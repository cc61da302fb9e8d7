"""Mints tests/golden/ref_ceres_*.npz from the REFERENCE'S OWN Ceres residual functor:
CPhotoconsistencyOdometryCeres.h:156-269 + third_party/sample.h + third_party/jet_extras.h,
compiled unmodified into oracle/_ref/libphovo_ref.so against the ceres::Jet / ceres::Problem
stand-ins of oracle/shim/ceres (Ceres itself is not installed here; see oracle/shim/ceres/jet.h for
what the stand-in assumes).  Run in the build container (needs /root/reference):

    python tests/golden/make_reference_ceres_golden.py

ref_ceres_640x480_cfg5.npz: BASELINE configs[2] -- config_5_level_optimization_ceres on a 640x480
pair.  For each of the 5 levels and each of 3 states: J^T J (21), J^T r (6), cost and the number of
non-zero residual slots formed from the functor's full output, and the functor's residual +
1x6 Jacobian themselves on a subset of target slots (the whole level for the two coarsest levels;
for the finer ones the two outermost rows / columns on every side -- where sample.h:36-49 clamps and
extrapolates -- plus a seeded random sample), of which a seeded quarter is stored so that the file
stays under 1 MB.  State 0 is the IDENTITY the apps start from
(every projected coordinate on an integer, CE:250-251 truncates), states 1 and 2 lie along the way.
"""
import importlib
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import ref_py  # noqa: E402

phovo = importlib.import_module("photoconsistency-visual-odometry_b200")

IDX = [(a, b) for a in range(6) for b in range(a, 6)]
KEEP = 0.25   # share of the sampled slots whose residual + Jacobian are stored
STATES = np.array([np.zeros(6),
                   [0.004, -0.003, 0.006, 0.003, -0.002, 0.0015],
                   [0.0195, -0.0102, 0.0153, 0.0099, -0.0081, 0.0061]])


def level_shapes(rows, cols, levels):
    import oracle_py
    return [oracle_py.level_size(rows, cols, l) for l in range(levels)]


def sample_slots(shape, n_random, seed, full_below=2000):
    r, c = shape
    if r * c <= full_below:
        return np.arange(r * c, dtype=np.int32)
    m = np.zeros(shape, bool)
    m[:2] = m[-2:] = True
    m[:, :2] = m[:, -2:] = True
    rng = np.random.default_rng(seed)
    m.ravel()[rng.choice(r * c, n_random, replace=False)] = True
    return np.flatnonzero(m.ravel()).astype(np.int32)


def normal_equations(res, jac):
    H = np.array([np.dot(jac[:, a], jac[:, b]) for a, b in IDX])
    return H, jac.T @ res, 0.5 * float(res @ res)


def main():
    rows, cols, seed, cfg = 480, 640, 51, "config_5_level_optimization_ceres"
    K = phovo.synth.K_FRAME_ALIGNMENT
    g0, d0, g1, _ = phovo.synth.make_pair(rows, cols, K=K, seed=seed)
    yml = phovo.configs.write_yaml(cfg, tempfile.mkdtemp())
    ref = ref_py.ReferenceCeres(yml, K)
    ref.set_frames(g0, d0, g1)
    out = dict(gray0=g0, depth0=d0.astype(np.float32), gray1=g1, K=K, config=np.array(cfg), states=STATES)
    for lvl, shape in enumerate(level_shapes(rows, cols, 5)):
        idx = sample_slots(shape, [1000, 800, 600, 600, 0][lvl], 100 + lvl)
        idx = np.sort(np.random.default_rng(200 + lvl).choice(idx, size=int(round(KEEP * len(idx))), replace=False))
        out["idx%d" % lvl] = idx
        for s, st in enumerate(STATES):
            res, jac = ref.evaluate(shape, st)
            res_d, _ = ref.evaluate(shape, st, want_jacobian=False)
            res = res.ravel()
            H, g, cost = normal_equations(res, jac)
            tag = "_l%d_s%d" % (lvl, s)
            out["H" + tag], out["g" + tag], out["cost" + tag] = H, g, np.array(cost)
            out["nnz" + tag] = np.array(int(np.count_nonzero(res)))
            out["res" + tag], out["jac" + tag] = res[idx], jac[idx]
            # the functor on T = double (cost-only evaluations): same scatter away from the identity
            out["nnz_double" + tag] = np.array(int(np.count_nonzero(res_d)))
            out["cost_double" + tag] = np.array(0.5 * float(res_d.ravel() @ res_d.ravel()))
            print("level", lvl, shape, "state", s, "non-zero slots", out["nnz" + tag], "(T=double:", out["nnz_double" + tag], ") cost", cost)
    np.savez_compressed(os.path.join(HERE, "ref_ceres_640x480_cfg5.npz"), **out)
    print("ref_ceres_640x480_cfg5.npz", os.path.getsize(os.path.join(HERE, "ref_ceres_640x480_cfg5.npz")) // 1024, "KiB")


if __name__ == "__main__":
    main()
