"""SURVEY row a10 pinned on the REFERENCE'S OWN residual functor.

oracle/_ref/libphovo_ref.so now also holds CPhotoconsistencyOdometryCeres.h (CE:156-269) with
third_party/sample.h and third_party/jet_extras.h, compiled UNMODIFIED from /root/reference against
the ceres::Jet / ceres::Problem stand-ins of oracle/shim/ceres (Ceres is not installed in this image).
The stand-in AutoDiffCostFunction evaluates the reference functor on T = double and on
T = Jet<double,6>, as Ceres' autodiff does.

  * live (wherever the library was built or travelled): the oracle's closed-form restatement equals
    the functor -- residuals bit for bit, Jacobians to 1e-13 -- on fresh pairs, every level, INCLUDING
    the identity state (every coordinate on an integer: the Jet quotient's rounding decides the slot);
    and the oracle's restated LM run on the reference functor ends where the oracle does;
  * committed fixture tests/golden/ref_ceres_640x480_cfg5.npz (tests/golden/make_reference_ceres_golden.py):
    BASELINE configs[2] at its full size; the oracle on CPU and K5 on the GPU are checked against it.

Still unpinned, and said so: the trajectory of Ceres' own trust-region minimiser (ceres::Solve is
third-party and absent; oracle and device run a restatement of its documented algorithm).
"""
import os

import numpy as np
import pytest

from helpers import GOLDEN, g_rel_err, h_rel_err
from test_gpu_parity import conv_cfg, make_odo

NAME = "ref_ceres_640x480_cfg5"
N_LEVELS, N_STATES = 5, 3


def golden():
    return dict(np.load(os.path.join(GOLDEN, NAME + ".npz")))


def padded_yaml(phovo, name, directory):
    """The reference's ceres configs list 4 min_trust_region_radius values for 5 levels (the reference
    then reads past the vector, CE:473): write every per-level list at full length."""
    v = dict(phovo.configs._lookup(name))
    n = v[phovo.configs.K_LEVELS]
    for k, val in list(v.items()):
        if isinstance(val, (list, tuple)) and len(val) < n:
            v[k] = list(val) + [val[-1]] * (n - len(val))
    path = os.path.join(directory, name + "_padded.yml")
    with open(path, "w") as f:
        f.write(phovo.configs.to_yaml(v))
    return path


def check_against_golden(gd, lvl, s, res, jac, H, g, cost, tol_jac, tol_res):
    tag = "_l%d_s%d" % (lvl, s)
    idx = gd["idx%d" % lvl]
    rg, jg = gd["res" + tag], gd["jac" + tag]
    assert np.max(np.abs(res.ravel()[idx] - rg)) <= tol_res
    # same scatter: a slot holds a residual here iff it does in the reference (CE:253-254 truncation, CE:261)
    assert np.array_equal(np.abs(res.ravel()[idx]) > 1e-9, np.abs(rg) > 1e-9)
    assert np.max(np.abs(jac[idx] - jg)) <= tol_jac * np.max(np.abs(jg))
    assert h_rel_err(H, gd["H" + tag]) < 1e-11 and g_rel_err(g, gd["g" + tag]) < 1e-11
    assert abs(cost - float(gd["cost" + tag])) <= 1e-12 * float(gd["cost" + tag])


def test_golden_exercises_the_sampler_edge_cases():
    """The fixture holds rows in the first half pixel (sample.h:36-49: ix = (int)x truncates towards 0, so
    x in [-0.5, 0) extrapolates with dx in (1, 1.5]) and on the last row / column clamp."""
    gd = golden()
    assert str(gd["config"]) == "config_5_level_optimization_ceres" and gd["gray0"].shape == (480, 640)
    for lvl in range(N_LEVELS):
        rows, cols = gd["gray0"].shape[0] >> lvl, gd["gray0"].shape[1] >> lvl
        idx = gd["idx%d" % lvl]
        r, c = idx // cols, idx % cols
        hit = np.zeros(4, bool)
        for s in range(N_STATES):
            nz = gd["res_l%d_s%d" % (lvl, s)] != 0
            hit |= [np.any(nz & (r == 0)), np.any(nz & (c == 0)), np.any(nz & (r == rows - 1)), np.any(nz & (c == cols - 1))]
        assert hit.all(), (lvl, hit)       # truncated slots of t < 1, and the clamp at the far edge
    # at the identity the two instantiations of the functor scatter differently, away from it they agree
    assert int(gd["nnz_l0_s0"]) != int(gd["nnz_double_l0_s0"])
    assert abs(int(gd["nnz_l0_s2"]) - int(gd["nnz_double_l0_s2"])) <= 2


def test_oracle_ceres_matches_reference_golden(phovo, oracle):
    gd = golden()
    cfg = phovo.configs.to_config(str(gd["config"]), phovo.capi)
    o = oracle.Oracle(conv_cfg(oracle, cfg), gd["K"])
    o.set_source(gd["gray0"], gd["depth0"].astype(np.float64))
    o.set_target(gd["gray1"])
    for lvl in range(N_LEVELS):
        for s, st in enumerate(gd["states"]):
            r = o.eval(lvl, st, want_residuals=True, want_jacobian=True)
            check_against_golden(gd, lvl, s, r["residuals"], r["jacobian"], r["H"], r["g"], r["cost"], 1e-13, 0.)
            assert int(np.count_nonzero(r["residuals"])) == int(gd["nnz_l%d_s%d" % (lvl, s)])


@pytest.mark.parametrize("cfg_name,shape,seed", [
    ("config_5_level_optimization_ceres", (480, 640), 61),
    ("config_4_level_optimization_ceres", (135, 241), 62),
    ("config_3_level_optimization_ceres", (96, 128), 63),     # blur 3 at level 2
])
def test_oracle_ceres_matches_reference_functor_live(phovo, oracle, tmp_path, cfg_name, shape, seed):
    import ref_py
    if not ref_py.available():
        pytest.skip("oracle/_ref not built: set REF to a checkout of the original project")
    K = phovo.synth.K_FRAME_ALIGNMENT.copy()
    K[:2] *= shape[1] / 640.
    g0, d0, g1, _ = phovo.synth.make_pair(shape[0], shape[1], K=K, seed=seed)
    ref = ref_py.ReferenceCeres(padded_yaml(phovo, cfg_name, str(tmp_path)), K)
    ref.set_frames(g0, d0, g1)
    cfg = phovo.configs.to_config(cfg_name, phovo.capi)
    o = oracle.Oracle(conv_cfg(oracle, cfg), K)
    o.set_source(g0, d0)
    o.set_target(g1)
    rng = np.random.default_rng(seed)
    states = [np.zeros(6), phovo.synth.XI_CONFIG1 * 0.4, rng.uniform(-0.02, 0.02, 6) * [1, 1, 1, .5, .5, .5]]
    for lvl in range(cfg.num_levels):
        if cfg.max_num_iterations[lvl] <= 0:
            continue
        lshape = o.level_image(0, lvl).shape
        for st in states:
            res, jac = ref.evaluate(lshape, st)
            r = o.eval(lvl, st, want_residuals=True, want_jacobian=True)
            assert np.array_equal(res.ravel(), r["residuals"])                       # bit for bit, scatter included
            assert np.max(np.abs(jac - r["jacobian"])) <= 1e-13 * np.max(np.abs(jac))
    # closed loop: the restated LM on the reference functor vs the oracle, from the apps' identity start
    s_ref, log_ref = ref.optimize()
    o.set_initial_state(np.zeros(6))
    o.optimize()
    log = o.iter_stats()
    assert [e["accepted"] for e in log] == [e["accepted"] for e in log_ref] and len(log) > 0
    for a, b in zip(log, log_ref):
        assert abs(a["cost"] - b["cost"]) <= 1e-11 * b["cost"]
        assert h_rel_err(a["H"], b["H"]) < 1e-11 and g_rel_err(a["g"], b["g"]) < 1e-10
    assert np.max(np.abs(o.state() - s_ref)) < 1e-11


@pytest.mark.gpu
def test_cuda_ceres_matches_reference_golden(phovo):
    """K5 (k_normal_eq<2>) against outputs of the reference functor at BASELINE configs[2]'s size: all 5
    levels, 3 states incl. the identity, residual + 1x6 Jacobian per sampled slot (incl. the
    extrapolation band of sample.h:36-49 and the truncation scatter CE:253-254), J^T J, J^T r, cost."""
    gd = golden()
    cfg = phovo.configs.to_config(str(gd["config"]), phovo.capi)
    odo = make_odo(phovo, cfg, gd["K"])
    odo.SetSourceFrame(gd["gray0"], gd["depth0"])
    odo.SetTargetFrame(gd["gray1"])
    for lvl in range(N_LEVELS):
        shape = odo.LevelImage(0, lvl).shape
        for s, st in enumerate(gd["states"]):
            res, jac = odo.EvalResiduals(lvl, st, shape)
            e = odo.EvalNormalEquations(lvl, st)
            check_against_golden(gd, lvl, s, res, jac, e["H"], e["g"], e["cost"], 1e-11, 1e-13)
            if s > 0:   # (at the identity many residuals are differences of equal pixels: 0 or rounding noise)
                assert abs(int(np.count_nonzero(np.abs(res) > 1e-12)) - int(gd["nnz_l%d_s%d" % (lvl, s)])) <= 64


@pytest.mark.gpu
def test_cuda_ceres_matches_reference_functor_live(phovo, tmp_path):
    """Whole levels, not samples: K5 against the reference functor run on the spot (the prebuilt
    oracle/_ref library travels to the GPU box)."""
    import ref_py
    if not ref_py.available():
        pytest.skip("oracle/_ref library not present on this box")
    K = phovo.synth.K_FRAME_ALIGNMENT
    g0, d0, g1, _ = phovo.synth.make_pair(480, 640, K=K, seed=64)
    name = "config_5_level_optimization_ceres"
    ref = ref_py.ReferenceCeres(padded_yaml(phovo, name, str(tmp_path)), K)
    ref.set_frames(g0, d0, g1)
    cfg = phovo.configs.to_config(name, phovo.capi)
    odo = make_odo(phovo, cfg, K)
    odo.SetSourceFrame(g0, d0)
    odo.SetTargetFrame(g1)
    for lvl in range(cfg.num_levels):
        shape = odo.LevelImage(0, lvl).shape
        for st in (np.zeros(6), phovo.synth.XI_CONFIG1 * 0.7):
            res_ref, jac_ref = ref.evaluate(shape, st)
            res_ref = res_ref.ravel()
            res, jac = odo.EvalResiduals(lvl, st, shape)
            assert np.array_equal(np.abs(res) > 1e-9, np.abs(res_ref) > 1e-9)          # same scatter, also at the identity
            assert np.max(np.abs(res - res_ref)) <= 1e-13
            assert np.max(np.abs(jac - jac_ref)) <= 1e-11 * np.max(np.abs(jac_ref))
    # closed loop at the stated size of BASELINE configs[2]: the CUDA LM (cooperative kernel and a wave of slots) against
    # "the reference functor under the restated LM" -- every LM decision (accepted / rejected steps) and the final state
    s_ref, log_ref = ref.optimize()
    odo.SetInitialStateVector(np.zeros(6))
    odo.Optimize()
    log = odo.IterationStats()
    assert len(log) == len(log_ref) > 0
    assert [e["accepted"] for e in log] == [e["accepted"] for e in log_ref]
    assert np.max(np.abs(odo.GetOptimalStateVector() - s_ref)) < 1e-10
    odo.BatchSetDebugFlags(8)
    st, it = odo.BatchAlign(g0[None], d0[None], g1[None])
    assert odo.BatchLastPath() == 3 and int(it.sum()) == len(log_ref)
    assert np.max(np.abs(st[0] - s_ref)) < 1e-10
