"""Parity pinned on the REFERENCE'S OWN SOURCE.

oracle/_ref/libphovo_ref.so is the reference's CPhotoconsistencyOdometryAnalytic.h compiled unmodified
from /root/reference against stand-ins for OpenCV/Eigen (oracle/shim; the image arithmetic behind
the stand-ins is the oracle's, pinned against the real OpenCV in test_oracle_pins.py).  Everything
first-party -- the per-pixel loop with its temp1..26 Jacobian, the residual scatter, the
Gauss-Newton update, TestTerminationCriteria, the YAML reader calls -- is the reference's code.

  * live (build container / wherever the prebuilt library travelled): oracle == reference on fresh
    random pairs, for every analytic reference config;
  * committed fixtures tests/golden/ref_*.npz (minted by tests/golden/make_reference_golden.py from
    that library): the oracle (CPU) and the CUDA path (GPU) are checked against them.
"""
import glob
import os

import numpy as np
import pytest

from helpers import GOLDEN, REL_NORMAL_EQ, assert_pose_close, g_rel_err, h_rel_err
from test_gpu_parity import conv_cfg, make_odo

REF_FIXTURES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "ref_pair_*.npz")))
IDX = [(a, b) for a in range(6) for b in range(a, 6)]


def pack(H):
    return np.array([H[i, j] for i, j in IDX])


def run_oracle(phovo, oracle, cfg_name, K, g0, d0, g1):
    cfg = phovo.configs.to_config(cfg_name, phovo.capi)
    o = oracle.Oracle(conv_cfg(oracle, cfg), K)
    o.set_source(g0, d0)
    o.set_target(g1)
    o.set_initial_state(np.zeros(6))
    o.optimize()
    return o


def test_fixtures_exist():
    assert len(REF_FIXTURES) >= 4


@pytest.mark.parametrize("name", REF_FIXTURES)
def test_oracle_matches_reference_golden(phovo, oracle, name):
    gd = dict(np.load(os.path.join(GOLDEN, name + ".npz")))
    o = run_oracle(phovo, oracle, str(gd["config"]), gd["K"], gd["gray0"], gd["depth0"].astype(np.float64), gd["gray1"])
    log = o.iter_stats()
    assert len(log) == len(gd["n"])                       # executed iterations (data dependent)
    for e, n, H, g in zip(log, gd["n"], gd["H"], gd["g"]):
        lr, lc = o.level_image(0, e["level"]).shape
        assert lr * lc == n
        # same doubles summed in a different order at most: far below the 1e-5 bar
        assert h_rel_err(e["H"], pack(H)) < 1e-12 and g_rel_err(e["g"], g) < 1e-12
    assert np.max(np.abs(o.state() - gd["state"])) < 1e-12
    assert np.max(np.abs(o.rt() - gd["rt"])) < 1e-12


@pytest.mark.parametrize("cfg_name,shape,K_name", [
    ("config_4_level_optimization_analytic", (480, 640), "K_FRAME_ALIGNMENT"),
    ("config_5_level_optimization_analytic", (480, 640), "K_VISUAL_ODOMETRY"),
    ("config_6_level_optimization_analytic", (270, 480), "K_FRAME_ALIGNMENT"),
    ("test_3_level_all_active", (101, 77), "K_FRAME_ALIGNMENT"),
])
def test_oracle_matches_reference_source_live(phovo, oracle, tmp_path, cfg_name, shape, K_name):
    import ref_py
    if not ref_py.available():
        pytest.skip("oracle/_ref not built: set REF to a checkout of the original project")
    K = getattr(phovo.synth, K_name).copy()
    if shape != (480, 640):
        K[:2] *= shape[1] / 640.
    yml = phovo.configs.write_yaml(cfg_name, str(tmp_path))
    ref = ref_py.Reference(yml, K)
    for seed in (41, 42):
        g0, d0, g1, _ = phovo.synth.make_pair(shape[0], shape[1], K=K, seed=seed)
        s, rt, iters = ref.align(g0, d0, g1)
        o = run_oracle(phovo, oracle, cfg_name, K, g0, d0, g1)
        log = o.iter_stats()
        assert len(log) == len(iters) and len(log) > 0
        for e, it in zip(log, iters):
            assert h_rel_err(e["H"], pack(it["H"])) < 1e-12 and g_rel_err(e["g"], it["g"]) < 1e-12
        assert np.max(np.abs(o.state() - s)) < 1e-12
        assert np.max(np.abs(o.rt() - rt)) < 1e-12


@pytest.mark.gpu
@pytest.mark.parametrize("name", REF_FIXTURES)
def test_cuda_matches_reference_golden(phovo, name):
    """The CUDA path against outputs of the reference's own code: normal equations per executed
    iteration within 1e-5 relative (north star), identical iteration counts, pose within
    1e-4 m / 1e-5 rad -- and in fact ten orders tighter."""
    gd = dict(np.load(os.path.join(GOLDEN, name + ".npz")))
    cfg = phovo.configs.to_config(str(gd["config"]), phovo.capi)
    odo = make_odo(phovo, cfg, gd["K"])
    odo.SetSourceFrame(gd["gray0"], gd["depth0"])
    odo.SetTargetFrame(gd["gray1"], None)
    odo.SetInitialStateVector(np.zeros(6))
    odo.Optimize()
    log = odo.IterationStats()
    assert len(log) == len(gd["n"])
    for e, H, g in zip(log, gd["H"], gd["g"]):
        assert h_rel_err(e["H"], pack(H)) < REL_NORMAL_EQ and g_rel_err(e["g"], g) < REL_NORMAL_EQ
        assert h_rel_err(e["H"], pack(H)) < 1e-11 and g_rel_err(e["g"], g) < 1e-10
    assert_pose_close(odo.GetOptimalStateVector(), gd["state"], name)
    assert np.max(np.abs(odo.GetOptimalStateVector() - gd["state"])) < 1e-10
    assert np.max(np.abs(odo.GetOptimalRigidTransformationMatrix() - gd["rt"])) < 1e-10
    # the batch entry on the same pair: the shared-memory-resident kernels when its levels fit, else (one pair) the pool
    st, it = odo.BatchAlign(gd["gray0"][None], gd["depth0"][None], gd["gray1"][None])
    assert odo.BatchLastPath() in (1, 2)
    assert int(it.sum()) == len(gd["n"])
    assert_pose_close(st[0], gd["state"], name + " (batch)")
    assert np.max(np.abs(st[0] - gd["state"])) < 1e-10
