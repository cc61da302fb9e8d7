"""The float64 restatement of the photometric + depth solver (oracle/bi_restatement.py) against the reference's own
outputs, tests/golden/ref_bi_*.npz, on the CPU.  The GPU tests of that solver (test_gpu_biobjective_restatement.py)
take the restatement as their reference, so it is pinned here first, and the negative cases show that the fixtures
tell its two aliasing rules apart."""
import glob
import importlib
import os

import numpy as np
import pytest

from helpers import GOLDEN, g_rel_err, h_rel_err

FIXTURES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "ref_bi_*.npz")))


def restate(name, rules="reference"):
    import bi_restatement
    import oracle_py
    configs = importlib.import_module("photoconsistency-visual-odometry_b200.configs")
    gd = dict(np.load(os.path.join(GOLDEN, name + ".npz")))
    cfg = configs.to_config(str(gd["config"]), oracle_py, mode=3)
    lv = bi_restatement.BiLevels(cfg, gd["K"], gd["gray0"], gd["depth0"], gd["gray1"], gd["depth1"])
    s, log = bi_restatement.optimize(lv, np.zeros(6), rules)
    return gd, lv, s, log


def worst_errors(gd, log):
    iu = np.triu_indices(6)
    eh = max(h_rel_err(e["H"], H[iu]) for e, H in zip(log, gd["H"]))
    eg = max(g_rel_err(e["g"], g) for e, g in zip(log, gd["g"]))
    return eh, eg


@pytest.mark.parametrize("name", FIXTURES)
def test_restatement_reproduces_reference_fixture(name):
    assert len(FIXTURES) >= 2
    gd, lv, s, log = restate(name)
    assert len(log) == len(gd["n"])
    for e, n in zip(log, gd["n"]):
        # the fixtures' n is the reference's row count 2N of the iteration's level
        assert 2 * lv.levels[e["level"]]["I0"].size == n
        assert 0 < e["num_valid"] <= n // 2
    eh, eg = worst_errors(gd, log)
    assert eh <= 1e-10 and eg <= 1e-10, (eh, eg)
    assert np.max(np.abs(s - gd["state"])) <= 1e-12


@pytest.mark.parametrize("rules", ["no_row0_rule", "swapped_keys"])
@pytest.mark.parametrize("name", FIXTURES)
def test_fixtures_reject_a_restatement_with_a_wrong_aliasing_rule(name, rules):
    """Row 0 taken by pixel 0's intensity row instead of its depth row, or depth writes beating intensity writes of the
    same pixel: either must fail the comparison the reference restatement passes."""
    gd, _, s, log = restate(name, rules)
    eh, eg = worst_errors(gd, log)
    assert len(log) != len(gd["n"]) or eh > 1e-8 or eg > 1e-8 or np.max(np.abs(s - gd["state"])) > 1e-10


def test_restatement_aliasing_rules_on_a_small_level():
    """The write-order rules spelled out on one evaluation: residual slot s holds the write with the largest key, row
    k of the Jacobian the last of pixel k's intensity row and pixel k/2's depth row; pixel 0's depth row owns row 0."""
    import bi_restatement
    gd, lv, _, _ = restate(FIXTURES[0])
    level = max(lv.levels)
    e = bi_restatement.evaluate(lv.levels[level], lv.K, level, np.array([0.01, -0.02, 0.01, 0.01, 0.02, -0.01]))
    N = lv.levels[level]["I0"].size
    valid = e["valid"]
    for k in range(2 * N):
        vk = k < N and valid[k]
        vh = k % 2 == 0 and valid[k >> 1]
        want = 2 * k if (vk and k > 0) else (k + 1 if vh else -1)
        assert e["row_owner"][k] == want, k
    assert (e["J"][e["row_owner"] < 0] == 0).all() and (e["res"][e["keys"] == 0] == 0).all()
    assert e["num_valid"] == int(valid.sum())
    assert e["cost"] == pytest.approx(0.5 * float(e["res"] @ e["res"]), rel=1e-15)
