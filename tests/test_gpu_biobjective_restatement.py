"""The photometric + depth solver (PHOVO_MODE_BIOBJECTIVE) against the float64 restatement of
oracle/bi_restatement.py, which test_bi_restatement.py pins to the reference's own outputs.

Every driver that runs this solver is checked on the same pairs: the per-pair Optimize with plain stream launches,
the CUDA graph and the cooperative kernel (SetExecution 0 / 1 / 2 / 3), and the batch entry through the waves of
per-pair slots (one CTA or a 2 / 4 / 8-CTA cluster per pair) and through the pool of per-pair contexts.  The
single evaluations (EvalNormalEquations, EvalResiduals with its 2N rows) are checked slot by slot and row by row at
states chosen to exercise the row and slot aliasing of the reference's stacked system."""
import numpy as np
import pytest

import bi_restatement as br
from helpers import g_rel_err, h_rel_err

pytestmark = pytest.mark.gpu

U16_SCALE = 1. / 5000.


def intrinsics(phovo, rows, cols, off_centre):
    """The app's K scaled to the frame; the off-centre set also has fx != fy."""
    K = phovo.synth.K_FRAME_ALIGNMENT.copy()
    f = 525. * cols / 640.
    K[0, 0], K[1, 1], K[0, 2], K[1, 2] = f, f, (cols - 1) / 2., (rows - 1) / 2.
    if off_centre:
        K[1, 1], K[0, 2], K[1, 2] = 1.04 * f, 0.41 * cols + 0.25, 0.58 * rows - 0.5
    return K


def as_type(d, kind):
    """metres (f64) -> the caller's depth type; u16 is raw * U16_SCALE"""
    if kind == "u16":
        return np.clip(np.rint(d / U16_SCALE), 0, 65535).astype(np.uint16)
    return d.astype(np.float32) if kind == "f32" else d.copy()


def make_cfg(phovo, name):
    if name in ("blur", "zero_middle"):
        cfg = phovo.configs.to_config("test_3_level_all_active", phovo.capi, mode=phovo.MODE_BIOBJECTIVE)
        if name == "blur":
            for l, b in enumerate((3, 0, 5)):
                cfg.blur_filter_size[l] = b
        else:                                                  # level 1 does nothing; the run starts off zero
            for l, (m, lam) in enumerate(((4, 1.), (0, 1.), (6, 0.7))):
                cfg.max_num_iterations[l], cfg.lambda_step[l], cfg.min_gradient_norm[l] = m, lam, 1e-3
        return cfg
    return phovo.configs.to_config(name, phovo.capi, mode=phovo.MODE_BIOBJECTIVE)


def make_pair(phovo, shape, K, seed, t0, t1):
    rows, cols = shape
    g0, d0, g1, d1 = phovo.synth.make_pair(rows, cols, K=K, xi=phovo.synth.random_motion(seed), seed=seed, depth_f32=False)
    return g0, as_type(d0, t0), g1, as_type(d1, t1)


def initial_state(phovo, seed, nonzero):
    return 0.5 * phovo.synth.random_motion(500 + seed) if nonzero else np.zeros(6)


def new_odo(phovo, cfg, K):
    odo = phovo.CPhotoconsistencyOdometryCuda()
    odo.SetConfig(cfg)
    odo.SetIntrinsicMatrix(K)
    return odo


def optimize(phovo, odo, g0, d0, g1, d1, s0, expect_numeric=False):
    odo.SetSourceFrame(g0, d0, depth_scale=U16_SCALE)
    odo.SetTargetFrame(g1, d1, depth_scale=U16_SCALE)
    odo.SetInitialStateVector(s0)
    if expect_numeric:
        with pytest.raises(phovo.PhovoError) as e:
            odo.Optimize()
        assert e.value.code == phovo.capi.E_NUMERIC
    else:
        odo.Optimize()
    return odo.GetOptimalStateVector(), odo.IterationStats()


def assert_log_matches(log, ref, what):
    assert [(e["level"], e["iteration"]) for e in log] == [(e["level"], e["iteration"]) for e in ref], what
    for a, b in zip(log, ref):
        w = (what, a["level"], a["iteration"])
        assert a["num_valid"] == b["num_valid"], w
        assert h_rel_err(a["H"], b["H"]) < 1e-9, (w, h_rel_err(a["H"], b["H"]))
        assert g_rel_err(a["g"], b["g"]) < 1e-8, (w, g_rel_err(a["g"], b["g"]))
        assert abs(a["cost"] - b["cost"]) <= 1e-10 * abs(b["cost"]), (w, a["cost"], b["cost"])
        assert np.max(np.abs(a["state_in"] - b["state_in"])) < 1e-9, w
        assert np.max(np.abs(a["state_out"] - b["state_out"])) < 1e-9, w


def iterations_per_level(log):
    it = np.zeros(10, np.int32)
    for e in log:
        it[e["level"]] += 1
    return it


# (shape, configuration, source depth, target depth, off-centre K, seed, non-zero initial state).  Half of an odd size
# rounds to even, so no frame is odd at every level: the three levels of 107x203 are 107x203, 54x102 and 27x51 (odd at
# levels 0 and 2), those of 106x150 are 106x150, 53x75 and 26x38 (odd at level 1).  15x21 ends in a 4x5 level (smaller
# coarse levels leave the normal equations singular).
CASES = {
    "480x640-cfg4-f32": ((480, 640), "config_4_level_optimization_analytic", "f32", "f32", False, 0, False),
    "480x640-all-u16": ((480, 640), "test_3_level_all_active", "u16", "u16", True, 1, False),
    "480x640-blur-f64-f32": ((480, 640), "blur", "f64", "f32", False, 2, False),
    "480x640-zeromid-f32-f64": ((480, 640), "zero_middle", "f32", "f64", True, 3, True),
    "135x241-all-f32-u16": ((135, 241), "test_3_level_all_active", "f32", "u16", True, 4, False),
    "135x241-cfg4-f64": ((135, 241), "config_4_level_optimization_analytic", "f64", "f64", False, 5, False),
    "135x241-zeromid-u16-f64": ((135, 241), "zero_middle", "u16", "f64", False, 6, True),
    "107x203-all-f64-u16": ((107, 203), "test_3_level_all_active", "f64", "u16", True, 7, False),
    "107x203-blur-u16-f32": ((107, 203), "blur", "u16", "f32", True, 8, False),
    "106x150-all-f32": ((106, 150), "test_3_level_all_active", "f32", "f32", False, 9, True),
    "15x21-all-f32": ((15, 21), "test_3_level_all_active", "f32", "f32", False, 10, False),
    "15x21-zeromid-u16-f64": ((15, 21), "zero_middle", "u16", "f64", True, 11, True),
}


@pytest.mark.parametrize("case", list(CASES))
def test_optimize_matches_restatement_on_every_driver(phovo, case):
    shape, cfg_name, t0, t1, off, seed, nonzero = CASES[case]
    cfg = make_cfg(phovo, cfg_name)
    K = intrinsics(phovo, *shape, off)
    g0, d0, g1, d1 = make_pair(phovo, shape, K, seed, t0, t1)
    s0 = initial_state(phovo, seed, nonzero)
    sref, ref = br.optimize(br.BiLevels(cfg, K, g0, d0, g1, d1, U16_SCALE), s0)
    assert len(ref) > 0 and np.isfinite(sref).all()
    odo = new_odo(phovo, cfg, K)
    out = {}
    for ex in (0, 1, 2, 3):
        odo.SetExecution(ex)
        s, log = optimize(phovo, odo, g0, d0, g1, d1, s0)
        if ex < 3:
            assert odo.LastPath() == ex, (case, ex, odo.GraphError())
        assert_log_matches(log, ref, (case, ex))
        assert np.max(np.abs(s - sref)) < 1e-9, (case, ex)
        out[ex] = (s, log)
    # the cluster driver does not take this solver: SetExecution(3) runs the cooperative kernel, bit for bit
    assert np.array_equal(out[3][0], out[2][0])
    for a, b in zip(out[3][1], out[2][1]):
        assert np.array_equal(a["H"], b["H"]) and np.array_equal(a["g"], b["g"]) and a["cost"] == b["cost"]
    odo.close()


# ---------------------------------------------------------------------------------------------
# batch entry: distinct pairs, each with its own target depth and initial state
BATCHES = {
    "135x241-all-u16": ((135, 241), "test_3_level_all_active", "u16", True, 20),
    "107x203-blur-f32": ((107, 203), "blur", "f32", False, 30),
    "480x640-cfg4-f64": ((480, 640), "config_4_level_optimization_analytic", "f64", False, 40),
    "15x21-zeromid-f32": ((15, 21), "zero_middle", "f32", True, 50),
}


def make_batch(phovo, shape, kind, K, seed0, P):
    pairs = [make_pair(phovo, shape, K, seed0 + p, kind, kind) for p in range(P)]
    g0, d0, g1, d1 = (np.stack([q[k] for q in pairs]) for k in range(4))
    init = np.stack([initial_state(phovo, seed0 + p, p % 2 == 1) for p in range(P)])
    return g0, d0, g1, d1, init


@pytest.mark.parametrize("batch", list(BATCHES))
def test_batch_matches_restatement_pair_by_pair(phovo, monkeypatch, batch):
    shape, cfg_name, kind, off, seed0 = BATCHES[batch]
    P = 5
    cfg = make_cfg(phovo, cfg_name)
    K = intrinsics(phovo, *shape, off)
    g0, d0, g1, d1, init = make_batch(phovo, shape, kind, K, seed0, P)
    refs = [br.optimize(br.BiLevels(cfg, K, g0[p], d0[p], g1[p], d1[p], U16_SCALE), init[p]) for p in range(P)]
    perm = np.array([3, 0, 4, 2, 1])
    odo = new_odo(phovo, cfg, K)
    runs = [("waves", 8, c) for c in ("1", "2", "4", "8")] + [("pool", 4, None)]
    for what, flags, cluster in runs:
        if cluster is None:
            monkeypatch.delenv("PHOVO_WAVE_CLUSTER", raising=False)
        else:
            monkeypatch.setenv("PHOVO_WAVE_CLUSTER", cluster)
        odo.BatchSetDebugFlags(flags)
        st, it = odo.BatchAlign(g0, d0, g1, init, depth_scale=U16_SCALE, depth1=d1)
        assert odo.BatchLastPath() == (3 if what == "waves" else 2), what
        for p, (sref, log) in enumerate(refs):
            assert np.array_equal(it[p], iterations_per_level(log)), (batch, what, cluster, p, it[p])
            assert np.max(np.abs(st[p] - sref)) < 1e-9, (batch, what, cluster, p)
        # the result of a pair does not depend on where it sits in the batch
        st2, it2 = odo.BatchAlign(g0[perm], d0[perm], g1[perm], init[perm], depth_scale=U16_SCALE, depth1=d1[perm])
        assert np.array_equal(st2, st[perm]) and np.array_equal(it2, it[perm]), (batch, what, cluster)
    monkeypatch.delenv("PHOVO_WAVE_CLUSTER", raising=False)
    odo.BatchSetDebugFlags(0)
    odo.close()


# ---------------------------------------------------------------------------------------------
# single evaluations at given states
EVAL_STATES = {
    "identity": np.zeros(6),                                                   # t(i) = i: slot 2i is pixel 2i's and pixel i's
    "motion": np.array([0.03, -0.02, 0.04, 0.015, -0.02, 0.01]),
    "zoom_out": np.array([0.05, -0.03, 6.0, 0.01, 0.02, -0.01]),              # every slot near the centre takes many pixels
    "rotated": np.array([-0.1, 0.08, -0.2, 0.06, -0.05, 0.04]),
}


def check_aliasing_is_exercised(name, e, N):
    t = e["target"][e["valid"]]
    assert (e["keys"][N:] > 0).any(), name                                    # depth slots 2 t >= N
    if name != "zoom_out":                                                    # (there every pixel lands near the centre)
        assert np.intersect1d(t, 2 * t).size > 0, name                       # an intensity and a depth write share a slot
    if name == "identity":
        assert e["valid"][0] and e["row_owner"][0] == 1                       # row 0 is pixel 0's depth row
        assert e["keys"][0] == 2                                              # and slot 0 its depth residual
    if name == "zoom_out":
        assert np.bincount(t).max() >= 8, np.bincount(t).max()


@pytest.mark.parametrize("shape,t0,t1,off", [((135, 241), "f32", "u16", True), ((107, 203), "u16", "f64", False),
                                            ((480, 640), "f64", "f32", True)])
def test_eval_normal_equations_and_residuals_match_restatement(phovo, shape, t0, t1, off):
    cfg = make_cfg(phovo, "test_3_level_all_active")
    K = intrinsics(phovo, *shape, off)
    g0, d0, g1, d1 = make_pair(phovo, shape, K, 60, t0, t1)
    d0[0, 0] = d0[1, 1] if d0[1, 1] else d0[2, 2]                             # pixel 0 valid: the row-0 rule applies
    lv = br.BiLevels(cfg, K, g0, d0, g1, d1, U16_SCALE)
    odo = new_odo(phovo, cfg, K)
    odo.SetSourceFrame(g0, d0, depth_scale=U16_SCALE)
    odo.SetTargetFrame(g1, d1, depth_scale=U16_SCALE)
    for level in range(3):
        rows, cols = lv.levels[level]["I0"].shape
        N = rows * cols
        for name, s in EVAL_STATES.items():
            e = br.evaluate(lv.levels[level], lv.K, level, s)
            check_aliasing_is_exercised(name, e, N)
            w = (shape, level, name)
            st = odo.EvalNormalEquations(level, s)
            assert st["num_valid"] == e["num_valid"], w
            assert h_rel_err(st["H"], br.pack_upper(e["H"])) < 1e-9 and g_rel_err(st["g"], e["g"]) < 1e-8, w
            assert abs(st["cost"] - e["cost"]) <= 1e-10 * e["cost"], w
            res, jac = odo.EvalResiduals(level, s, (rows, cols))
            assert res.shape == (2 * N,) and jac.shape == (2 * N, 6), w
            res2, jac2 = odo.EvalResiduals(level, s)                   # sized from the level the context built
            assert np.array_equal(res2, res) and np.array_equal(jac2, jac), w
            assert np.array_equal(res != 0, e["res"] != 0), (w, np.flatnonzero((res != 0) != (e["res"] != 0))[:10])
            assert np.array_equal((jac != 0).any(1), (e["J"] != 0).any(1)), w
            assert np.max(np.abs(res - e["res"])) <= 1e-12 * np.max(np.abs(e["res"])), w
            assert np.max(np.abs(jac - e["J"])) <= 1e-12 * np.max(np.abs(e["J"])), w
            assert st["cost"] == pytest.approx(0.5 * float(res @ res), rel=1e-12), w
        with pytest.raises(ValueError):                                # a shape that is not the level's is refused
            odo.EvalResiduals(level, EVAL_STATES["identity"], (rows, cols + 1))
    odo.close()


# ---------------------------------------------------------------------------------------------
# how the target depth arrives, and target depths that are not a clean depth map
def test_target_depth_inputs_give_the_same_results(phovo):
    import torch
    shape, kind = (135, 241), "u16"
    cfg = make_cfg(phovo, "test_3_level_all_active")
    K = intrinsics(phovo, *shape, True)
    g0, d0, g1, d1 = make_pair(phovo, shape, K, 70, kind, kind)
    s0 = initial_state(phovo, 70, True)
    sref, ref = br.optimize(br.BiLevels(cfg, K, g0, d0, g1, d1, U16_SCALE), s0)
    odo = new_odo(phovo, cfg, K)
    s, log = optimize(phovo, odo, g0, d0, g1, d1, s0)
    assert_log_matches(log, ref, "numpy")
    assert np.max(np.abs(s - sref)) < 1e-9

    def tensor(a):
        return torch.from_numpy(a.view(np.int16) if a.dtype == np.uint16 else a)
    wide = np.zeros((shape[0], shape[1] + 19), d1.dtype)
    wide[:, :shape[1]] = d1
    assert not wide[:, :shape[1]].flags.c_contiguous
    for what, t in (("strided", wide[:, :shape[1]]), ("pinned", tensor(d1).pin_memory()), ("device", tensor(d1).cuda())):
        s2, log2 = optimize(phovo, odo, g0, d0, g1, t, s0)
        torch.cuda.synchronize()
        assert np.array_equal(s2, s), what
        assert [(e["num_valid"], e["cost"]) for e in log2] == [(e["num_valid"], e["cost"]) for e in log], what
    # the batch entry: numpy, strided numpy, pinned and device inputs, and strided device views (the library reads dense
    # [P, rows, cols] frames; the wrapper copies views)
    P = 3
    bg0, bd0, bg1, bd1, init = make_batch(phovo, shape, kind, K, 80, P)

    def strided(a, device=False):                              # a view that starts inside a wider buffer
        wide = np.zeros((a.shape[0], a.shape[1] + 3, a.shape[2] + 11), a.dtype)
        inner = (slice(None), slice(2, 2 + a.shape[1]), slice(5, 5 + a.shape[2]))
        wide[inner] = a
        view = tensor(wide).cuda()[inner] if device else wide[inner]
        assert not (view.is_contiguous() if device else view.flags.c_contiguous)
        return view
    refs = [br.optimize(br.BiLevels(cfg, K, bg0[p], bd0[p], bg1[p], bd1[p], U16_SCALE), init[p])[0] for p in range(P)]
    for flags in (8, 4):
        odo.BatchSetDebugFlags(flags)
        st, it = odo.BatchAlign(bg0, bd0, bg1, init, depth_scale=U16_SCALE, depth1=bd1)
        for p in range(P):
            assert np.max(np.abs(st[p] - refs[p])) < 1e-9, (flags, p)
        for what, conv in (("strided", strided), ("pinned", lambda a: tensor(a).pin_memory()), ("device", lambda a: tensor(a).cuda()),
                           ("strided device", lambda a: strided(a, device=True))):
            args = [conv(a) for a in (bg0, bd0, bg1)]
            st2, it2 = odo.BatchAlign(*args, init, depth_scale=U16_SCALE, depth1=conv(bd1))
            torch.cuda.synchronize()
            assert np.array_equal(st2, st) and np.array_equal(it2, it), (flags, what)
    # one depth type is passed for both depths: a target depth of another type is refused, not misread
    with pytest.raises(TypeError):
        odo.BatchAlign(bg0, bd0, bg1, init, depth_scale=U16_SCALE, depth1=bd1.astype(np.float32))
    odo.BatchSetDebugFlags(0)
    odo.close()


def damaged(d1, how):
    d = d1.astype(np.float64)
    if how == "holes_and_out_of_range":
        d[10:30, 20:60] = 0.                                                   # a hole
        d[40:60, 100:140] = 7.5                                                # beyond max_depth
        d[-20:, :35] = -1.                                                     # negative
        d[70:75, :] = 0.25                                                     # below min_depth
    elif how == "all_zero":
        d[:] = 0.
    elif how == "nan":
        d[50, 60] = np.nan
    return d


@pytest.mark.parametrize("how", ["holes_and_out_of_range", "all_zero", "nan"])
def test_damaged_target_depth(phovo, how):
    """Holes and depths outside (min_depth, max_depth) are data like any other; an all-zero target depth (gain =
    mean(I1) / 0) or a NaN in it (gain NaN) makes the state non-finite: Optimize returns PHOVO_E_NUMERIC, the batch
    returns the non-finite state, and both agree with the restatement on every iteration's valid count."""
    shape = (135, 241)
    cfg = make_cfg(phovo, "test_3_level_all_active")
    K = intrinsics(phovo, *shape, False)
    g0, d0, g1, d1 = make_pair(phovo, shape, K, 90, "f64", "f64")
    d1 = damaged(d1, how)
    s0 = np.zeros(6)
    sref, ref = br.optimize(br.BiLevels(cfg, K, g0, d0, g1, d1, U16_SCALE), s0)
    finite = how == "holes_and_out_of_range"
    assert np.isfinite(sref).all() == finite
    odo = new_odo(phovo, cfg, K)
    for ex in (0, 1, 2):
        odo.SetExecution(ex)
        s, log = optimize(phovo, odo, g0, d0, g1, d1, s0, expect_numeric=not finite)
        if finite:
            assert_log_matches(log, ref, (how, ex))
            assert np.max(np.abs(s - sref)) < 1e-9
        else:
            assert not np.isfinite(s).all(), ex
            assert [(e["level"], e["iteration"], e["num_valid"]) for e in log] == \
                [(e["level"], e["iteration"], e["num_valid"]) for e in ref], ex
            assert np.array_equal(np.isfinite(s), np.isfinite(sref)), ex
    for flags in (8, 4):
        odo.BatchSetDebugFlags(flags)
        st, it = odo.BatchAlign(np.stack([g0, g0]), np.stack([d0, d0]), np.stack([g1, g1]), depth1=np.stack([d1, d1]))
        for p in range(2):
            assert np.array_equal(it[p], iterations_per_level(ref)), (how, flags, it[p])
            if finite:
                assert np.max(np.abs(st[p] - sref)) < 1e-9, (how, flags)
            else:
                assert np.array_equal(np.isfinite(st[p]), np.isfinite(sref)), (how, flags, st[p])
    odo.BatchSetDebugFlags(0)
    odo.close()


# ---------------------------------------------------------------------------------------------
def test_visual_odometry_chain_with_promoted_target(phovo):
    """Four frames: after each alignment the target becomes the source (PromoteTargetToSource with its depth) and the
    next frame comes with a fresh target depth; every step matches a restatement started from the previous state."""
    rows, cols = 120, 160
    cfg = make_cfg(phovo, "test_3_level_all_active")
    K = phovo.synth.K_VISUAL_ODOMETRY * np.array([[cols / 640.], [rows / 480.], [1.]])
    frames = [phovo.synth.make_sequence_frame(40 * k, rows, cols, K=K, n=1000) for k in range(4)]
    frames = [(g, as_type(d, "u16")) for g, d in frames]
    odo = new_odo(phovo, cfg, K)
    odo.SetSourceFrame(frames[0][0], frames[0][1], depth_scale=U16_SCALE)
    s = np.zeros(6)
    for k in range(1, 4):
        g, d = frames[k]
        odo.SetTargetFrame(g, d, depth_scale=U16_SCALE)
        odo.SetInitialStateVector(s)
        odo.Optimize()
        sref, ref = br.optimize(br.BiLevels(cfg, K, frames[k - 1][0], frames[k - 1][1], g, d, U16_SCALE), s)
        assert_log_matches(odo.IterationStats(), ref, ("step", k))
        s = odo.GetOptimalStateVector()
        assert np.max(np.abs(s - sref)) < 1e-9, k
        odo.PromoteTargetToSource(d, depth_scale=U16_SCALE)
    # a target without its depth is refused by this solver, also after runs with one
    odo.SetTargetFrame(frames[0][0])
    for call in (odo.Optimize, lambda: odo.EvalNormalEquations(0, np.zeros(6))):
        with pytest.raises(phovo.PhovoError) as e:
            call()
        assert e.value.code == phovo.capi.E_INVALID
    odo.close()
