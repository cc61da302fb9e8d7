"""The photometric + depth solver (MODE_BIOBJECTIVE) on device batches and recorded sequences.

phovo_batch_eval_normal_equations_with_target_depth must return, pair by pair, what EvalNormalEquations returns on a
context that built every level after SetSourceFrame / SetTargetFrame(gray1, depth1), to the bars of the analytic batch
evaluation, be bitwise reproducible and independent of which pairs share a call; BatchAlignDevice(depth1=),
AlignSequence and run_visual_odometry must run this solver as the per-pair API does."""

import importlib

import numpy as np
import pytest

import bi_restatement as br
from helpers import g_rel_err, h_rel_err
from test_gpu_batch_eval import assert_close, packed, pair
from test_gpu_biobjective_restatement import EVAL_STATES, U16_SCALE, as_type, damaged, intrinsics, make_cfg, make_pair

pytestmark = pytest.mark.gpu

CFG4 = "config_4_level_optimization_analytic"


def new_ctx(phovo, cfg, K, build_all=False):
    odo = phovo.CPhotoconsistencyOdometryCuda()
    odo.SetConfig(cfg)
    odo.SetIntrinsicMatrix(K)
    if build_all:
        odo.SetBuildAllLevels(True)
    return odo


def frames_of(phovo, shape, kind, K, seed0, P):
    pairs = [make_pair(phovo, shape, K, seed0 + p, kind, kind) for p in range(P)]
    return tuple(np.stack([q[k] for q in pairs]) for k in range(4))


def per_pair(ref, g0, d0, g1, d1, level, state):
    ref.SetSourceFrame(g0, d0, depth_scale=U16_SCALE)
    ref.SetTargetFrame(g1, d1, depth_scale=U16_SCALE)
    return ref.EvalNormalEquations(level, state)


def abi(odo, g0, d0, dtype, g1, d1, states, level, H, g, cost, nv, P=None, R=None, Cc=None):
    """phovo_batch_eval_normal_equations_with_target_depth straight through the C ABI (any mix of host / device buffers)."""
    capi = importlib.import_module("photoconsistency-visual-odometry_b200").capi
    if P is None:
        P, R, Cc = g0.shape
    return odo._L.phovo_batch_eval_normal_equations_with_target_depth(
        odo._h, P, R, Cc, capi._ptr(g0), capi._ptr(d0), dtype, float(U16_SCALE), capi._ptr(g1), capi._ptr(d1),
        capi._ptr(states), level, capi._ptr(H), capi._ptr(g), capi._ptr(cost), capi._ptr(nv))


def level1_unsupported(shape):
    return shape[0] % 4 == 3 or shape[1] % 4 == 3


# ---------------------------------------------------------------------------------------------
# 1. the per-pair path, at every level
@pytest.mark.parametrize("kind", ["f64", "f32", "u16"])
@pytest.mark.parametrize("shape", [(480, 640), (135, 241), (107, 203)])
def test_matches_per_pair_path_at_every_level(phovo, shape, kind):
    cfg = make_cfg(phovo, CFG4)
    K = intrinsics(phovo, *shape, shape != (480, 640))
    P = 2
    g0, d0, g1, d1 = frames_of(phovo, shape, kind, K, 100, P)
    odo = new_ctx(phovo, cfg, K)
    aligned, _ = odo.BatchAlign(g0, d0, g1, depth_scale=U16_SCALE, depth1=d1)
    rng = np.random.default_rng(7)
    states = [rng.uniform(-0.04, 0.04, 6), aligned] + list(EVAL_STATES.values())
    # every state for every pair: one batch of P * len(states) pairs
    idx = [p for _ in states for p in range(P)]
    S = np.concatenate([np.broadcast_to(s, (P, 6)) for s in states])
    ref = new_ctx(phovo, cfg, K, build_all=True)
    for level in range(4):
        if level == 1 and level1_unsupported(shape):
            with pytest.raises(phovo.PhovoError) as e:
                odo.BatchEvalNormalEquations(g0[idx], d0[idx], g1[idx], S, level=level, depth_scale=U16_SCALE, depth1=d1[idx])
            assert e.value.code == phovo.capi.E_UNSUPPORTED
            continue
        r = odo.BatchEvalNormalEquations(g0[idx], d0[idx], g1[idx], S, level=level, depth_scale=U16_SCALE, depth1=d1[idx])
        for k, p in enumerate(idx):
            st = per_pair(ref, g0[p], d0[p], g1[p], d1[p], level, S[k])
            assert_close(pair(r, k), st, (shape, kind, level, k))
    odo.close()
    ref.close()


def test_input_and_output_placements_are_bitwise_equal(phovo):
    import torch
    capi = phovo.capi
    shape = (120, 160)
    cfg = make_cfg(phovo, CFG4)
    K = intrinsics(phovo, *shape, True)
    g0, d0, g1, d1 = frames_of(phovo, shape, "u16", K, 130, 3)
    S = np.stack([EVAL_STATES["motion"], EVAL_STATES["identity"], EVAL_STATES["rotated"]])
    odo = new_ctx(phovo, cfg, K)

    def tensor(a):
        return torch.from_numpy(a.view(np.int16) if a.dtype == np.uint16 else a)
    for level in (0, 1, 2):
        r = odo.BatchEvalNormalEquations(g0, d0, g1, S, level=level, depth_scale=U16_SCALE, depth1=d1)
        for what, conv in (("pinned", lambda a: tensor(a).pin_memory()), ("device", lambda a: tensor(a).cuda())):
            r2 = odo.BatchEvalNormalEquations(*(conv(a) for a in (g0, d0, g1)), conv(S), level=level, depth_scale=U16_SCALE,
                                              depth1=conv(d1))
            for key in r:
                assert np.array_equal(r[key], r2[key]), (level, what, key)
        # device outputs and partial output sets through the C ABI
        gd0, dd0, gd1, dd1, sd = (tensor(a).cuda() for a in (g0, d0, g1, d1, S))
        H = torch.zeros((3, 21), dtype=torch.float64, device="cuda")
        g = torch.zeros((3, 6), dtype=torch.float64, device="cuda")
        cost = torch.zeros(3, dtype=torch.float64, device="cuda")
        nv = torch.zeros(3, dtype=torch.int32, device="cuda")
        assert abi(odo, gd0, dd0, capi.DEPTH_U16, gd1, dd1, sd, level, H, g, cost, nv) == capi.OK
        torch.cuda.synchronize()
        assert np.array_equal(H.cpu().numpy(), packed(r["H"])) and np.array_equal(g.cpu().numpy(), r["g"])
        assert np.array_equal(cost.cpu().numpy(), r["cost"]) and np.array_equal(nv.cpu().numpy(), r["num_valid"])
        Hh, ch = np.zeros((3, 21)), np.zeros(3)
        assert abi(odo, g0, d0, capi.DEPTH_U16, g1, d1, S, level, Hh, None, ch, None) == capi.OK
        assert np.array_equal(Hh, packed(r["H"])) and np.array_equal(ch, r["cost"])
    odo.close()


# ---------------------------------------------------------------------------------------------
# 2. the float64 restatement
def test_matches_restatement_at_eval_states(phovo):
    shape = (106, 150)
    cfg = make_cfg(phovo, "test_3_level_all_active")
    K = intrinsics(phovo, *shape, True)
    g0, d0, g1, d1 = make_pair(phovo, shape, K, 140, "f32", "f32")
    lv = br.BiLevels(cfg, K, g0, d0, g1, d1, U16_SCALE)
    odo = new_ctx(phovo, cfg, K)
    names = list(EVAL_STATES)
    S = np.stack([EVAL_STATES[n] for n in names])
    P = len(names)
    for level in range(3):
        r = odo.BatchEvalNormalEquations(np.stack([g0] * P), np.stack([d0] * P), np.stack([g1] * P), S, level=level,
                                         depth1=np.stack([d1] * P))
        for k, name in enumerate(names):
            e = br.evaluate(lv.levels[level], lv.K, level, S[k])
            w = (level, name)
            assert r["num_valid"][k] == e["num_valid"], w
            assert h_rel_err(packed(r["H"][k]), br.pack_upper(e["H"])) < 1e-9, (w, h_rel_err(packed(r["H"][k]), br.pack_upper(e["H"])))
            assert g_rel_err(r["g"][k], e["g"]) < 1e-8, w
            assert abs(r["cost"][k] - e["cost"]) <= 1e-10 * e["cost"], w
    odo.close()


# ---------------------------------------------------------------------------------------------
# 3. the iterations a batch alignment logs
def test_reproduces_the_alignment_log(phovo):
    shape = (120, 160)
    cfg = make_cfg(phovo, CFG4)
    K = intrinsics(phovo, *shape, False)
    P = 3
    g0, d0, g1, d1 = frames_of(phovo, shape, "u16", K, 150, P)
    odo = new_ctx(phovo, cfg, K)
    odo.BatchSetRecordStats(True)
    odo.BatchAlign(g0, d0, g1, depth_scale=U16_SCALE, depth1=d1)
    assert odo.BatchLastPath() == 2
    logs = [odo.BatchIterationStats(p) for p in range(P)]
    odo.BatchSetRecordStats(False)
    checked = 0
    for level in range(4):
        entries = [(p, e) for p in range(P) for e in logs[p] if e["level"] == level]
        if not entries:
            continue
        idx = [p for p, _ in entries]
        S = np.stack([e["state_in"] for _, e in entries])
        r = odo.BatchEvalNormalEquations(g0[idx], d0[idx], g1[idx], S, level=level, depth_scale=U16_SCALE, depth1=d1[idx])
        for k, (p, e) in enumerate(entries):
            w = (level, p, e["iteration"])
            assert r["num_valid"][k] == e["num_valid"], w
            assert h_rel_err(packed(r["H"][k]), e["H"]) < 1e-10, w
            assert g_rel_err(r["g"][k], e["g"]) < 1e-9, w
            checked += 1
    assert checked == sum(len(l) for l in logs) and checked > P
    odo.close()


# ---------------------------------------------------------------------------------------------
# 4. determinism and composition over several chunks
@pytest.fixture(scope="module")
def many(phovo):
    import torch
    P = 160
    K = phovo.synth.K_FRAME_ALIGNMENT
    g0, d0, g1, _ = phovo.synth.render_batch_torch(P, 480, 640, K, torch.device("cuda", 0), seed0=170)
    d1 = torch.roll(d0, 1, dims=0).flip(2).contiguous()        # another pair's depth, mirrored: a different target depth
    rng = np.random.default_rng(171)
    S = torch.from_numpy(rng.uniform(-0.03, 0.03, (P, 6))).cuda()
    return K, g0, d0, g1, d1, S


@pytest.mark.parametrize("level", [0, 2])
def test_bitwise_reproducible_and_independent_of_the_batch(phovo, many, level):
    import torch
    K, g0, d0, g1, d1, S = many
    odo = new_ctx(phovo, make_cfg(phovo, CFG4), K)
    r = odo.BatchEvalNormalEquations(g0, d0, g1, S, level=level, depth1=d1)
    assert np.all(r["num_valid"] > 0)
    r2 = odo.BatchEvalNormalEquations(g0, d0, g1, S, level=level, depth1=d1)
    for key in r:
        assert np.array_equal(r[key], r2[key]), key
    perm = torch.from_numpy(np.random.default_rng(level).permutation(g0.shape[0])).cuda()
    rp = odo.BatchEvalNormalEquations(g0[perm], d0[perm], g1[perm], S[perm], level=level, depth1=d1[perm])
    pc = perm.cpu().numpy()
    for key in r:
        assert np.array_equal(rp[key], r[key][pc]), key
    for k in (0, 77, 159):
        r1 = odo.BatchEvalNormalEquations(g0[k:k + 1], d0[k:k + 1], g1[k:k + 1], S[k:k + 1], level=level, depth1=d1[k:k + 1])
        for key in r:
            assert np.array_equal(r1[key][0], r[key][k]), (k, key)
    odo.close()


# ---------------------------------------------------------------------------------------------
# 5. target depths that are not a clean depth map
@pytest.mark.parametrize("how", ["holes_and_out_of_range", "all_zero", "nan"])
def test_damaged_target_depth(phovo, how):
    shape = (135, 241)
    cfg = make_cfg(phovo, CFG4)
    K = intrinsics(phovo, *shape, False)
    g0, d0, g1, d1 = make_pair(phovo, shape, K, 190, "f64", "f64")
    d1 = damaged(d1, how)
    S = np.stack([np.zeros(6), EVAL_STATES["motion"]])
    odo = new_ctx(phovo, cfg, K)
    ref = new_ctx(phovo, cfg, K, build_all=True)
    for level in (0, 2):
        r = odo.BatchEvalNormalEquations(np.stack([g0] * 2), np.stack([d0] * 2), np.stack([g1] * 2), S, level=level,
                                         depth1=np.stack([d1] * 2))
        for k in range(2):
            st = per_pair(ref, g0, d0, g1, d1, level, S[k])
            w = (how, level, k)
            assert r["num_valid"][k] == st["num_valid"], w
            Hb, Hr = packed(r["H"][k]), np.asarray(st["H"])
            assert np.array_equal(np.isfinite(Hb), np.isfinite(Hr)), w
            assert np.array_equal(np.isfinite(r["g"][k]), np.isfinite(np.asarray(st["g"]))), w
            assert np.isfinite(r["cost"][k]) == np.isfinite(st["cost"]), w
            if how == "holes_and_out_of_range":
                assert_close(pair(r, k), st, w)
    odo.close()
    ref.close()


# ---------------------------------------------------------------------------------------------
# 6. errors and recovery
def test_errors_and_recovery(phovo):
    capi = phovo.capi
    shape = (120, 160)
    K = intrinsics(phovo, *shape, False)
    g0, d0, g1, d1 = frames_of(phovo, shape, "f32", K, 200, 2)
    S = np.stack([EVAL_STATES["motion"], EVAL_STATES["rotated"]])
    odo = new_ctx(phovo, make_cfg(phovo, CFG4), K)
    H = np.zeros((2, 21))
    good = odo.BatchEvalNormalEquations(g0, d0, g1, S, level=1, depth1=d1)
    assert abi(odo, g0, d0, capi.DEPTH_F32, g1, None, S, 1, H, None, None, None) == capi.E_INVALID
    # the entry without a target depth keeps refusing this solver
    assert odo._L.phovo_batch_eval_normal_equations(odo._h, 2, 120, 160, capi._ptr(g0), capi._ptr(d0), capi.DEPTH_F32, 1.0,
                                                    capi._ptr(g1), capi._ptr(S), 1, capi._ptr(H), None, None, None) == capi.E_UNSUPPORTED
    # frames of 2^31 pixels are refused before any input is read
    assert abi(odo, g0, d0, capi.DEPTH_F32, g1, d1, S, 0, H, None, None, None, P=2, R=1 << 16, Cc=1 << 15) == capi.E_UNSUPPORTED
    blur = make_cfg(phovo, CFG4)
    blur.blur_filter_size[1] = 3
    ob = new_ctx(phovo, blur, K)
    assert abi(ob, g0, d0, capi.DEPTH_F32, g1, d1, S, 1, H, None, None, None) == capi.E_UNSUPPORTED
    assert abi(ob, g0, d0, capi.DEPTH_F32, g1, d1, S, 2, H, None, None, None) == capi.OK
    ob.close()
    after_fail = odo.BatchEvalNormalEquations(g0, d0, g1, S, level=1, depth1=d1)
    odo.BatchReleaseMemory()
    after_release = odo.BatchEvalNormalEquations(g0, d0, g1, S, level=1, depth1=d1)
    for key in good:
        assert np.array_equal(after_fail[key], good[key]) and np.array_equal(after_release[key], good[key]), key
    odo.close()
    # Ceres mode: the new entry forwards to the old one, which refuses it
    oc = new_ctx(phovo, phovo.configs.to_config(CFG4, capi, mode=capi.MODE_CERES), K)
    assert abi(oc, g0, d0, capi.DEPTH_F32, g1, d1, S, 0, H, None, None, None) == capi.E_UNSUPPORTED
    oc.close()
    # analytic modes: the new entry is the old one, bit for bit (the target depth is ignored)
    for mode in (capi.MODE_ANALYTIC_REF, capi.MODE_ANALYTIC_FIXED):
        oa = new_ctx(phovo, phovo.configs.to_config(CFG4, capi, mode=mode), K)
        for level in (0, 2):
            a = oa.BatchEvalNormalEquations(g0, d0, g1, S, level=level)
            b = oa.BatchEvalNormalEquations(g0, d0, g1, S, level=level, depth1=d1)
            for key in a:
                assert np.array_equal(a[key], b[key]), (mode, level, key)
        oa.close()


# ---------------------------------------------------------------------------------------------
# 7. device-resident batch alignment
@pytest.mark.parametrize("P", [5, 30])
def test_batch_align_device_with_target_depth(phovo, P):
    import torch
    shape = (120, 160)
    cfg = make_cfg(phovo, CFG4)
    K = intrinsics(phovo, *shape, True)
    g0, d0, g1, d1 = frames_of(phovo, shape, "u16", K, 210, P)
    init = np.stack([0.3 * phovo.synth.random_motion(210 + p) for p in range(P)])
    odo = new_ctx(phovo, cfg, K)
    st, it = odo.BatchAlign(g0, d0, g1, init, depth_scale=U16_SCALE, depth1=d1)
    path = odo.BatchLastPath()
    assert path == (2 if P < 24 else 3)

    def dev(a):
        return torch.from_numpy(a.view(np.int16) if a.dtype == np.uint16 else a).cuda()
    states = torch.zeros((P, 6), dtype=torch.float64, device="cuda")
    iters = torch.zeros((P, phovo.capi.MAXL), dtype=torch.int32, device="cuda")
    odo.BatchAlignDevice(dev(g0), dev(d0), dev(g1), states, iters, initial_states=dev(init), depth_scale=U16_SCALE,
                         depth1=dev(d1))
    torch.cuda.synchronize()
    assert odo.BatchLastPath() == path
    assert np.array_equal(iters.cpu().numpy(), it)
    assert np.array_equal(states.cpu().numpy(), st)
    odo.close()


# ---------------------------------------------------------------------------------------------
# 8. AlignSequence and 9. run_visual_odometry in mode 3
def sequence(phovo, n, rows=120, cols=160):
    K = phovo.synth.K_VISUAL_ODOMETRY * np.array([[cols / 640.], [rows / 480.], [1.]])
    fr = [phovo.synth.make_sequence_frame(3 * k, rows, cols, K=K, n=300) for k in range(n)]
    return K, np.stack([g for g, _ in fr]), np.stack([as_type(d, "u16") for _, d in fr])


def per_frame_loop(phovo, cfg, K, gray, depth):
    odo = new_ctx(phovo, cfg, K)
    odo.SetSourceFrame(gray[0], depth[0], depth_scale=U16_SCALE)
    states, iters, poses = [], [], [np.eye(4)]
    for k in range(1, len(gray)):
        if k > 1:
            odo.PromoteTargetToSource(depth[k - 1], depth_scale=U16_SCALE)
        odo.SetTargetFrame(gray[k], depth[k], depth_scale=U16_SCALE)
        odo.SetInitialStateVector(np.zeros(6))
        odo.Optimize()
        states.append(odo.GetOptimalStateVector())
        it = np.zeros(phovo.capi.MAXL, np.int32)
        for e in odo.IterationStats():
            it[e["level"]] += 1
        iters.append(it)
        poses.append(poses[-1] @ np.linalg.inv(odo.GetOptimalRigidTransformationMatrix()))
    odo.close()
    return np.array(states), np.array(iters), np.array(poses)


@pytest.mark.parametrize("n", [12, 30])
def test_align_sequence(phovo, n):
    cfg = make_cfg(phovo, CFG4)
    K, gray, depth = sequence(phovo, n)
    odo = new_ctx(phovo, cfg, K)
    st, it, poses = odo.AlignSequence(gray, depth, depth_scale=U16_SCALE)
    assert odo.BatchLastPath() == (2 if n - 1 < 24 else 3)
    rs, ri, rp = per_frame_loop(phovo, cfg, K, gray, depth)
    assert np.array_equal(it, ri)
    assert np.max(np.abs(st - rs)) < 1e-9
    assert np.max(np.abs(poses - rp)) < 1e-8
    level = 2
    st2, it2, poses2, diag = odo.AlignSequence(gray, depth, depth_scale=U16_SCALE, diagnostics=True, information_level=level)
    assert np.array_equal(st2, st) and np.array_equal(it2, it)
    for key in ("num_landed", "sum_abs_diff", "mean_abs_diff"):
        assert diag[key].shape == (n - 1,), key
    direct = odo.BatchEvalNormalEquations(gray[:-1], depth[:-1], gray[1:], st, level=level, depth_scale=U16_SCALE,
                                          depth1=depth[1:])
    for key in direct:
        assert np.array_equal(diag[key], direct[key]), key
    odo.close()


@pytest.mark.parametrize("promote", [True, False])
def test_run_visual_odometry(phovo, tmp_path, promote):
    pytest.importorskip("cv2")
    from test_dataset_reader import write_sequence
    ds = phovo.dataset
    n = 6
    K, frames = write_sequence(phovo, str(tmp_path), n=n, rows=120, cols=160)
    cfg = make_cfg(phovo, "test_3_level_all_active")
    odo = new_ctx(phovo, cfg, K)
    got = ds.run_visual_odometry(odo, ds.open_rgbd_dataset(str(tmp_path)), promote=promote)
    assert len(got) == n - 1
    gray = np.stack([g for _, g, _ in frames])
    depth = np.stack([d for _, _, d in frames])
    _, _, poses = odo.AlignSequence(gray, depth, depth_scale=1. / 5000.)
    for k in range(1, n):
        assert np.max(np.abs(got[k - 1][1] - poses[k])) < 1e-8, k
    odo.close()
