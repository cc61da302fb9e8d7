"""Batched normal equations at given states (phovo_batch_eval_normal_equations / BatchEvalNormalEquations).

For every pair the call must return what the per-pair path (EvalNormalEquations after SetSourceFrame / SetTargetFrame)
returns, to the bars the per-pair path itself meets against the CPU oracle; it must agree with the oracle, the
reference solver and the resident batch kernels that produce the poses, and be bitwise reproducible and independent
of which pairs share a call."""

import numpy as np
import pytest

from helpers import g_rel_err, h_rel_err

pytestmark = pytest.mark.gpu

K640 = np.array([[525., 0., 319.5], [0., 525., 239.5], [0., 0., 1.]])
K241 = np.array([[198., 0., 120.], [0., 198., 67.], [0., 0., 1.]])      # a 135x241 frame
IU = np.triu_indices(6)


def packed(H):
    return np.asarray(H)[..., IU[0], IU[1]]


def assert_close(b, ref, what=""):
    """b: one pair of a batch result (H packed), ref: an IterStats-like dict.  Bars of the per-pair path vs the oracle;
    where the reference sums are zero (nothing valid) they must be exactly zero."""
    assert b["num_valid"] == ref["num_valid"], (what, b["num_valid"], ref["num_valid"])
    Hr, gr = np.asarray(ref["H"], dtype=np.float64), np.asarray(ref["g"], dtype=np.float64)
    if ref["num_valid"] == 0 or not np.all(Hr[[0, 6, 11, 15, 18, 20]] > 0):
        assert np.array_equal(b["H"], Hr) and np.array_equal(b["g"], gr), what
    else:
        assert h_rel_err(b["H"], Hr) < 1e-10, (what, h_rel_err(b["H"], Hr))
        assert g_rel_err(b["g"], gr) < 1e-9, (what, g_rel_err(b["g"], gr))
    if ref["cost"] == 0:
        assert b["cost"] == 0, what
    else:
        assert abs(b["cost"] - ref["cost"]) < 1e-10 * ref["cost"], (what, b["cost"], ref["cost"])


def pair(r, k):
    return dict(H=packed(r["H"][k]), g=r["g"][k], cost=r["cost"][k], num_valid=int(r["num_valid"][k]))


def depth_variants(d32):
    return {"f64": (d32.astype(np.float64), 1.0), "f32": (d32, 1.0),
            "u16": (np.clip(np.rint(d32 * 5000.), 0, 65535).astype(np.uint16), 1. / 5000.)}


def make_ctx(phovo, mode=0, K=K640, cfg_name="config_4_level_optimization_analytic", build_all=False):
    odo = phovo.CPhotoconsistencyOdometryCuda()
    odo.SetConfig(phovo.configs.to_config(cfg_name, phovo.capi, mode=mode))
    odo.SetIntrinsicMatrix(K)
    if build_all:
        odo.SetBuildAllLevels(True)
    return odo


def abi(odo, g0, d0, dtype, scale, g1, states, level, H, g, cost, nv):
    """phovo_batch_eval_normal_equations straight through the C ABI (any mix of host / device buffers)."""
    from importlib import import_module
    capi = import_module("photoconsistency-visual-odometry_b200").capi
    P, R, Cc = g0.shape
    return odo._L.phovo_batch_eval_normal_equations(odo._h, P, R, Cc, capi._ptr(g0), capi._ptr(d0), dtype, float(scale),
                                                    capi._ptr(g1), capi._ptr(states), level, capi._ptr(H), capi._ptr(g),
                                                    capi._ptr(cost), capi._ptr(nv))


@pytest.fixture(scope="module")
def frames(phovo):
    """Four seeded pairs at 640x480 and at 135x241 (host numpy: gray0, depth0 f32, gray1)."""
    import torch
    out = {}
    for (R, C, K) in ((480, 640, K640), (135, 241, K241)):
        g0, d0, g1, _ = phovo.synth.render_batch_torch(4, R, C, K, torch.device("cuda", 0), seed0=31)
        out[(R, C)] = (g0.cpu().numpy(), d0.cpu().numpy(), g1.cpu().numpy(), K)
    return out


@pytest.mark.parametrize("depth", ["f64", "f32", "u16"])
@pytest.mark.parametrize("size", [(480, 640), (135, 241)])
@pytest.mark.parametrize("mode", [0, 1])
def test_matches_per_pair_path(phovo, frames, mode, size, depth):
    import torch
    capi = phovo.capi
    g0, d32, g1, K = frames[size]
    d, scale = depth_variants(d32)[depth]
    P = len(g0)
    # states: two random ones and the one a batch alignment returns, for every pair
    rng = np.random.default_rng(5 + mode)
    rand = [np.concatenate([rng.uniform(-0.05, 0.05, (P, 3)), rng.uniform(-0.03, 0.03, (P, 3))], axis=1) for _ in range(2)]
    aligned, _ = make_ctx(phovo, mode, K).BatchAlign(g0, d, g1, depth_scale=scale)
    sets = rand + [aligned]
    idx = np.repeat(np.arange(P), len(sets))                      # pair p with each state set
    st = np.stack([sets[s][p] for p in range(P) for s in range(len(sets))])
    bg0, bd, bg1 = g0[idx], d[idx], g1[idx]
    # the per-pair path, every level built
    ref = make_ctx(phovo, mode, K, build_all=True)
    expect = {}
    for p in range(P):
        ref.SetSourceFrame(g0[p], d[p], depth_scale=scale)
        ref.SetTargetFrame(g1[p])
        for level in range(4):
            for s in range(len(sets)):
                expect[(level, p * len(sets) + s)] = ref.EvalNormalEquations(level, sets[s][p])
    odo = make_ctx(phovo, mode, K)
    dev = torch.device("cuda", 0)
    tg0, td, tg1 = (torch.from_numpy(a.view(np.int16) if a.dtype == np.uint16 else a) for a in (bg0, bd, bg1))
    inputs = {"numpy": (bg0, bd, bg1), "pinned": tuple(t.pin_memory() for t in (tg0, td, tg1)),
              "cuda": tuple(t.to(dev) for t in (tg0, td, tg1))}
    code = {"f64": capi.DEPTH_F64, "f32": capi.DEPTH_F32, "u16": capi.DEPTH_U16}[depth]
    for level in range(4):
        if size == (135, 241) and level == 1:                     # cells cut by the border: not in the integer records
            H = np.zeros((len(st), 21))
            assert abi(odo, bg0, bd, code, scale, bg1, st, 1, H, None, None, None) == capi.E_UNSUPPORTED
            continue
        first = None
        for kind, (a0, a1, a2) in inputs.items():
            r = odo.BatchEvalNormalEquations(a0, a1, a2, st if kind != "cuda" else torch.from_numpy(st).to(dev),
                                             level=level, depth_scale=scale)
            assert np.array_equal(r["H"], np.swapaxes(r["H"], 1, 2))
            if first is None:
                first = r
                for k in range(len(st)):
                    assert_close(pair(r, k), expect[(level, k)], (mode, size, depth, level, k))
            else:
                for key in ("H", "g", "cost", "num_valid"):
                    assert np.array_equal(r[key], first[key]), (kind, key)
        # outputs on the device and partial output sets through the C ABI
        for out_dev in (False, True):
            mk = (lambda shape, dt: torch.zeros(shape, dtype=dt, device=dev)) if out_dev else \
                 (lambda shape, dt: torch.zeros(shape, dtype=dt))
            H, g, c, n = mk((len(st), 21), torch.float64), mk((len(st), 6), torch.float64), mk((len(st),), torch.float64), \
                mk((len(st),), torch.int32)
            assert abi(odo, *inputs["cuda"][:2], code, scale, inputs["cuda"][2], st, level, H, g, c, n) == 0
            assert np.array_equal(H.cpu().numpy(), packed(first["H"])) and np.array_equal(g.cpu().numpy(), first["g"])
            assert np.array_equal(c.cpu().numpy(), first["cost"]) and np.array_equal(n.cpu().numpy(), first["num_valid"])
            n2 = mk((len(st),), torch.int32)
            assert abi(odo, bg0, bd, code, scale, bg1, st, level, None, None, None, n2) == 0
            assert np.array_equal(n2.cpu().numpy(), first["num_valid"])


@pytest.mark.parametrize("size", [(96, 128), (120, 160)])
def test_matches_oracle_and_reference(phovo, oracle, size):
    from test_gpu_parity import conv_cfg
    R, C = size
    K = phovo.synth.K_FRAME_ALIGNMENT * np.array([[C / 640.], [R / 480.], [1.]])
    g0, d0, g1, _ = phovo.synth.make_pair(R, C, K=K, seed=12)
    rng = np.random.default_rng(13)
    st = np.concatenate([rng.uniform(-0.05, 0.05, (3, 3)), rng.uniform(-0.03, 0.03, (3, 3))], axis=1)
    st = np.vstack([np.zeros(6), st])
    P = len(st)
    for mode in (0, 1):
        cfg = phovo.configs.to_config("config_4_level_optimization_analytic", phovo.capi, mode=mode)
        for l in range(cfg.num_levels):
            cfg.max_num_iterations[l] = 1
        o = oracle.Oracle(conv_cfg(oracle, cfg), K)
        o.set_source(g0, d0)
        o.set_target(g1)
        odo = make_ctx(phovo, mode, K)                       # iterations [0, 0, 20, 50]: levels 0 and 1 are not configured
        for level in range(4):
            r = odo.BatchEvalNormalEquations(np.stack([g0] * P), np.stack([d0] * P), np.stack([g1] * P), st, level=level)
            for k in range(P):
                assert_close(pair(r, k), o.eval(level, st[k]), (size, mode, level, k))
    import ref_py
    if not ref_py.available():
        pytest.skip("oracle/_ref (the reference solver built from the original project) is not present")
    import tempfile
    c = phovo.configs
    odo = make_ctx(phovo, 0, K)
    for level in range(4):
        n = level + 1
        yml = c.to_yaml({c.K_LEVELS: n, c.K_BLUR: [0] * n, c.K_GRAD: [0.0625] * n, c.K_LAMBDA: [1] * n,
                         c.K_ITERS: [0] * level + [1], c.K_MINGRAD: [0.] * n, "visualizeIterations": 0})
        path = tempfile.mktemp(suffix=".yml")
        with open(path, "w") as f:
            f.write(yml)
        for k in range(P):
            _, _, iters = ref_py.Reference(path, K).align(g0, d0, g1, state0=st[k])
            r = odo.BatchEvalNormalEquations(g0[None], d0[None], g1[None], st[k][None], level=level)
            Hr, gr = packed(iters[0]["H"]), iters[0]["g"]
            assert int(r["num_valid"][0]) == iters[0]["n"], (level, k)
            assert h_rel_err(packed(r["H"][0]), Hr) < 1e-10 and g_rel_err(r["g"][0], gr) < 1e-9, (level, k)


def test_matches_resident_batch_kernels(phovo):
    """At every state the resident batch kernels logged, the batch evaluation gives their num_valid, H and g."""
    import torch
    dev = torch.device("cuda", 0)
    g0, d0, g1, _ = phovo.synth.render_batch_torch(4, 480, 640, K640, dev, seed0=55)
    for mode in (0, 1):
        odo = make_ctx(phovo, mode)
        odo.BatchSetRecordStats(True)
        odo.BatchAlign(g0, d0, g1)
        assert odo.BatchLastPath() == 1
        for p in range(4):
            log = odo.BatchIterationStats(p)
            assert len(log) > 0
            for level in sorted({e["level"] for e in log}):
                ent = [e for e in log if e["level"] == level]
                E = len(ent)
                st = np.stack([e["state_in"] for e in ent])
                r = odo.BatchEvalNormalEquations(g0[p].expand(E, -1, -1).contiguous(), d0[p].expand(E, -1, -1).contiguous(),
                                                 g1[p].expand(E, -1, -1).contiguous(), st, level=level)
                for k, e in enumerate(ent):
                    assert int(r["num_valid"][k]) == e["num_valid"], (mode, p, level, k)
                    assert h_rel_err(packed(r["H"][k]), e["H"]) < 1e-10, (mode, p, level, k)
                    assert g_rel_err(r["g"][k], e["g"]) < 1e-9, (mode, p, level, k)


def test_deterministic_and_independent_of_batch_composition(phovo):
    import torch
    dev = torch.device("cuda", 0)
    g0, d0, g1, _ = phovo.synth.render_batch_torch(160, 480, 640, K640, dev, seed0=91)
    rng = np.random.default_rng(17)
    st = np.concatenate([rng.uniform(-0.05, 0.05, (160, 3)), rng.uniform(-0.03, 0.03, (160, 3))], axis=1)
    odo = make_ctx(phovo, 0)
    keys = ("H", "g", "cost", "num_valid")
    a = odo.BatchEvalNormalEquations(g0, d0, g1, st, level=0)          # several L2-sized chunks
    b = odo.BatchEvalNormalEquations(g0, d0, g1, st, level=0)
    for k in keys:
        assert np.array_equal(a[k], b[k]), k
    perm = np.random.default_rng(4).permutation(160)
    pt = torch.from_numpy(perm).to(dev)
    c = odo.BatchEvalNormalEquations(g0[pt].contiguous(), d0[pt].contiguous(), g1[pt].contiguous(), st[perm], level=0)
    for k in keys:
        assert np.array_equal(c[k], a[k][perm]), k
    for p in (0, 77, 159):
        one = odo.BatchEvalNormalEquations(g0[p:p + 1], d0[p:p + 1], g1[p:p + 1], st[p:p + 1], level=0)
        for k in keys:
            assert np.array_equal(one[k][0], a[k][p]), (p, k)
    # level 2 (records of the pyramid kernel): permutation and single pairs too
    a2 = odo.BatchEvalNormalEquations(g0, d0, g1, st, level=2)
    c2 = odo.BatchEvalNormalEquations(g0[pt].contiguous(), d0[pt].contiguous(), g1[pt].contiguous(), st[perm], level=2)
    one = odo.BatchEvalNormalEquations(g0[5:6], d0[5:6], g1[5:6], st[5:6], level=2)
    for k in keys:
        assert np.array_equal(c2[k], a2[k][perm]) and np.array_equal(one[k][0], a2[k][5]), k


def test_degenerate_inputs_equal_per_pair_path(phovo, frames):
    g0, d32, g1, K = frames[(480, 640)]
    g0, d32, g1 = g0[:1], d32[:1], g1[:1]
    st0 = np.array([0.01, -0.02, 0.03, 0.01, 0.005, -0.01])
    cases = {"zero depth": (np.zeros_like(d32), st0), "nan depth": (np.full_like(d32, np.nan), st0),
             "nan state": (d32, np.array([np.nan, 0., 0., 0., 0., 0.])),
             "behind the camera": (d32, np.array([0., 0., -20., 0., 0., 0.]))}
    odo = make_ctx(phovo, 0)
    ref = make_ctx(phovo, 0, build_all=True)
    for name, (d, st) in cases.items():
        ref.SetSourceFrame(g0[0], d[0])
        ref.SetTargetFrame(g1[0])
        for level in (0, 2):
            r = odo.BatchEvalNormalEquations(g0, d, g1, st[None], level=level)
            e = ref.EvalNormalEquations(level, st)
            assert_close(pair(r, 0), e, (name, level))
            if name != "behind the camera":
                assert r["num_valid"][0] == 0 and not r["H"].any() and not r["g"].any(), name


def test_errors_and_release(phovo, frames):
    capi = phovo.capi
    g0, d32, g1, K = frames[(480, 640)]
    g0, d32, g1 = g0[:2], d32[:2], g1[:2]
    st = np.zeros((2, 6)); st[:, 0] = 0.01
    F32, EI, EU = capi.DEPTH_F32, capi.E_INVALID, capi.E_UNSUPPORTED
    odo = make_ctx(phovo, 0)
    ref = odo.BatchEvalNormalEquations(g0, d32, g1, st, level=2)
    H = np.zeros((2, 21))
    assert abi(odo, g0, d32, F32, 1., g1, st, 2, H, None, None, None) == 0
    assert np.array_equal(H, packed(ref["H"]))
    # PHOVO_E_INVALID
    fresh = phovo.CPhotoconsistencyOdometryCuda()                            # no intrinsics
    assert abi(fresh, g0, d32, F32, 1., g1, st, 0, H, None, None, None) == EI
    assert abi(odo, g0, d32, F32, 1., g1, st, -1, H, None, None, None) == EI
    assert abi(odo, g0, d32, F32, 1., g1, st, 4, H, None, None, None) == EI          # config 4 has 4 levels
    assert abi(odo, g0, d32, 7, 1., g1, st, 0, H, None, None, None) == EI
    assert abi(odo, g0, d32, F32, 1., g1, st, 0, None, None, None, None) == EI
    Pfn = odo._L.phovo_batch_eval_normal_equations
    for P, R, C in ((0, 480, 640), (2, 0, 640), (2, 480, 0)):
        assert Pfn(odo._h, P, R, C, capi._ptr(g0), capi._ptr(d32), F32, 1., capi._ptr(g1), capi._ptr(st), 0,
                   capi._ptr(H), None, None, None) == EI
    # PHOVO_E_UNSUPPORTED: frames of 2^31 px (rejected before any input is read), level 1 of a 3 mod 4 size,
    # a blurred level, the Ceres-mode and photometric + depth solvers
    assert Pfn(odo._h, 1, 1 << 16, 1 << 15, capi._ptr(g0), capi._ptr(d32), F32, 1., capi._ptr(g1), capi._ptr(st), 0,
               capi._ptr(H), None, None, None) == EU
    assert Pfn(odo._h, 1, 479, 640, capi._ptr(g0), capi._ptr(d32), F32, 1., capi._ptr(g1), capi._ptr(st), 1,
               capi._ptr(H), None, None, None) == EU
    cfg = odo.GetConfig()
    cfg.blur_filter_size[2] = 3
    blurred = phovo.CPhotoconsistencyOdometryCuda()
    blurred.SetConfig(cfg); blurred.SetIntrinsicMatrix(K)
    assert abi(blurred, g0, d32, F32, 1., g1, st, 2, H, None, None, None) == EU
    assert abi(blurred, g0, d32, F32, 1., g1, st, 3, H, None, None, None) == 0
    for mode in (capi.MODE_CERES, capi.MODE_BIOBJECTIVE):
        other = make_ctx(phovo, mode)
        assert abi(other, g0, d32, F32, 1., g1, st, 2, H, None, None, None) == EU
    # the next valid call after a failure, and after a release, gives the same results
    again = odo.BatchEvalNormalEquations(g0, d32, g1, st, level=2)
    odo.BatchReleaseMemory()
    released = odo.BatchEvalNormalEquations(g0, d32, g1, st, level=2)
    for k in ("H", "g", "cost", "num_valid"):
        assert np.array_equal(ref[k], again[k]) and np.array_equal(ref[k], released[k]), k


def test_align_sequence_information(phovo):
    import torch
    Kv = phovo.synth.K_VISUAL_ODOMETRY
    g, d = phovo.synth.render_sequence_torch(10, 480, 640, Kv, torch.device("cuda", 0))
    seq = make_ctx(phovo, 0, Kv, cfg_name="config_5_level_optimization_analytic")
    st, it, poses = seq.AlignSequence(g, d)
    st2, it2, poses2, info = seq.AlignSequence(g, d, information_level=0)
    assert np.array_equal(st, st2) and np.array_equal(it, it2) and np.array_equal(poses, poses2)
    assert set(info) == {"H", "g", "cost", "num_valid"}
    r = seq.BatchEvalNormalEquations(g[:-1].contiguous(), d[:-1].contiguous(), g[1:].contiguous(), st, level=0)
    for k in ("H", "g", "cost", "num_valid"):
        assert np.array_equal(info[k], r[k]), k
    assert (info["num_valid"] > 0).all()
    _, _, _, both = seq.AlignSequence(g, d, diagnostics=True, information_level=0)
    assert set(both) == {"num_landed", "sum_abs_diff", "mean_abs_diff", "H", "g", "cost", "num_valid"}
    assert np.array_equal(both["H"], info["H"])
