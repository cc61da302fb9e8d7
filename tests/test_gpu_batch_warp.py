"""Batched phovo::warpImage + absdiff (phovo_batch_warp_image / BatchWarpImage) and its per-pair summary.

Every image must equal, bit for bit, the reference's own function (golden file, live oracle when present) and the
per-pair path (WarpImage); the summary (landed pixels, summed |target - warped| over them) is an integer sum and
must not depend on chunking or order."""

import numpy as np
import pytest

from helpers import load_golden

pytestmark = pytest.mark.gpu

K = np.array([[525., 0., 319.5], [0., 525., 239.5], [0., 0., 1.]])


@pytest.fixture(scope="module")
def odo(phovo):
    return phovo.CPhotoconsistencyOdometryCuda()


@pytest.fixture(scope="module")
def pairs(phovo):
    """160 seeded 640x480 pairs (several chunks of the L2-sized key buffer), gray0 >= 1, and one pose per pair."""
    import torch
    g0, d0, g1, _ = phovo.synth.render_batch_torch(160, 480, 640, K, torch.device("cuda", 0), seed0=77)
    rng = np.random.default_rng(3)
    states = np.concatenate([rng.uniform(-0.05, 0.05, (160, 3)), rng.uniform(-0.03, 0.03, (160, 3))], axis=1)
    rts = np.stack([phovo.state_to_rt(s) for s in states])
    g0 = np.maximum(g0.cpu().numpy(), 1)
    return g0, d0.cpu().numpy(), g1.cpu().numpy(), rts


def depth_variants(d32):
    return {"f64": (d32.astype(np.float64), 1.0), "f32": (d32, 1.0),
            "u16": (np.clip(np.rint(d32 * 5000.), 0, 65535).astype(np.uint16), 1. / 5000.)}


def loop(odo, g0, d0, rts, K, level, g1, depth_scale):
    out = [odo.WarpImage(g0[p], d0[p], rts[p], K, level=level, targetImage=g1[p], depth_scale=depth_scale) for p in range(len(g0))]
    return np.stack([w for w, _ in out]), np.stack([d for _, d in out])


def summary_of(warped, diff):
    """With gray0 >= 1 a pixel landed iff warped > 0."""
    m = warped > 0
    return m.reshape(len(m), -1).sum(1), np.where(m, diff, 0).reshape(len(m), -1).sum(1, dtype=np.int64)


def abi(odo, g0, d0, dtype, scale, rts, K, level, g1, warped, diff, landed, sums):
    """phovo_batch_warp_image straight through the C ABI (any mix of host / device outputs); returns the code."""
    from importlib import import_module
    capi = import_module("photoconsistency-visual-odometry_b200").capi
    P, R, Cc = g0.shape
    Kc = np.ascontiguousarray(K, dtype=np.float64).reshape(9)
    return odo._L.phovo_batch_warp_image(odo._h, P, R, Cc, capi._ptr(g0), capi._ptr(d0), dtype, float(scale), capi._ptr(rts),
                                         Kc.ctypes.data_as(capi._dp), level, capi._ptr(g1), capi._ptr(warped), capi._ptr(diff),
                                         capi._ptr(landed), capi._ptr(sums))


def test_batch_matches_reference_golden(odo):
    gd = load_golden("ref_warp_image_120x160")
    P = 3
    g0, d0 = np.stack([gd["gray0"]] * P), np.stack([gd["depth0"].astype(np.float64)] * P)
    rts = np.stack([gd["rt"]] * P)
    for level in (0, 1):
        r = odo.BatchWarpImage(g0, d0, rts, gd["K"], level=level, gray1=np.stack([gd["gray1"]] * P))
        for p in range(P):
            assert np.array_equal(r["warped"][p], gd["warped_l%d" % level]), level
            ref_diff = np.abs(gd["gray1"].astype(np.int16) - gd["warped_l%d" % level].astype(np.int16)).astype(np.uint8)
            assert np.array_equal(r["diff"][p], ref_diff), level


def test_batch_matches_reference_source_live(phovo, odo, pairs):
    import ref_py
    if not ref_py.available():
        pytest.skip("oracle/_ref library not present")
    g0, d32, g1, _ = pairs
    rng = np.random.default_rng(11)
    st = np.concatenate([rng.uniform(-0.2, 0.2, (4, 3)), rng.uniform(-0.1, 0.1, (4, 3))], axis=1)
    rts = np.stack([phovo.state_to_rt(s) for s in st])
    for name, (d, scale) in depth_variants(d32[:4]).items():
        w = odo.BatchWarpImage(g0[:4], d, rts, K, depth_scale=scale)["warped"]
        for p in range(4):
            dm = d[p].astype(np.float64) * scale if name == "u16" else d[p].astype(np.float64)
            assert np.array_equal(w[p], ref_py.warp_image(g0[p], dm, rts[p], K)), (name, p)


@pytest.mark.parametrize("level", [0, 2])
@pytest.mark.parametrize("depth", ["f64", "f32", "u16"])
def test_batch_matches_per_pair_path(phovo, odo, pairs, depth, level):
    import torch
    capi = phovo.capi
    g0, d32, g1, rts = pairs
    if level == 2:                      # a level-2 frame (120x160) warped with K / 4
        g0, d32, g1 = (np.ascontiguousarray(a[:, 1::4, 1::4]) for a in (g0, d32, g1))
    d, scale = depth_variants(d32)[depth]
    wl, dl = loop(odo, g0, d, rts, K, level, g1, scale)
    nl, sl = summary_of(wl, dl)
    # numpy, pinned and CUDA inputs through the Python entry
    dev = torch.device("cuda", 0)
    tg0, td, tg1 = (torch.from_numpy(a.view(np.int16) if a.dtype == np.uint16 else a) for a in (g0, d, g1))
    for kind, args in (("numpy", (g0, d, g1)), ("pinned", tuple(t.pin_memory() for t in (tg0, td, tg1))),
                       ("cuda", tuple(t.to(dev) for t in (tg0, td, tg1)))):
        r = odo.BatchWarpImage(args[0], args[1], rts, K, level=level, gray1=args[2], depth_scale=scale)
        w = r["warped"] if kind != "cuda" else r["warped"].cpu().numpy()
        df = r["diff"] if kind != "cuda" else r["diff"].cpu().numpy()
        assert np.array_equal(w, wl), kind
        assert np.array_equal(df, dl), kind
        assert np.array_equal(r["num_landed"], nl) and np.array_equal(r["sum_abs_diff"], sl), kind
        assert np.array_equal(r["mean_abs_diff"], sl / np.maximum(nl, 1))
    # every combination of outputs, host and device, host and device inputs, through the C ABI
    code = {"f64": capi.DEPTH_F64, "f32": capi.DEPTH_F32, "u16": capi.DEPTH_U16}[depth]
    P = len(g0)
    cin = tuple(t.to(dev) for t in (tg0, td, tg1))
    for inputs in ((g0, d, g1), cin):
        for mask in (1, 2, 4, 8, 15):   # bits: warped, diff, num_landed, sum_abs_diff
            for out_dev in (False, True):
                mk = (lambda shape, dt: torch.zeros(shape, dtype=dt, device=dev)) if out_dev else \
                     (lambda shape, dt: torch.zeros(shape, dtype=dt))
                w = mk(g0.shape, torch.uint8) if mask & 1 else None
                df = mk(g0.shape, torch.uint8) if mask & 2 else None
                n = mk((P,), torch.int32) if mask & 4 else None
                s = mk((P,), torch.int64) if mask & 8 else None
                assert abi(odo, inputs[0], inputs[1], code, scale, rts, K, level, inputs[2], w, df, n, s) == 0, (mask, out_dev)
                if w is not None:
                    assert np.array_equal(w.cpu().numpy(), wl), (mask, out_dev)
                if df is not None:
                    assert np.array_equal(df.cpu().numpy(), dl), (mask, out_dev)
                if n is not None:
                    assert np.array_equal(n.cpu().numpy(), nl), (mask, out_dev)
                if s is not None:
                    assert np.array_equal(s.cpu().numpy(), sl), (mask, out_dev)


def test_summary_and_invisible_landed_pixels(odo, pairs):
    g0, d32, g1, rts = (a[:24] for a in pairs)
    r = odo.BatchWarpImage(g0, d32, rts, K, gray1=g1)
    m = r["warped"] > 0
    assert np.array_equal(r["num_landed"], m.reshape(24, -1).sum(1))
    assert np.array_equal(r["sum_abs_diff"], np.where(m, r["diff"], 0).reshape(24, -1).sum(1, dtype=np.int64))
    assert (r["num_landed"] > 0).all()
    # gray 0 everywhere: nothing visible, but landing is decided by geometry alone
    z = odo.BatchWarpImage(np.zeros_like(g0), d32, rts, K, gray1=g1)
    assert not z["warped"].any()
    assert np.array_equal(z["num_landed"], r["num_landed"])
    assert np.array_equal(z["diff"], g1)
    # summary only (no image buffers) gives the same numbers
    s = odo.BatchWarpImage(g0, d32, rts, K, gray1=g1, images=False)
    assert s["warped"] is None and s["diff"] is None
    assert np.array_equal(s["num_landed"], r["num_landed"]) and np.array_equal(s["sum_abs_diff"], r["sum_abs_diff"])
    # without gray1: warped and num_landed only
    o = odo.BatchWarpImage(g0, d32, rts, K)
    assert o["diff"] is None and o["sum_abs_diff"] is None and o["mean_abs_diff"] is None
    assert np.array_equal(o["warped"], r["warped"]) and np.array_equal(o["num_landed"], r["num_landed"])


def test_deterministic_and_permutation_equivariant(odo, pairs):
    g0, d32, g1, rts = pairs
    a = odo.BatchWarpImage(g0, d32, rts, K, gray1=g1)
    b = odo.BatchWarpImage(g0, d32, rts, K, gray1=g1)
    for k in ("warped", "diff", "num_landed", "sum_abs_diff"):
        assert np.array_equal(a[k], b[k]), k
    perm = np.random.default_rng(8).permutation(len(g0))
    c = odo.BatchWarpImage(g0[perm], d32[perm], rts[perm], K, gray1=g1[perm])
    for k in ("warped", "diff", "num_landed", "sum_abs_diff"):
        assert np.array_equal(c[k], a[k][perm]), k


def test_memset_cleared_keys_give_the_same_results(odo, pairs):
    g0, d32, g1, rts = (a[:60] for a in pairs)
    a = odo.BatchWarpImage(g0, d32, rts, K, gray1=g1)
    odo.BatchSetDebugFlags(16)
    try:
        b = odo.BatchWarpImage(g0, d32, rts, K, gray1=g1)
    finally:
        odo.BatchSetDebugFlags(0)
    c = odo.BatchWarpImage(g0, d32, rts, K, gray1=g1)     # keys left by the memset path: the next call starts clean
    for k in ("warped", "diff", "num_landed", "sum_abs_diff"):
        assert np.array_equal(a[k], b[k]) and np.array_equal(a[k], c[k]), k


def test_degenerate_inputs_land_nothing(odo, pairs):
    g0, d32, g1, rts = (a[:4].copy() for a in pairs)
    cases = {"zero depth": (np.zeros_like(d32), rts), "nan depth": (np.full_like(d32, np.nan), rts)}
    bad = rts.copy(); bad[:, 0, 3] = np.nan
    cases["non-finite Rt"] = (d32, bad)
    # every point on the camera's plane (Z = 0): the projection divides by zero
    flat = rts.copy(); flat[:, 2, :] = 0.
    cases["Z = 0"] = (d32, flat)
    for name, (d, rt) in cases.items():
        r = odo.BatchWarpImage(g0, d, rt, K, gray1=g1)
        assert not r["warped"].any() and (r["num_landed"] == 0).all() and (r["sum_abs_diff"] == 0).all(), name
        assert np.array_equal(r["diff"], g1), name


def test_points_behind_the_camera_follow_the_reference(odo, pairs):
    """The reference tests the SOURCE depth only (BASE:106), not Z > 0 after the transform: points behind the camera
    project mirrored through the principal point.  The batch does what the per-pair path does."""
    g0, d32, g1, rts = (a[:4].copy() for a in pairs)
    back = rts.copy(); back[:, 2, 3] = -20.       # every point ends up 15+ m behind the camera
    r = odo.BatchWarpImage(g0, d32, back, K, gray1=g1)
    wl, dl = loop(odo, g0, d32, back, K, 0, g1, 1.0)
    assert np.array_equal(r["warped"], wl) and np.array_equal(r["diff"], dl)
    assert np.array_equal(r["num_landed"], summary_of(wl, dl)[0])


def test_align_sequence_diagnostics(phovo, odo):
    import torch
    Kv = phovo.synth.K_VISUAL_ODOMETRY
    g, d = phovo.synth.render_sequence_torch(12, 480, 640, Kv, torch.device("cuda", 0))
    seq = phovo.CPhotoconsistencyOdometryCuda()
    seq.SetConfig(phovo.configs.to_config("config_5_level_optimization_analytic", phovo.capi))
    seq.SetIntrinsicMatrix(Kv)
    st, it, poses = seq.AlignSequence(g, d)
    st2, it2, poses2, diag = seq.AlignSequence(g, d, diagnostics=True)
    assert np.array_equal(st, st2) and np.array_equal(it, it2) and np.array_equal(poses, poses2)
    gn, dn = g.cpu().numpy(), d.cpu().numpy()
    for k in range(1, len(gn)):
        rt = phovo.state_to_rt(st[k - 1])
        w, df = odo.WarpImage(gn[k - 1], dn[k - 1], rt, Kv, targetImage=gn[k])
        # a landed pixel of gray 0 is invisible in w: count landing from a gray0 >= 1 copy
        w1 = odo.WarpImage(np.maximum(gn[k - 1], 1), dn[k - 1], rt, Kv)
        m = w1 > 0
        assert diag["num_landed"][k - 1] == m.sum(), k
        assert diag["sum_abs_diff"][k - 1] == np.where(m, df, 0).sum(dtype=np.int64), k
    assert np.array_equal(diag["mean_abs_diff"], diag["sum_abs_diff"] / np.maximum(diag["num_landed"], 1))


def test_error_paths_and_release(phovo, odo, pairs):
    capi = phovo.capi
    g0, d32, g1, rts = (a[:2] for a in pairs)
    w = np.zeros_like(g0); n = np.zeros(2, np.int32); s = np.zeros(2, np.int64)
    E = capi.E_INVALID
    assert abi(odo, g0, d32, capi.DEPTH_F32, 1., rts, K, 0, g1, w, None, None, None) == 0
    assert abi(odo, g0, d32, capi.DEPTH_F32, 1., rts, K, -1, g1, w, None, None, None) == E        # level
    assert abi(odo, g0, d32, capi.DEPTH_F32, 1., rts, K, 31, g1, w, None, None, None) == E
    assert abi(odo, g0, d32, 7, 1., rts, K, 0, g1, w, None, None, None) == E                      # depth type
    assert abi(odo, g0, d32, capi.DEPTH_F32, 1., rts, K, 0, None, w, w, None, None) == E          # diff without gray1
    assert abi(odo, g0, d32, capi.DEPTH_F32, 1., rts, K, 0, None, None, None, n, s) == E          # sum without gray1
    assert abi(odo, g0, d32, capi.DEPTH_F32, 1., rts, K, 0, g1, None, None, None, None) == E      # no output
    Kc = K.reshape(9).copy()
    assert odo._L.phovo_batch_warp_image(odo._h, 0, 480, 640, capi._ptr(g0), capi._ptr(d32), capi.DEPTH_F32, 1.,
                                         capi._ptr(rts), Kc.ctypes.data_as(capi._dp), 0, None, capi._ptr(w), None, None, None) == E
    assert odo._L.phovo_batch_warp_image(odo._h, 2, 0, 640, capi._ptr(g0), capi._ptr(d32), capi.DEPTH_F32, 1.,
                                         capi._ptr(rts), Kc.ctypes.data_as(capi._dp), 0, None, capi._ptr(w), None, None, None) == E
    ref = odo.BatchWarpImage(g0, d32, rts, K, gray1=g1)
    odo.BatchReleaseMemory()
    again = odo.BatchWarpImage(g0, d32, rts, K, gray1=g1)
    for k in ("warped", "diff", "num_landed", "sum_abs_diff"):
        assert np.array_equal(ref[k], again[k]), k
    # the per-pair path shares the keys: it still works after the release too
    assert np.array_equal(odo.WarpImage(g0[0], d32[0], rts[0], K), ref["warped"][0])
