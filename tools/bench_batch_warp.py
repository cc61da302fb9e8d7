#!/usr/bin/env python
"""Throughput of phovo_batch_warp_image (BatchWarpImage): 4096 device-resident 640x480 pairs with u16 depth, summary only
and with both images, against the per-pair WarpImage loop and a device-to-device copy peak measured in the same run;
AlignSequence on 1000 frames with and without `diagnostics`.  Prints one JSON line (profiles/r03_batch_warp.json).
usage (GPU box): python tools/bench_batch_warp.py [--pairs 4096] [--loop-pairs 256] [--frames 1000] [--reps 5]"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines() or [","])[0].split(",")[:2]
    return {"gpu": name.strip(), "power_limit": power.strip()}


def timed(fn, reps):
    """Median device time (CUDA events on the current stream) and host wall time of `fn`, ms; `fn` blocks."""
    import torch
    dev, wall = [], []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        wall.append((time.perf_counter() - t0) * 1e3)
        dev.append(a.elapsed_time(b))
    return float(np.median(dev)), float(np.median(wall))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=4096)
    ap.add_argument("--loop-pairs", type=int, default=256)
    ap.add_argument("--frames", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    phovo = importlib.import_module("photoconsistency-visual-odometry_b200")
    phovo.build()
    dev = torch.device("cuda", 0)
    out = {"tool": "bench_batch_warp", **gpu_info(), "rows": 480, "cols": 640, "depth": "u16 * 1/5000", "pairs": args.pairs}

    # ---- inputs: seeded, device-resident; 4096 pairs are 5 GB, far beyond the L2 ----
    K = phovo.synth.K_FRAME_ALIGNMENT
    P, n = args.pairs, 480 * 640
    g0, d32, g1, _ = phovo.synth.render_batch_torch(P, 480, 640, K, dev, seed0=2024)
    raw = torch.clamp(torch.round(d32.double() * 5000.), 0, 65535).to(torch.int32)
    d0 = torch.where(raw > 32767, raw - 65536, raw).to(torch.int16)       # u16 bits in an int16 tensor
    del raw
    del d32
    rng = np.random.default_rng(2024)
    states = np.concatenate([rng.uniform(-0.05, 0.05, (P, 3)), rng.uniform(-0.03, 0.03, (P, 3))], axis=1)
    rts = np.stack([phovo.state_to_rt(s) for s in states])
    rts_dev = torch.from_numpy(rts).to(dev)
    odo = phovo.CPhotoconsistencyOdometryCuda()
    scale = 1. / 5000.

    # ---- device-to-device copy peak (>= 1 GiB each way) ----
    src = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
    dst = torch.empty_like(src)
    dst.copy_(src)
    copy_ms, _ = timed(lambda: dst.copy_(src), args.reps)
    peak = 2 * src.numel() / (copy_ms * 1e-3)
    del src, dst
    out["d2d_copy_peak_GBps"] = round(peak / 1e9, 1)

    # ---- the batch: summary only, both images; keys cleared in the resolve pass (default) or by a memset per chunk ----
    warped = torch.empty((P, 480, 640), dtype=torch.uint8, device=dev)
    diff = torch.empty_like(warped)
    landed = torch.empty(P, dtype=torch.int32, device=dev)
    sums = torch.empty(P, dtype=torch.int64, device=dev)
    capi = phovo.capi
    Kc = np.ascontiguousarray(K, dtype=np.float64).reshape(9)
    torch_stream = torch.cuda.current_stream(dev).cuda_stream
    odo.SetStream(torch_stream)

    def call(images):
        rc = odo._L.phovo_batch_warp_image(odo._h, P, 480, 640, g0.data_ptr(), d0.data_ptr(), capi.DEPTH_U16, scale, rts_dev.data_ptr(),
                                           Kc.ctypes.data_as(capi._dp), 0, g1.data_ptr(), warped.data_ptr() if images else None,
                                           diff.data_ptr() if images else None, landed.data_ptr(), sums.data_ptr())
        assert rc == 0, rc

    compulsory = {"summary": 4 * n, "images": 6 * n}     # gray0 + u16 depth0 + gray1 in (+ warped + diff out), bytes per pair
    for key, images in (("summary", False), ("images", True)):
        for flags, suffix in ((0, ""), (16, "_memset_keys")):
            odo.BatchSetDebugFlags(flags)
            call(images)                                   # warm-up: keys, Rt buffer, summaries
            ms, wall = timed(lambda: call(images), args.reps)
            r = {"ms_per_call": round(ms, 3), "wall_ms_per_call": round(wall, 3), "pairs_per_s": round(P / (ms * 1e-3)),
                 "compulsory_bytes_per_pair": compulsory[key],
                 "achieved_GBps": round(compulsory[key] * P / (ms * 1e-3) / 1e9, 1),
                 "fraction_of_d2d_copy_peak": round(compulsory[key] * P / (ms * 1e-3) / peak, 3)}
            out["batch_" + key + suffix] = r
    odo.BatchSetDebugFlags(0)
    call(True)
    torch.cuda.synchronize()
    batch_landed, batch_sums = landed.cpu().numpy(), sums.cpu().numpy()

    # ---- per-pair WarpImage loop on the first pairs (host inputs, as the per-pair API takes them) ----
    L = min(args.loop_pairs, P)
    hg0, hd0, hg1 = g0[:L].cpu().numpy(), d0[:L].cpu().numpy().view(np.uint16), g1[:L].cpu().numpy()
    odo.WarpImage(hg0[0], hd0[0], rts[0], K, targetImage=hg1[0], depth_scale=scale)
    t0 = time.perf_counter()
    res = [odo.WarpImage(hg0[p], hd0[p], rts[p], K, targetImage=hg1[p], depth_scale=scale) for p in range(L)]
    loop_s = time.perf_counter() - t0
    wl, dl = np.stack([w for w, _ in res]), np.stack([d for _, d in res])
    bw, bd = warped[:L].cpu().numpy(), diff[:L].cpu().numpy()
    out["per_pair_loop"] = {"pairs": L, "ms_per_pair": round(1e3 * loop_s / L, 4), "pairs_per_s": round(L / loop_s, 1)}
    out["speedup_batch_images_vs_loop"] = round(out["batch_images"]["pairs_per_s"] / (L / loop_s), 1)
    m = bw > 0
    out["bitwise_equal_batch_vs_loop"] = bool(np.array_equal(bw, wl) and np.array_equal(bd, dl) and
                                              (batch_landed[:L] >= m.reshape(L, -1).sum(1)).all())
    out["mean_abs_diff_per_landed_pixel"] = round(float(batch_sums.sum() / max(batch_landed.sum(), 1)), 3)
    out["landed_fraction"] = round(float(batch_landed.sum()) / (P * n), 4)
    del g0, d0, g1, warped, diff

    # ---- AlignSequence with and without the per-frame summary ----
    Kv = phovo.synth.K_VISUAL_ODOMETRY
    gs, ds = phovo.synth.render_sequence_torch(args.frames, 480, 640, Kv, dev)
    seq = phovo.CPhotoconsistencyOdometryCuda()
    seq.SetConfig(phovo.configs.to_config("config_5_level_optimization_analytic", phovo.capi))
    seq.SetIntrinsicMatrix(Kv)
    for diag in (False, True):
        seq.AlignSequence(gs, ds, diagnostics=diag)
        ms, wall = timed(lambda: seq.AlignSequence(gs, ds, diagnostics=diag), 3)
        out["align_sequence" + ("_diagnostics" if diag else "")] = {"frames": args.frames, "wall_ms": round(wall, 2),
                                                                     "frames_per_s": round((args.frames - 1) / (wall * 1e-3))}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
