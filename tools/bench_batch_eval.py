#!/usr/bin/env python
"""Throughput of phovo_batch_eval_normal_equations (BatchEvalNormalEquations): 4096 device-resident 640x480 pairs with
u16 depth at levels 0 and 2, its split by kernel (torch.profiler, after the timed runs), algorithmic HBM bytes and FP64
instructions from the shapes against the measured peaks, and the per-pair loop (SetSourceFrame + SetTargetFrame +
EvalNormalEquations) on 64 of the same pairs.  Prints one JSON line (profiles/r04_batch_eval.json).
--mode 3: the photometric + depth solver through phovo_batch_eval_normal_equations_with_target_depth, with a target
depth per pair (the next pair's depth0), its per-pair loop with SetTargetFrame(gray1, depth1), and AlignSequence on
--sequence-frames frames with and without information_level=0 (profiles/r05_batch_eval_bi.json).
usage (GPU box): python tools/bench_batch_eval.py [--mode 0] [--pairs 4096] [--loop-pairs 64] [--reps 5]
                 [--sequence-frames 1000] [--out FILE]"""
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

# FP64 thread instructions per pixel, static counts of the kernels' SASS (sm_100a, u16 depth, mode 0): the winner pass
# (exact warp with a true division, unrolled 8 pixels per thread) per source pixel, the accumulate pass (Jacobian,
# 21 + 6 + 1 FMAs of the sums) per valid pixel.  The per-tile reduction and the pyramid are not counted.
FP64_WINNER_PER_PX = 53
FP64_ACCUMULATE_PER_VALID_PX = 85
# mode 3: the accumulate pass of the 2N-row system (residual, bi_jacobian_core with its true division, 27 FMAs of the
# sums) per non-zero row, estimated from the kernel's static count (152 with the per-tile reduction); at most 2 rows per
# valid source pixel are non-zero, which is what the bound below assumes
FP64_ACCUMULATE_BI_PER_ROW = 95
# measured FP64 peak of this pool's B200 (tools/fp64_peak.cu, profiles/r01_fp64_peak.jsonl): DFMA thread instructions / s
FP64_PEAK_INST_PER_S = 1.7055e13


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


def kernel_split(fn, calls=3):
    """Device ms per kernel name (torch.profiler, CUDA activities), mean over `calls` calls."""
    import torch
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    agg = {}
    for e in prof.events():
        if e.device_type.name == "CUDA":
            name = e.name
            for short in ("k_eval_winner_bi", "k_eval_accumulate_bi", "k_eval_target_depth", "k_eval_gain", "k_eval_winner",
                          "k_eval_accumulate", "k_eval_reduce", "k_eval_poses", "k_batch_pyramid"):
                if short in name:
                    name = short
                    break
            agg[name] = agg.get(name, 0.) + e.device_time_total / calls / 1e3
    return {k: round(v, 3) for k, v in sorted(agg.items(), key=lambda x: -x[1])[:8]}


def align_sequence(phovo, frames, R, C, reps):
    """AlignSequence (mode 3) on `frames` device-resident frames of the synthetic VO sequence, u16 depth: wall time of
    the call (it blocks) without and with information_level=0."""
    import torch
    K = phovo.synth.K_VISUAL_ODOMETRY
    gray = np.empty((frames, R, C), np.uint8)
    depth = np.empty((frames, R, C), np.uint16)
    for k in range(frames):
        g, d = phovo.synth.make_sequence_frame(k, R, C, K=K, n=frames)
        gray[k], depth[k] = g, np.clip(np.rint(d * 5000.), 0, 65535).astype(np.uint16)
    dev = torch.device("cuda", 0)
    gd, dd = torch.from_numpy(gray).to(dev), torch.from_numpy(depth.view(np.int16)).to(dev)
    odo = phovo.CPhotoconsistencyOdometryCuda()
    odo.SetConfig(phovo.configs.to_config("config_4_level_optimization_analytic", phovo.capi, mode=3))
    odo.SetIntrinsicMatrix(K)
    res = {"frames": frames, "rows": R, "cols": C}
    for what, kw in (("align", {}), ("align_and_information_level0", {"information_level": 0})):
        odo.AlignSequence(gd, dd, depth_scale=1. / 5000., **kw)              # warm-up
        walls = []
        for _ in range(reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = odo.AlignSequence(gd, dd, depth_scale=1. / 5000., **kw)
            torch.cuda.synchronize()
            walls.append(time.perf_counter() - t0)
        res[what] = {"s_per_call": round(float(np.median(walls)), 4), "frames_per_s": round((frames - 1) / float(np.median(walls)), 1),
                     "path": odo.BatchLastPath() if not kw else None}
        if not kw:
            res["mean_iterations_per_pair"] = round(float(out[1].sum(1).mean()), 2)
    odo.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=4096)
    ap.add_argument("--loop-pairs", type=int, default=64)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--mode", type=int, default=0, choices=(0, 1, 3), help="solver mode (3: photometric + depth)")
    ap.add_argument("--sequence-frames", type=int, default=0, help="mode 3: AlignSequence on this many 640x480 frames")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    phovo = importlib.import_module("photoconsistency-visual-odometry_b200")
    phovo.build()
    dev = torch.device("cuda", 0)
    R, C = 480, 640
    bi = args.mode == 3
    out = {"tool": "bench_batch_eval", **gpu_info(), "rows": R, "cols": C, "depth": "u16 * 1/5000", "pairs": args.pairs,
           "config": "config_4_level_optimization_analytic (mode %d)" % args.mode}
    if bi:
        out["target_depth"] = "depth0 of the next pair (pair P-1 takes pair 0's)"

    # ---- inputs: seeded, device-resident; 4096 pairs are 5 GB, far beyond the L2 ----
    K = phovo.synth.K_FRAME_ALIGNMENT
    P, n = args.pairs, R * C
    g0, d32, g1, _ = phovo.synth.render_batch_torch(P, R, C, K, dev, seed0=2024)
    raw = torch.clamp(torch.round(d32.double() * 5000.), 0, 65535).to(torch.int32)
    d0 = torch.where(raw > 32767, raw - 65536, raw).to(torch.int16)       # u16 bits in an int16 tensor
    del raw, d32
    d1 = torch.roll(d0, -1, dims=0).contiguous() if bi else None
    rng = np.random.default_rng(2024)
    states = np.concatenate([rng.uniform(-0.05, 0.05, (P, 3)), rng.uniform(-0.03, 0.03, (P, 3))], axis=1)
    st_dev = torch.from_numpy(states).to(dev)
    odo = phovo.CPhotoconsistencyOdometryCuda()
    odo.SetConfig(phovo.configs.to_config("config_4_level_optimization_analytic", phovo.capi, mode=args.mode or None))
    odo.SetIntrinsicMatrix(K)
    odo.SetStream(torch.cuda.current_stream(dev).cuda_stream)
    scale = 1. / 5000.
    capi = phovo.capi
    H = torch.empty((P, 21), dtype=torch.float64, device=dev)
    g = torch.empty((P, 6), dtype=torch.float64, device=dev)
    cost = torch.empty(P, dtype=torch.float64, device=dev)
    nv = torch.empty(P, dtype=torch.int32, device=dev)

    def call(level):
        if bi:
            rc = odo._L.phovo_batch_eval_normal_equations_with_target_depth(
                odo._h, P, R, C, g0.data_ptr(), d0.data_ptr(), capi.DEPTH_U16, scale, g1.data_ptr(), d1.data_ptr(),
                st_dev.data_ptr(), level, H.data_ptr(), g.data_ptr(), cost.data_ptr(), nv.data_ptr())
            assert rc == 0, rc
            return
        rc = odo._L.phovo_batch_eval_normal_equations(odo._h, P, R, C, g0.data_ptr(), d0.data_ptr(), capi.DEPTH_U16, scale,
                                                      g1.data_ptr(), st_dev.data_ptr(), level, H.data_ptr(), g.data_ptr(),
                                                      cost.data_ptr(), nv.data_ptr())
        assert rc == 0, rc

    results = {}
    for level in (0, 2):
        call(level)                                    # warm-up: keys, records, partials
        ms, wall = timed(lambda: call(level), args.reps)
        torch.cuda.synchronize()
        valid = int(nv.sum().item())
        ln = (R >> level) * (C >> level)
        # compulsory HBM: gray0 + u16 depth0 + gray1 (4 B per full-resolution pixel) at level 0; above level 0 the pyramid
        # kernel reads the two central rows of every 2^level, i.e. 2 / 2^level of the frames; keys, validity, level
        # records and partials stay in the L2 (chunks sized to half of it)
        hbm = 4 * n * P if level == 0 else 4 * n * P * 2 // (1 << level)
        fp64 = FP64_WINNER_PER_PX * ln * P + FP64_ACCUMULATE_PER_VALID_PX * valid
        if bi:
            # + the target depth (2 B per full-resolution pixel at level 0; the taps of the central 2 of every 2^level
            # rows above it) and, per level pixel, D1 / GxD / GyD written and read back (L2-resident by the chunking)
            hbm += 2 * n * P if level == 0 else 2 * n * P * 2 // (1 << level)
            fp64 = FP64_WINNER_PER_PX * ln * P + FP64_ACCUMULATE_BI_PER_ROW * 2 * valid
        t_hbm, t_fp64 = hbm / 7.7e12, fp64 / FP64_PEAK_INST_PER_S
        results[level] = dict(H=H.cpu().numpy().copy(), g=g.cpu().numpy().copy(), cost=cost.cpu().numpy().copy(),
                              nv=nv.cpu().numpy().copy())
        out["level%d" % level] = {
            "level_rows": R >> level, "level_cols": C >> level, "ms_per_call": round(ms, 3), "wall_ms_per_call": round(wall, 3),
            "pairs_per_s": round(P / (ms * 1e-3)), "valid_fraction": round(valid / (ln * P), 4),
            "hbm_bytes": hbm, "fp64_thread_inst": fp64,
            "min_ms_hbm_7.7TBps": round(t_hbm * 1e3, 3), "min_ms_fp64_measured_peak": round(t_fp64 * 1e3, 3),
            "bound": "fp64" if t_fp64 > t_hbm else "hbm",
            "fraction_of_bound": round(max(t_hbm, t_fp64) * 1e3 / ms, 3)}

    # ---- per-pair loop on the first pairs (host inputs, as the per-pair API takes them) ----
    L = min(args.loop_pairs, P)
    hg0, hd0, hg1 = g0[:L].cpu().numpy(), d0[:L].cpu().numpy().view(np.uint16), g1[:L].cpu().numpy()
    ref = phovo.CPhotoconsistencyOdometryCuda()
    ref.SetConfig(phovo.configs.to_config("config_4_level_optimization_analytic", phovo.capi, mode=args.mode or None))
    ref.SetIntrinsicMatrix(K)
    ref.SetBuildAllLevels(True)
    hd1 = d1[:L].cpu().numpy().view(np.uint16) if bi else [None] * L
    ref.SetSourceFrame(hg0[0], hd0[0], depth_scale=scale)
    ref.SetTargetFrame(hg1[0], hd1[0], depth_scale=scale)
    ref.EvalNormalEquations(0, states[0])
    loop = {}
    worst = {0: [0., 0., 0.], 2: [0., 0., 0.]}
    iu = np.triu_indices(6)
    for level in (0, 2):
        t0 = time.perf_counter()
        per = []
        for p in range(L):
            ref.SetSourceFrame(hg0[p], hd0[p], depth_scale=scale)
            ref.SetTargetFrame(hg1[p], hd1[p], depth_scale=scale)
            per.append(ref.EvalNormalEquations(level, states[p]))
        loop_s = time.perf_counter() - t0
        loop[level] = L / loop_s
        r = results[level]
        same_valid = all(int(r["nv"][p]) == per[p]["num_valid"] for p in range(L))
        for p in range(L):
            Hr, gr = np.asarray(per[p]["H"]), np.asarray(per[p]["g"])
            d = np.sqrt(np.abs(Hr[[0, 6, 11, 15, 18, 20]]))
            scale_h = np.outer(d, d)[iu]
            worst[level][0] = max(worst[level][0], float(np.max(np.abs(r["H"][p] - Hr) / scale_h)))
            worst[level][1] = max(worst[level][1], float(np.max(np.abs(r["g"][p] - gr)) / np.max(np.abs(gr))))
            worst[level][2] = max(worst[level][2], abs(r["cost"][p] - per[p]["cost"]) / per[p]["cost"])
        out["level%d" % level]["per_pair_loop"] = {
            "pairs": L, "ms_per_pair": round(1e3 * loop_s / L, 4), "pairs_per_s": round(L / loop_s, 1),
            "speedup_batch_vs_loop": round(out["level%d" % level]["pairs_per_s"] / (L / loop_s), 1),
            "num_valid_equal": bool(same_valid), "max_h_rel_err": worst[level][0], "max_g_rel_err": worst[level][1],
            "max_cost_rel_err": worst[level][2]}

    # ---- split by kernel: a profiled pass after the timed ones ----
    for level in (0, 2):
        out["level%d" % level]["kernel_ms"] = kernel_split(lambda: call(level))
    if bi and args.sequence_frames > 1:
        out["align_sequence"] = align_sequence(phovo, args.sequence_frames, R, C, args.reps)
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
