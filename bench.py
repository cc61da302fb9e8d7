#!/usr/bin/env python
"""bench.py -- headline benchmark: aligned RGB-D pairs/sec @640x480, 4-level Gauss-Newton.

Workload (BASELINE.json configs[3]): a batch of independent synthetic 640x480 RGB-D pairs aligned
with config_4_level_optimization_analytic (levels 3 and 2 active, <=50 / <=20 iterations,
gradient-norm stop at 300), sharded by pair across the GPUs: every rank aligns `--pairs` pairs
(weak scaling, no data-path collective; one final pose gather per step when N > 1).

  value   : pairs/s with the inputs already resident in HBM (CUDA events, max over ranks)
  e2e     : pairs/s through the reference-facing C ABI with HOST (pinned) buffers: the H2D copy of
            every pair and the D2H read of the poses are inside the timed region
  roofline: the dominant kernel (k_batch_level, one launch per active level) -- algorithmic bytes per SURVEY 8(d)
            (20 B/px per executed GN iteration + 216 B of sums) / its CUDA-event time, against the
            measured HBM copy bandwidth in MEASURED_PEAKS.json; the kernel is bound by the FP64 pipe
            (`bound: "fp64"`, `roofline.fp64`), the HBM figure is the contract's number
  cpu_baseline / --impl reference: the CPU oracle (faithful port of the reference's analytic path,
            the reference itself cannot be built here: no OpenCV/Eigen) on the host cores
  secondary: (N = 1) the other BASELINE configs measured in the same run, each with its own clock
            samples and the CPU oracle beside it: one 640x480 pair through SetSourceFrame ->
            SetTargetFrame -> Optimize from host buffers (configs[0]), the VO loop per frame
            (configs[1]), config_5_level_optimization_ceres (configs[2]), the 7680x4320 pair on one
            GPU (configs[4]).  What the reference times: FrameAlignment.cpp:99-101, VisualOdometry.cpp:227-230.

One JSON line on stdout (rank 0).
"""
import argparse
import ctypes as C
import importlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
PKG = "photoconsistency-visual-odometry_b200"
ROWS, COLS = 480, 640
CONFIG = "config_4_level_optimization_analytic"
METRIC = "aligned RGB-D pairs/sec @640x480 4-level GN"


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock, power and throttle reasons sampled DURING the timed region (NVML, ~2 ms period;
    nvidia-smi -lms as the fallback when pynvml cannot be loaded)."""
    BAD = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, index, period=0.001):
        self.index, self.samples, self.stop_flag, self.thread, self.nvml, self.err = index, [], False, None, None, None
        self.period = period      # sleep between samples; NVML queries take driver locks, so host-launch-heavy regions use a longer one

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.index
            if visible:
                try:
                    idx = int(visible.split(",")[self.index])
                except ValueError:
                    idx = self.index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.nvml = pynvml
            self.smax = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
            # the first call of each query can take tens of milliseconds: pay for it before the timed region
            pynvml.nvmlDeviceGetClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
            pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
            pynvml.nvmlDeviceGetPowerUsage(self.handle)
        except Exception as e:  # pragma: no cover
            self.err = repr(e)
            return
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def _run(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                reasons = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                # power is a slow query: every 8th sample is enough for the maximum
                power = n.nvmlDeviceGetPowerUsage(self.handle) / 1000.0 if len(self.samples) % 8 == 0 else 0.0
                self.samples.append((sm, reasons, power))
            except Exception as e:  # pragma: no cover
                self.err = repr(e)
                break
            time.sleep(self.period)

    def stop(self):
        self.stop_flag = True
        if self.thread:
            self.thread.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples: %s" % (self.err or "timed region too short")]}
        sm = sorted(x[0] for x in self.samples)
        mask = 0
        for x in self.samples:
            mask |= x[1]
        return {"sm_mhz": float(sm[len(sm) // 2]), "sm_max_mhz": float(self.smax), "power_w_max": max(x[2] for x in self.samples),
                "samples": len(self.samples), "reasons": sorted(k for k, b in self.BAD.items() if mask & b)}


def bind_to_gpu_numa_node(index):
    """Pin this process to the CPUs NVML reports as local to GPU `index`, so that its pinned host buffers are
    allocated on (and copied from) the GPU's own NUMA node.  Matters for `e2e` when several ranks upload at once."""
    try:
        import pynvml
        pynvml.nvmlInit()
        visible = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = index
        if visible:
            try:
                idx = int(visible.split(",")[index])
            except ValueError:
                idx = index
        h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def rows_read_fraction(cfg, rows):
    """Fraction of the source rows the active pyramid levels tap: level l >= 1 is decimated from the ORIGINAL
    image and reads the two central rows of each 2^l-row cell (AN:132), level 0 reads every row."""
    need = set()
    for lvl in range(cfg.num_levels):
        if cfg.max_num_iterations[lvl] <= 0:
            continue
        if lvl == 0:
            return 1.0
        cell = 1 << lvl
        for y in range(int(round(rows * 0.5 ** lvl))):
            need.update((min(y * cell + cell // 2 - 1, rows - 1), min(y * cell + cell // 2, rows - 1)))
    return len(need) / float(rows)


def algorithmic_bytes(cfg, iters, rows, cols, depth_bytes):
    """SURVEY 8(d): 20 B/px per executed GN iteration at a level of N px + 216 B out per iteration.
    Frame set-up (k_batch_pyramid): the COMPULSORY traffic -- the source rows the active levels tap of
    gray0, gray1 (1 B/px) and depth0 (`depth_bytes` B/px; whole 32-byte sectors, so every column of such
    a row counts) in, the packed record (f64 D0 + u16 I0 + u16 I1 = 12 B per active-level pixel) out."""
    import numpy as np
    total_iter_bytes, active_px = 0.0, 0
    for lvl in range(cfg.num_levels):
        if cfg.max_num_iterations[lvl] <= 0:
            continue
        n = int(round(rows * 0.5 ** lvl)) * int(round(cols * 0.5 ** lvl))
        active_px += n
        total_iter_bytes += float(np.sum(iters[:, lvl])) * (20.0 * n + 216.0)
    setup = iters.shape[0] * (rows_read_fraction(cfg, rows) * rows * cols * (2.0 + depth_bytes) + 12.0 * active_px)
    return total_iter_bytes, setup


DEPTH_SCALE = 1. / 5000.   # raw u16 sensor units -> metres (TUM convention, VisualOdometry.cpp:163)


def quantise_depth(d_metres):
    """metres -> raw u16 sensor units, the format both reference apps read from disk."""
    import numpy as np
    return np.clip(np.rint(d_metres * 5000.), 0, 65535).astype(np.uint16)


def oracle_config(phovo, name):
    """The named reference configuration as the ORACLE's POD (same layout as phovo_config) -- built without
    touching capi, so the CPU arm never maps libphovo_b200.so."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_py
    return phovo.configs.to_config(name, oracle_py)


def cpu_reference(phovo, K, pairs, threads, steps, warmup, lean=False, depth="u16"):
    """The CPU arm: the oracle port of the reference's analytic path, `threads` independent
    single-threaded alignments at a time (the reference itself is single-threaded, OpenMP off)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np
    import oracle_py
    oracle_py.build()
    distinct = min(pairs, 32)          # rendering on the host is slow; the sample repeats 32 distinct pairs
    g0, d0, g1, _ = phovo.synth.make_batch(distinct, ROWS, COLS, K=K, seed0=0)
    raw = quantise_depth(d0) if depth == "u16" else None
    if raw is not None:
        d0 = raw.astype(np.float64) * DEPTH_SCALE      # what the apps hand to SetSourceFrame (cv::Mat_<double>)
    reps = (pairs + distinct - 1) // distinct
    g0, d0, g1 = (np.tile(a, (reps, 1, 1))[:pairs] for a in (g0, d0, g1))
    raw = np.tile(raw, (reps, 1, 1))[:pairs] if raw is not None else None
    cfg = oracle_config(phovo, CONFIG)
    times, opt_times = [], []
    for s in range(warmup + steps):
        st, it, wall, opt = oracle_py.align_batch(cfg, K, g0, d0, g1, num_threads=threads, lean=lean)
        if s >= warmup:
            times.append(wall)
            opt_times.append(opt)
    wall = float(np.mean(times))
    return {"value": pairs / wall, "ms_per_step": wall * 1e3, "optimize_only_pairs_per_core_s": pairs / float(np.mean(opt_times)),
            "states": st, "iters": it, "inputs": (g0, d0, g1), "raw_depth": raw,
            "mean_iterations_per_pair": {str(l): float(it[:, l].mean()) for l in range(cfg.num_levels) if cfg.max_num_iterations[l] > 0}}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """--dump-outputs: the arrays the timed path returned in its last step, as <out_dir>/<name>.npy in float64,
    so that two builds can be compared output for output on the same seeded inputs.  When together they exceed
    64 MB, the arrays (which then share their first axis, the pair) keep a fixed, seeded sample of pairs whose
    indices are written as pair_index.npy."""
    import numpy as np
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        n = {a.shape[0] for a in arrays.values()}
        assert len(n) == 1, "outputs larger than the dump limit must share their first axis"
        n = n.pop()
        keep = DUMP_LIMIT_BYTES * n // (total + 8 * n)      # the index costs 8 B per kept pair
        idx = np.sort(np.random.default_rng(0).choice(n, size=keep, replace=False))
        arrays = {k: a[idx] for k, a in arrays.items()}
        arrays["pair_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


def workload_config(pairs_per_gpu, depth, world):
    """`config` of the JSON line: the workload and nothing measured, identical in both arms."""
    return {"workload": "batched independent 640x480 RGB-D pairs, %s (BASELINE configs[3]), %d pairs per GPU per step" % (CONFIG, pairs_per_gpu),
            "pairs_per_gpu": pairs_per_gpu, "rows": ROWS, "cols": COLS,
            "depth_dtype": "u16 raw x 1/5000 m" if depth == "u16" else "f32 metres",
            "parallelism": "pairs sharded x%d, final pose all_gather" % world,
            "l2_policy": "inputs larger than L2 (%.1f GB of frames per step)" % (pairs_per_gpu * ROWS * COLS * (2 + (2 if depth == "u16" else 4)) / 1e9)}


def pinned_h2d_peak(torch, dev, stream, nbytes=1 << 30, reps=5):
    """Best-of-`reps` bandwidth of one cudaMemcpyAsync of `nbytes` from pinned host memory to the device:
    the ceiling `e2e` can be compared with (measured in this run, on this rank's link)."""
    host = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    host.fill_(1)
    buf = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    best = 0.0
    for _ in range(reps + 1):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        buf.copy_(host, non_blocking=True)
        b.record(stream)
        b.synchronize()
        best = max(best, nbytes / (a.elapsed_time(b) * 1e-3) / 1e9)
    del host, buf
    return best


def median(xs):
    import numpy as np
    return float(np.median(xs)) if len(xs) else None


def secondary_block(phovo, torch, dev, local_rank, frames):
    """BASELINE configs[0], [1], [2] and [4] through the reference-facing per-pair API, host buffers in -> pose
    out, each under its own clock sampler, with the single-threaded CPU oracle (the reference is single-threaded)
    on the same inputs.  Device times are CUDA events recorded by the library around the frame set-up
    (uploads + pyramid kernels) and around Optimize() -- what the apps' TickMeter brackets."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np
    import oracle_py
    oracle_py.build()
    out = {}

    def pin(a):
        return torch.from_numpy(np.ascontiguousarray(a)).pin_memory()

    def timed_alignments(odo, src, tgt, reps, warm):
        """`warm` untimed alignments, and at least half a second of them: after an idle stretch (the CPU baseline runs
        just before this) the first host-to-device copies run at the PCIe link's idle speed -- set-up measures 0.28 ms
        instead of 0.10 ms until the link is back up (same code, measured both ways)."""
        setup, opt, wall = [], [], []
        sampler = ClockSampler(local_rank)

        def align():
            odo.SetSourceFrame(*src)
            odo.SetTargetFrame(tgt)
            odo.SetInitialStateVector(np.zeros(6))
            odo.Optimize()
            return odo.GetOptimalStateVector()
        t_warm, n_warm = time.perf_counter() + 0.5, 0
        while n_warm < warm or (time.perf_counter() < t_warm and n_warm < 2000):
            align(); n_warm += 1
        sampler.start()
        for rep in range(reps):
            t0 = time.perf_counter()
            s = align()
            t1 = time.perf_counter()
            a, b = odo.Timings()
            setup.append(a); opt.append(b); wall.append((t1 - t0) * 1e3)
        return s, setup, opt, wall, sampler.stop()

    def oracle_alignment(cfg_name, K, g0, d0, g1, reps):
        o = oracle_py.Oracle(oracle_config(phovo, cfg_name), K)
        t_opt, t_all = [], []
        for _ in range(reps):
            t0 = time.perf_counter()
            o.set_source(g0, d0); o.set_target(g1); o.set_initial_state(np.zeros(6))
            t1 = time.perf_counter()
            o.optimize()
            t2 = time.perf_counter()
            t_opt.append((t2 - t1) * 1e3); t_all.append((t2 - t0) * 1e3)
        return o, median(t_opt), median(t_all)

    # ---- configs[0]: PhotoconsistencyFrameAlignment, one 640x480 pair (depth cv::Mat_<double>, like the app)
    for key, cfg_name, reps, what in (
            ("single_pair_640x480", CONFIG, 200, "BASELINE configs[0]: PhotoconsistencyFrameAlignment, one 640x480 pair, 4-level analytic"),
            ("ceres_config_640x480", "config_5_level_optimization_ceres", 30, "BASELINE configs[2]: config_5_level_optimization_ceres on a 640x480 pair (levels 0 and 1 optimised); LM restated, Ceres itself absent")):
        K = phovo.synth.K_FRAME_ALIGNMENT
        g0, d0, g1, _ = phovo.synth.make_pair(ROWS, COLS, K=K, seed=0)
        odo = phovo.CPhotoconsistencyOdometryCuda(device=local_rank)
        odo.SetConfig(phovo.configs.to_config(cfg_name, phovo.capi)); odo.SetIntrinsicMatrix(K)
        s, setup, opt, wall, clocks = timed_alignments(odo, (pin(g0), pin(d0)), pin(g1), reps, 5)
        l0 = odo.LaunchCount()
        odo.SetSourceFrame(g0, d0); odo.SetTargetFrame(g1); odo.SetInitialStateVector(np.zeros(6)); odo.Optimize()
        launches = odo.LaunchCount() - l0
        log = odo.IterationStats()
        o, cpu_opt, cpu_all = oracle_alignment(cfg_name, K, g0, d0, g1, 3)
        out[key] = {"what": what, "iterations": len(log), "driver": odo.LastPath(), "reps": reps,
                    "optimize_ms_device": median(opt), "setup_ms_device": median(setup), "host_in_pose_out_ms_wall": median(wall),
                    "host_in_pose_out_ms_wall_p99": float(np.percentile(wall, 99)), "kernel_launches_per_alignment": launches,
                    "h2d_bytes_per_alignment": int(g0.nbytes + g1.nbytes + d0.nbytes),
                    "cpu_oracle": {"optimize_ms": cpu_opt, "setframes_plus_optimize_ms": cpu_all, "cores": 1, "kind": "port"},
                    "iterations_equal_cpu": len(log) == len(o.iter_stats()), "pose_abs_diff_vs_cpu": float(np.max(np.abs(s - o.state()))),
                    "clocks": clocks}
        odo.close()

    # ---- configs[1]: PhotoconsistencyVisualOdometry loop, sequential, per-frame latency
    K = phovo.synth.K_VISUAL_ODOMETRY
    name = "config_5_level_optimization_analytic"
    gray, depth = phovo.synth.render_sequence_torch(frames, ROWS, COLS, K, dev)
    hg = torch.empty(gray.shape, dtype=gray.dtype, pin_memory=True); hg.copy_(gray)
    hd = torch.empty(depth.shape, dtype=torch.float64, pin_memory=True); hd.copy_(depth.to(torch.float64))   # the app's Mat_<double>
    del gray, depth
    torch.cuda.synchronize(dev)
    odo = phovo.CPhotoconsistencyOdometryCuda(device=local_rank)
    odo.SetConfig(phovo.configs.to_config(name, phovo.capi)); odo.SetIntrinsicMatrix(K)
    for rep in range(2):                        # first pass over a short prefix warms up
        n = min(frames, 20) if rep == 0 else frames
        lat, states, iters, opt = [], [], 0, []
        sampler = ClockSampler(local_rank)
        if rep == 1:
            sampler.start()
        odo.SetSourceFrame(hg[0], hd[0])
        for k in range(1, n):
            t0 = time.perf_counter()
            if k > 1:
                odo.PromoteTargetToSource(hd[k - 1])            # VisualOdometry.cpp:222,256-257 without re-uploading the gray image
            odo.SetTargetFrame(hg[k])
            odo.SetInitialStateVector(np.zeros(6))              # :224 (always zero, :175)
            odo.Optimize()                                      # :227-230 is what the app times
            states.append(odo.GetOptimalStateVector())
            lat.append((time.perf_counter() - t0) * 1e3)
            opt.append(odo.Timings()[1])
            iters += len(odo.IterationStats())
        clocks = sampler.stop() if rep == 1 else None
    o = oracle_py.Oracle(oracle_config(phovo, name), K)
    cpu, err, it_equal = [], 0.0, True
    gn, dn = hg.numpy(), hd.numpy()
    for k in range(1, min(frames, 9)):
        t0 = time.perf_counter()
        o.set_source(gn[k - 1], dn[k - 1]); o.set_target(gn[k]); o.set_initial_state(np.zeros(6)); o.optimize()
        cpu.append((time.perf_counter() - t0) * 1e3)
        err = max(err, float(np.max(np.abs(o.state() - states[k - 1]))))
    out["vo_sequence_640x480"] = {"what": "BASELINE configs[1]: PhotoconsistencyVisualOdometry loop, %d synthetic frames, 5-level analytic, sequential on one GPU, target pyramid promoted to source between frames" % frames,
                                  "frames": frames, "ms_per_frame_wall": median(lat), "ms_per_frame_wall_p99": float(np.percentile(lat, 99)),
                                  "optimize_ms_device": median(opt), "frames_per_s": 1e3 / float(np.mean(lat)), "mean_iterations_per_frame": iters / float(len(lat)),
                                  "cpu_oracle": {"ms_per_frame": median(cpu), "cores": 1, "kind": "port", "frames": len(cpu)},
                                  "pose_abs_diff_vs_cpu_first_frames": err, "clocks": clocks}
    odo.close()
    del hg, hd

    # ---- configs[4]: one 7680x4320 pair on ONE GPU (the row-sharded runs are `--workload 8k --gpus N`)
    K = phovo.synth.K_8K
    name = "config_6_level_optimization_analytic"
    g0, d0, g1, _ = phovo.synth.render_batch_torch(1, 4320, 7680, K, dev, seed0=7, chunk=1, xis=phovo.synth.XI_CONFIG1[None])
    hg0 = torch.empty(g0[0].shape, dtype=torch.uint8, pin_memory=True); hg0.copy_(g0[0])
    hg1 = torch.empty(g1[0].shape, dtype=torch.uint8, pin_memory=True); hg1.copy_(g1[0])
    hd0 = torch.empty(d0[0].shape, dtype=torch.float32, pin_memory=True); hd0.copy_(d0[0])
    del g0, d0, g1
    torch.cuda.synchronize(dev)
    odo = phovo.CPhotoconsistencyOdometryCuda(device=local_rank)
    odo.SetConfig(phovo.configs.to_config(name, phovo.capi)); odo.SetIntrinsicMatrix(K)
    s, setup, opt, wall, clocks = timed_alignments(odo, (hg0, hd0), hg1, 10, 2)
    log = odo.IterationStats()
    o, cpu_opt, cpu_all = oracle_alignment(name, K, hg0.numpy(), hd0.numpy().astype(np.float64), hg1.numpy(), 1)
    out["single_pair_7680x4320"] = {"what": "BASELINE configs[4] on one GPU: one 7680x4320 pair, config_6_level_optimization_analytic (f32 depth at the boundary)",
                                    "iterations": len(log), "driver": odo.LastPath(), "reps": 10,
                                    "optimize_ms_device": median(opt), "setup_ms_device": median(setup), "host_in_pose_out_ms_wall": median(wall),
                                    "h2d_bytes_per_alignment": int(hg0.numel() + hg1.numel() + 4 * hd0.numel()),
                                    "cpu_oracle": {"optimize_ms": cpu_opt, "setframes_plus_optimize_ms": cpu_all, "cores": 1, "kind": "port"},
                                    "iterations_equal_cpu": len(log) == len(o.iter_stats()), "pose_abs_diff_vs_cpu": float(np.max(np.abs(s - o.state()))),
                                    "clocks": clocks}
    odo.close()

    # ---- the batch entry for the other two solvers of the apps' METHOD macro (FrameAlignment.cpp:34-44): waves of per-pair
    # slots, one CTA per pair through every level (k_align_slots); device-resident 640x480 pairs, wall clock around the call
    K = phovo.synth.K_FRAME_ALIGNMENT
    P = 1184
    g0, d0, g1, _ = phovo.synth.render_batch_torch(P + 1, ROWS, COLS, K, dev, seed0=11)
    waves = {}
    for key, cfg_name, mode in (("photometric_plus_depth", CONFIG, phovo.MODE_BIOBJECTIVE), ("ceres_mode", "config_5_level_optimization_ceres", None)):
        odo = phovo.CPhotoconsistencyOdometryCuda(device=local_rank)
        odo.SetConfig(phovo.configs.to_config(cfg_name, phovo.capi, mode=mode) if mode is not None else phovo.configs.to_config(cfg_name, phovo.capi))
        odo.SetIntrinsicMatrix(K)
        kw = {"depth1": d0[1:P + 1].contiguous()} if mode is not None else {}
        odo.BatchAlign(g0[:P], d0[:P], g1[:P], **kw)        # slots, arena, pinned result buffers
        torch.cuda.synchronize(dev)
        # (the wave path launches thousands of small set-up kernels from four host threads: a 2 ms NVML polling loop slows it by
        # up to 30 % through the driver's locks -- measured 84 ms steady without, 84-116 ms with -- so this block samples at 20 Hz)
        sampler = ClockSampler(local_rank, period=0.05)
        sampler.start()
        times = []
        for rep in range(3):                                  # median of three calls
            l0 = odo.LaunchCount()
            t0 = time.perf_counter()
            st, it = odo.BatchAlign(g0[:P], d0[:P], g1[:P], **kw)
            times.append(time.perf_counter() - t0)
        dt = median(times)
        waves[key] = {"config": cfg_name, "pairs": P, "pairs_per_s": P / dt, "ms_per_step": 1e3 * dt, "ms_per_step_all": [1e3 * t for t in times],
                      "path": odo.BatchLastPath(), "mean_iterations_per_pair": float(it.sum()) / P, "finite": bool(np.isfinite(st).all()),
                      "gpu_launches": int(odo.LaunchCount() - l0), "clocks": sampler.stop()}
        odo.close()
    out["batch_other_solvers_640x480"] = dict(waves, what="phovo_batch_align for the Ceres-mode and the photometric + depth solver: waves of per-pair slots (path 3), device-resident inputs, poses on the host")
    del g0, d0, g1
    return out


def run_8k(args, phovo, rank, world, local_rank, host_threads):
    """BASELINE configs[4]: ONE synthetic 7680x4320 pair, config_6_level_optimization_analytic, the per-pixel pass of the
    large levels sharded by source rows over the ranks, the 29 sums exchanged every iteration INSIDE the persistent
    kernel over NVLink peer memory (phovo_shard_optimize).  A step is one Optimize(); strong scaling; lower is better.
    Beside it, from the same run: the unsharded Optimize() on one GPU, the equality of the results, and the latency
    of an NCCL all-reduce of the same 32 doubles."""
    import numpy as np
    METRIC_8K = "Optimize() of one 7680x4320 RGB-D pair, 6-level GN, rows sharded over the GPUs"
    name = "config_6_level_optimization_analytic"
    K = phovo.synth.K_8K
    if args.impl == "reference":
        if rank != 0:
            return 0
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import oracle_py
        oracle_py.build()
        g0, d0, g1, _ = phovo.synth.make_pair(4320, 7680, K=K, seed=7)
        o = oracle_py.Oracle(oracle_config(phovo, name), K)
        o.set_source(g0, d0); o.set_target(g1)
        ts = []
        for s_ in range(max(args.warmup, 0) + args.steps):
            o.set_initial_state(np.zeros(6))
            t0 = time.perf_counter(); o.optimize(); t1 = time.perf_counter()
            if s_ >= args.warmup:
                ts.append((t1 - t0) * 1e3)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"state": o.state(),
                                             "iterations_per_level": np.bincount([e["level"] for e in o.iter_stats()], minlength=phovo.MAXL)})
        v = float(np.mean(ts))
        assert "libphovo_b200" not in open("/proc/self/maps").read()
        print(json.dumps({"impl": "reference", "metric": METRIC_8K, "value": v, "unit": "ms", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                          "ms_per_step": v, "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                          "config": {"workload": "one 7680x4320 RGB-D pair, %s (BASELINE configs[4])" % name, "rows": 4320, "cols": 7680},
                          "cpu_baseline": {"value": v, "unit": "ms", "cores": 1, "kind": "port", "sample": "the whole Optimize() of the pair, single thread (the reference is single-threaded)"},
                          "e2e": {"value": v, "unit": "ms", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return 0
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    phovo.build()
    cfg = phovo.configs.to_config(name, phovo.capi)
    stream = torch.cuda.current_stream(dev)
    g0, d0, g1, _ = phovo.synth.render_batch_torch(1, 4320, 7680, K, dev, seed0=7, chunk=1, xis=phovo.synth.XI_CONFIG1[None])
    g0, d0, g1 = g0[0].contiguous(), d0[0].contiguous(), g1[0].contiguous()

    def new_odo():
        odo = phovo.CPhotoconsistencyOdometryCuda(device=local_rank)
        odo.SetConfig(cfg); odo.SetIntrinsicMatrix(K); odo.SetStream(stream.cuda_stream)
        odo.SetSourceFrame(g0, d0); odo.SetTargetFrame(g1)
        return odo

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # the unsharded Optimize() on this GPU: the number sharding has to beat, and the result it has to reproduce
    single = new_odo()
    single_ms = []
    for _ in range(max(args.warmup, 3) + 5):
        single.SetInitialStateVector(np.zeros(6)); single.Optimize()
        single_ms.append(single.Timings()[1])
    s_single, log_single = single.GetOptimalStateVector(), single.IterationStats()
    single_ms = float(np.median(single_ms[-5:]))
    per_level = {}
    for e in log_single:
        per_level[e["level"]] = per_level.get(e["level"], 0) + 1

    odo = new_odo()
    ra = phovo.sharded.RowShardedAlignment(odo, rank, world, local_rank, exchange="peer")
    for _ in range(max(args.warmup, 3)):
        barrier()
        st, executed = ra.optimize_fused(min_shard_pixels=args.min_shard_pixels)
    sampler = ClockSampler(local_rank)
    sampler.start()
    dev_ms, wall_ms = [], []
    barrier()
    t_all0 = time.perf_counter()
    for _ in range(args.steps):
        barrier()                       # the ranks enter a step together: a rank waiting for a late peer is not what is measured
        t0 = time.perf_counter()
        st, executed = ra.optimize_fused(min_shard_pixels=args.min_shard_pixels)
        wall_ms.append((time.perf_counter() - t0) * 1e3)
        dev_ms.append(odo.Timings()[1])        # CUDA events around this rank's launches of the step
    barrier()
    t_all = time.perf_counter() - t_all0
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"state": st, "iterations_per_level": [executed.get(l, 0) for l in range(phovo.MAXL)]})
    t = torch.tensor([float(np.mean(dev_ms)), float(np.mean(wall_ms))], dtype=torch.float64, device=dev)
    mine = torch.tensor(st, dtype=torch.float64, device=dev)
    gathered = torch.zeros((world, 6), dtype=torch.float64, device=dev)
    nccl_us = None
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_gather_into_tensor(gathered, mine)
        buf = torch.zeros(32, dtype=torch.float64, device=dev)
        for _ in range(20):
            dist.all_reduce(buf)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier(); e0.record(stream)
        for _ in range(200):
            dist.all_reduce(buf)
        e1.record(stream); barrier()
        nccl_us = e0.elapsed_time(e1) / 200 * 1e3
    else:
        gathered[0] = mine
    value, wall = float(t[0].item()), float(t[1].item())
    iters = sum(executed.values())
    sharded_levels = [l for l in range(cfg.num_levels) if cfg.max_num_iterations[l] > 0 and world > 1 and
                      int(round(4320 * 0.5 ** l)) * int(round(7680 * 0.5 ** l)) >= args.min_shard_pixels]
    if rank == 0:
        line = {"metric": METRIC_8K, "value": value, "unit": "ms", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": value, "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": "one 7680x4320 RGB-D pair, %s (BASELINE configs[4])" % name, "rows": 4320, "cols": 7680,
                           "parallelism": "source rows of the levels with >= %d px sharded x%d, 29 sums exchanged per iteration inside the persistent kernel over NVLink peer memory; smaller levels replicated" % (args.min_shard_pixels, world),
                           "l2_policy": "frames resident in HBM (set once); the active levels (55 MB of fp64 images) are re-read every iteration"},
                "timing": "value = device time of one Optimize() (CUDA events around the rank's launches), mean over the steps, max over ranks; the ranks enter every step through a barrier",
                "wall_ms_per_step": wall, "timed_region_wall_s": t_all,
                "iterations": iters, "iterations_per_level": {str(k): v for k, v in sorted(executed.items())}, "sharded_levels": sharded_levels,
                "single_gpu": {"optimize_ms_device": single_ms, "iterations_per_level": {str(k): v for k, v in sorted(per_level.items())}},
                "speedup_vs_single_gpu": single_ms / value,
                "max_abs_state_diff_vs_single_gpu": float(np.max(np.abs(st - s_single))), "iterations_equal_single_gpu": executed == per_level,
                "ranks_bitwise_identical": bool((gathered == gathered[0]).all().item()),
                "nccl_allreduce_32_doubles_us": nccl_us,
                "e2e": {"value": wall, "unit": "ms", "h2d_bytes_per_step": 48, "d2h_bytes_per_step": 48 + 256 + 352 * iters,
                        "note": "the call a user makes (SetInitialStateVector + ShardOptimize + GetOptimalStateVector) timed on the host; the frames are set once and stay resident, per step the initial state (48 B) goes up and the device pose block (256 B) + one 352-byte log entry per executed iteration come back"},
                "gpu_launches": int(len(executed) + 1), "clocks": clocks}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--pairs", type=int, default=4096, help="pairs per GPU per step")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="batch", choices=["batch", "8k"],
                    help="batch: BASELINE configs[3] (the headline, default); 8k: BASELINE configs[4], ONE 7680x4320 pair whose rows are sharded over the --gpus ranks")
    ap.add_argument("--min-shard-pixels", type=int, default=262144, help="8k workload: levels with fewer pixels run unsharded on every rank")
    ap.add_argument("--cpu-pairs", type=int, default=0, help="pairs in the bounded CPU sample (0: 2 per host thread, >= 64)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the per-pair measurements of BASELINE configs[0], [1], [2], [4]")
    ap.add_argument("--secondary-frames", type=int, default=1000, help="frames of the synthetic VO sequence (BASELINE configs[1])")
    ap.add_argument("--depth", default="u16", choices=["u16", "f32"],
                    help="depth format at the boundary: raw u16 sensor units x 1/5000 m (what the reference apps read, default) or f32 metres")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (poses and iteration counts) as DIR/<name>.npy (rank 0); "
                         "with --impl reference the number of pairs is --cpu-pairs, which defaults to one depending on the host's core count")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    phovo = importlib.import_module(PKG)
    import numpy as np
    K = phovo.synth.K_FRAME_ALIGNMENT
    host_threads = os.cpu_count() or 1

    if args.workload == "8k":
        return run_8k(args, phovo, rank, world, local_rank, host_threads)
    if args.impl == "reference":
        if rank != 0:
            return 0
        pairs = args.cpu_pairs or max(64, 2 * host_threads)
        r = cpu_reference(phovo, K, pairs, host_threads, args.steps, max(args.warmup, 1), depth=args.depth)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"states": r["states"], "iterations": r["iters"]})
        line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": "pairs/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": workload_config(args.pairs, args.depth, args.gpus),
                "mean_iterations_per_pair": r["mean_iterations_per_pair"],
                "cpu_baseline": {"value": r["value"], "unit": "pairs/s", "cores": host_threads, "kind": "port",
                                 "sample": "each step aligns a bounded sample of %d pairs of the workload (32 distinct, %d threads x single-threaded alignments: SetSourceFrame + SetTargetFrame + Optimize), faithful cost structure (materialised Nx6 Jacobian, per-pass setZero); oracle/_ref (the reference's own loop over stand-in Eigen products) is 2-3x slower than this port" % (pairs, host_threads)},
                "e2e": {"value": r["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        # this arm is the CPU implementation alone: the CUDA library must not even be mapped
        assert "libphovo_b200" not in open("/proc/self/maps").read(), "the reference arm loaded the product library"
        print(json.dumps(line))
        return 0

    import torch
    import torch.distributed as dist
    numa = bind_to_gpu_numa_node(local_rank)       # before any pinned allocation (first touch decides the node)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL prints its version banner (NCCL_DEBUG=VERSION/INFO) to stdout by default; stdout carries the JSON line only
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    phovo.build()
    P = args.pairs
    cfg = phovo.configs.to_config(CONFIG, phovo.capi)
    odo = phovo.CPhotoconsistencyOdometryCuda(device=local_rank)
    odo.SetConfig(cfg)
    odo.SetIntrinsicMatrix(K)
    stream = torch.cuda.current_stream(dev)
    odo.SetStream(stream.cuda_stream)

    # ---- synthetic inputs (not timed): P pairs per rank, generated on the GPU, then mirrored to pinned host memory
    g0, d0, g1, xis = phovo.synth.render_batch_torch(P, ROWS, COLS, K, dev, seed0=rank * P)
    depth_scale = 1.0
    if args.depth == "u16":
        # raw sensor units (values < 32768: the int16 tensor carries the same bits as u16)
        d0 = torch.clamp(torch.round(d0.to(torch.float64) * 5000.), 0, 32767).to(torch.int16)
        depth_scale = DEPTH_SCALE
    states = torch.zeros((P, 6), dtype=torch.float64, device=dev)
    iters = torch.zeros((P, phovo.MAXL), dtype=torch.int32, device=dev)
    gathered = torch.zeros((world * P, 6), dtype=torch.float64, device=dev) if world > 1 else None
    torch.cuda.synchronize(dev)

    def step():
        odo.BatchAlignDevice(g0, d0, g1, states, iters, depth_scale=depth_scale)
        if world > 1:
            dist.all_gather_into_tensor(gathered, states)     # the final pose gather

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(args.warmup):
        step()
    barrier()
    launches0 = odo.LaunchCount()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pyr_ms, align_ms = [], []
    barrier()
    ev0.record(stream)
    for _ in range(args.steps):
        step()
    ev1.record(stream)
    barrier()
    clocks = sampler.stop()
    elapsed_ms = ev0.elapsed_time(ev1)
    if args.dump_outputs:
        iters_all = iters
        if world > 1:
            iters_all = torch.zeros((world * P, phovo.MAXL), dtype=torch.int32, device=dev)
            dist.all_gather_into_tensor(iters_all, iters)
        if rank == 0:
            dump_outputs(args.dump_outputs, {"states": (gathered if world > 1 else states).cpu().numpy(),
                                             "iterations": iters_all.cpu().numpy()})
    launches = odo.LaunchCount() - launches0
    # per-kernel CUDA-event times (recorded inside the library on the same stream), one more step
    for _ in range(3):
        odo.BatchAlignDevice(g0, d0, g1, states, iters, depth_scale=depth_scale)
        a, b = odo.BatchKernelTimes()
        pyr_ms.append(a); align_ms.append(b)
    t = torch.tensor([elapsed_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms = float(t.item())
    value = world * P * args.steps / (elapsed_ms * 1e-3)
    it_host = iters.cpu().numpy()
    st_host = states.cpu().numpy()

    # ---- end to end through the C ABI with HOST buffers (pinned): H2D of every input + D2H of the poses in the timed region
    hg0 = torch.empty(g0.shape, dtype=g0.dtype, pin_memory=True); hg0.copy_(g0)
    hd0 = torch.empty(d0.shape, dtype=d0.dtype, pin_memory=True); hd0.copy_(d0)
    hg1 = torch.empty(g1.shape, dtype=g1.dtype, pin_memory=True); hg1.copy_(g1)
    torch.cuda.synchronize(dev)
    for _ in range(2):
        st_e2e, it_e2e = odo.BatchAlign(hg0, hd0, hg1, depth_scale=depth_scale)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record(stream)
    e2e_steps = max(2, min(args.steps, 5))
    for _ in range(e2e_steps):
        st_e2e, it_e2e = odo.BatchAlign(hg0, hd0, hg1, depth_scale=depth_scale)
    e1.record(stream)
    barrier()
    wall_e2e = time.perf_counter() - t0
    e2e_ms = max(e0.elapsed_time(e1), 0.0)
    te = torch.tensor([max(e2e_ms, wall_e2e * 1e3)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * P * e2e_steps / (float(te.item()) * 1e-3)
    assert np.array_equal(st_e2e, st_host), "host-buffer path and device-resident path disagree"
    h2d_full = P * (2 * ROWS * COLS + ROWS * COLS * d0.element_size())
    h2d = odo.BatchLastH2DBytes()          # counted by the library from the copies it issued
    d2h = P * (6 * 8 + phovo.MAXL * 4)
    del hg0, hd0, hg1
    # the ceiling `e2e` can be held against, measured in this run: one big copy from pinned memory per rank,
    # (a) one rank at a time with the other links idle, (b) all ranks at once (what the e2e steps do)
    h2d_solo = 0.0
    for r in range(world):
        barrier()
        if r == rank:
            h2d_solo = pinned_h2d_peak(torch, dev, stream, reps=3)
    barrier()
    h2d_peak = pinned_h2d_peak(torch, dev, stream)
    tp = torch.tensor([h2d_peak, h2d_solo], dtype=torch.float64, device=dev)
    if world > 1:
        gathered_peaks = [torch.zeros_like(tp) for _ in range(world)]
        dist.all_gather(gathered_peaks, tp)
        h2d_peaks = [float(x[0].item()) for x in gathered_peaks]
        h2d_solos = [float(x[1].item()) for x in gathered_peaks]
    else:
        h2d_peaks, h2d_solos = [h2d_peak], [h2d_solo]

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- roofline of the dominant kernel
    peak, peak_src = hbm_peak()
    iter_bytes, setup_bytes = algorithmic_bytes(cfg, it_host, ROWS, COLS, d0.element_size())
    align_t = float(np.mean(align_ms)) * 1e-3
    pyr_t = float(np.mean(pyr_ms)) * 1e-3
    achieved = iter_bytes / align_t / 1e9
    px_iters = 0.0
    for lvl in range(cfg.num_levels):
        if cfg.max_num_iterations[lvl] > 0:
            px_iters += float(it_host[:, lvl].sum()) * int(round(ROWS * 0.5 ** lvl)) * int(round(COLS * 0.5 ** lvl))
    prof = {}
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "roofline_inputs.json")))
    except Exception:
        pass
    fp64 = None
    if prof.get("fp64_thread_inst_per_px_iter"):
        rate = px_iters * prof["fp64_thread_inst_per_px_iter"] / align_t
        fp64 = {"achieved": rate / 1e12, "peak": prof["fp64_peak_thread_inst_per_s"] / 1e12, "unit": "T fp64 thread-instructions/s",
                "frac": rate / prof["fp64_peak_thread_inst_per_s"], "inst_per_px_iter": prof["fp64_thread_inst_per_px_iter"],
                "source": "ncu op counters of %s / executed pixel-iterations; peak = %s" % (prof.get("tag"), prof.get("fp64_peak_source"))}
    issue = None
    if prof.get("issue_cycles_floor_per_32_px_iter") and clocks.get("sm_mhz"):
        sms = torch.cuda.get_device_properties(dev).multi_processor_count
        cyc = align_t * clocks["sm_mhz"] * 1e6 * 4 * sms / (px_iters / 32.0)      # scheduler cycles per 32 pixel-iterations (one warp's worth)
        issue = {"achieved_cycles_per_32_px_iter": cyc, "floor_cycles_per_32_px_iter": prof["issue_cycles_floor_per_32_px_iter"],
                 "frac": prof["issue_cycles_floor_per_32_px_iter"] / cyc,
                 "warp_inst_per_32_px_iter": prof["warp_inst_per_32_px_iter"], "fp64_warp_inst_per_32_px_iter": prof["fp64_warp_inst_per_32_px_iter"],
                 "source": "instruction counts from ncu (%s); an FP64-pipe instruction costs two issue cycles, nothing issues in its shadow (tools/issue_probe.cu, profiles/r02_issue_probe.jsonl): floor = all warp instructions + the fp64 ones once more" % prof.get("tag")}
    roofline = {"bound": "fp64", "kernel": "k_batch_level (one launch per active pyramid level; figures are the sum over the level launches)", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak,
                "traffic": (prof["dram_bytes_per_pair"] * P) if prof.get("dram_bytes_per_pair") else None,
                "traffic_source": "ncu --set full dram__bytes_read+write of one launch (%s, %d pairs) scaled by pairs" % (prof.get("tag"), prof.get("profiled_pairs", 0)) if prof else None,
                "peak_source": peak_src,
                "algorithmic_bytes_per_launch": iter_bytes, "kernel_ms": align_t * 1e3,
                "share_of_step": align_t / (align_t + pyr_t),
                "pixel_iterations_per_launch": px_iters,
                "ncu_dram_gbs": prof.get("dram_gbs"), "ncu_l2_gbs": prof.get("l2_gbs"),       # achieved DRAM / L2 bandwidth of the level kernels under ncu (north star: both beside the HBM peak)
                "note": "achieved / peak / frac are the contract's HBM figure: algorithmic bytes = SURVEY 8(d), 20 B per pixel per executed GN iteration + 216 B of sums, over the measured HBM copy bandwidth. The level is resident in shared memory, so DRAM traffic is the packed record read once (traffic) and the unit that binds the kernel is the FP64 pipe together with the issue slots it blocks: see fp64 (thread-instructions per pixel-iteration from ncu x executed pixel-iterations / kernel time, over the measured DFMA peak) and issue (issue cycles the kernel's instruction counts need at the least / scheduler cycles it takes)",
                "fp64": fp64, "issue": issue,
                "other_kernels": {"k_batch_pyramid": {"kernel_ms": pyr_t * 1e3, "algorithmic_bytes_per_launch": setup_bytes,
                                                      "achieved": setup_bytes / pyr_t / 1e9, "frac": setup_bytes / pyr_t / 1e9 / peak,
                                                      "bound": "hbm", "traffic": (prof["pyramid_dram_bytes_per_pair"] * P) if prof.get("pyramid_dram_bytes_per_pair") else None,
                                                      "note": "compulsory traffic: the source rows the active levels tap (%.0f%% of the rows) of gray0, gray1 and depth0 (%d B/px) in whole sectors + the 12 B/px packed record out" % (100 * rows_read_fraction(cfg, ROWS), d0.element_size())}}}
    # ---- CPU baseline on this box's host cores, bounded sample of the same workload
    cpu = None
    if not args.no_cpu_baseline:
        pairs = args.cpu_pairs or max(64, 2 * host_threads)
        r = cpu_reference(phovo, K, pairs, host_threads, 1, 0, depth=args.depth)
        # same inputs through the GPU: iteration counts and poses must agree with the CPU port
        cg0, cd0, cg1 = r["inputs"]
        if args.depth == "u16":
            st_chk, it_chk = odo.BatchAlign(cg0, r["raw_depth"], cg1, depth_scale=DEPTH_SCALE)
        else:
            st_chk, it_chk = odo.BatchAlign(cg0, cd0.astype(np.float32), cg1)
        iters_equal = bool(np.array_equal(it_chk, r["iters"]))
        pose_err = float(np.max(np.abs(st_chk - r["states"])))
        cpu = {"value": r["value"], "unit": "pairs/s", "cores": host_threads, "kind": "port",
               "sample": "%d pairs, %d threads x single-threaded alignments (SetSourceFrame+SetTargetFrame+Optimize)" % (pairs, host_threads),
               "optimize_only_pairs_per_core_s": r["optimize_only_pairs_per_core_s"],
               "gpu_vs_cpu_iterations_equal": iters_equal, "gpu_vs_cpu_max_pose_abs_diff": pose_err}
    sec = None
    if world == 1 and not args.no_secondary:
        del g0, d0, g1
        torch.cuda.empty_cache()
        sec = secondary_block(phovo, torch, dev, local_rank, args.secondary_frames)
    e2e_step_s = float(te.item()) / e2e_steps * 1e-3
    line = {"metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": workload_config(P, args.depth, world),
            "mean_iterations_per_pair": {str(l): float(it_host[:, l].mean()) for l in range(cfg.num_levels) if cfg.max_num_iterations[l] > 0},
            "e2e": {"value": e2e_value, "unit": "pairs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_step_s * 1e3, "steps": e2e_steps,
                    "link_gbs": h2d / e2e_step_s / 1e9, "h2d_peak_gbs": min(h2d_peaks), "h2d_peak_gbs_per_rank": h2d_peaks,
                    "h2d_peak_gbs_per_rank_alone": h2d_solos, "h2d_aggregate_gbs": h2d * world / e2e_step_s / 1e9,
                    "h2d_aggregate_peak_gbs": sum(h2d_peaks),
                    "link_frac_of_h2d_peak": h2d / e2e_step_s / 1e9 / min(h2d_peaks),
                    "host_cpus_bound_to_gpu_numa_node": numa,
                    "upload": "rows no active level reads are not uploaded: %d of %d input bytes cross PCIe per rank; link_gbs = per-rank H2D bytes / e2e step time (all ranks upload at once), h2d_peak_gbs = one 1 GiB cudaMemcpyAsync from pinned memory per rank, all ranks copying at once (slowest rank; per rank in h2d_peak_gbs_per_rank), h2d_peak_gbs_per_rank_alone = the same copy with the other ranks idle: the gap between the two is the host fabric (PCIe root complexes / memory), not this library" % (h2d, h2d_full)},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
            "latency_us_per_pair_per_sm": align_t / (P / min(P, 148)) * 1e6, "secondary": sec}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
