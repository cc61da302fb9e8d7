#!/usr/bin/env python
"""Device time per kernel (torch.profiler, CUDA activities) of one phovo_batch_warp_image call on the inputs of
tools/bench_batch_warp.py: 4096 device-resident 640x480 pairs, u16 depth; summary only, then with both images.
Mean of three calls, ms.  A run of its own: the profiler slows the host.  (profiles/r03_batch_warp_kernels.txt)"""
import importlib, sys, os, json
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
phovo = importlib.import_module("photoconsistency-visual-odometry_b200"); phovo.build()
dev = torch.device("cuda", 0); K = phovo.synth.K_FRAME_ALIGNMENT; P = 4096
g0, d32, g1, _ = phovo.synth.render_batch_torch(P, 480, 640, K, dev, seed0=2024)
raw = torch.clamp(torch.round(d32.double() * 5000.), 0, 65535).to(torch.int32)
d0 = torch.where(raw > 32767, raw - 65536, raw).to(torch.int16); del raw, d32
rng = np.random.default_rng(2024)
st = np.concatenate([rng.uniform(-0.05, 0.05, (P, 3)), rng.uniform(-0.03, 0.03, (P, 3))], axis=1)
rts = torch.from_numpy(np.stack([phovo.state_to_rt(s) for s in st])).to(dev)
odo = phovo.CPhotoconsistencyOdometryCuda(); odo.SetStream(torch.cuda.current_stream().cuda_stream)
for images in (False, True):
    odo.BatchWarpImage(g0, d0, rts, K, gray1=g1, images=images, depth_scale=1/5000.)
    torch.cuda.synchronize()
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            odo.BatchWarpImage(g0, d0, rts, K, gray1=g1, images=images, depth_scale=1/5000.)
        torch.cuda.synchronize()
    agg = {}
    for e in prof.events():
        if e.device_type.name == "CUDA":
            k = e.name[:60]; agg[k] = agg.get(k, 0) + e.device_time_total / 3 / 1e3
    print("images" if images else "summary", json.dumps({k: round(v, 3) for k, v in sorted(agg.items(), key=lambda x: -x[1])[:6]}))
