"""Per-stage timing of the fused path for one configuration; prints one line.
Usage: python profiles/tune_stage.py [variant] [frames] [--empty] [--memset]"""
import ctypes
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import lidar_vision_vqa_b200 as L  # noqa: E402
from lidar_vision_vqa_b200 import _native, ops, synth  # noqa: E402
from oracle import pillar_oracle as po  # noqa: E402

variant = sys.argv[1] if len(sys.argv) > 1 else "auto"
nb = int(sys.argv[2]) if len(sys.argv) > 2 else 16
dev = torch.device("cuda:0")
model, gc, _ = synth.WORKLOADS["cfg2_nuscenes32_b16_pillar0.2_bev512"]
grid = L.GridSpec.from_range(gc.point_cloud_range, gc.voxel_size, 32, 30000)
pts, offs = synth.make_batch(nb, model, 5)
if "--empty" in sys.argv:
    pts = pts + 1000.0  # nothing in range: every tile of the canvas is empty
sd = po.random_pfn_params(11, [64], True, seed=0)
pfn = ops.fold_pfn(sd["pfn_layers.0.linear.weight"], (sd["pfn_layers.0.norm.weight"], sd["pfn_layers.0.norm.bias"],
                   sd["pfn_layers.0.norm.running_mean"], sd["pfn_layers.0.norm.running_var"], 1e-3), None, c_point=5,
                   use_absolute_xyz=True, with_distance=False, voxel_size=grid.voxel_size,
                   point_cloud_range=grid.point_cloud_range, device=dev)
p, o = torch.from_numpy(pts).to(dev), torch.from_numpy(offs).to(dev)
bufs = ops.EncodeBuffers(len(pts), nb, grid, 64, dev)
if "--tightcap" in sys.argv:  # size the per-pillar outputs by the pillar count actually seen (+5 %)
    r0 = ops.encode_bev(p, o, grid, pfn, buffers=bufs, scatter_variant=variant)
    m0 = int(r0["pillar_count"][-1].item())
    bufs = ops.EncodeBuffers(len(pts), nb, grid, 64, dev, capacity=int(m0 * 1.05) + 16)
lib = _native.load()
K = 30
evs = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(K)]
for e4 in evs:
    for e in e4:
        e.record()
torch.cuda.synchronize()
arrs = [(ctypes.c_void_p * 4)(*[e.cuda_event for e in e4]) for e4 in evs]
for _ in range(5):
    ops.encode_bev(p, o, grid, pfn, buffers=bufs, scatter_variant=variant)
torch.cuda.synchronize()
for k in range(K):
    lib.pillars_set_stage_events(arrs[k])
    ops.encode_bev(p, o, grid, pfn, buffers=bufs, scatter_variant=variant)
lib.pillars_set_stage_events(None)
torch.cuda.synchronize()
st = np.array([[e4[i].elapsed_time(e4[i + 1]) for i in range(3)] for e4 in evs]) * 1e3
med = np.median(st, axis=0)
extra = ""
if "--memset" in sys.argv:
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t = []
    for _ in range(10):
        s.record(); bufs.bev.zero_(); e.record(); torch.cuda.synchronize(); t.append(s.elapsed_time(e) * 1e3)
    src = torch.empty_like(bufs.bev)
    t2 = []
    for _ in range(10):
        s.record(); bufs.bev.copy_(src); e.record(); torch.cuda.synchronize(); t2.append(s.elapsed_time(e) * 1e3)
    gb = bufs.bev.numel() * 4 / 1e9
    extra = f" | memset {min(t):.1f}us = {gb / min(t) * 1e6:.0f} GB/s | copy {min(t2):.1f}us = {2 * gb / min(t2) * 1e6:.0f} GB/s"
gbs = bufs.bev.numel() * 4 / (med[2] * 1e-6) / 1e9
print(f"{variant:7s} nb={nb} group={med[0]:.1f}us feat={med[1]:.1f}us scatter={med[2]:.1f}us ({gbs:.0f} GB/s write){extra}", flush=True)
