"""Scatter stage on a reused canvas (EncodeBuffers' occupancy bitmaps), timed with the library's stage events.
Regimes, one EncodeBuffers each: `empty` (an empty batch on a canvas whose bitmap is all clear: nothing is stored, the
stage is one pass over the index map and the bitmaps), `same` (one batch, re-encoded), `cycle5` (5 batches cycling through
the buffers) and `invalidated` (invalidate_canvas() before every call: the whole canvas is written, as without bitmaps).  Reports the 32-byte
canvas sectors written (popcount of prev | next times the channels), the bytes that makes, the minimum traffic of the stage
(those writes + the index map + the feature rows) and its rate against MEASURED_PEAKS.json.
Usage: python profiles/scripts/scatter_reuse.py [out.json]   (B200; cfg2 and cfg4, fp32 canvas)"""
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import lidar_vision_vqa_b200 as L  # noqa: E402
from lidar_vision_vqa_b200 import _native, ops, synth  # noqa: E402
from oracle import pillar_oracle as po  # noqa: E402

WORKLOADS = ("cfg2_nuscenes32_b16_pillar0.2_bev512", "cfg4_waymo64_pillar0.1_bev1024")
F, CALLS = 64, 25


def peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        return float(json.load(open(path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (copy, read + write)"
    return 6650.0, "fallback 6.65 TB/s"


def popcount(t):
    b = t.contiguous().view(torch.uint8).cpu().numpy()
    return int(np.unpackbits(b).sum())


def run(name, dev, lib, peak):
    model, gc, nb = synth.WORKLOADS[name]
    grid = L.GridSpec.from_range(gc.point_cloud_range, gc.voxel_size, gc.max_points_per_voxel, gc.max_voxels)
    nx, ny, _ = grid.grid_size
    sd = po.random_pfn_params(11, [F], True, seed=0)
    pfn = ops.fold_pfn(sd["pfn_layers.0.linear.weight"], (sd["pfn_layers.0.norm.weight"], sd["pfn_layers.0.norm.bias"],
                       sd["pfn_layers.0.norm.running_mean"], sd["pfn_layers.0.norm.running_var"], 1e-3), None,
                       c_point=5, use_absolute_xyz=True, with_distance=False, voxel_size=grid.voxel_size,
                       point_cloud_range=grid.point_cloud_range, device=dev)
    batches = []
    for r in range(5):  # the batches bench.py builds (seed0 = r * nb)
        pts, offs = synth.make_batch(nb, model, 5, seed0=r * nb)
        batches.append((torch.from_numpy(pts).to(dev), torch.from_numpy(offs).to(dev)))
    n_max = max(p.shape[0] for p, _ in batches)
    batches.append((torch.zeros((0, 5), dtype=torch.float32, device=dev), torch.zeros(nb + 1, dtype=torch.int32, device=dev)))
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(CALLS)]
    for e4 in evs:  # torch only reports times of events it recorded itself once
        for e in e4:
            e.record()
    torch.cuda.synchronize()
    arrs = [(ctypes.c_void_p * 4)(*[e.cuda_event for e in e4]) for e4 in evs]
    sectors_total = nb * ((nx * ny + 255) // 256) * 32
    out = {"grid": [nx, ny], "frames": nb, "canvas_bytes": 4 * F * nx * ny * nb}
    for regime, pick in (("empty", lambda k: 5), ("same", lambda k: 0), ("cycle5", lambda k: k % 5),
                         ("invalidated", lambda k: k % 5)):
        bufs = ops.EncodeBuffers(n_max, nb, grid, F, dev)
        for k in range(6):
            ops.encode_bev(*batches[pick(k)], grid, pfn, buffers=bufs)
        torch.cuda.synchronize()
        ms, sec, rows = [], [], []
        for k in range(CALLS):
            if regime == "invalidated":
                bufs.invalidate_canvas()
            lib.pillars_set_stage_events(arrs[k])
            res = ops.encode_bev(*batches[pick(k)], grid, pfn, buffers=bufs)
            lib.pillars_set_stage_events(None)
            torch.cuda.synchronize()
            ms.append(evs[k][2].elapsed_time(evs[k][3]))
            sec.append(sectors_total if regime == "invalidated" else popcount(bufs._occupancy[0] | bufs._occupancy[1]))
            rows.append(int(res["pillar_count"][-1].item()))
        t = float(np.median(ms))
        written = float(np.mean(sec)) * F * 32
        traffic = written + 4 * nx * ny * nb + 4 * F * float(np.mean(rows)) + 8 * nb * ((nx * ny + 255) // 256)
        out[regime] = {"scatter_ms_median": t, "scatter_ms_min": float(np.min(ms)), "scatter_ms_max": float(np.max(ms)),
                       "sectors_written_frac": float(np.mean(sec)) / sectors_total, "bytes_written": written,
                       "min_traffic_bytes": traffic, "written_gbs": written / (t * 1e-3) / 1e9,
                       "traffic_gbs": traffic / (t * 1e-3) / 1e9, "traffic_frac_of_peak": traffic / (t * 1e-3) / 1e9 / peak}
    return out


def main():
    dev = torch.device("cuda:0")
    lib = _native.load()
    peak, src = peak_gbs()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    res = {"gpu": smi, "peak_gbs": peak, "peak_source": src, "calls_per_regime": CALLS,
           "timing": "scatter stage between the library's stage events [2] and [3], one stream, synchronised per call",
           "traffic": "bytes written (sectors of prev | next x 64 channels x 32 B) + index map (4 B per cell) + feature "
                      "rows (256 B per pillar) + both bitmaps"}
    for name in WORKLOADS:
        res[name] = run(name, dev, lib, peak)
    text = json.dumps(res, indent=1)
    print(text)
    if len(sys.argv) > 1:
        os.makedirs(os.path.dirname(os.path.abspath(sys.argv[1])), exist_ok=True)
        open(sys.argv[1], "w").write(text + "\n")


if __name__ == "__main__":
    main()
