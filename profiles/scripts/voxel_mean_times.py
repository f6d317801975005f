"""Points -> MeanVFE voxel_features on VoxelNeXt's nuScenes grid (1440 x 1440 x 40, P = 10, 160 000 voxels per frame):
ms per batch for

  fused     ops.voxelize_mean (pillars_voxelize_mean: grouping + k_voxel_mean, no padded voxels), on the B200;
  padded    ops.voxelize with padded voxels [M, 10, C] (pillars_voxelize), then the reference's three torch lines on the
            B200 (mean_vfe.py:25-29);
  cpu       the C voxeliser (oracle/voxelize_ref.c) on one CPU thread, frame after frame, plus torch-CPU MeanVFE on one
            thread: what the product's data loader does with spconv's CPU voxeliser and one worker;

for 16 single nuScenes-like sweeps (C = 4, the product's input) and 8 ten-sweep clouds (C = 5).  GPU times are CUDA
events around one call, median of --calls after --warmup; the CPU time is the median of --cpu-calls host-clock runs.  The
points are on the device before the GPU timings start (the H2D copy is not counted on either GPU path).  A second pass
with the library's stage events splits the fused call into grouping and k_voxel_mean (the events break the PDL overlap,
so the two parts add up to a little more than the fused time).  `fill_ms` is a standalone 0xFF fill of the B * nx * ny
int32 index map that the hash grouping otherwise writes and pillars_voxelize_mean skips.  Writes one JSON file (--out).

    python profiles/scripts/voxel_mean_times.py --out out/r06_voxel_mean.json
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _gpu_ms(torch, fn, warmup, calls):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(calls):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return statistics.median(times), times


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--calls", type=int, default=30)
    ap.add_argument("--cpu-calls", type=int, default=3)
    args = ap.parse_args()

    import ctypes

    import numpy as np
    import torch

    import lidar_vision_vqa_b200 as L
    from lidar_vision_vqa_b200 import _native, ops, synth
    from mean_vfe_ref import mean_vfe, mean_vfe_sequential
    from oracle import pillar_oracle as po

    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    gc = synth.VOXELNEXT_NUSCENES
    grid = L.GridSpec(gc.point_cloud_range, gc.voxel_size, gc.grid_size, gc.max_points_per_voxel, gc.max_voxels)
    nx, ny, _ = gc.grid_size
    lib = _native.load()
    result = {"gpu": smi, "grid": list(gc.grid_size), "max_points": gc.max_points_per_voxel, "max_voxels": gc.max_voxels,
              "torch_threads_cpu_leg": 1, "workloads": {}}
    for name, model, nb, c in (("b16_single_c4", synth.NUSCENES_32, 16, 4), ("b8_10sweep_c5", synth.NUSCENES_10SWEEP, 8, 5)):
        pts, offs = synth.make_batch(nb, model, c, seed0=1000)
        p_d, o_d = torch.from_numpy(pts).to(dev), torch.from_numpy(offs).to(dev)
        res = ops.voxelize_mean(p_d, o_d, grid)
        torch.cuda.synchronize()
        m = int(res["pillar_count"][-1].item())
        fused_ms, fused_all = _gpu_ms(torch, lambda: ops.voxelize_mean(p_d, o_d, grid), args.warmup, args.calls)

        def padded():
            r = ops.voxelize(p_d, o_d, grid, want_voxels=True)
            return mean_vfe(r["voxels"][:m], r["voxel_num_points"][:m])

        padded_ms, _ = _gpu_ms(torch, padded, args.warmup, args.calls)
        fused = ops.voxelize_mean(p_d, o_d, grid)["voxel_features"][:m]
        via_padded = padded()
        r = ops.voxelize(p_d, o_d, grid, want_voxels=True)
        seq = mean_vfe_sequential(r["voxels"][:m].cpu().numpy(), r["voxel_num_points"][:m].cpu().numpy())
        bit_exact_vs_sequential = bool(np.array_equal(fused.cpu().numpy().view(np.uint32), seq.view(np.uint32)))
        rel = ((fused - via_padded).abs() / via_padded.abs().clamp_min(1e-30)).max().item()

        # grouping | k_voxel_mean split through the stage events
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        for e in ev:  # torch times only events it has recorded itself once
            e.record()
        arr = (ctypes.c_void_p * 4)(*[e.cuda_event for e in ev])
        lib.pillars_set_stage_events(arr)
        split = []
        for i in range(args.warmup + args.calls):
            ops.voxelize_mean(p_d, o_d, grid)
            ev[3].synchronize()
            if i >= args.warmup:
                split.append((ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2])))
        lib.pillars_set_stage_events(None)
        fill_ms, _ = _gpu_ms(torch, lambda: torch.full((nb, ny, nx), -1, dtype=torch.int32, device=dev), args.warmup,
                             args.calls)

        # the data loader's way: one CPU thread, frame after frame
        torch.set_num_threads(1)
        cpu = []
        for _ in range(args.cpu_calls):
            t0 = time.perf_counter()
            for b in range(nb):
                v = po.voxelize_hard(pts[offs[b]:offs[b + 1]], gc.point_cloud_range, gc.voxel_size,
                                     gc.max_points_per_voxel, gc.max_voxels)
                mean_vfe(torch.from_numpy(v["voxels"]), torch.from_numpy(v["num_points"]))
            cpu.append((time.perf_counter() - t0) * 1e3)
        result["workloads"][name] = {
            "frames": nb, "c_point": c, "points": int(len(pts)), "voxels": m,
            "voxels_at_p": int((r["voxel_num_points"][:m] == gc.max_points_per_voxel).sum().item()),
            "fused_ms": fused_ms, "fused_ms_min_max": [min(fused_all), max(fused_all)],
            "fused_grouping_ms": statistics.median(s[0] for s in split),
            "fused_voxel_mean_kernel_ms": statistics.median(s[1] for s in split),
            "padded_plus_torch_ms": padded_ms,
            "cpu_one_thread_ms": statistics.median(cpu),
            "index_map_fill_ms": fill_ms, "index_map_bytes": 4 * nb * nx * ny,
            "fused_bit_exact_vs_sequential_sum": bit_exact_vs_sequential,
            "fused_vs_padded_torch_max_rel": rel,
            "workspace_bytes": int(lib.pillars_workspace_bytes(len(pts), nb, ctypes.byref(grid.native()))),
        }
        print(name, json.dumps(result["workloads"][name]))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
