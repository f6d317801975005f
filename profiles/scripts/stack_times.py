"""Two-layer PFN ([64,64], waymo_models/pointpillar_1x.yaml:34) through pillars_encode_stack vs the single-layer path.
Usage: python profiles/scripts/stack_times.py [--generic] [workload]   (--generic: the general kernel, ops.force_generic_features)"""
import os, sys, numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import lidar_vision_vqa_b200 as L
from lidar_vision_vqa_b200 import _native, ops, synth
from oracle import pillar_oracle as po
argv = [a for a in sys.argv[1:] if a != "--generic"]
wl = argv[0] if argv else "cfg2_nuscenes32_b16_pillar0.2_bev512"
ops.force_generic_features("--generic" in sys.argv)
dev = torch.device("cuda:0")
model, gc, nb = synth.WORKLOADS[wl]
grid = L.GridSpec.from_range(gc.point_cloud_range, gc.voxel_size, gc.max_points_per_voxel, gc.max_voxels)
pts, offs = synth.make_batch(nb, model, 5)
p, o = torch.from_numpy(pts).to(dev), torch.from_numpy(offs).to(dev)
def timed(fn, n=10):
    for _ in range(3): fn()
    torch.cuda.synchronize(); ts = []
    for _ in range(n):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize(); ts.append(a.elapsed_time(b))
    return float(np.median(ts))
for filters in ([64], [64, 64]):
    sd = po.random_pfn_params(11, filters, True, seed=0)
    layers = []
    for i in range(len(filters)):
        layers.append((torch.as_tensor(sd[f"pfn_layers.{i}.linear.weight"]),
                       tuple(torch.as_tensor(sd[f"pfn_layers.{i}.norm.{k}"]) for k in ("weight", "bias", "running_mean", "running_var")) + (1e-3,), None))
    st = ops.fold_pfn_stack(layers, c_point=5, use_absolute_xyz=True, with_distance=False, voxel_size=grid.voxel_size,
                            point_cloud_range=grid.point_cloud_range, device=dev)
    t = timed(lambda: ops.encode_stack(p, o, grid, st, with_bev=False))
    print(f"{wl} NUM_FILTERS {filters}: encode_stack without canvas {t * 1e3:.1f} us per batch of {nb} ({len(pts)} points)")
