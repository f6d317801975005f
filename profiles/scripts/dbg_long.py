import sys, numpy as np, torch
sys.path.insert(0, '/root/repo')
import lidar_vision_vqa_b200 as L
from lidar_vision_vqa_b200 import ops, synth
from oracle import pillar_oracle as po
dev=torch.device('cuda:0')
model, gc, nb = synth.WORKLOADS["cfg2_nuscenes32_b16_pillar0.2_bev512"]
grid = L.GridSpec.from_range(gc.point_cloud_range, gc.voxel_size, 32, 30000)
pts, offs = synth.make_batch(nb, model, 5)
sd = po.random_pfn_params(11, [64], True, seed=0)
pfn = ops.fold_pfn(sd["pfn_layers.0.linear.weight"], (sd["pfn_layers.0.norm.weight"], sd["pfn_layers.0.norm.bias"], sd["pfn_layers.0.norm.running_mean"], sd["pfn_layers.0.norm.running_var"], 1e-3), None, c_point=5, use_absolute_xyz=True, with_distance=False, voxel_size=grid.voxel_size, point_cloud_range=grid.point_cloud_range, device=dev)
ops.set_grouping('hash')
p, o = torch.from_numpy(pts).to(dev), torch.from_numpy(offs).to(dev)
bufs = ops.EncodeBuffers(len(pts), nb, grid, 64, dev)
for _ in range(3):
    r = ops.encode_bev(p, o, grid, pfn, buffers=bufs)
    torch.cuda.synchronize()

h=bufs.ws[:64].view(torch.int32).cpu().tolist(); print('hdr',h); k=max(h[4],1); print('loop duration histogram (4us buckets):', h[4:12], 'slowest ns', h[12], 'gw', h[13], 'block', h[14], 'smid', h[15])
print('max num points', int(r['voxel_num_points'].max()))
