"""MeanVFE restated for the tests of pillars_voxelize_mean (test_gpu_voxel_mean.py, test_voxel_mean_cpu.py) and for
profiles/scripts/voxel_mean_times.py, on the padded voxels of ``oracle.pillar_oracle.voxelize_batch``.

Source: ``pcdet/models/backbones_3d/vfe/mean_vfe.py:25-29`` (MeanVFE.forward) of upstream OpenPCDet, which the vendored
reference copies; the vendored file itself was not available to check the line numbers against.  Not pinned by a golden.
"""
import numpy as np
import torch


def mean_vfe(voxels, num_points) -> torch.Tensor:
    """The reference's three lines in torch fp32: ``voxels [M,P,C]`` zero padded, ``num_points [M]`` -> ``[M, C]``.
    torch picks the order of the sum, so this equals the reference up to rounding."""
    v = torch.as_tensor(voxels, dtype=torch.float32)
    points_mean = v[:, :, :].sum(dim=1, keepdim=False)
    normalizer = torch.clamp_min(torch.as_tensor(num_points).view(-1, 1), min=1.0).type_as(v)
    return (points_mean / normalizer).contiguous()


def mean_vfe_sequential(voxels, num_points) -> np.ndarray:
    """The same mean with the sum pinned down: slot 0 + slot 1 + ... + slot P-1 in IEEE fp32 (padding slots included),
    then one fp32 division by ``max(num_points, 1)``.  What pillars_voxelize_mean computes bit for bit."""
    v = np.asarray(voxels, dtype=np.float32)
    s = v[:, 0, :].copy()
    for j in range(1, v.shape[1]):
        s = s + v[:, j, :]
    d = np.maximum(np.asarray(num_points), 1).astype(np.float32)
    return s / d[:, None]
