"""Seeded synthetic LiDAR sweeps shaped like the datasets BASELINE.json's configs name.

No dataset can be downloaded here, so every test and benchmark feeds these.  The generator is a
spinning multi-beam sensor over a ground plane with gamma-distributed obstacle ranges, per-ray
dropout and a final permutation -- the permutation mirrors ``DataProcessor.shuffle_points``
(reference: src/lidar-encoder/pcdet/datasets/processor/data_processor.py:95-105, enabled at test time
by tools/cfgs/nuscenes_models/cbgs_pp_multihead.yaml:12-16), so pillar ids come out in a scattered
first-appearance order exactly as they do after the reference's data pipeline.

Channels: (x, y, z, intensity in [0,255], t) float32 -- nuScenes layout
(reference: src/lidar-encoder/pcdet/datasets/nuscenes/nuscenes_dataset.py:85-118 for the multi-sweep form).
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import List, Sequence, Tuple

import numpy as np


@dataclass(frozen=True)
class SweepModel:
    beams: int = 32
    az_steps: int = 1084
    elev_deg: Tuple[float, float] = (-30.67, 10.67)
    sensor_height: float = 1.84
    max_range: float = 75.0
    dropout: float = 0.08
    n_sweeps: int = 1
    ego_step: float = 0.45  # metres travelled between consecutive sweeps (multi-sweep clouds)
    sweep_dt: float = 0.05
    ground_slope: float = 0.15  # amplitude of the slow ground undulation (m)
    ground_rough: float = 0.06  # per-ray ground height noise (m)


@dataclass(frozen=True)
class GridConfig:
    """Voxel grid + grouping limits (the DATA_PROCESSOR block of a PCDet yaml)."""

    point_cloud_range: Tuple[float, ...] = (-51.2, -51.2, -5.0, 51.2, 51.2, 3.0)
    voxel_size: Tuple[float, ...] = (0.2, 0.2, 8.0)
    max_points_per_voxel: int = 32
    max_voxels: int = 30000

    @property
    def grid_size(self) -> Tuple[int, int, int]:
        # reference: data_processor.py:135-136  grid = round((max - min) / voxel), computed in float64 numpy
        r = np.asarray(self.point_cloud_range, dtype=np.float64)
        g = np.round((r[3:6] - r[0:3]) / np.asarray(self.voxel_size, dtype=np.float64)).astype(np.int64)
        return int(g[0]), int(g[1]), int(g[2])


NUSCENES_32 = SweepModel()
NUSCENES_10SWEEP = SweepModel(n_sweeps=10)
WAYMO_64 = SweepModel(beams=64, az_steps=2810, elev_deg=(-17.6, 2.4), sensor_height=2.0)

# name -> (sweep model, grid config, batch) for BASELINE.json configs[0..3]
WORKLOADS = {
    "cfg1_nuscenes32_b1": (NUSCENES_32, GridConfig(), 1),
    "cfg2_nuscenes32_b16_pillar0.2_bev512": (NUSCENES_32, GridConfig(max_voxels=30000), 16),
    "cfg3_10sweep_p32_b8": (NUSCENES_10SWEEP, GridConfig(max_voxels=200000), 8),
    "cfg4_waymo64_pillar0.1_bev1024": (
        WAYMO_64,
        GridConfig(point_cloud_range=(-51.2, -51.2, -2.0, 51.2, 51.2, 4.0), voxel_size=(0.1, 0.1, 6.0),
                   max_points_per_voxel=32, max_voxels=200000),
        8,
    ),
}

# VoxelNeXt's nuScenes grid (tools/cfgs/nuscenes_models/cbgs_voxel0075_voxelnext.yaml:69-79): 1440 x 1440 x 40 voxels with
# MAX_POINTS_PER_VOXEL 10 and MAX_NUMBER_OF_VOXELS {train: 120000, test: 160000} (the test value here).  Not a WORKLOAD of
# bench.py: it feeds MeanVFEFromPoints (tests/test_gpu_voxel_mean.py, profiles/scripts/voxel_mean_times.py).
VOXELNEXT_NUSCENES = GridConfig(point_cloud_range=(-54.0, -54.0, -5.0, 54.0, 54.0, 3.0), voxel_size=(0.075, 0.075, 0.2),
                                max_points_per_voxel=10, max_voxels=160000)


def _one_revolution(rng: np.random.Generator, m: SweepModel) -> np.ndarray:
    az = (np.arange(m.az_steps, dtype=np.float64) + rng.uniform()) * (2.0 * np.pi / m.az_steps)
    el = np.deg2rad(np.linspace(m.elev_deg[0], m.elev_deg[1], m.beams))
    az_g, el_g = np.meshgrid(az, el, indexing="ij")  # firing order: all beams of one azimuth step
    # ground return; a gently undulating, rough ground spreads the rings radially (flat ground would stack ~10
    # points per near-field pillar and give 2.6 points/pillar overall instead of the ~2.1 of a real 32-beam sweep)
    h = m.sensor_height + m.ground_slope * np.sin(3.0 * az_g + rng.uniform(0.0, 2.0 * np.pi)) \
        + rng.normal(scale=m.ground_rough, size=az_g.shape)
    with np.errstate(divide="ignore", invalid="ignore"):
        r_ground = np.where(el_g < -1e-3, h / np.sin(-el_g), np.inf)
    # obstacles: a piecewise-constant range profile per azimuth sector gives object-like coherence,
    # plus a per-ray gamma draw for clutter
    n_sect = 96
    sect_r = rng.gamma(shape=2.2, scale=11.0, size=n_sect) + 2.0
    sect_h = rng.uniform(0.3, 3.5, size=n_sect)  # obstacle height above ground
    sect = (az_g / (2.0 * np.pi) * n_sect).astype(np.int64) % n_sect
    r_obj = sect_r[sect]
    z_at_obj = r_obj * np.sin(el_g)  # height relative to the sensor where the ray meets the obstacle plane
    hits_obj = (z_at_obj > -m.sensor_height) & (z_at_obj < sect_h[sect] - m.sensor_height)
    r_clutter = rng.gamma(shape=2.0, scale=14.0, size=az_g.shape) + 1.0
    use_clutter = rng.uniform(size=az_g.shape) < 0.12
    use_clutter |= ~np.isfinite(r_ground) & ~hits_obj  # rays that meet neither ground nor object end on far structure
    r = np.where(hits_obj, np.minimum(r_obj, r_ground), r_ground)
    r = np.where(use_clutter, np.minimum(r, r_clutter), r)
    r = r + rng.normal(scale=0.02, size=r.shape)
    keep = np.isfinite(r) & (r > 0.8) & (r < m.max_range) & (rng.uniform(size=r.shape) >= m.dropout)
    r, az_k, el_k = r[keep], az_g[keep], el_g[keep]
    x = r * np.cos(el_k) * np.cos(az_k)
    y = r * np.cos(el_k) * np.sin(az_k)
    z = r * np.sin(el_k)
    inten = rng.uniform(0.0, 255.0, size=r.shape)
    return np.stack([x, y, z, inten, np.zeros_like(r)], axis=1)


def make_sweep(seed: int, model: SweepModel = NUSCENES_32, num_features: int = 5, shuffle: bool = True) -> np.ndarray:
    """One frame: ``[N, num_features]`` float32, ``num_features`` in {4, 5} (4 drops the time channel, the
    product's own nuScenes yaml: tools/cfgs/dataset_configs/nuscenes_dataset.yaml:59-60)."""
    rng = np.random.default_rng(seed)
    parts = []
    for k in range(model.n_sweeps):
        p = _one_revolution(rng, model)
        p[:, 0] -= k * model.ego_step  # older sweeps sit behind the ego in the key-frame's coordinates
        p[:, 4] = k * model.sweep_dt
        parts.append(p)
    pts = np.concatenate(parts, axis=0)
    if shuffle:
        pts = pts[rng.permutation(pts.shape[0])]
    return np.ascontiguousarray(pts[:, :num_features], dtype=np.float32)


def make_batch(batch: int, model: SweepModel = NUSCENES_32, num_features: int = 5, seed0: int = 0,
               shuffle: bool = True) -> Tuple[np.ndarray, np.ndarray]:
    """Frames ``seed0 .. seed0+batch-1`` packed back to back.

    Returns ``(points [sum N, num_features] f32, frame_offsets [batch+1] i32)``.
    """
    frames = [make_sweep(seed0 + b, model, num_features, shuffle) for b in range(batch)]
    offs = np.zeros(batch + 1, dtype=np.int32)
    offs[1:] = np.cumsum([f.shape[0] for f in frames])
    return np.concatenate(frames, axis=0), offs


def to_pcdet_points(points: np.ndarray, frame_offsets: np.ndarray) -> np.ndarray:
    """Packed frames -> the collated ``batch_dict['points']`` layout ``[sum N, 1+C]`` with the batch index in
    column 0 (reference: src/lidar-encoder/pcdet/datasets/dataset.py:237-244)."""
    out = np.empty((points.shape[0], points.shape[1] + 1), dtype=np.float32)
    out[:, 1:] = points
    for b in range(len(frame_offsets) - 1):
        out[frame_offsets[b]:frame_offsets[b + 1], 0] = b
    return out
