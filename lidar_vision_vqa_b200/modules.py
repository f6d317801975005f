"""Drop-in modules for the pillar path, mirroring the reference's operator interface (names, constructor kwargs,
``forward(batch_dict) -> batch_dict``, state-dict keys) so they can be registered in pcdet's registries unchanged:

  reference (src/lidar-encoder/pcdet/...)                                  here
  models/backbones_3d/vfe/vfe_template.py:4-22        VFETemplate            VFETemplate
  models/backbones_3d/vfe/pillar_vfe.py:8-49          PFNLayer               PFNLayer (parameter container)
  models/backbones_3d/vfe/pillar_vfe.py:52-123        PillarVFE              PillarVFE        ('voxels' input)
  models/backbones_3d/vfe/dynamic_pillar_vfe.py:49-142 (point-input contract) PillarVFEFromPoints ('points' input,
                                                                              hard-voxeliser semantics, fused grouping)
  models/backbones_3d/vfe/mean_vfe.py:6-31            MeanVFE                MeanVFEFromPoints ('points' input, hard
                                                                              voxeliser + voxel mean, any 3-D grid)
  models/backbones_2d/map_to_bev/pointpillar_scatter.py:5-37  PointPillarScatter  PointPillarScatter

The PFN modules are inference only: BatchNorm is folded from the running statistics, so ``forward`` raises in training
mode.  MeanVFEFromPoints has no parameters and runs in either mode.
The compute is in libpillars_b200.so; a missing library or a non-sm_100 device raises (no eager fallback).
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch
import torch.nn as nn

from . import ops
from ._native import NativeLibraryError


_MISSING = object()


def _cfg_get(cfg, key, default=_MISSING):
    """EasyDict-style attribute access, plain dicts and dict subclasses whose __getattr__ raises KeyError."""
    try:
        return getattr(cfg, key)
    except (AttributeError, KeyError):
        pass
    if isinstance(cfg, dict) and key in cfg:
        return cfg[key]
    if default is _MISSING:
        raise AttributeError(f"model_cfg has no {key}")
    return default


def _tensor_version(t: torch.Tensor) -> int:
    """In-place modification counter, or -1 for inference tensors (a module moved under ``torch.inference_mode``), which do
    not track one."""
    try:
        return t._version
    except RuntimeError:
        return -1


def _dtype_of(name) -> torch.dtype:
    if isinstance(name, torch.dtype):
        return name
    table = {"float32": torch.float32, "fp32": torch.float32, "float16": torch.float16, "fp16": torch.float16,
             "half": torch.float16}
    if str(name) not in table:
        raise ValueError(f"OUT_DTYPE {name!r}: float32 or float16")
    return table[str(name)]


def _points_on_device(points: torch.Tensor) -> torch.Tensor:
    """A host batch (pinned or not) is copied as part of the call; without a GPU the call fails loudly."""
    if not points.is_cuda:
        if not torch.cuda.is_available():
            raise NativeLibraryError("the pillar path runs on a B200 only: no CUDA device (no CPU fallback)")
        points = points.cuda(non_blocking=True)
    return points.contiguous()


def _point_batch(batch_dict):
    """``(points on the device, batch size, frame offsets [B+1] int32 on the device, col0)`` of a point-input batch:
    ``points [N, 1+C]`` with the frame index in column 0, or packed ``[N, C]`` rows with ``points_frame_offsets``."""
    points = _points_on_device(batch_dict["points"])
    batch_size = int(batch_dict["batch_size"])
    packed_offs = batch_dict.get("points_frame_offsets")
    if packed_offs is None:
        return points, batch_size, ops.frame_offsets_from_points(points, batch_size), 1
    # packed [N, C] rows + explicit offsets instead of the frame-index column
    offs = torch.as_tensor(packed_offs, dtype=torch.int32)
    if not offs.is_cuda:
        offs = offs.to(points.device, non_blocking=True)
    if offs.numel() != batch_size + 1:
        raise ValueError("points_frame_offsets must have batch_size + 1 entries")
    return points, batch_size, offs, 0


class VFETemplate(nn.Module):
    def __init__(self, model_cfg, **kwargs):
        super().__init__()
        self.model_cfg = model_cfg

    def get_output_feature_dim(self):
        raise NotImplementedError

    def forward(self, **kwargs):
        raise NotImplementedError


class PFNLayer(nn.Module):
    """Holds ``linear`` / ``norm`` exactly like pillar_vfe.py:9-27 so reference checkpoints load by key and shape.
    It has no eager forward: the owning VFE folds it and calls the fused kernel."""

    def __init__(self, in_channels, out_channels, use_norm=True, last_layer=False):
        super().__init__()
        self.last_vfe = last_layer
        self.use_norm = use_norm
        if not self.last_vfe:
            out_channels = out_channels // 2
        if self.use_norm:
            self.linear = nn.Linear(in_channels, out_channels, bias=False)
            self.norm = nn.BatchNorm1d(out_channels, eps=1e-3, momentum=0.01)
        else:
            self.linear = nn.Linear(in_channels, out_channels, bias=True)

    def forward(self, inputs):  # pragma: no cover
        raise NativeLibraryError("PFNLayer has no eager path; call the owning VFE (libpillars_b200.so)")


class _PillarVFEBase(VFETemplate):
    def __init__(self, model_cfg, num_point_features, voxel_size, point_cloud_range, grid_size=None, **kwargs):
        super().__init__(model_cfg=model_cfg)
        self.use_norm = _cfg_get(model_cfg, "USE_NORM")
        self.with_distance = _cfg_get(model_cfg, "WITH_DISTANCE")
        self.use_absolute_xyz = _cfg_get(model_cfg, "USE_ABSLOTE_XYZ")
        self.num_raw_point_features = int(num_point_features)
        num_point_features += 6 if self.use_absolute_xyz else 3
        if self.with_distance:
            num_point_features += 1
        self.num_filters = list(_cfg_get(model_cfg, "NUM_FILTERS"))
        assert len(self.num_filters) > 0
        num_filters = [num_point_features] + list(self.num_filters)
        layers = []
        for i in range(len(num_filters) - 1):
            layers.append(PFNLayer(num_filters[i], num_filters[i + 1], self.use_norm,
                                   last_layer=(i >= len(num_filters) - 2)))
        self.pfn_layers = nn.ModuleList(layers)
        self.voxel_size = [float(v) for v in voxel_size]
        self.point_cloud_range = [float(v) for v in np.asarray(point_cloud_range).tolist()]
        self.voxel_x, self.voxel_y, self.voxel_z = self.voxel_size
        self.x_offset = self.voxel_x / 2 + self.point_cloud_range[0]
        self.y_offset = self.voxel_y / 2 + self.point_cloud_range[1]
        self.z_offset = self.voxel_z / 2 + self.point_cloud_range[2]
        self.grid_size = None if grid_size is None else [int(v) for v in np.asarray(grid_size).tolist()]
        self._folded = None
        self._folded_key = None
        self._stack_folded = None
        self._stack_key = None

    def get_output_feature_dim(self):
        return self.num_filters[-1]

    LAYOUT = 0  # ops / _native LAYOUT_PILLAR_VFE

    def _layer_tensors(self):
        out = []
        for layer in self.pfn_layers:
            out += [layer.linear.weight] + ([layer.norm.weight, layer.norm.bias, layer.norm.running_mean,
                                             layer.norm.running_var] if self.use_norm else [layer.linear.bias])
        return out

    def _check_eval(self):
        if self.training:
            raise RuntimeError("the B200 pillar path is inference-only (BatchNorm is folded from running statistics); "
                               "call .eval()")

    def _single_layer(self) -> bool:
        """What the streaming / single-layer kernels are instantiated for; everything else runs the general kernel."""
        return len(self.pfn_layers) == 1 and self.LAYOUT == 0 and int(self.num_filters[-1]) == 64

    def _cache_key(self, device):
        """Identifies the folded form: the device plus storage and version of every parameter and statistic."""
        self._check_eval()
        return (str(device),) + tuple((t.data_ptr(), _tensor_version(t)) for t in self._layer_tensors())

    def _fold_args(self, layer):
        """(linear weight, BatchNorm tuple or None, bias or None) of one PFNLayer, as ops.fold_layer takes them."""
        if not self.use_norm:
            return layer.linear.weight, None, layer.linear.bias
        norm = layer.norm
        return layer.linear.weight, (norm.weight, norm.bias, norm.running_mean, norm.running_var, norm.eps), None

    def _params(self, device) -> ops.PfnParams:
        """The single-layer form consumed by the streaming / dense kernels."""
        key = self._cache_key(device)
        if self._folded is None or key != self._folded_key:
            self._folded = ops.fold_pfn(*self._fold_args(self.pfn_layers[0]),
                                        c_point=self.num_raw_point_features, use_absolute_xyz=self.use_absolute_xyz,
                                        with_distance=self.with_distance, voxel_size=self.voxel_size,
                                        point_cloud_range=self.point_cloud_range, device=device)
            self._folded_key = key
        return self._folded

    def _stack(self, device) -> ops.PfnStackParams:
        """Any one- or two-layer configuration, for the general feature kernel (csrc/pfn_multi.cu)."""
        key = self._cache_key(device)
        if len(self.pfn_layers) > 2:
            raise NotImplementedError("PFN stacks of more than two layers are not built (no reference config uses one)")
        if self._stack_folded is None or key != self._stack_key:
            layers = [self._fold_args(layer) for layer in self.pfn_layers]
            self._stack_folded = ops.fold_pfn_stack(layers, c_point=self.num_raw_point_features,
                                                    use_absolute_xyz=self.use_absolute_xyz,
                                                    with_distance=self.with_distance, voxel_size=self.voxel_size,
                                                    point_cloud_range=self.point_cloud_range, device=device,
                                                    layout=self.LAYOUT)
            self._stack_key = key
        return self._stack_folded


class PillarVFE(_PillarVFEBase):
    """Reads ``voxels [M,P,C]``, ``voxel_num_points [M]``, ``voxel_coords [M,4] (b,z,y,x)`` (fp32 after
    ``load_data_to_gpu``, models/__init__.py:36, or int32) and writes ``pillar_features`` -- pillar_vfe.py:94-123."""

    def forward(self, batch_dict, **kwargs):
        voxels = batch_dict["voxels"]
        if self._single_layer():
            feats = ops.pfn_dense(voxels, batch_dict["voxel_num_points"], batch_dict["voxel_coords"],
                                  self._params(voxels.device), self.voxel_size)
        else:  # NUM_FILTERS with two entries: pillar_vfe.py:44-49,119-120
            ops._require_device(voxels)
            feats = ops.pfn_dense_stack(voxels, batch_dict["voxel_num_points"], batch_dict["voxel_coords"],
                                        self._stack(voxels.device), self.voxel_size)
        batch_dict["pillar_features"] = feats.squeeze()  # pillar_vfe.py:121 (M == 1 collapses to [F] there too)
        return batch_dict


def _mode_value(v, training: bool):
    if isinstance(v, dict) or hasattr(v, "keys"):
        return int(v["train" if training else "test"])
    return int(v)


class PillarVFEFromPoints(_PillarVFEBase):
    """Point-input variant: reads ``points [N, 1+C] (b,x,y,z,...)`` like DynamicPillarVFE (dynamic_pillar_vfe.py:90-91)
    but groups with the HARD voxeliser's semantics (first-appearance ids, first ``MAX_POINTS_PER_VOXEL`` points, at most
    ``MAX_NUMBER_OF_VOXELS`` pillars per frame), so its output equals ``transform_points_to_voxels`` + ``PillarVFE``.
    Writes ``pillar_features``, ``voxel_features`` (alias), ``voxel_coords [M,4] int32``, ``voxel_num_points``; with
    ``FUSE_SCATTER`` also ``spatial_features`` (the scatter then becomes a no-op).

    Extra model_cfg keys (all optional): MAX_POINTS_PER_VOXEL (32), MAX_NUMBER_OF_VOXELS (40000, int or
    {'train','test'}), FUSE_SCATTER (False), SCATTER_VARIANT ('auto'), SYNC_COUNTS (True), OUTPUT_RING (0),
    EMIT_INDEX_MAP (False).

    ``EMIT_INDEX_MAP: True`` adds ``batch_dict['bev_index_map'] [B, ny, nx] int32`` (row of the pillar in each cell, -1 =
    empty; a view of the call's workspace): with it ``BaseBEVBackbone`` (backbone.py) and the BEV tokeniser read the pillar
    rows directly and the dense canvas need not exist at all.

    ``SYNC_COUNTS: False`` removes the call's only host synchronisation: the per-pillar outputs then keep their CAPACITY
    (rows beyond the pillar count are undefined), and the counts stay on the
    device as ``batch_dict['pillar_count'] [B+1] int32`` (per frame, total last).  ``PointPillarScatter`` and the BEV
    tokeniser honour that count; with ``FUSE_SCATTER`` the canvas is already complete.  The default (True) reads the counts
    back and returns exactly the reference's shapes -- the reference itself synchronises at the same place
    (pointpillar_scatter.py:17).

    ``OUTPUT_RING: n`` (n > 0) makes the module own ``n`` sets of output buffers + workspace and hand them out round-robin
    instead of allocating fresh tensors per call: the outputs of call k stay valid until call k + n (issue those two calls on
    the same stream, or synchronise in between).  This is what a streaming extractor wants -- the canvas alone is 1 GiB per
    call at cfg2 -- and it is the configuration `bench.py` times end to end.

    Optional input key ``points_frame_offsets`` (``[B+1]`` int32, host or device): ``points`` is then the PACKED ``[N, C]``
    layout without the frame-index column (17 % fewer host->device bytes at C = 5)."""

    def __init__(self, model_cfg, num_point_features, voxel_size, point_cloud_range, grid_size, **kwargs):
        super().__init__(model_cfg, num_point_features, voxel_size, point_cloud_range, grid_size, **kwargs)
        self.max_points = int(_cfg_get(model_cfg, "MAX_POINTS_PER_VOXEL", 32))
        self.max_voxels = _mode_value(_cfg_get(model_cfg, "MAX_NUMBER_OF_VOXELS", 40000), training=False)
        self.fuse_scatter = bool(_cfg_get(model_cfg, "FUSE_SCATTER", False))
        self.scatter_variant = str(_cfg_get(model_cfg, "SCATTER_VARIANT", "auto"))
        self.sync_counts = bool(_cfg_get(model_cfg, "SYNC_COUNTS", True))
        self.output_ring = int(_cfg_get(model_cfg, "OUTPUT_RING", 0))
        self.emit_index_map = bool(_cfg_get(model_cfg, "EMIT_INDEX_MAP", False))
        self._ring, self._ring_next = [], 0
        self.grid = ops.GridSpec(self.point_cloud_range, self.voxel_size, self.grid_size, self.max_points,
                                 self.max_voxels)

    def forward(self, batch_dict, **kwargs):
        points, batch_size, offs, col0 = _point_batch(batch_dict)
        if self._single_layer():
            params, encode = self._params(points.device), ops.encode_bev
        else:
            params, encode = self._stack(points.device), ops.encode_stack
        buffers = None
        if self.output_ring > 0:
            buffers = self._ring_buffers(points.shape[0], batch_size, points.device)
        if self.emit_index_map and buffers is None:  # the map is a view of the workspace: keep that alive with the result
            buffers = ops.EncodeBuffers(points.shape[0], batch_size, self.grid, int(self.num_filters[-1]), points.device,
                                        with_bev=self.fuse_scatter)
        res = encode(points, offs, self.grid, params, col0=col0, buffers=buffers, with_bev=self.fuse_scatter,
                     scatter_variant=self.scatter_variant, want_index_map=self.emit_index_map)
        if self.emit_index_map:
            batch_dict["bev_index_map"] = res["cell_row"]
        if self.fuse_scatter:
            batch_dict["spatial_features"] = res["bev"]
            batch_dict["_b200_scatter_done"] = True
        batch_dict["pillar_count"] = res["pillar_count"]  # device, [B+1]
        if not self.sync_counts:
            # no host synchronisation: capacity-sized outputs, rows beyond the device-side count are padding
            batch_dict["voxel_features"] = batch_dict["pillar_features"] = res["pillar_features"]
            batch_dict["voxel_coords"] = res["voxel_coords"]
            batch_dict["voxel_num_points"] = res["voxel_num_points"]
            return batch_dict
        # the one host sync of the call: per-frame pillar counts (B+1 ints) size the returned views
        # (the reference syncs at the same place for the batch size, pointpillar_scatter.py:17)
        counts = res["pillar_count"].cpu()
        m = int(counts[-1])
        if m > res["pillar_features"].shape[0]:
            raise RuntimeError("pillar capacity overflow")
        batch_dict["voxel_features"] = batch_dict["pillar_features"] = res["pillar_features"][:m]
        batch_dict["voxel_coords"] = res["voxel_coords"][:m]
        batch_dict["voxel_num_points"] = res["voxel_num_points"][:m]
        batch_dict["pillars_per_frame"] = counts[:-1]  # host tensor
        return batch_dict


    def _ring_buffers(self, n_points: int, batch_size: int, device) -> "ops.EncodeBuffers":
        """OUTPUT_RING: the next of ``n`` module-owned buffer sets, grown when a batch has more points than any before."""
        if len(self._ring) != self.output_ring:
            self._ring = [None] * self.output_ring
        i = self._ring_next % self.output_ring
        self._ring_next += 1
        b = self._ring[i]
        if b is None or b.n_points < n_points or b.n_frames != batch_size or b.pillar_features.device != device \
                or (b.bev is None) != (not self.fuse_scatter):
            cap_points = int(n_points * 1.1) + 1024
            b = ops.EncodeBuffers(cap_points, batch_size, self.grid, int(self.num_filters[-1]), device,
                                  with_bev=self.fuse_scatter)
            self._ring[i] = b
        return b


class MeanVFEFromPoints(VFETemplate):
    """Point-input MeanVFE (mean_vfe.py:6-31) with the hard voxeliser in front: the equivalent of
    ``transform_points_to_voxels`` (data_processor.py:133-180) + ``MeanVFE`` on any 3-D grid, e.g. VoxelNeXt's
    1440 x 1440 x 40 (cbgs_voxel0075_voxelnext.yaml), with no padded ``voxels`` in between.  Reads ``points [N, 1+C]
    (b,x,y,z,...)``, or packed ``[N, C]`` rows with ``points_frame_offsets`` (as :class:`PillarVFEFromPoints`).  Writes
    ``voxel_features [M, C]`` (bit-identical to a sequential fp32 sum over the padded slots divided by the capped count),
    ``voxel_coords [M, 4] int32 (b, z, y, x)`` (what spconv's ``SparseConvTensor`` takes), ``voxel_num_points``,
    ``pillar_count [B+1]`` (device) and, with synced counts, ``pillars_per_frame`` (host).

    model_cfg keys (all optional): MAX_POINTS_PER_VOXEL (10), MAX_NUMBER_OF_VOXELS (160000; an int or {'train', 'test'},
    chosen by the module's training flag), SYNC_COUNTS (True; False keeps capacity-sized outputs and the counts on the
    device, as for :class:`PillarVFEFromPoints`).  The defaults are VoxelNeXt's nuScenes test values.  The module has no
    parameters, so it runs in training mode too."""

    def __init__(self, model_cfg, num_point_features, voxel_size, point_cloud_range, grid_size, **kwargs):
        super().__init__(model_cfg=model_cfg)
        self.num_point_features = int(num_point_features)
        self.max_points = int(_cfg_get(model_cfg, "MAX_POINTS_PER_VOXEL", 10))
        self.max_voxels_cfg = _cfg_get(model_cfg, "MAX_NUMBER_OF_VOXELS", 160000)
        _mode_value(self.max_voxels_cfg, training=False)  # an int or a {train, test} dict, checked here
        self.sync_counts = bool(_cfg_get(model_cfg, "SYNC_COUNTS", True))
        self.voxel_size = [float(v) for v in voxel_size]
        self.point_cloud_range = [float(v) for v in np.asarray(point_cloud_range).tolist()]
        self.grid_size = [int(v) for v in np.asarray(grid_size).tolist()]

    def get_output_feature_dim(self):
        return self.num_point_features

    def forward(self, batch_dict, **kwargs):
        points, batch_size, offs, col0 = _point_batch(batch_dict)
        grid = ops.GridSpec(self.point_cloud_range, self.voxel_size, self.grid_size, self.max_points,
                            _mode_value(self.max_voxels_cfg, self.training))
        res = ops.voxelize_mean(points, offs, grid, col0=col0, c_point=self.num_point_features)
        batch_dict["pillar_count"] = res["pillar_count"]  # device, [B+1]
        keys = ("voxel_features", "voxel_coords", "voxel_num_points")
        if not self.sync_counts:  # capacity-sized outputs, rows beyond the device-side count are padding
            batch_dict.update({k: res[k] for k in keys})
            return batch_dict
        counts = res["pillar_count"].cpu()  # the call's one host synchronisation
        m = int(counts[-1])
        batch_dict.update({k: res[k][:m] for k in keys})
        batch_dict["pillars_per_frame"] = counts[:-1]  # host tensor
        return batch_dict


class DynamicPillarVFE(_PillarVFEBase):
    """dynamic_pillar_vfe.py:49-142 (registry name ``DynPillarVFE``): reads ``points [N, 1+C] (b,x,y,z,...)``; quantises x,y
    on the device (z is not range checked), groups with NO per-pillar cap, ``scatter_mean`` / ``PFNLayerV2`` /
    ``scatter_max``; rows come out in the order of the merged key ``b*nx*ny + ix*ny + iy`` (``torch.unique``, :99-103) and
    ``voxel_coords`` is ``(b, 0, iy, ix)`` int32 (:132-138).  Writes ``pillar_features``, ``voxel_features``,
    ``voxel_coords`` (and ``voxel_num_points``, the uncapped counts, which the reference does not emit)."""

    COORDS_COLS = 4
    COORDS_KEY = "voxel_coords"

    def __init__(self, model_cfg, num_point_features, voxel_size, grid_size, point_cloud_range, **kwargs):
        super().__init__(model_cfg, num_point_features, voxel_size, point_cloud_range, grid_size, **kwargs)
        nx, ny, _ = self.grid_size
        # nz = 1 for the key: the dynamic variants collapse z (the reference builds its key from ix, iy only)
        self.grid = ops.GridSpec(self.point_cloud_range, self.voxel_size, (nx, ny, 1), 2 ** 31 - 1, 2 ** 31 - 1)

    def forward(self, batch_dict, **kwargs):
        points = _points_on_device(batch_dict["points"])
        if "batch_size" in batch_dict:
            batch_size = int(batch_dict["batch_size"])
        else:
            batch_size = int(points[:, 0].max().item()) + 1 if points.shape[0] else 0
        offs = ops.frame_offsets_from_points(points, batch_size)
        res = ops.encode_stack(points, offs, self.grid, self._stack(points.device), col0=1, dynamic=True,
                               coords_cols=self.COORDS_COLS)
        m = int(res["pillar_count"][-1].item())  # the reference syncs here too (torch.unique returns a sized tensor)
        feats = res["pillar_features"][:m]
        batch_dict["pillar_features"] = feats
        if self.COORDS_KEY == "voxel_coords":
            batch_dict["voxel_features"] = feats
        batch_dict[self.COORDS_KEY] = res["voxel_coords"][:m]
        batch_dict["voxel_num_points"] = res["voxel_num_points"][:m]
        return batch_dict


class DynamicPillarVFESimple2D(DynamicPillarVFE):
    """dynamic_pillar_vfe.py:145-240: features ``[f_center, point channels (, distance)]`` (no cluster offset), so the
    first linear has ``C + 3`` inputs (:151-157); writes ``pillar_features`` and ``pillar_coords [M,3] (b, iy, ix)``."""

    LAYOUT = 1
    COORDS_COLS = 3
    COORDS_KEY = "pillar_coords"

    def __init__(self, model_cfg, num_point_features, voxel_size, grid_size, point_cloud_range, **kwargs):
        nn.Module.__init__(self)
        self.model_cfg = model_cfg
        self.use_norm = _cfg_get(model_cfg, "USE_NORM")
        self.with_distance = _cfg_get(model_cfg, "WITH_DISTANCE")
        self.use_absolute_xyz = _cfg_get(model_cfg, "USE_ABSLOTE_XYZ")
        self.num_raw_point_features = int(num_point_features)
        c_in = int(num_point_features)
        if self.use_absolute_xyz:
            c_in += 3
        if self.with_distance:
            c_in += 1
        self.num_filters = list(_cfg_get(model_cfg, "NUM_FILTERS"))
        assert len(self.num_filters) > 0
        dims = [c_in] + list(self.num_filters)
        self.pfn_layers = nn.ModuleList([PFNLayer(dims[i], dims[i + 1], self.use_norm, last_layer=(i >= len(dims) - 2))
                                         for i in range(len(dims) - 1)])
        self.voxel_size = [float(v) for v in voxel_size]
        self.point_cloud_range = [float(v) for v in np.asarray(point_cloud_range).tolist()]
        self.voxel_x, self.voxel_y, self.voxel_z = self.voxel_size
        self.x_offset = self.voxel_x / 2 + self.point_cloud_range[0]
        self.y_offset = self.voxel_y / 2 + self.point_cloud_range[1]
        self.z_offset = self.voxel_z / 2 + self.point_cloud_range[2]
        self.grid_size = [int(v) for v in np.asarray(grid_size).tolist()]
        self._folded = self._folded_key = self._stack_folded = self._stack_key = None
        nx, ny = self.grid_size[0], self.grid_size[1]
        self.grid = ops.GridSpec(self.point_cloud_range, self.voxel_size, (nx, ny, 1), 2 ** 31 - 1, 2 ** 31 - 1)


class PointPillarScatter(nn.Module):
    """pointpillar_scatter.py:5-37.  ``batch_dict['batch_size']`` is used when present (the reference derives the
    batch from ``coords[:,0].max()+1`` with a host sync, :17 -- identical unless trailing frames are empty)."""

    def __init__(self, model_cfg, grid_size, **kwargs):
        super().__init__()
        self.model_cfg = model_cfg
        self.num_bev_features = _cfg_get(model_cfg, "NUM_BEV_FEATURES")
        self.nx, self.ny, self.nz = (int(v) for v in np.asarray(grid_size).tolist())
        assert self.nz == 1
        self.variant = str(_cfg_get(model_cfg, "SCATTER_VARIANT", "auto"))
        # optional: 'float16' writes the canvas in the dtype the product's extractor stores
        # (src/get-data/precompute_bev_features.py:394); the default float32 is the reference module's output
        self.out_dtype = _dtype_of(_cfg_get(model_cfg, "OUT_DTYPE", "float32"))

    def forward(self, batch_dict, **kwargs):
        if batch_dict.get("_b200_scatter_done", False) and "spatial_features" in batch_dict:
            return batch_dict
        feats, coords = batch_dict["pillar_features"], batch_dict["voxel_coords"]
        if "batch_size" in batch_dict:
            batch_size = int(batch_dict["batch_size"])
        else:
            batch_size = int(coords[:, 0].max().int().item()) + 1
        if feats.shape[-1] != self.num_bev_features:
            raise ValueError(f"pillar_features have {feats.shape[-1]} channels, NUM_BEV_FEATURES={self.num_bev_features}")
        m_dev = None
        pc = batch_dict.get("pillar_count")
        if torch.is_tensor(pc) and pc.is_cuda and pc.numel() == batch_size + 1 and feats.shape[0] >= 1:
            m_dev = pc[-1:]  # device-side live row count (PillarVFEFromPoints with SYNC_COUNTS false)
        batch_dict["spatial_features"] = ops.scatter_bev(feats, coords, batch_size, self.nx, self.ny, m_dev=m_dev,
                                                         variant=self.variant, out_dtype=self.out_dtype)
        return batch_dict


class PointPillarScatter3d(nn.Module):
    """pointpillar_scatter.py:40-73: grid from ``INPUT_SHAPE``, ``NUM_BEV_FEATURES // nz`` channels per pillar, canvas
    index ``z*ny*nx + y*nx + x``, output ``[B, NUM_BEV_FEATURES, ny, nx]``."""

    def __init__(self, model_cfg, grid_size=None, **kwargs):
        super().__init__()
        self.model_cfg = model_cfg
        self.nx, self.ny, self.nz = (int(v) for v in _cfg_get(model_cfg, "INPUT_SHAPE"))
        self.num_bev_features = _cfg_get(model_cfg, "NUM_BEV_FEATURES")
        self.num_bev_features_before_compression = self.num_bev_features // self.nz
        self.variant = str(_cfg_get(model_cfg, "SCATTER_VARIANT", "auto"))

    def forward(self, batch_dict, **kwargs):
        feats, coords = batch_dict["pillar_features"], batch_dict["voxel_coords"]
        if "batch_size" in batch_dict:
            batch_size = int(batch_dict["batch_size"])
        else:
            batch_size = int(coords[:, 0].max().int().item()) + 1
        if feats.shape[-1] != self.num_bev_features_before_compression:
            raise ValueError("pillar_features channels != NUM_BEV_FEATURES // nz")
        batch_dict["spatial_features"] = ops.scatter_bev(feats, coords, batch_size, self.nx, self.ny, self.nz,
                                                         variant=self.variant)
        return batch_dict


# name-keyed registries shaped like pcdet's (models/backbones_3d/vfe/__init__.py:9-18,
# models/backbones_2d/map_to_bev/__init__.py:5-10); INTEGRATION.md shows the two-line merge into them.
VFE_REGISTRY = {
    "VFETemplate": VFETemplate,
    "PillarVFE": PillarVFE,
    "PillarVFEFromPoints": PillarVFEFromPoints,
    "MeanVFEFromPoints": MeanVFEFromPoints,
    "DynPillarVFE": DynamicPillarVFE,
    "DynamicPillarVFESimple2D": DynamicPillarVFESimple2D,
}
MAP_TO_BEV_REGISTRY = {
    "PointPillarScatter": PointPillarScatter,
    "PointPillarScatter3d": PointPillarScatter3d,
}
