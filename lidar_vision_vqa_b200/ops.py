"""Tensor-level wrappers over the C ABI (include/pillars_b200.h).  PyTorch is used for device memory and the current
stream only; every byte of compute happens in libpillars_b200.so.  All functions require CUDA tensors and raise
:class:`NativeLibraryError` when the library or an sm_100 device is missing -- there is no fallback path."""
from __future__ import annotations

import ctypes
from dataclasses import dataclass
from typing import Dict, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _native
from ._native import NativeLibraryError, PillarsOutputs, PillarsPfn, PillarsPfnStack, check, make_grid

FOLDED_FLOATS = 13 * 64  # PILLARS_FOLDED_FLOATS
SCATTER_VARIANTS = {"auto": 0, "plain": 1, "wide": 4}

_WORKSPACES: Dict[Tuple[int, int], torch.Tensor] = {}
_DEVICE_OK: Dict[int, bool] = {}


def _require_device(t: torch.Tensor) -> None:
    if not t.is_cuda:
        raise NativeLibraryError("the pillar path runs on a B200 only: expected a CUDA tensor (no CPU fallback)")
    idx = t.device.index if t.device.index is not None else torch.cuda.current_device()
    if idx not in _DEVICE_OK:
        check(_native.load().pillars_device_ok(idx), "pillars_device_ok")
        _DEVICE_OK[idx] = True


def _stream_ptr() -> int:
    return int(torch.cuda.current_stream().cuda_stream)


def workspace(nbytes: int, device: torch.device, slot: int = 0) -> torch.Tensor:
    """A cached scratch tensor (grown geometrically); one per (device, slot).  Use different slots for concurrent
    streams."""
    key = (device.index if device.index is not None else torch.cuda.current_device(), slot)
    ws = _WORKSPACES.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(max(int(nbytes * 1.25), 1 << 20), dtype=torch.uint8, device=device)
        _WORKSPACES[key] = ws
    return ws


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


@dataclass
class GridSpec:
    point_cloud_range: Sequence[float]
    voxel_size: Sequence[float]
    grid_size: Sequence[int]
    max_points: int
    max_voxels: int

    @staticmethod
    def from_range(point_cloud_range, voxel_size, max_points: int, max_voxels: int) -> "GridSpec":
        # reference: datasets/processor/data_processor.py:135-136
        r = np.asarray(point_cloud_range, dtype=np.float64)
        g = np.round((r[3:6] - r[0:3]) / np.asarray(voxel_size, dtype=np.float64)).astype(np.int64)
        return GridSpec(tuple(float(v) for v in point_cloud_range), tuple(float(v) for v in voxel_size),
                        tuple(int(v) for v in g), int(max_points), int(max_voxels))

    def native(self):
        return make_grid(self.point_cloud_range, self.voxel_size, self.grid_size, self.max_points, self.max_voxels)


@dataclass
class PfnParams:
    """One PFN layer with BatchNorm folded (eval mode), resident on the device."""

    weight: torch.Tensor  # [F, C_in] fp32
    scale: torch.Tensor   # [F]
    shift: torch.Tensor   # [F]
    c_point: int
    use_absolute_xyz: bool
    with_distance: bool
    offset: Tuple[float, float, float]
    # the layer regrouped around the pillar centre for the streaming feature kernel (pillars_fold_pfn), or None when
    # the configuration is outside what that kernel covers
    folded: Optional[torch.Tensor] = None

    def native(self) -> PillarsPfn:
        p = PillarsPfn()
        p.c_point = self.c_point
        p.c_in = int(self.weight.shape[1])
        p.f_out = int(self.weight.shape[0])
        p.use_absolute_xyz = int(self.use_absolute_xyz)
        p.with_distance = int(self.with_distance)
        for i in range(3):
            p.offset[i] = float(self.offset[i])
        p.weight = self.weight.data_ptr()
        p.scale = self.scale.data_ptr()
        p.shift = self.shift.data_ptr()
        p.folded = _ptr(self.folded)
        return p

    def prepare(self) -> "PfnParams":
        """Folds the table of the streaming feature kernel once (device side); a no-op without a device."""
        if self.folded is None and self.weight.is_cuda and self.use_absolute_xyz and not self.with_distance \
                and self.c_point <= 5 and self.weight.shape[0] == 64:
            _require_device(self.weight)
            folded = torch.empty(FOLDED_FLOATS, dtype=torch.float32, device=self.weight.device)
            nat = self.native()
            check(_native.load().pillars_fold_pfn(ctypes.byref(nat), folded.data_ptr(), _stream_ptr()), "pillars_fold_pfn")
            # built once, then read by every later call on ANY stream: finish it here (one-time cost)
            torch.cuda.current_stream(self.weight.device).synchronize()
            self.folded = folded
        return self


def fold_pfn(weight: torch.Tensor, bn: Optional[Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, float]],
             bias: Optional[torch.Tensor], *, c_point: int, use_absolute_xyz: bool, with_distance: bool, voxel_size,
             point_cloud_range, device) -> PfnParams:
    """One PFN layer folded by :func:`fold_layer`, with the streaming kernel's table prepared where it applies."""
    # pillar_vfe.py:79-81: python floats (double), later promoted into fp32 tensor arithmetic
    off = tuple(float(voxel_size[i]) / 2 + float(point_cloud_range[i]) for i in range(3))
    return PfnParams(*fold_layer(weight, bn, bias, device), int(c_point), bool(use_absolute_xyz), bool(with_distance),
                     off).prepare()


@dataclass
class PfnStackParams:
    """A one- or two-layer PFN stack with BatchNorm folded (eval mode), resident on the device: what the general
    feature kernel (csrc/pfn_multi.cu) consumes."""

    layers: Sequence[PfnParams]  # folded layers in order; only weight / scale / shift of each are used
    c_point: int
    use_absolute_xyz: bool
    with_distance: bool
    offset: Tuple[float, float, float]
    layout: int = _native.LAYOUT_PILLAR_VFE

    @property
    def f_out(self) -> int:
        return int(self.layers[-1].weight.shape[0])

    def native(self) -> PillarsPfnStack:
        s = PillarsPfnStack()
        s.n_layers = len(self.layers)
        s.c_point = self.c_point
        s.use_absolute_xyz = int(self.use_absolute_xyz)
        s.with_distance = int(self.with_distance)
        s.layout = int(self.layout)
        for i in range(3):
            s.offset[i] = float(self.offset[i])
        for i, layer in enumerate(self.layers):
            s.out_features[i] = int(layer.weight.shape[0])
            s.weight[i] = layer.weight.data_ptr()
            s.scale[i] = layer.scale.data_ptr()
            s.shift[i] = layer.shift.data_ptr()
        return s


def fold_layer(weight: torch.Tensor, bn, bias, device) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """(weight fp32, scale, shift) of one layer on `device`.  BatchNorm1d(eval) folded in float64 on the host:
    scale = gamma/sqrt(var+eps), shift = beta - mean*scale (pillar_vfe.py:21-25,38-40); USE_NORM false: scale 1,
    shift = linear.bias."""
    w = weight.detach().to(device=device, dtype=torch.float32).contiguous()
    f = w.shape[0]
    if bn is not None:
        gamma, beta, mean, var, eps = bn
        sc = gamma.detach().double().cpu() / torch.sqrt(var.detach().double().cpu() + eps)
        sh = beta.detach().double().cpu() - mean.detach().double().cpu() * sc
    else:
        sc = torch.ones(f, dtype=torch.float64)
        sh = bias.detach().double().cpu() if bias is not None else torch.zeros(f, dtype=torch.float64)
    return w, sc.to(torch.float32).contiguous().to(device), sh.to(torch.float32).contiguous().to(device)


def fold_pfn_stack(layers, *, c_point: int, use_absolute_xyz: bool, with_distance: bool, voxel_size, point_cloud_range,
                   device, layout: int = _native.LAYOUT_PILLAR_VFE) -> PfnStackParams:
    """``layers``: sequence of ``(linear_weight, bn_tuple_or_None, bias_or_None)`` in order."""
    off = tuple(float(voxel_size[i]) / 2 + float(point_cloud_range[i]) for i in range(3))
    folded = []
    for (w, bn, bias) in layers:
        wf, sc, sh = fold_layer(w, bn, bias, device)
        folded.append(PfnParams(wf, sc, sh, int(c_point), bool(use_absolute_xyz), bool(with_distance), off))
    return PfnStackParams(folded, int(c_point), bool(use_absolute_xyz), bool(with_distance), off, int(layout))


def frame_offsets_from_points(points_b: torch.Tensor, batch_size: int) -> torch.Tensor:
    """``batch_dict['points']`` ``[N, 1+C]`` (frame index in column 0, datasets/dataset.py:237-244) -> ``[B+1]`` int32."""
    _require_device(points_b)
    assert points_b.dtype == torch.float32 and points_b.dim() == 2 and points_b.is_contiguous()
    offs = torch.empty(batch_size + 1, dtype=torch.int32, device=points_b.device)
    lib = _native.load()
    check(lib.pillars_frame_offsets(points_b.data_ptr(), points_b.shape[0], points_b.shape[1], batch_size,
                                    offs.data_ptr(), _stream_ptr()), "pillars_frame_offsets")
    return offs


def _check_points(points: torch.Tensor, frame_offsets: torch.Tensor):
    _require_device(points)
    if points.dtype != torch.float32 or points.dim() != 2 or not points.is_contiguous():
        raise ValueError("points must be a contiguous float32 [N, row] tensor")
    if frame_offsets.dtype != torch.int32 or not frame_offsets.is_cuda:
        raise ValueError("frame_offsets must be an int32 CUDA tensor")


_OUTPUT_KEYS = ("pillar_features", "voxel_coords", "voxel_num_points", "voxels", "point_pillar", "point_slot", "pillar_count")


def _outputs(res: Dict[str, torch.Tensor], capacity: int, want_index_map: bool = False) -> PillarsOutputs:
    """The library's view of the output tensors in ``res``; an output without a key is skipped."""
    out = PillarsOutputs()
    out.pillar_capacity = capacity
    for key in _OUTPUT_KEYS:
        setattr(out, key, _ptr(res.get(key)))
    bev = res.get("bev")
    if bev is not None:
        setattr(out, "bev_half" if bev.dtype == torch.float16 else "bev", bev.data_ptr())
    out.want_index_map = int(want_index_map)
    return out


def voxelize(points: torch.Tensor, frame_offsets: torch.Tensor, grid: GridSpec, *, col0: int = 0,
             c_point: Optional[int] = None, capacity: Optional[int] = None, want_voxels: bool = True,
             want_membership: bool = False, ws_slot: int = 0) -> Dict[str, torch.Tensor]:
    """Hard voxelisation of a packed batch on the GPU.  Returns tensors sized ``capacity`` (default: the upper bound
    ``min(N, B*max_voxels)``) plus ``pillar_count [B+1]``; slice with the count (``trim``) after a sync."""
    _check_points(points, frame_offsets)
    lib = _native.load()
    n, stride = points.shape
    nb = frame_offsets.numel() - 1
    c_point = stride - col0 if c_point is None else c_point
    cap = min(n, nb * grid.max_voxels) if capacity is None else capacity
    cap = max(int(cap), 1)
    dev = points.device
    g = grid.native()
    res = {
        "voxel_coords": torch.empty((cap, 4), dtype=torch.int32, device=dev),
        "voxel_num_points": torch.empty((cap,), dtype=torch.int32, device=dev),
        "pillar_count": torch.empty((nb + 1,), dtype=torch.int32, device=dev),
    }
    if want_voxels:
        res["voxels"] = torch.empty((cap, grid.max_points, c_point), dtype=torch.float32, device=dev)
    if want_membership:
        res["point_pillar"] = torch.empty((n,), dtype=torch.int32, device=dev)
        res["point_slot"] = torch.empty((n,), dtype=torch.int32, device=dev)
    out = _outputs(res, cap)
    need = lib.pillars_workspace_bytes(n, nb, ctypes.byref(g))
    ws = workspace(need, dev, ws_slot)
    check(lib.pillars_voxelize(points.data_ptr(), n, stride, col0, c_point, frame_offsets.data_ptr(), nb,
                               ctypes.byref(g), ctypes.byref(out), ws.data_ptr(), ws.numel(), _stream_ptr()),
          "pillars_voxelize")
    return res


def _padded_inputs(voxels: torch.Tensor, num_points: torch.Tensor, coords: torch.Tensor, c_point: int):
    """Checks the reference's padded input and brings ``num_points`` and ``coords`` to what the library reads, with a
    flag that is 1 for float32: float32 and int32 pass through, other floating types become float32, other integer types
    int32; bool and complex tensors are refused."""
    _require_device(voxels)
    if voxels.dtype != torch.float32 or voxels.dim() != 3:
        raise ValueError("voxels must be float32 [M,P,C]")
    if voxels.shape[2] != c_point:
        raise ValueError(f"voxels have {voxels.shape[2]} channels, the PFN was built for {c_point}")

    def norm(t, name):
        if t.dtype == torch.bool or t.dtype.is_complex:
            raise ValueError(f"{name}: unsupported dtype {t.dtype}")
        is_float = t.dtype.is_floating_point
        return t.to(torch.float32 if is_float else torch.int32).contiguous(), int(is_float)

    return (voxels.contiguous(), *norm(num_points, "voxel_num_points"), *norm(coords, "voxel_coords"))


def pfn_dense(voxels: torch.Tensor, num_points: torch.Tensor, coords: torch.Tensor, pfn: PfnParams,
              voxel_size) -> torch.Tensor:
    """PillarVFE.forward on the reference's padded input: ``voxels [M,P,C]``, ``num_points [M]``, ``coords [M,4]``
    (int32 or float32 each).  Returns ``[M, F]``."""
    voxels, npts, np_f, crd, crd_f = _padded_inputs(voxels, num_points, coords, pfn.c_point)
    m, p, _ = voxels.shape
    out = torch.empty((m, pfn.weight.shape[0]), dtype=torch.float32, device=voxels.device)
    vs = (ctypes.c_float * 3)(*[float(v) for v in voxel_size])
    nat = pfn.native()
    check(_native.load().pillars_pfn_dense(voxels.data_ptr(), npts.data_ptr(), np_f, crd.data_ptr(), crd_f, m, p,
                                           ctypes.byref(nat), vs, out.data_ptr(), _stream_ptr()), "pillars_pfn_dense")
    return out


def pfn_dense_stack(voxels: torch.Tensor, num_points: torch.Tensor, coords: torch.Tensor, stack: PfnStackParams,
                    voxel_size) -> torch.Tensor:
    """PillarVFE.forward on padded voxels through a one- or two-layer stack (pillar_vfe.py:94-123 with :44-49)."""
    voxels, npts, np_f, crd, crd_f = _padded_inputs(voxels, num_points, coords, stack.c_point)
    m, p, _ = voxels.shape
    out = torch.empty((m, stack.f_out), dtype=torch.float32, device=voxels.device)
    vs = (ctypes.c_float * 3)(*[float(v) for v in voxel_size])
    nat = stack.native()
    check(_native.load().pillars_pfn_dense_stack(voxels.data_ptr(), npts.data_ptr(), np_f, crd.data_ptr(), crd_f, m, p,
                                                 ctypes.byref(nat), vs, out.data_ptr(), _stream_ptr()),
          "pillars_pfn_dense_stack")
    return out


def encode_stack(points: torch.Tensor, frame_offsets: torch.Tensor, grid: GridSpec, stack: PfnStackParams, *,
                 col0: int = 0, dynamic: bool = False, coords_cols: int = 4, with_bev: bool = False,
                 capacity: Optional[int] = None, scatter_variant: str = "auto", ws_slot: int = 0,
                 buffers: Optional["EncodeBuffers"] = None, want_index_map: bool = False) -> Dict[str, torch.Tensor]:
    """Raw points -> pillar features through a feature stack.  ``dynamic=False``: hard-voxeliser semantics (the fused
    equivalent of ``transform_points_to_voxels`` + a multi-layer ``PillarVFE``; NUM_FILTERS [64, 64] in the standard
    feature layout runs on the streaming kernel's two-layer variant, everything else on the general kernel);
    ``dynamic=True``: DynamicPillarVFE / DynamicPillarVFESimple2D semantics (dynamic_pillar_vfe.py:90-142, :193-240).
    ``buffers`` (hard mode, 4-column coords): pre-allocated outputs + workspace, as for :func:`encode_bev`;
    ``want_index_map`` (needs ``buffers``, whose workspace it is a view of): ``cell_row`` as in :func:`encode_bev`."""
    if buffers is not None and (dynamic or coords_cols != 4):
        raise ValueError("EncodeBuffers hold hard-mode outputs with (b, z, y, x) coordinates")
    if want_index_map and buffers is None:
        raise ValueError("want_index_map needs EncodeBuffers (the map is a view of their workspace)")

    def fresh(n, nb, need):  # outputs of this call alone; the workspace is the cached one of `ws_slot`
        cap = capacity
        if cap is None:
            cap = n if dynamic else min(n, nb * grid.max_voxels)
        cap = max(int(cap), 1)  # an empty batch still needs non-NULL output pointers
        dev = points.device
        nx, ny, nz = grid.grid_size
        res = {
            "pillar_features": torch.empty((cap, stack.f_out), dtype=torch.float32, device=dev),
            "voxel_coords": torch.empty((cap, coords_cols), dtype=torch.int32, device=dev),
            "voxel_num_points": torch.empty((cap,), dtype=torch.int32, device=dev),
            "pillar_count": torch.empty((nb + 1,), dtype=torch.int32, device=dev),
        }
        if with_bev:
            res["bev"] = torch.empty((nb, stack.f_out * nz, ny, nx), dtype=torch.float32, device=dev)
        return res, workspace(need, dev, ws_slot)

    nat = stack.native()
    mode = _native.MODE_DYNAMIC if dynamic else _native.MODE_HARD
    return _encode("pillars_encode_stack", (ctypes.byref(nat), mode, coords_cols), points, frame_offsets, grid,
                   stack.f_out, stack.c_point, col0, buffers, with_bev, want_index_map, scatter_variant, fresh)


def scatter_bev(pillar_features: torch.Tensor, coords: torch.Tensor, batch_size: int, nx: int, ny: int, nz: int = 1, *,
                m_dev: Optional[torch.Tensor] = None, variant: str = "auto", ws_slot: int = 0,
                out: Optional[torch.Tensor] = None, out_dtype: torch.dtype = torch.float32) -> torch.Tensor:
    """PointPillarScatter.forward: ``[B, F, ny, nx]`` float32, zero where no pillar; with ``nz > 1`` the 3-D variant
    (PointPillarScatter3d, pointpillar_scatter.py:40-73): ``[B, F*nz, ny, nx]``.  ``out_dtype=torch.float16`` fuses the
    extractor's ``astype(np.float16)`` (src/get-data/precompute_bev_features.py:394) into the same pass."""
    _require_device(pillar_features)
    feats = pillar_features.reshape(-1, pillar_features.shape[-1]).contiguous()
    if feats.dtype != torch.float32:
        raise ValueError("pillar_features must be float32")
    m, f = feats.shape
    if coords.dtype == torch.float32:
        crd, crd_f = coords.contiguous(), 1
    else:
        crd, crd_f = coords.to(torch.int32).contiguous(), 0
    dev = feats.device
    if out_dtype not in (torch.float32, torch.float16):
        raise ValueError("out_dtype must be float32 or float16")
    bev = out if out is not None else torch.empty((batch_size, f * nz, ny, nx), dtype=out_dtype, device=dev)
    if bev.dtype != out_dtype:
        raise ValueError("out has the wrong dtype")
    need = 4 * batch_size * nx * ny * nz
    ws = workspace(need, dev, ws_slot)
    if out_dtype == torch.float16:
        check(_native.load().pillars_scatter_bev_half(feats.data_ptr(), crd.data_ptr(), crd_f, m, _ptr(m_dev), batch_size,
                                                      f, nx, ny, nz, bev.data_ptr(), ws.data_ptr(), ws.numel(),
                                                      _stream_ptr()), "pillars_scatter_bev_half")
        return bev
    check(_native.load().pillars_scatter_bev(feats.data_ptr(), crd.data_ptr(), crd_f, m, _ptr(m_dev), batch_size, f, nx,
                                             ny, nz, bev.data_ptr(), ws.data_ptr(), ws.numel(), SCATTER_VARIANTS[variant],
                                             _stream_ptr()), "pillars_scatter_bev")
    return bev


class EncodeBuffers:
    """Pre-allocated outputs + workspace for repeated :func:`encode_bev` calls on same-shaped batches (no allocator
    traffic inside a timed loop).

    The BEV canvas is reused, and a canvas the library wrote last is mostly zeros already: the buffers keep two occupancy
    bitmaps (pillars_set_canvas_occupancy) so that the next call writes only the cells that are or were occupied.  Writes
    to ``bev`` through torch (in place, through views, ``out=``) are seen by its version counter and make the next call
    write the whole canvas again.  Writes torch cannot see (raw pointers, DLPack, other native libraries) must be
    followed by :meth:`invalidate_canvas` before the buffers are used again."""

    def __init__(self, n_points: int, n_frames: int, grid: GridSpec, f_out: int, device, *, with_bev: bool = True,
                 capacity: Optional[int] = None, ws_slot: int = 0, bev_dtype: torch.dtype = torch.float32,
                 wire_slab: bool = False):
        """``wire_slab``: ``pillar_features``, ``voxel_coords`` and ``pillar_count`` are views of ONE contiguous byte buffer
        ``self.wire`` (features | coordinates | counts), so the whole compact result of a step travels as a single message
        (:class:`sharding.TokenGatherer`)."""
        cap = min(n_points, n_frames * grid.max_voxels) if capacity is None else capacity
        cap = max(int(cap), 1)  # an empty batch still needs non-NULL output pointers
        nx, ny, nz = grid.grid_size
        self.capacity = cap
        self.n_points, self.n_frames = int(n_points), int(n_frames)
        self.wire = None
        if wire_slab:
            a, b = cap * f_out * 4, cap * 16
            c = (4 * (n_frames + 1) + 15) // 16 * 16
            self.wire = torch.zeros(a + b + c, dtype=torch.uint8, device=device)
            self.pillar_features = self.wire[:a].view(torch.float32).view(cap, f_out)
            self.voxel_coords = self.wire[a:a + b].view(torch.int32).view(cap, 4)
            self.pillar_count = self.wire[a + b:a + b + 4 * (n_frames + 1)].view(torch.int32)
        else:
            self.pillar_features = torch.empty((cap, f_out), dtype=torch.float32, device=device)
            self.voxel_coords = torch.empty((cap, 4), dtype=torch.int32, device=device)
            self.pillar_count = torch.empty((n_frames + 1,), dtype=torch.int32, device=device)
        self.voxel_num_points = torch.empty((cap,), dtype=torch.int32, device=device)
        self.bev = None
        if with_bev:
            with torch.inference_mode(False):  # an inference tensor has no version counter
                self.bev = torch.empty((n_frames, f_out * nz, ny, nx), dtype=bev_dtype, device=device)
            # [2, n_frames, ceil(ny*nx / 256)] bitmaps, all dirty; the library reads [parity] and writes [1 - parity]
            self._occupancy = torch.full((2, n_frames, (ny * nx + 255) // 256), -1, dtype=torch.int32, device=device)
            self._parity = 0
            self._canvas_version = self.bev._version  # of the library's last write; None: contents unknown
        g = grid.native()
        need = _native.load().pillars_workspace_bytes(n_points, n_frames, ctypes.byref(g))
        self.ws = torch.empty(need, dtype=torch.uint8, device=device)
        self.ws_slot = ws_slot

    def invalidate_canvas(self) -> None:
        """The next call writes the whole canvas: call after writing ``bev`` in a way torch's version counter does not
        see."""
        self._canvas_version = None

    def _set_canvas_occupancy(self, lib) -> None:
        """Hands the bitmaps to the next native call on this thread; immediately before that call."""
        prev = self._occupancy[self._parity].data_ptr() if self._canvas_version == self.bev._version else None
        check(lib.pillars_set_canvas_occupancy(prev, self._occupancy[1 - self._parity].data_ptr()),
              "pillars_set_canvas_occupancy")

    def _canvas_written(self, ok: bool) -> None:
        if ok:
            self._parity ^= 1
            self._canvas_version = self.bev._version
        else:
            self._canvas_version = None


def _encode_canvas(buffers: Optional[EncodeBuffers], lib, call) -> int:
    """Runs the native `call` (returns its code) with the canvas occupancy of `buffers`, when it writes their canvas."""
    if buffers is None:
        return call()
    buffers._set_canvas_occupancy(lib)
    rc = 1
    try:
        rc = call()
    finally:
        buffers._canvas_written(rc == 0)
    return rc


def _encode(entry: str, features: tuple, points: torch.Tensor, frame_offsets: torch.Tensor, grid: GridSpec, f_out: int,
            c_point: int, col0: int, buffers: Optional[EncodeBuffers], with_bev: bool, want_index_map: bool,
            scatter_variant: str, fresh=None, want_membership: bool = False, want_voxels: bool = False
            ) -> Dict[str, torch.Tensor]:
    """What :func:`encode_bev` and :func:`encode_stack` share: the checks, the outputs, the ``cell_row`` view and the
    native call ``entry``, whose feature arguments are ``features``.  The outputs and the workspace are those of
    ``buffers``, or without buffers ``fresh(n, nb, workspace_bytes) -> (result dict, workspace)``."""
    lib = _native.load()
    n, nb = points.shape[0], frame_offsets.numel() - 1
    g = grid.native()
    need = lib.pillars_workspace_bytes(n, nb, ctypes.byref(g))
    if buffers is not None:  # (the library would write past them)
        if buffers.pillar_features.shape[1] != f_out or buffers.n_frames != nb:
            raise ValueError("buffers were created for another feature width / batch size")
        if buffers.ws.numel() < need:
            raise ValueError("EncodeBuffers workspace too small for this batch")
        if with_bev and buffers.bev is None:
            raise ValueError("buffers were created without a BEV canvas")
    _check_points(points, frame_offsets)
    stride = points.shape[1]
    if stride - col0 < c_point:
        raise ValueError("points have fewer channels than the PFN expects")
    if buffers is not None:
        res = {"pillar_features": buffers.pillar_features, "voxel_coords": buffers.voxel_coords,
               "voxel_num_points": buffers.voxel_num_points, "pillar_count": buffers.pillar_count}
        if with_bev:
            res["bev"] = buffers.bev
        ws = buffers.ws
    else:
        res, ws = fresh(n, nb, need)
    cap = res["pillar_features"].shape[0]
    if want_membership:
        res["point_pillar"] = torch.empty((n,), dtype=torch.int32, device=points.device)
        res["point_slot"] = torch.empty((n,), dtype=torch.int32, device=points.device)
    if want_voxels:
        res["voxels"] = torch.empty((cap, grid.max_points, c_point), dtype=torch.float32, device=points.device)
    out = _outputs(res, cap, want_index_map)
    if want_index_map:
        # the workspace layout depends on the point count of THIS call
        off = lib.pillars_workspace_cell_row_offset(n, nb, ctypes.byref(g))
        nx, ny, _ = grid.grid_size
        res["cell_row"] = ws[off:off + 4 * nb * ny * nx].view(torch.int32).view(nb, ny, nx)
    call = getattr(lib, entry)
    args = (points.data_ptr(), n, stride, col0, frame_offsets.data_ptr(), nb, ctypes.byref(g), *features, ctypes.byref(out),
            ws.data_ptr(), ws.numel(), SCATTER_VARIANTS[scatter_variant], _stream_ptr())
    check(_encode_canvas(buffers if with_bev else None, lib, lambda: call(*args)), entry)
    return res


def encode_bev(points: torch.Tensor, frame_offsets: torch.Tensor, grid: GridSpec, pfn: PfnParams, *, col0: int = 0,
               buffers: Optional[EncodeBuffers] = None, with_bev: bool = True, scatter_variant: str = "auto",
               want_membership: bool = False, want_voxels: bool = False, want_index_map: bool = False
               ) -> Dict[str, torch.Tensor]:
    """The fused path: raw points -> pillar_features / voxel_coords / voxel_num_points / pillar_count / bev.
    ``want_index_map`` adds ``cell_row`` [n_frames, ny, nx] int32 (row of the pillar in each cell, -1 = empty): a view of
    the workspace, valid until ``buffers`` is reused -- the input of the BEV tokeniser (tokens.py) and of the backbone's
    first layer (backbone.py); it does not need a canvas (``with_bev=False``).
    Everything is enqueued on the current stream; nothing synchronises."""
    f_out = int(pfn.weight.shape[0])
    if buffers is None:  # the call's own, so that the cell_row view keeps its workspace alive
        _require_device(points)
        buffers = EncodeBuffers(points.shape[0], frame_offsets.numel() - 1, grid, f_out, points.device, with_bev=with_bev)
    nat = pfn.native()
    return _encode("pillars_encode_bev", (ctypes.byref(nat),), points, frame_offsets, grid, f_out, pfn.c_point, col0,
                   buffers, with_bev, want_index_map, scatter_variant, want_membership=want_membership,
                   want_voxels=want_voxels)


def rebase_segments(coords: torch.Tensor, segment_counts: torch.Tensor, frames_per_segment: int,
                    overflow: Optional[torch.Tensor] = None) -> torch.Tensor:
    """In place on gathered ``coords [S, R, 4]`` int32 (S rank segments of R rows each, rank-local frame indices; the
    segments may be strided views of a larger buffer) with ``segment_counts [S, k]`` int32 whose LAST column is each
    segment's live row count: live rows get ``s * frames_per_segment`` added to their frame index, padding rows get frame
    ``-1`` (skipped by the scatter and the tokeniser).  ``overflow`` (int32 [1], device) is set when a count exceeds R.  No
    host synchronisation."""
    _require_device(coords)
    if coords.dtype != torch.int32 or coords.dim() != 3 or coords.shape[2] != 4 or coords.stride(2) != 1 \
            or coords.stride(1) != 4:
        raise ValueError("coords must be an int32 [S, R, 4] tensor with contiguous rows")
    if segment_counts.dtype != torch.int32 or segment_counts.dim() != 2 or segment_counts.shape[0] != coords.shape[0] \
            or segment_counts.stride(1) != 1 or not segment_counts.is_cuda:
        raise ValueError("segment_counts must be an int32 CUDA [S, k] tensor with contiguous rows")
    k = segment_counts.shape[1]
    s_n = coords.shape[0]
    check(_native.load().pillars_rebase_segments(coords.data_ptr(), s_n, coords.shape[1],
                                                 coords.stride(0) if s_n > 1 else 4 * coords.shape[1],
                                                 segment_counts.data_ptr() + 4 * (k - 1),
                                                 segment_counts.stride(0) if s_n > 1 else k, int(frames_per_segment),
                                                 _ptr(overflow), _stream_ptr()), "pillars_rebase_segments")
    return coords


GROUPING_MODES = {"auto": 0, "hash": 1, "dense": 2}


def set_grouping(mode: str) -> None:
    """Grouping implementation (thread-local): 'auto', 'hash' (open-addressing table) or 'dense' (direct-mapped cell
    table whenever n_frames * cells < 2^31).  Outputs are bit-identical."""
    check(_native.load().pillars_set_grouping(GROUPING_MODES[mode]), "pillars_set_grouping")


def force_generic_features(on: bool) -> None:
    """Test / measurement hook: run the generic feature kernel even when the fast one is eligible."""
    _native.load().pillars_force_generic_features(int(bool(on)))


def last_launch_count() -> int:
    return int(_native.load().pillars_last_launch_count())
