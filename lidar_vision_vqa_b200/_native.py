"""ctypes binding of libpillars_b200.so (include/pillars_b200.h).  There is no fallback: if the shared library is
missing or the device is not an sm_100 part, the callers raise."""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_float, c_int, c_int32, c_int64, c_size_t, c_void_p
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_build", "libpillars_b200.so")

EXPORTED_SYMBOLS = (
    "pillars_abi_version",
    "pillars_last_error",
    "pillars_device_ok",
    "pillars_workspace_bytes",
    "pillars_frame_offsets",
    "pillars_voxelize",
    "pillars_fold_pfn",
    "pillars_pfn_dense",
    "pillars_scatter_bev",
    "pillars_encode_bev",
    "pillars_last_launch_count",
    "pillars_set_stage_events",
    "pillars_force_generic_features",
    "pillars_set_grouping",
    "pillars_set_debug_times",
    "pillars_rebase_segments",
    "pillars_pfn_stack_in_features",
    "pillars_pfn_dense_stack",
    "pillars_encode_stack",
    "pillars_scatter_bev_half",
    "pillars_tokens_prepare",
    "pillars_tokens_workspace_bytes",
    "pillars_bev_tokens",
    "pillars_bev_tokens_map",
    "pillars_bev_tokens_dense",
    "pillars_workspace_cell_row_offset",
    "pillars_conv_weight_bytes",
    "pillars_conv_prepare",
    "pillars_conv_forward",
    "pillars_conv_forward_residual",
    "pillars_canvas_to_rows",
    "pillars_set_canvas_occupancy",
)

ABI_VERSION = 5
LAYOUT_PILLAR_VFE, LAYOUT_SIMPLE2D = 0, 1
MODE_HARD, MODE_DYNAMIC = 0, 1


class PillarsGrid(Structure):
    _fields_ = [("range", c_float * 6), ("voxel", c_float * 3), ("grid", c_int32 * 3), ("max_points", c_int32),
                ("max_voxels", c_int32)]


class PillarsPfn(Structure):
    _fields_ = [("c_point", c_int32), ("c_in", c_int32), ("f_out", c_int32), ("use_absolute_xyz", c_int32),
                ("with_distance", c_int32), ("offset", c_float * 3), ("weight", c_void_p), ("scale", c_void_p),
                ("shift", c_void_p), ("folded", c_void_p)]


class PillarsPfnStack(Structure):
    _fields_ = [("n_layers", c_int32), ("c_point", c_int32), ("out_features", c_int32 * 2),
                ("use_absolute_xyz", c_int32), ("with_distance", c_int32), ("layout", c_int32), ("offset", c_float * 3),
                ("weight", c_void_p * 2), ("scale", c_void_p * 2), ("shift", c_void_p * 2)]


class PillarsOutputs(Structure):
    _fields_ = [("pillar_capacity", c_int64), ("pillar_features", c_void_p), ("voxel_coords", c_void_p),
                ("voxel_num_points", c_void_p), ("voxels", c_void_p), ("point_pillar", c_void_p),
                ("point_slot", c_void_p), ("pillar_count", c_void_p), ("bev", c_void_p), ("bev_half", c_void_p),
                ("want_index_map", c_int32)]


class PillarsTokenizer(Structure):
    _fields_ = [("c_in", c_int32), ("d_model", c_int32), ("dw_weight", c_void_p), ("dw_bias", c_void_p),
                ("proj_weight_t", c_void_p), ("proj_bias", c_void_p), ("ln_weight", c_void_p), ("ln_bias", c_void_p),
                ("ln_eps", c_float), ("pe", c_void_p), ("background", c_void_p), ("proj_umma", c_void_p)]


class PillarsConv(Structure):
    _fields_ = [("c_in", c_int32), ("c_out", c_int32), ("k", c_int32), ("stride", c_int32), ("pad", c_int32), ("up", c_int32),
                ("relu", c_int32), ("round_out", c_int32)]


class NativeLibraryError(RuntimeError):
    pass


_LIB: Optional[ctypes.CDLL] = None


def load(build_if_missing: bool = True) -> ctypes.CDLL:
    """Loads (building first if the .so is absent or stale and nvcc is available)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if build_if_missing:
        from . import build as _build

        if _build.needs_build():
            try:
                _build.build()  # serialised across processes by a file lock, installed with an atomic rename
            except RuntimeError:
                if not os.path.isfile(LIB_PATH):  # no nvcc and nothing built: fail below with the library error
                    pass
                # (a shipped .so that is merely older than the sources is still loaded when nvcc is absent)
    if not os.path.isfile(LIB_PATH):
        raise NativeLibraryError(f"{LIB_PATH} is missing: run `python -m lidar_vision_vqa_b200.build` "
                                 "(there is no CPU/PyTorch fallback for the pillar path)")
    lib = ctypes.CDLL(LIB_PATH)
    lib.pillars_abi_version.restype = c_int
    lib.pillars_last_error.restype = c_char_p
    lib.pillars_last_launch_count.restype = c_int
    lib.pillars_device_ok.restype = c_int
    lib.pillars_device_ok.argtypes = [c_int]
    lib.pillars_workspace_bytes.restype = c_size_t
    lib.pillars_workspace_bytes.argtypes = [c_int64, c_int32, POINTER(PillarsGrid)]
    lib.pillars_frame_offsets.restype = c_int
    lib.pillars_frame_offsets.argtypes = [c_void_p, c_int64, c_int32, c_int32, c_void_p, c_void_p]
    lib.pillars_voxelize.restype = c_int
    lib.pillars_voxelize.argtypes = [c_void_p, c_int64, c_int32, c_int32, c_int32, c_void_p, c_int32,
                                     POINTER(PillarsGrid), POINTER(PillarsOutputs), c_void_p, c_size_t, c_void_p]
    lib.pillars_fold_pfn.restype = c_int
    lib.pillars_fold_pfn.argtypes = [POINTER(PillarsPfn), c_void_p, c_void_p]
    lib.pillars_pfn_dense.restype = c_int
    lib.pillars_pfn_dense.argtypes = [c_void_p, c_void_p, c_int32, c_void_p, c_int32, c_int64, c_int32,
                                      POINTER(PillarsPfn), POINTER(c_float), c_void_p, c_void_p]
    lib.pillars_scatter_bev.restype = c_int
    lib.pillars_scatter_bev.argtypes = [c_void_p, c_void_p, c_int32, c_int64, c_void_p, c_int32, c_int32, c_int32,
                                        c_int32, c_int32, c_void_p, c_void_p, c_size_t, c_int32, c_void_p]
    lib.pillars_scatter_bev_half.restype = c_int
    lib.pillars_scatter_bev_half.argtypes = [c_void_p, c_void_p, c_int32, c_int64, c_void_p, c_int32, c_int32, c_int32,
                                             c_int32, c_int32, c_void_p, c_void_p, c_size_t, c_void_p]
    lib.pillars_encode_bev.restype = c_int
    lib.pillars_encode_bev.argtypes = [c_void_p, c_int64, c_int32, c_int32, c_void_p, c_int32, POINTER(PillarsGrid),
                                       POINTER(PillarsPfn), POINTER(PillarsOutputs), c_void_p, c_size_t, c_int32,
                                       c_void_p]
    lib.pillars_pfn_stack_in_features.restype = c_int
    lib.pillars_pfn_stack_in_features.argtypes = [POINTER(PillarsPfnStack)]
    lib.pillars_pfn_dense_stack.restype = c_int
    lib.pillars_pfn_dense_stack.argtypes = [c_void_p, c_void_p, c_int32, c_void_p, c_int32, c_int64, c_int32,
                                            POINTER(PillarsPfnStack), POINTER(c_float), c_void_p, c_void_p]
    lib.pillars_encode_stack.restype = c_int
    lib.pillars_encode_stack.argtypes = [c_void_p, c_int64, c_int32, c_int32, c_void_p, c_int32, POINTER(PillarsGrid),
                                         POINTER(PillarsPfnStack), c_int32, c_int32, POINTER(PillarsOutputs), c_void_p,
                                         c_size_t, c_int32, c_void_p]
    lib.pillars_tokens_prepare.restype = c_int
    lib.pillars_tokens_prepare.argtypes = [POINTER(PillarsTokenizer), c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_void_p,
                                           c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]
    lib.pillars_tokens_workspace_bytes.restype = c_size_t
    lib.pillars_tokens_workspace_bytes.argtypes = [c_int32, c_int32, c_int32, c_int32, c_int32]
    lib.pillars_bev_tokens.restype = c_int
    lib.pillars_bev_tokens.argtypes = [c_void_p, c_void_p, c_int32, c_int64, c_void_p, c_int32, c_int32, c_int32,
                                       POINTER(PillarsTokenizer), c_void_p, c_void_p, c_size_t, c_void_p]
    lib.pillars_bev_tokens_map.restype = c_int
    lib.pillars_bev_tokens_map.argtypes = [c_void_p, c_void_p, c_int32, c_int32, c_int32, POINTER(PillarsTokenizer), c_void_p,
                                           c_void_p, c_size_t, c_void_p]
    lib.pillars_bev_tokens_dense.restype = c_int
    lib.pillars_bev_tokens_dense.argtypes = [c_void_p, c_int32, c_int32, c_int32, POINTER(PillarsTokenizer), c_void_p,
                                             c_void_p, c_size_t, c_void_p]
    lib.pillars_workspace_cell_row_offset.restype = c_size_t
    lib.pillars_workspace_cell_row_offset.argtypes = [c_int64, c_int32, POINTER(PillarsGrid)]
    lib.pillars_conv_weight_bytes.restype = c_size_t
    lib.pillars_conv_weight_bytes.argtypes = [POINTER(PillarsConv)]
    lib.pillars_conv_prepare.restype = c_int
    lib.pillars_conv_prepare.argtypes = [POINTER(PillarsConv), c_void_p, c_void_p, c_void_p, c_void_p]
    lib.pillars_conv_forward.restype = c_int
    lib.pillars_conv_forward.argtypes = [POINTER(PillarsConv), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32,
                                         c_int32, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p]
    lib.pillars_conv_forward_residual.restype = c_int
    lib.pillars_conv_forward_residual.argtypes = [POINTER(PillarsConv), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32,
                                                  c_int32, c_int32, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p,
                                                  c_void_p]
    lib.pillars_canvas_to_rows.restype = c_int
    lib.pillars_canvas_to_rows.argtypes = [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p]
    lib.pillars_rebase_segments.restype = c_int
    lib.pillars_rebase_segments.argtypes = [c_void_p, c_int32, c_int64, c_int64, c_void_p, c_int64, c_int32, c_void_p, c_void_p]
    lib.pillars_set_debug_times.restype = c_int
    lib.pillars_set_debug_times.argtypes = [c_void_p]
    lib.pillars_set_canvas_occupancy.restype = c_int
    lib.pillars_set_canvas_occupancy.argtypes = [c_void_p, c_void_p]
    lib.pillars_set_grouping.restype = c_int
    lib.pillars_set_grouping.argtypes = [c_int]
    lib.pillars_force_generic_features.restype = c_int
    lib.pillars_force_generic_features.argtypes = [c_int]
    lib.pillars_set_stage_events.restype = c_int
    lib.pillars_set_stage_events.argtypes = [POINTER(c_void_p)]
    _LIB = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().pillars_last_error().decode(errors="replace")
        raise NativeLibraryError(f"{what} failed (code {rc}): {msg}")


def make_grid(point_cloud_range, voxel_size, grid_size, max_points: int, max_voxels: int) -> PillarsGrid:
    g = PillarsGrid()
    for i in range(6):
        g.range[i] = float(point_cloud_range[i])
    for i in range(3):
        g.voxel[i] = float(voxel_size[i])
        g.grid[i] = int(grid_size[i])
    g.max_points = int(max_points)
    g.max_voxels = int(max_voxels)
    return g
