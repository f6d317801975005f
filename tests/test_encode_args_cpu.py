"""Host-side argument checking of the three fused-encoder entry points (pillars_voxelize, pillars_encode_bev,
pillars_encode_stack) and of the Python wrappers' buffer checks.  Every pointer is a fake, 256-byte aligned address and every
call has exactly one fault, so each call must fail in host validation: none reaches a launch, with or without a GPU."""
import ctypes

import pytest
import torch

from lidar_vision_vqa_b200 import _native, ops

BADARG, WORKSPACE, UNSUPPORTED = -1, -2, -3
FAKE = 1 << 32  # fake device addresses: FAKE * k, never dereferenced
BIG_WS = 1 << 40


@pytest.fixture(scope="module")
def lib():
    return _native.load()


def _grid(nz=1):
    return _native.make_grid((-1.6, -1.6, -4.0, 1.6, 1.6, 4.0), (0.2, 0.2, 8.0 / nz), (16, 16, nz), 32, 1000)


def _pfn():
    p = _native.PillarsPfn()
    p.c_point, p.c_in, p.f_out, p.use_absolute_xyz = 4, 10, 64, 1
    p.weight, p.scale, p.shift = FAKE * 1, FAKE * 2, FAKE * 3
    return p


def _stack():
    s = _native.PillarsPfnStack()
    s.n_layers, s.c_point, s.use_absolute_xyz = 2, 4, 1
    s.out_features[0], s.out_features[1] = 32, 64
    for i in range(2):
        s.weight[i], s.scale[i], s.shift[i] = FAKE * (4 + i), FAKE * (6 + i), FAKE * (8 + i)
    return s


def _outputs(**kw):
    o = _native.PillarsOutputs()
    o.pillar_capacity = 100
    o.pillar_features, o.voxel_coords, o.voxel_num_points, o.pillar_count = FAKE * 10, FAKE * 11, FAKE * 12, FAKE * 13
    for k, v in kw.items():
        setattr(o, k, v)
    return o


def _call(lib, entry, *, points=FAKE * 20, n=1000, nb=2, offsets=FAKE * 21, grid=True, nz=1, pfn=True, stack=True,
          mode=_native.MODE_HARD, coords_cols=4, out=True, out_kw=None, ws=FAKE * 22, ws_bytes=BIG_WS):
    """One call of `entry` with the given single fault (everything else valid)."""
    g = ctypes.byref(_grid(nz)) if grid else None
    o = ctypes.byref(_outputs(**(out_kw or {}))) if out else None
    if entry == "voxelize":
        return lib.pillars_voxelize(points, n, 5, 0, 4, offsets, nb, g, o, ws, ws_bytes, None)
    if entry == "encode_bev":
        p = ctypes.byref(_pfn()) if pfn else None
        return lib.pillars_encode_bev(points, n, 5, 0, offsets, nb, g, p, o, ws, ws_bytes, 0, None)
    s = ctypes.byref(_stack()) if stack else None
    return lib.pillars_encode_stack(points, n, 5, 0, offsets, nb, g, s, mode, coords_cols, o, ws, ws_bytes, 0, None)


ALL = ("voxelize", "encode_bev", "encode_stack")
CANVAS = {"bev": FAKE * 30}
FAULTS = [
    # (name, entry points, call arguments, expected code)
    ("grid_null", ALL, dict(grid=False), BADARG),
    ("pfn_null", ("encode_bev",), dict(pfn=False), BADARG),
    ("stack_null", ("encode_stack",), dict(stack=False), BADARG),
    ("out_null", ALL, dict(out=False), BADARG),
    ("frame_offsets_null", ALL, dict(offsets=None), BADARG),
    ("bad_mode", ("encode_stack",), dict(mode=7), BADARG),
    ("bad_coords_cols", ("encode_stack",), dict(coords_cols=5), BADARG),
    ("canvas_needs_nz1", ("encode_bev", "encode_stack"), dict(nz=2, out_kw=CANVAS), UNSUPPORTED),
    ("index_map_needs_nz1", ALL, dict(nz=2, out_kw={"want_index_map": 1}), UNSUPPORTED),
    ("dynamic_with_canvas", ("encode_stack",), dict(mode=_native.MODE_DYNAMIC, out_kw=CANVAS), UNSUPPORTED),
    ("membership_to_stack", ("encode_stack",), dict(out_kw={"point_pillar": FAKE * 31}), UNSUPPORTED),
    ("workspace_misaligned", ALL, dict(ws=FAKE * 22 + 16), WORKSPACE),
    ("workspace_too_small", ALL, dict(ws_bytes=16), WORKSPACE),
    ("points_without_frames", ALL, dict(nb=0), BADARG),
]


@pytest.mark.parametrize("name,entries,kw,code", FAULTS, ids=[f[0] for f in FAULTS])
def test_single_fault_return_codes(lib, name, entries, kw, code):
    for entry in entries:
        assert _call(lib, entry, **kw) == code, entry
        assert lib.pillars_last_error()


@pytest.mark.parametrize("entry", ["encode_bev", "encode_stack"])
def test_canvas_occupancy_is_one_shot(lib, entry):
    both = dict(out_kw={"bev": FAKE * 30, "bev_half": FAKE * 32}, ws_bytes=16)
    assert lib.pillars_set_canvas_occupancy(FAKE * 40, FAKE * 41) == 0
    assert _call(lib, entry, **both) == BADARG  # occupancy with both canvases
    assert _call(lib, entry, **both) == WORKSPACE  # consumed by the failed call


def test_voxelize_leaves_the_canvas_occupancy_in_place(lib):
    both = dict(out_kw={"bev": FAKE * 30, "bev_half": FAKE * 32}, ws_bytes=16)
    assert lib.pillars_set_canvas_occupancy(FAKE * 40, FAKE * 41) == 0
    assert _call(lib, "voxelize", ws_bytes=16) == WORKSPACE
    assert _call(lib, "encode_bev", **both) == BADARG
    assert _call(lib, "encode_bev", **both) == WORKSPACE


@pytest.mark.parametrize("f_out,n_frames", [(64, 3), (32, 2)], ids=["batch_size", "feature_width"])
def test_encode_bev_checks_buffers_without_a_canvas(f_out, n_frames):
    """Buffers made for another batch size or feature width are refused even when no canvas is written: the library
    would write past pillar_count / the feature rows."""
    grid = ops.GridSpec.from_range((-1.6, -1.6, -4.0, 1.6, 1.6, 4.0), (0.2, 0.2, 8.0), 32, 1000)
    pfn = ops.fold_pfn(torch.zeros(64, 10), None, None, c_point=4, use_absolute_xyz=True, with_distance=False,
                       voxel_size=grid.voxel_size, point_cloud_range=grid.point_cloud_range, device="cpu")
    bufs = ops.EncodeBuffers(100, n_frames, grid, f_out, "cpu", with_bev=False)
    points = torch.zeros(100, 4)
    offsets = torch.tensor([0, 50, 100], dtype=torch.int32)
    with pytest.raises(ValueError):
        ops.encode_bev(points, offsets, grid, pfn, buffers=bufs, with_bev=False)
