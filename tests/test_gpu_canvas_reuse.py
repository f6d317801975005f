"""GPU tests (``-m gpu``, B200) of canvas reuse: ``EncodeBuffers`` keep occupancy bitmaps so that a call writes only the
canvas cells that are or were occupied.  After every call of a sequence of different batches through one set of
buffers, the canvas must be bit-identical to a fresh call whose canvas was filled with NaN first (every element written)."""
import numpy as np
import pytest
import torch
from torch.utils import dlpack

from lidar_vision_vqa_b200 import synth

pytestmark = pytest.mark.gpu

CFG2_RANGE, CFG2_VOXEL = (-51.2, -51.2, -5.0, 51.2, 51.2, 3.0), (0.2, 0.2, 8.0)
NB = 2


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _bn(sd, i):
    return tuple(sd[f"pfn_layers.{i}.norm.{k}"] for k in ("weight", "bias", "running_mean", "running_var")) + (1e-3,)


def _encoder(path, oracle, grid, dev):
    """encode(points, offsets, grid, buffers, variant) -> result dict, through encode_bev or the two-layer encode_stack."""
    from lidar_vision_vqa_b200 import ops

    if path == "bev":
        sd = oracle.random_pfn_params(11, [64], True, seed=2)
        pfn = ops.fold_pfn(sd["pfn_layers.0.linear.weight"], _bn(sd, 0), None, c_point=5, use_absolute_xyz=True,
                           with_distance=False, voxel_size=grid.voxel_size, point_cloud_range=grid.point_cloud_range,
                           device=dev)
        return lambda p, o, g, b, v="auto": ops.encode_bev(p, o, g, pfn, buffers=b, scatter_variant=v)
    sd = oracle.random_pfn_params(11, [64, 64], True, seed=3)
    stack = ops.fold_pfn_stack([(sd[f"pfn_layers.{i}.linear.weight"], _bn(sd, i), None) for i in range(2)], c_point=5,
                               use_absolute_xyz=True, with_distance=False, voxel_size=grid.voxel_size,
                               point_cloud_range=grid.point_cloud_range, device=dev)
    return lambda p, o, g, b, v="auto": ops.encode_stack(p, o, g, stack, with_bev=True, buffers=b, scatter_variant=v)


def _fresh(encode, p, o, grid, dtype, dev, variant="auto"):
    """The canvas of a call on new buffers whose canvas holds NaN everywhere."""
    from lidar_vision_vqa_b200 import ops

    b = ops.EncodeBuffers(p.shape[0], o.numel() - 1, grid, 64, dev, bev_dtype=dtype)
    b.bev.fill_(float("nan"))
    return encode(p, o, grid, b, variant)["bev"].clone()


def _dev(batch, dev):
    return torch.from_numpy(batch[0]).to(dev), torch.from_numpy(batch[1]).to(dev)


def _cfg2(seed):
    return synth.make_batch(NB, synth.NUSCENES_32, 5, seed0=seed)


def _empty():
    return np.zeros((0, 5), np.float32), np.zeros(NB + 1, np.int32)


def _single_pillar():
    return np.array([[1.0, 2.0, 0.0, 0.5, 0.0]], np.float32), np.array([0, 0, 1], np.int32)


def _check_sequence(encode, bufs, steps, dtype, dev):
    for i, (batch, grid, variant) in enumerate(steps):
        p, o = _dev(batch, dev)
        got = encode(p, o, grid, bufs, variant)["bev"]
        ref = _fresh(encode, p, o, grid, dtype, dev, variant)
        torch.cuda.synchronize()
        assert got is bufs.bev
        assert torch.equal(got, ref), f"step {i}"


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
@pytest.mark.parametrize("path", ["bev", "stack"])
def test_reused_canvas_equals_fresh_canvas(path, dtype, dev, oracle):
    from lidar_vision_vqa_b200 import ops

    grid = ops.GridSpec.from_range(CFG2_RANGE, CFG2_VOXEL, 32, 30000)
    capped = ops.GridSpec.from_range(CFG2_RANGE, CFG2_VOXEL, 32, 300)  # max_voxels binds: fewer pillars than cells hit
    encode = _encoder(path, oracle, grid, dev)
    batches = [_cfg2(s) for s in (0, 7, 30, 11)]
    bufs = ops.EncodeBuffers(max(b[0].shape[0] for b in batches), NB, grid, 64, dev, bev_dtype=dtype)
    plain = "plain" if dtype == torch.float32 else "auto"  # the float16 canvas has one kernel
    _check_sequence(encode, bufs, [
        (batches[0], grid, "auto"), (batches[0], grid, "auto"), (batches[1], grid, "auto"), (_empty(), grid, "auto"),
        (_single_pillar(), grid, "auto"), (batches[2], grid, "auto"), (batches[2], capped, "auto"),
        (batches[0], grid, plain), (batches[3], grid, "auto"), (batches[1], capped, "auto"),
    ], dtype, dev)

    # a torch write to the returned canvas is seen by its version counter
    bufs.bev[:, :, 100:140].fill_(float("nan"))
    bufs.bev[0].add_(1)
    _check_sequence(encode, bufs, [(batches[3], grid, "auto")], dtype, dev)

    # a write torch cannot see, announced with invalidate_canvas()
    alias = dlpack.from_dlpack(dlpack.to_dlpack(bufs.bev))
    version = bufs.bev._version
    alias.fill_(float("nan"))
    assert bufs.bev._version == version
    bufs.invalidate_canvas()
    _check_sequence(encode, bufs, [(batches[0], grid, "auto"), (batches[1], grid, "auto")], dtype, dev)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
def test_fully_occupied_small_grid(dtype, dev, oracle):
    """Every cell of a 32 x 32 grid holds a pillar in frame 0, alternating with sparse batches."""
    from lidar_vision_vqa_b200 import ops

    rng, vs = (-3.2, -3.2, -5.0, 3.2, 3.2, 3.0), (0.2, 0.2, 8.0)
    grid = ops.GridSpec.from_range(rng, vs, 32, 30000)
    encode = _encoder("bev", oracle, grid, dev)
    g = np.random.default_rng(5)
    yy, xx = np.meshgrid(np.arange(32), np.arange(32), indexing="ij")
    full0 = np.stack([-3.1 + 0.2 * xx.ravel(), -3.1 + 0.2 * yy.ravel(), g.uniform(-1, 1, 1024), g.uniform(0, 1, 1024),
                      np.zeros(1024)], 1).astype(np.float32)
    sparse = g.uniform([-3.2, -3.2, -1, 0, 0], [3.2, 3.2, 1, 1, 0], (40, 5)).astype(np.float32)
    full = (np.concatenate([full0, sparse]), np.array([0, 1024, 1064], np.int32))
    thin = (sparse[::2].copy(), np.array([0, 10, 20], np.int32))
    bufs = ops.EncodeBuffers(1064, NB, grid, 64, dev, bev_dtype=dtype)
    _check_sequence(encode, bufs, [(full, grid, "auto"), (thin, grid, "auto"), (full, grid, "auto"), (full, grid, "auto"),
                                   (thin, grid, "auto")], dtype, dev)


def test_plane_on_the_plain_kernel(dev, oracle):
    """30 x 25 cells (not a multiple of 8): the plain kernel writes everything and marks the canvas all dirty."""
    from lidar_vision_vqa_b200 import ops

    rng, vs = (0.0, 0.0, -5.0, 6.0, 5.0, 3.0), (0.2, 0.2, 8.0)
    grid = ops.GridSpec.from_range(rng, vs, 32, 30000)
    assert tuple(grid.grid_size) == (30, 25, 1)
    encode = _encoder("bev", oracle, grid, dev)
    g = np.random.default_rng(6)
    batches = [(g.uniform([0, 0, -1, 0, 0], [6, 5, 1, 1, 0], (n, 5)).astype(np.float32), np.array([0, n // 2, n], np.int32))
               for n in (300, 40, 300)]
    bufs = ops.EncodeBuffers(300, NB, grid, 64, dev)
    _check_sequence(encode, bufs, [(b, grid, "auto") for b in batches + batches[:1]], torch.float32, dev)


def test_output_ring_over_streams(dev, oracle):
    """The module's OUTPUT_RING buffers, each used on several streams in turn, return the canvas of a fresh call."""
    import lidar_vision_vqa_b200 as L
    from lidar_vision_vqa_b200 import ops

    grid = ops.GridSpec.from_range(CFG2_RANGE, CFG2_VOXEL, 32, 30000)
    sd = oracle.random_pfn_params(11, [64], True, seed=2)
    cfg = dict(USE_NORM=True, WITH_DISTANCE=False, USE_ABSLOTE_XYZ=True, NUM_FILTERS=[64], MAX_POINTS_PER_VOXEL=32,
               MAX_NUMBER_OF_VOXELS=30000, FUSE_SCATTER=True, OUTPUT_RING=2, SYNC_COUNTS=False)

    class C(dict):
        __getattr__ = dict.__getitem__

    def module(ring):
        vfe = L.PillarVFEFromPoints(model_cfg=C(cfg, OUTPUT_RING=ring), num_point_features=5, voxel_size=list(CFG2_VOXEL),
                                    point_cloud_range=list(CFG2_RANGE), grid_size=np.array(grid.grid_size))
        vfe.load_state_dict(sd, strict=True)
        return vfe.eval().to(dev)

    vfe, fresh = module(2), module(0)  # OUTPUT_RING 0: new buffers, whole canvas written, on every call
    batches = [_cfg2(s) for s in (0, 7, 30)]
    pcdet = [torch.from_numpy(synth.to_pcdet_points(*b)).to(dev) for b in batches]
    refs = [fresh({"points": p, "batch_size": NB})["spatial_features"].clone() for p in pcdet]
    streams = [torch.cuda.Stream(device=dev) for _ in range(3)]
    torch.cuda.synchronize()
    for k in range(9):
        with torch.cuda.stream(streams[k % 3]):
            bd = vfe({"points": pcdet[k % 3], "batch_size": NB})
        torch.cuda.synchronize()
        assert torch.equal(bd["spatial_features"], refs[k % 3]), f"call {k}"


def test_batch_size_must_match_buffers(dev, oracle):
    from lidar_vision_vqa_b200 import ops

    grid = ops.GridSpec.from_range(CFG2_RANGE, CFG2_VOXEL, 32, 30000)
    encode = _encoder("bev", oracle, grid, dev)
    p, o = _dev(synth.make_batch(NB + 1, synth.NUSCENES_32, 5, seed0=0), dev)
    bufs = ops.EncodeBuffers(4 * p.shape[0], NB, grid, 64, dev)  # workspace large enough: the canvas is what is too small
    with pytest.raises(ValueError, match="batch size"):
        encode(p, o, grid, bufs)
