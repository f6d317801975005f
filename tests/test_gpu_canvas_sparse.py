"""GPU tests (``-m gpu``, B200) of the scatter on a reused canvas (``k_scatter_sparse``): one CTA reads a span of the index
map, lists the 8-cell groups that are occupied now or were last time, and writes only those.  After every call of a
sequence through one set of buffers, the canvas must be bit-identical to a fresh call on a NaN-filled canvas."""
import numpy as np
import pytest
import torch

from lidar_vision_vqa_b200 import synth

pytestmark = pytest.mark.gpu

VS = (0.2, 0.2, 8.0)


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _grid(nx, ny):
    from lidar_vision_vqa_b200 import ops

    grid = ops.GridSpec.from_range((0.0, 0.0, -5.0, nx * VS[0], ny * VS[1], 3.0), VS, 32, 200000)
    assert tuple(grid.grid_size) == (nx, ny, 1)
    return grid


def _encoder(oracle, grid, dev):
    from lidar_vision_vqa_b200 import ops

    sd = oracle.random_pfn_params(11, [64], True, seed=4)
    bn = tuple(sd[f"pfn_layers.0.norm.{k}"] for k in ("weight", "bias", "running_mean", "running_var")) + (1e-3,)
    pfn = ops.fold_pfn(sd["pfn_layers.0.linear.weight"], bn, None, c_point=5, use_absolute_xyz=True, with_distance=False,
                       voxel_size=grid.voxel_size, point_cloud_range=grid.point_cloud_range, device=dev)
    return lambda p, o, g, b: ops.encode_bev(p, o, g, pfn, buffers=b)


def _cells(nx, cells, rng):
    """One point in each listed cell (flat index y * nx + x) of a frame."""
    cells = np.asarray(cells, np.int64)
    x, y = cells % nx, cells // nx
    return np.stack([(x + rng.uniform(0.2, 0.8, x.size)) * VS[0], (y + rng.uniform(0.2, 0.8, y.size)) * VS[1],
                     rng.uniform(-1, 1, x.size), rng.uniform(0, 1, x.size), np.zeros(x.size)], 1).astype(np.float32)


def _batch(frames):
    pts = np.concatenate(frames) if frames else np.zeros((0, 5), np.float32)
    return pts, np.concatenate([[0], np.cumsum([f.shape[0] for f in frames])]).astype(np.int32)


def _check_sequence(encode, grid, n_frames, batches, dtype, dev):
    from lidar_vision_vqa_b200 import ops

    n_max = max(1, max(b[0].shape[0] for b in batches))
    bufs = ops.EncodeBuffers(n_max, n_frames, grid, 64, dev, bev_dtype=dtype)
    for i, (pts, offs) in enumerate(batches):
        p, o = torch.from_numpy(pts).to(dev), torch.from_numpy(offs).to(dev)
        got = encode(p, o, grid, bufs)["bev"]
        fresh = ops.EncodeBuffers(n_max, n_frames, grid, 64, dev, bev_dtype=dtype)
        fresh.bev.fill_(float("nan"))
        ref = encode(p, o, grid, fresh)["bev"]
        torch.cuda.synchronize()
        assert got is bufs.bev
        assert torch.equal(got, ref), f"step {i}"


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
@pytest.mark.parametrize("nb", [1, 2])
@pytest.mark.parametrize("shape", [(128, 64), (40, 40), (36, 26)])
def test_sparse_sequence(shape, nb, dtype, dev, oracle):
    """(128, 64): 8192 cells, every group of every span dirty (full lists);  (40, 40): 1600 cells, a plane that ends inside a
    bitmap word and inside a span (tail CTA);  (36, 26): 936 cells, the last float16 lane pair lies half outside the plane.
    Each sequence has full frames, sparse ones, an empty batch after a full one (prev set, now empty) and single pillars
    whose float16 lane pair has one dirty lane."""
    nx, ny = shape
    plane = nx * ny
    grid = _grid(nx, ny)
    encode = _encoder(oracle, grid, dev)
    rng = np.random.default_rng(nx * 1000 + ny + nb)
    full = _batch([_cells(nx, np.arange(plane), rng) for _ in range(nb)])
    sparse = [_batch([_cells(nx, rng.choice(plane, plane // d, replace=False), rng) for _ in range(nb)]) for d in (5, 40)]
    single = [_batch([_cells(nx, [c], rng)] + [_cells(nx, [], rng)] * (nb - 1)) for c in (8, 16 * 3 + 8, plane - 8)]
    empty = _batch([_cells(nx, [], rng)] * nb)
    _check_sequence(encode, grid, nb, [full, full, sparse[0], empty, single[0], single[1], full, empty, empty, sparse[1],
                                       single[2], sparse[0], full, sparse[1]], dtype, dev)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
def test_cfg4_shape(dtype, dev, oracle):
    """cfg4's canvas: 8 frames of 1024 x 1024 cells, 5 Waymo-like batches cycling through one set of buffers."""
    from lidar_vision_vqa_b200 import ops

    model, gc, nb = synth.WORKLOADS["cfg4_waymo64_pillar0.1_bev1024"]
    grid = ops.GridSpec.from_range(gc.point_cloud_range, gc.voxel_size, gc.max_points_per_voxel, gc.max_voxels)
    assert tuple(grid.grid_size)[:2] == (1024, 1024)
    encode = _encoder(oracle, grid, dev)
    batches = [synth.make_batch(nb, model, 5, seed0=r * nb) for r in range(3)]
    _check_sequence(encode, grid, nb, [batches[0], batches[1], batches[2], batches[0], batches[0], batches[2]], dtype, dev)
