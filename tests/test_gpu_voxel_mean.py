"""pillars_voxelize_mean / ops.voxelize_mean / MeanVFEFromPoints on a B200 (run with ``-m gpu``): the hard voxeliser on
VoxelNeXt's nuScenes grid (1440 x 1440 x 40, synth.VOXELNEXT_NUSCENES) followed by MeanVFE, against the CPU voxeliser
(oracle.voxelize_batch) and MeanVFE restated on its padded voxels (mean_vfe_ref.py).

Bars: coordinates, counts and per-frame counts bit-exact; voxel_features bit-exact against the sequential fp32 sum over
the padded slots, and within rtol 1e-6 of the reference's torch formula."""
import numpy as np
import pytest
import torch

from mean_vfe_ref import mean_vfe, mean_vfe_sequential
from lidar_vision_vqa_b200 import synth

GC = synth.VOXELNEXT_NUSCENES
RNG, VS, P = GC.point_cloud_range, GC.voxel_size, GC.max_points_per_voxel


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def L():
    import lidar_vision_vqa_b200 as pkg
    from lidar_vision_vqa_b200 import ops

    pkg.ops = ops
    return pkg


@pytest.fixture(params=["auto", "dense"])
def grouping(request, L):
    """Automatic grouping (the hash table on VoxelNeXt's grid) and the direct-mapped table forced."""
    L.ops.set_grouping(request.param)
    yield request.param
    L.ops.set_grouping("auto")


def _run(L, dev, pts, offs, p=P, mv=GC.max_voxels, rng=RNG, vs=VS):
    grid = L.GridSpec.from_range(rng, vs, p, mv)
    res = L.ops.voxelize_mean(torch.from_numpy(pts).to(dev), torch.from_numpy(offs).to(dev), grid)
    torch.cuda.synchronize()
    m = int(res["pillar_count"][-1].item())
    return {k: (v.cpu().numpy() if k == "pillar_count" else v[:m].cpu().numpy()) for k, v in res.items()}


def _check(got, pts, offs, p=P, mv=GC.max_voxels, rng=RNG, vs=VS, oracle=None):
    ref = oracle.voxelize_batch(pts, offs, rng, vs, p, mv)
    np.testing.assert_array_equal(got["pillar_count"][:-1], ref["pillars_per_frame"])
    assert got["pillar_count"][-1] == ref["coords"].shape[0]
    np.testing.assert_array_equal(got["voxel_coords"], ref["coords"])
    np.testing.assert_array_equal(got["voxel_num_points"], ref["num_points"])
    want = mean_vfe_sequential(ref["voxels"], ref["num_points"])
    np.testing.assert_array_equal(got["voxel_features"].view(np.uint32), want.view(np.uint32))
    np.testing.assert_allclose(got["voxel_features"], mean_vfe(ref["voxels"], ref["num_points"]).numpy(), rtol=1e-6, atol=0)
    return ref


FULL_CASES = {
    # name: (frames, sweep model, C, max_voxels, whether the cap binds in every frame)
    "b16_single_c4": (16, synth.NUSCENES_32, 4, 160000, False),
    "b16_single_c5": (16, synth.NUSCENES_32, 5, 160000, False),
    "b16_single_c4_cap_binds": (16, synth.NUSCENES_32, 4, 12000, True),
    "b8_10sweep_c5": (8, synth.NUSCENES_10SWEEP, 5, 160000, True),  # ~250k occupied voxels per ten-sweep cloud
    "b8_10sweep_c4_uncapped": (8, synth.NUSCENES_10SWEEP, 4, 400000, False),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(FULL_CASES))
def test_voxelnext_grid_full_size(name, dev, L, oracle):
    nb, model, c, mv, binds = FULL_CASES[name]
    pts, offs = synth.make_batch(nb, model, c, seed0=300 + len(name))
    got = _run(L, dev, pts, offs, mv=mv)
    ref = _check(got, pts, offs, mv=mv, oracle=oracle)
    n = ref["num_points"]
    assert (n > 1).any() and (n == 1).any()
    assert (ref["pillars_per_frame"] == mv).all() if binds else (ref["pillars_per_frame"] < mv).all()
    if model is synth.NUSCENES_10SWEEP:  # P = 10 binds in hundreds of voxels per ten-sweep cloud
        assert (n == P).sum() > 100 * nb
    # a second run gives the same bits
    again = _run(L, dev, pts, offs, mv=mv)
    for k in got:
        np.testing.assert_array_equal(again[k], got[k])


def _voxel_points(g, cell, count, c):
    """`count` points strictly inside voxel `cell` = (x, y, z), random channels."""
    lo = np.array([RNG[i] + cell[i] * VS[i] for i in range(3)], np.float64)
    xyz = lo + g.uniform(0.05, 0.95, (count, 3)) * np.asarray(VS)
    rest = g.uniform(0.0, 255.0, (count, c - 3))
    return np.concatenate([xyz, rest], 1).astype(np.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("p", [10, 40])
def test_long_voxels(p, grouping, dev, L, oracle):
    """Voxels of ~1000, 64, 33, 32, 31 points (lists longer than a 16-lane group and a warp) among ordinary ones, in
    shuffled order: the kept set is the p smallest indices and the sum runs in index order."""
    g = np.random.default_rng(5)
    parts = [_voxel_points(g, (700, 720, 20), 1000, 5)]
    for k, cnt in enumerate((64, 33, 32, 31, 17, 16, 15, 1)):
        parts.append(_voxel_points(g, (710 + 3 * k, 700, 25), cnt, 5))
    frame0 = np.concatenate(parts)
    frame0 = frame0[g.permutation(len(frame0))]
    frame1 = synth.make_sweep(9, synth.NUSCENES_32, 5)
    pts = np.concatenate([frame0, frame1])
    offs = np.array([0, len(frame0), len(pts)], np.int32)
    got = _run(L, dev, pts, offs, p=p)
    ref = _check(got, pts, offs, p=p, oracle=oracle)
    # frame 0 holds exactly these nine voxels, numbered in order of first appearance
    assert sorted(ref["num_points"][:ref["pillars_per_frame"][0]]) == sorted(min(n, p) for n in (1000, 64, 33, 32, 31, 17, 16, 15, 1))


@pytest.mark.gpu
def test_faces_z_rejection_and_zero_signs(grouping, dev, L, oracle):
    """Points exactly on every face of the range (x == 54.0 and z == 3.0 are outside, -54 and -5 inside), points rejected
    in z only, and -0.0 channels: a full voxel of -0.0 keeps its sign, a padded one ends at +0.0."""
    pts = [
        [-54.0, 0.1, 0.1, 1, 0], [54.0, 0.1, 0.1, 2, 0], [0.1, -54.0, 0.1, 3, 0], [0.1, 54.0, 0.1, 4, 0],
        [0.1, 0.1, -5.0, 5, 0], [0.1, 0.1, 3.0, 6, 0], [53.99999, 53.99999, 2.99999, 7, 0], [-54.0, -54.0, -5.0, 8, 0],
        [1.0, 1.0, -5.0001, 9, 0], [1.0, 1.0, 3.5, 10, 0], [1.0, 1.0, -7.0, 11, 0], [1.0, 1.0, np.nan, 12, 0],
    ]
    g = np.random.default_rng(1)
    full = _voxel_points(g, (100, 100, 10), P, 5)
    full[:, 3:] = -0.0
    part = _voxel_points(g, (101, 100, 10), 3, 5)
    part[:, 3:] = -0.0
    frame = np.concatenate([np.asarray(pts, np.float32), full, part])
    offs = np.array([0, len(frame)], np.int32)
    got = _run(L, dev, frame, offs)
    ref = _check(got, frame, offs, oracle=oracle)
    bits = got["voxel_features"][:, 3].view(np.uint32)
    assert (bits == 0x80000000).sum() == 1 and ref["coords"].shape[0] == 7  # 5 points inside the faces + the two voxels


@pytest.mark.gpu
def test_empty_frames_and_empty_batch(grouping, dev, L, oracle):
    sweep = synth.make_sweep(3, synth.NUSCENES_32, 4)
    out_of_range = np.full((40, 4), 100.0, np.float32)
    pts = np.concatenate([sweep, out_of_range])
    offs = np.array([0, 0, len(sweep), len(sweep), len(pts)], np.int32)  # frames 0 and 2 empty, frame 3 all rejected
    got = _run(L, dev, pts, offs)
    _check(got, pts, offs, oracle=oracle)
    assert got["pillar_count"].tolist()[:4] == [0, got["pillar_count"][1], 0, 0]
    empty = _run(L, dev, np.zeros((0, 4), np.float32), np.zeros(3, np.int32))
    assert empty["pillar_count"].tolist() == [0, 0, 0] and empty["voxel_features"].shape == (0, 4)


@pytest.mark.gpu
@pytest.mark.parametrize("col0,c", [(0, 16), (3, 13)])
def test_wide_rows(col0, c, dev, L, oracle):
    """Rows of 16 floats (the widest the library takes): every channel of the mean is written, from column col0 on."""
    sweep = synth.make_sweep(21, synth.NUSCENES_10SWEEP, 5)
    g = np.random.default_rng(3)
    # extra channels are non-negative like intensity and time, so the rtol bound against torch holds (no cancellation)
    rows = np.concatenate([g.uniform(0, 9, (len(sweep), col0)), sweep, g.uniform(0, 9, (len(sweep), 16 - col0 - 5))],
                          1).astype(np.float32)
    offs = np.array([0, len(rows) // 2, len(rows)], np.int32)
    grid = L.GridSpec.from_range(RNG, VS, P, GC.max_voxels)
    res = L.ops.voxelize_mean(torch.from_numpy(rows).to(dev), torch.from_numpy(offs).to(dev), grid, col0=col0)
    torch.cuda.synchronize()
    m = int(res["pillar_count"][-1].item())
    got = {k: (v.cpu().numpy() if k == "pillar_count" else v[:m].cpu().numpy()) for k, v in res.items()}
    assert got["voxel_features"].shape == (m, c)
    pts = np.ascontiguousarray(rows[:, col0:])
    ref = _check(got, pts, offs, oracle=oracle)
    assert (ref["num_points"] == P).any()


def _cfg(**kw):
    cfg = {"NAME": "MeanVFEFromPoints", "MAX_POINTS_PER_VOXEL": P,
           "MAX_NUMBER_OF_VOXELS": {"train": 120000, "test": 160000}}
    cfg.update(kw)
    return cfg


@pytest.mark.gpu
@pytest.mark.parametrize("sync", [True, False])
def test_module(sync, dev, L, oracle):
    """MeanVFEFromPoints on the collated [N, 1+C] layout and on packed rows + points_frame_offsets; SYNC_COUNTS False
    keeps capacity-sized outputs and the counts on the device."""
    pts, offs = synth.make_batch(4, synth.NUSCENES_32, 4, seed0=40)
    vfe = L.MeanVFEFromPoints(_cfg(SYNC_COUNTS=sync), 4, VS, RNG, GC.grid_size).eval()
    assert vfe.get_output_feature_dim() == 4
    ref = oracle.voxelize_batch(pts, offs, RNG, VS, P, 160000)
    m = ref["coords"].shape[0]
    want = mean_vfe_sequential(ref["voxels"], ref["num_points"])
    collated = synth.to_pcdet_points(pts, offs)
    for bd in ({"points": torch.from_numpy(collated).to(dev), "batch_size": 4},
               {"points": torch.from_numpy(pts).to(dev), "batch_size": 4, "points_frame_offsets": offs}):
        out = vfe(bd)
        pc = out["pillar_count"]
        assert pc.is_cuda and pc.cpu().tolist() == ref["pillars_per_frame"].tolist() + [m]
        feats, coords, npts = out["voxel_features"], out["voxel_coords"], out["voxel_num_points"]
        assert feats.dtype == torch.float32 and coords.dtype == torch.int32 and coords.shape[1] == 4
        if sync:
            assert feats.shape == (m, 4) and out["pillars_per_frame"].tolist() == ref["pillars_per_frame"].tolist()
        else:
            assert feats.shape[0] >= m and "pillars_per_frame" not in out
        np.testing.assert_array_equal(feats[:m].cpu().numpy().view(np.uint32), want.view(np.uint32))
        np.testing.assert_array_equal(coords[:m].cpu().numpy(), ref["coords"])
        np.testing.assert_array_equal(npts[:m].cpu().numpy(), ref["num_points"])
    # training mode takes the train cap
    vfe.train()
    out = vfe({"points": torch.from_numpy(collated).to(dev), "batch_size": 4})
    assert int(out["pillar_count"][-1].item()) == m  # 4 sweeps stay under either cap
