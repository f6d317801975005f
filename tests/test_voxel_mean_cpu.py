"""pillars_voxelize_mean and MeanVFEFromPoints without a GPU: the workspace query on VoxelNeXt's grid and on the pillar
workloads, argument errors of the new entry point, the module's contract, and the MeanVFE restatement itself."""
import ctypes

import numpy as np
import pytest
import torch

from mean_vfe_ref import mean_vfe, mean_vfe_sequential


@pytest.fixture(scope="module")
def lib():
    from lidar_vision_vqa_b200 import _native

    return _native.load()


def _grid(gc):
    from lidar_vision_vqa_b200 import GridSpec

    return GridSpec(gc.point_cloud_range, gc.voxel_size, gc.grid_size, gc.max_points_per_voxel, gc.max_voxels).native()


def test_workspace_on_the_voxelnext_grid_is_the_hash_layout(lib):
    """16 frames of 1440 x 1440 x 40 cells: the direct-mapped table is possible (< 2^31 cells) but not chosen, so the
    query reports the hash layout (the parent reported the dense layout's ~10.6 GB).  Forcing the dense table still
    gets a workspace that fits it."""
    from lidar_vision_vqa_b200 import ops, synth

    g = _grid(synth.VOXELNEXT_NUSCENES)
    n = 16 * 34_000
    auto = lib.pillars_workspace_bytes(n, 16, ctypes.byref(g))
    try:
        ops.set_grouping("hash")
        hash_only = lib.pillars_workspace_bytes(n, 16, ctypes.byref(g))
        ops.set_grouping("dense")
        dense = lib.pillars_workspace_bytes(n, 16, ctypes.byref(g))
    finally:
        ops.set_grouping("auto")
    assert auto == hash_only < 200_000_000
    assert dense > 16 * 1440 * 1440 * 40 * 8  # two 4-byte planes per (frame, cell)


# pillars_workspace_bytes of the parent commit for BASELINE.json's workloads, from no point at all through batches of
# single-sweep and ten-sweep size; the small counts on cfg4's 1024^2 canvas are where the dense table is possible but not
# preferred, so automatic grouping runs the hash table there
PARENT_WORKSPACE = {
    "cfg1_nuscenes32_b1": [(0, 1074176), (1000, 2196736), (20000, 3583744), (100000, 10777344), (34000, 4606464),
                           (300000, 30180608)],
    "cfg2_nuscenes32_b16_pillar0.2_bev512": [(0, 16810496), (1000, 33661696), (20000, 35048704), (100000, 40890112),
                                             (544000, 73308160), (4800000, 482486272)],
    "cfg3_10sweep_p32_b8": [(0, 8417792), (1000, 16880384), (20000, 18267392), (100000, 24108800), (272000, 36666624),
                            (2400000, 241256192)],
    "cfg4_waymo64_pillar0.1_bev1024": [(0, 33595904), (1000, 67224320), (20000, 68611328), (100000, 74452736),
                                       (272000, 87010560), (2400000, 266434304)],
}


@pytest.mark.parametrize("name", list(PARENT_WORKSPACE))
def test_workspace_of_the_pillar_workloads_is_unchanged(name, lib):
    """Pillar grids keep the parent's figure at every point count and under every grouping mode."""
    from lidar_vision_vqa_b200 import ops, synth

    _, gc, nb = synth.WORKLOADS[name]
    g = _grid(gc)
    try:
        for mode in ("auto", "hash", "dense"):
            ops.set_grouping(mode)
            for n, want in PARENT_WORKSPACE[name]:
                assert lib.pillars_workspace_bytes(n, nb, ctypes.byref(g)) == want, (name, mode, n)
    finally:
        ops.set_grouping("auto")


def test_voxelnext_grid_is_not_a_bench_workload():
    from lidar_vision_vqa_b200 import synth

    assert synth.VOXELNEXT_NUSCENES.grid_size == (1440, 1440, 40)
    assert all(gc != synth.VOXELNEXT_NUSCENES for _, gc, _ in synth.WORKLOADS.values())


def test_voxelize_mean_argument_errors(lib):
    """Every refusal is reported through the return code and pillars_last_error before any device work."""
    from lidar_vision_vqa_b200 import _native

    g = _native.make_grid((-54, -54, -5, 54, 54, 3), (0.075, 0.075, 0.2), (1440, 1440, 40), 10, 160000)
    dummy, ws = 4096, 1 << 20  # never dereferenced: every call below is refused first

    def call(grid=ctypes.byref(g), out=None, mean=dummy, workspace=ws, wbytes=1 << 40, stride=5, col0=0, c_point=5):
        o = out if out is not None else _native.PillarsOutputs(pillar_capacity=16)
        return lib.pillars_voxelize_mean(dummy, 100, stride, col0, c_point, dummy, 2, grid, ctypes.byref(o), mean,
                                         workspace, wbytes, None)

    assert call(mean=None) == -1  # PILLARS_E_BADARG
    assert lib.pillars_last_error()
    for field in ("pillar_features", "voxels", "point_pillar", "point_slot", "bev", "bev_half"):
        o = _native.PillarsOutputs(pillar_capacity=16)
        setattr(o, field, dummy)
        assert call(out=o) == -3, field  # PILLARS_E_UNSUPPORTED
    o = _native.PillarsOutputs(pillar_capacity=16, want_index_map=1)
    assert call(out=o) == -3
    big = _native.make_grid((-54, -54, -5, 54, 54, 3), (0.075, 0.075, 0.2), (1440, 1440, 40), 513, 160000)
    assert call(grid=ctypes.byref(big)) == -3 and b"512" in lib.pillars_last_error()
    assert call(grid=None) == -1
    assert call(stride=5, col0=1, c_point=5) == -1  # columns past the row
    assert call(stride=17, c_point=17) == -3  # rows of more than 16 floats are refused, so c_point <= 16
    assert call(workspace=None) == -2  # PILLARS_E_WORKSPACE
    assert call(workspace=ws + 16) == -2  # not 256-byte aligned
    assert call(wbytes=1024) == -2


def test_module_contract():
    import lidar_vision_vqa_b200 as L
    from lidar_vision_vqa_b200 import NativeLibraryError, synth

    gc = synth.VOXELNEXT_NUSCENES
    cfg = {"NAME": "MeanVFEFromPoints", "MAX_POINTS_PER_VOXEL": 10, "MAX_NUMBER_OF_VOXELS": {"train": 120000, "test": 160000}}
    assert L.VFE_REGISTRY["MeanVFEFromPoints"] is L.MeanVFEFromPoints
    vfe = L.MeanVFEFromPoints(model_cfg=cfg, num_point_features=4, voxel_size=gc.voxel_size,
                              point_cloud_range=np.asarray(gc.point_cloud_range), grid_size=np.asarray(gc.grid_size),
                              depth_downsample_factor=None)
    assert vfe.get_output_feature_dim() == 4 and list(vfe.state_dict()) == []
    assert vfe.max_points == 10 and vfe.grid_size == [1440, 1440, 40] and vfe.sync_counts
    assert L.MeanVFEFromPoints({}, 5, gc.voxel_size, gc.point_cloud_range, gc.grid_size).max_voxels_cfg == 160000
    with pytest.raises((KeyError, TypeError, ValueError)):
        L.MeanVFEFromPoints({"MAX_NUMBER_OF_VOXELS": {"train": 1}}, 4, gc.voxel_size, gc.point_cloud_range, gc.grid_size)
    if not torch.cuda.is_available():
        with pytest.raises(NativeLibraryError):
            vfe({"points": torch.zeros((10, 5)), "batch_size": 1})


def test_mean_vfe_restatements_agree():
    """The sequential restatement equals the torch formula up to rounding, divides by max(n, 1), and keeps -0.0 only
    where no padding slot follows."""
    g = np.random.default_rng(0)
    m, p, c = 500, 10, 5
    n = g.integers(0, p + 1, m)
    v = g.normal(size=(m, p, c)).astype(np.float32) * (np.arange(p)[None, :, None] < n[:, None, None])
    seq = mean_vfe_sequential(v, n)
    np.testing.assert_allclose(seq, mean_vfe(v, n).numpy(), rtol=1e-5, atol=1e-6)
    assert np.array_equal(seq[n == 0], np.zeros((int((n == 0).sum()), c), np.float32))
    z = np.zeros((2, p, 1), np.float32)
    z[0, :, 0] = -0.0
    z[1, :3, 0] = -0.0
    assert mean_vfe_sequential(z, np.array([p, 3])).view(np.uint32).ravel().tolist() == [0x80000000, 0]
