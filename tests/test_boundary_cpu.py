"""CPU tests of the drop-in boundary: the C-ABI library builds, loads and exports everything include/*.h declares;
the host modules mirror the reference's constructor / state-dict contract; compute calls fail loudly without a GPU."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT, load_golden, vfe_golden_names


class Cfg(dict):
    __getattr__ = dict.__getitem__


@pytest.fixture(scope="module")
def lib():
    from lidar_vision_vqa_b200 import _native

    return _native.load()


def test_library_exports_every_declared_symbol(lib):
    from lidar_vision_vqa_b200 import _native

    hdr = open(os.path.join(ROOT, "include", "pillars_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(pillars_[a-z_0-9]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    assert declared == set(_native.EXPORTED_SYMBOLS)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.pillars_abi_version() == _native.ABI_VERSION == 5


def test_struct_layouts_match_header_sizes():
    from lidar_vision_vqa_b200 import _native

    assert ctypes.sizeof(_native.PillarsGrid) == 6 * 4 + 3 * 4 + 3 * 4 + 4 + 4
    assert ctypes.sizeof(_native.PillarsPfn) == 5 * 4 + 3 * 4 + 4 * 8
    assert ctypes.sizeof(_native.PillarsOutputs) == 10 * 8 + 8  # + want_index_map (int32, padded)
    assert ctypes.sizeof(_native.PillarsConv) == 8 * 4
    assert ctypes.sizeof(_native.PillarsTokenizer) == 2 * 4 + 6 * 8 + 8 + 3 * 8  # eps padded to 8


def test_workspace_query_and_argument_errors(lib):
    from lidar_vision_vqa_b200 import _native

    g = _native.make_grid((-51.2, -51.2, -5, 51.2, 51.2, 3), (0.2, 0.2, 8), (512, 512, 1), 32, 30000)
    a = lib.pillars_workspace_bytes(100_000, 4, ctypes.byref(g))
    b = lib.pillars_workspace_bytes(200_000, 4, ctypes.byref(g))
    c = lib.pillars_workspace_bytes(200_000, 8, ctypes.byref(g))
    assert 0 < a < b < c
    assert lib.pillars_workspace_bytes(0, 4, ctypes.byref(g)) >= 4 * 4 * 512 * 512
    # bad arguments are reported through the return code + pillars_last_error, never a crash
    rc = lib.pillars_scatter_bev(None, None, 0, 5, None, 1, 64, 8, 8, 1, None, None, 0, 0, None)
    assert rc != 0 and lib.pillars_last_error()
    out = _native.PillarsOutputs()
    rc = lib.pillars_voxelize(None, 10, 5, 0, 5, None, 1, ctypes.byref(g), ctypes.byref(out), None, 0, None)
    assert rc == -1


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_no_gpu_means_loud_failure(lib):
    import lidar_vision_vqa_b200 as L

    assert lib.pillars_device_ok(-1) != 0
    vfe = L.PillarVFE(model_cfg=Cfg(USE_NORM=True, WITH_DISTANCE=False, USE_ABSLOTE_XYZ=True, NUM_FILTERS=[64]),
                      num_point_features=5, voxel_size=[0.2, 0.2, 8], point_cloud_range=[-1, -1, -1, 1, 1, 1]).eval()
    with pytest.raises(L.NativeLibraryError):
        vfe({"voxels": torch.zeros(3, 4, 5), "voxel_num_points": torch.ones(3), "voxel_coords": torch.zeros(3, 4)})
    sc = L.PointPillarScatter(model_cfg=Cfg(NUM_BEV_FEATURES=64), grid_size=[8, 8, 1])
    with pytest.raises(L.NativeLibraryError):
        sc({"pillar_features": torch.zeros(3, 64), "voxel_coords": torch.zeros(3, 4), "batch_size": 1})


@pytest.mark.parametrize("name", vfe_golden_names())
def test_state_dict_keys_and_shapes_match_reference(name):
    """Reference checkpoints load by key + shape (detectors/detector3d_template.py:330-359)."""
    import lidar_vision_vqa_b200 as L

    g = load_golden(name)
    cfg = Cfg(USE_NORM=bool(g["use_norm"]), WITH_DISTANCE=bool(g["with_distance"]), USE_ABSLOTE_XYZ=bool(g["use_abs"]),
              NUM_FILTERS=[int(v) for v in g["num_filters"]])
    for cls in (L.PillarVFE, L.PillarVFEFromPoints):
        m = cls(model_cfg=cfg, num_point_features=g["voxels"].shape[2], voxel_size=list(g["voxel_size"]),
                point_cloud_range=g["range"], grid_size=g["grid_size"], depth_downsample_factor=None)
        mine = {k: tuple(v.shape) for k, v in m.state_dict().items()}
        ref = {k: tuple(np.asarray(v).shape) for k, v in g["state_dict"].items()}
        assert mine == ref
        assert m.get_output_feature_dim() == int(g["num_filters"][-1])


def test_registries_and_scatter_contract():
    import lidar_vision_vqa_b200 as L

    assert L.VFE_REGISTRY["PillarVFE"] is L.PillarVFE
    assert L.MAP_TO_BEV_REGISTRY["PointPillarScatter"] is L.PointPillarScatter
    sc = L.PointPillarScatter(model_cfg=Cfg(NUM_BEV_FEATURES=64), grid_size=np.array([512, 512, 1]))
    assert (sc.nx, sc.ny, sc.nz, sc.num_bev_features) == (512, 512, 1, 64)
    with pytest.raises(AssertionError):
        L.PointPillarScatter(model_cfg=Cfg(NUM_BEV_FEATURES=64), grid_size=[8, 8, 2])  # pointpillar_scatter.py:12


def test_grid_size_rule_and_bn_fold():
    import lidar_vision_vqa_b200 as L
    from lidar_vision_vqa_b200 import ops

    g = L.GridSpec.from_range((-51.2, -51.2, -5.0, 51.2, 51.2, 3.0), (0.2, 0.2, 8.0), 32, 30000)
    assert g.grid_size == (512, 512, 1)
    g = L.GridSpec.from_range((0, -39.68, -3, 69.12, 39.68, 1), (0.16, 0.16, 4), 32, 16000)  # kitti pointpillar.yaml
    assert g.grid_size == (432, 496, 1)
    w = torch.randn(64, 11)
    gamma, beta, mean, var = torch.rand(64) + 0.5, torch.randn(64), torch.randn(64), torch.rand(64) + 0.5
    p = ops.fold_pfn(w, (gamma, beta, mean, var, 1e-3), None, c_point=5, use_absolute_xyz=True, with_distance=False,
                     voxel_size=(0.2, 0.2, 8.0), point_cloud_range=(-51.2, -51.2, -5, 51.2, 51.2, 3), device="cpu")
    x = torch.randn(7, 11)
    bn = torch.nn.BatchNorm1d(64, eps=1e-3)
    bn.weight.data, bn.bias.data, bn.running_mean, bn.running_var = gamma, beta, mean, var
    bn.eval()
    torch.testing.assert_close((x @ w.t()) * p.scale + p.shift, bn(x @ w.t()), rtol=1e-5, atol=1e-5)
    assert p.offset == (0.2 / 2 + -51.2, 0.2 / 2 + -51.2, 8.0 / 2 + -5)


@pytest.mark.parametrize("name", ["dyn_c5", "dyn_c5_2layer_zout", "dyn2d_c5_f32", "dyn_c4_dist_noabs"])
def test_dynamic_vfe_state_dict_contract(name):
    """DynPillarVFE / DynamicPillarVFESimple2D: constructor kwargs of dynamic_pillar_vfe.py:50,146, registry names of
    backbones_3d/vfe/__init__.py:9-18, reference state-dict keys load strictly, get_output_feature_dim."""
    import lidar_vision_vqa_b200 as L

    g = load_golden(name)
    reg = "DynamicPillarVFESimple2D" if bool(g["simple2d"]) else "DynPillarVFE"
    cls = L.VFE_REGISTRY[reg]
    cfg = Cfg(USE_NORM=True, WITH_DISTANCE=bool(g["with_distance"]), USE_ABSLOTE_XYZ=bool(g["use_abs"]),
              NUM_FILTERS=[int(v) for v in g["num_filters"]])
    vfe = cls(model_cfg=cfg, num_point_features=int(g["c"]), voxel_size=[float(v) for v in g["voxel_size"]],
              grid_size=g["grid_size"], point_cloud_range=g["range"], depth_downsample_factor=None)
    sd = {k: torch.from_numpy(v) for k, v in g["state_dict"].items()}
    vfe.load_state_dict(sd, strict=True)
    assert vfe.get_output_feature_dim() == int(g["num_filters"][-1])
    assert set(vfe.state_dict().keys()) == set(sd.keys())
    if not torch.cuda.is_available():
        with pytest.raises(L.NativeLibraryError):
            vfe.eval()({"points": torch.from_numpy(g["points_b"]), "batch_size": int(g["batch"])})


# ---- BEV tokeniser (VATLiDAR head, vat_lidar.py:63-121,206-253) -------------------------------------------------------------
def test_tokenizer_state_dict_contract_and_host_tables():
    """Parameter names/shapes are the reference's (so its checkpoints load), geometry tables equal the oracle's."""
    from lidar_vision_vqa_b200 import tokens as T
    from oracle import tokens_oracle as to

    tk = T.VATLiDARTokenizer(c_in=64, d_model=256)
    sd = to.random_token_params(64, 256, seed=0)
    assert {k: tuple(v.shape) for k, v in tk.state_dict().items()} == {k: tuple(v.shape) for k, v in sd.items()}
    res = tk.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()}, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    assert tk.norm_tokens.eps == to.LN_EPS
    for h, w in [(13, 9), (50, 50), (96, 64), (1, 7)]:
        geom, sid = T.grid_tables(h, w)
        g2, s2 = to.grid_geometry(h, w)
        np.testing.assert_array_equal(sid.numpy(), s2)
        np.testing.assert_allclose(geom.numpy(), g2, rtol=0, atol=1e-6)


def test_tokenizer_argument_errors(lib):
    from lidar_vision_vqa_b200 import _native

    t = _native.PillarsTokenizer()
    t.c_in, t.d_model = 64, 100  # d_model must be a multiple of 128
    assert lib.pillars_bev_tokens_map(None, None, 1, 8, 8, ctypes.byref(t), None, None, 0, None) == -3
    assert b"d_model" in lib.pillars_last_error()
    assert lib.pillars_bev_tokens_map(None, None, 1, 8, 8, None, None, None, 0, None) == -1
    a = lib.pillars_tokens_workspace_bytes(2, 64, 16, 16, 0)
    b = lib.pillars_tokens_workspace_bytes(2, 64, 16, 16, 1)
    assert 2 * 2 * 16 * 16 * 4 <= a < b and b >= a + 2 * 16 * 16 * 64 * 4
    g = _native.make_grid((-51.2, -51.2, -5, 51.2, 51.2, 3), (0.2, 0.2, 8), (512, 512, 1), 32, 30000)
    off = lib.pillars_workspace_cell_row_offset(100_000, 4, ctypes.byref(g))
    assert 0 < off and off + 4 * 4 * 512 * 512 <= lib.pillars_workspace_bytes(100_000, 4, ctypes.byref(g))


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_tokenizer_without_gpu_fails_loudly():
    import lidar_vision_vqa_b200 as L
    from lidar_vision_vqa_b200 import tokens as T

    tk = T.VATLiDARTokenizer(c_in=8, d_model=128).eval()
    with pytest.raises(L.NativeLibraryError):
        tk(torch.zeros(1, 8, 4, 4))
    with pytest.raises(L.NativeLibraryError):
        tk.forward_pillars(torch.zeros(2, 8), torch.zeros(2, 4), 1, (4, 4))


BACKBONE_CFGS = [
    dict(LAYER_NUMS=[3, 5, 5], LAYER_STRIDES=[2, 2, 2], NUM_FILTERS=[64, 128, 256], UPSAMPLE_STRIDES=[0.5, 1, 2],
         NUM_UPSAMPLE_FILTERS=[128, 128, 128]),                       # nuscenes_models/cbgs_pp_multihead.yaml:39-46
    dict(LAYER_NUMS=[3, 5, 5], LAYER_STRIDES=[2, 2, 2], NUM_FILTERS=[64, 128, 256], UPSAMPLE_STRIDES=[1, 2, 4],
         NUM_UPSAMPLE_FILTERS=[128, 128, 128]),                       # kitti_models/pointpillar.yaml
    dict(LAYER_NUMS=[2], LAYER_STRIDES=[1], NUM_FILTERS=[64], UPSAMPLE_STRIDES=[1], NUM_UPSAMPLE_FILTERS=[64],
         USE_CONV_FOR_NO_STRIDE=True),
]


@pytest.mark.parametrize("cfg", BACKBONE_CFGS, ids=["multihead", "kitti", "conv_for_no_stride"])
def test_backbone_mirrors_the_reference_module_tree(cfg):
    """Same constructor, same sub-module tree => the reference's checkpoints load by key and shape (f-3 boundary)."""
    from oracle import ref_loader as R
    from lidar_vision_vqa_b200 import BaseBEVBackbone

    if not R.reference_available():
        pytest.skip("reference tree / oracle/_ref copy not present")
    ref = R.load_bev_backbone()(R.AttrDict(cfg), 64)
    mine = BaseBEVBackbone(cfg, 64)
    a, b = ref.state_dict(), mine.state_dict()
    assert list(a.keys()) == list(b.keys())
    assert all(a[k].shape == b[k].shape for k in a)
    assert mine.num_bev_features == ref.num_bev_features
    mine.load_state_dict(a, strict=True)
    for m in mine.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            assert m.eps == 1e-3 and m.momentum == 0.01  # base_bev_backbone.py:36


def test_backbone_has_no_cpu_or_training_path():
    import lidar_vision_vqa_b200 as L

    m = L.BaseBEVBackbone(BACKBONE_CFGS[0], 64)
    with pytest.raises(NotImplementedError):
        m({"spatial_features": torch.zeros(1, 64, 32, 32)})
    with pytest.raises(L.NativeLibraryError):
        m.eval()({"spatial_features": torch.zeros(1, 64, 32, 32)})


def test_conv_weight_bytes_only_for_launchable_transposed_shapes(lib):
    """A ConvTranspose2d keeps its two dx phases side by side in one accumulator of 2 * c_out columns, and the kernel is
    instantiated up to 256: c_out = 256 must be refused by the size query, so that `prepare` raises NotImplementedError before
    it touches a device, instead of the launch failing later."""
    from lidar_vision_vqa_b200 import _native
    from lidar_vision_vqa_b200.backbone import _Layer

    def nbytes(c_in, c_out, up):
        cv = _native.PillarsConv(c_in, c_out, 1, 1, 0, up, 1, 0)
        return lib.pillars_conv_weight_bytes(ctypes.byref(cv))

    assert nbytes(256, 256, 2) == 0 and nbytes(256, 256, 4) == 0
    # [up * up phases][c_in / 32 channel blocks][c_out rows of 128 bytes]
    assert nbytes(256, 128, 2) == 4 * (256 // 32) * 128 * 128
    assert nbytes(128, 64, 4) == 16 * (128 // 32) * 64 * 128
    layer = _Layer(torch.nn.ConvTranspose2d(256, 256, 2, stride=2, bias=False), torch.nn.BatchNorm2d(256), True)
    with pytest.raises(NotImplementedError):
        layer.prepare(torch.device("cpu"))


def test_backbone_output_shape_and_flop_count_match_the_reference_module():
    """`output_shape` against the reference module's actual output, `bench.backbone_flops` against a count over its layers."""
    import importlib.util
    import os

    from oracle import ref_loader as R
    from lidar_vision_vqa_b200 import BaseBEVBackbone

    if not R.reference_available():
        pytest.skip("reference tree / oracle/_ref copy not present")
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(os.path.dirname(os.path.dirname(__file__)), "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    for cfg in BACKBONE_CFGS[:2]:
        ref = R.load_bev_backbone()(R.AttrDict(cfg), 64).eval()
        h, w, nb = 64, 48, 2
        flops = []

        def hook(mod, inp, out):
            if isinstance(mod, torch.nn.Conv2d):
                flops.append(2.0 * out.numel() * mod.in_channels * mod.kernel_size[0] * mod.kernel_size[1])
            else:  # ConvTranspose2d with kernel == stride: every input pixel feeds k*k outputs once
                flops.append(2.0 * inp[0].numel() // mod.in_channels * mod.in_channels * mod.out_channels
                             * mod.kernel_size[0] * mod.kernel_size[1])

        hs = [m.register_forward_hook(hook) for m in ref.modules() if isinstance(m, (torch.nn.Conv2d, torch.nn.ConvTranspose2d))]
        with torch.inference_mode():
            out = ref({"spatial_features": torch.zeros(nb, 64, h, w)})["spatial_features_2d"]
        for x in hs:
            x.remove()
        assert BaseBEVBackbone(cfg, 64).output_shape(h, w) == tuple(out.shape[1:])
        assert abs(bench.backbone_flops(cfg, 64, h, w, nb) - sum(flops)) <= 1e-6 * sum(flops)


def test_bench_side_measurements_are_guarded():
    """A failing optional section of bench.py (tokeniser, extractor, backbone, sub-lines) is recorded under its key and does
    not cost the run its main JSON line."""
    import importlib.util

    spec = importlib.util.spec_from_file_location("bench_mod2", os.path.join(os.path.dirname(os.path.dirname(__file__)), "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)

    def boom():
        raise ValueError("no such workload")

    assert bench.guarded("ok", lambda: {"value": 1}) == {"value": 1}
    got = bench.guarded("broken", boom)
    assert set(got) == {"error"} and "ValueError" in got["error"] and "no such workload" in got["error"]


def test_workspace_holds_the_second_layer_table(lib):
    """The two-layer streaming path folds layer 1 into the workspace (kFolded2Floats floats): the query must have grown by at
    least that over what the single-layer path needs of it, for every workload shape."""
    from lidar_vision_vqa_b200 import GridSpec
    import ctypes

    grid = GridSpec.from_range((-51.2, -51.2, -5.0, 51.2, 51.2, 3.0), (0.2, 0.2, 8.0), 32, 30000)
    g = grid.native()
    for n, nb in ((0, 1), (1000, 1), (503251, 16)):
        need = lib.pillars_workspace_bytes(n, nb, ctypes.byref(g))
        assert need >= 4 * (2 * 32 * 64 + 64)
        assert need % 16 == 0 or need > 0
