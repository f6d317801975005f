"""CPU tests of BaseBEVResBackbone's boundary: the module tree and state-dict keys of the reference's residual backbone
(against the restatement in oracle/bev_res_oracle.py and, where oracle/_ref holds it, the live class), the launch plan, the
refusals, and the fault codes of pillars_conv_forward_residual (all returned before anything touches a device)."""
import ctypes
import sys

import pytest
import torch

from oracle import bev_res_oracle as ro
from oracle import ref_loader as R

RES_CFGS = {
    "4level_s1222": dict(LAYER_NUMS=[1, 2, 2, 2], LAYER_STRIDES=[1, 2, 2, 2], NUM_FILTERS=[64, 128, 256, 256],
                         UPSAMPLE_STRIDES=[0.5, 1, 2, 4], NUM_UPSAMPLE_FILTERS=[128, 128, 128, 128]),
    "3level_s222_up124": dict(LAYER_NUMS=[2, 3, 3], LAYER_STRIDES=[2, 2, 2], NUM_FILTERS=[64, 128, 256],
                              UPSAMPLE_STRIDES=[1, 2, 4], NUM_UPSAMPLE_FILTERS=[128, 128, 128]),
    "1level_no_up": dict(LAYER_NUMS=[2], LAYER_STRIDES=[2], NUM_FILTERS=[128]),
}
E_BADARG, E_UNSUPPORTED = -1, -3


@pytest.mark.parametrize("name", sorted(RES_CFGS))
def test_module_tree_and_state_dict_match_the_restatement(name):
    from lidar_vision_vqa_b200 import BaseBEVResBackbone

    cfg = RES_CFGS[name]
    ref = ro.randomise(ro.BaseBEVResBackbone(cfg, 64), 1)
    mine = BaseBEVResBackbone(cfg, 64)
    a, b = ref.state_dict(), mine.state_dict()
    assert list(a) == list(b)
    assert all(a[k].shape == b[k].shape for k in a)
    assert mine.num_bev_features == ref.num_bev_features
    res = mine.load_state_dict(a, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    assert all(torch.equal(v, mine.state_dict()[k]) for k, v in a.items())
    for m in mine.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            assert m.eps == 1e-3 and m.momentum == 0.01
    assert "blocks.0.0.downsample_layer.0.weight" in b and "blocks.0.0.bn1.running_var" in b
    assert "blocks.0.1.downsample_layer.0.weight" not in b


@pytest.mark.parametrize("name", sorted(RES_CFGS))
def test_output_shape_matches_the_restatement(name):
    from lidar_vision_vqa_b200 import BaseBEVResBackbone

    cfg = RES_CFGS[name]
    ref = ro.BaseBEVResBackbone(cfg, 64).eval()
    for h, w in ((64, 48), (128, 80)):
        with torch.inference_mode():
            out = ref({"spatial_features": torch.zeros(1, 64, h, w)})["spatial_features_2d"]
        assert BaseBEVResBackbone(cfg, 64).output_shape(h, w) == tuple(out.shape[1:])


def test_launch_plan_projection_first_block_only_and_no_relu_on_it():
    from lidar_vision_vqa_b200 import BaseBEVResBackbone

    m = BaseBEVResBackbone(RES_CFGS["3level_s222_up124"], 64)
    m._build_plan()
    levels, de = m._plan
    assert [len(steps) for steps in levels] == [3, 4, 4]
    for steps in levels:
        assert steps[0].proj is not None and all(st.proj is None for st in steps[1:])
        assert steps[0].proj.desc == dict(c_in=steps[0].conv1.desc["c_in"], c_out=steps[0].conv1.desc["c_out"], k=1, stride=2,
                                          pad=0, up=1)
        assert not steps[0].proj.relu and all(st.conv1.relu and st.conv2.relu for st in steps)
        assert steps[0].proj.native(False).relu == 0 and steps[0].conv2.native(True).relu == 1
    assert [d.desc["up"] for d in de] == [1, 2, 4]  # stride 1 is a ConvTranspose2d in the residual class, always
    assert len(m._layers()) == sum(2 * len(s) + 1 for s in levels) + len(de)


def test_training_mode_and_cpu_input_raise():
    import lidar_vision_vqa_b200 as L

    m = L.BaseBEVResBackbone(RES_CFGS["1level_no_up"], 64)
    with pytest.raises(NotImplementedError):
        m({"spatial_features": torch.zeros(1, 64, 32, 32)})
    with pytest.raises(L.NativeLibraryError):
        m.eval()({"spatial_features": torch.zeros(1, 64, 32, 32)})


def test_shapes_outside_the_set_raise_at_prepare():
    from lidar_vision_vqa_b200 import BaseBEVResBackbone

    m = BaseBEVResBackbone(dict(LAYER_NUMS=[1], LAYER_STRIDES=[2], NUM_FILTERS=[96]), 64)
    m._build_plan()
    with pytest.raises(NotImplementedError):
        m._plan[0][0][0].proj.prepare(torch.device("cpu"))
    with pytest.raises(NotImplementedError):
        BaseBEVResBackbone(dict(LAYER_NUMS=[1, 1], LAYER_STRIDES=[1, 2], NUM_FILTERS=[64, 64]), 64).output_shape(32, 32)


@pytest.fixture(scope="module")
def lib():
    from lidar_vision_vqa_b200 import _native

    return _native.load()


def test_projection_geometry_is_accepted(lib):
    from lidar_vision_vqa_b200 import _native

    def nbytes(c_in, c_out, k, stride, pad):
        return lib.pillars_conv_weight_bytes(ctypes.byref(_native.PillarsConv(c_in, c_out, k, stride, pad, 1, 0, 0)))

    assert nbytes(64, 128, 1, 2, 0) == (64 // 32) * 128 * 128
    assert nbytes(128, 256, 1, 2, 0) == (128 // 32) * 256 * 128
    assert nbytes(64, 128, 1, 2, 1) == 0 and nbytes(64, 128, 3, 2, 0) == 0


def test_residual_entry_fault_codes(lib):
    from lidar_vision_vqa_b200 import _native

    buf = ctypes.create_string_buffer(4096 + 64)
    base = (ctypes.addressof(buf) + 63) & ~63  # (host memory: every case below fails before any device access)
    img, shift, x, out, res = base, base + 1024, base + 2048, base + 3072, base + 3584

    def call(cv, image=img, out_nchw=0, residual=res):
        return lib.pillars_conv_forward_residual(ctypes.byref(cv), image, shift, x, None, None, 1, 8, 8, out, cv.c_out, 0,
                                                 out_nchw, residual, None, None)

    plain = _native.PillarsConv(64, 64, 3, 1, 1, 1, 1, 1)
    assert call(_native.PillarsConv(64, 64, 1, 1, 0, 2, 1, 0)) == E_UNSUPPORTED  # transposed (up > 1)
    assert call(plain, out_nchw=1) == E_UNSUPPORTED
    assert call(plain, image=None) == E_BADARG
    assert call(plain, residual=res + 4) == E_BADARG  # misaligned residual
    assert call(plain, residual=None) == E_BADARG
    assert b"residual" in lib.pillars_last_error()
    assert call(_native.PillarsConv(64, 96, 3, 1, 1, 1, 1, 0)) == E_UNSUPPORTED


@pytest.mark.skipif(not R.reference_available(), reason="reference tree / oracle/_ref copy not present")
@pytest.mark.parametrize("name", sorted(RES_CFGS))
def test_restatement_matches_the_live_reference_class(name):
    """Keys, and fp32 CPU outputs bit for bit, of the restatement and the reference's own BaseBEVResBackbone."""
    R.load_bev_backbone()
    live = getattr(sys.modules["_ref_pcdet.base_bev_backbone"], "BaseBEVResBackbone", None)
    if live is None:
        pytest.skip("the reference's base_bev_backbone.py defines no BaseBEVResBackbone")
    cfg = RES_CFGS[name]
    torch.manual_seed(0)
    ref = ro.randomise(live(R.AttrDict(cfg), 64), 2).eval()
    mine = ro.BaseBEVResBackbone(R.AttrDict(cfg), 64).eval()
    assert list(ref.state_dict()) == list(mine.state_dict())
    mine.load_state_dict(ref.state_dict(), strict=True)
    assert mine.num_bev_features == ref.num_bev_features
    g = torch.Generator().manual_seed(3)
    canvas = torch.rand((2, 64, 48, 40), generator=g) * (torch.rand((2, 1, 48, 40), generator=g) < 0.1)
    with torch.inference_mode():
        a = ref({"spatial_features": canvas.clone()})["spatial_features_2d"]
        b = mine({"spatial_features": canvas.clone()})["spatial_features_2d"]
    assert torch.equal(a, b)
