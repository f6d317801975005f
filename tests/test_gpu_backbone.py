"""GPU parity of the BEV backbone row (SURVEY 8 f-3): the tcgen05 convolution kernel through the C ABI.

Two kinds of checks:
  * single layers on inputs whose values are exactly representable in tf32 (small integers): the tensor core's products and the
    fp32 accumulation are then exact, so every geometry (taps, stride, halo, parity planes, gathered input, transposed phases,
    NHWC / NCHW channel windows, ragged image borders) must match a float64 convolution BIT FOR BIT;
  * the whole `BaseBEVBackbone` against the reference's own module (oracle/_ref copy, CPU fp32) with random weights.  The kernel
    multiplies in tf32 -- as the reference's nn.Conv2d itself does on this GPU under PyTorch's default
    `torch.backends.cudnn.allow_tf32 = True` -- so the tolerance is stated against the output's scale:
    |err| <= 4e-3 * max|ref| over the 11 / 16 stacked layers (measured: 1.0e-3 at 16 x 512^2, where the reference's own TF32
    run deviates from its fp32 run by 0.8e-3: bench.py `backbone`).
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _dev():
    return torch.device("cuda:0")


def _int_tensor(shape, lo, hi, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(lo, hi + 1, shape, generator=g).to(torch.float32)


class _FakeBN:
    def __init__(self, c, shift):
        self.weight = torch.ones(c)
        self.bias = shift.clone()
        self.running_mean = torch.zeros(c)
        self.running_var = torch.ones(c) - 1e-3
        self.eps = 1e-3


def _run_layer(conv, shift, x_nchw, *, gather=False, out_nchw=False, c_total=None, c_off=0):
    from lidar_vision_vqa_b200 import backbone as B

    dev = _dev()
    transposed = isinstance(conv, torch.nn.ConvTranspose2d)
    layer = B._Layer(conv, _FakeBN(shift.numel(), shift), transposed)
    layer.prepare(dev)
    nb, c, h, w = x_nchw.shape
    d = layer.desc
    oh, ow = B.BaseBEVBackbone._out_hw(h, w, d)
    c_total = c_total or d["c_out"]
    if out_nchw:
        out = torch.full((nb, c_total, oh, ow), -7.0, device=dev)
    else:
        out = torch.full((nb, oh, ow, c_total), -7.0, device=dev)
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    if gather:
        occupied = (x_nchw != 0).any(dim=1)  # [nb, h, w]
        idx = torch.full((nb, h, w), -1, dtype=torch.int32)
        pos = occupied.nonzero()
        perm = torch.randperm(len(pos), generator=torch.Generator().manual_seed(5))
        rows = torch.empty((max(len(pos), 1), c))
        for r, k in enumerate(perm.tolist()):
            b, y, x = pos[k].tolist()
            idx[b, y, x] = r
            rows[r] = x_nchw[b, :, y, x]
        B.conv_forward(layer, out, c_total, c_off, out_nchw, nb, h, w, rows=rows.to(dev), cell_row=idx.to(dev), round_out=False,
                       error=err)
    else:
        x = x_nchw.permute(0, 2, 3, 1).contiguous().to(dev)
        B.conv_forward(layer, out, c_total, c_off, out_nchw, nb, h, w, x_nhwc=x, round_out=False, error=err)
    torch.cuda.synchronize()
    assert int(err.item()) == 0, hex(int(err.item()))
    return out.cpu(), d


def _reference_layer(conv, shift, x_nchw):
    with torch.no_grad():
        if isinstance(conv, torch.nn.ConvTranspose2d):
            y = F.conv_transpose2d(x_nchw.double(), conv.weight.double(), stride=conv.stride)
        else:
            pad = 1 if conv.kernel_size[0] == 3 else 0
            y = F.conv2d(x_nchw.double(), conv.weight.double(), stride=conv.stride, padding=pad)
        # eval BatchNorm with weight 1, mean 0, var + eps = 1: y + shift
        return torch.relu(y + shift.double().view(1, -1, 1, 1)).float()


LAYER_CASES = [
    # (c_in, c_out, k, stride, transposed, h, w, frames)
    (64, 64, 3, 1, False, 64, 16, 2),     # four stacked patches per CTA
    (64, 64, 3, 1, False, 40, 20, 1),     # ragged: image not a multiple of the patch in either direction
    (128, 128, 3, 1, False, 32, 24, 1),
    (256, 256, 3, 1, False, 32, 8, 1),
    (64, 128, 3, 2, False, 64, 32, 1),    # stride 2: parity planes
    (128, 256, 3, 2, False, 34, 18, 1),   # stride 2, ragged
    (64, 64, 3, 2, False, 64, 48, 2),
    (64, 128, 2, 2, False, 32, 32, 1),    # UPSAMPLE_STRIDES 0.5: Conv2d kernel 2 stride 2
    (128, 128, 1, 1, False, 16, 16, 1),   # 1x1
    (128, 128, 1, 1, True, 16, 24, 1),    # ConvTranspose2d kernel 1 stride 1 ([in, out] weights)
    (256, 128, 2, 2, True, 16, 8, 1),     # ConvTranspose2d kernel 2 stride 2: four phases
    (256, 128, 4, 4, True, 16, 8, 1),     # kernel 4 stride 4: sixteen phases
]


@pytest.mark.parametrize("case", LAYER_CASES, ids=lambda c: "x".join(map(str, c)))
def test_conv_layer_exact_on_tf32_representable_values(case):
    c_in, c_out, k, stride, transposed, h, w, nb = case
    if transposed:
        conv = torch.nn.ConvTranspose2d(c_in, c_out, k, stride=stride, bias=False)
    else:
        conv = torch.nn.Conv2d(c_in, c_out, k, stride=stride, padding=0, bias=False)
    with torch.no_grad():
        conv.weight.copy_(_int_tensor(tuple(conv.weight.shape), -3, 3, 11))
    shift = _int_tensor((c_out,), -40, 40, 12)
    x = _int_tensor((nb, c_in, h, w), -4, 4, 13)
    ref = _reference_layer(conv, shift, x)
    got, _ = _run_layer(conv, shift, x)
    assert got.shape == ref.permute(0, 2, 3, 1).shape
    assert torch.equal(got, ref.permute(0, 2, 3, 1).contiguous())


def test_conv_layer_nchw_channel_window_and_untouched_neighbours():
    conv = torch.nn.ConvTranspose2d(256, 128, 2, stride=2, bias=False)
    with torch.no_grad():
        conv.weight.copy_(_int_tensor(tuple(conv.weight.shape), -3, 3, 21))
    shift = _int_tensor((128,), -40, 40, 22)
    x = _int_tensor((2, 256, 16, 16), -4, 4, 23)
    ref = _reference_layer(conv, shift, x)
    got, _ = _run_layer(conv, shift, x, out_nchw=True, c_total=384, c_off=128)
    assert torch.equal(got[:, 128:256], ref)
    assert bool((got[:, :128] == -7.0).all()) and bool((got[:, 256:] == -7.0).all())


@pytest.mark.parametrize("stride,c_out", [(2, 64), (1, 64), (1, 128), (2, 128)])
def test_first_layer_gathers_from_pillar_rows(stride, c_out):
    """Input given as (pillar rows, BEV index map): 5 % of the cells occupied, rows in random order; several tile sets per CTA
    would need > 148 tiles, so the image is tall: the sparse loader's un-write of the previous tile set is exercised."""
    conv = torch.nn.Conv2d(64, c_out, 3, stride=stride, padding=0, bias=False)
    with torch.no_grad():
        conv.weight.copy_(_int_tensor(tuple(conv.weight.shape), -3, 3, 31))
    shift = _int_tensor((c_out,), -40, 40, 32)
    x = _int_tensor((6, 64, 320, 72), -4, 4, 33)
    g = torch.Generator().manual_seed(34)
    keep = (torch.rand((6, 1, 320, 72), generator=g) < 0.05).float()
    x = x * keep
    ref = _reference_layer(conv, shift, x)
    got, _ = _run_layer(conv, shift, x, gather=True)
    assert torch.equal(got, ref.permute(0, 2, 3, 1).contiguous())


def _randomise_bn(model, seed):
    g = torch.Generator().manual_seed(seed)
    for m in model.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            with torch.no_grad():
                m.weight.copy_(0.5 + torch.rand(m.weight.shape, generator=g))
                m.bias.copy_(0.2 * torch.randn(m.bias.shape, generator=g))
                m.running_mean.copy_(0.2 * torch.randn(m.bias.shape, generator=g))
                m.running_var.copy_(0.5 + 1.5 * torch.rand(m.bias.shape, generator=g))


BACKBONE_CASES = {
    # cbgs_pp_multihead.yaml:41-46 (the product's pillar config), layer counts as in the file
    "nuscenes_multihead": dict(LAYER_NUMS=[3, 5, 5], LAYER_STRIDES=[2, 2, 2], NUM_FILTERS=[64, 128, 256],
                               UPSAMPLE_STRIDES=[0.5, 1, 2], NUM_UPSAMPLE_FILTERS=[128, 128, 128]),
    # first block without down-sampling, plain convolutions in the branches (USE_CONV_FOR_NO_STRIDE)
    "stride1_first": dict(LAYER_NUMS=[1, 1], LAYER_STRIDES=[1, 2], NUM_FILTERS=[64, 128], UPSAMPLE_STRIDES=[1, 2],
                          NUM_UPSAMPLE_FILTERS=[64, 64], USE_CONV_FOR_NO_STRIDE=True),
    # kitti pointpillar.yaml: strides [2,2,2] / up-sampling [1,2,4]
    "kitti_pointpillar": dict(LAYER_NUMS=[3, 5, 5], LAYER_STRIDES=[2, 2, 2], NUM_FILTERS=[64, 128, 256],
                              UPSAMPLE_STRIDES=[1, 2, 4], NUM_UPSAMPLE_FILTERS=[128, 128, 128]),
}


@pytest.mark.parametrize("name", sorted(BACKBONE_CASES))
@pytest.mark.parametrize("fused_input", [False, True], ids=["canvas", "rows+map"])
def test_backbone_matches_reference_module(name, fused_input):
    from oracle import ref_loader as R
    from lidar_vision_vqa_b200.backbone import BaseBEVBackbone

    if not R.reference_available():
        pytest.skip("reference copy (oracle/_ref) not present")
    cfg = BACKBONE_CASES[name]
    ref = R.load_bev_backbone()(R.AttrDict(cfg), 64).eval()
    _randomise_bn(ref, 3)
    mine = BaseBEVBackbone(cfg, 64).eval()
    missing = mine.load_state_dict(ref.state_dict(), strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    assert mine.num_bev_features == ref.num_bev_features

    # a pillar-like canvas: 6 % occupied cells, 64 non-negative channels (PFN outputs are post-ReLU maxima)
    g = torch.Generator().manual_seed(7)
    nb, h, w = 2, 128, 96
    occupied = torch.rand((nb, 1, h, w), generator=g) < 0.06
    canvas = torch.rand((nb, 64, h, w), generator=g) * occupied
    with torch.inference_mode():
        want = ref({"spatial_features": canvas.clone()})["spatial_features_2d"]
    dev = _dev()
    mine = mine.to(dev)
    if fused_input:
        pos = occupied[:, 0].nonzero()
        idx = torch.full((nb, h, w), -1, dtype=torch.int32)
        idx[pos[:, 0], pos[:, 1], pos[:, 2]] = torch.arange(len(pos), dtype=torch.int32)
        rows = canvas.permute(0, 2, 3, 1)[pos[:, 0], pos[:, 1], pos[:, 2]].contiguous()
        d = {"pillar_features": rows.to(dev), "bev_index_map": idx.to(dev)}
    else:
        d = {"spatial_features": canvas.to(dev)}
    with torch.inference_mode():
        out = mine(d)
    torch.cuda.synchronize()
    assert int(out["_conv_error_word"].item()) == 0
    got = out["spatial_features_2d"].cpu()
    assert got.shape == want.shape
    scale = float(want.abs().max())
    err = float((got - want).abs().max())
    assert err <= 4e-3 * scale, (err, scale)
    # and not merely small on average: the bulk of the elements agree to tf32 accuracy
    assert float(((got - want).abs() <= 2e-3 * scale).float().mean()) > 0.99


def test_backbone_refuses_training_mode_and_cpu_input():
    from lidar_vision_vqa_b200 import _native
    from lidar_vision_vqa_b200.backbone import BaseBEVBackbone

    m = BaseBEVBackbone(BACKBONE_CASES["kitti_pointpillar"], 64)
    with pytest.raises(NotImplementedError):
        m({"spatial_features": torch.zeros(1, 64, 32, 32, device=_dev())})
    with pytest.raises(_native.NativeLibraryError):
        m.eval()({"spatial_features": torch.zeros(1, 64, 32, 32)})


def test_points_to_backbone_without_a_canvas_equals_the_canvas_route():
    """points -> PillarVFEFromPoints(EMIT_INDEX_MAP) -> BaseBEVBackbone reads pillar rows through the index map; the same
    sweeps through FUSE_SCATTER's dense canvas must give the identical tensor (same operands, same order of accumulation)."""
    from lidar_vision_vqa_b200 import synth
    from lidar_vision_vqa_b200.backbone import BaseBEVBackbone
    from lidar_vision_vqa_b200.modules import PillarVFEFromPoints

    dev = _dev()
    rng, vs = [-51.2, -51.2, -5.0, 51.2, 51.2, 3.0], [0.2, 0.2, 8.0]
    pts, offs = synth.make_batch(2, synth.NUSCENES_32, 5, seed0=3)
    b = np.repeat(np.arange(2), np.diff(offs)).astype(np.float32)[:, None]
    points = torch.from_numpy(np.concatenate([b, pts], axis=1)).to(dev)
    base = dict(USE_NORM=True, WITH_DISTANCE=False, USE_ABSLOTE_XYZ=True, NUM_FILTERS=[64], MAX_POINTS_PER_VOXEL=32,
                MAX_NUMBER_OF_VOXELS=30000)
    torch.manual_seed(0)
    vfe_map = PillarVFEFromPoints(dict(base, EMIT_INDEX_MAP=True), 5, vs, rng, [512, 512, 1]).eval().to(dev)
    vfe_canvas = PillarVFEFromPoints(dict(base, FUSE_SCATTER=True), 5, vs, rng, [512, 512, 1]).eval().to(dev)
    vfe_canvas.load_state_dict(vfe_map.state_dict())
    bb = BaseBEVBackbone(BACKBONE_CASES["nuscenes_multihead"], 64).eval().to(dev)
    _randomise_bn(bb, 9)
    with torch.inference_mode():
        d1 = vfe_map({"points": points, "batch_size": 2})
        assert "spatial_features" not in d1 and d1["bev_index_map"].shape == (2, 512, 512)
        m = d1["pillar_features"].shape[0]
        assert int((d1["bev_index_map"] >= 0).sum()) == m
        out1 = bb(d1)["spatial_features_2d"].clone()
        d2 = vfe_canvas({"points": points, "batch_size": 2})
        out2 = bb({"spatial_features": d2["spatial_features"]})["spatial_features_2d"]
    torch.cuda.synchronize()
    assert out1.shape == (2, 384, 128, 128)
    assert torch.equal(out1, out2)


@pytest.mark.parametrize("name", ["bb_2level_half_stride", "bb_3level_up124"])
def test_backbone_against_committed_reference_goldens(name):
    """tests/golden/bb_*.npz: config, state dict, canvas and the output of the reference's own BaseBEVBackbone.forward
    (made by tests/golden/make_golden_backbone.py).  A compact file holds the seed of the state dict and canvas instead: they
    are rebuilt here and must hash to what the reference module was run on, in the reference's state-dict key order."""
    import json
    import os

    from lidar_vision_vqa_b200.backbone import BaseBEVBackbone
    from oracle import pillar_oracle as po

    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name + ".npz"))
    cfg = json.loads(bytes(z["cfg"]).decode())
    if "gen.seed" in z.files:
        torch.manual_seed(int(z["gen.seed"]))
        m = BaseBEVBackbone(cfg, 64).eval()
        sd, canvas, sha = po.golden_backbone_inputs(m, int(z["gen.seed"]), *(int(v) for v in z["gen.shape"]))
        assert list(sd.keys()) == json.loads(bytes(z["sd_keys"]).decode())
        assert np.array_equal(sha, z["gen.sha256"]), "regenerated state dict / canvas differ from the reference's inputs"
    else:
        m = BaseBEVBackbone(cfg, 64).eval()
        sd = {k[3:]: torch.from_numpy(z[k].astype(np.float32) if z[k].dtype == np.float16 else z[k]) for k in z.files
              if k.startswith("sd.")}
        canvas = torch.from_numpy(z["canvas"].astype(np.float32))
    m.load_state_dict(sd, strict=True)
    assert m.num_bev_features == z["out"].shape[1]
    dev = _dev()
    m = m.to(dev)
    canvas = canvas.to(dev)
    with torch.inference_mode():
        out = m({"spatial_features": canvas})
    torch.cuda.synchronize()
    assert int(out["_conv_error_word"].item()) == 0
    got, want = out["spatial_features_2d"].cpu().numpy(), z["out"]
    assert got.shape == want.shape
    scale = float(np.abs(want).max())
    assert float(np.abs(got - want).max()) <= 4e-3 * scale
    assert float((np.abs(got - want) <= 2e-3 * scale).mean()) > 0.99


def test_extractor_ships_spatial_features_2d():
    """BevExtractor(ship='features2d'): per-token float16 [384, H/4, W/4] maps == float16 of BaseBEVBackbone run on the canvas of
    the same frame alone (frames are independent: batching and pipelining change nothing)."""
    from lidar_vision_vqa_b200 import synth
    from lidar_vision_vqa_b200.backbone import BaseBEVBackbone
    from lidar_vision_vqa_b200.extract import BevExtractor
    from lidar_vision_vqa_b200.modules import PillarVFEFromPoints

    dev = _dev()
    rng, vs = [-25.6, -25.6, -5.0, 25.6, 25.6, 3.0], [0.2, 0.2, 8.0]
    frames = [synth.make_sweep(700 + i, synth.NUSCENES_32, 5)[:7000 + 300 * i] for i in range(5)]
    base = dict(USE_NORM=True, WITH_DISTANCE=False, USE_ABSLOTE_XYZ=True, NUM_FILTERS=[64], MAX_POINTS_PER_VOXEL=32,
                MAX_NUMBER_OF_VOXELS=20000)
    torch.manual_seed(1)
    vfe = PillarVFEFromPoints(dict(base), 5, vs, rng, [256, 256, 1]).eval().to(dev)
    vfe_c = PillarVFEFromPoints(dict(base, FUSE_SCATTER=True), 5, vs, rng, [256, 256, 1]).eval().to(dev)
    vfe_c.load_state_dict(vfe.state_dict())
    bb = BaseBEVBackbone(BACKBONE_CASES["nuscenes_multihead"], 64).eval().to(dev)
    _randomise_bn(bb, 4)
    ex = BevExtractor(vfe, batch_size=2, max_points_per_frame=9000, depth=2, ship="features2d", backbone=bb)
    items = [(f"t{i}", f) for i, f in enumerate(frames)]
    got = {tok: np.array(arr) for tok, arr in ex.run(items)}
    assert list(got) == [t for t, _ in items]
    for tok, f in items:
        pts = torch.from_numpy(np.concatenate([np.zeros((len(f), 1), np.float32), f], axis=1)).to(dev)
        with torch.inference_mode():
            canvas = vfe_c({"points": pts, "batch_size": 1})["spatial_features"]
            want = bb({"spatial_features": canvas})["spatial_features_2d"][0].to(torch.float16).cpu().numpy()
        assert got[tok].dtype == np.float16 and got[tok].shape == (384, 64, 64)
        np.testing.assert_array_equal(got[tok].view(np.uint16), want.view(np.uint16))


@pytest.mark.parametrize("case", [(128, 128, 1, 1, 12, 64), (256, 128, 2, 2, 10, 40), (256, 128, 4, 4, 6, 33), (128, 64, 1, 1, 5, 96)],
                         ids=lambda c: "x".join(map(str, c)))
def test_wide_images_writing_nchw(case):
    """1x1 / transposed layers writing an NCHW channel window on images wider than a few patches, ragged widths included."""
    c_in, c_out, k, stride, h, w = case
    conv = torch.nn.ConvTranspose2d(c_in, c_out, k, stride=stride, bias=False)
    with torch.no_grad():
        conv.weight.copy_(_int_tensor(tuple(conv.weight.shape), -3, 3, 41))
    shift = _int_tensor((c_out,), -40, 40, 42)
    x = _int_tensor((2, c_in, h, w), -4, 4, 43)
    ref = _reference_layer(conv, shift, x)
    got, _ = _run_layer(conv, shift, x, out_nchw=True, c_total=c_out + 64, c_off=32)
    assert torch.equal(got[:, 32:32 + c_out], ref)
    assert bool((got[:, :32] == -7.0).all()) and bool((got[:, 32 + c_out:] == -7.0).all())
