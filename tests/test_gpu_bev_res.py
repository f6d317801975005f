"""GPU tests of BaseBEVResBackbone (the residual variant of f-3) and of what it adds to the tcgen05 convolution kernel: the
residual epilogue (y = relu(acc + shift + residual), pillars_conv_forward_residual), the 1x1 stride-2 projection and
BatchNorm without ReLU.

  * single launches on tf32-representable values (small integers, integer residuals): products, fp32 sums and the residual
    addition are exact, so every case must equal a float64 computation BIT FOR BIT -- with and without ReLU, with and
    without tf32-rounded output, every residual instantiation, ragged images, NHWC and gathered input, several frames;
  * the whole module against the torch restatement (oracle/bev_res_oracle.py, fp32 on the same GPU with TF32 off) on
    canvases of synthetic sweeps, at the f-3 bar: max error <= 4e-3 * max|ref|, 99 % of elements within 2e-3 * max|ref|.
    Measured on a B200 (2 frames, 256^2 grid; max |err| / max|ref|, share within 2e-3 * max|ref|): 4level_s1222 9.1e-4 / 1.0,
    3level_s222_up124 1.3e-3 / 1.0, 1level_no_up 1.1e-3 / 1.0; full size (16 x 512^2, frame 0, 4level_s1222) 9.4e-4 / 1.0.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import bev_res_oracle as ro

RES_CFGS = {
    "4level_s1222": dict(LAYER_NUMS=[1, 2, 2, 2], LAYER_STRIDES=[1, 2, 2, 2], NUM_FILTERS=[64, 128, 256, 256],
                         UPSAMPLE_STRIDES=[0.5, 1, 2, 4], NUM_UPSAMPLE_FILTERS=[128, 128, 128, 128]),
    "3level_s222_up124": dict(LAYER_NUMS=[2, 3, 3], LAYER_STRIDES=[2, 2, 2], NUM_FILTERS=[64, 128, 256],
                              UPSAMPLE_STRIDES=[1, 2, 4], NUM_UPSAMPLE_FILTERS=[128, 128, 128]),
    "1level_no_up": dict(LAYER_NUMS=[2], LAYER_STRIDES=[2], NUM_FILTERS=[128]),
}


def _dev():
    return torch.device("cuda:0")


def _ints(shape, lo, hi, seed, dev=None):
    g = torch.Generator(dev or "cpu").manual_seed(seed)
    return torch.randint(lo, hi + 1, shape, generator=g, device=dev).to(torch.float32)


def _rna_tf32(t):
    """cvt.rna.tf32.f32: keep 10 mantissa bits, round half away from zero."""
    return ((t.contiguous().view(torch.int32) + 0x1000) & -0x2000).view(torch.float32)


class _FakeBN:  # weight 1, mean 0, var + eps = 1: the BatchNorm is exactly "+ shift"
    def __init__(self, shift):
        c = shift.numel()
        self.weight, self.bias, self.running_mean, self.running_var, self.eps = torch.ones(c), shift.clone(), torch.zeros(c), \
            torch.ones(c) - 1e-3, 1e-3


def _gathered(x):
    """(rows in random order, index map with -1 for empty cells) of an NCHW tensor's non-zero cells."""
    nb, c, h, w = x.shape
    pos = (x != 0).any(dim=1).nonzero()
    pos = pos[torch.randperm(len(pos), generator=torch.Generator().manual_seed(5)).to(x.device)]
    idx = torch.full((nb, h, w), -1, dtype=torch.int32, device=x.device)
    idx[pos[:, 0], pos[:, 1], pos[:, 2]] = torch.arange(len(pos), dtype=torch.int32, device=x.device)
    rows = x.permute(0, 2, 3, 1)[pos[:, 0], pos[:, 1], pos[:, 2]].contiguous()
    return (rows if len(pos) else torch.zeros((1, c), device=x.device)), idx


# (c_in, c_out, k, stride, h, w, frames, gathered): every residual instantiation (stride, N, T) of launch_conv_umma --
# (1, 64, 4) (1, 64, 2) (1, 64, 1) (1, 128, 2) (1, 128, 1) (1, 256, 1) (2, 64, 1) (2, 128, 1) (2, 256, 1) -- and the projection
RES_CASES = [
    (64, 64, 3, 1, 67, 43, 3, False),     # four stacked patches, two MMA warps; ragged (67 = 4 * 16 + 3, 43 = 5 * 8 + 3)
    (64, 64, 3, 1, 29, 21, 2, False),     # two patches
    (64, 64, 3, 1, 13, 517, 2, True),     # one patch, gathered, wide
    (128, 128, 3, 1, 31, 19, 3, False),   # N 128, two patches
    (128, 128, 3, 1, 15, 33, 2, False),
    (256, 256, 3, 1, 17, 9, 2, False),
    (64, 64, 3, 2, 33, 31, 2, True),      # stride 2, gathered
    (64, 128, 3, 2, 45, 27, 2, False),
    (128, 256, 3, 2, 35, 23, 2, False),   # stride 2, N 256: one halo stage
    (64, 128, 1, 2, 61, 45, 3, False),    # the projection, 64 -> 128
    (128, 256, 1, 2, 33, 39, 2, False),   # the projection, 128 -> 256
    (64, 128, 1, 2, 71, 53, 2, True),     # the projection from pillar rows (level 0 of a stride-2 backbone)
    (64, 64, 1, 1, 40, 24, 2, True),      # the stride-1 projection from pillar rows (level 0 of a stride-1 backbone)
]


def _case_id(c):
    return "x".join(map(str, c[:6])) + f"_nb{c[6]}" + ("_rows" if c[7] else "")


def _run(c, relu, round_out, residual):
    from lidar_vision_vqa_b200 import backbone as B

    c_in, c_out, k, stride, h, w, nb, gathered = c
    dev = _dev()
    conv = torch.nn.Conv2d(c_in, c_out, k, stride=stride, padding=0, bias=False)
    with torch.no_grad():
        conv.weight.copy_(_ints(tuple(conv.weight.shape), -3, 3, 11))
    shift = _ints((c_out,), -40, 40, 12)
    x = _ints((nb, c_in, h, w), -4, 4, 13, dev)
    if gathered:
        x = x * (torch.rand((nb, 1, h, w), generator=torch.Generator(dev).manual_seed(14), device=dev) < 0.3)
    layer = B._Layer(conv, _FakeBN(shift), False, relu=relu)
    layer.prepare(dev)
    pad = 1 if k == 3 else 0
    oh, ow = (h + 2 * pad - k) // stride + 1, (w + 2 * pad - k) // stride + 1
    # integer residuals up to 3000: sums reach past 2048, where tf32's spacing exceeds 1 (the rounding matters, with ties)
    r = _ints((nb, oh, ow, c_out), -3000, 3000, 15, dev) if residual else None
    out = torch.full((nb, oh, ow, c_out), -7.0, device=dev)
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    if gathered:
        rows, idx = _gathered(x)
        B.conv_forward(layer, out, c_out, 0, False, nb, h, w, rows=rows, cell_row=idx, round_out=round_out, error=err,
                       residual=r)
    else:
        B.conv_forward(layer, out, c_out, 0, False, nb, h, w, x_nhwc=x.permute(0, 2, 3, 1).contiguous(), round_out=round_out,
                       error=err, residual=r)
    torch.cuda.synchronize()
    assert int(err.item()) == 0
    with torch.no_grad(), torch.backends.cudnn.flags(enabled=False):
        y = F.conv2d(x.double(), conv.weight.detach().to(dev, torch.float64), stride=stride, padding=pad)
        y = y + shift.to(dev, torch.float64).view(1, -1, 1, 1)
        if residual:
            y = y + r.permute(0, 3, 1, 2).double()
        if relu:
            y = torch.relu(y)
        y0 = y.float()
    ref = _rna_tf32(y0) if round_out else y0
    return out.permute(0, 3, 1, 2), ref, y0


@pytest.mark.gpu
@pytest.mark.parametrize("case", RES_CASES, ids=_case_id)
@pytest.mark.parametrize("relu,round_out", [(True, True), (True, False), (False, True), (False, False)],
                         ids=["relu_round", "relu", "round", "plain"])
def test_residual_epilogue_exact(case, relu, round_out):
    got, ref, ref0 = _run(case, relu, round_out, residual=True)
    if round_out:
        assert bool((ref != ref0).any()) and bool(((ref0.view(torch.int32) & 0x1FFF) == 0x1000).any())
    if not relu:
        assert bool((ref < 0).any())
    assert torch.equal(got, ref), f"{int((got != ref).sum())} of {ref.numel()} outputs differ"


@pytest.mark.gpu
@pytest.mark.parametrize("case", [c for c in RES_CASES if c[2] == 1], ids=_case_id)
def test_projection_without_residual_exact(case):
    """The projection as BaseBEVResBackbone launches it: BatchNorm, no ReLU, fp32 output."""
    got, ref, _ = _run(case, relu=False, round_out=False, residual=False)
    assert bool((ref < 0).any())
    assert torch.equal(got, ref)


@pytest.mark.gpu
def test_residual_epilogue_persistent_grid():
    """Enough tiles that every CTA of the persistent grid walks several tile sets (accumulator buffers wrap)."""
    got, ref, _ = _run((64, 64, 3, 1, 128, 256, 4, False), relu=True, round_out=True, residual=True)
    assert torch.equal(got, ref)


# ---- the whole module ---------------------------------------------------------------------------------------------------
def _sweep_inputs(nb, grid, seed):
    """pillar rows + index map, and the dense canvas, of ``nb`` synthetic nuScenes-like sweeps through PillarVFEFromPoints."""
    from lidar_vision_vqa_b200 import synth
    from lidar_vision_vqa_b200.modules import PillarVFEFromPoints

    dev = _dev()
    half = 0.2 * grid / 2
    rng, vs = [-half, -half, -5.0, half, half, 3.0], [0.2, 0.2, 8.0]
    pts, offs = synth.make_batch(nb, synth.NUSCENES_32, 5, seed0=seed)
    b = np.repeat(np.arange(nb), np.diff(offs)).astype(np.float32)[:, None]
    points = torch.from_numpy(np.concatenate([b, pts], axis=1)).to(dev)
    base = dict(USE_NORM=True, WITH_DISTANCE=False, USE_ABSLOTE_XYZ=True, NUM_FILTERS=[64], MAX_POINTS_PER_VOXEL=32,
                MAX_NUMBER_OF_VOXELS=60000)
    torch.manual_seed(seed)
    vfe_map = PillarVFEFromPoints(dict(base, EMIT_INDEX_MAP=True), 5, vs, rng, [grid, grid, 1]).eval().to(dev)
    vfe_canvas = PillarVFEFromPoints(dict(base, FUSE_SCATTER=True), 5, vs, rng, [grid, grid, 1]).eval().to(dev)
    vfe_canvas.load_state_dict(vfe_map.state_dict())
    with torch.inference_mode():
        d1 = vfe_map({"points": points, "batch_size": nb})
        d2 = vfe_canvas({"points": points, "batch_size": nb})
    return {"pillar_features": d1["pillar_features"], "bev_index_map": d1["bev_index_map"]}, d2["spatial_features"]


def _pair(cfg, seed):
    from lidar_vision_vqa_b200 import BaseBEVResBackbone

    torch.manual_seed(seed)
    ref = ro.randomise(ro.BaseBEVResBackbone(cfg, 64), seed).eval()
    mine = BaseBEVResBackbone(cfg, 64).eval()
    mine.load_state_dict(ref.state_dict(), strict=True)
    return ref.to(_dev()), mine.to(_dev())


def _reference_fp32(ref, canvas):
    tf32 = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.inference_mode():
            return ref({"spatial_features": canvas.clone()})["spatial_features_2d"]
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32


def _errors(got, want):
    scale = float(want.abs().max())
    d = (got - want).abs()
    return float(d.max()) / scale, float((d <= 2e-3 * scale).float().mean())


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(RES_CFGS))
def test_module_matches_the_restatement(name):
    ref, mine = _pair(RES_CFGS[name], 3)
    rows_map, canvas = _sweep_inputs(2, 256, 21)
    want = _reference_fp32(ref, canvas)
    with torch.inference_mode():
        out = mine(dict(rows_map))
        got = out["spatial_features_2d"].clone()
        again = mine(dict(rows_map))["spatial_features_2d"]
        via_canvas = mine({"spatial_features": canvas})["spatial_features_2d"]
    torch.cuda.synchronize()
    assert int(out["_conv_error_word"].item()) == 0
    assert got.shape == want.shape == (2, *mine.output_shape(256, 256))
    assert torch.equal(got, again)  # two runs, equal bits
    assert torch.equal(got, via_canvas)  # the canvas route compacts to the same rows: same operands, same order
    rel, share = _errors(got, want)
    print(f"{name}: max err / max|ref| = {rel:.2e}, within 2e-3: {share:.5f}")
    assert rel <= 4e-3 and share > 0.99


@pytest.mark.gpu
def test_refuses_training_mode_cpu_input_and_shapes_outside_the_set():
    from lidar_vision_vqa_b200 import BaseBEVResBackbone, _native

    m = BaseBEVResBackbone(RES_CFGS["1level_no_up"], 64)
    with pytest.raises(NotImplementedError):
        m({"spatial_features": torch.zeros(1, 64, 32, 32, device=_dev())})
    with pytest.raises(_native.NativeLibraryError):
        m.eval()({"spatial_features": torch.zeros(1, 64, 32, 32)})
    odd = BaseBEVResBackbone(dict(LAYER_NUMS=[1], LAYER_STRIDES=[2], NUM_FILTERS=[96]), 64).eval().to(_dev())
    with pytest.raises(NotImplementedError):
        odd({"spatial_features": torch.zeros(1, 64, 32, 32, device=_dev())})


@pytest.mark.gpu
def test_full_size_points_to_residual_backbone():
    """16 frames x 64 channels x 512^2 (the nuScenes pillar workload): rows + index map straight from the VFE, equal to the
    canvas route bit for bit, and frame 0 against the restatement."""
    ref, mine = _pair(RES_CFGS["4level_s1222"], 5)
    rows_map, canvas = _sweep_inputs(16, 512, 40)
    assert int((rows_map["bev_index_map"] >= 0).sum()) == rows_map["pillar_features"].shape[0]
    with torch.inference_mode():
        out = mine(dict(rows_map))
        got = out["spatial_features_2d"].clone()
        via_canvas = mine({"spatial_features": canvas})["spatial_features_2d"]
    torch.cuda.synchronize()
    assert int(out["_conv_error_word"].item()) == 0
    assert got.shape == (16, 512, 256, 256)
    assert torch.equal(got, via_canvas)
    want = _reference_fp32(ref, canvas[:1])
    rel, share = _errors(got[:1], want)
    print(f"full size frame 0: max err / max|ref| = {rel:.2e}, within 2e-3: {share:.5f}")
    assert rel <= 4e-3 and share > 0.99


@pytest.mark.gpu
def test_extractor_and_pipeline_take_the_residual_backbone():
    """BevExtractor(ship='features2d', backbone=BaseBEVResBackbone) (which runs it through PillarEncoderPipeline) yields
    float16(module(canvas of that frame alone)) per token, in input order."""
    from lidar_vision_vqa_b200 import synth
    from lidar_vision_vqa_b200.backbone import BaseBEVResBackbone
    from lidar_vision_vqa_b200.extract import BevExtractor
    from lidar_vision_vqa_b200.modules import PillarVFEFromPoints

    dev = _dev()
    rng, vs = [-25.6, -25.6, -5.0, 25.6, 25.6, 3.0], [0.2, 0.2, 8.0]
    frames = [synth.make_sweep(900 + i, synth.NUSCENES_32, 5)[:7000 + 300 * i] for i in range(5)]
    base = dict(USE_NORM=True, WITH_DISTANCE=False, USE_ABSLOTE_XYZ=True, NUM_FILTERS=[64], MAX_POINTS_PER_VOXEL=32,
                MAX_NUMBER_OF_VOXELS=20000)
    torch.manual_seed(1)
    vfe = PillarVFEFromPoints(dict(base), 5, vs, rng, [256, 256, 1]).eval().to(dev)
    vfe_c = PillarVFEFromPoints(dict(base, FUSE_SCATTER=True), 5, vs, rng, [256, 256, 1]).eval().to(dev)
    vfe_c.load_state_dict(vfe.state_dict())
    bb = ro.randomise(BaseBEVResBackbone(RES_CFGS["3level_s222_up124"], 64), 4).eval().to(dev)
    ex = BevExtractor(vfe, batch_size=2, max_points_per_frame=9000, depth=2, ship="features2d", backbone=bb)
    items = [(f"t{i}", f) for i, f in enumerate(frames)]
    got = {tok: np.array(arr) for tok, arr in ex.run(items)}
    assert list(got) == [t for t, _ in items]
    for tok, f in items:
        pts = torch.from_numpy(np.concatenate([np.zeros((len(f), 1), np.float32), f], axis=1)).to(dev)
        with torch.inference_mode():
            canvas = vfe_c({"points": pts, "batch_size": 1})["spatial_features"]
            want = bb({"spatial_features": canvas})["spatial_features_2d"][0].to(torch.float16).cpu().numpy()
        assert got[tok].dtype == np.float16 and got[tok].shape == (384, 128, 128)
        np.testing.assert_array_equal(got[tok].view(np.uint16), want.view(np.uint16))
