"""GPU parity of the BEV backbone row (SURVEY 8 f-3): the tcgen05 convolution kernel through the C ABI.

Three kinds of checks:
  * single layers on inputs whose values are exactly representable in tf32 (small integers): the tensor core's products and the
    fp32 accumulation are then exact, so every geometry (taps, stride, halo, parity planes, gathered input, transposed phases,
    NHWC / NCHW channel windows, ragged image borders, tf32-rounded outputs) must match a float64 convolution BIT FOR BIT.
    The case table reaches every instantiation `launch_conv_umma` can pick, at the product's per-layer image sizes, with
    enough frames that every CTA of the persistent grid walks at least three tile sets;
  * every launch of `BaseBEVBackbone.forward` at the product's image sizes, against float64 computed from that launch's own
    recorded input, within an error bound derived from the kernel's rounding points;
  * the whole `BaseBEVBackbone` against the reference's own module (oracle/_ref copy, CPU fp32) with random weights.  The kernel
    multiplies in tf32 -- as the reference's nn.Conv2d itself does on this GPU under PyTorch's default
    `torch.backends.cudnn.allow_tf32 = True` -- so the tolerance is stated against the output's scale:
    |err| <= 4e-3 * max|ref| over the 11 / 16 stacked layers (measured: 1.0e-3 at 16 x 512^2, where the reference's own TF32
    run deviates from its fp32 run by 0.8e-3: bench.py `backbone`).
"""
from typing import NamedTuple, Optional

import numpy as np
import pytest
import torch
import torch.nn.functional as F


def _dev():
    return torch.device("cuda:0")


def _int_tensor(shape, lo, hi, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(lo, hi + 1, shape, generator=g).to(torch.float32)


def _rna_tf32(t):
    """cvt.rna.tf32.f32 on float32 values: keep 10 mantissa bits, round half away from zero."""
    return ((t.contiguous().view(torch.int32) + 0x1000) & -0x2000).view(torch.float32)


class _FakeBN:
    def __init__(self, c, shift):
        self.weight = torch.ones(c)
        self.bias = shift.clone()
        self.running_mean = torch.zeros(c)
        self.running_var = torch.ones(c) - 1e-3
        self.eps = 1e-3


def _run_layer(conv, shift, x_nchw, *, gather=False, out_nchw=False, c_total=None, c_off=0, round_out=False):
    """One launch of `conv_forward`; returns the whole output buffer (on the device, -7 wherever the layer does not write)."""
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
    x = x_nchw.to(dev)
    if gather:  # the occupied cells' channels as pillar rows in random order, plus the BEV index map
        pos = (x != 0).any(dim=1).nonzero()
        perm = torch.randperm(len(pos), generator=torch.Generator().manual_seed(5)).to(dev)
        pos = pos[perm]
        idx = torch.full((nb, h, w), -1, dtype=torch.int32, device=dev)
        idx[pos[:, 0], pos[:, 1], pos[:, 2]] = torch.arange(len(pos), dtype=torch.int32, device=dev)
        rows = x.permute(0, 2, 3, 1)[pos[:, 0], pos[:, 1], pos[:, 2]].contiguous() if len(pos) else torch.zeros((1, c), device=dev)
        B.conv_forward(layer, out, c_total, c_off, out_nchw, nb, h, w, rows=rows, cell_row=idx, round_out=round_out, error=err)
    else:
        B.conv_forward(layer, out, c_total, c_off, out_nchw, nb, h, w, x_nhwc=x.permute(0, 2, 3, 1).contiguous(),
                       round_out=round_out, error=err)
    torch.cuda.synchronize()
    assert int(err.item()) == 0, hex(int(err.item()))
    return out, d


def _reference_layer(conv, shift, x_nchw, round_out=False):
    """float64 on the device with cuDNN off (a plain GEMM over the products: no FFT / Winograd).  On integer operands every
    partial sum is an integer below 2^24, so this is the exact result, in any summation order."""
    dev = _dev()
    with torch.no_grad(), torch.backends.cudnn.flags(enabled=False):
        x, wt = x_nchw.to(dev, torch.float64), conv.weight.detach().to(dev, torch.float64)
        if isinstance(conv, torch.nn.ConvTranspose2d):
            y = F.conv_transpose2d(x, wt, stride=conv.stride)
        else:
            pad = 1 if conv.kernel_size[0] == 3 else 0
            y = F.conv2d(x, wt, stride=conv.stride, padding=pad)
        # eval BatchNorm with weight 1, mean 0, var + eps = 1: y + shift
        y = torch.relu(y + shift.to(dev, torch.float64).view(1, -1, 1, 1)).float()
    return _rna_tf32(y) if round_out else y


def _conv_module(c_in, c_out, k, stride, transposed):
    if transposed:
        return torch.nn.ConvTranspose2d(c_in, c_out, k, stride=stride, bias=False)
    return torch.nn.Conv2d(c_in, c_out, k, stride=stride, padding=0, bias=False)


# k_conv_umma instantiations (CONV_CASE rows of launch_conv_umma): (stride, n_eff, T)
CONV_INSTANCES = {(1, 64, 4), (1, 64, 2), (1, 64, 1), (1, 128, 2), (1, 128, 1), (1, 256, 1), (2, 64, 1), (2, 128, 1), (2, 256, 1)}


def _launch_config(desc, h, w, gathered, nchw):
    """`launch_conv_umma`'s choice for a layer (csrc/conv_umma.cu), restated: n_eff accumulator columns per patch (a transposed
    convolution holds its two dx phases side by side: the "pair" epilogue), T stacked 16 x 8 patches per tile, SA halo stages,
    whether gathered input takes the sparse loader (it needs SA channel blocks), the epilogue branch and the tiles per frame."""
    n_eff = 2 * desc["c_out"] if desc["up"] > 1 else desc["c_out"]
    stride = desc["stride"]
    h_out = (h + 2 * desc["pad"] - desc["k"]) // stride + 1
    w_out = (w + 2 * desc["pad"] - desc["k"]) // stride + 1
    t = {64: 4, 128: 2}.get(n_eff, 1) if stride == 1 else 1
    while t > 1 and 16 * (t // 2) >= h_out:
        t //= 2
    sa = 1 if (stride == 2 and n_eff == 256) else 2
    pair = desc["up"] > 1
    return dict(n_eff=n_eff, T=t, stride=stride, pair=pair, sa=sa, mma_warps=2 if (stride == 1 and n_eff == 64 and t > 1) else 1,
                gathered=gathered, sparse=gathered and desc["c_in"] // 32 >= sa,
                epilogue=("nchw" if nchw else "nhwc") + ("_pair" if pair else ""),
                tiles_per_frame=-(-h_out // (16 * t)) * -(-w_out // 8))


class _Case(NamedTuple):
    name: str
    conv: tuple                        # (c_in, c_out, k, stride, transposed): Conv2d, or ConvTranspose2d(kernel = stride = k)
    h: int
    w: int
    nchw: bool = False                 # NCHW channel window with -7 neighbours, as the deblocks write (else NHWC, as blocks)
    round_out: bool = False            # tf32-rounded outputs, as every block layer stores them
    occupancy: Optional[float] = None  # gathered input (pillar rows + index map) with this share of occupied cells
    frames: Optional[int] = None       # None: enough frames that every CTA walks >= 3 tile sets

    def config(self):
        from lidar_vision_vqa_b200 import backbone as B

        desc = B._Layer(_conv_module(*self.conv), None, self.conv[4]).desc
        return _launch_config(desc, self.h, self.w, self.occupancy is not None, self.nchw)


def _product_layers(tag, h, w, strides, ups):
    """The distinct layer shapes of BaseBEVBackbone(LAYER_NUMS [3, 5, 5], NUM_FILTERS [64, 128, 256], NUM_UPSAMPLE_FILTERS
    [128] * 3) on an h x w canvas of 64 channels: as the module launches them (first layer gathered, blocks NHWC + round_out,
    deblocks into their NCHW window)."""
    cases, c_in = [], 64
    for i, (c, s) in enumerate(zip((64, 128, 256), strides)):
        first = dict(occupancy=0.3) if i == 0 else {}
        cases.append(_Case(f"{tag}.block{i}.0", (c_in, c, 3, s, False), h, w, round_out=True, **first))
        h, w = (h - 1) // s + 1, (w - 1) // s + 1
        cases.append(_Case(f"{tag}.block{i}.n", (c, c, 3, 1, False), h, w, round_out=True))
        u = ups[i]
        cases.append(_Case(f"{tag}.deblock{i}", (c, 128, 2, 2, False) if u == 0.5 else (c, 128, u, u, True), h, w, nchw=True))
        c_in = c
    return cases


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
] + [
    # the product's per-layer shapes: nuScenes multihead (512^2, strides 2/2/2, up-sampling 0.5/1/2), KITTI pointpillar
    # (496 x 432, 2/2/2, 1/2/4: ragged at every level) and Waymo pointpillar (468^2, 1/2/2, 1/2/4: the first layer is the
    # stride-1 four-patch two-MMA-warp configuration, gathered; 117^2 is odd)
    *_product_layers("nuscenes", 512, 512, (2, 2, 2), (0.5, 1, 2)),
    *_product_layers("kitti", 496, 432, (2, 2, 2), (1, 2, 4)),
    *_product_layers("waymo", 468, 468, (1, 2, 2), (1, 2, 4)),
    # instantiated, but reached by none of those
    _Case("s1_n64_T2.nchw_round", (64, 64, 3, 1, False), 32, 512, nchw=True, round_out=True),
    _Case("s1_n64_T1.nhwc", (64, 64, 3, 1, False), 16, 520),
    _Case("s1_n128_T1.nchw", (128, 128, 3, 1, False), 16, 512, nchw=True),
    _Case("pair_n128_T2.nhwc_round", (256, 64, 2, 2, True), 64, 128, round_out=True),
    _Case("pair_n128_T1.nhwc", (128, 64, 4, 4, True), 16, 256),
    _Case("pair_n256.nchw_round", (256, 128, 2, 2, True), 16, 256, nchw=True, round_out=True),
    _Case("c_in32.gathered_plain_loader", (32, 128, 3, 2, False), 256, 256, occupancy=0.1),
    _Case("c_in96.odd_channel_blocks", (96, 128, 3, 1, False), 128, 128, round_out=True),
    _Case("s2_n256_SA1.gathered", (64, 256, 3, 2, False), 256, 256, occupancy=0.06),
]


def _case_id(case):
    return case.name if isinstance(case, _Case) else "x".join(map(str, case))


def test_layer_cases_reach_every_instantiation():
    """Runs without a GPU: the table reaches every CONV_CASE row, both pair widths at both patch stacks, the gathered loader
    in its sparse, plain and one-stage forms, and every epilogue branch with and without tf32-rounded outputs."""
    cfgs = [c.config() for c in LAYER_CASES if isinstance(c, _Case)]
    assert {(c["stride"], c["n_eff"], c["T"]) for c in cfgs} == CONV_INSTANCES
    assert {(c["n_eff"], c["T"]) for c in cfgs if c["pair"]} == {(128, 1), (128, 2), (256, 1)}
    assert {c["sparse"] for c in cfgs if c["gathered"]} == {False, True}
    assert any(c["gathered"] and c["sa"] == 1 for c in cfgs)
    assert any(c["gathered"] and c["mma_warps"] == 2 for c in cfgs)
    branches = {(c.config()["epilogue"], c.round_out) for c in LAYER_CASES if isinstance(c, _Case)}
    assert branches == {(e, r) for e in ("nhwc", "nchw", "nchw_pair", "nhwc_pair") for r in (False, True)}
    assert {c.conv[0] for c in LAYER_CASES if isinstance(c, _Case)} >= {32, 64, 96, 128, 256}


def _case_operands(case, seed):
    """Integers in x in [-4, 4], w in [-3, 3], shift in [-40, 40]: every partial sum is an integer below 9 * 384 * 12 + 40 <
    2^24, exact in fp32 in any order.  With round_out the outputs must reach 2048, where tf32's spacing exceeds 1: there the
    input is non-negative and the even output channels' weights are positive (the odd ones keep both signs, for the ReLU)."""
    c_in, c_out, k, stride, transposed = case.conv
    conv = _conv_module(*case.conv)
    wt = _int_tensor(tuple(conv.weight.shape), -3, 3, seed)
    x_lo = -4
    if case.round_out:
        k_eff = c_in * (1 if transposed else k * k) * (case.occupancy or 1.0)
        x_lo, w_lo = (0, 1) if k_eff >= 512 else (3, 2)  # mean product 4 or 8.75
        pos = _int_tensor(tuple(conv.weight.shape), w_lo, 3, seed + 2)
        even = torch.zeros(c_out, dtype=torch.bool)
        even[0::2] = True
        even = even.view(1, -1, 1, 1) if transposed else even.view(-1, 1, 1, 1)
        wt = torch.where(even, pos, wt)
    with torch.no_grad():
        conv.weight.copy_(wt)
    shift = _int_tensor((c_out,), -40, 40, seed + 1)
    return conv, shift, x_lo


@pytest.mark.gpu
@pytest.mark.parametrize("case", LAYER_CASES, ids=_case_id)
def test_conv_layer_exact_on_tf32_representable_values(case):
    if not isinstance(case, _Case):
        c_in, c_out, k, stride, transposed, h, w, nb = case
        case = _Case(_case_id(case), (c_in, c_out, k, stride, transposed), h, w, frames=nb)
    dev = _dev()
    cfg = case.config()
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    nb = case.frames or -(-3 * sms // cfg["tiles_per_frame"])
    if case.frames is None:  # the persistent loop: accumulator buffers, stage barriers and frame decoding wrap
        assert nb * cfg["tiles_per_frame"] >= 3 * sms
    conv, shift, x_lo = _case_operands(case, 11)
    if case.frames is not None:
        x = _int_tensor((nb, case.conv[0], case.h, case.w), x_lo, 4, 13)
    else:  # (large: drawn on the device)
        g = torch.Generator(dev).manual_seed(13)
        x = torch.randint(x_lo, 5, (nb, case.conv[0], case.h, case.w), generator=g, device=dev).to(torch.float32)
        if case.occupancy is not None:
            x = x * (torch.rand((nb, 1, case.h, case.w), generator=g, device=dev) < case.occupancy)
    ref0 = _reference_layer(conv, shift, x)
    ref = _rna_tf32(ref0) if case.round_out else ref0
    if case.round_out:  # the rounding must matter: values it moves, ties among them (rn and rna differ only there)
        assert bool((ref != ref0).any())
        assert bool(((ref0.view(torch.int32) & 0x1FFF) == 0x1000).any())
    c_out = case.conv[1]
    c_total, c_off = (c_out + 64, 32) if (case.nchw or cfg["pair"]) and case.frames is None else (c_out, 0)
    got, _ = _run_layer(conv, shift, x, gather=case.occupancy is not None, out_nchw=case.nchw, c_total=c_total, c_off=c_off,
                        round_out=case.round_out)
    if case.nchw:
        win, rest = got[:, c_off:c_off + c_out], torch.cat([got[:, :c_off], got[:, c_off + c_out:]], dim=1)
    else:
        win, rest = got[..., c_off:c_off + c_out].permute(0, 3, 1, 2), torch.cat([got[..., :c_off], got[..., c_off + c_out:]], dim=-1)
    assert win.shape == ref.shape
    assert torch.equal(win, ref), f"{int((win != ref).sum())} of {ref.numel()} outputs differ"
    assert bool((rest == -7.0).all())


@pytest.mark.gpu
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


@pytest.mark.gpu
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


@pytest.mark.gpu
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


@pytest.mark.gpu
def test_backbone_refuses_training_mode_and_cpu_input():
    from lidar_vision_vqa_b200 import _native
    from lidar_vision_vqa_b200.backbone import BaseBEVBackbone

    m = BaseBEVBackbone(BACKBONE_CASES["kitti_pointpillar"], 64)
    with pytest.raises(NotImplementedError):
        m({"spatial_features": torch.zeros(1, 64, 32, 32, device=_dev())})
    with pytest.raises(_native.NativeLibraryError):
        m.eval()({"spatial_features": torch.zeros(1, 64, 32, 32)})


@pytest.mark.gpu
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


@pytest.mark.gpu
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


@pytest.mark.gpu
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


@pytest.mark.gpu
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


# ---- the accepted set is the launched set ----------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("geometry", [(3, 1, False), (1, 1, False), (3, 2, False), (2, 2, False), (2, 2, True), (4, 4, True)],
                         ids=["3x3s1", "1x1", "3x3s2", "2x2s2", "up2", "up4"])
@pytest.mark.parametrize("c_out", [64, 128, 256])
@pytest.mark.parametrize("c_in", [32, 64, 96, 256])
def test_every_accepted_descriptor_runs_exactly(c_in, c_out, geometry):
    """Whatever `pillars_conv_weight_bytes` accepts, `pillars_conv_forward` launches, exactly; what it refuses, `prepare`
    refuses with NotImplementedError."""
    from lidar_vision_vqa_b200 import _native
    from lidar_vision_vqa_b200 import backbone as B

    k, stride, transposed = geometry
    conv = _conv_module(c_in, c_out, k, stride, transposed)
    with torch.no_grad():
        conv.weight.copy_(_int_tensor(tuple(conv.weight.shape), -3, 3, 51))
    shift = _int_tensor((c_out,), -40, 40, 52)
    layer = B._Layer(conv, _FakeBN(c_out, shift), transposed)
    if _native.load().pillars_conv_weight_bytes(layer.native(False)) == 0:
        assert transposed and c_out == 256  # (n_eff = 512 is not instantiated)
        with pytest.raises(NotImplementedError):
            layer.prepare(_dev())
        return
    x = _int_tensor((2, c_in, 21, 19), -4, 4, 53)
    got, _ = _run_layer(conv, shift, x)
    ref = _reference_layer(conv, shift, x)
    assert torch.equal(got.permute(0, 3, 1, 2), ref)


# ---- every launch of the module at the product's image sizes ---------------------------------------------------------------
PRODUCT_BACKBONES = {
    "nuscenes_multihead_512": (BACKBONE_CASES["nuscenes_multihead"], 512, 512),
    "kitti_pointpillar_496x432": (BACKBONE_CASES["kitti_pointpillar"], 496, 432),
    # waymo_models/pointpillar_1x.yaml: the first block keeps the 468 x 468 grid
    "waymo_pointpillar_468": (dict(LAYER_NUMS=[3, 5, 5], LAYER_STRIDES=[1, 2, 2], NUM_FILTERS=[64, 128, 256],
                                   UPSAMPLE_STRIDES=[1, 2, 4], NUM_UPSAMPLE_FILTERS=[128, 128, 128]), 468, 468),
}


def _launch_error(call, dev):
    """float64 result of one recorded launch from its own input, and the bound on the kernel's deviation from it.

    The kernel's rounding points: weights w' = rna_tf32(fp32(w * scale)) (k_conv_wimg), inputs already tf32, products exact in
    fp32, K = taps * c_in of them summed in fp32 by the tensor core, then fp32 + shift, ReLU, and rna_tf32 with round_out.
    A sum of K terms in fp32 errs by at most K * u * (sum of |terms|); u = 2^-24 for round-to-nearest, and the factor 2
    (u = 2^-23) allows for truncation, as the tensor core's order and rounding of its accumulation are not documented.  The
    shift is one more term of that sum.  With round_out, the stored value may move by half a tf32 ulp more."""
    layer = call["layer"]
    d, bn = layer.desc, layer.bn
    if call["x"] is not None:
        x = call["x"].permute(0, 3, 1, 2)
    else:
        cell_row, rows = call["cell_row"], call["rows"]
        x = torch.zeros((*cell_row.shape, rows.shape[1]), dtype=torch.float32, device=dev)
        occ = cell_row >= 0
        x[occ] = rows[cell_row[occ].long()]
        x = x.permute(0, 3, 1, 2)
    assert torch.equal(_rna_tf32(x), x), "a layer's input is not tf32-representable"
    with torch.no_grad():  # as _Layer.prepare computes them
        scale = (bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + bn.eps)).to(dev)
        shift = bn.bias.detach().float().to(dev) - bn.running_mean.detach().float().to(dev) * scale
        w = layer.conv.weight.detach().to(dev, torch.float32)
        w = _rna_tf32(w * (scale.view(1, -1, 1, 1) if layer.transposed else scale.view(-1, 1, 1, 1))).double()
        x = x.double()
        with torch.backends.cudnn.flags(enabled=False):
            if layer.transposed:
                conv = lambda a, b: F.conv_transpose2d(a, b, stride=d["up"])  # noqa: E731
            else:
                conv = lambda a, b: F.conv2d(a, b, stride=d["stride"], padding=d["pad"])  # noqa: E731
            acc, s = conv(x, w), conv(x.abs(), w.abs())
    shift = shift.double().view(1, -1, 1, 1)
    ref = torch.relu(acc + shift)
    k = d["c_in"] * (1 if layer.transposed else d["k"] * d["k"])
    bound = 2 * (k + 1) * 2.0 ** -24 * (s + shift.abs())
    if call["round_out"]:
        bound = bound + torch.where(ref > 0, torch.exp2(torch.floor(torch.log2(ref.clamp_min(1e-300))) - 10), 0.0)
    return x, ref, bound


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(PRODUCT_BACKBONES))
@pytest.mark.parametrize("fused_input", [False, True], ids=["canvas", "rows+map"])
def test_backbone_launches_against_float64_at_product_size(name, fused_input, monkeypatch):
    """BaseBEVBackbone.forward on two frames at 6 % occupancy, random float weights and BatchNorm statistics: every launch is
    recorded with a copy of its input and checked against float64 computed from that input (teacher forcing: an error cannot
    compound over the 19 launches), within the bound `_launch_error` derives."""
    from lidar_vision_vqa_b200 import backbone as B

    cfg, h, w = PRODUCT_BACKBONES[name]
    dev = _dev()
    torch.manual_seed(17)
    m = B.BaseBEVBackbone(cfg, 64).eval()
    _randomise_bn(m, 5)
    m = m.to(dev)
    nb = 2
    g = torch.Generator(dev).manual_seed(19)
    occupied = torch.rand((nb, 1, h, w), generator=g, device=dev) < 0.06
    canvas = _rna_tf32(torch.rand((nb, 64, h, w), generator=g, device=dev)) * occupied  # tf32 already: no assumption
    if fused_input:  # about how the tensor core reads a non-tf32 fp32 value
        pos = occupied[:, 0].nonzero()
        idx = torch.full((nb, h, w), -1, dtype=torch.int32, device=dev)
        idx[pos[:, 0], pos[:, 1], pos[:, 2]] = torch.arange(len(pos), dtype=torch.int32, device=dev)
        d = {"pillar_features": canvas.permute(0, 2, 3, 1)[pos[:, 0], pos[:, 1], pos[:, 2]].contiguous(), "bev_index_map": idx}
    else:
        d = {"spatial_features": canvas}

    calls, launch = [], B.conv_forward

    def record(layer, out, out_c_total, out_c_off, out_nchw, n_frames, h_in, w_in, x_nhwc=None, rows=None, cell_row=None,
               round_out=True, error=None):
        calls.append(dict(layer=layer, out=out, c_total=out_c_total, c_off=out_c_off, nchw=out_nchw, hw=(n_frames, h_in, w_in),
                          x=None if x_nhwc is None else x_nhwc.clone(), rows=None if rows is None else rows.clone(),
                          cell_row=None if cell_row is None else cell_row.clone(), round_out=round_out))
        launch(layer, out, out_c_total, out_c_off, out_nchw, n_frames, h_in, w_in, x_nhwc=x_nhwc, rows=rows, cell_row=cell_row,
               round_out=round_out, error=error)

    monkeypatch.setattr(B, "conv_forward", record)
    with torch.inference_mode():
        out = m(d)
    torch.cuda.synchronize()
    assert int(out["_conv_error_word"].item()) == 0
    result = out["spatial_features_2d"]
    blocks, de = m._plan
    assert len(calls) == sum(len(layers) for layers in blocks) + len(de)
    assert result.shape == (nb, *m.output_shape(h, w))
    deblock_calls = [c for c in calls if c["layer"] in de]
    assert [c["layer"] for c in deblock_calls] == de
    assert all(c["out"] is result and c["nchw"] for c in deblock_calls)
    offs = [c["c_off"] for c in deblock_calls]
    assert offs == [sum(l.desc["c_out"] for l in de[:i]) for i in range(len(de))] and offs[-1] + de[-1].desc["c_out"] == result.shape[1]

    for i, call in enumerate(calls):
        x, ref, bound = _launch_error(call, dev)
        if i == 0:  # the first layer reads the canvas' cells (through pillars_canvas_to_rows on the canvas route)
            assert call["x"] is None and torch.equal(x.float(), canvas)
        c_out = call["layer"].desc["c_out"]
        if call["nchw"]:
            got = call["out"][:, call["c_off"]:call["c_off"] + c_out]  # the channel window of spatial_features_2d
        else:
            got = call["out"].permute(0, 3, 1, 2)
        assert got.shape == ref.shape, i
        excess = (got.double() - ref).abs() - bound
        assert float(excess.max()) <= 0, (i, call["layer"].desc, float(excess.max()), int((excess > 0).sum()))
