"""BaseBEVBackbone and BaseBEVResBackbone on the tcgen05 convolution kernel (SURVEY 8 f-3).

Mirrors `pcdet/models/backbones_2d/base_bev_backbone.py:6-112`: same constructor arguments, same sub-module tree -- so the
state-dict keys (`blocks.0.1.weight`, `blocks.0.2.running_mean`, `deblocks.2.0.weight`, ...) and therefore the reference's
checkpoints load unchanged -- same `forward(data_dict) -> data_dict` writing `spatial_features_2d` (NCHW fp32).

What differs is how eval-mode forward computes: every Conv2d/ConvTranspose2d + BatchNorm2d + ReLU triple is ONE launch of
`pillars_conv_forward` (csrc/conv_umma.cu), activations stay NHWC between layers, the three up-sampling branches write their
channel windows of the concatenated output directly (no `torch.cat`), and the first layer gathers its input from the pillar
rows through the BEV index map when the VFE left them in `data_dict` (`pillar_features` + `bev_index_map`): the dense
`spatial_features` canvas is then not read at all.  Given only `spatial_features`, the canvas is first compacted into that
form (`pillars_canvas_to_rows`).  There is no PyTorch fallback: training mode and shapes outside the kernel's set raise.

`BaseBEVResBackbone`, the reference's residual variant of the same file (ResNet BasicBlocks), shares all of that; its
blocks add the identity in the epilogue of their second convolution (`pillars_conv_forward_residual`)."""
from __future__ import annotations

from typing import List, Optional

import torch
import torch.nn as nn

from . import _native

_EPS, _MOMENTUM = 1e-3, 0.01  # base_bev_backbone.py:36


def _cfg_get(cfg, key, default=None):
    if isinstance(cfg, dict):
        return cfg.get(key, default)
    getter = getattr(cfg, "get", None)
    if callable(getter):
        return getter(key, default)
    return getattr(cfg, key, default)


class _Layer:
    """One fused conv + BN (+ ReLU) launch: geometry plus the prepared weight image."""

    def __init__(self, conv: nn.Module, bn: nn.BatchNorm2d, transposed: bool, relu: bool = True):
        self.conv, self.bn, self.transposed, self.relu = conv, bn, transposed, relu
        w = conv.weight
        if transposed:
            c_in, c_out, k = w.shape[0], w.shape[1], w.shape[2]
            stride = conv.stride[0]
            if k != stride or k not in (1, 2, 4):
                raise NotImplementedError(f"ConvTranspose2d kernel {k} stride {stride}: only kernel == stride in (1, 2, 4)")
            self.desc = dict(c_in=c_in, c_out=c_out, k=1, stride=1, pad=0, up=k)
        else:
            c_out, c_in, k = w.shape[0], w.shape[1], w.shape[2]
            self.desc = dict(c_in=c_in, c_out=c_out, k=k, stride=conv.stride[0], pad=1 if k == 3 else 0, up=1)
        self.image: Optional[torch.Tensor] = None
        self.shift: Optional[torch.Tensor] = None
        self._key = None

    def native(self, round_out: bool) -> _native.PillarsConv:
        d = self.desc
        return _native.PillarsConv(d["c_in"], d["c_out"], d["k"], d["stride"], d["pad"], d["up"], 1 if self.relu else 0,
                                   1 if round_out else 0)

    def prepare(self, device: torch.device) -> None:
        params = (self.conv.weight, self.bn.weight, self.bn.bias, self.bn.running_mean, self.bn.running_var)
        def version(t):  # inference tensors (a module moved under torch.inference_mode) do not track one
            try:
                return t._version
            except RuntimeError:
                return -1

        key = tuple((t.data_ptr(), version(t)) for t in params) + (str(device),)
        if key == self._key:
            return
        lib = _native.load()
        with torch.no_grad():
            w = self.conv.weight.detach().to(device=device, dtype=torch.float32)
            if self.transposed and self.desc["up"] == 1:  # ConvTranspose2d(k=1, s=1) is a 1x1 convolution with [in, out] weights
                w = w.permute(1, 0, 2, 3)
            w = w.contiguous()
            scale = (self.bn.weight.detach().float() / torch.sqrt(self.bn.running_var.detach().float() + self.bn.eps)).to(device)
            shift = (self.bn.bias.detach().float().to(device) - self.bn.running_mean.detach().float().to(device) * scale)
            scale, shift = scale.contiguous(), shift.contiguous()
        cv = self.native(False)
        nbytes = lib.pillars_conv_weight_bytes(cv)
        if nbytes == 0:
            raise NotImplementedError(f"convolution {self.desc} is outside the set the tcgen05 kernel is instantiated for")
        image = torch.empty(nbytes // 4, dtype=torch.float32, device=device)
        stream = torch.cuda.current_stream(device).cuda_stream
        _native.check(lib.pillars_conv_prepare(cv, w.data_ptr(), scale.data_ptr(), image.data_ptr(), stream), "pillars_conv_prepare")
        # built once, then read by every later call on ANY stream (a pipeline runs each batch on its own): finish it here
        torch.cuda.current_stream(device).synchronize()
        self.image, self.shift, self._key = image, shift, key


def conv_forward(layer: _Layer, out: torch.Tensor, out_c_total: int, out_c_off: int, out_nchw: bool, n_frames: int, h_in: int,
                 w_in: int, x_nhwc: Optional[torch.Tensor] = None, rows: Optional[torch.Tensor] = None,
                 cell_row: Optional[torch.Tensor] = None, round_out: bool = True, error: Optional[torch.Tensor] = None,
                 residual: Optional[torch.Tensor] = None) -> None:
    """One launch.  ``residual`` (NHWC, laid out like ``out``) is added after the BatchNorm shift, before the ReLU."""
    lib = _native.load()
    dev = out.device
    stream = torch.cuda.current_stream(dev).cuda_stream
    args = (layer.native(round_out), layer.image.data_ptr(), layer.shift.data_ptr(), x_nhwc.data_ptr() if x_nhwc is not None else None,
            rows.data_ptr() if rows is not None else None, cell_row.data_ptr() if cell_row is not None else None, n_frames, h_in,
            w_in, out.data_ptr(), out_c_total, out_c_off, 1 if out_nchw else 0)
    err = error.data_ptr() if error is not None else None
    if residual is None:
        _native.check(lib.pillars_conv_forward(*args, err, stream), "pillars_conv_forward")
    else:
        _native.check(lib.pillars_conv_forward_residual(*args, residual.data_ptr(), err, stream), "pillars_conv_forward_residual")


def _bev_cfg(model_cfg, input_channels):
    """The per-level lists of a BaseBEVBackbone-style config (base_bev_backbone.py:11-24)."""
    layer_nums = _cfg_get(model_cfg, "LAYER_NUMS")
    if layer_nums is not None:
        layer_strides, num_filters = _cfg_get(model_cfg, "LAYER_STRIDES"), _cfg_get(model_cfg, "NUM_FILTERS")
        assert len(layer_nums) == len(layer_strides) == len(num_filters)
    else:
        layer_nums = layer_strides = num_filters = []
    upsample_strides = _cfg_get(model_cfg, "UPSAMPLE_STRIDES")
    if upsample_strides is not None:
        num_upsample_filters = _cfg_get(model_cfg, "NUM_UPSAMPLE_FILTERS")
        assert len(upsample_strides) == len(num_upsample_filters)
    else:
        upsample_strides = num_upsample_filters = []
    c_in_list = [input_channels, *num_filters[:-1]]
    return layer_nums, layer_strides, num_filters, upsample_strides, num_upsample_filters, c_in_list


def _bn(c):
    return nn.BatchNorm2d(c, eps=_EPS, momentum=_MOMENTUM)


def _gathered_input(data_dict):
    """The first layer's input as (pillar rows, BEV index map, device, frames, h, w): the VFE's own rows + index map when it
    left them, otherwise the ``spatial_features`` canvas compacted into that form (``pillars_canvas_to_rows``)."""
    if data_dict.get("bev_index_map") is not None and data_dict.get("pillar_features") is not None:
        rows = data_dict["pillar_features"]
        cell_row = data_dict["bev_index_map"]
        dev = rows.device
        nb, h, w = cell_row.shape
    else:
        canvas = data_dict["spatial_features"]
        if canvas.dtype != torch.float32 or not canvas.is_cuda:
            raise _native.NativeLibraryError("spatial_features must be a float32 CUDA tensor (no CPU path)")
        canvas = canvas.contiguous()
        dev = canvas.device
        nb, c, h, w = canvas.shape
        lib = _native.load()
        cell_row = torch.empty((nb, h, w), dtype=torch.int32, device=dev)
        rows = torch.empty((max(nb * h * w, 1), c), dtype=torch.float32, device=dev)
        counter = torch.empty(1, dtype=torch.int32, device=dev)
        _native.check(lib.pillars_canvas_to_rows(canvas.data_ptr(), nb, c, h, w, cell_row.data_ptr(), rows.data_ptr(),
                                                 counter.data_ptr(), torch.cuda.current_stream(dev).cuda_stream),
                      "pillars_canvas_to_rows")
    if rows.dtype != torch.float32 or cell_row.dtype != torch.int32:
        raise _native.NativeLibraryError("pillar rows must be float32 and the index map int32")
    return rows.contiguous(), cell_row.contiguous(), dev, nb, h, w


class _FusedBEVBackbone(nn.Module):
    """What the plain and the residual backbone share: the input forms, the weight images, the output geometry and the
    up-sampling branches writing their channel windows of the NCHW result.  A subclass builds ``self._plan = (levels, de)``
    in ``_build_plan`` and runs one level in ``_run_level``; ``_chain(level)`` lists the layers whose geometries compose to
    that level's output size."""

    def _build_plan(self):
        raise NotImplementedError

    def _chain(self, level):
        raise NotImplementedError

    def _layers(self):
        raise NotImplementedError

    def _check_plan(self, n_levels, de):
        if len(de) > n_levels:
            raise NotImplementedError("the trailing deblock over the concatenated branches is not instantiated")
        if len(de) == 0 and n_levels != 1:
            raise NotImplementedError("multi-level backbone without up-sampling branches")

    @staticmethod
    def _out_hw(h, w, d):
        if d["up"] > 1:
            return d["up"] * h, d["up"] * w
        return (h + 2 * d["pad"] - d["k"]) // d["stride"] + 1, (w + 2 * d["pad"] - d["k"]) // d["stride"] + 1

    def _level_shapes(self, h, w):
        shapes = []
        for i in range(len(self._plan[0])):
            for l in self._chain(i):
                h, w = self._out_hw(h, w, l.desc)
            shapes.append((h, w))
        return shapes

    def output_shape(self, h: int, w: int):
        """(channels, height, width) of ``spatial_features_2d`` for an ``h x w`` input canvas."""
        if self._plan is None:
            self._build_plan()
        de = self._plan[1]
        shapes = self._level_shapes(h, w)
        if de:
            oh, ow = self._out_hw(*shapes[0], de[0].desc)
            return sum(l.desc["c_out"] for l in de), oh, ow
        return self._chain(0)[-1].desc["c_out"], shapes[0][0], shapes[0][1]

    def forward(self, data_dict):
        if self.training:
            raise NotImplementedError(f"{type(self).__name__} (B200) is an inference path: call .eval(); training runs the "
                                      "reference module")
        if self._plan is None:
            self._build_plan()
        levels, de = self._plan
        rows, cell_row, dev, nb, h, w = _gathered_input(data_dict)
        for l in self._layers():
            l.prepare(dev)
        error = torch.zeros(1, dtype=torch.int32, device=dev)

        # output geometry first: every branch must land on the same image
        shapes = self._level_shapes(h, w)
        if de:
            outs = [self._out_hw(*shapes[i], de[i].desc) for i in range(len(levels))]
            if any(o != outs[0] for o in outs):
                raise ValueError(f"up-sampling branches disagree on the output size: {outs}")
            oh, ow = outs[0]
            c_total = sum(l.desc["c_out"] for l in de)
        else:
            oh, ow = shapes[0]
            c_total = self._chain(0)[-1].desc["c_out"]
        result = torch.empty((nb, c_total, oh, ow), dtype=torch.float32, device=dev)

        c_off, x = 0, None
        for i in range(len(levels)):
            # without up-sampling the (single) level's last layer produces spatial_features_2d itself
            x = self._run_level(i, x, rows, cell_row, nb, h, w, None if de else result, error)
            h, w = shapes[i]
            if de:
                conv_forward(de[i], result, c_total, c_off, True, nb, h, w, x_nhwc=x, round_out=False, error=error)
                c_off += de[i].desc["c_out"]
        data_dict["spatial_features_2d"] = result
        data_dict["_conv_error_word"] = error
        return data_dict


class BaseBEVBackbone(_FusedBEVBackbone):
    """Drop-in for the reference class of the same name (registry `backbones_2d.__all__['BaseBEVBackbone']`)."""

    def __init__(self, model_cfg, input_channels):
        super().__init__()
        self.model_cfg = model_cfg
        layer_nums, layer_strides, num_filters, upsample_strides, num_upsample_filters, c_in_list = _bev_cfg(model_cfg,
                                                                                                            input_channels)
        levels = len(layer_nums)
        self.blocks, self.deblocks = nn.ModuleList(), nn.ModuleList()
        for i in range(levels):
            # sub-module positions are part of the checkpoint format: [pad, conv, bn, relu] + [conv, bn, relu] * n
            seq: List[nn.Module] = [nn.ZeroPad2d(1),
                                    nn.Conv2d(c_in_list[i], num_filters[i], 3, stride=layer_strides[i], padding=0, bias=False),
                                    _bn(num_filters[i]), nn.ReLU()]
            for _ in range(layer_nums[i]):
                seq += [nn.Conv2d(num_filters[i], num_filters[i], 3, padding=1, bias=False), _bn(num_filters[i]), nn.ReLU()]
            self.blocks.append(nn.Sequential(*seq))
            if len(upsample_strides) > 0:
                s = upsample_strides[i]
                if s > 1 or (s == 1 and not _cfg_get(model_cfg, "USE_CONV_FOR_NO_STRIDE", False)):
                    up = nn.ConvTranspose2d(num_filters[i], num_upsample_filters[i], s, stride=s, bias=False)
                else:
                    k = int(round(1 / s))
                    up = nn.Conv2d(num_filters[i], num_upsample_filters[i], k, stride=k, bias=False)
                self.deblocks.append(nn.Sequential(up, _bn(num_upsample_filters[i]), nn.ReLU()))
        c_in = sum(num_upsample_filters)
        if len(upsample_strides) > levels:
            s = upsample_strides[-1]
            self.deblocks.append(nn.Sequential(nn.ConvTranspose2d(c_in, c_in, s, stride=s, bias=False), _bn(c_in), nn.ReLU()))
        self.num_bev_features = c_in
        self._plan = None

    # ---- the fused plan ---------------------------------------------------------------------------------------------------
    def _build_plan(self):
        blocks = []
        for seq in self.blocks:
            mods = list(seq)
            layers = [_Layer(mods[1], mods[2], False)]
            for j in range(4, len(mods), 3):
                layers.append(_Layer(mods[j], mods[j + 1], False))
            blocks.append(layers)
        de = [_Layer(seq[0], seq[1], isinstance(seq[0], nn.ConvTranspose2d)) for seq in self.deblocks]
        self._check_plan(len(blocks), de)
        self._plan = (blocks, de)

    def _chain(self, level):
        return self._plan[0][level]

    def _layers(self):
        blocks, de = self._plan
        return [l for layers in blocks for l in layers] + de

    def _run_level(self, i, x, rows, cell_row, nb, h, w, final, error):
        """Level i's 3x3 convolutions, NHWC with tf32-rounded outputs; the last one into ``final`` (NCHW) when given."""
        layers = self._plan[0][i]
        dev = rows.device
        for j, l in enumerate(layers):
            oh_l, ow_l = self._out_hw(h, w, l.desc)
            if final is not None and j == len(layers) - 1:
                conv_forward(l, final, final.shape[1], 0, True, nb, h, w, x_nhwc=x, rows=rows if x is None else None,
                             cell_row=cell_row if x is None else None, round_out=False, error=error)
            else:
                y = torch.empty((nb, oh_l, ow_l, l.desc["c_out"]), dtype=torch.float32, device=dev)
                conv_forward(l, y, l.desc["c_out"], 0, False, nb, h, w, x_nhwc=x, rows=rows if x is None else None,
                             cell_row=cell_row if x is None else None, round_out=True, error=error)
                x = y
            h, w = oh_l, ow_l
        return x


class BasicBlock(nn.Module):
    """The residual unit of BaseBEVResBackbone (base_bev_backbone.py: ResNet BasicBlock): conv3x3(stride) + BN + ReLU,
    conv3x3 + BN, plus the identity -- or, with ``downsample``, a 1x1(stride) + BN projection of it -- then ReLU.  Holds
    the parameters under the reference's names; the B200 forward is BaseBEVResBackbone's."""

    def __init__(self, inplanes, planes, stride=1, padding=1, downsample=False):
        super().__init__()
        self.conv1 = nn.Conv2d(inplanes, planes, kernel_size=3, stride=stride, padding=padding, bias=False)
        self.bn1 = _bn(planes)
        self.relu1 = nn.ReLU()
        self.conv2 = nn.Conv2d(planes, planes, kernel_size=3, padding=1, bias=False)
        self.bn2 = _bn(planes)
        self.relu2 = nn.ReLU()
        self.downsample = downsample
        if self.downsample:
            self.downsample_layer = nn.Sequential(nn.Conv2d(inplanes, planes, kernel_size=1, stride=stride, padding=0, bias=False),
                                                  _bn(planes))
        self.stride = stride


class _ResStep:
    """One BasicBlock as launches: the projection (1x1 + BN, no ReLU; None = the block's input is the identity), conv1 and
    conv2, the latter adding the identity in its epilogue."""

    def __init__(self, blk: BasicBlock):
        if blk.conv1.padding[0] != 1:
            raise NotImplementedError(f"BasicBlock padding {blk.conv1.padding[0]}: only 1 is instantiated")
        self.proj = _Layer(blk.downsample_layer[0], blk.downsample_layer[1], False, relu=False) if blk.downsample else None
        self.conv1 = _Layer(blk.conv1, blk.bn1, False)
        self.conv2 = _Layer(blk.conv2, blk.bn2, False)


class BaseBEVResBackbone(_FusedBEVBackbone):
    """Drop-in for the reference's residual variant (registry `backbones_2d.__all__['BaseBEVResBackbone']`): every level is
    BasicBlock(c_in, f, stride, 1, downsample=True) followed by LAYER_NUMS[i] BasicBlock(f, f), the branches as in
    BaseBEVBackbone except that every stride >= 1 is a ConvTranspose2d (USE_CONV_FOR_NO_STRIDE is not read).

    Eval-mode forward: three launches per block with a projection (the projection, conv1, conv2 + residual) and two per block
    without; activations stay NHWC between them and the identity is added in conv2's epilogue before its ReLU.  The first
    block's projection and conv1 both gather their input from the pillar rows: the canvas is never materialised.  Training
    mode and shapes outside the kernel's set raise, as in BaseBEVBackbone."""

    def __init__(self, model_cfg, input_channels):
        super().__init__()
        self.model_cfg = model_cfg
        layer_nums, layer_strides, num_filters, upsample_strides, num_upsample_filters, c_in_list = _bev_cfg(model_cfg,
                                                                                                            input_channels)
        levels = len(layer_nums)
        self.blocks, self.deblocks = nn.ModuleList(), nn.ModuleList()
        for i in range(levels):
            seq = [BasicBlock(c_in_list[i], num_filters[i], layer_strides[i], 1, True)]
            for _ in range(layer_nums[i]):
                seq.append(BasicBlock(num_filters[i], num_filters[i]))
            self.blocks.append(nn.Sequential(*seq))
            if len(upsample_strides) > 0:
                s = upsample_strides[i]
                if s >= 1:
                    up = nn.ConvTranspose2d(num_filters[i], num_upsample_filters[i], s, stride=s, bias=False)
                else:
                    k = int(round(1 / s))
                    up = nn.Conv2d(num_filters[i], num_upsample_filters[i], k, stride=k, bias=False)
                self.deblocks.append(nn.Sequential(up, _bn(num_upsample_filters[i]), nn.ReLU()))
        c_in = sum(num_upsample_filters) if len(num_upsample_filters) > 0 else sum(num_filters)
        if len(upsample_strides) > levels:
            s = upsample_strides[-1]
            self.deblocks.append(nn.Sequential(nn.ConvTranspose2d(c_in, c_in, s, stride=s, bias=False), _bn(c_in), nn.ReLU()))
        self.num_bev_features = c_in
        self._plan = None

    def _build_plan(self):
        levels = [[_ResStep(blk) for blk in seq] for seq in self.blocks]
        de = [_Layer(seq[0], seq[1], isinstance(seq[0], nn.ConvTranspose2d)) for seq in self.deblocks]
        self._check_plan(len(levels), de)
        self._plan = (levels, de)

    def _chain(self, level):  # (a projection has its block's conv1 geometry: k 1 pad 0 and k 3 pad 1 agree at either stride)
        return [l for st in self._plan[0][level] for l in (st.conv1, st.conv2)]

    def _layers(self):
        levels, de = self._plan
        return [l for steps in levels for st in steps for l in (st.proj, st.conv1, st.conv2) if l is not None] + de

    def _run_level(self, i, x, rows, cell_row, nb, h, w, final, error):
        """Level i's blocks, NHWC; conv1 outputs and block outputs tf32-rounded (the next layer multiplies them), projections
        kept in fp32 (they are only ever added).  ``final`` (NCHW) receives the last block's output when given: the residual
        epilogue writes NHWC, so that one is copied over."""
        steps = self._plan[0][i]
        dev = rows.device
        for j, st in enumerate(steps):
            last = final is not None and j == len(steps) - 1
            oh, ow = self._out_hw(h, w, st.conv1.desc)
            c = st.conv1.desc["c_out"]
            src = dict(x_nhwc=x, rows=rows if x is None else None, cell_row=cell_row if x is None else None)
            if st.proj is not None:
                ident = torch.empty((nb, oh, ow, c), dtype=torch.float32, device=dev)
                conv_forward(st.proj, ident, c, 0, False, nb, h, w, round_out=False, error=error, **src)
            else:
                ident = x
            t = torch.empty((nb, oh, ow, c), dtype=torch.float32, device=dev)
            conv_forward(st.conv1, t, c, 0, False, nb, h, w, round_out=True, error=error, **src)
            y = torch.empty((nb, oh, ow, c), dtype=torch.float32, device=dev)
            conv_forward(st.conv2, y, c, 0, False, nb, oh, ow, x_nhwc=t, round_out=not last, error=error, residual=ident)
            if last:
                final.copy_(y.permute(0, 3, 1, 2))
            x, h, w = y, oh, ow
        return x
