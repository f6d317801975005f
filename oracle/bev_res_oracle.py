"""TEST INFRASTRUCTURE ONLY -- a torch restatement of ``BasicBlock`` / ``BaseBEVResBackbone``
(pcdet/models/backbones_2d/base_bev_backbone.py, OpenPCDet v0.6.0), used as the checker of the B200 class
``lidar_vision_vqa_b200.backbone.BaseBEVResBackbone``.  Same constructor, same sub-module tree (so the same state-dict
keys), eager fp32 forward.  Where the reference copy is present (oracle/_ref), ``tests/test_bev_res_oracle.py`` checks
this restatement against the live class: keys and CPU fp32 outputs must be identical.

    BasicBlock(inplanes, planes, stride=1, padding=1, downsample=False):
        out = relu2(bn2(conv2(relu1(bn1(conv1(x))))) + identity),  identity = downsample_layer(x) or x
        downsample_layer = Sequential(Conv2d(inplanes, planes, 1, stride, 0), BatchNorm2d)   (no ReLU)
    blocks[i] = Sequential(BasicBlock(c_in_i, f_i, stride_i, 1, True), BasicBlock(f_i, f_i) x LAYER_NUMS[i])
    deblocks[i] = ConvTranspose2d(k = s) for s >= 1, Conv2d(k = 1/s) below 1; + BN + ReLU (USE_CONV_FOR_NO_STRIDE unread)
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn as nn


def _get(cfg, key, default=None):
    return cfg.get(key, default) if hasattr(cfg, "get") else getattr(cfg, key, default)


def _bn(c):
    return nn.BatchNorm2d(c, eps=1e-3, momentum=0.01)


class BasicBlock(nn.Module):
    expansion = 1

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

    def forward(self, x):
        identity = x
        out = self.relu1(self.bn1(self.conv1(x)))
        out = self.bn2(self.conv2(out))
        if self.downsample:
            identity = self.downsample_layer(x)
        return self.relu2(out + identity)


class BaseBEVResBackbone(nn.Module):
    def __init__(self, model_cfg, input_channels):
        super().__init__()
        self.model_cfg = model_cfg
        if _get(model_cfg, "LAYER_NUMS") is not None:
            layer_nums, layer_strides = _get(model_cfg, "LAYER_NUMS"), _get(model_cfg, "LAYER_STRIDES")
            num_filters = _get(model_cfg, "NUM_FILTERS")
            assert len(layer_nums) == len(layer_strides) == len(num_filters)
        else:
            layer_nums = layer_strides = num_filters = []
        if _get(model_cfg, "UPSAMPLE_STRIDES") is not None:
            upsample_strides, num_upsample_filters = _get(model_cfg, "UPSAMPLE_STRIDES"), _get(model_cfg, "NUM_UPSAMPLE_FILTERS")
            assert len(upsample_strides) == len(num_upsample_filters)
        else:
            upsample_strides = num_upsample_filters = []
        num_levels = len(layer_nums)
        c_in_list = [input_channels, *num_filters[:-1]]
        self.blocks = nn.ModuleList()
        self.deblocks = nn.ModuleList()
        for idx in range(num_levels):
            cur_layers = [BasicBlock(c_in_list[idx], num_filters[idx], layer_strides[idx], 1, True)]
            for _ in range(layer_nums[idx]):
                cur_layers.append(BasicBlock(num_filters[idx], num_filters[idx]))
            self.blocks.append(nn.Sequential(*cur_layers))
            if len(upsample_strides) > 0:
                stride = upsample_strides[idx]
                if stride >= 1:
                    up = nn.ConvTranspose2d(num_filters[idx], num_upsample_filters[idx], upsample_strides[idx],
                                            stride=upsample_strides[idx], bias=False)
                else:
                    stride = int(np.round(1 / stride))
                    up = nn.Conv2d(num_filters[idx], num_upsample_filters[idx], stride, stride=stride, bias=False)
                self.deblocks.append(nn.Sequential(up, _bn(num_upsample_filters[idx]), nn.ReLU()))
        c_in = sum(num_upsample_filters) if len(num_upsample_filters) > 0 else sum(num_filters)
        if len(upsample_strides) > num_levels:
            self.deblocks.append(nn.Sequential(
                nn.ConvTranspose2d(c_in, c_in, upsample_strides[-1], stride=upsample_strides[-1], bias=False), _bn(c_in), nn.ReLU()))
        self.num_bev_features = c_in

    def forward(self, data_dict):
        spatial_features = data_dict["spatial_features"]
        ups = []
        x = spatial_features
        for i in range(len(self.blocks)):
            x = self.blocks[i](x)
            ups.append(self.deblocks[i](x) if len(self.deblocks) > 0 else x)
        if len(ups) > 1:
            x = torch.cat(ups, dim=1)
        elif len(ups) == 1:
            x = ups[0]
        if len(self.deblocks) > len(self.blocks):
            x = self.deblocks[-1](x)
        data_dict["spatial_features_2d"] = x
        return data_dict


def randomise(module: nn.Module, seed: int) -> nn.Module:
    """Non-trivial BatchNorm statistics and affine parameters (default-initialised BN would hide the shift and scale folds)."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for m in module.modules():
            if isinstance(m, nn.BatchNorm2d):
                m.weight.copy_(0.5 + torch.rand(m.weight.shape, generator=g))
                m.bias.copy_(0.2 * torch.randn(m.bias.shape, generator=g))
                m.running_mean.copy_(0.2 * torch.randn(m.bias.shape, generator=g))
                m.running_var.copy_(0.5 + 1.5 * torch.rand(m.bias.shape, generator=g))
    return module
