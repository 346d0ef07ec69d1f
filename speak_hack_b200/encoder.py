"""ResNet-50 feature encoder (identity / emotion / pose) on sm_100a kernels.

The reference builds each encoder as `nn.Sequential(*list(torchvision.models.resnet50().children())[:-1])`
(model.py:60-62).  `ResNet50Encoder` is an nn.Sequential with the same child indices, sub-module attribute names and
state_dict keys (`0.weight`, `1.running_mean`, `4.0.conv1.weight`, `4.0.downsample.1.bias`, ...), constructed in the
same order as torchvision so a seeded construction consumes the RNG identically, but its forward/backward are one
autograd node that launches libirfd_b200.so: tcgen05 implicit-GEMM convs whose epilogue gathers the train-mode
BatchNorm statistics, fused BN-apply+ReLU(+residual) passes, NHWC bf16 activations.  No torchvision import.
The forward, backward and inference passes live in encoder_group.py: a call runs as the one-member
`EncoderGroup([encoder])`.
"""
from __future__ import annotations

from typing import List

import torch
import torch.nn as nn

from . import ops

BN_EPS = 1e-5
BN_MOMENTUM = 0.1
# widest image the stem's im2col stages (21 input rows of W + 6 fp32 in 48 KB of shared memory)
MAX_STEM_W = 579
MIN_HW = 32


def check_inference_shape(x) -> None:
    """The eval-mode, no-autograd pass runs at any 32 <= H, W with W <= 579 (box-tiled convs where 128 consecutive
    pixels are not one tile, ceil-sized stride-2 layers like torchvision)."""
    h, w = x.shape[2], x.shape[3]
    if h < MIN_HW or w < MIN_HW or w > MAX_STEM_W:
        raise ops._lib.IrfdError(f"ResNet50Encoder: eval-mode inference needs {MIN_HW} <= H, W and W <= {MAX_STEM_W}, "
                                 f"got {tuple(x.shape)}")


def trainable_shape(n: int, h: int, w: int) -> bool:
    """Train-mode and differentiated passes (batch statistics in the conv epilogues, the backward kernels) need H and W
    multiples of 32 and every conv of the n-image batch on the linear pixel-tile geometry (ops.conv_geometry)."""
    if h % 32 or w % 32 or w > MAX_STEM_W:
        return False
    for i, (hs, ws) in enumerate(ops.resnet_stage_hw(h, w)):
        for k in ((1, 3) if i > 0 else (1,)):  # 3x3 stride-1 convs from layer1 on; 1x1 GEMMs at every stage
            g = ops.conv_geometry(n, hs, ws, k)
            if g is None or g[0]:
                return False
    return True


class Bottleneck(nn.Module):
    """Parameter container laid out like torchvision.models.resnet.Bottleneck (resnet.py:108-141)."""

    expansion = 4

    def __init__(self, inplanes, planes, stride=1, downsample=None):
        super().__init__()
        self.conv1 = nn.Conv2d(inplanes, planes, kernel_size=1, stride=1, bias=False)
        self.bn1 = nn.BatchNorm2d(planes)
        self.conv2 = nn.Conv2d(planes, planes, kernel_size=3, stride=stride, padding=1, bias=False)
        self.bn2 = nn.BatchNorm2d(planes)
        self.conv3 = nn.Conv2d(planes, planes * self.expansion, kernel_size=1, stride=1, bias=False)
        self.bn3 = nn.BatchNorm2d(planes * self.expansion)
        self.relu = nn.ReLU(inplace=True)
        self.downsample = downsample
        self.stride = stride


def _make_layer(inplanes, planes, blocks, stride):
    downsample = None
    if stride != 1 or inplanes != planes * 4:
        downsample = nn.Sequential(
            nn.Conv2d(inplanes, planes * 4, kernel_size=1, stride=stride, bias=False), nn.BatchNorm2d(planes * 4)
        )
    layers = [Bottleneck(inplanes, planes, stride, downsample)]
    for _ in range(1, blocks):
        layers.append(Bottleneck(planes * 4, planes))
    return nn.Sequential(*layers)


class ResNet50Encoder(nn.Sequential):
    """`nn.Sequential(conv1, bn1, relu, maxpool, layer1..4, avgpool)` with fused sm_100a forward/backward."""

    def __init__(self):
        conv1 = nn.Conv2d(3, 64, kernel_size=7, stride=2, padding=3, bias=False)
        bn1 = nn.BatchNorm2d(64)
        relu = nn.ReLU(inplace=True)
        maxpool = nn.MaxPool2d(kernel_size=3, stride=2, padding=1)
        layer1 = _make_layer(64, 64, 3, 1)
        layer2 = _make_layer(256, 128, 4, 2)
        layer3 = _make_layer(512, 256, 6, 2)
        layer4 = _make_layer(1024, 512, 3, 2)
        avgpool = nn.AdaptiveAvgPool2d((1, 1))
        fc = nn.Linear(2048, 1000)  # constructed (RNG parity with torchvision's ResNet.__init__) and dropped
        del fc
        super().__init__(conv1, bn1, relu, maxpool, layer1, layer2, layer3, layer4, avgpool)
        # torchvision's init loop (resnet.py:208-213)
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")
            elif isinstance(m, nn.BatchNorm2d):
                nn.init.constant_(m.weight, 1)
                nn.init.constant_(m.bias, 0)
        self._recompute_bn_update = False

    def _flat_params(self) -> List[nn.Parameter]:
        return [p for p in self.parameters()]

    def _bn_counters(self) -> List[torch.Tensor]:
        return [m.num_batches_tracked for m in self.modules() if isinstance(m, nn.BatchNorm2d)]

    def forward(self, x):
        return self._run(x, 1, None)

    def forward_groups(self, x, groups: int, stem_cols=None):
        """x = `groups` batches stacked along dim 0; equivalent to `groups` consecutive calls (per-call BN stats).
        stem_cols: optional `ops.im2col_stem(x, 192)` computed by the caller (shared by encoders fed the same x)."""
        return self._run(x, groups, stem_cols)

    def _run(self, x, groups, stem_cols):
        from .encoder_group import EncoderGroup  # encoder_group imports this module

        if not x.is_cuda:
            raise ops._lib.IrfdError("ResNet50Encoder: CUDA tensors only (no CPU fallback on the IRFD hot path)")
        if x.dim() != 4 or x.shape[1] != 3:
            raise ops._lib.IrfdError(f"ResNet50Encoder: expected [N,3,H,W], got {tuple(x.shape)}")
        recorded = torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self.parameters()))
        # refused before any launch, so the BatchNorm running buffers and counters stay untouched
        if not self.training and not recorded:
            check_inference_shape(x)
        elif not trainable_shape(x.size(0), x.shape[2], x.shape[3]):
            mode = "train-mode" if self.training else "differentiated eval-mode"
            raise ops._lib.IrfdError(f"ResNet50Encoder: a {mode} pass needs H, W multiples of 32 (W <= {MAX_STEM_W}) and "
                                     f"128-pixel tiles of whole rows / images at every stage, got {tuple(x.shape)}; "
                                     "eval-mode inference under no_grad runs at any 32 <= H, W")
        grp = EncoderGroup([self])
        if not grp.can_run(x, groups, recorded):
            raise ops._lib.IrfdError(f"ResNet50Encoder.forward_groups: shape {tuple(x.shape)} cannot form {groups} groups")
        return grp(x, groups, stem_cols)[0]
