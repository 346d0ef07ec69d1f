"""ResNet-50 feature encoder (identity / emotion / pose) on sm_100a kernels.

The reference builds each encoder as `nn.Sequential(*list(torchvision.models.resnet50().children())[:-1])`
(model.py:60-62).  `ResNet50Encoder` is an nn.Sequential with the same child indices, sub-module attribute names and
state_dict keys (`0.weight`, `1.running_mean`, `4.0.conv1.weight`, `4.0.downsample.1.bias`, ...), constructed in the
same order as torchvision so a seeded construction consumes the RNG identically, but its forward/backward are one
autograd node that launches libirfd_b200.so: tcgen05 implicit-GEMM convs whose epilogue gathers the train-mode
BatchNorm statistics, fused BN-apply+ReLU(+residual) passes, NHWC bf16 activations.  No torchvision import.
"""
from __future__ import annotations

from typing import List, Optional

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


class _BNState:
    """Per-BN forward record: batch (or running) mean/rstd + count, needed by backward and the second buffer update."""

    __slots__ = ("mean", "rstd", "count")

    def __init__(self, mean, rstd, count):
        self.mean, self.rstd, self.count = mean, rstd, count


def _bn_stats(bn: nn.BatchNorm2d, ssum, ssq, rows, train: bool, groups: int = 1, updates: int = 1):
    """Finalize batch statistics (train; one set per statistic group, running buffers updated group by group like
    consecutive nn.BatchNorm2d calls) or fetch the running ones (eval).  `rows` = total rows over all groups."""
    if train:
        count = rows // groups
        mean, rstd = ops.bn_finalize(ssum, ssq, count, BN_EPS, BN_MOMENTUM, bn.running_mean, bn.running_var, updates,
                                     groups)
        return _BNState(mean, rstd, count)
    return _BNState(bn.running_mean, ops.bn_eval_rstd(bn.running_var, BN_EPS), rows)


def _conv_stats(x, wk, ksize, train):
    if train:
        return ops.conv_gemm(x, wk, ksize, ops.EPI_STATS)
    return ops.conv_gemm(x, wk, ksize, ops.EPI_PLAIN), None, None


def _encoder_inference(enc, x, col0=None):
    """Eval-mode, no-autograd forward: every BatchNorm (+ReLU, + the Bottleneck residual add) is folded into the
    epilogue of the conv that feeds it (irfd_conv_gemm_affine), so a layer is ONE kernel and the pre-BN tensor is never
    rounded to bf16 or written to HBM.  Same arithmetic as torchvision's Bottleneck in eval mode (resnet.py:143-164)."""
    x = x.contiguous().to(torch.float32)
    n, _, h, w = x.shape
    if col0 is None:
        col0 = ops.im2col_stem(x, 192)
    m0 = col0.shape[0]
    sc, sh = ops.bn_eval_affine(enc[1])
    a0 = ops.conv_gemm_affine(col0.view(1, 1, m0, 192), ops.pack_conv_weight(enc[0].weight, ops.PACK_FLAT, kpad=192), 1,
                              sc, sh, relu=True).view(n, ops.half_up(h), ops.half_up(w), 64)
    cur, _ = ops.maxpool_fwd(a0)
    for li in range(4, 8):
        for blk in enc[li]:
            nb, hh, ww, _cin = cur.shape
            sc, sh = ops.bn_eval_affine(blk.bn1)
            a1 = ops.conv_gemm_affine(cur, ops.pack_conv_weight(blk.conv1.weight, ops.PACK_FPROP), 1, sc, sh, relu=True)
            planes = a1.shape[-1]
            sc, sh = ops.bn_eval_affine(blk.bn2)
            wk2 = ops.pack_conv_weight(blk.conv2.weight, ops.PACK_FPROP)
            if blk.stride == 1:
                a2 = ops.conv_gemm_affine(a1, wk2, 3, sc, sh, relu=True)
            else:
                col2 = ops.im2col_3x3s2(a1)
                a2 = ops.conv_gemm_affine(col2.view(1, 1, col2.shape[0], 9 * planes), wk2, 1, sc, sh,
                                          relu=True).view(nb, ops.half_up(hh), ops.half_up(ww), planes)
            if blk.downsample is not None:
                xs = ops.subsample2(cur) if blk.stride == 2 else cur
                sc, sh = ops.bn_eval_affine(blk.downsample[1])
                idn = ops.conv_gemm_affine(xs, ops.pack_conv_weight(blk.downsample[0].weight, ops.PACK_FPROP), 1, sc, sh,
                                           relu=False)
            else:
                idn = cur
            sc, sh = ops.bn_eval_affine(blk.bn3)
            cur = ops.conv_gemm_affine(a2, ops.pack_conv_weight(blk.conv3.weight, ops.PACK_FPROP), 1, sc, sh, res=idn,
                                       relu=True)
    return ops.avgpool_fwd(cur).view(n, -1, 1, 1)


class _EncoderFn(torch.autograd.Function):
    """forward(x [N,3,H,W] fp32, enc, groups, *params) -> features [N,2048,1,1] fp32.  params = enc._flat_params().

    groups > 1: x stacks `groups` independent batches along dim 0 (IRFD: source and target images); train-mode BN
    statistics are computed per group and the running buffers updated group by group, so the result is the same as
    `groups` separate encoder calls in that order (model.py:84-90 calls Ei(x_s) then Ei(x_t)), at half the launches.
    """

    @staticmethod
    def forward(ctx, x, enc, groups, col0, recorded, *params):
        train = enc.training
        G = groups if train else 1  # eval-mode BN uses the shared running statistics: no groups needed
        # The reference wraps every encoder call in a reentrant checkpoint (model.py:84-90): a differentiated pass
        # re-runs the forward during backward and so updates the BN running buffers twice (SURVEY Q3).  Both updates are
        # applied here, in the order the reference would produce them (forward order, then reverse order).
        # `recorded` (computed by the caller, where grad mode is visible) says a backward pass can follow
        U = 2 if (train and getattr(enc, "_recompute_bn_update", False) and recorded) else 1
        x = x.contiguous().to(torch.float32)
        n, _, h, w = x.shape
        S = {}  # saved activations
        # ---- stem: 7x7/2 conv as explicit im2col + GEMM, BN, ReLU, maxpool
        conv0, bn0 = enc[0], enc[1]
        if col0 is None:  # the stem's im2col matrix depends only on the images: callers may share it across encoders
            col0 = ops.im2col_stem(x, 192)
        wk0 = ops.pack_conv_weight(conv0.weight, ops.PACK_FLAT, kpad=192)
        if train:
            z0, s, q = ops.gemm_rows(col0, wk0, ops.EPI_STATS)
        else:
            z0, s, q = ops.gemm_rows(col0, wk0, ops.EPI_PLAIN), None, None
        h1, w1 = h // 2, w // 2
        z0 = z0.view(n, h1, w1, 64)
        st0 = _bn_stats(bn0, s, q, n * h1 * w1, train, G, U)
        a0 = ops.bn_apply(z0, st0.mean, st0.rstd, bn0.weight, bn0.bias, relu=True, groups=G)
        p0, arg0 = ops.maxpool_fwd(a0)
        S["stem"] = (col0, z0, st0, a0, arg0)
        cur = p0
        S["blocks"] = []
        for li in range(4, 8):
            for blk in enc[li]:
                xin = cur
                nb, hh, ww, cin = xin.shape
                z1, s, q = _conv_stats(xin, ops.pack_conv_weight(blk.conv1.weight, ops.PACK_FPROP), 1, train)
                st1 = _bn_stats(blk.bn1, s, q, nb * hh * ww, train, G, U)
                a1 = ops.bn_apply(z1, st1.mean, st1.rstd, blk.bn1.weight, blk.bn1.bias, relu=True, groups=G)
                planes = a1.shape[-1]
                wk2 = ops.pack_conv_weight(blk.conv2.weight, ops.PACK_FPROP)
                col2 = None
                if blk.stride == 1:
                    z2, s, q = _conv_stats(a1, wk2, 3, train)
                    ho, wo = hh, ww
                else:
                    col2 = ops.im2col_3x3s2(a1)
                    ho, wo = hh // 2, ww // 2
                    if train:
                        z2, s, q = ops.gemm_rows(col2, wk2, ops.EPI_STATS)
                    else:
                        z2, s, q = ops.gemm_rows(col2, wk2, ops.EPI_PLAIN), None, None
                    z2 = z2.view(nb, ho, wo, planes)
                st2 = _bn_stats(blk.bn2, s, q, nb * ho * wo, train, G, U)
                a2 = ops.bn_apply(z2, st2.mean, st2.rstd, blk.bn2.weight, blk.bn2.bias, relu=True, groups=G)
                z3, s, q = _conv_stats(a2, ops.pack_conv_weight(blk.conv3.weight, ops.PACK_FPROP), 1, train)
                st3 = _bn_stats(blk.bn3, s, q, nb * ho * wo, train, G, U)
                xs = zd = std = None
                if blk.downsample is not None:
                    dconv, dbn = blk.downsample[0], blk.downsample[1]
                    xs = ops.subsample2(xin) if blk.stride == 2 else xin
                    zd, s, q = _conv_stats(xs, ops.pack_conv_weight(dconv.weight, ops.PACK_FPROP), 1, train)
                    std = _bn_stats(dbn, s, q, nb * ho * wo, train, G, U)
                    out = ops.bn_apply(z3, st3.mean, st3.rstd, blk.bn3.weight, blk.bn3.bias, res=zd,
                                       bn2=(std.mean, std.rstd, dbn.weight, dbn.bias), relu=True, groups=G)
                else:
                    out = ops.bn_apply(z3, st3.mean, st3.rstd, blk.bn3.weight, blk.bn3.bias, res=xin, relu=True, groups=G)
                S["blocks"].append((blk, xin, z1, st1, a1, col2, z2, st2, a2, z3, st3, xs, zd, std, out))
                cur = out
        feat = ops.avgpool_fwd(cur)
        if train:  # nn.BatchNorm2d bookkeeping: one fused increment for all 53 counters
            torch._foreach_add_(enc._bn_counters(), G * U)
        S["final_hw"] = (cur.shape[1], cur.shape[2])
        ctx.enc = enc
        ctx.S = S
        ctx.train = train
        ctx.G = G
        return feat.view(n, -1, 1, 1)

    @staticmethod
    def backward(ctx, dfeat):
        enc, S = ctx.enc, ctx.S
        train, G = ctx.train, ctx.G
        grads = {}
        dfeat = dfeat.contiguous().view(dfeat.shape[0], -1).to(torch.float32)
        fh, fw = S["final_hw"]
        g, g2 = ops.avgpool_bwd(dfeat, fh, fw), None

        def bn_bwd(bn, st, g1, g2_, act, z, want_g_out=False, mask_from_z=False):
            r = ops.bn_backward(g1, g2_, None if mask_from_z else act, z, st.mean, st.rstd, bn.weight,
                                want_g_out=want_g_out, batch_stats=train, groups=G,
                                beta=bn.bias if mask_from_z else None)
            grads[bn.weight], grads[bn.bias] = r[1], r[2]
            return (r[0], r[3]) if want_g_out else r[0]

        for rec in reversed(S["blocks"]):
            blk, xin, z1, st1, a1, col2, z2, st2, a2, z3, st3, xs, zd, std, out = rec
            nb, hh, ww, cin = xin.shape
            planes = a1.shape[-1]
            dz3, gmask = bn_bwd(blk.bn3, st3, g, g2, out, z3, want_g_out=True)
            grads[blk.conv3.weight] = ops.conv_wgrad(a2, dz3, 1)
            d_a2 = ops.conv_gemm(dz3, ops.pack_conv_weight(blk.conv3.weight, ops.PACK_DGRAD), 1)
            dz2 = bn_bwd(blk.bn2, st2, d_a2, None, a2, z2, mask_from_z=True)
            if blk.stride == 1:
                grads[blk.conv2.weight] = ops.conv_wgrad(a1, dz2, 3)
                d_a1 = ops.conv_gemm(dz2, ops.pack_conv_weight(blk.conv2.weight, ops.PACK_DGRAD), 3)
            else:
                m2 = dz2.numel() // planes
                grads[blk.conv2.weight] = ops.conv_wgrad(col2.view(1, 1, m2, 9 * planes), dz2.view(1, 1, m2, planes), 1,
                                                         reduce_cin=planes, reduce_taps=9,
                                                         out_shape=(planes, planes, 3, 3))
                dcol = ops.gemm_rows(dz2.view(m2, planes), ops.pack_conv_weight(blk.conv2.weight, ops.PACK_DCOL))
                d_a1 = ops.col2im_3x3s2(dcol, nb, hh, ww, planes)
            dz1 = bn_bwd(blk.bn1, st1, d_a1, None, a1, z1, mask_from_z=True)
            grads[blk.conv1.weight] = ops.conv_wgrad(xin, dz1, 1)
            d_in = ops.conv_gemm(dz1, ops.pack_conv_weight(blk.conv1.weight, ops.PACK_DGRAD), 1)
            if blk.downsample is not None:
                dconv, dbn = blk.downsample[0], blk.downsample[1]
                dzd = bn_bwd(dbn, std, gmask, None, None, zd)
                grads[dconv.weight] = ops.conv_wgrad(xs, dzd, 1)
                d_xs = ops.conv_gemm(dzd, ops.pack_conv_weight(dconv.weight, ops.PACK_DGRAD), 1)
                if blk.stride == 2:
                    g, g2 = ops.scatter_add_s2(d_in, d_xs), None
                else:
                    g, g2 = d_in, d_xs
            else:
                g, g2 = d_in, gmask
        col0, z0, st0, a0, arg0 = S["stem"]
        d_a0 = ops.maxpool_bwd(g, arg0, g2)
        dz0 = bn_bwd(enc[1], st0, d_a0, None, a0, z0, mask_from_z=True)
        m0 = dz0.numel() // 64
        grads[enc[0].weight] = ops.conv_wgrad(col0.view(1, 1, m0, 192), dz0.view(1, 1, m0, 64), 1, reduce_cin=147,
                                              reduce_taps=1, out_shape=(64, 3, 7, 7))
        ctx.S = None
        # dL/dx of the stem is not produced: nothing on the IRFD path consumes the image gradient (train.py only sets
        # requires_grad on the batch as a side effect of the R1 penalty, SURVEY Q2).
        return (None, None, None, None, None) + tuple(grads.get(p) for p in enc._flat_params())


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
        if not x.is_cuda:
            raise ops._lib.IrfdError("ResNet50Encoder: CUDA tensors only (no CPU fallback on the IRFD hot path)")
        if x.dim() != 4 or x.shape[1] != 3:
            raise ops._lib.IrfdError(f"ResNet50Encoder: expected [N,3,H,W], got {tuple(x.shape)}")
        return self._run(x, 1, None)

    def _run(self, x, groups, stem_cols):
        params = self._flat_params()
        recorded = torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in params))
        if not self.training and not recorded:
            check_inference_shape(x)
            return _encoder_inference(self, x, stem_cols)  # inference: BN/ReLU/residual folded into the convs
        # refused before any launch, so the BatchNorm running buffers and counters stay untouched
        if not trainable_shape(x.size(0), x.shape[2], x.shape[3]):
            mode = "train-mode" if self.training else "differentiated eval-mode"
            raise ops._lib.IrfdError(f"ResNet50Encoder: a {mode} pass needs H, W multiples of 32 (W <= {MAX_STEM_W}) and "
                                     f"128-pixel tiles of whole rows / images at every stage, got {tuple(x.shape)}; "
                                     "eval-mode inference under no_grad runs at any 32 <= H, W")
        return _EncoderFn.apply(x, self, groups, stem_cols, recorded, *params)

    def can_group(self, x: torch.Tensor, groups: int) -> bool:
        """Grouped statistics need every layer's per-group row count to be a whole number of 128-pixel GEMM tiles."""
        if x.dim() != 4 or x.size(0) % groups:
            return False
        per_group = x.size(0) // groups
        return (per_group * (x.shape[2] // 32) * (x.shape[3] // 32)) % 128 == 0

    def forward_groups(self, x, groups: int, stem_cols=None):
        """x = `groups` batches stacked along dim 0; equivalent to `groups` consecutive calls (per-call BN stats).
        stem_cols: optional `ops.im2col_stem(x, 192)` computed by the caller (shared by encoders fed the same x)."""
        if not x.is_cuda:
            raise ops._lib.IrfdError("ResNet50Encoder: CUDA tensors only (no CPU fallback on the IRFD hot path)")
        if not self.can_group(x, groups):
            raise ops._lib.IrfdError(f"ResNet50Encoder.forward_groups: shape {tuple(x.shape)} cannot form {groups} groups")
        return self._run(x, groups, stem_cols)
