"""The three IRFD encoders (model.py:33-35: Ei, Ee, Ep) as ONE launch sequence.

`IRFD.forward` feeds the same images to three independent ResNet-50s (model.py:84-90), so layer l of Ei, Ee and Ep has
the same shape, the same input geometry and different weights.  Run one after the other (or on three streams) every
one of their 53 convs is a short launch dominated by prologue, first-load latency and tile quantisation (round 1: 22-32 %
of the tensor peak, 18-55 us launches against 6-26 us bounds).  `EncoderGroup` runs them in lockstep instead:

* activations of the E encoders are stacked encoder-major, `[E*N, H, W, C]` (N images per encoder);
* every conv is one grouped implicit GEMM (`irfd_conv_gemm_grouped`): the packed weights are stacked `[E*Cout, K]` and
  pixel tile t multiplies the rows of encoder t / tiles_per_encoder; the stem's im2col matrix is shared by all E;
* every BatchNorm is one launch sequence over `E x groups` statistic groups with per-encoder parameter sets
  (`irfd_bn_*_sets`): per-call batch statistics and running-buffer updates exactly as E x groups separate
  nn.BatchNorm2d calls (the reference calls each encoder on x_s and then on x_t);
* layout kernels (maxpool, stride-2 gathers, pools) are per image and run on the stacked tensor unchanged;
* weight gradients are one grouped split-K launch per layer (`irfd_conv_wgrad_grouped`: the CTAs of the three encoders
  share the single wave, a third of the fp32 partials), written straight into the caller's gradient buffers when
  `grad_targets` is set.

* the backward of every BatchNorm that feeds a conv (bn1, bn2) has its reduce pass inside the epilogue of that conv's
  data-gradient GEMM (`irfd_conv_gemm_bnbwd_grouped`: ReLU mask recomputed from z, per-tile sums of g and g*xhat), so the
  activation gradient is written once, already masked, and read once; the block outputs keep their ReLU mask as a bit
  plane (`irfd_bn_apply_sets(mask_bits)`) that bn3's backward reads instead of the activation.

This module is the only implementation of the encoder forward, backward and inference: a lone encoder call
(`ResNet50Encoder.forward` / `forward_groups`) runs as the one-member group `EncoderGroup([enc])`.

Numerically the forward of an E-encoder pass is E one-encoder passes: same kernels, same tiles, same summation order
per tile (tests/test_gpu_encoder_group.py: features and BN buffers bit-identical).  With E > 1 the backward sums the
BatchNorm statistics of bn1 / bn2 per 128-pixel tile instead of per row block: same terms in a different fp32 order
(IRFD_BN_FOLD=0 restores the separate launches and gradients equal to 3e-6).  A lone encoder never folds, so its
gradients do not depend on the setting.
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional

import torch
import torch.nn as nn

from . import ops
from .encoder import BN_EPS, BN_MOMENTUM, MAX_STEM_W, MIN_HW, ResNet50Encoder, trainable_shape


# IRFD_BN_FOLD (default 1): the reduce pass of bn1 / bn2's backward runs in the epilogue of the dgrad GEMM that produces
# their activation gradient (irfd_conv_gemm_bnbwd_grouped); 0 = separate reduce launch (experiments, A/B timing).
# IRFD_BN3_FOLD (default 0): the same for bn3 of every Bottleneck that is followed by an identity-shortcut block: the
# next block's conv1 data gradient adds the shortcut gradient, applies the ReLU mask and sums in its epilogue
# (irfd_conv_gemm_bnbwd_res_grouped).  Measured (B=32 pairs, same box): the BatchNorm family drops 7.3 -> 5.7 ms/step but
# the GEMM family grows 13.3 -> 15.7 ms (its epilogue streams two more wide tensors at < 3 TB/s) and the step gets
# slower (35.8 -> 36.3 ms), so it stays off.
fold_bn_reduce = os.environ.get("IRFD_BN_FOLD", "1") != "0"
fold_bn3_reduce = os.environ.get("IRFD_BN3_FOLD", "0") != "0"


def _stack_pack(convs, mode, kpad=0):
    return ops.pack_conv_weights_stacked([c.weight for c in convs], mode, kpad)


class _Stats:
    __slots__ = ("mean", "rstd")

    def __init__(self, mean, rstd):
        self.mean, self.rstd = mean, rstd


def _group_inference(grp: "EncoderGroup", x, col0=None):
    """Eval-mode, no-autograd forward of all encoders: every conv is ONE grouped kernel with the eval-mode BatchNorm,
    the ReLU and the Bottleneck residual add folded into its epilogue (per-encoder scale/shift vectors)."""
    encs = grp.encoders
    E = len(encs)
    x = x.contiguous().to(torch.float32)
    n, _, h, w = x.shape
    if col0 is None:
        col0 = ops.im2col_stem(x, 192)
    sc, sh = ops.bn_eval_affine_sets([e[1] for e in encs])
    a0 = ops.conv_gemm_affine_grouped(col0, _stack_pack([e[0] for e in encs], ops.PACK_FLAT, 192), 1, sc, sh, relu=True,
                                      wgroups=E, a_shared=True).view(E * n, ops.half_up(h), ops.half_up(w), 64)
    cur, _ = ops.maxpool_fwd(a0)
    for li in range(4, 8):
        for bi in range(len(encs[0][li])):
            blks = [e[li][bi] for e in encs]
            nb, hh, ww, _cin = cur.shape
            sc, sh = ops.bn_eval_affine_sets([b.bn1 for b in blks])
            a1 = ops.conv_gemm_affine_grouped(cur, _stack_pack([b.conv1 for b in blks], ops.PACK_FPROP), 1, sc, sh,
                                              relu=True, wgroups=E)
            planes = a1.shape[-1]
            sc, sh = ops.bn_eval_affine_sets([b.bn2 for b in blks])
            wk2 = _stack_pack([b.conv2 for b in blks], ops.PACK_FPROP)
            if blks[0].stride == 1:
                a2 = ops.conv_gemm_affine_grouped(a1, wk2, 3, sc, sh, relu=True, wgroups=E)
            else:
                col2 = ops.im2col_3x3s2(a1)
                a2 = ops.conv_gemm_affine_grouped(col2.view(1, 1, col2.shape[0], 9 * planes), wk2, 1, sc, sh, relu=True,
                                                  wgroups=E).view(nb, ops.half_up(hh), ops.half_up(ww), planes)
            if blks[0].downsample is not None:
                xs = ops.subsample2(cur) if blks[0].stride == 2 else cur
                sc, sh = ops.bn_eval_affine_sets([b.downsample[1] for b in blks])
                idn = ops.conv_gemm_affine_grouped(xs, _stack_pack([b.downsample[0] for b in blks], ops.PACK_FPROP), 1,
                                                   sc, sh, relu=False, wgroups=E)
            else:
                idn = cur
            sc, sh = ops.bn_eval_affine_sets([b.bn3 for b in blks])
            cur = ops.conv_gemm_affine_grouped(a2, _stack_pack([b.conv3 for b in blks], ops.PACK_FPROP), 1, sc, sh,
                                               res=idn, relu=True, wgroups=E)
    return ops.avgpool_fwd(cur).view(E, n, -1, 1, 1)


class _EncoderGroupFn(torch.autograd.Function):
    """forward(x [N,3,H,W], group, stat_groups, col0, recorded, image_grad, *params) -> features [E, N, 2048, 1, 1] fp32.

    Train mode, and eval mode with autograd (E == 1 only); eval-mode forwards without autograd go through
    _group_inference.  params = the encoders' parameters, encoder after encoder, in _flat_params() order.
    In train mode x stacks `stat_groups` independent batches along dim 0 (IRFD: source and target images): BatchNorm
    statistics are per (encoder, group) and each encoder's running buffers are updated group by group, like separate
    calls.  In eval mode every BatchNorm normalises with its running statistics and no buffer changes.
    image_grad: the backward also returns dL/dx, summed over the E encoders (the caller's image came out of a
    differentiable computation); otherwise x gets no gradient and no launch is spent on it."""

    @staticmethod
    def forward(ctx, x, grp, stat_groups, col0, recorded, image_grad, *params):
        encs: List[ResNet50Encoder] = grp.encoders
        E = len(encs)
        train = encs[0].training
        assert train or E == 1
        G = stat_groups if train else 1  # eval mode: the shared running statistics, no groups needed
        GT = E * G  # statistic groups of a stacked tensor: encoder-major, then the caller's groups
        # reentrant-checkpoint semantics of the reference (model.py:84-90, SURVEY Q3): a differentiated pass updates the
        # BN running buffers twice, forward order then reverse order
        U = 2 if (train and recorded and all(getattr(e, "_recompute_bn_update", False) for e in encs)) else 1
        ctx.image_grad = image_grad and ctx.needs_input_grad[0]
        ctx.x_dtype = x.dtype
        x = x.contiguous().to(torch.float32)
        n, _, h, w = x.shape
        # the stem's dcol GEMM gives each encoder whole 128-pixel tiles of the linear geometry (trainable shapes: H and
        # W are multiples of 32, so n * H/2 * W/2 is a multiple of 256)
        assert not ctx.image_grad or (n * (h // 2) * (w // 2)) % 128 == 0

        def conv(xx, wk, ksize, **kw):
            """Forward conv; in train mode its epilogue also gathers the BatchNorm statistics."""
            if train:
                return ops.conv_gemm_grouped(xx, wk, ksize, ops.EPI_STATS, wgroups=E, **kw)
            return ops.conv_gemm_grouped(xx, wk, ksize, wgroups=E, **kw), None, None

        def stats(bns, s, q, rows_total):
            if not train:
                return _Stats(bns[0].running_mean, ops.bn_eval_rstd(bns[0].running_var, BN_EPS))
            mean, rstd = ops.bn_finalize_sets(s, q, rows_total // GT, BN_EPS, BN_MOMENTUM,
                                              [b.running_mean for b in bns], [b.running_var for b in bns], U, G, E)
            return _Stats(mean, rstd)

        def apply(z, st, bns, relu=True, res=None, bn2=None, want_mask=False):
            return ops.bn_apply_sets(z, st.mean, st.rstd, [b.weight for b in bns], [b.bias for b in bns], res=res,
                                     bn2=bn2, relu=relu, groups=GT, want_mask=want_mask)

        S = {}
        if col0 is None:
            col0 = ops.im2col_stem(x, 192)
        bn0 = [e[1] for e in encs]
        z0, s, q = conv(col0, _stack_pack([e[0] for e in encs], ops.PACK_FLAT, 192), 1, a_shared=True)
        h1, w1 = h // 2, w // 2
        z0 = z0.view(E * n, h1, w1, 64)
        st0 = stats(bn0, s, q, E * n * h1 * w1)
        a0 = apply(z0, st0, bn0)
        cur, arg0 = ops.maxpool_fwd(a0)
        S["stem"] = (col0, z0, st0, a0, arg0)
        S["blocks"] = []
        for li in range(4, 8):
            for bi in range(len(encs[0][li])):
                blks = [e[li][bi] for e in encs]
                xin = cur
                nb, hh, ww, _cin = xin.shape
                z1, s, q = conv(xin, _stack_pack([b.conv1 for b in blks], ops.PACK_FPROP), 1)
                bn1 = [b.bn1 for b in blks]
                st1 = stats(bn1, s, q, nb * hh * ww)
                a1 = apply(z1, st1, bn1)
                planes = a1.shape[-1]
                wk2 = _stack_pack([b.conv2 for b in blks], ops.PACK_FPROP)
                col2 = None
                if blks[0].stride == 1:
                    z2, s, q = conv(a1, wk2, 3)
                    ho, wo = hh, ww
                else:
                    col2 = ops.im2col_3x3s2(a1)
                    ho, wo = hh // 2, ww // 2
                    z2, s, q = conv(col2.view(1, 1, col2.shape[0], 9 * planes), wk2, 1)
                    z2 = z2.view(nb, ho, wo, planes)
                bn2 = [b.bn2 for b in blks]
                st2 = stats(bn2, s, q, nb * ho * wo)
                a2 = apply(z2, st2, bn2)
                z3, s, q = conv(a2, _stack_pack([b.conv3 for b in blks], ops.PACK_FPROP), 1)
                bn3 = [b.bn3 for b in blks]
                st3 = stats(bn3, s, q, nb * ho * wo)
                xs = zd = std = None
                if blks[0].downsample is not None:
                    xs = ops.subsample2(xin) if blks[0].stride == 2 else xin
                    zd, s, q = conv(xs, _stack_pack([b.downsample[0] for b in blks], ops.PACK_FPROP), 1)
                    dbn = [b.downsample[1] for b in blks]
                    std = stats(dbn, s, q, nb * ho * wo)
                    out = apply(z3, st3, bn3, res=zd, want_mask=recorded,
                                bn2=(std.mean, std.rstd, [b.weight for b in dbn], [b.bias for b in dbn]))
                else:
                    out = apply(z3, st3, bn3, res=xin, want_mask=recorded)
                out, obits = out if recorded else (out, None)
                # the backward pass needs the block output only as a ReLU mask: keep the bit plane (1/16 of the bytes
                # to read back), the tensor itself lives on as the next block's input
                S["blocks"].append((li, blks, xin, z1, st1, a1, col2, z2, st2, a2, z3, st3, xs, zd, std, obits))
                cur = out
        feat = ops.avgpool_fwd(cur)
        if train:  # nn.BatchNorm2d bookkeeping (one fused increment)
            torch._foreach_add_([c for e in encs for c in e._bn_counters()], G * U)
        S["final_hw"] = (cur.shape[1], cur.shape[2])
        S["x_shape"] = (n, h, w)
        ctx.grp, ctx.S, ctx.G, ctx.train = grp, S, G, train
        return feat.view(E, n, -1, 1, 1)

    @staticmethod
    def backward(ctx, dfeat):
        grp, S, G, train = ctx.grp, ctx.S, ctx.G, ctx.train
        encs = grp.encoders
        E = len(encs)
        GT = E * G
        # the folded reduce passes sum in another fp32 order, which the train-mode stack amplifies
        # (scripts/fold_probe.py): a lone encoder keeps the separate launches, so its gradients do not depend on the
        # setting
        fold, fold3 = fold_bn_reduce and E > 1, fold_bn3_reduce and E > 1
        cb = grp._bwd_cb
        # parameter gradients of the generator's dense layers may still be in flight on the side stream (_FCFn.backward)
        ops.side_stream(dfeat.device).join()
        if cb is not None:
            cb("pre", None)
        targets: Optional[Dict[nn.Parameter, torch.Tensor]] = grp.grad_targets
        grads = {}
        dfeat = dfeat.contiguous().view(dfeat.shape[0] * dfeat.shape[1], -1).to(torch.float32)
        fh, fw = S["final_hw"]
        g, g2 = ops.avgpool_bwd(dfeat, fh, fw), None

        def tgt(p):
            """Where a parameter's gradient goes: the caller's buffer (written in place) or a fresh tensor."""
            if targets is not None:
                return targets[p]
            t = torch.empty_like(p, dtype=torch.float32)
            grads[p] = t
            return t

        def bn_bwd(bns, st, g1, g2_, act, z, want_g_out=False, mask_from_z=False, act_bits=None):
            r = ops.bn_backward_sets(g1, g2_, None if mask_from_z else act, z, st.mean, st.rstd,
                                     [b.weight for b in bns], [b.bias for b in bns] if mask_from_z else None,
                                     dgammas=[tgt(b.weight) for b in bns], dbetas=[tgt(b.bias) for b in bns],
                                     want_g_out=want_g_out, batch_stats=train, groups=GT, act_bits=act_bits)
            return (r[0], r[3]) if want_g_out else r[0]

        def dgrad_bn(dy, convs, ksize, bns, st, z):
            """Data gradient through `convs` into relu(BN(z)), then that BatchNorm's backward.  Launches the dgrad GEMM
            and returns the closure that launches the rest (the caller forks the weight gradient in between, so that it
            runs beside the HBM-bound BN pass) and returns dz."""
            wk = _stack_pack(convs, ops.PACK_DGRAD)
            if not fold:
                d_a = ops.conv_gemm_grouped(dy, wk, ksize, wgroups=E)
                return lambda: bn_bwd(bns, st, d_a, None, None, z, mask_from_z=True)
            gm, part = ops.conv_gemm_bnbwd_grouped(dy, wk, ksize, z, st.mean, st.rstd, [b.weight for b in bns],
                                                   [b.bias for b in bns], GT)
            return lambda: ops.bn_backward_finish_sets(gm, z, st.mean, st.rstd, [b.weight for b in bns], part,
                                                       dgammas=[tgt(b.weight) for b in bns],
                                                       dbetas=[tgt(b.bias) for b in bns], groups=GT)[0]

        side = ops.side_stream(dfeat.device)

        def wgrad(convs, xx, dy, ksize, **kw):
            """All E weight gradients of one layer in one split-K launch pair (the CTAs of the three encoders share the
            wave, so each encoder needs a third of the fp32 partials three separate launches would write), on the side
            stream: the tensor-bound wgrad overlaps the HBM-bound BatchNorm backward of the next layer."""
            dws = [tgt(c.weight) for c in convs]   # allocated on the main stream
            side.launch(lambda: ops.conv_wgrad_grouped(xx, dy, ksize, dws, **kw), xx, dy, *dws)

        cur_li = None
        pre = None   # (masked output gradient, partial sums) of this block's bn3 when the previous iteration formed them
        blocks = S["blocks"]
        for bidx in range(len(blocks) - 1, -1, -1):
            li, blks, xin, z1, st1, a1, col2, z2, st2, a2, z3, st3, xs, zd, std, obits = blocks[bidx]
            if cur_li is not None and li != cur_li and cb is not None:
                cb("stage", cur_li)  # every gradient of ResNet stage `cur_li` (all encoders) has been written
            cur_li = li
            nb, hh, ww, _cin = xin.shape
            planes = a1.shape[-1]
            if pre is not None:
                gmask, part3 = pre
                bn3 = [b.bn3 for b in blks]
                dz3 = ops.bn_backward_finish_sets(gmask, z3, st3.mean, st3.rstd, [b.weight for b in bn3], part3,
                                                  dgammas=[tgt(b.weight) for b in bn3],
                                                  dbetas=[tgt(b.bias) for b in bn3], groups=GT)[0]
                pre = None
            else:
                dz3, gmask = bn_bwd([b.bn3 for b in blks], st3, g, g2, None, z3, want_g_out=True, act_bits=obits)
            # dgrad first, wgrad second: the persistent dgrad takes the SMs, the wgrad (side stream) follows it and
            # runs beside the BatchNorm backward that consumes the dgrad's output
            finish = dgrad_bn(dz3, [b.conv3 for b in blks], 1, [b.bn2 for b in blks], st2, z2)
            wgrad([b.conv3 for b in blks], a2, dz3, 1)
            dz2 = finish()
            if blks[0].stride == 1:
                finish = dgrad_bn(dz2, [b.conv2 for b in blks], 3, [b.bn1 for b in blks], st1, z1)
                wgrad([b.conv2 for b in blks], a1, dz2, 3)
                dz1 = finish()
            else:
                m2 = dz2.numel() // planes
                dcol = ops.conv_gemm_grouped(dz2.view(1, 1, m2, planes),
                                             _stack_pack([b.conv2 for b in blks], ops.PACK_DCOL), 1, wgroups=E)
                wgrad([b.conv2 for b in blks], col2, dz2.view(m2, planes), 1, reduce_cin=planes, reduce_taps=9)
                d_a1 = ops.col2im_3x3s2(dcol.view(m2, 9 * planes), nb, hh, ww, planes)
                dz1 = bn_bwd([b.bn1 for b in blks], st1, d_a1, None, a1, z1, mask_from_z=True)
            wk1 = _stack_pack([b.conv1 for b in blks], ops.PACK_DGRAD)
            if blks[0].downsample is None and fold3:
                # identity shortcut: this block's input gradient is conv1's data gradient + the masked output gradient,
                # and the input is the previous block's relu(bn3(z3) + shortcut): that BatchNorm's reduce pass runs here
                prev = blocks[bidx - 1]
                pre = ops.conv_gemm_bnbwd_res_grouped(dz1, wk1, 1, prev[10], prev[11].mean, prev[11].rstd, gmask,
                                                      prev[15], GT, wgroups=E)
                wgrad([b.conv1 for b in blks], xin, dz1, 1)
                continue
            d_in = ops.conv_gemm_grouped(dz1, wk1, 1, wgroups=E)
            wgrad([b.conv1 for b in blks], xin, dz1, 1)
            if blks[0].downsample is not None:
                dzd = bn_bwd([b.downsample[1] for b in blks], std, gmask, None, None, zd)
                d_xs = ops.conv_gemm_grouped(dzd, _stack_pack([b.downsample[0] for b in blks], ops.PACK_DGRAD), 1,
                                             wgroups=E)
                wgrad([b.downsample[0] for b in blks], xs, dzd, 1)
                if blks[0].stride == 2:
                    g, g2 = ops.scatter_add_s2(d_in, d_xs), None
                else:
                    g, g2 = d_in, d_xs
            else:
                g, g2 = d_in, gmask
        if cb is not None and cur_li is not None:
            cb("stage", cur_li)
        col0, z0, st0, a0, arg0 = S["stem"]
        d_a0 = ops.maxpool_bwd(g, arg0, g2)
        dz0 = bn_bwd([e[1] for e in encs], st0, d_a0, None, a0, z0, mask_from_z=True)
        # the stem's im2col matrix is shared: every encoder reads the same rows
        wgrad([e[0] for e in encs], col0, dz0.view(-1, 64), 1, x_shared=True, reduce_cin=147, reduce_taps=1)
        dx = None
        if ctx.image_grad:
            # dL/dx of the 7x7/2 stem conv: dcol = dz0 @ W per encoder (one grouped GEMM, [E*P, 192] bf16), then the
            # col2im gather sums the E encoders' columns onto the image; it runs beside the stem's weight gradient
            dcol = ops.conv_gemm_grouped(dz0.view(1, 1, -1, 64), _stack_pack([e[0] for e in encs], ops.PACK_FLAT_T, 192),
                                         1, wgroups=E)
            dx = ops.col2im_stem(dcol.view(-1, 192), E, *S["x_shape"])
            if ctx.x_dtype != torch.float32:
                dx = dx.to(ctx.x_dtype)
        side.join()
        if cb is not None:
            cb("stage", 3)   # the stem (Sequential indices 0, 1)
            cb("post", None)
        ctx.S = None
        if targets is not None:
            return (dx,) + (None,) * (5 + sum(len(e._flat_params()) for e in encs))
        return (dx, None, None, None, None, None) + tuple(grads.get(p) for e in encs for p in e._flat_params())


class EncoderGroup:
    """Lockstep runner for encoders of identical architecture fed the same images (not an nn.Module: the encoders stay
    registered where the reference has them, `IRFD.Ei / .Ee / .Ep`)."""

    def __init__(self, encoders: List[ResNet50Encoder]):
        self.encoders = list(encoders)
        # optional {parameter: fp32 tensor of the parameter's shape}: backward WRITES each gradient there (overwrite,
        # one backward per step) and returns no gradient to autograd — the trainer's flat gradient buffers
        self.grad_targets: Optional[Dict[nn.Parameter, torch.Tensor]] = None
        self._bwd_cb = None  # data-parallel trainer: called with ("pre"|"stage"|"post", stage index) during backward

    def can_run(self, x: torch.Tensor, groups: int, recorded: bool = False) -> bool:
        """Whether x ([N,3,H,W], `groups` batches stacked along dim 0) runs as one grouped pass.  recorded: autograd
        records the pass, so an eval-mode pass needs the train-mode kernels' shapes too (the backward runs them)."""
        encs = self.encoders
        if not (x.is_cuda and x.dim() == 4 and x.shape[1] == 3 and x.size(0) % groups == 0):
            return False
        if len({e.training for e in encs}) != 1:
            return False
        E, n = len(encs), x.size(0)
        h, w = x.shape[2], x.shape[3]
        if not encs[0].training and not recorded:
            # eval mode: every grouped launch must give each encoder whole tiles of its x.size(0) images (ONE statistic
            # group, the running statistics): the flat GEMMs (stem, 1x1, stride-2 im2col) need a multiple of 128 pixels
            # per encoder, the 3x3 convs a tile geometry with whole images per encoder
            if h < MIN_HW or w < MIN_HW or w > MAX_STEM_W:
                return False
            for i, (hs, ws) in enumerate(ops.resnet_stage_hw(h, w)):
                for k in ((1, 3) if i > 0 else (1,)):
                    if ops.conv_geometry(E * n, hs, ws, k, E) is None:
                        return False
            return True
        if not trainable_shape(n, h, w):
            return False
        # more than one (encoder, statistic group): each needs whole 128-pixel tiles at every stage (layer4 is the
        # smallest, (H/32) x (W/32) pixels per image)
        return E * groups == 1 or (n // groups * (h // 32) * (w // 32)) % 128 == 0

    def __call__(self, x: torch.Tensor, groups: int = 1, stem_cols=None, image_grad: Optional[bool] = None):
        """Returns features [E, N, 2048, 1, 1]: out[e] == encoders[e].forward_groups(x, groups).
        image_grad: whether the backward returns dL/dx.  Default: when x came out of a differentiable computation
        (x.grad_fn is set); a leaf image, such as a batch of training data, gets no gradient, as before.  A caller that
        stacks its images first decides from its own tensors, since the stacking op always has a grad_fn."""
        encs = self.encoders
        recorded = torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for e in encs
                                                                       for p in e.parameters()))
        if not self.can_run(x, groups, recorded):
            raise ops._lib.IrfdError(f"EncoderGroup: shape {tuple(x.shape)} / modes cannot run as one grouped pass")
        if not encs[0].training:
            if not recorded:
                return _group_inference(self, x, stem_cols)
            if len(encs) > 1:
                raise ops._lib.IrfdError("EncoderGroup: eval-mode passes with autograd run one encoder at a time")
        if image_grad is None:
            image_grad = x.grad_fn is not None
        params = [p for e in encs for p in e._flat_params()]
        return _EncoderGroupFn.apply(x, self, groups, stem_cols, recorded, bool(image_grad), *params)
