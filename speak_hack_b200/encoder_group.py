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

Numerically the forward of the grouped pass is the per-encoder pass: same kernels, same tiles, same summation order
per tile (tests/test_gpu_encoder_group.py: features and BN buffers bit-identical).  The backward sums the BatchNorm
statistics of bn1 / bn2 per 128-pixel tile instead of per row block: same terms in a different fp32 order
(IRFD_BN_FOLD=0 restores the per-encoder launches and gradients equal to 3e-6).
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
    """forward(x [N,3,H,W] fp32, group, stat_groups, col0, recorded, *params) -> features [E, N, 2048, 1, 1] fp32.

    Train mode only (eval-mode forwards without autograd go through _group_inference; eval-mode forwards WITH autograd
    through the per-encoder path).  params = the encoders' parameters, encoder after encoder, in _flat_params() order.
    x stacks `stat_groups` independent batches along dim 0 (IRFD: source and target images): BatchNorm statistics are
    per (encoder, group) and each encoder's running buffers are updated group by group, like separate calls."""

    @staticmethod
    def forward(ctx, x, grp, stat_groups, col0, recorded, *params):
        encs: List[ResNet50Encoder] = grp.encoders
        E = len(encs)
        G = stat_groups
        GT = E * G  # statistic groups of a stacked tensor: encoder-major, then the caller's groups
        # reentrant-checkpoint semantics of the reference (model.py:84-90, SURVEY Q3): a differentiated pass updates the
        # BN running buffers twice, forward order then reverse order
        U = 2 if (recorded and all(getattr(e, "_recompute_bn_update", False) for e in encs)) else 1
        x = x.contiguous().to(torch.float32)
        n, _, h, w = x.shape

        def stats(bns, s, q, rows_total):
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
        z0, s, q = ops.conv_gemm_grouped(col0, _stack_pack([e[0] for e in encs], ops.PACK_FLAT, 192), 1, ops.EPI_STATS,
                                         wgroups=E, a_shared=True)
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
                z1, s, q = ops.conv_gemm_grouped(xin, _stack_pack([b.conv1 for b in blks], ops.PACK_FPROP), 1,
                                                 ops.EPI_STATS, wgroups=E)
                bn1 = [b.bn1 for b in blks]
                st1 = stats(bn1, s, q, nb * hh * ww)
                a1 = apply(z1, st1, bn1)
                planes = a1.shape[-1]
                wk2 = _stack_pack([b.conv2 for b in blks], ops.PACK_FPROP)
                col2 = None
                if blks[0].stride == 1:
                    z2, s, q = ops.conv_gemm_grouped(a1, wk2, 3, ops.EPI_STATS, wgroups=E)
                    ho, wo = hh, ww
                else:
                    col2 = ops.im2col_3x3s2(a1)
                    ho, wo = hh // 2, ww // 2
                    z2, s, q = ops.conv_gemm_grouped(col2.view(1, 1, col2.shape[0], 9 * planes), wk2, 1, ops.EPI_STATS,
                                                     wgroups=E)
                    z2 = z2.view(nb, ho, wo, planes)
                bn2 = [b.bn2 for b in blks]
                st2 = stats(bn2, s, q, nb * ho * wo)
                a2 = apply(z2, st2, bn2)
                z3, s, q = ops.conv_gemm_grouped(a2, _stack_pack([b.conv3 for b in blks], ops.PACK_FPROP), 1,
                                                 ops.EPI_STATS, wgroups=E)
                bn3 = [b.bn3 for b in blks]
                st3 = stats(bn3, s, q, nb * ho * wo)
                xs = zd = std = None
                if blks[0].downsample is not None:
                    xs = ops.subsample2(xin) if blks[0].stride == 2 else xin
                    zd, s, q = ops.conv_gemm_grouped(xs, _stack_pack([b.downsample[0] for b in blks], ops.PACK_FPROP), 1,
                                                     ops.EPI_STATS, wgroups=E)
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
        counters = [c for e in encs for c in e._bn_counters()]
        torch._foreach_add_(counters, G * U)  # nn.BatchNorm2d bookkeeping (one fused increment)
        S["final_hw"] = (cur.shape[1], cur.shape[2])
        ctx.grp, ctx.S, ctx.G = grp, S, G
        return feat.view(E, n, -1, 1, 1)

    @staticmethod
    def backward(ctx, dfeat):
        grp, S, G = ctx.grp, ctx.S, ctx.G
        encs = grp.encoders
        E = len(encs)
        GT = E * G
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
                                     want_g_out=want_g_out, batch_stats=True, groups=GT, act_bits=act_bits)
            return (r[0], r[3]) if want_g_out else r[0]

        def dgrad_bn(dy, convs, ksize, bns, st, z):
            """Data gradient through `convs` into relu(BN(z)), then that BatchNorm's backward.  Launches the dgrad GEMM
            and returns the closure that launches the rest (the caller forks the weight gradient in between, so that it
            runs beside the HBM-bound BN pass) and returns dz."""
            wk = _stack_pack(convs, ops.PACK_DGRAD)
            if not fold_bn_reduce:
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
            if blks[0].downsample is None and fold_bn3_reduce:
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
        side.join()
        if cb is not None:
            cb("stage", 3)   # the stem (Sequential indices 0, 1)
            cb("post", None)
        ctx.S = None
        # dL/dx of the stem is not produced (nothing on the IRFD path consumes the image gradient, SURVEY Q2)
        if targets is not None:
            return (None,) * (5 + sum(len(e._flat_params()) for e in encs))
        return (None, None, None, None, None) + tuple(grads.get(p) for e in encs for p in e._flat_params())


class EncoderGroup:
    """Lockstep runner for encoders of identical architecture fed the same images (not an nn.Module: the encoders stay
    registered where the reference has them, `IRFD.Ei / .Ee / .Ep`)."""

    def __init__(self, encoders: List[ResNet50Encoder]):
        self.encoders = list(encoders)
        # optional {parameter: fp32 tensor of the parameter's shape}: backward WRITES each gradient there (overwrite,
        # one backward per step) and returns no gradient to autograd — the trainer's flat gradient buffers
        self.grad_targets: Optional[Dict[nn.Parameter, torch.Tensor]] = None
        self._bwd_cb = None  # data-parallel trainer: called with ("pre"|"stage"|"post", stage index) during backward

    def can_run(self, x: torch.Tensor, groups: int) -> bool:
        encs = self.encoders
        if not (x.is_cuda and x.dim() == 4 and x.shape[1] == 3 and x.size(0) % groups == 0):
            return False
        if len({e.training for e in encs}) != 1:
            return False
        h, w = x.shape[2], x.shape[3]
        if not encs[0].training:
            # eval mode: every grouped launch must give each encoder whole tiles of its x.size(0) images (ONE statistic
            # group, the running statistics): the flat GEMMs (stem, 1x1, stride-2 im2col) need a multiple of 128 pixels
            # per encoder, the 3x3 convs a tile geometry with whole images per encoder
            if h < MIN_HW or w < MIN_HW or w > MAX_STEM_W:
                return False
            E, n = len(encs), x.size(0)
            for i, (hs, ws) in enumerate(ops.resnet_stage_hw(h, w)):
                for k in ((1, 3) if i > 0 else (1,)):
                    if ops.conv_geometry(E * n, hs, ws, k, E) is None:
                        return False
            return True
        if h % 32 or w % 32 or not trainable_shape(x.size(0), h, w):
            return False
        per_group = x.size(0) // groups
        return (per_group * (h // 32) * (w // 32)) % 128 == 0

    def __call__(self, x: torch.Tensor, groups: int = 1, stem_cols=None):
        """Returns features [E, N, 2048, 1, 1]: out[e] == encoders[e].forward_groups(x, groups)."""
        if not self.can_run(x, groups):
            raise ops._lib.IrfdError(f"EncoderGroup: shape {tuple(x.shape)} / modes cannot run as one grouped pass")
        encs = self.encoders
        params = [p for e in encs for p in e._flat_params()]
        recorded = torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in params))
        if not encs[0].training:
            if recorded:
                raise ops._lib.IrfdError("EncoderGroup: eval-mode passes with autograd run per encoder")
            return _group_inference(self, x, stem_cols)
        return _EncoderGroupFn.apply(x, self, groups, stem_cols, recorded, *params)
