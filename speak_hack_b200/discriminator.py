"""StyleDiscriminator — styleganv1.py:637-695 (SURVEY.md §8(f) row N1).

Same classes, constructor signatures and state_dict keys as the reference (`D.*`, spectral-norm `weight_orig / weight_u /
weight_v`), so checkpoints move both ways and a seeded construction consumes the RNG identically.

Forward, first-order backward (gradient w.r.t. the image AND all parameters) and the second-order path of the R1
penalty run on the sm_100a kernels: `irfd_from_rgb_fwd` for the 1x1 RGB stem, the tcgen05 implicit-GEMM convs with the
`+ bias -> leaky_relu(0.2)` tail fused as their epilogue (3x3 stride 1 directly, 3x3 stride 2 through the same NHWC
im2col the encoders use), NHWC bf16 activations, fp32 dense head.  That covers the reference's generator step
(train.py:197-201: `D(x_recon)` -> BCE -> backward into Gd) and its discriminator step (train.py:157-183).

R1 (train.py:246-255) differentiates THROUGH the image gradient: `torch.autograd.grad(D(x).sum(), x,
create_graph=True)` followed by a backward of `grad.pow(2).sum()`.  The reference's own `compute_r1_reg` works on this
module unchanged: when `_DiscFn.backward` runs with grad mode enabled (create_graph=True) it returns the image gradient
as the output of a second autograd node, `_DiscGradFn`, whose backward is the closed-form second-order chain.  D is
piecewise linear in x, so with the leaky-ReLU masks m_l of the forward pass held fixed

    g_{l-1} = C_l^T (m_l * g_l)                         (image-gradient chain, u_l = m_l * g_l)
    d<g_x, p_x>/dW_l = wgrad(input = p_{l-1}, output gradient = u_l),   p_l = m_l * (C_l p_{l-1})

i.e. one masked forward chain on p_x (the gradient arriving at g_x) and one wgrad per layer, all on the same kernels
as the first-order path.  Biases only enter through the masks: their second-order gradient is zero, and so is the
image's.  `D.r1_penalty(x)` is the same computation fused into one node (it skips the first-order weight gradients a
generic double backward cannot know it does not need).

Spectral normalisation itself (one power iteration on each [Cout, Cin*k*k] matrix, styleganv1.py:643-654 via
torch.nn.utils.spectral_norm) runs in its torch hook by default, which keeps `weight_u / weight_v` updates and the
backward through sigma exactly the reference's.  Inside `D.native_spectral_norm()` (the graphed discriminator step,
trainer.IRFDDiscriminatorStep(use_cuda_graph=True)) the same computation runs on the sm_100a kernels instead, all
layers of a call in 3 launches forward and 2 backward (_SpectralNormFn).  There is no PyTorch composition of the
network in this module: inputs the kernels cannot take (CPU tensors, other resolutions, channel counts that are not
multiples of 64) raise.
"""
from __future__ import annotations

import contextlib

import numpy as np
import torch
import torch.nn as nn
from torch.autograd.function import once_differentiable
from torch.nn.utils import spectral_norm

from . import ops


class DiscriminatorBlock(nn.Module):
    def __init__(self, in_channels, out_channels):
        super().__init__()
        self.conv1 = spectral_norm(nn.Conv2d(in_channels, in_channels, kernel_size=3, padding=1))
        self.conv2 = spectral_norm(nn.Conv2d(in_channels, out_channels, kernel_size=3, padding=1, stride=2))

    def forward(self, x):
        raise ops._lib.IrfdError("DiscriminatorBlock runs fused inside StyleDiscriminator (NHWC bf16 activations between "
                                 "its convs); call StyleDiscriminator")


def _normalized_weight(m: nn.Module) -> torch.Tensor:
    """Run the module's spectral-norm pre-forward hook (power iteration in train mode, buffers updated in place exactly
    like a call of the module would) and return `weight = weight_orig / sigma`, attached to autograd."""
    for hook in m._forward_pre_hooks.values():
        hook(m, None)
    return m.weight


class _SpectralNormFn(torch.autograd.Function):
    """forward(power_iteration, n, weight_orig x n, weight_u x n, weight_v x n) -> n spectrally normalised weights
    W_sn = weight_orig / sigma, on the sm_100a kernels (ops.spectral_norm_fwd): in train mode one power iteration per
    layer updates weight_u / weight_v in place, as torch.nn.utils.spectral_norm's hook does.  Backward treats u and v as
    constants, like the hook (it differentiates weight_orig / sigma with u, v cloned):
    dL/dweight_orig = (G - <G, W_sn> u v^T) / sigma."""

    @staticmethod
    def forward(ctx, power_iteration, n, *tensors):
        ws, us, vs = tensors[:n], tensors[n: 2 * n], tensors[2 * n:]
        outs, u_save, v_save, sigma = ops.spectral_norm_fwd(ws, us, vs, power_iteration)
        ctx.n = n
        ctx.save_for_backward(u_save, v_save, sigma, *outs)
        return tuple(outs)

    @staticmethod
    @once_differentiable
    def backward(ctx, *grads):
        u_save, v_save, sigma, *outs = ctx.saved_tensors
        dws = ops.spectral_norm_bwd(grads, outs, u_save, v_save, sigma)
        return (None, None) + tuple(dws) + (None,) * (2 * ctx.n)


_ones_cache = {}


def _ones(c: int, device) -> torch.Tensor:
    key = (c, device.index)
    if key not in _ones_cache:
        _ones_cache[key] = torch.ones(c, dtype=torch.float32, device=device)
    return _ones_cache[key]


def _pack(w: torch.Tensor, mode: int) -> torch.Tensor:
    # the normalised weight is a fresh tensor every forward: repack without the (pointer-keyed) cache
    return ops._pack_conv_weight(w.contiguous(), mode)


def _disc_forward(x, nblocks, wb):
    """Returns (logits [B,1], saved).  Layer order in wb: rgb, (conv1, conv2) x nblocks, final, dense0, dense1; each as
    (spectrally normalised weight, bias)."""
    x = x.contiguous().to(torch.float32)
    dev = x.device
    w_rgb, b_rgb = wb[0], wb[1]
    c0 = w_rgb.shape[0]
    a = ops.from_rgb_fwd(x, w_rgb.reshape(c0, 3).contiguous(), b_rgb.contiguous())
    acts, cols = [a], []
    i = 2
    for _ in range(nblocks):
        w1, b1, w2, b2 = wb[i], wb[i + 1], wb[i + 2], wb[i + 3]
        i += 4
        cin, cout = w1.shape[0], w2.shape[0]
        y1 = ops.conv_gemm_affine(a, _pack(w1, ops.PACK_FPROP), 3, _ones(cin, dev), b1.contiguous(), relu=2)
        nb, hh, ww, _ = y1.shape
        col = ops.im2col_3x3s2(y1)
        y2 = ops.conv_gemm_affine(col.view(1, 1, col.shape[0], 9 * cin), _pack(w2, ops.PACK_FPROP), 1, _ones(cout, dev),
                                  b2.contiguous(), relu=2).view(nb, hh // 2, ww // 2, cout)
        acts += [y1, y2]
        cols.append(col)
        a = y2
    w_f, b_f = wb[i], wb[i + 1]
    yf = ops.conv_gemm_affine(a, _pack(w_f, ops.PACK_FPROP), 3, _ones(w_f.shape[0], dev), b_f.contiguous(), relu=2)
    acts.append(yf)
    pooled = ops.avgpool_fwd(yf)
    wd0, bd0, wd1, bd1 = wb[i + 2], wb[i + 3], wb[i + 4], wb[i + 5]
    hdn = ops.linear_fwd(pooled, wd0.contiguous(), bd0.contiguous(), 1.0, 1.0, lrelu=True)
    out = ops.linear_fwd(hdn, wd1.contiguous(), bd1.contiguous(), 1.0, 1.0, lrelu=False)
    return out, {"x": x, "acts": acts, "cols": cols, "pooled": pooled, "hdn": hdn}


def _disc_backward(S, nblocks, wb, dout, need_dx=True, need_dw=True, keep_u=False):
    """First-order backward chain.  Returns (dx or None, grads aligned with wb (None where not computed), U) where U
    holds every layer's masked upstream gradient u_l = lrelu'(z_l) * dL/dy_l (the R1 chain needs them)."""
    acts, cols, pooled, hdn = S["acts"], S["cols"], S["pooled"], S["hdn"]
    grads = [None] * len(wb)
    U = {"blk": [None] * nblocks}
    i = 2 + 4 * nblocks
    wd0, wd1 = wb[i + 2], wb[i + 4]
    dout = dout.contiguous().to(torch.float32)
    dh, dw1_, db1_ = ops.linear_bwd(dout, hdn, wd1.contiguous(), 1.0, 1.0, need_dw=need_dw)
    dz0 = ops.lrelu_bwd(dh, hdn)
    dpool, dw0_, db0_ = ops.linear_bwd(dz0, pooled, wd0.contiguous(), 1.0, 1.0, need_dw=need_dw)
    grads[i + 2], grads[i + 3], grads[i + 4], grads[i + 5] = dw0_, db0_, dw1_, db1_
    U["head"] = dz0
    yf = acts[-1]
    g = ops.avgpool_bwd(dpool, yf.shape[1], yf.shape[2])
    dz, grads[i + 1] = ops.bias_lrelu_bwd(g, yf)
    U["final"] = dz
    if need_dw:
        grads[i] = ops.conv_wgrad(acts[-2], dz, 3)
    g = ops.conv_gemm(dz, _pack(wb[i], ops.PACK_DGRAD), 3)
    for bi in reversed(range(nblocks)):
        j = 2 + 4 * bi
        w1, w2 = wb[j], wb[j + 2]
        a_in, y1, y2 = acts[2 * bi], acts[2 * bi + 1], acts[2 * bi + 2]
        cin, cout = w1.shape[0], w2.shape[0]
        col = cols[bi]
        m2 = col.shape[0]
        dz2, grads[j + 3] = ops.bias_lrelu_bwd(g, y2)
        if need_dw:
            grads[j + 2] = ops.conv_wgrad(col.view(1, 1, m2, 9 * cin), dz2.view(1, 1, m2, cout), 1, reduce_cin=cin,
                                          reduce_taps=9, out_shape=(cout, cin, 3, 3))
        dcol = ops.gemm_rows(dz2.view(m2, cout), _pack(w2, ops.PACK_DCOL))
        nb, hh, ww, _ = y1.shape
        g = ops.col2im_3x3s2(dcol, nb, hh, ww, cin)
        dz1, grads[j + 1] = ops.bias_lrelu_bwd(g, y1)
        if need_dw:
            grads[j] = ops.conv_wgrad(a_in, dz1, 3)
        g = ops.conv_gemm(dz1, _pack(w1, ops.PACK_DGRAD), 3)
        U["blk"][bi] = (dz1, dz2)
    # RGB stem: z = W x + b per pixel
    a0 = acts[0]
    c0 = a0.shape[-1]
    dz, grads[1] = ops.bias_lrelu_bwd(g, a0)
    U["rgb"] = dz
    w_rgb_t = wb[0].reshape(c0, 3).t().contiguous()
    if need_dw:
        # dW[c][k] = sum_pix dz[pix][c] * x[k][pix]: the 1x1 to_rgb backward with the roles of image and activation
        # swapped (its dy output is a by-product here)
        _, dwt, _ = ops.to_rgb_bwd(S["x"], dz, w_rgb_t)
        grads[0] = dwt.view(3, c0).t().contiguous().view_as(wb[0])
    dx = None
    if need_dx:  # dx[k][pix] = sum_c W[c][k] dz[pix][c]: the 1x1 to_rgb forward with W^T and no bias
        dx = ops.to_rgb_fwd(dz, w_rgb_t, torch.zeros(3, dtype=torch.float32, device=dz.device))
    if not need_dw:
        grads = [None] * len(wb)
    return dx, grads, (U if keep_u else None)


def _second_order_chain(S, U, nblocks, wb, px, dout):
    """Given p_x (fp32 [B,3,H,W], the gradient arriving at the image gradient g_x), the forward record S and the masked
    upstream gradients U of the first-order chain, returns (grads aligned with wb, d<g_x,p_x>/d dout [B,1])."""
    acts, hdn = S["acts"], S["hdn"]
    grads = [None] * len(wb)
    px = px.contiguous().to(torch.float32)
    c0 = acts[0].shape[-1]
    w_rgb = wb[0].reshape(c0, 3).contiguous()
    _, dwt, _ = ops.to_rgb_bwd(px, U["rgb"], w_rgb.t().contiguous())
    grads[0] = dwt.view(3, c0).t().contiguous().view_as(wb[0])
    p, _ = ops.bias_lrelu_bwd(ops.from_rgb_fwd(px, w_rgb, None, lrelu=False), acts[0])
    for bi in range(nblocks):
        j = 2 + 4 * bi
        w1, w2 = wb[j], wb[j + 2]
        y1, y2 = acts[2 * bi + 1], acts[2 * bi + 2]
        cin, cout = w1.shape[0], w2.shape[0]
        u1, u2 = U["blk"][bi]
        grads[j] = ops.conv_wgrad(p, u1, 3)
        p, _ = ops.bias_lrelu_bwd(ops.conv_gemm(p, _pack(w1, ops.PACK_FPROP), 3), y1)
        pcol = ops.im2col_3x3s2(p)
        m2 = pcol.shape[0]
        grads[j + 2] = ops.conv_wgrad(pcol.view(1, 1, m2, 9 * cin), u2.view(1, 1, m2, cout), 1, reduce_cin=cin,
                                      reduce_taps=9, out_shape=(cout, cin, 3, 3))
        q = ops.gemm_rows(pcol, _pack(w2, ops.PACK_FPROP)).view(y2.shape)
        p, _ = ops.bias_lrelu_bwd(q, y2)
    i = 2 + 4 * nblocks
    grads[i] = ops.conv_wgrad(p, U["final"], 3)
    p, _ = ops.bias_lrelu_bwd(ops.conv_gemm(p, _pack(wb[i], ops.PACK_FPROP), 3), acts[-1])
    ppool = ops.avgpool_fwd(p)
    wd0, wd1 = wb[i + 2].contiguous(), wb[i + 4].contiguous()
    t = ops.linear_fwd(ppool, wd0, None, 1.0, 1.0, lrelu=False)
    _, grads[i + 2], _ = ops.linear_bwd(U["head"], ppool, wd0, 1.0, 1.0, need_dx=False, has_bias=False)
    pdh = ops.lrelu_bwd(t, hdn)
    dout = dout.contiguous().to(torch.float32)
    _, grads[i + 4], _ = ops.linear_bwd(dout, pdh, wd1, 1.0, 1.0, need_dx=False, has_bias=False)
    d_dout = ops.linear_fwd(pdh, wd1, None, 1.0, 1.0, lrelu=False)
    return grads, d_dout


class _DiscGradFn(torch.autograd.Function):
    """The image gradient of D as a differentiable function of (dout, weights): forward = the first-order dgrad chain,
    backward = _second_order_chain.  Created by _DiscFn.backward when it runs under create_graph=True."""

    @staticmethod
    def forward(ctx, dout, holder, nblocks, *wb):
        dx, grads, U = _disc_backward(holder["S"], nblocks, wb, dout, need_dx=True, need_dw=holder["need_dw"],
                                      keep_u=True)
        holder["grads"] = grads
        ctx.S, ctx.U, ctx.nblocks, ctx.wb = holder["S"], U, nblocks, wb
        ctx.save_for_backward(dout)
        return dx

    @staticmethod
    @once_differentiable
    def backward(ctx, ddx):
        (dout,) = ctx.saved_tensors
        grads, d_dout = _second_order_chain(ctx.S, ctx.U, ctx.nblocks, ctx.wb, ddx, dout)
        ctx.S = ctx.U = None
        return (d_dout, None, None) + tuple(grads)


class _DiscFn(torch.autograd.Function):
    """forward(x [B,3,H,W] fp32, nblocks, w_rgb, b_rgb, (w1, b1, w2, b2) x nblocks, w_final, b_final, wd0, bd0, wd1, bd1)
    -> logits [B,1] fp32.  The weights are the spectrally normalised ones (autograd continues into weight_orig)."""

    @staticmethod
    def forward(ctx, x, nblocks, *wb):
        out, S = _disc_forward(x, nblocks, wb)
        ctx.nblocks, ctx.S, ctx.wb = nblocks, S, wb
        ctx.need_dx = ctx.needs_input_grad[0]
        ctx.need_dw = any(ctx.needs_input_grad[2:])
        return out

    @staticmethod
    def backward(ctx, dout):
        if torch.is_grad_enabled() and ctx.need_dx:
            # create_graph=True (train.py:250-252): the image gradient must remain a function of the weights
            holder = {"S": ctx.S, "need_dw": ctx.need_dw}
            dx = _DiscGradFn.apply(dout, holder, ctx.nblocks, *ctx.wb)
            return (dx, None) + tuple(holder["grads"])
        dx, grads, _ = _disc_backward(ctx.S, ctx.nblocks, ctx.wb, dout, need_dx=ctx.need_dx, need_dw=ctx.need_dw)
        ctx.S = None
        return (dx, None) + tuple(grads)


class _R1Fn(torch.autograd.Function):
    """R1 penalty  mean_b || d D(x).sum() / dx ||^2  (train.py:246-255) and its gradient w.r.t. the (normalised) weights
    as ONE node: forward, dgrad chain (no first-order weight gradients), second-order chain with p_x = 2 g_x / B."""

    @staticmethod
    def forward(ctx, x, nblocks, *wb):
        bsz = x.shape[0]
        out, S = _disc_forward(x, nblocks, wb)
        dout = torch.ones_like(out)
        gx, _, U = _disc_backward(S, nblocks, wb, dout, need_dx=True, need_dw=False, keep_u=True)
        pen = ops.sumsq(gx) / bsz
        ctx.grads, _ = _second_order_chain(S, U, nblocks, wb, ops.scale_copy(gx, 2.0 / bsz), dout)
        del S, U
        return pen.view(())

    @staticmethod
    @once_differentiable
    def backward(ctx, dpen):
        grads, ctx.grads = ctx.grads, None
        return (None, None) + tuple(None if g is None else g * dpen for g in grads)


class StyleDiscriminator(nn.Module):
    def __init__(self, resolution=256, fmap_base=8192, num_channels=3, fmap_max=512):
        super().__init__()
        self.resolution_log2 = int(np.log2(resolution))

        def nf(stage):
            return min(int(fmap_base / (2.0 ** stage)), fmap_max)

        self.fromrgb = spectral_norm(nn.Conv2d(num_channels, nf(self.resolution_log2 - 1), kernel_size=1))
        self.blocks = nn.ModuleList()
        for res in range(self.resolution_log2, 2, -1):
            self.blocks.append(DiscriminatorBlock(nf(res - 1), nf(res - 2)))
        self.final_conv = spectral_norm(nn.Conv2d(nf(2), nf(1), kernel_size=3, padding=1))
        self.adaptive_pool = nn.AdaptiveAvgPool2d((1, 1))
        self.dense0 = spectral_norm(nn.Linear(nf(1), nf(0)))
        self.dense1 = spectral_norm(nn.Linear(nf(0), 1))

    def _native_ok(self, x) -> bool:
        if not (x.is_cuda and x.dim() == 4 and x.shape[1] == 3):
            return False
        # every conv input must map onto the GEMM tiles (64-channel multiples, 128-pixel tile geometry)
        if x.shape[2] != x.shape[3] or x.shape[2] != 2 ** self.resolution_log2 or self.fromrgb.weight_orig.shape[0] % 64:
            return False
        return all(b.conv1.weight_orig.shape[0] % 64 == 0 and b.conv2.weight_orig.shape[0] % 64 == 0 for b in self.blocks)

    def _sn_modules(self):
        mods = [self.fromrgb]
        for blk in self.blocks:
            mods += [blk.conv1, blk.conv2]
        return mods + [self.final_conv, self.dense0, self.dense1]

    @contextlib.contextmanager
    def native_spectral_norm(self):
        """Within this context every call normalises its weights with the sm_100a spectral-norm kernels (one
        _SpectralNormFn node per call) instead of the torch hooks: same u / v updates and gradients, a fixed number of
        launches, capturable in a CUDA graph.  Outside it the hooks run, exactly as in the reference."""
        prev, self._native_sn = self.__dict__.get("_native_sn", False), True
        try:
            yield self
        finally:
            self._native_sn = prev

    def _weights_and_biases(self):
        mods = self._sn_modules()
        if self.__dict__.get("_native_sn", False):
            ws = _SpectralNormFn.apply(self.training, len(mods), *[m.weight_orig for m in mods],
                                       *[m.weight_u for m in mods], *[m.weight_v for m in mods])
        else:
            ws = [_normalized_weight(m) for m in mods]
        wb = []
        for m, w in zip(mods, ws):
            wb += [w, m.bias]
        return wb

    def r1_penalty(self, real_img):
        """`compute_r1_reg(D, real_img)` of train.py:246-255 fused into one node: the penalty (scalar) with gradients
        w.r.t. the parameters.  Like the reference it marks the batch as requiring grad (SURVEY Q2) and runs the
        spectral-norm hooks once (one power iteration in train mode, as `D(real_img)` would)."""
        real_img.requires_grad_(True)
        self._require_native(real_img, "r1_penalty")
        return _R1Fn.apply(real_img.detach(), len(self.blocks), *self._weights_and_biases())

    def _require_native(self, x, what):
        if not self._native_ok(x):  # no fallback: the sm_100a path either runs or the call fails
            raise ops._lib.IrfdError(
                f"StyleDiscriminator.{what}: input {tuple(x.shape)} on {x.device} does not fit the sm_100a path (CUDA, "
                f"square {2 ** self.resolution_log2}x{2 ** self.resolution_log2} RGB images, 64-channel multiples)")

    def forward(self, x):
        self._require_native(x, "forward")
        return _DiscFn.apply(x, len(self.blocks), *self._weights_and_biases())


def compute_r1_reg(D: StyleDiscriminator, real_img):
    """train.py:246-255, verbatim semantics: the generic double backward, which the native node supports.
    (`D.r1_penalty(real_img)` computes the same value and gradients in one fused node.)"""
    real_img = real_img.requires_grad_(True)
    real_pred = D(real_img)
    grad_real = torch.autograd.grad(outputs=real_pred.sum(), inputs=real_img, create_graph=True)[0]
    return grad_real.pow(2).reshape(grad_real.shape[0], -1).sum(1).mean()
