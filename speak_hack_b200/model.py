"""IRFD (Inter-Reconstructed Feature Disentanglement) — drop-in for the reference's model.py:28-137, 356-372.

Same class names, constructor signatures, `forward()` signatures, attribute names (.Ei .Ee .Ep .Gd .D .Cm
.current_resolution) and state_dict keys as the reference, so train.py / test_irfd.py / inference.py can use it
unchanged.  The encoders, generator and losses run on the hand-written sm_100a kernels of libirfd_b200.so; there is
no CPU fallback and no ATen compute on the hot path (torch is used for memory, autograd graph plumbing, RNG draws in
the reference's order and the [B,6144] concatenation, which is a bit-exact copy).
"""
from __future__ import annotations

import logging

import torch
import torch.nn as nn

from . import ops
from .discriminator import StyleDiscriminator
from .encoder import ResNet50Encoder, _encoder_inference, check_inference_shape
from .encoder_group import EncoderGroup
from .generator import StyleGenerator


class _MSEFn(torch.autograd.Function):
    """nn.MSELoss(reduction='mean') on fp32 CUDA tensors (model.py:206, 358, 367)."""

    @staticmethod
    def forward(ctx, a, b, scale):
        a = a.contiguous().to(torch.float32)
        b = b.contiguous().to(torch.float32)
        ctx.save_for_backward(a, b)
        ctx.scale = scale
        out = ops.mse_fwd(a, b)
        if scale != 1.0:
            out = ops.scale_copy(out, scale)
        return out.view(())

    @staticmethod
    def backward(ctx, g):
        a, b = ctx.saved_tensors
        need_a, need_b = ctx.needs_input_grad[:2]
        gs = g.contiguous().view(1).to(torch.float32)
        if ctx.scale != 1.0:
            gs = ops.scale_copy(gs, ctx.scale)
        da, db = ops.mse_bwd(a, b, gs, need_da=need_a, need_db=need_b)
        return da, db, None


def mse_loss(a: torch.Tensor, b: torch.Tensor, scale: float = 1.0) -> torch.Tensor:
    """scale * mean((a - b)^2) (nn.MSELoss, model.py:206, 358, 367); scale folds a sum of equally sized MSE terms."""
    if a.shape != b.shape:
        raise ValueError(f"mse_loss: shape mismatch {tuple(a.shape)} vs {tuple(b.shape)}")
    return _MSEFn.apply(a, b, float(scale))


class IRFD(nn.Module):
    def __init__(self, max_resolution=256):
        super().__init__()
        # construction order == reference (model.py:33-41): it fixes how a seeded construction consumes the RNG
        self.Ei = self._create_encoder()  # identity
        self.Ee = self._create_encoder()  # emotion
        self.Ep = self._create_encoder()  # pose
        self.Gd = StyleGenerator(input_dim=6144)
        self.D = StyleDiscriminator()
        self.Cm = nn.Linear(2048, 8)
        self.max_resolution = max_resolution
        self.current_resolution = max_resolution
        self.logger = logging.getLogger(__name__)
        self.apply(self._init_weights)

    def _init_weights(self, m):
        # model.py:50-54: every nn.Conv2d / nn.Linear is re-initialised, the "pretrained" encoders included
        if isinstance(m, nn.Conv2d) or isinstance(m, nn.Linear):
            nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")
            if m.bias is not None:
                nn.init.constant_(m.bias, 0)

    def adjust_for_resolution(self, resolution):
        self.current_resolution = resolution

    def _create_encoder(self):
        return ResNet50Encoder()

    def _prepare_generator_input(self, *features):
        # model.py:64-69 — flatten and concatenate: identity, emotion, pose (a pure copy, bit-exact)
        return torch.cat([f.view(f.size(0), -1) for f in features], dim=1)

    def _encode(self, enc, x):
        """`checkpoint(enc, x)` of the reference (model.py:84-90), reentrant flavour: the encoder is differentiated
        only when the INPUT requires grad (SURVEY Q2), and a differentiated pass updates the BN running buffers a
        second time during backward (SURVEY Q3).  Activations are kept instead of recomputed (180 GB of HBM)."""
        if torch.is_grad_enabled() and x.requires_grad:
            enc._recompute_bn_update = enc.training
            try:
                return enc(x)
            finally:
                enc._recompute_bn_update = False
        with torch.no_grad():
            return enc(x)

    @property
    def encoder_group(self):
        """Lockstep runner of the three encoders (encoder_group.EncoderGroup), created on first use."""
        grp = self.__dict__.get("_encoder_group")
        if grp is None or grp.encoders != [self.Ei, self.Ee, self.Ep]:
            grp = EncoderGroup([self.Ei, self.Ee, self.Ep])
            self.__dict__["_encoder_group"] = grp
        return grp

    def _encode_all(self, x_s, x_t):
        """The six encoder passes of model.py:84-90.  When shapes allow, the three encoders run in lockstep on the
        stacked source+target batch: ONE launch per layer (grouped GEMM over the three weight sets, BatchNorm over
        3 encoders x 2 statistic groups) — numerically the same as Ei(x_s), Ee(x_s), Ep(x_s), Ei(x_t), ... (per-call
        batch statistics, each encoder's running buffers updated source first), at a sixth of the kernel launches."""
        same = x_s.shape == x_t.shape and x_s.requires_grad == x_t.requires_grad and x_s.is_cuda
        grp = self.encoder_group
        diff = torch.is_grad_enabled() and x_s.requires_grad
        if same and x_s.dim() == 4 and (grp.encoders[0].training or not diff):
            x = torch.cat([x_s, x_t], dim=0)  # cat keeps requires_grad (SURVEY Q2 semantics)
            if grp.can_run(x, 2):
                B = x_s.size(0)
                if diff:
                    for enc in grp.encoders:
                        enc._recompute_bn_update = enc.training
                    try:
                        f = grp(x, 2)
                    finally:
                        for enc in grp.encoders:
                            enc._recompute_bn_update = False
                else:
                    with torch.no_grad():
                        f = grp(x, 2)
                return f[0, :B], f[1, :B], f[2, :B], f[0, B:], f[1, B:], f[2, B:]
        return (self._encode(self.Ei, x_s), self._encode(self.Ee, x_s), self._encode(self.Ep, x_s),
                self._encode(self.Ei, x_t), self._encode(self.Ee, x_t), self._encode(self.Ep, x_t))

    def forward(self, x_s, x_t):
        fi_s, fe_s, fp_s, fi_t, fe_t, fp_t = self._encode_all(x_s, x_t)

        # model.py:97-104 — one CPU-generator draw per forward; whole-tensor S<->T swap of one code type
        swap_type = torch.randint(0, 3, (1,)).item()
        if swap_type == 0:
            fi_s, fi_t = fi_t, fi_s
        elif swap_type == 1:
            fe_s, fe_t = fe_t, fe_s
        else:
            fp_s, fp_t = fp_t, fp_s

        x_s_recon = self.Gd(self._prepare_generator_input(fi_s, fe_s, fp_s))
        x_t_recon = self.Gd(self._prepare_generator_input(fi_t, fe_t, fp_t))

        # model.py:121-122 — the predictions are discarded by train.py:190 and the emotion loss is hard-wired to 0
        # (model.py:354), so they are computed without an autograd graph.
        with torch.no_grad():
            emotion_pred_s = self._emotion(fe_s)
            emotion_pred_t = self._emotion(fe_t)
        return x_s_recon, x_t_recon, fi_s, fe_s, fp_s, fi_t, fe_t, fp_t, emotion_pred_s, emotion_pred_t

    def _emotion(self, fe):
        logits = ops.linear_fwd(fe.detach().reshape(fe.size(0), -1).contiguous(), self.Cm.weight, self.Cm.bias, 1.0, 1.0,
                                lrelu=False)
        return ops.softmax_rows(logits)


class StyleGANLoss(nn.Module):
    """model.py:130-137."""

    def __init__(self, device):
        super().__init__()
        self.device = device

    def forward(self, real, fake):
        return mse_loss(fake, torch.ones_like(fake)) + mse_loss(real, torch.zeros_like(real))


class IRFDLoss(nn.Module):
    """The differentiable part of the reference's IRFDLoss (model.py:182-386): identity and reconstruction MSE.

    The pose term needs SixDRepNet weights fetched from a URL and goes through `.item()` (zero gradient); the emotion
    term is hard-wired to 0.0 (model.py:354).  Both are returned as zeros here (SURVEY F4; out of scope rows of §2).
    """

    def __init__(self, config=None, device=None):
        super().__init__()
        self.device = device
        w = (config or {}).get("weights", {}) if isinstance(config, dict) else {}
        self.face_recognition_weight = w.get("face_recognition", 1.0)
        self.emotion_weight = w.get("emotion", 1.0)
        self.landmark_weight = w.get("landmark", 1.0)

    def identity_loss(self, fi_s, fi_t):
        return mse_loss(fi_s, fi_t)

    def reconstruction_loss(self, x_s, x_t, x_s_recon, x_t_recon):
        return mse_loss(x_s, x_s_recon) + mse_loss(x_t, x_t_recon)

    def forward(self, x_s, x_t, x_s_recon, x_t_recon, fi_s, fe_s, fp_s, fi_t, fe_t, fp_t, emotion_labels_s=None,
                emotion_labels_t=None):
        zero = torch.zeros((), device=x_s.device)
        l_identity = self.identity_loss(fi_s, fi_t)
        l_recon = self.reconstruction_loss(x_s, x_t, x_s_recon, x_t_recon)
        return zero, zero.clone(), l_identity, l_recon


# ----------------------------------------------------------------------------------------------------------------------
# Static-graph variant of IRFD.forward (used by trainer.IRFDTrainer(use_cuda_graph=True) and inference.IRFDInference)
# ----------------------------------------------------------------------------------------------------------------------
class _SwapCatFn(torch.autograd.Function):
    """Device-side S<->T swap + concat: ctrl[0] = swap_type.  Pure copies (bit-exact), see csrc/control.cu."""

    @staticmethod
    def forward(ctx, ctrl, *feats):
        flat = [f.reshape(f.size(0), -1).contiguous() for f in feats]
        ctx.ctrl = ctrl
        ctx.c = flat[0].shape[1]
        ctx.shapes = [f.shape for f in feats]
        return ops.swap_cat_fwd(flat, ctrl)

    @staticmethod
    def backward(ctx, dgen_s, dgen_t):
        outs = ops.swap_cat_bwd(dgen_s.contiguous(), dgen_t.contiguous(), ctx.ctrl, ctx.c)
        return (None,) + tuple(o.view(s) for o, s in zip(outs, ctx.shapes))


class _SwapCatStackedFn(torch.autograd.Function):
    """The same on the stacked layout of the lockstep encoder pass: f [3, 2B, C, 1, 1] (encoder-major; source rows then
    target rows) -> gen [2B, 3C] whose first B rows are the source generator input and the rest the target's
    (model.py:97-114).  Backward scatters into ONE [3, 2B, C] gradient buffer (six slices written by one kernel)."""

    @staticmethod
    def forward(ctx, ctrl, f):
        e, n2, c = f.shape[0], f.shape[1], f.shape[2]
        b = n2 // 2
        f2 = f.reshape(e, n2, c)
        gen = torch.empty((n2, e * c), dtype=torch.float32, device=f.device)
        ops.swap_cat_fwd([f2[0, :b], f2[1, :b], f2[2, :b], f2[0, b:], f2[1, b:], f2[2, b:]], ctrl, out=gen)
        ctx.ctrl, ctx.shape = ctrl, f.shape
        return gen

    @staticmethod
    def backward(ctx, dgen):
        dgen = dgen.contiguous()
        e, n2, c = ctx.shape[0], ctx.shape[1], ctx.shape[2]
        b = n2 // 2
        df = torch.empty((e, n2, c), dtype=torch.float32, device=dgen.device)
        ops.swap_cat_bwd(dgen[:b], dgen[b:], ctx.ctrl, c,
                         outs=[df[0, :b], df[1, :b], df[2, :b], df[0, b:], df[1, b:], df[2, b:]])
        return None, df.view(ctx.shape)


def _irfd_forward_static(self: IRFD, x_s, x_t, ctrl):
    """IRFD.forward with the swap / style-mixing decisions taken on the device from `ctrl` (int32 [3]).
    Returns (x_s_recon, x_t_recon, fi_s, fi_t) with fi_* UNswapped (the identity MSE is symmetric in them)."""
    img, f, b = self.forward_static_stacked(torch.cat([x_s, x_t], dim=0), ctrl)
    return img[:b], img[b:], f[0, :b], f[0, b:]


def _irfd_forward_static_stacked(self: IRFD, x, ctrl):
    """The whole forward on the stacked batch x = [x_s; x_t] ([2B, 3, H, W]): the three encoders in lockstep (one launch
    per layer), device-side swap + concat, ONE generator call over the 2B stacked codes.
    Returns (images [2B, 3, R, R] (source reconstructions first), features [3, 2B, 2048, 1, 1] unswapped, B)."""
    grp = self.encoder_group
    b = x.size(0) // 2
    diff = torch.is_grad_enabled() and x.requires_grad
    training = grp.encoders[0].training
    if not training and not diff and not grp.can_run(x, 2):
        # eval-mode inference at a size the lockstep pass cannot tile: the three encoders one after the other on the
        # stacked batch (same arithmetic per pixel, so the same features), sharing the stem's im2col matrix
        encs = grp.encoders
        if not (x.is_cuda and x.dim() == 4 and x.shape[1] == 3) or len({e.training for e in encs}) != 1:
            raise ops._lib.IrfdError(f"IRFD.forward_static: bad batch {tuple(x.shape)} / encoder modes")
        check_inference_shape(x)
        with torch.no_grad():
            xf = x.contiguous().to(torch.float32)
            col0 = ops.im2col_stem(xf, 192)
            f = torch.stack([_encoder_inference(e, xf, col0) for e in encs])
        gen = _SwapCatStackedFn.apply(ctrl, f)
        return self.Gd.forward_static(gen, ctrl, 1, b_first=b), f, b
    if not grp.can_run(x, 2) or (diff and not training):
        raise ops._lib.IrfdError(f"IRFD.forward_static: batch {tuple(x.shape)} cannot run as one lockstep encoder pass "
                                 "(needs pairs x (H/32) x (W/32) to be a multiple of 128); use IRFD.forward")
    if diff:
        for enc in grp.encoders:
            enc._recompute_bn_update = enc.training
        try:
            f = grp(x, 2)
        finally:
            for enc in grp.encoders:
                enc._recompute_bn_update = False
    else:
        with torch.no_grad():
            f = grp(x, 2)
    gen = _SwapCatStackedFn.apply(ctrl, f)
    img = self.Gd.forward_static(gen, ctrl, 1, b_first=b)
    return img, f, b


IRFD.forward_static = _irfd_forward_static
IRFD.forward_static_stacked = _irfd_forward_static_stacked
