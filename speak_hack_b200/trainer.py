"""IRFD generator-step trainer: the reference's G step (train.py:186-210) on the sm_100a path, single- or multi-GPU.

One process per GPU.  Each rank runs the IRFD forward/backward on its shard of the global batch (per-rank BatchNorm
statistics, like the reference under accelerate/DDP without SyncBN); gradients are averaged by bucketed all-reduce
overlapped with backward (dp.py); Adam (train.py:346: Gd.parameters() only, lr 2e-4) is one fused kernel over a flat
parameter buffer, optionally preceded by clip_grad_norm_ over ALL model parameters (train.py:207-208).

Loss: l_identity + l_recon, the differentiable terms of the reference's criterion (model.py:356-372; the pose and
emotion terms carry no gradient, SURVEY F4) — SURVEY §8(d) config 3.  The reference's G step additionally adds
`stylegan_loss_weight * BCE(D(x_recon), real)` (train.py:197-203); pass `adv_weight` to include it: D(x_s_recon) and
D(x_t_recon) run through the native discriminator, their gradient reaches Gd, and D's own parameter gradients (which
the reference's clip_grad_norm_ over model.parameters() also sees) enter the clipping norm.

Gradient buffers are flat: all of Gd in one fp32 buffer, the encoders in one buffer per ResNet stage holding that
stage's parameters of Ei, Ee and Ep.  The lockstep encoder backward (encoder_group.py) writes every encoder gradient
straight into its slot (no autograd accumulation kernels), and each buffer is one all-reduce bucket.

`use_cuda_graph=True` captures the WHOLE step (zero_grad, forward, losses, backward, all-reduce, Adam) into one CUDA
graph on ONE stream (plus the communication stream).  The reference's CPU-generator decisions (swap type, style-mixing
cuts) are still drawn on the host in the reference's order every step, but reach the kernels through a 3-int control
tensor (csrc/control.cu) so the launch sequence is static.  Differences from eager mode: source and target images live
in one stacked [2B,3,H,W] buffer, the two generator calls run as ONE call over the 2B stacked codes (the generator has
no batch statistics), and the encoders' bf16 weight repacks are captured as constants (encoders have no optimizer in
the reference, train.py:346).
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional

import torch

from . import ops
from .dp import BucketSchedule, GradBuckets, broadcast_buffers
from .model import IRFD, mse_loss

_PREPACK = os.environ.get("IRFD_PREPACK", "1") != "0"   # 0: conv weights are repacked lazily on the main stream
REAL_LABEL, FAKE_LABEL = 0.9, 0.1   # train.py:145-146 (one-sided label smoothing on both sides)
STAGES = (7, 6, 5, 4, 3)  # ResNet50Encoder child indices 7..4 = layer4..layer1; 3 stands for the stem (children 0, 1)


def flatten_parameters(params: List[torch.nn.Parameter]):
    """Re-home parameters (and their .grad) as views of flat fp32 buffers: Adam and all-reduce become single launches."""
    total = sum(p.numel() for p in params)
    dev = params[0].device
    flat = torch.empty(total, dtype=torch.float32, device=dev)
    gflat = torch.zeros(total, dtype=torch.float32, device=dev)
    off = 0
    for p in params:
        n = p.numel()
        flat[off: off + n].copy_(p.data.reshape(-1))
        p.data = flat[off: off + n].view_as(p.data)
        p.grad = gflat[off: off + n].view_as(p.data)
        off += n
    return flat, gflat


def _stage_of(name: str) -> int:
    idx = int(name.split(".")[0])
    return idx if idx >= 4 else 3


def flat_encoder_gradients(encoders) -> (Dict[int, torch.Tensor], Dict[torch.nn.Parameter, torch.Tensor]):
    """One flat fp32 gradient buffer per ResNet stage (all encoders' parameters of that stage, encoder after encoder);
    every parameter's .grad becomes a view of its slot.  Returns ({stage: flat}, {parameter: view})."""
    dev = next(encoders[0].parameters()).device
    by_stage: Dict[int, List[torch.nn.Parameter]] = {k: [] for k in STAGES}
    for enc in encoders:
        for name, p in enc.named_parameters():
            by_stage[_stage_of(name)].append(p)
    flats, targets = {}, {}
    for k, ps in by_stage.items():
        flat = torch.zeros(sum(p.numel() for p in ps), dtype=torch.float32, device=dev)
        off = 0
        for p in ps:
            v = flat[off: off + p.numel()].view_as(p)
            p.grad = v
            targets[p] = v
            off += p.numel()
        flats[k] = flat
    return flats, targets


class _BCELogitsFn(torch.autograd.Function):
    """mean(BCEWithLogits(x, target)) for a constant target in {0, 1} on a [B, 1] logit tensor (train.py:200-201).
    B values: evaluated with the fp32 softplus form, gradient (sigmoid(x) - t) / B."""

    @staticmethod
    def forward(ctx, logits, target: float):
        x = logits.detach().to(torch.float32)
        ctx.save_for_backward(x)
        ctx.target = target
        return (torch.clamp(x, min=0) - x * target + torch.log1p(torch.exp(-x.abs()))).mean()

    @staticmethod
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        return g * (torch.sigmoid(x) - ctx.target) / x.numel(), None


class StepGraph:
    """The graph-mode plumbing the generator step (IRFDTrainer) and the discriminator step (IRFDDiscriminatorStep)
    share: the reference's CPU-generator draws uploaded as a device control tensor, the device step counter of the
    captured Adam, and capture with rollback of the warm-up passes."""

    def __init__(self, model: IRFD, device: torch.device):
        self.model = model
        self.device = device
        self.ctrl = torch.zeros(3, dtype=torch.int32, device=device)
        # ring of pinned control buffers: an async H2D copy reads its pinned source when the STREAM reaches it, and the
        # CPU runs several graph replays ahead, so a slot is rewritten only after the copy that read it has completed
        self._ring = ([(torch.zeros(3, dtype=torch.int32).pin_memory(), torch.cuda.Event()) for _ in range(8)]
                      if device.type == "cuda" else [])
        self._slot = 0
        self.last_ctrl = None
        self.step_dev = torch.zeros(1, dtype=torch.int32, device=device)

    def draw_ctrl(self):
        """The reference's CPU-generator draws of one IRFD.forward, in its order: swap (model.py:98), then per Gd call
        rand(1) and, when mixing, randint(1, L) (styleganv1.py:548, 552)."""
        gd = self.model.Gd
        L = gd.synthesis.num_layers
        vals = [int(torch.randint(0, 3, (1,)).item())]
        for g in range(2):
            cut = L
            if gd.training and gd.style_mixing_prob > 0:
                if torch.rand(1) < gd.style_mixing_prob:
                    cut = int(torch.randint(1, L, (1,)).item())
            vals.append(cut)
        self.upload_ctrl(vals)

    def upload_ctrl(self, vals):
        host, ev = self._ring[self._slot]
        self._slot = (self._slot + 1) % len(self._ring)
        ev.synchronize()  # no-op unless the CPU is a whole ring ahead of the device
        host[0], host[1], host[2] = vals
        self.ctrl.copy_(host, non_blocking=True)
        ev.record()
        self.last_ctrl = tuple(vals)

    def capture(self, owner, body, state):
        """Capture body() (one step of `owner`) into a CUDA graph.  Two warm-up passes run first (allocator, lazy
        function attributes, pack caches); they are real steps, so everything they mutate is put back: the tensors in
        `state`, owner.step_count, the device step counter and both RNG streams.  Returns (graph, launches)."""
        dev = self.device
        self.step_dev.fill_(owner.step_count)
        snap = [t.clone() for t in state]
        snap_step = owner.step_count
        cpu_rng, cuda_rng = torch.get_rng_state(), torch.cuda.get_rng_state(dev)
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                self.draw_ctrl()
                body()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        before = ops.launch_count
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            body()
        launches = ops.launch_count - before
        # the captured pass was only recorded, not executed; the warm-up passes are rolled back
        for t, c in zip(state, snap):
            t.copy_(c)
        owner.step_count = snap_step
        self.step_dev.fill_(snap_step)
        torch.set_rng_state(cpu_rng)
        torch.cuda.set_rng_state(cuda_rng, dev)
        return graph, launches


class IRFDTrainer:
    def __init__(self, model: IRFD, lr: float = 2e-4, betas=(0.9, 0.999), eps: float = 1e-8,
                 grad_clip: Optional[float] = None, encoder_grads: bool = True, use_cuda_graph: bool = False,
                 adv_weight: Optional[float] = None):
        if adv_weight is not None and use_cuda_graph:
            raise ops._lib.IrfdError("IRFDTrainer: the adversarial term runs the discriminator's spectral-norm hooks "
                                     "(torch code) every step; use the eager step (use_cuda_graph=False) with adv_weight")
        self.model = model
        self.lr, self.betas, self.eps = lr, betas, eps
        self.grad_clip = grad_clip
        self.encoder_grads = encoder_grads
        self.adv_weight = adv_weight
        self.gd_params = list(model.Gd.parameters())
        self.flat, self.gflat = flatten_parameters(self.gd_params)
        self._gd_targets = {p.data_ptr(): p.grad for p in self.gd_params}
        self._gd_conv_weights = [p for p in self.gd_params if p.dim() == 4 and p.shape[-1] == 3]
        self.m = torch.zeros_like(self.flat)
        self.v = torch.zeros_like(self.flat)
        self.step_count = 0
        self.encoders = [model.Ei, model.Ee, model.Ep]
        self.device = self.flat.device
        self.stage_flats, self._enc_targets = flat_encoder_gradients(self.encoders)
        self._enc_params = [p for e in self.encoders for p in e.parameters()]
        self.buckets = GradBuckets(self.device)
        if self.device.type == "cuda":
            side = ops.side_stream(self.device)
            self.buckets.producers = lambda: [side.stream] if side.active else []
        self.world = self.buckets.world
        self.schedule = BucketSchedule(self.buckets, self.gflat, self.stage_flats)
        self.last_losses = None
        # static-graph state
        self.use_cuda_graph = use_cuda_graph
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        self.graph_launches = 0
        self._graphed = StepGraph(model, self.device)
        self.ctrl, self.step_dev = self._graphed.ctrl, self._graphed.step_dev
        self._graph_key = None
        self._static = None

    # ---------------------------------------------------------------------------------------------- shared pieces
    def zero_grad(self, encoders_direct: bool = True, gd_direct: bool = False):
        """Gd gradients are accumulated by autograd into the flat buffer: zero it — unless the step writes them in place
        (static step: one generator call, generator.GRAD_TARGETS).  Encoder gradients are overwritten by the lockstep
        backward; only the per-encoder fallback path (autograd accumulation) needs them zeroed."""
        if not gd_direct:
            self.gflat.zero_()
        for p in self.gd_params:  # keep .grad pointing into the flat buffer
            t = self._gd_targets[p.data_ptr()]
            if p.grad is not t:
                p.grad = t
        if self.adv_weight is not None:
            for p in self.model.D.parameters():
                p.grad = None
        for p in self._enc_params:  # keep .grad pointing into the flat stage buffers
            if p.grad is not self._enc_targets[p]:
                p.grad = self._enc_targets[p]
        if not encoders_direct:
            for f in self.stage_flats.values():
                f.zero_()

    def _direct(self, x_s) -> bool:
        """Will a batch of this shape run as ONE lockstep encoder pass (source and target stacked) that writes its
        gradients in place?  Mirrors IRFD._encode_all / EncoderGroup.can_run for 2 statistic groups of x_s.size(0)."""
        ok = (x_s.is_cuda and x_s.dim() == 4 and x_s.shape[1] == 3 and x_s.shape[2] % 32 == 0 and x_s.shape[3] % 32 == 0
              and (x_s.size(0) * (x_s.shape[2] // 32) * (x_s.shape[3] // 32)) % 128 == 0)
        return bool(ok and self.encoder_grads and all(e.training for e in self.encoders))

    def _backward_and_update(self, loss, static: bool):
        grp = self.model.encoder_group
        if self.world > 1:
            self.schedule.reset()
            grp._bwd_cb = self.schedule.on_event
        try:
            loss.backward()
        finally:
            grp._bwd_cb = None
        ops.side_stream(self.gflat.device).join()   # side-stream gradient launches (no-op when the encoders joined)
        if self.world > 1:
            self.schedule.final()
        self.step_count += 1
        total_sumsq = None
        if self.grad_clip is not None:
            total_sumsq = ops.sumsq(self.gflat)
            for f in self.stage_flats.values():
                ops.sumsq(f, out=total_sumsq, out_beta=1.0)
            if self.adv_weight is not None:  # clip_grad_norm_(model.parameters()) also sees D's gradients
                for p in self.model.D.parameters():
                    if p.grad is not None:
                        ops.sumsq(p.grad.reshape(-1).contiguous(), out=total_sumsq, out_beta=1.0)
        ops.adam_step(self.flat, self.gflat, self.m, self.v, self.lr, self.betas[0], self.betas[1], self.eps,
                      self.step_count, total_sumsq=total_sumsq, max_norm=self.grad_clip or 0.0,
                      step_dev=self.step_dev if static else None)
        ops.invalidate_packed(self._gd_conv_weights)  # Adam wrote through the flat buffer: bf16 repacks are stale

    def _prep(self, x):
        # train.py's R1 penalty leaves requires_grad=True on the batch, which is what lets the reference's reentrant
        # checkpoints differentiate the encoders (SURVEY Q2)
        return x.detach().requires_grad_(True) if self.encoder_grads else x.detach()

    def _adversarial(self, recon):
        """stylegan_loss_weight * mean over the two reconstructions of BCE(D(x_recon), real) (train.py:197-203)."""
        d = self.model.D(recon)
        return _BCELogitsFn.apply(d, REAL_LABEL)

    # ---------------------------------------------------------------------------------------------- eager step
    def train_step_eager(self, x_s: torch.Tensor, x_t: torch.Tensor):
        """zero_grad -> forward -> MSE losses -> backward (+ overlapped all-reduce) -> [clip] -> Adam on Gd."""
        direct = self._direct(x_s)
        self.zero_grad(encoders_direct=direct)
        grp = self.model.encoder_group
        grp.grad_targets = self._enc_targets if direct else None
        try:
            x_s, x_t = self._prep(x_s), self._prep(x_t)
            out = self.model(x_s, x_t)
            x_s_recon, x_t_recon, fi_s, _, _, fi_t = out[:6]
            l_identity = mse_loss(fi_s, fi_t)
            l_recon = mse_loss(x_s.detach(), x_s_recon) + mse_loss(x_t.detach(), x_t_recon)
            loss = l_identity + l_recon
            if self.adv_weight is not None:
                loss = loss + self.adv_weight * 0.5 * (self._adversarial(x_s_recon) + self._adversarial(x_t_recon))
            self._backward_and_update(loss, static=False)
        finally:
            grp.grad_targets = None
        self.last_losses = (l_identity.detach(), l_recon.detach())
        return loss.detach()

    # ---------------------------------------------------------------------------------------------- static-graph step
    def _static_body(self):
        x_all, loss_out, lid_out, lrec_out = self._static
        b = x_all.size(0) // 2
        from . import generator

        self.zero_grad(encoders_direct=True, gd_direct=True)
        grp = self.model.encoder_group
        grp.grad_targets = self._enc_targets
        generator.GRAD_TARGETS = self._gd_targets   # ONE generator call per step: its backward writes gflat in place
        try:
            if _PREPACK:   # the generator's conv repacks (its weights changed in the last Adam step) behind the encoders
                ops.prepack_conv_weights(generator.synthesis_pack_items(self.model.Gd.synthesis),
                                         ops.side_stream(self.device))
            x = self._prep(x_all)
            img, f, _ = self.model.forward_static_stacked(x, self.ctrl)
            l_identity = mse_loss(f[0, :b], f[0, b:])
            # MSE(x_s, x_s_recon) + MSE(x_t, x_t_recon) with equally sized halves == 2 * MSE over the stacked batch
            l_recon = mse_loss(x_all, img, scale=2.0)
            loss = l_identity + l_recon
            if self.adv_weight is not None:
                loss = loss + self.adv_weight * self._adversarial(img)  # mean over 2B logits == (BCE_s + BCE_t) / 2
            self._backward_and_update(loss, static=True)
        finally:
            grp.grad_targets = None
            generator.GRAD_TARGETS = None
        loss_out.copy_(loss.detach())
        lid_out.copy_(l_identity.detach())
        lrec_out.copy_(l_recon.detach())

    def _ensure_static(self, x_s):
        """The stacked static batch [x_s; x_t] and the three loss scalars the static step reads / writes."""
        dev = self.device
        if not self._direct(x_s):
            raise ops._lib.IrfdError(
                f"IRFDTrainer static step: batch {tuple(x_s.shape)} cannot run as one lockstep encoder pass (pairs x "
                "(H/32) x (W/32) must be a multiple of 128, encoders in train mode with gradients); use "
                "train_step_eager")
        b = x_s.size(0)
        shape = (2 * b,) + tuple(x_s.shape[1:])
        if self._static is None or tuple(self._static[0].shape) != shape:
            self._static = (torch.empty(shape, dtype=torch.float32, device=dev), torch.zeros((), device=dev),
                            torch.zeros((), device=dev), torch.zeros((), device=dev))

    def _capture(self, x_s, x_t):
        self._ensure_static(x_s)
        b = x_s.size(0)
        self._static[0][:b].copy_(x_s)
        self._static[0][b:].copy_(x_t)
        bufs = [bf for e in self.encoders for bf in e.buffers()]
        bufs += [bf for bf in self.model.D.buffers()] if self.adv_weight is not None else []
        return self._graphed.capture(self, self._static_body, [self.flat, self.m, self.v] + bufs)

    def _graph_state(self, x_s):
        """What a captured graph bakes in besides the buffers it owns: the train/eval mode of every sub-network, the
        input shape, and the encoders' bf16 weight repacks (constants in the graph; keyed by the weights' version
        counters so load_state_dict / an external optimizer on the encoders forces a recapture)."""
        m = self.model
        enc_ver = tuple(e[0].weight._version for e in self.encoders)
        return (m.training, m.Gd.training, tuple(e.training for e in self.encoders), tuple(x_s.shape), enc_ver,
                float(m.Gd.style_mixing_prob), self.buckets.enabled)

    def train_step_graph(self, x_s: torch.Tensor, x_t: torch.Tensor):
        key = self._graph_state(x_s)
        if self.graph is not None and key != self._graph_key:
            self.graph = None
        if self.graph is None:
            self.graph, self.graph_launches = self._capture(x_s, x_t)
            self._graph_key = key
        b = x_s.size(0)
        self._static[0][:b].copy_(x_s, non_blocking=True)   # straight into the stacked static batch: no torch.cat
        self._static[0][b:].copy_(x_t, non_blocking=True)
        self._graphed.draw_ctrl()
        self.graph.replay()
        self.step_count += 1
        ops.launch_count += self.graph_launches
        self.last_losses = (self._static[2], self._static[3])
        return self._static[1]

    def train_step_static_eager(self, x_s: torch.Tensor, x_t: torch.Tensor):
        """The launch sequence of the captured step, launched kernel by kernel (bench.py times every GEMM launch with
        CUDA events this way — events cannot be recorded inside a graph replay — and ncu lists its launches)."""
        self._ensure_static(x_s)
        b = x_s.size(0)
        self._static[0][:b].copy_(x_s, non_blocking=True)
        self._static[0][b:].copy_(x_t, non_blocking=True)
        self._graphed.draw_ctrl()
        self.step_dev.fill_(self.step_count)
        self._static_body()
        return self._static[1]

    def train_step(self, x_s: torch.Tensor, x_t: torch.Tensor):
        """use_cuda_graph: one graph replay.  Otherwise the reference-ordered eager step (IRFD.forward: two generator
        calls, the reference's RNG consumption order)."""
        if self.use_cuda_graph:
            return self.train_step_graph(x_s, x_t)
        return self.train_step_eager(x_s, x_t)

    def snapshot(self):
        """Everything a step mutates (Gd parameters, Adam moments, BN buffers, step counters), for restore()."""
        bufs = [bf for e in self.encoders for bf in e.buffers()]
        return ([t.clone() for t in (self.flat, self.m, self.v)], [bf.clone() for bf in bufs], self.step_count)

    def restore(self, snap) -> None:
        tensors, bufs, step = snap
        for t, c in zip((self.flat, self.m, self.v), tensors):
            t.copy_(c)
        for bf, c in zip([bf for e in self.encoders for bf in e.buffers()], bufs):
            bf.copy_(c)
        self.step_count = step
        self.step_dev.fill_(step)
        ops.invalidate_packed(self._gd_conv_weights)

    def gradient_buffers(self):
        """The flat gradient buffers in bucket order: all of Gd, then the encoders' stages 4..1 and the stem."""
        return [self.gflat] + [self.stage_flats[k] for k in STAGES]

    def sync_buffers(self) -> None:
        """DDP `broadcast_buffers=True` (train.py:399 default): every rank takes rank 0's BatchNorm running buffers.
        Call before evaluating or checkpointing a data-parallel run (save_checkpoint does)."""
        broadcast_buffers(self.encoders)

    # ---------------------------------------------------------------------------------------------- checkpoints
    # The reference saves {'model_state_dict', 'optimizer_G', 'optimizer_D', 'epoch', 'resolution', 'config'}
    # (train.py:232-240) and resumes with load_state_dict on each (train.py:362-368).  optimizer_G is
    # torch.optim.Adam(model.Gd.parameters(), lr=2e-4) (train.py:346); the fused trainer keeps the same state in flat
    # buffers, exported / imported here in torch.optim.Adam's state_dict layout so checkpoints move both ways.
    def optimizer_state_dict(self) -> dict:
        state, off = {}, 0
        for i, p in enumerate(self.gd_params):
            n = p.numel()
            if self.step_count > 0:
                state[i] = {"step": torch.tensor(float(self.step_count)),
                            "exp_avg": self.m[off: off + n].view_as(p).clone(),
                            "exp_avg_sq": self.v[off: off + n].view_as(p).clone()}
            off += n
        group = {"lr": self.lr, "betas": tuple(self.betas), "eps": self.eps, "weight_decay": 0, "amsgrad": False,
                 "maximize": False, "foreach": None, "capturable": False, "differentiable": False, "fused": None,
                 "params": list(range(len(self.gd_params)))}
        return {"state": state, "param_groups": [group]}

    def load_optimizer_state_dict(self, sd: dict) -> None:
        groups = sd["param_groups"]
        if len(groups) != 1 or len(groups[0]["params"]) != len(self.gd_params):
            raise ValueError("optimizer_G state does not match Gd.parameters() (one group, %d tensors expected)"
                             % len(self.gd_params))
        g = groups[0]
        if g.get("weight_decay", 0) or g.get("amsgrad", False) or g.get("maximize", False):
            raise ValueError("the fused Adam step implements torch.optim.Adam without weight_decay/amsgrad/maximize")
        self.lr, self.betas, self.eps = float(g["lr"]), tuple(g["betas"]), float(g["eps"])
        steps, off = set(), 0
        self.m.zero_()
        self.v.zero_()
        for i, p in zip(g["params"], self.gd_params):
            n = p.numel()
            st = sd["state"].get(i)
            if st is not None:
                if tuple(st["exp_avg"].shape) != tuple(p.shape):
                    raise ValueError(f"optimizer_G state {i}: shape {tuple(st['exp_avg'].shape)} != {tuple(p.shape)}")
                self.m[off: off + n].copy_(st["exp_avg"].reshape(-1))
                self.v[off: off + n].copy_(st["exp_avg_sq"].reshape(-1))
                steps.add(int(float(st["step"])))
            off += n
        if len(steps) > 1:
            raise ValueError("optimizer_G state has different step counts per parameter; the fused step keeps one")
        self.step_count = steps.pop() if steps else 0
        self.step_dev.fill_(self.step_count)
        self.graph = None  # a captured graph is still valid (it reads the buffers), but lr/betas are baked in: recapture

    def save_checkpoint(self, path: str, epoch: int = 0, config=None, optimizer_d: Optional[dict] = None) -> None:
        """Writes the reference's checkpoint dictionary (train.py:232-240); loadable by the reference's resume code."""
        self.sync_buffers()
        torch.save({"model_state_dict": self.model.state_dict(), "optimizer_G": self.optimizer_state_dict(),
                    "optimizer_D": optimizer_d if optimizer_d is not None else {}, "epoch": epoch,
                    "resolution": getattr(self.model, "current_resolution", 256), "config": config}, path)

    def load_checkpoint(self, path: str, map_location=None) -> dict:
        """Resume from a checkpoint written by save_checkpoint OR by the reference's train.py; returns the dictionary
        (the caller restores optimizer_D / epoch / config, which are outside the hot path)."""
        ckpt = torch.load(path, map_location=map_location or self.device, weights_only=False)
        self.graph = None  # the graph holds the encoders' bf16 repacks as constants: always recapture after a load
        self.model.load_state_dict(ckpt["model_state_dict"])  # copies INTO the flat parameter views
        ops.invalidate_packed(list(self.model.parameters()))
        if ckpt.get("optimizer_G"):
            self.load_optimizer_state_dict(ckpt["optimizer_G"])
        return ckpt


class IRFDDiscriminatorStep:
    """The reference's discriminator step (train.py:157-183) on the native discriminator.

        D(x_s + n), D(x_t + n)                      -> BCE against real_label 0.9       (instance noise std 0.1)
        x_recon = model(x_s, x_t)[:2] under no_grad  (train mode: the encoders' BN buffers move, as in the reference)
        D(x_s_recon + n), D(x_t_recon + n)          -> BCE against fake_label 0.1
        R1 = (r1(x_s) + r1(x_t)) / 2                 (train.py:246-255; fused second-order node, D.r1_penalty)
        loss_D = real + fake + r1_weight * R1 -> backward -> Adam(lr 5e-5) on D.parameters()   (train.py:347)

    Every D call is its own forward (one spectral-norm power iteration each, like the reference's six calls).  D's
    parameters and gradients are views of flat fp32 buffers, so zero_grad and Adam are one launch each.  By default the
    step launches eagerly and D normalises its weights in the torch spectral-norm hooks.

    `use_cuda_graph=True` captures the whole step into one CUDA graph: the six D calls, each with its own power
    iteration on the native spectral-norm kernels (D.native_spectral_norm()), the instance noise (drawn in the graph
    from the CUDA generator), the no-grad IRFD forward as IRFD.forward_static_stacked (source and target stacked, ONE
    generator call over both, so the generator's noise planes are drawn over the stacked batch), BCE, the fused R1
    node, backward, the data-parallel gradient average and Adam.  The swap and style-mixing draws are taken from the
    CPU generator every step in the order IRFD.forward takes them (StepGraph.draw_ctrl), so a loop that alternates G
    and D steps sees the same CPU RNG stream in either mode.  The generator's bf16 weight repacks run inside the graph
    (the G step's Adam rewrites its weights between D steps); the encoders' are graph constants, so a change of their
    weights (load_state_dict), of any module's mode, of the batch shape, style_mixing_prob, lr, betas, eps, r1_weight
    or noise_std recaptures."""

    def __init__(self, model: IRFD, lr: float = 5e-5, betas=(0.9, 0.999), eps: float = 1e-8, r1_weight: float = 1.0,
                 noise_std: float = 0.1, use_cuda_graph: bool = False):
        self.model = model
        self.lr, self.betas, self.eps = lr, betas, eps
        self.r1_weight, self.noise_std = r1_weight, noise_std
        self.params = list(model.D.parameters())
        self.flat, self.gflat = flatten_parameters(self.params)
        self._grad_views = [p.grad for p in self.params]
        self.m = torch.zeros_like(self.flat)
        self.v = torch.zeros_like(self.flat)
        self.step_count = 0
        self.last = None
        # static-graph state
        self.use_cuda_graph = use_cuda_graph
        self.device = self.flat.device
        self.encoders = [model.Ei, model.Ee, model.Ep]
        self._gd_conv_weights = [p for p in model.Gd.parameters() if p.dim() == 4 and p.shape[-1] == 3]
        self._graphed = StepGraph(model, self.device)
        self.ctrl, self.step_dev = self._graphed.ctrl, self._graphed.step_dev
        self.buckets = GradBuckets(self.device)
        self.world = self.buckets.world
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        self.graph_launches = 0
        self.captures = 0
        self._graph_key = None
        self._static = None

    def _noisy(self, x):
        return torch.add(x.detach(), torch.randn_like(x), alpha=self.noise_std)   # add_instance_noise, train.py:148-149

    def step(self, x_s: torch.Tensor, x_t: torch.Tensor):
        """use_cuda_graph: one graph replay (step_graph).  Otherwise the eager step (step_eager)."""
        if self.use_cuda_graph:
            return self.step_graph(x_s, x_t)
        return self.step_eager(x_s, x_t)

    def step_eager(self, x_s: torch.Tensor, x_t: torch.Tensor):
        model, D = self.model, self.model.D
        # the reference's R1 helper marks the batch as requiring grad (train.py:247); do that to private views so the
        # caller's (possibly reused, in-place refilled) input buffers stay plain tensors
        x_s, x_t = x_s.detach(), x_t.detach()
        self.gflat.zero_()
        for p, v in zip(self.params, self._grad_views):  # keep .grad pointing into the flat buffer
            if p.grad is not v:
                p.grad = v
        d_real_s, d_real_t = D(self._noisy(x_s)), D(self._noisy(x_t))
        loss_real = 0.5 * (_BCELogitsFn.apply(d_real_s, REAL_LABEL) + _BCELogitsFn.apply(d_real_t, REAL_LABEL))
        with torch.no_grad():
            out = model(x_s, x_t)
        d_fake_s, d_fake_t = D(self._noisy(out[0])), D(self._noisy(out[1]))
        loss_fake = 0.5 * (_BCELogitsFn.apply(d_fake_s, FAKE_LABEL) + _BCELogitsFn.apply(d_fake_t, FAKE_LABEL))
        r1 = 0.5 * (D.r1_penalty(x_s) + D.r1_penalty(x_t))
        loss = loss_real + loss_fake + self.r1_weight * r1
        loss.backward()
        self.step_count += 1
        ops.adam_step(self.flat, self.gflat, self.m, self.v, self.lr, self.betas[0], self.betas[1], self.eps,
                      self.step_count)
        self.last = (loss_real.detach(), loss_fake.detach(), r1.detach())
        return loss.detach()

    # ---------------------------------------------------------------------------------------------- static-graph step
    def _static_body(self):
        x_all, out = self._static
        b = x_all.size(0) // 2
        model, D = self.model, self.model.D
        from . import generator

        self.gflat.zero_()
        for p, v in zip(self.params, self._grad_views):
            if p.grad is not v:
                p.grad = v
        x_s, x_t = x_all[:b].detach(), x_all[b:].detach()
        with D.native_spectral_norm():
            d_real_s, d_real_t = D(self._noisy(x_s)), D(self._noisy(x_t))
            loss_real = 0.5 * (_BCELogitsFn.apply(d_real_s, REAL_LABEL) + _BCELogitsFn.apply(d_real_t, REAL_LABEL))
            with torch.no_grad():
                # the G step's Adam rewrote Gd since the last D step: repack its conv weights inside the graph
                ops.invalidate_packed(self._gd_conv_weights)
                if _PREPACK:
                    ops.prepack_conv_weights(generator.synthesis_pack_items(model.Gd.synthesis),
                                             ops.side_stream(self.device))
                img, _, _ = model.forward_static_stacked(x_all, self.ctrl)
            ops.side_stream(self.device).join()
            d_fake_s, d_fake_t = D(self._noisy(img[:b])), D(self._noisy(img[b:]))
            loss_fake = 0.5 * (_BCELogitsFn.apply(d_fake_s, FAKE_LABEL) + _BCELogitsFn.apply(d_fake_t, FAKE_LABEL))
            r1 = 0.5 * (D.r1_penalty(x_s) + D.r1_penalty(x_t))
        loss = loss_real + loss_fake + self.r1_weight * r1
        loss.backward()
        if self.world > 1:   # DDP's gradient average over the ranks (D sits inside the reference's wrapped model)
            self.buckets.launch(self.gflat)
            self.buckets.finish()
        self.step_count += 1
        ops.adam_step(self.flat, self.gflat, self.m, self.v, self.lr, self.betas[0], self.betas[1], self.eps,
                      self.step_count, step_dev=self.step_dev)
        for o, t in zip(out, (loss, loss_real, loss_fake, r1)):
            o.copy_(t.detach())
        # under capture the repacks above were only recorded: eager code must not take them from the pack cache
        ops.invalidate_packed(self._gd_conv_weights)

    def _load_static(self, x_s, x_t):
        """Copy the pair into the stacked static batch [x_s; x_t] (allocated, with the 4 loss scalars, on first use)."""
        if x_s.shape != x_t.shape:
            raise ops._lib.IrfdError(f"IRFDDiscriminatorStep static step: x_s {tuple(x_s.shape)} and x_t "
                                     f"{tuple(x_t.shape)} differ; use step_eager")
        b = x_s.size(0)
        shape = (2 * b,) + tuple(x_s.shape[1:])
        if self._static is None or tuple(self._static[0].shape) != shape:
            self._static = (torch.empty(shape, dtype=torch.float32, device=self.device),
                            torch.zeros(4, dtype=torch.float32, device=self.device))
        self._static[0][:b].copy_(x_s, non_blocking=True)
        self._static[0][b:].copy_(x_t, non_blocking=True)

    def _graph_state(self, x_s):
        """What a captured graph bakes in besides the buffers it reads: module modes, the batch shape, the encoders'
        bf16 repacks (keyed by their weights' version counters), style_mixing_prob and the hyper-parameters that are
        kernel arguments."""
        m = self.model
        enc_ver = tuple(e[0].weight._version for e in self.encoders)
        return (m.training, m.D.training, m.Gd.training, tuple(e.training for e in self.encoders), tuple(x_s.shape),
                enc_ver, float(m.Gd.style_mixing_prob), float(self.lr), tuple(self.betas), float(self.eps),
                float(self.r1_weight), float(self.noise_std), self.buckets.enabled)

    def _finish(self):
        out = self._static[1]
        self.last = (out[1], out[2], out[3])
        return out[0]

    def step_graph(self, x_s: torch.Tensor, x_t: torch.Tensor):
        """One replay of the captured step (captured first, or again when _graph_state changed).  The returned loss
        and `last` are the graph's static outputs: the next step overwrites them."""
        key = self._graph_state(x_s)
        if self.graph is not None and key != self._graph_key:
            self.graph = None
        if self.graph is None:
            self._load_static(x_s, x_t)
            state = [self.flat, self.m, self.v] + list(self.model.D.buffers())
            state += [bf for e in self.encoders for bf in e.buffers()]
            self.graph, self.graph_launches = self._graphed.capture(self, self._static_body, state)
            self._graph_key = key
            self.captures += 1
        self._load_static(x_s, x_t)
        self._graphed.draw_ctrl()
        self.graph.replay()
        self.step_count += 1
        ops.launch_count += self.graph_launches
        return self._finish()

    def step_static_eager(self, x_s: torch.Tensor, x_t: torch.Tensor):
        """The launch sequence of the captured step, launched kernel by kernel: the reference the replay is tested
        against, and a way to time the step per launch (events cannot be recorded inside a replay)."""
        self._load_static(x_s, x_t)
        self._graphed.draw_ctrl()
        self.step_dev.fill_(self.step_count)
        self._static_body()
        return self._finish()
