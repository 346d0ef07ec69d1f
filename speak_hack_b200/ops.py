"""Tensor-level wrappers over the C ABI: validate, allocate outputs with torch (device-memory plumbing), launch.

Nothing in here computes with PyTorch; every function either launches kernels from libirfd_b200.so or raises.
Activations are NHWC bf16 tensors; parameters and reductions are fp32.
"""
from __future__ import annotations

import ctypes
import os
import weakref
from typing import Optional

import torch

from . import _lib

BF16 = torch.bfloat16
F32 = torch.float32

EPI_PLAIN, EPI_STATS, EPI_STYLE = 0, 1, 2
PACK_FPROP, PACK_DGRAD, PACK_DCOL, PACK_FLAT = 0, 1, 2, 3

# kernels launched through this module since the last reset (bench.py's gpu_launches claim)
launch_count = 0


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _chk(t: torch.Tensor, dtype, name: str) -> None:
    if not t.is_cuda:
        raise _lib.IrfdError(f"{name}: expected a CUDA tensor (the IRFD hot path has no CPU fallback)")
    if t.dtype != dtype:
        raise _lib.IrfdError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise _lib.IrfdError(f"{name}: expected a contiguous tensor")


def _call(name: str, *args, launches: int = 1) -> None:
    global launch_count
    rc = getattr(_lib.load(), name)(*args)
    _lib.check(rc, name)
    launch_count += launches


# Optional per-launch CUDA-event timing of the tensor-core GEMM launches (bench.py's roofline pass).
_gemm_timing = None


def gemm_timing_begin() -> None:
    global _gemm_timing
    _gemm_timing = []


def gemm_timing_end():
    """Returns {family: {name, ms, flops, bytes, launches, records}}; call after torch.cuda.synchronize().
    `records` keeps (ms, flops, bytes) per launch so the caller can form a per-launch roofline bound."""
    global _gemm_timing
    rec, _gemm_timing = _gemm_timing or [], None
    fam = {}
    for name, flops, nbytes, e0, e1 in rec:
        f = fam.setdefault(name, {"name": name, "ms": 0.0, "flops": 0.0, "bytes": 0.0, "launches": 0, "records": []})
        ms = e0.elapsed_time(e1)
        f["ms"] += ms
        f["flops"] += flops
        f["bytes"] += nbytes
        f["launches"] += 1
        f["records"].append((ms, flops, nbytes))
    return fam


class _timed:
    """flops: algorithmic flops of the launch (for memory-bound families the historical convention is bytes here);
    nbytes: algorithmic HBM bytes of the launch (inputs read once + outputs written once)."""

    def __init__(self, name, flops, nbytes=0.0):
        self.name, self.flops, self.nbytes = name, flops, nbytes

    def __enter__(self):
        if _gemm_timing is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e1 = torch.cuda.Event(enable_timing=True)
            self.e0.record()
        return self

    def __exit__(self, *exc):
        if _gemm_timing is not None:
            self.e1.record()
            _gemm_timing.append((self.name, self.flops, self.nbytes, self.e0, self.e1))
        return False


# ----------------------------------------------------------------------------------------------------------------------
# Side stream for weight-gradient launches
# ----------------------------------------------------------------------------------------------------------------------
# In a backward pass the weight gradient of a layer is off the critical path: dz feeds (a) the wgrad GEMM and (b) the
# dgrad GEMM -> BatchNorm / style backward of the next layer.  (a) is tensor-bound, the BN / style passes in (b) are
# HBM-bound, and a persistent GEMM CTA (one per SM, ~210 KB of shared memory) leaves room for a row-streaming block on
# the same SM, so running (a) on a second stream hides most of it.  Fork/join are events, capturable in a CUDA graph.
use_side_stream = os.environ.get("IRFD_SIDE_STREAM", "1") != "0"   # 0: everything on one stream (experiments)
_side_streams = {}


class SideStream:
    def __init__(self, device):
        self.stream = torch.cuda.Stream(device)
        self.keep = []       # tensors the side stream still reads/writes: kept alive (no allocator reuse) until join()
        self.active = False

    def launch(self, fn, *keep):
        """Run fn() (kernel launches only, no allocations) on the side stream, ordered after everything enqueued so far
        on the current stream."""
        if not use_side_stream:
            fn()
            return
        ev = torch.cuda.Event()
        ev.record()
        self.stream.wait_event(ev)
        with torch.cuda.stream(self.stream):
            fn()
        self.keep.extend(keep)
        self.active = True

    def join(self):
        """Order the current stream after the side stream's work; release the kept tensors."""
        if self.active:
            torch.cuda.current_stream().wait_stream(self.stream)
            self.active = False
        self.keep.clear()


def side_stream(device) -> SideStream:
    key = device.index if device.index is not None else torch.cuda.current_device()
    s = _side_streams.get(key)
    if s is None:
        s = _side_streams[key] = SideStream(device)
    return s


_workspace = {}
_workspace_retired = []  # outgrown buffers stay alive: a captured CUDA graph may still hold their addresses


def workspace(nbytes: int, device) -> torch.Tensor:
    """Grow-only scratch buffer (split-K partials, reduction partials), one per (device, stream): every use is
    stream-ordered, and the weight-gradient launches run on their own side stream."""
    key = (device.type, device.index, torch.cuda.current_stream(device).cuda_stream if device.type == "cuda" else 0)
    buf = _workspace.get(key)
    if buf is None or buf.numel() < nbytes:
        if buf is not None:
            _workspace_retired.append(buf)
        buf = torch.empty(max(int(nbytes), 1 << 22), dtype=torch.uint8, device=device)
        _workspace[key] = buf
    return buf


# ----------------------------------------------------------------------------------------------------------------------
# tensor-core GEMMs
# ----------------------------------------------------------------------------------------------------------------------
def conv_gemm(x, wk, ksize, mode=EPI_PLAIN, bias=None, nw=None, noise=None, sp1=None, s1=None, force_block_n=0,
              split_y=False):
    """Stride-1 same-padding conv as implicit GEMM.  x [N,H,W,Cin] bf16, wk [Cout, k*k*Cin] bf16.
    Returns out (mode 0), (out, stat_sum, stat_sq) (mode 1), (a, y) (mode 2), (a, y, y_lo) (mode 2, split_y)."""
    lib = _lib.load()
    _chk(x, BF16, "x")
    _chk(wk, BF16, "wk")
    n, h, w, cin = x.shape
    cout = wk.shape[0]
    if wk.shape[1] != ksize * ksize * cin:
        raise _lib.IrfdError(f"wk shape {tuple(wk.shape)} does not match ksize={ksize}, cin={cin}")
    out = torch.empty((n, h, w, cout), dtype=BF16, device=x.device)
    out2 = torch.empty_like(out) if mode == EPI_STYLE else None
    ssum = ssq = None
    if mode == EPI_STATS:
        mt = lib.irfd_conv_gemm_m_tiles(n, h, w)
        ssum = torch.empty((mt, cout), dtype=F32, device=x.device)
        ssq = torch.empty((mt, cout), dtype=F32, device=x.device)
    for t, nm in ((bias, "bias"), (nw, "nw"), (noise, "noise"), (sp1, "sp1"), (s1, "s1")):
        if t is not None:
            _chk(t, F32, nm)
    m = n * h * w
    nbytes = 2.0 * m * cin + 2.0 * m * cout * (2 if mode == EPI_STYLE else 1) + 2.0 * cin * cout * ksize * ksize
    out_lo = torch.empty_like(out) if (mode == EPI_STYLE and split_y) else None
    with _timed("conv_gemm_kernel (tcgen05 fprop/dgrad)", 2.0 * m * cout * cin * ksize * ksize, nbytes):
        if out_lo is not None:
            _call("irfd_conv_gemm_style_split", x.data_ptr(), n, h, w, cin, wk.data_ptr(), cout, ksize, out.data_ptr(),
                  out2.data_ptr(), out_lo.data_ptr(), _ptr(bias), _ptr(nw), _ptr(noise), _ptr(sp1), _ptr(s1),
                  force_block_n, _stream())
        else:
            _call("irfd_conv_gemm", x.data_ptr(), n, h, w, cin, wk.data_ptr(), cout, ksize, out.data_ptr(), _ptr(out2),
                  mode, _ptr(bias), _ptr(nw), _ptr(noise), _ptr(sp1), _ptr(s1), _ptr(ssum), _ptr(ssq), force_block_n,
                  _stream())
    if mode == EPI_STATS:
        return out, ssum, ssq
    if mode == EPI_STYLE:
        return (out, out2, out_lo) if split_y else (out, out2)
    return out


def conv_gemm_affine(x, wk, ksize, scale, shift, res=None, relu=True, force_block_n=0):
    """Conv with y = act(acc*scale + shift [+ res]) folded into the epilogue (eval-mode BN + ReLU + residual of the
    encoders; conv + bias + leaky ReLU of the discriminator).  relu: False/0 none, True/1 ReLU, 2 leaky ReLU(0.2).
    Returns out [N,H,W,Cout] bf16."""
    _chk(x, BF16, "x")
    _chk(wk, BF16, "wk")
    n, h, w, cin = x.shape
    cout = wk.shape[0]
    out = torch.empty((n, h, w, cout), dtype=BF16, device=x.device)
    if res is not None:
        _chk(res, BF16, "res")
        if res.numel() != out.numel():
            raise _lib.IrfdError("conv_gemm_affine: residual shape mismatch")
    m = n * h * w
    nbytes = 2.0 * m * cin + 2.0 * m * cout * (2 if res is not None else 1) + 2.0 * cin * cout * ksize * ksize
    with _timed("conv_gemm_kernel (tcgen05 fprop/dgrad)", 2.0 * m * cout * cin * ksize * ksize, nbytes):
        _call("irfd_conv_gemm_affine", x.data_ptr(), n, h, w, cin, wk.data_ptr(), cout, ksize, out.data_ptr(),
              scale.data_ptr(), shift.data_ptr(), _ptr(res), int(relu), force_block_n, _stream())
    return out


def conv_gemm_grouped(x, wk, ksize, mode=EPI_PLAIN, wgroups=3, a_shared=False, rows=None, force_block_n=0):
    """One launch for `wgroups` weight sets (the three IRFD encoders).  x [N,H,W,Cin] bf16 stacks the groups' images
    group-major (N = wgroups * images per group); wk [wgroups*Cout, k*k*Cin].  a_shared: x is a 2-D [rows_per_group, K]
    matrix read by every group (the stem's im2col); the output then has wgroups * rows_per_group rows.
    Returns out (mode 0) or (out, stat_sum, stat_sq) (mode 1; partials are [m_tiles, Cout], group-major tiles)."""
    lib = _lib.load()
    _chk(x, BF16, "x")
    _chk(wk, BF16, "wk")
    if wk.shape[0] % wgroups:
        raise _lib.IrfdError(f"conv_gemm_grouped: {wk.shape[0]} weight rows do not split into {wgroups} groups")
    cout = wk.shape[0] // wgroups
    if a_shared:
        m_g, cin = x.shape
        n, h, w = 1, 1, m_g * wgroups
        out = torch.empty((m_g * wgroups, cout), dtype=BF16, device=x.device)
    else:
        n, h, w, cin = x.shape
        out = torch.empty((n, h, w, cout), dtype=BF16, device=x.device)
    if wk.shape[1] != ksize * ksize * cin:
        raise _lib.IrfdError(f"wk shape {tuple(wk.shape)} does not match ksize={ksize}, cin={cin}")
    m = n * h * w
    ssum = ssq = None
    if mode == EPI_STATS:
        mt = lib.irfd_conv_gemm_m_tiles(n, h, w)
        ssum = torch.empty((mt, cout), dtype=F32, device=x.device)
        ssq = torch.empty((mt, cout), dtype=F32, device=x.device)
    nbytes = 2.0 * m * cin / (wgroups if a_shared else 1) + 2.0 * m * cout + 2.0 * wgroups * cin * cout * ksize * ksize
    with _timed("conv_gemm_kernel (tcgen05 fprop/dgrad)", 2.0 * m * cout * cin * ksize * ksize, nbytes):
        _call("irfd_conv_gemm_grouped", x.data_ptr(), n, h, w, cin, wk.data_ptr(), cout, ksize, out.data_ptr(), mode,
              _ptr(ssum), _ptr(ssq), wgroups, 1 if a_shared else 0, force_block_n, _stream())
    if mode == EPI_STATS:
        return out, ssum, ssq
    return out


def conv_gemm_bnbwd_grouped(dy, wk, ksize, z, mean, rstd, gammas, betas, stat_groups, force_block_n=0):
    """Data gradient of a conv whose input was relu(BN(z)), with that BatchNorm's backward reduce pass in the epilogue.
    dy [N,H,W,Cin'] bf16 (groups stacked group-major), wk the stacked dgrad weights [len(gammas)*C, k*k*Cin'], z
    [N,H,W,C].  Returns (g, partial): g = dgrad * (gamma*xhat+beta > 0) bf16, partial [m_tiles, 2, C] fp32 per-tile sums
    of g and g*xhat.  Finish with bn_backward_finish_sets."""
    lib = _lib.load()
    _chk(dy, BF16, "dy")
    _chk(wk, BF16, "wk")
    _chk(z, BF16, "z")
    wgroups = len(gammas)
    n, h, w, cin = dy.shape
    cout = wk.shape[0] // wgroups
    if wk.shape[0] % wgroups or wk.shape[1] != ksize * ksize * cin or z.shape != (n, h, w, cout):
        raise _lib.IrfdError(f"conv_gemm_bnbwd_grouped: wk {tuple(wk.shape)} / z {tuple(z.shape)} do not match dy "
                             f"{tuple(dy.shape)}, ksize={ksize}, {wgroups} groups")
    m = n * h * w
    out = torch.empty((n, h, w, cout), dtype=BF16, device=dy.device)
    partial = torch.empty((lib.irfd_conv_gemm_m_tiles(n, h, w), 2, cout), dtype=F32, device=dy.device)
    nbytes = 2.0 * m * cin + 2 * 2.0 * m * cout + 2.0 * wgroups * cin * cout * ksize * ksize
    with _timed("conv_gemm_kernel (tcgen05 fprop/dgrad)", 2.0 * m * cout * cin * ksize * ksize, nbytes):
        _call("irfd_conv_gemm_bnbwd_grouped", dy.data_ptr(), n, h, w, cin, wk.data_ptr(), cout, ksize, out.data_ptr(),
              z.data_ptr(), mean.data_ptr(), rstd.data_ptr(), _ptr_array(gammas), _ptr_array(betas), partial.data_ptr(),
              stat_groups, wgroups, force_block_n, _stream())
    return out, partial


def conv_gemm_bnbwd_res_grouped(dy, wk, ksize, z, mean, rstd, g2, bits, stat_groups, wgroups=3, force_block_n=0):
    """conv_gemm_bnbwd_grouped for the BatchNorm that closes a Bottleneck: g = (dgrad + g2) * mask with the mask from
    the bit plane `bits` (bn_apply_sets(want_mask=True)).  Returns (g, partial)."""
    lib = _lib.load()
    _chk(dy, BF16, "dy")
    _chk(wk, BF16, "wk")
    _chk(z, BF16, "z")
    _chk(g2, BF16, "g2")
    n, h, w, cin = dy.shape
    cout = wk.shape[0] // wgroups
    m = n * h * w
    if (wk.shape[0] % wgroups or wk.shape[1] != ksize * ksize * cin or z.shape != (n, h, w, cout) or g2.shape != z.shape
            or bits.dtype != torch.uint8 or bits.numel() != m * cout // 8):
        raise _lib.IrfdError(f"conv_gemm_bnbwd_res_grouped: wk {tuple(wk.shape)} / z {tuple(z.shape)} / g2 "
                             f"{tuple(g2.shape)} / bits {tuple(bits.shape)} do not match dy {tuple(dy.shape)}")
    out = torch.empty((n, h, w, cout), dtype=BF16, device=dy.device)
    partial = torch.empty((lib.irfd_conv_gemm_m_tiles(n, h, w), 2, cout), dtype=F32, device=dy.device)
    nbytes = 2.0 * m * cin + (3 + 1.0 / 16) * 2.0 * m * cout + 2.0 * wgroups * cin * cout * ksize * ksize
    with _timed("conv_gemm_kernel (tcgen05 fprop/dgrad)", 2.0 * m * cout * cin * ksize * ksize, nbytes):
        _call("irfd_conv_gemm_bnbwd_res_grouped", dy.data_ptr(), n, h, w, cin, wk.data_ptr(), cout, ksize, out.data_ptr(),
              z.data_ptr(), mean.data_ptr(), rstd.data_ptr(), g2.data_ptr(), bits.data_ptr(), partial.data_ptr(),
              stat_groups, wgroups, force_block_n, _stream())
    return out, partial


def conv_gemm_affine_grouped(x, wk, ksize, scale, shift, res=None, relu=True, wgroups=3, a_shared=False,
                             force_block_n=0):
    """Grouped conv with y = act(acc*scale[g] + shift[g] [+ res]) in the epilogue; scale/shift are [wgroups, Cout]."""
    _chk(x, BF16, "x")
    _chk(wk, BF16, "wk")
    _chk(scale, F32, "scale")
    _chk(shift, F32, "shift")
    cout = wk.shape[0] // wgroups
    if a_shared:
        m_g, cin = x.shape
        n, h, w = 1, 1, m_g * wgroups
        out = torch.empty((m_g * wgroups, cout), dtype=BF16, device=x.device)
    else:
        n, h, w, cin = x.shape
        out = torch.empty((n, h, w, cout), dtype=BF16, device=x.device)
    if scale.numel() != wgroups * cout or shift.numel() != wgroups * cout:
        raise _lib.IrfdError("conv_gemm_affine_grouped: scale/shift must be [wgroups, Cout]")
    if res is not None:
        _chk(res, BF16, "res")
        if res.numel() != out.numel():
            raise _lib.IrfdError("conv_gemm_affine_grouped: residual shape mismatch")
    m = n * h * w
    nbytes = (2.0 * m * cin / (wgroups if a_shared else 1) + 2.0 * m * cout * (2 if res is not None else 1)
              + 2.0 * wgroups * cin * cout * ksize * ksize)
    with _timed("conv_gemm_kernel (tcgen05 fprop/dgrad)", 2.0 * m * cout * cin * ksize * ksize, nbytes):
        _call("irfd_conv_gemm_affine_grouped", x.data_ptr(), n, h, w, cin, wk.data_ptr(), cout, ksize, out.data_ptr(),
              scale.data_ptr(), shift.data_ptr(), _ptr(res), int(relu), wgroups, 1 if a_shared else 0, force_block_n,
              _stream())
    return out


def bn_eval_affine(bn):
    """(scale, shift) of an eval-mode nn.BatchNorm2d, cached on nothing: two tiny launches per call."""
    c = bn.weight.numel()
    scale = torch.empty(c, dtype=F32, device=bn.weight.device)
    shift = torch.empty(c, dtype=F32, device=bn.weight.device)
    _call("irfd_bn_eval_affine", bn.running_mean.data_ptr(), bn.running_var.data_ptr(), bn.weight.data_ptr(),
          bn.bias.data_ptr(), float(bn.eps), scale.data_ptr(), shift.data_ptr(), c, _stream())
    return scale, shift


def gemm_rows(a2d, wk, mode=EPI_PLAIN):
    """Plain GEMM out[M, N] = a2d[M, K] @ wk[N, K]^T through the conv kernel (1x1 conv over a single row of pixels)."""
    m, k = a2d.shape
    r = conv_gemm(a2d.view(1, 1, m, k), wk, 1, mode)
    if mode == EPI_STATS:
        return r[0].view(m, -1), r[1], r[2]
    return r.view(m, -1)


def conv_wgrad(x, dy, ksize, dw=None, beta=0.0, reduce_cin=0, reduce_taps=0, out_shape=None):
    """dW (fp32, OIHW) of a stride-1 same-padding conv from its NHWC bf16 input and output gradient."""
    lib = _lib.load()
    _chk(x, BF16, "x")
    _chk(dy, BF16, "dy")
    n, h, w, cin = x.shape
    cout = dy.shape[-1]
    if dw is None:
        shape = out_shape if out_shape is not None else (cout, cin, ksize, ksize)
        dw = torch.empty(shape, dtype=F32, device=x.device)
        beta = 0.0
    _chk(dw, F32, "dw")
    need = lib.irfd_wgrad_workspace_bytes(n, h, w, cin, cout, ksize)
    ws = workspace(need, x.device)
    nbytes = 2.0 * n * h * w * (cin + cout) + 4.0 * cin * cout * ksize * ksize
    with _timed("wgrad_gemm_kernel (tcgen05 split-K + reduce)", 2.0 * n * h * w * cout * cin * ksize * ksize, nbytes):
        _call("irfd_conv_wgrad", x.data_ptr(), dy.data_ptr(), n, h, w, cin, cout, ksize, dw.data_ptr(), beta,
              reduce_cin, reduce_taps, ws.data_ptr(), ws.numel(), _stream(), launches=2)
    return dw


def conv_wgrad_grouped(x, dy, ksize, dws, x_shared=False, reduce_cin=0, reduce_taps=0):
    """Weight gradients of `len(dws)` weight groups (the same layer of the three encoders) in ONE launch pair.
    x [N,H,W,Cin] / dy [N,H,W,Cout] stack the groups' images group-major (2-D [rows, K] matrices are accepted too);
    x_shared: x is one group's [rows, K] matrix read by every group.  dws: fp32 OIHW destinations (overwritten)."""
    lib = _lib.load()
    _chk(x, BF16, "x")
    _chk(dy, BF16, "dy")
    groups = len(dws)
    for d in dws:
        _chk(d, F32, "dw")
    cin, cout = x.shape[-1], dy.shape[-1]
    if dy.dim() == 4 and not x_shared:
        n, h, w = dy.shape[0], dy.shape[1], dy.shape[2]
    else:
        n, h, w = 1, 1, dy.numel() // cout
    need = lib.irfd_wgrad_workspace_bytes_grouped(n, h, w, cin, cout, ksize, groups)
    if need < 0:
        raise _lib.IrfdError(f"conv_wgrad_grouped: {groups} groups not supported")
    ws = workspace(need, x.device)
    m = n * h * w
    nbytes = 2.0 * m * cout + 2.0 * m * cin / (groups if x_shared else 1) + 4.0 * groups * cin * cout * ksize * ksize
    with _timed("wgrad_gemm_kernel (tcgen05 split-K + reduce)", 2.0 * m * cout * cin * ksize * ksize, nbytes):
        _call("irfd_conv_wgrad_grouped", x.data_ptr(), dy.data_ptr(), n, h, w, cin, cout, ksize, _ptr_array(dws), 0.0,
              reduce_cin, reduce_taps, groups, 1 if x_shared else 0, ws.data_ptr(), ws.numel(), _stream(), launches=2)
    return dws


_pack_cache = {}


def invalidate_packed(params) -> None:
    """Drop cached bf16 repacks of `params` (call after updating them through a raw pointer, e.g. irfd_adam_step)."""
    ptrs = {p.data_ptr() for p in params}
    def hit(k0):  # single-weight entries key on one pointer, stacked entries on a tuple of pointers
        return any(q in ptrs for q in k0) if isinstance(k0, tuple) else k0 in ptrs

    for key in [k for k in _pack_cache if hit(k[0])]:
        del _pack_cache[key]


def pack_conv_weight(w: torch.Tensor, mode: int, kpad: int = 0) -> torch.Tensor:
    """fp32 OIHW parameter -> bf16 GEMM operand, cached until the parameter changes (private repack, SURVEY §8(b)).

    The cache key is (storage pointer, mode); an entry is valid while the tensor's autograd version counter is
    unchanged, which covers every torch-side in-place update (optimizers, load_state_dict, init)."""
    key = (w.data_ptr(), mode, kpad, tuple(w.shape))
    hit = _pack_cache.get(key)
    # the weakref guards against address reuse: a NEW tensor allocated where a freed one lived must not hit
    if hit is not None and hit[0] == w._version and hit[2]() is w:
        return hit[1]
    packed = _pack_conv_weight(w, mode, kpad)
    _pack_cache[key] = (w._version, packed, weakref.ref(w))
    return packed


def prepack_conv_weights(items, side) -> int:
    """Refresh the cached bf16 operands of `items` = [(fp32 OIHW weight, mode), ...] whose parameter changed, with the
    pack kernels on the side stream (`side`: ops.SideStream): the generator's 3x3 weights change at every optimizer step,
    and packed lazily each repack sits on the main stream right before the GEMM that needs it (24 launches per step).
    Issued at the start of a step they hide behind the encoders' forward.  The destinations are allocated here, on the
    calling stream; consumers must be ordered after the side stream's work (the synthesis forward waits, per layer, for a
    style event recorded later on the same side stream).  Returns the number of repacks launched."""
    todo = []
    for w, mode in items:
        key = (w.data_ptr(), mode, 0, tuple(w.shape))
        hit = _pack_cache.get(key)
        if hit is not None and hit[0] == w._version and hit[2]() is w:
            continue
        o, i, kh, kw = w.shape
        shape = (o, kh * kw * i) if mode == PACK_FPROP else (i, kh * kw * o)
        dst = torch.empty(shape, dtype=BF16, device=w.device)
        todo.append((w, mode, dst))
        _pack_cache[key] = (w._version, dst, weakref.ref(w))
    if todo:
        side.launch(lambda: [_pack_conv_weight(w, m, out=d) for w, m, d in todo], *[d for _, _, d in todo])
    return len(todo)


def pack_conv_weights_stacked(ws, mode: int, kpad: int = 0) -> torch.Tensor:
    """Packed bf16 operands of several same-shape conv weights stacked along the rows ([len(ws)*rows, K]) for the
    grouped launches; cached until any of the weights changes (same validity rule as pack_conv_weight)."""
    key = (tuple(w.data_ptr() for w in ws), mode, kpad, tuple(ws[0].shape))
    vers = tuple(w._version for w in ws)
    hit = _pack_cache.get(key)
    if hit is not None and hit[0] == vers and all(r() is w for r, w in zip(hit[2], ws)):
        return hit[1]
    o, i, kh, kw = ws[0].shape
    taps = kh * kw
    rows, cols = {PACK_FPROP: (o, taps * i), PACK_DGRAD: (i, taps * o), PACK_DCOL: (taps * i, o)}.get(mode, (o, kpad))
    dst = torch.empty((len(ws) * rows, cols), dtype=BF16, device=ws[0].device)
    for e, w in enumerate(ws):
        _pack_conv_weight(w, mode, kpad, out=dst[e * rows: (e + 1) * rows])
    _pack_cache[key] = (vers, dst, [weakref.ref(w) for w in ws])
    return dst


def _pack_conv_weight(w: torch.Tensor, mode: int, kpad: int = 0, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _chk(w, F32, "w")
    o, i, kh, kw = w.shape
    taps = kh * kw
    if mode == PACK_FPROP:
        shape = (o, taps * i)
    elif mode == PACK_DGRAD:
        shape = (i, taps * o)
    elif mode == PACK_DCOL:
        shape = (taps * i, o)
    else:
        shape = (o, kpad)
    dst = out if out is not None else torch.empty(shape, dtype=BF16, device=w.device)
    if tuple(dst.shape) != tuple(shape) or not dst.is_contiguous():
        raise _lib.IrfdError(f"_pack_conv_weight: destination {tuple(dst.shape)} != {tuple(shape)}")
    _call("irfd_pack_conv_weight", w.data_ptr(), dst.data_ptr(), o, i, taps, mode, kpad, _stream())
    return dst


# ----------------------------------------------------------------------------------------------------------------------
# BatchNorm
# ----------------------------------------------------------------------------------------------------------------------
def bn_finalize(ssum, ssq, count, eps, momentum, running_mean=None, running_var=None, running_updates=1, groups=1):
    """count = rows PER GROUP.  Returns mean, rstd of shape [groups, C] ([C] when groups == 1)."""
    tiles, c = ssum.shape
    if tiles % groups:
        raise _lib.IrfdError(f"bn_finalize: {tiles} tiles do not split into {groups} groups")
    shape = (c,) if groups == 1 else (groups, c)
    mean = torch.empty(shape, dtype=F32, device=ssum.device)
    rstd = torch.empty(shape, dtype=F32, device=ssum.device)
    _call("irfd_bn_finalize", ssum.data_ptr(), ssq.data_ptr(), tiles // groups, c, int(count), eps, momentum,
          mean.data_ptr(), rstd.data_ptr(), _ptr(running_mean), _ptr(running_var), running_updates, groups, _stream())
    return mean, rstd


def bn_running_update(mean, rstd, eps, count, momentum, running_mean, running_var):
    _call("irfd_bn_running_update", mean.data_ptr(), rstd.data_ptr(), eps, int(count), momentum,
          running_mean.data_ptr(), running_var.data_ptr(), mean.numel(), _stream())


def bn_eval_rstd(running_var, eps):
    rstd = torch.empty_like(running_var)
    _call("irfd_bn_eval_rstd", running_var.data_ptr(), eps, rstd.data_ptr(), running_var.numel(), _stream())
    return rstd


def bn_apply(z, mean, rstd, gamma, beta, res=None, bn2=None, relu=True, groups=1):
    """out = [relu](BN(z) [+ res | + BN2(res)]); bn2 = (mean2, rstd2, gamma2, beta2)."""
    _chk(z, BF16, "z")
    c = z.shape[-1]
    rows = z.numel() // c
    out = torch.empty_like(z)
    m2 = r2 = g2 = b2 = None
    if bn2 is not None:
        m2, r2, g2, b2 = bn2
    _call("irfd_bn_apply", z.data_ptr(), mean.data_ptr(), rstd.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
          _ptr(res), _ptr(m2), _ptr(r2), _ptr(g2), _ptr(b2), out.data_ptr(), rows, c, 1 if relu else 0, groups,
          _stream())
    return out


def bn_backward(g1, g2, act, z, mean, rstd, gamma, want_g_out=False, batch_stats=True, groups=1, beta=None):
    """Returns dz (bf16), dgamma, dbeta (fp32) [, masked g (bf16)]."""
    lib = _lib.load()
    c = z.shape[-1]
    rows = z.numel() // c
    dz = torch.empty_like(z)
    g_out = torch.empty_like(z) if want_g_out else None
    dgamma = torch.empty(c, dtype=F32, device=z.device)
    dbeta = torch.empty(c, dtype=F32, device=z.device)
    ws = workspace(lib.irfd_bn_bwd_workspace_bytes(rows, c, groups), z.device)
    # algorithmic HBM bytes: both passes read g1 [, g2] [, act], z; the apply pass writes dz [, g_out]
    nbytes = _bn_bwd_bytes(rows, c, g2 is not None, 1.0 if act is not None else 0.0, want_g_out)
    with _timed("bn_backward (reduce+finalize+apply, HBM)", nbytes):
        _bn_backward_call(g1, g2, act, z, mean, rstd, gamma, beta, dz, g_out, dgamma, dbeta, batch_stats, rows, c, groups,
                          ws)
    if want_g_out:
        return dz, dgamma, dbeta, g_out
    return dz, dgamma, dbeta


def _bn_backward_call(g1, g2, act, z, mean, rstd, gamma, beta, dz, g_out, dgamma, dbeta, batch_stats, rows, c, groups, ws):
    _call("irfd_bn_backward", g1.data_ptr(), _ptr(g2), _ptr(act), z.data_ptr(), mean.data_ptr(), rstd.data_ptr(),
          gamma.data_ptr(), _ptr(beta), dz.data_ptr(), _ptr(g_out), dgamma.data_ptr(), dbeta.data_ptr(), 0.0,
          1 if batch_stats else 0, rows, c, groups,
          ws.data_ptr(), ws.numel(), _stream(), launches=3)


def _ptr_array(tensors):
    """Host array of device pointers (one per parameter set) for the *_sets entry points; None when no tensor given."""
    if tensors is None:
        return None
    return (ctypes.c_void_p * len(tensors))(*[None if t is None else t.data_ptr() for t in tensors])


def bn_eval_affine_sets(bns):
    """(scale, shift) [nsets, C] of eval-mode nn.BatchNorm2d layers of one shape, one launch."""
    c = bns[0].weight.numel()
    dev = bns[0].weight.device
    scale = torch.empty((len(bns), c), dtype=F32, device=dev)
    shift = torch.empty((len(bns), c), dtype=F32, device=dev)
    _call("irfd_bn_eval_affine_sets", _ptr_array([b.running_mean for b in bns]), _ptr_array([b.running_var for b in bns]),
          _ptr_array([b.weight for b in bns]), _ptr_array([b.bias for b in bns]), float(bns[0].eps), scale.data_ptr(),
          shift.data_ptr(), c, len(bns), _stream())
    return scale, shift


def bn_finalize_sets(ssum, ssq, count, eps, momentum, running_means, running_vars, running_updates, groups, nsets):
    """`nsets` BatchNorm layers of one shape (same layer of the three encoders) x `groups` statistic groups each.
    ssum/ssq: [tiles, C] with the tiles stacked set-major, group-major inside a set.  count = rows PER GROUP.
    Returns mean, rstd [nsets*groups, C]; each set's running buffers are updated in place."""
    tiles, c = ssum.shape
    tot = groups * nsets
    if tiles % tot:
        raise _lib.IrfdError(f"bn_finalize_sets: {tiles} tiles do not split into {nsets} sets x {groups} groups")
    mean = torch.empty((tot, c), dtype=F32, device=ssum.device)
    rstd = torch.empty((tot, c), dtype=F32, device=ssum.device)
    _call("irfd_bn_finalize_sets", ssum.data_ptr(), ssq.data_ptr(), tiles // tot, c, int(count), eps, momentum,
          mean.data_ptr(), rstd.data_ptr(), _ptr_array(running_means), _ptr_array(running_vars), running_updates, groups,
          nsets, _stream())
    return mean, rstd


def bn_apply_sets(z, mean, rstd, gammas, betas, res=None, bn2=None, relu=True, groups=1, want_mask=False):
    """out = [relu](BN(z) [+ res | + BN2(res)]) with per-set gamma/beta lists (len = nsets) and per-group statistics
    (`groups` = TOTAL statistic groups); bn2 = (mean2, rstd2, gammas2, betas2).  want_mask: also return the ReLU mask as
    a bit plane ([rows, C/8] uint8) for bn_backward_sets(act_bits=...)."""
    _chk(z, BF16, "z")
    c = z.shape[-1]
    rows = z.numel() // c
    out = torch.empty_like(z)
    bits = torch.empty((rows, c // 8), dtype=torch.uint8, device=z.device) if want_mask else None
    m2 = r2 = g2 = b2 = None
    if bn2 is not None:
        m2, r2, g2, b2 = bn2
    _call("irfd_bn_apply_sets", z.data_ptr(), mean.data_ptr(), rstd.data_ptr(), _ptr_array(gammas), _ptr_array(betas),
          _ptr(res), _ptr(m2), _ptr(r2), _ptr_array(g2) if g2 is not None else _ptr_array([None] * len(gammas)),
          _ptr_array(b2) if b2 is not None else _ptr_array([None] * len(gammas)), out.data_ptr(), _ptr(bits), rows, c,
          1 if relu else 0, groups, len(gammas), _stream())
    return (out, bits) if want_mask else out


def _bn_bwd_bytes(rows, c, has_g2, mask_units, want_g_out):
    """Algorithmic HBM bytes of reduce + apply.  Without g_out both passes read g1 [, g2] [, mask], z and the apply pass
    writes dz; with g_out the reduce pass also writes the masked gradient and the apply pass reads only that and z."""
    n_in = 2 + (1 if has_g2 else 0) + mask_units
    if want_g_out:
        return 2.0 * rows * c * (n_in + 1 + 3)
    return 2.0 * rows * c * (2 * n_in + 1)


def bn_backward_sets(g1, g2, act, z, mean, rstd, gammas, betas=None, dgammas=None, dbetas=None, want_g_out=False,
                     batch_stats=True, groups=1, act_bits=None):
    """BN backward for `len(gammas)` parameter sets in one launch sequence.  dgammas/dbetas: optional lists of [C] fp32
    output tensors (written, not accumulated); allocated as one [nsets, C] tensor each when omitted.  The ReLU mask comes
    from `act` (post-ReLU tensor), `act_bits` (bn_apply_sets(want_mask=True)) or is recomputed from z when betas is given.
    Returns dz, dgamma(s), dbeta(s) [, masked g]."""
    lib = _lib.load()
    c = z.shape[-1]
    rows = z.numel() // c
    nsets = len(gammas)
    dz = torch.empty_like(z)
    g_out = torch.empty_like(z) if want_g_out else None
    if dgammas is None:
        dg_all = torch.empty((nsets, c), dtype=F32, device=z.device)
        db_all = torch.empty((nsets, c), dtype=F32, device=z.device)
        dgammas, dbetas = list(dg_all.unbind(0)), list(db_all.unbind(0))
    ws = workspace(lib.irfd_bn_bwd_workspace_bytes(rows, c, groups), z.device)
    if act_bits is not None and act is not None:
        raise _lib.IrfdError("bn_backward_sets: pass act or act_bits, not both")
    mask_units = 1.0 if act is not None else (1.0 / 16 if act_bits is not None else 0.0)
    nbytes = _bn_bwd_bytes(rows, c, g2 is not None, mask_units, want_g_out)
    with _timed("bn_backward (reduce+finalize+apply, HBM)", nbytes):
        _call("irfd_bn_backward_sets", g1.data_ptr(), _ptr(g2), _ptr(act if act_bits is None else act_bits),
              0 if act_bits is None else 1, z.data_ptr(), mean.data_ptr(),
              rstd.data_ptr(), _ptr_array(gammas), _ptr_array(betas) if betas is not None else None, dz.data_ptr(),
              _ptr(g_out), _ptr_array(dgammas), _ptr_array(dbetas), 0.0, 1 if batch_stats else 0, rows, c, groups, nsets,
              ws.data_ptr(), ws.numel(), _stream(), launches=3)
    if want_g_out:
        return dz, dgammas, dbetas, g_out
    return dz, dgammas, dbetas


def bn_backward_finish_sets(g, z, mean, rstd, gammas, partial, dgammas=None, dbetas=None, batch_stats=True, groups=1):
    """Second half of a BN backward whose reduce pass ran in conv_gemm_bnbwd_grouped: g is the masked gradient, partial
    [groups * tiles, 2, C] the per-tile sums.  Returns dz, dgammas, dbetas."""
    c = z.shape[-1]
    rows = z.numel() // c
    nsets = len(gammas)
    dz = torch.empty_like(z)
    if dgammas is None:
        dg_all = torch.empty((nsets, c), dtype=F32, device=z.device)
        db_all = torch.empty((nsets, c), dtype=F32, device=z.device)
        dgammas, dbetas = list(dg_all.unbind(0)), list(db_all.unbind(0))
    if partial.shape[0] % groups:
        raise _lib.IrfdError("bn_backward_finish_sets: partial rows do not split into the statistic groups")
    ws = workspace(2 * groups * c * 4, z.device)
    with _timed("bn_backward (reduce+finalize+apply, HBM)", 2.0 * rows * c * 3):
        _call("irfd_bn_backward_finish_sets", g.data_ptr(), z.data_ptr(), mean.data_ptr(), rstd.data_ptr(),
              _ptr_array(gammas), dz.data_ptr(), _ptr_array(dgammas), _ptr_array(dbetas), 0.0, 1 if batch_stats else 0,
              rows, c, groups, nsets, partial.data_ptr(), partial.shape[0] // groups, ws.data_ptr(), ws.numel(), _stream(),
              launches=2)
    return dz, dgammas, dbetas


def conv_geometry(n: int, h: int, w: int, ksize: int, wgroups: int = 1):
    """Pixel-tile geometry the conv GEMM uses for this shape (irfd_conv_gemm_geometry, host-only, no CUDA call):
    (boxed, tw, th, tn, tiles_w, tiles_h, tiles_n), or None when no geometry serves the shape."""
    out = (ctypes.c_int * 7)()
    if _lib.load().irfd_conv_gemm_geometry(n, h, w, ksize, wgroups, out) != _lib.IRFD_OK:
        return None
    return tuple(out)


# ----------------------------------------------------------------------------------------------------------------------
# layout / pooling
# ----------------------------------------------------------------------------------------------------------------------
def half_up(x: int) -> int:
    """Output size of every stride-2 layer of ResNet-50 (7x7/2 p3, MaxPool 3/2 p1, 3x3/2 p1, 1x1/2): ceil(x / 2)."""
    return (x + 1) // 2


def resnet_stage_hw(h: int, w: int):
    """Feature-map sizes of a ResNet-50 on an h x w image: [stem conv, layer1 (after the maxpool), layer2, layer3,
    layer4], each (H, W) — torchvision's arithmetic for any size."""
    sizes = [(half_up(h), half_up(w))]
    for _ in range(4):  # the maxpool (layer1 keeps its size), then the stride-2 first blocks of layer2..4
        sizes.append((half_up(sizes[-1][0]), half_up(sizes[-1][1])))
    return sizes


def im2col_stem(x: torch.Tensor, kpad: int = 192) -> torch.Tensor:
    _chk(x, F32, "x")
    n, c, h, w = x.shape
    if c != 3:
        raise _lib.IrfdError("im2col_stem expects 3 input channels")
    col = torch.empty((n * half_up(h) * half_up(w), kpad), dtype=BF16, device=x.device)
    _call("irfd_im2col_stem", x.data_ptr(), col.data_ptr(), n, h, w, kpad, _stream())
    return col


def im2col_3x3s2(a: torch.Tensor) -> torch.Tensor:
    n, h, w, c = a.shape
    col = torch.empty((n * half_up(h) * half_up(w), 9 * c), dtype=BF16, device=a.device)
    _call("irfd_im2col_3x3s2", a.data_ptr(), col.data_ptr(), n, h, w, c, _stream())
    return col


def col2im_3x3s2(dcol: torch.Tensor, n, h, w, c) -> torch.Tensor:
    dx = torch.empty((n, h, w, c), dtype=BF16, device=dcol.device)
    _call("irfd_col2im_3x3s2", dcol.data_ptr(), dx.data_ptr(), n, h, w, c, _stream())
    return dx


def subsample2(a: torch.Tensor) -> torch.Tensor:
    n, h, w, c = a.shape
    out = torch.empty((n, half_up(h), half_up(w), c), dtype=BF16, device=a.device)
    _call("irfd_subsample2", a.data_ptr(), out.data_ptr(), n, h, w, c, _stream())
    return out


def scatter_add_s2(a: Optional[torch.Tensor], b: torch.Tensor) -> torch.Tensor:
    n, h2, w2, c = b.shape
    out = torch.empty((n, h2 * 2, w2 * 2, c), dtype=BF16, device=b.device)
    _call("irfd_scatter_add_s2", _ptr(a), b.data_ptr(), out.data_ptr(), n, h2 * 2, w2 * 2, c, _stream())
    return out


def maxpool_fwd(a: torch.Tensor):
    n, h, w, c = a.shape
    out = torch.empty((n, half_up(h), half_up(w), c), dtype=BF16, device=a.device)
    arg = torch.empty((n, half_up(h), half_up(w), c), dtype=torch.uint8, device=a.device)
    _call("irfd_maxpool_fwd", a.data_ptr(), out.data_ptr(), arg.data_ptr(), n, h, w, c, _stream())
    return out, arg


def maxpool_bwd(dout: torch.Tensor, arg: torch.Tensor, dout2: Optional[torch.Tensor] = None) -> torch.Tensor:
    n, h2, w2, c = dout.shape
    dx = torch.empty((n, h2 * 2, w2 * 2, c), dtype=BF16, device=dout.device)
    _call("irfd_maxpool_bwd", dout.data_ptr(), _ptr(dout2), arg.data_ptr(), dx.data_ptr(), n, h2 * 2, w2 * 2, c,
          _stream())
    return dx


def avgpool_fwd(a: torch.Tensor) -> torch.Tensor:
    n, h, w, c = a.shape
    out = torch.empty((n, c), dtype=F32, device=a.device)
    _call("irfd_avgpool_fwd", a.data_ptr(), out.data_ptr(), n, h * w, c, _stream())
    return out


def avgpool_bwd(dfeat: torch.Tensor, h: int, w: int) -> torch.Tensor:
    _chk(dfeat, F32, "dfeat")
    n, c = dfeat.shape
    g = torch.empty((n, h, w, c), dtype=BF16, device=dfeat.device)
    _call("irfd_avgpool_bwd", dfeat.data_ptr(), g.data_ptr(), n, h * w, c, _stream())
    return g


# ----------------------------------------------------------------------------------------------------------------------
# synthesis-network pieces
# ----------------------------------------------------------------------------------------------------------------------
def const_input_fwd(cst, bias, nw, noise, sp1, s1, split_y=False):
    """Returns (a0, y0) or, with split_y, (a0, y0, y0_lo): y0 + y0_lo is the split-bf16 source of the first upsample."""
    b, c = sp1.shape
    a0 = torch.empty((b, 4, 4, c), dtype=BF16, device=sp1.device)
    y0 = torch.empty_like(a0)
    y0_lo = torch.empty_like(a0) if split_y else None
    _call("irfd_const_input_split_fwd", cst.data_ptr(), bias.data_ptr(), nw.data_ptr(), noise.data_ptr(),
          sp1.data_ptr(), s1.data_ptr(), a0.data_ptr(), y0.data_ptr(), _ptr(y0_lo), b, c, _stream())
    return (a0, y0, y0_lo) if split_y else (a0, y0)


def const_input_bwd(dy, a0, noise, sp1, outs=None):
    """outs: optional (dconst, dbias, dnw) fp32 destinations (overwritten)."""
    b, c = sp1.shape
    dev = sp1.device
    dsp1 = torch.empty((b, c), dtype=F32, device=dev)
    ds1 = torch.empty((b, c), dtype=F32, device=dev)
    if outs is not None:
        dconst, dbias, dnw = outs
    else:
        dconst = torch.empty((1, c, 4, 4), dtype=F32, device=dev)
        dbias = torch.empty(c, dtype=F32, device=dev)
        dnw = torch.empty(c, dtype=F32, device=dev)
    _call("irfd_const_input_bwd", dy.data_ptr(), a0.data_ptr(), noise.data_ptr(), sp1.data_ptr(), dsp1.data_ptr(),
          ds1.data_ptr(), dconst.data_ptr(), dbias.data_ptr(), dnw.data_ptr(), b, c, _stream())
    return dsp1, ds1, dconst, dbias, dnw


def upsample2x_fwd(x: torch.Tensor, x_lo: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Bilinear x2 of x (+ x_lo when the source is split bf16)."""
    _chk(x, BF16, "x")
    if x_lo is not None:
        _chk(x_lo, BF16, "x_lo")
        if x_lo.shape != x.shape:
            raise _lib.IrfdError("upsample2x_fwd: x_lo shape mismatch")
    b, h, w, c = x.shape
    out = torch.empty((b, 2 * h, 2 * w, c), dtype=BF16, device=x.device)
    _call("irfd_upsample2x_split_fwd", x.data_ptr(), _ptr(x_lo), out.data_ptr(), b, h, w, c, _stream())
    return out


def upsample2x_bwd(dout: torch.Tensor) -> torch.Tensor:
    _chk(dout, BF16, "dout")
    b, h2, w2, c = dout.shape
    din = torch.empty((b, h2 // 2, w2 // 2, c), dtype=BF16, device=dout.device)
    _call("irfd_upsample2x_bwd", dout.data_ptr(), din.data_ptr(), b, h2 // 2, w2 // 2, c, _stream())
    return din


def style_bwd(dy, a, noise, sp1, dbias_out=None, dnw_out=None):
    """Backward of the fused conv epilogue.  Returns dz (bf16), ds1, dsp1 [B,C], dbias, dnw [C] (the last two written
    into dbias_out / dnw_out when given)."""
    lib = _lib.load()
    b, h, w, c = dy.shape
    dev = dy.device
    dz = torch.empty_like(dy)
    ds1 = torch.empty((b, c), dtype=F32, device=dev)
    dsp1 = torch.empty((b, c), dtype=F32, device=dev)
    dbias = dbias_out if dbias_out is not None else torch.empty(c, dtype=F32, device=dev)
    dnw = dnw_out if dnw_out is not None else torch.empty(c, dtype=F32, device=dev)
    ws = workspace(lib.irfd_style_bwd_workspace_bytes(b, h * w, c), dev)
    _call("irfd_style_bwd", dy.data_ptr(), a.data_ptr(), noise.data_ptr(), sp1.data_ptr(), dz.data_ptr(),
          ds1.data_ptr(), dsp1.data_ptr(), dbias.data_ptr(), dnw.data_ptr(), b, h * w, c, ws.data_ptr(), ws.numel(),
          _stream(), launches=2)
    return dz, ds1, dsp1, dbias, dnw


def to_rgb_fwd(y, w, bias):
    b, h, wd, c = y.shape
    out = torch.empty((b, 3, h, wd), dtype=F32, device=y.device)
    _call("irfd_to_rgb_fwd", y.data_ptr(), w.data_ptr(), bias.data_ptr(), out.data_ptr(), b, h * wd, c, _stream())
    return out


def to_rgb_bwd(drgb, y, w, dw_out=None, db_out=None):
    lib = _lib.load()
    _chk(drgb, F32, "drgb")
    b, h, wd, c = y.shape
    dy = torch.empty_like(y)
    dw = dw_out if dw_out is not None else torch.empty((3, c, 1, 1), dtype=F32, device=y.device)
    dbias = db_out if db_out is not None else torch.empty(3, dtype=F32, device=y.device)
    ws = workspace(lib.irfd_to_rgb_bwd_workspace_bytes(b, h * wd, c), y.device)
    _call("irfd_to_rgb_bwd", drgb.data_ptr(), y.data_ptr(), w.data_ptr(), dy.data_ptr(), dw.data_ptr(),
          dbias.data_ptr(), b, h * wd, c, ws.data_ptr(), ws.numel(), _stream(), launches=2)
    return dy, dw, dbias


def nchw_to_nhwc(x: torch.Tensor, c_pad: Optional[int] = None) -> torch.Tensor:
    """[B,C,H,W] fp32 -> [B,H,W,c_pad] bf16 (channels >= C zero)."""
    _chk(x, F32, "x")
    b, c, h, w = x.shape
    cp = c if c_pad is None else c_pad
    out = torch.empty((b, h, w, cp), dtype=BF16, device=x.device)
    _call("irfd_nchw_to_nhwc_bf16", x.data_ptr(), out.data_ptr(), b, c, h * w, cp, _stream())
    return out


def nhwc_to_nchw(x: torch.Tensor, c: Optional[int] = None) -> torch.Tensor:
    """[B,H,W,c_pad] bf16 -> [B,c,H,W] fp32 (first c channels)."""
    _chk(x, BF16, "x")
    b, h, w, cp = x.shape
    c = cp if c is None else c
    out = torch.empty((b, c, h, w), dtype=F32, device=x.device)
    _call("irfd_nhwc_bf16_to_nchw", x.data_ptr(), out.data_ptr(), b, c, h * w, cp, _stream())
    return out


def apply_noise_nchw(x, w, noise):
    _chk(x, F32, "x")
    _chk(w, F32, "w")
    _chk(noise, F32, "noise")
    b, c, h, wd = x.shape
    if noise.numel() != b * h * wd or w.numel() != c:
        raise _lib.IrfdError("apply_noise_nchw: noise must be [B,1,H,W] and weight [C]")
    out = torch.empty_like(x)
    _call("irfd_apply_noise_nchw", x.data_ptr(), w.data_ptr(), noise.data_ptr(), out.data_ptr(), b, c, h * wd, _stream())
    return out


def apply_style_nchw(x, style):
    _chk(x, F32, "x")
    _chk(style, F32, "style")
    b, c, h, wd = x.shape
    if tuple(style.shape) != (b, 2 * c):
        raise _lib.IrfdError(f"apply_style_nchw: style must be [B, 2C] = {(b, 2 * c)}, got {tuple(style.shape)}")
    out = torch.empty_like(x)
    _call("irfd_apply_style_nchw", x.data_ptr(), style.data_ptr(), out.data_ptr(), b, c, h * wd, _stream())
    return out


# ----------------------------------------------------------------------------------------------------------------------
# discriminator pieces
# ----------------------------------------------------------------------------------------------------------------------
def from_rgb_fwd(x, w, bias, lrelu=True):
    """x [B,3,H,W] fp32, w [C,3] fp32, bias [C] or None -> [leaky_relu](conv1x1 + bias) as NHWC bf16 [B,H,W,C]."""
    _chk(x, F32, "x")
    _chk(w, F32, "w")
    if bias is not None:
        _chk(bias, F32, "bias")
    b, ch, h, wd = x.shape
    if ch != 3 or w.shape[1] != 3:
        raise _lib.IrfdError("from_rgb_fwd expects 3 input channels")
    c = w.shape[0]
    out = torch.empty((b, h, wd, c), dtype=BF16, device=x.device)
    _call("irfd_from_rgb_fwd", x.data_ptr(), w.data_ptr(), _ptr(bias), out.data_ptr(), b, h * wd, c,
          1 if lrelu else 0, _stream())
    return out


def bias_lrelu_bwd(g, y):
    """Backward of y = leaky_relu(conv + bias): returns dz (bf16, shape of y) and dbias [C] fp32."""
    lib = _lib.load()
    _chk(g, BF16, "g")
    _chk(y, BF16, "y")
    c = y.shape[-1]
    rows = y.numel() // c
    dz = torch.empty_like(y)
    dbias = torch.empty(c, dtype=F32, device=y.device)
    ws = workspace(lib.irfd_bias_lrelu_bwd_workspace_bytes(rows, c), y.device)
    _call("irfd_bias_lrelu_bwd", g.data_ptr(), y.data_ptr(), dz.data_ptr(), dbias.data_ptr(), rows, c, ws.data_ptr(),
          ws.numel(), _stream(), launches=2)
    return dz, dbias


# ----------------------------------------------------------------------------------------------------------------------
# fp32 dense layers
# ----------------------------------------------------------------------------------------------------------------------
def linear_fwd(x, w, bias, wmul=1.0, bmul=1.0, lrelu=True):
    _chk(x, F32, "x")
    _chk(w, F32, "w")
    b, k = x.shape
    n = w.shape[0]
    y = torch.empty((b, n), dtype=F32, device=x.device)
    _call("irfd_linear_fwd", x.data_ptr(), w.data_ptr(), _ptr(bias), y.data_ptr(), b, n, k, wmul, bmul,
          1 if lrelu else 0, _stream())
    return y


def lrelu_bwd(dy, y):
    _chk(dy, F32, "dy")
    dz = torch.empty_like(dy)
    _call("irfd_lrelu_bwd", dy.data_ptr(), y.data_ptr(), dz.data_ptr(), dy.numel(), _stream())
    return dz


def linear_bwd(dz, x, w, wmul=1.0, bmul=1.0, need_dx=True, dx=None, dx_beta=0.0, need_dw=True, has_bias=True, dw_out=None,
               db_out=None):
    """Returns (dx, dw, db); dx may be accumulated into an existing buffer (dx_beta=1); dw_out / db_out: optional fp32
    destinations of the parameter gradients (overwritten), e.g. views of the trainer's flat gradient buffer."""
    b, n = dz.shape
    k = w.shape[1]
    dev = dz.device
    if need_dx and dx is None:
        dx = torch.empty((b, k), dtype=F32, device=dev)
        dx_beta = 0.0
    dw = (dw_out if dw_out is not None else torch.empty((n, k), dtype=F32, device=dev)) if need_dw else None
    db = (db_out if db_out is not None else torch.empty(n, dtype=F32, device=dev)) if (need_dw and has_bias) else None
    for r0 in range(0, b, 64):  # the kernels keep one accumulator per batch row in registers (<= 64 rows per launch)
        r1 = min(b, r0 + 64)
        _call("irfd_linear_bwd", dz[r0:r1].data_ptr(), _ptr(x[r0:r1]) if x is not None else None, w.data_ptr(),
              dx[r0:r1].data_ptr() if need_dx else None, dx_beta, _ptr(dw), _ptr(db), 0.0 if r0 == 0 else 1.0, r1 - r0,
              n, k, wmul, bmul, _stream(), launches=int(need_dx) + int(need_dw))
    return dx, dw, db


def softmax_rows(x):
    y = torch.empty_like(x)
    _call("irfd_softmax_rows", x.data_ptr(), y.data_ptr(), x.shape[0], x.shape[1], _stream())
    return y


def scale_copy(src, scale):
    dst = torch.empty_like(src)
    _call("irfd_scale_copy", src.data_ptr(), dst.data_ptr(), scale, src.numel(), _stream())
    return dst


def split_style(style, c):
    b = style.shape[0]
    sp1 = torch.empty((b, c), dtype=F32, device=style.device)
    s1 = torch.empty((b, c), dtype=F32, device=style.device)
    _call("irfd_split_style", style.data_ptr(), sp1.data_ptr(), s1.data_ptr(), b, c, _stream())
    return sp1, s1


def merge_style_grad(dsp1, ds1):
    b, c = dsp1.shape
    d = torch.empty((b, 2 * c), dtype=F32, device=dsp1.device)
    _call("irfd_merge_style_grad", dsp1.data_ptr(), ds1.data_ptr(), d.data_ptr(), b, c, _stream())
    return d


# ----------------------------------------------------------------------------------------------------------------------
# losses / optimiser
# ----------------------------------------------------------------------------------------------------------------------
def mse_fwd(a, b, out=None, out_beta=0.0):
    lib = _lib.load()
    _chk(a, F32, "a")
    _chk(b, F32, "b")
    if out is None:
        out = torch.empty(1, dtype=F32, device=a.device)
        out_beta = 0.0
    ws = workspace(lib.irfd_reduce_workspace_bytes(), a.device)
    _call("irfd_mse_fwd", a.data_ptr(), b.data_ptr(), a.numel(), out.data_ptr(), out_beta, ws.data_ptr(), ws.numel(),
          _stream(), launches=2)
    return out


def mse_bwd(a, b, gscale, need_da=True, need_db=False):
    da = torch.empty_like(a) if need_da else None
    db = torch.empty_like(a) if need_db else None
    _call("irfd_mse_bwd", a.data_ptr(), b.data_ptr(), a.numel(), gscale.data_ptr(), _ptr(da), _ptr(db), _stream())
    return da, db


def sumsq(g, out=None, out_beta=0.0):
    lib = _lib.load()
    if out is None:
        out = torch.empty(1, dtype=F32, device=g.device)
        out_beta = 0.0
    ws = workspace(lib.irfd_reduce_workspace_bytes(), g.device)
    _call("irfd_sumsq", g.data_ptr(), g.numel(), out.data_ptr(), out_beta, ws.data_ptr(), ws.numel(), _stream(),
          launches=2)
    return out


def adam_step(p, g, m, v, lr, beta1, beta2, eps, step, total_sumsq=None, max_norm=0.0, step_dev=None):
    _call("irfd_adam_step", p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel(), lr, beta1, beta2, eps,
          step, _ptr(step_dev), _ptr(total_sumsq), max_norm, _stream(), launches=1 if step_dev is None else 2)


# ----------------------------------------------------------------------------------------------------------------------
# device-side routing (static-graph mode)
# ----------------------------------------------------------------------------------------------------------------------
def style_rows_fwd(w, w2, ctrl, ctrl_idx, psi, cutoff, num_layers, b_first=None):
    """b_first: the batch stacks two generator calls; rows [0, b_first) use ctrl[ctrl_idx], the rest ctrl[ctrl_idx+1]."""
    b, k = w.shape
    rows_t = torch.empty((num_layers, b, k), dtype=F32, device=w.device)
    _call("irfd_style_rows_pair_fwd", w.data_ptr(), w2.data_ptr(), ctrl.data_ptr(), ctrl_idx, psi, cutoff,
          rows_t.data_ptr(), num_layers, b, k, b if b_first is None else b_first, _stream())
    return rows_t


def style_rows_bwd(drows_t, psi, cutoff):
    l, b, k = drows_t.shape
    dw = torch.empty((b, k), dtype=F32, device=drows_t.device)
    _call("irfd_style_rows_bwd", drows_t.data_ptr(), psi, cutoff, dw.data_ptr(), l, b, k, _stream())
    return dw


def swap_cat_fwd(feats, ctrl, out=None):
    """feats = (fi_s, fe_s, fp_s, fi_t, fe_t, fp_t), each [B, C] fp32 contiguous.  out: optional [2B, 3C] buffer whose
    halves receive the source and the target generator inputs (one stacked generator call)."""
    b, c = feats[0].shape
    if out is not None:
        _chk(out, F32, "out")
        gen_s, gen_t = out[:b], out[b:]
    else:
        gen_s = torch.empty((b, 3 * c), dtype=F32, device=feats[0].device)
        gen_t = torch.empty_like(gen_s)
    _call("irfd_swap_cat_fwd", *[f.data_ptr() for f in feats], ctrl.data_ptr(), gen_s.data_ptr(), gen_t.data_ptr(), b,
          c, _stream())
    return gen_s, gen_t


def swap_cat_bwd(dgen_s, dgen_t, ctrl, c, outs=None):
    """outs: optional six [B, C] fp32 destinations (e.g. slices of one stacked feature-gradient buffer)."""
    b = dgen_s.shape[0]
    if outs is None:
        outs = [torch.empty((b, c), dtype=F32, device=dgen_s.device) for _ in range(6)]
    _call("irfd_swap_cat_bwd", dgen_s.data_ptr(), dgen_t.data_ptr(), ctrl.data_ptr(), *[o.data_ptr() for o in outs], b,
          c, _stream())
    return outs
