"""-m gpu: the ResNet-50 encoders back-propagate to an image that a differentiable computation produced.

The stem's data gradient is one grouped dcol GEMM (dz0 @ W, pack mode FLAT_T) and the col2im_stem gather, which sums
the encoders that read the same image.  Checked: the gather and the whole chain against float64 torch on the same bf16
operands, a lone eval-mode encoder against torchvision fp32, the lockstep pass against the one-encoder passes, the
dz0 the kernels actually receive in a train step, the generator chain Ei(Gd(f)), IRFD.forward with non-leaf inputs,
and that leaf images keep their old behaviour (no gradient, no extra launch, bit-identical results)."""
import os
import sys

import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

pytestmark = pytest.mark.gpu


def _rel(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def _images(n, seed, dev, h=256, w=256):
    return (torch.rand(n, 3, h, w, generator=torch.Generator().manual_seed(seed)) * 2 - 1).to(dev)


def _encoder(dev, seed=5, train=True):
    import speak_hack_b200 as P

    torch.manual_seed(seed)
    enc = P.ResNet50Encoder().to(dev)
    return enc.train(train)


def _stem_weights(e, dev, seed=11):
    g = torch.Generator().manual_seed(seed)
    return [(torch.randn(64, 3, 7, 7, generator=g) * 0.05).to(dev) for _ in range(e)]


@pytest.mark.parametrize("hw", [(256, 256), (128, 256), (512, 512), (250, 250), (63, 95)])
@pytest.mark.parametrize("n", [1, 3])
@pytest.mark.parametrize("e", [1, 3])
def test_col2im_stem_matches_fold(cuda_device, e, n, hw):
    from speak_hack_b200 import ops

    h, w = hw
    ho, wo = (h + 1) // 2, (w + 1) // 2
    g = torch.Generator().manual_seed(e * 100 + n * 10 + h)
    dcol = torch.randn(e * n * ho * wo, 192, generator=g).to(cuda_device, torch.bfloat16)
    dx = ops.col2im_stem(dcol, e, n, h, w)
    cols = dcol.double()[:, :147].view(e, n, ho * wo, 147).permute(0, 1, 3, 2)
    ref = sum(F.fold(cols[i], (h, w), 7, padding=3, stride=2) for i in range(e))
    torch.cuda.synchronize()
    err = _rel(dx, ref)
    assert dx.shape == (n, 3, h, w) and err < 1e-5, err
    assert torch.equal(dx, ops.col2im_stem(dcol, e, n, h, w))   # a gather in a fixed order: deterministic


@pytest.mark.parametrize("hw", [(256, 256), (128, 256)])
@pytest.mark.parametrize("e", [1, 3])
def test_stem_dgrad_chain_matches_conv2d_input(cuda_device, e, hw):
    """Pack (FLAT_T) + grouped dcol GEMM + col2im_stem against float64 conv2d_input on the same bf16 dz0 and weights."""
    from speak_hack_b200 import ops

    n, (h, w) = 2, hw
    ws = _stem_weights(e, cuda_device)
    dz0 = torch.randn(e * n, h // 2, w // 2, 64, generator=torch.Generator().manual_seed(3)).to(cuda_device,
                                                                                                 torch.bfloat16)
    wk = ops.pack_conv_weights_stacked(ws, ops.PACK_FLAT_T, 192)
    assert wk.shape == (e * 192, 64) and not wk.view(e, 192, 64)[:, 147:].any()
    dcol = ops.conv_gemm_grouped(dz0.view(1, 1, -1, 64), wk, 1, wgroups=e)
    dx = ops.col2im_stem(dcol.view(-1, 192), e, n, h, w)
    d = dz0.double().view(e, n, h // 2, w // 2, 64).permute(0, 1, 4, 2, 3)
    ref = sum(torch.nn.grad.conv2d_input((n, 3, h, w), ws[i].to(torch.bfloat16).double(), d[i], stride=2, padding=3)
              for i in range(e))
    torch.cuda.synchronize()
    err = _rel(dx, ref)
    print(f"[image-grad] pack + dcol GEMM + col2im_stem vs float64, E={e} {h}x{w}: rel-L2 {err:.3e}")
    assert err < 4e-3, err


def test_eval_lone_encoder_matches_torchvision(cuda_device):
    """Eval mode with autograd, non-leaf input: dL/dx against torchvision's ResNet-50 in fp32 with the same weights, in
    the well-conditioned regime of the eval-mode parameter-gradient check (fresh running statistics, MSE to a target
    far from the features)."""
    import irfd_oracle as O
    import speak_hack_b200 as P

    enc = _encoder(cuda_device, train=False)
    ref = O.make_encoder_ref().to(cuda_device)
    ref.load_state_dict(enc.state_dict())
    ref.eval()
    x, _ = O.synthetic_pair(2, seed=9)
    tgt = (torch.randn(2, 2048, 1, 1, generator=torch.Generator().manual_seed(10)) * 100).to(cuda_device)
    x0 = x.to(cuda_device).requires_grad_(True)
    xr = x0.detach().clone().requires_grad_(True)
    P.mse_loss(enc(x0 * 1), tgt).backward()
    F.mse_loss(ref(xr), tgt).backward()
    torch.cuda.synchronize()
    err = _rel(x0.grad, xr.grad)
    e_w = _rel(enc[0].weight.grad, ref[0].weight.grad)
    print(f"[image-grad] eval lone encoder dL/dx vs torchvision fp32: rel-L2 {err:.3e} (stem weight grad {e_w:.3e})")
    # measured 2.2e-1 on a B200: the bf16 error of dz0 itself, which the stem weight gradient (6.1e-2) averages over
    # every pixel and dL/dx does not; the stem's own data gradient adds 1.7e-3 (test_train_in_context_dz0)
    assert torch.isfinite(x0.grad).all() and err < 0.45, err


def _grp_dx(encs, x0, groups, wt):
    from speak_hack_b200.encoder_group import EncoderGroup

    x0 = x0.detach().clone().requires_grad_(True)
    f = EncoderGroup(encs)(x0 * 1, groups)
    (f * wt[: len(encs)]).sum().backward()
    return x0.grad


def test_train_lockstep_matches_one_encoder_passes(cuda_device, monkeypatch):
    """Train mode, three encoders in lockstep on two statistic groups: dL/dx equals the sum of the three one-member
    passes' dL/dx (the BatchNorm-reduce folds off, so both sum the same terms in the same order per encoder)."""
    from speak_hack_b200 import encoder_group

    monkeypatch.setattr(encoder_group, "fold_bn_reduce", False)
    encs = [_encoder(cuda_device, seed=s) for s in (5, 6, 7)]
    x0 = _images(4, 8, cuda_device)
    wt = torch.randn(3, 4, 2048, 1, 1, generator=torch.Generator().manual_seed(9)).to(cuda_device)
    dx3 = _grp_dx(encs, x0, 2, wt)
    dx1 = sum(_grp_dx([encs[i]], x0, 2, wt[i:i + 1]) for i in range(3))
    torch.cuda.synchronize()
    err = _rel(dx3, dx1)
    print(f"[image-grad] lockstep dL/dx vs sum of one-encoder passes: rel-L2 {err:.3e}")
    assert err <= 1e-5, err


def test_train_in_context_dz0(cuda_device, monkeypatch):
    """Train mode, lockstep: the dz0 the dcol GEMM actually receives, taken to dL/dx by float64 conv2d_input, against
    the image gradient the pass returns.  (End to end, train-mode gradients differ from fp32 by O(0.3), DESIGN §5.)"""
    from speak_hack_b200 import ops
    from speak_hack_b200.encoder_group import EncoderGroup

    encs = [_encoder(cuda_device, seed=s) for s in (5, 6, 7)]
    grp = EncoderGroup(encs)
    x0 = _images(4, 8, cuda_device).requires_grad_(True)
    wt = torch.randn(3, 4, 2048, 1, 1, generator=torch.Generator().manual_seed(9)).to(cuda_device)
    (grp(x0 * 1, 2) * wt).sum().backward()   # caches the packs
    ws = [e[0].weight for e in encs]
    pack = ops.pack_conv_weights_stacked(ws, ops.PACK_FLAT_T, 192)
    seen = []
    orig = ops.conv_gemm_grouped

    def gemm(x, wk, ksize, *a, **kw):
        if wk is pack:
            seen.append(x.clone())
        return orig(x, wk, ksize, *a, **kw)

    monkeypatch.setattr(ops, "conv_gemm_grouped", gemm)
    x0.grad = None
    (grp(x0 * 1, 2) * wt).sum().backward()
    torch.cuda.synchronize()
    assert len(seen) == 1
    d = seen[0].double().view(3, 4, 128, 128, 64).permute(0, 1, 4, 2, 3)
    ref = sum(torch.nn.grad.conv2d_input(tuple(x0.shape), ws[i].to(torch.bfloat16).double(), d[i], stride=2, padding=3)
              for i in range(3))
    err = _rel(x0.grad, ref)
    print(f"[image-grad] train lockstep dL/dx vs conv2d_input on the kernels' dz0: rel-L2 {err:.3e}")
    assert err < 4e-3, err


def test_generator_chain(cuda_device):
    """mse(Ei(Gd(f)), t) in eval mode: Gd receives the encoder's image gradient (at the parent commit its .grad stayed
    None), bit-identical to Gd's backward fed that gradient explicitly, and close to the fp32 oracle chain."""
    import irfd_oracle as O
    import speak_hack_b200 as P
    from parity_util import oracle_noise, product_noise

    dev = cuda_device
    torch.manual_seed(O.WEIGHT_SEED)
    gref = O.StyleGeneratorRef(input_dim=6144)
    O.perturb_noise_weights(gref)
    gd = P.StyleGenerator(input_dim=6144)
    gd.load_state_dict(gref.state_dict())
    gref, gd = gref.to(dev).eval(), gd.to(dev).eval()
    enc = _encoder(dev, train=False)
    eref = O.make_encoder_ref().to(dev)
    eref.load_state_dict(enc.state_dict())
    eref.eval()
    feat = (torch.randn(2, 6144, generator=torch.Generator().manual_seed(3)).abs() * 0.5).to(dev)
    t = torch.randn(2, 2048, 1, 1, generator=torch.Generator().manual_seed(4)).to(dev)

    product_noise(gd, 21)
    img = gd(feat)
    img.retain_grad()
    P.mse_loss(enc(img), t).backward()
    g_chain = {k: p.grad.clone() for k, p in gd.named_parameters() if p.grad is not None}
    assert any(k.startswith("mapping") for k in g_chain) and any(k.startswith("synthesis") for k in g_chain)
    gd.zero_grad(set_to_none=True)
    product_noise(gd, 21)
    img2 = gd(feat)
    img2.backward(img.grad)
    for k, p in gd.named_parameters():
        assert (p.grad is None) == (k not in g_chain) and (p.grad is None or torch.equal(p.grad, g_chain[k])), k

    oracle_noise(gref, 21)
    F.mse_loss(eref(gref(feat)), t).backward()
    torch.cuda.synchronize()
    rr = dict(gref.named_parameters())
    errs = {k: _rel(g, rr[k].grad) for k, g in g_chain.items() if rr[k].grad.norm() > 0}
    worst = max(errs, key=errs.get)
    whole = _rel(torch.cat([g.flatten() for g in g_chain.values()]),
                 torch.cat([rr[k].grad.flatten() for k in g_chain]))
    print(f"[image-grad] Gd grads through Ei vs oracle chain: all params rel-L2 {whole:.3e}, worst {worst} "
          f"{errs[worst]:.3e}")
    assert whole < 3.5e-2 and errs[worst] < 7.8e-2, (whole, worst, errs[worst])   # measured 1.7e-2 / 3.9e-2 on a B200


@pytest.mark.parametrize("batch, train", [(2, True), (1, True), (2, False)])
def test_irfd_forward_non_leaf_inputs(cuda_device, batch, train):
    """IRFD.forward on images produced by a computation: the lockstep pass (B = 2, train) and the per-encoder fallback
    (B = 1: half a tile per statistic group; eval mode with autograd) both send gradients to what produced them."""
    import speak_hack_b200 as P

    torch.manual_seed(0)
    model = P.IRFD().to(cuda_device).train(train)
    a = _images(batch, 1, cuda_device).requires_grad_(True)
    b = _images(batch, 2, cuda_device).requires_grad_(True)
    out = model(a * 0.5, b * 0.5)
    fi_s, fi_t = out[2], out[5]
    (P.mse_loss(fi_s, fi_t) + P.mse_loss(out[0], a.detach()) + P.mse_loss(out[1], b.detach())).backward()
    torch.cuda.synchronize()
    for t in (a, b):
        assert t.grad is not None and torch.isfinite(t.grad).all() and t.grad.abs().sum() > 0


def test_forward_static_stacked_non_leaf(cuda_device):
    import speak_hack_b200 as P

    torch.manual_seed(0)
    model = P.IRFD().to(cuda_device).train()
    x0 = torch.cat([_images(2, 1, cuda_device), _images(2, 2, cuda_device)]).requires_grad_(True)
    ctrl = torch.tensor([0, 14, 14], dtype=torch.int32, device=cuda_device)
    img, f, b = model.forward_static_stacked(x0 * 1, ctrl)
    P.mse_loss(f[0, :b], f[0, b:]).backward()
    torch.cuda.synchronize()
    assert x0.grad is not None and torch.isfinite(x0.grad).all() and x0.grad.abs().sum() > 0
    x1 = x0.detach().clone().requires_grad_(True)   # a leaf: no gradient, as before
    img, f, b = model.forward_static_stacked(x1, ctrl)
    P.mse_loss(f[0, :b], f[0, b:]).backward()
    assert x1.grad is None


def test_leaf_inputs_unchanged(cuda_device):
    """A leaf image gets no gradient and no extra launch; a non-leaf call makes exactly two more launches (the dcol
    GEMM and col2im_stem) and otherwise computes bit for bit what the leaf call computes."""
    from speak_hack_b200 import ops

    enc = _encoder(cuda_device)
    bufs = {k: v.clone() for k, v in enc.named_buffers()}   # restoring the parameters would invalidate the packs
    x = _images(2, 6, cuda_device)
    wt = torch.randn(2, 2048, 1, 1, generator=torch.Generator().manual_seed(7)).to(cuda_device)

    def run(non_leaf):
        with torch.no_grad():
            for k, v in enc.named_buffers():
                v.copy_(bufs[k])
        enc.zero_grad(set_to_none=True)
        x0 = x.clone().requires_grad_(True)
        n0 = ops.launch_count
        f = enc(x0 * 1 if non_leaf else x0)
        (f * wt).sum().backward()
        torch.cuda.synchronize()
        return (ops.launch_count - n0, x0.grad, f.detach().clone(),
                {k: p.grad.clone() for k, p in enc.named_parameters()},
                {k: v.clone() for k, v in enc.state_dict().items()})

    run(True)   # caches every pack, FLAT_T included
    n_nl, dx_nl, f_nl, g_nl, s_nl = run(True)
    n_l, dx_l, f_l, g_l, s_l = run(False)
    assert dx_l is None and dx_nl is not None and torch.isfinite(dx_nl).all()
    assert n_nl - n_l == 2, (n_nl, n_l)
    assert torch.equal(f_nl, f_l)
    assert all(torch.equal(g_nl[k], g_l[k]) for k in g_l)
    assert all(torch.equal(s_nl[k], s_l[k]) for k in s_l)
