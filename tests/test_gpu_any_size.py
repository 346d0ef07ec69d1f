"""-m gpu: eval-mode encoders and IRFD inference at any image size — the box-tiled conv geometry (PLAIN / AFFINE, weight
groups, no writes outside the output), the ceil-sized stride-2 layout kernels, the encoder and the full eval forward
against the fp32 oracle at sizes that are not a power of two, graph replay equal to the eager forward, and clean
refusals of the passes that keep the old shape rules."""
import ctypes
import os
import sys

import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))

pytestmark = pytest.mark.gpu

BOX_SHAPES = [(56, 56), (28, 28), (14, 14), (7, 7), (80, 80), (40, 40), (10, 10), (96, 96), (48, 48), (12, 12),
              (63, 63), (32, 19), (19, 32), (144, 144), (200, 72)]


def rel_l2(a, b):
    a = a.double()
    b = b.double()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def _mk(n, h, w, cin, cout, dev, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, h, w, cin, generator=g).to(dev).to(torch.bfloat16)
    wt = (torch.randn(cout, cin, 3, 3, generator=g) / (cin * 9) ** 0.5).to(dev).to(torch.bfloat16)
    wk = wt.permute(0, 2, 3, 1).contiguous().reshape(cout, 9 * cin)
    return x, wt, wk


def _ref(x, wt):
    return F.conv2d(x.float().permute(0, 3, 1, 2), wt.float(), padding=1).permute(0, 2, 3, 1)


@pytest.mark.parametrize("h,w", BOX_SHAPES)
def test_box_tiled_conv_matches_conv2d(cuda_device, h, w):
    from speak_hack_b200 import ops

    dev = cuda_device
    for n in (1, 2, 3, 5):
        geo = ops.conv_geometry(n, h, w, 3)
        assert geo is not None and geo[0] == 1, (n, h, w, geo)
        for bn in (64, 128, 256):
            cin, cout = (64, 256) if bn != 128 else (128, 128)
            x, wt, wk = _mk(n, h, w, cin, cout, dev, seed=n * 1000 + h * 7 + w)
            g = torch.Generator().manual_seed(bn + n)
            bias = torch.randn(cout, generator=g).to(dev)
            scale = (torch.rand(cout, generator=g) + 0.5).to(dev)
            shift = torch.randn(cout, generator=g).to(dev)
            res = torch.randn(n, h, w, cout, generator=g).to(dev).to(torch.bfloat16)
            ref = _ref(x, wt)
            y = ops.conv_gemm(x, wk, 3, ops.EPI_PLAIN, force_block_n=bn)
            yb = ops.conv_gemm(x, wk, 3, ops.EPI_PLAIN, bias=bias, force_block_n=bn)
            ya = ops.conv_gemm_affine(x, wk, 3, scale, shift, relu=True, force_block_n=bn)
            yr = ops.conv_gemm_affine(x, wk, 3, scale, shift, res=res, relu=False, force_block_n=bn)
            torch.cuda.synchronize()
            aff = ref * scale + shift
            for got, want, what in ((y, ref, "plain"), (yb, ref + bias, "plain+bias"), (ya, aff.clamp_min(0), "affine relu"),
                                    (yr, aff + res.float(), "affine+res")):
                assert rel_l2(got.float(), want) < 4e-3, (n, h, w, bn, what)


@pytest.mark.parametrize("n,h,w,cin,cout", [(2, 7, 7, 512, 512), (3, 14, 14, 256, 256), (1, 28, 28, 128, 512),
                                            (5, 63, 63, 64, 64), (2, 19, 32, 512, 128)])
def test_box_tiled_conv_wide_channels(cuda_device, n, h, w, cin, cout):
    from speak_hack_b200 import ops

    x, wt, wk = _mk(n, h, w, cin, cout, cuda_device, seed=3)
    scale = torch.ones(cout, device=cuda_device)
    shift = torch.zeros(cout, device=cuda_device)
    y = ops.conv_gemm(x, wk, 3, ops.EPI_PLAIN)
    ya = ops.conv_gemm_affine(x, wk, 3, scale, shift, relu=False)
    torch.cuda.synchronize()
    ref = _ref(x, wt)
    assert rel_l2(y.float(), ref) < 4e-3 and torch.equal(y, ya)


@pytest.mark.parametrize("h,w", BOX_SHAPES)
def test_box_tiled_conv_writes_nothing_outside_the_output(cuda_device, h, w):
    """Called through the C ABI with the output inside a larger buffer: the sentinel bytes before and after it stay."""
    from speak_hack_b200 import _lib, ops

    lib = _lib.load()
    dev = cuda_device
    for n in (1, 2, 3, 5):
        for bn, cout in ((64, 64), (128, 128), (256, 256)):
            x, wt, wk = _mk(n, h, w, 64, cout, dev, seed=11)
            scale = torch.ones(cout, device=dev)
            shift = torch.zeros(cout, device=dev)
            numel = n * h * w * cout
            pad = 128 * 256 + 1000  # more than one whole tile of rows on each side
            buf = torch.full((numel + 2 * pad,), -7.25, dtype=torch.bfloat16, device=dev)
            out_ptr = buf.data_ptr() + pad * 2
            for mode in ("plain", "affine"):
                if mode == "plain":
                    rc = lib.irfd_conv_gemm(x.data_ptr(), n, h, w, 64, wk.data_ptr(), cout, 3, out_ptr, None, 0, None,
                                            None, None, None, None, None, None, bn, ops._stream())
                else:
                    rc = lib.irfd_conv_gemm_affine(x.data_ptr(), n, h, w, 64, wk.data_ptr(), cout, 3, out_ptr,
                                                   scale.data_ptr(), shift.data_ptr(), None, 0, bn, ops._stream())
                _lib.check(rc, mode)
                torch.cuda.synchronize()
                assert (buf[:pad] == -7.25).all() and (buf[pad + numel:] == -7.25).all(), (n, h, w, bn, mode)
                got = buf[pad:pad + numel].view(n, h, w, cout)
                assert rel_l2(got.float(), _ref(x, wt)) < 4e-3, (n, h, w, bn, mode)


@pytest.mark.parametrize("per,h,w,cout", [(1, 56, 56, 64), (2, 7, 7, 512), (3, 14, 14, 256), (2, 19, 32, 128),
                                          (1, 28, 28, 128), (5, 10, 10, 256)])
def test_grouped_box_tiled_conv_equals_per_group(cuda_device, per, h, w, cout):
    from speak_hack_b200 import ops

    dev = cuda_device
    E = 3
    assert ops.conv_geometry(E * per, h, w, 3, E)[0] == 1
    g = torch.Generator().manual_seed(per * 31 + h)
    x = torch.randn(E * per, h, w, 64, generator=g).to(dev).to(torch.bfloat16)
    wks = [(torch.randn(cout, 9 * 64, generator=g) / 24).to(dev).to(torch.bfloat16) for _ in range(E)]
    sc = (torch.rand(E, cout, generator=g) + 0.5).to(dev)
    sh = torch.randn(E, cout, generator=g).to(dev)
    res = torch.randn(E * per, h, w, cout, generator=g).to(dev).to(torch.bfloat16)
    for r, relu in ((None, True), (res, True), (res, False)):
        got = ops.conv_gemm_affine_grouped(x, torch.cat(wks).contiguous(), 3, sc, sh, res=r, relu=relu, wgroups=E)
        for e in range(E):
            rs = None if r is None else r[e * per:(e + 1) * per].contiguous()
            want = ops.conv_gemm_affine(x[e * per:(e + 1) * per].contiguous(), wks[e], 3, sc[e].contiguous(),
                                        sh[e].contiguous(), res=rs, relu=relu)
            torch.cuda.synchronize()
            assert torch.equal(got[e * per:(e + 1) * per], want), (per, h, w, e)


LAYOUT_SIZES = [(31, 30), (30, 31), (33, 47), (34, 38), (224, 224), (250, 250), (27, 81), (7, 5), (64, 64)]


@pytest.mark.parametrize("h,w", LAYOUT_SIZES)
def test_layout_kernels_at_any_size(cuda_device, h, w):
    from speak_hack_b200 import ops

    dev = cuda_device
    g = torch.Generator().manual_seed(h * 1000 + w)
    n = 2
    # stem im2col: 7x7 / 2, pad 3, k = c * 49 + kh * 7 + kw, zero padded to 192 columns
    x = (torch.rand(n, 3, h, w, generator=g) * 2 - 1).to(dev)
    col = ops.im2col_stem(x, 192)
    ho, wo = ops.half_up(h), ops.half_up(w)
    ref = F.unfold(x, 7, padding=3, stride=2).transpose(1, 2).reshape(n * ho * wo, 147).to(torch.bfloat16)
    torch.cuda.synchronize()
    assert col.shape == (n * ho * wo, 192)
    assert torch.equal(col[:, :147], ref) and (col[:, 147:] == 0).all()
    # NHWC bf16 activations
    c = 64
    a = torch.randn(n, h, w, c, generator=g).to(dev).to(torch.bfloat16)
    an = a.float().permute(0, 3, 1, 2)
    mp, _ = ops.maxpool_fwd(a)
    want = F.max_pool2d(an, 3, 2, 1).permute(0, 2, 3, 1).to(torch.bfloat16)
    col2 = ops.im2col_3x3s2(a)
    want2 = F.unfold(an, 3, padding=1, stride=2).view(n, c, 9, ho * wo).permute(0, 3, 2, 1).reshape(n * ho * wo, 9 * c)
    sub = ops.subsample2(a)
    torch.cuda.synchronize()
    assert mp.shape == (n, ho, wo, c) and torch.equal(mp, want)
    assert torch.equal(col2, want2.to(torch.bfloat16))
    assert torch.equal(sub, a[:, ::2, ::2, :])


@pytest.fixture(scope="module")
def nets(cuda_device):
    import irfd_oracle as O
    import speak_hack_b200 as P

    torch.manual_seed(O.WEIGHT_SEED)
    ref = O.IRFDRef().eval()
    net = P.IRFD()
    net.load_state_dict(ref.state_dict())
    return ref, net.to(cuda_device).eval()


@pytest.mark.parametrize("h,w", [(224, 224), (320, 320), (384, 384), (250, 250), (300, 200), (33, 47)])
def test_encoder_features_at_any_size(cuda_device, nets, h, w):
    ref, net = nets
    g = torch.Generator().manual_seed(h + w)
    x = torch.rand(2, 3, h, w, generator=g) * 2 - 1
    with torch.no_grad():
        f_ref = ref.Ei(x)
        f = net.Ei(x.to(cuda_device))
    torch.cuda.synchronize()
    e = rel_l2(f.cpu(), f_ref)
    print(f"[any-size] encoder eval {h}x{w}: features rel-L2 {e:.3e}")
    assert f.shape == (2, 2048, 1, 1) and e < 6e-3


def test_full_eval_forward_224(cuda_device, nets):
    import irfd_oracle as O

    ref, net = nets
    x_s, x_t = O.synthetic_pair(2, res=224)
    torch.manual_seed(O.FORWARD_SEED)
    with torch.no_grad():
        o_ref = ref(x_s, x_t)
    torch.manual_seed(O.FORWARD_SEED)
    with torch.no_grad():
        o = net(x_s.to(cuda_device), x_t.to(cuda_device))
    torch.cuda.synchronize()
    e_feat = max(O.rel_l2(a, b) for a, b in zip(o[2:8], o_ref[2:8]))
    e_img = max(O.rel_l2(o[0], o_ref[0]), O.rel_l2(o[1], o_ref[1]))
    print(f"[any-size] IRFD eval forward 224^2: features {e_feat:.3e}, images {e_img:.3e}")
    assert e_feat < 8e-3 and e_img < 8e-2


def test_mixed_source_and_target_sizes(cuda_device, nets):
    _, net = nets
    g = torch.Generator().manual_seed(4)
    xs = (torch.rand(2, 3, 224, 224, generator=g) * 2 - 1).to(cuda_device)
    xt = (torch.rand(2, 3, 250, 200, generator=g) * 2 - 1).to(cuda_device)
    with torch.no_grad():
        o = net(xs, xt)
        fi_t = net.Ei(xt)
    torch.cuda.synchronize()
    assert o[0].shape == o[1].shape == (2, 3, 256, 256)
    assert torch.isfinite(o[0]).all() and torch.isfinite(o[1]).all()
    assert torch.equal(o[5], fi_t) or torch.equal(o[2], fi_t)  # swap type 0 exchanges the identity codes


@pytest.fixture(scope="module")
def warmed_net(cuda_device):
    """IRFD with realistic BatchNorm running buffers (two train-mode forwards at 256^2; fresh buffers blow the
    eval-mode activations up), in eval mode."""
    import irfd_oracle as O
    import speak_hack_b200 as P

    torch.manual_seed(O.WEIGHT_SEED)
    net = P.IRFD().to(cuda_device).train()
    x_s, x_t = O.synthetic_pair(2)
    with torch.no_grad():
        for _ in range(2):
            net(x_s.to(cuda_device), x_t.to(cuda_device))
    return net.eval()


@pytest.mark.parametrize("b,lockstep", [(2, False), (64, True)])
def test_graph_replay_equals_eager_at_224(cuda_device, warmed_net, b, lockstep):
    import irfd_oracle as O
    from speak_hack_b200.inference import IRFDInference

    net = warmed_net
    x_s, x_t = O.synthetic_pair(b, res=224)
    xs, xt = x_s.to(cuda_device), x_t.to(cuda_device)
    assert net.encoder_group.can_run(torch.cat([xs, xt]), 2) == lockstep
    run = IRFDInference(net, xs, xt)
    seen = set()
    for seed in range(12):
        torch.manual_seed(seed)
        swap = int(torch.randint(0, 3, (1,)))
        if swap in seen:
            continue
        seen.add(swap)
        torch.manual_seed(seed)
        with torch.no_grad():
            want = net(xs, xt)
        torch.manual_seed(seed)
        got = [t.clone() for t in run(xs, xt)]
        torch.cuda.synchronize()
        assert torch.isfinite(want[0]).all()
        assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1]), f"swap {swap}"
        fi_s, fi_t = (want[5], want[2]) if swap == 0 else (want[2], want[5])
        assert torch.equal(got[2], fi_s) and torch.equal(got[3], fi_t)
    assert seen == {0, 1, 2}


def _bn_state(net):
    return {k: v.clone() for k, v in net.state_dict().items() if "running" in k or "num_batches" in k}


def test_clean_refusals(cuda_device, warmed_net):
    from speak_hack_b200._lib import IrfdError

    net = warmed_net
    dev = cuda_device
    g = torch.Generator().manual_seed(9)
    x = (torch.rand(2, 3, 224, 224, generator=g) * 2 - 1).to(dev)
    before = _bn_state(net)
    try:
        net.train()
        with torch.no_grad():
            with pytest.raises(IrfdError):
                net.Ei(x)
            with pytest.raises(IrfdError):
                net(x, x)
        with pytest.raises(IrfdError):   # differentiated train-mode pass
            net.Ee(x.clone().requires_grad_(True))
        net.eval()
        with pytest.raises(IrfdError):   # eval mode with autograd (the parameters require grad)
            net.Ep(x)
        torch.cuda.synchronize()
        after = _bn_state(net)
        assert all(torch.equal(before[k], after[k]) for k in before)
        with torch.no_grad():
            for shape in ((1, 3, 64, 580), (1, 3, 31, 64), (1, 3, 64, 31), (1, 3, 16, 16)):
                with pytest.raises(IrfdError):
                    net.Ei(torch.zeros(shape, device=dev))
            f = net.Ei(torch.zeros((1, 3, 32, 579), device=dev))   # the limits themselves run
        torch.cuda.synchronize()
        assert f.shape == (1, 2048, 1, 1)
    finally:
        net.eval()
