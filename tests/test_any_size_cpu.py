"""CPU: the pixel-tile geometry of the conv GEMM (irfd_conv_gemm_geometry) covers every output pixel exactly once at
any size, keeps the linear geometry for every shape it served before, refuses the modes the box-tiled instances do not
implement before any CUDA call, and the stage-size helper matches torchvision's ResNet-50 at any image size."""
import ctypes

import numpy as np
import pytest
import torch


@pytest.fixture(scope="module")
def lib():
    import os

    from speak_hack_b200 import _lib, build

    if not os.path.exists(_lib.LIB_PATH):
        build.build(verbose=False)
    return _lib.load()


def _geo(lib, n, h, w, k, g):
    out = (ctypes.c_int * 7)()
    rc = lib.irfd_conv_gemm_geometry(n, h, w, k, g, out)
    return rc, tuple(out)


def _old_rule_accepts(n, h, w, k, g):
    """The 3x3 / pointwise shape rule of the linear geometry, as conv_gemm_impl applied it before box tiles existed."""
    m = n * h * w
    if g > 1 and m % (128 * g):
        return False
    H, W = (1, m) if k == 1 else (h, w)
    if W >= 128:
        return k == 1 or W % 128 == 0
    if 128 % W:
        return False
    rows = 128 // W
    return H % rows == 0 if H >= rows else rows % H == 0


def test_box_tiles_cover_every_pixel_exactly_once(lib):
    checked = boxed = 0
    for g in (1, 3):
        for n in range(1, 6):
            for h in range(1, 161):
                for w in range(1, 601):
                    rc, (bx, tw, th, tn, tiles_w, tiles_h, tiles_n) = _geo(lib, n, h, w, 3, g)
                    if g > 1 and n % g and not _old_rule_accepts(n, h, w, 3, g):
                        assert rc == -1, (n, h, w, g)  # images cannot split into the weight groups
                        continue
                    assert rc == 0, (n, h, w, g)
                    checked += 1
                    if not bx:
                        continue
                    boxed += 1
                    assert 1 <= tw * th * tn <= 128, (n, h, w, g)
                    assert tw <= 128 and th <= 128 and tn <= n
                    # a regular grid of boxes: disjoint by construction, so "exactly once" == the grid covers the image
                    # and no box row / column / image slot starts past it
                    assert (tiles_w - 1) * tw < w <= tiles_w * tw, (n, h, w, g)
                    assert (tiles_h - 1) * th < h <= tiles_h * th, (n, h, w, g)
                    assert (tiles_n - 1) * tn < n <= tiles_n * tn, (n, h, w, g)
                    if w < 128:
                        assert tw == w and th == min(h, 128 // w)
                        if th < h:
                            assert tn == 1
                    else:
                        assert tw == 128 and th == 1 and tn == 1
                    if g > 1:  # whole tiles per weight group: every box holds images of one group only
                        assert (n // g) % tn == 0 and (tiles_n % g) == 0, (n, h, w, g)
    assert checked > 500000 and boxed > checked // 2


@pytest.mark.parametrize("n,h,w,g", [(1, 7, 7, 1), (3, 7, 7, 1), (2, 14, 14, 1), (5, 19, 32, 1), (1, 144, 200, 1),
                                     (6, 7, 7, 3), (3, 13, 9, 3), (6, 56, 56, 3), (2, 1, 131, 1)])
def test_box_tiles_enumerated(lib, n, h, w, g):
    """Explicit enumeration: every pixel of the [n, h, w] output lies in exactly one box, in tile order image-major,
    then rows, then columns, and with weight groups every box lies inside one group's images."""
    rc, (bx, tw, th, tn, tiles_w, tiles_h, tiles_n) = _geo(lib, n, h, w, 3, g)
    assert rc == 0 and bx == 1
    hits = np.zeros((n, h, w), dtype=np.int32)
    per_group = n // g
    for t in range(tiles_w * tiles_h * tiles_n):
        wt, rest = t % tiles_w, t // tiles_w
        ht, nt = rest % tiles_h, rest // tiles_h
        n0, h0, w0 = nt * tn, ht * th, wt * tw
        hits[n0:n0 + tn, h0:h0 + th, w0:w0 + tw] += 1
        if g > 1:
            group = t // (tiles_w * tiles_h * tiles_n // g)
            assert n0 // per_group == group and (min(n0 + tn, n) - 1) // per_group == group
    assert (hits == 1).all()


def test_old_shapes_keep_the_linear_geometry(lib):
    count = 0
    for k in (1, 3):
        for g in (1, 3):
            for n in range(1, 7):
                for h in list(range(1, 34)) + [48, 56, 64, 96, 112, 128, 256]:
                    for w in list(range(1, 34)) + [48, 56, 64, 96, 112, 128, 256, 384, 512]:
                        if not _old_rule_accepts(n, h, w, k, g):
                            continue
                        rc, o = _geo(lib, n, h, w, k, g)
                        assert rc == 0 and o[0] == 0, (n, h, w, k, g, o)
                        assert o[4] * o[5] * o[6] == lib.irfd_conv_gemm_m_tiles(n, h, w), (n, h, w, k, g, o)
                        count += 1
    assert count > 1000


def test_pointwise_shapes(lib):
    # a pointwise conv is one long row: linear from 128 pixels on, box-tiled (one short row) below when 128 % M != 0
    assert _geo(lib, 1, 1, 1000, 1, 1) == (0, (0, 128, 1, 1, 8, 1, 1))
    assert _geo(lib, 2, 7, 7, 1, 1) == (0, (1, 98, 1, 1, 1, 1, 1))
    assert _geo(lib, 1, 8, 8, 1, 1)[1][0] == 0
    # grouped pointwise launches keep needing whole 128-pixel tiles per group
    assert _geo(lib, 3, 7, 7, 1, 3)[0] == -1
    assert _geo(lib, 384, 7, 7, 1, 3)[1][0] == 0


def test_box_tiled_shapes_refuse_other_modes_before_any_cuda_call(lib):
    buf = ctypes.create_string_buffer(1 << 12)
    p = ctypes.cast(buf, ctypes.c_void_p)
    for mode in (1, 2):  # STATS, STYLE
        rc = lib.irfd_conv_gemm(p, 2, 56, 56, 64, p, 64, 3, p, p, mode, p, p, p, p, p, p, p, 0, None)
        assert rc == -1 and b"box tiles" in lib.irfd_last_error(), (mode, lib.irfd_last_error())
    rc = lib.irfd_conv_gemm_grouped(p, 6, 28, 28, 64, p, 64, 3, p, 1, p, p, 3, 0, 0, None)
    assert rc == -1 and b"box tiles" in lib.irfd_last_error()
    ptrs = (ctypes.c_void_p * 3)(p.value, p.value, p.value)
    rc = lib.irfd_conv_gemm_bnbwd_grouped(p, 6, 14, 14, 64, p, 64, 3, p, p, p, p, ptrs, ptrs, p, 3, 3, 0, None)
    assert rc == -1 and b"box tiles" in lib.irfd_last_error()
    rc = lib.irfd_conv_gemm_bnbwd_res_grouped(p, 3, 7, 7, 64, p, 64, 3, p, p, p, p, p, p, p, 3, 3, 0, None)
    assert rc == -1 and b"box tiles" in lib.irfd_last_error()


def _torchvision_sizes(h, w):
    from torchvision.models import resnet50

    net = resnet50().to("meta").eval()
    x = torch.empty(1, 3, h, w, device="meta")
    out = []
    x = net.conv1(x)
    out.append(tuple(x.shape[2:]))
    x = net.maxpool(net.relu(net.bn1(x)))
    for layer in (net.layer1, net.layer2, net.layer3, net.layer4):
        x = layer(x)
        out.append(tuple(x.shape[2:]))
    return out


@pytest.mark.parametrize("h,w", [(224, 224), (256, 256), (320, 320), (384, 384), (250, 250), (300, 200), (33, 47),
                                 (32, 32), (63, 95), (129, 31), (1, 1), (2, 3), (577, 579), (200, 72)])
def test_stage_shapes_match_torchvision(h, w):
    from speak_hack_b200 import ops

    assert ops.resnet_stage_hw(h, w) == _torchvision_sizes(h, w)
