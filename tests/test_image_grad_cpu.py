"""CPU: the image-gradient entry points of the encoders' stem (irfd_col2im_stem, pack mode FLAT_T) validate their
arguments before any CUDA call, and the stem's dcol GEMM gets whole 128-pixel tiles per encoder on the linear geometry
at every shape a differentiated encoder pass accepts."""
import ctypes
import os

import pytest


@pytest.fixture(scope="module")
def lib():
    from speak_hack_b200 import _lib, build

    if not os.path.exists(_lib.LIB_PATH):
        build.build(verbose=False)
    return _lib.load()


def _buf(nbytes=4096, offset=0):
    buf = ctypes.create_string_buffer(nbytes + 32)
    base = (ctypes.addressof(buf) + 15) // 16 * 16   # 16-byte aligned
    return buf, ctypes.c_void_p(base + offset)


def test_header_declares_col2im_stem():
    from speak_hack_b200 import _lib

    res, args = _lib.SIGNATURES["irfd_col2im_stem"]
    assert res is ctypes.c_int and len(args) == 8


@pytest.mark.parametrize("case, msg", [
    (dict(dcol=None), b"null or unaligned"),
    (dict(offset=8), b"null or unaligned"),
    (dict(dx=None), b"null or unaligned"),
    (dict(nsets=0), b"column sets"),
    (dict(nsets=5), b"column sets"),
    (dict(kpad=144), b"kpad"),
    (dict(kpad=196), b"kpad"),
    (dict(n=0), b"bad shape"),
    (dict(h=0), b"bad shape"),
    (dict(w=-4), b"bad shape"),
    (dict(n=70000), b"bad shape"),
])
def test_col2im_stem_rejects_bad_arguments(lib, case, msg):
    keep, p = _buf(offset=case.get("offset", 0))
    a = dict(dcol=p, dx=p, n=1, h=64, w=64, kpad=192, nsets=3)
    a.update({k: v for k, v in case.items() if k != "offset"})
    rc = lib.irfd_col2im_stem(a["dcol"], a["dx"], a["n"], a["h"], a["w"], a["kpad"], a["nsets"], None)
    assert rc == -1 and msg in lib.irfd_last_error(), lib.irfd_last_error()


def test_pack_flat_t_rejects_bad_arguments(lib):
    keep, p = _buf()
    assert lib.irfd_pack_conv_weight(p, p, 64, 3, 49, 4, 144, None) == -1   # kpad < 147 rows
    assert b"FLAT_T" in lib.irfd_last_error()
    assert lib.irfd_pack_conv_weight(p, p, 64, 3, 49, 5, 192, None) == -1   # no mode 5
    assert lib.irfd_pack_conv_weight(None, p, 64, 3, 49, 4, 192, None) == -1


@pytest.mark.parametrize("b", [1, 2, 32])
@pytest.mark.parametrize("e", [1, 3])
def test_stem_dcol_gemm_is_linear_at_every_trainable_shape(lib, b, e):
    """P = n * H/2 * W/2 pixels per encoder, n = B (a lone encoder) or 2B (the paired lockstep pass): the dcol GEMM
    [E*P, 64] x [64, 192] gives each of the E weight groups whole 128-pixel tiles (boxed = 0)."""
    from speak_hack_b200 import ops
    from speak_hack_b200.encoder import MAX_STEM_W, trainable_shape

    checked = 0
    for n in (b, 2 * b):
        for h in range(32, 1025, 32):
            for w in range(32, MAX_STEM_W + 1, 32):
                if not trainable_shape(n, h, w):
                    continue
                p = n * (h // 2) * (w // 2)
                g = ops.conv_geometry(1, 1, e * p, 1, e)
                assert g is not None and g[0] == 0 and p % 256 == 0, (n, h, w, e, g)
                checked += 1
    assert checked >= 10
