"""CPU: the spectral-norm entry points are bound from the header, and reject bad arguments before any CUDA call."""
import ctypes
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from speak_hack_b200 import _lib, build

    if not os.path.exists(_lib.LIB_PATH):
        build.build(verbose=False)
    return _lib.load()


def _d_shapes():
    """[rows, cols] of the 16 spectrally normalised matrices of the 256^2 StyleDiscriminator."""
    from speak_hack_b200.discriminator import StyleDiscriminator

    d = StyleDiscriminator()
    ws = [m.weight_orig for m in d._sn_modules()]
    return [(w.shape[0], w.numel() // w.shape[0]) for w in ws]


def _arrays(shapes):
    n = len(shapes)
    return (ctypes.c_int * n)(*[r for r, _ in shapes]), (ctypes.c_int * n)(*[c for _, c in shapes])


def test_header_binding():
    from ctypes import c_float, c_int, c_longlong, c_void_p

    from speak_hack_b200 import _lib

    sig = _lib.SIGNATURES
    assert sig["irfd_spectral_norm_workspace_bytes"] == (c_longlong, [c_void_p, c_void_p, c_int])
    assert sig["irfd_spectral_norm_fwd"] == (c_int, [c_void_p] * 9 + [c_int, c_int, c_float, c_void_p, c_longlong,
                                                                     c_void_p])
    assert sig["irfd_spectral_norm_bwd"] == (c_int, [c_void_p] * 8 + [c_int, c_void_p, c_longlong, c_void_p])


def test_discriminator_layer_table():
    shapes = _d_shapes()
    assert len(shapes) == 16
    assert shapes[0] == (64, 3) and shapes[-3] == (512, 4608) and shapes[-2] == (512, 512) and shapes[-1] == (1, 512)
    assert sum(r * c for r, c in shapes) == 19_100_352   # 76.4 MB of fp32 weights read twice per D call


def test_workspace_bytes(lib):
    shapes = _d_shapes()
    rows, cols = _arrays(shapes)
    fwd = sum(c + (c + 31) // 32 + r + (r + 7) // 8 for r, c in shapes)
    bwd = sum((r * c + 8191) // 8192 for r, c in shapes)
    assert lib.irfd_spectral_norm_workspace_bytes(rows, cols, len(shapes)) == 4 * max(fwd, bwd)
    assert lib.irfd_spectral_norm_workspace_bytes(rows, cols, 0) < 0


def test_invalid_arguments_return_error_codes_without_a_gpu(lib):
    shapes = [(64, 576), (1, 512)]
    rows, cols = _arrays(shapes)
    buf = ctypes.create_string_buffer(64)
    p = ctypes.cast(buf, ctypes.c_void_p)
    ptrs = (ctypes.c_void_p * 2)(p, p)
    ws_bytes = lib.irfd_spectral_norm_workspace_bytes(rows, cols, 2)
    fwd, bwd = lib.irfd_spectral_norm_fwd, lib.irfd_spectral_norm_bwd

    def err(rc, text):
        return rc == -1 and text in lib.irfd_last_error()

    assert err(fwd(ptrs, ptrs, ptrs, ptrs, None, None, None, rows, cols, 2, 1, 1e-12, p, ws_bytes, None),
               b"null pointer")
    assert err(fwd(ptrs, ptrs, ptrs, ptrs, None, None, p, rows, cols, 0, 1, 1e-12, p, ws_bytes, None), b"layers")
    assert err(fwd(ptrs, ptrs, ptrs, ptrs, None, None, p, rows, cols, 33, 1, 1e-12, p, ws_bytes, None), b"layers")
    assert err(fwd(ptrs, ptrs, ptrs, ptrs, None, None, p, rows, cols, 2, 1, 0.0, p, ws_bytes, None), b"eps")
    assert err(fwd(ptrs, ptrs, ptrs, ptrs, None, None, p, rows, cols, 2, 1, 1e-12, p, ws_bytes - 4, None),
               b"workspace too small")
    assert err(fwd(ptrs, ptrs, ptrs, ptrs, None, None, p, None, cols, 2, 1, 1e-12, p, ws_bytes, None), b"rows/cols")
    holes = (ctypes.c_void_p * 2)(p, None)
    assert err(fwd(ptrs, holes, ptrs, ptrs, None, None, p, rows, cols, 2, 1, 1e-12, p, ws_bytes, None), b"layer 1")
    empty_rows, _ = _arrays([(0, 576), (1, 512)])
    assert err(fwd(ptrs, ptrs, ptrs, ptrs, None, None, p, empty_rows, cols, 2, 1, 1e-12, p, ws_bytes, None), b"empty")
    big_rows, big_cols = _arrays([(1 << 16, 1 << 16), (1, 512)])
    assert err(fwd(ptrs, ptrs, ptrs, ptrs, None, None, p, big_rows, big_cols, 2, 1, 1e-12, p, ws_bytes, None),
               b"2^31")
    assert err(bwd(ptrs, ptrs, p, p, None, ptrs, rows, cols, 2, p, ws_bytes, None), b"null pointer")
    assert err(bwd(ptrs, ptrs, p, p, p, ptrs, rows, cols, 2, p, 4, None), b"workspace too small")
    assert err(bwd(ptrs, holes, p, p, p, ptrs, rows, cols, 2, p, ws_bytes, None), b"layer 1")


def test_native_spectral_norm_context_is_scoped():
    """Outside D.native_spectral_norm() the torch hooks run; the context restores the previous setting."""
    from speak_hack_b200.discriminator import StyleDiscriminator

    d = StyleDiscriminator()
    assert not d.__dict__.get("_native_sn", False)
    with d.native_spectral_norm():
        assert d._native_sn
        with d.native_spectral_norm():
            assert d._native_sn
        assert d._native_sn
    assert not d._native_sn
    with pytest.raises(RuntimeError):
        with d.native_spectral_norm():
            raise RuntimeError("boom")
    assert not d._native_sn
