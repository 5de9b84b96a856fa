"""CPU: the one-launch 3-channel layer's entry point -- declared and exported, argument checks answered on the host
before any launch, and unsupported shapes handed back to the caller, which then keeps the tap GEMM + col2im3 path."""
import ctypes
import os

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
IPR_E_NULL, IPR_E_SHAPE, IPR_E_UNSUPPORTED, IPR_E_ALIGN = -1, -2, -3, -4
P = ctypes.c_void_p(0x10000)            # never dereferenced: every call below returns before a launch


def _lib():
    from ipr_gan_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        from ipr_gan_b200 import build
        build.build()
    return _lib.lib()


def test_symbol_declared_and_exported():
    from ipr_gan_b200 import _lib
    header = open(os.path.join(ROOT, "include", "ipr_b200.h")).read()
    assert "int ipr_tapfold3_f32(" in header
    assert "ipr_tapfold3_f32" in _lib.SIGNATURES
    assert hasattr(_lib_handle(), "ipr_tapfold3_f32")


def _lib_handle():
    from ipr_gan_b200 import _lib as m
    _lib()
    return ctypes.CDLL(m.LIB_PATH)


def test_null_pointers():
    L = _lib()
    assert L.ipr_tapfold3_f32(None, P, None, P, 4, 32, 32, 1, None) == IPR_E_NULL
    assert L.ipr_tapfold3_f32(P, None, None, P, 4, 32, 32, 1, None) == IPR_E_NULL
    assert L.ipr_tapfold3_f32(P, P, None, None, 4, 32, 32, 1, None) == IPR_E_NULL


@pytest.mark.parametrize("batch,h,w", [(0, 32, 32), (-1, 32, 32), (4, 0, 32), (4, 32, 0), (1 << 31, 32, 32)])
def test_bad_shapes(batch, h, w):
    assert _lib().ipr_tapfold3_f32(P, P, None, P, batch, h, w, 1, None) == IPR_E_SHAPE


def test_alignment():
    L = _lib()
    odd = ctypes.c_void_p(0x10008)
    assert L.ipr_tapfold3_f32(odd, P, None, P, 4, 32, 32, 1, None) == IPR_E_ALIGN
    assert L.ipr_tapfold3_f32(P, odd, None, P, 4, 32, 32, 1, None) == IPR_E_ALIGN
    assert L.ipr_tapfold3_f32(P, P, None, ctypes.c_void_p(0x10002), 4, 32, 32, 1, None) == IPR_E_ALIGN


@pytest.mark.parametrize("h,w", [(64, 64), (20, 20), (4, 96), (32, 256), (1024, 1), (12, 24)])
def test_unsupported_shapes(h, w):
    # more than 1024 pixels, pixels not a multiple of 128, a width that does not divide 128, or a staged image that
    # does not fit in shared memory
    assert _lib().ipr_tapfold3_f32(P, P, None, P, 4, h, w, 1, None) == IPR_E_UNSUPPORTED


def test_engine_falls_back_on_unsupported_shape(monkeypatch):
    """tapfold3 returns None (the caller runs the two-launch path) for shapes the kernel does not cover, and for every
    shape when IPR_NO_TAPFOLD=1."""
    from ipr_gan_b200 import engine
    _lib()
    monkeypatch.setattr(engine, "_st", lambda: None)
    pack = torch.zeros(1, 32, 64, dtype=torch.bfloat16)
    a = torch.zeros(2, 64, 64, 64, dtype=torch.bfloat16)
    assert engine.tapfold3(a, pack, True) is None
    monkeypatch.setenv("IPR_NO_TAPFOLD", "1")
    assert engine.tapfold3(torch.zeros(2, 32, 32, 64, dtype=torch.bfloat16), pack, True) is None
