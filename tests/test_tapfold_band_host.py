"""CPU: the banded one-launch 3-channel layer's entry point (ipr_tapfold3_band_f32, for the 64 x 64 networks) --
declared and exported, argument checks answered on the host before any launch, unsupported shapes handed back."""
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
    from ipr_gan_b200 import _lib as m
    header = open(os.path.join(ROOT, "include", "ipr_b200.h")).read()
    assert "int ipr_tapfold3_band_f32(" in header
    assert m.SIGNATURES["ipr_tapfold3_band_f32"] == m.SIGNATURES["ipr_tapfold3_f32"]
    _lib()
    assert hasattr(ctypes.CDLL(m.LIB_PATH), "ipr_tapfold3_band_f32")


def test_null_pointers():
    L = _lib()
    assert L.ipr_tapfold3_band_f32(None, P, None, P, 4, 64, 64, 1, None) == IPR_E_NULL
    assert L.ipr_tapfold3_band_f32(P, None, None, P, 4, 64, 64, 1, None) == IPR_E_NULL
    assert L.ipr_tapfold3_band_f32(P, P, None, None, 4, 64, 64, 1, None) == IPR_E_NULL


@pytest.mark.parametrize("batch,h,w", [(0, 64, 64), (-1, 64, 64), (4, 0, 64), (4, 64, 0), (1 << 31, 64, 64),
                                       (1 << 30, 64, 64)])
def test_bad_shapes(batch, h, w):
    # the last case: 6 bands an image, more work items than an int counts
    assert _lib().ipr_tapfold3_band_f32(P, P, None, P, batch, h, w, 1, None) == IPR_E_SHAPE


def test_alignment():
    L = _lib()
    odd = ctypes.c_void_p(0x10008)
    assert L.ipr_tapfold3_band_f32(odd, P, None, P, 4, 64, 64, 1, None) == IPR_E_ALIGN
    assert L.ipr_tapfold3_band_f32(P, odd, None, P, 4, 64, 64, 1, None) == IPR_E_ALIGN
    assert L.ipr_tapfold3_band_f32(P, P, None, ctypes.c_void_p(0x10002), 4, 64, 64, 1, None) == IPR_E_ALIGN


@pytest.mark.parametrize("h,w", [
    (32, 96), (64, 48), (12, 24),          # widths that do not divide 128
    (20, 20), (3, 32), (1, 64),            # pixel counts that are not a multiple of 128
    (32, 256), (64, 512),                  # wider than one 128-row sub-tile
])
def test_unsupported_shapes(h, w):
    assert _lib().ipr_tapfold3_band_f32(P, P, None, P, 4, h, w, 1, None) == IPR_E_UNSUPPORTED


def test_whole_image_entry_still_declines_64x64():
    """The banded entry point takes 64 x 64; the whole-image one keeps handing it back."""
    assert _lib().ipr_tapfold3_f32(P, P, None, P, 4, 64, 64, 1, None) == IPR_E_UNSUPPORTED


def test_engine_band_fold_off_under_switch(monkeypatch):
    """IPR_NO_TAPFOLD=1 selects the tap GEMM + col2im3 path for every shape: tapfold3_band returns None before it
    calls the library (CPU tensors, no stream)."""
    from ipr_gan_b200 import engine
    _lib()
    monkeypatch.setattr(engine, "_st", lambda: None)
    monkeypatch.setenv("IPR_NO_TAPFOLD", "1")
    pack = torch.zeros(1, 32, 64, dtype=torch.bfloat16)
    for h in (64, 32):
        a = torch.zeros(2, h, h, 64, dtype=torch.bfloat16)
        assert engine.tapfold3_band(a, pack, True) is None
        assert engine._fold3(a, pack, False, sigma=None) is None
