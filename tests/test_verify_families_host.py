"""CPU: host side of the image-generator verification sweep -- the clamp(0, 1) crop entry point's argument checks, the
post-processing mode selection and the rank slicing."""
import ctypes
import os

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_clamp01_crop_is_declared_and_exported():
    from ipr_gan_b200 import _lib
    header = open(os.path.join(ROOT, "include", "ipr_b200.h")).read()
    assert "int ipr_crop_clamp01_f32(" in header
    assert hasattr(ctypes.CDLL(_lib.LIB_PATH), "ipr_crop_clamp01_f32")
    assert _lib.SIGNATURES["ipr_crop_clamp01_f32"] == _lib.SIGNATURES["ipr_crop_postproc_f32"]


def test_clamp01_crop_argument_checks():
    """The documented error codes come from the host before any launch (the pointers are never dereferenced)."""
    from ipr_gan_b200 import _lib
    lib = _lib.lib()
    f = lib.ipr_crop_clamp01_f32
    p = ctypes.c_void_p(256)
    assert f(None, p, p, 2, 3, 96, 96, 48, 0, 0, None) == -1
    assert f(p, None, p, 2, 3, 96, 96, 48, 0, 0, None) == -1
    assert f(p, p, None, 2, 3, 96, 96, 48, 0, 0, None) == -1
    assert f(p, p, p, 0, 3, 96, 96, 48, 0, 0, None) == -2             # empty batch
    assert f(p, p, p, 2, 0, 96, 96, 48, 0, 0, None) == -2
    assert f(p, p, p, 2, 3, 96, 96, 0, 0, 0, None) == -2              # empty window
    assert f(p, p, p, 2, 3, 96, 96, 48, 49, 0, None) == -2            # window leaves the image
    assert f(p, p, p, 2, 3, 96, 96, 48, 0, 49, None) == -2
    assert f(p, p, p, 2, 3, 96, 96, 48, -1, 0, None) == -2
    # same checks, same codes as the [-1, 1] variant
    for args in ((None, p, p, 2, 3, 96, 96, 48, 0, 0, None), (p, p, p, 2, 3, 96, 96, 48, 49, 0, None)):
        assert f(*args) == lib.ipr_crop_postproc_f32(*args)


def test_postproc_mode_and_refusals():
    from ipr_gan_b200 import ops
    assert ops.postproc_mode(True) == "signed" and ops.postproc_mode(False) == "unit"
    with pytest.raises(ops.IprError):
        ops.crop_patch(torch.zeros(1, 3, 8, 8), torch.zeros(1, 1, 4, 4), "tl", 4, postproc="clamp")
    with pytest.raises(ops.IprError):                                 # no CPU fallback for the new mode either
        ops.crop_patch(torch.zeros(1, 3, 8, 8), torch.zeros(1, 1, 4, 4), "tl", 4, postproc="unit")


@pytest.mark.parametrize("world", [1, 2, 3, 4, 5, 7, 8])
def test_rank_slices_cover_every_input_once(world):
    from ipr_gan_b200 import verify
    for n in list(range(0, 40)) + [97, 1000, 1003]:
        seen = []
        prev_hi = 0
        for r in range(world):
            lo, hi = verify.rank_slice(n, r, world)
            assert 0 <= lo <= hi <= n and lo == prev_hi           # contiguous, in rank order
            seen.extend(range(lo, hi))
            prev_hi = hi
        assert seen == list(range(n)), (n, world)


def test_image_sweep_rejects_bad_inputs():
    from ipr_gan_b200 import verify
    for bad in (torch.zeros(3, 24, 24), torch.zeros(0, 3, 24, 24), torch.zeros(2, 3, 24, 24, dtype=torch.float64)):
        with pytest.raises(ValueError):
            verify.image_verification_sweep(None, None, None, bad)
    with pytest.raises(ValueError):
        verify.image_verification_sweep(None, None, None, torch.zeros(2, 3, 24, 24), batch=0)
