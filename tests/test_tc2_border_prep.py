"""The border pre-pass of the 8-bit tensor-core RMD kernel (rmd_border_prep_kernel), replayed on the CPU (tests/emul/rmd_tc2_prep_emul.cpp):
the store and DC sums its images give an RMD CTA after the bulk copies are the ones the CTA's own prologue built from the reconstruction
before the pre-pass existed, at every depth, for partial CTUs at the picture's right and bottom edges, with strong smoothing on and off."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from _util import P, i16p, pseudo_recon, textured_plane

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def prep(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("prep_emul") / "librmd_tc2_prep_emul.so")
    csrc = os.path.join(os.path.dirname(HERE), "fast-cu-decision-hevc_b200", "csrc")
    subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-I" + csrc, "-o", so,
                    os.path.join(HERE, "emul", "rmd_tc2_prep_emul.cpp")], check=True, capture_output=True)
    lib = C.CDLL(so)
    lib.emul_tc2_prep_check.restype = C.c_longlong
    return lib


def _rec(W, H, seed):
    rec = pseudo_recon(textured_plane(W, H, 8, seed=seed), 8)
    rec[:, : W // 2] = (np.arange(H)[:, None] // 3 + np.arange(W // 2)[None, :] // 5 + 40).astype(np.int16)   # flat: strong smoothing
    return np.ascontiguousarray(rec)


@pytest.mark.parametrize("strong", [0, 1])
@pytest.mark.parametrize("W,H,seed", [(200, 136, 5), (328, 72, 9), (64, 64, 1)])
def test_prepass_images_match_in_kernel_prologue(prep, strong, W, H, seed):
    rec = _rec(W, H, seed)
    compared = C.c_longlong(0)
    bad = prep.emul_tc2_prep_check(strong, P(rec, i16p), W, W, H, C.byref(compared))
    assert compared.value > 0
    assert bad == 0


def test_prepass_strong_smoothing_changes_images(prep):
    """the flat half of the picture takes the strong (bilinear) 32x32 filter: the images with and without it differ"""
    W, H = 200, 136
    rec = _rec(W, H, 5)
    n = prep.emul_tc2_prep_ctu_bytes() * ((W + 63) // 64) * ((H + 63) // 64)
    img = [np.zeros(n, np.uint8) for _ in range(2)]
    for strong in (0, 1):
        assert prep.emul_tc2_prep_images(strong, P(rec, i16p), W, W, H, img[strong].ctypes.data_as(C.POINTER(C.c_uint8))) == 0
    assert not np.array_equal(img[0], img[1])
