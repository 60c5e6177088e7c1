"""CPU replay of me_mc_chroma_kernel (tests/emul/mc_chroma_emul.cpp emul_mc_chroma: the host plan of cucd_me_mc_chroma and the kernel's
__host__ __device__ phases for every thread id of every CTA) against the checker tests/mc_chroma_oracle.c, SSE and samples: the
chroma blocks of the 22 PU shapes, uni L0, uni L1, bi and bi with identical motion, all 64 fraction pairs, supports at the corners
of the chroma margin, classes fuller than one CTA, 8 and 10 bits."""
import numpy as np
import pytest

from mc_chroma_util import emul_mc_chroma, load_mc_chroma_emul, load_mc_chroma_oracle, mcc_candidates, mcc_scene, oracle_mc_chroma
from mc_util import MC_SHAPES


@pytest.fixture(scope="module")
def mco():
    return load_mc_chroma_oracle()


@pytest.fixture(scope="module")
def emul():
    return load_mc_chroma_emul()


def check(emul, mco, sc, descs):
    want_s, want_p = oracle_mc_chroma(mco, sc, descs)
    got_s, got_p, n_cta = emul_mc_chroma(emul, sc, descs)
    assert n_cta > 0
    for i, d in enumerate(descs):
        for c in range(2):
            assert np.array_equal(got_p[i][c], want_p[i][c]), (d, c)
        assert np.array_equal(got_s[i], want_s[i]), d
    return n_cta


@pytest.mark.parametrize("bd", [8, 10])
def test_emul_mc_chroma_matches_oracle_in_one_mixed_batch(emul, mco, bd):
    sc = mcc_scene(bd, seed=bd)
    rng = np.random.default_rng(bd + 1)
    descs = mcc_candidates(sc, rng) + mcc_candidates(sc, rng) + mcc_candidates(sc, rng)
    rng.shuffle(descs)
    n_cta = check(emul, mco, sc, descs)
    assert n_cta < len(descs)                                # small candidates share CTAs


@pytest.mark.parametrize("bd", [8, 10])
def test_emul_mc_chroma_packs_many_small_candidates(emul, mco, bd):
    """more candidates of one class than a CTA holds (64 of a 2x4 chroma block): the last CTA of a class is partial"""
    sc = mcc_scene(bd, seed=20 + bd)
    rng = np.random.default_rng(bd + 2)
    descs = []
    for _ in range(70):
        descs += mcc_candidates(sc, rng, shapes=[(4, 8), (8, 8), (16, 16)], modes=("l0", "bi"), edge=False)
    n_cta = check(emul, mco, sc, descs)
    assert n_cta > 6                                         # six classes; 70 uni 2x4 blocks take two CTAs


@pytest.mark.parametrize("bd", [8, 10])
def test_emul_mc_chroma_every_fraction_pair(emul, mco, bd):
    sc = mcc_scene(bd, seed=30 + bd)
    descs = []
    for f0 in range(64):
        for f1 in range(0, 64, 9):
            descs.append(dict(x=64, y=32, w=8, h=8, ref_idx=(0, 3), mvx=(-40 + (f0 & 7), 16 + (f1 & 7)), mvy=(24 + (f0 >> 3), -8 + (f1 >> 3)), use_hadamard=0))
        descs.append(dict(x=40, y=8, w=12, h=16, ref_idx=(-1, 3), mvx=(0, 8 * 9 + (f0 & 7)), mvy=(0, -8 * 7 + (f0 >> 3)), use_hadamard=1))
        descs.append(dict(x=100, y=60, w=4, h=8, ref_idx=(3, 0), mvx=(-8 * 3 + (f0 >> 3), 5), mvy=(8 * 2 + (f0 & 7), 67), use_hadamard=0))
    check(emul, mco, sc, descs)


def test_mc_shapes_give_every_chroma_shape():
    """the 22 luma PU shapes give 2- and 6-wide (and high) chroma blocks as well as 32 x 32"""
    chroma = {(w // 2, h // 2) for w, h in MC_SHAPES}
    assert len(chroma) == 22 and {(2, 4), (4, 2), (2, 8), (6, 8), (8, 6), (32, 32), (24, 32), (32, 8)} <= chroma
