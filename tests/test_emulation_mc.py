"""CPU replay of me_mc_kernel (tests/emul/mc_emul.cpp emul_mc_cost: the host plan of cucd_me_mc_cost and the kernel's __host__
__device__ phases for every thread id of every CTA) against the checker tests/mc_oracle.c, distortion and samples: the 22 PU shapes,
uni L0, uni L1, bi and bi with identical motion, random and extreme fractions, SAD and Hadamard, 8 and 10 bits, supports at the
edge of the margin."""
import numpy as np
import pytest

from mc_util import MC_SHAPES, emul_mc, load_mc_emul, load_mc_oracle, mc_candidates, mc_scene, oracle_mc


@pytest.fixture(scope="module")
def mco():
    return load_mc_oracle()


@pytest.fixture(scope="module")
def emul():
    return load_mc_emul()


def check(emul, mco, sc, descs):
    want_d, want_p = oracle_mc(mco, sc, descs)
    got_d, got_p, n_cta = emul_mc(emul, sc, descs)
    assert n_cta > 0
    for i, d in enumerate(descs):
        assert np.array_equal(got_p[i], want_p[i]), d
        assert got_d[i] == want_d[i], d
    return n_cta


@pytest.mark.parametrize("bd", [8, 10])
def test_emul_mc_matches_oracle_in_one_mixed_batch(emul, mco, bd):
    sc = mc_scene(bd, seed=bd)
    rng = np.random.default_rng(bd + 1)
    descs = mc_candidates(sc, rng) + mc_candidates(sc, rng)
    rng.shuffle(descs)
    n_cta = check(emul, mco, sc, descs)
    assert n_cta < len(descs)                                # small candidates share CTAs


@pytest.mark.parametrize("bd", [8, 10])
def test_emul_mc_packs_many_small_candidates(emul, mco, bd):
    """one class per shape with more candidates than a CTA holds: the last CTA of a class is partial"""
    sc = mc_scene(bd, seed=20 + bd)
    rng = np.random.default_rng(bd + 2)
    descs = []
    for _ in range(24):
        descs += mc_candidates(sc, rng, shapes=[(4, 4), (8, 8), (8, 4), (16, 16)], modes=("l0", "bi"), hads=(1,), edge=False)
    check(emul, mco, sc, descs)


@pytest.mark.parametrize("bd", [8, 10])
def test_emul_mc_every_fraction_pair(emul, mco, bd):
    sc = mc_scene(bd, seed=30 + bd)
    descs = []
    for f0 in range(16):
        for f1 in range(16):
            descs.append(dict(x=64, y=32, w=8, h=8, ref_idx=(0, 3), mvx=(-40 + (f0 & 3), 12 + (f1 & 3)), mvy=(20 + (f0 >> 2), -8 + (f1 >> 2)), use_hadamard=f0 & 1))
        descs.append(dict(x=40, y=8, w=12, h=16, ref_idx=(-1, 3), mvx=(0, 4 * 9 + (f0 & 3)), mvy=(0, -4 * 7 + (f0 >> 2)), use_hadamard=0))
    check(emul, mco, sc, descs)


def test_emul_mc_shapes_cover_the_subpel_test():
    assert len(MC_SHAPES) == 22 and len(set(MC_SHAPES)) == 22
