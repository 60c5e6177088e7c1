"""CPU replay of me_tz_kernel (tests/emul/me_tz_emul.cpp: the me_tz_* phases of csrc/me_core.cuh with the kernel's lane mapping and its
two xor butterflies) against the checker tests/me_tz_oracle.c: the points of every stage with their values, in HM's order, and the
final integer result, at 8, 9 and 10 bit, with extreme sample values."""
import numpy as np
import pytest

from me_tz_util import FRAC, HAD, MC_SHAPES, TZ2N, emul_tz, lambda_cost, load_me_tz_emul, load_me_tz_oracle, mc_scene, oracle_tz, tz_desc


@pytest.fixture(scope="module")
def tz():
    return load_me_tz_oracle()


@pytest.fixture(scope="module")
def emul():
    return load_me_tz_emul()


def check(tz, emul, sc, descs):
    lanes, extra = set(), 0
    for d in descs:
        want, wtrace, nprobe = oracle_tz(tz, sc, dict(d, flags=d["flags"] & ~(FRAC | HAD)), trace_cap=200000)
        got, gtrace, ev, g = emul_tz(emul, sc, d)
        assert np.array_equal(got[:3], want[:3]), d
        assert np.array_equal(gtrace, wtrace), d                       # every stage's points, values and order
        assert ev >= nprobe
        extra += ev - nprobe
        lanes.add(g)
    return lanes, extra


def descs_for(sc, rng, shapes=MC_SHAPES):
    out = []
    for w, h in shapes:
        for R, fl in ((64, FRAC | HAD), (64, TZ2N), (8, FRAC | TZ2N), (1, 0)):
            x = int(rng.integers(0, (sc["W"] - w) // 4 + 1)) * 4
            y = int(rng.integers(0, (sc["H"] - h) // 4 + 1)) * 4
            if len(out) % 5 == 4:
                x, y = [(0, 0), (sc["W"] - w, 0), (0, sc["H"] - h), (sc["W"] - w, sc["H"] - h)][len(out) // 5 % 4]
            pred = tuple(int(v) for v in rng.integers(-400, 401, 2)) if rng.random() < 0.3 else tuple(int(v) for v in rng.integers(-30, 31, 2))
            out.append(tz_desc(sc, x, y, w, h, sc["slots"][len(out) % 2], pred, R, sub_shift=int(rng.integers(0, 2)),
                               lam=int([0, lambda_cost(22), lambda_cost(37), 0xFFFFFFFF][len(out) % 4]), flags=fl,
                               mv2n=tuple(int(v) for v in rng.integers(-20, 21, 2))))
    return out


@pytest.mark.parametrize("bd", [8, 9, 10])
def test_replay_matches_checker_on_pictures(tz, emul, bd):
    sc = mc_scene(bd, seed=bd + 90)
    lanes, extra = check(tz, emul, sc, descs_for(sc, np.random.default_rng(bd + 90)))
    assert lanes == {1, 2, 4, 8, 16, 32}                               # every lane mapping took part
    assert extra > 0                                                   # chunks past the first search's stop were evaluated and dropped


@pytest.mark.parametrize("bd", [8, 9, 10])
def test_replay_matches_checker_on_extreme_samples(tz, emul, bd):
    """source at 2^bd - 1, references of 0 and 2^bd - 1: the largest SADs and sums the kernel forms"""
    sc = mc_scene(bd, seed=bd + 95)
    hi = (1 << bd) - 1
    rng = np.random.default_rng(bd + 95)
    sc = dict(sc, org=np.full_like(sc["org"], hi), refs={s: np.where(rng.random(p.shape) < 0.9, 0, hi).astype(np.int16) for s, p in sc["refs"].items()})
    check(tz, emul, sc, descs_for(sc, rng, shapes=MC_SHAPES[:8]))
