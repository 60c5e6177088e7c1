"""The checker of cucd_me_search (tests/me_search_oracle.c) against the semantics stated in include/cucudecide.h: xGetComponentBits,
the wrapping motion-vector cost, and an independent numpy statement of the integer search (a lexicographic argmin over (cost, raster
index) on the oracle's SAD surfaces) and of the two-stage refinement walk over the oracle's sub-pel tables."""
import ctypes as C

import numpy as np
import pytest

from _util import load_oracle
from me_search_util import (FRAC, HAD, HM_H, HM_Q, MC_SHAPES, mc_scene, np_bits, np_cost, np_search, np_walk, load_me_search_oracle, oracle_search,
                            search_desc, search_descs, walk_batch)


@pytest.fixture(scope="module")
def mso():
    return load_me_search_oracle()


@pytest.fixture(scope="module")
def oracle():
    return load_oracle()


def loop_bits(v):
    """xGetComponentBits as HM writes it"""
    t = (-v << 1) + 1 if v <= 0 else v << 1
    n = 1
    while t != 1:
        t >>= 1
        n += 2
    return n


def test_bits_match_the_loop_form(mso):
    vs = np.arange(-70000, 70001)
    got = np.array([mso.oracle_mv_bits(int(v)) for v in vs], np.int64)
    assert np.array_equal(got, np.array([loop_bits(int(v)) for v in vs], np.int64))
    assert np.array_equal(got, np_bits(vs))


def test_cost_wraps_32_bits(mso):
    rng = np.random.default_rng(5)
    for lam in (0xFFFFFFFF, 0x80000001, 0x12345678, 1 << 20, 888605):
        for _ in range(200):
            x, y = (int(v) for v in rng.integers(-9000, 9000, 2))
            px, py = (int(v) for v in rng.integers(-32768, 32768, 2))
            s = int(rng.integers(0, 3))
            bits = loop_bits(x * (1 << s) - px) + loop_bits(y * (1 << s) - py)
            want = ((lam * bits) & 0xFFFFFFFF) >> 16
            assert mso.oracle_mv_cost(lam, x, y, s, px, py) == want == int(np_cost(lam, x, y, s, px, py))
    assert ((0xFFFFFFFF * 40) >> 16) != mso.oracle_mv_cost(0xFFFFFFFF, 0, 0, 0, 1 << 9, 1 << 9)     # the product does wrap


@pytest.mark.parametrize("bd", [8, 10])
def test_checker_matches_numpy_statement(mso, oracle, bd):
    """the 22 PU shapes, +-64 / +-4 / 1x1 windows, windows clipped at picture corners, sub_shift 0 and 1, Hadamard and SAD, all lambdas"""
    sc = mc_scene(bd, seed=bd + 3)
    rng = np.random.default_rng(bd)
    descs = search_descs(sc, rng)
    assert len(descs) == len(MC_SHAPES) * 9
    assert any(d["right"] - d["left"] < 128 and d["right"] - d["left"] > 8 for d in descs)          # +-64 windows clipped at a corner
    assert {d["right"] - d["left"] for d in descs} >= {0, 8, 128} and {d["sub_shift"] for d in descs} == {0, 1}
    got = oracle_search(mso, sc, descs)
    want = np_search(oracle, sc, descs)
    for i, d in enumerate(descs):
        assert np.array_equal(got[i], want[i]), (d, got[i], want[i])


def test_checker_matches_numpy_statement_signed_keys(mso, oracle):
    sc = mc_scene(10, seed=9)
    rng = np.random.default_rng(9)
    descs = search_descs(sc, rng, shapes=MC_SHAPES[::3], radii=(4, 0))
    src = rng.integers(-1500, 2600, sum(d["w"] * d["h"] for d in descs)).astype(np.int16)
    assert np.array_equal(oracle_search(mso, sc, descs, src), np_search(oracle, sc, descs, src))


@pytest.mark.parametrize("bd", [8, 10])
def test_ties_on_constant_planes(mso, bd):
    """every candidate has the same SAD: lambda 0 keeps the window's top-left, lambda > 0 the fewest-bits MV first in raster order"""
    sc = mc_scene(bd, seed=1)
    v = 77 if bd == 8 else 300
    sc["org"] = np.full_like(sc["org"], v)
    sc["refs"] = {s: np.full_like(p, v + 5) for s, p in sc["refs"].items()}
    for w, h in [(16, 16), (8, 4), (64, 32)]:
        d = search_desc(sc, 64, 32, w, h, sc["slots"][0], 3, -2, 6, sub_shift=0, pred=(0, 0), lam=0, flags=0)
        r = oracle_search(mso, sc, [d])[0]
        assert (r[0], r[1]) == (d["left"], d["top"])
        for pred in [(0, 0), (13, -7), (-40, 22)]:
            d = search_desc(sc, 64, 32, w, h, sc["slots"][0], 3, -2, 6, sub_shift=0, pred=pred, lam=157084, flags=0)
            r = oracle_search(mso, sc, [d])[0]
            ys, xs = np.mgrid[d["top"]:d["bottom"] + 1, d["left"]:d["right"] + 1]
            bits = np_bits(4 * xs - pred[0]) + np_bits(4 * ys - pred[1])
            k = int(np.argmin(bits.ravel()))                  # the first of the fewest bits in raster order
            assert (r[0], r[1]) == (int(xs.ravel()[k]), int(ys.ravel()[k]))


def two_way_tie_table(a, b, base=1000, lo=10):
    """a 49-table whose two positions a and b are equal and lowest, everything else high"""
    T = np.full(49, base, np.uint32)
    T[a] = lo
    T[b] = lo
    return T


def test_walk_orders_on_two_way_ties(mso):
    """lambda 0: the walk keeps the first of two tied candidates in HM's order; H and Q differ at their entries 3..6"""
    d = dict(pred_x=0, pred_y=0, **{"lambda": 0})
    for i in range(1, 9):
        for j in range(i + 1, 9):
            hx, hy = HM_H[i]
            gx, gy = HM_H[j]
            T = two_way_tie_table((2 * hy + 3) * 7 + 2 * hx + 3, (2 * gy + 3) * 7 + 2 * gx + 3)
            qmv, fc = np.zeros(2, np.int32), np.zeros(1, np.uint32)
            mso.oracle_me_frac_walk(T.ctypes.data, 5, -3, 0, 0, 0, qmv.ctypes.data, fc.ctypes.data)
            assert (qmv[0], qmv[1]) == (20 + 2 * hx, -12 + 2 * hy), (i, j)       # the half stage keeps H_i; the quarter stage stays
            assert tuple(qmv) + (fc[0],) == np_walk(T, 5, -3, d)
    for i in range(1, 9):
        for j in range(i + 1, 9):
            qx, qy = HM_Q[i]
            rx, ry = HM_Q[j]
            T = np.full(49, 1000, np.uint32)
            T[3 * 7 + 3] = 500                                                  # the half stage stays at (0, 0)
            T[(qy + 3) * 7 + qx + 3] = 10
            T[(ry + 3) * 7 + rx + 3] = 10
            qmv, fc = np.zeros(2, np.int32), np.zeros(1, np.uint32)
            mso.oracle_me_frac_walk(T.ctypes.data, 0, 0, 0, 0, 0, qmv.ctypes.data, fc.ctypes.data)
            assert (qmv[0], qmv[1], fc[0]) == (qx, qy, 10), (i, j)
            assert tuple(qmv) + (fc[0],) == np_walk(T, 0, 0, d)
    # (-1, 0) comes before (-1, -1) in H but after it in Q
    assert HM_H.index((-1, 0)) < HM_H.index((-1, -1)) and HM_Q.index((-1, 0)) > HM_Q.index((-1, -1))


def test_walk_adds_the_scaled_costs(mso):
    rng = np.random.default_rng(11)
    for _ in range(400):
        T = rng.integers(0, 1 << 14, 49).astype(np.uint32)
        mvx, mvy = (int(v) for v in rng.integers(-64, 65, 2))
        px, py = (int(v) for v in rng.integers(-300, 300, 2))
        lam = int(rng.choice([0, 157084, 888605, 0xFFFFFFFF, int(rng.integers(0, 1 << 32))]))
        qmv, fc = np.zeros(2, np.int32), np.zeros(1, np.uint32)
        mso.oracle_me_frac_walk(T.ctypes.data, mvx, mvy, px, py, lam, qmv.ctypes.data, fc.ctypes.data)
        assert (int(qmv[0]), int(qmv[1]), int(fc[0])) == np_walk(T, mvx, mvy, dict(pred_x=px, pred_y=py, **{"lambda": lam}))


def test_batched_walk_of_the_gpu_tests(mso):
    """walk_batch (the surface route of test_gpu_me_search.py and bench_rows.py) equals the checker's walk"""
    rng = np.random.default_rng(12)
    T = rng.integers(0, 1 << 12, (500, 49)).astype(np.uint32)
    T[::7, 24] = T[::7, 17]                                                              # ties
    mv, pred = rng.integers(-64, 65, (500, 2)), rng.integers(-32768, 32768, (500, 2))
    for lam in (0, 888605, 0xFFFFFFFF):
        qmv, fc = walk_batch(T, mv, pred, lam)
        for i in range(0, 500, 3):
            q, f = np.zeros(2, np.int32), np.zeros(1, np.uint32)
            mso.oracle_me_frac_walk(T[i].ctypes.data, int(mv[i, 0]), int(mv[i, 1]), int(pred[i, 0]), int(pred[i, 1]), lam, q.ctypes.data, f.ctypes.data)
            assert (int(qmv[i, 0]), int(qmv[i, 1]), int(fc[i])) == (int(q[0]), int(q[1]), int(f[0]))


def test_frac_flag_names():
    assert (FRAC, HAD) == (1, 2) and C.sizeof(C.c_int) == 4
