"""CPU replay of the motion-search phases of cucd_me_search (tests/emul/me_search_emul.cpp) against the checker tests/me_search_oracle.c:
the Argmin epilogue of the SAD kernels with its warp key reduction (dy-lane tiles with their own SAD arithmetic, dx-lane tiles on the
oracle's SADs), the prep phase and the walk phase, for every thread id."""
import ctypes as C

import numpy as np
import pytest

from _util import P, i16p, load_oracle, u32p
from me_search_util import (FRAC, MC_SHAPES, eff_sub_shift, load_me_search_emul, load_me_search_oracle, mc_scene, oracle_search, oracle_surface,
                            search_descs, src_blocks)


@pytest.fixture(scope="module")
def mso():
    return load_me_search_oracle()


@pytest.fixture(scope="module")
def oracle():
    return load_oracle()


@pytest.fixture(scope="module")
def emul():
    return load_me_search_emul()


def replay_keys(emul, oracle, sc, descs, src=None):
    keys, counts = [], np.zeros(3, np.int64)
    for d, blk in zip(descs, src_blocks(sc, descs, src)):
        surf = np.ascontiguousarray(oracle_surface(oracle, sc, d, blk))
        p = sc["refs"][d["ref_idx"]]
        M = sc["M"]
        win = C.c_void_p(p.ctypes.data + 2 * ((d["y"] + d["top"] + M) * p.shape[1] + d["x"] + d["left"] + M))
        fast = int(src is None and d["w"] in (4, 8, 12, 16, 24, 32, 48, 64))
        kernel_o = int(src is None and sc["bd"] == 8)
        cnt = np.zeros(3, np.int32)
        k = emul.emul_me_search_key(sc["bd"], P(blk, i16p), d["w"], d["w"], d["h"], win, p.shape[1], d["left"], d["right"], d["top"], d["bottom"], eff_sub_shift(d),
                                    fast, kernel_o, P(surf, u32p), d["lambda"] & 0xFFFFFFFF, d["pred_x"], d["pred_y"], cnt.ctypes.data)
        keys.append(int(k))
        counts += cnt
    return keys, counts


def want_keys(mso, sc, descs, src=None):
    res = oracle_search(mso, sc, descs, src)
    out = []
    for d, r in zip(descs, res):
        cols = d["right"] - d["left"] + 1
        cost = mso.oracle_mv_cost(d["lambda"] & 0xFFFFFFFF, int(r[0]), int(r[1]), 2, d["pred_x"], d["pred_y"])
        out.append(((int(r[2]) + cost) << 32) | ((int(r[1]) - d["top"]) * cols + int(r[0]) - d["left"]))
    return out


@pytest.mark.parametrize("bd", [8, 9, 10])
def test_argmin_epilogue_matches_checker(emul, mso, oracle, bd):
    sc = mc_scene(bd, seed=50 + bd)
    rng = np.random.default_rng(bd + 7)
    descs = search_descs(sc, rng, flag_sets=(0,))
    got, counts = replay_keys(emul, oracle, sc, descs)
    assert got == want_keys(mso, sc, descs)
    assert counts[0] > 0 and counts[1] > 0 and counts[2] > 0            # O, M and E tiles all took part


def test_argmin_epilogue_signed_keys(emul, mso, oracle):
    sc = mc_scene(8, seed=61)
    rng = np.random.default_rng(61)
    descs = search_descs(sc, rng, shapes=MC_SHAPES[::2], radii=(64, 4), flag_sets=(0,))
    src = rng.integers(-700, 900, sum(d["w"] * d["h"] for d in descs)).astype(np.int16)
    got, counts = replay_keys(emul, oracle, sc, descs, src)
    assert got == want_keys(mso, sc, descs, src)
    assert counts[1] == 0 and counts[2] == 0                            # caller-supplied blocks: dx-lane tiles only


def test_prep_decodes_every_key(emul, mso):
    rng = np.random.default_rng(3)
    n = 300
    job, cost, keys, want = np.zeros((n, 5), np.int32), np.zeros((n, 4), np.int32), np.zeros(n, np.uint64), []
    stride, ref_in, frac_of = 608, [], []
    for i in range(n):
        left, top = (int(v) for v in rng.integers(-80, 10, 2))
        cols, rows = (int(v) for v in rng.integers(1, 130, 2))
        lam = int(rng.choice([0, 157084, 888605, 0xFFFFFFFF]))
        px, py = (int(v) for v in rng.integers(-32768, 32768, 2))
        dx, dy = int(rng.integers(0, cols)), int(rng.integers(0, rows))
        sad = int(rng.integers(0, 1 << 23))
        c = mso.oracle_mv_cost(lam, left + dx, top + dy, 2, px, py)
        keys[i] = ((sad + c) << 32) | (dy * cols + dx)
        frac = len(ref_in) if i % 3 else -1
        base = int(rng.integers(0, 1 << 20))
        if frac >= 0:
            ref_in.append(base)
            frac_of.append((i, base + (top + dy) * stride + left + dx))
        job[i] = (left, left + cols - 1, top, top + rows - 1, base)
        cost[i] = (lam - (1 << 32) if lam > 0x7FFFFFFF else lam, px, py, frac)
        want.append((left + dx, top + dy, sad, 4 * (left + dx), 4 * (top + dy), 0))
    out = np.zeros((n, 6), np.int32)
    ref_out = np.zeros(max(1, len(ref_in)), np.int32)
    ref_in = np.array(ref_in or [0], np.int32)
    emul.emul_me_search_prep(n, keys.ctypes.data, job.ctypes.data, cost.ctypes.data, stride, len(frac_of), ref_in.ctypes.data, ref_out.ctypes.data, out.ctypes.data)
    got = out.astype(np.int64)
    got[:, [2, 5]] = out[:, [2, 5]].view(np.uint32)
    assert [tuple(r) for r in got] == want
    assert [int(ref_out[f]) for f in range(len(frac_of))] == [r for _, r in frac_of]


def test_walk_matches_checker(emul, mso):
    rng = np.random.default_rng(4)
    for _ in range(2000):
        T = rng.integers(0, 1 << int(rng.integers(4, 20)), 49).astype(np.uint32)
        if rng.random() < 0.3:                                          # ties
            T[rng.integers(0, 49, 6)] = T.min()
        mvx, mvy = (int(v) for v in rng.integers(-200, 200, 2))
        px, py = (int(v) for v in rng.integers(-32768, 32768, 2))
        lam = int(rng.choice([0, 157084, 888605, 0xFFFFFFFF]))
        res = np.array([mvx, mvy, 0, 0, 0, 0], np.int32)
        emul.emul_me_search_walk(T.ctypes.data, lam, px, py, res.ctypes.data)
        qmv, fc = np.zeros(2, np.int32), np.zeros(1, np.uint32)
        mso.oracle_me_frac_walk(T.ctypes.data, mvx, mvy, px, py, lam, qmv.ctypes.data, fc.ctypes.data)
        assert (res[3], res[4], np.uint32(res[5])) == (qmv[0], qmv[1], fc[0])


def test_flags_constant():
    assert FRAC == 1
