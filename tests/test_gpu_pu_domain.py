"""Every PU shape and row sub-sampling the ME calls accept, not only the 22 HEVC shapes: against the oracles at 8, 9 and 10 bit.

cucd_me_desc / cucd_search_desc / cucd_tz_desc take any width that is a multiple of 4 in 4..64, any height in 4..64 (h % 4 is checked
only with FRAC) and sub_shift 0..4.  Widths outside HM's list (20, 28, 36, ...) ignore sub_shift, as the generic xGetSAD does, and run on
the dx-lane kernels; the TZ kernel stages ceil(h / 2^sub_shift) source rows.  Sub-pel, MC and chroma MC take every multiple-of-4 shape,
4x4 (chroma 2x2) included, and small ones such as 20x12 or 4x60 go to me_subpel_small_kernel.

The tests marked gpu run the sweep through the C ABI; the others run the same sweep through the CPU replays of the kernel code
(tests/emul), so that a change of the tiling, the staging or the sub-sampling rule is caught without a GPU as well."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from _util import P, ROOT, i16p, u32p
from mc_chroma_util import emul_mc_chroma, load_mc_chroma_emul, load_mc_chroma_oracle, mcc_candidates, mcc_scene, oracle_mc_chroma
from mc_util import emul_mc, load_mc_emul, load_mc_oracle, mc_candidates, mc_scene, oracle_mc
from me_search_util import FRAC, HAD, LAMBDAS, as_rows, eff_sub_shift, load_me_search_oracle, oracle_search, oracle_surface, search_desc, src_blocks
from me_tz_util import TZ2N, emul_tz, load_me_tz_emul, load_me_tz_oracle, oracle_tz, oracle_tz_rows, ref_base, src_block, tz_desc

BDS = (8, 9, 10)
WIDTHS = tuple(range(4, 65, 4))
HM_WIDTHS = (4, 8, 12, 16, 24, 32, 48, 64)
HEIGHTS = (4, 5, 6, 7, 9, 16, 33, 63, 64)                 # every h % 4 class, odd heights at both ends of the range
SUB_SHIFTS = tuple(range(5))
SHAPES4 = [(w, h) for w in WIDTHS for h in range(4, 65, 4)]   # the 256 shapes of pu_shape_ok
# windows (left, right, top, bottom) of the SAD sweep.  For HM's widths: 67 x 69 candidates = M tiles + an E strip (3 columns) + O rows;
# 37 x 33 = an M tile + an O strip (5 columns) + an O row; 9 x 9 = one O tile
WINDOWS = ((-33, 33, -40, 28), (-20, 16, -16, 16), (-4, 4, -3, 5))


with open(os.path.join(ROOT, "fast-cu-decision-hevc_b200", "csrc", "me_core.cuh")) as _f:
    _a, _b = re.search(r"kSpHorCap = (\d+) \* (\d+);", _f.read()).groups()
SP_HOR_CAP = int(_a) * int(_b)


def subpel_is_small(w, h):
    """me_core.cuh subpel_is_small: the PUs me_subpel_small_kernel takes"""
    return w * h <= 256 and 7 * (h + 9) * w <= SP_HOR_CAP


def sad_sweep(bd):
    """(scene, descs): one PU per width, height and sub_shift, the windows of WINDOWS in turn"""
    sc = mc_scene(bd, W=192, H=128, slots=(0,), seed=bd + 500)
    rng = np.random.default_rng(bd + 500)
    descs = []
    for w in WIDTHS:
        for h in HEIGHTS:
            for s in SUB_SHIFTS:
                l, r, t, b = WINDOWS[len(descs) % len(WINDOWS)]
                x, y = int(rng.integers(0, (sc["W"] - w) // 4 + 1)) * 4, int(rng.integers(0, sc["H"] - h + 1))
                descs.append(dict(x=x, y=y, w=w, h=h, ref_idx=0, left=l, right=r, top=t, bottom=b, sub_shift=s))
    assert {d["w"] for d in descs} == set(WIDTHS) and {d["h"] % 4 for d in descs} == {0, 1, 2, 3}
    assert {d["sub_shift"] for d in descs} == set(SUB_SHIFTS)
    assert {(d["w"], d["left"]) for d in descs} == {(w, W[0]) for w in WIDTHS for W in WINDOWS}     # every window for every width
    return sc, descs


def odd_pus(sc, rng, make):
    """generic widths with every sub_shift, and HM's widths at heights that are not multiples of 4 (nor of 2^sub_shift): make(x, y, w, h,
    sub_shift, n) builds the descriptor"""
    out = []
    shapes = [(w, h) for w in WIDTHS if w not in HM_WIDTHS for h in (4, 7, 12, 33, 64)] + [(w, h) for w in HM_WIDTHS for h in (5, 6, 9, 63)]
    for w, h in shapes:
        n = len(out)
        x, y = int(rng.integers(0, (sc["W"] - w) // 4 + 1)) * 4, int(rng.integers(0, sc["H"] - h + 1))
        out.append(make(x, y, w, h, n % 5, n))
    assert {d["w"] for d in out} == set(WIDTHS) and {d["h"] % 4 for d in out} == {0, 1, 2, 3} and {d["sub_shift"] for d in out} == set(SUB_SHIFTS)
    assert any(d["w"] in HM_WIDTHS and d["h"] % (1 << d["sub_shift"]) for d in out)              # a partial last row group
    assert any(d["w"] not in HM_WIDTHS and d["sub_shift"] > 0 for d in out)
    return out


def search_sweep(bd):
    sc = mc_scene(bd, seed=bd + 510)
    rng = np.random.default_rng(bd + 510)

    def make(x, y, w, h, s, n):
        fl = (FRAC | HAD, FRAC)[n % 2] if h % 4 == 0 else 0
        cx, cy = int(rng.integers(-10, 11)), int(rng.integers(-10, 11))
        return search_desc(sc, x, y, w, h, sc["slots"][n % 2], cx, cy, 12 if n % 3 else 40, sub_shift=s, pred=(4 * cx + 3, 4 * cy - 5),
                           lam=LAMBDAS[n % 3], flags=fl)
    return sc, odd_pus(sc, rng, make)


def tz_sweep(bd):
    sc = mc_scene(bd, seed=bd + 520)
    rng = np.random.default_rng(bd + 520)

    def make(x, y, w, h, s, n):
        fl = ((FRAC | HAD, FRAC | TZ2N)[n % 2] if h % 4 == 0 else (0, TZ2N)[n % 2])
        pred = (int(rng.integers(-60, 61)), int(rng.integers(-60, 61)))
        return tz_desc(sc, x, y, w, h, sc["slots"][n % 2], pred, (16, 64)[n % 2], sub_shift=s, lam=LAMBDAS[n % 3], flags=fl,
                       mv2n=tuple(int(v) for v in rng.integers(-8, 9, 2)))
    return sc, odd_pus(sc, rng, make)


def subpel_sweep(bd):
    sc = mc_scene(bd, seed=bd + 530)
    rng = np.random.default_rng(bd + 530)
    descs = []
    for w, h in SHAPES4:
        for had in (1, 0):
            x, y = int(rng.integers(0, (sc["W"] - w) // 4 + 1)) * 4, int(rng.integers(0, (sc["H"] - h) // 4 + 1)) * 4
            mvx, mvy = int(rng.integers(-x - 70, sc["W"] - x - w + 70)), int(rng.integers(-y - 70, sc["H"] - y - h + 70))
            descs.append(dict(x=x, y=y, w=w, h=h, ref_idx=sc["slots"][len(descs) % 2], mvx=mvx, mvy=mvy, use_hadamard=had))
    return sc, descs


def subpel_want(oracle, sc, descs):
    out = np.zeros((len(descs), 49), np.uint32)
    for i, d in enumerate(descs):
        blk = src_block(sc, d)
        oracle.oracle_subpel_surface(sc["bd"], P(blk, i16p), d["w"], d["w"], d["h"], ref_base(sc, d), sc["refs"][d["ref_idx"]].shape[1], d["mvx"], d["mvy"],
                                     d["use_hadamard"], P(out[i], u32p))
    return out


def mc_sweep(bd):
    sc = mc_scene(bd, seed=bd + 540)
    descs = mc_candidates(sc, np.random.default_rng(bd + 540), shapes=SHAPES4, modes=("l0", "l1", "bi"))
    assert {(d["w"], d["h"]) for d in descs} == set(SHAPES4) and {d["use_hadamard"] for d in descs} == {0, 1}
    return sc, descs


def mcc_sweep(bd):
    sc = mcc_scene(bd, seed=bd + 550)
    descs = mcc_candidates(sc, np.random.default_rng(bd + 550), shapes=SHAPES4, modes=("l0", "l1", "bi"))
    return sc, descs


@pytest.fixture(scope="module")
def mso():
    return load_me_search_oracle()


@pytest.fixture(scope="module")
def tzo():
    return load_me_tz_oracle()


@pytest.fixture(scope="module")
def mco():
    return load_mc_oracle()


@pytest.fixture(scope="module")
def mcco():
    return load_mc_chroma_oracle()


def engine(cucd, sc):
    eng = cucd.Engine(sc["W"], sc["H"], bit_depth=sc["bd"])
    eng.set_cur_picture(sc["org"])
    for s, p in sc["refs"].items():
        eng.set_ref_picture(s, p, sc["M"], sc["M"])
    return eng


# ---- through the C ABI -----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("bd", BDS)
def test_sad_surface_every_width_height_and_sub_shift(cucd, oracle, bd):
    """cucd_me_sad_surface (dy-lane and dx-lane kernels) and cucd_me_sad_surface_src (the signed dx-lane kernel) on the same PUs; a
    generic width's surface equals its sub_shift 0 surface"""
    sc, descs = sad_sweep(bd)
    blocks = src_blocks(sc, descs)
    with engine(cucd, sc) as eng:
        got = eng.me_sad_surface(descs)
        got_src = eng.me_sad_surface(descs, src=np.concatenate([b.ravel() for b in blocks]))
        generic = [d for d in descs if d["w"] not in HM_WIDTHS]
        got0 = eng.me_sad_surface([dict(d, sub_shift=0) for d in generic])
    for d, blk, g, gs in zip(descs, blocks, got, got_src):
        want = oracle_surface(oracle, sc, d, blk)
        assert np.array_equal(g, want), d
        assert np.array_equal(gs, want), ("src", d)
    for d, g, g0 in zip(generic, [g for d, g in zip(descs, got) if d["w"] not in HM_WIDTHS], got0):
        assert np.array_equal(g, g0), d


@pytest.mark.gpu
@pytest.mark.parametrize("bd", BDS)
def test_search_generic_widths_and_odd_heights(cucd, mso, bd):
    """cucd_me_search: integer only where h % 4 != 0, FRAC (Hadamard and SAD) otherwise"""
    sc, descs = search_sweep(bd)
    want = oracle_search(mso, sc, descs)
    with engine(cucd, sc) as eng:
        got = as_rows(eng.me_search(descs))
    for i, d in enumerate(descs):
        assert np.array_equal(got[i], want[i]), (d, got[i], want[i])


@pytest.mark.gpu
@pytest.mark.parametrize("bd", BDS)
def test_tz_search_generic_widths_and_odd_heights(cucd, tzo, bd):
    sc, descs = tz_sweep(bd)
    want = oracle_tz_rows(tzo, sc, descs)
    with engine(cucd, sc) as eng:
        got = as_rows(eng.me_tz_search(descs))
    for i, d in enumerate(descs):
        assert np.array_equal(got[i], want[i]), (d, got[i], want[i])


@pytest.mark.gpu
@pytest.mark.parametrize("bd", BDS)
def test_subpel_every_multiple_of_4_shape(cucd, oracle, bd):
    """all 256 shapes, Hadamard and SAD: both sub-pel kernels take part"""
    sc, descs = subpel_sweep(bd)
    small = [subpel_is_small(d["w"], d["h"]) for d in descs]
    assert 0 < sum(small) < len(descs)
    want = subpel_want(oracle, sc, descs)
    with engine(cucd, sc) as eng:
        got = eng.me_subpel_cost(descs)
    for i, d in enumerate(descs):
        assert np.array_equal(got[i].ravel(), want[i]), d


@pytest.mark.gpu
@pytest.mark.parametrize("bd", BDS)
def test_mc_cost_every_multiple_of_4_shape(cucd, mco, bd):
    sc, descs = mc_sweep(bd)
    want_d, want_p = oracle_mc(mco, sc, descs)
    with engine(cucd, sc) as eng:
        got_d, got_p = eng.me_mc_cost(descs, want_pred=True)
    for i, d in enumerate(descs):
        assert np.array_equal(got_p[i], want_p[i]) and got_d[i] == want_d[i], d


@pytest.mark.gpu
@pytest.mark.parametrize("bd", BDS)
def test_mc_chroma_every_multiple_of_4_shape(cucd, mcco, bd):
    """chroma blocks 2x2 .. 32x32"""
    sc, descs = mcc_sweep(bd)
    want_s, want_p = oracle_mc_chroma(mcco, sc, descs)
    with engine(cucd, sc) as eng:
        eng.set_cur_picture_chroma(*sc["org_c"])
        for s, (cb, cr) in sc["refs_c"].items():
            eng.set_ref_picture_chroma(s, cb, cr, sc["Mc"], sc["Mc"])
        got_s, got_p = eng.me_mc_chroma(descs, want_pred=True)
    for i, d in enumerate(descs):
        assert np.array_equal(got_s[i], want_s[i]) and all(np.array_equal(got_p[i][c], want_p[i][c]) for c in range(2)), d


# ---- the same sweeps through the CPU replays of the kernel code -------------------------------------------------------------------
@pytest.mark.parametrize("bd", BDS)
def test_sad_sweep_dy_lane_kernel_code(emul, oracle, bd):
    """HM's widths (the dy-lane kernel's): every height and sub_shift, the tiles M, E and O of the large window each taken"""
    sc, descs = sad_sweep(bd)
    p, M = sc["refs"][0], sc["M"]
    seen = set()
    for d, blk in zip(descs, src_blocks(sc, descs)):
        if d["w"] not in HM_WIDTHS:
            continue
        cols, rows = d["right"] - d["left"] + 1, d["bottom"] - d["top"] + 1
        got = np.full((rows, cols), 0xdeadbeef, np.uint32)
        hits = np.zeros((rows, cols), np.uint8)
        counts = (C.c_int * 3)()
        win = C.c_void_p(p.ctypes.data + 2 * ((d["y"] + M + d["top"]) * p.shape[1] + d["x"] + M + d["left"]))
        emul.emul_me_sad_surface(bd, P(blk, i16p), d["w"], d["w"], d["h"], win, p.shape[1], cols, rows, d["sub_shift"], P(got, u32p),
                                 hits.ctypes.data_as(C.c_void_p), counts)
        assert (hits == 1).all(), d
        want = oracle_surface(oracle, sc, d, blk)
        dy = got != 0xffffffff
        assert np.array_equal(got[dy], want[dy]), d
        if (d["left"], d["right"], d["top"], d["bottom"]) == WINDOWS[0]:
            assert all(counts), (d, list(counts))
            seen.add((d["w"], d["h"], d["sub_shift"]))
    assert {(w, s) for w, _, s in seen} == {(w, s) for w in HM_WIDTHS for s in SUB_SHIFTS}
    assert {h % 4 for _, h, _ in seen} == {0, 1, 2, 3}


@pytest.mark.parametrize("bd", BDS)
def test_tz_sweep_kernel_code(bd, tzo):
    """the replay of me_tz_kernel (its sub-sampling rule and row count) on the TZ sweep's PUs, integer result and every folded probe"""
    emul = load_me_tz_emul()
    sc, descs = tz_sweep(bd)
    for d in descs:
        want, wtrace, _ = oracle_tz(tzo, sc, dict(d, flags=d["flags"] & ~(FRAC | HAD)), trace_cap=200000)
        got, trace, _, _ = emul_tz(emul, sc, d)
        assert np.array_equal(got[:3], want[:3]), d
        assert np.array_equal(trace, wtrace), d
    assert {eff_sub_shift(d) for d in descs} == set(SUB_SHIFTS)


@pytest.mark.parametrize("bd", BDS)
def test_subpel_sweep_small_pu_kernel_code(emul, oracle, bd):
    """every shape me_subpel_small_kernel takes, and no other, through its replay"""
    sc, descs = subpel_sweep(bd)
    want = subpel_want(oracle, sc, descs)
    n_small = 0
    for i, d in enumerate(descs):
        got = np.full(49, 0xdeadbeef, np.uint32)
        p = sc["refs"][d["ref_idx"]]
        at_mv = C.c_void_p(p.ctypes.data + 2 * ((d["y"] + sc["M"] + d["mvy"]) * p.shape[1] + d["x"] + sc["M"] + d["mvx"]))
        small = emul.emul_subpel_small(bd, P(src_block(sc, d), i16p), d["w"], d["w"], d["h"], at_mv, p.shape[1], d["use_hadamard"], P(got, u32p))
        assert small == subpel_is_small(d["w"], d["h"]), d
        if small:
            assert np.array_equal(got, want[i]), d
            n_small += 1
    assert 0 < n_small < len(descs)


@pytest.mark.parametrize("bd", BDS)
def test_mc_sweep_kernel_code(mco, bd):
    sc, descs = mc_sweep(bd)
    want_d, want_p = oracle_mc(mco, sc, descs)
    got_d, got_p, n_cta = emul_mc(load_mc_emul(), sc, descs)
    assert n_cta > 0
    for i, d in enumerate(descs):
        assert np.array_equal(got_p[i], want_p[i]) and got_d[i] == want_d[i], d


@pytest.mark.parametrize("bd", BDS)
def test_mc_chroma_sweep_kernel_code(mcco, bd):
    sc, descs = mcc_sweep(bd)
    want_s, want_p = oracle_mc_chroma(mcco, sc, descs)
    got_s, got_p, n_cta = emul_mc_chroma(load_mc_chroma_emul(), sc, descs)
    assert n_cta > 0
    for i, d in enumerate(descs):
        assert np.array_equal(got_s[i], want_s[i]) and all(np.array_equal(got_p[i][c], want_p[i][c]) for c in range(2)), d
