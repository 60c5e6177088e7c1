"""The checker of cucd_me_mc_cost (tests/mc_oracle.c) against statements that do not share its code: an independent numpy statement
of HM's four xPredInterBlk branches and addAvg, constant planes, bi-prediction with identical motion (the arithmetic fact behind
xCheckIdenticalMotion), and the uni-directional costs of oracle_subpel_surface, which the encoder dumps tests/golden/frac_*.npz pin."""
import ctypes as C

import numpy as np
import pytest

from _util import P, golden, frac_records, i16p, u32p
from mc_util import load_mc_oracle

TAPS = np.array([[0, 0, 0, 64, 0, 0, 0, 0], [-1, 4, -10, 58, 17, -5, 1, 0], [-1, 4, -11, 40, 40, -11, 4, -1], [0, 1, -5, 17, 58, -10, 4, -1]], np.int64)
OFFS = 1 << 13                                        # IF_INTERNAL_OFFS


@pytest.fixture(scope="module")
def mco():
    return load_mc_oracle()


# ---- numpy statement of TComInterpolationFilter::filter / filterCopy and TComPrediction::xPredInterBlk ----------------------------
def np_copy(bd, src, is_first, is_last):
    shift = max(2, 14 - bd)
    s = src.astype(np.int64)
    if is_first == is_last:
        return s
    if is_first:
        return (s << shift) - OFFS
    return np.clip((s + OFFS + (1 << (shift - 1))) >> shift, 0, (1 << bd) - 1)


def np_filter(bd, src, frac, vertical, is_first, is_last, w, h):
    """src: the samples rows -3 .. h + 3 (vertical) or columns -3 .. w + 3 (horizontal) around the block"""
    head = 14 - bd
    if is_last:
        shift = 6 + (0 if is_first else head)
        offset = (1 << (shift - 1)) + (0 if is_first else OFFS << 6)
    else:
        shift = 6 - (head if is_first else 0)
        offset = -OFFS * (1 << shift) if is_first else 0
    s = src.astype(np.int64)
    acc = sum(TAPS[frac][k] * (s[k:k + h, :] if vertical else s[:, k:k + w]) for k in range(8))
    v = (acc + offset) >> shift
    return np.clip(v, 0, (1 << bd) - 1) if is_last else v


def np_pred_blk(bd, plane, y, x, w, h, fx, fy, bi):
    """xPredInterBlk (luma) of the block at integer position (y, x) of `plane`"""
    last = not bi
    if fy == 0:
        return np_copy(bd, plane[y:y + h, x:x + w], True, last) if fx == 0 else np_filter(bd, plane[y:y + h, x - 3:x + w + 4], fx, False, True, last, w, h)
    if fx == 0:
        return np_filter(bd, plane[y - 3:y + h + 4, x:x + w], fy, True, True, last, w, h)
    tmp = np_filter(bd, plane[y - 3:y + h + 4, x - 3:x + w + 4], fx, False, True, False, w, h + 7)
    return np_filter(bd, tmp, fy, True, False, last, w, h)


def np_add_avg(bd, p0, p1):
    shift = max(2, 14 - bd) + 1
    return np.clip((p0 + p1 + (1 << (shift - 1)) + 2 * OFFS) >> shift, 0, (1 << bd) - 1)


def random_plane(bd, rng, H=48, W=96):
    """noise with runs of 0 and 2^bd - 1 (rows, columns and a checkerboard patch) so that every clip and extreme is reached"""
    hi = (1 << bd) - 1
    p = rng.integers(0, hi + 1, (H, W))
    p[4:7, :] = hi
    p[:, 20:23] = 0
    p[30:40, 50:80] = np.where(np.indices((10, 30)).sum(0) % 2 == 0, hi, 0)
    return np.ascontiguousarray(p.astype(np.int16))


def mc_pred(mco, bd, plane, lists, w, h):
    """oracle_mc_pred; lists: [(y, x, fx, fy)] with one or two entries, integer positions inside `plane`"""
    S = plane.shape[1]
    a = [(C.c_void_p(plane.ctypes.data + 2 * (y * S + x)), S, fx, fy) for y, x, fx, fy in lists]
    b = a[1] if len(a) == 2 else (None, 0, 0, 0)
    out = np.zeros((h, w), np.int16)
    mco.oracle_mc_pred(bd, len(a), a[0][0], a[0][1], a[0][2], a[0][3], b[0], b[1], b[2], b[3], w, h, P(out, i16p))
    return out


@pytest.mark.parametrize("bd", [8, 10])
@pytest.mark.parametrize("w,h", [(8, 8), (16, 4), (4, 12), (12, 16)])
def test_oracle_matches_numpy_statement_of_the_four_branches(mco, bd, w, h):
    """all 16 fraction pairs of list 0 against all 16 of list 1 (bi), and all 16 uni; the blocks sit on and around the extreme runs"""
    rng = np.random.default_rng(bd * 100 + w + h)
    plane = random_plane(bd, rng)
    fr = [(fx, fy) for fy in range(4) for fx in range(4)]
    for i, (fx0, fy0) in enumerate(fr):
        y0, x0 = int(rng.integers(3, 48 - h - 4)), int(rng.integers(3, 96 - w - 4))
        p0 = np_pred_blk(bd, plane, y0, x0, w, h, fx0, fy0, bi=False)
        assert np.array_equal(mc_pred(mco, bd, plane, [(y0, x0, fx0, fy0)], w, h), p0), ("uni", fx0, fy0)
        i0 = np_pred_blk(bd, plane, y0, x0, w, h, fx0, fy0, bi=True)
        assert i0.min() >= -32768 and i0.max() <= 32767
        for fx1, fy1 in fr:
            y1, x1 = int(rng.integers(3, 48 - h - 4)), int(rng.integers(3, 96 - w - 4))
            i1 = np_pred_blk(bd, plane, y1, x1, w, h, fx1, fy1, bi=True)
            want = np_add_avg(bd, i0, i1)
            got = mc_pred(mco, bd, plane, [(y0, x0, fx0, fy0), (y1, x1, fx1, fy1)], w, h)
            assert np.array_equal(got, want), ("bi", fx0, fy0, fx1, fy1)


@pytest.mark.parametrize("bd", [8, 10])
def test_constant_reference_predicts_the_constant(mco, bd):
    for c in (0, 1, (1 << bd) // 3, (1 << bd) - 1):
        plane = np.full((40, 40), c, np.int16)
        for fx in range(4):
            for fy in range(4):
                assert (mc_pred(mco, bd, plane, [(8, 8, fx, fy)], 16, 8) == c).all()
                assert (mc_pred(mco, bd, plane, [(8, 8, fx, fy), (10, 12, 3 - fy, fx)], 16, 8) == c).all()


@pytest.mark.parametrize("bd", [8, 10])
def test_bi_with_identical_motion_equals_uni(mco, bd):
    rng = np.random.default_rng(bd)
    plane = random_plane(bd, rng)
    for fx in range(4):
        for fy in range(4):
            for w, h in ((8, 8), (4, 16), (32, 24)):
                y, x = int(rng.integers(3, 48 - h - 4)), int(rng.integers(3, 96 - w - 4))
                assert np.array_equal(mc_pred(mco, bd, plane, [(y, x, fx, fy)] * 2, w, h), mc_pred(mco, bd, plane, [(y, x, fx, fy)], w, h)), (fx, fy, w, h)


@pytest.mark.parametrize("clip", ["had8", "sad10"])
def test_uni_cost_equals_the_pinned_subpel_surface(mco, clip):
    """every record of the encoder dump: oracle_mc_cost at the record's quarter-pel offset equals oracle_subpel_surface's entry, and
    that entry equals the distortion the encoder computed"""
    n = 0
    for r in frac_records(golden(f"frac_{clip}.npz")):
        bd, w, h = r["bd"], r["w"], r["h"]
        org = np.ascontiguousarray(r["org"], np.int16)
        win = np.ascontiguousarray(r["win"], np.int16)               # (h + 9) x (w + 9), origin (-4, -4) from zero MV
        S = win.shape[1]
        zero = win.ctypes.data + 2 * (4 * S + 4)
        surf = np.zeros(49, np.uint32)
        mco.oracle_subpel_surface(bd, P(org, i16p), w, w, h, C.c_void_p(zero), S, 0, 0, r["had"], P(surf, u32p))
        qx, qy = r["qx"], r["qy"]
        at = C.c_void_p(zero + 2 * ((qy >> 2) * S + (qx >> 2)))
        got = mco.oracle_mc_cost(bd, P(org, i16p), w, 1, at, S, qx & 3, qy & 3, None, 0, 0, 0, w, h, r["had"], None)
        assert got == surf[(qy + 3) * 7 + qx + 3] == r["dist"], (w, h, qx, qy)
        n += 1
    assert n > 0
