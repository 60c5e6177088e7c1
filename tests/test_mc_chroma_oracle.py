"""The checker of cucd_me_mc_chroma (tests/mc_chroma_oracle.c) against statements that do not share its code: an independent numpy
statement of HM's four xPredInterBlk chroma branches and addAvg, integer MVs that copy the reference, constant planes, bi-prediction
with identical motion, the mirror symmetry of the half-sample filter, and its SSE against oracle_sse of the prediction it returns."""
import ctypes as C

import numpy as np
import pytest

from _util import P, i16p
from mc_chroma_util import load_mc_chroma_oracle

TAPS = np.array([[0, 64, 0, 0], [-2, 58, 10, -2], [-4, 54, 16, -2], [-6, 46, 28, -4], [-4, 36, 36, -4], [-4, 28, 46, -6], [-2, 16, 54, -4],
                 [-2, 10, 58, -2]], np.int64)
OFFS = 1 << 13                                        # IF_INTERNAL_OFFS
FRACS = [(fx, fy) for fy in range(8) for fx in range(8)]


@pytest.fixture(scope="module")
def mco():
    return load_mc_chroma_oracle()


# ---- numpy statement of TComInterpolationFilter::filter<4> / filterCopy and the chroma branch of xPredInterBlk ----------------------
def np_copy(bd, src, is_first, is_last):
    shift = max(2, 14 - bd)
    s = src.astype(np.int64)
    if is_first == is_last:
        return s
    if is_first:
        return (s << shift) - OFFS
    return np.clip((s + OFFS + (1 << (shift - 1))) >> shift, 0, (1 << bd) - 1)


def np_filter(bd, src, frac, vertical, is_first, is_last, w, h):
    """src: the samples rows -1 .. h + 2 (vertical) or columns -1 .. w + 2 (horizontal) around the block"""
    head = 14 - bd
    if is_last:
        shift = 6 + (0 if is_first else head)
        offset = (1 << (shift - 1)) + (0 if is_first else OFFS << 6)
    else:
        shift = 6 - (head if is_first else 0)
        offset = -OFFS * (1 << shift) if is_first else 0
    s = src.astype(np.int64)
    acc = sum(TAPS[frac][k] * (s[k:k + h, :] if vertical else s[:, k:k + w]) for k in range(4))
    v = (acc + offset) >> shift
    return np.clip(v, 0, (1 << bd) - 1) if is_last else v


def np_pred_blk(bd, plane, y, x, w, h, fx, fy, bi):
    """xPredInterBlk (chroma) of the block at integer position (y, x) of `plane`"""
    last = not bi
    if fy == 0:
        return np_copy(bd, plane[y:y + h, x:x + w], True, last) if fx == 0 else np_filter(bd, plane[y:y + h, x - 1:x + w + 2], fx, False, True, last, w, h)
    if fx == 0:
        return np_filter(bd, plane[y - 1:y + h + 2, x:x + w], fy, True, True, last, w, h)
    tmp = np_filter(bd, plane[y - 1:y + h + 2, x - 1:x + w + 2], fx, False, True, False, w, h + 3)
    return np_filter(bd, tmp, fy, True, False, last, w, h)


def np_add_avg(bd, p0, p1):
    shift = max(2, 14 - bd) + 1
    return np.clip((p0 + p1 + (1 << (shift - 1)) + 2 * OFFS) >> shift, 0, (1 << bd) - 1)


def random_plane(bd, rng, H=40, W=72):
    """noise with runs of 0 and 2^bd - 1 (rows, columns and a checkerboard patch) so that every clip and extreme is reached"""
    hi = (1 << bd) - 1
    p = rng.integers(0, hi + 1, (H, W))
    p[4:6, :] = hi
    p[:, 20:22] = 0
    p[24:34, 40:64] = np.where(np.indices((10, 24)).sum(0) % 2 == 0, hi, 0)
    return np.ascontiguousarray(p.astype(np.int16))


def mc_pred(mco, bd, plane, lists, w, h):
    """oracle_mc_chroma_pred; lists: [(y, x, fx, fy)] with one or two entries, integer positions inside `plane`"""
    S = plane.shape[1]
    a = [(C.c_void_p(plane.ctypes.data + 2 * (y * S + x)), S, fx, fy) for y, x, fx, fy in lists]
    b = a[1] if len(a) == 2 else (None, 0, 0, 0)
    out = np.zeros((h, w), np.int16)
    mco.oracle_mc_chroma_pred(bd, len(a), a[0][0], a[0][1], a[0][2], a[0][3], b[0], b[1], b[2], b[3], w, h, P(out, i16p))
    return out


def pos(rng, plane, w, h):
    return int(rng.integers(1, plane.shape[0] - h - 2)), int(rng.integers(1, plane.shape[1] - w - 2))


@pytest.mark.parametrize("bd", [8, 10])
@pytest.mark.parametrize("w,h", [(2, 4), (4, 2), (6, 8), (8, 8), (16, 4)])
def test_oracle_matches_numpy_statement_of_the_four_branches(mco, bd, w, h):
    """all 64 fraction pairs of list 0 uni, and each against all 64 of list 1 (bi); the blocks sit on and around the extreme runs"""
    rng = np.random.default_rng(bd * 100 + 7 * w + h)
    plane = random_plane(bd, rng)
    for fx0, fy0 in FRACS:
        y0, x0 = pos(rng, plane, w, h)
        p0 = np_pred_blk(bd, plane, y0, x0, w, h, fx0, fy0, bi=False)
        assert np.array_equal(mc_pred(mco, bd, plane, [(y0, x0, fx0, fy0)], w, h), p0), ("uni", fx0, fy0)
        i0 = np_pred_blk(bd, plane, y0, x0, w, h, fx0, fy0, bi=True)
        lo, hi = (-10750, 10733) if fy0 == 0 else (-14107, 14089)                   # the bounds of me_core.cuh: stage 1 (fy = 0), stage 2
        assert lo <= i0.min() and i0.max() <= hi
        for fx1, fy1 in FRACS:
            y1, x1 = pos(rng, plane, w, h)
            i1 = np_pred_blk(bd, plane, y1, x1, w, h, fx1, fy1, bi=True)
            got = mc_pred(mco, bd, plane, [(y0, x0, fx0, fy0), (y1, x1, fx1, fy1)], w, h)
            assert np.array_equal(got, np_add_avg(bd, i0, i1)), ("bi", fx0, fy0, fx1, fy1)


@pytest.mark.parametrize("bd", [8, 10])
def test_integer_motion_copies_the_reference(mco, bd):
    rng = np.random.default_rng(bd + 11)
    plane = random_plane(bd, rng)
    for w, h in ((2, 4), (4, 2), (6, 8), (12, 16), (32, 32)):
        y, x = pos(rng, plane, w, h)
        want = plane[y:y + h, x:x + w]
        assert np.array_equal(mc_pred(mco, bd, plane, [(y, x, 0, 0)], w, h), want), (w, h)
        assert np.array_equal(mc_pred(mco, bd, plane, [(y, x, 0, 0)] * 2, w, h), want), (w, h)


@pytest.mark.parametrize("bd", [8, 10])
def test_constant_reference_predicts_the_constant(mco, bd):
    for c in (0, 1, (1 << bd) // 3, (1 << bd) - 1):
        plane = np.full((24, 24), c, np.int16)
        for fx, fy in FRACS:
            assert (mc_pred(mco, bd, plane, [(4, 4, fx, fy)], 8, 4) == c).all()
            assert (mc_pred(mco, bd, plane, [(4, 4, fx, fy), (6, 5, 7 - fy, fx)], 8, 4) == c).all()


@pytest.mark.parametrize("bd", [8, 10])
def test_bi_with_identical_motion_equals_uni(mco, bd):
    rng = np.random.default_rng(bd)
    plane = random_plane(bd, rng)
    for fx, fy in FRACS:
        for w, h in ((2, 8), (8, 8), (16, 12)):
            y, x = pos(rng, plane, w, h)
            assert np.array_equal(mc_pred(mco, bd, plane, [(y, x, fx, fy)] * 2, w, h), mc_pred(mco, bd, plane, [(y, x, fx, fy)], w, h)), (fx, fy, w, h)


@pytest.mark.parametrize("bd", [8, 10])
def test_half_sample_filter_is_mirror_symmetric(mco, bd):
    """fraction 4 has symmetric taps: the plane mirrored in both axes predicts the mirrored block.  A half-sample position x + c + 1/2
    of a plane W wide lands on (W - 2 - x - c) + 1/2 of the mirrored plane, a whole-sample position x + c on W - 1 - x - c"""
    rng = np.random.default_rng(bd + 5)
    plane = random_plane(bd, rng)
    mirror = np.ascontiguousarray(plane[::-1, ::-1])
    Hp, Wp = plane.shape
    for fx in (0, 4):
        for fy in (0, 4):
            for w, h in ((2, 4), (6, 8), (16, 16)):
                y, x = pos(rng, plane, w, h)
                ym, xm = Hp - h - y - (1 if fy else 0), Wp - w - x - (1 if fx else 0)
                for bi in (False, True):
                    a = [(y, x, fx, fy)] * (2 if bi else 1)
                    b = [(ym, xm, fx, fy)] * (2 if bi else 1)
                    assert np.array_equal(mc_pred(mco, bd, plane, a, w, h)[::-1, ::-1], mc_pred(mco, bd, mirror, b, w, h)), (fx, fy, w, h, bi)


@pytest.mark.parametrize("bd", [8, 10])
def test_sse_is_oracle_sse_of_the_prediction(mco, bd):
    rng = np.random.default_rng(bd + 9)
    plane = random_plane(bd, rng)
    for w, h in ((2, 4), (8, 6), (32, 32)):
        org = np.ascontiguousarray(rng.integers(0, 1 << bd, (h, w)).astype(np.int16))
        for fx, fy in FRACS[::5]:
            (y0, x0), (y1, x1) = pos(rng, plane, w, h), pos(rng, plane, w, h)
            for nl in (1, 2):
                S = plane.shape[1]
                r0, r1 = C.c_void_p(plane.ctypes.data + 2 * (y0 * S + x0)), C.c_void_p(plane.ctypes.data + 2 * (y1 * S + x1))
                pred = np.zeros((h, w), np.int16)
                sse = mco.oracle_mc_chroma_cost(bd, P(org, i16p), w, nl, r0, S, fx, fy, r1 if nl == 2 else None, S, fy, fx, w, h, P(pred, i16p))
                assert sse == mco.oracle_sse(bd, P(org, i16p), w, P(pred, i16p), w, w, h)
                d = org.astype(np.int64) - pred
                assert sse == int(((d * d) >> (2 * (bd - 8))).sum())
