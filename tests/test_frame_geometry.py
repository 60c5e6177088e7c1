"""The frame RMD paths at every picture-edge residue, at the strong-smoothing threshold and on the border pre-pass images of the 8-bit
tensor-core kernel, replayed on the CPU (tests/emul) against the plain-C oracle, bit for bit.

- the closed-form availability of the frame kernels (tc2::pu_avail) against the oracle's per-unit flags, and those against a statement
  of HEVC 6.4.1 z-scan availability written here;
- the ALU, tc2 and tc3 replays over EDGE_SIZES;
- the tc2 replay of the path the GPU runs (border pre-pass images, bulk copies) over several pictures, with fork-aware masks and a
  scratch that holds stale bytes where the pre-pass writes no image;
- the pre-pass images against the in-CTA prologue over several pictures and with masks;
- 32x32 borders whose strong-smoothing deviations sit at the threshold and one below it.
The replays of one test run in a few threads: the emulators release no shared state and ctypes drops the GIL."""
import ctypes as C
import os
import subprocess
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from _util import EDGE_SIZES, P, edge_content, i16p, oracle_rmd_frame, strong_filter_pus, threshold_picture, u8p, u32p

HERE = os.path.dirname(os.path.abspath(__file__))
COST_PRUNED, COST_NOT_INSIDE = np.uint32(0xFFFFFFFE), np.uint32(0xFFFFFFFF)
DEPTH_RANGES = [(0, 1), (1, 5), (5, 21), (21, 85), (85, 341)]     # PUs of each depth in a CTU's 341-entry table (N = 64 .. 4)
CTA_CTUS = [4, 4, 2, 2, 2]                                         # CTUs per CTA of the tensor-core kernels at each depth


def _pool():
    return ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1))


@pytest.fixture(scope="module")
def prep(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("prep_emul") / "librmd_tc2_prep_emul.so")
    csrc = os.path.join(os.path.dirname(HERE), "fast-cu-decision-hevc_b200", "csrc")
    subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-I" + csrc, "-o", so,
                    os.path.join(HERE, "emul", "rmd_tc2_prep_emul.cpp")], check=True, capture_output=True)
    lib = C.CDLL(so)
    lib.emul_tc2_prep_check.restype = C.c_longlong
    return lib


def _ctus(W, H):
    return ((W + 63) // 64) * ((H + 63) // 64)


# ---- the geometry list itself ----------------------------------------------------------------------------------------------------
def test_edge_sizes_cover_every_residue_and_small_pictures():
    for r in range(8, 64, 8):
        assert any(W % 64 == r and W > 64 for W, _ in EDGE_SIZES), r
        assert any(H % 64 == r and H > 64 for _, H in EDGE_SIZES), r
    assert any(W < 64 for W, _ in EDGE_SIZES) and any(H < 64 for _, H in EDGE_SIZES) and (8, 8) in EDGE_SIZES
    assert any(_ctus(W, H) % 2 == 1 and _ctus(W, H) > 1 for W, H in EDGE_SIZES)
    assert all(W % 8 == 0 and H % 8 == 0 for W, H in EDGE_SIZES)
    assert sum(_ctus(W, H) > 4 for W, H in EDGE_SIZES) == 0          # 2 x 2 CTUs or fewer: the replays stay cheap


# ---- availability ----------------------------------------------------------------------------------------------------------------
def _zscan_address(x, y, W):
    """MinTbAddrZs of the 4x4 unit holding sample (x, y) (HEVC 6.5.2 with one slice and one tile, CTB 64, min TB 4): CTBs in raster
    order, the 256 units of a CTB in z order"""
    ctb = (y // 64) * ((W + 63) // 64) + x // 64
    ux, uy, z = (x % 64) // 4, (y % 64) // 4, 0
    for b in range(4):
        z |= ((ux >> b) & 1) << (2 * b) | ((uy >> b) & 1) << (2 * b + 1)
    return ctb * 256 + z


def _available(xc, yc, xn, yn, W, H):
    """HEVC 6.4.1: a neighbour outside the picture, or later in z-scan order than the current block, is not available"""
    if xn < 0 or yn < 0 or xn >= W or yn >= H:
        return False
    return _zscan_address(xn, yn, W) < _zscan_address(xc, yc, W)


def _pus_inside(W, H):
    for d in range(5):
        n = 64 >> d
        for y0 in range(0, H - n + 1, n):
            for x0 in range(0, W - n + 1, n):
                yield n, x0, y0


def _check_availability(emul, oracle, W, H):
    """For every PU inside the picture: the oracle's bNeighborFlags (TComPattern.cpp:550-727) are HEVC 6.4.1 availability, and the
    available units are the prefix runs of tc2::pu_avail: the left column and its below-left extension from the top (lenL samples),
    the above row and its above-right extension from the left (lenT samples), and the corner (availC)"""
    out = (C.c_int * 3)()
    checked = 0
    cut = [0, 0]
    for n, x0, y0 in _pus_inside(W, H):
        half = n // 2
        flags = np.zeros(n + 1, np.uint8)
        oracle.oracle_neighbour_flags(x0, y0, n, W, H, P(flags, u8p))
        want = [_available(x0, y0, x0 - 1, y0 + (half - 1 - u) * 4, W, H) for u in range(half)]
        want += [_available(x0, y0, x0 - 1, y0 - 1, W, H)]
        want += [_available(x0, y0, x0 + u * 4, y0 - 1, W, H) for u in range(half)]
        assert flags.astype(bool).tolist() == want, (n, x0, y0)
        assert emul.emul_pu_avail(n.bit_length() - 1, x0, y0, W, H, out) == 0
        lenL, lenT, availC = out
        left = flags[:half][::-1]                    # top to bottom
        above = flags[half + 1:]
        assert left.tolist() == [int(k < lenL // 4) for k in range(half)], ("left", n, x0, y0, lenL)
        assert above.tolist() == [int(k < lenT // 4) for k in range(half)], ("above", n, x0, y0, lenT)
        assert int(flags[half]) == availC, ("corner", n, x0, y0)
        cut[0] += n // 4 < lenL // 4 < half          # a below-left run cut short by the picture's bottom edge
        cut[1] += n // 4 < lenT // 4 < half          # an above-right run cut short by the right edge
        checked += 1
    assert checked > 0
    return cut


@pytest.mark.parametrize("W,H", EDGE_SIZES)
def test_closed_form_availability_vs_per_unit_flags(emul, oracle, W, H):
    _check_availability(emul, oracle, W, H)


def test_edge_sizes_cut_the_extension_runs(emul, oracle):
    """the list holds PUs whose below-left run the bottom edge cuts short, and PUs whose above-right run the right edge cuts short"""
    cuts = np.array([_check_availability(emul, oracle, W, H) for W, H in EDGE_SIZES])
    assert (cuts[:, 0] > 0).sum() >= 3 and (cuts[:, 1] > 0).sum() >= 3


# ---- the replays over EDGE_SIZES ---------------------------------------------------------------------------------------------------
def _tc2(emul, strong, org, rec, need=None):
    H, W = org.shape
    got = np.zeros((_ctus(W, H), 341, 35), np.uint32)
    emul.emul_rmd_frame_tc2(strong, P(org, i16p), W, P(rec, i16p), W, W, H, P(got, u32p), None if need is None else P(need, u8p))
    return got


def _tc2_prep(emul, strong, orgs, recs, need=None, poison=0xC3, stride=None):
    """the replay of the GPU's frame path (pre-pass images + bulk copies) over the pictures orgs / recs, planes of `stride` samples"""
    n, H, W = orgs.shape
    S = stride or W
    o = np.zeros((n, H, S), np.int16); o[:, :, :W] = orgs
    r = np.zeros((n, H, S), np.int16); r[:, :, :W] = recs
    got = np.zeros((n * _ctus(W, H), 341, 35), np.uint32)
    emul.emul_rmd_frames_tc2_prep(strong, n, P(o, i16p), C.c_longlong(H * S), S, P(r, i16p), C.c_longlong(H * S), S, W, H, P(got, u32p),
                                  None if need is None else P(need, u8p), poison)
    return got


def _tc3(emul, bd, strong, org, rec):
    H, W = org.shape
    got = np.zeros((_ctus(W, H), 341, 35), np.uint32)
    emul.emul_rmd_frame_tc3(bd, strong, P(org, i16p), W, P(rec, i16p), W, W, H, P(got, u32p), None)
    return got


def _alu(emul, bd, strong, org, rec):
    H, W = org.shape
    got = np.zeros((_ctus(W, H), 341, 35), np.uint32)
    emul.emul_rmd_frame(bd, strong, P(org, i16p), W, P(rec, i16p), W, W, H, 0, got.shape[0], P(got, u32p))
    return got


def test_edge_content_fires_strong_smoothing_beside_cut_runs(oracle):
    """edge_content puts the strong filter next to a below-left run and next to an above-right run that the picture edge cuts short"""
    fired = [p for W, H in EDGE_SIZES for p in strong_filter_pus(oracle, *edge_content(W, H, 8, seed=W * 7 + H), 8)]
    assert any(8 < left < 16 for _, _, left, _ in fired)
    assert any(8 < above < 16 for _, _, _, above in fired)


@pytest.mark.parametrize("W,H", EDGE_SIZES)
def test_frame_replays_vs_oracle_at_edge_sizes(emul, oracle, W, H):
    """ALU (8 / 10 bit), tc2 (its prologue and the pre-pass images) and tc3 (8 / 9 / 10 bit), strong smoothing off and on"""
    runs = []
    for bd in (8, 9, 10):
        org, rec = edge_content(W, H, bd, seed=W * 7 + H)
        if W >= 32 and H >= 32:                        # a 32x32 PU fits: the strong filter changes its table
            assert strong_filter_pus(oracle, org, rec, bd), bd
        for strong in (0, 1):
            want = oracle_rmd_frame(oracle, org, rec, bd, strong)
            runs.append((("tc3", bd, strong), lambda o=org, r=rec, b=bd, s=strong: _tc3(emul, b, s, o, r), want))
            if bd != 9:
                runs.append((("alu", bd, strong), lambda o=org, r=rec, b=bd, s=strong: _alu(emul, b, s, o, r), want))
            if bd == 8:
                runs.append((("tc2", bd, strong), lambda o=org, r=rec, s=strong: _tc2(emul, s, o, r), want))
                runs.append((("tc2 images", bd, strong), lambda o=org, r=rec, s=strong: _tc2_prep(emul, s, o[None], r[None]), want))
    with _pool() as ex:
        futs = [(tag, ex.submit(fn), want) for tag, fn, want in runs]
        for tag, f, want in futs:
            assert np.array_equal(f.result(), want), tag


# ---- the tc2 replay of the GPU's frame path: several pictures, fork-aware masks, stale scratch ------------------------------------
def _expected(full, need):
    inside = full[:, :, 0] != COST_NOT_INSIDE
    return np.where(need.astype(bool)[:, :, None], full, np.where(inside[:, :, None], COST_PRUNED, COST_NOT_INSIDE))


def _skips_inside_live_ctas(full, need):
    """(CTU, depth) pairs that have no PU to evaluate (so no image) while another CTU of their CTA has one"""
    ev = (full[:, :, 0] != COST_NOT_INSIDE) & need.astype(bool)
    n = 0
    for d, (a, b) in enumerate(DEPTH_RANGES):
        live = ev[:, a:b].any(axis=1)
        k = CTA_CTUS[d]
        for cg in range(len(live)):
            unit = range(cg // k * k, min(len(live), cg // k * k + k))
            n += (not live[cg]) and any(live[c] for c in unit)
    return n


def _masks(full, seed):
    """random masks, the pattern of the fork-aware emulator test, and masks that prune a whole CTU at one depth while the other
    CTUs of its CTA are evaluated"""
    rng = np.random.default_rng(seed)
    nctu = full.shape[0]
    out = []
    for p in (0.5, 0.85):
        m = (rng.random((nctu, 341)) < p).astype(np.uint8)
        m[:, 85:] = np.repeat(m[:, 85::4], 4, axis=1)                 # 4x4 PUs: NxN of an 8x8 CU is pruned as a whole
        out.append(m)
    m = (rng.random((nctu, 341)) < 0.5).astype(np.uint8)
    m[:, 1:5] = 0
    m[:, 85:] = np.repeat(m[:, 85::4], 4, axis=1)
    out.append(m)
    for shift in (0, 1):
        m = np.ones((nctu, 341), np.uint8)
        for d, (a, b) in enumerate(DEPTH_RANGES):
            for cg in range(nctu):
                if cg % CTA_CTUS[d] == (d + shift) % CTA_CTUS[d]:
                    m[cg, a:b] = 0
        out.append(m)
    return out


def test_tc2_prepass_path_multi_picture_masks_and_stale_scratch(emul, oracle):
    """3 pictures of 3 CTUs (CTAs of 2 and 4 CTUs straddle the pictures): every picture against the oracle, without a mask and with
    masks; the image buffer starts as one poison byte or another, and the tables do not depend on it"""
    W, H = 136, 40
    assert _ctus(W, H) == 3
    pics = [edge_content(W, H, 8, seed=s) for s in (11, 12, 13)]
    orgs = np.stack([p[0] for p in pics]); recs = np.stack([p[1] for p in pics])
    full = np.concatenate([oracle_rmd_frame(oracle, o, r, 8) for o, r in pics])
    masks = _masks(full, 3)
    assert _skips_inside_live_ctas(full, masks[-1]) > 0 and _skips_inside_live_ctas(full, masks[-2]) > 0
    runs = [(None, 0x00), (None, 0xFF)] + [(m, p) for m in masks for p in (0x00, 0xFF)]
    with _pool() as ex:
        futs = [ex.submit(_tc2_prep, emul, 1, orgs, recs, m, p) for m, p in runs]
        got = [f.result() for f in futs]
    assert np.array_equal(got[0], full) and np.array_equal(got[1], full)
    for i, m in enumerate(masks):
        want = _expected(full, m)
        assert np.array_equal(got[2 + 2 * i], want), i
        assert np.array_equal(got[3 + 2 * i], want), i


def test_tc2_prepass_path_strided_planes(emul, oracle):
    """planes whose stride exceeds the picture width (W + 72 samples), 2 pictures"""
    W, H = 88, 104
    pics = [edge_content(W, H, 8, seed=s) for s in (21, 22)]
    got = _tc2_prep(emul, 1, np.stack([p[0] for p in pics]), np.stack([p[1] for p in pics]), stride=W + 72)
    assert np.array_equal(got, np.concatenate([oracle_rmd_frame(oracle, o, r, 8) for o, r in pics]))


# ---- the pre-pass images against the in-CTA prologue beyond one picture ------------------------------------------------------------
def _prep_check(prep, strong, recs, need=None):
    n, H, W = recs.shape
    recs = np.ascontiguousarray(recs)
    compared = C.c_longlong(0)
    bad = prep.emul_tc2_prep_check(strong, n, P(recs, i16p), C.c_longlong(H * W), W, W, H, None if need is None else P(need, u8p), C.byref(compared))
    return bad, compared.value


@pytest.mark.parametrize("W,H", EDGE_SIZES)
def test_prepass_images_match_prologue_at_edge_sizes(prep, W, H):
    recs = np.stack([edge_content(W, H, 8, seed=W + H + k)[1] for k in range(2)])
    for strong in (0, 1):
        bad, compared = _prep_check(prep, strong, recs)
        assert compared > 0 and bad == 0, strong


def test_prepass_images_match_prologue_multi_picture_with_masks(prep, oracle):
    W, H = 136, 40
    pics = [edge_content(W, H, 8, seed=s) for s in (11, 12, 13)]
    recs = np.stack([p[1] for p in pics])
    full = np.concatenate([oracle_rmd_frame(oracle, o, r, 8) for o, r in pics])
    for need in [None] + _masks(full, 4):
        bad, compared = _prep_check(prep, 1, recs, need)
        assert compared > 0 and bad == 0


# ---- strong smoothing at its threshold ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("bd", [8, 10])
def test_strong_smoothing_threshold_replays_vs_oracle(emul, oracle, bd):
    org, rec = threshold_picture(oracle, bd)
    want = oracle_rmd_frame(oracle, org, rec, bd, 1)
    assert not np.array_equal(want, oracle_rmd_frame(oracle, org, rec, bd, 0))
    runs = [("tc3", lambda: _tc3(emul, bd, 1, org, rec)), ("alu", lambda: _alu(emul, bd, 1, org, rec))]
    if bd == 8:
        runs += [("tc2", lambda: _tc2(emul, 1, org, rec)), ("tc2 images", lambda: _tc2_prep(emul, 1, org[None], rec[None]))]
    with _pool() as ex:
        futs = [(tag, ex.submit(fn)) for tag, fn in runs]
        for tag, f in futs:
            assert np.array_equal(f.result(), want), tag
