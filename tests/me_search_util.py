"""Helpers of the cucd_me_search tests (full-search motion estimation and the sub-pel refinement walk): loaders for the checker and the
CPU replay, search descriptors, the checker's answers and an independent numpy statement of the search.

tests/emul/libcucd_me_search_oracle.so - oracle/cucd_oracle.c plus tests/me_search_oracle.c, the checker of the motion search
tests/emul/libme_search_emul.so        - tests/emul/me_search_emul.cpp, the CPU replay of the search phases
"""
import ctypes as C
import os
import subprocess

import numpy as np

from _util import PKG, ROOT, P, _newer, i16p, i32p, u32p
from mc_util import MC_SHAPES, mc_scene  # noqa: F401  (the scene and PU shapes of the motion-compensation tests)

FRAC, HAD = 1, 2
HM_H = [(0, 0), (0, -1), (0, 1), (-1, 0), (1, 0), (-1, -1), (1, -1), (-1, 1), (1, 1)]
HM_Q = [(0, 0), (0, -1), (0, 1), (-1, -1), (1, -1), (-1, 0), (1, 0), (-1, 1), (1, 1)]


def lambda_cost(qp):
    """m_uiCost = floor(65536 sqrt(lambda)) with HM's lambda = 0.57 2^((QP - 12) / 3)"""
    return int(np.floor(65536.0 * np.sqrt(0.57 * 2.0 ** ((qp - 12) / 3.0))))


LAMBDAS = (0, lambda_cost(22), lambda_cost(37), 0xFFFFFFFF)


def load_me_search_oracle():
    d = os.path.join(ROOT, "oracle")
    so = os.path.join(ROOT, "tests", "emul", "libcucd_me_search_oracle.so")
    srcs = [os.path.join(ROOT, "tests", "me_search_oracle.c"), os.path.join(d, "cucd_oracle.c"), os.path.join(d, "cucd_oracle.h")]
    if not _newer(so, srcs):
        subprocess.run(["gcc", "-O2", "-fPIC", "-std=c99", "-Wall", "-Wextra", "-ffp-contract=off", "-fno-fast-math", "-shared", "-I" + d, "-o", so,
                        srcs[0], srcs[1], "-lm"], check=True, capture_output=True)
    lib = C.CDLL(so)
    lib.oracle_mv_bits.restype = C.c_uint32
    lib.oracle_mv_cost.restype = C.c_uint32
    lib.oracle_mv_cost.argtypes = [C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.oracle_me_frac_walk.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_void_p, C.c_void_p]
    lib.oracle_me_search.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int] + [C.c_int] * 7 + [C.c_uint32, C.c_int, C.c_void_p]
    return lib


def load_me_search_emul():
    d = os.path.join(ROOT, "tests", "emul")
    so = os.path.join(d, "libme_search_emul.so")
    csrc = os.path.join(ROOT, PKG, "csrc")
    cpp = os.path.join(d, "me_search_emul.cpp")
    srcs = [cpp] + [os.path.join(csrc, f) for f in ("rmd_core.cuh", "me_core.cuh")]
    if not _newer(so, srcs):
        subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-Wall", "-Wno-unknown-pragmas", "-I" + csrc, "-o", so, cpp], check=True, capture_output=True)
    lib = C.CDLL(so)
    lib.emul_me_search_key.restype = C.c_uint64
    lib.emul_me_search_key.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int] + [C.c_int] * 7 + [C.c_void_p, C.c_uint32, C.c_int,
                                                                                                                              C.c_int, C.c_void_p]
    lib.emul_me_search_walk.argtypes = [C.c_void_p, C.c_uint32, C.c_int, C.c_int, C.c_void_p]
    lib.emul_me_search_prep.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    return lib


# ---------------------------------------------------------------------------------------------------
def window_limits(sc, x, y, w, h, frac=True):
    """least left / top and largest right / bottom whose support stays inside the padded planes: the 8-tap support of cucd_me_search's
    FRAC rule (x + left - 4 >= -M, x + right + w + 4 <= W - 1 + M), else the integer window alone"""
    M, W, H = sc["M"], sc["W"], sc["H"]
    e = 4 if frac else 0
    return (e - M - x, W - 1 + M - w - e - x, e - M - y, H - 1 + M - h - e - y)


def search_desc(sc, x, y, w, h, ref_idx, cx, cy, R, sub_shift=1, pred=(0, 0), lam=0, flags=FRAC | HAD):
    """a +-R window around (cx, cy), clipped like xSetSearchRange: the centre clipped into the legal range (clipMv), then the window"""
    lo_x, hi_x, lo_y, hi_y = window_limits(sc, x, y, w, h, bool(flags & FRAC))
    cx, cy = min(max(cx, lo_x), hi_x), min(max(cy, lo_y), hi_y)
    return dict(x=x, y=y, w=w, h=h, ref_idx=ref_idx, left=max(cx - R, lo_x), right=min(cx + R, hi_x), top=max(cy - R, lo_y), bottom=min(cy + R, hi_y),
                sub_shift=sub_shift, pred_x=int(pred[0]), pred_y=int(pred[1]), **{"lambda": int(lam)}, flags=flags)


def search_descs(sc, rng, shapes=MC_SHAPES, radii=(64, 4, 0), flag_sets=(FRAC | HAD, FRAC, 0), lambdas=LAMBDAS, corners=True):
    """per shape, radius and flag set one PU with a random position, window centre, predictor and lambda; with corners every third
    PU sits at a picture corner with its window centre pushed beyond the margin, so that the window is clipped"""
    W, H = sc["W"], sc["H"]
    slots = sc["slots"]
    out = []
    for w, h in shapes:
        for R in radii:
            for fl in flag_sets:
                n = len(out)
                if corners and n % 3 == 2:
                    x, y = [(0, 0), (W - w, 0), (0, H - h), (W - w, H - h)][n // 3 % 4]
                    cx = -200 if x == 0 else 200
                    cy = -200 if y == 0 else 200
                else:
                    x = int(rng.integers(0, (W - w) // 4 + 1)) * 4
                    y = int(rng.integers(0, (H - h) // 4 + 1)) * 4
                    cx, cy = int(rng.integers(-12, 13)), int(rng.integers(-12, 13))
                pred = (int(rng.integers(-32768, 32768)), int(rng.integers(-32768, 32768))) if rng.random() < 0.3 else (4 * cx + int(rng.integers(-9, 10)),
                                                                                                                       4 * cy + int(rng.integers(-9, 10)))
                lam = int(lambdas[n % len(lambdas)])
                d = search_desc(sc, x, y, w, h, slots[n % len(slots)], cx, cy, R, sub_shift=int(rng.integers(0, 2)), pred=pred, lam=lam, flags=fl)
                if d["left"] > d["right"] or d["top"] > d["bottom"]:
                    continue
                out.append(d)
    return out


def ref_base(sc, d):
    """pointer to the co-located sample (mv 0) of the PU in its padded reference plane"""
    p, M = sc["refs"][d["ref_idx"]], sc["M"]
    return C.c_void_p(p.ctypes.data + 2 * ((d["y"] + M) * p.shape[1] + d["x"] + M))


def src_blocks(sc, descs, src=None):
    """the source block of every PU: its own block of `src` (back to back) or the block of the current picture"""
    out, off = [], 0
    for d in descs:
        if src is None:
            out.append(np.ascontiguousarray(sc["org"][d["y"]:d["y"] + d["h"], d["x"]:d["x"] + d["w"]]))
        else:
            out.append(np.ascontiguousarray(src[off:off + d["w"] * d["h"]].reshape(d["h"], d["w"])))
        off += d["w"] * d["h"]
    return out


def eff_sub_shift(d):
    """the generic xGetSAD (widths outside HM's list) ignores iSubShift, as cucd_me_sad_surface does"""
    return d["sub_shift"] if d["w"] in (4, 8, 12, 16, 24, 32, 48, 64) else 0


def oracle_search(lib, sc, descs, src=None):
    """(n, 6) int64: mvx, mvy, sad, qmvx, qmvy, frac_cost of tests/me_search_oracle.c oracle_me_search"""
    res = np.zeros((len(descs), 6), np.int32)
    for i, (d, blk) in enumerate(zip(descs, src_blocks(sc, descs, src))):
        r = np.zeros(6, np.int32)
        rc = lib.oracle_me_search(sc["bd"], P(blk, i16p), d["w"], d["w"], d["h"], ref_base(sc, d), sc["refs"][d["ref_idx"]].shape[1], d["left"], d["right"],
                                  d["top"], d["bottom"], eff_sub_shift(d), d["pred_x"], d["pred_y"], d["lambda"] & 0xFFFFFFFF, d["flags"], P(r, i32p))
        assert rc == 0
        res[i] = r
    out = res.astype(np.int64)
    out[:, [2, 5]] = res[:, [2, 5]].view(np.uint32).astype(np.int64)
    return out


def oracle_surface(oracle, sc, d, blk):
    cols, rows = d["right"] - d["left"] + 1, d["bottom"] - d["top"] + 1
    s = np.zeros((rows, cols), np.uint32)
    oracle.oracle_sad_surface(sc["bd"], P(blk, i16p), d["w"], d["w"], d["h"], ref_base(sc, d), sc["refs"][d["ref_idx"]].shape[1], d["left"], d["right"],
                              d["top"], d["bottom"], eff_sub_shift(d), P(s, u32p))
    return s


def oracle_table(oracle, sc, d, blk, mvx, mvy, had):
    t = np.zeros(49, np.uint32)
    oracle.oracle_subpel_surface(sc["bd"], P(blk, i16p), d["w"], d["w"], d["h"], ref_base(sc, d), sc["refs"][d["ref_idx"]].shape[1], mvx, mvy, had, P(t, u32p))
    return t


# ---- an independent numpy statement ---------------------------------------------------------------
def np_bits(v):
    """xGetComponentBits, closed form: 1 + 2 floor(log2 t)"""
    v = np.asarray(v, np.int64)
    t = np.where(v <= 0, -2 * v + 1, 2 * v)
    return 1 + 2 * (np.floor(np.log2(t.astype(np.float64))).astype(np.int64))


def np_cost(lam, x, y, s, px, py):
    return ((np.uint64(lam) * (np_bits(np.asarray(x, np.int64) * (1 << s) - px) + np_bits(np.asarray(y, np.int64) * (1 << s) - py)).astype(np.uint64))
            & np.uint64(0xFFFFFFFF)) >> np.uint64(16)


def np_integer_search(surface, d):
    """lexicographic argmin over (sad + cost_2, raster index): (mvx, mvy, sad)"""
    rows, cols = surface.shape
    ys, xs = np.mgrid[d["top"]:d["bottom"] + 1, d["left"]:d["right"] + 1]
    c = surface.astype(np.uint64) + np_cost(d["lambda"], xs, ys, 2, d["pred_x"], d["pred_y"])
    order = np.lexsort((np.arange(rows * cols), c.ravel()))
    k = int(order[0])
    return d["left"] + k % cols, d["top"] + k // cols, int(surface.ravel()[k])


def np_walk(T, mvx, mvy, d):
    """the two 9-point stages: (qmvx, qmvy, frac_cost)"""
    T = np.asarray(T, np.uint64).ravel()
    hd = [int((T[(2 * hy + 3) * 7 + 2 * hx + 3] + np_cost(d["lambda"], 2 * mvx + hx, 2 * mvy + hy, 1, d["pred_x"], d["pred_y"])) & 0xFFFFFFFF) for hx, hy in HM_H]
    bx, by = HM_H[int(np.argmin(hd))]                   # argmin returns the first of equal minima
    qd = [int((T[(2 * by + qy + 3) * 7 + 2 * bx + qx + 3] + np_cost(d["lambda"], 4 * mvx + 2 * bx + qx, 4 * mvy + 2 * by + qy, 0, d["pred_x"], d["pred_y"]))
              & 0xFFFFFFFF) for qx, qy in HM_Q]
    q = int(np.argmin(qd))
    return 4 * mvx + 2 * bx + HM_Q[q][0], 4 * mvy + 2 * by + HM_Q[q][1], qd[q]


def np_search(oracle, sc, descs, src=None):
    """the search stated with numpy on the oracle's surfaces and tables: (n, 6) int64"""
    out = np.zeros((len(descs), 6), np.int64)
    for i, (d, blk) in enumerate(zip(descs, src_blocks(sc, descs, src))):
        mvx, mvy, sad = np_integer_search(oracle_surface(oracle, sc, d, blk), d)
        q = (4 * mvx, 4 * mvy, 0)
        if d["flags"] & FRAC:
            q = np_walk(oracle_table(oracle, sc, d, blk, mvx, mvy, 1 if d["flags"] & HAD else 0), mvx, mvy, d)
        out[i] = (mvx, mvy, sad, *q)
    return out


def walk_batch(T, mv, pred, lam):
    """np_walk for many PUs at once: T (n, 49) uint32, mv (n, 2), pred (n, 2), lam scalar"""
    n = T.shape[0]
    idx = np.arange(n)
    best = np.full(n, np.iinfo(np.int64).max, np.int64)
    hb = np.zeros((n, 2), np.int64)
    for hx, hy in HM_H:
        d = (T[:, (2 * hy + 3) * 7 + 2 * hx + 3].astype(np.uint64) + np_cost(lam, 2 * mv[:, 0] + hx, 2 * mv[:, 1] + hy, 1, pred[:, 0], pred[:, 1])) & 0xFFFFFFFF
        d = d.astype(np.int64)
        take = d < best
        best = np.where(take, d, best)
        hb[take] = (hx, hy)
    best[:] = np.iinfo(np.int64).max
    qb = np.zeros((n, 2), np.int64)
    for qx, qy in HM_Q:
        d = (T[idx, (2 * hb[:, 1] + qy + 3) * 7 + 2 * hb[:, 0] + qx + 3].astype(np.uint64)
             + np_cost(lam, 4 * mv[:, 0] + 2 * hb[:, 0] + qx, 4 * mv[:, 1] + 2 * hb[:, 1] + qy, 0, pred[:, 0], pred[:, 1])) & 0xFFFFFFFF
        d = d.astype(np.int64)
        take = d < best
        best = np.where(take, d, best)
        qb[take] = (qx, qy)
    return 4 * mv + 2 * hb + qb, best


def as_rows(res):
    """a SEARCH_RESULT array as (n, 6) int64"""
    return np.stack([res[k].astype(np.int64) for k in ("mvx", "mvy", "sad", "qmvx", "qmvy", "frac_cost")], axis=1)
