"""Helpers of the cucd_me_tz_search tests (HM's TZ integer search and the refinement walk): loaders for the checker and the CPU replay,
TZ descriptors built the way xMotionEstimation builds its window and clip box, the checker's answers and an independent pure-Python
statement of the walk.

tests/emul/libcucd_me_tz_oracle.so - oracle/cucd_oracle.c, tests/me_search_oracle.c and tests/me_tz_oracle.c: the checker
tests/emul/libme_tz_emul.so        - tests/emul/me_tz_emul.cpp, the CPU replay of me_tz_kernel
"""
import ctypes as C
import os
import subprocess

import numpy as np

from _util import PKG, ROOT, P, _newer, i16p, i32p
from me_search_util import FRAC, HAD, LAMBDAS, MC_SHAPES, as_rows, lambda_cost, mc_scene, ref_base  # noqa: F401

TZ2N = 4
FIELDS = ("x", "y", "w", "h", "ref_idx", "left", "right", "top", "bottom", "sub_shift", "pred_x", "pred_y", "lambda", "flags", "search_range",
          "clip_left", "clip_right", "clip_top", "clip_bottom", "mv2n_x", "mv2n_y")


def load_me_tz_oracle():
    d = os.path.join(ROOT, "oracle")
    so = os.path.join(ROOT, "tests", "emul", "libcucd_me_tz_oracle.so")
    srcs = [os.path.join(ROOT, "tests", "me_tz_oracle.c"), os.path.join(ROOT, "tests", "me_search_oracle.c"), os.path.join(d, "cucd_oracle.c"),
            os.path.join(d, "cucd_oracle.h")]
    if not _newer(so, srcs):
        subprocess.run(["gcc", "-O2", "-fPIC", "-std=c99", "-Wall", "-Wextra", "-ffp-contract=off", "-fno-fast-math", "-shared", "-I" + d, "-o", so,
                        srcs[0], srcs[1], srcs[2], "-lm"], check=True, capture_output=True)
    lib = C.CDLL(so)
    lib.oracle_mv_cost.restype = C.c_uint32
    lib.oracle_mv_cost.argtypes = [C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.oracle_me_tz_search.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p] + [C.c_int] * 4 + [C.c_void_p, C.c_void_p,
                                                                                                                                         C.c_int, C.c_void_p]
    return lib


def load_me_tz_emul():
    d = os.path.join(ROOT, "tests", "emul")
    so = os.path.join(d, "libme_tz_emul.so")
    csrc = os.path.join(ROOT, PKG, "csrc")
    cpp = os.path.join(d, "me_tz_emul.cpp")
    srcs = [cpp] + [os.path.join(csrc, f) for f in ("rmd_core.cuh", "me_core.cuh")]
    if not _newer(so, srcs):
        subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-Wall", "-Wno-unknown-pragmas", "-I" + csrc, "-o", so, cpp], check=True, capture_output=True)
    lib = C.CDLL(so)
    lib.emul_me_tz_search.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    return lib


# ---------------------------------------------------------------------------------------------------
def clip_box(sc, x, y, w, h, frac=True):
    """the largest box whose blocks (with FRAC their 8-tap support) stay inside the padded planes: what HM's clipMv area with its
    80-sample margin gives, and what cucd_me_tz_search checks"""
    M, W, H = sc["M"], sc["W"], sc["H"]
    e = 4 if frac else 0
    f = 5 if frac else 0
    return (e - M - x, W - 1 + M - (w - 1) - f - x, e - M - y, H - 1 + M - (h - 1) - f - y)


def tz_desc(sc, x, y, w, h, ref_idx, pred, R, sub_shift=1, lam=0, flags=FRAC | HAD, mv2n=(0, 0), box=None):
    """xMotionEstimation's descriptor: box = the clip box; win = xSetSearchRange: the quarter-pel predictor clipped into the box,
    +- R samples, clipped again, >> 2"""
    cl, cr, ct, cb = box if box is not None else clip_box(sc, x, y, w, h, bool(flags & FRAC))
    px = min(max(int(pred[0]), 4 * cl), 4 * cr)
    py = min(max(int(pred[1]), 4 * ct), 4 * cb)
    left, right = max(px - 4 * R, 4 * cl) >> 2, min(px + 4 * R, 4 * cr) >> 2
    top, bottom = max(py - 4 * R, 4 * ct) >> 2, min(py + 4 * R, 4 * cb) >> 2
    return dict(x=x, y=y, w=w, h=h, ref_idx=ref_idx, left=left, right=right, top=top, bottom=bottom, sub_shift=sub_shift, pred_x=int(pred[0]),
                pred_y=int(pred[1]), flags=flags, search_range=R, clip_left=cl, clip_right=cr, clip_top=ct, clip_bottom=cb, mv2n_x=int(mv2n[0]),
                mv2n_y=int(mv2n[1]), **{"lambda": int(lam)})


def desc_row(d):
    """the 21 int32 of a cucd_tz_desc"""
    return np.array([(int(d[k]) & 0xFFFFFFFF) - (1 << 32) if k == "lambda" and int(d[k]) > 0x7FFFFFFF else int(d.get(k, 0)) for k in FIELDS], np.int32)


def src_block(sc, d):
    return np.ascontiguousarray(sc["org"][d["y"]:d["y"] + d["h"], d["x"]:d["x"] + d["w"]])


def oracle_tz(lib, sc, d, surface=None, trace_cap=0):
    """(res (6,) int64, trace (n, 6) int64 or None, probe count) of tests/me_tz_oracle.c for one PU.  surface: (array, left, top) to
    take the SADs from instead of the planes"""
    res = np.zeros(6, np.int32)
    tr = np.zeros((max(trace_cap, 1), 6), np.int32)
    n = C.c_int(0)
    row = desc_row(d)
    blk = src_block(sc, d) if "org" in sc else None
    if surface is not None:
        s, sl, st = surface
        s = np.ascontiguousarray(s, np.uint32)
        sarg, lims = s.ctypes.data, (sl, sl + s.shape[1] - 1, st, st + s.shape[0] - 1)
    else:
        sarg, lims = None, (0, 0, 0, 0)
    ref = ref_base(sc, d) if "refs" in sc else None
    stride = sc["refs"][d["ref_idx"]].shape[1] if "refs" in sc else 0
    rc = lib.oracle_me_tz_search(sc.get("bd", 8), None if blk is None else P(blk, i16p), d["w"], ref, stride, P(row, i32p), sarg, *lims, P(res, i32p),
                                 tr.ctypes.data if trace_cap else None, trace_cap, C.byref(n))
    if rc != 0:
        raise ValueError(f"oracle_me_tz_search returned {rc}")
    out = res.astype(np.int64)
    out[[2, 5]] = res[[2, 5]].view(np.uint32)
    trace = None
    if trace_cap:
        trace = tr[:min(n.value, trace_cap)].astype(np.int64)
        trace[:, 5] &= 0xFFFFFFFF
    return out, trace, n.value


def oracle_tz_rows(lib, sc, descs):
    """(n, 6) int64 checker results"""
    return np.stack([oracle_tz(lib, sc, d)[0] for d in descs]) if descs else np.zeros((0, 6), np.int64)


def emul_tz(emul, sc, d, cap=200000):
    """(res (6,) int64, trace (n, 6) int64, points evaluated, lanes per probe) of the CPU replay of me_tz_kernel for one PU: the integer
    result and the points of every folded segment"""
    res = np.zeros(6, np.int32)
    tr = np.zeros((cap, 6), np.int32)
    ev, lanes = np.zeros(1, np.int32), np.zeros(1, np.int32)
    blk = src_block(sc, d)
    row = desc_row(d)
    n = emul.emul_me_tz_search(sc["bd"], P(blk, i16p), d["w"], ref_base(sc, d), sc["refs"][d["ref_idx"]].shape[1], P(row, i32p), P(res, i32p), tr.ctypes.data,
                               cap, ev.ctypes.data, lanes.ctypes.data)
    assert 0 <= n <= cap
    out = res.astype(np.int64)
    out[2] = int(res[2]) & 0xFFFFFFFF
    t = tr[:n].astype(np.int64)
    t[:, 5] &= 0xFFFFFFFF
    return out, t, int(ev[0]), int(lanes[0])


# ---- an independent statement of the walk --------------------------------------------------------------------------------------
def py_bits(v):
    t = -2 * v + 1 if v <= 0 else 2 * v
    return 2 * (t.bit_length() - 1) + 1


def py_cost(d, x, y):
    return ((int(d["lambda"]) & 0xFFFFFFFF) * (py_bits(4 * x - d["pred_x"]) + py_bits(4 * y - d["pred_y"])) & 0xFFFFFFFF) >> 16


def _diamond_points(D):
    """(dx, dy, p, d) of xTZ8PointDiamondSearch in HM's order"""
    if D == 1:
        return [(0, -1, 2, 1), (-1, 0, 4, 1), (1, 0, 5, 1), (0, 1, 7, 1)]
    if D <= 8:
        h = D // 2
        return [(0, -D, 2, D), (-h, -h, 1, h), (h, -h, 3, h), (-D, 0, 4, D), (D, 0, 5, D), (-h, h, 6, h), (h, h, 8, h), (0, D, 7, D)]
    q = D // 4
    pts = [(0, -D, 0, D), (-D, 0, 0, D), (D, 0, 0, D), (0, D, 0, D)]
    for k in (1, 2, 3):
        pts += [(-q * k, -D + q * k, 0, D), (q * k, -D + q * k, 0, D), (-q * k, D - q * k, 0, D), (q * k, D - q * k, 0, D)]
    return pts


TWO_POINT = {1: [(-1, 0), (0, -1)], 2: [(-1, -1), (1, -1)], 3: [(0, -1), (1, 0)], 4: [(-1, 1), (-1, -1)], 5: [(1, -1), (1, 1)], 6: [(-1, 0), (0, 1)],
             7: [(-1, 1), (1, 1)], 8: [(1, 0), (0, 1)]}


def py_tz_walk(d, sad):
    """the walk of include/cucudecide.h, probe by probe: sad(x, y) gives the SAD.  Returns ((mvx, mvy, sad), trace of (x, y, p, d, stage,
    c)) with the checker's stage numbers"""
    win = (d["left"], d["right"], d["top"], d["bottom"])
    box = (d["clip_left"], d["clip_right"], d["clip_top"], d["clip_bottom"])
    R = d["search_range"]
    s = dict(best=(1 << 32) - 1, b=(0, 0), dist=0, round=0, pt=0, stage=0)
    trace = []

    def probe(x, y, p, dd):
        c = (sad(x, y) + py_cost(d, x, y)) & 0xFFFFFFFF
        trace.append((x, y, p, dd, s["stage"], c))
        if c < s["best"]:
            s.update(best=c, b=(x, y), dist=dd, round=0, pt=p)

    def inside(cx, cy, dx, dy):
        x, y = cx + dx, cy + dy
        return (dx >= 0 or x >= win[0]) and (dx <= 0 or x <= win[1]) and (dy >= 0 or y >= win[2]) and (dy <= 0 or y <= win[3])

    def diamond(c, D):
        s["round"] += 1
        for dx, dy, p, dd in _diamond_points(D):
            if inside(c[0], c[1], dx, dy):
                probe(c[0] + dx, c[1] + dy, p, dd)

    def two_point():
        c = s["b"]
        for dx, dy in TWO_POINT.get(s["pt"], []):
            if inside(c[0], c[1], dx, dy):
                probe(c[0] + dx, c[1] + dy, 0, 2)

    def clamp(v, lo, hi):
        return min(max(v, lo), hi)

    dists = []
    D = 1
    while D <= R:
        dists.append(D)
        D *= 2
    probe(clamp(d["pred_x"], 4 * box[0], 4 * box[1]) >> 2, clamp(d["pred_y"], 4 * box[2], 4 * box[3]) >> 2, 0, 0)
    probe(0, 0, 0, 0)
    rwin = win
    if d["flags"] & TZ2N:
        probe(clamp(d.get("mv2n_x", 0), box[0], box[1]), clamp(d.get("mv2n_y", 0), box[2], box[3]), 0, 0)
        bx, by = s["b"]
        rwin = (clamp(bx - R, box[0], box[1]), clamp(bx + R, box[0], box[1]), clamp(by - R, box[2], box[3]), clamp(by + R, box[2], box[3]))
    s["stage"] = 1
    c = s["b"]
    for D in dists:
        diamond(c, D)
        if s["round"] >= 3:
            break
    if s["dist"] == 1:
        s["dist"] = 0
        s["stage"] = 2
        two_point()
    if s["dist"] > 5:
        s["dist"] = 5
        s["stage"] = 3
        for y in range(rwin[2], rwin[3] + 1, 5):
            for x in range(rwin[0], rwin[1] + 1, 5):
                probe(x, y, 0, 5)
    star = 0
    while s["dist"] > 0:
        c = s["b"]
        s.update(dist=0, pt=0, stage=4 + 2 * star)
        for D in dists:
            diamond(c, D)
        if s["dist"] == 1:
            s["dist"] = 0
            s["stage"] = 5 + 2 * star
            if s["pt"] != 0:
                two_point()
        star += 1
    bx, by = s["b"]
    return (bx, by, (s["best"] - py_cost(d, bx, by)) & 0xFFFFFFFF), trace


def surface_sad(surface, left, top):
    """sad(x, y) over a (rows, cols) array whose entry (0, 0) is mv (left, top)"""
    return lambda x, y: int(surface[y - top, x - left])
