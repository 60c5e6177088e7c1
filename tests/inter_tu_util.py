"""Helpers of the cucd_inter_tu_* tests (transform, quantisation and distortion of inter residual quadtrees): the checker's loader and
its per-TU answers, and seeded residual batches.

tests/emul/libcucd_inter_tu_oracle.so - oracle/cucd_oracle.c plus tests/inter_tu_oracle.c, the checker of the inter TU chain
"""
import ctypes as C
import os
import subprocess

import numpy as np

from _util import ROOT, P, _newer, i16p, i32p


def load_inter_tu_oracle():
    """tests/inter_tu_oracle.c linked with the oracle it is composed from, as one library"""
    d = os.path.join(ROOT, "oracle")
    so = os.path.join(ROOT, "tests", "emul", "libcucd_inter_tu_oracle.so")
    srcs = [os.path.join(ROOT, "tests", "inter_tu_oracle.c"), os.path.join(d, "cucd_oracle.c"), os.path.join(d, "cucd_oracle.h")]
    if not _newer(so, srcs):
        subprocess.run(["gcc", "-O2", "-fPIC", "-std=c99", "-Wall", "-Wextra", "-ffp-contract=off", "-fno-fast-math", "-shared", "-I" + d, "-o", so,
                        srcs[0], srcs[1], "-lm"], check=True, capture_output=True)
    lib = C.CDLL(so)
    lib.oracle_sse.restype = C.c_uint32
    lib.oracle_quant.restype = C.c_int
    return lib


def oracle_inter_tu(lib, bd, n, qp, ts, chroma, sbh, stage, resi, level_in=None):
    """oracle_inter_tu on one n x n residual block: dict(coef, level, rresi, dist, dist_zero, abs_sum)"""
    resi = np.ascontiguousarray(resi, np.int16).reshape(n, n)
    coef = np.zeros(n * n, np.int32)
    level = np.zeros(n * n, np.int32) if level_in is None else np.ascontiguousarray(level_in, np.int32).ravel().copy()
    rresi = np.zeros(n * n, np.int16)
    dist, dist_zero, abs_sum = C.c_uint32(0), C.c_uint32(0), C.c_int32(0)
    lib.oracle_inter_tu(bd, n, int(qp), int(ts), int(chroma), int(sbh), stage, P(resi, i16p), n, P(coef, i32p), P(level, i32p), P(rresi, i16p),
                        C.byref(dist), C.byref(dist_zero), C.byref(abs_sum))
    return dict(coef=coef, level=level, rresi=rresi, dist=dist.value, dist_zero=dist_zero.value, abs_sum=abs_sum.value)


def oracle_sse(lib, bd, a, b):
    """oracle_sse of two equally shaped blocks"""
    a = np.ascontiguousarray(a, np.int16); b = np.ascontiguousarray(b, np.int16)
    h, w = a.shape if a.ndim == 2 else (1, a.size)
    return int(lib.oracle_sse(bd, P(a, i16p), w, P(b, i16p), w, w, h))


def random_residual(rng, n, bd, kind):
    """an n x n residual in [-(2^bd - 1), 2^bd - 1]: 0 full-range noise, 1 small noise (many zero levels), 2 the two extremes,
    3 a smooth ramp plus noise (what motion compensation leaves)"""
    hi = (1 << bd) - 1
    if kind == 0:
        r = rng.integers(-hi, hi + 1, (n, n))
    elif kind == 1:
        r = rng.integers(-3, 4, (n, n))
    elif kind == 2:
        r = rng.choice([-hi, hi], (n, n))
    else:
        y, x = np.mgrid[0:n, 0:n]
        r = (int(rng.integers(-hi // 4, hi // 4 + 1)) * (x + y) // (2 * n) + rng.integers(-hi // 16 - 1, hi // 16 + 2, (n, n)))
    return np.clip(r, -hi, hi).astype(np.int16)


def tu_golden_inter_records(g):
    """the records of a tests/golden/tu_*.npz file whose intra chain ran the DCT or transform skip (every record but luma 4x4 without
    transform skip), with resi = org - pred"""
    from _util import tu_records
    out = []
    for r in tu_records(g):
        if r["n"] == 4 and not r["chroma"] and not r["ts"]:
            continue
        r["resi"] = (np.asarray(r["org"], np.int32) - np.asarray(r["pred"], np.int32)).astype(np.int16).ravel()
        out.append(r)
    return out


def wrap_case(ito, seed=0):
    """levels of +-32767 at 32x32, 10 bit, and a residual of -+1023 against the sign of the rresi they give: the SSE passes 2^32"""
    bd, n = 10, 32
    level = np.random.default_rng(seed).choice([-32767, 32767], n * n).astype(np.int32)
    rresi = oracle_inter_tu(ito, bd, n, 51, 0, 0, 1, 2, np.zeros(n * n, np.int16), level_in=level)["rresi"]
    resi = np.where(rresi > 0, -1023, 1023).astype(np.int16)
    return level, resi
