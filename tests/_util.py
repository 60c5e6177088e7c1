"""Shared helpers of the test-suite: loaders for the checker libraries and seeded synthetic content.

oracle/libcucd_oracle.so  - the plain-C restatement (the checker)
oracle/_ref/libhmref.so   - the reference's own compiled functions (only where it was built)
tests/emul/librmd_emul.so - CPU replay of the CUDA kernels' per-thread code
"""
import ctypes as C
import importlib
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
PKG = "fast-cu-decision-hevc_b200"

i16p = C.POINTER(C.c_int16)
i32p = C.POINTER(C.c_int32)
u8p = C.POINTER(C.c_uint8)
u32p = C.POINTER(C.c_uint32)
f64p = C.POINTER(C.c_double)


def P(a, t):
    return a.ctypes.data_as(t)


def _newer(target, sources):
    if not os.path.exists(target):
        return False
    t = os.path.getmtime(target)
    return all(os.path.getmtime(s) <= t for s in sources)


def load_oracle():
    d = os.path.join(ROOT, "oracle")
    so = os.path.join(d, "libcucd_oracle.so")
    if not _newer(so, [os.path.join(d, "cucd_oracle.c"), os.path.join(d, "cucd_oracle.h")]):
        subprocess.run(["make", "-C", d, "libcucd_oracle.so"], check=True, capture_output=True)
    lib = C.CDLL(so)
    lib.oracle_satd.restype = C.c_uint32
    lib.oracle_sad.restype = C.c_uint32
    lib.oracle_tcm_yc.restype = C.c_double
    lib.oracle_aq_activity.restype = C.c_double
    return lib


def load_hmref():
    so = os.path.join(ROOT, "oracle", "_ref", "libhmref.so")
    if not os.path.exists(so):
        return None
    lib = C.CDLL(so)
    lib.hmref_hads.restype = C.c_uint32
    lib.hmref_sad.restype = C.c_uint32
    lib.hmref_init(8)
    return lib


def load_emul():
    d = os.path.join(ROOT, "tests", "emul")
    so = os.path.join(d, "librmd_emul.so")
    csrc = os.path.join(ROOT, PKG, "csrc")
    cpps = [os.path.join(d, "rmd_emul.cpp"), os.path.join(d, "rmd_tc2_emul.cpp"), os.path.join(d, "rmd_tc3_emul.cpp"), os.path.join(d, "me_emul.cpp")]
    srcs = cpps + [os.path.join(d, "tc2_prep_replay.h")] + [os.path.join(csrc, f) for f in ("rmd_core.cuh", "rmd_chunk.cuh", "rmd_tc2.cuh", "rmd_tc3.cuh", "rmd_tc_frame.cuh", "feature_core.cuh", "me_core.cuh")]
    if not _newer(so, srcs):
        subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-I" + csrc, "-o", so] + cpps,
                       check=True, capture_output=True)
    return C.CDLL(so)


def load_package():
    return importlib.import_module(PKG)


def golden(name):
    return np.load(os.path.join(GOLDEN, name))


# ---------------------------------------------------------------------------------------------------
# seeded synthetic content
# ---------------------------------------------------------------------------------------------------
def textured_plane(W, H, bit_depth=8, seed=20261018, t=0):
    """The "textured motion" luma of SURVEY.md 8d: 8x8-blocky random texture translated (2,1) px per
    frame + two low-frequency sinusoids + uniform noise, clipped; scaled for >8 bit."""
    rng = np.random.default_rng(seed)
    field = rng.integers(0, 256, (H // 8 + 2 + 16, W // 8 + 2 + 32)).astype(np.float64)
    tex = np.kron(field, np.ones((8, 8)))[t: t + H, 2 * t: 2 * t + W]
    x = np.arange(W)[None, :]
    y = np.arange(H)[:, None]
    noise = np.random.default_rng(seed + 1000 + t).uniform(-6, 6, (H, W))
    Y = 0.6 * tex + 30 + 20 * np.sin((x + 3 * t) / 37.0) + 15 * np.cos((y - 2 * t) / 29.0) + noise
    Y = np.clip(np.rint(Y), 0, 255).astype(np.int64)
    if bit_depth > 8:
        sh = bit_depth - 8
        Y = (Y << sh) + np.random.default_rng(seed + 2000 + t).integers(0, 1 << sh, (H, W))
    return Y.astype(np.int16)


def full_range_keys(rng, shape):
    """caller-supplied source keys from all of int16 (the `_src` calls accept any value): uniform samples with runs of -32768 and of
    32767 along the last axis.  Against a reference sample r, a key k gives |k - r| up to 65535, beyond the int16 range of a half-word"""
    k = rng.integers(-32768, 32768, shape)
    flat = k.reshape(-1)
    for v in (-32768, 32767):
        for s in rng.integers(0, flat.size, max(1, flat.size // 64)):
            flat[s:s + int(rng.integers(4, 40))] = v
    return k.astype(np.int16)


def pseudo_recon(org, bit_depth=8, seed=7):
    """A stand-in reconstruction: the source low-passed a little plus small noise (what a codec's
    reconstruction looks like statistically), so that borders differ from the source."""
    o = org.astype(np.int32)
    pad = np.pad(o, 1, mode="edge")
    blur = (pad[:-2, 1:-1] + pad[2:, 1:-1] + pad[1:-1, :-2] + pad[1:-1, 2:] + 4 * o + 4) >> 3
    noise = np.random.default_rng(seed).integers(-2, 3, o.shape)
    return np.clip(blur + noise, 0, (1 << bit_depth) - 1).astype(np.int16)


def oracle_rmd_frame(lib, org, rec, bit_depth, strong=1, ctu_begin=0, ctu_end=None):
    H, W = org.shape
    nctu = ((W + 63) // 64) * ((H + 63) // 64)
    if ctu_end is None:
        ctu_end = nctu
    org = np.ascontiguousarray(org)
    rec = np.ascontiguousarray(rec)
    out = np.zeros((ctu_end - ctu_begin, 341, 35), np.uint32)
    lib.oracle_rmd_frame(bit_depth, strong, P(org, i16p), W, P(rec, i16p), W, W, H, ctu_begin, ctu_end, P(out, u32p))
    return out


def oracle_outlier_frame(lib, org, bit_depth):
    H, W = org.shape
    org = np.ascontiguousarray(org)
    obf = np.zeros((H // 4, W // 4), np.int16)
    outl = np.zeros((H, W), np.int16)
    yc = np.zeros(16, np.float64)
    lib.oracle_outlier_frame(bit_depth, P(org, i16p), W, W, H, P(obf, i16p), P(outl, i16p), P(yc, f64p))
    return obf, outl, yc


def oracle_cu_sums(lib, obf, W, H, depth):
    s = 64 >> depth
    a = np.zeros((H // s, W // s), np.int32)
    b = np.zeros((H // s, W // s), np.int32)
    obf = np.ascontiguousarray(obf)
    if a.size:
        lib.oracle_cu_sums(P(obf, i16p), W, H, depth, P(a, i32p), P(b, i32p))
    return a, b


def oracle_ctu_src_had(lib, org):
    H, W = org.shape
    org = np.ascontiguousarray(org)
    out = np.zeros(((W + 63) // 64) * ((H + 63) // 64), np.int32)
    lib.oracle_ctu_src_had(P(org, i16p), W, W, H, P(out, i32p))
    return out


def oracle_tmv_features(lib, org, cus):
    """cus: (x, y, log2_size) -> (nCU, 5, 26) float64 of oracle_tmv_features."""
    H, W = org.shape
    org = np.ascontiguousarray(org)
    out = np.zeros((len(cus), 5, 26), np.float64)
    for i, (x, y, l) in enumerate(cus):
        lib.oracle_tmv_features(C.c_void_p(org.ctypes.data + 2 * (y * W + x)), W, 1 << l, C.c_void_p(out[i].ctypes.data))
    return out


def oracle_aq_activity(lib, org, max_aq_depth):
    H, W = org.shape
    org = np.ascontiguousarray(org)
    acts, avg = [], np.zeros(max_aq_depth, np.float64)
    for d in range(max_aq_depth):
        u = 64 >> d
        a = np.zeros(((H + u - 1) // u, (W + u - 1) // u), np.float64)
        avg[d] = lib.oracle_aq_activity(P(org, i16p), W, W, H, u, P(a, f64p))
        acts.append(a)
    return acts, avg


def all_cus(W, H, depths=(0, 1, 2, 3)):
    """every whole CU of the picture at the given depths as (x, y, log2_size)"""
    out = []
    for d in depths:
        n = 64 >> d
        out += [(x, y, 6 - d) for y in range(0, H - n + 1, n) for x in range(0, W - n + 1, n)]
    return out


def oracle_intra_tu(lib, bd, n, mode, qp, ts, org, border, stage, strong=1, intra=1, sbh=1, level_in=None, chroma=0):
    """oracle_intra_tu on one TU: returns dict(coef, level, pred, reco, dist, abs_sum)."""
    org = np.ascontiguousarray(org, np.int16)
    border = np.ascontiguousarray(border, np.int16)
    coef = np.zeros(n * n, np.int32)
    level = np.zeros(n * n, np.int32) if level_in is None else np.ascontiguousarray(level_in, np.int32).copy()
    pred = np.zeros(n * n, np.int16)
    reco = np.zeros(n * n, np.int16)
    dist = C.c_uint32(0)
    abs_sum = C.c_int32(0)
    lib.oracle_intra_tu_c(bd, n, int(mode), int(qp), int(ts), int(chroma), strong, intra, sbh, stage, P(org, i16p), n, P(border, i16p), P(coef, i32p), P(level, i32p),
                        P(pred, i16p), P(reco, i16p), C.byref(dist), C.byref(abs_sum))
    return dict(coef=coef, level=level, pred=pred, reco=reco, dist=dist.value, abs_sum=abs_sum.value)


TU_HDR = ("poc", "x", "y", "mode", "bd", "ts", "load", "qp", "intra", "sbh", "rdoq", "abs_sum", "dist", "comp")


def tu_records(g):
    """iterate the records of a tests/golden/tu_*.npz file as dicts"""
    for tag in sorted(k[:-4] for k in g.files if k.endswith("_hdr")):
        n = int(tag[1:].rstrip("ts"))
        for i, h in enumerate(g[tag + "_hdr"]):
            r = dict(zip(TU_HDR, (int(v) for v in h)))
            r["n"] = n
            r["chroma"] = int(tag[0] == "c")
            for k in ("border", "org", "pred", "coef", "level", "reco"):
                r[k] = g[tag + "_" + k][i]
            yield r


def frac_records(g):
    """iterate tests/golden/frac_*.npz: dict(w, h, bd, had, qx, qy, dist, org (h,w), win (h+9, w+9) with origin at (-4,-4))"""
    oo = wo = 0
    for w, h, bd, had, qx, qy, dist in g["hdr"]:
        w, h = int(w), int(h)
        org = g["org"][oo:oo + w * h].reshape(h, w); oo += w * h
        win = g["win"][wo:wo + (w + 9) * (h + 9)].reshape(h + 9, w + 9); wo += (w + 9) * (h + 9)
        yield dict(w=w, h=h, bd=int(bd), had=int(had), qx=int(qx), qy=int(qy), dist=int(dist) & 0xFFFFFFFF, org=org, win=win)


def pu_table_index(x, y, n):
    """index of the PU at picture position (x, y) of size n inside its CTU's 341-entry cost table (depth-major, z-order)"""
    d = {64: 0, 32: 1, 16: 2, 8: 3, 4: 4}[n]
    px, py, z = (x % 64) // n, (y % 64) // n, 0
    for b in range(4):
        z |= ((px >> b) & 1) << (2 * b) | ((py >> b) & 1) << (2 * b + 1)
    return (0, 1, 5, 21, 85)[d] + z


def oracle_prune_mask(lib, obf, W, H, skip, term):
    obf = np.ascontiguousarray(obf, np.int16); skip = np.ascontiguousarray(skip, np.uint8); term = np.ascontiguousarray(term, np.uint8)
    need = np.zeros((((W + 63) // 64) * ((H + 63) // 64), 341), np.uint8)
    lib.oracle_prune_mask(C.c_void_p(obf.ctypes.data), W, H, C.c_void_p(skip.ctypes.data), C.c_void_p(term.ctypes.data), C.c_void_p(need.ctypes.data))
    return need


# ---------------------------------------------------------------------------------------------------
# picture geometries of the frame paths
# ---------------------------------------------------------------------------------------------------
# The frame kernels build their borders in closed form (rmd_tc2.cuh pu_avail): the below-left and above-right runs are cut by the
# picture edge, so they depend on W % 64 and H % 64.  Every residue 8 .. 56 occurs in both dimensions of a picture wider / taller than
# one CTU; pictures narrower, shorter and smaller than one CTU, and odd CTU counts (CTAs of 2 and 4 CTUs straddle pictures of a
# multi-picture launch), are in the list too.  Most sizes are 2 x 2 CTUs or fewer, so that the CPU replays stay cheap.
EDGE_SIZES = [(72, 120), (80, 112), (88, 104), (96, 96), (104, 88), (112, 80), (120, 72),
              (8, 8), (24, 136), (136, 40), (40, 24)]


def edge_content(W, H, bd, seed):
    """source and reconstruction for the geometry sweeps.  The source is textured.  The reconstruction is a gentle ramp everywhere but
    its lower right quadrant, which is textured and holds full-range noise in its own lower right quarter: the ramp covers the whole
    border of the 32x32 PUs along the top and the left, cut runs at the picture edge included, so the strong filter fires there"""
    org = textured_plane(W, H, bd, seed=seed)
    rec = pseudo_recon(org, bd, seed=seed + 1)
    ramp = ((np.arange(H)[:, None] // 8 + np.arange(W)[None, :] // 6 + 40) << (bd - 8)).astype(np.int16)
    y0, x0 = H // 2 // 8 * 8, W // 2 // 8 * 8
    keep = np.zeros((H, W), bool)
    keep[y0:, x0:] = True
    rec = np.where(keep, rec, ramp)
    y1, x1 = (H + y0) // 2, (W + x0) // 2
    rec[y1:, x1:] = np.random.default_rng(seed + 2).integers(0, 1 << bd, (H - y1, W - x1))
    return np.ascontiguousarray(org), np.ascontiguousarray(rec.astype(np.int16))


def strong_filter_pus(oracle, org, rec, bd):
    """the 32x32 PUs whose oracle costs differ between strong smoothing on and off, as (x0, y0, left units, above units): the number of
    available 4-sample units of the left column with its below-left run and of the above row with its above-right run (16 each at most)"""
    H, W = org.shape
    diff = (oracle_rmd_frame(oracle, org, rec, bd, 1) != oracle_rmd_frame(oracle, org, rec, bd, 0)).any(axis=2)
    out = []
    for y0 in range(0, H - 31, 32):
        for x0 in range(0, W - 31, 32):
            if diff[(y0 // 64) * ((W + 63) // 64) + x0 // 64, pu_table_index(x0, y0, 32)]:
                flags = np.zeros(33, np.uint8)
                oracle.oracle_neighbour_flags(x0, y0, 32, W, H, P(flags, u8p))
                out.append((x0, y0, int(flags[:16].sum()), int(flags[17:].sum())))
    return out


def threshold_recon(W, H, bd, seed):
    """a ramp with noise of +-(1 << (bd - 6)) (+-4 at 8 bit, +-16 at 10 bit): the strong-smoothing deviations of its 32x32 PUs fall
    around the threshold 1 << (bd - 5)"""
    a = 1 << (bd - 6)
    ramp = ((np.arange(H)[:, None] + np.arange(W)[None, :]) // 4 + 60) << (bd - 8)
    noise = np.random.default_rng(seed).integers(-a, a + 1, (H, W))
    return np.ascontiguousarray(np.clip(ramp + noise, 0, (1 << bd) - 1).astype(np.int16))


def strong_deviations(lib, rec, bd):
    """(|bl + tl - 2 L[N]|, |tl + tr - 2 T[N]|) of the unfiltered border (oracle_neighbour_flags + oracle_fill_border) of every 32x32 PU
    inside the picture: the two values the strong-smoothing decision compares with 1 << (bd - 5)"""
    H, W = rec.shape
    rec = np.ascontiguousarray(rec, np.int16)
    n = 32
    out = []
    for y0 in range(0, H - n + 1, n):
        for x0 in range(0, W - n + 1, n):
            flags = np.zeros(n + 1, np.uint8)                 # 2N / 4 units on each side and the corner
            lib.oracle_neighbour_flags(x0, y0, n, W, H, P(flags, u8p))
            b = np.zeros(4 * n + 1, np.int16)
            lib.oracle_fill_border(bd, n, C.c_void_p(rec.ctypes.data + 2 * (y0 * W + x0)), W, P(flags, u8p), P(b, i16p))
            b = b.astype(np.int64)
            out.append((abs(b[0] + b[2 * n] - 2 * b[n]), abs(b[2 * n] + b[4 * n] - 2 * b[3 * n])))
    return out


THRESHOLD_PICTURES = {8: (192, 128, 0), 10: (192, 128, 48)}     # bit depth: W, H, seed of threshold_recon


def threshold_picture(oracle, bd):
    """source and reconstruction whose 32x32 borders put both strong-smoothing deviations, on the left and on the above side, at
    1 << (bd - 5) and one below it; asserted here, so that a change of content cannot silently drop the case"""
    W, H, seed = THRESHOLD_PICTURES[bd]
    rec = threshold_recon(W, H, bd, seed)
    thr = 1 << (bd - 5)
    dev = strong_deviations(oracle, rec, bd)
    for side in (0, 1):
        vals = {d[side] for d in dev}
        assert thr - 1 in vals and thr in vals, (bd, side)
    assert any(max(d) == thr for d in dev)            # the decision fails only by reaching the threshold
    assert any(max(d) == thr - 1 for d in dev)        # the decision holds one below it
    return textured_plane(W, H, bd, seed=seed + 5), rec
