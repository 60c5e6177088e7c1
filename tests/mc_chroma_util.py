"""Helpers of the cucd_me_mc_chroma tests (4:2:0 chroma motion compensation of inter candidates): loaders for the checker and the
CPU replay, a seeded scene with chroma planes, candidates and the checker's answers.

tests/emul/libcucd_mc_chroma_oracle.so - oracle/cucd_oracle.c plus tests/mc_chroma_oracle.c, the checker of chroma motion compensation
tests/emul/libmc_chroma_emul.so        - tests/emul/mc_chroma_emul.cpp, the CPU replay of me_mc_chroma_kernel's per-thread code
"""
import ctypes as C
import os
import subprocess

import numpy as np

from _util import PKG, ROOT, P, _newer, i16p, i32p, pseudo_recon, textured_plane, u32p
from mc_util import MC_MODES, MC_SHAPES, mc_desc_array, mc_scene


def load_mc_chroma_oracle():
    """tests/mc_chroma_oracle.c linked with the oracle it builds on, as one library"""
    d = os.path.join(ROOT, "oracle")
    so = os.path.join(ROOT, "tests", "emul", "libcucd_mc_chroma_oracle.so")
    srcs = [os.path.join(ROOT, "tests", "mc_chroma_oracle.c"), os.path.join(d, "cucd_oracle.c"), os.path.join(d, "cucd_oracle.h")]
    if not _newer(so, srcs):
        subprocess.run(["gcc", "-O2", "-fPIC", "-std=c99", "-Wall", "-Wextra", "-ffp-contract=off", "-fno-fast-math", "-shared", "-I" + d, "-o", so,
                        srcs[0], srcs[1], "-lm"], check=True, capture_output=True)
    lib = C.CDLL(so)
    lib.oracle_sse.restype = C.c_uint32
    lib.oracle_mc_chroma_cost.restype = C.c_uint32
    return lib


def load_mc_chroma_emul():
    """tests/emul/mc_chroma_emul.cpp: the host plan of cucd_me_mc_chroma and the __host__ __device__ phases of me_mc_chroma_kernel,
    compiled for the CPU"""
    d = os.path.join(ROOT, "tests", "emul")
    so = os.path.join(d, "libmc_chroma_emul.so")
    csrc = os.path.join(ROOT, PKG, "csrc")
    cpp = os.path.join(d, "mc_chroma_emul.cpp")
    srcs = [cpp, os.path.join(ROOT, "include", "cucudecide.h")] + [os.path.join(csrc, f) for f in ("rmd_core.cuh", "me_core.cuh")]
    if not _newer(so, srcs):
        subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-Wall", "-Wno-unknown-pragmas", "-I" + csrc, "-o", so, cpp], check=True, capture_output=True)
    return C.CDLL(so)


# ---------------------------------------------------------------------------------------------------
def mcc_scene(bd, W=256, H=144, M=80, slots=(0, 3), seed=0):
    """mc_scene (luma) plus 4:2:0 chroma: source planes org_c = (Cb, Cr) of (H/2, W/2) and, per slot, padded reference planes
    refs_c[slot] = (Cb, Cr) with margin M/2 (replicated edges, HM's luma margin >> 1), carrying runs of 0 and 2^bd - 1"""
    sc = mc_scene(bd, W, H, M, slots, seed)
    hi, Wc, Hc, Mc = (1 << bd) - 1, W // 2, H // 2, M // 2
    sc["org_c"] = tuple(textured_plane(Wc, Hc, bd, seed=seed + 140 + c) for c in range(2))
    sc["refs_c"] = {}
    for k, s in enumerate(slots):
        pl = []
        for c in range(2):
            rec = pseudo_recon(textured_plane(Wc, Hc, bd, seed=seed + 150 + 2 * k + c, t=k + 1), bd)
            rec[3 + 2 * k + c::11, :] = hi
            rec[:, 5 + k + c::9] = 0
            rec[30:38, 50 + 4 * k:70 + 4 * k] = np.where(np.indices((8, 20)).sum(0) % 2 == c, hi, 0)
            pl.append(np.ascontiguousarray(np.pad(rec, Mc, mode="edge")))
        sc["refs_c"][s] = tuple(pl)
    sc["Mc"] = Mc
    return sc


def mcc_mv_range(sc, cx, cw, size_c):
    """inclusive range of the integer chroma MV part whose 4-tap support stays inside the padded chroma plane (cx + mv - 1 >= -Mc,
    cx + mv + cw + 1 <= size_c - 1 + Mc; size_c = W/2 horizontally, H/2 vertically)"""
    return 1 - sc["Mc"] - cx, size_c - 2 + sc["Mc"] - cw - cx


def mcc_candidates(sc, rng, shapes=MC_SHAPES, modes=MC_MODES, edge=True):
    """per luma PU shape and mode one candidate with random eighth-pel chroma MVs (luma quarter-pel); with edge, every fourth candidate
    puts the support of each list exactly at a corner of the chroma margin, and fractions are drawn from the extremes 0, 4 and 7 half
    of the time"""
    W, H = sc["W"], sc["H"]
    s0, s1 = sc["slots"][0], sc["slots"][-1]
    out = []
    for w, h in shapes:
        for mode in modes:
            x = int(rng.integers(0, (W - w) // 4 + 1)) * 4
            y = int(rng.integers(0, (H - h) // 4 + 1)) * 4
            n = len(out)

            def mv(lo_hi, corner):
                lo, hi = lo_hi
                i = (lo if corner == 0 else hi) if edge and n % 4 == 3 else int(rng.integers(lo, hi + 1))
                f = int(rng.choice([0, 4, 7])) if rng.random() < 0.5 else int(rng.integers(0, 8))
                return 8 * i + f
            c = [int(rng.integers(0, 2)) for _ in range(4)]
            rx, ry = mcc_mv_range(sc, x // 2, w // 2, W // 2), mcc_mv_range(sc, y // 2, h // 2, H // 2)
            mvs = [(mv(rx, c[0]), mv(ry, c[1])), (mv(rx, c[2]), mv(ry, c[3]))]
            if mode == "l0":
                ref, mvs = (s0, -1), [mvs[0], (0, 0)]
            elif mode == "l1":
                ref, mvs = (-1, s1), [(0, 0), mvs[1]]
            elif mode == "bi":
                ref = (s0, s1)
            else:
                ref, mvs = (s0, s0), [mvs[0], mvs[0]]
            out.append(dict(x=x, y=y, w=w, h=h, ref_idx=ref, mvx=(mvs[0][0], mvs[1][0]), mvy=(mvs[0][1], mvs[1][1]), use_hadamard=int(rng.integers(0, 2))))
    return out


def oracle_mc_chroma(lib, sc, descs):
    """(sse uint32 (n, 2), [(Cb, Cr) predictions]) of tests/mc_chroma_oracle.c oracle_mc_chroma_cost for the candidates"""
    Mc = sc["Mc"]
    sse = np.zeros((len(descs), 2), np.uint32)
    preds = []
    for i, d in enumerate(descs):
        cx, cy, cw, ch = d["x"] // 2, d["y"] // 2, d["w"] // 2, d["h"] // 2
        lists = [l for l in (0, 1) if d["ref_idx"][l] >= 0]
        pair = []
        for c in range(2):
            a = []
            for l in lists:
                p = sc["refs_c"][d["ref_idx"][l]][c]
                y0, x0 = cy + (d["mvy"][l] >> 3) + Mc, cx + (d["mvx"][l] >> 3) + Mc
                assert y0 >= 1 and x0 >= 1 and y0 + ch + 1 < p.shape[0] and x0 + cw + 1 < p.shape[1], d      # the support lies inside
                a.append((C.c_void_p(p.ctypes.data + 2 * (y0 * p.shape[1] + x0)), p.shape[1], d["mvx"][l] & 7, d["mvy"][l] & 7))
            b = a[1] if len(a) == 2 else (None, 0, 0, 0)
            blk = np.ascontiguousarray(sc["org_c"][c][cy:cy + ch, cx:cx + cw])
            pred = np.zeros((ch, cw), np.int16)
            sse[i, c] = lib.oracle_mc_chroma_cost(sc["bd"], P(blk, i16p), cw, len(a), a[0][0], a[0][1], a[0][2], a[0][3], b[0], b[1], b[2], b[3], cw, ch,
                                                  P(pred, i16p))
            pair.append(pred)
        preds.append(tuple(pair))
    return sse, preds


def split_pred(descs, flat):
    """the flat pred array of cucd_me_mc_chroma -> [(Cb, Cr)]"""
    out, off = [], 0
    for d in descs:
        cw, ch = d["w"] // 2, d["h"] // 2
        out.append((flat[off:off + cw * ch].reshape(ch, cw), flat[off + cw * ch:off + 2 * cw * ch].reshape(ch, cw)))
        off += 2 * cw * ch
    return out


def emul_mc_chroma(emul, sc, descs):
    """(sse (n, 2), [(Cb, Cr)], CTA count) of the CPU replay of me_mc_chroma_kernel"""
    n = len(descs)
    nslot = max(sc["refs_c"]) + 1
    planes = (C.c_void_p * (2 * nslot))()
    strides, mx = np.zeros(nslot, np.int32), np.full(nslot, sc["Mc"], np.int32)
    for s, (cb, cr) in sc["refs_c"].items():
        planes[2 * s], planes[2 * s + 1] = cb.ctypes.data, cr.ctypes.data
        strides[s] = cb.shape[1]
    org = [np.ascontiguousarray(p) for p in sc["org_c"]]
    cur = (C.c_void_p * 2)(org[0].ctypes.data, org[1].ctypes.data)
    arr = mc_desc_array(descs)
    sse = np.zeros((n, 2), np.uint32)
    pred = np.zeros(max(1, sum(d["w"] * d["h"] // 2 for d in descs)), np.int16)
    nCta = emul.emul_mc_chroma(sc["bd"], cur, org[0].shape[1], planes, P(strides, i32p), P(mx, i32p), P(mx, i32p), n, P(arr, i32p), P(sse, u32p),
                               P(pred, i16p))
    return sse, split_pred(descs, pred), nCta
