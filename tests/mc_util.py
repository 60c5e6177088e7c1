"""Helpers of the cucd_me_mc_cost tests (motion compensation of inter candidates): loaders for the checker and the CPU replay, a seeded
scene, candidates and the checker's answers.

tests/emul/libcucd_mc_oracle.so - oracle/cucd_oracle.c plus tests/mc_oracle.c, the checker of motion compensation
tests/emul/libmc_emul.so        - tests/emul/mc_emul.cpp, the CPU replay of me_mc_kernel's per-thread code
"""
import ctypes as C
import os
import subprocess

import numpy as np

from _util import PKG, ROOT, P, _newer, i16p, i32p, pseudo_recon, textured_plane, u32p


def load_mc_oracle():
    """tests/mc_oracle.c (motion compensation of inter candidates) linked with the oracle it builds on, as one library"""
    d = os.path.join(ROOT, "oracle")
    so = os.path.join(ROOT, "tests", "emul", "libcucd_mc_oracle.so")
    srcs = [os.path.join(ROOT, "tests", "mc_oracle.c"), os.path.join(d, "cucd_oracle.c"), os.path.join(d, "cucd_oracle.h")]
    if not _newer(so, srcs):
        subprocess.run(["gcc", "-O2", "-fPIC", "-std=c99", "-Wall", "-Wextra", "-ffp-contract=off", "-fno-fast-math", "-shared", "-I" + d, "-o", so,
                        srcs[0], srcs[1], "-lm"], check=True, capture_output=True)
    lib = C.CDLL(so)
    lib.oracle_satd.restype = C.c_uint32
    lib.oracle_sad.restype = C.c_uint32
    lib.oracle_mc_cost.restype = C.c_uint32
    return lib


def load_mc_emul():
    """tests/emul/mc_emul.cpp: the host plan of cucd_me_mc_cost and the __host__ __device__ phases of me_mc_kernel, compiled for the CPU"""
    d = os.path.join(ROOT, "tests", "emul")
    so = os.path.join(d, "libmc_emul.so")
    csrc = os.path.join(ROOT, PKG, "csrc")
    cpp = os.path.join(d, "mc_emul.cpp")
    srcs = [cpp, os.path.join(ROOT, "include", "cucudecide.h")] + [os.path.join(csrc, f) for f in ("rmd_core.cuh", "me_core.cuh")]
    if not _newer(so, srcs):
        subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-Wall", "-Wno-unknown-pragmas", "-I" + csrc, "-o", so, cpp], check=True, capture_output=True)
    return C.CDLL(so)


# ---------------------------------------------------------------------------------------------------
MC_SHAPES = [(64, 64), (64, 32), (32, 64), (32, 32), (64, 16), (64, 48), (16, 64), (48, 64), (32, 8), (32, 24), (8, 32), (24, 32), (16, 16), (16, 4),
             (16, 12), (4, 16), (12, 16), (16, 8), (8, 16), (8, 8), (8, 4), (4, 8)]      # the PU shapes of test_gpu_subpel.py
MC_MODES = ("l0", "l1", "bi", "bi_same")


def mc_scene(bd, W=256, H=144, M=80, slots=(0, 3), seed=0):
    """source plane and padded reference planes (margin M, replicated edges) in the given slots; the references carry runs of 0 and
    2^bd - 1 so that the clip and the intermediates' extremes are reached"""
    hi = (1 << bd) - 1
    org = textured_plane(W, H, bd, seed=seed + 40)
    refs = {}
    for k, s in enumerate(slots):
        rec = pseudo_recon(textured_plane(W, H, bd, seed=seed + 41 + k, t=k + 1), bd)
        rec[5 + 3 * k::17, :] = hi
        rec[:, 7 + k::13] = 0
        rec[60:76, 100 + 8 * k:140 + 8 * k] = np.where(np.indices((16, 40)).sum(0) % 2 == 0, hi, 0)
        refs[s] = np.ascontiguousarray(np.pad(rec, M, mode="edge"))
    return dict(bd=bd, W=W, H=H, M=M, org=org, refs=refs, slots=tuple(slots))


def mc_mv_range(sc, x, w, size):
    """inclusive range of the integer MV part whose 8-tap support stays inside the padded plane (x + mv - 3 >= -M,
    x + mv + w + 3 <= size - 1 + M; size = W horizontally, H vertically)"""
    return 3 - sc["M"] - x, size - 1 + sc["M"] - w - 3 - x


def mc_candidates(sc, rng, shapes=MC_SHAPES, modes=MC_MODES, hads=(1, 0), edge=True):
    """per shape, mode and distortion one candidate with random quarter-pel MVs; with edge, every fourth candidate puts the support
    of each list exactly at a corner of the margin, and fractions are drawn from the extremes 0 and 3 half of the time"""
    W, H = sc["W"], sc["H"]
    s0, s1 = sc["slots"][0], sc["slots"][-1]
    out = []
    for w, h in shapes:
        for mode in modes:
            for had in hads:
                x = int(rng.integers(0, (W - w) // 4 + 1)) * 4
                y = int(rng.integers(0, (H - h) // 4 + 1)) * 4
                n = len(out)

                def mv(lo_hi, corner):
                    lo, hi = lo_hi
                    i = (lo if corner == 0 else hi) if edge and n % 4 == 3 else int(rng.integers(lo, hi + 1))
                    f = int(rng.choice([0, 3])) if rng.random() < 0.5 else int(rng.integers(0, 4))
                    return 4 * i + f
                c = [int(rng.integers(0, 2)) for _ in range(4)]
                rx, ry = mc_mv_range(sc, x, w, W), mc_mv_range(sc, y, h, H)
                mvs = [(mv(rx, c[0]), mv(ry, c[1])), (mv(rx, c[2]), mv(ry, c[3]))]
                if mode == "l0":
                    ref, mvs = (s0, -1), [mvs[0], (0, 0)]
                elif mode == "l1":
                    ref, mvs = (-1, s1), [(0, 0), mvs[1]]
                elif mode == "bi":
                    ref = (s0, s1)
                else:
                    ref, mvs = (s0, s0), [mvs[0], mvs[0]]
                out.append(dict(x=x, y=y, w=w, h=h, ref_idx=ref, mvx=(mvs[0][0], mvs[1][0]), mvy=(mvs[0][1], mvs[1][1]), use_hadamard=had))
    return out


def mc_ref_at(sc, slot, x, y, mvx, mvy):
    """pointer to the sample at the integer part of the MV of the block at (x, y) in the padded plane of `slot`"""
    p, M = sc["refs"][slot], sc["M"]
    return C.c_void_p(p.ctypes.data + 2 * ((y + (mvy >> 2) + M) * p.shape[1] + x + (mvx >> 2) + M))


def oracle_mc(lib, sc, descs):
    """(dist uint32[n], predictions) of tests/mc_oracle.c oracle_mc_cost for the candidates"""
    org = np.ascontiguousarray(sc["org"])
    dist = np.zeros(len(descs), np.uint32)
    preds = []
    for i, d in enumerate(descs):
        lists = [l for l in (0, 1) if d["ref_idx"][l] >= 0]
        for l in lists:                                    # the 8-tap support lies inside the padded plane
            rows, cols = sc["refs"][d["ref_idx"][l]].shape
            y0, x0 = d["y"] + (d["mvy"][l] >> 2) + sc["M"], d["x"] + (d["mvx"][l] >> 2) + sc["M"]
            assert y0 >= 3 and x0 >= 3 and y0 + d["h"] + 3 < rows and x0 + d["w"] + 3 < cols, d
        a = [(mc_ref_at(sc, d["ref_idx"][l], d["x"], d["y"], d["mvx"][l], d["mvy"][l]), sc["refs"][d["ref_idx"][l]].shape[1], d["mvx"][l] & 3, d["mvy"][l] & 3)
             for l in lists]
        b = a[1] if len(a) == 2 else (None, 0, 0, 0)
        blk = np.ascontiguousarray(org[d["y"]:d["y"] + d["h"], d["x"]:d["x"] + d["w"]])
        pred = np.zeros((d["h"], d["w"]), np.int16)
        dist[i] = lib.oracle_mc_cost(sc["bd"], P(blk, i16p), d["w"], len(a), a[0][0], a[0][1], a[0][2], a[0][3], b[0], b[1], b[2], b[3], d["w"], d["h"],
                                     d["use_hadamard"], P(pred, i16p))
        preds.append(pred)
    return dist, preds


def mc_desc_array(descs):
    """cucd_mc_desc records (11 int32 each) for the CPU replay"""
    return np.array([[d["x"], d["y"], d["w"], d["h"], *d["ref_idx"], *d["mvx"], *d["mvy"], d["use_hadamard"]] for d in descs], np.int32).reshape(-1, 11)


def emul_mc(emul, sc, descs):
    """(dist, predictions, CTA count) of the CPU replay of me_mc_kernel"""
    n = len(descs)
    nslot = max(sc["refs"]) + 1
    planes = (C.c_void_p * nslot)()
    strides, mx = np.zeros(nslot, np.int32), np.full(nslot, sc["M"], np.int32)
    for s, p in sc["refs"].items():
        planes[s] = p.ctypes.data
        strides[s] = p.shape[1]
    arr = mc_desc_array(descs)
    org = np.ascontiguousarray(sc["org"])
    dist = np.zeros(n, np.uint32)
    pred = np.zeros(max(1, sum(d["w"] * d["h"] for d in descs)), np.int16)
    nCta = emul.emul_mc_cost(sc["bd"], P(org, i16p), sc["W"], planes, P(strides, i32p), P(mx, i32p), P(mx, i32p), n, P(arr, i32p), P(dist, u32p), P(pred, i16p))
    preds, off = [], 0
    for d in descs:
        preds.append(pred[off:off + d["w"] * d["h"]].reshape(d["h"], d["w"]))
        off += d["w"] * d["h"]
    return dist, preds, nCta
