#!/usr/bin/env python3
"""bench_rows.py - secondary measurements: the SURVEY.md section-8 rows that bench.py's headline line does not cover.

bench.py times the frame path (a1-a5, a8-a11).  This script times the other operators of include/cucudecide.h on one B200,
each on a 1080p-sized workload, and prints ONE JSON line per row:
  kernel   throughput from the device time between the first and last kernel of the call (cucd_last_kernel_time: CUDA events
           on the library's stream, copies outside) and the HBM roofline fraction of that time for the row's ALGORITHMIC bytes
           (every input read once, every output written once; DESIGN.md section 4 states the per-unit figures)
  e2e      the same C-ABI call with host buffers, wall clock around the bare call (descriptor arrays prebuilt, copies inside): the caller's
           buffers page-locked once through cucd_pin_host_buffer (what an encoder does with its long-lived buffers); e2e_pageable: the same
           buffers before they were pinned.  h2d_bytes / d2h_bytes let the reader subtract the PCIe time
  cpu      the reference's own function (oracle/_ref/libhmref.so, kind "reference") or the oracle port (kind "port") on a
           bounded sample, on `cores` host threads
Rows: s2 (cucd_intra_rmd_batch), f1 (cucd_queue_*: K concurrent instances), s3 (cucd_me_sad_surface), f3 (cucd_me_subpel_cost),
a12 (cucd_tmv_features), a13 (cucd_aq_activity), f2 (cucd_intra_tu_code / _forward / _recon).  Usage: python bench_rows.py [--iters 5] > gpurun_out/rows.jsonl
Last rows: f5 (cucd_me_mc_cost, motion compensation + distortion of inter candidates; row_f5 runs it on its own), f6
(cucd_inter_tu_forward / _code / _recon, the TUs of inter residual quadtrees; row_f6) and f7 (cucd_me_mc_chroma, the 4:2:0 chroma of
f5's candidates; row_f7) and f8 (cucd_me_search / _src, the motion search of bench.py's inter workloads against the surface route it
replaces; row_f8) and f9 (cucd_me_tz_search, the TZ search of the same workloads, depth by depth; row_f9).  --only f5 / f6 / f7 / f8 / f9
runs one of them alone.
"""
import argparse
import ctypes as C
import importlib
import json
import os
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import _util  # noqa: E402
from _util import P, i16p, i32p, u32p, f64p  # noqa: E402

W, H = 1920, 1080


def hbm_peak():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"], "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        return 7700.0, "fallback (B200_PROFILING.md nominal)"


def timed(fn, eng, iters, pin=()):
    """returns (kernel s, call s with the buffers in `pin` page-locked, call s with pageable buffers)"""
    fn()                                     # warm-up (allocations inside the handle)
    fn()
    ps = []
    for _ in range(max(2, iters // 2)):
        t0 = time.perf_counter()
        fn()
        ps.append(time.perf_counter() - t0)
    for a in pin:
        eng.pin_host_buffer(a)
    fn()
    ks, ws = [], []
    for _ in range(iters):
        t0 = time.perf_counter()
        fn()
        ws.append(time.perf_counter() - t0)
        ks.append(eng.last_kernel_time_ms() * 1e-3)
    for a in pin:
        eng.unpin_host_buffer(a)
    return float(np.median(ks)), float(np.median(ws)), float(np.median(ps))


def cpu_parallel(work, n_items, threads):
    """run work(i) for i in range(n_items) on `threads` host threads (ctypes releases the GIL); returns seconds"""
    t0 = time.perf_counter()
    with ThreadPoolExecutor(threads) as ex:
        list(ex.map(work, range(n_items)))
    return time.perf_counter() - t0


def emit(row, unit, units, k_s, w_s, algo_bytes, cpu, extra=None, p_s=None, h2d=None, d2h=None):
    peak, src = hbm_peak()
    gbs = algo_bytes / k_s / 1e9
    d = {"row": row, "unit": unit, "units_per_call": units,
         "kernel": {"value": units / k_s, "ms": k_s * 1e3, "algorithmic_bytes": algo_bytes, "achieved_gbs": gbs, "hbm_peak_gbs": peak,
                    "frac": gbs / peak, "peak_source": src},
         "e2e": {"value": units / w_s, "ms": w_s * 1e3, "call_over_kernel": w_s / k_s, "h2d_bytes": h2d, "d2h_bytes": d2h},
         "e2e_pageable": None if p_s is None else {"value": units / p_s, "ms": p_s * 1e3},
         "cpu": cpu}
    if extra:
        d.update(extra)
    print(json.dumps(d), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--cpu-threads", type=int, default=min(16, os.cpu_count() or 1))
    ap.add_argument("--only", choices=["f5", "f6", "f7", "f8", "f9"], default=None, help="run one of the last rows alone")
    a = ap.parse_args()
    cucd = importlib.import_module("fast-cu-decision-hevc_b200")
    if a.only:
        {"f5": row_f5, "f6": row_f6, "f7": row_f7, "f8": row_f8, "f9": row_f9}[a.only](cucd, a.iters, a.cpu_threads)
        return
    oracle = _util.load_oracle()
    ref = _util.load_hmref()
    T = a.cpu_threads
    org = _util.textured_plane(W, H, 8, seed=5)
    rec = _util.pseudo_recon(org, 8)
    rng = np.random.default_rng(1)
    eng = cucd.Engine(W, H, bit_depth=8)

    # ---- S2: batched RMD with caller-supplied borders: the 341 PUs of 510 CTUs' worth of blocks (mixed sizes) -------------
    sizes, orgs, brds = [], [], []
    for n, cnt in ((64, 480), (32, 1980), (16, 8040), (8, 32400), (4, 129600)):
        cnt = cnt // 4                      # a quarter picture per call keeps the host-side packing small
        sizes += [int(np.log2(n))] * cnt
        orgs.append(rng.integers(0, 256, cnt * n * n).astype(np.int16))
        brds.append(rng.integers(0, 256, cnt * (4 * n + 1)).astype(np.int16))
    o, b = np.concatenate(orgs), np.concatenate(brds)
    n_pu = len(sizes)
    pu_arr, _ = cucd.Engine.pu_descs(sizes)
    sad_out = np.zeros((n_pu, 35), np.uint32)
    k_s, w_s, p_s = timed(lambda: eng.intra_rmd_batch_raw(pu_arr, n_pu, o, b, sad_out), eng, a.iters, pin=(o, b, sad_out))
    algo = o.nbytes + b.nbytes + n_pu * 35 * 4
    # CPU: the reference's own prediction + Hadamard functions per PU
    samp = list(range(0, n_pu, 97))
    off_o = np.cumsum([0] + [1 << (2 * s) for s in sizes]); off_b = np.cumsum([0] + [(4 << s) + 1 for s in sizes])
    lib, kind = (ref, "reference") if ref is not None else (oracle, "port")
    fn = lib.hmref_rmd_pu if ref is not None else lib.oracle_rmd_pu

    def work_s2(i):
        j = samp[i]; n = 1 << sizes[j]
        out = np.zeros(35, np.uint32)
        fn(8, n, 1, C.c_void_p(o.ctypes.data + 2 * int(off_o[j])), n, C.c_void_p(b.ctypes.data + 2 * int(off_b[j])), P(out, u32p))
    sec = cpu_parallel(work_s2, len(samp), T)
    emit("s2_intra_rmd_batch", "PU/s", n_pu, k_s, w_s, algo,
         {"value": len(samp) / sec, "unit": "PU/s", "cores": T, "kind": kind, "sample": f"every 97th PU of the batch ({len(samp)} PUs, same size mix) in {sec:.2f} s"},
         p_s=p_s, h2d=int(o.nbytes + b.nbytes + n_pu * 16), d2h=int(sad_out.nbytes))

    # ---- f1: the coalescing queue: K encoder instances (host threads), each submitting one CU's worth of PUs per request and waiting
    #      for it (the live encoder's serial dependency), for K = 1, 4, 16: what coalescing buys over one-request-per-launch ----------------
    #      (a C++ driver: Python threads would measure the GIL) ------------------------------------------------------------------------------
    import subprocess
    exe = os.path.join(ROOT, "profiles", "ubench", "queue_bench")
    pkg = os.path.join(ROOT, "fast-cu-decision-hevc_b200")
    try:
        subprocess.run(["g++", "-O2", "-std=c++17", "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "profiles", "ubench", "queue_bench.cpp"),
                        "-L" + pkg, "-lcucudecide", "-Wl,-rpath," + pkg, "-lpthread", "-o", exe], check=True, capture_output=True)
        sys.stdout.write(subprocess.run([exe, "2000"], check=True, capture_output=True, text=True).stdout)
        sys.stdout.flush()
    except (subprocess.CalledProcessError, OSError) as e:
        print(json.dumps({"row": "f1_rmd_queue", "unavailable": str(e)[:200]}), flush=True)

    # ---- S3: integer-ME SAD surfaces: every whole 32x32 PU of the picture, +-32 window, FEN row sub-sampling ---------------
    pad = 80
    refp = np.pad(rec, pad, mode="edge")
    eng.set_cur_picture(org); eng.set_ref_picture(0, refp, pad, pad)
    descs = [dict(x=x, y=y, w=32, h=32, ref_idx=0, left=-32, right=32, top=-32, bottom=32, sub_shift=1)
             for y in range(0, H - 31, 32) for x in range(0, W - 31, 32)]
    n_pu = len(descs)
    me_arr, _, me_total = cucd.Engine.me_descs(descs)
    surf = np.zeros(me_total, np.uint32)
    k_s, w_s, p_s = timed(lambda: eng.me_sad_surface_raw(me_arr, n_pu, surf), eng, a.iters, pin=(surf,))
    algo = n_pu * (32 * 32 * 2 + 96 * 96 * 2 + 65 * 65 * 4)
    samp = descs[::40]
    Wp = W + 2 * pad
    fn = ref.hmref_sad_surface if ref is not None else oracle.oracle_sad_surface

    def work_s3(i):
        d = samp[i]
        blk = np.ascontiguousarray(org[d["y"]:d["y"] + 32, d["x"]:d["x"] + 32])
        out = np.zeros(65 * 65, np.uint32)
        base = refp.ctypes.data + 2 * ((d["y"] + pad) * Wp + d["x"] + pad)
        fn(8, P(blk, i16p), 32, 32, 32, C.c_void_p(base), Wp, -32, 32, -32, 32, 1, P(out, u32p))
    sec = cpu_parallel(work_s3, len(samp), T)
    emit("s3_me_sad_surface", "candidate SAD/s", n_pu * 65 * 65, k_s, w_s, algo,
         {"value": len(samp) * 65 * 65 / sec, "unit": "candidate SAD/s", "cores": T, "kind": kind,
          "sample": f"{len(samp)} of the {n_pu} PUs (32x32, 65x65 window, iSubShift 1) in {sec:.2f} s"},
         {"pus_per_call": n_pu}, p_s=p_s, h2d=int(n_pu * 40), d2h=int(surf.nbytes))

    # ---- f3: fractional-pel refinement of the same PUs around a pseudo-random integer MV, Hadamard -------------------------------------------
    sdescs = [dict(x=d["x"], y=d["y"], w=32, h=32, ref_idx=0, mvx=int(rng.integers(-16, 17)), mvy=int(rng.integers(-16, 17)), use_hadamard=1) for d in descs]
    sp_arr, _ = cucd.Engine.subpel_descs(sdescs)
    sp_out = np.zeros((len(sdescs), 49), np.uint32)
    k_s, w_s, p_s = timed(lambda: eng.me_subpel_cost_raw(sp_arr, len(sdescs), sp_out), eng, a.iters, pin=(sp_out,))
    algo = len(sdescs) * (32 * 32 * 2 + 41 * 41 * 2 + 49 * 4)
    samp = sdescs[::40]

    def work_f3(i):
        d = samp[i]
        blk = np.ascontiguousarray(org[d["y"]:d["y"] + 32, d["x"]:d["x"] + 32])
        out = np.zeros(49, np.uint32)
        base = refp.ctypes.data + 2 * ((d["y"] + pad) * Wp + d["x"] + pad)
        oracle.oracle_subpel_surface(8, P(blk, i16p), 32, 32, 32, C.c_void_p(base), Wp, d["mvx"], d["mvy"], 1, P(out, u32p))
    sec = cpu_parallel(work_f3, len(samp), T)
    emit("f3_me_subpel_cost", "PU refinement/s", len(sdescs), k_s, w_s, algo,
         {"value": len(samp) / sec, "unit": "PU refinement/s", "cores": T, "kind": "port",
          "sample": f"{len(samp)} of the {len(sdescs)} PUs (32x32, 49 quarter-pel positions, Hadamard) through the oracle in {sec:.2f} s"},
         p_s=p_s, h2d=int(len(sdescs) * 32), d2h=int(sp_out.nbytes))

    # ---- a12: TMV features of every whole CU of the picture (depths 0..3) -------------------------------------------------------
    cus = _util.all_cus(W, H)
    cu_arr, n_cu = cucd.Engine.cu_descs(cus)
    feat = np.zeros((n_cu, 5, 26))
    k_s, w_s, p_s = timed(lambda: eng.tmv_features_raw(cu_arr, n_cu, feat), eng, a.iters, pin=(feat,))
    algo = sum((1 << (2 * l)) * 2 + 130 * 8 for _, _, l in cus)
    samp = cus[::61]

    def work_a12(i):
        x, y, l = samp[i]
        out = np.zeros(130)
        if ref is not None:
            ref.hmref_tmv_features(P(org, i16p), W, W, H, x, y, 1 << l, P(out, f64p))
        else:
            oracle.oracle_tmv_features(C.c_void_p(org.ctypes.data + 2 * (y * W + x)), W, 1 << l, P(out, f64p))
    sec = cpu_parallel(work_a12, len(samp), 1)          # the reference shim copies the whole plane per call: 1 thread, plane copy included
    emit("a12_tmv_features", "CU/s", len(cus), k_s, w_s, algo,
         {"value": len(samp) / sec, "unit": "CU/s", "cores": 1, "kind": kind, "sample": f"every 61st CU ({len(samp)}) in {sec:.2f} s (driver copies the plane per call)"},
         p_s=p_s, h2d=int(n_cu * 12), d2h=int(feat.nbytes))

    # ---- a13: AQ activity, 4 layers ------------------------------------------------------------------------------------------------
    k_s, w_s, _ = timed(lambda: eng.aq_activity(4), eng, a.iters)
    units = sum(((W + (64 >> d) - 1) // (64 >> d)) * ((H + (64 >> d) - 1) // (64 >> d)) for d in range(4))
    algo = 4 * W * H * 2 + units * 8
    t0 = time.perf_counter()
    _util.oracle_aq_activity(oracle, org, 4)
    sec = time.perf_counter() - t0
    emit("a13_aq_activity", "AQ unit/s", units, k_s, w_s, algo,
         {"value": units / sec, "unit": "AQ unit/s", "cores": 1, "kind": "port", "sample": f"one 1080p picture, 4 layers, in {sec:.3f} s"})

    # ---- f2: intra TU coding: every whole TU position of the picture at 32/16/8/4 with a random mode ------------------------------------
    tus, orgs, brds = [], [], []
    for n in (32, 16, 8, 4):
        for y in range(0, H - n + 1, n):
            rows = org[y:y + n]
            for x in range(0, W - n + 1, n):
                tus.append((int(np.log2(n)), int(rng.integers(0, 35)), 32, 0))
                orgs.append(rows[:, x:x + n].ravel())
    o = np.concatenate(orgs)
    nb = sum((4 << t[0]) + 1 for t in tus)
    b = np.resize(o, nb).astype(np.int16)            # borders drawn from the picture's own samples
    n_tu = len(tus)
    samples = o.size
    _, tu_arr, _ = cucd.Engine._tu_descs(tus)
    coef = np.zeros(samples, np.int32); pix = np.zeros(samples, np.int16); dist = np.zeros(n_tu, np.uint32); asum = np.zeros(n_tu, np.int32)
    pins = (o, b, coef, pix, dist, asum)
    for name, stage, out_bytes in (("f2_intra_tu_forward", 0, samples * 6), ("f2_intra_tu_code", 1, samples * 6 + n_tu * 8), ("f2_intra_tu_recon", 2, samples * 2 + n_tu * 4)):
        k_s, w_s, p_s = timed(lambda: eng.intra_tu_raw(stage, tu_arr, n_tu, o, b, coef, pix, dist, asum), eng, a.iters, pin=pins)
        algo = o.nbytes + b.nbytes + out_bytes + (samples * 4 if stage == 2 else 0)
        cpu = None
        if name == "f2_intra_tu_code":
            samp = list(range(0, n_tu, 53))
            off_o = np.cumsum([0] + [1 << (2 * t[0]) for t in tus]); off_b = np.cumsum([0] + [(4 << t[0]) + 1 for t in tus])

            def work_tu(i):
                j = samp[i]; n = 1 << tus[j][0]
                _util.oracle_intra_tu(oracle, 8, n, tus[j][1], 32, 0, o[off_o[j]:off_o[j + 1]], b[off_b[j]:off_b[j + 1]], 1)
            sec = cpu_parallel(work_tu, len(samp), T)
            cpu = {"value": len(samp) / sec, "unit": "TU/s", "cores": T, "kind": "port",
                   "sample": f"every 53rd TU ({len(samp)}, same size mix) through the oracle's matrix-form chain in {sec:.2f} s"}
        emit(name, "TU/s", n_tu, k_s, w_s, algo, cpu, {"luma_samples_per_call": int(samples)}, p_s=p_s,
             h2d=int(o.nbytes + b.nbytes + n_tu * 16 + (samples * 4 if stage == 2 else 0)), d2h=int(out_bytes))
    eng.close()
    row_f5(cucd, a.iters, T)
    row_f6(cucd, a.iters, T)
    row_f7(cucd, a.iters, T)
    row_f8(cucd, a.iters, T)
    row_f9(cucd, a.iters, T)


def gpu_identity():
    """name and power limit of the card the row ran on, read in the same run as the measurement"""
    import subprocess
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        return "unknown"


def f5_candidates(rng):
    """the candidates of row_f5: every whole 32x32, 16x16 and 8x8 PU of a 1920x1080 picture carries five (quarter-pel MVs within
    +-64 samples; a third uni L0, a third uni L1, a third bi; Hadamard)"""
    descs = []
    for n in (32, 16, 8):
        for y in range(0, H - n + 1, n):
            for x in range(0, W - n + 1, n):
                for c in range(5):
                    mv = [int(v) for v in rng.integers(-256, 257, 4)]
                    kind = (len(descs)) % 3
                    ref = ((0, -1), (-1, 1), (0, 1))[kind]
                    descs.append(dict(x=x, y=y, w=n, h=n, ref_idx=ref, mvx=(mv[0], mv[1]), mvy=(mv[2], mv[3]), use_hadamard=1))
    return descs


def row_f5(cucd, iters=5, threads=8):
    """f5: motion compensation + distortion of inter candidates (cucd_me_mc_cost) on a 1920x1080 10-bit picture with two references.
    Batched: every whole 32x32, 16x16 and 8x8 PU carries five merge-like candidates (quarter-pel MVs within +-64 samples; a third uni
    L0, a third uni L1, a third bi; Hadamard), one call for the picture.  Latency: one request of one 16x16 bi candidate, what an
    encoder pays per call when it sends a PU at a time."""
    bd, pad = 10, 80
    org = _util.textured_plane(W, H, bd, seed=51)
    refs = [np.pad(_util.pseudo_recon(_util.textured_plane(W, H, bd, seed=51, t=k + 1), bd), pad, mode="edge") for k in range(2)]
    rng = np.random.default_rng(5)
    eng = cucd.Engine(W, H, bit_depth=bd)
    eng.set_cur_picture(org)
    for k, r in enumerate(refs):
        eng.set_ref_picture(k, r, pad, pad)
    descs = f5_candidates(rng)
    arr, n_c, samples = cucd.Engine.mc_descs(descs)
    dist = np.zeros(n_c, np.uint32)
    pred = np.zeros(samples, np.int16)
    k_s, w_s, p_s = timed(lambda: eng.me_mc_cost_raw(arr, n_c, dist), eng, iters, pin=(dist,))
    kp_s, wp_s, _ = timed(lambda: eng.me_mc_cost_raw(arr, n_c, dist, pred), eng, iters, pin=(dist, pred))
    n_lists = sum(2 if d["ref_idx"][0] >= 0 and d["ref_idx"][1] >= 0 else 1 for d in descs)
    algo = sum(d["w"] * d["h"] * 2 + 4 + 44 for d in descs) + sum((d["w"] + 7) * (d["h"] + 7) * 2 for d in descs for r in d["ref_idx"] if r >= 0)
    # CPU: the oracle on host threads, every 97th candidate
    import mc_util
    mco = mc_util.load_mc_oracle()
    samp = descs[::97]
    Wp = W + 2 * pad

    def work(i):
        d = samp[i]
        blk = np.ascontiguousarray(org[d["y"]:d["y"] + d["h"], d["x"]:d["x"] + d["w"]])
        a = [(C.c_void_p(refs[r].ctypes.data + 2 * ((d["y"] + (d["mvy"][l] >> 2) + pad) * Wp + d["x"] + (d["mvx"][l] >> 2) + pad)), d["mvx"][l] & 3, d["mvy"][l] & 3)
             for l, r in enumerate(d["ref_idx"]) if r >= 0]
        b = a[1] if len(a) == 2 else (None, 0, 0)
        mco.oracle_mc_cost(bd, P(blk, i16p), d["w"], len(a), a[0][0], Wp, a[0][1], a[0][2], b[0], Wp, b[1], b[2], d["w"], d["h"], 1, None)
    sec = cpu_parallel(work, len(samp), threads)
    # single-candidate latency: wall clock of one call, median over many
    one = [dict(x=960, y=528, w=16, h=16, ref_idx=(0, 1), mvx=(37, -90), mvy=(-13, 58), use_hadamard=1)]
    one_arr, _, _ = cucd.Engine.mc_descs(one)
    one_dist = np.zeros(1, np.uint32)
    for _ in range(50):
        eng.me_mc_cost_raw(one_arr, 1, one_dist)
    lat = []
    for _ in range(2000):
        t0 = time.perf_counter()
        eng.me_mc_cost_raw(one_arr, 1, one_dist)
        lat.append(time.perf_counter() - t0)
    eng.close()
    emit("f5_me_mc_cost", "candidate/s", n_c, k_s, w_s, algo,
         {"value": len(samp) / sec, "unit": "candidate/s", "cores": threads, "kind": "port",
          "sample": f"every 97th candidate ({len(samp)}) through tests/mc_oracle.c in {sec:.2f} s"},
         {"gpu": gpu_identity(), "bit_depth": bd, "pus": n_c // 5, "candidates_per_call": n_c, "lists_per_call": n_lists,
          "with_pred": {"kernel_ms": kp_s * 1e3, "e2e_ms": wp_s * 1e3, "d2h_bytes": int(dist.nbytes + pred.nbytes)},
          "single_candidate_latency_us": {"median": float(np.median(lat)) * 1e6, "p10": float(np.percentile(lat, 10)) * 1e6,
                                          "p90": float(np.percentile(lat, 90)) * 1e6, "calls": len(lat), "candidate": "16x16 bi, Hadamard"}},
         p_s=p_s, h2d=int(n_c * 44), d2h=int(dist.nbytes))


def row_f7(cucd, iters=5, threads=8):
    """f7: 4:2:0 chroma motion compensation + SSE (cucd_me_mc_chroma) of exactly the f5 workload: the same 1920x1080 10-bit picture
    size, two references, the same candidate array (five per whole 32/16/8 PU), one call; chroma planes 960x540 with an 80 / 2 margin.
    Latency: one request of one 16x16 bi candidate (its 8x8 Cb and Cr blocks)."""
    bd, pad = 10, 40
    Wc, Hc = W // 2, H // 2
    org_c = [_util.textured_plane(Wc, Hc, bd, seed=71 + c) for c in range(2)]
    refs_c = [[np.pad(_util.pseudo_recon(_util.textured_plane(Wc, Hc, bd, seed=71 + c, t=k + 1), bd), pad, mode="edge") for c in range(2)] for k in range(2)]
    eng = cucd.Engine(W, H, bit_depth=bd)
    eng.set_cur_picture_chroma(*org_c)
    for k in range(2):
        eng.set_ref_picture_chroma(k, *refs_c[k], pad, pad)
    descs = f5_candidates(np.random.default_rng(5))
    arr, n_c, samples = cucd.Engine.mc_descs(descs)
    sse = np.zeros(2 * n_c, np.uint32)
    pred = np.zeros(samples // 2, np.int16)
    k_s, w_s, p_s = timed(lambda: eng.me_mc_chroma_raw(arr, n_c, sse), eng, iters, pin=(sse,))
    kp_s, wp_s, _ = timed(lambda: eng.me_mc_chroma_raw(arr, n_c, sse, pred), eng, iters, pin=(sse, pred))
    n_lists = sum(2 if d["ref_idx"][0] >= 0 and d["ref_idx"][1] >= 0 else 1 for d in descs)
    # per candidate: the two source blocks, 44 descriptor bytes, two sse words, and per used list two (w/2 + 3)(h/2 + 3) windows
    algo = sum(d["w"] * d["h"] // 2 * 2 + 44 + 8 for d in descs) + sum(2 * (d["w"] // 2 + 3) * (d["h"] // 2 + 3) * 2 for d in descs for r in d["ref_idx"] if r >= 0)
    import mc_chroma_util
    mco = mc_chroma_util.load_mc_chroma_oracle()
    samp = descs[::97]
    Wp = Wc + 2 * pad

    def work(i):
        d = samp[i]
        cx, cy, cw, ch = d["x"] // 2, d["y"] // 2, d["w"] // 2, d["h"] // 2
        for c in range(2):
            blk = np.ascontiguousarray(org_c[c][cy:cy + ch, cx:cx + cw])
            a = [(C.c_void_p(refs_c[r][c].ctypes.data + 2 * ((cy + (d["mvy"][l] >> 3) + pad) * Wp + cx + (d["mvx"][l] >> 3) + pad)), d["mvx"][l] & 7, d["mvy"][l] & 7)
                 for l, r in enumerate(d["ref_idx"]) if r >= 0]
            b = a[1] if len(a) == 2 else (None, 0, 0)
            mco.oracle_mc_chroma_cost(bd, P(blk, i16p), cw, len(a), a[0][0], Wp, a[0][1], a[0][2], b[0], Wp, b[1], b[2], cw, ch, None)
    sec = cpu_parallel(work, len(samp), threads)
    one = [dict(x=960, y=528, w=16, h=16, ref_idx=(0, 1), mvx=(37, -90), mvy=(-13, 58), use_hadamard=1)]
    one_arr, _, _ = cucd.Engine.mc_descs(one)
    one_sse = np.zeros(2, np.uint32)
    for _ in range(50):
        eng.me_mc_chroma_raw(one_arr, 1, one_sse)
    lat = []
    for _ in range(2000):
        t0 = time.perf_counter()
        eng.me_mc_chroma_raw(one_arr, 1, one_sse)
        lat.append(time.perf_counter() - t0)
    eng.close()
    emit("f7_me_mc_chroma", "candidate/s", n_c, k_s, w_s, algo,
         {"value": len(samp) / sec, "unit": "candidate/s", "cores": threads, "kind": "port",
          "sample": f"every 97th candidate ({len(samp)}, Cb and Cr) through tests/mc_chroma_oracle.c in {sec:.2f} s"},
         {"gpu": gpu_identity(), "bit_depth": bd, "chroma_format": "4:2:0", "pus": n_c // 5, "candidates_per_call": n_c, "lists_per_call": n_lists,
          "with_pred": {"kernel_ms": kp_s * 1e3, "e2e_ms": wp_s * 1e3, "d2h_bytes": int(sse.nbytes + pred.nbytes)},
          "single_candidate_latency_us": {"median": float(np.median(lat)) * 1e6, "p10": float(np.percentile(lat, 10)) * 1e6,
                                          "p90": float(np.percentile(lat, 90)) * 1e6, "calls": len(lat), "candidate": "16x16 bi (8x8 Cb + Cr)"}},
         p_s=p_s, h2d=int(n_c * 44), d2h=int(sse.nbytes))


def row_f6(cucd, iters=5, threads=8):
    """f6: inter TU coding (cucd_inter_tu_forward / _code / _recon) on the residual of one 1920x1080 8-bit picture: the source minus a
    copy shifted by (3, 2) samples, tiled at every luma RQT level 32/16/8/4 (whole TUs) and, for each 4:2:0 chroma plane (the source
    sub-sampled at two phases, minus its shifted copy), at 16/8/4; QP 32 (chroma 31), sign hiding; one call for the picture."""
    bd = 8
    org = _util.textured_plane(W, H, bd, seed=61).astype(np.int32)
    planes = [(org - np.roll(org, (2, 3), axis=(0, 1)), (32, 16, 8, 4), 32, 0)]
    for ph in (0, 1):
        c = org[ph::2, ph::2]
        planes.append((c - np.roll(c, (1, 2), axis=(0, 1)), (16, 8, 4), 31, 1))
    tus, blocks = [], []
    for plane, sizes, qp, chroma in planes:
        for n in sizes:
            ph, pw = plane.shape[0] // n * n, plane.shape[1] // n * n
            b = plane[:ph, :pw].reshape(ph // n, n, pw // n, n).transpose(0, 2, 1, 3).reshape(-1, n * n)
            tus += [(int(np.log2(n)), qp, 0, chroma)] * b.shape[0]
            blocks.append(b.ravel())
    resi = np.concatenate(blocks).astype(np.int16)
    n_tu, samples = len(tus), int(resi.size)
    _, arr, total = cucd.Engine._inter_tu_descs(tus)
    assert total == samples
    coef = np.zeros(samples, np.int32); rresi = np.zeros(samples, np.int16)
    dist = np.zeros(n_tu, np.uint32); dz = np.zeros(n_tu, np.uint32); asum = np.zeros(n_tu, np.int32)
    pins = (resi, coef, rresi, dist, dz, asum)
    eng = cucd.Engine(W, H, bit_depth=bd)
    import inter_tu_util
    ito = inter_tu_util.load_inter_tu_oracle()
    offs = np.cumsum([0] + [1 << (2 * t[0]) for t in tus])
    gpu = gpu_identity()
    rows = (("f6_inter_tu_forward", 0, samples * 4 + n_tu * 4, samples * 2),
            ("f6_inter_tu_code", 1, samples * 6 + n_tu * 12, samples * 2),
            ("f6_inter_tu_recon", 2, samples * 2 + n_tu * 4, samples * 6))
    for name, stage, out_bytes, in_bytes in rows:
        k_s, w_s, p_s = timed(lambda: eng.inter_tu_raw(stage, arr, n_tu, resi, coef, rresi=None if stage == 0 else rresi,
                                                       dist=None if stage == 0 else dist, dist_zero=None if stage == 2 else dz,
                                                       abs_sum=asum if stage == 1 else None), eng, iters, pin=pins)
        cpu = None
        if stage == 1:
            samp = list(range(0, n_tu, 53))

            def work(i):
                j = samp[i]; t = tus[j]
                inter_tu_util.oracle_inter_tu(ito, bd, 1 << t[0], t[1], t[2], t[3], 1, 1, resi[offs[j]:offs[j + 1]])
            sec = cpu_parallel(work, len(samp), threads)
            cpu = {"value": len(samp) / sec, "unit": "TU/s", "cores": threads, "kind": "port",
                   "sample": f"every 53rd TU ({len(samp)}, same size mix) through tests/inter_tu_oracle.c in {sec:.2f} s"}
        emit(name, "TU/s", n_tu, k_s, w_s, in_bytes + out_bytes, cpu,
             {"gpu": gpu, "bit_depth": bd, "samples_per_call": samples, "tus_per_call": n_tu, "luma_tus": sum(1 for t in tus if not t[3]),
              "qp": "32 luma / 31 chroma", "sign_hiding": True},
             p_s=p_s, h2d=int(in_bytes + n_tu * 16), d2h=int(out_bytes))
    eng.close()



def row_f8(cucd, iters=5, threads=8):
    """f8: motion search (cucd_me_search) on the ME part of bench.py's inter workloads: the 42 900 square PUs of a 1920x1080 picture
    (bench.inter_pus), +-64 windows, FEN sub_shift (1 above 8x8), FRAC with Hadamard, lambda = floor(65536 sqrt(0.57 2^((32 - 12) / 3)))
    (QP 32), predictors drawn in +-64 samples.  ldp1080p: 8-bit, one reference; ra1080p10: 10-bit, two references (one call for both).
    Baseline in the same run: the surface route to the same answer (cucd_me_sad_surface + host argmin, cucd_me_subpel_cost + host walk),
    whose results must equal the search's.  f8_me_search_src: +-4 windows with signed keys (cucd_me_search_src) on the same PUs."""
    import bench
    import me_search_util as msu
    R, M = bench.ME_RANGE, bench.ME_MARGIN
    pus = bench.inter_pus(W, H)
    lam = msu.lambda_cost(32)
    mso = msu.load_me_search_oracle()
    gpu = gpu_identity()
    for cfg, bd, nref in (("ldp1080p", 8, 1), ("ra1080p10", 10, 2)):
        org = _util.textured_plane(W, H, bd, seed=81)
        refs = [np.ascontiguousarray(np.pad(_util.pseudo_recon(_util.textured_plane(W, H, bd, seed=82 + k), bd), M, mode="edge")) for k in range(nref)]
        rng = np.random.default_rng(83)
        eng = cucd.Engine(W, H, bit_depth=bd)
        eng.set_cur_picture(org)
        for k, r in enumerate(refs):
            eng.set_ref_picture(k, r, M, M)
        for row, rad, signed in (("f8_me_search", R, False), ("f8_me_search_src", 4, True)):
            descs = []
            for k in range(nref):
                preds = rng.integers(-4 * R, 4 * R + 1, (len(pus), 2))
                descs += [dict(x=x, y=y, w=s, h=s, ref_idx=k, left=-rad, right=rad, top=-rad, bottom=rad, sub_shift=1 if s > 8 else 0, pred_x=int(p[0]),
                               pred_y=int(p[1]), flags=msu.FRAC | msu.HAD, **{"lambda": lam}) for (x, y, s), p in zip(pus, preds)]
            arr, n = cucd.Engine.search_descs(descs)
            res = np.zeros(n, cucd.SEARCH_RESULT)
            src = None
            if signed:
                src = rng.integers(-(1 << bd), 2 << bd, sum(d["w"] * d["h"] for d in descs)).astype(np.int16)
            k_s, w_s, p_s = timed(lambda: eng.me_search_raw(arr, n, res, src), eng, iters, pin=(res,) + ((src,) if signed else ()))
            h2d = n * 56 + (0 if src is None else src.nbytes)
            d2h = n * 24
            # algorithmic bytes: per PU its source block, its (w + 2 rad)^2 reference window, the (w + 9)^2 window of the sub-pel stage,
            # the descriptor and the result
            algo = sum(d["w"] * d["h"] * 2 + (d["w"] + 2 * rad) * (d["h"] + 2 * rad) * 2 + (d["w"] + 9) * (d["h"] + 9) * 2 + 56 + 24 for d in descs)
            # the checker on host threads, every 97th PU
            samp = descs[::97]
            blocks = msu.src_blocks(dict(org=org), samp)
            sc = dict(bd=bd, M=M, refs={k: r for k, r in enumerate(refs)})

            def work(i):
                d = samp[i]
                blk, r = blocks[i], np.zeros(6, np.int32)
                mso.oracle_me_search(bd, P(blk, i16p), d["w"], d["w"], d["h"], msu.ref_base(sc, d), refs[d["ref_idx"]].shape[1], d["left"], d["right"], d["top"],
                                     d["bottom"], d["sub_shift"], d["pred_x"], d["pred_y"], lam, d["flags"], P(r, i32p))
            cpu = None
            if src is None:                 # the signed-key row: the same checker, not timed twice
                sec = cpu_parallel(work, len(samp), threads)
                cpu = {"value": len(samp) / sec, "unit": "PU/s", "cores": threads, "kind": "port",
                       "sample": f"every 97th PU ({len(samp)}) through tests/me_search_oracle.c in {sec:.2f} s"}
            extra = {"gpu": gpu, "config": cfg, "bit_depth": bd, "refs": nref, "pus_per_call": n, "window": f"+-{rad}", "flags": "FRAC|HADAMARD",
                     "lambda": lam, "lambda_note": "floor(65536 sqrt(0.57 2^((QP - 12) / 3))) at QP 32", "signed_keys": signed}
            if not signed:
                extra["surface_route"] = surface_route(cucd, eng, descs, res, R, lam)
            emit(row, "PU/s", n, k_s, w_s, algo, cpu, extra, p_s=p_s, h2d=int(h2d), d2h=int(d2h))
        eng.close()


def surface_route(cucd, eng, descs, res, R, lam):
    """today's route to cucd_me_search's answer, timed once on the wall clock: cucd_me_sad_surface in chunks + numpy argmin of
    sad + cost_2, cucd_me_subpel_cost at the argmin + numpy walk.  Checks that it gives the search's results."""
    import me_search_util as msu
    n = len(descs)
    side = 2 * R + 1
    xs = np.arange(-R, R + 1)
    mv = np.zeros((n, 2), np.int64)
    sad = np.zeros(n, np.int64)
    preds = np.array([(d["pred_x"], d["pred_y"]) for d in descs], np.int64)
    chunk = 4096
    surf = np.zeros(chunk * side * side, np.uint32)
    eng.pin_host_buffer(surf)
    t_gpu = t_host = 0.0
    t0 = time.perf_counter()
    for c0 in range(0, n, chunk):
        part = descs[c0:c0 + chunk]
        arr, m, total = cucd.Engine.me_descs(part)
        ta = time.perf_counter()
        eng.me_sad_surface_raw(arr, m, surf[:total])
        tb = time.perf_counter()
        s = surf[:total].reshape(m, side, side).astype(np.uint64)
        p = preds[c0:c0 + m]
        bits = msu.np_bits(4 * xs[None, :] - p[:, :1])[:, None, :] + msu.np_bits(4 * xs[None, :] - p[:, 1:])[:, :, None]
        cost = ((np.uint64(lam) * bits.astype(np.uint64)) & np.uint64(0xFFFFFFFF)) >> np.uint64(16)
        k = np.argmin((s + cost).reshape(m, -1), axis=1)
        mv[c0:c0 + m, 0] = k % side - R
        mv[c0:c0 + m, 1] = k // side - R
        sad[c0:c0 + m] = s.reshape(m, -1)[np.arange(m), k].astype(np.int64)
        t_gpu += tb - ta
        t_host += time.perf_counter() - tb
    eng.unpin_host_buffer(surf)
    sp = [dict(x=d["x"], y=d["y"], w=d["w"], h=d["h"], ref_idx=d["ref_idx"], mvx=int(m_[0]), mvy=int(m_[1]), use_hadamard=1) for d, m_ in zip(descs, mv)]
    ta = time.perf_counter()
    arr, m = cucd.Engine.subpel_descs(sp)
    T = np.zeros((m, 49), np.uint32)
    eng.me_subpel_cost_raw(arr, m, T)
    tb = time.perf_counter()
    qmv, fc = msu.walk_batch(T, mv, preds, lam)
    t1 = time.perf_counter()
    t_gpu += tb - ta
    t_host += t1 - tb
    want = np.concatenate([mv, sad[:, None], qmv, fc[:, None]], axis=1)
    same = bool(np.array_equal(msu.as_rows(res), want))
    return {"wall_ms": (t1 - t0) * 1e3, "gpu_calls_ms": t_gpu * 1e3, "host_argmin_walk_ms": t_host * 1e3, "d2h_bytes": int(n * side * side * 4 + n * 49 * 4),
            "h2d_bytes": int(n * 40 + n * 32), "round_trips": 2, "results_equal": same}


def row_f9(cucd, iters=5, threads=8):
    """f9: TZ search (cucd_me_tz_search) on the ME part of bench.py's inter workloads: the 42 900 square PUs of a 1920x1080 picture
    (bench.inter_pus), source textured_plane(t=1), references pseudo_recon of t=0 (real (2, 1) motion); ldp1080p 8-bit with one
    reference, ra1080p10 10-bit with two (one call per depth for both).  +-64, FEN sub_shift, FRAC with Hadamard, lambda of QP 32; the
    calls go depth by depth (64, 32, 16, 8): a PU's predictor is its parent's quarter-pel result and its TZ_2NX2N start its parent's
    integer result (depth 0: predictor (0, 0), no 2Nx2N start).  Box = the legal area of the 80-sample margin, window = xSetSearchRange
    around the predictor.  Times are summed over the four calls.  In the same run: HM's probes per PU and the kernel's evaluated points
    (checker and CPU replay on every 97th PU), the checker's rate on host threads, the surface route to the same answers (cucd_me_sad_surface
    over the bounding box of each PU's probes, the checker's walk on it, cucd_me_subpel_cost + host walk; must be equal) and
    cucd_me_search +-64 on the same PUs and windows, for scale."""
    import bench
    import me_search_util as msu
    import me_tz_util as mtu
    R, M = bench.ME_RANGE, bench.ME_MARGIN
    pus = bench.inter_pus(W, H)
    lam = msu.lambda_cost(32)
    tz = mtu.load_me_tz_oracle()
    emul = mtu.load_me_tz_emul()
    gpu = gpu_identity()
    for cfg, bd, nref in (("ldp1080p", 8, 1), ("ra1080p10", 10, 2)):
        org = _util.textured_plane(W, H, bd, seed=91, t=1)
        refs = [np.ascontiguousarray(np.pad(_util.pseudo_recon(_util.textured_plane(W, H, bd, seed=91, t=0), bd, seed=92 + k), M, mode="edge"))
                for k in range(nref)]
        sc = dict(bd=bd, W=W, H=H, M=M, org=org, refs={k: r for k, r in enumerate(refs)})
        eng = cucd.Engine(W, H, bit_depth=bd)
        eng.set_cur_picture(org)
        for k, r in enumerate(refs):
            eng.set_ref_picture(k, r, M, M)
        # one pass depth by depth builds every depth's descriptors from its parents' results
        parent = {}
        depths = []
        for size in (64, 32, 16, 8):
            descs = []
            for k in range(nref):
                for x, y, s in pus:
                    if s != size:
                        continue
                    p = parent.get((k, x & ~(2 * s - 1), y & ~(2 * s - 1), 2 * s))
                    pred = (0, 0) if p is None else (p[3], p[4])
                    fl = msu.FRAC | msu.HAD | (0 if p is None else mtu.TZ2N)
                    descs.append(mtu.tz_desc(sc, x, y, s, s, k, pred, R, sub_shift=1 if s > 8 else 0, lam=lam, flags=fl,
                                             mv2n=(0, 0) if p is None else (p[0], p[1])))
            arr = cucd.Engine.tz_descs(descs)
            res = np.zeros(len(arr), cucd.SEARCH_RESULT)
            eng.me_tz_search_raw(arr, res)
            for d, r in zip(descs, res):
                parent[(d["ref_idx"], d["x"], d["y"], d["w"])] = tuple(int(r[f]) for f in ("mvx", "mvy", "sad", "qmvx", "qmvy"))
            depths.append((descs, arr, res))
        n = sum(len(a) for _, a, _ in depths)
        k_s = w_s = p_s = 0.0
        direct = []
        for _, arr, res in depths:
            try:
                k1, w1, p1 = timed(lambda: eng.me_tz_search_raw(arr, res), eng, iters, pin=(res,))
            except cucd.CucdError:            # a call small enough for the zero-copy path is not timed: its call time stands for the kernel
                direct.append(len(arr))
                ws = []
                for _ in range(iters):
                    t0 = time.perf_counter()
                    eng.me_tz_search_raw(arr, res)
                    ws.append(time.perf_counter() - t0)
                k1 = w1 = p1 = float(np.median(ws))
            k_s, w_s, p_s = k_s + k1, w_s + w1, p_s + p1
        descs = [d for ds, _, _ in depths for d in ds]
        got = np.concatenate([msu.as_rows(r) for _, _, r in depths])
        # cucd_me_search over the same windows, for scale
        sarr, sn = cucd.Engine.search_descs([dict(d, flags=msu.FRAC | msu.HAD) for d in descs])
        sres = np.zeros(sn, cucd.SEARCH_RESULT)
        fk, fw, _ = timed(lambda: eng.me_search_raw(sarr, sn, sres), eng, iters, pin=(sres,))
        # HM's probes (checker) and the kernel's evaluated points (CPU replay) on a sample; the checker's rate on host threads
        samp = descs[::97]
        probes, raster, evals, first_hm, first_all = [], [], [], [], []
        for d in samp:
            _, tr, cnt = mtu.oracle_tz(tz, sc, d, trace_cap=20000)
            probes.append(cnt)
            raster.append(int((tr[:, 4] == 3).sum()))
            first_hm.append(int((tr[:, 4] == 1).sum()))
            first_all.append(first_search_points(mtu, d, tr))
            res6 = np.zeros(6, np.int32)
            tr2 = np.zeros((20000, 6), np.int32)
            ev, g = np.zeros(1, np.int32), np.zeros(1, np.int32)
            blk = mtu.src_block(sc, d)
            emul.emul_me_tz_search(bd, P(blk, i16p), d["w"], mtu.ref_base(sc, d), refs[d["ref_idx"]].shape[1], P(mtu.desc_row(d), i32p), P(res6, i32p),
                                   tr2.ctypes.data, 20000, ev.ctypes.data, g.ctypes.data)
            evals.append(int(ev[0]))

        def work(i):
            mtu.oracle_tz(tz, sc, samp[i])
        sec = cpu_parallel(work, len(samp), threads)
        cpu = {"value": len(samp) / sec, "unit": "PU/s", "cores": threads, "kind": "port",
               "sample": f"every 97th PU ({len(samp)}) through tests/me_tz_oracle.c in {sec:.2f} s"}
        h2d = n * (16 + 20 + 4 + 48) + sum(4 * (len(a) // 4 + 2) for _, a, _ in depths)
        d2h = n * 24
        # algorithmic bytes: per PU its source block, the reference block of every HM probe (sample mean), the sub-pel window, the records
        mean_probes = float(np.mean(probes))
        algo = int(sum(d["w"] * d["h"] * 2 * (1 + mean_probes) + (d["w"] + 9) * (d["h"] + 9) * 2 + 88 + 24 for d in descs))
        extra = {"gpu": gpu, "config": cfg, "bit_depth": bd, "refs": nref, "pus_per_call": n, "calls": 4, "window": f"+-{R}", "flags": "FRAC|HADAMARD (+TZ_2NX2N below depth 0)",
                 "lambda": lam, "lambda_note": "floor(65536 sqrt(0.57 2^((QP - 12) / 3))) at QP 32",
                 "hm_probes_per_pu": {"mean": mean_probes, "max": int(max(probes)), "raster_share": float(sum(raster) / max(1, sum(probes))),
                                      "sample": len(samp)},
                 "kernel_points_per_pu": {"mean": float(np.mean(evals)), "over_hm": float(sum(evals) / max(1, sum(probes))),
                                          "first_search_hm_mean": float(np.mean(first_hm)), "first_search_all_distances_mean": float(np.mean(first_all))},
                 "zero_copy_calls_pus": direct, "zero_copy_note": "calls on the zero-copy path are not timed: their call time is counted as kernel time",
                 "me_search_same_pus": {"kernel_ms": fk * 1e3, "e2e_ms": fw * 1e3},
                 "surface_route": tz_surface_route(cucd, eng, tz, mtu, msu, sc, descs, got, threads)}
        emit("f9_me_tz_search", "PU/s", n, k_s, w_s, algo, cpu, extra, p_s=p_s, h2d=int(h2d), d2h=int(d2h))
        eng.close()


def first_search_points(mtu, d, tr):
    """points the first search would probe if all its distances were evaluated at once (guards applied, no three-round stop)"""
    st0 = tr[tr[:, 4] == 0]
    cx, cy = (int(v) for v in st0[int(np.argmin(st0[:, 5])), :2])      # argmin: the first of equal values, as the strict '<'
    cnt, D = 0, 1
    while D <= d["search_range"]:
        for dx, dy, _, _ in mtu._diamond_points(D):
            x, y = cx + dx, cy + dy
            cnt += (dx >= 0 or x >= d["left"]) and (dx <= 0 or x <= d["right"]) and (dy >= 0 or y >= d["top"]) and (dy <= 0 or y <= d["bottom"])
        D *= 2
    return cnt


def tz_surface_route(cucd, eng, tz, mtu, msu, sc, descs, got, threads):
    """the surface route to cucd_me_tz_search's answer: cucd_me_sad_surface over the bounding box of each PU's probes (from the
    checker's trace), the checker's walk on that surface on host threads, cucd_me_subpel_cost at its result and the host walk"""
    n = len(descs)
    boxes = [None] * n

    def trace(i):
        tr = mtu.oracle_tz(tz, sc, descs[i], trace_cap=20000)[1]
        boxes[i] = (int(tr[:, 0].min()), int(tr[:, 0].max()), int(tr[:, 1].min()), int(tr[:, 1].max()))
    cpu_parallel(trace, n, threads)
    ints = np.zeros((n, 3), np.int64)
    t_gpu = t_host = 0.0
    t0 = time.perf_counter()
    chunk = 2048
    for c0 in range(0, n, chunk):
        part = [dict(d, left=b[0], right=b[1], top=b[2], bottom=b[3]) for d, b in zip(descs[c0:c0 + chunk], boxes[c0:c0 + chunk])]
        arr, m, total = cucd.Engine.me_descs(part)
        surf = np.zeros(total, np.uint32)
        ta = time.perf_counter()
        eng.me_sad_surface_raw(arr, m, surf)
        tb = time.perf_counter()
        offs = np.cumsum([0] + [(d["right"] - d["left"] + 1) * (d["bottom"] - d["top"] + 1) for d in part])

        def walk(i):
            d = part[i]
            s = surf[offs[i]:offs[i + 1]].reshape(d["bottom"] - d["top"] + 1, d["right"] - d["left"] + 1)
            r = mtu.oracle_tz(tz, {"bd": sc["bd"]}, dict(descs[c0 + i], flags=descs[c0 + i]["flags"] & mtu.TZ2N), surface=(s, d["left"], d["top"]))[0]
            ints[c0 + i] = r[:3]
        cpu_parallel(walk, m, threads)
        t_gpu += tb - ta
        t_host += time.perf_counter() - tb
    sp = [dict(x=d["x"], y=d["y"], w=d["w"], h=d["h"], ref_idx=d["ref_idx"], mvx=int(r[0]), mvy=int(r[1]), use_hadamard=1) for d, r in zip(descs, ints)]
    ta = time.perf_counter()
    arr, m = cucd.Engine.subpel_descs(sp)
    T = np.zeros((m, 49), np.uint32)
    eng.me_subpel_cost_raw(arr, m, T)
    tb = time.perf_counter()
    preds = np.array([(d["pred_x"], d["pred_y"]) for d in descs], np.int64)
    qmv, fc = msu.walk_batch(T, ints[:, :2], preds, descs[0]["lambda"])
    t1 = time.perf_counter()
    t_gpu += tb - ta
    t_host += t1 - tb
    want = np.concatenate([ints, qmv, fc[:, None]], axis=1)
    return {"wall_ms": (t1 - t0) * 1e3, "gpu_calls_ms": t_gpu * 1e3, "host_walks_ms": t_host * 1e3,
            "d2h_bytes": int(sum((b[1] - b[0] + 1) * (b[3] - b[2] + 1) for b in boxes) * 4 + n * 49 * 4), "results_equal": bool(np.array_equal(got, want)),
            "pus_equal": int((got == want).all(axis=1).sum()), "pus": n}


if __name__ == "__main__":
    main()
