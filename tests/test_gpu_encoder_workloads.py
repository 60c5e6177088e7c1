"""The workloads of tests/test_gpu_encoder_md5.py without the reference encoder.  That module encodes with HM binaries built
from the reference's sources (oracle/_ref), which a checkout does not contain.  Here the same clips (gen_golden.synth_clip:
same sizes, bit depths, picture counts and seeds) go through the entry points the integrated encoder calls - the frame
features and rough-mode-decision tables, integer-ME SAD surfaces over the +-64 TZ window, the 49-point sub-pel tables (with
the bi-predictive key for random access), the TU coding chain, texture features, and cucd_server shared by three client
processes - and every answer must equal the oracle's (pinned to the reference by tests/test_oracle_golden.py and
tests/test_oracle_vs_ref.py).  With no encoder there is no reconstruction: _util.pseudo_recon of each picture stands in for
it, as the neighbours of the intra search and as the reference picture of the next picture."""
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import pytest

from _util import (P, i16p, u32p, all_cus, oracle_aq_activity, oracle_cu_sums, oracle_intra_tu, oracle_outlier_frame, oracle_rmd_frame,
                   oracle_tmv_features, pseudo_recon)

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
M = 80          # TComPicYuv margin


def luma_planes(W, H, frames, bd, seed):
    import gen_golden as gg
    clip = np.frombuffer(gg.synth_clip(W, H, frames, bd, seed), np.uint8 if bd == 8 else "<u2")
    per = W * H * 3 // 2
    return [clip[t * per: t * per + W * H].reshape(H, W).astype(np.int16) for t in range(frames)]


def check_frame(eng, oracle, org, rec, bd, ctus=None):
    """features + RMD tables of one picture against the oracle (every CTU, or the given subset)"""
    H, W = org.shape
    out = eng.frame(org, rec)
    obf, outl, yc = oracle_outlier_frame(oracle, org, bd)
    assert np.array_equal(out["obf"], obf) and np.array_equal(out["outlier"], outl) and np.array_equal(out["yc"][1:], yc[1:])
    for d in range(4):
        num, tot = oracle_cu_sums(oracle, obf, W, H, d)
        assert np.array_equal(out[f"num_obf{d}"], num) and np.array_equal(out[f"n_outlier{d}"], tot), d
    for c in (range(eng.ctus_per_pic) if ctus is None else ctus):
        assert np.array_equal(out["rmd_cost"][c], oracle_rmd_frame(oracle, org, rec, bd, ctu_begin=c, ctu_end=c + 1)[0]), c


def check_inter(eng, oracle, cur, refs, bd, rng, n_pu):
    """integer-ME surfaces over the full +-64 window and sub-pel tables of sampled square PUs against every reference picture;
    with two references (random access) also the bi-predictive search key 2 * org - prediction of the other list"""
    H, W = cur.shape
    padded = [np.ascontiguousarray(np.pad(r, M, mode="edge")) for r in refs]
    eng.set_cur_picture(cur)
    for k, p in enumerate(padded):
        eng.set_ref_picture(k, p, M, M)
    S = W + 2 * M
    pus = []
    for _ in range(n_pu):
        s = int(rng.choice([64, 32, 16, 8]))
        pus.append((int(rng.integers(0, (W - s) // s + 1)) * s, int(rng.integers(0, (H - s) // s + 1)) * s, s))
    for k, p in enumerate(padded):
        me = [dict(x=x, y=y, w=s, h=s, ref_idx=k, left=-64, right=64, top=-64, bottom=64, sub_shift=1 if s > 8 else 0) for x, y, s in pus]
        sp = [dict(x=x, y=y, w=s, h=s, ref_idx=k, mvx=int(rng.integers(-40, 41)), mvy=int(rng.integers(-40, 41)), use_hadamard=1) for x, y, s in pus]
        surf, frac = eng.me_sad_surface(me), eng.me_subpel_cost(sp)
        key = None
        if len(padded) == 2:
            other = refs[1 - k].astype(np.int32)
            key = [np.ascontiguousarray((2 * cur[y:y + s, x:x + s].astype(np.int32) - other[y:y + s, x:x + s]).astype(np.int16)) for x, y, s in pus]
            me_bi = [dict(d, left=-4, right=4, top=-4, bottom=4) for d in me]
            surf_bi = eng.me_sad_surface(me_bi, src=np.concatenate([b.ravel() for b in key]))
            frac_bi = eng.me_subpel_cost(sp, src=np.concatenate([b.ravel() for b in key]))
        for i, (x, y, s) in enumerate(pus):
            zero = C.c_void_p(p.ctypes.data + 2 * ((y + M) * S + x + M))
            blocks = [(np.ascontiguousarray(cur[y:y + s, x:x + s]), me[i], surf[i], frac[i])]
            if key is not None:
                blocks.append((key[i], me_bi[i], surf_bi[i], frac_bi[i]))
            for blk, d, got, got49 in blocks:
                want = np.zeros_like(got)
                oracle.oracle_sad_surface(bd, P(blk, i16p), s, s, s, zero, S, d["left"], d["right"], d["top"], d["bottom"], d["sub_shift"], P(want, u32p))
                assert np.array_equal(got, want), (k, d)
                want49 = np.zeros(49, np.uint32)
                oracle.oracle_subpel_surface(bd, P(blk, i16p), s, s, s, zero, S, sp[i]["mvx"], sp[i]["mvy"], 1, P(want49, u32p))
                assert np.array_equal(got49.ravel(), want49), (k, sp[i])


def check_tus(eng, oracle, org, rec, bd, qp, rng):
    """the TU coding chain (cucd_intra_tu_code) on luma TUs of every size and 4x4 chroma blocks taken from the picture"""
    H, W = org.shape
    tus, orgs, brds, want = [], [], [], []
    for i in range(120):
        chroma = int(i % 6 == 5)
        l = 2 if chroma else int(rng.integers(2, 6))
        n = 1 << l
        x, y = int(rng.integers(1, (W - n) // n)) * n, int(rng.integers(1, (H - n) // n)) * n
        mode, ts = int(rng.integers(0, 35)), int(n == 4 and rng.integers(0, 2))
        o = np.ascontiguousarray(org[y:y + n, x:x + n]).ravel()
        left = rec[y:y + 2 * n, x - 1][::-1] if y + 2 * n <= H else np.full(2 * n, rec[y, x - 1], np.int16)
        top = rec[y - 1, x:x + 2 * n] if x + 2 * n <= W else np.full(2 * n, rec[y - 1, x], np.int16)
        b = np.concatenate([left, [rec[y - 1, x - 1]], top]).astype(np.int16)
        tus.append((l, mode, qp, ts, chroma)); orgs.append(o); brds.append(b)
        want.append(oracle_intra_tu(oracle, bd, n, mode, qp, ts, o, b, 1, chroma=chroma))
    level, reco, dist, abs_sum = eng.intra_tu_code(tus, np.concatenate(orgs), np.concatenate(brds))
    assert np.array_equal(level, np.concatenate([w["level"] for w in want]))
    assert np.array_equal(reco, np.concatenate([w["reco"] for w in want]))
    assert list(dist) == [w["dist"] for w in want] and list(abs_sum) == [w["abs_sum"] for w in want]


@pytest.mark.parametrize("cfg,bd,frames,qp", [("AI", 8, 5, 32), ("AI", 10, 2, 27), ("LDP", 8, 3, 32), ("RA", 10, 9, 32), ("AITU", 8, 1, 32), ("AITU", 10, 1, 27)])
def test_encoder_clip_through_the_entry_points(cucd, oracle, cfg, bd, frames, qp):
    """the 416x240 clips of test_bitstream_md5_matches_reference_encoder: every picture's frame outputs in full; LDP (I + P
    pictures, one reference) and RA (GOP8 B pictures, the pictures on either side as the two references) add ME and sub-pel;
    AITU adds the TU coding chain at the clip's QP; 8-bit AI adds the texture features and AQ activity of every picture"""
    W, H = 416, 240
    orgs = luma_planes(W, H, frames, bd, 20261030 + bd)
    recs = [pseudo_recon(o, bd, seed=t) for t, o in enumerate(orgs)]
    rng = np.random.default_rng(frames * 100 + bd)
    with cucd.Engine(W, H, bit_depth=bd) as eng:
        for t, (org, rec) in enumerate(zip(orgs, recs)):
            check_frame(eng, oracle, org, rec, bd)
            if cfg == "LDP" and t > 0:
                check_inter(eng, oracle, org, [recs[t - 1]], bd, rng, 24)
            if cfg == "RA" and 0 < t < frames - 1:
                check_inter(eng, oracle, org, [recs[t - 1], recs[t + 1]], bd, rng, 12)
            if cfg == "AITU":
                check_tus(eng, oracle, org, rec, bd, qp, rng)
            if cfg == "AI" and bd == 8:
                eng.set_cur_picture(org)
                cus = all_cus(W, H)[t::5]
                assert np.array_equal(eng.tmv_features(cus), oracle_tmv_features(oracle, org, cus))
                acts, avg = eng.aq_activity(4)
                wacts, wavg = oracle_aq_activity(oracle, org, 4)
                assert all(np.array_equal(a, b) for a, b in zip(acts, wacts)) and np.array_equal(avg, wavg)


def _fullsize_cases():
    return sorted(json.load(open(os.path.join(ROOT, "tests", "golden", "encoder_md5.json"))).items())


@pytest.mark.parametrize("name,ref", _fullsize_cases(), ids=[n for n, _ in _fullsize_cases()])
def test_fullsize_clip_through_the_entry_points(cucd, oracle, name, ref):
    """the BASELINE-size clips of test_fullsize_bitstream_md5_matches_recorded_reference: the first picture's features in full and
    its RMD tables on corner, edge (partial bottom row at 1080p) and seeded interior CTUs; LDP / RA: the second picture's ME
    surfaces over the full +-64 window and sub-pel tables at real picture size (RA with the bi-predictive key)"""
    W, H, bd = ref["width"], ref["height"], ref["bit_depth"]
    inter = ref["structure"] != "AI"
    orgs = luma_planes(W, H, 3 if ref["structure"] == "RA" else 2 if inter else 1, bd, ref["seed"])
    recs = [pseudo_recon(o, bd, seed=t) for t, o in enumerate(orgs)]
    rng = np.random.default_rng(ref["seed"])
    with cucd.Engine(W, H, bit_depth=bd) as eng:
        wc, nctu = eng.ctus_per_row, eng.ctus_per_pic
        subset = sorted(set([0, wc - 1, nctu - wc, nctu - 1] + [int(c) for c in rng.integers(0, nctu, 8)]))
        check_frame(eng, oracle, orgs[0], recs[0], bd, subset)
        if inter:
            check_inter(eng, oracle, orgs[1], [recs[0]] + recs[2:], bd, rng, 16)


def test_three_client_processes_through_cucd_server(oracle, tmp_path):
    """the set-up of test_three_encoder_instances_through_cucd_server_stay_byte_identical with the encoders replaced by
    tests/ipc_replay.cpp (the header-only client of include/cucd_ipc.h): three processes - All-Intra 8 bit, low-delay P 8 bit,
    All-Intra 10 bit on the same clips - share the GPU through cucd_server.  Their one-PU rough-mode-decision requests must be
    coalesced into common batches, and every answer (features, RMD costs, ME surfaces, sub-pel tables) must equal the oracle's."""
    server = os.path.join(ROOT, "fast-cu-decision-hevc_b200", "cucd_server")
    assert os.path.exists(server), "cucd_server not built"
    exe = str(tmp_path / "ipc_replay")
    subprocess.run(["g++", "-std=c++17", "-O2", "-I" + os.path.join(ROOT, "include"), "-o", exe, os.path.join(ROOT, "tests", "ipc_replay.cpp"), "-lrt"],
                   check=True, capture_output=True)
    W, H = 416, 240
    jobs = [(8, 3, False), (8, 3, True), (10, 2, False)]
    want, files = [], []
    for i, (bd, frames, inter) in enumerate(jobs):
        orgs = luma_planes(W, H, frames, bd, 20261300 + i)
        rng = np.random.default_rng(i)
        pus = [(int(rng.integers(1, 416 // (1 << l) - 1)) << l, int(rng.integers(1, 240 // (1 << l) - 1)) << l, l) for l in map(int, rng.integers(2, 6, 400))]
        rec = pseudo_recon(orgs[0], bd)
        porg = [np.ascontiguousarray(orgs[0][y:y + (1 << l), x:x + (1 << l)]).ravel() for x, y, l in pus]
        pbrd = [np.concatenate([rec[y:y + (2 << l), x - 1][::-1] if y + (2 << l) <= H else np.full(2 << l, rec[y, x - 1]), [rec[y - 1, x - 1]],
                                rec[y - 1, x:x + (2 << l)] if x + (2 << l) <= W else np.full(2 << l, rec[y - 1, x])]).astype(np.int16) for x, y, l in pus]
        me = [(x, y, 1 << l, 1 << l, 0, -64, 64, -64, 64, 1 if l > 3 else 0) for x, y, l in pus[:20] if l >= 3] if inter else []
        sp = [(d[0], d[1], d[2], d[3], 0, int(rng.integers(-30, 31)), int(rng.integers(-30, 31)), 1) for d in me]
        refp = np.ascontiguousarray(np.pad(rec, M, mode="edge"))
        hdr = np.array([W, H, bd, frames, len(pus), sum(a.size for a in porg), sum(b.size for b in pbrd), len(me), len(sp), M], np.int32)
        path = str(tmp_path / f"job{i}.bin")
        with open(path, "wb") as f:
            for a in [hdr] + orgs + [np.array([l for _, _, l in pus], np.int32)] + porg + pbrd + ([refp] if me else []):
                f.write(np.ascontiguousarray(a).tobytes())
            f.write(np.array(me, np.int32).tobytes() + np.array(sp, np.int32).tobytes())
        files.append(path)
        w = [a for o in orgs for a in oracle_outlier_frame(oracle, o, bd)[:2]]
        for o, b, (x, y, l) in zip(porg, pbrd, pus):
            r = np.zeros(35, np.uint32)
            oracle.oracle_rmd_pu(bd, 1 << l, 1, P(o, i16p), 1 << l, P(b, i16p), P(r, u32p))
            w.append(r)
        S = W + 2 * M
        for d, s in zip(me, sp):
            blk = np.ascontiguousarray(orgs[1][d[1]:d[1] + d[3], d[0]:d[0] + d[2]])
            zero = C.c_void_p(refp.ctypes.data + 2 * ((d[1] + M) * S + d[0] + M))
            r = np.zeros(129 * 129, np.uint32)
            oracle.oracle_sad_surface(bd, P(blk, i16p), d[2], d[2], d[3], zero, S, -64, 64, -64, 64, d[9], P(r, u32p))
            r49 = np.zeros(49, np.uint32)
            oracle.oracle_subpel_surface(bd, P(blk, i16p), s[2], s[2], s[3], zero, S, s[5], s[6], 1, P(r49, u32p))
            w += [r, r49]
        want.append(w)
    name = f"/cucd_test_{os.getpid()}"
    srv = subprocess.Popen([server, "--name", name, "--clients", str(len(jobs))], stdout=subprocess.PIPE, text=True)
    procs = []
    try:
        time.sleep(1.0)
        procs = [subprocess.Popen([exe, name, f, f + ".out"], stderr=subprocess.PIPE, text=True) for f in files]
        errs = [p.communicate(timeout=600)[1] for p in procs]
        for p, e in zip(procs, errs):
            assert p.returncode == 0, e[-1500:]
        stats = json.loads(srv.communicate(timeout=60)[0].strip().splitlines()[-1])
    finally:
        for p in procs + [srv]:
            if p.poll() is None:
                p.kill()
                p.wait()
    assert stats["closed"] == 3 and stats["frames"] == 8 and stats["rmd_requests"] == 1200 and stats["me_surfaces"] > 0 and stats["subpel"] > 0
    assert stats["rmd_batches"] < stats["rmd_requests"]            # requests of different processes really shared batches
    for f, w in zip(files, want):
        got = np.fromfile(f + ".out", np.uint8)
        off = 0
        for a in w:
            n = a.nbytes
            assert np.array_equal(got[off:off + n].view(a.dtype), a.ravel()), (f, off)
            off += n
        assert off == got.size
