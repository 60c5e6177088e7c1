"""cucd_me_mc_chroma through the C ABI (and through cucd_server) against the checker tests/mc_chroma_oracle.c: 4:2:0 chroma motion
compensation of uni- and bi-predictive inter candidates and the SSE of each plane, samples and sums.  Integer work: bit-exact."""
import json
import os
import subprocess
import time

import numpy as np
import pytest

from _util import ROOT
from mc_chroma_util import load_mc_chroma_oracle, mcc_candidates, mcc_scene, oracle_mc_chroma
from mc_util import MC_SHAPES

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def mco():
    return load_mc_chroma_oracle()


def engine(cucd, sc):
    eng = cucd.Engine(sc["W"], sc["H"], bit_depth=sc["bd"])
    eng.set_cur_picture(sc["org"])
    eng.set_cur_picture_chroma(*sc["org_c"])
    for s, p in sc["refs"].items():
        eng.set_ref_picture(s, p, sc["M"], sc["M"])
        eng.set_ref_picture_chroma(s, *sc["refs_c"][s], sc["Mc"], sc["Mc"])
    return eng


def assert_equal(descs, got_s, got_p, want_s, want_p):
    for i, d in enumerate(descs):
        for c in range(2):
            assert np.array_equal(got_p[i][c], want_p[i][c]), (d, c)
        assert np.array_equal(got_s[i], want_s[i]), d


@pytest.mark.parametrize("bd", [8, 9, 10])
def test_mc_chroma_vs_oracle_mixed_batch_and_single_candidates(cucd, mco, bd):
    """the coverage of test_emulation_mc_chroma.py: the chroma blocks of 22 PU shapes x (uni L0, uni L1, bi, bi with identical
    motion), random and extreme eighth-pel fractions, supports at the chroma margin's corners; in one mixed batch and one per call"""
    sc = mcc_scene(bd, seed=bd)
    rng = np.random.default_rng(bd + 1)
    descs = mcc_candidates(sc, rng) + mcc_candidates(sc, rng) + mcc_candidates(sc, rng)
    rng.shuffle(descs)
    want_s, want_p = oracle_mc_chroma(mco, sc, descs)
    with engine(cucd, sc) as eng:
        got_s, got_p = eng.me_mc_chroma(descs, want_pred=True)
        assert_equal(descs, got_s, got_p, want_s, want_p)
        assert np.array_equal(eng.me_mc_chroma(descs), got_s)                 # pred = NULL: the same sums
        for i, d in enumerate(descs):
            s1, p1 = eng.me_mc_chroma([d], want_pred=True)
            assert_equal([d], s1, p1, want_s[i:i + 1], want_p[i:i + 1])


@pytest.mark.parametrize("bd", [8, 10])
def test_mc_chroma_large_batch_spans_several_waves(cucd, mco, bd):
    """>= 10 000 candidates of mixed shapes and modes; every 7th is checked in full against the oracle, all against the single-shape
    batches of the same candidates"""
    sc = mcc_scene(bd, W=416, H=240, seed=50 + bd)
    rng = np.random.default_rng(bd + 3)
    descs = []
    while len(descs) < 10500:
        descs += mcc_candidates(sc, rng, shapes=[MC_SHAPES[int(i)] for i in rng.integers(0, 22, 6)] + [(8, 8), (16, 16), (4, 8)])
    with engine(cucd, sc) as eng:
        got_s, got_p = eng.me_mc_chroma(descs, want_pred=True)
        samp = list(range(0, len(descs), 7))
        want_s, want_p = oracle_mc_chroma(mco, sc, [descs[i] for i in samp])
        assert_equal([descs[i] for i in samp], got_s[samp], [got_p[i] for i in samp], want_s, want_p)
        assert np.array_equal(eng.me_mc_chroma(descs), got_s)
        assert eng.last_kernel_time_ms() > 0
        by_shape = {}
        for i, d in enumerate(descs):
            by_shape.setdefault((d["w"], d["h"]), []).append(i)
        for idx in by_shape.values():
            assert np.array_equal(eng.me_mc_chroma([descs[i] for i in idx]), got_s[idx])


@pytest.mark.parametrize("bd", [8, 10])
def test_mc_chroma_lists_on_the_same_and_on_different_slots(cucd, mco, bd):
    """bi on one slot and on two slots in either order; uni on list 0 and on list 1 of each slot: a motion on list 1 predicts what
    the same motion on list 0 predicts"""
    sc = mcc_scene(bd, seed=70 + bd, slots=(2, 5))
    descs = []
    for r0, r1 in ((2, 2), (5, 5), (2, 5), (5, 2)):
        for w, h in ((16, 16), (4, 8), (24, 32)):
            descs.append(dict(x=48, y=32, w=w, h=h, ref_idx=(r0, r1), mvx=(-37, 22), mvy=(13, -54), use_hadamard=1))
            descs.append(dict(x=48, y=32, w=w, h=h, ref_idx=(r0, -1), mvx=(-37, 0), mvy=(13, 0), use_hadamard=0))
            descs.append(dict(x=48, y=32, w=w, h=h, ref_idx=(-1, r0), mvx=(0, -37), mvy=(0, 13), use_hadamard=0))
    want_s, want_p = oracle_mc_chroma(mco, sc, descs)
    with engine(cucd, sc) as eng:
        got_s, got_p = eng.me_mc_chroma(descs, want_pred=True)
    assert_equal(descs, got_s, got_p, want_s, want_p)
    for i in range(0, len(descs), 3):
        assert np.array_equal(got_s[i + 1], got_s[i + 2]) and all(np.array_equal(got_p[i + 1][c], got_p[i + 2][c]) for c in range(2))
    assert not np.array_equal(got_p[0][0], got_p[2 * 9][0])            # the slots hold different pictures


def test_mc_chroma_stale_planes(cucd, mco):
    """setting a slot's luma unsets its chroma, setting the current luma unsets the current chroma; the calls fail until the chroma is
    set again, and the luma call is not affected"""
    sc = mcc_scene(8, seed=5)
    d = [dict(x=16, y=16, w=16, h=8, ref_idx=(0, 3), mvx=(5, -7), mvy=(2, 9), use_hadamard=1)]
    want, _ = oracle_mc_chroma(mco, sc, d)
    with engine(cucd, sc) as eng:
        assert np.array_equal(eng.me_mc_chroma(d), want)
        eng.set_ref_picture(3, sc["refs"][3], sc["M"], sc["M"])
        with pytest.raises(cucd.CucdError, match="chroma of the reference picture not set"):
            eng.me_mc_chroma(d)
        assert eng.me_mc_cost(d).shape == (1,)
        eng.set_ref_picture_chroma(3, *sc["refs_c"][3], sc["Mc"], sc["Mc"])
        assert np.array_equal(eng.me_mc_chroma(d), want)
        eng.set_cur_picture(sc["org"])
        with pytest.raises(cucd.CucdError, match="cucd_set_cur_picture_chroma"):
            eng.me_mc_chroma(d)
        assert eng.me_mc_cost(d).shape == (1,)
        eng.set_cur_picture_chroma(*sc["org_c"])
        assert np.array_equal(eng.me_mc_chroma(d), want)


def test_destroy_releases_the_chroma_planes(cucd):
    """cucd_destroy frees the chroma planes and tables: handles that set eight 1080p reference slots' chroma (about 23 MB of device
    memory each, more in allocation pages) come and go without the device's free memory shrinking"""
    import torch
    W, H, Mc = 1920, 1080, 40
    cb = np.zeros((H // 2 + 2 * Mc, W // 2 + 2 * Mc), np.int16)
    cur = np.zeros((H // 2, W // 2), np.int16)
    d = [dict(x=64, y=64, w=16, h=16, ref_idx=(0, 7), mvx=(3, -5), mvy=(7, 2), use_hadamard=0)]

    def cycle():
        with cucd.Engine(W, H, bit_depth=8) as eng:
            for s in range(8):
                eng.set_ref_picture_chroma(s, cb, cb, Mc, Mc)
            eng.set_cur_picture_chroma(cur, cur)
            assert eng.me_mc_chroma(d).shape == (1, 2)
    for _ in range(2):
        cycle()
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info(0)[0]
    for _ in range(30):                                                     # a leak would lose > 680 MB
        cycle()
    torch.cuda.synchronize()
    assert free0 - torch.cuda.mem_get_info(0)[0] < 128 << 20


def test_mc_chroma_rejections_and_empty_batch(cucd):
    sc = mcc_scene(8, seed=3)
    W, H, M, Mc = sc["W"], sc["H"], sc["M"], sc["Mc"]
    Wc, Hc = W // 2, H // 2
    ok = dict(x=16, y=16, w=16, h=16, ref_idx=(0, 3), mvx=(5, -7), mvy=(2, 9), use_hadamard=1)
    with cucd.Engine(W, H, bit_depth=8) as eng:
        eng.set_cur_picture(sc["org"])
        with pytest.raises(cucd.CucdError, match="cucd_set_cur_picture_chroma"):
            eng.me_mc_chroma([ok])
        eng.set_cur_picture_chroma(*sc["org_c"])
        for s in (0, 3):
            eng.set_ref_picture(s, sc["refs"][s], M, M)
        with pytest.raises(cucd.CucdError, match="chroma of the reference picture not set"):
            eng.me_mc_chroma([ok])                                        # luma set, chroma not
        eng.set_ref_picture_chroma(0, *sc["refs_c"][0], Mc, Mc)
        with pytest.raises(cucd.CucdError, match="chroma of the reference picture not set"):
            eng.me_mc_chroma([ok])                                        # slot 3 still without chroma
        eng.set_ref_picture_chroma(3, *sc["refs_c"][3], Mc, Mc)
        assert eng.me_mc_chroma([ok]).shape == (1, 2)
        s, p = eng.me_mc_chroma([], want_pred=True)
        assert s.shape == (0, 2) and p == []
        # the support of a 16x16 PU at (16, 16): chroma block (8, 8, 8, 8); integer chroma MV i is inside for 1 - Mc - 8 <= i <= Wc - 2 + Mc - 16
        lo, hx, hy = 1 - Mc - 8, Wc - 2 + Mc - 16, Hc - 2 + Mc - 16
        bad = [dict(ok, w=6), dict(ok, h=2), dict(ok, w=68), dict(ok, h=66), dict(ok, x=-4), dict(ok, y=H - 8), dict(ok, x=W - 12),
               dict(ok, ref_idx=(-1, -1)), dict(ok, ref_idx=(0, 64)), dict(ok, ref_idx=(7, -1)),
               dict(ok, mvx=(8 * (lo - 1) + 7, 0)),                   # left edge of the support one sample outside, list 0
               dict(ok, mvx=(0, 8 * (hx + 1))),                       # right edge, list 1
               dict(ok, mvy=(8 * (lo - 1) + 7, 0)),                   # top
               dict(ok, mvy=(0, 8 * (hy + 1)))]                       # bottom
        for b in bad:
            with pytest.raises(cucd.CucdError):
                eng.me_mc_chroma([ok, b])
        # the corners themselves are accepted, at every fraction
        for f in (0, 7):
            edge = [dict(ok, mvx=(8 * lo + f, 8 * hx + f), mvy=(8 * lo + f, 8 * hy + f)), dict(ok, mvx=(8 * hx + f, 8 * lo + f), mvy=(8 * hy + f, 8 * lo + f))]
            assert eng.me_mc_chroma(edge).shape == (2, 2)
        lib = cucd.load_library()
        arr, n, _ = eng.mc_descs([ok])
        sse = np.zeros(2, np.uint32)
        assert lib.cucd_me_mc_chroma(eng.h, -1, arr, sse.ctypes.data, None) == -1
        assert lib.cucd_me_mc_chroma(eng.h, 1, None, sse.ctypes.data, None) == -1
        assert lib.cucd_me_mc_chroma(eng.h, 1, arr, None, None) == -1
        assert lib.cucd_me_mc_chroma(None, 1, arr, sse.ctypes.data, None) == -1
        assert lib.cucd_me_mc_chroma(eng.h, 0, None, None, None) == 0
        cb, cr = sc["refs_c"][0]
        assert lib.cucd_set_ref_picture_chroma(eng.h, 0, None, cr.ctypes.data, cr.shape[1], Mc, Mc) == -1
        assert lib.cucd_set_ref_picture_chroma(eng.h, 64, cb.ctypes.data, cr.ctypes.data, cr.shape[1], Mc, Mc) == -1
        assert lib.cucd_set_ref_picture_chroma(eng.h, 0, cb.ctypes.data, cr.ctypes.data, Wc + 2 * Mc - 1, Mc, Mc) == -1
        assert lib.cucd_set_ref_picture_chroma(eng.h, 0, cb.ctypes.data, cr.ctypes.data, cr.shape[1], -1, Mc) == -1
        assert lib.cucd_set_cur_picture_chroma(eng.h, cb.ctypes.data, None, Wc) == -1
        assert lib.cucd_set_cur_picture_chroma(eng.h, cb.ctypes.data, cr.ctypes.data, Wc - 1) == -1
        assert eng.me_mc_chroma([ok]).shape == (1, 2)                     # the handle still works


@pytest.mark.parametrize("bd", [8, 10])
def test_chroma_from_motion_compensation_to_the_residual_quadtree(cucd, bd):
    """a 64x64 bi and a uni candidate: luma prediction from cucd_me_mc_cost(pred), chroma from cucd_me_mc_chroma(pred); org - pred for
    Y, Cb and Cr, and every TU of the luma (32, 16, 8, 4) and chroma (16, 8, 4) RQT depths of both candidates through one
    cucd_inter_tu_code call.  Per plane and depth the chroma dist_zero sum to the candidate's sse; Cb + Cr sse plus the luma SSE of
    the prediction is the skip distortion before chroma weighting"""
    from inter_tu_util import load_inter_tu_oracle, oracle_inter_tu, oracle_sse
    from mc_util import load_mc_oracle, oracle_mc
    ito = load_inter_tu_oracle()
    sc = mcc_scene(bd, seed=20 + bd)
    x, y = 64, 32
    descs = [dict(x=x, y=y, w=64, h=64, ref_idx=(0, 3), mvx=(13, -22), mvy=(-7, 30), use_hadamard=1),
             dict(x=x, y=y, w=64, h=64, ref_idx=(-1, 3), mvx=(0, 6), mvy=(0, -5), use_hadamard=0)]
    with engine(cucd, sc) as eng:
        _, lp = eng.me_mc_cost(descs, want_pred=True)
        sse, cp = eng.me_mc_chroma(descs, want_pred=True)
        want_d, want_lp = oracle_mc(load_mc_oracle(), sc, descs)
        want_s, want_cp = oracle_mc_chroma(load_mc_chroma_oracle(), sc, descs)
        assert all(np.array_equal(a, b) for a, b in zip(lp, want_lp))
        assert_equal(descs, sse, cp, want_s, want_cp)
        planes = [(sc["org"][y:y + 64, x:x + 64], (5, 4, 3, 2), 0)] + [(sc["org_c"][c][y // 2:y // 2 + 32, x // 2:x // 2 + 32], (4, 3, 2), 1) for c in range(2)]
        tus, res, owner = [], [], []
        for k in range(len(descs)):
            preds = (lp[k], cp[k][0], cp[k][1])
            for comp, (org, sizes, chroma) in enumerate(planes):
                resi = (org.astype(np.int32) - preds[comp]).astype(np.int16)
                for lg in sizes:
                    n = 1 << lg
                    for by in range(0, org.shape[0], n):
                        for bx in range(0, org.shape[1], n):
                            tus.append((lg, 30 + k - chroma, 0, chroma))
                            res.append(np.ascontiguousarray(resi[by:by + n, bx:bx + n]).ravel())
                            owner.append((k, comp, lg))
        level, rresi, dist, dz, abs_sum = eng.inter_tu_code(tus, np.concatenate(res))
    offs = np.cumsum([0] + [r.size for r in res])
    for i in range(0, len(tus), 5):
        lg, qp, ts, ch = tus[i]
        w = oracle_inter_tu(ito, bd, 1 << lg, qp, ts, ch, 1, 1, res[i])
        assert np.array_equal(level[offs[i]:offs[i + 1]], w["level"]) and (dist[i], dz[i]) == (w["dist"], w["dist_zero"]), i
    for k in range(len(descs)):
        for comp in (1, 2):
            for lg in (4, 3, 2):
                assert sum(int(dz[i]) for i, o in enumerate(owner) if o == (k, comp, lg)) == sse[k, comp - 1], (k, comp, lg)
        skip = oracle_sse(ito, bd, sc["org"][y:y + 64, x:x + 64], want_lp[k]) + sum(
            oracle_sse(ito, bd, sc["org_c"][c][y // 2:y // 2 + 32, x // 2:x // 2 + 32], want_cp[k][c]) for c in range(2))
        assert oracle_sse(ito, bd, sc["org"][y:y + 64, x:x + 64], lp[k]) + int(sse[k, 0]) + int(sse[k, 1]) == skip, k


def test_mc_chroma_through_cucd_server(cucd, tmp_path):
    """tests/ipc_mc_chroma_replay.cpp sends set-cur (luma + chroma), set-ref (luma + chroma) and cucd_me_mc_chroma requests to
    cucd_server --clients 1; every reply equals the direct call's"""
    server = os.path.join(ROOT, "fast-cu-decision-hevc_b200", "cucd_server")
    assert os.path.exists(server), "cucd_server not built"
    exe = str(tmp_path / "ipc_mc_chroma_replay")
    subprocess.run(["g++", "-std=c++17", "-O2", "-I" + os.path.join(ROOT, "include"), "-o", exe, os.path.join(ROOT, "tests", "ipc_mc_chroma_replay.cpp"),
                    "-lrt"], check=True, capture_output=True)
    sc = mcc_scene(10, seed=11)
    rng = np.random.default_rng(12)
    descs = mcc_candidates(sc, rng, shapes=MC_SHAPES[::3])
    slots = sorted(sc["refs"])
    with engine(cucd, sc) as eng:
        s_all, p_all = eng.me_mc_chroma(descs, want_pred=True)
    flat = lambda ps: np.concatenate([q.ravel() for p in ps for q in p])
    want = [s_all, flat(p_all), s_all]
    for i in range(len(descs)):
        want += [s_all[i], flat(p_all[i:i + 1])]
    job = str(tmp_path / "mcc_job.bin")
    with open(job, "wb") as f:
        f.write(np.array([sc["W"], sc["H"], sc["bd"], sc["M"], len(slots), len(descs)] + slots, np.int32).tobytes())
        f.write(np.ascontiguousarray(sc["org"]).tobytes())
        for c in range(2):
            f.write(np.ascontiguousarray(sc["org_c"][c]).tobytes())
        for s in slots:
            f.write(sc["refs"][s].tobytes())
            for c in range(2):
                f.write(sc["refs_c"][s][c].tobytes())
        f.write(np.array([[d["x"], d["y"], d["w"], d["h"], *d["ref_idx"], *d["mvx"], *d["mvy"], d["use_hadamard"]] for d in descs], np.int32).tobytes())
    name = f"/cucd_mcc_test_{os.getpid()}"
    srv = subprocess.Popen([server, "--name", name, "--clients", "1"], stdout=subprocess.PIPE, text=True)
    try:
        time.sleep(1.0)
        proc = subprocess.run([exe, name, job, job + ".out"], capture_output=True, text=True, timeout=600)
        assert proc.returncode == 0, proc.stderr[-1500:]
        stats = json.loads(srv.communicate(timeout=60)[0].strip().splitlines()[-1])
    finally:
        if srv.poll() is None:
            srv.kill()
            srv.wait()
    assert stats["closed"] == 1 and stats["mc_chroma"] == 2 + len(descs) and stats["set_ref"] == len(slots)
    got = np.fromfile(job + ".out", np.uint8)
    off = 0
    for a in want:
        n = a.nbytes
        assert np.array_equal(got[off:off + n].view(a.dtype), a.ravel()), off
        off += n
    assert off == got.size
