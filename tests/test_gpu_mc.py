"""cucd_me_mc_cost through the C ABI (and through cucd_server) against the checker tests/mc_oracle.c: uni- and bi-predictive motion
compensation of inter candidates and their distortion, samples and sums.  Integer work: bit-exact."""
import json
import os
import subprocess
import time

import numpy as np
import pytest

from _util import ROOT
from mc_util import MC_SHAPES, load_mc_oracle, mc_candidates, mc_scene, oracle_mc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def mco():
    return load_mc_oracle()


def engine(cucd, sc):
    eng = cucd.Engine(sc["W"], sc["H"], bit_depth=sc["bd"])
    eng.set_cur_picture(sc["org"])
    for s, p in sc["refs"].items():
        eng.set_ref_picture(s, p, sc["M"], sc["M"])
    return eng


def assert_equal(descs, got_d, got_p, want_d, want_p):
    for i, d in enumerate(descs):
        assert np.array_equal(got_p[i], want_p[i]), d
        assert got_d[i] == want_d[i], d


@pytest.mark.parametrize("bd", [8, 10])
def test_mc_vs_oracle_mixed_batch_and_single_candidates(cucd, mco, bd):
    """the coverage of test_emulation_mc.py: 22 shapes x (uni L0, uni L1, bi, bi with identical motion) x (Hadamard, SAD), random and
    extreme fractions, supports at the margin's corners; in one mixed batch and as batches of one candidate"""
    sc = mc_scene(bd, seed=bd)
    rng = np.random.default_rng(bd + 1)
    descs = mc_candidates(sc, rng) + mc_candidates(sc, rng)
    rng.shuffle(descs)
    want_d, want_p = oracle_mc(mco, sc, descs)
    with engine(cucd, sc) as eng:
        got_d, got_p = eng.me_mc_cost(descs, want_pred=True)
        assert_equal(descs, got_d, got_p, want_d, want_p)
        assert np.array_equal(eng.me_mc_cost(descs), got_d)                  # pred off: the same sums
        for i, d in enumerate(descs):
            d1, p1 = eng.me_mc_cost([d], want_pred=True)
            assert d1[0] == want_d[i] and np.array_equal(p1[0], want_p[i]), d


@pytest.mark.parametrize("bd", [8, 10])
def test_mc_large_batch_spans_several_waves(cucd, mco, bd):
    """>= 10 000 candidates of mixed shapes and modes; every 7th is checked in full against the oracle, all against the single-shape
    batches of the same candidates"""
    sc = mc_scene(bd, W=416, H=240, seed=50 + bd)
    rng = np.random.default_rng(bd + 3)
    descs = []
    while len(descs) < 10500:
        descs += mc_candidates(sc, rng, shapes=[MC_SHAPES[int(i)] for i in rng.integers(0, 22, 6)] + [(8, 8), (16, 16), (32, 32)])
    with engine(cucd, sc) as eng:
        got_d, got_p = eng.me_mc_cost(descs, want_pred=True)
        samp = list(range(0, len(descs), 7))
        want_d, want_p = oracle_mc(mco, sc, [descs[i] for i in samp])
        assert_equal([descs[i] for i in samp], got_d[samp], [got_p[i] for i in samp], want_d, want_p)
        assert np.array_equal(eng.me_mc_cost(descs), got_d)
        ms = eng.last_kernel_time_ms()
        assert ms > 0
        by_shape = {}
        for i, d in enumerate(descs):
            by_shape.setdefault((d["w"], d["h"]), []).append(i)
        for idx in by_shape.values():
            assert np.array_equal(eng.me_mc_cost([descs[i] for i in idx]), got_d[idx])


@pytest.mark.parametrize("bd", [8, 10])
def test_mc_lists_on_the_same_and_on_different_slots(cucd, mco, bd):
    """bi on one slot and on two slots in either order; uni on list 0 and on list 1 of each slot: a motion on list 1 predicts what
    the same motion on list 0 predicts"""
    sc = mc_scene(bd, seed=70 + bd, slots=(2, 5))
    descs = []
    for r0, r1 in ((2, 2), (5, 5), (2, 5), (5, 2)):
        for w, h in ((16, 16), (8, 4), (24, 32)):
            descs.append(dict(x=48, y=32, w=w, h=h, ref_idx=(r0, r1), mvx=(-37, 22), mvy=(13, -54), use_hadamard=1))
            descs.append(dict(x=48, y=32, w=w, h=h, ref_idx=(r0, -1), mvx=(-37, 0), mvy=(13, 0), use_hadamard=0))
            descs.append(dict(x=48, y=32, w=w, h=h, ref_idx=(-1, r0), mvx=(0, -37), mvy=(0, 13), use_hadamard=0))
    want_d, want_p = oracle_mc(mco, sc, descs)
    with engine(cucd, sc) as eng:
        got_d, got_p = eng.me_mc_cost(descs, want_pred=True)
    assert_equal(descs, got_d, got_p, want_d, want_p)
    for i in range(0, len(descs), 3):
        assert got_d[i + 1] == got_d[i + 2] and np.array_equal(got_p[i + 1], got_p[i + 2])
    assert not np.array_equal(got_p[0], got_p[2 * 9])                  # the slots hold different pictures


@pytest.mark.parametrize("bd", [8, 10])
def test_uni_equals_subpel_cost_entries(cucd, bd):
    """a uni candidate at integer MV + (dx, dy) quarter pels costs what cucd_me_subpel_cost's table holds at (dx, dy)"""
    sc = mc_scene(bd, seed=90 + bd)
    rng = np.random.default_rng(bd + 9)
    sp, mc, where = [], [], []
    for k, (w, h) in enumerate(MC_SHAPES):
        for had in (1, 0):
            x = int(rng.integers(0, (sc["W"] - w) // 4 + 1)) * 4; y = int(rng.integers(0, (sc["H"] - h) // 4 + 1)) * 4
            mvx, mvy = int(rng.integers(-20, 21)), int(rng.integers(-20, 21))
            sp.append(dict(x=x, y=y, w=w, h=h, ref_idx=3, mvx=mvx, mvy=mvy, use_hadamard=had))
            for dy in range(-3, 4):
                for dx in range(-3, 4):
                    mc.append(dict(x=x, y=y, w=w, h=h, ref_idx=(-1, 3) if (dx + dy) % 2 else (3, -1), mvx=(4 * mvx + dx,) * 2, mvy=(4 * mvy + dy,) * 2,
                                   use_hadamard=had))
                    where.append((len(sp) - 1, dy + 3, dx + 3))
    with engine(cucd, sc) as eng:
        table = eng.me_subpel_cost(sp)
        got = eng.me_mc_cost(mc)
    for g, (i, r, c) in zip(got, where):
        assert g == table[i, r, c], (sp[i], r, c)


def test_mc_rejections_and_empty_batch(cucd):
    sc = mc_scene(8, seed=3)
    W, H, M = sc["W"], sc["H"], sc["M"]
    ok = dict(x=16, y=16, w=16, h=16, ref_idx=(0, 3), mvx=(5, -7), mvy=(2, 9), use_hadamard=1)
    with cucd.Engine(W, H, bit_depth=8) as eng:
        with pytest.raises(cucd.CucdError, match="cucd_set_cur_picture"):
            eng.me_mc_cost([ok])
        eng.set_cur_picture(sc["org"])
        eng.set_ref_picture(0, sc["refs"][0], M, M)
        with pytest.raises(cucd.CucdError, match="reference picture not set"):
            eng.me_mc_cost([ok])                                          # slot 3 is not set yet
        eng.set_ref_picture(3, sc["refs"][3], M, M)
        assert eng.me_mc_cost([ok]).shape == (1,)
        d, p = eng.me_mc_cost([], want_pred=True)
        assert d.shape == (0,) and p == []
        assert eng.me_mc_cost([]).shape == (0,)
        bad = [dict(ok, w=6), dict(ok, h=2), dict(ok, w=68), dict(ok, h=66), dict(ok, x=-4), dict(ok, y=H - 8), dict(ok, x=W - 12),
               dict(ok, ref_idx=(-1, -1)), dict(ok, ref_idx=(0, 64)), dict(ok, ref_idx=(7, -1)),
               dict(ok, mvx=(4 * (3 - M - 16) - 1, 0)),                 # left edge of the support one sample outside
               dict(ok, mvx=(0, 4 * (W - 1 + M - 16 - 3 - 16) + 4)),   # right edge, list 1
               dict(ok, mvy=(4 * (3 - M - 16) - 4, 0)),
               dict(ok, mvy=(0, 4 * (H - 1 + M - 16 - 3 - 16) + 4))]
        for b in bad:
            with pytest.raises(cucd.CucdError):
                eng.me_mc_cost([ok, b])
        # the corners themselves are accepted
        edge = [dict(ok, mvx=(4 * (3 - M - 16), 4 * (W - 1 + M - 16 - 3 - 16) + 3), mvy=(4 * (3 - M - 16), 4 * (H - 1 + M - 16 - 3 - 16) + 3))]
        assert eng.me_mc_cost(edge).shape == (1,)
        lib = cucd.load_library()
        arr, n, _ = eng.mc_descs([ok])
        dist = np.zeros(1, np.uint32)
        assert lib.cucd_me_mc_cost(eng.h, -1, arr, dist.ctypes.data, None) == -1
        assert lib.cucd_me_mc_cost(eng.h, 1, None, dist.ctypes.data, None) == -1
        assert lib.cucd_me_mc_cost(eng.h, 1, arr, None, None) == -1
        assert lib.cucd_me_mc_cost(None, 1, arr, dist.ctypes.data, None) == -1
        assert lib.cucd_me_mc_cost(eng.h, 0, None, None, None) == 0


def test_mc_through_cucd_server(cucd, tmp_path):
    """tests/ipc_mc_replay.cpp sends set-cur, set-ref and cucd_me_mc_cost requests to cucd_server --clients 1; every reply equals the
    direct call's"""
    server = os.path.join(ROOT, "fast-cu-decision-hevc_b200", "cucd_server")
    assert os.path.exists(server), "cucd_server not built"
    exe = str(tmp_path / "ipc_mc_replay")
    subprocess.run(["g++", "-std=c++17", "-O2", "-I" + os.path.join(ROOT, "include"), "-o", exe, os.path.join(ROOT, "tests", "ipc_mc_replay.cpp"), "-lrt"],
                   check=True, capture_output=True)
    sc = mc_scene(10, seed=11)
    rng = np.random.default_rng(12)
    descs = mc_candidates(sc, rng, shapes=MC_SHAPES[::3])
    slots = sorted(sc["refs"])
    with engine(cucd, sc) as eng:
        d_all, p_all = eng.me_mc_cost(descs, want_pred=True)
    want = [d_all, np.concatenate([p.ravel() for p in p_all]), d_all]
    for i in range(len(descs)):
        want += [d_all[i:i + 1], p_all[i].ravel()]
    job = str(tmp_path / "mc_job.bin")
    with open(job, "wb") as f:
        f.write(np.array([sc["W"], sc["H"], sc["bd"], sc["M"], len(slots), len(descs)] + slots, np.int32).tobytes())
        f.write(np.ascontiguousarray(sc["org"]).tobytes())
        for s in slots:
            f.write(sc["refs"][s].tobytes())
        f.write(np.array([[d["x"], d["y"], d["w"], d["h"], *d["ref_idx"], *d["mvx"], *d["mvy"], d["use_hadamard"]] for d in descs], np.int32).tobytes())
    name = f"/cucd_mc_test_{os.getpid()}"
    srv = subprocess.Popen([server, "--name", name, "--clients", "1"], stdout=subprocess.PIPE, text=True)
    proc = None
    try:
        time.sleep(1.0)
        proc = subprocess.run([exe, name, job, job + ".out"], capture_output=True, text=True, timeout=600)
        assert proc.returncode == 0, proc.stderr[-1500:]
        stats = json.loads(srv.communicate(timeout=60)[0].strip().splitlines()[-1])
    finally:
        if srv.poll() is None:
            srv.kill()
            srv.wait()
    assert stats["closed"] == 1 and stats["mc"] == 2 + len(descs) and stats["set_ref"] == len(slots)
    got = np.fromfile(job + ".out", np.uint8)
    off = 0
    for a in want:
        n = a.nbytes
        assert np.array_equal(got[off:off + n].view(a.dtype), a.ravel()), off
        off += n
    assert off == got.size
