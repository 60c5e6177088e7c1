"""cucd_me_tz_search through the C ABI (and through cucd_server) against the checker tests/me_tz_oracle.c, and against the surface route:
cucd_me_sad_surface over the bounding box of the walk's probes, the checker's walk on that surface, then cucd_me_subpel_cost at its
result and the refinement walk on the host.  Integer work: bit-exact."""
import json
import os
import subprocess
import time

import numpy as np
import pytest

from _util import ROOT, pseudo_recon, textured_plane
from me_search_util import np_walk
from me_tz_util import (FRAC, HAD, LAMBDAS, MC_SHAPES, TZ2N, as_rows, lambda_cost, load_me_tz_oracle, mc_scene, oracle_tz, oracle_tz_rows,
                        tz_desc)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def tz():
    return load_me_tz_oracle()


def engine(cucd, sc):
    eng = cucd.Engine(sc["W"], sc["H"], bit_depth=sc["bd"])
    eng.set_cur_picture(sc["org"])
    for s, p in sc["refs"].items():
        eng.set_ref_picture(s, p, sc["M"], sc["M"])
    return eng


def scene(kind, bd, seed):
    """moving: the source is textured_plane(t=1), the reference pseudo_recon of t=0 (real (2, 1) motion); unrelated: mc_scene's planes
    (the walk mostly ends in the raster); constant: flat planes (ties everywhere)"""
    sc = mc_scene(bd, seed=seed)
    if kind == "moving":
        W, H, M = sc["W"], sc["H"], sc["M"]
        sc = dict(sc, org=textured_plane(W, H, bd, seed=seed, t=1),
                  refs={s: np.ascontiguousarray(np.pad(pseudo_recon(textured_plane(W, H, bd, seed=seed, t=0), bd, seed=s + 1), M, mode="edge"))
                        for s in sc["slots"]})
    elif kind == "constant":
        v = (1 << bd) // 3
        sc = dict(sc, org=np.full_like(sc["org"], v), refs={s: np.full_like(p, v + 5 * k) for k, (s, p) in enumerate(sc["refs"].items())})
    return sc


def tz_descs(sc, rng, shapes=MC_SHAPES, R=64, flag_sets=(FRAC | HAD, FRAC, 0), tz2n=(0, TZ2N)):
    """per shape and flag set one PU; every fifth sits at a picture corner (its box clipped there), predictors near the motion or
    anywhere in int16, lambdas cycling through LAMBDAS"""
    W, H = sc["W"], sc["H"]
    out = []
    for w, h in shapes:
        for fl in flag_sets:
            for t in tz2n:
                n = len(out)
                if n % 5 == 4:
                    x, y = [(0, 0), (W - w, 0), (0, H - h), (W - w, H - h)][n // 5 % 4]
                else:
                    x = int(rng.integers(0, (W - w) // 4 + 1)) * 4
                    y = int(rng.integers(0, (H - h) // 4 + 1)) * 4
                pred = (int(rng.integers(-32768, 32768)), int(rng.integers(-32768, 32768))) if rng.random() < 0.2 else \
                    (-8 + int(rng.integers(-12, 13)), -4 + int(rng.integers(-12, 13)))
                out.append(tz_desc(sc, x, y, w, h, sc["slots"][n % len(sc["slots"])], pred, R, sub_shift=int(rng.integers(0, 2)),
                                   lam=int(LAMBDAS[n % len(LAMBDAS)]), flags=fl | t, mv2n=tuple(int(v) for v in rng.integers(-6, 7, 2))))
    return out


def assert_rows(descs, got, want):
    for i, d in enumerate(descs):
        assert np.array_equal(got[i], want[i]), (d, got[i], want[i])


@pytest.mark.parametrize("bd", [8, 9, 10])
@pytest.mark.parametrize("kind", ["moving", "unrelated", "constant"])
def test_tz_search_vs_checker(cucd, tz, bd, kind):
    """22 shapes x (FRAC + Hadamard, FRAC + SAD, integer only) x (with and without TZ_2NX2N), lambdas {0, QP 22, QP 37, 2^32 - 1}: one
    shuffled batch, then single-PU calls (the zero-copy path)"""
    sc = scene(kind, bd, seed=bd + 10 * len(kind))
    rng = np.random.default_rng(bd + len(kind))
    descs = tz_descs(sc, rng)
    rng.shuffle(descs)
    assert {d["lambda"] for d in descs} == set(LAMBDAS)
    want = oracle_tz_rows(tz, sc, descs)
    with engine(cucd, sc) as eng:
        assert_rows(descs, as_rows(eng.me_tz_search(descs)), want)
        for i in range(0, len(descs), 7):
            assert np.array_equal(as_rows(eng.me_tz_search([descs[i]]))[0], want[i]), descs[i]
    if kind == "unrelated":
        probes = [oracle_tz(tz, sc, d, trace_cap=100000)[1] for d in descs]
        assert sum(bool((t[:, 4] == 3).any()) for t in probes) > len(descs) // 2          # the raster ran on most PUs


@pytest.mark.parametrize("bd", [8, 10])
def test_tz_search_agrees_with_surface_route(cucd, tz, bd):
    """cucd_me_sad_surface over the bounding box of the checker's probes, the checker's walk on that surface, cucd_me_subpel_cost at
    its result and the host walk: the same answer as cucd_me_tz_search"""
    sc = scene("moving", bd, seed=bd + 300)
    rng = np.random.default_rng(bd + 300)
    descs = tz_descs(sc, rng, shapes=MC_SHAPES[::2], flag_sets=(FRAC | HAD, FRAC))
    with engine(cucd, sc) as eng:
        res = as_rows(eng.me_tz_search(descs))
        boxes = []
        for d in descs:
            tr = oracle_tz(tz, sc, d, trace_cap=100000)[1]
            boxes.append((int(tr[:, 0].min()), int(tr[:, 0].max()), int(tr[:, 1].min()), int(tr[:, 1].max())))
        surf = eng.me_sad_surface([dict(d, left=b[0], right=b[1], top=b[2], bottom=b[3]) for d, b in zip(descs, boxes)])
        ints = [oracle_tz(tz, {"bd": bd}, dict(d, flags=d["flags"] & TZ2N), surface=(s, b[0], b[2]))[0] for d, b, s in zip(descs, boxes, surf)]
        tabs = eng.me_subpel_cost([dict(x=d["x"], y=d["y"], w=d["w"], h=d["h"], ref_idx=d["ref_idx"], mvx=int(r[0]), mvy=int(r[1]),
                                        use_hadamard=1 if d["flags"] & HAD else 0) for d, r in zip(descs, ints)])
    for d, r, i, t in zip(descs, res, ints, tabs):
        walk = np_walk(t, int(i[0]), int(i[1]), d)
        assert tuple(int(v) for v in r) == (int(i[0]), int(i[1]), int(i[2])) + tuple(int(v) for v in walk), d


def test_rejections_keep_the_handle_usable(cucd, tz):
    sc = mc_scene(8, seed=5)
    W, H, M = sc["W"], sc["H"], sc["M"]
    ok = tz_desc(sc, 32, 32, 16, 16, 0, (3, -5), 16, lam=lambda_cost(27), flags=FRAC | HAD | TZ2N, mv2n=(2, 1))
    want = oracle_tz(tz, sc, ok)[0]
    with cucd.Engine(W, H, bit_depth=8) as eng:
        with pytest.raises(cucd.CucdError, match="cucd_set_cur_picture"):
            eng.me_tz_search([ok])
        eng.set_cur_picture(sc["org"])
        with pytest.raises(cucd.CucdError, match="reference picture not set"):
            eng.me_tz_search([ok])
        eng.set_ref_picture(0, sc["refs"][0], M, M)
        assert np.array_equal(as_rows(eng.me_tz_search([ok]))[0], want)
        assert eng.me_tz_search([]).shape == (0,)
        cl, cr, ct, cb = ok["clip_left"], ok["clip_right"], ok["clip_top"], ok["clip_bottom"]
        bad = [dict(ok, w=6), dict(ok, h=2), dict(ok, w=68), dict(ok, x=-4), dict(ok, y=H - 8), dict(ok, sub_shift=5), dict(ok, sub_shift=-1),
               dict(ok, ref_idx=7), dict(ok, ref_idx=64), dict(ok, ref_idx=-1), dict(ok, flags=8), dict(ok, flags=-1),
               dict(ok, pred_x=32768), dict(ok, pred_y=-32769), dict(ok, mv2n_x=32768), dict(ok, mv2n_y=-32769),
               dict(ok, left=3, right=2), dict(ok, top=3, bottom=2),                                    # empty window
               dict(ok, left=cl - 1), dict(ok, right=cr + 1), dict(ok, top=ct - 1), dict(ok, bottom=cb + 1),   # window outside the box
               dict(ok, clip_left=1, left=1), dict(ok, clip_right=-1, right=-1, left=-2), dict(ok, clip_top=1, top=1),
               dict(ok, clip_bottom=-1, bottom=-1, top=-2),                                             # box without (0, 0)
               dict(ok, clip_left=cl - 1), dict(ok, clip_right=cr + 1), dict(ok, clip_top=ct - 1), dict(ok, clip_bottom=cb + 1),   # 8-tap support
               dict(ok, clip_left=cl - 5, flags=0), dict(ok, clip_bottom=cb + 6, flags=0),             # the blocks themselves
               dict(ok, search_range=-1), dict(ok, search_range=4096),
               dict(ok, h=6, w=16)]                                                                      # FRAC needs h % 4 == 0
        for b in bad:
            with pytest.raises(cucd.CucdError):
                eng.me_tz_search([ok, b])
            assert np.array_equal(as_rows(eng.me_tz_search([ok]))[0], want), b
        # the limits themselves are accepted: the FRAC box, the integer box (4 / 5 samples wider), h = 6 without FRAC, range 4095
        edge = [dict(ok, left=cl, right=cr, top=ct, bottom=cb),
                dict(ok, clip_left=cl - 4, clip_right=cr + 5, clip_top=ct - 4, clip_bottom=cb + 5, left=cl - 4, bottom=cb + 5, flags=TZ2N),
                dict(ok, h=6, flags=0), dict(ok, search_range=4095, flags=0)]
        assert_rows(edge, as_rows(eng.me_tz_search(edge)), oracle_tz_rows(tz, sc, edge))
        lib = cucd.load_library()
        arr = cucd.Engine.tz_descs([ok])
        out = np.zeros(1, cucd.SEARCH_RESULT)
        assert lib.cucd_me_tz_search(eng.h, -1, arr.ctypes.data, out.ctypes.data) == -1
        assert lib.cucd_me_tz_search(eng.h, 1, None, out.ctypes.data) == -1
        assert lib.cucd_me_tz_search(eng.h, 1, arr.ctypes.data, None) == -1
        assert lib.cucd_me_tz_search(None, 1, arr.ctypes.data, out.ctypes.data) == -1
        assert lib.cucd_me_tz_search(eng.h, 0, None, None) == 0
        assert np.array_equal(as_rows(eng.me_tz_search([ok]))[0], want)


def test_slot_reset_between_calls(cucd, tz):
    sc = mc_scene(10, seed=6)
    sc2 = mc_scene(10, seed=7)
    descs = tz_descs(sc, np.random.default_rng(6), shapes=MC_SHAPES[::4], flag_sets=(FRAC | HAD,))
    with engine(cucd, sc) as eng:
        assert_rows(descs, as_rows(eng.me_tz_search(descs)), oracle_tz_rows(tz, sc, descs))
        for s in sc["slots"]:
            eng.set_ref_picture(s, sc2["refs"][s], sc["M"], sc["M"])
        assert_rows(descs, as_rows(eng.me_tz_search(descs)), oracle_tz_rows(tz, dict(sc, refs=sc2["refs"]), descs))


def test_last_kernel_time_covers_the_search(cucd):
    sc = mc_scene(8, W=1920, H=1080, seed=8)
    rng = np.random.default_rng(8)
    descs = [tz_desc(sc, int(x), int(y), 16, 16, sc["slots"][0], (0, 0), 64, lam=lambda_cost(30)) for x, y in zip(rng.integers(0, 119, 3000) * 16,
                                                                                                                 rng.integers(0, 67, 3000) * 16)]
    with engine(cucd, sc) as eng:
        n0 = eng.launch_count
        eng.me_tz_search(descs)
        ms = eng.last_kernel_time_ms()
        assert eng.launch_count - n0 >= 3                      # TZ walk, sub-pel, refinement walk
    assert 0 < ms < 5000


def test_tz_search_through_cucd_server_three_clients(cucd, tz, tmp_path):
    """three tests/ipc_me_tz_replay.cpp processes send set-cur, set-ref and cucd_me_tz_search requests to cucd_server --clients 3;
    every reply equals the checker"""
    server = os.path.join(ROOT, "fast-cu-decision-hevc_b200", "cucd_server")
    assert os.path.exists(server), "cucd_server not built"
    exe = str(tmp_path / "ipc_me_tz_replay")
    subprocess.run(["g++", "-std=c++17", "-O2", "-I" + os.path.join(ROOT, "include"), "-o", exe, os.path.join(ROOT, "tests", "ipc_me_tz_replay.cpp"), "-lrt"],
                   check=True, capture_output=True)
    from me_tz_util import FIELDS, desc_row
    assert len(FIELDS) == 21
    jobs, wants = [], []
    for c in range(3):
        sc = scene("moving" if c != 1 else "unrelated", 8 + 2 * (c % 2), seed=40 + c)
        descs = tz_descs(sc, np.random.default_rng(40 + c), shapes=MC_SHAPES[c::3], flag_sets=(FRAC | HAD, 0))
        slots = sorted(sc["refs"])
        want = oracle_tz_rows(tz, sc, descs)
        wants.append(np.concatenate([want, want]))
        job = str(tmp_path / f"tz_job{c}.bin")
        with open(job, "wb") as f:
            f.write(np.array([sc["W"], sc["H"], sc["bd"], sc["M"], len(slots), len(descs)] + slots, np.int32).tobytes())
            f.write(np.ascontiguousarray(sc["org"]).tobytes())
            for s in slots:
                f.write(sc["refs"][s].tobytes())
            f.write(np.stack([desc_row(d) for d in descs]).tobytes())
        jobs.append((job, len(descs)))
    name = f"/cucd_tz_test_{os.getpid()}"
    srv = subprocess.Popen([server, "--name", name, "--clients", "3"], stdout=subprocess.PIPE, text=True)
    procs = []
    try:
        time.sleep(1.0)
        procs = [subprocess.Popen([exe, name, j, j + ".out"], stderr=subprocess.PIPE, text=True) for j, _ in jobs]
        for p in procs:
            _, err = p.communicate(timeout=600)
            assert p.returncode == 0, err[-1500:]
        stats = json.loads(srv.communicate(timeout=60)[0].strip().splitlines()[-1])
    finally:
        for p in procs:
            if p.poll() is None:
                p.kill()
                p.wait()
        if srv.poll() is None:
            srv.kill()
            srv.wait()
    assert stats["closed"] == 3 and stats["tz"] == sum(1 + n for _, n in jobs)
    for (job, n), want in zip(jobs, wants):
        got = np.fromfile(job + ".out", np.int32).reshape(-1, 6).astype(np.int64)
        got[:, [2, 5]] &= 0xFFFFFFFF
        assert got.shape[0] == 2 * n
        assert np.array_equal(got, want)
