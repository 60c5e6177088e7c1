"""cucd_me_search / cucd_me_search_src through the C ABI (and cucd_me_search through cucd_server) against the checker
tests/me_search_oracle.c and against the surface route it replaces: cucd_me_sad_surface, then cucd_me_subpel_cost at the integer
result, then the argmin and the walk on the host.  Integer work: bit-exact."""
import json
import os
import subprocess
import time

import numpy as np
import pytest

from _util import ROOT, full_range_keys, pseudo_recon, textured_plane
from me_search_util import (FRAC, HAD, LAMBDAS, MC_SHAPES, as_rows, lambda_cost, load_me_search_oracle, mc_scene, np_bits, np_walk, oracle_search,
                            search_desc, search_descs, walk_batch)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def mso():
    return load_me_search_oracle()


def engine(cucd, sc):
    eng = cucd.Engine(sc["W"], sc["H"], bit_depth=sc["bd"])
    eng.set_cur_picture(sc["org"])
    for s, p in sc["refs"].items():
        eng.set_ref_picture(s, p, sc["M"], sc["M"])
    return eng


def assert_rows(descs, got, want):
    for i, d in enumerate(descs):
        assert np.array_equal(got[i], want[i]), (d, got[i], want[i])


@pytest.mark.parametrize("bd", [8, 9, 10])
def test_search_vs_checker_mixed_batch_and_single_pus(cucd, mso, bd):
    """22 shapes x (+-64, +-4, 1x1) x (FRAC + Hadamard, FRAC + SAD, integer only), lambdas {0, QP 22, QP 37, 2^32 - 1}, predictors
    anywhere in int16, windows clipped at the corners, sub_shift 0 and 1: one shuffled batch, then batches of one PU"""
    sc = mc_scene(bd, seed=bd + 100)
    rng = np.random.default_rng(bd + 100)
    descs = search_descs(sc, rng) + search_descs(sc, rng)
    rng.shuffle(descs)
    assert {d["lambda"] for d in descs} == set(LAMBDAS)
    want = oracle_search(mso, sc, descs)
    with engine(cucd, sc) as eng:
        assert_rows(descs, as_rows(eng.me_search(descs)), want)
        for i in range(0, len(descs), 5):
            assert np.array_equal(as_rows(eng.me_search([descs[i]]))[0], want[i]), descs[i]


@pytest.mark.parametrize("bd,keys", [pytest.param(bd, k, id=str(bd) if k == "hm" else f"{bd}-{k}") for k in ("hm", "int16") for bd in (8, 9, 10)])
def test_search_src_signed_keys(cucd, mso, bd, keys):
    """caller-supplied keys outside [0, 2^bd), as the bi-predictive refinement sends them.  keys "int16": samples from all of int16 with
    runs of both ends and whole blocks of -32768 against the scene's reference runs of 0 and 2^bd - 1, in +-40 windows (several dx-lane
    tiles a row)"""
    sc = mc_scene(bd, seed=bd + 200)
    rng = np.random.default_rng(bd + 200)
    descs = search_descs(sc, rng, radii=(8, 4, 0) if keys == "hm" else (40, 8, 0))
    hi = 1 << bd
    n = sum(d["w"] * d["h"] for d in descs)
    if keys == "hm":
        src = rng.integers(-hi, 2 * hi, n).astype(np.int16)
    else:
        src = full_range_keys(rng, n)
        off = 0
        for i, d in enumerate(descs):
            if i % 4 == 0:
                src[off:off + d["w"] * d["h"]] = -32768
            off += d["w"] * d["h"]
        assert max(d["right"] - d["left"] + 1 for d in descs) > 64
    want = oracle_search(mso, sc, descs, src)
    with cucd.Engine(sc["W"], sc["H"], bit_depth=bd) as eng:                 # no current picture needed
        for s, p in sc["refs"].items():
            eng.set_ref_picture(s, p, sc["M"], sc["M"])
        assert_rows(descs, as_rows(eng.me_search(descs, src=src)), want)


@pytest.mark.parametrize("bd", [8, 10])
def test_search_agrees_with_surface_and_subpel_calls(cucd, bd):
    """sad = the cucd_me_sad_surface entry at mv; qmv / frac_cost = the walk over cucd_me_subpel_cost's table; a 1x1 window at mv
    reproduces the refinement alone"""
    sc = mc_scene(bd, seed=bd + 300)
    rng = np.random.default_rng(bd + 300)
    descs = [d for d in search_descs(sc, rng, radii=(16,), flag_sets=(FRAC | HAD, FRAC))]
    with engine(cucd, sc) as eng:
        res = eng.me_search(descs)
        surf = eng.me_sad_surface(descs)
        tabs = eng.me_subpel_cost([dict(x=d["x"], y=d["y"], w=d["w"], h=d["h"], ref_idx=d["ref_idx"], mvx=int(r["mvx"]), mvy=int(r["mvy"]),
                                        use_hadamard=1 if d["flags"] & HAD else 0) for d, r in zip(descs, res)])
        one = [dict(d, left=int(r["mvx"]), right=int(r["mvx"]), top=int(r["mvy"]), bottom=int(r["mvy"])) for d, r in zip(descs, res)]
        res1 = eng.me_search(one)
    for d, r, s, t, r1 in zip(descs, res, surf, tabs, res1):
        assert r["sad"] == s[r["mvy"] - d["top"], r["mvx"] - d["left"]], d
        assert (int(r["qmvx"]), int(r["qmvy"]), int(r["frac_cost"])) == np_walk(t, int(r["mvx"]), int(r["mvy"]), d), d
        assert tuple(r1) == tuple(r), d


def test_ldp1080p_workload_matches_surface_route(cucd):
    """the ME part of bench.py's ldp1080p: 42 900 square PUs of a 1920x1080 8-bit picture, +-64, FEN sub_shift, FRAC with Hadamard.
    Every PU equals the surface route: cucd_me_sad_surface, numpy argmin, cucd_me_subpel_cost at the argmin, numpy walk."""
    import bench
    W, H, R, M = 1920, 1080, bench.ME_RANGE, bench.ME_MARGIN
    pus = bench.inter_pus(W, H)
    assert len(pus) == 42900
    org = textured_plane(W, H, 8, seed=31)
    ref = np.ascontiguousarray(np.pad(pseudo_recon(textured_plane(W, H, 8, seed=32), 8), M, mode="edge"))
    rng = np.random.default_rng(33)
    lam = lambda_cost(32)
    preds = rng.integers(-4 * R, 4 * R + 1, (len(pus), 2))
    descs = [dict(x=x, y=y, w=s, h=s, ref_idx=0, left=-R, right=R, top=-R, bottom=R, sub_shift=1 if s > 8 else 0, pred_x=int(p[0]), pred_y=int(p[1]),
                  flags=FRAC | HAD, **{"lambda": lam}) for (x, y, s), p in zip(pus, preds)]
    with cucd.Engine(W, H, bit_depth=8) as eng:
        eng.set_cur_picture(org)
        eng.set_ref_picture(0, ref, M, M)
        got = as_rows(eng.me_search(descs))
        # the surface route, in chunks of PUs
        xs = np.arange(-R, R + 1)
        mv = np.zeros((len(pus), 2), np.int64)
        sad = np.zeros(len(pus), np.int64)
        for c0 in range(0, len(pus), 2048):
            chunk = descs[c0:c0 + 2048]
            arr, n, total = cucd.Engine.me_descs(chunk)
            surf = np.zeros(total, np.uint32)
            eng.me_sad_surface_raw(arr, n, surf)
            surf = surf.reshape(n, 2 * R + 1, 2 * R + 1).astype(np.uint64)
            p = preds[c0:c0 + n]
            bits = np_bits(4 * xs[None, :] - p[:, :1])[:, None, :] + np_bits(4 * xs[None, :] - p[:, 1:])[:, :, None]
            cost = ((np.uint64(lam) * bits.astype(np.uint64)) & np.uint64(0xFFFFFFFF)) >> np.uint64(16)
            k = np.argmin((surf + cost).reshape(n, -1), axis=1)                                     # first minimum = least raster index
            mv[c0:c0 + n, 0] = k % (2 * R + 1) - R
            mv[c0:c0 + n, 1] = k // (2 * R + 1) - R
            sad[c0:c0 + n] = surf.reshape(n, -1)[np.arange(n), k].astype(np.int64)
        sp = [dict(x=d["x"], y=d["y"], w=d["w"], h=d["h"], ref_idx=0, mvx=int(m[0]), mvy=int(m[1]), use_hadamard=1) for d, m in zip(descs, mv)]
        arr, n = cucd.Engine.subpel_descs(sp)
        T = np.zeros((n, 49), np.uint32)
        eng.me_subpel_cost_raw(arr, n, T)
    qmv, fc = walk_batch(T, mv, preds, lam)
    want = np.concatenate([mv, sad[:, None], qmv, fc[:, None]], axis=1)
    bad = np.nonzero((got != want).any(axis=1))[0]
    assert bad.size == 0, (bad.size, descs[bad[0]], got[bad[0]], want[bad[0]])
    assert len(np.unique(mv, axis=0)) > 100                                                         # the search moves


def test_rejections_keep_the_handle_usable(cucd, mso):
    sc = mc_scene(8, seed=5)
    W, H, M = sc["W"], sc["H"], sc["M"]
    ok = search_desc(sc, 32, 32, 16, 16, 0, 0, 0, 8, pred=(3, -5), lam=lambda_cost(27))
    want = oracle_search(mso, sc, [ok])[0]
    with cucd.Engine(W, H, bit_depth=8) as eng:
        with pytest.raises(cucd.CucdError, match="cucd_set_cur_picture"):
            eng.me_search([ok])
        eng.set_cur_picture(sc["org"])
        with pytest.raises(cucd.CucdError, match="reference picture not set"):
            eng.me_search([ok])
        eng.set_ref_picture(0, sc["refs"][0], M, M)
        assert np.array_equal(as_rows(eng.me_search([ok]))[0], want)
        assert eng.me_search([]).shape == (0,)
        x = 32
        bad = [dict(ok, w=6), dict(ok, h=2), dict(ok, w=68), dict(ok, x=-4), dict(ok, y=H - 8), dict(ok, left=3, right=2), dict(ok, sub_shift=5),
               dict(ok, ref_idx=7), dict(ok, ref_idx=64), dict(ok, flags=4), dict(ok, flags=-1),
               dict(ok, pred_x=32768), dict(ok, pred_y=-32769),
               dict(ok, h=6, w=16),                                                       # FRAC needs h % 4 == 0
               dict(ok, left=4 - M - x - 1), dict(ok, right=W - 1 + M - 16 - 4 - x + 1),  # 8-tap support one sample outside
               dict(ok, top=4 - M - 32 - 1), dict(ok, bottom=H - 1 + M - 16 - 4 - 32 + 1),
               dict(ok, left=-M - x - 1, flags=0)]                                        # the integer window itself outside
        for b in bad:
            with pytest.raises(cucd.CucdError):
                eng.me_search([ok, b])
            assert np.array_equal(as_rows(eng.me_search([ok]))[0], want), b
        # the FRAC limits themselves are accepted, and without FRAC the integer window may reach the margin
        edge = [dict(ok, left=4 - M - x, right=W - 1 + M - 16 - 4 - x, top=4 - M - 32, bottom=H - 1 + M - 16 - 4 - 32),
                dict(ok, left=-M - x, right=W - 1 + M - 16 - x, top=-M - 32, bottom=H - 1 + M - 16 - 32, flags=0)]
        assert_rows(edge, as_rows(eng.me_search(edge)), oracle_search(mso, sc, edge))
        lib = cucd.load_library()
        arr, n = eng.search_descs([ok])
        out = np.zeros(1, cucd.SEARCH_RESULT)
        src = np.zeros(256, np.int16)
        assert lib.cucd_me_search(eng.h, -1, arr, out.ctypes.data) == -1
        assert lib.cucd_me_search(eng.h, 1, None, out.ctypes.data) == -1
        assert lib.cucd_me_search(eng.h, 1, arr, None) == -1
        assert lib.cucd_me_search(None, 1, arr, out.ctypes.data) == -1
        assert lib.cucd_me_search(eng.h, 0, None, None) == 0
        assert lib.cucd_me_search_src(eng.h, 1, arr, None, out.ctypes.data) == -1
        assert lib.cucd_me_search_src(eng.h, -1, arr, src.ctypes.data, out.ctypes.data) == -1
        assert lib.cucd_me_search_src(eng.h, 0, None, None, None) == 0
        assert np.array_equal(as_rows(eng.me_search([ok]))[0], want)


def test_slot_reset_between_calls(cucd, mso):
    sc = mc_scene(10, seed=6)
    sc2 = mc_scene(10, seed=7)
    rng = np.random.default_rng(6)
    descs = search_descs(sc, rng, shapes=MC_SHAPES[::4], radii=(8,), flag_sets=(FRAC | HAD,))
    with engine(cucd, sc) as eng:
        assert_rows(descs, as_rows(eng.me_search(descs)), oracle_search(mso, sc, descs))
        for s in sc["slots"]:
            eng.set_ref_picture(s, sc2["refs"][s], sc["M"], sc["M"])
        mixed = dict(sc, refs=sc2["refs"])
        assert_rows(descs, as_rows(eng.me_search(descs)), oracle_search(mso, mixed, descs))


def test_last_kernel_time_covers_the_search(cucd):
    sc = mc_scene(8, W=1920, H=1080, seed=8)
    rng = np.random.default_rng(8)
    descs = [search_desc(sc, int(x), int(y), 16, 16, sc["slots"][0], 0, 0, 64, lam=lambda_cost(30)) for x, y in zip(rng.integers(0, 119, 3000) * 16,
                                                                                                                      rng.integers(0, 67, 3000) * 16)]
    with engine(cucd, sc) as eng:
        n0 = eng.launch_count
        eng.me_search(descs)
        ms = eng.last_kernel_time_ms()
        assert eng.launch_count - n0 >= 4                      # SAD kernels, prep, sub-pel, walk
    assert 0 < ms < 5000


def test_search_through_cucd_server_three_clients(cucd, mso, tmp_path):
    """three tests/ipc_me_search_replay.cpp processes send set-cur, set-ref and cucd_me_search requests to cucd_server --clients 3;
    every reply equals the checker"""
    server = os.path.join(ROOT, "fast-cu-decision-hevc_b200", "cucd_server")
    assert os.path.exists(server), "cucd_server not built"
    exe = str(tmp_path / "ipc_me_search_replay")
    subprocess.run(["g++", "-std=c++17", "-O2", "-I" + os.path.join(ROOT, "include"), "-o", exe, os.path.join(ROOT, "tests", "ipc_me_search_replay.cpp"), "-lrt"],
                   check=True, capture_output=True)
    jobs, wants = [], []
    for c in range(3):
        sc = mc_scene(8 + 2 * (c % 2), seed=40 + c)
        rng = np.random.default_rng(40 + c)
        descs = search_descs(sc, rng, shapes=MC_SHAPES[c::3], radii=(16, 0))
        slots = sorted(sc["refs"])
        want = oracle_search(mso, sc, descs)
        wants.append(np.concatenate([want, want]))
        job = str(tmp_path / f"search_job{c}.bin")
        with open(job, "wb") as f:
            f.write(np.array([sc["W"], sc["H"], sc["bd"], sc["M"], len(slots), len(descs)] + slots, np.int32).tobytes())
            f.write(np.ascontiguousarray(sc["org"]).tobytes())
            for s in slots:
                f.write(sc["refs"][s].tobytes())
            f.write(np.array([[d["x"], d["y"], d["w"], d["h"], d["ref_idx"], d["left"], d["right"], d["top"], d["bottom"], d["sub_shift"], d["pred_x"],
                               d["pred_y"], np.uint32(d["lambda"]).view(np.int32), d["flags"]] for d in descs], np.int32).tobytes())
        jobs.append((job, len(descs)))
    name = f"/cucd_search_test_{os.getpid()}"
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
    assert stats["closed"] == 3 and stats["search"] == sum(1 + n for _, n in jobs)
    for (job, n), want in zip(jobs, wants):
        got = np.fromfile(job + ".out", np.int32).reshape(-1, 6).astype(np.int64)
        got[:, [2, 5]] &= 0xFFFFFFFF
        assert got.shape[0] == 2 * n
        assert np.array_equal(got, want)
