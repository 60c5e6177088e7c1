"""The checker of cucd_me_tz_search (tests/me_tz_oracle.c, written probe by probe in HM's branch structure) against the independent
Python statement of the walk in tests/me_tz_util.py (point lists and one directional guard rule), on synthetic SAD surfaces and on
pictures; literal probe orders for the diamonds, the border guards, the two-point cases and the raster."""
import numpy as np
import pytest

from me_tz_util import FRAC, HAD, MC_SHAPES, TZ2N, lambda_cost, load_me_tz_oracle, mc_scene, oracle_tz, py_tz_walk, surface_sad, tz_desc

B = 100                                    # synthetic surfaces cover the box [-B, B] x [-B, B]


@pytest.fixture(scope="module")
def tz():
    return load_me_tz_oracle()


def synth(f, win=(-64, 64, -64, 64), R=64, pred=(0, 0), lam=0, flags=0, mv2n=(0, 0)):
    """a descriptor over the box [-B, B]^2 with the given window, and the surface f(x, y) over the box"""
    ys, xs = np.mgrid[-B:B + 1, -B:B + 1]
    s = np.asarray(f(xs, ys), np.int64)
    s = np.broadcast_to(s, xs.shape).astype(np.uint32)
    d = dict(x=0, y=0, w=8, h=8, ref_idx=0, left=win[0], right=win[1], top=win[2], bottom=win[3], sub_shift=0, pred_x=pred[0], pred_y=pred[1],
             flags=flags, search_range=R, clip_left=-B, clip_right=B, clip_top=-B, clip_bottom=B, mv2n_x=mv2n[0], mv2n_y=mv2n[1], **{"lambda": lam})
    return d, s


def run(tz, d, s):
    """checker on the surface == the Python statement; returns the checker's trace as (x, y, p, d, stage, c) tuples"""
    res, trace, n = oracle_tz(tz, {"bd": 8}, d, surface=(s, -B, -B), trace_cap=100000)
    (mx, my, sad), want = py_tz_walk(d, surface_sad(s, -B, -B))
    got = [tuple(int(v) for v in t) for t in trace]
    assert got == [tuple(t) for t in want]
    assert (int(res[0]), int(res[1]), int(res[2])) == (mx, my, sad)
    assert n == len(got)
    return got, res


def stage(trace, k, cx=0, cy=0):
    """the (dx, dy, p, d) of stage k relative to (cx, cy)"""
    return [(x - cx, y - cy, p, d) for x, y, p, d, st, _ in trace if st == k]


def test_first_search_stops_after_three_rounds_on_a_flat_surface(tz):
    """nothing beats (0, 0): D = 1, 2, 4 run, then round 3 stops the first search; no raster, no star"""
    trace, res = run(tz, *synth(lambda x, y: 500 + 0 * x))
    assert [t[:2] for t in trace if t[4] == 0] == [(0, 0), (0, 0)]
    assert stage(trace, 1) == [(0, -1, 2, 1), (-1, 0, 4, 1), (1, 0, 5, 1), (0, 1, 7, 1),
                               (0, -2, 2, 2), (-1, -1, 1, 1), (1, -1, 3, 1), (-2, 0, 4, 2), (2, 0, 5, 2), (-1, 1, 6, 1), (1, 1, 8, 1), (0, 2, 7, 2),
                               (0, -4, 2, 4), (-2, -2, 1, 2), (2, -2, 3, 2), (-4, 0, 4, 4), (4, 0, 5, 4), (-2, 2, 6, 2), (2, 2, 8, 2), (0, 4, 7, 4)]
    assert max(t[4] for t in trace) == 1 and tuple(res[:2]) == (0, 0)


def test_diamond_16_inside_the_window(tz):
    """(0, -2) wins the D = 2 round, so D = 4, 8, 16 follow and the stop comes after D = 16"""
    trace, _ = run(tz, *synth(lambda x, y: np.where((x == 0) & (y == -2), 100, 500)))
    d16 = [t for t in stage(trace, 1) if t[3] == 16]
    assert d16 == [(0, -16, 0, 16), (-16, 0, 0, 16), (16, 0, 0, 16), (0, 16, 0, 16),
                   (-4, -12, 0, 16), (4, -12, 0, 16), (-4, 12, 0, 16), (4, 12, 0, 16),
                   (-8, -8, 0, 16), (8, -8, 0, 16), (-8, 8, 0, 16), (8, 8, 0, 16),
                   (-12, -4, 0, 16), (12, -4, 0, 16), (-12, 4, 0, 16), (12, 4, 0, 16)]
    assert not [t for t in stage(trace, 1) if t[3] == 32]


@pytest.mark.parametrize("border", ["top", "left", "right", "bottom"])
def test_border_guards(tz, border):
    """a window whose `border` lies 1 sample from the start: every point that crosses it is skipped, in the D <= 8 and D > 8 lists;
    points that move only along the border stay"""
    win = dict(top=(-64, 64, -1, 64), left=(-1, 64, -64, 64), right=(-64, 1, -64, 64), bottom=(-64, 64, -64, 1))[border]
    f = lambda x, y: np.where((x == 0) & (y == 0), 400, np.where((x == 3) & (y == 7), 300, 500))   # noqa: E731  (nothing in reach wins)
    d, s = synth(f, win=win, R=32)
    trace, _ = run(tz, d, s)
    pts = stage(trace, 1)
    assert all(win[0] <= x <= win[1] and win[2] <= y <= win[3] for x, y, _, _ in pts)
    full = [(0, -1), (-1, 0), (1, 0), (0, 1), (0, -2), (-1, -1), (1, -1), (-2, 0), (2, 0), (-1, 1), (1, 1), (0, 2),
            (0, -4), (-2, -2), (2, -2), (-4, 0), (4, 0), (-2, 2), (2, 2), (0, 4)]
    assert [p[:2] for p in pts] == [p for p in full if win[0] <= p[0] <= win[1] and win[2] <= p[1] <= win[3]]


def test_border_guards_far_diamond(tz):
    """D = 32 around a centre 20 samples below the top border: only the points whose own y stays inside are probed, per side"""
    f = lambda x, y: np.where((x == 0) & (y == 4), 100, 500)   # noqa: E731  D = 4 wins: D = 8, 16 and 32 follow
    d, s = synth(f, win=(-64, 64, -20, 64), R=32)
    trace, _ = run(tz, d, s)
    d32 = [t[:2] for t in stage(trace, 1) if t[3] == 32]
    want = [(-32, 0), (32, 0), (0, 32)]
    for k in (1, 2, 3):
        q = 8 * k
        if -32 + q >= -20:
            want += [(-q, -32 + q), (q, -32 + q)]
        want += [(-q, 32 - q), (q, 32 - q)]
    assert d32 == want


TWO = {1: [(-1, 0), (0, -1)], 2: [(-1, -1), (1, -1)], 3: [(0, -1), (1, 0)], 4: [(-1, 1), (-1, -1)], 5: [(1, -1), (1, 1)], 6: [(-1, 0), (0, 1)],
       7: [(-1, 1), (1, 1)], 8: [(1, 0), (0, 1)]}
WINNER = {1: (-1, -1), 2: (0, -1), 3: (1, -1), 4: (-1, 0), 5: (1, 0), 6: (-1, 1), 7: (0, 1), 8: (1, 1)}


@pytest.mark.parametrize("pt", range(1, 9))
def test_two_point_cases(tz, pt):
    """the first search ends at distance 1 with point pt: the two-point search probes its two points (d 2, p 0) around the winner"""
    wx, wy = WINNER[pt]
    d, s = synth(lambda x, y: np.where((x == wx) & (y == wy), 100, 500), R=8)
    trace, _ = run(tz, d, s)
    assert [t for t in stage(trace, 1) if (t[0], t[1]) == (wx, wy)][0][2] == pt
    assert stage(trace, 2, wx, wy) == [(dx, dy, 0, 2) for dx, dy in TWO[pt]]


def test_raster_order_and_star(tz):
    """the first search ends at distance 8 > 5: the raster visits the window in steps of 5, rows outer, columns inner; a star
    refinement follows"""
    f = lambda x, y: np.where((x == 0) & (y == -4), 200, np.where((x == 0) & (y == -8), 100, 500))   # noqa: E731
    d, s = synth(f, win=(-12, 12, -10, 8), R=8)
    trace, _ = run(tz, d, s)
    assert [(x, y) for x, y, p, dd, st, _ in trace if st == 3] == [(x, y) for y in (-10, -5, 0, 5) for x in (-12, -7, -2, 3, 8)]
    assert all(p == 0 and dd == 5 for _, _, p, dd, st, _ in trace if st == 3)
    assert any(t[4] == 4 for t in trace)


def test_raster_not_taken_at_distance_4(tz):
    trace, _ = run(tz, *synth(lambda x, y: np.where((x == 4) & (y == 0), 100, 500), R=64))
    assert not [t for t in trace if t[4] == 3]


def test_2nx2n_start_moves_the_raster_window(tz):
    """the 2Nx2N start (20, 30) wins the starts, so the raster window is +-R around it, clipped into the box"""
    f = lambda x, y: np.select([(x == 20) & (y == 30), (x == 20) & (y == 26), (x == 20) & (y == 22)], [200, 150, 100], 500)   # noqa: E731
    d, s = synth(f, win=(-16, 16, -16, 16), R=16, flags=TZ2N, mv2n=(20, 30))
    trace, _ = run(tz, d, s)
    assert [t[:2] for t in trace if t[4] == 0] == [(0, 0), (0, 0), (20, 30)]
    r = [t[:2] for t in trace if t[4] == 3]
    assert r[0] == (4, 14) and r[-1] == (34, 44)


def test_2nx2n_start_clamped_into_the_box(tz):
    d, s = synth(lambda x, y: 300 + (x - 7) ** 2 + (y + 3) ** 2, flags=TZ2N, mv2n=(500, -700))
    trace, _ = run(tz, d, s)
    assert [t[:2] for t in trace if t[4] == 0][2] == (B, -B)


def test_star_refinement_of_several_iterations(tz):
    """a bowl far from the start, distances up to 4 (no raster): the star refinement walks down to its bottom in many iterations"""
    trace, res = run(tz, *synth(lambda x, y: 3 * np.abs(x - 37) + 2 * np.abs(y + 23) + 10, pred=(12, -9), R=4))
    assert max(t[4] for t in trace) >= 4 + 2 * 5
    assert tuple(res[:2]) == (37, -23)


@pytest.mark.parametrize("R", [0, 1])
def test_small_search_ranges(tz, R):
    d, s = synth(lambda x, y: 300 + np.abs(x - 1) + np.abs(y + 1), R=R, win=(-R, R, -R, R))
    trace, _ = run(tz, d, s)
    assert stage(trace, 1) == ([] if R == 0 else [(0, -1, 2, 1), (-1, 0, 4, 1), (1, 0, 5, 1), (0, 1, 7, 1)])


def test_random_surfaces_windows_and_predictors(tz):
    """many walks on random surfaces, windows, predictors and lambdas: checker == Python statement, probe for probe"""
    rng = np.random.default_rng(5)
    for it in range(300):
        kind = it % 3
        if kind == 0:
            base = rng.integers(0, 1 << 12, (2 * B + 1, 2 * B + 1))
        elif kind == 1:                                                    # smooth bowls with noise: long walks
            cx, cy = rng.integers(-60, 61, 2)
            ys, xs = np.mgrid[-B:B + 1, -B:B + 1]
            base = 4 * np.abs(xs - cx) + 3 * np.abs(ys - cy) + rng.integers(0, 40, xs.shape)
        else:                                                              # few levels: ties everywhere
            base = rng.integers(0, 3, (2 * B + 1, 2 * B + 1)) * 50
        R = int(rng.choice([0, 1, 2, 3, 5, 8, 16, 33, 64]))
        l0, t0 = (int(v) for v in rng.integers(-B, B - 1, 2))
        win = (l0, int(rng.integers(l0, B + 1)), t0, int(rng.integers(t0, B + 1)))
        pred = tuple(int(v) for v in rng.integers(-4 * B - 40, 4 * B + 40, 2))
        lam = int(rng.choice([0, lambda_cost(22), lambda_cost(37), 0xFFFFFFFF]))
        flags = int(rng.choice([0, TZ2N]))
        mv2n = tuple(int(v) for v in rng.integers(-B - 20, B + 20, 2))
        d, s = synth(lambda x, y: base, win=win, R=R, pred=pred, lam=lam, flags=flags, mv2n=mv2n)
        run(tz, d, s)


def np_sad(sc, d, x, y):
    """xGetSAD* with numpy: rows stepped by 1 << sub_shift (generic widths: every row), sum << sub_shift >> (bd - 8)"""
    ss = d["sub_shift"] if d["w"] in (4, 8, 12, 16, 24, 32, 48, 64) else 0
    M = sc["M"]
    org = sc["org"][d["y"]:d["y"] + d["h"]:1 << ss, d["x"]:d["x"] + d["w"]].astype(np.int64)
    ref = sc["refs"][d["ref_idx"]][d["y"] + y + M:d["y"] + y + M + d["h"]:1 << ss, d["x"] + x + M:d["x"] + x + M + d["w"]].astype(np.int64)
    return (int(np.abs(org - ref).sum()) << ss) >> (sc["bd"] - 8)


@pytest.mark.parametrize("bd", [8, 10])
def test_pictures_against_the_statement(tz, bd):
    """real planes (moving texture, runs of 0 and 2^bd - 1): the checker's walk and SADs equal the statement on numpy SADs"""
    sc = mc_scene(bd, seed=bd + 70)
    rng = np.random.default_rng(bd)
    for w, h in MC_SHAPES[::3]:
        for R, fl in ((64, FRAC | HAD), (16, TZ2N), (3, FRAC)):
            x = int(rng.integers(0, (sc["W"] - w) // 4 + 1)) * 4
            y = int(rng.integers(0, (sc["H"] - h) // 4 + 1)) * 4
            pred = tuple(int(v) for v in rng.integers(-40, 41, 2))
            d = tz_desc(sc, x, y, w, h, sc["slots"][0], pred, R, sub_shift=int(rng.integers(0, 2)), lam=lambda_cost(30), flags=fl,
                        mv2n=tuple(int(v) for v in rng.integers(-10, 11, 2)))
            res, trace, _ = oracle_tz(tz, sc, d, trace_cap=100000)
            (mx, my, sad), want = py_tz_walk(d, lambda px, py: np_sad(sc, d, px, py))
            assert [tuple(int(v) for v in t) for t in trace] == [tuple(t) for t in want], d
            assert (int(res[0]), int(res[1]), int(res[2])) == (mx, my, sad)


def test_constant_planes_tie_on_cost(tz):
    """equal SADs everywhere: the motion-vector cost and HM's order decide, in both statements"""
    sc = mc_scene(8, seed=3)
    sc = dict(sc, org=np.full_like(sc["org"], 77), refs={s: np.full_like(p, 77) for s, p in sc["refs"].items()})
    for pred in ((0, 0), (13, -7), (-90, 41)):
        d = tz_desc(sc, 64, 32, 16, 16, sc["slots"][0], pred, 64, lam=lambda_cost(27), flags=TZ2N, mv2n=(3, 3))
        res, trace, _ = oracle_tz(tz, sc, d, trace_cap=100000)
        (mx, my, sad), want = py_tz_walk(d, lambda px, py: 0)
        assert [tuple(int(v) for v in t) for t in trace] == [tuple(t) for t in want]
        assert (int(res[0]), int(res[1]), int(res[2])) == (mx, my, 0)


def test_surface_must_cover_every_probe(tz):
    d, s = synth(lambda x, y: 500 + 0 * x)
    with pytest.raises(ValueError):
        oracle_tz(tz, {"bd": 8}, d, surface=(s[B - 2:B + 3, B - 2:B + 3], -2, -2))
