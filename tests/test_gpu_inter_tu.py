"""cucd_inter_tu_forward / _recon / _code through the C ABI against the checker tests/inter_tu_oracle.c: transform, quantisation and
distortion of the TUs of inter residual quadtrees (xEstimateResidualQT).  Integer work: bit-exact."""
import numpy as np
import pytest

from _util import P, golden, i16p, i32p, load_oracle, oracle_intra_tu
from inter_tu_util import load_inter_tu_oracle, oracle_inter_tu, oracle_sse, random_residual, tu_golden_inter_records, wrap_case

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ito():
    return load_inter_tu_oracle()


def random_tus(rng, bd, count):
    """(log2, qp, ts, chroma) records and their residuals: every size, luma and chroma, transform skip at 4x4, QPs over 0..51"""
    tus, res = [], []
    for i in range(count):
        lg = int(rng.integers(2, 6))
        chroma = int(lg < 5 and rng.random() < 0.35)
        ts = int(lg == 2 and rng.random() < 0.4)
        qp = int(rng.choice([0, 1, 9, 17, 22, 27, 32, 37, 42, 47, 51])) if i % 3 else int(rng.integers(0, 52))
        tus.append((lg, qp, ts, chroma))
        res.append(random_residual(rng, 1 << lg, bd, i % 4).ravel())
    return tus, res


def check_all_calls(eng, ito, bd, tus, res):
    """the three calls on one batch against the checker, per TU: coef, dist_zero; level, rresi, dist, abs_sum (sign hiding on
    and off); the reconstruction half on the levels of the whole chain"""
    resi = np.concatenate(res)
    offs = np.cumsum([0] + [r.size for r in res])
    coef, dz0 = eng.inter_tu_forward(tus, resi)
    for sbh in (1, 0):
        level, rresi, dist, dz, abs_sum = eng.inter_tu_code(tus, resi, sign_hiding=bool(sbh))
        rresi2, dist2 = eng.inter_tu_recon(tus, resi, level)
        assert np.array_equal(rresi2, rresi) and np.array_equal(dist2, dist) and np.array_equal(dz, dz0)
        for i, (lg, qp, ts, ch) in enumerate(tus):
            n, sl = 1 << lg, slice(offs[i], offs[i + 1])
            w = oracle_inter_tu(ito, bd, n, qp, ts, ch, sbh, 1, res[i])
            key = (i, n, qp, ts, ch, sbh)
            assert np.array_equal(coef[sl], w["coef"]) and dz0[i] == w["dist_zero"], key
            assert abs_sum[i] == w["abs_sum"] and np.array_equal(level[sl], w["level"]), key
            assert np.array_equal(rresi[sl], w["rresi"]) and dist[i] == w["dist"], key


@pytest.mark.parametrize("bd", [8, 9, 10])
def test_random_batches_vs_checker(cucd, ito, bd):
    """shuffled sizes (size bucketing and the scatter back to caller order), in a small batch and in one of 6000 TUs that spans
    several waves of CTAs"""
    rng = np.random.default_rng(70 + bd)
    with cucd.Engine(64, 64, bit_depth=bd) as eng:
        for count in (300, 6000):
            tus, res = random_tus(rng, bd, count)
            check_all_calls(eng, ito, bd, tus, res)


@pytest.mark.parametrize("clip", ["rdoq8", "hdq8", "hdq10"])
def test_encoder_tu_records_through_the_inter_calls(cucd, ito, clip):
    """the intra TU records the reference encoder dumped whose transform is the inter chain's (DCT or transform skip): forward on
    org - pred gives the dumped coef, the reconstruction half on the dumped levels gives the dumped reco and dist"""
    recs = tu_golden_inter_records(golden(f"tu_{clip}.npz"))
    recs = [recs[i] for i in np.random.default_rng(6).permutation(len(recs))]
    bd = recs[0]["bd"]
    tus = [(int(np.log2(r["n"])), r["qp"], r["ts"], r["chroma"]) for r in recs]
    resi = np.concatenate([r["resi"] for r in recs])
    offs = np.cumsum([0] + [r["n"] ** 2 for r in recs])
    with cucd.Engine(64, 64, bit_depth=bd) as eng:
        coef, dz = eng.inter_tu_forward(tus, resi)
        assert np.array_equal(coef, np.concatenate([np.asarray(r["coef"]).ravel() for r in recs]))
        rresi, dist = eng.inter_tu_recon(tus, resi, np.concatenate([np.asarray(r["level"]).ravel() for r in recs]))
    for i, r in enumerate(recs):
        sl = slice(offs[i], offs[i + 1])
        reco = np.clip(np.asarray(r["pred"], np.int32).ravel() + rresi[sl], 0, (1 << bd) - 1).astype(np.int16)
        assert np.array_equal(reco, np.asarray(r["reco"]).ravel()), i
        assert oracle_sse(ito, bd, reco, np.asarray(r["org"], np.int16).ravel()) == r["dist"]
        w = oracle_inter_tu(ito, bd, r["n"], r["qp"], r["ts"], r["chroma"], 1, 2, r["resi"], level_in=np.asarray(r["level"]).ravel())
        assert np.array_equal(rresi[sl], w["rresi"]) and dist[i] == w["dist"] and dz[i] == w["dist_zero"]


@pytest.mark.parametrize("bd", [8, 9, 10])
def test_extreme_residuals(cucd, ito, bd):
    """+-(2^bd - 1) constant and checkerboard blocks at every size (luma, chroma, transform skip), low and high QP; an all-zero
    residual gives abs_sum 0 and dist 0"""
    hi = (1 << bd) - 1
    tus, res = [], []
    for lg in (2, 3, 4, 5):
        n = 1 << lg
        cb = np.where(np.indices((n, n)).sum(0) % 2 == 0, hi, -hi)
        for blk in (np.full((n, n), hi), np.full((n, n), -hi), cb, -cb, np.zeros((n, n))):
            for qp in (0, 22, 51):
                for ts, ch in ((0, 0), (0, 1)) + (((1, 0), (1, 1)) if lg == 2 else ()):
                    if ch and lg == 5:
                        continue
                    tus.append((lg, qp, ts, ch))
                    res.append(blk.astype(np.int16).ravel())
    with cucd.Engine(64, 64, bit_depth=bd) as eng:
        check_all_calls(eng, ito, bd, tus, res)
        level, rresi, dist, dz, abs_sum = eng.inter_tu_code(tus, np.concatenate(res))
    zero = [i for i, r in enumerate(res) if not r.any()]
    assert zero and all(abs_sum[i] == 0 and dist[i] == 0 and dz[i] == 0 for i in zero)


def test_recon_distortion_wraps_past_2_32(cucd, ito):
    """_recon with levels of +-32767 at 32x32, 10 bit: the SSE passes 2^32 and dist is the checker's wrapped uint32"""
    level, resi = wrap_case(ito)
    w = oracle_inter_tu(ito, 10, 32, 51, 0, 0, 1, 2, resi, level_in=level)
    exact = int((((resi.astype(np.int64) - w["rresi"]) ** 2) >> 4).sum())
    assert exact >= 1 << 32
    with cucd.Engine(64, 64, bit_depth=10) as eng:
        rresi, dist = eng.inter_tu_recon([(5, 51, 0, 0)] * 2, np.concatenate([resi, resi]), np.concatenate([level, level]))
    assert np.array_equal(rresi[:1024], w["rresi"]) and list(dist) == [w["dist"], w["dist"]] == [exact % (1 << 32)] * 2


def test_luma_4x4_is_the_dct(cucd, ito):
    """a luma 4x4 residual whose intra DST and DCT coefficients differ: the inter coefficients are the DCT's"""
    bd = 8
    resi = random_residual(np.random.default_rng(3), 4, bd, 0)
    dct = oracle_inter_tu(ito, bd, 4, 30, 0, 0, 1, 0, resi)["coef"]
    dst = np.zeros(16, np.int32)
    ito.oracle_fwd_transform(bd, 4, 1, P(np.ascontiguousarray(resi), i16p), 4, P(dst, i32p))
    assert not np.array_equal(dct, dst)
    with cucd.Engine(64, 64, bit_depth=bd) as eng:
        coef, _ = eng.inter_tu_forward([(2, 30, 0, 0)], resi)
    assert np.array_equal(coef, dct)


@pytest.mark.parametrize("bd", [8, 10])
def test_from_motion_compensation_to_the_residual_quadtree(cucd, ito, bd):
    """bi- and uni-predictive 64x64 candidates through cucd_me_mc_cost(..., pred), resi = org - pred on the host, and every TU of the
    CU's inter RQT (32, 16, 8, 4) of all candidates in one cucd_inter_tu_code call; the dist_zero of the TUs that tile the PU at
    each depth sum to oracle_sse(org, pred)"""
    from mc_util import load_mc_oracle, mc_scene, oracle_mc
    sc = mc_scene(bd, seed=20 + bd)
    x, y = 64, 32
    descs = [dict(x=x, y=y, w=64, h=64, ref_idx=(0, 3), mvx=(13, -22), mvy=(-7, 30), use_hadamard=1),
             dict(x=x, y=y, w=64, h=64, ref_idx=(0, -1), mvx=(-41, 0), mvy=(18, 0), use_hadamard=0),
             dict(x=x, y=y, w=64, h=64, ref_idx=(-1, 3), mvx=(0, 6), mvy=(0, -5), use_hadamard=1)]
    eng = cucd.Engine(sc["W"], sc["H"], bit_depth=bd)
    try:
        eng.set_cur_picture(sc["org"])
        for s, p in sc["refs"].items():
            eng.set_ref_picture(s, p, sc["M"], sc["M"])
        dist_mc, preds = eng.me_mc_cost(descs, want_pred=True)
        want_d, want_p = oracle_mc(load_mc_oracle(), sc, descs)
        assert np.array_equal(dist_mc, want_d) and all(np.array_equal(a, b) for a, b in zip(preds, want_p))
        org = sc["org"][y:y + 64, x:x + 64].astype(np.int32)
        tus, res, owner = [], [], []
        for c, pred in enumerate(preds):
            resi = (org - pred).astype(np.int16)
            for lg in (5, 4, 3, 2):
                n = 1 << lg
                for by in range(0, 64, n):
                    for bx in range(0, 64, n):
                        tus.append((lg, 27 + c, 0, 0))
                        res.append(np.ascontiguousarray(resi[by:by + n, bx:bx + n]).ravel())
                        owner.append((c, lg))
        level, rresi, dist, dz, abs_sum = eng.inter_tu_code(tus, np.concatenate(res))
    finally:
        eng.close()
    offs = np.cumsum([0] + [r.size for r in res])
    for i, (lg, qp, ts, ch) in enumerate(tus):
        w = oracle_inter_tu(ito, bd, 1 << lg, qp, ts, ch, 1, 1, res[i])
        sl = slice(offs[i], offs[i + 1])
        assert np.array_equal(level[sl], w["level"]) and np.array_equal(rresi[sl], w["rresi"]), i
        assert (dist[i], dz[i], abs_sum[i]) == (w["dist"], w["dist_zero"], w["abs_sum"]), i
    for c, pred in enumerate(preds):
        want = oracle_sse(ito, bd, sc["org"][y:y + 64, x:x + 64], pred)
        for lg in (5, 4, 3, 2):
            assert sum(int(dz[i]) for i, o in enumerate(owner) if o == (c, lg)) == want, (c, lg)


def test_rejections_and_the_empty_call(cucd, ito):
    """every invalid argument returns an error and leaves the handle usable; nTU == 0 is a no-op; an intra TU call afterwards still
    matches its oracle"""
    eng = cucd.Engine(64, 64, bit_depth=8)
    lib, h = eng.lib, eng.h
    resi = np.zeros(32 * 32 * 2, np.int16)
    out32 = np.zeros(32 * 32 * 2, np.int32); out16 = np.zeros(32 * 32 * 2, np.int16)
    u1, u2, s1 = np.zeros(2, np.uint32), np.zeros(2, np.uint32), np.zeros(2, np.int32)
    good = tu_desc_array([(3, 0, 30, 0)])
    R, O, L = resi.ctypes.data, out32.ctypes.data, out16.ctypes.data
    fwd = lambda n, d, r=R, c=O: lib.cucd_inter_tu_forward(h, n, d, r, c, u1.ctypes.data)
    rec = lambda n, d, r=R, lv=O, dist=u1.ctypes.data: lib.cucd_inter_tu_recon(h, n, d, r, lv, L, dist)
    code = lambda n, d, flags=2, r=R, lv=O, rr=L, dist=u1.ctypes.data: lib.cucd_inter_tu_code(h, n, d, r, flags, lv, rr, dist, u2.ctypes.data, s1.ctypes.data)
    try:
        for call in (fwd, rec, code):
            assert call(0, None) == 0 and call(0, good, r=None) == 0                       # nTU == 0: no-op, nothing read
            assert call(-1, good) == -1
            assert call(1, None) == -1
            assert call(1, good, r=None) == -1
            for bad, rc in (((1, 0, 30, 0), -1), ((6, 0, 30, 0), -1), ((3, 0, -1, 0), -1), ((3, 0, 52, 0), -1), ((3, 1, 30, 0), -1),
                            ((3, 26, 30, 0), -1), ((3, 0, 30, 4), -1), ((3, 0, 30, 0x80), -1), ((3, 0, 30, 1), -2), ((5, 0, 30, 3), -2)):
                assert call(1, tu_desc_array([bad])) == rc, (call, bad)
        assert fwd(1, good, c=None) == -1
        assert rec(1, good, lv=None) == -1 and rec(1, good, dist=None) == -1
        assert code(1, good, lv=None) == -1 and code(1, good, rr=None) == -1 and code(1, good, dist=None) == -1
        assert code(1, good, flags=1) == -1 and code(1, good, flags=3) == -1 and code(1, good, flags=4) == -1
        # optional outputs may be NULL
        assert lib.cucd_inter_tu_forward(h, 1, good, R, O, None) == 0
        assert lib.cucd_inter_tu_recon(h, 1, good, R, O, None, u1.ctypes.data) == 0
        assert lib.cucd_inter_tu_code(h, 1, good, R, 0, O, L, u1.ctypes.data, None, None) == 0
        # the handle still works: an inter call and an intra TU call match their checkers
        rng = np.random.default_rng(8)
        r8 = random_residual(rng, 8, 8, 0)
        level, rresi, dist, dz, abs_sum = eng.inter_tu_code([(3, 30, 0, 0)], r8)
        w = oracle_inter_tu(ito, 8, 8, 30, 0, 0, 1, 1, r8)
        assert np.array_equal(level, w["level"]) and dist[0] == w["dist"]
        t_org = rng.integers(0, 256, 64).astype(np.int16); t_brd = rng.integers(0, 256, 33).astype(np.int16)
        lv, reco, d, a = eng.intra_tu_code([(3, 18, 32, 0)], t_org, t_brd)
        wi = oracle_intra_tu(load_oracle(), 8, 8, 18, 32, 0, t_org, t_brd, 1)
        assert np.array_equal(lv, wi["level"]) and np.array_equal(reco, wi["reco"]) and d[0] == wi["dist"]
    finally:
        eng.close()


def tu_desc_array(descs):
    """raw cucd_tu_desc records (log2_size, mode, qp, flags), unchecked"""
    import importlib
    T = importlib.import_module("fast-cu-decision-hevc_b200.binding")._TuDesc
    arr = (T * len(descs))()
    for i, (l, m, q, f) in enumerate(descs):
        arr[i].log2_size, arr[i].mode, arr[i].qp, arr[i].flags = l, m, q, f
    return arr
