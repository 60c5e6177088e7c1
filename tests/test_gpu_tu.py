"""Parity of the intra TU coding kernels, luma and 4:2:0 chroma blocks (SURVEY.md 8f.2 / 8f.4, xIntraCodingTUBlock TEncSearch.cpp:1092-1387) through the C ABI:
against the TU records dumped from the reference encoder's own call sites (tests/golden/tu_*.npz) and against the oracle on
seeded random TUs.  Integer work: bit-exact."""
import numpy as np
import pytest

from _util import golden, oracle_intra_tu, tu_records

pytestmark = pytest.mark.gpu


def _pack(recs):
    tus = [(int(np.log2(r["n"])), r["mode"], r["qp"], r["ts"], r.get("chroma", 0)) for r in recs]
    org = np.concatenate([np.asarray(r["org"], np.int16).ravel() for r in recs])
    brd = np.concatenate([np.asarray(r["border"], np.int16).ravel() for r in recs])
    offs = np.cumsum([0] + [r["n"] ** 2 for r in recs])
    return tus, org, brd, offs


@pytest.mark.parametrize("clip", ["rdoq8", "hdq8", "hdq10"])
def test_tu_kernels_vs_reference_encoder_dump(cucd, clip):
    g = golden(f"tu_{clip}.npz")
    recs = list(tu_records(g))
    order = np.random.default_rng(5).permutation(len(recs))          # mixed sizes: exercises the size bucketing and scatter
    recs = [recs[i] for i in order]
    bd = recs[0]["bd"]
    tus, org, brd, offs = _pack(recs)
    with cucd.Engine(64, 64, bit_depth=bd) as eng:
        coef, pred = eng.intra_tu_forward(tus, org, brd)
        assert np.array_equal(pred, np.concatenate([r["pred"] for r in recs]))
        assert np.array_equal(coef, np.concatenate([r["coef"] for r in recs]))
        reco, dist = eng.intra_tu_recon(tus, org, brd, np.concatenate([r["level"] for r in recs]))
        assert np.array_equal(reco, np.concatenate([r["reco"] for r in recs]))
        assert np.array_equal(dist, np.array([r["dist"] for r in recs], np.uint32))
        if not recs[0]["rdoq"]:
            flags = (cucd.TU_INTRA_SLICE if recs[0]["intra"] else 0) | (cucd.TU_SIGN_HIDING if recs[0]["sbh"] else 0)
            level, reco2, dist2, abs_sum = eng.intra_tu_code(tus, org, brd, flags)
            assert np.array_equal(abs_sum, np.array([r["abs_sum"] for r in recs], np.int32))
            assert np.array_equal(level, np.concatenate([r["level"] for r in recs]))
            assert np.array_equal(reco2, reco) and np.array_equal(dist2, dist)


@pytest.mark.parametrize("bd", [8, 9, 10])
def test_tu_kernels_vs_oracle_random(cucd, oracle, bd):
    """every size x every mode, low and high QP, extreme samples, transform skip, sign hiding on/off, P-slice rounding"""
    rng = np.random.default_rng(40 + bd)
    hi = (1 << bd) - 1
    recs = []
    for n in (4, 8, 16, 32):
        for mode in range(35):
            for rep in range(2 if n < 32 else 1):
                kind = (mode + rep) % 3
                if kind == 0:
                    org = rng.integers(0, hi + 1, n * n)
                    brd = rng.integers(0, hi + 1, 4 * n + 1)
                elif kind == 1:                                       # smooth: small residuals, many zero levels, strong smoothing at 32
                    base = rng.integers(8, hi - 8)
                    org = base + rng.integers(-3, 4, n * n)
                    brd = base + rng.integers(-1, 2, 4 * n + 1)
                else:
                    org = rng.choice([0, hi], n * n)
                    brd = rng.choice([0, hi], 4 * n + 1)
                recs.append(dict(n=n, mode=mode, qp=int(rng.choice([0, 4, 17, 22, 27, 32, 37, 45, 51])), ts=int(n == 4 and rep == 1),
                                 chroma=int((mode + n) % 4 == 1),
                                 org=org.astype(np.int16), border=brd.astype(np.int16)))
    tus, org, brd, offs = _pack(recs)
    with cucd.Engine(64, 64, bit_depth=bd) as eng:
        coef, pred = eng.intra_tu_forward(tus, org, brd)
        for flags in (cucd.TU_INTRA_SLICE | cucd.TU_SIGN_HIDING, 0):
            level, reco, dist, abs_sum = eng.intra_tu_code(tus, org, brd, flags)
            reco2, dist2 = eng.intra_tu_recon(tus, org, brd, level)
            assert np.array_equal(reco2, reco) and np.array_equal(dist2, dist)          # stage 2 on stage 1's levels = stage 1
            for i, r in enumerate(recs):
                sl = slice(offs[i], offs[i + 1])
                w0 = oracle_intra_tu(oracle, bd, r["n"], r["mode"], r["qp"], r["ts"], r["org"], r["border"], 0, chroma=r["chroma"])
                assert np.array_equal(pred[sl], w0["pred"]) and np.array_equal(coef[sl], w0["coef"]), (r["n"], r["mode"], r["ts"])
                w1 = oracle_intra_tu(oracle, bd, r["n"], r["mode"], r["qp"], r["ts"], r["org"], r["border"], 1,
                                     intra=int(bool(flags & cucd.TU_INTRA_SLICE)), sbh=int(bool(flags & cucd.TU_SIGN_HIDING)), chroma=r["chroma"])
                assert abs_sum[i] == w1["abs_sum"] and np.array_equal(level[sl], w1["level"]), (r["n"], r["mode"], r["qp"], r["ts"], flags)
                assert np.array_equal(reco[sl], w1["reco"]) and dist[i] == w1["dist"]


def test_tu_edge_cases(cucd, oracle):
    with cucd.Engine(64, 64, bit_depth=8) as eng:
        c, p = eng.intra_tu_forward([], np.zeros(0, np.int16), np.zeros(0, np.int16))
        assert c.size == 0 and p.size == 0
        with pytest.raises(cucd.CucdError):
            eng.intra_tu_forward([(6, 0, 30, 0)], np.zeros(4096, np.int16), np.zeros(257, np.int16))      # 64x64 is not a TU size
        with pytest.raises(cucd.CucdError):
            eng.intra_tu_code([(3, 0, 30, 1)], np.zeros(64, np.int16), np.zeros(33, np.int16))            # transform skip is 4x4 only
        # ragged counts: not a multiple of the TUs-per-CTA chunk (16 for 4x4, 4 for 8x8)
        rng = np.random.default_rng(2)
        for n, cnt in ((4, 1), (4, 17), (4, 33), (8, 5), (16, 3), (32, 2)):
            recs = [dict(n=n, mode=int(rng.integers(0, 35)), qp=30, ts=0, org=rng.integers(0, 256, n * n).astype(np.int16),
                         border=rng.integers(0, 256, 4 * n + 1).astype(np.int16)) for _ in range(cnt)]
            tus, org, brd, offs = _pack(recs)
            level, reco, dist, abs_sum = eng.intra_tu_code(tus, org, brd)
            for i, r in enumerate(recs):
                w = oracle_intra_tu(oracle, 8, n, r["mode"], 30, 0, r["org"], r["border"], 1)
                assert np.array_equal(level[offs[i]:offs[i + 1]], w["level"]) and dist[i] == w["dist"] and abs_sum[i] == w["abs_sum"]
