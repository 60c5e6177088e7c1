"""The checker of the inter TU chain (tests/inter_tu_oracle.c, oracle_inter_tu) pinned on the CPU.  No encoder dump of
xEstimateResidualQT exists, so it is pinned through data that does: the intra TU records the reference encoder dumped
(tests/golden/tu_*.npz) for every TU whose intra chain ran the same transform (the DCT or transform skip), the reference's DCT
answers in tests/golden/ref_functions.npz for the 4x4 luma DCT that no intra TU uses, and the two semantics of the inter
chain that the intra one does not have (diagonal scan for sign hiding, rresi = 0 for zero levels)."""
import hashlib

import numpy as np
import pytest

from _util import P, golden, i16p, i32p
from inter_tu_util import load_inter_tu_oracle, oracle_inter_tu, oracle_sse, random_residual, tu_golden_inter_records, wrap_case


def digest(a):
    """the 64-bit digest tests/golden/ref_functions.npz records per answer (test_oracle_vs_ref.py)"""
    return np.frombuffer(hashlib.blake2b(np.ascontiguousarray(a).tobytes(), digest_size=8).digest(), np.uint64)[0]


@pytest.fixture(scope="module")
def ito():
    return load_inter_tu_oracle()


@pytest.mark.parametrize("clip", ["rdoq8", "hdq8", "hdq10"])
def test_forward_and_reconstruction_match_encoder_tu_records(ito, clip):
    recs = tu_golden_inter_records(golden(f"tu_{clip}.npz"))
    assert len(recs) > 100
    kinds = {(r["n"], r["chroma"], r["ts"]) for r in recs}
    assert {(4, 1, 0), (8, 0, 0), (32, 0, 0)} <= kinds and any(k[2] for k in kinds)
    for r in recs:
        n, bd = r["n"], r["bd"]
        w0 = oracle_inter_tu(ito, bd, n, r["qp"], r["ts"], r["chroma"], 1, 0, r["resi"])
        assert np.array_equal(w0["coef"], np.asarray(r["coef"]).ravel()), (n, r["chroma"], r["ts"])
        assert w0["dist_zero"] == oracle_sse(ito, bd, r["resi"], np.zeros(n * n, np.int16))
        w2 = oracle_inter_tu(ito, bd, n, r["qp"], r["ts"], r["chroma"], 1, 2, r["resi"], level_in=np.asarray(r["level"]).ravel())
        reco = np.clip(np.asarray(r["pred"], np.int32).ravel() + w2["rresi"], 0, (1 << bd) - 1).astype(np.int16)
        assert np.array_equal(reco, np.asarray(r["reco"]).ravel()), (n, r["chroma"], r["ts"])
        assert oracle_sse(ito, bd, reco, np.asarray(r["org"], np.int16).ravel()) == r["dist"]


@pytest.mark.parametrize("bd", [8, 10])
def test_4x4_dct_pair_is_the_one_the_reference_answers_pin(ito, bd):
    """The checker's 4x4 forward is oracle_fwd_transform(useDST = 0); its inverse on dequantised levels is
    oracle_inv_transform(useDST = 0).  Both are pinned here again on the inputs of the recorded reference answers
    (test_oracle_vs_ref.py::test_core_transforms_match_reference, n = 4): the DCT answers come from the checker's stage 0."""
    n = 4
    rng = np.random.default_rng(200 + n + bd)
    hi = (1 << bd) - 1
    answers = []
    for trial in range(40):
        kind = trial % 4
        if kind == 0:
            resi = rng.integers(-hi, hi + 1, (n, n))
        elif kind == 1:
            resi = rng.choice([-hi, hi], size=(n, n))
        elif kind == 2:
            resi = np.full((n, n), hi if trial % 8 < 4 else -hi)
        else:
            resi = rng.integers(-6, 7, (n, n))
        resi16 = np.ascontiguousarray(resi.astype(np.int16))
        for dst in (0, 1):
            got = np.zeros(n * n, np.int32)
            if dst == 0:
                got = oracle_inter_tu(ito, bd, n, 30, 0, 0, 0, 0, resi16)["coef"]
            else:
                ito.oracle_fwd_transform(bd, n, 1, P(resi16, i16p), n, P(got, i32p))
            answers.append(got)
            for coef in (got, rng.choice([-32768, 32767], size=n * n).astype(np.int32), (got * 3).clip(-32768, 32767).astype(np.int32)):
                gres = np.zeros(n * n, np.int16)
                ito.oracle_inv_transform(bd, n, dst, P(np.ascontiguousarray(coef), i32p), P(gres, i16p), n)
                answers.append(gres)
    want = golden("ref_functions.npz")[f"transforms_n4_bd{bd}"]
    assert np.array_equal(np.array([digest(a) for a in answers], np.uint64), want)
    # the inverse of stage 2 is the DCT one: rresi = xIT(useDST = 0) of the dequantised levels, and differs from the DST's
    for qp in (4, 22, 37):
        level = rng.integers(-40, 41, n * n).astype(np.int32)
        deq = np.zeros(n * n, np.int32)
        ito.oracle_dequant(bd, n, qp, P(level, i32p), P(deq, i32p))
        dct, dst = np.zeros(n * n, np.int16), np.zeros(n * n, np.int16)
        ito.oracle_inv_transform(bd, n, 0, P(deq, i32p), P(dct, i16p), n)
        ito.oracle_inv_transform(bd, n, 1, P(deq, i32p), P(dst, i16p), n)
        w = oracle_inter_tu(ito, bd, n, qp, 0, 0, 1, 2, np.zeros(n * n, np.int16), level_in=level)
        assert np.array_equal(w["rresi"], dct) and not np.array_equal(dct, dst)


def test_sign_hiding_uses_the_diagonal_scan(ito):
    """a seeded block where oracle_quant with the horizontal / vertical scan hides a different sign than with the diagonal one:
    the checker gives the diagonal scan's levels"""
    bd, n = 8, 8
    found = 0
    for seed in range(400):
        resi = random_residual(np.random.default_rng(seed), n, bd, seed % 4)
        qp = 22 + seed % 15
        c = oracle_inter_tu(ito, bd, n, qp, 0, 0, 1, 0, resi)["coef"]
        lv = {}
        for scan in (0, 1, 2):
            lv[scan] = np.zeros(n * n, np.int32)
            ito.oracle_quant(bd, n, qp, 0, 1, scan, P(c, i32p), P(lv[scan], i32p))
        if np.array_equal(lv[0], lv[1]) and np.array_equal(lv[0], lv[2]):
            continue
        w = oracle_inter_tu(ito, bd, n, qp, 0, 0, 1, 1, resi)
        assert np.array_equal(w["level"], lv[0]), seed
        found += 1
    assert found >= 5


@pytest.mark.parametrize("bd", [8, 10])
def test_zero_levels_give_zero_rresi_and_the_zero_distortion(ito, bd):
    rng = np.random.default_rng(bd)
    for n in (4, 8, 16, 32):
        for ts in ((0, 1) if n == 4 else (0,)):
            resi = random_residual(rng, n, bd, 0)
            w = oracle_inter_tu(ito, bd, n, 30, ts, 0, 1, 2, resi, level_in=np.zeros(n * n, np.int32))
            assert not w["rresi"].any() and w["abs_sum"] == 0
            assert w["dist"] == w["dist_zero"] == oracle_sse(ito, bd, resi, np.zeros((n, n), np.int16))
            # a residual the quantiser zeroes: stage 1 gives the same
            small = np.ones((n, n), np.int16)
            w1 = oracle_inter_tu(ito, bd, n, 51, ts, 0, 1, 1, small)
            assert w1["abs_sum"] == 0 and not w1["level"].any() and not w1["rresi"].any() and w1["dist"] == w1["dist_zero"] == (n * n if bd == 8 else 0)


def test_distortion_wraps_like_a_uint32(ito):
    """the checker keeps HM's wrapped uint32 Distortion"""
    level, resi = wrap_case(ito)
    w = oracle_inter_tu(ito, 10, 32, 51, 0, 0, 1, 2, resi, level_in=level)
    exact = int((((resi.astype(np.int64) - w["rresi"]) ** 2) >> 4).sum())
    assert exact >= 1 << 32 and w["dist"] == exact % (1 << 32)
