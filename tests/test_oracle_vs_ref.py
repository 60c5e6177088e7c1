"""The oracle against the reference's own compiled functions (oracle/_ref/libhmref.so) on seeded random
inputs - covers what the encoder dumps cannot reach (arbitrary availability patterns, extreme sample
values, every mode's raw prediction block).

Where oracle/_ref was built, every answer is compared with the live reference.  Everywhere, the answers
are compared with the reference's answers to the same inputs recorded as 64-bit digests in
tests/golden/ref_functions.npz (tests/golden/gen_golden_ref_functions.py), so a checkout without the
reference runs the same comparison."""
import hashlib

import numpy as np
import pytest

from _util import P, golden, i16p, i32p, u8p, u32p, f64p, oracle_outlier_frame, oracle_ctu_src_had, textured_plane

SIZES = [4, 8, 16, 32, 64]
RECORD = None          # tests/golden/gen_golden_ref_functions.py sets a dict here: answers are recorded instead of checked
_recorded = None


def digest(a):
    return np.frombuffer(hashlib.blake2b(np.ascontiguousarray(a).tobytes(), digest_size=8).digest(), np.uint64)[0]


def check_recorded(key, answers):
    """the oracle's answers of one test case, in order, against the digests of the reference's answers to the same inputs"""
    global _recorded
    got = np.array([digest(a) for a in answers], np.uint64)
    if RECORD is not None:
        RECORD[key] = got
        return
    if _recorded is None:
        _recorded = golden("ref_functions.npz")
    want = _recorded[key]
    assert len(got) == len(want), key
    bad = np.nonzero(got != want)[0]
    assert not len(bad), f"{key}: the oracle differs from the reference at answers {bad[:20].tolist()} of {len(want)}"


def rand_border(rng, n, bd, kind):
    hi = (1 << bd) - 1
    if kind == 0:
        return rng.integers(0, hi + 1, 4 * n + 1).astype(np.int16)
    if kind == 1:  # smooth ramp: makes strong smoothing fire
        return np.clip(np.linspace(rng.integers(0, hi), rng.integers(0, hi), 4 * n + 1) + rng.integers(-1, 2, 4 * n + 1), 0, hi).astype(np.int16)
    return np.full(4 * n + 1, rng.integers(0, hi + 1), np.int16)


@pytest.mark.parametrize("bd", [8, 10])
@pytest.mark.parametrize("n", SIZES)
def test_fill_border_random_flags(oracle, hmref, n, bd):
    rng = np.random.default_rng(100 + n + bd)
    S = 2 * n + 40
    answers = []
    for trial in range(60):
        rec = rng.integers(0, 1 << bd, (S, S)).astype(np.int16)
        flags = (rng.random(n + 1) < rng.choice([0.0, 0.3, 0.7, 1.0])).astype(np.uint8)
        if trial == 0:
            flags[:] = 0
        a = np.zeros(4 * n + 1, np.int16)
        base = rec.ctypes.data + 2 * (20 * S + 20)
        import ctypes as C
        oracle.oracle_fill_border(bd, n, C.c_void_p(base), S, P(flags, u8p), P(a, i16p))
        if hmref:
            b = np.zeros(4 * n + 1, np.int16)
            hmref.hmref_fill_border(bd, n, C.c_void_p(base), S, P(flags, u8p), P(b, i16p))
            assert np.array_equal(a, b), (trial, flags)
        answers.append(a)
    check_recorded(f"fill_border_n{n}_bd{bd}", answers)


@pytest.mark.parametrize("bd", [8, 10])
@pytest.mark.parametrize("n", SIZES)
def test_every_mode_prediction_block(oracle, hmref, n, bd):
    rng = np.random.default_rng(200 + n + bd)
    answers = []
    for trial in range(6):
        border = rand_border(rng, n, bd, trial % 3)
        fil = np.zeros(4 * n + 1, np.int16)
        oracle.oracle_filter_border(bd, n, 1, P(border, i16p), P(fil, i16p))
        for mode in range(35):
            a = np.zeros(n * n, np.int16)
            oracle.oracle_predict(bd, n, mode, P(border, i16p), P(fil, i16p), P(a, i16p))
            if hmref:
                b = np.zeros(n * n, np.int16)
                hmref.hmref_predict(bd, n, mode, P(border, i16p), 0, 1, P(b, i16p))
                assert np.array_equal(a, b), (trial, mode)
            answers.append(a)
    check_recorded(f"predict_n{n}_bd{bd}", answers)


@pytest.mark.parametrize("bd", [8, 10])
@pytest.mark.parametrize("n", SIZES)
def test_rmd_pu_random(oracle, hmref, n, bd):
    rng = np.random.default_rng(300 + n + bd)
    answers = []
    for trial in range(8):
        border = rand_border(rng, n, bd, trial % 3)
        org = rng.integers(0, 1 << bd, n * n).astype(np.int16) if trial % 2 else np.full(n * n, (1 << bd) - 1, np.int16)
        a = np.zeros(35, np.uint32)
        oracle.oracle_rmd_pu(bd, n, 1, P(org, i16p), n, P(border, i16p), P(a, u32p))
        if hmref:
            b = np.zeros(35, np.uint32)
            hmref.hmref_rmd_pu(bd, n, 1, P(org, i16p), n, P(border, i16p), P(b, u32p))
            assert np.array_equal(a, b), trial
        answers.append(a)
    check_recorded(f"rmd_pu_n{n}_bd{bd}", answers)


@pytest.mark.parametrize("bd", [8, 10])
def test_satd_and_sad_shapes(oracle, hmref, bd):
    rng = np.random.default_rng(400 + bd)
    answers = []
    for (w, h) in [(4, 4), (8, 8), (16, 16), (32, 32), (64, 64), (8, 4), (4, 8), (16, 4), (12, 16), (24, 32), (48, 64), (64, 16), (16, 64)]:
        o = rng.integers(0, 1 << bd, (h, w)).astype(np.int16)
        r = rng.integers(0, 1 << bd, (h, w)).astype(np.int16)
        satd = oracle.oracle_satd(bd, P(o, i16p), w, P(r, i16p), w, w, h)
        if hmref:
            assert satd == hmref.hmref_hads(bd, P(o, i16p), w, P(r, i16p), w, w, h)
        answers.append(np.uint32(satd))
        for sub in (0, 1, 2):
            if h >> sub < 1 or (h % (1 << sub)):
                continue
            sad = oracle.oracle_sad(bd, P(o, i16p), w, P(r, i16p), w, w, h, sub)
            if hmref:
                assert sad == hmref.hmref_sad(bd, P(o, i16p), w, P(r, i16p), w, w, h, sub), (w, h, sub)
            answers.append(np.uint32(sad))
    check_recorded(f"satd_sad_bd{bd}", answers)


@pytest.mark.parametrize("bd,W,H", [(8, 192, 128), (10, 136, 72)])
def test_outlier_frame_and_src_had(oracle, hmref, bd, W, H):
    org = textured_plane(W, H, bd, seed=31 + bd)
    obf, outl, _ = oracle_outlier_frame(oracle, org, bd)
    if hmref:
        robf = np.zeros_like(obf)
        rout = np.zeros_like(outl)
        hmref.hmref_outlier_frame(bd, P(org, i16p), W, W, H, P(robf, i16p), P(rout, i16p))
        assert np.array_equal(obf, robf)
        assert np.array_equal(outl, rout)
    had = oracle_ctu_src_had(oracle, org)
    if hmref:
        wc = (W + 63) // 64
        for ctu in range(len(had)):
            cx, cy = (ctu % wc) * 64, (ctu // wc) * 64
            tot = 0
            for y in range(cy, min(cy + 64, H) - 7, 8):
                for x in range(cx, min(cx + 64, W) - 7, 8):
                    blk = np.ascontiguousarray(org[y:y + 8, x:x + 8])
                    tot += hmref.hmref_src_had8x8(P(blk, i16p), 8)
            assert had[ctu] == tot
    check_recorded(f"outlier_src_had_bd{bd}_{W}x{H}", [obf, outl, had])


def test_rmd_frame_enumeration(oracle, hmref):
    """replay-mode enumeration (z-scan availability + fill + 35 modes) on a picture with partial CTUs"""
    from _util import oracle_rmd_frame, pseudo_recon
    W, H, bd = 136, 88, 8
    org = textured_plane(W, H, bd, seed=77)
    rec = pseudo_recon(org, bd)
    a = oracle_rmd_frame(oracle, org, rec, bd)
    if hmref:
        b = np.zeros_like(a)
        hmref.hmref_rmd_frame(bd, 1, P(org, i16p), W, P(rec, i16p), W, W, H, 0, a.shape[0], 2, P(b, u32p))
        assert np.array_equal(a, b)
    check_recorded("rmd_frame", list(a))


@pytest.mark.parametrize("bd,W,H", [(8, 200, 136), (10, 136, 72), (8, 64, 64)])
def test_tmv_features_and_aq_activity_match_reference(oracle, hmref, bd, W, H):
    """a12 / a13: the oracle against the reference's own getTMVFeature and TEncPreanalyzer::xPreanalyze (doubles, bit-exact)."""
    import ctypes as C
    from _util import all_cus, oracle_aq_activity, oracle_tmv_features, f64p
    org = textured_plane(W, H, bd, seed=3)
    # extreme content too: the quirky triangle entries and the truncation toward zero depend on signs
    ext = np.random.default_rng(5).choice([0, (1 << bd) - 1], size=(H, W)).astype(np.int16)
    answers = []
    for plane in (org, ext):
        cus = all_cus(W, H)[::3]
        got = oracle_tmv_features(oracle, plane, cus)
        if hmref:
            want = np.zeros((len(cus), 5, 26))
            for i, (x, y, l) in enumerate(cus):
                hmref.hmref_tmv_features(P(plane, i16p), W, W, H, x, y, 1 << l, C.c_void_p(want[i].ctypes.data))
            assert np.array_equal(got, want)
        acts, avg = oracle_aq_activity(oracle, plane, 4)
        if hmref:
            ref = [np.zeros_like(a) for a in acts]
            ptrs = (C.c_void_p * 4)(*[a.ctypes.data for a in ref])
            ravg = np.zeros(4)
            hmref.hmref_aq_activity(P(plane, i16p), W, W, H, 4, ptrs, P(ravg, f64p))
            for a, b in zip(acts, ref):
                assert np.array_equal(a, b)
            assert np.array_equal(avg, ravg)
        answers += list(got) + acts + [avg]
    check_recorded(f"tmv_aq_bd{bd}_{W}x{H}", answers)


@pytest.mark.parametrize("bd", [8, 10])
@pytest.mark.parametrize("n", [4, 8, 16, 32])
def test_core_transforms_match_reference(oracle, hmref, n, bd):
    """xTrMxN / xITrMxN (TComTrQuant.cpp:860-985) on random and extreme inputs, DCT and (4x4) DST; the restated matrices
    against the reference's partial butterflies, including the 16-bit clipping of the inverse's first stage."""
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
        resi16 = resi.astype(np.int16)
        for dst in ([0, 1] if n == 4 else [0]):
            got = np.zeros(n * n, np.int32)
            oracle.oracle_fwd_transform(bd, n, dst, P(resi16, i16p), n, P(got, i32p))
            if hmref:
                want = np.zeros(n * n, np.int32)
                hmref.hmref_fwd_transform(bd, n, dst, P(np.ascontiguousarray(resi.astype(np.int32)), i32p), P(want, i32p))
                assert np.array_equal(got, want)
            answers.append(got)
            # inverse on the forward output and on extreme coefficient blocks
            for coef in (got, rng.choice([-32768, 32767], size=n * n).astype(np.int32), (got * 3).clip(-32768, 32767).astype(np.int32)):
                gres = np.zeros(n * n, np.int16)
                oracle.oracle_inv_transform(bd, n, dst, P(np.ascontiguousarray(coef), i32p), P(gres, i16p), n)
                if hmref:
                    wres = np.zeros(n * n, np.int32)
                    hmref.hmref_inv_transform(bd, n, dst, P(np.ascontiguousarray(coef), i32p), P(wres, i32p))
                    assert np.array_equal(gres.astype(np.int32), wres)
                answers.append(gres)
    check_recorded(f"transforms_n{n}_bd{bd}", answers)


def test_sse_matches_reference(oracle, hmref):
    oracle.oracle_sse.restype = __import__("ctypes").c_uint32
    if hmref:
        hmref.hmref_sse.restype = __import__("ctypes").c_uint32
    rng = np.random.default_rng(9)
    answers = []
    for bd in (8, 10):
        for n in (4, 8, 16, 32):
            a = rng.integers(0, 1 << bd, (n, n)).astype(np.int16)
            b = rng.integers(0, 1 << bd, (n, n)).astype(np.int16)
            sse = oracle.oracle_sse(bd, P(a, i16p), n, P(b, i16p), n, n, n)
            if hmref:
                assert sse == hmref.hmref_sse(bd, P(a, i16p), n, P(b, i16p), n, n, n)
            answers.append(np.uint32(sse))
    check_recorded("sse", answers)
