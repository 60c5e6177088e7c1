"""CPU replay of the CUDA kernels' per-thread code (tests/emul, built from the same __host__ __device__
headers the sm_100a kernels compile) against the golden vectors and the oracle.  Lets the kernel
arithmetic be checked where there is no GPU; the -m gpu tests check the real kernels."""
import numpy as np
import pytest

from _util import P, golden, i16p, i32p, u8p, u32p, oracle_outlier_frame, oracle_rmd_frame, pseudo_recon, textured_plane


@pytest.mark.parametrize("clip", ["ai8", "ai10"])
@pytest.mark.parametrize("n", [4, 8, 16, 32, 64])
def test_batch_kernel_code_vs_golden(emul, clip, n):
    g = golden(f"rmd_{clip}.npz")
    bd = int(g["meta"][2])
    org = np.ascontiguousarray(g[f"n{n}_org"])
    unf = np.ascontiguousarray(g[f"n{n}_unf"])
    out = np.zeros((len(org), 35), np.uint32)
    assert emul.emul_rmd_batch(bd, 1, int(np.log2(n)), len(org), P(org, i16p), P(unf, i16p), P(out, u32p)) == 0
    assert np.array_equal(out, g[f"n{n}_sad"])


@pytest.mark.parametrize("bd,W,H", [(8, 200, 136), (10, 136, 72)])
def test_frame_kernel_code_vs_oracle(emul, oracle, bd, W, H):
    org = textured_plane(W, H, bd, seed=5)
    rec = pseudo_recon(org, bd)
    rec[:, : W // 2] = (np.arange(H)[:, None] // 3 + np.arange(W // 2)[None, :] // 5 + 40).astype(np.int16)  # flat: strong smoothing
    want = oracle_rmd_frame(oracle, org, rec, bd)
    S = (W + 7) // 8 * 8
    orgp = np.zeros((H, S), np.int16)
    orgp[:, :W] = org
    got = np.zeros_like(want)
    emul.emul_rmd_frame(bd, 1, P(orgp, i16p), S, P(rec, i16p), W, W, H, 0, want.shape[0], P(got, u32p))
    assert np.array_equal(got, want)


@pytest.mark.parametrize("W,H,seed", [(200, 136, 5), (64, 64, 1), (328, 72, 9)])
def test_tensor_core_frame_kernel_code_vs_oracle(emul, oracle, W, H, seed):
    """rmd_tc2: prediction and Hadamard as exact integer matmuls through the kernel's own weight tables,
    window gather, row map and byte packing (tests/emul/rmd_tc2_emul.cpp)"""
    org = textured_plane(W, H, 8, seed=seed)
    rec = pseudo_recon(org, 8)
    rec[:, : W // 2] = (np.arange(H)[:, None] // 3 + np.arange(W // 2)[None, :] // 5 + 40).astype(np.int16)
    want = oracle_rmd_frame(oracle, org, rec, 8)
    got = np.zeros_like(want)
    emul.emul_rmd_frame_tc2(1, P(org, i16p), W, P(rec, i16p), W, W, H, P(got, u32p), None)
    assert np.array_equal(got, want)


@pytest.mark.parametrize("bd,W,H,seed", [(10, 200, 136, 5), (10, 64, 64, 1), (9, 328, 72, 9), (8, 136, 72, 2)])
def test_half_precision_tensor_core_frame_kernel_code_vs_oracle(emul, oracle, bd, W, H, seed):
    """rmd_tc3 (9/10-bit content on tcgen05 kind::f16): the kernel's fp16 weight tables, record / window operands, magic-number
    accumulator read-out and FADD |x| epilogue, replayed with exact products (tests/emul/rmd_tc3_emul.cpp)"""
    org = textured_plane(W, H, bd, seed=seed)
    rec = pseudo_recon(org, bd)
    rec[:, : W // 2] = ((np.arange(H)[:, None] // 3 + np.arange(W // 2)[None, :] // 5 + 40) << (bd - 8)).astype(np.int16)   # flat: strong smoothing
    want = oracle_rmd_frame(oracle, org, rec, bd)
    S = (W + 7) // 8 * 8
    orgp = np.zeros((H, S), np.int16); orgp[:, :W] = org
    recp = np.zeros((H, S), np.int16); recp[:, :W] = rec
    got = np.zeros_like(want)
    emul.emul_rmd_frame_tc3(bd, 1, P(orgp, i16p), S, P(recp, i16p), S, W, H, P(got, u32p), None)
    assert np.array_equal(got, want)


def test_half_precision_tensor_core_frame_kernel_code_extreme_values(emul, oracle):
    """0 / 1023 checkerboards and stripes: the largest accumulators (2^23 + 65535) and Hadamard sums the fp32 path sees"""
    W = H = 64
    yy, xx = np.mgrid[0:H, 0:W]
    rng = np.random.default_rng(3)
    cases = [(np.where((xx + yy) & 1, 1023, 0), np.where((xx + yy) & 1, 0, 1023)), (np.full((H, W), 1023), np.zeros((H, W))),
             (np.where(xx & 1, 1023, 0), np.full((H, W), 1023)), (rng.integers(0, 1024, (H, W)), rng.integers(0, 1024, (H, W)))]
    for org, rec in cases:
        org = np.ascontiguousarray(org.astype(np.int16)); rec = np.ascontiguousarray(rec.astype(np.int16))
        want = oracle_rmd_frame(oracle, org, rec, 10)
        got = np.zeros_like(want)
        emul.emul_rmd_frame_tc3(10, 1, P(org, i16p), W, P(rec, i16p), W, W, H, P(got, u32p), None)
        assert np.array_equal(got, want)


@pytest.mark.parametrize("bd,W,H", [(8, 200, 136), (10, 136, 72)])
def test_tensor_core_frame_kernel_code_fork_aware_mask(emul, oracle, bd, W, H):
    """fork-aware mode of rmd_tc2 / rmd_tc3: a random `needed` mask, every 32x32 PU pruned (each of those CTAs takes the early exit);
    the table is the oracle's with CUCD_COST_PRUNED for a pruned PU and CUCD_COST_NOT_INSIDE outside the picture"""
    org = textured_plane(W, H, bd, seed=6)
    rec = pseudo_recon(org, bd)
    full = oracle_rmd_frame(oracle, org, rec, bd)
    need = (np.random.default_rng(bd).random(full.shape[:2]) < 0.5).astype(np.uint8)
    need[:, 1:5] = 0
    need[:, 85:] = np.repeat(need[:, 85::4], 4, axis=1)               # 4x4 PUs: NxN of an 8x8 CU is pruned as a whole
    inside = full[:, :, 0] != 0xFFFFFFFF
    want = np.where(((need == 0) & inside)[:, :, None], np.uint32(0xFFFFFFFE), full)
    got = np.zeros_like(full)
    if bd == 8:
        emul.emul_rmd_frame_tc2(1, P(org, i16p), W, P(rec, i16p), W, W, H, P(got, u32p), P(need, u8p))
    else:
        emul.emul_rmd_frame_tc3(bd, 1, P(org, i16p), W, P(rec, i16p), W, W, H, P(got, u32p), P(need, u8p))
    assert (~inside).any() and (inside & (need == 0)).any() and (inside & (need == 1)).any()
    assert np.array_equal(got, want)


@pytest.mark.parametrize("n", [4, 8, 16, 32, 64])
def test_tensor_core_batch_kernel_code_vs_golden(emul, n):
    """S2 batches on the tensor-core code path against the vectors dumped from the reference encoder's own RMD loop"""
    g = golden("rmd_ai8.npz")
    org = np.ascontiguousarray(g[f"n{n}_org"])
    unf = np.ascontiguousarray(g[f"n{n}_unf"])
    out = np.zeros((len(org), 35), np.uint32)
    assert emul.emul_rmd_batch_tc2(1, int(np.log2(n)), len(org), P(org, i16p), P(unf, i16p), P(out, u32p)) == 0
    assert np.array_equal(out, g[f"n{n}_sad"])


def test_tensor_core_frame_kernel_code_extreme_values(emul, oracle):
    """the byte-1 extraction must be exact at 0 / 255 and for alternating content"""
    W = H = 64
    yy, xx = np.mgrid[0:H, 0:W]
    rng = np.random.default_rng(3)
    cases = [(np.where((xx + yy) & 1, 255, 0), np.where((xx + yy) & 1, 0, 255)), (np.full((H, W), 255), np.zeros((H, W))),
             (np.where(xx & 1, 255, 0), np.full((H, W), 255)), (rng.integers(0, 256, (H, W)), rng.integers(0, 256, (H, W)))]
    for org, rec in cases:
        org = np.ascontiguousarray(org.astype(np.int16)); rec = np.ascontiguousarray(rec.astype(np.int16))
        want = oracle_rmd_frame(oracle, org, rec, 8)
        got = np.zeros_like(want)
        emul.emul_rmd_frame_tc2(1, P(org, i16p), W, P(rec, i16p), W, W, H, P(got, u32p), None)
        assert np.array_equal(got, want)


@pytest.mark.parametrize("bd", [8, 10])
def test_extreme_values_do_not_overflow_packed_lanes(emul, oracle, bd):
    """worst case for the 16-bit packed butterflies: full-scale checkerboards against 0 / max borders"""
    hi = (1 << bd) - 1
    for n in (4, 8, 16, 32, 64):
        yy, xx = np.mgrid[0:n, 0:n]
        pats = [np.where((xx + yy) & 1, hi, 0), np.where(xx & 1, hi, 0), np.full((n, n), hi), np.where((xx // 4 + yy // 4) & 1, hi, 0)]
        borders = [np.zeros(4 * n + 1), np.full(4 * n + 1, hi), np.where(np.arange(4 * n + 1) & 1, hi, 0)]
        org = np.concatenate([p.ravel() for p in pats for _ in borders]).astype(np.int16)
        brd = np.concatenate([b for _ in pats for b in borders]).astype(np.int16)
        cnt = len(pats) * len(borders)
        got = np.zeros((cnt, 35), np.uint32)
        emul.emul_rmd_batch(bd, 1, int(np.log2(n)), cnt, P(org, i16p), P(brd, i16p), P(got, u32p))
        for k in range(cnt):
            want = np.zeros(35, np.uint32)
            o = np.ascontiguousarray(org[k * n * n:(k + 1) * n * n])
            b = np.ascontiguousarray(brd[k * (4 * n + 1):(k + 1) * (4 * n + 1)])
            oracle.oracle_rmd_pu(bd, n, 1, P(o, i16p), n, P(b, i16p), P(want, u32p))
            assert np.array_equal(got[k], want), (n, k)


@pytest.mark.parametrize("clip", ["ai8", "ai10"])
def test_feature_kernel_code_vs_golden(emul, cucd, clip):
    """DCT + histogram (pass 1) -> host TCM fit of the library -> threshold/OBF/Outlier (pass 2)"""
    g = golden(f"obf_{clip}.npz")
    _, W, H, bd = [int(v) for v in g["f0_meta"]]
    org = np.ascontiguousarray(g["f0_org"])
    hist = np.zeros(16 * 4096, np.uint32)
    emul.emul_feature_hist(bd, P(org, i16p), W, W, H, P(hist, u32p))
    yc, thr = cucd.tcm_fit(hist, (W // 4) * (H // 4))
    assert np.array_equal(yc[1:], g["f0_yc"][1:])
    obf = np.zeros((H // 4, W // 4), np.int16)
    outl = np.zeros((H, W), np.int16)
    emul.emul_feature_obf(bd, P(org, i16p), W, W, H, P(thr, i32p), P(obf, i16p), P(outl, i16p))
    assert np.array_equal(obf, g["f0_obf"])
    assert np.array_equal(outl, g["f0_outlier"])


def test_fork_aware_enumeration_kernel_code_vs_oracle_walk(emul, oracle):
    """prune_mask_ctu (the kernel's iterative walk over per-depth Num_OBF grids) == the oracle's recursive restatement of
    TEncCu::xCompressCU on the OBF plane, for every switch combination, on pictures with partial CTUs (1080p-like 56-row edge)"""
    import ctypes as C
    import itertools
    from _util import oracle_cu_sums
    rng = np.random.default_rng(12)
    for W, H in ((200, 136), (256, 120), (64, 64)):
        obf = (rng.integers(0, 16, (H // 4, W // 4)) * (rng.random((H // 4, W // 4)) < 0.08)).astype(np.int16)
        obf[: H // 8] = 0                                             # a flat band: Num_OBF == 0 up to depth 0
        grids = [oracle_cu_sums(oracle, obf, W, H, d)[0] for d in range(4)]
        nctu = ((W + 63) // 64) * ((H + 63) // 64)
        for bits in itertools.product((0, 1), repeat=4):
            for skip, term in ((bits, (0, 0, 0, 0)), ((0, 0, 0, 0), bits), (bits, bits[::-1]), ((1, 1, 1, 1), bits)):
                a = (C.c_uint8 * 4)(*skip); b = (C.c_uint8 * 4)(*term)
                want = np.zeros((nctu, 341), np.uint8); got = np.full((nctu, 341), 7, np.uint8)
                oracle.oracle_prune_mask(obf.ctypes.data_as(C.c_void_p), W, H, a, b, want.ctypes.data_as(C.c_void_p))
                emul.emul_prune_mask(W, H, *[g.ctypes.data_as(C.c_void_p) for g in grids], a, b, got.ctypes.data_as(C.c_void_p))
                assert np.array_equal(got, want), (W, H, skip, term)
        # no switch on: the full enumeration of everything inside the picture
        a = (C.c_uint8 * 4)(0, 0, 0, 0)
        full = np.zeros((nctu, 341), np.uint8)
        oracle.oracle_prune_mask(obf.ctypes.data_as(C.c_void_p), W, H, a, a, full.ctypes.data_as(C.c_void_p))
        assert full.sum() > 0 and (W % 64 or H % 64 or full.all())


# ---- integer-ME SAD: the dy-lane kernel's tiling, staging and sliding SAD (csrc/me_core.cuh) ---------------------------------
def _emul_me_surface(emul, oracle, bd, cur, refp, M, x, y, w, h, left, right, top, bottom, sub):
    import ctypes as C
    S = refp.shape[1]
    cols, rows = right - left + 1, bottom - top + 1
    o = np.ascontiguousarray(cur[y:y + h, x:x + w])
    base = refp.ctypes.data + 2 * ((y + M) * S + x + M)
    want = np.zeros((rows, cols), np.uint32)
    oracle.oracle_sad_surface(bd, P(o, i16p), w, w, h, C.c_void_p(base), S, left, right, top, bottom, sub, P(want, u32p))
    got = np.full((rows, cols), 0xdeadbeef, np.uint32); hits = np.zeros((rows, cols), np.uint8); counts = (C.c_int * 3)()
    win = refp.ctypes.data + 2 * ((y + M + top) * S + x + M + left)
    emul.emul_me_sad_surface(bd, P(o, i16p), w, w, h, C.c_void_p(win), S, cols, rows, sub, P(got, u32p), hits.ctypes.data_as(C.c_void_p), counts)
    assert (hits == 1).all(), "every candidate is written by exactly one tile"
    dy_lane = got != 0xffffffff                                     # candidates of the O tiles carry the sentinel
    assert np.array_equal(got[dy_lane], want[dy_lane]), (bd, w, h, cols, rows, sub)
    return list(counts), int(dy_lane.sum())


@pytest.mark.parametrize("bd", [8, 9, 10])
def test_me_dy_lane_kernel_code_vs_oracle(emul, oracle, bd):
    """TComRdCost::xGetSAD* (TComRdCost.cpp:465-962) over whole windows: every PU width HM has (AMP 12 / 24 / 48 included), the +-64
    window of TEncSearch::xSetSearchRange, windows whose width / height leave every kind of strip, row sub-sampling 0 / 1 / 2"""
    W, H, M = 192, 128, 80
    cur = textured_plane(W, H, bd, seed=31, t=1)
    refp = np.pad(pseudo_recon(textured_plane(W, H, bd, seed=31, t=0), bd), M, mode="edge")
    cases = [(64, 64, 64, 64, -64, 64, -64, 64, 1),       # the production window: 8 M + 2 E + 4 O tiles
             (0, 0, 16, 16, -72, 8, -72, 8, 1), (176, 112, 16, 16, -5, 72, -3, 72, 0), (32, 16, 12, 16, -40, 9, -30, 40, 1),
             (40, 24, 24, 32, -33, 0, 0, 31, 1), (8, 8, 8, 4, -20, 20, -20, 20, 0), (8, 8, 4, 8, -16, 17, -16, 50, 0),
             (64, 32, 48, 64, -16, 19, -40, 30, 1), (64, 32, 64, 16, -40, -5, -2, 61, 1), (96, 64, 32, 32, -64, 64, -64, 63, 2),
             (16, 16, 8, 8, -16, 15, -16, 15, 0), (100, 60, 4, 4, -32, 34, -32, 31, 0), (64, 64, 64, 64, 0, 71, 0, 32, 0),
             (16, 8, 32, 8, -3, 3, -3, 3, 0), (48, 48, 16, 32, -8, 8, -64, 64, 1)]
    total_dy = 0
    for x, y, w, h, l, r, t, b, sub in cases:
        counts, n = _emul_me_surface(emul, oracle, bd, cur, refp, M, x, y, w, h, l, r, t, b, sub)
        total_dy += n
        if (r - l + 1, b - t + 1) == (129, 129):
            assert counts == [4, 8, 2]
        if r - l + 1 < 32 or b - t + 1 < 32:
            assert counts[1] == 0 and counts[2] == 0
    assert total_dy > 50000


@pytest.mark.parametrize("bd", [8, 9, 10])
def test_me_dy_lane_kernel_code_extreme_values(emul, oracle, bd):
    """source at one end of the sample range, reference at the other (and mixed): the packed 16-bit partial sums of the 9/10-bit path
    must be folded before they overflow, for the widest PU and the smallest"""
    W, H, M = 128, 128, 72
    top = (1 << bd) - 1
    rng = np.random.default_rng(5)
    for pattern in range(3):
        cur = np.full((H, W), top if pattern != 1 else 0, np.int16)
        ref = np.full((H, W), 0 if pattern != 1 else top, np.int16)
        if pattern == 2:
            ref = (rng.integers(0, 2, (H, W)) * top).astype(np.int16)
        refp = np.pad(ref, M, mode="edge")
        for x, y, w, h, sub in ((32, 32, 64, 64, 0), (32, 32, 64, 64, 1), (40, 40, 4, 4, 0), (32, 48, 48, 16, 0), (64, 64, 8, 64, 0)):
            _emul_me_surface(emul, oracle, bd, cur, refp, M, x, y, w, h, -32, 32, -40, 31, sub)


@pytest.mark.parametrize("bd", [8, 9, 10])
def test_subpel_small_pu_kernel_code_vs_oracle(emul, oracle, bd):
    """me_subpel_small_kernel (one CTA per PU, all 49 quarter-pel positions; csrc/me_core.cuh) against the oracle's restatement of
    xPatternSearchFracDIF (TEncSearch.cpp:4340-4376): every PU shape with w * h <= 256 HM has, Hadamard and SAD, textured and
    extreme content"""
    import ctypes as C
    W, H, M = 96, 96, 16
    top = (1 << bd) - 1
    rng = np.random.default_rng(8)
    shapes = [(8, 8), (4, 8), (8, 4), (16, 16), (16, 8), (8, 16), (16, 4), (4, 16), (12, 16), (16, 12), (32, 8), (8, 32), (4, 4)]
    n_small = 0
    for content in range(3):
        if content == 0:
            cur = textured_plane(W, H, bd, seed=41, t=1); ref = pseudo_recon(textured_plane(W, H, bd, seed=41, t=0), bd)
        elif content == 1:
            cur = np.full((H, W), top, np.int16); ref = ((np.indices((H, W)).sum(0) & 1) * top).astype(np.int16)
        else:
            cur = (rng.integers(0, 2, (H, W)) * top).astype(np.int16); ref = (rng.integers(0, 2, (H, W)) * top).astype(np.int16)
        refp = np.pad(ref, M, mode="edge")
        S = W + 2 * M
        for k, (w, h) in enumerate(shapes):
            x, y = 8 + 4 * (k % 5), 12 + 4 * (k % 3)
            mvx, mvy = (-3 + k) % 7 - 3, (2 * k) % 5 - 2
            for had in (1, 0):
                blk = np.ascontiguousarray(cur[y:y + h, x:x + w])
                zero = C.c_void_p(refp.ctypes.data + 2 * ((y + M) * S + x + M))
                want = np.zeros(49, np.uint32); got = np.full(49, 0xdeadbeef, np.uint32)
                oracle.oracle_subpel_surface(bd, P(blk, i16p), w, w, h, zero, S, mvx, mvy, had, P(want, u32p))
                at_mv = C.c_void_p(refp.ctypes.data + 2 * ((y + M + mvy) * S + x + M + mvx))
                n_small += emul.emul_subpel_small(bd, P(blk, i16p), w, w, h, at_mv, S, had, P(got, u32p))
                assert np.array_equal(got, want), (bd, content, w, h, had)
    assert n_small == 3 * len(shapes) * 2
