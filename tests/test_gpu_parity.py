"""Parity of the CUDA path, called through the C ABI (libcucudecide.so), against the golden vectors of
the real reference encoder and against the oracle on seeded inputs.  Everything is integer work:
the bar is bit-exact."""
import numpy as np
import pytest

from _util import (P, golden, i16p, u32p, oracle_ctu_src_had, oracle_cu_sums, oracle_outlier_frame, oracle_rmd_frame,
                   pseudo_recon, textured_plane)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng8(cucd):
    e = cucd.Engine(416, 240, bit_depth=8, max_pictures=3)
    yield e
    e.close()


@pytest.fixture(scope="module")
def eng10(cucd):
    e = cucd.Engine(416, 240, bit_depth=10, max_pictures=2)
    yield e
    e.close()


# ---- S2: batched RMD with caller-supplied borders vs the encoder's own uiSad[35] --------------------
@pytest.mark.parametrize("clip", ["ai8", "ai10"])
def test_rmd_batch_vs_reference_encoder_dump(eng8, eng10, clip):
    g = golden(f"rmd_{clip}.npz")
    eng = eng8 if clip == "ai8" else eng10
    sizes, orgs, brds, want = [], [], [], []
    for n in (4, 8, 16, 32, 64):
        k = len(g[f"n{n}_org"])
        sizes += [int(np.log2(n))] * k
        orgs.append(g[f"n{n}_org"].ravel()); brds.append(g[f"n{n}_unf"].ravel()); want.append(g[f"n{n}_sad"])
    # interleave the sizes so that the library's size bucketing and output scatter are exercised
    order = np.random.default_rng(3).permutation(len(sizes))
    sizes = np.array(sizes)
    org_list, brd_list, o_off, b_off = [], [], 0, 0
    flat_org, flat_brd = np.concatenate(orgs), np.concatenate(brds)
    offs_o, offs_b = [], []
    for s in sizes:
        n = 1 << s
        offs_o.append(o_off); offs_b.append(b_off)
        o_off += n * n; b_off += 4 * n + 1
    for i in order:
        n = 1 << sizes[i]
        org_list.append(flat_org[offs_o[i]: offs_o[i] + n * n]); brd_list.append(flat_brd[offs_b[i]: offs_b[i] + 4 * n + 1])
    got = eng.intra_rmd_batch(sizes[order], np.concatenate(org_list), np.concatenate(brd_list))
    assert np.array_equal(got, np.concatenate(want)[order])


def test_rmd_batch_edge_cases(eng8, oracle):
    assert eng8.intra_rmd_batch([], np.zeros(0, np.int16), np.zeros(0, np.int16)).shape == (0, 35)
    rng = np.random.default_rng(11)
    for n, cnt in ((4, 1), (4, 5), (4, 257), (8, 65), (16, 17), (32, 5), (64, 3)):   # ragged: not a multiple of a chunk
        org = rng.integers(0, 256, (cnt, n * n)).astype(np.int16)
        brd = rng.integers(0, 256, (cnt, 4 * n + 1)).astype(np.int16)
        got = eng8.intra_rmd_batch([int(np.log2(n))] * cnt, org, brd)
        for k in range(cnt):
            want = np.zeros(35, np.uint32)
            oracle.oracle_rmd_pu(8, n, 1, P(org[k], i16p), n, P(brd[k], i16p), P(want, u32p))
            assert np.array_equal(got[k], want), (n, k)


@pytest.mark.parametrize("bd", [8, 9, 10])
def test_rmd_batch_extreme_values(cucd, oracle, bd):
    hi = (1 << bd) - 1
    with cucd.Engine(64, 64, bit_depth=bd) as eng:
        for n in (4, 8, 16, 32, 64):
            yy, xx = np.mgrid[0:n, 0:n]
            pats = [np.where((xx + yy) & 1, hi, 0), np.where(xx & 1, hi, 0), np.full((n, n), hi), np.zeros((n, n))]
            borders = [np.zeros(4 * n + 1), np.full(4 * n + 1, hi), np.where(np.arange(4 * n + 1) & 1, hi, 0)]
            org = np.stack([p.ravel() for p in pats for _ in borders]).astype(np.int16)
            brd = np.stack([b for _ in pats for b in borders]).astype(np.int16)
            got = eng.intra_rmd_batch([int(np.log2(n))] * len(org), org, brd)
            for k in range(len(org)):
                want = np.zeros(35, np.uint32)
                oracle.oracle_rmd_pu(bd, n, 1, P(org[k], i16p), n, P(brd[k], i16p), P(want, u32p))
                assert np.array_equal(got[k], want), (n, k)


# ---- S1/S4 + replay S2 through cuCUDecide_frame(s) ----------------------------------------------------
@pytest.mark.parametrize("clip", ["ai8", "ai10"])
def test_frame_features_vs_reference_encoder_dump(eng8, eng10, oracle, clip):
    g = golden(f"obf_{clip}.npz")
    eng = eng8 if clip == "ai8" else eng10
    nf = int(g["nframes"][0])
    orgs = [np.ascontiguousarray(g[f"f{k}_org"]) for k in range(nf)]
    outs = eng.frames(orgs)                    # no reconstruction plane: features only
    for k in range(nf):
        _, W, H, bd = [int(v) for v in g[f"f{k}_meta"]]
        o = outs[k]
        assert np.array_equal(o["yc"][1:], g[f"f{k}_yc"][1:])
        assert np.array_equal(o["obf"], g[f"f{k}_obf"])
        assert np.array_equal(o["outlier"], g[f"f{k}_outlier"])
        cu = g[f"f{k}_cu"]
        for depth in range(4):
            sel = cu[cu[:, 0] == depth]
            s = 64 >> depth
            assert np.array_equal(o[f"num_obf{depth}"][sel[:, 2] // s, sel[:, 1] // s], sel[:, 4])
            assert np.array_equal(o[f"n_outlier{depth}"][sel[:, 2] // s, sel[:, 1] // s], sel[:, 5])
        assert np.array_equal(o["ctu_src_had"], oracle_ctu_src_had(oracle, orgs[k]))


@pytest.mark.parametrize("bd,W,H", [(8, 416, 240), (10, 200, 136), (8, 64, 64), (8, 8, 72), (10, 72, 136)])
def test_frame_replay_vs_oracle(cucd, oracle, bd, W, H):
    """full enumeration (341 PUs x 35 modes per CTU), partial CTUs on the right and bottom edges.
    (The one-CU-wide case used to be 8x8: on some tiny pictures the reference's lambda iteration of the TCM fit,
    TEncSlice.cpp:221-226, needs minutes to converge - oracle and product reproduce that faithfully, the suite avoids it.)"""
    org = textured_plane(W, H, bd, seed=W + H)
    rec = pseudo_recon(org, bd)
    if W >= 128:
        rec[:, : W // 2] = ((np.arange(H)[:, None] // 3 + np.arange(W // 2)[None, :] // 5 + 40) << (bd - 8)).astype(np.int16)
    with cucd.Engine(W, H, bit_depth=bd) as eng:
        out = eng.frame(org, rec)
    want = oracle_rmd_frame(oracle, org, rec, bd)
    assert np.array_equal(out["rmd_cost"], want)
    obf, outl, yc = oracle_outlier_frame(oracle, org, bd)
    assert np.array_equal(out["yc"][1:], yc[1:])
    assert np.array_equal(out["obf"], obf)
    assert np.array_equal(out["outlier"], outl)
    for d in range(4):
        a, b = oracle_cu_sums(oracle, obf, W, H, d)
        assert np.array_equal(out[f"num_obf{d}"], a) and np.array_equal(out[f"n_outlier{d}"], b)
    assert np.array_equal(out["ctu_src_had"], oracle_ctu_src_had(oracle, org))


def test_frames_batch_equals_single_pictures(cucd):
    """a batch of pictures (also larger than max_pictures -> grouped) gives what one picture at a time gives"""
    W, H = 200, 136
    orgs = [textured_plane(W, H, 8, seed=9, t=t) for t in range(5)]
    recs = [pseudo_recon(o, 8, seed=t) for t, o in enumerate(orgs)]
    with cucd.Engine(W, H, max_pictures=2) as eng:
        batch = eng.frames(orgs, recs)
        for t in range(5):
            one = eng.frame(orgs[t], recs[t], poc=t)
            for k in one:
                assert np.array_equal(one[k], batch[t][k]), (t, k)


def test_strong_smoothing_flag_is_honoured(cucd, oracle):
    W, H = 128, 128
    org = textured_plane(W, H, 8, seed=2)
    rec = np.full((H, W), 100, np.int16) + (np.arange(W)[None, :] // 9).astype(np.int16)
    for strong in (0, 1):
        with cucd.Engine(W, H, strong_intra_smoothing=strong) as eng:
            got = eng.frame(org, rec)["rmd_cost"]
        assert np.array_equal(got, oracle_rmd_frame(oracle, org, rec, 8, strong=strong))


def test_strided_host_planes(cucd, oracle):
    """HM hands over planes with stride W+160 and an 80-sample margin (TComPicYuv.cpp:83-101)"""
    W, H = 136, 72
    org = textured_plane(W, H, 8, seed=4)
    rec = pseudo_recon(org, 8)
    big_o = np.zeros((H + 160, W + 160), np.int16); big_o[80:80 + H, 80:80 + W] = org
    big_r = np.zeros((H + 160, W + 160), np.int16); big_r[80:80 + H, 80:80 + W] = rec
    with cucd.Engine(W, H) as eng:
        out = eng.frame(big_o[80:80 + H, 80:80 + W], big_r[80:80 + H, 80:80 + W])
    assert np.array_equal(out["rmd_cost"], oracle_rmd_frame(oracle, org, rec, 8))


def test_invalid_arguments_are_rejected(cucd):
    with pytest.raises(cucd.CucdError):
        cucd.Engine(100, 64)              # not a multiple of 8
    with pytest.raises(cucd.CucdError):
        cucd.Engine(64, 64, bit_depth=12)  # packed 16-bit butterflies are valid up to 10 bit
    with cucd.Engine(64, 64) as eng:
        with pytest.raises(cucd.CucdError):
            eng.intra_rmd_batch([7], np.zeros(128 * 128, np.int16), np.zeros(513, np.int16))


# ---- S3: integer-ME SAD ---------------------------------------------------------------------------------
def test_me_probes_vs_reference_encoder_dump(cucd):
    """every sampled xTZSearchHelp probe: place PU and reference block into planes, ask for the 1x1 window"""
    g = golden("me_ldp8.npz")
    hdr, org, ref = g["hdr"], g["org"], g["ref"]
    W = H = 128
    with cucd.Engine(W, H) as eng:
        off = 0
        for cols, rows, sub, bd, _, _, sad in hdr[:120]:
            cols, rows = int(cols), int(rows)
            cur = np.zeros((H, W), np.int16); refp = np.zeros((H + 16, W + 16), np.int16)
            cur[8:8 + rows, 16:16 + cols] = org[off: off + cols * rows].reshape(rows, cols)
            refp[8 + 8 + 3:8 + 8 + 3 + rows, 8 + 16 - 2:8 + 16 - 2 + cols] = ref[off: off + cols * rows].reshape(rows, cols)
            off += cols * rows
            eng.set_cur_picture(cur)
            eng.set_ref_picture(0, refp, 8, 8)
            s = eng.me_sad_surface([dict(x=16, y=8, w=cols, h=rows, ref_idx=0, left=-2, right=-2, top=3, bottom=3, sub_shift=int(sub))])[0]
            assert s.shape == (1, 1) and int(s[0, 0]) == int(sad), (cols, rows, sub)


@pytest.mark.parametrize("bd", [8, 9, 10])
def test_me_surfaces_vs_oracle(cucd, oracle, bd):
    W, H, M = 192, 128, 80
    cur = textured_plane(W, H, bd, seed=21, t=1)
    ref = pseudo_recon(textured_plane(W, H, bd, seed=21, t=0), bd)
    refp = np.pad(ref, M, mode="edge")
    descs = [dict(x=64, y=64, w=64, h=64, ref_idx=1, left=-64, right=64, top=-64, bottom=64, sub_shift=1),
             dict(x=0, y=0, w=16, h=16, ref_idx=1, left=-72, right=8, top=-72, bottom=8, sub_shift=1),
             dict(x=176, y=112, w=16, h=16, ref_idx=1, left=-5, right=72, top=-3, bottom=72, sub_shift=1),
             dict(x=32, y=16, w=12, h=16, ref_idx=1, left=-7, right=9, top=-4, bottom=4, sub_shift=1),
             dict(x=40, y=24, w=24, h=32, ref_idx=1, left=-33, right=0, top=0, bottom=9, sub_shift=1),
             dict(x=8, y=8, w=8, h=4, ref_idx=1, left=-3, right=3, top=-3, bottom=3, sub_shift=0),
             dict(x=8, y=8, w=4, h=8, ref_idx=1, left=0, right=0, top=0, bottom=0, sub_shift=0),
             dict(x=64, y=32, w=48, h=64, ref_idx=1, left=-16, right=15, top=-8, bottom=7, sub_shift=1),
             dict(x=64, y=32, w=64, h=16, ref_idx=1, left=-40, right=-9, top=-2, bottom=2, sub_shift=1),
             dict(x=96, y=64, w=32, h=32, ref_idx=1, left=-64, right=64, top=-64, bottom=63, sub_shift=2)]
    with cucd.Engine(W, H, bit_depth=bd) as eng:
        eng.set_cur_picture(cur)
        eng.set_ref_picture(1, refp, M, M)
        got = eng.me_sad_surface(descs)
    S = W + 2 * M
    for d, g_ in zip(descs, got):
        want = np.zeros_like(g_)
        o = np.ascontiguousarray(cur[d["y"]:d["y"] + d["h"], d["x"]:d["x"] + d["w"]])
        base = refp.ctypes.data + 2 * ((d["y"] + M) * S + d["x"] + M)
        import ctypes as C
        oracle.oracle_sad_surface(bd, P(o, i16p), d["w"], d["w"], d["h"], C.c_void_p(base), S, d["left"], d["right"], d["top"], d["bottom"],
                                  d["sub_shift"], P(want, u32p))
        assert np.array_equal(g_, want), d
    # zero motion on identical planes is zero; window leaving the padded plane is refused
    with cucd.Engine(W, H, bit_depth=bd) as eng:
        eng.set_cur_picture(cur)
        eng.set_ref_picture(0, np.pad(cur, M, mode="edge"), M, M)
        assert int(eng.me_sad_surface([dict(x=64, y=64, w=32, h=32, ref_idx=0, left=0, right=0, top=0, bottom=0, sub_shift=1)])[0][0, 0]) == 0
        with pytest.raises(cucd.CucdError):
            eng.me_sad_surface([dict(x=0, y=0, w=16, h=16, ref_idx=0, left=-81, right=0, top=0, bottom=0, sub_shift=0)])


# ---- the two frame-RMD implementations (integer ALU, tcgen05 prediction + Hadamard) must agree bit for bit -------
@pytest.mark.parametrize("W,H", [(416, 240), (200, 136), (64, 64), (328, 72)])
def test_tensor_core_path_equals_alu_path_and_oracle(cucd, oracle, W, H):
    org = textured_plane(W, H, 8, seed=W)
    rec = pseudo_recon(org, 8)
    rec[:, : W // 2] = (np.arange(H)[:, None] // 3 + np.arange(W // 2)[None, :] // 5 + 40).astype(np.int16)
    with cucd.Engine(W, H, max_pictures=3) as eng:
        eng.set_rmd_path(1)
        tc = eng.frames([org, rec, org], [rec, org, org])      # 3 pictures: CTU groups of 4 straddle pictures
        eng.set_rmd_path(0)
        alu = eng.frames([org, rec, org], [rec, org, org])
    want = oracle_rmd_frame(oracle, org, rec, 8)
    assert np.array_equal(tc[0]["rmd_cost"], want)
    assert np.array_equal(alu[0]["rmd_cost"], want)
    for k in range(3):
        assert np.array_equal(tc[k]["rmd_cost"], alu[k]["rmd_cost"])


def test_tensor_core_path_extreme_values(cucd, oracle):
    W = H = 64
    yy, xx = np.mgrid[0:H, 0:W]
    for org, rec in [(np.where((xx + yy) & 1, 255, 0), np.where((xx + yy) & 1, 0, 255)), (np.full((H, W), 255), np.zeros((H, W))),
                     (np.where(xx & 1, 255, 0), np.full((H, W), 255))]:
        org = org.astype(np.int16); rec = rec.astype(np.int16)
        with cucd.Engine(W, H) as eng:
            with pytest.raises(cucd.CucdError):
                eng.set_rmd_path(3)                       # 0 / 1 / 2 are the paths of the ABI
            got = eng.frame(org, rec)["rmd_cost"]
        assert np.array_equal(got, oracle_rmd_frame(oracle, org, rec, 8))


# ---- 9/10-bit content: tcgen05 kind::f16 kernel (exact integers in fp16 operands / fp32 accumulators) == integer ALU == oracle ----
@pytest.mark.parametrize("bd,W,H", [(10, 416, 240), (10, 200, 136), (9, 328, 72), (10, 64, 64), (8, 200, 136)])
def test_half_precision_tensor_core_path_equals_alu_path_and_oracle(cucd, oracle, bd, W, H):
    org = textured_plane(W, H, bd, seed=W + bd)
    rec = pseudo_recon(org, bd)
    rec[:, : W // 2] = ((np.arange(H)[:, None] // 3 + np.arange(W // 2)[None, :] // 5 + 40) << (bd - 8)).astype(np.int16)
    with cucd.Engine(W, H, bit_depth=bd, max_pictures=3) as eng:
        eng.set_rmd_path(2)                                    # the half-precision kernel whatever the bit depth
        tc = eng.frames([org, rec, org], [rec, org, org])      # 3 pictures: CTU groups of 4 straddle pictures
        eng.set_rmd_path(0)
        alu = eng.frames([org, rec, org], [rec, org, org])
        eng.set_rmd_path(1)                                    # the default: kind::f16 above 8 bit, kind::i8 at 8 bit
        dflt = eng.frame(org, rec)
    want = oracle_rmd_frame(oracle, org, rec, bd)
    assert np.array_equal(tc[0]["rmd_cost"], want)
    assert np.array_equal(dflt["rmd_cost"], want)
    for k in range(3):
        assert np.array_equal(tc[k]["rmd_cost"], alu[k]["rmd_cost"])


def test_half_precision_tensor_core_path_extreme_values(cucd, oracle):
    """0 / 1023 checkerboards and stripes: the largest accumulators (2^23 + 65535) and Hadamard sums; random full-range content"""
    W = H = 64
    yy, xx = np.mgrid[0:H, 0:W]
    rng = np.random.default_rng(3)
    for org, rec in [(np.where((xx + yy) & 1, 1023, 0), np.where((xx + yy) & 1, 0, 1023)), (np.full((H, W), 1023), np.zeros((H, W))),
                     (np.where(xx & 1, 1023, 0), np.full((H, W), 1023)), (rng.integers(0, 1024, (H, W)), rng.integers(0, 1024, (H, W)))]:
        org = np.ascontiguousarray(org.astype(np.int16)); rec = np.ascontiguousarray(rec.astype(np.int16))
        with cucd.Engine(W, H, bit_depth=10) as eng:
            got = eng.frame(org, rec)["rmd_cost"]
        assert np.array_equal(got, oracle_rmd_frame(oracle, org, rec, 10))


# ---- packed cost tables (cucd_frame_out.rmd_cost_packed) carry the same numbers -------------------------------
@pytest.mark.parametrize("bd,W,H", [(8, 200, 136), (9, 104, 88), (10, 136, 72)])
def test_packed_cost_tables_equal_wide_tables(cucd, oracle, bd, W, H):
    org = textured_plane(W, H, bd, seed=11)
    rec = pseudo_recon(org, bd)
    with cucd.Engine(W, H, bit_depth=bd, max_pictures=2) as eng:
        wide = eng.frames([org, rec], [rec, org])
        outs = [eng.alloc_frame_out(True, packed=True) for _ in range(2)]
        eng.frames([org, rec], [rec, org], outs)
    want = oracle_rmd_frame(oracle, org, rec, bd)
    for k in range(2):
        got = cucd.unpack_costs(outs[k]["rmd_cost_packed"])
        assert np.array_equal(got, wide[k]["rmd_cost"])
    assert np.array_equal(cucd.unpack_costs(outs[0]["rmd_cost_packed"]), want)
    assert (want == 0xFFFFFFFF).any()          # partial CTUs: the 0xFFFF / 0x1FFF markers are exercised
    with cucd.Engine(W, H, bit_depth=bd) as eng:                     # the C helpers a host encoder would use
        assert np.array_equal(eng.unpack_costs_c(outs[0]["rmd_cost_packed"]), want)
        t = np.ascontiguousarray(outs[0]["rmd_cost_packed"][1])
        for pu, mode in [(0, 0), (4, 34), (20, 7), (21, 0), (84, 34), (85, 0), (86, 1), (200, 17), (340, 34)]:
            assert eng.lib.cucd_packed_cost(t.ctypes.data, pu, mode) == int(want[1, pu, mode])


# ---- ABI v4: byte planes in, byte feature planes out, pinned caller buffers, begin / end ------------------------
def test_u8_planes_and_narrow_outputs_equal_the_int16_call(cucd):
    W, H = 200, 136
    org = textured_plane(W, H, 8, seed=21); rec = pseudo_recon(org, 8)
    with cucd.Engine(W, H, max_pictures=2) as eng:
        wide = eng.frames([org, rec], [rec, org])
        outs = [eng.alloc_frame_out(True, packed=True, narrow=True) for _ in range(2)]
        # HM-layout byte planes: stride W + 160, the plane starts 80 samples into its row
        def hm(a):
            buf = np.zeros((H, W + 160), np.uint8); buf[:, 80:80 + W] = a
            return buf[:, 80:80 + W]
        eng.frames([hm(org), hm(rec)], [hm(rec), hm(org)], outs)
        for k in range(2):
            assert np.array_equal(cucd.unpack_costs(outs[k]["rmd_cost_packed"]), wide[k]["rmd_cost"])
            assert np.array_equal(outs[k]["obf_u8"].astype(np.int16), wide[k]["obf"])
            assert np.array_equal(outs[k]["outlier_u8"].astype(np.int16), wide[k]["outlier"])
            assert np.array_equal(outs[k]["num_obf3"], wide[k]["num_obf3"]) and np.array_equal(outs[k]["yc"], wide[k]["yc"])
    with cucd.Engine(W, H, bit_depth=10) as eng10:
        with pytest.raises(cucd.CucdError):
            eng10.frames([org.astype(np.uint8)], [rec.astype(np.uint8)])      # byte planes need an 8-bit handle


def test_outlier_plane_fits_a_byte_at_the_extremes(cucd, oracle):
    """|AC coefficient| / 100 <= 163 (include/cucudecide.h): blocks that maximise single AC coefficients"""
    from test_capi_load import _extreme_outlier_plane
    for bd in (8, 10):
        org = _extreme_outlier_plane(bd, 3)
        obf, outl, _ = oracle_outlier_frame(oracle, org, bd)
        assert 160 <= outl.max() <= 163
        with cucd.Engine(org.shape[1], org.shape[0], bit_depth=bd) as eng:
            out = eng.alloc_frame_out(False, narrow=True)
            eng.frame(org, None, out=out)
        assert np.array_equal(out["outlier_u8"].astype(np.int16), outl) and np.array_equal(out["obf_u8"].astype(np.int16), obf)


def test_pinned_and_auto_pinned_caller_buffers(cucd):
    W, H = 416, 240
    org = textured_plane(W, H, 8, seed=31); rec = pseudo_recon(org, 8)
    with cucd.Engine(W, H) as eng:
        want = eng.frame(org, rec)
    def hm(a):
        buf = np.zeros((H + 160, W + 160), np.int16); buf[80:80 + H, 80:80 + W] = a
        return buf, buf[80:80 + H, 80:80 + W]
    bo, vo = hm(org); br, vr = hm(rec)
    with cucd.Engine(W, H) as eng:
        eng.pin_host_buffer(bo); eng.pin_host_buffer(br)
        eng.pin_host_buffer(bo)                                # pinning twice is fine
        got = eng.frame(vo, vr)
        assert np.array_equal(got["rmd_cost"], want["rmd_cost"]) and np.array_equal(got["obf"], want["obf"])
        eng.unpin_host_buffer(bo)
        with pytest.raises(cucd.CucdError):
            eng.unpin_host_buffer(bo)
        got = eng.frame(vo, vr)                                # pageable again
        assert np.array_equal(got["rmd_cost"], want["rmd_cost"])
    with cucd.Engine(W, H, auto_pin_host=1) as eng:
        for _ in range(2):
            got = eng.frame(vo, vr)
            assert np.array_equal(got["rmd_cost"], want["rmd_cost"]) and np.array_equal(got["outlier"], want["outlier"])
        log2s, o, b = [3] * 4000, np.tile(org[:8, :8].ravel(), 4000), np.tile(rec[0, :33], 4000)      # > 64 KB arrays: registered on first sight
        a1 = eng.intra_rmd_batch(log2s, o, b)
        a2 = eng.intra_rmd_batch(log2s, o, b)
        assert np.array_equal(a1, a2) and (a1 == a1[0]).all()


def test_dev_frames_begin_end_pipelined(cucd):
    import torch
    W, H, P = 200, 136, 2
    dev = torch.device("cuda", 0)
    pitch = (W + 63) // 64 * 64
    batches = []
    with cucd.Engine(W, H, max_pictures=P) as eng:
        for b in range(3):
            orgs = [textured_plane(W, H, 8, seed=40 + 2 * b + p) for p in range(P)]
            recs = [pseudo_recon(o, 8) for o in orgs]
            d_org = torch.zeros((P, H, pitch), dtype=torch.int16, device=dev); d_rec = torch.zeros_like(d_org)
            for p in range(P):
                d_org[p, :, :W] = torch.from_numpy(orgs[p]).to(dev); d_rec[p, :, :W] = torch.from_numpy(recs[p]).to(dev)
            d_cost = torch.zeros((P, eng.ctus_per_pic, 341, 35), dtype=torch.int32, device=dev)
            d_obf = torch.zeros((P, H // 4, W // 4), dtype=torch.int16, device=dev)
            d_outl = torch.zeros((P, H, W), dtype=torch.int16, device=dev)
            yc = np.zeros((P, 16))
            batches.append((orgs, recs, d_org, d_rec, d_cost, d_obf, d_outl, yc))
        st = torch.cuda.current_stream().cuda_stream
        def begin(b):
            _, _, d_org, d_rec, d_cost, d_obf, d_outl, yc = batches[b]
            eng.dev_frames(st, P, d_org.data_ptr(), H * pitch, pitch, d_rec.data_ptr(), H * pitch, pitch,
                           {"obf": d_obf.data_ptr(), "outlier": d_outl.data_ptr(), "rmd_cost": d_cost.data_ptr()}, yc_host=yc, begin_only=True)
        begin(0); begin(1)
        with pytest.raises(cucd.CucdError):
            begin(2)                                          # at most two batches in flight
        eng.dev_frames_end(); begin(2); eng.dev_frames_end(); eng.dev_frames_end()
        with pytest.raises(cucd.CucdError):
            eng.dev_frames_end()
        torch.cuda.synchronize()
        for orgs, recs, _, _, d_cost, d_obf, d_outl, yc in batches:
            want = eng.frames(orgs, recs)
            for p in range(P):
                assert np.array_equal(d_cost[p].cpu().numpy().view(np.uint32), want[p]["rmd_cost"])
                assert np.array_equal(d_obf[p].cpu().numpy(), want[p]["obf"]) and np.array_equal(d_outl[p].cpu().numpy(), want[p]["outlier"])
                assert np.array_equal(yc[p], want[p]["yc"])


def test_misaligned_device_planes_are_rejected_not_faulted(cucd):
    import torch
    W, H = 128, 64
    dev = torch.device("cuda", 0)
    buf = torch.zeros(4 * H * (W + 64) + 64, dtype=torch.int16, device=dev)
    cost = torch.zeros((2, 341, 35), dtype=torch.int32, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    with cucd.Engine(W, H) as eng:
        base = buf.data_ptr()
        for rec_ptr, rec_stride in [(base + 2, W), (base, W + 4), (base, W - 8)]:          # 2-byte offset, stride not multiple of 8, stride < width
            with pytest.raises(cucd.CucdError):
                eng.dev_rmd_frames(st, 1, base, H * W, W, rec_ptr, H * rec_stride, rec_stride, cost.data_ptr())
        eng.dev_rmd_frames(st, 1, base, H * W, W, base, H * W, W, cost.data_ptr())
        torch.cuda.synchronize()


# ---- S2 batches: the integer-ALU kernels stay bit-exact for 8-bit content too (the default 8-bit path is tcgen05) ----
def test_rmd_batch_alu_path_8bit_vs_reference_encoder_dump(cucd):
    g = golden("rmd_ai8.npz")
    with cucd.Engine(416, 240, bit_depth=8) as eng:
        for path in (0, 1):
            eng.set_rmd_path(path)
            for n in (4, 8, 16, 32, 64):
                got = eng.intra_rmd_batch([int(np.log2(n))] * len(g[f"n{n}_org"]), g[f"n{n}_org"], g[f"n{n}_unf"])
                assert np.array_equal(got, g[f"n{n}_sad"]), (path, n)


# ---- S2 async coalescing queue: several host threads, one batch stream --------------------------------------------
def test_rmd_queue_coalesces_concurrent_requests(cucd, oracle):
    import threading
    rng = np.random.default_rng(5)
    reqs = []
    for t in range(4):
        mine = []
        for k in range(12):
            sizes = rng.integers(2, 7, rng.integers(1, 9))
            org = np.concatenate([rng.integers(0, 256, (1 << s) ** 2) for s in sizes]).astype(np.int16)
            brd = np.concatenate([rng.integers(0, 256, 4 * (1 << s) + 1) for s in sizes]).astype(np.int16)
            mine.append((sizes, org, brd))
        reqs.append(mine)
    results = [[None] * 12 for _ in range(4)]
    with cucd.Engine(64, 64, bit_depth=8) as eng, cucd.RmdQueue(eng) as q:
        def client(t):
            tickets = [q.submit(*r) for r in reqs[t]]          # fire everything, then collect: requests pile up behind the worker
            for k, (ticket, sad) in enumerate(tickets):
                q.wait(ticket)
                results[t][k] = sad
        ths = [threading.Thread(target=client, args=(t,)) for t in range(4)]
        for th in ths:
            th.start()
        for th in ths:
            th.join()
        st = q.stats()
    assert st["requests"] == 48 and st["batches"] <= st["requests"]
    for t in range(4):
        for (sizes, org, brd), got in zip(reqs[t], results[t]):
            oo = bo = 0
            for i, s in enumerate(sizes):
                n = 1 << int(s)
                want = np.zeros(35, np.uint32)
                o = np.ascontiguousarray(org[oo:oo + n * n]); b = np.ascontiguousarray(brd[bo:bo + 4 * n + 1])
                oracle.oracle_rmd_pu(8, n, 1, P(o, i16p), n, P(b, i16p), P(want, u32p))
                assert np.array_equal(got[i], want)
                oo += n * n; bo += 4 * n + 1


# ---- a12 / a13: CU texture features and AQ activity (doubles, bit-exact) ---------------------------
@pytest.mark.parametrize("tag", ["a8", "b10"])
def test_texture_features_vs_reference_golden(cucd, tag):
    g = golden("texture.npz")
    W, H, bd = [int(v) for v in g[f"{tag}_meta"]]
    with cucd.Engine(W, H, bit_depth=bd) as eng:
        eng.set_cur_picture(g[f"{tag}_org"])
        got = eng.tmv_features([tuple(int(v) for v in c) for c in g[f"{tag}_cus"]])
        assert np.array_equal(got, g[f"{tag}_tmv"])
        acts, avg = eng.aq_activity(4)
        for d in range(4):
            assert np.array_equal(acts[d], g[f"{tag}_act{d}"])
        assert np.array_equal(avg, g[f"{tag}_avg"])
        assert eng.tmv_features([]).shape == (0, 5, 26)
        with pytest.raises(cucd.CucdError):
            eng.tmv_features([(4, 0, 3)])            # not aligned to the CU size
        with pytest.raises(cucd.CucdError):
            eng.aq_activity(5)


@pytest.mark.parametrize("bd", [8, 9, 10])
def test_texture_features_vs_oracle_1080p_rows(cucd, oracle, bd):
    from _util import all_cus, oracle_aq_activity, oracle_tmv_features
    W, H = 1920, 1080
    org = textured_plane(W, H, bd, seed=77)
    with cucd.Engine(W, H, bit_depth=bd) as eng:
        eng.set_cur_picture(org)
        cus = all_cus(W, H)
        got = eng.tmv_features(cus)                   # all 43 k whole CUs of the picture in one launch
        sel = np.random.default_rng(1).choice(len(cus), 600, replace=False)
        want = oracle_tmv_features(oracle, org, [cus[i] for i in sel])
        assert np.array_equal(got[sel], want)
        acts, avg = eng.aq_activity(4)
        wacts, wavg = oracle_aq_activity(oracle, org, 4)
        for a, b in zip(acts, wacts):
            assert np.array_equal(a, b)               # includes the clipped 56-row units of the last CTU row
        assert np.array_equal(avg, wavg)


# ---- fork-aware frame mode (cucd_set_decision_switches) ------------------------------------------------------------------
@pytest.mark.parametrize("name", ["a8", "b8"])
def test_fork_aware_frame_mode_vs_real_encoder_visits(cucd, oracle, name):
    """On the Testing pictures of a real encode (fork_ai8.npz: source planes, the switches the encoder held) the pruned frame
    call evaluates exactly the PUs the encoder's RMD loop visited, with the costs of the full enumeration; every other PU inside
    the picture carries CUCD_COST_PRUNED.  Host-buffer call (wide and packed tables) and the device-resident begin / end call."""
    import torch
    from _util import oracle_prune_mask, pu_table_index
    g = golden("fork_ai8.npz")
    W, H, bd = [int(v) for v in g[f"{name}_meta"]]
    pocs = [int(p) for p in g[f"{name}_pocs"]]
    orgs = [g[f"{name}_p{p}_org"] for p in pocs]
    recs = [pseudo_recon(o, bd) for o in orgs]
    nctu = ((W + 63) // 64) * ((H + 63) // 64)
    with cucd.Engine(W, H, bit_depth=bd, max_pictures=len(pocs)) as eng:
        full = eng.frames(orgs, recs)
        for k, poc in enumerate(pocs):
            sk, te = g[f"{name}_p{poc}_skip"], g[f"{name}_p{poc}_term"]
            eng.set_decision_switches(1, sk, te)
            got = eng.frames([orgs[k]], [recs[k]])[0]
            outp = eng.alloc_frame_out(True, packed=True, narrow=True)
            eng.frames([orgs[k]], [recs[k]], [outp])
            assert np.array_equal(got["obf"], g[f"{name}_p{poc}_obf"]) and np.array_equal(got["obf"], full[k]["obf"])
            vis = np.zeros((nctu, 341), bool)
            for x, y, n in g[f"{name}_p{poc}_visited"]:
                vis[(int(y) // 64) * ((W + 63) // 64) + int(x) // 64, pu_table_index(int(x), int(y), int(n))] = True
            assert np.array_equal(vis, oracle_prune_mask(oracle, got["obf"], W, H, sk, te).astype(bool))
            inside = full[k]["rmd_cost"][:, :, 0] != cucd.COST_NOT_INSIDE
            want = np.where(vis[:, :, None], full[k]["rmd_cost"], np.where(inside[:, :, None], np.uint32(cucd.COST_PRUNED), np.uint32(cucd.COST_NOT_INSIDE)))
            assert np.array_equal(got["rmd_cost"], want), (name, poc)
            assert np.array_equal(cucd.unpack_costs(outp["rmd_cost_packed"]), want)
            assert np.array_equal(eng.unpack_costs_c(outp["rmd_cost_packed"]), want)
            # device-resident, split call
            dev = torch.device("cuda", 0); pitch = (W + 63) // 64 * 64
            d_org = torch.zeros((1, H, pitch), dtype=torch.int16, device=dev); d_rec = torch.zeros_like(d_org)
            d_org[0, :, :W] = torch.from_numpy(orgs[k]).to(dev); d_rec[0, :, :W] = torch.from_numpy(recs[k]).to(dev)
            d_cost = torch.zeros((1, nctu, 341, 35), dtype=torch.int32, device=dev)
            st = torch.cuda.current_stream().cuda_stream
            eng.dev_frames(st, 1, d_org.data_ptr(), H * pitch, pitch, d_rec.data_ptr(), H * pitch, pitch, {"rmd_cost": d_cost.data_ptr()}, begin_only=True)
            eng.dev_frames_end()
            torch.cuda.synchronize()
            assert np.array_equal(d_cost[0].cpu().numpy().view(np.uint32), want)
            eng.set_decision_switches(0)
        again = eng.frames(orgs, recs)
        assert all(np.array_equal(a["rmd_cost"], b["rmd_cost"]) for a, b in zip(again, full))


@pytest.mark.parametrize("bd,path", [(8, 1), (8, 0), (10, 0), (10, 1)])
def test_fork_aware_frame_mode_all_switch_patterns(cucd, oracle, bd, path):
    """every Skip2Nx2N / TerminateCU pattern on a picture with flat and textured regions and partial CTUs, tensor-core and ALU kernels"""
    import itertools
    from _util import oracle_prune_mask
    W, H = 328, 200
    org = textured_plane(W, H, bd, seed=51)
    org[:72, :] = 100 << (bd - 8)                        # flat: Num_OBF == 0 there
    org[:, 200:264] = 60 << (bd - 8)
    rec = pseudo_recon(org, bd)
    with cucd.Engine(W, H, bit_depth=bd) as eng:
        eng.set_rmd_path(path)
        full = eng.frame(org, rec)
        inside = full["rmd_cost"][:, :, 0] != cucd.COST_NOT_INSIDE
        for i, bits in enumerate(itertools.product((0, 1), repeat=4)):
            sk, te = bits, bits[::-1] if i % 2 else (1, 1, 1, 1)
            eng.set_decision_switches(1, sk, te)
            got = eng.frame(org, rec)
            need = oracle_prune_mask(oracle, full["obf"], W, H, sk, te).astype(bool)
            want = np.where(need[:, :, None], full["rmd_cost"], np.where(inside[:, :, None], np.uint32(cucd.COST_PRUNED), np.uint32(cucd.COST_NOT_INSIDE)))
            assert np.array_equal(got["rmd_cost"], want), (sk, te)
            assert np.array_equal(got["obf"], full["obf"]) and np.array_equal(got["num_obf2"], full["num_obf2"])
