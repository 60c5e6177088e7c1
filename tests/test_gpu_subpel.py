"""Parity of the fractional-pel refinement kernel (SURVEY.md 8f.3, xPatternSearchFracDIF TEncSearch.cpp:4340-4376) through the
C ABI: against candidates dumped from the reference encoder's xPatternRefinement (tests/golden/frac_*.npz) and against the oracle
on seeded pictures.  Integer work: bit-exact."""
import ctypes as C

import numpy as np
import pytest

from _util import P, frac_records, full_range_keys, golden, i16p, u32p, pseudo_recon, textured_plane

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("clip", ["had8", "sad10"])
def test_subpel_vs_reference_encoder_dump(cucd, clip):
    """each record is laid out in its own 96x96 cell of a canvas pair (source block / reference window at zero integer MV)"""
    recs = list(frac_records(golden(f"frac_{clip}.npz")))
    bd = recs[0]["bd"]
    CELL, PER = 96, 10
    S = CELL * PER
    done = 0
    with cucd.Engine(S, S, bit_depth=bd) as eng:
        for first in range(0, len(recs), PER * PER):
            chunk = recs[first:first + PER * PER]
            cur = np.zeros((S, S), np.int16); ref = np.zeros((S + 32, S + 32), np.int16)
            descs = []
            for i, r in enumerate(chunk):
                x0, y0 = (i % PER) * CELL + 8, (i // PER) * CELL + 8
                cur[y0:y0 + r["h"], x0:x0 + r["w"]] = r["org"]
                ref[16 + y0 - 4:16 + y0 + r["h"] + 5, 16 + x0 - 4:16 + x0 + r["w"] + 5] = r["win"]
                descs.append(dict(x=x0, y=y0, w=r["w"], h=r["h"], ref_idx=0, mvx=0, mvy=0, use_hadamard=r["had"]))
            eng.set_cur_picture(cur); eng.set_ref_picture(0, ref, 16, 16)
            got = eng.me_subpel_cost(descs)
            for i, r in enumerate(chunk):
                assert got[i, r["qy"] + 3, r["qx"] + 3] == r["dist"], (r["w"], r["h"], r["qx"], r["qy"], r["had"])
                done += 1
    assert done == len(recs)


@pytest.mark.parametrize("bd", [8, 9, 10])
def test_subpel_vs_oracle(cucd, oracle, bd):
    W, H, M = 416, 240, 80
    org = textured_plane(W, H, bd, seed=21)
    rec = pseudo_recon(textured_plane(W, H, bd, seed=21, t=1), bd)
    refp = np.pad(rec, M, mode="edge")
    rng = np.random.default_rng(6)
    shapes = [(64, 64), (64, 32), (32, 64), (32, 32), (64, 16), (64, 48), (16, 64), (48, 64), (32, 8), (32, 24), (8, 32), (24, 32), (16, 16), (16, 4), (16, 12),
              (4, 16), (12, 16), (16, 8), (8, 16), (8, 8), (8, 4), (4, 8)]
    descs = []
    for w, h in shapes:
        for had in (1, 0):
            x = int(rng.integers(0, (W - w) // 4 + 1)) * 4; y = int(rng.integers(0, (H - h) // 4 + 1)) * 4
            # include MVs that push the 8-tap support into the replicated margin
            mvx = int(rng.integers(-x - 70, W - x - w + 70)); mvy = int(rng.integers(-y - 70, H - y - h + 70))
            descs.append(dict(x=x, y=y, w=w, h=h, ref_idx=0, mvx=mvx, mvy=mvy, use_hadamard=had))
    with cucd.Engine(W, H, bit_depth=bd) as eng:
        eng.set_cur_picture(org); eng.set_ref_picture(0, refp, M, M)
        got = eng.me_subpel_cost(descs)
        assert eng.me_subpel_cost([]).shape == (0, 7, 7)
        with pytest.raises(cucd.CucdError):
            eng.me_subpel_cost([dict(x=0, y=0, w=8, h=8, ref_idx=0, mvx=-78, mvy=0, use_hadamard=1)])     # support leaves the margin
        with pytest.raises(cucd.CucdError):
            eng.me_subpel_cost([dict(x=0, y=0, w=6, h=8, ref_idx=0, mvx=0, mvy=0, use_hadamard=1)])
    Wp = W + 2 * M
    for i, d in enumerate(descs):
        blk = np.ascontiguousarray(org[d["y"]:d["y"] + d["h"], d["x"]:d["x"] + d["w"]])
        want = np.zeros(49, np.uint32)
        zero = C.c_void_p(refp.ctypes.data + 2 * ((d["y"] + M) * Wp + d["x"] + M))
        oracle.oracle_subpel_surface(bd, P(blk, i16p), d["w"], d["w"], d["h"], zero, Wp, d["mvx"], d["mvy"], d["use_hadamard"], P(want, u32p))
        assert np.array_equal(got[i].ravel(), want), d


@pytest.mark.parametrize("bd,keys", [pytest.param(bd, k, id=str(bd) if k == "hm" else f"{bd}-{k}") for k in ("hm", "int16") for bd in (8, 9, 10)])
def test_bipred_key_blocks_vs_oracle(cucd, oracle, bd, keys):
    """cucd_me_sad_surface_src / cucd_me_subpel_cost_src: the bi-predictive refinement of xMotionEstimation (TEncSearch.cpp:3787-3849)
    searches with the key 2 * org - prediction of the other list (TComYuv::removeHighFreq): samples below 0 and above the bit depth's
    range, caller-supplied blocks instead of the current picture.  Integer search (+-4, xPatternSearch) and the 49 sub-pel positions.
    keys "int16": what the header allows beyond HM's keys - samples from all of int16 with runs of both ends, whole blocks of -32768
    against reference runs of 0 and 2^bd - 1 (|key - ref| up to 32768 + 2^bd - 1), and +-40 windows (several dx-lane tiles a row)."""
    W, H, M = 256, 128, 80
    hi = (1 << bd) - 1
    rec = pseudo_recon(textured_plane(W, H, bd, seed=33, t=1), bd)
    if keys == "hm":
        org = textured_plane(W, H, bd, seed=33).astype(np.int32)
        other = pseudo_recon(textured_plane(W, H, bd, seed=34, t=2), bd).astype(np.int32)
        other[:, ::3] = hi; other[::5, :] = 0                  # push 2 * org - other to both ends of [-hi, 2 * hi]
        key = (2 * org - other).astype(np.int16)
        assert key.min() < 0 and key.max() > hi
        R = 4
    else:
        key = full_range_keys(np.random.default_rng(bd + 60), (H, W))
        rec[3::7, :] = hi; rec[:, 5::11] = 0
        R = 40
    refp = np.pad(rec, M, mode="edge")
    rng = np.random.default_rng(8)
    shapes = [(64, 64), (32, 32), (16, 16), (8, 8), (64, 32), (16, 64), (32, 24), (12, 16), (8, 4), (4, 8)]
    me, sp, blocks = [], [], []
    for k, (w, h) in enumerate(shapes):
        x = int(rng.integers(0, (W - w) // 4 + 1)) * 4; y = int(rng.integers(0, (H - h) // 4 + 1)) * 4
        cx, cy = int(rng.integers(-20, 21)), int(rng.integers(-20, 21))
        me.append(dict(x=x, y=y, w=w, h=h, ref_idx=0, left=cx - R, right=cx + R, top=cy - R, bottom=cy + R, sub_shift=1 if h > 8 else 0))
        sp.append(dict(x=x, y=y, w=w, h=h, ref_idx=0, mvx=cx, mvy=cy, use_hadamard=int(rng.integers(0, 2))))
        blk = np.array(key[y:y + h, x:x + w])
        if keys == "int16" and k % 3 == 0:
            blk[:] = -32768 if k % 2 == 0 else 32767
        blocks.append(blk)
    if keys == "int16":
        assert sum(b.min() == b.max() == -32768 for b in blocks) >= 2 and sum(b.min() == b.max() == 32767 for b in blocks) >= 1
    src = np.concatenate([b.ravel() for b in blocks])
    with cucd.Engine(W, H, bit_depth=bd) as eng:
        eng.set_ref_picture(0, refp, M, M)                     # no cucd_set_cur_picture: the source blocks are the caller's
        surf = eng.me_sad_surface(me, src=src)
        frac = eng.me_subpel_cost(sp, src=src)
        with pytest.raises(cucd.CucdError):
            eng.me_sad_surface(me)                             # the plain call still needs the current picture
    Wp = W + 2 * M
    for i, (d, f, blk) in enumerate(zip(me, sp, blocks)):
        zero = C.c_void_p(refp.ctypes.data + 2 * ((d["y"] + M) * Wp + d["x"] + M))
        want = np.zeros_like(surf[i])
        oracle.oracle_sad_surface(bd, P(blk, i16p), d["w"], d["w"], d["h"], zero, Wp, d["left"], d["right"], d["top"], d["bottom"], d["sub_shift"], P(want, u32p))
        assert np.array_equal(surf[i], want), d
        want49 = np.zeros(49, np.uint32)
        oracle.oracle_subpel_surface(bd, P(blk, i16p), f["w"], f["w"], f["h"], zero, Wp, f["mvx"], f["mvy"], f["use_hadamard"], P(want49, u32p))
        assert np.array_equal(frac[i].ravel(), want49), f
