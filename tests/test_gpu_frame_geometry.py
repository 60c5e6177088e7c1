"""The frame RMD kernels on the GPU at every picture-edge residue (EDGE_SIZES), at the strong-smoothing threshold, across growth and
stream hand-off of the 8-bit kernel's border scratch, and in fork-aware mode on a scratch that holds stale images.  Every picture of
every launch is compared with the plain-C oracle, bit for bit.  cucd_dev_rmd_frames runs no feature pass, so it takes pictures smaller
than a CTU without the TCM fit."""
import numpy as np
import pytest

from _util import EDGE_SIZES, edge_content, oracle_prune_mask, oracle_rmd_frame, pseudo_recon, strong_filter_pus, textured_plane, threshold_picture

pytestmark = pytest.mark.gpu

COST_PRUNED, COST_NOT_INSIDE = np.uint32(0xFFFFFFFE), np.uint32(0xFFFFFFFF)


def _upload(pics, stride):
    """pictures (list of (H, W) int16) as one device tensor (n, H, stride)"""
    import torch
    H, W = pics[0].shape
    a = np.zeros((len(pics), H, stride), np.int16)
    for k, p in enumerate(pics):
        a[k, :, :W] = p
    return torch.from_numpy(a).to("cuda:0")


def _enqueue(eng, orgs, recs, stride=None, stream=None):
    """cucd_dev_rmd_frames over the pictures on `stream` (default: torch's current stream), with the uploads on that stream too, so
    that nothing synchronises the host with launches already queued; returns the device tensors"""
    import torch
    H, W = orgs[0].shape
    S = stride or W
    stream = stream or torch.cuda.current_stream()
    with torch.cuda.stream(stream):
        d_org, d_rec = _upload(orgs, S), _upload(recs, S)
        d_cost = torch.full((len(orgs), eng.ctus_per_pic, 341, 35), -1, dtype=torch.int32, device="cuda:0")
    eng.dev_rmd_frames(stream.cuda_stream, len(orgs), d_org.data_ptr(), H * S, S, d_rec.data_ptr(), H * S, S, d_cost.data_ptr())
    return d_org, d_rec, d_cost


def _costs(d_cost):
    return d_cost.cpu().numpy().view(np.uint32)


def _check_every_picture(oracle, got, orgs, recs, bd, strong, tag):
    for k, (o, r) in enumerate(zip(orgs, recs)):
        assert np.array_equal(got[k], oracle_rmd_frame(oracle, o, r, bd, strong)), (tag, k)


# ---- the sweep -------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("bd", [8, 9, 10])
@pytest.mark.parametrize("W,H", EDGE_SIZES)
def test_dev_rmd_frames_at_edge_sizes_vs_oracle(cucd, oracle, W, H, bd):
    """3 pictures of different content per launch; 8 bit: ALU, kind::i8 (border pre-pass + bulk copies) and kind::f16 kernels;
    9 / 10 bit: ALU and kind::f16.  One size also runs with planes whose stride exceeds the width (W + 72 samples)."""
    import torch
    pics = [edge_content(W, H, bd, seed=W * 3 + H + 100 * k) for k in range(3)]
    orgs = [p[0] for p in pics]; recs = [p[1] for p in pics]
    if W >= 32 and H >= 32:                            # a 32x32 PU fits: the strong filter changes its table
        assert strong_filter_pus(oracle, orgs[0], recs[0], bd)
    strides = [None, W + 72] if (W, H) == (88, 104) else [None]
    with cucd.Engine(W, H, bit_depth=bd, max_pictures=3) as eng:
        for path in ((0, 1, 2) if bd == 8 else (0, 1)):
            eng.set_rmd_path(path)
            for S in strides:
                _, _, d_cost = _enqueue(eng, orgs, recs, S)
                torch.cuda.synchronize()
                _check_every_picture(oracle, _costs(d_cost), orgs, recs, bd, 1, (path, S))


@pytest.mark.parametrize("bd", [8, 10])
@pytest.mark.parametrize("strong", [0, 1])
def test_dev_rmd_frames_at_the_strong_smoothing_threshold(cucd, oracle, bd, strong):
    """32x32 borders whose deviations sit at 1 << (bd - 5) and one below it (threshold_picture asserts that they do)"""
    import torch
    org, rec = threshold_picture(oracle, bd)
    H, W = org.shape
    orgs, recs = [org, rec, org], [rec, org, org]     # the threshold reconstruction first, then other borders
    with cucd.Engine(W, H, bit_depth=bd, strong_intra_smoothing=strong, max_pictures=3) as eng:
        for path in ((0, 1, 2) if bd == 8 else (0, 1)):
            eng.set_rmd_path(path)
            _, _, d_cost = _enqueue(eng, orgs, recs)
            torch.cuda.synchronize()
            _check_every_picture(oracle, _costs(d_cost), orgs, recs, bd, strong, path)


# ---- the border scratch of the 8-bit kernel ------------------------------------------------------------------------------------------
def test_border_scratch_grows_beyond_max_pictures(cucd, oracle):
    """the handle sizes its scratch for max_pictures = 1; cucd_dev_rmd_frames then asks for 4 pictures and 2"""
    import torch
    W, H = 200, 136
    with cucd.Engine(W, H, max_pictures=1) as eng:
        eng.set_rmd_path(1)
        for n, seed in ((1, 300), (4, 310), (2, 320)):
            pics = [edge_content(W, H, 8, seed=seed + k) for k in range(n)]
            orgs = [p[0] for p in pics]; recs = [p[1] for p in pics]
            _, _, d_cost = _enqueue(eng, orgs, recs)
            torch.cuda.synchronize()
            _check_every_picture(oracle, _costs(d_cost), orgs, recs, 8, 1, n)


def test_border_scratch_two_streams(cucd, oracle):
    """A 4-picture launch on one stream and a launch of other content on a second stream.  Both launches' inputs are on the device
    first; then the two are enqueued back to back, with no synchronisation between them, so that the second launch's border pre-pass
    would rewrite the scratch while the first launch's RMD CTAs may still read it unless the handle orders the two.  One attempt."""
    import torch
    W, H = 416, 240
    a = [edge_content(W, H, 8, seed=400 + k) for k in range(4)]
    b = [(textured_plane(W, H, 8, seed=500 + k), np.random.default_rng(500 + k).integers(0, 256, (H, W)).astype(np.int16)) for k in range(4)]
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    with cucd.Engine(W, H, max_pictures=4) as eng:
        eng.set_rmd_path(1)
        bufs = []
        for pics in (a, b):
            bufs.append((_upload([p[0] for p in pics], W), _upload([p[1] for p in pics], W),
                         torch.full((4, eng.ctus_per_pic, 341, 35), -1, dtype=torch.int32, device="cuda:0")))
        torch.cuda.synchronize()
        for (d_org, d_rec, d_cost), s in zip(bufs, (s1, s2)):
            eng.dev_rmd_frames(s.cuda_stream, 4, d_org.data_ptr(), H * W, W, d_rec.data_ptr(), H * W, W, d_cost.data_ptr())
        torch.cuda.synchronize()
        _check_every_picture(oracle, _costs(bufs[0][2]), [p[0] for p in a], [p[1] for p in a], 8, 1, "stream 1")
        _check_every_picture(oracle, _costs(bufs[1][2]), [p[0] for p in b], [p[1] for p in b], 8, 1, "stream 2")


def test_dev_frames_two_batches_on_two_streams(cucd):
    """cucd_dev_frames_begin on two streams with both batches in flight, then the two ends: the same tables and features as the
    host frames() call.  One attempt."""
    import torch
    W, H, P = 416, 240, 2
    batches = []
    for b in range(2):
        orgs = [textured_plane(W, H, 8, seed=600 + 10 * b + k) for k in range(P)]
        batches.append((orgs, [pseudo_recon(o, 8) for o in orgs]))
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    with cucd.Engine(W, H, max_pictures=P) as eng:
        dev = []
        for (orgs, recs), s in zip(batches, streams):
            with torch.cuda.stream(s):
                d_org, d_rec = _upload(orgs, W), _upload(recs, W)
                d_cost = torch.full((P, eng.ctus_per_pic, 341, 35), -1, dtype=torch.int32, device="cuda:0")
                d_obf = torch.zeros((P, H // 4, W // 4), dtype=torch.int16, device="cuda:0")
            eng.dev_frames(s.cuda_stream, P, d_org.data_ptr(), H * W, W, d_rec.data_ptr(), H * W, W,
                           {"obf": d_obf.data_ptr(), "rmd_cost": d_cost.data_ptr()}, begin_only=True)
            dev.append((d_org, d_rec, d_cost, d_obf))
        eng.dev_frames_end()
        eng.dev_frames_end()
        torch.cuda.synchronize()
        for (orgs, recs), (_, _, d_cost, d_obf) in zip(batches, dev):
            want = eng.frames(orgs, recs)
            for p in range(P):
                assert np.array_equal(_costs(d_cost)[p], want[p]["rmd_cost"]), p
                assert np.array_equal(d_obf[p].cpu().numpy(), want[p]["obf"]), p


# ---- fork-aware mode on a scratch that holds stale images --------------------------------------------------------------------------
@pytest.mark.parametrize("path", [1, 0])
def test_fork_aware_first_call_and_after_other_content(cucd, oracle, path):
    """A fork-aware call writes no image for a (CTU, depth) with nothing to evaluate, while the RMD CTAs still copy that CTU's slot.
    On a fresh handle the first call is fork-aware; on another, a full call on noise comes first.  Both equal the full enumeration of a
    separate handle with the pruned and outside-picture codes filled in.  Every handle is created before the full enumeration runs and
    stays open to the end, so no handle's scratch can be memory that held this picture's correct images."""
    import torch
    W, H = 328, 200
    org = textured_plane(W, H, 8, seed=51)
    org[:72, :] = 100
    org[:, 200:264] = 60
    rec = pseudo_recon(org, 8)
    noise = np.random.default_rng(9).integers(0, 256, (2, H, W)).astype(np.int16)
    patterns = [((1, 1, 1, 1), (1, 1, 1, 1)), ((0, 1, 0, 1), (1, 0, 1, 0)), ((1, 0, 0, 0), (0, 0, 1, 1))]
    engines = [cucd.Engine(W, H) for _ in range(2 * len(patterns) + 1)]
    try:
        ref = engines[-1]
        for eng in engines:
            eng.set_rmd_path(path)
        full = ref.frame(org, rec)
        assert np.array_equal(full["rmd_cost"], oracle_rmd_frame(oracle, org, rec, 8))
        inside = full["rmd_cost"][:, :, 0] != COST_NOT_INSIDE
        for i, (sk, te) in enumerate(patterns):
            need = oracle_prune_mask(oracle, full["obf"], W, H, sk, te).astype(bool)
            want = np.where(need[:, :, None], full["rmd_cost"], np.where(inside[:, :, None], COST_PRUNED, COST_NOT_INSIDE))
            assert (inside & ~need).any() and need.any()
            for stale in (False, True):
                eng = engines[2 * i + stale]
                if stale:                                   # a full launch on noise fills the scratch with other images
                    _, _, d_cost = _enqueue(eng, [noise[0]], [noise[1]])
                    torch.cuda.synchronize()
                    assert np.array_equal(_costs(d_cost)[0], oracle_rmd_frame(oracle, noise[0], noise[1], 8))
                eng.set_decision_switches(1, sk, te)
                got = eng.frame(org, rec)
                assert np.array_equal(got["rmd_cost"], want), (sk, te, stale)
    finally:
        for eng in engines:
            eng.close()
