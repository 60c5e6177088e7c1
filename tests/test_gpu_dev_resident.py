"""The device-resident ME and feature-pass calls checked value by value: cucd_dev_me_sad_surface / cucd_dev_me_subpel_cost on the
benchmark's inter workloads, their stream and buffer-reuse contract, and cucd_dev_feature_hist -> cucd_tcm_fit -> cucd_dev_feature_obf
step by step.  These calls have plumbing of their own (job records through the handle's own pinned and device blocks, guarded by
events; kernels left queued on the caller's stream), so they are compared with the oracle and with the host-buffer calls, which
tests/test_gpu_parity.py, tests/test_gpu_subpel.py and tests/test_gpu_encoder_workloads.py pin to the oracle.  Integer work:
bit-exact."""
import ctypes as C

import numpy as np
import pytest

import bench
from _util import (P, i16p, u32p, oracle_ctu_src_had, oracle_cu_sums, oracle_outlier_frame, pseudo_recon, textured_plane)
from test_capi_load import _extreme_outlier_plane

pytestmark = pytest.mark.gpu

SPIN_CYCLES = 50_000_000          # torch.cuda._sleep: ~25 ms at the B200's ~2 GHz SM clock


def _torch():
    import torch
    return torch, torch.device("cuda", 0)


def _me_setup(W, H, bd, n_refs, seed):
    """the planes of run_inter in bench.py: current picture t = 1, references pseudo_recon(t = 0 / 2) padded by ME_MARGIN"""
    M = bench.ME_MARGIN
    cur = textured_plane(W, H, bd, seed, 1)
    refs = [np.ascontiguousarray(np.pad(pseudo_recon(textured_plane(W, H, bd, seed, (0, 2)[k]), bd, 10 + k), M, mode="edge")) for k in range(n_refs)]
    return cur, refs


def _me_descs(pus, k):
    R = bench.ME_RANGE
    return [dict(x=x, y=y, w=s, h=s, ref_idx=k, left=-R, right=R, top=-R, bottom=R, sub_shift=1 if s > 8 else 0) for x, y, s in pus]


def _subpel_descs(pus, k, W, H, M, rng):
    """seeded integer MVs for the 49-point tables: every eighth PU puts the 8-tap support exactly on one side of the padded plane
    (x + mvx - 4 == -M, x + mvx + w + 4 == W - 1 + M, and the same vertically), the others lie in the +-64 window or anywhere
    in the plane; use_hadamard alternates at random"""
    out = []
    for i, (x, y, s) in enumerate(pus):
        lox, hix = -M + 4 - x, W - 1 + M - 4 - s - x
        loy, hiy = -M + 4 - y, H - 1 + M - 4 - s - y
        if i % 8 < 4 or i % 8 == 7:
            mvx, mvy = int(rng.integers(lox, hix + 1)), int(rng.integers(loy, hiy + 1))
        else:
            mvx, mvy = int(rng.integers(max(lox, -64), min(hix, 64) + 1)), int(rng.integers(max(loy, -64), min(hiy, 64) + 1))
        side = i % 8
        mvx = lox if side == 0 else hix if side == 1 else mvx
        mvy = loy if side == 2 else hiy if side == 3 else mvy
        out.append(dict(x=x, y=y, w=s, h=s, ref_idx=k, mvx=mvx, mvy=mvy, use_hadamard=int(rng.integers(0, 2))))
    return out


def _support_sides(d, W, H, M):
    """the sides of the padded plane the 8-tap support of a sub-pel descriptor touches"""
    return {side for side, hit in (("left", d["x"] + d["mvx"] - 4 == -M), ("right", d["x"] + d["mvx"] + d["w"] + 4 == W - 1 + M),
                                   ("top", d["y"] + d["mvy"] - 4 == -M), ("bottom", d["y"] + d["mvy"] + d["h"] + 4 == H - 1 + M)) if hit}


def _oracle_sad(oracle, bd, cur, refp, M, d):
    S = refp.shape[1]
    blk = np.ascontiguousarray(cur[d["y"]:d["y"] + d["h"], d["x"]:d["x"] + d["w"]])
    out = np.zeros((d["bottom"] - d["top"] + 1) * (d["right"] - d["left"] + 1), np.uint32)
    zero = C.c_void_p(refp.ctypes.data + 2 * ((d["y"] + M) * S + d["x"] + M))
    oracle.oracle_sad_surface(bd, P(blk, i16p), d["w"], d["w"], d["h"], zero, S, d["left"], d["right"], d["top"], d["bottom"], d["sub_shift"], P(out, u32p))
    return out


def _oracle_subpel(oracle, bd, cur, refp, M, d):
    S = refp.shape[1]
    blk = np.ascontiguousarray(cur[d["y"]:d["y"] + d["h"], d["x"]:d["x"] + d["w"]])
    out = np.zeros(49, np.uint32)
    zero = C.c_void_p(refp.ctypes.data + 2 * ((d["y"] + M) * S + d["x"] + M))
    oracle.oracle_subpel_surface(bd, P(blk, i16p), d["w"], d["w"], d["h"], zero, S, d["mvx"], d["mvy"], d["use_hadamard"], P(out, u32p))
    return out


def _offsets(descs):
    sizes = [(d["bottom"] - d["top"] + 1) * (d["right"] - d["left"] + 1) for d in descs]
    return np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)


def _u32(t):
    return t.cpu().numpy().view(np.uint32)


class _MeCall:
    """descriptor arrays of one cucd_dev_me_sad_surface + cucd_dev_me_subpel_cost pair and device buffers for their results, filled
    with 0xFFFFFFFF so that an entry the kernels miss cannot pass.  The fills run on torch's stream: synchronise before enqueue()
    puts the calls on another stream."""

    def __init__(self, eng, me, sp):
        torch, dev = _torch()
        self.eng, self.me, self.sp = eng, me, sp
        self.arr, self.n, total = eng.me_descs(me)
        self.sarr, self.sn = eng.subpel_descs(sp)
        self.d_sad = torch.full((total,), -1, dtype=torch.int32, device=dev)
        self.d_sub = torch.full((self.sn, 49), -1, dtype=torch.int32, device=dev)

    def enqueue(self, stream):
        self.eng.dev_me_sad_surface(stream, self.arr, self.n, self.d_sad.data_ptr())
        self.eng.dev_me_subpel_cost(stream, self.sarr, self.sn, self.d_sub.data_ptr())
        return self.d_sad, self.d_sub


def _dev_me(eng, stream, me, sp):
    """one _MeCall enqueued on `stream`: returns the two buffers, still being written there"""
    torch, _ = _torch()
    call = _MeCall(eng, me, sp)
    torch.cuda.synchronize()
    return call.enqueue(stream)


def _check_me_vs_oracle(oracle, bd, cur, refs, margins, me, sp, d_sad, d_sub, which=None):
    """every PU of the device buffers against the oracle; refs / margins per reference slot"""
    sad, sub = _u32(d_sad), _u32(d_sub)
    offs = _offsets(me)
    assert offs[-1] == sad.size
    for i in (range(len(me)) if which is None else which):
        d, f = me[i], sp[i]
        assert np.array_equal(sad[offs[i]:offs[i + 1]], _oracle_sad(oracle, bd, cur, refs[d["ref_idx"]], margins[d["ref_idx"]], d)), d
        assert np.array_equal(sub[i], _oracle_subpel(oracle, bd, cur, refs[f["ref_idx"]], margins[f["ref_idx"]], f)), f


def _sample_pus(pus, W, H, rng, per_size=64):
    """indices of the four corner PUs of every size and a seeded sample of `per_size` more per size, half of it on the picture edges"""
    index = {pu: i for i, pu in enumerate(pus)}
    picked = []
    for s in sorted({s for _, _, s in pus}):
        xmax, ymax = (W - s) // s * s, (H - s) // s * s
        corners = [index[(x, y, s)] for x, y in ((0, 0), (xmax, 0), (0, ymax), (xmax, ymax))]
        mine = [i for i, (x, y, t) in enumerate(pus) if t == s]
        edge = [i for i in mine if pus[i][0] in (0, xmax) or pus[i][1] in (0, ymax)]
        picked += corners + list(rng.choice(edge, min(len(edge), per_size // 2), replace=False)) + list(rng.choice(mine, per_size // 2, replace=False))
    return sorted(set(int(i) for i in picked))


# ---- a. the benchmark's ME workloads, device-resident ----------------------------------------------------------------------
@pytest.mark.parametrize("name", ["ldp1080p", "ra1080p10"])
def test_bench_me_workload_device_resident(cucd, oracle, name):
    """ldp1080p (8 bit, one reference) and ra1080p10 (10 bit, two reference slots): every square PU of bench.inter_pus with the
    benchmark's +-64 window and sub_shift in one device-resident call per reference, and seeded sub-pel MVs (both DistFuncs, supports
    ending exactly at the margin).  The whole output equals the host-buffer calls on consecutive slices of the same descriptors;
    the corner PUs of every size and a seeded sample, partly on the picture edges, equal the oracle."""
    torch, dev = _torch()
    cfg = bench.CONFIGS[name]
    W, H, bd, NR, M = cfg["width"], cfg["height"], cfg["bit_depth"], cfg["refs"], bench.ME_MARGIN
    cur, refs = _me_setup(W, H, bd, NR, 20261018)
    pus = bench.inter_pus(W, H)
    rng = np.random.default_rng(bd * 10 + NR)
    me = [_me_descs(pus, k) for k in range(NR)]
    sp = [_subpel_descs(pus, k, W, H, M, rng) for k in range(NR)]
    with cucd.Engine(W, H, bit_depth=bd) as eng:
        eng.set_cur_picture(cur)
        for k in range(NR):
            eng.set_ref_picture(k, refs[k], M, M)
        calls = [_MeCall(eng, me[k], sp[k]) for k in range(NR)]
        out = [c.enqueue(torch.cuda.current_stream().cuda_stream) for c in calls]
        torch.cuda.synchronize()
        SLICE = 2000
        for k, (d_sad, d_sub) in enumerate(out):
            off = 0
            for a in range(0, len(pus), SLICE):
                arr, n, total = eng.me_descs(me[k][a:a + SLICE])
                host = np.empty(total, np.uint32)
                eng.me_sad_surface_raw(arr, n, host)
                assert torch.equal(d_sad[off:off + total], torch.from_numpy(host.view(np.int32)).to(dev)), (name, k, a)
                off += total
                assert np.array_equal(_u32(d_sub[a:a + n]), eng.me_subpel_cost(sp[k][a:a + SLICE]).reshape(n, 49)), (name, k, a)
            assert off == d_sad.numel()
        sample = _sample_pus(pus, W, H, rng)
        for k, (d_sad, d_sub) in enumerate(out):
            assert {"left", "right", "top", "bottom"} <= set().union(*(_support_sides(sp[k][i], W, H, M) for i in sample))
            offs = _offsets(me[k])
            for i in sample:
                got = _u32(d_sad[offs[i]:offs[i + 1]])
                assert np.array_equal(got, _oracle_sad(oracle, bd, cur, refs[k], M, me[k][i])), (name, k, me[k][i])
                assert np.array_equal(_u32(d_sub[i]), _oracle_subpel(oracle, bd, cur, refs[k], M, sp[k][i])), (name, k, sp[k][i])


@pytest.mark.parametrize("bd,n_refs", [(8, 1), (9, 2), (10, 2)])
def test_small_picture_me_device_resident_vs_oracle(cucd, oracle, bd, n_refs):
    """416x240 (partial CTUs on the bottom edge): every square PU, every candidate and every sub-pel table against the oracle"""
    torch, _ = _torch()
    W, H, M = 416, 240, bench.ME_MARGIN
    cur, refs = _me_setup(W, H, bd, n_refs, 20261019)
    pus = bench.inter_pus(W, H)
    rng = np.random.default_rng(bd)
    with cucd.Engine(W, H, bit_depth=bd) as eng:
        eng.set_cur_picture(cur)
        for k in range(n_refs):
            eng.set_ref_picture(k, refs[k], M, M)
        st = torch.cuda.current_stream().cuda_stream
        for k in range(n_refs):
            me, sp = _me_descs(pus, k), _subpel_descs(pus, k, W, H, M, rng)
            d_sad, d_sub = _dev_me(eng, st, me, sp)
            torch.cuda.synchronize()
            _check_me_vs_oracle(oracle, bd, cur, refs, [M] * n_refs, me, sp, d_sad, d_sub)


# ---- b. stream and buffer-reuse contract of the device-resident ME calls ----------------------------------------------------
def _random_me(rng, W, H, M, n, win, k=0):
    """n PUs of HM's shapes with windows of up to +-win inside the padded plane, and their sub-pel descriptors"""
    shapes = [(64, 64), (32, 32), (16, 16), (8, 8), (64, 32), (16, 64), (32, 24), (12, 16), (8, 4), (4, 8), (48, 64), (16, 12)]
    me, sp = [], []
    for _ in range(n):
        w, h = shapes[int(rng.integers(0, len(shapes)))]
        x, y = int(rng.integers(0, (W - w) // 4 + 1)) * 4, int(rng.integers(0, (H - h) // 4 + 1)) * 4
        left, top = max(-win, -M - x), max(-win, -M - y)
        right, bottom = min(win, W - 1 + M - x - w + 1), min(win, H - 1 + M - y - h + 1)
        l2, t2 = int(rng.integers(left, right + 1)), int(rng.integers(top, bottom + 1))
        r2, b2 = int(rng.integers(l2, right + 1)), int(rng.integers(t2, bottom + 1))
        me.append(dict(x=x, y=y, w=w, h=h, ref_idx=k, left=l2, right=r2, top=t2, bottom=b2, sub_shift=1 if h > 8 else 0))
        mvx = int(rng.integers(max(-M + 4 - x, -win), min(W - 1 + M - 4 - w - x, win) + 1))
        mvy = int(rng.integers(max(-M + 4 - y, -win), min(H - 1 + M - 4 - h - y, win) + 1))
        sp.append(dict(x=x, y=y, w=w, h=h, ref_idx=k, mvx=mvx, mvy=mvy, use_hadamard=int(rng.integers(0, 2))))
    return me, sp


def test_dev_me_back_to_back_growing_records_and_host_call_between(cucd, oracle):
    """two device-resident SAD calls back to back on one stream, the second with more PUs and larger windows (its records no
    longer fit the device block of the first), a host-buffer call, then a device-resident sub-pel call; nothing waits in between"""
    torch, dev = _torch()
    W, H, bd, M = 416, 240, 8, bench.ME_MARGIN
    cur, refs = _me_setup(W, H, bd, 1, 31)
    rng = np.random.default_rng(31)
    me1, _ = _random_me(rng, W, H, M, 40, 8)
    me2, _ = _random_me(rng, W, H, M, 400, 40)
    me3, _ = _random_me(rng, W, H, M, 30, 16)
    _, sp4 = _random_me(rng, W, H, M, 300, 64)
    with cucd.Engine(W, H, bit_depth=bd) as eng:
        eng.set_cur_picture(cur)
        eng.set_ref_picture(0, refs[0], M, M)
        bufs = []
        for me in (me1, me2):
            arr, n, total = eng.me_descs(me)
            bufs.append(torch.full((total,), -1, dtype=torch.int32, device=dev))
        sarr, sn = eng.subpel_descs(sp4)
        d_sub = torch.full((sn, 49), -1, dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        st = torch.cuda.Stream()
        for me, buf in zip((me1, me2), bufs):
            arr, n, _ = eng.me_descs(me)
            eng.dev_me_sad_surface(st.cuda_stream, arr, n, buf.data_ptr())
        host = eng.me_sad_surface(me3)
        eng.dev_me_subpel_cost(st.cuda_stream, sarr, sn, d_sub.data_ptr())
        st.synchronize()
    for d, got in zip(me3, host):
        assert np.array_equal(got.ravel(), _oracle_sad(oracle, bd, cur, refs[0], M, d)), d
    for me, buf in zip((me1, me2), bufs):
        sad, offs = _u32(buf), _offsets(me)
        for i, d in enumerate(me):
            assert np.array_equal(sad[offs[i]:offs[i + 1]], _oracle_sad(oracle, bd, cur, refs[0], M, d)), d
    sub = _u32(d_sub)
    for i, f in enumerate(sp4):
        assert np.array_equal(sub[i], _oracle_subpel(oracle, bd, cur, refs[0], M, f)), f


def test_dev_me_calls_alternating_streams(cucd, oracle):
    """successive device-resident calls alternating between two streams, then on stream 0 (the legacy default stream)"""
    torch, dev = _torch()
    W, H, bd, M = 416, 240, 10, bench.ME_MARGIN
    cur, refs = _me_setup(W, H, bd, 2, 32)
    rng = np.random.default_rng(32)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    plan = [s1.cuda_stream, s2.cuda_stream, s1.cuda_stream, s2.cuda_stream, None]
    calls = [_random_me(rng, W, H, M, 60 + 20 * j, 24, k=j % 2) for j in range(len(plan))]
    with cucd.Engine(W, H, bit_depth=bd) as eng:
        eng.set_cur_picture(cur)
        for k in range(2):
            eng.set_ref_picture(k, refs[k], M, M)
        pending = [_MeCall(eng, me, sp) for me, sp in calls]
        torch.cuda.synchronize()
        outs = [c.enqueue(stream) for stream, c in zip(plan, pending)]          # nothing waits between the calls
        torch.cuda.synchronize()
    for (me, sp), (d_sad, d_sub) in zip(calls, outs):
        _check_me_vs_oracle(oracle, bd, cur, refs, [M, M], me, sp, d_sad, d_sub)


def test_picture_replacement_while_dev_me_work_is_queued(cucd, oracle):
    """A caller enqueues the device-resident ME of picture A and uploads picture B at once (include/cucudecide.h): the queued
    work must see A and its references, the next call B.  A bounded spin on the stream keeps the work queued while the setters
    run, so that the order is deterministic.  The sub-pel call waits on the host for the records of the SAD call to be uploaded,
    which the first spin delays; a second spin between the two keeps the sub-pel kernel queued when the setters run.  Slot 1 is
    replaced with a smaller margin (a new stride in the reference table, same device block).  Once on a side stream, once on
    stream 0.  The kernels run once beforehand: with lazy module loading the first launch of a kernel waits for the device to go
    idle, which would end the spins before the setters run."""
    torch, dev = _torch()
    W, H, bd, M, M1 = 416, 240, 8, bench.ME_MARGIN, 72
    curA, (refA0, refA1) = _me_setup(W, H, bd, 2, 41)
    curB, (refB0,) = _me_setup(W, H, bd, 1, 42)
    refB1 = np.ascontiguousarray(np.pad(pseudo_recon(textured_plane(W, H, bd, 43, 2), bd, 3), M1, mode="edge"))
    refsA, refsB = ([refA0, refA1], [M, M]), ([refB0, refB1], [M, M1])
    rng = np.random.default_rng(41)
    rounds = []
    for _ in range(2):
        me, sp = [], []
        for k in (0, 1):                         # windows and supports inside margin M1: the same descriptors are valid for B
            a, b = _random_me(rng, W, H, M1, 40, 64, k=k)
            me += a; sp += b
        rounds.append((me, sp))
    errors = []
    with cucd.Engine(W, H, bit_depth=bd) as eng:
        eng.set_cur_picture(curA); eng.set_ref_picture(0, refA0, M, M); eng.set_ref_picture(1, refA1, M, M)
        _dev_me(eng, torch.cuda.current_stream().cuda_stream, rounds[0][0] + rounds[1][0], rounds[0][1] + rounds[1][1])
        torch.cuda.synchronize()
        for stream, (me, sp) in zip((torch.cuda.Stream(), torch.cuda.default_stream()), rounds):
            eng.set_cur_picture(curA); eng.set_ref_picture(0, refA0, M, M); eng.set_ref_picture(1, refA1, M, M)
            call = _MeCall(eng, me, sp)
            torch.cuda.synchronize()
            st = stream.cuda_stream
            with torch.cuda.stream(stream):
                torch.cuda._sleep(SPIN_CYCLES)
            eng.dev_me_sad_surface(st, call.arr, call.n, call.d_sad.data_ptr())
            with torch.cuda.stream(stream):
                torch.cuda._sleep(SPIN_CYCLES)
            eng.dev_me_subpel_cost(st, call.sarr, call.sn, call.d_sub.data_ptr())
            eng.set_cur_picture(curB); eng.set_ref_picture(0, refB0, M, M); eng.set_ref_picture(1, refB1, M1, M1)
            stream.synchronize()
            sad, sub, offs = _u32(call.d_sad), _u32(call.d_sub), _offsets(me)
            tally = {"sad": [0, 0, 0], "subpel": [0, 0, 0]}          # PUs with picture A's values, with picture B's, with neither
            for i, (d, f) in enumerate(zip(me, sp)):
                k, g = d["ref_idx"], sad[offs[i]:offs[i + 1]]
                t = tally["sad"]
                if np.array_equal(g, _oracle_sad(oracle, bd, curA, refsA[0][k], refsA[1][k], d)):
                    t[0] += 1
                else:
                    t[1 if np.array_equal(g, _oracle_sad(oracle, bd, curB, refsB[0][k], refsB[1][k], d)) else 2] += 1
                k, g, t = f["ref_idx"], sub[i], tally["subpel"]
                if np.array_equal(g, _oracle_subpel(oracle, bd, curA, refsA[0][k], refsA[1][k], f)):
                    t[0] += 1
                else:
                    t[1 if np.array_equal(g, _oracle_subpel(oracle, bd, curB, refsB[0][k], refsB[1][k], f)) else 2] += 1
            if tally["sad"][0] != len(me) or tally["subpel"][0] != len(sp):
                errors.append(f"stream {st}: PUs with picture A's / picture B's / other values: SAD surfaces {tally['sad']}, "
                              f"sub-pel tables {tally['subpel']}")
            # the next call sees B, the new margin of slot 1 included
            d_sad, d_sub = _dev_me(eng, st, me, sp)
            stream.synchronize()
            _check_me_vs_oracle(oracle, bd, curB, refsB[0], refsB[1], me, sp, d_sad, d_sub)
    assert not errors, errors


# ---- c. the device-resident feature pass, step by step ------------------------------------------------------------------------
def _feature_pictures(W, H, bd):
    """three pictures; the second carries the 4x4 patterns that maximise single AC coefficients (|c| >= 4096: histogram bins
    >= 512, which the kernel counts with global atomics)"""
    a = textured_plane(W, H, bd, seed=W + bd)
    b = textured_plane(W, H, bd, seed=W + bd + 1, t=2).copy()
    b[:128, :128] = _extreme_outlier_plane(bd, 5)
    c = pseudo_recon(textured_plane(W, H, bd, seed=W + bd + 2), bd)
    return [np.ascontiguousarray(p) for p in (a, b, c)]


def _device_planes(pics, bd, pitch, pic_stride, offset, seed):
    """the pictures in one device buffer: picture p at offset + p * pic_stride samples, rows `pitch` apart; the samples between and
    after the rows are in-range noise, so that a kernel reading them would give other answers.  Returns (buffer, base pointer)."""
    torch, dev = _torch()
    H, W = pics[0].shape
    host = np.random.default_rng(seed).integers(0, 1 << bd, offset + len(pics) * pic_stride + 64).astype(np.int16)
    for p, pic in enumerate(pics):
        start = offset + p * pic_stride
        host[start:start + H * pitch].reshape(H, pitch)[:, :W] = pic
    buf = torch.from_numpy(host).to(dev)
    return buf, buf.data_ptr() + 2 * offset


def _oracle_hist(oracle, org, bd):
    """[16][4096] counts of min(|c| >> 3, 4095) of oracle_dct4x4 over the whole 4x4 blocks, frequencies 1..15"""
    H, W = org.shape
    coef = np.zeros((H // 4 * (W // 4), 16), np.int32)
    i = 0
    for by in range(H // 4):
        for bx in range(W // 4):
            oracle.oracle_dct4x4(bd, C.c_void_p(org.ctypes.data + 2 * (4 * by * W + 4 * bx)), W, C.c_void_p(coef.ctypes.data + 64 * i))
            i += 1
    hist = np.zeros((16, 4096), np.uint32)
    for f in range(1, 16):
        hist[f] = np.bincount(np.minimum(np.abs(coef[:, f]) >> 3, 4095), minlength=4096)
    return hist


@pytest.mark.parametrize("W,H", [(200, 136), (1920, 1080)])
@pytest.mark.parametrize("bd", [8, 10])
def test_dev_feature_pass_step_by_step(cucd, oracle, bd, W, H):
    """cucd_dev_feature_hist -> cucd_tcm_fit per picture -> thresholds yc * 8 -> cucd_dev_feature_obf on three pictures in one
    device buffer whose rows are wider than the picture and whose pictures are further apart than H rows; against the oracle and
    against cucd_dev_frames on the same planes.  Alignment: the histogram pass takes an 8-byte aligned base with strides that are
    multiples of 4 samples (and gives the same histograms there), the OBF pass wants 16 bytes and multiples of 8."""
    torch, dev = _torch()
    pics = _feature_pictures(W, H, bd)
    n, nb = len(pics), (W // 4) * (H // 4)
    pitch = W + 40
    pic_stride = (H + 3) * pitch + 64
    buf, base = _device_planes(pics, bd, pitch, pic_stride, 0, bd)
    assert base % 16 == 0
    want_hist = [_oracle_hist(oracle, p, bd) for p in pics]
    assert want_hist[1][:, 512:].sum() > 0                   # the global-atomic bins are populated
    with cucd.Engine(W, H, bit_depth=bd, max_pictures=n) as eng:
        st = torch.cuda.current_stream().cuda_stream
        grid = [eng.cu_grid(d) for d in range(4)]
        d_hist = torch.full((n, 16, 4096), -1, dtype=torch.int32, device=dev)
        eng.dev_feature_hist(st, n, base, pic_stride, pitch, d_hist.data_ptr())
        hist = _u32(d_hist)
        for p in range(n):
            assert np.array_equal(hist[p], want_hist[p]), p
        fits = [cucd.tcm_fit(hist[p], nb) for p in range(n)]
        thr = np.stack([(yc * 8).astype(np.int32) for yc, _ in fits])
        for p, (yc, t) in enumerate(fits):
            assert np.array_equal(t[1:], thr[p, 1:])
        d_thr = torch.from_numpy(thr).to(dev)
        d_obf = torch.full((n, H // 4, W // 4), -1, dtype=torch.int16, device=dev)
        d_outl = torch.full((n, H, W), -1, dtype=torch.int16, device=dev)
        d_num = [torch.full((n,) + grid[d], -1, dtype=torch.int32, device=dev) for d in range(4)]
        d_sum = [torch.full((n,) + grid[d], -1, dtype=torch.int32, device=dev) for d in range(4)]
        d_had = torch.full((n, eng.ctus_per_pic), -1, dtype=torch.int32, device=dev)
        eng.dev_feature_obf(st, n, base, pic_stride, pitch, d_thr.data_ptr(), d_obf.data_ptr(), d_outl.data_ptr(),
                            [t.data_ptr() for t in d_num], [t.data_ptr() for t in d_sum], d_had.data_ptr())
        got = {"obf": d_obf.cpu().numpy(), "outlier": d_outl.cpu().numpy(), "ctu_src_had": d_had.cpu().numpy()}
        for d in range(4):
            got[f"num_obf{d}"], got[f"n_outlier{d}"] = d_num[d].cpu().numpy(), d_sum[d].cpu().numpy()
        for p, pic in enumerate(pics):
            obf, outl, yc = oracle_outlier_frame(oracle, pic, bd)
            assert np.array_equal(fits[p][0][1:], yc[1:]), p
            assert np.array_equal(got["obf"][p], obf) and np.array_equal(got["outlier"][p], outl), p
            for d in range(4):
                num, tot = oracle_cu_sums(oracle, obf, W, H, d)
                assert np.array_equal(got[f"num_obf{d}"][p], num) and np.array_equal(got[f"n_outlier{d}"][p], tot), (p, d)
            assert np.array_equal(got["ctu_src_had"][p], oracle_ctu_src_had(oracle, pic)), p
        # cucd_dev_frames (features only) on the same planes
        f_obf, f_outl = torch.full_like(d_obf, -1), torch.full_like(d_outl, -1)
        f_num, f_sum = [torch.full_like(t, -1) for t in d_num], [torch.full_like(t, -1) for t in d_sum]
        f_had = torch.full_like(d_had, -1)
        yc_host = np.zeros((n, 16))
        eng.dev_frames(st, n, base, pic_stride, pitch, None, 0, 0,
                       {"obf": f_obf.data_ptr(), "outlier": f_outl.data_ptr(), "num_obf": [t.data_ptr() for t in f_num],
                        "n_outlier": [t.data_ptr() for t in f_sum], "ctu_src_had": f_had.data_ptr()}, yc_host=yc_host)
        torch.cuda.synchronize()
        assert np.array_equal(f_obf.cpu().numpy(), got["obf"]) and np.array_equal(f_outl.cpu().numpy(), got["outlier"])
        assert np.array_equal(f_had.cpu().numpy(), got["ctu_src_had"])
        for d in range(4):
            assert np.array_equal(f_num[d].cpu().numpy(), got[f"num_obf{d}"]) and np.array_equal(f_sum[d].cpu().numpy(), got[f"n_outlier{d}"]), d
        for p in range(n):
            assert np.array_equal(yc_host[p, 1:], fits[p][0][1:]), p

        # alignment: an 8-byte (not 16-byte) aligned base, strides multiples of 4 (not 8) samples
        pitch4 = W + 36
        pic_stride4 = (H + 3) * pitch4 + 4
        buf4, base4 = _device_planes(pics, bd, pitch4, pic_stride4, 4, bd + 1)
        assert base4 % 16 == 8
        d_hist.fill_(-1)
        eng.dev_feature_hist(st, n, base4, pic_stride4, pitch4, d_hist.data_ptr())
        hist4 = _u32(d_hist)
        for p in range(n):
            assert np.array_equal(hist4[p], want_hist[p]), p
        for b, ps, s in ((base4 - 4, pic_stride4, pitch4), (base4, pic_stride4, pitch4 + 2), (base4, pic_stride4 + 2, pitch4),
                         (base4, pic_stride4, W - 4)):
            with pytest.raises(cucd.CucdError):
                eng.dev_feature_hist(st, n, b, ps, s, d_hist.data_ptr())
        for b, ps, s in ((base4, pic_stride4, pitch4), (base, pic_stride, pitch4), (base, pic_stride + 4, pitch), (base + 8, pic_stride, pitch)):
            with pytest.raises(cucd.CucdError):
                eng.dev_feature_obf(st, n, b, ps, s, d_thr.data_ptr(), d_obf.data_ptr(), d_outl.data_ptr(),
                                    [t.data_ptr() for t in d_num], [t.data_ptr() for t in d_sum], d_had.data_ptr())
        torch.cuda.synchronize()
        del buf, buf4
