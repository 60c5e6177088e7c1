#!/usr/bin/env python3
"""bench.py - CU-decision CTUs/s at 1080p All-Intra (BASELINE.json's metric) on N B200s of one node.

A "step" is one pass of the hot path over one batch of P synthetic 1080p pictures: the per-picture
outlier/OBF feature pass (GPU pass 1 -> host TCM fit -> GPU pass 2, per-CU block sums, per-CTU source
Hadamard) plus the full rough-mode-decision enumeration (341 PUs x 35 modes per CTU, borders built
from a reconstruction plane).  Workload = BASELINE.json configs[1] (1920x1080 8-bit All-Intra).

  value      whole-job CTUs/s with inputs resident in HBM (cucd_dev_frames on torch's stream, CUDA events)
  e2e        the same pass through the host-buffer C-ABI call cuCUDecide_frames: pinned host planes in,
             every output back on the host, copies inside the timed region (wall clock around the calls)
  roofline   the RMD kernel (the one dominant launch of a step): algorithmic bytes / its event-timed duration
  cpu_baseline  the reference's own CPU functions (oracle/_ref/libhmref.so) or the oracle port on a bounded sample

`--impl reference` times the reference's CPU implementation of the same path on the host cores.
Multi-GPU: pictures shard across ranks (weak scaling, no collective on the data path).
"""
import argparse
import ctypes as C
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = "fast-cu-decision-hevc_b200"
METRIC = "cu_decision_ctus_per_s_1080p_all_intra"
ALGO_BYTES_PER_CTU = 72484          # SURVEY.md 8d: source 8192 + borders 16552 + cost tables 47740 (int16 samples)


def textured_plane(W, H, bit_depth, seed, t):
    """SURVEY.md 8d 'textured motion' luma: 8x8-blocky random field translated (2,1) px/frame + two
    sinusoids + uniform noise +-6, clipped to 8 bit (scaled with random LSBs for >8 bit)."""
    rng = np.random.default_rng(seed)
    field = rng.integers(0, 256, (H // 8 + 2 + 16, W // 8 + 2 + 32)).astype(np.float32)
    tex = np.kron(field, np.ones((8, 8), np.float32))[t % 64: t % 64 + H, (2 * t) % 128: (2 * t) % 128 + W]
    x = np.arange(W, dtype=np.float32)[None, :]
    y = np.arange(H, dtype=np.float32)[:, None]
    noise = np.random.default_rng(seed + 1000 + t).uniform(-6, 6, (H, W)).astype(np.float32)
    Y = 0.6 * tex + 30 + 20 * np.sin((x + 3 * t) / 37.0) + 15 * np.cos((y - 2 * t) / 29.0) + noise
    Y = np.clip(np.rint(Y), 0, 255).astype(np.int32)
    if bit_depth > 8:
        sh = bit_depth - 8
        Y = (Y << sh) + np.random.default_rng(seed + 2000 + t).integers(0, 1 << sh, (H, W))
    return Y.astype(np.int16)


def pseudo_recon(org, bit_depth, seed):
    o = org.astype(np.int32)
    pad = np.pad(o, 1, mode="edge")
    blur = (pad[:-2, 1:-1] + pad[2:, 1:-1] + pad[1:-1, :-2] + pad[1:-1, 2:] + 4 * o + 4) >> 3
    noise = np.random.default_rng(seed).integers(-2, 3, o.shape)
    return np.clip(blur + noise, 0, (1 << bit_depth) - 1).astype(np.int16)


# ---------------------------------------------------------------------------------------------------
# CPU reference arm / cpu_baseline
# ---------------------------------------------------------------------------------------------------
def load_cpu_checker():
    ref = os.path.join(ROOT, "oracle", "_ref", "libhmref.so")
    if os.path.exists(ref):
        lib = C.CDLL(ref)
        lib.hmref_init(8)
        return lib, "reference"
    so = os.path.join(ROOT, "oracle", "libcucd_oracle.so")
    if not os.path.exists(so):
        subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "libcucd_oracle.so"], check=True, capture_output=True)
    return C.CDLL(so), "port"


def _feature_pass(lib, kind, org, bd):
    """one picture through the reference's single-threaded feature pass (TEncSlice::getOutlierWithDCT)"""
    H, W = org.shape
    obf, outl, yc = np.zeros((H // 4, W // 4), np.int16), np.zeros((H, W), np.int16), np.zeros(16)
    vp = lambda a: C.c_void_p(a.ctypes.data)  # noqa: E731
    if kind == "reference":
        lib.hmref_outlier_frame(bd, vp(org), W, W, H, vp(obf), vp(outl))
    else:
        lib.oracle_outlier_frame(bd, vp(org), W, W, H, vp(obf), vp(outl), vp(yc))


def cpu_path_sample(lib, kind, pics, bit_depth, threads, ctus_per_pic_limit=None, feature_rows=None):
    """One CPU step: every picture in `pics` [(org, rec), ...] through the RMD enumeration (CTUs spread over
    `threads` host threads inside the reference driver) and through the per-picture feature pass.  The
    reference's feature pass is single-threaded and not re-entrant, so pictures run concurrently in
    forked child processes (up to `threads` of them) while the parent runs the RMD enumeration.
    Returns (ctus_per_s, seconds, ctus)."""
    H, W = pics[0][0].shape
    nctu_pic = ((W + 63) // 64) * ((H + 63) // 64)
    n_ctus = nctu_pic if ctus_per_pic_limit is None else min(nctu_pic, ctus_per_pic_limit)

    def vp(a):
        return C.c_void_p(a.ctypes.data)
    out = np.zeros((n_ctus, 341, 35), np.uint32)
    nproc = max(1, min(threads, len(pics)))
    sys.stdout.flush()
    t0 = time.perf_counter()
    def spawn(k):
        pid = os.fork()
        if pid == 0:
            try:
                devnull = os.open(os.devnull, os.O_WRONLY)
                os.dup2(devnull, 1)        # the reference prints diagnostics from its TCM fit
                for i in range(k, len(pics), nproc):
                    _feature_pass(lib, kind, pics[i][0] if feature_rows is None else np.ascontiguousarray(pics[i][0][:feature_rows]), bit_depth)
            finally:
                os._exit(0)
        return pid
    kids = [(k, spawn(k)) for k in range(nproc)]
    for org, rec in pics:
        if kind == "reference":
            lib.hmref_rmd_frame(bit_depth, 1, vp(org), W, vp(rec), W, W, H, 0, n_ctus, threads, vp(out))
        else:
            lib.oracle_rmd_frame(bit_depth, 1, vp(org), W, vp(rec), W, W, H, 0, n_ctus, vp(out))
    for k, pid in kids:
        _, status = os.waitpid(pid, 0)
        for _ in range(2):                 # the reference's feature pass has been seen to die once in a run on the GPU box: run that worker's pictures again
            if status == 0:
                break
            print(f"[bench] CPU feature-pass worker {k} ended with wait status {status}; retrying", file=sys.stderr)
            _, status = os.waitpid(spawn(k), 0)
        if status != 0:
            raise RuntimeError(f"a CPU feature-pass worker failed (wait status {status})")
    dt = time.perf_counter() - t0
    ctus = n_ctus * len(pics)
    return ctus / dt, dt, ctus


def cpu_me_sample(lib, kind, cur, refs_padded, pus, bit_depth, threads):
    """The inter part of one CPU step on `pus` [(x, y, size)]: per reference the whole +-64 SAD surface (the reference's own xGetSAD*
    through hmref_sad_surface, or the oracle port) and the 49-point sub-pel Hadamard table (oracle port of TComInterpolationFilter +
    xGetHADs - the reference has no separable entry point for it), PUs spread over `threads` host threads.  Returns seconds."""
    from concurrent.futures import ThreadPoolExecutor
    so = os.path.join(ROOT, "oracle", "libcucd_oracle.so")
    port = C.CDLL(so)
    R, M = ME_RANGE, ME_MARGIN
    H, W = cur.shape

    def one(pu):
        x, y, s = pu
        blk = np.ascontiguousarray(cur[y:y + s, x:x + s])
        out = np.empty((2 * R + 1) ** 2, np.uint32)
        o49 = np.empty(49, np.uint32)
        for rp in refs_padded:
            stride = rp.shape[1]
            base = C.c_void_p(rp.ctypes.data + 2 * ((y + M) * stride + x + M))
            sub = 1 if s > 8 else 0
            if kind == "reference":
                lib.hmref_sad_surface(bit_depth, C.c_void_p(blk.ctypes.data), s, s, s, base, stride, -R, R, -R, R, sub, C.c_void_p(out.ctypes.data))
            else:
                port.oracle_sad_surface(bit_depth, C.c_void_p(blk.ctypes.data), s, s, s, base, stride, -R, R, -R, R, sub, C.c_void_p(out.ctypes.data))
            port.oracle_subpel_surface(bit_depth, C.c_void_p(blk.ctypes.data), s, s, s, base, stride, 1, -1, 1, C.c_void_p(o49.ctypes.data))
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=max(1, threads)) as ex:
        list(ex.map(one, pus))
    return time.perf_counter() - t0


def cpu_reference_run_inter(args, steps, warmup):
    """Reference arm of the inter configurations on a bounded sample: the first four CTU rows of one picture through the intra path (as
    the All-Intra arm; the feature pass on those 256 picture rows) and through the ME part; CTU/s = CTUs / (intra seconds + ME seconds)."""
    lib, kind = load_cpu_checker()
    threads = os.cpu_count() or 1
    W, H, bd = args.width, args.height, args.bit_depth
    n_ctus = 4 * ((W + 63) // 64)
    cur = textured_plane(W, H, bd, 20261018, 1)
    recs = [pseudo_recon(textured_plane(W, H, bd, 20261018, t), bd, t) for t in (0, 2)][:args.refs]
    refs_padded = [np.ascontiguousarray(np.pad(r, ME_MARGIN, mode="edge")) for r in recs]
    ctus_per_row = (W + 63) // 64
    # PUs of the first n_ctus CTUs (raster order)
    pus = [(x, y, s) for (x, y, s) in inter_pus(W, H) if (y // 64) * ctus_per_row + x // 64 < n_ctus]
    vals, secs = [], 0.0
    for i in range(warmup + steps):
        _, dt_intra, _ = cpu_path_sample(lib, kind, [(cur, recs[0])], bd, threads, n_ctus, feature_rows=256)
        dt_me = cpu_me_sample(lib, kind, cur, refs_padded, pus, bd, threads)
        if i >= warmup:
            vals.append(n_ctus / (dt_intra + dt_me)); secs += dt_intra + dt_me
    desc = (f"{steps} steps x {n_ctus} CTUs (4 CTU rows) of one {W}x{H} picture: intra path + {len(pus)} PUs x {args.refs} reference(s) x {(2 * ME_RANGE + 1) ** 2} SAD candidates "
            f"(reference xGetSAD*) + 49-point sub-pel Hadamard (oracle port), {secs:.1f} s on {threads} thread(s)")
    return float(np.mean(vals)), {"value": float(np.mean(vals)), "unit": "CTU/s", "cores": threads, "kind": kind, "sample": desc}


def cpu_reference_run(args, steps, warmup, target_step_s=2.0):
    if args.refs:
        return cpu_reference_run_inter(args, steps, warmup)
    """The reference's CPU implementation of the path on all host threads: returns (mean CTU/s, dict)."""
    lib, kind = load_cpu_checker()
    threads = (os.cpu_count() or 1) if kind == "reference" else 1
    W, H, bd = args.width, args.height, args.bit_depth
    base = [(textured_plane(W, H, bd, 20261018, t), None) for t in range(2)]
    base = [(o, pseudo_recon(o, bd, t)) for t, (o, _) in enumerate(base)]
    if kind == "reference":
        rate, dt, _ = cpu_path_sample(lib, kind, base[:1], bd, threads)            # calibration picture
        n_pics = int(max(1, min(64, round(target_step_s / max(dt, 1e-3)))))
        limit = None
    else:                                                                         # scalar port: a slice of one picture
        n_pics, limit = 1, 48
    pics = [base[i % len(base)] for i in range(n_pics)]
    vals, secs, ctus = [], 0.0, 0
    for i in range(warmup + steps):
        v, dt, n = cpu_path_sample(lib, kind, pics, bd, threads, limit)
        if i >= warmup:
            vals.append(v); secs += dt; ctus += n
    desc = (f"{steps} steps x {n_pics} picture(s) of {W}x{H}" + (f" ({limit} CTUs each)" if limit else "") +
            f": RMD enumeration 341 PUs x 35 modes per CTU + feature pass, {ctus} CTUs in {secs:.1f} s on {threads} thread(s)")
    return float(np.mean(vals)), {"value": float(np.mean(vals)), "unit": "CTU/s", "cores": threads, "kind": kind, "sample": desc}


def run_reference(args, rank, world):
    if rank != 0:
        return
    t_all = time.perf_counter()
    value, base = cpu_reference_run(args, args.steps, args.warmup)
    ctus_per_step = args.pics * ((args.width + 63) // 64) * ((args.height + 63) // 64)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "CTU/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * ctus_per_step / value, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int32", "data": "synthetic", "config": workload_config(args), "cpu_baseline": base,
            "e2e": {"value": value, "unit": "CTU/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": time.perf_counter() - t_all}
    print(json.dumps(line))


# BASELINE.json configs[1..4] as bench workloads (configs[0] is the reference's own 416x240 CPU run: a parity-test case)
CONFIGS = {
    "ai1080p8": dict(width=1920, height=1080, bit_depth=8, pics=16, refs=0, label="BASELINE configs[1]: 1920x1080 8-bit All-Intra Main"),
    "ai2160p10": dict(width=3840, height=2160, bit_depth=10, pics=4, refs=0, label="BASELINE configs[2]: 3840x2160 10-bit All-Intra Main10"),
    "ldp1080p": dict(width=1920, height=1080, bit_depth=8, pics=1, refs=1, label="BASELINE configs[3]: 1920x1080 low-delay P Main, integer-ME SAD on the GPU, search range 64"),
    "ra1080p10": dict(width=1920, height=1080, bit_depth=10, pics=1, refs=2, label="BASELINE configs[4]: 1920x1080 Random Access GOP8 Main10 (one reference per list)"),
}
ME_RANGE = 64          # --SearchRange=64
ME_MARGIN = 80         # TComPicYuv margin: CTU + 16 (TComPicYuv.cpp:83-84)


DUMP_BUDGET_BYTES = 60 << 20


def dump_outputs(out_dir, arrays):
    """--dump-outputs: write each output of the timed path's last step as out_dir/<name>.npy, exact in float64 (float32 for
    16-bit outputs).  `arrays` maps name -> (device tensor, numpy dtype the tensor's bits hold).  An array larger than its share
    of DUMP_BUDGET_BYTES is reduced to a fixed sample: the sorted, de-duplicated flat indices drawn by default_rng(0), the same
    for every run of the same arguments, so that two builds can be compared output for output."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    cap = DUMP_BUDGET_BYTES // (8 * len(arrays))
    for name, (t, dtype) in arrays.items():
        flat = t.reshape(-1)
        if flat.numel() > cap:
            idx = np.unique(np.random.default_rng(0).integers(0, flat.numel(), cap))
            flat = flat[torch.from_numpy(idx).to(flat.device)]
        a = flat.cpu().numpy().view(dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32 if a.itemsize <= 2 else np.float64))


def inter_pus(W, H):
    """the square 2Nx2N PUs of every CU at depths 0..3 that lies inside the picture (85 per whole CTU): (x, y, size)"""
    pus = []
    for size in (64, 32, 16, 8):
        for y in range(0, H - size + 1, size):
            for x in range(0, W - size + 1, size):
                pus.append((x, y, size))
    return pus


def me_algo_bytes(pus):
    """SURVEY.md 8d: per PU cur w*h*2 + ref (w+2R)(h+2R)*2 + out (2R+1)^2*4"""
    R = ME_RANGE
    return sum(s * s * 2 + (s + 2 * R) * (s + 2 * R) * 2 + (2 * R + 1) ** 2 * 4 for _, _, s in pus)


def workload_config(args):
    which = args.label or "not a BASELINE configuration"
    if args.refs:
        npu = len(inter_pus(args.width, args.height))
        return {"workload": f"{args.width}x{args.height} {args.bit_depth}-bit ({which}): per picture the intra path (feature pass + RMD enumeration 341 PUs x 35 modes per CTU) "
                            f"plus, per reference picture ({args.refs}), the integer-ME SAD surface of every square PU of depths 0-3 ({npu} PUs, window +-{ME_RANGE} = "
                            f"{(2 * ME_RANGE + 1) ** 2} candidates each, FEN row sub-sampling) and its 49-point quarter-pel Hadamard refinement; {args.pics} picture(s) per step per GPU",
                "pictures_per_step_per_gpu": args.pics, "ctus_per_picture": ((args.width + 63) // 64) * ((args.height + 63) // 64), "reference_pictures": args.refs,
                "me_pus_per_picture": npu,
                "l2_policy": f"inputs larger than L2: a step writes {npu * (2 * ME_RANGE + 1) ** 2 * 4 * args.refs / 1e9:.2f} GB of SAD surfaces",
                "parallelism": f"pictures sharded over {args.gpus} GPU(s), no collective"}
    enum = ("FORK-AWARE (Testing-picture) enumeration - NOT the headline workload: Num_OBF first, then only the PUs TEncCu::xCompressCU still reaches with Skip2Nx2N on at "
            "every depth and TerminateCU on at depths 0-2; pruned PUs carry CUCD_COST_PRUNED" if getattr(args, "fork_aware", False) else "full intra RMD enumeration")
    return {"workload": f"{args.width}x{args.height} {args.bit_depth}-bit All-Intra ({which}): {enum} "
                        f"341 PUs x 35 modes per CTU + OBF/outlier feature pass, {args.pics} pictures per step per GPU",
            "pictures_per_step_per_gpu": args.pics, "ctus_per_picture": ((args.width + 63) // 64) * ((args.height + 63) // 64),
            "l2_policy": "inputs larger than L2: one step reads 2 planes x pictures and writes the cost tables (> 126 MB) before any reuse",
            "parallelism": f"pictures sharded over {args.gpus} GPU(s), no collective"}


# ---------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(device)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            pass

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        out, _ = self.proc.communicate(timeout=10)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in out.splitlines():
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "samples": len(sm),
                "reasons": sorted(reasons)}


def bind_to_gpu_numa_node(local_rank):
    """Run this rank (and allocate its pinned host buffers: first touch) on the CPUs of the NUMA node the GPU hangs off, as a
    production host would place an encoder instance.  Pinned buffers on the remote socket cost ~20 % of the PCIe D2H rate, and
    the host-buffer call is D2H bound.  Returns a description for the JSON line; any failure leaves the affinity untouched."""
    if os.environ.get("BENCH_NO_NUMA_BIND"):
        return "disabled"
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(local_rank)],
                           capture_output=True, text=True, timeout=20).stdout.strip().lower()
        bus = q[-12:] if len(q) >= 12 else q           # 00000000:1B:00.0 -> 0000:1b:00.0
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        n_nodes = len([d for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit()])
        if node < 0 or n_nodes < 2:
            return f"single node (numa_node={node}, nodes={n_nodes})"
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return f"node {node}: no allowed CPUs"
        os.sched_setaffinity(0, cpus)
        return f"node {node} of {n_nodes} ({len(cpus)} CPUs)"
    except Exception as e:   # noqa: BLE001
        return f"unavailable ({type(e).__name__})"


# ---------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------
def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    cucd = importlib.import_module(PKG)
    no_gpu = "bench.py: no CUDA device - the product has no CPU path (use --impl reference for the CPU arm)"
    if not os.path.exists("/dev/nvidiactl") and not torch.cuda.is_available():      # a GPU-less box fails at once; on a GPU box CUDA is first touched below
        raise SystemExit(no_gpu)
    # The CPU baseline forks worker processes (the reference's feature pass is not re-entrant): it runs BEFORE this process creates
    # its CUDA context, page-locked buffers and worker threads - a fork after that is not safe.
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not args.fork_aware:
        _, cpu_baseline = cpu_reference_run(args, steps=3, warmup=1, target_step_s=3.0)
    if not torch.cuda.is_available():
        raise SystemExit(no_gpu)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # NCCL's version banner must not share stdout with the JSON line
        dist.init_process_group("nccl", device_id=dev)

    W, H, bd, P = args.width, args.height, args.bit_depth, args.pics
    # host threads of the TCM fits: cores / ranks, so that 8 ranks do not oversubscribe a 32-core host
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    host_threads = max(1, min(8, cores // max(1, world)))
    eng = cucd.Engine(W, H, bit_depth=bd, device=local_rank, max_pictures=P, host_threads=host_threads)
    nctu = eng.ctus_per_pic
    pitch = (W + 63) // 64 * 64
    FORK_SW = ((1, 1, 1, 1), (1, 1, 1, 0))      # tests/golden/fork_ai8.npz: what SetDecisionSwitch left after the verify picture of a real encode
    if args.fork_aware:
        eng.set_decision_switches(1, *FORK_SW)
    # the job is a clip of world x P pictures per step; ranks deal its pictures out round-robin (no schedule coupling between the
    # synthetic pictures: fast-cu-decision-hevc_b200/sharding.py shard_independent) - weak scaling, P pictures per rank and step
    my_pictures = list(cucd.shard_independent(world * P, rank, world))
    orgs = [textured_plane(W, H, bd, 20261018, t) for t in my_pictures]
    recs = [pseudo_recon(o, bd, t) for t, o in enumerate(orgs)]

    def pinned(shape, dtype):
        tdt = {np.int16: torch.int16, np.int32: torch.int32, np.uint32: torch.int32, np.float64: torch.float64, np.uint8: torch.uint8}[dtype]
        t = torch.empty(shape, dtype=tdt, pin_memory=True)
        pinned.keep.append(t)
        a = t.numpy()
        return a.view(np.uint32) if dtype is np.uint32 else a
    pinned.keep = []

    # host side of the e2e call: 8-bit content travels as bytes (cuCUDecide_frames_u8), 10-bit as HM's Pel; outputs in the
    # narrowest exact formats (packed cost tables, byte OBF / Outlier planes)
    hdt = np.uint8 if bd == 8 else np.int16
    h_org = [pinned((H, W), hdt) for _ in range(P)]
    h_rec = [pinned((H, W), hdt) for _ in range(P)]
    for p in range(P):
        h_org[p][:] = orgs[p]; h_rec[p][:] = recs[p]
    h_outs = [eng.alloc_frame_out(True, pinned_alloc=pinned, packed=True, narrow=True) for _ in range(P)]

    # ---- device-resident buffers -------------------------------------------------------------------
    d_org = torch.zeros((P, H, pitch), dtype=torch.int16, device=dev)
    d_rec = torch.zeros((P, H, pitch), dtype=torch.int16, device=dev)
    for p in range(P):
        d_org[p, :, :W] = torch.from_numpy(orgs[p]).to(dev)
        d_rec[p, :, :W] = torch.from_numpy(recs[p]).to(dev)
    d_cost = torch.empty((P, nctu, 341, 35), dtype=torch.int32, device=dev)
    d_obf = torch.empty((P, H // 4, W // 4), dtype=torch.int16, device=dev)
    d_outl = torch.empty((P, H, W), dtype=torch.int16, device=dev)
    d_num = [torch.empty((P,) + eng.cu_grid(d), dtype=torch.int32, device=dev) for d in range(4)]
    d_sum = [torch.empty((P,) + eng.cu_grid(d), dtype=torch.int32, device=dev) for d in range(4)]
    d_had = torch.empty((P, nctu), dtype=torch.int32, device=dev)
    d_out = {"obf": d_obf.data_ptr(), "outlier": d_outl.data_ptr(), "num_obf": [t.data_ptr() for t in d_num],
             "n_outlier": [t.data_ptr() for t in d_sum], "ctu_src_had": d_had.data_ptr(), "rmd_cost": d_cost.data_ptr()}
    stream = torch.cuda.current_stream().cuda_stream

    def dev_steps(n):
        """n steps through the split call: the host fit of step i runs while the GPU is already on the RMD kernel of step i+1
        (cucd_dev_frames_begin / _end, at most two steps in flight); every step is complete when the stream drains."""
        for i in range(n):
            eng.dev_frames(stream, P, d_org.data_ptr(), H * pitch, pitch, d_rec.data_ptr(), H * pitch, pitch, d_out, begin_only=True)
            if i > 0:
                eng.dev_frames_end()
        eng.dev_frames_end()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- kernel-resident timing ----------------------------------------------------------------------
    # nvidia-smi needs a few hundred ms to start: launch the sampler before the warm-up so that it is already reporting when the
    # (tens of ms long) timed region runs, and keep it running through the end-to-end region, which is timed under load too
    clocks = ClockSampler(local_rank)
    dev_steps(max(args.warmup, 3))
    barrier()
    l0 = eng.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    dev_steps(args.steps)
    e1.record()
    barrier()
    launches = eng.launch_count - l0
    dev_ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"rmd_cost": (d_cost, np.uint32), "obf": (d_obf, np.int16), "outlier": (d_outl, np.int16),
                                         "ctu_src_had": (d_had, np.int32), **{f"num_obf{d}": (t, np.int32) for d, t in enumerate(d_num)},
                                         **{f"n_outlier{d}": (t, np.int32) for d, t in enumerate(d_sum)}})
    rmd_ms, n_timed = eng.rmd_kernel_time_ms(min(args.steps, 64))

    # ---- end to end through the host-buffer ABI -------------------------------------------------------
    # One encoder instance = one handle, calls are synchronous (HM is single-threaded).  The deployment the
    # reference implies is several encoder instances per GPU (SURVEY.md 8b/8f), so the headline e2e figure runs
    # `--e2e-instances` handles from as many host threads (each with its own pinned buffers; ctypes drops the GIL
    # inside the call): while one instance drains its cost tables over PCIe the other uploads and computes.
    def e2e_run(engines, outs_list, steps, planes=None):
        import threading
        po, pr = planes or (h_org, h_rec)
        def work(e, o):
            for _ in range(steps):
                e.frames(po, pr, o)
        ths = [threading.Thread(target=work, args=(e, o)) for e, o in zip(engines, outs_list)]
        t0 = time.perf_counter()
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    n_inst = max(1, args.e2e_instances)
    inst_threads = max(1, host_threads // n_inst)
    engines = [eng] + [cucd.Engine(W, H, bit_depth=bd, device=local_rank, max_pictures=P, host_threads=inst_threads) for _ in range(n_inst - 1)]
    if args.fork_aware:
        for e in engines[1:]:
            e.set_decision_switches(1, *FORK_SW)
    outs_list = [h_outs] + [[e.alloc_frame_out(True, pinned_alloc=pinned, packed=True, narrow=True) for _ in range(P)] for e in engines[1:]]
    e2e_steps = max(1, min(args.steps, 5))
    e2e_run(engines[:1], outs_list[:1], max(1, min(args.warmup, 2)))
    barrier()
    e2e_single_s = e2e_run(engines[:1], outs_list[:1], e2e_steps)
    if n_inst > 1:
        e2e_run(engines, outs_list, 1)
        barrier()
        e2e_s = e2e_run(engines, outs_list, e2e_steps)
    else:
        e2e_s = e2e_single_s
    clk = clocks.stop()
    h2d = 2 * P * W * H * np.dtype(hdt).itemsize
    d2h = sum(int(a.nbytes) for o in h_outs for a in o.values())

    # ---- the documented integration (INTEGRATION.md): HM's own planes - Pel = int16, stride W + 160, xMalloc'ed (pageable,
    #      TComPicYuv.cpp:97) - and plain caller-owned output buffers, one encoder instance.  (a) as they are, (b) page-locked once
    #      through cucd_pin_host_buffer / auto_pin_host, as a maintainer would do at TComPicYuv::create.  Rank 0 only. ----------
    hm_e2e = None
    if rank == 0 and not args.no_hm_planes and not args.fork_aware:
        def hm_plane(a):
            buf = np.zeros((H + 160, W + 160), np.int16)
            buf[80:80 + H, 80:80 + W] = a
            return buf[80:80 + H, 80:80 + W]
        hm_org = [hm_plane(o) for o in orgs]
        hm_rec = [hm_plane(r) for r in recs]
        hm_e2e = {"planes": "int16, stride W+160, heap memory (HM TComPicYuv layout); outputs in heap memory, packed / byte formats", "instances": 1}
        for key, auto in (("pageable", 0), ("page_locked_once", 1)):
            with cucd.Engine(W, H, bit_depth=bd, device=local_rank, max_pictures=P, host_threads=host_threads, auto_pin_host=auto) as e:
                outs = [e.alloc_frame_out(True, packed=True, narrow=True) for _ in range(P)]
                e2e_run([e], [outs], 2, (hm_org, hm_rec))                 # warm-up (and, with auto_pin_host, the one-time registration)
                dt = e2e_run([e], [outs], 3, (hm_org, hm_rec))
                hm_e2e[key] = {"value": P * nctu * 3 / dt, "unit": "CTU/s", "ms_per_step": 1e3 * dt / 3}
                ok_hm = bool(np.array_equal(outs[0]["rmd_cost_packed"], h_outs[0]["rmd_cost_packed"]) and np.array_equal(outs[P - 1]["obf_u8"], h_outs[P - 1]["obf_u8"]))
                hm_e2e[key]["agrees_with_pinned_run"] = ok_hm

    # spot-check that both paths produced the same tables (device-resident vs host-buffer)
    same = all(bool(np.array_equal(d_cost[p].cpu().numpy().view(np.uint32), cucd.unpack_costs(h_outs[p]["rmd_cost_packed"]))) for p in (0, P - 1))

    # ---- reduce over ranks ---------------------------------------------------------------------------
    t = torch.tensor([dev_ms, e2e_s, rmd_ms, e2e_single_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_s, rmd_ms, e2e_single_s = [float(v) for v in t.tolist()]
    ctus_step_gpu = P * nctu
    value = world * ctus_step_gpu * args.steps / (dev_ms * 1e-3)
    e2e_value = world * n_inst * ctus_step_gpu * e2e_steps / e2e_s
    e2e_single = world * ctus_step_gpu * e2e_steps / e2e_single_s

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    else:
        peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
    achieved = ALGO_BYTES_PER_CTU * ctus_step_gpu / (rmd_ms * 1e-3) / 1e9
    kernel_name = "rmd_frame_kernel" if os.environ.get("CUCD_RMD_PATH") == "alu" else ("rmd_frame_tc2_kernel" if bd == 8 else "rmd_frame_tc3_kernel")
    # DRAM bytes per launch: dram__bytes_read + dram__bytes_write per CTU of the committed ncu --set full capture of the SAME kernel
    # (profiles/r02/rmd_traffic.json, cold-cache 2040-CTU launches) x the CTUs of this launch; null when that kernel has no capture
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "r02", "rmd_traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        if kernel_name in tj:
            traffic = float(tj[kernel_name]["dram_bytes_per_ctu"]) * ctus_step_gpu
            traffic_src = "profiles/r02/rmd_traffic.json: %.0f B/CTU measured by ncu on a %d-CTU launch, scaled to this launch; cost-table lines still dirty in L2 at kernel end are not counted" % (
                tj[kernel_name]["dram_bytes_per_ctu"], tj[kernel_name]["ctus_per_launch"])
    roofline = {"bound": "hbm", "kernel": kernel_name, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src, "launch_ms": rmd_ms, "launches_timed": n_timed, "algorithmic_bytes_per_launch": ALGO_BYTES_PER_CTU * ctus_step_gpu,
                "peak_source": peak_src,
                "note": "launch_ms is the CUDA-event window around the RMD launch on the caller's stream; the small feature kernels run beside it on a high-priority stream and take part of that window. RMD is compute bound by construction (~140 int-op/B, SURVEY.md 8d): predictions and Hadamard run on tcgen05 (kind::i8 for 8-bit content, kind::f16 with exact integer operands for 9/10-bit content), "
                        "the epilogues on the integer ALU; the HBM fraction is small; see profiles/ for pipe utilisation"}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "CTU/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "int32", "data": "synthetic", "config": workload_config(args), "clocks": clk,
                "e2e": {"value": e2e_value, "unit": "CTU/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                        "ms_per_step": 1e3 * e2e_s / (e2e_steps * n_inst), "instances_per_gpu": n_inst,
                        "single_instance_value": e2e_single, "single_instance_ms_per_step": 1e3 * e2e_single_s / e2e_steps,
                        "api": ("cuCUDecide_frames_u8 (8-bit content as bytes)" if bd == 8 else "cuCUDecide_frames (int16 planes)") +
                               ": pinned host planes in, every output back on the host in its narrowest exact format",
                        "outputs_copied": sorted(h_outs[0].keys()), "hm_layout_planes": hm_e2e,
                        "host_numa_binding": numa, "host_threads_per_handle": host_threads},
                "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu_baseline,
                "paths_agree": same}
        if args.fork_aware:
            t0 = d_cost[0].cpu().numpy().view(np.uint32)[:, :, 0]
            line["fork_aware"] = {"label": "separate line, not the headline", "skip2Nx2N": FORK_SW[0], "terminateCU": FORK_SW[1],
                                  "pus_evaluated_fraction_picture0": float(((t0 != 0xFFFFFFFE) & (t0 != 0xFFFFFFFF)).sum() / max(1, (t0 != 0xFFFFFFFF).sum()))}
            line["cpu_baseline"] = None        # the CPU arm enumerates everything: not comparable with this line
        print(json.dumps(line))
    eng.close()
    if world > 1:
        dist.destroy_process_group()


def run_inter(args, rank, world, local_rank):
    """BASELINE configs[3] / [4]: the CU-decision cost path of an inter picture - the intra path of the picture plus, per reference
    picture, integer-ME SAD surfaces and quarter-pel refinement tables of every square PU.  value: everything resident in HBM
    (cucd_dev_frames + cucd_dev_me_sad_surface + cucd_dev_me_subpel_cost on torch's stream, CUDA events); e2e: the host-buffer
    calls (cuCUDecide_frames, cucd_set_cur/ref_picture, cucd_me_sad_surface, cucd_me_subpel_cost), planes up and every table down."""
    import torch
    import torch.distributed as dist
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    cucd = importlib.import_module(PKG)
    no_gpu = "bench.py: no CUDA device - the product has no CPU path (use --impl reference for the CPU arm)"
    if not os.path.exists("/dev/nvidiactl") and not torch.cuda.is_available():      # a GPU-less box fails at once; on a GPU box CUDA is first touched below
        raise SystemExit(no_gpu)
    cpu_baseline = None                     # before the CUDA context exists (the CPU arm forks)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        _, cpu_baseline = cpu_reference_run(args, steps=2, warmup=1)
    if not torch.cuda.is_available():
        raise SystemExit(no_gpu)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    W, H, bd, P, NR = args.width, args.height, args.bit_depth, args.pics, args.refs
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    host_threads = max(1, min(8, cores // max(1, world)))
    eng = cucd.Engine(W, H, bit_depth=bd, device=local_rank, max_pictures=1, host_threads=host_threads)
    nctu, pitch, R, M = eng.ctus_per_pic, (W + 63) // 64 * 64, ME_RANGE, ME_MARGIN
    # per picture of the step: the current picture (t = 1 + 3p), its reconstruction stand-in, NR reference reconstructions (t - 1, t + 1)
    seed = 20261018 + 97 * rank
    curs = [textured_plane(W, H, bd, seed, 1 + 3 * p) for p in range(P)]
    recs = [pseudo_recon(c, bd, p) for p, c in enumerate(curs)]
    refs = [[np.ascontiguousarray(np.pad(pseudo_recon(textured_plane(W, H, bd, seed, 3 * p + (0, 2)[k]), bd, 10 + k), M, mode="edge")) for k in range(NR)] for p in range(P)]
    pus = inter_pus(W, H)
    n_pu, cand = len(pus), (2 * R + 1) ** 2
    me_arr, me_n, me_total = [], 0, 0
    for k in range(NR):
        arr, me_n, me_total = cucd.Engine.me_descs([dict(x=x, y=y, w=s, h=s, ref_idx=k, left=-R, right=R, top=-R, bottom=R, sub_shift=1 if s > 8 else 0) for x, y, s in pus])
        me_arr.append(arr)
    sp_arr = [cucd.Engine.subpel_descs([dict(x=x, y=y, w=s, h=s, ref_idx=k, mvx=1, mvy=-1, use_hadamard=1) for x, y, s in pus])[0] for k in range(NR)]

    # ---- device-resident buffers ---------------------------------------------------------------------
    d_org = torch.zeros((1, H, pitch), dtype=torch.int16, device=dev); d_rec = torch.zeros_like(d_org)
    d_cost = torch.empty((1, nctu, 341, 35), dtype=torch.int32, device=dev)
    d_obf = torch.empty((1, H // 4, W // 4), dtype=torch.int16, device=dev); d_outl = torch.empty((1, H, W), dtype=torch.int16, device=dev)
    d_had = torch.empty((1, nctu), dtype=torch.int32, device=dev)
    d_out = {"obf": d_obf.data_ptr(), "outlier": d_outl.data_ptr(), "ctu_src_had": d_had.data_ptr(), "rmd_cost": d_cost.data_ptr()}
    d_sad = [torch.empty(me_total, dtype=torch.int32, device=dev) for _ in range(NR)]
    d_sub = [torch.empty((n_pu, 49), dtype=torch.int32, device=dev) for _ in range(NR)]
    stream = torch.cuda.current_stream().cuda_stream
    me_ev = []

    def resident_picture(p):
        """a picture and its references become resident (untimed for `value`: inputs are in HBM when the timed region starts)"""
        d_org[0, :, :W] = torch.from_numpy(curs[p]).to(dev); d_rec[0, :, :W] = torch.from_numpy(recs[p]).to(dev)
        eng.set_cur_picture(curs[p])
        for k in range(NR):
            eng.set_ref_picture(k, refs[p][k], M, M)

    def dev_step(timed):
        eng.dev_frames(stream, 1, d_org.data_ptr(), H * pitch, pitch, d_rec.data_ptr(), H * pitch, pitch, d_out)
        for k in range(NR):
            if timed:
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
            eng.dev_me_sad_surface(stream, me_arr[k], me_n, d_sad[k].data_ptr())
            if timed:
                b.record(); me_ev.append((a, b))
            eng.dev_me_subpel_cost(stream, sp_arr[k], me_n, d_sub[k].data_ptr())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # `pics` pictures per step: the same resident picture is processed P times per step (P = 1 by default) - uploading between
    # the timed calls would turn `value` into an e2e figure
    resident_picture(0)
    clocks = ClockSampler(local_rank)
    for _ in range(max(args.warmup, 3)):
        for _ in range(P):
            dev_step(False)
    barrier()
    l0 = eng.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        for _ in range(P):
            dev_step(True)
    e1.record()
    barrier()
    launches = eng.launch_count - l0
    dev_ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"rmd_cost": (d_cost, np.uint32), "obf": (d_obf, np.int16), "outlier": (d_outl, np.int16),
                                         "ctu_src_had": (d_had, np.int32), **{f"me_sad_ref{k}": (d_sad[k], np.uint32) for k in range(NR)},
                                         **{f"me_subpel_ref{k}": (d_sub[k], np.uint32) for k in range(NR)}})
    me_ms = float(np.mean([a.elapsed_time(b) for a, b in me_ev]))

    # ---- end to end: host planes up, every table down ---------------------------------------------------
    def pinned(shape, dtype):
        tdt = {np.int16: torch.int16, np.int32: torch.int32, np.uint32: torch.int32, np.float64: torch.float64, np.uint8: torch.uint8}[dtype]
        t = torch.empty(shape, dtype=tdt, pin_memory=True)
        pinned.keep.append(t)
        a = t.numpy()
        return a.view(np.uint32) if dtype is np.uint32 else a
    pinned.keep = []
    hdt = np.uint8 if bd == 8 else np.int16
    h_cur = [pinned((H, W), hdt) for _ in range(P)]; h_rec = [pinned((H, W), hdt) for _ in range(P)]
    h_cur16 = [pinned((H, W), np.int16) for _ in range(P)]
    h_refs = [[pinned(refs[p][k].shape, np.int16) for k in range(NR)] for p in range(P)]
    for p in range(P):
        h_cur[p][:] = curs[p]; h_rec[p][:] = recs[p]; h_cur16[p][:] = curs[p]
        for k in range(NR):
            h_refs[p][k][:] = refs[p][k]
    h_out = eng.alloc_frame_out(True, pinned_alloc=pinned, packed=True, narrow=True)
    h_sad = pinned((me_total,), np.uint32)              # one surface block, reused per reference (an encoder consumes it before the next)
    h_sub = pinned((n_pu, 49), np.uint32)

    def e2e_step():
        for p in range(P):
            eng.frames([h_cur[p]], [h_rec[p]], [h_out])
            eng.set_cur_picture(h_cur16[p])
            for k in range(NR):
                eng.set_ref_picture(k, h_refs[p][k], M, M)
                eng.me_sad_surface_raw(me_arr[k], me_n, h_sad)
                eng.me_subpel_cost_raw(sp_arr[k], me_n, h_sub)
    e2e_steps = max(1, min(args.steps, 3))
    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    clk = clocks.stop()
    h2d = P * (2 * W * H * np.dtype(hdt).itemsize + W * H * 2 + NR * int(refs[0][0].nbytes))
    d2h = P * (sum(int(a.nbytes) for a in h_out.values()) + NR * (int(h_sad.nbytes) + int(h_sub.nbytes)))
    # the two paths agree (last reference of the last picture)
    resident_picture(P - 1)
    dev_step(False)
    torch.cuda.synchronize()
    same = bool(np.array_equal(d_sad[NR - 1].cpu().numpy().view(np.uint32), h_sad) and np.array_equal(d_sub[NR - 1].cpu().numpy().view(np.uint32), h_sub) and
                np.array_equal(d_cost[0].cpu().numpy().view(np.uint32), cucd.unpack_costs(h_out["rmd_cost_packed"])))

    t = torch.tensor([dev_ms, e2e_s, me_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_s, me_ms = [float(v) for v in t.tolist()]
    ctus_step_gpu = P * nctu
    value = world * ctus_step_gpu * args.steps / (dev_ms * 1e-3)
    e2e_value = world * ctus_step_gpu * e2e_steps / e2e_s
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    else:
        peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
    algo = me_algo_bytes(pus)
    achieved = algo / (me_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": "me_sad_dy_kernel<u8>" if bd == 8 else "me_sad_dy_kernel<s16>", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": None, "launch_ms": me_ms, "launches_timed": len(me_ev), "algorithmic_bytes_per_launch": algo, "peak_source": peak_src,
                "note": "the dominant launch of an inter step: one SAD surface call per reference = the dy-lane kernel (tiles M / E of csrc/me_core.cuh) "
                        "plus the dx-lane kernel for the last row of the window (CUDA events on the launching stream around the "
                        "call; includes the upload of its job records).  Algorithmic bytes per PU = source + reference window + surface (SURVEY.md 8d); "
                        f"the work is {(2 * ME_RANGE + 1) ** 2} candidates x w x h absolute differences per PU: integer-ALU bound (VABSDIFF4), see profiles/"}
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "CTU/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "int32", "data": "synthetic", "config": workload_config(args), "clocks": clk,
                "e2e": {"value": e2e_value, "unit": "CTU/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                        "ms_per_step": 1e3 * e2e_s / e2e_steps, "instances_per_gpu": 1,
                        "api": "cuCUDecide_frames(_u8) + cucd_set_cur_picture / cucd_set_ref_picture + cucd_me_sad_surface + cucd_me_subpel_cost: pinned host planes in, "
                               "cost tables, feature planes, every SAD surface and refinement table back on the host",
                        "host_numa_binding": numa},
                "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu_baseline, "paths_agree": same}
        print(json.dumps(line))
    eng.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="ai1080p8", choices=sorted(CONFIGS), help="BASELINE.json workload (default: configs[1], the one the metric is quoted on)")
    ap.add_argument("--pics", type=int, default=None, help="pictures per step per GPU (default: the configuration's)")
    ap.add_argument("--width", type=int, default=None)
    ap.add_argument("--height", type=int, default=None)
    ap.add_argument("--bit-depth", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-hm-planes", action="store_true", help="skip the pageable / page-locked HM-layout e2e measurement")
    ap.add_argument("--fork-aware", action="store_true",
                    help="SEPARATE, labelled line (never the headline): Testing-picture mode of the fork - the frame calls prune the PUs the encoder's "
                         "early decisions would skip (cucd_set_decision_switches; switches as a real 416x240 encode held them: Skip2Nx2N on at every depth, "
                         "TerminateCU on at depths 0-2)")
    ap.add_argument("--e2e-instances", type=int, default=2, help="encoder instances (handles + host threads) per GPU in the e2e measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (rank 0's device-resident outputs) as DIR/<name>.npy, "
                         "float32/float64, at most 60 MiB in all (larger arrays as a fixed seeded sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    cfg = CONFIGS[args.config]
    custom = any(v is not None for v in (args.width, args.height, args.bit_depth))
    args.width, args.height = args.width or cfg["width"], args.height or cfg["height"]
    args.bit_depth, args.pics, args.refs = args.bit_depth or cfg["bit_depth"], args.pics or cfg["pics"], cfg["refs"]
    args.label = None if custom else cfg["label"]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    args.gpus = world if world > 1 else args.gpus
    if args.refs:
        run_inter(args, rank, world, local_rank)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
