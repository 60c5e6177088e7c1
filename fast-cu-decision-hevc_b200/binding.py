"""ctypes binding of include/cucudecide.h (one Python method per C entry point).

Argument meaning follows the header, which in turn cites the reference call site each entry point
replaces.  numpy arrays go in and out for the host-buffer API; the ``dev_*`` methods take raw device
pointers (ints) and a CUDA stream handle so that callers holding data in HBM (bench.py through
torch) can launch the kernels on their own stream.
"""
import ctypes as C
import os
import re

import numpy as np

NUM_MODES = 35
PUS_PER_CTU = 341
COST_NOT_INSIDE, COST_PRUNED = 0xFFFFFFFF, 0xFFFFFFFE     # table codes (CUCD_COST_NOT_INSIDE / CUCD_COST_PRUNED)
PACKED_WIDE_PUS = 21                     # CUCD_PACKED_WIDE_PUS: PUs 0..20 stay uint32
PACKED_U16_PUS = 64                      # CUCD_PACKED_U16_PUS: the 8x8 PUs as uint16
PACKED_U16_OFFSET = PACKED_WIDE_PUS * 35 * 4
PACKED_B13_OFFSET = PACKED_U16_OFFSET + PACKED_U16_PUS * 35 * 2
PACKED_CTU_BYTES = PACKED_B13_OFFSET + 256 * 35 * 13 // 8   # CUCD_PACKED_CTU_BYTES = 21980


def unpack_costs(packed):
    """(nCtu, PACKED_CTU_BYTES) uint8 packed CTU tables (cucd_frame_out.rmd_cost_packed) -> (nCtu, 341, 35) uint32,
    a numpy restatement of cucd_unpack_costs() (uint32 | uint16 | 13-bit little-endian bit stream)."""
    packed = np.ascontiguousarray(packed, np.uint8).reshape(-1, PACKED_CTU_BYTES)
    n = packed.shape[0]
    out = np.empty((n, PUS_PER_CTU, NUM_MODES), np.uint32)
    out[:, :PACKED_WIDE_PUS] = packed[:, :PACKED_U16_OFFSET].copy().view(np.uint32).reshape(n, PACKED_WIDE_PUS, NUM_MODES)
    mid = packed[:, PACKED_U16_OFFSET:PACKED_B13_OFFSET].copy().view(np.uint16).reshape(n, PACKED_U16_PUS, NUM_MODES)
    out[:, PACKED_WIDE_PUS:PACKED_WIDE_PUS + PACKED_U16_PUS] = np.where(mid >= 0xFFFE, mid.astype(np.uint32) | np.uint32(0xFFFF0000), mid.astype(np.uint32))
    # 8 values = 13 bytes = 104 bits
    grp = packed[:, PACKED_B13_OFFSET:].reshape(n, -1, 13).astype(np.uint64)
    lo = sum(grp[:, :, k] << np.uint64(8 * k) for k in range(8))
    hi = sum(grp[:, :, 8 + k] << np.uint64(8 * k) for k in range(5))
    vals = np.empty(grp.shape[:2] + (8,), np.uint32)
    for k in range(8):
        bit = 13 * k
        if bit + 13 <= 64:
            v = (lo >> np.uint64(bit)) & np.uint64(0x1FFF)
        elif bit >= 64:
            v = (hi >> np.uint64(bit - 64)) & np.uint64(0x1FFF)
        else:
            v = ((lo >> np.uint64(bit)) | (hi << np.uint64(64 - bit))) & np.uint64(0x1FFF)
        vals[:, :, k] = v.astype(np.uint32)
    small = vals.reshape(n, 256, NUM_MODES)
    out[:, PACKED_WIDE_PUS + PACKED_U16_PUS:] = np.where(small >= 0x1FFE, small | np.uint32(0xFFFFE000), small)
    return out


HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libcucudecide.so")
HEADER_PATH = os.path.join(os.path.dirname(HERE), "include", "cucudecide.h")

_i16p = C.POINTER(C.c_int16)
_i32p = C.POINTER(C.c_int32)
_u32p = C.POINTER(C.c_uint32)
_f64p = C.POINTER(C.c_double)


class CucdError(RuntimeError):
    pass


class _Config(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("width", "height", "bit_depth", "ctu_size", "max_depth", "strong_intra_smoothing",
                                       "device", "max_pictures", "host_threads", "auto_pin_host")]


class _FrameOut(C.Structure):
    _fields_ = [("obf", _i16p), ("outlier", _i16p), ("yc", _f64p), ("num_obf", _i32p * 4), ("n_outlier", _i32p * 4),
                ("ctu_src_had", _i32p), ("rmd_cost", _u32p), ("rmd_cost_packed", C.POINTER(C.c_uint8)),
                ("obf_u8", C.POINTER(C.c_uint8)), ("outlier_u8", C.POINTER(C.c_uint8))]


class _DevOut(C.Structure):
    _fields_ = [("obf", C.c_void_p), ("outlier", C.c_void_p), ("num_obf", C.c_void_p * 4), ("n_outlier", C.c_void_p * 4),
                ("ctu_src_had", C.c_void_p), ("rmd_cost", C.c_void_p)]


class _PuDesc(C.Structure):
    _fields_ = [("log2_size", C.c_uint8), ("reserved", C.c_uint8 * 3)]


class _MeDesc(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("x", "y", "w", "h", "ref_idx", "left", "right", "top", "bottom", "sub_shift")]


class _SubpelDesc(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("x", "y", "w", "h", "ref_idx", "mvx", "mvy", "use_hadamard")]


class _McDesc(C.Structure):
    _fields_ = [("x", C.c_int), ("y", C.c_int), ("w", C.c_int), ("h", C.c_int), ("ref_idx", C.c_int * 2), ("mvx", C.c_int * 2), ("mvy", C.c_int * 2),
                ("use_hadamard", C.c_int)]


class _TuDesc(C.Structure):
    _fields_ = [("log2_size", C.c_uint8), ("mode", C.c_uint8), ("qp", C.c_int8), ("flags", C.c_uint8)]


TU_INTRA_SLICE, TU_SIGN_HIDING = 1, 2


class _CuDesc(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("x", "y", "log2_size")]


TMV_FEATURES = 5 * 26


def declared_symbols():
    """Every function name include/cucudecide.h declares."""
    text = open(HEADER_PATH).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(cucd_[a-z_0-9]+|cuCUDecide_[a-z]+)\s*\(", text)))


_lib = None


def load_library():
    """Load libcucudecide.so (built in-tree by __graft_entry__.build / make). Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CucdError(f"{LIB_PATH} is missing - run `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    lib.cucd_last_error.restype = C.c_char_p
    lib.cucd_last_error.argtypes = [C.c_void_p]
    lib.cucd_launch_count.restype = C.c_longlong
    lib.cucd_launch_count.argtypes = [C.c_void_p]
    lib.cucd_create.argtypes = [C.POINTER(_Config), C.POINTER(C.c_void_p)]
    lib.cucd_destroy.argtypes = [C.c_void_p]
    lib.cuCUDecide_frames.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.c_int, C.POINTER(C.c_void_p), C.c_int,
                                      C.POINTER(_FrameOut)]
    lib.cuCUDecide_frames_u8.argtypes = lib.cuCUDecide_frames.argtypes
    lib.cucd_pin_host_buffer.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    lib.cucd_unpin_host_buffer.argtypes = [C.c_void_p, C.c_void_p]
    lib.cucd_unpack_costs.argtypes = [C.c_void_p, C.c_void_p]
    lib.cucd_unpack_costs.restype = None
    lib.cucd_packed_cost.argtypes = [C.c_void_p, C.c_int, C.c_int]
    lib.cucd_packed_cost.restype = C.c_uint32
    lib.cucd_set_rmd_path.argtypes = [C.c_void_p, C.c_int]
    lib.cucd_set_decision_switches.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    lib.cuCUDecide_frame.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.POINTER(_FrameOut)]
    lib.cucd_intra_rmd_batch.argtypes = [C.c_void_p, C.c_int, C.POINTER(_PuDesc), C.c_void_p, C.c_void_p, C.c_void_p]
    lib.cucd_set_ref_picture.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int]
    lib.cucd_set_cur_picture.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    lib.cucd_me_sad_surface.argtypes = [C.c_void_p, C.c_int, C.POINTER(_MeDesc), C.c_void_p]
    lib.cucd_me_subpel_cost.argtypes = [C.c_void_p, C.c_int, C.POINTER(_SubpelDesc), C.c_void_p]
    lib.cucd_me_sad_surface_src.argtypes = [C.c_void_p, C.c_int, C.POINTER(_MeDesc), C.c_void_p, C.c_void_p]
    lib.cucd_me_subpel_cost_src.argtypes = [C.c_void_p, C.c_int, C.POINTER(_SubpelDesc), C.c_void_p, C.c_void_p]
    lib.cucd_me_mc_cost.argtypes = [C.c_void_p, C.c_int, C.POINTER(_McDesc), C.c_void_p, C.c_void_p]
    lib.cucd_set_ref_picture_chroma.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]
    lib.cucd_set_cur_picture_chroma.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    lib.cucd_me_mc_chroma.argtypes = [C.c_void_p, C.c_int, C.POINTER(_McDesc), C.c_void_p, C.c_void_p]
    lib.cucd_intra_tu_forward.argtypes = [C.c_void_p, C.c_int, C.POINTER(_TuDesc), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.cucd_intra_tu_recon.argtypes = [C.c_void_p, C.c_int, C.POINTER(_TuDesc), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.cucd_intra_tu_code.argtypes = [C.c_void_p, C.c_int, C.POINTER(_TuDesc), C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p]
    lib.cucd_inter_tu_forward.argtypes = [C.c_void_p, C.c_int, C.POINTER(_TuDesc), C.c_void_p, C.c_void_p, C.c_void_p]
    lib.cucd_inter_tu_recon.argtypes = [C.c_void_p, C.c_int, C.POINTER(_TuDesc), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.cucd_inter_tu_code.argtypes = [C.c_void_p, C.c_int, C.POINTER(_TuDesc), C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p]
    lib.cucd_tmv_features.argtypes = [C.c_void_p, C.c_int, C.POINTER(_CuDesc), C.c_void_p]
    lib.cucd_aq_activity.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.c_void_p]
    lib.cucd_dev_rmd_frames.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_longlong, C.c_int, C.c_void_p,
                                        C.c_longlong, C.c_int, C.c_void_p]
    lib.cucd_dev_feature_hist.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_longlong, C.c_int, C.c_void_p]
    lib.cucd_dev_feature_obf.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_longlong, C.c_int, C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_void_p]
    lib.cucd_dev_frames.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_longlong, C.c_int, C.c_void_p, C.c_longlong,
                                    C.c_int, C.POINTER(_DevOut), C.c_void_p]
    lib.cucd_dev_me_sad_surface.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(_MeDesc), C.c_void_p]
    lib.cucd_dev_me_subpel_cost.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(_SubpelDesc), C.c_void_p]
    lib.cucd_dev_frames_begin.argtypes = lib.cucd_dev_frames.argtypes
    lib.cucd_dev_frames_end.argtypes = [C.c_void_p]
    lib.cucd_queue_create.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
    lib.cucd_queue_destroy.argtypes = [C.c_void_p]
    lib.cucd_queue_submit.argtypes = [C.c_void_p, C.c_int, C.POINTER(_PuDesc), C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64)]
    lib.cucd_queue_wait.argtypes = [C.c_void_p, C.c_uint64]
    lib.cucd_queue_stats.argtypes = [C.c_void_p, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]
    lib.cucd_last_kernel_time.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
    lib.cucd_rmd_kernel_time.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_float)]
    lib.cucd_tcm_fit.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    _lib = lib
    return lib


def tcm_fit(hist, n_blocks):
    """cucd_tcm_fit: 16x4096 uint32 histogram of one picture -> (yc[16] float64, thr[16] int32)."""
    lib = load_library()
    hist = np.ascontiguousarray(hist, np.uint32)
    assert hist.size == 16 * 4096
    yc = np.zeros(16, np.float64)
    thr = np.zeros(16, np.int32)
    rc = lib.cucd_tcm_fit(hist.ctypes.data, int(n_blocks), yc.ctypes.data, thr.ctypes.data)
    if rc != 0:
        raise CucdError(f"cucd_tcm_fit failed ({rc})")
    return yc, thr


def _plane(a, dtype=np.int16):
    a = np.asarray(a)
    isz = np.dtype(dtype).itemsize
    if a.dtype != dtype or a.ndim != 2 or a.strides[1] != isz or a.strides[0] % isz:
        raise ValueError(f"planes must be 2-D {np.dtype(dtype).name} arrays with contiguous rows")
    return a, a.strides[0] // isz


class Engine:
    """One cucd_handle: one encoder instance on one GPU."""

    def __init__(self, width, height, bit_depth=8, strong_intra_smoothing=1, device=0, max_pictures=1, host_threads=0, auto_pin_host=0):
        self.lib = load_library()
        self.width, self.height, self.bit_depth = int(width), int(height), int(bit_depth)
        self.ctus_per_row = (self.width + 63) // 64
        self.ctus_per_pic = self.ctus_per_row * ((self.height + 63) // 64)
        cfg = _Config(self.width, self.height, self.bit_depth, 64, 4, int(strong_intra_smoothing), int(device), int(max_pictures),
                      int(host_threads), int(auto_pin_host))
        self.h = C.c_void_p()
        rc = self.lib.cucd_create(C.byref(cfg), C.byref(self.h))
        if rc != 0:
            msg = self.lib.cucd_last_error(None).decode()
            self.h = None
            raise CucdError(f"cucd_create failed ({rc}): {msg}")

    # ---- plumbing -------------------------------------------------------------------------------
    def _check(self, rc, what):
        if rc != 0:
            raise CucdError(f"{what} failed ({rc}): {self.lib.cucd_last_error(self.h).decode()}")

    def close(self):
        if getattr(self, "h", None):
            self.lib.cucd_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    @property
    def launch_count(self):
        return int(self.lib.cucd_launch_count(self.h))

    def cu_grid(self, depth):
        s = 64 >> depth
        return self.height // s, self.width // s

    # ---- S1/S4 (+ replay S2) --------------------------------------------------------------------
    def alloc_frame_out(self, want_rmd=True, pinned_alloc=None, packed=False, narrow=False):
        """numpy output buffers for one picture (pinned_alloc(shape, dtype) may supply pinned memory).
        packed=True asks for the cost tables in the packed CTU format (rmd_cost_packed) instead of uint32,
        narrow=True for the OBF / Outlier planes as bytes (obf_u8 / outlier_u8) instead of int16."""
        mk = pinned_alloc or (lambda shape, dtype: np.zeros(shape, dtype))
        W, H = self.width, self.height
        out = {"yc": mk((16,), np.float64), "ctu_src_had": mk((self.ctus_per_pic,), np.int32)}
        if narrow:
            out["obf_u8"] = mk((H // 4, W // 4), np.uint8); out["outlier_u8"] = mk((H, W), np.uint8)
        else:
            out["obf"] = mk((H // 4, W // 4), np.int16); out["outlier"] = mk((H, W), np.int16)
        for d in range(4):
            out[f"num_obf{d}"] = mk(self.cu_grid(d), np.int32)
            out[f"n_outlier{d}"] = mk(self.cu_grid(d), np.int32)
        if want_rmd and packed:
            out["rmd_cost_packed"] = mk((self.ctus_per_pic, PACKED_CTU_BYTES), np.uint8)
        elif want_rmd:
            out["rmd_cost"] = mk((self.ctus_per_pic, PUS_PER_CTU, NUM_MODES), np.uint32)
        return out

    def _frame_out_struct(self, o):
        fo = _FrameOut()

        def ptr(name, t):
            a = o.get(name)
            return a.ctypes.data_as(t) if a is not None and a.size else t()

        fo.obf = ptr("obf", _i16p)
        fo.outlier = ptr("outlier", _i16p)
        fo.yc = ptr("yc", _f64p)
        for d in range(4):
            fo.num_obf[d] = ptr(f"num_obf{d}", _i32p)
            fo.n_outlier[d] = ptr(f"n_outlier{d}", _i32p)
        fo.ctu_src_had = ptr("ctu_src_had", _i32p)
        fo.rmd_cost = ptr("rmd_cost", _u32p)
        fo.rmd_cost_packed = ptr("rmd_cost_packed", C.POINTER(C.c_uint8))
        fo.obf_u8 = ptr("obf_u8", C.POINTER(C.c_uint8))
        fo.outlier_u8 = ptr("outlier_u8", C.POINTER(C.c_uint8))
        return fo

    def frames(self, orgs, recs=None, outs=None, want_rmd=True):
        """cuCUDecide_frames (int16 planes) / cuCUDecide_frames_u8 (uint8 planes) on host planes; returns the list of output dicts."""
        n = len(orgs)
        dt = np.uint8 if np.asarray(orgs[0]).dtype == np.uint8 else np.int16
        fn = self.lib.cuCUDecide_frames_u8 if dt == np.uint8 else self.lib.cuCUDecide_frames
        planes = [_plane(a, dt) for a in orgs]
        stride = planes[0][1]
        assert all(s == stride and p.shape == (self.height, self.width) for p, s in planes)
        org_ptrs = (C.c_void_p * n)(*[p.ctypes.data for p, _ in planes])
        rec_ptrs, rstride = None, 0
        if recs is not None:
            rp = [_plane(a, dt) for a in recs]
            rstride = rp[0][1]
            assert len(rp) == n and all(s == rstride and p.shape == (self.height, self.width) for p, s in rp)
            rec_ptrs = (C.c_void_p * n)(*[p.ctypes.data for p, _ in rp])
        if outs is None:
            outs = [self.alloc_frame_out(want_rmd and recs is not None) for _ in range(n)]
        fos = (_FrameOut * n)(*[self._frame_out_struct(o) for o in outs])
        self._check(fn(self.h, n, org_ptrs, stride, rec_ptrs, rstride, fos), "cuCUDecide_frames")
        return outs

    def pin_host_buffer(self, a):
        """cucd_pin_host_buffer on the memory of a numpy array (page-locks it for the lifetime of the handle)"""
        a = np.asarray(a)
        lo = a.ctypes.data
        nbytes = (a.shape[0] - 1) * a.strides[0] + a.shape[1] * a.strides[1] if a.ndim == 2 else a.nbytes
        self._check(self.lib.cucd_pin_host_buffer(self.h, lo, nbytes), "cucd_pin_host_buffer")

    def unpin_host_buffer(self, a):
        self._check(self.lib.cucd_unpin_host_buffer(self.h, np.asarray(a).ctypes.data), "cucd_unpin_host_buffer")

    def unpack_costs_c(self, packed):
        """cucd_unpack_costs per CTU (the C helper a host encoder would call)"""
        packed = np.ascontiguousarray(packed, np.uint8).reshape(-1, PACKED_CTU_BYTES)
        out = np.empty((packed.shape[0], PUS_PER_CTU, NUM_MODES), np.uint32)
        for i in range(packed.shape[0]):
            self.lib.cucd_unpack_costs(packed[i].ctypes.data, out[i].ctypes.data)
        return out

    def frame(self, org, rec=None, poc=0, out=None, want_rmd=True):
        """cuCUDecide_frame: one picture."""
        p, stride = _plane(org)
        rptr, rstride = None, 0
        if rec is not None:
            r, rstride = _plane(rec)
            rptr = r.ctypes.data
        if out is None:
            out = self.alloc_frame_out(want_rmd and rec is not None)
        fo = self._frame_out_struct(out)
        self._check(self.lib.cuCUDecide_frame(self.h, p.ctypes.data, stride, rptr, rstride, int(poc), C.byref(fo)), "cuCUDecide_frame")
        return out

    # ---- S2 ---------------------------------------------------------------------------------------
    def intra_rmd_batch(self, log2_sizes, org, border):
        """cucd_intra_rmd_batch: PUs of mixed sizes, org/border packed back to back. Returns (nPU, 35) uint32."""
        log2_sizes = np.asarray(log2_sizes, np.uint8)
        n = int(log2_sizes.size)
        org = np.ascontiguousarray(org, np.int16).ravel()
        border = np.ascontiguousarray(border, np.int16).ravel()
        sizes = 1 << log2_sizes.astype(np.int64)
        assert org.size == int((sizes * sizes).sum()) and border.size == int((4 * sizes + 1).sum())
        desc = (_PuDesc * max(n, 1))()
        for i in range(n):
            desc[i].log2_size = int(log2_sizes[i])
        sad = np.zeros((n, NUM_MODES), np.uint32)
        self._check(self.lib.cucd_intra_rmd_batch(self.h, n, desc, org.ctypes.data, border.ctypes.data, sad.ctypes.data), "cucd_intra_rmd_batch")
        return sad

    @staticmethod
    def pu_descs(log2_sizes):
        """ctypes descriptor array for cucd_intra_rmd_batch (build once, reuse): (array, n)"""
        log2_sizes = np.asarray(log2_sizes, np.uint8)
        desc = (_PuDesc * max(int(log2_sizes.size), 1))()
        np.frombuffer(desc, np.uint8)[: 4 * log2_sizes.size: 4] = log2_sizes
        return desc, int(log2_sizes.size)

    def intra_rmd_batch_raw(self, desc, n, org, border, sad):
        """the bare C call on prebuilt descriptors and caller-owned numpy buffers (what an encoder's own call costs)"""
        self._check(self.lib.cucd_intra_rmd_batch(self.h, n, desc, org.ctypes.data, border.ctypes.data, sad.ctypes.data), "cucd_intra_rmd_batch")

    def intra_tu_raw(self, stage, arr, n, org, border, coef_or_level, pix, dist, abs_sum, flags=TU_INTRA_SLICE | TU_SIGN_HIDING):
        """stage 0: cucd_intra_tu_forward (coef out, pix = pred), 1: cucd_intra_tu_code, 2: cucd_intra_tu_recon (level in) on prebuilt descriptors"""
        if stage == 0:
            rc = self.lib.cucd_intra_tu_forward(self.h, n, arr, org.ctypes.data, border.ctypes.data, coef_or_level.ctypes.data, pix.ctypes.data)
        elif stage == 1:
            rc = self.lib.cucd_intra_tu_code(self.h, n, arr, org.ctypes.data, border.ctypes.data, int(flags), coef_or_level.ctypes.data, pix.ctypes.data,
                                             dist.ctypes.data, abs_sum.ctypes.data)
        else:
            rc = self.lib.cucd_intra_tu_recon(self.h, n, arr, org.ctypes.data, border.ctypes.data, coef_or_level.ctypes.data, pix.ctypes.data, dist.ctypes.data)
        self._check(rc, "cucd_intra_tu_*")

    def inter_tu_raw(self, stage, arr, n, resi, coef_or_level, rresi=None, dist=None, dist_zero=None, abs_sum=None, flags=TU_SIGN_HIDING):
        """stage 0: cucd_inter_tu_forward (coef out), 1: cucd_inter_tu_code, 2: cucd_inter_tu_recon (level in) on prebuilt descriptors;
        outputs are caller-owned numpy arrays, None where the call allows NULL"""
        ptr = lambda a: None if a is None else a.ctypes.data
        if stage == 0:
            rc = self.lib.cucd_inter_tu_forward(self.h, n, arr, resi.ctypes.data, coef_or_level.ctypes.data, ptr(dist_zero))
        elif stage == 1:
            rc = self.lib.cucd_inter_tu_code(self.h, n, arr, resi.ctypes.data, int(flags), coef_or_level.ctypes.data, ptr(rresi), ptr(dist),
                                             ptr(dist_zero), ptr(abs_sum))
        else:
            rc = self.lib.cucd_inter_tu_recon(self.h, n, arr, resi.ctypes.data, coef_or_level.ctypes.data, ptr(rresi), ptr(dist))
        self._check(rc, "cucd_inter_tu_*")

    # ---- S3 ---------------------------------------------------------------------------------------
    def set_ref_picture(self, ref_idx, padded, margin_x, margin_y):
        """padded: (H+2my, W+2mx) int16 plane including the replicated margins."""
        p, stride = _plane(padded)
        assert p.shape == (self.height + 2 * margin_y, self.width + 2 * margin_x)
        origin = p.ctypes.data + 2 * (margin_y * stride + margin_x)
        self._check(self.lib.cucd_set_ref_picture(self.h, int(ref_idx), origin, stride, int(margin_x), int(margin_y)), "cucd_set_ref_picture")

    def set_cur_picture(self, org):
        p, stride = _plane(org)
        self._check(self.lib.cucd_set_cur_picture(self.h, p.ctypes.data, stride), "cucd_set_cur_picture")

    @staticmethod
    def me_descs(descs):
        """list of dicts(x,y,w,h,ref_idx,left,right,top,bottom,sub_shift) -> (ctypes array, n, total candidates): build once, reuse"""
        arr = (_MeDesc * max(len(descs), 1))()
        total = 0
        for i, d in enumerate(descs):
            for k in ("x", "y", "w", "h", "ref_idx", "left", "right", "top", "bottom", "sub_shift"):
                setattr(arr[i], k, int(d[k]))
            total += (d["bottom"] - d["top"] + 1) * (d["right"] - d["left"] + 1)
        return arr, len(descs), total

    @staticmethod
    def subpel_descs(descs):
        arr = (_SubpelDesc * max(len(descs), 1))()
        for i, d in enumerate(descs):
            for k in ("x", "y", "w", "h", "ref_idx", "mvx", "mvy", "use_hadamard"):
                setattr(arr[i], k, int(d[k]))
        return arr, len(descs)

    def me_sad_surface_raw(self, arr, n, out):
        """cucd_me_sad_surface with a prebuilt descriptor array; out: uint32 host array of `total` candidates"""
        self._check(self.lib.cucd_me_sad_surface(self.h, n, arr, out.ctypes.data), "cucd_me_sad_surface")

    def me_subpel_cost_raw(self, arr, n, out):
        self._check(self.lib.cucd_me_subpel_cost(self.h, n, arr, out.ctypes.data), "cucd_me_subpel_cost")

    def dev_me_sad_surface(self, stream, arr, n, d_out):
        """cucd_dev_me_sad_surface: surfaces stay in HBM at device pointer d_out"""
        self._check(self.lib.cucd_dev_me_sad_surface(self.h, stream, n, arr, d_out), "cucd_dev_me_sad_surface")

    def dev_me_subpel_cost(self, stream, arr, n, d_out):
        self._check(self.lib.cucd_dev_me_subpel_cost(self.h, stream, n, arr, d_out), "cucd_dev_me_subpel_cost")

    def me_sad_surface(self, descs, src=None):
        """descs: list of dicts(x,y,w,h,ref_idx,left,right,top,bottom,sub_shift). Returns list of (rows, cols) uint32 surfaces.
        src: optional int16 array with the PUs' own w x h source blocks back to back (cucd_me_sad_surface_src: bi-predictive search)."""
        n = len(descs)
        arr = (_MeDesc * max(n, 1))()
        total = 0
        shapes = []
        for i, d in enumerate(descs):
            for k in ("x", "y", "w", "h", "ref_idx", "left", "right", "top", "bottom", "sub_shift"):
                setattr(arr[i], k, int(d[k]))
            shapes.append((d["bottom"] - d["top"] + 1, d["right"] - d["left"] + 1))
            total += shapes[-1][0] * shapes[-1][1]
        out = np.zeros(max(total, 1), np.uint32)
        if src is None:
            self._check(self.lib.cucd_me_sad_surface(self.h, n, arr, out.ctypes.data), "cucd_me_sad_surface")
        else:
            src = np.ascontiguousarray(src, np.int16)
            assert src.size == sum(int(d["w"]) * int(d["h"]) for d in descs)
            self._check(self.lib.cucd_me_sad_surface_src(self.h, n, arr, src.ctypes.data, out.ctypes.data), "cucd_me_sad_surface_src")
        res, off = [], 0
        for r, c in shapes:
            res.append(out[off:off + r * c].reshape(r, c))
            off += r * c
        return res

    def me_subpel_cost(self, descs, src=None):
        """descs: list of dicts(x,y,w,h,ref_idx,mvx,mvy,use_hadamard). Returns (n, 7, 7) uint32: [dy+3][dx+3], quarter-pel offsets.
        src: optional int16 array with the PUs' own source blocks back to back (cucd_me_subpel_cost_src)."""
        n = len(descs)
        arr = (_SubpelDesc * max(n, 1))()
        for i, d in enumerate(descs):
            for k in ("x", "y", "w", "h", "ref_idx", "mvx", "mvy", "use_hadamard"):
                setattr(arr[i], k, int(d[k]))
        out = np.zeros((n, 7, 7), np.uint32)
        if src is None:
            self._check(self.lib.cucd_me_subpel_cost(self.h, n, arr, out.ctypes.data), "cucd_me_subpel_cost")
        else:
            src = np.ascontiguousarray(src, np.int16)
            assert src.size == sum(int(d["w"]) * int(d["h"]) for d in descs)
            self._check(self.lib.cucd_me_subpel_cost_src(self.h, n, arr, src.ctypes.data, out.ctypes.data), "cucd_me_subpel_cost_src")
        return out

    @staticmethod
    def mc_descs(descs):
        """list of dicts(x,y,w,h,ref_idx=(r0,r1),mvx=(..),mvy=(..),use_hadamard) -> (ctypes array, n, prediction samples)"""
        arr = (_McDesc * max(len(descs), 1))()
        samples = 0
        for i, d in enumerate(descs):
            for k in ("x", "y", "w", "h", "use_hadamard"):
                setattr(arr[i], k, int(d[k]))
            for k in ("ref_idx", "mvx", "mvy"):
                a, b = d[k]
                getattr(arr[i], k)[0] = int(a)
                getattr(arr[i], k)[1] = int(b)
            samples += int(d["w"]) * int(d["h"])
        return arr, len(descs), samples

    def me_mc_cost_raw(self, arr, n, dist, pred=None):
        """cucd_me_mc_cost with a prebuilt descriptor array; dist: uint32 host array of n, pred: int16 host array or None"""
        self._check(self.lib.cucd_me_mc_cost(self.h, n, arr, dist.ctypes.data, None if pred is None else pred.ctypes.data), "cucd_me_mc_cost")

    def me_mc_cost(self, descs, want_pred=False):
        """Motion compensation + distortion of inter candidates (cucd_me_mc_cost).  descs: list of dicts(x, y, w, h, ref_idx=(r0, r1),
        mvx=(mx0, mx1), mvy=(my0, my1), use_hadamard); ref_idx -1 = list unused, MVs in quarter pels.  Returns dist, (n,) uint32, and
        with want_pred=True also the list of (h, w) int16 predictions: (dist, preds)."""
        arr, n, samples = self.mc_descs(descs)
        dist = np.zeros(n, np.uint32)
        pred = np.zeros(max(samples, 1), np.int16) if want_pred else None
        self.me_mc_cost_raw(arr, n, dist, pred)
        if not want_pred:
            return dist
        res, off = [], 0
        for d in descs:
            w, h = int(d["w"]), int(d["h"])
            res.append(pred[off:off + w * h].reshape(h, w))
            off += w * h
        return dist, res

    # ---- 4:2:0 chroma of inter candidates (cucd_me_mc_chroma) ------------------------------------------------
    def set_ref_picture_chroma(self, ref_idx, cb_padded, cr_padded, margin_x, margin_y):
        """cb_padded, cr_padded: (H/2 + 2my, W/2 + 2mx) int16 planes including the replicated margins (chroma samples), one stride.
        Call after set_ref_picture(ref_idx, ...): that call marks the slot's chroma unset."""
        (cb, stride), (cr, stride_r) = _plane(cb_padded), _plane(cr_padded)
        assert cb.shape == cr.shape == (self.height // 2 + 2 * margin_y, self.width // 2 + 2 * margin_x) and stride == stride_r
        off = 2 * (margin_y * stride + margin_x)
        self._check(self.lib.cucd_set_ref_picture_chroma(self.h, int(ref_idx), cb.ctypes.data + off, cr.ctypes.data + off, stride, int(margin_x),
                                                         int(margin_y)), "cucd_set_ref_picture_chroma")

    def set_cur_picture_chroma(self, cb, cr):
        """cb, cr: (H/2, W/2) int16 planes of the current picture, one stride.  Call after set_cur_picture."""
        (cb, stride), (cr, stride_r) = _plane(cb), _plane(cr)
        assert cb.shape == cr.shape == (self.height // 2, self.width // 2) and stride == stride_r
        self._check(self.lib.cucd_set_cur_picture_chroma(self.h, cb.ctypes.data, cr.ctypes.data, stride), "cucd_set_cur_picture_chroma")

    def me_mc_chroma_raw(self, arr, n, sse, pred=None):
        """cucd_me_mc_chroma with a prebuilt descriptor array (mc_descs); sse: uint32 host array of 2 n, pred: int16 host array of
        n_samples / 2 (the luma sample count of mc_descs) or None"""
        self._check(self.lib.cucd_me_mc_chroma(self.h, n, arr, sse.ctypes.data, None if pred is None else pred.ctypes.data), "cucd_me_mc_chroma")

    def me_mc_chroma(self, descs, want_pred=False):
        """4:2:0 chroma motion compensation + SSE of inter candidates (cucd_me_mc_chroma) on the descriptors of me_mc_cost.  Returns sse,
        (n, 2) uint32 (Cb, Cr), and with want_pred=True also the list of (Cb, Cr) pairs of (h/2, w/2) int16 predictions: (sse, preds)."""
        arr, n, samples = self.mc_descs(descs)
        sse = np.zeros((n, 2), np.uint32)
        pred = np.zeros(max(samples // 2, 1), np.int16) if want_pred else None
        self.me_mc_chroma_raw(arr, n, sse, pred)
        if not want_pred:
            return sse
        res, off = [], 0
        for d in descs:
            cw, ch = int(d["w"]) // 2, int(d["h"]) // 2
            res.append((pred[off:off + cw * ch].reshape(ch, cw), pred[off + cw * ch:off + 2 * cw * ch].reshape(ch, cw)))
            off += 2 * cw * ch
        return sse, res

    # ---- intra luma TU coding (xIntraCodingTUBlock) ------------------------------------------------
    @staticmethod
    def _tu_descs(tus):
        """tus: iterable of (log2_size, mode, qp, transform_skip[, chroma])"""
        tus = list(tus)
        arr = (_TuDesc * max(len(tus), 1))()
        total = 0
        for i, tu in enumerate(tus):
            l, m, q, ts = tu[:4]
            chroma = tu[4] if len(tu) > 4 else 0
            arr[i].log2_size, arr[i].mode, arr[i].qp, arr[i].flags = int(l), int(m), int(q), (1 if ts else 0) | (2 if chroma else 0)
            total += 1 << (2 * int(l))
        return tus, arr, total

    def intra_tu_forward(self, tus, org, border, want_pred=True):
        """Returns (coef int32, pred int16), both flat in the packing of org."""
        tus, arr, total = self._tu_descs(tus)
        org = np.ascontiguousarray(org, np.int16).ravel(); border = np.ascontiguousarray(border, np.int16).ravel()
        coef = np.zeros(total, np.int32)
        pred = np.zeros(total, np.int16) if want_pred else None
        self._check(self.lib.cucd_intra_tu_forward(self.h, len(tus), arr, org.ctypes.data, border.ctypes.data, coef.ctypes.data,
                                                   pred.ctypes.data if want_pred else None), "cucd_intra_tu_forward")
        return coef, pred

    def intra_tu_recon(self, tus, org, border, level):
        """Returns (reco int16 flat, dist uint32 per TU)."""
        tus, arr, total = self._tu_descs(tus)
        org = np.ascontiguousarray(org, np.int16).ravel(); border = np.ascontiguousarray(border, np.int16).ravel()
        level = np.ascontiguousarray(level, np.int32).ravel()
        assert level.size == total
        reco = np.zeros(total, np.int16)
        dist = np.zeros(len(tus), np.uint32)
        self._check(self.lib.cucd_intra_tu_recon(self.h, len(tus), arr, org.ctypes.data, border.ctypes.data, level.ctypes.data, reco.ctypes.data,
                                                 dist.ctypes.data), "cucd_intra_tu_recon")
        return reco, dist

    def intra_tu_code(self, tus, org, border, flags=TU_INTRA_SLICE | TU_SIGN_HIDING):
        """Whole chain with the plain quantiser. Returns (level int32 flat, reco int16 flat, dist uint32, abs_sum int32)."""
        tus, arr, total = self._tu_descs(tus)
        org = np.ascontiguousarray(org, np.int16).ravel(); border = np.ascontiguousarray(border, np.int16).ravel()
        level = np.zeros(total, np.int32); reco = np.zeros(total, np.int16)
        dist = np.zeros(len(tus), np.uint32); abs_sum = np.zeros(len(tus), np.int32)
        self._check(self.lib.cucd_intra_tu_code(self.h, len(tus), arr, org.ctypes.data, border.ctypes.data, int(flags), level.ctypes.data,
                                                reco.ctypes.data, dist.ctypes.data, abs_sum.ctypes.data), "cucd_intra_tu_code")
        return level, reco, dist, abs_sum

    # ---- inter TU coding (xEstimateResidualQT): the TUs of inter residual quadtrees ------------------------------------
    @staticmethod
    def _inter_tu_descs(tus):
        """tus: iterable of (log2_size, qp, transform_skip[, chroma]); the mode of every descriptor is 0"""
        tus = [(t[0], 0) + tuple(t[1:]) for t in tus]
        return Engine._tu_descs(tus)

    def inter_tu_forward(self, tus, resi):
        """resi: the residual blocks org - pred, N*N int16 per TU back to back.  Returns (coef int32 flat, dist_zero uint32 per TU)."""
        tus, arr, total = self._inter_tu_descs(tus)
        resi = np.ascontiguousarray(resi, np.int16).ravel()
        assert resi.size == total
        coef = np.zeros(total, np.int32)
        dist_zero = np.zeros(len(tus), np.uint32)
        self.inter_tu_raw(0, arr, len(tus), resi, coef, dist_zero=dist_zero)
        return coef, dist_zero

    def inter_tu_recon(self, tus, resi, level):
        """levels chosen by the caller (RDOQ).  Returns (rresi int16 flat, dist uint32 per TU)."""
        tus, arr, total = self._inter_tu_descs(tus)
        resi = np.ascontiguousarray(resi, np.int16).ravel()
        level = np.ascontiguousarray(level, np.int32).ravel()
        assert resi.size == total and level.size == total
        rresi = np.zeros(total, np.int16)
        dist = np.zeros(len(tus), np.uint32)
        self.inter_tu_raw(2, arr, len(tus), resi, level, rresi=rresi, dist=dist)
        return rresi, dist

    def inter_tu_code(self, tus, resi, sign_hiding=True):
        """Whole chain with the plain quantiser.  Returns (level int32 flat, rresi int16 flat, dist uint32, dist_zero uint32, abs_sum int32)."""
        tus, arr, total = self._inter_tu_descs(tus)
        resi = np.ascontiguousarray(resi, np.int16).ravel()
        assert resi.size == total
        level = np.zeros(total, np.int32); rresi = np.zeros(total, np.int16)
        dist = np.zeros(len(tus), np.uint32); dist_zero = np.zeros(len(tus), np.uint32); abs_sum = np.zeros(len(tus), np.int32)
        self.inter_tu_raw(1, arr, len(tus), resi, level, rresi=rresi, dist=dist, dist_zero=dist_zero, abs_sum=abs_sum,
                          flags=TU_SIGN_HIDING if sign_hiding else 0)
        return level, rresi, dist, dist_zero, abs_sum

    def tmv_features(self, cus):
        """cus: iterable of (x, y, log2_size) of the picture given to set_cur_picture. Returns (nCU, 5, 26) float64
        = TMVFeature::m_adFeature of getTMVFeature (tools_YS.cpp:1682-1839)."""
        cus = list(cus)
        arr = (_CuDesc * max(len(cus), 1))()
        for i, (x, y, l) in enumerate(cus):
            arr[i].x, arr[i].y, arr[i].log2_size = int(x), int(y), int(l)
        out = np.zeros((len(cus), 5, 26), np.float64)
        self._check(self.lib.cucd_tmv_features(self.h, len(cus), arr, out.ctypes.data), "cucd_tmv_features")
        return out

    @staticmethod
    def cu_descs(cus):
        arr = (_CuDesc * max(len(cus), 1))()
        for i, (x, y, l) in enumerate(cus):
            arr[i].x, arr[i].y, arr[i].log2_size = int(x), int(y), int(l)
        return arr, len(cus)

    def tmv_features_raw(self, arr, n, out):
        self._check(self.lib.cucd_tmv_features(self.h, n, arr, out.ctypes.data), "cucd_tmv_features")

    def aq_activity(self, max_aq_depth):
        """TEncPreanalyzer::xPreanalyze of the current picture: ([per-layer (rows, cols) float64 activity], avg[max_aq_depth])."""
        acts = []
        for d in range(max_aq_depth):
            u = 64 >> d
            acts.append(np.zeros(((self.height + u - 1) // u, (self.width + u - 1) // u), np.float64))
        ptrs = (C.c_void_p * max_aq_depth)(*[a.ctypes.data for a in acts])
        avg = np.zeros(max_aq_depth, np.float64)
        self._check(self.lib.cucd_aq_activity(self.h, int(max_aq_depth), ptrs, avg.ctypes.data), "cucd_aq_activity")
        return acts, avg

    # ---- device-resident entry points (raw pointers) ----------------------------------------------
    def dev_rmd_frames(self, stream, n_pics, d_org, org_pic_stride, org_stride, d_rec, rec_pic_stride, rec_stride, d_cost):
        self._check(self.lib.cucd_dev_rmd_frames(self.h, stream, n_pics, d_org, org_pic_stride, org_stride, d_rec, rec_pic_stride,
                                                 rec_stride, d_cost), "cucd_dev_rmd_frames")

    def dev_feature_hist(self, stream, n_pics, d_org, org_pic_stride, org_stride, d_hist):
        self._check(self.lib.cucd_dev_feature_hist(self.h, stream, n_pics, d_org, org_pic_stride, org_stride, d_hist), "cucd_dev_feature_hist")

    def dev_feature_obf(self, stream, n_pics, d_org, org_pic_stride, org_stride, d_thr, d_obf, d_outlier, d_num, d_sum, d_ctu_had):
        num = (C.c_void_p * 4)(*d_num)
        summ = (C.c_void_p * 4)(*d_sum)
        self._check(self.lib.cucd_dev_feature_obf(self.h, stream, n_pics, d_org, org_pic_stride, org_stride, d_thr, d_obf, d_outlier,
                                                  num, summ, d_ctu_had), "cucd_dev_feature_obf")

    def dev_frames(self, stream, n_pics, d_org, org_pic_stride, org_stride, d_rec, rec_pic_stride, rec_stride, d_out, yc_host=None, begin_only=False):
        """cucd_dev_frames (or, with begin_only, cucd_dev_frames_begin - pair it with dev_frames_end):
        d_out = dict of device pointers (obf, outlier, num_obf[4], n_outlier[4], ctu_src_had, rmd_cost)."""
        o = _DevOut()
        o.obf = d_out.get("obf")
        o.outlier = d_out.get("outlier")
        for d in range(4):
            o.num_obf[d] = (d_out.get("num_obf") or [None] * 4)[d]
            o.n_outlier[d] = (d_out.get("n_outlier") or [None] * 4)[d]
        o.ctu_src_had = d_out.get("ctu_src_had")
        o.rmd_cost = d_out.get("rmd_cost")
        yc = yc_host.ctypes.data if yc_host is not None else None
        fn = self.lib.cucd_dev_frames_begin if begin_only else self.lib.cucd_dev_frames
        self._check(fn(self.h, stream, n_pics, d_org, org_pic_stride, org_stride, d_rec, rec_pic_stride, rec_stride, C.byref(o), yc), "cucd_dev_frames")

    def dev_frames_end(self):
        self._check(self.lib.cucd_dev_frames_end(self.h), "cucd_dev_frames_end")

    def last_kernel_time_ms(self):
        ms = C.c_float(0)
        self._check(self.lib.cucd_last_kernel_time(self.h, C.byref(ms)), "cucd_last_kernel_time")
        return ms.value

    def rmd_kernel_time_ms(self, n_calls):
        """mean device duration of the RMD launch over the last n_calls dev_frames calls (stream must be synchronised)"""
        ms = C.c_float(0)
        n = self.lib.cucd_rmd_kernel_time(self.h, int(n_calls), C.byref(ms))
        if n < 0:
            self._check(n, "cucd_rmd_kernel_time")
        return float(ms.value), int(n)

    def set_decision_switches(self, enable, skip2nx2n=(0, 0, 0, 0), terminate_cu=(0, 0, 0, 0)):
        """cucd_set_decision_switches: fork-aware enumeration of the frame calls (Testing pictures); per-depth switch lists of 4"""
        a = (C.c_uint8 * 4)(*[int(bool(v)) for v in skip2nx2n]); b = (C.c_uint8 * 4)(*[int(bool(v)) for v in terminate_cu])
        self._check(self.lib.cucd_set_decision_switches(self.h, int(bool(enable)), a, b), "cucd_set_decision_switches")

    def set_rmd_path(self, path):
        """0 / False: integer ALU; 1 / True: predictions + Hadamard on the tensor cores (kind::i8 at 8 bit, kind::f16 above);
        2: the half-precision tensor-core kernel whatever the bit depth"""
        self._check(self.lib.cucd_set_rmd_path(self.h, int(path)), "cucd_set_rmd_path")


class RmdQueue:
    """cucd_queue: asynchronous, coalescing front end of cucd_intra_rmd_batch shared by several host threads."""

    def __init__(self, engine):
        self.lib, self.engine = engine.lib, engine
        self.q = C.c_void_p()
        rc = self.lib.cucd_queue_create(engine.h, C.byref(self.q))
        if rc != 0:
            raise CucdError(f"cucd_queue_create failed ({rc})")

    def submit(self, log2_sizes, org, border):
        """returns (ticket, sad) - sad (nPU, 35) uint32 is valid after wait(ticket)"""
        log2_sizes = np.asarray(log2_sizes, np.uint8)
        n = int(log2_sizes.size)
        org = np.ascontiguousarray(org, np.int16).ravel()
        border = np.ascontiguousarray(border, np.int16).ravel()
        desc = (_PuDesc * max(n, 1))()
        for i in range(n):
            desc[i].log2_size = int(log2_sizes[i])
        sad = np.zeros((n, NUM_MODES), np.uint32)
        t = C.c_uint64(0)
        rc = self.lib.cucd_queue_submit(self.q, n, desc, org.ctypes.data, border.ctypes.data, sad.ctypes.data, C.byref(t))
        if rc != 0:
            raise CucdError(f"cucd_queue_submit failed ({rc})")
        return int(t.value), sad

    def wait(self, ticket):
        rc = self.lib.cucd_queue_wait(self.q, C.c_uint64(ticket))
        if rc != 0:
            raise CucdError(f"cucd_queue_wait failed ({rc}): {self.lib.cucd_last_error(self.engine.h).decode()}")

    def stats(self):
        r, p, b = C.c_longlong(0), C.c_longlong(0), C.c_longlong(0)
        self.lib.cucd_queue_stats(self.q, C.byref(r), C.byref(p), C.byref(b))
        return {"requests": int(r.value), "pus": int(p.value), "batches": int(b.value)}

    def close(self):
        if getattr(self, "q", None):
            self.lib.cucd_queue_destroy(self.q)
            self.q = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
