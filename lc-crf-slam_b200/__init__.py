"""lc-crf-slam_b200 -- B200 (sm_100a) implementation of LC-CRF-SLAM's CRF hot path.

The product is `liblccrf.so` (CUDA kernels behind the C ABI of include/lccrf.h) plus the C++
header mirror of the reference's DenseCRF API in `densecrf/`.  This Python module is plumbing
only: a ctypes binding used by tests/ and bench.py.  There is no CPU fallback -- every call
fails loudly when the library or a B200 is missing.

Import with `importlib.import_module("lc-crf-slam_b200")` (the directory name is not a valid
identifier).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import weakref

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "liblccrf.so")
INCLUDE_DIR = os.path.join(os.path.dirname(HERE), "include")
DENSECRF_INCLUDE_DIR = os.path.join(HERE, "densecrf")

from . import synth  # noqa: E402,F401


def build(verbose: bool = False) -> str:
    """Compile liblccrf.so in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    subprocess.run(["make", "-C", os.path.join(HERE, "csrc"), "-j8"], check=True,
                   stdout=None if verbose else subprocess.DEVNULL)
    return LIB_PATH


class LccrfError(RuntimeError):
    pass


class SlamParams(C.Structure):
    """lccrf_slam_params (TUM3.yaml:81-101)."""
    _fields_ = [(n, C.c_float) for n in (
        "w1", "w2", "u_alpha", "stdev_alpha", "u_beta", "stdev_beta", "u_gamma", "stdev_gamma",
        "point3d_stdev", "point2d_stdev", "u_depth", "pth", "confidence")] + [("iters", C.c_int)]

    @classmethod
    def make(cls, **kw) -> "SlamParams":
        p = cls()
        d = dict(synth.SLAM_PARAMS)
        d.update(kw)
        for k, v in d.items():
            setattr(p, k, v)
        return p


class ImageKernel(C.Structure):
    """lccrf_image_kernel: one PottsPotentialCPU<M,F>::FromImage potential (F = 2: Gaussian, F = C + 2: bilateral)."""
    _fields_ = [("F", C.c_int), ("w", C.c_float), ("posdev", C.c_float), ("featuredev", C.c_float)]


_fp = C.POINTER(C.c_float)
_ip = C.POINTER(C.c_int)
_sp = C.POINTER(C.c_short)
_vp = C.c_void_p
_byref = C.byref  # Images takes a parameter named C

# every symbol include/lccrf.h declares: (restype, argtypes)
SYMBOLS = {
    "lccrf_version": (C.c_char_p, []),
    "lccrf_last_error": (C.c_char_p, []),
    "lccrf_device_count": (C.c_int, []),
    "lccrf_ctx_create": (C.c_int, [C.c_int, C.POINTER(_vp)]),
    "lccrf_ctx_destroy": (None, [_vp]),
    "lccrf_ctx_set_stream": (C.c_int, [_vp, _vp]),
    "lccrf_ctx_sync": (C.c_int, [_vp]),
    "lccrf_ctx_kernel_launches": (C.c_uint64, [_vp]),
    "lccrf_ctx_build_scratch_in_use": (C.c_int, [_vp, _vp]),
    "lccrf_ctx_set_option": (C.c_int, [_vp, C.c_char_p, C.c_int]),
    "lccrf_ctx_profile_report": (C.c_int, [_vp, C.c_char_p, C.c_int]),
    "lccrf_lattice_create": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.POINTER(_vp)]),
    "lccrf_lattice_destroy": (None, [_vp]),
    "lccrf_lattice_sizes": (C.c_int, [_vp, _ip, _ip, _ip]),
    "lccrf_lattice_export": (C.c_int, [_vp, _vp, _vp, _vp]),
    "lccrf_lattice_filter": (C.c_int, [_vp, _vp, _vp, C.c_int]),
    "lccrf_lattice_filter_window": (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "lccrf_lattice_debug_counters": (C.c_int, [_vp, _vp]),
    "lccrf_crf_create": (C.c_int, [_vp, C.c_int, C.c_int, C.POINTER(_vp)]),
    "lccrf_crf_destroy": (None, [_vp]),
    "lccrf_crf_set_unary": (C.c_int, [_vp, _vp]),
    "lccrf_crf_set_unary_from_label": (C.c_int, [_vp, _vp, C.c_float, _vp, _vp]),
    "lccrf_crf_set_unary_entry": (C.c_int, [_vp, C.c_int, C.c_int, C.c_float]),
    "lccrf_crf_add_potts": (C.c_int, [_vp, _vp, C.c_int, C.c_float]),
    "lccrf_crf_add_potts_image": (C.c_int, [_vp, C.c_int, C.c_int, C.c_float, C.c_float, _vp, C.c_int, C.c_int, C.c_float]),
    "lccrf_crf_start": (C.c_int, [_vp]),
    "lccrf_crf_step": (C.c_int, [_vp, C.c_float]),
    "lccrf_crf_inference": (C.c_int, [_vp, C.c_int, C.c_int, C.c_float]),
    "lccrf_crf_build_map": (C.c_int, [_vp]),
    "lccrf_crf_map": (_sp, [_vp]),
    "lccrf_crf_prob": (_fp, [_vp]),
    "lccrf_crf_potts_vertices": (C.c_int, [_vp, C.c_int, _ip]),
    "lccrf_crf_num_potts": (C.c_int, [_vp]),
    "lccrf_crf_step_init": (C.c_int, [_vp, _vp]),
    "lccrf_crf_set_prob": (C.c_int, [_vp, _vp]),
    "lccrf_crf_potts_apply": (C.c_int, [_vp, C.c_int, _vp, _vp, _vp]),
    "lccrf_exp_and_normalize": (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_int, C.c_float, C.c_float]),
    "lccrf_map_point_unary": (C.c_int, [_vp, C.c_int, _vp, _vp, _vp, _vp, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp]),
    "lccrf_rough_classify": (C.c_int, [_vp, C.c_int, _vp, _vp, _vp, _vp, C.POINTER(SlamParams), _vp]),
    "lccrf_epipolar_prior": (C.c_int, [_vp, C.c_int, _vp, _vp, _vp, _vp, C.c_float, C.c_float, C.c_int, _vp, _vp, _vp, _vp]),
    "lccrf_bf_match": (C.c_int, [_vp, C.c_int, _vp, C.c_int, _vp, C.c_double, _vp, _vp, _ip]),
    "lccrf_bf_match_batch": (C.c_int, [_vp, C.c_int, _vp, _vp, _vp, _vp, C.c_double, _vp, _vp, _ip]),
    "lccrf_frames_create": (C.c_int, [_vp, C.c_int, _vp, C.POINTER(SlamParams), _vp, C.POINTER(_vp)]),
    "lccrf_frames_destroy": (None, [_vp]),
    "lccrf_frames_set_inputs": (C.c_int, [_vp, _vp, _vp, _vp, _vp]),
    "lccrf_frames_set_map_inputs": (C.c_int, [_vp, _vp, _vp, _vp, _vp, C.c_int, _vp, _vp, _vp, _vp, _vp]),
    "lccrf_frames_run": (C.c_int, [_vp]),
    "lccrf_frames_get_outputs": (C.c_int, [_vp, _vp, _vp]),
    "lccrf_frames_submit_map": (C.c_int, [_vp, C.c_int, _vp, _vp, _vp, C.c_int, _vp, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "lccrf_frames_set_keyframe_keypoints": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, _vp]),
    "lccrf_frames_set_map_inputs_indexed": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int, C.c_int, _vp, _vp, _vp, _vp, _vp]),
    "lccrf_frames_submit_map_indexed": (C.c_int, [_vp, C.c_int, _vp, _vp, _vp, C.c_int, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "lccrf_frames_submit": (C.c_int, [_vp, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp]),
    "lccrf_frames_wait": (C.c_int, [_vp, C.c_int]),
    "lccrf_frames_partition": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "lccrf_frames_get_debug": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "lccrf_frames_debug_counters": (C.c_int, [_vp, C.c_int, _vp]),
    "lccrf_frames_algorithmic_bytes": (C.c_int, [_vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "lccrf_images_create": (C.c_int, [_vp, C.c_int, _vp, _vp, C.c_int, C.c_int, C.c_int, C.POINTER(ImageKernel), C.POINTER(_vp)]),
    "lccrf_images_destroy": (None, [_vp]),
    "lccrf_images_set_inputs": (C.c_int, [_vp, _vp, C.c_int, _vp]),
    "lccrf_images_set_inputs_from_label": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_float, _vp, _vp]),
    "lccrf_images_run": (C.c_int, [_vp, C.c_int, C.c_float]),
    "lccrf_images_get_outputs": (C.c_int, [_vp, _vp, _vp]),
    "lccrf_images_vertices": (C.c_int, [_vp, _vp]),
    "lccrf_map_create": (C.c_int, [_vp, C.c_int, C.POINTER(_vp)]),
    "lccrf_map_destroy": (None, [_vp]),
    "lccrf_map_apply": (C.c_int, [_vp, _vp]),
    "lccrf_map_set_observations": (C.c_int, [_vp, C.c_int, C.c_int, _vp, _vp]),
    "lccrf_map_reserve_observations": (C.c_int, [_vp, C.c_longlong]),
    "lccrf_map_sizes": (C.c_int, [_vp, _ip, _ip, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]),
    "lccrf_map_export": (C.c_int, [_vp, C.c_int, _vp, _vp, _vp, _vp, C.c_longlong, _vp]),
    "lccrf_frames_set_visible": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "lccrf_frames_submit_visible": (C.c_int, [_vp, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "lccrf_frames_set_prior": (C.c_int, [_vp, C.c_int, _vp, _vp]),
    "lccrf_frames_set_partition_outputs": (C.c_int, [_vp, C.c_int, _vp, _vp, _vp, _vp, _vp]),
    "lccrf_snapshot_writer_open": (C.c_int, [C.c_char_p, C.c_int, C.POINTER(_vp)]),
    "lccrf_snapshot_write_frame": (C.c_int, [_vp, C.c_longlong, C.c_double, C.c_int, _vp, _vp, _vp, _vp, C.c_int, _vp, _vp, _vp, _vp, _vp]),
    "lccrf_snapshot_writer_close": (C.c_int, [_vp]),
    "lccrf_snapshot_reader_open": (C.c_int, [C.c_char_p, C.POINTER(_vp)]),
    "lccrf_snapshot_reader_close": (None, [_vp]),
    "lccrf_snapshot_num_frames": (C.c_int, [_vp]),
    "lccrf_snapshot_truncated": (C.c_int, [_vp]),
    "lccrf_snapshot_frame_info": (C.c_int, [_vp, C.c_int, _vp]),
    "lccrf_snapshot_read_frame": (C.c_int, [_vp, C.c_int, _vp, _vp, _vp, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp]),
}

# names of the eight long-row splat counters (lccrf_lattice_debug_counters, lccrf_frames_debug_counters)
_SCAN_COUNTERS = ("long_rows", "chunks", "pieces", "tickets", "rec_fast", "rec_cross", "rec_fallback", "rec_zero")

_lib = None


def load_library() -> C.CDLL:
    """dlopen liblccrf.so and bind every declared symbol.  Raises if the library is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise LccrfError(f"{LIB_PATH} is missing: run __graft_entry__.build() (there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def _ptr(a):
    return None if a is None else a.ctypes.data


def _arr(a, dtype):
    return None if a is None else np.ascontiguousarray(a, dtype=dtype)


_libm = None


def _logf(x) -> np.float32:
    """glibc logf -- what std::log(float) resolves to in src/Tracking.cc's translation unit."""
    global _libm
    if _libm is None:
        _libm = C.CDLL("libm.so.6")
        _libm.logf.restype = C.c_float
        _libm.logf.argtypes = [C.c_float]
    return np.float32(_libm.logf(C.c_float(float(x))))


def label_energies(L: int, conf: float) -> np.ndarray:
    """{u, n, p} of densecrf3d.h:109-114 for one shared confidence: -log(1/M), -log((1-c)/(M-1)), -log(c)."""
    f = np.float32
    return np.array([-_logf(f(1.0) / f(L)), -_logf((f(1.0) - f(conf)) / f(L - 1)), -_logf(f(conf))], dtype=np.float32)


class Context:
    """lccrf_ctx: one per GPU."""

    def __init__(self, device: int = 0, stream: int | None = None):
        self.lib = load_library()
        h = _vp()
        self._check(self.lib.lccrf_ctx_create(device, C.byref(h)))
        self.h = h
        self.device = device
        self._children = weakref.WeakSet()  # handles created from this context: closed before the context goes
        if stream is not None:
            self._check(self.lib.lccrf_ctx_set_stream(self.h, _vp(stream)))

    def _check(self, rc: int):
        if rc != 0:
            raise LccrfError(f"liblccrf error {rc}: {self.lib.lccrf_last_error().decode()}")

    def close(self):
        if getattr(self, "h", None):
            for child in list(getattr(self, "_children", ())):
                try:
                    child.close()
                except Exception:
                    pass
            self.lib.lccrf_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sync(self):
        self._check(self.lib.lccrf_ctx_sync(self.h))

    def set_option(self, name: str, value: int):
        self._check(self.lib.lccrf_ctx_set_option(self.h, name.encode(), value))

    def profile_report(self) -> dict:
        """{kernel name: (launches, total_ms)} since profiling was switched on; clears the records."""
        buf = C.create_string_buffer(1 << 16)
        n = self.lib.lccrf_ctx_profile_report(self.h, buf, len(buf))
        if n < 0:
            self._check(n)
        out = {}
        for line in buf.value.decode().splitlines():
            name, cnt, ms = line.split()
            out[name] = (int(cnt), float(ms))
        return out

    @property
    def kernel_launches(self) -> int:
        return int(self.lib.lccrf_ctx_kernel_launches(self.h))

    def build_scratch_in_use(self) -> int:
        """slots of the lattice-build hash scratch that are not empty (0 between builds); synchronises"""
        n = C.c_longlong(0)
        self._check(self.lib.lccrf_ctx_build_scratch_in_use(self.h, C.byref(n)))
        return n.value

    # ---- free functions ----
    def exp_and_normalize(self, x, scale: float, relax: float = 1.0, prev=None) -> np.ndarray:
        x = _arr(x, np.float32)
        N, L = x.shape
        out = _arr(prev, np.float32).copy() if prev is not None else np.zeros_like(x)
        self._check(self.lib.lccrf_exp_and_normalize(self.h, _ptr(out), _ptr(x), N, L, scale, relax))
        return out

    def map_point_unary(self, snap):
        N = snap.n
        ob, er, de = (np.empty(N, dtype=np.float32) for _ in range(3))
        self._check(self.lib.lccrf_map_point_unary(
            self.h, N, _ptr(snap.xyz), _ptr(snap.obs_ptr), _ptr(snap.obs_kf), _ptr(snap.obs_uv),
            snap.kf_pose.shape[0], _ptr(snap.kf_pose), _ptr(snap.kf_intr), _ptr(snap.kf_bounds),
            _ptr(ob), _ptr(er), _ptr(de)))
        return ob, er, de

    def rough_classify(self, observs, error, depth, prm: SlamParams, p4=None) -> np.ndarray:
        observs, error, depth = (_arr(a, np.float32) for a in (observs, error, depth))
        p4 = _arr(p4, np.float64)
        lab = np.empty(observs.size, dtype=np.int16)
        self._check(self.lib.lccrf_rough_classify(self.h, observs.size, _ptr(observs), _ptr(error), _ptr(depth),
                                                  _ptr(p4), C.byref(prm), _ptr(lab)))
        return lab


    def epipolar_prior(self, fid1, pt1, pt2, F, u_gamma, stdev_gamma, n_feat=0):
        """GetFeature2EpipolarDis (Tracking.cc:2030-2047): returns (dis[M], prob[M], dis_by_fid[n_feat], prob_by_fid[n_feat])."""
        pt1, pt2 = _arr(pt1, np.float32), _arr(pt2, np.float32)
        M = pt1.shape[0]
        fid = _arr(fid1, np.int32) if fid1 is not None else None
        F9 = np.ascontiguousarray(F, dtype=np.float64).reshape(9)
        dis, prob = np.empty(M, np.float64), np.empty(M, np.float64)
        dbf, pbf = np.empty(n_feat, np.float64), np.empty(n_feat, np.float64)
        self._check(self.lib.lccrf_epipolar_prior(self.h, M, _ptr(fid), _ptr(pt1), _ptr(pt2), _ptr(F9), u_gamma, stdev_gamma,
                                                  n_feat, _ptr(dbf) if n_feat and fid is not None else None,
                                                  _ptr(pbf) if n_feat and fid is not None else None, _ptr(dis), _ptr(prob)))
        return dis, prob, dbf, pbf

    def bf_match(self, desc_q, desc_t, ratio=0.6, want_knn=True):
        """BfMatch (Tracking.cc:1747-1766): returns (match[nq], knn[nq,4] or None, n_match)."""
        dq = np.ascontiguousarray(desc_q, dtype=np.uint8).reshape(-1, 32)
        dt = np.ascontiguousarray(desc_t, dtype=np.uint8).reshape(-1, 32)
        match = np.empty(dq.shape[0], np.int32)
        knn = np.empty((dq.shape[0], 4), np.int32) if want_knn else None
        n = C.c_int(0)
        self._check(self.lib.lccrf_bf_match(self.h, dq.shape[0], _ptr(dq), dt.shape[0], _ptr(dt), ratio, _ptr(match),
                                            _ptr(knn), C.byref(n)))
        return match, knn, n.value

    def bf_match_batch(self, q_ptr, desc_q, t_ptr, desc_t, ratio=0.6, want_knn=False):
        q_ptr, t_ptr = _arr(q_ptr, np.int32), _arr(t_ptr, np.int32)
        dq = np.ascontiguousarray(desc_q, dtype=np.uint8).reshape(-1, 32)
        dt = np.ascontiguousarray(desc_t, dtype=np.uint8).reshape(-1, 32)
        match = np.empty(dq.shape[0], np.int32)
        knn = np.empty((dq.shape[0], 4), np.int32) if want_knn else None
        n = C.c_int(0)
        self._check(self.lib.lccrf_bf_match_batch(self.h, q_ptr.size - 1, _ptr(q_ptr), _ptr(dq), _ptr(t_ptr), _ptr(dt), ratio,
                                                  _ptr(match), _ptr(knn), C.byref(n)))
        return match, knn, n.value


class Lattice:
    """lccrf_lattice: PermutohedralLatticeCPU replacement."""

    def __init__(self, ctx: Context, features):
        self.ctx = ctx
        f = _arr(features, np.float32)
        self.N, self.d = f.shape
        h = _vp()
        ctx._check(ctx.lib.lccrf_lattice_create(ctx.h, _ptr(f), self.d, self.N, C.byref(h)))
        self.h = h
        ctx._children.add(self)
        v = C.c_int()
        ctx._check(ctx.lib.lccrf_lattice_sizes(self.h, None, None, C.byref(v)))
        self.V = v.value

    def export(self):
        D = self.d + 1
        off = np.empty((self.N, D), dtype=np.int32)
        bary = np.empty((self.N, D), dtype=np.float32)
        nbr = np.empty((D, self.V, 2), dtype=np.int32)
        self.ctx._check(self.ctx.lib.lccrf_lattice_export(self.h, _ptr(off), _ptr(bary), _ptr(nbr)))
        return off, bary, nbr

    def filter(self, x) -> np.ndarray:
        x = _arr(x, np.float32)
        L = x.size // self.N if self.N else 1
        out = np.empty_like(x)
        self.ctx._check(self.ctx.lib.lccrf_lattice_filter(self.h, _ptr(out), _ptr(x), L))
        return out

    def filter_window(self, x, L, in_offset=0, out_offset=0, in_size=-1, out_size=-1) -> np.ndarray:
        """compute() with its windowing arguments: x holds the in_size input points, the result the out_size points"""
        x = _arr(x, np.float32)
        n_out = self.N - out_offset if out_size == -1 else out_size
        out = np.empty((max(n_out, 0), L), dtype=np.float32)
        self.ctx._check(self.ctx.lib.lccrf_lattice_filter_window(self.h, _ptr(out), _ptr(x), L, in_offset, out_offset, in_size, out_size))
        return out

    def debug_counters(self):
        """long-row splat counters; rec_* accumulate over the filter calls since the lattice was built"""
        out = np.zeros(8, dtype=np.int32)
        self.ctx._check(self.ctx.lib.lccrf_lattice_debug_counters(self.h, _ptr(out)))
        return dict(zip(_SCAN_COUNTERS, out.tolist()))

    def close(self):
        if getattr(self, "h", None):
            self.ctx.lib.lccrf_lattice_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class DenseCRF:
    """lccrf_crf: DenseCRF3D<M> / DenseCRFCPU<M> replacement (method names follow densecrf_base.h)."""

    def __init__(self, ctx: Context, N: int, L: int):
        self.ctx, self.N, self.L = ctx, N, L
        h = _vp()
        ctx._check(ctx.lib.lccrf_crf_create(ctx.h, N, L, C.byref(h)))
        self.h = h
        ctx._children.add(self)

    def setUnaryEnergy(self, unary):
        u = _arr(unary, np.float32)
        self.ctx._check(self.ctx.lib.lccrf_crf_set_unary(self.h, _ptr(u)))

    def setUnaryEnergyFromLabel(self, label, confidence=0.5, energies=None):
        lab = _arr(label, np.int16)
        if energies is None:
            energies = label_energies(self.L, confidence)
        n_en = np.full(self.L, energies[1], dtype=np.float32)
        p_en = np.full(self.L, energies[2], dtype=np.float32)
        self.ctx._check(self.ctx.lib.lccrf_crf_set_unary_from_label(self.h, _ptr(lab), float(energies[0]), _ptr(n_en), _ptr(p_en)))

    def SetUnaryEnergtForPositiveNode(self, idx, m, value):
        self.ctx._check(self.ctx.lib.lccrf_crf_set_unary_entry(self.h, idx, m, value))

    def addPairwiseEnergy(self, features, w: float):
        f = _arr(features, np.float32)
        self.ctx._check(self.ctx.lib.lccrf_crf_add_potts(self.h, _ptr(f), f.shape[1], w))

    def addPairwiseFromImage(self, W, H, w, posdev, img=None, featuredev=0.0):
        if img is None:
            self.ctx._check(self.ctx.lib.lccrf_crf_add_potts_image(self.h, W, H, w, posdev, None, 0, 2, 0.0))
        else:
            is_u8 = img.dtype == np.uint8
            a = np.ascontiguousarray(img) if is_u8 else _arr(img, np.float32)
            F = 2 + a.size // (W * H)
            self.ctx._check(self.ctx.lib.lccrf_crf_add_potts_image(self.h, W, H, w, posdev, _ptr(a), int(is_u8), F, featuredev))

    def potts_vertices(self, k: int) -> int:
        v = C.c_int()
        self.ctx._check(self.ctx.lib.lccrf_crf_potts_vertices(self.h, k, C.byref(v)))
        return v.value

    def potts_apply(self, k, out, inp):
        out = _arr(out, np.float32).copy()
        inp = _arr(inp, np.float32)
        tmp = np.empty_like(out)
        self.ctx._check(self.ctx.lib.lccrf_crf_potts_apply(self.h, k, _ptr(out), _ptr(inp), _ptr(tmp)))
        return out, tmp

    def startInference(self):
        self.ctx._check(self.ctx.lib.lccrf_crf_start(self.h))

    def stepInference(self, relax=1.0):
        self.ctx._check(self.ctx.lib.lccrf_crf_step(self.h, relax))

    def inference(self, n_iterations, with_map=False, relax=1.0):
        self.ctx._check(self.ctx.lib.lccrf_crf_inference(self.h, n_iterations, int(with_map), relax))

    def buildMap(self):
        self.ctx._check(self.ctx.lib.lccrf_crf_build_map(self.h))

    def getMap(self):
        p = self.ctx.lib.lccrf_crf_map(self.h)
        if not p:
            return None
        return np.ctypeslib.as_array(p, shape=(max(self.N, 1),))[:self.N].copy()

    def getProbability(self):
        p = self.ctx.lib.lccrf_crf_prob(self.h)
        if not p:
            return None
        return np.ctypeslib.as_array(p, shape=(max(self.N, 1) * self.L,))[:self.N * self.L].copy().reshape(self.N, self.L)

    def close(self):
        if getattr(self, "h", None):
            self.ctx.lib.lccrf_crf_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MapDelta(C.Structure):
    """lccrf_map_delta: the map changes of one step (include/lccrf.h).  Build with MapDelta.make(...): the numpy arrays
    are converted once and kept alive by the object; nothing is copied per use."""
    _fields_ = [("kf_first", C.c_int), ("kf_count", C.c_int), ("kf_pose", _vp), ("kf_intr", _vp), ("kf_bounds", _vp),
                ("kf_keypoints", _vp), ("n_pose", C.c_int), ("pose_kf", _vp), ("pose", _vp), ("n_xyz", C.c_int),
                ("xyz_id", _vp), ("xyz", _vp), ("n_erase", C.c_int), ("erase_pt", _vp), ("erase_kf", _vp),
                ("n_bad", C.c_int), ("bad_pt", _vp), ("n_add", C.c_int), ("add_pt", _vp), ("add_kf", _vp), ("add_fid", _vp),
                ("n_erase_seg", C.c_int), ("erase_seg_ptr", _vp), ("n_add_seg", C.c_int), ("add_seg_ptr", _vp)]

    @classmethod
    def make(cls, kf_first=0, kf_pose=None, kf_intr=None, kf_bounds=None, kf_keypoints=None, pose_kf=None, pose=None,
             xyz_id=None, xyz=None, erase_pt=None, erase_kf=None, bad_pt=None, add_pt=None, add_kf=None, add_fid=None,
             erase_seg_ptr=None, add_seg_ptr=None, pin=None) -> "MapDelta":
        """pin: optional callable array -> page-locked copy (bench.py passes a torch pin_memory wrapper)"""
        d = cls()
        keep = []

        def f32(a):
            if a is None:
                return None
            a = np.ascontiguousarray(a, dtype=np.float32)
            a = pin(a) if pin else a
            keep.append(a)
            return a

        def i32(a):
            if a is None:
                return None
            a = np.ascontiguousarray(a, dtype=np.int32)
            a = pin(a) if pin else a
            keep.append(a)
            return a

        kf_pose, kf_intr, kf_bounds, kf_keypoints, pose, xyz = (f32(a) for a in (kf_pose, kf_intr, kf_bounds, kf_keypoints, pose, xyz))
        pose_kf, xyz_id, erase_pt, erase_kf, bad_pt, add_pt, add_kf, add_fid = (
            i32(a) for a in (pose_kf, xyz_id, erase_pt, erase_kf, bad_pt, add_pt, add_kf, add_fid))
        d.kf_first = int(kf_first)
        d.kf_count = 0 if kf_pose is None else int(kf_pose.size // 12)
        d.kf_pose, d.kf_intr, d.kf_bounds, d.kf_keypoints = _ptr(kf_pose), _ptr(kf_intr), _ptr(kf_bounds), _ptr(kf_keypoints)
        d.n_pose = 0 if pose is None else int(pose.size // 12)
        d.pose_kf, d.pose = _ptr(pose_kf), _ptr(pose)
        d.n_xyz = 0 if xyz is None else int(xyz.size // 3)
        d.xyz_id, d.xyz = _ptr(xyz_id), _ptr(xyz)
        d.n_erase = 0 if erase_pt is None else int(erase_pt.size)
        d.erase_pt, d.erase_kf = _ptr(erase_pt), _ptr(erase_kf)
        d.n_bad = 0 if bad_pt is None else int(bad_pt.size)
        d.bad_pt = _ptr(bad_pt)
        d.n_add = 0 if add_pt is None else int(add_pt.size)
        d.add_pt, d.add_kf, d.add_fid = _ptr(add_pt), _ptr(add_kf), _ptr(add_fid)
        d._seg = [None if a is None else np.ascontiguousarray(a, dtype=np.int32) for a in (erase_seg_ptr, add_seg_ptr)]
        d.n_erase_seg = 0 if d._seg[0] is None else int(d._seg[0].size - 1)
        d.n_add_seg = 0 if d._seg[1] is None else int(d._seg[1].size - 1)
        d.erase_seg_ptr, d.add_seg_ptr = _ptr(d._seg[0]), _ptr(d._seg[1])
        if pose_kf is not None and pose_kf.size != d.n_pose or xyz_id is not None and xyz_id.size != d.n_xyz:
            raise LccrfError("MapDelta: id arrays must match their value arrays")
        if d.n_erase and (erase_kf is None or erase_kf.size != d.n_erase):
            raise LccrfError("MapDelta: erase_pt / erase_kf sizes differ")
        if d.n_add and (add_kf is None or add_fid is None or add_kf.size != d.n_add or add_fid.size != d.n_add):
            raise LccrfError("MapDelta: add_pt / add_kf / add_fid sizes differ")
        d._keep = keep
        return d

    @property
    def nbytes(self) -> int:
        """bytes this delta moves host -> device"""
        return int(sum(a.nbytes for a in self._keep))


class Map:
    """lccrf_map: the device-resident SLAM map (keyframes, map points, observation lists)."""

    def __init__(self, ctx: Context, kp_stride: int):
        self.ctx, self.kp_stride = ctx, int(kp_stride)
        h = _vp()
        ctx._check(ctx.lib.lccrf_map_create(ctx.h, self.kp_stride, C.byref(h)))
        self.h = h
        ctx._children.add(self)

    def apply(self, delta: MapDelta = None, **kw):
        d = delta if delta is not None else MapDelta.make(**kw)
        self.ctx._check(self.ctx.lib.lccrf_map_apply(self.h, C.byref(d)))

    def set_observations(self, obs_ptr, obs_ref, pt_first=0):
        obs_ptr = _arr(obs_ptr, np.int32)
        obs_ref = _arr(obs_ref, np.int32)
        assert obs_ref.ndim == 2 and obs_ref.shape[1] == 2
        self.ctx._check(self.ctx.lib.lccrf_map_set_observations(self.h, int(pt_first), int(obs_ptr.size - 1), _ptr(obs_ptr), _ptr(obs_ref)))

    def reserve_observations(self, entries: int):
        self.ctx._check(self.ctx.lib.lccrf_map_reserve_observations(self.h, int(entries)))

    def sizes(self) -> dict:
        nk, npnt = C.c_int(), C.c_int()
        no, pu, pc = C.c_longlong(), C.c_longlong(), C.c_longlong()
        self.ctx._check(self.ctx.lib.lccrf_map_sizes(self.h, C.byref(nk), C.byref(npnt), C.byref(no), C.byref(pu), C.byref(pc)))
        return dict(n_kf=nk.value, n_points=npnt.value, n_obs=no.value, pool_used=pu.value, pool_cap=pc.value)

    def export(self, point_id):
        """observation lists of the given points in the set_map_inputs layout: (obs_ptr, obs_kf, obs_uv, xyz)"""
        ids = _arr(point_id, np.int32)
        n = int(ids.size)
        ptr = np.zeros(n + 1, np.int32)
        self.ctx._check(self.ctx.lib.lccrf_map_export(self.h, n, _ptr(ids), _ptr(ptr), None, None, 0, None))
        nnz = int(ptr[-1])
        kf, uv, xyz = np.empty(nnz, np.int32), np.empty((nnz, 2), np.float32), np.empty((n, 3), np.float32)
        self.ctx._check(self.ctx.lib.lccrf_map_export(self.h, n, _ptr(ids), _ptr(ptr), _ptr(kf), _ptr(uv), nnz, _ptr(xyz)))
        return ptr, kf, uv, xyz

    def close(self):
        if getattr(self, "h", None):
            self.ctx.lib.lccrf_map_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Frames:
    """lccrf_frames: B independent per-frame CRF problems (Tracking.cc:1871-1930) in one launch sequence."""

    def __init__(self, ctx: Context, n_points, prm: SlamParams | None = None, energies=None):
        self.ctx = ctx
        self.prm = prm or SlamParams.make()
        n_points = np.asarray(n_points, dtype=np.int64)
        self.B = int(n_points.size)
        self.prob_ptr = np.zeros(self.B + 1, dtype=np.int32)
        np.cumsum(n_points, out=self.prob_ptr[1:])
        self.NT = int(self.prob_ptr[-1])
        self.energies = label_energies(2, self.prm.confidence) if energies is None else _arr(energies, np.float32)
        h = _vp()
        ctx._check(ctx.lib.lccrf_frames_create(ctx.h, self.B, _ptr(self.prob_ptr), C.byref(self.prm), _ptr(self.energies), C.byref(h)))
        self.h = h
        ctx._children.add(self)

    def set_inputs(self, observs, error, depth, kp2d):
        a = [_arr(x, np.float32) for x in (observs, error, depth, kp2d)]
        self._keep = a
        self.ctx._check(self.ctx.lib.lccrf_frames_set_inputs(self.h, *[_ptr(x) for x in a]))

    def set_map_inputs(self, xyz, obs_ptr, obs_kf, obs_uv, kf_pose, kf_intr, kf_bounds, kp2d, kf_ptr=None):
        xyz, obs_uv, kf_pose, kf_intr, kf_bounds, kp2d = (_arr(x, np.float32) for x in (xyz, obs_uv, kf_pose, kf_intr, kf_bounds, kp2d))
        obs_ptr, obs_kf, kf_ptr = _arr(obs_ptr, np.int32), _arr(obs_kf, np.int32), _arr(kf_ptr, np.int32)
        self._keep = [xyz, obs_ptr, obs_kf, obs_uv, kf_pose, kf_intr, kf_bounds, kp2d, kf_ptr]
        self.ctx._check(self.ctx.lib.lccrf_frames_set_map_inputs(
            self.h, _ptr(xyz), _ptr(obs_ptr), _ptr(obs_kf), _ptr(obs_uv), kf_pose.shape[0], _ptr(kf_pose),
            _ptr(kf_intr), _ptr(kf_bounds), _ptr(kp2d), _ptr(kf_ptr)))

    def run(self):
        self.ctx._check(self.ctx.lib.lccrf_frames_run(self.h))

    def get_outputs(self, map_out=None, prob_out=None, want_prob=True):
        mp = np.empty(self.NT, dtype=np.int16) if map_out is None else map_out
        pr = (np.empty((self.NT, 2), dtype=np.float32) if prob_out is None else prob_out) if want_prob else None
        self.ctx._check(self.ctx.lib.lccrf_frames_get_outputs(self.h, _ptr(mp), _ptr(pr)))
        return mp, pr

    def submit_map(self, slot, xyz, obs_ptr, obs_kf, obs_uv, kf_pose, kf_intr, kf_bounds, kp2d, kf_ptr, map_out, prob_out):
        """Pipelined step through HOST buffers (no conversion or copy here: pass contiguous, ideally pinned, arrays;
        obs_kf may be int32 or uint16).  Returns immediately; call wait(slot) before reading map_out / prob_out."""
        kb = obs_kf.dtype.itemsize
        assert obs_kf.dtype in (np.int32, np.uint16)
        self.ctx._check(self.ctx.lib.lccrf_frames_submit_map(
            self.h, slot, _ptr(xyz), _ptr(obs_ptr), _ptr(obs_kf), kb, _ptr(obs_uv), kf_pose.shape[0], _ptr(kf_pose),
            _ptr(kf_intr), _ptr(kf_bounds), _ptr(kp2d), _ptr(kf_ptr), _ptr(map_out), _ptr(prob_out)))

    def set_keyframe_keypoints(self, kp_table, kf_first=0):
        """Resident keyframe keypoints (KeyFrame::mvKeysUn): kp_table [n_kf][stride][2] float32 for keyframes
        [kf_first, kf_first + n_kf).  Uploaded once per keyframe, not per step."""
        kp_table = _arr(kp_table, np.float32)
        assert kp_table.ndim == 3 and kp_table.shape[2] == 2
        self.ctx._check(self.ctx.lib.lccrf_frames_set_keyframe_keypoints(self.h, kf_first, kp_table.shape[0], kp_table.shape[1], _ptr(kp_table)))

    def set_map_inputs_indexed(self, xyz, obs_ptr, obs_ref, kf_pose, kf_intr, kf_bounds, kp2d, kf_ptr=None):
        """set_map_inputs with {keyframe, feature index} pairs (obs_ref [nnz][2], uint16 or int32) instead of
        (obs_kf, obs_uv): keypoints come from the resident table."""
        xyz, kf_pose, kf_intr, kf_bounds, kp2d = (_arr(x, np.float32) for x in (xyz, kf_pose, kf_intr, kf_bounds, kp2d))
        obs_ptr, kf_ptr = _arr(obs_ptr, np.int32), _arr(kf_ptr, np.int32)
        obs_ref = np.ascontiguousarray(obs_ref)
        assert obs_ref.dtype in (np.int32, np.uint16) and obs_ref.ndim == 2 and obs_ref.shape[1] == 2
        self._keep = [xyz, obs_ptr, obs_ref, kf_pose, kf_intr, kf_bounds, kp2d, kf_ptr]
        self.ctx._check(self.ctx.lib.lccrf_frames_set_map_inputs_indexed(
            self.h, _ptr(xyz), _ptr(obs_ptr), _ptr(obs_ref), obs_ref.dtype.itemsize, kf_pose.shape[0], _ptr(kf_pose),
            _ptr(kf_intr), _ptr(kf_bounds), _ptr(kp2d), _ptr(kf_ptr)))

    def submit_map_indexed(self, slot, xyz, obs_ptr, obs_ref, kf_pose, kf_intr, kf_bounds, kp2d, kf_ptr, map_out, prob_out):
        """Pipelined step through HOST buffers with indexed observations (4 bytes per observation with uint16 pairs)."""
        assert obs_ref.dtype in (np.int32, np.uint16) and obs_ref.ndim == 2 and obs_ref.shape[1] == 2
        self.ctx._check(self.ctx.lib.lccrf_frames_submit_map_indexed(
            self.h, slot, _ptr(xyz), _ptr(obs_ptr), _ptr(obs_ref), obs_ref.dtype.itemsize, kf_pose.shape[0], _ptr(kf_pose),
            _ptr(kf_intr), _ptr(kf_bounds), _ptr(kp2d), _ptr(kf_ptr), _ptr(map_out), _ptr(prob_out)))

    def submit(self, slot, observs, error, depth, kp2d, map_out, prob_out):
        self.ctx._check(self.ctx.lib.lccrf_frames_submit(self.h, slot, _ptr(observs), _ptr(error), _ptr(depth), _ptr(kp2d),
                                                          _ptr(map_out), _ptr(prob_out)))

    def wait(self, slot):
        self.ctx._check(self.ctx.lib.lccrf_frames_wait(self.h, slot))

    def set_visible(self, mp: "Map", point_id, kp2d, delta: MapDelta = None, kf_ptr=None):
        """frame points = ids of the resident map's points (+ optional delta applied first); follow with run()"""
        ids, kp, kfp = _arr(point_id, np.int32), _arr(kp2d, np.float32), _arr(kf_ptr, np.int32)
        self.ctx._check(self.ctx.lib.lccrf_frames_set_visible(self.h, mp.h, C.byref(delta) if delta is not None else None,
                                                            _ptr(ids), _ptr(kp), _ptr(kfp)))

    def submit_visible(self, slot, mp: "Map", point_id, kp2d, map_out, prob_out, delta: MapDelta = None, kf_ptr=None):
        """pipelined step against the resident map through HOST buffers (no conversion here: pass contiguous int32 /
        float32 arrays, ideally pinned; they and the delta must stay alive until wait(slot))"""
        assert point_id.dtype == np.int32 and kp2d.dtype == np.float32 and (kf_ptr is None or kf_ptr.dtype == np.int32)
        self._vis_keep = getattr(self, "_vis_keep", {})
        self._vis_keep[slot] = (point_id, kp2d, delta, kf_ptr)
        self.ctx._check(self.ctx.lib.lccrf_frames_submit_visible(
            self.h, slot, mp.h, C.byref(delta) if delta is not None else None, _ptr(point_id), _ptr(kp2d), _ptr(kf_ptr),
            _ptr(map_out), _ptr(prob_out)))

    def set_prior(self, slot, p4=None, has_prior=None):
        """epipolar prior p4 [NT] float64 (+ per-problem flags [B] uint8) of the next run / submission of `slot`"""
        p4 = _arr(p4, np.float64)
        hp = _arr(has_prior, np.uint8)
        self._prior_keep = getattr(self, "_prior_keep", {})
        self._prior_keep[slot] = (p4, hp)
        self.ctx._check(self.ctx.lib.lccrf_frames_set_prior(self.h, slot, _ptr(p4), _ptr(hp)))

    def set_partition_outputs(self, slot, fid=None, enable=True):
        """label-application lists delivered by submit_*(slot); returns the dict of host arrays they land in"""
        self._part_keep = getattr(self, "_part_keep", {})
        if not enable:
            self._part_keep.pop(slot, None)
            self.ctx._check(self.ctx.lib.lccrf_frames_set_partition_outputs(self.h, slot, None, None, None, None, None))
            return None
        out = dict(fid=_arr(fid, np.int32), dyn_ptr=np.zeros(self.B + 1, np.int32), dyn=np.zeros(max(self.NT, 1), np.int32),
                   stat_ptr=np.zeros(self.B + 1, np.int32), stat=np.zeros(max(self.NT, 1), np.int32))
        self._part_keep[slot] = out
        self.ctx._check(self.ctx.lib.lccrf_frames_set_partition_outputs(
            self.h, slot, _ptr(out["fid"]), _ptr(out["dyn_ptr"]), _ptr(out["dyn"]), _ptr(out["stat_ptr"]), _ptr(out["stat"])))
        return out

    def partition(self, fid=None):
        """Label application (Tracking.cc:1945-1955): per-problem lists of moving / static points in point order.
        Returns (dyn_ptr, dyn_list, stat_ptr, stat_list); list elements are fid[i] when fid is given, else the
        point's index inside its problem."""
        fid = _arr(fid, np.int32)
        if fid is not None and fid.size != self.NT:
            raise LccrfError("fid must have one entry per point")
        dyn_ptr, stat_ptr = np.empty(self.B + 1, dtype=np.int32), np.empty(self.B + 1, dtype=np.int32)
        dyn, stat = np.empty(self.NT, dtype=np.int32), np.empty(self.NT, dtype=np.int32)
        self.ctx._check(self.ctx.lib.lccrf_frames_partition(self.h, _ptr(fid), _ptr(dyn_ptr), _ptr(dyn), _ptr(stat_ptr), _ptr(stat)))
        return dyn_ptr, dyn[:dyn_ptr[-1]].copy(), stat_ptr, stat[:stat_ptr[-1]].copy()

    def get_debug(self):
        lab = np.empty(self.NT, dtype=np.int16)
        ob, er, de = (np.empty(self.NT, dtype=np.float32) for _ in range(3))
        V = np.empty((self.B, 2), dtype=np.int32)
        self.ctx._check(self.ctx.lib.lccrf_frames_get_debug(self.h, _ptr(lab), _ptr(ob), _ptr(er), _ptr(de), _ptr(V)))
        return dict(init_label=lab, observs=ob, error=er, depth=de, V=V)

    def debug_counters(self, k):
        out = np.zeros(8, dtype=np.int32)
        self.ctx._check(self.ctx.lib.lccrf_frames_debug_counters(self.h, k, _ptr(out)))
        return dict(zip(_SCAN_COUNTERS, out.tolist()))

    def algorithmic_bytes(self):
        t, i, u = C.c_double(), C.c_double(), C.c_double()
        self.ctx._check(self.ctx.lib.lccrf_frames_algorithmic_bytes(self.h, C.byref(t), C.byref(i), C.byref(u)))
        return dict(total=t.value, per_iteration=i.value, unary=u.value)

    def close(self):
        if getattr(self, "h", None):
            self.ctx.lib.lccrf_frames_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Images:
    """lccrf_images: B full-image DenseCRFs (DenseCRFCPU<M> + PottsPotentialCPU<M,F>::FromImage) in one launch sequence.

    sizes: [(W, H), ...] per image; kernels: [(F, w, posdev, featuredev), ...] in addPairwiseEnergy order (F = 2 Gaussian,
    F = C + 2 bilateral); C: channels per pixel.  Arrays are concatenated over the images in order."""

    def __init__(self, ctx: Context, sizes, L: int, kernels, C: int = 3):
        self.ctx, self.L, self.C = ctx, int(L), int(C)
        wh = np.asarray(sizes, dtype=np.int32).reshape(-1, 2)
        self.W, self.H = np.ascontiguousarray(wh[:, 0]), np.ascontiguousarray(wh[:, 1])
        self.B = int(wh.shape[0])
        self.ptr = np.zeros(self.B + 1, dtype=np.int64)
        np.cumsum(self.W.astype(np.int64) * self.H, out=self.ptr[1:])
        self.NT = int(self.ptr[-1])
        self.K = len(kernels)
        ks = (ImageKernel * max(self.K, 1))(*[ImageKernel(int(F), w, posdev, fd) for F, w, posdev, fd in kernels])
        h = _vp()
        ctx._check(ctx.lib.lccrf_images_create(ctx.h, self.B, _ptr(self.W), _ptr(self.H), self.C, self.L, self.K, ks, _byref(h)))
        self.h = h
        ctx._children.add(self)

    def _cat(self, a, dtype=None):
        if isinstance(a, (list, tuple)):
            a = np.concatenate([np.asarray(x).reshape(-1) for x in a]) if a else np.zeros(0, dtype or np.float32)
        return None if a is None else np.ascontiguousarray(a, dtype=dtype)

    def set_inputs(self, img, unary=None, label=None, energies=None):
        """img: [NT, C] (or a list per image) uint8 or float32, None without bilateral kernels.  Either unary [NT, L]
        (setUnaryEnergy) or label [NT] with energies = {u, n, p} of label_energies, or (u, n_en[L], p_en[L])."""
        img = self._cat(img)
        u8 = img is None or img.dtype == np.uint8
        if img is not None and not u8:
            img = np.ascontiguousarray(img, dtype=np.float32)
        if unary is not None:
            u = self._cat(unary, np.float32)
            self.ctx._check(self.ctx.lib.lccrf_images_set_inputs(self.h, _ptr(img), int(u8), _ptr(u)))
            return
        lab = self._cat(label, np.int16)
        if energies is None or len(energies) == 3 and np.ndim(energies[1]) == 0:
            e = label_energies(self.L, 0.5) if energies is None else np.asarray(energies, np.float32)
            u_en, n_en, p_en = float(e[0]), np.full(self.L, e[1], np.float32), np.full(self.L, e[2], np.float32)
        else:
            u_en, n_en, p_en = float(energies[0]), _arr(energies[1], np.float32), _arr(energies[2], np.float32)
        self.ctx._check(self.ctx.lib.lccrf_images_set_inputs_from_label(self.h, _ptr(img), int(u8), _ptr(lab), u_en,
                                                                        _ptr(n_en), _ptr(p_en)))

    def run(self, T: int, relax: float = 1.0):
        self.ctx._check(self.ctx.lib.lccrf_images_run(self.h, int(T), float(relax)))

    def get_outputs(self, want_prob=True, map_out=None, prob_out=None):
        """(map [NT], prob [NT, L] or None, [(map_b, prob_b), ...] views per image); synchronises"""
        mp = np.empty(self.NT, dtype=np.int16) if map_out is None else map_out
        pr = (np.empty((self.NT, self.L), dtype=np.float32) if prob_out is None else prob_out) if want_prob else None
        self.ctx._check(self.ctx.lib.lccrf_images_get_outputs(self.h, _ptr(mp), _ptr(pr)))
        split = [(mp[a:b], None if pr is None else pr[a:b]) for a, b in zip(self.ptr[:-1], self.ptr[1:])]
        return mp, pr, split

    def vertices(self) -> np.ndarray:
        """[B, K] lattice vertex counts (M_) of the last run"""
        V = np.zeros((self.B, self.K), dtype=np.int32)
        self.ctx._check(self.ctx.lib.lccrf_images_vertices(self.h, _ptr(V)))
        return V

    def close(self):
        if getattr(self, "h", None):
            self.ctx.lib.lccrf_images_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ------------------------------------------------------------------ snapshot / replay files (host only)
class SnapshotInfo(C.Structure):
    _fields_ = [("N", C.c_int), ("nKF", C.c_int), ("nnz", C.c_longlong), ("frame_id", C.c_longlong),
                ("timestamp", C.c_double), ("stored_kf_bytes", C.c_int)]


def _snap_check(lib, rc):
    if rc != 0:
        raise LccrfError(f"liblccrf error {rc}: {lib.lccrf_last_error().decode()}")


class SnapshotWriter:
    """Appends CRF-input frames (the lccrf_frames_set_map_inputs layout + feature ids) to an LCCRFSNP file."""

    def __init__(self, path: str, append: bool = False):
        self.lib = load_library()
        self.h = _vp()
        _snap_check(self.lib, self.lib.lccrf_snapshot_writer_open(os.fsencode(path), int(append), C.byref(self.h)))

    def write(self, snap, frame_id: int = 0, timestamp: float = 0.0, fid=None):
        """snap: any object with xyz, obs_ptr, obs_kf, obs_uv, kf_pose, kf_intr, kf_bounds, kp2d (synth.MapSnapshot)."""
        xyz, ptr, kf, uv = _arr(snap.xyz, np.float32), _arr(snap.obs_ptr, np.int32), _arr(snap.obs_kf, np.int32), _arr(snap.obs_uv, np.float32)
        pose, intr, bnd, kp = (_arr(a, np.float32) for a in (snap.kf_pose, snap.kf_intr, snap.kf_bounds, snap.kp2d))
        fid = _arr(fid, np.int32)
        n = int(xyz.shape[0])
        if ptr.size != n + 1 or kp.size != 2 * n or (fid is not None and fid.size != n):
            raise LccrfError("inconsistent snapshot arrays")
        _snap_check(self.lib, self.lib.lccrf_snapshot_write_frame(
            self.h, int(frame_id), float(timestamp), n, _ptr(xyz), _ptr(ptr), _ptr(kf), _ptr(uv), int(pose.shape[0]),
            _ptr(pose), _ptr(intr), _ptr(bnd), _ptr(kp), _ptr(fid)))

    def close(self):
        if getattr(self, "h", None):
            h, self.h = self.h, None
            _snap_check(self.lib, self.lib.lccrf_snapshot_writer_close(h))

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


class SnapshotFrame:
    """One frame read back from a snapshot file (same attribute names as synth.MapSnapshot)."""

    def __init__(self, info, xyz, obs_ptr, obs_kf, obs_uv, kf_pose, kf_intr, kf_bounds, kp2d, fid):
        self.frame_id, self.timestamp = int(info.frame_id), float(info.timestamp)
        self.xyz, self.obs_ptr, self.obs_kf, self.obs_uv = xyz, obs_ptr, obs_kf, obs_uv
        self.kf_pose, self.kf_intr, self.kf_bounds, self.kp2d, self.fid = kf_pose, kf_intr, kf_bounds, kp2d, fid

    @property
    def n(self):
        return int(self.xyz.shape[0])

    @property
    def nnz(self):
        return int(self.obs_kf.shape[0])


class SnapshotReader:
    """Random access to the frames of an LCCRFSNP file; every read verifies checksum and structure."""

    def __init__(self, path: str):
        self.lib = load_library()
        self.h = _vp()
        _snap_check(self.lib, self.lib.lccrf_snapshot_reader_open(os.fsencode(path), C.byref(self.h)))

    def __len__(self):
        return int(self.lib.lccrf_snapshot_num_frames(self.h))

    @property
    def truncated(self) -> bool:
        return bool(self.lib.lccrf_snapshot_truncated(self.h))

    def info(self, i: int) -> SnapshotInfo:
        inf = SnapshotInfo()
        _snap_check(self.lib, self.lib.lccrf_snapshot_frame_info(self.h, int(i), C.byref(inf)))
        return inf

    def read(self, i: int, kf_dtype=np.int32) -> SnapshotFrame:
        inf = self.info(i)
        n, nnz, nkf = inf.N, int(inf.nnz), inf.nKF
        xyz, ptr = np.empty((n, 3), np.float32), np.empty(n + 1, np.int32)
        kf, uv = np.empty(nnz, kf_dtype), np.empty((nnz, 2), np.float32)
        pose, intr, bnd = np.empty((nkf, 12), np.float32), np.empty((nkf, 4), np.float32), np.empty((nkf, 4), np.float32)
        kp, fid = np.empty((n, 2), np.float32), np.empty(n, np.int32)
        _snap_check(self.lib, self.lib.lccrf_snapshot_read_frame(
            self.h, int(i), _ptr(xyz), _ptr(ptr), _ptr(kf), int(np.dtype(kf_dtype).itemsize), _ptr(uv), _ptr(pose), _ptr(intr),
            _ptr(bnd), _ptr(kp), _ptr(fid)))
        return SnapshotFrame(inf, xyz, ptr, kf, uv, pose, intr, bnd, kp, fid)

    def close(self):
        if getattr(self, "h", None):
            self.lib.lccrf_snapshot_reader_close(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def concat_frames(frames):
    """Concatenate map snapshots / snapshot frames into one batch for Frames.set_map_inputs / submit_map: CSR pointers
    and keyframe indices are rebased, kf_ptr [B+1] names every problem's keyframe slice, fid is carried along."""
    ptr, kf, eo, ko = [np.zeros(1, np.int64)], [], 0, 0
    for s in frames:
        ptr.append(s.obs_ptr[1:].astype(np.int64) + eo)
        kf.append(s.obs_kf.astype(np.int64) + ko)
        eo += int(s.obs_kf.shape[0])
        ko += int(s.kf_pose.shape[0])
    kf_ptr = np.zeros(len(frames) + 1, dtype=np.int32)
    np.cumsum([s.kf_pose.shape[0] for s in frames], out=kf_ptr[1:])
    cat = lambda k, shape: (np.concatenate([getattr(s, k).reshape(shape) for s in frames]) if frames else np.zeros(shape if shape[0] != -1 else (0,) + shape[1:], np.float32))
    out = dict(xyz=cat("xyz", (-1, 3)), obs_ptr=np.concatenate(ptr).astype(np.int32),
               obs_kf=(np.concatenate(kf) if kf else np.zeros(0)).astype(np.int32), obs_uv=cat("obs_uv", (-1, 2)),
               kf_pose=cat("kf_pose", (-1, 12)), kf_intr=cat("kf_intr", (-1, 4)), kf_bounds=cat("kf_bounds", (-1, 4)),
               kp2d=cat("kp2d", (-1, 2)), kf_ptr=kf_ptr)
    if frames and all(getattr(s, "fid", None) is not None for s in frames):
        out["fid"] = np.concatenate([s.fid for s in frames]).astype(np.int32)
    return out
