"""Host-side mirror of go-muse's exported API over the muse_b200 C ABI (ctypes).

The reference is a Go package; there is no Go toolchain in this image, so this module
plays the part of the Go facade in `go-muse_b200/go/` for tests and benchmarks: the same
names, argument meaning and error behaviour as go-muse
(labels.go / series.go / group.go / results.go / scores.go / muse_batch.go), with every
numeric step delegated to libmuse_b200.so through include/muse_b200.h.

There is NO CPU fallback: importing works anywhere (so the symbol table can be checked
without a GPU) but creating a context without a CUDA device raises MuseError.
"""
from __future__ import annotations

import ctypes as C
import heapq
import math
import os
import subprocess
import uuid
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
# MUSE_B200_LIB: an alternative build of the same library (kernel A/B runs); default = the in-tree build
LIB_PATH = os.environ.get("MUSE_B200_LIB") or os.path.join(_HERE, "libmuse_b200.so")

MUSE_OK = 0
MUSE_ERR_INVALID_ARG = 1
MUSE_ERR_CUDA = 2
MUSE_ERR_LENGTH_MISMATCH = 3
MUSE_ERR_STDDEV_ZERO = 4
MUSE_ERR_NO_DEVICE = 5
MUSE_ERR_UNSUPPORTED = 6
MUSE_ERR_OUT_OF_MEMORY = 7

MODE_AUTO, MODE_EXACT, MODE_SCREEN = 0, 1, 2

SignFilter_POS = 1    # results.go:23
SignFilter_NEG = -1   # results.go:24
SignFilter_ANY = 0    # results.go:25
DefaultLabel = "uid"  # labels.go:7

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC"]
# translation units of libmuse_b200.so: the C ABI and one file per family of kernel instantiations
SOURCES = ["muse_api.cu", "kernels_exact.cu", "kernels_screen_warp.cu", "kernels_screen_big.cu", "kernels_screen_big13_a.cu", "kernels_screen_big13_b.cu", "kernels_screen_big13_c.cu",
           "kernels_screen_big13_d.cu", "kernels_screen_multi.cu", "kernels_bounds_tc.cu", "kernels_long.cu",
           "kernels_screen_sub1.cu", "kernels_screen_sub2.cu", "kernels_screen_sub3.cu", "kernels_screen_sub4.cu", "kernels_roll.cu",
           "kernels_remove.cu"]


class MuseError(Exception):
    """An `error` return of the Go API."""

    def __init__(self, code: int, msg: str):
        super().__init__(msg)
        self.code = code


class Partial(C.Structure):
    _fields_ = [("group_key", C.c_uint64), ("score", C.c_double), ("series_idx", C.c_int64),
                ("lag", C.c_int32), ("flags", C.c_int32)]


class Timing(C.Structure):
    _fields_ = [("total_ms", C.c_float), ("score_ms", C.c_float), ("rescore_ms", C.c_float),
                ("select_ms", C.c_float), ("n_rescored", C.c_int64), ("n_refined", C.c_int64),
                ("mode", C.c_int32), ("n_launches", C.c_int32)]


PARTIAL_DTYPE = np.dtype([("group_key", "<u8"), ("score", "<f8"), ("series_idx", "<i8"),
                          ("lag", "<i4"), ("flags", "<i4")])


def build(verbose: bool = False, out: Optional[str] = None, extra_flags: Sequence[str] = (), tag: str = "") -> str:
    """Compile libmuse_b200.so for sm_100a with nvcc (cross-compiles without a GPU): one object per translation
    unit, compiled side by side, then one link.  out / extra_flags / tag: a variant build for kernel A/B runs
    (tools/build_variant.py; loaded with MUSE_B200_LIB)."""
    from concurrent.futures import ThreadPoolExecutor
    csrc = os.path.join(_HERE, "csrc")
    lib_path = out or LIB_PATH
    hdrs = [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith((".cuh", ".h"))]
    hdrs.append(os.path.join(_ROOT, "include", "muse_b200.h"))
    objdir = os.path.join(_ROOT, "build", "obj" + ("_" + tag if tag else ""))
    os.makedirs(objdir, exist_ok=True)
    srcs = [os.path.join(csrc, f) for f in SOURCES if os.path.exists(os.path.join(csrc, f))]
    objs = [os.path.join(objdir, os.path.basename(f)[:-3] + ".o") for f in srcs]

    def stale(target, deps):
        return not os.path.exists(target) or any(os.path.getmtime(target) < os.path.getmtime(d) for d in deps)

    def compile_one(pair):
        src, obj = pair
        if not stale(obj, [src] + hdrs):
            return
        cmd = ["nvcc"] + NVCC_FLAGS + list(extra_flags) + ["-c", "-o", obj, src]
        if verbose:
            print(" ".join(cmd), flush=True)
        subprocess.check_call(cmd)

    with ThreadPoolExecutor(max_workers=max(1, min(len(srcs), os.cpu_count() or 1))) as ex:
        list(ex.map(compile_one, zip(srcs, objs)))
    if stale(lib_path, objs):
        cmd = ["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", lib_path] + objs
        if verbose:
            print(" ".join(cmd), flush=True)
        subprocess.check_call(cmd)
    return lib_path


_lib = None

# name -> (restype, argtypes); every symbol include/muse_b200.h declares
_dp, _ip64, _ip32 = C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_int32)
_vp = C.c_void_p
ABI = {
    "muse_last_error": (C.c_char_p, []),
    "muse_version": (C.c_char_p, []),
    "muse_ctx_create": (C.c_int, [C.c_int, C.POINTER(_vp)]),
    "muse_ctx_destroy": (None, [_vp]),
    "muse_ctx_synchronize": (C.c_int, [_vp]),
    "muse_ctx_set_stream": (C.c_int, [_vp, _vp]),
    "muse_host_alloc": (C.c_int, [C.POINTER(_vp), C.c_int64]),
    "muse_host_free": (None, [_vp]),
    "muse_held_bytes": (C.c_int, [_ip64, _ip64]),
    "muse_group_create": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int64, C.POINTER(_vp)]),
    "muse_group_destroy": (None, [_vp]),
    "muse_group_append": (C.c_int, [_vp, _vp, C.c_int64, C.c_int64, _vp]),
    "muse_group_append_device": (C.c_int, [_vp, _vp, C.c_int64, C.c_int64, _vp]),
    "muse_group_append_synthetic": (C.c_int, [_vp, C.c_int64, C.c_uint64, C.c_int64]),
    "muse_group_append_synthetic_ex": (C.c_int, [_vp, C.c_int64, C.c_uint64, C.c_int64, C.c_int32]),
    "muse_multi_last_timing": (C.c_int, [_vp, C.POINTER(C.c_float)]),
    "muse_group_set_synthetic_labels": (C.c_int, [_vp, _ip64, _ip64]),
    "muse_synth_row": (None, [C.c_uint64, C.c_int64, C.c_int64, _dp]),
    "muse_synth_reference": (None, [C.c_uint64, C.c_int64, _dp]),
    "muse_group_size": (C.c_int64, [_vp]),
    "muse_group_series_len": (C.c_int64, [_vp]),
    "muse_group_set_global_offset": (C.c_int, [_vp, C.c_int64]),
    "muse_group_clear": (C.c_int, [_vp]),
    "muse_group_read_row": (C.c_int, [_vp, C.c_int64, _dp]),
    "muse_group_read_rows": (C.c_int, [_vp, C.c_int64, C.c_int64, _vp]),
    "muse_group_roll": (C.c_int, [_vp, C.c_int64, C.c_int64, _vp, C.c_int64]),
    "muse_group_roll_device": (C.c_int, [_vp, C.c_int64, C.c_int64, _vp, C.c_int64]),
    "muse_group_remove": (C.c_int, [_vp, _ip64, C.c_int64, _ip64, _ip64, _ip64]),
    "muse_batch_create": (C.c_int, [_vp, _vp, _dp, C.c_int64, C.POINTER(_vp)]),
    "muse_batch_destroy": (None, [_vp]),
    "muse_batch_fft_len": (C.c_int64, [_vp]),
    "muse_batch_run": (C.c_int, [_vp, _ip32, C.c_int32, C.c_int64, C.c_int64, C.c_double, C.c_int32,
                                 _dp, _ip64, _ip64, _ip64]),
    "muse_batch_run_ex": (C.c_int, [_vp, _ip32, C.c_int32, C.c_int64, C.c_int64, C.c_double, C.c_int32,
                                    C.c_int32, C.c_int32, _dp, _ip64, _ip64, _ip64]),
    "muse_batch_run_where": (C.c_int, [_vp, _ip32, _ip32, C.c_int32, _ip32, C.c_int32, C.c_int64, C.c_int64, C.c_double,
                                       C.c_int32, C.c_int32, C.c_int32, _dp, _ip64, _ip64, _ip64]),
    "muse_batch_score_all": (C.c_int, [_vp, C.c_int32, _dp, _ip32]),
    "muse_batch_xcorr": (C.c_int, [_vp, C.c_int64, _dp, _ip32]),
    "muse_batch_screen_bounds": (C.c_int, [_vp, C.c_int32, C.c_int64, _vp, _vp]),
    "muse_batch_run_partial": (C.c_int, [_vp, _ip32, C.c_int32, C.c_int64, C.c_int64, C.c_double, C.c_int32,
                                         C.c_int32, _vp, C.c_int64, _ip64]),
    "muse_batch_run_partial_device": (C.c_int, [_vp, C.c_int64, C.c_int64, C.c_double, C.c_int32, C.c_int32, _vp, C.c_int64]),
    "muse_multi_run": (C.c_int, [_vp, _vp, _dp, C.c_int64, C.c_int64, _ip32, C.c_int32, C.c_int64, C.c_int64, C.c_double,
                                 C.c_int32, C.c_int32, _dp, _ip64, _ip64, _ip64]),
    "muse_multi_run_where": (C.c_int, [_vp, _vp, _dp, C.c_int64, C.c_int64, _ip32, _ip32, C.c_int32, _ip32, C.c_int32, C.c_int64,
                                       C.c_int64, C.c_double, C.c_int32, C.c_int32, _dp, _ip64, _ip64, _ip64]),
    "muse_multi_last_stats": (C.c_int, [_vp, _ip64, _ip64]),
    "muse_multi_bounds_tc": (C.c_int, [_vp, _vp, _dp, C.c_int64, C.c_int64, _vp]),
    "muse_xcorr": (C.c_int, [_vp, _dp, C.c_int64, _dp, C.c_int64, C.c_int64, C.c_int32, _dp, C.c_int64, _ip64, _ip64,
                             C.POINTER(C.c_double), _ip32]),
    "muse_exchange_create": (C.c_int, [_vp, C.c_int32, C.c_int32, C.c_int64, C.POINTER(_vp)]),
    "muse_exchange_ipc_handle": (C.c_int, [_vp, _vp]),
    "muse_exchange_open_peers": (C.c_int, [_vp, _vp]),
    "muse_exchange_destroy": (None, [_vp]),
    "muse_batch_run_exchange": (C.c_int, [_vp, _vp, C.c_int64, C.c_int64, C.c_double, C.c_int32, C.c_int32,
                                          _dp, _ip64, _ip64, _ip64]),
    "muse_batch_run_exchange_ex": (C.c_int, [_vp, _vp, _ip32, C.c_int32, C.c_int64, C.c_int64, C.c_double, C.c_int32, C.c_int32,
                                             _dp, _ip64, _ip64, _ip64]),
    "muse_multi_run_exchange": (C.c_int, [_vp, _vp, _dp, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_double, C.c_int32,
                                          C.c_int32, _dp, _ip64, _ip64, _ip64]),
    "muse_merge_partials_many": (C.c_int, [_vp, _vp, C.c_int32, C.c_int64, C.c_int64, _dp, _ip64, _ip64, _ip64]),
    "muse_batch_partial_capacity": (C.c_int64, [_vp, _ip32, C.c_int32, C.c_int64]),
    "muse_merge_partials": (C.c_int, [_vp, C.c_int64, C.c_int64, C.c_int64, C.c_double, C.c_int32,
                                      _dp, _ip64, _ip64, _ip64]),
    "muse_batch_last_timing": (C.c_int, [_vp, C.POINTER(Timing)]),
}


def lib():
    """The C-ABI library.  Fails loudly when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MuseError(MUSE_ERR_CUDA, "libmuse_b200.so is not built (run __graft_entry__.build()); "
                                           "there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in ABI.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def _check(rc: int):
    if rc != MUSE_OK:
        raise MuseError(rc, lib().muse_last_error().decode("utf-8", "replace"))


def _d(a: np.ndarray):
    return a.ctypes.data_as(_dp)


# ----------------------------------------------------------------------------------
# low level handles
# ----------------------------------------------------------------------------------
class Context:
    def __init__(self, device: int = 0):
        self.h = _vp()
        _check(lib().muse_ctx_create(device, C.byref(self.h)))
        self.device = device

    def synchronize(self):
        _check(lib().muse_ctx_synchronize(self.h))

    def set_stream(self, cuda_stream: Optional[int]):
        """Run on the given cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream)."""
        _check(lib().muse_ctx_set_stream(self.h, _vp(cuda_stream) if cuda_stream else None))

    def close(self):
        if self.h:
            lib().muse_ctx_destroy(self.h)
            self.h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_default_ctx: Dict[int, Context] = {}


def default_context(device: Optional[int] = None) -> Context:
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0")) if "MUSE_DEVICE" not in os.environ else int(os.environ["MUSE_DEVICE"])
    if device not in _default_ctx:
        _default_ctx[device] = Context(device)
    return _default_ctx[device]


class DeviceStore:
    """muse_group handle: the device slab + label-id table."""

    def __init__(self, ctx: Context, series_len: int, n_label_keys: int, capacity: int = 0):
        self.ctx = ctx
        self.h = _vp()
        self.series_len = series_len
        self.n_label_keys = n_label_keys
        _check(lib().muse_group_create(ctx.h, series_len, n_label_keys, capacity, C.byref(self.h)))

    def append(self, rows: np.ndarray, label_ids: Optional[np.ndarray] = None):
        rows = np.ascontiguousarray(rows, dtype=np.float64)
        if rows.ndim == 1:
            rows = rows[None, :]
        ids_p = None
        if label_ids is not None:
            label_ids = np.ascontiguousarray(label_ids, dtype=np.int32)
            ids_p = label_ids.ctypes.data_as(_vp)
        _check(lib().muse_group_append(self.h, rows.ctypes.data_as(_vp), rows.shape[0], rows.shape[1], ids_p))

    def append_host_ptr(self, ptr: int, n_series: int, series_len: int, ids_ptr: Optional[int] = None):
        _check(lib().muse_group_append(self.h, _vp(ptr), n_series, series_len, _vp(ids_ptr) if ids_ptr else None))

    def append_device(self, d_rows_ptr: int, n_series: int, series_len: int, d_ids_ptr: Optional[int] = None):
        _check(lib().muse_group_append_device(self.h, _vp(d_rows_ptr), n_series, series_len,
                                              _vp(d_ids_ptr) if d_ids_ptr else None))

    def append_synthetic(self, n_series: int, seed: int, first_index: int, variant: int = 0):
        _check(lib().muse_group_append_synthetic_ex(self.h, n_series, seed, first_index, variant))

    def set_synthetic_labels(self, div: Sequence[int], mod: Sequence[int]):
        """label id of key k for global series index i = (i / div[k]) % mod[k] (call after set_global_offset)."""
        d = np.asarray(list(div), dtype=np.int64)
        m = np.asarray(list(mod), dtype=np.int64)
        assert d.size >= self.n_label_keys and m.size >= self.n_label_keys
        _check(lib().muse_group_set_synthetic_labels(self.h, d.ctypes.data_as(_ip64), m.ctypes.data_as(_ip64)))

    def set_global_offset(self, off: int):
        _check(lib().muse_group_set_global_offset(self.h, off))

    def size(self) -> int:
        return int(lib().muse_group_size(self.h))

    def clear(self):
        _check(lib().muse_group_clear(self.h))

    def read_rows(self, first: int, n_rows: int, out: Optional[np.ndarray] = None) -> np.ndarray:
        if out is None:
            out = np.empty((n_rows, self.series_len))
        _check(lib().muse_group_read_rows(self.h, first, n_rows, out.ctypes.data_as(_vp)))
        return out

    def roll(self, samples: np.ndarray, first: int = 0):
        """muse_group_roll: rows [first, first + n_rows) slide forward by k samples in place, row <- row[k:] ++ samples[i],
        where samples is a host array [n_rows][k] (page-locked memory, e.g. from muse_host_alloc, is copied directly)."""
        X = np.ascontiguousarray(samples, dtype=np.float64)
        if X.ndim != 2:
            raise MuseError(MUSE_ERR_INVALID_ARG, "roll: samples must be [n_rows][k], got shape %r" % (X.shape,))
        n_rows, k = X.shape
        if k > self.series_len:
            raise MuseError(MUSE_ERR_INVALID_ARG, "roll: k = %d new samples exceed the series length %d" % (k, self.series_len))
        if first < 0:
            raise MuseError(MUSE_ERR_INVALID_ARG, "roll: first = %d < 0" % first)
        _check(lib().muse_group_roll(self.h, first, n_rows, X.ctypes.data_as(_vp), k))

    def roll_device(self, ptr: int, first: int, n_rows: int, k: int):
        """muse_group_roll_device: as roll, the [n_rows][k] samples in DEVICE memory at address ptr."""
        _check(lib().muse_group_roll_device(self.h, first, n_rows, _vp(ptr), k))

    def remove(self, rows) -> Tuple[np.ndarray, np.ndarray]:
        """muse_group_remove: the local rows `rows` (strictly ascending) leave the store, in place.  Returns (moved_from,
        moved_to): the kept rows at or above the new size that took the places of removed rows below it, in that order."""
        r = np.ascontiguousarray(rows, dtype=np.int64).reshape(-1)
        moved_from = np.zeros(max(r.size, 1), dtype=np.int64)
        moved_to = np.zeros(max(r.size, 1), dtype=np.int64)
        n_moved = C.c_int64(0)
        _check(lib().muse_group_remove(self.h, r.ctypes.data_as(_ip64) if r.size else None, r.size, moved_from.ctypes.data_as(_ip64),
                                       moved_to.ctypes.data_as(_ip64), C.byref(n_moved)))
        return moved_from[:n_moved.value], moved_to[:n_moved.value]

    def read_rows_ptr(self, first: int, n_rows: int, ptr: int):
        _check(lib().muse_group_read_rows(self.h, first, n_rows, _vp(ptr)))

    def read_row(self, i: int) -> np.ndarray:
        out = np.zeros(self.series_len)
        _check(lib().muse_group_read_row(self.h, i, _d(out)))
        return out

    def close(self):
        if self.h:
            lib().muse_group_destroy(self.h)
            self.h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def synth_row(seed: int, index: int, series_len: int) -> np.ndarray:
    out = np.zeros(series_len)
    lib().muse_synth_row(seed, index, series_len, _d(out))
    return out


def synth_reference(seed: int, series_len: int) -> np.ndarray:
    out = np.zeros(series_len)
    lib().muse_synth_reference(seed, series_len, _d(out))
    return out


class DeviceBatch:
    """muse_batch handle."""

    def __init__(self, ctx: Context, store: DeviceStore, ref: np.ndarray):
        self.ctx = ctx
        self.store = store
        self.h = _vp()
        ref = np.ascontiguousarray(ref, dtype=np.float64)
        _check(lib().muse_batch_create(ctx.h, store.h, _d(ref), ref.size, C.byref(self.h)))

    def fft_len(self) -> int:
        return int(lib().muse_batch_fft_len(self.h))

    def run(self, key_cols: Sequence[int], max_lag: int, top_n: int, threshold: float, sign_filter: int = 0,
            mode: int = MODE_AUTO, signed_scores: bool = False):
        cap = max(1, int(top_n))
        sc = np.zeros(cap)
        lg = np.zeros(cap, dtype=np.int64)
        ix = np.zeros(cap, dtype=np.int64)
        n_out = C.c_int64(0)
        kc = np.asarray(list(key_cols), dtype=np.int32)
        _check(lib().muse_batch_run_ex(self.h, kc.ctypes.data_as(_ip32) if kc.size else None, kc.size, max_lag, top_n,
                                       threshold, sign_filter, mode, int(signed_scores), _d(sc),
                                       lg.ctypes.data_as(_ip64), ix.ctypes.data_as(_ip64), C.byref(n_out)))
        k = int(n_out.value)
        return sc[:k], lg[:k], ix[:k]

    def run_where(self, where_cols: Sequence[int], where_ids: Sequence[int], key_cols: Sequence[int], max_lag: int, top_n: int,
                  threshold: float, sign_filter: int = 0, mode: int = MODE_AUTO, signed_scores: bool = False):
        """muse_batch_run_where: run() over the series whose label id in column where_cols[j] is where_ids[j] for every j;
        indices are those of the whole store."""
        wc = np.asarray(list(where_cols), dtype=np.int32)
        wi = np.asarray(list(where_ids), dtype=np.int32)
        if wc.size != wi.size:
            raise MuseError(MUSE_ERR_INVALID_ARG, "run_where: %d where columns, %d ids" % (wc.size, wi.size))
        cap = max(1, int(top_n))
        sc = np.zeros(cap)
        lg = np.zeros(cap, dtype=np.int64)
        ix = np.zeros(cap, dtype=np.int64)
        n_out = C.c_int64(0)
        kc = np.asarray(list(key_cols), dtype=np.int32)
        _check(lib().muse_batch_run_where(self.h, wc.ctypes.data_as(_ip32) if wc.size else None,
                                          wi.ctypes.data_as(_ip32) if wi.size else None, wc.size,
                                          kc.ctypes.data_as(_ip32) if kc.size else None, kc.size, max_lag, top_n, threshold,
                                          sign_filter, mode, int(signed_scores), _d(sc), lg.ctypes.data_as(_ip64),
                                          ix.ctypes.data_as(_ip64), C.byref(n_out)))
        k = int(n_out.value)
        return sc[:k], lg[:k], ix[:k]

    def score_all(self, signed_scores: bool = False):
        S = self.store.size()
        sc = np.zeros(max(S, 1))
        lg = np.zeros(max(S, 1), dtype=np.int32)
        _check(lib().muse_batch_score_all(self.h, int(signed_scores), _d(sc), lg.ctypes.data_as(_ip32)))
        return sc[:S], lg[:S].astype(np.int64)

    def screen_bounds(self, refine: bool = False, max_lag: int = 0):
        """fp32 bounds of every series (diagnostic).  refine=False: the spectral upper bound (> 1 means
        undecided).  refine=True: (upper, lower) of the fused second stage for the lag window max_lag:
        upper == -1: certainly outside the window; lower >= 0: certainly inside, score >= lower."""
        S = self.store.size()
        u = np.zeros(max(S, 1), dtype=np.float32)
        lo = np.full(max(S, 1), -1.0, dtype=np.float32)
        _check(lib().muse_batch_screen_bounds(self.h, int(refine), int(max_lag), u.ctypes.data_as(_vp),
                                              lo.ctypes.data_as(_vp)))
        return (u[:S], lo[:S]) if refine else u[:S]

    def xcorr(self, local_index: int):
        cc = np.zeros(self.fft_len())
        z = C.c_int32(0)
        _check(lib().muse_batch_xcorr(self.h, local_index, _d(cc), C.byref(z)))
        return (None if z.value else cc), bool(z.value)

    def run_partial(self, key_cols: Sequence[int], max_lag: int, top_n: int, threshold: float, sign_filter: int = 0,
                    mode: int = MODE_AUTO) -> np.ndarray:
        kc = np.asarray(list(key_cols), dtype=np.int32)
        kcp = kc.ctypes.data_as(_ip32) if kc.size else None
        cap = max(1, int(lib().muse_batch_partial_capacity(self.h, kcp, kc.size, top_n)))
        out = np.zeros(cap, dtype=PARTIAL_DTYPE)
        n_out = C.c_int64(0)
        _check(lib().muse_batch_run_partial(self.h, kcp, kc.size, max_lag, top_n, threshold, sign_filter, mode,
                                            out.ctypes.data_as(_vp), cap, C.byref(n_out)))
        return out[:int(n_out.value)]

    def run_partial_device(self, max_lag: int, top_n: int, threshold: float, sign_filter: int, mode: int,
                           d_out_ptr: int, capacity: int):
        """Ungrouped shard partials written to DEVICE memory at d_out_ptr (capacity records of 32 bytes) by work
        queued on the context's stream; nothing is synchronised (see muse_batch_run_partial_device)."""
        _check(lib().muse_batch_run_partial_device(self.h, max_lag, top_n, threshold, sign_filter, mode,
                                                   _vp(d_out_ptr), capacity))

    def timing(self) -> Timing:
        t = Timing()
        _check(lib().muse_batch_last_timing(self.h, C.byref(t)))
        return t

    def close(self):
        if self.h:
            lib().muse_batch_destroy(self.h)
            self.h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def merge_partials(parts: np.ndarray, max_lag: int, top_n: int, threshold: float, sign_filter: int = 0):
    parts = np.ascontiguousarray(parts, dtype=PARTIAL_DTYPE)
    cap = max(1, int(top_n))
    sc = np.zeros(cap)
    lg = np.zeros(cap, dtype=np.int64)
    ix = np.zeros(cap, dtype=np.int64)
    n_out = C.c_int64(0)
    _check(lib().muse_merge_partials(parts.ctypes.data_as(_vp), parts.size, max_lag, top_n, threshold, sign_filter,
                                     _d(sc), lg.ctypes.data_as(_ip64), ix.ctypes.data_as(_ip64), C.byref(n_out)))
    k = int(n_out.value)
    return sc[:k], lg[:k], ix[:k]


def multi_run(store: "DeviceStore", refs, key_cols: Sequence[int], max_lag: int, top_n: int, threshold: float,
              sign_filter: int = 0, mode: int = MODE_AUTO, raw: bool = False):
    """muse_multi_run: every row of refs as a NewBatch + Run against the resident store.  Returns one
    (scores, lags, series_idx) triple per reference, None where the reference has zero std; raw=True returns the
    call's own outputs instead: (scores[Q, top_n], lags[Q, top_n], series_idx[Q, top_n], n_out[Q]), n_out -1 for such
    a reference."""
    R = np.ascontiguousarray(refs, dtype=np.float64)
    assert R.ndim == 2
    Q, cap = R.shape[0], max(1, int(top_n))
    kc = np.asarray(list(key_cols), dtype=np.int32)
    sc = np.zeros((max(Q, 1), cap))
    lg = np.zeros((max(Q, 1), cap), dtype=np.int64)
    ix = np.zeros((max(Q, 1), cap), dtype=np.int64)
    n_out = np.zeros(max(Q, 1), dtype=np.int64)
    _check(lib().muse_multi_run(store.ctx.h, store.h, _d(R), Q, R.shape[1], kc.ctypes.data_as(_ip32) if kc.size else None,
                                kc.size, max_lag, top_n, threshold, sign_filter, mode, _d(sc), lg.ctypes.data_as(_ip64),
                                ix.ctypes.data_as(_ip64), n_out.ctypes.data_as(_ip64)))
    if raw:
        return sc[:Q], lg[:Q], ix[:Q], n_out[:Q]
    return [None if n_out[q] < 0 else (sc[q, :n_out[q]].copy(), lg[q, :n_out[q]].copy(), ix[q, :n_out[q]].copy())
            for q in range(Q)]


def multi_run_where(store: "DeviceStore", refs, where_cols: Sequence[int], where_ids: Sequence[int], key_cols: Sequence[int],
                    max_lag: int, top_n: int, threshold: float, sign_filter: int = 0, mode: int = MODE_AUTO, raw: bool = False):
    """muse_multi_run_where: multi_run over the series whose label id in column where_cols[j] is where_ids[j] for every j (one
    selection for all references); indices are those of the whole store.  Returns as multi_run."""
    R = np.ascontiguousarray(refs, dtype=np.float64)
    assert R.ndim == 2
    wc = np.asarray(list(where_cols), dtype=np.int32)
    wi = np.asarray(list(where_ids), dtype=np.int32)
    if wc.size != wi.size:
        raise MuseError(MUSE_ERR_INVALID_ARG, "multi_run_where: %d where columns, %d ids" % (wc.size, wi.size))
    Q, cap = R.shape[0], max(1, int(top_n))
    kc = np.asarray(list(key_cols), dtype=np.int32)
    sc = np.zeros((max(Q, 1), cap))
    lg = np.zeros((max(Q, 1), cap), dtype=np.int64)
    ix = np.zeros((max(Q, 1), cap), dtype=np.int64)
    n_out = np.zeros(max(Q, 1), dtype=np.int64)
    _check(lib().muse_multi_run_where(store.ctx.h, store.h, _d(R), Q, R.shape[1], wc.ctypes.data_as(_ip32) if wc.size else None,
                                      wi.ctypes.data_as(_ip32) if wi.size else None, wc.size,
                                      kc.ctypes.data_as(_ip32) if kc.size else None, kc.size, max_lag, top_n, threshold,
                                      sign_filter, mode, _d(sc), lg.ctypes.data_as(_ip64), ix.ctypes.data_as(_ip64),
                                      n_out.ctypes.data_as(_ip64)))
    if raw:
        return sc[:Q], lg[:Q], ix[:Q], n_out[:Q]
    return _triples(sc[:Q], lg[:Q], ix[:Q], n_out[:Q])


def multi_records(sc: np.ndarray, lg: np.ndarray, ix: np.ndarray, n_out: np.ndarray) -> np.ndarray:
    """multi_run(raw=True) outputs as [Q, top_n] muse_partial records: row q holds query q's list in its order
    (group_key = global series index), padded with flags = 1 -- the layout muse_merge_partials_many merges."""
    Q, top_n = sc.shape
    rec = np.zeros((Q, top_n), dtype=PARTIAL_DTYPE)
    valid = np.arange(top_n)[None, :] < np.maximum(n_out, 0)[:, None]
    rec["group_key"] = np.where(valid, ix, 0).astype(np.uint64)
    rec["score"] = np.where(valid, sc, 0.0)
    rec["series_idx"] = np.where(valid, ix, 0)
    rec["lag"] = np.where(valid, lg, 0).astype(np.int32)
    rec["flags"] = np.where(valid, 0, 1)
    return rec


def merge_partials_many(ctx: Context, d_parts: int, world: int, n_refs: int, top_n: int):
    """muse_merge_partials_many: merge the per-query lists of `world` shards, gathered in DEVICE memory at address d_parts as
    [world][n_refs][top_n] records (multi_records of each shard), into the global top_n of every query.  Returns
    (scores[Q, top_n], lags[Q, top_n], series_idx[Q, top_n], n_out[Q])."""
    cap = max(1, int(top_n))
    sc = np.zeros((max(n_refs, 1), cap))
    lg = np.zeros((max(n_refs, 1), cap), dtype=np.int64)
    ix = np.zeros((max(n_refs, 1), cap), dtype=np.int64)
    n_out = np.zeros(max(n_refs, 1), dtype=np.int64)
    _check(lib().muse_merge_partials_many(ctx.h, _vp(d_parts), world, n_refs, top_n, _d(sc), lg.ctypes.data_as(_ip64),
                                          ix.ctypes.data_as(_ip64), n_out.ctypes.data_as(_ip64)))
    return sc[:n_refs], lg[:n_refs], ix[:n_refs], n_out[:n_refs]


def _triples(sc, lg, ix, n_out):
    return [None if n_out[q] < 0 else (sc[q, :n_out[q]].copy(), lg[q, :n_out[q]].copy(), ix[q, :n_out[q]].copy())
            for q in range(len(n_out))]


def multi_last_stats(ctx: Context) -> Tuple[int, int]:
    """(second stages, fp64 re-scorings) of the context's last multi_run, summed over its queries."""
    a, b = C.c_int64(0), C.c_int64(0)
    _check(lib().muse_multi_last_stats(ctx.h, C.byref(a), C.byref(b)))
    return int(a.value), int(b.value)


def multi_last_timing(ctx: Context) -> Tuple[float, float, float, float]:
    """Device ms of the last launch group of the tensor-core multi-query path: (magnitudes, bounds GEMM, second stages, tails)."""
    ms = (C.c_float * 4)()
    _check(lib().muse_multi_last_timing(ctx.h, ms))
    return tuple(float(x) for x in ms)


def multi_bounds_tc(store: "DeviceStore", refs) -> np.ndarray:
    """muse_multi_bounds_tc: [Q, S] upper bounds of every series' score against every reference, computed as one bf16
    contraction on the tensor cores (diagnostic)."""
    R = np.ascontiguousarray(refs, dtype=np.float64)
    assert R.ndim == 2
    out = np.zeros((R.shape[0], max(store.size(), 1)), dtype=np.float32)
    _check(lib().muse_multi_bounds_tc(store.ctx.h, store.h, _d(R), R.shape[0], R.shape[1], out.ctypes.data_as(_vp)))
    return out[:, :store.size()]


def xCorr(x, y, n: int, normalize: bool, ctx: Optional[Context] = None):
    """xcorr.go:102-153 on the device, any n: (cc, lag, value); (None, 0, 0.0) when a normalised input has
    zero std (:109-126).  n is raised to max(n, len(x), len(y)) (:104-106)."""
    ctx = ctx or default_context()
    xa = np.ascontiguousarray(x, dtype=np.float64)
    ya = np.ascontiguousarray(y, dtype=np.float64)
    nn = max(int(n), xa.size, ya.size)
    cc = np.zeros(max(nn, 1))
    n_out, lag, val, z = C.c_int64(0), C.c_int64(0), C.c_double(0.0), C.c_int32(0)
    _check(lib().muse_xcorr(ctx.h, _d(xa), xa.size, _d(ya), ya.size, int(n), int(bool(normalize)), _d(cc), cc.size,
                            C.byref(n_out), C.byref(lag), C.byref(val), C.byref(z)))
    if z.value:
        return None, 0, 0.0
    return cc[:int(n_out.value)], int(lag.value), float(val.value)


# ----------------------------------------------------------------------------------
# go-muse API mirror
# ----------------------------------------------------------------------------------
LabelMap = dict   # labels.go:11


class Labels:
    """labels.go:14-73."""

    def __init__(self, labels: Dict[str, str]):
        self.labels = dict(labels)
        self.keys = sorted(self.labels.keys())

    def Len(self) -> int:
        return len(self.labels)

    def Keys(self) -> List[str]:
        return self.keys

    def Get(self, key: str) -> Tuple[str, bool]:
        if key in self.labels:
            return self.labels[key], True
        return "", False

    def ID(self, labels: Optional[List[str]] = None) -> str:
        # labels.go:54-73: sorted requested keys (the caller's list is sorted in place), absent keys skipped
        if not labels:
            labels = self.keys
        else:
            labels.sort()
        return ",".join(k + ":" + self.labels[k] for k in labels if k in self.labels)

    def __repr__(self):
        return "Labels(%r)" % (self.labels,)


def NewLabels(labels: Dict[str, str]) -> Labels:
    return Labels(labels)


class Series:
    """series.go:8-42.  The values are never modified in place (go-muse z-normalises in place); Group.Roll replaces them by
    the rolled window."""

    def __init__(self, y, labels: Optional[Labels] = None):
        if labels is None or labels.Len() == 0:
            labels = Labels({DefaultLabel: str(uuid.uuid4())})   # series.go:16-18
        self.y = np.asarray(y, dtype=np.float64)
        self.labels = labels

    def Length(self) -> int:
        return int(self.y.size)

    def Values(self) -> np.ndarray:
        return self.y

    def Labels(self) -> Labels:
        return self.labels

    def UID(self) -> str:
        return self.labels.ID(list(self.labels.Keys()))


def NewSeries(y, labels: Optional[Labels] = None) -> Series:
    return Series(y, labels)


class Group:
    """group.go:7-104 over a device store.

    Strings stay here: every label key becomes a column and every value an int32 id
    (dictionary encoded at Add); the device sees only the id table."""

    def __init__(self, name: str, ctx: Optional[Context] = None):
        self.Name = name
        self.n = 0
        self.registry: Dict[str, int] = {}       # uid -> series index
        self.series: List[Series] = []
        self._ctx = ctx
        self._store: Optional[DeviceStore] = None
        self._cols: List[str] = []                # label key per device column
        self._dict: Dict[str, Dict[str, int]] = {}
        self._uploaded = 0

    def Length(self) -> int:
        return self.n

    def Add(self, *series: Series):
        for s in series:
            if len(s.labels.Keys()) == 0:                                   # group.go:33-36
                raise MuseError(MUSE_ERR_INVALID_ARG, "Invalid Series with no labels, %r" % (s,))
            uid = s.UID()
            if uid in self.registry:                                        # group.go:39-41
                raise MuseError(MUSE_ERR_INVALID_ARG, "Series with label:values, %s, already exists within group, %s"
                                % (uid, self.Name))
            if len(self.registry) == 0:                                     # group.go:45-51
                self.n = s.Length()
            elif s.Length() != self.n:
                raise MuseError(MUSE_ERR_LENGTH_MISMATCH, "Timeseries has length %d, but current group has length %d"
                                % (s.Length(), self.n))
            self.registry[uid] = len(self.series)
            self.series.append(s)
        return None

    def Roll(self, samples):
        """Every series slides forward by k new samples, y <- y[k:] ++ samples[i] for the i-th series in Add order, on the
        device store in place (no re-upload) and in each Series' values (a later store rebuild uploads from those).
        samples: [len(series)][k], 0 <= k <= Length(); checked before any device call."""
        rows = [np.asarray(r, dtype=np.float64) for r in samples]
        if len(rows) != len(self.series):
            raise MuseError(MUSE_ERR_INVALID_ARG, "Roll: %d rows of samples for %d series" % (len(rows), len(self.series)))
        if not rows:
            return None
        k = rows[0].size
        for i, r in enumerate(rows):
            if r.ndim != 1 or r.size != k:
                raise MuseError(MUSE_ERR_INVALID_ARG, "Roll: row %d has shape %r, row 0 has %d samples" % (i, r.shape, k))
        if k > self.n:
            raise MuseError(MUSE_ERR_INVALID_ARG, "Roll: %d new samples exceed the series length %d" % (k, self.n))
        if k == 0:
            return None
        store = self._sync_device()
        try:
            store.roll(np.stack(rows), 0)
        except MuseError:
            # rows rolled before a device failure: drop the store, the next call rebuilds it from the unchanged values
            store.close()
            self._store = None
            raise
        for s, r in zip(self.series, rows):
            s.y = np.concatenate([s.y[k:], r])
        return None

    def Remove(self, *series: Series):
        """Takes series out of the group, matched by UID(); a series that is not a member raises MuseError and nothing is
        removed (a series named twice is removed once).  With a device store the removal is in place (muse_group_remove):
        the remaining series keep their positions, except that the last ones move into the places of removed ones, and
        self.series makes the same moves (the library's pairs).  Without a store, or when the device call fails (the store
        is then dropped and rebuilt by the next call that needs it), the remaining series keep their order.  A group that
        becomes empty forgets its length, as a new Group.  Remove then Add of the same UID replaces a series."""
        idx = set()
        for s in series:
            i = self.registry.get(s.UID())
            if i is None:
                raise MuseError(MUSE_ERR_INVALID_ARG, "Series with label:values, %s, is not within group, %s" % (s.UID(), self.Name))
            idx.add(i)
        if not idx:
            return None
        if len(idx) == len(self.series) or self._store is None:
            if self._store is not None:
                self._store.close()
                self._store = None
            self._remove_in_order(idx)
            return None
        store = self._sync_device()
        rows = sorted(idx)
        try:
            moved_from, moved_to = store.remove(rows)
        except MuseError:
            store.close()
            self._store = None
            self._remove_in_order(idx)
            raise
        for i in rows:
            del self.registry[self.series[i].UID()]
        for f, t in zip(moved_from.tolist(), moved_to.tolist()):
            self.series[t] = self.series[f]
            self.registry[self.series[t].UID()] = t
        del self.series[len(self.series) - len(rows):]
        self._uploaded = len(self.series)
        return None

    def _remove_in_order(self, idx):
        self.series = [s for i, s in enumerate(self.series) if i not in idx]
        self.registry = {s.UID(): i for i, s in enumerate(self.series)}
        if not self.series:
            self.n = 0

    def FilterByLabelValues(self, labels: Labels) -> List[Series]:
        """group.go:60-71: members whose values match on every key of `labels`."""
        keys = labels.Keys()
        out = []
        for s in self.series:
            if s.labels.ID(list(keys)) == labels.ID(list(keys)):
                out.append(s)
        return out if keys else []

    # -- device side ---------------------------------------------------------------
    def _sync_device(self) -> DeviceStore:
        ctx = self._ctx or default_context()
        keys = sorted({k for s in self.series for k in s.labels.Keys()})
        # a new key needs a column; a key that Remove took from every series keeps its column (all ids -1 now), which groups
        # and filters as an absent key does, so the store is not rebuilt
        if self._store is None or not set(keys) <= set(self._cols):
            if self._store is not None:
                self._store.close()
            self._cols = keys
            self._dict = {k: {} for k in keys}
            # one extra column that nobody has (all ids -1): grouping by an unknown key
            self._store = DeviceStore(ctx, self.n, len(keys) + 1, len(self.series))
            self._uploaded = 0
        if self._uploaded < len(self.series):
            new = self.series[self._uploaded:]
            rows = np.stack([s.y for s in new])
            ids = np.full((len(new), len(self._cols) + 1), -1, dtype=np.int32)
            for i, s in enumerate(new):
                for c, k in enumerate(self._cols):
                    v, ok = s.labels.Get(k)
                    if ok:
                        d = self._dict[k]
                        ids[i, c] = d.setdefault(v, len(d))
            self._store.append(rows, ids)
            self._uploaded = len(self.series)
        return self._store

    def _where(self, labels: Labels) -> Optional[Tuple[List[int], List[int]]]:
        """(columns, ids) of the equalities of FilterByLabelValues(labels) on the device store; None when no series can
        match: empty labels, or a key or value no series of the store has."""
        keys = labels.Keys()
        if not keys:
            return None
        cols, ids = [], []
        for k in keys:
            v, _ = labels.Get(k)
            if k not in self._cols or v not in self._dict[k]:
                return None
            cols.append(self._cols.index(k))
            ids.append(self._dict[k][v])
        return cols, ids

    def _key_cols(self, group_by: Optional[List[str]]) -> List[int]:
        if not group_by:
            return []
        cols = []
        for name in sorted(set(group_by)):
            if name in self._cols:
                cols.append(self._cols.index(name))
        if not cols:
            cols = [len(self._cols)]       # every series lacks the key(s): one group (labels.go:61-65)
        return cols


def NewGroup(name: str) -> Group:
    return Group(name)


def _go_float(f: float) -> str:
    """encoding/json's float64 formatting: shortest digits that round-trip, %f form for 1e-6 <= |f| < 1e21, else
    %e form with a one- or two-digit exponent cleaned up as Go does (1e-07 -> 1e-7)."""
    from decimal import Decimal
    if f == 0:
        return "-0" if str(f).startswith("-") else "0"
    d = Decimal(repr(f))
    if 1e-6 <= abs(f) < 1e21:
        t = format(d, "f")
        return t.rstrip("0").rstrip(".") if "." in t else t
    sign, digits, exp = d.as_tuple()
    ds = "".join(map(str, digits)).rstrip("0") or "0"
    e10 = exp + len(digits) - 1
    mant = ds[0] + ("." + ds[1:] if len(ds) > 1 else "")
    return "%s%se%s%d" % ("-" if sign else "", mant, "-" if e10 < 0 else "+", abs(e10))


class Score:
    """scores.go:11-15."""

    __slots__ = ("Labels", "Lag", "PercentScore")

    def __init__(self, Labels: Optional[Labels] = None, Lag: int = 0, PercentScore: float = 0.0):
        self.Labels = Labels
        self.Lag = Lag
        self.PercentScore = PercentScore

    def to_json(self):
        return {"labels": self.Labels.labels if self.Labels else None, "lag": self.Lag,
                "percentScore": self.PercentScore}

    def MarshalJSON(self) -> str:
        """What encoding/json writes for the Go struct (scores.go:11-15): keys labels / lag / percentScore in
        field order; *Labels has only unexported fields (labels.go:14-17), so a non-nil one is `{}`."""
        import json
        if self.PercentScore != self.PercentScore or abs(self.PercentScore) == float("inf"):
            raise ValueError("json: unsupported value: %r" % self.PercentScore)     # as encoding/json
        return '{"labels":%s,"lag":%d,"percentScore":%s}' % ("{}" if self.Labels is not None else "null", self.Lag,
                                                           _go_float(float(self.PercentScore)))


class Results:
    """results.go:11-87: filter + top-N min-heap on |score|; not reset between Runs."""

    def __init__(self, maxLag: int, topN: int, threshold: float, signFilter: int):
        self.MaxLag = maxLag
        self.TopN = topN
        self.Threshold = threshold
        self.SignFilter = signFilter
        self._heap: List[Tuple[float, int, Score]] = []
        self._seq = 0

    def passed(self, s: Score) -> bool:
        return (abs(float(s.Lag)) <= float(self.MaxLag) and abs(s.PercentScore) >= self.Threshold
                and (self.SignFilter == SignFilter_ANY
                     or (s.PercentScore > 0 and self.SignFilter == SignFilter_POS)
                     or (s.PercentScore < 0 and self.SignFilter == SignFilter_NEG)))

    def Update(self, s: Score):
        if s.Labels is None:                                                # results.go:56-59
            return
        if not self.passed(s):
            return
        self._seq += 1
        item = (abs(s.PercentScore), -self._seq, s)   # equal scores: earlier arrival ranks higher
        if len(self._heap) == self.TopN:
            if self.TopN > 0 and abs(s.PercentScore) > self._heap[0][0]:    # strictly greater, :62-66
                heapq.heapreplace(self._heap, item)
        else:
            heapq.heappush(self._heap, item)

    def Fetch(self) -> Tuple[List[Score], float]:
        """Descending |score| (results.go:81-85) and the mean |score| (NaN when empty); drains the heap."""
        items = sorted(self._heap, key=lambda it: (-it[0], -it[1]))
        self._heap = []
        scores = [it[2] for it in items]
        total = sum(abs(s.PercentScore) for s in scores)
        return scores, (total / len(scores) if scores else float("nan"))


def NewResults(maxLag: int, topN: int, threshold: float, signFilter: int) -> Results:
    return Results(maxLag, topN, threshold, signFilter)


class Batch:
    """muse_batch.go:13-130."""

    def __init__(self, ref: Series, comp: Group, results: Results, cc: int, mode: int = MODE_AUTO):
        for s in comp.series:                                               # muse_batch.go:24-28
            if ref.Length() != s.Length():
                raise MuseError(MUSE_ERR_LENGTH_MISMATCH,
                                "%s from comparison group series does not have the same length as the reference"
                                % s.UID())
        if cc < 1:
            cc = 1
        self.Comparison = comp
        self.Results = results
        self.Concurrency = cc     # kept for API parity; the device schedules the work
        self.mode = mode
        self._ref = np.array(ref.Values(), dtype=np.float64, copy=True)
        self._batch: Optional[DeviceBatch] = None
        if comp.series:
            store = comp._sync_device()
            self._batch = DeviceBatch(store.ctx, store, self._ref)        # MuseError on std == 0
        else:
            # empty comparison group: still validate the query as muse_batch.go:38-41 does
            ctx = comp._ctx or default_context()
            tmp = DeviceStore(ctx, max(ref.Length(), 2), 0, 1)
            try:
                DeviceBatch(ctx, tmp, self._ref).close()
            finally:
                tmp.close()
        self.n = self._batch.fft_len() if self._batch else 0

    def Run(self, groupByLabels: Optional[List[str]] = None):
        """muse_batch.go:99-130; always returns None (nil)."""
        comp = self.Comparison
        if not comp.series:
            return None
        store = comp._sync_device()
        if self._batch is None or self._batch.store is not store:
            self._batch = DeviceBatch(store.ctx, store, self._ref)
        r = self.Results
        cols = comp._key_cols(groupByLabels)
        # the device applies the Results filter and keeps the TopN best; pushing those through
        # Results.Update leaves the heap exactly as pushing every group score would
        sc, lg, ix = self._batch.run(cols, r.MaxLag, r.TopN, r.Threshold, r.SignFilter, mode=self.mode)
        for s, l, i in zip(sc, lg, ix):
            r.Update(Score(comp.series[int(i)].Labels(), int(l), float(s)))
        return None


    def RunWhere(self, labels: Labels, groupByLabels: Optional[List[str]] = None):
        """Run over the series of Comparison.FilterByLabelValues(labels) only, on the resident store: Results end up as
        NewBatch(ref, <a Group of those series>, ...).Run(groupByLabels) leaves them.  Nothing matches (empty labels, a key
        or value no series has): no device call, Results untouched.  Always returns None (nil)."""
        comp = self.Comparison
        if not comp.series or not labels.Keys():
            return None
        store = comp._sync_device()          # uploads series added since the last call; the dictionary then knows every value
        where = comp._where(labels)
        if where is None:
            return None
        if self._batch is None or self._batch.store is not store:
            self._batch = DeviceBatch(store.ctx, store, self._ref)
        r = self.Results
        cols = comp._key_cols(groupByLabels)
        sc, lg, ix = self._batch.run_where(where[0], where[1], cols, r.MaxLag, r.TopN, r.Threshold, r.SignFilter,
                                           mode=self.mode)
        for s, l, i in zip(sc, lg, ix):
            r.Update(Score(comp.series[int(i)].Labels(), int(l), float(s)))
        return None


def NewBatch(ref: Series, comp: Group, results: Results, cc: int) -> Batch:
    return Batch(ref, comp, results, cc)


def RunMany(refs: Sequence[Series], comp: Group, results: Sequence[Results], groupByLabels: Optional[List[str]] = None):
    """go/muse/multi.go RunMany: a loop of NewBatch(refs[q], comp, results[q], cc).Run(groupByLabels) in one call
    (muse_multi_run).  Returns (errs, err) as the Go function: err a MuseError (nothing was run), else errs[q] the
    MuseError of a constant reference (results[q] untouched) or None."""
    return _run_many(refs, comp, results, False, None, groupByLabels)


def RunManyWhere(refs: Sequence[Series], comp: Group, results: Sequence[Results], labels: Optional[Labels],
                 groupByLabels: Optional[List[str]] = None):
    """go/muse/multi.go RunManyWhere: RunMany over comp.FilterByLabelValues(labels) only, on the resident store
    (muse_multi_run_where) -- a loop of NewBatch(refs[q], comp, results[q], cc).RunWhere(labels, groupByLabels).  The checks
    of RunMany; nothing can match (empty labels, a key or value no series has): no device call, results untouched and
    every errs[q] None."""
    return _run_many(refs, comp, results, True, labels, groupByLabels)


def _run_many(refs, comp: Group, results, filter_: bool, labels: Optional[Labels], groupByLabels):
    if len(refs) != len(results):
        return None, MuseError(MUSE_ERR_INVALID_ARG, "%d references but %d results" % (len(refs), len(results)))
    errs: List[Optional[MuseError]] = [None] * len(refs)
    if len(refs) == 0 or len(comp.series) == 0:
        return errs, None
    n = comp.Length()
    r0 = results[0]
    for ref, rq in zip(refs, results):
        if ref.Length() != n:
            return None, MuseError(MUSE_ERR_INVALID_ARG, "%s does not have the same length as the comparison group" % ref.UID())
        if (rq.MaxLag, rq.TopN, rq.Threshold, rq.SignFilter) != (r0.MaxLag, r0.TopN, r0.Threshold, r0.SignFilter):
            return None, MuseError(MUSE_ERR_INVALID_ARG, "RunMany needs the same MaxLag, TopN, Threshold and SignFilter on every Results")
    if r0.TopN < 1 or (filter_ and (labels is None or not labels.Keys())):
        return errs, None
    R = np.stack([np.asarray(ref.Values(), dtype=np.float64) for ref in refs])
    try:
        store = comp._sync_device()      # uploads series added since the last call: the dictionary then knows every value
        cols = comp._key_cols(groupByLabels)
        if filter_:
            where = comp._where(labels)
            if where is None:
                return errs, None
            out = multi_run_where(store, R, where[0], where[1], cols, r0.MaxLag, r0.TopN, r0.Threshold, r0.SignFilter)
        else:
            out = multi_run(store, R, cols, r0.MaxLag, r0.TopN, r0.Threshold, r0.SignFilter)
    except MuseError as e:
        return None, e
    for q, got in enumerate(out):
        if got is None:
            errs[q] = MuseError(MUSE_ERR_STDDEV_ZERO, "Invalid input query, Standard deviation of zero")
            continue
        for s, l, i in zip(*got):
            results[q].Update(Score(comp.series[int(i)].Labels(), int(l), float(s)))
    return errs, None


class Muse:
    """muse.go:12-92: one reference, Run(compGraphs) scores ONE group of series with SIGNED scores
    (clamped to [-1, 1], muse.go:72-76), keeps the one with the largest |score| (strictly greater,
    first always taken, muse.go:86) and pushes it through Results.Update."""

    def __init__(self, ref: Series, results: Results, ctx: Optional[Context] = None):
        if ref.Length() < 1:                                                # muse.go:24-26
            raise MuseError(MUSE_ERR_INVALID_ARG, "Reference series length must be greater than zero")
        self.Results = results
        self.refN = ref.Length()
        self._ctx = ctx or default_context()
        self._ref = np.array(ref.Values(), dtype=np.float64, copy=True)
        self._store = DeviceStore(self._ctx, self.refN, 0, 1)
        self._batch = DeviceBatch(self._ctx, self._store, self._ref)        # MuseError "Invalid input query" on std == 0
        self.n = self._batch.fft_len()

    def Run(self, compGraphs: Sequence[Series]):
        if len(compGraphs) == 0:                                            # muse.go:48-51
            return None
        for s in compGraphs:                                                # muse.go:70-72
            if s.Length() != self.refN:
                return MuseError(MUSE_ERR_LENGTH_MISMATCH,
                                 "Encountered a comparison graph with differing length than the reference, %r" % s.Labels())
        self._store.clear()
        self._store.append(np.stack([np.asarray(s.Values(), dtype=np.float64) for s in compGraphs]))
        sc, lg = self._batch.score_all(signed_scores=True)
        best = 0
        for i in range(1, len(sc)):                                         # muse.go:86: strictly greater |score|
            if abs(sc[i]) > abs(sc[best]):
                best = i
        self.Results.Update(Score(compGraphs[best].Labels(), int(lg[best]), float(sc[best])))
        return None


def New(ref: Series, results: Results) -> Muse:
    return Muse(ref, results)


# ----------------------------------------------------------------------------------
# multi-GPU: one process per GPU, shards merged with one small all-gather
# ----------------------------------------------------------------------------------
def allgather_merge(parts: np.ndarray, max_lag: int, top_n: int, threshold: float, sign_filter: int = 0,
                    fixed_capacity: Optional[int] = None):
    """All-gather this rank's muse_partial records over torch.distributed (NCCL on GPUs, gloo on
    CPU) and merge them (muse_merge_partials) -- every rank returns the same global result.

    fixed_capacity: when every rank emits at most that many records (ungrouped runs: top_n) the
    size exchange is skipped and ONE all-gather is issued; otherwise the counts are gathered first.
    """
    import torch
    import torch.distributed as dist

    world = dist.get_world_size()
    backend = dist.get_backend()
    dev = torch.device("cuda", torch.cuda.current_device()) if backend == "nccl" else torch.device("cpu")
    parts = np.ascontiguousarray(parts, dtype=PARTIAL_DTYPE)
    if fixed_capacity is None:
        n_local = torch.tensor([parts.size], dtype=torch.int64, device=dev)
        counts = torch.zeros(world, dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(counts, n_local)
        counts = counts.cpu().numpy()
        cap = int(counts.max())
    else:
        cap = int(fixed_capacity)
        counts = None
    rec = np.zeros(max(cap, 1), dtype=PARTIAL_DTYPE)
    rec["flags"] = 1                                   # padding records are ignored by the merge
    rec[:parts.size] = parts
    t = torch.from_numpy(rec.view(np.uint8)).to(dev)
    out = torch.empty(world * t.numel(), dtype=torch.uint8, device=dev)
    dist.all_gather_into_tensor(out, t)
    allp = out.cpu().numpy().view(PARTIAL_DTYPE)
    return merge_partials(allp, max_lag, top_n, threshold, sign_filter)


_gather_buffers: Dict[Tuple[int, int, int], tuple] = {}


def allgather_merge_device(batch: DeviceBatch, max_lag: int, top_n: int, threshold: float, sign_filter: int = 0,
                           mode: int = MODE_AUTO):
    """One multi-GPU step of an UNGROUPED run with the partials kept on the device: the shard's top_n
    records are written by the library on the context's stream (which must be torch's current stream:
    Context.set_stream), all-gathered by NCCL on that same stream, copied to the host once and merged
    (muse_merge_partials).  Falls back to the host path when the device-side select reports an overflow."""
    import torch
    import torch.distributed as dist

    world = dist.get_world_size()
    dev = torch.cuda.current_device()
    cap = max(1, int(top_n))
    key = (dev, world, cap)
    if key not in _gather_buffers:
        t = torch.empty(cap * PARTIAL_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
        out = torch.empty(world * t.numel(), dtype=torch.uint8, device="cuda")
        host = torch.empty(world * t.numel(), dtype=torch.uint8, pin_memory=True)
        _gather_buffers[key] = (t, out, host)
    t, out, host = _gather_buffers[key]
    batch.run_partial_device(max_lag, top_n, threshold, sign_filter, mode, t.data_ptr(), cap)
    dist.all_gather_into_tensor(out, t)
    host.copy_(out, non_blocking=True)
    torch.cuda.current_stream().synchronize()
    allp = host.numpy().view(PARTIAL_DTYPE)
    if np.any(allp["flags"] == 2):      # some shard's candidate list did not fit the device-side select
        parts = batch.run_partial([], max_lag, top_n, threshold, sign_filter, mode=mode)
        return allgather_merge(parts, max_lag, top_n, threshold, sign_filter, fixed_capacity=top_n)
    return merge_partials(allp, max_lag, top_n, threshold, sign_filter)


def allgather_merge_many(store: DeviceStore, refs, max_lag: int, top_n: int, threshold: float, sign_filter: int = 0,
                         mode: int = MODE_AUTO):
    """Many references against a sharded store without the peer-memory exchange (CUDA IPC closed): multi_run on this rank's
    shard, its per-query lists as records in device memory, ONE NCCL all-gather, then the per-query merge on the device
    (muse_merge_partials_many).  Returns what Exchange.run_many returns -- identical on every rank."""
    import torch
    import torch.distributed as dist

    world = dist.get_world_size()
    sc, lg, ix, n_out = multi_run(store, refs, [], max_lag, top_n, threshold, sign_filter, mode=mode, raw=True)
    Q = len(n_out)
    if Q == 0 or top_n < 1:
        return _triples(sc, lg, ix, n_out)
    mine = torch.from_numpy(multi_records(sc, lg, ix, n_out).view(np.uint8).reshape(-1)).cuda()
    allr = torch.empty(world * mine.numel(), dtype=torch.uint8, device=mine.device)
    dist.all_gather_into_tensor(allr, mine)
    torch.cuda.current_stream().synchronize()
    msc, mlg, mix, mn = merge_partials_many(store.ctx, allr.data_ptr(), world, Q, top_n)
    mn = np.where(n_out < 0, -1, mn)          # std(ref) == 0: the same on every rank
    return _triples(msc, mlg, mix, mn)


class Exchange:
    """muse_exchange: the shard's top_n records go into every rank's receive buffer over NVLink peer memory,
    written by the selection kernel itself (no library collective on the data path).  Setup exchanges the CUDA
    IPC handles once with torch.distributed (any backend); ranks must call run() the same number of times."""

    def __init__(self, ctx: Context, capacity: int):
        import torch.distributed as dist
        self.ctx = ctx
        self.h = _vp()
        self.capacity = int(capacity)
        if not (dist.is_available() and dist.is_initialized()):      # a single process: the push targets only itself
            _check(lib().muse_exchange_create(ctx.h, 0, 1, self.capacity, C.byref(self.h)))
            return
        rank, world = dist.get_rank(), dist.get_world_size()
        # every rank takes every collective below whatever happened locally, and all of them raise together
        # when any rank failed (CUDA IPC closed in this container, no peer access): callers fall back as one
        err, mine = None, C.create_string_buffer(64)
        try:
            _check(lib().muse_exchange_create(ctx.h, rank, world, self.capacity, C.byref(self.h)))
            _check(lib().muse_exchange_ipc_handle(self.h, C.cast(mine, _vp)))
        except MuseError as e:
            err = str(e)
        handles = [None] * world
        dist.all_gather_object(handles, (bytes(mine.raw), err))
        if all(e is None for _, e in handles):
            try:
                blob = C.create_string_buffer(b"".join(h for h, _ in handles), 64 * world)
                _check(lib().muse_exchange_open_peers(self.h, C.cast(blob, _vp)))
            except MuseError as e:
                err = str(e)
        errs = [None] * world
        dist.all_gather_object(errs, err)
        bad = [(r, e) for r, e in enumerate(errs) if e is not None]
        if bad:
            self.close()
            raise MuseError(MUSE_ERR_UNSUPPORTED, "peer-memory exchange unavailable (rank %d: %s)" % bad[0])
        dist.barrier()

    def run(self, batch: DeviceBatch, max_lag: int, top_n: int, threshold: float, sign_filter: int = 0,
            mode: int = MODE_AUTO, key_cols: Sequence[int] = ()):
        """One multi-GPU step; returns the merged (scores, lags, series_idx) -- identical on every rank -- or None
        when every rank must take the host path (a record list too long for the device-side select or merge).
        key_cols: grouped run (every group representative of the shard is exchanged; the capacity must hold them)."""
        cap = max(1, int(top_n))
        sc = np.zeros(cap)
        lg = np.zeros(cap, dtype=np.int64)
        ix = np.zeros(cap, dtype=np.int64)
        n_out = C.c_int64(0)
        kc = np.asarray(list(key_cols), dtype=np.int32)
        rc = lib().muse_batch_run_exchange_ex(batch.h, self.h, kc.ctypes.data_as(_ip32) if kc.size else None, kc.size, max_lag, top_n,
                                              threshold, sign_filter, mode, _d(sc), lg.ctypes.data_as(_ip64),
                                              ix.ctypes.data_as(_ip64), C.byref(n_out))
        if rc == MUSE_ERR_UNSUPPORTED:
            return None
        _check(rc)
        k = int(n_out.value)
        return sc[:k], lg[:k], ix[:k]

    def run_many(self, store: DeviceStore, refs, max_lag: int, top_n: int, threshold: float, sign_filter: int = 0,
                 mode: int = MODE_AUTO):
        """muse_multi_run_exchange: every row of refs against the WHOLE sharded store (ungrouped), as multi_run on one store
        holding every shard would return it -- one (scores, lags, series_idx) triple per reference, None where the reference
        has zero std -- identical on every rank.  Every rank passes the same refs and arguments."""
        R = np.ascontiguousarray(refs, dtype=np.float64)
        assert R.ndim == 2
        Q, cap = R.shape[0], max(1, int(top_n))
        sc = np.zeros((max(Q, 1), cap))
        lg = np.zeros((max(Q, 1), cap), dtype=np.int64)
        ix = np.zeros((max(Q, 1), cap), dtype=np.int64)
        n_out = np.zeros(max(Q, 1), dtype=np.int64)
        _check(lib().muse_multi_run_exchange(store.h, self.h, _d(R), Q, R.shape[1], max_lag, top_n, threshold, sign_filter, mode,
                                             _d(sc), lg.ctypes.data_as(_ip64), ix.ctypes.data_as(_ip64),
                                             n_out.ctypes.data_as(_ip64)))
        return _triples(sc[:Q], lg[:Q], ix[:Q], n_out[:Q])

    def close(self):
        if self.h:
            lib().muse_exchange_destroy(self.h)
            self.h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
