"""garage_b200 -- B200 (sm_100a) erasure-coding block path for Garage.

The product is ``libgarage_ec.so`` (CUDA kernels + the C ABI declared in
``include/garage_ec.h``).  This module is the thin ctypes harness the tests and the bench
drive it with; it mirrors the C ABI one to one (same names minus the ``garage_ec_`` prefix,
same argument meaning, same error codes) and adds nothing of its own.  There is no CPU
fallback: if the library cannot be loaded or no sm_100 device is present, calls raise.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _build

__all__ = ["GarageEc", "EcError", "load_library", "lib_path", "ABI_SYMBOLS",
           "MEM_HOST", "MEM_DEVICE", "VANDERMONDE", "CAUCHY"]

OK = 0
E_INVALID, E_CUDA, E_NOMEM, E_UNRECOVERABLE, E_NODEVICE, E_ALIGN = -1, -2, -3, -4, -5, -6
E_UNCORRECTABLE = -7
VANDERMONDE, CAUCHY = 0, 1
MEM_HOST, MEM_DEVICE = 0, 1
MAX_K, MAX_M = 32, 8

# every symbol include/garage_ec.h declares (tests check the .so exports each one)
ABI_SYMBOLS = [
    "garage_ec_create", "garage_ec_create_with_matrix", "garage_ec_destroy", "garage_ec_matrix",
    "garage_ec_params", "garage_ec_strerror", "garage_ec_last_error", "garage_ec_abi_version",
    "garage_ec_shard_len", "garage_ec_stride_for", "garage_ec_encode", "garage_ec_reconstruct",
    "garage_ec_verify", "garage_ec_encode_blocks", "garage_ec_decode_blocks",
    "garage_ec_fill_random", "garage_ec_host_alloc", "garage_ec_host_alloc_wc", "garage_ec_host_free",
    "garage_ec_launch_count", "garage_ec_set_timing", "garage_ec_timing_read",
    "garage_ec_shard_sums", "garage_ec_check_sums", "garage_ec_blake2sum",
    "garage_ec_encode_blocks_with_sums", "garage_ec_scrub_repair",
    "garage_ec_numa_info", "garage_ec_bind_thread", "garage_ec_debug_fail_after",
    "garage_ec_set_sum_kind", "garage_ec_set_wait_mode", "garage_ec_copy_for_dma", "garage_ec_shard_sum_host", "garage_ec_reconstruct_stripes",
    "garage_ec_correct",
]


class EcError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("garage_ec error %d: %s" % (code, msg))
        self.code = code


def lib_path():
    return _build.SO


_lib = None


def load_library(build=True):
    """Load libgarage_ec.so (building it in-tree first if sources are newer).  Raises if the
    CUDA extension is missing -- the product path never falls back to CPU code."""
    global _lib
    if _lib is not None:
        return _lib
    if build:
        try:
            _build.build()
        except Exception:
            if not os.path.exists(_build.SO):
                raise
    if not os.path.exists(_build.SO):
        raise RuntimeError("garage_b200: %s missing -- build it with __graft_entry__.build()" % _build.SO)
    L = C.CDLL(_build.SO)
    vp, sz, i32, u32, u64 = C.c_void_p, C.c_size_t, C.c_int, C.c_uint32, C.c_uint64
    L.garage_ec_create.argtypes = [C.POINTER(vp), i32, i32, i32, i32]
    L.garage_ec_create_with_matrix.argtypes = [C.POINTER(vp), i32, i32, i32, vp]
    L.garage_ec_destroy.argtypes = [vp]
    L.garage_ec_destroy.restype = None
    L.garage_ec_matrix.argtypes = [vp, vp]
    L.garage_ec_params.argtypes = [vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]
    L.garage_ec_strerror.argtypes = [i32]
    L.garage_ec_strerror.restype = C.c_char_p
    L.garage_ec_last_error.argtypes = [vp]
    L.garage_ec_last_error.restype = C.c_char_p
    L.garage_ec_abi_version.restype = i32
    L.garage_ec_shard_len.argtypes = [u32, i32]
    L.garage_ec_shard_len.restype = u32
    L.garage_ec_stride_for.argtypes = [u32]
    L.garage_ec_stride_for.restype = sz
    L.garage_ec_encode.argtypes = [vp, vp, vp, vp, sz, sz, i32, vp]
    L.garage_ec_reconstruct.argtypes = [vp, vp, vp, vp, vp, vp, sz, sz, i32, vp]
    L.garage_ec_verify.argtypes = [vp, vp, vp, vp, sz, sz, i32, vp]
    L.garage_ec_correct.argtypes = [vp, vp, vp, vp, vp, vp, sz, sz, i32, vp]
    L.garage_ec_encode_blocks.argtypes = [vp, vp, vp, sz, vp, sz]
    L.garage_ec_encode_blocks_with_sums.argtypes = [vp, vp, vp, sz, vp, vp, sz]
    L.garage_ec_scrub_repair.argtypes = [vp, vp, vp, vp, vp, vp, sz, sz, i32, vp]
    L.garage_ec_shard_sums.argtypes = [vp, vp, vp, sz, sz, i32, vp, i32, vp]
    L.garage_ec_check_sums.argtypes = [vp, vp, vp, vp, sz, sz, i32, vp, i32, vp]
    L.garage_ec_blake2sum.argtypes = [vp, sz, vp]
    L.garage_ec_blake2sum.restype = None
    L.garage_ec_decode_blocks.argtypes = [vp, vp, vp, vp, sz, sz, vp, vp]
    L.garage_ec_fill_random.argtypes = [vp, vp, sz, u64, u64, vp]
    L.garage_ec_host_alloc.argtypes = [vp, C.POINTER(vp), sz]
    L.garage_ec_host_alloc_wc.argtypes = [vp, C.POINTER(vp), sz]
    L.garage_ec_host_free.argtypes = [vp, vp]
    L.garage_ec_host_free.restype = None
    L.garage_ec_launch_count.argtypes = [vp]
    L.garage_ec_launch_count.restype = u64
    L.garage_ec_set_timing.argtypes = [vp, i32]
    L.garage_ec_timing_read.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(u64)]
    L.garage_ec_numa_info.argtypes = [vp, C.POINTER(i32), C.POINTER(i32)]
    L.garage_ec_bind_thread.argtypes = [vp]
    L.garage_ec_debug_fail_after.argtypes = [vp, C.c_long]
    L.garage_ec_reconstruct_stripes.argtypes = [vp, vp, vp, vp, vp, vp, sz, sz]
    L.garage_ec_set_sum_kind.argtypes = [vp, i32]
    L.garage_ec_set_wait_mode.argtypes = [vp, i32]
    L.garage_ec_copy_for_dma.argtypes = [vp, vp, C.c_size_t]
    L.garage_ec_copy_for_dma.restype = None
    L.garage_ec_shard_sum_host.argtypes = [i32, vp, sz, vp]
    _lib = L
    return L


def blake2sum(data) -> bytes:
    """Garage's blake2sum (BLAKE2b-512 truncated to 32 bytes) through the library's host code."""
    L = load_library()
    a = np.frombuffer(bytes(data), dtype=np.uint8) if not isinstance(data, np.ndarray) else np.ascontiguousarray(data)
    out = np.zeros(32, dtype=np.uint8)
    L.garage_ec_blake2sum(C.c_void_p(a.ctypes.data) if a.size else None, a.size, C.c_void_p(out.ctypes.data))
    return out.tobytes()


SUM_BLAKE2, SUM_ADLER8 = 0, 1


def shard_sum_host(kind, data) -> bytes:
    """the 32-byte per-shard tag of `kind` computed by the library's host code"""
    L = load_library()
    a = np.frombuffer(bytes(data), dtype=np.uint8) if not isinstance(data, np.ndarray) else np.ascontiguousarray(data)
    out = np.zeros(32, dtype=np.uint8)
    rc = L.garage_ec_shard_sum_host(kind, C.c_void_p(a.ctypes.data) if a.size else None, a.size, C.c_void_p(out.ctypes.data))
    if rc:
        raise EcError(rc, "shard_sum_host")
    return out.tobytes()


def copy_for_dma(dst, src):
    """copy `src` into `dst` (numpy uint8 views, dst normally pinned) with non-temporal stores: garage_ec_copy_for_dma"""
    assert dst.dtype == np.uint8 and src.dtype == np.uint8 and dst.size >= src.size
    load_library().garage_ec_copy_for_dma(C.c_void_p(dst.ctypes.data), C.c_void_p(src.ctypes.data), src.size)


def _ptr(x):
    """device tensor / numpy array / int / None -> void*"""
    if x is None:
        return None
    if isinstance(x, int):
        return C.c_void_p(x)
    if isinstance(x, np.ndarray):
        return C.c_void_p(x.ctypes.data)
    if hasattr(x, "data_ptr"):
        return C.c_void_p(x.data_ptr())
    raise TypeError(type(x))


def _is_device(x):
    return hasattr(x, "data_ptr") and getattr(x, "is_cuda", False)


class GarageEc:
    """One context = (GPU, k, m, matrix): mirrors ``garage_ec_ctx``.

    Buffers are torch CUDA uint8 tensors (DEVICE mode: enqueued on torch's current stream)
    or numpy uint8 arrays (HOST mode: synchronous, staged through the library's lanes).
    """

    def __init__(self, device=0, k=10, m=4, kind=VANDERMONDE, matrix=None):
        self._L = load_library()
        h = C.c_void_p()
        if matrix is not None:
            mat = np.ascontiguousarray(matrix, dtype=np.uint8)
            if mat.shape != (m, k):
                raise ValueError("matrix must be m x k")
            rc = self._L.garage_ec_create_with_matrix(C.byref(h), device, k, m, _ptr(mat))
        else:
            rc = self._L.garage_ec_create(C.byref(h), device, k, m, kind)
        if rc != OK:
            raise EcError(rc, self._L.garage_ec_strerror(rc).decode())
        self._h = h
        self.device, self.k, self.m = device, k, m

    # -- lifecycle
    def close(self):
        if getattr(self, "_h", None):
            self._L.garage_ec_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc, allow=()):
        if rc != OK and rc not in allow:
            msg = self._L.garage_ec_strerror(rc).decode()
            if rc == E_CUDA:
                msg += " (" + self._L.garage_ec_last_error(self._h).decode() + ")"
            raise EcError(rc, msg)
        return rc

    def _stream(self, *bufs):
        if any(_is_device(b) for b in bufs):
            import torch

            return MEM_DEVICE, C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        return MEM_HOST, None

    # -- introspection
    def matrix(self):
        out = np.zeros((self.m, self.k), dtype=np.uint8)
        self._check(self._L.garage_ec_matrix(self._h, _ptr(out)))
        return out

    def shard_len(self, block_len):
        return int(self._L.garage_ec_shard_len(block_len, self.k))

    def stride_for(self, shard_len):
        return int(self._L.garage_ec_stride_for(shard_len))

    def launch_count(self):
        return int(self._L.garage_ec_launch_count(self._h))

    def set_timing(self, on=True):
        self._check(self._L.garage_ec_set_timing(self._h, 1 if on else 0))

    def timing_read(self):
        ms, n = C.c_double(0), C.c_uint64(0)
        self._check(self._L.garage_ec_timing_read(self._h, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    # -- the three batch operations (shard layout; see include/garage_ec.h)
    def encode(self, data, parity, stride, n, shard_len=None):
        kind, st = self._stream(data, parity)
        return self._check(self._L.garage_ec_encode(self._h, _ptr(data), _ptr(parity), _ptr(shard_len),
                                                    stride, n, kind, st))

    def reconstruct(self, shards, present, stride, n, want=None, status=None, shard_len=None,
                    allow_unrecoverable=True):
        kind, st = self._stream(shards)
        allow = (E_UNRECOVERABLE,) if allow_unrecoverable else ()
        return self._check(self._L.garage_ec_reconstruct(self._h, _ptr(shards), _ptr(present), _ptr(want),
                                                         _ptr(status), _ptr(shard_len), stride, n, kind, st),
                           allow)

    def reconstruct_stripes(self, stripes, present, stride, want=None, status=None, shard_len=None):
        """gather form: `stripes` is a list of numpy arrays, one (k+m)*stride buffer per stripe"""
        n = len(stripes)
        ptrs = (C.c_void_p * n)(*[a.ctypes.data for a in stripes])
        return self._check(self._L.garage_ec_reconstruct_stripes(self._h, C.cast(ptrs, C.c_void_p), _ptr(present),
                                                                 _ptr(want), _ptr(status), _ptr(shard_len), stride, n),
                           (E_UNRECOVERABLE,))

    def verify(self, shards, mismatch, stride, n, shard_len=None):
        kind, st = self._stream(shards)
        return self._check(self._L.garage_ec_verify(self._h, _ptr(shards), _ptr(mismatch), _ptr(shard_len),
                                                    stride, n, kind, st))

    def correct(self, shards, stride, n, present=None, status=None, fixed=None, shard_len=None):
        """error-locating decode: find and repair wrong shards from the parity alone (garage_ec_correct).
        HOST mode returns 0, E_UNRECOVERABLE or E_UNCORRECTABLE (per-stripe detail in `status`)."""
        kind, st = self._stream(shards)
        return self._check(self._L.garage_ec_correct(self._h, _ptr(shards), _ptr(present), _ptr(status), _ptr(fixed),
                                                     _ptr(shard_len), stride, n, kind, st),
                           (E_UNRECOVERABLE, E_UNCORRECTABLE))

    # -- per-shard integrity (blake2sum of every shard)
    def shard_sums(self, shards, sums_out, stride, n, per_stripe, shard_len=None):
        kind, st = self._stream(shards)
        return self._check(self._L.garage_ec_shard_sums(self._h, _ptr(shards), _ptr(shard_len), stride, n,
                                                        per_stripe, _ptr(sums_out), kind, st))

    def check_sums(self, shards, expect, bad_out, stride, n, per_stripe, shard_len=None):
        kind, st = self._stream(shards)
        return self._check(self._L.garage_ec_check_sums(self._h, _ptr(shards), _ptr(expect), _ptr(shard_len),
                                                        stride, n, per_stripe, _ptr(bad_out), kind, st))

    def scrub_repair(self, shards, expect_sums, bad_out, stride, n, status=None, shard_len=None):
        """config-5 sweep: hash every shard, rebuild the corrupt ones in place."""
        kind, st = self._stream(shards)
        return self._check(self._L.garage_ec_scrub_repair(self._h, _ptr(shards), _ptr(expect_sums), _ptr(bad_out),
                                                          _ptr(status), _ptr(shard_len), stride, n, kind, st),
                           (E_UNRECOVERABLE,))

    # -- block-level host API
    def encode_blocks(self, blocks, parity_out, stride, sums_out=None):
        """blocks: list of 1-D uint8 numpy arrays; parity_out: numpy (n*m*stride);
        sums_out: optional numpy n*(k+m)*32 for the per-shard blake2sums."""
        n = len(blocks)
        ptrs = (C.c_void_p * n)(*[b.ctypes.data for b in blocks])
        lens = np.array([b.size for b in blocks], dtype=np.uint32)
        return self._check(self._L.garage_ec_encode_blocks_with_sums(self._h, C.cast(ptrs, C.c_void_p), _ptr(lens),
                                                                     n, _ptr(parity_out), _ptr(sums_out), stride))

    def decode_blocks(self, shards, present, block_lens, stride, blocks_out, status=None):
        n = len(blocks_out)
        ptrs = (C.c_void_p * n)(*[b.ctypes.data for b in blocks_out])
        lens = np.ascontiguousarray(block_lens, dtype=np.uint32)
        return self._check(self._L.garage_ec_decode_blocks(self._h, _ptr(shards), _ptr(present), _ptr(lens), n,
                                                           stride, C.cast(ptrs, C.c_void_p), _ptr(status)),
                           (E_UNRECOVERABLE,))

    # -- harness utilities
    def fill_random(self, dst, nbytes, seed, offset=0):
        import torch

        st = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        return self._check(self._L.garage_ec_fill_random(self._h, _ptr(dst), nbytes, seed, offset, st))

    def host_alloc(self, nbytes, write_combined=False):
        """pinned host buffer as a numpy uint8 array (freed with host_free)."""
        p = C.c_void_p()
        fn = self._L.garage_ec_host_alloc_wc if write_combined else self._L.garage_ec_host_alloc
        self._check(fn(self._h, C.byref(p), nbytes))
        arr = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(nbytes,))
        return arr, p

    def host_free(self, p):
        self._L.garage_ec_host_free(self._h, p)

    def numa_info(self):
        """(NUMA node of the GPU, node the last host_alloc landed on); -1 = unknown"""
        a, b = C.c_int(-1), C.c_int(-1)
        self._check(self._L.garage_ec_numa_info(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def bind_thread(self):
        """pin the calling thread to the CPUs of the GPU's NUMA node; True if bound"""
        return self._L.garage_ec_bind_thread(self._h) == 0

    def set_wait_mode(self, blocking):
        """HOST-mode calls wait by sleeping on an event (True) instead of spinning in the driver (False, default)"""
        self._check(self._L.garage_ec_set_wait_mode(self._h, 1 if blocking else 0))

    def set_sum_kind(self, kind):
        self._check(self._L.garage_ec_set_sum_kind(self._h, kind))

    def debug_fail_after(self, n_calls):
        self._check(self._L.garage_ec_debug_fail_after(self._h, n_calls))
