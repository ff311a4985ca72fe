"""bwtc_b200 — B200-native forward Burrows-Wheeler transform engine for pjmikkol/bwtc.

Python is only the test / bench harness language here.  The product is
``bwtc_b200/libbwtc_cuda.so`` (hand-written sm_100a kernels + C++ host code behind the C-ABI of
``include/bwtc_cuda.h``) and the C++ mirror of the reference's ``BWTransform`` / ``BWTManager`` interface in
``bwtc_b200/host/``.  This module binds the C-ABI with ctypes and mirrors the reference's names
(``BWTBlock``, ``BWTManager``, ``CudaBWTransform``; reference: BWTBlock.hpp:39-72,
bwtransforms/BWTManager.hpp:40-58, bwtransforms/BWTransform.hpp:48-70) so parity tests read like the
reference's own tests (test/InverseBwtTest.cpp:57-66).

There is NO CPU fallback: if the CUDA library is missing or fails to load, importing the engine classes
raises ``BwtcCudaUnavailable``; nothing in this package ever calls ``oracle/``.
"""
from __future__ import annotations

import ctypes
import os
from typing import List, Optional, Sequence, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libbwtc_cuda.so")
GEN_LIB_PATH = os.path.join(_HERE, "libbwtc_gen.so")
INTEGRATION_LIB_PATH = os.path.join(_HERE, "libbwtc_integration.so")

MAX_ROUNDS = 40
MAX_BLOCK = 0x7FFFFFFD            # BWTC_CUDA_MAX_BLOCK
SCRATCH_BYTES_PER_SUFFIX = 40     # BWTC_CUDA_SCRATCH_BYTES_PER_SUFFIX
SCRATCH_FIXED_BYTES = 8 << 20     # BWTC_CUDA_SCRATCH_FIXED_BYTES
ECORRUPT = -6                     # BWTC_CUDA_ECORRUPT: an inverse input that is not the BWT of any text
EVERIFY = -7                      # BWTC_CUDA_EVERIFY: a verified forward output did not restore its input
FLAG_VERIFIED = 1 << 6            # stats flags bit 6: the forward output was verified on the device
FLAG_CORRUPT = 1 << 7             # stats flags bit 7: this inverse block is corrupt
FLAG_SA = 1 << 8                  # stats flags bit 8: this call produced a suffix array (divsufsort)
FLAG_LCP = 1 << 9                 # stats flags bit 9: this call produced an LCP array (divsufsort_lcp)
FLAG_ROUND0_BUCKETS = 1 << 10     # stats flags bit 10: round 0 sorted its low key digits bucket by bucket (k_bucket_sort)
FLAG_SEARCH = 1 << 11             # stats flags bit 11: this call was a pattern search (sa_search)
FLAG_LZ77 = 1 << 12               # stats flags bit 12: this call produced an LZ77 factorisation (lz77)


class BwtcCudaUnavailable(RuntimeError):
    """The CUDA engine library is not built / not loadable.  There is no fallback path."""


class BwtcCudaError(RuntimeError):
    def __init__(self, code: int, msg: str, blocks: Optional[List[int]] = None):
        super().__init__(f"bwtc_cuda error {code}: {msg}")
        self.code = code
        self.blocks = blocks  # ECORRUPT from inverse_blocks: the indices of the corrupt blocks


class Stats(ctypes.Structure):
    """Mirror of ``bwtc_cuda_stats`` (include/bwtc_cuda.h)."""

    _fields_ = [
        ("n_suffixes", ctypes.c_uint32),
        ("sigma", ctypes.c_uint32),
        ("bits_per_char", ctypes.c_uint32),
        ("chars_round0", ctypes.c_uint32),
        ("key_bytes_round0", ctypes.c_uint32),
        ("rounds", ctypes.c_uint32),
        ("live", ctypes.c_uint32 * MAX_ROUNDS),
        ("passes", ctypes.c_uint32 * MAX_ROUNDS),
        ("prefix_len", ctypes.c_uint32 * MAX_ROUNDS),
        ("kernel_launches", ctypes.c_uint64),
        ("algorithmic_bytes", ctypes.c_uint64),
        ("gpu_ms", ctypes.c_float),
        ("sort_ms", ctypes.c_float),
        ("sort_bytes", ctypes.c_uint64),
        ("sort_launches", ctypes.c_uint32),
        ("sort0_launches", ctypes.c_uint32),
        ("sort0_bytes", ctypes.c_uint64),
        ("sort0_ms", ctypes.c_float),
        ("flags", ctypes.c_uint32),
        ("batch_blocks", ctypes.c_uint32),
        ("round0_big_buckets", ctypes.c_uint32),
    ]

    def as_dict(self) -> dict:
        r = int(self.rounds)
        return {
            "n_suffixes": int(self.n_suffixes), "sigma": int(self.sigma), "bits_per_char": int(self.bits_per_char),
            "chars_round0": int(self.chars_round0), "key_bytes_round0": int(self.key_bytes_round0), "rounds": r,
            "live": [int(self.live[i]) for i in range(r)], "passes": [int(self.passes[i]) for i in range(r)],
            "prefix_len": [int(self.prefix_len[i]) for i in range(r)],
            "kernel_launches": int(self.kernel_launches), "algorithmic_bytes": int(self.algorithmic_bytes),
            "gpu_ms": float(self.gpu_ms), "sort_ms": float(self.sort_ms), "sort_bytes": int(self.sort_bytes),
            "sort_launches": int(self.sort_launches), "sort0_launches": int(self.sort0_launches),
            "sort0_bytes": int(self.sort0_bytes), "sort0_ms": float(self.sort0_ms), "flags": int(self.flags),
            "batch_blocks": int(self.batch_blocks), "round0_big_buckets": int(self.round0_big_buckets),
        }


RUNS_OVERFLOW = 0xFFFFFFFF


class Runs(ctypes.Structure):
    """Mirror of ``bwtc_cuda_runs`` (include/bwtc_cuda.h)."""

    _fields_ = [("capacity", ctypes.c_uint32), ("count", ctypes.c_uint32), ("symbol", ctypes.c_void_p), ("start", ctypes.c_void_p)]


_u8p = ctypes.POINTER(ctypes.c_uint8)
_u32p = ctypes.POINTER(ctypes.c_uint32)
_vp = ctypes.c_void_p

# every symbol include/bwtc_cuda.h declares: (name, restype, argtypes)
C_ABI = [
    ("bwtc_cuda_device_count", ctypes.c_int, []),
    ("bwtc_cuda_version", ctypes.c_char_p, []),
    ("bwtc_cuda_stats_sizeof", ctypes.c_uint32, []),
    ("bwtc_cuda_global_error", ctypes.c_char_p, []),
    ("bwtc_cuda_ctx_create", ctypes.c_int, [ctypes.POINTER(_vp), ctypes.c_int, ctypes.c_uint32]),
    ("bwtc_cuda_ctx_destroy", None, [_vp]),
    ("bwtc_cuda_scratch_bytes", ctypes.c_uint64, [ctypes.c_uint32]),
    ("bwtc_cuda_last_error", ctypes.c_char_p, [_vp]),
    ("bwtc_cuda_get_stats", ctypes.c_int, [_vp, ctypes.POINTER(Stats)]),
    ("bwtc_cuda_ctx_set_round0", ctypes.c_int, [_vp, ctypes.c_uint32, ctypes.c_uint32]),
    ("bwtc_cuda_ctx_set_timing", ctypes.c_int, [_vp, ctypes.c_int]),
    ("bwtc_cuda_ctx_set_verify", ctypes.c_int, [_vp, ctypes.c_int]),
    ("bwtc_cuda_ctx_set_debug", ctypes.c_int, [_vp, ctypes.c_uint32]),
    ("bwtc_cuda_debug_read", ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_uint64, _vp, ctypes.c_uint64]),
    ("bwtc_cuda_divbwtf", ctypes.c_int64, [_vp, _vp, _vp, ctypes.c_uint32, _vp, ctypes.c_uint32, _vp]),
    ("bwtc_cuda_divbwt", ctypes.c_int64, [_vp, _vp, _vp, ctypes.c_uint32, _vp, ctypes.c_uint32]),
    ("bwtc_cuda_divsufsort", ctypes.c_int, [_vp, _vp, _vp, ctypes.c_uint32]),
    ("bwtc_cuda_divsufsort_device", ctypes.c_int, [_vp, _vp, _vp, ctypes.c_uint32]),
    ("bwtc_cuda_sufcheck", ctypes.c_int, [_vp, _vp, _vp, ctypes.c_uint32]),
    ("bwtc_cuda_divsufsort_lcp", ctypes.c_int, [_vp, _vp, _vp, _vp, ctypes.c_uint32]),
    ("bwtc_cuda_divsufsort_lcp_device", ctypes.c_int, [_vp, _vp, _vp, _vp, ctypes.c_uint32]),
    ("bwtc_cuda_sa_search", ctypes.c_int,
     [_vp, _vp, ctypes.c_uint32, _vp, ctypes.c_uint32, _vp, _vp, ctypes.c_uint32, _vp, _vp]),
    ("bwtc_cuda_sa_search_device", ctypes.c_int,
     [_vp, _vp, ctypes.c_uint32, _vp, ctypes.c_uint32, _vp, _vp, ctypes.c_uint32, _vp, _vp]),
    ("bwtc_cuda_lz77", ctypes.c_int64, [_vp, _vp, ctypes.c_uint32, _vp, _vp, ctypes.c_uint32]),
    ("bwtc_cuda_lz77_device", ctypes.c_int64, [_vp, _vp, ctypes.c_uint32, _vp, _vp, ctypes.c_uint32]),
    ("bwtc_cuda_bwt_block", ctypes.c_int64, [_vp, _vp, ctypes.c_uint32, _vp, ctypes.c_uint32, _vp]),
    ("bwtc_cuda_bwt_block_device", ctypes.c_int64, [_vp, _vp, _vp, ctypes.c_uint32, _vp, ctypes.c_uint32, _vp]),
    ("bwtc_cuda_bwt_block_runs", ctypes.c_int64, [_vp, _vp, ctypes.c_uint32, _vp, ctypes.c_uint32, _vp, _vp]),
    ("bwtc_cuda_inverse_block", ctypes.c_int64, [_vp, _vp, ctypes.c_uint32, _vp, ctypes.c_uint32]),
    ("bwtc_cuda_inverse_block_device", ctypes.c_int64, [_vp, _vp, _vp, ctypes.c_uint32, ctypes.c_uint32]),
    ("bwtc_cuda_inverse_raw", ctypes.c_int64, [_vp, _vp, ctypes.c_uint32, _vp, ctypes.c_uint32]),
    ("bwtc_cuda_inverse_blocks", ctypes.c_int, [_vp, _vp, _vp, _vp, ctypes.c_uint32, ctypes.c_int, _vp, _vp]),
    ("bwtc_cuda_bwt_blocks", ctypes.c_int,
     [_vp, _vp, _vp, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_int, _vp, _vp, _vp]),
    ("bwtc_cuda_num_starting_points", ctypes.c_uint32, [ctypes.c_uint32, ctypes.c_uint32]),
    ("bwtc_cuda_pipeline_create", ctypes.c_int, [ctypes.POINTER(_vp), ctypes.c_int, ctypes.c_int, ctypes.c_uint32]),
    ("bwtc_cuda_pipeline_destroy", None, [_vp]),
    ("bwtc_cuda_pipeline_error", ctypes.c_char_p, [_vp]),
    ("bwtc_cuda_pipeline_set_round0", ctypes.c_int, [_vp, ctypes.c_uint32, ctypes.c_uint32]),
    ("bwtc_cuda_pipeline_set_timing", ctypes.c_int, [_vp, ctypes.c_int]),
    ("bwtc_cuda_pipeline_set_verify", ctypes.c_int, [_vp, ctypes.c_int]),
    ("bwtc_cuda_pipeline_run", ctypes.c_int,
     [_vp, _vp, _vp, _vp, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_int, _vp, _vp, _vp, _vp]),
    ("bwtc_cuda_pipeline_submit", ctypes.c_int,
     [_vp, _vp, _vp, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_int, _vp, _vp, _vp, _vp, ctypes.POINTER(ctypes.c_uint64)]),
    ("bwtc_cuda_pipeline_wait", ctypes.c_int, [_vp, ctypes.c_uint64]),
    ("bwtc_cuda_pipeline_submit_inverse", ctypes.c_int,
     [_vp, _vp, _vp, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_int, _vp, ctypes.POINTER(ctypes.c_uint64)]),
    ("bwtc_cuda_pipeline_submit_runs", ctypes.c_int,
     [_vp, _vp, _vp, ctypes.c_uint32, ctypes.c_uint32, _vp, _vp, _vp, _vp, ctypes.POINTER(ctypes.c_uint64)]),
    ("bwtc_cuda_pipeline_timing_begin", ctypes.c_int, [_vp]),
    ("bwtc_cuda_pipeline_timing_end", ctypes.c_float, [_vp]),
]

_lib = None


def load_library(path: Optional[str] = None) -> ctypes.CDLL:
    """dlopen the C-ABI library and bind every declared symbol.  Raises if it is missing: no fallback."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise BwtcCudaUnavailable(
            f"{p} not found - build it with `python -c 'import __graft_entry__ as g; g.build()'`; "
            "the engine has no CPU fallback")
    try:
        lib = ctypes.CDLL(p)
    except OSError as e:  # pragma: no cover - depends on the box
        raise BwtcCudaUnavailable(f"cannot load {p}: {e}") from e
    for name, res, args in C_ABI:
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    if path is None:
        _lib = lib
    return lib


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data


def pack_patterns(seq) -> Tuple[np.ndarray, np.ndarray]:
    """Patterns (bytes, str as latin-1, or uint8 arrays) as the (P, P_off) pair sa_search takes: P = their bytes one
    after the other (uint8), P_off = len(seq) + 1 offsets (uint64), pattern i = P[P_off[i]:P_off[i+1]]."""
    parts = [np.frombuffer(p.encode("latin-1") if isinstance(p, str) else bytes(p), np.uint8) for p in seq]
    P_off = np.zeros(len(parts) + 1, np.uint64)
    if parts:
        P_off[1:] = np.cumsum([p.size for p in parts], dtype=np.uint64)
    P = np.concatenate(parts) if parts else np.zeros(0, np.uint8)
    return np.ascontiguousarray(P, np.uint8), P_off


def num_starting_points(block_bytes: int, starts: int) -> int:
    """BWTManager::setStartingPoints clamp + BWTBlock::prepareLFpowers (BWTManager.cpp:60-64, BWTBlock.cpp:104-108)."""
    return int(load_library().bwtc_cuda_num_starting_points(block_bytes, starts))


class CudaContext:
    """One in-flight block: a CUDA stream + device scratch (bwtc_cuda_ctx)."""

    def __init__(self, max_block_bytes: int, device: int = 0, lib_path: Optional[str] = None):
        self._lib = load_library(lib_path)
        h = _vp()
        rc = self._lib.bwtc_cuda_ctx_create(ctypes.byref(h), device, max_block_bytes)
        if rc != 0:
            raise BwtcCudaError(rc, self._lib.bwtc_cuda_global_error().decode())
        self._h = h
        self.max_block_bytes = max_block_bytes

    def close(self):
        if getattr(self, "_h", None):
            self._lib.bwtc_cuda_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int) -> int:
        if rc < 0:
            raise BwtcCudaError(rc, self._lib.bwtc_cuda_last_error(self._h).decode())
        return rc

    def set_round0(self, chars: int = 0, key_bytes: int = 0):
        self._check(self._lib.bwtc_cuda_ctx_set_round0(self._h, chars, key_bytes))

    def set_timing(self, detail: int):
        self._check(self._lib.bwtc_cuda_ctx_set_timing(self._h, detail))

    def set_debug(self, max_rounds: int):
        self._check(self._lib.bwtc_cuda_ctx_set_debug(self._h, max_rounds))

    def set_verify(self, on: bool):
        """bwtc_cuda_ctx_set_verify: every forward call, block contract and raw (divbwtf), inverts its output on the device
        and compares it with the input, and checks every LFpowers entry against the inversion, before it returns; a
        mismatch raises BwtcCudaError with code EVERIFY and leaves the input, LFpowers and freqs in place.  The initial
        value comes from BWTC_VERIFY (read when the context is created, default off); this call overrides it."""
        self._check(self._lib.bwtc_cuda_ctx_set_verify(self._h, 1 if on else 0))

    def debug_read(self, which: int, dtype, count: int, offset_bytes: int = 0) -> np.ndarray:
        out = np.empty(count, dtype=dtype)
        self._check(self._lib.bwtc_cuda_debug_read(self._h, which, offset_bytes, out.ctypes.data, out.nbytes))
        return out

    def stats(self) -> dict:
        s = Stats()
        self._lib.bwtc_cuda_get_stats(self._h, ctypes.byref(s))
        return s.as_dict()

    # raw contract: divbwtf(T, U, A=NULL, n, LFpowers, nLFpowers, freqs) — divsufsort.h:91-94
    def divbwtf(self, T: np.ndarray, U: np.ndarray, LFpowers: np.ndarray, freqs: Optional[np.ndarray]) -> int:
        assert T.dtype == np.uint8 and U.dtype == np.uint8 and LFpowers.dtype == np.uint32
        return self._check(self._lib.bwtc_cuda_divbwtf(self._h, T.ctypes.data, U.ctypes.data, T.size,
                                                        LFpowers.ctypes.data, LFpowers.size, _ptr(freqs)))

    def last_error(self) -> str:
        return self._lib.bwtc_cuda_last_error(self._h).decode()

    # suffix array of a raw text: libdivsufsort's divsufsort(T, SA, n) / sufcheck(T, SA, n, verbose)
    def divsufsort(self, T: np.ndarray, SA: Optional[np.ndarray] = None) -> np.ndarray:
        """The suffix array of T (uint8) under the raw contract's order: int32[T.size], or written into SA (int32,
        pageable or pinned) when given.  Raises BwtcCudaError on failure (EVERIFY with verification on: SA untouched)."""
        assert T.dtype == np.uint8 and T.flags.c_contiguous
        if SA is None:
            SA = np.empty(T.size, dtype=np.int32)
        assert SA.dtype == np.int32 and SA.size >= T.size and SA.flags.c_contiguous
        self._check(self._lib.bwtc_cuda_divsufsort(self._h, T.ctypes.data, SA.ctypes.data, T.size))
        return SA

    def divsufsort_device(self, d_T: int, d_SA: int, n: int) -> None:
        """divsufsort with T (n bytes) and SA (n int32, 4-byte aligned) in device memory (e.g. torch data_ptr())."""
        self._check(self._lib.bwtc_cuda_divsufsort_device(self._h, d_T, d_SA, n))

    def divsufsort_lcp(self, T: np.ndarray, SA: Optional[np.ndarray] = None,
                       LCP: Optional[np.ndarray] = None) -> Tuple[np.ndarray, np.ndarray]:
        """(SA, LCP) of T (uint8): the suffix array as divsufsort returns it and its LCP array (LCP[0] = 0, LCP[r] = the
        longest common prefix of suffixes SA[r-1] and SA[r]), int32[T.size] each, or written into SA / LCP (int32,
        pageable or pinned) when given.  Raises BwtcCudaError on failure (EVERIFY with verification on: both untouched)."""
        assert T.dtype == np.uint8 and T.flags.c_contiguous
        if SA is None:
            SA = np.empty(T.size, dtype=np.int32)
        if LCP is None:
            LCP = np.empty(T.size, dtype=np.int32)
        for a in (SA, LCP):
            assert a.dtype == np.int32 and a.size >= T.size and a.flags.c_contiguous
        self._check(self._lib.bwtc_cuda_divsufsort_lcp(self._h, T.ctypes.data, SA.ctypes.data, LCP.ctypes.data, T.size))
        return SA, LCP

    def divsufsort_lcp_device(self, d_T: int, d_SA: int, d_LCP: int, n: int) -> None:
        """divsufsort_lcp with T (n bytes, any alignment), SA and LCP (n int32 each, 4-byte aligned, not overlapping) in
        device memory (e.g. torch data_ptr())."""
        self._check(self._lib.bwtc_cuda_divsufsort_lcp_device(self._h, d_T, d_SA, d_LCP, n))

    def sufcheck(self, T: np.ndarray, SA: np.ndarray) -> bool:
        """True if SA (int32) is the suffix array of T (uint8); False if not (last_error() names the first offending row).
        Other failures raise BwtcCudaError."""
        assert T.dtype == np.uint8 and SA.dtype == np.int32 and SA.size == T.size
        assert T.flags.c_contiguous and SA.flags.c_contiguous
        rc = self._lib.bwtc_cuda_sufcheck(self._h, T.ctypes.data, SA.ctypes.data, T.size)
        if rc == ECORRUPT:
            return False
        self._check(rc)
        return True

    # pattern search in a suffix array: libdivsufsort's sa_search(T, Tsize, P, Psize, SA, SAsize, &idx), batched
    def sa_search(self, T: np.ndarray, SA: np.ndarray, P: np.ndarray, P_off: np.ndarray,
                  left: Optional[np.ndarray] = None, size: Optional[np.ndarray] = None) -> Tuple[np.ndarray, np.ndarray]:
        """(left, size), int32[count] each (or written into left / size when given): pattern i = P[P_off[i]:P_off[i+1]]
        (see pack_patterns) matches the rows SA[left[i] : left[i] + size[i]] of SA (int32, sorted suffixes of T, entries
        outside [0, T.size) stand for the empty suffix); with no match, left[i] is where it would be inserted.  Host arrays,
        pageable or pinned.  Raises BwtcCudaError on failure (decreasing offsets: EARG, left / size untouched)."""
        assert T.dtype == np.uint8 and SA.dtype == np.int32 and P.dtype == np.uint8 and P_off.dtype == np.uint64
        for a in (T, SA, P, P_off):
            assert a.flags.c_contiguous
        count = P_off.size - 1
        assert count >= 0
        if left is None:
            left = np.empty(count, np.int32)
        if size is None:
            size = np.empty(count, np.int32)
        for a in (left, size):
            assert a.dtype == np.int32 and a.size >= count and a.flags.c_contiguous
        self._check(self._lib.bwtc_cuda_sa_search(self._h, T.ctypes.data, T.size, SA.ctypes.data, SA.size, P.ctypes.data,
                                                  P_off.ctypes.data, count, left.ctypes.data, size.ctypes.data))
        return left, size

    def sa_search_device(self, d_T: int, n: int, d_SA: int, SAsize: int, d_P: int, d_P_off: int, count: int,
                         d_left: int, d_size: int) -> None:
        """sa_search with every array in device memory (e.g. torch data_ptr()): T (n bytes) and P at any alignment, SA,
        left and size (int32) 4-byte aligned, P_off (count + 1 uint64) 8-byte aligned."""
        self._check(self._lib.bwtc_cuda_sa_search_device(self._h, d_T, n, d_SA, SAsize, d_P, d_P_off, count, d_left,
                                                         d_size))

    # greedy LZ77 factorisation (self-reference allowed, KKP's source rule; include/bwtc_cuda.h)
    def lz77(self, T: np.ndarray, src: Optional[np.ndarray] = None,
             len: Optional[np.ndarray] = None) -> Tuple[np.ndarray, np.ndarray]:
        """(src, len), int32[z] each: the greedy LZ77 phrases of T (uint8).  Phrase k is a literal when len[k] == 0 (src[k]
        is the byte) and otherwise copies len[k] bytes from position src[k], before its start.  The call runs with capacity
        min(src.size, len.size), T.size for fresh arrays (z <= T.size always, so no count query is needed), and returns
        views of the first z entries.  Given arrays (int32, pageable or pinned) too small for z raise ValueError and stay
        untouched.  Raises BwtcCudaError on failure (EVERIFY with verification on: src / len untouched)."""
        assert T.dtype == np.uint8 and T.flags.c_contiguous
        n = T.size
        if src is None:
            src = np.empty(n, np.int32)
        if len is None:
            len = np.empty(n, np.int32)
        for a in (src, len):
            assert a.dtype == np.int32 and a.flags.c_contiguous
        cap = min(src.size, len.size)
        z = self._check(self._lib.bwtc_cuda_lz77(self._h, T.ctypes.data, n, src.ctypes.data, len.ctypes.data, cap))
        if z > cap:
            raise ValueError(f"lz77: {z} phrases do not fit arrays of {cap} entries (src / len untouched)")
        return src[:z], len[:z]

    def lz77_device(self, d_T: int, n: int, d_src: int, d_len: int, capacity: int) -> int:
        """lz77 with T (n bytes, any alignment) and the phrase arrays (capacity int32 each, 4-byte aligned, not
        overlapping) in device memory (e.g. torch data_ptr()).  Returns z; the arrays are written only when z <= capacity
        (capacity 0 with null arrays: a count query)."""
        return self._check(self._lib.bwtc_cuda_lz77_device(self._h, d_T, n, d_src or None, d_len or None, capacity))

    # block contract: BWTransform::doTransform(BWTBlock&, freqs) — BWTransform.cpp:52-64
    def bwt_block(self, block: np.ndarray, LFpowers: np.ndarray, freqs: Optional[np.ndarray]) -> int:
        assert block.dtype == np.uint8 and LFpowers.dtype == np.uint32
        return self._check(self._lib.bwtc_cuda_bwt_block(self._h, block.ctypes.data, block.size,
                                                          LFpowers.ctypes.data, LFpowers.size, _ptr(freqs)))

    def bwt_block_runs(self, block: np.ndarray, LFpowers: np.ndarray, freqs: Optional[np.ndarray], capacity: int):
        """bwtc_cuda_bwt_block_runs: the block transform + the maximal runs of its output (symbol[], start[]) when there
        are at most `capacity` of them, else None (SURVEY.md §8f row f3)."""
        sym = np.zeros(max(capacity, 1), np.uint8)
        start = np.zeros(max(capacity, 1), np.uint32)
        r = Runs(capacity, 0, sym.ctypes.data, start.ctypes.data)
        pidx = self._check(self._lib.bwtc_cuda_bwt_block_runs(self._h, block.ctypes.data, block.size, LFpowers.ctypes.data,
                                                               LFpowers.size, _ptr(freqs), ctypes.addressof(r)))
        if r.count == RUNS_OVERFLOW:
            return pidx, None
        return pidx, (sym[: r.count].copy(), start[: r.count].copy())

    # inverse, block level: InverseBWTransform::doTransform(BWTBlock&) — InverseBWT.cpp:47-51
    def inverse_block(self, block: np.ndarray, LFpowers: np.ndarray) -> int:
        assert block.dtype == np.uint8 and LFpowers.dtype == np.uint32
        return self._check(self._lib.bwtc_cuda_inverse_block(self._h, block.ctypes.data, block.size, LFpowers.ctypes.data,
                                                              LFpowers.size))

    def inverse_block_device(self, d_in: int, d_out: int, n: int, eob: int) -> int:
        return self._check(self._lib.bwtc_cuda_inverse_block_device(self._h, d_in, d_out, n, eob))

    # inverse, raw virtual: doTransform(byte* bwt, uint32 N, LFpow) — InverseBWT.hpp:49-50
    def inverse_raw(self, bwt: np.ndarray, LFpowers: np.ndarray) -> int:
        assert bwt.dtype == np.uint8 and LFpowers.dtype == np.uint32
        return self._check(self._lib.bwtc_cuda_inverse_raw(self._h, bwt.ctypes.data, bwt.size, LFpowers.ctypes.data, LFpowers.size))

    def inverse_blocks(self, blocks, LF, on_device: bool = False, out=None) -> None:
        """bwtc_cuda_inverse_blocks: restore the given blocks (uint8 arrays, or CUDA tensors / (pointer, size) pairs when
        on_device) IN PLACE, or into `out` (same kinds, same sizes).  LF: per block its LFpowers row (e.g. what bwt_blocks
        returned) or just its end-of-block row; only LF[k][0] is used.  Equal-sized runs are inverted as one device-side
        problem; stats() then describes the last run.  Corrupt blocks (not the BWT of any text with their end-of-block row)
        raise BwtcCudaError with code ECORRUPT and .blocks = their indices, after every valid block has been restored; a
        corrupt block's buffer is left as it was."""
        count = len(blocks)
        ptrs, sizes = zip(*[_block_ptr(b, on_device) for b in blocks]) if count else ((), ())
        a_in = (ctypes.c_void_p * count)(*ptrs)
        a_out = None
        if out is not None:
            assert len(out) == count
            optrs, osizes = zip(*[_block_ptr(b, on_device) for b in out]) if count else ((), ())
            assert tuple(osizes) == tuple(sizes), "out[k] must have the size of blocks[k]"
            a_out = (ctypes.c_void_p * count)(*optrs)
        a_sz = np.asarray(sizes, dtype=np.uint32)
        eob = np.asarray(LF, dtype=np.uint32)
        eob = eob.reshape(count, -1)[:, 0] if eob.size else eob
        rows = np.zeros((count, 256), dtype=np.uint32)
        rows[:, 0] = eob
        stats = (Stats * max(count, 1))()
        rc = self._lib.bwtc_cuda_inverse_blocks(self._h, a_in, a_out, a_sz.ctypes.data, count, 1 if on_device else 0,
                                                rows.ctypes.data, ctypes.addressof(stats))
        if rc == ECORRUPT:
            raise BwtcCudaError(rc, self._lib.bwtc_cuda_last_error(self._h).decode(),
                                [k for k in range(count) if stats[k].flags & FLAG_CORRUPT])
        self._check(rc)

    def bwt_blocks(self, blocks, starts: int, want_freqs: bool = True, on_device: bool = False):
        """bwtc_cuda_bwt_blocks: transform the given blocks (uint8 arrays, or CUDA tensors / (pointer, size) pairs when
        on_device) IN PLACE (equal-sized runs are batched into one device-side sort).  Returns (LFpowers[count, 256],
        nLF[count], freqs[count, 256] or None)."""
        count = len(blocks)
        ptrs, sizes = zip(*[_block_ptr(b, on_device) for b in blocks]) if count else ((), ())
        a_ptrs = (ctypes.c_void_p * count)(*ptrs)
        a_sz = np.asarray(sizes, dtype=np.uint32)
        LF = np.zeros((count, 256), dtype=np.uint32)
        nLF = np.zeros(count, dtype=np.uint32)
        fr = np.zeros((count, 256), dtype=np.uint32) if want_freqs else None
        self._check(self._lib.bwtc_cuda_bwt_blocks(self._h, a_ptrs, a_sz.ctypes.data, count, starts, 1 if on_device else 0,
                                                   LF.ctypes.data, nLF.ctypes.data, _ptr(fr)))
        return LF, nLF, fr

    def bwt_block_device(self, d_in: int, d_out: int, n: int, LFpowers: np.ndarray,
                         freqs: Optional[np.ndarray]) -> int:
        return self._check(self._lib.bwtc_cuda_bwt_block_device(self._h, d_in, d_out, n, LFpowers.ctypes.data,
                                                                 LFpowers.size, _ptr(freqs)))


def _block_ptr(b, on_device: bool):
    """(address, bytes) of a block argument: a uint8 numpy array (host), a CUDA tensor, or a (pointer, size) pair."""
    if isinstance(b, tuple):
        return int(b[0]), int(b[1])
    if on_device:
        return int(b.data_ptr()), int(b.numel() * b.element_size())
    assert isinstance(b, np.ndarray) and b.dtype == np.uint8
    return b.ctypes.data, b.size


class BWTBlock:
    """Mirror of bwtc::BWTBlock (BWTBlock.hpp:39-72): a view (begin, size) into a caller-owned byte buffer
    plus the LFpowers vector and the transformed flag."""

    def __init__(self, data: np.ndarray, length: Optional[int] = None, is_transformed: bool = False):
        assert data.dtype == np.uint8 and data.ndim == 1
        self._data = data
        self._length = data.size if length is None else int(length)
        self._LFpowers = np.zeros(1, dtype=np.uint32)
        self._transformed = bool(is_transformed)

    def size(self) -> int:
        return self._length

    def begin(self) -> np.ndarray:
        return self._data[: self._length]

    def LFpowers(self) -> np.ndarray:
        return self._LFpowers

    def isTransformed(self) -> bool:
        return self._transformed

    def setTransformed(self, t: bool):
        assert self._transformed != t
        self._transformed = t

    def prepareLFpowers(self, startingPoints: int):  # BWTBlock.cpp:104-108
        if self._length <= 256 or startingPoints == 0:
            k = 1
        elif startingPoints <= 256:
            k = startingPoints
        else:
            k = 256
        self._LFpowers = np.zeros(k, dtype=np.uint32)


class CudaBWTransform:
    """The new BWTransform subclass (mirror of bwtc_b200/host/CudaBWTransform.hpp).  Same two contract
    levels as the reference (bwtransforms/BWTransform.hpp:53-61)."""

    def __init__(self, max_block_bytes: int = 1 << 20, device: int = 0):
        self._device = device
        self._ctx = CudaContext(max_block_bytes, device)

    @property
    def context(self) -> CudaContext:
        return self._ctx

    def _ensure(self, n: int):
        if n > self._ctx.max_block_bytes:
            want = max(n, 2 * self._ctx.max_block_bytes)
            self._ctx.close()  # release the old scratch first: peak device memory stays one context
            self._ctx = CudaContext(want, self._device)

    # raw virtual: doTransform(byte* begin, uint32 length, vector<uint32>& LF[, freqs])
    def doTransformRaw(self, begin: np.ndarray, LFpowers: np.ndarray, freqs: Optional[np.ndarray] = None) -> int:
        self._ensure(begin.size)
        return self._ctx.divbwtf(begin, begin, LFpowers, freqs)

    # block level: doTransform(BWTBlock&[, freqs]) — reverse/sentinel/hole-fill fused on the device
    def doTransform(self, block: BWTBlock, freqs: Optional[np.ndarray] = None) -> int:
        self._ensure(block.size())
        pidx = self._ctx.bwt_block(block.begin(), block.LFpowers(), freqs)
        block.setTransformed(True)
        return pidx

    # sizing hooks of BWTransform (return 0 in both reference engines, Divsufsorter.hpp:67-70); here real
    def maxSizeInBytes(self, block_size: int) -> int:
        """Exact device scratch of a context for blocks of this size (bwtc_cuda_scratch_bytes)."""
        return int(load_library().bwtc_cuda_scratch_bytes(block_size))

    def maxBlockSize(self, memory_budget: int) -> int:
        """Largest block whose scratch fits the budget (BWTC_CUDA_SCRATCH_BYTES_PER_SUFFIX = 40 is an upper bound from
        1 MiB on; the fixed part is below 8 MiB)."""
        b = max(0, (memory_budget - SCRATCH_FIXED_BYTES) // SCRATCH_BYTES_PER_SUFFIX - 1)
        return min(b, MAX_BLOCK)

    def suggestedBlockSize(self, memory_budget: int) -> int:
        return min(self.maxBlockSize(memory_budget), 32 << 20)


class BWTManager:
    """Mirror of bwtc::BWTManager (bwtransforms/BWTManager.hpp:40-58) with one new choice char 'c' (CUDA).
    The reference's 'd' / 's' / 'a' choices are CPU engines that this package deliberately does not carry."""

    def __init__(self, startingPoints: int = 1, max_block_bytes: int = 1 << 20, device: int = 0):
        self.m_startingPoints = 1
        self.setStartingPoints(startingPoints)
        self._transformers: List[CudaBWTransform] = []
        self._max_block = max_block_bytes
        self._device = device

    @staticmethod
    def isValidChoice(c: str) -> bool:
        return c == "c"

    def initialize(self, choice: str = "c"):
        if not self.isValidChoice(choice):
            raise ValueError("bwtc_b200 carries only the CUDA transformer (choice 'c'); there is no CPU fallback")
        self._transformers.append(CudaBWTransform(self._max_block, self._device))

    def setStartingPoints(self, startingPoints: int):  # BWTManager.cpp:60-64
        self.m_startingPoints = min(256, max(1, int(startingPoints)))

    def getStartingPoints(self) -> int:
        return self.m_startingPoints

    def doTransform(self, block: BWTBlock, freqs: Optional[np.ndarray] = None) -> int:  # BWTManager.cpp:46-58
        assert not block.isTransformed()
        block.prepareLFpowers(self.m_startingPoints)
        return self._transformers[0].doTransform(block, freqs)


class Pipeline:
    """Batched look-ahead driver over independent blocks on one GPU (bwtc_cuda_pipeline)."""

    def __init__(self, max_block_bytes: int, depth: int = 3, device: int = 0):
        self._lib = load_library()
        h = _vp()
        rc = self._lib.bwtc_cuda_pipeline_create(ctypes.byref(h), device, depth, max_block_bytes)
        if rc != 0:
            raise BwtcCudaError(rc, self._lib.bwtc_cuda_global_error().decode())
        self._h = h
        self.depth = depth

    def close(self):
        if getattr(self, "_h", None):
            self._lib.bwtc_cuda_pipeline_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_round0(self, chars: int = 0, key_bytes: int = 0):
        self._lib.bwtc_cuda_pipeline_set_round0(self._h, chars, key_bytes)

    def set_timing(self, detail: int):
        self._lib.bwtc_cuda_pipeline_set_timing(self._h, detail)

    def set_verify(self, on: bool):
        """bwtc_cuda_pipeline_set_verify: forward blocks and their LFpowers are verified on the device (see
        CudaContext.set_verify); overrides BWTC_VERIFY for every context of the pipeline."""
        rc = self._lib.bwtc_cuda_pipeline_set_verify(self._h, 1 if on else 0)
        if rc < 0:
            raise BwtcCudaError(rc, self._lib.bwtc_cuda_pipeline_error(self._h).decode())

    def run_ptrs(self, in_ptrs: Sequence[int], out_ptrs: Sequence[int], sizes: Sequence[int], starts: int,
                 on_device: bool, want_freqs: bool = True, want_stats: bool = True):
        nb = len(sizes)
        a_in = (ctypes.c_void_p * nb)(*in_ptrs)
        a_out = (ctypes.c_void_p * nb)(*out_ptrs)
        a_sz = np.asarray(sizes, dtype=np.uint32)
        LF = np.zeros((nb, 256), dtype=np.uint32)
        nLF = np.zeros(nb, dtype=np.uint32)
        freqs = np.zeros((nb, 256), dtype=np.uint32) if want_freqs else None
        stats = (Stats * nb)() if want_stats else None
        rc = self._lib.bwtc_cuda_pipeline_run(self._h, ctypes.addressof(a_in), ctypes.addressof(a_out), a_sz.ctypes.data,
                                              nb, starts, 1 if on_device else 0, LF.ctypes.data, nLF.ctypes.data,
                                              _ptr(freqs), ctypes.addressof(stats) if stats is not None else None)
        if rc < 0:
            raise BwtcCudaError(rc, self._lib.bwtc_cuda_pipeline_error(self._h).decode())
        return LF, nLF, freqs, ([s.as_dict() for s in stats] if stats is not None else None)

    def submit(self, block: np.ndarray, starts: int = 8, want_freqs: bool = True):
        """Streaming form (bwtc_cuda_pipeline_submit): queues one host block for an in-place transform and returns a
        handle; call wait(handle) to get (LFpowers, freqs).  The block must stay alive until then."""
        h = {"block": block, "LF": np.zeros(256, np.uint32), "nLF": ctypes.c_uint32(0),
             "freqs": np.zeros(256, np.uint32) if want_freqs else None, "ticket": ctypes.c_uint64(0)}
        rc = self._lib.bwtc_cuda_pipeline_submit(self._h, block.ctypes.data, block.ctypes.data, block.size, starts, 0,
                                                 h["LF"].ctypes.data, ctypes.addressof(h["nLF"]), _ptr(h["freqs"]), None,
                                                 ctypes.byref(h["ticket"]))
        if rc < 0:
            raise BwtcCudaError(rc, self._lib.bwtc_cuda_pipeline_error(self._h).decode())
        return h

    def submit_runs(self, block: np.ndarray, capacity: int, starts: int = 8, out: Optional[np.ndarray] = None):
        """Streaming transform with run statistics (bwtc_cuda_pipeline_submit_runs): queues one host block, transformed in
        place or into `out` (same size; `block` is then left as it is), and returns a handle; wait(handle) returns
        (LFpowers, freqs, runs) with runs = (symbol[], start[]) of the output's maximal runs, or None when there are more
        than `capacity`.  Such a block is never batched with others.  The buffers must stay alive until then."""
        assert block.dtype == np.uint8
        dst = block if out is None else out
        assert dst.dtype == np.uint8 and dst.size == block.size
        sym = np.zeros(max(capacity, 1), np.uint8)
        start = np.zeros(max(capacity, 1), np.uint32)
        h = {"kind": "runs", "block": block, "out": dst, "LF": np.zeros(256, np.uint32), "nLF": ctypes.c_uint32(0),
             "freqs": np.zeros(256, np.uint32), "sym": sym, "start": start,
             "runs": Runs(capacity, 0, sym.ctypes.data, start.ctypes.data), "ticket": ctypes.c_uint64(0)}
        rc = self._lib.bwtc_cuda_pipeline_submit_runs(self._h, block.ctypes.data, dst.ctypes.data, block.size, starts,
                                                      h["LF"].ctypes.data, ctypes.addressof(h["nLF"]), h["freqs"].ctypes.data,
                                                      ctypes.addressof(h["runs"]), ctypes.byref(h["ticket"]))
        if rc < 0:
            raise BwtcCudaError(rc, self._lib.bwtc_cuda_pipeline_error(self._h).decode())
        return h

    def submit_inverse(self, block: np.ndarray, LF):
        """Streaming inverse (bwtc_cuda_pipeline_submit_inverse): queues one host block (the output of a forward block
        transform) to be restored in place and returns a handle; wait(handle) returns the block.  LF: the block's
        LFpowers (only LF[0] is used) or its end-of-block row.  The block must stay alive until then."""
        assert block.dtype == np.uint8
        eob = int(np.asarray(LF, dtype=np.uint32).reshape(-1)[0])
        h = {"kind": "inverse", "block": block, "ticket": ctypes.c_uint64(0)}
        rc = self._lib.bwtc_cuda_pipeline_submit_inverse(self._h, block.ctypes.data, block.ctypes.data, block.size, eob, 0,
                                                         None, ctypes.byref(h["ticket"]))
        if rc < 0:
            raise BwtcCudaError(rc, self._lib.bwtc_cuda_pipeline_error(self._h).decode())
        return h

    def wait(self, h):
        """Waits for a handle of submit (returns (LFpowers, freqs)), of submit_runs (returns (LFpowers, freqs, runs or None))
        or of submit_inverse (returns the restored block).  Raises for a failed handle only: a corrupt inverse block (code
        ECORRUPT) does not fail the other blocks of its group."""
        rc = self._lib.bwtc_cuda_pipeline_wait(self._h, h["ticket"])
        if rc < 0:
            raise BwtcCudaError(rc, self._lib.bwtc_cuda_pipeline_error(self._h).decode())
        if h.get("kind") == "inverse":
            return h["block"]
        if h.get("kind") == "runs":
            cnt = h["runs"].count
            runs = None if cnt == RUNS_OVERFLOW else (h["sym"][:cnt].copy(), h["start"][:cnt].copy())
            return h["LF"][: h["nLF"].value].copy(), h["freqs"], runs
        return h["LF"][: h["nLF"].value].copy(), h["freqs"]

    def run(self, blocks: Sequence[np.ndarray], starts: int = 8):
        """Transforms host blocks in place."""
        ptrs = [b.ctypes.data for b in blocks]
        return self.run_ptrs(ptrs, ptrs, [b.size for b in blocks], starts, on_device=False)

    def run_inverse(self, blocks: Sequence[np.ndarray], LF) -> None:
        """Restores host blocks in place: submit_inverse for all, then wait for all (LF[k][0] = block k's end-of-block
        row).  Raises the first error after every block has been waited for."""
        LF = np.asarray(LF, dtype=np.uint32).reshape(len(blocks), -1)
        handles, first = [], None
        for k, b in enumerate(blocks):
            try:
                handles.append(self.submit_inverse(b, LF[k]))
            except BwtcCudaError as e:  # (the blocks already queued are still waited for)
                first = e
                break
        for h in handles:
            try:
                self.wait(h)
            except BwtcCudaError as e:
                first = first or e
        if first is not None:
            raise first

    def timing_begin(self):
        rc = self._lib.bwtc_cuda_pipeline_timing_begin(self._h)
        if rc < 0:
            raise BwtcCudaError(rc, "timing_begin failed")

    def timing_end(self) -> float:
        ms = float(self._lib.bwtc_cuda_pipeline_timing_end(self._h))
        if ms < 0:
            raise BwtcCudaError(int(ms), "timing_end failed")
        return ms


# ---- synthetic workload generators (bwtc_b200/tools/gen_inputs.c) --------------------------------------
_gen = None


def _gen_lib() -> ctypes.CDLL:
    global _gen
    if _gen is None:
        if not os.path.exists(GEN_LIB_PATH):
            raise RuntimeError(f"{GEN_LIB_PATH} not found - run __graft_entry__.build()")
        g = ctypes.CDLL(GEN_LIB_PATH)
        g.bwtc_gen_random.argtypes = [_vp, ctypes.c_uint64, ctypes.c_uint64]
        g.bwtc_gen_dna.argtypes = [_vp, ctypes.c_uint64, ctypes.c_uint64]
        g.bwtc_gen_repetitive.argtypes = [_vp, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_double]
        g.bwtc_gen_markov2.argtypes = [_vp, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint32,
                                       ctypes.c_uint32, ctypes.c_double]
        for f in (g.bwtc_gen_random, g.bwtc_gen_dna, g.bwtc_gen_repetitive, g.bwtc_gen_markov2):
            f.restype = None
        _gen = g
    return _gen


def generate(kind: str, n: int, seed: int = 1, out: Optional[np.ndarray] = None) -> np.ndarray:
    """The four synthetic input families of BASELINE.json (SURVEY.md §8d), fixed seeds.
    kind: 'markov' | 'dna' | 'repetitive' | 'random'."""
    buf = np.empty(n, dtype=np.uint8) if out is None else out
    assert buf.dtype == np.uint8 and buf.size >= n
    g = _gen_lib()
    if kind == "markov":
        g.bwtc_gen_markov2(buf.ctypes.data, n, 7, seed, 64, 32, 0.05)
    elif kind == "dna":
        g.bwtc_gen_dna(buf.ctypes.data, n, seed)
    elif kind == "repetitive":
        g.bwtc_gen_repetitive(buf.ctypes.data, n, seed, 4096, 0.001)
    elif kind == "random":
        g.bwtc_gen_random(buf.ctypes.data, n, seed)
    else:
        raise ValueError(kind)
    return buf[:n]
