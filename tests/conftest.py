"""Shared fixtures.  GPU tests are marked @pytest.mark.gpu; everything else runs on CPU.

Only tests/ (plus __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs) may load
oracle/liboracle.so or oracle/_ref/libbwtc_ref.so — they are checkers, never the product path.
"""
import ctypes
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def _ensure_built():
    need = [os.path.join(ROOT, "oracle", "liboracle.so"), os.path.join(ROOT, "bwtc_b200", "libbwtc_gen.so"),
            os.path.join(ROOT, "bwtc_b200", "libbwtc_cuda.so")]
    if not all(os.path.exists(p) for p in need):
        subprocess.run([sys.executable, "-c", "import __graft_entry__ as g; g.build()"], cwd=ROOT, check=True)


_ensure_built()


class Oracle:
    """ctypes view of oracle/liboracle.so (the C restatement)."""

    def __init__(self):
        self.lib = ctypes.CDLL(os.path.join(ROOT, "oracle", "liboracle.so"))
        self.lib.oracle_bwt_block.restype = ctypes.c_int64
        self.lib.oracle_bwt_block.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_void_p,
                                              ctypes.c_void_p, ctypes.c_void_p]
        self.lib.oracle_bwt_raw.restype = ctypes.c_int64
        self.lib.oracle_bwt_raw.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint32, ctypes.c_void_p,
                                            ctypes.c_uint32, ctypes.c_void_p]
        self.lib.oracle_suffix_array.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_void_p, ctypes.c_void_p]
        self.lib.oracle_inverse_block.restype = ctypes.c_int64
        self.lib.oracle_inverse_block.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint32]
        self.lib.oracle_inverse_raw.restype = ctypes.c_int64
        self.lib.oracle_inverse_raw.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint32]
        self.lib.oracle_num_starting_points.restype = ctypes.c_uint32
        self.lib.oracle_num_starting_points.argtypes = [ctypes.c_uint32, ctypes.c_uint32]

    def block(self, x, starts, guard=0xAB):
        buf = np.concatenate([x, np.array([guard], np.uint8)])
        LF = np.zeros(256, np.uint32)
        n = ctypes.c_uint32(0)
        fr = np.zeros(256, np.uint32)
        pidx = self.lib.oracle_bwt_block(buf.ctypes.data, x.size, starts, LF.ctypes.data, ctypes.byref(n), fr.ctypes.data)
        assert buf[-1] == guard
        assert pidx >= 0
        return buf[:-1].copy(), LF[: n.value].copy(), fr

    def raw(self, T, nLF, want_freqs=True):
        buf = T.copy()
        LF = np.zeros(max(nLF, 1), np.uint32)
        fr = np.zeros(256, np.uint32)
        rc = self.lib.oracle_bwt_raw(buf.ctypes.data, buf.ctypes.data, T.size, LF.ctypes.data, nLF,
                                     fr.ctypes.data if want_freqs else None)
        return rc, buf, LF, fr

    def inverse_block(self, bwt, eob, guard=0xAB):
        buf = np.concatenate([bwt, np.array([guard], np.uint8)])
        rc = self.lib.oracle_inverse_block(buf.ctypes.data, bwt.size, int(eob))
        assert buf[-1] == guard and rc == bwt.size, rc
        return buf[:-1].copy()

    def suffix_array(self, T):
        SA = np.zeros(T.size, np.uint32)
        ISA = np.zeros(T.size, np.uint32)
        self.lib.oracle_suffix_array(T.ctypes.data, T.size, SA.ctypes.data, ISA.ctypes.data)
        return SA, ISA


class Reference:
    """ctypes view of oracle/_ref/libbwtc_ref.so (the unmodified reference, compiled by oracle/Makefile)."""

    def __init__(self, path):
        self.lib = ctypes.CDLL(path)
        self.lib.ref_compress.restype = ctypes.c_longlong
        self.lib.ref_uncompress.restype = ctypes.c_longlong

    def block(self, x, starts, algo=b"d", guard=0xAB, want_freqs=True):
        buf = np.concatenate([x, np.array([guard], np.uint8)])
        LF = np.zeros(256, np.uint32)
        n = ctypes.c_uint32(0)
        fr = np.zeros(256, np.uint32)
        self.lib.ref_bwt_block(ctypes.c_void_p(buf.ctypes.data), ctypes.c_uint(x.size), ctypes.c_uint(starts),
                               ctypes.c_char(algo), ctypes.c_void_p(LF.ctypes.data), ctypes.byref(n),
                               ctypes.c_void_p(fr.ctypes.data) if want_freqs else None)
        assert buf[-1] == guard
        return buf[:-1].copy(), LF[: n.value].copy(), fr

    def raw(self, T, nLF, algo=b"d", want_freqs=True):
        buf = T.copy()
        LF = np.zeros(max(nLF, 1), np.uint32)
        fr = np.zeros(256, np.uint32)
        self.lib.ref_bwt_raw(ctypes.c_void_p(buf.ctypes.data), ctypes.c_uint(T.size), ctypes.c_uint(nLF),
                             ctypes.c_char(algo), ctypes.c_void_p(LF.ctypes.data),
                             ctypes.c_void_p(fr.ctypes.data) if want_freqs else None)
        return buf, LF, fr

    def inverse_block(self, bwt, LF):
        buf = np.concatenate([bwt, np.zeros(1, np.uint8)])
        lf = np.ascontiguousarray(LF, dtype=np.uint32)
        self.lib.ref_inverse_block(ctypes.c_void_p(buf.ctypes.data), ctypes.c_uint(bwt.size),
                                   ctypes.c_void_p(lf.ctypes.data), ctypes.c_uint(lf.size))
        return buf[:-1].copy()

    def compress(self, src, dst, mem_limit, coder=b"H", algo=b"d", starts=8):
        return int(self.lib.ref_compress(src.encode(), dst.encode(), ctypes.c_ulonglong(mem_limit),
                                         ctypes.c_char(coder), ctypes.c_char(algo), ctypes.c_uint(starts)))

    def uncompress(self, src, dst):
        return int(self.lib.ref_uncompress(src.encode(), dst.encode()))


def digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


class OracleRecord:
    """The C oracle's forward transform of the GPU tests' full-size generated blocks, recorded in
    tests/golden/oracle_bwt_digests.json by tests/golden/make_oracle_digests.py: digests of the transformed bytes and
    freqs, and the LFpowers, keyed by the digest of the input."""

    def __init__(self):
        with open(os.path.join(ROOT, "tests", "golden", "oracle_bwt_digests.json")) as f:
            self.rec = json.load(f)

    def check(self, x, starts, out, LF, fr=None):
        key = f"{digest(x)}:{starts}"
        e = self.rec.get(key)
        assert e is not None, f"no recorded oracle output for this input ({key}): run tests/golden/make_oracle_digests.py"
        assert [int(v) for v in LF] == e["LF"], (LF, e["LF"])
        assert fr is None or digest(fr) == e["freqs"], "freqs differ from the oracle's"
        assert digest(out) == e["bwt"], "BWT bytes differ from the oracle's"


@pytest.fixture(scope="session")
def oracle():
    return Oracle()


@pytest.fixture(scope="session")
def oracle_record():
    return OracleRecord()


@pytest.fixture(scope="session")
def reference():
    p = os.path.join(ROOT, "oracle", "_ref", "libbwtc_ref.so")
    if not os.path.exists(p):
        pytest.skip("oracle/_ref/libbwtc_ref.so not built (no /root/reference here and no prebuilt copy)")
    return Reference(p)


@pytest.fixture(scope="session")
def golden():
    z = np.load(os.path.join(ROOT, "tests", "golden", "forward_bwt_golden.npz"))
    names = sorted({k.split("/")[0] for k in z.files})
    return {n: {f: z[f"{n}/{f}"] for f in ("in", "starts", "out", "LF", "freqs")} for n in names}


def has_cuda():
    try:
        import bwtc_b200 as bw

        return bw.load_library().bwtc_cuda_device_count() > 0
    except Exception:
        return False
