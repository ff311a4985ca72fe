"""CPU side of block integrity (DESIGN.md §3.7 single-cycle check, §3.10 verification): the new setters refuse a null
handle with a message, the header's new codes match the binding, and a CPU classifier of "is (L, eob) the BWT of any
text?" — the reference the GPU tests (tests/test_gpu_verify.py) judge mutated blocks by — is checked on every binary text
of up to 10 bytes."""
import itertools
import os
import re

import numpy as np

import bwtc_b200 as bw
from conftest import ROOT

EARG = -1
INV_K = 32  # splitter spacing of ibwt_kernels.cuh


def psi_of(out, eob):
    """Psi of a block-contract forward output (n bytes, hole at eob filled with L[N-1]) with end-of-block row eob: the
    stable order of the keys L + 1 (0 at the sentinel row), exactly as k_inv_keys + the two digit passes build it."""
    n = out.size
    N = n + 1
    keys = np.empty(N, np.int32)
    keys[:n] = out.astype(np.int32) + 1
    if eob < n:
        keys[n] = int(out[eob]) + 1
    keys[eob] = 0
    return np.argsort(keys, kind="stable")


def cycle_labels(psi):
    """Smallest row of each row's Psi cycle (pointer jumping, log2 N rounds)."""
    lab = np.arange(psi.size)
    p = psi.copy()
    for _ in range(max(1, int(np.ceil(np.log2(psi.size)))) + 1):
        lab = np.minimum(lab, lab[p])
        p = p[p]
    return lab


def classify(out, eob, k=INV_K):
    """(valid, a_fails, b_fails) at splitter spacing k: valid = Psi is one cycle; (a) some cycle holds no splitter (the
    walk-1 lengths do not sum to N); (b) some splitter lies off the cycle through row 0 (its chain never reaches NIL)."""
    lab = cycle_labels(psi_of(np.asarray(out, np.uint8), int(eob)))
    split = np.arange(0, lab.size, k)
    has = np.zeros(lab.size, bool)
    has[lab[split]] = True
    a_fails = not bool(has[np.unique(lab)].all())
    b_fails = bool((lab[split] != 0).any())
    return bool((lab == 0).all()), a_fails, b_fails


def is_bwt(out, eob):
    return classify(out, eob)[0]


def test_setters_refuse_null_handles():
    lib = bw.load_library()
    assert lib.bwtc_cuda_ctx_set_verify(None, 1) == EARG
    assert b"null context" in lib.bwtc_cuda_global_error()
    assert lib.bwtc_cuda_pipeline_set_verify(None, 1) == EARG
    assert b"null pipeline" in lib.bwtc_cuda_global_error()


def test_header_codes_match_binding():
    src = open(os.path.join(ROOT, "include", "bwtc_cuda.h")).read()
    codes = {m.group(1): int(m.group(2)) for m in re.finditer(r"#define\s+BWTC_CUDA_(E[A-Z]+)\s+\((-?\d+)\)", src)}
    assert codes["ECORRUPT"] == bw.ECORRUPT == -6
    assert codes["EVERIFY"] == bw.EVERIFY == -7
    assert len(set(codes.values())) == len(codes), codes


def test_classifier_accepts_oracle_outputs_and_counts_a_bijection(oracle):
    for n in range(1, 11):
        valid = set()
        for bits in itertools.product((0, 1), repeat=n):
            x = np.array(bits, np.uint8)
            out, LF, _ = oracle.block(x, 1)
            assert is_bwt(out, LF[0]), (bits, out, LF[0])
            valid.add((out.tobytes(), int(LF[0])))
        assert len(valid) == 2 ** n  # distinct texts give distinct (L, eob)
        count = 0
        for bits in itertools.product((0, 1), repeat=n):
            out = np.array(bits, np.uint8)
            for eob in range(n + 1):
                v, a_fails, b_fails = classify(out, eob)
                assert v == (not a_fails and not b_fails)
                assert not b_fails  # N <= 32: row 0 is the only splitter
                if v:
                    assert (out.tobytes(), eob) in valid
                    count += 1
        assert count == 2 ** n  # the BWT is a bijection onto the valid pairs


def test_classifier_labels_both_failure_kinds():
    rng = np.random.default_rng(7)
    out = rng.integers(0, 4, 4000).astype(np.uint8)
    kinds = {classify(out, e)[1:] for e in rng.integers(0, 4001, 40)}
    assert any(a for a, _ in kinds) and any(b for _, b in kinds)
