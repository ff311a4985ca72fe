"""GPU parity of the INVERSE transform (SURVEY.md §8f row f4; bwtc_cuda_inverse_block / _raw, kernels in
bwtc_b200/csrc/ibwt_kernels.cuh): bit-exact against the oracle's restatement, on the outputs of the oracle's forward
transform — the inverse must not merely undo this repo's forward path — and at BASELINE block sizes.  The reference's
own inverse (MtlSaInverseBWT) pins the oracle's in tests/test_oracle.py where the reference is built."""
import numpy as np
import pytest

import bwtc_b200 as bw

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = bw.CudaContext(4 << 20)
    yield c
    c.close()


def _gpu_inverse(ctx, bwt, LF):
    buf = np.concatenate([bwt, np.array([0x77], np.uint8)])
    view = buf[:-1]
    rc = ctx.inverse_block(view, np.ascontiguousarray(LF, dtype=np.uint32))
    assert rc == bwt.size and buf[-1] == 0x77, "byte after the block must be preserved"
    return view.copy()


def test_inverse_of_oracle_forward_small_and_structured(ctx, oracle):
    rng = np.random.default_rng(61)
    cases = []
    for n in (1, 2, 3, 7, 127, 128, 129, 255, 256, 257, 1000, 4095, 4096, 4097, 65537, 300000):
        for sigma in (1, 2, 4, 64, 256):
            cases.append(rng.integers(0, sigma, n).astype(np.uint8))
    cases += [np.zeros(5000, np.uint8), np.full(70000, 0xFF, np.uint8), np.frombuffer(b"ab" * 30000, np.uint8).copy(),
              np.frombuffer(b"abc" * 20000 + b"z", np.uint8).copy(), (255 - (np.arange(100000) % 256)).astype(np.uint8),
              np.tile(rng.integers(0, 256, 777).astype(np.uint8), 200)]
    for x in cases:
        for starts in (1, 8):
            b, LF, fr = oracle.block(x, starts)
            back = _gpu_inverse(ctx, b, LF)
            assert np.array_equal(back, x), (x.size, starts)
            assert np.array_equal(oracle.inverse_block(b, LF[0]), x)


@pytest.mark.parametrize("kind", ["markov", "dna", "repetitive", "random"])
def test_inverse_of_reference_forward_matches_reference_inverse(ctx, oracle, kind):
    """The forward output of the oracle (the restatement of the reference's forward transform): the GPU's inverse equals
    the oracle's inverse (the restatement of the reference's) and restores x."""
    x = bw.generate(kind, (1 << 20) + 13, seed=71)
    b, LF, fr = oracle.block(x, 8)
    back = _gpu_inverse(ctx, b, LF)
    assert np.array_equal(back, oracle.inverse_block(b, LF[0]))
    assert np.array_equal(back, x)


def test_inverse_raw_contract(ctx, oracle):
    """doTransform(byte* bwt, uint32 N, LFpow) (InverseBWT.hpp:49-50): N rows with the end-of-block row ignored."""
    rng = np.random.default_rng(62)
    for n in (1, 2, 500, 100000):
        x = rng.integers(0, 5, n).astype(np.uint8)
        b, LF, fr = oracle.block(x, 1)
        moved = b[LF[0]] if LF[0] < n else 0  # (eob == N-1: the last row IS the end-of-block row, nothing was moved)
        raw = np.concatenate([b, np.array([moved], np.uint8)])  # re-open the hole as InverseBWT.cpp:49 does
        raw[LF[0]] = 0xEE                                           # the end-of-block row: any value
        rc = ctx.inverse_raw(raw, LF)
        assert rc == n and np.array_equal(raw[:n], x), n


def test_forward_then_inverse_on_the_device_in_place():
    import torch

    n = 3 << 20
    x = bw.generate("markov", n, seed=72)
    ctx = bw.CudaContext(n)
    try:
        d = torch.from_numpy(x.copy()).cuda()
        LF = np.zeros(8, np.uint32)
        ctx.bwt_block_device(d.data_ptr(), d.data_ptr(), n, LF, None)
        ctx.inverse_block_device(d.data_ptr(), d.data_ptr(), n, int(LF[0]))
        torch.cuda.synchronize()
        assert np.array_equal(d.cpu().numpy(), x)
    finally:
        ctx.close()


@pytest.mark.parametrize("kind,mib", [("markov", 32), ("dna", 64), ("repetitive", 16), ("random", 128)])
def test_inverse_full_size_blocks(oracle_record, kind, mib):
    """BASELINE block sizes: GPU forward (bit-exact to the reference, tests/test_gpu_fullsize.py) then GPU inverse restores
    the block; up to 32 MiB the forward output that was inverted is also checked against the oracle's recorded one."""
    n = mib << 20
    x = bw.generate(kind, n, seed=73)
    ctx = bw.CudaContext(n)
    try:
        b = x.copy()
        LF = np.zeros(8, np.uint32)
        ctx.bwt_block(b, LF, None)
        fwd = b.copy()
        ctx.inverse_block(b, LF)
        st = ctx.stats()
    finally:
        ctx.close()
    assert np.array_equal(b, x), kind
    if mib <= 32:
        oracle_record.check(x, 8, fwd, LF)
    print(f"inverse {kind} {mib} MiB: gpu_ms={st['gpu_ms']:.3f} = {n / 1e6 / (st['gpu_ms'] / 1e3):.0f} MB/s, {st['kernel_launches']} launches")


def test_inverse_rejects_bad_arguments(ctx):
    with pytest.raises(bw.BwtcCudaError):
        ctx.inverse_block(np.zeros(10, np.uint8), np.array([11], np.uint32))  # end-of-block position outside [0, N)
    with pytest.raises(bw.BwtcCudaError):
        ctx.inverse_block(np.zeros((4 << 20) + 1, np.uint8), np.array([0], np.uint32))  # above the context capacity
