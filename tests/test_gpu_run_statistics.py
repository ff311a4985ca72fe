"""GPU tests of the run statistics gathered with the BWT (SURVEY.md §8f row f3): bwtc_cuda_bwt_block_runs must return
exactly the maximal runs of the transformed block (what utils::calculateRunFrequenciesAndStoreRuns, Utils.cpp:150-170,
finds by scanning), report overflow instead of truncating, and the pipelined compressor that feeds them to the reference's
HuffmanEncoder must still write byte-identical .bwtc files."""
import json

import numpy as np
import pytest

import bwtc_b200 as bw
from test_pipelined_compressor import REFTOOL, need_libs, run_tool

pytestmark = pytest.mark.gpu


def _runs_of(b):
    heads = np.flatnonzero(np.concatenate([[True], b[1:] != b[:-1]]))
    return b[heads], heads.astype(np.uint32)


@pytest.mark.parametrize("kind,n", [("repetitive", 1 << 20), ("repetitive", (9 << 20) + 5), ("markov", 300001), ("dna", 1 << 18),
                                    ("random", 70000), ("zeros", 100000), ("tiny", 1), ("tiny", 2), ("tiny", 4097)])
def test_runs_equal_a_scan_of_the_output(oracle, kind, n):
    if kind == "zeros":
        x = np.zeros(n, np.uint8)
    elif kind == "tiny":
        x = (np.arange(n) % 3).astype(np.uint8)
    else:
        x = bw.generate(kind, n, seed=81)
    ctx = bw.CudaContext(n)
    try:
        blk = x.copy()
        LF = np.zeros(bw.num_starting_points(n, 8), np.uint32)
        fr = np.zeros(256, np.uint32)
        pidx, runs = ctx.bwt_block_runs(blk, LF, fr, capacity=n)
        assert runs is not None
        if n <= (2 << 20):
            w = oracle.block(x, 8)
            assert np.array_equal(blk, w[0]) and (LF == w[1]).all() and (fr == w[2]).all()
        sym, start = _runs_of(blk)
        assert runs[0].size == sym.size and np.array_equal(runs[0], sym) and np.array_equal(runs[1], start), (kind, n)
        # a capacity below the run count: overflow is reported, nothing is truncated silently
        if sym.size > 1:
            blk2 = x.copy()
            pidx2, runs2 = ctx.bwt_block_runs(blk2, LF, None, capacity=sym.size - 1)
            assert runs2 is None and np.array_equal(blk2, blk)
            blk3 = x.copy()
            pidx3, runs3 = ctx.bwt_block_runs(blk3, LF, None, capacity=sym.size)
            assert runs3 is not None and runs3[0].size == sym.size
    finally:
        ctx.close()


@pytest.mark.parametrize("kind", ["repetitive", "markov"])
def test_pipelined_compress_with_gpu_run_statistics_is_byte_identical(tmp_path, kind):
    """16 MiB blocks (run statistics apply to blocks above 8 MiB): the repetitive input has few runs (the GPU's runs are
    used, the coder never scans), the Markov input overflows the capacity (the coder scans as before).  Same bytes."""
    need_libs()
    x = bw.generate(kind, (40 << 20) + 321, seed=82)
    src = tmp_path / "in.bin"
    x.tofile(src)
    mem = 90687655  # 16 MiB blocks
    run_tool("compress", "cpu", src, tmp_path / "ref.bwtc", mem, "H", 8, tool=REFTOOL)
    out = json.loads(run_tool("pipe_compress", src, tmp_path / "pipe.bwtc", mem, "H", "c", 8, 4, 0, "0", 3))
    assert (tmp_path / "ref.bwtc").read_bytes() == (tmp_path / "pipe.bwtc").read_bytes()
    served = out.get("run_statistics_served", 0)
    if kind == "repetitive":
        assert served > 0, "the GPU's runs should have replaced the coder's scans"
    else:
        assert served == 0


def test_pipelined_compress_mixed_blocks_with_and_without_run_statistics(tmp_path, monkeypatch):
    """One file, three kinds of block (16 MiB blocks): repetitive (few runs: the GPU's runs are served to the coder),
    Markov (over the size/8 capacity: the coder scans), and a last block below 8 MiB (no runs asked for).  Byte-identical
    to the reference, and again with BWTC_RUN_STATS=0."""
    need_libs()
    x = np.concatenate([bw.generate("repetitive", 16 << 20, seed=83), bw.generate("markov", 16 << 20, seed=84),
                        bw.generate("random", (3 << 20) + 77, seed=85)])
    src = tmp_path / "in.bin"
    x.tofile(src)
    mem = 90687655  # 16 MiB blocks
    run_tool("compress", "cpu", src, tmp_path / "ref.bwtc", mem, "H", 8, tool=REFTOOL)
    ref = (tmp_path / "ref.bwtc").read_bytes()
    out = json.loads(run_tool("pipe_compress", src, tmp_path / "pipe.bwtc", mem, "H", "c", 8, 4, 0, "0", 2))
    assert (tmp_path / "pipe.bwtc").read_bytes() == ref
    assert out.get("run_statistics_served", 0) > 0, "the repetitive block's runs should have been served"
    monkeypatch.setenv("BWTC_RUN_STATS", "0")
    out = json.loads(run_tool("pipe_compress", src, tmp_path / "off.bwtc", mem, "H", "c", 8, 4, 0, "0", 2))
    assert (tmp_path / "off.bwtc").read_bytes() == ref
    assert out.get("run_statistics_served", 0) == 0
