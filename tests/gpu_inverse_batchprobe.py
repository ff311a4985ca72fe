#!/usr/bin/env python
"""Batched vs one-by-one inverse transform (not a pytest).  Prints the card and its power limit, then for each shape the
device time (stats gpu_ms, summed over the calls) and the host wall time including copies of
  - CudaContext.inverse_blocks (equal-sized runs inverted as one problem) against a loop of inverse_block, same context;
  - Pipeline.run_inverse over 256 pinned 1 MiB blocks (depth 3, device time by timing_begin/end) against a loop of
    inverse_block on one context;
  - the single 32 MiB Markov inverse against a library built from an earlier commit (--parent-lib), alternated;
and a torch.profiler per-kernel summary of the 64 x 256 KiB shape both ways.
  python tests/gpu_inverse_batchprobe.py [--reps 5] [--parent-lib path/to/libbwtc_cuda.so]"""
import argparse
import ctypes
import os
import statistics
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bwtc_b200 as bw  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--parent-lib", default=None)
args = ap.parse_args()


def spread(v):
    return f"median {statistics.median(v):8.3f}  min {min(v):8.3f}  max {max(v):8.3f}"


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "nvidia-smi unavailable"


print(f"card: {card()}  (name, power limit, max SM clock)", flush=True)


def forward(ctx, xs):
    blocks = [x.copy() for x in xs]
    LF, nLF, _ = ctx.bwt_blocks(blocks, 8, want_freqs=False)
    return blocks, LF


def time_batch(ctx, bwts, LF, work):
    for w, b in zip(work, bwts):
        w[:] = b
    t0 = time.perf_counter()
    ctx.inverse_blocks(work, LF)
    wall = (time.perf_counter() - t0) * 1e3
    st = ctx.stats()
    return st["gpu_ms"], wall, st


def time_single(ctx, bwts, LF, work):
    for w, b in zip(work, bwts):
        w[:] = b
    gpu = 0.0
    t0 = time.perf_counter()
    for k, w in enumerate(work):
        ctx.inverse_block(w, LF[k, :1])
        gpu += ctx.stats()["gpu_ms"]
    return gpu, (time.perf_counter() - t0) * 1e3


def probe_context(kind, count, kib):
    n = kib << 10
    xs = [bw.generate(kind, n, seed=2000 + k) for k in range(count)]
    ctx = bw.CudaContext(count * (n + 1))
    try:
        bwts, LF = forward(ctx, xs)
        work = [np.empty(n, np.uint8) for _ in range(count)]
        time_batch(ctx, bwts, LF, work)  # warm-up of both paths
        assert all(np.array_equal(w, x) for w, x in zip(work, xs)), "batch result differs"
        time_single(ctx, bwts, LF, work)
        assert all(np.array_equal(w, x) for w, x in zip(work, xs)), "single result differs"
        bg, bw_, sg, sw = [], [], [], []
        for _ in range(args.reps):  # alternated
            g, w, st = time_batch(ctx, bwts, LF, work)
            bg.append(g); bw_.append(w)
            g, w = time_single(ctx, bwts, LF, work)
            sg.append(g); sw.append(w)
        assert all(np.array_equal(w, x) for w, x in zip(work, xs))
    finally:
        ctx.close()
    mb = count * n / 1e6
    print(f"{kind:7s} {count:3d} x {kib:5d} KiB  batch  gpu_ms {spread(bg)} | wall_ms {spread(bw_)}  "
          f"({st['kernel_launches']} launches, {mb / statistics.median(bw_) * 1e3:.0f} MB/s wall)", flush=True)
    print(f"{'':26s} single gpu_ms {spread(sg)} | wall_ms {spread(sw)}  ({mb / statistics.median(sw) * 1e3:.0f} MB/s wall)",
          flush=True)
    print(f"{'':26s} speed-up: device {statistics.median(sg) / statistics.median(bg):.2f}x, wall "
          f"{statistics.median(sw) / statistics.median(bw_):.2f}x", flush=True)


def probe_pipeline(count=256, kib=1024, depth=3):
    import torch

    n = kib << 10
    xs = [bw.generate("markov", n, seed=3000 + k) for k in range(count)]
    pinned = [torch.from_numpy(x.copy()).pin_memory() for x in xs]
    blocks = [t.numpy() for t in pinned]
    p = bw.Pipeline(n, depth=depth)
    ctx = bw.CudaContext(n)
    try:
        LF, nLF, _, _ = p.run(blocks, 8)
        bwts = [b.copy() for b in blocks]
        pg, pw, sw = [], [], []
        for rep in range(args.reps + 1):
            for b, s in zip(blocks, bwts):
                b[:] = s
            p.timing_begin()
            t0 = time.perf_counter()
            p.run_inverse(blocks, LF)
            w = (time.perf_counter() - t0) * 1e3
            g = p.timing_end()
            assert all(np.array_equal(b, x) for b, x in zip(blocks, xs)), "pipeline result differs"
            for b, s in zip(blocks, bwts):
                b[:] = s
            t0 = time.perf_counter()
            for k, b in enumerate(blocks):
                ctx.inverse_block(b, LF[k, :1])
            s_w = (time.perf_counter() - t0) * 1e3
            assert all(np.array_equal(b, x) for b, x in zip(blocks, xs)), "single result differs"
            if rep:  # rep 0 is the warm-up
                pg.append(g); pw.append(w); sw.append(s_w)
    finally:
        p.close()
        ctx.close()
    mb = count * n / 1e6
    print(f"pipeline {count} x {kib} KiB pinned, depth {depth}: run_inverse device_ms {spread(pg)} | wall_ms {spread(pw)}  "
          f"({mb / statistics.median(pw) * 1e3:.0f} MB/s wall)", flush=True)
    print(f"{'':26s} inverse_block loop wall_ms {spread(sw)}  ({mb / statistics.median(sw) * 1e3:.0f} MB/s wall); "
          f"speed-up {statistics.median(sw) / statistics.median(pw):.2f}x", flush=True)


def parent_context(n, path):
    """A context on a library from an earlier commit: bind only the symbols it exports."""
    saved = bw.C_ABI
    lib = ctypes.CDLL(path)
    bw.C_ABI = [e for e in saved if hasattr(lib, e[0])]
    try:
        return bw.CudaContext(n, lib_path=path)
    finally:
        bw.C_ABI = saved


def probe_single_vs_parent(path, mib=32):
    n = mib << 20
    x = bw.generate("markov", n, seed=73)
    cur = bw.CudaContext(n)
    par = parent_context(n, path)
    try:
        b = x.copy()
        LF = np.zeros(8, np.uint32)
        cur.bwt_block(b, LF, None)
        fwd = b.copy()
        res = {"this": [], "parent": []}
        for rep in range(2 * args.reps + 1):
            for name, c in (("this", cur), ("parent", par)) if rep % 2 == 0 else (("parent", par), ("this", cur)):
                b[:] = fwd
                c.inverse_block(b, LF)
                assert np.array_equal(b, x), name
                if rep:
                    res[name].append(c.stats()["gpu_ms"])
    finally:
        cur.close()
        par.close()
    for name in ("this", "parent"):
        print(f"single {mib} MiB markov inverse, {name:6s} library: gpu_ms {spread(res[name])}", flush=True)
    print(f"{'':26s} this / parent (medians): {statistics.median(res['this']) / statistics.median(res['parent']):.4f}",
          flush=True)


def profile_kernels(count=64, kib=256):
    import torch
    from torch.profiler import ProfilerActivity, profile

    n = kib << 10
    xs = [bw.generate("markov", n, seed=2000 + k) for k in range(count)]
    ctx = bw.CudaContext(count * (n + 1))
    try:
        bwts, LF = forward(ctx, xs)
        work = [np.empty(n, np.uint8) for _ in range(count)]
        time_batch(ctx, bwts, LF, work)
        time_single(ctx, bwts, LF, work)
        for name, fn in (("batch", time_batch), ("single", time_single)):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                fn(ctx, bwts, LF, work)
                torch.cuda.synchronize()
            print(f"--- per-kernel device time, {count} x {kib} KiB markov, {name}")
            print(prof.key_averages().table(sort_by="cuda_time_total", row_limit=12), flush=True)
    finally:
        ctx.close()


for kind, count, kib in (("markov", 64, 256), ("markov", 32, 1024), ("markov", 16, 1024), ("random", 32, 1024)):
    probe_context(kind, count, kib)
probe_pipeline()
if args.parent_lib:
    probe_single_vs_parent(args.parent_lib)
profile_kernels()
