#!/usr/bin/env python
"""Cost of block integrity (not a pytest; profiles/r04_verify.md).  Prints the card and its power limit, then, alternated in
one process (medians with min / max over --reps):
  - the inverse with its single-cycle check against a library built from an earlier commit (--parent-lib): the single
    32 MiB Markov block, 64 x 256 KiB and 32 x 1 MiB through inverse_blocks — device time (stats gpu_ms) and wall time;
  - the forward with verification off against on (and off against the earlier library, with both launch counts): 32 MiB
    Markov, a 32 x 1 MiB batch, and 256 pinned 1 MiB blocks through the pipeline at depth 3.
  python tests/gpu_verify_probe.py --parent-lib path/to/earlier/libbwtc_cuda.so [--reps 7]"""
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
ap.add_argument("--reps", type=int, default=7)
ap.add_argument("--parent-lib", required=True)
args = ap.parse_args()


def spread(v):
    return f"median {statistics.median(v):8.3f}  min {min(v):8.3f}  max {max(v):8.3f}"


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "nvidia-smi unavailable"


def parent_context(n):
    """A context on the earlier library: bind only the symbols it exports."""
    saved = bw.C_ABI
    lib = ctypes.CDLL(args.parent_lib)
    bw.C_ABI = [e for e in saved if hasattr(lib, e[0])]
    try:
        return bw.CudaContext(n, lib_path=args.parent_lib)
    finally:
        bw.C_ABI = saved


def alternate(arms, reps):
    """arms: {name: fn() -> (gpu_ms, wall_ms)}; one warm-up round, then reps rounds in alternating order."""
    res = {k: ([], []) for k in arms}
    names = list(arms)
    for rep in range(reps + 1):
        for k in (names if rep % 2 else names[::-1]):
            g, w = arms[k]()
            if rep:
                res[k][0].append(g)
                res[k][1].append(w)
    return res


def report(title, res, base):
    for k, (g, w) in res.items():
        print(f"{title:34s} {k:12s} gpu_ms {spread(g)} | wall_ms {spread(w)}", flush=True)
    for k, (g, w) in res.items():
        if k != base:
            print(f"{'':34s} {k} / {base} (medians): device {statistics.median(g) / statistics.median(res[base][0]):.4f}, "
                  f"wall {statistics.median(w) / statistics.median(res[base][1]):.4f}", flush=True)


def inverse_arm(ctx, bwts, LF, xs):
    work = [np.empty(b.size, np.uint8) for b in bwts]

    def run():
        for w, b in zip(work, bwts):
            w[:] = b
        t0 = time.perf_counter()
        if len(work) == 1:
            ctx.inverse_block(work[0], LF[0, :1])
        else:
            ctx.inverse_blocks(work, LF)
        wall = (time.perf_counter() - t0) * 1e3
        assert all(np.array_equal(w, x) for w, x in zip(work, xs))
        return ctx.stats()["gpu_ms"], wall
    return run


def probe_inverse(count, kib):
    n = kib << 10
    xs = [bw.generate("markov", n, seed=(73 if count == 1 else 2000 + k)) for k in range(count)]
    cur, par = bw.CudaContext(count * (n + 1)), parent_context(count * (n + 1))
    try:
        bwts = [x.copy() for x in xs]
        LF, _, _ = cur.bwt_blocks(bwts, 8, want_freqs=False)
        res = alternate({"this": inverse_arm(cur, bwts, LF, xs), "parent": inverse_arm(par, bwts, LF, xs)}, args.reps)
    finally:
        cur.close()
        par.close()
    report(f"inverse {count} x {kib} KiB markov", res, "parent")


def forward_arm(ctx, xs, launches):
    work = [np.empty(x.size, np.uint8) for x in xs]
    ref = {}

    def run():
        for w, x in zip(work, xs):
            w[:] = x
        t0 = time.perf_counter()
        if len(work) == 1:
            LF = np.zeros(8, np.uint32)
            ctx.bwt_block(work[0], LF, None)
        else:
            LF, _, _ = ctx.bwt_blocks(work, 8, want_freqs=False)
        wall = (time.perf_counter() - t0) * 1e3
        st = ctx.stats()
        launches.append(st["kernel_launches"])
        if not ref:
            ref["out"] = [w.copy() for w in work]
        assert all(np.array_equal(w, r) for w, r in zip(work, ref["out"]))
        return st["gpu_ms"], wall
    return run


def probe_forward(count, kib):
    n = kib << 10
    xs = [bw.generate("markov", n, seed=(73 if count == 1 else 2000 + k)) for k in range(count)]
    cap = count * (n + 1)
    off, on, par = bw.CudaContext(cap), bw.CudaContext(cap), parent_context(cap)
    on.set_verify(True)
    la = {"verify_off": [], "verify_on": [], "parent": []}
    try:
        res = alternate({"verify_off": forward_arm(off, xs, la["verify_off"]), "verify_on": forward_arm(on, xs, la["verify_on"]),
                         "parent": forward_arm(par, xs, la["parent"])}, args.reps)
    finally:
        off.close()
        on.close()
        par.close()
    report(f"forward {count} x {kib} KiB markov", res, "verify_off")
    print(f"{'':34s} kernel launches per call: " + ", ".join(f"{k} {sorted(set(v))}" for k, v in la.items()), flush=True)
    assert set(la["verify_off"]) == set(la["parent"]), "verification off must launch what the earlier library launches"


def probe_pipeline(count=256, kib=1024, depth=3):
    import torch

    n = kib << 10
    xs = [bw.generate("markov", n, seed=3000 + k) for k in range(count)]
    pinned = [torch.from_numpy(x.copy()).pin_memory() for x in xs]
    blocks = [t.numpy() for t in pinned]
    ptrs = [b.ctypes.data for b in blocks]
    pipes = {"verify_off": bw.Pipeline(n, depth=depth), "verify_on": bw.Pipeline(n, depth=depth)}
    pipes["verify_on"].set_verify(True)
    ref = {}

    def arm(p):
        def run():
            for b, x in zip(blocks, xs):
                b[:] = x
            p.timing_begin()
            t0 = time.perf_counter()
            p.run_ptrs(ptrs, ptrs, [n] * count, 8, on_device=False, want_freqs=False, want_stats=False)
            w = (time.perf_counter() - t0) * 1e3
            g = p.timing_end()
            if not ref:
                ref["out"] = [b.copy() for b in blocks]
            assert all(np.array_equal(b, r) for b, r in zip(blocks, ref["out"]))
            return g, w
        return run
    try:
        res = alternate({k: arm(p) for k, p in pipes.items()}, args.reps)
    finally:
        for p in pipes.values():
            p.close()
    report(f"pipeline {count} x {kib} KiB pinned d{depth}", res, "verify_off")
    mb = count * n / 1e6
    for k, (g, w) in res.items():
        print(f"{'':34s} {k}: {mb / statistics.median(w) * 1e3:.0f} MB/s wall", flush=True)


print(f"card: {card()}  (name, power limit, max SM clock)", flush=True)
for count, kib in ((1, 32 << 10), (64, 256), (32, 1024)):
    probe_inverse(count, kib)
for count, kib in ((1, 32 << 10), (32, 1024)):
    probe_forward(count, kib)
probe_pipeline()
