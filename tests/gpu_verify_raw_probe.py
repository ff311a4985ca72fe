#!/usr/bin/env python
"""Cost of verifying the raw contract and every LFpowers entry (not a pytest; profiles/r05_verify_raw.md).  Prints the card
and its power limit, then, alternated in one process (medians with min / max over --reps; gpu_ms = stats.gpu_ms, CUDA
events around the call's device work):
  - a raw 32 MiB Markov text (divbwtf, pageable, last byte as generated) with verification off and on, and off on a
    library built from an earlier commit (--parent-lib);
  - the block contract with verification on, this library (which also checks LFpowers[1..]) against the earlier one:
    32 MiB Markov (bwt_block) and a 32 x 1 MiB batch (bwt_blocks);
  - the plain inverse against the earlier library: 32 MiB Markov (inverse_block) and 64 x 256 KiB (inverse_blocks).
  python tests/gpu_verify_raw_probe.py --parent-lib path/to/earlier/libbwtc_cuda.so [--reps 7]"""
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


def report(title, res, base, launches=None):
    for k, (g, w) in res.items():
        print(f"{title:34s} {k:12s} gpu_ms {spread(g)} | wall_ms {spread(w)}", flush=True)
    for k, (g, w) in res.items():
        if k != base:
            print(f"{'':34s} {k} / {base} (medians): device {statistics.median(g) / statistics.median(res[base][0]):.4f}, "
                  f"wall {statistics.median(w) / statistics.median(res[base][1]):.4f}", flush=True)
    if launches:
        print(f"{'':34s} kernel launches per call: " + ", ".join(f"{k} {sorted(set(v))}" for k, v in launches.items()),
              flush=True)


def timed(ctx, fn, launches, flags=None):
    t0 = time.perf_counter()
    fn()
    wall = (time.perf_counter() - t0) * 1e3
    st = ctx.stats()
    launches.append(st["kernel_launches"])
    if flags is not None:
        assert bool(st["flags"] & bw.FLAG_VERIFIED) == flags
    return st["gpu_ms"], wall


def probe_raw():
    T = bw.generate("markov", 32 << 20, seed=73)
    off, on, par = bw.CudaContext(T.size), bw.CudaContext(T.size), parent_context(T.size)
    on.set_verify(True)
    la = {"verify_off": [], "verify_on": [], "parent": []}
    ref = {}

    def arm(ctx, name, flag):
        U = np.empty_like(T)
        LF = np.zeros(8, np.uint32)

        def run():
            r = timed(ctx, lambda: ctx.divbwtf(T, U, LF, None), la[name], flag)
            ref.setdefault("U", U.copy())
            ref.setdefault("LF", LF.copy())
            keep = np.arange(T.size) != LF[0]
            assert np.array_equal(U[keep], ref["U"][keep]) and np.array_equal(LF, ref["LF"])
            return r
        return run
    try:
        res = alternate({"verify_off": arm(off, "verify_off", False), "verify_on": arm(on, "verify_on", True),
                         "parent": arm(par, "parent", None)}, args.reps)
    finally:
        off.close()
        on.close()
        par.close()
    report(f"raw 32 MiB markov (last byte {int(T[-1])})", res, "verify_off", la)
    assert set(la["verify_off"]) == set(la["parent"]), "verification off must launch what the earlier library launches"


def probe_block_verify(count, kib):
    n = kib << 10
    xs = [bw.generate("markov", n, seed=(73 if count == 1 else 2000 + k)) for k in range(count)]
    cap = count * (n + 1)
    cur, par = bw.CudaContext(cap), parent_context(cap)
    cur.set_verify(True)
    par._check(par._lib.bwtc_cuda_ctx_set_verify(par._h, 1))
    la = {"this": [], "parent": []}
    ref = {}

    def arm(ctx, name):
        work = [np.empty(x.size, np.uint8) for x in xs]

        def run():
            for w, x in zip(work, xs):
                w[:] = x
            if count == 1:
                r = timed(ctx, lambda: ctx.bwt_block(work[0], np.zeros(8, np.uint32), None), la[name], True)
            else:
                r = timed(ctx, lambda: ctx.bwt_blocks(work, 8, want_freqs=False), la[name], True)
            ref.setdefault("out", [w.copy() for w in work])
            assert all(np.array_equal(w, o) for w, o in zip(work, ref["out"]))
            return r
        return run
    try:
        res = alternate({"this": arm(cur, "this"), "parent": arm(par, "parent")}, args.reps)
    finally:
        cur.close()
        par.close()
    report(f"verified block {count} x {kib} KiB", res, "parent", la)


def probe_inverse(count, kib):
    n = kib << 10
    xs = [bw.generate("markov", n, seed=(73 if count == 1 else 2000 + k)) for k in range(count)]
    cur, par = bw.CudaContext(count * (n + 1)), parent_context(count * (n + 1))
    la = {"this": [], "parent": []}
    try:
        bwts = [x.copy() for x in xs]
        LF, _, _ = cur.bwt_blocks(bwts, 8, want_freqs=False)

        def arm(ctx, name):
            work = [np.empty(b.size, np.uint8) for b in bwts]

            def run():
                for w, b in zip(work, bwts):
                    w[:] = b
                if count == 1:
                    r = timed(ctx, lambda: ctx.inverse_block(work[0], LF[0, :1]), la[name])
                else:
                    r = timed(ctx, lambda: ctx.inverse_blocks(work, LF), la[name])
                assert all(np.array_equal(w, x) for w, x in zip(work, xs))
                return r
            return run
        res = alternate({"this": arm(cur, "this"), "parent": arm(par, "parent")}, args.reps)
    finally:
        cur.close()
        par.close()
    report(f"inverse {count} x {kib} KiB markov", res, "parent", la)


print(f"card: {card()}  (name, power limit, max SM clock)", flush=True)
probe_raw()
for count, kib in ((1, 32 << 10), (32, 1024)):
    probe_block_verify(count, kib)
for count, kib in ((1, 32 << 10), (64, 256)):
    probe_inverse(count, kib)
