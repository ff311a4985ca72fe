#!/usr/bin/env python
"""Cost of the LCP array (not a pytest; profiles/r09_lcp.md).  Prints the card and its power limit, then, alternated in one
process (medians with min / max over --reps; gpu_ms = stats.gpu_ms, CUDA events around the call's device work):
  - divsufsort_lcp_device against divsufsort_device on the same bytes (device-resident buffers), and their difference:
    32 MiB Markov, 64 MiB DNA, 256 MiB random, 16 MiB repetitive, 32 MiB of real source text, one byte at 256 MiB; beside
    them the LCP stage's device counters (irreducible rows, bytes compared, pairs in the long tier, window segments), the
    maximum and mean LCP, and stats.rounds;
  - the host variant divsufsort_lcp into pinned and into pageable arrays (wall time: 8 bytes per input byte come back);
  - divsufsort_device, divbwtf and bwt_block_device on this library against a library built from an earlier commit
    (--parent-lib), with launch counts: the existing paths must run what they ran before.
With --out PATH the numbers are also written there as JSON.
  python tests/gpu_lcp_probe.py --parent-lib path/to/earlier/libbwtc_cuda.so [--reps 5]"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import bwtc_b200 as bw  # noqa: E402
from _inputs import real_source_text  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--parent-lib", required=True)
ap.add_argument("--out", default=None, help="also write the numbers to this JSON file")
args = ap.parse_args()

MiB = 1 << 20
CASES = [("markov", 32), ("dna", 64), ("random", 256), ("repetitive", 16), ("source", 32), ("one_byte", 256)]
RESULTS = {}


def spread(v):
    return {"median": statistics.median(v), "min": min(v), "max": max(v)}


def fmt(v):
    s = spread(v)
    return f"median {s['median']:8.3f}  min {s['min']:8.3f}  max {s['max']:8.3f}"


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "nvidia-smi unavailable"


def text(kind, mib, seed):
    n = mib * MiB
    if kind == "source":
        return real_source_text(n)  # (fewer bytes where the interpreter's tree is smaller: the report prints n)
    if kind == "one_byte":
        return np.full(n, 0x61, np.uint8)
    return bw.generate(kind, n, seed=seed)


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


def report(title, res, base=None, extra=None):
    out = {}
    for k, (g, w) in res.items():
        print(f"{title:30s} {k:24s} gpu_ms {fmt(g)} | wall_ms {fmt(w)}", flush=True)
        out[k] = {"gpu_ms": spread(g), "wall_ms": spread(w)}
    if base:
        for k, (g, w) in res.items():
            if k != base:
                dg = statistics.median(g) - statistics.median(res[base][0])
                rg = statistics.median(g) / statistics.median(res[base][0])
                rw = statistics.median(w) / statistics.median(res[base][1])
                print(f"{'':30s} {k} - {base} (medians): device {dg:+.3f} ms; ratio device {rg:.4f}, wall {rw:.4f}", flush=True)
                out[k]["minus_" + base] = dg
                out[k]["ratio_to_" + base] = {"device": rg, "wall": rw}
    if extra:
        for line in extra if isinstance(extra, list) else [extra]:
            print(f"{'':30s} {line}", flush=True)
        out["note"] = extra
    RESULTS[title] = out


def timed(ctx, fn, sync=None):
    t0 = time.perf_counter()
    fn()
    if sync:
        sync()
    wall = (time.perf_counter() - t0) * 1e3
    st = ctx.stats()
    return st["gpu_ms"], wall, st


def lcp_counters(ctx):
    """LcpCtl of the last divsufsort_lcp (bwtc_cuda_debug_read 9): 4 x u64, then the window list lengths."""
    c = ctx.debug_read(9, np.uint64, 4)
    lists = ctx.debug_read(9, np.uint32, 33, offset_bytes=32)
    return {"irreducible": int(c[0]), "short_bytes": int(c[1]), "window_bytes": int(c[2]), "segments": int(c[3]),
            "long_pairs": int(lists[0]), "windows_used": int(np.count_nonzero(lists))}


def probe_device(kind, mib):
    import torch

    T = text(kind, mib, 91)
    n = T.size
    dT = torch.from_numpy(T).cuda()
    dSA = torch.empty(n, dtype=torch.int32, device="cuda")
    dLCP = torch.empty(n, dtype=torch.int32, device="cuda")
    ctx = bw.CudaContext(n)
    launches = {"divsufsort_device": set(), "divsufsort_lcp_device": set()}
    info = {}
    try:
        def sa():
            g, w, st = timed(ctx, lambda: ctx.divsufsort_device(dT.data_ptr(), dSA.data_ptr(), n), torch.cuda.synchronize)
            assert st["flags"] & bw.FLAG_SA and not st["flags"] & bw.FLAG_LCP
            launches["divsufsort_device"].add(st["kernel_launches"])
            return g, w

        def lcp():
            g, w, st = timed(ctx, lambda: ctx.divsufsort_lcp_device(dT.data_ptr(), dSA.data_ptr(), dLCP.data_ptr(), n),
                             torch.cuda.synchronize)
            assert st["flags"] & bw.FLAG_LCP
            launches["divsufsort_lcp_device"].add(st["kernel_launches"])
            info["rounds"] = st["rounds"]
            return g, w
        res = alternate({"divsufsort_device": sa, "divsufsort_lcp_device": lcp}, args.reps)
        cnt = lcp_counters(ctx)
        L = dLCP.cpu().numpy().astype(np.int64)
        cnt.update({"n": n, "irreducible_fraction": cnt["irreducible"] / max(n - 1, 1), "max_lcp": int(L.max()),
                    "mean_lcp": float(L.mean()), "rounds": info["rounds"]})
        if kind == "one_byte":
            assert np.array_equal(L, np.arange(n))
        report(f"device {kind} {mib} MiB", res, "divsufsort_device",
               ["kernel launches per call: " + ", ".join(f"{k} {sorted(v)}" for k, v in launches.items()),
                "LCP stage: " + ", ".join(f"{k} {v:.4g}" if isinstance(v, float) else f"{k} {v}" for k, v in cnt.items())])
        RESULTS[f"device {kind} {mib} MiB"]["lcp_stage"] = cnt
    finally:
        ctx.close()
        del dT, dSA, dLCP
        torch.cuda.empty_cache()


def probe_host(kind, mib):
    import torch

    T = text(kind, mib, 92)
    n = T.size
    pin = (torch.empty(n, dtype=torch.int32).pin_memory().numpy(), torch.empty(n, dtype=torch.int32).pin_memory().numpy())
    page = (np.empty(n, np.int32), np.empty(n, np.int32))
    ctx = bw.CudaContext(n)
    try:
        def arm(bufs):
            def run():
                g, w, _ = timed(ctx, lambda: ctx.divsufsort_lcp(T, *bufs))
                return g, w
            return run
        res = alternate({"pinned SA+LCP": arm(pin), "pageable SA+LCP": arm(page)}, args.reps)
        assert np.array_equal(pin[0], page[0]) and np.array_equal(pin[1], page[1])
        report(f"host {kind} {mib} MiB", res, "pinned SA+LCP")
    finally:
        ctx.close()


def probe_parent(kind, mib):
    import torch

    T = text(kind, mib, 93)
    n = T.size
    dT = torch.from_numpy(T).cuda()
    cur, par = bw.CudaContext(n), parent_context(n)
    la = {}
    ref = {}
    try:
        def arm(ctx, name, what):
            la[name] = set()
            dU = torch.empty(n, dtype=torch.uint8, device="cuda")
            dS = torch.empty(n, dtype=torch.int32, device="cuda")
            U = np.empty_like(T)

            def run():
                LF = np.zeros(8, np.uint32)
                if what == "raw":
                    g, w, st = timed(ctx, lambda: ctx.divbwtf(T, U, LF, None))
                    out = U
                elif what == "block":
                    g, w, st = timed(ctx, lambda: ctx.bwt_block_device(dT.data_ptr(), dU.data_ptr(), n, LF, None),
                                     torch.cuda.synchronize)
                    out = dU.cpu().numpy()
                else:
                    g, w, st = timed(ctx, lambda: ctx.divsufsort_device(dT.data_ptr(), dS.data_ptr(), n), torch.cuda.synchronize)
                    out = dS.cpu().numpy()
                la[name].add(st["kernel_launches"])
                assert not st["flags"] & bw.FLAG_LCP
                if what not in ref:
                    ref[what] = (out.copy(), LF.copy())
                keep = np.arange(n) != LF[0] if what == "raw" else slice(None)
                assert np.array_equal(out[keep], ref[what][0][keep]) and np.array_equal(LF, ref[what][1])
                return g, w
            return run
        for what, call in (("sa", "divsufsort_device"), ("raw", "divbwtf"), ("block", "bwt_block_device")):
            a, b = f"this {call}", f"parent {call}"
            res = alternate({a: arm(cur, a, what), b: arm(par, b, what)}, args.reps)
            report(f"parent {kind} {mib} MiB {what}", res, b,
                   "kernel launches per call: " + ", ".join(f"{k} {sorted(la[k])}" for k in (a, b)))
            assert la[a] == la[b]
    finally:
        cur.close()
        par.close()


if __name__ == "__main__":
    c = card()
    print("card:", c, flush=True)
    RESULTS["card"] = c
    for kind, mib in CASES:
        probe_device(kind, mib)
    for kind, mib in (("markov", 32), ("dna", 64)):
        probe_host(kind, mib)
    for kind, mib in (("markov", 32), ("dna", 64)):
        probe_parent(kind, mib)
    print("card:", card(), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(RESULTS, f, indent=1)
