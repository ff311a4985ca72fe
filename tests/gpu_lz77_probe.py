#!/usr/bin/env python
"""Cost of the LZ77 factorisation (not a pytest; profiles/r12_lz77.md).  Prints the card and its power limit, then,
alternated in one process (medians with min / max over --reps; gpu_ms = stats.gpu_ms, CUDA events around the call's
device work):
  - lz77_device against divsufsort_lcp_device on the same bytes (device-resident buffers), and their difference: 32 MiB
    Markov, 64 MiB DNA, 256 MiB random, 16 MiB repetitive, 32 MiB of real source text, one byte at 256 MiB; beside them
    the phrase count, the stage's counters (rows outside their tile, marking rounds), launches, and the time of the
    sequential C oracle (tests/lz77_oracle.c) parsing the same text from its SA on one host core;
  - the host variant lz77 into pinned and into pageable arrays (wall time: 8 bytes per phrase come back);
  - divsufsort_lcp_device, divsufsort_device, divbwtf and bwt_block_device on this library against a library built from
    an earlier commit (--parent-lib), with launch counts and outputs: the existing paths must run what they ran before.
With --out PATH the numbers are also written there as JSON.
  python tests/gpu_lz77_probe.py --parent-lib path/to/earlier/libbwtc_cuda.so [--reps 5]"""
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
from test_lz77_keys import decode, oracle_lz77  # noqa: E402

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


def lz_counters(ctx):
    """LzCtl of the last lz77 (bwtc_cuda_debug_read 11): phrases, rows outside their tile (u64), HBM rounds (u32)."""
    c = ctx.debug_read(11, np.uint64, 2)
    return {"phrases": int(c[0]), "rows_outside_tile": int(c[1]),
            "marking_rounds": int(ctx.debug_read(11, np.uint32, 1, offset_bytes=16)[0])}


def probe_device(kind, mib):
    import torch

    T = text(kind, mib, 91)
    n = T.size
    dT = torch.from_numpy(T).cuda()
    dSA = torch.empty(n, dtype=torch.int32, device="cuda")
    dLCP = torch.empty(n, dtype=torch.int32, device="cuda")
    d_src = torch.empty(n, dtype=torch.int32, device="cuda")
    d_len = torch.empty(n, dtype=torch.int32, device="cuda")
    ctx = bw.CudaContext(n)
    launches = {"divsufsort_lcp_device": set(), "lz77_device": set()}
    info = {}
    try:
        def lcp():
            g, w, st = timed(ctx, lambda: ctx.divsufsort_lcp_device(dT.data_ptr(), dSA.data_ptr(), dLCP.data_ptr(), n),
                             torch.cuda.synchronize)
            assert st["flags"] & bw.FLAG_LCP and not st["flags"] & bw.FLAG_LZ77
            launches["divsufsort_lcp_device"].add(st["kernel_launches"])
            return g, w

        def lz():
            g, w, st = timed(ctx, lambda: info.__setitem__("z", ctx.lz77_device(dT.data_ptr(), n, d_src.data_ptr(),
                                                                                 d_len.data_ptr(), n)), torch.cuda.synchronize)
            assert st["flags"] & bw.FLAG_LZ77
            launches["lz77_device"].add(st["kernel_launches"])
            return g, w
        res = alternate({"divsufsort_lcp_device": lcp, "lz77_device": lz}, args.reps)
        z = info["z"]
        cnt = lz_counters(ctx)
        assert cnt["phrases"] == z
        src, ln = d_src[:z].cpu().numpy(), d_len[:z].cpu().numpy()
        SA = dSA.cpu().numpy()
        t0 = time.perf_counter()
        want_src, want_len = oracle_lz77(T, SA)
        oracle_ms = (time.perf_counter() - t0) * 1e3
        assert np.array_equal(src, want_src) and np.array_equal(ln, want_len), kind
        assert np.array_equal(decode(src, ln, n), T), kind
        cnt.update({"n": n, "bytes_per_phrase": n / z, "max_len": int(ln.max()), "literals": int((ln == 0).sum()),
                    "oracle_parse_ms_one_core": oracle_ms})
        report(f"device {kind} {mib} MiB", res, "divsufsort_lcp_device",
               ["kernel launches per call: " + ", ".join(f"{k} {sorted(v)}" for k, v in launches.items()),
                "LZ77 stage: " + ", ".join(f"{k} {v:.4g}" if isinstance(v, float) else f"{k} {v}" for k, v in cnt.items())])
        RESULTS[f"device {kind} {mib} MiB"]["lz77_stage"] = cnt
    finally:
        ctx.close()
        del dT, dSA, dLCP, d_src, d_len
        torch.cuda.empty_cache()


def probe_host(kind, mib):
    import torch

    T = text(kind, mib, 92)
    n = T.size
    pin = (torch.empty(n, dtype=torch.int32).pin_memory().numpy(), torch.empty(n, dtype=torch.int32).pin_memory().numpy())
    page = (np.empty(n, np.int32), np.empty(n, np.int32))
    ctx = bw.CudaContext(n)
    got = {}
    try:
        def arm(name, bufs):
            def run():
                g, w, _ = timed(ctx, lambda: got.__setitem__(name, ctx.lz77(T, *bufs)))
                return g, w
            return run
        res = alternate({"pinned src+len": arm("pinned", pin), "pageable src+len": arm("pageable", page)}, args.reps)
        z = got["pinned"][0].size
        assert np.array_equal(got["pinned"][0], got["pageable"][0]) and np.array_equal(got["pinned"][1], got["pageable"][1])
        report(f"host {kind} {mib} MiB", res, "pinned src+len", f"phrases {z} ({8 * z / MiB:.2f} MiB back)")
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
            dL = torch.empty(n, dtype=torch.int32, device="cuda")
            U = np.empty_like(T)

            def run():
                LF = np.zeros(8, np.uint32)
                if what == "raw":
                    g, w, st = timed(ctx, lambda: ctx.divbwtf(T, U, LF, None))
                    out = U.copy()
                elif what == "block":
                    g, w, st = timed(ctx, lambda: ctx.bwt_block_device(dT.data_ptr(), dU.data_ptr(), n, LF, None),
                                     torch.cuda.synchronize)
                    out = dU.cpu().numpy()
                elif what == "lcp":
                    g, w, st = timed(ctx, lambda: ctx.divsufsort_lcp_device(dT.data_ptr(), dS.data_ptr(), dL.data_ptr(), n),
                                     torch.cuda.synchronize)
                    out = np.concatenate([dS.cpu().numpy(), dL.cpu().numpy()])
                else:
                    g, w, st = timed(ctx, lambda: ctx.divsufsort_device(dT.data_ptr(), dS.data_ptr(), n), torch.cuda.synchronize)
                    out = dS.cpu().numpy()
                la[name].add(st["kernel_launches"])
                assert not st["flags"] & bw.FLAG_LZ77
                if what not in ref:
                    ref[what] = (out.copy(), LF.copy())
                keep = np.arange(n) != LF[0] if what == "raw" else slice(None)
                assert np.array_equal(out[keep], ref[what][0][keep]) and np.array_equal(LF, ref[what][1])
                return g, w
            return run
        for what, call in (("lcp", "divsufsort_lcp_device"), ("sa", "divsufsort_device"), ("raw", "divbwtf"),
                           ("block", "bwt_block_device")):
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
