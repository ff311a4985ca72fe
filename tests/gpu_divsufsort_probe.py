#!/usr/bin/env python
"""Cost of the suffix array (not a pytest; profiles/r06_divsufsort.md).  Prints the card and its power limit, then, alternated
in one process (medians with min / max over --reps; gpu_ms = stats.gpu_ms, CUDA events around the call's device work):
  - divsufsort_device against bwt_block_device on the same bytes (device-resident input and output): 32 MiB Markov,
    64 MiB DNA, 256 MiB random, 16 MiB repetitive; and sufcheck's device time on each SA;
  - the host variant divsufsort from a pinned and from a pageable SA (wall time: it copies 4 bytes per input byte back);
  - bwt_block_device and divbwtf on this library against a library built from an earlier commit (--parent-lib), with
    launch counts: with the SA off the forward paths must run what they ran before.
With --out PATH the numbers are also written there as JSON.
  python tests/gpu_divsufsort_probe.py --parent-lib path/to/earlier/libbwtc_cuda.so [--reps 5]"""
import argparse
import ctypes
import json
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
ap.add_argument("--parent-lib", required=True)
ap.add_argument("--out", default=None, help="also write the numbers to this JSON file")
args = ap.parse_args()

MiB = 1 << 20
CASES = [("markov", 32), ("dna", 64), ("random", 256), ("repetitive", 16)]
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
        print(f"{title:30s} {k:18s} gpu_ms {fmt(g)} | wall_ms {fmt(w)}", flush=True)
        out[k] = {"gpu_ms": spread(g), "wall_ms": spread(w)}
    if base:
        for k, (g, w) in res.items():
            if k != base:
                rg = statistics.median(g) / statistics.median(res[base][0])
                rw = statistics.median(w) / statistics.median(res[base][1])
                print(f"{'':30s} {k} / {base} (medians): device {rg:.4f}, wall {rw:.4f}", flush=True)
                out[k]["ratio_to_" + base] = {"device": rg, "wall": rw}
    if extra:
        print(f"{'':30s} {extra}", flush=True)
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


def probe_device(kind, mib):
    import torch

    T = bw.generate(kind, mib * MiB, seed=81)
    n = T.size
    dT = torch.from_numpy(T).cuda()
    dSA = torch.empty(n, dtype=torch.int32, device="cuda")
    dU = torch.empty(n, dtype=torch.uint8, device="cuda")
    ctx = bw.CudaContext(n)
    launches = {"bwt_block_device": set(), "divsufsort_device": set()}
    try:
        def bwt():
            g, w, st = timed(ctx, lambda: ctx.bwt_block_device(dT.data_ptr(), dU.data_ptr(), n, np.zeros(8, np.uint32), None),
                             torch.cuda.synchronize)
            launches["bwt_block_device"].add(st["kernel_launches"])
            return g, w

        def sa():
            g, w, st = timed(ctx, lambda: ctx.divsufsort_device(dT.data_ptr(), dSA.data_ptr(), n), torch.cuda.synchronize)
            assert st["flags"] & bw.FLAG_SA
            launches["divsufsort_device"].add(st["kernel_launches"])
            return g, w
        res = alternate({"bwt_block_device": bwt, "divsufsort_device": sa}, args.reps)
        report(f"device {kind} {mib} MiB", res, "bwt_block_device",
               "kernel launches per call: " + ", ".join(f"{k} {sorted(v)}" for k, v in launches.items()))
        # sufcheck of that SA (host entry: T and SA are uploaded first; gpu_ms covers the check kernels only)
        SA = dSA.cpu().numpy()
        gs, ws = [], []
        for rep in range(args.reps + 1):
            t0 = time.perf_counter()
            assert ctx.sufcheck(T, SA)
            w = (time.perf_counter() - t0) * 1e3
            if rep:
                gs.append(ctx.stats()["gpu_ms"])
                ws.append(w)
        report(f"sufcheck {kind} {mib} MiB", {"sufcheck": (gs, ws)})
    finally:
        ctx.close()
        del dT, dSA, dU
        torch.cuda.empty_cache()


def probe_host(kind, mib):
    import torch

    T = bw.generate(kind, mib * MiB, seed=82)
    n = T.size
    pinned = torch.empty(n, dtype=torch.int32).pin_memory().numpy()
    pageable = np.empty(n, np.int32)
    ctx = bw.CudaContext(n)
    try:
        def arm(SA):
            def run():
                g, w, _ = timed(ctx, lambda: ctx.divsufsort(T, SA))
                return g, w
            return run
        res = alternate({"pinned SA": arm(pinned), "pageable SA": arm(pageable)}, args.reps)
        assert np.array_equal(pinned, pageable)
        report(f"host {kind} {mib} MiB", res, "pinned SA")
    finally:
        ctx.close()


def probe_parent(kind, mib):
    import torch

    T = bw.generate(kind, mib * MiB, seed=83)
    n = T.size
    dT = torch.from_numpy(T).cuda()
    cur, par = bw.CudaContext(n), parent_context(n)
    la = {}
    ref = {}
    try:
        def arm(ctx, name, raw):
            la[name] = set()
            dU = torch.empty(n, dtype=torch.uint8, device="cuda")
            U = np.empty_like(T)

            def run():
                LF = np.zeros(8, np.uint32)
                if raw:
                    g, w, st = timed(ctx, lambda: ctx.divbwtf(T, U, LF, None))
                    out = U
                else:
                    g, w, st = timed(ctx, lambda: ctx.bwt_block_device(dT.data_ptr(), dU.data_ptr(), n, LF, None),
                                     torch.cuda.synchronize)
                    out = dU.cpu().numpy()
                la[name].add(st["kernel_launches"])
                assert not st["flags"] & bw.FLAG_SA
                key = "raw" if raw else "block"
                if key not in ref:
                    ref[key] = (out.copy(), LF.copy())
                keep = np.arange(n) != LF[0] if raw else slice(None)
                assert np.array_equal(out[keep], ref[key][0][keep]) and np.array_equal(LF, ref[key][1])
                return g, w
            return run
        res = alternate({"this bwt_block_device": arm(cur, "this bwt_block_device", False),
                         "parent bwt_block_device": arm(par, "parent bwt_block_device", False)}, args.reps)
        report(f"parent {kind} {mib} MiB block", res, "parent bwt_block_device",
               "kernel launches per call: " + ", ".join(f"{k} {sorted(v)}" for k, v in la.items()))
        assert la["this bwt_block_device"] == la["parent bwt_block_device"]
        res = alternate({"this divbwtf": arm(cur, "this divbwtf", True), "parent divbwtf": arm(par, "parent divbwtf", True)},
                        args.reps)
        report(f"parent {kind} {mib} MiB raw", res, "parent divbwtf",
               "kernel launches per call: " + ", ".join(f"{k} {sorted(v)}" for k, v in la.items() if "divbwtf" in k))
        assert la["this divbwtf"] == la["parent divbwtf"]
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
