#!/usr/bin/env python
"""Cost of the pattern search (not a pytest; profiles/r11_sa_search.md).  Prints the card and its power limit, then:
  - sa_search_device (device-resident text, SA, patterns and results; the SA built by divsufsort_device) on 32 MiB Markov,
    64 MiB DNA, 256 MiB random and 16 MiB repetitive text, for --count patterns of 8, 32, 256 and 4096 bytes, as hits
    (substrings at random positions) and as mutated substrings (one byte changed in the middle: nearly all misses):
    stats.gpu_ms (CUDA events around the two kernels) with its spread over --reps calls, patterns per second, and the
    probes and text bytes compared per pattern (bwtc_cuda_debug_read 10);
  - the host variant sa_search with every array pageable and every array pinned (wall time, 32-byte hits; the call copies
    T and the SA to the device);
  - the C oracle (tests/sa_search_oracle.c) over all host cores, one thread per core on slices of the batch, with the core
    count printed, on --oracle-count of the same patterns; its results are compared with the device's;
  - with --parent-lib: divsufsort_device, divbwtf and bwt_block_device on this library against a library built from an
    earlier commit, alternating in one process, with launch counts: the existing paths must run what they ran before.
With --out PATH the numbers are also written there as JSON.
  python tests/gpu_sa_search_probe.py [--parent-lib path/to/earlier/libbwtc_cuda.so] [--out r11.json]"""
import argparse
import concurrent.futures
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
from test_sa_search_keys import _oracle_lib, oracle_sa_search  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--count", type=int, default=1_000_000)
ap.add_argument("--oracle-count", type=int, default=100_000)
ap.add_argument("--parent-lib", default=None)
ap.add_argument("--out", default=None, help="also write the numbers to this JSON file")
args = ap.parse_args()

MiB = 1 << 20
CASES = [("markov", 32), ("dna", 64), ("random", 256), ("repetitive", 16)]
LENGTHS = (8, 32, 256, 4096)
RESULTS = {}


def spread(v):
    return {"median": statistics.median(v), "min": min(v), "max": max(v)}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "nvidia-smi unavailable"


def device_patterns(torch, dT, n, L, count, miss, seed):
    """count patterns of L bytes cut from the device text at random positions (one byte changed when miss)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    starts = torch.randint(0, n - L + 1, (count,), device="cuda", generator=g)
    dP = torch.empty(count * L, dtype=torch.uint8, device="cuda")
    ar = torch.arange(L, device="cuda")
    step = max(1, (1 << 28) // (L * 8))
    for a in range(0, count, step):
        b = min(count, a + step)
        rows = dT[(starts[a:b, None] + ar[None, :]).reshape(-1)].view(b - a, L)
        if miss:
            rows[:, L // 2] ^= 0x5A
        dP[a * L:b * L] = rows.reshape(-1)
    dO = torch.arange(count + 1, device="cuda", dtype=torch.int64) * L
    return dP, dO


def probe_kind(kind, mib):
    import torch

    n = mib * MiB
    T = bw.generate(kind, n, seed=111)
    dT = torch.from_numpy(T).cuda()
    dSA = torch.empty(n, dtype=torch.int32, device="cuda")
    ctx = bw.CudaContext(n)
    out = {"n": n}
    try:
        ctx.divsufsort_device(dT.data_ptr(), dSA.data_ptr(), n)
        out["divsufsort_device_gpu_ms"] = ctx.stats()["gpu_ms"]
        count = args.count
        dL = torch.empty(count, dtype=torch.int32, device="cuda")
        dS = torch.empty(count, dtype=torch.int32, device="cuda")
        SA = dSA.cpu().numpy()
        for L in LENGTHS:
            for miss in (False, True):
                name = f"{'mutated' if miss else 'hits'} {L}"
                dP, dO = device_patterns(torch, dT, n, L, count, miss, seed=L * 2 + miss)
                torch.cuda.synchronize()

                def run():
                    ctx.sa_search_device(dT.data_ptr(), n, dSA.data_ptr(), n, dP.data_ptr(), dO.data_ptr(), count,
                                         dL.data_ptr(), dS.data_ptr())
                    return ctx.stats()
                run()  # warm-up
                sts = [run() for _ in range(args.reps)]
                g = [s["gpu_ms"] for s in sts]
                probes, nbytes = (int(v) for v in ctx.debug_read(10, np.uint64, 2))
                sizes = dS.cpu().numpy()
                row = {"gpu_ms": spread(g), "patterns_per_s": count / (statistics.median(g) / 1e3),
                       "probes_per_pattern": probes / count, "bytes_per_pattern": nbytes / count,
                       "kernel_launches": sts[-1]["kernel_launches"], "found_fraction": float(np.mean(sizes > 0)),
                       "mean_size": float(sizes.mean())}
                if args.oracle_count:
                    k = min(args.oracle_count, count)
                    P = dP[:k * L].cpu().numpy()
                    P_off = dO[:k + 1].cpu().numpy().view(np.uint64)
                    ncore = os.cpu_count() or 1
                    left = np.empty(k, np.int32)
                    size = np.empty(k, np.int32)
                    bounds = np.linspace(0, k, ncore + 1).astype(int)
                    t0 = time.perf_counter()
                    with concurrent.futures.ThreadPoolExecutor(ncore) as ex:
                        list(ex.map(lambda i: oracle_sa_search(T, SA, P, P_off, int(bounds[i]), int(bounds[i + 1] - bounds[i]),
                                                               left[bounds[i]:], size[bounds[i]:]), range(ncore)))
                    wall = time.perf_counter() - t0
                    same = bool(np.array_equal(left, dL[:k].cpu().numpy()) and np.array_equal(size, sizes[:k]))
                    row["oracle"] = {"cores": ncore, "patterns": k, "wall_ms": wall * 1e3, "patterns_per_s": k / wall,
                                     "same_results": same}
                    assert same, (kind, name)
                out[name] = row
                print(f"{kind:10s} {mib:4d} MiB {name:13s} gpu_ms {row['gpu_ms']['median']:8.3f} "
                      f"(min {row['gpu_ms']['min']:.3f} max {row['gpu_ms']['max']:.3f})  {row['patterns_per_s'] / 1e6:8.2f} M/s  "
                      f"probes {row['probes_per_pattern']:6.2f}  bytes {row['bytes_per_pattern']:9.1f}  found "
                      f"{row['found_fraction']:.3f}" + (f"  oracle {row['oracle']['cores']} cores "
                                                         f"{row['oracle']['patterns_per_s'] / 1e6:.3f} M/s" if "oracle" in row else ""),
                      flush=True)
                del dP, dO
        # host variant: every array pageable, then every array pinned (32-byte hits)
        L = 32
        dP, dO = device_patterns(torch, dT, n, L, count, False, seed=7)
        page = {"T": T, "SA": SA, "P": dP.cpu().numpy(), "P_off": dO.cpu().numpy().view(np.uint64),
                "left": np.empty(count, np.int32), "size": np.empty(count, np.int32)}
        keep = []
        pin = {}
        for k, v in page.items():
            t = torch.from_numpy(v.view(np.int64) if v.dtype == np.uint64 else v).pin_memory()
            keep.append(t)
            pin[k] = t.numpy().view(np.uint64) if v.dtype == np.uint64 else t.numpy()
        host = {}
        for label, a in (("pageable", page), ("pinned", pin)):
            walls, gms = [], []
            for rep in range(args.reps + 1):
                t0 = time.perf_counter()
                ctx.sa_search(a["T"], a["SA"], a["P"], a["P_off"], a["left"], a["size"])
                w = (time.perf_counter() - t0) * 1e3
                if rep:
                    walls.append(w)
                    gms.append(ctx.stats()["gpu_ms"])
            host[label] = {"wall_ms": spread(walls), "gpu_ms": spread(gms)}
            print(f"{kind:10s} {mib:4d} MiB host {label:9s} 32-byte hits wall_ms {statistics.median(walls):9.3f} "
                  f"(min {min(walls):.3f} max {max(walls):.3f})  gpu_ms {statistics.median(gms):.3f}", flush=True)
        assert np.array_equal(page["left"], pin["left"]) and np.array_equal(page["size"], pin["size"])
        out["host 32-byte hits"] = host
    finally:
        ctx.close()
        torch.cuda.empty_cache()
    RESULTS[f"{kind} {mib} MiB"] = out


def parent_context(n):
    """A context on the earlier library: bind only the symbols it exports."""
    saved = bw.C_ABI
    lib = ctypes.CDLL(args.parent_lib)
    bw.C_ABI = [e for e in saved if hasattr(lib, e[0])]
    try:
        return bw.CudaContext(n, lib_path=args.parent_lib)
    finally:
        bw.C_ABI = saved


def probe_parent(kind, mib):
    """divsufsort_device, divbwtf and bwt_block_device, this library and the parent's alternating: device time, launches,
    identical outputs."""
    import torch

    n = mib * MiB
    T = bw.generate(kind, n, seed=93)
    dT = torch.from_numpy(T).cuda()
    cur, par = bw.CudaContext(n), parent_context(n)
    res = {}
    try:
        for what in ("divsufsort_device", "divbwtf", "bwt_block_device"):
            rows = {"this": ([], set(), []), "parent": ([], set(), [])}
            for rep in range(args.reps + 1):
                for name in (("this", "parent") if rep % 2 else ("parent", "this")):
                    ctx = cur if name == "this" else par
                    LF = np.zeros(8, np.uint32)
                    if what == "divsufsort_device":
                        dS = torch.empty(n, dtype=torch.int32, device="cuda")
                        ctx.divsufsort_device(dT.data_ptr(), dS.data_ptr(), n)
                        outv = dS.cpu().numpy()
                    elif what == "divbwtf":
                        U = np.empty_like(T)
                        ctx.divbwtf(T, U, LF, None)
                        U[LF[0]] = 0
                        outv = U
                    else:
                        dU = torch.empty(n, dtype=torch.uint8, device="cuda")
                        ctx.bwt_block_device(dT.data_ptr(), dU.data_ptr(), n, LF, None)
                        outv = dU.cpu().numpy()
                    st = ctx.stats()
                    if rep:
                        rows[name][0].append(st["gpu_ms"])
                    rows[name][1].add(st["kernel_launches"])
                    rows[name][2].append(hash(outv.tobytes()) ^ hash(LF.tobytes()))
            same = len(set(rows["this"][2]) | set(rows["parent"][2])) == 1
            r = {k: {"gpu_ms": spread(v[0]), "kernel_launches": sorted(v[1])} for k, v in rows.items()}
            r["ratio_this_to_parent"] = statistics.median(rows["this"][0]) / statistics.median(rows["parent"][0])
            r["same_outputs"] = same
            res[what] = r
            print(f"parent {kind} {mib} MiB {what:18s} this {r['this']['gpu_ms']['median']:8.3f} ms "
                  f"(min {r['this']['gpu_ms']['min']:.3f} max {r['this']['gpu_ms']['max']:.3f}) launches {r['this']['kernel_launches']} | "
                  f"parent {r['parent']['gpu_ms']['median']:8.3f} ms (min {r['parent']['gpu_ms']['min']:.3f} "
                  f"max {r['parent']['gpu_ms']['max']:.3f}) launches {r['parent']['kernel_launches']} | ratio "
                  f"{r['ratio_this_to_parent']:.4f} same outputs {same}", flush=True)
            assert same and rows["this"][1] == rows["parent"][1], what
    finally:
        cur.close()
        par.close()
    RESULTS[f"parent {kind} {mib} MiB"] = res


if __name__ == "__main__":
    _oracle_lib()  # compiled once, before any timing
    c = card()
    print("card:", c, flush=True)
    RESULTS["card (name, power.limit)"] = c
    RESULTS["settings"] = {"count": args.count, "reps": args.reps, "oracle_count": args.oracle_count}
    for kind, mib in CASES:
        probe_kind(kind, mib)
    if args.parent_lib:
        probe_parent("markov", 32)
    print("card:", card(), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(RESULTS, f, indent=1)
