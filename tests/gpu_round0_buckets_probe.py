"""Cost of the round-0 bucket sort (k_bucket_sort) against the digit passes it replaces: per-block device time and
per-kernel CUDA time (torch.profiler) for every top-pass count, on generated blocks; outputs compared with the 8-pass
mode.  Prints one JSON row per run; with a path as the first argument the rows are also written there as JSON
(profiles/r10_round0_buckets_probe.json)."""
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bwtc_b200 as bw  # noqa: E402

MiB = 1 << 20


def run(x, top, reps):
    os.environ["BWTC_ROUND0_TOP"] = str(top)
    ctx = bw.CudaContext(x.size)
    try:
        LF = np.zeros(bw.num_starting_points(x.size, 8), np.uint32)
        ms, out = [], None
        for _ in range(reps):
            blk = x.copy()
            ctx.bwt_block(blk, LF, None)
            ms.append(ctx.stats()["gpu_ms"])
            out = blk
        st = ctx.stats()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                ctx.bwt_block(x.copy(), LF, None)
            torch.cuda.synchronize()
        kern = {}
        for e in prof.key_averages():
            if e.device_type == torch.autograd.DeviceType.CUDA and ("k_bucket_sort" in e.key or "k_radix_pass" in e.key):
                name = "k_bucket_sort" if "k_bucket_sort" in e.key else "k_radix_pass"
                kern.setdefault(name, [0.0, 0])
                kern[name][0] += e.device_time_total / 1e3 / 3  # ms per block
                kern[name][1] += e.count // 3
        return out, LF.copy(), statistics.median(ms), st, kern
    finally:
        ctx.close()


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else None
    torch.zeros(1).cuda()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    res = {"gpu": gpu, "rows": []}
    cases = [("markov", 32, 1000), ("markov", 32, 1001), ("markov", 16, 1000), ("markov", 64, 1000)]
    for kind, mib, seed in cases:
        x = bw.generate(kind, mib * MiB, seed=seed)
        base = None
        for top in (0, 4, 5, 6, -1):
            os.environ.pop("BWTC_ROUND0_TOP", None)
            out, LF, ms, st, kern = run(x, top, 7) if top >= 0 else _run_env(x)
            if base is None:
                base = (out, LF)
            same = bool(np.array_equal(out, base[0]) and np.array_equal(LF, base[1]))
            row = {"kind": kind, "mib": mib, "seed": seed, "top": top, "gpu_ms": ms, "passes0": st["passes"][0],
                   "flags": st["flags"], "big": st["round0_big_buckets"], "same_as_8pass": same, "kernels": kern}
            print(json.dumps(row), flush=True)
            res["rows"].append(row)
    if path:
        with open(path, "w") as f:
            json.dump(res, f, indent=1)
    print(gpu)


def _run_env(x):
    # default policy: no BWTC_ROUND0_TOP in the environment
    ctx = bw.CudaContext(x.size)
    try:
        LF = np.zeros(bw.num_starting_points(x.size, 8), np.uint32)
        ms = []
        for _ in range(7):
            blk = x.copy()
            ctx.bwt_block(blk, LF, None)
            ms.append(ctx.stats()["gpu_ms"])
        return blk, LF.copy(), statistics.median(ms), ctx.stats(), {}
    finally:
        ctx.close()


if __name__ == "__main__":
    main()
