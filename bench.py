#!/usr/bin/env python
"""bench.py — forward-BWT throughput of the B200-native engine (BASELINE.json metric) + roofline + CPU baseline.

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W   (the reference's own CPU path)
    python bench.py --gpus N ... --dump-outputs DIR    also write what the last timed step computed as DIR/<name>.npy
                                                     (N > 1: DIR/<name>_rank<r>.npy, one set per rank)

A "step" is one pass of the hot path over one batch of synthetic input: BLOCKS_PER_STEP independent 32 MiB blocks
of order-2 Markov text per GPU (BASELINE.json config 5 at one GPU's share), transformed through the batched
look-ahead pipeline (bwtc_cuda_pipeline_run, include/bwtc_cuda.h).
  value        : MB/s of input text, inputs and outputs resident in HBM, timed with CUDA events over all pipeline streams.
  e2e          : the same metric through the host-buffer C-ABI call (pinned host in/out, H2D + D2H inside the timed region).
  e2e_pageable : ... with malloc'ed (pageable) host buffers, what a bwtc PrecompressorBlock is: staged through the engine's
                 pinned ring on copy streams of their own.
  roofline     : the dominant kernel (k_radix_pass): algorithmic bytes per launch / average launch duration, measured
                 live with CUDA events on the launching stream in a separate single-stream leg.
  configs      : one entry per BASELINE.json config (1 MiB Markov batched, 64 MiB DNA, 16 MiB repetitive, 256 MiB random,
                 32 MiB Markov): value / e2e / rounds / live / passes / algorithmic bytes / whole-block roofline fraction.
  compress_e2e : BASELINE config 5 end to end — bwtc::PipelinedCompressor (reader -> GPU BWT look-ahead -> parallel CPU
                 Huffman coding with the reference's own HuffmanEncoder -> ordered writer), MB/s of input, cores stated.
  cpu_baseline : the UNMODIFIED reference (oracle/_ref, divsufsort path) on the host cores, bounded sample.
No oracle/ code is on the measured GPU path; oracle/_ref is executed only by the cpu_baseline / --impl reference legs.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BLOCK_BYTES = 32 << 20
BLOCKS_PER_STEP = 16
STARTS = 8
KIND = "markov"
WORKLOAD = ("order-2 Markov text (sigma 64, Dirichlet 0.05), 32 MiB blocks, %d blocks (512 MiB) per GPU per step, "
            "8 starting points, block contract (BWTransform::doTransform(BWTBlock&, freqs))" % BLOCKS_PER_STEP)
METRIC = "forward BWT MB/s (SA+BWT, 32 MiB blocks)"
DTYPE = "u8 text / u32 ranks / u64 sort keys (integer)"
MEM_32MIB = 181375309  # Compressor memLimit with floor(0.185 * mem) = 32 MiB (Compressor.cpp:78)


def make_config(**kw):
    """Both arms print the same keys (the driver compares the two config dicts)."""
    cfg = {"workload": WORKLOAD, "pipeline_depth": None, "l2": None,
           "parallelism": "independent blocks sharded by rank (block i -> rank i mod G), no collective on the data path",
           "host": None, "lookback_tile_ids": None, "host_wait": None, "sample": None}
    cfg.update(kw)
    return cfg


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def _gen_blocks(count, seed0, nbytes=BLOCK_BYTES, kind=KIND, out=None):
    import bwtc_b200 as bw

    bufs = out if out is not None else [np.empty(nbytes, np.uint8) for _ in range(count)]
    with ThreadPoolExecutor(max_workers=min(count, os.cpu_count() or 1)) as ex:
        list(ex.map(lambda i: bw.generate(kind, nbytes, seed=seed0 + i, out=bufs[i]), range(count)))
    return bufs


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md clocks line)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                pw.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "power_w_max": float(max(pw)), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ reference
class RefLib:
    def __init__(self):
        p = os.path.join(ROOT, "oracle", "_ref", "libbwtc_ref.so")
        self.kind = "reference"
        if not os.path.exists(p):
            raise RuntimeError("oracle/_ref/libbwtc_ref.so missing (build with __graft_entry__.build() where "
                               "/root/reference exists)")
        self.lib = ctypes.CDLL(p)

    def bwt_block(self, buf, n):
        """BWTManager('d', 8 starting points).doTransform(block, freqs) — the reference's divsufsort path."""
        LF = np.zeros(256, np.uint32)
        k = ctypes.c_uint32(0)
        fr = np.zeros(256, np.uint32)
        self.lib.ref_bwt_block(ctypes.c_void_p(buf.ctypes.data), ctypes.c_uint(n), ctypes.c_uint(STARTS),
                               ctypes.c_char(b"d"), ctypes.c_void_p(LF.ctypes.data), ctypes.byref(k),
                               ctypes.c_void_p(fr.ctypes.data))


def run_reference_threads(ref, blocks_src, cores):
    """One worker thread per core with private buffers over independent blocks (ctypes drops the GIL).
    Returns wall seconds for transforming len(blocks_src) blocks."""
    work = [np.concatenate([b, np.zeros(1, np.uint8)]) for b in blocks_src]
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=cores) as ex:
        list(ex.map(lambda w: ref.bwt_block(w, w.size - 1), work))
    return time.perf_counter() - t0


def cpu_baseline_sample(cores, blocks_per_core=1):
    ref = RefLib()
    nb = cores * blocks_per_core
    blocks = _gen_blocks(nb, seed0=9000)
    dt = run_reference_threads(ref, blocks, cores)
    mbps = nb * BLOCK_BYTES / 1e6 / dt
    return {"value": mbps, "unit": "MB/s", "cores": cores, "kind": "reference",
            "per_core_mbps": mbps / cores,
            "sample": "%d x 32 MiB Markov blocks (same generator as the GPU arm), one block per host thread, "
                      "reference Divsufsorter via BWTManager('d'), 8 starting points, %.1f s wall" % (nb, dt)}


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    ref = RefLib()
    blocks = _gen_blocks(cores, seed0=9000)
    for _ in range(args.warmup):
        run_reference_threads(ref, blocks[: max(1, cores // 4)], cores)
    t = 0.0
    for _ in range(args.steps):
        t += run_reference_threads(ref, blocks, cores)
    mbps = args.steps * cores * BLOCK_BYTES / 1e6 / t
    sample = ("each step = %d x 32 MiB Markov blocks, one per host thread (%d threads), reference Divsufsorter via "
              "BWTManager('d'), 8 starting points" % (cores, cores))
    line = {"impl": "reference", "metric": METRIC, "value": mbps, "unit": "MB/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE,
            "data": "synthetic", "config": make_config(sample=sample, host="%d host threads" % cores),
            "cpu_baseline": {"value": mbps, "unit": "MB/s", "cores": cores, "kind": "reference", "sample": sample},
            "e2e": {"value": mbps, "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------------ compress leg (config 5)
def compress_leg(device, nblocks, threads, depth, seed0):
    """BASELINE config 5 end to end, in a process of its own (libbwtc_integration.so contains the reference's objects and
    must not share a process with oracle/_ref): nblocks x 32 MiB of Markov text in host memory ->
    bwtc::PipelinedCompressor(choice 'c', coder 'H') -> .bwtc bytes (counted).  Prints one JSON line."""
    import bwtc_b200 as bw

    lib = ctypes.CDLL(bw.INTEGRATION_LIB_PATH)
    lib.b200_pipelined_compress_mem.restype = ctypes.c_longlong
    n = nblocks * BLOCK_BYTES
    data = np.empty(n, np.uint8)
    _gen_blocks(nblocks, seed0, out=[data[i * BLOCK_BYTES:(i + 1) * BLOCK_BYTES] for i in range(nblocks)])
    devs = (ctypes.c_int * 1)(device)
    err = ctypes.create_string_buffer(1024)
    res = []
    for rep in range(2):  # first pass warms the pipeline (context allocation, page faults of the staging buffers)
        tm = (ctypes.c_double * 10)()
        t0 = time.perf_counter()
        r = lib.b200_pipelined_compress_mem(ctypes.c_void_p(data.ctypes.data), ctypes.c_ulonglong(n), ctypes.c_ulonglong(MEM_32MIB),
                                            ctypes.c_char(b"H"), ctypes.c_char(b"c"), ctypes.c_uint(STARTS), ctypes.c_uint(threads),
                                            ctypes.c_uint(0), devs, ctypes.c_uint(1), ctypes.c_int(depth), None,
                                            ctypes.c_ulonglong(0), tm, err, ctypes.c_uint(1024))
        dt = time.perf_counter() - t0
        if r < 0:
            print(json.dumps({"error": err.value.decode(errors="replace")}))
            return 1
        res.append((dt, int(r), list(tm)))
    dt, size, tm = res[-1]
    try:
        lib.b200_shutdown()
    except Exception:  # noqa: BLE001
        pass
    print(json.dumps({"seconds": dt, "input_bytes": n, "compressed_bytes": size, "encoder_threads": threads, "pipeline_depth": depth,
                      "encoder_busy_core_s": tm[2], "reader_busy_s": tm[1], "writer_busy_s": tm[3], "first_pass_seconds": res[0][0]}))
    return 0


def run_compress_leg(local_rank, world, rank):
    cores = os.cpu_count() or 1
    threads = max(1, cores // world)
    nblocks = 32 if world == 1 else 16
    cmd = [sys.executable, os.path.abspath(__file__), "--leg", "compress", "--leg-device", str(local_rank), "--leg-blocks",
           str(nblocks), "--leg-threads", str(threads), "--leg-seed", str(5000 + 1000 * rank)]
    env = dict(os.environ)
    # glibc: back malloc's mmap'ed chunks with transparent huge pages (the reference allocates and frees ~5 block sizes of
    # scratch per block — PrecompressorBlock.cpp:41, HuffmanCoders.cpp:125-126 — one page fault per 4 KiB otherwise)
    env.setdefault("GLIBC_TUNABLES", "glibc.malloc.hugetlb=1")
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
        out = json.loads(r.stdout.strip().splitlines()[-1])
    except Exception as e:  # noqa: BLE001
        return {"error": "compress leg failed: %s" % e}
    return out


# ------------------------------------------------------------------------------------------------ GPU arm
def measure_workload(bw, torch, dev, local_rank, kind, nbytes, nblocks, depth, reps, seed0, want_e2e=True):
    """One BASELINE config on this GPU: device-resident throughput through the pipeline, the host-buffer (pinned) figure,
    and the per-block execution record of the first block."""
    host_in = [torch.empty(nbytes, dtype=torch.uint8).pin_memory() for _ in range(nblocks)]
    _gen_blocks(nblocks, seed0, nbytes, kind, out=[t.numpy() for t in host_in])
    host_out = [torch.empty(nbytes, dtype=torch.uint8).pin_memory() for _ in range(nblocks)]
    dev_in = [t.to(dev) for t in host_in]
    dev_out = [torch.empty_like(t) for t in dev_in]
    sizes = [nbytes] * nblocks
    pipe = bw.Pipeline(nbytes, depth=depth, device=local_rank)
    try:
        d_in, d_out = [t.data_ptr() for t in dev_in], [t.data_ptr() for t in dev_out]
        h_in, h_out = [t.data_ptr() for t in host_in], [t.data_ptr() for t in host_out]
        pipe.run_ptrs(d_in, d_out, sizes, STARTS, on_device=True, want_stats=False)
        torch.cuda.synchronize()
        pipe.timing_begin()
        for _ in range(reps):
            LF, nLF, fr, stats = pipe.run_ptrs(d_in, d_out, sizes, STARTS, on_device=True)
        ms = pipe.timing_end()
        value = reps * nblocks * nbytes / 1e6 / (ms / 1e3)
        e2e = None
        if want_e2e:
            pipe.run_ptrs(h_in, h_out, sizes, STARTS, on_device=False, want_stats=False)
            t0 = time.perf_counter()
            for _ in range(reps):
                LFh, _, frh, _ = pipe.run_ptrs(h_in, h_out, sizes, STARTS, on_device=False, want_stats=False)
            e2e = reps * nblocks * nbytes / 1e6 / (time.perf_counter() - t0)
            assert (LFh == LF).all() and (frh == fr).all()
            assert torch.equal(dev_out[0].cpu(), host_out[0]) and torch.equal(dev_out[-1].cpu(), host_out[-1])
    finally:
        pipe.close()
    seen, alg, gms, launches = set(), 0, 0.0, 0
    for i, s in enumerate(stats):  # a batch's record is shared by its blocks: count it once
        key = i if s["batch_blocks"] <= 1 else ("b", s["n_suffixes"], s["gpu_ms"])
        if key in seen:
            continue
        seen.add(key)
        alg += s["algorithmic_bytes"]
        gms += s["gpu_ms"]
        launches += s["kernel_launches"]
    s0 = stats[0]
    return {"value": value, "e2e": e2e, "stats0": s0, "alg_bytes_per_input_byte": alg / float(nblocks * nbytes),
            "launches_per_step": launches, "sum_block_gpu_ms": gms}


DUMP_SAMPLES_PER_BLOCK = 1 << 19


def dump_outputs(directory, suffix, dev_out, LF, nLF, freqs):
    """What the last timed step handed its caller for this rank's blocks, as float arrays: the transformed bytes at a
    fixed sample of distinct positions (seed 0, float32, 32 MiB per rank), and the LFpowers and freqs (float64: exact
    for the u32 values).  The inputs are seeded too, so two builds given the same arguments can be compared file by
    file."""
    import torch

    os.makedirs(directory, exist_ok=True)
    n = dev_out[0].numel()
    pos = np.sort(np.random.default_rng(0).choice(n, DUMP_SAMPLES_PER_BLOCK, replace=False))
    idx = torch.from_numpy(pos).to(dev_out[0].device)
    sample = torch.stack([t[idx] for t in dev_out]).float().cpu().numpy()
    np.save(os.path.join(directory, "bwt_sample%s.npy" % suffix), sample)
    np.save(os.path.join(directory, "lfpowers%s.npy" % suffix),
            np.stack([LF[i, : nLF[i]] for i in range(len(dev_out))]).astype(np.float64))
    np.save(os.path.join(directory, "freqs%s.npy" % suffix), np.asarray(freqs, np.float64))


def main_gpu(args):
    import torch
    import torch.distributed as dist

    import bwtc_b200 as bw

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    from bwtc_b200 import sharding
    bound_cpus = sharding.bind_host_to_gpu(local_rank) if world > 1 else 0  # NUMA-local staging buffers and workers
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    nb, n = BLOCKS_PER_STEP, BLOCK_BYTES
    # synthetic input: different blocks on every rank (weak scaling: per-GPU work fixed)
    host_in = [torch.empty(n, dtype=torch.uint8).pin_memory() for _ in range(nb)]
    host_out = [torch.empty(n, dtype=torch.uint8).pin_memory() for _ in range(nb)]
    # block i of the global stream -> rank i mod G (bwtc_b200/sharding.py); seeds follow the GLOBAL block index
    mine = sharding.blocks_for_rank(nb * world, rank, world)
    assert len(mine) == nb
    with ThreadPoolExecutor(max_workers=min(nb, os.cpu_count() or 1)) as ex:
        list(ex.map(lambda j: bw.generate(KIND, n, seed=1000 + mine[j], out=host_in[j].numpy()), range(nb)))
    dev_in = [t.to(dev) for t in host_in]
    dev_out = [torch.empty_like(t) for t in dev_in]
    torch.cuda.synchronize()

    if args.depth <= 0:
        args.depth = 6  # in-flight blocks per GPU; waiting workers sleep, so this no longer depends on the host core count
    pipe = bw.Pipeline(n, depth=args.depth, device=local_rank)
    sizes = [n] * nb
    d_in = [t.data_ptr() for t in dev_in]
    d_out = [t.data_ptr() for t in dev_out]
    h_in = [t.data_ptr() for t in host_in]
    h_out = [t.data_ptr() for t in host_out]

    # ---- value: device-resident inputs/outputs, CUDA events over every pipeline stream
    for _ in range(args.warmup):
        pipe.run_ptrs(d_in, d_out, sizes, STARTS, on_device=True)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches = 0
    pipe.timing_begin()
    t0 = time.perf_counter()
    last_stats = None
    for _ in range(args.steps):
        LF, nLF, freqs, stats = pipe.run_ptrs(d_in, d_out, sizes, STARTS, on_device=True)
        launches += sum(s["kernel_launches"] for s in stats)
        last_stats = stats
    ms_dev = pipe.timing_end()
    barrier()
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, "_rank%d" % rank if world > 1 else "", dev_out, LF, nLF, freqs)

    # ---- e2e: host (pinned) buffers through the same C-ABI call, H2D + D2H inside the timed region
    for _ in range(max(1, args.warmup // 2)):
        pipe.run_ptrs(h_in, h_out, sizes, STARTS, on_device=False)
    barrier()
    t1 = time.perf_counter()
    for _ in range(args.steps):
        LFh, nLFh, freqsh, _ = pipe.run_ptrs(h_in, h_out, sizes, STARTS, on_device=False)
    barrier()
    e2e_s = time.perf_counter() - t1
    # the two paths must agree (device result vs host result of the same blocks)
    assert (LFh == LF).all() and (freqsh == freqs).all()
    assert torch.equal(dev_out[0].cpu(), host_out[0]) and torch.equal(dev_out[-1].cpu(), host_out[-1])

    # ---- e2e with PAGEABLE host buffers (malloc'ed, like PrecompressorBlock.cpp:37-49): pinned staging ring inside the engine
    page_in = [t.numpy().copy() for t in host_in]
    page_out = [np.empty(n, np.uint8) for _ in range(nb)]
    p_in, p_out = [a.ctypes.data for a in page_in], [a.ctypes.data for a in page_out]
    pipe.run_ptrs(p_in, p_out, sizes, STARTS, on_device=False, want_stats=False)
    barrier()
    t2 = time.perf_counter()
    psteps = max(1, args.steps // 2)
    for _ in range(psteps):
        LFp, _, freqsp, _ = pipe.run_ptrs(p_in, p_out, sizes, STARTS, on_device=False, want_stats=False)
    barrier()
    page_s = time.perf_counter() - t2
    assert (LFp == LF).all() and np.array_equal(page_out[0], host_out[0].numpy()) and np.array_equal(page_out[-1], host_out[-1].numpy())

    # ---- max over ranks
    times = torch.tensor([ms_dev, e2e_s * 1e3, wall * 1e3, page_s * 1e3], dtype=torch.float64, device=dev)
    ltot = torch.tensor([launches], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
        dist.all_reduce(ltot, op=dist.ReduceOp.SUM)
    ms_dev_max, e2e_ms_max, wall_ms_max, page_ms_max = [float(v) for v in times.tolist()]
    total_bytes = world * args.steps * nb * n
    value = total_bytes / 1e6 / (ms_dev_max / 1e3)
    e2e_value = total_bytes / 1e6 / (e2e_ms_max / 1e3)
    page_value = world * psteps * nb * n / 1e6 / (page_ms_max / 1e3)
    pipe.close()
    del dev_in, dev_out, page_in, page_out
    torch.cuda.empty_cache()

    # ---- copy-only ceiling of this box at this N: every rank moves 32 MiB pinned buffers in and out concurrently, no
    # kernels.  The end-to-end figure moves n bytes in and n bytes out per block, so this bounds it from above.
    ceiling = None
    try:
        s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
        cb_d = [torch.empty(n, dtype=torch.uint8, device=dev) for _ in range(4)]
        cb_e = [torch.empty(n, dtype=torch.uint8, device=dev) for _ in range(4)]
        for rep in range(2):
            barrier()
            tcp = time.perf_counter()
            iters = 24
            for it in range(iters):
                with torch.cuda.stream(s_in):
                    cb_d[it % 4].copy_(host_in[it % nb], non_blocking=True)
                with torch.cuda.stream(s_out):
                    host_out[it % nb].copy_(cb_e[it % 4], non_blocking=True)
            torch.cuda.synchronize()
            dtc = time.perf_counter() - tcp
        tc_t = torch.tensor([dtc], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tc_t, op=dist.ReduceOp.MAX)
        ceiling = {"value": world * iters * n / 1e6 / float(tc_t.item()), "unit": "MB/s per direction, both directions concurrently",
                   "note": "pinned 32 MiB buffers, two copy streams per GPU, no kernels, max over ranks: the upper bound of `e2e` "
                           "on this box at this GPU count (host memory / PCIe root)"}
        del cb_d, cb_e
    except Exception as e:  # noqa: BLE001
        ceiling = {"error": str(e)}

    # ---- BASELINE config 5 end to end: PipelinedCompressor with CPU Huffman coding overlapped (every rank, own stream)
    comp = None
    if not args.no_compress:
        barrier()
        tc0 = time.perf_counter()
        mine_c = run_compress_leg(local_rank, world, rank)
        barrier()
        tc = time.perf_counter() - tc0
        vals = torch.tensor([float(mine_c.get("seconds", 1e9)), float(mine_c.get("input_bytes", 0)),
                             float(mine_c.get("compressed_bytes", 0)), float(mine_c.get("encoder_busy_core_s", 0))],
                            dtype=torch.float64, device=dev)
        mx = vals.clone()
        if world > 1:
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            dist.all_reduce(vals, op=dist.ReduceOp.SUM)
        if "error" in mine_c:
            comp = mine_c
        else:
            comp = {"value": float(vals[1]) / 1e6 / float(mx[0]), "unit": "MB/s of input (whole job)",
                    "workload": "%d x 32 MiB Markov blocks per rank from host memory -> bwtc::PipelinedCompressor(BWT 'c' on the GPU, "
                                "coder 'H' = the reference's HuffmanEncoder on %d host threads per rank) -> .bwtc bytes"
                                % (mine_c["input_bytes"] // BLOCK_BYTES, mine_c["encoder_threads"]),
                    "seconds_max_over_ranks": float(mx[0]), "input_bytes": float(vals[1]), "compressed_bytes": float(vals[2]),
                    "encoder_threads_per_rank": mine_c["encoder_threads"], "host_cores": os.cpu_count(),
                    "encoder_busy_core_s": float(vals[3]),
                    "coder_mb_per_core_s": float(vals[1]) / 1e6 / max(float(vals[3]), 1e-9),
                    "gpu_pipeline_depth": mine_c["pipeline_depth"], "leg_wall_s": tc,
                    "reader_busy_s_rank0": mine_c.get("reader_busy_s"), "writer_busy_s_rank0": mine_c.get("writer_busy_s"),
                    "first_pass_seconds_rank0": mine_c.get("first_pass_seconds"),
                    "note": "bound by the CPU entropy coder (MB per core-second above x cores); the GPU BWT stage runs "
                            "ahead of it (see `value` / `e2e`)"}

    line = None
    if rank == 0:
        peak, peak_src = _peaks()
        # ---- roofline leg: one context, one stream, every radix pass bracketed by CUDA events
        dev_in = [t.to(dev) for t in host_in[:4]]
        dev_out = [torch.empty_like(t) for t in dev_in]
        ctx = bw.CudaContext(n, device=local_rank)
        ctx.set_timing(1)
        LF1 = np.zeros(STARTS, np.uint32)
        sort_ms = sort_bytes = sort_launches = all_sort_ms = 0
        gpu_ms = alg_bytes = 0
        ROOF_WARM, ROOF_TIMED = 4, 48  # the GPU idled while the context was allocated: warm up, then average 384 launches
        rsampler = ClockSampler(local_rank)
        for i in range(ROOF_WARM + ROOF_TIMED):
            if i == ROOF_WARM:
                rsampler.start()
            ctx.bwt_block_device(dev_in[i % 4].data_ptr(), dev_out[i % 4].data_ptr(), n, LF1, None)
            if i < ROOF_WARM:
                continue  # warm-up
            st = ctx.stats()
            sort_ms += st["sort0_ms"]            # round-0 passes: every launch sorts all N records of the block
            sort_bytes += st["sort0_bytes"]
            sort_launches += st["sort0_launches"]
            all_sort_ms += st["sort_ms"]
            gpu_ms += st["gpu_ms"]
            alg_bytes += st["algorithmic_bytes"]
        roof_clocks = rsampler.stop()
        ctx.close()
        del dev_in, dev_out
        achieved = sort_bytes / 1e9 / (sort_ms / 1e3)
        traffic, traffic_src = None, None
        for tp in ("r02_radix_pass_traffic.json", "r01_radix_pass_traffic.json"):
            tp = os.path.join(ROOT, "profiles", tp)
            if os.path.exists(tp):
                try:
                    tj = json.load(open(tp))
                    traffic = tj.get("dram_bytes_per_launch")
                    traffic_src = "offline `ncu --set full` capture %s (kernel source at commit %s)" % (
                        os.path.basename(tp), tj.get("commit", "unrecorded"))
                    break
                except Exception:
                    traffic = None
        st0 = last_stats[0]
        roofline = {"bound": "hbm", "kernel": "k_radix_pass<u64,256,16> (one 8-bit LSD digit pass over (key, suffix id) records)",
                    "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "peak_source": peak_src, "traffic": traffic, "traffic_source": traffic_src,
                    "bytes_per_launch": sort_bytes / max(sort_launches, 1),
                    "avg_launch_ms": sort_ms / max(sort_launches, 1), "launches_timed": sort_launches, "clocks_during_leg": roof_clocks,
                    "share_of_block_gpu_time": all_sort_ms / gpu_ms,
                    "launch_shape": "the 8 round-0 digit passes: 33 554 433 records of (u64 key, u32 id) per launch "
                                    "(later rounds of this workload are sort-free: k_seg_round / k_small_rounds)",
                    "whole_block": {"algorithmic_bytes_per_input_byte": alg_bytes / float(ROOF_TIMED * n),
                                    "achieved_gbs": alg_bytes / 1e9 / (gpu_ms / 1e3),
                                    "frac_of_peak": alg_bytes / 1e9 / (gpu_ms / 1e3) / peak,
                                    "frac_of_nominal_8000": alg_bytes / 1e9 / (gpu_ms / 1e3) / 8000.0,
                                    "ms_per_block_single_stream": gpu_ms / ROOF_TIMED,
                                    "rounds": st0["rounds"], "live": st0["live"], "passes": st0["passes"],
                                    "chars_round0": st0["chars_round0"], "key_bytes_round0": st0["key_bytes_round0"]}}
        # ---- one entry per BASELINE.json config (device-resident through the pipeline + pinned host figure)
        configs = []
        if world == 1 and not args.no_configs:
            plan = [("1: Markov 16 MiB, 1 MiB blocks (batched 32 per device-side sort)", "markov", 1 << 20, 64, 3, 4),
                    ("2: DNA (4 symbols), 64 MiB blocks", "dna", 64 << 20, 6, 3, 2),
                    ("3: repetitive (4 KiB seed tiled, 0.1% mutations), 16 MiB blocks", "repetitive", 16 << 20, 6, 3, 2),
                    ("4: uniform random bytes, 256 MiB blocks", "random", 256 << 20, 3, 2, 2),
                    ("5: Markov stream, 32 MiB blocks (the headline workload)", "markov", 32 << 20, 8, 4, 3)]
            for name, kind, nbytes, nblk, dpt, reps in plan:
                try:
                    r = measure_workload(bw, torch, dev, local_rank, kind, nbytes, nblk, dpt, reps, seed0=7000)
                    s0 = r["stats0"]
                    rr = s0["rounds"]
                    configs.append({"config": name, "value": r["value"], "e2e": r["e2e"], "unit": "MB/s", "blocks": nblk,
                                    "pipeline_depth": dpt, "rounds": rr, "live_over_N": [round(v / s0["n_suffixes"], 4) for v in s0["live"][:rr]],
                                    "passes": s0["passes"][:rr], "chars_round0": s0["chars_round0"], "key_bytes_round0": s0["key_bytes_round0"],
                                    "algorithmic_bytes_per_input_byte": r["alg_bytes_per_input_byte"],
                                    "whole_block_gbs": r["alg_bytes_per_input_byte"] * r["value"] / 1e3,
                                    "whole_block_frac_of_peak": r["alg_bytes_per_input_byte"] * r["value"] / 1e3 / peak,
                                    "kernel_launches_per_step": r["launches_per_step"]})
                except Exception as e:  # noqa: BLE001
                    configs.append({"config": name, "error": str(e)})
                torch.cuda.empty_cache()
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            try:
                cpu = cpu_baseline_sample(os.cpu_count() or 1)
            except Exception as e:  # noqa: BLE001
                cpu = {"value": None, "unit": "MB/s", "cores": 0, "kind": "reference", "sample": "unavailable: %s" % e}
        line = {"metric": METRIC, "value": value, "unit": "MB/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_dev_max / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": DTYPE,
                "data": "synthetic",
                "config": make_config(
                    pipeline_depth=args.depth,
                    l2="the same 16 device-resident blocks (512 MiB) per GPU are re-transformed every step; each in-flight block "
                       "streams through ~1.3 GB of scratch, far larger than the 126 MB L2 (no flush needed)",
                    host="rank 0 bound to %s host cores (NVML affinity of its GPU)" % (bound_cpus if bound_cpus else "all"),
                    lookback_tile_ids="tickets (watchdog fallback)" if any(s["flags"] & 1 for s in last_stats) else "block index",
                    host_wait=os.environ.get("BWTC_WAIT_MODE", "adaptive poll (default)")),
                "e2e": {"value": e2e_value, "unit": "MB/s", "h2d_bytes_per_step": nb * n,
                        "d2h_bytes_per_step": nb * (n + 4 * STARTS + 256 * 4)},
                "e2e_pageable": {"value": page_value, "unit": "MB/s",
                                 "note": "malloc'ed host buffers (what a bwtc PrecompressorBlock is): staged through the engine's "
                                         "pinned ring, memcpy + DMA overlapped on copy streams"},
                "e2e_copy_ceiling": ceiling,
                "gpu_launches": int(ltot.item()),
                "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu, "configs": configs, "compress_e2e": comp,
                "wall_ms_per_step": wall_ms_max / args.steps}
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(line), flush=True)
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--depth", type=int, default=0, help="in-flight blocks (contexts + sleeping host workers) per GPU; 0 = 6")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true")
    ap.add_argument("--no-compress", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the last timed step's outputs (sampled BWT bytes, LFpowers, freqs) as DIR/<name>.npy, "
                         "or DIR/<name>_rank<r>.npy for each rank with several GPUs; GPU path only")
    ap.add_argument("--leg", default="")
    ap.add_argument("--leg-device", type=int, default=0)
    ap.add_argument("--leg-blocks", type=int, default=32)
    ap.add_argument("--leg-threads", type=int, default=0)
    ap.add_argument("--leg-depth", type=int, default=4)
    ap.add_argument("--leg-seed", type=int, default=5000)
    args = ap.parse_args()
    if args.leg == "compress":
        return compress_leg(args.leg_device, args.leg_blocks, args.leg_threads or (os.cpu_count() or 1), args.leg_depth, args.leg_seed)
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the GPU path's outputs; --impl reference has none to write")
        return main_reference(args)
    return main_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
