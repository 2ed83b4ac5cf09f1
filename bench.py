#!/usr/bin/env python
"""bench.py -- RS(k,m) encode+decode GiB/s on 1 MiB blocks (BASELINE.json's metric).

One step = one pass of the hot path over one batch: RS(10,4) ENCODE of `blocks` x 1 MiB
synthetic blocks (BASELINE config 2) followed by RS(10,4) RECONSTRUCT of the same number of
stripes with 4 random erasures each (config 3), device-resident, through the C ABI
(libgarage_ec.so).  value = payload bytes (2 x blocks x 1 MiB per step, per GPU, all GPUs
summed) / time.  The K timed steps replay a CUDA graph of one captured step (same library calls,
host out of the way); an eager pass of the same K steps just before it carries the per-kernel
CUDA events the roofline is computed from.  `e2e` repeats the step through the HOST-buffer entry
points (pinned host memory, H2D + D2H inside the timed region).  The CPU arm (`cpu_baseline`, `--impl
reference`) times oracle/rs_simd.c -- the reference itself has no RS code (SURVEY.md 0.1).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR writes what the last timed step returned (see dump_outputs) as float32 .npy files;
the inputs depend only on the arguments, so two builds can be compared file for file.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CPU_KEYS = ("value", "unit", "cores", "kind", "sample", "isa", "encode_gibs", "decode_gibs", "blocks", "per_thread_gibs", "host")
METRIC = "RS(k,m) encode+decode GiB/s on 1 MiB blocks; % HBM roofline @1/2/4/8 GPU"
SEED = 0x6761726167650010
B = 1 << 20
GIB = float(1 << 30)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--m", type=int, default=4)
    ap.add_argument("--blocks", type=int, default=0,
                    help="1 MiB blocks per GPU per pass (0 = 4096, BASELINE configs 2+3; 8192 at 8 GPUs = the 65 536 "
                         "blocks of config 4)")
    ap.add_argument("--e2e-blocks", type=int, default=0, help="blocks per e2e step (0 = --blocks)")
    ap.add_argument("--cpu-blocks", type=int, default=0,
                    help="blocks per CPU-arm step (0 = auto: max(512, 16 per host thread), capped at 4096 -- "
                         "with fewer blocks per thread the pthread fan-out dominates and the CPU looks slower than it is)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-sweep", action="store_true", help="skip the config-5 scrub/repair sweep extra")
    ap.add_argument("--sweep-stripes", type=int, default=4096, help="stripes per code per GPU in the sweep extra")
    ap.add_argument("--sweep-e2e-stripes", type=int, default=512,
                    help="stripes per code per GPU in the HOST-buffer (end-to-end) sweep companion")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write rank 0's outputs of the last step to DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs records the GPU path (--impl ours)")
    if a.blocks <= 0:
        a.blocks = 8192 if int(os.environ.get("WORLD_SIZE", "1")) >= 8 else 4096
    return a


# ------------------------------------------------------------------ helpers
def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy read+write)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic():
    """dram bytes per launch of the streaming kernels from the COMMITTED ncu capture (profiles/, not
    measured in this run: ncu replays every kernel ~40 times and must not run inside a bench), or {}"""
    p = os.path.join(ROOT, "profiles", "dominant_kernel_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return {}
    return {}


def host_info():
    """what the CPU arm actually ran on: the ratio GPU/CPU swings with it (round 1: the same code did
    20 GiB/s on one box and 100 GiB/s on another, both reporting 128 threads)"""
    info = {"affinity_cpus": len(os.sched_getaffinity(0)), "logical_cpus": os.cpu_count()}
    try:
        cores, models, mhz = set(), set(), []
        phys = core = None
        for line in open("/proc/cpuinfo"):
            if line.startswith("physical id"):
                phys = line.split(":")[1].strip()
            elif line.startswith("core id"):
                core = line.split(":")[1].strip()
                cores.add((phys, core))
            elif line.startswith("model name"):
                models.add(line.split(":", 1)[1].strip())
            elif line.startswith("cpu MHz"):
                mhz.append(float(line.split(":")[1]))
        info["physical_cores"] = len(cores) or None
        info["sockets"] = len({c[0] for c in cores}) or None
        info["cpu_model"] = sorted(models)[0] if models else None
        info["cpu_mhz_now_median"] = statistics.median(mhz) if mhz else None
    except Exception:  # noqa: BLE001
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            info["cgroup_cpu_max"] = open(path).read().strip()
            break
        except Exception:  # noqa: BLE001
            continue
    try:
        info["numa_nodes"] = len([d for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit()])
    except Exception:  # noqa: BLE001
        pass
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemTotal"):
                info["mem_total_gib"] = round(int(line.split()[1]) / 2**20, 1)
    except Exception:  # noqa: BLE001
        pass
    return info


class ClockSampler:
    """SM clock + throttle reasons of one GPU, sampled by the MAIN thread after all timed steps have
    been enqueued and until their end event completes: every sample is taken under load inside the
    timed region, and no NVML call competes with a kernel launch for the driver (a background
    sampler thread did: one run showed 0.7 ms of launch gaps per 2 ms step)."""

    def __init__(self, index):
        self.index, self.samples, self.reasons = index, [], set()
        self.max_mhz, self.err, self.raw_mask, self.power_w = None, None, 0, []
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # noqa: BLE001
            self.nv, self.err = None, repr(e)

    def sample(self):
        nv = self.nv
        if not nv:
            return
        names = {"gpu_idle": 0x1, "applications_clocks_setting": 0x2, "sw_power_cap": 0x4, "hw_slowdown": 0x8,
                 "sync_boost": 0x10, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
                 "hw_power_brake": 0x80, "display_clock_setting": 0x100}
        try:
            self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
            try:
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            except Exception:  # older binding name
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            self.raw_mask |= int(r)
            for n, bit in names.items():
                if r & bit:
                    self.reasons.add(n)
            try:
                self.power_w.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            except Exception:  # noqa: BLE001
                pass
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)

    def sample_until(self, end_event, max_samples=200):
        """poll while the GPU is still inside the timed region"""
        while not end_event.query() and len(self.samples) < max_samples:
            self.sample()
            time.sleep(0.004)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "error": self.err or "no samples"}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "reasons_raw_mask": self.raw_mask, "samples": len(self.samples),
                "sm_mhz_min": min(self.samples), "sm_mhz_max_seen": max(self.samples),
                "power_w_max": max(self.power_w) if self.power_w else None,
                "note": "sampled by NVML while the timed steps execute; an HBM-bound kernel does not hold the SM "
                        "clock at its maximum (DVFS), no clock lock is set by this program"}


def alg_bytes_per_pass(k, m, e, n, L):
    """ALGORITHMIC bytes (SURVEY.md 8(d)): encode reads k*L, writes m*L per stripe; reconstruct
    with e erasures reads k*L, writes e*L.  (k*L = B up to the <k bytes of tail padding.)"""
    return n * (k + m) * L, n * (k + e) * L


DUMP_SHARD_BYTES = 56_000_000  # float32 budget of the two shard samples; with the rest the dump stays under 64 MB


def dump_outputs(out_dir, parity, shards, present, status, k, m, n, L, stride):
    """Write what the step's caller receives, as float32 .npy files: `encode_parity` and `reconstruct_shards`
    (the rebuilt erased shards, in shard order) of a fixed seeded sample of stripes `sample_stripes`, each
    shard cut to its length L (and, if one stripe alone would not fit the budget, to its first bytes), and
    `reconstruct_status` of every stripe."""
    import torch

    s = min(n, 16, max(1, DUMP_SHARD_BYTES // (2 * m * L * 4)))
    w = min(L, DUMP_SHARD_BYTES // (2 * m * s * 4))
    idx = np.sort(np.random.default_rng(SEED).choice(n, s, replace=False))
    it = torch.from_numpy(idx).to(parity.device)
    erased = (present[torch.from_numpy(idx)] == 0).to(parity.device)
    out = {
        "sample_stripes": idx,
        "encode_parity": parity.view(n, m, stride)[it, :, :w],
        "reconstruct_shards": shards.view(n, k + m, stride)[it][erased].view(s, m, stride)[:, :, :w],
        "reconstruct_status": status,
    }
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        a = a.cpu().numpy() if hasattr(a, "cpu") else a
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))


# ------------------------------------------------------------------ CPU arm (oracle port)
def cpu_arm(k, m, nblocks, steps, warmup, budget_s=None):
    """times oracle/rs_simd.c (all host threads) on `nblocks` x 1 MiB: encode + reconstruct
    with m erasures per stripe.  Returns dict with GiB/s (same payload definition)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O

    L = O.lib().rs_oracle_shard_len(B, k)
    stride = (L + 127) // 128 * 128
    tot = k + m
    threads = O.lib().rs_simd_max_threads()
    if nblocks <= 0:
        nblocks = min(4096, max(512, 16 * threads))
    P = O.build_matrix(k, m, 0)
    shards = np.zeros((nblocks, tot, stride), dtype=np.uint8)
    for s in range(nblocks):
        blk = O.fill_random(B, SEED, s * B)
        shards[s, :k] = O.split_block(blk, k, stride).reshape(k, stride)
    data = np.ascontiguousarray(shards[:, :k]).reshape(-1)
    lens = np.full(nblocks, L, dtype=np.uint32)
    rng = np.random.default_rng(1234)
    present = np.ones((nblocks, tot), dtype=np.uint8)
    for s in range(nblocks):
        present[s, rng.choice(tot, m, replace=False)] = 0
    par = O.encode(k, m, P, data, stride, nblocks, lens, simd=True)
    shards[:, k:] = par.reshape(nblocks, m, stride)
    # NUMA: place every stripe on the memory node of the worker thread that processes it
    data = O.numa_local_copy(data, k * stride, nblocks, threads)
    par = O.numa_local_copy(par, m * stride, nblocks, threads)
    flat = O.numa_local_copy(shards.reshape(-1), tot * stride, nblocks, threads)
    del shards
    t_enc = t_dec = 0.0
    done = 0
    t_start = time.perf_counter()
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        O.lib().rs_simd_encode(k, m, P.ctypes.data, data.ctypes.data, par.ctypes.data, lens.ctypes.data,
                               stride, nblocks, threads)
        t1 = time.perf_counter()
        O.lib().rs_simd_reconstruct(k, m, P.ctypes.data, flat.ctypes.data, present.ctypes.data, None,
                                    lens.ctypes.data, stride, nblocks, threads)
        t2 = time.perf_counter()
        if it >= warmup:
            t_enc += t1 - t0
            t_dec += t2 - t1
            done += 1
        if budget_s and done >= 1 and time.perf_counter() - t_start > budget_s:
            break
    payload = nblocks * B * done
    return {
        "value": 2 * payload / (t_enc + t_dec) / GIB, "unit": "GiB/s", "cores": threads, "kind": "port",
        "blocks": nblocks, "per_thread_gibs": 2 * payload / (t_enc + t_dec) / GIB / max(threads, 1), "host": host_info(),
        "isa": O.lib().rs_simd_isa().decode(),
        "encode_gibs": payload / t_enc / GIB, "decode_gibs": payload / t_dec / GIB,
        "sample": "%d x 1 MiB blocks RS(%d,%d): encode + reconstruct(%d erasures/stripe), %d timed passes, "
                  "oracle/rs_simd.c (%s) on %d threads" % (nblocks, k, m, m, done, O.lib().rs_simd_isa().decode(), threads),
        "ms_per_step": 1e3 * (t_enc + t_dec) / done, "steps": done,
    }


def run_reference(args, rank, world):
    if rank != 0:
        return
    r = cpu_arm(args.k, args.m, args.cpu_blocks, args.steps, args.warmup)
    nref = r["blocks"]
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": "GiB/s", "n_gpus": args.gpus,
        "steps": r["steps"], "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": "BASELINE configs 2+3: RS(%d,%d) encode + reconstruct(%d erasures/stripe) of 1 MiB blocks; "
                               "each step is a bounded sample of %d blocks of that workload (the GPU arm runs %d per "
                               "GPU); GiB/s is size-independent at these sizes" % (args.k, args.m, args.m, nref, args.blocks),
                   "sample_blocks_per_step": nref,
                   "note": "the reference (garage v1.2.0) has no RS code; this is the CPU oracle port oracle/rs_simd.c"},
        "cpu_baseline": {k: r[k] for k in CPU_KEYS},
        "e2e": {"value": r["value"], "unit": "GiB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------ GPU arm
def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist

    import garage_b200 as G

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    k, m, n = args.k, args.m, args.blocks
    tot = k + m

    # rank 0 owns the generator matrix and the block ranges; one NCCL broadcast (SURVEY.md 8(e))
    if world > 1:
        from garage_b200 import dist as D

        P0 = ranges0 = None
        if rank == 0:
            with G.GarageEc(local_rank, k, m, G.VANDERMONDE) as tmp:
                P0 = tmp.matrix()
            ranges0 = D.partition_blocks(n * world, world)
        P, ranges = D.broadcast_control(k, m, P0, ranges0, dev, dist)
        first_block = ranges[rank][0]
        assert ranges[rank][1] - first_block == n
        enc = G.GarageEc(local_rank, k, m, matrix=P)
        dec = G.GarageEc(local_rank, k, m, matrix=P)
    else:
        first_block = 0
        enc = G.GarageEc(local_rank, k, m, G.VANDERMONDE)
        dec = G.GarageEc(local_rank, k, m, G.VANDERMONDE)

    # this rank's host threads and pinned buffers live on the GPU's NUMA node (8-GPU hosts: 4 GPUs per socket)
    bound = enc.bind_thread()
    L = enc.shard_len(B)
    stride = enc.stride_for(L)
    # device-resident inputs (inputs >> L2: %.1f GB) generated from the shared counter stream
    shards = torch.zeros(n * tot * stride, dtype=torch.uint8, device=dev)
    sh3 = shards.view(n, tot, stride)
    data = torch.empty(n * k * stride, dtype=torch.uint8, device=dev)
    enc.fill_random(data, n * k * stride, SEED, first_block * k * stride)
    d3 = data.view(n, k, stride)
    d3[:, :, L:] = 0
    if k * L > B:
        d3[:, k - 1, L - (k * L - B):] = 0
    lens = torch.full((n,), L, dtype=torch.int32, device=dev)
    parity = torch.zeros(n * m * stride, dtype=torch.uint8, device=dev)
    enc.encode(data, parity, stride, n, shard_len=lens)
    sh3[:, :k] = d3
    sh3[:, k:] = parity.view(n, m, stride)
    # digest of the stripes the timed work must reproduce: the blake2sum of every shard, computed on the
    # device by the library (garage_ec_shard_sums) -- 32 bytes per shard, compared after every timed region
    sums_ref = torch.zeros(n * tot * 32, dtype=torch.uint8, device=dev)
    enc.shard_sums(shards, sums_ref, stride, n, tot, shard_len=lens)
    sums_now = torch.zeros_like(sums_ref)

    def check_results(tag):
        assert int(status.abs().sum()) == 0, tag
        enc.shard_sums(shards, sums_now, stride, n, tot, shard_len=lens)
        assert torch.equal(sums_now, sums_ref), "reconstruct output differs from the original stripes (%s)" % tag
        assert torch.equal(parity, sh3[:, k:].reshape(-1)), "encode output differs (%s)" % tag

    # parity of sampled stripes against the CPU oracle (the checker; scalar normative arithmetic)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O

    oracle_checked = []
    Pm = O.build_matrix(k, m, 0)
    for s_i in sorted({0, 1, n // 3, n // 2, n - 2, n - 1}):
        dd = d3[s_i].cpu().numpy().reshape(-1)
        want = O.encode(k, m, Pm, dd, stride, 1, np.array([L], dtype=np.uint32))
        got = parity.view(n, m, stride)[s_i].cpu().numpy().reshape(-1)
        assert np.array_equal(got, want), "encode differs from the CPU oracle at stripe %d" % s_i
        oracle_checked.append(first_block + s_i)
    g = torch.Generator().manual_seed(1234 + rank)
    erased = torch.rand(n, tot, generator=g).argsort(dim=1)[:, :m]
    present = torch.ones(n, tot, dtype=torch.uint8)
    present.scatter_(1, erased, 0)
    present_d = present.to(dev)
    sh3[~present_d.bool()] = 0
    status = torch.zeros(n, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()

    def step():
        enc.encode(data, parity, stride, n, shard_len=lens)
        dec.reconstruct(shards, present_d, stride, n, status=status, shard_len=lens)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()

    # ---- the timed region of the headline: K steps with the host out of the way.
    # One step (the same two library calls) is captured into a CUDA graph -- the DEVICE entry points
    # only enqueue kernels and stream-ordered allocations -- and replayed K times; on the eager pass
    # the Python/ctypes/driver path left 30-140 us of launch gaps per 1.9 ms step depending on the
    # host.  If capture is not possible the steps run eagerly (without the per-kernel events).
    g_step, graph_note = None, None
    try:
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            step()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize()
        g_step = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g_step):
            step()
        for _ in range(3):
            g_step.replay()
        torch.cuda.synchronize()
    except Exception as e:  # noqa: BLE001
        g_step, graph_note = None, "graph capture failed (%r): timed steps ran eagerly" % (e,)
    run_step = g_step.replay if g_step is not None else step
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    clk = ClockSampler(local_rank)
    barrier()
    ev0.record()
    for _ in range(args.steps):
        run_step()
    ev1.record()
    clk.sample_until(ev1)  # the host is ahead of the GPU: these samples fall inside the timed region
    barrier()
    ms = ev0.elapsed_time(ev1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, parity, shards, present, status, k, m, n, L, stride)
    # parity of the timed work: reconstructed shards == originals (per-shard blake2sums), parity unchanged
    check_results("graph-replayed timed region")
    graph_used = g_step is not None
    del g_step

    # ---- second pass (eager, per-kernel CUDA events recorded by the library on the launch stream):
    # the kernel durations the roofline is computed from, same K steps, same inputs.  A short pause
    # and fresh warm-up steps first: straight after ~100 ms of sustained load the SM/memory clocks
    # of some boxes sag (DVFS, no throttle reason reported) and the second region measured 2-4 % slow.
    time.sleep(1.0)
    for _ in range(3):
        step()
    barrier()
    enc.set_timing(True)
    dec.set_timing(True)
    enc.timing_read(), dec.timing_read()
    l0 = enc.launch_count() + dec.launch_count()
    ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ea.record()
    for _ in range(args.steps):
        step()
    eb.record()
    barrier()
    eager_ms = ea.elapsed_time(eb)
    launches = enc.launch_count() + dec.launch_count() - l0
    enc_ms, enc_n = enc.timing_read()
    dec_ms, dec_n = dec.timing_read()
    check_results("eager pass")
    # ---- scrub-verify of the same stripes (third streaming kernel; not part of the step): K launches
    mm = torch.zeros(n, dtype=torch.int32, device=dev)
    time.sleep(1.0)  # same pause + fresh warm-up as before the eager pass (clocks sag after sustained load)
    for _ in range(3):
        enc.verify(shards, mm, stride, n, shard_len=lens)
    barrier()
    enc.timing_read()
    for _ in range(args.steps):
        enc.verify(shards, mm, stride, n, shard_len=lens)
    barrier()
    ver_ms, ver_n = enc.timing_read()
    enc.set_timing(False)
    dec.set_timing(False)
    assert int(mm.abs().sum()) == 0, "verify flagged a clean stripe"

    step_mode = {"mode": "cuda-graph replay of one captured step" if graph_used else "eager",
                 "eager_ms_per_step_with_kernel_events": eager_ms / args.steps, "note": graph_note}

    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    lt = torch.tensor([launches], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(lt, op=dist.ReduceOp.SUM)
    ms_max = float(t.item())
    payload_per_step = 2 * n * B * world
    value = payload_per_step * args.steps / (ms_max * 1e-3) / GIB

    # ---- what a plain device copy reaches on THIS GPU right now (SURVEY.md 8(d): report the
    # practically achievable ceiling measured in the same run next to the driver's figure) -----
    cp_n = min(1 << 30, shards.numel() // 2 // 4096 * 4096)
    cp_src = shards[:cp_n]
    cp_dst = shards[cp_n: 2 * cp_n]
    snap = cp_dst.clone()
    best = None
    for _ in range(6):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        cp_dst.copy_(cp_src)
        b.record()
        torch.cuda.synchronize()
        t_ms = a.elapsed_time(b)
        best = t_ms if best is None else min(best, t_ms)
    cp_dst.copy_(snap)
    del snap
    copy_gbs_now = 2 * cp_n / (best * 1e-3) / 1e9

    # ---- roofline: the three streaming kernels, the time-dominant one of the step on top -----
    peak, peak_src = peaks()
    enc_alg, dec_alg = alg_bytes_per_pass(k, m, m, n, L)
    ver_alg = enc_alg  # verify reads k data + m parity shards
    enc_avg_ms = enc_ms / max(enc_n, 1)
    dec_avg_ms = dec_ms / max(dec_n, 1)
    ver_avg_ms = ver_ms / max(ver_n, 1)
    tr = ncu_traffic()

    def kern(name, alg, avg_ms, launches, key):
        ach = alg / (avg_ms * 1e-3) / 1e9
        t = (tr.get("kernels") or {}).get(key) or {}
        return {"kernel": name, "achieved": ach, "frac": ach / peak, "avg_launch_ms": avg_ms, "launches_timed": launches,
                "algorithmic_bytes_per_launch": alg, "frac_of_copy_this_run": ach / copy_gbs_now,
                "traffic": t.get("dram_bytes_per_launch"), "traffic_at_blocks": t.get("blocks")}

    kernels = {
        "encode": kern("rs_apply_kernel<%d, encode>" % k, enc_alg, enc_avg_ms, enc_n, "encode"),
        "reconstruct": kern("rs_apply_kernel<%d, reconstruct>" % k, dec_alg, dec_avg_ms, dec_n, "reconstruct"),
        "verify": kern("rs_apply_kernel<%d, verify>" % k, ver_alg, ver_avg_ms, ver_n, "verify"),
    }
    step_ms = enc_avg_ms + dec_avg_ms
    kernels["encode"]["share_of_step"] = enc_avg_ms / step_ms
    kernels["reconstruct"]["share_of_step"] = dec_avg_ms / step_ms
    kernels["verify"]["share_of_step"] = None  # scrub kernel: timed in its own K launches, not part of the step
    dom = "encode" if enc_avg_ms >= dec_avg_ms else "reconstruct"
    d = kernels[dom]
    roofline = {
        "bound": "hbm", "kernel": d["kernel"], "achieved": d["achieved"], "peak": peak, "unit": "GB/s", "frac": d["frac"],
        "dominant": "largest share of the step's kernel time (%.1f %%)" % (100 * d["share_of_step"]),
        "peak_source": peak_src, "traffic": d["traffic"],
        "traffic_note": tr.get("note", "no ncu capture committed yet") + " -- read from the committed file "
                        "profiles/dominant_kernel_traffic.json, NOT measured in this run",
        "algorithmic_bytes_per_launch": d["algorithmic_bytes_per_launch"], "avg_launch_ms": d["avg_launch_ms"],
        "launches_timed": d["launches_timed"],
        "timing": "CUDA events recorded by the library around every rs_apply launch, on the launch stream, over the "
                  "eager pass of the same K steps that follows the graph-replayed timed region (verify: K launches of its own)",
        "hbm_read_frac_encode": (n * k * L) / (enc_avg_ms * 1e-3) / 1e9 / peak,
        "copy_gbs_this_run": copy_gbs_now,
        "copy_note": "torch d2d copy of <= 1 GiB (read+write bytes, best of 6) on this GPU in this run; the streaming kernels' "
                     "traffic is 71% reads / 29% writes (verify: reads only), a copy is 50/50",
        "whole_step": {"achieved": (enc_alg + dec_alg) / (ms_max / args.steps * 1e-3) / 1e9,
                       "frac": (enc_alg + dec_alg) / (ms_max / args.steps * 1e-3) / 1e9 / peak,
                       "note": "algorithmic bytes of encode + reconstruct / graph-replayed step time (includes rs_plan_kernel)"},
        "kernels": kernels,
    }

    # ---- e2e: the same step through the HOST-buffer entry points (pinned memory) ------------
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(args, torch, dist, enc, dec, rank, world, dev, shards, data, present, L, stride)

    sweep = None
    if not args.no_sweep:
        del sh3, d3
        torch.cuda.empty_cache()
        sweep = {"workload": "BASELINE config 5: mixed RS(6,3)/RS(10,4) stripes of 1 MiB blocks, 10% corrupted shards, "
                             "detect (per-shard tag) + reconstruct + rewrite through garage_ec_scrub_repair; "
                             "GiB/s = payload bytes healed-or-verified per second, all GPUs"}
        variants = (("device_adler8", 1, False), ("device_blake2", 0, False), ("e2e_host_adler8", 1, True))
        for name, kind, host in variants:
            sw_ms, sw_detail, sw_err = 0.0, None, None
            try:
                sw_ms, sw_detail = run_sweep(args, torch, dist, rank, world, dev, local_rank, kind, host)
            except Exception as e:  # noqa: BLE001  (an extra must never cost the headline line)
                sw_err = repr(e)
            flag = torch.tensor([0.0 if sw_err else 1.0, sw_ms], dtype=torch.float64, device=dev)
            if world > 1:  # every rank reaches these collectives whether or not its sweep worked
                okf = flag[:1].clone()
                dist.all_reduce(okf, op=dist.ReduceOp.MIN)
                dist.all_reduce(flag[1:], op=dist.ReduceOp.MAX)
                flag[0] = okf[0]
            stripes = args.sweep_e2e_stripes if host else args.sweep_stripes
            if float(flag[0]) > 0:
                sweep[name] = {"value": 2 * stripes * B * world / (float(flag[1]) * 1e-3) / GIB, "unit": "GiB/s",
                               "stripes_per_code_per_gpu": stripes,
                               "tag": "adler8 (8 x Adler-32 per shard)" if kind == 1 else "blake2sum per shard",
                               "memory": "pinned host buffers, H2D + D2H inside the timed region (wall clock, max over ranks)"
                                         if host else "device-resident (CUDA events, max over ranks)",
                               "detail_rank0": sw_detail}
            else:
                sweep[name] = {"error": sw_err or "failed on another rank"}
        if "value" in sweep.get("device_adler8", {}):
            sweep["value"], sweep["unit"] = sweep["device_adler8"]["value"], "GiB/s"

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = cpu_arm(k, m, args.cpu_blocks, 1000, 1, budget_s=12.0)
        cpu = {kk: cpu[kk] for kk in CPU_KEYS}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "GiB/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {
                "workload": "BASELINE configs 2+3: RS(%d,%d) encode of %d x 1 MiB blocks + reconstruct of %d stripes "
                            "with %d random erasures each, per GPU, device-resident" % (k, m, n, n, m),
                "blocks_per_gpu": n, "blocks_total": n * world, "shard_len": L, "stride": stride, "matrix": "vandermonde-systematic",
                "l2": "inputs larger than L2 (%.1f GB per pass vs 126 MB), no flush needed" % (enc_alg / 1e9),
                "parallelism": "independent block ranges per GPU, NCCL broadcast of matrix+ranges only" if world > 1 else "1 GPU",
                "reference_arm": "bench.py --impl reference times a bounded sample (see its config.sample_blocks_per_step) of "
                                 "this same workload on the host cores; GiB/s is size-independent at these sizes",
                "rank0_thread_bound_to_gpu_numa_node": bool(bound),
                "timed_region": "K steps = K replays of a CUDA graph holding one step's library calls (garage_ec_encode + "
                                "garage_ec_reconstruct, DEVICE mode): every replay re-executes all kernels on the same "
                                "device-resident inputs; per-kernel CUDA events come from an eager pass of the same K steps",
            },
            "encode_gibs": n * B * world / (enc_avg_ms * 1e-3) / GIB,
            "decode_gibs": n * B * world / (dec_avg_ms * 1e-3) / GIB,
            "verify_gibs": n * B * world / (ver_avg_ms * 1e-3) / GIB,
            "checked": {"per_shard_blake2sums_after_every_region": True, "oracle_parity_stripes": oracle_checked},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "config5_sweep": sweep,
            "timed_steps": step_mode,
            "gpu_launches": int(lt.item()),
            "clocks": clk.summary(),
        }
        print(json.dumps(line))
    enc.close()
    dec.close()


def run_sweep(args, torch, dist, rank, world, dev, local_rank, sum_kind=1, host=False):
    """BASELINE config 5 (extra, outside the timed step): mixed RS(6,3)/RS(10,4) stripes of 1 MiB blocks,
    every shard corrupted with p = 0.10, one garage_ec_scrub_repair sweep per code = detect (per-shard
    integrity tag) -> reconstruct -> rewrite in place; payload bytes healed-or-verified per second.
    sum_kind: 1 = adler8 tag (HBM-bound), 0 = blake2sum (Garage's Hash, compute-bound).
    host=True: the stripes live in pinned HOST memory (NUMA-local) and cross PCIe inside the timed
    region -- the end-to-end companion (ScrubWorker reading shard files, repair.rs:438-490)."""
    import garage_b200 as G

    n = args.sweep_e2e_stripes if host else args.sweep_stripes
    total_ms, detail = 0.0, {}
    for (k, m) in ((6, 3), (10, 4)):
        tot = k + m
        with G.GarageEc(local_rank, k, m) as ec:
            ec.set_sum_kind(sum_kind)
            L = ec.shard_len(B)
            stride = ec.stride_for(L)
            data = torch.empty(n * k * stride, dtype=torch.uint8, device=dev)
            ec.fill_random(data, n * k * stride, SEED + 77 + rank, 0)
            data.view(n, k, stride)[:, :, L:] = 0
            lens = torch.full((n,), L, dtype=torch.int32, device=dev)
            par = torch.zeros(n * m * stride, dtype=torch.uint8, device=dev)
            ec.encode(data, par, stride, n, shard_len=lens)
            shards = torch.cat([data.view(n, k, stride), par.view(n, m, stride)], dim=1).contiguous()
            del data, par
            sums = torch.zeros(n * tot * 32, dtype=torch.uint8, device=dev)
            ec.shard_sums(shards.view(-1), sums, stride, n, tot, shard_len=lens)
            orig = shards.clone()
            g = torch.Generator().manual_seed(99 + rank)
            hit = (torch.rand(n, tot, generator=g) < 0.10).to(dev)
            pos = torch.randint(0, L, (n, tot), generator=g).to(dev)
            bad = torch.zeros(n * tot, dtype=torch.uint8, device=dev)
            status = torch.zeros(n, dtype=torch.int32, device=dev)
            sidx, iidx = torch.nonzero(hit, as_tuple=True)
            nbad = hit.sum(dim=1)
            if host:
                h_sh, p1 = ec.host_alloc(n * tot * stride)
                h_sums = sums.cpu().numpy()
                h_lens = np.full(n, L, dtype=np.uint32)
                h_bad = np.zeros(n * tot, dtype=np.uint8)
                h_st = np.zeros(n, dtype=np.int32)
                hurt = orig.clone()
                hurt[sidx, iidx, pos[sidx, iidx]] ^= 0x5A
                ms, iters, warm = 0.0, 3, 1
                for it in range(iters + warm):
                    torch.from_numpy(h_sh).copy_(hurt.view(-1))
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    ec.scrub_repair(h_sh, h_sums, h_bad, stride, n, status=h_st, shard_len=h_lens)
                    if it >= warm:
                        ms += (time.perf_counter() - t0) * 1e3
                ms /= iters
                ok_h = h_st == 0
                assert np.array_equal(h_bad.reshape(n, tot) != 0, hit.cpu().numpy())
                assert int((~ok_h).sum()) == int((nbad > m).sum())
                assert np.array_equal(h_sh.reshape(n, tot, stride)[ok_h], orig.cpu().numpy()[ok_h])
                ec.host_free(p1)
                unrec = int((~ok_h).sum())
            else:
                ms, iters, warm = 0.0, 4, 3  # warm-up also lets the SM clock ramp back up after the PCIe-bound e2e phase
                for it in range(iters + warm):
                    shards.copy_(orig)
                    shards[sidx, iidx, pos[sidx, iidx]] ^= 0x5A
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    torch.cuda.synchronize()
                    a.record()
                    ec.scrub_repair(shards.view(-1), sums, bad, stride, n, status=status, shard_len=lens)
                    b.record()
                    torch.cuda.synchronize()
                    if it >= warm:
                        ms += a.elapsed_time(b)
                ms /= iters
                assert torch.equal(bad.view(n, tot).bool(), hit)
                ok = status == 0
                assert int((~ok).sum()) == int((nbad > m).sum())
                assert torch.equal(shards[ok], orig[ok])
                unrec = int((~ok).sum())
            detail["rs%d_%d" % (k, m)] = {"ms": ms, "stripes": n, "unrecoverable": unrec, "corrupt_shards": int(hit.sum())}
            total_ms += ms
            del shards, orig, sums
            torch.cuda.empty_cache()
    return total_ms, detail


def run_e2e(args, torch, dist, enc, dec, rank, world, dev, shards_d, data_d, present, L, stride):
    """encode: host data (pinned) -> parity (pinned); reconstruct: host shards (pinned) in place.
    H2D/D2H inside the timed region, through garage_ec_encode / garage_ec_reconstruct HOST mode."""
    import garage_b200 as G

    k, m = args.k, args.m
    tot = k + m
    n = min(args.e2e_blocks or 4096, args.blocks)  # 12 GB of pinned host memory per rank at 4096 blocks
    bufs = []
    while True:
        try:
            h_data, p1 = enc.host_alloc(n * k * stride)
            bufs.append(p1)
            h_par, p2 = enc.host_alloc(n * m * stride)
            bufs.append(p2)
            h_sh, p3 = enc.host_alloc(n * tot * stride)
            bufs.append(p3)
            break
        except G.EcError:
            for p in bufs:
                enc.host_free(p)
            bufs = []
            n //= 2
            if n < 64:
                break
    if n < 64:  # no pinned memory on this rank: still take part in the collectives below, then report the failure
        if world > 1:
            dist.barrier()
            dummy = torch.zeros(7, dtype=torch.float64, device=dev)
            dist.all_gather([torch.zeros_like(dummy) for _ in range(world)], dummy)
        return {"value": None, "unit": "GiB/s", "error": "pinned allocation failed on rank %d" % rank}
    torch.from_numpy(h_data).copy_(data_d[: n * k * stride])
    torch.from_numpy(h_sh).copy_(shards_d[: n * tot * stride])
    h_present = np.ascontiguousarray(present[:n].numpy())
    h_sh.reshape(n, tot, stride)[h_present == 0] = 0  # the erased shards really are gone
    h_lens = np.full(n, L, dtype=np.uint32)
    h_status = np.zeros(n, dtype=np.int32)
    torch.cuda.synchronize()

    t_enc = t_dec = 0.0

    def step(timed=False):
        nonlocal t_enc, t_dec
        t0 = time.perf_counter()
        enc.encode(h_data, h_par, stride, n, shard_len=h_lens)
        t1 = time.perf_counter()
        dec.reconstruct(h_sh, h_present, stride, n, status=h_status, shard_len=h_lens)
        t2 = time.perf_counter()
        if timed:
            t_enc += t1 - t0
            t_dec += t2 - t1

    for _ in range(2):
        step()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    steps = max(2, min(args.steps, 5))
    for _ in range(steps):
        step(True)
    torch.cuda.synchronize()
    el = time.perf_counter() - t0
    gpu_node, buf_node = enc.numa_info()
    mine = torch.tensor([el, t_enc, t_dec, float(gpu_node), float(buf_node), float(len(os.sched_getaffinity(0))), float(n)],
                        dtype=torch.float64, device=dev)
    if world > 1:
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
    else:
        allr = [mine]
    allr = [[float(x) for x in t.tolist()] for t in allr]
    if any(r[6] <= 0 for r in allr):
        for p in bufs:
            enc.host_free(p)
        return {"value": None, "unit": "GiB/s", "error": "pinned allocation failed on another rank"}
    el = max(r[0] for r in allr)
    n_all = sum(int(r[6]) for r in allr)  # blocks per e2e step over all ranks (a rank short of pinned memory runs fewer)
    # the e2e results are the same bytes the device-resident pass produced (sampled stripes)
    ref = shards_d.view(-1, tot, stride)
    ok = not h_status.any()
    for s in sorted(set([0, 1, n // 2, n - 1])):
        r = ref[s].cpu().numpy()
        ok = ok and np.array_equal(h_par.reshape(n, m, stride)[s], r[k:])
        ok = ok and np.array_equal(h_sh.reshape(n, tot, stride)[s], r)
    assert ok, "e2e results differ from the device-resident pass"
    up_enc, dn_enc = n * k * stride + n * 4, n * m * stride
    up_dec, dn_dec = n * k * stride + n * 4 + n * tot, n * m * ((L + 15) // 16 * 16) + n * 4
    res = {
        "value": 2 * n_all * B * steps / el / GIB, "unit": "GiB/s", "steps": steps, "blocks_per_step": n,
        "blocks_per_step_all_ranks": n_all,
        # whole job (all ranks): encode data + the k survivors up; parity + rebuilt shards + status down
        "h2d_bytes_per_step": int(world * (up_enc + up_dec)),
        "d2h_bytes_per_step": int(world * (dn_enc + dn_dec)),
        "api": "garage_ec_encode + garage_ec_reconstruct, GARAGE_EC_MEM_HOST, pinned buffers from garage_ec_host_alloc "
               "(NUMA-local to the GPU), calling thread bound to the GPU's node (garage_ec_bind_thread); encode stages 48 MB "
               "chunks through three lanes, reconstruct reads the survivors and writes the rebuilt shards in the pinned host "
               "buffer directly from the kernel (both inside the timed region, both over PCIe)",
        "timer": "host wall clock around synchronous calls (max over ranks)", "checked": bool(ok),
        # per-rank link numbers: which rank (which socket / root complex) limits the job
        "per_rank": [{"rank": i, "GiBs": 2 * int(r[6]) * B * steps / r[0] / GIB,
                      "encode_h2d_GBs": up_enc * steps / r[1] / 1e9, "encode_d2h_GBs": dn_enc * steps / r[1] / 1e9,
                      "reconstruct_h2d_GBs": up_dec * steps / r[2] / 1e9, "reconstruct_d2h_GBs": dn_dec * steps / r[2] / 1e9,
                      "gpu_numa_node": int(r[3]), "pinned_buffer_numa_node": int(r[4]), "thread_affinity_cpus": int(r[5])}
                     for i, r in enumerate(allr)],
    }
    slow = min(res["per_rank"], key=lambda x: x["GiBs"])
    fast = max(res["per_rank"], key=lambda x: x["GiBs"])
    local_ok = all(r["gpu_numa_node"] < 0 or r["gpu_numa_node"] == r["pinned_buffer_numa_node"] for r in res["per_rank"])
    if world == 1:
        res["limiter"] = ("the PCIe link: encode H2D %.1f GB/s + D2H %.1f GB/s, reconstruct H2D %.1f GB/s + D2H %.1f GB/s "
                          "(PCIe 5.0 x16: ~55 GB/s one way, ~47 GB/s per direction under bidirectional load); the kernels are "
                          "~100x faster (device-resident `value`)" % (slow["encode_h2d_GBs"], slow["encode_d2h_GBs"],
                                                                    slow["reconstruct_h2d_GBs"], slow["reconstruct_d2h_GBs"]))
    else:
        res["limiter"] = ("%d ranks at %.1f-%.1f GiB/s each (slowest rank %d: encode H2D %.1f GB/s, reconstruct H2D %.1f GB/s); pinned "
                          "buffers %s. A rank alone on such a host reaches ~48 GiB/s (53 GB/s H2D staged encode, 50 + 20 GB/s zero-copy reconstruct): a uniform per-rank drop with "
                          "all ranks active and NUMA-local buffers points at the shared host memory / IO system (aggregate DMA "
                          "%.0f GB/s up + %.0f GB/s down), not at placement and not at the kernels"
                          % (world, slow["GiBs"], fast["GiBs"], slow["rank"], slow["encode_h2d_GBs"], slow["reconstruct_h2d_GBs"],
                             "on every GPU's own NUMA node" if local_ok else "NOT all on their GPU's NUMA node",
                             res["h2d_bytes_per_step"] * steps / el / 1e9, res["d2h_bytes_per_step"] * steps / el / 1e9))
    for p in bufs:
        enc.host_free(p)
    return res


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist

        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist

            dist.destroy_process_group()


if __name__ == "__main__":
    main()
