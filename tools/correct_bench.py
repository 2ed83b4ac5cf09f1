#!/usr/bin/env python
"""Device-resident timing of garage_ec_correct against garage_ec_verify (same bytes read) on
4096 x 1 MiB RS(10,4), with the device-to-device copy peak of the same run as the roofline.
Not the contract bench (bench.py).

    python tools/correct_bench.py [--blocks 4096 --iters 12 --warmup 2] [--out profiles/x.json]

Scenarios: clean batch; one stale shard in 1 % / 100 % of the stripes; two stale shards in every
stripe; byte flips (each shard of each stripe has one byte flipped with probability 0.10).  Each
iteration restores the corrupted input (untimed), then times verify and correct back to back with
CUDA events; the median of the iterations is reported.
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ap = argparse.ArgumentParser()
ap.add_argument("--blocks", type=int, default=4096)
ap.add_argument("--iters", type=int, default=12)
ap.add_argument("--warmup", type=int, default=2)
ap.add_argument("--out", default=None)
args = ap.parse_args()

import torch  # noqa: E402

import garage_b200 as G  # noqa: E402

k, m, n = 10, 4, args.blocks
tot = k + m
ec = G.GarageEc(0, k, m)
L = ec.shard_len(1 << 20)
stride = ec.stride_for(L)
orig = torch.zeros(n * tot * stride, dtype=torch.uint8, device="cuda")
o3 = orig.view(n, tot, stride)
data = torch.empty(n * k * stride, dtype=torch.uint8, device="cuda")
ec.fill_random(data, data.numel(), 11)
data.view(n, k, stride)[:, :, L:] = 0
par = torch.zeros(n * m * stride, dtype=torch.uint8, device="cuda")
lens = torch.full((n,), L, dtype=torch.int32, device="cuda")
ec.encode(data, par, stride, n, shard_len=lens)
o3[:, :k] = data.view(n, k, stride)
o3[:, k:] = par.view(n, m, stride)
del data, par
sh = torch.empty_like(orig)
src = torch.empty_like(orig)
mm = torch.zeros(n, dtype=torch.int32, device="cuda")
st = torch.zeros(n, dtype=torch.int32, device="cuda")
fx = torch.zeros(n * tot, dtype=torch.uint8, device="cuda")
g = torch.Generator(device="cuda").manual_seed(5)


def scenario(name):
    src.copy_(orig)
    s3 = src.view(n, tot, stride)
    if name.startswith("stale"):
        nshards, frac = (2, 1.0) if name == "stale2_100pct" else (1, 0.01 if name == "stale1_1pct" else 1.0)
        rows = torch.randperm(n, device="cuda", generator=g)[: max(1, int(n * frac))]
        for j in range(nshards):
            idx = torch.randint(0, tot, (rows.numel(),), device="cuda", generator=g)
            if j:
                idx = (idx0 + 1 + idx % (tot - 1)) % tot  # a different shard than the first one
            idx0 = idx
            s3[rows, idx, :L] = torch.randint(0, 256, (rows.numel(), L), dtype=torch.uint8, device="cuda", generator=g)
    elif name == "flip_p0.10":
        hit = torch.rand(n, tot, device="cuda", generator=g) < 0.10
        s_idx, r_idx = hit.nonzero(as_tuple=True)
        cols = torch.randint(0, L, (s_idx.numel(),), device="cuda", generator=g)
        s3[s_idx, r_idx, cols] ^= torch.randint(1, 256, (s_idx.numel(),), dtype=torch.uint8, device="cuda", generator=g)


def time_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(torch.cuda.current_device())
        info["power_limit_w"] = pynvml.nvmlDeviceGetEnforcedPowerLimit(h) / 1000.0
        info["sm_clock_max_mhz"] = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
    except Exception as e:  # noqa: BLE001
        info["nvml_error"] = repr(e)
    return info


read_bytes = n * tot * L
res = {"tool": "tools/correct_bench.py", "workload": "RS(10,4), %d x 1 MiB blocks, DEVICE mode" % n,
       "bytes_read_per_call": read_bytes, "iters": args.iters, "warmup": args.warmup, **gpu_info(), "scenarios": {}}
copy_ms = []
for i in range(args.warmup + args.iters):
    t = time_ms(lambda: sh.copy_(orig))
    if i >= args.warmup:
        copy_ms.append(t)
res["copy_peak"] = {"median_ms": statistics.median(copy_ms), "GBps_read_plus_write": 2 * orig.numel() / statistics.median(copy_ms) / 1e6}
for name in ["clean", "stale1_1pct", "stale1_100pct", "stale2_100pct", "flip_p0.10"]:
    scenario(name)
    ver, cor = [], []
    for i in range(args.warmup + args.iters):
        sh.copy_(src)
        tv = time_ms(lambda: ec.verify(sh, mm, stride, n, shard_len=lens))
        tc = time_ms(lambda: ec.correct(sh, stride, n, status=st, fixed=fx, shard_len=lens))
        if i >= args.warmup:
            ver.append(tv)
            cor.append(tc)
    ok = bool(torch.equal(sh, orig)) and int(st.abs().sum()) == 0
    mv, mc = statistics.median(ver), statistics.median(cor)
    res["scenarios"][name] = {
        "verify_median_ms": mv, "correct_median_ms": mc, "correct_over_verify": mc / mv,
        "verify_GBps": read_bytes / mv / 1e6, "correct_GBps": read_bytes / mc / 1e6,
        "stripes_with_fixed_shards": int((fx.view(n, tot).sum(dim=1) > 0).sum()),
        "restored_exactly": ok,
        "verify_ms_all": ver, "correct_ms_all": cor,
    }
print(json.dumps(res, indent=1))
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
