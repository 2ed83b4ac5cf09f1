"""The bench contract: `bench.py --impl reference` prints exactly one JSON line with the keys a caller
reads and non-zero ranks stay silent (CPU only); `--dump-outputs` writes the results of the last timed
step (GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(env_extra=None):
    env = dict(os.environ)
    env.update(env_extra or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                           "--warmup", "1", "--cpu-blocks", "16"], capture_output=True, text=True, env=env, timeout=300)


def test_reference_arm_line():
    r = run()
    assert r.returncode == 0, r.stderr
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "GiB/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("RS(k,m) encode+decode GiB/s on 1 MiB blocks")
    assert d["value"] > 0 and d["steps"] == 2 and d["dtype"] == "u8" and d["data"] == "synthetic"
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": "GiB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_other_ranks_do_nothing():
    r = run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_bad_arguments_are_rejected():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True,
                           timeout=60)
        assert r.returncode == 2 and "error" in r.stderr, extra


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_steps_results(tmp_path):
    """--dump-outputs: parity of the sampled stripes == the CPU oracle's encode of the bench's input stream,
    rebuilt shards == the erased shards of the original stripe, every stripe recovered, under 64 MB"""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O

    k, m, n, B = 10, 4, 48, 1 << 20
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--blocks", str(n), "--steps", "2",
                        "--warmup", "1", "--no-e2e", "--no-cpu", "--no-sweep", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    names = sorted(p.name for p in tmp_path.iterdir())
    assert names == ["encode_parity.npy", "reconstruct_shards.npy", "reconstruct_status.npy", "sample_stripes.npy"]
    assert sum(p.stat().st_size for p in tmp_path.iterdir()) <= 64_000_000
    d = {name[:-4]: np.load(tmp_path / name) for name in names}
    assert all(a.dtype == np.float32 for a in d.values())
    assert d["reconstruct_status"].shape == (n,) and not d["reconstruct_status"].any()
    L = int(O.lib().rs_oracle_shard_len(B, k))
    stride = (L + 127) // 128 * 128
    P = O.build_matrix(k, m, 0)
    idx = d["sample_stripes"].astype(np.int64)
    assert len(idx) == len(set(idx.tolist())) and d["encode_parity"].shape == (len(idx), m, L)
    for j, s in enumerate(idx):
        data = O.fill_random(k * stride, 0x6761726167650010, int(s) * k * stride).reshape(k, stride)
        data[:, L:] = 0
        data[k - 1, L - (k * L - B):] = 0
        par = O.encode(k, m, P, data.reshape(-1), stride, 1, np.array([L], dtype=np.uint32)).reshape(m, stride)
        assert np.array_equal(d["encode_parity"][j], par[:, :L]), s
        stripe = np.concatenate([data, par])[:, :L]
        rows = [next((i for i in range(k + m) if np.array_equal(stripe[i], got)), -1) for got in d["reconstruct_shards"][j]]
        assert -1 not in rows and rows == sorted(set(rows)), (s, rows)
