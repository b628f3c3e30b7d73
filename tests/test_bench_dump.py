"""bench.py --dump-outputs: the arrays the timed path computed in its last step, written so that two builds (or two
runs) can be compared output for output."""
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d)) if f.endswith(".npy")}


def test_write_outputs_dtypes_and_seeded_sample(tmp_path):
    n = 1000
    rng = np.random.default_rng(3)
    arrays = {"price": rng.standard_normal((n, 4)), "window": rng.standard_normal((n, 8, 4)).astype(np.float32),
              "done": rng.random(n) < .1, "risk": rng.integers(0, 4, (n, 4)).astype(np.uint8),
              "timestamp": np.arange(n, dtype=np.int64) * 7}
    bench.write_outputs(tmp_path / "all", arrays, env_offset=5000)
    got = load(tmp_path / "all")
    assert {k: v.dtype for k, v in got.items()} == {"price": np.float64, "window": np.float32, "done": np.float32,
                                                   "risk": np.float32, "timestamp": np.float64, "env_index": np.float64}
    np.testing.assert_array_equal(got["env_index"], np.arange(n) + 5000)
    for k, a in arrays.items():
        np.testing.assert_array_equal(got[k], a)

    limit = 100 * (8 * 4 + 4 * 32 + 4 + 16 + 8 + 8)  # 100 envs' worth
    for d in ("s1", "s2"):
        bench.write_outputs(tmp_path / d, arrays, env_offset=5000, limit=limit)
    s1, s2 = load(tmp_path / "s1"), load(tmp_path / "s2")
    assert sum(a.nbytes for a in s1.values()) <= limit
    idx = s1["env_index"].astype(np.int64) - 5000
    assert len(idx) == 100 and np.all(np.diff(idx) > 0)
    for k, a in arrays.items():
        np.testing.assert_array_equal(s1[k], a[idx])
        np.testing.assert_array_equal(s1[k], s2[k])


def run_bench(out, *args):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--warmup", "1", "--slabs", "8",
           "--streams", "8", "--setup-steps", "1024", "--no-cpu-baseline", "--dump-outputs", str(out)] + list(args)
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    return load(out)


@pytest.mark.gpu
def test_dump_is_the_last_timed_step_and_reproducible(tmp_path):
    """Six timed steps as two CUDA-graph repeats of three and as one eager region of six give the same outputs bit for
    bit.  Fourteen steps end on the same slab (step index 14 after one warm-up step, 14 % 8 == 6) eight steps later:
    the same envs, other values, so the dump is the slab's state after the last timed step.  Eight slabs on eight
    streams for 1,024 steps each, so that blocks of the slabs' step and refill kernels share SMs: the TMA-staged step
    kernel then needs its proxy fence before each shared-memory copy to stay bit-reproducible."""
    a = run_bench(tmp_path / "a", "--steps", "3", "--repeats", "2", "--graph", "on")
    b = run_bench(tmp_path / "b", "--steps", "6", "--repeats", "1", "--graph", "off")
    c = run_bench(tmp_path / "c", "--steps", "14", "--repeats", "1", "--graph", "off")
    assert sum(x.nbytes for x in a.values()) <= bench.DUMP_LIMIT
    assert a.keys() == b.keys() and {"state_price", "reward", "done", "transaction_units", "shaped_reward"} <= a.keys()
    assert a["state_price"].shape == (bench.ENVS_PER_GPU, bench.N_ASSETS)
    for k in a:
        assert a[k].dtype in (np.float32, np.float64), k
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    np.testing.assert_array_equal(a["env_index"], c["env_index"])
    assert not np.array_equal(a["state_timestamp"], c["state_timestamp"])
    assert not np.array_equal(a["state_price"], c["state_price"])
