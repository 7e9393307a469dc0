"""CPU: the parts of bench.py the driver depends on that need no GPU -- the reference arm prints one JSON line with the
contract's keys, the same `config` object as the GPU arm, and times only the hashing call."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_line():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                          "--log2-batch", "12"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1                                       # exactly one JSON line on stdout
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "hades_permutations_per_sec" and d["unit"] == "perm/s"
    assert d["steps"] == 2 and d["warmup"] == 1 and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0
    # value = digests hashed / time spent inside the hashing call
    assert abs(d["value"] - (1 << 12) / (d["ms_per_step"] * 1e-3)) / d["value"] < 1e-6
    sys.path.insert(0, ROOT)
    import bench
    assert d["config"] == bench.workload_config(12, 1)           # identical to the GPU arm's config object


def test_non_zero_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--gpus", "2", "--log2-batch", "10"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert res.returncode == 0 and res.stdout.strip() == ""


import pytest


def _merkle4_oracle_words(data):
    """Merkle4 digests of (n, 4, 4) limbs by the C oracle, as dump_outputs writes them: 32-bit words in float64."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    sys.path.insert(0, ROOT)
    import c_oracle
    import hades_oracle as o
    from poseidon252_b200.scalar import to_mont
    tag = to_mont(o.hash_to_scalar(o.tag_input([o.Absorb(4), o.Squeeze(1)], o.Domain.Merkle4)))
    return c_oracle.digest(tag, data, 4, 1).reshape(len(data), 4).view(np.uint32).astype(np.float64)


def test_reference_arm_dump_outputs(tmp_path):
    """--dump-outputs: the last step's digests, one float64 row of 8 exact 32-bit words per item, identical from run
    to run and equal to the oracle on the arm's seeded inputs."""
    import numpy as np
    from poseidon252_b200.scalar import random_limbs_fast
    dumps = []
    for run in range(2):
        d = tmp_path / str(run)
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                              "--warmup", "0", "--log2-batch", "10", "--dump-outputs", str(d)],
                             capture_output=True, text=True, timeout=300, cwd=ROOT)
        assert res.returncode == 0, res.stderr[-2000:]
        assert sorted(os.listdir(d)) == ["digests.npy"]
        dumps.append(np.load(d / "digests.npy"))
    assert dumps[0].dtype == np.float64 and dumps[0].shape == (1 << 10, 8)
    assert np.array_equal(dumps[0], dumps[1])
    assert np.array_equal(dumps[0], _merkle4_oracle_words(random_limbs_fast(np.random.default_rng(123), (1 << 10, 4))))


def test_steps_must_be_positive():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert res.returncode != 0 and "--steps" in res.stderr


@pytest.mark.gpu
def test_gpu_arm_dump_outputs(tmp_path):
    """--dump-outputs on the GPU arm: the digests of the last timed step (input buffer (steps - 1) % 4 of the seeded
    rotation), bit-exact against the oracle."""
    import numpy as np
    from poseidon252_b200.scalar import random_limbs_fast
    steps, log2 = 3, 12
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "3",
                          "--log2-batch", str(log2), "--no-tree", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-3000:]
    assert json.loads(res.stdout)["steps"] == steps
    got = np.load(tmp_path / "digests.npy")
    rng = np.random.default_rng(0xC10D)
    ins = [random_limbs_fast(rng, (1 << log2, 4)) for _ in range(4)]
    assert got.dtype == np.float64 and np.array_equal(got, _merkle4_oracle_words(ins[(steps - 1) % 4]))


@pytest.mark.gpu
def test_gpu_arm_line_small():
    """the GPU arm end to end on a reduced batch: one JSON line, contract keys, roofline / imad / e2e / tree blocks,
    tree parity ok"""
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "3", "--log2-batch", "14",
                          "--log4-leaves", "7", "--no-cpu-baseline"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-3000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "clocks", "gpu_launches", "roofline", "e2e", "tree"):
        assert k in d, k
    assert d["gpu_launches"] == 3 and d["n_gpus"] == 1 and d["value"] > 1e6
    assert d["roofline"]["bound"] == "hbm" and 0 < d["roofline"]["frac"] < 1
    assert d["roofline"]["imad"]["bound"] == "imad" and 0 < d["roofline"]["imad"]["frac"] < 1
    assert d["e2e"]["h2d_bytes_per_step"] == (1 << 14) * 128 and d["e2e"]["d2h_bytes_per_step"] == (1 << 14) * 32
    assert d["tree"]["parity"] == "ok" and d["tree"]["leaves_log4"] == 7 and len(d["tree"]["per_level_rank0"]) == 7
