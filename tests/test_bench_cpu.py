"""CPU-side checks of bench.py's host logic: the known-answer arithmetic that verifies the
timed MSMs, the reference arm's JSON line and its step / budget handling, the output dump."""
import json
import os
import random
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

R = bench.R_MODULUS


def test_dot_mod_r_matches_big_integers():
    rnd = random.Random(4)
    n = 5000
    a = [rnd.getrandbits(250) for _ in range(n)] + [(1 << 256) - 1, 0]
    s = [rnd.getrandbits(250) for _ in range(n)] + [(1 << 256) - 1, 12345]
    A = torch.from_numpy(np.frombuffer(b"".join(x.to_bytes(32, "little") for x in a), np.uint8).reshape(-1, 32).copy())
    S = torch.from_numpy(np.frombuffer(b"".join(x.to_bytes(32, "little") for x in s), np.uint8).reshape(-1, 32).copy())
    assert bench.dot_mod_r(torch, A, S) == sum(x * y for x, y in zip(a, s)) % R


def test_known_answer_identity_on_the_oracle():
    """sum s_i (a_i G) == (sum a_i s_i mod r) G: the identity bench.py's verification rests on."""
    from oracle import decaf377_ref as o
    rnd = random.Random(5)
    a = [rnd.randrange(R) for _ in range(6)]
    s = [rnd.randrange(R) for _ in range(6)]
    pts = [o.scalar_mul(o.GENERATOR, x) for x in a]
    lhs = o.compress(o.vartime_multiscalar_mul(s, pts))
    assert lhs == bench.expected_encoding(sum(x * y for x, y in zip(a, s)) % R)


def test_reference_arm_line_and_budget():
    def run(*extra):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", *extra],
                           capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 0, r.stderr
        return json.loads(r.stdout.strip().splitlines()[-1])

    line = run("--logn", "12", "--steps", "3", "--warmup", "2")
    assert line["impl"] == "reference" and line["steps"] == 3 and line["warmup"] == 2
    assert line["unit"] == "Mpoints/s" and line["value"] > 0 and line["higher_is_better"] is True
    assert line["config"]["same_size_as_gpu_arm"] is True and "2^12" in line["config"]["workload"]
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0,
                           "d2h_bytes_per_step": 0}
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    # a budget that one step already exhausts still yields one timed step, honestly reported
    line = run("--logn", "14", "--steps", "20", "--warmup", "5", "--ref-budget-s", "0.01")
    assert line["steps"] == 1 and line["warmup"] == 1
    # other ranks of a torchrun launch print nothing
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--logn", "10"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT, env=dict(os.environ, RANK="1"))
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_steps_below_one_are_refused():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0 and "--steps" in r.stderr


def test_dump_outputs_float32_and_seeded_row_sample(tmp_path):
    small = {"element_xy": torch.arange(64, dtype=torch.uint8), "encoding": torch.arange(32, dtype=torch.uint8)}
    bench.dump_outputs(str(tmp_path / "small"), small)
    for name, t in small.items():
        got = np.load(tmp_path / "small" / (name + ".npy"))
        assert got.dtype == np.float32 and np.array_equal(got, t.numpy())
    assert not (tmp_path / "small" / "rows.npy").exists()
    # larger than the budget: every output keeps the same seeded sample of rows
    n = 600000
    g = torch.Generator().manual_seed(1)
    big = {"elements": torch.randint(0, 256, (n, 128), dtype=torch.uint8, generator=g),
           "ok": torch.randint(0, 2, (n,), dtype=torch.uint8, generator=g)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), big)
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= bench.DUMP_BUDGET
    rows = np.load(tmp_path / "a" / "rows.npy")
    assert rows.dtype == np.float64 and 0 < len(rows) < n and np.all(np.diff(rows) > 0)
    rows = rows.astype(np.int64)
    for name, t in big.items():
        got = np.load(tmp_path / "a" / (name + ".npy"))
        assert got.dtype == np.float32 and np.array_equal(got, t.numpy()[rows])
    for f in ("rows.npy", "elements.npy", "ok.npy"):
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f))
