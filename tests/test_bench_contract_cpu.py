"""bench.py contract on the CPU side: the reference arm (the oracle timed on the host cores)
prints one JSON line with the keys the driver reads, and needs neither a GPU nor the CUDA
library."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line(oracle):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload",
                          "tiny", "--steps", "2", "--warmup", "1", "--ref-sample-sweeps", "40"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "spin_flip_attempts_per_sec" and d["unit"] == "flips/s"
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 1 and d["higher_is_better"] is True
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["scaling"] == "strong" and isinstance(d["dtype"], str) and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    e2e = d["e2e"]
    assert e2e["value"] == d["value"] and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0
    assert d["gpu_launches"] == 0


import numpy as np
import pytest


def test_dump_outputs_unpacks_and_bounds_what_it_writes(tmp_path, monkeypatch):
    """--dump-outputs: the spins of the packed words land at [replica, site] (a seeded sample of the
    sites when they do not fit), and an array above the per-array bound is cut to a sample."""
    monkeypatch.setenv("NCCL_DEBUG", "WARN")     # what importing bench would set in this process
    import bench

    rng = np.random.default_rng(1)
    E, n = 70, 50
    st = rng.integers(0, 2, (E, n)).astype(bool)
    words = (E + 31) // 32
    bits = np.zeros((words * 32, n), dtype=np.uint64)
    bits[:E] = st
    packed = (bits.reshape(words, 32, n) << np.arange(32, dtype=np.uint64)[None, :, None]).sum(1).T
    packed = packed.astype(np.uint32)
    got = bench.sampled_states(packed, E)
    assert got.dtype == np.float32 and (got == st).all()
    part = bench.sampled_states(packed, E, nbytes=4 * E * 7)
    assert part.shape == (E, 7)
    assert all(any((part[:, k] == st[:, s]).all() for s in range(n)) for k in range(7))
    assert (part == bench.sampled_states(packed, E, nbytes=4 * E * 7)).all()
    big = np.arange(bench.DUMP_BYTES // 8 + 5, dtype=np.float64)
    bench.dump_outputs(str(tmp_path), 0, 1, energies=big[:10], big=big)
    assert (np.load(tmp_path / "energies.npy") == big[:10]).all()
    cut = np.load(tmp_path / "big.npy")
    assert cut.nbytes == bench.DUMP_BYTES and np.isin(cut, big).all()


@pytest.mark.gpu
def test_b200_arm_prints_the_contract_line(native, tmp_path):
    """The product arm on the CI-size workload: one JSON line with value / e2e / roofline /
    clocks / gpu_launches, all measured (no CPU baseline leg here, it has its own test), and with
    --dump-outputs the per-sweep energies and the spins its last timed step left behind."""
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tiny", "--steps", "3",
                          "--warmup", "3", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert "impl" not in d or d["impl"] != "reference"
    assert d["metric"] == "spin_flip_attempts_per_sec" and d["unit"] == "flips/s" and d["n_gpus"] == 1
    assert d["steps"] == 3 and d["warmup"] == 3 and d["value"] > 0 and d["higher_is_better"] is True
    assert d["gpu_launches"] > 0
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and r["peak"] > 0
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    e2e = d["e2e"]
    assert e2e["value"] > 0 and e2e["h2d_bytes_per_step"] >= 0 and e2e["d2h_bytes_per_step"] > 0
    assert e2e["value"] <= d["value"] * 1.05      # host copies inside the timed region cannot make it faster
    assert "sm_mhz" in d["clocks"] and "reasons" in d["clocks"]
    # tiny: 3D +-J L = 16 (j_seed 2024), 64 replicas, 20 sweeps per step; all 4096 sites fit the dump
    en = np.load(tmp_path / "energies.npy")
    st = np.load(tmp_path / "states.npy")
    assert en.dtype == np.float64 and en.shape == (64, 20)
    assert st.dtype == np.float32 and st.shape == (64, 16 ** 3)
    g = native.Graph.torus(native.Context.get(0), (16, 16, 16), j0=1.0, pmj=True, j_seed=2024)
    a, b, j = g.edges()
    s = st.astype(np.int64) * 2 - 1
    assert (en[:, -1] == (s[:, a.astype(np.int64)] * s[:, b.astype(np.int64)] * j).sum(1)).all()
