#!/usr/bin/env python
"""Benchmark of the classical Ising Monte-Carlo hot path (BASELINE.json metric: spin-flip
attempts / s, device-timed, max over ranks, + fraction of the HBM roofline).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload c3|c2]
                  [--dump-outputs DIR]

Workload c3 (default; the configuration BASELINE.json's target is quoted on): 3D Edwards-
Anderson +-J spin glass, L = 64 periodic, 1024 replicas IN TOTAL, one step =
run_monte_carlo_annealing_and_get_energies with a (0, 0.1) -> (T, 1.2) schedule of T sweeps and
the energy of every replica after every sweep.  Replicas are the sharding unit (the reference's
rayon axis, lattice.rs:192-197): with N ranks every rank simulates 1024 / N of them ("sharded
across 8 B200" in BASELINE.json's config 3), no data-path collective, scaling = strong.  The
1024-replicas-per-GPU figure (weak scaling) is reported beside it as `weak_value`.

`value`  : all ranks' flip attempts / device time of K steps, state resident in HBM.
`e2e`    : the same metric through Lattice.run_monte_carlo_annealing_and_get_energies with host
           buffers (initial state H2D, energies + bool[E, N] states D2H inside the timed region).
`roofline`: the sweep kernel alone (algorithmic bytes per launch / its mean launch time).
`--impl reference`: the CPU restatement of the reference algorithm (oracle/, all host threads)
           on a bounded sample of the same workload.
`--dump-outputs DIR`: after the `value` region, DIR/energies.npy (float64[E, sweeps], the per-sweep
           energies its last step returned) and DIR/states.npy (float32[E, k], 1 = up, the spins at
           a fixed seeded sample of k sites); the same arguments give the same inputs on every run.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

# the contract is ONE line on stdout: keep NCCL's "NCCL version ..." banner (printed to stdout at
# NCCL_DEBUG=VERSION, which some launchers export) out of it
if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
    os.environ["NCCL_DEBUG"] = "WARN"

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

WORKLOADS = {
    # name: (dims, pmj, j0, replicas per GPU, sweeps per step, schedule ends)
    "c3": dict(dims=(64, 64, 64), pmj=True, j0=1.0, replicas=1024, sweeps=1000, beta=(0.1, 1.2),
               desc="3D EA +-J spin glass L=64 periodic, 1024 replicas in total (sharded over the ranks), "
                    "run_monte_carlo_annealing_and_get_energies, 1000 sweeps/step"),
    "c2": dict(dims=(4096, 4096), pmj=False, j0=-1.0, replicas=1024, sweeps=20, beta=(0.43, 0.43),
               desc="2D square ferromagnet 4096x4096 checkerboard, 1024 experiments/GPU, "
                    "beta=0.43, 20 sweeps/step"),
    "c4": dict(kind="tempering", n=1_000_000, degree=3, replicas=64, sweeps=100, swap_every=10,
               beta=(0.1, 1.5), dims=(1_000_000,), pmj=False, j0=-1.0,
               desc="random 3-regular graph N=1e6 (greedy colouring), parallel tempering: ONE ladder of 64 betas "
                    "geometric in [0.1, 1.5] sharded over the ranks, swap every 10 sweeps, 100 sweeps/step"),
    "c5": dict(kind="single", dims=(65536, 65536), pmj=False, j0=-1.0, sweeps=20, beta=(0.44, 0.44), replicas=1,
               desc="2D ferromagnet 65536x65536 single lattice bit-packed along x, row strips over the "
                    "ranks with halo exchange, beta=0.44, 20 sweeps/step"),
    "tiny": dict(dims=(16, 16, 16), pmj=True, j0=1.0, replicas=64, sweeps=20, beta=(0.1, 1.2),
                 desc="3D +-J L=16, 64 replicas (CI-size)"),
}
# SURVEY.md 8(d): every spin bit read once and written once per sweep (2 bits / flip) plus the
# coupling bits and the per-sweep energy write amortised over the replicas.
def algorithmic_bytes_per_flip(w):
    n = int(np.prod(w["dims"]))
    dim = len(w["dims"])
    b = 0.25
    if w["pmj"]:
        b += dim / 8.0 / w["replicas"]
    return b, n


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "250"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except Exception:
                continue
            for k, n in enumerate(names):
                if len(r) > 2 + k and r[2 + k].lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(mx)) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def dist_setup(ngpus):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return world, rank, local


def betas_for(w):
    b0, b1 = w["beta"]
    # documented linear ramp (0, b0) -> (T, b1): every sweep has its own beta and thresholds
    return np.linspace(b0, b1, w["sweeps"], endpoint=False)


# ------------------------------------------------------------------------------------------------
# reference arm: CPU restatement of the reference algorithm, all host threads
# ------------------------------------------------------------------------------------------------
def oracle_sample(w, steps, warmup, sample_sweeps=None, with_energies=True):
    import oracle_lib

    # all host cores, also under torchrun (which exports OMP_NUM_THREADS=1)
    try:
        ncores = len(os.sched_getaffinity(0))
    except AttributeError:
        ncores = os.cpu_count() or 1
    oracle_lib.lib().orc_set_num_threads(ncores)
    threads = oracle_lib.lib().orc_num_threads()
    dims = w["dims"]
    n = int(np.prod(dims))
    rng = np.random.default_rng(2024)
    # same lattice family: periodic torus, +-J iid (or uniform) couplings
    idx = np.arange(n)
    coords = np.unravel_index(idx, dims[::-1])[::-1]  # x fastest
    a, b, j = [], [], []
    for d in range(len(dims)):
        c = [x.copy() for x in coords]
        c[d] = (c[d] + 1) % dims[d]
        nb = np.ravel_multi_index(c[::-1], dims[::-1])
        a.append(idx)
        b.append(nb)
        j.append(rng.integers(0, 2, n) * 2.0 - 1.0 if w["pmj"] else np.full(n, w["j0"]))
    g = oracle_lib.Graph(arrays=(np.concatenate(a), np.concatenate(b), np.concatenate(j)), nvars=n)
    E = threads
    if sample_sweeps is None:
        # measured on this image's Xeon: ~60 ns per attempt + energy term while the lattice is
        # cache-resident, ~300 ns once adjacency + state exceed L2; size one step to ~6 s
        per_attempt = 60e-9 if n <= 65536 else 300e-9
        sample_sweeps = max(1, int(6.0 / (n * per_attempt)))
    stops = [(0, w["beta"][0]), (sample_sweeps, w["beta"][1])]
    seeds = oracle_lib.make_seeds(1, E)
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        g.run_annealing(stops, sample_sweeps, seeds, q1_compat=False, per_step_energies=with_energies)
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    attempts = E * n * sample_sweeps
    total = sum(times)
    return dict(value=attempts * len(times) / total, ms_per_step=1e3 * total / len(times), cores=threads,
                sample=f"{E} experiments (one per host thread) x {sample_sweeps} timesteps of {n} "
                       f"random-site attempts{' + get_energy' if with_energies else ''} each, "
                       f"lattice {'x'.join(map(str, dims))}")


def regular_graph(n, d, seed):
    """random d-regular graph, pairing model with rejection of self loops / multi-edges"""
    rng = np.random.default_rng(seed)
    while True:
        stubs = np.repeat(np.arange(n, dtype=np.int64), d)
        rng.shuffle(stubs)
        a, b = stubs[0::2], stubs[1::2]
        key = np.minimum(a, b) * n + np.maximum(a, b)
        if not (a == b).any() and len(np.unique(key)) == len(key):
            return a, b


def oracle_sample_tempering(w, steps, warmup):
    """CPU restatement of the tempering loop (oracle/ising_oracle.c: orc_pt_run, cadence of
    tempering.rs:156-222, random-site Metropolis per replica) on a bounded sample: the same graph
    family at N = 50 000 sites, the same 64 betas and swap cadence, all host threads over replicas."""
    import oracle_lib

    try:
        ncores = len(os.sched_getaffinity(0))
    except AttributeError:
        ncores = os.cpu_count() or 1
    oracle_lib.lib().orc_set_num_threads(ncores)
    threads = oracle_lib.lib().orc_num_threads()
    n = 50_000
    a, b = regular_graph(n, w["degree"], 2026)
    g = oracle_lib.Graph(arrays=(a, b, np.full(len(a), w["j0"])), nvars=n)
    betas = np.geomspace(w["beta"][0], w["beta"][1], w["replicas"])
    sweeps = 2 * w["swap_every"]
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        g.pt_run(betas, 7, sweeps, w["swap_every"], sweeps)
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    total = sum(times)
    return dict(value=w["replicas"] * n * sweeps * len(times) / total, ms_per_step=1e3 * total / len(times),
                cores=threads,
                sample=f"{w['replicas']} betas x {sweeps} timesteps of {n} random-site attempts each on a random "
                       f"{w['degree']}-regular graph of N = {n} (full size: N = {w['n']}), swap every {w['swap_every']}")


def cpu_sample_for(w, steps, warmup, ref_sample_sweeps=None):
    if w.get("kind") == "tempering":
        return oracle_sample_tempering(w, steps, warmup)
    if w.get("kind") == "single":
        # the reference cannot hold a 65536^2 lattice (206 GB of edges, lattice.rs:31): its algorithm
        # is timed on 2048^2 lattices, one per host thread
        ws = dict(w)
        ws["dims"] = (2048, 2048)
        r = oracle_sample(ws, steps, warmup, ref_sample_sweeps, with_energies=False)
        r["sample"] += " (config 5 is ONE 65536x65536 lattice, which the reference cannot hold)"
        return r
    return oracle_sample(w, steps, warmup, ref_sample_sweeps)


def run_reference(args, w, world, rank):
    if rank != 0:
        return
    r = cpu_sample_for(w, args.steps, args.warmup, args.ref_sample_sweeps or None)
    line = {
        "impl": "reference", "metric": "spin_flip_attempts_per_sec", "value": r["value"],
        "unit": "flips/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": args.workload + ": " + w["desc"], "parallelism": "host threads over experiments"},
        "cpu_baseline": {"value": r["value"], "unit": "flips/s", "cores": r["cores"], "kind": "port",
                         "sample": r["sample"]},
        "e2e": {"value": r["value"], "unit": "flips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
def _dist_helpers(world, local):
    import torch

    if world > 1:
        import torch.distributed as dist

        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local))
    else:
        dist = None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce(x, op):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=getattr(dist.ReduceOp, op))
        return float(t.item())

    return dist, barrier, reduce


def run_tempering(args, w, world, rank, local):
    """config 4 as BASELINE states it: ONE ladder of 64 betas on a random 3-regular graph of 10^6
    sites, its configurations sharded over the N ranks (rank r holds block r of the betas; the
    energies of a swap step travel in one NCCL all-gather issued by the library).  A temperature
    is one replica BIT, so a rank that owns 8 of the 64 configurations still sweeps whole 32-bit
    words: the stated split cannot go faster than one GPU (DESIGN.md 7) - `ladders_value` beside
    it is what N GPUs are good for on this workload, one independent ladder per GPU."""
    import torch

    import pyisingmontecarlo_b200 as pkg
    from pyisingmontecarlo_b200 import _native as nat
    from pyisingmontecarlo_b200.tempering import shard_range

    torch.cuda.set_device(local)
    dist, barrier, reduce = _dist_helpers(world, local)
    n, d = w["n"], w["degree"]
    a, b = regular_graph(n, d, 2026)
    ctx = nat.Context.get(local)
    g = nat.Graph.from_edges(ctx, n, a.astype(np.uint64), b.astype(np.uint64), np.full(len(a), w["j0"]))
    betas = np.geomspace(w["beta"][0], w["beta"][1], w["replicas"])
    lo, hi = shard_range(w["replicas"], rank, world)
    pt = nat.Tempering(g, betas, seed=7, cfg_lo=lo, cfg_hi=hi, planes=args.planes, rounds=args.rounds)
    comm = None
    if world > 1:
        comm = nat.Comm.from_torch(ctx)
        pt.set_comm(comm)
    T, swap = w["sweeps"], w["swap_every"]

    def step(the_pt):   # device-resident loop of tempering.rs:156-222, no samples
        the_pt.timesteps_sample(T, swap, T + 1)

    for _ in range(args.warmup):
        step(pt)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    l0 = pt.sim_stats()["kernel_launches"]
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step(pt)
    barrier()
    dt = reduce(time.perf_counter() - t0, "MAX")
    launches = pt.sim_stats()["kernel_launches"] - l0
    clocks = sampler.stop() if rank == 0 else None
    flips = float(w["replicas"]) * n * T * args.steps
    value = flips / dt

    # one independent ladder per GPU (weak), for comparison
    ladders_value = None
    if world > 1:
        own = nat.Tempering(g, betas, seed=100 + rank, planes=args.planes, rounds=args.rounds)
        step(own)
        barrier()
        t0 = time.perf_counter()
        step(own)
        barrier()
        ladders_value = world * float(w["replicas"]) * n * T / reduce(time.perf_counter() - t0, "MAX")
        own.close()

    # e2e: the public LatticeTempering API with host buffers: the sampled states of all 64 betas
    # (64 x 10^6 bools) are read back once per step
    edges = list(zip(zip(a.tolist(), b.tolist()), [w["j0"]] * len(a)))
    lt = pkg.LatticeTempering(edges, seed=7, device=local)
    for beta in betas:
        lt.add_graph(0.0, 0.0, float(beta))
    lt.qmc_timesteps_sample(T, swap, T)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        st, en = lt.qmc_timesteps_sample(T, swap, T)
        _ = float(en[0]) + float(st[0, 0, 0])
    barrier()
    e2e_s = reduce(time.perf_counter() - t0, "MAX")
    e2e = {"value": flips / e2e_s, "unit": "flips/s", "h2d_bytes_per_step": 0,
           "d2h_bytes_per_step": int(w["replicas"] * n + 8 * w["replicas"]), "ms_per_step": 1e3 * e2e_s / args.steps,
           "api": "LatticeTempering.qmc_timesteps_sample (states of all betas + time-averaged energies to host; "
                  "graph and ladder stay resident between calls, so there is no per-step H2D)"}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r = oracle_sample_tempering(w, 1, 0)
        cpu = {"value": r["value"], "unit": "flips/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]}
    # SURVEY 8(d): 2 spin bits + CSR indices streamed once per sweep per replica block
    bpf = (2 * w["replicas"] / 8 + d * 4 + 4 + 4) / w["replicas"]
    peak, peak_src = peaks()
    att, acc = pt.pair_stats()
    if rank == 0:
        print(json.dumps({
            "metric": "spin_flip_attempts_per_sec", "value": value, "unit": "flips/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u32 bit-sliced (1 bit per spin per replica)", "data": "synthetic",
            "config": {"workload": args.workload + ": " + w["desc"], "ncolors": g.ncolors,
                       "parallelism": f"one ladder, configurations sharded x{world}, NCCL all-gather of the "
                                      "energies per swap step inside the library",
                       "timing": "host clock around device-synchronised steps; the loop itself never waits for the host",
                       "l2": "8 MiB of spins + 12 MB of indices per rank: L2-resident"},
            "ladders_value": ladders_value,
            "ladders_note": "N independent ladders, one per GPU (weak scaling)" if ladders_value else None,
            "roofline": {"bound": "hbm", "achieved": bpf * flips / dt / 1e9 / world, "peak": peak, "unit": "GB/s",
                         "frac": bpf * flips / dt / 1e9 / world / peak, "traffic": None, "peak_source": peak_src,
                         "kernel": "k_sweep_general (whole step, per GPU)", "algorithmic_bytes_per_flip": bpf},
            "swap_acceptance": float(acc.sum()) / max(1.0, float(att.sum())),
            "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
            "total_swaps": pt.total_swaps(),
        }), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_single(args, w, world, rank, local):
    """config 5: ONE lattice split in row strips (strong scaling: total work fixed); halo rows by
    ncclSend/ncclRecv inside the library, one deep exchange per 8 sweeps."""
    import torch

    import pyisingmontecarlo_b200 as pkg

    torch.cuda.set_device(local)
    dist, barrier, reduce = _dist_helpers(world, local)
    Lx, Ly = w["dims"]
    lat = pkg.SingleLattice2D(Lx, Ly, j=w["j0"], seed=9, device=local, planes=args.planes, rounds=args.rounds)
    betas = [w["beta"][0]] * w["sweeps"]
    for _ in range(args.warmup):
        lat.sweeps(betas)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    lat.strip.stats(reset=True)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        lat.sweeps(betas)
    barrier()
    wall = reduce(time.perf_counter() - t0, "MAX")
    stt = lat.strip.stats()
    dev_ms = reduce(stt["device_ms"], "MAX")
    clocks = sampler.stop() if rank == 0 else None
    flips = float(Lx) * Ly * w["sweeps"] * args.steps
    launches = stt["launches"]
    value = flips / (dev_ms * 1e-3)

    # e2e: public API, a fresh all-up lattice every step, the energy of the final state to the host
    def step_e2e():
        lat.set_all(True)
        lat.sweeps(betas)
        return lat.energy()

    step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    barrier()
    e2e_s = reduce(time.perf_counter() - t0, "MAX")
    e2e = {"value": flips / e2e_s, "unit": "flips/s", "h2d_bytes_per_step": int(8 * len(betas)),
           "d2h_bytes_per_step": 16 * world, "ms_per_step": 1e3 * e2e_s / args.steps,
           "api": "SingleLattice2D.set_all + sweeps + energy (the lattice lives on the device: the inputs of a "
                  "step are its betas, the result its energy)"}
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r = cpu_sample_for(w, 1, 0)
        cpu = {"value": r["value"], "unit": "flips/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]}
    peak, peak_src = peaks()
    bpf = 0.25
    per_launch_ms = dev_ms / max(1, launches)
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(tpath) and world == 1:
        tj = json.load(open(tpath)).get(args.workload)
        if tj:
            traffic = tj["dram_bytes_read_per_launch"] + tj["dram_bytes_write_per_launch"]
    if rank == 0:
        ach = bpf * (flips / world / max(1, launches)) / (per_launch_ms * 1e-3) / 1e9
        print(json.dumps({
            "metric": "spin_flip_attempts_per_sec", "value": value, "unit": "flips/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u32 bit-sliced (1 bit per spin)", "data": "synthetic",
            "config": {"workload": args.workload + ": " + w["desc"],
                       "parallelism": f"row strips x{world}, ncclSend/ncclRecv of 16 boundary rows per side every 8 sweeps",
                       "timing": "CUDA events of the library around each batch of sweeps (kernels + halo exchange), "
                                 "max over ranks",
                       "l2": "512 MiB lattice, larger than L2" if world == 1 else "%d MiB per rank" % (512 // world)},
            "wall_ms_per_step": 1e3 * wall / args.steps,
            "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "traffic": traffic,
                         "peak_source": peak_src, "frac": ach / peak, "kernel": "k_strip_phase (one colour phase, per GPU)",
                         "kernel_ms": per_launch_ms, "algorithmic_bytes_per_flip": bpf},
            "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
        }), flush=True)
    if world > 1:
        dist.destroy_process_group()


def instruction_bound(kind):
    """Model time of one site group (4 replica words) of the sweep kernel from its SASS instruction
    mix (profiles/r02_sass_mix.json) and the pipe rates measured by profiles/microbench/pipe_bench.cu
    (profiles/r02_pipe_bench.json): cycles = 2.07 per ALU-pipe instruction + ~2.4 per 32x32->64
    multiply that does not overlap + ~0.85 per IMAD + 1 per other issue slot."""
    try:
        mix = json.load(open(os.path.join(ROOT, "profiles", "r02_sass_mix.json")))[kind]
        rates = json.load(open(os.path.join(ROOT, "profiles", "r02_pipe_bench.json")))["model"]
    except Exception:
        return None
    cyc = (mix["alu"] * rates["alu"] + mix["mul_wide_or_hi"] * rates["mul_wide_or_hi"] +
           mix["imad"] * rates["imad"] + mix["other"] * rates["other"])
    return {"cycles_per_site_group": cyc, "mix": mix, "rates": rates}


DUMP_BYTES = 32 << 20   # per array: --dump-outputs writes at most 64 MB in all


def sampled_states(packed, E, nbytes=DUMP_BYTES):
    """float32[E, k] spins (1 = up) at a fixed, seeded sample of k sites (all sites when they fit in
    nbytes) from the packed words uint32[nvars, ceil(E / 32)] (bit r of word w = replica 32 w + r)"""
    nvars = packed.shape[0]
    k = min(nvars, nbytes // (4 * E))
    sites = np.sort(np.random.default_rng(0).choice(nvars, k, replace=False)) if k < nvars else np.arange(nvars)
    bits = (packed[sites, :, None] >> np.arange(32, dtype=np.uint32)) & 1
    return bits.reshape(k, -1)[:, :E].T.astype(np.float32)


def dump_outputs(path, rank, world, **arrays):
    """--dump-outputs DIR: what the timed path returned in its last step, as DIR/<name>.npy, so that
    two builds can be compared output for output.  An array larger than DUMP_BYTES is cut to a
    fixed, seeded sample of its elements; with several ranks every rank writes its own shard."""
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        if a.nbytes > DUMP_BYTES:
            idx = np.sort(np.random.default_rng(0).choice(a.size, DUMP_BYTES // a.itemsize, replace=False))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(path, name + (f".rank{rank}" if world > 1 else "") + ".npy"), a)


def run_b200(args, w, world, rank, local):
    import torch

    import pyisingmontecarlo_b200 as pkg
    from pyisingmontecarlo_b200 import _native as nat

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a B200; there is no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    ctx = nat.Context.get(local)
    E_total = w["replicas"]
    if E_total % (32 * world):
        raise SystemExit(f"{E_total} replicas do not split into whole 32-replica words over {world} ranks")
    E = E_total // world                      # strong scaling: the replicas are sharded over the ranks
    n = int(np.prod(w["dims"]))
    betas = betas_for(w)
    graph = nat.Graph.torus(ctx, w["dims"], j0=w["j0"], pmj=w["pmj"], j_seed=2024)
    sim = nat.Sim(graph, E, seed=31337, replica_offset=rank * E, planes=args.planes, rounds=args.rounds)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    def timed(the_sim, per_sweep_energies, steps):
        """steps x (L2 flush, all sweeps) -> stats of the timed region (device time from the library's
        CUDA events on its stream, max over ranks taken by the caller), its wall time and what the
        last step returned"""
        the_sim.reset_stats()
        barrier()
        t0 = time.perf_counter()
        out = None
        for _ in range(steps):
            flush.zero_()
            torch.cuda.synchronize()
            out = the_sim.sweeps(betas, per_sweep_energies=per_sweep_energies)
        barrier()
        return the_sim.stats(), time.perf_counter() - t0, out

    # -------- value: device-resident, sweeps + per-sweep energies
    for _ in range(args.warmup):
        flush.zero_()
        sim.sweeps(betas, per_sweep_energies=True)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    st, wall, energies = timed(sim, True, args.steps)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, rank, world, energies=energies, states=sampled_states(sim.packed(), E))
    dev_ms = max_over_ranks(st["sweep_device_ms"])
    launches = st["kernel_launches"]
    flips_all = sum_over_ranks(float(st["flip_attempts"]))
    value = flips_all / (dev_ms * 1e-3)

    # -------- the plain colour phase alone (same state, same betas, no energy accumulation)
    st2, _, _ = timed(sim, False, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    plain_ms = max_over_ranks(st2["sweep_kernel_ms"] / max(1, st2["sweep_kernel_launches"]))
    sweep_only_value = sum_over_ranks(float(st2["flip_attempts"])) / (max_over_ranks(st2["sweep_device_ms"]) * 1e-3)
    # the accumulating colour phase (second launch of every sweep of the `value` region): what is
    # left of a sweep after one plain phase (this charges it the per-chunk memset / conversion too)
    per_sweep_ms = dev_ms / (args.steps * len(betas))
    acc_ms = max(per_sweep_ms - plain_ms, 1e-9)
    bpf, _ = algorithmic_bytes_per_flip(w)
    flips_per_launch = E * n / 2.0  # one colour class per launch, per rank
    peak, peak_src = peaks()
    traffic = None   # dram__bytes_read + write per launch, from the committed ncu capture (1-GPU shape)
    tpath = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(tpath) and world == 1:
        tj = json.load(open(tpath)).get(args.workload)
        if tj:
            traffic = tj["dram_bytes_read_per_launch"] + tj["dram_bytes_write_per_launch"]

    def roof(ms, kernel, kind):
        ach = bpf * flips_per_launch / (ms * 1e-3) / 1e9
        d = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
             "traffic": traffic, "peak_source": peak_src, "kernel": kernel, "kernel_ms": ms,
             "algorithmic_bytes_per_flip": bpf, "algorithmic_bytes_per_launch": int(bpf * flips_per_launch)}
        ib = instruction_bound(kind) if world == 1 and args.workload == "c3" and not args.rounds else None
        if ib and clocks and clocks.get("sm_mhz"):
            site_groups = flips_per_launch / 128.0           # 4 words x 32 replicas per thread item
            smsp = 4 * torch.cuda.get_device_properties(local).multi_processor_count
            model_ms = ib["cycles_per_site_group"] * (site_groups / 32.0) / smsp / (clocks["sm_mhz"] * 1e3)
            d["instruction_bound"] = {"model_ms": model_ms, "frac_of_instruction_bound": model_ms / ms,
                                      "cycles_per_site_group": ib["cycles_per_site_group"], "mix": ib["mix"],
                                      "note": "kernel is bound by the integer pipes, not by HBM: see DESIGN.md 5 and "
                                              "profiles/microbench/pipe_bench.cu"}
        return d

    roofline = roof(acc_ms, "k_sweep_rows<ACC=1> (second colour phase + fused per-sweep energies): the kernel "
                            "that dominates `value`", "acc")
    roofline["plain_phase"] = roof(plain_ms, "k_sweep_rows<ACC=0> (first colour phase)", "plain")
    roofline["whole_step_frac"] = bpf * (flips_all / world) / (dev_ms * 1e-3) / 1e9 / peak

    # -------- the same sweep-only region with Philox4x32-10 (the library default is 7 rounds)
    philox10_value = None
    if not args.rounds and world == 1:
        sim10 = nat.Sim(graph, E, seed=31337, replica_offset=rank * E, planes=args.planes, rounds=10)
        sim10.sweeps(betas[: max(1, len(betas) // 10)])
        sim10.reset_stats()
        barrier()
        sim10.sweeps(betas)
        barrier()
        s10 = sim10.stats()
        philox10_value = float(s10["flip_attempts"]) / (s10["sweep_device_ms"] * 1e-3)
        sim10.close()

    # -------- weak scaling beside it: 1024 replicas on every GPU (what round 1 reported as `value`)
    weak_value = None
    if world > 1:
        simw = nat.Sim(graph, E_total, seed=31337, replica_offset=rank * E_total, planes=args.planes,
                       rounds=args.rounds)
        simw.sweeps(betas[: max(1, len(betas) // 10)], per_sweep_energies=True)
        simw.reset_stats()
        barrier()
        simw.sweeps(betas, per_sweep_energies=True)
        barrier()
        sw = simw.stats()
        weak_value = sum_over_ranks(float(sw["flip_attempts"])) / (max_over_ranks(sw["sweep_device_ms"]) * 1e-3)
        simw.close()

    # -------- e2e: the public API with host buffers; the ranks shard the experiments exactly as
    # above (Lattice.distributed), every rank reads back its own rows
    if len(w["dims"]) == 3 or args.e2e_full:
        lat = pkg.Lattice.torus(w["dims"], j=w["j0"], pmj=w["pmj"], j_seed=2024, seed_gen=31337, device=local)
        lat.linear_annealing = True
        if world > 1:
            lat.distributed = True
            lat.gather_results = False
        rng = np.random.default_rng(0)
        init = rng.integers(0, 2, n).astype(bool)
        stops = [(0, w["beta"][0]), (w["sweeps"], w["beta"][1])]

        def step_e2e():
            lat.set_initial_state(init)  # N bools H2D inside the call
            en, stt = lat.run_monte_carlo_annealing_and_get_energies(stops, w["sweeps"], E_total, only_basic_moves=True)
            return float(en[0, -1]) + float(stt[0, 0])

        for _ in range(min(args.warmup, 2)):
            step_e2e()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step_e2e()
        barrier()
        e2e_s = max_over_ranks(time.perf_counter() - t0)
        e2e = {"value": E_total * n * w["sweeps"] * args.steps / e2e_s, "unit": "flips/s",
               "h2d_bytes_per_step": int(world * (n + 16 * len(stops))),
               "d2h_bytes_per_step": int(E_total * w["sweeps"] * 8 + E_total * n),
               "ms_per_step": 1e3 * e2e_s / args.steps,
               "api": "Lattice.run_monte_carlo_annealing_and_get_energies (host buffers in/out; "
                      "experiments sharded over the ranks, bytes summed over the ranks)"}
    else:
        e2e = None

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r = oracle_sample(w, 1, 0)
        cpu = {"value": r["value"], "unit": "flips/s", "cores": r["cores"], "kind": "port",
               "sample": r["sample"]}

    if rank == 0:
        line = {
            "metric": "spin_flip_attempts_per_sec", "value": value, "unit": "flips/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u32 bit-sliced (1 bit per spin per replica)",
            "data": "synthetic",
            "config": {"workload": args.workload + ": " + w["desc"], "replicas_total": E_total,
                       "replicas_per_gpu": E,
                       "parallelism": f"replicas sharded x{world} (no collective)",
                       "l2": "256 MiB flush between steps; within a step the %d MiB state is L2-resident by design"
                             % (n * E // 8 >> 20) if n * E / 8 < 100e6 else "state larger than L2",
                       "msc_planes": args.planes or 6, "philox_rounds": args.rounds or 7},
            "wall_ms_per_step": 1e3 * wall / args.steps,
            "sweep_only_value": sweep_only_value,
            "sweep_only_value_philox10": philox10_value,
            "weak_value": weak_value,
            "weak_note": "all ranks' flips/s with 1024 replicas on EVERY GPU (round 1's `value`)" if weak_value else None,
            "roofline": roofline,
            "cpu_baseline": cpu,
            "e2e": e2e,
            "gpu_launches": int(launches),
            "clocks": clocks,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--planes", type=int, default=0)
    ap.add_argument("--rounds", type=int, default=0)
    ap.add_argument("--sweeps", type=int, default=0, help="override sweeps per step (profiling)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ref-sample-sweeps", type=int, default=0,
                    help="reference arm: timesteps per step of the bounded CPU sample (0 = sized to ~10 s)")
    ap.add_argument("--e2e-full", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the energies and a sample of the states of the last timed step to DIR/*.npy")
    args = ap.parse_args()
    w = dict(WORKLOADS[args.workload])
    if args.dump_outputs and (args.impl == "reference" or w.get("kind")):
        raise SystemExit("--dump-outputs covers the replica workloads of the b200 arm (c2, c3, tiny)")
    if args.sweeps:
        w["sweeps"] = args.sweeps
        w["desc"] += f" [sweeps/step overridden to {args.sweeps}]"
    world, rank, local = dist_setup(args.gpus)
    if args.impl == "reference":
        run_reference(args, w, world, rank)
    elif w.get("kind") == "tempering":
        run_tempering(args, w, world, rank, local)
    elif w.get("kind") == "single":
        run_single(args, w, world, rank, local)
    else:
        run_b200(args, w, world, rank, local)


if __name__ == "__main__":
    main()
