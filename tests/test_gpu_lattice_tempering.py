"""Parallel tempering on square and cubic tori (LatticeTempering, native.Tempering on a 2D / 3D
torus) compared bit for bit with the scalar mirror (oracle/msc_mirror.c: msc_mirror_pt_ex) on the
device, at every instantiation and launch shape the library picks (run with -m gpu on a B200).

A lattice ladder runs its own kernels: the thread-block-cluster chunk with per-replica threshold
tables, k_sweep_stencil_cluster<DIM, PMJ, 6, ROUNDS, V, ACC, PERBETA = true> (with ACC its last
sweep leaves the swap cycle's satisfied-bond counts), k_sweep_stencil_perbeta + k_nsat_stencil
above the cluster limit, k_pt_cycle (energies, time averages, swaps, per-pair counters, replica ->
slot map, bit-sliced tables) and k_pt_gather_rows for the slot-ordered samples.  The swaps couple
every replica word, so every case runs the mirror on the whole ladder and compares the samples, the
time-averaged energies, the total swap count, the final slot permutation and the per-pair attempts
and accepts.  Every run records its kernels (torch.profiler) and asserts the instantiations and
cluster sizes that the launcher's rules, restated below, give (none of these rules depends on the
SM count); each case also asserts the branch it exists for, so a case that loses its path fails
under its own name.
"""
import json
import os
import re
import subprocess
import sys
import tempfile
from dataclasses import dataclass, field

import numpy as np
import pytest

from mirror_check import instances, pow2_ceil

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SW_MAX_ITEMS = ((1 << 7) - 1) // 6          # msc_device.cuh: fused counter capacity per thread
ALL_CLUSTER = {(D, P, 6, R, V, acc, True) for D in (2, 3) for P in (True, False) for R in (7, 10)
               for V in (1, 2, 4) for acc in (True, False) if not (V == 4 and acc)}
ALL_PERBETA = {(D, P, R, V, False) for D in (2, 3) for P in (True, False) for R in (7, 10) for V in (1, 2, 4)}
KNOBS = ("ISING_PT_NO_FUSED_COUNTS", "ISING_NO_PDL", "ISING_NO_CLUSTER", "ISING_CLUSTER_MAX",
         "ISING_CLUSTER_WORDS")


# ---------------------------------------------------------------------------------------------
# the launcher's dispatch restated (api_sim.cu: sim_enqueue_sweeps_counting, sim_sweeps_coop;
# sweep_cluster.cu: launch_sweeps_stencil_cluster, cluster_launch, cluster_launch_n;
# sweep_stencil.cu: launch_sweep_stencil, launch_nsat_stencil)
# ---------------------------------------------------------------------------------------------
def cluster_ctas(dims, W, V, ncta, acc):
    """CTAs of k_sweep_stencil_cluster launched for `ncta`, or None when cluster_launch_n declines"""
    Lxh, rows = dims[0] // 2, int(np.prod(dims[1:]))
    groups = W // V
    wx = 32 if groups >= 32 else pow2_ceil(groups)
    by_row = pow2_ceil(Lxh)
    if wx * by_row > 256:
        by_row = 256 // wx
    per_row = wx * by_row
    want = -(-rows * per_row // ncta)
    threads = max(pow2_ceil(min(want, 256)), per_row, 32)
    rpb = threads // per_row
    if rpb == 0:
        return None
    g = min(-(-rows // rpb), ncta)
    if acc:
        items = -(-rows // (g * rpb)) * -(-Lxh // by_row)
        if items >= SW_MAX_ITEMS or by_row * rpb < V:
            return None
    return g


def dispatch(dims, E, env):
    """the path of a tempering chunk on a sim of E replicas: cluster (counted or not, V, CTAs) or
    one launch per colour phase (V)"""
    halfN = int(np.prod(dims)) // 2
    W = -(-E // 32)
    words = halfN * W
    max_words = int(env.get("ISING_CLUSTER_WORDS", 16384))
    max_cta = int(env.get("ISING_CLUSTER_MAX", 16))
    if "ISING_NO_CLUSTER" not in env and words <= max_words:
        V = 1
        if words > 4096 and W % 2 == 0:
            V = 2
        if words > 8192 and W % 4 == 0:
            V = 4

        def ctas(acc):
            if words > 2048 and max_cta >= 16:
                g = cluster_ctas(dims, W, V, 16, acc)
                if g is not None:
                    return g
            return cluster_ctas(dims, W, V, 8 if max_cta >= 8 else max(1, max_cta), acc)

        counted = "ISING_PT_NO_FUSED_COUNTS" not in env and words <= 8192 and ctas(True) is not None
        return dict(path="cluster", V=V, counted=counted, ctas=ctas(counted), W=W, words=words)
    V = 4 if W % 4 == 0 else 2 if W % 2 == 0 else 1
    return dict(path="phase", V=V, counted=False, ctas=None, W=W, words=words)


def chunks(timesteps, swap, sample):
    """sweep counts of the chunks of ising_pt_timesteps_sample (tempering.rs:156-222)"""
    out, remaining, to_swap, to_sample = [], timesteps, swap, sample
    while remaining:
        t = min(to_sample, to_swap, remaining)
        out.append(t)
        to_sample -= t
        to_swap -= t
        remaining -= t
        to_swap = to_swap or swap
        to_sample = to_sample or sample
    return out


def expected_kernels(dims, pmj, rounds, E, env, chunk_list):
    """{kernel: instantiations} the chunks of a ladder must run"""
    D = dispatch(dims, E, env)
    DIM, V, W = len(dims), D["V"], D["W"]
    want = {"k_sweep_stencil_cluster": set(), "k_sweep_stencil_perbeta": set(), "k_nsat_stencil": set()}
    if D["path"] == "phase":
        want["k_sweep_stencil_perbeta"].add((DIM, pmj, rounds, V, False))
    elif D["counted"]:
        want["k_sweep_stencil_cluster"].add((DIM, pmj, 6, rounds, V, True, True))
        if any(t > 4096 for t in chunk_list):    # split: the leading part runs uncounted
            want["k_sweep_stencil_cluster"].add((DIM, pmj, 6, rounds, V, False, True))
    else:
        want["k_sweep_stencil_cluster"].add((DIM, pmj, 6, rounds, V, False, True))
    if not D["counted"]:
        want["k_nsat_stencil"].add((DIM, pmj, 4 if W % 4 == 0 else 2 if W % 2 == 0 else 1))
    return D, want


# ---------------------------------------------------------------------------------------------
# kernels and cluster sizes from the profiler
# ---------------------------------------------------------------------------------------------
def launched_grids(fn):
    """(fn(), kernel names, {name: set of grid.x}) of the CUDA kernels launched meanwhile"""
    import torch
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = sorted({e.name for e in prof.events()})
    grids = {}
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            trace = json.load(f)
    for ev in trace.get("traceEvents", []):
        if ev.get("cat") == "kernel" and "grid" in ev.get("args", {}):
            grids.setdefault(ev["name"], set()).add(int(ev["args"]["grid"][0]))
    return out, names, grids


def short(names):
    return {m.group(1) for n in names for m in [re.search(r"\b(k_\w+)", n)] if m}


def cluster_grid(grids):
    """grid sizes of the k_sweep_stencil_cluster launches"""
    return set().union(*[g for n, g in grids.items() if "k_sweep_stencil_cluster" in n] or [set()])


# ---------------------------------------------------------------------------------------------
# the runs
# ---------------------------------------------------------------------------------------------
@dataclass
class Case:
    name: str
    dims: tuple
    R: int
    pmj: bool
    j0: float
    rounds: int
    timesteps: int
    swap: int
    sample: int
    seed: int
    reach: dict = field(default_factory=dict)   # dispatch property -> value
    beta_hi: float = 1.0

    @property
    def betas(self):
        """an even ladder from 0.1 towards beta_hi, its steps no wider than 0.6 / sqrt(N), so that
        neighbouring energies overlap and swaps happen on large lattices too"""
        step = min((self.beta_hi - 0.1) / (self.R - 1), 0.6 / np.sqrt(np.prod(self.dims)))
        return 0.1 + step * np.arange(self.R)


def env_knobs():
    return {k: v for k, v in os.environ.items() if k in KNOBS}


def torus(native, dims, pmj, j0, j_seed=7):
    return native.Graph.torus(native.Context.get(0), dims, j0=j0, pmj=pmj, j_seed=j_seed)


def compare_ladder(label, got, ref):
    """got / ref: (states, energies, total swaps, slot_of_cfg, attempts, accepts)"""
    st, en, sw, sl, att, acc = got
    st_r, en_r, sw_r, sl_r, att_r, acc_r = ref
    assert sw_r > 0, f"{label}: the mirror swapped nothing"
    if st is not None:
        assert st.shape == st_r.shape, (label, st.shape, st_r.shape)
        bad = np.argwhere(st != st_r)
        assert len(bad) == 0, f"{label}: {len(bad)} sample spins differ, first (slot, sample, site) {bad[0]}"
    bad = np.flatnonzero(en != en_r)
    assert len(bad) == 0, f"{label}: {len(bad)} energies differ, first slot {bad[0]}: {en[bad[0]]} vs {en_r[bad[0]]}"
    assert sw == sw_r, f"{label}: {sw} swaps vs {sw_r}"
    assert (sl == sl_r).all(), f"{label}: slot permutations differ"
    assert (att == att_r).all(), f"{label}: per-pair attempts differ at pairs {np.flatnonzero(att != att_r)[:8]}"
    assert (acc == acc_r).all(), f"{label}: per-pair accepts differ at pairs {np.flatnonzero(acc != acc_r)[:8]}"


def run_case(native, oracle, case):
    """One ladder through ising_pt_timesteps_sample against msc_mirror_pt_ex.  -> kernel names"""
    env = env_knobs()
    g = torus(native, case.dims, case.pmj, case.j0, case.seed)
    assert g.kind == len(case.dims) and g.integer_classes
    cl = chunks(case.timesteps, case.swap, case.sample)
    D, want = expected_kernels(case.dims, case.pmj, case.rounds, case.R, env, cl)
    for k, v in case.reach.items():
        if k == "split":
            assert any(t > 4096 for t in cl) == v, (case.name, cl)
        elif k == "one_sweep_chunks":
            assert cl.count(1) >= v, (case.name, cl)
        elif not env:       # a knob moves the case off its branch on purpose (test_knob_changes_no_bit)
            assert D[k] == v, f"{case.name}: reaches {k} = {D[k]}, meant for {v} ({D})"
    label = (f"{case.name} [{'x'.join(map(str, case.dims))} x {case.R}, {'pmj' if case.pmj else 'uniform'} "
             f"j0={case.j0} R={case.rounds}, {D['path']} V={D['V']}{' counted' if D['counted'] else ''}]")
    pt = native.Tempering(g, case.betas, case.seed, rounds=case.rounds)
    (states, energies), names, grids = launched_grids(
        lambda: pt.timesteps_sample(case.timesteps, replica_swap_freq=case.swap, sampling_freq=case.sample))
    att, acc = pt.pair_stats()
    got = (states, energies, pt.total_swaps(), pt.slots(), att, acc)
    pt.close()
    k = short(names)
    print(f"{label}: {sorted(k)}, cluster grids {sorted(cluster_grid(grids))}", flush=True)
    for kern, inst in want.items():
        seen = instances(names, kern)
        assert seen == inst, (label, kern, sorted(seen), "expected", sorted(inst))
    assert "k_pt_cycle" in k, (label, sorted(k))
    assert ("k_pt_gather_rows" in k) == (case.timesteps >= case.sample), (label, sorted(k))
    if D["path"] == "cluster":
        assert cluster_grid(grids) == {D["ctas"]}, (label, "cluster CTAs", grids, "expected", D["ctas"])
    a, b, j = g.edges()
    ref = oracle.msc_mirror_pt_ex(a, b, j, g.nvars, g.colors(), case.betas, case.seed, case.timesteps,
                                  case.swap, case.sample, rounds=case.rounds)
    compare_ladder(label, got, ref)
    return names


# shapes: (name, dims, R, reach); each runs over (+-J, uniform) x Philox-7 / 10
SHAPES = [
    ("c3d_v1_counted_8cta", (8, 8, 8), 64, dict(path="cluster", V=1, counted=True, ctas=8)),
    ("c3d_v1_counted_16cta", (12, 12, 12), 128, dict(path="cluster", V=1, counted=True, ctas=16)),
    ("c2d_v1_counted", (16, 16), 32, dict(path="cluster", V=1, counted=True)),
    ("c3d_v2_counted", (16, 16, 16), 128, dict(path="cluster", V=2, counted=True, words=8192)),
    ("c2d_v2_counted", (64, 64), 128, dict(path="cluster", V=2, counted=True, words=8192)),
    ("c3d_v1_uncounted", (16, 16, 24), 96, dict(path="cluster", V=1, counted=False)),
    ("c2d_v1_uncounted", (128, 64), 96, dict(path="cluster", V=1, counted=False)),
    ("c3d_v2_uncounted", (16, 16, 16), 192, dict(path="cluster", V=2, counted=False)),
    ("c2d_v2_uncounted", (64, 64), 192, dict(path="cluster", V=2, counted=False)),
    ("c3d_v4", (16, 16, 16), 256, dict(path="cluster", V=4, counted=False, words=16384)),
    ("c2d_v4", (128, 64), 128, dict(path="cluster", V=4, counted=False, words=16384)),
    ("p3d_v1", (32, 32, 34), 32, dict(path="phase", V=1)),
    ("p3d_v2", (32, 32, 32), 64, dict(path="phase", V=2)),
    ("p3d_v4", (32, 32, 32), 128, dict(path="phase", V=4)),
    ("p2d_v1", (256, 256), 32, dict(path="phase", V=1)),
    ("p2d_v2", (256, 256), 64, dict(path="phase", V=2)),
    ("p2d_v4", (256, 256), 128, dict(path="phase", V=4)),
]
# (timesteps, swap, sample): swap every sweep; sample coprime to swap (1-sweep chunks, cycles
# without a swap, timesteps not a multiple of the sample cadence); longer chunks
CADENCES = [(6, 1, 2), (7, 2, 3), (8, 4, 3), (6, 3, 2)]
UNIFORM_J = (-1.0, 1.0, -0.5, 2.0)            # ferro, antiferro, |J| = 0.5, |J| = 2
PMJ_J = (1.0, 0.5, 2.0)
CASES = []
for i, (nm, dims, R, reach) in enumerate(SHAPES):
    for k, (pmj, rounds) in enumerate(((True, 7), (False, 7), (True, 10), (False, 10))):
        j0 = PMJ_J[(i + k) % 3] if pmj else UNIFORM_J[(i + k) % 4]
        T, sw, sa = CADENCES[(i + k) % 4]
        CASES.append(Case(f"{nm}_{'pmj' if pmj else 'uni'}_r{rounds}", dims, R, pmj, j0, rounds, T, sw, sa,
                          100 + 4 * i + k, reach, beta_hi=1.0 / abs(j0) ** 0.5))
CASES += [
    # k_pt_cycle past its first pass: 96 table warps, e32 = 1024, 1023 pairs
    Case("r1024_4cubed", (4, 4, 4), 1024, True, 1.0, 7, 6, 1, 4, 301,
         dict(path="cluster", V=1, counted=True, words=1024), beta_hi=2.0),
    # R = 1100: W = 35, ragged last word, 1099 pairs; N = 216 (byte path of the sample gather)
    Case("r1100_6cubed", (6, 6, 6), 1100, False, -1.0, 10, 7, 2, 3, 302,
         dict(path="cluster", V=1, counted=True, W=35), beta_hi=1.5),
    Case("r1024_16cubed_phase", (16, 16, 16), 1024, True, 0.5, 7, 4, 2, 3, 303, dict(path="phase", V=4)),
    # sample cadence coprime to the swap cadence: 1-sweep counted chunks, cycles without a swap
    Case("coprime_cadence_2d", (16, 16), 64, True, 1.0, 7, 13, 3, 2, 304,
         dict(path="cluster", counted=True, one_sweep_chunks=2)),
    # a chunk of 4099 sweeps: 3 uncounted, then 4096 counted
    Case("split_chunk_3d", (4, 4, 4), 32, True, 1.0, 7, 4101, 4099, 4100, 305,
         dict(path="cluster", counted=True, split=True), beta_hi=0.6),
    Case("split_chunk_2d", (8, 8), 64, False, 1.0, 10, 4200, 4099, 4150, 306,
         dict(path="cluster", counted=True, split=True), beta_hi=0.6),
    # N % 16 != 0: the byte path of k_pt_gather_rows (6 x 10 = 60 sites, 6^3 = 216)
    Case("bytes_6x10", (6, 10), 64, True, 2.0, 7, 9, 2, 1, 307, dict(path="cluster", counted=True)),
    Case("bytes_6cubed", (6, 6, 6), 96, False, 0.5, 10, 10, 3, 4, 308, dict(path="cluster", counted=True)),
]
CASE = {c.name: c for c in CASES}


# ---------------------------------------------------------------------------------------------
# shards of one ladder in one process (word_lo = 1 and 2)
# ---------------------------------------------------------------------------------------------
SHARD_SPLITS = (((0, 40), (40, 100)), ((0, 64), (64, 100)))


def check_shards(native, oracle, dims, pmj, j0, path):
    """[0, 40) + [40, 100) and [0, 64) + [64, 100) of a 100-beta ladder, stepped by hand with
    concatenated energies (what the all-gather does), equal the unsharded ladder, and that ladder
    equals the mirror: energies of every step, slots, total swaps, pair statistics, states"""
    env = env_knobs()
    R, t, steps, seed = 100, 2, 5, 401
    betas = np.geomspace(0.1, 1.0, R)
    g = torus(native, dims, pmj, j0, 5)
    full = native.Tempering(g, betas, seed)
    shards = [[native.Tempering(g, betas, seed, cfg_lo=lo, cfg_hi=hi) for lo, hi in split]
              for split in SHARD_SPLITS]
    for split in SHARD_SPLITS:
        for lo, hi in split:
            E = min(((hi + 31) // 32 - lo // 32) * 32, R - (lo // 32) * 32)
            assert dispatch(dims, E, env)["path"] == path, (dims, lo, hi, dispatch(dims, E, env))
    acc = np.zeros(R)
    seen_names = []
    for step in range(steps):
        cfg_of_slot = np.argsort(full.slots())
        ef = full.sweeps(t)
        for s in range(R):
            acc[s] += ef[cfg_of_slot[s]] * float(t)
        full.swap_step(ef)
        for si, pair in enumerate(shards):
            (es, names, _) = launched_grids(lambda: np.concatenate([p.sweeps(t) for p in pair]))
            assert (es == ef).all(), f"split {SHARD_SPLITS[si]} step {step}: energies differ"
            _, names2, _ = launched_grids(lambda: [p.swap_step(es) for p in pair])
            seen_names += names + names2
    k = short(seen_names)
    assert "k_pt_swap" in k and "k_pt_cycle" not in k, sorted(k)
    assert ("k_sweep_stencil_cluster" in k) == (path == "cluster"), sorted(k)
    assert ("k_sweep_stencil_perbeta" in k) == (path == "phase"), sorted(k)
    st_full = full.local_states()
    att_f, acc_f = full.pair_stats()
    for split, pair in zip(SHARD_SPLITS, shards):
        for p in pair:
            assert (p.slots() == full.slots()).all(), f"{split}: slots differ"
            assert p.total_swaps() == full.total_swaps(), f"{split}: swap counts differ"
            att, accp = p.pair_stats()
            assert (att == att_f).all() and (accp == acc_f).all(), f"{split}: pair statistics differ"
        assert (np.concatenate([p.local_states() for p in pair]) == st_full).all(), f"{split}: states differ"
    a, b, j = g.edges()
    T = steps * t
    ref = oracle.msc_mirror_pt_ex(a, b, j, g.nvars, g.colors(), betas, seed, T, t, T)
    slots = full.slots()
    got = (st_full[np.argsort(slots)][:, None, :], acc / T, full.total_swaps(), slots, att_f, acc_f)
    compare_ladder(f"unsharded {dims} x {R}", got, ref)
    for pair in shards:
        for p in pair:
            p.close()
    full.close()
    return seen_names


# ---------------------------------------------------------------------------------------------
# the Python face
# ---------------------------------------------------------------------------------------------
def check_lattice_tempering(native, oracle):
    """LatticeTempering over a +-J cubic edge list: recognised as a stencil, runs the checkerboard
    kernels, and qmc_timesteps_sample equals the mirror at the seed the class passes on"""
    import pyisingmontecarlo_b200 as pkg

    L = 8
    rng = np.random.default_rng(12)
    signs = np.where(rng.random((L ** 3, 3)) < 0.5, -1.0, 1.0)
    edges = oracle.cubic_edges(L, lambda n, d: signs[n, d])
    lt = pkg.LatticeTempering(edges, seed=8128)
    betas = np.geomspace(0.15, 1.3, 40)
    for b in betas:
        lt.add_graph(0.0, 0.0, float(b))
    (states, energies), names, _ = launched_grids(lambda: lt.qmc_timesteps_sample(11, replica_swap_freq=2,
                                                                                 sampling_freq=4))
    g = lt._graph
    assert g.kind == 3 and g.dims == (L, L, L), (g.kind, g.dims)
    k = short(names)
    assert "k_sweep_stencil_cluster" in k and "k_pt_cycle" in k and "k_sweep_general" not in k, sorted(k)
    a, b, j = g.edges()
    ref = oracle.msc_mirror_pt_ex(a, b, j, g.nvars, g.colors(), betas, lt._seed, 11, 2, 4)
    pt = lt._pt
    att, acc = pt.pair_stats()
    compare_ladder("LatticeTempering 8^3 +-J x 40", (states, energies, lt.get_total_swaps(), pt.slots(), att, acc),
                   ref)
    return names


# ---------------------------------------------------------------------------------------------
# the device runs, in child processes
# ---------------------------------------------------------------------------------------------
# Every check runs in one child process and the tests below report its outcomes: the profiler
# attaches CUPTI to the process it runs in, and later profiler sessions in the same process can miss
# kernels that other tests load meanwhile (DESIGN.md section 2, item 7).
CHECKS = {f"case/{c.name}": (run_case, (c,)) for c in CASES}
CHECKS["shards/cluster"] = (check_shards, ((8, 8, 8), True, 1.0, "cluster"))
CHECKS["shards/phase"] = (check_shards, ((32, 32, 34), False, -1.0, "phase"))
CHECKS["python_face"] = (check_lattice_tempering, ())


def run_checks(path, names):
    """child: run the named checks, write {name: "ok" or the traceback} and the union of the
    sweep instantiations recorded to path"""
    import time
    import traceback

    import oracle_lib
    from pyisingmontecarlo_b200 import _native as nat

    nat.Context.get(0)
    res, seen = {}, {"k_sweep_stencil_cluster": set(), "k_sweep_stencil_perbeta": set()}
    for name in names:
        fn, args = CHECKS[name]
        t0 = time.time()
        try:
            kn = fn(nat, oracle_lib, *args)
            for kern in seen:
                seen[kern] |= instances(kn or [], kern)
            res[name] = "ok"
        except Exception:
            res[name] = traceback.format_exc()
        print(name, "ok" if res[name] == "ok" else "FAILED", f"{time.time() - t0:.1f} s", flush=True)
    with open(path, "w") as f:
        json.dump({"outcomes": res, "instances": {k: sorted(v) for k, v in seen.items()}}, f)


_CHILD = (
    "import sys\n"
    "sys.path[:0] = [%r, %r]\n"
    "import test_gpu_lattice_tempering as T\n"
    "T.run_checks(sys.argv[1], sys.argv[2:])\n") % (ROOT, os.path.join(ROOT, "tests"))


def child(names, env=None, timeout=1500):
    """{"outcomes": {name: outcome}, "instances": {...}} of the named checks, run in a child process
    (the ISING_ knobs from env only; ISING_B200_LIB, which names the library, is kept)"""
    e = {k: v for k, v in os.environ.items() if not k.startswith("ISING_") or k == "ISING_B200_LIB"}
    e.update(env or {})
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "outcomes.json")
        res = subprocess.run([sys.executable, "-c", _CHILD, path] + list(names), env=e, timeout=timeout,
                             capture_output=True, text=True)
        assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-6000:]
        with open(path) as f:
            return json.load(f)


@pytest.fixture(scope="module")
def results(native, oracle):
    return child(CHECKS)


def _report(results, name):
    assert results["outcomes"][name] == "ok", results["outcomes"][name]


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_lattice_ladder_matches_mirror(results, case):
    _report(results, f"case/{case.name}")


@pytest.mark.parametrize("path", ["cluster", "phase"])
def test_shards_equal_unsharded_ladder_and_mirror(results, path):
    """shards at word_lo = 1 and 2 (configurations [40, 100) and [64, 100))"""
    _report(results, f"shards/{path}")


def test_lattice_tempering_class_matches_mirror(results):
    _report(results, "python_face")


def test_every_instantiation_ran(results):
    """the runs above cover all 40 reachable tempering instantiations of the cluster chunk and all
    24 of the per-phase per-replica sweep"""
    for kern, every in (("k_sweep_stencil_cluster", ALL_CLUSTER), ("k_sweep_stencil_perbeta", ALL_PERBETA)):
        seen = {tuple(t) for t in results["instances"][kern]}
        assert seen == every, (kern, "missing", sorted(every - seen), "unexpected", sorted(seen - every))


# knob -> (value, the cases run under it in one child process)
KNOB_RUNS = {
    "ISING_PT_NO_FUSED_COUNTS": ("1", ["c3d_v1_counted_8cta_pmj_r7", "c2d_v2_counted_uni_r10", "r1024_4cubed",
                                       "split_chunk_3d"]),
    "ISING_NO_PDL": ("1", ["c3d_v1_counted_16cta_pmj_r10", "c2d_v4_uni_r7", "p3d_v2_pmj_r7", "r1100_6cubed"]),
    "ISING_NO_CLUSTER": ("1", ["c3d_v1_counted_8cta_uni_r7", "c2d_v1_uncounted_pmj_r10", "c3d_v4_pmj_r7"]),
    "ISING_CLUSTER_MAX": ("8", ["c3d_v1_counted_16cta_pmj_r7", "c3d_v2_counted_uni_r7", "c2d_v2_uncounted_pmj_r7"]),
    "ISING_CLUSTER_WORDS": ("4096", ["c3d_v2_counted_pmj_r10", "c2d_v2_counted_uni_r7"]),
}


@pytest.mark.parametrize("knob", list(KNOB_RUNS))
def test_knob_changes_no_bit(native, oracle, knob):
    """each A/B knob, read once per process, in its own child: no bit changes, and the knob takes
    effect on every case listed (the restated dispatch changes, and each run asserts that the kernels
    and cluster sizes follow it).  ISING_NO_PDL is the exception: it only drops the programmatic
    stream serialization attribute of the launches, which changes no kernel, instantiation or grid
    the profiler records, so that child checks the bits alone."""
    value, names = KNOB_RUNS[knob]
    for n in names:
        c = CASE[n]
        before, after = dispatch(c.dims, c.R, {}), dispatch(c.dims, c.R, {knob: value})
        if knob == "ISING_PT_NO_FUSED_COUNTS":
            assert before["counted"] and not after["counted"], (n, before, after)
        elif knob == "ISING_NO_CLUSTER":
            assert before["path"] == "cluster" and after["path"] == "phase", (n, before, after)
        elif knob == "ISING_CLUSTER_MAX":
            assert before["ctas"] > 8 and after["ctas"] == 8, (n, before, after)
        elif knob == "ISING_CLUSTER_WORDS":
            assert before["words"] == 8192 and before["path"] == "cluster" and after["path"] == "phase", (n, after)
    res = child([f"case/{n}" for n in names], {knob: value})
    for n in names:
        _report(res, f"case/{n}")
