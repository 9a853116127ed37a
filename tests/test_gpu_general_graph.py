"""The general-graph sweep (k_sweep_general, csrc/sweep_general.cu) and its energy count
(k_nsat_general) compared bit for bit with the scalar mirror (oracle/msc_mirror.c) on the device,
at every instantiation and launch shape the library picks, and BASELINE config 4 at full size (run
with -m gpu on a B200).

Every general graph and every general_layout sim runs on these kernels.  A decision depends only
on (seed, site, global replica word, sweep), so msc_mirror(E = 32 k, replica_offset = 32 w)
reproduces words w .. w + k - 1 of a larger run: large runs are checked word by word.  Every run
records its kernels (torch.profiler) and asserts the k_sweep_general<K, ROUNDS, PERBETA, DEG, V>
instantiations that the launcher's rules, restated below with the device's SM count, give; each
case also asserts the branch it exists for, so a case that loses its path fails under its own name.
"""
import json
import os
import subprocess
import sys
import tempfile
from dataclasses import dataclass, field

import numpy as np
import pytest

from mirror_check import (assert_same, check_words, device_sms, families, instances, launched,
                          pow2_ceil, random_regular, word_bits)

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GEN_MAX_DEG = 15


# ---------------------------------------------------------------------------------------------
# the launcher's dispatch restated (api_core.cu: ensure_general_on_device; api_sim.cu:
# ising_sim_create_ex; sweep_general.cu: gen_launch, gen_launch_degree, launch_nsat_general)
# ---------------------------------------------------------------------------------------------
def gen_launch(W, count, sms):
    """launch shape of k_sweep_general over one (colour, degree) group of `count` sites"""
    V = 2 if W % 2 == 0 else 1
    groups = W // V
    wx = 32 if groups >= 32 else pow2_ceil(groups)
    by = 256 // wx
    blocks = min(-(-count // by), 16 * sms)
    return dict(V=V, wx=wx, by=by, blocks=blocks, site_passes=-(-count // (blocks * by)),
                w0_passes=-(-W // (wx * V)))


def gen_deg(K, rounds, deg):
    """DEG template argument: compile-time degree for 3 / 4 / 6 at the default (K, ROUNDS) only"""
    return deg if K == 6 and rounds == 7 and deg in (3, 4, 6) else 0


def nsat_launch(W, nvars, sms):
    """launch shape of k_nsat_general"""
    wx = min(32, pow2_ceil(W))
    by = 256 // wx
    grid = max(1, min(-(-nvars // by), 8 * sms))
    return dict(wx=wx, by=by, grid=grid, site_passes=-(-nvars // (grid * by)), w0_passes=-(-W // wx))


def degrees(nvars, a, b):
    """adjacency entries per site (a multi-edge counts twice)"""
    return np.bincount(a.astype(np.int64), minlength=nvars) + np.bincount(b.astype(np.int64), minlength=nvars)


def gen_groups(colors, deg):
    """{(colour, degree): sites}: one k_sweep_general launch each per sweep"""
    keys, counts = np.unique(colors.astype(np.int64) * (GEN_MAX_DEG + 1) + deg, return_counts=True)
    return {(int(k) // (GEN_MAX_DEG + 1), int(k) % (GEN_MAX_DEG + 1)): int(c) for k, c in zip(keys, counts)}


def sweep_instances(groups, W, K, rounds, perbeta):
    V = 2 if W % 2 == 0 else 1
    return {(K, rounds, perbeta, gen_deg(K, rounds, d), V) for _, d in groups}


# ---------------------------------------------------------------------------------------------
# graphs
# ---------------------------------------------------------------------------------------------
def signs(rng, m):
    return np.where(rng.random(m) < 0.5, -1.0, 1.0)


def mixed_degree_edges():
    """Degrees 0 .. 15 in one graph, +-0.5: six sites of every degree (isolated sites and leaves
    included) among 1200 sites of degree 1 .. 5, and one double bond (sites 0 and 1, counted
    twice towards their degrees)."""
    rng = np.random.default_rng(8)
    target = np.concatenate([[9, 12], np.repeat(np.arange(16), 6), rng.integers(1, 6, 1200)])
    n = len(target)
    if target.sum() % 2:
        target[-1] += 1 if target[-1] < 5 else -1
    pre_a, pre_b = np.array([0, 0]), np.array([1, 1])
    rest = target.copy()
    rest[0] -= 2
    rest[1] -= 2
    while True:
        stubs = np.repeat(np.arange(n), rest)
        rng.shuffle(stubs)
        a, b = stubs[0::2], stubs[1::2]
        if not (a == b).any():
            break
    a, b = np.concatenate([pre_a, a]), np.concatenate([pre_b, b])
    return n, a, b, 0.5 * signs(rng, len(a))


def circulant15(n):
    """15-regular ferromagnet: i ~ i +- 1 .. 7 and i ~ i + n/2 (n even)"""
    i = np.arange(n, dtype=np.int64)
    a = np.concatenate([i for _ in range(7)] + [i[:n // 2]])
    b = np.concatenate([(i + k) % n for k in range(1, 8)] + [i[:n // 2] + n // 2])
    return a, b


def _rr(n, seed, j):
    rng = np.random.default_rng(seed)
    a, b = random_regular(n, 3, rng)
    return n, a, b, (signs(rng, len(a)) if j == "pmj" else np.full(len(a), float(j)))


GRAPHS = {
    # name: (builder -> (nvars, a, b, j)) or torus arguments; general_layout
    "rr3_120k_pmj": (lambda: _rr(120_000, 5, "pmj"), False),
    "rr3_4000_ferro": (lambda: _rr(4000, 6, -1.0), False),
    "rr3_2000_anti": (lambda: _rr(2000, 7, 1.0), False),
    "mixed_half": (mixed_degree_edges, False),
    "torus2d_anti": (dict(dims=(512, 512), j0=1.0), True),
    "torus3d_pmj_half": (dict(dims=(64, 64, 64), j0=0.5, pmj=True, j_seed=3), True),
}
_graph_cache = {}


@dataclass
class G:
    g: object
    general_layout: bool
    edges: tuple
    colors: np.ndarray
    deg: np.ndarray
    groups: dict


def graph(native, name):
    if name not in _graph_cache:
        spec, general = GRAPHS[name]
        ctx = native.Context.get(0)
        if isinstance(spec, dict):
            g = native.Graph.torus(ctx, **spec)
        else:
            n, a, b, j = spec()
            g = native.Graph.from_edges(ctx, n, a, b, j)
        a, b, j = g.edges()
        colors = g.colors()
        deg = degrees(g.nvars, a, b)
        _graph_cache[name] = G(g, general, (a, b, j), colors, deg, gen_groups(colors, deg))
    return _graph_cache[name]


# ---------------------------------------------------------------------------------------------
# 1. shape matrix against the mirror
# ---------------------------------------------------------------------------------------------
BETAS = np.array([0.35, 0.8, 1.2, 1.2])
NSWEEPS = 4             # sweeps of a per-replica-beta run


def replica_betas(E):
    return np.linspace(0.2, 1.6, E)


@dataclass
class Case:
    name: str
    graph: str
    E: int
    seed: int
    perbeta: bool = False
    offset: int = 0
    planes: int = 6
    rounds: int = 7
    words: tuple = None     # None: every replica in one mirror run
    reach: dict = field(default_factory=dict)   # launch-shape property -> value in every group

    @property
    def W(self):
        return -(-self.E // 32)


def _torus_cases(tag, gname, deg):
    out = []
    for E, V in ((1024, 2), (470, 1)):
        W = -(-E // 32)
        for pb in (False, True):
            out.append(Case(f"{tag}_deg{deg}_v{V}" + ("_perbeta" if pb else ""), gname, E, 50 + E % 7 + pb,
                            perbeta=pb, words=(0, W // 2, W - 1),
                            reach=dict(V=V, wx=16, by=16, DEG=deg, min_site_passes=2)))
    return out


CASES = [
    # config 4's graph family at 1.2 * 10^5 sites: every colour group wraps the grid
    Case("rr3_wrap", "rr3_120k_pmj", 2048, 31, words=(0, 31, 63),
         reach=dict(V=2, wx=32, by=8, DEG=3, min_site_passes=2)),
    Case("rr3_wrap_perbeta", "rr3_120k_pmj", 2048, 32, perbeta=True, words=(0, 31, 63),
         reach=dict(V=2, wx=32, by=8, DEG=3, min_site_passes=2)),
    # the replica-word loop: two passes with 31 idle lanes in the second, three passes
    Case("ragged_w33", "rr3_4000_ferro", 1051, 33, reach=dict(V=1, wx=32, w0_passes=2, DEG=3)),
    Case("ragged_w33_perbeta", "rr3_4000_ferro", 1051, 34, perbeta=True, reach=dict(V=1, wx=32, w0_passes=2, DEG=3)),
    Case("w130", "rr3_2000_anti", 4160, 35, reach=dict(V=2, wx=32, w0_passes=3)),
    # lane widths 16 and 32 with one word per thread
    Case("wx16_v1", "rr3_2000_anti", 470, 36, reach=dict(V=1, wx=16, w0_passes=1)),
    Case("wx32_v1", "rr3_2000_anti", 990, 37, reach=dict(V=1, wx=32, w0_passes=1)),
    # sharded runs: the global word gw0 != 0 enters the Philox counter
    Case("offset_gw0", "rr3_4000_ferro", 200, 38, offset=320, reach=dict(V=1, wx=8)),
    Case("offset_gw0_perbeta", "rr3_4000_ferro", 256, 39, perbeta=True, offset=2048, reach=dict(V=2, wx=4)),
] + _torus_cases("torus2d", "torus2d_anti", 4) + _torus_cases("torus3d", "torus3d_pmj_half", 6)
CASE = {c.name: c for c in CASES}


def check_reach(case, gr, sms):
    """the case still reaches the branch it is meant for, in every (colour, degree) group"""
    for (col, d), count in gr.groups.items():
        sh = gen_launch(case.W, count, sms)
        sh["DEG"] = gen_deg(case.planes, case.rounds, d)
        for k, want in case.reach.items():
            if k == "min_site_passes":
                assert sh["site_passes"] >= want, f"{case.name}: group ({col}, {d}) runs {sh['site_passes']} grid passes"
            else:
                assert sh[k] == want, f"{case.name}: group ({col}, {d}) reaches {k} = {sh[k]}, meant for {want}"


def run_case(native, oracle, sms, case):
    """One run of per-sweep energies against the mirror (all replicas, or case.words), bit for
    bit; energies() too.  Asserts the instantiations.  Returns the kernel names."""
    gr = graph(native, case.graph)
    g = gr.g
    check_reach(case, gr, sms)
    label = f"{case.name} [{g.nvars} sites x {case.E}, K={case.planes} R={case.rounds}]"
    sim = native.Sim(g, case.E, case.seed, replica_offset=case.offset, planes=case.planes, rounds=case.rounds,
                     general_layout=gr.general_layout)
    pb = replica_betas(case.E) if case.perbeta else None
    if case.perbeta:
        sim.set_betas(pb)
    en, names = launched(lambda: sim.sweeps(NSWEEPS if case.perbeta else BETAS, per_sweep_energies=True))
    got = instances(names, "k_sweep_general")
    want = sweep_instances(gr.groups, case.W, case.planes, case.rounds, case.perbeta)
    print(f"{label}: {sorted(got)}")
    assert got == want, (label, "k_sweep_general instances", sorted(got), "expected", sorted(want))
    assert families(names) == {"k_sweep_general", "k_nsat_general"}, (label, names)
    assert (sim.energies() == en[:, -1]).all(), label
    kw = dict(planes=case.planes, rounds=case.rounds)
    if case.words is None:
        st = sim.states()
        a, b, j = gr.edges
        en_ref, st_ref = oracle.msc_mirror(a, b, j, g.nvars, gr.colors, case.E, case.seed,
                                           None if case.perbeta else BETAS, replica_offset=case.offset,
                                           per_sweep=True, per_replica_beta=pb,
                                           nsweeps=NSWEEPS if case.perbeta else None, **kw)
        assert_same(st, st_ref, en, en_ref, label, case.offset)
    else:
        packed = sim.packed()
        check_words(oracle, g, case.E, case.seed, NSWEEPS if case.perbeta else BETAS, case.words, en,
                    lambda w: word_bits(packed, w, min(32, case.E - 32 * w)), label, offset=case.offset,
                    edges=gr.edges, per_replica_beta=pb, **kw)
    sim.close()
    return names


MIXED = [(K, R, pb) for K in (5, 6, 7) for R in (7, 10) for pb in (False, True)]


def check_mixed_degrees(native, oracle, sms, K, R, perbeta):
    """Degrees 0 .. 15 with +-0.5 couplings: the run-time-degree kernel (DEG = 0: four counter
    planes, up to eight uphill classes) next to the degree-specialised ones at K = 6, R = 7"""
    gr = graph(native, "mixed_half")
    degs = {d for _, d in gr.groups}
    assert degs == set(range(16)), degs
    assert all(sum(c for (_, d), c in gr.groups.items() if d == dd) >= 6 for dd in range(8, 16))
    a, b, _ = gr.edges
    key = np.minimum(a, b) * gr.g.nvars + np.maximum(a, b)
    assert len(np.unique(key)) < len(key), "no multi-edge"
    case = Case(f"mixed_K{K}_R{R}", "mixed_half", 64 if perbeta else 70, 60 + K + R, perbeta=perbeta,
                planes=K, rounds=R)
    names = run_case(native, oracle, sms, case)
    assert 0 in {t[3] for t in instances(names, "k_sweep_general")}


def check_integer_float_boundary(native, oracle, sms):
    """Max degree 15 stays on the integer kernel (and equals the mirror); one more bond at a
    degree-15 site (degree 16) sends the graph to k_sweep_real (test_gpu_float_path.py checks it)."""
    gr = graph(native, "mixed_half")
    assert gr.g.max_degree == 15 and gr.g.integer_classes
    run_case(native, oracle, sms, Case("max_degree_15", "mixed_half", 40, 71))
    a, b, j = gr.edges
    hub = int(np.flatnonzero(gr.deg == 15)[0])
    other = int(np.flatnonzero(gr.deg == 0)[0])
    ctx = native.Context.get(0)
    g16 = native.Graph.from_edges(ctx, gr.g.nvars, np.append(a, hub), np.append(b, other), np.append(j, 0.5))
    assert g16.max_degree == 16 and g16.integer_classes
    sim = native.Sim(g16, 40, 71)
    _, names = launched(lambda: sim.sweeps([0.5]))
    assert families(names) == {"k_sweep_real"}, names
    sim.close()


# ---------------------------------------------------------------------------------------------
# 2. energies as exact integers: every replica after every sweep
# ---------------------------------------------------------------------------------------------
def int_energies(states, a, b, j):
    """int64 numpy energy (in units of |J|) of every replica"""
    ai, bi = a.astype(np.intp), b.astype(np.intp)
    sg = np.sign(j).astype(np.int64)
    s = states.view(np.int8)
    out = np.empty(len(s), dtype=np.int64)
    for r in range(0, len(s), 256):
        x = s[r:r + 256] * np.int8(2) - np.int8(1)
        out[r:r + 256] = ((x[:, ai] * x[:, bi]).astype(np.int64) * sg).sum(1)
    return out


EXACT = [("w_loop_W130", "rr3_2000_anti", 4160, dict(w0_passes=5)),
         ("grid_wrap", "rr3_120k_pmj", 320, dict(min_site_passes=2)),
         ("degree15_W35", "mixed_half", 1100, dict(w0_passes=2))]


def check_every_replica_every_sweep(native, oracle, sms, name, gname, E, reach):
    """Single-sweep calls with per-sweep energies: every replica's energy equals an int64
    recomputation from the returned states, and so does energies().  This checks k_nsat_general and
    k_energy_from_hist independently of the mirror (its word loop; its grid-stride wrap)."""
    gr = graph(native, gname)
    g = gr.g
    sh = nsat_launch(-(-E // 32), g.nvars, sms)
    for k, want in reach.items():
        assert (sh["site_passes"] >= want) if k == "min_site_passes" else sh[k] == want, (name, sh)
    a, b, j = gr.edges
    jabs = abs(j[0])
    sim = native.Sim(g, E, 90 + E)
    for t, beta in enumerate((0.45, 1.2, 1.2)):
        en, names = launched(lambda: sim.sweeps([beta], per_sweep_energies=True))
        assert "k_nsat_general" in families(names), names
        e_np = int_energies(sim.states(), a, b, j) * jabs
        bad = np.flatnonzero(en[:, 0] != e_np)
        assert len(bad) == 0, (f"{name} sweep {t}: {len(bad)} per-sweep energies differ, first replica "
                               f"{bad[:1]}: {en[bad[:1], 0]} vs {e_np[bad[:1]]}")
        assert (sim.energies() == e_np).all(), f"{name} sweep {t}: energies()"
    sim.close()


def check_nsat_flushes_at_degree_15(native, oracle, sms):
    """A 15-regular ferromagnet large enough that every thread of k_nsat_general counts about 300
    sites: all up, a thread's satisfied bonds (15 per site) pass the 4095 its 12-plane counter holds,
    so the result is right only if the counter is flushed inside the site loop.  Then one sweep of
    the run-time-degree sweep kernel over groups that wrap its grid, checked on words 0 and 31."""
    E, W = 1024, 32
    n = 8 * sms * (256 // 32) * 300
    sh = nsat_launch(W, n, sms)
    assert sh["site_passes"] * 15 > 4095, sh
    a, b = circulant15(n)
    ctx = native.Context.get(0)
    g = native.Graph.from_edges(ctx, n, a, b, np.full(len(a), -1.0))
    assert g.max_degree == 15 and g.integer_classes
    sim = native.Sim(g, E, 2025)
    sim.set_state(np.ones(n, dtype=bool))
    assert (sim.energies() == -float(len(a))).all()
    en, names = launched(lambda: sim.sweeps([0.05], per_sweep_energies=True))   # flips ~5 % of the sites
    assert instances(names, "k_sweep_general") == {(6, 7, False, 0, 2)}, names
    groups = gen_groups(g.colors(), degrees(n, a, b))
    wrapped = sum(c for c in groups.values() if gen_launch(W, c, sms)["site_passes"] >= 2)
    assert wrapped > 0.9 * n, groups
    packed = sim.packed()
    sim.close()
    for w in (0, 31):
        x = packed[a, w] ^ packed[b, w]          # bit b set: bond of replica 32 w + b unsatisfied
        unsat = np.array([np.count_nonzero((x >> np.uint32(bit)) & np.uint32(1)) for bit in range(32)])
        e_np = -float(len(a)) + 2.0 * unsat
        assert (en[32 * w:32 * w + 32, 0] == e_np).all(), (w, en[32 * w:32 * w + 32, 0], e_np)
    assert (en[:, 0] > -float(len(a))).all()


# ---------------------------------------------------------------------------------------------
# 3. BASELINE config 4 at full size
# ---------------------------------------------------------------------------------------------
C4_BETAS = np.geomspace(0.1, 1.5, 64)


def config4(native):
    """bench.py's config 4 graph: random 3-regular, N = 10^6, J = -1 (seed 2026)"""
    import pyisingmontecarlo_b200 as pkg

    if "config4" not in _graph_cache:
        a, b = random_regular(1_000_000, 3, np.random.default_rng(2026))
        g = pkg.Lattice.from_arrays(a, b, np.full(len(a), -1.0)).graph()
        assert g.kind == native.KIND_GENERAL and g.max_degree == 3
        _graph_cache["config4"] = (g, g.edges(), g.colors())
    return _graph_cache["config4"]


def check_config4_sweeps(native, oracle, sms):
    """64 replicas at the ladder's 64 betas (per-replica tables), 10 sweeps: all replicas"""
    g, (a, b, j), colors = config4(native)
    sim = native.Sim(g, 64, 7)
    sim.set_betas(C4_BETAS)
    en, names = launched(lambda: sim.sweeps(10, per_sweep_energies=True))
    assert instances(names, "k_sweep_general") == {(6, 7, True, 3, 2)}, names
    st = sim.states()
    sim.close()
    en_ref, st_ref = oracle.msc_mirror(a, b, j, g.nvars, colors, 64, 7, None, per_replica_beta=C4_BETAS,
                                       nsweeps=10, per_sweep=True)
    assert_same(st, st_ref, en, en_ref, "config 4 sweeps")


def check_config4_ladder(native, oracle, sms):
    """The ladder as bench.py runs it (device-resident timesteps_sample, seed 7, swap every 10):
    states, time-averaged energies, swap count and slot permutation equal msc_mirror_pt"""
    g, (a, b, j), colors = config4(native)
    pt = native.Tempering(g, C4_BETAS, seed=7)
    (states, energies), names = launched(lambda: pt.timesteps_sample(20, replica_swap_freq=10, sampling_freq=20))
    assert instances(names, "k_sweep_general") == {(6, 7, True, 3, 2)}, names
    assert any("k_pt_cycle" in n for n in names) and any("k_build_tables" in n for n in names), names
    swaps, slots = pt.total_swaps(), pt.slots()
    pt.close()
    st_ref, en_ref, swaps_ref, slots_ref = oracle.msc_mirror_pt(a, b, j, g.nvars, colors, C4_BETAS, 7, 20,
                                                                replica_swap_freq=10, sampling_freq=20)
    assert swaps_ref >= 1
    assert swaps == swaps_ref and (slots == slots_ref).all(), (swaps, swaps_ref)
    assert (energies == en_ref).all(), np.flatnonzero(energies != en_ref)
    assert_same(states[:, 0], st_ref[:, 0], None, None, "config 4 ladder")


# ---------------------------------------------------------------------------------------------
# 4. the device runs, in child processes
# ---------------------------------------------------------------------------------------------
# Every check above runs in one child process and the tests below report its outcomes.  The
# profiler attaches CUPTI to the process it runs in, and later sessions in the same process can
# miss kernels that other tests load while it is detached (seen for the row-walk file when this
# file ran before it in one pytest process); a child keeps the pytest process free of CUPTI.
CHECKS = {f"shape/{c.name}": (run_case, (c,)) for c in CASES}
CHECKS.update({f"mixed/{K}/{R}/{pb}": (check_mixed_degrees, (K, R, pb)) for K, R, pb in MIXED})
CHECKS["boundary"] = (check_integer_float_boundary, ())
CHECKS.update({f"exact/{e[0]}": (check_every_replica_every_sweep, e) for e in EXACT})
CHECKS["flush"] = (check_nsat_flushes_at_degree_15, ())
CHECKS["config4/sweeps"] = (check_config4_sweeps, ())
CHECKS["config4/ladder"] = (check_config4_ladder, ())


def run_checks(path, names):
    """child: run the named checks, write {name: "ok" or the traceback} to path"""
    import traceback

    import oracle_lib
    from pyisingmontecarlo_b200 import _native as nat

    nat.Context.get(0)
    sms = device_sms()
    res = {}
    for name in names:
        fn, args = CHECKS[name]
        try:
            fn(nat, oracle_lib, sms, *args)
            res[name] = "ok"
        except Exception:
            res[name] = traceback.format_exc()
        print(name, "ok" if res[name] == "ok" else "FAILED", flush=True)
    with open(path, "w") as f:
        json.dump(res, f)


_CHILD = (
    "import sys\n"
    "sys.path[:0] = [%r, %r]\n"
    "import test_gpu_general_graph as T\n"
    "T.run_checks(sys.argv[1], sys.argv[2:])\n") % (ROOT, os.path.join(ROOT, "tests"))


def child(names, env=None, timeout=1500):
    """{name: outcome} of the named checks, run in a child process (ISING_ knobs from env only)"""
    e = {k: v for k, v in os.environ.items() if not k.startswith("ISING_")}
    e.update(env or {})
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "outcomes.json")
        res = subprocess.run([sys.executable, "-c", _CHILD, path] + list(names), env=e, timeout=timeout,
                             capture_output=True, text=True)
        assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-6000:]
        with open(path) as f:
            return json.load(f)


@pytest.fixture(scope="module")
def outcomes(native, oracle):
    return child(CHECKS)


def _report(outcomes, name):
    assert outcomes[name] == "ok", outcomes[name]


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_shape_matrix_matches_mirror(outcomes, case):
    _report(outcomes, f"shape/{case.name}")


@pytest.mark.parametrize("K,R,perbeta", MIXED, ids=[f"K{K}_R{R}" + ("_perbeta" if pb else "") for K, R, pb in MIXED])
def test_mixed_degrees_match_mirror(outcomes, K, R, perbeta):
    """Degrees 0 .. 15 with +-0.5 couplings at K = 5 / 6 / 7 and Philox-7 / 10"""
    _report(outcomes, f"mixed/{K}/{R}/{perbeta}")


def test_integer_float_boundary(outcomes):
    _report(outcomes, "boundary")


@pytest.mark.parametrize("name", [e[0] for e in EXACT])
def test_every_replica_every_sweep(outcomes, name):
    _report(outcomes, f"exact/{name}")


def test_nsat_flushes_at_degree_15(outcomes):
    _report(outcomes, "flush")


def test_config4_sweeps_match_mirror(outcomes):
    _report(outcomes, "config4/sweeps")


def test_config4_ladder_matches_mirror(outcomes):
    _report(outcomes, "config4/ladder")


def test_no_pdl_changes_no_result(native, oracle):
    """ISING_NO_PDL=1 (read once per process): without programmatic dependent launch the general
    sweep's prefetch before griddepcontrol.wait still sees the previous group's spins, and the
    results equal the mirror"""
    names = ["shape/rr3_wrap", "shape/ragged_w33_perbeta"]
    res = child(names, {"ISING_NO_PDL": "1"})
    for n in names:
        _report(res, n)
