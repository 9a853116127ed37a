"""The bit-sliced two-spin edge move (k_edge_general, csrc/moves.cu) compared bit for bit with the
scalar mirror (oracle/msc_mirror.c: msc_mirror_moves) on the device, at every instantiation and
launch shape the library picks, and at config 3's size (run with -m gpu on a B200).

Every equal-|J|, bias-free graph runs its non-basic edge moves on this kernel (Lattice with
non_basic_moves, ClassicIsing(nedgeupdates=...), ising_sim_set_moves).  It has its own decision
machinery (edge_flip_mask) and its own host-side layout (api_core.cu: ensure_edge_general_on_device),
so the sweep gates say nothing about it.  A decision depends only on (seed, edge id, global replica
word, timestep, pass), so msc_mirror_moves(E = 32 k, replica_offset = 32 w) reproduces words
w .. w + k - 1 of a larger run: large runs are checked word by word, the words on a thread pool
(the mirror's edge pass is serial; ctypes releases the GIL).  Every run records its kernels
(torch.profiler) and asserts the k_edge_general<K, ROUNDS, V, DEG> instantiations that the
launcher's rules, restated below with the device's SM count, give; each case also asserts the
branch it exists for, so a case that loses its path fails under its own name.
"""
import json
import os
import re
import subprocess
import sys
import tempfile
from concurrent.futures import ThreadPoolExecutor
from dataclasses import dataclass, field

import numpy as np
import pytest

from mirror_check import device_sms, first_diff, instances, launched, pow2_ceil, random_regular, word_bits

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GEN_MAX_DEG = 15
ALL_INSTANCES = ({(K, R, V, 0) for K in (5, 6, 7) for R in (7, 10) for V in (1, 2)}
                 | {(6, 7, V, D) for V in (1, 2) for D in (4, 6, 10)})


# ---------------------------------------------------------------------------------------------
# the launcher's dispatch restated (api_core.cu: ensure_edge_general_on_device; moves.cu:
# edge_general_launch, edge_general_degree; api_sim.cu: sim_non_basic_moves)
# ---------------------------------------------------------------------------------------------
def edge_launch(W, count, sms):
    """launch shape of k_edge_general over one (class, outer degree) group of `count` bonds"""
    V = 2 if W % 2 == 0 else 1
    groups = W // V
    wx = 32 if groups >= 32 else pow2_ceil(groups)
    by = 256 // wx
    blocks = min(-(-count // by), 16 * sms)
    w_passes = -(-W // (wx * V))
    return dict(V=V, wx=wx, by=by, blocks=blocks, bond_passes=-(-count // (blocks * by)), w_passes=w_passes,
                idle_lanes=wx * w_passes - groups)


def edge_deg(K, rounds, d):
    """DEG template argument: compile-time outer degree 4 / 6 / 10 at the default (K, ROUNDS) only"""
    return d if K == 6 and rounds == 7 and d in (4, 6, 10) else 0


def outer_degrees(nvars, a, b):
    """D of every bond: adjacency entries of both ends that do not lead to the other end"""
    a, b = a.astype(np.int64), b.astype(np.int64)
    deg = np.bincount(a, minlength=nvars) + np.bincount(b, minlength=nvars)
    key = np.minimum(a, b) * nvars + np.maximum(a, b)
    _, inv, mult = np.unique(key, return_inverse=True, return_counts=True)
    return deg, deg[a] + deg[b] - 2 * mult[inv]


def edge_groups(cls, D):
    """{(class, D): bonds}: one k_edge_general launch each per pass"""
    keys, counts = np.unique(cls.astype(np.int64) * 64 + D, return_counts=True)
    return {(int(k) // 64, int(k) % 64): int(c) for k, c in zip(keys, counts)}


def edge_instances(groups, W, K, rounds):
    V = 2 if W % 2 == 0 else 1
    return {(K, rounds, V, edge_deg(K, rounds, d)) for _, d in groups}


def kernels(names):
    out = set()
    for n in names:
        m = re.search(r"\b(k_\w+)", n)
        if m:
            out.add(m.group(1))
    return out


# ---------------------------------------------------------------------------------------------
# graphs
# ---------------------------------------------------------------------------------------------
def signs(rng, m):
    return np.where(rng.random(m) < 0.5, -1.0, 1.0)


def outer_degree_edges(copies=6, seed=21):
    """Every outer degree D = 0 .. 15, +-0.5: per D, `copies` bonds (u, v) with deg(u) = (D + 3) // 2
    and deg(v) = (D + 2) // 2 made up by leaves (a leaf of a hub of degree p has D = p - 1), and one
    double bond with three leaves at each end (D = 6).  Site degrees stay <= 9."""
    rng = np.random.default_rng(seed)
    a, b, n = [], [], 0
    for D in range(16):
        p, q = (D + 3) // 2, (D + 2) // 2
        for _ in range(copies):
            u, v = n, n + 1
            n += 2
            a.append(u)
            b.append(v)
            for hub, k in ((u, p - 1), (v, q - 1)):
                for _ in range(k):
                    a.append(hub)
                    b.append(n)
                    n += 1
    u, v = n, n + 1
    n += 2
    a += [u, u]
    b += [v, v]
    for hub in (u, v):
        for _ in range(3):
            a.append(hub)
            b.append(n)
            n += 1
    a, b = np.array(a), np.array(b)
    return n, a, b, 0.5 * signs(rng, len(a))


def irregular_edges():
    """300 sites of degree 1 .. 5 (random pairing), a multi-edge, a leaf and an isolated pair, +-1"""
    rng = np.random.default_rng(17)
    n = 300
    target = rng.integers(1, 6, n)
    if target.sum() % 2:
        target[0] += 1
    while True:
        stubs = np.repeat(np.arange(n), target)
        rng.shuffle(stubs)
        a, b = stubs[0::2], stubs[1::2]
        if not (a == b).any():
            break
    # a double bond 300 = 301, a leaf 302 on site 0, an isolated pair 303 - 304
    a = np.concatenate([a, [300, 300, 301, 302, 303]])
    b = np.concatenate([b, [301, 301, 1, 0, 304]])
    return n + 5, a, b, signs(rng, len(a))


def _rr(n, seed):
    rng = np.random.default_rng(seed)
    a, b = random_regular(n, 3, rng)
    return n, a, b, signs(rng, len(a))


GRAPHS = {
    # name: builder -> (nvars, a, b, j), or torus arguments; general_layout
    "torus3d_pmj": (dict(dims=(8, 8, 8), j0=1.0, pmj=True, j_seed=4), False),
    "torus3d_pmj_gen": (dict(dims=(8, 8, 8), j0=1.0, pmj=True, j_seed=4), True),
    "torus2d_anti": (dict(dims=(16, 12), j0=1.0), False),
    "torus2d_ferro_gen": (dict(dims=(16, 12), j0=-1.0), True),
    "rr3_2000_pmj": (lambda: _rr(2000, 3), False),
    "irregular": (irregular_edges, False),
    "outer_degrees": (outer_degree_edges, False),
    "rr3_300k_pmj": (lambda: _rr(300_000, 9), False),
    "square1024_ferro": (dict(dims=(1024, 1024), j0=-1.0), False),
    # bench.py's config 3 lattice
    "config3": (dict(dims=(64, 64, 64), j0=1.0, pmj=True, j_seed=2024), False),
}
_graph_cache = {}


@dataclass
class G:
    g: object
    general_layout: bool
    edges: tuple
    colors: np.ndarray
    cls: np.ndarray
    D: np.ndarray
    groups: dict


def make_graph(native, spec, general_layout=False):
    ctx = native.Context.get(0)
    if isinstance(spec, dict):
        g = native.Graph.torus(ctx, **spec)
    else:
        n, a, b, j = spec
        g = native.Graph.from_edges(ctx, n, a, b, j)
    a, b, j = g.edges()
    cls = g.edge_classes()
    _, D = outer_degrees(g.nvars, a, b)
    return G(g, general_layout, (a, b, j), g.colors(), cls, D, edge_groups(cls, D))


def graph(native, name):
    if name not in _graph_cache:
        spec, general = GRAPHS[name]
        _graph_cache[name] = make_graph(native, spec if isinstance(spec, dict) else spec(), general)
    return _graph_cache[name]


# ---------------------------------------------------------------------------------------------
# comparison with the mirror
# ---------------------------------------------------------------------------------------------
def mirror_words(oracle, gr, E, seed, betas, words, offset=0, planes=6, rounds=7, spin_sweeps=1, passes=1):
    """{w: (energies[k, T], states bool[k, nvars], continuation decisions)} of msc_mirror_moves run
    on replica word w alone (k = 32, or the ragged last word's true tail), words concurrently"""
    a, b, j = gr.edges

    def one(w):
        k = min(32, E - 32 * w)
        cont = np.zeros(1, dtype=np.uint64)
        en, st = oracle.msc_mirror_moves(a, b, j, gr.g.nvars, gr.colors, gr.cls, k, seed, betas,
                                         spin_sweeps=spin_sweeps, edge_passes=passes,
                                         replica_offset=offset + 32 * w, planes=planes, rounds=rounds,
                                         per_step=True, continuations=cont)
        return en, st, int(cont[0])

    with ThreadPoolExecutor(max_workers=max(1, min(len(words), os.cpu_count() or 1))) as ex:
        return dict(zip(words, ex.map(one, words)))


def check_against_mirror(oracle, gr, sim, E, seed, betas, words, en, label, offset=0, **kw):
    """states and per-timestep energies of `words` equal the mirror's; -> continuation decisions"""
    packed = sim.packed()
    ref = mirror_words(oracle, gr, E, seed, betas, words, offset, **kw)
    cont = 0
    for w in words:
        k = min(32, E - 32 * w)
        en_ref, st_ref, c = ref[w]
        cont += c
        st = word_bits(packed, w, k)
        ok = (st == st_ref).all() and (en[32 * w:32 * w + k] == en_ref).all()
        assert ok, f"{label} word {w}: {first_diff(st, st_ref, en[32 * w:32 * w + k], en_ref, offset + 32 * w)}"
    return cont


# ---------------------------------------------------------------------------------------------
# 1. shape matrix, grid wrap, config 3
# ---------------------------------------------------------------------------------------------
SHAPE_BETAS = np.array([0.2, 0.7, 2.0])


@dataclass
class Case:
    name: str
    graph: str
    E: int
    seed: int
    betas: np.ndarray = field(default_factory=lambda: SHAPE_BETAS)
    moves: tuple = (1, 2)        # (spin_sweeps, edge_passes)
    offset: int = 0
    planes: int = 6
    rounds: int = 7
    words: tuple = None          # None: every word
    importance: bool = False
    reach: dict = field(default_factory=dict)   # launch-shape property -> value in every group

    @property
    def W(self):
        return -(-self.E // 32)


def check_reach(case, gr, sms):
    """the case still reaches the branch it is meant for.  V / wx / w_passes / idle_lanes hold
    in every group; DEG: some group runs it; wrapped: at least that many groups take >= 2 grid
    passes over their bonds"""
    shapes = {key: edge_launch(case.W, c, sms) for key, c in gr.groups.items()}
    for k, want in case.reach.items():
        if k == "DEG":
            got = {edge_deg(case.planes, case.rounds, d) for _, d in gr.groups}
            assert want in got, f"{case.name}: DEG {want} not among {sorted(got)}"
        elif k == "wrapped":
            n = sum(sh["bond_passes"] >= 2 for sh in shapes.values())
            assert n >= want, f"{case.name}: {n} groups wrap the grid, meant for >= {want}"
        elif k == "min_idle_lanes":
            assert all(sh["idle_lanes"] >= want for sh in shapes.values()), (case.name, shapes)
        else:
            for key, sh in shapes.items():
                assert sh[k] == want, f"{case.name}: group {key} reaches {k} = {sh[k]}, meant for {want}"
    return shapes


def run_case(native, oracle, sms, case):
    """One run with per-timestep energies against the mirror, word by word, bit for bit.
    Asserts the instantiations.  Returns the kernel names."""
    gr = graph(native, case.graph)
    g = gr.g
    shapes = check_reach(case, gr, sms)
    assert g.integer_classes and g.max_degree <= GEN_MAX_DEG and gr.D.max() <= GEN_MAX_DEG
    label = f"{case.name} [{g.nvars} sites x {case.E}, K={case.planes} R={case.rounds}]"
    sim = native.Sim(g, case.E, case.seed, replica_offset=case.offset, planes=case.planes, rounds=case.rounds,
                     general_layout=gr.general_layout)
    sim.set_moves(case.moves[0], case.moves[1], 0, edge_importance=case.importance)
    en, names = launched(lambda: sim.sweeps(case.betas, per_sweep_energies=True))
    got = instances(names, "k_edge_general")
    want = edge_instances(gr.groups, case.W, case.planes, case.rounds)
    print(f"{label}: {sorted(got)}, {len(gr.groups)} groups, max bond passes "
          f"{max(sh['bond_passes'] for sh in shapes.values())}", flush=True)
    assert got == want, (label, "k_edge_general instances", sorted(got), "expected", sorted(want))
    assert "k_edge_moves" not in kernels(names), (label, names)
    assert (sim.energies() == en[:, -1]).all(), label
    words = tuple(range(case.W)) if case.words is None else case.words
    cont = check_against_mirror(oracle, gr, sim, case.E, case.seed, case.betas, words, en, label, case.offset,
                                planes=case.planes, rounds=case.rounds, spin_sweeps=case.moves[0],
                                passes=case.moves[1])
    sim.close()
    return names, cont


CASES = [
    # the lane shapes: wx = 1, 1, 4, 8, 4 with V = 1, 2, 1, 1, 2 (idle x-lanes at E = 96 and 160)
    Case("e32_torus3d_deg10", "torus3d_pmj", 32, 11, reach=dict(V=1, wx=1, DEG=10)),
    Case("e64_torus2d_deg6", "torus2d_anti", 64, 12, reach=dict(V=2, wx=1, DEG=6)),
    Case("e96_rr3_deg4", "rr3_2000_pmj", 96, 13, reach=dict(V=1, wx=4, DEG=4, min_idle_lanes=1)),
    Case("e160_irregular", "irregular", 160, 14, reach=dict(V=1, wx=8, DEG=0, min_idle_lanes=3)),
    Case("e256_torus3d_general", "torus3d_pmj_gen", 256, 15, reach=dict(V=2, wx=4, DEG=10)),
    # wx = 16 and 32
    Case("e1024_torus2d_general", "torus2d_ferro_gen", 1024, 16, reach=dict(V=2, wx=16, DEG=6)),
    Case("e2048_torus3d", "torus3d_pmj", 2048, 17, reach=dict(V=2, wx=32, DEG=10)),
    # the word loop: two passes with a 27-replica tail word, three passes
    Case("e1051_rr3", "rr3_2000_pmj", 1051, 18, reach=dict(V=1, wx=32, w_passes=2, DEG=4)),
    Case("e1051_torus2d", "torus2d_anti", 1051, 19, reach=dict(V=1, wx=32, w_passes=2)),
    Case("e4160_irregular", "irregular", 4160, 20, reach=dict(V=2, wx=32, w_passes=3)),
    Case("e4160_torus3d", "torus3d_pmj", 4160, 21, reach=dict(V=2, wx=32, w_passes=3, DEG=10)),
    # sharded runs: the global word gw0 != 0 enters the Philox counter and the initial state
    Case("offset320_torus3d", "torus3d_pmj", 200, 22, offset=320, reach=dict(V=1, wx=8)),
    Case("offset2048_rr3", "rr3_2000_pmj", 256, 23, offset=2048, reach=dict(V=2, wx=4, DEG=4)),
    # edge moves alone, and importance sampling (every bond weighs alike: no bit may change)
    Case("moves_alone_irregular", "irregular", 96, 24, moves=(0, 3)),
    Case("importance_torus3d", "torus3d_pmj", 256, 25, importance=True, reach=dict(DEG=10)),
    Case("importance_irregular", "irregular", 70, 26, importance=True),
    # grid wrap: 8 of 11 classes wrap (cap 18944 bonds at 148 SMs); 9 classes wrap about 7 times
    Case("wrap_rr3_300k", "rr3_300k_pmj", 2048, 27, betas=np.array([0.5, 1.5]), moves=(1, 1), words=(0, 31, 63),
         reach=dict(V=2, wx=32, DEG=4, wrapped=6)),
    Case("wrap_square1024", "square1024_ferro", 1024, 28, betas=np.array([0.42, 0.46]), moves=(1, 1),
         words=(0, 31), reach=dict(V=2, wx=16, DEG=6, wrapped=6)),
    # config 3 with edge moves: 12 classes wrap, 19 small or one-bond classes
    Case("config3_64cubed", "config3", 1024, 29, betas=np.array([0.21, 0.22, 0.23]), moves=(1, 1),
         words=(0, 31), reach=dict(V=2, wx=16, DEG=10, wrapped=10)),
]
CASE = {c.name: c for c in CASES}


# ---------------------------------------------------------------------------------------------
# 2. every instantiation: outer degrees 0 .. 15 at K = 5 / 6 / 7, Philox-7 / 10, V = 1 / 2
# ---------------------------------------------------------------------------------------------
DEG_BETAS = np.array([0.3, 3.0, 3.0, 3.0])     # high beta: ties (32 / 2^K per uphill word) are common
MIXED = [(K, R, V) for K in (5, 6, 7) for R in (7, 10) for V in (1, 2)]


def check_outer_degrees(native, oracle, sms, K, R, V):
    """Every outer degree 0 .. 15 in one +-0.5 graph: the run-time-degree kernel (DEG = 0: four
    counter planes, up to eight uphill classes) and, at K = 6, R = 7, the DEG = 4 / 6 / 10 ones.  At
    high beta some decisions read continuation rounds (philox4x32_more): the 4th tie of a word at
    K = 5, the 3rd at K = 6, the 2nd at K = 7; the mirror counts them."""
    gr = graph(native, "outer_degrees")
    assert set(gr.D.tolist()) == set(range(16)), sorted(set(gr.D.tolist()))
    assert all((gr.D == d).sum() >= 6 for d in range(16))
    E = 64 if V == 2 else 96
    case = Case(f"outer_degrees_K{K}_R{R}_V{V}", "outer_degrees", E, 40 + K + R + V, betas=DEG_BETAS,
                planes=K, rounds=R, reach=dict(V=V, DEG=0))
    names, cont = run_case(native, oracle, sms, case)
    print(f"{case.name}: {cont} decisions read continuation rounds", flush=True)
    assert cont > 0, f"{case.name}: no decision reached a continuation round"
    assert 0 in {t[3] for t in instances(names, "k_edge_general")}
    return names


def check_float_boundary(native, oracle, sms):
    """One more leaf at the larger end of a D = 15 pair makes that pair D = 16: the whole graph's
    edge moves go to k_edge_moves, while the sweep stays on the integer kernel"""
    gr = graph(native, "outer_degrees")
    a, b, j = gr.edges
    i = int(np.flatnonzero(gr.D == 15)[0])
    deg, _ = outer_degrees(gr.g.nvars, a, b)
    hub = int(a[i]) if deg[a[i]] >= deg[b[i]] else int(b[i])
    n = gr.g.nvars + 1
    g16 = make_graph(native, (n, np.append(a, hub), np.append(b, n - 1), np.append(j, 0.5)))
    assert g16.D.max() == 16 and g16.g.max_degree <= GEN_MAX_DEG and g16.g.integer_classes
    sim = native.Sim(g16.g, 64, 71)
    sim.set_moves(1, 1, 0)
    _, names = launched(lambda: sim.sweeps([0.5, 1.0]))
    sim.close()
    k = kernels(names)
    assert "k_edge_moves" in k and "k_edge_general" not in k, names
    assert "k_sweep_general" in k, names


# ---------------------------------------------------------------------------------------------
# 3. a shard against the matching words of the unsharded run
# ---------------------------------------------------------------------------------------------
def check_shard(native, oracle, sms):
    """E = 96 at replica_offset 128 (W = 3: one word per thread) equals words 4 .. 6 of the
    unsharded E = 256 run (W = 8: two words per thread)"""
    gr = graph(native, "torus3d_pmj")
    runs = []
    for E, off, V in ((256, 0, 2), (96, 128, 1)):
        sim = native.Sim(gr.g, E, 33, replica_offset=off)
        sim.set_moves(1, 2, 0)
        en, names = launched(lambda: sim.sweeps(SHAPE_BETAS, per_sweep_energies=True))
        assert instances(names, "k_edge_general") == {(6, 7, V, 10)}, names
        runs.append((en, sim.packed()))
        sim.close()
    (en_full, p_full), (en_shard, p_shard) = runs
    assert (p_shard == p_full[:, 4:7]).all(), "shard states differ from words 4 .. 6 of the full run"
    assert (en_shard == en_full[128:224]).all(), "shard energies differ"


# ---------------------------------------------------------------------------------------------
# 4. every replica after every timestep against an int64 numpy energy
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


# (name, graph, E, (spin_sweeps, edge_passes), energy kernel); stencil: W = 1 / 8 / 32 / 64 give
# 16 / 16 / 4 / 2 copies of a timestep's counters
EXACT = [("stencil_w1", "torus3d_pmj", 32, (1, 1), "k_nsat_stencil"),
         ("stencil_w8", "torus2d_anti", 256, (0, 2), "k_nsat_stencil"),
         ("stencil_w32", "torus3d_pmj", 1024, (1, 2), "k_nsat_stencil"),
         ("stencil_w64", "torus3d_pmj", 2048, (0, 1), "k_nsat_stencil"),
         ("general_w33", "irregular", 1051, (1, 1), "k_nsat_general"),
         ("general_alone", "torus3d_pmj_gen", 200, (0, 2), "k_nsat_general")]


def check_every_replica_every_step(native, oracle, sms, name, gname, E, moves, nsat):
    gr = graph(native, gname)
    a, b, j = gr.edges
    jabs = abs(j[0])
    sim = native.Sim(gr.g, E, 90 + E, general_layout=gr.general_layout)
    sim.set_moves(moves[0], moves[1], 0)
    for t, beta in enumerate((0.3, 1.0, 2.0)):
        en, names = launched(lambda: sim.sweeps([beta], per_sweep_energies=True))
        k = kernels(names)
        assert nsat in k and "k_edge_general" in k and "k_edge_moves" not in k, names
        e_np = int_energies(sim.states(), a, b, j) * jabs
        bad = np.flatnonzero(en[:, 0] != e_np)
        assert len(bad) == 0, (f"{name} step {t}: {len(bad)} per-step energies differ, first replica "
                               f"{bad[:1]}: {en[bad[:1], 0]} vs {e_np[bad[:1]]}")
        assert (sim.energies() == e_np).all(), f"{name} step {t}: energies()"
    sim.close()


# ---------------------------------------------------------------------------------------------
# 5. the device runs, in child processes
# ---------------------------------------------------------------------------------------------
# Every check runs in one child process and the tests below report its outcomes: the profiler
# attaches CUPTI to the process it runs in, and later profiler sessions in the same process can miss
# kernels that other tests load meanwhile (DESIGN.md section 2, item 7).
CHECKS = {f"shape/{c.name}": (run_case, (c,)) for c in CASES}
CHECKS.update({f"degrees/{K}/{R}/{V}": (check_outer_degrees, (K, R, V)) for K, R, V in MIXED})
CHECKS["boundary"] = (check_float_boundary, ())
CHECKS["shard"] = (check_shard, ())
CHECKS.update({f"exact/{e[0]}": (check_every_replica_every_step, e) for e in EXACT})


def run_checks(path, names):
    """child: run the named checks, write {name: "ok" or the traceback} and the union of the
    k_edge_general instantiations recorded to path"""
    import time
    import traceback

    import oracle_lib
    from pyisingmontecarlo_b200 import _native as nat

    nat.Context.get(0)
    sms = device_sms()
    res, seen = {}, set()
    for name in names:
        fn, args = CHECKS[name]
        t0 = time.time()
        try:
            out = fn(nat, oracle_lib, sms, *args)
            kn = out[0] if isinstance(out, tuple) else out
            if kn:
                seen |= instances(kn, "k_edge_general")
            res[name] = "ok"
        except Exception:
            res[name] = traceback.format_exc()
        print(name, "ok" if res[name] == "ok" else "FAILED", f"{time.time() - t0:.1f} s", flush=True)
    with open(path, "w") as f:
        json.dump({"outcomes": res, "instances": sorted(seen)}, f)


_CHILD = (
    "import sys\n"
    "sys.path[:0] = [%r, %r]\n"
    "import test_gpu_edge_moves as T\n"
    "T.run_checks(sys.argv[1], sys.argv[2:])\n") % (ROOT, os.path.join(ROOT, "tests"))


def child(names, env=None, timeout=1500):
    """{"outcomes": {name: outcome}, "instances": [...]} of the named checks, run in a child process
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
def test_edge_moves_match_mirror(results, case):
    _report(results, f"shape/{case.name}")


@pytest.mark.parametrize("K,R,V", MIXED, ids=[f"K{K}_R{R}_V{V}" for K, R, V in MIXED])
def test_outer_degrees_0_to_15_match_mirror(results, K, R, V):
    """D = 0 .. 15 at K = 5 / 6 / 7, Philox-7 / 10, V = 1 / 2, with continuation rounds"""
    _report(results, f"degrees/{K}/{R}/{V}")


def test_outer_degree_16_takes_the_float_kernel(results):
    _report(results, "boundary")


def test_shard_equals_words_of_the_unsharded_run(results):
    _report(results, "shard")


@pytest.mark.parametrize("name", [e[0] for e in EXACT])
def test_every_replica_every_step(results, name):
    _report(results, f"exact/{name}")


def test_every_instantiation_ran(results):
    """the checks above ran all 18 instantiations of k_edge_general"""
    seen = {tuple(t) for t in results["instances"]}
    assert seen == ALL_INSTANCES, (sorted(ALL_INSTANCES - seen), sorted(seen - ALL_INSTANCES))


def test_no_pdl_changes_no_result(native, oracle):
    """ISING_NO_PDL=1 (read once per process): the per-group launches without programmatic
    dependent launch give the same bits"""
    names = ["shape/e1051_rr3", "shape/e4160_torus3d", "degrees/6/7/2"]
    res = child(names, {"ISING_NO_PDL": "1"})
    for n in names:
        _report(res, n)
