"""The float-field path on the GPU, decision by decision (tests/float_reference.py).

Graphs outside the integer classes (real couplings, a bias, degree > 15) run on k_sweep_real,
k_edge_moves and k_worm_moves.  Each accept / reject is a Philox word against exp(-beta dE) in
f32 and __expf; the f64 reference knows every decision except the few whose word falls in the
rounding band, and a replica that meets one is dropped from the comparison.  Every other replica
must equal the reference bit for bit, at least 99 % of them must stay determined, and every
returned energy must lie within the explicit f64 summation bound of the exact energy.  Everything
goes through the C ABI (Sim, Tempering, Lattice); the start is read back before the first sweep
or set by the test."""
import numpy as np
import pytest

import float_reference as fr

pytestmark = pytest.mark.gpu

BETAS = [0.0, 0.3, 1.0, 3.0, 1e6]


def report(name, ch):
    print(f"\nfloat-gate {name}: in band {ch.in_band} of {ch.decisions} decisions, "
          f"determined {ch.determined.sum()} of {ch.E} replicas")


def assert_gate(ch, got, name, min_determined=0.99):
    report(name, ch)
    bad = np.nonzero((np.asarray(got) != ch.s).any(axis=1) & ch.determined)[0]
    assert len(bad) == 0, f"{name}: replicas {bad[:10]} differ from the reference outside the band"
    assert ch.determined.mean() >= min_determined, (ch.determined.sum(), ch.E)
    assert ch.in_band < 1e-3 * max(ch.decisions, 1)


def assert_energies(g, states, energies):
    ref = g.energies(states)
    err = np.abs(np.asarray(energies) - ref)
    assert (err <= g.energy_bound()).all(), (err.max(), g.energy_bound())


def lattice_edges(L, rng):
    n = np.arange(L ** 3)
    x, y, z = n % L, (n // L) % L, n // (L * L)
    b = np.concatenate([(x + 1) % L + L * (y + L * z), x + L * ((y + 1) % L + L * z), x + L * (y + L * ((z + 1) % L))])
    a = np.concatenate([n, n, n])
    return L ** 3, a, b, rng.normal(size=len(a)), rng.normal(size=L ** 3)


def regular_edges(n, d, rng):
    """a simple d-regular graph (d even): the circulant i ~ i + 1 .. i + d / 2, randomly relabelled"""
    perm = rng.permutation(n)
    i = np.repeat(np.arange(n), d // 2)
    k = np.tile(np.arange(1, d // 2 + 1), n)
    return perm[i], perm[(i + k) % n]


def make_graph(native, kind, rng):
    """-> (native Graph, reference Graph, bias)"""
    ctx = native.Context.get(0)
    bias = None
    if kind == "lattice12":
        n, a, b, j, bias = lattice_edges(12, rng)
    elif kind == "sk256":
        n = 256
        a, b = np.triu_indices(n, 1)
        j = rng.normal(size=len(a)) / np.sqrt(n)
    elif kind == "regular20":
        n = 300
        a, b = regular_edges(n, 20, rng)
        j = rng.choice([-1.0, 1.0], size=len(a))
    elif kind == "torus_field":
        n, a, b, _, _ = lattice_edges(6, rng)
        j = np.full(len(a), -1.0)
        bias = np.full(n, 0.3)
    else:   # real couplings, a leaf (site 10), an isolated site (11), a double bond (1-4)
        n = 12
        edges = [(0, 1), (1, 2), (2, 0), (2, 3), (3, 4), (1, 4), (1, 4), (4, 5), (5, 6), (6, 7), (7, 8), (8, 9),
                 (9, 5), (0, 8), (3, 10)]
        a = np.array([e[0] for e in edges]); b = np.array([e[1] for e in edges])
        j = rng.normal(size=len(a))
        bias = rng.normal(size=n) * 0.4
        bias[11] = 0.0
    g = native.Graph.from_edges(ctx, n, a.astype(np.uint64), b.astype(np.uint64), j, bias)
    assert not g.integer_classes or g.max_degree > 15
    return g, fr.Graph.from_native(g, bias), bias


@pytest.mark.parametrize("kind", ["lattice12", "sk256", "regular20", "torus_field"])
@pytest.mark.parametrize("E,rounds", [(1, 7), (33, 10), (1031, 7)])
def test_sweeps_take_the_reference_decisions(native, kind, E, rounds):
    rng = np.random.default_rng(len(kind) * 10000 + E)
    g, ref, _ = make_graph(native, kind, rng)
    seed = 0xF10A7 + E
    sim = native.Sim(g, E, seed, rounds=rounds)
    ch = fr.Chain(ref, sim.states(), seed, rounds=rounds)
    sim.sweeps(np.array(BETAS))
    for t, beta in enumerate(BETAS):
        ch.sweep(t, beta)
    got = sim.states()
    assert_gate(ch, got, f"sweeps {kind} E={E} rounds={rounds}")
    assert_energies(ref, got, sim.energies())


def test_sharded_sim_equals_the_unsharded_one(native):
    """Sim(E=40, replica_offset=64) == replicas 64..103 of Sim(E=104) with sweeps, edge passes and worms:
    gw0 in all three float kernels, the replica offset in the worms; the reference at offset 64 agrees"""
    rng = np.random.default_rng(64)
    g, ref, _ = make_graph(native, "moves", rng)
    seed, betas = 0xABCDEF, np.array([0.3, 1.0, 3.0, 0.0, 1e6, 0.7])
    init = rng.integers(0, 2, size=(104, g.nvars)).astype(bool)
    full = native.Sim(g, 104, seed)
    part = native.Sim(g, 40, seed, replica_offset=64)
    full.set_states(init)
    part.set_states(init[64:])
    ch = fr.Chain(ref, init[64:], seed, rep0=64)
    for sim in (full, part):
        sim.set_moves(1, 2, 3, worm_len=3)
        sim.sweeps(betas)
    for t, beta in enumerate(betas):
        ch.timestep(t, beta, 1, 2, 3, 3)
    got = part.states()
    assert (got == full.states()[64:]).all()
    assert_gate(ch, got, "sharded sim at offset 64", min_determined=0.97)
    assert_energies(ref, got, part.energies())


@pytest.mark.parametrize("moves", [
    dict(spin_sweeps=0, edge_passes=2, worms=2, worm_len=1),
    dict(spin_sweeps=1, edge_passes=2, worms=2, worm_len=2, edge_importance=True),
    dict(spin_sweeps=0, edge_passes=2, worms=3, worm_len=5, edge_importance=True),
    dict(spin_sweeps=1, edge_passes=2, worms=2, worm_len=8),
])
def test_moves_take_the_reference_decisions(native, moves):
    rng = np.random.default_rng(7 + moves["worm_len"])
    g, ref, _ = make_graph(native, "moves", rng)
    E, seed = 1031, 0x3A0E5 + moves["worm_len"]
    betas = np.array([0.3, 1.0, 3.0, 1e6, 0.0, 0.6])
    sim = native.Sim(g, E, seed)
    ch = fr.Chain(ref, sim.states(), seed)
    sim.set_moves(**moves)
    sim.sweeps(betas)
    for t, beta in enumerate(betas):
        ch.timestep(t, beta, moves["spin_sweeps"], moves["edge_passes"], moves["worms"], moves["worm_len"],
                    moves.get("edge_importance", False))
    got = sim.states()
    assert_gate(ch, got, f"moves {moves}", min_determined=0.97)
    assert_energies(ref, got, sim.energies())


def test_worms_alone_on_the_checkerboard_layout(native):
    """a +-J torus keeps the checkerboard layout; worms alone run there (set_moves(0, 0, 4, 5))"""
    ctx = native.Context.get(0)
    g = native.Graph.torus(ctx, (8, 6), j0=1.0, pmj=True, j_seed=4)
    ref = fr.Graph.from_native(g)
    E, seed = 70, 0x77
    betas = np.array([0.2, 0.8, 1e6, 0.0, 0.5])
    sim = native.Sim(g, E, seed)
    ch = fr.Chain(ref, sim.states(), seed)
    sim.set_moves(0, 0, 4, 5)
    sim.sweeps(betas)
    for t, beta in enumerate(betas):
        ch.timestep(t, beta, 0, 0, 4, 5)
    assert_gate(ch, sim.states(), "worms on the checkerboard layout")


def test_per_replica_betas(native):
    rng = np.random.default_rng(3)
    g, ref, _ = make_graph(native, "lattice12", rng)
    E, seed = 1031, 0xBE7A5
    sim = native.Sim(g, E, seed)
    betas = np.linspace(0.0, 3.0, E)
    sim.set_betas(betas)
    ch = fr.Chain(ref, sim.states(), seed)
    sim.sweeps(4)
    for t in range(4):
        ch.sweep(t, betas)
    got = sim.states()
    assert_gate(ch, got, "set_betas linspace(0, 3, 1031)")
    assert_energies(ref, got, sim.energies())


def test_tempering_on_real_couplings_with_a_field(native):
    """R = 40 (two replica words) on a Gaussian graph with biases: each configuration sweeps at
    betas[slot], Philox replica = configuration; slots follow decide_swaps on the same energies.
    Shards [0, 12) + [12, 40) and [0, 32) + [32, 40), stepped with the concatenated energies, equal
    the single ladder in states, slots and swap counts."""
    rng = np.random.default_rng(40)
    n = 500
    a, b = regular_edges(n, 4, rng)
    extra = rng.integers(0, n, size=(200, 2))
    extra = extra[extra[:, 0] != extra[:, 1]]
    a, b = np.concatenate([a, extra[:, 0]]), np.concatenate([b, extra[:, 1]])
    j, bias = rng.normal(size=len(a)), rng.normal(size=n) * 0.3
    ctx = native.Context.get(0)
    g = native.Graph.from_edges(ctx, n, a.astype(np.uint64), b.astype(np.uint64), j, bias)
    ref = fr.Graph.from_native(g, bias)
    R, seed, k = 40, 0x7E3, 2
    betas = np.linspace(0.1, 2.0, R)
    full = native.Tempering(g, betas, seed)
    shards = [[native.Tempering(g, betas, seed, cfg_lo=lo, cfg_hi=hi) for lo, hi in split]
              for split in ([(0, 12), (12, 40)], [(0, 32), (32, 40)])]
    ch = fr.Chain(ref, full.local_states(), seed)
    for sh in shards:
        assert (np.concatenate([p.local_states() for p in sh]) == ch.s).all()
    slot_of_cfg, cfg_of_slot = np.arange(R, dtype=np.uint32), np.arange(R, dtype=np.uint32)
    swaps, t = 0, 0
    for step in range(6):
        ef = full.sweeps(k)
        for _ in range(k):
            ch.sweep(t, betas[slot_of_cfg])
            t += 1
        got = full.local_states()
        assert_energies(ref, got, ef)
        full.swap_step(ef)
        swaps += native.decide_swaps(betas, ef, seed, step, slot_of_cfg, cfg_of_slot)
        assert (full.slots() == slot_of_cfg).all()
        for sh in shards:
            es = np.concatenate([p.sweeps(k) for p in sh])
            assert_energies(ref, got, es)
            for p in sh:
                p.swap_step(es)
                assert (p.slots() == slot_of_cfg).all()
            assert (np.concatenate([p.local_states() for p in sh]) == got).all()
    assert full.total_swaps() == swaps > 0
    for sh in shards:
        assert all(p.total_swaps() == swaps for p in sh)
    assert_gate(ch, full.local_states(), "tempering R=40", min_determined=0.97)


@pytest.mark.parametrize("driver", ["run", "sampling", "annealing", "linear_annealing"])
def test_lattice_drivers(native, driver):
    """Lattice with real edges, biases, seed_gen (the sim seed) and an initial state, against the
    reference replaying the same timesteps"""
    import pyisingmontecarlo_b200 as pkg

    rng = np.random.default_rng(11)
    n, a, b, j, bias = lattice_edges(6, rng)
    edges = [((int(x), int(y)), float(w)) for x, y, w in zip(a, b, j)]
    lat = pkg.Lattice(edges, seed_gen=0x5EED)
    for i, v in enumerate(bias):
        lat.set_individual_bias(i, float(v))
    init = rng.integers(0, 2, size=n).astype(bool)
    lat.set_initial_state(init)
    ref = fr.Graph(n, a, b, j, bias, lat.graph().colors())
    E, T = 70, 12
    ch = fr.Chain(ref, np.broadcast_to(init, (E, n)), 0x5EED)
    if driver == "run":
        en, st = lat.run_monte_carlo(0.8, T, E, only_basic_moves=True)
        for t in range(T):
            ch.sweep(t, 0.8)
    elif driver == "sampling":
        en, st = lat.run_monte_carlo_sampling(0.8, T, E, only_basic_moves=True, thermalization_time=3, sampling_freq=4)
        assert st.shape == (E, 3, n)
        for t in range(3 + T):
            ch.sweep(t, 0.8)
            if t >= 3 and (t - 2) % 4 == 0:
                k = (t - 2) // 4 - 1
                assert not ((st[:, k] != ch.s).any(axis=1) & ch.determined).any(), k
                assert_energies(ref, st[:, k], en[:, k])
        st = st[:, -1]
        en = en[:, -1]
    else:
        lat.linear_annealing = driver == "linear_annealing"
        stops = [(0, 0.1), (5, 2.0), (9, 0.5)]
        en, st = lat.run_monte_carlo_annealing_and_get_energies(stops, T, E, only_basic_moves=True)
        sched = native.schedule_betas(stops, T, linear=driver == "linear_annealing")
        for t in range(T):
            ch.sweep(t, sched[t])
        en = en[:, -1]
    assert_gate(ch, st, f"Lattice {driver}")
    assert_energies(ref, st, en)
