"""The non-basic moves (two-spin edge moves, worm moves) as the oracle restates them keep the
Boltzmann distribution: chains made of those moves alone reproduce exact enumeration."""
import numpy as np
import pytest

from moves_cases import boltzmann, histogram_z, irregular_graph  # noqa: E402


@pytest.mark.parametrize("moves", [
    dict(nedge=7, nworm=2, worm_len=3),                       # no single-spin move at all
    dict(nedge=7, nworm=2, worm_len=3, importance=True),      # edges drawn with probability ~ |J|
    dict(nworm=6, worm_len=1),                                # worm of one site = random-site attempt
    dict(nedge=7, nworm=4, worm_len=4),                       # even moves only: parity sectors
    dict(nspin=6, nedge=7, nworm=1, worm_len=2),              # everything together
])
def test_moves_alone_sample_the_boltzmann_law(oracle, moves):
    edges, n, biases = irregular_graph()
    beta = 0.8
    g = oracle.Graph(edges, biases=biases)
    E = 40000
    seeds = oracle.make_seeds(11, E)
    _, st = g.run_moves(beta, 60, seeds, **moves)
    _, p, _ = boltzmann(edges, n, beta, biases)
    # chains of even-length moves only keep the parity of the number of up spins: compare per sector
    if moves.get("nspin", 0) == 0 and moves.get("worm_len", 1) % 2 == 0:
        par = st.sum(1) % 2
        parity_of_state = np.array([bin(i).count("1") % 2 for i in range(2 ** n)])
        for sector in (0, 1):
            sel = st[par == sector]
            ps = np.where(parity_of_state == sector, p, 0.0)
            ps = ps / ps.sum()
            z = histogram_z(sel, ps)[parity_of_state == sector]
            assert np.abs(z).max() < 4.5, z
        return
    z = histogram_z(st, p)
    assert np.abs(z).max() < 4.5, z


def test_edge_move_leaves_the_shared_bond_alone(oracle):
    # one bond, strong coupling: flipping both ends never changes the energy, so every edge move
    # is accepted and the pair keeps its relative orientation
    g = oracle.Graph([((0, 1), -5.0)])
    seeds = oracle.make_seeds(3, 64)
    en, st = g.run_moves(3.0, 9, seeds, nedge=1, initial_state=[True, True])
    assert (en == -5.0).all() and (st[:, 0] == st[:, 1]).all()
    assert (st[:, 0] == False).all()      # 9 accepted double flips


def test_bit_sliced_edge_pass_of_the_mirror_samples_the_boltzmann_law(oracle, native):
    """The device's bit-sliced edge move (restated in oracle/msc_mirror.c, to which the GPU kernel is
    compared bit for bit) against exact enumeration: 4x4 torus, sweeps + edge passes, and edge
    passes alone within a parity sector."""
    L = 4
    a = [x + L * y for y in range(L) for x in range(L)] * 2
    b = [(x + 1) % L + L * y for y in range(L) for x in range(L)] + [x + L * ((y + 1) % L) for y in range(L) for x in range(L)]
    j = [-1.0] * len(a)
    edges = [((int(x), int(y)), w) for x, y, w in zip(a, b, j)]
    colors = np.array([(n % L + n // L) & 1 for n in range(L * L)], dtype=np.uint32)
    cls, ncls = native.strong_edge_colouring(L * L, a, b)
    beta = 0.35
    _, p, en = boltzmann(edges, L * L, beta)
    exact = float((p * en).sum())
    var = float((p * en * en).sum()) - exact ** 2
    E = 2048
    en_m, st = oracle.msc_mirror_moves(a, b, j, L * L, colors, cls, E, 5, np.full(40, beta), spin_sweeps=1,
                                       edge_passes=1, per_step=True)
    e = en_m[:, -1]
    assert abs(e.mean() - exact) < 4 * np.sqrt(var / E), (e.mean(), exact)
    # edge passes alone keep the parity of the number of up spins: compare within the even sector
    _, st2 = oracle.msc_mirror_moves(a, b, j, L * L, colors, cls, E, 9, np.full(60, beta), spin_sweeps=0,
                                     edge_passes=2)
    even = st2[st2.sum(1) % 2 == 0]
    parity = np.array([bin(i).count("1") % 2 for i in range(2 ** (L * L))])
    pe = np.where(parity == 0, p, 0.0)
    pe /= pe.sum()
    exact_even = float((pe * en).sum())
    var_even = float((pe * en * en).sum()) - exact_even ** 2
    g = oracle.Graph(edges)
    e_even = np.array([g.energy(s) for s in even])
    assert len(even) > E // 4
    assert abs(e_even.mean() - exact_even) < 4 * np.sqrt(var_even / len(even)), (e_even.mean(), exact_even)


@pytest.mark.parametrize("planes", [1, 2, 6])
def test_tie_words_of_the_mirror_are_sound_uniforms(oracle, planes):
    """The production rule takes the resolver words beyond the calls a site update makes anyway from
    continuation rounds of its last Philox block (philox.h: philox4x32_more).  With six planes only
    one word in a hundred gets that far; with ONE plane every second uphill decision is a tie, so a
    word meets ~8 of them and most decisions hang on continuation words (R_4 .. of a single call).
    The sweep must still sample the Boltzmann law: 4 x 4 ferromagnet and a frustrated +-J torus
    against exact enumeration, the mean energy at 4 sigma and the histogram of the energy levels at
    4.5 sigma."""
    L = 4
    a = [x + L * y for y in range(L) for x in range(L)] * 2
    b = [(x + 1) % L + L * y for y in range(L) for x in range(L)] + [x + L * ((y + 1) % L) for y in range(L) for x in range(L)]
    rng = np.random.default_rng(4)
    colors = np.array([(n % L + n // L) & 1 for n in range(L * L)], dtype=np.uint32)
    for j, beta in (([-1.0] * len(a), 0.4), (list(rng.choice([-1.0, 1.0], len(a))), 0.9)):
        edges = [((int(x), int(y)), w) for x, y, w in zip(a, b, j)]
        _, p, en = boltzmann(edges, L * L, beta)
        exact = float((p * en).sum())
        var = float((p * en * en).sum()) - exact ** 2
        E = 4096
        en_m, _ = oracle.msc_mirror(a, b, j, L * L, colors, E, 77 + planes, np.full(50, beta), planes=planes,
                                    per_sweep=True)
        e = en_m[:, -1]
        assert abs(e.mean() - exact) < 4 * np.sqrt(var / E), (planes, beta, e.mean(), exact)
        # energy-level histogram (levels are multiples of 4 |J|)
        levels = np.unique(en)
        pl = np.array([p[en == lv].sum() for lv in levels])
        counts = np.array([(e == lv).sum() for lv in levels])
        z = (counts - E * pl) / np.sqrt(np.maximum(E * pl * (1 - pl), 1e-12))
        assert np.abs(z[pl * E > 5]).max() < 4.5, (planes, beta, z)


def test_mirror_counts_continuation_rounds_without_changing_a_bit(oracle, native):
    """msc_mirror_moves_ex counts the edge-move decisions that read a continuation round (a resolver
    word beyond the K/4 + 1 Philox calls of a decision: philox4x32_more on the device).  Its states
    and energies equal msc_mirror_moves'; at high beta such decisions occur at K = 1 (the 4th tie of
    a word) and at K = 7 (the 2nd); a run without edge passes counts none."""
    rng = np.random.default_rng(6)
    L = 6
    a = [x + L * y for y in range(L) for x in range(L)] * 2
    b = [(x + 1) % L + L * y for y in range(L) for x in range(L)] + [x + L * ((y + 1) % L) for y in range(L) for x in range(L)]
    j = list(rng.choice([-1.0, 1.0], len(a)))
    colors = np.array([(n % L + n // L) & 1 for n in range(L * L)], dtype=np.uint32)
    cls, _ = native.strong_edge_colouring(L * L, a, b)
    betas = np.array([0.3, 3.0, 3.0, 3.0])
    for planes, rounds in ((1, 7), (7, 10)):
        kw = dict(spin_sweeps=1, edge_passes=2, planes=planes, rounds=rounds, per_step=True)
        en, st = oracle.msc_mirror_moves(a, b, j, L * L, colors, cls, 100, 8, betas, **kw)
        cont = np.zeros(1, dtype=np.uint64)
        en2, st2 = oracle.msc_mirror_moves(a, b, j, L * L, colors, cls, 100, 8, betas, continuations=cont, **kw)
        assert (st == st2).all() and (en == en2).all()
        assert cont[0] > 0, (planes, rounds)
        oracle.msc_mirror_moves(a, b, j, L * L, colors, cls, 100, 8, betas, spin_sweeps=1, edge_passes=0,
                                planes=planes, rounds=rounds, continuations=cont)
        assert cont[0] == 0
