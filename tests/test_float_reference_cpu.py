"""The f64 reference of the float-field path (tests/float_reference.py) pinned on its own, without
any kernel: its Philox equals the oracle's, and its sweeps, edge passes and worms are a sound
Metropolis chain (exact enumeration of the Boltzmann law), so the decision-level gates built on it
(test_device_source_on_host.py, test_gpu_float_path.py) compare the kernels with a correct chain."""
import numpy as np
import pytest

import float_reference as fr
from moves_cases import boltzmann, histogram_z, irregular_graph


@pytest.mark.parametrize("rounds", [7, 10])
def test_philox_equals_the_oracle(oracle, rounds):
    rng = np.random.default_rng(rounds)
    ctr = rng.integers(0, 2**32, size=(40, 4), dtype=np.uint64)
    ctr[:, 3] = (ctr[:, 3] & 0xFF) | (rng.integers(0, 256, 40, dtype=np.uint64) << 8) | \
        (rng.integers(0, 6, 40, dtype=np.uint64) << 24)            # call | pass << 8 | tag << 24
    key = rng.integers(0, 2**32, size=2, dtype=np.uint64)
    got = fr.philox(ctr[:, 0], ctr[:, 1], ctr[:, 2], ctr[:, 3], key[0], key[1], rounds)
    for i in range(len(ctr)):
        want = oracle.philox4x32([int(x) for x in ctr[i]], [int(key[0]), int(key[1])], rounds)
        assert [int(w[i]) for w in got] == list(want)


def _sparse_graph():
    """the graph of test_float_kernels_on_the_host_sample_the_boltzmann_law"""
    from test_device_source_on_host import greedy_colouring, random_sparse

    rng = np.random.default_rng(17)
    n = 10
    a, b = random_sparse(n, 18, rng, 6)
    j = rng.normal(size=len(a))
    bias = rng.normal(size=n) * 0.4
    col, _ = greedy_colouring(n, a, b)
    return n, a, b, j, bias, col


def test_reference_sweeps_sample_the_boltzmann_law():
    n, a, b, j, bias, col = _sparse_graph()
    g = fr.Graph(n, a, b, j, bias, col)
    beta, E = 0.6, 4096
    edges = [((int(x), int(y)), float(w)) for x, y, w in zip(a, b, g.jq)]
    states, p, en = boltzmann(edges, n, beta, g.bq)
    rng = np.random.default_rng(1)
    ch = fr.Chain(g, rng.integers(0, 2, size=(E, n)).astype(bool), 0xF10A7)
    for t in range(40):
        ch.sweep(t, beta)
    # <E> and every <s_i> within 4.5 sigma of the enumeration (many states are too rare for a histogram)
    s = ch.s * 2.0 - 1
    obs = np.concatenate([(s[:, a] * s[:, b] * g.jq).sum(1, keepdims=True) - s @ g.bq[:, None], s], axis=1)
    exact = np.concatenate([[(p * en).sum()], p @ (states * 2.0 - 1)])
    z = (obs.mean(0) - exact) / (obs.std(0, ddof=1) / np.sqrt(E))
    assert np.abs(z).max() < 4.5, z
    assert ch.in_band < 1e-3 * ch.decisions


@pytest.mark.parametrize("moves", [
    dict(spin_sweeps=0, edge_passes=1, worms=2, worm_len=3),
    dict(spin_sweeps=0, edge_passes=2, worms=1, worm_len=2, importance=True),
    dict(spin_sweeps=0, edge_passes=0, worms=6, worm_len=1),
    dict(spin_sweeps=0, edge_passes=1, worms=3, worm_len=4),
    dict(spin_sweeps=1, edge_passes=1, worms=2, worm_len=5, importance=True),
    dict(spin_sweeps=0, edge_passes=1, worms=2, worm_len=8),
])
def test_reference_moves_sample_the_boltzmann_law(moves):
    """edge passes (with and without importance weights) and worms of every length on the irregular
    graph of the move tests; chains of moves that conserve the parity of the up spins are compared
    per parity sector"""
    from test_device_source_on_host import greedy_colouring, strong_edge_colouring

    edges, n, biases = irregular_graph()
    a = np.array([e[0][0] for e in edges]); b = np.array([e[0][1] for e in edges])
    j = np.array([e[1] for e in edges])
    col, _ = greedy_colouring(n, a, b)
    g = fr.Graph(n, a, b, j, biases, col, strong_edge_colouring(n, a, b))
    beta, E = 0.8, 8192
    _, p, _ = boltzmann([((int(x), int(y)), float(w)) for x, y, w in zip(a, b, g.jq)], n, beta, g.bq)
    rng = np.random.default_rng(moves["worm_len"])
    ch = fr.Chain(g, rng.integers(0, 2, size=(E, n)).astype(bool), 2025 + moves["worm_len"])
    for t in range(60):
        ch.timestep(t, beta, moves["spin_sweeps"], moves["edge_passes"], moves["worms"], moves["worm_len"],
                    moves.get("importance", False))
    st = ch.s
    if moves["spin_sweeps"] == 0 and (moves["worm_len"] % 2 == 0 or moves["worm_len"] > n):
        par = st.sum(1) % 2
        parity_of_state = np.array([bin(i).count("1") % 2 for i in range(2 ** n)])
        for sector in (0, 1):
            ps = np.where(parity_of_state == sector, p, 0.0)
            z = histogram_z(st[par == sector], ps / ps.sum())[parity_of_state == sector]
            assert np.abs(z).max() < 4.5, z
    else:
        z = histogram_z(st, p)
        assert np.abs(z).max() < 4.5, z


def test_decide_limits():
    """beta = 0 accepts everything (the sweep rejects only u = 2^32 - 1, in band), beta = 1e6 rejects
    every uphill move, an exact zero field with beta = 1e6 stays determined"""
    u = np.array([0, 2**31, 2**32 - 2, 2**32 - 1], dtype=np.uint64)
    acc, band = fr.decide(u, np.full(4, 2.0), np.full(4, 1e-6), 0.0)
    assert acc.all() and (band == [False, False, True, True]).all()      # 2^32 - 2 lies within 4 ulp of 1
    acc, band = fr.decide(u, np.full(4, 0.5), np.full(4, 1e-6), 1e6)
    assert not acc.any() and not band.any()
    acc, band = fr.decide(u, np.full(4, -0.5), np.full(4, 1e-6), 1e6)
    assert acc.all() and not band.any()
    acc, band = fr.decide(u, np.zeros(4), np.zeros(4), 1e6, kind="edge")
    assert acc.all() and not band.any()
