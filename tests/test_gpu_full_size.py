"""Full BASELINE sizes on one B200: size-independent properties (configs 2 and 4)."""
import json
import os
import time

import numpy as np
import pytest

from mirror_check import random_regular

pytestmark = pytest.mark.gpu

GOLD = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "exact_2d_ising.json")))


def test_config2_full_size_vs_onsager(native):
    """2D ferromagnet 4096 x 4096, 1024 experiments (2 GiB of packed spins, larger than L2).
    Away from T_c the infinite-lattice Onsager energy is reached within tens of sweeps:
    beta = 0.30 from a random start, beta = 0.60 from the ordered state."""
    ctx = native.Context.get(0)
    L, E = 4096, 1024
    g = native.Graph.torus(ctx, (L, L), j0=-1.0)
    assert g.kind == native.KIND_STENCIL2D
    sim = native.Sim(g, E, 2025)
    sim.sweeps([0.30] * 57)
    per = sim.sweeps([0.30] * 3, per_sweep_energies=True)      # fused accumulation ...
    assert (per[:, -1] == sim.energies()).all()                 # ... == the separate energy pass
    assert (per[:, 0] != per[:, 2]).any()
    e = sim.energies() / (L * L)
    exact = GOLD["onsager"]["b0.3"]["e_per_site"]
    assert abs(e.mean() - exact) < 2e-4, (e.mean(), exact)
    assert e.std() < 5e-4                      # 1.7e7 sites: per-experiment noise ~ 2e-4
    m = sim.magnetization() / (L * L)
    assert np.abs(m).max() < 5e-3
    # a 32-experiment shard at offset 992 reproduces experiments 992..1023 (multi-GPU split)
    shard = native.Sim(g, 32, 2025, replica_offset=992)
    shard.sweeps([0.30] * 60)
    assert (shard.energies() == sim.energies()[992:]).all()
    shard.close()
    sim.set_state(np.ones(L * L, dtype=bool))
    sim.sweeps([0.60] * 60)
    e = sim.energies() / (L * L)
    exact = GOLD["onsager"]["b0.6"]
    assert abs(e.mean() - exact["e_per_site"]) < 3e-4, (e.mean(), exact)
    m = sim.magnetization() / (L * L)
    assert abs(m.mean() - exact["m"]) < 3e-4, (m.mean(), exact["m"])
    st = sim.stats()
    assert st["flip_attempts"] == 120 * E * L * L
    sim.close()


def test_config4_full_size_tempering(native):
    """Random 3-regular graph, N = 10^6, 64 betas geometric in [0.1, 1.5], swap every 10 sweeps."""
    import pyisingmontecarlo_b200 as pkg

    rng = np.random.default_rng(2026)
    n = 1_000_000
    a, b = random_regular(n, 3, rng)
    lat = pkg.Lattice.from_arrays(a, b, np.full(len(a), -1.0))
    g = lat.graph()
    assert g.kind == native.KIND_GENERAL and g.max_degree == 3 and 3 <= g.ncolors <= 4
    colors = g.colors()
    assert (colors[a] != colors[b]).all()
    betas = np.geomspace(0.1, 1.5, 64)
    pt = native.Tempering(g, betas, seed=7)
    acc = np.zeros(64)
    for step in range(12):
        en = pt.sweeps(10)
        acc[pt.slots()] += en
        pt.swap_step(en)
    assert pt.total_swaps() > 0
    slots = pt.slots()
    e_by_slot = np.empty(64)
    e_by_slot[slots] = en
    # hotter slots have higher energy; the hottest matches the Bethe-lattice paramagnet
    assert (np.diff(e_by_slot) < 0).mean() > 0.9
    assert abs(e_by_slot[0] / n + 1.5 * np.tanh(0.1)) < 2e-3, e_by_slot[0] / n
    assert e_by_slot[-1] / n < -1.2
    st = pt.local_states()
    assert st.shape == (64, n)
    # energy of one returned configuration recomputed on the host
    s = st[5].astype(np.int8) * 2 - 1
    assert en[5] == float(-(s[a].astype(np.int64) * s[b]).sum())


def test_config2_beta_sweep_around_tc_vs_onsager(native):
    """BASELINE config 2 as stated: 4096 x 4096 ferromagnet, 1024 experiments, a beta sweep around
    T_c (beta_c = 0.4407) against Onsager's infinite-lattice energy (L = 4096 is 170+ correlation
    lengths at every point, so finite-size corrections are far below the error bar).  Hot starts
    above T_c, ordered starts below (a hot start below T_c coarsens for ~L^2 sweeps); the number
    of sweeps is >= 8 autocorrelation times xi^2.17 of the checkerboard Metropolis dynamics, and
    >= 2000.  Tolerance: 3 sigma of the mean over the 1024 independent experiments, measured from
    their spread, plus 5e-5 for the residual of the exponential relaxation."""
    ctx = native.Context.get(0)
    L, E = 4096, 1024
    g = native.Graph.torus(ctx, (L, L), j0=-1.0)
    plan = [(0.40, 2000, False), (0.42, 3000, False), (0.43, 10000, False),
            (0.45, 4000, True), (0.46, 2000, True), (0.48, 2000, True)]
    sim = native.Sim(g, E, 4242)
    for beta, sweeps, cold in plan:
        if cold:
            sim.set_state(np.ones(L * L, dtype=bool))
        else:
            sim.randomize()
        sim.sweeps(np.full(sweeps, beta))
        e = sim.energies() / (L * L)
        exact = GOLD["onsager"][f"b{beta}"]
        sigma = e.std(ddof=1) / np.sqrt(E)
        assert abs(e.mean() - exact["e_per_site"]) < 3 * sigma + 5e-5, (beta, e.mean(), exact, sigma)
        m = np.abs(sim.magnetization()) / (L * L)
        if cold:
            sm = m.std(ddof=1) / np.sqrt(E)
            assert abs(m.mean() - exact["m"]) < 3 * sm + 2e-4, (beta, m.mean(), exact["m"], sm)
        else:
            # |m| of a 4096^2 lattice at xi ~ 23 (beta = 0.43): chi / N fluctuations of a few 1e-3
            assert m.mean() < 0.02 and m.max() < 0.08, (beta, m.mean(), m.max())
    sim.close()


def test_config1_full_replay_1000_timesteps(native, oracle):
    """North-star check 1 at BASELINE config 1's full length: 32 x 32 ferromagnet, beta = 0.44, 64
    experiments, 1000 timesteps of 1024 attempts.  The oracle emits the reference algorithm's own
    (site, uniform) trace (786 MB); the device must reproduce states and energies bit for bit."""
    import pyisingmontecarlo_b200 as pkg

    edges = oracle.square_edges(32)
    og = oracle.Graph(edges)
    lat = pkg.Lattice(edges, seed_gen=0)
    seeds = np.array(lat.make_seeds(64), dtype=np.uint64)
    sites, u, init, en_o, st_o = og.trace(0.44, seeds, 1000 * 1024)
    assert sites.shape == (64, 1000 * 1024)
    en_r, st_r = lat.replay(0.44, sites, u, init)
    assert (st_r == st_o).all() and (en_r == en_o).all()
    kauf = GOLD["kaufman"]["L32_b0.44"]
    sd = np.sqrt(kauf["c_per_site"] / (0.44 ** 2 * 1024))
    assert abs(en_r.mean() / 1024 - kauf["e_per_site"]) < 4 * sd / np.sqrt(64)


def test_config5_full_size_band_vs_mirror(native, oracle):
    """BASELINE config 5 on one GPU: a 65536 x 65536 lattice (512 MiB packed).  The CPU mirror can
    not sweep 4.3e9 sites, but a decision depends only on global coordinates, so a band of rows
    recomputed from the same Philox initial state must equal the device's rows wherever the
    band's neighbours are known (oracle/msc_mirror.c: msc_mirror_single_band) - at the top of the
    lattice, in the middle, and across the word boundary rows of a strip's interior."""
    import pyisingmontecarlo_b200 as pkg

    L = 65536
    lat = pkg.SingleLattice2D(L, seed=31)
    betas = [0.44, 0.30]
    lat.sweeps(betas)
    n = len(betas)
    for y0 in (1, 32760, L - 14):
        nrows = 13 if y0 != 32760 else 17
        if y0 + nrows >= L:
            nrows = L - 1 - y0
        band = oracle.msc_mirror_single_band(L, y0, nrows, -1.0, 31, betas)
        got = lat.strip.rows(y0 + 2 * n, y0 + nrows - 2 * n)
        assert (got == band[2 * n: nrows - 2 * n]).all(), y0
    nsat, up = lat.strip.global_sums()
    assert lat.energy() == 2.0 * L * L - 2.0 * nsat
