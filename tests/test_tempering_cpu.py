"""Host-side tempering logic: swap decisions (C ABI, no device) and the sharded replica loop
over torch.distributed with the gloo backend (world_size 2, runs on CPU)."""
import math
import os
import socket
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_shard_range_partitions():
    from pyisingmontecarlo_b200.tempering import shard_range

    for n, world in [(64, 8), (10, 3), (5, 5), (7, 2), (1024, 8)]:
        blocks = [shard_range(n, r, world) for r in range(world)]
        assert blocks[0][0] == 0 and blocks[-1][1] == n
        assert all(blocks[r][1] == blocks[r + 1][0] for r in range(world - 1))
        sizes = [hi - lo for lo, hi in blocks]
        assert max(sizes) - min(sizes) <= 1


def test_decide_swaps_rule(native, oracle):
    """even pairs then odd pairs; always swap when (b_a-b_b)(E_a-E_b) >= 0; otherwise with
    probability exp(.) from Philox(seed; slot, parity, step)."""
    R = 9
    betas = np.linspace(0.2, 1.0, R)
    rng = np.random.default_rng(0)
    slot_of = np.arange(R, dtype=np.uint32)
    cfg_of = np.arange(R, dtype=np.uint32)
    py_slot, py_cfg = slot_of.copy(), cfg_of.copy()
    total = 0
    for step in range(50):
        en = rng.normal(size=R) * 3
        n = native.decide_swaps(betas, en, 1234, step, slot_of, cfg_of)
        cnt = 0
        for parity in (0, 1):
            for a in range(parity, R - 1, 2):
                ca, cb = py_cfg[a], py_cfg[a + 1]
                d = (betas[a] - betas[a + 1]) * (en[ca] - en[cb])
                acc = True
                if d < 0:
                    r = oracle.philox4x32([a, parity, step, 2 << 24], [1234, 0], 10)
                    acc = (float(r[0]) + 0.5) / 2**32 < math.exp(d)
                if acc:
                    py_cfg[a], py_cfg[a + 1] = cb, ca
                    py_slot[cb], py_slot[ca] = a, a + 1
                    cnt += 1
        assert n == cnt
        assert (slot_of == py_slot).all() and (cfg_of == py_cfg).all()
        assert (cfg_of[slot_of] == np.arange(R)).all()
        total += n
    assert 0 < total < 50 * (R - 1)


class FakeStepper:
    """Deterministic stand-in for the device stepper: configuration c's 'energy' and 'state'
    depend only on (c, its current beta, time), so any sharding must give the same history."""

    def __init__(self, native, betas, seed, lo, hi, nvars):
        self.native, self.betas, self.seed = native, np.asarray(betas, float), seed
        self.R, self.lo, self.hi, self.nvars = len(betas), lo, hi, nvars
        self.slot_of = np.arange(self.R, dtype=np.uint32)
        self.cfg_of = np.arange(self.R, dtype=np.uint32)
        self.time, self.step, self.swaps = 0, 0, 0
        self.x = np.arange(self.R, dtype=float)          # per-configuration 'state'

    def sweeps(self, t):
        self.time += t
        for c in range(self.R):                            # every rank evolves all: cheap fake
            self.x[c] = math.sin(self.x[c] * 1.7 + self.betas[self.slot_of[c]] * self.time)
        return -10 * self.x[self.lo:self.hi] * np.arange(self.lo + 1, self.hi + 1)

    def swap_step(self, all_e):
        self.swaps += self.native.decide_swaps(self.betas, all_e, self.seed, self.step, self.slot_of,
                                               self.cfg_of)
        self.step += 1

    def slots(self):
        return self.slot_of.copy()

    def local_states(self):
        s = np.zeros((self.hi - self.lo, self.nvars), dtype=np.bool_)
        for c in range(self.lo, self.hi):
            s[c - self.lo] = (np.arange(self.nvars) * (c + 1) + int(1e3 * self.x[c])) % 3 == 0
        return s


def _worker(rank, world, port, out):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist

    from pyisingmontecarlo_b200 import _native as nat
    from pyisingmontecarlo_b200.tempering import _Collective, run_tempering_loop, shard_range

    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    R, nvars = 11, 13
    betas = np.linspace(0.1, 1.3, R)
    lo, hi = shard_range(R, rank, world)
    counts = [shard_range(R, r, world)[1] - shard_range(R, r, world)[0] for r in range(world)]
    st = FakeStepper(nat, betas, 99, lo, hi, nvars)
    states, en = run_tempering_loop(st, R, nvars, 23, 3, 4, _Collective(), counts)
    np.savez(out + f".{rank}.npz", states=states, en=en, swaps=st.swaps, slots=st.slots())
    dist.destroy_process_group()


def test_sharded_loop_over_gloo_equals_single_process(native, tmp_path):
    import torch.multiprocessing as mp

    from pyisingmontecarlo_b200.tempering import run_tempering_loop

    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    out = str(tmp_path / "pt")
    mp.spawn(_worker, args=(2, port, out), nprocs=2, join=True)
    R, nvars = 11, 13
    betas = np.linspace(0.1, 1.3, R)
    single = FakeStepper(native, betas, 99, 0, R, nvars)
    states, en = run_tempering_loop(single, R, nvars, 23, 3, 4)
    assert single.swaps > 0
    for rank in range(2):
        d = np.load(out + f".{rank}.npz")
        assert (d["states"] == states).all()
        assert np.array_equal(d["en"], en)
        assert int(d["swaps"]) == single.swaps and (d["slots"] == single.slots()).all()


def test_cadence_matches_reference_loop(native):
    """tempering.rs:177-212: run min(to_sample, to_swap, remaining); swap before sample."""
    from pyisingmontecarlo_b200.tempering import run_tempering_loop

    calls = []

    class Probe(FakeStepper):
        def sweeps(self, t):
            calls.append(("run", t))
            return super().sweeps(t)

        def swap_step(self, e):
            calls.append(("swap",))
            super().swap_step(e)

        def local_states(self):
            calls.append(("sample",))
            return super().local_states()

    st = Probe(native, [0.3, 0.6], 1, 0, 2, 4)
    states, en = run_tempering_loop(st, 2, 4, 10, 4, 3)
    assert states.shape == (2, 3, 4)
    assert calls == [("run", 3), ("sample",), ("run", 1), ("swap",), ("run", 2), ("sample",),
                     ("run", 2), ("swap",), ("run", 1), ("sample",), ("run", 1)]
    with pytest.raises(ValueError):
        run_tempering_loop(st, 2, 4, 10, 0, 3)


def test_lattice_tempering_surface_without_gpu():
    """The argument handling of LatticeTempering (tempering.rs:43-117) needs no device: replicas are
    classical (transverse field 0), share the lattice and one longitudinal field, and nothing is
    compiled before the first run."""
    import pyisingmontecarlo_b200 as pkg

    with pytest.raises(ValueError, match="Must supply some edges for graph"):
        pkg.LatticeTempering([])
    edges = [((0, 1), -1.0), ((1, 2), 0.5), ((2, 0), 1.25)]
    lt = pkg.LatticeTempering(edges, seed=3)
    assert lt.nvars == 3 and lt.get_num_graphs() == 0 and lt.get_total_swaps() == 0
    lt.add_graph(0.0, 0.25, 0.4)
    lt.add_graph(0.0, 0.25, 0.8, None, None, None)
    assert lt.get_num_graphs() == 2
    with pytest.raises(NotImplementedError, match="transverse"):
        lt.add_graph(0.5, 0.25, 1.0)
    with pytest.raises(NotImplementedError, match="share the longitudinal field"):
        lt.add_graph(0.0, 0.0, 1.0)
    with pytest.raises(NotImplementedError, match="per-replica edge lists"):
        lt.add_graph(0.0, 0.25, 1.0, edges)
    assert lt.get_num_graphs() == 2
    cp = lt.clone()                       # nothing on the device yet: a host-side copy
    assert cp.get_num_graphs() == 2 and cp.nvars == 3 and cp is not lt
    cp.add_graph(0.0, 0.25, 1.2)
    assert lt.get_num_graphs() == 2 and cp.get_num_graphs() == 3
    with pytest.raises(ValueError, match="Attempted to get graph 5 of 2"):
        lt.get_graph_itime(5)
    with pytest.raises(NotImplementedError):
        lt.run_quantum_monte_carlo_and_measure_variable_autocorrelation
    with pytest.raises(AttributeError):
        lt.no_such_method


@pytest.mark.parametrize("R,timesteps,swap_freq,rounds", [(21, 37, 3, 7), (16, 20, 1, 10), (9, 11, 4, 7)])
def test_mirror_pair_statistics(oracle, R, timesteps, swap_freq, rounds):
    """msc_mirror_pt_ex returns what msc_mirror_pt returns, bit for bit, and the swaps tried and taken
    per pair of neighbouring slots: every pair is tried once per swap step (even pairs, then odd
    pairs), and the accepts add up to the total swap count."""
    L = 6
    rng = np.random.default_rng(R)
    a = np.array([x * L + y for x in range(L) for y in range(L)] * 2)
    b = np.array([((x + 1) % L) * L + y for x in range(L) for y in range(L)]
                 + [x * L + (y + 1) % L for x in range(L) for y in range(L)])
    j = np.where(rng.random(len(a)) < 0.5, -1.0, 1.0)
    colors = np.array([(n // L + n % L) & 1 for n in range(L * L)], dtype=np.uint32)
    betas = np.geomspace(0.1, 2.0, R)
    args = (a, b, j, L * L, colors, betas, 99, timesteps, swap_freq, 5)
    st, en, swaps, slots = oracle.msc_mirror_pt(*args, rounds=rounds)
    st2, en2, swaps2, slots2, attempts, accepts = oracle.msc_mirror_pt_ex(*args, rounds=rounds)
    assert (st == st2).all() and (en == en2).all() and swaps == swaps2 and (slots == slots2).all()
    assert attempts.shape == accepts.shape == (R - 1,)
    steps = timesteps // swap_freq
    assert (attempts == steps).all(), (attempts, steps)
    assert int(accepts.sum()) == swaps > 0
    assert (accepts <= attempts).all() and (accepts < attempts).any()
