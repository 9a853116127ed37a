"""ctypes wrapper of the CPU oracle (oracle/ising_oracle.c, oracle/msc_mirror.c).

Test infrastructure: imported by tests/, __graft_entry__.smoke() and bench.py's CPU-baseline
legs only.  Builds oracle/_build/libising_oracle.so with `make -C oracle` when it is missing.
"""
import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
LIB_PATH = os.path.join(ORACLE_DIR, "_build", "libising_oracle.so")

_lib = None
_P = C.c_void_p
_U64 = C.c_uint64


def build(force=False):
    srcs = [os.path.join(ORACLE_DIR, f) for f in ("ising_oracle.c", "msc_mirror.c", "Makefile")]
    stale = (not os.path.exists(LIB_PATH)) or any(
        os.path.exists(s) and os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in srcs)
    if force or stale:
        res = subprocess.run(["make", "-C", ORACLE_DIR] + (["-B"] if force else []),
                             capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("oracle build failed:\n" + res.stdout + res.stderr)
    return LIB_PATH


def lib():
    global _lib
    if _lib is None:
        build()
        h = C.CDLL(LIB_PATH)
        h.orc_next_u64.restype = _U64
        h.orc_next_u64.argtypes = [_P]
        h.orc_gen_range.restype = _U64
        h.orc_gen_range.argtypes = [_P, _U64]
        h.orc_gen_f64.restype = C.c_double
        h.orc_gen_f64.argtypes = [_P]
        h.orc_gen_bool.restype = C.c_int
        h.orc_gen_bool.argtypes = [_P]
        h.orc_seed_from_u64.restype = None
        h.orc_seed_from_u64.argtypes = [_U64, _P]
        h.orc_make_seeds.restype = None
        h.orc_make_seeds.argtypes = [_U64, _U64, _P]
        h.orc_graph_new.restype = _P
        h.orc_graph_new.argtypes = [_U64, _U64, _P, _P, _P, _P]
        h.orc_graph_free.restype = None
        h.orc_graph_free.argtypes = [_P]
        h.orc_energy.restype = C.c_double
        h.orc_energy.argtypes = [_P, _P]
        h.orc_run_monte_carlo.restype = C.c_int
        h.orc_run_monte_carlo.argtypes = [_P, C.c_double, _U64, _U64, _P, _P, _U64, _P, _P]
        h.orc_run_moves.restype = C.c_int
        h.orc_run_moves.argtypes = [_P, _P, _P, _P, C.c_double, _U64, _U64, _P, _P, _U64, _U64, _U64, _U64,
                                    C.c_int, _P, _P]
        h.orc_run_sampling.restype = C.c_int
        h.orc_run_sampling.argtypes = [_P, C.c_double, _U64, _U64, _P, _P, _U64, _U64, _U64, _P, _P]
        h.orc_schedule_betas.restype = C.c_int
        h.orc_schedule_betas.argtypes = [_P, _P, _U64, _U64, C.c_int, _P]
        h.orc_run_annealing.restype = C.c_int
        h.orc_run_annealing.argtypes = [_P, _P, _U64, _U64, _P, _P, _U64, C.c_int, _P, _P]
        h.orc_trace.restype = C.c_int
        h.orc_trace.argtypes = [_P, C.c_double, _U64, _P, _P, _U64, _P, _P, _P, _P, _P]
        h.orc_replay.restype = C.c_int
        h.orc_replay.argtypes = [_P, C.c_double, _U64, _U64, _P, _P, _P, _P, _P]
        h.orc_pt_run.restype = C.c_int
        h.orc_pt_run.argtypes = [_P, _U64, _P, _U64, _U64, _U64, _U64, _U64, _P, _P, _P]
        h.orc_num_threads.restype = C.c_int
        h.orc_num_threads.argtypes = []
        h.orc_set_num_threads.restype = None
        h.orc_set_num_threads.argtypes = [C.c_int]
        h.msc_philox4x32.restype = None
        h.msc_philox4x32.argtypes = [C.c_int, _P, _P, _P]
        h.msc_mirror_run.restype = C.c_int
        h.msc_mirror_run.argtypes = [_U64, _U64, _P, _P, _P, _P, C.c_uint32, _U64, _U64, _U64,
                                     C.c_int, C.c_int, C.c_int, _P, _P, _U64, _U64, _P, _P, _P,
                                     C.c_int]
        h.msc_mirror_pt.restype = C.c_int
        h.msc_mirror_pt.argtypes = [_U64, _U64, _P, _P, _P, _P, C.c_uint32, _U64, _P, _U64, C.c_int,
                                    C.c_int, _U64, _U64, _U64, _P, _P, _P, _P]
        h.msc_mirror_pt_ex.restype = C.c_int
        h.msc_mirror_pt_ex.argtypes = h.msc_mirror_pt.argtypes + [_P, _P]
        h.msc_mirror_single.restype = C.c_int
        h.msc_mirror_single.argtypes = [_U64, _U64, C.c_double, _U64, C.c_int, C.c_int, C.c_int, _P,
                                        _U64, _P, _P]
        _lib = h
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Rng:
    """rand 0.8 SmallRng restated (xoshiro256++)."""

    def __init__(self, seed=None, state=None):
        self.s = np.zeros(4, dtype=np.uint64)
        if state is not None:
            self.s[:] = state
        else:
            lib().orc_seed_from_u64(int(seed), _p(self.s))

    def next_u64(self):
        return int(lib().orc_next_u64(_p(self.s)))

    def gen_range(self, n):
        return int(lib().orc_gen_range(_p(self.s), int(n)))

    def gen_f64(self):
        return float(lib().orc_gen_f64(_p(self.s)))

    def gen_bool(self):
        return bool(lib().orc_gen_bool(_p(self.s)))


def make_seeds(seed_gen, n):
    out = np.empty(n, dtype=np.uint64)
    lib().orc_make_seeds(int(seed_gen), n, _p(out))
    return out


class Graph:
    def __init__(self, edges=None, arrays=None, nvars=None, biases=None):
        if arrays is not None:
            a, b, j = arrays
        else:
            a = [e[0][0] for e in edges]
            b = [e[0][1] for e in edges]
            j = [e[1] for e in edges]
        self.a = np.ascontiguousarray(a, dtype=np.uint64)
        self.b = np.ascontiguousarray(b, dtype=np.uint64)
        self.j = np.ascontiguousarray(j, dtype=np.float64)
        self.nvars = int(max(self.a.max(), self.b.max())) + 1 if nvars is None else int(nvars)
        self.biases = None if biases is None else np.ascontiguousarray(biases, dtype=np.float64)
        self.h = lib().orc_graph_new(self.nvars, len(self.a), _p(self.a), _p(self.b), _p(self.j),
                                     _p(self.biases))

    def __del__(self):
        try:
            lib().orc_graph_free(self.h)
        except Exception:
            pass

    def energy(self, state):
        s = np.ascontiguousarray(state, dtype=np.uint8)
        return float(lib().orc_energy(self.h, _p(s)))

    def _init(self, initial_state):
        return None if initial_state is None else np.ascontiguousarray(initial_state, dtype=np.uint8)

    def run_monte_carlo(self, beta, timesteps, seeds, initial_state=None, attempts_per_step=0):
        seeds = np.ascontiguousarray(seeds, dtype=np.uint64)
        E = len(seeds)
        energies = np.zeros(E)
        states = np.zeros((E, self.nvars), dtype=np.uint8)
        init = self._init(initial_state)
        rc = lib().orc_run_monte_carlo(self.h, float(beta), timesteps, E, _p(seeds), _p(init),
                                       attempts_per_step, _p(energies), _p(states))
        assert rc == 0
        return energies, states.astype(bool)

    def run_moves(self, beta, timesteps, seeds, nspin=0, nedge=0, nworm=0, worm_len=4, importance=False,
                  initial_state=None):
        """Timesteps of explicit move counts (orc_run_moves) -> (energies[E], states bool[E, nvars])."""
        seeds = np.ascontiguousarray(seeds, dtype=np.uint64)
        E = len(seeds)
        energies = np.zeros(E)
        states = np.zeros((E, self.nvars), dtype=np.uint8)
        init = self._init(initial_state)
        rc = lib().orc_run_moves(self.h, _p(self.a), _p(self.b), _p(self.j), float(beta), timesteps, E,
                                 _p(seeds), _p(init), nspin, nedge, nworm, worm_len, int(importance),
                                 _p(energies), _p(states))
        assert rc == 0
        return energies, states.astype(bool)

    def run_sampling(self, beta, timesteps, seeds, initial_state=None, attempts_per_step=0,
                     thermalization=0, sampling_freq=1):
        seeds = np.ascontiguousarray(seeds, dtype=np.uint64)
        E = len(seeds)
        ns = timesteps // sampling_freq
        energies = np.zeros((E, ns))
        states = np.zeros((E, ns, self.nvars), dtype=np.uint8)
        init = self._init(initial_state)
        rc = lib().orc_run_sampling(self.h, float(beta), timesteps, E, _p(seeds), _p(init),
                                    attempts_per_step, thermalization, sampling_freq,
                                    _p(energies), _p(states))
        assert rc == 0
        return energies, states.astype(bool)

    def run_annealing(self, stops, timesteps, seeds, initial_state=None, attempts_per_step=0,
                      q1_compat=True, per_step_energies=False):
        betas = schedule_betas(stops, timesteps, q1_compat)
        seeds = np.ascontiguousarray(seeds, dtype=np.uint64)
        E = len(seeds)
        energies = np.zeros((E, timesteps) if per_step_energies else (E,))
        states = np.zeros((E, self.nvars), dtype=np.uint8)
        init = self._init(initial_state)
        rc = lib().orc_run_annealing(self.h, _p(betas), timesteps, E, _p(seeds), _p(init),
                                     attempts_per_step, int(per_step_energies), _p(energies),
                                     _p(states))
        assert rc == 0
        return energies, states.astype(bool)

    def trace(self, beta, seeds, nattempts, initial_state=None):
        seeds = np.ascontiguousarray(seeds, dtype=np.uint64)
        E = len(seeds)
        sites = np.zeros((E, nattempts), dtype=np.uint32)
        u = np.zeros((E, nattempts), dtype=np.float64)
        init_out = np.zeros((E, self.nvars), dtype=np.uint8)
        energies = np.zeros(E)
        states = np.zeros((E, self.nvars), dtype=np.uint8)
        init = self._init(initial_state)
        rc = lib().orc_trace(self.h, float(beta), E, _p(seeds), _p(init), nattempts, _p(sites),
                             _p(u), _p(init_out), _p(energies), _p(states))
        assert rc == 0
        return sites, u, init_out.astype(bool), energies, states.astype(bool)

    def replay(self, beta, sites, u, init):
        sites = np.ascontiguousarray(sites, dtype=np.uint32)
        u = np.ascontiguousarray(u, dtype=np.float64)
        init = np.ascontiguousarray(init, dtype=np.uint8)
        E, A = sites.shape
        energies = np.zeros(E)
        states = np.zeros((E, self.nvars), dtype=np.uint8)
        rc = lib().orc_replay(self.h, float(beta), E, A, _p(sites), _p(u), _p(init), _p(energies),
                              _p(states))
        assert rc == 0
        return energies, states.astype(bool)

    def pt_run(self, betas, container_seed, timesteps, replica_swap_freq=1, sampling_freq=1,
               attempts_per_step=0):
        betas = np.ascontiguousarray(betas, dtype=np.float64)
        R = len(betas)
        ns = timesteps // sampling_freq
        states = np.zeros((R, ns, self.nvars), dtype=np.uint8)
        energies = np.zeros(R)
        swaps = C.c_uint64(0)
        rc = lib().orc_pt_run(self.h, R, _p(betas), int(container_seed), timesteps,
                              replica_swap_freq, sampling_freq, attempts_per_step, _p(states),
                              _p(energies), C.byref(swaps))
        assert rc == 0
        return states.astype(bool), energies, int(swaps.value)


def schedule_betas(stops, timesteps, q1_compat=True):
    t = np.ascontiguousarray([s[0] for s in stops], dtype=np.uint64)
    b = np.ascontiguousarray([s[1] for s in stops], dtype=np.float64)
    out = np.zeros(timesteps)
    rc = lib().orc_schedule_betas(_p(t), _p(b), len(t), timesteps, int(q1_compat), _p(out))
    assert rc == 0
    return out


def msc_mirror_moves(a, b, j, nvars, colors, edge_cls, E, seed, betas, *, spin_sweeps=1, edge_passes=1,
                     replica_offset=0, planes=6, rounds=7, per_step=False, states=None, continuations=None):
    """Timesteps of a colour-class sweep + passes of bit-sliced edge moves as the device runs them
    (oracle/msc_mirror.c: msc_mirror_moves) -> (energies[E, n] or None, states bool[E, nvars]);
    starts from `states` when given, else from the Philox initial state.  continuations: uint64[1]
    or None; receives the number of edge-move decisions that read a continuation-round word (a
    resolver word beyond the K/4 + 1 Philox calls every decision makes)."""
    a = np.ascontiguousarray(a, dtype=np.uint64)
    b = np.ascontiguousarray(b, dtype=np.uint64)
    j = np.ascontiguousarray(j, dtype=np.float64)
    colors = np.ascontiguousarray(colors, dtype=np.uint32)
    edge_cls = np.ascontiguousarray(edge_cls, dtype=np.uint32)
    betas = np.ascontiguousarray(betas, dtype=np.float64)
    st = np.zeros((E, nvars), dtype=np.uint8) if states is None else np.ascontiguousarray(
        states, dtype=np.uint8).copy()
    en = np.zeros((E, len(betas))) if per_step else None
    argtypes = [_U64, _U64, _P, _P, _P, _P, C.c_uint32, _P, C.c_uint32, _U64, _U64, _U64, C.c_int, C.c_int,
                C.c_int, _P, _U64, C.c_int, C.c_uint32, _P, _P]
    args = [nvars, len(a), _p(a), _p(b), _p(j), _p(colors), int(colors.max()) + 1, _p(edge_cls),
            int(edge_cls.max()) + 1, E, int(seed), replica_offset, planes, rounds, int(states is None), _p(betas),
            len(betas), int(spin_sweeps), int(edge_passes), _p(st), _p(en)]
    if continuations is None:
        fn = lib().msc_mirror_moves
    else:
        assert continuations.dtype == np.uint64 and continuations.shape == (1,)
        continuations[0] = 0
        fn = lib().msc_mirror_moves_ex
        argtypes.append(_P)
        args.append(_p(continuations))
    fn.restype = C.c_int
    fn.argtypes = argtypes
    rc = fn(*args)
    assert rc == 0, rc
    return en, st.astype(bool)


OPTIONS = {"uniform_always": 0, "zero_draws": 1, "init_draws": 2, "bias_sign": 3, "pt_pairs": 4}


class options:
    """with oracle_lib.options(uniform_always=1): ...  -- the named alternatives of the recalled
    crate semantics (oracle/ising_oracle.c: ORC_OPT_*); the defaults come back on exit."""

    def __init__(self, **kw):
        self.kw = kw

    def __enter__(self):
        h = lib()
        h.orc_set_option.restype = C.c_int
        h.orc_set_option.argtypes = [C.c_int, C.c_int]
        for k, v in self.kw.items():
            rc = h.orc_set_option(OPTIONS[k], int(v))
            if rc:
                h.orc_reset_options()
                raise ValueError(f"oracle option {k} = {v} rejected")
        return self

    def __exit__(self, *exc):
        lib().orc_reset_options()
        return False


def get_option(name):
    h = lib()
    h.orc_get_option.restype = C.c_int
    h.orc_get_option.argtypes = [C.c_int]
    return int(h.orc_get_option(OPTIONS[name]))


def philox4x32(ctr, key, rounds=10):
    c = np.ascontiguousarray(ctr, dtype=np.uint32)
    k = np.ascontiguousarray(key, dtype=np.uint32)
    out = np.zeros(4, dtype=np.uint32)
    lib().msc_philox4x32(rounds, _p(c), _p(k), _p(out))
    return out


def msc_mirror(a, b, j, nvars, colors, E, seed, betas, *, replica_offset=0, planes=6, rounds=7,
               init_state=None, states=None, sweep0=0, per_sweep=False, per_replica_beta=None,
               nsweeps=None):
    """Scalar restatement of the production sweep (oracle/msc_mirror.c).

    betas: one per sweep; or pass per_replica_beta=[E values] and nsweeps for a run where
    experiment e stays at its own beta (parallel-tempering style)."""
    a = np.ascontiguousarray(a, dtype=np.uint64)
    b = np.ascontiguousarray(b, dtype=np.uint64)
    j = np.ascontiguousarray(j, dtype=np.float64)
    colors = np.ascontiguousarray(colors, dtype=np.uint32)
    if per_replica_beta is not None:
        betas = np.ascontiguousarray(per_replica_beta, dtype=np.float64)
        assert len(betas) == E and nsweeps is not None
        nsw = int(nsweeps)
    else:
        betas = np.ascontiguousarray(betas, dtype=np.float64)
        nsw = len(betas)
    randomize = int(states is None and init_state is None)
    st = np.zeros((E, nvars), dtype=np.uint8) if states is None else np.ascontiguousarray(
        states, dtype=np.uint8).copy()
    init = None if init_state is None else np.ascontiguousarray(init_state, dtype=np.uint8)
    eps = np.zeros((E, nsw)) if per_sweep else None
    fin = np.zeros(E)
    rc = lib().msc_mirror_run(nvars, len(a), _p(a), _p(b), _p(j), _p(colors), int(colors.max()) + 1,
                              E, int(seed), replica_offset, planes, rounds, randomize, _p(init),
                              _p(betas), nsw, sweep0, _p(st), _p(eps), _p(fin),
                              int(per_replica_beta is not None))
    assert rc == 0, rc
    return (eps if per_sweep else fin), st.astype(bool)


def msc_mirror_pt(a, b, j, nvars, colors, betas, seed, timesteps, replica_swap_freq=1,
                  sampling_freq=1, planes=6, rounds=7):
    """Parallel tempering as the device runs it (oracle/msc_mirror.c: msc_mirror_pt)."""
    return _mirror_pt(a, b, j, nvars, colors, betas, seed, timesteps, replica_swap_freq, sampling_freq,
                      planes, rounds, False)


def msc_mirror_pt_ex(a, b, j, nvars, colors, betas, seed, timesteps, replica_swap_freq=1,
                     sampling_freq=1, planes=6, rounds=7):
    """msc_mirror_pt and the per-pair swap statistics (oracle/msc_mirror.c: msc_mirror_pt_ex)
    -> (states, energies, total swaps, slot_of_cfg, attempts uint64[R - 1], accepts uint64[R - 1]);
    pair a is slots (a, a + 1), as ising_pt_get_pair_stats returns them."""
    return _mirror_pt(a, b, j, nvars, colors, betas, seed, timesteps, replica_swap_freq, sampling_freq,
                      planes, rounds, True)


def _mirror_pt(a, b, j, nvars, colors, betas, seed, timesteps, replica_swap_freq, sampling_freq, planes,
               rounds, pair_stats):
    a = np.ascontiguousarray(a, dtype=np.uint64)
    b = np.ascontiguousarray(b, dtype=np.uint64)
    j = np.ascontiguousarray(j, dtype=np.float64)
    colors = np.ascontiguousarray(colors, dtype=np.uint32)
    betas = np.ascontiguousarray(betas, dtype=np.float64)
    R = len(betas)
    ns = timesteps // sampling_freq
    states = np.zeros((R, ns, nvars), dtype=np.uint8)
    energies = np.zeros(R)
    swaps = C.c_uint64(0)
    slots = np.zeros(R, dtype=np.uint32)
    args = [nvars, len(a), _p(a), _p(b), _p(j), _p(colors), int(colors.max()) + 1, R, _p(betas), int(seed),
            planes, rounds, timesteps, replica_swap_freq, sampling_freq, _p(states), _p(energies),
            C.byref(swaps), _p(slots)]
    if not pair_stats:
        rc = lib().msc_mirror_pt(*args)
        assert rc == 0, rc
        return states.astype(bool), energies, int(swaps.value), slots
    attempts = np.zeros(max(R - 1, 0), dtype=np.uint64)
    accepts = np.zeros(max(R - 1, 0), dtype=np.uint64)
    rc = lib().msc_mirror_pt_ex(*args, _p(attempts), _p(accepts))
    assert rc == 0, rc
    return states.astype(bool), energies, int(swaps.value), slots, attempts, accepts


def msc_mirror_single_band(Lx, y0, nrows, j, seed, betas, planes=6, rounds=7):
    """Rows y0 .. y0 + nrows - 1 of a large lattice from its Philox initial state; after len(betas)
    sweeps the rows [2 n, nrows - 2 n) of the result equal the full lattice's (msc_mirror.c)."""
    betas = np.ascontiguousarray(betas, dtype=np.float64)
    st = np.zeros((nrows, Lx), dtype=np.uint8)
    fn = lib().msc_mirror_single_band
    fn.restype = C.c_int
    fn.argtypes = [_U64, _U64, _U64, C.c_double, _U64, C.c_int, C.c_int, C.c_int, _P, _U64, _P]
    rc = fn(Lx, y0, nrows, float(j), int(seed), planes, rounds, 1, _p(betas), len(betas), _p(st))
    assert rc == 0, rc
    return st.astype(bool)


def msc_mirror_single(Lx, Ly, j, seed, betas, planes=6, rounds=7, state=None):
    """One bit-packed 2D lattice as the device runs it (oracle/msc_mirror.c: msc_mirror_single)."""
    betas = np.ascontiguousarray(betas, dtype=np.float64)
    st = np.zeros((Ly, Lx), dtype=np.uint8) if state is None else np.ascontiguousarray(state, dtype=np.uint8).copy()
    en = np.zeros(len(betas))
    rc = lib().msc_mirror_single(Lx, Ly, float(j), int(seed), planes, rounds, int(state is None),
                                 _p(betas), len(betas), _p(st), _p(en))
    assert rc == 0, rc
    return en, st.astype(bool)


# ---- lattice helpers shared by the tests ---------------------------------------------------
def square_edges(L, j=-1.0, order="xy"):
    """BASELINE config 1: [((x*L+y, ((x+1)%L)*L+y), j), ((x*L+y, x*L+(y+1)%L), j)]"""
    edges = []
    for x in range(L):
        for y in range(L):
            edges.append(((x * L + y, ((x + 1) % L) * L + y), j))
            edges.append(((x * L + y, x * L + (y + 1) % L), j))
    return edges


def cubic_edges(L, jfun):
    edges = []
    idx = lambda x, y, z: x + L * (y + L * z)
    for z in range(L):
        for y in range(L):
            for x in range(L):
                n = idx(x, y, z)
                edges.append(((n, idx((x + 1) % L, y, z)), jfun(n, 0)))
                edges.append(((n, idx(x, (y + 1) % L, z)), jfun(n, 1)))
                edges.append(((n, idx(x, y, (z + 1) % L)), jfun(n, 2)))
    return edges
