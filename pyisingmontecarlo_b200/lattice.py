"""`Lattice` -- host-side mirror of the reference pyclass (src/lattice.rs:27-470) for the
classical Monte-Carlo path, running on libising_b200 (CUDA, sm_100a) through its C ABI.

Same names, argument order, defaults, return dtypes/shapes and error behaviour as the
reference's `py_monte_carlo.Lattice`; the quantum methods (lattice.rs:472-1069) stay on the
reference.  Documented deviations of the GPU path (SURVEY.md 8b):
  D1  with `only_basic_moves` None / False the reference's timestep also performs two-spin edge
      moves and worm moves whose rules live in the out-of-tree `qmc` crate.  By default only
      single-spin sweeps run (warned once per process); `Lattice.non_basic_moves = True` makes
      such calls also run one pass of two-spin edge moves and one 4-site worm move per
      experiment in every timestep (this engine's restatement of those moves, csrc/moves.cu);
  D2  `edge_move_importance_sampling=True` needs `non_basic_moves` (it only affects the edge
      moves) and raises NotImplementedError without it;
  D3  a timestep is one colour-class sweep (every site attempted once) instead of nvars
      attempts at uniformly random sites: same Boltzmann law, different transient.
"""
import secrets
import warnings

import numpy as np

from . import _native as nat

_U64 = 2**64 - 1
_warned_basic_moves = False


def _user_stacklevel():
    """stacklevel that points a warning at the first frame outside this package"""
    import sys

    here = __name__.rsplit(".", 1)[0]
    level, f = 1, sys._getframe(1)
    while f is not None and f.f_globals.get("__name__", "").startswith(here):
        level, f = level + 1, f.f_back
    return level


def warn_non_basic_moves(only_basic_moves):
    """Deviation D1, said out loud once per process: with only_basic_moves None / False the
    reference's timestep also performs two-spin edge flips and worm updates (lattice.rs:205,
    classicising.rs:100-106; their rules live in the out-of-tree `qmc` crate).  The GPU path
    performs single-spin Metropolis sweeps - the same Boltzmann distribution, other dynamics."""
    global _warned_basic_moves
    if only_basic_moves or _warned_basic_moves:
        return
    _warned_basic_moves = True
    warnings.warn("only_basic_moves is None/False: the reference would also perform edge-flip and worm "
                  "moves in each timestep; the B200 engine performs single-spin Metropolis sweeps only "
                  "(same equilibrium distribution, different dynamics; see DESIGN.md deviation D1). "
                  "Pass only_basic_moves=True to state that this is what you want, or set "
                  "Lattice.non_basic_moves = True to run this engine's edge and worm moves as well.",
                  UserWarning, stacklevel=_user_stacklevel())


def _edges_to_arrays(edges):
    n = len(edges)
    a = np.empty(n, dtype=np.uint64)
    b = np.empty(n, dtype=np.uint64)
    j = np.empty(n, dtype=np.float64)
    for k, ((x, y), w) in enumerate(edges):
        if x < 0 or y < 0:
            raise OverflowError("can't convert negative int to unsigned")  # pyo3's usize conversion
        a[k], b[k], j[k] = x, y, w
    return a, b, j


class Lattice:
    """A lattice for running ising monte carlo simulations. Takes a list of edges: ((a, b), j), ...

    Creates new initial conditions each time simulations are run, does not preserve any internal
    state for the lattice variables (spins).  (lattice.rs:24-39)
    """

    def __init__(self, edges, seed_gen=None, use_allocator=None, *, device=None):
        # lattice.rs:46-73
        if len(edges) == 0:
            raise ValueError("Must supply some edges for graph")
        self._a, self._b, self._j = _edges_to_arrays(edges)
        self._init_common(int(max(self._a.max(), self._b.max())) + 1, seed_gen, use_allocator, device)

    def _init_common(self, nvars, seed_gen, use_allocator, device):
        self.nvars = nvars
        self._torus = None
        self._bias_global = 0.0
        self._bias_individual = None
        self._transverse = None
        self._initial_state = None
        self._enable_rvb_updates = False
        self._enable_heatbath = False
        self._seed_gen = None if seed_gen is None else int(seed_gen) & _U64
        self._use_allocator = True if use_allocator is None else bool(use_allocator)
        self._device = device
        self._graph = None
        # knobs of the device path that do not exist in the reference (defaults = parity mode)
        self.linear_annealing = False   # False reproduces the reference's schedule quirk Q1
        # True: calls with only_basic_moves None / False also run two-spin edge moves and worm
        # moves in every timestep (deviation D1); False: single-spin sweeps only, with a warning
        self.non_basic_moves = False
        # multi-GPU (one process per GPU, torch.distributed initialised): shard the experiments
        # over the ranks in blocks of 32 (the reference's rayon axis, lattice.rs:192-197) and,
        # when gather_results is set, all-gather so that every rank returns the full arrays
        self.distributed = False
        self.gather_results = True
        self.process_group = None
        self.msc_planes = 0             # 0 = library default
        self.philox_rounds = 0

    # ---- additive constructors (the edge-list form cannot express configs 2/3/5) -------------
    @classmethod
    def from_arrays(cls, a, b, j, seed_gen=None, *, device=None):
        """Edge list as three arrays instead of a list of ((a, b), j) tuples."""
        self = cls.__new__(cls)
        self._a = np.ascontiguousarray(a, dtype=np.uint64)
        self._b = np.ascontiguousarray(b, dtype=np.uint64)
        self._j = np.ascontiguousarray(j, dtype=np.float64)
        if len(self._a) == 0:
            raise ValueError("Must supply some edges for graph")
        self._init_common(int(max(self._a.max(), self._b.max())) + 1, seed_gen, None, device)
        return self

    @classmethod
    def torus(cls, dims, j=-1.0, pmj=False, j_seed=0, seed_gen=None, *, device=None):
        """Periodic square / cubic lattice, site index x + Lx*(y + Ly*z); pmj=True draws every
        bond as +-|j| (one disorder sample shared by all experiments, as lattice.rs:199 shares
        `&self.edges`).  set_global_bias(h) puts it in the uniform field h (bit-sliced field kernel);
        individual biases are not supported on a torus."""
        self = cls.__new__(cls)
        dims = tuple(int(d) for d in dims)
        n = 1
        for d in dims:
            n *= d
        self._a = self._b = self._j = None
        self._init_common(n, seed_gen, None, device)
        self._torus = (dims, float(j), bool(pmj), int(j_seed))
        return self

    # ---- configuration surface, lattice.rs:76-161 ---------------------------------------------
    def set_seed_gen(self, seed_gen=None):
        self._seed_gen = None if seed_gen is None else int(seed_gen) & _U64

    def make_seeds(self, num_experiments):
        """lattice.rs:83-91: master SmallRng(seed_gen | entropy) -> one u64 per experiment."""
        seed = self._seed_gen if self._seed_gen is not None else secrets.randbits(64)
        return [int(s) for s in nat.make_seeds(seed, num_experiments)]

    def set_enable_rvb_update(self, enable_updates):
        self._enable_rvb_updates = bool(enable_updates)

    def set_enable_heatbath_update(self, enable_heatbath):
        self._enable_heatbath = bool(enable_heatbath)

    def set_individual_bias(self, var, bias):
        if not 0 <= var < self.nvars:
            raise ValueError(f"Index out of bounds: variable {var} out of {self.nvars}")
        if self._bias_individual is None:
            self._bias_individual = np.full(self.nvars, self._bias_global, dtype=np.float64)
        self._bias_individual[var] = bias
        self._graph = None

    def set_global_bias(self, bias):
        self._bias_global = float(bias)
        self._bias_individual = None
        self._graph = None

    def set_transverse_field(self, transverse):
        if transverse > 0.0:
            self._transverse = float(transverse)
        elif transverse == 0.0:
            self._transverse = None
        else:
            raise ValueError("Transverse field must be positive")

    def set_initial_state(self, initial_state):
        initial_state = np.asarray(initial_state, dtype=np.bool_).ravel()
        if len(initial_state) == self.nvars:
            self._initial_state = initial_state.copy()
        elif len(initial_state) == 0:
            self._initial_state = None
        else:
            raise ValueError("Initial state must be of the same size as biases, or 0.")

    def clone(self):
        import copy

        other = copy.copy(self)
        if self._bias_individual is not None:
            other._bias_individual = self._bias_individual.copy()
        return other

    # ---- plumbing --------------------------------------------------------------------------
    def _biases(self):
        if self._bias_individual is not None:
            return self._bias_individual
        if self._bias_global != 0.0:
            return np.full(self.nvars, self._bias_global, dtype=np.float64)
        return None

    def graph(self):
        """Compiled device graph (cached until the biases change)."""
        if self._graph is None:
            ctx = nat.Context.get(self._device)
            if self._torus is not None:
                if self._bias_individual is not None:
                    raise NotImplementedError("individual biases (set_individual_bias) on Lattice.torus lattices "
                                              "are not supported; set_global_bias applies a uniform field")
                dims, j, pmj, j_seed = self._torus
                # a global bias is a uniform field (bit-sliced field kernel); none keeps the plain torus
                field = self._bias_global if self._bias_global != 0.0 else None
                self._graph = nat.Graph.torus(ctx, dims, j, pmj, j_seed, field=field)
            else:
                self._graph = nat.Graph.from_edges(ctx, self.nvars, self._a, self._b, self._j,
                                                   self._biases())
        return self._graph

    def _check_classical(self, edge_move_importance_sampling, only_basic_moves=True):
        """-> flags of the run: which moves a timestep performs (lattice.rs:181, 200, 205)."""
        if self._transverse is not None:
            raise ValueError("Cannot run classic monte carlo with transverse field")
        if only_basic_moves:
            return nat.FLAG_ONLY_BASIC_MOVES      # importance sampling has no move to act on
        if self.non_basic_moves:
            return nat.FLAG_NON_BASIC_MOVES | (nat.FLAG_EDGE_IMPORTANCE if edge_move_importance_sampling else 0)
        warn_non_basic_moves(only_basic_moves)
        return nat.FLAG_EDGE_IMPORTANCE if edge_move_importance_sampling else 0   # -> NotImplementedError (D2)

    def _run_seed(self):
        return self._seed_gen if self._seed_gen is not None else secrets.randbits(64)

    def _args(self, flags, **kw):
        init = None
        if self._initial_state is not None:
            init = np.ascontiguousarray(self._initial_state, dtype=np.uint8)
        return nat.run_args(flags=flags, seed=self._run_seed(), initial_state=init, **kw)

    def _call(self, fn, args, energies, states):
        g = self.graph()
        if self.msc_planes or self.philox_rounds:
            raise NotImplementedError("msc_planes/philox_rounds are set per Sim; use pyisingmontecarlo_b200.Sim")
        if self.distributed:
            return self._call_sharded(fn, args, energies, states, g)
        nat.check(fn(g.ctx.handle, g.handle, args, nat.ptr(energies), nat.ptr(states)), g.ctx.handle)
        return energies, states

    def _call_sharded(self, fn, args, energies, states, g):
        """This rank runs experiments [32 w_lo, min(E, 32 w_hi)); replica_offset keeps every
        experiment on the random stream it has in the unsharded run."""
        from .tempering import _Collective, shard_range

        if self._seed_gen is None:
            raise ValueError("a seed_gen is required when experiments are sharded across ranks")
        coll = _Collective(self.process_group)
        E = int(args.num_experiments)
        words = (E + 31) // 32
        blocks = [shard_range(words, r, coll.world) for r in range(coll.world)]
        counts = [max(0, min(E, 32 * hi) - 32 * lo) for lo, hi in blocks]
        lo = 32 * blocks[coll.rank][0]
        n = counts[coll.rank]
        loc_e = np.zeros((n,) + energies.shape[1:], dtype=np.float64)
        loc_s = nat.PinnedPool.empty((n,) + states.shape[1:], np.bool_)
        if n:
            args.num_experiments = n
            args.replica_offset = lo
            nat.check(fn(g.ctx.handle, g.handle, args, nat.ptr(loc_e), nat.ptr(loc_s)), g.ctx.handle)
        self.local_range = (lo, lo + n)
        if not self.gather_results or not coll.active:
            return loc_e, loc_s
        return coll.allgather_concat(loc_e, counts), coll.allgather_concat(loc_s, counts)

    # ---- classical runs, lattice.rs:163-470 -------------------------------------------------
    def run_monte_carlo(self, beta, timesteps, num_experiments, only_basic_moves=None,
                        edge_move_importance_sampling=None):
        """lattice.rs:171-221 -> (energies float64[E], states bool[E, nvars])

        only_basic_moves=None/False: single-spin sweeps only (deviation D1, warned once) unless
        `non_basic_moves` is set, which adds an edge-move pass and a worm move to every timestep."""
        flags = self._check_classical(edge_move_importance_sampling, only_basic_moves)
        energies = np.zeros(num_experiments, dtype=np.float64)
        states = nat.PinnedPool.empty((num_experiments, self.nvars), np.bool_)
        args = self._args(flags, beta=float(beta), timesteps=int(timesteps),
                          num_experiments=int(num_experiments))
        return self._call(nat.lib().ising_run_monte_carlo, args, energies, states)

    def run_monte_carlo_sampling(self, beta, timesteps, num_experiments, only_basic_moves=None,
                                 thermalization_time=None, sampling_freq=None,
                                 edge_move_importance_sampling=None):
        """lattice.rs:231-299 -> (energies float64[E, n_s], states bool[E, n_s, nvars])"""
        flags = self._check_classical(edge_move_importance_sampling, only_basic_moves)
        thermalization_time = 0 if thermalization_time is None else int(thermalization_time)
        sampling_freq = 1 if sampling_freq is None else int(sampling_freq)
        if sampling_freq == 0:
            raise ZeroDivisionError("sampling_freq must be non-zero (the reference panics)")
        n_samples = int(timesteps) // sampling_freq
        energies = np.zeros((num_experiments, n_samples), dtype=np.float64)
        states = nat.PinnedPool.empty((num_experiments, n_samples, self.nvars), np.bool_)
        args = self._args(flags, beta=float(beta), timesteps=int(timesteps),
                          num_experiments=int(num_experiments), thermalization=thermalization_time,
                          sampling_freq=sampling_freq)
        return self._call(nat.lib().ising_run_monte_carlo_sampling, args, energies, states)

    def run_monte_carlo_observables(self, beta, timesteps, num_experiments, thermalization_time=None,
                                    sampling_freq=None, overlaps=True):
        """Additive (SURVEY 8(f)2): the loop of lattice.rs:231-299 with the per-sample state copy
        replaced by on-device reductions.  Same trajectories as run_monte_carlo_sampling for the
        same seed_gen -> (energies[E, n_s], M[E, n_s] = sum_i s_i, Q[E // 2, n_s] = overlap of
        the experiment pairs (2p, 2p+1)); Binder ratios etc. follow on the host from M and Q."""
        self._check_classical(None)
        if self.distributed:
            raise NotImplementedError("run_monte_carlo_observables on a sharded Lattice")
        thermalization_time = 0 if thermalization_time is None else int(thermalization_time)
        sampling_freq = 1 if sampling_freq is None else int(sampling_freq)
        if sampling_freq == 0:
            raise ZeroDivisionError("sampling_freq must be non-zero (the reference panics)")
        sim = nat.Sim(self.graph(), int(num_experiments), self._run_seed(),
                      planes=self.msc_planes or 0, rounds=self.philox_rounds or 0)
        try:
            if self._initial_state is not None:
                sim.set_state(self._initial_state)
            return sim.run_observables(beta, thermalization_time, sampling_freq,
                                       int(timesteps) // sampling_freq, overlaps)
        finally:
            sim.close()

    def _annealing(self, betas, timesteps, num_experiments, only_basic_moves,
                   edge_move_importance_sampling, per_step):
        flags = self._check_classical(edge_move_importance_sampling, only_basic_moves)
        if per_step:
            flags |= nat.FLAG_PER_STEP_ENERGIES
        if self.linear_annealing:
            flags |= nat.FLAG_LINEAR_SCHEDULE
        betas = list(betas)
        st = np.ascontiguousarray([int(t) for t, _ in betas], dtype=np.uint64)
        sb = np.ascontiguousarray([float(v) for _, v in betas], dtype=np.float64)
        shape = (num_experiments, int(timesteps)) if per_step else (num_experiments,)
        energies = nat.PinnedPool.empty(shape, np.float64)
        states = nat.PinnedPool.empty((num_experiments, self.nvars), np.bool_)
        args = self._args(flags, sched_t=st if len(st) else None, sched_beta=sb if len(sb) else None,
                          sched_len=len(st), timesteps=int(timesteps),
                          num_experiments=int(num_experiments))
        return self._call(nat.lib().ising_run_monte_carlo_annealing, args, energies, states)

    def run_monte_carlo_annealing(self, betas, timesteps, num_experiments, only_basic_moves=None,
                                  edge_move_importance_sampling=None):
        """lattice.rs:309-385 -> (energies float64[E], states bool[E, nvars])"""
        return self._annealing(betas, timesteps, num_experiments, only_basic_moves,
                               edge_move_importance_sampling, False)

    def run_monte_carlo_annealing_and_get_energies(self, betas, timesteps, num_experiments,
                                                   only_basic_moves=None,
                                                   edge_move_importance_sampling=None):
        """lattice.rs:395-470 -> (energies float64[E, timesteps], states bool[E, nvars])"""
        return self._annealing(betas, timesteps, num_experiments, only_basic_moves,
                               edge_move_importance_sampling, True)

    # ---- replay mode (north-star correctness check 1) -----------------------------------------
    def replay(self, beta, sites, uniforms, init_states):
        """Re-runs the reference's own (site, uniform) sequence on the GPU, bit-exactly.

        sites uint32[E, A], uniforms float64[E, A] (ignored where dE <= 0), init bool[E, nvars]."""
        sites = np.ascontiguousarray(sites, dtype=np.uint32)
        uniforms = np.ascontiguousarray(uniforms, dtype=np.float64)
        init = np.ascontiguousarray(init_states, dtype=np.uint8)
        E, A = sites.shape
        if uniforms.shape != (E, A) or init.shape != (E, self.nvars):
            raise ValueError("replay trace shapes disagree")
        g = self.graph()
        energies = np.zeros(E, dtype=np.float64)
        states = np.zeros((E, self.nvars), dtype=np.bool_)
        nat.check(nat.lib().ising_replay(g.ctx.handle, g.handle, float(beta), E, A, nat.ptr(sites),
                                         nat.ptr(uniforms), nat.ptr(init), nat.ptr(energies),
                                         nat.ptr(states)), g.ctx.handle)
        return energies, states

    # ---- quantum path: out of scope, stays on the reference (lattice.rs:472-1069) -------------
    def __getattr__(self, name):
        if name.startswith("run_quantum_monte_carlo") or name in (
                "average_on_and_off_diagonal_and_consts", "get_offset"):
            raise NotImplementedError(
                f"{name}: the SSE quantum Monte Carlo path is out of scope of the B200 engine and "
                "remains on the reference py_monte_carlo build")
        raise AttributeError(name)
