"""ctypes binding of libising_b200.so (include/ising_b200.h).

This is the only door to the compute path: if the shared library (built by
``pyisingmontecarlo_b200._build.build_native`` / ``__graft_entry__.build``) is missing, or no
sm_100 device is visible, the calls fail loudly -- there is no CPU or eager fallback.
"""
import ctypes as C
import os
import threading

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
# ISING_B200_LIB lets kernel experiments point at an alternative build of the same library
LIB_PATH = os.environ.get("ISING_B200_LIB") or os.path.join(HERE, "libising_b200.so")

ISING_OK, ISING_E_INVALID, ISING_E_CUDA, ISING_E_UNSUPPORTED, ISING_E_AMBIGUOUS, ISING_E_NOMEM = range(6)

FLAG_ONLY_BASIC_MOVES = 1 << 0
FLAG_PER_STEP_ENERGIES = 1 << 1
FLAG_LINEAR_SCHEDULE = 1 << 2
FLAG_EDGE_IMPORTANCE = 1 << 3
FLAG_NON_BASIC_MOVES = 1 << 4

KIND_GENERAL, KIND_STENCIL2D, KIND_STENCIL3D = 0, 2, 3


class NativeLibraryMissing(ImportError):
    pass


class AmbiguousReplay(RuntimeError):
    pass


class GraphInfo(C.Structure):
    _fields_ = [
        ("nvars", C.c_uint64),
        ("nedges", C.c_uint64),
        ("kind", C.c_int32),
        ("ncolors", C.c_int32),
        ("max_degree", C.c_int32),
        ("integer_classes", C.c_int32),
        ("dims", C.c_uint64 * 3),
        ("jabs", C.c_double),
    ]


class SimStats(C.Structure):
    _fields_ = [
        ("kernel_launches", C.c_uint64),
        ("sweeps", C.c_uint64),
        ("flip_attempts", C.c_uint64),
        ("sweep_device_ms", C.c_double),
        ("sweep_kernel_ms", C.c_double),
        ("sweep_kernel_launches", C.c_uint64),
        ("edge_attempts", C.c_uint64),
        ("worm_attempts", C.c_uint64),
    ]


class Moves(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32),
        ("spin_sweeps", C.c_uint32),
        ("edge_passes", C.c_uint32),
        ("worms", C.c_uint32),
        ("worm_len", C.c_uint32),
        ("edge_importance", C.c_uint32),
    ]


class RunArgs(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32),
        ("flags", C.c_uint32),
        ("beta", C.c_double),
        ("sched_t", C.c_void_p),
        ("sched_beta", C.c_void_p),
        ("sched_len", C.c_uint64),
        ("timesteps", C.c_uint64),
        ("num_experiments", C.c_uint64),
        ("thermalization", C.c_uint64),
        ("sampling_freq", C.c_uint64),
        ("seed", C.c_uint64),
        ("replica_offset", C.c_uint64),
        ("initial_state", C.c_void_p),
    ]


_P = C.c_void_p
_SIGNATURES = {
    # name: (restype, argtypes)
    "ising_abi_version": (C.c_int, []),
    "ising_ctx_create": (C.c_int, [C.c_int, C.POINTER(_P)]),
    "ising_ctx_create_on_stream": (C.c_int, [C.c_int, _P, C.POINTER(_P)]),
    "ising_ctx_destroy": (None, [_P]),
    "ising_last_error": (C.c_char_p, [_P]),
    "ising_host_alloc": (C.c_int, [C.c_size_t, C.POINTER(_P)]),
    "ising_host_free": (None, [_P]),
    "ising_graph_from_edges": (C.c_int, [_P, C.c_uint64, C.c_uint64, _P, _P, _P, _P, C.POINTER(_P)]),
    "ising_graph_torus": (C.c_int, [_P, C.c_int, _P, C.c_double, C.c_int, C.c_uint64, C.POINTER(_P)]),
    "ising_graph_torus_field": (C.c_int, [_P, C.c_int, _P, C.c_double, C.c_int, C.c_uint64, C.c_double, C.POINTER(_P)]),
    "ising_graph_destroy": (None, [_P]),
    "ising_graph_get_info": (C.c_int, [_P, C.POINTER(GraphInfo)]),
    "ising_graph_get_colors": (C.c_int, [_P, _P]),
    "ising_graph_get_edges": (C.c_int, [_P, _P, _P, _P]),
    "ising_graph_get_edge_classes": (C.c_int, [_P, _P]),
    "ising_strong_edge_colouring": (C.c_int, [C.c_uint64, C.c_uint64, _P, _P, _P, C.POINTER(C.c_uint32)]),
    "ising_make_seeds": (C.c_int, [C.c_uint64, C.c_uint64, _P]),
    "ising_sim_create": (C.c_int, [_P, _P, C.c_uint64, C.c_uint64, C.c_uint64, C.POINTER(_P)]),
    "ising_sim_create_ex": (C.c_int, [_P, _P, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint32, C.POINTER(_P)]),
    "ising_sim_set_betas": (C.c_int, [_P, _P]),
    "ising_sim_destroy": (None, [_P]),
    "ising_sim_configure": (C.c_int, [_P, C.c_int, C.c_int]),
    "ising_sim_set_moves": (C.c_int, [_P, C.POINTER(Moves)]),
    "ising_sim_randomize": (C.c_int, [_P]),
    "ising_sim_set_state": (C.c_int, [_P, _P]),
    "ising_sim_set_states": (C.c_int, [_P, _P]),
    "ising_sim_sweeps": (C.c_int, [_P, _P, C.c_uint64, _P]),
    "ising_sim_run_sampling": (C.c_int, [_P, C.c_double, C.c_uint64, C.c_uint64, C.c_uint64, _P, _P]),
    "ising_sim_run_sampling_packed": (C.c_int, [_P, C.c_double, C.c_uint64, C.c_uint64, C.c_uint64, _P, _P]),
    "ising_sim_run_observables": (C.c_int, [_P, C.c_double, C.c_uint64, C.c_uint64, C.c_uint64, _P, _P, _P]),
    "ising_sim_get_energies": (C.c_int, [_P, _P]),
    "ising_sim_get_states": (C.c_int, [_P, _P]),
    "ising_sim_get_packed": (C.c_int, [_P, _P]),
    "ising_sim_get_magnetization": (C.c_int, [_P, _P]),
    "ising_sim_step_acceptance": (C.c_int, [_P, C.c_double, _P]),
    "ising_sim_set_packed": (C.c_int, [_P, _P]),
    "ising_sim_get_counter": (C.c_int, [_P, C.POINTER(C.c_uint64)]),
    "ising_sim_set_counter": (C.c_int, [_P, C.c_uint64]),
    "ising_pt_get_sim": (C.c_int, [_P, C.POINTER(_P)]),
    "ising_pt_get_counters": (C.c_int, [_P, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "ising_pt_restore": (C.c_int, [_P, _P, C.c_uint64, C.c_uint64]),
    "ising_sim_get_stats": (C.c_int, [_P, C.POINTER(SimStats)]),
    "ising_sim_reset_stats": (C.c_int, [_P]),
    "ising_run_monte_carlo": (C.c_int, [_P, _P, C.POINTER(RunArgs), _P, _P]),
    "ising_run_monte_carlo_sampling": (C.c_int, [_P, _P, C.POINTER(RunArgs), _P, _P]),
    "ising_run_monte_carlo_annealing": (C.c_int, [_P, _P, C.POINTER(RunArgs), _P, _P]),
    "ising_schedule_betas": (C.c_int, [_P, _P, C.c_uint64, C.c_uint64, C.c_int, _P]),
    "ising_pt_create": (C.c_int, [_P, _P, _P, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.POINTER(_P)]),
    "ising_pt_destroy": (None, [_P]),
    "ising_pt_configure": (C.c_int, [_P, C.c_int, C.c_int]),
    "ising_pt_sweeps": (C.c_int, [_P, C.c_uint64, _P]),
    "ising_pt_swap_step": (C.c_int, [_P, _P]),
    "ising_pt_decide_swaps": (C.c_int, [_P, C.c_uint64, _P, C.c_uint64, C.c_uint64, _P, _P, C.POINTER(C.c_uint64)]),
    "ising_pt_get_slots": (C.c_int, [_P, _P]),
    "ising_pt_get_local_states": (C.c_int, [_P, _P]),
    "ising_pt_total_swaps": (C.c_int, [_P, C.POINTER(C.c_uint64)]),
    "ising_pt_timesteps_sample": (C.c_int, [_P, C.c_uint64, C.c_uint64, C.c_uint64, _P, _P]),
    "ising_strip_get_row_range": (C.c_int, [_P, C.c_uint64, C.c_uint64, _P]),
    "ising_strip_sweeps": (C.c_int, [_P, _P, _P, C.c_uint64, C.c_uint32]),
    "ising_strip_set_field": (C.c_int, [_P, C.c_double]),
    "ising_strip_sweeps_field": (C.c_int, [_P, _P, _P, _P, C.c_uint64, C.c_uint32]),
    "ising_strip_global_sums": (C.c_int, [_P, _P, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "ising_pt_set_comm": (C.c_int, [_P, _P]),
    "ising_pt_get_pair_stats": (C.c_int, [_P, _P, _P]),
    "ising_comm_unique_id": (C.c_int, [_P, C.c_uint64]),
    "ising_comm_create": (C.c_int, [_P, _P, C.c_int, C.c_int, C.POINTER(_P)]),
    "ising_comm_destroy": (None, [_P]),
    "ising_comm_info": (C.c_int, [_P, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "ising_strip_create": (C.c_int, [_P, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_double, C.c_uint64, C.POINTER(_P)]),
    "ising_strip_create_ex": (C.c_int, [_P, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_double, C.c_uint64, C.c_uint32, C.POINTER(_P)]),
    "ising_strip_phase_ext": (C.c_int, [_P, C.c_int, C.c_double, C.c_uint32, C.c_int, C.c_int]),
    "ising_strip_halo_deep": (C.c_int, [_P, C.c_int, C.c_uint32, _P, C.c_int]),
    "ising_strip_wrap_deep": (C.c_int, [_P, C.c_uint32]),
    "ising_strip_destroy": (None, [_P]),
    "ising_strip_configure": (C.c_int, [_P, C.c_int, C.c_int]),
    "ising_strip_set_all": (C.c_int, [_P, C.c_int]),
    "ising_strip_phase": (C.c_int, [_P, C.c_int, C.c_double]),
    "ising_strip_phase_rows": (C.c_int, [_P, C.c_int, C.c_double, C.c_uint64, C.c_uint64, C.c_int, C.c_int]),
    "ising_strip_halo_async": (C.c_int, [_P, C.c_int, C.c_int, _P]),
    "ising_strip_get_boundary": (C.c_int, [_P, C.c_int, C.c_int, _P]),
    "ising_strip_set_ghost": (C.c_int, [_P, C.c_int, C.c_int, _P]),
    "ising_strip_wrap_local": (C.c_int, [_P, C.c_int]),
    "ising_strip_observables": (C.c_int, [_P, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "ising_strip_get_rows": (C.c_int, [_P, _P]),
    "ising_strip_get_stats": (C.c_int, [_P, C.POINTER(C.c_uint64), C.POINTER(C.c_double), C.c_int]),
    "ising_replay": (C.c_int, [_P, _P, C.c_double, C.c_uint64, C.c_uint64, _P, _P, _P, _P, _P]),
}

_lib = None
_lock = threading.Lock()


def exported_symbols():
    """Every entry point include/ising_b200.h declares."""
    return sorted(_SIGNATURES)


def lib():
    """Loads libising_b200.so once; raises NativeLibraryMissing if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise NativeLibraryMissing(
                    f"{LIB_PATH} is missing: run `python __graft_entry__.py build` (nvcc, sm_100a). "
                    "pyisingmontecarlo_b200 has no CPU fallback."
                )
            handle = C.CDLL(LIB_PATH)
            for name, (res, args) in _SIGNATURES.items():
                fn = getattr(handle, name)
                fn.restype = res
                fn.argtypes = args
            _lib = handle
    return _lib


def _err(ctx):
    msg = lib().ising_last_error(ctx)
    return msg.decode("utf-8", "replace") if msg else "unknown error"


def check(rc, ctx=None):
    if rc == ISING_OK:
        return
    msg = _err(ctx)
    if rc == ISING_E_INVALID:
        raise ValueError(msg)
    if rc == ISING_E_UNSUPPORTED:
        raise NotImplementedError(msg)
    if rc == ISING_E_AMBIGUOUS:
        raise AmbiguousReplay(msg)
    if rc == ISING_E_NOMEM:
        raise MemoryError(msg)
    raise RuntimeError(msg)


def ptr(arr):
    return None if arr is None else arr.ctypes.data_as(C.c_void_p)


class PinnedPool:
    """Output arrays in page-locked host memory, recycled when the numpy array is collected.

    The reference allocates its outputs in the host layer and hands them to numpy without a
    copy (lattice.rs:183-184, 213-214); doing the same here with cudaHostAlloc memory makes the
    device->host copies of bool[E, N] run at PCIe speed.  Blocks go back to a free list keyed
    by size when the last view of the array dies, so steady-state calls allocate nothing."""

    GRAIN = 1 << 21
    MAX_CACHED = 8 << 30
    _free = {}
    _cached = 0
    _lk = threading.Lock()

    @classmethod
    def _release(cls, addr, size):
        with cls._lk:
            if cls._cached + size <= cls.MAX_CACHED:
                cls._free.setdefault(size, []).append(addr)
                cls._cached += size
                return
        lib().ising_host_free(addr)

    @classmethod
    def empty(cls, shape, dtype):
        import weakref

        dtype = np.dtype(dtype)
        nbytes = int(np.prod(shape, dtype=np.int64)) * dtype.itemsize
        if nbytes < (1 << 20):
            return np.empty(shape, dtype=dtype)
        size = (nbytes + cls.GRAIN - 1) // cls.GRAIN * cls.GRAIN
        addr = None
        with cls._lk:
            lst = cls._free.get(size)
            if lst:
                addr = lst.pop()
                cls._cached -= size
        if addr is None:
            p = C.c_void_p()
            check(lib().ising_host_alloc(size, C.byref(p)))
            addr = p.value
        buf = (C.c_uint8 * size).from_address(addr)
        weakref.finalize(buf, cls._release, addr, size)
        return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape, dtype=np.int64))).reshape(shape)


class Context:
    """One CUDA device + stream (ising_ctx)."""

    _cache = {}

    def __init__(self, device=0, stream=None):
        """stream: a cudaStream_t as integer (e.g. torch.cuda.current_stream().cuda_stream) to run
        on the caller's stream instead of a private one."""
        self.device = int(device)
        h = C.c_void_p()
        if stream is None:
            check(lib().ising_ctx_create(self.device, C.byref(h)), None)
        else:
            check(lib().ising_ctx_create_on_stream(self.device, C.c_void_p(int(stream)), C.byref(h)), None)
        self.handle = h

    @classmethod
    def get(cls, device=None):
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", "0")) if "LOCAL_RANK" in os.environ else 0
        key = (os.getpid(), int(device))
        if key not in cls._cache:
            cls._cache[key] = Context(device)
        return cls._cache[key]

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                lib().ising_ctx_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class Graph:
    """Compiled coupling graph (ising_graph): CSR + colouring, or a checkerboard stencil."""

    def __init__(self, ctx, handle):
        self.ctx = ctx
        self.handle = handle
        info = GraphInfo()
        check(lib().ising_graph_get_info(handle, C.byref(info)), ctx.handle)
        self.nvars = int(info.nvars)
        self.nedges = int(info.nedges)
        self.kind = int(info.kind)
        self.ncolors = int(info.ncolors)
        self.max_degree = int(info.max_degree)
        self.integer_classes = bool(info.integer_classes)
        self.dims = tuple(int(d) for d in info.dims)
        self.jabs = float(info.jabs)
        self.field = None   # uniform field of a torus built with Graph.torus(field=...)

    @classmethod
    def from_edges(cls, ctx, nvars, a, b, j, biases=None):
        a = np.ascontiguousarray(a, dtype=np.uint64)
        b = np.ascontiguousarray(b, dtype=np.uint64)
        j = np.ascontiguousarray(j, dtype=np.float64)
        bias = None if biases is None else np.ascontiguousarray(biases, dtype=np.float64)
        h = C.c_void_p()
        check(lib().ising_graph_from_edges(ctx.handle, int(nvars), len(a), ptr(a), ptr(b), ptr(j),
                                           ptr(bias), C.byref(h)), ctx.handle)
        return cls(ctx, h)

    @classmethod
    def torus(cls, ctx, dims, j0=-1.0, pmj=False, j_seed=0, field=None):
        """field=None: no field (ising_graph_torus); a number h, 0.0 included: the torus in the uniform
        field h, E = sum J s s' - h sum s, on the bit-sliced field kernel (ising_graph_torus_field)."""
        L = np.ascontiguousarray(list(dims) + [1] * (3 - len(dims)), dtype=np.uint64)
        h = C.c_void_p()
        if field is None:
            check(lib().ising_graph_torus(ctx.handle, len(dims), ptr(L), float(j0), int(bool(pmj)),
                                          int(j_seed), C.byref(h)), ctx.handle)
        else:
            check(lib().ising_graph_torus_field(ctx.handle, len(dims), ptr(L), float(j0), int(bool(pmj)),
                                                int(j_seed), float(field), C.byref(h)), ctx.handle)
        g = cls(ctx, h)
        g.field = None if field is None else float(field)
        return g

    def colors(self):
        out = np.empty(self.nvars, dtype=np.uint32)
        check(lib().ising_graph_get_colors(self.handle, ptr(out)), self.ctx.handle)
        return out

    def edge_classes(self):
        """class of every bond in the strong edge colouring of the edge moves (uint32[nedges])"""
        out = np.empty(self.nedges, dtype=np.uint32)
        check(lib().ising_graph_get_edge_classes(self.handle, ptr(out)), self.ctx.handle)
        return out

    def edges(self):
        a = np.empty(self.nedges, dtype=np.uint64)
        b = np.empty(self.nedges, dtype=np.uint64)
        j = np.empty(self.nedges, dtype=np.float64)
        check(lib().ising_graph_get_edges(self.handle, ptr(a), ptr(b), ptr(j)), self.ctx.handle)
        return a, b, j

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                lib().ising_graph_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class Sim:
    """Device-resident replica-bit-packed experiments (ising_sim)."""

    def __init__(self, graph, num_experiments, seed, replica_offset=0, planes=0, rounds=0,
                 general_layout=False):
        self.graph = graph
        self.ctx = graph.ctx
        self.E = int(num_experiments)
        h = C.c_void_p()
        check(lib().ising_sim_create_ex(self.ctx.handle, graph.handle, self.E, int(seed) & (2**64 - 1),
                                        int(replica_offset), 1 if general_layout else 0,
                                        C.byref(h)), self.ctx.handle)
        self.handle = h
        if planes or rounds:
            check(lib().ising_sim_configure(h, int(planes), int(rounds)), self.ctx.handle)

    def randomize(self):
        check(lib().ising_sim_randomize(self.handle), self.ctx.handle)

    def set_moves(self, spin_sweeps=1, edge_passes=0, worms=0, worm_len=4, edge_importance=False):
        """What a timestep consists of (ising_sim_set_moves); set_moves() alone restores the
        default of one colour-class sweep."""
        m = Moves(C.sizeof(Moves), int(spin_sweeps), int(edge_passes), int(worms), int(worm_len),
                  1 if edge_importance else 0)
        check(lib().ising_sim_set_moves(self.handle, C.byref(m)), self.ctx.handle)

    def set_state(self, state):
        s = np.ascontiguousarray(state, dtype=np.uint8)
        if s.shape != (self.graph.nvars,):
            raise ValueError("state must have nvars entries")
        check(lib().ising_sim_set_state(self.handle, ptr(s)), self.ctx.handle)

    def set_states(self, states):
        s = np.ascontiguousarray(states, dtype=np.uint8)
        if s.shape != (self.E, self.graph.nvars):
            raise ValueError("states must be [num_experiments, nvars]")
        check(lib().ising_sim_set_states(self.handle, ptr(s)), self.ctx.handle)

    def sweeps(self, betas, per_sweep_energies=False):
        """betas: one inverse temperature per sweep, or an int = number of sweeps at the
        per-experiment betas installed with set_betas()."""
        if isinstance(betas, (int, np.integer)):
            n, b = int(betas), None
        else:
            b = np.ascontiguousarray(betas, dtype=np.float64)
            n = len(b)
        out = np.empty((self.E, n), dtype=np.float64) if per_sweep_energies else None
        check(lib().ising_sim_sweeps(self.handle, ptr(b), n, ptr(out)), self.ctx.handle)
        return out

    def set_betas(self, betas):
        b = np.ascontiguousarray(betas, dtype=np.float64)
        if b.shape != (self.E,):
            raise ValueError("betas must have one entry per experiment")
        check(lib().ising_sim_set_betas(self.handle, ptr(b)), self.ctx.handle)

    def run_sampling(self, beta, thermalization, sampling_freq, n_samples, packed=False):
        """(energies[E, n_s], states bool[E, n_s, nvars]); packed=True returns the samples as
        uint32[n_s, nvars, ceil(E/32)] instead (bit e%32 of word e/32 = experiment e)."""
        energies = np.empty((self.E, n_samples), dtype=np.float64)
        if packed:
            words = PinnedPool.empty((n_samples, self.graph.nvars, (self.E + 31) // 32), np.uint32)
            check(lib().ising_sim_run_sampling_packed(self.handle, float(beta), int(thermalization),
                                                      int(sampling_freq), int(n_samples), ptr(energies),
                                                      ptr(words)), self.ctx.handle)
            return energies, words
        states = PinnedPool.empty((self.E, n_samples, self.graph.nvars), np.bool_)
        check(lib().ising_sim_run_sampling(self.handle, float(beta), int(thermalization),
                                           int(sampling_freq), int(n_samples), ptr(energies),
                                           ptr(states)), self.ctx.handle)
        return energies, states

    def run_observables(self, beta, thermalization, sampling_freq, n_samples, overlaps=True):
        """(energies[E, n_s], magnetisations[E, n_s], overlaps[E // 2, n_s] or None), reduced on
        the device: no state read-back."""
        energies = np.zeros((self.E, n_samples), dtype=np.float64)
        mags = np.zeros((self.E, n_samples), dtype=np.float64)
        q = np.zeros((self.E // 2, n_samples), dtype=np.float64) if overlaps else None
        check(lib().ising_sim_run_observables(self.handle, float(beta), int(thermalization),
                                              int(sampling_freq), int(n_samples), ptr(energies),
                                              ptr(mags), ptr(q)), self.ctx.handle)
        return energies, mags, q

    def energies(self):
        out = np.empty(self.E, dtype=np.float64)
        check(lib().ising_sim_get_energies(self.handle, ptr(out)), self.ctx.handle)
        return out

    def step_acceptance(self, beta):
        """one timestep at beta -> spins changed per experiment (uint64[E]): the accepted flips"""
        out = np.empty(self.E, dtype=np.uint64)
        check(lib().ising_sim_step_acceptance(self.handle, float(beta), ptr(out)), self.ctx.handle)
        return out

    def magnetization(self):
        out = np.empty(self.E, dtype=np.float64)
        check(lib().ising_sim_get_magnetization(self.handle, ptr(out)), self.ctx.handle)
        return out

    def states(self, out=None):
        if out is None:
            out = np.empty((self.E, self.graph.nvars), dtype=np.bool_)
        check(lib().ising_sim_get_states(self.handle, ptr(out)), self.ctx.handle)
        return out

    def packed(self):
        out = np.empty((self.graph.nvars, (self.E + 31) // 32), dtype=np.uint32)
        check(lib().ising_sim_get_packed(self.handle, ptr(out)), self.ctx.handle)
        return out

    def set_packed(self, words):
        w = np.ascontiguousarray(words, dtype=np.uint32)
        if w.shape != (self.graph.nvars, (self.E + 31) // 32):
            raise ValueError("packed state must be uint32[nvars, ceil(E/32)]")
        check(lib().ising_sim_set_packed(self.handle, ptr(w)), self.ctx.handle)

    @property
    def counter(self):
        n = C.c_uint64(0)
        check(lib().ising_sim_get_counter(self.handle, C.byref(n)), self.ctx.handle)
        return int(n.value)

    @counter.setter
    def counter(self, value):
        check(lib().ising_sim_set_counter(self.handle, int(value)), self.ctx.handle)

    def stats(self):
        st = SimStats()
        check(lib().ising_sim_get_stats(self.handle, C.byref(st)), self.ctx.handle)
        return {k: getattr(st, k) for k, _ in SimStats._fields_}

    def reset_stats(self):
        check(lib().ising_sim_reset_stats(self.handle), self.ctx.handle)

    def close(self):
        if getattr(self, "handle", None):
            lib().ising_sim_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


COMM_ID_BYTES = 128


class Comm:
    """NCCL communicator owned by the library (ising_comm), one rank per process / GPU.  The
    collectives of the hot path (tempering energies, strip halos) are issued by the C library on
    the context's stream; the host layer only has to get rank 0's unique id to every rank."""

    def __init__(self, ctx, unique_id, rank, world):
        self.ctx = ctx
        idb = np.frombuffer(bytes(unique_id), dtype=np.uint8).copy()
        if idb.size != COMM_ID_BYTES:
            raise ValueError("unique id must be %d bytes" % COMM_ID_BYTES)
        h = C.c_void_p()
        check(lib().ising_comm_create(ctx.handle, ptr(idb), int(rank), int(world), C.byref(h)), ctx.handle)
        self.handle = h
        self.rank, self.world = int(rank), int(world)

    @staticmethod
    def unique_id():
        out = np.zeros(COMM_ID_BYTES, dtype=np.uint8)
        check(lib().ising_comm_unique_id(ptr(out), COMM_ID_BYTES), None)
        return out.tobytes()

    @classmethod
    def from_torch(cls, ctx, group=None):
        """Bootstraps over an initialised torch.distributed group (any backend): rank 0 creates
        the id, a broadcast carries its 128 bytes.  torch is used for this exchange only."""
        import torch
        import torch.distributed as dist

        rank, world = dist.get_rank(group), dist.get_world_size(group)
        backend = dist.get_backend(group)
        dev = torch.device("cuda", ctx.device) if backend == "nccl" else torch.device("cpu")
        buf = torch.zeros(COMM_ID_BYTES, dtype=torch.uint8, device=dev)
        if rank == 0:
            buf.copy_(torch.frombuffer(bytearray(cls.unique_id()), dtype=torch.uint8))
        dist.broadcast(buf, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
        return cls(ctx, bytes(buf.cpu().numpy().tobytes()), rank, world)

    def close(self):
        if getattr(self, "handle", None):
            lib().ising_comm_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Tempering:
    """Classical parallel tempering on the device (ising_pt): configurations [cfg_lo, cfg_hi)
    of a ladder of `betas` live on this rank."""

    def __init__(self, graph, betas, seed, cfg_lo=0, cfg_hi=None, planes=0, rounds=0):
        self.graph = graph
        self.ctx = graph.ctx
        self.betas = np.ascontiguousarray(betas, dtype=np.float64)
        self.seed = int(seed) & (2**64 - 1)
        self.R = len(self.betas)
        self.lo = int(cfg_lo)
        self.hi = self.R if cfg_hi is None else int(cfg_hi)
        h = C.c_void_p()
        check(lib().ising_pt_create(self.ctx.handle, graph.handle, ptr(self.betas), self.R, self.lo,
                                    self.hi, int(seed) & (2**64 - 1), C.byref(h)), self.ctx.handle)
        self.handle = h
        if planes or rounds:
            check(lib().ising_pt_configure(h, int(planes), int(rounds)), self.ctx.handle)

    def sweeps(self, t, want_energies=True):
        out = np.empty(self.hi - self.lo, dtype=np.float64) if want_energies else None
        check(lib().ising_pt_sweeps(self.handle, int(t), ptr(out)), self.ctx.handle)
        return out

    def swap_step(self, all_energies):
        e = np.ascontiguousarray(all_energies, dtype=np.float64)
        if e.shape != (self.R,):
            raise ValueError("all_energies must have one entry per configuration")
        check(lib().ising_pt_swap_step(self.handle, ptr(e)), self.ctx.handle)

    def slots(self):
        out = np.empty(self.R, dtype=np.uint32)
        check(lib().ising_pt_get_slots(self.handle, ptr(out)), self.ctx.handle)
        return out

    def local_states(self):
        out = np.empty((self.hi - self.lo, self.graph.nvars), dtype=np.bool_)
        check(lib().ising_pt_get_local_states(self.handle, ptr(out)), self.ctx.handle)
        return out

    def total_swaps(self):
        n = C.c_uint64(0)
        check(lib().ising_pt_total_swaps(self.handle, C.byref(n)), self.ctx.handle)
        return int(n.value)

    def sim_stats(self):
        """Launch / sweep counters of the sim behind the ladder (ising_sim_stats)."""
        sim = C.c_void_p()
        check(lib().ising_pt_get_sim(self.handle, C.byref(sim)), self.ctx.handle)
        st = SimStats()
        check(lib().ising_sim_get_stats(sim, C.byref(st)), self.ctx.handle)
        return {k: getattr(st, k) for k, _ in SimStats._fields_}

    def set_comm(self, comm):
        """Shards the ladder over the ranks of `comm` (this object must hold the rank's block):
        timesteps_sample then gathers energies and samples with NCCL inside the library."""
        check(lib().ising_pt_set_comm(self.handle, comm.handle if comm is not None else None), self.ctx.handle)
        self._comm = comm

    def pair_stats(self):
        """(attempts, accepts) uint64[R - 1] of the swaps between neighbouring betas."""
        att = np.zeros(max(self.R - 1, 0), dtype=np.uint64)
        acc = np.zeros(max(self.R - 1, 0), dtype=np.uint64)
        check(lib().ising_pt_get_pair_stats(self.handle, ptr(att), ptr(acc)), self.ctx.handle)
        return att, acc

    def checkpoint(self):
        """Everything needed to continue this ladder bit for bit (see restore)."""
        sim = C.c_void_p()
        check(lib().ising_pt_get_sim(self.handle, C.byref(sim)), self.ctx.handle)
        E = min(((self.hi + 31) // 32 - self.lo // 32) * 32, self.R - (self.lo // 32) * 32)
        words = np.empty((self.graph.nvars, (E + 31) // 32), dtype=np.uint32)
        check(lib().ising_sim_get_packed(sim, ptr(words)), self.ctx.handle)
        cnt, a, b = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        check(lib().ising_sim_get_counter(sim, C.byref(cnt)), self.ctx.handle)
        check(lib().ising_pt_get_counters(self.handle, C.byref(a), C.byref(b)), self.ctx.handle)
        return {"packed": words, "sweeps": int(cnt.value), "slots": self.slots(),
                "swap_step": int(a.value), "total_swaps": int(b.value)}

    def restore(self, ck):
        sim = C.c_void_p()
        check(lib().ising_pt_get_sim(self.handle, C.byref(sim)), self.ctx.handle)
        words = np.ascontiguousarray(ck["packed"], dtype=np.uint32)
        slots = np.ascontiguousarray(ck["slots"], dtype=np.uint32)
        E = min(((self.hi + 31) // 32 - self.lo // 32) * 32, self.R - (self.lo // 32) * 32)
        if words.shape != (self.graph.nvars, (E + 31) // 32):
            raise ValueError(f"checkpoint holds packed spins of shape {words.shape}, this ladder needs "
                             f"{(self.graph.nvars, (E + 31) // 32)}")
        if slots.shape != (self.R,):
            raise ValueError(f"checkpoint holds {slots.size} slots, this ladder has {self.R}")
        check(lib().ising_sim_set_packed(sim, ptr(words)), self.ctx.handle)
        check(lib().ising_sim_set_counter(sim, int(ck["sweeps"])), self.ctx.handle)
        check(lib().ising_pt_restore(self.handle, ptr(slots), int(ck["swap_step"]), int(ck["total_swaps"])),
              self.ctx.handle)

    def timesteps_sample(self, timesteps, replica_swap_freq=1, sampling_freq=1):
        ns = int(timesteps) // int(sampling_freq) if sampling_freq else 0
        states = PinnedPool.empty((self.R, ns, self.graph.nvars), np.bool_) if ns else \
            np.zeros((self.R, 0, self.graph.nvars), dtype=np.bool_)
        energies = np.empty(self.R, dtype=np.float64)
        check(lib().ising_pt_timesteps_sample(self.handle, int(timesteps), int(replica_swap_freq),
                                              int(sampling_freq), ptr(states), ptr(energies)),
              self.ctx.handle)
        return states, energies

    def close(self):
        if getattr(self, "handle", None):
            lib().ising_pt_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Strip:
    """Rows [row_lo, row_hi) of one large bit-packed 2D lattice (ising_strip)."""

    def __init__(self, ctx, Lx, Ly, row_lo, row_hi, j=-1.0, seed=0, planes=0, rounds=0, ghost=1):
        self.ctx, self.Lx, self.Ly = ctx, int(Lx), int(Ly)
        self.row_lo, self.row_hi = int(row_lo), int(row_hi)
        self.words = self.Lx // 64
        self.ghost = int(ghost)
        h = C.c_void_p()
        check(lib().ising_strip_create_ex(ctx.handle, self.Lx, self.Ly, self.row_lo, self.row_hi, float(j),
                                          int(seed) & (2**64 - 1), self.ghost, C.byref(h)), ctx.handle)
        self.handle = h
        if planes or rounds:
            check(lib().ising_strip_configure(h, int(planes), int(rounds)), ctx.handle)

    def set_all(self, up):
        check(lib().ising_strip_set_all(self.handle, int(bool(up))), self.ctx.handle)

    def set_field(self, h):
        """uniform longitudinal field h (E = sum J s s' - h sum s) of every later phase and sweep"""
        check(lib().ising_strip_set_field(self.handle, float(h)), self.ctx.handle)

    def sweeps(self, betas, comm=None, exchange_every=8, fields=None):
        """One checkerboard sweep per beta with the halo exchange inside the library
        (ising_strip_sweeps): comm = None for a strip that holds the whole lattice.  fields: one
        field h per beta (ising_strip_sweeps_field; the last one stays set), None = the strip's field."""
        b = np.ascontiguousarray(np.atleast_1d(betas), dtype=np.float64)
        c = comm.handle if comm is not None else None
        if fields is None:
            check(lib().ising_strip_sweeps(self.handle, c, ptr(b), len(b), int(exchange_every)), self.ctx.handle)
            return
        f = np.ascontiguousarray(np.atleast_1d(fields), dtype=np.float64)
        if f.shape != b.shape:
            raise ValueError(f"fields: one value per beta ({len(b)}), got {len(f)}")
        check(lib().ising_strip_sweeps_field(self.handle, c, ptr(b), ptr(f), len(b), int(exchange_every)),
              self.ctx.handle)

    def global_sums(self, comm=None):
        """(satisfied bonds, up spins) of the whole lattice over all ranks of comm."""
        a, b = C.c_uint64(0), C.c_uint64(0)
        check(lib().ising_strip_global_sums(self.handle, comm.handle if comm is not None else None,
                                            C.byref(a), C.byref(b)), self.ctx.handle)
        return int(a.value), int(b.value)

    def phase(self, colour, beta):
        check(lib().ising_strip_phase(self.handle, int(colour), float(beta)), self.ctx.handle)

    def phase_rows(self, colour, beta, r0, r1, advance=False, sync=False):
        check(lib().ising_strip_phase_rows(self.handle, int(colour), float(beta), int(r0), int(r1),
                                           int(advance), int(sync)), self.ctx.handle)

    def phase_ext(self, colour, beta, ext, advance=False, sync=False):
        """local rows + ext ghost rows on each side (communication-avoiding batches)"""
        check(lib().ising_strip_phase_ext(self.handle, int(colour), float(beta), int(ext), int(advance),
                                          int(sync)), self.ctx.handle)

    def halo_deep(self, direction, depth, buf, sync=True):
        """buf: numpy uint32[2, 2, depth, words] (host) or an integer device pointer."""
        p = ptr(buf) if isinstance(buf, np.ndarray) else C.c_void_p(int(buf))
        check(lib().ising_strip_halo_deep(self.handle, int(direction), int(depth), p, int(sync)),
              self.ctx.handle)

    def wrap_deep(self, depth):
        check(lib().ising_strip_wrap_deep(self.handle, int(depth)), self.ctx.handle)

    def halo_async(self, colour, direction, buf_ptr):
        check(lib().ising_strip_halo_async(self.handle, int(colour), int(direction),
                                           C.c_void_p(int(buf_ptr))), self.ctx.handle)

    def get_boundary(self, colour, which, dst=None):
        """dst: numpy uint32[words] (host) or an integer device pointer."""
        if dst is None:
            dst = np.empty(self.words, dtype=np.uint32)
        p = ptr(dst) if isinstance(dst, np.ndarray) else C.c_void_p(int(dst))
        check(lib().ising_strip_get_boundary(self.handle, int(colour), int(which), p), self.ctx.handle)
        return dst

    def set_ghost(self, colour, which, src):
        if isinstance(src, np.ndarray):
            src = np.ascontiguousarray(src, dtype=np.uint32)
            p = ptr(src)
        else:
            p = C.c_void_p(int(src))
        check(lib().ising_strip_set_ghost(self.handle, int(colour), int(which), p), self.ctx.handle)

    def wrap_local(self, colour):
        check(lib().ising_strip_wrap_local(self.handle, int(colour)), self.ctx.handle)

    def observables(self):
        a, b = C.c_uint64(0), C.c_uint64(0)
        check(lib().ising_strip_observables(self.handle, C.byref(a), C.byref(b)), self.ctx.handle)
        return int(a.value), int(b.value)

    def rows(self, r0=None, r1=None):
        """bool[rows, Lx] of all local rows, or of the local rows [r0, r1)."""
        if r0 is None and r1 is None:
            out = np.empty((self.row_hi - self.row_lo, self.Lx), dtype=np.bool_)
            check(lib().ising_strip_get_rows(self.handle, ptr(out)), self.ctx.handle)
            return out
        r0 = 0 if r0 is None else int(r0)
        r1 = self.row_hi - self.row_lo if r1 is None else int(r1)
        out = np.empty((r1 - r0, self.Lx), dtype=np.bool_)
        check(lib().ising_strip_get_row_range(self.handle, r0, r1, ptr(out)), self.ctx.handle)
        return out

    def stats(self, reset=False):
        a, b = C.c_uint64(0), C.c_double(0)
        check(lib().ising_strip_get_stats(self.handle, C.byref(a), C.byref(b), int(reset)), self.ctx.handle)
        return {"launches": int(a.value), "device_ms": float(b.value)}

    def close(self):
        if getattr(self, "handle", None):
            lib().ising_strip_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def strong_edge_colouring(nvars, a, b):
    """Host only: class of every bond such that two bonds of a class share no site and no bond
    joins them (ising_strong_edge_colouring) -> (uint32[nedges], number of classes)."""
    a = np.ascontiguousarray(a, dtype=np.uint64)
    b = np.ascontiguousarray(b, dtype=np.uint64)
    cls = np.empty(len(a), dtype=np.uint32)
    n = C.c_uint32(0)
    check(lib().ising_strong_edge_colouring(int(nvars), len(a), ptr(a), ptr(b), ptr(cls), C.byref(n)))
    return cls, int(n.value)


def decide_swaps(betas, all_energies, seed, swap_step, slot_of_config, config_of_slot):
    """Host-only swap decisions of one tempering step (ising_pt_decide_swaps); the two
    permutation arrays (uint32) are updated in place, returns the number of swaps."""
    b = np.ascontiguousarray(betas, dtype=np.float64)
    e = np.ascontiguousarray(all_energies, dtype=np.float64)
    assert slot_of_config.dtype == np.uint32 and config_of_slot.dtype == np.uint32
    n = C.c_uint64(0)
    check(lib().ising_pt_decide_swaps(ptr(b), len(b), ptr(e), int(seed) & (2**64 - 1), int(swap_step),
                                      ptr(slot_of_config), ptr(config_of_slot), C.byref(n)))
    return int(n.value)


def make_seeds(seed_gen, n):
    out = np.empty(int(n), dtype=np.uint64)
    check(lib().ising_make_seeds(int(seed_gen) & (2**64 - 1), int(n), ptr(out)))
    return out


def schedule_betas(stops, timesteps, linear=False):
    """Per-timestep betas of the annealing entry points (lattice.rs:320-334, 357-365)."""
    t = np.ascontiguousarray([s[0] for s in stops], dtype=np.uint64)
    b = np.ascontiguousarray([s[1] for s in stops], dtype=np.float64)
    out = np.empty(int(timesteps), dtype=np.float64)
    check(lib().ising_schedule_betas(ptr(t), ptr(b), len(t), int(timesteps), int(bool(linear)), ptr(out)))
    return out


def run_args(**kw):
    a = RunArgs()
    a.struct_size = C.sizeof(RunArgs)
    keep = []
    for k, v in kw.items():
        if k in ("sched_t", "sched_beta", "initial_state"):
            if v is not None:
                keep.append(v)
                setattr(a, k, v.ctypes.data)
        else:
            setattr(a, k, v)
    a._keepalive = keep
    return a
