/*
 * ising_b200.h -- C ABI of libising_b200.so, the B200 (sm_100a) engine behind the classical
 * Monte-Carlo path of py_monte_carlo (Renmusxd/PyIsingMonteCarlo).
 *
 * The reference has no FFI seam on this path: src/lattice.rs calls the out-of-tree Rust type
 * qmc::classical::graph::GraphState by static linkage (lattice.rs:5,199).  Each entry point
 * below names the reference call it replaces; INTEGRATION.md shows the Rust `extern "C"`
 * block and the patched call sites a maintainer would add.
 *
 * Conventions: every function returns ISING_OK (0) or an ISING_E_* code and never aborts;
 * the message of the last failure is ising_last_error(ctx) (ctx may be NULL for failures of
 * ising_ctx_create itself).  All buffers are caller-owned HOST memory unless a name ends in
 * `_dev`.  A context is bound to one CUDA device and one stream and is not re-entrant.
 * Energies use the reference's convention E = sum_edges J s_a s_b - sum_i b_i s_i with
 * s = +1 for `true`, so J > 0 is antiferromagnetic (README.md:45-46, lattice.rs:43-44).
 */
#ifndef ISING_B200_H
#define ISING_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ISING_ABI_VERSION 1

#if defined(__GNUC__)
#define ISING_API __attribute__((visibility("default")))
#else
#define ISING_API
#endif

enum {
    ISING_OK = 0,
    ISING_E_INVALID = 1,     /* bad argument (reference: PyValueError)                      */
    ISING_E_CUDA = 2,        /* CUDA runtime failure, no device, or wrong architecture      */
    ISING_E_UNSUPPORTED = 3, /* valid in the reference but not on the GPU path (D1/D2)      */
    ISING_E_AMBIGUOUS = 4,   /* replay: a uniform fell within rounding of exp(-beta dE)     */
    ISING_E_NOMEM = 5
};

typedef struct ising_ctx ising_ctx;
typedef struct ising_graph ising_graph;
typedef struct ising_sim ising_sim;
typedef struct ising_pt ising_pt;
typedef struct ising_strip ising_strip;
typedef struct ising_comm ising_comm;

/* ---- context ---------------------------------------------------------------------------- */
ISING_API int ising_abi_version(void);
ISING_API int ising_ctx_create(int device, ising_ctx **out);
/* Same, on the caller's CUDA stream (cudaStream_t passed as void*): launches are then ordered
 * with the caller's own kernels and NCCL calls without host synchronisation. */
ISING_API int ising_ctx_create_on_stream(int device, void *cuda_stream, ising_ctx **out);
ISING_API void ising_ctx_destroy(ising_ctx *ctx);
ISING_API const char *ising_last_error(const ising_ctx *ctx);

/* Page-locked host memory for output arrays.  The reference allocates its outputs itself
 * (lattice.rs:183-184) and hands them to numpy; a host layer that allocates them here gets
 * D2H copies at PCIe speed instead of pageable staging. */
ISING_API int ising_host_alloc(size_t bytes, void **out);
ISING_API void ising_host_free(void *p);

/* ---- graph layout (replaces GraphState::new's adjacency build, lattice.rs:199) ----------- */
enum { ISING_KIND_GENERAL = 0, ISING_KIND_STENCIL2D = 2, ISING_KIND_STENCIL3D = 3 };

typedef struct ising_graph_info {
    uint64_t nvars;
    uint64_t nedges;
    int32_t kind;         /* ISING_KIND_*                                                  */
    int32_t ncolors;      /* colour classes of the sweep                                   */
    int32_t max_degree;
    int32_t integer_classes; /* 1: all |J| equal and no bias -> bit-sliced integer kernel  */
    uint64_t dims[3];     /* stencil extents (x fastest), 1 where unused                   */
    double jabs;          /* common |J| when integer_classes                               */
} ising_graph_info;

/* Edge list in SoA form, a copy of Lattice.edges: Vec<((usize,usize),f64)> (lattice.rs:31);
 * biases = nvars values or NULL for 0 (lattice.rs:186-189).  The host compiles CSR + a
 * greedy colouring and recognises row-major square / cubic tori (checkerboard layout). */
ISING_API int ising_graph_from_edges(ising_ctx *ctx, uint64_t nvars, uint64_t nedges, const uint64_t *a,
                           const uint64_t *b, const double *j, const double *biases,
                           ising_graph **out);
/* Additive constructor for lattices too large for a Python edge list: dim in {2,3}, periodic,
 * site index x + Lx*(y + Ly*z).  pmj = 0: every bond = j0;  pmj = 1: bond = +-|j0| iid with
 * probability 1/2 from Philox(j_seed) (one disorder sample shared by all experiments). */
ISING_API int ising_graph_torus(ising_ctx *ctx, int dim, const uint64_t *L, double j0, int pmj,
                      uint64_t j_seed, ising_graph **out);
/* The same torus in a uniform longitudinal field h: E = sum_edges J s_a s_b - h sum_i s_i, so h > 0
 * favours up spins.  Runs on the bit-sliced field kernel with exact integer thresholds per
 * (spin, satisfied bonds) class, also for h = 0 (then bit for bit what ising_graph_torus runs).
 * Non-finite h -> ISING_E_INVALID.  Per-replica betas (ising_sim_set_betas), edge / worm moves,
 * ISING_SIM_GENERAL_LAYOUT, tempering (ising_pt_create) and ising_replay refuse such a graph with
 * ISING_E_UNSUPPORTED. */
ISING_API int ising_graph_torus_field(ising_ctx *ctx, int dim, const uint64_t *L, double j0, int pmj,
                            uint64_t j_seed, double h, ising_graph **out);
ISING_API void ising_graph_destroy(ising_graph *g);
ISING_API int ising_graph_get_info(const ising_graph *g, ising_graph_info *out);
ISING_API int ising_graph_get_colors(const ising_graph *g, uint32_t *colors /* nvars */);
ISING_API int ising_graph_get_edges(const ising_graph *g, uint64_t *a, uint64_t *b, double *j);
/* Class of every bond in the strong edge colouring the two-spin edge moves are launched by
 * (ising_sim_set_moves): cls[nedges], two bonds of a class share no site and no bond joins them.
 * The CPU mirror of the tests needs it to replay a pass in the library's order. */
ISING_API int ising_graph_get_edge_classes(ising_graph *g, uint32_t *cls);
/* The colouring alone, on the host (no context, no device): cls[nedges], *nclasses. */
ISING_API int ising_strong_edge_colouring(uint64_t nvars, uint64_t nedges, const uint64_t *a, const uint64_t *b,
                                uint32_t *cls, uint32_t *nclasses);

/* ---- seeds (Lattice::make_seeds, lattice.rs:83-91, seed_gen = Some(seed)) ---------------- */
ISING_API int ising_make_seeds(uint64_t seed_gen, uint64_t n, uint64_t *out);

/* ---- device-resident simulation: E experiments of one graph, replica-bit-packed ---------- */
/* replica_offset = global index of this shard's first experiment (multiple of 32); it only
 * enters the Philox counters, so a sharded run reproduces the unsharded one bit for bit.   */
ISING_API int ising_sim_create(ising_ctx *ctx, const ising_graph *g, uint64_t num_experiments,
                     uint64_t seed, uint64_t replica_offset, ising_sim **out);
/* flags: ISING_SIM_GENERAL_LAYOUT runs a recognised torus through the general (colour x degree
 * group) kernels in natural site order (cross-check of the two kernel families). */
enum { ISING_SIM_GENERAL_LAYOUT = 1u << 0 };
ISING_API int ising_sim_create_ex(ising_ctx *ctx, const ising_graph *g, uint64_t num_experiments,
                        uint64_t seed, uint64_t replica_offset, uint32_t flags, ising_sim **out);
ISING_API void ising_sim_destroy(ising_sim *sim);
/* Experiment e runs at betas[e] from now on (parallel tempering: one replica bit per
 * temperature); afterwards ising_sim_sweeps takes betas = NULL.  Graphs with integer energy
 * classes (all |J| equal, no bias) get bit-sliced per-replica threshold tables (on lattices for
 * planes = 6); real couplings / biases run on the float-field kernel with one beta per replica bit. */
ISING_API int ising_sim_set_betas(ising_sim *sim, const double *betas /* E */);
/* Tuning knobs of the multi-spin-coded kernel; 0 keeps the default.  planes = bit-planes
 * compared before the per-bit resolver (5..7), rounds = Philox4x32 rounds (7 or 10).      */
ISING_API int ising_sim_configure(ising_sim *sim, int planes, int rounds);
/* What one timestep consists of: the arguments of qmc GraphState::do_time_step(beta,
 * nspinupdates, nedgeupdates, nwormupdates, only_basic_moves) as the reference passes them at
 * lattice.rs:205, 272, 278, 366, 452 and classicising.rs:100-106, 146-165, in units of whole
 * passes.  Default (never called, or moves = NULL): one colour-class sweep, no other move.
 *   spin_sweeps      0 or 1 colour-class sweeps of single-spin Metropolis attempts
 *   edge_passes      passes over all bonds of two-spin moves (both ends of a bond flip together),
 *                    one launch per class of a strong edge colouring
 *   worms, worm_len  worm moves per experiment: a self-avoiding chain of worm_len (1..8) sites
 *                    from a uniformly random site, flipped as a whole; worm_len = 1 is the
 *                    reference's attempt at a uniformly random site
 *   edge_importance  GraphState::enable_edge_importance_sampling (lattice.rs:200, classicising.rs:76):
 *                    a bond is attempted at a rate proportional to |J|
 * All are Metropolis moves with symmetric (or ratio-corrected) proposals, so any mix keeps the
 * Boltzmann distribution; their rules inside the `qmc` crate could not be read (DESIGN.md D1). */
typedef struct ising_moves {
    uint32_t struct_size;      /* sizeof(ising_moves) */
    uint32_t spin_sweeps;
    uint32_t edge_passes;
    uint32_t worms;
    uint32_t worm_len;
    uint32_t edge_importance;
} ising_moves;
ISING_API int ising_sim_set_moves(ising_sim *sim, const ising_moves *moves);
/* Random start (GraphState::new's make_random_spin_state, one Philox bit per spin) ...     */
ISING_API int ising_sim_randomize(ising_sim *sim);
/* ... or the same given state for every experiment (Lattice.set_initial_state, :201-203).  */
ISING_API int ising_sim_set_state(ising_sim *sim, const uint8_t *state /* nvars */);
/* Per-experiment states, bool[E, nvars] (ClassicIsing.add_graph(initial_state)).           */
ISING_API int ising_sim_set_states(ising_sim *sim, const uint8_t *states /* E*nvars */);
/* nsweeps colour-class sweeps (1 sweep = every site attempted once = one reference
 * "timestep" of nvars attempts); sweep k runs at betas[k].  If energies_per_sweep != NULL it
 * receives double[E, nsweeps] (GraphState::get_energy after every timestep, lattice.rs:454). */
ISING_API int ising_sim_sweeps(ising_sim *sim, const double *betas, uint64_t nsweeps,
                     double *energies_per_sweep);
/* thermalization sweeps, then n_samples x (sampling_freq sweeps, state copy, energy) on the
 * resident state: ClassicIsing::run_monte_carlo_sampling (classicising.rs:119-179) and the body
 * of Lattice::run_monte_carlo_sampling.  energies[E, n_samples], states bool[E, n_samples, nvars] */
ISING_API int ising_sim_run_sampling(ising_sim *sim, double beta, uint64_t thermalization,
                           uint64_t sampling_freq, uint64_t n_samples, double *energies,
                           uint8_t *states);
/* Opt-in packed form of the same loop (additive, SURVEY 8(f)2): samples as
 * uint32[n_samples, nvars, ceil(E/32)] in natural site order (bit e%32 of word e/32 is
 * experiment e, as ising_sim_get_packed) -- 8x less D2H than bool[E, n_samples, nvars], the only
 * practical form at config 2 size (2 GiB instead of 17 GB per sample). */
ISING_API int ising_sim_run_sampling_packed(ising_sim *sim, double beta, uint64_t thermalization,
                                  uint64_t sampling_freq, uint64_t n_samples, double *energies,
                                  uint32_t *words);
/* The same loop without the state read-back (additive; feeds SURVEY 8(f)2): per sample the
 * energy, the magnetisation M = sum_i s_i and the overlap Q = sum_i s_i^(2p) s_i^(2p+1) of the
 * experiment pairs (2p, 2p+1), all reduced on the device.  energies / mags double[E, n_samples],
 * overlaps double[E / 2, n_samples]; any of the three may be NULL.                           */
ISING_API int ising_sim_run_observables(ising_sim *sim, double beta, uint64_t thermalization,
                              uint64_t sampling_freq, uint64_t n_samples, double *energies,
                              double *mags, double *overlaps);
ISING_API int ising_sim_get_energies(ising_sim *sim, double *energies /* E */);
ISING_API int ising_sim_get_states(ising_sim *sim, uint8_t *states /* E*nvars, bool */);
/* Opt-in packed read-back: uint32[nvars, ceil(E/32)] in natural site order (bit e%32 of word
 * e/32 is experiment e) -- 8x less D2H than bool[E, nvars].                                 */
ISING_API int ising_sim_get_packed(ising_sim *sim, uint32_t *words);
/* Checkpointing (the reference saves only its QMC classes, tempering.rs:307-347, and never the
 * RNG state; here seed + sweep counter + packed spins are the complete state, so a restored
 * run continues bit for bit).  words: uint32[nvars, ceil(E/32)] as from ising_sim_get_packed. */
ISING_API int ising_sim_set_packed(ising_sim *sim, const uint32_t *words);
ISING_API int ising_sim_get_counter(const ising_sim *sim, uint64_t *sweeps_done);
ISING_API int ising_sim_set_counter(ising_sim *sim, uint64_t sweeps_done);
/* One timestep at beta and, per experiment, the number of spins it changed (= accepted single-spin
 * flips for the default timestep, in which every site is attempted exactly once).  The per-run
 * acceptance metric; measured by differencing the packed state, at no cost to the sweep kernels. */
ISING_API int ising_sim_step_acceptance(ising_sim *sim, double beta, uint64_t *changed /* E */);
/* per-experiment magnetisation sum_i s_i */
ISING_API int ising_sim_get_magnetization(ising_sim *sim, double *m /* E */);

typedef struct ising_sim_stats {
    uint64_t kernel_launches;  /* kernels launched by this sim since creation / last reset   */
    uint64_t sweeps;
    uint64_t flip_attempts;    /* E_padded-free count: E * nvars * sweeps                    */
    double sweep_device_ms;    /* CUDA-event time of the sweep kernels (on the ctx stream)   */
    double sweep_kernel_ms;    /* same, summed over sweep-kernel launches only               */
    uint64_t sweep_kernel_launches;
    uint64_t edge_attempts;    /* two-spin edge moves attempted (ising_sim_set_moves)        */
    uint64_t worm_attempts;    /* worm moves attempted                                       */
} ising_sim_stats;
ISING_API int ising_sim_get_stats(ising_sim *sim, ising_sim_stats *out);
ISING_API int ising_sim_reset_stats(ising_sim *sim);

/* ---- one blocking call per pymethod (host buffers in, host buffers out) ------------------ */
enum {
    ISING_FLAG_ONLY_BASIC_MOVES = 1u << 0,  /* informational: the GPU path is always basic  */
    ISING_FLAG_PER_STEP_ENERGIES = 1u << 1, /* annealing_and_get_energies                   */
    ISING_FLAG_LINEAR_SCHEDULE = 1u << 2,   /* documented interpolation instead of quirk Q1 */
    ISING_FLAG_EDGE_IMPORTANCE = 1u << 3,   /* needs ISING_FLAG_NON_BASIC_MOVES, else ISING_E_UNSUPPORTED */
    ISING_FLAG_NON_BASIC_MOVES = 1u << 4    /* every timestep also runs one pass of edge moves and one
                                               worm of 4 sites per experiment (ising_sim_set_moves) */
};

typedef struct ising_run_args {
    uint32_t struct_size;        /* sizeof(ising_run_args)                                  */
    uint32_t flags;
    double beta;                 /* run / sampling                                          */
    const uint64_t *sched_t;     /* annealing stops (time, beta), any order, may be empty   */
    const double *sched_beta;
    uint64_t sched_len;
    uint64_t timesteps;
    uint64_t num_experiments;
    uint64_t thermalization;     /* sampling                                                */
    uint64_t sampling_freq;      /* sampling; 0 -> ISING_E_INVALID                          */
    uint64_t seed;               /* Philox key (Lattice.seed_gen or entropy drawn by caller) */
    uint64_t replica_offset;     /* see ising_sim_create                                    */
    const uint8_t *initial_state; /* nvars bools or NULL                                    */
} ising_run_args;

/* Lattice::run_monte_carlo, lattice.rs:171-221: energies[E], states bool[E, nvars]. */
ISING_API int ising_run_monte_carlo(ising_ctx *ctx, const ising_graph *g, const ising_run_args *args,
                          double *energies, uint8_t *states);
/* Lattice::run_monte_carlo_sampling, lattice.rs:231-299: energies[E, n_s], states[E, n_s, nvars]
 * with n_s = timesteps / sampling_freq. */
ISING_API int ising_run_monte_carlo_sampling(ising_ctx *ctx, const ising_graph *g,
                                   const ising_run_args *args, double *energies,
                                   uint8_t *states);
/* Lattice::run_monte_carlo_annealing (lattice.rs:309-385; energies[E]) and
 * ..._and_get_energies (395-470; ISING_FLAG_PER_STEP_ENERGIES, energies[E, timesteps]). */
ISING_API int ising_run_monte_carlo_annealing(ising_ctx *ctx, const ising_graph *g,
                                    const ising_run_args *args, double *energies,
                                    uint8_t *states);
/* The per-timestep betas the annealing entry points use (schedule normalisation of
 * lattice.rs:320-334 and the beta expression of :357-365).  out[timesteps]. */
ISING_API int ising_schedule_betas(const uint64_t *sched_t, const double *sched_beta, uint64_t sched_len,
                         uint64_t timesteps, int linear, double *out);

/* ---- replay mode: the reference's own (site, uniform) sequence, bit-exact ---------------- */
/* Sequential random-site Metropolis exactly as GraphState::do_spin_flip / should_flip:
 * dE summed over the adjacency in ascending neighbour order in f64, accept iff
 * !(dE > 0) || u < exp(-beta dE).  sites[E, nattempts], u[E, nattempts] (entries of attempts
 * with dE <= 0 are ignored), init bool[E, nvars]; energies[E], states bool[E, nvars]. */
ISING_API int ising_replay(ising_ctx *ctx, const ising_graph *g, double beta, uint64_t num_experiments,
                 uint64_t nattempts, const uint32_t *sites, const double *u,
                 const uint8_t *init, double *energies, uint8_t *states);

/* ---- communicator of the multi-GPU paths (one process per GPU) ----------------------------- */
/* The reference's only parallel axes are rayon loops inside one process (experiments,
 * lattice.rs:192-197; tempering replicas, tempering.rs:179-186).  Across GPUs the same axes are
 * sharded over processes, and what the hot path exchanges - the replica energies of a tempering
 * swap step, the boundary rows of a strip decomposition - moves through NCCL calls this library
 * makes on the context's stream.  NCCL is bound at run time (dlopen of libnccl.so.2, shared with
 * whatever copy the process already loaded).  Rank 0 obtains an id, the host layer broadcasts
 * its ISING_COMM_ID_BYTES bytes by any means, every rank creates its communicator from it. */
#define ISING_COMM_ID_BYTES 128
ISING_API int ising_comm_unique_id(uint8_t *out, uint64_t capacity);
ISING_API int ising_comm_create(ising_ctx *ctx, const uint8_t *id, int rank, int world, ising_comm **out);
ISING_API void ising_comm_destroy(ising_comm *comm);
ISING_API int ising_comm_info(const ising_comm *comm, int *rank, int *world);

/* ---- classical parallel tempering with the cadence of tempering.rs:156-222 --------------- */
/* One configuration per inverse temperature ("slot"), every configuration one replica bit of
 * the packed layout, so a whole temperature ladder advances in one sweep.  A swap exchanges the
 * betas of two configurations (equivalent to exchanging the configurations, tempering.rs:192),
 * nothing moves.  Multi-GPU: rank r owns configurations [cfg_lo, cfg_hi); after an all-gather
 * of the per-configuration energies every rank takes identical swap decisions (Philox keyed
 * by seed and swap step), so there is no second collective.  Any graph ising_sim_create takes:
 * integer-class graphs are bit-exact against the CPU mirror; real couplings / biases (a longitudinal
 * field, tempering.rs:70-75) use the float-field kernel and f64 energies from the device, whose
 * atomic summation order can move a swap decision that sits within an ulp of its threshold. */
ISING_API int ising_pt_create(ising_ctx *ctx, const ising_graph *g, const double *betas, uint64_t nbetas,
                    uint64_t cfg_lo, uint64_t cfg_hi, uint64_t seed, ising_pt **out);
ISING_API void ising_pt_destroy(ising_pt *pt);
ISING_API int ising_pt_configure(ising_pt *pt, int planes, int rounds);
/* t sweeps of the local configurations, then their energies, local_energies[cfg_hi - cfg_lo]
 * (may be NULL).  Replaces graph.timesteps(t, beta) of tempering.rs:179-186. */
ISING_API int ising_pt_sweeps(ising_pt *pt, uint64_t t, double *local_energies);
/* TemperingContainer::parallel_tempering_step (tempering.rs:192); all_energies[nbetas] by
 * configuration. */
ISING_API int ising_pt_swap_step(ising_pt *pt, const double *all_energies);
/* The decision rule alone (host only, no device): even pairs then odd pairs of slots, pair
 * (a, a+1) swaps with probability min(1, exp((b_a - b_{a+1})(E_a - E_{a+1}))), uniform =
 * Philox(seed; a, parity, swap_step).  Updates the two permutations in place. */
ISING_API int ising_pt_decide_swaps(const double *betas, uint64_t nbetas, const double *all_energies,
                          uint64_t seed, uint64_t swap_step, uint32_t *slot_of_config,
                          uint32_t *config_of_slot, uint64_t *nswaps);
ISING_API int ising_pt_get_slots(const ising_pt *pt, uint32_t *slot_of_config /* nbetas */);
ISING_API int ising_pt_get_local_states(ising_pt *pt, uint8_t *states /* (cfg_hi-cfg_lo)*nvars */);
/* checkpoint support: the sim holding the ladder's configurations (borrowed, do not destroy),
 * the swap counters, and restoring the slot permutation */
ISING_API int ising_pt_get_sim(ising_pt *pt, ising_sim **out);
ISING_API int ising_pt_get_counters(const ising_pt *pt, uint64_t *swap_step, uint64_t *total_swaps);
ISING_API int ising_pt_restore(ising_pt *pt, const uint32_t *slot_of_config, uint64_t swap_step,
                     uint64_t total_swaps);
/* LatticeTempering::get_total_swaps, tempering.rs:297-299 */
ISING_API int ising_pt_total_swaps(const ising_pt *pt, uint64_t *out);
/* Swaps attempted / accepted per pair of neighbouring betas (pair a = slots a and a + 1;
 * attempts[nbetas - 1], accepts[nbetas - 1]): the per-pair view of get_total_swaps. */
ISING_API int ising_pt_get_pair_stats(const ising_pt *pt, uint64_t *attempts, uint64_t *accepts);
/* Shards the ladder over the ranks of a communicator (tempering.rs:179-186 is the reference's
 * replica axis): rank r must have been created with the r-th contiguous block of configurations
 * (blocks of nbetas / world, remainder to the first ranks).  From then on
 * ising_pt_timesteps_sample all-gathers the energies (and the sampled states) with NCCL on the
 * context's stream and every rank returns the full arrays. */
ISING_API int ising_pt_set_comm(ising_pt *pt, ising_comm *comm);
/* LatticeTempering::qmc_timesteps_sample (tempering.rs:156-222):
 * states bool[R, timesteps / sampling_freq, nvars], energies[R].  Device-resident: sweeps,
 * energies, swap decisions (Philox + a fixed-sequence exp, identical to ising_pt_decide_swaps),
 * threshold tables and samples are all enqueued on the context's stream; the host waits once. */
ISING_API int ising_pt_timesteps_sample(ising_pt *pt, uint64_t timesteps, uint64_t replica_swap_freq,
                              uint64_t sampling_freq, uint8_t *states, double *energies);

/* ---- one large 2D lattice, domain-decomposed in row strips (BASELINE config 5) ---------- */
/* The reference cannot run this at all (one experiment = one thread, lattice.rs:197-212; the
 * 8.6e9-edge list would not fit).  One uniform-J periodic Lx x Ly lattice, spins bit-packed along
 * x; this rank owns rows [row_lo, row_hi) plus two ghost rows.  Per colour phase the caller
 * moves one boundary row (Lx/64 words) to each neighbouring strip -- get_boundary / set_ghost
 * take host or device pointers, so the exchange can be NCCL send/recv between ranks -- or calls
 * wrap_local when a single strip holds the whole lattice.  The random numbers are keyed by the
 * global row, so any strip decomposition produces the same configuration. */
ISING_API int ising_strip_create(ising_ctx *ctx, uint64_t Lx, uint64_t Ly, uint64_t row_lo, uint64_t row_hi,
                       double j, uint64_t seed, ising_strip **out);
/* Communication-avoiding variant: `ghost` ghost rows on each side (1 <= ghost <= rows).  After
 * ONE exchange of 2k boundary rows of both colours (halo_deep / wrap_deep) the strip runs k
 * sweeps without talking to its neighbours: phase q = 0 .. 2k-1 of the batch updates the local
 * rows plus ext = 2k-1-q ghost rows on each side (phase_ext); the redundant ghost updates
 * reproduce the neighbour's bits because the random numbers are keyed by the global row. */
ISING_API int ising_strip_create_ex(ising_ctx *ctx, uint64_t Lx, uint64_t Ly, uint64_t row_lo, uint64_t row_hi,
                          double j, uint64_t seed, uint32_t ghost, ising_strip **out);
ISING_API int ising_strip_phase_ext(ising_strip *s, int colour, double beta, uint32_t ext, int advance_sweep,
                          int sync);
/* buf = uint32[2 sides][2 colours][depth][Lx/64], host or device.  dir 0: side 0 <- first `depth`
 * local rows, side 1 <- last `depth` local rows; dir 1: side 0 -> ghost rows above, side 1 ->
 * ghost rows below.  A strip sends side 0 up and side 1 down. */
ISING_API int ising_strip_halo_deep(ising_strip *s, int dir, uint32_t depth, void *buf, int sync);
ISING_API int ising_strip_wrap_deep(ising_strip *s, uint32_t depth);
ISING_API void ising_strip_destroy(ising_strip *s);
ISING_API int ising_strip_configure(ising_strip *s, int planes, int rounds);
ISING_API int ising_strip_set_all(ising_strip *s, int up);
ISING_API int ising_strip_phase(ising_strip *s, int colour, double beta);
/* local rows [r0, r1) of a colour phase; sync = 0 only enqueues on the context's stream */
ISING_API int ising_strip_phase_rows(ising_strip *s, int colour, double beta, uint64_t r0, uint64_t r1,
                           int advance_sweep, int sync);
/* device-side halo staging without host wait: dir 0 = boundary rows -> buf_dev[2*Lx/64 words],
 * dir 1 = buf_dev -> ghost rows */
ISING_API int ising_strip_halo_async(ising_strip *s, int colour, int dir, void *buf_dev);
ISING_API int ising_strip_get_boundary(ising_strip *s, int colour, int which, void *dst_words);
ISING_API int ising_strip_set_ghost(ising_strip *s, int colour, int which, const void *src_words);
ISING_API int ising_strip_wrap_local(ising_strip *s, int colour);
ISING_API int ising_strip_observables(ising_strip *s, uint64_t *nsat_local, uint64_t *up_local);
/* nsweeps whole sweeps of a lattice split in row strips over the ranks of `comm` (NULL: this
 * strip holds the whole lattice): batches of `exchange_every` sweeps, one deep halo exchange of
 * 2 * exchange_every boundary rows per side (ncclSend / ncclRecv on the context's stream) per
 * batch, ghost rows updated redundantly in between.  exchange_every is clipped to ghost / 2. */
ISING_API int ising_strip_sweeps(ising_strip *s, ising_comm *comm, const double *betas, uint64_t nsweeps,
                       uint32_t exchange_every);
/* Uniform longitudinal field h (E = sum J s s' - h sum s, s = +1 for an up spin) for every later
 * phase (_phase, _phase_rows, _phase_ext) and sweep (_sweeps) of the strip; ISING_E_INVALID unless
 * finite.  h = 0 (either sign) runs the zero-field kernel with its bits. */
ISING_API int ising_strip_set_field(ising_strip *s, double h);
/* ising_strip_sweeps with one (betas[t], fields[t]) per sweep, e.g. a field reversal or ramp; the
 * strip's field is fields[nsweeps - 1] afterwards.  ISING_STRIP_FUSE=1 has no field variant: sweeps
 * with h != 0 run the two phase launches. */
ISING_API int ising_strip_sweeps_field(ising_strip *s, ising_comm *comm, const double *betas, const double *fields,
                             uint64_t nsweeps, uint32_t exchange_every);
/* satisfied bonds and up spins of the WHOLE lattice (halo exchange + all-reduce inside) */
ISING_API int ising_strip_global_sums(ising_strip *s, ising_comm *comm, uint64_t *nsat, uint64_t *up);
ISING_API int ising_strip_get_rows(ising_strip *s, uint8_t *rows_out /* (row_hi-row_lo)*Lx bool */);
/* local rows [r0, r1) only: bool[r1 - r0, Lx] */
ISING_API int ising_strip_get_row_range(ising_strip *s, uint64_t r0, uint64_t r1, uint8_t *rows_out);
ISING_API int ising_strip_get_stats(ising_strip *s, uint64_t *launches, double *device_ms, int reset);

#ifdef __cplusplus
}
#endif
#endif /* ISING_B200_H */
