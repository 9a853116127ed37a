// C ABI: the device-resident simulation object (ising_sim_*): state, sweeps, energies, read-back.
#include "api_internal.h"

// ------------------------------------------------------------------------------------------
// simulation object
// ------------------------------------------------------------------------------------------
void count_launch(ising_sim* s, int n) {
    if (n > 0) s->stats.kernel_launches += (uint64_t)n;
}

extern "C" int ising_sim_create_ex(ising_ctx* ctx, const ising_graph* g, uint64_t E, uint64_t seed,
                                   uint64_t replica_offset, uint32_t flags, ising_sim** out) {
    CtxLock _lk(ctx);
    if (!ctx || !g || !out) return fail(ctx, ISING_E_INVALID, "ctx/graph/out is NULL");
    *out = nullptr;
    if (g->ctx != ctx) return fail(ctx, ISING_E_INVALID, "graph belongs to another context");
    if (E == 0) return fail(ctx, ISING_E_INVALID, "num_experiments must be > 0");
    if (replica_offset % 32) return fail(ctx, ISING_E_INVALID, "replica_offset must be a multiple of 32");
    const HostGraph& h = g->h;
    // Philox counter word 0 is the 32-bit site index
    if (h.nvars > 0xFFFFFFFFull)
        return fail(ctx, ISING_E_UNSUPPORTED, "graphs of 2^32 or more sites are not supported (32-bit site index in the RNG counter)");
    if (h.field_graph && (flags & ISING_SIM_GENERAL_LAYOUT))
        return fail(ctx, ISING_E_UNSUPPORTED, "a torus in a field runs on the stencil layout only (no ISING_SIM_GENERAL_LAYOUT)");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    // integer energy classes (all |J| equal, no bias, degree <= 15) use the bit-sliced kernels;
    // anything else the reference accepts runs on the float-field kernel
    // (max_degree is known without the CSR: compile_from_edges builds it, make_torus sets 2*dim)
    const bool real = !h.integer_classes || (h.kind == ISING_KIND_GENERAL && h.max_degree > GEN_MAX_DEG);
    const bool general = real || h.kind == ISING_KIND_GENERAL || (flags & ISING_SIM_GENERAL_LAYOUT);
    if (real) {
        const int rc = ensure_real_on_device(ctx, const_cast<ising_graph*>(g));
        if (rc) return rc;
    } else if (general) {
        const int rc = ensure_general_on_device(ctx, const_cast<ising_graph*>(g));
        if (rc) return rc;
    }
    std::unique_ptr<ising_sim> s(new ising_sim);
    s->ctx = ctx;
    s->g = g;
    s->E = E;
    s->seed = seed;
    s->replica_offset = replica_offset;
    s->general = general;
    s->real = real;
    s->field = h.field_graph;
    Layout& L = s->lay;
    L.kind = general ? ISING_KIND_GENERAL : h.kind;
    L.Lx = (uint32_t)h.dims[0];
    L.Ly = (uint32_t)h.dims[1];
    L.Lz = (uint32_t)h.dims[2];
    L.Lxh = L.Lx / 2;
    L.rows = L.Ly * L.Lz;
    L.W = (uint32_t)((E + 31) / 32);
    L.nvars = h.nvars;
    L.halfN = h.nvars / 2;
    if (!general && (uint64_t)L.Lxh * L.W > 0xFFFFFFFFull)
        return fail(ctx, ISING_E_UNSUPPORTED, "lattice row too long for 32-bit word offsets");
    const size_t words = (size_t)h.nvars * L.W;
    s->spins_bytes = words * sizeof(uint32_t);
    s->counts_bytes = (size_t)L.W * 32 * sizeof(unsigned long long) * (s->field ? 2 : 1);
    void* p = nullptr;
    CUDA_TRY(ctx, ctx_buf_get(ctx, s->spins_bytes, &p));
    s->d_spins = (uint32_t*)p;
    cudaError_t ce = ctx_buf_get(ctx, s->counts_bytes, &p);
    if (ce != cudaSuccess) {
        ctx_buf_put(ctx, s->d_spins, s->spins_bytes);
        CUDA_TRY(ctx, ce);
    }
    s->d_counts = (unsigned long long*)p;
    *out = s.release();
    ctx_retain(ctx);
    return ising_sim_randomize(*out);
}

extern "C" int ising_sim_create(ising_ctx* ctx, const ising_graph* g, uint64_t E, uint64_t seed,
                                uint64_t replica_offset, ising_sim** out) {
    CtxLock _lk(ctx);
    return ising_sim_create_ex(ctx, g, E, seed, replica_offset, 0u, out);
}

extern "C" void ising_sim_destroy(ising_sim* s) {
    if (!s) return;
    struct Release { ising_ctx* c; ~Release() { ctx_release(c); } } _rel{s->ctx};   // after the lock is gone
    CtxLock _lk(s->ctx);
    cudaSetDevice(s->ctx->device);
    cudaStreamSynchronize(s->ctx->stream);
    ctx_buf_put(s->ctx, s->d_spins, s->spins_bytes);
    ctx_buf_put(s->ctx, s->d_counts, s->counts_bytes);
    cudaFree(s->d_t64);
    cudaFree(s->d_slot);
    cudaFree(s->d_tplane);
    cudaFree(s->d_tlow);
    delete s;
}

extern "C" int ising_sim_configure(ising_sim* s, int planes, int rounds) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s) return fail(nullptr, ISING_E_INVALID, "sim is NULL");
    if (planes) {
        if (planes < 5 || planes > 7) return fail(s->ctx, ISING_E_INVALID, "planes must be 5..7");
        s->planes = planes;
    }
    if (rounds) {
        if (rounds != 7 && rounds != 10) return fail(s->ctx, ISING_E_INVALID, "rounds must be 7 or 10");
        s->rounds = rounds;
    }
    return ISING_OK;
}

extern "C" int ising_sim_randomize(ising_sim* s) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s) return fail(nullptr, ISING_E_INVALID, "sim is NULL");
    ising_ctx* ctx = s->ctx;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    count_launch(s, launch_init_random(s->d_spins, s->lay, (uint32_t)s->seed,
                                       (uint32_t)(s->seed >> 32),
                                       (uint32_t)(s->replica_offset / 32), ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return ISING_OK;
}

extern "C" int ising_sim_set_state(ising_sim* s, const uint8_t* state) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s || !state) return fail(s ? s->ctx : nullptr, ISING_E_INVALID, "sim/state is NULL");
    ising_ctx* ctx = s->ctx;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    void* dv = nullptr;
    CUDA_TRY(ctx, ctx_scratch(ctx, 0, s->lay.nvars, &dv));
    uint8_t* d = (uint8_t*)dv;
    cudaError_t e = cudaMemcpyAsync(d, state, s->lay.nvars, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) {
        count_launch(s, launch_init_broadcast(s->d_spins, s->lay, d, ctx->stream));
        e = cudaStreamSynchronize(ctx->stream);
    }
    CUDA_TRY(ctx, e);
    return ISING_OK;
}

extern "C" int ising_sim_set_states(ising_sim* s, const uint8_t* states) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s || !states) return fail(s ? s->ctx : nullptr, ISING_E_INVALID, "sim/states is NULL");
    ising_ctx* ctx = s->ctx;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const size_t bytes = (size_t)s->E * s->lay.nvars;
    void* dv = nullptr;
    CUDA_TRY(ctx, ctx_scratch(ctx, 0, bytes, &dv));
    uint8_t* d = (uint8_t*)dv;
    cudaError_t e = cudaMemcpyAsync(d, states, bytes, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) {
        count_launch(s, launch_pack_states(s->d_spins, s->lay, d, s->E, ctx->stream));
        e = cudaStreamSynchronize(ctx->stream);
    }
    CUDA_TRY(ctx, e);
    return ISING_OK;
}

// dE of the uphill classes in units of |J|: stencil 2D {4, 8}, 3D {4, 8, 12}
void fill_thresholds(const HostGraph& h, double beta, int K, MscThresholds* th) {
    const int dim = h.kind == ISING_KIND_STENCIL3D ? 3 : 2;
    memset(th, 0, sizeof *th);
    for (int c = 0; c < dim; ++c) {
        const double de = 4.0 * (c + 1) * h.jabs;
        const double p = exp(-beta * de);
        const double scaled = ldexp(p, K + 32);
        const uint64_t tmax = (1ull << (K + 32)) - 1;
        uint64_t T;
        if (!(scaled >= 0.0)) T = 0;  // NaN beta: never accept uphill
        else if (scaled >= (double)tmax) T = tmax;
        else T = (uint64_t)floor(scaled);
        for (int pl = 0; pl < K; ++pl)
            th->plane[c][pl] = ((T >> (K + 31 - pl)) & 1ull) ? 0xFFFFFFFFu : 0u;
        th->low[c] = (uint32_t)(T & 0xFFFFFFFFull);
    }
}

// T = floor(exp(-beta dE) 2^(K+32)) clipped to K+32 bits; NaN -> 0 (never accept uphill)
uint64_t threshold64(double beta, double de, int K) {
    const double scaled = ldexp(exp(-beta * de), K + 32);
    const uint64_t tmax = (1ull << (K + 32)) - 1;
    if (!(scaled >= 0.0)) return 0;
    if (scaled >= (double)tmax) return tmax;
    return (uint64_t)floor(scaled);
}

// uphill classes of a degree-d site: n_sat = d/2+1 .. d, dE = 2|J|(2 n_sat - d)
void fill_gen_thresholds(double jabs, double beta, int K, uint32_t deg, GenThresholds* th) {
    memset(th, 0, sizeof *th);
    const uint32_t cmin = deg / 2 + 1, ncls = deg - deg / 2;
    for (uint32_t j = 0; j < ncls && j < (uint32_t)GEN_MAX_CLS; ++j) {
        const int cls = 2 * (int)(cmin + j) - (int)deg;
        const uint64_t T = threshold64(beta, 2.0 * jabs * (double)cls, K);
        for (int pl = 0; pl < K; ++pl)
            th->plane[j][pl] = ((T >> (K + 31 - pl)) & 1ull) ? 0xFFFFFFFFu : 0u;
        th->low[j] = (uint32_t)(T & 0xFFFFFFFFull);
    }
}

static int sim_one_sweep_general(ising_sim* s, double beta) {
    ising_ctx* ctx = s->ctx;
    const ising_graph* g = s->g;
    const HostGraph& h = g->h;
    GenSweepArgs a;
    a.spins = s->d_spins;
    a.W = s->lay.W;
    a.sweep = (uint32_t)s->sweep_counter;
    a.key0 = (uint32_t)s->seed;
    a.key1 = (uint32_t)(s->seed >> 32);
    a.gw0 = (uint32_t)(s->replica_offset / 32);
    a.planes = s->planes;
    a.rounds = s->rounds;
    a.tables.plane = s->perbeta ? s->d_tplane : nullptr;
    a.tables.low = s->perbeta ? s->d_tlow : nullptr;
    memset(&a.th, 0, sizeof a.th);
    int launches = 0;
    for (int c = 0; c < g->gen_ncolors; ++c)
        for (size_t k = 0; k < g->gen_groups.size(); ++k) {
            if (g->gen_group_color[k] != c) continue;
            const GenGroup& gg = g->gen_groups[k];
            // (an isolated site has dE = 0 and, as in the reference's dE <= 0 rule, always flips)
            if (!s->perbeta) fill_gen_thresholds(h.jabs, beta, s->planes, gg.deg, &a.th);
            const int n = launch_sweep_general(a, gg, ctx->stream);
            if (n < 0) return fail(ctx, ISING_E_CUDA, "general sweep launch failed: %s",
                                   cudaGetErrorString(cudaGetLastError()));
            launches += n;
        }
    count_launch(s, launches);
    s->stats.sweep_kernel_launches += (uint64_t)launches;
    s->sweep_counter++;
    s->stats.sweeps++;
    s->stats.flip_attempts += s->E * h.nvars;
    return ISING_OK;
}

static int sim_one_sweep_real(ising_sim* s, double beta) {
    ising_ctx* ctx = s->ctx;
    const ising_graph* g = s->g;
    RealSweepArgs a;
    a.spins = s->d_spins;
    a.row = g->d_row32;
    a.nbr = g->d_nbr32;
    a.jf = g->d_jf;
    a.biasf = g->d_biasf;
    a.W = s->lay.W;
    a.beta = (float)beta;
    a.beta_slots = s->perbeta ? s->d_t64 : nullptr;   // real sims keep the betas themselves in d_t64
    a.slot_of_replica = s->perbeta ? s->d_slot : nullptr;
    a.sweep = (uint32_t)s->sweep_counter;
    a.key0 = (uint32_t)s->seed;
    a.key1 = (uint32_t)(s->seed >> 32);
    a.gw0 = (uint32_t)(s->replica_offset / 32);
    a.rounds = s->rounds;
    int launches = 0;
    for (int c = 0; c < g->h.ncolors; ++c) {
        a.sites = g->d_csites + g->color_off[c];
        a.count = g->color_off[c + 1] - g->color_off[c];
        const int n = launch_sweep_real(a, ctx->stream);
        if (n < 0) return fail(ctx, ISING_E_CUDA, "real-coupling sweep launch failed: %s",
                               cudaGetErrorString(cudaGetLastError()));
        launches += n;
    }
    count_launch(s, launches);
    s->stats.sweep_kernel_launches += (uint64_t)launches;
    s->sweep_counter++;
    s->stats.sweeps++;
    s->stats.flip_attempts += s->E * g->h.nvars;
    return ISING_OK;
}

// f64 energies of a real-coupling sim into d_out[e * estride + eoff]
static int sim_energy_real(ising_sim* s, double* d_tmp /* [32 W] */) {
    ising_ctx* ctx = s->ctx;
    const ising_graph* g = s->g;
    CUDA_TRY(ctx, cudaMemsetAsync(d_tmp, 0, (size_t)s->lay.W * 32 * sizeof(double), ctx->stream));
    const int n = launch_energy_real(s->d_spins, s->lay.nvars, s->lay.W, g->d_row32, g->d_nbr32,
                                     g->d_jv, g->d_bias, d_tmp, ctx->stream);
    if (n < 0) return fail(ctx, ISING_E_CUDA, "energy launch failed");
    count_launch(s, n);
    return ISING_OK;
}

// Thresholds of the (spin, n_sat) classes of a torus or a strip in a field: dE = 2|J|(2 n_sat - 2 dim)
// + 2 h sigma, evaluated left to right in f64 (at h = 0 the doubles fill_thresholds and the strip's plain
// thresholds use); dE <= 0 flips always.
void fill_field_thresholds(double jabs, double field, int dim, double beta, int K, FieldThresholds* th) {
    memset(th, 0, sizeof *th);
    for (int sp = 0; sp < 2; ++sp)
        for (int n = 0; n <= 2 * dim; ++n) {
            const double sigma = sp ? 1.0 : -1.0;
            const double de = 2.0 * jabs * (double)(2 * n - 2 * dim) + 2.0 * field * sigma;
            if (!(de > 0.0)) continue;
            const uint64_t T = threshold64(beta, de, K);
            th->up[sp][n] = 0xFFFFFFFFu;
            for (int pl = 0; pl < K; ++pl) th->plane[pl][sp][n] = ((T >> (K + 31 - pl)) & 1ull) ? 0xFFFFFFFFu : 0u;
            th->low[sp][n] = (uint32_t)(T & 0xFFFFFFFFull);
        }
}

static int sim_one_sweep_field(ising_sim* s, double beta) {
    ising_ctx* ctx = s->ctx;
    const HostGraph& h = s->g->h;
    SweepArgs a;
    memset(&a, 0, sizeof a);
    a.spins = s->d_spins;
    a.jmask = s->g->d_jmask;
    a.lay = s->lay;
    a.sweep = (uint32_t)s->sweep_counter;
    a.key0 = (uint32_t)s->seed;
    a.key1 = (uint32_t)(s->seed >> 32);
    a.gw0 = (uint32_t)(s->replica_offset / 32);
    a.antiferro = h.uniform_antiferro ? 0xFFFFFFFFu : 0u;
    a.planes = s->planes;
    a.rounds = s->rounds;
    FieldThresholds th;
    fill_field_thresholds(h.jabs, h.field, h.kind == ISING_KIND_STENCIL3D ? 3 : 2, beta, s->planes, &th);
    const int n = launch_sweep_field(a, th, ctx->stream);
    if (n < 0) return fail(ctx, ISING_E_CUDA, "field sweep launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    count_launch(s, n);
    s->stats.sweep_kernel_launches += (uint64_t)n;
    s->sweep_counter++;
    s->stats.sweeps++;
    s->stats.flip_attempts += s->E * h.nvars;
    return ISING_OK;
}

// satisfied bonds into nsat[W * 32] and up spins into up[W * 32] (both zeroed by the caller)
static int sim_count_field(ising_sim* s, unsigned long long* nsat, unsigned long long* up) {
    ising_ctx* ctx = s->ctx;
    const int n = launch_nsat_stencil(s->d_spins, s->g->d_jmask, s->lay, s->g->h.uniform_antiferro ? 0xFFFFFFFFu : 0u,
                                      nsat, ctx->stream);
    if (n < 0) return fail(ctx, ISING_E_CUDA, "energy launch failed");
    count_launch(s, n);
    count_launch(s, launch_count_up(s->d_spins, s->lay, up, ctx->stream));
    return ISING_OK;
}

static int sim_one_sweep_basic(ising_sim* s, double beta, unsigned long long* nsat_out = nullptr,
                               uint32_t nsat_copies = 1) {
    if (s->real) return sim_one_sweep_real(s, beta);
    if (s->field) return sim_one_sweep_field(s, beta);
    if (s->general) return sim_one_sweep_general(s, beta);
    ising_ctx* ctx = s->ctx;
    const HostGraph& h = s->g->h;
    SweepArgs a;
    a.spins = s->d_spins;
    a.jmask = s->g->d_jmask;
    a.jmask8 = s->g->d_jmask8;
    a.sm_count = ctx->sm_count;
    a.lay = s->lay;
    a.sweep = (uint32_t)s->sweep_counter;
    a.key0 = (uint32_t)s->seed;
    a.key1 = (uint32_t)(s->seed >> 32);
    a.gw0 = (uint32_t)(s->replica_offset / 32);
    a.antiferro = h.uniform_antiferro ? 0xFFFFFFFFu : 0u;
    a.planes = s->planes;
    a.rounds = s->rounds;
    if (s->perbeta) memset(&a.th, 0, sizeof a.th);
    else fill_thresholds(h, beta, s->planes, &a.th);
    a.nsat_out = nsat_out;
    a.nsat_copies = nsat_copies;
    a.nsat_stride = s->lay.W * 32;
    a.tplane = s->perbeta ? s->d_tplane : nullptr;
    a.tlow = s->perbeta ? s->d_tlow : nullptr;
    const int n = launch_sweep_stencil(a, ctx->stream);
    if (n < 0) return fail(ctx, ISING_E_CUDA, "sweep launch failed: %s",
                           cudaGetErrorString(cudaGetLastError()));
    count_launch(s, n);
    s->stats.sweep_kernel_launches += (uint64_t)n;
    s->sweep_counter++;
    s->stats.sweeps++;
    s->stats.flip_attempts += s->E * h.nvars;
    return ISING_OK;
}

// The non-basic part of a timestep (ising_sim_set_moves): passes of two-spin edge moves over the
// classes of the strong edge colouring, then the worm moves.  t = index of the timestep.
static int sim_non_basic_moves(ising_sim* s, double beta, uint64_t t) {
    ising_ctx* ctx = s->ctx;
    const ising_graph* g = s->g;
    const MoveGraph mg{g->d_row32, g->d_nbr32, g->d_jf, g->d_biasf};
    int launches = 0;
    // all |J| equal, no bias, <= 15 outer bonds per pair: the bit-sliced kernel with exact integer
    // thresholds (importance sampling weights every bond alike there); else float local fields
    const ising_graph::EdgeGen& eg = g->edge_gen[s->general ? 0 : 1];
    static const bool force_float = getenv("ISING_EDGE_FLOAT") != nullptr;   // A/B knob
    const bool bitsliced = eg.usable && !s->real && !force_float;
    for (uint32_t pass = 0; bitsliced && pass < s->mv.edge_passes; ++pass) {
        GenSweepArgs ga;
        ga.spins = s->d_spins;
        ga.W = s->lay.W;
        ga.sweep = (uint32_t)t;
        ga.key0 = (uint32_t)s->seed;
        ga.key1 = (uint32_t)(s->seed >> 32);
        ga.gw0 = (uint32_t)(s->replica_offset / 32);
        ga.planes = s->planes;
        ga.rounds = s->rounds;
        ga.tables.plane = nullptr;
        ga.tables.low = nullptr;
        uint32_t th_deg = 0xFFFFFFFFu;
        for (const EdgeGroup& gr : eg.groups) {
            if (gr.deg != th_deg) {
                fill_gen_thresholds(g->h.jabs, beta, s->planes, gr.deg, &ga.th);
                th_deg = gr.deg;
            }
            const int n = launch_edge_general(ga, gr, pass, ctx->stream);
            if (n < 0) return fail(ctx, ISING_E_CUDA, "edge-move launch failed: %s",
                                   cudaGetErrorString(cudaGetLastError()));
            launches += n;
        }
    }
    for (uint32_t pass = 0; !bitsliced && pass < s->mv.edge_passes; ++pass)
        for (size_t c = 0; c + 1 < g->medge_off.size(); ++c) {
            EdgeMoveArgs a;
            a.spins = s->d_spins;
            a.lay = s->lay;
            a.g = mg;
            const uint32_t o = g->medge_off[c];
            a.ea = g->d_mea + o;
            a.eb = g->d_meb + o;
            a.eid = g->d_meid + o;
            a.wrel = s->mv.edge_importance ? g->d_mwrel + o : nullptr;
            a.count = g->medge_off[c + 1] - o;
            a.beta = (float)beta;
            a.sweep = (uint32_t)t;
            a.key0 = (uint32_t)s->seed;
            a.key1 = (uint32_t)(s->seed >> 32);
            a.gw0 = (uint32_t)(s->replica_offset / 32);
            a.pass = pass;
            a.rounds = s->rounds;
            const int n = launch_edge_moves(a, ctx->stream);
            if (n < 0) return fail(ctx, ISING_E_CUDA, "edge-move launch failed: %s",
                                   cudaGetErrorString(cudaGetLastError()));
            launches += n;
        }
    if (s->mv.worms) {
        WormArgs a;
        a.spins = s->d_spins;
        a.lay = s->lay;
        a.g = mg;
        a.E = s->E;
        a.replica_offset = s->replica_offset;
        a.nworms = s->mv.worms;
        a.worm0 = 0;
        a.len = s->mv.worm_len;
        a.beta = (float)beta;
        a.sweep = (uint32_t)t;
        a.key0 = (uint32_t)s->seed;
        a.key1 = (uint32_t)(s->seed >> 32);
        a.rounds = s->rounds;
        const int n = launch_worm_moves(a, ctx->stream);
        if (n < 0) return fail(ctx, ISING_E_CUDA, "worm-move launch failed: %s",
                               cudaGetErrorString(cudaGetLastError()));
        launches += n;
    }
    count_launch(s, launches);
    s->stats.edge_attempts += (uint64_t)s->mv.edge_passes * s->g->h.nedges * s->E;
    s->stats.worm_attempts += (uint64_t)s->mv.worms * s->E;
    return ISING_OK;
}

// One timestep: the colour-class sweep and, when ising_sim_set_moves asked for them, the non-basic
// moves.  nsat_out (fused per-sweep energy accumulation) only without non-basic moves.
static int sim_one_sweep(ising_sim* s, double beta, unsigned long long* nsat_out = nullptr,
                         uint32_t nsat_copies = 1) {
    if (!s->moves_active) return sim_one_sweep_basic(s, beta, nsat_out, nsat_copies);
    const uint64_t t = s->sweep_counter;
    if (s->mv.spin_sweeps) {
        const int rc = sim_one_sweep_basic(s, beta);
        if (rc) return rc;
    } else {
        s->sweep_counter++;
        s->stats.sweeps++;
    }
    return sim_non_basic_moves(s, beta, t);
}

extern "C" int ising_sim_set_moves(ising_sim* s, const ising_moves* mv) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s) return fail(nullptr, ISING_E_INVALID, "sim is NULL");
    ising_ctx* ctx = s->ctx;
    if (!mv) {   // back to the default timestep
        s->moves_active = false;
        return ISING_OK;
    }
    if (mv->struct_size != sizeof(ising_moves))
        return fail(ctx, ISING_E_INVALID, "ising_moves.struct_size mismatch (%u != %zu)", mv->struct_size,
                    sizeof(ising_moves));
    if (mv->spin_sweeps > 1)
        return fail(ctx, ISING_E_UNSUPPORTED, "spin_sweeps must be 0 or 1 (a timestep holds at most one colour-class sweep)");
    if (mv->worms && (mv->worm_len < 1 || mv->worm_len > (uint32_t)WORM_MAX_LEN))
        return fail(ctx, ISING_E_INVALID, "worm_len must be 1..%d", WORM_MAX_LEN);
    if (mv->edge_passes > 255) return fail(ctx, ISING_E_INVALID, "edge_passes must be <= 255");
    const bool non_basic = mv->edge_passes || mv->worms;
    if (non_basic && s->field)
        return fail(ctx, ISING_E_UNSUPPORTED, "edge and worm moves do not take a field (a torus in a field runs single-spin sweeps)");
    if (non_basic && s->perbeta)
        return fail(ctx, ISING_E_UNSUPPORTED, "non-basic moves run at one beta per timestep, not at per-experiment betas");
    if (non_basic) {
        CUDA_TRY(ctx, cudaSetDevice(ctx->device));
        int rc = ensure_moves_on_device(ctx, const_cast<ising_graph*>(s->g));
        if (rc == ISING_OK && mv->edge_passes)
            rc = ensure_edge_general_on_device(ctx, const_cast<ising_graph*>(s->g), !s->general);
        if (rc) return rc;
    }
    s->mv = *mv;
    s->moves_active = non_basic || mv->spin_sweeps == 0;
    return ISING_OK;
}

// Launch-bound sizes: a whole chunk of sweeps in one cooperative launch.  Returns 1 when done
// that way, 0 when the caller should fall back to per-phase launches, < 0 on error (rc in *err).
// counts_last (per-replica betas only): hist[e] receives the counts of the LAST sweep of the chunk
// (k_sweep_stencil_cluster<ACC, PERBETA>) instead of a history of all sweeps.
static int sim_sweeps_coop(ising_sim* s, const double* betas, uint64_t nt, unsigned long long* hist,
                           int* err, uint32_t hist_stride = 0, bool counts_last = false) {
    if (hist_stride == 0) hist_stride = s->lay.W * 32;   // words of history per sweep
    *err = ISING_OK;
    if (s->general || s->real || s->field || s->moves_active || nt == 0) return 0;
    if (s->perbeta ? (s->planes != 6 || (hist != nullptr) != counts_last) : counts_last) return 0;
    if ((uint64_t)s->lay.halfN * s->lay.W > (1ull << 19)) return 0;  // big enough to fill the GPU
    ising_ctx* ctx = s->ctx;
    const HostGraph& h = s->g->h;
    // per-sweep thresholds (one beta per sweep); per-replica betas use the sim's device tables
    std::vector<MscThresholds> th(s->perbeta ? 0 : nt);
    for (uint64_t t = 0; t < th.size(); ++t) fill_thresholds(h, betas[t], s->planes, &th[t]);
    void* dv = nullptr;
    cudaError_t e = ctx_scratch(ctx, 3, std::max<size_t>(1, th.size()) * sizeof(MscThresholds), &dv);
    if (e == cudaSuccess && !th.empty())
        e = cudaMemcpyAsync(dv, th.data(), nt * sizeof(MscThresholds), cudaMemcpyHostToDevice, ctx->stream);
    if (e != cudaSuccess) {
        *err = fail(ctx, ISING_E_CUDA, "threshold table upload: %s", cudaGetErrorString(e));
        return -1;
    }
    SweepArgs a;
    a.spins = s->d_spins;
    a.jmask = s->g->d_jmask;
    a.jmask8 = s->g->d_jmask8;
    a.sm_count = ctx->sm_count;
    a.lay = s->lay;
    a.sweep = (uint32_t)s->sweep_counter;
    a.key0 = (uint32_t)s->seed;
    a.key1 = (uint32_t)(s->seed >> 32);
    a.gw0 = (uint32_t)(s->replica_offset / 32);
    a.antiferro = h.uniform_antiferro ? 0xFFFFFFFFu : 0u;
    a.planes = s->planes;
    a.rounds = s->rounds;
    a.nsat_out = nullptr;
    a.tplane = s->perbeta ? s->d_tplane : nullptr;
    a.tlow = s->perbeta ? s->d_tlow : nullptr;
    memset(&a.th, 0, sizeof a.th);
    // smallest lattices: one thread-block cluster, hardware barrier between the phases
    static const bool no_cluster = getenv("ISING_NO_CLUSTER") != nullptr;  // A/B knob
    int rc = 0;
    if (!no_cluster) {
        rc = launch_sweeps_stencil_cluster(a, (const MscThresholds*)dv, (uint32_t)nt, hist, hist_stride,
                                           ctx->stream);
        if (rc < 0) {
            cudaGetLastError();
            rc = 0;
        }
    }
    // Above the cluster limit one launch per colour phase wins: with programmatic dependent launch
    // a phase of 64^3 x 128 replicas takes 5.8 us, the cooperative kernel (two grid barriers per
    // sweep) 13.6 us.  ISING_COOP=1 keeps the cooperative kernel reachable for A/B runs.
    static const bool use_coop = getenv("ISING_COOP") != nullptr;
    if (rc == 0 && use_coop && !s->perbeta && !(hist && s->lay.W > 8))
        rc = launch_sweeps_stencil_coop(a, (const MscThresholds*)dv, (uint32_t)nt, hist, hist_stride,
                                        ctx->stream);
    if (rc < 0) {
        cudaGetLastError();
        return 0;  // e.g. too many blocks to be co-resident: use the per-phase launches
    }
    if (rc == 0) return 0;
    // (the pageable host table has been staged by the time cudaMemcpyAsync returned; per-replica
    // betas upload nothing)  Launch errors of the chunk surface here when a table was used.
    if (!th.empty()) {
        e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) {
            *err = fail(ctx, ISING_E_CUDA, "multi-sweep launch: %s", cudaGetErrorString(e));
            return -1;
        }
    }
    count_launch(s, 1);
    s->stats.sweep_kernel_launches += 1;
    s->sweep_counter += nt;
    s->stats.sweeps += nt;
    s->stats.flip_attempts += nt * s->E * h.nvars;
    return 1;
}

// n_sat per experiment into s->d_counts (zeroed first)
int sim_count_nsat(ising_sim* s, unsigned long long* d_counts, bool zero_first) {
    ising_ctx* ctx = s->ctx;
    const HostGraph& h = s->g->h;
    if (zero_first)
        CUDA_TRY(ctx, cudaMemsetAsync(d_counts, 0, (size_t)s->lay.W * 32 * sizeof(unsigned long long),
                                      ctx->stream));
    if (s->general) {
        const int n = launch_nsat_general(s->d_spins, s->lay.nvars, s->lay.W, s->g->d_row32,
                                          s->g->d_nbr32, s->g->d_anti8, d_counts, ctx->stream);
        if (n < 0) return fail(ctx, ISING_E_CUDA, "energy launch failed");
        count_launch(s, n);
        return ISING_OK;
    }
    const int n = launch_nsat_stencil(s->d_spins, s->g->d_jmask, s->lay,
                                      h.uniform_antiferro ? 0xFFFFFFFFu : 0u, d_counts,
                                      ctx->stream);
    if (n < 0) return fail(ctx, ISING_E_CUDA, "energy launch failed");
    count_launch(s, n);
    return ISING_OK;
}

// The sweeps of one tempering chunk (per-replica betas), enqueued like sim_enqueue_sweeps; when the
// lattice runs inside one thread-block cluster the last sweep also leaves the satisfied-bond counts
// of the final configuration in d_counts (zeroed by the caller) and *counted is set: the swap cycle
// then needs no separate count pass.  ISING_PT_NO_FUSED_COUNTS=1 is the A/B knob.
int sim_enqueue_sweeps_counting(ising_sim* s, uint64_t nsweeps, unsigned long long* d_counts, bool* counted) {
    *counted = false;
    static const bool off = getenv("ISING_PT_NO_FUSED_COUNTS") != nullptr;
    if (off || !s->perbeta || nsweeps == 0) return sim_enqueue_sweeps(s, nullptr, nsweeps);
    if (nsweeps > 4096) {
        const int rc = sim_enqueue_sweeps(s, nullptr, nsweeps - 4096);
        if (rc) return rc;
        nsweeps = 4096;
    }
    if (s->sweep_counter + nsweeps > 0xFFFFFFFFull) return sim_enqueue_sweeps(s, nullptr, nsweeps);  // reports the wrap
    int err = ISING_OK;
    const int done = sim_sweeps_coop(s, nullptr, nsweeps, d_counts, &err, 0, true);
    if (done < 0) return err;
    if (done) {
        *counted = true;
        return ISING_OK;
    }
    return sim_enqueue_sweeps(s, nullptr, nsweeps);
}

// nsweeps sweeps enqueued on the context's stream, no host wait and no timing (the tempering
// loop synchronises once per swap step, when it reads the energies)
int sim_enqueue_sweeps(ising_sim* s, const double* betas, uint64_t nsweeps) {
    // Philox counter word 2 is the 32-bit sweep index: refuse to wrap (a wrapped counter would
    // silently replay the random streams of sweeps 0, 1, ...)
    if (s->sweep_counter + nsweeps > 0xFFFFFFFFull || s->sweep_counter + nsweeps < nsweeps)
        return fail(s->ctx, ISING_E_UNSUPPORTED,
                    "sweep counter would pass 2^32 (%llu done, %llu requested): start a new simulation or seed",
                    (unsigned long long)s->sweep_counter, (unsigned long long)nsweeps);
    uint64_t t = 0;
    while (t < nsweeps) {
        const uint64_t nt = std::min<uint64_t>(4096, nsweeps - t);
        int err = ISING_OK;
        const int done = (betas || s->perbeta) ? sim_sweeps_coop(s, betas ? betas + t : nullptr, nt, nullptr, &err) : 0;
        if (done < 0) return err;
        if (done) { t += nt; continue; }
        for (uint64_t k = 0; k < nt; ++k) {
            const int rc = sim_one_sweep(s, betas ? betas[t + k] : 0.0);
            if (rc) return rc;
        }
        t += nt;
    }
    return ISING_OK;
}

extern "C" int ising_sim_sweeps(ising_sim* s, const double* betas, uint64_t nsweeps,
                                double* energies_per_sweep) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s) return fail(nullptr, ISING_E_INVALID, "sim is NULL");
    if (s->perbeta ? betas != nullptr : (nsweeps && !betas))
        return fail(s->ctx, ISING_E_INVALID,
                    s->perbeta ? "sim runs at per-experiment betas (ising_sim_set_betas): pass betas = NULL"
                               : "betas is NULL");
    ising_ctx* ctx = s->ctx;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const HostGraph& h = s->g->h;
    const uint64_t E = s->E;
    const int mult = s->general ? 1 : 2;
    if (s->sweep_counter + nsweeps > 0xFFFFFFFFull || s->sweep_counter + nsweeps < nsweeps)
        return fail(ctx, ISING_E_UNSUPPORTED,
                    "sweep counter would pass 2^32 (%llu done, %llu requested): start a new simulation or seed",
                    (unsigned long long)s->sweep_counter, (unsigned long long)nsweeps);
    if (!energies_per_sweep) {
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
        const int rc0 = sim_enqueue_sweeps(s, betas, nsweeps);
        if (rc0) return rc0;
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
        float ms = 0.f;
        CUDA_TRY(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        s->stats.sweep_device_ms += ms;
        s->stats.sweep_kernel_ms += ms;
        return ISING_OK;
    }
    // per-sweep energies: integer n_sat history on the device, converted and transposed to
    // double[E, nsweeps] there, one D2H per chunk
    const uint64_t chunk_max = 2048;
    const size_t cw = (size_t)s->lay.W * 32;
    // lattices: several copies of a sweep's counters, so that the blocks of the accumulating
    // phase do not serialise their atomics on W * 32 addresses (SweepArgs::nsat_copies)
    const uint32_t copies = (s->general || s->real || s->field) ? 1u
                            : (uint32_t)std::max<size_t>(1, std::min<size_t>(16, 4096 / std::max<size_t>(cw, 1)));
    const size_t hstride = cw * copies;   // words of history per sweep
    unsigned long long* d_hist = nullptr;
    double* d_out = nullptr;
    void* sp = nullptr;
    // a field adds the up-spin counts of every sweep behind the satisfied-bond history
    const size_t hist_words = hstride * std::min(chunk_max, nsweeps);
    CUDA_TRY(ctx, ctx_scratch(ctx, 1, hist_words * (s->field ? 2 : 1) * sizeof(unsigned long long), &sp));
    d_hist = (unsigned long long*)sp;
    unsigned long long* d_up_hist = d_hist + hist_words;
    CUDA_TRY(ctx, ctx_scratch(ctx, 2, (size_t)E * std::min(chunk_max, nsweeps) * sizeof(double), &sp));
    d_out = (double*)sp;
    cudaError_t e = cudaSuccess;
    int rc = ISING_OK;
    for (uint64_t t0 = 0; t0 < nsweeps && rc == ISING_OK; t0 += chunk_max) {
        const uint64_t nt = std::min(chunk_max, nsweeps - t0);
        cudaEventRecord(ctx->ev0, ctx->stream);
        cudaMemsetAsync(d_hist, 0, hstride * nt * sizeof(unsigned long long), ctx->stream);
        if (s->field) cudaMemsetAsync(d_up_hist, 0, hstride * nt * sizeof(unsigned long long), ctx->stream);
        // the second colour phase of every sweep adds its post-flip satisfied-bond counts
        // into that sweep's slot of the history (fused, no separate energy pass)
        int coop_err = ISING_OK;
        const int coop = betas ? sim_sweeps_coop(s, betas + t0, nt, d_hist, &coop_err, (uint32_t)hstride) : 0;
        if (coop < 0) rc = coop_err;
        for (uint64_t t = 0; coop == 0 && t < nt && rc == ISING_OK; ++t) {
            rc = sim_one_sweep(s, betas ? betas[t0 + t] : 0.0, d_hist + t * hstride, copies);
            if (rc == ISING_OK && s->real) {
                rc = sim_energy_real(s, reinterpret_cast<double*>(d_hist + t * cw));
            } else if (rc == ISING_OK && s->field) {
                rc = sim_count_field(s, d_hist + t * cw, d_up_hist + t * cw);
            } else if (rc == ISING_OK && s->moves_active && !s->general) {
                // the non-basic moves ran after the sweep: count the satisfied bonds of the result
                const int n = launch_nsat_stencil(s->d_spins, s->g->d_jmask, s->lay,
                                                  h.uniform_antiferro ? 0xFFFFFFFFu : 0u,
                                                  d_hist + t * hstride, ctx->stream);
                if (n < 0) rc = fail(ctx, ISING_E_CUDA, "energy launch failed");
                else count_launch(s, n);
            } else if (rc == ISING_OK && s->general) {  // no fused accumulation on general graphs
                const int n = launch_nsat_general(s->d_spins, s->lay.nvars, s->lay.W, s->g->d_row32,
                                                  s->g->d_nbr32, s->g->d_anti8, d_hist + t * cw,
                                                  ctx->stream);
                if (n < 0) rc = fail(ctx, ISING_E_CUDA, "energy launch failed");
                else count_launch(s, n);
            }
        }
        if (rc == ISING_OK && s->field)
            count_launch(s, launch_energy_field(d_hist, d_up_hist, E, cw, nt, h.jabs, h.nedges, h.field, h.nvars, d_out,
                                                nt, 0, ctx->stream));
        else if (rc == ISING_OK && s->real)
            count_launch(s, launch_transpose_hist_f64(reinterpret_cast<double*>(d_hist), E, cw, nt,
                                                      d_out, ctx->stream));
        else if (rc == ISING_OK)
            count_launch(s, launch_energy_from_hist(d_hist, E, cw, nt, h.jabs, h.nedges, mult,
                                                    d_out, ctx->stream, copies));
        cudaEventRecord(ctx->ev1, ctx->stream);
        if (rc != ISING_OK) break;
        // rows [e][t0 .. t0 + nt) straight into the caller's double[E, nsweeps] (strided copy)
        e = copy_rows_d2h(energies_per_sweep + t0, (size_t)nsweeps * sizeof(double), d_out,
                          (size_t)nt * sizeof(double), (size_t)nt * sizeof(double), E, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) { rc = fail(ctx, ISING_E_CUDA, "energy read-back: %s", cudaGetErrorString(e)); break; }
        float ms = 0.f;
        cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
        s->stats.sweep_device_ms += ms;
    }
    return rc;
}

// current energies of all experiments into d_out[e * estride + eoff] (device)
int sim_energies_to_device(ising_sim* s, double* d_out, uint64_t estride, uint64_t eoff) {
    ising_ctx* ctx = s->ctx;
    const HostGraph& h = s->g->h;
    if (s->real) {
        double* tmp = reinterpret_cast<double*>(s->d_counts);  // same size as the u64 counters
        const int rc = sim_energy_real(s, tmp);
        if (rc) return rc;
        count_launch(s, launch_copy_strided_f64(tmp, s->E, d_out, estride, eoff, ctx->stream));
        return ISING_OK;
    }
    if (s->field) {
        const size_t cw = (size_t)s->lay.W * 32;
        CUDA_TRY(ctx, cudaMemsetAsync(s->d_counts, 0, 2 * cw * sizeof(unsigned long long), ctx->stream));
        const int rc = sim_count_field(s, s->d_counts, s->d_counts + cw);
        if (rc) return rc;
        count_launch(s, launch_energy_field(s->d_counts, s->d_counts + cw, s->E, cw, 1, h.jabs, h.nedges, h.field,
                                            h.nvars, d_out, estride, eoff, ctx->stream));
        return ISING_OK;
    }
    const int rc = sim_count_nsat(s, s->d_counts);
    if (rc) return rc;
    count_launch(s, launch_energy_from_nsat(s->d_counts, s->E, h.jabs, h.nedges, s->general ? 1 : 2,
                                            d_out, estride, eoff, ctx->stream));
    return ISING_OK;
}

extern "C" int ising_sim_get_energies(ising_sim* s, double* energies) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s || !energies) return fail(s ? s->ctx : nullptr, ISING_E_INVALID, "sim/energies is NULL");
    ising_ctx* ctx = s->ctx;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    void* dv = nullptr;
    CUDA_TRY(ctx, ctx_scratch(ctx, 2, s->E * sizeof(double), &dv));
    double* d_out = (double*)dv;
    const int rc = sim_energies_to_device(s, d_out, 1, 0);
    if (rc) return rc;
    CUDA_TRY(ctx, cudaMemcpyAsync(energies, d_out, s->E * sizeof(double), cudaMemcpyDeviceToHost,
                                  ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return ISING_OK;
}

// Accepted flips of ONE timestep at beta, per experiment: the packed state is copied, the timestep
// runs, and the positional popcount of before ^ after counts the spins that changed - every site
// is attempted exactly once per colour-class sweep, so with the default timestep this is the number
// of accepted single-spin flips (SURVEY 5.5).  Costs nothing on the sweep kernels' own path.
extern "C" int ising_sim_step_acceptance(ising_sim* s, double beta, uint64_t* changed) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s || !changed) return fail(s ? s->ctx : nullptr, ISING_E_INVALID, "sim/changed is NULL");
    if (s->perbeta) return fail(s->ctx, ISING_E_UNSUPPORTED, "per-experiment betas: use ising_sim_sweeps");
    ising_ctx* ctx = s->ctx;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    void* dv = nullptr;
    CUDA_TRY(ctx, ctx_scratch(ctx, 0, s->spins_bytes, &dv));
    uint32_t* before = (uint32_t*)dv;
    CUDA_TRY(ctx, cudaMemcpyAsync(before, s->d_spins, s->spins_bytes, cudaMemcpyDeviceToDevice, ctx->stream));
    const int rc = sim_enqueue_sweeps(s, &beta, 1);
    if (rc) return rc;
    const size_t cw = (size_t)s->lay.W * 32;
    count_launch(s, launch_xor_words(before, s->d_spins, s->spins_bytes / 4, ctx->stream));
    CUDA_TRY(ctx, cudaMemsetAsync(s->d_counts, 0, cw * sizeof(unsigned long long), ctx->stream));
    count_launch(s, launch_count_up(before, s->lay, s->d_counts, ctx->stream));
    std::vector<unsigned long long> h(cw);
    CUDA_TRY(ctx, cudaMemcpyAsync(h.data(), s->d_counts, cw * sizeof(unsigned long long), cudaMemcpyDeviceToHost,
                                  ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    for (uint64_t e = 0; e < s->E; ++e) changed[e] = h[e];
    return ISING_OK;
}

extern "C" int ising_sim_get_magnetization(ising_sim* s, double* m) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s || !m) return fail(s ? s->ctx : nullptr, ISING_E_INVALID, "sim/m is NULL");
    ising_ctx* ctx = s->ctx;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const size_t cw = (size_t)s->lay.W * 32;
    CUDA_TRY(ctx, cudaMemsetAsync(s->d_counts, 0, cw * sizeof(unsigned long long), ctx->stream));
    count_launch(s, launch_count_up(s->d_spins, s->lay, s->d_counts, ctx->stream));
    std::vector<unsigned long long> up(cw);
    CUDA_TRY(ctx, cudaMemcpyAsync(up.data(), s->d_counts, cw * sizeof(unsigned long long),
                                  cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    for (uint64_t e = 0; e < s->E; ++e)
        m[e] = 2.0 * (double)up[e] - (double)s->lay.nvars;
    return ISING_OK;
}

// bool[E, nvars] to host memory, staged through a device buffer in slabs of experiments
int sim_states_to_host(ising_sim* s, uint8_t* states) {
    ising_ctx* ctx = s->ctx;
    const uint64_t N = s->lay.nvars;
    const size_t bytes = (size_t)s->E * N;
    void* dv = nullptr;
    CUDA_TRY(ctx, ctx_scratch(ctx, 0, bytes, &dv));
    uint8_t* d = (uint8_t*)dv;
    count_launch(s, launch_unpack_states(s->d_spins, s->lay, d, s->E, N, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(states, d, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return ISING_OK;
}

extern "C" int ising_sim_get_states(ising_sim* s, uint8_t* states) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s || !states) return fail(s ? s->ctx : nullptr, ISING_E_INVALID, "sim/states is NULL");
    CUDA_TRY(s->ctx, cudaSetDevice(s->ctx->device));
    return sim_states_to_host(s, states);
}

extern "C" int ising_sim_get_packed(ising_sim* s, uint32_t* words) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s || !words) return fail(s ? s->ctx : nullptr, ISING_E_INVALID, "sim/words is NULL");
    ising_ctx* ctx = s->ctx;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const size_t n = (size_t)s->lay.nvars * s->lay.W;
    void* dv = nullptr;
    CUDA_TRY(ctx, ctx_scratch(ctx, 0, n * 4, &dv));
    uint32_t* d = (uint32_t*)dv;
    count_launch(s, launch_export_natural(s->d_spins, s->lay, d, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(words, d, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return ISING_OK;
}

// checkpoint support: the packed state in natural order plus the sweep counter are the whole
// state of a sim (the RNG is counter-based: seed + counter, nothing else to save)
extern "C" int ising_sim_set_packed(ising_sim* s, const uint32_t* words) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s || !words) return fail(s ? s->ctx : nullptr, ISING_E_INVALID, "sim/words is NULL");
    ising_ctx* ctx = s->ctx;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const size_t n = (size_t)s->lay.nvars * s->lay.W;
    void* dv = nullptr;
    CUDA_TRY(ctx, ctx_scratch(ctx, 0, n * 4, &dv));
    CUDA_TRY(ctx, cudaMemcpyAsync(dv, words, n * 4, cudaMemcpyHostToDevice, ctx->stream));
    count_launch(s, launch_import_natural(s->d_spins, s->lay, (const uint32_t*)dv, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return ISING_OK;
}

extern "C" int ising_sim_get_counter(const ising_sim* s, uint64_t* sweeps_done) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s || !sweeps_done) return fail(nullptr, ISING_E_INVALID, "sim/out is NULL");
    *sweeps_done = s->sweep_counter;
    return ISING_OK;
}

extern "C" int ising_sim_set_counter(ising_sim* s, uint64_t sweeps_done) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s) return fail(nullptr, ISING_E_INVALID, "sim is NULL");
    s->sweep_counter = sweeps_done;
    return ISING_OK;
}

extern "C" int ising_sim_get_stats(ising_sim* s, ising_sim_stats* out) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s || !out) return fail(nullptr, ISING_E_INVALID, "sim/out is NULL");
    *out = s->stats;
    return ISING_OK;
}

extern "C" int ising_sim_reset_stats(ising_sim* s) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s) return fail(nullptr, ISING_E_INVALID, "sim is NULL");
    s->stats = ising_sim_stats{};
    return ISING_OK;
}
