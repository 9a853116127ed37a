// C ABI: per-experiment inverse temperatures and classical parallel tempering (ising_pt_*).
#include "api_internal.h"
#include "pt_exp.h"

// ------------------------------------------------------------------------------------------
// per-experiment inverse temperatures and classical parallel tempering
// ------------------------------------------------------------------------------------------
extern "C" int ising_sim_set_betas(ising_sim* s, const double* betas) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s || !betas) return fail(s ? s->ctx : nullptr, ISING_E_INVALID, "sim/betas is NULL");
    ising_ctx* ctx = s->ctx;
    if (s->field) return fail(ctx, ISING_E_UNSUPPORTED, "per-experiment betas on a torus in a field are not supported");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const HostGraph& h = s->g->h;
    const uint32_t W = s->lay.W, E32 = 32 * W;
    if (s->real) {
        // float-field kernel: no tables, the betas themselves (f64 bit patterns) by replica bit
        std::vector<unsigned long long> bits(E32);
        std::vector<uint32_t> slot(E32);
        for (uint32_t e = 0; e < E32; ++e) {
            const double beta = betas[e < s->E ? e : 0];
            memcpy(&bits[e], &beta, sizeof beta);
            slot[e] = e;
        }
        if (!s->d_t64 || s->t64_rows != E32) {
            cudaFree(s->d_t64); cudaFree(s->d_slot);
            s->d_t64 = nullptr; s->d_slot = nullptr;
            CUDA_TRY(ctx, dev_alloc(&s->d_t64, (size_t)E32));
            CUDA_TRY(ctx, dev_alloc(&s->d_slot, (size_t)E32));
            s->t64_rows = E32;
        }
        CUDA_TRY(ctx, cudaMemcpyAsync(s->d_t64, bits.data(), bits.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
        CUDA_TRY(ctx, cudaMemcpyAsync(s->d_slot, slot.data(), slot.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));   // locals
        s->perbeta = true;
        return ISING_OK;
    }
    if (!s->general) {
        // checkerboard layout: classes dE = 4|J|, 8|J| (, 12|J|); tables are built for 6 planes
        if (s->planes != 6)
            return fail(ctx, ISING_E_UNSUPPORTED, "per-experiment betas on a lattice need planes = 6");
        std::vector<unsigned long long> t64((size_t)E32 * 3, 0ull);
        const int ncls = h.kind == ISING_KIND_STENCIL3D ? 3 : 2;
        for (uint32_t e = 0; e < E32; ++e) {
            const double beta = betas[e < s->E ? e : 0];
            for (int c = 0; c < ncls; ++c)
                t64[(size_t)e * 3 + c] = threshold64(beta, 4.0 * (c + 1) * h.jabs, s->planes);
        }
        if (!s->d_t64 || s->t64_rows != E32) {
            cudaFree(s->d_t64); cudaFree(s->d_slot); cudaFree(s->d_tplane); cudaFree(s->d_tlow);
            s->d_t64 = nullptr; s->d_slot = nullptr; s->d_tplane = nullptr; s->d_tlow = nullptr;
            CUDA_TRY(ctx, dev_alloc(&s->d_t64, t64.size()));
            CUDA_TRY(ctx, dev_alloc(&s->d_tplane, (size_t)W * 3 * 8));
            CUDA_TRY(ctx, dev_alloc(&s->d_tlow, (size_t)E32 * 3));
            s->t64_rows = E32;
        }
        CUDA_TRY(ctx, cudaMemcpyAsync(s->d_t64, t64.data(), t64.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
        // no host wait: cudaMemcpyAsync from pageable memory returns once the buffer is staged
        count_launch(s, launch_build_tables_stencil(s->d_t64, nullptr, W, s->planes, s->d_tplane, s->d_tlow, ctx->stream));
        s->perbeta = true;
        return ISING_OK;
    }
    const size_t per = (size_t)(GEN_MAX_DEG + 1) * GEN_MAX_CLS;
    std::vector<unsigned long long> t64((size_t)E32 * per, 0ull);
    std::vector<uint32_t> slot(E32);
    if (s->beta_rows_planes != s->planes || s->beta_rows.size() > 65536) {
        s->beta_rows.clear();
        s->beta_rows_planes = s->planes;
    }
    for (uint32_t e = 0; e < E32; ++e) {
        slot[e] = e;
        const double beta = betas[e < s->E ? e : 0];  // padding bits: any valid beta
        uint64_t key;
        memcpy(&key, &beta, sizeof key);
        auto it = s->beta_rows.find(key);
        if (it == s->beta_rows.end()) {
            std::vector<unsigned long long> row(per, 0ull);
            for (uint32_t deg = 1; deg <= (uint32_t)GEN_MAX_DEG; ++deg) {
                const uint32_t cmin = deg / 2 + 1, ncls = deg - deg / 2;
                for (uint32_t j = 0; j < ncls; ++j) {
                    const int cls = 2 * (int)(cmin + j) - (int)deg;
                    row[(size_t)deg * GEN_MAX_CLS + j] = threshold64(beta, 2.0 * h.jabs * (double)cls, s->planes);
                }
            }
            it = s->beta_rows.emplace(key, std::move(row)).first;
        }
        memcpy(&t64[(size_t)e * per], it->second.data(), per * sizeof(unsigned long long));
    }
    if (!s->d_t64 || s->t64_rows != E32) {
        cudaFree(s->d_t64); cudaFree(s->d_slot); cudaFree(s->d_tplane); cudaFree(s->d_tlow);
        s->d_t64 = nullptr; s->d_slot = nullptr; s->d_tplane = nullptr; s->d_tlow = nullptr;
        s->t64_rows = E32;
        CUDA_TRY(ctx, dev_alloc(&s->d_t64, t64.size()));
        CUDA_TRY(ctx, dev_alloc(&s->d_slot, (size_t)E32));
        CUDA_TRY(ctx, dev_alloc(&s->d_tplane, (size_t)(GEN_MAX_DEG + 1) * W * GEN_MAX_CLS * 8));
        CUDA_TRY(ctx, dev_alloc(&s->d_tlow, (size_t)(GEN_MAX_DEG + 1) * E32 * GEN_MAX_CLS));
    }
    CUDA_TRY(ctx, cudaMemcpyAsync(s->d_t64, t64.data(), t64.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(s->d_slot, slot.data(), slot.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    count_launch(s, launch_build_tables(s->d_t64, s->d_slot, W, s->planes, s->d_tplane, s->d_tlow,
                                        ctx->stream));
    // no host wait: cudaMemcpyAsync from pageable memory returns once t64 / slot are staged
    s->perbeta = true;
    return ISING_OK;
}

// Thresholds by SLOT (one row per inverse temperature of a ladder) plus a device-resident
// replica -> slot indirection: a swap step only permutes slot_of_replica on the device and
// rebuilds the bit-sliced tables from the resident rows - no exp(), no upload, no host wait.
static int sim_set_slot_thresholds(ising_sim* s, const double* betas_by_slot, uint64_t R) {
    ising_ctx* ctx = s->ctx;
    const HostGraph& h = s->g->h;
    const uint32_t W = s->lay.W, E32 = 32 * W;
    if (s->real) {
        // real couplings / biases: the float-field kernel takes exp(-beta dE) per replica bit, so the
        // "rows" are the betas themselves (f64 bit patterns by slot) behind the same replica -> slot map
        std::vector<unsigned long long> bits(R);
        for (uint64_t r = 0; r < R; ++r) memcpy(&bits[r], &betas_by_slot[r], sizeof(double));
        CUDA_TRY(ctx, cudaSetDevice(ctx->device));
        cudaFree(s->d_t64); s->d_t64 = nullptr;
        cudaFree(s->d_slot); s->d_slot = nullptr;
        CUDA_TRY(ctx, dev_alloc(&s->d_t64, (size_t)R));
        CUDA_TRY(ctx, dev_alloc(&s->d_slot, (size_t)E32));
        CUDA_TRY(ctx, cudaMemsetAsync(s->d_slot, 0, (size_t)E32 * 4, ctx->stream));
        CUDA_TRY(ctx, cudaMemcpyAsync(s->d_t64, bits.data(), bits.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));   // bits is a local
        s->perbeta = true;
        s->t64_rows = (uint32_t)R;
        return ISING_OK;
    }
    const size_t per = s->general ? (size_t)(GEN_MAX_DEG + 1) * GEN_MAX_CLS : 3;
    if (!s->general && s->planes != 6)
        return fail(ctx, ISING_E_UNSUPPORTED, "per-experiment betas on a lattice need planes = 6");
    std::vector<unsigned long long> t64((size_t)R * per, 0ull);
    for (uint64_t r = 0; r < R; ++r) {
        const double beta = betas_by_slot[r];
        if (s->general) {
            for (uint32_t deg = 1; deg <= (uint32_t)GEN_MAX_DEG; ++deg) {
                const uint32_t cmin = deg / 2 + 1, ncls = deg - deg / 2;
                for (uint32_t j = 0; j < ncls; ++j) {
                    const int cls = 2 * (int)(cmin + j) - (int)deg;
                    t64[r * per + (size_t)deg * GEN_MAX_CLS + j] = threshold64(beta, 2.0 * h.jabs * (double)cls, s->planes);
                }
            }
        } else {
            const int ncls = h.kind == ISING_KIND_STENCIL3D ? 3 : 2;
            for (int c = 0; c < ncls; ++c) t64[r * per + c] = threshold64(beta, 4.0 * (c + 1) * h.jabs, s->planes);
        }
    }
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    cudaFree(s->d_t64); s->d_t64 = nullptr;
    cudaFree(s->d_slot); s->d_slot = nullptr;
    cudaFree(s->d_tplane); s->d_tplane = nullptr;
    cudaFree(s->d_tlow); s->d_tlow = nullptr;
    CUDA_TRY(ctx, dev_alloc(&s->d_t64, t64.size()));
    CUDA_TRY(ctx, dev_alloc(&s->d_slot, (size_t)E32));
    if (s->general) {
        CUDA_TRY(ctx, dev_alloc(&s->d_tplane, (size_t)(GEN_MAX_DEG + 1) * W * GEN_MAX_CLS * 8));
        CUDA_TRY(ctx, dev_alloc(&s->d_tlow, (size_t)(GEN_MAX_DEG + 1) * E32 * GEN_MAX_CLS));
    } else {
        CUDA_TRY(ctx, dev_alloc(&s->d_tplane, (size_t)W * 3 * 8));
        CUDA_TRY(ctx, dev_alloc(&s->d_tlow, (size_t)E32 * 3));
    }
    CUDA_TRY(ctx, cudaMemcpyAsync(s->d_t64, t64.data(), t64.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));   // t64 is a local
    s->perbeta = true;
    s->t64_rows = (uint32_t)R;
    return ISING_OK;
}

// bit-sliced threshold tables of the sim from its resident rows and slot_of_replica (enqueue only)
static int sim_tables_from_slots(ising_sim* s) {
    ising_ctx* ctx = s->ctx;
    if (s->real) return ISING_OK;   // the float-field kernel reads the betas through the slot map
    const int n = s->general ? launch_build_tables(s->d_t64, s->d_slot, s->lay.W, s->planes, s->d_tplane,
                                                   s->d_tlow, ctx->stream)
                             : launch_build_tables_stencil(s->d_t64, s->d_slot, s->lay.W, s->planes,
                                                           s->d_tplane, s->d_tlow, ctx->stream);
    if (n < 0) return fail(ctx, ISING_E_CUDA, "threshold table launch failed");
    count_launch(s, n);
    return ISING_OK;
}

struct ising_pt {
    ising_ctx* ctx = nullptr;
    const ising_graph* g = nullptr;
    ising_sim* sim = nullptr;
    ising_comm* comm = nullptr;       // borrowed; NULL = this rank holds every configuration
    uint64_t R = 0, lo = 0, hi = 0;   // this rank owns configurations [lo, hi)
    uint64_t word_lo = 0;             // first replica word held locally
    std::vector<double> betas;        // by slot
    uint64_t seed = 0;
    // host mirrors of the device-resident state (valid unless host_stale)
    std::vector<uint32_t> slot_of_cfg, cfg_of_slot;
    std::vector<unsigned long long> stats;   // swap_step, total_swaps, attempts[R], accepts[R]
    bool host_stale = false;
    // device-resident state of the exchange cycle
    double* d_betas = nullptr;
    uint32_t* d_slot_of_cfg = nullptr;
    uint32_t* d_cfg_of_slot = nullptr;
    uint32_t* d_gidx = nullptr;       // configuration -> index in the gathered arrays
    std::vector<uint32_t> gidx;
    double* d_e_local = nullptr;      // [32 W] energies of the locally held replica bits
    double* d_e_all = nullptr;        // [world * cmax] gathered, rank-major
    double* d_acc = nullptr;          // [R] sum of E * t by slot
    unsigned long long* d_nsat = nullptr;   // [32 W] satisfied-bond counters of the cycle (kept zeroed by k_pt_cycle)
    unsigned long long* d_stats = nullptr;
    uint64_t cmax = 0;                // configurations per rank in the gathered arrays
    int world = 1, rank = 0;
};

int comm_rank(const ising_comm* c);
int comm_world(const ising_comm* c);
int comm_allgather_bytes(ising_comm* c, const void* send, void* recv, size_t bytes, cudaStream_t st);

// block of configurations of rank r when R configurations are split over `world` ranks
static void pt_block(uint64_t R, int world, int r, uint64_t* lo, uint64_t* hi) {
    const uint64_t base = R / (uint64_t)world, rem = R % (uint64_t)world;
    *lo = (uint64_t)r * base + std::min<uint64_t>((uint64_t)r, rem);
    *hi = *lo + base + ((uint64_t)r < rem ? 1 : 0);
}

// gathered-array layout for `world` ranks (world = 1: identity)
static void pt_layout(ising_pt* pt, int world) {
    pt->world = world;
    pt->cmax = (pt->R + (uint64_t)world - 1) / (uint64_t)world;
    pt->gidx.assign(pt->R, 0);
    for (int r = 0; r < world; ++r) {
        uint64_t lo, hi;
        pt_block(pt->R, world, r, &lo, &hi);
        for (uint64_t c = lo; c < hi; ++c) pt->gidx[c] = (uint32_t)((uint64_t)r * pt->cmax + (c - lo));
    }
}

static int pt_upload_layout(ising_pt* pt) {
    ising_ctx* ctx = pt->ctx;
    cudaFree(pt->d_e_all);
    pt->d_e_all = nullptr;
    CUDA_TRY(ctx, dev_alloc(&pt->d_e_all, (size_t)pt->world * pt->cmax + 32));
    CUDA_TRY(ctx, cudaMemsetAsync(pt->d_e_all, 0, ((size_t)pt->world * pt->cmax + 32) * sizeof(double), ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(pt->d_gidx, pt->gidx.data(), pt->R * 4, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return ISING_OK;
}

// host permutation / counters -> device, then the replica -> slot map and the threshold tables
static int pt_push_state(ising_pt* pt) {
    ising_ctx* ctx = pt->ctx;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, cudaMemcpyAsync(pt->d_slot_of_cfg, pt->slot_of_cfg.data(), pt->R * 4, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(pt->d_cfg_of_slot, pt->cfg_of_slot.data(), pt->R * 4, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(pt->d_stats, pt->stats.data(), pt->stats.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
    count_launch(pt->sim, launch_pt_local_slots(pt->d_slot_of_cfg, (uint32_t)pt->R, pt->sim->d_slot,
                                                (uint32_t)pt->word_lo, pt->sim->lay.W * 32, ctx->stream));
    const int rc = sim_tables_from_slots(pt->sim);
    if (rc) return rc;
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));   // the host vectors may change after return
    pt->host_stale = false;
    return ISING_OK;
}

// device permutation / counters -> host mirrors (one wait; only when the host asks for them)
static int pt_sync_host(ising_pt* pt) {
    if (!pt->host_stale) return ISING_OK;
    ising_ctx* ctx = pt->ctx;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, cudaMemcpyAsync(pt->slot_of_cfg.data(), pt->d_slot_of_cfg, pt->R * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(pt->cfg_of_slot.data(), pt->d_cfg_of_slot, pt->R * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(pt->stats.data(), pt->d_stats, pt->stats.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    pt->host_stale = false;
    return ISING_OK;
}

static void pt_free_device(ising_pt* pt) {
    cudaFree(pt->d_betas);
    cudaFree(pt->d_slot_of_cfg);
    cudaFree(pt->d_cfg_of_slot);
    cudaFree(pt->d_gidx);
    cudaFree(pt->d_e_local);
    cudaFree(pt->d_e_all);
    cudaFree(pt->d_acc);
    cudaFree(pt->d_nsat);
    cudaFree(pt->d_stats);
}

extern "C" int ising_pt_create(ising_ctx* ctx, const ising_graph* g, const double* betas,
                               uint64_t nbetas, uint64_t cfg_lo, uint64_t cfg_hi, uint64_t seed,
                               ising_pt** out) {
    CtxLock _lk(ctx);
    if (!ctx || !g || !betas || !out) return fail(ctx, ISING_E_INVALID, "ctx/graph/betas/out is NULL");
    *out = nullptr;
    if (nbetas == 0 || cfg_lo >= cfg_hi || cfg_hi > nbetas)
        return fail(ctx, ISING_E_INVALID, "need 0 <= cfg_lo < cfg_hi <= nbetas");
    if (nbetas > 0xFFFFFFFFull) return fail(ctx, ISING_E_UNSUPPORTED, "too many replicas");
    if (g->h.field_graph)
        return fail(ctx, ISING_E_UNSUPPORTED, "tempering on a torus in a field is not supported (give the field as biases of an edge list)");
    std::unique_ptr<ising_pt> pt(new ising_pt);
    pt->ctx = ctx;
    pt->g = g;
    pt->R = nbetas;
    pt->lo = cfg_lo;
    pt->hi = cfg_hi;
    pt->seed = seed;
    pt->betas.assign(betas, betas + nbetas);
    pt->slot_of_cfg.resize(nbetas);
    pt->cfg_of_slot.resize(nbetas);
    pt->stats.assign(2 + 2 * nbetas, 0ull);
    for (uint64_t r = 0; r < nbetas; ++r) pt->slot_of_cfg[r] = pt->cfg_of_slot[r] = (uint32_t)r;
    // whole replica words: configuration c always lives at bit c%32 of global word c/32, so a
    // sharded run draws exactly the random numbers of the unsharded one
    pt->word_lo = cfg_lo / 32;
    const uint64_t word_hi = (cfg_hi + 31) / 32;
    const uint64_t E = std::min<uint64_t>((word_hi - pt->word_lo) * 32, nbetas - pt->word_lo * 32);
    // lattices temper on the checkerboard kernels, other graphs on the colour x degree kernels
    int rc = ising_sim_create_ex(ctx, g, E, seed, pt->word_lo * 32, 0u, &pt->sim);
    if (rc) return rc;
    auto bail = [&](int code) {
        pt_free_device(pt.get());
        ising_sim_destroy(pt->sim);
        return code;
    };
    rc = sim_set_slot_thresholds(pt->sim, pt->betas.data(), nbetas);
    if (rc) return bail(rc);
    const size_t e32 = (size_t)pt->sim->lay.W * 32;
    cudaError_t e = dev_alloc(&pt->d_betas, nbetas);
    if (e == cudaSuccess) e = dev_alloc(&pt->d_slot_of_cfg, nbetas);
    if (e == cudaSuccess) e = dev_alloc(&pt->d_cfg_of_slot, nbetas);
    if (e == cudaSuccess) e = dev_alloc(&pt->d_gidx, nbetas);
    if (e == cudaSuccess) e = dev_alloc(&pt->d_e_local, e32 + nbetas);
    if (e == cudaSuccess) e = dev_alloc(&pt->d_acc, nbetas);
    if (e == cudaSuccess) e = dev_alloc(&pt->d_stats, pt->stats.size());
    if (e == cudaSuccess) e = dev_alloc(&pt->d_nsat, e32);
    if (e == cudaSuccess) e = cudaMemsetAsync(pt->d_nsat, 0, e32 * sizeof(unsigned long long), ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(pt->d_acc, 0, nbetas * sizeof(double), ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(pt->d_e_local, 0, (e32 + nbetas) * sizeof(double), ctx->stream);
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(pt->d_betas, pt->betas.data(), nbetas * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
    if (e != cudaSuccess) return bail(fail(ctx, ISING_E_CUDA, "tempering state allocation: %s", cudaGetErrorString(e)));
    // until a communicator is attached the gathered array is this rank's view: identity layout
    // when it holds everything, otherwise the layout of the ranks implied by [cfg_lo, cfg_hi)
    pt_layout(pt.get(), 1);
    rc = pt_upload_layout(pt.get());
    if (rc == ISING_OK) rc = pt_push_state(pt.get());
    if (rc) return bail(rc);
    *out = pt.release();
    ctx_retain(ctx);
    return ISING_OK;
}

extern "C" int ising_pt_set_comm(ising_pt* pt, ising_comm* comm) {
    CtxLock _lk(pt ? pt->ctx : nullptr);
    if (!pt) return fail(nullptr, ISING_E_INVALID, "pt is NULL");
    const int world = comm_world(comm), rank = comm_rank(comm);
    uint64_t lo, hi;
    pt_block(pt->R, world, rank, &lo, &hi);
    if (lo != pt->lo || hi != pt->hi)
        return fail(pt->ctx, ISING_E_INVALID,
                    "rank %d of %d must own configurations [%llu, %llu) (contiguous blocks, remainder to the "
                    "first ranks); this ladder was created for [%llu, %llu)", rank, world,
                    (unsigned long long)lo, (unsigned long long)hi, (unsigned long long)pt->lo,
                    (unsigned long long)pt->hi);
    pt->comm = comm;
    pt->rank = rank;
    pt_layout(pt, world);
    return pt_upload_layout(pt);
}

extern "C" void ising_pt_destroy(ising_pt* pt) {
    if (!pt) return;
    struct Release { ising_ctx* c; ~Release() { ctx_release(c); } } _rel{pt->ctx};   // after the lock is gone
    CtxLock _lk(pt->ctx);
    cudaSetDevice(pt->ctx->device);
    cudaStreamSynchronize(pt->ctx->stream);
    pt_free_device(pt);
    ising_sim_destroy(pt->sim);
    delete pt;
}

extern "C" int ising_pt_configure(ising_pt* pt, int planes, int rounds) {
    CtxLock _lk(pt ? pt->ctx : nullptr);
    if (!pt) return fail(nullptr, ISING_E_INVALID, "pt is NULL");
    int rc = ising_sim_configure(pt->sim, planes, rounds);
    if (rc) return rc;
    rc = pt_sync_host(pt);
    if (rc) return rc;
    rc = sim_set_slot_thresholds(pt->sim, pt->betas.data(), pt->R);   // thresholds depend on the plane count
    return rc ? rc : pt_push_state(pt);
}

extern "C" int ising_pt_sweeps(ising_pt* pt, uint64_t t, double* local_energies) {
    CtxLock _lk(pt ? pt->ctx : nullptr);
    if (!pt) return fail(nullptr, ISING_E_INVALID, "pt is NULL");
    if (!local_energies) return ising_sim_sweeps(pt->sim, nullptr, t, nullptr);
    // enqueue only: the energy read-back below is the one host wait of the swap cycle
    CUDA_TRY(pt->ctx, cudaSetDevice(pt->ctx->device));
    int rc = sim_enqueue_sweeps(pt->sim, nullptr, t);
    if (rc) return rc;
    std::vector<double> en(pt->sim->E);
    rc = ising_sim_get_energies(pt->sim, en.data());
    if (rc) return rc;
    for (uint64_t c = pt->lo; c < pt->hi; ++c) local_energies[c - pt->lo] = en[c - pt->word_lo * 32];
    return ISING_OK;
}

// One tempering step (the shape of TemperingContainer::parallel_tempering_step as driven from
// tempering.rs:191-194): even slot pairs (0,1),(2,3).. then odd pairs (1,2),(3,4)..; the pair
// (a, a+1) exchanges configurations with probability min(1, exp((b_a - b_{a+1})(E_a - E_{a+1}))).
// The uniform is Philox(seed; slot a, swap step), so every rank takes the same decisions from
// the all-gathered energies.  all_energies is indexed by CONFIGURATION.  Host restatement of
// k_pt_swap (same operations in the same order; exp is the fixed sequence of pt_exp.h).
extern "C" int ising_pt_decide_swaps(const double* betas, uint64_t R, const double* all_energies,
                                     uint64_t seed, uint64_t swap_step, uint32_t* slot_of_cfg,
                                     uint32_t* cfg_of_slot, uint64_t* nswaps) {
    if (!betas || !all_energies || !slot_of_cfg || !cfg_of_slot)
        return fail(nullptr, ISING_E_INVALID, "ising_pt_decide_swaps: NULL argument");
    uint64_t swaps = 0;
    for (int parity = 0; parity < 2; ++parity)
        for (uint64_t a = parity; a + 1 < R; a += 2) {
            const uint32_t ca = cfg_of_slot[a], cb = cfg_of_slot[a + 1];
            const double db = betas[a] - betas[a + 1], de = all_energies[ca] - all_energies[cb];
            const double d = db * de;
            bool acc = true;
            if (d < 0.0) {
                const u32x4 r = philox4x32<10>((uint32_t)a, (uint32_t)parity, (uint32_t)swap_step,
                                               TAG_SWAP << 24, (uint32_t)seed, (uint32_t)(seed >> 32));
                const double uu = ((double)r.x + 0.5) * (1.0 / 4294967296.0);
                acc = uu < pt_exp_nonpos(d);
            }
            if (acc) {
                cfg_of_slot[a] = cb;
                cfg_of_slot[a + 1] = ca;
                slot_of_cfg[cb] = (uint32_t)a;
                slot_of_cfg[ca] = (uint32_t)(a + 1);
                ++swaps;
            }
        }
    if (nswaps) *nswaps = swaps;
    return ISING_OK;
}

// swap decisions + slot map + threshold tables on the device from d_e_all (enqueue only)
static int pt_device_swap(ising_pt* pt) {
    ising_ctx* ctx = pt->ctx;
    const int n = launch_pt_swap(pt->d_betas, pt->d_e_all, pt->d_gidx, pt->d_slot_of_cfg, pt->d_cfg_of_slot,
                                 (uint32_t)pt->R, pt->seed, pt->d_stats, pt->sim->d_slot,
                                 (uint32_t)pt->word_lo, pt->sim->lay.W * 32, ctx->stream);
    if (n < 0) return fail(ctx, ISING_E_CUDA, "swap kernel launch failed");
    count_launch(pt->sim, n);
    pt->host_stale = true;
    return sim_tables_from_slots(pt->sim);
}

// One launch for everything between two batches of sweeps (see k_pt_cycle); with a communicator
// the energies are computed first, gathered, and the rest follows in one launch.
// counted: the sweeps before left the satisfied-bond counts in pt->d_nsat (sim_enqueue_sweeps_counting)
static int pt_cycle(ising_pt* pt, uint64_t t, bool do_swap, bool counted = false) {
    ising_ctx* ctx = pt->ctx;
    ising_sim* sim = pt->sim;
    const HostGraph& h = pt->g->h;
    const bool multi = pt->comm && pt->world > 1;
    int rc = ISING_OK;
    if (sim->real) {
        // real couplings / biases: f64 energies from the CSR energy kernel instead of bond counters
        rc = sim_energies_to_device(sim, pt->d_e_local, 1, 0);
        if (rc == ISING_OK && !multi)
            CUDA_TRY(ctx, cudaMemcpyAsync(pt->d_e_all, pt->d_e_local, sim->E * sizeof(double),
                                          cudaMemcpyDeviceToDevice, ctx->stream));
    } else if (!counted) {
        rc = sim_count_nsat(sim, pt->d_nsat, false);
    }
    if (rc) return rc;
    PtCycleArgs a;
    a.nsat = sim->real ? nullptr : pt->d_nsat;
    a.e_local = pt->d_e_local;
    a.e_all = pt->d_e_all;
    a.E = (uint32_t)sim->E;
    a.e32 = sim->lay.W * 32;
    a.identity = multi ? 0u : 1u;
    a.scale = h.jabs;
    a.nbonds = h.nedges;
    a.mult = sim->general ? 1 : 2;
    a.gidx = pt->d_gidx;
    a.betas = pt->d_betas;
    a.slot_of_cfg = pt->d_slot_of_cfg;
    a.cfg_of_slot = pt->d_cfg_of_slot;
    a.R = (uint32_t)pt->R;
    a.key0 = (uint32_t)pt->seed;
    a.key1 = (uint32_t)(pt->seed >> 32);
    a.stats = pt->d_stats;
    a.slot_of_replica = sim->d_slot;
    a.word_lo = (uint32_t)pt->word_lo;
    a.acc = pt->d_acc;
    a.t = (double)t;
    a.do_swap = do_swap ? 1 : 0;
    const bool fuse_tables = do_swap && !sim->general;
    a.t64 = fuse_tables ? sim->d_t64 : nullptr;
    a.W = sim->lay.W;
    a.K = sim->planes;
    a.tplane = sim->d_tplane;
    a.tlow = sim->d_tlow;
    if (multi) {
        // energies first (no accumulate / swap: R = 0), all-gather, then the rest without the energy part
        if (!sim->real) {
            PtCycleArgs e = a;
            e.R = 0;
            e.do_swap = 0;
            e.t64 = nullptr;
            if (launch_pt_cycle(e, ctx->stream) < 0) return fail(ctx, ISING_E_CUDA, "tempering cycle launch failed");
            count_launch(sim, 1);
        }
        const double* mine = pt->d_e_local + (pt->lo - pt->word_lo * 32);
        rc = comm_allgather_bytes(pt->comm, mine, pt->d_e_all, pt->cmax * sizeof(double), ctx->stream);
        if (rc) return rc;
        a.nsat = nullptr;
    } else if (!(pt->lo == 0 && pt->hi == pt->R)) {
        return fail(ctx, ISING_E_INVALID, "a sharded ladder needs a communicator (ising_pt_set_comm)");
    }
    if (launch_pt_cycle(a, ctx->stream) < 0) return fail(ctx, ISING_E_CUDA, "tempering cycle launch failed");
    count_launch(sim, 1);
    if (do_swap) {
        pt->host_stale = true;
        if (!fuse_tables) return sim_tables_from_slots(sim);
    }
    return ISING_OK;
}

extern "C" int ising_pt_swap_step(ising_pt* pt, const double* all_energies) {
    CtxLock _lk(pt ? pt->ctx : nullptr);
    if (!pt || !all_energies) return fail(pt ? pt->ctx : nullptr, ISING_E_INVALID, "pt/energies is NULL");
    ising_ctx* ctx = pt->ctx;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    // host-provided energies (by configuration) into the gathered layout, then the device step
    std::vector<double> staged((size_t)pt->world * pt->cmax, 0.0);
    for (uint64_t c = 0; c < pt->R; ++c) staged[pt->gidx[c]] = all_energies[c];
    CUDA_TRY(ctx, cudaMemcpyAsync(pt->d_e_all, staged.data(), staged.size() * sizeof(double),
                                  cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));   // `staged` is a local
    return pt_device_swap(pt);
}

extern "C" int ising_pt_get_slots(const ising_pt* cpt, uint32_t* slot_of_config) {
    ising_pt* pt = const_cast<ising_pt*>(cpt);
    CtxLock _lk(pt ? pt->ctx : nullptr);
    if (!pt || !slot_of_config) return fail(nullptr, ISING_E_INVALID, "pt/out is NULL");
    const int rc = pt_sync_host(pt);
    if (rc) return rc;
    for (uint64_t c = 0; c < pt->R; ++c) slot_of_config[c] = pt->slot_of_cfg[c];
    return ISING_OK;
}

extern "C" int ising_pt_get_local_states(ising_pt* pt, uint8_t* states) {
    CtxLock _lk(pt ? pt->ctx : nullptr);
    if (!pt || !states) return fail(pt ? pt->ctx : nullptr, ISING_E_INVALID, "pt/states is NULL");
    const uint64_t N = pt->g->h.nvars;
    std::vector<uint8_t> all((size_t)pt->sim->E * N);
    const int rc = ising_sim_get_states(pt->sim, all.data());
    if (rc) return rc;
    for (uint64_t c = pt->lo; c < pt->hi; ++c)
        memcpy(states + (c - pt->lo) * N, all.data() + (c - pt->word_lo * 32) * N, N);
    return ISING_OK;
}

// checkpoint support: the sim behind the ladder, and the permutation / counters
extern "C" int ising_pt_get_sim(ising_pt* pt, ising_sim** out) {
    CtxLock _lk(pt ? pt->ctx : nullptr);
    if (!pt || !out) return fail(nullptr, ISING_E_INVALID, "pt/out is NULL");
    *out = pt->sim;
    return ISING_OK;
}

extern "C" int ising_pt_get_counters(const ising_pt* cpt, uint64_t* swap_step, uint64_t* total_swaps) {
    ising_pt* pt = const_cast<ising_pt*>(cpt);
    CtxLock _lk(pt ? pt->ctx : nullptr);
    if (!pt || !swap_step || !total_swaps) return fail(nullptr, ISING_E_INVALID, "pt/out is NULL");
    const int rc = pt_sync_host(pt);
    if (rc) return rc;
    *swap_step = pt->stats[0];
    *total_swaps = pt->stats[1];
    return ISING_OK;
}

// SURVEY 5.5: swaps attempted / accepted per pair of neighbouring betas (pair a = slots a, a+1)
extern "C" int ising_pt_get_pair_stats(const ising_pt* cpt, uint64_t* attempts, uint64_t* accepts) {
    ising_pt* pt = const_cast<ising_pt*>(cpt);
    CtxLock _lk(pt ? pt->ctx : nullptr);
    if (!pt || !attempts || !accepts) return fail(nullptr, ISING_E_INVALID, "pt/out is NULL");
    const int rc = pt_sync_host(pt);
    if (rc) return rc;
    for (uint64_t a = 0; a + 1 < pt->R; ++a) {
        attempts[a] = pt->stats[2 + a];
        accepts[a] = pt->stats[2 + pt->R + a];
    }
    return ISING_OK;
}

extern "C" int ising_pt_restore(ising_pt* pt, const uint32_t* slot_of_config, uint64_t swap_step,
                                uint64_t total_swaps) {
    CtxLock _lk(pt ? pt->ctx : nullptr);
    if (!pt || !slot_of_config) return fail(pt ? pt->ctx : nullptr, ISING_E_INVALID, "pt/slots is NULL");
    std::vector<uint8_t> seen(pt->R, 0);
    for (uint64_t c = 0; c < pt->R; ++c) {
        if (slot_of_config[c] >= pt->R || seen[slot_of_config[c]])
            return fail(pt->ctx, ISING_E_INVALID, "slot_of_config is not a permutation");
        seen[slot_of_config[c]] = 1;
    }
    int rc = pt_sync_host(pt);
    if (rc) return rc;
    for (uint64_t c = 0; c < pt->R; ++c) {
        pt->slot_of_cfg[c] = slot_of_config[c];
        pt->cfg_of_slot[slot_of_config[c]] = (uint32_t)c;
    }
    pt->stats[0] = swap_step;
    pt->stats[1] = total_swaps;
    return pt_push_state(pt);
}

extern "C" int ising_pt_total_swaps(const ising_pt* cpt, uint64_t* out) {
    ising_pt* pt = const_cast<ising_pt*>(cpt);
    CtxLock _lk(pt ? pt->ctx : nullptr);
    if (!pt || !out) return fail(nullptr, ISING_E_INVALID, "pt/out is NULL");
    const int rc = pt_sync_host(pt);
    if (rc) return rc;
    *out = pt->stats[1];
    return ISING_OK;
}

// LatticeTempering::qmc_timesteps_sample, tempering.rs:156-222: run min(to_sample, to_swap,
// remaining) -> swap step -> sample; states[R, n_s, nvars] holds "the configuration currently at
// beta_r", energies[R] = sum(E_r after chunk * chunk) / timesteps.
//
// The whole loop is enqueued on the context's stream: sweeps, energies, (multi-GPU) the NCCL
// all-gather of the R energies, the swap kernel, the table rebuild, the slot-ordered samples
// and their copies to the caller's array - the host waits once, at the end.  A ladder that is
// sharded over ranks (ising_pt_set_comm) runs the same loop on every rank and every rank
// returns the full arrays.
extern "C" int ising_pt_timesteps_sample(ising_pt* pt, uint64_t timesteps, uint64_t replica_swap_freq,
                                         uint64_t sampling_freq, uint8_t* states, double* energies) {
    CtxLock _lk(pt ? pt->ctx : nullptr);
    if (!pt || !energies) return fail(pt ? pt->ctx : nullptr, ISING_E_INVALID, "pt/energies is NULL");
    ising_ctx* ctx = pt->ctx;
    const bool whole = pt->lo == 0 && pt->hi == pt->R;
    if (!whole && !(pt->comm && pt->world > 1))
        return fail(ctx, ISING_E_INVALID,
                    "ising_pt_timesteps_sample needs all configurations on this rank or a communicator");
    if (replica_swap_freq == 0 || sampling_freq == 0)
        return fail(ctx, ISING_E_INVALID,
                    "replica_swap_freq and sampling_freq must be > 0 (the reference loops forever on 0)");
    const uint64_t R = pt->R, N = pt->g->h.nvars, ns = timesteps / sampling_freq;
    if (ns && !states) return fail(ctx, ISING_E_INVALID, "states is NULL");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, cudaMemsetAsync(pt->d_acc, 0, R * sizeof(double), ctx->stream));
    // sample staging: the local rows (unpacked), the gathered rows, the slot-ordered rows
    uint8_t *d_rows = nullptr, *d_all = nullptr, *d_sorted = nullptr;
    const uint64_t E = pt->sim->E;
    const size_t rows_local = (size_t)(E + pt->cmax) * N;
    if (ns) {
        void* dv = nullptr;
        CUDA_TRY(ctx, ctx_scratch(ctx, 0, rows_local, &dv));
        d_rows = (uint8_t*)dv;
        CUDA_TRY(ctx, ctx_scratch(ctx, 4, (size_t)pt->world * pt->cmax * N, &dv));
        d_all = (uint8_t*)dv;
        CUDA_TRY(ctx, ctx_scratch(ctx, 5, (size_t)R * N, &dv));
        d_sorted = (uint8_t*)dv;
    }
    uint64_t remaining = timesteps, to_swap = replica_swap_freq, to_sample = sampling_freq, k = 0;
    int rc = ISING_OK;
    while (remaining > 0 && rc == ISING_OK) {
        const uint64_t t = std::min(std::min(to_sample, to_swap), remaining);
        bool counted = false;
        rc = sim_enqueue_sweeps_counting(pt->sim, t, pt->d_nsat, &counted);
        if (rc) break;
        to_sample -= t; to_swap -= t; remaining -= t;
        rc = pt_cycle(pt, t, to_swap == 0, counted);    // energies, (all-gather,) time average, swap step, tables
        if (rc) break;
        if (to_swap == 0) to_swap = replica_swap_freq;
        if (to_sample == 0) {
            if (k < ns) {
                count_launch(pt->sim, launch_unpack_states(pt->sim->d_spins, pt->sim->lay, d_rows, E, N, ctx->stream));
                const uint8_t* mine = d_rows + (pt->lo - pt->word_lo * 32) * N;
                const uint8_t* gathered = mine;
                if (pt->comm && pt->world > 1) {
                    rc = comm_allgather_bytes(pt->comm, mine, d_all, (size_t)pt->cmax * N, ctx->stream);
                    if (rc) break;
                    gathered = d_all;
                }
                count_launch(pt->sim, launch_pt_gather_rows(gathered, N, pt->d_gidx, pt->d_cfg_of_slot,
                                                            (uint32_t)R, d_sorted, ctx->stream));
                cudaError_t e = copy_rows_d2h(states + k * N, (size_t)ns * N, d_sorted, (size_t)N, (size_t)N, R,
                                              ctx->stream);
                if (e != cudaSuccess) { rc = fail(ctx, ISING_E_CUDA, "sample read-back: %s", cudaGetErrorString(e)); break; }
            }
            ++k;
            to_sample = sampling_freq;
        }
    }
    std::vector<double> acc(R, 0.0);
    cudaError_t e = cudaMemcpyAsync(acc.data(), pt->d_acc, R * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
    cudaError_t e2 = cudaStreamSynchronize(ctx->stream);   // the one host wait (also on error paths)
    if (rc) return rc;
    if (e != cudaSuccess || e2 != cudaSuccess)
        return fail(ctx, ISING_E_CUDA, "tempering loop: %s", cudaGetErrorString(e != cudaSuccess ? e : e2));
    for (uint64_t slot = 0; slot < R; ++slot) energies[slot] = acc[slot] / (double)timesteps;
    return ISING_OK;
}
