// C ABI: one blocking call per reference pymethod (ising_run_*), sampling / observables loops, replay.
#include "api_internal.h"

// ------------------------------------------------------------------------------------------
// one blocking call per pymethod
// ------------------------------------------------------------------------------------------
static int check_run_args(ising_ctx* ctx, const ising_graph* g, const ising_run_args* a,
                          const void* energies, const void* states) {
    if (!ctx || !g || !a) return fail(ctx, ISING_E_INVALID, "ctx/graph/args is NULL");
    if (a->struct_size != sizeof(ising_run_args))
        return fail(ctx, ISING_E_INVALID, "ising_run_args.struct_size mismatch (%u != %zu)",
                    a->struct_size, sizeof(ising_run_args));
    if ((a->flags & ISING_FLAG_EDGE_IMPORTANCE) && !(a->flags & ISING_FLAG_NON_BASIC_MOVES))
        return fail(ctx, ISING_E_UNSUPPORTED,
                    "edge_move_importance_sampling only affects the non-basic edge moves: pass "
                    "ISING_FLAG_NON_BASIC_MOVES as well");
    if ((a->flags & ISING_FLAG_NON_BASIC_MOVES) && (a->flags & ISING_FLAG_ONLY_BASIC_MOVES))
        return fail(ctx, ISING_E_INVALID, "ISING_FLAG_NON_BASIC_MOVES contradicts ISING_FLAG_ONLY_BASIC_MOVES");
    if (a->num_experiments && (!energies || !states))
        return fail(ctx, ISING_E_INVALID, "output buffers are NULL");
    return ISING_OK;
}

static int make_sim_for_run(ising_ctx* ctx, const ising_graph* g, const ising_run_args* a,
                            ising_sim** sim) {
    int rc = ising_sim_create(ctx, g, a->num_experiments, a->seed, a->replica_offset, sim);
    if (rc) return rc;
    if (a->initial_state) rc = ising_sim_set_state(*sim, a->initial_state);
    if (rc == ISING_OK && (a->flags & ISING_FLAG_NON_BASIC_MOVES)) {
        ising_moves mv{};
        mv.struct_size = sizeof mv;
        mv.spin_sweeps = 1;
        mv.edge_passes = 1;
        mv.worms = 1;
        mv.worm_len = 4;
        mv.edge_importance = (a->flags & ISING_FLAG_EDGE_IMPORTANCE) ? 1u : 0u;
        rc = ising_sim_set_moves(*sim, &mv);
    }
    if (rc) { ising_sim_destroy(*sim); *sim = nullptr; }
    return rc;
}

extern "C" int ising_run_monte_carlo(ising_ctx* ctx, const ising_graph* g,
                                     const ising_run_args* a, double* energies, uint8_t* states) {
    CtxLock _lk(ctx);
    int rc = check_run_args(ctx, g, a, energies, states);
    if (rc) return rc;
    if (a->num_experiments == 0) return ISING_OK;
    ising_sim* sim = nullptr;
    rc = make_sim_for_run(ctx, g, a, &sim);
    if (rc) return rc;
    std::vector<double> betas(a->timesteps, a->beta);
    rc = ising_sim_sweeps(sim, betas.data(), a->timesteps, nullptr);
    if (rc == ISING_OK) rc = ising_sim_get_energies(sim, energies);
    if (rc == ISING_OK) rc = ising_sim_get_states(sim, states);
    ising_sim_destroy(sim);
    return rc;
}

static cudaError_t ctx_copy_stream(ising_ctx* ctx) {
    if (ctx->copy_stream) return cudaSuccess;
    cudaError_t e = cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking);
    for (int b = 0; b < 2 && e == cudaSuccess; ++b) {
        e = cudaEventCreateWithFlags(&ctx->ev_filled[b], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_drained[b], cudaEventDisableTiming);
    }
    return e;
}

// thermalise, then n_s x (sampling_freq sweeps, copy state, energy): lattice.rs:271-287 and
// classicising.rs:146-171 on a device-resident sim.  energies[E, n_s], states[E, n_s, nvars].
// At scale: samples are unpacked into one of two device slabs laid out
// [E, nk, N]; while the sweeps of the next slab run, the copy stream drains the previous one
// straight into the caller's [E, ns, N] array with a strided (2D) copy -- no host staging.
// packed != nullptr: samples are returned as uint32[ns, nvars, W] (natural site order, bit e%32 of
// word e/32 = experiment e; 8x less device-to-host traffic) instead of bool[E, ns, nvars].
static int sim_run_sampling_impl(ising_sim* sim, double beta, uint64_t thermalization, uint64_t sampling_freq,
                                 uint64_t ns, double* energies, uint8_t* states, uint32_t* packed) {
    ising_ctx* ctx = sim->ctx;
    if (ns && (!energies || (!states && !packed))) return fail(ctx, ISING_E_INVALID, "output buffers are NULL");
    if (sim->perbeta) return fail(ctx, ISING_E_INVALID, "sampling runs at one beta");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const uint64_t E = sim->E, N = sim->lay.nvars, W = sim->lay.W;
    std::vector<double> betas(std::max<uint64_t>(thermalization, sampling_freq), beta);
    int rc = ising_sim_sweeps(sim, betas.data(), thermalization, nullptr);
    if (rc || ns == 0) return rc;
    CUDA_TRY(ctx, ctx_copy_stream(ctx));
    // Every exit below - also the error returns inside the slab loop - first drains both streams:
    // copies into the caller's arrays and reads of the scratch slabs must not outlive the call.
    struct Drain {
        ising_ctx* c;
        ~Drain() {
            cudaStreamSynchronize(c->copy_stream);
            cudaStreamSynchronize(c->stream);
        }
    } drain{ctx};
    uint64_t slab_bytes = 1ull << 29;
    if (const char* env = getenv("ISING_SAMPLING_SLAB_BYTES")) slab_bytes = strtoull(env, nullptr, 10);  // test knob
    const uint64_t sample_bytes = packed ? N * W * 4 : E * N;   // one sample on the device
    const uint64_t slab = std::max<uint64_t>(1, std::min<uint64_t>(ns, slab_bytes / std::max<uint64_t>(1, sample_bytes)));
    const int nbuf = slab < ns ? 2 : 1;
    uint8_t* d_st[2] = {nullptr, nullptr};
    double* d_en[2] = {nullptr, nullptr};
    for (int b = 0; b < nbuf; ++b) {
        void* dv = nullptr;
        CUDA_TRY(ctx, ctx_scratch(ctx, b ? 4 : 0, (size_t)sample_bytes * slab, &dv));
        d_st[b] = (uint8_t*)dv;
        CUDA_TRY(ctx, ctx_scratch(ctx, b ? 5 : 2, (size_t)E * slab * sizeof(double), &dv));
        d_en[b] = (double*)dv;
    }
    uint64_t islab = 0;
    for (uint64_t k0 = 0; k0 < ns; k0 += slab, ++islab) {
        const uint64_t nk = std::min(slab, ns - k0);
        const int b = (int)(islab & 1);
        if (islab >= 2) CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_drained[b], 0));
        for (uint64_t k = 0; k < nk; ++k) {
            rc = ising_sim_sweeps(sim, betas.data(), sampling_freq, nullptr);
            if (rc) return rc;
            if (packed)   // device slab [nk][N][W]
                count_launch(sim, launch_export_natural(sim->d_spins, sim->lay,
                                                        reinterpret_cast<uint32_t*>(d_st[b]) + k * N * W,
                                                        ctx->stream));
            else          // device slab [E][nk][N]
                count_launch(sim, launch_unpack_states(sim->d_spins, sim->lay, d_st[b] + k * N, E, nk * N,
                                                       ctx->stream));
            rc = sim_energies_to_device(sim, d_en[b], nk, k);
            if (rc) return rc;
        }
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev_filled[b], ctx->stream));
        CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_filled[b], 0));
        if (packed)
            CUDA_TRY(ctx, cudaMemcpyAsync(packed + k0 * N * W, d_st[b], (size_t)nk * sample_bytes,
                                          cudaMemcpyDeviceToHost, ctx->copy_stream));
        else
            CUDA_TRY(ctx, copy_rows_d2h(states + k0 * N, (size_t)ns * N, d_st[b], (size_t)nk * N,
                                        (size_t)nk * N, E, ctx->copy_stream));
        CUDA_TRY(ctx, copy_rows_d2h(energies + k0, (size_t)ns * 8, d_en[b], (size_t)nk * 8,
                                    (size_t)nk * 8, E, ctx->copy_stream));
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev_drained[b], ctx->copy_stream));
    }
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->copy_stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return ISING_OK;
}

extern "C" int ising_sim_run_sampling(ising_sim* sim, double beta, uint64_t thermalization,
                                      uint64_t sampling_freq, uint64_t ns, double* energies,
                                      uint8_t* states) {
    CtxLock _lk(sim ? sim->ctx : nullptr);
    if (!sim) return fail(nullptr, ISING_E_INVALID, "sim is NULL");
    if (ns && !states) return fail(sim->ctx, ISING_E_INVALID, "output buffers are NULL");
    return sim_run_sampling_impl(sim, beta, thermalization, sampling_freq, ns, energies, states, nullptr);
}

extern "C" int ising_sim_run_sampling_packed(ising_sim* sim, double beta, uint64_t thermalization,
                                             uint64_t sampling_freq, uint64_t ns, double* energies,
                                             uint32_t* words) {
    CtxLock _lk(sim ? sim->ctx : nullptr);
    if (!sim) return fail(nullptr, ISING_E_INVALID, "sim is NULL");
    if (ns && !words) return fail(sim->ctx, ISING_E_INVALID, "output buffers are NULL");
    return sim_run_sampling_impl(sim, beta, thermalization, sampling_freq, ns, energies, nullptr, words);
}

// The sampling loop without the state read-back (a sample of config 2 is 17 GB of bools):
// per sample the energy, the magnetisation M = sum_i s_i and, when asked for, the overlap
// Q = sum_i s_i^(2p) s_i^(2p+1) of adjacent experiment pairs (the spin-glass order parameter
// when all experiments share the couplings, lattice.rs:199).  Outputs are [E, ns] / [E/2, ns].
extern "C" int ising_sim_run_observables(ising_sim* sim, double beta, uint64_t thermalization,
                                         uint64_t sampling_freq, uint64_t ns, double* energies,
                                         double* mags, double* overlaps) {
    CtxLock _lk(sim ? sim->ctx : nullptr);
    if (!sim) return fail(nullptr, ISING_E_INVALID, "sim is NULL");
    ising_ctx* ctx = sim->ctx;
    if (sim->perbeta) return fail(ctx, ISING_E_INVALID, "sampling runs at one beta");
    if (sampling_freq == 0) return fail(ctx, ISING_E_INVALID, "sampling_freq must be > 0");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const uint64_t E = sim->E, N = sim->lay.nvars, P = E / 2;
    const size_t cw = (size_t)sim->lay.W * 32;
    std::vector<double> betas(std::max<uint64_t>(thermalization, sampling_freq), beta);
    int rc = ising_sim_sweeps(sim, betas.data(), thermalization, nullptr);
    if (rc || ns == 0) return rc;
    const uint64_t chunk = std::max<uint64_t>(1, std::min<uint64_t>(ns, (1ull << 23) / std::max<uint64_t>(1, E)));
    void* dv = nullptr;
    CUDA_TRY(ctx, ctx_scratch(ctx, 2, (size_t)E * chunk * sizeof(double), &dv));
    double* d_en = (double*)dv;
    CUDA_TRY(ctx, ctx_scratch(ctx, 4, (size_t)E * chunk * sizeof(double), &dv));
    double* d_m = (double*)dv;
    CUDA_TRY(ctx, ctx_scratch(ctx, 5, (size_t)std::max<uint64_t>(P, 1) * chunk * sizeof(double), &dv));
    double* d_q = (double*)dv;
    for (uint64_t k0 = 0; k0 < ns; k0 += chunk) {
        const uint64_t nk = std::min(chunk, ns - k0);
        for (uint64_t k = 0; k < nk; ++k) {
            rc = ising_sim_sweeps(sim, betas.data(), sampling_freq, nullptr);
            if (rc) return rc;
            if (energies) {
                rc = sim_energies_to_device(sim, d_en, nk, k);
                if (rc) return rc;
            }
            if (mags) {
                CUDA_TRY(ctx, cudaMemsetAsync(sim->d_counts, 0, cw * sizeof(unsigned long long), ctx->stream));
                count_launch(sim, launch_count_up(sim->d_spins, sim->lay, sim->d_counts, ctx->stream));
                // M = 2 up - N = -(N - 2 up)
                count_launch(sim, launch_energy_from_nsat(sim->d_counts, E, -1.0, N, 2, d_m, nk, k, ctx->stream));
            }
            if (overlaps && P) {
                CUDA_TRY(ctx, cudaMemsetAsync(sim->d_counts, 0, cw * sizeof(unsigned long long), ctx->stream));
                count_launch(sim, launch_count_up(sim->d_spins, sim->lay, sim->d_counts, ctx->stream, true));
                count_launch(sim, launch_overlap_from_counts(sim->d_counts, P, N, d_q, nk, k, ctx->stream));
            }
        }
        if (energies)
            CUDA_TRY(ctx, copy_rows_d2h(energies + k0, (size_t)ns * 8, d_en, (size_t)nk * 8, (size_t)nk * 8, E,
                                        ctx->stream));
        if (mags)
            CUDA_TRY(ctx, copy_rows_d2h(mags + k0, (size_t)ns * 8, d_m, (size_t)nk * 8, (size_t)nk * 8, E,
                                        ctx->stream));
        if (overlaps && P)
            CUDA_TRY(ctx, copy_rows_d2h(overlaps + k0, (size_t)ns * 8, d_q, (size_t)nk * 8, (size_t)nk * 8, P,
                                        ctx->stream));
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return ISING_OK;
}

extern "C" int ising_run_monte_carlo_sampling(ising_ctx* ctx, const ising_graph* g,
                                              const ising_run_args* a, double* energies,
                                              uint8_t* states) {
    CtxLock _lk(ctx);
    int rc = check_run_args(ctx, g, a, energies, states);
    if (rc) return rc;
    if (a->sampling_freq == 0)
        return fail(ctx, ISING_E_INVALID, "sampling_freq must be > 0 (the reference divides by it)");
    if (a->num_experiments == 0) return ISING_OK;
    ising_sim* sim = nullptr;
    rc = make_sim_for_run(ctx, g, a, &sim);
    if (rc) return rc;
    rc = ising_sim_run_sampling(sim, a->beta, a->thermalization, a->sampling_freq,
                                a->timesteps / a->sampling_freq, energies, states);
    ising_sim_destroy(sim);
    return rc;
}

extern "C" int ising_run_monte_carlo_annealing(ising_ctx* ctx, const ising_graph* g,
                                               const ising_run_args* a, double* energies,
                                               uint8_t* states) {
    CtxLock _lk(ctx);
    int rc = check_run_args(ctx, g, a, energies, states);
    if (rc) return rc;
    if (a->sched_len && (!a->sched_t || !a->sched_beta))
        return fail(ctx, ISING_E_INVALID, "schedule arrays are NULL");
    std::vector<double> betas(a->timesteps);
    if (!schedule_betas(a->sched_t, a->sched_beta, a->sched_len, a->timesteps,
                        (a->flags & ISING_FLAG_LINEAR_SCHEDULE) != 0, betas.data()))
        return fail(ctx, ISING_E_INVALID, "annealing schedule has fewer than two stops");
    if (a->num_experiments == 0) return ISING_OK;
    ising_sim* sim = nullptr;
    rc = make_sim_for_run(ctx, g, a, &sim);
    if (rc) return rc;
    if (a->flags & ISING_FLAG_PER_STEP_ENERGIES) {
        rc = ising_sim_sweeps(sim, betas.data(), a->timesteps, energies);
    } else {
        rc = ising_sim_sweeps(sim, betas.data(), a->timesteps, nullptr);
        if (rc == ISING_OK) rc = ising_sim_get_energies(sim, energies);
    }
    if (rc == ISING_OK) rc = ising_sim_get_states(sim, states);
    ising_sim_destroy(sim);
    return rc;
}

// ------------------------------------------------------------------------------------------
// replay
// ------------------------------------------------------------------------------------------
extern "C" int ising_replay(ising_ctx* ctx, const ising_graph* g, double beta, uint64_t E,
                            uint64_t A, const uint32_t* sites, const double* u,
                            const uint8_t* init, double* energies, uint8_t* states) {
    CtxLock _lk(ctx);
    if (!ctx || !g) return fail(ctx, ISING_E_INVALID, "ctx/graph is NULL");
    if (g->h.field_graph)
        return fail(ctx, ISING_E_UNSUPPORTED, "replay does not take the field of a torus (give it as biases of an edge list)");
    if (E == 0) return ISING_OK;
    if (!init || !energies || !states || (A && (!sites || !u)))
        return fail(ctx, ISING_E_INVALID, "replay buffers are NULL");
    const uint64_t N = g->h.nvars;
    for (uint64_t i = 0; i < E * A; ++i)
        if (sites[i] >= N) return fail(ctx, ISING_E_INVALID, "trace site %u out of range", sites[i]);
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    int rc = ensure_csr_on_device(ctx, const_cast<ising_graph*>(g));
    if (rc) return rc;
    uint32_t* d_sites = nullptr;
    double* d_u = nullptr;
    uint8_t* d_states = nullptr;
    double* d_en = nullptr;
    unsigned int* d_amb = nullptr;
    cudaError_t e = dev_alloc(&d_sites, E * A);
    if (e == cudaSuccess) e = dev_alloc(&d_u, E * A);
    if (e == cudaSuccess) e = dev_alloc(&d_states, E * N);
    if (e == cudaSuccess) e = dev_alloc(&d_en, E);
    if (e == cudaSuccess) e = dev_alloc(&d_amb, 1);
    unsigned int amb = 0;
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_sites, sites, E * A * 4, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_u, u, E * A * 8, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_states, init, E * N, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_amb, 0, sizeof(unsigned int), ctx->stream);
    if (e == cudaSuccess) {
        ReplayArgs ra;
        ra.E = E; ra.N = N; ra.A = A;
        ra.row = g->d_row; ra.nbr = g->d_nbr; ra.jv = g->d_jv; ra.bias = g->d_bias;
        ra.sites = d_sites; ra.u = d_u; ra.states = d_states; ra.energies = d_en;
        ra.beta = beta; ra.ambiguous = d_amb;
        if (launch_replay(ra, ctx->stream) < 0) e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(states, d_states, E * N, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(energies, d_en, E * 8, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(&amb, d_amb, sizeof amb, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(d_sites); cudaFree(d_u); cudaFree(d_states); cudaFree(d_en); cudaFree(d_amb);
    CUDA_TRY(ctx, e);
    if (amb)
        return fail(ctx, ISING_E_AMBIGUOUS,
                    "%u replayed decisions had u within 4e-15 of exp(-beta dE); not certified", amb);
    return ISING_OK;
}
