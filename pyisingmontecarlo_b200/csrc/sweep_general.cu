// sm_100a kernels: colour-class sweeps on arbitrary graphs (K4), per-replica threshold tables for
// parallel tempering, energies on CSR graphs, float-field sweeps for real couplings and biases.
#include "msc_device.cuh"

namespace ising {

// ------------------------------------------------------------------------------------------
// K4: colour-class sweep on an arbitrary graph (CSR/ELL), all |J| equal, no bias.
// Same decision rule and Philox stream as the stencil kernel (DESIGN.md "Production sweep"),
// generic in the degree: n_sat is a 4-plane vertical counter, the uphill classes are
// n_sat = deg/2+1 .. deg.  PERBETA: thresholds differ per replica (parallel tempering).
// ------------------------------------------------------------------------------------------
// DEG > 0: compile-time degree (neighbour loads unrolled and in flight together); DEG = 0: runtime.
// V consecutive replica words of a site per thread: one index load / address computation and one
// 4V-byte gather per neighbour for V words (needs W % V == 0).
#ifndef ISING_GEN_MINB
#define ISING_GEN_MINB 4   // resident blocks per SM the general sweep is compiled for
#endif
template <int K, int ROUNDS, bool PERBETA, int DEG, int V>
__global__ void __launch_bounds__(256, ISING_GEN_MINB)
k_sweep_general(uint32_t* __restrict__ spins, GenGroup g, uint32_t W, uint32_t sweep, PhiloxKeys pk,
                uint32_t gw0, GenThresholds th, GenTables tab) {
    constexpr int NCALL = K / 4 + 1;
    // planes of the n_sat counter: enough for DEG when it is known at compile time
    constexpr int NPL = DEG == 0 ? 4 : (DEG < 2 ? 1 : (DEG < 4 ? 2 : (DEG < 8 ? 3 : 4)));
    const uint32_t deg = DEG > 0 ? (uint32_t)DEG : g.deg;
    const uint32_t cmin = deg / 2 + 1, ncls = deg - deg / 2;
    // Programmatic dependent launch (as the row walk, sweep_rows.cuh): the next colour group may be
    // scheduled while this one drains; the graph arrays of this thread's first site - constant data -
    // are pulled towards the SM before the wait, the spins are not touched until after it.
    asm volatile("griddepcontrol.launch_dependents;");
    {
        const uint32_t i0 = blockIdx.x * blockDim.y + threadIdx.y;
        if (i0 < g.count) {
            asm volatile("prefetch.global.L2 [%0];" ::"l"(g.sites + i0));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(g.anti + i0));
            for (uint32_t k = 0; k < deg; ++k) asm volatile("prefetch.global.L2 [%0];" ::"l"(g.nbr + (size_t)k * g.count + i0));
        }
    }
    asm volatile("griddepcontrol.wait;" ::: "memory");
    // block = (wx lanes over replica word groups, by over sites): no division to split an item index
    for (uint32_t i = blockIdx.x * blockDim.y + threadIdx.y; i < g.count; i += gridDim.x * blockDim.y)
    for (uint32_t w0 = threadIdx.x * V; w0 < W; w0 += blockDim.x * V) {
        const uint32_t n = g.sites[i];
        const uint32_t ab = g.anti[i];
        uint32_t sv[V];
        load_words<V>(spins + (size_t)n * W + w0, sv);
        uint32_t cntv[V][4];
#pragma unroll
        for (int v = 0; v < V; ++v)
#pragma unroll
            for (int l = 0; l < 4; ++l) cntv[v][l] = 0;
        if constexpr (DEG > 0) {
            uint32_t x[DEG][V];
#pragma unroll
            for (int k = 0; k < DEG; ++k)
                load_words<V>(spins + (size_t)g.nbr[(size_t)k * g.count + i] * W + w0, x[k]);
#pragma unroll
            for (int k = 0; k < DEG; ++k) {
                const uint32_t m = 0u - ((ab >> k) & 1u);
#pragma unroll
                for (int v = 0; v < V; ++v) {
                    uint32_t c = ~(sv[v] ^ x[k][v] ^ m);  // satisfied bond
#pragma unroll
                    for (int l = 0; l < NPL; ++l) {
                        const uint32_t t = cntv[v][l] & c;
                        cntv[v][l] ^= c;
                        c = t;
                    }
                }
            }
        } else {
            for (uint32_t k = 0; k < deg; ++k) {
                const uint32_t nb = g.nbr[(size_t)k * g.count + i];
                uint32_t x[V];
                load_words<V>(spins + (size_t)nb * W + w0, x);
                const uint32_t m = 0u - ((ab >> k) & 1u);
#pragma unroll
                for (int v = 0; v < V; ++v) {
                    uint32_t c = ~(sv[v] ^ x[v] ^ m);  // satisfied bond
#pragma unroll
                    for (int l = 0; l < 4; ++l) {
                        const uint32_t t = cntv[v][l] & c;
                        cntv[v][l] ^= c;
                        c = t;
                    }
                }
            }
        }
#pragma unroll
        for (int v = 0; v < V; ++v) {
        const uint32_t w = w0 + v;
        const uint32_t (&cnt)[4] = cntv[v];
        // one-hot masks of the uphill classes
        uint32_t oh[GEN_MAX_CLS];
        uint32_t up = 0;
#pragma unroll
        for (int j = 0; j < GEN_MAX_CLS; ++j) {
            oh[j] = 0;
            if ((uint32_t)j < ncls) {
                const uint32_t val = cmin + j;
                uint32_t o = 0xFFFFFFFFu;
#pragma unroll
                for (int l = 0; l < NPL; ++l) o &= ((val >> l) & 1u) ? cnt[l] : ~cnt[l];
                oh[j] = o;
                up |= o;
            }
        }
        uint32_t r[NCALL * 4];
#pragma unroll
        for (int q = 0; q < NCALL; ++q) {
            const u32x4 o = philox4x32_keys<ROUNDS>(n, gw0 + w, sweep, (uint32_t)q | (TAG_ACCEPT << 24), pk);
            r[4 * q + 0] = o.x; r[4 * q + 1] = o.y; r[4 * q + 2] = o.z; r[4 * q + 3] = o.w;
        }
        const uint32_t* tp = PERBETA ? tab.plane + ((size_t)deg * W + w) * GEN_MAX_CLS * 8 : nullptr;
        uint32_t eq = up, borrow = 0;
#pragma unroll
        for (int p = K - 1; p >= 0; --p) {
            uint32_t t = 0;
#pragma unroll
            for (int j = 0; j < GEN_MAX_CLS; ++j)
                if ((uint32_t)j < ncls) t |= oh[j] & (PERBETA ? __ldg(tp + j * 8 + p) : th.plane[j][p]);
            borrow = maj3(~r[p], t, borrow);
            eq &= ~(r[p] ^ t);
        }
        uint32_t flip = ~up | (borrow & ~eq);
        // tied bits: the first SPARE in straight-line code on the words left over from the calls
        // above (as in msc_flip_mask), the rare rest in a loop
        constexpr int SPARE = (4 * NCALL - K) < 2 ? (4 * NCALL - K) : 2;
#pragma unroll
        for (int j2 = 0; j2 < SPARE; ++j2) {
            const uint32_t bit = eq & (0u - eq);
            const int b = (__ffs((int)eq) - 1) & 31;
            uint32_t cls = 0;
#pragma unroll
            for (int j = 1; j < GEN_MAX_CLS; ++j)
                if ((uint32_t)j < ncls && (oh[j] & bit)) cls = j;
            uint32_t lo;
            if (PERBETA) {
                lo = __ldg(tab.low + ((size_t)deg * 32 * W + (size_t)w * 32 + b) * GEN_MAX_CLS + cls);
            } else {
                lo = th.low[0];
#pragma unroll
                for (int j = 1; j < GEN_MAX_CLS; ++j)
                    if (cls == (uint32_t)j) lo = th.low[j];
            }
            if (r[K + j2] < lo) flip |= bit;
            eq ^= bit;
        }
        if (eq) {
            int jj = K + SPARE;
            u32x4 cur = {r[4 * (NCALL - 1)], r[4 * (NCALL - 1) + 1], r[4 * (NCALL - 1) + 2],
                         r[4 * (NCALL - 1) + 3]};
            do {
                const int b = __ffs((int)eq) - 1;
                if ((jj & 3) == 0 && jj >= 4 * NCALL)
                    cur = philox4x32_more(cur, (uint32_t)(ROUNDS + (jj >> 2) - NCALL), pk.k[0], pk.k[1]);
                const int m = jj & 3;
                const uint32_t val = m == 0 ? cur.x : (m == 1 ? cur.y : (m == 2 ? cur.z : cur.w));
                uint32_t cls = 0;
#pragma unroll
                for (int j = 1; j < GEN_MAX_CLS; ++j)
                    if ((oh[j] >> b) & 1u) cls = j;
                const uint32_t lo = PERBETA
                    ? __ldg(tab.low + ((size_t)deg * 32 * W + (size_t)w * 32 + b) * GEN_MAX_CLS + cls)
                    : th.low[cls];
                if (val < lo) flip |= 1u << b;
                eq &= eq - 1;
                ++jj;
            } while (eq);
        }
        sv[v] ^= flip;
        }
        store_words<V>(spins + (size_t)n * W + w0, sv);
    }
}

template <int K, int ROUNDS, int DEG, int V>
static void gen_launch(const GenSweepArgs& a, const GenGroup& g, cudaStream_t st) {
    const uint32_t groups = a.W / V;
    const uint32_t wx = groups >= 32 ? 32 : pow2_ceil(groups);
    const dim3 block(wx, 256 / wx, 1);
    uint64_t blocks = ((uint64_t)g.count + block.y - 1) / block.y;
    if (blocks > (uint64_t)device_sms() * 16) blocks = (uint64_t)device_sms() * 16;
    const dim3 grid((unsigned)blocks);
    const PhiloxKeys pk = philox_round_keys(a.key0, a.key1);
    if (a.tables.plane != nullptr)
        launch_pdl_v(k_sweep_general<K, ROUNDS, true, DEG, V>, grid, block, 0, st, a.spins, g, a.W, a.sweep, pk, a.gw0,
                     a.th, a.tables);
    else
        launch_pdl_v(k_sweep_general<K, ROUNDS, false, DEG, V>, grid, block, 0, st, a.spins, g, a.W, a.sweep, pk, a.gw0,
                     a.th, a.tables);
}

// degree-specialised kernels only for the default (K, rounds)
template <int K, int ROUNDS, int V>
static void gen_launch_degree(const GenSweepArgs& a, const GenGroup& g, cudaStream_t st) {
    if constexpr (K == 6 && ROUNDS == kDefaultRounds) {
        if (g.deg == 3) return gen_launch<K, ROUNDS, 3, V>(a, g, st);
        if (g.deg == 4) return gen_launch<K, ROUNDS, 4, V>(a, g, st);
        if (g.deg == 6) return gen_launch<K, ROUNDS, 6, V>(a, g, st);
    }
    gen_launch<K, ROUNDS, 0, V>(a, g, st);
}

template <int K, int ROUNDS>
static void gen_launch_vec(const GenSweepArgs& a, const GenGroup& g, cudaStream_t st) {
    if (a.W % 2 == 0) gen_launch_degree<K, ROUNDS, 2>(a, g, st);
    else gen_launch_degree<K, ROUNDS, 1>(a, g, st);
}

int launch_sweep_general(const GenSweepArgs& a, const GenGroup& g, cudaStream_t st) {
    if (g.count == 0) return 0;
    if (g.deg > (uint32_t)GEN_MAX_DEG) return -1;
#define GEN_ROUNDS(KK)                                                                            \
    do { if (a.rounds == 7) gen_launch_vec<KK, 7>(a, g, st); else gen_launch_vec<KK, 10>(a, g, st); } while (0)
    switch (a.planes) {
        case 5: GEN_ROUNDS(5); break;
        case 6: GEN_ROUNDS(6); break;
        case 7: GEN_ROUNDS(7); break;
        default: return -1;
    }
#undef GEN_ROUNDS
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

// per-replica threshold tables from host-computed 64-bit thresholds (integer work only, so the
// bits are exactly the host's): T64[(slot * (GEN_MAX_DEG+1) + deg) * GEN_MAX_CLS + cls]
// one warp per (degree, word, class); lane b = replica bit b, plane masks by ballot
__global__ void k_build_tables(const unsigned long long* __restrict__ t64,
                               const uint32_t* __restrict__ slot_of_replica, uint32_t W, int K,
                               uint32_t* __restrict__ plane_out, uint32_t* __restrict__ low_out) {
    const uint32_t total = (GEN_MAX_DEG + 1) * W * GEN_MAX_CLS;
    const uint32_t b = threadIdx.x & 31u;
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t idx = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; idx < total; idx += warps) {
        const uint32_t cls = idx % GEN_MAX_CLS;
        const uint32_t w = (idx / GEN_MAX_CLS) % W;
        const uint32_t deg = idx / (GEN_MAX_CLS * W);
        const uint32_t e = w * 32 + b;
        const uint32_t slot = slot_of_replica[e];
        const unsigned long long T = t64[((size_t)slot * (GEN_MAX_DEG + 1) + deg) * GEN_MAX_CLS + cls];
        low_out[((size_t)deg * 32 * W + e) * GEN_MAX_CLS + cls] = (uint32_t)(T & 0xFFFFFFFFull);
        uint32_t mine = 0;  // lane p keeps plane p
        for (int p = 0; p < 8; ++p) {
            const uint32_t m = p < K ? __ballot_sync(0xFFFFFFFFu, (T >> (K + 31 - p)) & 1ull) : 0u;
            if (b == (uint32_t)p) mine = m;
        }
        if (b < 8) plane_out[(((size_t)deg * W + w) * GEN_MAX_CLS + cls) * 8 + b] = mine;
    }
}

// stencil variant: T64[e * 3 + cls] per replica -> tplane[(w * 3 + cls) * 8 + p], tlow[(e) * 3 + cls]
__global__ void k_build_tables_stencil(const unsigned long long* __restrict__ t64,
                                       const uint32_t* __restrict__ slot_of_replica, uint32_t W, int K,
                                       uint32_t* __restrict__ plane_out, uint32_t* __restrict__ low_out) {
    const uint32_t b = threadIdx.x & 31u;
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t idx = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; idx < W * 3; idx += warps) {
        const uint32_t cls = idx % 3, w = idx / 3;
        const uint32_t e = w * 32 + b;
        const uint32_t row = slot_of_replica ? slot_of_replica[e] : e;
        const unsigned long long T = t64[(size_t)row * 3 + cls];
        low_out[(size_t)e * 3 + cls] = (uint32_t)(T & 0xFFFFFFFFull);
        uint32_t mine = 0;
        for (int p = 0; p < 8; ++p) {
            const uint32_t m = p < K ? __ballot_sync(0xFFFFFFFFu, (T >> (K + 31 - p)) & 1ull) : 0u;
            if (b == (uint32_t)p) mine = m;
        }
        if (b < 8) plane_out[((size_t)w * 3 + cls) * 8 + b] = mine;
    }
}

int launch_build_tables_stencil(const unsigned long long* t64, const uint32_t* slot_of_replica, uint32_t W,
                                int K, uint32_t* plane_out, uint32_t* low_out, cudaStream_t st) {
    const uint32_t blocks = (W * 3 + 3) / 4;   // 4 warps per block
    const uint32_t cap = device_sms() * 8u;
    k_build_tables_stencil<<<blocks < cap ? blocks : cap, 128, 0, st>>>(t64, slot_of_replica, W, K, plane_out,
                                                                        low_out);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

int launch_build_tables(const unsigned long long* t64, const uint32_t* slot_of_replica, uint32_t W,
                        int K, uint32_t* plane_out, uint32_t* low_out, cudaStream_t st) {
    const uint32_t total = (GEN_MAX_DEG + 1) * W * GEN_MAX_CLS;
    const uint32_t blocks = (total + 3) / 4;
    const uint32_t cap = device_sms() * 8u;
    k_build_tables<<<blocks < cap ? blocks : cap, 128, 0, st>>>(t64, slot_of_replica, W, K, plane_out, low_out);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

// satisfied bonds per experiment on a general graph (each bond seen from both ends)
__global__ void __launch_bounds__(256)
k_nsat_general(const uint32_t* __restrict__ spins, uint64_t nvars, uint32_t W,
               const uint32_t* __restrict__ row, const uint32_t* __restrict__ nbr,
               const uint8_t* __restrict__ anti, unsigned long long* __restrict__ nsat2) {
    __shared__ int sm[32 * 256];
    const int nthreads = blockDim.x * blockDim.y;
    const int tid = threadIdx.y * blockDim.x + threadIdx.x;
    for (uint32_t w0 = 0; w0 < W; w0 += blockDim.x) {
        for (int b = 0; b < 32; ++b) sm[b * nthreads + tid] = 0;
        const uint32_t w = w0 + threadIdx.x;
        VCount<VC_PLANES> vc;
        vc.clear();
        int pending = 0;
        if (w < W) {
            for (uint64_t n = (uint64_t)blockIdx.x * blockDim.y + threadIdx.y; n < nvars;
                 n += (uint64_t)gridDim.x * blockDim.y) {
                const uint32_t s = spins[(size_t)n * W + w];
                const uint32_t lo = row[n], hi = row[n + 1];
                // satisfied bonds of this site in a 4-plane counter (degree <= 15 on this path),
                // neighbours four at a time so that the gathers are in flight together
                uint32_t cnt[4] = {0, 0, 0, 0};
                for (uint32_t k = lo; k < hi; k += 4) {
                    uint32_t c4[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const bool ok = k + u < hi;
                        const uint32_t x = spins[(size_t)(ok ? nbr[k + u] : n) * W + w];
                        const uint32_t m = (ok && anti[k + u]) ? 0xFFFFFFFFu : 0u;
                        c4[u] = ok ? ~(s ^ x ^ m) : 0u;
                    }
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        uint32_t c = c4[u];
#pragma unroll
                        for (int l = 0; l < 4; ++l) {
                            const uint32_t t = cnt[l] & c;
                            cnt[l] ^= c;
                            c = t;
                        }
                    }
                }
                vadd<VC_PLANES, 4>(vc.v, cnt);
                pending += 15;
                if (pending > VC_FLUSH_ADD1 - 15) {
                    vc.flush(sm, tid, nthreads);
                    pending = 0;
                }
            }
            vc.flush(sm, tid, nthreads);
        }
        block_reduce_counts(sm, nsat2, w0, W);
    }
}

int launch_nsat_general(const uint32_t* spins, uint64_t nvars, uint32_t W, const uint32_t* row,
                        const uint32_t* nbr, const uint8_t* anti, unsigned long long* nsat2,
                        cudaStream_t st) {
    const uint32_t wx = W >= 32 ? 32 : pow2_ceil(W);
    dim3 block(wx, 256 / wx, 1);
    uint64_t g = (nvars + block.y - 1) / block.y;
    if (g > device_sms() * 8u) g = device_sms() * 8u;
    if (g == 0) g = 1;
    k_nsat_general<<<dim3((unsigned)g), block, 0, st>>>(spins, nvars, W, row, nbr, anti, nsat2);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

// ------------------------------------------------------------------------------------------
// Colour-class sweep for arbitrary real couplings and biases (lattice.rs:31, 104-131): the local
// field is not an integer class, so every replica bit gets its own float field, its own
// exp(-beta dE) and its own 32-bit uniform (word b%4 of Philox call b/4 on the usual counter).
// dE = -2 s_i sum_k J_ik s_k + 2 b_i s_i  (qmc GraphState::do_spin_flip); accept iff dE <= 0 or
// R < floor(exp(-beta dE) 2^32).  Not bit-exact against f64 (f32 field, __expf): every decision
// outside the rounding band of those equals the f64 reference's (tests/float_reference.py).
// ------------------------------------------------------------------------------------------
template <int ROUNDS>
__global__ void __launch_bounds__(256)
k_sweep_real(RealSweepArgs a) {
    for (uint32_t i = blockIdx.x * blockDim.y + threadIdx.y; i < a.count; i += gridDim.x * blockDim.y)
    for (uint32_t w = threadIdx.x; w < a.W; w += blockDim.x) {
        const uint32_t n = a.sites[i];
        const uint32_t s = a.spins[(size_t)n * a.W + w];
        const uint32_t lo = a.row[n], hi = a.row[n + 1];
        const float bias = a.biasf[n];
        uint32_t flip = 0;
        for (uint32_t b0 = 0; b0 < 32; b0 += 4) {
            const u32x4 r = philox4x32<ROUNDS>(n, a.gw0 + w, a.sweep, (b0 >> 2) | (TAG_ACCEPT << 24),
                                               a.key0, a.key1);
            const uint32_t rr[4] = {r.x, r.y, r.z, r.w};
            float h[4] = {0.f, 0.f, 0.f, 0.f};
            for (uint32_t k = lo; k < hi; ++k) {
                const uint32_t x = a.spins[(size_t)a.nbr[k] * a.W + w] >> b0;
                const uint32_t jb = __float_as_uint(a.jf[k]);
#pragma unroll
                for (int q = 0; q < 4; ++q)  // J * s_k: flip the sign bit where the spin is down
                    h[q] += __uint_as_float(jb ^ ((~(x >> q) & 1u) << 31));
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const float si = ((s >> (b0 + q)) & 1u) ? 1.f : -1.f;
                const float de = 2.f * si * (bias - h[q]);
                bool acc = true;
                if (de > 0.f) {
                    const float beta = a.beta_slots
                        ? (float)__longlong_as_double((long long)__ldg(a.beta_slots + __ldg(a.slot_of_replica + w * 32u + b0 + q)))
                        : a.beta;
                    const float pth = __expf(-beta * de) * 4294967296.f;
                    acc = rr[q] < __float2uint_rz(pth);  // saturating conversion
                }
                if (acc) flip |= 1u << (b0 + q);
            }
        }
        a.spins[(size_t)n * a.W + w] = s ^ flip;
    }
}

int launch_sweep_real(const RealSweepArgs& a, cudaStream_t st) {
    if (a.count == 0) return 0;
    const uint32_t wx = a.W >= 32 ? 32 : pow2_ceil(a.W);
    const dim3 block(wx, 256 / wx, 1);
    uint64_t blocks = ((uint64_t)a.count + block.y - 1) / block.y;
    if (blocks > (uint64_t)device_sms() * 16) blocks = (uint64_t)device_sms() * 16;
    if (a.rounds == 7) k_sweep_real<7><<<(unsigned)blocks, block, 0, st>>>(a);
    else k_sweep_real<10><<<(unsigned)blocks, block, 0, st>>>(a);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

__global__ void __launch_bounds__(256)
k_energy_real(const uint32_t* __restrict__ spins, uint64_t nvars, uint32_t W,
              const uint32_t* __restrict__ row, const uint32_t* __restrict__ nbr,
              const double* __restrict__ jv, const double* __restrict__ bias,
              double* __restrict__ energies) {
    // block = (wx word columns, by site lanes); each thread keeps 32 f64 partial energies
    const uint32_t w = blockIdx.y * blockDim.x + threadIdx.x;
    if (w >= W) return;
    double acc[32];
#pragma unroll
    for (int b = 0; b < 32; ++b) acc[b] = 0.0;
    for (uint64_t n = (uint64_t)blockIdx.x * blockDim.y + threadIdx.y; n < nvars;
         n += (uint64_t)gridDim.x * blockDim.y) {
        const uint32_t s = spins[(size_t)n * W + w];
        const double bi = bias[n];
        for (uint32_t k = row[n]; k < row[n + 1]; ++k) {
            const uint32_t eqm = ~(s ^ spins[(size_t)nbr[k] * W + w]);  // 1 where s_i == s_k
            const double hj = 0.5 * jv[k];
#pragma unroll
            for (int b = 0; b < 32; ++b) acc[b] += ((eqm >> b) & 1u) ? hj : -hj;
        }
#pragma unroll
        for (int b = 0; b < 32; ++b) acc[b] += ((s >> b) & 1u) ? -bi : bi;
    }
#pragma unroll
    for (int b = 0; b < 32; ++b) atomicAdd(energies + (size_t)w * 32 + b, acc[b]);
}

int launch_energy_real(const uint32_t* spins, uint64_t nvars, uint32_t W, const uint32_t* row,
                       const uint32_t* nbr, const double* jv, const double* bias, double* energies,
                       cudaStream_t st) {
    const uint32_t wx = W >= 32 ? 32 : pow2_ceil(W);
    dim3 block(wx, 128 / wx, 1);
    uint64_t g = (nvars + block.y - 1) / block.y;
    if (g > device_sms() * 4u) g = device_sms() * 4u;
    if (g == 0) g = 1;
    dim3 grid((unsigned)g, (W + wx - 1) / wx, 1);
    k_energy_real<<<grid, block, 0, st>>>(spins, nvars, W, row, nbr, jv, bias, energies);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

}  // namespace ising
