// sm_100a kernels: one large 2D lattice bit-packed along x in row strips (K7).
#include "sweep_rows.cuh"

namespace ising {

// ------------------------------------------------------------------------------------------
// K7: one large 2D lattice bit-packed along x (config 5).  Same decision rule as the replica-
// packed kernels; here the 32 bits of a word are 32 same-colour sites of one row, so the two
// x neighbours are the other-colour word at the same index and that word funnel-shifted by one
// bit (carry from the adjacent word).  Philox counter = (global row, colour << 30 | word, sweep,
// call): a draw does not depend on how rows are split into strips.
// ------------------------------------------------------------------------------------------
// V consecutive words of a row per thread (128-bit loads when V == 4; needs Wr % V == 0).  The
// site update is the row walk's (sweep_rows.cuh: update_site): Philox rounds 1-3 shared over the
// V words and both calls (counter = (row, colour << 30 | word, sweep, call), i.e. the words of a
// thread differ in counter word 1 only), threshold planes selected with IMAD, rare ties deferred.
template <int K, int ROUNDS, int V>
__global__ void __launch_bounds__(256, 3)
k_strip_phase(uint32_t* __restrict__ spins, const __grid_constant__ StripGeom g, uint32_t c, uint32_t sweep,
              const __grid_constant__ PhiloxKeys pk, uint32_t antiferro, const __grid_constant__ MscMux mx,
              uint32_t r_begin, uint32_t r_count) {
    const uint32_t groups = g.Wr / V;
    const uint32_t o = 1u - c;
    VCount<1> unused[V];
    // programmatic dependent launch: the next phase is scheduled while this one drains
    asm volatile("griddepcontrol.launch_dependents;");
    asm volatile("griddepcontrol.wait;" ::: "memory");
    // block = (x over the word groups of a row, y over rows): storage rows [r_begin, r_begin + r_count)
    for (uint32_t rr = blockIdx.y * blockDim.y + threadIdx.y; rr < r_count; rr += gridDim.y * blockDim.y)
    for (uint32_t jg = blockIdx.x * blockDim.x + threadIdx.x; jg < groups; jg += gridDim.x * blockDim.x) {
        const uint32_t j = jg * V;
        const uint32_t r = r_begin + rr;
        const uint32_t y = strip_global_row(g, r);
        const uint32_t p = (y + c) & 1u;
        uint32_t s[V], n[4][V];
        uint32_t* own = strip_load_site<V>(spins, g, c, o, r, j, p, s, n);
        const uint32_t m[4] = {antiferro, antiferro, antiferro, antiferro};
        update_site<2, K, ROUNDS, V, false>(s, n, m, y, (c << 30) | j, sweep, pk, mx, unused);
        store_words<V>(own, s);
    }
}

template <int V>
static int strip_phase_dispatch(const StripSweepArgs& a, cudaStream_t st) {
    dim3 grid, block;
    strip_phase_shape(a, V, &grid, &block);
#define STRIP_LAUNCH(KK, RR)                                                                     \
    launch_pdl_v(k_strip_phase<KK, RR, V>, grid, block, 0, st, a.spins, a.g, a.colour, a.sweep,    \
                 philox_round_keys(a.key0, a.key1), a.antiferro, make_mux(a.th), a.r_begin, a.r_count)
#define STRIP_ROUNDS(KK)                                                                         \
    do { if (a.rounds == 7) STRIP_LAUNCH(KK, 7); else STRIP_LAUNCH(KK, 10); } while (0)
    switch (a.planes) {
        case 5: STRIP_ROUNDS(5); break;
        case 6: STRIP_ROUNDS(6); break;
        case 7: STRIP_ROUNDS(7); break;
        default: return -1;
    }
#undef STRIP_ROUNDS
#undef STRIP_LAUNCH
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

int launch_strip_phase(const StripSweepArgs& a, cudaStream_t st) {
    if (a.r_count == 0 || a.g.Wr == 0) return 0;
    // rows are 16-byte aligned when Wr % 4 == 0 (every row starts at a multiple of Wr words)
    if (a.g.Wr % 4 == 0) return strip_phase_dispatch<4>(a, st);
    if (a.g.Wr % 2 == 0) return strip_phase_dispatch<2>(a, st);
    return strip_phase_dispatch<1>(a, st);
}

// block = (x over the V-word groups of a row, y over rows), 256 threads; at most 64 blocks along x
// and 32 blocks per SM in all: the kernels stride over what the grid does not cover
void strip_phase_shape(const StripSweepArgs& a, uint32_t V, dim3* grid, dim3* block) {
    const uint32_t groups = a.g.Wr / V;
    const uint32_t bx = groups >= 256 ? 256 : pow2_ceil(groups);
    *block = dim3(bx, 256 / bx, 1);
    uint32_t gx = (groups + bx - 1) / bx;
    if (gx > 64) gx = 64;
    uint32_t gy = (a.r_count + block->y - 1) / block->y;
    const uint32_t gy_cap = (device_sms() * 32u + gx - 1) / gx;
    if (gy > gy_cap) gy = gy_cap;
    *grid = dim3(gx, gy, 1);
}

// ------------------------------------------------------------------------------------------
// Both colour phases of a sweep in ONE pass over the lattice (temporal blocking, out of place).
// OPT-IN (ISING_STRIP_FUSE=1): it cuts the DRAM traffic of the 65536^2 lattice from 1.43x to ~1.0x
// the algorithmic bytes and is bit-identical, but it is SLOWER than the two phase launches -
// 4.49 (rows staged by TMA) / 4.34 (rows loaded by the warps) / 3.62 (neighbour-warp flags instead
// of the row barrier) against 4.82 x 10^12 flips/s (profiles/r02_strip_fused_ab.log): the kernel is
// bound by the integer pipes, not by HBM, and the row-by-row dependence of colour 1 on colour 0
// takes away the freedom of 24 independent warps per SM that the phase kernel has.
//
// The two-launch sweep reads both colours and writes one per phase: 6 bits of DRAM traffic per
// site and sweep for a lattice that does not fit the L2 (profiles/r02_traffic.json: 1.43x the
// algorithmic 4 bits).  Here a block owns a band of rows and walks down it: it updates colour 0
// of row r from the OLD colour-1 rows r-1, r, r+1 (read from `src`), keeps the new row in a
// four-slot ring in shared memory, and then updates colour 1 of row r-1 from the NEW colour-0
// rows r-2, r-1, r in the ring.  Every word is read once from `src` and written once to `dst`.
// Bands are independent: the new colour-0 rows just outside a band (a-1 and e) are computed
// redundantly and not written - a draw is a function of the global row, so both owners agree
// (the argument that makes the deep halo exchange between GPUs work, DESIGN.md 7).  Writing to
// a second array keeps the old rows intact for the neighbouring bands.
//   colour 0: storage rows [r0, r0 + n0);  colour 1: [r0 + 1, r0 + n0 - 1)
// block = (bx word groups of a row) x (by bands); a thread keeps its word group.
// ------------------------------------------------------------------------------------------
template <int K, int ROUNDS, int V>
__global__ void __launch_bounds__(256, 3)
k_strip_sweep_fused(const uint32_t* __restrict__ src, uint32_t* __restrict__ dst, const __grid_constant__ StripGeom g,
                    uint32_t sweep, const __grid_constant__ PhiloxKeys pk, uint32_t antiferro,
                    const __grid_constant__ MscMux mx, uint32_t r0, uint32_t n0, uint32_t nbands) {
    extern __shared__ uint32_t ring_all[];                       // [by][4][Wr]
    const uint32_t Wr = g.Wr;
    uint32_t* ring = ring_all + (size_t)threadIdx.y * 4u * Wr;
    const uint32_t band = blockIdx.x * blockDim.y + threadIdx.y;
    const uint32_t q = n0 / nbands, rem = n0 % nbands;
    const bool live = band < nbands;
    const uint32_t a = r0 + band * q + (band < rem ? band : rem);   // colour-0 rows [a, e) are this band's
    const uint32_t e = live ? a + q + (band < rem ? 1u : 0u) : a;
    const uint32_t j = threadIdx.x * V;
    const bool col = live && j < Wr;
    const uint32_t jp = j + V == Wr ? 0u : j + V, jm = j == 0 ? Wr - V : j - V;   // first word of the next / previous group
    VCount<1> unused[V];
    const uint32_t m[4] = {antiferro, antiferro, antiferro, antiferro};
    const uint32_t end0 = r0 + n0;
    // q + 3 steps for every band (bands of q and q + 1 rows share the barriers)
    for (uint32_t it = 0; it < q + 3; ++it) {
        const uint32_t r = a + it - 1u;                            // colour-0 row of this step (a - 1 .. e)
        if (col && r + 1u >= a && r <= e && r >= r0 && r < end0) {
            const uint32_t y = strip_global_row(g, r);
            const uint32_t p = y & 1u;
            uint32_t s[V], n[4][V];
            const uint32_t* orow = src + strip_off(g, 1, r, 0);
            load_words<V>(src + strip_off(g, 0, r, j), s);
            load_words<V>(orow + j, n[0]);
            load_words<V>(orow + j - Wr, n[2]);
            load_words<V>(orow + j + Wr, n[3]);
            const uint32_t edge = p ? orow[jp] : orow[jm + V - 1];
#pragma unroll
            for (int v = 0; v < V; ++v) {
                if (p) n[1][v] = __funnelshift_r(n[0][v], v + 1 < V ? n[0][v + 1 < V ? v + 1 : v] : edge, 1);
                else n[1][v] = __funnelshift_l(v > 0 ? n[0][v > 0 ? v - 1 : 0] : edge, n[0][v], 1);
            }
            update_site<2, K, ROUNDS, V, false>(s, n, m, y, j, sweep, pk, mx, unused);
            store_words<V>(ring + (r & 3u) * Wr + j, s);
            if (r >= a && r < e) store_words<V>(dst + strip_off(g, 0, r, j), s);
        }
        __syncthreads();
        const uint32_t r1 = r - 1u;                                // colour-1 row of this step (a .. e - 1)
        if (col && it >= 2u && r1 < e && r1 > r0 && r1 + 1u < end0) {
            const uint32_t y = strip_global_row(g, r1);
            const uint32_t p = (y + 1u) & 1u;
            uint32_t s[V], n[4][V];
            const uint32_t* nrow = ring + (r1 & 3u) * Wr;
            load_words<V>(src + strip_off(g, 1, r1, j), s);
            load_words<V>(nrow + j, n[0]);
            load_words<V>(ring + ((r1 - 1u) & 3u) * Wr + j, n[2]);
            load_words<V>(ring + ((r1 + 1u) & 3u) * Wr + j, n[3]);
            const uint32_t edge = p ? nrow[jp] : nrow[jm + V - 1];
#pragma unroll
            for (int v = 0; v < V; ++v) {
                if (p) n[1][v] = __funnelshift_r(n[0][v], v + 1 < V ? n[0][v + 1 < V ? v + 1 : v] : edge, 1);
                else n[1][v] = __funnelshift_l(v > 0 ? n[0][v > 0 ? v - 1 : 0] : edge, n[0][v], 1);
            }
            update_site<2, K, ROUNDS, V, false>(s, n, m, y, (1u << 30) | j, sweep, pk, mx, unused);
            store_words<V>(dst + strip_off(g, 1, r1, j), s);
        }
    }
}

// The same pass with every row staged in shared memory by the TMA unit (cp.async.bulk, completion
// on an mbarrier): the barrier per row makes the warps of a block move in step, so loads issued by
// the warps themselves are not hidden behind other warps' arithmetic the way they are in the
// free-running phase kernel (measured: 4.33 instead of 4.81 x 10^12 flips/s on the 65536^2 lattice).
// Here thread 0 asks for the rows of the NEXT step right after the barrier of the current one:
//   OC1  old colour-1 rows, ring of 4 (row x is read by the colour-0 steps x-1, x, x+1 and as the
//        spin word of colour-1 step x)        OC0  old colour-0 rows, ring of 2
//   NC0  new colour-0 rows, ring of 4 (written by the threads, never by the TMA unit)
// and the compute reads shared memory only.  One band per block, block = the word groups of a row.
template <int K, int ROUNDS>
__global__ void __launch_bounds__(256, 3)
k_strip_sweep_fused_tma(const uint32_t* __restrict__ src, uint32_t* __restrict__ dst, const __grid_constant__ StripGeom g,
                        uint32_t sweep, const __grid_constant__ PhiloxKeys pk, uint32_t antiferro,
                        const __grid_constant__ MscMux mx, uint32_t r0, uint32_t n0, uint32_t nbands) {
    constexpr int V = 4;
    extern __shared__ __align__(128) uint32_t smem_rows[];       // OC1[4][Wr] | OC0[2][Wr] | NC0[4][Wr]
    __shared__ __align__(8) unsigned long long bar_c1[4], bar_c0[2];
    const uint32_t Wr = g.Wr, RB = Wr * 4u;
    uint32_t* oc1 = smem_rows;
    uint32_t* oc0 = smem_rows + 4u * Wr;
    uint32_t* nc0 = smem_rows + 6u * Wr;
    const uint32_t band = blockIdx.x;
    const uint32_t q = n0 / nbands, rem = n0 % nbands;
    const uint32_t a = r0 + band * q + (band < rem ? band : rem);
    const uint32_t e = a + q + (band < rem ? 1u : 0u);
    const uint32_t end0 = r0 + n0;
    const uint32_t c0lo = a - 1u > r0 ? a - 1u : r0;              // colour-0 rows this band computes: [c0lo, c0hi]
    const uint32_t c0hi = e < end0 - 1u ? e : end0 - 1u;
    const uint32_t j = threadIdx.x * V;
    const uint32_t jp = j + V == Wr ? 0u : j + V, jm = j == 0 ? Wr - V : j - V;
    VCount<1> unused[V];
    const uint32_t m[4] = {antiferro, antiferro, antiferro, antiferro};
    const bool producer = threadIdx.x == 0;
    // old colour-1 row x (c0lo - 1 <= x <= c0hi + 1) / old colour-0 row x (c0lo <= x <= c0hi) into their rings
    auto fetch_c1 = [&](uint32_t x) {
        const uint32_t k = x - (c0lo - 1u), bar = smem_u32(&bar_c1[k & 3u]);
        mbar_expect_tx(bar, RB);
        tma_load_1d(smem_u32(oc1 + (k & 3u) * Wr), src + strip_off(g, 1, x, 0), RB, bar);
    };
    auto fetch_c0 = [&](uint32_t x) {
        const uint32_t k = x - c0lo, bar = smem_u32(&bar_c0[k & 1u]);
        mbar_expect_tx(bar, RB);
        tma_load_1d(smem_u32(oc0 + (k & 1u) * Wr), src + strip_off(g, 0, x, 0), RB, bar);
    };
    auto wait_c1 = [&](uint32_t x) {
        const uint32_t k = x - (c0lo - 1u);
        mbar_wait(smem_u32(&bar_c1[k & 3u]), (k >> 2) & 1u);
    };
    if (producer) {
        for (int i = 0; i < 4; ++i) mbar_init(smem_u32(&bar_c1[i]), 1u);
        for (int i = 0; i < 2; ++i) mbar_init(smem_u32(&bar_c0[i]), 1u);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (producer) {   // everything the first colour-0 step reads
        fetch_c1(c0lo - 1u);
        fetch_c1(c0lo);
        fetch_c1(c0lo + 1u);
        fetch_c0(c0lo);
    }
    for (uint32_t r = c0lo; r <= c0hi; ++r) {
        {
            const uint32_t k1 = r - (c0lo - 1u), k0 = r - c0lo;    // ring indices of old rows r (colour 1 / 0)
            if (r == c0lo) { wait_c1(r - 1u); wait_c1(r); }
            wait_c1(r + 1u);
            mbar_wait(smem_u32(&bar_c0[k0 & 1u]), (k0 >> 1) & 1u);
            const uint32_t y = strip_global_row(g, r);
            const uint32_t p = y & 1u;
            uint32_t s[V], n[4][V];
            const uint32_t* orow = oc1 + (k1 & 3u) * Wr;
            load_words<V>(oc0 + (k0 & 1u) * Wr + j, s);
            load_words<V>(orow + j, n[0]);
            load_words<V>(oc1 + ((k1 - 1u) & 3u) * Wr + j, n[2]);
            load_words<V>(oc1 + ((k1 + 1u) & 3u) * Wr + j, n[3]);
            const uint32_t edge = p ? orow[jp] : orow[jm + V - 1];
#pragma unroll
            for (int v = 0; v < V; ++v) {
                if (p) n[1][v] = __funnelshift_r(n[0][v], v + 1 < V ? n[0][v + 1 < V ? v + 1 : v] : edge, 1);
                else n[1][v] = __funnelshift_l(v > 0 ? n[0][v > 0 ? v - 1 : 0] : edge, n[0][v], 1);
            }
            update_site<2, K, ROUNDS, V, false>(s, n, m, y, j, sweep, pk, mx, unused);
            store_words<V>(nc0 + (r & 3u) * Wr + j, s);
            if (r >= a && r < e) store_words<V>(dst + strip_off(g, 0, r, j), s);
        }
        __syncthreads();
        // every thread is past colour-1 step r-2 and colour-0 step r: old colour-1 row r-2 and old
        // colour-0 row r-1 are dead, their slots take the rows of the next step
        if (producer) {
            if (r + 2u <= c0hi + 1u) fetch_c1(r + 2u);
            if (r + 1u <= c0hi) fetch_c0(r + 1u);
        }
        const uint32_t r1 = r - 1u;                                // colour-1 row of this step
        if (r1 >= c0lo + 1u && r1 + 1u <= c0hi && r1 >= a && r1 < e) {
            const uint32_t y = strip_global_row(g, r1);
            const uint32_t p = (y + 1u) & 1u;
            uint32_t s[V], n[4][V];
            const uint32_t* nrow = nc0 + (r1 & 3u) * Wr;
            load_words<V>(oc1 + ((r1 - (c0lo - 1u)) & 3u) * Wr + j, s);
            load_words<V>(nrow + j, n[0]);
            load_words<V>(nc0 + ((r1 - 1u) & 3u) * Wr + j, n[2]);
            load_words<V>(nc0 + ((r1 + 1u) & 3u) * Wr + j, n[3]);
            const uint32_t edge = p ? nrow[jp] : nrow[jm + V - 1];
#pragma unroll
            for (int v = 0; v < V; ++v) {
                if (p) n[1][v] = __funnelshift_r(n[0][v], v + 1 < V ? n[0][v + 1 < V ? v + 1 : v] : edge, 1);
                else n[1][v] = __funnelshift_l(v > 0 ? n[0][v > 0 ? v - 1 : 0] : edge, n[0][v], 1);
            }
            update_site<2, K, ROUNDS, V, false>(s, n, m, y, (1u << 30) | j, sweep, pk, mx, unused);
            store_words<V>(dst + strip_off(g, 1, r1, j), s);
        }
    }
}

// 1 when launched, 0 when the geometry does not fit (caller runs the two colour phases), -1 on error
int launch_strip_sweep_fused(const StripSweepArgs& a, const uint32_t* src, uint32_t* dst, cudaStream_t st) {
    constexpr int V = 4;
    static const bool enabled = getenv("ISING_STRIP_FUSE") != nullptr;
    if (!enabled || a.planes != 6 || a.rounds != kDefaultRounds) return 0;
    if (a.g.Wr % V || a.g.Wr / V > 256u || a.r_count < 4) return 0;
    const uint32_t groups = a.g.Wr / V;
    static const int min_rows = getenv("ISING_STRIP_FUSE_MIN_ROWS") ? atoi(getenv("ISING_STRIP_FUSE_MIN_ROWS")) : 48;
    static const bool no_tma = getenv("ISING_STRIP_NO_TMA") != nullptr;   // A/B knob: rows loaded by the warps
    if (!no_tma && groups >= 32u && (groups & (groups - 1u)) == 0u) {
        // TMA-staged rows: the block is exactly the word groups of a row, one band per block
        auto kt = k_strip_sweep_fused_tma<6, kDefaultRounds>;
        const size_t smem_t = (size_t)10u * a.g.Wr * sizeof(uint32_t);
        static int per_sm_t = 0;
        static size_t per_sm_t_smem = 0;
        static uint32_t per_sm_t_threads = 0;
        if (per_sm_t == 0 || per_sm_t_smem != smem_t || per_sm_t_threads != groups) {
            int n = 0;
            if (cudaFuncSetAttribute(kt, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_t) != cudaSuccess ||
                cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kt, (int)groups, smem_t) != cudaSuccess || n < 1) {
                cudaGetLastError();
                n = -1;
            }
            per_sm_t = n;
            per_sm_t_smem = smem_t;
            per_sm_t_threads = groups;
        }
        if (per_sm_t > 0) {
            uint32_t nb = device_sms() * (uint32_t)per_sm_t;
            if (nb > a.r_count / 2) nb = a.r_count / 2;
            if (nb >= 1 && a.r_count / nb >= (uint32_t)min_rows) {
                kt<<<nb, groups, smem_t, st>>>(src, dst, a.g, a.sweep, philox_round_keys(a.key0, a.key1), a.antiferro,
                                               make_mux(a.th), a.r_begin, a.r_count, nb);
                return cudaGetLastError() == cudaSuccess ? 1 : -1;
            }
        }
    }
    const uint32_t bx = pow2_ceil(groups) < 32u ? 32u : pow2_ceil(groups);
    const uint32_t by = 256u / bx;
    const size_t smem = (size_t)by * 4u * a.g.Wr * sizeof(uint32_t);
    auto kern = k_strip_sweep_fused<6, kDefaultRounds, V>;
    static int per_sm = 0;
    static size_t per_sm_smem = 0;
    if (per_sm == 0 || per_sm_smem != smem) {
        int n = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kern, 256, smem) != cudaSuccess || n < 1) {
            cudaGetLastError();
            return 0;
        }
        per_sm = n;
        per_sm_smem = smem;
    }
    // one resident wave of blocks; a band pays two redundant colour-0 rows, so it must not be short
    uint32_t nbands = device_sms() * (uint32_t)per_sm * by;
    if (nbands > a.r_count / 2) nbands = a.r_count / 2;
    if (nbands < 1 || a.r_count / nbands < (uint32_t)min_rows) return 0;
    const uint32_t blocks = (nbands + by - 1) / by;
    kern<<<blocks, dim3(bx, by, 1), smem, st>>>(src, dst, a.g, a.sweep, philox_round_keys(a.key0, a.key1), a.antiferro,
                                                make_mux(a.th), a.r_begin, a.r_count, nbands);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

__global__ void k_strip_init_random(uint32_t* __restrict__ spins, StripGeom g, uint32_t k0,
                                    uint32_t k1) {
    const uint64_t total = 2ull * g.rows * g.Wr;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t c = (uint32_t)(i / ((uint64_t)g.rows * g.Wr));
        const uint64_t rem = i - (uint64_t)c * g.rows * g.Wr;
        const uint32_t r = (uint32_t)(rem / g.Wr) + g.ghost, j = (uint32_t)(rem % g.Wr);
        const u32x4 v = philox4x32<10>(g.row0 + r - g.ghost, (c << 30) | j, 0u, TAG_INIT << 24, k0, k1);
        spins[strip_off(g, c, r, j)] = v.x;
    }
}

int launch_strip_init_random(uint32_t* spins, const StripGeom& g, uint32_t key0, uint32_t key1,
                             cudaStream_t st) {
    k_strip_init_random<<<device_sms() * 8, 256, 0, st>>>(spins, g, key0, key1);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

// per-lattice observables are plain popcounts in this layout
__global__ void __launch_bounds__(256)
k_strip_observables(const uint32_t* __restrict__ spins, StripGeom g, uint32_t antiferro,
                    unsigned long long* __restrict__ acc) {
    unsigned long long nsat = 0, up = 0;
    const uint64_t total = (uint64_t)g.rows * g.Wr;
    for (uint64_t item = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; item < total;
         item += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t r = (uint32_t)(item / g.Wr) + g.ghost, j = (uint32_t)(item % g.Wr);
        const uint32_t y = g.row0 + r - g.ghost;
        const uint32_t p = y & 1u;  // colour 0
        const uint32_t s = spins[strip_off(g, 0, r, j)];
        const uint32_t nx = spins[strip_off(g, 1, r, j)];
        uint32_t nsh;
        if (p) nsh = __funnelshift_r(nx, spins[strip_off(g, 1, r, j + 1 == g.Wr ? 0 : j + 1)], 1);
        else nsh = __funnelshift_l(spins[strip_off(g, 1, r, j == 0 ? g.Wr - 1 : j - 1)], nx, 1);
        const uint32_t nu = spins[strip_off(g, 1, r - 1, j)];
        const uint32_t nd = spins[strip_off(g, 1, r + 1, j)];
        nsat += __popc(~(s ^ nx ^ antiferro)) + __popc(~(s ^ nsh ^ antiferro)) +
                __popc(~(s ^ nu ^ antiferro)) + __popc(~(s ^ nd ^ antiferro));
        up += __popc(s) + __popc(nx);
    }
    for (int off = 16; off; off >>= 1) {
        nsat += __shfl_xor_sync(0xFFFFFFFFu, nsat, off);
        up += __shfl_xor_sync(0xFFFFFFFFu, up, off);
    }
    if ((threadIdx.x & 31) == 0) {
        if (nsat) atomicAdd(acc, nsat);
        if (up) atomicAdd(acc + 1, up);
    }
}

int launch_strip_observables(const uint32_t* spins, const StripGeom& g, uint32_t antiferro,
                             unsigned long long* acc, cudaStream_t st) {
    k_strip_observables<<<device_sms() * 4, 256, 0, st>>>(spins, g, antiferro, acc);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

__global__ void k_strip_unpack(const uint32_t* __restrict__ spins, StripGeom g,
                               uint8_t* __restrict__ out, uint32_t l0, uint32_t nrows) {
    const uint64_t Lx = 64ull * g.Wr;
    const uint64_t total = (uint64_t)nrows * Lx;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t r = (uint32_t)(i / Lx) + l0 + g.ghost;
        const uint32_t x = (uint32_t)(i % Lx);
        const uint32_t y = g.row0 + r - g.ghost;
        const uint32_t c = (x + y) & 1u, xh = x >> 1;
        out[i] = (uint8_t)((spins[strip_off(g, c, r, xh >> 5)] >> (xh & 31u)) & 1u);
    }
}

int launch_strip_unpack(const uint32_t* spins, const StripGeom& g, uint8_t* out_dev, cudaStream_t st,
                        uint32_t l0, uint32_t nrows) {
    if (nrows == 0xFFFFFFFFu) nrows = g.rows - l0;
    k_strip_unpack<<<device_sms() * 8, 256, 0, st>>>(spins, g, out_dev, l0, nrows);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

}  // namespace ising
