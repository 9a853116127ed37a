// sm_100a kernel: one colour phase of the large bit-packed 2D lattice (strip.cu: k_strip_phase) in a
// uniform longitudinal field h (energy E = sum J s s' - h sum s).  The class of a site becomes
// (sigma, n_sat), n_sat = 0..4, so dE = 2|J|(2 n_sat - 4) + 2 h sigma takes at most 10 values and the
// thresholds stay exact host integers (FieldThresholds, kernels.h).  Rows, loads, x neighbours, the
// Philox counter (global row, colour << 30 | word, sweep, call), the tie order and the continuation
// rounds are those of k_strip_phase, so a draw still depends on the global row only: the redundant
// ghost-row updates of the deep halo exchange stay exact (a uniform field is the same on every row).
#include "sweep_rows.cuh"

namespace ising {

// V consecutive words of a row per thread; Philox rounds 1-3 shared over the V words and both calls
// (sweep_rows.cuh: PhiloxSite), the uphill bits and threshold planes selected per bit by (spin, n_sat)
// (msc_device.cuh: field_flip_mask_words).
template <int K, int ROUNDS, int V>
__global__ void __launch_bounds__(256, 3)
k_strip_phase_field(uint32_t* __restrict__ spins, const __grid_constant__ StripGeom g, uint32_t c, uint32_t sweep,
                    const __grid_constant__ PhiloxKeys pk, uint32_t antiferro,
                    const __grid_constant__ FieldThresholds th, uint32_t r_begin, uint32_t r_count) {
    static_assert(K >= 4 && K <= 7, "two Philox calls: K planes + (8 - K) resolver words");
    const uint32_t groups = g.Wr / V;
    const uint32_t o = 1u - c;
    // programmatic dependent launch: the next phase is scheduled while this one drains
    asm volatile("griddepcontrol.launch_dependents;");
    asm volatile("griddepcontrol.wait;" ::: "memory");
    // block = (x over the word groups of a row, y over rows): storage rows [r_begin, r_begin + r_count)
    for (uint32_t rr = blockIdx.y * blockDim.y + threadIdx.y; rr < r_count; rr += gridDim.y * blockDim.y)
    for (uint32_t jg = blockIdx.x * blockDim.x + threadIdx.x; jg < groups; jg += gridDim.x * blockDim.x) {
        const uint32_t j = jg * V;
        const uint32_t r = r_begin + rr;
        const uint32_t y = strip_global_row(g, r);
        uint32_t s[V], n[4][V];
        uint32_t* own = strip_load_site<V>(spins, g, c, o, r, j, (y + c) & 1u, s, n);
        PhiloxSite<ROUNDS, V> ph;
        ph.prepare(y, (c << 30) | j, sweep, pk);
#pragma unroll
        for (int v = 0; v < V; ++v) {
            uint32_t rw[8];
            ph.finish(v, 0, pk, rw);
            ph.finish(v, 1, pk, rw + 4);
            uint32_t a[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) a[k] = ~(s[v] ^ n[k][v] ^ antiferro);
            uint32_t b0, b1, b2;
            count_sat<2>(a, b0, b1, b2);
            s[v] ^= field_flip_mask_words<2, K, ROUNDS>(s[v], b0, b1, b2, th, rw, pk);
        }
        store_words<V>(own, s);
    }
}

template <int V>
static int strip_field_dispatch(const StripSweepArgs& a, const FieldThresholds& th, cudaStream_t st) {
    dim3 grid, block;
    strip_phase_shape(a, V, &grid, &block);
    const PhiloxKeys pk = philox_round_keys(a.key0, a.key1);
#define FIELD_LAUNCH(KK, RR)                                                                           \
    launch_pdl_v(k_strip_phase_field<KK, RR, V>, grid, block, 0, st, a.spins, a.g, a.colour, a.sweep, pk, \
                 a.antiferro, th, a.r_begin, a.r_count)
#define FIELD_ROUNDS(KK)                                                                               \
    do { if (a.rounds == 7) FIELD_LAUNCH(KK, 7); else FIELD_LAUNCH(KK, 10); } while (0)
    switch (a.planes) {
        case 5: FIELD_ROUNDS(5); break;
        case 6: FIELD_ROUNDS(6); break;
        case 7: FIELD_ROUNDS(7); break;
        default: return -1;
    }
#undef FIELD_ROUNDS
#undef FIELD_LAUNCH
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

int launch_strip_phase_field(const StripSweepArgs& a, const FieldThresholds& th, cudaStream_t st) {
    if (a.r_count == 0 || a.g.Wr == 0) return 0;
    // V and launch shape as launch_strip_phase picks them
    if (a.g.Wr % 4 == 0) return strip_field_dispatch<4>(a, th, st);
    if (a.g.Wr % 2 == 0) return strip_field_dispatch<2>(a, th, st);
    return strip_field_dispatch<1>(a, th, st);
}

}  // namespace ising
