// sm_100a kernels: checkerboard sweeps of a square / cubic torus in a uniform longitudinal field
// h (energy E = sum J s s' - h sum s), and the conversion of the per-sweep counts to energies.
// The bit-sliced Metropolis rule of msc_flip_mask (msc_device.cuh) with a class that also depends
// on the spin: dE = 2|J|(2 n_sat - 2 DIM) + 2 h sigma takes at most 2 (2 DIM + 1) values, so the
// thresholds stay exact integers computed on the host (FieldThresholds, kernels.h).
#include "msc_device.cuh"

namespace ising {

// Flip mask of one word: the K/4 + 1 Philox calls of (site, word, sweep) and field_flip_mask_words
// (msc_device.cuh) on their words.
template <int DIM, int K, int ROUNDS>
__device__ __forceinline__ uint32_t field_flip_mask(uint32_t s, uint32_t b0, uint32_t b1, uint32_t b2,
                                                    const FieldThresholds& th, uint32_t site, uint32_t gw,
                                                    uint32_t sweep, const PhiloxKeys& pk) {
    constexpr int NCALL = K / 4 + 1;
    uint32_t r[NCALL * 4];
#pragma unroll
    for (int q = 0; q < NCALL; ++q) {
        const u32x4 o = philox4x32_keys<ROUNDS>(site, gw, sweep, (uint32_t)q | (TAG_ACCEPT << 24), pk);
        r[4 * q + 0] = o.x;
        r[4 * q + 1] = o.y;
        r[4 * q + 2] = o.z;
        r[4 * q + 3] = o.w;
    }
    return field_flip_mask_words<DIM, K, ROUNDS>(s, b0, b1, b2, th, r, pk);
}

// One colour phase on the stencil layout (kernels.h: Layout).  block = (lanes over groups of V
// replica words, half-row positions); the blocks walk the rows with stride gridDim.x.
// (3 blocks per SM: left to itself ptxas caps one instantiation at 64 registers and spills.)
template <int DIM, bool PMJ, int K, int ROUNDS, int V>
__global__ void __launch_bounds__(256, 3)
k_sweep_field(uint32_t* __restrict__ own, const uint32_t* __restrict__ oth, const uint32_t* __restrict__ jm,
              Layout L, uint32_t c, uint32_t sweep, PhiloxKeys pk, uint32_t gw0, uint32_t antiferro,
              FieldThresholds th) {
    const uint32_t Lxh = L.Lxh, W = L.W, Ly = L.Ly, Lz = L.Lz;
    const uint32_t rowlen = Lxh * W;
    for (uint32_t w = V * threadIdx.x; w < W; w += V * blockDim.x) {
        for (uint32_t row = blockIdx.x; row < L.rows; row += gridDim.x) {
            const uint32_t z = row / Ly, y = row - z * Ly;
            const uint32_t p = (y + z + c) & 1u;
            const uint32_t ym = y == 0 ? Ly - 1 : y - 1, yp = y + 1 == Ly ? 0 : y + 1;
            uint32_t* __restrict__ o_c = own + (size_t)row * rowlen;
            const uint32_t* __restrict__ n_x = oth + (size_t)row * rowlen;
            const uint32_t* __restrict__ n_ym = oth + (size_t)(z * Ly + ym) * rowlen;
            const uint32_t* __restrict__ n_yp = oth + (size_t)(z * Ly + yp) * rowlen;
            const uint32_t* __restrict__ n_zm = nullptr;
            const uint32_t* __restrict__ n_zp = nullptr;
            if (DIM == 3) {
                const uint32_t zm = z == 0 ? Lz - 1 : z - 1, zp = z + 1 == Lz ? 0 : z + 1;
                n_zm = oth + (size_t)(zm * Ly + y) * rowlen;
                n_zp = oth + (size_t)(zp * Ly + y) * rowlen;
            }
            for (uint32_t xh = threadIdx.y; xh < Lxh; xh += blockDim.y) {
                const uint32_t xs = p ? (xh + 1 == Lxh ? 0 : xh + 1) : (xh == 0 ? Lxh - 1 : xh - 1);
                uint32_t m[2 * DIM];
#pragma unroll
                for (int k = 0; k < 2 * DIM; ++k)
                    m[k] = PMJ ? __ldg(jm + (size_t)k * L.halfN + (size_t)row * Lxh + xh) : antiferro;
                const uint32_t site = row * L.Lx + 2 * xh + p;
                const uint32_t i = xh * W + w;
                uint32_t s[V], n[2 * DIM][V];
                load_words<V>(o_c + i, s);
                load_words<V>(n_x + i, n[0]);
                load_words<V>(n_x + xs * W + w, n[1]);
                load_words<V>(n_ym + i, n[2]);
                load_words<V>(n_yp + i, n[3]);
                if (DIM == 3) {
                    load_words<V>(n_zm + i, n[4]);
                    load_words<V>(n_zp + i, n[5]);
                }
#pragma unroll
                for (int v = 0; v < V; ++v) {
                    uint32_t a[2 * DIM];
#pragma unroll
                    for (int k = 0; k < 2 * DIM; ++k) a[k] = ~(s[v] ^ n[k][v] ^ m[k]);
                    uint32_t b0, b1, b2;
                    count_sat<DIM>(a, b0, b1, b2);
                    s[v] ^= field_flip_mask<DIM, K, ROUNDS>(s[v], b0, b1, b2, th, site, gw0 + w + v, sweep, pk);
                }
                store_words<V>(o_c + i, s);
            }
        }
    }
}

// out[e * estride + eoff + t] = |J| (nbonds - 2 nsat) + h (nsites - 2 up), two rounded products and
// one rounded sum (no contraction), for nt sweeps of counts nsat[t * cw + e], up[t * cw + e]
__global__ void k_energy_field(const unsigned long long* __restrict__ nsat, const unsigned long long* __restrict__ up,
                               uint64_t E, uint64_t cw, uint64_t nt, double jabs, uint64_t nbonds, double h,
                               uint64_t nsites, double* __restrict__ out, uint64_t estride, uint64_t eoff) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= E * nt) return;
    const uint64_t e = i / nt, t = i - e * nt;
    const long long bonds = (long long)nbonds - 2ll * (long long)nsat[t * cw + e];
    const long long spins = (long long)nsites - 2ll * (long long)up[t * cw + e];
    out[e * estride + eoff + t] = __dadd_rn(__dmul_rn(jabs, (double)bonds), __dmul_rn(h, (double)spins));
}

// block = (wx lanes over the V-word groups of a site, by half-row positions), at least one warp;
// grid = one block per row up to 32 blocks per SM, rows beyond that are walked with the grid stride
static void field_launch_shape(const Layout& L, uint32_t V, dim3* grid, dim3* block) {
    const uint32_t groups = (L.W + V - 1) / V;
    const uint32_t wx = groups >= 32 ? 32 : pow2_ceil(groups);
    uint32_t by = 256 / wx;
    const uint32_t need = pow2_ceil(L.Lxh);
    if (by > need) by = need;
    if (wx * by < 32) by = 32 / wx;
    *block = dim3(wx, by, 1);
    const uint32_t cap = device_sms() * 32u;
    *grid = dim3(L.rows < cap ? L.rows : cap, 1, 1);
}

template <int DIM, bool PMJ, int K, int ROUNDS, int V>
static int field_launch(const SweepArgs& a, const FieldThresholds& th, cudaStream_t st) {
    const Layout& L = a.lay;
    dim3 grid, block;
    field_launch_shape(L, V, &grid, &block);
    const size_t csz = (size_t)L.halfN * L.W;
    const size_t jsz = (size_t)2 * DIM * L.halfN;
    const PhiloxKeys pk = philox_round_keys(a.key0, a.key1);
    for (uint32_t c = 0; c < 2; ++c)
        k_sweep_field<DIM, PMJ, K, ROUNDS, V><<<grid, block, 0, st>>>(
            a.spins + c * csz, a.spins + (1 - c) * csz, PMJ ? a.jmask + c * jsz : nullptr, L, c, a.sweep, pk, a.gw0,
            a.antiferro, th);
    return cudaGetLastError() == cudaSuccess ? 2 : -1;
}

template <int DIM, bool PMJ, int V>
static int field_dispatch(const SweepArgs& a, const FieldThresholds& th, cudaStream_t st) {
    const bool r7 = a.rounds == 7;
    switch (a.planes) {
        case 5: return r7 ? field_launch<DIM, PMJ, 5, 7, V>(a, th, st) : field_launch<DIM, PMJ, 5, 10, V>(a, th, st);
        case 6: return r7 ? field_launch<DIM, PMJ, 6, 7, V>(a, th, st) : field_launch<DIM, PMJ, 6, 10, V>(a, th, st);
        case 7: return r7 ? field_launch<DIM, PMJ, 7, 7, V>(a, th, st) : field_launch<DIM, PMJ, 7, 10, V>(a, th, st);
        default: return -1;
    }
}

template <int V>
static int field_dispatch_kind(const SweepArgs& a, const FieldThresholds& th, cudaStream_t st) {
    const bool pmj = a.jmask != nullptr;
    if (a.lay.kind == ISING_KIND_STENCIL3D)
        return pmj ? field_dispatch<3, true, V>(a, th, st) : field_dispatch<3, false, V>(a, th, st);
    if (a.lay.kind == ISING_KIND_STENCIL2D)
        return pmj ? field_dispatch<2, true, V>(a, th, st) : field_dispatch<2, false, V>(a, th, st);
    return -1;
}

int launch_sweep_field(const SweepArgs& a, const FieldThresholds& th, cudaStream_t st) {
    if (a.rounds != 7 && a.rounds != 10) return -1;
    // widest vector the replica-word count allows, as the stencil launcher picks it
    if (a.lay.W % 4 == 0) return field_dispatch_kind<4>(a, th, st);
    if (a.lay.W % 2 == 0) return field_dispatch_kind<2>(a, th, st);
    return field_dispatch_kind<1>(a, th, st);
}

int launch_energy_field(const unsigned long long* nsat, const unsigned long long* up, uint64_t E, uint64_t cw,
                        uint64_t nt, double jabs, uint64_t nbonds, double h, uint64_t nsites, double* out_dev,
                        uint64_t estride, uint64_t eoff, cudaStream_t st) {
    const uint64_t n = E * nt;
    const unsigned g = (unsigned)((n + 255) / 256);
    k_energy_field<<<g ? g : 1, 256, 0, st>>>(nsat, up, E, cw, nt, jabs, nbonds, h, nsites, out_dev, estride, eoff);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

}  // namespace ising
