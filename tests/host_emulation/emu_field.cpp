// TEST INFRASTRUCTURE (CPU suite only).  Runs the field kernels from their own source on the host
// (cuda_on_host.h) for tests/test_field_on_host.py:
//   k_sweep_field (csrc/sweep_field.cu)   both colour phases of a sweep of a torus in a uniform field,
//                                         in the block / grid shape of the library's field_launch_shape()
//   k_energy_field                        per-sweep energies from the satisfied-bond and up-spin counts
// Thresholds as fill_field_thresholds() of api_sim.cu.
#include "cuda_on_host.h"

#include <math.h>
#include <string.h>

namespace ising { unsigned device_sms(); }
#include "prepared/field_kernels.cuh"

namespace ising {
static unsigned g_sms = 2;
unsigned device_sms() { return g_sms; }
}  // namespace ising

using namespace ising;

namespace {

uint64_t threshold64(double beta, double de, int K) {
    const double scaled = ldexp(exp(-beta * de), K + 32);
    const uint64_t tmax = (1ull << (K + 32)) - 1;
    if (!(scaled >= 0.0)) return 0;
    if (scaled >= (double)tmax) return tmax;
    return (uint64_t)floor(scaled);
}

void thresholds(int dim, double jabs, double h, double beta, int K, FieldThresholds* th) {
    memset(th, 0, sizeof *th);
    for (int sp = 0; sp < 2; ++sp)
        for (int n = 0; n <= 2 * dim; ++n) {
            const double sigma = sp ? 1.0 : -1.0;
            const double de = 2.0 * jabs * (double)(2 * n - 2 * dim) + 2.0 * h * sigma;
            if (!(de > 0.0)) continue;
            const uint64_t T = threshold64(beta, de, K);
            th->up[sp][n] = 0xFFFFFFFFu;
            for (int pl = 0; pl < K; ++pl) th->plane[pl][sp][n] = ((T >> (K + 31 - pl)) & 1ull) ? 0xFFFFFFFFu : 0u;
            th->low[sp][n] = (uint32_t)(T & 0xFFFFFFFFull);
        }
}

// field_launch() of sweep_field.cu
template <int DIM, bool PMJ, int K, int ROUNDS, int V>
void sweep(const Layout& L, uint32_t* spins, const uint32_t* jmask, uint32_t antiferro, uint64_t seed,
           uint32_t sweep_idx, uint32_t gw0, const FieldThresholds& th) {
    dim3 grid, block;
    field_launch_shape(L, V, &grid, &block);
    const size_t csz = (size_t)L.halfN * L.W, jsz = (size_t)2 * DIM * L.halfN;
    const PhiloxKeys pk = philox_round_keys((uint32_t)seed, (uint32_t)(seed >> 32));
    for (uint32_t c = 0; c < 2; ++c)
        emu::launch_v(k_sweep_field<DIM, PMJ, K, ROUNDS, V>, grid, block, 0, spins + c * csz,
                      (const uint32_t*)spins + (1 - c) * csz, PMJ ? jmask + c * jsz : nullptr, L, c, sweep_idx, pk,
                      gw0, antiferro, th);
}

template <int DIM, bool PMJ, int V>
int by_planes(const Layout& L, uint32_t* spins, const uint32_t* jmask, uint32_t antiferro, uint64_t seed,
              uint32_t sweep_idx, uint32_t gw0, int K, int rounds, const FieldThresholds& th) {
#define RUN(KK, RR) sweep<DIM, PMJ, KK, RR, V>(L, spins, jmask, antiferro, seed, sweep_idx, gw0, th)
    if (K == 5 && rounds == 7) RUN(5, 7);
    else if (K == 5 && rounds == 10) RUN(5, 10);
    else if (K == 6 && rounds == 7) RUN(6, 7);
    else if (K == 6 && rounds == 10) RUN(6, 10);
    else if (K == 7 && rounds == 7) RUN(7, 7);
    else if (K == 7 && rounds == 10) RUN(7, 10);
    else return -2;
#undef RUN
    return 0;
}

}  // namespace

// One sweep (both colour phases) of the stencil layout spins[2][rows][Lxh][W]; jmask = [2][2 dim][halfN]
// bond masks or NULL (uniform sign: antiferro).  sms = SM count the launch shape is computed for.
extern "C" int emu_sweep_field(int dim, uint32_t Lx, uint32_t Ly, uint32_t Lz, uint32_t W, int V, const uint32_t* jmask,
                               uint32_t antiferro, uint32_t* spins, uint64_t seed, uint32_t sweep_idx, uint32_t gw0,
                               int K, int rounds, double beta, double jabs, double h, uint32_t sms) {
    if (W % V) return -1;
    Layout L;
    memset(&L, 0, sizeof L);
    L.kind = dim == 3 ? ISING_KIND_STENCIL3D : ISING_KIND_STENCIL2D;
    L.Lx = Lx; L.Ly = Ly; L.Lz = dim == 3 ? Lz : 1; L.Lxh = Lx / 2; L.rows = L.Ly * L.Lz; L.W = W;
    L.nvars = (uint64_t)Lx * L.Ly * L.Lz;
    L.halfN = L.nvars / 2;
    g_sms = sms;
    FieldThresholds th;
    thresholds(dim, jabs, h, beta, K, &th);
    const bool pmj = jmask != nullptr;
#define SHAPE(D, P, VV) if (dim == D && pmj == P && V == VV) \
        return by_planes<D, P, VV>(L, spins, jmask, antiferro, seed, sweep_idx, gw0, K, rounds, th)
    SHAPE(3, true, 4); SHAPE(3, true, 2); SHAPE(3, true, 1);
    SHAPE(3, false, 4); SHAPE(3, false, 2); SHAPE(3, false, 1);
    SHAPE(2, true, 4); SHAPE(2, true, 2); SHAPE(2, true, 1);
    SHAPE(2, false, 4); SHAPE(2, false, 2); SHAPE(2, false, 1);
#undef SHAPE
    return -9;
}

// launch_energy_field() of sweep_field.cu
extern "C" void emu_energy_field(const unsigned long long* nsat, const unsigned long long* up, uint64_t E, uint64_t cw,
                                 uint64_t nt, double jabs, uint64_t nbonds, double h, uint64_t nsites, double* out,
                                 uint64_t estride, uint64_t eoff) {
    const uint64_t n = E * nt;
    const unsigned g = (unsigned)((n + 255) / 256);
    emu::launch_v(k_energy_field, dim3(g ? g : 1), dim3(256), 0, nsat, up, E, cw, nt, jabs, nbonds, h, nsites, out,
                  estride, eoff);
}
