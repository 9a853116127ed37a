// TEST INFRASTRUCTURE (CPU suite only).  Runs the field strip kernel (k_strip_phase_field of
// csrc/strip_field.cu: one large 2D lattice bit-packed along x, in a uniform longitudinal field) from its
// own source on the host (cuda_on_host.h) for tests/test_strip_field_on_host.py, which compares the
// result with tests/strip_field_mirror.c.  Block and grid shape are strip_phase_shape()'s (strip.cu), with
// the SM count of the grid cap given; the thresholds restate fill_field_thresholds() of api_sim.cu for 2D.
#include "cuda_on_host.h"

#include <math.h>
#include <string.h>

#include "prepared/strip_field_kernel.cuh"

using namespace ising;

namespace {

uint64_t threshold64(double beta, double de, int K) {
    const double scaled = ldexp(exp(-beta * de), K + 32);
    const uint64_t tmax = (1ull << (K + 32)) - 1;
    if (!(scaled >= 0.0)) return 0;
    if (scaled >= (double)tmax) return tmax;
    return (uint64_t)floor(scaled);
}

void thresholds2d(double jabs, double h, double beta, int K, FieldThresholds* th) {
    memset(th, 0, sizeof *th);
    for (int sp = 0; sp < 2; ++sp)
        for (int n = 0; n <= 4; ++n) {
            const double sigma = sp ? 1.0 : -1.0;
            const double de = 2.0 * jabs * (double)(2 * n - 4) + 2.0 * h * sigma;
            if (!(de > 0.0)) continue;
            const uint64_t T = threshold64(beta, de, K);
            th->up[sp][n] = 0xFFFFFFFFu;
            for (int pl = 0; pl < K; ++pl) th->plane[pl][sp][n] = ((T >> (K + 31 - pl)) & 1ull) ? 0xFFFFFFFFu : 0u;
            th->low[sp][n] = (uint32_t)(T & 0xFFFFFFFFull);
        }
}

template <int K, int ROUNDS, int V>
void run(uint32_t* spins, const StripGeom& g, uint32_t c, uint32_t sweep, uint64_t seed, uint32_t antiferro,
         const FieldThresholds& th, uint32_t r_begin, uint32_t r_count, uint32_t sms) {
    const uint32_t groups = g.Wr / V;
    const uint32_t bx = groups >= 256 ? 256 : pow2_ceil(groups);
    const dim3 block(bx, 256 / bx, 1);
    uint32_t gx = (groups + bx - 1) / bx;
    if (gx > 64) gx = 64;
    uint32_t gy = (r_count + block.y - 1) / block.y;
    const uint32_t gy_cap = (sms * 32u + gx - 1) / gx;
    if (gy > gy_cap) gy = gy_cap;                 // the kernel strides over the rows by the grid
    emu::launch_v(k_strip_phase_field<K, ROUNDS, V>, dim3(gx, gy, 1), block, 0, spins, g, c, sweep,
                  philox_round_keys((uint32_t)seed, (uint32_t)(seed >> 32)), antiferro, th, r_begin, r_count);
}

template <int V>
int by_planes(uint32_t* spins, const StripGeom& g, uint32_t c, uint32_t sweep, uint64_t seed, uint32_t antiferro,
              const FieldThresholds& th, uint32_t r_begin, uint32_t r_count, uint32_t sms, int K, int rounds) {
#define RUN(KK, RR) run<KK, RR, V>(spins, g, c, sweep, seed, antiferro, th, r_begin, r_count, sms)
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

// One colour phase in the field h on the storage rows [r_begin, r_begin + r_count) of
// spins[2][rows + 2 ghost][Wr]; V as launch_strip_phase_field picks it.
extern "C" int emu_strip_phase_field(uint32_t* spins, uint32_t Wr, uint32_t rows, uint32_t row0, uint32_t Ly,
                                     uint32_t ghost, uint32_t colour, uint32_t sweep, uint64_t seed, uint32_t antiferro,
                                     double beta, double jabs, double h, int K, int rounds, uint32_t r_begin,
                                     uint32_t r_count, uint32_t sms) {
    if (Wr == 0 || r_count == 0) return 0;
    StripGeom g{Wr, rows, row0, Ly, ghost};
    FieldThresholds th;
    thresholds2d(jabs, h, beta, K, &th);
    if (Wr % 4 == 0) return by_planes<4>(spins, g, colour, sweep, seed, antiferro, th, r_begin, r_count, sms, K, rounds);
    if (Wr % 2 == 0) return by_planes<2>(spins, g, colour, sweep, seed, antiferro, th, r_begin, r_count, sms, K, rounds);
    return by_planes<1>(spins, g, colour, sweep, seed, antiferro, th, r_begin, r_count, sms, K, rounds);
}
