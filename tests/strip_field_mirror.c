/*
 * tests/strip_field_mirror.c -- the scalar mirror (oracle/msc_mirror.c: msc_mirror_single) of the large
 * bit-packed 2D lattice in a uniform longitudinal field (pyisingmontecarlo_b200/csrc/strip_field.cu), for
 * bit-exact checks of the field strip kernel.  TEST INFRASTRUCTURE ONLY.  The mirror's source is included
 * as it is, so that this file shares its Philox, thresholds, resolver streams and initial state; only the
 * class of a site gains the field term.  Built by tests/strip_field_check.py with the oracle's flags
 * (-ffp-contract=off: the products and sums below must not be fused).
 */
#include "../oracle/msc_mirror.c"

/* The 32 decisions of word j of colour c in global row y (sweep t): own = the row's sites, up / dn = the
 * rows y - 1 / y + 1.  E = sum J s s' - h sum s (s = +1 for a set bit): dE = 2|J|(2 n_sat - 4) + 2 h sigma
 * (left to right in f64); dE <= 0 flips without a resolver word, else U < T(dE) with the planes and the
 * tie rule of msc_mirror_single. */
static void field_word(uint8_t *own, const uint8_t *up, const uint8_t *dn, uint64_t Lx, uint64_t y, uint32_t c,
                       uint64_t j, uint32_t t, double beta, double h, double jabs, int anti, int K, int rounds,
                       uint32_t k0, uint32_t k1) {
    int tie_rank = 0;
    for (uint32_t b = 0; b < 32; ++b) {
        const uint64_t x = 2 * (32 * j + b) + ((y + c) & 1);
        const uint8_t s = own[x];
        const uint8_t nb[4] = {own[(x + 1) % Lx], own[(x + Lx - 1) % Lx], dn[x], up[x]};
        int nsat = 0;
        for (int k = 0; k < 4; ++k) nsat += anti ? (s != nb[k]) : (s == nb[k]);
        const double sigma = s ? 1.0 : -1.0;
        const double de = 2.0 * jabs * (double)(2 * nsat - 4) + 2.0 * h * sigma;
        if (de <= 0.0) { own[x] ^= 1; continue; }
        const uint64_t T = threshold(beta, de, K);
        const uint32_t gw = (c << 30) | (uint32_t)j;
        int decided = 0, accept = 0;
        for (int p = 0; p < K && !decided; ++p) {
            const uint32_t rb = (stream_word(rounds, K, (uint32_t)y, gw, t, (uint32_t)p, k0, k1) >> b) & 1u;
            const uint32_t tb = (uint32_t)((T >> (K + 31 - p)) & 1ull);
            if (rb != tb) { decided = 1; accept = rb < tb; }
        }
        if (!decided) {
            const uint32_t v = stream_word(rounds, K, (uint32_t)y, gw, t, (uint32_t)(K + tie_rank), k0, k1);
            accept = v < (uint32_t)(T & 0xFFFFFFFFull);
            ++tie_rank;
        }
        if (accept) own[x] ^= 1;
    }
}

/* msc_mirror_single with one (betas[t], fields[t]) per sweep.  state: bool[Ly, Lx] in/out (the Philox
 * initial state when randomize != 0).  nsat_out / up_out (or NULL): int64[nsweeps], the satisfied bonds
 * and up spins after each sweep. */
ORC_EXPORT int msc_mirror_single_field(uint64_t Lx, uint64_t Ly, double jcoupling, uint64_t seed, int K, int rounds,
                                       int randomize, const double *betas, const double *fields, uint64_t nsweeps,
                                       uint8_t *state, long long *nsat_out, long long *up_out) {
    if (Lx % 64 || (Ly & 1) || K < 1 || K > 8) return -1;
    if (randomize) msc_mirror_single(Lx, Ly, jcoupling, seed, K, rounds, 1, betas, 0, state, NULL);
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    const double jabs = fabs(jcoupling);
    const int anti = jcoupling > 0;
    for (uint64_t t = 0; t < nsweeps; ++t) {
        for (uint32_t c = 0; c < 2; ++c)
            for (uint64_t y = 0; y < Ly; ++y)
                for (uint64_t j = 0; j < Lx / 64; ++j)
                    field_word(state + y * Lx, state + ((y + Ly - 1) % Ly) * Lx, state + ((y + 1) % Ly) * Lx, Lx, y, c,
                               j, (uint32_t)t, betas[t], fields[t], jabs, anti, K, rounds, k0, k1);
        long long nsat = 0, up = 0;
        for (uint64_t y = 0; y < Ly; ++y)
            for (uint64_t x = 0; x < Lx; ++x) {
                const uint8_t s = state[y * Lx + x];
                const uint8_t r = state[y * Lx + (x + 1) % Lx], d = state[((y + 1) % Ly) * Lx + x];
                nsat += anti ? (s != r) : (s == r);
                nsat += anti ? (s != d) : (s == d);
                up += s;
            }
        if (nsat_out) nsat_out[t] = nsat;
        if (up_out) up_out[t] = up;
    }
    return 0;
}

/* msc_mirror_single_band in the field schedule: rows y0 .. y0 + nrows - 1 (0 < y0, y0 + nrows < Ly); after
 * nsweeps sweeps the rows [2 nsweeps, nrows - 2 nsweeps) equal those of the full lattice. */
ORC_EXPORT int msc_mirror_single_band_field(uint64_t Lx, uint64_t y0, uint64_t nrows, double jcoupling, uint64_t seed,
                                            int K, int rounds, int randomize, const double *betas,
                                            const double *fields, uint64_t nsweeps, uint8_t *state) {
    if (Lx % 64 || K < 1 || K > 8 || nrows < 4 * nsweeps + 1) return -1;
    if (randomize) msc_mirror_single_band(Lx, y0, nrows, jcoupling, seed, K, rounds, 1, betas, 0, state);
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    const double jabs = fabs(jcoupling);
    const int anti = jcoupling > 0;
    for (uint64_t t = 0; t < nsweeps; ++t)
        for (uint32_t c = 0; c < 2; ++c) {
            const uint64_t q = 2 * t + c;
            for (uint64_t r = q + 1; r + q + 1 < nrows; ++r)
                for (uint64_t j = 0; j < Lx / 64; ++j)
                    field_word(state + r * Lx, state + (r - 1) * Lx, state + (r + 1) * Lx, Lx, y0 + r, c, j,
                               (uint32_t)t, betas[t], fields[t], jabs, anti, K, rounds, k0, k1);
        }
    return 0;
}
