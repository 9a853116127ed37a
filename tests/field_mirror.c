/*
 * tests/field_mirror.c -- the scalar mirror (oracle/msc_mirror.c) of the sweep of a torus in a uniform
 * longitudinal field (pyisingmontecarlo_b200/csrc/sweep_field.cu), for bit-exact checks of the field
 * kernels.  TEST INFRASTRUCTURE ONLY.  The mirror's source is included as it is, so that this file
 * shares its Philox, thresholds, resolver streams, initial state and bond counting; only the class of
 * a site and the energy gain the field term.  Built by tests/field_check.py with the oracle's flags
 * (-ffp-contract=off: the products and sums below must not be fused).
 */
#include "../oracle/msc_mirror.c"

/* A uniform longitudinal field h (E = sum J s s' - h sum s, s = +1 for a set bit): the same sweep with
 * dE = 2|J|(2 n_sat - d) + 2 h sigma (left to right in f64), flip when dE <= 0 without a resolver word,
 * else U < T(dE) with the planes / resolver rule of mirror_sweep (pyisingmontecarlo_b200/csrc/sweep_field.cu). */
static void mirror_sweep_field(const mirror_t *m, uint64_t E, uint8_t *states, double beta, double h, uint32_t sweep) {
    const uint64_t W = (E + 31) / 32, nvars = m->nvars;
    const int K = m->K;
    const uint32_t nwords = 4u * ((uint32_t)K / 4 + 1);
    for (uint32_t col = 0; col < m->ncolors; ++col)
#pragma omp parallel for schedule(static) if (m->proper && nvars > 4096)
        for (uint64_t n = 0; n < nvars; ++n) {
            if (m->colors[n] != col) continue;
            const int d = (int)(m->row[n + 1] - m->row[n]);
            uint32_t R[12];
            for (uint64_t w = 0; w < W; ++w) {
                int j = 0, have_r = 0;
                for (uint64_t b = 0; b < 32 && w * 32 + b < E; ++b) {
                    uint8_t *st = states + (w * 32 + b) * nvars;
                    int nsat = 0;
                    for (uint64_t k = m->row[n]; k < m->row[n + 1]; ++k) {
                        const int equal = st[n] == st[m->nbr[k]];
                        nsat += m->anti[k] ? !equal : equal;
                    }
                    const double sigma = st[n] ? 1.0 : -1.0;
                    const double de = 2.0 * m->jabs * (double)(2 * nsat - d) + 2.0 * h * sigma;
                    if (de <= 0.0) { st[n] ^= 1; continue; }
                    const uint64_t T = threshold(beta, de, K);
                    if (!have_r) {
                        for (uint32_t call = 0; call < nwords / 4; ++call) {
                            uint32_t c[4] = {(uint32_t)n, m->gw0 + (uint32_t)w, sweep, call};
                            philox4x32(m->rounds, c, m->k0, m->k1);
                            memcpy(R + 4 * call, c, sizeof c);
                        }
                        have_r = 1;
                    }
                    int decided = 0, accept = 0;
                    for (int p = 0; p < K && !decided; ++p) {
                        const uint32_t rb = (R[p] >> b) & 1u;
                        const uint32_t tb = (uint32_t)((T >> (K + 31 - p)) & 1ull);
                        if (rb != tb) { decided = 1; accept = rb < tb; }
                    }
                    if (!decided) {
                        const uint32_t q = (uint32_t)(K + j);
                        const uint32_t v = q < nwords ? R[q]
                                                      : stream_word(m->rounds, K, (uint32_t)n, m->gw0 + (uint32_t)w,
                                                                    sweep, q, m->k0, m->k1);
                        accept = v < (uint32_t)(T & 0xFFFFFFFFull);
                        ++j;
                    }
                    if (accept) st[n] ^= 1;
                }
            }
        }
}

/* |J| (n_edges - 2 n_sat) + h (N - 2 up): two products and one sum */
static double mirror_energy_field(const mirror_t *m, const uint8_t *st, double h) {
    long long up = 0;
    for (uint64_t n = 0; n < m->nvars; ++n) up += st[n];
    const double bonds = mirror_energy(m, st);
    return bonds + h * (double)((long long)m->nvars - 2 * up);
}

/* msc_mirror_run in a uniform field h (one beta per sweep; per_replica_beta != 0 is refused with -4) */
ORC_EXPORT int msc_mirror_run_field(uint64_t nvars, uint64_t nedges, const uint64_t *ea,
                                    const uint64_t *eb, const double *ej, const uint32_t *colors,
                                    uint32_t ncolors, uint64_t E, uint64_t seed,
                                    uint64_t replica_offset, int K, int rounds, int randomize,
                                    const uint8_t *init_state, const double *betas, uint64_t nsweeps,
                                    uint64_t sweep0, uint8_t *states, double *energies_per_sweep,
                                    double *final_energies, int per_replica_beta, double field) {
    if (per_replica_beta) return -4;
    mirror_t m;
    int rc = mirror_init(&m, nvars, nedges, ea, eb, ej, colors, ncolors, seed, replica_offset, K, rounds);
    if (rc) return rc;
    if (randomize) mirror_randomize(&m, E, states);
    else if (init_state)
        for (uint64_t e = 0; e < E; ++e) memcpy(states + e * nvars, init_state, nvars);
    for (uint64_t t = 0; t < nsweeps; ++t) {
        mirror_sweep_field(&m, E, states, betas[t], field, (uint32_t)(sweep0 + t));
        if (energies_per_sweep) {
#pragma omp parallel for schedule(static)
            for (uint64_t e = 0; e < E; ++e)
                energies_per_sweep[e * nsweeps + t] = mirror_energy_field(&m, states + e * nvars, field);
        }
    }
    if (final_energies) {
#pragma omp parallel for schedule(static)
        for (uint64_t e = 0; e < E; ++e) final_energies[e] = mirror_energy_field(&m, states + e * nvars, field);
    }
    mirror_free(&m);
    return 0;
}
