/*
 * oracle/msc_mirror.c -- scalar CPU restatement of the PRODUCTION-RNG sweep of libising_b200
 * (DESIGN.md "Production sweep"), one spin at a time, for bit-exact checks of the CUDA kernels.
 *
 * TEST INFRASTRUCTURE ONLY (see ising_oracle.c).  This file does not restate the reference: the
 * reference updates uniformly random sites sequentially with xoshiro256++ (restated in
 * ising_oracle.c), whereas the device path sweeps colour classes with Philox randomness.  The
 * two agree in distribution (tests/test_statistics*.py), not draw by draw; this mirror pins the
 * device path's exact bits so that a kernel optimisation cannot silently change results.
 *
 * Algorithm (graphs with all |J| equal and no bias):
 *   for sweep t, colour c = 0..C-1, every site n of colour c, every replica word w:
 *     n_sat = satisfied bonds (J s s' < 0) of n, d = degree;  dE = 2|J|(2 n_sat - d)
 *     dE <= 0 -> flip.  dE > 0 -> flip iff U < T(dE), T = floor(exp(-beta dE) 2^(K+32)):
 *       words R_m = output m%4 of Philox4x32-R(key = seed, ctr = (n, w, t, m/4));
 *       bit b of R_0..R_{K-1} are the K most significant bits of U for replica 32w+b, compared
 *       MSB first; bits of the word still tied after K planes are taken in ascending b and the
 *       j-th of them accepts iff R_{K+j} < T mod 2^32.  Words beyond the K/4 + 1 calls every
 *       update makes are continuation rounds of the last block (stream_word_tag below).
 *   initial state: bit b of Philox4x32-10(key, ctr = (n, w, 0, 1<<24)).x
 *   energy: |J| (n_edges - 2 n_sat_total)
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define ORC_EXPORT __attribute__((visibility("default")))

static void philox4x32(int rounds, uint32_t c[4], uint32_t k0, uint32_t k1) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
    for (int r = 0; r < rounds; ++r) {
        uint64_t p0 = (uint64_t)M0 * c[0], p1 = (uint64_t)M1 * c[2];
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1;
        c[1] = (uint32_t)p1;
        c[3] = (uint32_t)p0;
        c[0] = n0;
        c[2] = n2;
        k0 += W0;
        k1 += W1;
    }
}

/* known-answer hook for the tests */
ORC_EXPORT void msc_philox4x32(int rounds, const uint32_t ctr[4], const uint32_t key[2],
                               uint32_t out[4]) {
    uint32_t c[4] = {ctr[0], ctr[1], ctr[2], ctr[3]};
    philox4x32(rounds, c, key[0], key[1]);
    memcpy(out, c, sizeof c);
}

/* Word R_m of a decision stream with K planes on counter (c0, c1, c2, call | tag): the NCALL =
 * K/4 + 1 calls every update makes give R_0 .. R_{4 NCALL - 1}; later words (third and later
 * ties of a word) are continuation rounds of the last block: R_m = output m%4 of
 * Philox4x32-(rounds + m/4 - NCALL + 1) on the counter of call NCALL - 1 (msc_device.cuh). */
static uint32_t stream_word_tag(int rounds, int K, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t tag,
                                uint32_t m, uint32_t k0, uint32_t k1) {
    const uint32_t ncall = (uint32_t)K / 4 + 1;
    uint32_t call = m >> 2;
    int extra = 0;
    if (call >= ncall) {
        extra = (int)(call - ncall) + 1;
        call = ncall - 1;
    }
    uint32_t c[4] = {c0, c1, c2, call | tag};
    philox4x32(rounds + extra, c, k0, k1);
    return c[m & 3];
}

static uint32_t stream_word(int rounds, int K, uint32_t site, uint32_t gw, uint32_t sweep, uint32_t m,
                            uint32_t k0, uint32_t k1) {
    return stream_word_tag(rounds, K, site, gw, sweep, 0u, m, k0, k1);
}

static uint64_t threshold(double beta, double de, int K) {
    const double scaled = ldexp(exp(-beta * de), K + 32);
    const uint64_t tmax = (1ull << (K + 32)) - 1;
    if (!(scaled >= 0.0)) return 0;
    if (scaled >= (double)tmax) return tmax;
    return (uint64_t)floor(scaled);
}

typedef struct {
    uint64_t nvars, nedges;
    const uint64_t *ea, *eb;
    const double *ej;
    const uint32_t *colors;
    uint32_t ncolors;
    uint64_t *row, *nbr;
    uint8_t *anti;
    double jabs;
    uint32_t k0, k1, gw0;
    int K, rounds;
    int proper;   /* no bond joins two sites of one colour */
} mirror_t;

static int mirror_init(mirror_t *m, uint64_t nvars, uint64_t nedges, const uint64_t *ea,
                       const uint64_t *eb, const double *ej, const uint32_t *colors,
                       uint32_t ncolors, uint64_t seed, uint64_t replica_offset, int K, int rounds) {
    if (nedges == 0 || K < 1 || K > 8) return -1;
    m->jabs = fabs(ej[0]);
    for (uint64_t e = 0; e < nedges; ++e)
        if (fabs(ej[e]) != m->jabs) return -2;
    m->nvars = nvars; m->nedges = nedges; m->ea = ea; m->eb = eb; m->ej = ej;
    m->colors = colors; m->ncolors = ncolors;
    m->k0 = (uint32_t)seed; m->k1 = (uint32_t)(seed >> 32);
    m->gw0 = (uint32_t)(replica_offset / 32);
    m->K = K; m->rounds = rounds;
    m->proper = 1;
    for (uint64_t e = 0; e < nedges; ++e)
        if (colors[ea[e]] == colors[eb[e]]) m->proper = 0;
    m->row =(uint64_t *)calloc(nvars + 1, sizeof(uint64_t));
    for (uint64_t e = 0; e < nedges; ++e) { m->row[ea[e] + 1]++; m->row[eb[e] + 1]++; }
    for (uint64_t i = 0; i < nvars; ++i) m->row[i + 1] += m->row[i];
    m->nbr = (uint64_t *)malloc(sizeof(uint64_t) * 2 * nedges);
    m->anti = (uint8_t *)malloc(2 * nedges);
    uint64_t *fill = (uint64_t *)calloc(nvars, sizeof(uint64_t));
    for (uint64_t e = 0; e < nedges; ++e) {
        uint64_t a = ea[e], b = eb[e];
        m->nbr[m->row[a] + fill[a]] = b; m->anti[m->row[a] + fill[a]++] = ej[e] > 0;
        m->nbr[m->row[b] + fill[b]] = a; m->anti[m->row[b] + fill[b]++] = ej[e] > 0;
    }
    free(fill);
    return 0;
}

static void mirror_free(mirror_t *m) { free(m->row); free(m->nbr); free(m->anti); }

static void mirror_randomize(const mirror_t *m, uint64_t E, uint8_t *states) {
    const uint64_t W = (E + 31) / 32;
    for (uint64_t n = 0; n < m->nvars; ++n)
        for (uint64_t w = 0; w < W; ++w) {
            uint32_t c[4] = {(uint32_t)n, m->gw0 + (uint32_t)w, 0u, 1u << 24};
            philox4x32(10, c, m->k0, m->k1);
            for (uint64_t b = 0; b < 32 && w * 32 + b < E; ++b)
                states[(w * 32 + b) * m->nvars + n] = (c[0] >> b) & 1u;
        }
}

/* one colour-class sweep; replica e runs at beta[e] (beta_stride = 0: one beta for all) */
static void mirror_sweep(const mirror_t *m, uint64_t E, uint8_t *states, const double *beta,
                         int beta_stride, uint32_t sweep) {
    const uint64_t W = (E + 31) / 32, nvars = m->nvars;
    const int K = m->K;
    /* Memoised values only (same arithmetic as computing them at every use): the thresholds of a
     * shared beta per class, and the words R_0 .. R_{4 NCALL - 1} of one (site, word) stream, which
     * every replica bit of the word reads. */
    enum { TCACHE = 64 };
    uint64_t tcache[TCACHE];
    if (!beta_stride)
        for (int cls = 1; cls < TCACHE; ++cls) tcache[cls] = threshold(beta[0], 2.0 * m->jabs * (double)cls, K);
    const uint32_t nwords = 4u * ((uint32_t)K / 4 + 1);
    /* the sites of one colour share no bond when the colouring is proper: any update order (and
     * so threads) gives the same bits; otherwise they run in ascending order on one thread */
    for (uint32_t col = 0; col < m->ncolors; ++col)
#pragma omp parallel for schedule(static) if (m->proper && nvars > 4096)
        for (uint64_t n = 0; n < nvars; ++n) {
            if (m->colors[n] != col) continue;
            const int d = (int)(m->row[n + 1] - m->row[n]);
            uint32_t R[12];
            for (uint64_t w = 0; w < W; ++w) {
                int j = 0; /* resolver rank within the word */
                int have_r = 0;
                for (uint64_t b = 0; b < 32 && w * 32 + b < E; ++b) {
                    uint8_t *st = states + (w * 32 + b) * nvars;
                    int nsat = 0;
                    for (uint64_t k = m->row[n]; k < m->row[n + 1]; ++k) {
                        const int equal = st[n] == st[m->nbr[k]];
                        nsat += m->anti[k] ? !equal : equal;
                    }
                    const int cls = 2 * nsat - d;
                    if (cls <= 0) { st[n] ^= 1; continue; }
                    const double bt = beta[beta_stride ? (w * 32 + b) : 0];
                    const uint64_t T = (!beta_stride && cls < TCACHE) ? tcache[cls]
                                                                      : threshold(bt, 2.0 * m->jabs * (double)cls, K);
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

static double mirror_energy(const mirror_t *m, const uint8_t *st) {
    long long nsat = 0;
    for (uint64_t k = 0; k < m->nedges; ++k) {
        const int equal = st[m->ea[k]] == st[m->eb[k]];
        nsat += (m->ej[k] > 0) ? !equal : equal;
    }
    return m->jabs * (double)((long long)m->nedges - 2 * nsat);
}

/* states: bool[E, nvars], in/out (filled from Philox when randomize != 0, or broadcast from
 * init_state when given).  energies_per_sweep: double[E, nsweeps] or NULL.  final_energies:
 * double[E] or NULL.  per_replica_beta != 0: betas is double[E] (one per replica, constant over
 * the sweeps) instead of double[nsweeps]. */
ORC_EXPORT int msc_mirror_run(uint64_t nvars, uint64_t nedges, const uint64_t *ea,
                              const uint64_t *eb, const double *ej, const uint32_t *colors,
                              uint32_t ncolors, uint64_t E, uint64_t seed,
                              uint64_t replica_offset, int K, int rounds, int randomize,
                              const uint8_t *init_state, const double *betas, uint64_t nsweeps,
                              uint64_t sweep0, uint8_t *states, double *energies_per_sweep,
                              double *final_energies, int per_replica_beta) {
    mirror_t m;
    int rc = mirror_init(&m, nvars, nedges, ea, eb, ej, colors, ncolors, seed, replica_offset, K, rounds);
    if (rc) return rc;
    if (randomize) mirror_randomize(&m, E, states);
    else if (init_state)
        for (uint64_t e = 0; e < E; ++e) memcpy(states + e * nvars, init_state, nvars);
    for (uint64_t t = 0; t < nsweeps; ++t) {
        if (per_replica_beta) mirror_sweep(&m, E, states, betas, 1, (uint32_t)(sweep0 + t));
        else mirror_sweep(&m, E, states, betas + t, 0, (uint32_t)(sweep0 + t));
        if (energies_per_sweep) {
#pragma omp parallel for schedule(static)
            for (uint64_t e = 0; e < E; ++e)
                energies_per_sweep[e * nsweeps + t] = mirror_energy(&m, states + e * nvars);
        }
    }
    if (final_energies) {
#pragma omp parallel for schedule(static)
        for (uint64_t e = 0; e < E; ++e) final_energies[e] = mirror_energy(&m, states + e * nvars);
    }
    mirror_free(&m);
    return 0;
}

/* One pass of two-spin edge moves (pyisingmontecarlo_b200/csrc/moves.cu: k_edge_general), the
 * classes of the library's strong edge colouring one after the other.  The pair (a, b) counts the
 * satisfied bonds among its D outer bonds (adjacency entries of a and b that do not lead to the
 * other end); dE = 2|J|(2 n_sat - D); same threshold / plane / resolver rule as a site of degree D,
 * on the stream (edge, replica word, timestep, call | pass << 8 | 4 << 24). */
static uint32_t edge_stream_word(int rounds, int K, uint32_t eid, uint32_t gw, uint32_t sweep, uint32_t pass,
                                 uint32_t m, uint32_t k0, uint32_t k1) {
    return stream_word_tag(rounds, K, eid, gw, sweep, (pass << 8) | (4u << 24), m, k0, k1);
}

static void mirror_edge_pass(const mirror_t *m, const uint32_t *edge_cls, uint32_t ncls, uint64_t E,
                             uint8_t *states, double beta, uint32_t sweep, uint32_t pass, uint64_t *continuations) {
    const uint64_t W = (E + 31) / 32, nvars = m->nvars;
    const int K = m->K;
    const uint32_t nwords = 4u * ((uint32_t)K / 4 + 1);   /* words of the calls every decision makes */
    for (uint32_t c = 0; c < ncls; ++c)
        for (uint64_t e = 0; e < m->nedges; ++e) {
            if (edge_cls[e] != c) continue;
            const uint64_t end[2] = {m->ea[e], m->eb[e]};
            for (uint64_t w = 0; w < W; ++w) {
                int j = 0;
                for (uint64_t b = 0; b < 32 && w * 32 + b < E; ++b) {
                    uint8_t *st = states + (w * 32 + b) * nvars;
                    int nsat = 0, d = 0;
                    for (int s = 0; s < 2; ++s) {
                        const uint64_t u = end[s], other = end[1 - s];
                        for (uint64_t k = m->row[u]; k < m->row[u + 1]; ++k) {
                            if (m->nbr[k] == other) continue;
                            const int equal = st[u] == st[m->nbr[k]];
                            nsat += m->anti[k] ? !equal : equal;
                            ++d;
                        }
                    }
                    const int cls = 2 * nsat - d;
                    int accept = 1;
                    if (cls > 0) {
                        const uint64_t T = threshold(beta, 2.0 * m->jabs * (double)cls, K);
                        int decided = 0;
                        accept = 0;
                        for (int p = 0; p < K && !decided; ++p) {
                            const uint32_t rb = (edge_stream_word(m->rounds, K, (uint32_t)e, m->gw0 + (uint32_t)w, sweep,
                                                                  pass, (uint32_t)p, m->k0, m->k1) >> b) & 1u;
                            const uint32_t tb = (uint32_t)((T >> (K + 31 - p)) & 1ull);
                            if (rb != tb) { decided = 1; accept = rb < tb; }
                        }
                        if (!decided) {
                            const uint32_t v = edge_stream_word(m->rounds, K, (uint32_t)e, m->gw0 + (uint32_t)w, sweep,
                                                                pass, (uint32_t)(K + j), m->k0, m->k1);
                            accept = v < (uint32_t)(T & 0xFFFFFFFFull);
                            if (continuations && (uint32_t)(K + j) >= nwords) ++*continuations;
                            ++j;
                        }
                    }
                    if (accept) { st[end[0]] ^= 1; st[end[1]] ^= 1; }
                }
            }
        }
}

/* Timesteps of [one colour-class sweep] + edge_passes passes of edge moves, one beta per timestep
 * (ising_sim_set_moves with worms = 0).  states bool[E, nvars] in/out, filled from Philox when
 * randomize != 0; energies_per_step double[E, nsteps] or NULL.  continuations (or NULL) receives
 * the number of edge-move decisions that read a resolver word beyond the K/4 + 1 calls every
 * decision makes, i.e. a continuation round of the last block. */
ORC_EXPORT int msc_mirror_moves_ex(uint64_t nvars, uint64_t nedges, const uint64_t *ea, const uint64_t *eb,
                                   const double *ej, const uint32_t *colors, uint32_t ncolors,
                                   const uint32_t *edge_cls, uint32_t nedge_cls, uint64_t E, uint64_t seed,
                                   uint64_t replica_offset, int K, int rounds, int randomize, const double *betas,
                                   uint64_t nsteps, int spin_sweeps, uint32_t edge_passes, uint8_t *states,
                                   double *energies_per_step, uint64_t *continuations) {
    mirror_t m;
    int rc = mirror_init(&m, nvars, nedges, ea, eb, ej, colors, ncolors, seed, replica_offset, K, rounds);
    if (rc) return rc;
    if (randomize) mirror_randomize(&m, E, states);
    for (uint64_t t = 0; t < nsteps; ++t) {
        if (spin_sweeps) mirror_sweep(&m, E, states, betas + t, 0, (uint32_t)t);
        for (uint32_t pass = 0; pass < edge_passes; ++pass)
            mirror_edge_pass(&m, edge_cls, nedge_cls, E, states, betas[t], (uint32_t)t, pass, continuations);
        if (energies_per_step)
            for (uint64_t e = 0; e < E; ++e)
                energies_per_step[e * nsteps + t] = mirror_energy(&m, states + e * nvars);
    }
    mirror_free(&m);
    return 0;
}

ORC_EXPORT int msc_mirror_moves(uint64_t nvars, uint64_t nedges, const uint64_t *ea, const uint64_t *eb,
                                const double *ej, const uint32_t *colors, uint32_t ncolors,
                                const uint32_t *edge_cls, uint32_t nedge_cls, uint64_t E, uint64_t seed,
                                uint64_t replica_offset, int K, int rounds, int randomize, const double *betas,
                                uint64_t nsteps, int spin_sweeps, uint32_t edge_passes, uint8_t *states,
                                double *energies_per_step) {
    return msc_mirror_moves_ex(nvars, nedges, ea, eb, ej, colors, ncolors, edge_cls, nedge_cls, E, seed,
                               replica_offset, K, rounds, randomize, betas, nsteps, spin_sweeps, edge_passes,
                               states, energies_per_step, NULL);
}

/* exp(d), d <= 0, as the fixed sequence of IEEE double operations the device's swap kernel and
 * ising_pt_decide_swaps use (pyisingmontecarlo_b200/csrc/pt_exp.h), restated here so that the
 * mirror's swap decisions are bit-identical to the device's: d = k ln2 + r, degree-13 Taylor
 * polynomial of exp(r) in Horner form, 2^k from the exponent bits.  Compiled without FMA
 * contraction (the Makefile passes -ffp-contract=off). */
static double pt_exp_nonpos(double d) {
    if (!(d <= 0.0)) return 1.0;
    if (d < -700.0) return 0.0;
    const double INV_LN2 = 1.4426950408889634074;
    const double LN2_HI = 6.93147180369123816490e-01;
    const double LN2_LO = 1.90821492927058770002e-10;
    const double t = d * INV_LN2;
    const long long ki = (long long)(t + -0.5);
    const double kf = (double)ki;
    double r = d + -(kf * LN2_HI);
    r = r + -(kf * LN2_LO);
    static const double c[13] = {1.6059043836821613e-10, 2.0876756987868098e-09, 2.5052108385441720e-08,
                                 2.7557319223985888e-07, 2.7557319223985893e-06, 2.4801587301587302e-05,
                                 1.9841269841269841e-04, 1.3888888888888889e-03, 8.3333333333333332e-03,
                                 4.1666666666666664e-02, 1.6666666666666666e-01, 5.0000000000000000e-01,
                                 1.0000000000000000e+00};
    double p = c[0];
    for (int i = 1; i < 13; ++i) p = p * r + c[i];
    p = p * r + 1.0;
    const uint64_t bits = (uint64_t)(1023 + ki) << 52;
    double scale;
    memcpy(&scale, &bits, sizeof scale);
    return p * scale;
}

/* Parallel tempering exactly as libising_b200 runs it (ising_pt_timesteps_sample): one
 * configuration per replica bit, betas[R] by slot, cadence of tempering.rs:156-222, swap rule
 * and Philox draw of ising_pt_decide_swaps.  states[R, n_s, nvars], energies[R].  attempts and
 * accepts (or NULL): uint64[R - 1], the swaps tried and taken per pair of neighbouring slots,
 * indexed by the lower slot (ising_pt_get_pair_stats). */
ORC_EXPORT int msc_mirror_pt_ex(uint64_t nvars, uint64_t nedges, const uint64_t *ea,
                                const uint64_t *eb, const double *ej, const uint32_t *colors,
                                uint32_t ncolors, uint64_t R, const double *betas, uint64_t seed, int K,
                                int rounds, uint64_t timesteps, uint64_t swap_freq,
                                uint64_t sampling_freq, uint8_t *states_out, double *energies_out,
                                uint64_t *total_swaps, uint32_t *slot_of_cfg_out, uint64_t *attempts,
                                uint64_t *accepts) {
    if (swap_freq == 0 || sampling_freq == 0) return -3;
    mirror_t m;
    int rc = mirror_init(&m, nvars, nedges, ea, eb, ej, colors, ncolors, seed, 0, K, rounds);
    if (rc) return rc;
    uint8_t *cfg = (uint8_t *)malloc(R * nvars);
    mirror_randomize(&m, R, cfg);
    uint32_t *slot_of_cfg = (uint32_t *)malloc(sizeof(uint32_t) * R);
    uint32_t *cfg_of_slot = (uint32_t *)malloc(sizeof(uint32_t) * R);
    double *bcfg = (double *)malloc(sizeof(double) * R), *en = (double *)malloc(sizeof(double) * R);
    double *acc = (double *)calloc(R, sizeof(double));
    for (uint64_t r = 0; r < R; ++r) slot_of_cfg[r] = cfg_of_slot[r] = (uint32_t)r;
    for (uint64_t a = 0; a + 1 < R; ++a) {
        if (attempts) attempts[a] = 0;
        if (accepts) accepts[a] = 0;
    }
    const uint64_t ns = timesteps / sampling_freq;
    uint64_t remaining = timesteps, to_swap = swap_freq, to_sample = sampling_freq, k = 0;
    uint64_t swaps = 0, swap_step = 0, sweep = 0;
    while (remaining > 0) {
        uint64_t t = to_sample < to_swap ? to_sample : to_swap;
        if (remaining < t) t = remaining;
        for (uint64_t c = 0; c < R; ++c) bcfg[c] = betas[slot_of_cfg[c]];
        for (uint64_t i = 0; i < t; ++i) mirror_sweep(&m, R, cfg, bcfg, 1, (uint32_t)sweep++);
        for (uint64_t c = 0; c < R; ++c) en[c] = mirror_energy(&m, cfg + c * nvars);
        for (uint64_t s = 0; s < R; ++s) acc[s] += en[cfg_of_slot[s]] * (double)t;
        to_sample -= t; to_swap -= t; remaining -= t;
        if (to_swap == 0) {
            for (int parity = 0; parity < 2; ++parity)
                for (uint64_t a = parity; a + 1 < R; a += 2) {
                    const uint32_t ca = cfg_of_slot[a], cb = cfg_of_slot[a + 1];
                    const double d = (betas[a] - betas[a + 1]) * (en[ca] - en[cb]);
                    int accept = 1;
                    if (d < 0.0) {
                        uint32_t c4[4] = {(uint32_t)a, (uint32_t)parity, (uint32_t)swap_step, 2u << 24};
                        philox4x32(10, c4, m.k0, m.k1);
                        const double uu = ((double)c4[0] + 0.5) * (1.0 / 4294967296.0);
                        accept = uu < pt_exp_nonpos(d);
                    }
                    if (attempts) ++attempts[a];
                    if (accept) {
                        cfg_of_slot[a] = cb; cfg_of_slot[a + 1] = ca;
                        slot_of_cfg[cb] = (uint32_t)a; slot_of_cfg[ca] = (uint32_t)(a + 1);
                        ++swaps;
                        if (accepts) ++accepts[a];
                    }
                }
            ++swap_step;
            to_swap = swap_freq;
        }
        if (to_sample == 0) {
            if (k < ns)
                for (uint64_t s = 0; s < R; ++s)
                    memcpy(states_out + (s * ns + k) * nvars, cfg + (uint64_t)cfg_of_slot[s] * nvars, nvars);
            ++k;
            to_sample = sampling_freq;
        }
    }
    for (uint64_t s = 0; s < R; ++s) energies_out[s] = acc[s] / (double)timesteps;
    if (total_swaps) *total_swaps = swaps;
    if (slot_of_cfg_out) memcpy(slot_of_cfg_out, slot_of_cfg, sizeof(uint32_t) * R);
    free(cfg); free(slot_of_cfg); free(cfg_of_slot); free(bcfg); free(en); free(acc);
    mirror_free(&m);
    return 0;
}

ORC_EXPORT int msc_mirror_pt(uint64_t nvars, uint64_t nedges, const uint64_t *ea,
                             const uint64_t *eb, const double *ej, const uint32_t *colors,
                             uint32_t ncolors, uint64_t R, const double *betas, uint64_t seed, int K,
                             int rounds, uint64_t timesteps, uint64_t swap_freq,
                             uint64_t sampling_freq, uint8_t *states_out, double *energies_out,
                             uint64_t *total_swaps, uint32_t *slot_of_cfg_out) {
    return msc_mirror_pt_ex(nvars, nedges, ea, eb, ej, colors, ncolors, R, betas, seed, K, rounds, timesteps,
                            swap_freq, sampling_freq, states_out, energies_out, total_swaps, slot_of_cfg_out,
                            NULL, NULL);
}

/* One large 2D lattice, bit-packed along x (libising_b200 ising_strip_*, DESIGN.md "Single
 * lattice"): same decision rule, but the word of a decision is (row y, colour c, j = (x/2)/32),
 * its bit (x/2)%32, and the Philox counter (y, c << 30 | j, sweep, call).  state: bool[Ly, Lx]. */
ORC_EXPORT int msc_mirror_single(uint64_t Lx, uint64_t Ly, double jcoupling, uint64_t seed, int K,
                                 int rounds, int randomize, const double *betas, uint64_t nsweeps,
                                 uint8_t *state, double *energies_per_sweep) {
    if (Lx % 64 || (Ly & 1) || K < 1 || K > 8) return -1;
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    const double jabs = fabs(jcoupling);
    const int anti = jcoupling > 0;
    const uint64_t Wr = Lx / 64;
    if (randomize)
        for (uint64_t y = 0; y < Ly; ++y)
            for (uint32_t c = 0; c < 2; ++c)
                for (uint64_t j = 0; j < Wr; ++j) {
                    uint32_t ctr[4] = {(uint32_t)y, (c << 30) | (uint32_t)j, 0u, 1u << 24};
                    philox4x32(10, ctr, k0, k1);
                    for (uint32_t b = 0; b < 32; ++b) {
                        const uint64_t x = 2 * (32 * j + b) + ((y + c) & 1);
                        state[y * Lx + x] = (ctr[0] >> b) & 1u;
                    }
                }
    for (uint64_t t = 0; t < nsweeps; ++t) {
        for (uint32_t c = 0; c < 2; ++c)
            for (uint64_t y = 0; y < Ly; ++y)
                for (uint64_t j = 0; j < Wr; ++j) {
                    int tie_rank = 0;
                    for (uint32_t b = 0; b < 32; ++b) {
                        const uint64_t x = 2 * (32 * j + b) + ((y + c) & 1);
                        const uint8_t s = state[y * Lx + x];
                        const uint8_t nb[4] = {state[y * Lx + (x + 1) % Lx], state[y * Lx + (x + Lx - 1) % Lx],
                                               state[((y + 1) % Ly) * Lx + x], state[((y + Ly - 1) % Ly) * Lx + x]};
                        int nsat = 0;
                        for (int k = 0; k < 4; ++k) nsat += anti ? (s != nb[k]) : (s == nb[k]);
                        const int cls = 2 * nsat - 4;
                        if (cls <= 0) { state[y * Lx + x] ^= 1; continue; }
                        const uint64_t T = threshold(betas[t], 2.0 * jabs * (double)cls, K);
                        const uint32_t gw = (c << 30) | (uint32_t)j;
                        int decided = 0, accept = 0;
                        for (int p = 0; p < K && !decided; ++p) {
                            const uint32_t rb = (stream_word(rounds, K, (uint32_t)y, gw, (uint32_t)t, (uint32_t)p, k0, k1) >> b) & 1u;
                            const uint32_t tb = (uint32_t)((T >> (K + 31 - p)) & 1ull);
                            if (rb != tb) { decided = 1; accept = rb < tb; }
                        }
                        if (!decided) {
                            const uint32_t v = stream_word(rounds, K, (uint32_t)y, gw, (uint32_t)t, (uint32_t)(K + tie_rank), k0, k1);
                            accept = v < (uint32_t)(T & 0xFFFFFFFFull);
                            ++tie_rank;
                        }
                        if (accept) state[y * Lx + x] ^= 1;
                    }
                }
        if (energies_per_sweep) {
            long long nsat = 0;
            for (uint64_t y = 0; y < Ly; ++y)
                for (uint64_t x = 0; x < Lx; ++x) {
                    const uint8_t s = state[y * Lx + x];
                    const uint8_t r = state[y * Lx + (x + 1) % Lx], d = state[((y + 1) % Ly) * Lx + x];
                    nsat += anti ? (s != r) : (s == r);
                    nsat += anti ? (s != d) : (s == d);
                }
            energies_per_sweep[t] = jabs * (double)(2 * (long long)(Lx * Ly) - 2 * nsat);
        }
    }
    return 0;
}

/* A band of rows of the same lattice: state = bool[nrows, Lx] holds the global rows
 * y0 .. y0 + nrows - 1 (0 < y0, y0 + nrows < Ly: no periodic wrap inside the band).  The decision
 * of a site depends only on its global coordinates, so the band reproduces the big lattice
 * wherever its neighbours are known: colour phase q (q = 0 .. 2 nsweeps - 1) updates the rows
 * [q + 1, nrows - q - 1), and after nsweeps sweeps the rows [2 nsweeps, nrows - 2 nsweeps) equal
 * those of the full lattice - the check a 65536^2 lattice allows on a CPU. */
ORC_EXPORT int msc_mirror_single_band(uint64_t Lx, uint64_t y0, uint64_t nrows, double jcoupling, uint64_t seed,
                                      int K, int rounds, int randomize, const double *betas, uint64_t nsweeps,
                                      uint8_t *state) {
    if (Lx % 64 || K < 1 || K > 8 || nrows < 4 * nsweeps + 1) return -1;
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    const double jabs = fabs(jcoupling);
    const int anti = jcoupling > 0;
    const uint64_t Wr = Lx / 64;
    if (randomize)
        for (uint64_t r = 0; r < nrows; ++r)
            for (uint32_t c = 0; c < 2; ++c)
                for (uint64_t j = 0; j < Wr; ++j) {
                    const uint64_t y = y0 + r;
                    uint32_t ctr[4] = {(uint32_t)y, (c << 30) | (uint32_t)j, 0u, 1u << 24};
                    philox4x32(10, ctr, k0, k1);
                    for (uint32_t b = 0; b < 32; ++b) {
                        const uint64_t x = 2 * (32 * j + b) + ((y + c) & 1);
                        state[r * Lx + x] = (ctr[0] >> b) & 1u;
                    }
                }
    for (uint64_t t = 0; t < nsweeps; ++t)
        for (uint32_t c = 0; c < 2; ++c) {
            const uint64_t q = 2 * t + c;
            for (uint64_t r = q + 1; r + q + 1 < nrows; ++r)
                for (uint64_t j = 0; j < Wr; ++j) {
                    const uint64_t y = y0 + r;
                    int tie_rank = 0;
                    for (uint32_t b = 0; b < 32; ++b) {
                        const uint64_t x = 2 * (32 * j + b) + ((y + c) & 1);
                        const uint8_t s = state[r * Lx + x];
                        const uint8_t nb[4] = {state[r * Lx + (x + 1) % Lx], state[r * Lx + (x + Lx - 1) % Lx],
                                               state[(r + 1) * Lx + x], state[(r - 1) * Lx + x]};
                        int nsat = 0;
                        for (int k = 0; k < 4; ++k) nsat += anti ? (s != nb[k]) : (s == nb[k]);
                        const int cls = 2 * nsat - 4;
                        if (cls <= 0) { state[r * Lx + x] ^= 1; continue; }
                        const uint64_t T = threshold(betas[t], 2.0 * jabs * (double)cls, K);
                        const uint32_t gw = (c << 30) | (uint32_t)j;
                        int decided = 0, accept = 0;
                        for (int p = 0; p < K && !decided; ++p) {
                            const uint32_t rb = (stream_word(rounds, K, (uint32_t)y, gw, (uint32_t)t, (uint32_t)p, k0, k1) >> b) & 1u;
                            const uint32_t tb = (uint32_t)((T >> (K + 31 - p)) & 1ull);
                            if (rb != tb) { decided = 1; accept = rb < tb; }
                        }
                        if (!decided) {
                            const uint32_t v = stream_word(rounds, K, (uint32_t)y, gw, (uint32_t)t, (uint32_t)(K + tie_rank), k0, k1);
                            accept = v < (uint32_t)(T & 0xFFFFFFFFull);
                            ++tie_rank;
                        }
                        if (accept) state[r * Lx + x] ^= 1;
                    }
                }
        }
    return 0;
}
