// Launch wrappers of the sm_100a kernels (sweep_stencil.cu, sweep_general.cu, strip.cu, observables.cu, state_io.cu).  Host-callable, no CUDA types beyond
// cudaStream_t so that api.cpp stays plain C++.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace ising {

// Philox4x32 rounds of the production streams: 7 is the Crush-resistant minimum of the Random123
// paper (Salmon et al., SC'11, table 2) and the default; 10 is the paper's recommended safety
// margin, selectable per simulation (ising_sim_configure).  The launch-bound fast paths
// (cooperative kernel, degree-specialised general kernels, row walk) are built for the default.
constexpr int kDefaultRounds = 7;

// SM count of the current device (cudaDevAttrMultiProcessorCount, cached per device): grids of the
// persistent / grid-stride kernels are sized in multiples of it, never from a literal.
unsigned device_sms();

// Replica-bit-packed spin storage.  One 32-bit word = one site in 32 experiments.
//   general graph : word(n, w) at n * W + w                          (natural site order)
//   stencil       : colour-compacted checkerboard, word(c, row, xh, w) at
//                   ((c * rows + row) * Lxh + xh) * W + w, row = z * Ly + y,
//                   x = 2 * xh + ((y + z + c) & 1)
struct Layout {
    int32_t kind;  // ISING_KIND_*
    uint32_t Lx, Ly, Lz, Lxh, rows;
    uint32_t W;    // words per site = ceil(E / 32)
    uint64_t nvars;
    uint64_t halfN;  // sites per colour (stencil)
};

// Acceptance thresholds of the multi-spin-coded Metropolis step for <= 3 uphill classes.
// T_c = floor(exp(-beta dE_c) * 2^(K+32)); plane[c][p] is all-ones iff bit (K+31-p) of T_c
// is set (MSB first), low[c] = T_c mod 2^32 is what the per-bit resolver compares against.
struct MscThresholds {
    uint32_t plane[3][8];
    uint32_t low[3];
};

struct SweepArgs {
    uint32_t* spins;
    const uint32_t* jmask;  // stencil +-J: [colour][6 or 4][halfN] bond masks, else nullptr
    const uint32_t* jmask8 = nullptr;  // the same, site-major [colour][halfN][8] (row-walk kernel)
    int sm_count = 0;       // SMs of the device (persistent grids)
    Layout lay;
    uint32_t sweep;         // global sweep index (Philox counter word 2)
    uint32_t key0, key1;    // Philox key = seed
    uint32_t gw0;           // global replica-word index of local word 0
    uint32_t antiferro;     // uniform-sign lattices: all-ones iff J > 0
    int planes, rounds;
    MscThresholds th;
    // when non-null the second colour phase also accumulates the per-experiment satisfied-bond
    // count after the sweep into nsat_out[W * 32] (must be zeroed by the caller)
    unsigned long long* nsat_out;
    // The blocks of the accumulating phase add into nsat_out[(block % nsat_copies) * nsat_stride + e]:
    // a few hundred blocks finishing together would otherwise serialise their atomics on the same
    // W * 32 addresses (measured: ~4 us of a 13 us phase at 128 replicas).  The reader sums the copies.
    uint32_t nsat_copies = 1;
    uint32_t nsat_stride = 0;
    // per-replica inverse temperatures (planes must be 6): bit-sliced threshold tables
    //   tplane[(w * 3 + cls) * 8 + p], tlow[(w * 32 + b) * 3 + cls];  nullptr = one beta (th)
    const uint32_t* tplane;
    const uint32_t* tlow;
};
// ---- uniform longitudinal field on a torus (sweep_field.cu) ----------------------------------
// The class of a site is (spin s, n_sat): s = 1 for an up spin (sigma = +1), n_sat = 0 .. 2*DIM
// satisfied bonds, dE = 2|J|(2 n_sat - 2 DIM) + 2 h sigma.  plane[p][s][n] is all-ones iff bit
// (K+31-p) of the class threshold T is set, low[s][n] = T mod 2^32, up[s][n] all-ones iff dE > 0
// (other classes flip unconditionally).  Entries n > 2*DIM are never read.
struct FieldThresholds {
    uint32_t plane[8][2][8];
    uint32_t low[2][8];
    uint32_t up[2][8];
};
// both colour phases of one sweep in a field (2 launches, a.th unused); returns launches or -1
int launch_sweep_field(const SweepArgs& a, const FieldThresholds& th, cudaStream_t st);
// out[e * estride + eoff + t] = jabs (nbonds - 2 nsat[t * cw + e]) + h (nsites - 2 up[t * cw + e])
int launch_energy_field(const unsigned long long* nsat, const unsigned long long* up, uint64_t E, uint64_t cw,
                        uint64_t nt, double jabs, uint64_t nbonds, double h, uint64_t nsites, double* out_dev,
                        uint64_t estride, uint64_t eoff, cudaStream_t st);

// T64[row * 3 + cls], row = slot_of_replica[e] (nullptr: row = e) -> tplane / tlow of the stencil kernels
int launch_build_tables_stencil(const unsigned long long* t64, const uint32_t* slot_of_replica, uint32_t W,
                                int K, uint32_t* plane_out, uint32_t* low_out, cudaStream_t st);

// both colour phases of one sweep (2 launches); returns launches made or -1
int launch_sweep_stencil(const SweepArgs& a, cudaStream_t st);
// the same through the persistent row-walk kernels (sweep_rows.cuh); 0 = configuration not covered
int launch_sweep_rows_2d(const SweepArgs& a, cudaStream_t st);
int launch_sweep_rows_3d(const SweepArgs& a, cudaStream_t st);
// A chunk of nsweeps whole sweeps in ONE cooperative launch (grid barrier between colour phases):
// for lattices so small that a colour phase is launch-bound.  th_dev[nsweeps] = thresholds per
// sweep (device memory); hist (or nullptr) receives the per-sweep n_sat at hist[t * cw + e].
// Returns 1 if launched, 0 if this configuration has no cooperative variant, -1 on error.
int launch_sweeps_stencil_coop(const SweepArgs& a, const MscThresholds* th_dev, uint32_t nsweeps,
                               unsigned long long* hist, uint32_t cw, cudaStream_t st);
// The same for lattices of at most 8192 site-words per colour, inside ONE thread-block cluster
// (hardware cluster barrier between the colour phases); K = 6.  hist as above.
int launch_sweeps_stencil_cluster(const SweepArgs& a, const MscThresholds* th_dev, uint32_t nsweeps,
                                  unsigned long long* hist, uint32_t cw, cudaStream_t st);
// n_sat[e] += number of satisfied bonds of experiment e (one colour's sites cover every bond)
int launch_nsat_stencil(const uint32_t* spins, const uint32_t* jmask, const Layout& lay,
                        uint32_t antiferro, unsigned long long* nsat, cudaStream_t st);
// up[e] += number of up spins of experiment e
int launch_count_up(const uint32_t* spins, const Layout& lay, unsigned long long* up,
                    cudaStream_t st, bool pair = false);
// a[i] ^= b[i] for n words
int launch_xor_words(uint32_t* a, const uint32_t* b, uint64_t n, cudaStream_t st);
int launch_overlap_from_counts(const unsigned long long* dis, uint64_t P, uint64_t nsites,
                               double* out_dev, uint64_t stride, uint64_t off, cudaStream_t st);
int launch_init_random(uint32_t* spins, const Layout& lay, uint32_t key0, uint32_t key1,
                       uint32_t gw0, cudaStream_t st);
int launch_init_broadcast(uint32_t* spins, const Layout& lay, const uint8_t* state_dev,
                          cudaStream_t st);
int launch_pack_states(uint32_t* spins, const Layout& lay, const uint8_t* states_dev,
                       uint64_t E, cudaStream_t st);
// bool[E, nvars] (row stride = out_stride bytes between experiments) from packed words
int launch_unpack_states(const uint32_t* spins, const Layout& lay, uint8_t* out_dev, uint64_t E,
                         uint64_t out_stride, cudaStream_t st);
int launch_import_natural(uint32_t* spins, const Layout& lay, const uint32_t* in_dev, cudaStream_t st);
// packed words in natural order [nvars][W]
int launch_export_natural(const uint32_t* spins, const Layout& lay, uint32_t* out_dev,
                          cudaStream_t st);
// energies[e * estride + eoff] = scale * (double)(nbonds - mult * nsat[e]); mult = 2 when
// nsat counts every satisfied bond once (stencil), 1 when it counts it from both ends
int launch_energy_from_nsat(const unsigned long long* nsat, uint64_t E, double scale,
                            uint64_t nbonds, int mult, double* out_dev, uint64_t estride,
                            uint64_t eoff, cudaStream_t st);

// hist[(t * copies + c) * cw + e], summed over the copies c
int launch_energy_from_hist(const unsigned long long* hist, uint64_t E, uint64_t cw, uint64_t nt,
                            double scale, uint64_t nbonds, int mult, double* out_dev,
                            cudaStream_t st, uint32_t copies = 1);

// ---- general graphs (arbitrary edge list, greedy colouring), all |J| equal, no bias -----------
constexpr int GEN_MAX_DEG = 15;   // satisfied-bond count fits 4 bit-planes
constexpr int GEN_MAX_CLS = 8;    // uphill classes of one degree: n_sat = deg/2+1 .. deg

struct GenGroup {             // the sites of one colour that have the same degree
    const uint32_t* sites;    // [count] natural site index
    const uint32_t* nbr;      // [deg][count] neighbour site index
    const uint32_t* anti;     // [count] bit k set iff the bond to neighbour k has J > 0
    uint32_t count, deg;
};

// thresholds of one degree, same for every replica (uniform beta)
struct GenThresholds {
    uint32_t plane[GEN_MAX_CLS][8];
    uint32_t low[GEN_MAX_CLS];
};

// thresholds that differ per replica (parallel tempering): bit-sliced in device memory
//   plane[((deg * W + w) * GEN_MAX_CLS + cls) * 8 + p]: bit b = threshold bit p of replica 32w+b
//   low[((deg * E32 + e) * GEN_MAX_CLS + cls)],  E32 = 32 * W
struct GenTables {
    const uint32_t* plane;
    const uint32_t* low;
};

struct GenSweepArgs {
    uint32_t* spins;          // [nvars][W]
    uint32_t W;
    uint32_t sweep, key0, key1, gw0;
    int planes, rounds;
    GenThresholds th;         // used when tables.plane == nullptr
    GenTables tables;
};
int launch_sweep_general(const GenSweepArgs& a, const GenGroup& g, cudaStream_t st);
// T64[slot][deg 0..GEN_MAX_DEG][cls] (host-computed) + slot_of_replica[E32] -> GenTables
int launch_build_tables(const unsigned long long* t64, const uint32_t* slot_of_replica,
                        uint32_t W, int K, uint32_t* plane_out, uint32_t* low_out,
                        cudaStream_t st);
// nsat2[e] += sum over sites of the satisfied bonds at that site (every bond counted twice)
int launch_nsat_general(const uint32_t* spins, uint64_t nvars, uint32_t W, const uint32_t* row,
                        const uint32_t* nbr, const uint8_t* anti, unsigned long long* nsat2,
                        cudaStream_t st);

// ---- device-resident replica exchange (pt_device.cu) ------------------------------------------
int launch_pt_swap(const double* betas, const double* e_all, const uint32_t* gidx, uint32_t* slot_of_cfg,
                   uint32_t* cfg_of_slot, uint32_t R, uint64_t seed, unsigned long long* stats,
                   uint32_t* slot_of_replica, uint32_t word_lo, uint32_t e32, cudaStream_t st);
int launch_pt_local_slots(const uint32_t* slot_of_cfg, uint32_t R, uint32_t* slot_of_replica,
                          uint32_t word_lo, uint32_t e32, cudaStream_t st);
int launch_pt_gather_rows(const uint8_t* rows, uint64_t n, const uint32_t* gidx, const uint32_t* cfg_of_slot,
                          uint32_t R, uint8_t* out, cudaStream_t st);

// fused post-sweep part of a tempering cycle (one block), see pt_device.cu
struct PtCycleArgs {
    unsigned long long* nsat;      // [e32] local satisfied-bond counters (zeroed on exit), or nullptr
    double* e_local;               // [e32] local energies (written when nsat != nullptr)
    double* e_all;                 // gathered energies; written from e_local when `identity`
    uint32_t E, e32, identity;     // local experiments; 32 W; 1: one rank holds everything (gidx = id)
    double scale;                  // |J|
    unsigned long long nbonds;
    int mult;
    const uint32_t* gidx;
    const double* betas;
    uint32_t* slot_of_cfg;
    uint32_t* cfg_of_slot;
    uint32_t R, key0, key1;
    unsigned long long* stats;
    uint32_t* slot_of_replica;
    uint32_t word_lo;
    double* acc;
    double t;                      // sweeps since the last energies (weight of the time average)
    int do_swap;
    // stencil threshold tables (W * 3 rows), nullptr: the caller rebuilds tables itself
    const unsigned long long* t64;
    uint32_t W;
    int K;
    uint32_t* tplane;
    uint32_t* tlow;
};
int launch_pt_cycle(const PtCycleArgs& a, cudaStream_t st);

// ---- arbitrary real couplings and biases (float local field per replica bit) -----------------
struct RealSweepArgs {
    uint32_t* spins;          // [nvars][W]
    const uint32_t* sites;    // sites of the colour being updated
    uint32_t count;
    const uint32_t* row;      // CSR (u32 offsets), neighbours ascending
    const uint32_t* nbr;
    const float* jf;          // coupling per CSR entry
    const float* biasf;       // per site
    uint32_t W;
    float beta;
    // per-replica inverse temperatures (tempering): replica bit e of this sim runs at the f64 whose
    // bit pattern is beta_slots[slot_of_replica[e]]; nullptr = `beta` for every replica
    const unsigned long long* beta_slots;
    const uint32_t* slot_of_replica;
    uint32_t sweep, key0, key1, gw0;
    int rounds;
};
int launch_sweep_real(const RealSweepArgs& a, cudaStream_t st);
// energies[e] += sum_edges J s s - sum_i b_i s_i in f64 (every bond seen from both ends, halved)
int launch_energy_real(const uint32_t* spins, uint64_t nvars, uint32_t W, const uint32_t* row,
                       const uint32_t* nbr, const double* jv, const double* bias,
                       double* energies /* [32 W], zeroed */, cudaStream_t st);

// ---- non-basic moves of a timestep (moves.cu): two-spin edge moves and worm (chain) moves ------
struct MoveGraph {            // CSR with f32 couplings and biases (ensure_real_on_device)
    const uint32_t* row;
    const uint32_t* nbr;
    const float* jf;
    const float* biasf;
};
struct EdgeMoveArgs {
    uint32_t* spins;
    Layout lay;
    MoveGraph g;
    const uint32_t* ea;       // one class of the strong edge colouring
    const uint32_t* eb;
    const uint32_t* eid;      // index of the edge in the edge list (Philox counter word 0)
    const float* wrel;        // |J| / max |J| per edge (importance sampling) or nullptr
    uint32_t count;
    float beta;
    uint32_t sweep, key0, key1, gw0, pass;
    int rounds;
};
int launch_edge_moves(const EdgeMoveArgs& a, cudaStream_t st);
// bit-sliced edge moves (all |J| equal, no bias): the bonds of one class of the strong edge
// colouring that see the same number of outer bonds, in ELL form; spins addressed by slot
struct EdgeGroup {
    const uint32_t* sa;       // [count] slot (word base / W) of end a
    const uint32_t* sb;       // [count] slot of end b
    const uint32_t* eid;      // [count] index in the edge list (Philox counter word 0)
    const uint32_t* anti;     // [count] bit k set iff outer bond k has J > 0
    const uint32_t* endp;     // [count] bit k set iff outer bond k hangs on end b
    const uint32_t* nbr;      // [deg][count] slot of the far end of outer bond k
    uint32_t count, deg;
};
// a.th = thresholds of degree g.deg (fill_gen_thresholds), a.sweep = timestep
int launch_edge_general(const GenSweepArgs& a, const EdgeGroup& g, uint32_t pass, cudaStream_t st);
constexpr int WORM_MAX_LEN = 8;
struct WormArgs {
    uint32_t* spins;
    Layout lay;
    MoveGraph g;
    uint64_t E, replica_offset;
    uint32_t nworms, worm0, len;   // worms per experiment of this launch, index of the first, sites per worm
    float beta;
    uint32_t sweep, key0, key1;
    int rounds;
};
int launch_worm_moves(const WormArgs& a, cudaStream_t st);

int launch_copy_strided_f64(const double* in, uint64_t E, double* out, uint64_t estride,
                            uint64_t eoff, cudaStream_t st);
int launch_transpose_hist_f64(const double* hist, uint64_t E, uint64_t cw, uint64_t nt, double* out,
                              cudaStream_t st);

// ---- one large 2D lattice, bit-packed along x (config 5), uniform J, row strips ---------------
// Colour-compacted: S[c][r][j], r = 0 .. rows + 2 ghost - 1 (the first and last `ghost` rows
// hold copies of the neighbouring strips' boundary rows; local row l is r = ghost + l),
// j = 0 .. Wr-1, Wr = Lx / 64 words per colour row; bit b of word j of global row y is site
// x = 2 (32 j + b) + ((y + c) & 1).
struct StripGeom {
    uint32_t Wr;        // words per colour row
    uint32_t rows;      // local rows
    uint32_t row0;      // global index of the first local row
    uint32_t Ly;        // global number of rows
    uint32_t ghost;     // ghost rows on each side (>= 1)
};
// global row of storage row r (ghost rows wrap around the torus)
#if defined(__CUDACC__)
__host__ __device__
#endif
inline uint32_t strip_global_row(const StripGeom& g, uint32_t r) {
    uint32_t y = g.row0 + r;          // row0 + r - ghost, modulo Ly
    if (y < g.ghost) y += g.Ly;
    y -= g.ghost;
    if (y >= g.Ly) y -= g.Ly;
    return y;
}
struct StripSweepArgs {
    uint32_t* spins;    // [2][rows + 2 ghost][Wr]
    StripGeom g;
    uint32_t colour, sweep, key0, key1, antiferro;
    int planes, rounds;
    MscThresholds th;   // classes: n_sat = 3 -> dE = 4|J|, n_sat = 4 -> dE = 8|J|
    uint32_t r_begin, r_count;  // storage rows to update: [r_begin, r_begin + r_count) within [1, rows + 2 ghost - 1)
};
int launch_strip_phase(const StripSweepArgs& a, cudaStream_t st);
// grid / block of a strip colour phase with V words per thread (strip.cu)
void strip_phase_shape(const StripSweepArgs& a, uint32_t V, dim3* grid, dim3* block);
// the same colour phase in a uniform field h (strip_field.cu): classes (spin, n_sat = 0..4) with the
// thresholds th of dE = 2|J|(2 n_sat - 4) + 2 h sigma; a.th unused
int launch_strip_phase_field(const StripSweepArgs& a, const FieldThresholds& th, cudaStream_t st);
// Both colour phases of one sweep in a single out-of-place pass (src -> dst): colour 0 on storage
// rows [r_begin, r_begin + r_count), colour 1 on [r_begin + 1, r_begin + r_count - 1); a.colour is
// ignored.  Returns 1 when launched, 0 when the geometry is not covered, -1 on error.
int launch_strip_sweep_fused(const StripSweepArgs& a, const uint32_t* src, uint32_t* dst, cudaStream_t st);
int launch_strip_init_random(uint32_t* spins, const StripGeom& g, uint32_t key0, uint32_t key1,
                             cudaStream_t st);
// acc[0] += satisfied bonds seen from colour-0 sites (every bond once), acc[1] += up spins
int launch_strip_observables(const uint32_t* spins, const StripGeom& g, uint32_t antiferro,
                             unsigned long long* acc, cudaStream_t st);
// bool rows [nrows][Lx] of local rows l0 .. l0 + nrows - 1 from the packed strip (default: all)
int launch_strip_unpack(const uint32_t* spins, const StripGeom& g, uint8_t* out_dev, cudaStream_t st,
                        uint32_t l0 = 0, uint32_t nrows = 0xFFFFFFFFu);

struct ReplayArgs {
    uint64_t E, N, A;
    const uint64_t* row;   // CSR offsets (nvars + 1)
    const uint32_t* nbr;
    const double* jv;
    const double* bias;
    const uint32_t* sites;  // [E, A]
    const double* u;        // [E, A]
    uint8_t* states;        // [E, N], holds init on entry, final state on exit
    double* energies;       // [E]
    double beta;
    unsigned int* ambiguous;  // incremented when u is within rounding of exp(-beta dE)
};
int launch_replay(const ReplayArgs& a, cudaStream_t st);

}  // namespace ising
