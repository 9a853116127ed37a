// TEST INFRASTRUCTURE (CPU suite only).  The float-field kernels - colour-class sweeps on real
// couplings and biases (k_sweep_real, k_energy_real of csrc/sweep_general.cu), the float two-spin
// edge moves and the worm moves (k_edge_moves, k_worm_moves of csrc/moves.cu) - from their own
// source on the host (cuda_on_host.h), for tests/test_device_source_on_host.py: the statistical
// check against exact enumeration, and the decision-by-decision check against the f64 reference of
// tests/float_reference.py (every accept / reject outside the rounding band of the f32 field and
// the fast exponential equals the reference's; the same gate runs on the GPU in
// tests/test_gpu_float_path.py).  Every argument the library's launchers set is an argument here:
// Philox rounds, the global replica word of local word 0 (gw0), the replica offset of the worms,
// per-replica betas through a slot map, and the checkerboard spin layout for the moves.
#include "cuda_on_host.h"

#include "prepared/real_kernels.cuh"
#include "prepared/float_moves_kernels.cuh"

using namespace ising;

namespace {
Layout make_layout(int kind, uint32_t Lx, uint32_t Ly, uint32_t Lz, uint64_t nvars, uint32_t W) {
    Layout L;
    memset(&L, 0, sizeof L);
    L.kind = kind;
    L.W = W;
    L.nvars = nvars;
    if (kind != ISING_KIND_GENERAL) {
        L.Lx = Lx; L.Ly = Ly; L.Lz = kind == ISING_KIND_STENCIL3D ? Lz : 1;
        L.Lxh = Lx / 2; L.rows = L.Ly * L.Lz;
        L.halfN = nvars / 2;
    }
    return L;
}
dim3 site_block(uint32_t W) {
    const uint32_t wx = W >= 32 ? 32 : pow2_ceil(W);
    return dim3(wx, 256 / wx, 1);
}
}  // namespace

// beta_slots / slot_of_replica: nullptr = `beta` for every replica (RealSweepArgs)
extern "C" void emu_sweep_real(uint32_t* spins, const uint32_t* sites, uint32_t count, const uint32_t* row,
                               const uint32_t* nbr, const float* jf, const float* biasf, uint32_t W, float beta,
                               uint32_t sweep, uint64_t seed, uint32_t gw0, int rounds,
                               const unsigned long long* beta_slots, const uint32_t* slot_of_replica) {
    if (count == 0) return;
    RealSweepArgs a;
    memset(&a, 0, sizeof a);
    a.spins = spins; a.sites = sites; a.count = count; a.row = row; a.nbr = nbr; a.jf = jf; a.biasf = biasf;
    a.W = W; a.beta = beta; a.sweep = sweep; a.key0 = (uint32_t)seed; a.key1 = (uint32_t)(seed >> 32); a.gw0 = gw0;
    a.beta_slots = beta_slots; a.slot_of_replica = slot_of_replica;
    a.rounds = rounds;
    const dim3 block = site_block(W);
    if (rounds == 7) emu::launch_v(k_sweep_real<7>, dim3((count + block.y - 1) / block.y), block, 0, a);
    else emu::launch_v(k_sweep_real<10>, dim3((count + block.y - 1) / block.y), block, 0, a);
}

extern "C" void emu_energy_real(const uint32_t* spins, uint64_t nvars, uint32_t W, const uint32_t* row,
                                const uint32_t* nbr, const double* jv, const double* bias, double* energies) {
    const uint32_t wx = W >= 32 ? 32 : pow2_ceil(W);
    const dim3 block(wx, 128 / wx, 1);
    uint64_t g = (nvars + block.y - 1) / block.y;
    if (g > 3) g = 3;
    emu::launch_v(k_energy_real, dim3((unsigned)g, (W + wx - 1) / wx, 1), block, 0, spins, nvars, W, row, nbr, jv, bias,
                  energies);
}

extern "C" void emu_edge_moves(uint32_t* spins, uint64_t nvars, uint32_t W, const uint32_t* row, const uint32_t* nbr,
                               const float* jf, const float* biasf, const uint32_t* ea, const uint32_t* eb,
                               const uint32_t* eid, const float* wrel, uint32_t count, float beta, uint32_t sweep,
                               uint64_t seed, uint32_t gw0, uint32_t pass, int rounds) {
    if (count == 0) return;
    EdgeMoveArgs a;
    memset(&a, 0, sizeof a);
    a.spins = spins; a.lay = make_layout(ISING_KIND_GENERAL, 0, 0, 0, nvars, W); a.g = MoveGraph{row, nbr, jf, biasf};
    a.ea = ea; a.eb = eb; a.eid = eid; a.wrel = wrel; a.count = count; a.beta = beta;
    a.sweep = sweep; a.key0 = (uint32_t)seed; a.key1 = (uint32_t)(seed >> 32); a.gw0 = gw0; a.pass = pass;
    a.rounds = rounds;
    const dim3 block = site_block(W);
    if (rounds == 7) emu::launch_v(k_edge_moves<7>, dim3((count + block.y - 1) / block.y), block, 0, a);
    else emu::launch_v(k_edge_moves<10>, dim3((count + block.y - 1) / block.y), block, 0, a);
}

// kind / Lx / Ly / Lz: the spin layout (ISING_KIND_GENERAL = natural order, else the checkerboard)
extern "C" void emu_worm_moves(uint32_t* spins, int kind, uint32_t Lx, uint32_t Ly, uint32_t Lz, uint64_t nvars,
                               uint32_t W, const uint32_t* row, const uint32_t* nbr, const float* jf, const float* biasf,
                               uint64_t E, uint64_t replica_offset, uint32_t nworms, uint32_t len, float beta,
                               uint32_t sweep, uint64_t seed, int rounds) {
    WormArgs a;
    memset(&a, 0, sizeof a);
    a.spins = spins; a.lay = make_layout(kind, Lx, Ly, Lz, nvars, W); a.g = MoveGraph{row, nbr, jf, biasf};
    a.E = E; a.replica_offset = replica_offset; a.nworms = nworms; a.worm0 = 0; a.len = len; a.beta = beta;
    a.sweep = sweep; a.key0 = (uint32_t)seed; a.key1 = (uint32_t)(seed >> 32); a.rounds = rounds;
    if (rounds == 7) emu::launch_v(k_worm_moves<7>, dim3((unsigned)((E + 127) / 128)), dim3(128), 0, a);
    else emu::launch_v(k_worm_moves<10>, dim3((unsigned)((E + 127) / 128)), dim3(128), 0, a);
}
