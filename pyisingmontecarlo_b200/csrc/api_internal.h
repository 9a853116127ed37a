// Internals shared by the translation units that implement the C ABI (api_*.cu): the opaque
// objects behind the handles, error reporting, the context's buffer caches.  Nothing here is
// exported (the library is built with -fvisibility=hidden).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <memory>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/ising_b200.h"
#include "graph.h"
#include "kernels.h"
#include "philox.h"

using namespace ising;

// ------------------------------------------------------------------------------------------
// objects
// ------------------------------------------------------------------------------------------
struct ising_ctx {
    // Every extern "C" entry point that touches a context holds this for the call: the scratch
    // buffers, the free list, the timing events and the copy stream are per-context state, and
    // ctypes releases the GIL (the pyo3 reference holds it, so its calls were serialised too).
    // Recursive because entry points are built from each other (create -> randomize, ...).
    std::recursive_mutex mu;
    // Objects created from a context (graphs, sims, ladders, strips, communicators) keep it alive:
    // ising_ctx_destroy with live children only marks the context, the last child to go frees it.
    // Host languages with garbage collection destroy handles in no particular order.
    int children = 0;
    bool destroy_requested = false;
    int device = 0;
    cudaStream_t stream = nullptr;
    bool owns_stream = true;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::string err;
    int sm_count = 0;
    // grow-only device scratch (staging of outputs), so that repeated calls do not pay
    // cudaMalloc/cudaFree of hundreds of MB every time
    void* scratch[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    size_t scratch_bytes[6] = {0, 0, 0, 0, 0, 0};
    // second stream + events for the double-buffered device-to-host copies of the sampling path
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_filled[2] = {nullptr, nullptr}, ev_drained[2] = {nullptr, nullptr};
    // free list of device buffers released by destroyed sims: a stateless Lattice run creates
    // and destroys a sim per call, and cudaMalloc/cudaFree (device-wide synchronising, tens
    // of ms with large pinned regions mapped) must not be on that path
    std::vector<std::pair<void*, size_t>> free_bufs;
    size_t free_bytes = 0;
};

struct ising_graph {
    ising_ctx* ctx = nullptr;
    HostGraph h;
    // device copies
    uint32_t* d_jmask = nullptr;   // stencil +-J bond masks [2][2*dim][halfN]
    uint32_t* d_jmask8 = nullptr;  // the same, site-major [2][halfN][8]
    uint64_t* d_row = nullptr;     // CSR for replay / general kernels (uploaded on demand)
    uint32_t* d_nbr = nullptr;
    double* d_jv = nullptr;
    double* d_bias = nullptr;
    // general-graph sweep data (built on demand): colour x degree groups in ELL form
    bool gen_built = false;
    std::vector<GenGroup> gen_groups;
    std::vector<int> gen_group_color;
    int gen_ncolors = 0;
    uint32_t* d_gsites = nullptr;
    uint32_t* d_gnbr = nullptr;
    uint32_t* d_ganti = nullptr;
    uint32_t* d_row32 = nullptr;   // CSR for the energy kernel
    uint32_t* d_nbr32 = nullptr;
    uint8_t* d_anti8 = nullptr;
    // real couplings / biases: sites ordered by colour + float CSR values
    bool real_built = false;
    uint32_t* d_csites = nullptr;
    std::vector<uint32_t> color_off;   // ncolors + 1 offsets into d_csites
    float* d_jf = nullptr;
    float* d_biasf = nullptr;
    // non-basic moves: classes of the strong edge colouring (built on demand)
    bool moves_built = false;
    uint32_t* d_mea = nullptr;
    uint32_t* d_meb = nullptr;
    uint32_t* d_meid = nullptr;
    float* d_mwrel = nullptr;
    std::vector<uint32_t> medge_off;   // nclasses + 1 offsets into the four arrays
    EdgeClasses medge;                 // host copy (class of every bond: ising_graph_get_edge_classes)
    // bit-sliced edge moves (integer classes): (class, outer degree) groups in ELL form, built on
    // demand once per spin layout ([0] natural order, [1] checkerboard) because they hold slots
    struct EdgeGen {
        bool built = false, usable = false;
        std::vector<EdgeGroup> groups;   // in class order
        uint32_t* d_blob = nullptr;
    } edge_gen[2];
};

struct ising_comm;

struct ising_sim {
    ising_ctx* ctx = nullptr;
    const ising_graph* g = nullptr;
    uint64_t E = 0;
    uint64_t seed = 0;
    uint64_t replica_offset = 0;
    Layout lay{};
    uint32_t* d_spins = nullptr;
    unsigned long long* d_counts = nullptr;  // per-experiment integer accumulator [W*32]
    size_t spins_bytes = 0, counts_bytes = 0;
    uint64_t sweep_counter = 0;
    int planes = 6, rounds = kDefaultRounds;
    ising_sim_stats stats{};
    bool general = false;          // natural-order layout + colour/degree groups
    bool real = false;             // general layout, float local fields (real J / biases)
    // per-replica inverse temperatures (parallel tempering); general layout only
    bool perbeta = false;
    unsigned long long* d_t64 = nullptr;
    uint32_t* d_slot = nullptr;
    uint32_t t64_rows = 0;         // rows of d_t64 (per replica bit, or per ladder slot)
    uint32_t* d_tplane = nullptr;
    uint32_t* d_tlow = nullptr;
    // host cache of the general-graph threshold rows T64[deg][cls] by beta (bit pattern): in
    // parallel tempering the set of betas is fixed and only their assignment to replicas moves,
    // so a swap step must not recompute thousands of exp()
    std::unordered_map<uint64_t, std::vector<unsigned long long>> beta_rows;
    int beta_rows_planes = 0;
    // uniform longitudinal field (ising_graph_torus_field): stencil layout, field kernel; d_counts
    // then holds 2 * W * 32 counters (satisfied bonds, up spins)
    bool field = false;
    // what a timestep consists of (ising_sim_set_moves); default: one colour-class sweep
    bool moves_active = false;
    ising_moves mv{};
};

int fail(ising_ctx* ctx, int code, const char* fmt, ...);

void ctx_really_destroy(ising_ctx* ctx);   // api_core.cu
inline void ctx_retain(ising_ctx* ctx) {
    if (!ctx) return;
    std::lock_guard<std::recursive_mutex> g(ctx->mu);
    ++ctx->children;
}
inline void ctx_release(ising_ctx* ctx) {
    if (!ctx) return;
    bool last;
    {
        std::lock_guard<std::recursive_mutex> g(ctx->mu);
        last = --ctx->children == 0 && ctx->destroy_requested;
    }
    if (last) ctx_really_destroy(ctx);
}

struct CtxLock {
    ising_ctx* c;
    explicit CtxLock(const ising_ctx* ctx) : c(const_cast<ising_ctx*>(ctx)) { if (c) c->mu.lock(); }
    ~CtxLock() { if (c) c->mu.unlock(); }
    CtxLock(const CtxLock&) = delete;
    CtxLock& operator=(const CtxLock&) = delete;
};

#define CUDA_TRY(ctx, call)                                                          \
    do {                                                                             \
        cudaError_t _e = (call);                                                     \
        if (_e != cudaSuccess)                                                       \
            return fail((ctx), ISING_E_CUDA, "%s failed: %s", #call, cudaGetErrorString(_e)); \
    } while (0)

template <typename T>
static inline cudaError_t dev_alloc(T** p, size_t count) {
    return cudaMalloc((void**)p, std::max<size_t>(count, 1) * sizeof(T));
}

// context buffer caches (api_core.cu)
cudaError_t ctx_buf_get(ising_ctx* ctx, size_t bytes, void** out);
void ctx_buf_put(ising_ctx* ctx, void* p, size_t bytes);
cudaError_t ctx_scratch(ising_ctx* ctx, int slot, size_t bytes, void** out);
// rows of `width` bytes from device (pitch spitch) to host (pitch dpitch), enqueued on st
cudaError_t copy_rows_d2h(void* dst, size_t dpitch, const void* src, size_t spitch, size_t width,
                          size_t height, cudaStream_t st);
// on-demand device copies of a graph (api_core.cu)
int ensure_csr_on_device(ising_ctx* ctx, ising_graph* g);
int ensure_csr32_on_device(ising_ctx* ctx, ising_graph* g);
int ensure_real_on_device(ising_ctx* ctx, ising_graph* g);
int ensure_general_on_device(ising_ctx* ctx, ising_graph* g);
int ensure_moves_on_device(ising_ctx* ctx, ising_graph* g);
int ensure_edge_general_on_device(ising_ctx* ctx, ising_graph* g, bool stencil_layout);
// simulation object (api_sim.cu)
void count_launch(ising_sim* s, int n);
uint64_t threshold64(double beta, double de, int K);
void fill_field_thresholds(double jabs, double field, int dim, double beta, int K, FieldThresholds* th);
int sim_enqueue_sweeps(ising_sim* s, const double* betas, uint64_t nsweeps);
int sim_enqueue_sweeps_counting(ising_sim* s, uint64_t nsweeps, unsigned long long* d_counts, bool* counted);
// zero_first = false: the caller guarantees a zeroed buffer (the tempering cycle zeroes it in k_pt_cycle)
int sim_count_nsat(ising_sim* s, unsigned long long* d_counts, bool zero_first = true);
int sim_energies_to_device(ising_sim* s, double* d_out, uint64_t estride, uint64_t eoff);
