// TEST INFRASTRUCTURE (CPU suite only): just enough of the CUDA execution model to run the
// library's own kernel sources (pyisingmontecarlo_b200/csrc/*.cu, *.cuh) on the host, one OS thread
// per CUDA thread, so that the kernel source itself - row geometry, shared Philox rounds, bit-sliced
// compare, tie words, vertical counters and their block reduction, the tempering cycle - is compared
// bit for bit with oracle/msc_mirror.c without a GPU, and can be run under Thread / Address /
// UndefinedBehavior sanitizers.  Nothing of the product links or loads this.
//
// What stands in for what:
//   threadIdx / blockIdx / blockDim / gridDim   thread_local variables set by emu::launch()
//   __syncthreads()                             a pthread barrier over the block's threads
//   __shared__ (static)                         a function-local static: blocks run one at a time
//   extern __shared__ (dynamic)                 emu::dyn_smem, allocated per launch (per block when resident)
//   cg::this_grid().sync(), this_cluster().sync()  a barrier over all threads of a resident launch
//   atomicAdd, __ldg, __umulhi, __ffs, __popc   their plain C++ meaning (atomicAdd under a mutex)
//   __ballot_sync, __shfl_xor_sync (full mask)  a barrier over the warp's 32 threads around a scratch row
// The prepared copies of the sources (tests/test_device_source_on_host.py: prepare_sources) have the
// griddepcontrol PTX, the TMA-staged variants and the <<< >>> launch wrappers cut out; every cut is
// an asserted exact-text edit there.
#pragma once
#include <cuda_runtime.h>   // vector types (uint2, uint4, dim3) and the host API's typedefs only
#include <math.h>
#include <pthread.h>
#include <string.h>
#include <stdint.h>

#include <mutex>
#include <thread>
#include <tuple>
#include <vector>

#define __launch_bounds__(...)
#define __grid_constant__
// (host_defines.h leaves this one to nvcc; defined after the standard headers, which spell the
// attribute with the same token)
#define __noinline__ __attribute__((noinline))
#define EMU_SHARED static

namespace emu {
inline thread_local uint3 t_threadIdx, t_blockIdx;
inline thread_local dim3 t_blockDim, t_gridDim;
inline thread_local pthread_barrier_t* t_barrier = nullptr;
inline thread_local uint32_t* dyn_smem = nullptr;   // the block's dynamic shared memory
inline thread_local pthread_barrier_t* t_grid_barrier = nullptr;   // cooperative / cluster launches only
inline thread_local pthread_barrier_t* t_warp_barrier = nullptr;   // the 32 consecutive threads of a warp
inline thread_local uint64_t* t_warp_scratch = nullptr;            // 32 slots per warp (votes, shuffles)
inline std::mutex atomic_mu;
}  // namespace emu

// what the kernels use of <cooperative_groups.h>: the grid barrier of a cooperative launch and the
// barrier of a thread-block cluster, both a barrier over every thread of an emu::launch_resident
namespace cooperative_groups {
struct grid_group { void sync() const { pthread_barrier_wait(emu::t_grid_barrier); } };
struct cluster_group { void sync() const { pthread_barrier_wait(emu::t_grid_barrier); } };
inline grid_group this_grid() { return {}; }
inline cluster_group this_cluster() { return {}; }
}  // namespace cooperative_groups

#define threadIdx emu::t_threadIdx
#define blockIdx emu::t_blockIdx
#define blockDim emu::t_blockDim
#define gridDim emu::t_gridDim

static inline void __syncthreads() { pthread_barrier_wait(emu::t_barrier); }
static inline uint32_t __umulhi(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * b) >> 32); }
static inline int __ffs(int v) { return __builtin_ffs(v); }
static inline int __popc(uint32_t v) { return __builtin_popcount(v); }
// (lo, hi) as one 64-bit value shifted by n & 31: the low word (_r) / the high word (_l) of the result
static inline uint32_t __funnelshift_r(uint32_t lo, uint32_t hi, uint32_t n) {
    return (uint32_t)((((uint64_t)hi << 32) | lo) >> (n & 31));
}
static inline uint32_t __funnelshift_l(uint32_t lo, uint32_t hi, uint32_t n) {
    return (uint32_t)(((((uint64_t)hi << 32) | lo) << (n & 31)) >> 32);
}
template <typename T>
static inline T __ldg(const T* p) { return *p; }
// round-to-nearest add / multiply that the compiler must not contract into a fused multiply-add:
// plain operations here (the emulation is built with -ffp-contract=off)
static inline double __dadd_rn(double a, double b) { return a + b; }
static inline double __dmul_rn(double a, double b) { return a * b; }
static inline double __dsub_rn(double a, double b) { return a - b; }
// float kernels (real couplings, float moves): bit casts, the fast exponential as libm's expf (inside
// the error bound of __expf that tests/float_reference.py allows for), the saturating float -> uint32
// conversion
static inline uint32_t __float_as_uint(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }
static inline float __uint_as_float(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }
static inline double __longlong_as_double(long long v) { double d; memcpy(&d, &v, 8); return d; }
#define __expf(x) expf(x)   /* (glibc declares a function of this name itself) */
static inline uint32_t __float2uint_rz(float f) {
    if (!(f > 0.f)) return 0u;                       // NaN and negatives
    if (f >= 4294967296.f) return 0xFFFFFFFFu;
    return (uint32_t)f;
}
static inline uint64_t __umul64hi(uint64_t a, uint64_t b) { return (uint64_t)(((unsigned __int128)a * b) >> 64); }
template <typename T>
static inline T __ldcg(const T* p) { return *(const volatile T*)p; }
static inline unsigned int atomicAdd(unsigned int* p, unsigned int v) {
    std::lock_guard<std::mutex> g(emu::atomic_mu);
    const unsigned int old = *p;
    *p = old + v;
    return old;
}
static inline unsigned int atomicXor(unsigned int* p, unsigned int v) {
    std::lock_guard<std::mutex> g(emu::atomic_mu);
    const unsigned int old = *p;
    *p = old ^ v;
    return old;
}
static inline double atomicAdd(double* p, double v) {
    std::lock_guard<std::mutex> g(emu::atomic_mu);
    const double old = *p;
    *p = old + v;
    return old;
}
static inline unsigned long long atomicAdd(unsigned long long* p, unsigned long long v) {
    std::lock_guard<std::mutex> g(emu::atomic_mu);
    const unsigned long long old = *p;
    *p = old + v;
    return old;
}

// warp vote over the full warp: lanes post their predicate, meet, read all 32
static inline uint32_t __ballot_sync(uint32_t, int pred) {
    const unsigned lane = (threadIdx.x + blockDim.x * (threadIdx.y + blockDim.y * threadIdx.z)) & 31u;
    emu::t_warp_scratch[lane] = pred ? 1u : 0u;
    pthread_barrier_wait(emu::t_warp_barrier);
    uint32_t r = 0;
    for (unsigned l = 0; l < 32; ++l) r |= (uint32_t)emu::t_warp_scratch[l] << l;
    pthread_barrier_wait(emu::t_warp_barrier);
    return r;
}
// butterfly exchange over the full warp (values of up to 64 bits)
template <typename T>
static inline T __shfl_xor_sync(uint32_t, T v, int lane_mask) {
    static_assert(sizeof(T) <= 8, "shuffle of at most 64 bits");
    const unsigned lane = (threadIdx.x + blockDim.x * (threadIdx.y + blockDim.y * threadIdx.z)) & 31u;
    uint64_t raw = 0;
    memcpy(&raw, &v, sizeof(T));
    emu::t_warp_scratch[lane] = raw;
    pthread_barrier_wait(emu::t_warp_barrier);
    raw = emu::t_warp_scratch[lane ^ (unsigned)lane_mask];
    pthread_barrier_wait(emu::t_warp_barrier);
    T out;
    memcpy(&out, &raw, sizeof(T));
    return out;
}

namespace emu {
// <<<grid, block, smem_bytes>>> of a kernel taking one by-value argument: blocks one after the
// other, the threads of a block concurrently
template <typename Args>
void launch(void (*kern)(const Args), dim3 grid, dim3 block, size_t smem_bytes, const Args& args) {
    const unsigned nthreads = block.x * block.y * block.z;
    std::vector<uint32_t> smem(smem_bytes / 4 + 1);
    uint32_t* const smem_p = smem.data();
    const unsigned nwarps = nthreads % 32 == 0 ? nthreads / 32 : 0;   // warp votes need whole warps
    std::vector<pthread_barrier_t> wbar(nwarps);
    std::vector<uint64_t> wscratch((size_t)nwarps * 32 + 1);
    for (auto& w : wbar) pthread_barrier_init(&w, nullptr, 32);
    pthread_barrier_t* const wbar_p = wbar.data();
    uint64_t* const wscratch_p = wscratch.data();
    for (unsigned b = 0; b < grid.x * grid.y; ++b) {
        pthread_barrier_t bar;
        pthread_barrier_init(&bar, nullptr, nthreads);
        std::vector<std::thread> th;
        th.reserve(nthreads);
        for (unsigned t = 0; t < nthreads; ++t)
            th.emplace_back([=, &bar, &args] {
                t_threadIdx = uint3{t % block.x, (t / block.x) % block.y, t / (block.x * block.y)};
                t_blockIdx = uint3{b % grid.x, b / grid.x, 0};
                t_blockDim = block;
                t_gridDim = grid;
                t_barrier = &bar;
                dyn_smem = smem_p;
                t_warp_barrier = nwarps ? wbar_p + t / 32 : nullptr;
                t_warp_scratch = wscratch_p + (size_t)(t / 32) * 32;
                kern(args);
            });
        for (auto& x : th) x.join();
        pthread_barrier_destroy(&bar);
    }
    for (auto& w : wbar) pthread_barrier_destroy(&w);
}

// Cooperative / cluster launch: all blocks resident at once (every thread of the grid is an OS
// thread), so that a grid-wide or cluster-wide barrier can be waited on.  Function-local statics
// standing in for __shared__ are then shared by the blocks: fine for the kernels run this way,
// whose static shared data is the same in every block (the thresholds of the current sweep).
template <typename Args>
void launch_resident(void (*kern)(const Args), dim3 grid, dim3 block, size_t smem_bytes, const Args& args) {
    const unsigned nthreads = block.x * block.y * block.z, nblocks = grid.x * grid.y;
    std::vector<std::vector<uint32_t>> smem(nblocks, std::vector<uint32_t>(smem_bytes / 4 + 1));
    std::vector<pthread_barrier_t> bars(nblocks);
    pthread_barrier_t all;
    pthread_barrier_init(&all, nullptr, nthreads * nblocks);
    for (auto& b : bars) pthread_barrier_init(&b, nullptr, nthreads);
    std::vector<std::thread> th;
    th.reserve((size_t)nthreads * nblocks);
    for (unsigned b = 0; b < nblocks; ++b)
        for (unsigned t = 0; t < nthreads; ++t)
            th.emplace_back([=, &bars, &all, &smem, &args] {
                t_threadIdx = uint3{t % block.x, (t / block.x) % block.y, t / (block.x * block.y)};
                t_blockIdx = uint3{b % grid.x, b / grid.x, 0};
                t_blockDim = block;
                t_gridDim = grid;
                t_barrier = &bars[b];
                t_grid_barrier = &all;
                dyn_smem = smem[b].data();
                kern(args);
            });
    for (auto& x : th) x.join();
    for (auto& b : bars) pthread_barrier_destroy(&b);
    pthread_barrier_destroy(&all);
}
}  // namespace emu

namespace emu {
// the same for kernels that take several parameters
template <bool RESIDENT = false, typename... KArgs, typename... Args>
void launch_v(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem_bytes, Args... args) {
    struct Pack { void (*k)(KArgs...); std::tuple<KArgs...> a; };
    Pack p{kern, std::tuple<KArgs...>(KArgs(args)...)};
    const Pack* pp = &p;
    void (*tramp)(const Pack*) = [](const Pack* q) { std::apply(q->k, q->a); };
    if (RESIDENT) launch_resident<const Pack*>(tramp, grid, block, smem_bytes, pp);
    else launch<const Pack*>(tramp, grid, block, smem_bytes, pp);
}
}  // namespace emu
