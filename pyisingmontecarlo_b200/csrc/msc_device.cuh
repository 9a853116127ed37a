// Device-side building blocks shared by the kernel translation units: bit-sliced neighbour
// counting, vertical counters and their block reduction, the Metropolis flip mask, vector
// loads.  See DESIGN.md sections 4-5.
#pragma once
#include "kernels.h"

#include <cooperative_groups.h>

#include <stdlib.h>

#include "../../include/ising_b200.h"
#include "philox.h"

namespace cg = cooperative_groups;

namespace ising {


// ------------------------------------------------------------------------------------------
// layout helpers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ size_t site_word_base(const Layout& L, uint64_t n) {
    if (L.kind == ISING_KIND_GENERAL) return (size_t)n * L.W;
    const uint32_t x = (uint32_t)(n % L.Lx);
    const uint32_t r = (uint32_t)(n / L.Lx);  // row = z * Ly + y
    const uint32_t y = r % L.Ly, z = r / L.Ly;
    const uint32_t c = (x + y + z) & 1u;
    return (((size_t)c * L.rows + r) * L.Lxh + (x >> 1)) * L.W;
}

// ------------------------------------------------------------------------------------------
// bit-sliced satisfied-bond count of one word: planes (b0, b1, b2) of n_sat in 0..2*DIM
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t maj3(uint32_t a, uint32_t b, uint32_t c) {
    return (a & b) | (c & (a ^ b));
}

template <int DIM>
__device__ __forceinline__ void count_sat(const uint32_t (&a)[2 * DIM], uint32_t& b0,
                                          uint32_t& b1, uint32_t& b2) {
    if (DIM == 3) {
        const uint32_t s0 = a[0] ^ a[1] ^ a[2], c0 = maj3(a[0], a[1], a[2]);
        const uint32_t s1 = a[3] ^ a[4] ^ a[5], c1 = maj3(a[3], a[4], a[5]);
        const uint32_t k = s0 & s1;
        b0 = s0 ^ s1;
        b1 = c0 ^ c1 ^ k;
        b2 = maj3(c0, c1, k);
    } else {
        const uint32_t s0 = a[0] ^ a[1] ^ a[2], c0 = maj3(a[0], a[1], a[2]);
        const uint32_t k = s0 & a[3];
        b0 = s0 ^ a[3];
        b1 = c0 ^ k;
        b2 = c0 & k;
    }
}

// ------------------------------------------------------------------------------------------
// vertical (bit-sliced) counters: plane l holds bit l of 32 independent per-replica counters
// ------------------------------------------------------------------------------------------
template <int NP>
struct VCount {
    uint32_t v[NP];
    __device__ __forceinline__ void clear() {
#pragma unroll
        for (int l = 0; l < NP; ++l) v[l] = 0;
    }
    // counters += b0 + 2 b1 + 4 b2
    __device__ __forceinline__ void add3(uint32_t b0, uint32_t b1, uint32_t b2) {
        uint32_t c = v[0] & b0;
        v[0] ^= b0;
        uint32_t t = v[1] ^ b1, c2 = (v[1] & b1) | (c & t);
        v[1] = t ^ c;
        c = c2;
        t = v[2] ^ b2;
        c2 = (v[2] & b2) | (c & t);
        v[2] = t ^ c;
        c = c2;
#pragma unroll
        for (int l = 3; l < NP; ++l) {
            t = v[l] & c;
            v[l] ^= c;
            c = t;
        }
    }
    __device__ __forceinline__ void add1(uint32_t b0) {
        uint32_t c = b0;
#pragma unroll
        for (int l = 0; l < NP; ++l) {
            const uint32_t t = v[l] & c;
            v[l] ^= c;
            c = t;
        }
    }
    // sm is int[32][nthreads]; adds this thread's 32 counters to its column
    __device__ __forceinline__ void flush(int* sm, int tid, int nthreads) {
#pragma unroll 4
        for (int b = 0; b < 32; ++b) {
            int cnt = 0;
#pragma unroll
            for (int l = 0; l < NP; ++l) cnt |= (int)((v[l] >> b) & 1u) << l;
            sm[b * nthreads + tid] += cnt;
        }
        clear();
    }
};

// --- bit-sliced helpers for the cross-thread reduction of vertical counters --------------------
// acc (NR planes) += x (NX planes), both little-endian bit-sliced integers
template <int NR, int NX>
__device__ __forceinline__ void vadd(uint32_t (&acc)[NR], const uint32_t (&x)[NX]) {
    uint32_t c = 0;
#pragma unroll
    for (int l = 0; l < NR; ++l) {
        const uint32_t xi = l < NX ? x[l] : 0u;
        const uint32_t t = acc[l] ^ xi;
        const uint32_t c2 = (acc[l] & xi) | (c & t);
        acc[l] = t ^ c;
        c = c2;
    }
}

#ifndef ISING_SW_NP
#define ISING_SW_NP 7
#endif
constexpr int SW_NP = ISING_SW_NP;                       // fused n_sat counter planes per thread
constexpr int SW_MAX_ITEMS = ((1 << SW_NP) - 1) / 6;    // sites a thread may accumulate (n_sat <= 6)

constexpr int NS_NR = 20;  // block-level counter planes: 256 threads x 1023 fits 18 bits

// Block-wide reduction of per-thread vertical counters (NP planes, V replica words per thread,
// block = (wx, by)) into per-experiment integers: bit-sliced tree through shared memory, then
// one SWAR bit-transpose per word column and 32 integer atomics per column.
//   sm: max(NP * V, NR) * nthreads words;  out[(w0 + column) * 32 + bit] += count
//   NR = planes of the block-level counters: nthreads * (2^NP - 1) must stay below 2^NR
template <int NP, int V, int NR = NS_NR>
__device__ __forceinline__ void block_reduce_vcount(const VCount<NP> (&vc)[V], uint32_t* sm,
                                                    unsigned long long* __restrict__ out,
                                                    uint32_t w0, uint32_t W) {
    const uint32_t wx = blockDim.x, by = blockDim.y, nthreads = wx * by;
    const uint32_t tid = threadIdx.y * wx + threadIdx.x;
    const uint32_t C = wx * V;  // word columns of this chunk (C divides nthreads)
    __syncthreads();
#pragma unroll
    for (int v = 0; v < V; ++v)
#pragma unroll
        for (int l = 0; l < NP; ++l) sm[(l * V + v) * nthreads + tid] = vc[v].v[l];
    __syncthreads();
    // stage A: thread (column c, part q) adds the counters of every Q-th row-thread
    const uint32_t Q = nthreads / C;
    const uint32_t c = tid % C, q = tid / C;
    const uint32_t cx = c / V, cv = c % V;
    uint32_t acc[NR];
#pragma unroll
    for (int l = 0; l < NR; ++l) acc[l] = 0;
    for (uint32_t ty = q; ty < by; ty += Q) {
        uint32_t x[NP];
#pragma unroll
        for (int l = 0; l < NP; ++l) x[l] = sm[(l * V + cv) * nthreads + ty * wx + cx];
        vadd<NR, NP>(acc, x);
    }
    __syncthreads();
#pragma unroll
    for (int l = 0; l < NR; ++l) sm[l * nthreads + tid] = acc[l];  // [plane][q][c]
    __syncthreads();
    // stage B1: tree over the Q parts of every column (all threads of the surviving parts work)
    for (uint32_t half = Q >> 1; half >= 1; half >>= 1) {
        if (q < half) {
            uint32_t x[NR];
#pragma unroll
            for (int l = 0; l < NR; ++l) x[l] = sm[l * nthreads + (q + half) * C + c];
            vadd<NR, NR>(acc, x);
#pragma unroll
            for (int l = 0; l < NR; ++l) sm[l * nthreads + tid] = acc[l];
        }
        __syncthreads();
    }
    // stage B2: SWAR bit-transpose of the column totals (part 0), byte-lane group g per thread:
    // bits g, g+8, g+16, g+24 of the planes land in four byte lanes; 4 integer atomics each
    if (w0 + c < W) {
        if (q != 0) {
#pragma unroll
            for (int l = 0; l < NR; ++l) acc[l] = sm[l * nthreads + c];
        }
        unsigned long long* o = out + (size_t)(w0 + c) * 32;
        for (uint32_t g = q; g < 8; g += Q) {
            uint32_t lo = 0, hi = 0, top = 0;
#pragma unroll
            for (int l = 0; l < 8; ++l) {
                lo += ((acc[l] >> g) & 0x01010101u) << l;
                if (l + 8 < NR) hi += ((acc[l + 8] >> g) & 0x01010101u) << l;
                if (l + 16 < NR) top += ((acc[l + 16] >> g) & 0x01010101u) << l;
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const uint32_t cnt = ((lo >> (8 * k)) & 0xFFu) | (((hi >> (8 * k)) & 0xFFu) << 8) |
                                     (((top >> (8 * k)) & 0xFFu) << 16);
                if (cnt) atomicAdd(o + g + 8 * k, (unsigned long long)cnt);
            }
        }
    }
    __syncthreads();
}

// ------------------------------------------------------------------------------------------
// Metropolis acceptance of the uphill bits of one word.
//   up   : bits with dE > 0;  (sel1, sel0) select the class of each such bit
//   K bit-planes R_0..R_{K-1} are the K most significant bits of a uniform U per replica and
//   are compared against the class threshold T: U_top < T_top is the borrow of the bit-sliced
//   subtraction U_top - T_top (one majority LOP3 per plane, LSB first); bits whose top K bits
//   tie (probability 2^-K) are resolved by a fresh 32-bit word against the low 32 threshold
//   bits, tied bits taken in ascending position.  Word R_m is output m%4 of Philox call m/4
//   on counter (site, replica word, sweep, call) for the NCALL = K/4 + 1 calls every update
//   makes; later words (the third tie of a word and beyond, 1 word in 100) are the outputs of
//   continuation rounds of the last of those blocks: R_m = output m%4 of
//   Philox4x32-(ROUNDS + m/4 - NCALL + 1) on the counter of call NCALL - 1.
// returns the flip mask (downhill bits always flip)
// ------------------------------------------------------------------------------------------
// PERBETA: every replica bit has its own inverse temperature (parallel tempering): the plane
// masks are words tp[cls * 8 + p] whose bit b is the threshold bit of replica b of this word,
// the resolver thresholds tl[b * 3 + cls].
template <int NCLS, int K, int ROUNDS, bool PERBETA = false>
__device__ __forceinline__ uint32_t msc_flip_mask(uint32_t up, uint32_t sel0, uint32_t sel1,
                                                  const MscThresholds& th, uint32_t site,
                                                  uint32_t gw, uint32_t sweep, const PhiloxKeys& pk,
                                                  const uint32_t* __restrict__ tp = nullptr,
                                                  const uint32_t* __restrict__ tl = nullptr) {
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
    uint32_t eq = up, borrow = 0;
#pragma unroll
    for (int p = K - 1; p >= 0; --p) {
        const uint32_t P0 = PERBETA ? __ldg(tp + 0 * 8 + p) : th.plane[0][p];
        const uint32_t P1 = PERBETA ? __ldg(tp + 1 * 8 + p) : th.plane[1][p];
        uint32_t t = (sel0 & P1) | (~sel0 & P0);
        if (NCLS == 3) {
            const uint32_t P2 = PERBETA ? __ldg(tp + 2 * 8 + p) : th.plane[2][p];
            t = (sel1 & P2) | (~sel1 & t);
        }
        borrow = maj3(~r[p], t, borrow);
        eq &= ~(r[p] ^ t);
    }
    uint32_t flip = ~up | (borrow & ~eq);
    // Tied bits (2^-K each).  The first SPARE of them use the words left over from the calls
    // above in straight-line predicated code (no divergent loop for the common case); anything
    // beyond that, rare, takes further rounds of the last block in a loop.
    constexpr int SPARE = (4 * NCALL - K) < 2 ? (4 * NCALL - K) : 2;
#pragma unroll
    for (int j = 0; j < SPARE; ++j) {
        const uint32_t bit = eq & (0u - eq);  // lowest tied bit, 0 when nothing is tied
        uint32_t lo;
        if (PERBETA) {
            const int b = (__ffs((int)eq) - 1) & 31;
            const uint32_t cls = (NCLS == 3 && (sel1 & bit)) ? 2u : ((sel0 & bit) ? 1u : 0u);
            lo = __ldg(tl + b * 3 + cls);
        } else {
            lo = (sel0 & bit) ? th.low[1] : th.low[0];
            if (NCLS == 3 && (sel1 & bit)) lo = th.low[2];
        }
        if (r[K + j] < lo) flip |= bit;
        eq ^= bit;
    }
    if (eq) {
        int j = K + SPARE;
        u32x4 cur = {r[4 * (NCALL - 1)], r[4 * (NCALL - 1) + 1], r[4 * (NCALL - 1) + 2],
                     r[4 * (NCALL - 1) + 3]};
        do {
            const int b = __ffs((int)eq) - 1;
            if ((j & 3) == 0 && j >= 4 * NCALL)
                cur = philox4x32_more(cur, (uint32_t)(ROUNDS + (j >> 2) - NCALL), pk.k[0], pk.k[1]);
            const int m = j & 3;
            const uint32_t v = m == 0 ? cur.x : (m == 1 ? cur.y : (m == 2 ? cur.z : cur.w));
            uint32_t lo;
            if (PERBETA) {
                const uint32_t cls = (NCLS == 3 && ((sel1 >> b) & 1u)) ? 2u : (((sel0 >> b) & 1u) ? 1u : 0u);
                lo = __ldg(tl + b * 3 + cls);
            } else {
                lo = ((sel0 >> b) & 1u) ? th.low[1] : th.low[0];
                if (NCLS == 3 && ((sel1 >> b) & 1u)) lo = th.low[2];
            }
            if (v < lo) flip |= 1u << b;
            eq &= eq - 1;
            ++j;
        } while (eq);
    }
    return flip;
}

// V consecutive replica words as one vector load / store (128-bit when V == 4)
template <int V> struct WordVec;
template <> struct WordVec<1> { typedef uint32_t type; };
template <> struct WordVec<2> { typedef uint2 type; };
template <> struct WordVec<4> { typedef uint4 type; };

template <int V>
__device__ __forceinline__ void load_words(const uint32_t* p, uint32_t (&out)[V]) {
    typedef typename WordVec<V>::type T;
    const T v = *reinterpret_cast<const T*>(p);
    const uint32_t* w = reinterpret_cast<const uint32_t*>(&v);
#pragma unroll
    for (int k = 0; k < V; ++k) out[k] = w[k];
}

template <int V>
__device__ __forceinline__ void store_words(uint32_t* p, const uint32_t (&in)[V]) {
    typedef typename WordVec<V>::type T;
    T v;
    uint32_t* w = reinterpret_cast<uint32_t*>(&v);
#pragma unroll
    for (int k = 0; k < V; ++k) w[k] = in[k];
    *reinterpret_cast<T*>(p) = v;
}

// ------------------------------------------------------------------------------------------
// uniform longitudinal field (sweep_field.cu, strip_field.cu): the class of a bit is (spin, n_sat)
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t bit_select(uint32_t x, uint32_t one, uint32_t zero) {
    return (x & one) | (~x & zero);
}

// v[n_sat] per replica bit, n_sat given by its planes (b0, b1, b2); patterns above 2 DIM do not occur
template <int DIM>
__device__ __forceinline__ uint32_t nsat_select(uint32_t b0, uint32_t b1, uint32_t b2, const uint32_t (&v)[8]) {
    const uint32_t lo = bit_select(b1, bit_select(b0, v[3], v[2]), bit_select(b0, v[1], v[0]));
    if (DIM == 3) return bit_select(b2, bit_select(b1, v[6], bit_select(b0, v[5], v[4])), lo);
    return bit_select(b2, v[4], lo);
}

// v[s][n_sat] per replica bit, s = the spin word
template <int DIM>
__device__ __forceinline__ uint32_t class_select(uint32_t s, uint32_t b0, uint32_t b1, uint32_t b2,
                                                 const uint32_t (&v)[2][8]) {
    return bit_select(s, nsat_select<DIM>(b0, b1, b2, v[1]), nsat_select<DIM>(b0, b1, b2, v[0]));
}

// Flip mask of one word from the words r of its K/4 + 1 Philox calls: msc_flip_mask's planes, resolver
// words, continuation rounds and tie order, with the uphill bits and the threshold bits selected by
// (spin, n_sat).  Bits with dE <= 0 flip without a resolver word.
template <int DIM, int K, int ROUNDS>
__device__ __forceinline__ uint32_t field_flip_mask_words(uint32_t s, uint32_t b0, uint32_t b1, uint32_t b2,
                                                          const FieldThresholds& th, const uint32_t (&r)[4 * (K / 4 + 1)],
                                                          const PhiloxKeys& pk) {
    constexpr int NCALL = K / 4 + 1;
    const uint32_t up = class_select<DIM>(s, b0, b1, b2, th.up);
    uint32_t eq = up, borrow = 0;
#pragma unroll
    for (int p = K - 1; p >= 0; --p) {
        const uint32_t t = class_select<DIM>(s, b0, b1, b2, th.plane[p]);
        borrow = maj3(~r[p], t, borrow);
        eq &= ~(r[p] ^ t);
    }
    uint32_t flip = ~up | (borrow & ~eq);
    // tied bits (2^-K each), ascending bit position: the words left over from the calls above,
    // then further rounds of the last block
    int j = K;
    u32x4 cur = {r[4 * (NCALL - 1)], r[4 * (NCALL - 1) + 1], r[4 * (NCALL - 1) + 2], r[4 * (NCALL - 1) + 3]};
    while (eq) {
        const int b = __ffs((int)eq) - 1;
        if ((j & 3) == 0 && j >= 4 * NCALL)
            cur = philox4x32_more(cur, (uint32_t)(ROUNDS + (j >> 2) - NCALL), pk.k[0], pk.k[1]);
        const int m = j & 3;
        const uint32_t v = m == 0 ? cur.x : (m == 1 ? cur.y : (m == 2 ? cur.z : cur.w));
        const uint32_t n = ((b0 >> b) & 1u) | (((b1 >> b) & 1u) << 1) | (((b2 >> b) & 1u) << 2);
        if (v < th.low[(s >> b) & 1u][n]) flip |= 1u << b;
        eq &= eq - 1;
        ++j;
    }
    return flip;
}

// ------------------------------------------------------------------------------------------
// one large 2D lattice bit-packed along x in row strips (strip.cu, strip_field.cu; kernels.h: StripGeom)
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ size_t strip_off(const StripGeom& g, uint32_t c, uint32_t r, uint32_t j) {
    return ((size_t)c * (g.rows + 2 * g.ghost) + r) * g.Wr + j;
}

// Words j .. j + V - 1 of colour c in storage row r (s) and their four neighbour words: the other
// colour o = 1 - c at the same index (n[0]), those funnel-shifted by one bit with the carry from the
// adjacent word (n[1], the other x neighbour; p = (y + c) & 1 gives the side), the rows above and
// below (n[2], n[3]).  Returns the address of s.
template <int V>
__device__ __forceinline__ uint32_t* strip_load_site(uint32_t* spins, const StripGeom& g, uint32_t c, uint32_t o,
                                                     uint32_t r, uint32_t j, uint32_t p, uint32_t (&s)[V],
                                                     uint32_t (&n)[4][V]) {
    uint32_t* own = spins + strip_off(g, c, r, j);
    const uint32_t* orow = spins + strip_off(g, o, r, 0);
    load_words<V>(own, s);
    load_words<V>(orow + j, n[0]);
    load_words<V>(orow + j - g.Wr, n[2]);
    load_words<V>(orow + j + g.Wr, n[3]);
    const uint32_t edge = p ? orow[j + V == g.Wr ? 0 : j + V] : orow[j == 0 ? g.Wr - 1 : j - 1];
#pragma unroll
    for (int v = 0; v < V; ++v) {
        if (p) n[1][v] = __funnelshift_r(n[0][v], v + 1 < V ? n[0][v + 1 < V ? v + 1 : v] : edge, 1);
        else n[1][v] = __funnelshift_l(v > 0 ? n[0][v > 0 ? v - 1 : 0] : edge, n[0][v], 1);
    }
    return own;
}

// ------------------------------------------------------------------------------------------
// K3: positional popcount (per-experiment integer observables from packed words)
// vertical counters: plane l of VCount holds bit l of 32 independent counters
// ------------------------------------------------------------------------------------------
constexpr int VC_PLANES = 12;           // counters up to 4095
constexpr int VC_FLUSH_ADD1 = 4095;

// reduce sm[32][nthreads] over threadIdx.y and add to out[(w0 + tx) * 32 + b]
__device__ __forceinline__ void block_reduce_counts(int* sm, unsigned long long* out, uint32_t w0,
                                                    uint32_t W) {
    const int wx = blockDim.x, by = blockDim.y, nthreads = wx * by;
    const int tid = threadIdx.y * wx + threadIdx.x;
    __syncthreads();
    for (int idx = tid; idx < 32 * wx; idx += nthreads) {
        const int b = idx / wx, tx = idx - b * wx;
        if (w0 + tx >= W) continue;
        long long sum = 0;
        for (int ty = 0; ty < by; ++ty) sum += sm[b * nthreads + ty * wx + tx];
        if (sum) atomicAdd(out + (size_t)(w0 + tx) * 32 + b, (unsigned long long)sum);
    }
    __syncthreads();
}

// Launch with programmatic stream serialisation: consecutive colour phases overlap launch latency
// and preamble with the tail of the previous phase (the kernels order themselves with
// griddepcontrol.wait).  Measured on BASELINE config 3: 61.8 -> 59.3 us per sweep at 1024
// replicas, 16.4 -> 11.5 us at 128 replicas per GPU (the 8-GPU split).  ISING_NO_PDL=1 launches
// the ordinary way (A/B knob).
template <typename Kern, typename Args>
static inline cudaError_t launch_pdl(Kern kern, dim3 grid, dim3 block, size_t smem, cudaStream_t st, const Args& args) {
    static const bool no_pdl = getenv("ISING_NO_PDL") != nullptr;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = no_pdl ? 0 : 1;
    return cudaLaunchKernelEx(&cfg, kern, args);
}

// the same for kernels that take several parameters
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl_v(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                       Args... args) {
    static const bool no_pdl = getenv("ISING_NO_PDL") != nullptr;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = no_pdl ? 0 : 1;
    return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

static inline uint32_t pow2_ceil(uint32_t v) {
    uint32_t p = 1;
    while (p < v) p <<= 1;
    return p;
}

}  // namespace ising
