// C ABI: one large 2D lattice in row strips (ising_strip_*).
#include "api_internal.h"

// ------------------------------------------------------------------------------------------
// one large 2D lattice in row strips (config 5)
// ------------------------------------------------------------------------------------------
struct ising_strip {
    ising_ctx* ctx = nullptr;
    StripGeom g{};
    uint64_t Lx = 0;
    uint32_t* d_spins = nullptr;
    uint32_t* d_alt = nullptr;     // second array of the fused (out-of-place) sweep, allocated on first use
    size_t bytes = 0;
    unsigned long long* d_acc = nullptr;
    double j = -1.0;
    double field = 0.0;            // uniform longitudinal field h of the next sweeps (ising_strip_set_field)
    uint64_t seed = 0, sweep = 0, launches = 0;
    int planes = 6, rounds = kDefaultRounds;
    double device_ms = 0.0;
};

extern "C" int ising_strip_create_ex(ising_ctx* ctx, uint64_t Lx, uint64_t Ly, uint64_t row_lo,
                                     uint64_t row_hi, double j, uint64_t seed, uint32_t ghost,
                                     ising_strip** out) {
    CtxLock _lk(ctx);
    if (!ctx || !out) return fail(ctx, ISING_E_INVALID, "ctx/out is NULL");
    *out = nullptr;
    if (ghost < 1 || ghost > row_hi - row_lo || ghost > 1024)
        return fail(ctx, ISING_E_INVALID, "ghost depth must be 1..min(rows, 1024)");
    if (Lx < 64 || Lx % 64) return fail(ctx, ISING_E_INVALID, "Lx must be a positive multiple of 64");
    if (Ly < 2 || (Ly & 1)) return fail(ctx, ISING_E_INVALID, "Ly must be even");
    if (row_lo >= row_hi || row_hi > Ly) return fail(ctx, ISING_E_INVALID, "need 0 <= row_lo < row_hi <= Ly");
    if (Ly > 0xFFFFFFFFull || Lx / 64 > 0x3FFFFFFFull) return fail(ctx, ISING_E_INVALID, "lattice too large");
    if (!(fabs(j) > 0.0) || !std::isfinite(j)) return fail(ctx, ISING_E_INVALID, "j must be finite and non-zero");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    std::unique_ptr<ising_strip> s(new ising_strip);
    s->ctx = ctx;
    s->Lx = Lx;
    s->g.Wr = (uint32_t)(Lx / 64);
    s->g.rows = (uint32_t)(row_hi - row_lo);
    s->g.row0 = (uint32_t)row_lo;
    s->g.Ly = (uint32_t)Ly;
    s->g.ghost = ghost;
    s->j = j;
    s->seed = seed;
    s->bytes = (size_t)2 * (s->g.rows + 2 * ghost) * s->g.Wr * sizeof(uint32_t);
    void* p = nullptr;
    CUDA_TRY(ctx, ctx_buf_get(ctx, s->bytes, &p));
    s->d_spins = (uint32_t*)p;
    cudaError_t e = ctx_buf_get(ctx, 2 * sizeof(unsigned long long), &p);
    if (e != cudaSuccess) { ctx_buf_put(ctx, s->d_spins, s->bytes); CUDA_TRY(ctx, e); }
    s->d_acc = (unsigned long long*)p;
    CUDA_TRY(ctx, cudaMemsetAsync(s->d_spins, 0, s->bytes, ctx->stream));
    if (launch_strip_init_random(s->d_spins, s->g, (uint32_t)seed, (uint32_t)(seed >> 32), ctx->stream) < 0)
        return fail(ctx, ISING_E_CUDA, "strip init launch failed");
    s->launches++;
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    *out = s.release();
    ctx_retain(ctx);
    return ISING_OK;
}

extern "C" int ising_strip_create(ising_ctx* ctx, uint64_t Lx, uint64_t Ly, uint64_t row_lo,
                                  uint64_t row_hi, double j, uint64_t seed, ising_strip** out) {
    CtxLock _lk(ctx);
    return ising_strip_create_ex(ctx, Lx, Ly, row_lo, row_hi, j, seed, 1, out);
}

extern "C" void ising_strip_destroy(ising_strip* s) {
    if (!s) return;
    struct Release { ising_ctx* c; ~Release() { ctx_release(c); } } _rel{s->ctx};   // after the lock is gone
    CtxLock _lk(s->ctx);
    cudaSetDevice(s->ctx->device);
    cudaStreamSynchronize(s->ctx->stream);
    ctx_buf_put(s->ctx, s->d_spins, s->bytes);
    if (s->d_alt) ctx_buf_put(s->ctx, s->d_alt, s->bytes);
    ctx_buf_put(s->ctx, s->d_acc, 2 * sizeof(unsigned long long));
    delete s;
}

extern "C" int ising_strip_configure(ising_strip* s, int planes, int rounds) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s) return fail(nullptr, ISING_E_INVALID, "strip is NULL");
    if (planes) {
        if (planes < 5 || planes > 7) return fail(s->ctx, ISING_E_INVALID, "planes must be 5..7");
        s->planes = planes;
    }
    if (rounds) {
        if (rounds != 7 && rounds != 10) return fail(s->ctx, ISING_E_INVALID, "rounds must be 7 or 10");
        s->rounds = rounds;
    }
    return ISING_OK;
}

extern "C" int ising_strip_set_all(ising_strip* s, int up) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s) return fail(nullptr, ISING_E_INVALID, "strip is NULL");
    CUDA_TRY(s->ctx, cudaSetDevice(s->ctx->device));
    CUDA_TRY(s->ctx, cudaMemsetAsync(s->d_spins, up ? 0xFF : 0x00, s->bytes, s->ctx->stream));
    CUDA_TRY(s->ctx, cudaStreamSynchronize(s->ctx->stream));
    return ISING_OK;
}

static void strip_fill_args(const ising_strip* s, double beta, StripSweepArgs* a) {
    a->spins = s->d_spins;
    a->g = s->g;
    a->sweep = (uint32_t)s->sweep;
    a->key0 = (uint32_t)s->seed;
    a->key1 = (uint32_t)(s->seed >> 32);
    a->antiferro = s->j > 0 ? 0xFFFFFFFFu : 0u;
    a->planes = s->planes;
    a->rounds = s->rounds;
    memset(&a->th, 0, sizeof a->th);
    for (int c = 0; c < 2; ++c) {
        const uint64_t T = threshold64(beta, 4.0 * (c + 1) * fabs(s->j), s->planes);
        for (int pl = 0; pl < s->planes; ++pl)
            a->th.plane[c][pl] = ((T >> (s->planes + 31 - pl)) & 1ull) ? 0xFFFFFFFFu : 0u;
        a->th.low[c] = (uint32_t)(T & 0xFFFFFFFFull);
    }
}

// One whole sweep as a single out-of-place pass (launch_strip_sweep_fused): colour 0 on storage rows
// [r0, r1), colour 1 on [r0 + 1, r1 - 1).  Returns 1 when done that way (the two arrays swap roles),
// 0 when the caller should run the two colour phases, < 0 on error (message set).
static int strip_sweep_fused(ising_strip* s, double beta, uint64_t r0, uint64_t r1) {
    static const bool on = getenv("ISING_STRIP_FUSE") != nullptr;   // opt-in: measured slower, see strip.cu
    if (!on || s->field != 0.0 || r1 < r0 + 4) return 0;   // no field variant: two phase launches
    ising_ctx* ctx = s->ctx;
    if (s->sweep > 0xFFFFFFFFull) return 0;   // the phase path reports the overflow
    if (!s->d_alt) {
        void* p = nullptr;
        if (ctx_buf_get(ctx, s->bytes, &p) != cudaSuccess) {   // no room for a second array: two phases
            cudaGetLastError();
            return 0;
        }
        s->d_alt = (uint32_t*)p;
        // rows the sweeps never write (outermost ghost rows) must not hold garbage the observables read
        if (cudaMemcpyAsync(s->d_alt, s->d_spins, s->bytes, cudaMemcpyDeviceToDevice, ctx->stream) != cudaSuccess)
            return -fail(ctx, ISING_E_CUDA, "strip: copy into the second array failed");
    }
    StripSweepArgs a;
    strip_fill_args(s, beta, &a);
    a.colour = 0;
    a.r_begin = (uint32_t)r0;
    a.r_count = (uint32_t)(r1 - r0);
    const int n = launch_strip_sweep_fused(a, s->d_spins, s->d_alt, ctx->stream);
    if (n < 0) return -fail(ctx, ISING_E_CUDA, "fused strip sweep launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    if (n == 0) return 0;
    std::swap(s->d_spins, s->d_alt);
    s->launches++;
    s->sweep++;
    return 1;
}

// Local rows [r0, r1) of one colour phase; the ghost rows of the OTHER colour must hold the
// neighbours' boundary rows when r0 == 0 or r1 == rows.  sync = 0 only enqueues (no host wait,
// no event timing); advance != 0 bumps the sweep counter (call it on the last piece of colour 1).
static int strip_phase_storage_rows(ising_strip* s, int colour, double beta, uint64_t r0, uint64_t r1,
                                    int advance, int sync) {
    ising_ctx* ctx = s->ctx;
    if (s->sweep > 0xFFFFFFFFull)   // 32-bit sweep index in the Philox counter: refuse to wrap
        return fail(ctx, ISING_E_UNSUPPORTED, "sweep counter passed 2^32: start a new lattice or seed");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    StripSweepArgs a;
    strip_fill_args(s, beta, &a);
    a.colour = (uint32_t)colour;
    a.r_begin = (uint32_t)r0;
    a.r_count = (uint32_t)(r1 - r0);
    if (sync) CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    int n;
    if (s->field != 0.0) {   // h = +-0 runs the plain kernel: the same bits, at its speed
        FieldThresholds th;
        fill_field_thresholds(fabs(s->j), s->field, 2, beta, s->planes, &th);
        n = launch_strip_phase_field(a, th, ctx->stream);
    } else {
        n = launch_strip_phase(a, ctx->stream);
    }
    if (n < 0) return fail(ctx, ISING_E_CUDA, "strip phase launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    if (a.r_count) s->launches++;
    if (sync) {
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
        float ms = 0.f;
        CUDA_TRY(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        s->device_ms += ms;
    }
    if (advance) s->sweep++;
    return ISING_OK;
}

extern "C" int ising_strip_phase_rows(ising_strip* s, int colour, double beta, uint64_t r0, uint64_t r1,
                                      int advance, int sync) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s || colour < 0 || colour > 1) return fail(s ? s->ctx : nullptr, ISING_E_INVALID, "bad strip/colour");
    if (r0 > r1 || r1 > s->g.rows) return fail(s->ctx, ISING_E_INVALID, "bad row range");
    return strip_phase_storage_rows(s, colour, beta, s->g.ghost + r0, s->g.ghost + r1, advance, sync);
}

// The local rows plus `ext` ghost rows on each side (ext < ghost): the redundant update of
// ghost rows reproduces the neighbour's bits (Philox is keyed by the global row), so that after
// one deep exchange of 2k rows a strip can run k sweeps without communicating: phase q of the
// batch (q = 0 .. 2k-1) is called with ext = 2k - 1 - q.
extern "C" int ising_strip_phase_ext(ising_strip* s, int colour, double beta, uint32_t ext, int advance,
                                     int sync) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s || colour < 0 || colour > 1) return fail(s ? s->ctx : nullptr, ISING_E_INVALID, "bad strip/colour");
    if (ext >= s->g.ghost) return fail(s->ctx, ISING_E_INVALID, "ext must be < ghost depth");
    return strip_phase_storage_rows(s, colour, beta, s->g.ghost - ext, s->g.ghost + s->g.rows + ext,
                                    advance, sync);
}

// one whole colour phase, blocking; the sweep counter advances after colour 1
extern "C" int ising_strip_phase(ising_strip* s, int colour, double beta) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s) return fail(nullptr, ISING_E_INVALID, "strip is NULL");
    return ising_strip_phase_rows(s, colour, beta, 0, s->g.rows, colour == 1, 1);
}

// Uniform longitudinal field h (E = sum J s s' - h sum s, s = +1 for an up spin) of every later phase
// and sweep of this strip; h = 0 runs the zero-field kernel.
extern "C" int ising_strip_set_field(ising_strip* s, double h) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s) return fail(nullptr, ISING_E_INVALID, "strip is NULL");
    if (!std::isfinite(h)) return fail(s->ctx, ISING_E_INVALID, "field must be finite");
    s->field = h;
    return ISING_OK;
}

// storage row r of a colour (local row l is r = ghost + l)
static uint32_t* strip_row_ptr(ising_strip* s, int colour, uint32_t r) {
    return s->d_spins + ((size_t)colour * (s->g.rows + 2 * s->g.ghost) + r) * s->g.Wr;
}

// Deep halo staging, both colours at once.  buf = uint32[2 sides][2 colours][depth][Lx/64]
// (host or device memory).  dir = 0: side 0 <- the first `depth` local rows, side 1 <- the last
// `depth` local rows; dir = 1: side 0 -> the `depth` ghost rows above the first local row,
// side 1 -> the ghost rows below the last one.  Rows are in increasing global order.  A strip
// sends side 0 to the strip above and side 1 to the strip below and receives the upper
// neighbour's side 1 into its side 0.  sync = 0 only enqueues.
extern "C" int ising_strip_halo_deep(ising_strip* s, int dir, uint32_t depth, void* buf, int sync) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s || !buf) return fail(s ? s->ctx : nullptr, ISING_E_INVALID, "bad argument");
    ising_ctx* ctx = s->ctx;
    const StripGeom& g = s->g;
    if (depth < 1 || depth > g.ghost || depth > g.rows)
        return fail(ctx, ISING_E_INVALID, "depth must be 1..min(ghost, rows)");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const size_t nb = (size_t)depth * g.Wr * 4;
    uint8_t* b = (uint8_t*)buf;
    for (int side = 0; side < 2; ++side)
        for (int c = 0; c < 2; ++c) {
            uint8_t* slot = b + (size_t)(side * 2 + c) * nb;
            if (dir == 0) {
                const uint32_t r = side ? g.ghost + g.rows - depth : g.ghost;
                CUDA_TRY(ctx, cudaMemcpyAsync(slot, strip_row_ptr(s, c, r), nb, cudaMemcpyDefault, ctx->stream));
            } else {
                const uint32_t r = side ? g.ghost + g.rows : g.ghost - depth;
                CUDA_TRY(ctx, cudaMemcpyAsync(strip_row_ptr(s, c, r), slot, nb, cudaMemcpyDefault, ctx->stream));
            }
        }
    if (sync) CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return ISING_OK;
}

// single strip covering the whole lattice: periodic wrap of `depth` rows of both colours
extern "C" int ising_strip_wrap_deep(ising_strip* s, uint32_t depth) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s) return fail(nullptr, ISING_E_INVALID, "strip is NULL");
    ising_ctx* ctx = s->ctx;
    const StripGeom& g = s->g;
    if (depth < 1 || depth > g.ghost || depth > g.rows)
        return fail(ctx, ISING_E_INVALID, "depth must be 1..min(ghost, rows)");
    if (g.rows != g.Ly) return fail(ctx, ISING_E_INVALID, "wrap needs a strip that holds the whole lattice");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const size_t nb = (size_t)depth * g.Wr * 4;
    for (int c = 0; c < 2; ++c) {
        CUDA_TRY(ctx, cudaMemcpyAsync(strip_row_ptr(s, c, g.ghost - depth), strip_row_ptr(s, c, g.ghost + g.rows - depth),
                                      nb, cudaMemcpyDeviceToDevice, ctx->stream));
        CUDA_TRY(ctx, cudaMemcpyAsync(strip_row_ptr(s, c, g.ghost + g.rows), strip_row_ptr(s, c, g.ghost), nb,
                                      cudaMemcpyDeviceToDevice, ctx->stream));
    }
    return ISING_OK;
}

// which = 0: first local row, 1: last local row.  dst holds Lx/64 words, host or device memory.
extern "C" int ising_strip_get_boundary(ising_strip* s, int colour, int which, void* dst) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s || !dst || colour < 0 || colour > 1) return fail(s ? s->ctx : nullptr, ISING_E_INVALID, "bad argument");
    ising_ctx* ctx = s->ctx;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, cudaMemcpyAsync(dst, strip_row_ptr(s, colour, which ? s->g.ghost + s->g.rows - 1 : s->g.ghost),
                                  (size_t)s->g.Wr * 4, cudaMemcpyDefault, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return ISING_OK;
}

// Device-to-device halo staging without a host wait, for contexts created on the caller's
// stream: dir = 0 copies both boundary rows of `colour` into buf_dev[0..Wr) (first row) and
// buf_dev[Wr..2Wr) (last row); dir = 1 copies buf_dev[0..Wr) into the ghost row above the first
// row and buf_dev[Wr..2Wr) into the ghost row below the last row.
extern "C" int ising_strip_halo_async(ising_strip* s, int colour, int dir, void* buf_dev) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s || !buf_dev || colour < 0 || colour > 1) return fail(s ? s->ctx : nullptr, ISING_E_INVALID, "bad argument");
    ising_ctx* ctx = s->ctx;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const size_t nb = (size_t)s->g.Wr * 4;
    uint8_t* b = (uint8_t*)buf_dev;
    if (dir == 0) {
        CUDA_TRY(ctx, cudaMemcpyAsync(b, strip_row_ptr(s, colour, s->g.ghost), nb, cudaMemcpyDeviceToDevice, ctx->stream));
        CUDA_TRY(ctx, cudaMemcpyAsync(b + nb, strip_row_ptr(s, colour, s->g.ghost + s->g.rows - 1), nb, cudaMemcpyDeviceToDevice, ctx->stream));
    } else {
        CUDA_TRY(ctx, cudaMemcpyAsync(strip_row_ptr(s, colour, s->g.ghost - 1), b, nb, cudaMemcpyDeviceToDevice, ctx->stream));
        CUDA_TRY(ctx, cudaMemcpyAsync(strip_row_ptr(s, colour, s->g.ghost + s->g.rows), b + nb, nb, cudaMemcpyDeviceToDevice, ctx->stream));
    }
    return ISING_OK;
}

// which = 0: ghost row above the first local row, 1: ghost row below the last local row
extern "C" int ising_strip_set_ghost(ising_strip* s, int colour, int which, const void* src) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s || !src || colour < 0 || colour > 1) return fail(s ? s->ctx : nullptr, ISING_E_INVALID, "bad argument");
    ising_ctx* ctx = s->ctx;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, cudaMemcpyAsync(strip_row_ptr(s, colour, which ? s->g.ghost + s->g.rows : s->g.ghost - 1), src,
                                  (size_t)s->g.Wr * 4, cudaMemcpyDefault, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return ISING_OK;
}

// single strip covering the whole lattice: periodic wrap of its own boundary rows
extern "C" int ising_strip_wrap_local(ising_strip* s, int colour) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s || colour < 0 || colour > 1) return fail(s ? s->ctx : nullptr, ISING_E_INVALID, "bad argument");
    ising_ctx* ctx = s->ctx;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const size_t nb = (size_t)s->g.Wr * 4;
    CUDA_TRY(ctx, cudaMemcpyAsync(strip_row_ptr(s, colour, s->g.ghost - 1), strip_row_ptr(s, colour, s->g.ghost + s->g.rows - 1), nb,
                                  cudaMemcpyDeviceToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(strip_row_ptr(s, colour, s->g.ghost + s->g.rows), strip_row_ptr(s, colour, s->g.ghost), nb,
                                  cudaMemcpyDeviceToDevice, ctx->stream));
    return ISING_OK;
}

// local sums: satisfied bonds (colour-0 sites see every bond once; needs colour-1 ghosts) and up spins
extern "C" int ising_strip_observables(ising_strip* s, uint64_t* nsat, uint64_t* up) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s || !nsat || !up) return fail(s ? s->ctx : nullptr, ISING_E_INVALID, "bad argument");
    ising_ctx* ctx = s->ctx;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, cudaMemsetAsync(s->d_acc, 0, 2 * sizeof(unsigned long long), ctx->stream));
    if (launch_strip_observables(s->d_spins, s->g, s->j > 0 ? 0xFFFFFFFFu : 0u, s->d_acc, ctx->stream) < 0)
        return fail(ctx, ISING_E_CUDA, "strip observables launch failed");
    s->launches++;
    unsigned long long h[2];
    CUDA_TRY(ctx, cudaMemcpyAsync(h, s->d_acc, sizeof h, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    *nsat = h[0];
    *up = h[1];
    return ISING_OK;
}

int comm_world(const ising_comm* c);
int comm_ring_exchange(ising_comm* c, const void* send_up, const void* send_down, void* recv_up,
                       void* recv_down, size_t bytes, cudaStream_t st);
int comm_allreduce_sum_u64(ising_comm* c, const void* send, void* recv, size_t count, cudaStream_t st);

// `depth` boundary rows of both colours to the neighbouring strips' ghost rows (periodic ring of
// ranks), straight from / into the spin array: the rows of one colour are contiguous, so a
// message is one ncclSend of depth * Lx/64 words.  comm = NULL (or one rank): the strip wraps
// onto itself.  Enqueue only.
static int strip_exchange_deep(ising_strip* s, ising_comm* comm, uint32_t depth) {
    if (!comm || comm_world(comm) == 1) return ising_strip_wrap_deep(s, depth);
    const StripGeom& g = s->g;
    if (depth < 1 || depth > g.ghost || depth > g.rows)
        return fail(s->ctx, ISING_E_INVALID, "depth must be 1..min(ghost, rows)");
    const size_t nb = (size_t)depth * g.Wr * 4;
    for (int c = 0; c < 2; ++c) {
        const int rc = comm_ring_exchange(comm, strip_row_ptr(s, c, g.ghost), strip_row_ptr(s, c, g.ghost + g.rows - depth),
                                          strip_row_ptr(s, c, g.ghost - depth), strip_row_ptr(s, c, g.ghost + g.rows), nb,
                                          s->ctx->stream);
        if (rc) return rc;
    }
    return ISING_OK;
}

// nsweeps checkerboard sweeps of a lattice that is split in row strips over the ranks of `comm`
// (BASELINE config 5; the reference cannot run it, lattice.rs:197-212): batches of k =
// exchange_every sweeps, each one deep halo exchange of 2k rows per side (NCCL send/recv over
// NVLink, issued here on the context's stream) followed by 2k colour phases that update the
// shrinking valid part of the ghost rows redundantly.  The host waits once, at the end.
// fields = NULL: every sweep in the strip's field; else sweep t runs in fields[t], which stays set.
static int strip_sweeps(ising_strip* s, ising_comm* comm, const double* betas, const double* fields,
                        uint64_t nsweeps, uint32_t exchange_every) {
    if (!s || (nsweeps && !betas)) return fail(s ? s->ctx : nullptr, ISING_E_INVALID, "strip/betas is NULL");
    ising_ctx* ctx = s->ctx;
    for (uint64_t t = 0; fields && t < nsweeps; ++t)
        if (!std::isfinite(fields[t])) return fail(ctx, ISING_E_INVALID, "fields must be finite");
    const StripGeom& g = s->g;
    uint32_t k = exchange_every ? exchange_every : 1;
    if (2 * k > g.ghost) k = g.ghost / 2;
    if (2 * k > g.rows) k = g.rows / 2;
    if (k < 1) return fail(ctx, ISING_E_INVALID, "strip needs >= 2 ghost rows and >= 2 local rows for batched sweeps");
    if ((!comm || comm_world(comm) == 1) && g.rows != g.Ly)
        return fail(ctx, ISING_E_INVALID, "a strip that holds only part of the lattice needs a communicator");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    int rc = ISING_OK;
    for (uint64_t i = 0; i < nsweeps && rc == ISING_OK;) {
        const uint32_t nb = (uint32_t)std::min<uint64_t>(k, nsweeps - i);
        rc = strip_exchange_deep(s, comm, 2 * nb);
        for (uint32_t q = 0; q < 2 * nb && rc == ISING_OK; q += 2) {
            if (fields) s->field = fields[i + q / 2];
            // ISING_STRIP_FUSE=1: both colours in one out-of-place pass (6 -> 4 bits of DRAM traffic per
            // site and sweep, but measured 7 % slower: strip.cu); default: the two phase launches
            const int fused = strip_sweep_fused(s, betas[i + q / 2], g.ghost - (2 * nb - 1 - q),
                                                g.ghost + g.rows + (2 * nb - 1 - q));
            if (fused < 0) rc = -fused;
            for (uint32_t c = 0; c < 2 && fused == 0 && rc == ISING_OK; ++c)
                rc = strip_phase_storage_rows(s, (int)c, betas[i + q / 2], g.ghost - (2 * nb - 1 - q - c),
                                              g.ghost + g.rows + (2 * nb - 1 - q - c), (int)c, 0);
        }
        i += nb;
    }
    cudaEventRecord(ctx->ev1, ctx->stream);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (rc) return rc;
    if (e != cudaSuccess) return fail(ctx, ISING_E_CUDA, "strip sweeps: %s", cudaGetErrorString(e));
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) s->device_ms += ms;
    return ISING_OK;
}

extern "C" int ising_strip_sweeps(ising_strip* s, ising_comm* comm, const double* betas, uint64_t nsweeps,
                                  uint32_t exchange_every) {
    CtxLock _lk(s ? s->ctx : nullptr);
    return strip_sweeps(s, comm, betas, nullptr, nsweeps, exchange_every);
}

// the same loop with one (beta, h) per sweep; the kernel is chosen per sweep by fields[t] != 0
extern "C" int ising_strip_sweeps_field(ising_strip* s, ising_comm* comm, const double* betas, const double* fields,
                                        uint64_t nsweeps, uint32_t exchange_every) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (s && nsweeps && !fields) return fail(s->ctx, ISING_E_INVALID, "fields is NULL");
    return strip_sweeps(s, comm, betas, fields, nsweeps, exchange_every);
}

// Global sums over all strips: satisfied bonds and up spins of the whole lattice (halo exchange
// of one colour-1 row, local reduction, NCCL all-reduce).
extern "C" int ising_strip_global_sums(ising_strip* s, ising_comm* comm, uint64_t* nsat, uint64_t* up) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s || !nsat || !up) return fail(s ? s->ctx : nullptr, ISING_E_INVALID, "bad argument");
    ising_ctx* ctx = s->ctx;
    const StripGeom& g = s->g;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    if (!comm || comm_world(comm) == 1) {
        if (g.rows != g.Ly) return fail(ctx, ISING_E_INVALID, "a partial strip needs a communicator");
        const int rc = ising_strip_wrap_local(s, 1);
        if (rc) return rc;
    } else {
        const size_t nb = (size_t)g.Wr * 4;
        const int rc = comm_ring_exchange(comm, strip_row_ptr(s, 1, g.ghost), strip_row_ptr(s, 1, g.ghost + g.rows - 1),
                                          strip_row_ptr(s, 1, g.ghost - 1), strip_row_ptr(s, 1, g.ghost + g.rows), nb,
                                          ctx->stream);
        if (rc) return rc;
    }
    CUDA_TRY(ctx, cudaMemsetAsync(s->d_acc, 0, 2 * sizeof(unsigned long long), ctx->stream));
    if (launch_strip_observables(s->d_spins, s->g, s->j > 0 ? 0xFFFFFFFFu : 0u, s->d_acc, ctx->stream) < 0)
        return fail(ctx, ISING_E_CUDA, "strip observables launch failed");
    s->launches++;
    if (comm && comm_world(comm) > 1) {
        const int rc = comm_allreduce_sum_u64(comm, s->d_acc, s->d_acc, 2, ctx->stream);
        if (rc) return rc;
    }
    unsigned long long h[2];
    CUDA_TRY(ctx, cudaMemcpyAsync(h, s->d_acc, sizeof h, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    *nsat = h[0];
    *up = h[1];
    return ISING_OK;
}

extern "C" int ising_strip_get_rows(ising_strip* s, uint8_t* rows_out) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s || !rows_out) return fail(s ? s->ctx : nullptr, ISING_E_INVALID, "bad argument");
    ising_ctx* ctx = s->ctx;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const size_t bytes = (size_t)s->g.rows * s->Lx;
    void* dv = nullptr;
    CUDA_TRY(ctx, ctx_scratch(ctx, 0, bytes, &dv));
    if (launch_strip_unpack(s->d_spins, s->g, (uint8_t*)dv, ctx->stream) < 0)
        return fail(ctx, ISING_E_CUDA, "strip unpack launch failed");
    s->launches++;
    CUDA_TRY(ctx, cudaMemcpyAsync(rows_out, dv, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return ISING_OK;
}

// local rows [r0, r1) only (a band of a lattice too large to read back whole)
extern "C" int ising_strip_get_row_range(ising_strip* s, uint64_t r0, uint64_t r1, uint8_t* rows_out) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s || !rows_out) return fail(s ? s->ctx : nullptr, ISING_E_INVALID, "bad argument");
    if (r0 > r1 || r1 > s->g.rows) return fail(s->ctx, ISING_E_INVALID, "bad row range");
    ising_ctx* ctx = s->ctx;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const size_t bytes = (size_t)(r1 - r0) * s->Lx;
    if (bytes == 0) return ISING_OK;
    void* dv = nullptr;
    CUDA_TRY(ctx, ctx_scratch(ctx, 0, bytes, &dv));
    if (launch_strip_unpack(s->d_spins, s->g, (uint8_t*)dv, ctx->stream, (uint32_t)r0, (uint32_t)(r1 - r0)) < 0)
        return fail(ctx, ISING_E_CUDA, "strip unpack launch failed");
    s->launches++;
    CUDA_TRY(ctx, cudaMemcpyAsync(rows_out, dv, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return ISING_OK;
}

extern "C" int ising_strip_get_stats(ising_strip* s, uint64_t* launches, double* device_ms, int reset) {
    CtxLock _lk(s ? s->ctx : nullptr);
    if (!s) return fail(nullptr, ISING_E_INVALID, "strip is NULL");
    if (launches) *launches = s->launches;
    if (device_ms) *device_ms = s->device_ms;
    if (reset) { s->launches = 0; s->device_ms = 0.0; }
    return ISING_OK;
}
