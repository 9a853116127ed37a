// C ABI of libising_b200.so (include/ising_b200.h).  Host orchestration only: argument
// checks with the reference's error behaviour, device buffers, kernel launches, CUDA-event
// timing.  There is deliberately no CPU implementation behind these entry points: without a
// CUDA device every compute call fails with ISING_E_CUDA.
#include "api_internal.h"

// ------------------------------------------------------------------------------------------
// error reporting, context buffer caches
// ------------------------------------------------------------------------------------------
static thread_local std::string g_global_error;

int fail(ising_ctx* ctx, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf;
    g_global_error = buf;
    return code;
}

cudaError_t ctx_buf_get(ising_ctx* ctx, size_t bytes, void** out) {
    bytes = std::max<size_t>(bytes, 256);
    for (size_t i = 0; i < ctx->free_bufs.size(); ++i)
        if (ctx->free_bufs[i].second >= bytes && ctx->free_bufs[i].second <= bytes + bytes / 4 + 4096) {
            *out = ctx->free_bufs[i].first;
            ctx->free_bytes -= ctx->free_bufs[i].second;
            ctx->free_bufs.erase(ctx->free_bufs.begin() + i);
            return cudaSuccess;
        }
    return cudaMalloc(out, bytes);
}


void ctx_buf_put(ising_ctx* ctx, void* p, size_t bytes) {
    if (!p) return;
    bytes = std::max<size_t>(bytes, 256);
    const size_t cap = (size_t)8 << 30;
    if (ctx->free_bytes + bytes > cap || ctx->free_bufs.size() >= 64) {
        cudaFree(p);
        return;
    }
    ctx->free_bufs.emplace_back(p, bytes);
    ctx->free_bytes += bytes;
}

cudaError_t ctx_scratch(ising_ctx* ctx, int slot, size_t bytes, void** out) {
    if (ctx->scratch_bytes[slot] < bytes) {
        if (ctx->scratch[slot]) cudaFree(ctx->scratch[slot]);
        ctx->scratch[slot] = nullptr;
        ctx->scratch_bytes[slot] = 0;
        const size_t want = std::max<size_t>(bytes, 1 << 20);
        cudaError_t e = cudaMalloc(&ctx->scratch[slot], want);
        if (e != cudaSuccess) return e;
        ctx->scratch_bytes[slot] = want;
    }
    *out = ctx->scratch[slot];
    return cudaSuccess;
}

// rows of `width` bytes, device (pitch spitch) to host (pitch dpitch); the 2D copy engine path
// is limited to pitches below 2^31, longer rows go one by one
cudaError_t copy_rows_d2h(void* dst, size_t dpitch, const void* src, size_t spitch, size_t width,
                                 size_t height, cudaStream_t st) {
    if (width == 0 || height == 0) return cudaSuccess;
    if (dpitch < (1ull << 31) && spitch < (1ull << 31))
        return cudaMemcpy2DAsync(dst, dpitch, src, spitch, width, height, cudaMemcpyDeviceToHost, st);
    for (size_t r = 0; r < height; ++r) {
        cudaError_t e = cudaMemcpyAsync((char*)dst + r * dpitch, (const char*)src + r * spitch, width,
                                        cudaMemcpyDeviceToHost, st);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}


// ------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------
extern "C" int ising_abi_version(void) { return ISING_ABI_VERSION; }

extern "C" const char* ising_last_error(const ising_ctx* ctx) {
    return ctx ? ctx->err.c_str() : g_global_error.c_str();
}

static int ctx_create_impl(int device, cudaStream_t external, bool use_external, ising_ctx** out);

extern "C" int ising_ctx_create(int device, ising_ctx** out) {
    return ctx_create_impl(device, nullptr, false, out);
}

// Same, but every launch and copy of this context goes to the caller's stream (e.g. torch's
// current stream): work is then ordered with the caller's own kernels and NCCL calls without
// host synchronisation.
extern "C" int ising_ctx_create_on_stream(int device, void* cuda_stream, ising_ctx** out) {
    return ctx_create_impl(device, (cudaStream_t)cuda_stream, true, out);
}

static int ctx_create_impl(int device, cudaStream_t external, bool use_external, ising_ctx** out) {
    if (!out) return fail(nullptr, ISING_E_INVALID, "out is NULL");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, ISING_E_CUDA,
                    "no CUDA device available (%s); libising_b200 has no CPU fallback",
                    e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    if (device < 0 || device >= ndev)
        return fail(nullptr, ISING_E_INVALID, "device %d out of range (0..%d)", device, ndev - 1);
    CUDA_TRY(nullptr, cudaSetDevice(device));
    cudaDeviceProp prop;
    CUDA_TRY(nullptr, cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(nullptr, ISING_E_CUDA,
                    "device %d is sm_%d%d; this library is built for sm_100a (B200) only", device,
                    prop.major, prop.minor);
    std::unique_ptr<ising_ctx> ctx(new ising_ctx);
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    if (use_external) {
        ctx->stream = external;
        ctx->owns_stream = false;
    } else {
        CUDA_TRY(nullptr, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    }
    CUDA_TRY(nullptr, cudaEventCreate(&ctx->ev0));
    CUDA_TRY(nullptr, cudaEventCreate(&ctx->ev1));
    *out = ctx.release();
    return ISING_OK;
}

extern "C" void ising_ctx_destroy(ising_ctx* ctx) {
    if (!ctx) return;
    bool now;
    {
        std::lock_guard<std::recursive_mutex> g(ctx->mu);
        ctx->destroy_requested = true;
        now = ctx->children == 0;
    }
    if (now) ctx_really_destroy(ctx);
}

void ctx_really_destroy(ising_ctx* ctx) {
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    for (int b = 0; b < 2; ++b) {
        if (ctx->ev_filled[b]) cudaEventDestroy(ctx->ev_filled[b]);
        if (ctx->ev_drained[b]) cudaEventDestroy(ctx->ev_drained[b]);
    }
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->stream && ctx->owns_stream) cudaStreamDestroy(ctx->stream);
    for (void* p : ctx->scratch) cudaFree(p);
    for (auto& b : ctx->free_bufs) cudaFree(b.first);
    delete ctx;
}

extern "C" int ising_host_alloc(size_t bytes, void** out) {
    if (!out) return fail(nullptr, ISING_E_INVALID, "out is NULL");
    *out = nullptr;
    cudaError_t e = cudaHostAlloc(out, std::max<size_t>(bytes, 1), cudaHostAllocPortable);
    if (e != cudaSuccess)
        return fail(nullptr, ISING_E_NOMEM, "cudaHostAlloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
    return ISING_OK;
}

extern "C" void ising_host_free(void* p) {
    if (p) cudaFreeHost(p);
}

// ------------------------------------------------------------------------------------------
// graph
// ------------------------------------------------------------------------------------------
static int upload_stencil_masks(ising_ctx* ctx, ising_graph* g) {
    const HostGraph& h = g->h;
    if (h.kind == ISING_KIND_GENERAL || h.uniform_sign) return ISING_OK;
    const int dim = h.kind == ISING_KIND_STENCIL3D ? 3 : 2;
    const uint64_t Lx = h.dims[0], Ly = h.dims[1], Lz = h.dims[2];
    const uint64_t Lxh = Lx / 2, rows = Ly * Lz, halfN = h.nvars / 2;
    std::vector<uint32_t> m((size_t)2 * 2 * dim * halfN);
    auto sgn = [&](uint64_t x, uint64_t y, uint64_t z, int d) -> uint32_t {
        const uint64_t n = x + Lx * (y + Ly * z);
        return ((h.fwd_sign[n] >> d) & 1) ? 0xFFFFFFFFu : 0u;
    };
    for (uint32_t c = 0; c < 2; ++c)
        for (uint64_t r = 0; r < rows; ++r) {
            const uint64_t z = r / Ly, y = r % Ly;
            const uint32_t p = (uint32_t)((y + z + c) & 1);
            for (uint64_t xh = 0; xh < Lxh; ++xh) {
                const uint64_t x = 2 * xh + p;
                const uint64_t xm = x == 0 ? Lx - 1 : x - 1;
                const uint64_t ym = y == 0 ? Ly - 1 : y - 1, zm = z == 0 ? Lz - 1 : z - 1;
                uint32_t* base = m.data() + (size_t)c * 2 * dim * halfN + r * Lxh + xh;
                // k = 0: neighbour stored at the same half-index (x+1 if p == 0 else x-1)
                // k = 1: the other x neighbour;  2: y-1  3: y+1  4: z-1  5: z+1
                const uint32_t jxp = sgn(x, y, z, 0), jxm = sgn(xm, y, z, 0);
                base[0 * halfN] = p == 0 ? jxp : jxm;
                base[1 * halfN] = p == 0 ? jxm : jxp;
                base[2 * halfN] = sgn(x, ym, z, 1);
                base[3 * halfN] = sgn(x, y, z, 1);
                if (dim == 3) {
                    base[4 * halfN] = sgn(x, y, zm, 2);
                    base[5 * halfN] = sgn(x, y, z, 2);
                }
            }
        }
    CUDA_TRY(ctx, dev_alloc(&g->d_jmask, m.size()));
    CUDA_TRY(ctx, cudaMemcpy(g->d_jmask, m.data(), m.size() * sizeof(uint32_t),
                             cudaMemcpyHostToDevice));
    // the same masks site-major, [colour][halfN][8] (k = 0..2*dim-1, rest 0): two 128-bit loads
    // per site in the row-walk kernel instead of 2*dim scalar ones
    std::vector<uint32_t> m8((size_t)2 * halfN * 8, 0u);
    for (uint32_t c = 0; c < 2; ++c)
        for (uint64_t i = 0; i < halfN; ++i)
            for (int k = 0; k < 2 * dim; ++k)
                m8[((size_t)c * halfN + i) * 8 + k] = m[(size_t)c * 2 * dim * halfN + (size_t)k * halfN + i];
    CUDA_TRY(ctx, dev_alloc(&g->d_jmask8, m8.size()));
    CUDA_TRY(ctx, cudaMemcpy(g->d_jmask8, m8.data(), m8.size() * sizeof(uint32_t),
                             cudaMemcpyHostToDevice));
    return ISING_OK;
}

int ensure_csr_on_device(ising_ctx* ctx, ising_graph* g) {
    if (g->d_row) return ISING_OK;
    g->h.build_csr();
    const HostGraph& h = g->h;
    CUDA_TRY(ctx, dev_alloc(&g->d_row, h.row.size()));
    CUDA_TRY(ctx, dev_alloc(&g->d_nbr, h.nbr.size()));
    CUDA_TRY(ctx, dev_alloc(&g->d_jv, h.jv.size()));
    CUDA_TRY(ctx, dev_alloc(&g->d_bias, h.nvars));
    CUDA_TRY(ctx, cudaMemcpy(g->d_row, h.row.data(), h.row.size() * 8, cudaMemcpyHostToDevice));
    CUDA_TRY(ctx, cudaMemcpy(g->d_nbr, h.nbr.data(), h.nbr.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(ctx, cudaMemcpy(g->d_jv, h.jv.data(), h.jv.size() * 8, cudaMemcpyHostToDevice));
    std::vector<double> b(h.nvars, 0.0);
    if (h.has_bias) b = h.bias;
    CUDA_TRY(ctx, cudaMemcpy(g->d_bias, b.data(), h.nvars * 8, cudaMemcpyHostToDevice));
    return ISING_OK;
}

int ensure_csr32_on_device(ising_ctx* ctx, ising_graph* g) {
    if (g->d_row32) return ISING_OK;
    HostGraph& h = g->h;
    h.build_csr();
    if (2 * h.nedges > 0xFFFFFFFFull) return fail(ctx, ISING_E_UNSUPPORTED, "too many edges");
    const uint64_t N = h.nvars;
    std::vector<uint32_t> row32(N + 1);
    for (uint64_t n = 0; n <= N; ++n) row32[n] = (uint32_t)h.row[n];
    std::vector<uint8_t> anti8(h.jv.size());
    for (size_t k = 0; k < h.jv.size(); ++k) anti8[k] = h.jv[k] > 0;
    CUDA_TRY(ctx, dev_alloc(&g->d_row32, row32.size()));
    CUDA_TRY(ctx, dev_alloc(&g->d_nbr32, h.nbr.size()));
    CUDA_TRY(ctx, dev_alloc(&g->d_anti8, anti8.size()));
    CUDA_TRY(ctx, cudaMemcpy(g->d_row32, row32.data(), row32.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(ctx, cudaMemcpy(g->d_nbr32, h.nbr.data(), h.nbr.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(ctx, cudaMemcpy(g->d_anti8, anti8.data(), anti8.size(), cudaMemcpyHostToDevice));
    return ISING_OK;
}

// arbitrary real couplings and biases: colour-ordered site list + float CSR values
int ensure_real_on_device(ising_ctx* ctx, ising_graph* g) {
    if (g->real_built) return ISING_OK;
    int rc = ensure_csr32_on_device(ctx, g);
    if (rc) return rc;
    rc = ensure_csr_on_device(ctx, g);  // f64 couplings / biases for the energy kernel
    if (rc) return rc;
    HostGraph& h = g->h;
    const uint64_t N = h.nvars;
    std::vector<uint32_t> order(N);
    g->color_off.assign(h.ncolors + 1, 0);
    for (uint64_t n = 0; n < N; ++n) g->color_off[h.color_of(n) + 1]++;
    for (int c = 0; c < h.ncolors; ++c) g->color_off[c + 1] += g->color_off[c];
    std::vector<uint32_t> fill(g->color_off.begin(), g->color_off.end() - 1);
    for (uint64_t n = 0; n < N; ++n) order[fill[h.color_of(n)]++] = (uint32_t)n;
    std::vector<float> jf(h.jv.begin(), h.jv.end());
    std::vector<float> bf(N, 0.f);
    if (h.has_bias) for (uint64_t n = 0; n < N; ++n) bf[n] = (float)h.bias[n];
    CUDA_TRY(ctx, dev_alloc(&g->d_csites, order.size()));
    CUDA_TRY(ctx, dev_alloc(&g->d_jf, jf.size()));
    CUDA_TRY(ctx, dev_alloc(&g->d_biasf, bf.size()));
    CUDA_TRY(ctx, cudaMemcpy(g->d_csites, order.data(), order.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(ctx, cudaMemcpy(g->d_jf, jf.data(), jf.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(ctx, cudaMemcpy(g->d_biasf, bf.data(), bf.size() * 4, cudaMemcpyHostToDevice));
    g->real_built = true;
    return ISING_OK;
}

// non-basic moves: f32 CSR + the classes of a strong edge colouring
int ensure_moves_on_device(ising_ctx* ctx, ising_graph* g) {
    if (g->moves_built) return ISING_OK;
    int rc = ensure_real_on_device(ctx, g);
    if (rc) return rc;
    if (g->h.nedges > 0xFFFFFFFFull) return fail(ctx, ISING_E_UNSUPPORTED, "too many edges");
    EdgeClasses ec;
    strong_edge_colouring(&g->h, &ec);
    CUDA_TRY(ctx, dev_alloc(&g->d_mea, ec.ea.size()));
    CUDA_TRY(ctx, dev_alloc(&g->d_meb, ec.eb.size()));
    CUDA_TRY(ctx, dev_alloc(&g->d_meid, ec.eid.size()));
    CUDA_TRY(ctx, dev_alloc(&g->d_mwrel, ec.wrel.size()));
    CUDA_TRY(ctx, cudaMemcpy(g->d_mea, ec.ea.data(), ec.ea.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(ctx, cudaMemcpy(g->d_meb, ec.eb.data(), ec.eb.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(ctx, cudaMemcpy(g->d_meid, ec.eid.data(), ec.eid.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(ctx, cudaMemcpy(g->d_mwrel, ec.wrel.data(), ec.wrel.size() * 4, cudaMemcpyHostToDevice));
    g->medge_off = ec.off;
    g->medge = std::move(ec);
    g->moves_built = true;
    return ISING_OK;
}

// (class, outer degree) groups of the bit-sliced edge-move kernel (moves.cu: k_edge_general)
int ensure_edge_general_on_device(ising_ctx* ctx, ising_graph* g, bool stencil_layout) {
    ising_graph::EdgeGen& eg = g->edge_gen[stencil_layout ? 1 : 0];
    if (eg.built) return ISING_OK;
    int rc = ensure_moves_on_device(ctx, g);
    if (rc) return rc;
    HostGraph& h = g->h;
    eg.built = true;
    eg.usable = false;
    if (!h.integer_classes) return ISING_OK;
    const EdgeClasses& ec = g->medge;
    const uint64_t M = ec.ea.size();
    const uint64_t Lx = h.dims[0], Ly = h.dims[1], Lxh = Lx / 2, rows = h.dims[1] * h.dims[2];
    auto slot = [&](uint32_t n) -> uint32_t {
        if (!stencil_layout) return n;
        const uint64_t x = n % Lx, r = n / Lx, y = r % Ly, z = r / Ly;
        const uint64_t c = (x + y + z) & 1u;
        return (uint32_t)((c * rows + r) * Lxh + (x >> 1));
    };
    // outer bonds of every edge: the adjacency entries of a and of b that do not lead to the other end
    struct Item { uint32_t sa, sb, eid, anti, endp, deg; uint32_t nb[GEN_MAX_DEG]; };
    std::vector<Item> items(M);
    for (uint64_t i = 0; i < M; ++i) {
        Item& it = items[i];
        const uint32_t a = ec.ea[i], b = ec.eb[i];
        it.sa = slot(a); it.sb = slot(b); it.eid = ec.eid[i]; it.anti = 0; it.endp = 0; it.deg = 0;
        for (int end = 0; end < 2; ++end) {
            const uint32_t u = end ? b : a, other = end ? a : b;
            for (uint64_t k = h.row[u]; k < h.row[u + 1]; ++k) {
                if (h.nbr[k] == other) continue;
                if (it.deg >= (uint32_t)GEN_MAX_DEG) return ISING_OK;   // too many outer bonds: float kernel
                if (h.jv[k] > 0) it.anti |= 1u << it.deg;
                if (end) it.endp |= 1u << it.deg;
                it.nb[it.deg++] = slot(h.nbr[k]);
            }
        }
    }
    // blob layout per group: sa | sb | eid | anti | endp | nbr[deg][count]
    std::vector<uint32_t> blob;
    struct Off { size_t at; uint32_t count, deg; };
    std::vector<Off> offs;
    for (size_t c = 0; c + 1 < ec.off.size(); ++c)
        for (uint32_t d = 0; d <= (uint32_t)GEN_MAX_DEG; ++d) {
            std::vector<uint32_t> idx;
            for (uint32_t i = ec.off[c]; i < ec.off[c + 1]; ++i)
                if (items[i].deg == d) idx.push_back(i);
            if (idx.empty()) continue;
            const uint32_t n = (uint32_t)idx.size();
            Off o{blob.size(), n, d};
            blob.resize(blob.size() + (size_t)(5 + d) * n);
            uint32_t* p = blob.data() + o.at;
            for (uint32_t q = 0; q < n; ++q) {
                const Item& it = items[idx[q]];
                p[q] = it.sa; p[n + q] = it.sb; p[2 * n + q] = it.eid; p[3 * n + q] = it.anti; p[4 * n + q] = it.endp;
                for (uint32_t k = 0; k < d; ++k) p[(size_t)(5 + k) * n + q] = it.nb[k];
            }
            offs.push_back(o);
        }
    CUDA_TRY(ctx, dev_alloc(&eg.d_blob, blob.size()));
    CUDA_TRY(ctx, cudaMemcpy(eg.d_blob, blob.data(), blob.size() * 4, cudaMemcpyHostToDevice));
    for (const Off& o : offs) {
        EdgeGroup gr;
        const uint32_t* p = eg.d_blob + o.at;
        gr.sa = p; gr.sb = p + o.count; gr.eid = p + 2 * (size_t)o.count; gr.anti = p + 3 * (size_t)o.count;
        gr.endp = p + 4 * (size_t)o.count; gr.nbr = p + 5 * (size_t)o.count;
        gr.count = o.count; gr.deg = o.deg;
        eg.groups.push_back(gr);
    }
    eg.usable = true;
    return ISING_OK;
}

// host only: no context, no device
extern "C" int ising_strong_edge_colouring(uint64_t nvars, uint64_t nedges, const uint64_t* a, const uint64_t* b,
                                           uint32_t* cls, uint32_t* nclasses) {
    if ((nedges && (!a || !b || !cls)) || !nclasses) return fail(nullptr, ISING_E_INVALID, "null argument");
    if (nedges > 0xFFFFFFFFull || nvars > 0xFFFFFFFFull) return fail(nullptr, ISING_E_UNSUPPORTED, "graph too large");
    HostGraph h;
    h.nvars = nvars;
    h.nedges = nedges;
    h.ea.assign(a, a + nedges);
    h.eb.assign(b, b + nedges);
    h.ej.assign(nedges, 1.0);
    for (uint64_t e = 0; e < nedges; ++e)
        if (a[e] >= nvars || b[e] >= nvars || a[e] == b[e])
            return fail(nullptr, ISING_E_INVALID, "edge %llu: end points must be distinct sites below nvars",
                        (unsigned long long)e);
    EdgeClasses ec;
    strong_edge_colouring(&h, &ec);
    for (size_t c = 0; c + 1 < ec.off.size(); ++c)
        for (uint32_t i = ec.off[c]; i < ec.off[c + 1]; ++i) cls[ec.eid[i]] = (uint32_t)c;
    *nclasses = (uint32_t)(ec.off.size() - 1);
    return ISING_OK;
}

extern "C" int ising_graph_get_edge_classes(ising_graph* g, uint32_t* cls) {
    CtxLock _lk(g ? g->ctx : nullptr);
    if (!g || !cls) return fail(nullptr, ISING_E_INVALID, "graph/cls is NULL");
    CUDA_TRY(g->ctx, cudaSetDevice(g->ctx->device));
    const int rc = ensure_moves_on_device(g->ctx, g);
    if (rc) return rc;
    const EdgeClasses& ec = g->medge;
    for (size_t c = 0; c + 1 < ec.off.size(); ++c)
        for (uint32_t i = ec.off[c]; i < ec.off[c + 1]; ++i) cls[ec.eid[i]] = (uint32_t)c;
    return ISING_OK;
}

// colour x degree groups of a graph whose couplings all have the same magnitude
int ensure_general_on_device(ising_ctx* ctx, ising_graph* g) {
    if (g->gen_built) return ISING_OK;
    HostGraph& h = g->h;
    if (!h.integer_classes)
        return fail(ctx, ISING_E_INVALID, "internal: integer-class kernels on a real-valued graph");
    {
        const int rc32 = ensure_csr32_on_device(ctx, g);
        if (rc32) return rc32;
    }
    const uint64_t N = h.nvars;
    const int ncol = h.ncolors;
    // bucket sites by (colour, degree)
    std::vector<std::vector<uint32_t>> bucket((size_t)ncol * (GEN_MAX_DEG + 1));
    for (uint64_t n = 0; n < N; ++n) {
        const uint32_t deg = (uint32_t)(h.row[n + 1] - h.row[n]);
        bucket[(size_t)h.color_of(n) * (GEN_MAX_DEG + 1) + deg].push_back((uint32_t)n);
    }
    std::vector<uint32_t> sites, nbr, anti;
    struct Off { size_t s, n; uint32_t count, deg; int color; };
    std::vector<Off> offs;
    for (int c = 0; c < ncol; ++c)
        for (int d = 0; d <= GEN_MAX_DEG; ++d) {
            const auto& b = bucket[(size_t)c * (GEN_MAX_DEG + 1) + d];
            if (b.empty()) continue;
            Off o{sites.size(), nbr.size(), (uint32_t)b.size(), (uint32_t)d, c};
            sites.insert(sites.end(), b.begin(), b.end());
            nbr.resize(nbr.size() + (size_t)d * b.size());
            for (size_t i = 0; i < b.size(); ++i) {
                const uint64_t lo = h.row[b[i]];
                uint32_t bits = 0;
                for (int k = 0; k < d; ++k) {
                    nbr[o.n + (size_t)k * b.size() + i] = h.nbr[lo + k];
                    if (h.jv[lo + k] > 0) bits |= 1u << k;
                }
                anti.push_back(bits);
            }
            offs.push_back(o);
        }
    CUDA_TRY(ctx, dev_alloc(&g->d_gsites, sites.size()));
    CUDA_TRY(ctx, dev_alloc(&g->d_gnbr, nbr.size()));
    CUDA_TRY(ctx, dev_alloc(&g->d_ganti, anti.size()));
    CUDA_TRY(ctx, cudaMemcpy(g->d_gsites, sites.data(), sites.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(ctx, cudaMemcpy(g->d_gnbr, nbr.data(), nbr.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(ctx, cudaMemcpy(g->d_ganti, anti.data(), anti.size() * 4, cudaMemcpyHostToDevice));
    for (const Off& o : offs) {
        GenGroup gg;
        gg.sites = g->d_gsites + o.s;
        gg.nbr = g->d_gnbr + o.n;
        gg.anti = g->d_ganti + o.s;
        gg.count = o.count;
        gg.deg = o.deg;
        g->gen_groups.push_back(gg);
        g->gen_group_color.push_back(o.color);
    }
    g->gen_ncolors = ncol;
    g->gen_built = true;
    return ISING_OK;
}

extern "C" int ising_graph_from_edges(ising_ctx* ctx, uint64_t nvars, uint64_t nedges,
                                      const uint64_t* a, const uint64_t* b, const double* j,
                                      const double* biases, ising_graph** out) {
    CtxLock _lk(ctx);
    if (!ctx || !out) return fail(ctx, ISING_E_INVALID, "ctx/out is NULL");
    *out = nullptr;
    if (nedges && (!a || !b || !j)) return fail(ctx, ISING_E_INVALID, "edge arrays are NULL");
    std::unique_ptr<ising_graph> g(new ising_graph);
    g->ctx = ctx;
    const std::string msg = compile_from_edges(nvars, nedges, a, b, j, biases, &g->h);
    if (!msg.empty()) return fail(ctx, ISING_E_INVALID, "%s", msg.c_str());
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const int rc = upload_stencil_masks(ctx, g.get());
    if (rc) return rc;
    *out = g.release();
    ctx_retain(ctx);
    return ISING_OK;
}

extern "C" int ising_graph_torus(ising_ctx* ctx, int dim, const uint64_t* L, double j0, int pmj,
                                 uint64_t j_seed, ising_graph** out) {
    CtxLock _lk(ctx);
    if (!ctx || !out || !L) return fail(ctx, ISING_E_INVALID, "ctx/out/L is NULL");
    *out = nullptr;
    std::unique_ptr<ising_graph> g(new ising_graph);
    g->ctx = ctx;
    const std::string msg = make_torus(dim, L, j0, pmj, j_seed, &g->h);
    if (!msg.empty()) return fail(ctx, ISING_E_INVALID, "%s", msg.c_str());
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const int rc = upload_stencil_masks(ctx, g.get());
    if (rc) return rc;
    *out = g.release();
    ctx_retain(ctx);
    return ISING_OK;
}

extern "C" int ising_graph_torus_field(ising_ctx* ctx, int dim, const uint64_t* L, double j0, int pmj,
                                       uint64_t j_seed, double h, ising_graph** out) {
    CtxLock _lk(ctx);
    if (!ctx || !out || !L) return fail(ctx, ISING_E_INVALID, "ctx/out/L is NULL");
    *out = nullptr;
    if (!std::isfinite(h)) return fail(ctx, ISING_E_INVALID, "field must be finite");
    const int rc = ising_graph_torus(ctx, dim, L, j0, pmj, j_seed, out);
    if (rc) return rc;
    (*out)->h.field_graph = true;
    (*out)->h.field = h;
    return ISING_OK;
}

extern "C" void ising_graph_destroy(ising_graph* g) {
    if (!g) return;
    ising_ctx* owner = g->ctx;
    struct Release { ising_ctx* c; ~Release() { ctx_release(c); } } _rel{owner};   // after the lock is gone
    CtxLock _lk(owner);
    if (g->ctx) cudaSetDevice(g->ctx->device);
    cudaFree(g->d_jmask);
    cudaFree(g->d_jmask8);
    cudaFree(g->d_row);
    cudaFree(g->d_nbr);
    cudaFree(g->d_jv);
    cudaFree(g->d_bias);
    cudaFree(g->d_gsites);
    cudaFree(g->d_gnbr);
    cudaFree(g->d_ganti);
    cudaFree(g->d_row32);
    cudaFree(g->d_nbr32);
    cudaFree(g->d_anti8);
    cudaFree(g->d_csites);
    cudaFree(g->d_jf);
    cudaFree(g->d_biasf);
    cudaFree(g->d_mea);
    cudaFree(g->d_meb);
    cudaFree(g->d_meid);
    cudaFree(g->d_mwrel);
    cudaFree(g->edge_gen[0].d_blob);
    cudaFree(g->edge_gen[1].d_blob);
    delete g;
}

extern "C" int ising_graph_get_info(const ising_graph* g, ising_graph_info* out) {
    CtxLock _lk(g ? g->ctx : nullptr);
    if (!g || !out) return fail(nullptr, ISING_E_INVALID, "graph/out is NULL");
    const HostGraph& h = g->h;
    out->nvars = h.nvars;
    out->nedges = h.nedges;
    out->kind = h.kind;
    out->ncolors = h.ncolors;
    out->max_degree = h.max_degree;
    out->integer_classes = h.integer_classes ? 1 : 0;
    out->dims[0] = h.dims[0];
    out->dims[1] = h.dims[1];
    out->dims[2] = h.dims[2];
    out->jabs = h.jabs;
    return ISING_OK;
}

extern "C" int ising_graph_get_colors(const ising_graph* g, uint32_t* colors) {
    CtxLock _lk(g ? g->ctx : nullptr);
    if (!g || !colors) return fail(nullptr, ISING_E_INVALID, "graph/colors is NULL");
    for (uint64_t n = 0; n < g->h.nvars; ++n) colors[n] = g->h.color_of(n);
    return ISING_OK;
}

extern "C" int ising_graph_get_edges(const ising_graph* g, uint64_t* a, uint64_t* b, double* j) {
    CtxLock _lk(g ? g->ctx : nullptr);
    if (!g || !a || !b || !j) return fail(nullptr, ISING_E_INVALID, "graph/arrays NULL");
    for (uint64_t e = 0; e < g->h.nedges; ++e) g->h.edge_at(e, a + e, b + e, j + e);
    return ISING_OK;
}

extern "C" int ising_make_seeds(uint64_t seed_gen, uint64_t n, uint64_t* out) {
    if (n && !out) return fail(nullptr, ISING_E_INVALID, "out is NULL");
    make_seeds(seed_gen, n, out);
    return ISING_OK;
}

extern "C" int ising_schedule_betas(const uint64_t* st, const double* sb, uint64_t n,
                                    uint64_t timesteps, int linear, double* out) {
    if ((n && (!st || !sb)) || (timesteps && !out))
        return fail(nullptr, ISING_E_INVALID, "schedule arrays are NULL");
    if (!schedule_betas(st, sb, n, timesteps, linear != 0, out))
        return fail(nullptr, ISING_E_INVALID, "annealing schedule has fewer than two stops");
    return ISING_OK;
}
