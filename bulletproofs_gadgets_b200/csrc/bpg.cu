// bpg.cu -- libbpg: context, resident generators, MSM driver and the C ABI (include/bpg.h).
// Single translation unit: device kernels live in kernels_*.cuh, host protocol code in host_*.h / prover.inl.
#include "bpg_internal.h"
#include "consts.h"
#include "host_merlin.h"
#include "host_rng_service.h"
#include "host_scalar64.h"
#include "kernels_core.cuh"
#include "kernels_msm.cuh"
#include "kernels_vec.cuh"
#include "kernels_batch.cuh"

#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <atomic>
#include <mutex>
#include <thread>

#include <strings.h>

static thread_local std::string g_cuda_err;
void bpg_set_cuda_error(cudaError_t e, const char *file, int line) {
    char buf[512];
    snprintf(buf, sizeof buf, "%s:%d: %s (%s)", file, line, cudaGetErrorString(e), cudaGetErrorName(e));
    g_cuda_err = buf;
}
#define CTX_TRY(x) do { int rc_ = (x); if (rc_ != BPG_OK) { if (rc_ == BPG_E_CUDA) ctx->last_error = g_cuda_err; return rc_; } } while (0)
#define KCHECK() do { ctx->launches++; cudaError_t e_ = cudaGetLastError(); if (e_ != cudaSuccess) { bpg_set_cuda_error(e_, __FILE__, __LINE__); ctx->last_error = g_cuda_err; return BPG_E_CUDA; } } while (0)

int dev_buf::ensure(size_t bytes) {
    if (bytes <= cap) return BPG_OK;
    if (p) { cudaFree(p); p = nullptr; cap = 0; }
    size_t want = bytes + bytes / 8 + 256;
    CUDA_TRY(cudaMalloc(&p, want));
    cap = want;
    return BPG_OK;
}
void dev_buf::release() { if (p) cudaFree(p); p = nullptr; cap = 0; }

// Wait for the context's stream.  With BPG_BLOCKING_SYNC=1 the host thread sleeps on an event created with
// cudaEventBlockingSync instead of spinning, which leaves the core to the other provers' transcript RNG.
// (process-wide switches are atomics: prover threads read them while another thread may call the setter)
static std::atomic<int> g_blocking_sync{-1};
static inline int blocking_sync_now() {
    int v = g_blocking_sync.load(std::memory_order_relaxed);
    if (v < 0) { const char *e = getenv("BPG_BLOCKING_SYNC"); v = (e && e[0] == '1') ? 1 : 0; int exp = -1; g_blocking_sync.compare_exchange_strong(exp, v); v = g_blocking_sync.load(); }
    return v;
}
int bpg_stream_sync(bpg_ctx *ctx, cudaStream_t s) {
    if (!blocking_sync_now() || s != ctx->stream) { CUDA_TRY(cudaStreamSynchronize(s)); return BPG_OK; }
    CUDA_TRY(cudaEventRecord(ctx->ev, s));
    CUDA_TRY(cudaEventSynchronize(ctx->ev));
    return BPG_OK;
}
extern "C" void bpg_set_blocking_sync(int on) { g_blocking_sync.store(on ? 1 : 0); }
#define SYNC_TRY(ctx, s) CTX_TRY(bpg_stream_sync(ctx, s))
// Device -> pageable host copies return only when the copy is done, and the driver SPINS for everything queued before
// them (measured: 47 ms of host CPU per proof with 48 provers sharing a GPU, starving the transcript-RNG lanes).  In
// blocking-sync mode the thread first sleeps on the stream's event, so the copy finds an idle stream.
#define D2H_TRY(ctx, dst, src, bytes, s) do { if (blocking_sync_now() == 1) SYNC_TRY(ctx, s); CUDA_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, s)); } while (0)

// ================================================================ context
extern "C" const char *bpg_strerror(int code) {
    switch (code) {
    case BPG_OK: return "ok";
    case BPG_E_CUDA: return "CUDA error";
    case BPG_E_SIZE: return "invalid size / generator capacity";
    case BPG_E_DECOMPRESS: return "point decompression failed";
    case BPG_E_ARG: return "invalid argument";
    case BPG_E_FORMAT: return "proof format error";
    case BPG_E_NOMEM: return "out of memory";
    case BPG_E_COMM: return "NCCL communicator error";
    }
    return "unknown";
}
extern "C" void bpg_set_sizing_mode(int mode);
extern "C" void bpg_ctx_destroy(bpg_ctx *ctx);
// __constant__ symbols are per-device globals: uploaded once per device, under a lock, and complete (device-wide sync) before
// any kernel of any context can run -- the contexts' streams are cudaStreamNonBlocking and do not order against the legacy
// default stream the symbol copy uses.
static std::mutex g_const_mu;
static bool g_const_done[64] = {false};
static int upload_device_constants(int device) {
    std::lock_guard<std::mutex> lk(g_const_mu);
    if (device < 64 && g_const_done[device]) return BPG_OK;
    if (bpg_init_constants_host() != 0) return BPG_E_ARG;
    CUDA_TRY(cudaMemcpyToSymbol(c_K, &h_K, sizeof(bpg_consts)));
    CUDA_TRY(cudaDeviceSynchronize());
    if (device < 64) g_const_done[device] = true;
    return BPG_OK;
}
extern "C" int bpg_ctx_create(int device, bpg_ctx **out) {
    if (!out) return BPG_E_ARG;
    *out = nullptr;
    int ndev = 0;
    CUDA_TRY(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return BPG_E_ARG;
    CUDA_TRY(cudaSetDevice(device));
    int rc = upload_device_constants(device);
    if (rc != BPG_OK) return rc;
    (void)blocking_sync_now();
    static std::once_flag sizing_once;
    std::call_once(sizing_once, [] { if (const char *e = getenv("BPG_SIZING_MODE")) bpg_set_sizing_mode(atoi(e)); });
    bpg_ctx *ctx = new bpg_ctx();
    ctx->device = device;
    // BPG_ACC_PRIO=0 switches the priority split off (every kernel on one default-priority stream, as in round 1)
    static const int acc_prio = [] { const char *e2 = getenv("BPG_ACC_PRIO"); return e2 ? atoi(e2) : 1; }();
    int prio_lo = 0, prio_hi = 0;
    cudaError_t e = cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi); // (numerically: lowest priority = largest value)
    if (!acc_prio) prio_lo = prio_hi = 0;
    if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&ctx->stream, cudaStreamNonBlocking, prio_hi);
    if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&ctx->stream2, cudaStreamNonBlocking, prio_hi);
    if (e == cudaSuccess && acc_prio) {
        e = cudaStreamCreateWithPriority(&ctx->acc_stream, cudaStreamNonBlocking, prio_lo);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_acc[0], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_acc[1], cudaEventDisableTiming);
    }
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev, cudaEventDisableTiming | cudaEventBlockingSync);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev2, cudaEventDisableTiming);
    if (e != cudaSuccess) { // nothing of a half-built context may leak
        bpg_set_cuda_error(e, __FILE__, __LINE__);
        bpg_ctx_destroy(ctx);
        return BPG_E_CUDA;
    }
    *out = ctx;
    return BPG_OK;
}
extern "C" void bpg_ctx_destroy(bpg_ctx *ctx) {
    if (!ctx) return;
    const bool dbg = getenv("BPG_TRACE_DESTROY") != nullptr;
#define DSTEP(name) do { if (dbg) { fprintf(stderr, "[bpg destroy %p] %s\n", (void *)ctx, name); fflush(stderr); } } while (0)
    DSTEP("begin");
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    DSTEP("synced");
    if (ctx->comm) bpg_comm_destroy(ctx);
    for (int i = 0; i < 2; i++) { prefetch_slot_free(ctx->pre[i]); ctx->pre[i] = nullptr; }
    for (cudaEvent_t e : ctx->prof_ev) cudaEventDestroy(e);
    ctx->prof_ev.clear();
    DSTEP("prof events destroyed");
    // prover secrets (witness, blindings, transcript-RNG draws) do not outlive the context
    for (int i : {8, 9, 12, 13}) if (ctx->scratch[i].p) cudaMemset(ctx->scratch[i].p, 0, ctx->scratch[i].cap);
    if (ctx->h_pinned) explicit_bzero(ctx->h_pinned, ctx->h_pinned_cap);
    ctx->gens.reset(); // the tables are freed with their last user
    ctx->tab = nullptr; ctx->comb = nullptr;
    DSTEP("tables freed");
    dev_buf *bufs[] = {&ctx->counts, &ctx->offsets, &ctx->cursor, &ctx->sorted, &ctx->partial, &ctx->buckets, &ctx->lvlP, &ctx->lvlQ, &ctx->heavy, &ctx->results};
    for (dev_buf *b : bufs) b->release();
    for (dev_buf &b : ctx->scratch) b.release();
    ctx->batch_gh.release();
    ctx->vb_sums.release(); ctx->comm_recv.release();
    ctx->mat_pts.release(); ctx->mat_ext.release(); ctx->mat_tab.release(); ctx->heavy_part.release();
    DSTEP("buffers freed");
    if (ctx->h_pinned) cudaFreeHost(ctx->h_pinned);
    if (ctx->prof_pairs) cudaFreeHost(ctx->prof_pairs);
    DSTEP("pinned freed");
    for (int i = 0; i < 16; i++) if (ctx->tev[i]) { if (dbg) fprintf(stderr, "[bpg destroy] tev[%d]=%p\n", i, (void *)ctx->tev[i]); cudaEventDestroy(ctx->tev[i]); }
    DSTEP("timer events destroyed");
    for (int i = 0; i < 2; i++) if (ctx->ev_stage[i]) cudaEventDestroy(ctx->ev_stage[i]);
    if (ctx->ev) cudaEventDestroy(ctx->ev);
    if (ctx->ev2) cudaEventDestroy(ctx->ev2);
    DSTEP("events destroyed");
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    if (ctx->stream2) cudaStreamDestroy(ctx->stream2);
    if (ctx->acc_stream) cudaStreamDestroy(ctx->acc_stream);
    for (cudaEvent_t &ev : ctx->ev_acc) if (ev) cudaEventDestroy(ev);
    DSTEP("streams destroyed");
    delete ctx;
#undef DSTEP
}
extern "C" const char *bpg_last_error(bpg_ctx *ctx) { return ctx ? ctx->last_error.c_str() : g_cuda_err.c_str(); }
extern "C" uint64_t bpg_launch_count(bpg_ctx *ctx) { return ctx ? ctx->launches : 0; }
extern "C" int bpg_sync(bpg_ctx *ctx) { if (!ctx) return BPG_E_ARG; SYNC_TRY(ctx, ctx->stream); return BPG_OK; }

extern "C" int bpg_dev_alloc(bpg_ctx *ctx, size_t bytes, void **d_ptr) { if (!ctx || !d_ptr) return BPG_E_ARG; CUDA_TRY(cudaSetDevice(ctx->device)); CUDA_TRY(cudaMalloc(d_ptr, bytes ? bytes : 1)); return BPG_OK; }
extern "C" int bpg_dev_free(bpg_ctx *ctx, void *d_ptr) { if (!ctx) return BPG_E_ARG; CUDA_TRY(cudaFree(d_ptr)); return BPG_OK; }
extern "C" int bpg_host_alloc(bpg_ctx *ctx, size_t bytes, void **h_ptr) { if (!ctx || !h_ptr) return BPG_E_ARG; CUDA_TRY(cudaSetDevice(ctx->device)); CUDA_TRY(cudaHostAlloc(h_ptr, bytes ? bytes : 1, cudaHostAllocPortable)); return BPG_OK; }
extern "C" int bpg_host_free(bpg_ctx *ctx, void *h_ptr) { if (!ctx) return BPG_E_ARG; CUDA_TRY(cudaFreeHost(h_ptr)); return BPG_OK; }
extern "C" int bpg_dev_upload(bpg_ctx *ctx, void *d_dst, const void *h_src, size_t bytes) {
    if (!ctx) return BPG_E_ARG;
    CUDA_TRY(cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    SYNC_TRY(ctx, ctx->stream);
    return BPG_OK;
}
extern "C" int bpg_dev_download(bpg_ctx *ctx, void *h_dst, const void *d_src, size_t bytes) {
    if (!ctx) return BPG_E_ARG;
    D2H_TRY(ctx, h_dst, d_src, bytes, ctx->stream);
    SYNC_TRY(ctx, ctx->stream);
    return BPG_OK;
}

// ================================================================ generators
static const uint8_t RISTRETTO_BASEPOINT[32] = {0xe2, 0xf2, 0xae, 0x0a, 0x6a, 0xbc, 0x4e, 0x71, 0xa8, 0x84, 0xa9, 0x61, 0xc5, 0x00, 0x51, 0x5f,
                                                0x58, 0xe3, 0x0b, 0x6a, 0xa5, 0x82, 0xdd, 0x8d, 0xb6, 0xa6, 0x59, 0x45, 0xe0, 0x8d, 0x2d, 0x76};

extern "C" size_t bpg_gens_capacity(bpg_ctx *ctx) { return ctx ? ctx->cap : 0; }

gens_tables::~gens_tables() {
    cudaSetDevice(device);
    if (tab) cudaFree(tab);
    if (comb) cudaFree(comb);
}
static std::mutex g_gens_mu;
static std::weak_ptr<gens_tables> g_gens[64]; // per device: the largest table set currently alive

static int gens_build(bpg_ctx *ctx, size_t cap, std::shared_ptr<gens_tables> &out) {
    std::shared_ptr<gens_tables> g = std::make_shared<gens_tables>();
    g->device = ctx->device;
    uint32_t ptotal = (uint32_t)(2 * cap + 2);
    size_t tab_bytes = (size_t)BPG_NWIN * ptotal * sizeof(ge_an);
    if (cudaMalloc((void **)&g->tab, tab_bytes) != cudaSuccess) { cudaGetLastError(); return BPG_E_NOMEM; }
    CUDA_TRY(cudaMalloc((void **)&g->comb, (size_t)2 * 32 * 128 * sizeof(ge_an)));
    // SHAKE256 streams on two host threads (sequential squeeze, ~0.3 us per 136 bytes)
    size_t sbytes = 64 * cap;
    // pageable staging: this is a one-off upload, and freeing / re-allocating a large pinned buffer after timing events had
    // been used made cudaEventDestroy crash on this driver (580.159) -- see tools/repro_teardown.py
    std::vector<uint8_t> stage(2 * sbytes + 128);
    uint8_t *hs = stage.data();
    std::thread tg([&] { bpgh::generators_chain_stream('G', 0, hs, cap); });
    bpgh::generators_chain_stream('H', 0, hs + sbytes, cap);
    tg.join();
    // B~ = from_uniform_bytes(SHA3-512(compress(B)))
    bpgh::sha3_512(hs + 2 * sbytes, RISTRETTO_BASEPOINT, 32);
    memcpy(hs + 2 * sbytes + 64, RISTRETTO_BASEPOINT, 32);
    CTX_TRY(ctx->scratch[0].ensure(2 * sbytes + 128));
    uint8_t *ds = (uint8_t *)ctx->scratch[0].p;
    CUDA_TRY(cudaMemcpyAsync(ds, hs, 2 * sbytes + 128, cudaMemcpyHostToDevice, ctx->stream));
    k_gens_tables<<<LAUNCH_1D(2 * cap, 128), 0, ctx->stream>>>(ds, (uint32_t)(2 * cap), 0, ptotal, g->tab);
    KCHECK();
    CTX_TRY(ctx->scratch[1].ensure(16));
    uint32_t one = 1;
    CUDA_TRY(cudaMemcpyAsync(ctx->scratch[1].p, &one, 4, cudaMemcpyHostToDevice, ctx->stream));
    k_point_tables<<<1, 32, 0, ctx->stream>>>(ds + 2 * sbytes + 64, 1, (uint32_t)(2 * cap), ptotal, g->tab, (uint32_t *)ctx->scratch[1].p);
    KCHECK();
    k_gens_tables<<<1, 32, 0, ctx->stream>>>(ds + 2 * sbytes, 1, (uint32_t)(2 * cap + 1), ptotal, g->tab);
    KCHECK();
    k_build_comb<<<1, 64, 0, ctx->stream>>>(g->tab, ptotal, (uint32_t)(2 * cap), g->comb);
    KCHECK();
    SYNC_TRY(ctx, ctx->stream); // complete before any other context (other stream) can see the tables
    g->cap = cap;
    g->ptotal = ptotal;
    out = g;
    return BPG_OK;
}

extern "C" int bpg_gens_ensure(bpg_ctx *ctx, size_t capacity) {
    if (!ctx) return BPG_E_ARG;
    if (capacity <= ctx->cap) return BPG_OK;
    if (capacity > (1u << 22)) return BPG_E_SIZE;
    CUDA_TRY(cudaSetDevice(ctx->device));
    size_t cap = 64;
    while (cap < capacity) cap <<= 1;
    static int private_tables = -1;
    if (private_tables < 0) { const char *e = getenv("BPG_PRIVATE_TABLES"); private_tables = (e && e[0] == '1') ? 1 : 0; }
    std::shared_ptr<gens_tables> g;
    {
        // held while building: contexts asking for the same tables at the same time wait for the first one instead of
        // building their own copy
        std::lock_guard<std::mutex> lk(g_gens_mu);
        if (!private_tables && ctx->device < 64) g = g_gens[ctx->device].lock();
        if (!g || g->cap < cap) {
            g.reset();
            CTX_TRY(gens_build(ctx, cap, g));
            if (!private_tables && ctx->device < 64) g_gens[ctx->device] = g;
        }
    }
    SYNC_TRY(ctx, ctx->stream); // nothing of this context may still read the tables it is about to release
    ctx->gens = g;
    ctx->tab = g->tab; ctx->comb = g->comb;
    ctx->cap = g->cap; ctx->ptotal = g->ptotal;
    return BPG_OK;
}

extern "C" int bpg_gens_export(bpg_ctx *ctx, size_t i0, size_t n, uint8_t *G32, uint8_t *H32) {
    if (!ctx) return BPG_E_ARG;
    if (i0 + n > ctx->cap) return BPG_E_SIZE;
    if (n == 0) return BPG_OK;
    CUDA_TRY(cudaSetDevice(ctx->device));
    CTX_TRY(ctx->scratch[0].ensure(64 * n));
    uint8_t *d = (uint8_t *)ctx->scratch[0].p;
    k_export_kernel<<<LAUNCH_1D(n, 64), 0, ctx->stream>>>(ctx->tab, (uint32_t)i0, (uint32_t)n, d);
    KCHECK();
    k_export_kernel<<<LAUNCH_1D(n, 64), 0, ctx->stream>>>(ctx->tab, (uint32_t)(ctx->cap + i0), (uint32_t)n, d + 32 * n);
    KCHECK();
    if (G32) D2H_TRY(ctx, G32, d, 32 * n, ctx->stream);
    if (H32) D2H_TRY(ctx, H32, d + 32 * n, 32 * n, ctx->stream);
    SYNC_TRY(ctx, ctx->stream);
    return BPG_OK;
}
extern "C" int bpg_pedersen_gens(bpg_ctx *ctx, uint8_t B32[32], uint8_t Bb32[32]) {
    if (!ctx || !ctx->cap) return BPG_E_ARG;
    CUDA_TRY(cudaSetDevice(ctx->device));
    CTX_TRY(ctx->scratch[0].ensure(64));
    uint8_t *d = (uint8_t *)ctx->scratch[0].p;
    k_export_kernel<<<1, 32, 0, ctx->stream>>>(ctx->tab, (uint32_t)(2 * ctx->cap), 2, d);
    KCHECK();
    uint8_t h[64];
    D2H_TRY(ctx, h, d, 64, ctx->stream);
    SYNC_TRY(ctx, ctx->stream);
    if (B32) memcpy(B32, h, 32);
    if (Bb32) memcpy(Bb32, h + 32, 32);
    return BPG_OK;
}

// ================================================================ device op wrappers
static int run_compress(bpg_ctx *ctx, cudaStream_t s, const ge *d_pts, size_t n, uint8_t *d_out32) {
    if (!n) return BPG_OK;
    if (n <= 32) k_compress_kernel<<<1, 32, 0, s>>>(d_pts, (uint32_t)n, d_out32);
    else k_compress_kernel<<<LAUNCH_1D(n, 128), 0, s>>>(d_pts, (uint32_t)n, d_out32);
    KCHECK();
    return BPG_OK;
}
// tree-sum n points into d_out[0] using scratch d_tmp (>= n/64+1 points); d_pts is clobbered when n > 64
static int run_points_sum(bpg_ctx *ctx, cudaStream_t s, ge *d_pts, size_t n, ge *d_tmp, ge *d_out) {
    ge *src = d_pts, *dst = d_tmp;
    while (true) {
        size_t nb = (n + 63) / 64;
        ge *o = nb == 1 ? d_out : dst;
        k_points_sum_kernel<<<(unsigned)nb, 64, 0, s>>>(src, (uint32_t)n, o);
        KCHECK();
        if (nb == 1) break;
        n = nb;
        ge *t = src; src = dst; dst = t;
    }
    return BPG_OK;
}

// Protocol calls in flight in this process.  With several provers / verifiers sharing the GPU the kernels are sized for
// work efficiency (long accumulate chunks: fewer bucket runs cut at chunk borders, measured +5 % proofs/s at half a wave;
// work-lean row/column reduction); a lone caller gets the latency-oriented sizes (two waves, shallow reductions).
static std::atomic<int> g_inflight{0};
struct bpg_inflight_guard {
    bpg_inflight_guard() { g_inflight.fetch_add(1, std::memory_order_relaxed); }
    ~bpg_inflight_guard() { g_inflight.fetch_sub(1, std::memory_order_relaxed); }
};
static std::atomic<int> g_sizing_mode{-1}; // -1 auto, 0 latency, 1 throughput (bpg_set_sizing_mode)
extern "C" void bpg_set_sizing_mode(int mode) { g_sizing_mode.store(mode < 0 ? -1 : (mode ? 1 : 0)); }
static inline int bpg_lean_now() {
    int m = g_sizing_mode.load(std::memory_order_relaxed);
    return m >= 0 ? m : (g_inflight.load(std::memory_order_relaxed) >= 4 ? 1 : 0);
}

// Common front half of every bucket MSM: histogram -> scan -> counting-sort scatter -> chunked accumulation -> per-bucket
// finish.  `digits(scatter, counters_or_cursor, sorted)` launches the recoding kernel of the caller (k_msm_digits for plain
// MSMs, k_mat_digits for the multi-output fold).  Leaves the nb bucket sums in ctx->buckets.
template <class DigitsLaunch>
static int msm_bucketize(bpg_ctx *ctx, cudaStream_t s, uint32_t nb, size_t maxpairs, bool any, const ge_an *tab, int lean, DigitsLaunch &&digits) {
    // chunk = sorted pairs summed by one thread.  Latency sizing: two full waves of 4 blocks x 128 threads on 148 SMs
    // (151 552 threads).  Throughput sizing (lean): half a wave of longer chunks -- other proofs fill the rest of the GPU.
    size_t tgt = lean ? 37888 : 151552;
    uint32_t cap = lean ? 2 * BPG_CHUNK : BPG_CHUNK;
    uint32_t CH = (uint32_t)((maxpairs + tgt - 1) / tgt);
    if (CH < 8) CH = 8;
    if (CH > cap) CH = cap;
    size_t nchunks = (maxpairs + CH - 1) / CH + 1;
    uint32_t ntiles = (nb + 1023) / 1024;
    CTX_TRY(ctx->counts.ensure(((size_t)nb + 2 + ntiles + 2) * 4)); // counters, then the scan's ticket + per-tile totals
    CTX_TRY(ctx->offsets.ensure(((size_t)nb + 2) * 4));
    CTX_TRY(ctx->cursor.ensure(((size_t)nb + 2) * 4));
    CTX_TRY(ctx->sorted.ensure((maxpairs + 1) * 4));
    CTX_TRY(ctx->partial.ensure(2 * nchunks * sizeof(ge)));
    CTX_TRY(ctx->buckets.ensure((size_t)nb * sizeof(ge)));
    CTX_TRY(ctx->heavy.ensure(((size_t)nb + 2) * 4));
    uint32_t *counts = (uint32_t *)ctx->counts.p, *offsets = (uint32_t *)ctx->offsets.p, *cursor = (uint32_t *)ctx->cursor.p;
    uint32_t *heavy = (uint32_t *)ctx->heavy.p;
    CUDA_TRY(cudaMemsetAsync(counts, 0, ((size_t)nb + 2 + ntiles + 2) * 4, s));
    CUDA_TRY(cudaMemsetAsync(heavy + nb + 1, 0, 4, s));
    if (any) {
        digits(0, counts, (uint32_t *)nullptr);
        KCHECK();
    }
    k_msm_scan<<<ntiles, 256, 0, s>>>(counts, nb, offsets, cursor, counts + nb + 2);
    KCHECK();
    if (any) {
        digits(1, cursor, (uint32_t *)ctx->sorted.p);
        KCHECK();
        bool prof = ctx->prof_on && ctx->prof_n < 64; // the first 64 launches after bpg_prof_enable are timed
        // the accumulation runs on the context's low-priority stream (bpg_internal.h), fenced on both sides
        cudaStream_t sa = (ctx->acc_stream && s == ctx->stream) ? ctx->acc_stream : s;
        if (sa != s) { CUDA_TRY(cudaEventRecord(ctx->ev_acc[0], s)); CUDA_TRY(cudaStreamWaitEvent(sa, ctx->ev_acc[0], 0)); }
        if (prof) CUDA_TRY(cudaEventRecord(ctx->prof_ev[2 * ctx->prof_n], sa)); // events are pre-created by bpg_prof_enable
        k_msm_accumulate<<<LAUNCH_1D(nchunks, 128), 0, sa>>>((const uint32_t *)ctx->sorted.p, offsets, nb, tab, (ge *)ctx->buckets.p, (ge *)ctx->partial.p, CH);
        KCHECK();
        if (prof) CUDA_TRY(cudaEventRecord(ctx->prof_ev[2 * ctx->prof_n + 1], sa));
        if (sa != s) { CUDA_TRY(cudaEventRecord(ctx->ev_acc[1], sa)); CUDA_TRY(cudaStreamWaitEvent(s, ctx->ev_acc[1], 0)); }
        if (prof) {
            CUDA_TRY(cudaMemcpyAsync(&ctx->prof_pairs[ctx->prof_n], offsets + nb, 4, cudaMemcpyDeviceToHost, s));
            ctx->prof_n++;
        }
    }
    k_msm_finish<<<LAUNCH_1D(nb, 64), 0, s>>>(offsets, nb, (ge *)ctx->buckets.p, (const ge *)ctx->partial.p, heavy, heavy + nb + 1, CH);
    KCHECK();
    if (any) {
        // heavy buckets: at most (pairs / (BPG_HEAVY_SPAN * CH)) of them can exist; segment sums, then one block per bucket
        size_t max_heavy = maxpairs / ((size_t)BPG_HEAVY_SPAN * CH) + 1;
        CTX_TRY(ctx->heavy_part.ensure(max_heavy * BPG_HEAVY_SEGS * sizeof(ge)));
        unsigned hb = (unsigned)std::min<size_t>(max_heavy, 64);
        k_msm_heavy<<<dim3(hb, BPG_HEAVY_SEGS), 64, 0, s>>>(offsets, (const ge *)ctx->partial.p, heavy, heavy + nb + 1, CH, (ge *)ctx->heavy_part.p);
        KCHECK();
        k_msm_heavy_final<<<hb, 32, 0, s>>>((ge *)ctx->buckets.p, heavy, heavy + nb + 1, (const ge *)ctx->heavy_part.p);
        KCHECK();
    }
    return BPG_OK;
}

static int msm_run_local(bpg_ctx *ctx, cudaStream_t s, msm_plan *plan, ge *d_out) {
    uint32_t total = 0;
    for (int i = 0; i < plan->nseg; i++) { plan->seg[i].start = total; total += plan->seg[i].n; }
    plan->total = total;
    const int vb = plan->varbase ? 1 : 0;
    const int Gout = plan->ngroups;
    int G = vb ? 16 * Gout : Gout; // bucket groups: with variable points every window of an output is a group of its own
    msm_params P;
    memcpy(P.seg, plan->seg, sizeof(P.seg));
    P.nseg = plan->nseg; P.total = total; P.ptotal = plan->tab ? plan->ptotal : ctx->ptotal; P.varbase = (uint32_t)vb;
    const ge_an *tab = plan->tab ? plan->tab : ctx->tab;
    ge *d_final = d_out;
    if (vb) { // the bucket engine writes the window sums, k_msm_horner16 recombines them into d_final
        CTX_TRY(ctx->vb_sums.ensure((size_t)G * sizeof(ge)));
        d_out = (ge *)ctx->vb_sums.p;
    }
    if (total <= BPG_SMALL_MSM_TERMS) {
        // Small MSM (late IPP rounds over the materialised generators, small circuits): the 2 x 2^15-bucket reduction below
        // would cost more than the accumulation.  Split every 16-bit digit into two 8-bit digits instead (two pairs per
        // digit, 2 x 129 buckets per group) and reduce each group with one k_mat_reduce block.
        uint32_t nb = (uint32_t)G * 2u * BPG_MAT_NB;
        CTX_TRY(msm_bucketize(ctx, s, nb, (size_t)total * BPG_NWIN * 2, total != 0, tab, plan->lean, [&](int scatter, uint32_t *cc, uint32_t *sorted) {
            if (scatter) k_msm_digits<1, 1><<<LAUNCH_1D(total, 256), 0, s>>>(P, cc, sorted);
            else k_msm_digits<0, 1><<<LAUNCH_1D(total, 256), 0, s>>>(P, cc, sorted);
        }));
        CTX_TRY(ctx->lvlQ.ensure(8 * (size_t)G * sizeof(ge)));
        k_small_reduce<<<2 * G, 128, 0, s>>>((const ge *)ctx->buckets.p, (ge *)ctx->lvlQ.p);
        KCHECK();
        k_small_combine<<<(G + 31) / 32, 32, 0, s>>>((const ge *)ctx->lvlQ.p, (uint32_t)G, d_out);
        KCHECK();
        if (vb) { k_msm_horner16<<<(Gout + 31) / 32, 32, 0, s>>>(d_out, (uint32_t)Gout, d_final); KCHECK(); }
        return BPG_OK;
    }
    uint32_t nb = (uint32_t)G * BPG_NBP;
    CTX_TRY(ctx->lvlP.ensure((size_t)G * (BPG_NROWS + BPG_NCOLS) * sizeof(ge)));
    CTX_TRY(ctx->lvlQ.ensure(8 * (size_t)G * sizeof(ge)));
    // large single-group MSMs: shared-memory privatised histogram / scatter (one block per SM), see kernels_msm.cuh
    bool priv = (!vb && G <= BPG_MAX_GROUPS && total >= BPG_PRIV_MSM_TERMS);
    int sms = 0;
    // upper bound of the terms any one group receives (a segment whose group alternates by halves gives each of the two half)
    uint32_t max_group_terms = 0;
    {
        uint32_t per[2 * BPG_MAX_GROUPS] = {0};
        for (int i = 0; i < plan->nseg && G <= BPG_MAX_GROUPS; i++) {
            const msm_seg &sg = plan->seg[i];
            if (sg.alt) { per[sg.group] += (sg.n + 1) / 2 + 1; per[sg.group ^ 1u] += (sg.n + 1) / 2 + 1; }
            else per[sg.group] += sg.n;
        }
        for (uint32_t v : per) max_group_terms = std::max(max_group_terms, v);
    }
    if (priv) {
        // (idempotent and cheap; setting it per call keeps it correct for every device without shared mutable state)
        CUDA_TRY(cudaFuncSetAttribute(k_msm_hist_smem, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(BPG_NBP * 4)));
        CUDA_TRY(cudaFuncSetAttribute(k_msm_scatter_smem, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(BPG_NBP * 4)));
        CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device));
    }
    CTX_TRY(msm_bucketize(ctx, s, nb, (size_t)total * BPG_NWIN, total != 0, tab, plan->lean, [&](int scatter, uint32_t *cc, uint32_t *sorted) {
        if (priv) {
            // the privatised scatter keeps one open range per (block, bucket): beyond ~2^20 terms those ranges no longer fit
            // the 126 MB L2 and the plain cursor-ordered scatter (33 K open sectors) is faster again
            // (measured 2^19 / 2^20 / 2^21 / 2^22 terms: 1.14 / 1.90 / 3.85 / 8.11 ms privatised vs 1.18 / 1.99 / 3.60 / 6.89 ms plain)
            const bool priv_scatter = total <= (1u << 20);
            // several groups of at most 2^20 terms each (the L / R pair of an IPP round over 2 x 2^20 generators, A_I / A_O):
            // one privatised launch per group, one after the other (BPG_SCATTER_PG=0 switches this off for A/B runs)
            static const int scatter_pg = [] { const char *e = getenv("BPG_SCATTER_PG"); return e ? atoi(e) : 1; }();
            // (block size of the privatised kernels, profiles/r02_sort_variants.jsonl: 1024 / 512 / 256 threads -> 57.8 / 59.5 / 60.4 ms per
            // solo 2^20 proof, 24.3 / 24.4 proofs/s with 48 provers: smaller blocks leave more registers to co-resident accumulate
            // blocks but are slower themselves)
            const bool per_group = scatter_pg && !priv_scatter && G > 1 && max_group_terms <= (1u << 20) + 64;
            if (scatter && per_group) { for (int g = 0; g < G; g++) k_msm_scatter_smem<<<dim3(sms, 1), 1024, BPG_NBP * 4, s>>>(P, cc, sorted, (uint32_t)g); }
            else if (scatter && priv_scatter) k_msm_scatter_smem<<<dim3(sms, G), 1024, BPG_NBP * 4, s>>>(P, cc, sorted, 0u);
            else if (scatter) k_msm_digits<1, 0><<<LAUNCH_1D(total, 256), 0, s>>>(P, cc, sorted);
            else k_msm_hist_smem<<<dim3(sms, G), 1024, BPG_NBP * 4, s>>>(P, cc);
        } else {
            if (scatter) k_msm_digits<1, 0><<<LAUNCH_1D(total, 256), 0, s>>>(P, cc, sorted);
            else k_msm_digits<0, 0><<<LAUNCH_1D(total, 256), 0, s>>>(P, cc, sorted);
        }
    }));
    // weighted sum over the 129 x 256 bucket matrix: row/column sums, small-weight multiples, combine
    ge *rc = (ge *)ctx->lvlP.p, *out2 = (ge *)ctx->lvlQ.p;
    // protocol drivers (many proofs in flight) ask for the work-lean reduction; the stand-alone MSM entry points keep the
    // shallower one (measured: lean = +4 % proofs/s, +25 us per solo MSM)
    if (plan->lean) k_msm_rowcol_lean<<<dim3(BPG_NROWS + BPG_NCOLS / 4, G), 32, 0, s>>>((const ge *)ctx->buckets.p, rc);
    else k_msm_rowcol<<<dim3(BPG_NROWS + BPG_NCOLS, G), 64, 0, s>>>((const ge *)ctx->buckets.p, rc);
    KCHECK();
    k_msm_wfinal<<<dim3(8, G), 64, 0, s>>>(rc, out2);
    KCHECK();
    k_msm_combine<<<G, 32, 0, s>>>(out2, d_out);
    KCHECK();
    if (vb) { k_msm_horner16<<<(Gout + 31) / 32, 32, 0, s>>>(d_out, (uint32_t)Gout, d_final); KCHECK(); }
    return BPG_OK;
}

// ---------------------------------------------------------------- NCCL exchange of partial points (K10)
// The library owns a communicator per sharded context and enqueues ncclAllGather on the context's OWN stream, between the
// kernel that produced the partial points and the kernel that adds the world's partials: no host synchronisation, no
// callback, ~35 exchanges per 2^20 proof cost their NVLink latency only.  NCCL is resolved at run time (dlopen of
// libnccl.so.2: the copy already loaded by the host application -- e.g. torch's bundled one -- or the system one), so
// libbpg has no link-time dependency on it and single-GPU users never load it.
#include <dlfcn.h>
#include <nccl.h>
namespace {
struct nccl_api {
    void *h = nullptr;
    decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
    decltype(&ncclCommInitRank) CommInitRank = nullptr;
    decltype(&ncclAllGather) AllGather = nullptr;
    decltype(&ncclCommDestroy) CommDestroy = nullptr;
    decltype(&ncclGetErrorString) GetErrorString = nullptr;
    bool ok = false;
};
nccl_api &nccl() {
    static nccl_api a;
    static std::once_flag once;
    std::call_once(once, [] {
        const char *names[] = {getenv("BPG_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
        for (const char *nm : names) {
            if (!nm) continue;
            a.h = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
            if (a.h) break;
        }
        if (!a.h) return;
        a.GetUniqueId = (decltype(a.GetUniqueId))dlsym(a.h, "ncclGetUniqueId");
        a.CommInitRank = (decltype(a.CommInitRank))dlsym(a.h, "ncclCommInitRank");
        a.AllGather = (decltype(a.AllGather))dlsym(a.h, "ncclAllGather");
        a.CommDestroy = (decltype(a.CommDestroy))dlsym(a.h, "ncclCommDestroy");
        a.GetErrorString = (decltype(a.GetErrorString))dlsym(a.h, "ncclGetErrorString");
        a.ok = a.GetUniqueId && a.CommInitRank && a.AllGather && a.CommDestroy;
    });
    return a;
}
} // namespace
extern "C" int bpg_comm_unique_id(uint8_t out128[128]) {
    if (!out128) return BPG_E_ARG;
    if (!nccl().ok) return BPG_E_COMM;
    ncclUniqueId id;
    if (nccl().GetUniqueId(&id) != ncclSuccess) return BPG_E_COMM;
    static_assert(sizeof id == 128, "ncclUniqueId is 128 bytes");
    memcpy(out128, &id, 128);
    return BPG_OK;
}
extern "C" int bpg_comm_destroy(bpg_ctx *ctx) {
    if (!ctx) return BPG_E_ARG;
    if (ctx->comm) {
        cudaSetDevice(ctx->device);
        cudaStreamSynchronize(ctx->stream);
        nccl().CommDestroy((ncclComm_t)ctx->comm);
        ctx->comm = nullptr;
        ctx->shard_rank = 0; ctx->shard_world = 1; ctx->shard_cap = 0;
    }
    return BPG_OK;
}
// collective: every rank of the group calls it with the id rank 0 obtained from bpg_comm_unique_id
extern "C" int bpg_comm_init(bpg_ctx *ctx, int rank, int world, const uint8_t id128[128]) {
    if (!ctx || !id128 || world < 1 || rank < 0 || rank >= world) return BPG_E_ARG;
    if (!nccl().ok) { ctx->last_error = "libnccl.so.2 not found (set BPG_NCCL_LIB)"; return BPG_E_COMM; }
    CUDA_TRY(cudaSetDevice(ctx->device));
    bpg_comm_destroy(ctx);
    ncclUniqueId id;
    memcpy(&id, id128, 128);
    ncclComm_t c = nullptr;
    ncclResult_t r = nccl().CommInitRank(&c, world, id, rank);
    if (r != ncclSuccess) { ctx->last_error = std::string("ncclCommInitRank: ") + (nccl().GetErrorString ? nccl().GetErrorString(r) : "error"); return BPG_E_COMM; }
    ctx->comm = c;
    ctx->shard_rank = rank; ctx->shard_world = world;
    ctx->shard_send = nullptr; ctx->shard_recv = nullptr; ctx->shard_fn = nullptr; ctx->shard_user = nullptr;
    ctx->shard_cap = (size_t)1 << 40; // exchange buffers are the library's own and grow on demand
    return BPG_OK;
}

extern "C" int bpg_ctx_set_shard(bpg_ctx *ctx, int rank, int world, void *d_send, void *d_recv, size_t send_cap, bpg_allgather_fn allgather, void *user) {
    if (!ctx || world < 1 || rank < 0 || rank >= world) return BPG_E_ARG;
    if (world > 1 && (!d_send || !d_recv || !allgather || send_cap < (256u << 10))) return BPG_E_ARG;
    if (ctx->comm) bpg_comm_destroy(ctx);
    for (int i = 0; i < 2; i++) { prefetch_slot_free(ctx->pre[i]); ctx->pre[i] = nullptr; }
    ctx->shard_rank = rank; ctx->shard_world = world;
    ctx->shard_send = d_send; ctx->shard_recv = d_recv; ctx->shard_cap = send_cap;
    ctx->shard_fn = allgather; ctx->shard_user = user;
    return BPG_OK;
}
// contiguous slice [lo, hi) of n items owned by `rank` (same rule as parallel.shard_range)
static inline void shard_slice(uint32_t n, int rank, int world, uint32_t &lo, uint32_t &hi) {
    uint32_t base = n / (uint32_t)world, rem = n % (uint32_t)world, r = (uint32_t)rank;
    lo = r * base + (r < rem ? r : rem);
    hi = lo + base + (r < rem ? 1u : 0u);
}
// K partial points of this rank (d_pts, on stream s) -> all-gather -> d_pts[k] = sum over ranks
static int shard_exchange_sum(bpg_ctx *ctx, cudaStream_t s, ge *d_pts, uint32_t K) {
    size_t bytes = (size_t)K * sizeof(ge);
    if (bytes > ctx->shard_cap) return BPG_E_SIZE;
    if (ctx->comm) { // stream-ordered: partials -> all-gather over NVLink -> sum, nothing waits on the host
        CTX_TRY(ctx->comm_recv.ensure(bytes * (size_t)ctx->shard_world));
        ncclResult_t r = nccl().AllGather(d_pts, ctx->comm_recv.p, bytes, ncclUint8, (ncclComm_t)ctx->comm, s);
        if (r != ncclSuccess) { ctx->last_error = std::string("ncclAllGather: ") + (nccl().GetErrorString ? nccl().GetErrorString(r) : "error"); return BPG_E_COMM; }
        ctx->launches++;
        k_sum_ranks<<<LAUNCH_1D(K, 64), 0, s>>>((const ge *)ctx->comm_recv.p, K, (uint32_t)ctx->shard_world, d_pts);
        KCHECK();
        return BPG_OK;
    }
    CUDA_TRY(cudaMemcpyAsync(ctx->shard_send, d_pts, bytes, cudaMemcpyDeviceToDevice, s));
    SYNC_TRY(ctx, s);
    if (ctx->shard_fn(ctx->shard_user, bytes) != 0) { ctx->last_error = "all-gather callback failed"; return BPG_E_ARG; }
    k_sum_ranks<<<LAUNCH_1D(K, 64), 0, s>>>((const ge *)ctx->shard_recv, K, (uint32_t)ctx->shard_world, d_pts);
    KCHECK();
    return BPG_OK;
}

int msm_run(bpg_ctx *ctx, cudaStream_t s, msm_plan *plan_in, ge *d_out) {
    msm_plan sliced;
    msm_plan *plan = plan_in;
    const bool sharded = plan_in->shard && ctx->shard_world > 1;
    if (sharded) {
        // every vector segment is cut by point range; single terms (blinding / Q scalars) stay with rank 0
        sliced = *plan_in;
        sliced.nseg = 0;
        for (int i = 0; i < plan_in->nseg; i++) {
            msm_seg g = plan_in->seg[i];
            if (g.n == 1) { if (ctx->shard_rank != 0) continue; }
            else {
                uint32_t lo, hi;
                shard_slice(g.n, ctx->shard_rank, ctx->shard_world, lo, hi);
                if (hi == lo) continue;
                g.scalars += lo; g.p0 += lo; g.j0 += lo; g.n = hi - lo;
            }
            sliced.seg[sliced.nseg++] = g;
        }
        plan = &sliced;
    }
    CTX_TRY(msm_run_local(ctx, s, plan, d_out));
    if (sharded) CTX_TRY(shard_exchange_sum(ctx, s, d_out, (uint32_t)plan->ngroups));
    return BPG_OK;
}

// Late fold (see kernels_msm.cuh): G^(k)_i, H^(k)_i for i < n' from the per-generator factors EG, EH (length N), then the
// 16-window affine-Niels tables of those 2 n' points (+ B) in ctx->mat_tab with 2 n' + 2 points per window.
int msm_materialise_fold(bpg_ctx *ctx, cudaStream_t s, uint32_t N, uint32_t nprime, const sc *d_EG, const sc *d_EH, int lean, int shard) {
    uint32_t nout = 2 * nprime;
    uint32_t nb = 2 * nout * BPG_MAT_NB;
    uint32_t pt_small = nout + 2;
    CTX_TRY(ctx->mat_pts.ensure((size_t)nout * sizeof(ge)));
    CTX_TRY(ctx->mat_ext.ensure((size_t)BPG_NWIN * nout * sizeof(ge)));
    CTX_TRY(ctx->mat_tab.ensure((size_t)BPG_NWIN * pt_small * sizeof(ge_an)));
    uint32_t cap = (uint32_t)ctx->cap, ptotal = ctx->ptotal;
    const bool sharded = shard && ctx->shard_world > 1;
    uint32_t p0 = 0, p1 = N; // this rank's point range of BOTH vectors (the per-segment slices of the round MSMs)
    if (sharded) shard_slice(N, ctx->shard_rank, ctx->shard_world, p0, p1);
    uint32_t nt = 2 * (p1 - p0);
    CTX_TRY(msm_bucketize(ctx, s, nb, (size_t)nt * BPG_NWIN * 2, nt != 0, ctx->tab, lean, [&](int scatter, uint32_t *cc, uint32_t *sorted) {
        // one block per output, no global atomics (BPG_MAT_BLOCK=0 keeps the term-parallel kernels for A/B runs)
        static const int mat_block = [] { const char *e = getenv("BPG_MAT_BLOCK"); return e ? atoi(e) : 1; }();
        if (mat_block) {
            if (scatter) k_mat_block<1><<<nout, 256, 0, s>>>(p0, p1, nprime, cap, ptotal, d_EG, d_EH, nullptr, (const uint32_t *)ctx->offsets.p, sorted);
            else k_mat_block<0><<<nout, 256, 0, s>>>(p0, p1, nprime, cap, ptotal, d_EG, d_EH, cc, nullptr, nullptr);
        }
        else if (scatter) k_mat_digits<1><<<LAUNCH_1D(nt, 256), 0, s>>>(N, nprime, cap, ptotal, d_EG, d_EH, p0, p1, cc, sorted);
        else k_mat_digits<0><<<LAUNCH_1D(nt, 256), 0, s>>>(N, nprime, cap, ptotal, d_EG, d_EH, p0, p1, cc, sorted);
    }));
    k_mat_reduce<<<nout, 32, 0, s>>>((const ge *)ctx->buckets.p, nout, (ge *)ctx->mat_pts.p);
    KCHECK();
    if (sharded) CTX_TRY(shard_exchange_sum(ctx, s, (ge *)ctx->mat_pts.p, nout));
    k_mat_chain<<<LAUNCH_1D(nout, 64), 0, s>>>((const ge *)ctx->mat_pts.p, nout, (ge *)ctx->mat_ext.p);
    KCHECK();
    k_mat_affine<<<LAUNCH_1D(nout + BPG_NWIN, 64), 0, s>>>((const ge *)ctx->mat_ext.p, nout, pt_small, (ge_an *)ctx->mat_tab.p, ctx->tab, ptotal,
                                                                      2 * cap);
    KCHECK();
    return BPG_OK;
}

// ================================================================ Pedersen / MSM entry points
extern "C" int bpg_pedersen_commit(bpg_ctx *ctx, const uint8_t *v, const uint8_t *r, size_t n, uint8_t *out32) {
    if (!ctx || (n && (!v || !r || !out32))) return BPG_E_ARG;
    if (!ctx->cap) CTX_TRY(bpg_gens_ensure(ctx, 64));
    if (!n) return BPG_OK;
    CUDA_TRY(cudaSetDevice(ctx->device));
    CTX_TRY(ctx->scratch[0].ensure(96 * n));
    uint8_t *d = (uint8_t *)ctx->scratch[0].p;
    CUDA_TRY(cudaMemcpyAsync(d, v, 32 * n, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(d + 32 * n, r, 32 * n, cudaMemcpyHostToDevice, ctx->stream));
    if (n <= 512) // few commitments: one warp each (latency); many: one thread each (throughput)
        k_pedersen_warp<<<(unsigned)n, 32, 0, ctx->stream>>>((const sc *)d, (const sc *)(d + 32 * n), (uint32_t)n, ctx->comb, d + 64 * n, nullptr);
    else
        k_pedersen_kernel<<<LAUNCH_1D(n, 128), 0, ctx->stream>>>((const sc *)d, (const sc *)(d + 32 * n), (uint32_t)n, ctx->comb, d + 64 * n, nullptr);
    KCHECK();
    D2H_TRY(ctx, out32, d + 64 * n, 32 * n, ctx->stream);
    SYNC_TRY(ctx, ctx->stream);
    return BPG_OK;
}

// variable-base part -> d_out (1 point).  Few terms (the 13 + 2 lg N + m points of a proof): decompress + one windowed scalar
// multiplication per thread + tree sum (latency of ONE scalar multiplication).  Many terms (bpg_msm, circuits with thousands
// of commitments, batch verification): decompress to affine Niels + the bucket engine over the points themselves.
#define BPG_VARBASE_BUCKET_TERMS 8192
static int varbase_msm_dev(bpg_ctx *ctx, cudaStream_t s, const uint8_t *d_scalars, const uint8_t *d_points32, size_t k, ge *d_out, uint32_t *d_ok,
                           dev_buf &pts_buf, dev_buf &blk_buf) {
    if (k >= BPG_VARBASE_BUCKET_TERMS) {
        CTX_TRY(pts_buf.ensure((k + 1) * sizeof(ge_an)));
        ge_an *pts = (ge_an *)pts_buf.p;
        k_decompress_an_kernel<<<LAUNCH_1D(k, 128), 0, s>>>(d_points32, (uint32_t)k, pts, d_ok);
        KCHECK();
        msm_plan plan;
        memset(&plan, 0, sizeof plan);
        plan.ngroups = 1; plan.varbase = 1; plan.tab = pts; plan.ptotal = (uint32_t)k; plan.lean = bpg_lean_now();
        msm_seg &g = plan.seg[plan.nseg++];
        g.scalars = (const sc *)d_scalars; g.n = (uint32_t)k; g.p0 = 0; g.group = 0; g.reduce = 1;
        return msm_run(ctx, s, &plan, d_out);
    }
    CTX_TRY(pts_buf.ensure((k + 1) * sizeof(ge)));
    size_t nb = (k + 63) / 64;
    CTX_TRY(blk_buf.ensure(2 * (nb + 64) * sizeof(ge)));
    ge *pts = (ge *)pts_buf.p, *blk = (ge *)blk_buf.p;
    k_decompress_kernel<<<LAUNCH_1D(k, 128), 0, s>>>(d_points32, (uint32_t)k, pts, d_ok);
    KCHECK();
    k_varbase_kernel<<<(unsigned)nb, 64, 0, s>>>((const sc *)d_scalars, pts, (uint32_t)k, blk);
    KCHECK();
    return run_points_sum(ctx, s, blk, nb, blk + nb + 32, d_out);
}

static int msm_gens_impl(bpg_ctx *ctx, const void *d_sG, const void *d_sH, const uint8_t *h_sG, const uint8_t *h_sH, size_t n, size_t offset,
                         const uint8_t *extra_scalars, const uint8_t *extra_points32, size_t k, uint8_t *out32, uint8_t *out128, void *d_out128 = nullptr,
                         bool exchange = false) {
    if (!ctx) return BPG_E_ARG;
    if (k && (!extra_scalars || !extra_points32)) return BPG_E_ARG;
    CUDA_TRY(cudaSetDevice(ctx->device));
    if (offset + n > ctx->cap) return BPG_E_SIZE;
    if (!ctx->cap) CTX_TRY(bpg_gens_ensure(ctx, 64));
    cudaStream_t s = ctx->stream;
    // stage host inputs
    size_t nG = (d_sG || h_sG) ? n : 0, nH = (d_sH || h_sH) ? n : 0;
    size_t hbytes = 32 * ((h_sG ? n : 0) + (h_sH ? n : 0)) + 64 * k;
    CTX_TRY(ctx->scratch[2].ensure(hbytes + 64));
    uint8_t *d = (uint8_t *)ctx->scratch[2].p;
    size_t off = 0;
    if (h_sG) { CUDA_TRY(cudaMemcpyAsync(d + off, h_sG, 32 * n, cudaMemcpyHostToDevice, s)); d_sG = d + off; off += 32 * n; }
    if (h_sH) { CUDA_TRY(cudaMemcpyAsync(d + off, h_sH, 32 * n, cudaMemcpyHostToDevice, s)); d_sH = d + off; off += 32 * n; }
    const uint8_t *d_es = nullptr, *d_ep = nullptr;
    if (k) {
        CUDA_TRY(cudaMemcpyAsync(d + off, extra_scalars, 32 * k, cudaMemcpyHostToDevice, s)); d_es = d + off; off += 32 * k;
        CUDA_TRY(cudaMemcpyAsync(d + off, extra_points32, 32 * k, cudaMemcpyHostToDevice, s)); d_ep = d + off; off += 32 * k;
    }
    CTX_TRY(ctx->results.ensure(8 * sizeof(ge) + 64));
    ge *res = (ge *)ctx->results.p;
    uint32_t *d_ok = (uint32_t *)(res + 8);
    uint32_t one = 1;
    CUDA_TRY(cudaMemcpyAsync(d_ok, &one, 4, cudaMemcpyHostToDevice, s));
    msm_plan plan;
    memset(&plan, 0, sizeof plan);
    plan.ngroups = 1;
    bool host_scalars = h_sG || h_sH;
    if (nG) { msm_seg &g = plan.seg[plan.nseg++]; g.scalars = (const sc *)d_sG; g.n = (uint32_t)n; g.p0 = (uint32_t)offset; g.group = 0; g.reduce = host_scalars || true; }
    if (nH) { msm_seg &g = plan.seg[plan.nseg++]; g.scalars = (const sc *)d_sH; g.n = (uint32_t)n; g.p0 = (uint32_t)(ctx->cap + offset); g.group = 0; g.reduce = host_scalars || true; }
    CTX_TRY(msm_run(ctx, s, &plan, res));
    if (exchange && ctx->shard_world > 1) CTX_TRY(shard_exchange_sum(ctx, s, res, 1)); // this rank's slice -> sum over the ranks
    size_t npts = 1;
    if (k) {
        CTX_TRY(varbase_msm_dev(ctx, s, d_es, d_ep, k, res + 1, d_ok, ctx->scratch[3], ctx->scratch[4]));
        npts = 2;
    }
    if (npts == 2) { k_points_sum_kernel<<<1, 64, 0, s>>>(res, 2, res + 2); KCHECK(); }
    ge *final_pt = npts == 2 ? res + 2 : res;
    uint32_t ok = 1;
    if (out32) {
        uint8_t *d32 = (uint8_t *)(res + 4);
        CTX_TRY(run_compress(ctx, s, final_pt, 1, d32));
        D2H_TRY(ctx, out32, d32, 32, s);
    }
    if (out128) D2H_TRY(ctx, out128, final_pt, 128, s);
    if (d_out128) CUDA_TRY(cudaMemcpyAsync(d_out128, final_pt, 128, cudaMemcpyDeviceToDevice, s));
    D2H_TRY(ctx, &ok, d_ok, 4, s);
    SYNC_TRY(ctx, s);
    return ok ? BPG_OK : BPG_E_DECOMPRESS;
}
extern "C" int bpg_msm_gens(bpg_ctx *ctx, const uint8_t *sG, const uint8_t *sH, size_t n, size_t offset, const uint8_t *extra_scalars,
                            const uint8_t *extra_points32, size_t k, uint8_t out32[32]) {
    if (!out32) return BPG_E_ARG;
    return msm_gens_impl(ctx, nullptr, nullptr, sG, sH, n, offset, extra_scalars, extra_points32, k, out32, nullptr);
}
extern "C" int bpg_msm_gens_dev(bpg_ctx *ctx, const void *d_sG, const void *d_sH, size_t n, size_t offset, uint8_t out32[32]) {
    if (!out32) return BPG_E_ARG;
    return msm_gens_impl(ctx, d_sG, d_sH, nullptr, nullptr, n, offset, nullptr, nullptr, 0, out32, nullptr);
}
extern "C" int bpg_msm_gens_partial_dev(bpg_ctx *ctx, const void *d_sG, const void *d_sH, size_t n, size_t offset, uint8_t out128[128]) {
    if (!out128) return BPG_E_ARG;
    return msm_gens_impl(ctx, d_sG, d_sH, nullptr, nullptr, n, offset, nullptr, nullptr, 0, nullptr, out128);
}
extern "C" int bpg_msm_gens_partial_to_dev(bpg_ctx *ctx, const void *d_sG, const void *d_sH, size_t n, size_t offset, void *d_out128) {
    if (!d_out128) return BPG_E_ARG;
    return msm_gens_impl(ctx, d_sG, d_sH, nullptr, nullptr, n, offset, nullptr, nullptr, 0, nullptr, nullptr, d_out128);
}
extern "C" int bpg_msm_gens_sharded_dev(bpg_ctx *ctx, const void *d_sG, const void *d_sH, size_t n_local, size_t offset, uint8_t out32[32]) {
    if (!ctx || !out32) return BPG_E_ARG;
    if (ctx->shard_world > 1 && !ctx->comm) return BPG_E_ARG; // needs bpg_comm_init
    return msm_gens_impl(ctx, d_sG, d_sH, nullptr, nullptr, n_local, offset, nullptr, nullptr, 0, out32, nullptr, nullptr, /*exchange=*/true);
}
extern "C" int bpg_points_sum_compress_dev(bpg_ctx *ctx, const void *d_ext128, size_t n, uint8_t out32[32]) {
    if (!ctx || !d_ext128 || !out32 || n == 0 || n > 64) return BPG_E_ARG;
    CUDA_TRY(cudaSetDevice(ctx->device));
    CTX_TRY(ctx->results.ensure(8 * sizeof(ge) + 64));
    ge *res = (ge *)ctx->results.p;
    k_points_sum_kernel<<<1, 64, 0, ctx->stream>>>((const ge *)d_ext128, (uint32_t)n, res);
    KCHECK();
    CTX_TRY(run_compress(ctx, ctx->stream, res, 1, (uint8_t *)(res + 4)));
    D2H_TRY(ctx, out32, res + 4, 32, ctx->stream);
    SYNC_TRY(ctx, ctx->stream);
    return BPG_OK;
}
extern "C" int bpg_points_sum_compress(bpg_ctx *ctx, const uint8_t *ext128, size_t n, uint8_t out32[32]) {
    if (!ctx || !ext128 || !out32 || n == 0 || n > 64) return BPG_E_ARG;
    CUDA_TRY(cudaSetDevice(ctx->device));
    CTX_TRY(ctx->results.ensure(8 * sizeof(ge) + 64));
    CTX_TRY(ctx->scratch[3].ensure(64 * sizeof(ge)));
    ge *pts = (ge *)ctx->scratch[3].p, *res = (ge *)ctx->results.p;
    CUDA_TRY(cudaMemcpyAsync(pts, ext128, 128 * n, cudaMemcpyHostToDevice, ctx->stream));
    k_points_sum_kernel<<<1, 64, 0, ctx->stream>>>(pts, (uint32_t)n, res);
    KCHECK();
    CTX_TRY(run_compress(ctx, ctx->stream, res, 1, (uint8_t *)(res + 4)));
    D2H_TRY(ctx, out32, res + 4, 32, ctx->stream);
    SYNC_TRY(ctx, ctx->stream);
    return BPG_OK;
}
extern "C" int bpg_msm(bpg_ctx *ctx, const uint8_t *scalars, const uint8_t *points32, size_t n, uint8_t out32[32]) {
    if (!ctx || !out32 || (n && (!scalars || !points32))) return BPG_E_ARG;
    if (n == 0) { memset(out32, 0, 32); return BPG_OK; }
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    CTX_TRY(ctx->scratch[2].ensure(64 * n));
    uint8_t *d = (uint8_t *)ctx->scratch[2].p;
    CUDA_TRY(cudaMemcpyAsync(d, scalars, 32 * n, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(d + 32 * n, points32, 32 * n, cudaMemcpyHostToDevice, s));
    CTX_TRY(ctx->results.ensure(8 * sizeof(ge) + 64));
    ge *res = (ge *)ctx->results.p;
    uint32_t *d_ok = (uint32_t *)(res + 8);
    uint32_t one = 1, ok = 1;
    CUDA_TRY(cudaMemcpyAsync(d_ok, &one, 4, cudaMemcpyHostToDevice, s));
    CTX_TRY(varbase_msm_dev(ctx, s, d, d + 32 * n, n, res, d_ok, ctx->scratch[3], ctx->scratch[4]));
    CTX_TRY(run_compress(ctx, s, res, 1, (uint8_t *)(res + 4)));
    D2H_TRY(ctx, out32, res + 4, 32, s);
    D2H_TRY(ctx, &ok, d_ok, 4, s);
    SYNC_TRY(ctx, s);
    return ok ? BPG_OK : BPG_E_DECOMPRESS;
}
extern "C" int bpg_fold_points(bpg_ctx *ctx, const uint8_t sl[32], const uint8_t sr[32], const uint8_t *PL32, const uint8_t *PR32, size_t n, uint8_t *out32) {
    if (!ctx || !sl || !sr || (n && (!PL32 || !PR32 || !out32))) return BPG_E_ARG;
    if (!n) return BPG_OK;
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    CTX_TRY(ctx->scratch[2].ensure(96 * n + 128));
    CTX_TRY(ctx->scratch[3].ensure(3 * n * sizeof(ge)));
    uint8_t *d = (uint8_t *)ctx->scratch[2].p;
    ge *pts = (ge *)ctx->scratch[3].p;
    CUDA_TRY(cudaMemcpyAsync(d, sl, 32, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(d + 32, sr, 32, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(d + 64, PL32, 32 * n, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(d + 64 + 32 * n, PR32, 32 * n, cudaMemcpyHostToDevice, s));
    CTX_TRY(ctx->results.ensure(8 * sizeof(ge) + 64));
    uint32_t *d_ok = (uint32_t *)((ge *)ctx->results.p + 8);
    uint32_t one = 1, ok = 1;
    CUDA_TRY(cudaMemcpyAsync(d_ok, &one, 4, cudaMemcpyHostToDevice, s));
    k_decompress_kernel<<<LAUNCH_1D(2 * n, 128), 0, s>>>(d + 64, (uint32_t)(2 * n), pts, d_ok);
    KCHECK();
    for (int e = 12; e < 14; e++) if (!ctx->tev[e]) CUDA_TRY(cudaEventCreate(&ctx->tev[e]));
    CUDA_TRY(cudaEventRecord(ctx->tev[12], s)); // event slots 12 / 13 bracket the fold kernel (bpg_event_elapsed_ms)
    k_fold_kernel<<<LAUNCH_1D(n, 64), 0, s>>>((const sc *)d, (const sc *)(d + 32), pts, pts + n, (uint32_t)n, pts + 2 * n);
    KCHECK();
    CUDA_TRY(cudaEventRecord(ctx->tev[13], s));
    CTX_TRY(run_compress(ctx, s, pts + 2 * n, n, d + 64));
    D2H_TRY(ctx, out32, d + 64, 32 * n, s);
    D2H_TRY(ctx, &ok, d_ok, 4, s);
    SYNC_TRY(ctx, s);
    return ok ? BPG_OK : BPG_E_DECOMPRESS;
}

extern "C" int bpg_event_record(bpg_ctx *ctx, int slot) {
    if (!ctx || slot < 0 || slot >= 16) return BPG_E_ARG;
    CUDA_TRY(cudaSetDevice(ctx->device));
    if (!ctx->tev[slot]) CUDA_TRY(cudaEventCreate(&ctx->tev[slot]));
    CUDA_TRY(cudaEventRecord(ctx->tev[slot], ctx->stream));
    return BPG_OK;
}
extern "C" int bpg_event_elapsed_ms(bpg_ctx *ctx, int a, int b, float *ms) {
    if (!ctx || !ms || a < 0 || b < 0 || a >= 16 || b >= 16 || !ctx->tev[a] || !ctx->tev[b]) return BPG_E_ARG;
    CUDA_TRY(cudaEventSynchronize(ctx->tev[b]));
    CUDA_TRY(cudaEventElapsedTime(ms, ctx->tev[a], ctx->tev[b]));
    return BPG_OK;
}
extern "C" int bpg_prof_enable(bpg_ctx *ctx, int on) {
    if (!ctx) return BPG_E_ARG;
    CUDA_TRY(cudaSetDevice(ctx->device));
    SYNC_TRY(ctx, ctx->stream);
    if (on && !ctx->prof_pairs) CUDA_TRY(cudaMallocHost((void **)&ctx->prof_pairs, 4096 * 4));
    if (!on) { // profiling off: release the events right away (after the sync above)
        for (cudaEvent_t e : ctx->prof_ev) cudaEventDestroy(e);
        ctx->prof_ev.clear();
        ctx->prof_n = 0;
    }
    // all events are created here, never in the launch path (event creation takes the context lock and was measured to
    // slow concurrent provers by a third when done lazily inside the timed region)
    while (on && ctx->prof_ev.size() < 2 * 64) { cudaEvent_t e; CUDA_TRY(cudaEventCreate(&e)); ctx->prof_ev.push_back(e); }
    ctx->prof_on = on;
    if (on) ctx->prof_n = 0;
    return BPG_OK;
}
extern "C" int bpg_prof_read(bpg_ctx *ctx, uint64_t *launches, double *ms_total, uint64_t *pairs_total) {
    if (!ctx || !launches || !ms_total || !pairs_total) return BPG_E_ARG;
    SYNC_TRY(ctx, ctx->stream);
    double ms = 0; uint64_t pairs = 0;
    for (size_t i = 0; i < ctx->prof_n; i++) {
        float t = 0;
        CUDA_TRY(cudaEventElapsedTime(&t, ctx->prof_ev[2 * i], ctx->prof_ev[2 * i + 1]));
        ms += t; pairs += ctx->prof_pairs[i];
    }
    *launches = ctx->prof_n; *ms_total = ms; *pairs_total = pairs;
    return BPG_OK;
}

extern "C" long bpg_prof_read_launches(bpg_ctx *ctx, float *ms, uint32_t *pairs, size_t cap) {
    if (!ctx || !ms || !pairs) return BPG_E_ARG;
    SYNC_TRY(ctx, ctx->stream);
    size_t n = ctx->prof_n < cap ? ctx->prof_n : cap;
    for (size_t i = 0; i < n; i++) {
        CUDA_TRY(cudaEventElapsedTime(&ms[i], ctx->prof_ev[2 * i], ctx->prof_ev[2 * i + 1]));
        pairs[i] = ctx->prof_pairs[i];
    }
    return (long)n;
}

extern "C" int bpg_bench_imad(bpg_ctx *ctx, int iters, float *ms, double *mac32) {
    if (!ctx || !ms || !mac32) return BPG_E_ARG;
    CUDA_TRY(cudaSetDevice(ctx->device));
    int sms = 0;
    CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device));
    int blocks = sms * 8, threads = 256;
    CTX_TRY(ctx->scratch[5].ensure((size_t)blocks * threads * 4));
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0)); CUDA_TRY(cudaEventCreate(&e1));
    k_bench_fe_mul<<<blocks, threads, 0, ctx->stream>>>((uint32_t *)ctx->scratch[5].p, 8); // warm-up
    KCHECK();
    CUDA_TRY(cudaEventRecord(e0, ctx->stream));
    k_bench_fe_mul<<<blocks, threads, 0, ctx->stream>>>((uint32_t *)ctx->scratch[5].p, iters);
    KCHECK();
    CUDA_TRY(cudaEventRecord(e1, ctx->stream));
    CUDA_TRY(cudaEventSynchronize(e1));
    CUDA_TRY(cudaEventElapsedTime(ms, e0, e1));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    *mac32 = (double)blocks * threads * (double)iters * 2.0 * 72.0; // 64 limb products + 8 fold-by-38 per field multiply
    return BPG_OK;
}

extern "C" int bpg_bench_latency(bpg_ctx *ctx, int iters, double cycles_per_op[8]) {
    if (!ctx || !cycles_per_op || iters <= 0) return BPG_E_ARG;
    CUDA_TRY(cudaSetDevice(ctx->device));
    CTX_TRY(ctx->scratch[5].ensure(256));
    unsigned long long *d = (unsigned long long *)ctx->scratch[5].p;
    for (int mode = 0; mode < 8; mode++) {
        k_bench_latency<<<1, 32, 0, ctx->stream>>>(mode, iters, d, (uint32_t *)(d + 16));
        KCHECK();
    }
    unsigned long long h[8];
    D2H_TRY(ctx, h, d, sizeof h, ctx->stream);
    SYNC_TRY(ctx, ctx->stream);
    for (int i = 0; i < 8; i++) cycles_per_op[i] = (double)h[i] / iters;
    return BPG_OK;
}

// ================================================================ Merlin transcript (host)
struct bpg_transcript { bpgh::Transcript t; };
extern "C" bpg_transcript *bpg_transcript_new(const uint8_t *label, size_t len) { bpg_transcript *t = new bpg_transcript(); t->t = bpgh::Transcript(label, len); return t; }
extern "C" void bpg_transcript_free(bpg_transcript *t) { delete t; }
extern "C" void bpg_transcript_append(bpg_transcript *t, const uint8_t *label, size_t ll, const uint8_t *msg, size_t ml) { t->t.append_raw(label, ll, msg, ml); }
extern "C" void bpg_transcript_challenge(bpg_transcript *t, const uint8_t *label, size_t ll, uint8_t *out, size_t n) { t->t.challenge_raw(label, ll, out, n); }

// host-only: `count` 64-byte draws of TranscriptRng(Transcript(label)).finalize(ext32) after `warm` scalar draws,
// through the lane-batched service (use_service = 1) or the scalar definition (0).  Needs no device (CPU tests).
extern "C" int bpg_host_rng_lanes(void) { return bpgh::RngService::get().lanes(); }
extern "C" int bpg_host_rng_draw64(const uint8_t *label, size_t label_len, const uint8_t ext32[32], size_t warm, size_t count, int use_service,
                                   uint8_t *out) {
    if (!label || !ext32 || (count && !out)) return BPG_E_ARG;
    bpgh::Transcript t(label, label_len);
    bpgh::TranscriptRng rng(t);
    rng.finalize(ext32);
    uint8_t tmp[64];
    for (size_t i = 0; i < warm; i++) rng.fill_bytes(tmp, 64);
    if (use_service) bpgh::RngService::get().draw64(rng, out, count);
    else for (size_t i = 0; i < count; i++) rng.fill_bytes(out + 64 * i, 64);
    rng.fill_bytes(out + 64 * count, 64); // one more scalar draw: proves that the stream state was handed back intact
    return BPG_OK;
}

#include "prover.inl"
#include "prover_batch.inl"
