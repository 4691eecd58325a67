// kb_core.cu -- context lifecycle, buffer pools, profiling hooks, store ingest (kb_load_sorted) and the
// NCCL revision-cursor exchange of libkbb200.so.
#include <dlfcn.h>
#include <stdarg.h>

#include <algorithm>

#include "kb_internal.cuh"
#include "kb_decode.cuh"

// ------------------------------------------------------------------------------------------------
// errors / buffers
// ------------------------------------------------------------------------------------------------
int kb_fail(kb_ctx *ctx, int code, const char *fmt, ...)
{
    if (ctx) {
        char buf[512];
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(buf, sizeof(buf), fmt, ap);
        va_end(ap);
        ctx->err = buf;
    }
    return code;
}

int kb_cuda_fail(kb_ctx *ctx, cudaError_t e, const char *what)
{
    return kb_fail(ctx, e == cudaErrorMemoryAllocation ? KB_ENOMEM : KB_ECUDA, "CUDA error %d (%s) at %s", (int)e,
                   cudaGetErrorString(e), what);
}

int dbuf_ensure(kb_ctx *ctx, DBuf &b, size_t bytes)
{
    if (bytes <= b.cap && b.p) return KB_OK;
    size_t want = std::max(bytes + bytes / 4, (size_t)4096);
    want = (want + 255) & ~(size_t)255;
    if (b.p) {
        KB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        if (ctx->stream_g) KB_CUDA(ctx, cudaStreamSynchronize(ctx->stream_g));
        cudaFree(b.p);
        b.p = nullptr;
        b.cap = 0;
    }
    KB_CUDA(ctx, cudaMalloc(&b.p, want));
    b.cap = want;
    return KB_OK;
}

int hbuf_ensure(kb_ctx *ctx, HBuf &b, size_t bytes)
{
    if (bytes <= b.cap && b.p) return KB_OK;
    size_t want = std::max(bytes + bytes / 4, (size_t)4096);
    if (b.p) {
        KB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        if (ctx->stream_g) KB_CUDA(ctx, cudaStreamSynchronize(ctx->stream_g));
        cudaFreeHost(b.p);
        b.p = nullptr;
        b.cap = 0;
    }
    KB_CUDA(ctx, cudaHostAlloc(&b.p, want, cudaHostAllocDefault));
    b.cap = want;
    return KB_OK;
}

template <typename B>
static bool pool_take(std::vector<B> &pool, size_t bytes, B *out)
{
    int best = -1;
    for (int i = 0; i < (int)pool.size(); i++)
        if (pool[i].cap >= bytes && (best < 0 || pool[i].cap < pool[best].cap)) best = i;
    if (best < 0) return false;
    *out = pool[best];
    pool.erase(pool.begin() + best);
    return true;
}

int pool_get_dev(kb_ctx *ctx, size_t bytes, DBuf *out)
{
    if (bytes == 0) bytes = 16;
    if (pool_take(ctx->free_dev, bytes, out)) return KB_OK;
    DBuf b;
    KB_TRY(dbuf_ensure(ctx, b, bytes));
    *out = b;
    return KB_OK;
}

int pool_get_host(kb_ctx *ctx, size_t bytes, HBuf *out)
{
    if (bytes == 0) bytes = 16;
    if (pool_take(ctx->free_host, bytes, out)) return KB_OK;
    HBuf b;
    KB_TRY(hbuf_ensure(ctx, b, bytes));
    *out = b;
    return KB_OK;
}

int pool_get_arena(kb_ctx *ctx, size_t bytes, DBuf *out)
{
    if (bytes == 0) bytes = 16;
    if (pool_take(ctx->free_arena, bytes, out)) return KB_OK;
    DBuf b;
    KB_TRY(dbuf_ensure(ctx, b, bytes));
    *out = b;
    return KB_OK;
}

void pool_put_arena(kb_ctx *ctx, DBuf b)
{
    if (!b.p) return;
    if (ctx->free_arena.size() >= 8) {
        cudaFree(b.p);  // implicit device synchronisation: nothing can still be writing it
        return;
    }
    ctx->free_arena.push_back(b);
}

int ctx_quiesce(kb_ctx *ctx)
{
    KB_TRY(kb_pending_harvest_all(ctx));  // submitted range batches: their kernels are done once their rows are back
    if (ctx->stream_g) KB_CUDA(ctx, cudaStreamSynchronize(ctx->stream_g));
    if (ctx->stream2) KB_CUDA(ctx, cudaStreamSynchronize(ctx->stream2));  // a prefetched bound search may still read the slabs
    return KB_OK;
}

void pool_put_dev(kb_ctx *ctx, DBuf b)
{
    if (!b.p) return;
    if (ctx->free_dev.size() >= 16) {
        cudaFree(b.p);
        return;
    }
    ctx->free_dev.push_back(b);
}

void pool_put_host(kb_ctx *ctx, HBuf b)
{
    if (!b.p) return;
    if (ctx->free_host.size() >= 16) {
        cudaFreeHost(b.p);
        return;
    }
    ctx->free_host.push_back(b);
}

// ------------------------------------------------------------------------------------------------
// profiling
// ------------------------------------------------------------------------------------------------
int prof_index(kb_ctx *ctx, const char *name)
{
    for (int i = 0; i < (int)ctx->prof.size(); i++)
        if (ctx->prof[i].name == name) return i;
    ProfEntry e;
    e.name = name;
    ctx->prof.push_back(e);
    return (int)ctx->prof.size() - 1;
}

static cudaEvent_t ev_get(kb_ctx *ctx)
{
    if (!ctx->ev_pool.empty()) {
        cudaEvent_t e = ctx->ev_pool.back();
        ctx->ev_pool.pop_back();
        return e;
    }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}

void prof_begin(kb_ctx *ctx, int idx, uint64_t alg_bytes, cudaStream_t strm)
{
    ProfPending p;
    p.idx = idx;
    p.a = ev_get(ctx);
    p.b = ev_get(ctx);
    cudaEventRecord(p.a, strm);
    ctx->prof_pending.push_back(p);
    ctx->prof[idx].launches++;
    ctx->prof[idx].bytes += alg_bytes;
}

void prof_end(kb_ctx *ctx, cudaStream_t strm) { cudaEventRecord(ctx->prof_pending.back().b, strm); }

static void prof_resolve(kb_ctx *ctx)
{
    if (ctx->prof_pending.empty()) return;
    cudaStreamSynchronize(ctx->stream);
    if (ctx->stream_g) cudaStreamSynchronize(ctx->stream_g);
    for (auto &p : ctx->prof_pending) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess) ctx->prof[p.idx].ms += ms;
        ctx->ev_pool.push_back(p.a);
        ctx->ev_pool.push_back(p.b);
    }
    ctx->prof_pending.clear();
}

extern "C" int kb_prof_enable(kb_ctx *ctx, int on)
{
    if (!ctx) return KB_EINVAL;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (!on) prof_resolve(ctx);
    ctx->prof_on = on;
    return KB_OK;
}

extern "C" int kb_prof_reset(kb_ctx *ctx)
{
    if (!ctx) return KB_EINVAL;
    std::lock_guard<std::mutex> g(ctx->mu);
    prof_resolve(ctx);
    ctx->prof.clear();
    return KB_OK;
}

extern "C" int kb_prof_read(kb_ctx *ctx, kb_prof_entry *entries, int cap, int *n)
{
    if (!ctx || !n) return KB_EINVAL;
    std::lock_guard<std::mutex> g(ctx->mu);
    prof_resolve(ctx);
    int k = 0;
    for (auto &e : ctx->prof) {
        if (k < cap && entries) {
            memset(&entries[k], 0, sizeof(kb_prof_entry));
            strncpy(entries[k].name, e.name.c_str(), sizeof(entries[k].name) - 1);
            entries[k].launches = e.launches;
            entries[k].total_ms = e.ms;
            entries[k].alg_bytes = e.bytes;
        }
        k++;
    }
    *n = k;
    return KB_OK;
}

extern "C" uint64_t kb_launch_count(kb_ctx *ctx) { return ctx ? ctx->launches : 0; }

// ------------------------------------------------------------------------------------------------
// lifecycle
// ------------------------------------------------------------------------------------------------
extern "C" int kb_abi_version(void) { return KB_ABI_VERSION; }

extern "C" int kb_open(int device_ordinal, const kb_config *cfg, kb_ctx **out)
{
    if (!out) return KB_EINVAL;
    const bool high = cfg && cfg->struct_size >= sizeof(kb_config) && (cfg->flags & KB_CFG_HIGH_PRIORITY);
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev <= 0 || device_ordinal < 0 || device_ordinal >= ndev) {
        // no CPU fallback: the product path refuses to run without a CUDA device
        return KB_ECUDA;
    }
    kb_ctx *ctx = new kb_ctx();
    ctx->device = device_ordinal;
    int prio_lo = 0, prio_hi = 0, prio_lane = 0;
    if (cudaSetDevice(device_ordinal) != cudaSuccess ||
        cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi) != cudaSuccess)
        prio_lo = prio_hi = 0;
    // three levels when the device has them (numerically lower = more urgent): bound search > lane streams (short kernels of a
    // batch) > bulk copies (gather / wire copy, by their stream)
    static const bool split = !(getenv("KB_PRIO_SPLIT") && atoi(getenv("KB_PRIO_SPLIT")) == 0);
    prio_lane = (split && prio_lo - prio_hi >= 2) ? prio_lo - 1 : prio_lo;
    if (
        cudaStreamCreateWithPriority(&ctx->stream, cudaStreamNonBlocking, high ? prio_hi : prio_lane) != cudaSuccess ||
        // the bound search is tiny and the host waits for it: always ahead of everything; the copy stream (gather / wire
        // copy) is throughput work that the next batch's short kernels should not queue behind: always behind
        cudaStreamCreateWithPriority(&ctx->stream2, cudaStreamNonBlocking, prio_hi) != cudaSuccess ||
        cudaStreamCreateWithPriority(&ctx->stream_g, cudaStreamNonBlocking, prio_lo) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_jobs, cudaEventDisableTiming) != cudaSuccess ||
        // second lane of range batches (kb_range_submit) and the stream of the device -> host answer copies
        cudaStreamCreateWithPriority(&ctx->stream_h, cudaStreamNonBlocking, prio_lo) != cudaSuccess ||
        // search counters + the error flag: zeroed once, before any stream can touch them
        cudaMalloc(&ctx->d_ctrs.p, 1024) != cudaSuccess || cudaMemset(ctx->d_ctrs.p, 0, 1024) != cudaSuccess ||
        cudaDeviceSynchronize() != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_gather[0], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_gather[1], cudaEventDisableTiming) != cudaSuccess) {
        delete ctx;
        return KB_ECUDA;
    }
    ctx->d_ctrs.cap = 1024;
    // the other lanes of range batches (kb_range_submit): KB_LANES batches in flight at most
    ctx->n_lanes = getenv("KB_LANES") ? std::min(std::max(atoi(getenv("KB_LANES")), 1), KB_MAX_LANES) : 3;
    ctx->prio_lane = high ? prio_hi : prio_lane;
    for (int l = 1; l < ctx->n_lanes; l++)  // their streams are created when a submission first rotates onto them
        ctx->parked[l - 1].id = l;
    *out = ctx;
    return KB_OK;
}

// exchange the current lane's fields with the other lane's (the enqueued work holds raw pointers, not these fields)
void lane_swap(kb_ctx *ctx)
{
    if (ctx->n_lanes < 2) return;
    ScanLane &a = ctx->parked[ctx->park_next];
    if (!a.stream) {  // first use of this lane (a context that never submits ahead -- the watch context -- has one lane)
        if (cudaStreamCreateWithPriority(&a.stream, cudaStreamNonBlocking, ctx->prio_lane) != cudaSuccess ||
            cudaEventCreateWithFlags(&a.ev_jobs, cudaEventDisableTiming) != cudaSuccess) {
            if (a.stream) cudaStreamDestroy(a.stream);
            a.stream = nullptr;
            cudaGetLastError();
            return;  // stay on the current lane: the next submission first reads this lane's rows back
        }
    }
    ctx->park_next = (ctx->park_next + 1) % (ctx->n_lanes - 1);
    std::swap(ctx->stream, a.stream);
    std::swap(ctx->ev_jobs, a.ev_jobs);
    std::swap(ctx->h_rout, a.h_rout);
    std::swap(ctx->h_rout_cap, a.h_rout_cap);
    std::swap(ctx->rout_epoch, a.rout_epoch);
    std::swap(ctx->d_bounds, a.d_bounds);
    std::swap(ctx->d_bres, a.d_bres);
    std::swap(ctx->d_reqs, a.d_reqs);
    std::swap(ctx->d_tiles, a.d_tiles);
    std::swap(ctx->d_tgt, a.d_tgt);
    std::swap(ctx->d_tcnt, a.d_tcnt);
    std::swap(ctx->d_tscan, a.d_tscan);
    std::swap(ctx->d_reqout, a.d_reqout);
    std::swap(ctx->d_sel, a.d_sel);
    std::swap(ctx->d_slot, a.d_slot);
    std::swap(ctx->h_stage, a.h_stage);
    std::swap(ctx->h_stage2, a.h_stage2);
    std::swap(ctx->search_pub, a.search_pub);
    std::swap(ctx->lane, a.id);
}

static void dfree(DBuf &b)
{
    if (b.p) cudaFree(b.p);
    b.p = nullptr;
    b.cap = 0;
}

extern "C" void kb_close(kb_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    kb_pending_drop_all(ctx);
    cudaStreamSynchronize(ctx->stream);
    for (auto &a : ctx->parked)
        if (a.stream) cudaStreamSynchronize(a.stream);
    if (ctx->stream_g) cudaStreamSynchronize(ctx->stream_g);
    if (ctx->stream2) cudaStreamSynchronize(ctx->stream2);
    if (ctx->stream_h) cudaStreamSynchronize(ctx->stream_h);
    watch_tables_free(ctx);
    for (auto &a : ctx->parked) {  // (d_tiles aliases d_reqs)
        DBuf *lane[] = {&a.d_bounds, &a.d_bres, &a.d_reqs, &a.d_tgt, &a.d_tcnt, &a.d_tscan, &a.d_reqout, &a.d_sel, &a.d_slot};
        for (DBuf *b : lane) dfree(*b);
        if (a.h_stage.p) cudaFreeHost(a.h_stage.p);
        if (a.h_stage2.p) cudaFreeHost(a.h_stage2.p);
        if (a.h_rout) cudaFreeHost(a.h_rout);
        if (a.search_pub.host) cudaFreeHost(a.search_pub.host);
        if (a.ev_jobs) cudaEventDestroy(a.ev_jobs);
        if (a.stream) cudaStreamDestroy(a.stream);
    }
    if (ctx->stream_h) cudaStreamDestroy(ctx->stream_h);
    DBuf *all[] = {&ctx->d_kslab, &ctx->d_koff16, &ctx->d_klen, &ctx->d_vslab, &ctx->d_voff16, &ctx->d_vlen, &ctx->d_dir,
                   &ctx->d_crev, &ctx->d_cword, &ctx->d_bounds, &ctx->d_bres, &ctx->d_reqs,
                   &ctx->d_tgt, &ctx->d_agg, &ctx->d_tcnt, &ctx->d_tscan, &ctx->d_reqout,
                   &ctx->d_sel, &ctx->d_slot, &ctx->d_jobs, &ctx->d_gjobs, &ctx->d_jobs2, &ctx->d_gjobs2, &ctx->d_flags, &ctx->d_cursor,
                   &ctx->d_ctrs, &ctx->s_koff16, &ctx->s_klen, &ctx->s_voff16, &ctx->s_vlen, &ctx->s_dir,
                   &ctx->s_crev, &ctx->s_cword};
    for (DBuf *b : all) dfree(*b);
    for (auto &b : ctx->free_dev) cudaFree(b.p);
    for (auto &b : ctx->free_host) cudaFreeHost(b.p);
    if (ctx->h_stage.p) cudaFreeHost(ctx->h_stage.p);
    if (ctx->h_stage2.p) cudaFreeHost(ctx->h_stage2.p);
    for (auto &p : ctx->prof_pending) {
        cudaEventDestroy(p.a);
        cudaEventDestroy(p.b);
    }
    for (auto e : ctx->ev_pool) cudaEventDestroy(e);
    for (size_t r = 0; r < ctx->p2p_peer.size(); r++)
        if (ctx->p2p_peer[r] && ctx->p2p_peer[r] != ctx->p2p_mine) cudaIpcCloseMemHandle(ctx->p2p_peer[r]);
    if (ctx->p2p_mine) cudaFree(ctx->p2p_mine);
    if (ctx->d_p2p_ptrs.p) cudaFree(ctx->d_p2p_ptrs.p);
    if (ctx->h_p2p_out) cudaFreeHost(ctx->h_p2p_out);
    if (ctx->nccl_comm) {
        void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);
        if (h) {
            typedef int (*destroy_t)(void *);
            destroy_t f = (destroy_t)dlsym(h, "ncclCommDestroy");
            if (f) f(ctx->nccl_comm);
        }
    }
    if (ctx->h_rout) cudaFreeHost(ctx->h_rout);
    if (ctx->h_wpub) cudaFreeHost(ctx->h_wpub);
    for (auto &b : ctx->free_arena) cudaFree(b.p);
    for (auto &sl : ctx->prefetch) {
        if (sl.stage.p) cudaFreeHost(sl.stage.p);
        if (sl.d_bounds.p) cudaFree(sl.d_bounds.p);
        if (sl.d_bres.p) cudaFree(sl.d_bres.p);
        if (sl.pub.host) cudaFreeHost(sl.pub.host);
    }
    if (ctx->search_pub.host) cudaFreeHost(ctx->search_pub.host);
    if (ctx->ev_jobs) cudaEventDestroy(ctx->ev_jobs);
    for (int i = 0; i < 2; i++)
        if (ctx->ev_gather[i]) cudaEventDestroy(ctx->ev_gather[i]);
    if (ctx->stream_g) cudaStreamDestroy(ctx->stream_g);
    if (ctx->stream2) cudaStreamDestroy(ctx->stream2);
    cudaStreamDestroy(ctx->stream);
    delete ctx;
}

extern "C" const char *kb_last_error(kb_ctx *ctx) { return ctx ? ctx->err.c_str() : "no context"; }
extern "C" void *kb_stream(kb_ctx *ctx) { return ctx ? (void *)ctx->stream : nullptr; }

extern "C" int kb_sync(kb_ctx *ctx)
{
    if (!ctx) return KB_EINVAL;
    std::lock_guard<std::mutex> g(ctx->mu);
    KB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (auto &a : ctx->parked)
        if (a.stream) KB_CUDA(ctx, cudaStreamSynchronize(a.stream));
    if (ctx->stream_g) KB_CUDA(ctx, cudaStreamSynchronize(ctx->stream_g));
    if (ctx->stream_h) KB_CUDA(ctx, cudaStreamSynchronize(ctx->stream_h));
    if (ctx->stream2) KB_CUDA(ctx, cudaStreamSynchronize(ctx->stream2));  // the delivery lists of the last watch match
    return KB_OK;
}

// ------------------------------------------------------------------------------------------------
// store ingest
// ------------------------------------------------------------------------------------------------
// one warp per record: copy the packed bytes into the 16-byte aligned slab (destination is pre-zeroed)
__global__ void k_repack(const uint8_t *__restrict__ src, const uint64_t *__restrict__ soff, uint8_t *__restrict__ dst,
                         const uint32_t *__restrict__ doff16_32, const uint64_t *__restrict__ doff16_64, uint32_t n)
{
    uint32_t w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    uint32_t nw = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t i = w; i < n; i += nw) {
        uint64_t s = soff[i], e = soff[i + 1];
        uint64_t d = (doff16_32 ? (uint64_t)doff16_32[i] : doff16_64[i]) * 16ull;
        for (uint64_t b = lane; b < e - s; b += 32) dst[d + b] = src[s + b];
    }
}

// thread per record: the decoded columns (kb_decode.cuh) and the strict ascending order of adjacent keys (storage.Iter
// contract) in one pass over the keys; bad = the first record that is not greater than its predecessor
__global__ void __launch_bounds__(256) k_col_build(StoreDev st, uint64_t *__restrict__ crev, uint32_t *__restrict__ cword,
                                                   uint32_t *__restrict__ bad)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= st.n) return;
    uint64_t r;
    uint32_t w;
    bool less;
    col_entry(st, i, &r, &w, &less);
    crev[i] = r;
    cword[i] = w;
    if (!less) atomicMin(bad, i);
}

__global__ void __launch_bounds__(256) k_pack_dir(StoreDev st, uint4 *__restrict__ dir)
{
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= st.n) return;
    const uint64_t vo = st.voff16[r];
    dir[r] = make_uint4(st.koff16[r], (uint32_t)st.klen[r] | ((uint32_t)(vo >> 32) << 16), st.vlen[r], (uint32_t)vo);
}

// the decoded columns of the loaded directory, and its key order (KB_EUNSORTED); waits for the device
static int store_build_columns(kb_ctx *ctx, const char *who)
{
    const uint64_t n = ctx->st.n;
    KB_TRY(dbuf_ensure(ctx, ctx->d_crev, (n + 1) * 8));
    KB_TRY(dbuf_ensure(ctx, ctx->d_cword, (n + 1) * 4));
    KB_TRY(dbuf_ensure(ctx, ctx->d_flags, 64));
    ctx->st.crev = (const uint64_t *)ctx->d_crev.p;
    ctx->st.cword = (const uint32_t *)ctx->d_cword.p;
    uint32_t bad = 0xFFFFFFFFu;
    if (n) {
        KB_CUDA(ctx, cudaMemcpyAsync(ctx->d_flags.p, &bad, 4, cudaMemcpyHostToDevice, ctx->stream));
        const uint64_t mean_key = ctx->key_bytes / n;
        KB_LAUNCH(ctx, "k_col_build", n * (2 * mean_key + 2 * 14 + 16 + 12),  // two keys, two entries, a value probe
                  (k_col_build<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(ctx->st, (uint64_t *)ctx->d_crev.p,
                                                                                    (uint32_t *)ctx->d_cword.p,
                                                                                    (uint32_t *)ctx->d_flags.p)));
        KB_CUDA(ctx, cudaGetLastError());
        KB_CUDA(ctx, cudaMemcpyAsync(&bad, ctx->d_flags.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
    }
    KB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (bad != 0xFFFFFFFFu) return kb_fail(ctx, KB_EUNSORTED, "%srecord %u is not greater than its predecessor", who, bad);
    return KB_OK;
}

int store_pack_dir(kb_ctx *ctx)
{
    const uint64_t n = ctx->st.n;
    // value offsets are 16-byte units: 48 bits cover 4 PiB
    KB_TRY(dbuf_ensure(ctx, ctx->d_dir, (n + 1) * 16));
    ctx->st.dir = (const uint4 *)ctx->d_dir.p;
    if (n) {
        k_pack_dir<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(ctx->st, (uint4 *)ctx->d_dir.p);
        KB_CUDA(ctx, cudaGetLastError());
    }
    return KB_OK;
}

extern "C" int kb_load_sorted(kb_ctx *ctx, const uint8_t *keys, const uint64_t *key_off, const uint8_t *vals,
                              const uint64_t *val_off, uint64_t n)
{
    if (!ctx || (n && (!keys || !key_off || !vals || !val_off))) return KB_EINVAL;
    std::lock_guard<std::mutex> g(ctx->mu);
    cudaSetDevice(ctx->device);
    KB_TRY(ctx_quiesce(ctx));
    if (n >= 0xFFFFFFFEull) return kb_fail(ctx, KB_ELIMIT, "too many records (%llu)", (unsigned long long)n);
    ctx->loaded = false;

    // destination offsets (host): every record padded to a 16-byte multiple
    std::vector<uint32_t> koff16(n + 1);
    std::vector<uint16_t> klen(n ? n : 1);
    std::vector<uint64_t> voff16(n + 1);
    std::vector<uint32_t> vlen(n ? n : 1);
    uint64_t kacc = 0, vacc = 0, max_kv = 0;
    for (uint64_t i = 0; i < n; i++) {
        uint64_t kl = key_off[i + 1] - key_off[i], vl = val_off[i + 1] - val_off[i];
        if (kl > 65535) return kb_fail(ctx, KB_ELIMIT, "key %llu longer than 65535 bytes", (unsigned long long)i);
        if (vl > 0xFFFFFFFFull) return kb_fail(ctx, KB_ELIMIT, "value %llu too long", (unsigned long long)i);
        koff16[i] = (uint32_t)kacc;
        voff16[i] = vacc;
        klen[i] = (uint16_t)kl;
        vlen[i] = (uint32_t)vl;
        kacc += (kl + 15) / 16;
        vacc += (vl + 15) / 16;
        max_kv = std::max<uint64_t>(max_kv, (kl + 15) / 16 + (vl + 15) / 16);
        if (kacc > 0xFFFFFFF0ull) return kb_fail(ctx, KB_ELIMIT, "key slab exceeds 64 GiB");
    }
    koff16[n] = (uint32_t)kacc;
    voff16[n] = vacc;
    ctx->key_bytes = kacc * 16;
    ctx->val_bytes = vacc * 16;
    ctx->max_kv_chunks = (uint32_t)std::min<uint64_t>(max_kv, 0xFFFFFFFFu);

    KB_TRY(dbuf_ensure(ctx, ctx->d_kslab, kacc * 16 + 64));
    KB_TRY(dbuf_ensure(ctx, ctx->d_vslab, vacc * 16 + 16));
    KB_TRY(dbuf_ensure(ctx, ctx->d_koff16, (n + 1) * 4));
    KB_TRY(dbuf_ensure(ctx, ctx->d_klen, (n + 1) * 2));
    KB_TRY(dbuf_ensure(ctx, ctx->d_voff16, (n + 1) * 8));
    KB_TRY(dbuf_ensure(ctx, ctx->d_vlen, (n + 1) * 4));
    KB_CUDA(ctx, cudaMemsetAsync(ctx->d_kslab.p, 0, kacc * 16 + 16, ctx->stream));
    KB_CUDA(ctx, cudaMemsetAsync(ctx->d_vslab.p, 0, vacc * 16 + 16, ctx->stream));
    KB_CUDA(ctx, cudaMemcpyAsync(ctx->d_koff16.p, koff16.data(), (n + 1) * 4, cudaMemcpyHostToDevice, ctx->stream));
    KB_CUDA(ctx, cudaMemcpyAsync(ctx->d_klen.p, klen.data(), n * 2, cudaMemcpyHostToDevice, ctx->stream));
    KB_CUDA(ctx, cudaMemcpyAsync(ctx->d_voff16.p, voff16.data(), (n + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    KB_CUDA(ctx, cudaMemcpyAsync(ctx->d_vlen.p, vlen.data(), n * 4, cudaMemcpyHostToDevice, ctx->stream));

    // packed source bytes -> device (temporary), then repack on the device
    uint64_t ksrc = n ? key_off[n] - key_off[0] : 0, vsrc = n ? val_off[n] - val_off[0] : 0;
    DBuf tmp_b, tmp_o;
    uint64_t maxsrc = std::max(ksrc, vsrc);
    KB_TRY(dbuf_ensure(ctx, tmp_b, maxsrc + 16));
    KB_TRY(dbuf_ensure(ctx, tmp_o, (n + 1) * 8));
    const int TB = 256;
    int rg = (int)std::min<uint64_t>((n * 32 + TB - 1) / TB + 1, 148 * 16);
    int rc = KB_OK;
    do {
        if (n == 0) break;
        // keys (offsets rebased to 0 if the caller's first offset is not 0)
        std::vector<uint64_t> rebased;
        const uint64_t *ko = key_off, *vo = val_off;
        if (key_off[0] != 0) {
            rebased.resize(n + 1);
            for (uint64_t i = 0; i <= n; i++) rebased[i] = key_off[i] - key_off[0];
            ko = rebased.data();
        }
        if (cudaMemcpyAsync(tmp_b.p, keys + key_off[0], ksrc, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess ||
            cudaMemcpyAsync(tmp_o.p, ko, (n + 1) * 8, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess) {
            rc = kb_fail(ctx, KB_ECUDA, "H2D of keys failed");
            break;
        }
        k_repack<<<rg, TB, 0, ctx->stream>>>((const uint8_t *)tmp_b.p, (const uint64_t *)tmp_o.p,
                                             (uint8_t *)ctx->d_kslab.p, (const uint32_t *)ctx->d_koff16.p, nullptr,
                                             (uint32_t)n);
        if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) {
            rc = kb_fail(ctx, KB_ECUDA, "key repack failed: %s", cudaGetErrorString(cudaGetLastError()));
            break;
        }
        std::vector<uint64_t> rebased_v;
        if (val_off[0] != 0) {
            rebased_v.resize(n + 1);
            for (uint64_t i = 0; i <= n; i++) rebased_v[i] = val_off[i] - val_off[0];
            vo = rebased_v.data();
        }
        if (cudaMemcpyAsync(tmp_b.p, vals + val_off[0], vsrc, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess ||
            cudaMemcpyAsync(tmp_o.p, vo, (n + 1) * 8, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess) {
            rc = kb_fail(ctx, KB_ECUDA, "H2D of values failed");
            break;
        }
        k_repack<<<rg, TB, 0, ctx->stream>>>((const uint8_t *)tmp_b.p, (const uint64_t *)tmp_o.p,
                                             (uint8_t *)ctx->d_vslab.p, nullptr, (const uint64_t *)ctx->d_voff16.p,
                                             (uint32_t)n);
        if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) {
            rc = kb_fail(ctx, KB_ECUDA, "value repack failed: %s", cudaGetErrorString(cudaGetLastError()));
            break;
        }
    } while (0);
    cudaFree(tmp_b.p);
    cudaFree(tmp_o.p);
    if (rc != KB_OK) return rc;

    ctx->st.kslab = (const uint4 *)ctx->d_kslab.p;
    ctx->st.koff16 = (const uint32_t *)ctx->d_koff16.p;
    ctx->st.klen = (const uint16_t *)ctx->d_klen.p;
    ctx->st.vslab = (const uint4 *)ctx->d_vslab.p;
    ctx->st.voff16 = (const uint64_t *)ctx->d_voff16.p;
    ctx->st.vlen = (const uint32_t *)ctx->d_vlen.p;
    ctx->st.n = (uint32_t)n;
    KB_TRY(store_pack_dir(ctx));
    ctx->kused16 = kacc;
    ctx->vused16 = vacc;
    ctx->store_gen++;
    ctx->garbage_k16 = ctx->garbage_v16 = ctx->displaced = 0;
    ctx->ttl_queue.clear();
    ctx->ttl_of.clear();

    // the decoded columns, and the iterator contract: strictly ascending unique keys
    KB_TRY(store_build_columns(ctx, ""));
    ctx->loaded = true;
    return KB_OK;
}

extern "C" int kb_store_info(kb_ctx *ctx, uint64_t *n_records, uint64_t *key_bytes, uint64_t *val_bytes)
{
    if (!ctx) return KB_EINVAL;
    if (!ctx->loaded) return kb_fail(ctx, KB_ESTATE, "no store loaded");
    if (n_records) *n_records = ctx->st.n;
    if (key_bytes) *key_bytes = ctx->key_bytes;
    if (val_bytes) *val_bytes = ctx->val_bytes;
    return KB_OK;
}

// ------------------------------------------------------------------------------------------------
// durable dump / restore of the snapshot (device layout, so restore is file -> pinned staging -> HBM with no repack)
// ------------------------------------------------------------------------------------------------
namespace {
struct DumpHeader {
    char     magic[8];  // "KBB200D1"
    uint32_t version, header_bytes;
    uint64_t n, key_chunks, val_chunks;
    uint64_t compact_present, compact_rev;
    uint32_t max_kv_chunks, pad;
    uint64_t sum_dir, sum_keys, sum_vals;  // FNV-1a 64 of the directory section and of the two slabs
};
constexpr size_t DUMP_STAGE = 64u << 20;  // bytes per host <-> device hop

inline uint64_t fnv1a64_update(uint64_t h, const uint8_t *p, size_t n)
{
    // 8 bytes per step (word-wise FNV-1a variant): the checksum only has to detect torn or foreign files
    size_t i = 0;
    for (; i + 8 <= n; i += 8) {
        uint64_t w;
        memcpy(&w, p + i, 8);
        h = (h ^ w) * 0x100000001b3ull;
    }
    for (; i < n; i++) h = (h ^ p[i]) * 0x100000001b3ull;
    return h;
}

// device -> file through the pinned staging buffer; returns the checksum of the bytes written
int dump_section(kb_ctx *ctx, FILE *f, const void *dev, uint64_t bytes, uint64_t *sum)
{
    uint64_t h = 0xcbf29ce484222325ull;
    for (uint64_t off = 0; off < bytes; off += DUMP_STAGE) {
        const size_t n = (size_t)std::min<uint64_t>(DUMP_STAGE, bytes - off);
        KB_CUDA(ctx, cudaMemcpyAsync(ctx->h_stage.p, (const uint8_t *)dev + off, n, cudaMemcpyDeviceToHost, ctx->stream));
        KB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        h = fnv1a64_update(h, (const uint8_t *)ctx->h_stage.p, n);
        if (fwrite(ctx->h_stage.p, 1, n, f) != n) return kb_fail(ctx, KB_EIO, "dump: short write");
    }
    *sum = h;
    return KB_OK;
}

int restore_section(kb_ctx *ctx, FILE *f, void *dev, uint64_t bytes, uint64_t *sum)
{
    uint64_t h = 0xcbf29ce484222325ull;
    for (uint64_t off = 0; off < bytes; off += DUMP_STAGE) {
        const size_t n = (size_t)std::min<uint64_t>(DUMP_STAGE, bytes - off);
        if (fread(ctx->h_stage.p, 1, n, f) != n) return kb_fail(ctx, KB_EINVAL, "restore: file truncated");
        h = fnv1a64_update(h, (const uint8_t *)ctx->h_stage.p, n);
        KB_CUDA(ctx, cudaMemcpyAsync((uint8_t *)dev + off, ctx->h_stage.p, n, cudaMemcpyHostToDevice, ctx->stream));
        KB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // the staging buffer is reused by the next hop
    }
    *sum = h;
    return KB_OK;
}
}  // namespace

extern "C" int kb_dump(kb_ctx *ctx, const char *path)
{
    if (!ctx || !path) return KB_EINVAL;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (!ctx->loaded) return kb_fail(ctx, KB_ESTATE, "no store loaded");
    cudaSetDevice(ctx->device);
    KB_TRY(ctx_quiesce(ctx));
    KB_TRY(store_compact_layout(ctx));  // the file holds the contiguous, key-ordered layout
    KB_TRY(hbuf_ensure(ctx, ctx->h_stage, DUMP_STAGE));
    // the record directory lives on the device only: fetch it for the directory section
    std::vector<uint32_t> h_koff16(ctx->st.n + 1), h_vlen(std::max<uint32_t>(ctx->st.n, 1));
    std::vector<uint16_t> h_klen(std::max<uint32_t>(ctx->st.n, 1));
    std::vector<uint64_t> h_voff16(ctx->st.n + 1);
    if (ctx->st.n) {
        const uint64_t nn = ctx->st.n;
        KB_CUDA(ctx, cudaMemcpyAsync(h_koff16.data(), ctx->st.koff16, nn * 4, cudaMemcpyDeviceToHost, ctx->stream));
        KB_CUDA(ctx, cudaMemcpyAsync(h_klen.data(), ctx->st.klen, nn * 2, cudaMemcpyDeviceToHost, ctx->stream));
        KB_CUDA(ctx, cudaMemcpyAsync(h_voff16.data(), ctx->st.voff16, nn * 8, cudaMemcpyDeviceToHost, ctx->stream));
        KB_CUDA(ctx, cudaMemcpyAsync(h_vlen.data(), ctx->st.vlen, nn * 4, cudaMemcpyDeviceToHost, ctx->stream));
        KB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    h_koff16[ctx->st.n] = (uint32_t)ctx->kused16;
    h_voff16[ctx->st.n] = ctx->vused16;
    const std::string tmp = std::string(path) + ".tmp";
    FILE *f = fopen(tmp.c_str(), "wb");
    if (!f) return kb_fail(ctx, KB_EIO, "dump: cannot create %s", tmp.c_str());
    const uint64_t n = ctx->st.n;
    DumpHeader h;
    memset(&h, 0, sizeof(h));
    memcpy(h.magic, "KBB200D1", 8);
    h.version = 1;
    h.header_bytes = (uint32_t)sizeof(DumpHeader);
    h.n = n;
    h.key_chunks = ctx->key_bytes / 16;
    h.val_chunks = ctx->val_bytes / 16;
    h.compact_present = ctx->compact_present ? 1 : 0;
    h.compact_rev = ctx->compact_rev;
    h.max_kv_chunks = ctx->max_kv_chunks;
    int rc = KB_OK;
    if (fwrite(&h, 1, sizeof(h), f) != sizeof(h)) rc = kb_fail(ctx, KB_EIO, "dump: short write");
    // directory section: the host copies are authoritative (kb_load_sorted / kb_apply_batch maintain them)
    uint64_t hd = 0xcbf29ce484222325ull;
    auto put = [&](const void *p, size_t bytes) {
        if (rc != KB_OK) return;
        hd = fnv1a64_update(hd, (const uint8_t *)p, bytes);
        if (bytes && fwrite(p, 1, bytes, f) != bytes) rc = kb_fail(ctx, KB_EIO, "dump: short write");
    };
    put(h_koff16.data(), (n + 1) * 4);
    put(h_klen.data(), n * 2);
    put(h_voff16.data(), (n + 1) * 8);
    put(h_vlen.data(), n * 4);
    h.sum_dir = hd;
    if (rc == KB_OK) rc = dump_section(ctx, f, ctx->d_kslab.p, ctx->key_bytes, &h.sum_keys);
    if (rc == KB_OK) rc = dump_section(ctx, f, ctx->d_vslab.p, ctx->val_bytes, &h.sum_vals);
    if (rc == KB_OK && (fseek(f, 0, SEEK_SET) != 0 || fwrite(&h, 1, sizeof(h), f) != sizeof(h)))
        rc = kb_fail(ctx, KB_EIO, "dump: cannot finish the header");
    if (fclose(f) != 0 && rc == KB_OK) rc = kb_fail(ctx, KB_EIO, "dump: close failed");
    if (rc == KB_OK && rename(tmp.c_str(), path) != 0) rc = kb_fail(ctx, KB_EIO, "dump: cannot rename to %s", path);
    if (rc != KB_OK) remove(tmp.c_str());
    return rc;
}

extern "C" int kb_restore(kb_ctx *ctx, const char *path)
{
    if (!ctx || !path) return KB_EINVAL;
    std::lock_guard<std::mutex> g(ctx->mu);
    cudaSetDevice(ctx->device);
    KB_TRY(ctx_quiesce(ctx));
    FILE *f = fopen(path, "rb");
    if (!f) return kb_fail(ctx, KB_EIO, "restore: cannot open %s", path);
    struct Closer {
        FILE *f;
        ~Closer() { fclose(f); }
    } closer{f};
    DumpHeader h;
    if (fread(&h, 1, sizeof(h), f) != sizeof(h) || memcmp(h.magic, "KBB200D1", 8) != 0 || h.version != 1 ||
        h.header_bytes != sizeof(DumpHeader))
        return kb_fail(ctx, KB_EINVAL, "restore: %s is not a kb_b200 dump (version 1)", path);
    const uint64_t n = h.n;
    if (n >= 0xFFFFFFFEull || h.key_chunks > 0xFFFFFFF0ull) return kb_fail(ctx, KB_ELIMIT, "restore: dump exceeds the format limits");
    ctx->loaded = false;
    std::vector<uint32_t> koff16(n + 1), vlen(n ? n : 1);
    std::vector<uint16_t> klen(n ? n : 1);
    std::vector<uint64_t> voff16(n + 1);
    uint64_t hd = 0xcbf29ce484222325ull;
    bool ok = true;
    auto get = [&](void *p, size_t bytes) {
        if (!ok) return;
        if (bytes && fread(p, 1, bytes, f) != bytes) ok = false;
        else hd = fnv1a64_update(hd, (const uint8_t *)p, bytes);
    };
    get(koff16.data(), (n + 1) * 4);
    get(klen.data(), n * 2);
    get(voff16.data(), (n + 1) * 8);
    get(vlen.data(), n * 4);
    if (!ok) return kb_fail(ctx, KB_EINVAL, "restore: file truncated");
    if (hd != h.sum_dir) return kb_fail(ctx, KB_EINVAL, "restore: directory checksum mismatch");
    // the directory must describe exactly the slabs that follow: monotone offsets, every record inside its slab
    if (koff16[0] != 0 || voff16[0] != 0 || koff16[n] != h.key_chunks || voff16[n] != h.val_chunks) ok = false;
    uint64_t max_kv = 0;
    for (uint64_t i = 0; ok && i < n; i++) {
        const uint64_t nk = ((uint32_t)klen[i] + 15) / 16, nv = ((uint64_t)vlen[i] + 15) / 16;
        if (koff16[i + 1] < koff16[i] || koff16[i + 1] - koff16[i] != nk) ok = false;
        if (voff16[i + 1] < voff16[i] || voff16[i + 1] - voff16[i] != nv) ok = false;
        max_kv = std::max(max_kv, nk + nv);
    }
    if (!ok) return kb_fail(ctx, KB_EINVAL, "restore: inconsistent record directory");
    KB_TRY(hbuf_ensure(ctx, ctx->h_stage, DUMP_STAGE));
    KB_TRY(dbuf_ensure(ctx, ctx->d_kslab, h.key_chunks * 16 + 64));
    KB_TRY(dbuf_ensure(ctx, ctx->d_vslab, h.val_chunks * 16 + 64));
    KB_TRY(dbuf_ensure(ctx, ctx->d_koff16, (n + 1) * 4));
    KB_TRY(dbuf_ensure(ctx, ctx->d_klen, (n + 1) * 2));
    KB_TRY(dbuf_ensure(ctx, ctx->d_voff16, (n + 1) * 8));
    KB_TRY(dbuf_ensure(ctx, ctx->d_vlen, (n + 1) * 4));
    KB_CUDA(ctx, cudaMemsetAsync((uint8_t *)ctx->d_kslab.p + h.key_chunks * 16, 0, 64, ctx->stream));
    KB_CUDA(ctx, cudaMemsetAsync((uint8_t *)ctx->d_vslab.p + h.val_chunks * 16, 0, 64, ctx->stream));
    uint64_t sk = 0, sv = 0;
    KB_TRY(restore_section(ctx, f, ctx->d_kslab.p, h.key_chunks * 16, &sk));
    KB_TRY(restore_section(ctx, f, ctx->d_vslab.p, h.val_chunks * 16, &sv));
    if (sk != h.sum_keys || sv != h.sum_vals) return kb_fail(ctx, KB_EINVAL, "restore: slab checksum mismatch");
    KB_CUDA(ctx, cudaMemcpyAsync(ctx->d_koff16.p, koff16.data(), (n + 1) * 4, cudaMemcpyHostToDevice, ctx->stream));
    KB_CUDA(ctx, cudaMemcpyAsync(ctx->d_klen.p, klen.data(), n * 2, cudaMemcpyHostToDevice, ctx->stream));
    KB_CUDA(ctx, cudaMemcpyAsync(ctx->d_voff16.p, voff16.data(), (n + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    KB_CUDA(ctx, cudaMemcpyAsync(ctx->d_vlen.p, vlen.data(), n * 4, cudaMemcpyHostToDevice, ctx->stream));
    ctx->st.kslab = (const uint4 *)ctx->d_kslab.p;
    ctx->st.koff16 = (const uint32_t *)ctx->d_koff16.p;
    ctx->st.klen = (const uint16_t *)ctx->d_klen.p;
    ctx->st.vslab = (const uint4 *)ctx->d_vslab.p;
    ctx->st.voff16 = (const uint64_t *)ctx->d_voff16.p;
    ctx->st.vlen = (const uint32_t *)ctx->d_vlen.p;
    ctx->st.n = (uint32_t)n;
    KB_TRY(store_pack_dir(ctx));
    ctx->key_bytes = h.key_chunks * 16;
    KB_TRY(store_build_columns(ctx, "restore: "));  // the decoded columns and the iterator contract, as in kb_load_sorted
    ctx->kused16 = h.key_chunks;
    ctx->vused16 = h.val_chunks;
    ctx->store_gen++;
    ctx->garbage_k16 = ctx->garbage_v16 = ctx->displaced = 0;
    ctx->ttl_queue.clear();
    ctx->ttl_of.clear();
    ctx->key_bytes = h.key_chunks * 16;
    ctx->val_bytes = h.val_chunks * 16;
    ctx->max_kv_chunks = (uint32_t)std::min<uint64_t>(max_kv, 0xFFFFFFFFu);
    ctx->compact_present = h.compact_present != 0;
    ctx->compact_rev = h.compact_rev;
    ctx->loaded = true;
    return KB_OK;
}

extern "C" int kb_set_compact_revision(kb_ctx *ctx, int present, uint64_t rev)
{
    if (!ctx) return KB_EINVAL;
    std::lock_guard<std::mutex> g(ctx->mu);
    ctx->compact_present = present != 0;
    ctx->compact_rev = rev;
    return KB_OK;
}

// ------------------------------------------------------------------------------------------------
// NCCL revision cursor (one ncclAllGather of one uint64 per rank; min over ranks on the device)
// ------------------------------------------------------------------------------------------------
struct IdBlob {
    char internal[KB_NCCL_ID_BYTES];
};

namespace {
struct NcclApi {
    void *h = nullptr;
    int (*GetUniqueId)(void *) = nullptr;
    int (*CommInitRank)(void **, int, /* ncclUniqueId by value */ IdBlob, int) = nullptr;
    int (*AllGather)(const void *, void *, size_t, int, void *, cudaStream_t) = nullptr;
    int (*CommDestroy)(void *) = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
};
}  // namespace

static NcclApi *nccl_api()
{
    static NcclApi api;
    static bool tried = false;
    if (tried) return api.h ? &api : nullptr;
    tried = true;
    // reuse the copy already mapped into the process (torch bundles one) before falling back to the system lib
    void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) return nullptr;
    api.GetUniqueId = (int (*)(void *))dlsym(h, "ncclGetUniqueId");
    api.CommInitRank = (int (*)(void **, int, IdBlob, int))dlsym(h, "ncclCommInitRank");
    api.AllGather = (int (*)(const void *, void *, size_t, int, void *, cudaStream_t))dlsym(h, "ncclAllGather");
    api.CommDestroy = (int (*)(void *))dlsym(h, "ncclCommDestroy");
    api.GetErrorString = (const char *(*)(int))dlsym(h, "ncclGetErrorString");
    if (!api.GetUniqueId || !api.CommInitRank || !api.AllGather) return nullptr;
    api.h = h;
    return &api;
}

extern "C" int kb_nccl_unique_id(uint8_t id[KB_NCCL_ID_BYTES])
{
    NcclApi *a = nccl_api();
    if (!a) return KB_ENCCL;
    IdBlob b;
    memset(&b, 0, sizeof(b));
    if (a->GetUniqueId(&b) != 0) return KB_ENCCL;
    memcpy(id, &b, KB_NCCL_ID_BYTES);
    return KB_OK;
}

// ---- peer-memory cursor exchange ------------------------------------------------------------------------------
// The one collective of the path moves 8 bytes per rank; ncclAllGather spends ~40 us of launch and protocol latency
// on it.  Here every rank owns a small slot buffer that all peers map (cudaIpc over NVLink / NVSwitch): a rank stores
// its cursor and then an epoch flag straight into every peer's buffer and spins on its own buffer until all flags
// of the epoch have arrived.  Two slot sets alternate by epoch parity: a rank can be at most one exchange ahead of
// the slowest peer (it needs that peer's flag to finish), so it never overwrites a set that is still being read.
constexpr int KB_P2P_MAX_RANKS = 1024;

__global__ void __launch_bounds__(KB_P2P_MAX_RANKS)
k_cursor_p2p(uint64_t *const *__restrict__ peers, int me, int n, uint64_t epoch, uint64_t local, uint64_t *out)
{
    __shared__ unsigned long long smin;
    __shared__ int failed;
    const int r = threadIdx.x;
    if (r == 0) {
        smin = ~0ull;
        failed = 0;
    }
    __syncthreads();
    const size_t set = (size_t)(epoch & 1) * n * 2;
    if (r < n) {
        volatile uint64_t *p = peers[r] + set + (size_t)me * 2;
        p[0] = local;
        __threadfence_system();
        p[1] = epoch;
        volatile uint64_t *mine = peers[me] + set + (size_t)r * 2;
        const long long t0 = clock64();
        bool ok = true;
        while (mine[1] < epoch) {  // a peer that is AHEAD (this rank skipped an exchange) also releases the wait
            if (clock64() - t0 > 8000000000ll) {  // ~4 s: a peer never joined this exchange
                ok = false;
                break;
            }
        }
        __threadfence_system();
        const uint64_t v = mine[0];
        out[r] = v;
        if (ok) atomicMin(&smin, (unsigned long long)v);
        else atomicExch(&failed, 1);
    }
    __syncthreads();
    if (r < n) __threadfence_system();  // the gathered values reach the mapped host buffer before the status word
    __syncthreads();
    if (r == 0) {
        out[n] = smin;
        __threadfence_system();
        *(volatile uint64_t *)&out[n + 1] = failed ? 2 : 1;  // status: 1 done, 2 timed out
    }
}

static void p2p_setup(kb_ctx *ctx, NcclApi *a)
{
    const int n = ctx->nccl_nranks, me = ctx->nccl_rank;
    if (n > KB_P2P_MAX_RANKS) return;
    const size_t slot_bytes = (size_t)2 * n * 2 * 8;
    void *mine = nullptr, *d_handles = nullptr;
    std::vector<cudaIpcMemHandle_t> handles(n);
    std::vector<void *> peer(n, nullptr);
    bool ok = cudaMalloc(&mine, slot_bytes) == cudaSuccess && cudaMemset(mine, 0, slot_bytes) == cudaSuccess &&
              cudaMalloc(&d_handles, (size_t)(n + 1) * sizeof(cudaIpcMemHandle_t) + 64) == cudaSuccess;
    cudaIpcMemHandle_t my_h;
    memset(&my_h, 0, sizeof(my_h));
    // a rank that cannot export its buffer still takes part in the handle all-gather (it is collective) and sends zeros
    const bool exported = ok && cudaIpcGetMemHandle(&my_h, mine) == cudaSuccess;
    if (d_handles) {
        uint8_t *dh = (uint8_t *)d_handles;
        cudaMemcpyAsync(dh, &my_h, sizeof(my_h), cudaMemcpyHostToDevice, ctx->stream);
        int rc = a->AllGather(dh, dh + sizeof(my_h), sizeof(my_h), /*ncclUint8*/ 1, ctx->nccl_comm, ctx->stream);
        if (rc != 0) ok = false;
        cudaMemcpyAsync(handles.data(), dh + sizeof(my_h), (size_t)n * sizeof(my_h), cudaMemcpyDeviceToHost, ctx->stream);
        if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) ok = false;
    }
    ok = ok && exported;
    static const cudaIpcMemHandle_t zero_h = {};
    for (int r = 0; ok && r < n; r++) {
        if (memcmp(&handles[r], &zero_h, sizeof(zero_h)) == 0) {
            ok = false;  // that peer could not export
        } else if (r == me) {
            peer[r] = mine;
        } else if (cudaIpcOpenMemHandle(&peer[r], handles[r], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
            peer[r] = nullptr;
            ok = false;
        }
    }
    if (ok) ok = dbuf_ensure(ctx, ctx->d_p2p_ptrs, (size_t)n * sizeof(void *)) == KB_OK &&
                 cudaMemcpy(ctx->d_p2p_ptrs.p, peer.data(), (size_t)n * sizeof(void *), cudaMemcpyHostToDevice) == cudaSuccess &&
                 cudaHostAlloc((void **)&ctx->h_p2p_out, (size_t)(n + 2) * 8, cudaHostAllocMapped) == cudaSuccess;
    // all ranks must take the same path: agree on the outcome (one more tiny all-gather, still collective on failure)
    if (d_handles) {
        uint8_t *dh = (uint8_t *)d_handles;
        const uint8_t mine_ok = ok ? 1 : 0;
        std::vector<uint8_t> all_ok(n, 0);
        cudaMemcpyAsync(dh, &mine_ok, 1, cudaMemcpyHostToDevice, ctx->stream);
        int rc = a->AllGather(dh, dh + 16, 1, /*ncclUint8*/ 1, ctx->nccl_comm, ctx->stream);
        cudaMemcpyAsync(all_ok.data(), dh + 16, (size_t)n, cudaMemcpyDeviceToHost, ctx->stream);
        if (rc != 0 || cudaStreamSynchronize(ctx->stream) != cudaSuccess) ok = false;
        for (int r = 0; r < n; r++) ok = ok && all_ok[r] == 1;
        cudaFree(d_handles);
    } else {
        ok = false;
    }
    cudaGetLastError();  // a failed IPC call must not poison later error checks
    if (!ok) {
        for (int r = 0; r < n; r++)
            if (peer[r] && peer[r] != mine) cudaIpcCloseMemHandle(peer[r]);
        if (mine) cudaFree(mine);
        return;
    }
    ctx->p2p_mine = mine;
    ctx->p2p_peer = peer;
    ctx->p2p_epoch = 0;
    ctx->p2p_ready = true;
}

extern "C" int kb_nccl_init(kb_ctx *ctx, const uint8_t id[KB_NCCL_ID_BYTES], int rank, int nranks)
{
    if (!ctx || !id || rank < 0 || rank >= nranks) return KB_EINVAL;
    std::lock_guard<std::mutex> g(ctx->mu);
    NcclApi *a = nccl_api();
    if (!a) return kb_fail(ctx, KB_ENCCL, "libnccl.so.2 not loadable");
    cudaSetDevice(ctx->device);
    IdBlob b;
    memcpy(&b, id, KB_NCCL_ID_BYTES);
    int rc = a->CommInitRank(&ctx->nccl_comm, nranks, b, rank);
    if (rc != 0) return kb_fail(ctx, KB_ENCCL, "ncclCommInitRank: %s", a->GetErrorString ? a->GetErrorString(rc) : "?");
    ctx->nccl_rank = rank;
    ctx->nccl_nranks = nranks;
    if (nranks > 1) p2p_setup(ctx, a);  // best effort: without it the cursor exchange stays on ncclAllGather
    return KB_OK;
}

extern "C" int kb_cursor_transport(kb_ctx *ctx)
{
    if (!ctx) return KB_EINVAL;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (!ctx->nccl_comm) return KB_CURSOR_NONE;
    if (ctx->nccl_nranks == 1) return KB_CURSOR_SINGLE;
    return ctx->p2p_ready && !ctx->cursor_force_nccl ? KB_CURSOR_P2P : KB_CURSOR_NCCL;
}

extern "C" int kb_cursor_force_nccl(kb_ctx *ctx, int on)
{
    if (!ctx) return KB_EINVAL;
    std::lock_guard<std::mutex> g(ctx->mu);
    ctx->cursor_force_nccl = on != 0;
    return KB_OK;
}

__global__ void k_cursor_min(const uint64_t *all, int n, uint64_t *out)
{
    uint64_t m = ~0ull;
    for (int i = 0; i < n; i++) m = all[i] < m ? all[i] : m;
    *out = m;
}

extern "C" int kb_cursor_allgather(kb_ctx *ctx, uint64_t local_rev, uint64_t *all_revs, uint64_t *min_rev)
{
    if (!ctx) return KB_EINVAL;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (!ctx->nccl_comm) return kb_fail(ctx, KB_ESTATE, "kb_nccl_init has not been called");
    NcclApi *a = nccl_api();
    cudaSetDevice(ctx->device);
    int n = ctx->nccl_nranks;
    if (n == 1) {
        // a single shard has nobody to exchange with: the readable revision is its own cursor
        if (all_revs) all_revs[0] = local_rev;
        if (min_rev) *min_rev = local_rev;
        return KB_OK;
    }
    if (ctx->p2p_ready && !ctx->cursor_force_nccl) {
        const uint64_t epoch = ++ctx->p2p_epoch;
        volatile uint64_t *out = ctx->h_p2p_out;
        out[n + 1] = 0;
        const int threads = ((n + 31) / 32) * 32;
        KB_LAUNCH(ctx, "k_cursor_p2p", (uint64_t)n * 16,
                  (k_cursor_p2p<<<1, threads, 0, ctx->stream>>>((uint64_t *const *)ctx->d_p2p_ptrs.p, ctx->nccl_rank, n, epoch,
                                                              local_rev, ctx->h_p2p_out)));
        // the kernel's last store is the status word in mapped pinned memory: polling it is a few microseconds cheaper
        // than a stream synchronisation; a launch failure or a hung device still ends in the synchronise below
        const auto t0 = std::chrono::steady_clock::now();
        for (uint64_t spins = 1; out[n + 1] == 0; spins++) {
            kb_cpu_relax();
            if ((spins & 0xFFFF) == 0 && std::chrono::steady_clock::now() - t0 > std::chrono::seconds(6)) break;
        }
        if (out[n + 1] == 0) KB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        if (out[n + 1] != 1) {
            // A peer never joined.  This rank leaves the peer-memory path for good: the late peer still finds this rank's
            // flag for the epoch it missed, then times out on the next one and falls back too, so the ranks meet again in
            // ncclAllGather instead of waiting 4 s on every exchange from here on.
            ctx->p2p_ready = false;
            return kb_fail(ctx, KB_ENCCL, "cursor exchange: a peer did not join epoch %llu (falling back to ncclAllGather)",
                           (unsigned long long)epoch);
        }
        if (all_revs)
            for (int r = 0; r < n; r++) all_revs[r] = out[r];
        if (min_rev) *min_rev = out[n];
        return KB_OK;
    }
    KB_TRY(dbuf_ensure(ctx, ctx->d_cursor, (size_t)(n + 2) * 8));
    uint64_t *d = (uint64_t *)ctx->d_cursor.p;  // [0]=local, [1..n]=gathered, [n+1]=min
    KB_TRY(hbuf_ensure(ctx, ctx->h_stage2, 64));
    *(uint64_t *)ctx->h_stage2.p = local_rev;
    KB_CUDA(ctx, cudaMemcpyAsync(d, ctx->h_stage2.p, 8, cudaMemcpyHostToDevice, ctx->stream));
    int rc = a->AllGather(d, d + 1, 1, /*ncclUint64*/ 5, ctx->nccl_comm, ctx->stream);
    if (rc != 0) return kb_fail(ctx, KB_ENCCL, "ncclAllGather: %s", a->GetErrorString ? a->GetErrorString(rc) : "?");
    KB_LAUNCH(ctx, "cursor_min", (uint64_t)n * 8, (k_cursor_min<<<1, 1, 0, ctx->stream>>>(d + 1, n, d + 1 + n)));
    std::vector<uint64_t> host(n + 1);
    KB_CUDA(ctx, cudaMemcpyAsync(host.data(), d + 1, (size_t)(n + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
    KB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (all_revs) memcpy(all_revs, host.data(), (size_t)n * 8);
    if (min_rev) *min_rev = host[n];
    return KB_OK;
}
