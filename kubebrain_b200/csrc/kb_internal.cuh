// kb_internal.cuh -- shared host/device plumbing of libkbb200.so (sm_100a only, no CPU fallback).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <chrono>
#include <map>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/kb_b200.h"

// ------------------------------------------------------------------------------------------------
// HBM layouts (DESIGN.md section 3)
// ------------------------------------------------------------------------------------------------
struct StoreDev {
    const uint4    *kslab;   // internal keys, every record starts on a 16-byte boundary, zero padded
    const uint32_t *koff16;  // n+1 offsets in 16-byte units
    const uint16_t *klen;    // n exact key lengths
    const uint4    *vslab;   // values, 16-byte aligned, zero padded
    const uint64_t *voff16;  // n+1 offsets in 16-byte units
    const uint32_t *vlen;    // n exact value lengths
    const uint4    *dir;     // n packed directory entries (one 16-byte load per record):
                             // {koff16, klen | (voff16 >> 32) << 16, vlen, (uint32_t)voff16}
    const uint64_t *crev;    // n decoded columns (kb_decode.cuh): revision of the key, or of a revision record's value
    const uint32_t *cword;   //   LCP with the preceding key | static flags (KB_C_*)
    uint32_t        n;
};

// fills StoreDev::dir from the four directory arrays (kb_core.cu); enqueued on ctx->stream
int store_pack_dir(struct kb_ctx *ctx);
// rewrites both slabs contiguously in key order when records are out of place or garbage exists (kb_scan.cu)
int store_compact_layout(struct kb_ctx *ctx);

// one scanner.Range / Count / Compact request, resolved to record indices
struct ReqDev {
    uint32_t lo, hi;       // record interval [lo, hi)
    uint32_t flat0;        // first slot of this request in the flat per-record scratch (multiple of TILE)
    uint32_t tile0;        // first tile of this request
    uint32_t ntiles;
    uint32_t sel_base;     // first slot of this request in the selection arrays
    uint64_t read_rev;
    int64_t  limit;
};

struct TileDev {
    uint32_t req;
    uint32_t rec0;   // first store record of the tile
    uint32_t n;      // records in the tile (<= TILE)
    uint32_t flat0;  // flat slot of rec0
    uint32_t lo;     // first record of the request (copy of ReqDev.lo)
    uint32_t pad;
    uint64_t read_rev;
};

struct ScanMode {
    int      compact;      // workerConfig.compact
    int      ttl_scan;     // !SupportTTL() && timeoutRevision != 0
    uint64_t timeout_rev;
    int      wire;         // 0: padded [key][value] arena; KB_WIRE_KVS_I / KB_WIRE_EVENTS_I: etcd protobuf elements
};
enum { KB_WIRE_NONE_I = 0, KB_WIRE_KVS_I = 1, KB_WIRE_EVENTS_I = 2 };

// per-record meta word of one request (col_meta, kb_decode.cuh)
#define KB_M_LCP_MASK 0x0000FFFFu
#define KB_M_DEC_OK   (1u << 16)
#define KB_M_REV0     (1u << 17)   // revision == 0 (revision record)
#define KB_M_TRIG     (1u << 18)   // takes part as "cur": decodable, not TTL-expired, rev <= read_rev
#define KB_M_TOMB     (1u << 19)   // value == "tombstone"
#define KB_M_PREVOK   (1u << 20)   // becomes "prev" (TRIG and not the Q5 skip)
#define KB_M_REVDEL   (1u << 21)   // class 3 victim
#define KB_M_TTLREV   (1u << 22)   // class 4 victim
#define KB_M_TTLOBJ   (1u << 23)   // class 5 victim
// static flags of a record's column word (cword bits 16..21; DEC_OK and REV0 keep their meta-word positions)
#define KB_C_TOMBV    (1u << 18)   // value == "tombstone"
#define KB_C_VL9      (1u << 19)   // value length == 9
#define KB_C_VL8      (1u << 20)   // value length >= 8
#define KB_C_EVENTS   (1u << 21)   // the user key contains "/events/"
#define KB_C_FLAGS    (KB_M_DEC_OK | KB_M_REV0 | KB_C_TOMBV | KB_C_VL9 | KB_C_VL8 | KB_C_EVENTS)
#define KB_LCP_INF    0xFFFFu
#define KB_NONE       0xFFFFFFFFu

#define KB_TILE       1024          // records per tile (256 threads x 4)

// ------------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 ldg_stream(const uint4 *p)
{
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}

__device__ __forceinline__ void stg_stream(uint4 *p, const uint4 &v)
{
    asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z),
                 "r"(v.w)
                 : "memory");
}

// first differing byte (memory order) of two 16-byte chunks, 16 when equal
__device__ __forceinline__ int first_diff16(const uint4 &a, const uint4 &b)
{
    uint32_t x;
    x = a.x ^ b.x; if (x) return (__ffs(x) - 1) >> 3;
    x = a.y ^ b.y; if (x) return 4 + ((__ffs(x) - 1) >> 3);
    x = a.z ^ b.z; if (x) return 8 + ((__ffs(x) - 1) >> 3);
    x = a.w ^ b.w; if (x) return 12 + ((__ffs(x) - 1) >> 3);
    return 16;
}

__device__ __forceinline__ uint32_t byte_of(const uint4 &a, int i)
{
    uint32_t w = (i < 4) ? a.x : (i < 8) ? a.y : (i < 12) ? a.z : a.w;
    return (w >> ((i & 3) * 8)) & 0xffu;
}

__device__ __forceinline__ uint64_t be64_bytes(const uint8_t *p)
{
    uint64_t v = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) v = (v << 8) | (uint64_t)p[i];
    return v;
}

__device__ __forceinline__ uint32_t pad16(uint32_t x) { return (x + 15u) & ~15u; }

// ---- mbarrier / bulk-copy helpers of the TMA copies (k_gather, k_wire_copy)
__device__ __forceinline__ uint32_t dsmem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
// Bounded wait (a bulk copy that faults never completes its barrier): gives up after ~2 s of polling and raises the
// context's error flag instead of hanging the stream; the results of that launch are then garbage and the host fails
// the call (kb_range_batch checks the flag).
__device__ __forceinline__ bool dmbar_wait(uint64_t *bar, uint32_t parity, unsigned int *err_flag)
{
    uint32_t done = 0;
    for (uint32_t spins = 0; spins < (1u << 26); spins++) {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(dsmem_u32(bar)), "r"(parity)
            : "memory");
        if (done) return true;
    }
    atomicExch(err_flag, 1u);
    return false;
}
// Streaming copies: the bytes are read once per answer, so they are the first to leave L2 (evict_first) -- the 126 MB L2
// then keeps what the latency-bound kernels running beside the copy re-read (directory arrays, decoded columns, the
// fan-out's tables and scratch) instead of cycling the answer's keys and values through it every step.
__device__ __forceinline__ uint64_t l2_evict_first_policy()
{
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}

// ------------------------------------------------------------------------------------------------
// host plumbing
// ------------------------------------------------------------------------------------------------
struct DBuf {
    void  *p = nullptr;
    size_t cap = 0;
};

struct HBuf {  // pinned host
    void  *p = nullptr;
    size_t cap = 0;
};

struct ProfEntry {
    std::string name;
    uint64_t launches = 0;
    double   ms = 0;
    uint64_t bytes = 0;
};

struct ProfPending {
    int idx;
    cudaEvent_t a, b;
};

struct Watcher {
    std::string prefix;
    uint64_t min_rev;
    bool live;
};

struct WatchTablesDev;  // kb_watch.cu

struct SearchPubBuf {  // mapped pinned: [flag u64 | pad to 64 bytes | results u32 x nb], written by k_search
    uint8_t *host = nullptr;
    size_t cap = 0;
    uint64_t epoch = 0;
};

// The per-batch state of a range call.  kb_ctx holds the CURRENT lane's fields directly (every entry point works on
// them); kb_range_submit leaves its batch in flight and exchanges them with a parked lane's, so that the next batch is laid out and
// launched on another stream / scratch set while the earlier ones' kernels run (lane_swap rotates through `parked`).
struct ScanLane {
    cudaStream_t stream = nullptr;
    cudaEvent_t ev_jobs = nullptr;
    uint8_t *h_rout = nullptr;
    size_t h_rout_cap = 0;
    uint64_t rout_epoch = 0;
    DBuf d_bounds, d_bres, d_reqs, d_tiles, d_tgt, d_tcnt, d_tscan, d_reqout, d_sel, d_slot;
    HBuf h_stage, h_stage2;
    SearchPubBuf search_pub;
    int id = 0;
};
constexpr int KB_MAX_LANES = 4;

struct kb_pending;  // a submitted range batch (kb_scan.cu)

struct kb_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t stream2 = nullptr;  // bound search of a range batch: runs beside the tail (gather) of the previous batch
    // The gather / wire copy of a range batch runs on its own stream, so the next batch's emit .. placement (main
    // stream) overlaps it.  Two sets of job buffers alternate between consecutive batches; ev_gather[set] marks the end
    // of the last gather that read a set, ev_jobs the end of the current batch's job construction.
    cudaStream_t stream_g = nullptr;
    cudaEvent_t ev_jobs = nullptr, ev_gather[2] = {nullptr, nullptr};
    uint64_t batch_seq = 0;
    ScanLane parked[KB_MAX_LANES - 1];            // the other lanes (kb_range_submit rotates through them)
    int n_lanes = 2, park_next = 0;
    int lane = 0;                                 // which lane the context's own fields are right now
    kb_pending *lane_pending[KB_MAX_LANES] = {nullptr, nullptr, nullptr, nullptr};  // submitted, rows not yet read back, per lane
    int prio_lane = 0;                            // priority of the lane streams (above the copy stream's when the device has levels)
    cudaStream_t stream_h = nullptr;              // device -> host copies of KB_OUT_HOST answers (behind the gather's event)
    // per-request results (ReqOut) published by the device into mapped pinned memory: [flag u64 | pad to 64 | rows]
    uint8_t *h_rout = nullptr;
    size_t   h_rout_cap = 0;
    uint64_t rout_epoch = 0;
    uint64_t *h_wpub = nullptr;      // watch match: [0] epoch flag, [1] total deliveries (mapped pinned, device-written)
    uint64_t wpub_epoch = 0;
    std::string err;
    std::mutex mu;

    // store
    bool loaded = false;
    StoreDev st{};
    DBuf d_kslab, d_koff16, d_klen, d_vslab, d_voff16, d_vlen, d_dir, d_crev, d_cword;
    uint64_t key_bytes = 0, val_bytes = 0;
    uint32_t max_kv_chunks = 0;  // largest padded [key][value] pair, in 16-byte chunks: sizes the gather's ring buffers
    // heap + sorted directory (kb_apply_batch): chunks in use at the slab tails, chunks no live record points at, records
    // appended out of key order since the last layout compaction; s_* = the spare directory set the next merge writes
    uint64_t kused16 = 0, vused16 = 0, garbage_k16 = 0, garbage_v16 = 0, displaced = 0, layout_compactions = 0;
    DBuf s_koff16, s_klen, s_voff16, s_vlen, s_dir, s_crev, s_cword;
    bool compact_present = false;
    uint64_t compact_rev = 0;
    // TTL puts: (expire_unix, internal key), ordered by time; ttl_of[key] = the expiry the key currently has (a later put
    // of the same key replaces or cancels it, a delete cancels it)
    std::multimap<uint64_t, std::string> ttl_queue;
    std::unordered_map<std::string, uint64_t> ttl_of;

    // scratch (grow only)
    DBuf d_bounds, d_bres, d_reqs, d_tiles /* alias into d_reqs */, d_tgt, d_agg, d_tcnt /* look-back states */, d_tscan, d_reqout,
        d_sel, d_slot, d_jobs, d_gjobs, d_jobs2, d_gjobs2 /* second job-buffer set */, d_flags,
        d_ctrs /* search counters and the copy kernels' error flag, kept at zero between kernels */;
    HBuf h_stage, h_stage2;

    // kb_range_prefetch: bound searches started ahead of the kb_range_batch that will use them (two in flight at most)
    typedef ::SearchPubBuf SearchPubBuf;
    SearchPubBuf search_pub;  // of the search a range call runs itself
    struct SearchSlot {
        HBuf stage;
        DBuf d_bounds, d_bres;
        SearchPubBuf pub;
        size_t ident_bytes = 0;
        uint64_t store_gen = 0, seq = 0;
        bool valid = false;
    } prefetch[2];
    uint32_t prefetch_next = 0;
    uint64_t store_gen = 0;  // bumped whenever the snapshot changes

    // buffer pools for results
    std::vector<DBuf> free_dev;
    std::vector<DBuf> free_arena;  // response arenas: only ever written by the gather stream (or after ctx_quiesce)
    std::vector<HBuf> free_host;

    // watchers
    std::vector<Watcher> watchers;
    std::vector<uint32_t> free_watch_ids;
    bool watch_dirty = true;
    WatchTablesDev *wt = nullptr;
    struct kb_events_dev *ev_scratch = nullptr;  // grow-only upload slab of kb_watch_match

    // NCCL (dlopen'ed)
    void *nccl_comm = nullptr;
    int nccl_rank = -1, nccl_nranks = 0;
    DBuf d_cursor;
    // peer-memory cursor exchange (set up by kb_nccl_init when every peer's slot buffer can be mapped over NVLink)
    bool p2p_ready = false;
    bool cursor_force_nccl = false;           // kb_cursor_force_nccl: measure / use the ncclAllGather path although peers map
    uint64_t p2p_epoch = 0;
    void *p2p_mine = nullptr;                 // this rank's slot buffer: 2 epochs x nranks x {value, flag}
    std::vector<void *> p2p_peer;             // every rank's slot buffer as seen from this device (own entry = p2p_mine)
    DBuf d_p2p_ptrs;                          // the same pointers on the device
    uint64_t *h_p2p_out = nullptr;            // pinned: [nranks] gathered cursors, [nranks] min, [nranks+1] status

    // profiling
    int prof_on = 0;  // 0 off, 1 every kernel, 2 only the HBM-bound copy (k_gather)
    std::vector<ProfEntry> prof;
    std::vector<ProfPending> prof_pending;
    std::vector<cudaEvent_t> ev_pool;
    uint64_t launches = 0;
    bool gather_attr_set = false, wire_attr_set = false;  // per-context (per-device) kernel attributes
};

struct kb_result {
    int type = 0;  // 1 range, 2 compact, 3 match
    int out_mode = 0;
    // range
    std::vector<uint64_t> req_first, req_count, req_examined;
    uint64_t n_kvs = 0, n_bytes = 0;
    HBuf h_meta, h_bytes;
    DBuf d_bytes;
    const uint32_t *rec_idx = nullptr;
    const uint64_t *rev = nullptr, *key_off = nullptr, *val_off = nullptr;
    const uint32_t *key_len = nullptr, *val_len = nullptr;
    cudaEvent_t done_ev = nullptr;         // recorded behind the gather on ctx->stream_g (device-resident range answers)
    int wire = 0;                          // KB_WIRE_*_I
    const uint64_t *elem_off = nullptr;    // wire modes: n_kvs + 1 element offsets into the arena
    // compact
    uint64_t n_victims = 0, count = 0, examined = 0, vic_cap = 0;
    HBuf h_vic;
    DBuf d_vic;
    // get
    uint64_t n_gets = 0;
    HBuf h_get;  // [status u8 n (padded)][mod_rev u64 n][val_off u64 n][rec u32 n][val_len u32 n]
    // match
    uint64_t n_watchers = 0, n_deliveries = 0;
    HBuf h_match;
    DBuf d_match;
};

kb_result *kb_result_new(int type, int out_mode);

int kb_fail(kb_ctx *ctx, int code, const char *fmt, ...);
int kb_cuda_fail(kb_ctx *ctx, cudaError_t e, const char *what);

#define KB_CUDA(ctx, call)                                               \
    do {                                                                 \
        cudaError_t _e = (call);                                         \
        if (_e != cudaSuccess) return kb_cuda_fail((ctx), _e, #call);    \
    } while (0)

#define KB_TRY(expr)              \
    do {                          \
        int _rc = (expr);         \
        if (_rc != KB_OK) return _rc; \
    } while (0)

int dbuf_ensure(kb_ctx *ctx, DBuf &b, size_t bytes);
int hbuf_ensure(kb_ctx *ctx, HBuf &b, size_t bytes);
int pool_get_dev(kb_ctx *ctx, size_t bytes, DBuf *out);
int pool_get_arena(kb_ctx *ctx, size_t bytes, DBuf *out);
void pool_put_arena(kb_ctx *ctx, DBuf b);
// read back the rows of every submitted range batch, then wait for the gather stream: every entry point other than the
// range calls starts with it
int ctx_quiesce(kb_ctx *ctx);
int kb_pending_harvest_all(kb_ctx *ctx);  // kb_scan.cu
void kb_pending_drop_all(kb_ctx *ctx);
void lane_swap(kb_ctx *ctx);
int pool_get_host(kb_ctx *ctx, size_t bytes, HBuf *out);
void pool_put_dev(kb_ctx *ctx, DBuf b);
void pool_put_host(kb_ctx *ctx, HBuf b);

// profiling: bracket a kernel launch with events when enabled
int prof_index(kb_ctx *ctx, const char *name);
static inline bool prof_major(const char *n) { return strcmp(n, "k_gather") == 0; }
void prof_begin(kb_ctx *ctx, int idx, uint64_t alg_bytes, cudaStream_t strm);
void prof_end(kb_ctx *ctx, cudaStream_t strm);

#define KB_LAUNCH_S(ctx, strm, name, bytes, ...)              \
    do {                                                      \
        static thread_local int _pi = -1;                     \
        const bool _p = (ctx)->prof_on == 1 || ((ctx)->prof_on == 2 && prof_major(name)); \
        if (_p) {                                             \
            _pi = prof_index((ctx), (name));                  \
            prof_begin((ctx), _pi, (bytes), (strm));          \
        }                                                     \
        __VA_ARGS__;                                          \
        (ctx)->launches++;                                    \
        if (_p) prof_end((ctx), (strm));                      \
    } while (0)
#define KB_LAUNCH(ctx, name, bytes, ...) KB_LAUNCH_S(ctx, (ctx)->stream, name, bytes, __VA_ARGS__)

// one polite spin of a host polling loop (the device publishes results into mapped pinned memory)
static inline void kb_cpu_relax()
{
#if defined(__x86_64__) || defined(__i386__)
    __builtin_ia32_pause();
#endif
}

// host wall-clock segments (with kb_prof_enable(ctx, 1 or 2)): where the non-kernel time of a call goes
typedef std::chrono::steady_clock::time_point kb_tp;
static inline kb_tp kb_now() { return std::chrono::steady_clock::now(); }
static inline void kb_seg(kb_ctx *ctx, const char *name, kb_tp &t)
{
    if (ctx->prof_on == 0) return;
    kb_tp n = kb_now();
    int i = prof_index(ctx, name);
    ctx->prof[i].launches++;
    ctx->prof[i].ms += std::chrono::duration<double, std::milli>(n - t).count();
    t = n;
}

// kb_watch.cu
void watch_tables_free(kb_ctx *ctx);
