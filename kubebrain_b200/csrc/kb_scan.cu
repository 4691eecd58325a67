// kb_scan.cu -- the MVCC range-scan and compaction-sweep path.
//
// Replaces (reference file:line):
//   storage.Iter over badger            pkg/storage/badger/iter.go:27-98        -> HBM slab + k_search
//   coder.Decode                        pkg/backend/coder/normal.go:58-70       -> decoded columns (kb_decode.cuh)
//   worker.run (range + compact)        pkg/backend/scanner/scanner.go:389-516  -> col_meta, k_emit, k_place
//   commonResultReceiver (limit)        pkg/backend/scanner/receiver.go:62-103  -> k_tile_scan, k_place, k_gather
//
// Kernel pipeline for one batch of requests (streams: S2 = bound search, S = main, SG = copy stream):
//   k_search      [S2] lower_bound of every [start,end) bound in the sorted slab (warp per bound, 32-ary); the only
//                 step the host waits for before it lays the requests out as tiles
//   k_emit        [S] per tile: every record's meta word from its decoded columns (crev / cword, written with the
//                 directory: kb_decode.cuh) and the request's read revision, then a segmented "last visible version"
//                 scan over the meta words (prev pointer + running min-LCP; the cross-tile carry by decoupled look-back)
//                 decides which record every key change emits / supersedes
//   k_tile_scan   [S] prefix sums of the per-tile counts / bytes (one CTA per 1024 tiles); k_req_totals: per-request rows
//   k_place       [S] ordered placement of the selection (limit applied) / ordered victim list
//   k_req_finalize [S] per-request prefix sums; publishes the per-request rows to mapped pinned memory (the host
//                 returns device-resident answers on that flag)
//   k_gather_jobs / k_wire_jobs [S] one copy job per emitted kv + the per-kv view arrays
//   k_gather / k_wire_copy [SG] bulk-TMA copy of the winners' key+value into the response arena (padded pairs, or
//                 etcd protobuf elements); overlaps the next batch's k_emit .. k_place
#include <algorithm>
#include <memory>

#include "kb_internal.cuh"
#include "kb_decode.cuh"
#include "kb_wire.cuh"

namespace {


constexpr unsigned FULL = 0xffffffffu;

// ------------------------------------------------------------------------------------------------
// k_search
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool key_less(const StoreDev &st, uint32_t rec, const uint4 *b, uint32_t blen)
{
    const uint4 *a = st.kslab + st.koff16[rec];
    uint32_t la = st.klen[rec];
    uint32_t m = la < blen ? la : blen;
    // Kubernetes keys share ~30 leading bytes: fetch the first three chunks together instead of one per round trip
    // (both slabs are padded, so the loads are in bounds; positions at or beyond m are ignored)
    {
        uint4 x0 = a[0], x1 = a[1], x2 = a[2];
        uint4 y0 = b[0], y1 = b[1], y2 = b[2];
        int p = first_diff16(x0, y0);
        if (p < 16) return p < (int)m ? byte_of(x0, p) < byte_of(y0, p) : la < blen;
        p = first_diff16(x1, y1);
        if (p < 16) return 16 + p < (int)m ? byte_of(x1, p) < byte_of(y1, p) : la < blen;
        p = first_diff16(x2, y2);
        if (p < 16) return 32 + p < (int)m ? byte_of(x2, p) < byte_of(y2, p) : la < blen;
    }
    for (uint32_t c = 3; c * 16 < m; c++) {
        uint4 x = a[c], y = b[c];
        int p = first_diff16(x, y);
        if (p < 16 && c * 16 + p < m) return byte_of(x, p) < byte_of(y, p);
    }
    return la < blen;
}

// out[w] = index of the first record whose key >= bound w (bytes.Compare order)
// pub (optional): mapped pinned memory [flag u64 | pad to 64 bytes | results u32 x nb].  Every warp stores its result there
// too; the warp that completes the count raises the flag to `epoch` -- the host polls it instead of paying a stream /
// event synchronisation (measured 70 us for an already finished search while another host thread was busy in the driver).
struct SearchPub {
    uint8_t *host;          // nullptr: results only in `out`
    unsigned int *done;     // device counter, zero between searches
    uint64_t epoch;
};

__global__ void __launch_bounds__(128) k_search(StoreDev st, const uint4 *__restrict__ bounds,
                                                const uint32_t *__restrict__ boff16,
                                                const uint32_t *__restrict__ blen, uint32_t nb,
                                                uint32_t *__restrict__ out, SearchPub pub)
{
    uint32_t w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    uint32_t lane = threadIdx.x & 31;
    if (w >= nb) return;
    const uint4 *b = bounds + boff16[w];
    uint32_t bl = blen[w];
    uint32_t lo = 0, hi = st.n;
    for (;;) {
        uint32_t span = hi - lo;
        if (span == 0) break;
        if (span <= 32) {
            bool less = lane < span ? key_less(st, lo + lane, b, bl) : false;
            lo += __popc(__ballot_sync(FULL, less));
            break;
        }
        uint32_t piv = lo + (uint32_t)(((uint64_t)span * (lane + 1)) / 33);
        bool less = key_less(st, piv, b, bl);
        int k = __popc(__ballot_sync(FULL, less));  // sorted slab: `less` holds for a prefix of the pivots
        uint32_t nlo = lo, nhi = hi;
        if (k > 0) nlo = __shfl_sync(FULL, piv, k - 1) + 1;
        if (k < 32) nhi = __shfl_sync(FULL, piv, k);
        lo = nlo;
        hi = nhi;
    }
    if (lane == 0) {
        out[w] = lo;
        if (pub.host) {
            ((volatile uint32_t *)(pub.host + 64))[w] = lo;
            __threadfence_system();
            if (atomicAdd(pub.done, 1u) == nb - 1) {
                *pub.done = 0;
                __threadfence_system();
                *(volatile uint64_t *)pub.host = pub.epoch;
            }
        }
    }
}


// ------------------------------------------------------------------------------------------------
// block-wide exclusive scan of the (last-prev slot, min-LCP-since) state
//   combine(A, B) = B.L != NONE ? B : (A.L, min(A.m, B.m))
// ------------------------------------------------------------------------------------------------
struct LM {
    uint32_t L, m;
};

__device__ __forceinline__ LM lm_combine(LM a, LM b)
{
    if (b.L != KB_NONE) return b;
    LM r;
    r.L = a.L;
    r.m = min(a.m, b.m);
    return r;
}

__device__ __forceinline__ LM block_excl_scan_lm(LM v, LM *warp_tot /* 8 */)
{
    const unsigned lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    LM inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        LM o;
        o.L = __shfl_up_sync(FULL, inc.L, d);
        o.m = __shfl_up_sync(FULL, inc.m, d);
        if (lane >= (unsigned)d) inc = lm_combine(o, inc);
    }
    if (lane == 31) warp_tot[w] = inc;
    __syncthreads();
    LM ex;  // exclusive within the warp
    ex.L = __shfl_up_sync(FULL, inc.L, 1);
    ex.m = __shfl_up_sync(FULL, inc.m, 1);
    if (lane == 0) {
        ex.L = KB_NONE;
        ex.m = KB_LCP_INF;
    }
    LM pre;
    pre.L = KB_NONE;
    pre.m = KB_LCP_INF;
    for (unsigned k = 0; k < w; k++) pre = lm_combine(pre, warp_tot[k]);
    __syncthreads();
    return lm_combine(pre, ex);
}

__device__ __forceinline__ uint64_t warp_incl_scan_u64(uint64_t v)
{
    const unsigned lane = threadIdx.x & 31;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint64_t o = __shfl_up_sync(FULL, v, d);
        if (lane >= (unsigned)d) v += o;
    }
    return v;
}

// exclusive scan of two u64 values per thread over 256 threads
__device__ __forceinline__ void block_excl_scan2(uint64_t a, uint64_t b, uint64_t &ea, uint64_t &eb, uint64_t &ta,
                                                 uint64_t &tb, uint64_t *ws /* 2*9 */)
{
    const unsigned lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    uint64_t ia = warp_incl_scan_u64(a), ib = warp_incl_scan_u64(b);
    if (lane == 31) {
        ws[w] = ia;
        ws[9 + w] = ib;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        uint64_t ra = 0, rb = 0;
        for (int k = 0; k < 8; k++) {
            uint64_t x = ws[k], y = ws[9 + k];
            ws[k] = ra;
            ws[9 + k] = rb;
            ra += x;
            rb += y;
        }
        ws[8] = ra;
        ws[17] = rb;
    }
    __syncthreads();
    ea = ia - a + ws[w];
    eb = ib - b + ws[9 + w];
    ta = ws[8];
    tb = ws[17];
    __syncthreads();
}

// ------------------------------------------------------------------------------------------------
// k_emit: the worker.run state machine, data-parallel.
// For every TRIG record i with prev p = last PREVOK record before it (inside the request):
//   same key  <=> klen[i] == klen[p] && min LCP over (p, i] >= klen[i] - 9
//   range  : key change && rev[p] > 0 && value[p] != tombstone  -> emit p         (scanner.go:457-462)
//   compact: same key && rev[p] > 0                             -> p superseded   (scanner.go:463-469)
// After the last record of a request the trailing prev is emitted (scanner.go:503-507).
// tgt[i] = flat slot of the emitted (range) / superseded (compact) record, or NONE.
// tcnt[2t] = emissions (range) or delete calls (compact) of tile t; tcnt[2t+1] = response bytes (range) or object
// count (compact).
//
// The (last PREVOK slot, min LCP since) carry into a tile comes from DECOUPLED LOOK-BACK over per-tile states: a tile
// (taken in ticket order) publishes its own aggregate at once, then warp 0 reads the states of up to 32 preceding tiles
// of the request per step until it meets an inclusive prefix or a tile that holds a PREVOK record (nothing before such a
// tile can matter).  Round 1 walked the sub-tile aggregates backwards with one thread until it met a visible record: a
// scan whose records are mostly invisible (read revision below the versions, compact at an old revision) cost O(tiles)
// dependent loads per tile; now it costs one step per tile.
// (Round 2 also tried resolving the output positions by look-back in the same pass -- one kernel instead of three: with
// ~1 200 tiles of 1 024 records in flight every tile walked ~5 windows back to the frontier of resolved prefixes, 2.5 ms
// per 100M records against 1.1 ms for emit + scan + place; profiles/r02_run2_decode_sweep.txt.)
// ------------------------------------------------------------------------------------------------
struct ReqOut {
    uint64_t total;        // emissions (range) / delete calls (compact)
    uint64_t total_aux;    // response bytes (range) / object count (compact)
    uint64_t capped_aux;   // response bytes of the first `limit` emissions (valid with KB_RO_CAPPED)
    uint32_t examined;     // records pulled from the iterator (valid with KB_RO_LIMIT_STOP, else hi - lo)
    uint32_t flags;
};
enum { KB_RO_LIMIT_STOP = 1u, KB_RO_CAPPED = 2u };

struct __align__(16) TileState {  // 32 bytes; zeroed by one memset per batch
    unsigned long long lm_agg, lm_pre;  // (last PREVOK slot | min LCP << 32): the tile alone / request start .. this tile
    uint32_t st_lm;                     // 0 empty, 1 aggregate valid, 2 inclusive prefix valid
    uint32_t pad[3];
};
enum { TS_EMPTY = 0, TS_AGG = 1, TS_PREFIX = 2 };

__device__ __forceinline__ unsigned long long lm_pack(LM v) { return ((unsigned long long)v.m << 32) | v.L; }
__device__ __forceinline__ LM lm_unpack(unsigned long long w)
{
    LM r;
    r.L = (uint32_t)w;
    r.m = (uint32_t)(w >> 32);
    return r;
}
__device__ __forceinline__ void ts_publish(uint32_t *status, uint32_t v)
{
    __threadfence();
    *(volatile uint32_t *)status = v;
}

// warp 0: exclusive (L, m) carry of tile t inside its request (tiles [t0, t))
__device__ __forceinline__ LM lookback_lm(TileState *ts, uint32_t t, uint32_t t0, uint32_t lane)
{
    LM acc;
    acc.L = KB_NONE;
    acc.m = KB_LCP_INF;
    for (uint32_t hi = t; hi > t0;) {  // this step looks at tiles hi-1, hi-2, .. (lane 0 = nearest)
        const bool in = lane < hi - t0;
        TileState *p = ts + (hi - 1 - (in ? lane : 0));
        uint32_t st;
        do {
            st = in ? *(volatile uint32_t *)&p->st_lm : (uint32_t)TS_PREFIX;
        } while (!__all_sync(FULL, st != TS_EMPTY));
        __threadfence();
        LM v;
        v.L = KB_NONE;
        v.m = KB_LCP_INF;
        if (in) v = lm_unpack(*(volatile unsigned long long *)(st == TS_PREFIX ? &p->lm_pre : &p->lm_agg));
        const unsigned term = __ballot_sync(FULL, in && (st == TS_PREFIX || v.L != KB_NONE));
        const uint32_t k = term ? (uint32_t)(__ffs(term) - 1) : 31u;  // farthest lane that still matters
        const uint32_t mm = __reduce_min_sync(FULL, (in && lane <= k) ? v.m : KB_LCP_INF);
        const uint32_t Lk = __shfl_sync(FULL, v.L, k);
        // combine(farther, nearer): nearer tiles (already in acc) hold no PREVOK, so only the minimum accumulates
        acc.m = min(acc.m, mm);
        if (term) {
            acc.L = Lk;
            break;
        }
        hi -= min(32u, hi - t0);
    }
    return acc;
}

// meta word of record `rec` for request `req` (col_meta over the record's decoded columns)
__device__ __forceinline__ uint32_t rec_meta(const StoreDev &st, const ScanMode &mode, const ReqDev &req, uint32_t rec)
{
    return col_meta(st.crev[rec], st.cword[rec], mode, req.read_rev, rec == req.lo);
}

template <bool COMPACT>
__global__ void __launch_bounds__(256, 8)  // <= 32 registers: must fit beside the gather CTAs and other batches' kernels
k_emit(StoreDev st, ScanMode mode, const ReqDev *__restrict__ reqs, const TileDev *__restrict__ tiles,
       TileState *__restrict__ ts, unsigned int *__restrict__ ticket, uint32_t *__restrict__ tgt,
       uint32_t *__restrict__ tail_tgt, uint64_t *__restrict__ tcnt)
{
    __shared__ LM warp_tot[8];
    __shared__ LM carry_s, agg_s;
    __shared__ uint64_t ws2[18];
    __shared__ uint32_t tile_s;
    if (threadIdx.x == 0) tile_s = atomicAdd(ticket, 1u);  // ticket order: every preceding tile has started
    __syncthreads();
    const uint32_t tix = tile_s;
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const TileDev tile = tiles[tix];
    const ReqDev req = reqs[tile.req];
    const bool first_tile = tix == req.tile0, last_tile = tix == req.tile0 + req.ntiles - 1;
    TileState *my = ts + tix;
    const uint32_t base = threadIdx.x * 4;
    const uint32_t flat = tile.flat0 + base;
    uint32_t w[4];
#pragma unroll
    for (int k = 0; k < 4; k++) w[k] = base + k < tile.n ? rec_meta(st, mode, req, tile.rec0 + base + k) : KB_LCP_INF;
    LM mine;
    mine.L = KB_NONE;
    mine.m = KB_LCP_INF;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        if (w[k] & KB_M_PREVOK) {
            mine.L = flat + k;
            mine.m = KB_LCP_INF;
        } else {
            mine.m = min(mine.m, w[k] & KB_M_LCP_MASK);
        }
    }
    const LM ex = block_excl_scan_lm(mine, warp_tot);
    if (threadIdx.x == 255) agg_s = lm_combine(ex, mine);
    __syncthreads();
    if (warp == 0) {
        const LM agg = agg_s;
        LM carry;
        carry.L = KB_NONE;
        carry.m = KB_LCP_INF;
        bool resolved = first_tile;
        if (!first_tile) {
            // Fast path: the meta word of any record can be computed from its columns, so the last PREVOK record is
            // looked for directly in the 256 records before the tile -- 32 per step, nearest first.  Almost every tile
            // ends here without waiting for anybody.
            for (uint32_t back = 0; back < 256 && !resolved; back += 32) {
                const uint32_t wd = rec_meta(st, mode, req, tile.rec0 - 1 - back - lane);  // lane 0 = the record right in front
                const unsigned pm = __ballot_sync(FULL, wd & KB_M_PREVOK);
                const uint32_t k = pm ? (uint32_t)(__ffs(pm) - 1) : 32u;  // nearest PREVOK lane; records nearer than it count
                const uint32_t mm = __reduce_min_sync(FULL, lane < k ? (wd & KB_M_LCP_MASK) : KB_LCP_INF);
                carry.m = min(carry.m, mm);
                if (pm) {
                    carry.L = tile.flat0 - 1 - back - k;
                    resolved = true;
                }
            }
        }
        if (resolved) {
            if (lane == 0) {
                my->lm_pre = lm_pack(lm_combine(carry, agg));
                ts_publish(&my->st_lm, TS_PREFIX);
            }
        } else {
            // long run without a visible record: decoupled look-back over the tile states
            if (lane == 0) {
                my->lm_agg = lm_pack(agg);
                ts_publish(&my->st_lm, TS_AGG);
            }
            carry = lookback_lm(ts, tix, req.tile0, lane);
            if (lane == 0) {
                my->lm_pre = lm_pack(lm_combine(carry, agg));
                ts_publish(&my->st_lm, TS_PREFIX);
            }
        }
        if (lane == 0) carry_s = carry;
    }
    __syncthreads();
    LM x = lm_combine(carry_s, ex);

    uint64_t cnt = 0, aux = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        if (base + k >= tile.n) break;
        const uint32_t i = flat + k;
        const uint32_t word = w[k];
        uint32_t t = KB_NONE;
        if (word & KB_M_TRIG) {
            if (x.L != KB_NONE) {
                const uint32_t mm = min(x.m, word & KB_M_LCP_MASK);
                const uint32_t irec = req.lo + (i - req.flat0), prec = req.lo + (x.L - req.flat0);
                const uint32_t pw = rec_meta(st, mode, req, prec);
                const uint32_t kl = st.klen[irec], pkl = st.klen[prec];
                const bool same = (kl == pkl) && (mm >= kl - 9);
                if (!same) {
                    if (!(pw & KB_M_REV0) && !(pw & KB_M_TOMB)) {
                        if (COMPACT) {
                            aux++;  // count++ only
                        } else {
                            t = x.L;
                            cnt++;
                            aux += kv_resp_bytes(st, prec, mode.wire);
                        }
                    }
                } else if (COMPACT && !(pw & KB_M_REV0)) {
                    t = x.L;  // superseded version
                    cnt++;
                }
            }
            if (COMPACT) {
                if (word & KB_M_TOMB) cnt++;
                if (word & KB_M_REVDEL) cnt++;
            }
        }
        if (COMPACT && (word & (KB_M_TTLREV | KB_M_TTLOBJ))) cnt++;
        if (word & KB_M_PREVOK) {
            x.L = i;
            x.m = KB_LCP_INF;
        } else {
            x.m = min(x.m, word & KB_M_LCP_MASK);
        }
        tgt[i] = t;
        if (last_tile && base + k == tile.n - 1) {
            // end of the request's iterator: the trailing prev (scanner.go:503-507)
            uint32_t tt = KB_NONE;
            if (x.L != KB_NONE) {
                const uint32_t prec = req.lo + (x.L - req.flat0);
                const uint32_t pw = rec_meta(st, mode, req, prec);
                if (!(pw & KB_M_REV0) && !(pw & KB_M_TOMB)) {
                    if (COMPACT) {
                        aux++;
                    } else {
                        tt = x.L;
                        cnt++;
                        aux += kv_resp_bytes(st, prec, mode.wire);
                    }
                }
            }
            tail_tgt[tile.req] = tt;
        }
    }
    uint64_t ea, eb, ta, tb;
    block_excl_scan2(cnt, aux, ea, eb, ta, tb, ws2);
    if (threadIdx.x == 0) {
        tcnt[2 * tix] = ta;
        tcnt[2 * tix + 1] = tb;
    }
}

// tile table from the request table: tile t belongs to the last request whose tile0 <= t (requests without records own
// no tile; their tile0 equals their successor's)
__global__ void __launch_bounds__(256)
k_fill_tiles(const ReqDev *__restrict__ reqs, uint32_t nreq, uint32_t nt, TileDev *__restrict__ tiles)
{
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nt) return;
    uint32_t lo = 0, hi = nreq;  // invariant: reqs[lo].tile0 <= t
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (reqs[mid].tile0 <= t) lo = mid; else hi = mid;
    }
    const ReqDev r = reqs[lo];  // among equal tile0 the LAST request is found: the one that really owns tile t
    const uint32_t k = t - r.tile0, n = r.hi - r.lo;
    TileDev td;
    td.req = lo;
    td.rec0 = r.lo + k * KB_TILE;
    td.n = min((uint32_t)KB_TILE, n - k * KB_TILE);
    td.flat0 = r.flat0 + k * KB_TILE;
    td.lo = r.lo;
    td.pad = 0;
    td.read_rev = r.read_rev;
    tiles[t] = td;
}

// ------------------------------------------------------------------------------------------------
// k_tile_scan: exclusive prefix of the per-tile (count, aux) pairs over ALL tiles of the batch, tscan[2 * (T + 1)].
// One CTA per chunk of 1024 tiles (round 1: one CTA for everything, 35 us per 10M records): a chunk scans its tiles,
// publishes its total, and adds the totals of the chunks in front of it (at most a few hundred: plain look-back).
// ------------------------------------------------------------------------------------------------
struct __align__(16) ChunkState {
    unsigned long long cnt, aux;
    uint32_t ready;
    uint32_t pad[3];
};

__global__ void __launch_bounds__(256, 8)  // <= 32 registers: must fit beside the persistent CTAs of other batches
k_tile_scan(const uint64_t *__restrict__ tcnt, uint64_t *__restrict__ tscan, uint32_t ntiles, ChunkState *__restrict__ cs)
{
    __shared__ uint64_t ws2[18];
    __shared__ uint64_t base_s[2];
    const uint32_t c = blockIdx.x, t0 = c * 1024 + threadIdx.x * 4;
    uint64_t a[4], b[4], sa = 0, sb = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        a[k] = t0 + k < ntiles ? tcnt[2 * (t0 + k)] : 0;
        b[k] = t0 + k < ntiles ? tcnt[2 * (t0 + k) + 1] : 0;
        sa += a[k];
        sb += b[k];
    }
    uint64_t ea, eb, ta, tb;
    block_excl_scan2(sa, sb, ea, eb, ta, tb, ws2);
    if (threadIdx.x == 0) {
        cs[c].cnt = ta;
        cs[c].aux = tb;
        ts_publish(&cs[c].ready, 1u);
    }
    if (threadIdx.x < 32) {
        // totals of the chunks in front, 32 at a time (each is ready as soon as its own 1024 counts are summed)
        const uint32_t lane = threadIdx.x;
        uint64_t pa = 0, pb = 0;
        for (uint32_t p0 = 0; p0 < c; p0 += 32) {
            const uint32_t p = p0 + lane;
            if (p < c) {
                while (*(volatile uint32_t *)&cs[p].ready == 0) {}
                __threadfence();
                pa += *(volatile unsigned long long *)&cs[p].cnt;
                pb += *(volatile unsigned long long *)&cs[p].aux;
            }
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            pa += __shfl_xor_sync(FULL, pa, d);
            pb += __shfl_xor_sync(FULL, pb, d);
        }
        if (lane == 0) {
            base_s[0] = pa;
            base_s[1] = pb;
        }
    }
    __syncthreads();
    uint64_t ra = base_s[0] + ea, rb = base_s[1] + eb;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        if (t0 + k < ntiles) {
            tscan[2 * (t0 + k)] = ra;
            tscan[2 * (t0 + k) + 1] = rb;
        }
        ra += a[k];
        rb += b[k];
        if (t0 + k == ntiles - 1) {
            tscan[2 * ntiles] = ra;
            tscan[2 * ntiles + 1] = rb;
        }
    }
}

// per-request totals from the tile prefix sums; every field of the row is written (no memset needed)
__global__ void __launch_bounds__(256)
k_req_totals(const ReqDev *__restrict__ reqs, uint32_t nreq, const uint64_t *__restrict__ tscan, ReqOut *__restrict__ rout)
{
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nreq) return;
    const ReqDev r = reqs[q];
    ReqOut o;
    o.total = o.total_aux = 0;
    if (r.ntiles) {
        o.total = tscan[2 * (r.tile0 + r.ntiles)] - tscan[2 * r.tile0];
        o.total_aux = tscan[2 * (r.tile0 + r.ntiles) + 1] - tscan[2 * r.tile0 + 1];
    }
    o.capped_aux = 0;
    o.examined = 0;
    o.flags = 0;
    rout[q] = o;
}

// ------------------------------------------------------------------------------------------------
// k_place: ordered selection (range) -- position = emissions before it in the request; the first `limit`
// positions are kept (commonResultReceiver.needMore, receiver.go:82-87).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256, 8)  // <= 32 registers: must fit beside the persistent CTAs of other batches
k_place(StoreDev st, const ReqDev *__restrict__ reqs, const TileDev *__restrict__ tiles,
        const uint32_t *__restrict__ tgt, const uint32_t *__restrict__ tail_tgt,
        const uint64_t *__restrict__ tscan, uint32_t *__restrict__ sel, uint64_t *__restrict__ slot,
        ReqOut *__restrict__ rout, int wire)
{
    __shared__ uint64_t ws2[18];
    const TileDev tile = tiles[blockIdx.x];
    const ReqDev req = reqs[tile.req];
    const uint32_t base = threadIdx.x * 4;
    const uint32_t flat = tile.flat0 + base;
    const bool last_tile = (blockIdx.x == req.tile0 + req.ntiles - 1);
    uint32_t t[5];
    uint32_t sz[5];
    uint64_t cnt = 0, bytes = 0;
#pragma unroll
    for (int k = 0; k < 5; k++) {
        t[k] = KB_NONE;
        sz[k] = 0;
    }
    if (base < tile.n) {
        uint4 tw = *(const uint4 *)(tgt + flat);
        t[0] = tw.x;
        t[1] = base + 1 < tile.n ? tw.y : KB_NONE;
        t[2] = base + 2 < tile.n ? tw.z : KB_NONE;
        t[3] = base + 3 < tile.n ? tw.w : KB_NONE;
        if (last_tile && tile.n - 1 >= base && tile.n - 1 < base + 4) t[4] = tail_tgt[tile.req];
    }
#pragma unroll
    for (int k = 0; k < 5; k++) {
        if (t[k] != KB_NONE) {
            const uint32_t prec = req.lo + (t[k] - req.flat0);
            sz[k] = (uint32_t)kv_resp_bytes(st, prec, wire);
            cnt++;
            bytes += sz[k];
        }
    }
    uint64_t ea, eb, ta, tb;
    block_excl_scan2(cnt, bytes, ea, eb, ta, tb, ws2);
    uint64_t pos = tscan[2 * blockIdx.x] - tscan[2 * req.tile0] + ea;
    uint64_t off = tscan[2 * blockIdx.x + 1] - tscan[2 * req.tile0 + 1] + eb;
    const bool limited = req.limit > 0;
#pragma unroll
    for (int k = 0; k < 5; k++) {
        if (t[k] == KB_NONE) continue;
        if (!limited || pos < (uint64_t)req.limit) {
            sel[req.sel_base + pos] = req.lo + (t[k] - req.flat0);
            slot[req.sel_base + pos] = off;
            if (limited && pos == (uint64_t)req.limit - 1) {
                rout[tile.req].capped_aux = off + sz[k];
                uint32_t fl = KB_RO_CAPPED;
                if (k < 4) {
                    // the limit-th append happened inside the loop: the iterator stops here (Q4)
                    rout[tile.req].examined = (flat + k) - req.flat0 + 1;
                    fl |= KB_RO_LIMIT_STOP;
                }
                rout[tile.req].flags = fl;
            }
        }
        pos++;
        off += sz[k];
    }
}

// ordered delete calls (compact): per record [superseded prev] [tombstone] [revision record] | [ttl]
__global__ void __launch_bounds__(256, 8)  // <= 32 registers: must fit beside the persistent CTAs of other batches
k_place_victims(StoreDev st, ScanMode mode, const ReqDev *__restrict__ reqs, const TileDev *__restrict__ tiles,
                const uint32_t *__restrict__ tgt, const uint64_t *__restrict__ tscan, uint32_t *__restrict__ vidx,
                uint8_t *__restrict__ vcls)
{
    __shared__ uint64_t ws2[18];
    const TileDev tile = tiles[blockIdx.x];
    const ReqDev req = reqs[tile.req];
    const uint32_t base = threadIdx.x * 4;
    const uint32_t flat = tile.flat0 + base;
    uint32_t t[4], w[4];
    uint64_t cnt = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        t[k] = KB_NONE;
        w[k] = 0;
    }
    if (base < tile.n) {
        const uint4 tw = *(const uint4 *)(tgt + flat);
        t[0] = tw.x;
        if (base + 1 < tile.n) t[1] = tw.y;
        if (base + 2 < tile.n) t[2] = tw.z;
        if (base + 3 < tile.n) t[3] = tw.w;
    }
#pragma unroll
    for (int k = 0; k < 4; k++)
        if (base + k < tile.n) w[k] = rec_meta(st, mode, req, tile.rec0 + base + k);
#pragma unroll
    for (int k = 0; k < 4; k++) {
        if (t[k] != KB_NONE) cnt++;
        if ((w[k] & KB_M_TRIG) && (w[k] & KB_M_TOMB)) cnt++;
        if (w[k] & KB_M_REVDEL) cnt++;
        if (w[k] & (KB_M_TTLREV | KB_M_TTLOBJ)) cnt++;
    }
    uint64_t ea, eb, ta, tb;
    block_excl_scan2(cnt, 0, ea, eb, ta, tb, ws2);
    uint64_t pos = req.sel_base + tscan[2 * blockIdx.x] - tscan[2 * req.tile0] + ea;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        if (base + k >= tile.n) break;
        const uint32_t irec = req.lo + (flat + k - req.flat0);
        if (t[k] != KB_NONE) {
            vidx[pos] = req.lo + (t[k] - req.flat0);
            vcls[pos++] = KB_V_SUPERSEDED;
        }
        if ((w[k] & KB_M_TRIG) && (w[k] & KB_M_TOMB)) {
            vidx[pos] = irec;
            vcls[pos++] = KB_V_TOMBSTONE;
        }
        if (w[k] & KB_M_REVDEL) {
            vidx[pos] = irec;
            vcls[pos++] = KB_V_REVRECORD;
        }
        if (w[k] & KB_M_TTLREV) {
            vidx[pos] = irec;
            vcls[pos++] = KB_V_TTL_REVREC;
        }
        if (w[k] & KB_M_TTLOBJ) {
            vidx[pos] = irec;
            vcls[pos++] = KB_V_TTL_OBJECT;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// k_gather: one warp per emitted kv; key (internal key, padded) then value (padded), 16-byte vector copies
// ------------------------------------------------------------------------------------------------
struct GatherOut {
    uint32_t *rec_idx;
    uint64_t *rev;
    uint64_t *key_off;
    uint32_t *key_len;
    uint64_t *val_off;
    uint32_t *val_len;
};

// one copy job per emitted kv (32 bytes): built thread-parallel so the per-kv lookups (request search, selection,
// offsets, lengths) do not sit in front of the streaming copy
struct GatherJob {
    uint64_t dst16;   // arena chunk index
    uint64_t vsrc16;  // value slab chunk index
    uint32_t ksrc16;  // key slab chunk index
    uint32_t nk, nv;  // 16-byte chunks of key / value
    uint32_t kl;      // exact key length
};

__global__ void __launch_bounds__(256)
k_gather_jobs(StoreDev st, const ReqDev *__restrict__ reqs, uint32_t nreq, const uint64_t *__restrict__ job_first,
              const uint64_t *__restrict__ arena_base, const uint32_t *__restrict__ sel,
              const uint64_t *__restrict__ slot, GatherJob *__restrict__ jobs, GatherOut out)
{
    const uint64_t n_kvs = job_first[nreq];  // written by k_req_finalize
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n_kvs; k += (uint64_t)gridDim.x * blockDim.x) {
    uint32_t lo = 0, hi = nreq;  // request of kv k: last q with job_first[q] <= k
    while (hi - lo > 1) {
        uint32_t mid = (lo + hi) >> 1;
        if (job_first[mid] <= k) lo = mid; else hi = mid;
    }
    const uint32_t q = lo;
    const uint64_t s = reqs[q].sel_base + (k - job_first[q]);
    const uint32_t rec = sel[s];
    const uint64_t dst_byte = arena_base[q] + slot[s];
    const uint32_t kl = st.klen[rec], vl = st.vlen[rec];
    GatherJob j;
    j.dst16 = dst_byte >> 4;
    j.vsrc16 = st.voff16[rec];
    j.ksrc16 = st.koff16[rec];
    j.nk = (kl + 15) >> 4;
    j.nv = (vl + 15) >> 4;
    j.kl = kl;
    jobs[k] = j;
    out.rec_idx[k] = rec;
    out.key_off[k] = dst_byte + 4;
    out.key_len[k] = kl - 13;
    out.val_off[k] = dst_byte + (uint64_t)j.nk * 16;
    out.val_len[k] = vl;
    out.rev[k] = st.crev[rec];  // an emitted record has a non-zero key revision: the column holds it
    }
}

// ---- k_gather: bulk-TMA copy of every winner's [internal key, padded][value, padded] into the response arena.
// One elected lane per warp drives a ring of `stages` shared-memory buffers: cp.async.bulk global->shared
// (completion on an mbarrier), then cp.async.bulk shared->global into the arena.  A kv larger than one buffer is
// moved in pieces.  The copy engine generates full-line requests; the SM only issues two or three instructions per
// 2.5 KB piece.
constexpr int GATHER_WARPS = 8;
constexpr int GATHER_MAX_STAGES = 8;
constexpr uint32_t GATHER_MAX_PIECE = 160;       // 16-byte chunks per buffer (2560 B)
constexpr uint32_t GATHER_WARP_CHUNKS = 880;     // shared memory per warp (13.75 KiB): two CTAs of 8 warps per SM

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// bounded like dmbar_wait (kb_internal.cuh): a bulk copy that faults never completes its barrier; give up after ~2 s of
// polling and raise the context's error flag instead of hanging the stream
__device__ __forceinline__ void mbar_wait_parity(uint64_t *bar, uint32_t parity, unsigned int *err_flag)
{
    dmbar_wait(bar, parity, err_flag);
}

// `piece` (chunks per ring buffer) and `stages` (buffers per warp) are chosen by the host from the store's largest
// [key][value] pair so that a typical kv is exactly one piece and two CTAs fit per SM.  Blocks of 32 jobs are handed
// out through a global counter (zeroed by the kernel that builds the jobs), so a CTA that starts late -- the SM was
// still busy with another stream's kernel -- simply takes fewer blocks.
__global__ void __launch_bounds__(GATHER_WARPS * 32, 8)  // 32 registers: only lane 0 of a warp does more than fetch jobs
k_gather(StoreDev st, const GatherJob *__restrict__ jobs, const uint64_t *__restrict__ n_kvs_dev,
         uint4 *__restrict__ arena, uint32_t piece, uint32_t stages, unsigned long long *__restrict__ work_ctr,
         unsigned int *__restrict__ err_flag)
{
    extern __shared__ __align__(128) uint4 gbuf[];  // GATHER_WARPS x stages x piece
    __shared__ uint64_t bars[GATHER_WARPS * GATHER_MAX_STAGES];
    __shared__ uint64_t ring_dst[GATHER_WARPS * GATHER_MAX_STAGES];
    __shared__ uint32_t ring_len[GATHER_WARPS * GATHER_MAX_STAGES];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // Lane 0 drives the copies (the data never passes through registers); the other lanes only help to fetch the
    // job descriptors: 32 jobs per coalesced load, handed to lane 0 by shuffles, next block prefetched.
    uint4 *buf = gbuf + (size_t)warp * stages * piece;
    uint64_t *bar = bars + warp * GATHER_MAX_STAGES;
    uint64_t *rdst = ring_dst + warp * GATHER_MAX_STAGES;
    uint32_t *rlen = ring_len + warp * GATHER_MAX_STAGES;
    if (lane == 0) {
        for (uint32_t s = 0; s < stages; s++)
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(bar + s)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();

    const uint64_t n_kvs = *n_kvs_dev;
    const uint64_t l2pol = l2_evict_first_policy();  // both directions stream: the copy must not flush L2 for its neighbours
    const uint32_t dist = stages - 2;   // pieces in flight per warp
    uint32_t in_flight = 0;             // pieces issued and not yet stored (lane 0 only)
    uint32_t si = 0, ss = 0, ph = 0;    // issue slot, store slot, parity of the store slot's current fill

    // wait for the oldest in-flight piece and send it to the arena
    auto retire = [&]() {
        mbar_wait_parity(bar + ss, ph, err_flag);
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(arena + rdst[ss]),
                     "r"(smem_u32(buf + ss * piece)), "r"(rlen[ss] * 16), "l"(l2pol)
                     : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        if (++ss == stages) {
            ss = 0;
            ph ^= 1;
        }
        in_flight--;
    };
    auto grab = [&]() -> uint64_t {  // next block of 32 jobs
        unsigned long long b = 0;
        if (lane == 0) b = atomicAdd(work_ctr, 32ull);
        const uint32_t lo = __shfl_sync(0xffffffffu, (uint32_t)b, 0), hi = __shfl_sync(0xffffffffu, (uint32_t)(b >> 32), 0);
        return ((uint64_t)hi << 32) | lo;
    };

    const uint4 zero4 = make_uint4(0, 0, 0, 0);
    uint64_t base = grab();
    uint4 n0 = zero4, n1 = zero4;  // this lane's job of the NEXT block (prefetched)
    if (base + lane < n_kvs) {
        const uint4 *jp = (const uint4 *)(jobs + base + lane);
        n0 = __ldg(jp);
        n1 = __ldg(jp + 1);
    }
    while (base < n_kvs) {
        const uint4 c0j = n0, c1j = n1;
        const uint64_t nb = grab();
        n0 = n1 = zero4;
        if (nb + lane < n_kvs) {
            const uint4 *jp = (const uint4 *)(jobs + nb + lane);
            n0 = __ldg(jp);
            n1 = __ldg(jp + 1);
        }
        const uint64_t left = n_kvs - base;
        const uint32_t cnt = left < 32 ? (uint32_t)left : 32u;
        for (uint32_t j = 0; j < cnt; j++) {
            const uint32_t d_lo = __shfl_sync(0xffffffffu, c0j.x, j), d_hi = __shfl_sync(0xffffffffu, c0j.y, j);
            const uint32_t v_lo = __shfl_sync(0xffffffffu, c0j.z, j), v_hi = __shfl_sync(0xffffffffu, c0j.w, j);
            const uint32_t ksrc16 = __shfl_sync(0xffffffffu, c1j.x, j);
            const uint32_t nk = __shfl_sync(0xffffffffu, c1j.y, j), nv = __shfl_sync(0xffffffffu, c1j.z, j);
            if (lane == 0) {
                const uint64_t dst16 = ((uint64_t)d_hi << 32) | d_lo, vsrc16 = ((uint64_t)v_hi << 32) | v_lo;
                const uint32_t n = nk + nv;
                for (uint32_t c0 = 0; c0 < n; c0 += piece) {
                    const uint32_t len = min(piece, n - c0);
                    if (in_flight >= dist) retire();
                    // the buffer was last read by the bulk store of the piece `stages` issues ago; at most two younger
                    // store groups can still be pending when it has finished reading shared memory
                    asm volatile("cp.async.bulk.wait_group.read 2;" ::: "memory");
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar + si)),
                                 "r"(len * 16)
                                 : "memory");
                    uint4 *dstbuf = buf + si * piece;
                    const uint32_t kpart = c0 < nk ? min(nk - c0, len) : 0;  // chunks of this piece from the key
                    if (kpart)
                        asm volatile(
                            "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
                                smem_u32(dstbuf)),
                            "l"(st.kslab + ksrc16 + c0), "r"(kpart * 16), "r"(smem_u32(bar + si)), "l"(l2pol)
                            : "memory");
                    if (len > kpart) {
                        const uint32_t v0c = (c0 + kpart) - nk;  // first value chunk of this piece
                        asm volatile(
                            "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
                                smem_u32(dstbuf + kpart)),
                            "l"(st.vslab + vsrc16 + v0c), "r"((len - kpart) * 16), "r"(smem_u32(bar + si)), "l"(l2pol)
                            : "memory");
                    }
                    rdst[si] = dst16 + c0;
                    rlen[si] = len;
                    if (++si == stages) si = 0;
                    in_flight++;
                }
            }
        }
        base = nb;
    }
    if (lane == 0) {
        while (in_flight) retire();
        asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    }
}

// ring geometry for a store whose largest padded [key][value] pair is `max_kv_chunks`
static inline void gather_geometry(uint32_t max_kv_chunks, uint32_t *piece, uint32_t *stages)
{
    uint32_t p = std::min<uint32_t>(std::max<uint32_t>(max_kv_chunks, 32), GATHER_MAX_PIECE);
    uint32_t s = std::min<uint32_t>(std::max<uint32_t>(GATHER_WARP_CHUNKS / p, 3), GATHER_MAX_STAGES);
    *piece = p;
    *stages = s;
}

// ---- k_get_resolve: one warp per point read.  cand = (first record > EncodeObjectKey(key, revision)) - 1 is what the
// reference's reverse iterator yields first (range.go:97-107); it answers the read iff it decodes to the same user
// key with a non-zero revision (range.go:109-117); a tombstone value maps to ErrKeyNotFound (range.go:82-86).
struct GetOut {
    uint8_t *status;
    uint64_t *mod_rev;
    uint64_t *voff16;  // value slab chunk of the answering record (the host builds the copy jobs from it)
    uint32_t *rec;
    uint32_t *vlen;
};

__global__ void __launch_bounds__(128)
k_get_resolve(StoreDev st, const uint4 *__restrict__ bounds, const uint32_t *__restrict__ boff16,
              const uint32_t *__restrict__ blen, const uint32_t *__restrict__ ub, uint32_t n, GetOut out)
{
    const uint32_t g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (g >= n) return;
    const uint32_t idx = ub[g];
    uint32_t status = KB_GET_NOT_FOUND, rec = 0, vl = 0;
    uint64_t mrev = 0, vo = 0;
    if (idx > 0) {
        rec = idx - 1;
        const uint32_t bl = blen[g];           // magic + key + '$' + rev(8) + one 0x00 byte
        const uint32_t pre = bl - 9;           // magic + key + '$'
        const uint32_t kl = st.klen[rec];
        if (kl == pre + 8) {
            const uint4 *a = st.kslab + st.koff16[rec];
            const uint4 *b = bounds + boff16[g];
            bool eq = true;
            for (uint32_t c = lane; c * 16 < pre; c += 32) {
                uint4 x = a[c], y = b[c];
                int p = first_diff16(x, y);
                if (p < 16 && c * 16 + p < pre) eq = false;
            }
            eq = __all_sync(0xffffffffu, eq);
            if (eq) {
                mrev = be64_bytes((const uint8_t *)a + kl - 8);
                if (mrev != 0) {
                    vl = st.vlen[rec];
                    vo = st.voff16[rec];
                    status = KB_GET_FOUND;
                    if (vl == 9) {
                        const uint4 v0 = st.vslab[vo];
                        if (v0.x == 0x626d6f74u && v0.y == 0x6e6f7473u && (v0.z & 0xffu) == 0x65u) status = KB_GET_TOMBSTONE;
                    }
                }
            }
        }
    }
    if (lane == 0) {
        out.status[g] = (uint8_t)status;
        out.mod_rev[g] = status == KB_GET_NOT_FOUND ? 0 : mrev;
        out.voff16[g] = vo;
        out.rec[g] = rec;
        out.vlen[g] = vl;
    }
}

// ---- kb_apply_batch helpers ------------------------------------------------------------------------------
// exists[i] = 1 iff the record at pos[i] (lower_bound of op key i) carries exactly that key; old_vchunks[i] = its value's
// 16-byte chunks (they become garbage when the op replaces or deletes the record)
__global__ void __launch_bounds__(128)
k_key_exists(StoreDev st, const uint4 *__restrict__ bounds, const uint32_t *__restrict__ boff16,
             const uint32_t *__restrict__ blen, const uint32_t *__restrict__ pos, uint32_t n, uint8_t *__restrict__ exists,
             uint32_t *__restrict__ old_vchunks)
{
    const uint32_t g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (g >= n) return;
    const uint32_t r = pos[g];
    bool eq = r < st.n;
    if (eq) {
        const uint32_t bl = blen[g];
        eq = st.klen[r] == bl;
        if (eq) {
            const uint4 *a = st.kslab + st.koff16[r];
            const uint4 *b = bounds + boff16[g];
            for (uint32_t c = lane; c * 16 < bl; c += 32) {
                uint4 x = a[c], y = b[c];
                int p = first_diff16(x, y);
                if (p < 16 && c * 16 + p < bl) eq = false;
            }
        }
        eq = __all_sync(0xffffffffu, eq);
    }
    if (lane == 0) {
        exists[g] = eq ? 1 : 0;
        old_vchunks[g] = eq ? (st.vlen[r] + 15) >> 4 : 0;
    }
}

// The store is a HEAP of key / value bytes plus a directory sorted by key.  A committed batch appends the bytes of its
// puts at the slab tails and rebuilds only the directory: every surviving record moves by (#inserts at or before it) -
// (#deletes before it), every insert lands at (its lower bound) + (#inserts before it) - (#deletes before it).
// ins_pos / del_pos / rep_pos are ascending; entries are packed like StoreDev::dir.  A surviving record's decoded columns
// travel with it; k_col_fix then recomputes the entries the batch made stale.
struct DirArrays {
    uint32_t *koff16;
    uint16_t *klen;
    uint64_t *voff16;
    uint32_t *vlen;
    uint4 *dir;
    uint64_t *crev;
    uint32_t *cword;
};

__device__ __forceinline__ uint32_t lower_bound_u32(const uint32_t *a, uint32_t n, uint32_t v)
{
    uint32_t lo = 0, hi = n;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (a[mid] < v) lo = mid + 1; else hi = mid;
    }
    return lo;
}

__device__ __forceinline__ void dir_store(const DirArrays &d, uint32_t at, const uint4 &e)
{
    d.koff16[at] = e.x;
    d.klen[at] = (uint16_t)(e.y & 0xffffu);
    d.voff16[at] = ((uint64_t)(e.y >> 16) << 32) | e.w;
    d.vlen[at] = e.z;
    d.dir[at] = e;
}

__global__ void __launch_bounds__(256)
k_dir_merge(StoreDev old, const uint32_t *__restrict__ ins_pos, const uint4 *__restrict__ ins_ent, uint32_t n_ins,
            const uint32_t *__restrict__ del_pos, uint32_t n_del, const uint32_t *__restrict__ rep_pos,
            const uint4 *__restrict__ rep_ent, uint32_t n_rep, DirArrays out)
{
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < old.n) {
        const uint32_t i = (uint32_t)t;
        const uint32_t db = lower_bound_u32(del_pos, n_del, i);
        if (db < n_del && del_pos[db] == i) return;  // deleted
        const uint32_t ib = lower_bound_u32(ins_pos, n_ins, i + 1);  // inserts with pos <= i sort in front of record i
        uint4 e = old.dir[i];
        const uint32_t rb = lower_bound_u32(rep_pos, n_rep, i);
        if (rb < n_rep && rep_pos[rb] == i) {  // same key, new value
            const uint4 r = rep_ent[rb];
            e.y = (e.y & 0xffffu) | (r.y & 0xffff0000u);
            e.z = r.z;
            e.w = r.w;
        }
        const uint32_t at = i + ib - db;
        dir_store(out, at, e);
        out.crev[at] = old.crev[i];  // stale for a replaced record or a changed predecessor: k_col_fix rewrites those
        out.cword[at] = old.cword[i];
    } else if (t < (uint64_t)old.n + n_ins) {
        const uint32_t k = (uint32_t)(t - old.n);
        const uint32_t p = ins_pos[k];
        dir_store(out, p + k - lower_bound_u32(del_pos, n_del, p), ins_ent[k]);
    }
}

// The column entries a merge made stale, recomputed from the new directory (`nd`) and the slab bytes.  A surviving
// record's entry depends on its own key and value and on its predecessor's key, so only these can change:
//   an inserted record, and the record behind it (its predecessor is new);
//   the record that takes a deleted record's place (its predecessor was the deleted one's);
//   a replaced record (its value changed: tombstone flag, revision in the value);
//   whatever ends up at position 0 (no predecessor).
// One thread per candidate, O(ops) key reads; a record that is a candidate twice gets the same entry twice.
__global__ void __launch_bounds__(256)
k_col_fix(StoreDev nd, const uint32_t *__restrict__ ins_pos, uint32_t n_ins, const uint32_t *__restrict__ del_pos,
          uint32_t n_del, const uint32_t *__restrict__ rep_pos, uint32_t n_rep, uint64_t *__restrict__ crev,
          uint32_t *__restrict__ cword)
{
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t q[2] = {KB_NONE, KB_NONE};
    if (t < n_ins) {
        const uint32_t p = ins_pos[t];
        q[0] = p + (uint32_t)t - lower_bound_u32(del_pos, n_del, p);
        q[1] = q[0] + 1;
    } else if (t < (uint64_t)n_ins + n_del) {
        // the first new record behind the deleted one's place: survivors before it + inserts at or before it
        const uint32_t k = (uint32_t)(t - n_ins), d = del_pos[k];
        q[0] = d - k + lower_bound_u32(ins_pos, n_ins, d + 1);
    } else if (t < (uint64_t)n_ins + n_del + n_rep) {
        const uint32_t i = rep_pos[t - n_ins - n_del];
        q[0] = i + lower_bound_u32(ins_pos, n_ins, i + 1) - lower_bound_u32(del_pos, n_del, i);
    } else if (t == (uint64_t)n_ins + n_del + n_rep) {
        q[0] = 0;
    }
#pragma unroll
    for (int j = 0; j < 2; j++) {
        if (q[j] >= nd.n) continue;
        uint64_t r;
        uint32_t w;
        bool less;
        col_entry(nd, q[j], &r, &w, &less);
        crev[q[j]] = r;
        cword[q[j]] = w;
    }
}

// layout compaction: every record's key and value copied to its place in fresh, contiguous, sorted slabs (warp per record)
__global__ void __launch_bounds__(256)
k_relocate(StoreDev old, const uint32_t *__restrict__ nkoff16, const uint64_t *__restrict__ nvoff16, uint4 *__restrict__ nk,
           uint4 *__restrict__ nv)
{
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t r = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < old.n; r += warps) {
        const uint32_t kc = ((uint32_t)old.klen[r] + 15) >> 4, vc = (old.vlen[r] + 15) >> 4;
        const uint4 *ks = old.kslab + old.koff16[r], *vs = old.vslab + old.voff16[r];
        uint4 *kd = nk + nkoff16[r], *vd = nv + nvoff16[r];
        for (uint32_t c = lane; c < kc; c += 32) kd[c] = ldg_stream(ks + c);
        for (uint32_t c = lane; c < vc; c += 32) stg_stream(vd + c, ldg_stream(vs + c));
    }
}

// The per-request rows are the only thing the host needs before it can return a device-resident answer: the device
// stores them into mapped pinned memory and then raises the epoch flag, the host polls the flag -- no copy, no stream
// synchronisation, and the gather that follows keeps running after the call has returned.
__device__ __forceinline__ void publish_rout(const ReqOut *__restrict__ rout, uint32_t nreq, uint8_t *host, uint64_t epoch,
                                             const unsigned int *err_flag)
{
    const uint4 *src = (const uint4 *)rout;
    uint4 *dst = (uint4 *)(host + 64);
    for (uint32_t i = threadIdx.x; i < nreq * 2; i += blockDim.x) dst[i] = src[i];
    if (threadIdx.x == 0) *(volatile uint64_t *)(host + 8) = *err_flag;  // a bulk copy of this batch never completed
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence_system();
        *(volatile uint64_t *)host = epoch;
    }
}

__global__ void __launch_bounds__(256) k_publish_rout(const ReqOut *__restrict__ rout, uint32_t nreq, uint8_t *host,
                                                      uint64_t epoch, const unsigned int *err_flag)
{
    publish_rout(rout, nreq, host, epoch, err_flag);
}

// single CTA: per-request emitted count / response bytes (limit applied) and their exclusive prefixes over the
// requests: job_first[q] = first kv of request q, arena_base[q] = first arena byte of request q; [nreq] = totals
__global__ void __launch_bounds__(256, 8)  // <= 32 registers: must fit beside the persistent CTAs of other batches
k_req_finalize(const ReqDev *__restrict__ reqs, uint32_t nreq, const ReqOut *__restrict__ rout,
               uint64_t *__restrict__ job_first, uint64_t *__restrict__ arena_base,
               unsigned long long *__restrict__ work_ctr, uint8_t *host_rout, uint64_t epoch,
               const unsigned int *__restrict__ err_flag)
{
    if (threadIdx.x == 0) *work_ctr = 0;  // the gather's block counter
    __shared__ uint64_t ws2[18];
    __shared__ uint64_t carry[2];
    if (threadIdx.x == 0) carry[0] = carry[1] = 0;
    __syncthreads();
    for (uint32_t c0 = 0; c0 < nreq; c0 += 256) {
        const uint32_t q = c0 + threadIdx.x;
        uint64_t ne = 0, nb = 0;
        if (q < nreq) {
            const ReqOut o = rout[q];
            const int64_t lim = reqs[q].limit;
            ne = (lim > 0 && o.total > (uint64_t)lim) ? (uint64_t)lim : o.total;
            nb = (lim > 0 && (o.flags & KB_RO_CAPPED)) ? o.capped_aux : o.total_aux;
        }
        uint64_t ea, eb, ta, tb;
        block_excl_scan2(ne, nb, ea, eb, ta, tb, ws2);
        const uint64_t ca = carry[0], cb = carry[1];
        if (q < nreq) {
            job_first[q] = ca + ea;
            arena_base[q] = cb + eb;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            carry[0] = ca + ta;
            carry[1] = cb + tb;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        job_first[nreq] = carry[0];
        arena_base[nreq] = carry[1];
    }
    publish_rout(rout, nreq, host_rout, epoch, err_flag);
}

}  // namespace

// ================================================================================================
// host orchestration
// ================================================================================================
kb_result *kb_result_new(int type, int out_mode)
{
    kb_result *r = new kb_result();
    r->type = type;
    r->out_mode = out_mode;
    return r;
}

// return every pooled buffer of a result; the caller holds ctx->mu
static void result_release_locked(kb_ctx *ctx, kb_result *res)
{
    if (!res) return;
    if (ctx) {
        pool_put_host(ctx, res->h_meta);
        pool_put_host(ctx, res->h_bytes);
        pool_put_arena(ctx, res->d_bytes);
        if (res->done_ev) ctx->ev_pool.push_back(res->done_ev);
        pool_put_host(ctx, res->h_vic);
        pool_put_dev(ctx, res->d_vic);
        pool_put_host(ctx, res->h_match);
        pool_put_dev(ctx, res->d_match);
        pool_put_host(ctx, res->h_get);
    }
    delete res;
}

void kb_result_release_locked(kb_ctx *ctx, kb_result *res) { result_release_locked(ctx, res); }

extern "C" void kb_result_free(kb_ctx *ctx, kb_result *res)
{
    if (!res) return;
    if (ctx) {
        std::lock_guard<std::mutex> g(ctx->mu);
        result_release_locked(ctx, res);
    } else {
        delete res;
    }
}

namespace {

struct Resolved {
    std::vector<ReqDev> reqs;
    uint32_t nt = 0;  // tiles of the batch (the tile table itself is filled on the device, k_fill_tiles)
    uint64_t total_flat = 0, total_sel = 0, key_bytes = 0, n_records = 0;
};

// lay the requests ([lo,hi) already known) out as tiles of KB_TILE records that never span two requests
int layout_requests(kb_ctx *ctx, bool cap_by_limit, Resolved &R)
{
    R.n_records = 0;
    uint64_t flat = 0, selb = 0, nt = 0;
    for (size_t q = 0; q < R.reqs.size(); q++) {
        ReqDev &r = R.reqs[q];
        r.flat0 = (uint32_t)flat;
        r.tile0 = (uint32_t)nt;
        uint32_t n = r.hi - r.lo;
        r.ntiles = (n + KB_TILE - 1) / KB_TILE;
        r.sel_base = (uint32_t)selb;
        nt += r.ntiles;
        flat += (uint64_t)r.ntiles * KB_TILE;
        uint64_t cap = n;
        if (cap_by_limit && r.limit > 0) cap = std::min<uint64_t>(cap, (uint64_t)r.limit);
        selb += cap;
        R.n_records += n;
        if (flat >= 0xFFFFF000ull || selb >= 0xFFFFF000ull)
            return kb_fail(ctx, KB_ELIMIT, "batch examines more than 2^32 records; split it");
    }
    R.total_flat = flat;
    R.total_sel = selb;
    R.nt = (uint32_t)nt;
    return KB_OK;
}

// upload the bound keys, run k_search, and lay the requests out as tiles
// pack the bounds of a batch the way k_search reads them: [keys, each padded to 16 bytes + 3 chunks of slack | offsets |
// lengths]; returns the bytes to upload (the search results land behind them)
int pack_bounds(kb_ctx *ctx, const kb_range_req *reqs, uint64_t nreq, HBuf &stage, uint64_t *chunks_out)
{
    uint64_t chunks = 0;
    for (uint64_t q = 0; q < nreq; q++) {
        if ((!reqs[q].start && reqs[q].start_len) || (!reqs[q].end && reqs[q].end_len)) return KB_EINVAL;
        if (reqs[q].start_len > 65535 || reqs[q].end_len > 65535) return kb_fail(ctx, KB_ELIMIT, "bound key too long");
        chunks += (reqs[q].start_len + 15) / 16 + (reqs[q].end_len + 15) / 16 + 6;
    }
    const uint64_t nb = 2 * nreq;
    KB_TRY(hbuf_ensure(ctx, stage, chunks * 16 + nb * 12 + 128));
    uint8_t *hs = (uint8_t *)stage.p;
    memset(hs, 0, chunks * 16);
    uint32_t *hboff = (uint32_t *)(hs + chunks * 16), *hblen = hboff + nb;
    uint64_t c = 0;
    for (uint64_t q = 0; q < nreq; q++) {
        const uint8_t *keys[2] = {reqs[q].start, reqs[q].end};
        const uint64_t lens[2] = {reqs[q].start_len, reqs[q].end_len};
        for (int j = 0; j < 2; j++) {
            hboff[2 * q + j] = (uint32_t)c;
            hblen[2 * q + j] = (uint32_t)lens[j];
            if (lens[j]) memcpy(hs + c * 16, keys[j], lens[j]);
            c += (lens[j] + 15) / 16 + 3;
        }
    }
    *chunks_out = chunks;
    return KB_OK;
}

// upload + k_search, asynchronous on `ss`; the results are published into `pub` (mapped pinned: [flag | pad | u32 x nb])
int enqueue_search(kb_ctx *ctx, HBuf &stage, DBuf &d_bounds, DBuf &d_bres, uint64_t chunks, uint64_t nb, cudaStream_t ss,
                   kb_ctx::SearchPubBuf &pb, int slot)
{
    uint8_t *hs = (uint8_t *)stage.p;
    KB_TRY(dbuf_ensure(ctx, d_bounds, chunks * 16 + nb * 8 + 64));
    KB_TRY(dbuf_ensure(ctx, d_bres, nb * 4 + 16));
    const size_t need = 64 + nb * 4 + 64;
    if (!pb.host || pb.cap < need) {
        if (pb.host) {
            KB_CUDA(ctx, cudaStreamSynchronize(ss));
            cudaFreeHost(pb.host);
            pb.host = nullptr;
        }
        KB_CUDA(ctx, cudaHostAlloc((void **)&pb.host, need * 2, cudaHostAllocMapped));
        memset(pb.host, 0, need * 2);
        pb.cap = need * 2;
        pb.epoch = 0;
    }
    KB_CUDA(ctx, cudaMemcpyAsync(d_bounds.p, hs, chunks * 16 + nb * 8, cudaMemcpyHostToDevice, ss));
    const uint32_t *d_boff = (const uint32_t *)((const uint8_t *)d_bounds.p + chunks * 16);
    const unsigned sgrid = (unsigned)((nb * 32 + 127) / 128);
    pb.epoch++;
    if (nb == 0) {
        *(volatile uint64_t *)pb.host = pb.epoch;  // nothing to search: already "published"
        return KB_OK;
    }
    SearchPub pub{pb.host, (unsigned int *)ctx->d_ctrs.p + 16 + slot, pb.epoch};
    KB_LAUNCH(ctx, "k_search", nb * 64,
              (k_search<<<sgrid, 128, 0, ss>>>(ctx->st, (const uint4 *)d_bounds.p, d_boff, d_boff + nb, (uint32_t)nb,
                                               (uint32_t *)d_bres.p, pub)));
    return KB_OK;
}

// wait for a published search; the stream is consulted now and then so that a failed launch is noticed
int search_wait(kb_ctx *ctx, kb_ctx::SearchPubBuf &pb, cudaStream_t ss)
{
    volatile uint64_t *flag = (volatile uint64_t *)pb.host;
    for (uint64_t spins = 1;; spins++) {
        if (*flag == pb.epoch) {
            if (ctx->prof_on) ctx->prof[prof_index(ctx, "host:search_wait_spins")].launches += spins;
            return KB_OK;
        }
        kb_cpu_relax();
        if ((spins & 0xFFFF) == 0) {
            const cudaError_t q = cudaStreamQuery(ss);
            if (q == cudaSuccess) return *flag == pb.epoch ? KB_OK : kb_fail(ctx, KB_ECUDA, "bound search: results were not published");
            if (q != cudaErrorNotReady) return kb_cuda_fail(ctx, q, "bound search");
        }
    }
}

// upload the bound keys, run k_search (or pick up the search kb_range_prefetch started for exactly these bounds), and lay
// the requests out as tiles
int resolve_requests(kb_ctx *ctx, const kb_range_req *reqs, uint64_t nreq, bool cap_by_limit, Resolved &R,
                     kb_tp *tseg = nullptr)
{
    uint64_t chunks = 0;
    KB_TRY(pack_bounds(ctx, reqs, nreq, ctx->h_stage, &chunks));
    if (tseg) kb_seg(ctx, "host:range_pack_bounds", *tseg);
    const uint64_t nb = 2 * nreq;
    uint8_t *hs = (uint8_t *)ctx->h_stage.p;
    const uint32_t *hres = nullptr;
    const size_t ident_bytes = chunks * 16 + nb * 8;
    // a prefetched search for the same bounds on the same snapshot?
    kb_ctx::SearchSlot *hit = nullptr;
    for (auto &sl : ctx->prefetch)  // the OLDEST matching one: a caller may already have submitted the batch after this one
        if (sl.valid && sl.ident_bytes == ident_bytes && sl.store_gen == ctx->store_gen &&
            memcmp(sl.stage.p, hs, ident_bytes) == 0 && (!hit || sl.seq < hit->seq))
            hit = &sl;
    if (hit && ctx->prof_on != 1) {
        if (tseg) kb_seg(ctx, "host:range_search_enqueue", *tseg);
        KB_TRY(search_wait(ctx, hit->pub, ctx->stream2));
        hres = (const uint32_t *)(hit->pub.host + 64);
        hit->valid = false;  // consumed
        if (tseg) kb_seg(ctx, "host:range_search_sync", *tseg);
    } else {
        // The search only reads the snapshot and its own bound slab, so it runs on the second stream: while the previous
        // batch's gather is still draining the host already learns the record intervals of this one.
        // (With every kernel bracketed by profiling events -- level 1 -- it stays on the main stream.)
        cudaStream_t ss = ctx->prof_on == 1 ? ctx->stream : ctx->stream2;
        KB_TRY(enqueue_search(ctx, ctx->h_stage, ctx->d_bounds, ctx->d_bres, chunks, nb, ss, ctx->search_pub, 2 + ctx->lane));
        if (tseg) kb_seg(ctx, "host:range_search_enqueue", *tseg);
        KB_TRY(search_wait(ctx, ctx->search_pub, ss));
        hres = (const uint32_t *)(ctx->search_pub.host + 64);
        if (tseg) kb_seg(ctx, "host:range_search_sync", *tseg);
    }

    R.reqs.resize(nreq);
    for (uint64_t q = 0; q < nreq; q++) {
        ReqDev &r = R.reqs[q];
        r.lo = hres[2 * q];
        r.hi = std::max(hres[2 * q + 1], r.lo);
        r.read_rev = reqs[q].read_rev;
        r.limit = reqs[q].limit;
    }
    return layout_requests(ctx, cap_by_limit, R);
}

int upload_layout(kb_ctx *ctx, const Resolved &R)
{
    const size_t nreq = R.reqs.size(), nt = R.nt;
    // the tile table starts on a 32-byte boundary behind the requests; only the requests travel, the device derives the
    // tiles from them (a 100M-record sweep has 97 656 tiles: 0.4 ms of host loop + 3 MB of upload in round 1)
    const size_t req_bytes = (nreq * sizeof(ReqDev) + 31) & ~(size_t)31;
    KB_TRY(dbuf_ensure(ctx, ctx->d_reqs, req_bytes + std::max<size_t>(nt, 1) * sizeof(TileDev) + 64));
    ctx->d_tiles.p = (uint8_t *)ctx->d_reqs.p + req_bytes;  // alias into d_reqs (never freed on its own)
    ctx->d_tiles.cap = 0;
    KB_TRY(dbuf_ensure(ctx, ctx->d_tgt, std::max<uint64_t>(R.total_flat, 4) * 4 + nreq * 4 + 16));
    // one zeroed region per batch: [ticket, padded to 64 bytes][one ChunkState per 1024 tiles][one TileState per tile]
    KB_TRY(dbuf_ensure(ctx, ctx->d_tscan, 64 + (std::max<size_t>(nt, 1) / 1024 + 1) * sizeof(ChunkState) +
                                              std::max<size_t>(nt, 1) * sizeof(TileState)));
    KB_TRY(dbuf_ensure(ctx, ctx->d_tcnt, (std::max<size_t>(nt, 1) * 2 + (nt + 1) * 2) * 8));  // tcnt | tscan
    KB_TRY(dbuf_ensure(ctx, ctx->d_reqout, std::max<size_t>(nreq, 1) * sizeof(ReqOut)));
    // pinned staging so the async copies really are asynchronous
    const size_t bytes = nreq * sizeof(ReqDev);
    KB_TRY(hbuf_ensure(ctx, ctx->h_stage2, bytes + 64));
    uint8_t *h = (uint8_t *)ctx->h_stage2.p;
    memcpy(h, R.reqs.data(), bytes);
    if (bytes) KB_CUDA(ctx, cudaMemcpyAsync(ctx->d_reqs.p, h, bytes, cudaMemcpyHostToDevice, ctx->stream));
    if (nt)
        KB_LAUNCH(ctx, "k_fill_tiles", nt * 32,
                  (k_fill_tiles<<<(unsigned)((nt + 255) / 256), 256, 0, ctx->stream>>>((const ReqDev *)ctx->d_reqs.p, (uint32_t)nreq,
                                                                                        (uint32_t)nt, (TileDev *)ctx->d_tiles.p)));
    return KB_OK;
}

}  // namespace

// bulk-TMA gather of `n_jobs` (upper bound) copy jobs into `arena`
static int launch_gather(kb_ctx *ctx, cudaStream_t strm, const GatherJob *d_jobs, const uint64_t *d_njobs,
                         unsigned long long *d_ctr, uint4 *arena, uint64_t n_jobs, uint64_t alg_bytes)
{
    uint32_t piece, stages;
    gather_geometry(ctx->max_kv_chunks, &piece, &stages);
    const size_t gsmem = (size_t)GATHER_WARPS * stages * piece * 16;
    if (!ctx->gather_attr_set) {
        KB_CUDA(ctx, cudaFuncSetAttribute(k_gather, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)(GATHER_WARPS * GATHER_WARP_CHUNKS * 16)));
        ctx->gather_attr_set = true;
    }
    static const unsigned per_sm = getenv("KB_GATHER_CTAS") ? (unsigned)std::max(1, atoi(getenv("KB_GATHER_CTAS"))) : 2;  // experiment knob
    const unsigned ggrid =
        (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((n_jobs + GATHER_WARPS * 32 - 1) / (GATHER_WARPS * 32), per_sm * 148));
    KB_LAUNCH_S(ctx, strm, "k_gather", alg_bytes,
                (k_gather<<<ggrid, GATHER_WARPS * 32, gsmem, strm>>>(ctx->st, d_jobs, d_njobs, arena, piece, stages, d_ctr,
                                                                     (unsigned int *)ctx->d_ctrs.p + 8)));
    return KB_OK;
}

// emit -> tile scan -> request totals -> (place) for an uploaded layout; everything stays enqueued on
// ctx->stream.  Range: the selection goes to ctx->d_sel / d_slot; compact: the delete calls go to vidx / vcls.
static int launch_scan_core(kb_ctx *ctx, const Resolved &R, const ScanMode &mode, bool with_place,
                            uint32_t *vidx = nullptr, uint8_t *vcls = nullptr)
{
    const uint32_t nt = R.nt;
    const uint32_t nreq = (uint32_t)R.reqs.size();
    const ReqDev *d_reqs = (const ReqDev *)ctx->d_reqs.p;
    const TileDev *d_tiles = (const TileDev *)ctx->d_tiles.p;
    uint32_t *d_tgt = (uint32_t *)ctx->d_tgt.p;
    uint32_t *d_tail = d_tgt + std::max<uint64_t>(R.total_flat, 4);
    const uint32_t nchunks = nt / 1024 + 1;
    unsigned int *d_ticket = (unsigned int *)ctx->d_tscan.p;
    ChunkState *d_cs = (ChunkState *)((uint8_t *)ctx->d_tscan.p + 64);
    TileState *d_ts = (TileState *)(d_cs + nchunks);
    uint64_t *d_tcnt = (uint64_t *)ctx->d_tcnt.p, *d_tscan = d_tcnt + (size_t)std::max<uint32_t>(nt, 1) * 2;
    ReqOut *d_rout = (ReqOut *)ctx->d_reqout.p;
    if (nt) {
        // the ticket and the look-back states start empty
        KB_CUDA(ctx, cudaMemsetAsync(ctx->d_tscan.p, 0, 64 + (size_t)nchunks * sizeof(ChunkState) + (size_t)nt * sizeof(TileState),
                                     ctx->stream));
        // per record: 12 bytes of decoded columns read, the 4-byte target written
        if (mode.compact) {
            KB_LAUNCH(ctx, "k_emit_compact", R.n_records * 16,
                      (k_emit<true><<<nt, 256, 0, ctx->stream>>>(ctx->st, mode, d_reqs, d_tiles, d_ts, d_ticket, d_tgt, d_tail,
                                                                d_tcnt)));
        } else {
            KB_LAUNCH(ctx, "k_emit", R.n_records * 16,
                      (k_emit<false><<<nt, 256, 0, ctx->stream>>>(ctx->st, mode, d_reqs, d_tiles, d_ts, d_ticket, d_tgt, d_tail,
                                                                 d_tcnt)));
        }
        KB_LAUNCH(ctx, "k_tile_scan", (uint64_t)nt * 32,
                  (k_tile_scan<<<nchunks, 256, 0, ctx->stream>>>(d_tcnt, d_tscan, nt, d_cs)));
    }
    if (nreq)
        KB_LAUNCH(ctx, "k_req_totals", (uint64_t)nreq * 64,
                  (k_req_totals<<<(nreq + 255) / 256, 256, 0, ctx->stream>>>(d_reqs, nreq, d_tscan, d_rout)));
    if (nt && with_place) {
        if (mode.compact) {
            KB_LAUNCH(ctx, "k_place_victims", R.n_records * 16,  // columns + targets (the victims are written on top)
                      (k_place_victims<<<nt, 256, 0, ctx->stream>>>(ctx->st, mode, d_reqs, d_tiles, d_tgt, d_tscan, vidx, vcls)));
        } else {
            KB_LAUNCH(ctx, "k_place", R.n_records * 4,
                      (k_place<<<nt, 256, 0, ctx->stream>>>(ctx->st, d_reqs, d_tiles, d_tgt, d_tail, d_tscan,
                                                            (uint32_t *)ctx->d_sel.p, (uint64_t *)ctx->d_slot.p, d_rout,
                                                            mode.wire)));
        }
    }
    KB_CUDA(ctx, cudaGetLastError());
    return KB_OK;
}

// `limit` requests over intervals much larger than the limit: find how far the reference's loop would read
// (worker.run stops pulling from the iterator once the receiver is full, scanner.go:416 / receiver.go:82-87) by
// scanning geometrically growing windows, then clip the request to exactly those records.  The final pass then
// sees what the reference saw, with work proportional to the answer instead of to the interval.
constexpr uint32_t KB_LIMIT_WINDOW_MIN = 8192;

// *reused: the probe pass WAS the final pass (every request of the batch was probed, all of them were settled by the first
// window, padded-arena sizes): its selection and request rows are already on the device, the caller skips its own scan
static int probe_limit_windows(kb_ctx *ctx, Resolved &R, int wire, bool *reused)
{
    *reused = false;
    struct Todo {
        uint32_t q, true_hi;
        uint64_t w;
    };
    std::vector<Todo> todo;
    for (uint32_t q = 0; q < R.reqs.size(); q++) {
        const ReqDev &r = R.reqs[q];
        if (r.limit <= 0) continue;
        uint64_t w0 = std::max<uint64_t>(KB_LIMIT_WINDOW_MIN, (uint64_t)r.limit * 8);
        w0 = (w0 + KB_TILE - 1) / KB_TILE * KB_TILE;
        if ((uint64_t)(r.hi - r.lo) > w0) todo.push_back(Todo{q, r.hi, w0});
    }
    if (todo.empty()) return KB_OK;
    ScanMode mode;
    mode.compact = 0;
    mode.ttl_scan = 0;
    mode.timeout_rev = 0;
    mode.wire = 0;
    for (int round = 0; !todo.empty(); round++) {
        Resolved P;
        P.reqs.resize(todo.size());
        for (size_t i = 0; i < todo.size(); i++) {
            P.reqs[i] = R.reqs[todo[i].q];
            P.reqs[i].hi = (uint32_t)std::min<uint64_t>(todo[i].true_hi, (uint64_t)P.reqs[i].lo + todo[i].w);
        }
        KB_TRY(layout_requests(ctx, true, P));
        KB_TRY(upload_layout(ctx, P));
        KB_TRY(dbuf_ensure(ctx, ctx->d_sel, std::max<uint64_t>(P.total_sel, 1) * 4));
        KB_TRY(dbuf_ensure(ctx, ctx->d_slot, std::max<uint64_t>(P.total_sel, 1) * 8));
        KB_TRY(launch_scan_core(ctx, P, mode, true));
        KB_TRY(hbuf_ensure(ctx, ctx->h_stage, P.reqs.size() * sizeof(ReqOut) + 64));
        KB_CUDA(ctx, cudaMemcpyAsync(ctx->h_stage.p, ctx->d_reqout.p, P.reqs.size() * sizeof(ReqOut),
                                     cudaMemcpyDeviceToHost, ctx->stream));
        KB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        const ReqOut *ro = (const ReqOut *)ctx->h_stage.p;
        std::vector<Todo> next;
        for (size_t i = 0; i < todo.size(); i++) {
            ReqDev &r = R.reqs[todo[i].q];
            if (ro[i].flags & KB_RO_LIMIT_STOP)
                r.hi = r.lo + ro[i].examined;  // exactly the records the reference's loop pulled
            else if (P.reqs[i].hi != todo[i].true_hi)
                next.push_back(Todo{todo[i].q, todo[i].true_hi, todo[i].w * 8});
            // else: the whole interval was examined and the limit was not reached inside the loop
        }
        if (round == 0 && next.empty() && wire == 0 && todo.size() == R.reqs.size()) {
            // every request of the batch sits in P in the same order; for a request the limit stopped, the window holds
            // more records than the reference's loop pulled, but the first `limit` emissions, the bytes of those and the
            // examined count (all in its request row) are the ones the clipped scan would produce
            R = P;
            *reused = true;
            return KB_OK;
        }
        todo.swap(next);
    }
    return layout_requests(ctx, true, R);
}

static_assert(sizeof(ReqOut) == 32, "publish_rout copies ReqOut rows as two 16-byte words");

static int rout_map_ensure(kb_ctx *ctx, uint64_t nreq)
{
    const size_t need = 64 + std::max<uint64_t>(nreq, 1) * sizeof(ReqOut);
    if (ctx->h_rout && ctx->h_rout_cap >= need) return KB_OK;
    if (ctx->h_rout) {
        KB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        cudaFreeHost(ctx->h_rout);
        ctx->h_rout = nullptr;
        ctx->h_rout_cap = 0;
    }
    const size_t cap = need + need / 2;
    KB_CUDA(ctx, cudaHostAlloc((void **)&ctx->h_rout, cap, cudaHostAllocMapped));
    memset(ctx->h_rout, 0, cap);
    ctx->h_rout_cap = cap;
    return KB_OK;
}

// wait until the device has published the rows of `epoch`; the stream is only consulted now and then, to notice a
// failed launch or kernel instead of spinning forever
static int rout_wait(kb_ctx *ctx, const uint8_t *h_rout, cudaStream_t strm, uint64_t epoch)
{
    volatile const uint64_t *flag = (volatile const uint64_t *)h_rout;
    for (uint64_t spins = 1;; spins++) {
        if (*flag == epoch) return KB_OK;
        kb_cpu_relax();
        if ((spins & 0xFFFF) == 0) {
            const cudaError_t q = cudaStreamQuery(strm);
            if (q == cudaSuccess) return *flag == epoch ? KB_OK : kb_fail(ctx, KB_ECUDA, "range scan: results were not published");
            if (q != cudaErrorNotReady) return kb_cuda_fail(ctx, q, "range scan");
        }
    }
}

// a range batch between its submission and the collection of its answer
struct kb_pending {
    int lane = 0;
    Resolved R;
    uint64_t nreq = 0;
    int out_mode = 0, wire = 0;
    bool want_kvs = false;
    kb_result *res = nullptr;
    DBuf d_om;
    GatherOut go;
    uint64_t *d_elem_off = nullptr;
    uint64_t epoch = 0;
    const uint8_t *h_rout = nullptr;  // the lane's mapped row buffer and stream at submission time
    cudaStream_t stream = nullptr;
    kb_tp t_submit;
    std::vector<ReqOut> rout;         // rows, once read back
    bool harvested = false;
    int harvest_rc = KB_OK;
};
static int pending_harvest(kb_ctx *ctx, kb_pending *P);

// first half of a range call: everything up to the launch of the last kernel; the batch is then in flight on the current lane
static int range_submit_locked(kb_ctx *ctx, const kb_range_req *reqs, uint64_t nreq, int out_mode, kb_pending **out)
{
    // wire modes: the arena holds etcd protobuf elements instead of padded [key][value] pairs (kb_wire.cuh)
    const int wire_flags = out_mode & (KB_WIRE_ETCD_KVS | KB_WIRE_ETCD_EVENTS);
    out_mode &= ~(KB_WIRE_ETCD_KVS | KB_WIRE_ETCD_EVENTS);
    if (out_mode != KB_OUT_HOST && out_mode != KB_OUT_DEVICE && out_mode != KB_OUT_COUNT) return KB_EINVAL;
    if (wire_flags == (KB_WIRE_ETCD_KVS | KB_WIRE_ETCD_EVENTS) || (wire_flags && out_mode == KB_OUT_COUNT)) return KB_EINVAL;
    const int wire = wire_flags == KB_WIRE_ETCD_KVS ? KB_WIRE_KVS_I : wire_flags == KB_WIRE_ETCD_EVENTS ? KB_WIRE_EVENTS_I : 0;
    *out = nullptr;
    if (!ctx->loaded) return kb_fail(ctx, KB_ESTATE, "no store loaded");
    cudaSetDevice(ctx->device);
    // this lane's previous batch still owns the lane's host-visible buffers until its rows have been read back
    if (ctx->lane_pending[ctx->lane]) KB_TRY(pending_harvest(ctx, ctx->lane_pending[ctx->lane]));
    for (uint64_t q = 0; q < nreq; q++) {
        // checkCompactRace (scanner.go:594-626)
        if (ctx->compact_present && ctx->compact_rev > reqs[q].read_rev)
            return kb_fail(ctx, KB_ECOMPACTED, "range stream revision %llu less than compact revision %llu",
                           (unsigned long long)reqs[q].read_rev, (unsigned long long)ctx->compact_rev);
    }
    kb_tp tseg = kb_now();
    std::unique_ptr<kb_pending> P(new kb_pending());
    Resolved &R = P->R;
    KB_TRY(resolve_requests(ctx, reqs, nreq, true, R, &tseg));
    kb_seg(ctx, "host:range_layout", tseg);
    bool probe_is_final = false;
    if (out_mode != KB_OUT_COUNT) {
        KB_TRY(probe_limit_windows(ctx, R, wire, &probe_is_final));
        kb_seg(ctx, "host:range_limit_probe", tseg);
    }
    if (!probe_is_final) {
        KB_TRY(upload_layout(ctx, R));
        KB_TRY(dbuf_ensure(ctx, ctx->d_sel, std::max<uint64_t>(R.total_sel, 1) * 4));
        KB_TRY(dbuf_ensure(ctx, ctx->d_slot, std::max<uint64_t>(R.total_sel, 1) * 8));
    }
    const ReqDev *d_reqs = (const ReqDev *)ctx->d_reqs.p;
    ReqOut *d_rout = (ReqOut *)ctx->d_reqout.p;
    ScanMode mode;
    mode.compact = 0;
    mode.ttl_scan = 0;
    mode.timeout_rev = 0;
    mode.wire = wire;
    if (!probe_is_final) KB_TRY(launch_scan_core(ctx, R, mode, out_mode != KB_OUT_COUNT));
    KB_TRY(rout_map_ensure(ctx, nreq));
    const uint64_t epoch = ++ctx->rout_epoch;

    // Response arena: sized by an upper bound the host knows without a round trip (all key+value bytes of the examined
    // record intervals), so the gather is enqueued right behind the placement and the only synchronisation left is
    // the final one (the arena is pooled, so steady-state calls reuse it).
    const bool want_kvs = out_mode != KB_OUT_COUNT && R.total_sel > 0;
    // (a heap has no "bytes of an interval": every examined record could be emitted with the store's largest pair, and
    // no answer can exceed one copy of everything per request that could return it all)
    uint64_t ub_bytes = 0;
    for (auto &r : R.reqs) {
        uint64_t cap = (uint64_t)(r.hi - r.lo);
        if (r.limit > 0) cap = std::min<uint64_t>(cap, (uint64_t)r.limit);
        ub_bytes += std::min<uint64_t>(cap * ctx->max_kv_chunks, ctx->kused16 + ctx->vused16) * 16;
    }
    // a wire element is at most 48 bytes of tags / varints longer than its key + value (and the key loses 13)
    if (wire) ub_bytes += (uint64_t)R.total_sel * 48;
    kb_result *res = kb_result_new(1, out_mode);
    res->wire = wire;
    DBuf d_om;
    // every early return below hands the pooled buffers back (the stream keeps later reuse ordered behind this call)
    struct Guard {
        kb_ctx *ctx;
        kb_result *&res;
        DBuf &d_om;
        bool armed = true;
        ~Guard()
        {
            if (!armed) return;
            pool_put_dev(ctx, d_om);
            result_release_locked(ctx, res);
        }
    } guard{ctx, res, d_om};
    GatherOut go;
    memset(&go, 0, sizeof(go));
    const uint64_t cap_kvs = R.total_sel;
    uint64_t *d_elem_off = nullptr;
    const size_t meta_cap = cap_kvs * (wire ? 44 : 36) + 64 + 8;
    int rc = KB_OK;
    // The copy into the arena runs on the gather stream.  Consecutive batches alternate between two sets of job
    // buffers, so this batch's job construction (main stream) may overlap the previous batch's copy; it only has to
    // wait for the copy that last READ this set (two batches ago).
    const int set = (int)(ctx->batch_seq++ & 1);
    DBuf &jb = set ? ctx->d_jobs2 : ctx->d_jobs;
    DBuf &gb = set ? ctx->d_gjobs2 : ctx->d_gjobs;
    cudaStream_t sg = ctx->stream_g;
    if (want_kvs) {
        rc = pool_get_dev(ctx, meta_cap, &d_om);
        if (rc == KB_OK) rc = pool_get_arena(ctx, ub_bytes + 64, &res->d_bytes);
        if (rc == KB_OK) rc = dbuf_ensure(ctx, jb, (nreq + 1) * 16 + 8);
        if (rc == KB_OK)
            rc = dbuf_ensure(ctx, gb, std::max<uint64_t>(cap_kvs, 1) * (wire ? sizeof(WireJob) : sizeof(GatherJob)));
        if (rc != KB_OK) return rc;
        uint8_t *om = (uint8_t *)d_om.p;
        go.rev = (uint64_t *)om;
        go.key_off = go.rev + cap_kvs;
        go.val_off = go.key_off + cap_kvs;
        d_elem_off = go.val_off + cap_kvs;  // wire modes only: cap_kvs + 1 entries
        go.rec_idx = (uint32_t *)(wire ? d_elem_off + cap_kvs + 1 : d_elem_off);
        go.key_len = go.rec_idx + cap_kvs;
        go.val_len = go.key_len + cap_kvs;
        uint64_t *d_jobfirst = (uint64_t *)jb.p, *d_arenabase = d_jobfirst + nreq + 1;
        unsigned long long *d_workctr = (unsigned long long *)(d_arenabase + nreq + 1);  // zeroed by k_req_finalize
        KB_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_gather[set], 0));
        KB_LAUNCH(ctx, "k_req_finalize", nreq * 64,
                  (k_req_finalize<<<1, 256, 0, ctx->stream>>>(d_reqs, (uint32_t)nreq, d_rout, d_jobfirst, d_arenabase,
                                                              d_workctr, ctx->h_rout, epoch,
                                                              (const unsigned int *)ctx->d_ctrs.p + 8)));
        const unsigned jgrid = (unsigned)std::min<uint64_t>((cap_kvs + 255) / 256, 148 * 8);
        if (wire) {
            WireOut wo;
            wo.rec_idx = go.rec_idx;
            wo.rev = go.rev;
            wo.key_off = go.key_off;
            wo.key_len = go.key_len;
            wo.val_off = go.val_off;
            wo.val_len = go.val_len;
            wo.elem_off = d_elem_off;
            WireJob *d_wj = (WireJob *)gb.p;
            KB_LAUNCH(ctx, "k_wire_jobs", cap_kvs * 20,
                      (k_wire_jobs<<<jgrid, 256, 0, ctx->stream>>>(ctx->st, d_reqs, (uint32_t)nreq, d_jobfirst, d_arenabase,
                                                                  (const uint32_t *)ctx->d_sel.p,
                                                                  (const uint64_t *)ctx->d_slot.p, wire, d_wj, wo)));
            KB_CUDA(ctx, cudaEventRecord(ctx->ev_jobs, ctx->stream));
            KB_CUDA(ctx, cudaStreamWaitEvent(sg, ctx->ev_jobs, 0));
            uint32_t slot_chunks, wstages;
            wire_geometry(ctx->max_kv_chunks, &slot_chunks, &wstages);
            const size_t wsmem = (size_t)WIRE_WARPS * wstages * slot_chunks * 16;
            if (!ctx->wire_attr_set) {
                cudaFuncSetAttribute(k_wire_copy, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)(WIRE_WARPS * WIRE_WARP_CHUNKS * 16));
                ctx->wire_attr_set = true;
            }
            const unsigned wgrid =
                (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((cap_kvs + WIRE_WARPS - 1) / WIRE_WARPS, 2 * 148));
            KB_LAUNCH_S(ctx, sg, "k_wire_copy", 0,
                        (k_wire_copy<<<wgrid, WIRE_WARPS * 32, wsmem, sg>>>(ctx->st, d_wj, d_jobfirst + nreq,
                                                                          (uint8_t *)res->d_bytes.p, slot_chunks, wstages,
                                                                          (unsigned int *)ctx->d_ctrs.p + 8)));
        } else {
            GatherJob *d_gj = (GatherJob *)gb.p;
            KB_LAUNCH(ctx, "k_gather_jobs", cap_kvs * 20,
                      (k_gather_jobs<<<jgrid, 256, 0, ctx->stream>>>(ctx->st, d_reqs, (uint32_t)nreq, d_jobfirst, d_arenabase,
                                                                    (const uint32_t *)ctx->d_sel.p,
                                                                    (const uint64_t *)ctx->d_slot.p, d_gj, go)));
            KB_CUDA(ctx, cudaEventRecord(ctx->ev_jobs, ctx->stream));
            KB_CUDA(ctx, cudaStreamWaitEvent(sg, ctx->ev_jobs, 0));
            KB_TRY(launch_gather(ctx, sg, d_gj, d_jobfirst + nreq, d_workctr, (uint4 *)res->d_bytes.p, cap_kvs, 0));
        }
        KB_CUDA(ctx, cudaEventRecord(ctx->ev_gather[set], sg));
        // the answer is complete when this event has fired (kb_result_wait, kb_sync)
        res->done_ev = nullptr;
        if (!ctx->ev_pool.empty()) {
            res->done_ev = ctx->ev_pool.back();
            ctx->ev_pool.pop_back();
        } else {
            KB_CUDA(ctx, cudaEventCreate(&res->done_ev));
        }
        KB_CUDA(ctx, cudaEventRecord(res->done_ev, sg));
    }
    if (!want_kvs && nreq) {  // count-only / empty answers: nothing ran k_req_finalize, publish the rows directly
        KB_LAUNCH(ctx, "k_publish_rout", nreq * 32,
                  (k_publish_rout<<<1, 256, 0, ctx->stream>>>(d_rout, (uint32_t)nreq, ctx->h_rout, epoch,
                                                              (const unsigned int *)ctx->d_ctrs.p + 8)));
    }
    kb_seg(ctx, "host:range_launch", tseg);
    guard.armed = false;
    P->lane = ctx->lane;
    P->nreq = nreq;
    P->out_mode = out_mode;
    P->wire = wire;
    P->want_kvs = want_kvs;
    P->res = res;
    P->d_om = d_om;
    P->go = go;
    P->d_elem_off = d_elem_off;
    P->epoch = epoch;
    P->h_rout = ctx->h_rout;
    P->stream = ctx->stream;
    P->t_submit = tseg;
    ctx->lane_pending[ctx->lane] = P.get();
    *out = P.release();
    return KB_OK;
}

// wait for the rows of a submitted batch and keep them with it: afterwards the lane's buffers are free again
static int pending_harvest(kb_ctx *ctx, kb_pending *P)
{
    if (P->harvested) return P->harvest_rc;
    P->harvested = true;
    if (ctx->lane_pending[P->lane] == P) ctx->lane_pending[P->lane] = nullptr;
    P->rout.resize(std::max<uint64_t>(P->nreq, 1));
    if (P->nreq) {
        P->harvest_rc = rout_wait(ctx, P->h_rout, P->stream, P->epoch);
        if (P->harvest_rc != KB_OK) return P->harvest_rc;
        memcpy(P->rout.data(), P->h_rout + 64, P->nreq * sizeof(ReqOut));
        if (*(volatile uint64_t *)(P->h_rout + 8) != 0)
            return P->harvest_rc = kb_fail(ctx, KB_ECUDA, "range scan: a bulk copy of the answer never completed");
    }
    return KB_OK;
}

int kb_pending_harvest_all(kb_ctx *ctx)
{
    for (int l = 0; l < KB_MAX_LANES; l++)
        if (ctx->lane_pending[l]) KB_TRY(pending_harvest(ctx, ctx->lane_pending[l]));
    return KB_OK;
}

static void pending_drop(kb_ctx *ctx, kb_pending *P)
{
    if (ctx->lane_pending[P->lane] == P) ctx->lane_pending[P->lane] = nullptr;
    pool_put_dev(ctx, P->d_om);
    result_release_locked(ctx, P->res);
    delete P;
}

void kb_pending_drop_all(kb_ctx *ctx)  // kb_close: batches nobody collected
{
    for (int l = 0; l < KB_MAX_LANES; l++)
        if (kb_pending *P = ctx->lane_pending[l]) {
            pending_harvest(ctx, P);
            pending_drop(ctx, P);
        }
}

// second half: rows -> the result's per-request arrays, host copies for KB_OUT_HOST
static int range_collect_locked(kb_ctx *ctx, kb_pending *P, kb_result **out)
{
    *out = nullptr;
    cudaSetDevice(ctx->device);
    const uint64_t nreq = P->nreq;
    const int out_mode = P->out_mode, wire = P->wire;
    const bool want_kvs = P->want_kvs;
    Resolved &R = P->R;
    kb_result *res = P->res;
    DBuf &d_om = P->d_om;
    GatherOut &go = P->go;
    uint64_t *d_elem_off = P->d_elem_off;
    kb_tp tseg = kb_now();
    struct Guard {  // every return below ends the batch: a failed one hands its buffers back
        kb_ctx *ctx;
        kb_pending *P;
        bool armed = true;
        ~Guard()
        {
            if (armed) pending_drop(ctx, P);
        }
    } guard{ctx, P};
    int rc = pending_harvest(ctx, P);
    if (rc != KB_OK) return rc;
    std::vector<ReqOut> &rout = P->rout;
    cudaStream_t sg = ctx->stream_g;
    kb_seg(ctx, "host:range_sync", tseg);

    res->req_first.resize(nreq + 1);
    res->req_count.resize(nreq);
    res->req_examined.resize(nreq);
    uint64_t nk = 0, nbytes = 0;
    for (uint64_t q = 0; q < nreq; q++) {
        uint64_t ne = rout[q].total;
        bool capped = R.reqs[q].limit > 0 && ne > (uint64_t)R.reqs[q].limit;
        if (capped) ne = (uint64_t)R.reqs[q].limit;
        res->req_first[q] = nk;
        if (out_mode == KB_OUT_COUNT) {
            res->req_count[q] = rout[q].total;  // emptyResultReceiver never stops the loop
            res->req_examined[q] = R.reqs[q].hi - R.reqs[q].lo;
        } else {
            const bool stop = rout[q].flags & KB_RO_LIMIT_STOP;
            res->req_count[q] = stop ? 0 : ne;  // (0, nil) when the limit stopped the loop (Q4)
            res->req_examined[q] = stop ? rout[q].examined : R.reqs[q].hi - R.reqs[q].lo;
            nk += ne;
            nbytes += (R.reqs[q].limit > 0 && (rout[q].flags & KB_RO_CAPPED)) ? rout[q].capped_aux : rout[q].total_aux;
        }
    }
    res->req_first[nreq] = nk;
    res->n_kvs = nk;
    res->n_bytes = nbytes;
    if (ctx->prof_on) {  // the gather's algorithmic bytes are only known now
        int gi = prof_index(ctx, wire ? "k_wire_copy" : "k_gather");
        ctx->prof[gi].bytes += 2 * nbytes + nk * 40;
    }

    if (want_kvs && nk > 0) {
        if (out_mode == KB_OUT_HOST) {
            // per-kv arrays: six strided pieces of the capacity-sized device layout -> one compact host layout
            rc = pool_get_host(ctx, nk * 44 + 64 + 8, &res->h_meta);
            if (rc == KB_OK) rc = pool_get_host(ctx, nbytes + 16, &res->h_bytes);
            if (rc == KB_OK) {
                uint8_t *hm = (uint8_t *)res->h_meta.p;
                const void *srcs[7] = {go.rev, go.key_off, go.val_off, d_elem_off, go.rec_idx, go.key_len, go.val_len};
                const size_t cnt[7] = {nk, nk, nk, wire ? nk + 1 : 0, nk, nk, nk};
                const size_t esz[7] = {8, 8, 8, 8, 4, 4, 4};
                size_t off = 0;
                // on the host-copy stream, behind this batch's gather: a later batch's gather (already queued on the copy
                // stream when batches are submitted ahead) does not sit between the answer and the host
                cudaStream_t sh = ctx->stream_h;
                if (res->done_ev) cudaStreamWaitEvent(sh, res->done_ev, 0);
                for (int i = 0; i < 7; i++) {
                    if (cnt[i]) cudaMemcpyAsync(hm + off, srcs[i], cnt[i] * esz[i], cudaMemcpyDeviceToHost, sh);
                    off += cnt[i] * esz[i];
                }
                cudaMemcpyAsync(res->h_bytes.p, res->d_bytes.p, nbytes, cudaMemcpyDeviceToHost, sh);
            }
            cudaError_t e = cudaStreamSynchronize(ctx->stream_h);  // behind the gather (which waited for the per-kv arrays)
            kb_seg(ctx, "host:range_d2h", tseg);
            if (rc == KB_OK && e != cudaSuccess) rc = kb_cuda_fail(ctx, e, "range D2H");
            if (rc != KB_OK) return rc;
            uint8_t *hm = (uint8_t *)res->h_meta.p;
            res->rev = (const uint64_t *)hm;
            res->key_off = res->rev + nk;
            res->val_off = res->key_off + nk;
            res->elem_off = wire ? res->val_off + nk : nullptr;
            res->rec_idx = (const uint32_t *)(res->val_off + nk + (wire ? nk + 1 : 0));
            res->key_len = res->rec_idx + nk;
            res->val_len = res->key_len + nk;
            pool_put_dev(ctx, d_om);
            d_om = DBuf();
            pool_put_arena(ctx, res->d_bytes);
            res->d_bytes = DBuf();
        } else {
            res->rev = go.rev;
            res->key_off = go.key_off;
            res->val_off = go.val_off;
            res->rec_idx = go.rec_idx;
            res->key_len = go.key_len;
            res->val_len = go.val_len;
            res->elem_off = wire ? d_elem_off : nullptr;
            res->d_vic = d_om;  // owned by the result (returned to the pool by kb_result_free)
            d_om = DBuf();
        }
    } else {
        pool_put_dev(ctx, d_om);
        d_om = DBuf();
        if (res->d_bytes.p) {
            pool_put_arena(ctx, res->d_bytes);
            res->d_bytes = DBuf();
        }
    }
    guard.armed = false;
    *out = res;
    delete P;
    kb_seg(ctx, "host:range_finish", tseg);
    return KB_OK;
}

extern "C" int kb_range_batch(kb_ctx *ctx, const kb_range_req *reqs, uint64_t nreq, int out_mode, kb_result **out)
{
    if (!ctx || !out || (nreq && !reqs)) return KB_EINVAL;
    *out = nullptr;
    std::lock_guard<std::mutex> g(ctx->mu);
    kb_pending *P = nullptr;
    KB_TRY(range_submit_locked(ctx, reqs, nreq, out_mode, &P));
    return range_collect_locked(ctx, P, out);
}

// The two halves on their own: a caller with a queue of batches submits batch n+1 before it collects batch n, so the
// host's part of n+1 (bound search round trip, layout, launches) and its first kernels overlap the kernels of n.  Each
// submission leaves its batch on the current lane and moves the context to the other one; two batches in flight at most
// (a third submission first reads back the rows of the batch that last used its lane).
extern "C" int kb_range_submit(kb_ctx *ctx, const kb_range_req *reqs, uint64_t nreq, int out_mode, kb_pending **out)
{
    if (!ctx || !out || (nreq && !reqs)) return KB_EINVAL;
    *out = nullptr;
    std::lock_guard<std::mutex> g(ctx->mu);
    KB_TRY(range_submit_locked(ctx, reqs, nreq, out_mode, out));
    lane_swap(ctx);
    return KB_OK;
}

extern "C" int kb_range_collect(kb_ctx *ctx, kb_pending *pending, kb_result **out)
{
    if (!ctx || !pending || !out) return KB_EINVAL;
    std::lock_guard<std::mutex> g(ctx->mu);
    return range_collect_locked(ctx, pending, out);
}

// give up a submitted batch without reading its answer
extern "C" void kb_pending_free(kb_ctx *ctx, kb_pending *pending)
{
    if (!ctx || !pending) return;
    std::lock_guard<std::mutex> g(ctx->mu);
    cudaSetDevice(ctx->device);
    pending_harvest(ctx, pending);  // its kernels must be done before its buffers go back to the pools
    pending_drop(ctx, pending);
}

// Start the bound search of a batch that a later kb_range_batch will ask for (same bounds, same snapshot): a caller with a
// queue of pending requests submits batch n+1 before it waits for batch n, so the search's host round trip (the one
// synchronisation a range call needs before it can lay its requests out) overlaps the previous batch's kernels.
extern "C" int kb_range_prefetch(kb_ctx *ctx, const kb_range_req *reqs, uint64_t nreq)
{
    if (!ctx || (nreq && !reqs)) return KB_EINVAL;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (!ctx->loaded) return kb_fail(ctx, KB_ESTATE, "no store loaded");
    cudaSetDevice(ctx->device);
    const int slot = (int)(ctx->prefetch_next++ & 1);
    kb_ctx::SearchSlot &sl = ctx->prefetch[slot];
    if (ctx->prof_on) {  // diagnostic: is the OTHER slot's (older) submission already complete when the next one is made?
        kb_ctx::SearchSlot &other = ctx->prefetch[slot ^ 1];
        if (other.valid && other.pub.host) {
            const bool ready = *(volatile uint64_t *)other.pub.host == other.pub.epoch;
            ctx->prof[prof_index(ctx, ready ? "host:prefetch_older_ready" : "host:prefetch_older_pending")].launches++;
        }
    }
    if (sl.valid) KB_TRY(search_wait(ctx, sl.pub, ctx->stream2));  // an unconsumed older submission still owns the buffers
    sl.valid = false;
    uint64_t chunks = 0;
    KB_TRY(pack_bounds(ctx, reqs, nreq, sl.stage, &chunks));
    KB_TRY(enqueue_search(ctx, sl.stage, sl.d_bounds, sl.d_bres, chunks, 2 * nreq, ctx->stream2, sl.pub, slot));
    sl.ident_bytes = chunks * 16 + 2 * nreq * 8;
    sl.store_gen = ctx->store_gen;
    sl.seq = ctx->prefetch_next;
    sl.valid = true;
    return KB_OK;
}

extern "C" int kb_result_wait(kb_ctx *ctx, const kb_result *res, void *cuda_stream)
{
    if (!ctx || !res) return KB_EINVAL;
    if (!res->done_ev) return KB_OK;
    cudaSetDevice(ctx->device);
    if (cuda_stream) {
        KB_CUDA(ctx, cudaStreamWaitEvent((cudaStream_t)cuda_stream, res->done_ev, 0));
    } else {
        KB_CUDA(ctx, cudaEventSynchronize(res->done_ev));
    }
    return KB_OK;
}

extern "C" int kb_range_view_get(const kb_result *res, kb_range_view *v)
{
    if (!res || !v || res->type != 1) return KB_EINVAL;
    memset(v, 0, sizeof(*v));
    v->n_req = res->req_count.size();
    v->req_first = res->req_first.data();
    v->req_count = res->req_count.data();
    v->req_examined = res->req_examined.data();
    v->n_kvs = res->n_kvs;
    v->rec_idx = res->rec_idx;
    v->rev = res->rev;
    v->key_off = res->key_off;
    v->key_len = res->key_len;
    v->val_off = res->val_off;
    v->val_len = res->val_len;
    v->n_bytes = res->n_bytes;
    v->elem_off = res->elem_off;
    v->wire = res->wire == KB_WIRE_KVS_I ? KB_WIRE_ETCD_KVS : res->wire == KB_WIRE_EVENTS_I ? KB_WIRE_ETCD_EVENTS : 0;
    v->on_device = res->out_mode == KB_OUT_DEVICE;
    v->bytes = res->out_mode == KB_OUT_DEVICE ? (const uint8_t *)res->d_bytes.p : (const uint8_t *)res->h_bytes.p;
    return KB_OK;
}

// ---- framing of the wire elements (host): etcdserverpb.ResponseHeader{revision} (pkg/server/etcd/kv.go:253-257) is
// field 1 of both responses; a header with revision 0 is still emitted (non-nil message of length 0)
static uint64_t host_put_varint(uint8_t *out, uint64_t v)
{
    uint64_t n = 0;
    while (v >= 0x80) {
        out[n++] = (uint8_t)(v | 0x80);
        v >>= 7;
    }
    out[n++] = (uint8_t)v;
    return n;
}

static uint64_t host_put_header(uint64_t header_rev, uint8_t *out)
{
    uint8_t body[12];
    uint64_t nb = 0;
    if (header_rev) {
        body[nb++] = 0x18;  // ResponseHeader.revision = 3, varint
        nb += host_put_varint(body + nb, header_rev);
    }
    uint64_t w = 0;
    out[w++] = 0x0a;  // field 1, length-delimited
    w += host_put_varint(out + w, nb);
    memcpy(out + w, body, nb);
    return w + nb;
}

extern "C" uint64_t kb_wire_range_head(uint64_t header_rev, uint8_t *out)
{
    return out ? host_put_header(header_rev, out) : 0;
}

extern "C" uint64_t kb_wire_range_tail(int more, int64_t count, uint8_t *out)
{
    if (!out) return 0;
    uint64_t w = 0;
    if (more) {  // RangeResponse.more = 3
        out[w++] = 0x18;
        out[w++] = 1;
    }
    if (count) {  // RangeResponse.count = 4
        out[w++] = 0x20;
        w += host_put_varint(out + w, (uint64_t)count);
    }
    return w;
}

extern "C" uint64_t kb_wire_watch_head(uint64_t header_rev, int canceled, const uint8_t *reason, uint64_t reason_len,
                                       uint8_t *out)
{
    if (!out || (reason_len && !reason)) return 0;
    uint64_t w = host_put_header(header_rev, out);
    if (canceled) {  // WatchResponse.canceled = 4
        out[w++] = 0x20;
        out[w++] = 1;
    }
    if (reason_len) {  // WatchResponse.cancel_reason = 6
        out[w++] = 0x32;
        w += host_put_varint(out + w, reason_len);
        memcpy(out + w, reason, reason_len);
        w += reason_len;
    }
    return w;
}

// ------------------------------------------------------------------------------------------------
// point reads
// ------------------------------------------------------------------------------------------------
extern "C" int kb_get_batch(kb_ctx *ctx, const kb_get_req *reqs, uint64_t n, int out_mode, kb_result **out)
{
    if (!ctx || !out || (n && !reqs)) return KB_EINVAL;
    if (out_mode != KB_OUT_HOST && out_mode != KB_OUT_DEVICE) return KB_EINVAL;
    *out = nullptr;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (!ctx->loaded) return kb_fail(ctx, KB_ESTATE, "no store loaded");
    cudaSetDevice(ctx->device);
    KB_TRY(ctx_quiesce(ctx));
    if (n >= 0x7FFFFFFFull) return kb_fail(ctx, KB_ELIMIT, "too many point reads in one batch");
    // bound of read i = EncodeObjectKey(key, revision or MaxUint64) + 0x00: its lower_bound is the first record
    // strictly greater than the start key of the reference's reverse iterator
    uint64_t chunks = 0;
    for (uint64_t i = 0; i < n; i++) {
        if (!reqs[i].key && reqs[i].key_len) return KB_EINVAL;
        if (reqs[i].key_len > 65000) return kb_fail(ctx, KB_ELIMIT, "key too long");
        chunks += (reqs[i].key_len + 14 + 15) / 16 + 3;
    }
    KB_TRY(hbuf_ensure(ctx, ctx->h_stage, chunks * 16 + n * 8 + n * 32 + 256));
    uint8_t *hs = (uint8_t *)ctx->h_stage.p;
    memset(hs, 0, chunks * 16);
    uint32_t *hboff = (uint32_t *)(hs + chunks * 16), *hblen = hboff + n;
    uint64_t c = 0;
    for (uint64_t i = 0; i < n; i++) {
        uint8_t *b = hs + c * 16;
        const uint64_t ul = reqs[i].key_len;
        const uint64_t rev = reqs[i].revision ? reqs[i].revision : ~0ull;
        b[0] = 0x57; b[1] = 0xfb; b[2] = 0x80; b[3] = 0x8b;
        if (ul) memcpy(b + 4, reqs[i].key, ul);
        b[4 + ul] = 0x24;
        for (int k = 0; k < 8; k++) b[5 + ul + k] = (uint8_t)(rev >> (8 * (7 - k)));
        b[13 + ul] = 0;
        hboff[i] = (uint32_t)c;
        hblen[i] = (uint32_t)(ul + 14);
        c += (ul + 14 + 15) / 16 + 3;
    }
    KB_TRY(dbuf_ensure(ctx, ctx->d_bounds, chunks * 16 + n * 8 + 64));
    KB_TRY(dbuf_ensure(ctx, ctx->d_bres, std::max<uint64_t>(n, 1) * 4));
    // per-read outputs on the device: [mod_rev u64][voff16 u64][rec u32][vlen u32][status u8]
    KB_TRY(dbuf_ensure(ctx, ctx->d_reqout, std::max<uint64_t>(n, 1) * 25 + 64));
    KB_CUDA(ctx, cudaMemcpyAsync(ctx->d_bounds.p, hs, chunks * 16 + n * 8, cudaMemcpyHostToDevice, ctx->stream));
    const uint32_t *d_boff = (const uint32_t *)((const uint8_t *)ctx->d_bounds.p + chunks * 16);
    GetOut go;
    go.mod_rev = (uint64_t *)ctx->d_reqout.p;
    go.voff16 = go.mod_rev + n;
    go.rec = (uint32_t *)(go.voff16 + n);
    go.vlen = go.rec + n;
    go.status = (uint8_t *)(go.vlen + n);
    if (n) {
        KB_LAUNCH(ctx, "k_search", n * 64,
                  (k_search<<<(unsigned)((n * 32 + 127) / 128), 128, 0, ctx->stream>>>(
                      ctx->st, (const uint4 *)ctx->d_bounds.p, d_boff, d_boff + n, (uint32_t)n, (uint32_t *)ctx->d_bres.p, SearchPub{nullptr, nullptr, 0})));
        KB_LAUNCH(ctx, "k_get_resolve", n * 320,
                  (k_get_resolve<<<(unsigned)((n * 32 + 127) / 128), 128, 0, ctx->stream>>>(
                      ctx->st, (const uint4 *)ctx->d_bounds.p, d_boff, d_boff + n, (const uint32_t *)ctx->d_bres.p,
                      (uint32_t)n, go)));
    }
    // host copy of the per-read outputs (same layout), behind the staging area used above
    kb_result *res = kb_result_new(4, out_mode);
    res->n_gets = n;
    const size_t st_off = (n + 7) & ~(size_t)7;  // h_get: [status (padded to 8)][mod_rev][val_off][rec][val_len]
    int rc = pool_get_host(ctx, st_off + n * 24 + 64, &res->h_get);
    if (rc != KB_OK) {
        result_release_locked(ctx, res);
        return rc;
    }
    uint8_t *hg = (uint8_t *)res->h_get.p;
    uint8_t *h_status = hg;
    uint64_t *h_mrev = (uint64_t *)(hg + st_off), *h_voff = h_mrev + n;
    uint32_t *h_rec = (uint32_t *)(h_voff + n), *h_vlen = h_rec + n;
    if (n) {
        cudaMemcpyAsync(h_voff, go.voff16, n * 8, cudaMemcpyDeviceToHost, ctx->stream);  // slab chunk; rewritten below
        cudaMemcpyAsync(h_mrev, go.mod_rev, n * 8, cudaMemcpyDeviceToHost, ctx->stream);
        cudaMemcpyAsync(h_rec, go.rec, n * 4, cudaMemcpyDeviceToHost, ctx->stream);
        cudaMemcpyAsync(h_vlen, go.vlen, n * 4, cudaMemcpyDeviceToHost, ctx->stream);
        cudaMemcpyAsync(h_status, go.status, n, cudaMemcpyDeviceToHost, ctx->stream);
    }
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        result_release_locked(ctx, res);
        return kb_cuda_fail(ctx, e, "get resolve");
    }
    // copy jobs for the found values (host side: offsets come from the host copies of the directory)
    std::vector<GatherJob> jobs;
    uint64_t nbytes = 0;
    for (uint64_t i = 0; i < n; i++) {
        const uint64_t src16 = h_voff[i];
        h_voff[i] = 0;
        if (h_status[i] != KB_GET_FOUND) {
            if (h_status[i] == KB_GET_NOT_FOUND) h_vlen[i] = 0;
            continue;
        }
        GatherJob j;
        j.dst16 = nbytes / 16;
        j.vsrc16 = src16;
        j.ksrc16 = 0;
        j.nk = 0;
        j.nv = (h_vlen[i] + 15) / 16;
        j.kl = 0;
        h_voff[i] = nbytes;
        nbytes += (uint64_t)j.nv * 16;
        if (j.nv) jobs.push_back(j);
    }
    res->n_bytes = nbytes;
    if (!jobs.empty()) {
        const uint64_t nj = jobs.size();
        rc = dbuf_ensure(ctx, ctx->d_gjobs, nj * sizeof(GatherJob));
        if (rc == KB_OK) rc = dbuf_ensure(ctx, ctx->d_jobs, 64);
        if (rc == KB_OK) rc = pool_get_arena(ctx, nbytes + 64, &res->d_bytes);
        if (rc == KB_OK) rc = hbuf_ensure(ctx, ctx->h_stage2, nj * sizeof(GatherJob) + 64);
        if (rc != KB_OK) {
            result_release_locked(ctx, res);
            return rc;
        }
        uint8_t *hj = (uint8_t *)ctx->h_stage2.p;
        memcpy(hj, &nj, 8);
        memset(hj + 8, 0, 8);  // the gather's block counter
        memcpy(hj + 64, jobs.data(), nj * sizeof(GatherJob));
        cudaMemcpyAsync(ctx->d_jobs.p, hj, 16, cudaMemcpyHostToDevice, ctx->stream);
        cudaMemcpyAsync(ctx->d_gjobs.p, hj + 64, nj * sizeof(GatherJob), cudaMemcpyHostToDevice, ctx->stream);
        rc = launch_gather(ctx, ctx->stream, (const GatherJob *)ctx->d_gjobs.p, (const uint64_t *)ctx->d_jobs.p,
                           (unsigned long long *)ctx->d_jobs.p + 1, (uint4 *)res->d_bytes.p, nj, 2 * nbytes);
        if (rc != KB_OK) {
            result_release_locked(ctx, res);
            return rc;
        }
        if (out_mode == KB_OUT_HOST) {
            rc = pool_get_host(ctx, nbytes + 16, &res->h_bytes);
            if (rc == KB_OK) cudaMemcpyAsync(res->h_bytes.p, res->d_bytes.p, nbytes, cudaMemcpyDeviceToHost, ctx->stream);
        }
        e = cudaStreamSynchronize(ctx->stream);
        if (rc == KB_OK && e != cudaSuccess) rc = kb_cuda_fail(ctx, e, "get gather");
        if (rc != KB_OK) {
            result_release_locked(ctx, res);
            return rc;
        }
        if (out_mode == KB_OUT_HOST) {
            pool_put_arena(ctx, res->d_bytes);
            res->d_bytes = DBuf();
        }
    }
    *out = res;
    return KB_OK;
}

extern "C" int kb_get_view_get(const kb_result *res, kb_get_view *v)
{
    if (!res || !v || res->type != 4) return KB_EINVAL;
    memset(v, 0, sizeof(*v));
    const uint64_t n = res->n_gets;
    const size_t st_off = (n + 7) & ~(size_t)7;
    const uint8_t *hg = (const uint8_t *)res->h_get.p;
    v->n = n;
    v->status = hg;
    v->mod_rev = (const uint64_t *)(hg + st_off);
    v->val_off = v->mod_rev + n;
    v->rec_idx = (const uint32_t *)(v->val_off + n);
    v->val_len = v->rec_idx + n;
    v->n_bytes = res->n_bytes;
    v->on_device = res->out_mode == KB_OUT_DEVICE;
    v->bytes = v->on_device ? (const uint8_t *)res->d_bytes.p : (const uint8_t *)res->h_bytes.p;
    return KB_OK;
}

// ------------------------------------------------------------------------------------------------
// compaction sweep
// ------------------------------------------------------------------------------------------------
extern "C" int kb_compact_sweep(kb_ctx *ctx, const uint8_t *start, uint64_t start_len, const uint8_t *end,
                                uint64_t end_len, uint64_t rev, uint64_t timeout_rev, int support_ttl, int out_mode,
                                kb_result **out)
{
    if (!ctx || !out) return KB_EINVAL;
    if (out_mode != KB_OUT_HOST && out_mode != KB_OUT_DEVICE && out_mode != KB_OUT_COUNT) return KB_EINVAL;
    *out = nullptr;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (!ctx->loaded) return kb_fail(ctx, KB_ESTATE, "no store loaded");
    cudaSetDevice(ctx->device);
    KB_TRY(ctx_quiesce(ctx));
    kb_range_req rq;
    rq.start = start;
    rq.start_len = start_len;
    rq.end = end;
    rq.end_len = end_len;
    rq.read_rev = rev;
    rq.limit = 0;
    Resolved R;
    KB_TRY(resolve_requests(ctx, &rq, 1, false, R));
    KB_TRY(upload_layout(ctx, R));
    ReqOut *d_rout = (ReqOut *)ctx->d_reqout.p;
    ScanMode mode;
    mode.compact = 1;
    mode.ttl_scan = (!support_ttl && timeout_rev != 0) ? 1 : 0;
    mode.timeout_rev = timeout_rev;
    mode.wire = 0;
    // One pass writes the ordered delete calls, so their buffer is sized before the count is known: a record is the
    // target of at most two calls (superseded as somebody's prev + tombstone / deleted revision record at its own turn,
    // or one TTL call).  The buffer is pooled; the host copy is cut to the real count.
    kb_result *res = kb_result_new(2, out_mode);
    const uint64_t nrec = R.n_records, cap_v = 2 * nrec;
    uint32_t *vidx = nullptr;
    uint8_t *vcls = nullptr;
    if (out_mode != KB_OUT_COUNT && nrec) {
        int rc = pool_get_dev(ctx, cap_v * 5 + 64, &res->d_vic);
        if (rc != KB_OK) {
            result_release_locked(ctx, res);
            return rc;
        }
        vidx = (uint32_t *)res->d_vic.p;
        vcls = (uint8_t *)(vidx + cap_v);
    }
    int rc = launch_scan_core(ctx, R, mode, vidx != nullptr, vidx, vcls);
    if (rc == KB_OK) rc = hbuf_ensure(ctx, ctx->h_stage, sizeof(ReqOut) + 64);
    if (rc == KB_OK && cudaMemcpyAsync(ctx->h_stage.p, d_rout, sizeof(ReqOut), cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess)
        rc = kb_fail(ctx, KB_ECUDA, "compact sweep: D2H");
    if (rc == KB_OK) {
        cudaError_t e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = kb_cuda_fail(ctx, e, "compact sweep");
    }
    if (rc != KB_OK) {
        result_release_locked(ctx, res);
        return rc;
    }
    ReqOut ro;
    memcpy(&ro, ctx->h_stage.p, sizeof(ro));

    // scan(compact=true) blindly stores the compact revision (checkCompactRace, scanner.go:596-604)
    ctx->compact_present = true;
    ctx->compact_rev = rev;

    res->n_victims = ro.total;
    res->count = ro.total_aux;
    res->examined = R.reqs[0].hi - R.reqs[0].lo;
    res->vic_cap = cap_v;
    if (out_mode == KB_OUT_HOST && ro.total > 0) {
        const uint64_t nv = ro.total;
        rc = pool_get_host(ctx, nv * 5 + 64, &res->h_vic);
        if (rc == KB_OK) {
            cudaMemcpyAsync(res->h_vic.p, vidx, nv * 4, cudaMemcpyDeviceToHost, ctx->stream);
            cudaMemcpyAsync((uint8_t *)res->h_vic.p + nv * 4, vcls, nv, cudaMemcpyDeviceToHost, ctx->stream);
            cudaError_t e = cudaStreamSynchronize(ctx->stream);
            if (e != cudaSuccess) rc = kb_cuda_fail(ctx, e, "compact sweep: victims D2H");
        }
        if (rc != KB_OK) {
            result_release_locked(ctx, res);
            return rc;
        }
    }
    if (out_mode != KB_OUT_DEVICE && res->d_vic.p) {
        pool_put_dev(ctx, res->d_vic);
        res->d_vic = DBuf();
    }
    *out = res;
    return KB_OK;
}

extern "C" int kb_compact_view_get(const kb_result *res, kb_compact_view *v)
{
    if (!res || !v || res->type != 2) return KB_EINVAL;
    memset(v, 0, sizeof(*v));
    v->n_victims = res->n_victims;
    v->count = res->count;
    v->examined = res->examined;
    v->on_device = res->out_mode == KB_OUT_DEVICE;
    const uint8_t *base = v->on_device ? (const uint8_t *)res->d_vic.p : (const uint8_t *)res->h_vic.p;
    if (base && res->out_mode != KB_OUT_COUNT) {
        v->victim_idx = (const uint32_t *)base;
        // device-resident answers keep the capacity-sized layout the sweep wrote into; the host copy is compact
        v->victim_class = base + (v->on_device ? res->vic_cap : res->n_victims) * 4;
    }
    return KB_OK;
}


// ------------------------------------------------------------------------------------------------
// kb_apply_batch: one committed BatchWrite merged into the HBM snapshot.
//
// Round 1 rebuilt both slabs and merged the whole directory on the host for every batch (O(store bytes)).  Now the
// store is a heap + a sorted directory: the bytes of the batch's puts are appended at the slab tails (a value that
// replaces an existing key leaves the old bytes behind as garbage; the key bytes are reused), and only the directory
// (46 bytes per record with the decoded columns) is rebuilt, on the device, by k_dir_merge + k_col_fix.  Records
// appended out of key order cost the copy kernels scattered reads, not wrong answers.  When more than 1/32 of the
// records are out of place, or a quarter of a slab is garbage, store_compact_layout rewrites the slabs contiguously in
// key order (O(store), amortised O(1) per op).
// ------------------------------------------------------------------------------------------------
namespace {
struct ApplyOp {
    std::string key, val;
    uint32_t type;
    uint64_t order;
};

// grow a slab to hold `need16` chunks (+ slack), keeping its first `used16` chunks
int slab_reserve(kb_ctx *ctx, DBuf &slab, uint64_t used16, uint64_t need16)
{
    const size_t need = (size_t)need16 * 16 + 64;
    if (slab.p && slab.cap >= need) return KB_OK;
    DBuf nb;
    KB_TRY(dbuf_ensure(ctx, nb, need + need / 2));
    if (slab.p && used16)
        KB_CUDA(ctx, cudaMemcpyAsync(nb.p, slab.p, (size_t)used16 * 16, cudaMemcpyDeviceToDevice, ctx->stream));
    KB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (slab.p) cudaFree(slab.p);
    slab = nb;
    return KB_OK;
}
}  // namespace

// the directory arrays that are NOT live (k_dir_merge / store_compact_layout write them, then the sets swap)
static int dir_spare_ensure(kb_ctx *ctx, uint64_t n)
{
    KB_TRY(dbuf_ensure(ctx, ctx->s_koff16, (n + 1) * 4));
    KB_TRY(dbuf_ensure(ctx, ctx->s_klen, (n + 1) * 2));
    KB_TRY(dbuf_ensure(ctx, ctx->s_voff16, (n + 1) * 8));
    KB_TRY(dbuf_ensure(ctx, ctx->s_vlen, (n + 1) * 4));
    KB_TRY(dbuf_ensure(ctx, ctx->s_dir, (n + 1) * 16));
    KB_TRY(dbuf_ensure(ctx, ctx->s_crev, (n + 1) * 8));
    KB_TRY(dbuf_ensure(ctx, ctx->s_cword, (n + 1) * 4));
    return KB_OK;
}

static void dir_swap(kb_ctx *ctx, uint64_t n)
{
    std::swap(ctx->d_koff16, ctx->s_koff16);
    std::swap(ctx->d_klen, ctx->s_klen);
    std::swap(ctx->d_voff16, ctx->s_voff16);
    std::swap(ctx->d_vlen, ctx->s_vlen);
    std::swap(ctx->d_dir, ctx->s_dir);
    std::swap(ctx->d_crev, ctx->s_crev);
    std::swap(ctx->d_cword, ctx->s_cword);
    ctx->st.koff16 = (const uint32_t *)ctx->d_koff16.p;
    ctx->st.klen = (const uint16_t *)ctx->d_klen.p;
    ctx->st.voff16 = (const uint64_t *)ctx->d_voff16.p;
    ctx->st.vlen = (const uint32_t *)ctx->d_vlen.p;
    ctx->st.dir = (const uint4 *)ctx->d_dir.p;
    ctx->st.crev = (const uint64_t *)ctx->d_crev.p;
    ctx->st.cword = (const uint32_t *)ctx->d_cword.p;
    ctx->st.kslab = (const uint4 *)ctx->d_kslab.p;
    ctx->st.vslab = (const uint4 *)ctx->d_vslab.p;
    ctx->st.n = (uint32_t)n;
    ctx->store_gen++;  // prefetched bound searches of the old snapshot are void
}

// rewrite both slabs contiguously in key order (also what kb_dump writes); the caller holds ctx->mu
int store_compact_layout(kb_ctx *ctx)
{
    const uint64_t n = ctx->st.n;
    if (ctx->displaced == 0 && ctx->garbage_k16 == 0 && ctx->garbage_v16 == 0) return KB_OK;
    std::vector<uint16_t> klen(std::max<uint64_t>(n, 1));
    std::vector<uint32_t> vlen(std::max<uint64_t>(n, 1)), nko(n + 1);
    std::vector<uint64_t> nvo(n + 1);
    if (n) {
        KB_CUDA(ctx, cudaMemcpyAsync(klen.data(), ctx->st.klen, n * 2, cudaMemcpyDeviceToHost, ctx->stream));
        KB_CUDA(ctx, cudaMemcpyAsync(vlen.data(), ctx->st.vlen, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
        KB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    uint64_t kacc = 0, vacc = 0;
    for (uint64_t i = 0; i < n; i++) {
        nko[i] = (uint32_t)kacc;
        nvo[i] = vacc;
        kacc += ((uint32_t)klen[i] + 15) / 16;
        vacc += ((uint64_t)vlen[i] + 15) / 16;
    }
    nko[n] = (uint32_t)kacc;
    nvo[n] = vacc;
    DBuf nk, nv;
    KB_TRY(dbuf_ensure(ctx, nk, kacc * 16 + 64));
    int rc = dbuf_ensure(ctx, nv, vacc * 16 + 64);
    if (rc == KB_OK) rc = dir_spare_ensure(ctx, n);
    if (rc != KB_OK) {
        cudaFree(nk.p);
        if (nv.p) cudaFree(nv.p);
        return rc;
    }
    cudaMemsetAsync((uint8_t *)nk.p + kacc * 16, 0, 64, ctx->stream);
    cudaMemsetAsync((uint8_t *)nv.p + vacc * 16, 0, 64, ctx->stream);
    cudaMemcpyAsync(ctx->s_koff16.p, nko.data(), (n + 1) * 4, cudaMemcpyHostToDevice, ctx->stream);
    cudaMemcpyAsync(ctx->s_voff16.p, nvo.data(), (n + 1) * 8, cudaMemcpyHostToDevice, ctx->stream);
    if (n) {
        KB_LAUNCH(ctx, "k_relocate", 2 * (kacc + vacc) * 16,
                  (k_relocate<<<148 * 8, 256, 0, ctx->stream>>>(ctx->st, (const uint32_t *)ctx->s_koff16.p,
                                                               (const uint64_t *)ctx->s_voff16.p, (uint4 *)nk.p, (uint4 *)nv.p)));
        cudaMemcpyAsync(ctx->s_klen.p, ctx->st.klen, n * 2, cudaMemcpyDeviceToDevice, ctx->stream);
        cudaMemcpyAsync(ctx->s_vlen.p, ctx->st.vlen, n * 4, cudaMemcpyDeviceToDevice, ctx->stream);
        // directory order does not change: the decoded columns stay valid
        cudaMemcpyAsync(ctx->s_crev.p, ctx->st.crev, n * 8, cudaMemcpyDeviceToDevice, ctx->stream);
        cudaMemcpyAsync(ctx->s_cword.p, ctx->st.cword, n * 4, cudaMemcpyDeviceToDevice, ctx->stream);
    }
    cudaError_t e = cudaStreamSynchronize(ctx->stream);  // the host vectors die here; the old slabs are released below
    if (e != cudaSuccess) {
        cudaFree(nk.p);
        cudaFree(nv.p);
        ctx->loaded = false;
        return kb_cuda_fail(ctx, e, "layout compaction");
    }
    cudaFree(ctx->d_kslab.p);
    cudaFree(ctx->d_vslab.p);
    ctx->d_kslab = nk;
    ctx->d_vslab = nv;
    dir_swap(ctx, n);
    rc = store_pack_dir(ctx);
    if (rc == KB_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess) rc = KB_ECUDA;
    if (rc != KB_OK) {
        ctx->loaded = false;
        return rc;
    }
    ctx->kused16 = kacc;
    ctx->vused16 = vacc;
    ctx->key_bytes = kacc * 16;
    ctx->val_bytes = vacc * 16;
    ctx->garbage_k16 = ctx->garbage_v16 = ctx->displaced = 0;
    ctx->layout_compactions++;
    return KB_OK;
}

static int apply_batch_locked(kb_ctx *ctx, const kb_write_op *ops, uint64_t n_ops);

extern "C" int kb_apply_batch(kb_ctx *ctx, const kb_write_op *ops, uint64_t n_ops)
{
    if (!ctx || (n_ops && !ops)) return KB_EINVAL;
    std::lock_guard<std::mutex> g(ctx->mu);
    KB_TRY(apply_batch_locked(ctx, ops, n_ops));
    // TTL bookkeeping, in op order: the last op on a key decides whether (and when) it expires
    for (uint64_t i = 0; i < n_ops; i++) {
        std::string k((const char *)ops[i].key, ops[i].key_len);
        if (ops[i].type == KB_OP_PUT && ops[i].expire_unix) {
            ctx->ttl_of[k] = ops[i].expire_unix;
            ctx->ttl_queue.emplace(ops[i].expire_unix, std::move(k));
        } else if (!ctx->ttl_of.empty()) {
            ctx->ttl_of.erase(k);  // deleted, or rewritten without a ttl: stale queue entries are skipped by kb_expire
        }
    }
    return KB_OK;
}

extern "C" int kb_expire(kb_ctx *ctx, uint64_t now_unix, uint64_t *n_dropped)
{
    if (!ctx) return KB_EINVAL;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (n_dropped) *n_dropped = 0;
    if (!ctx->loaded) return kb_fail(ctx, KB_ESTATE, "no store loaded");
    std::vector<std::string> due;
    auto end = ctx->ttl_queue.upper_bound(now_unix);
    for (auto it = ctx->ttl_queue.begin(); it != end; ++it) {
        auto cur = ctx->ttl_of.find(it->second);
        if (cur != ctx->ttl_of.end() && cur->second == it->first) {  // still the expiry the key has
            due.push_back(it->second);
            ctx->ttl_of.erase(cur);
        }
    }
    ctx->ttl_queue.erase(ctx->ttl_queue.begin(), end);
    if (due.empty()) return KB_OK;
    std::vector<kb_write_op> ops(due.size());
    for (size_t i = 0; i < due.size(); i++) {
        memset(&ops[i], 0, sizeof(kb_write_op));
        ops[i].type = KB_OP_DEL;
        ops[i].key = (const uint8_t *)due[i].data();
        ops[i].key_len = due[i].size();
    }
    const uint64_t before = ctx->st.n;
    KB_TRY(apply_batch_locked(ctx, ops.data(), ops.size()));
    if (n_dropped) *n_dropped = before - ctx->st.n;
    return KB_OK;
}

static int apply_batch_locked(kb_ctx *ctx, const kb_write_op *ops, uint64_t n_ops)
{
    if (!ctx->loaded) return kb_fail(ctx, KB_ESTATE, "no store loaded");
    cudaSetDevice(ctx->device);
    KB_TRY(ctx_quiesce(ctx));
    if (n_ops == 0) return KB_OK;
    // 1. last op per key wins; sort by key (bytes.Compare order)
    std::vector<ApplyOp> all(n_ops);
    for (uint64_t i = 0; i < n_ops; i++) {
        if ((!ops[i].key && ops[i].key_len) || (ops[i].type == KB_OP_PUT && !ops[i].val && ops[i].val_len)) return KB_EINVAL;
        if (ops[i].key_len > 65535) return kb_fail(ctx, KB_ELIMIT, "key longer than 65535 bytes");
        if (ops[i].val_len > 0xFFFFFFFFull) return kb_fail(ctx, KB_ELIMIT, "value too long");
        if (ops[i].type != KB_OP_PUT && ops[i].type != KB_OP_DEL) return KB_EINVAL;
        all[i].key.assign((const char *)ops[i].key, ops[i].key_len);
        if (ops[i].type == KB_OP_PUT) all[i].val.assign((const char *)ops[i].val, ops[i].val_len);
        all[i].type = ops[i].type;
        all[i].order = i;
    }
    std::sort(all.begin(), all.end(), [](const ApplyOp &a, const ApplyOp &b) {
        const int c = a.key.compare(b.key);  // std::string::compare is lexicographic on unsigned char via char_traits
        return c != 0 ? c < 0 : a.order < b.order;
    });
    std::vector<ApplyOp> m;
    for (size_t i = 0; i < all.size(); i++)
        if (i + 1 == all.size() || all[i + 1].key != all[i].key) m.push_back(std::move(all[i]));
    const uint64_t M = m.size();

    // 2. op keys as a padded bound slab on the device; lower bound and exact-match test of every op key
    uint64_t kchunks = 0;
    for (auto &o : m) kchunks += (o.key.size() + 15) / 16 + 3;
    KB_TRY(hbuf_ensure(ctx, ctx->h_stage, kchunks * 16 + M * 8 + 256));
    uint8_t *hs = (uint8_t *)ctx->h_stage.p;
    memset(hs, 0, kchunks * 16);
    uint32_t *hboff = (uint32_t *)(hs + kchunks * 16), *hblen = hboff + M;
    uint64_t kc = 0;
    for (uint64_t i = 0; i < M; i++) {
        hboff[i] = (uint32_t)kc;
        hblen[i] = (uint32_t)m[i].key.size();
        if (!m[i].key.empty()) memcpy(hs + kc * 16, m[i].key.data(), m[i].key.size());
        kc += (m[i].key.size() + 15) / 16 + 3;
    }
    KB_TRY(dbuf_ensure(ctx, ctx->d_bounds, kchunks * 16 + M * 8 + 64));
    KB_TRY(dbuf_ensure(ctx, ctx->d_bres, M * 9 + 64));
    KB_CUDA(ctx, cudaMemcpyAsync(ctx->d_bounds.p, hs, kchunks * 16 + M * 8, cudaMemcpyHostToDevice, ctx->stream));
    const uint32_t *d_boff = (const uint32_t *)((const uint8_t *)ctx->d_bounds.p + kchunks * 16);
    uint32_t *d_pos = (uint32_t *)ctx->d_bres.p, *d_oldv = d_pos + M;
    uint8_t *d_exists = (uint8_t *)(d_oldv + M);
    const unsigned sg = (unsigned)((M * 32 + 127) / 128);
    KB_LAUNCH(ctx, "k_search", M * 64,
              (k_search<<<sg, 128, 0, ctx->stream>>>(ctx->st, (const uint4 *)ctx->d_bounds.p, d_boff, d_boff + M, (uint32_t)M,
                                                     d_pos, SearchPub{nullptr, nullptr, 0})));
    KB_LAUNCH(ctx, "k_key_exists", M * 320,
              (k_key_exists<<<sg, 128, 0, ctx->stream>>>(ctx->st, (const uint4 *)ctx->d_bounds.p, d_boff, d_boff + M, d_pos,
                                                         (uint32_t)M, d_exists, d_oldv)));
    std::vector<uint32_t> pos(M), oldv(M);
    std::vector<uint8_t> exists(M);
    KB_CUDA(ctx, cudaMemcpyAsync(pos.data(), d_pos, M * 4, cudaMemcpyDeviceToHost, ctx->stream));
    KB_CUDA(ctx, cudaMemcpyAsync(oldv.data(), d_oldv, M * 4, cudaMemcpyDeviceToHost, ctx->stream));
    KB_CUDA(ctx, cudaMemcpyAsync(exists.data(), d_exists, M, cudaMemcpyDeviceToHost, ctx->stream));
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) return kb_cuda_fail(ctx, e, "apply: search");

    // 3. classify; lay the appended bytes out behind the slab tails
    const uint64_t N = ctx->st.n;
    std::vector<uint32_t> ins_pos, del_pos, rep_pos;
    std::vector<uint4> ins_ent, rep_ent;
    std::vector<uint8_t> kimg, vimg;  // images of the appended key / value chunks
    uint64_t ktail = ctx->kused16, vtail = ctx->vused16, garbage_k = 0, garbage_v = 0;
    uint32_t max_kv = ctx->max_kv_chunks;
    auto append = [](std::vector<uint8_t> &img, const std::string &b) {
        const size_t at = img.size(), n16 = (b.size() + 15) / 16;
        img.resize(at + n16 * 16, 0);
        if (!b.empty()) memcpy(img.data() + at, b.data(), b.size());
        return (uint64_t)n16;
    };
    auto entry = [](uint64_t ko, size_t kl, uint64_t vo, size_t vl) {
        return make_uint4((uint32_t)ko, (uint32_t)kl | ((uint32_t)(vo >> 32) << 16), (uint32_t)vl, (uint32_t)vo);
    };
    for (uint64_t i = 0; i < M; i++) {
        if (m[i].type == KB_OP_PUT) {
            const uint64_t vo = vtail;
            const uint64_t nv = append(vimg, m[i].val);
            vtail += nv;
            const uint64_t nk = (m[i].key.size() + 15) / 16;
            if (exists[i]) {  // same key: the key bytes stay where they are, the old value becomes garbage
                rep_pos.push_back(pos[i]);
                rep_ent.push_back(entry(0, 0, vo, m[i].val.size()));
                garbage_v += oldv[i];
            } else {
                ins_pos.push_back(pos[i]);
                ins_ent.push_back(entry(ktail, m[i].key.size(), vo, m[i].val.size()));
                ktail += append(kimg, m[i].key);
            }
            max_kv = std::max<uint32_t>(max_kv, (uint32_t)std::min<uint64_t>(nk + nv, 0xFFFFFFFFu));
        } else if (exists[i]) {
            del_pos.push_back(pos[i]);
            garbage_k += (m[i].key.size() + 15) / 16;
            garbage_v += oldv[i];
        }
    }
    const uint64_t n_ins = ins_pos.size(), n_del = del_pos.size(), n_rep = rep_pos.size();
    const uint64_t N2 = N + n_ins - n_del;
    if (N2 >= 0xFFFFFFFEull) return kb_fail(ctx, KB_ELIMIT, "too many records");
    if (ktail > 0xFFFFFFF0ull) return kb_fail(ctx, KB_ELIMIT, "key slab exceeds 64 GiB");
    if (n_ins + n_del + n_rep == 0) return KB_OK;  // only deletes of absent keys

    // 4. bytes to the slab tails (growing a slab copies its used part once; the live store is untouched until step 6)
    KB_TRY(slab_reserve(ctx, ctx->d_kslab, ctx->kused16, ktail));
    KB_TRY(slab_reserve(ctx, ctx->d_vslab, ctx->vused16, vtail));
    ctx->st.kslab = (const uint4 *)ctx->d_kslab.p;
    ctx->st.vslab = (const uint4 *)ctx->d_vslab.p;
    const size_t tab_bytes = (n_ins + n_del + n_rep) * 4 + (n_ins + n_rep) * 16 + 64;
    KB_TRY(hbuf_ensure(ctx, ctx->h_stage2, kimg.size() + vimg.size() + tab_bytes + 256));
    uint8_t *h2 = (uint8_t *)ctx->h_stage2.p;
    if (!kimg.empty()) memcpy(h2, kimg.data(), kimg.size());
    if (!vimg.empty()) memcpy(h2 + kimg.size(), vimg.data(), vimg.size());
    uint8_t *ht = h2 + ((kimg.size() + vimg.size() + 15) & ~(size_t)15);
    uint4 *t_ins_ent = (uint4 *)ht, *t_rep_ent = t_ins_ent + n_ins;
    uint32_t *t_ins_pos = (uint32_t *)(t_rep_ent + n_rep), *t_del_pos = t_ins_pos + n_ins, *t_rep_pos = t_del_pos + n_del;
    if (n_ins) memcpy(t_ins_ent, ins_ent.data(), n_ins * 16), memcpy(t_ins_pos, ins_pos.data(), n_ins * 4);
    if (n_rep) memcpy(t_rep_ent, rep_ent.data(), n_rep * 16), memcpy(t_rep_pos, rep_pos.data(), n_rep * 4);
    if (n_del) memcpy(t_del_pos, del_pos.data(), n_del * 4);
    KB_TRY(dbuf_ensure(ctx, ctx->d_bounds, tab_bytes + 64));  // the bound slab is no longer needed: reuse it for the tables
    KB_TRY(dir_spare_ensure(ctx, N2));
    if (!kimg.empty())
        KB_CUDA(ctx, cudaMemcpyAsync((uint8_t *)ctx->d_kslab.p + ctx->kused16 * 16, h2, kimg.size(), cudaMemcpyHostToDevice, ctx->stream));
    if (!vimg.empty())
        KB_CUDA(ctx, cudaMemcpyAsync((uint8_t *)ctx->d_vslab.p + ctx->vused16 * 16, h2 + kimg.size(), vimg.size(),
                                     cudaMemcpyHostToDevice, ctx->stream));
    // key_less reads up to three chunks past a key: keep the slack behind the tails zero
    KB_CUDA(ctx, cudaMemsetAsync((uint8_t *)ctx->d_kslab.p + ktail * 16, 0, 64, ctx->stream));
    KB_CUDA(ctx, cudaMemsetAsync((uint8_t *)ctx->d_vslab.p + vtail * 16, 0, 64, ctx->stream));
    KB_CUDA(ctx, cudaMemcpyAsync(ctx->d_bounds.p, ht, tab_bytes - 64, cudaMemcpyHostToDevice, ctx->stream));
    // 5. the directory, rebuilt on the device into the spare set
    const uint4 *d_ins_ent = (const uint4 *)ctx->d_bounds.p, *d_rep_ent = d_ins_ent + n_ins;
    const uint32_t *d_ins_pos = (const uint32_t *)(d_rep_ent + n_rep), *d_del_pos = d_ins_pos + n_ins, *d_rep_pos = d_del_pos + n_del;
    DirArrays out;
    out.koff16 = (uint32_t *)ctx->s_koff16.p;
    out.klen = (uint16_t *)ctx->s_klen.p;
    out.voff16 = (uint64_t *)ctx->s_voff16.p;
    out.vlen = (uint32_t *)ctx->s_vlen.p;
    out.dir = (uint4 *)ctx->s_dir.p;
    out.crev = (uint64_t *)ctx->s_crev.p;
    out.cword = (uint32_t *)ctx->s_cword.p;
    const uint64_t threads = N + n_ins;
    KB_LAUNCH(ctx, "k_dir_merge", (N + N2) * 46,
              (k_dir_merge<<<(unsigned)((threads + 255) / 256), 256, 0, ctx->stream>>>(ctx->st, d_ins_pos, d_ins_ent, (uint32_t)n_ins,
                                                                                       d_del_pos, (uint32_t)n_del, d_rep_pos,
                                                                                       d_rep_ent, (uint32_t)n_rep, out)));
    // the stale column entries, from the new directory: per candidate two keys, two directory entries, one value probe
    StoreDev nd = ctx->st;
    nd.koff16 = out.koff16;
    nd.klen = out.klen;
    nd.voff16 = out.voff16;
    nd.vlen = out.vlen;
    nd.dir = out.dir;
    nd.crev = out.crev;
    nd.cword = out.cword;
    nd.n = (uint32_t)N2;
    const uint64_t n_fix = 2 * n_ins + n_del + n_rep + 1;
    const uint64_t mean_key = ktail * 16 / std::max<uint64_t>(N2, 1);
    KB_LAUNCH(ctx, "k_col_fix", n_fix * (2 * mean_key + 2 * 14 + 16 + 12),
              (k_col_fix<<<(unsigned)((n_ins + n_del + n_rep + 1 + 255) / 256), 256, 0, ctx->stream>>>(
                  nd, d_ins_pos, (uint32_t)n_ins, d_del_pos, (uint32_t)n_del, d_rep_pos, (uint32_t)n_rep, out.crev, out.cword)));
    e = cudaStreamSynchronize(ctx->stream);  // the staging buffers are reused by the next call
    if (e != cudaSuccess) {
        ctx->loaded = false;
        return kb_cuda_fail(ctx, e, "apply: directory merge");
    }
    // 6. the new snapshot becomes visible
    dir_swap(ctx, N2);
    ctx->kused16 = ktail;
    ctx->vused16 = vtail;
    ctx->key_bytes = ktail * 16;
    ctx->val_bytes = vtail * 16;
    ctx->garbage_k16 += garbage_k;
    ctx->garbage_v16 += garbage_v;
    ctx->displaced += n_ins;
    ctx->max_kv_chunks = max_kv;
    if (ctx->displaced > std::max<uint64_t>(4096, N2 / 32) || ctx->garbage_k16 * 4 > ktail || ctx->garbage_v16 * 4 > vtail)
        KB_TRY(store_compact_layout(ctx));
    return KB_OK;
}
