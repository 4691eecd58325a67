// kb_watch.cu -- watch fan-out: one revision-ordered event slab x every registered watcher's
// (key-prefix, min-revision) predicate -> per-watcher ordered delivery lists.
//
// Replaces (reference file:line):
//   WatcherHub.Stream broadcast           pkg/backend/watcherhub.go:78-92   (every batch handed to every watcher)
//   processEvents / filterByRevision /    pkg/backend/watch.go:119-159      (per watcher: strip leading events below
//   filterByPrefix                                                           min_rev, keep bytes.HasPrefix matches)
//
// Brute force is W x E prefix tests (1e9 for 10k watchers x 100k events).  Here watchers are grouped by
// distinct prefix; an event probes a device hash table once per DISTINCT PREFIX LENGTH with the FNV-1a
// hash of its own leading bytes (verified byte-exactly), so the work is O(E * #lengths + deliveries).
//
// Round 2: the seven dependent launches of round 1 (each queueing again behind the scan context's persistent
// CTAs) are ONE cooperative kernel, k_fanout, whose phases are separated by grid barriers:
//   P1  per collector batch: running max of Event.Revision (the "leading strip" predicate becomes pm[i] >= min_rev)
//       and a flag "revisions globally non-decreasing"; per event and prefix length: the matched group (ematch) and
//       warp-aggregated group counts
//   P2  per event: the group's segment is claimed lazily from a bump allocator (segments need to be disjoint, not
//       ordered, so no prefix sum over the groups); groups are classified small (<= 32 matches), medium (<= big_t),
//       large (global bitmap); small/medium matches are scattered with warp-aggregated slot claims, for a large group
//       the warp's ballot IS the 32-event bitmap word
//   P3  medium groups: shared-memory bitmap windows -> ascending segment; large groups: ordered bitmap expansion
//   P4  warp per watcher: small groups are rank-sorted in registers here; deliveries = its group's ascending segment
//       filtered by min_rev (a suffix found by a 32-ary search when revisions are monotone)
//   P5  the last CTA to finish P4 computes the per-watcher output offsets and leaves the scratch clean for the next call
// followed by k_publish_total (mapped pinned flag: the host returns here) and k_expand_write (one thread per delivery).
#include <algorithm>
#include <map>
#include <unordered_map>

#include "kb_internal.cuh"

struct kb_events_dev {
    DBuf keys;       // n x stride bytes: the first `stride` bytes of every event key (zero padded)
    DBuf klen;       // n x u32 true key lengths
    DBuf rev;        // n x u64
    DBuf batch_off;  // (nb+1) x u64
    uint32_t n = 0, nb = 0, stride = 0;
};

struct WatchTablesDev {
    uint32_t n_ids = 0, n_groups = 0, n_lens = 0, table_size = 0, max_len = 0, pstride16 = 1;
    uint64_t d_hint = 0;  // deliveries of the previous match (sizes the next output buffer)
    DBuf gprefix, wgroup, wminrev, lens, table;
    // per-call scratch
    DBuf gstate /* gcnt | gfill | ctl */, galloc, lists, ematch, seg, seg_sorted, bitmaps, pm, wstate /* wcnt | wsrc | wn | wlo */,
        wstart, total;
    // Everything above is carved out of ONE allocation: [tables | per-call scratch].  The context's stream carries an L2
    // access-policy window over it (persisting): the scan context streams > 1 GB through the 126 MB L2 in every step, which
    // would otherwise evict the tables and the scratch between two phases of k_fanout (it then runs on HBM latency).
    DBuf arena;
    size_t tab_end = 0, scr_bytes = 0, scr_sig = 0;
    bool scratch_clean = false;   // the previous k_fanout left gstate / galloc / bitmaps in their initial state
    uint32_t scratch_groups = 0, scratch_large = 0, scratch_bm_words = 0;
    uint32_t fan_gen = 0;         // value of the grid-barrier generation word after the last launch
    uint32_t fan_set = 0;         // which of the two sets of group state the next k_fanout uses
    int fan_grid = 0;             // co-resident CTAs of k_fanout on this device (0: not queried yet)
    // The delivery lists are written by k_expand_write on the context's second stream, so the write of burst n overlaps
    // k_fanout of burst n+1: what the write reads (sorted segments, running max, per-watcher state, offsets, total) exists
    // twice, `wr_set` alternates.  ev_fan: end of the last k_fanout; ev_write[s]: end of the last write that read set s.
    uint32_t wr_set = 0;
    cudaEvent_t ev_fan = nullptr, ev_write[2] = {nullptr, nullptr};
};

namespace {

constexpr unsigned FULL = 0xffffffffu;
constexpr uint64_t FNV_OFFSET = 14695981039346656037ull;
constexpr uint64_t FNV_PRIME = 1099511628211ull;

__host__ __device__ __forceinline__ uint32_t slot_of(uint64_t h, uint32_t len, uint32_t mask)
{
    uint64_t m = h ^ ((uint64_t)len * 0x9E3779B97F4A7C15ull);
    m ^= m >> 29;
    return (uint32_t)(m ^ (m >> 32)) & mask;
}

struct EvDev {
    const uint4 *keys;
    const uint32_t *klen;
    const uint64_t *rev;
    const uint64_t *batch_off;
    uint32_t n, nb, stride16;
};

struct TabDev {
    const uint4 *gprefix;      // group g's prefix at gprefix + g * pstride16 (zero padded)
    const uint32_t *wgroup;
    const uint64_t *wminrev;
    const uint32_t *lens;      // distinct prefix lengths, ascending
    const uint4 *table;        // open addressing: {hash lo, hash hi, prefix length, group} ; group == NONE: empty
    uint32_t n_ids, n_groups, n_lens, mask, max_len, pstride16;
};

// control words of one match (gstate: [gcnt G+1][gfill G+1][ctl 16])
enum { FC_NONMONO = 0, FC_CURSOR = 1, FC_NLARGE = 2, FC_NMED = 3, FC_ARRIVE = 4, FC_GEN = 5, FC_DONE = 6, FC_ABORT = 7, FC_WORDS = 16 };
constexpr unsigned long long FAN_UNSET = ~0ull, FAN_BUSY = ~0ull - 1;
// One CTA per SM, < 2 KiB of shared memory (see fan_grid_sync).  Registers: 384 threads x 80 (k_fanout's cap, no spill)
// = 30 720; its neighbours on an SM are the scan context's two gather CTAs (2 x 256 x 32 = 16 384) and the short scan
// kernels (256 x 32 = 8 192 per CTA): 30 720 + 16 384 + 2 x 8 192 = 63 488 of 65 536.  Measured on a B200 (1 000 W,
// 1 965 MHz max SM clock, bench step, 3 runs each): cap 64 (28 B spilled) 4.26-4.52 G events/s, 72 (20 B) 4.55-4.59,
// 80 4.62-4.66 (profiles/r03_fanout_cap_ab.txt).
constexpr uint32_t FAN_THREADS = 384;
constexpr uint32_t BM_WORDS = 256;   // 8192 event indices per shared-memory window (1 KiB).  The scan context's two gather
                                     // CTAs leave ~6 KiB of an SM's shared memory (every resident CTA also costs 1 KiB of
                                     // reserve): with a 4 KiB window here NOTHING else of the scan context -- not even the
                                     // shared-memory-free k_search -- fitted beside them for the whole fan-out (measured:
                                     // k_search 10 us alone, 140 us in a step)

struct FanScratch {
    uint32_t *gcnt, *gfill, *ctl;
    unsigned long long *galloc;      // per group (bitmap slot or NONE) << 32 | segment base; FAN_UNSET between calls
    uint32_t *med_list, *large_list;
    uint32_t *ematch, *seg, *sorted, *bitmaps;
    uint64_t *pm;
    uint32_t *wcnt, *wsrc, *wn, *wlo;
    uint64_t *wstart, *total;
    uint32_t big_t, max_large, bm_words, chunks_per_group, gen_base;
    // group state is double buffered: this call uses gcnt / gfill / galloc / bitmaps and clears the OTHER set (used by the
    // previous call) in its first phase, fully parallel; *nlarge_w: bitmap slots this call used, *nlarge_r: the previous one
    uint32_t *z_gcnt, *z_bitmaps, *nlarge_w, *nlarge_r;
    unsigned long long *z_galloc;
    uint64_t *o_start, *h_start;   // the output buffer's offsets and their (pinned, device-visible) host copy
    uint64_t *h_pub, epoch;        // mapped flag: [0] epoch, [1] total deliveries, [2] a barrier timed out; [3..7] phase ends (ns)
};

// scratch written by one CTA and read by another inside the same launch goes around the (non-coherent) L1
__device__ __forceinline__ uint32_t ldcg32(const uint32_t *p) { return __ldcg(p); }
__device__ __forceinline__ uint64_t ldcg64(const uint64_t *p) { return __ldcg((const unsigned long long *)p); }

// Grid barrier.  The kernel is launched with ONE CTA per SM of modest size (384 threads, < 28 k registers, < 2 KiB of
// shared memory), which fits beside whatever the scan context has resident, so every CTA gets an SM while the others
// spin; nothing this kernel waits for depends on work queued behind it.  (A cooperative launch would guarantee the same
// but is gang-scheduled: measured, it waited for the scan context's persistent kernels to drain -- 247 us in a step
// against 90 us alone -- and held k_search behind it.)  `gen` only ever grows; the host passes its value before the launch.
// A barrier that does not complete within ~2 s raises FC_ABORT: every CTA then falls through to the end of the kernel
// and the host fails the call instead of hanging.
__device__ __forceinline__ void fan_grid_sync(uint32_t *ctl, uint32_t target)
{
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(&ctl[FC_ARRIVE], 1u) == gridDim.x - 1) {
            atomicExch(&ctl[FC_ARRIVE], 0u);  // nobody arrives at the next barrier before the release below
            __threadfence();
            atomicExch(&ctl[FC_GEN], target);
        } else {
            const long long t0 = clock64();
            while (*(volatile uint32_t *)&ctl[FC_GEN] != target) {
                __nanosleep(64);
                if (clock64() - t0 > 4000000000ll) {
                    atomicExch(&ctl[FC_ABORT], 1u);
                    break;
                }
                if (*(volatile uint32_t *)&ctl[FC_ABORT]) break;
            }
        }
        __threadfence();
    }
    __syncthreads();
}

// ---- running max of the revisions inside each collector batch (filterByRevision strips only the LEADING
//      events below min_rev, watch.go:153-159, so event i survives iff max(rev[batch start..i]) >= min_rev)
__device__ __forceinline__ void d_batch_pm(const EvDev &ev, uint64_t *__restrict__ pm, uint32_t *__restrict__ nonmono,
                                           uint32_t vblock)
{
    const uint32_t w = (vblock * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= ev.nb) return;
    const uint64_t lo = ev.batch_off[w], hi = ev.batch_off[w + 1];
    uint64_t carry = 0;
    bool bad = false;
    for (uint64_t c = lo; c < hi; c += 32) {
        const uint64_t i = c + lane;
        uint64_t v = i < hi ? ev.rev[i] : 0;
        if (i < hi && i > 0 && ev.rev[i - 1] > v) bad = true;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            uint64_t o = __shfl_up_sync(FULL, v, d);
            if (lane >= (unsigned)d) v = max(v, o);
        }
        v = max(v, carry);
        if (i < hi) pm[i] = v;
        carry = __shfl_sync(FULL, v, 31);
    }
    if (__any_sync(FULL, bad) && lane == 0) atomicOr(nonmono, 1u);
}

// ---- per event and distinct prefix length: the group whose prefix the key starts with (or NONE).
//      ematch[li * E + i]; group counts are aggregated inside the warp before touching memory.
//      A thread owns EPT events (i, i + blockDim, ..): the hash / probe / verify chains of its events are independent and
//      are written interleaved so that their loads are in flight together (the phase is a chain of ~4 dependent loads per
//      prefix length; one CTA per SM has 256 threads for ~680 events).
constexpr int FAN_EPT = 3;

__device__ __forceinline__ void d_match_count(const EvDev &ev, const TabDev &tb, uint32_t *__restrict__ ematch,
                                              uint32_t *__restrict__ gcnt, uint32_t vblock)
{
    const uint32_t lane = threadIdx.x & 31;
    uint32_t i[FAN_EPT], klen[FAN_EPT];
    const uint4 *kp[FAN_EPT];
    uint64_t h[FAN_EPT];
    uint4 chunk[FAN_EPT];
    bool valid[FAN_EPT];
#pragma unroll
    for (int e = 0; e < FAN_EPT; e++) {
        i[e] = (vblock * FAN_EPT + e) * blockDim.x + threadIdx.x;
        valid[e] = i[e] < ev.n;
        klen[e] = valid[e] ? ev.klen[i[e]] : 0;
        kp[e] = ev.keys + (uint64_t)(valid[e] ? i[e] : 0) * ev.stride16;
        h[e] = FNV_OFFSET;
        chunk[e] = make_uint4(0, 0, 0, 0);
    }
    uint32_t pos = 0;  // bytes hashed so far (the same for every event: lengths are visited in ascending order)
    for (uint32_t li = 0; li < tb.n_lens; li++) {  // uniform trip count: the warp collectives below need all lanes
        const uint32_t L = __ldg(tb.lens + li);
        for (; pos < L; pos++) {
            if ((pos & 15) == 0) {
#pragma unroll
                for (int e = 0; e < FAN_EPT; e++) chunk[e] = __ldg(kp[e] + (pos >> 4));  // in bounds: L <= stride
            }
#pragma unroll
            for (int e = 0; e < FAN_EPT; e++) h[e] = (h[e] ^ (uint64_t)byte_of(chunk[e], pos & 15)) * FNV_PRIME;
        }
        // probe (hash, length): one 16-byte entry per slot; the first probes of all events go out together
        uint32_t s[FAN_EPT], g[FAN_EPT];
        uint4 t[FAN_EPT];
#pragma unroll
        for (int e = 0; e < FAN_EPT; e++) {
            s[e] = slot_of(h[e], L, tb.mask);
            t[e] = __ldg(tb.table + s[e]);
            g[e] = KB_NONE;
        }
#pragma unroll
        for (int e = 0; e < FAN_EPT; e++) {
            if (!(valid[e] && L <= klen[e])) continue;
            for (;;) {
                if (t[e].w == KB_NONE) break;
                if (t[e].x == (uint32_t)h[e] && t[e].y == (uint32_t)(h[e] >> 32) && t[e].z == L) {
                    // verify the bytes so the result is exact
                    const uint4 *gp = tb.gprefix + (uint64_t)t[e].w * tb.pstride16;
                    bool eq = true;
                    for (uint32_t k = 0; k * 16 < L && eq; k++) {
                        uint4 a = __ldg(kp[e] + k), b = __ldg(gp + k);
                        int p = first_diff16(a, b);
                        if (p < 16 && k * 16 + p < L) eq = false;
                    }
                    if (eq) {
                        g[e] = t[e].w;
                        break;  // prefixes are unique per group
                    }
                }
                s[e] = (s[e] + 1) & tb.mask;
                t[e] = __ldg(tb.table + s[e]);
            }
        }
#pragma unroll
        for (int e = 0; e < FAN_EPT; e++) {
            if (valid[e]) ematch[(uint64_t)li * ev.n + i[e]] = g[e];
            const unsigned peers = __match_any_sync(FULL, g[e]);
            if (g[e] != KB_NONE && lane == (unsigned)(__ffs(peers) - 1)) atomicAdd(&gcnt[g[e]], (uint32_t)__popc(peers));
        }
    }
}

// ---- P2: claim the group's segment on first touch, then scatter
__device__ __forceinline__ unsigned long long d_group_alloc(const FanScratch &sc, uint32_t g)
{
    unsigned long long a = __ldcg(&sc.galloc[g]);
    if (a < FAN_BUSY) return a;
    const unsigned long long old = atomicCAS(&sc.galloc[g], FAN_UNSET, FAN_BUSY);
    if (old == FAN_UNSET) {
        const uint32_t n = ldcg32(&sc.gcnt[g]);
        uint32_t cls = KB_NONE;
        if (n > sc.big_t) {
            const uint32_t slot = atomicAdd(&sc.ctl[FC_NLARGE], 1u);
            if (slot < sc.max_large) {  // cannot overflow: sum(gcnt) <= E * n_lens
                cls = slot;
                sc.large_list[slot] = g;
            }
        } else if (n > 32) {
            sc.med_list[atomicAdd(&sc.ctl[FC_NMED], 1u)] = g;
        }
        const uint32_t base = atomicAdd(&sc.ctl[FC_CURSOR], n);
        a = ((unsigned long long)cls << 32) | base;
        __threadfence();
        atomicExch(&sc.galloc[g], a);
        return a;
    }
    if (old < FAN_BUSY) return old;
    // another warp is allocating (it never waits for anybody): spin until it has published
    do {
        __nanosleep(32);
        a = *(volatile unsigned long long *)&sc.galloc[g];
    } while (a >= FAN_BUSY);
    return a;
}

__device__ __forceinline__ void d_scatter(const FanScratch &sc, uint32_t n_events, uint32_t n_lens, uint32_t vblock)
{
    const uint32_t i = vblock * blockDim.x + threadIdx.x;
    const uint32_t lane = threadIdx.x & 31;
    const bool valid = i < n_events;
    for (uint32_t li = 0; li < n_lens; li++) {
        const uint32_t g = valid ? ldcg32(&sc.ematch[(uint64_t)li * n_events + i]) : KB_NONE;  // written by another CTA in P1
        const unsigned peers = __match_any_sync(FULL, g);
        if (g == KB_NONE) continue;
        const uint32_t leader = __ffs(peers) - 1;
        unsigned long long a = 0;
        uint32_t fill = 0;
        if (lane == leader) {
            a = d_group_alloc(sc, g);
            if ((uint32_t)(a >> 32) == KB_NONE) fill = atomicAdd(&sc.gfill[g], (uint32_t)__popc(peers));
        }
        const uint32_t base = __shfl_sync(peers, (uint32_t)a, leader);
        const uint32_t cls = __shfl_sync(peers, (uint32_t)(a >> 32), leader);
        fill = __shfl_sync(peers, fill, leader);
        if (cls != KB_NONE) {
            // the 32 events of this warp are exactly one bitmap word of the group
            if (lane == leader) sc.bitmaps[(uint64_t)cls * sc.bm_words + (i >> 5)] = peers;
        } else {
            sc.seg[base + fill + __popc(peers & ((1u << lane) - 1))] = i;
        }
    }
}

__device__ __forceinline__ uint32_t block_excl_scan_u32(uint32_t v, uint32_t *wsum /* 33 */, uint32_t &total)
{
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t o = __shfl_up_sync(FULL, inc, d);
        if (lane >= (unsigned)d) inc += o;
    }
    if (lane == 31) wsum[wid] = inc;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t run = 0;
        for (uint32_t k = 0; k < nw; k++) {
            uint32_t x = wsum[k];
            wsum[k] = run;
            run += x;
        }
        wsum[32] = run;
    }
    __syncthreads();
    const uint32_t ex = wsum[wid] + inc - v;
    total = wsum[32];
    __syncthreads();
    return ex;
}

// ---- P3a: one CTA per medium group (33..big_t entries): shared-memory bitmap over windows of its [min, max]
__device__ __forceinline__ void d_sort_medium(const FanScratch &sc, uint32_t *bm, uint32_t *wsum, uint32_t *red)
{
    const uint32_t nmed = ldcg32(&sc.ctl[FC_NMED]);
    for (uint32_t bi = blockIdx.x; bi < nmed; bi += gridDim.x) {
        const uint32_t g = ldcg32(&sc.med_list[bi]);
        const uint32_t n = ldcg32(&sc.gcnt[g]), base = (uint32_t)__ldcg(&sc.galloc[g]);
        if (threadIdx.x == 0) {
            red[0] = 0xFFFFFFFFu;
            red[1] = 0;
        }
        __syncthreads();
        uint32_t mn = 0xFFFFFFFFu, mx = 0;
        for (uint32_t j = threadIdx.x; j < n; j += blockDim.x) {
            const uint32_t v = ldcg32(&sc.seg[base + j]);
            mn = min(mn, v);
            mx = max(mx, v);
        }
        atomicMin(&red[0], mn);
        atomicMax(&red[1], mx);
        __syncthreads();
        mn = red[0];
        mx = red[1];
        uint32_t outpos = 0;
        for (uint64_t w0 = mn & ~31u; w0 <= mx; w0 += (uint64_t)BM_WORDS * 32) {
            const uint64_t need_words = ((uint64_t)mx - w0) / 32 + 1;
            const uint32_t nwords = need_words < BM_WORDS ? (uint32_t)need_words : BM_WORDS;
            for (uint32_t j = threadIdx.x; j < nwords; j += blockDim.x) bm[j] = 0;
            __syncthreads();
            for (uint32_t j = threadIdx.x; j < n; j += blockDim.x) {
                const uint64_t v = ldcg32(&sc.seg[base + j]);
                if (v >= w0 && v < w0 + (uint64_t)nwords * 32) {
                    const uint32_t d = (uint32_t)(v - w0);
                    atomicOr(&bm[d >> 5], 1u << (d & 31));
                }
            }
            __syncthreads();
            // ordered expansion: each thread owns a contiguous run of words
            const uint32_t per = (nwords + blockDim.x - 1) / blockDim.x;
            const uint32_t wlo = min(nwords, threadIdx.x * per), whi = min(nwords, wlo + per);
            uint32_t cnt = 0;
            for (uint32_t j = wlo; j < whi; j++) cnt += __popc(bm[j]);
            uint32_t total;
            uint32_t at = outpos + block_excl_scan_u32(cnt, wsum, total);
            for (uint32_t j = wlo; j < whi; j++) {
                uint32_t bits = bm[j];
                while (bits) {
                    const uint32_t b = __ffs(bits) - 1;
                    bits &= bits - 1;
                    sc.sorted[base + at++] = (uint32_t)(w0 + (uint64_t)j * 32 + b);
                }
            }
            outpos += total;
            __syncthreads();
        }
        __syncthreads();
    }
}

// ---- P3b: large groups: ordered expansion of the global bitmap; job = (large group, chunk of FAN_THREADS words)
__device__ __forceinline__ void d_expand_large(const FanScratch &sc, uint32_t *wsum, uint32_t *pre_sp)
{
    uint32_t &pre_s = *pre_sp;
    const uint32_t nlarge = min(ldcg32(&sc.ctl[FC_NLARGE]), sc.max_large);
    for (uint32_t job = blockIdx.x; job < nlarge * sc.chunks_per_group; job += gridDim.x) {
        const uint32_t slot = job / sc.chunks_per_group, chunk = job % sc.chunks_per_group;
        const uint32_t g = ldcg32(&sc.large_list[slot]);
        const uint32_t *bm = sc.bitmaps + (uint64_t)slot * sc.bm_words;
        // matches in the words before this chunk
        uint32_t part = 0;
        for (uint32_t j = threadIdx.x; j < chunk * FAN_THREADS; j += blockDim.x) part += __popc(ldcg32(&bm[j]));
        uint32_t tot;
        block_excl_scan_u32(part, wsum, tot);
        if (threadIdx.x == 0) pre_s = tot;
        __syncthreads();
        const uint32_t wi = chunk * FAN_THREADS + threadIdx.x;
        uint32_t bits = wi < sc.bm_words ? ldcg32(&bm[wi]) : 0;
        uint32_t total;
        uint32_t at = (uint32_t)__ldcg(&sc.galloc[g]) + pre_s + block_excl_scan_u32(__popc(bits), wsum, total);
        while (bits) {
            const uint32_t b = __ffs(bits) - 1;
            bits &= bits - 1;
            sc.sorted[at++] = wi * 32 + b;
        }
        __syncthreads();
    }
}

// ---- P4: deliveries per watcher.  A warp takes TWO watchers at a time, one per 16-lane half: a namespace watcher's
// group holds a handful of events (<= 16 in 99 % of the cases), which a half-warp rank-sorts in registers; a watcher whose
// group is larger (or medium / large: already sorted by P3) is then handled by the whole warp.
__device__ __forceinline__ void d_watcher_big(const TabDev &tb, const FanScratch &sc, bool mono, uint32_t w, uint32_t n,
                                              uint32_t base, uint32_t lane)
{
    const uint64_t mr = __ldg(tb.wminrev + w);
    uint32_t lo = 0, cnt = 0;
    if (n <= 32) {
        // small group: rank sort in registers; every watcher of the group writes the same ascending segment
        const uint32_t v = lane < n ? ldcg32(&sc.seg[base + lane]) : 0xFFFFFFFFu;
        uint32_t rank = 0;
#pragma unroll
        for (int j = 0; j < 32; j++) {
            const uint32_t o = __shfl_sync(FULL, v, j);
            rank += (o < v) ? 1u : 0u;  // event indices inside one group are distinct
        }
        if (lane < n) sc.sorted[base + rank] = v;
        const bool keep = lane < n && ldcg64(&sc.pm[v]) >= mr;
        cnt = __popc(__ballot_sync(FULL, keep));
        lo = mono ? n - cnt : 0;
    } else if (mono) {
        // survivors are a suffix of the ascending segment: 32-ary search for the first event at or above min_rev
        const uint32_t *M = sc.sorted + base;
        uint32_t hi = n;
        for (;;) {
            const uint32_t span = hi - lo;
            if (span == 0) break;
            if (span <= 32) {
                const bool ge = lane < span && ldcg64(&sc.pm[ldcg32(&M[lo + lane])]) >= mr;
                const unsigned m = __ballot_sync(FULL, ge);
                lo += m ? (uint32_t)(__ffs(m) - 1) : span;
                break;
            }
            const uint32_t piv = lo + (uint32_t)(((uint64_t)span * (lane + 1)) / 33);
            const bool ge = ldcg64(&sc.pm[ldcg32(&M[piv])]) >= mr;
            const int k = __popc(~__ballot_sync(FULL, ge));  // pivots below min_rev: a prefix of the lanes
            uint32_t nlo = lo, nhi = hi;
            if (k > 0) nlo = __shfl_sync(FULL, piv, k - 1) + 1;
            if (k < 32) nhi = __shfl_sync(FULL, piv, k);
            lo = nlo;
            hi = nhi;
        }
        cnt = n - lo;
    } else {
        const uint32_t *M = sc.sorted + base;
        for (uint32_t c = 0; c < n; c += 32) {
            const uint32_t j = c + lane;
            const bool keep = j < n && ldcg64(&sc.pm[ldcg32(&M[j])]) >= mr;
            cnt += __popc(__ballot_sync(FULL, keep));
        }
    }
    if (lane == 0) {
        sc.wcnt[w] = cnt;
        sc.wsrc[w] = base;
        sc.wn[w] = n;
        sc.wlo[w] = lo;
    }
}

__device__ __forceinline__ void d_watcher_count(const TabDev &tb, const FanScratch &sc, bool mono)
{
    const uint32_t lane = threadIdx.x & 31, half = lane >> 4, sub = lane & 15;
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t w0 = ((blockIdx.x * blockDim.x + threadIdx.x) >> 5) * 2; w0 < tb.n_ids; w0 += warps * 2) {
        const uint32_t w = w0 + half;
        const bool have = w < tb.n_ids;
        const uint32_t g = have ? __ldg(tb.wgroup + w) : KB_NONE;
        uint32_t n = 0, base = 0;
        unsigned long long a = FAN_UNSET;
        if (g != KB_NONE) a = __ldcg(&sc.galloc[g]);
        if (a < FAN_BUSY) {  // the group matched at least one event
            n = ldcg32(&sc.gcnt[g]);
            base = (uint32_t)a;
        }
        const unsigned hmask = half ? 0xFFFF0000u : 0x0000FFFFu;  // the halves may diverge: they only sync among themselves
        if (n <= 16) {
            // this half-warp's watcher: rank sort of <= 16 entries with 16-lane shuffles
            const uint64_t mr = have ? __ldg(tb.wminrev + w) : 0;
            const uint32_t v = sub < n ? ldcg32(&sc.seg[base + sub]) : 0xFFFFFFFFu;
            uint32_t rank = 0;
#pragma unroll
            for (int j = 0; j < 16; j++) {
                const uint32_t o = __shfl_sync(hmask, v, j, 16);
                rank += (o < v) ? 1u : 0u;
            }
            if (sub < n) sc.sorted[base + rank] = v;
            const bool keep = sub < n && ldcg64(&sc.pm[v]) >= mr;
            const uint32_t cnt = __popc(__ballot_sync(hmask, keep));
            if (sub == 0 && have) {
                sc.wcnt[w] = cnt;
                sc.wsrc[w] = base;
                sc.wn[w] = n;
                sc.wlo[w] = mono ? n - cnt : 0;
            }
        }
        __syncwarp();
        // watchers with a bigger group: the whole warp, one after the other
        const uint32_t n0 = __shfl_sync(FULL, n, 0), n1 = __shfl_sync(FULL, n, 16);
        const uint32_t b0 = __shfl_sync(FULL, base, 0), b1 = __shfl_sync(FULL, base, 16);
        if (n0 > 16) d_watcher_big(tb, sc, mono, w0, n0, b0, lane);
        if (n1 > 16 && w0 + 1 < tb.n_ids) d_watcher_big(tb, sc, mono, w0 + 1, n1, b1, lane);
    }
}

// ---- P5 (one CTA): exclusive prefix of the per-watcher delivery counts; scratch back to its initial state
__device__ __forceinline__ void d_finish(const TabDev &tb, const FanScratch &sc, uint64_t *ws /* 33 */)
{
    // Exclusive prefix of the per-watcher counts by ONE CTA with coalesced accesses: every warp owns a contiguous chunk
    // of watchers and walks it 32 at a time (first pass: chunk totals; second pass: warp scans with the running carry).
    // The offsets go to the device scratch, to the output buffer and -- 256 contiguous bytes per warp store -- to the
    // pinned host copy.  (The first version gave each thread a contiguous run: 8-byte PCIe writes 216 bytes apart; with
    // the scratch zeroing it made this tail ~50 us of a 110 us kernel.)
    const uint32_t W = tb.n_ids, lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const uint32_t per = ((W + nw - 1) / nw + 31) & ~31u;  // watchers per warp, a multiple of 32
    const uint32_t a = min(W, wid * per), b = min(W, a + per);
    uint64_t sum = 0;
    for (uint32_t w = a + lane; w < b; w += 32) sum += ldcg32(&sc.wcnt[w]);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) sum += __shfl_xor_sync(FULL, sum, d);
    if (lane == 0) ws[wid] = sum;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint64_t run = 0;
        for (uint32_t k = 0; k < nw; k++) {
            uint64_t x = ws[k];
            ws[k] = run;
            run += x;
        }
        ws[32] = run;
    }
    __syncthreads();
    uint64_t carry = ws[wid];
    for (uint32_t w0 = a; w0 < b; w0 += 32) {
        const uint32_t w = w0 + lane;
        const uint64_t c = w < b ? ldcg32(&sc.wcnt[w]) : 0;
        uint64_t inc = c;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            uint64_t o = __shfl_up_sync(FULL, inc, d);
            if (lane >= (unsigned)d) inc += o;
        }
        if (w < b) {
            const uint64_t at = carry + inc - c;
            sc.wstart[w] = at;
            sc.o_start[w] = at;
            sc.h_start[w] = at;
        }
        carry += __shfl_sync(FULL, inc, 31);
    }
    const uint32_t aborted = ldcg32(&sc.ctl[FC_ABORT]);
    if (threadIdx.x == 0) {
        sc.wstart[W] = ws[32];
        sc.o_start[W] = ws[32];
        sc.h_start[W] = ws[32];
        sc.total[0] = ws[32];
        // k_expand_write picks its path from this copy; bit 32 = a grid barrier timed out (the answer is void)
        sc.total[1] = (uint64_t)ldcg32(&sc.ctl[FC_NONMONO]) | ((uint64_t)aborted << 32);
        *sc.nlarge_w = min(ldcg32(&sc.ctl[FC_NLARGE]), sc.max_large);  // bitmap slots the NEXT call has to clear
    }
    __syncthreads();
    // the per-call control words back to zero (the group state itself is double buffered: the next call clears this set
    // in its first phase, see k_fanout)
    if (threadIdx.x < FC_WORDS && threadIdx.x != FC_GEN) sc.ctl[threadIdx.x] = 0;
    // the offsets in host memory, then the flag the host polls
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        sc.h_pub[1] = ws[32];
        sc.h_pub[2] = aborted;
        __threadfence_system();
        *(volatile uint64_t *)sc.h_pub = sc.epoch;
    }
}

__device__ __forceinline__ uint64_t fan_now_ns();

__device__ __forceinline__ uint64_t fan_now_ns()
{
    uint64_t t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

__global__ void __maxnreg__(80)  // 384 threads x 80 registers, see FAN_THREADS
k_fanout(EvDev ev, TabDev tb, FanScratch sc)
{
    // phase timestamps of CTA 0 (profiling: kb_prof_read reports them as fan:P1 .. fan:finish when profiling is on)
    const bool stamp = blockIdx.x == 0 && threadIdx.x == 0;
    uint64_t t_begin = 0;
    if (threadIdx.x == 0) {  // when did the LAST CTA of the grid get its SM? (ctl words 8..9 as one u64, zeroed at the end)
        t_begin = fan_now_ns();
        atomicMax((unsigned long long *)&sc.ctl[8], (unsigned long long)t_begin);
    }
    uint64_t t_p[4] = {0, 0, 0, 0};
    __shared__ uint32_t bm[BM_WORDS];
    __shared__ uint32_t wsum[33];
    __shared__ uint32_t red[2];
    __shared__ uint64_t ws64[33];
    __shared__ uint32_t last_s;
    // P1
    const uint32_t pm_blocks = (ev.nb * 32 + FAN_THREADS - 1) / FAN_THREADS;
    const uint32_t ev_blocks = tb.n_groups ? (ev.n + FAN_THREADS - 1) / FAN_THREADS : 0;
    const uint32_t ev_blocks3 = (ev_blocks + FAN_EPT - 1) / FAN_EPT;  // P1: a virtual block covers FAN_EPT x 256 events
    {   // the other set of group state (the previous call's) back to its initial state
        const uint64_t tid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (uint64_t)gridDim.x * blockDim.x;
        const uint32_t G = tb.n_groups;
        for (uint64_t i = tid; i < 2ull * (G + 1); i += nth) sc.z_gcnt[i] = 0;  // gcnt | gfill are contiguous
        for (uint64_t i = tid; i < G; i += nth) sc.z_galloc[i] = FAN_UNSET;
        const uint64_t zb = (uint64_t)min(ldcg32(sc.nlarge_r), sc.max_large) * sc.bm_words;
        for (uint64_t i = tid; i < zb; i += nth) sc.z_bitmaps[i] = 0;
    }
    for (uint32_t vb = blockIdx.x; vb < pm_blocks + ev_blocks3; vb += gridDim.x) {
        if (vb < pm_blocks)
            d_batch_pm(ev, sc.pm, &sc.ctl[FC_NONMONO], vb);
        else
            d_match_count(ev, tb, sc.ematch, sc.gcnt, vb - pm_blocks);
    }
    fan_grid_sync(sc.ctl, sc.gen_base + 1);
    if (stamp) t_p[0] = fan_now_ns();
    // P2
    for (uint32_t vb = blockIdx.x; vb < ev_blocks; vb += gridDim.x) d_scatter(sc, ev.n, tb.n_lens, vb);
    fan_grid_sync(sc.ctl, sc.gen_base + 2);
    if (stamp) t_p[1] = fan_now_ns();
    // P3
    d_sort_medium(sc, bm, wsum, red);
    d_expand_large(sc, wsum, red);
    fan_grid_sync(sc.ctl, sc.gen_base + 3);
    if (stamp) t_p[2] = fan_now_ns();
    // P4
    const bool mono = ldcg32(&sc.ctl[FC_NONMONO]) == 0;
    d_watcher_count(tb, sc, mono);
    if (stamp) {
        t_p[3] = fan_now_ns();
        sc.h_pub[3] = t_p[0] - t_begin;   // P1 + barrier
        sc.h_pub[4] = t_p[1] - t_p[0];    // P2 + barrier
        sc.h_pub[5] = t_p[2] - t_p[1];    // P3 + barrier
        sc.h_pub[6] = t_p[3] - t_p[2];    // P4 of this CTA
        sc.h_pub[7] = __ldcg((const unsigned long long *)&sc.ctl[8]) - t_begin;  // start of the last CTA - start of CTA 0
    }
    // P5: the last CTA to get here finishes alone; the end of the kernel is the barrier for what follows
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        last_s = atomicAdd(&sc.ctl[FC_DONE], 1u) == gridDim.x - 1;
        __threadfence();
    }
    __syncthreads();
    if (last_s) d_finish(tb, sc, ws64);
}

// monotone revisions: one thread per delivery (suffix copy)
__device__ __forceinline__ void d_expand_write(uint32_t n_ids, const uint32_t *__restrict__ wsrc,
                                               const uint32_t *__restrict__ wlo, const uint32_t *__restrict__ sorted,
                                               const uint64_t *__restrict__ wstart, uint64_t n_deliveries,
                                               uint32_t *__restrict__ out)
{
    for (uint64_t d = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; d < n_deliveries;
         d += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t lo = 0, hi = n_ids;  // last watcher with wstart[w] <= d
        while (hi - lo > 1) {
            const uint32_t mid = (lo + hi) >> 1;
            if (wstart[mid] <= d) lo = mid; else hi = mid;
        }
        const uint32_t w = lo;
        out[d] = sorted[wsrc[w] + wlo[w] + (uint32_t)(d - wstart[w])];
    }
}

// non-monotone revisions (general case): warp per watcher, ordered filtered copy
__device__ __forceinline__ void d_expand_write_general(uint32_t n_ids, const uint64_t *__restrict__ wminrev,
                                                       const uint32_t *__restrict__ wsrc, const uint32_t *__restrict__ wn,
                                                       const uint32_t *__restrict__ sorted,
                                                       const uint64_t *__restrict__ pm,
                                                       const uint64_t *__restrict__ wstart, uint32_t *__restrict__ out)
{
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < n_ids; w += warps) {
        const uint32_t n = wn[w];
        const uint32_t *M = sorted + wsrc[w];
        const uint64_t mr = wminrev[w];
        const uint64_t o = wstart[w];
        uint64_t total = 0;
        for (uint32_t c = 0; c < n; c += 32) {
            const uint32_t j = c + lane;
            const uint32_t e = j < n ? M[j] : 0;
            const bool keep = j < n && pm[e] >= mr;
            const unsigned m = __ballot_sync(FULL, keep);
            if (keep) out[o + total + __popc(m & ((1u << lane) - 1))] = e;
            total += __popc(m);
        }
    }
}

// one launch for both output paths: revisions monotone -> one thread per delivery; otherwise warp per watcher
__global__ void __launch_bounds__(256)
k_expand_write(uint32_t n_ids, const uint64_t *__restrict__ wminrev, const uint32_t *__restrict__ wsrc,
               const uint32_t *__restrict__ wn, const uint32_t *__restrict__ wlo, const uint32_t *__restrict__ sorted,
               const uint64_t *__restrict__ pm, const uint64_t *__restrict__ total /* [0] deliveries [1] non-monotone */,
               const uint64_t *__restrict__ wstart, uint64_t capacity, uint32_t *__restrict__ out)
{
    const uint64_t n_deliveries = wstart[n_ids];
    if (n_deliveries > capacity) return;  // the host sees the total, grows the buffer and launches again
    if ((total[1] >> 32) != 0) return;  // aborted match
    if ((uint32_t)total[1] == 0)
        d_expand_write(n_ids, wsrc, wlo, sorted, wstart, n_deliveries, out);
    else
        d_expand_write_general(n_ids, wminrev, wsrc, wn, sorted, pm, wstart, out);
}

uint64_t fnv1a(const std::string &s)
{
    uint64_t h = FNV_OFFSET;
    for (unsigned char c : s) h = (h ^ c) * FNV_PRIME;
    return h;
}

inline size_t arena_align(size_t x) { return (x + 255) & ~(size_t)255; }

// a view of `bytes` at `cursor` inside the arena (the caller made sure it fits); views are never freed on their own
void arena_view(WatchTablesDev &T, size_t &cursor, DBuf &view, size_t bytes)
{
    view.p = (uint8_t *)T.arena.p + cursor;
    view.cap = 0;
    cursor += arena_align(std::max<size_t>(bytes, 16));
}

// (re)allocate the arena for `need` bytes and put the L2 access-policy window of the context's stream over it
int arena_reserve(kb_ctx *ctx, WatchTablesDev &T, size_t need)
{
    if (T.arena.p && T.arena.cap >= need) return KB_OK;
    KB_TRY(dbuf_ensure(ctx, T.arena, need + need / 2));
    T.scratch_clean = false;
    ctx->watch_dirty = true;  // the tables lived in the old allocation
    cudaStreamAttrValue attr;
    memset(&attr, 0, sizeof(attr));
    int max_win = 0, persist_max = 0;
    cudaDeviceGetAttribute(&max_win, cudaDevAttrMaxAccessPolicyWindowSize, ctx->device);
    cudaDeviceGetAttribute(&persist_max, cudaDevAttrMaxPersistingL2CacheSize, ctx->device);
    const size_t setaside = std::min<size_t>((size_t)persist_max, (size_t)32 << 20);
    // Off unless KB_L2_PERSIST=1.  Measured (profiles/r02_l2_persist_ab.txt): with a 32 MB set-aside the fan-out itself does
    // not get faster inside a step (231 -> 290 us) and the scan context's gather loses the L2 it uses as a write buffer
    // (185 -> 250 us): 0.327 -> 0.381 ms per step.
    static const bool l2_persist = getenv("KB_L2_PERSIST") && atoi(getenv("KB_L2_PERSIST")) == 1;
    if (max_win > 0 && setaside > 0 && l2_persist) {
        cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, setaside);  // device-wide; the same value from every context
        attr.accessPolicyWindow.base_ptr = T.arena.p;
        attr.accessPolicyWindow.num_bytes = std::min<size_t>(T.arena.cap, (size_t)max_win);
        attr.accessPolicyWindow.hitRatio = (float)std::min(1.0, (double)setaside / (double)attr.accessPolicyWindow.num_bytes);
        attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
        cudaStreamSetAttribute(ctx->stream, cudaStreamAttributeAccessPolicyWindow, &attr);
    }
    cudaGetLastError();  // the window is an optimisation: a part that refuses it still computes the same answers
    return KB_OK;
}

int upload(kb_ctx *ctx, DBuf &b, const void *src, size_t bytes)
{
    if (bytes) KB_CUDA(ctx, cudaMemcpyAsync(b.p, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return KB_OK;
}

// rebuild the device tables after kb_watch_add / kb_watch_del
int rebuild_tables(kb_ctx *ctx)
{
    if (!ctx->wt) ctx->wt = new WatchTablesDev();
    WatchTablesDev &T = *ctx->wt;
    const uint32_t n_ids = (uint32_t)ctx->watchers.size();
    std::map<std::string, std::vector<uint32_t>> groups;  // ordered: deterministic group ids
    uint32_t max_len = 0;
    for (uint32_t w = 0; w < n_ids; w++)
        if (ctx->watchers[w].live) {
            groups[ctx->watchers[w].prefix].push_back(w);
            max_len = std::max<uint32_t>(max_len, (uint32_t)ctx->watchers[w].prefix.size());
        }
    const uint32_t G = (uint32_t)groups.size();
    // every prefix zero padded to the same stride, so an entry of the hash table (hash, length, group) is all a probe reads
    // before the byte-exact verify
    const uint32_t pstride16 = std::max<uint32_t>(1, (max_len + 15) / 16);
    if ((uint64_t)G * pstride16 * 16 > (1ull << 32)) return kb_fail(ctx, KB_ELIMIT, "watch prefixes exceed 4 GiB");
    std::vector<uint8_t> gprefix((size_t)std::max(G, 1u) * pstride16 * 16, 0);
    std::vector<uint32_t> glen(G), wgroup(std::max(n_ids, 1u), KB_NONE), lens;
    std::vector<uint64_t> ghash(std::max(G, 1u)), wminrev(std::max(n_ids, 1u), 0);
    uint32_t gi = 0;
    for (auto &kv : groups) {
        const std::string &p = kv.first;
        glen[gi] = (uint32_t)p.size();
        ghash[gi] = fnv1a(p);
        if (!p.empty()) memcpy(gprefix.data() + (size_t)gi * pstride16 * 16, p.data(), p.size());
        for (uint32_t w : kv.second) wgroup[w] = gi;
        lens.push_back((uint32_t)p.size());
        gi++;
    }
    for (uint32_t w = 0; w < n_ids; w++) wminrev[w] = ctx->watchers[w].min_rev;
    std::sort(lens.begin(), lens.end());
    lens.erase(std::unique(lens.begin(), lens.end()), lens.end());
    uint32_t tsize = 16;
    while (tsize < 2 * G + 2) tsize <<= 1;
    std::vector<uint4> table(tsize, make_uint4(0, 0, 0, KB_NONE));
    for (uint32_t g = 0; g < G; g++) {
        uint32_t s = slot_of(ghash[g], glen[g], tsize - 1);
        while (table[s].w != KB_NONE) s = (s + 1) & (tsize - 1);
        table[s] = make_uint4((uint32_t)ghash[g], (uint32_t)(ghash[g] >> 32), glen[g], g);
    }
    if (lens.empty()) lens.push_back(0);
    // tables at the head of the arena, the per-call scratch (sized by the last burst) behind them
    const size_t tab_bytes = arena_align(gprefix.size()) + arena_align(wgroup.size() * 4) + arena_align(wminrev.size() * 8) +
                             arena_align(lens.size() * 4) + arena_align(table.size() * 16);
    KB_TRY(arena_reserve(ctx, T, tab_bytes + T.scr_bytes + 4096));
    size_t cur = 0;
    arena_view(T, cur, T.gprefix, gprefix.size());
    arena_view(T, cur, T.wgroup, wgroup.size() * 4);
    arena_view(T, cur, T.wminrev, wminrev.size() * 8);
    arena_view(T, cur, T.lens, lens.size() * 4);
    arena_view(T, cur, T.table, table.size() * 16);
    if (cur != T.tab_end) T.scr_sig = 0;  // the scratch behind the tables moves
    T.tab_end = cur;
    KB_TRY(upload(ctx, T.gprefix, gprefix.data(), gprefix.size()));
    KB_TRY(upload(ctx, T.wgroup, wgroup.data(), wgroup.size() * 4));
    KB_TRY(upload(ctx, T.wminrev, wminrev.data(), wminrev.size() * 8));
    KB_TRY(upload(ctx, T.lens, lens.data(), lens.size() * 4));
    KB_TRY(upload(ctx, T.table, table.data(), table.size() * 16));
    KB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // the host vectors die here
    T.n_ids = n_ids;
    T.n_groups = G;
    T.n_lens = G ? (uint32_t)lens.size() : 0;
    T.table_size = tsize;
    T.max_len = max_len;
    T.pstride16 = pstride16;
    T.scratch_clean = false;  // the group count changed: the scratch is laid out again
    ctx->watch_dirty = false;
    return KB_OK;
}

uint32_t needed_stride(kb_ctx *ctx)
{
    uint32_t max_len = 0;
    for (auto &w : ctx->watchers)
        if (w.live) max_len = std::max<uint32_t>(max_len, (uint32_t)w.prefix.size());
    return std::max<uint32_t>(16, (max_len + 15) / 16 * 16);
}

int events_upload_locked(kb_ctx *ctx, const kb_events *ev, kb_events_dev *d)
{
    if (ev->n >= 0xFFFFFFF0ull) return kb_fail(ctx, KB_ELIMIT, "too many events");
    const uint32_t n = (uint32_t)ev->n;
    const uint32_t stride = needed_stride(ctx);
    const uint32_t nb = ev->batch_off && ev->n_batches ? (uint32_t)ev->n_batches : 1;
    // pinned staging: [keys n*stride][klen n*4][rev n*8][batch_off (nb+1)*8]
    const size_t kbytes = (size_t)n * stride, total = kbytes + (size_t)n * 12 + (size_t)(nb + 1) * 8 + 64;
    KB_TRY(hbuf_ensure(ctx, ctx->h_stage, total));
    uint8_t *h = (uint8_t *)ctx->h_stage.p;
    uint32_t *hl = (uint32_t *)(h + kbytes);
    uint64_t *hr = (uint64_t *)(h + kbytes + (size_t)n * 4);
    // keep 8-byte alignment for the u64 arrays
    size_t rev_off = (kbytes + (size_t)n * 4 + 7) & ~(size_t)7;
    hr = (uint64_t *)(h + rev_off);
    uint64_t *hb = hr + n;
    for (uint32_t i = 0; i < n; i++) {
        const uint64_t o = ev->key_off[i], l = ev->key_off[i + 1] - o;
        const uint32_t c = (uint32_t)std::min<uint64_t>(l, stride);
        uint8_t *dst = h + (size_t)i * stride;
        memcpy(dst, ev->keys + o, c);
        if (c < stride) memset(dst + c, 0, stride - c);
        hl[i] = (uint32_t)std::min<uint64_t>(l, 0xFFFFFFFFull);
    }
    if (n) memcpy(hr, ev->rev, (size_t)n * 8);
    if (ev->batch_off && ev->n_batches) {
        memcpy(hb, ev->batch_off, (size_t)(nb + 1) * 8);
    } else {
        hb[0] = 0;
        hb[1] = n;
    }
    KB_TRY(dbuf_ensure(ctx, d->keys, std::max<size_t>(kbytes, 16)));
    KB_TRY(dbuf_ensure(ctx, d->klen, std::max<size_t>((size_t)n * 4, 16)));
    KB_TRY(dbuf_ensure(ctx, d->rev, std::max<size_t>((size_t)n * 8, 16)));
    KB_TRY(dbuf_ensure(ctx, d->batch_off, (size_t)(nb + 1) * 8));
    if (n) {
        KB_CUDA(ctx, cudaMemcpyAsync(d->keys.p, h, kbytes, cudaMemcpyHostToDevice, ctx->stream));
        KB_CUDA(ctx, cudaMemcpyAsync(d->klen.p, hl, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream));
        KB_CUDA(ctx, cudaMemcpyAsync(d->rev.p, hr, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
    }
    KB_CUDA(ctx, cudaMemcpyAsync(d->batch_off.p, hb, (size_t)(nb + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    d->n = n;
    d->nb = nb;
    d->stride = stride;
    return KB_OK;
}

void events_release(kb_events_dev *d)
{
    if (d->keys.p) cudaFree(d->keys.p);
    if (d->klen.p) cudaFree(d->klen.p);
    if (d->rev.p) cudaFree(d->rev.p);
    if (d->batch_off.p) cudaFree(d->batch_off.p);
    d->keys = d->klen = d->rev = d->batch_off = DBuf();
}

}  // namespace

void watch_tables_free(kb_ctx *ctx)
{
    if (!ctx->wt) return;
    WatchTablesDev &T = *ctx->wt;
    if (T.arena.p) cudaFree(T.arena.p);  // every other buffer is a view into it
    if (T.ev_fan) cudaEventDestroy(T.ev_fan);
    for (auto e : T.ev_write)
        if (e) cudaEventDestroy(e);
    delete ctx->wt;
    ctx->wt = nullptr;
    if (ctx->ev_scratch) {
        events_release(ctx->ev_scratch);
        delete ctx->ev_scratch;
        ctx->ev_scratch = nullptr;
    }
}

extern "C" int kb_watch_add(kb_ctx *ctx, const uint8_t *prefix, uint64_t prefix_len, uint64_t min_rev, uint32_t *id)
{
    if (!ctx || !id || (prefix_len && !prefix)) return KB_EINVAL;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (prefix_len > 65535) return kb_fail(ctx, KB_ELIMIT, "watch prefix longer than 65535 bytes");
    Watcher w;
    w.prefix.assign((const char *)prefix, (size_t)prefix_len);
    w.min_rev = min_rev;
    w.live = true;
    if (!ctx->free_watch_ids.empty()) {  // ids of cancelled watches are reused so the id space stays dense
        *id = ctx->free_watch_ids.back();
        ctx->free_watch_ids.pop_back();
        ctx->watchers[*id] = w;
    } else {
        ctx->watchers.push_back(w);
        *id = (uint32_t)ctx->watchers.size() - 1;
    }
    ctx->watch_dirty = true;
    return KB_OK;
}

extern "C" int kb_watch_del(kb_ctx *ctx, uint32_t id)
{
    if (!ctx) return KB_EINVAL;
    std::lock_guard<std::mutex> g(ctx->mu);
    if (id >= ctx->watchers.size() || !ctx->watchers[id].live) return kb_fail(ctx, KB_EINVAL, "unknown watcher %u", id);
    ctx->watchers[id].live = false;
    ctx->free_watch_ids.push_back(id);
    ctx->watch_dirty = true;
    return KB_OK;
}

extern "C" int kb_watch_count(kb_ctx *ctx, uint64_t *n)
{
    if (!ctx || !n) return KB_EINVAL;
    std::lock_guard<std::mutex> g(ctx->mu);
    uint64_t c = 0;
    for (auto &w : ctx->watchers) c += w.live ? 1 : 0;
    *n = c;
    return KB_OK;
}

extern "C" int kb_events_upload(kb_ctx *ctx, const kb_events *ev, kb_events_dev **out)
{
    if (!ctx || !ev || !out || (ev->n && (!ev->keys || !ev->key_off || !ev->rev))) return KB_EINVAL;
    std::lock_guard<std::mutex> g(ctx->mu);
    cudaSetDevice(ctx->device);
    kb_events_dev *d = new kb_events_dev();
    int rc = events_upload_locked(ctx, ev, d);
    if (rc == KB_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess) rc = kb_fail(ctx, KB_ECUDA, "event upload");
    if (rc != KB_OK) {
        events_release(d);
        delete d;
        return rc;
    }
    *out = d;
    return KB_OK;
}

extern "C" void kb_events_free(kb_ctx *ctx, kb_events_dev *ev)
{
    if (!ev) return;
    if (ctx) {
        std::lock_guard<std::mutex> g(ctx->mu);
        cudaSetDevice(ctx->device);
        cudaStreamSynchronize(ctx->stream);
        events_release(ev);
    }
    delete ev;
}

// the delivery total, handed to the host through mapped pinned memory as soon as it is known (behind the offsets copy,
// in front of the write kernel): a device-resident match returns while its delivery lists are still being written
__global__ void k_publish_total(const uint64_t *__restrict__ total, uint64_t *host, uint64_t epoch)
{
    if (threadIdx.x == 0) {
        host[1] = total[0];
        host[2] = total[1] >> 32;  // 1: a grid barrier of k_fanout timed out
        __threadfence_system();
        *(volatile uint64_t *)host = epoch;
    }
}

static int wpub_wait(kb_ctx *ctx, uint64_t epoch)
{
    volatile uint64_t *flag = ctx->h_wpub;
    for (uint64_t spins = 1;; spins++) {
        if (*flag == epoch) return KB_OK;
        kb_cpu_relax();
        if ((spins & 0xFFFF) == 0) {
            const cudaError_t q = cudaStreamQuery(ctx->stream);
            if (q == cudaSuccess) return *flag == epoch ? KB_OK : kb_fail(ctx, KB_ECUDA, "watch match: total was not published");
            if (q != cudaErrorNotReady) return kb_cuda_fail(ctx, q, "watch match");
        }
    }
}

static int match_locked(kb_ctx *ctx, const kb_events_dev *d, int out_mode, kb_result **out)
{
    kb_tp tseg = kb_now();
    if (ctx->watch_dirty || !ctx->wt) {
        KB_CUDA(ctx, cudaStreamSynchronize(ctx->stream2));  // the previous burst's write still reads the tables
        KB_TRY(rebuild_tables(ctx));
    }
    WatchTablesDev &T = *ctx->wt;
    if (d->stride < needed_stride(ctx))
        return kb_fail(ctx, KB_ESTATE, "event slab was uploaded for shorter watcher prefixes (stride %u < %u); upload again",
                       d->stride, needed_stride(ctx));
    const uint32_t E = d->n, G = T.n_groups, W = T.n_ids, NL = std::max(T.n_lens, 1u);
    const uint64_t seg_cap = std::max<uint64_t>((uint64_t)E * NL, 1);
    if (seg_cap >= 0xFFFFFFF0ull) return kb_fail(ctx, KB_ELIMIT, "events x distinct prefix lengths exceeds 2^32");
    // groups matching more than big_t events get a global bitmap; at most E*NL/big_t of them can exist
    const uint32_t big_t = std::max<uint32_t>(1024, E / 64);
    const uint32_t max_large = (uint32_t)(seg_cap / big_t) + 1;
    const uint32_t bm_words = (E + 31) / 32;
    const uint32_t chunks_per_group = (bm_words + FAN_THREADS - 1) / FAN_THREADS;
    const size_t gstate_words = (size_t)4 * (G + 1) + FC_WORDS + 4;  // two sets of gcnt | gfill, control words, nlarge[2]
    const size_t bitmap_bytes = std::max<size_t>((size_t)max_large * bm_words * 4, 16);
    // per-call scratch behind the tables (one arena, see WatchTablesDev); a layout change voids the "clean" state
    // (group state -- gcnt | gfill, galloc, bitmaps -- twice: the sets alternate between calls)
    // (the last five exist twice -- see wr_set; each copy starts on an arena boundary)
    const size_t one[5] = {arena_align(seg_cap * 4), arena_align(std::max<size_t>((size_t)E * 8, 16)), arena_align((size_t)(W + 1) * 16),
                           arena_align((size_t)(W + 2) * 8), arena_align(16)};
    const size_t sizes[11] = {gstate_words * 4, (size_t)2 * (G + 1) * 8, 2 * bitmap_bytes, (size_t)(G + max_large + 2) * 4, seg_cap * 4,
                              seg_cap * 4, 2 * one[0], 2 * one[1], 2 * one[2], 2 * one[3], 2 * one[4]};
    size_t scr = 0, sig = 1469598103934665603ull;
    for (size_t x : sizes) {
        scr += arena_align(std::max<size_t>(x, 16));
        sig = (sig ^ x) * 1099511628211ull;
    }
    if (T.tab_end + scr > T.arena.cap) {
        KB_CUDA(ctx, cudaStreamSynchronize(ctx->stream2));
        T.scr_bytes = scr;
        KB_TRY(arena_reserve(ctx, T, T.tab_end + scr + 4096));
        KB_TRY(rebuild_tables(ctx));  // the tables moved with the arena
    }
    T.scr_bytes = std::max(T.scr_bytes, scr);
    if (sig != T.scr_sig) T.scratch_clean = false;
    T.scr_sig = sig;
    {
        size_t cur = T.tab_end;
        DBuf *views[11] = {&T.gstate, &T.galloc, &T.bitmaps, &T.lists, &T.ematch, &T.seg, &T.seg_sorted, &T.pm, &T.wstate,
                           &T.wstart, &T.total};
        for (int i = 0; i < 11; i++) arena_view(T, cur, *views[i], sizes[i]);
    }

    EvDev ev;
    ev.keys = (const uint4 *)d->keys.p;
    ev.klen = (const uint32_t *)d->klen.p;
    ev.rev = (const uint64_t *)d->rev.p;
    ev.batch_off = (const uint64_t *)d->batch_off.p;
    ev.n = E;
    ev.nb = d->nb;
    ev.stride16 = d->stride / 16;
    TabDev tb;
    tb.gprefix = (const uint4 *)T.gprefix.p;
    tb.wgroup = (const uint32_t *)T.wgroup.p;
    tb.wminrev = (const uint64_t *)T.wminrev.p;
    tb.lens = (const uint32_t *)T.lens.p;
    tb.table = (const uint4 *)T.table.p;
    tb.n_ids = W;
    tb.n_groups = G;
    tb.n_lens = T.n_lens;
    tb.mask = T.table_size - 1;
    tb.max_len = T.max_len;
    tb.pstride16 = T.pstride16;
    FanScratch sc;
    const uint32_t set = T.fan_set & 1;
    uint32_t *gs = (uint32_t *)T.gstate.p;
    sc.gcnt = gs + (size_t)set * 2 * (G + 1);
    sc.gfill = sc.gcnt + (G + 1);
    sc.z_gcnt = gs + (size_t)(set ^ 1) * 2 * (G + 1);
    sc.ctl = gs + (size_t)4 * (G + 1);
    sc.nlarge_w = sc.ctl + FC_WORDS + set;
    sc.nlarge_r = sc.ctl + FC_WORDS + (set ^ 1);
    sc.galloc = (unsigned long long *)T.galloc.p + (size_t)set * (G + 1);
    sc.z_galloc = (unsigned long long *)T.galloc.p + (size_t)(set ^ 1) * (G + 1);
    sc.med_list = (uint32_t *)T.lists.p;
    sc.large_list = sc.med_list + G + 1;
    sc.ematch = (uint32_t *)T.ematch.p;
    sc.seg = (uint32_t *)T.seg.p;
    const uint32_t ws = T.wr_set & 1;  // the set this burst's write reads
    sc.sorted = (uint32_t *)((uint8_t *)T.seg_sorted.p + ws * one[0]);
    sc.bitmaps = (uint32_t *)T.bitmaps.p + (size_t)set * (bitmap_bytes / 4);
    sc.z_bitmaps = (uint32_t *)T.bitmaps.p + (size_t)(set ^ 1) * (bitmap_bytes / 4);
    sc.pm = (uint64_t *)((uint8_t *)T.pm.p + ws * one[1]);
    sc.wcnt = (uint32_t *)((uint8_t *)T.wstate.p + ws * one[2]);
    sc.wsrc = sc.wcnt + (W + 1);
    sc.wn = sc.wsrc + (W + 1);
    sc.wlo = sc.wn + (W + 1);
    sc.wstart = (uint64_t *)((uint8_t *)T.wstart.p + ws * one[3]);
    sc.total = (uint64_t *)((uint8_t *)T.total.p + ws * one[4]);
    sc.big_t = big_t;
    sc.max_large = max_large;
    sc.bm_words = bm_words;
    sc.chunks_per_group = chunks_per_group;

    // The kernel leaves gcnt / gfill / ctl / galloc / the bitmaps it used in their initial state; they are only set from
    // the host after a table rebuild, a reallocation, a failed call, or when the geometry of the bitmaps changed.
    if (!T.scratch_clean || T.scratch_groups != G || T.scratch_large != max_large || T.scratch_bm_words != bm_words) {
        KB_CUDA(ctx, cudaMemsetAsync(T.gstate.p, 0, gstate_words * 4, ctx->stream));
        KB_CUDA(ctx, cudaMemsetAsync(T.galloc.p, 0xFF, (size_t)2 * (G + 1) * 8, ctx->stream));
        KB_CUDA(ctx, cudaMemsetAsync(T.bitmaps.p, 0, 2 * bitmap_bytes, ctx->stream));
        T.fan_gen = 0;
        T.scratch_groups = G;
        T.scratch_large = max_large;
        T.scratch_bm_words = bm_words;
    }
    T.scratch_clean = false;  // until this call has been enqueued completely
    const uint64_t ev_bytes = (uint64_t)E * (d->stride + 4);
    // Output [start (W+1) x u64][event_idx D x u32].  D is only known on the device; the buffer is sized from the
    // previous call's D (+25 %) and the write kernel refuses to run when it would not fit, so the steady state needs
    // no round trip before the write.  k_fanout's last CTA writes the offsets straight into the output buffer and into
    // the (pinned, device-visible) host copy and raises the epoch flag: the host returns on it.
    KB_TRY(hbuf_ensure(ctx, ctx->h_stage2, 64));
    if (!ctx->h_wpub) {
        KB_CUDA(ctx, cudaHostAlloc((void **)&ctx->h_wpub, 64, cudaHostAllocMapped));
        memset(ctx->h_wpub, 0, 64);
    }
    uint64_t cap = std::max<uint64_t>(T.d_hint + T.d_hint / 4 + 4096, 1 << 16);
    uint64_t D = 0;
    DBuf d_out;
    HBuf h_out;
    int rc = KB_OK;
    KB_TRY(pool_get_dev(ctx, (size_t)(W + 1) * 8 + cap * 4 + 16, &d_out));
    rc = pool_get_host(ctx, (size_t)(W + 1) * 8 + 16, &h_out);
    if (rc != KB_OK) {
        pool_put_dev(ctx, d_out);
        return rc;
    }
    if (!T.ev_fan) {
        cudaEventCreateWithFlags(&T.ev_fan, cudaEventDisableTiming);
        cudaEventCreateWithFlags(&T.ev_write[0], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&T.ev_write[1], cudaEventDisableTiming);
    }
    cudaStream_t sw = ctx->stream2;  // the write stream
    // this burst overwrites the set the write two bursts ago read
    KB_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, T.ev_write[ws], 0));
    const uint64_t wepoch = ++ctx->wpub_epoch;
    sc.o_start = (uint64_t *)d_out.p;
    sc.h_start = (uint64_t *)h_out.p;
    sc.h_pub = ctx->h_wpub;
    sc.epoch = wepoch;
    const bool run = E && W;
    if (run) {
        if (!T.fan_grid) {
            int per_sm = 0, sms = 0;
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_fanout, (int)FAN_THREADS, 0);
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
            if (per_sm < 1 || sms < 1) {
                pool_put_dev(ctx, d_out);
                pool_put_host(ctx, h_out);
                return kb_fail(ctx, KB_ECUDA, "k_fanout does not fit on an SM");
            }
            T.fan_grid = sms;  // one CTA per SM: all of them are resident together (see fan_grid_sync)
        }
        sc.gen_base = T.fan_gen;
        KB_LAUNCH(ctx, "k_fanout", ev_bytes + (uint64_t)E * NL * 12 + (uint64_t)E * 16 + (uint64_t)W * 44,
                  (k_fanout<<<(unsigned)T.fan_grid, FAN_THREADS, 0, ctx->stream>>>(ev, tb, sc)));
        T.fan_gen += 3;  // three grid barriers per launch
        T.fan_set ^= 1;  // the next call uses the other set of group state and clears this one
    } else {
        // no events or no watchers: every list is empty
        cudaMemsetAsync(sc.wstart, 0, (size_t)(W + 2) * 8, ctx->stream);
        cudaMemsetAsync(sc.total, 0, 16, ctx->stream);
        cudaMemsetAsync(d_out.p, 0, (size_t)(W + 1) * 8, ctx->stream);
        memset(h_out.p, 0, (size_t)(W + 1) * 8);
        k_publish_total<<<1, 32, 0, ctx->stream>>>(sc.total, ctx->h_wpub, wepoch);
    }
    auto launch_write = [&](uint32_t *o_idx, uint64_t capacity) {
        const unsigned wgrid = (unsigned)std::max<uint64_t>(std::min<uint64_t>((capacity + 255) / 256, 148 * 16),
                                                            std::min<uint64_t>(((uint64_t)W * 32 + 255) / 256, 148 * 16));
        KB_LAUNCH_S(ctx, sw, "k_expand_write", capacity * 8,
                    (k_expand_write<<<wgrid, 256, 0, sw>>>(W, tb.wminrev, sc.wsrc, sc.wn, sc.wlo, sc.sorted, sc.pm, sc.total,
                                                          sc.wstart, capacity, o_idx)));
    };
    cudaEventRecord(T.ev_fan, ctx->stream);
    cudaStreamWaitEvent(sw, T.ev_fan, 0);
    if (run) launch_write((uint32_t *)((uint64_t *)d_out.p + W + 1), cap);
    T.wr_set ^= 1;
    // the total (and the offsets) are published in front of the write kernel: a device-resident answer returns on the flag
    // while the delivery lists are still being written (they are valid in stream order)
    kb_seg(ctx, "host:match_launch", tseg);
    rc = wpub_wait(ctx, wepoch);
    kb_seg(ctx, "host:match_sync", tseg);
    if (rc == KB_OK && ctx->h_wpub[2]) rc = kb_fail(ctx, KB_ECUDA, "watch match: a grid barrier timed out");
    if (rc != KB_OK) {
        pool_put_dev(ctx, d_out);
        pool_put_host(ctx, h_out);
        return rc;
    }
    D = ctx->h_wpub[1];
    T.d_hint = D;
    if (ctx->prof_on && run) {  // phase spans of CTA 0 (ns -> ms), as pseudo kernels "fan:*"
        static const char *names[5] = {"fan:P1_match", "fan:P2_scatter", "fan:P3_sort", "fan:P4_watchers", "fan:last_cta_start"};
        for (int i = 0; i < 5; i++) {
            ProfEntry &pe = ctx->prof[prof_index(ctx, names[i])];
            pe.launches++;
            pe.ms += (double)ctx->h_wpub[3 + i] * 1e-6;
        }
    }
    if (D > cap) {
        // first call or a burst larger than the hint: a buffer that fits, the offsets again, and the write once more
        pool_put_dev(ctx, d_out);
        d_out = DBuf();
        cap = D;
        rc = pool_get_dev(ctx, (size_t)(W + 1) * 8 + cap * 4 + 16, &d_out);
        if (rc != KB_OK) {
            pool_put_host(ctx, h_out);
            return rc;
        }
        cudaMemcpyAsync(d_out.p, sc.wstart, (size_t)(W + 1) * 8, cudaMemcpyDeviceToDevice, sw);
        launch_write((uint32_t *)((uint64_t *)d_out.p + W + 1), cap);
    }
    cudaEventRecord(T.ev_write[ws], sw);  // the set may be overwritten (and the answer read) once this has fired
    T.scratch_clean = run;  // everything was enqueued: k_fanout restores the scratch before it ends
    if (out_mode == KB_OUT_HOST) {
        pool_put_host(ctx, h_out);
        h_out = HBuf();
        rc = pool_get_host(ctx, (size_t)(W + 1) * 8 + D * 4 + 16, &h_out);
        if (rc == KB_OK)
            cudaMemcpyAsync(h_out.p, d_out.p, (size_t)(W + 1) * 8 + D * 4, cudaMemcpyDeviceToHost, sw);
        cudaError_t e = cudaStreamSynchronize(sw);
        kb_seg(ctx, "host:match_d2h", tseg);
        if (rc == KB_OK && e != cudaSuccess) rc = kb_cuda_fail(ctx, e, "watch match");
    }
    if (rc != KB_OK) {
        T.scratch_clean = false;
        pool_put_dev(ctx, d_out);
        pool_put_host(ctx, h_out);
        return rc;
    }
    kb_result *res = kb_result_new(3, out_mode);
    if (out_mode == KB_OUT_HOST) {
        pool_put_dev(ctx, d_out);
        d_out = DBuf();
    }
    res->n_watchers = W;
    res->n_deliveries = D;
    res->h_match = h_out;
    res->d_match = d_out;
    if (out_mode == KB_OUT_DEVICE) {  // the lists are complete when the write stream gets here (kb_result_wait, kb_sync)
        if (!ctx->ev_pool.empty()) {
            res->done_ev = ctx->ev_pool.back();
            ctx->ev_pool.pop_back();
        } else if (cudaEventCreate(&res->done_ev) != cudaSuccess) {
            res->done_ev = nullptr;
        }
        if (res->done_ev) cudaEventRecord(res->done_ev, sw);
    }
    *out = res;
    return KB_OK;
}

extern "C" int kb_watch_match_dev(kb_ctx *ctx, const kb_events_dev *ev, int out_mode, kb_result **out)
{
    if (!ctx || !ev || !out || (out_mode != KB_OUT_HOST && out_mode != KB_OUT_DEVICE)) return KB_EINVAL;
    *out = nullptr;
    std::lock_guard<std::mutex> g(ctx->mu);
    cudaSetDevice(ctx->device);
    return match_locked(ctx, ev, out_mode, out);
}

extern "C" int kb_watch_match(kb_ctx *ctx, const kb_events *ev, int out_mode, kb_result **out)
{
    if (!ctx || !ev || !out || (out_mode != KB_OUT_HOST && out_mode != KB_OUT_DEVICE)) return KB_EINVAL;
    if (ev->n && (!ev->keys || !ev->key_off || !ev->rev)) return KB_EINVAL;
    *out = nullptr;
    std::lock_guard<std::mutex> g(ctx->mu);
    cudaSetDevice(ctx->device);
    if (!ctx->ev_scratch) ctx->ev_scratch = new kb_events_dev();
    KB_TRY(events_upload_locked(ctx, ev, ctx->ev_scratch));
    return match_locked(ctx, ctx->ev_scratch, out_mode, out);
}

extern "C" int kb_match_view_get(const kb_result *res, kb_match_view *v)
{
    if (!res || !v || res->type != 3) return KB_EINVAL;
    memset(v, 0, sizeof(*v));
    v->n_watchers = res->n_watchers;
    v->n_deliveries = res->n_deliveries;
    v->on_device = res->out_mode == KB_OUT_DEVICE;
    v->start = (const uint64_t *)res->h_match.p;  // offsets are always host readable
    if (v->on_device)
        v->event_idx = (const uint32_t *)((const uint64_t *)res->d_match.p + res->n_watchers + 1);
    else
        v->event_idx = (const uint32_t *)((const uint64_t *)res->h_match.p + res->n_watchers + 1);
    return KB_OK;
}
