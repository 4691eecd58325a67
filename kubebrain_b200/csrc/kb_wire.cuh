// kb_wire.cuh -- the scan answer as etcd protobuf elements, written by the device (included by kb_scan.cu).
//
// Replaces the per-kv materialisation of the etcd-compatible server: kvToEtcdKv (pkg/server/etcd/backendshim.go:427-436)
// + the gogo-protobuf Marshal of etcdserverpb.RangeResponse.kvs (List, backendshim.go:269-282) or of
// etcdserverpb.WatchResponse.events (range stream, backendshim.go:349-363; batches cut by receiver.go:119-138).
// A protobuf message is the concatenation of its fields, so the device writes the repeated-field ELEMENTS back to
// back (one per emitted kv, reference order) and the host only prepends / appends the few header and trailer bytes
// (kb_wire_range_head / _tail / kb_wire_watch_head): nothing is re-materialised per kv on the CPU.
//
//   KVS    element:  12 <len(kv)>  kv                       kv = [0a <ul> user key] [18 <rev>] [2a <vl> value]
//   EVENTS element:  5a <len(ev)>  ev,  ev = 12 <len(kv)> kv      (proto3: empty key / value and rev 0 are omitted)
//
// Field numbers: go.etcd.io/etcd/api/v3 v3.5.2 (reference go.mod:28), pinned by tests/test_wire.py.
#pragma once

#include "kb_internal.cuh"

namespace {

__device__ __forceinline__ uint32_t varint_len(uint64_t v) { return v ? (uint32_t)(70 - __clzll((long long)v)) / 7u : 1u; }

struct WireSizes {
    uint32_t ul, vl;
    uint64_t rev;
    uint64_t body, kv, elem;  // mvccpb.KeyValue body, kv field (tag + len + body), whole element
};

__device__ __forceinline__ WireSizes wire_sizes(uint32_t ul, uint32_t vl, uint64_t rev, int wire)
{
    WireSizes s;
    s.ul = ul;
    s.vl = vl;
    s.rev = rev;
    s.body = (ul ? 1 + varint_len(ul) + (uint64_t)ul : 0) + (rev ? 1 + varint_len(rev) : 0) +
             (vl ? 1 + varint_len(vl) + (uint64_t)vl : 0);
    s.kv = 1 + varint_len(s.body) + s.body;
    s.elem = wire == KB_WIRE_KVS_I ? s.kv : 1 + varint_len(s.kv) + s.kv;
    return s;
}

// response bytes of one emitted record: padded [key][value] in the arena modes, element bytes in the wire modes
__device__ __forceinline__ uint64_t kv_resp_bytes(const StoreDev &st, uint32_t rec, int wire)
{
    const uint32_t kl = st.klen[rec], vl = st.vlen[rec];
    if (!wire) return (uint64_t)pad16(kl) + pad16(vl);
    const uint64_t rev = be64_bytes((const uint8_t *)(st.kslab + st.koff16[rec]) + kl - 8);
    return wire_sizes(kl - 13, vl, rev, wire).elem;
}

struct __align__(16) WireJob {  // 96 bytes: six 16-byte loads, the same for every lane of the warp that copies it
    uint4 loc;     // {dst lo, dst hi, vsrc16 lo, vsrc16 hi}: first arena byte of the element, value slab chunk
    uint4 len;     // {ksrc16, ul, vl, n1 | n2 << 8}: key slab chunk (magic | user key | '$' | rev), lengths
    uint4 h1[2];   // bytes in front of the user key: [5a len] 12 len [0a len]   (n1 of them)
    uint4 h2[2];   // bytes between user key and value: [18 rev] [2a len]        (n2 of them)
};

struct WireOut {
    uint32_t *rec_idx;
    uint64_t *rev;
    uint64_t *key_off;
    uint32_t *key_len;
    uint64_t *val_off;
    uint32_t *val_len;
    uint64_t *elem_off;  // n_kvs + 1
};

__device__ __forceinline__ uint32_t put_varint(uint8_t *p, uint64_t v)
{
    uint32_t n = 0;
    while (v >= 0x80) {
        p[n++] = (uint8_t)(v | 0x80);
        v >>= 7;
    }
    p[n++] = (uint8_t)v;
    return n;
}

// the bytes in front of the user key and between the user key and the value
__device__ __forceinline__ void wire_headers(const WireSizes &s, int wire, uint8_t *h1, uint32_t &n1, uint8_t *h2,
                                             uint32_t &n2)
{
    n1 = 0;
    if (wire == KB_WIRE_EVENTS_I) {
        h1[n1++] = 0x5a;
        n1 += put_varint(h1 + n1, s.kv);
    }
    h1[n1++] = 0x12;
    n1 += put_varint(h1 + n1, s.body);
    if (s.ul) {
        h1[n1++] = 0x0a;
        n1 += put_varint(h1 + n1, s.ul);
    }
    n2 = 0;
    if (s.rev) {
        h2[n2++] = 0x18;
        n2 += put_varint(h2 + n2, s.rev);
    }
    if (s.vl) {
        h2[n2++] = 0x2a;
        n2 += put_varint(h2 + n2, s.vl);
    }
}

// thread per emitted kv: where its element goes and what the per-kv view arrays say
__global__ void __launch_bounds__(256)
k_wire_jobs(StoreDev st, const ReqDev *__restrict__ reqs, uint32_t nreq, const uint64_t *__restrict__ job_first,
            const uint64_t *__restrict__ arena_base, const uint32_t *__restrict__ sel,
            const uint64_t *__restrict__ slot, int wire, WireJob *__restrict__ jobs, WireOut out)
{
    const uint64_t n_kvs = job_first[nreq];
    if (n_kvs == 0 && blockIdx.x == 0 && threadIdx.x == 0) out.elem_off[0] = 0;
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n_kvs;
         k += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t lo = 0, hi = nreq;  // request of kv k: last q with job_first[q] <= k
        while (hi - lo > 1) {
            const uint32_t mid = (lo + hi) >> 1;
            if (job_first[mid] <= k) lo = mid; else hi = mid;
        }
        const uint32_t q = lo;
        const uint64_t s = reqs[q].sel_base + (k - job_first[q]);
        const uint32_t rec = sel[s];
        const uint64_t E = arena_base[q] + slot[s];
        const uint32_t kl = st.klen[rec], vl = st.vlen[rec];
        const uint32_t ksrc16 = st.koff16[rec];
        const uint64_t rev = st.crev[rec];  // an emitted record has a non-zero key revision: the column holds it
        const WireSizes ws = wire_sizes(kl - 13, vl, rev, wire);
        __align__(16) uint8_t h1[32], h2[32];
        uint32_t n1, n2;
#pragma unroll
        for (int b = 0; b < 32; b++) h1[b] = h2[b] = 0;
        wire_headers(ws, wire, h1, n1, h2, n2);
        const uint64_t vsrc16 = st.voff16[rec];
        WireJob j;
        j.loc = make_uint4((uint32_t)E, (uint32_t)(E >> 32), (uint32_t)vsrc16, (uint32_t)(vsrc16 >> 32));
        j.len = make_uint4(ksrc16, ws.ul, vl, n1 | (n2 << 8));
        j.h1[0] = ((const uint4 *)h1)[0];
        j.h1[1] = ((const uint4 *)h1)[1];
        j.h2[0] = ((const uint4 *)h2)[0];
        j.h2[1] = ((const uint4 *)h2)[1];
        jobs[k] = j;
        out.rec_idx[k] = rec;
        out.rev[k] = rev;
        out.key_off[k] = E + n1;
        out.key_len[k] = ws.ul;
        out.val_off[k] = E + n1 + ws.ul + n2;
        out.val_len[k] = vl;
        out.elem_off[k] = E;
        if (k == n_kvs - 1) out.elem_off[n_kvs] = E + ws.elem;
    }
}

// bytes [lo, hi) of a 16-byte chunk as a mask (0xff per selected byte); lo/hi are clamped to [0,16]
__device__ __forceinline__ uint4 byte_mask16(int lo, int hi)
{
    lo = max(lo, 0);
    hi = min(hi, 16);
    uint32_t w[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int a = max(lo - 4 * k, 0), b = min(hi - 4 * k, 4);  // byte range inside word k
        uint32_t m = 0;
        if (b > a) {
            const uint32_t upto_b = b >= 4 ? 0xffffffffu : ((1u << (8 * b)) - 1u);
            const uint32_t upto_a = a >= 4 ? 0xffffffffu : ((1u << (8 * a)) - 1u);
            m = upto_b & ~upto_a;
        }
        w[k] = m;
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}

// 16 bytes starting `s` bytes (0..15) into the 32-byte pair (lo, hi)
__device__ __forceinline__ uint4 funnel16(const uint4 &lo, const uint4 &hi, uint32_t s)
{
    const uint32_t w[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
    const uint32_t ws = s >> 2, bs = (s & 3) * 8;
    uint32_t o[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        uint32_t a = 0, b = 0;
#pragma unroll
        for (int t = 0; t < 4; t++) {  // ws is 0..3: select without dynamic register indexing
            if (ws == (uint32_t)t) {
                a = w[t + k];
                b = w[t + k + 1 < 8 ? t + k + 1 : 7];
            }
        }
        o[k] = __funnelshift_r(a, b, bs);
    }
    return make_uint4(o[0], o[1], o[2], o[3]);
}

// the part of the element's chunk [e0, e0+16) that comes from a global-memory segment: segment bytes
// [begin, begin+len) of the element are bytes [skip, skip+len) behind the 16-byte aligned pointer `base`
template <bool SMEM>
__device__ __forceinline__ uint4 wire_ld(const uint4 *p)
{
    return SMEM ? *p : __ldg(p);  // staged copy in shared memory, or the slab itself
}

template <bool SMEM, typename I>
__device__ __forceinline__ void seg_mem(uint4 &acc, I e0, I begin, uint32_t len, const uint4 *base, uint32_t skip)
{
    const I lo = begin - e0, hi = begin + (I)len - e0;  // segment range in chunk coordinates
    if (hi <= 0 || lo >= 16 || len == 0) return;
    const I t = (I)skip + (e0 - begin);  // source byte of chunk byte 0 (may be negative)
    const I ci = t >> 4;                          // floor
    const uint32_t s = (uint32_t)(t & 15);
    const I last = ((I)skip + len - 1) >> 4;  // last chunk holding segment bytes
    uint4 a = make_uint4(0, 0, 0, 0), b = a;
    if (ci >= 0 && ci <= last) a = wire_ld<SMEM>(base + ci);
    if (s != 0 && ci + 1 >= 0 && ci + 1 <= last) b = wire_ld<SMEM>(base + ci + 1);
    const uint4 v = funnel16(a, b, s);
    const uint4 m = byte_mask16((int)max(lo, (I)0), (int)min(hi, (I)16));
    acc.x |= v.x & m.x;
    acc.y |= v.y & m.y;
    acc.z |= v.z & m.z;
    acc.w |= v.w & m.w;
}

// ... and the part that comes from a short header (at most 32 bytes, held in two registers quads): chunk byte j is
// header byte j - lo, i.e. the 16 bytes at offset 16 - lo of the 64-byte string [16 zero bytes | h_lo | h_hi | 16 zero]
template <typename I>
__device__ __forceinline__ void seg_reg(uint4 &acc, I e0, I begin, uint32_t len, const uint4 &h_lo, const uint4 &h_hi)
{
    const I lo = begin - e0, hi = lo + (I)len;
    if (hi <= 0 || lo >= 16 || len == 0) return;
    const int o = 16 - (int)lo;  // 1 .. 47
    const uint4 z = make_uint4(0, 0, 0, 0);
    const int q = o >> 4;
    const uint4 a = q == 0 ? z : q == 1 ? h_lo : h_hi;
    const uint4 b = q == 0 ? h_lo : q == 1 ? h_hi : z;
    const uint4 v = funnel16(a, b, (uint32_t)(o & 15));
    const uint4 m = byte_mask16((int)max(lo, (I)0), (int)min(hi, (I)16));
    acc.x |= v.x & m.x;
    acc.y |= v.y & m.y;
    acc.z |= v.z & m.z;
    acc.w |= v.w & m.w;
}

constexpr int WIRE_WARPS = 8;

// 16 bytes starting 4*WS + bs/8 bytes into the pair (a, b): the word offset is a compile-time constant, the bit shift
// inside a word (bs = 0, 8, 16, 24) is a run-time operand of the funnel shift
template <int WS>
__device__ __forceinline__ uint4 funnel16_w(const uint4 &a, const uint4 &b, uint32_t bs)
{
    const uint32_t w0 = WS == 0 ? a.x : WS == 1 ? a.y : WS == 2 ? a.z : a.w;
    const uint32_t w1 = WS == 0 ? a.y : WS == 1 ? a.z : WS == 2 ? a.w : b.x;
    const uint32_t w2 = WS == 0 ? a.z : WS == 1 ? a.w : WS == 2 ? b.x : b.y;
    const uint32_t w3 = WS == 0 ? a.w : WS == 1 ? b.x : WS == 2 ? b.y : b.z;
    const uint32_t w4 = WS == 0 ? b.x : WS == 1 ? b.y : WS == 2 ? b.z : b.w;
    return make_uint4(__funnelshift_r(w0, w1, bs), __funnelshift_r(w1, w2, bs), __funnelshift_r(w2, w3, bs),
                      __funnelshift_r(w3, w4, bs));
}

// Interior chunks [c_lo, c_hi) of a destination that lie entirely inside one source segment: chunk c holds source
// bytes [t0 + 16 (c - c_lo), +16) behind `base`, so the byte shift is the same for all of them.  Per chunk: two
// 16-byte loads (the second is the neighbour lane's first), four funnel shifts, one 16-byte store; two chunks per
// lane and step.
template <bool SMEM, int WS, typename I>
__device__ __forceinline__ void copy_interior_w(uint4 *__restrict__ dst0, I c_lo, I c_hi,
                                                const uint4 *src, uint32_t bs, uint32_t lane)
{
    const I n = c_hi - c_lo;
    uint4 *d = dst0 + c_lo;
    for (I i = lane; i < n; i += 64) {
        const bool two = i + 32 < n;
        const uint4 a0 = wire_ld<SMEM>(src + i), b0 = wire_ld<SMEM>(src + i + 1);
        const uint4 a1 = two ? wire_ld<SMEM>(src + i + 32) : a0, b1 = two ? wire_ld<SMEM>(src + i + 33) : b0;
        stg_stream(d + i, funnel16_w<WS>(a0, b0, bs));
        if (two) stg_stream(d + i + 32, funnel16_w<WS>(a1, b1, bs));
    }
}

template <bool SMEM, typename I>
__device__ __forceinline__ void copy_interior(uint4 *__restrict__ dst0, I c_lo, I c_hi, const uint4 *base, I t0,
                                              uint32_t lane)
{
    if (c_hi <= c_lo) return;
    const uint4 *src = base + (t0 >> 4);
    const uint32_t s = (uint32_t)(t0 & 15), bs = (s & 3) * 8;
    switch (s >> 2) {  // warp-uniform
        case 0: copy_interior_w<SMEM, 0, I>(dst0, c_lo, c_hi, src, bs, lane); break;
        case 1: copy_interior_w<SMEM, 1, I>(dst0, c_lo, c_hi, src, bs, lane); break;
        case 2: copy_interior_w<SMEM, 2, I>(dst0, c_lo, c_hi, src, bs, lane); break;
        default: copy_interior_w<SMEM, 3, I>(dst0, c_lo, c_hi, src, bs, lane); break;
    }
}

// One element, by one warp.  The destination is produced in aligned 16-byte chunks.  Chunks that lie entirely inside
// the user key or inside the value (all but a handful) take the uniform-shift fast path; the few boundary chunks
// (headers, segment seams, the element's first and last chunk, which it shares with its neighbours) are assembled
// from the four segments [header | user key | rev + value header | value] and fall back to byte stores where they
// are partial.  ksrc points at the internal key (user key at +4), vsrc at the value; both 16-byte aligned.
template <bool SMEM, typename I>
__device__ __forceinline__ void wire_emit_element(const uint4 &loc, const uint4 &len, const uint4 &h1a, const uint4 &h1b,
                                                  const uint4 &h2a, const uint4 &h2b, const uint4 *ksrc,
                                                  const uint4 *vsrc, uint8_t *__restrict__ arena, uint32_t lane)
{
    const uint64_t dst = ((uint64_t)loc.y << 32) | loc.x;
    const uint32_t ul = len.y, vl = len.z, n1 = len.w & 0xffu, n2 = (len.w >> 8) & 0xffu;
    const I total = (I)n1 + ul + n2 + vl;
    const I lead = (I)(dst & 15);
    uint4 *dst0 = (uint4 *)(arena + (dst - lead));
    const I nchunks = (lead + total + 15) >> 4;
    const I b_key = n1, b_h2 = b_key + ul, b_val = b_h2 + n2;
    // interior chunk ranges of the two source segments (chunk c covers element bytes [16 c - lead, +16))
    const I ck_lo = (b_key + lead + 15) >> 4;
    const I ck_hi = max(ck_lo, (b_key + (I)ul + lead) >> 4);
    const I cv_lo = max(ck_hi, (b_val + lead + 15) >> 4);
    const I cv_hi = max(cv_lo, (b_val + (I)vl + lead) >> 4);
    copy_interior<SMEM, I>(dst0, ck_lo, ck_hi, ksrc, 4 + (ck_lo * 16 - lead - b_key), lane);
    copy_interior<SMEM, I>(dst0, cv_lo, cv_hi, vsrc, cv_lo * 16 - lead - b_val, lane);
    // boundary chunks: [0, ck_lo) u [ck_hi, cv_lo) u [cv_hi, nchunks)
    const I nb0 = ck_lo, nb1 = cv_lo - ck_hi, nb2 = nchunks - cv_hi;
    for (I i = lane; i < nb0 + nb1 + nb2; i += 32) {
        const I c = i < nb0 ? i : i < nb0 + nb1 ? ck_hi + (i - nb0) : cv_hi + (i - nb0 - nb1);
        const I e0 = c * 16 - lead;
        uint4 acc = make_uint4(0, 0, 0, 0);
        seg_reg<I>(acc, e0, 0, n1, h1a, h1b);
        seg_mem<SMEM, I>(acc, e0, b_key, ul, ksrc, 4);
        seg_reg<I>(acc, e0, b_h2, n2, h2a, h2b);
        seg_mem<SMEM, I>(acc, e0, b_val, vl, vsrc, 0);
        if (e0 >= 0 && e0 + 16 <= total) {
            stg_stream(dst0 + c, acc);
        } else {
            uint8_t *d = (uint8_t *)(dst0 + c);
#pragma unroll
            for (int b = 0; b < 16; b++)
                if (e0 + b >= 0 && e0 + b < total) d[b] = (uint8_t)byte_of(acc, b);
        }
    }
}

__device__ __forceinline__ uint32_t wsmem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void wmbar_wait(uint64_t *bar, uint32_t parity, unsigned int *err_flag)
{
    dmbar_wait(bar, parity, err_flag);  // bounded: see kb_internal.cuh
}

constexpr int WIRE_MAX_STAGES = 8;
constexpr uint32_t WIRE_JOB_CHUNKS = sizeof(WireJob) / 16;  // 6
constexpr uint32_t WIRE_WARP_CHUNKS = 880;                  // shared memory per warp: two CTAs of 8 warps per SM

// k_wire_copy: warp per element, sources staged by the copy engine.  Lane 0 runs `stages - 1` elements ahead and
// issues, per element, three bulk (TMA) copies into the warp's ring slot -- the 96-byte job, the internal key, the
// value -- completing on the slot's mbarrier; the whole warp then assembles the element from shared memory
// (wire_emit_element<true>) and writes it with 16-byte stores.  The loads in flight are therefore independent of the
// registers, exactly as in k_gather; only the unaligned destination forces the bytes through the lanes.  An element
// too large for a slot is copied straight from the slab (wire_emit_element<false>).
__global__ void __launch_bounds__(WIRE_WARPS * 32, 2)
k_wire_copy(StoreDev st, const WireJob *__restrict__ jobs, const uint64_t *__restrict__ n_kvs_dev,
            uint8_t *__restrict__ arena, uint32_t slot_chunks, uint32_t stages, unsigned int *__restrict__ err_flag)
{
    extern __shared__ __align__(128) uint4 wbuf[];  // WIRE_WARPS x stages x slot_chunks
    __shared__ uint64_t wbars[WIRE_WARPS * WIRE_MAX_STAGES];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint4 *ring = wbuf + (size_t)warp * stages * slot_chunks;
    uint64_t *bar = wbars + warp * WIRE_MAX_STAGES;
    if (lane == 0) {
        for (uint32_t s = 0; s < stages; s++)
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(wsmem_u32(bar + s)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    const uint64_t n_kvs = *n_kvs_dev;
    const uint64_t kstride = (uint64_t)gridDim.x * WIRE_WARPS;
    const uint64_t k0 = (uint64_t)blockIdx.x * WIRE_WARPS + warp;
    const uint32_t room = slot_chunks - WIRE_JOB_CHUNKS - 1;  // chunks of key + value a slot can stage

    // lane 0: issue the copies of element k into ring slot `slot`
    auto issue = [&](uint64_t k, uint32_t slot) {
        const uint4 *jp = (const uint4 *)(jobs + k);
        const uint4 loc = __ldg(jp), len = __ldg(jp + 1);
        const uint32_t nkc = (4 + len.y + 15) >> 4, nvc = (len.z + 15) >> 4;
        const bool fits = nkc + nvc <= room;
        uint4 *sl = ring + (size_t)slot * slot_chunks;
        const uint32_t b = wsmem_u32(bar + slot);
        // the slot was last read (generic proxy) by the warp before the __syncwarp that precedes this call
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(b),
                     "r"((WIRE_JOB_CHUNKS + (fits ? nkc + nvc : 0)) * 16)
                     : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                         wsmem_u32(sl)),
                     "l"(jp), "r"(WIRE_JOB_CHUNKS * 16), "r"(b)
                     : "memory");
        if (fits) {
            const uint64_t vsrc16 = ((uint64_t)loc.w << 32) | loc.z;
            if (nkc)
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                                 wsmem_u32(sl + WIRE_JOB_CHUNKS)),
                             "l"(st.kslab + len.x), "r"(nkc * 16), "r"(b)
                             : "memory");
            if (nvc)
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                                 wsmem_u32(sl + WIRE_JOB_CHUNKS + nkc)),
                             "l"(st.vslab + vsrc16), "r"(nvc * 16), "r"(b)
                             : "memory");
        }
    };

    uint64_t k_issue = k0, k_proc = k0;
    uint32_t s_issue = 0, s_proc = 0, ph = 0;
    // prologue: fill all but one slot
    for (uint32_t i = 0; i + 1 < stages && k_issue < n_kvs; i++, k_issue += kstride) {
        if (lane == 0) issue(k_issue, s_issue);
        if (++s_issue == stages) s_issue = 0;
    }
    for (; k_proc < n_kvs; k_proc += kstride) {
        if (k_issue < n_kvs) {  // the slot freed by the previous step (a __syncwarp ended that step)
            if (lane == 0) issue(k_issue, s_issue);
            if (++s_issue == stages) s_issue = 0;
            k_issue += kstride;
        }
        wmbar_wait(bar + s_proc, ph, err_flag);
        const uint4 *sl = ring + (size_t)s_proc * slot_chunks;
        const uint4 loc = sl[0], len = sl[1], h1a = sl[2], h1b = sl[3], h2a = sl[4], h2b = sl[5];
        const uint32_t nkc = (4 + len.y + 15) >> 4, nvc = (len.z + 15) >> 4;
        if (nkc + nvc <= room) {
            wire_emit_element<true, int>(loc, len, h1a, h1b, h2a, h2b, sl + WIRE_JOB_CHUNKS, sl + WIRE_JOB_CHUNKS + nkc, arena,
                                    lane);
        } else {
            const uint64_t vsrc16 = ((uint64_t)loc.w << 32) | loc.z;
            wire_emit_element<false, long long>(loc, len, h1a, h1b, h2a, h2b, st.kslab + len.x, st.vslab + vsrc16, arena, lane);
        }
        __syncwarp();  // every lane is done reading the slot before lane 0 refills it
        if (++s_proc == stages) {
            s_proc = 0;
            ph ^= 1;
        }
    }
}

// ring geometry of k_wire_copy for a store whose largest padded [key][value] pair is `max_kv_chunks`
static inline void wire_geometry(uint32_t max_kv_chunks, uint32_t *slot_chunks, uint32_t *stages)
{
    const uint32_t room = max_kv_chunks < 32 ? 32 : max_kv_chunks > 160 ? 160 : max_kv_chunks;
    const uint32_t slot = WIRE_JOB_CHUNKS + room + 1;  // job | key + value | one chunk of slack for the shifted reads
    uint32_t s = WIRE_WARP_CHUNKS / slot;
    s = s < 3 ? 3 : s > (uint32_t)WIRE_MAX_STAGES ? (uint32_t)WIRE_MAX_STAGES : s;
    *slot_chunks = slot;
    *stages = s;
}

}  // namespace
