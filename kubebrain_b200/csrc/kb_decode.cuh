// kb_decode.cuh -- the decoded columns of the record directory and the per-request meta word (included by kb_core.cu
// and kb_scan.cu).
//
// Almost everything coder.Decode (pkg/backend/coder/normal.go:58-70) and the per-record front half of worker.run
// (pkg/backend/scanner/scanner.go:430-453, 471-491, 566-591) compute about a record is a property of the snapshot, not of
// the request.  It is computed once, when the directory is written, and kept per record in directory order:
//   crev  u64  the key's revision when it is non-zero; for a revision record (revision 0) with a value of >= 8 bytes the
//              BE64 revision in the value's first 8 bytes; 0 otherwise
//   cword u32  bits 0..15  LCP with the preceding record's key (KB_LCP_INF for record 0)
//              bits 16..21 static flags: KB_M_DEC_OK, KB_M_REV0, KB_C_TOMBV, KB_C_VL9, KB_C_VL8, KB_C_EVENTS
// kb_load_sorted / kb_restore build both columns (k_col_build, which also checks the key order), k_dir_merge carries them
// through a write batch and k_col_fix recomputes the O(ops) entries the batch touched, the layout compaction copies them.
// A scan turns a record's entry into its meta word (col_meta): only the comparisons against the read revision, the
// compact revision and timeout_rev are left, so the scan reads 12 bytes per record instead of the record's key.
#pragma once

#include "kb_internal.cuh"

namespace {

constexpr uint32_t MAGIC_LE = 0x8b80fb57u;  // bytes 57 fb 80 8b (coder/normal.go:26)

// bytes.Contains(rawKey, "/events/") for the user key = key bytes [4, len - 9): one 16-byte load per chunk, the bytes
// shifted through a 64-bit window in registers
__device__ __forceinline__ bool key_has_events(const uint4 *kp, uint32_t len)
{
    const uint32_t end = len - 9;
    uint64_t w = 0;
    for (uint32_t c = 0; c * 16 < end; c++) {
        const uint4 x = kp[c];
#pragma unroll
        for (int b = 0; b < 16; b++) {
            const uint32_t p = c * 16 + b;
            if (p >= 4 && p < end) {
                w = (w << 8) | byte_of(x, b);
                if (p >= 11 && w == 0x2f6576656e74732full) return true;
            }
        }
    }
    return false;
}

// Column entry of record i of `st`, against record i - 1 (none for i == 0).  *less: record i - 1 sorts strictly before
// record i (bytes.Compare order; always true for i == 0).
__device__ __forceinline__ void col_entry(const StoreDev &st, uint32_t i, uint64_t *crev, uint32_t *cword, bool *less)
{
    const uint4 *kp = st.kslab + st.koff16[i];
    const uint32_t len = st.klen[i];
    uint32_t lcp = KB_LCP_INF;
    bool lt = true;
    if (i > 0) {
        const uint4 *pp = st.kslab + st.koff16[i - 1];
        const uint32_t plen = st.klen[i - 1];
        const uint32_t m = min(len, plen), nch = (m + 15) >> 4;
        lcp = m;
        lt = plen < len;  // all common bytes equal: the shorter key first; equal lengths: a duplicate
        // four chunk pairs per step, loaded together (the loads stay inside both keys: the index is clamped)
        bool found = false;
        for (uint32_t c0 = 0; c0 < nch && !found; c0 += 4) {
            uint4 x[4], y[4];
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const uint32_t c = min(c0 + j, nch - 1);
                x[j] = pp[c];
                y[j] = kp[c];
            }
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int p = first_diff16(x[j], y[j]);
                if (!found && c0 + j < nch && p < 16 && (c0 + j) * 16 + p < m) {
                    lcp = (c0 + j) * 16 + p;
                    lt = byte_of(x[j], p) < byte_of(y[j], p);
                    found = true;
                }
            }
        }
    }
    const uint8_t *kb = (const uint8_t *)kp;
    uint32_t flags = 0;
    uint64_t r = 0;
    // coder.Decode; keys shorter than 13 bytes are undecodable (Go would panic)
    if (len >= 13 && ((const uint32_t *)kp)[0] == MAGIC_LE && kb[len - 9] == 0x24) {
        const uint64_t rev = be64_bytes(kb + len - 8);
        const uint32_t vl = st.vlen[i];
        uint4 v = make_uint4(0, 0, 0, 0);
        if (vl >= 8) v = st.vslab[st.voff16[i]];
        flags |= KB_M_DEC_OK;
        r = rev;
        if (rev == 0) {
            flags |= KB_M_REV0;
            if (vl >= 8)  // BE64 of the value's first 8 bytes: the revision a deleted-flag revision record holds
                r = ((uint64_t)__byte_perm(v.x, 0, 0x0123) << 32) | __byte_perm(v.y, 0, 0x0123);
        }
        if (vl == 9) flags |= KB_C_VL9;
        if (vl >= 8) flags |= KB_C_VL8;
        if (vl == 9 && v.x == 0x626d6f74u && v.y == 0x6e6f7473u && (v.z & 0xffu) == 0x65u)
            flags |= KB_C_TOMBV;  // "tombstone" util.go:28
        if (key_has_events(kp, len)) flags |= KB_C_EVENTS;
    }
    *crev = r;
    *cword = lcp | flags;
    *less = lt;
}

// The meta word of one record for one request: LCP (KB_LCP_INF for the request's first record, which has no predecessor
// inside the request) + the decode / visibility / tombstone / compaction-class flags (KB_M_*).
__device__ __forceinline__ uint32_t col_meta(uint64_t crev, uint32_t cword, const ScanMode &mode, uint64_t read_rev,
                                             bool first)
{
    uint32_t w = first ? KB_LCP_INF : (cword & KB_M_LCP_MASK);
    if (!(cword & KB_M_DEC_OK)) return w;
    w |= cword & (KB_M_DEC_OK | KB_M_REV0);
    const bool rev0 = (cword & KB_M_REV0) != 0;
    bool expired = false;
    if (mode.ttl_scan && (cword & KB_C_EVENTS)) {  // compactIfExpired scanner.go:566-591
        if (rev0) {
            if ((cword & KB_C_VL8) && crev <= mode.timeout_rev) {
                expired = true;
                w |= KB_M_TTLREV;
            }
        } else if (crev <= mode.timeout_rev) {
            expired = true;
            w |= KB_M_TTLOBJ;
        }
    }
    if (!expired && (rev0 || crev <= read_rev)) {  // scanner.go:451-453
        w |= KB_M_TRIG;
        if (cword & KB_C_TOMBV) w |= KB_M_TOMB;
        bool prevok = true;
        if (mode.compact && rev0 && (cword & KB_C_VL9)) {  // scanner.go:476-491
            if (crev > read_rev)
                prevok = false;  // `continue` without updating prev (Q5)
            else
                w |= KB_M_REVDEL;
        }
        if (prevok) w |= KB_M_PREVOK;
    }
    return w;
}

}  // namespace
