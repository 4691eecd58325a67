/*
 * kb_b200.h -- C ABI of libkbb200.so: the B200-native MVCC range-scan / compaction-sweep /
 * watch fan-out engine that drops in behind KubeBrain's Go plugin surfaces.
 *
 * The reference (kubewharf/kubebrain) is 100 % Go and has NO native boundary today; the entry points
 * below are what a cgo shim for this path binds (INTEGRATION.md shows the binding).  Each symbol cites
 * the reference interface (file:line in the reference tree) whose hot loop it replaces.
 *
 * Conventions: every function returns 0 (KB_OK) or a negative kb_status; no exception crosses the
 * boundary; all pointers are plain host pointers unless a field says "device"; inputs are caller-owned
 * and may be released when the call returns; results are library-owned handles (kb_result) that stay
 * valid until kb_result_free (this is what lets the Go side keep slices alive after Iter.Close, as
 * worker.run requires -- pkg/backend/scanner/scanner.go:493-495).  A kb_ctx serialises its own calls
 * (one CUDA stream); use one ctx per goroutine-pool shard or guard it with a mutex.
 * There is NO CPU fallback: without a CUDA device kb_open fails with KB_ECUDA.
 */
#ifndef KB_B200_H
#define KB_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KB_ABI_VERSION 2  /* 2: kb_write_op.expire_unix, kb_expire, kb_range_prefetch, kb_range_submit / _collect, kb_cursor_transport / _force_nccl */

typedef enum kb_status {
    KB_OK = 0,
    KB_EINVAL = -1,      /* bad argument                                                         */
    KB_ECUDA = -2,       /* CUDA runtime / driver failure (kb_last_error has the text)            */
    KB_ENOMEM = -3,
    KB_EUNSORTED = -4,   /* kb_load_sorted: keys not strictly ascending (storage.Iter contract)   */
    KB_ECOMPACTED = -5,  /* range revision below the compact revision (scanner.go:618-624)        */
    KB_ESTATE = -6,      /* call out of order (no store loaded, NCCL not initialised, ...)         */
    KB_ENCCL = -7,
    KB_ELIMIT = -8,      /* input exceeds a documented format limit (key > 65535 B, n >= 2^32-1)   */
    KB_EIO = -9          /* kb_dump / kb_restore: file could not be opened, read or written        */
} kb_status;

typedef struct kb_ctx kb_ctx;
typedef struct kb_result kb_result;
typedef struct kb_events_dev kb_events_dev;

typedef struct kb_config {
    uint32_t struct_size;   /* sizeof(kb_config), for forward compatibility */
    uint32_t flags;         /* KB_CFG_* */
} kb_config;
/* the ctx's stream gets the highest CUDA stream priority: its kernels are scheduled ahead of those of other contexts
 * sharing the GPU (e.g. the latency-critical scan context next to a fan-out context) */
#define KB_CFG_HIGH_PRIORITY 1u

/* ---- lifecycle ------------------------------------------------------------------------------ */
int kb_abi_version(void);
int kb_open(int device_ordinal, const kb_config *cfg, kb_ctx **out);
void kb_close(kb_ctx *ctx);
const char *kb_last_error(kb_ctx *ctx);
/* the main cudaStream_t of this ctx (callers may record events on it).  Device-resident answers are completed on other
 * streams of the context: order consumers with kb_result_wait, not with this stream. */
void *kb_stream(kb_ctx *ctx);
int kb_sync(kb_ctx *ctx);

/* ---- store: replaces storage.Iter over badger (pkg/storage/badger/iter.go:27-98) --------------
 * Bulk-loads a snapshot of the engine: n unique internal keys in ascending bytes.Compare order with
 * their values, packed back to back (record i = keys[key_off[i]..key_off[i+1])).  The snapshot becomes
 * an HBM-resident slab (16-byte aligned records) that every scan below reads.  */
int kb_load_sorted(kb_ctx *ctx, const uint8_t *keys, const uint64_t *key_off, const uint8_t *vals,
                   const uint64_t *val_off, uint64_t n);
int kb_store_info(kb_ctx *ctx, uint64_t *n_records, uint64_t *key_bytes, uint64_t *val_bytes);

/* Durable dump / restore of the HBM snapshot (restart without re-iterating the engine; the on-disk format of the
 * engine itself -- badger / TiKV, pkg/storage/badger/badger.go:33-39 -- is untouched).  The file holds the record
 * directory and both slabs in device layout plus the compact-revision record, each section with an FNV-1a 64 checksum;
 * kb_restore validates header, sizes, checksums and the iterator contract (ascending unique keys) before the snapshot
 * becomes visible.  KB_EIO on file errors, KB_EINVAL on a corrupt or foreign file. */
int kb_dump(kb_ctx *ctx, const char *path);
int kb_restore(kb_ctx *ctx, const char *path);

/* Incremental maintenance from the write path: one committed storage.BatchWrite (pkg/storage/interface.go:81-106;
 * the backend issues CAS(revision record) + Put(object record) per write, pkg/backend/txn.go:249-265,
 * creator/naive.go:53-105) applied to the HBM snapshot.  Keys are INTERNAL keys.  The last op on a key wins;
 * deleting an absent key is a no-op.  The slab is rebuilt by a device-side merge (O(store bytes) of HBM copy), so
 * callers batch their commits (e.g. the <=300-event collector batches). */
enum { KB_OP_PUT = 0, KB_OP_DEL = 1 };
typedef struct kb_write_op {
    uint32_t type;                              /* KB_OP_PUT / KB_OP_DEL */
    const uint8_t *key;  uint64_t key_len;
    const uint8_t *val;  uint64_t val_len;      /* ignored for KB_OP_DEL */
    uint64_t expire_unix;                       /* KB_OP_PUT: 0 = never; else the wall-clock second at which the engine
                                                   stops returning the key (the backend writes /events/ keys with a ttl,
                                                   storage.BatchWrite.Put(key, val, ttl), badger WithTTL batch.go:47-93) */
} kb_write_op;
int kb_apply_batch(kb_ctx *ctx, const kb_write_op *ops, uint64_t n);
/* TTL: engines with SupportTTL() (badger) never delete expired keys explicitly -- they just stop returning them.  The
 * mirror keeps (expire_unix, key) of every TTL put and kb_expire removes from the snapshot every record whose time has
 * come (one kb_apply_batch-style merge).  The storage adaptor calls it from a ticker and in front of every compaction, so
 * the mirror lags the engine by at most one tick.  *n_dropped (optional) = records removed. */
int kb_expire(kb_ctx *ctx, uint64_t now_unix, uint64_t *n_dropped);
/* compact_key record used by checkCompactRace (scanner.go:594-626); present=0 clears it */
int kb_set_compact_revision(kb_ctx *ctx, int present, uint64_t rev);

/* ---- range scan: replaces scanner.Range / Count / RangeStream -> worker.run -------------------
 * (pkg/backend/scanner/scanner.go:83-145, 389-516; receivers scanner/receiver.go:62-103) */
enum {
    KB_OUT_HOST = 0,    /* results copied to pinned host memory inside the call                    */
    KB_OUT_DEVICE = 1,  /* results stay in HBM; the view holds device pointers.  kb_range_batch returns as soon
                           as the per-request counts are known, while the copy into the arena may still be
                           running on the context's copy stream: order consumers behind it with
                           kb_result_wait(ctx, res, their_stream), or call kb_result_wait(ctx, res, NULL) /
                           kb_sync(ctx) before touching the arena or the per-kv arrays from the host              */
    KB_OUT_COUNT = 2,   /* emptyResultReceiver: counts only (scanner.Count)                         */
    /* OR-ed into KB_OUT_HOST / KB_OUT_DEVICE: the arena holds the answer as etcd protobuf elements, one per
     * emitted kv in emission order, ready to be framed and sent (go.etcd.io/etcd/api/v3 v3.5.2 field numbers):
     *   KVS:    etcdserverpb.RangeResponse.kvs elements -- replaces kvToEtcdKv + Marshal of the List answer
     *           (pkg/server/etcd/backendshim.go:269-282, 427-436)
     *   EVENTS: etcdserverpb.WatchResponse.events elements, mvccpb.Event{kv} -- the range-stream answer
     *           (backendshim.go:349-363); batches are cut at elem_off[300*i] (receiver.go:119-138)            */
    KB_WIRE_ETCD_KVS = 0x10,
    KB_WIRE_ETCD_EVENTS = 0x20
};

typedef struct kb_range_req {
    const uint8_t *start;  uint64_t start_len;   /* internal keys: coder.EncodeObjectKey(key, 0)  */
    const uint8_t *end;    uint64_t end_len;     /* half-open [start, end); start >= end answers
                                                     nothing (backend.List refuses such ranges before
                                                     the scanner is reached, range.go:147-149)     */
    uint64_t read_rev;                            /* workerConfig.revision                         */
    int64_t  limit;                               /* scanner.Range limit; <= 0 means unlimited     */
} kb_range_req;

typedef struct kb_range_view {
    uint64_t n_req;
    const uint64_t *req_first;  /* n_req+1: kvs of request q are [req_first[q], req_first[q+1])   */
    const uint64_t *req_count;  /* n_req: worker.run's object count (for scanner.Count)            */
    const uint64_t *req_examined; /* n_req: records pulled from the iterator                      */
    uint64_t n_kvs;
    /* per emitted kv, in the reference's emission order */
    const uint32_t *rec_idx;    /* index of the store record that supplied key/value/revision     */
    const uint64_t *rev;        /* KeyValue.Revision                                              */
    const uint64_t *key_off;    /* offset of the USER key inside bytes                            */
    const uint32_t *key_len;
    const uint64_t *val_off;
    const uint32_t *val_len;
    const uint8_t  *bytes;      /* arena (host pinned for KB_OUT_HOST, device for KB_OUT_DEVICE)   */
    uint64_t n_bytes;
    int on_device;              /* 1: bytes AND the per-kv arrays are device pointers (req_* stay host) */
    /* wire modes: element k is bytes[elem_off[k] .. elem_off[k+1]); key_off / val_off point at the raw user-key and
     * value bytes inside it; the elements of request q are contiguous: elem_off[req_first[q]] .. elem_off[req_first[q+1]] */
    const uint64_t *elem_off;   /* n_kvs+1, NULL in the arena modes or when n_kvs == 0             */
    int wire;                   /* 0, KB_WIRE_ETCD_KVS or KB_WIRE_ETCD_EVENTS                       */
} kb_range_view;

/* One call = one batch of independent scanner.Range requests answered on one snapshot. */
int kb_range_batch(kb_ctx *ctx, const kb_range_req *reqs, uint64_t n_req, int out_mode, kb_result **out);
/* Optional: start the bound search of a batch ahead of the kb_range_batch call that will ask for it (identical bounds, same
 * snapshot; anything else is ignored).  A caller with a queue of pending requests submits batch n+1 before it waits for
 * batch n; the one host round trip of a range call then overlaps the previous batch's kernels. */
int kb_range_prefetch(kb_ctx *ctx, const kb_range_req *reqs, uint64_t n_req);
/* A range call in two halves (kb_range_batch == submit + collect): kb_range_submit lays the batch out and launches its
 * kernels, kb_range_collect waits for its rows and builds the result (host copies for KB_OUT_HOST happen here).  A caller
 * with a queue of batches (the shim under concurrent scanner.Range goroutines) submits batch n+1 before it collects batch
 * n: n+1's bound search, layout and first kernels then overlap n's kernels.  Two batches are in flight at most; a third
 * submission first waits for the rows of the batch two back.  Collect in any order; every pending ends in exactly one of
 * kb_range_collect (also on failure) or kb_pending_free.  Any other entry point may be called in between (it first
 * reads back the rows of what is in flight). */
typedef struct kb_pending kb_pending;
int kb_range_submit(kb_ctx *ctx, const kb_range_req *reqs, uint64_t n_req, int out_mode, kb_pending **out);
int kb_range_collect(kb_ctx *ctx, kb_pending *pending, kb_result **out);
void kb_pending_free(kb_ctx *ctx, kb_pending *pending);
int kb_range_view_get(const kb_result *res, kb_range_view *view);
/* Completion of a KB_OUT_DEVICE answer (range arena and per-kv arrays; delivery lists of a watch match): cuda_stream (a cudaStream_t) is made to wait for it on the device;
 * with cuda_stream == NULL the calling host thread blocks until it is complete.  No-op for host-resident results. */
int kb_result_wait(kb_ctx *ctx, const kb_result *res, void *cuda_stream);

/* Framing around the wire elements (host side, a few bytes each; return the byte count written, out >= 32 bytes
 * [+ reason_len for the watch head]):
 *   RangeResponse  = kb_wire_range_head(header.revision) | KVS elements | kb_wire_range_tail(more, count)
 *                    (backendshim.go:269-277: count = len(kvs) + (more ? 1 : 0))
 *   WatchResponse  = kb_wire_watch_head(header.revision, 0, NULL, 0) | EVENTS elements of one batch
 *   end of stream  = kb_wire_watch_head(revision, 1, err, len)       (backendshim.go:353-355, scanner.go:179-192) */
uint64_t kb_wire_range_head(uint64_t header_rev, uint8_t *out);
uint64_t kb_wire_range_tail(int more, int64_t count, uint8_t *out);
uint64_t kb_wire_watch_head(uint64_t header_rev, int canceled, const uint8_t *reason, uint64_t reason_len, uint8_t *out);

/* ---- point reads: replaces backend.get / getInternalVal (pkg/backend/range.go:81-121): a reverse iterator from
 * EncodeObjectKey(key, revision) down to EncodeObjectKey(key, 0) with limit 1.  revision 0 means "latest". */
enum { KB_GET_FOUND = 0, KB_GET_NOT_FOUND = 1, KB_GET_TOMBSTONE = 2 /* ErrKeyNotFound, but mod_rev is valid */ };

typedef struct kb_get_req {
    const uint8_t *key;  uint64_t key_len;   /* USER key */
    uint64_t revision;
} kb_get_req;

typedef struct kb_get_view {
    uint64_t n;
    const uint8_t  *status;    /* KB_GET_* per request (host)                                     */
    const uint64_t *mod_rev;   /* revision the returned value was written at (host)               */
    const uint32_t *rec_idx;   /* store record (host; undefined unless found / tombstone)         */
    const uint64_t *val_off;   /* offset of the value inside bytes (host; found only)             */
    const uint32_t *val_len;
    const uint8_t  *bytes;     /* values (host pinned for KB_OUT_HOST, device for KB_OUT_DEVICE)  */
    uint64_t n_bytes;
    int on_device;
} kb_get_view;

int kb_get_batch(kb_ctx *ctx, const kb_get_req *reqs, uint64_t n, int out_mode, kb_result **out);
int kb_get_view_get(const kb_result *res, kb_get_view *view);

/* ---- compaction sweep: replaces scanner.Compact -> worker.run(compact=true) --------------------
 * (scanner.go:195-199, 457-491, 538-591; driver pkg/backend/compact.go:31-127).
 * Classifies every record of [start,end) visible at `rev`; the deletes themselves are applied by the
 * caller in bulk (the reference issues one storage transaction per victim, scanner.go:538-564). */
enum {
    KB_V_SUPERSEDED = 1,  /* scanner.go:465-469 store.Del of an older version                     */
    KB_V_TOMBSTONE  = 2,  /* scanner.go:472-475 store.Del of a tombstone-valued version            */
    KB_V_REVRECORD  = 3,  /* scanner.go:477-491 store.DelCurrent of a deleted-flag revision record */
    KB_V_TTL_REVREC = 4,  /* scanner.go:576-581 (only when !SupportTTL and timeout_rev != 0)       */
    KB_V_TTL_OBJECT = 5   /* scanner.go:582-585                                                    */
};

typedef struct kb_compact_view {
    uint64_t n_victims;
    const uint32_t *victim_idx;    /* store record index of every delete call, in the reference's order */
    const uint8_t  *victim_class;
    uint64_t count;                /* worker.run's count (includes the Q5 double count)            */
    uint64_t examined;
    int on_device;                 /* 1: victim_idx / victim_class are device pointers              */
} kb_compact_view;

int kb_compact_sweep(kb_ctx *ctx, const uint8_t *start, uint64_t start_len, const uint8_t *end, uint64_t end_len,
                     uint64_t rev, uint64_t timeout_rev, int support_ttl, int out_mode, kb_result **out);
int kb_compact_view_get(const kb_result *res, kb_compact_view *view);

/* ---- watch fan-out: replaces WatcherHub.Stream + processEvents/filterByRevision/filterByPrefix --
 * (pkg/backend/watcherhub.go:78-92, pkg/backend/watch.go:119-159) */
int kb_watch_add(kb_ctx *ctx, const uint8_t *prefix, uint64_t prefix_len, uint64_t min_rev, uint32_t *id);
int kb_watch_del(kb_ctx *ctx, uint32_t id);
int kb_watch_count(kb_ctx *ctx, uint64_t *n);

typedef struct kb_events {
    const uint8_t  *keys;  const uint64_t *key_off;   /* Event.Kv.Key (user keys), n+1 offsets     */
    const uint64_t *rev;                               /* Event.Revision                            */
    uint64_t n;
    const uint64_t *batch_off; uint64_t n_batches;    /* collector batches (<=300, backend.go:41);
                                                          NULL/0 = one batch                        */
} kb_events;

typedef struct kb_match_view {
    uint64_t n_watchers;         /* number of registered watcher ids covered (max id + 1)          */
    const uint64_t *start;       /* n_watchers+1: deliveries of watcher id w = [start[w],start[w+1]) */
    const uint32_t *event_idx;   /* event indices, ascending per watcher (stream order)             */
    uint64_t n_deliveries;
    int on_device;               /* 1: event_idx is a device pointer, complete after kb_result_wait / kb_sync (start[]
                                    and n_deliveries are host values, final when the call returns)          */
} kb_match_view;

int kb_watch_match(kb_ctx *ctx, const kb_events *ev, int out_mode, kb_result **out);
/* device-resident event slabs (benchmarks / GPU-side producers) */
int kb_events_upload(kb_ctx *ctx, const kb_events *ev, kb_events_dev **out);
void kb_events_free(kb_ctx *ctx, kb_events_dev *ev);
int kb_watch_match_dev(kb_ctx *ctx, const kb_events_dev *ev, int out_mode, kb_result **out);
int kb_match_view_get(const kb_result *res, kb_match_view *view);

void kb_result_free(kb_ctx *ctx, kb_result *res);

/* ---- multi-GPU: the committed-revision cursor (tso.GetRevision, pkg/backend/tso/tso.go:47-49;
 * follower /status poll pkg/server/service/revision/revision.go:219-259) as ONE ncclAllGather of one
 * uint64 per rank; min over ranks = the globally readable revision. */
#define KB_NCCL_ID_BYTES 128
int kb_nccl_unique_id(uint8_t id[KB_NCCL_ID_BYTES]);
int kb_nccl_init(kb_ctx *ctx, const uint8_t id[KB_NCCL_ID_BYTES], int rank, int nranks);
int kb_cursor_allgather(kb_ctx *ctx, uint64_t local_rev, uint64_t *all_revs /* nranks */, uint64_t *min_rev);
/* which transport kb_cursor_allgather uses: stores into peer memory over NVLink (every peer's slot buffer could be
 * mapped at kb_nccl_init), ncclAllGather otherwise.  kb_cursor_force_nccl(ctx, 1) selects the NCCL path although peers
 * map -- collective: every rank has to switch before the next exchange. */
enum { KB_CURSOR_NONE = 0, KB_CURSOR_SINGLE = 1, KB_CURSOR_NCCL = 2, KB_CURSOR_P2P = 3 };
int kb_cursor_transport(kb_ctx *ctx);
int kb_cursor_force_nccl(kb_ctx *ctx, int on);

/* ---- measurement hooks (bench.py): per-kernel CUDA-event timing on the ctx stream -------------- */
typedef struct kb_prof_entry {
    char     name[32];
    uint64_t launches;
    double   total_ms;
    uint64_t alg_bytes;   /* algorithmic bytes the launches were asked to move (DESIGN.md section 4) */
} kb_prof_entry;
int kb_prof_enable(kb_ctx *ctx, int on); /* 0 off, 1 every kernel, 2 only k_gather */
int kb_prof_reset(kb_ctx *ctx);
int kb_prof_read(kb_ctx *ctx, kb_prof_entry *entries, int cap, int *n);
uint64_t kb_launch_count(kb_ctx *ctx); /* kernels launched by this ctx since open */

#ifdef __cplusplus
}
#endif
#endif
