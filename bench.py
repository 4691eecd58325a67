#!/usr/bin/env python
"""bench.py -- range-scan + watch-fanout throughput of the B200 path (and of the reference CPU path).

    python bench.py --gpus N --steps K --warmup W [--impl reference]

One STEP = one pass of the hot path over one batch of synthetic input (BASELINE.json configs[1]+[2]):
  * scan   : one full-range unlimited Range (RangeStream shape) + Q=256 namespace List requests (limit 10 001) on
             a 1M-record snapshot (200k objects x [1 revision record + 4 versions], 256 B keys, 2 KB values,
             5 % tombstoned, read revision = 90th percentile);
  * fan-out: a 100k-event burst (334 collector batches of <= 300) against 10k watchers
             (9 984 namespace prefixes + 16 cluster-wide);
  * at N > 1 every rank owns the namespaces that fnv1a64(prefix) maps to it (weak scaling: ~1M records, ~10k
    watchers, ~100k events per GPU) and the step starts with ONE ncclAllGather of the per-shard revision cursor.
Unit of work ("event") = one stored MVCC record examined by a scan, or one watch event matched against the whole
watcher set.  `value` = events/s with inputs resident in HBM; `e2e` = the same through the C-ABI with HOST buffers
(host->device and device->host copies inside the timed region).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

# more hardware work queues than the default 8: the bench drives two contexts x three streams (+ torch's); streams that
# share a queue serialise behind each other (must be set before the CUDA context exists)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from kubebrain_b200 import synth  # noqa: E402
from kubebrain_b200.coder import NormalCoder, prefix_end  # noqa: E402
from kubebrain_b200.packed import PackedEvents, PackedWatchers, Slab  # noqa: E402

CODER = NormalCoder()
METRIC = "range-scan + watch-fanout events/sec"
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent

N_OBJECTS, VERSIONS, LU, LV = 200_000, 4, 256, 2048
NS_STORE, NS_EVENTS, N_NS_WATCH, N_CLUSTER_WATCH, N_EVENTS, Q_LISTS = 1000, 11_000, 9984, 16, 100_000, 256
BURST_START = 2_000_000


ns_shard = synth.ns_shard


def build_workload(rank: int, world: int, mode: str = "weak"):
    """per-rank shard of the synthetic: store, list requests, watchers, event burst.
    weak  : every GPU gets ~1M records / ~10k watchers / ~100k events (the data set grows with N);
    strong: BASELINE configs[4] as written -- 8M records (1.6M objects), 50k namespace watchers (+16 cluster-wide,
            replicated) and ONE 100k-event burst in total, hash-sharded over the N GPUs."""
    t0 = time.time()
    if mode == "strong":
        n_obj, n_ns, n_nsw, n_ev, ns_ev = 1_600_000, 50_000, 50_000, N_EVENTS, 55_000
    else:
        n_obj, n_ns, n_nsw, n_ev, ns_ev = N_OBJECTS * world, NS_STORE * world, N_NS_WATCH * world, N_EVENTS * world, \
            NS_EVENTS * world
    store, meta = synth.gen_store(n_obj, VERSIONS, LU, LV, n_ns, config_id=2,
                                  shard=(rank, world) if world > 1 else None)
    lo, hi = CODER.encode_object_key(b"/registry/", 0), CODER.encode_object_key(b"/registry0", 0)
    reqs = [(lo, hi, meta.read_rev, 0)]
    owned = np.nonzero(ns_shard(np.arange(n_ns), world) == rank)[0]
    resn = [b"pods", b"configmaps", b"secrets", b"services", b"deployments", b"events"]
    for i in range(Q_LISTS):
        p = b"/registry/" + resn[i % 6] + b"/ns-%05d/" % int(owned[(i * 7) % len(owned)])
        reqs.append((CODER.encode_object_key(p, 0), CODER.encode_object_key(prefix_end(p), 0), meta.read_rev, 10001))
    # watchers: namespace watchers of the namespaces this rank owns + the cluster-wide ones (replicated)
    w_all = synth.gen_watchers(n_nsw, N_CLUSTER_WATCH, BURST_START, BURST_START + n_ev // 2)
    ns_ids = np.arange(n_nsw)
    keep = np.concatenate([ns_shard(ns_ids, world) == rank, np.ones(N_CLUSTER_WATCH, dtype=bool)])
    idx = np.nonzero(keep)[0]
    watchers = w_all if world == 1 else PackedWatchers(w_all.prefixes.take(idx), w_all.min_rev[idx])
    # events: the burst routed by the same hash
    ev_all = synth.gen_events(n_ev, LU, ns_ev, BURST_START)
    if world > 1:
        mat = ev_all.keys.data.reshape(-1, LU)
        digits = mat[:, 18:23].astype(np.int64) - 48  # "/registry/pods/ns-%05d/": the namespace number
        ev_ns = digits @ np.array([10000, 1000, 100, 10, 1], dtype=np.int64)
        sel = np.nonzero(ns_shard(ev_ns, world) == rank)[0]
        n = len(sel)
        ev = PackedEvents(Slab.from_fixed(mat[sel]), ev_all.rev[sel],
                          np.array(list(range(0, n, 300)) + [n], dtype=np.uint64))
    else:
        ev = ev_all
    return dict(store=store, meta=meta, reqs=reqs, watchers=watchers, events=ev, gen_s=time.time() - t0, mode=mode,
                n_obj_global=n_obj, n_ns_global=n_ns)


def bind_to_gpu_numa_node(local_rank: int):
    """Pin this process to the CPUs of the NUMA node its GPU hangs off BEFORE any pinned host memory is allocated, so
    the response pools are node-local (round 1: at N=8 the 8 x 484 MB of pinned-host writes per step reached only
    ~160 GB/s in aggregate).  Returns (original affinity, description) -- the caller restores the mask for CPU legs."""
    try:
        orig = os.sched_getaffinity(0)
    except AttributeError:
        return None, "no sched_getaffinity"
    try:
        import torch

        pr = torch.cuda.get_device_properties(local_rank)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        base = f"/sys/bus/pci/devices/{bdf}/"
        node = int(open(base + "numa_node").read().strip())
        cpus = set()
        for part in open(base + "local_cpulist").read().strip().split(","):
            lo_, _, hi_ = part.partition("-")
            cpus.update(range(int(lo_), int(hi_ or lo_) + 1))
        cpus &= orig
        if node < 0 or not cpus:
            return orig, f"gpu {bdf}: no NUMA information"
        os.sched_setaffinity(0, cpus)
        return orig, f"gpu {bdf} -> numa node {node}, {len(cpus)} cpus"
    except Exception as e:  # sysfs layout differs, attribute missing: run unbound
        return orig, f"unbound ({type(e).__name__})"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)"""

    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.p = None
        self.path = f"/tmp/kb_clocks_{os.getpid()}.csv"

    def start(self):
        try:
            self.f = open(self.path, "w")
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.FIELDS}",
                                       "--format=csv,noheader,nounits", "-lms", "20"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        for line in open(self.path):
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.unlink(self.path)
        except OSError:
            pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            for k in ("hbm_gbs", "hbm_gb_s", "hbm_copy_gbs"):
                if k in d:
                    return float(d[k]), "measured"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback"


def ncu_traffic(kernel: str):
    """dram bytes per launch of the dominant kernel from the committed ncu --set full capture, if any"""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(kernel)
        except Exception:
            return None
    return None


# ---------------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation of the path (C restatement, all usable host threads)
# ---------------------------------------------------------------------------------------------------------
def host_threads() -> int:
    """threads this process may really use: the scheduler affinity mask bounded by the cgroup CPU quota (os.cpu_count()
    reports the machine, not the container -- the round-1 reference arm oversubscribed a quota-limited box 5x)"""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:  # cgroup v2
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            n = min(n, max(1, int(float(q) / float(per) + 0.5)))
    except (OSError, ValueError):
        try:  # cgroup v1
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0 and per > 0:
                n = min(n, max(1, int(q / per + 0.5)))
        except (OSError, ValueError):
            pass
    return max(1, n)


CPU_LEGS = ("scan_faithful_s", "scan_zero_copy_s", "lists_s", "fanout_alloc_s", "fanout_prealloc_s")


def cpu_legs(ost, wl, threads: int):
    """one pass of the step's work on the host, every leg timed on its own:
      scan, faithful   : partition-parallel worker.run WITH the badger iterator's per-record copies (KeyCopy + 2x ValueCopy,
                         reference pkg/storage/badger/iter.go:85-92, scanner.go:441,495), P = threads (TiKV shape)
      scan, zero copy  : the same loop over borrowed slices (no per-record copies), P = threads
      lists            : 256 x List(limit 10001), one goroutine each (run back to back on one thread: ~170 records each)
      fan-out          : every watcher runs filterByRevision + filterByPrefix over all batches, watchers sharded over
                         `threads`; with (watch.go:141) and without the per-batch output allocation"""
    from oracle import binding as ko

    t = {}
    s, e, rev, _ = wl["reqs"][0]
    t0 = time.perf_counter()
    n_f, ex_f, _ = ko.bench_scan(ost, s, e, rev, 0, True, threads)
    t["scan_faithful_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    n_z, ex_z, _ = ko.bench_scan(ost, s, e, rev, 0, False, threads)
    t["scan_zero_copy_s"] = time.perf_counter() - t0
    assert (n_f, ex_f) == (n_z, ex_z)
    examined, emitted = ex_f, n_f
    t0 = time.perf_counter()
    for s, e, rev, lim in wl["reqs"][1:]:
        n, ex, _ = ko.bench_scan(ost, s, e, rev, lim, False, 1)
        examined += ex
        emitted += n
    t["lists_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    _, idx, _ = ko.fanout(wl["events"], wl["watchers"], threads=threads, alloc_per_batch=True)
    t["fanout_alloc_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    _, idx2, _ = ko.fanout(wl["events"], wl["watchers"], threads=threads, alloc_per_batch=False)
    t["fanout_prealloc_s"] = time.perf_counter() - t0
    assert len(idx) == len(idx2)
    return t, examined, emitted, len(idx)


def cpu_summary(legs_mean, events: int, threads: int):
    fastest = (min(legs_mean["scan_faithful_s"], legs_mean["scan_zero_copy_s"]) + legs_mean["lists_s"] +
               min(legs_mean["fanout_alloc_s"], legs_mean["fanout_prealloc_s"]))
    faithful = legs_mean["scan_faithful_s"] + legs_mean["lists_s"] + legs_mean["fanout_alloc_s"]
    return {
        "value": events / fastest, "unit": "events/s", "cores": threads, "kind": "port",
        "s_per_step": fastest, "legs_s": {k: legs_mean[k] for k in CPU_LEGS},
        "value_faithful": events / faithful, "s_per_step_faithful": faithful,
        "variant": "fastest of each leg: scan = min(faithful copies, zero copy) at P = cores; fan-out = min(per-batch "
                   "allocation, preallocated); `value_faithful` keeps the badger-style copies and watch.go:141 allocation",
    }


def run_reference(args, rank: int, world: int):
    if rank != 0:
        return
    from oracle import binding as ko

    wl = build_workload(0, 1)
    ost = ko.OracleStore(wl["store"])
    threads = host_threads()
    for _ in range(max(args.warmup, 1)):
        cpu_legs(ost, wl, threads)
    acc = {k: 0.0 for k in CPU_LEGS}
    for _ in range(args.steps):
        legs, examined, emitted, deliveries = cpu_legs(ost, wl, threads)
        for k in CPU_LEGS:
            acc[k] += legs[k]
    mean = {k: v / args.steps for k, v in acc.items()}
    events = examined + wl["events"].n
    summ = cpu_summary(mean, events, threads)
    # context: the badger shape (a single partition => the full scan is ONE goroutine, badger.go:52-54)
    t1 = time.perf_counter()
    s, e, rev, _ = wl["reqs"][0]
    ko.bench_scan(ost, s, e, rev, 0, True, 1)
    summ["badger_single_partition_scan_s"] = time.perf_counter() - t1
    summ["sample"] = (f"{args.steps} full steps, every leg timed separately on {threads} threads (affinity mask bounded by the "
                      "cgroup quota): 1 unlimited Range over 1M records + 256 List(limit 10001) + 100k-event burst x 10k "
                      "watchers; value = fastest variant of each leg (BASELINE.md section 3)")
    value = summ["value"]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "events/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": summ["s_per_step"] * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(1, wl),
        "cpu_baseline": summ,
        "e2e": {"value": value, "unit": "events/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def workload_config(world: int, wl):
    strong = wl.get("mode") == "strong"
    return {
        "workload": ("configs[4]: 8M MVCC records (256B key, 2KB val) + 50k watchers + one 100k-event burst hash-sharded over "
                     "the GPUs, per GPU 1 full Range + 256 List(limit 10001)") if strong else
                    ("configs[1]+[2]: 1M MVCC records/GPU (256B key, 2KB val), 1 full Range + 256 List(limit 10001), "
                     "100k-event burst x 10k watchers/GPU"),
        "records_per_gpu": int(wl["store"].n), "list_requests": Q_LISTS, "watchers_per_gpu": int(wl["watchers"].n),
        "events_per_gpu": int(wl["events"].n), "read_rev": int(wl["meta"].read_rev),
        "parallelism": f"hash-shard x{world}" if world > 1 else "single GPU",
        "l2": "inputs larger than L2 (>= 0.7 GB streamed from HBM per step)",
        "overlap": "scan and fan-out run concurrently on two kb_ctx of the same GPU, K batches and K bursts per timed region, "
                   "each half on its own host thread; range batches are submitted ahead (kb_range_submit / kb_range_collect, "
                   "`pipeline.range_batches_in_flight` on the B200 line), so one batch's host round trip and first kernels "
                   "overlap the previous batch's kernels",
        "unit_of_work": "records examined + events matched",
    }


# ---------------------------------------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------------------------------------
def run_b200(args, rank: int, local_rank: int, world: int):
    import torch

    from kubebrain_b200._lib import KB_OUT_DEVICE, KB_OUT_HOST, Engine

    torch.cuda.set_device(local_rank)
    orig_affinity, numa_note = bind_to_gpu_numa_node(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    wl = build_workload(rank, world, args.mode)
    # two contexts on the same GPU, as in the reference where scans and the watch hub are independent goroutines:
    # `eng` owns the HBM-resident snapshot (scans), `weng` owns the watcher tables (fan-out); each has its own stream
    prio = os.environ.get("KB_BENCH_PRIO", "fanout")  # which context gets the high-priority streams: scan | fanout | none
    # (measured: fanout 0.316 ms, scan 0.325 ms, none 0.336 ms per step -- the short fan-out kernels otherwise queue behind the
    # scan context's persistent CTAs)
    eng = Engine(local_rank, high_priority=(prio == "scan" and not args.serial))
    eng.load_sorted(wl["store"])
    weng = eng if args.serial else Engine(local_rank, high_priority=(prio == "fanout"))
    weng.watch_add_many(wl["watchers"])
    # the revision-cursor communicator (one uint64 per rank)
    uid = Engine.nccl_unique_id() if rank == 0 else bytes(128)
    if world > 1:
        t = torch.tensor(list(uid), dtype=torch.uint8, device="cuda")
        dist.broadcast(t, 0)
        uid = bytes(t.cpu().tolist())
    # the cursor exchange runs on the fan-out context: it is off the scan call's critical path (round 1: 12 -> 51 us in front
    # of every range batch at N = 1 -> 8) and the scan of step n reads at the revision the exchange of step n-1 agreed on
    ceng = weng
    ceng.nccl_init(uid, rank, world)
    evh = weng.events_upload(wl["events"])
    stream = torch.cuda.ExternalStream(eng.stream())
    wstream = torch.cuda.ExternalStream(weng.stream())
    # the kb_range_req[] a C / cgo caller passes directly; marshalled once so the timed call is the C-ABI call itself
    reqs = Engine.pack_range_reqs(wl["reqs"])
    local_rev = int(wl["meta"].last_rev)
    if not args.no_prefetch:
        # pipeline depth one: the FIRST step's bound search is submitted here, every step then submits the next step's
        # before it asks for its own answer (one submission and one consumption per step)
        eng.range_prefetch(reqs)

    # the fan-out half runs on a long-lived worker thread (ctypes releases the GIL inside the C ABI calls)
    import queue
    import threading

    jobs_q, done_q = queue.SimpleQueue(), queue.SimpleQueue()
    pyt = {"cursor": 0.0, "range_call": 0.0, "range_submit": 0.0, "range_collect": 0.0, "range_result": 0.0, "fan_call": 0.0, "n": 0}

    def worker():
        torch.cuda.set_device(local_rank)
        while True:
            fn = jobs_q.get()
            if fn is None:
                return
            try:
                done_q.put(fn())
            except Exception as e:  # surfaced on the main thread
                done_q.put(e)

    wthread = None
    if not args.serial:
        wthread = threading.Thread(target=worker, daemon=True)
        wthread.start()

    readable = {"rev": 0}
    # --dump-outputs: countdown[half] counts the timed steps of that half still to come.  The answer of the last one is kept
    # open (a result stays valid until kb_result_free) to be written after the timed region; every other answer is freed
    # as usual, so no step runs with more result buffers alive than without the dump.
    countdown, kept = {"scan": 0, "fan": 0}, {}

    def release(half, res):
        if countdown[half]:
            countdown[half] -= 1
            if countdown[half] == 0:
                kept[half] = res
                return
        res.close()

    def fan_device():
        t0 = time.perf_counter()
        _, readable["rev"] = ceng.cursor_allgather(local_rev)
        pyt["cursor"] += time.perf_counter() - t0
        m = weng.watch_match_dev(evh, KB_OUT_DEVICE)
        d = m.n_deliveries
        release("fan", m)
        pyt["fan_call"] = pyt.get("fan_call", 0.0) + time.perf_counter() - t0
        return d

    def fan_e2e():
        _, readable["rev"] = ceng.cursor_allgather(local_rev)
        m = weng.watch_match(wl["events"], KB_OUT_HOST)
        d = m.n_deliveries
        dbytes = d * 4 + (m.n_watchers + 1) * 8
        m.close()
        return dbytes

    def both(scan_fn, fan_fn):
        if args.serial:
            a = scan_fn()
            return a, fan_fn()
        jobs_q.put(fan_fn)
        a = scan_fn()
        b = done_q.get()
        if isinstance(b, Exception):
            raise b
        return a, b

    def scan_device():
        t1 = time.perf_counter()
        if not args.no_prefetch:
            eng.range_prefetch(reqs)  # the NEXT step's bound search (a server with queued requests submits ahead); this
            # step's call picks up the one submitted during the previous step: every step still does one search
        r = eng.range_batch(reqs, KB_OUT_DEVICE)
        t2 = time.perf_counter()
        ex = int(r.req_examined.sum())
        nk = r.n_kvs
        release("scan", r)
        t3 = time.perf_counter()
        pyt["range_call"] += t2 - t1
        pyt["range_result"] += t3 - t2
        pyt["n"] += 1
        return ex, nk

    def scan_e2e():
        if not args.no_prefetch:
            eng.range_prefetch(reqs)
        r = eng.range_batch(reqs, KB_OUT_HOST)
        ex = int(r.req_examined.sum())
        nbytes = r.n_bytes + r.n_kvs * 36
        checksum = int(r.arena[:: max(1, r.n_bytes // 4096)].sum()) if r.n_bytes else 0  # the host reads the result
        r.close()
        return ex, nbytes, checksum

    def step_device():
        (ex, nk), d = both(scan_device, fan_device)
        return ex, nk, d

    def step_e2e():
        (ex, nbytes, checksum), dbytes = both(scan_e2e, fan_e2e)
        return ex, nbytes + dbytes, checksum

    # Batches in flight (default 2): batch n+1 is submitted (bound search, layout, launches) before batch n is collected,
    # the way the shim serves concurrent scanner.Range goroutines; every step is still one whole batch, and all K batches
    # are submitted, answered and drained inside the timed region.  The fan-out bursts run on their own thread, K of them
    # in the same region (the reference's watcher hub is an independent goroutine, it does not wait for scans).
    def scan_pipelined(steps, e2e):
        mode = KB_OUT_HOST if e2e else KB_OUT_DEVICE
        out = None
        pend = []

        def finish(pd):
            t2 = time.perf_counter()
            r = pd.collect()
            t3 = time.perf_counter()
            ex = int(r.req_examined.sum())
            if e2e:
                nbytes = r.n_bytes + r.n_kvs * 36
                checksum = int(r.arena[:: max(1, r.n_bytes // 4096)].sum()) if r.n_bytes else 0  # the host reads the result
                o = (ex, nbytes, checksum)
            else:
                o = (ex, r.n_kvs)
            release("scan", r)
            pyt["range_collect"] += t3 - t2
            pyt["range_result"] += time.perf_counter() - t3
            return o

        for _ in range(steps):
            t1 = time.perf_counter()
            pend.append(eng.range_submit(reqs, mode))
            pyt["range_submit"] += time.perf_counter() - t1
            pyt["n"] += 1
            if len(pend) >= args.in_flight:
                out = finish(pend.pop(0))
        while pend:
            out = finish(pend.pop(0))
        return out

    def run_steps(steps, e2e):
        """K steps; returns what the last step of each half returned"""
        if args.serial or args.in_flight <= 1:
            out = None
            for _ in range(steps):
                out = step_e2e() if e2e else step_device()
            return out
        fan = fan_e2e if e2e else fan_device
        jobs_q.put(lambda: [fan() for _ in range(steps)][-1])
        sc = scan_pipelined(steps, e2e)
        f = done_q.get()
        if isinstance(f, Exception):
            raise f
        return (sc[0], sc[1], f) if not e2e else (sc[0], sc[1] + f, sc[2])

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(e2e, steps):
        barrier()
        a, b, bw = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        a.record(stream)
        t0 = time.perf_counter()
        out = run_steps(steps, e2e)
        # device-resident answers return while their last copy is still running on the context's copy stream:
        # drain both contexts before the end events so that the timed region holds ALL the work of the K steps
        eng.sync()
        if weng is not eng:
            weng.sync()
        b.record(stream)
        bw.record(wstream)
        barrier()
        wall = time.perf_counter() - t0
        dev_ms = max(a.elapsed_time(b), a.elapsed_time(bw))  # both streams must have drained
        if dist is not None:
            t = torch.tensor([dev_ms, wall * 1e3], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dev_ms, wall = float(t[0]), float(t[1]) / 1e3
        return dev_ms, wall, out

    # clocks / throttle reasons are sampled from the warm-up to the end of the e2e pass (the timed regions last
    # only tens of milliseconds, so sampling them alone would give one or two points)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    n_warm = max(args.warmup, 3, args.in_flight + 1)  # every lane of the range pipeline allocates its scratch on first use
    run_steps(n_warm, False)
    run_steps(n_warm, True)

    # timed region: CUDA events bracket only the two HBM-bound kernels (level 2) so the event records do not
    # perturb the step; a second, untimed pass with every kernel bracketed fills the per-kernel table
    engines = [eng] if weng is eng else [eng, weng]
    for e in engines:
        e.prof_reset()
        e.prof_enable(2)
    l0 = sum(e.launch_count() for e in engines)
    for k in list(pyt):
        pyt[k] = 0
    if args.dump_outputs:
        countdown.update(scan=args.steps, fan=args.steps)
    dev_ms, wall_s, (examined, n_kvs, deliveries) = timed(False, args.steps)
    if args.dump_outputs:
        last = (kept.pop("scan"), kept.pop("fan"))
        if rank == 0:
            dump_outputs(args.dump_outputs, eng, *last)
        for res in last:
            res.close()
    host_call_us = {k: 1e6 * v / max(pyt["n"], 1) for k, v in pyt.items() if k != "n"}
    launches = sum(e.launch_count() for e in engines) - l0
    prof_major = {}
    for e in engines:
        e.prof_enable(0)
        prof_major.update({p["name"]: p for p in e.prof_read()})
        e.prof_reset()
        e.prof_enable(1)
    prof_ms, _, _ = timed(False, args.steps)
    prof = []
    for e in engines:
        e.prof_enable(0)
        prof += e.prof_read()
    for p in prof:  # the timed-region measurement wins for the kernels it covers
        if p["name"] in prof_major:
            p.update(prof_major[p["name"]])
    e2e_ms, e2e_wall, (examined2, d2h_bytes, _) = timed(True, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    # the cursor exchange on its own, both transports (the timed loop uses the peer-memory kernel when peers map)
    cursor_us = {}
    if world > 1:
        for name, force_nccl in (("p2p" if ceng.cursor_mode() == "p2p" else "nccl", False), ("nccl", True)):
            if name in cursor_us:
                continue
            ceng.cursor_force_nccl(force_nccl)
            for _ in range(5):
                ceng.cursor_allgather(local_rev)
            barrier()
            t0 = time.perf_counter()
            for _ in range(50):
                ceng.cursor_allgather(local_rev)
            cursor_us[name] = (time.perf_counter() - t0) / 50 * 1e6
        ceng.cursor_force_nccl(False)
        t = torch.tensor([cursor_us.get("p2p", 0.0), cursor_us.get("nccl", 0.0)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        cursor_us = {k: float(v) for k, v in zip(("p2p", "nccl"), t.tolist()) if v > 0}
    # parity of the very answers that were timed, on every rank (raises -> rc != 0)
    parity = None if args.no_parity else parity_check(eng, weng, wl, evh, reqs, rank, world, dist)
    # the two bulk kernels with the GPU to themselves (untimed; CUDA events around each launch): inside the timed region their
    # event brackets include the time they wait for SM residency behind the other lane's bulk kernel
    alone = None
    if rank == 0:
        eng.sync()
        weng.sync()
        eng.prof_reset()
        eng.prof_enable(2)
        for _ in range(6):
            r = eng.range_batch(reqs, KB_OUT_DEVICE)
            r.wait()
            r.close()
            eng.sync()
        eng.prof_enable(0)
        alone = {p["name"]: p for p in eng.prof_read() if p["launches"]}
        eng.prof_reset()
    if orig_affinity is not None:
        os.sched_setaffinity(0, orig_affinity)  # CPU legs below use every core the container has

    events_local = examined + wl["events"].n
    if dist is not None:
        t = torch.tensor([events_local, launches], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        events_total, launches_total = float(t[0]), int(t[1])
    else:
        events_total, launches_total = float(events_local), int(launches)
    ms_per_step = dev_ms / args.steps
    value = events_total / (ms_per_step / 1e3)
    e2e_value = events_total / (e2e_ms / args.steps / 1e3)
    h2d_bytes = wl["events"].n * (32 + 12) + reqs.n * 2 * 300

    if rank == 0:
        peak, peak_src = measured_hbm_peak()
        kern = []
        for p in prof:
            if p["launches"] == 0:
                continue
            ms = p["total_ms"] / p["launches"]
            per_launch = p["alg_bytes"] / p["launches"]
            kern.append({"name": p["name"], "launches_per_step": p["launches"] / args.steps, "avg_us": ms * 1e3,
                         "alg_bytes_per_launch": per_launch,
                         "achieved_gbs": (per_launch / 1e9) / (ms / 1e3) if ms > 0 else None,
                         "share": p["total_ms"] / max(dev_ms if p["name"] in prof_major else prof_ms, 1e-9),
                         "timed_region": p["name"] in prof_major})
        host_segments = sorted([k for k in kern if k["name"].startswith("host:")], key=lambda k: -k["share"])
        kern = sorted([k for k in kern if not k["name"].startswith("host:")], key=lambda k: -k["share"])
        # dominant kernel = the one that moves the most algorithmic bytes per step (the latency-bound fan-out kernel is
        # longer inside a step, where it shares the GPU with the scan, but moves 40 MB against the gather's 950 MB)
        dom = max(kern, key=lambda k: k["alg_bytes_per_launch"] * k["launches_per_step"]) if kern else None
        roof = None
        if dom:
            roof = {"kernel": dom["name"], "bound": "hbm", "achieved": dom["achieved_gbs"], "peak": peak,
                    "peak_source": peak_src, "unit": "GB/s", "frac": dom["achieved_gbs"] / peak,
                    "traffic": ncu_traffic(dom["name"]), "share_of_step": dom["share"]}
            roof["others"] = [{"kernel": k["name"], "achieved": k["achieved_gbs"], "frac": (k["achieved_gbs"] or 0) / peak,
                               "avg_us": k["avg_us"], "traffic": ncu_traffic(k["name"])}
                              for k in kern if k["name"] in ("k_decode_lcp", "k_fanout") and k is not dom]
            # the streams of the two contexts overlap, so kernel times add up to more than the wall step: the share that
            # compares with a serialised ncu launch list is the one of the summed kernel time
            ksum = sum(k["avg_us"] * k["launches_per_step"] for k in kern)
            roof["share_of_kernel_time"] = dom["avg_us"] * dom["launches_per_step"] / ksum if ksum else None
            # the same kernels with the GPU to themselves, and the step as a whole (all algorithmic bytes of a step over the
            # step time): with batches in flight the event brackets of the bulk kernels overlap each other
            roof["alone"] = {}
            for name in ("k_gather", "k_decode_lcp"):
                a = (alone or {}).get(name)
                if a:
                    us = 1e3 * a["total_ms"] / a["launches"]
                    gbs = (a["alg_bytes"] / a["launches"] / 1e9) / (us / 1e6)
                    roof["alone"][name] = {"avg_us": us, "achieved": gbs, "frac": gbs / peak}
            step_bytes = sum(k["alg_bytes_per_launch"] * k["launches_per_step"] for k in kern)
            roof["step"] = {"alg_bytes": step_bytes, "achieved": step_bytes / 1e9 / (ms_per_step / 1e3),
                            "frac": step_bytes / 1e9 / (ms_per_step / 1e3) / peak}
            roof["note"] = ("achieved / frac: CUDA events around the kernel inside the timed region (includes waiting for SM "
                            "residency when another batch's bulk kernel holds the shared memory); alone: the same launch with the "
                            "GPU to itself; step: all algorithmic bytes of a step over ms_per_step")
        line = {
            "metric": METRIC, "value": value, "unit": "events/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.mode,
            "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": workload_config(world, wl),
            "pipeline": {"range_batches_in_flight": 1 if args.serial else max(1, args.in_flight),
                         "halves": "joined at every step" if (args.serial or args.in_flight <= 1) else "independent threads, K steps each"},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "events/s", "h2d_bytes_per_step": int(h2d_bytes),
                    "d2h_bytes_per_step": int(d2h_bytes), "ms_per_step": e2e_ms / args.steps},
            "gpu_launches": launches_total,
            "roofline": roof,
            "kernels": kern, "host_segments": host_segments,
            "scan_records_per_step": int(examined), "emitted_kvs_per_step": int(n_kvs),
            "fanout_events_per_step": int(wl["events"].n), "deliveries_per_step": int(deliveries),
            "wall_ms_per_step": wall_s * 1e3 / args.steps, "gen_s": wl["gen_s"],
            "host_call_us": host_call_us, "numa": numa_note,
            "parity_checked": bool(parity and parity.get("parity_checked")), "parity": parity,
        }
        if cursor_us:
            line["cursor_exchange_us"] = cursor_us
        if world == 1 and not args.no_extras:
            line["latency"] = latency_probe(eng, wl)
            line["fanout_alone"] = fanout_alone(weng, evh, wl, peak)
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(wl)
        if world == 1 and not args.no_extras:
            line["extra"] = {"compaction": compaction_extra(local_rank, peak, full=not args.small_compaction),
                             "wire": wire_extra(eng, wl), "write_path": write_rate_extra(eng, wl)}
        print(json.dumps(line), flush=True)
    if wthread is not None:
        jobs_q.put(None)
        wthread.join(timeout=5)
    weng.events_free(evh)
    if weng is not eng:
        weng.close()
    eng.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------
# parity of the timed answers (every rank, every N): the GPU answers of the bench workload against the oracle
# ---------------------------------------------------------------------------------------------------------
MASK64 = (1 << 64) - 1


def _dev_bytes(ptr: int, nbytes: int):
    """a torch uint8 view of raw device memory owned by libkbb200 (no copy)"""
    import torch

    class _H:
        pass

    h = _H()
    h.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (int(ptr), False), "version": 3}
    return torch.as_tensor(h, device="cuda")


def _digest_device(ptr: int, nbytes: int) -> int:
    """position-weighted checksum of ALL arena bytes, computed on the device: sum_i word_i * (2i+1) mod 2^64"""
    import torch

    assert nbytes % 8 == 0
    w = _dev_bytes(ptr, nbytes).view(torch.int64)
    tot = 0
    step = 1 << 24
    for a in range(0, w.numel(), step):  # chunked: bounds the temporaries to 128 MB
        b = min(a + step, w.numel())
        wt = torch.arange(a, b, device="cuda", dtype=torch.int64) * 2 + 1
        tot = (tot + int((w[a:b] * wt).sum().item())) & MASK64
    return tot


def _digest_expected(store, rec_idx: np.ndarray) -> int:
    """the same checksum of the arena the reference's answer would fill: per emitted kv [internal key, zero padded to
    16][value, zero padded to 16], in emission order"""
    koff, voff = store.keys.off.astype(np.int64), store.vals.off.astype(np.int64)
    idx = rec_idx.astype(np.int64)
    kl, vl = koff[idx + 1] - koff[idx], voff[idx + 1] - voff[idx]
    assert len(idx) == 0 or (kl.min() == kl.max() and vl.min() == vl.max()), "bench store emits fixed-size kvs"
    if len(idx) == 0:
        return 0
    klen, vlen = int(kl[0]), int(vl[0])
    kp, vp = (klen + 15) // 16 * 16, (vlen + 15) // 16 * 16
    slot_words = (kp + vp) // 8
    tot = 0
    rows = 4096
    with np.errstate(over="ignore"):
        for a in range(0, len(idx), rows):
            sl = idx[a : a + rows]
            m = np.zeros((len(sl), kp + vp), dtype=np.uint8)
            m[:, :klen] = store.keys.data[koff[sl][:, None] + np.arange(klen)]
            m[:, kp : kp + vlen] = store.vals.data[voff[sl][:, None] + np.arange(vlen)]
            w = m.view("<u8").reshape(-1)
            wt = (np.arange(a * slot_words, a * slot_words + w.size, dtype=np.uint64) * np.uint64(2) + np.uint64(1))
            tot = (tot + int((w * wt).sum(dtype=np.uint64))) & MASK64
    return tot


def parity_check(eng, weng, wl, evh, reqs, rank: int, world: int, dist):
    """After the timed region: (1) this rank's GPU answers of the step -- emitted record indices, examined / object counts,
    a device-computed digest of ALL arena bytes, the per-watcher delivery lists -- against the oracle on this rank's
    shard; (2) N > 1: one broad List answered by every shard, merged by sharded.merge_list_runs, against the oracle on the
    unsharded store.  Any mismatch raises (the bench exits non-zero)."""
    from kubebrain_b200 import sharded
    from kubebrain_b200._lib import KB_OUT_DEVICE, KB_OUT_HOST
    from oracle import binding as ko

    t0 = time.perf_counter()
    ost = ko.OracleStore(wl["store"])
    r = eng.range_batch(reqs, KB_OUT_DEVICE)
    rec = r.device_array("rec_idx", np.uint32)
    exp_all = []
    for q, (s, e, rev, lim) in enumerate(wl["reqs"]):
        exp = ko.range_(ost, s, e, rev, lim)
        a, b = int(r.req_first[q]), int(r.req_first[q + 1])
        if not np.array_equal(rec[a:b].astype(np.uint64), exp.emit):
            raise AssertionError(f"rank {rank}: request {q}: emitted records differ from the oracle")
        if int(r.req_examined[q]) != exp.examined or int(r.req_count[q]) != exp.count:
            raise AssertionError(f"rank {rank}: request {q}: examined / count differ from the oracle")
        exp_all.append(exp.emit)
    exp_idx = np.concatenate(exp_all) if exp_all else np.zeros(0, np.uint64)
    d_dev = _digest_device(r.bytes_ptr, r.n_bytes) if r.n_bytes else 0
    d_exp = _digest_expected(wl["store"], exp_idx)
    if d_dev != d_exp:
        raise AssertionError(f"rank {rank}: arena digest {d_dev:#x} differs from the oracle's {d_exp:#x}")
    n_kvs, n_bytes = r.n_kvs, r.n_bytes
    r.close()
    start, idx, _ = ko.fanout(wl["events"], wl["watchers"], threads=host_threads())
    m = weng.watch_match_dev(evh, KB_OUT_DEVICE)
    if m.start.tolist() != start.tolist() or not np.array_equal(m.device_event_idx(), idx.astype(np.uint32)):
        raise AssertionError(f"rank {rank}: fan-out delivery lists differ from the oracle")
    deliveries = m.n_deliveries
    m.close()
    out = {"parity_checked": True, "kvs": int(n_kvs), "arena_bytes_digested": int(n_bytes), "deliveries": int(deliveries),
           "requests": len(wl["reqs"])}
    if world > 1:
        broad = b"/registry/services/"
        assert sharded.owner_of_prefix(broad, world) is None
        blo, bhi = CODER.encode_object_key(broad, 0), CODER.encode_object_key(prefix_end(broad), 0)
        rev = int(wl["meta"].read_rev)
        g = eng.range_batch([(blo, bhi, rev, 0)], KB_OUT_HOST)
        run = [(k, len(v), rv) for k, v, rv in g.kvs(0)]
        g.close()
        runs = [None] * world
        dist.all_gather_object(runs, run)
        if rank == 0:
            # the unsharded store with short values: keys, revisions and tombstones do not depend on Lv
            gstore, gmeta = synth.gen_store(wl["n_obj_global"], VERSIONS, LU, 16, wl["n_ns_global"], config_id=2)
            gst = ko.OracleStore(gstore)
            assert gmeta.read_rev == rev
            for limit in (0, 5000):
                exp = ko.range_(gst, blo, bhi, rev, limit + 1 if limit else 0)  # backend.List asks for limit + 1
                exp_kv = [(k, rv) for k, _, rv in exp.kvs(gstore)]
                got, more = sharded.merge_list_runs(runs, limit)
                if [(k, rv) for k, _, rv in got] != (exp_kv[:limit] if limit else exp_kv) or \
                        more != (limit > 0 and len(exp_kv) > limit) or any(vl != LV for _, vl, _ in got):
                    raise AssertionError(f"merged broad List (limit {limit}) differs from the oracle on the unsharded store")
            out["merged_list_kvs"] = len(exp_kv)
        ok = [None] * world
        dist.all_gather_object(ok, True)  # every rank reached this point without raising
    out["seconds"] = time.perf_counter() - t0
    return out


DUMP_MAX_KVS = 1 << 20  # per-kv arrays: 24 B a kv in the dump
DUMP_MAX_DELIVERIES = 1 << 21  # delivery list: 4 B a delivery
DUMP_BYTES_KVS = 2048  # kvs whose key and value bytes are written: ~19 MB at the bench's 2 KB values
DUMP_LIMIT = 64 << 20


def _dump_positions(n: int, cap: int) -> np.ndarray:
    """all of 0..n-1, or a fixed seeded sorted sample of `cap` of them"""
    if n <= cap:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, cap, replace=False))


def dump_outputs(out_dir: str, eng, r, m):
    """Write one step's answers as DIR/<name>.npy (float64 for indices and revisions, float32 for lengths, bytes and
    delivered event indices) so that two builds can be compared output for output on the same seeded inputs.
      range_req_first / _count / _examined : per request of the batch
      range_rec_idx / _rev / _key_len / _val_len : per emitted kv (at the positions range_kv_pos when there are more
                                                   than DUMP_MAX_KVS)
      range_bytes_kv, range_key_bytes, range_value_bytes : the key and value bytes of a seeded sample of the emitted kvs,
                                                   concatenated in sample order (their lengths are in range_*_len)
      fan_start, fan_event_idx : per-watcher offsets into the delivery list, the delivered event indices (at the positions
                                 fan_delivery_pos when there are more than DUMP_MAX_DELIVERIES)"""
    out = {"range_req_first": r.req_first, "range_req_count": r.req_count, "range_req_examined": r.req_examined}
    r.wait()
    pos = _dump_positions(r.n_kvs, DUMP_MAX_KVS)
    if len(pos) < r.n_kvs:
        out["range_kv_pos"] = pos
    cols = {name: r.device_array(name, dt)[pos] for name, dt in (
        ("rec_idx", np.uint32), ("rev", np.uint64), ("key_off", np.uint64), ("key_len", np.uint32),
        ("val_off", np.uint64), ("val_len", np.uint32))}
    out["range_rec_idx"], out["range_rev"] = cols["rec_idx"], cols["rev"]
    out["range_key_len"], out["range_val_len"] = cols["key_len"].astype(np.float32), cols["val_len"].astype(np.float32)
    pick = _dump_positions(len(pos), DUMP_BYTES_KVS)
    out["range_bytes_kv"] = pos[pick]
    for what in ("key", "val"):
        chunks = [eng.read_device(r.bytes_ptr + int(o), int(n), sync=False)
                  for o, n in zip(cols[what + "_off"][pick], cols[what + "_len"][pick])]
        name = "range_key_bytes" if what == "key" else "range_value_bytes"
        out[name] = np.frombuffer(b"".join(chunks), dtype=np.uint8).astype(np.float32)
    out["fan_start"] = m.start
    idx = m.device_event_idx()
    dpos = _dump_positions(len(idx), DUMP_MAX_DELIVERIES)
    if len(dpos) < len(idx):
        out["fan_delivery_pos"] = dpos
    assert len(idx) == 0 or int(idx.max()) < 1 << 24, "event indices must be exact in float32"
    out["fan_event_idx"] = idx[dpos].astype(np.float32)
    out = {k: v if v.dtype == np.float32 else v.astype(np.float64) for k, v in out.items()}
    total = sum(v.nbytes for v in out.values())
    assert total <= DUMP_LIMIT, f"dump of {total} bytes exceeds {DUMP_LIMIT}"
    os.makedirs(out_dir, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def latency_probe(eng, wl):
    """SURVEY 8d config 2 latency run: ONE List(limit 10 000) over the whole prefix (backend.List asks the scanner for
    10 001, pkg/backend/range.go:153-171; worker.run stops pulling once the receiver is full).  Reported in microseconds:
    device-resident answer complete, host-resident answer complete (e2e), and the CPU port on one thread."""
    from kubebrain_b200._lib import KB_OUT_DEVICE, KB_OUT_HOST, Engine
    from oracle import binding as ko

    p = b"/registry/"
    s, e = CODER.encode_object_key(p, 0), CODER.encode_object_key(prefix_end(p), 0)
    rev = int(wl["meta"].read_rev)
    pk = Engine.pack_range_reqs([(s, e, rev, 10001)])
    ost = ko.OracleStore(wl["store"])
    exp = ko.range_(ost, s, e, rev, 10001)
    r = eng.range_batch(pk, KB_OUT_HOST)
    assert np.array_equal(r.rec_idx.astype(np.uint64), exp.emit) and int(r.req_examined[0]) == exp.examined
    n_bytes = r.n_bytes
    r.close()

    def rep(mode, n=40):
        ts = []
        for _ in range(n):
            eng.sync()
            t0 = time.perf_counter()
            r = eng.range_batch(pk, mode)
            if mode == KB_OUT_DEVICE:
                r.wait()
            ts.append(time.perf_counter() - t0)
            r.close()
        return statistics.median(ts[5:]) * 1e6

    dev_us, e2e_us = rep(KB_OUT_DEVICE), rep(KB_OUT_HOST)
    cpu = []
    for faithful in (True, False):
        ts = []
        for _ in range(7):
            t0 = time.perf_counter()
            ko.bench_scan(ost, s, e, rev, 10001, faithful, 1)
            ts.append(time.perf_counter() - t0)
        cpu.append(statistics.median(ts) * 1e6)
    return {"request": "List(/registry/ .. prefix end, limit 10000 -> 10001 asked)", "examined": int(exp.examined),
            "emitted": int(len(exp.emit)), "answer_bytes": int(n_bytes), "device_us": dev_us, "e2e_us": e2e_us,
            "cpu_port_faithful_us": cpu[0], "cpu_port_zero_copy_us": cpu[1], "parity_checked": True}


def fanout_alone(weng, evh, wl, peak: float, reps: int = 30):
    """BASELINE configs[2] on its own (no scan beside it): one 100k-event burst against the 10k watchers, device resident;
    roofline against SURVEY 8d's algorithmic bytes E*(Lu+8+4) + W*44 + D*8"""
    import torch

    from kubebrain_b200._lib import KB_OUT_DEVICE

    ws = torch.cuda.ExternalStream(weng.stream())
    for _ in range(5):
        weng.watch_match_dev(evh, KB_OUT_DEVICE).close()
    weng.sync()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = weng.launch_count()
    a.record(ws)
    for _ in range(reps):
        m = weng.watch_match_dev(evh, KB_OUT_DEVICE)
        d = m.n_deliveries
        m.close()
    weng.sync()
    b.record(ws)
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / reps
    # where the time goes: per-kernel events and the phase spans k_fanout's first CTA stamps (a separate, untimed pass)
    weng.prof_reset()
    weng.prof_enable(1)
    for _ in range(10):
        weng.watch_match_dev(evh, KB_OUT_DEVICE).close()
    weng.prof_enable(0)
    parts = {p["name"]: round(1e3 * p["total_ms"] / p["launches"], 1) for p in weng.prof_read()
             if p["launches"] and (p["name"].startswith("fan:") or p["name"] in ("k_fanout", "k_expand_write"))}
    weng.prof_reset()
    E, W = int(wl["events"].n), int(wl["watchers"].n)
    alg = E * (LU + 12) + W * 44 + d * 8
    return {"workload": "configs[2] alone: 100k-event burst x 10k watchers, device-resident slab and answer",
            "us_per_burst": ms * 1e3, "events_per_s": E / (ms / 1e3), "deliveries_per_s": d / (ms / 1e3),
            "launches_per_burst": (weng.launch_count() - l0) / reps, "parts_us": parts,
            "roofline": {"bound": "hbm", "achieved": alg / 1e9 / (ms / 1e3), "peak": peak, "unit": "GB/s",
                         "frac": alg / 1e9 / (ms / 1e3) / peak, "alg_bytes": alg,
                         "note": "latency bound: 41 MB of algorithmic traffic per burst"}}


def write_rate_extra(eng, wl):
    """extra, run last (it changes the snapshot): the write path behind the collector's <= 300-event batches on the bench
    store -- 150 updates per batch, each a CAS of the revision record + a Put of the new 2 KB version
    (pkg/backend/txn.go:249-265) -- through kb_apply_batch (heap + sorted directory: the cost of a batch does not grow with
    the bytes of the store)"""
    import random
    import struct

    keys = wl["store"].keys
    rng = random.Random(5)
    rev = int(wl["meta"].last_rev)
    n0 = eng.store_info()[0]
    batches, n_ops = 40, 0
    val = b"w" * LV
    plan = []
    for _ in range(batches):
        ops = []
        for i in rng.sample(range(keys.n), 150):
            uk = keys[i][4:-9]
            rev += 1
            ops.append((CODER.encode_object_key(uk, 0), struct.pack(">Q", rev)))
            ops.append((CODER.encode_object_key(uk, rev), val))
        plan.append(ops)
    eng.apply_batch(plan[0])
    t0 = time.perf_counter()
    for ops in plan[1:]:
        eng.apply_batch(ops)
        n_ops += len(ops)
    dt = time.perf_counter() - t0
    assert eng.store_info()[0] == n0 + batches * 150
    # the snapshot still answers: a count over everything at the new revision
    lo, hi = CODER.encode_object_key(b"/registry/", 0), CODER.encode_object_key(b"/registry0", 0)
    from kubebrain_b200._lib import KB_OUT_COUNT

    r = eng.range_batch([(lo, hi, rev, 0)], KB_OUT_COUNT)
    objects = int(r.req_count[0])
    r.close()
    return {"workload": f"{batches - 1} batches of 300 ops (150 updates) on the {n0}-record store",
            "ops_per_s": n_ops / dt, "ms_per_batch": dt / (batches - 1) * 1e3, "records_after": int(eng.store_info()[0]),
            "objects_visible_after": objects}


def wire_extra(eng, wl):
    """extra (not part of the headline): the full-range answer written as etcd protobuf elements by the device
    (KB_WIRE_ETCD_EVENTS, the range-stream shape) instead of padded [key][value] pairs"""
    from kubebrain_b200._lib import KB_OUT_DEVICE, KB_WIRE_ETCD_EVENTS, Engine

    reqs = Engine.pack_range_reqs(wl["reqs"][:1])
    for _ in range(3):
        eng.range_batch(reqs, KB_OUT_DEVICE | KB_WIRE_ETCD_EVENTS).close()
    eng.prof_reset()
    eng.prof_enable(1)
    reps = 5
    for _ in range(reps):
        r = eng.range_batch(reqs, KB_OUT_DEVICE | KB_WIRE_ETCD_EVENTS)
        nk, nb = r.n_kvs, r.n_bytes
        r.close()
    eng.prof_enable(0)
    kern = {p["name"]: {"avg_us": 1e3 * p["total_ms"] / p["launches"],
                        "achieved_gbs": (p["alg_bytes"] / p["launches"] / 1e9) / (p["total_ms"] / p["launches"] / 1e3)
                        if p["total_ms"] > 0 else None}
            for p in eng.prof_read() if p["launches"] and p["name"] in ("k_wire_copy", "k_wire_jobs", "k_decode_lcp", "k_emit")}
    return {"workload": "1 full Range of the bench store as WatchResponse.events elements, device resident",
            "kvs": int(nk), "wire_bytes": int(nb), "kernels": kern}


def compaction_extra(device: int, peak: float, full: bool = True):
    """BASELINE configs[3] (not part of the timed step): keep-latest sweep over 10M objects x (1 revision record + 9
    versions), Lu=64 -> 100M records, ~80M victims, device-resident victim list; the same sweep's ordered victim list is
    compared with the oracle in this run.  Falls back to 1/10 size when the host cannot hold the synthetic."""
    import torch

    from kubebrain_b200._lib import KB_OUT_DEVICE, KB_OUT_HOST, Engine
    from oracle import binding as ko

    if full:
        try:
            import psutil

            full = psutil.virtual_memory().available > 48 * 2**30
        except Exception:
            full = False
    n_obj, n_ns = (10_000_000, 50_000) if full else (1_000_000, 10_000)
    store, meta = synth.gen_store(n_obj, 9, 64, 64, n_ns, config_id=4, tomb_frac=0.02)
    eng = Engine(device)
    eng.load_sorted(store)
    lo, hi = CODER.encode_object_key(b"/registry/", 0), CODER.encode_object_key(b"/registry0", 0)
    for _ in range(2):
        eng.compact_sweep(lo, hi, meta.last_rev, out_mode=KB_OUT_DEVICE).close()
    stream = torch.cuda.ExternalStream(eng.stream())
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 4
    torch.cuda.synchronize()
    a.record(stream)
    for _ in range(reps):
        r = eng.compact_sweep(lo, hi, meta.last_rev, out_mode=KB_OUT_DEVICE)
        nv = r.n_victims
        r.close()
    b.record(stream)
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / reps
    # per-kernel times in a separate pass (the event pairs add gaps)
    eng.prof_reset()
    eng.prof_enable(1)
    for _ in range(2):
        eng.compact_sweep(lo, hi, meta.last_rev, out_mode=KB_OUT_DEVICE).close()
    eng.prof_enable(0)
    kern = {p["name"]: {"avg_us": 1e3 * p["total_ms"] / p["launches"],
                        "achieved_gbs": (p["alg_bytes"] / p["launches"] / 1e9) / (p["total_ms"] / p["launches"] / 1e3)
                        if p["total_ms"] > 0 else None}
            for p in eng.prof_read() if p["launches"] and not p["name"].startswith("host:")}
    # parity in the same run: the ordered victim list with classes against the oracle
    got = eng.compact_sweep(lo, hi, meta.last_rev, out_mode=KB_OUT_HOST)
    exp = ko.scan(ko.OracleStore(store), [lo, hi], meta.last_rev, compact=True, collect=False)
    ok = (got.n_victims == len(exp.victims) and got.count == exp.count and
          np.array_equal(got.victim_idx.astype(np.uint64), exp.victims) and np.array_equal(got.victim_class, exp.vclass))
    got.close()
    eng.close()
    if not ok:
        raise AssertionError("compaction sweep differs from the oracle")
    # SURVEY 8d config 4: per record Lk + 4 + 4 = 85 B, + 9 B for every 9-byte value and every revision record
    vl = store.vals.lengths()
    alg = int(store.n) * 85 + int(((vl == 9) | (np.arange(store.n) % 10 == 0)).sum()) * 9 + (int(store.n) + 7) // 8
    return {"workload": f"config 4 {'FULL size' if full else 'at 1/10'}: {store.n / 1e6:.0f}M records (Lk=77), compact at max revision",
            "records": int(store.n), "victims": int(nv), "ms_per_sweep": ms, "records_per_s": store.n / (ms / 1e3),
            "parity_checked": True,
            "roofline": {"bound": "hbm", "achieved": alg / 1e9 / (ms / 1e3), "peak": peak, "unit": "GB/s",
                         "frac": alg / 1e9 / (ms / 1e3) / peak, "alg_bytes": alg},
            "kernels": kern}


def cpu_baseline(wl):
    """the oracle port timed on this box's host cores on the same workload (bounded: 2 full steps, legs timed apart)"""
    from oracle import binding as ko

    ost = ko.OracleStore(wl["store"])
    threads = host_threads()
    cpu_legs(ost, wl, threads)
    reps = 2
    acc = {k: 0.0 for k in CPU_LEGS}
    for _ in range(reps):
        legs, examined, emitted, deliveries = cpu_legs(ost, wl, threads)
        for k in CPU_LEGS:
            acc[k] += legs[k]
    summ = cpu_summary({k: v / reps for k, v in acc.items()}, examined + wl["events"].n, threads)
    summ["sample"] = (f"{reps} full steps on {threads} threads, legs timed separately (1M-record Range faithful / zero copy, "
                      "256 Lists, 100k events x 10k watchers with / without the per-batch allocation)")
    return summ


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--serial", action="store_true", help="scan and fan-out back to back on one stream")
    ap.add_argument("--mode", default="weak", choices=["weak", "strong"],
                    help="weak: ~1M records / 10k watchers / 100k events per GPU; strong: configs[4] as written, 8M records + "
                         "50k watchers + one 100k burst in total")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle comparison of the timed answers")
    ap.add_argument("--prefetch", dest="no_prefetch", action="store_false", default=True,
                    help="submit the next step's bound search ahead (kb_range_prefetch).  Off by default: measured, it moves the "
                         "next decode under the previous gather and both HBM-bound kernels slow each other down (0.38 vs 0.33 ms)")
    ap.add_argument("--in-flight", type=int, default=2,
                    help="range batches in flight (kb_range_submit / kb_range_collect); 1 = one kb_range_batch per step, "
                         "joined with the fan-out burst at every step (the round-1 loop)")
    ap.add_argument("--small-compaction", action="store_true", help="extra: config 4 at 1/10 size instead of 100M records")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the range batch and watch match answers of the last timed step (rank "
                         "0's shard) as DIR/<name>.npy, at most 64 MB; the inputs are seeded, so two builds can be compared")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the answers of the B200 path; the reference arm returns counts only")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    run_b200(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
