"""bench.py --dump-outputs: the answers of the last timed step written as float32 / float64 .npy files of at most 64 MB.
The CPU test drives dump_outputs with stand-in results; the GPU test runs the bench and compares its dump with the oracle
on the same seeded workload, rebuilt in this process."""
from __future__ import annotations

import importlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import binding as ko

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture
def bench(monkeypatch):
    # importing bench.py sets a CUDA connection count for the process; keep it out of the other tests
    monkeypatch.delenv("CUDA_DEVICE_MAX_CONNECTIONS", raising=False)
    return importlib.import_module("bench")


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


class _Eng:
    def __init__(self, arena: bytes):
        self.arena = arena

    def read_device(self, ptr, nbytes, sync=True):
        return self.arena[ptr : ptr + nbytes]


class _Range:
    def __init__(self, n_kvs, rng):
        self.req_first = np.array([0, 7, n_kvs], np.uint64)
        self.req_count = np.array([3, 5], np.uint64)
        self.req_examined = np.array([11, n_kvs + 4], np.uint64)
        self.n_kvs = n_kvs
        self.bytes_ptr = 0
        klen = rng.integers(1, 9, n_kvs).astype(np.uint32)
        vlen = rng.integers(0, 13, n_kvs).astype(np.uint32)
        sizes = np.stack([klen, vlen], 1).reshape(-1).astype(np.uint64)
        off = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.uint64).reshape(-1, 2)
        self.cols = {"rec_idx": rng.permutation(n_kvs).astype(np.uint32), "rev": rng.integers(1, 2**40, n_kvs).astype(np.uint64),
                     "key_off": off[:, 0], "key_len": klen, "val_off": off[:, 1], "val_len": vlen}
        self.arena = rng.integers(0, 256, int(sizes.sum()), dtype=np.uint8).tobytes()

    def wait(self):
        pass

    def device_array(self, name, dtype):
        return self.cols[name].astype(dtype)


class _Match:
    def __init__(self, rng):
        self.start = np.array([0, 4, 4, 30], np.uint64)
        self.idx = rng.integers(0, 5000, 30).astype(np.uint32)

    def device_event_idx(self):
        return self.idx


def test_dump_outputs_writes_samples_within_the_limit(bench, tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_MAX_KVS", 40)
    monkeypatch.setattr(bench, "DUMP_BYTES_KVS", 9)
    monkeypatch.setattr(bench, "DUMP_MAX_DELIVERIES", 16)
    r, m = _Range(100, np.random.default_rng(1)), _Match(np.random.default_rng(2))
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), _Eng(r.arena), r, m)
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a)  # the sample is fixed
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    pos = a["range_kv_pos"].astype(np.int64)
    assert len(pos) == 40 and np.all(np.diff(pos) > 0)
    assert np.array_equal(a["range_rec_idx"], r.cols["rec_idx"][pos]) and np.array_equal(a["range_rev"], r.cols["rev"][pos])
    assert np.array_equal(a["range_val_len"], r.cols["val_len"][pos])
    assert np.array_equal(a["range_req_examined"], r.req_examined)
    kv = a["range_bytes_kv"].astype(np.int64)
    assert len(kv) == 9 and set(kv) <= set(pos)
    for what, name in (("key", "range_key_bytes"), ("val", "range_value_bytes")):
        exp = b"".join(r.arena[int(r.cols[what + "_off"][k]) : int(r.cols[what + "_off"][k] + r.cols[what + "_len"][k])]
                       for k in kv)
        assert a[name].astype(np.uint8).tobytes() == exp
    dpos = a["fan_delivery_pos"].astype(np.int64)
    assert np.array_equal(a["fan_start"], m.start) and np.array_equal(a["fan_event_idx"], m.idx[dpos])


@pytest.mark.gpu
def test_bench_dump_is_the_oracle_answer(bench, tmp_path):
    out = tmp_path / "dump"
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "1", "--no-extras",
                        "--no-cpu-baseline", "--no-parity", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-3000:]
    assert json.loads(p.stdout.strip().splitlines()[-1])["steps"] == 3
    d = _load(out)
    assert sum(v.nbytes for v in d.values()) <= 64 << 20
    wl = bench.build_workload(0, 1)
    store, ost = wl["store"], ko.OracleStore(wl["store"])
    exps = [ko.range_(ost, s, e, rev, lim) for s, e, rev, lim in wl["reqs"]]
    assert d["range_req_first"].tolist() == np.cumsum([0] + [len(x.emit) for x in exps]).tolist()
    assert d["range_req_count"].tolist() == [x.count for x in exps]
    assert d["range_req_examined"].tolist() == [x.examined for x in exps]
    emit = np.concatenate([x.emit for x in exps])
    assert "range_kv_pos" not in d and np.array_equal(d["range_rec_idx"], emit)
    kvs = ko.ScanResult(0, emit, None, None, 0, False, 0).kvs(store)  # (user key, value, revision) per emitted kv
    assert d["range_rev"].tolist() == [rev for _, _, rev in kvs]
    assert d["range_key_len"].tolist() == [len(k) for k, _, _ in kvs]
    assert d["range_val_len"].tolist() == [len(v) for _, v, _ in kvs]
    kv = d["range_bytes_kv"].astype(np.int64)
    assert len(kv) == 2048
    assert d["range_key_bytes"].astype(np.uint8).tobytes() == b"".join(kvs[i][0] for i in kv)
    assert d["range_value_bytes"].astype(np.uint8).tobytes() == b"".join(kvs[i][1] for i in kv)
    start, idx, _ = ko.fanout(wl["events"], wl["watchers"], threads=4)
    assert d["fan_start"].tolist() == start.tolist()
    assert "fan_delivery_pos" not in d and np.array_equal(d["fan_event_idx"], idx)
