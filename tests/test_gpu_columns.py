"""The decoded columns (crev / cword, kubebrain_b200/csrc/kb_decode.cuh) after write batches.

A write batch carries every surviving record's column entry through the directory merge and recomputes only the
entries it made stale.  A stale entry changes an answer only for some read revisions and some request bounds, so after
every batch three things are compared: the engine that took the writes, a fresh engine loaded from the same items
(columns built from scratch), and the oracle -- over read revisions below, between and above the versions, sub-ranges
that start on the changed records, and the compaction sweep with and without the TTL pass."""
from __future__ import annotations

import random
import struct

import pytest

from kubebrain_b200._lib import Engine
from kubebrain_b200.packed import PackedStore
from oracle import binding as ko
from tests import fuzz
from tests.test_gpu_parity import check_compact, check_ranges

pytestmark = pytest.mark.gpu

MAGIC = fuzz.MAGIC
TOMB = fuzz.TOMB


def _ik(uk: bytes, rev: int) -> bytes:
    return MAGIC + uk + b"$" + struct.pack(">Q", rev)


@pytest.fixture(scope="module")
def engines():
    a, b = Engine(0), Engine(0)
    yield a, b
    a.close()
    b.close()


def _ttl_safe(op):
    """a revision record of an /events/ key keeps a value of >= 8 bytes (the TTL sweep reads value[:8]; Go panics)"""
    k, v = op
    if v is not None and len(v) < 8 and len(k) >= 13 and k.startswith(MAGIC) and k[-9:] == b"$" + b"\x00" * 8 \
            and b"/events/" in k[4:-9]:
        v = struct.pack(">Q", 7)
    return (k, v)


def _apply(items: dict, ops):
    for op in ops:
        if op[1] is None:
            items.pop(op[0], None)
        else:
            items[op[0]] = op[1]


def _bounds(cur: PackedStore, touched, seed: int):
    """the whole store, random sub-ranges, and ranges that start on / right behind the records a batch touched (a
    request's first record has no predecessor inside the request; the one behind it does)"""
    keys = cur.keys.tolist()
    out = fuzz.fuzz_bounds(cur, seed, n=4)
    for k in list(touched)[:12]:
        out.append((k, b"\xff" * 4))
        out.append((k + b"\x00", b"\xff" * 4))
        out.append((k[: max(len(k) - 9, 1)], k + b"\x00"))
    out.append((keys[0], keys[min(3, len(keys) - 1)] + b"\x00"))
    return out


def check_all(engines, items: dict, revs, touched=(), timeouts=(0,), seed=0):
    """the written engine and a freshly loaded one, both against the oracle"""
    written, fresh = engines
    cur = PackedStore.from_items(list(items.items()))
    st = ko.OracleStore(cur)
    fresh.load_sorted(cur)
    assert written.store_info()[0] == cur.n
    bounds = _bounds(cur, touched, seed)
    for e in (written, fresh):
        e.set_compact_revision(None)
        reqs = [(s, t, r, lim) for (s, t) in bounds for r in revs for lim in (0, 3)]
        for i in range(0, len(reqs), 64):
            check_ranges(e, cur, st, reqs[i:i + 64])
        for s, t in bounds[:6]:
            for r in revs:
                check_compact(e, cur, st, s, t, r)
                for to in timeouts:
                    if to:
                        check_compact(e, cur, st, s, t, r, timeout_rev=to, support_ttl=False)
                e.set_compact_revision(None)


def _prefix_store():
    """user keys that are prefixes of each other, with '$' and bytes below it inside them: deleting or inserting one
    record changes the LCP of the record behind it"""
    uks = [b"a", b"a$", b"a$$", b"a#", b"a\x00", b"a\x00$", b"a/b", b"a/b$x", b"a/b#", b"ab", b"a" + b"x" * 40,
           b"a" + b"x" * 40 + b"$", b"b", b"b/events/x", b"b/events/x$"]
    items = {}
    for j, uk in enumerate(uks):
        for rev in (10 + j, 30 + j, 50 + j):
            items[_ik(uk, rev)] = b"v%d" % rev
        items[_ik(uk, 0)] = struct.pack(">Q", 50 + j)
    return items


def test_predecessor_changes(engines):
    written, _ = engines
    items = _prefix_store()
    written.load_sorted(PackedStore.from_items(list(items.items())))
    revs = (5, 20, 35, 60, 2**62)
    check_all(engines, items, revs)
    keys = sorted(items)
    batches = [
        # delete single records: the record behind each gets a new predecessor
        [(keys[5], None), (keys[17], None), (keys[40], None)],
        # delete a run of records, so the survivor behind it skips several
        [(k, None) for k in sorted(items)[20:26]],
        # inserts in front of existing records: a version between two others, a user key that sorts between two
        [(_ik(b"a$", 20), b"new"), (_ik(b"a\x00", 1), b"x"), (_ik(b"a$#", 40), b"y"), (_ik(b"a/", 33), TOMB)],
        # inserts and deletes landing on the same place
        [(sorted(items)[10], None), (sorted(items)[10][:-8] + struct.pack(">Q", 1), b"in front")],
        # several inserts in front of the same record
        [(_ik(b"a/b", r), b"z") for r in (1, 2, 3, 4)] + [(_ik(b"a/a", 9), b"q")],
    ]
    for n, ops in enumerate(batches):
        written.apply_batch(ops)
        _apply(items, ops)
        check_all(engines, items, revs, touched=[op[0] for op in ops], seed=n)


def test_value_rewrites(engines):
    """replacements that turn values into the tombstone literal and back; revision-record values whose revision moves
    across the read and compact revisions; /events/ keys under the TTL sweep"""
    written, _ = engines
    items = _prefix_store()
    written.load_sorted(PackedStore.from_items(list(items.items())))
    revs = (20, 35, 45, 2**62)
    timeouts = (25, 55)
    ev = [k for k in sorted(items) if b"/events/" in k]
    tomb_keys = [k for k in sorted(items) if k[-8:] != b"\x00" * 8][::4]
    revrec = [k for k in sorted(items) if k[-8:] == b"\x00" * 8]
    batches = [
        [(k, TOMB) for k in tomb_keys],
        [(k, b"back to a value") for k in tomb_keys[::2]] + [(k, b"tombstonf") for k in tomb_keys[1::2]],
        [(k, struct.pack(">Q", 40)) for k in revrec[::2]] + [(k, struct.pack(">Q", 40) + b"\x00") for k in revrec[1::2]],
        [(k, struct.pack(">Q", 2**40)) for k in revrec[::3]] + [_ttl_safe((k, b"short")) for k in revrec[1::3]],
        [(k, struct.pack(">Q", 20) + b"\x01") for k in revrec],
        [(k, struct.pack(">Q", r) + b"\x00") for k, r in zip(ev, (10, 30, 60, 90))],
        [(k, TOMB) for k in ev] + [(_ik(b"b/events/y", 5), b"e1"), (_ik(b"b/events/y", 0), struct.pack(">Q", 70))],
    ]
    for n, ops in enumerate(batches):
        written.apply_batch(ops)
        _apply(items, ops)
        check_all(engines, items, revs, touched=[op[0] for op in ops], timeouts=timeouts, seed=n)


def test_record_zero(engines):
    written, _ = engines
    items = _prefix_store()
    written.load_sorted(PackedStore.from_items(list(items.items())))
    revs = (5, 35, 2**62)
    for n in range(3):  # delete record 0 (the new first record loses its predecessor)
        k0 = min(items)
        written.apply_batch([(k0, None)])
        _apply(items, [(k0, None)])
        check_all(engines, items, revs, touched=[min(items)], seed=n)
    for n, k in enumerate([MAGIC + b"0$" + b"\x00" * 8, MAGIC + b"!", b"\x01"]):  # insert in front of record 0
        written.apply_batch([(k, b"first")])
        _apply(items, [(k, b"first")])
        check_all(engines, items, revs, touched=sorted(items)[:2], seed=n)
    ops = [(min(items), None), (b"\x00\x01", TOMB)]  # both at once
    written.apply_batch(ops)
    _apply(items, ops)
    check_all(engines, items, revs, touched=sorted(items)[:2])


@pytest.mark.parametrize("seed", range(3))
def test_random_batches(engines, tmp_path, seed):
    """random batches of all the above over the fuzz stores, through a layout compaction and a dump / restore (the
    restored engine then takes the remaining batches)"""
    written, fresh = engines
    rng = random.Random(seed)
    store = fuzz.fuzz_store(500 + seed, n_keys=120)
    items = dict(zip(store.keys.tolist(), store.vals.tolist()))
    written.load_sorted(store)
    revs = (0, 15, 30, 45, 2**64 - 1)
    timeouts = (20, 50)
    uks = sorted({k[4:-9] for k in items if k.startswith(MAGIC) and len(k) >= 13})
    cur_eng = written
    restored = None
    for rnd in range(8):
        keys = sorted(items)
        ops = []
        for _ in range(rng.randint(1, 40)):
            r = rng.random()
            if r < 0.25 and keys:
                ops.append((rng.choice(keys), None))
            elif r < 0.45 and keys:
                k = rng.choice(keys)
                ops.append((k, rng.choice([TOMB, b"", b"x" * rng.randint(1, 400), struct.pack(">Q", rng.randint(0, 60)),
                                           struct.pack(">Q", rng.randint(0, 60)) + b"\x00"])))
            elif r < 0.8:
                uk = rng.choice(uks) + rng.choice([b"", b"$", b"#", b"\x00", b"/events/", b"a"])
                ops.append((_ik(uk, rng.randint(0, 60)), rng.choice([TOMB, b"v", struct.pack(">Q", rng.randint(1, 60))])))
            else:
                k = rng.choice([MAGIC + b"\x00", b"\x00" + bytes([rng.randrange(256)]), b"\xff\xfe",
                                MAGIC + rng.choice(uks) + b"%" + b"\x00" * 8])
                ops.append((k, b"junk"))
        ops = [_ttl_safe(op) for op in ops]
        cur_eng.apply_batch(ops)
        _apply(items, ops)
        if rnd == 4:  # records are out of place: the dump compacts the layout first, the copy restores from the file
            path = str(tmp_path / "snap.kb")
            cur_eng.dump(path)
            restored = Engine(0)
            restored.restore(path)
            cur_eng = restored
        check_all((cur_eng, fresh), items, revs, touched=[op[0] for op in ops], timeouts=timeouts, seed=rnd)
    if restored is not None:
        restored.close()
