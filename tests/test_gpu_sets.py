"""The sets read back out of the device (include/ctmr.h, "the sets read back"): list, members, canonical export and
import, against the reference model on top of the CPU oracle (tests/sets_model.py), across shapes (single ctx, groups,
peer processes) and table sizes."""
import os
import sys

import numpy as np
import pytest

from conftest import NOW_NS, NOW_SEC, ROOT, pack
from sets_model import SetsModel, issuer_digests

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    from ct_mapreduce_b200 import build, engine
    build.build()
    return engine


def _gpu_shapes():
    import torch
    shapes = [[0, 0, 0]]
    if torch.cuda.device_count() >= 2:
        shapes.append(list(range(min(torch.cuda.device_count(), 8))))
    return shapes


def _batches(ora, golden, n=8000):
    """Two batches with twins inside and across them, the golden certificates and serials of 20..64 octets (the ones
    above 39 never enter a set)."""
    from test_oracle_properties import _cert_with_times
    cfg = ora.synth_cfg(n, dup_mode=1)
    blob, offs, idx = ora.synth_corpus(cfg, 0, n)
    iblob, ioffs = ora.synth_issuers(cfg)
    synth = [blob[int(offs[i]):int(offs[i + 1])].tobytes() for i in range(n)]
    issuers = [iblob[int(ioffs[k]):int(ioffs[k + 1])].tobytes() for k in range(len(ioffs) - 1)]
    longs = [_cert_with_times(b"900101000000Z", b"300615123045Z", serial=bytes([1]) + bytes([(m * 7 + 3) & 0xFF]) * (m - 1))
             for m in (20, 39, 40, 64)]
    extra = len(issuers)
    issuers.append(longs[0])
    gold = [fx["der"] for fx in golden.values()]
    h = n // 2
    a_ders = synth[:h] + gold + longs
    a_idx = list(idx[:h]) + [extra] * (len(gold) + len(longs))
    b_ders = synth[h:] + longs + synth[:40]
    b_idx = list(idx[h:]) + [extra] * len(longs) + list(idx[:40])
    ib, io = pack(issuers)
    out = []
    for ders, ii in ((a_ders, a_idx), (b_ders, b_idx)):
        bl, of = pack(ders)
        out.append((bl, of, ib, io, np.array(ii, np.uint32)))
    return out


KW = dict(issuer_cn_filter=b"", log_expired_entries=True, max_issuers=1024, pair_capacity_log2=16)


def _same_export(got, want):
    assert got.next_index == want.next_index
    assert np.array_equal(got.sets, want.sets), (got.sets.size, want.sets.size)
    assert np.array_equal(got.first_index, want.first_index)
    assert np.array_equal(got.serial_off, want.serial_off) and np.array_equal(got.serials, want.serials)
    assert got.tobytes() == want.tobytes()


def _fill(db, model, batches, flags=0, preload=True):
    """Batch A, a preload (new serials and one already known), batch B; db outputs checked against the model."""
    A, B = batches
    ra = db.store_batch(*A, NOW_NS, want_sha=not flags)
    _, na = model.process(*A, NOW_NS)
    assert np.array_equal(ra.was_unknown, na)
    if preload:
        d = issuer_digests(model.ora, A[2], A[3])[0]
        hour = NOW_SEC // 3600 + 24 * 400
        serials = [b"\x7f\x01", b"\x7f\x02", b"\x7f\x01"]
        db.preload_known(hour, d, serials)
        model.preload(hour, d, serials)
    rb = db.store_batch(*B, NOW_NS, want_sha=not flags)
    _, nb = model.process(*B, NOW_NS)
    assert np.array_equal(rb.was_unknown, nb)
    return ra, rb


@pytest.mark.parametrize("flags", [0, 1])   # 1 = CTMR_F_NO_FINGERPRINT: the light map kernel fills the table
def test_export_list_known_match_the_model(eng, ora, golden, flags):
    batches = _batches(ora, golden)
    model = SetsModel(ora, b"", True)
    with eng.GpuCertDatabase(table_capacity=1 << 15, flags=flags, **KW) as db:
        _fill(db, model, batches, flags)
        ex = db.export_sets()
        want = model.export()
        _same_export(ex, want)
        assert ex.sets.size > 50 and ex.n_members < model.next_index
        # serials above 39 octets never appear
        assert all(int(ex.serial_off[k + 1] - ex.serial_off[k]) <= 39 for k in range(ex.n_members))
        # list_sets over an hour range = the filtered model list
        hours = sorted({int(h) for h in ex.sets["exp_hour"]})
        lo, hi = hours[len(hours) // 4], hours[3 * len(hours) // 4]
        ls = db.list_sets(lo, hi)
        assert [(bytes(s["issuer_digest"]), int(s["exp_hour"]), int(s["count"])) for s in ls] == model.list_sets(lo, hi)
        assert np.array_equal(db.list_sets(), ex.sets)
        # Known() of a few sets, and cardinalities
        for j in (0, ex.sets.size // 2, ex.sets.size - 1):
            d, h = bytes(ex.sets[j]["issuer_digest"]), int(ex.sets[j]["exp_hour"])
            assert db.get_known_certificates(h, d).known() == [s for s, _ in model.members(h, d)]
            ser, fi = db.set_members(h, d)
            assert fi.tolist() == [f for _, f in model.members(h, d)]
            assert db.get_known_certificates(h, d).count() == len(ser)
        ser, fi = db.set_members(hours[0], b"\x00" * 32)   # an issuer the ctx never saw
        assert ser == [] and fi.size == 0


def test_export_after_eviction(eng, ora, golden):
    batches = _batches(ora, golden)
    model = SetsModel(ora, b"", True)
    with eng.GpuCertDatabase(table_capacity=1 << 15, **KW) as db:
        _fill(db, model, batches)
        before = db.export_sets()
        hours = sorted({int(h) for h in before.sets["exp_hour"]})
        cut = hours[len(hours) // 2] * 3600
        assert db.evict_expired(cut) > 0
        model.evict_expired(cut)
        after = db.export_sets()
        _same_export(after, model.export())
        assert after.sets.size < before.sets.size and (after.sets["exp_hour"] * 3600 > cut).all()
        keep = [j for j in range(before.sets.size) if int(before.sets[j]["exp_hour"]) * 3600 > cut]
        assert [before.members(j) for j in keep] == [after.members(j) for j in range(after.sets.size)]


def _owner_check(grp, shard_exports):
    from test_sharded_gloo import key_owner
    dense = {grp.issuer_digest(k): k for k in range(int(grp._lib.ctmr_issuer_count(grp.members[0]._h)))}
    W = len(shard_exports)
    for r, part in enumerate(shard_exports):
        for s in part.sets:
            assert key_owner(int(s["exp_hour"]), dense[bytes(s["issuer_digest"])], W) == r


def test_export_is_independent_of_the_shape(eng, ora, golden):
    batches = _batches(ora, golden)
    model = SetsModel(ora, b"", True)
    with eng.GpuCertDatabase(table_capacity=1 << 15, **KW) as db:
        _fill(db, model, batches)
        single = db.export_sets()
    _same_export(single, model.export())
    for devices in _gpu_shapes():
        m2 = SetsModel(ora, b"", True)
        grp = eng.GpuCertGroup(devices, table_capacity=1 << 14, **KW)
        try:
            _fill(grp, m2, batches)
            _same_export(grp.export_sets(), single)
            parts = [m.export_sets() for m in grp.members]
            assert sum(p.sets.size for p in parts) == single.sets.size
            _owner_check(grp, parts)
            _same_export(eng.SetExport.merge(parts), single)
            ls = grp.list_sets()
            assert np.array_equal(ls, single.sets)
            j = single.sets.size // 3
            d, h = bytes(single.sets[j]["issuer_digest"]), int(single.sets[j]["exp_hour"])
            assert grp.get_known_certificates(h, d).known() == [s for s, _ in single.members(j)]
        finally:
            grp.close()


def test_round_trip_into_other_shapes_then_continue(eng, ora, golden):
    from ct_mapreduce_b200 import capi
    A, B = _batches(ora, golden)
    model = SetsModel(ora, b"", True)
    src = eng.GpuCertDatabase(table_capacity=1 << 15, **KW)
    src.store_batch(*A, NOW_NS)
    model.process(*A, NOW_NS)
    ex = src.export_sets()
    _same_export(ex, model.export())
    targets = [eng.GpuCertDatabase(table_capacity=1 << 17, **KW), eng.GpuCertGroup([0, 0], table_capacity=1 << 15, **KW),
               eng.GpuCertGroup([0, 0, 0], table_capacity=1 << 15, **KW)]
    if len(_gpu_shapes()) > 1:
        targets.append(eng.GpuCertGroup(_gpu_shapes()[1], table_capacity=1 << 15, **KW))
    try:
        for t in targets:
            t.import_sets(ex)
            _same_export(t.export_sets(), ex)
        # the next batch on source, targets and the model continuing
        model.process(*B, NOW_NS)
        r_src = src.store_batch(*B, NOW_NS)
        ex2 = src.export_sets()
        _same_export(ex2, model.export())
        counts = {k: v for k, v in src.issuer_counts().items() if v}
        for t in targets:
            r = t.store_batch(*B, NOW_NS)
            for f in ("status", "was_unknown", "first_issuer_hour"):
                assert np.array_equal(getattr(r, f), getattr(r_src, f)), f
            assert {k: v for k, v in t.issuer_counts().items() if v} == counts
            _same_export(t.export_sets(), ex2)
        # refused: a non-empty target, a member of an in-process group
        with pytest.raises(capi.CtmrError):
            targets[0].import_sets(ex)
        fresh = eng.GpuCertGroup([0, 0], table_capacity=1 << 14, **KW)
        try:
            with pytest.raises(capi.CtmrError):
                fresh.members[0].import_sets(ex)
        finally:
            fresh.close()
        bad = eng.SetExport(ex.next_index, ex.sets, ex.serials, ex.serial_off.copy(), ex.first_index)
        bad.serial_off[1] = bad.serial_off[0]   # an empty serial
        with eng.GpuCertDatabase(table_capacity=1 << 15, **KW) as empty:
            with pytest.raises(capi.CtmrError):
                empty.import_sets(bad)
    finally:
        for t in targets:
            t.close()
        src.close()


def _peer_worker(rank, world, port, export, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, ROOT)
    try:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(0)
        dist.init_process_group("gloo", rank=rank, world_size=world)
        from ct_mapreduce_b200 import engine, sharded
        db = engine.GpuCertDatabase(device=0, table_capacity=1 << 15, max_issuers=1024, max_batch_entries=1500)
        sharded.attach_peers(db)
        dist.barrier()
        db.import_sets(engine.SetExport(*export))   # every rank gets the full export and keeps its own sets
        dist.barrier()
        part = db.export_sets()
        dense = {db.issuer_digest(k): k for k in range(int(db._lib.ctmr_issuer_count(db._h)))}
        dist.barrier()
        q.put((rank, (part.next_index, part.sets, part.serials, part.serial_off, part.first_index), dense, None))
        dist.barrier()
        db.close()
        dist.destroy_process_group()
    except Exception:
        import traceback
        q.put((rank, None, None, traceback.format_exc()))
        raise


@pytest.mark.timeout(600)
def test_peer_ranks_import_their_own_sets(eng, ora, golden):
    import torch.multiprocessing as mp
    from test_gpu_group import _free_port
    from test_sharded_gloo import key_owner
    batches = _batches(ora, golden, 4000)
    model = SetsModel(ora, b"", True)
    for b in batches:
        model.process(*b, NOW_NS)
    full = model.export()
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    args = (full.next_index, full.sets, full.serials, full.serial_off, full.first_index)
    procs = [ctx.Process(target=_peer_worker, args=(r, world, port, args, q)) for r in range(world)]
    for p in procs:
        p.start()
    outs = {}
    for _ in range(world):
        rank, part, dense, err = q.get(timeout=500)
        assert err is None, err
        outs[rank] = (eng.SetExport(*part), dense)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    parts = [outs[r][0] for r in range(world)]
    assert all(p.sets.size for p in parts)
    for r in range(world):
        for s in parts[r].sets:
            assert key_owner(int(s["exp_hour"]), outs[r][1][bytes(s["issuer_digest"])], world) == r
    _same_export(eng.SetExport.merge(parts), full)


@pytest.mark.timeout(900)
def test_full_scale_group_round_trip():
    """1 M entries (twins across batches) through a 3-shard group: members = new entries, every set's member count = its
    cardinality, and the round trip into a single ctx re-exports byte-identically."""
    import torch
    from ct_mapreduce_b200 import capi, engine
    n, parts = 1_000_000, 4
    cfg = capi.synth_cfg(n, len_mode=1, len_lo=400, len_hi=900, dup_mode=1)
    iblob, ioffs = engine.synth_issuers(cfg)
    grp = engine.GpuCertGroup([0, 0, 0], table_capacity=1 << 20, issuer_cn_filter=b"", log_expired_entries=True, max_issuers=1024)
    try:
        new = 0
        step = n // parts
        for k in range(parts):
            blob, offsets, idx, total = engine.synth_corpus_device(cfg, k * step, step, torch.device("cuda:0"))
            b, o, i = blob[:total].cpu().numpy(), offsets.cpu().numpy().astype(np.uint64), idx.cpu().numpy().astype(np.uint32)
            r = grp.store_batch(b, o, iblob, ioffs, i, NOW_NS, want_sha=False)
            new += int(r.was_unknown.sum())
        ex = grp.export_sets()
        assert ex.n_members == new and ex.next_index == n
        assert int(ex.sets["count"].sum()) == new
        for j in range(0, ex.sets.size, max(1, ex.sets.size // 50)):
            s = ex.sets[j]
            assert grp.get_known_certificates(int(s["exp_hour"]), bytes(s["issuer_digest"])).count() == int(s["count"])
        with engine.GpuCertDatabase(table_capacity=1 << 21, max_issuers=1024) as one:
            one.import_sets(ex)
            _same_export(one.export_sets(), ex)
    finally:
        grp.close()


def test_too_small_buffers_report_the_sizes(eng, ora, golden):
    """NULL buffers: sizes only.  Buffers one short: CTMR_E_BATCH_TOO_LARGE, the sizes still reported."""
    import ctypes as C
    from ct_mapreduce_b200 import capi
    A, _ = _batches(ora, golden, 3000)
    with eng.GpuCertDatabase(table_capacity=1 << 15, **KW) as db:
        db.store_batch(*A, NOW_NS)
        L, h = db._lib, db._h
        full = db.export_sets()
        lo, hi = -(1 << 63), (1 << 63) - 1
        n = C.c_uint64(0)
        assert L.ctmr_list_sets(h, lo, hi, None, 0, C.byref(n)) == 0 and n.value == full.sets.size
        buf = np.zeros(full.sets.size, capi.SET_INFO_DTYPE)
        n = C.c_uint64(0)
        assert L.ctmr_list_sets(h, lo, hi, capi.ptr(buf), full.sets.size - 1, C.byref(n)) == capi.E_BATCH_TOO_LARGE
        assert n.value == full.sets.size
        j = int(np.argmax(full.sets["count"]))
        s = full.sets[j]
        cnt = int(s["count"])
        assert cnt >= 2
        d = (C.c_uint8 * 32).from_buffer_copy(bytes(s["issuer_digest"]))
        blob, off, first = np.zeros(39 * cnt, np.uint8), np.zeros(cnt + 1, np.uint64), np.zeros(cnt, np.uint64)
        n = C.c_uint64(0)
        rc = L.ctmr_set_members(h, int(s["exp_hour"]), d, capi.ptr(blob), blob.size, capi.ptr(off), capi.ptr(first), cnt - 1, C.byref(n))
        assert rc == capi.E_BATCH_TOO_LARGE and n.value == cnt
        x = capi.SetExport()
        assert L.ctmr_export_sets(h, C.byref(x)) == 0
        assert (x.n_sets, x.n_members, x.serial_bytes, x.next_index) == (full.sets.size, full.n_members, full.serials.size, full.next_index)
        sets = np.zeros(full.sets.size, capi.SET_INFO_DTYPE)
        ser, off, first = np.zeros(full.serials.size, np.uint8), np.zeros(full.n_members + 1, np.uint64), np.zeros(full.n_members, np.uint64)
        for short in ("sets", "serials", "members"):
            x = capi.SetExport()
            x.sets, x.sets_cap = capi.ptr(sets), sets.size - (short == "sets")
            x.serials, x.serials_cap = capi.ptr(ser), ser.size - (short == "serials")
            x.serial_off, x.first_index, x.members_cap = capi.ptr(off), capi.ptr(first), full.n_members - (short == "members")
            assert L.ctmr_export_sets(h, C.byref(x)) == capi.E_BATCH_TOO_LARGE, short
            assert (x.n_sets, x.n_members, x.serial_bytes) == (full.sets.size, full.n_members, full.serials.size), short


def _peer_batch_worker(rank, world, port, batch, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, ROOT)
    try:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(0)
        dist.init_process_group("gloo", rank=rank, world_size=world)
        from ct_mapreduce_b200 import engine, sharded
        db = engine.GpuCertDatabase(device=0, table_capacity=1 << 15, max_batch_entries=PEER_E, **KW)
        sharded.attach_peers(db)
        dist.barrier()
        db.store_batch(*batch, NOW_NS)           # collective: one round, rank r's entry j at global index r * E + j
        dist.barrier()
        part = db.export_sets()                  # this rank's own sets, not collective
        dense = {db.issuer_digest(k): k for k in range(int(db._lib.ctmr_issuer_count(db._h)))}
        dist.barrier()
        q.put((rank, (part.next_index, part.sets, part.serials, part.serial_off, part.first_index), dense, None))
        dist.barrier()
        db.close()
        dist.destroy_process_group()
    except Exception:
        import traceback
        q.put((rank, None, None, traceback.format_exc()))
        raise


PEER_E = 4096


@pytest.mark.timeout(600)
def test_peer_ranks_export_their_shards_after_peer_batches(eng, ora):
    """State built by the peer data path (two processes, one GPU): every rank exports its own shard; the merge equals a
    single ctx over the same entries in the order the peer path defines (rank 0's batch, then rank 1's), with rank 1's
    first indices at E + j instead of n0 + j."""
    import torch.multiprocessing as mp
    from test_gpu_group import _free_port
    from test_sharded_gloo import key_owner
    n0, n1 = 3000, 2500
    cfg = ora.synth_cfg(n0 + n1, dup_mode=1)
    blob, offs, idx = ora.synth_corpus(cfg, 0, n0 + n1)
    iblob, ioffs = ora.synth_issuers(cfg)
    batches = [(blob, offs[:n0 + 1], iblob, ioffs, idx[:n0]), (blob, offs[n0:], iblob, ioffs, idx[n0:])]
    with eng.GpuCertDatabase(table_capacity=1 << 15, **KW) as one:
        for b in batches:
            one.store_batch(*b, NOW_NS)
        single = one.export_sets()
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_peer_batch_worker, args=(r, world, port, batches[r], q)) for r in range(world)]
    for p in procs:
        p.start()
    outs = {}
    for _ in range(world):
        rank, part, dense, err = q.get(timeout=500)
        assert err is None, err
        outs[rank] = (eng.SetExport(*part), dense)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    parts = [outs[r][0] for r in range(world)]
    assert all(p.sets.size for p in parts)
    for r in range(world):
        for s in parts[r].sets:
            assert key_owner(int(s["exp_hour"]), outs[r][1][bytes(s["issuer_digest"])], world) == r
    fi = single.first_index.astype(np.int64)
    want = eng.SetExport(world * PEER_E, single.sets, single.serials, single.serial_off,
                         np.where(fi < n0, fi, fi - n0 + PEER_E).astype(np.uint64))
    _same_export(eng.SetExport.merge(parts), want)
