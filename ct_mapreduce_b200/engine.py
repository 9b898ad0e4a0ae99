"""Host-side mirror of the reference interface for the CT map/reduce path, over the C ABI.

The reference is Go (no toolchain in this image), so this module plays the part the Go shim plays
in production (INTEGRATION.md): it packs batches, calls libctmr through the very same C entry
points, and exposes the results under the reference's names:

    GpuCertDatabase.store_batch        <- insertCTWorker loop body + FilesystemDatabase.Store
                                          (cmd/ct-fetch/ct-fetch.go:191-245, storage/filesystemdatabase.go:158-211)
    GpuCertDatabase.get_known_certificates(exp_hour, issuer).count()
                                       <- KnownCertificates.Count (storage/knowncertificates.go:57-63)
    GpuCertDatabase.issuer_counts      <- the per-issuer sum of cmd/storage-statistics/storage-statistics.go:44-53
    GpuCertDatabase.status_counters    <- metrics certIsFilteredOut.{CA,expired,cn-filtered}, insertCTWorker.Inserted
    GpuCertDatabase.list_sets          <- GetIssuerAndDatesFromCache + Count() (storage/filesystemdatabase.go:59-100)
    GpuCertDatabase.get_known_certificates(exp_hour, issuer).known()
                                       <- KnownCertificates.Known (storage/knowncertificates.go:65-96)
    GpuCertDatabase.export_sets / import_sets
                                       <- the Redis state in canonical form, portable across table sizes and group sizes

All arithmetic happens in the CUDA kernels; nothing here parses, hashes or de-duplicates.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import capi
from .capi import CtmrError


@dataclass
class BatchResult:
    """Per-entry outputs of one batch (numpy arrays in host memory)."""
    status: np.ndarray
    sha256: np.ndarray | None
    exp_hour: np.ndarray
    serial_off: np.ndarray
    serial_len: np.ndarray
    was_unknown: np.ndarray
    first_issuer_hour: np.ndarray
    # IssuerMetadata string reducers (only filled by store_batch(..., want_meta=True))
    issuer_name_off: np.ndarray | None = None
    issuer_name_len: np.ndarray | None = None
    crldp_off: np.ndarray | None = None
    crldp_len: np.ndarray | None = None
    first_issuer_dn: np.ndarray | None = None
    first_crldp: np.ndarray | None = None
    # PEM of the new certificates (want_pem=True): texts back to back, entry i = pem[pem_off[i]:pem_off[i+1]]
    pem: np.ndarray | None = None
    pem_off: np.ndarray | None = None

    def pem_of(self, i: int) -> bytes:
        return self.pem[int(self.pem_off[i]):int(self.pem_off[i + 1])].tobytes()


class KnownCertificatesView:
    """Read side of storage.KnownCertificates for one (expDate, issuer) (knowncertificates.go:57-63)."""

    def __init__(self, db: "GpuCertDatabase", exp_hour: int, issuer_digest: bytes):
        self._db, self.exp_hour, self.issuer_digest = db, int(exp_hour), bytes(issuer_digest)

    def count(self) -> int:
        out = C.c_uint64(0)
        d = (C.c_uint8 * 32).from_buffer_copy(self.issuer_digest)
        self._db._check(self._db._lib.ctmr_set_cardinality(self._db._h, self.exp_hour, d, C.byref(out)))
        return out.value

    def known(self) -> list:
        """The set's serials (raw octets), in first-seen order (KnownCertificates.Known, knowncertificates.go:65-96)."""
        return self._db.set_members(self.exp_hour, self.issuer_digest)[0]


@dataclass
class SetExport:
    """Canonical export of the known-certificate sets (include/ctmr.h, "the sets read back"): sets by (issuer digest,
    exp_hour), members of a set by first index.  Member k of set j: serials[serial_off[k]:serial_off[k+1]], first_index[k],
    for k in [sets[j]["member_off"], sets[j]["member_off"] + sets[j]["count"])."""
    next_index: int
    sets: np.ndarray         # capi.SET_INFO_DTYPE [n_sets]
    serials: np.ndarray      # uint8 [serial_bytes]
    serial_off: np.ndarray   # uint64 [n_members + 1]
    first_index: np.ndarray  # uint64 [n_members]

    @property
    def n_members(self) -> int:
        return int(self.first_index.size)

    def members(self, j: int):
        """[(serial bytes, first index)] of set j."""
        lo = int(self.sets[j]["member_off"])
        return [(self.serials[int(self.serial_off[k]):int(self.serial_off[k + 1])].tobytes(), int(self.first_index[k]))
                for k in range(lo, lo + int(self.sets[j]["count"]))]

    def tobytes(self) -> bytes:
        """Every array back to back: equal exports are equal byte strings."""
        return b"".join([np.uint64(self.next_index).tobytes(), self.sets.tobytes(), self.serials.tobytes(),
                         np.ascontiguousarray(self.serial_off, np.uint64).tobytes(),
                         np.ascontiguousarray(self.first_index, np.uint64).tobytes()])

    def __eq__(self, other) -> bool:
        return isinstance(other, SetExport) and self.tobytes() == other.tobytes()

    @staticmethod
    def merge(parts) -> "SetExport":
        """The exports of the shards of one group (disjoint sets) -> the group's export, canonical order."""
        parts = list(parts)
        order = sorted((bytes(p.sets[j]["issuer_digest"]), int(p.sets[j]["exp_hour"]), i, j)
                       for i, p in enumerate(parts) for j in range(p.sets.size))
        sets = np.zeros(len(order), capi.SET_INFO_DTYPE)
        serials, first, lens, run = [], [], [], 0
        for out_j, (_, _, i, j) in enumerate(order):
            sets[out_j] = parts[i].sets[j]
            sets[out_j]["member_off"] = run
            for ser, fi in parts[i].members(j):
                serials.append(ser)
                first.append(fi)
                lens.append(len(ser))
            run += int(parts[i].sets[j]["count"])
        off = np.zeros(len(lens) + 1, np.uint64)
        off[1:] = np.cumsum(lens, dtype=np.uint64)
        return SetExport(max([p.next_index for p in parts] or [0]), sets, np.frombuffer(b"".join(serials), np.uint8).copy(), off,
                         np.array(first, np.uint64))


def _attach_pem(o: "capi.Out", res: BatchResult, n: int, der_bytes: int):
    """Room for the PEM of every certificate of the batch (the worst case: all new)."""
    res.pem = np.zeros(der_bytes // 3 * 4 + der_bytes // 48 + 64 * n + 256, np.uint8)
    res.pem_off = np.zeros(n + 1, np.uint64)
    o.pem, o.pem_cap, o.pem_off = capi.ptr(res.pem), res.pem.size, capi.ptr(res.pem_off)


class RawBatchResult:
    """Outputs of ctmr_process_raw (ctmr_raw_out): the path's outputs plus what the wire format carried."""

    def __init__(self, n: int, want_sha: bool = True, want_meta: bool = False):
        self.path = BatchResult(np.zeros(n, np.uint8), np.zeros((n, 32), np.uint8) if want_sha else None, np.zeros(n, np.int64),
                                np.zeros(n, np.uint32), np.zeros(n, np.uint32), np.zeros(n, np.uint8), np.zeros(n, np.uint8))
        if want_meta:
            p = self.path
            p.issuer_name_off, p.issuer_name_len = np.zeros(n, np.uint32), np.zeros(n, np.uint32)
            p.crldp_off, p.crldp_len = np.zeros(n, np.uint32), np.zeros(n, np.uint32)
            p.first_issuer_dn, p.first_crldp = np.zeros(n, np.uint8), np.zeros(n, np.uint8)
        self.entry_status = np.zeros(n, np.uint8)
        self.entry_type = np.zeros(n, np.uint8)
        self.timestamp_ms = np.zeros(n, np.uint64)
        self.issuer = np.zeros(n, np.uint32)
        self.leaf_src = np.zeros(n, np.uint8)
        self.leaf_off = np.zeros(n, np.uint32)
        self.leaf_len = np.zeros(n, np.uint32)


class GpuCertDatabase:
    """One ctmr_ctx = one GPU's share of the known-certificate state."""

    _SETS = "ctmr_"   # prefix of the set read-back entry points this handle takes

    def __init__(self, device: int = 0, table_capacity: int = 1 << 22, issuer_cn_filter: bytes | str = b"",
                 log_expired_entries: bool = False, flags: int = 0, max_issuers: int = 0, max_batch_entries: int = 0,
                 max_batch_bytes: int = 0, pair_capacity_log2: int = 0, meta_capacity_log2: int = 0, max_round_entries: int = 0,
                 _adopt=None):
        self._lib = capi.load()
        if _adopt is not None:  # a member of a GpuCertGroup: the group owns the handle
            self._h, self.device, self.flags, self._owned = _adopt, device, flags, False
            return
        self._owned = True
        if isinstance(issuer_cn_filter, str):
            issuer_cn_filter = issuer_cn_filter.encode()
        self._filter = bytes(issuer_cn_filter)
        cfg = capi.Config()
        cfg.struct_size = C.sizeof(capi.Config)
        cfg.device = device
        cfg.table_capacity = table_capacity
        cfg.max_batch_entries = max_batch_entries
        cfg.max_batch_bytes = max_batch_bytes
        cfg.max_issuers = max_issuers
        cfg.pair_capacity_log2 = pair_capacity_log2
        cfg.meta_capacity_log2 = meta_capacity_log2
        cfg.max_round_entries = max_round_entries
        cfg.issuer_cn_filter = self._filter
        cfg.issuer_cn_filter_len = len(self._filter)
        cfg.log_expired_entries = int(bool(log_expired_entries))
        cfg.flags = flags
        h = C.c_void_p()
        rc = self._lib.ctmr_create(C.byref(cfg), C.byref(h))
        if rc != 0:
            raise CtmrError(rc, (self._lib.ctmr_last_error(None) or b"").decode())
        self._h = h
        self.device = device
        self.flags = flags

    # ------------------------------------------------------------------ plumbing
    def _check(self, rc: int):
        if rc != 0:
            raise CtmrError(rc, (self._lib.ctmr_last_error(self._h) or b"").decode())

    def close(self):
        if getattr(self, "_h", None):
            if getattr(self, "_owned", True):
                self._lib.ctmr_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def handle(self):
        return self._h

    # ------------------------------------------------------------------ issuers
    def register_issuers(self, issuer_blob: np.ndarray, issuer_offsets: np.ndarray) -> np.ndarray:
        """NewIssuer(x509.ParseCertificate(Chain[0])) for each certificate -> dense indices."""
        issuer_blob = np.ascontiguousarray(issuer_blob, np.uint8)
        issuer_offsets = np.ascontiguousarray(issuer_offsets, np.uint64)
        n = issuer_offsets.size - 1
        out = np.zeros(max(n, 1), np.uint32)
        self._check(self._lib.ctmr_register_issuers(self._h, capi.ptr(issuer_blob), capi.ptr(issuer_offsets), n, capi.ptr(out)))
        return out[:n]

    def issuer_digest(self, dense_idx: int) -> bytes:
        d = (C.c_uint8 * 32)()
        self._check(self._lib.ctmr_issuer_digest(self._h, dense_idx, d))
        return bytes(d)

    # ------------------------------------------------------------------ the hot path, host buffers
    def store_batch(self, blob, offsets, issuer_blob, issuer_offsets, issuer_idx, now_unix_ns: int,
                    want_sha: bool = True, out: BatchResult | None = None, want_meta: bool = False,
                    want_pem: bool = False) -> BatchResult:
        """One batch through ctmr_process_batch (HOST buffers in, HOST buffers out)."""
        blob = np.ascontiguousarray(blob, np.uint8)
        offsets = np.ascontiguousarray(offsets, np.uint64)
        n = offsets.size - 1
        n_iss = 0
        if issuer_offsets is not None:
            issuer_blob = np.ascontiguousarray(issuer_blob, np.uint8)
            issuer_offsets = np.ascontiguousarray(issuer_offsets, np.uint64)
            n_iss = issuer_offsets.size - 1
        if issuer_idx is not None:
            issuer_idx = np.ascontiguousarray(issuer_idx, np.uint32)
        if out is None:
            out = BatchResult(np.zeros(n, np.uint8), np.zeros((n, 32), np.uint8) if want_sha else None, np.zeros(n, np.int64),
                              np.zeros(n, np.uint32), np.zeros(n, np.uint32), np.zeros(n, np.uint8), np.zeros(n, np.uint8))
        if want_meta and out.first_issuer_dn is None:
            out.issuer_name_off, out.issuer_name_len = np.zeros(n, np.uint32), np.zeros(n, np.uint32)
            out.crldp_off, out.crldp_len = np.zeros(n, np.uint32), np.zeros(n, np.uint32)
            out.first_issuer_dn, out.first_crldp = np.zeros(n, np.uint8), np.zeros(n, np.uint8)
        o = capi.Out(capi.ptr(out.status), capi.ptr(out.sha256) if want_sha else None, capi.ptr(out.exp_hour),
                     capi.ptr(out.serial_off), capi.ptr(out.serial_len), capi.ptr(out.was_unknown),
                     capi.ptr(out.first_issuer_hour),
                     *([capi.ptr(out.issuer_name_off), capi.ptr(out.issuer_name_len), capi.ptr(out.crldp_off),
                        capi.ptr(out.crldp_len), capi.ptr(out.first_issuer_dn), capi.ptr(out.first_crldp)] if want_meta else [None] * 6))
        if want_pem:
            _attach_pem(o, out, n, int(blob.size))
        self._check(self._process_batch_fn()(self._h, capi.ptr(blob), capi.ptr(offsets), n,
                                             capi.ptr(issuer_blob) if n_iss else None,
                                             capi.ptr(issuer_offsets) if n_iss else None, n_iss,
                                             capi.ptr(issuer_idx), now_unix_ns, C.byref(o)))
        return out

    def _process_batch_fn(self):
        return self._lib.ctmr_process_batch

    # ------------------------------------------------------------------ CT wire-format front end (include/ctmr_frontend.h)
    def store_raw_entries(self, text, leaf_off, leaf_len, extra_off, extra_len, now_unix_ns: int, want_sha: bool = True,
                          want_meta: bool = False, want_pem: bool = False) -> "RawBatchResult":
        """get-entries strings (base64 leaf_input / extra_data, spans into `text`) through ctmr_process_raw:
        what GetRawEntries' JSON decode, ct.LogEntryFromLeaf (ct-fetch.go:424,452) and insertCTWorker + Store do."""
        text = np.frombuffer(text, np.uint8) if isinstance(text, (bytes, bytearray, memoryview)) else np.ascontiguousarray(text, np.uint8)
        leaf_off, extra_off = np.ascontiguousarray(leaf_off, np.uint64), np.ascontiguousarray(extra_off, np.uint64)
        leaf_len, extra_len = np.ascontiguousarray(leaf_len, np.uint32), np.ascontiguousarray(extra_len, np.uint32)
        n = leaf_off.size
        r = RawBatchResult(n, want_sha, want_meta)
        p = r.path
        o = capi.RawOut()
        o.path = capi.Out(capi.ptr(p.status), capi.ptr(p.sha256) if want_sha else None, capi.ptr(p.exp_hour), capi.ptr(p.serial_off),
                          capi.ptr(p.serial_len), capi.ptr(p.was_unknown), capi.ptr(p.first_issuer_hour),
                          *([capi.ptr(p.issuer_name_off), capi.ptr(p.issuer_name_len), capi.ptr(p.crldp_off), capi.ptr(p.crldp_len),
                             capi.ptr(p.first_issuer_dn), capi.ptr(p.first_crldp)] if want_meta else [None] * 6))
        for name in ("entry_status", "entry_type", "timestamp_ms", "issuer", "leaf_src", "leaf_off", "leaf_len"):
            setattr(o, name, capi.ptr(getattr(r, name)))
        if want_pem:
            _attach_pem(o.path, p, n, (int(leaf_len.sum()) + int(extra_len.sum())) // 4 * 3)
        b = capi.RawBatch(capi.ptr(text), text.size, capi.ptr(leaf_off), capi.ptr(leaf_len), capi.ptr(extra_off), capi.ptr(extra_len),
                          n, now_unix_ns)
        self._check(self._process_raw_fn()(self._h, C.byref(b), C.byref(o)))
        return r

    def _process_raw_fn(self):
        return self._lib.ctmr_process_raw

    def frontend_profile_last(self):
        """(frontend_ms, path_ms, frontend_launches) of the last store_raw_entries call (CUDA events inside the library)."""
        a, b, k = C.c_float(0), C.c_float(0), C.c_uint64(0)
        self._check(self._lib.ctmr_frontend_profile_last(self._h, C.byref(a), C.byref(b), C.byref(k)))
        return a.value, b.value, k.value

    # ------------------------------------------------------------------ device-resident variants (torch tensors / raw pointers)
    def map_device(self, batch: capi.DevBatch, out: capi.DevOut, stream=None):
        self._check(self._lib.ctmr_map_device(self._h, C.byref(batch), C.byref(out), stream))

    def reduce_device(self, keys, m: int, was_unknown, first_issuer_hour, stream=None):
        self._check(self._lib.ctmr_reduce_device(self._h, capi.ptr(keys), m, capi.ptr(was_unknown),
                                                 capi.ptr(first_issuer_hour), stream))

    def process_device(self, batch: capi.DevBatch, out: capi.DevOut, stream=None):
        self._check(self._lib.ctmr_process_device(self._h, C.byref(batch), C.byref(out), stream))

    def read_histogram_device(self, counts_dst, n_slots: int, status_dst=None, stream=None):
        self._check(self._lib.ctmr_read_histogram_device(self._h, capi.ptr(counts_dst), n_slots, capi.ptr(status_dst), stream))

    def profile_last(self):
        """(map_ms, total_ms) of the last process_device call, from the library's own CUDA events."""
        m, t = C.c_float(0), C.c_float(0)
        self._check(self._lib.ctmr_profile_last(self._h, C.byref(m), C.byref(t)))
        return m.value, t.value

    def sha256_ceiling(self, iters=2000, rolled=True, ctas_per_sm=2):
        """Register-only SHA-256 rate on this GPU: (GB/s of message bytes, ms)."""
        ms, blocks = C.c_float(0), C.c_uint64(0)
        self._check(self._lib.ctmr_sha256_ceiling_device(self._h, iters, int(rolled), ctas_per_sm, C.byref(ms), C.byref(blocks)))
        return blocks.value * 64 / (ms.value / 1e3) / 1e9, ms.value

    def reset_device(self, stream=None):
        self._check(self._lib.ctmr_reset_device(self._h, stream))

    def check_device(self, stream=None):
        self._check(self._lib.ctmr_check_device(self._h, stream))

    # ------------------------------------------------------------------ one process per GPU: peers over CUDA IPC (ctmr_peer_*)
    def peer_export(self, world: int) -> bytes:
        h = (C.c_uint8 * capi.PEER_HANDLE_BYTES)()
        self._check(self._lib.ctmr_peer_export(self._h, world, h))
        return bytes(h)

    def peer_attach(self, rank: int, world: int, handles: list):
        """handles[r] = rank r's peer_export().  Afterwards process_device / store_batch / reset_device are collective."""
        buf = (C.c_uint8 * (capi.PEER_HANDLE_BYTES * world)).from_buffer_copy(b"".join(handles))
        self._check(self._lib.ctmr_peer_attach(self._h, rank, world, buf))

    def peer_barrier_device(self, stream=None):
        self._check(self._lib.ctmr_peer_barrier_device(self._h, stream))

    def peer_allreduce_histogram_device(self, counts_dst, n_slots: int, status_dst=None, stream=None):
        self._check(self._lib.ctmr_peer_allreduce_histogram_device(self._h, capi.ptr(counts_dst), n_slots, capi.ptr(status_dst), stream))

    # ------------------------------------------------------------------ warm start / checkpoint (SURVEY §8(f)-4)
    def preload_known(self, exp_hour: int, issuer_digest: bytes, serials):
        """Seed one "serials::<expDate>::<issuer>" set (e.g. KnownCertificates.Known() read back from Redis)."""
        serials = [bytes(x) for x in serials]
        offs = np.zeros(len(serials) + 1, np.uint64)
        offs[1:] = np.cumsum([len(x) for x in serials], dtype=np.uint64)
        blob = np.frombuffer(b"".join(serials) or b"\0", np.uint8).copy()
        d = (C.c_uint8 * 32).from_buffer_copy(issuer_digest)
        self._check(self._lib.ctmr_preload_known(self._h, exp_hour, d, capi.ptr(blob), capi.ptr(offs), len(serials)))

    def snapshot(self) -> np.ndarray:
        need = C.c_uint64(0)
        self._check(self._lib.ctmr_snapshot_size(self._h, C.byref(need)))
        buf = np.empty(need.value, np.uint8)
        wrote = C.c_uint64(0)
        self._check(self._lib.ctmr_snapshot_save(self._h, capi.ptr(buf), buf.size, C.byref(wrote)))
        return buf[:wrote.value]

    def restore(self, snap: np.ndarray):
        snap = np.ascontiguousarray(snap, np.uint8)
        self._check(self._lib.ctmr_snapshot_load(self._h, capi.ptr(snap), snap.size))

    def evict_expired(self, now_unix_sec: int) -> int:
        """Apply the Redis TTLs (EXPIREAT(expDate) on every serials:: set, knowncertificates.go:98-104): sets with
        expDate <= now vanish.  Returns the number of serials dropped."""
        n = C.c_uint64(0)
        self._check(self._lib.ctmr_evict_expired(self._h, int(now_unix_sec), C.byref(n)))
        return int(n.value)

    # ------------------------------------------------------------------ reducers' read side
    def get_known_certificates(self, exp_hour: int, issuer_digest: bytes) -> KnownCertificatesView:
        return KnownCertificatesView(self, exp_hour, issuer_digest)

    def issuer_counts(self) -> dict:
        """{Issuer.ID digest (32 bytes): number of unique certificates} for every registered issuer."""
        n = C.c_size_t(self._lib.ctmr_issuer_count(self._h))
        cap = max(int(n.value), 1)
        dig = np.zeros((cap, 32), np.uint8)
        cnt = np.zeros(cap, np.uint64)
        self._check(self._lib.ctmr_issuer_counts(self._h, capi.ptr(dig), capi.ptr(cnt), C.byref(n)))
        return {bytes(dig[i]): int(cnt[i]) for i in range(n.value)}

    def status_counters(self) -> np.ndarray:
        out = np.zeros(capi.ST_COUNT, np.uint64)
        self._check(self._lib.ctmr_status_counters(self._h, capi.ptr(out)))
        return out

    def table_stats(self):
        used, cap = C.c_uint64(0), C.c_uint64(0)
        self._check(self._lib.ctmr_table_stats(self._h, C.byref(used), C.byref(cap)))
        return used.value, cap.value

    # ------------------------------------------------------------------ the sets read back (list, members, export / import)
    def _sets_fn(self, name):
        return getattr(self._lib, self._SETS + name)

    def list_sets(self, min_exp_hour: int | None = None, max_exp_hour: int | None = None) -> np.ndarray:
        """Live sets with min_exp_hour <= exp_hour <= max_exp_hour (None = unbounded), canonical order, as a
        capi.SET_INFO_DTYPE array (issuer_digest, exp_hour, count, member_off).  On a group member: that shard's sets."""
        lo = -(1 << 63) if min_exp_hour is None else int(min_exp_hour)
        hi = (1 << 63) - 1 if max_exp_hour is None else int(max_exp_hour)
        fn, n = self._sets_fn("list_sets"), C.c_uint64(0)
        self._check(fn(self._h, lo, hi, None, 0, C.byref(n)))
        out = np.zeros(max(n.value, 1), capi.SET_INFO_DTYPE)
        self._check(fn(self._h, lo, hi, capi.ptr(out), out.size, C.byref(n)))
        return out[:n.value]

    def set_members(self, exp_hour: int, issuer_digest: bytes):
        """(serials in first-seen order, their first indices) of one set."""
        fn, n = self._sets_fn("set_members"), C.c_uint64(0)
        d = (C.c_uint8 * 32).from_buffer_copy(bytes(issuer_digest))
        self._check(fn(self._h, int(exp_hour), d, None, 0, None, None, 0, C.byref(n)))
        cap = max(n.value, 1)
        blob, off, first = np.zeros(cap * capi.MAX_SERIAL, np.uint8), np.zeros(cap + 1, np.uint64), np.zeros(cap, np.uint64)
        self._check(fn(self._h, int(exp_hour), d, capi.ptr(blob), blob.size, capi.ptr(off), capi.ptr(first), cap, C.byref(n)))
        k = n.value
        return [blob[int(off[i]):int(off[i + 1])].tobytes() for i in range(k)], first[:k].copy()

    def export_sets(self) -> SetExport:
        """Canonical export of every live set (include/ctmr.h): portable to a ctx or group of any size."""
        fn, x = self._sets_fn("export_sets"), capi.SetExport()
        self._check(fn(self._h, C.byref(x)))
        sets = np.zeros(max(x.n_sets, 1), capi.SET_INFO_DTYPE)
        serials = np.zeros(max(x.serial_bytes, 1), np.uint8)
        off, first = np.zeros(x.n_members + 1, np.uint64), np.zeros(max(x.n_members, 1), np.uint64)
        x.sets, x.sets_cap = capi.ptr(sets), sets.size
        x.serials, x.serials_cap = capi.ptr(serials), serials.size
        x.serial_off, x.first_index, x.members_cap = capi.ptr(off), capi.ptr(first), x.n_members
        self._check(fn(self._h, C.byref(x)))
        return SetExport(int(x.next_index), sets[:x.n_sets], serials[:x.serial_bytes], off[:x.n_members + 1], first[:x.n_members])

    def import_sets(self, export: SetExport):
        """Load an export into this EMPTY ctx / group (CtmrError otherwise); members keep their first indices."""
        sets = np.ascontiguousarray(export.sets, capi.SET_INFO_DTYPE)
        serials = np.ascontiguousarray(export.serials, np.uint8)
        off, first = np.ascontiguousarray(export.serial_off, np.uint64), np.ascontiguousarray(export.first_index, np.uint64)
        keep = [np.zeros(1, np.uint8) if a.size == 0 else a for a in (sets, serials, first)]
        x = capi.SetExport(int(export.next_index), sets.size, first.size, serials.size, capi.ptr(keep[0]), sets.size,
                           capi.ptr(keep[1]), serials.size, capi.ptr(off), capi.ptr(keep[2]), first.size)
        self._check(self._sets_fn("import_sets")(self._h, C.byref(x)))


class GpuCertGroup(GpuCertDatabase):
    """Several GPUs of one box behind ONE handle (ctmr_group_*): what the Go host calls in place of the worker pool of
    StartDatabaseThreads (cmd/ct-fetch/ct-fetch.go:140-145).  Same methods, globally exact results: every set
    "serials::<expDate>::<issuer>" lives on one owner GPU and the map kernels insert into it over NVLink."""

    def __init__(self, devices, table_capacity: int = 1 << 22, issuer_cn_filter: bytes | str = b"", log_expired_entries: bool = False,
                 flags: int = 0, max_issuers: int = 0, max_batch_entries: int = 0, max_batch_bytes: int = 0,
                 pair_capacity_log2: int = 0, meta_capacity_log2: int = 0):
        self._lib = capi.load()
        if isinstance(issuer_cn_filter, str):
            issuer_cn_filter = issuer_cn_filter.encode()
        self._filter = bytes(issuer_cn_filter)
        cfg = capi.Config()
        cfg.struct_size = C.sizeof(capi.Config)
        cfg.table_capacity, cfg.max_batch_entries, cfg.max_batch_bytes = table_capacity, max_batch_entries, max_batch_bytes
        cfg.max_issuers, cfg.pair_capacity_log2, cfg.meta_capacity_log2 = max_issuers, pair_capacity_log2, meta_capacity_log2
        cfg.issuer_cn_filter, cfg.issuer_cn_filter_len = self._filter, len(self._filter)
        cfg.log_expired_entries, cfg.flags = int(bool(log_expired_entries)), flags
        devs = (C.c_int32 * len(devices))(*devices)
        h = C.c_void_p()
        rc = self._lib.ctmr_group_create(C.byref(cfg), devs, len(devices), C.byref(h))
        if rc != 0:
            raise CtmrError(rc, (self._lib.ctmr_group_last_error(None) or b"").decode())
        self._h, self._owned = h, True
        self._SETS = "ctmr_group_"
        self.devices, self.device, self.flags = list(devices), devices[0], flags
        self.members = [GpuCertDatabase(device=devices[r], flags=flags, _adopt=C.c_void_p(self._lib.ctmr_group_member(h, r)))
                        for r in range(len(devices))]

    def _check(self, rc: int):
        if rc != 0:
            raise CtmrError(rc, (self._lib.ctmr_group_last_error(self._h) or b"").decode())

    def close(self):
        if getattr(self, "_h", None):
            for m in self.members:
                m._h = None
            self._lib.ctmr_group_destroy(self._h)
            self._h = None

    def _process_batch_fn(self):
        return self._lib.ctmr_group_process_batch

    def _process_raw_fn(self):
        return self._lib.ctmr_group_process_raw

    def register_issuers(self, issuer_blob, issuer_offsets):
        return self.members[0].register_issuers(issuer_blob, issuer_offsets)   # the registry is the group's

    def issuer_digest(self, dense_idx: int) -> bytes:
        return self.members[0].issuer_digest(dense_idx)

    def preload_known(self, exp_hour: int, issuer_digest: bytes, serials):
        serials = [bytes(x) for x in serials]
        offs = np.zeros(len(serials) + 1, np.uint64)
        offs[1:] = np.cumsum([len(x) for x in serials], dtype=np.uint64)
        blob = np.frombuffer(b"".join(serials) or b"\0", np.uint8).copy()
        d = (C.c_uint8 * 32).from_buffer_copy(issuer_digest)
        self._check(self._lib.ctmr_group_preload_known(self._h, exp_hour, d, capi.ptr(blob), capi.ptr(offs), len(serials)))

    def evict_expired(self, now_unix_sec: int) -> int:
        n = C.c_uint64(0)
        self._check(self._lib.ctmr_group_evict_expired(self._h, int(now_unix_sec), C.byref(n)))
        return int(n.value)

    def reset(self):
        self._check(self._lib.ctmr_group_reset(self._h))

    def snapshot(self) -> np.ndarray:
        need = C.c_uint64(0)
        self._check(self._lib.ctmr_group_snapshot_size(self._h, C.byref(need)))
        buf = np.empty(need.value, np.uint8)
        wrote = C.c_uint64(0)
        self._check(self._lib.ctmr_group_snapshot_save(self._h, capi.ptr(buf), buf.size, C.byref(wrote)))
        return buf[:wrote.value]

    def restore(self, snap: np.ndarray):
        snap = np.ascontiguousarray(snap, np.uint8)
        self._check(self._lib.ctmr_group_snapshot_load(self._h, capi.ptr(snap), snap.size))

    def get_known_certificates(self, exp_hour: int, issuer_digest: bytes):
        grp = self

        class _View:
            def count(self_inner) -> int:
                out = C.c_uint64(0)
                d = (C.c_uint8 * 32).from_buffer_copy(bytes(issuer_digest))
                grp._check(grp._lib.ctmr_group_set_cardinality(grp._h, int(exp_hour), d, C.byref(out)))
                return out.value

            def known(self_inner) -> list:
                return grp.set_members(exp_hour, issuer_digest)[0]
        return _View()

    def issuer_counts(self) -> dict:
        n = C.c_size_t(self._lib.ctmr_issuer_count(self.members[0]._h))
        cap = max(int(n.value), 1)
        dig = np.zeros((cap, 32), np.uint8)
        cnt = np.zeros(cap, np.uint64)
        self._check(self._lib.ctmr_group_issuer_counts(self._h, capi.ptr(dig), capi.ptr(cnt), C.byref(n)))
        return {bytes(dig[i]): int(cnt[i]) for i in range(n.value)}

    def status_counters(self) -> np.ndarray:
        out = np.zeros(capi.ST_COUNT, np.uint64)
        self._check(self._lib.ctmr_group_status_counters(self._h, capi.ptr(out)))
        return out

    def table_stats(self):
        used, cap = C.c_uint64(0), C.c_uint64(0)
        self._check(self._lib.ctmr_group_table_stats(self._h, C.byref(used), C.byref(cap)))
        return used.value, cap.value

    def _single_ctx_only(self, *a, **k):
        raise CtmrError(capi.E_INVALID, "this entry point takes one ctx: use group.members[r] (read side) or the group's own methods")

    # the device-resident / per-ctx entry points of the base class do not take a group handle
    map_device = reduce_device = process_device = read_histogram_device = profile_last = sha256_ceiling = _single_ctx_only
    reset_device = check_device = peer_export = peer_attach = peer_barrier_device = _single_ctx_only
    peer_allreduce_histogram_device = frontend_profile_last = _single_ctx_only


# ---------------------------------------------------------------------- synthetic corpus (bench/test tooling)
def synth_issuers(cfg: capi.SynthCfg):
    """DER of the synthetic CA certificates (host side), (blob u8, offsets u64[n_issuers+1])."""
    L = capi.load()
    offsets = np.zeros(cfg.n_issuers + 1, np.uint64)
    total = L.ctmr_synth_issuers_host(C.byref(cfg), capi.ptr(offsets), None, 0)
    blob = np.zeros(total, np.uint8)
    L.ctmr_synth_issuers_host(C.byref(cfg), capi.ptr(offsets), capi.ptr(blob), total)
    return blob, offsets


def synth_corpus_device(cfg: capi.SynthCfg, first: int, n: int, device, want_issuer_idx=True):
    """Generate entries [first, first+n) in HBM: (blob u8, offsets i64-as-u64 [n+1], issuer_idx i32-as-u32 [n])."""
    import torch

    L = capi.load()
    dev = torch.device(device)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream or 1  # 0x1 = cudaStreamLegacy
        offsets = torch.empty(n + 1, dtype=torch.int64, device=dev)
        total = C.c_uint64(0)
        rc = L.ctmr_synth_offsets_device(C.byref(cfg), first, n, offsets.data_ptr(), C.byref(total), stream)
        if rc:
            raise CtmrError(rc, "ctmr_synth_offsets_device")
        blob = torch.empty(total.value + 64, dtype=torch.uint8, device=dev)  # readable past the end, 16-byte rounding
        idx = torch.empty(n, dtype=torch.int32, device=dev) if want_issuer_idx else None
        rc = L.ctmr_synth_write_device(C.byref(cfg), first, n, offsets.data_ptr(), blob.data_ptr(),
                                       idx.data_ptr() if idx is not None else None, stream)
        if rc:
            raise CtmrError(rc, "ctmr_synth_write_device")
        torch.cuda.synchronize(dev)
    return blob, offsets, idx, int(total.value)
