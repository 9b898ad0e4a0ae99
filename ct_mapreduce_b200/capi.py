"""ctypes binding of libctmr.so (include/ctmr.h) -- the same C ABI a Go host binds with cgo.

The library is hand-written CUDA for sm_100a; there is no Python or CPU implementation of the path
behind these calls.  `load()` raises if the shared object is missing instead of falling back.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libctmr.so")

# per-entry status (include/ctmr.h CTMR_ST_*)
ST_OK, ST_PARSE_ERR, ST_FILTER_CA, ST_FILTER_EXPIRED, ST_FILTER_CN, ST_NO_ISSUER, ST_ISSUER_PARSE_ERR, ST_SERIAL_TOO_LONG = range(8)
ST_COUNT = 8
ISSUER_NONE = 0xFFFFFFFF
MAX_SERIAL = 39
ISSUER_BAD = 0xFFFFFFFE
F_NO_FINGERPRINT = 1
E_INVALID = -1
E_TABLE_FULL = -4
E_TOO_MANY_ISSUERS = -5
E_NO_DEVICE = -6
E_BATCH_TOO_LARGE = -7

EXPORTS = [
    "ctmr_abi_version", "ctmr_create", "ctmr_destroy", "ctmr_last_error", "ctmr_host_alloc", "ctmr_host_free",
    "ctmr_register_issuers", "ctmr_issuer_digest", "ctmr_issuer_count", "ctmr_process_batch", "ctmr_issuer_counts",
    "ctmr_set_cardinality", "ctmr_status_counters", "ctmr_table_stats", "ctmr_map_device", "ctmr_reduce_device",
    "ctmr_process_device", "ctmr_read_histogram_device",
    "ctmr_check_device", "ctmr_reset_device", "ctmr_profile_last", "ctmr_preload_known", "ctmr_snapshot_size",
    "ctmr_snapshot_save", "ctmr_snapshot_load", "ctmr_evict_expired", "ctmr_sha256_ceiling_device", "ctmr_synth_offsets_device", "ctmr_synth_write_device", "ctmr_synth_truth_device", "ctmr_synth_issuers_host", "ctmr_synth_raw_pages_host",
    "ctmr_process_raw", "ctmr_group_process_raw", "ctmr_frontend_profile_last",  # include/ctmr_frontend.h
    # several GPUs: one process (group) / one process per GPU (peer)
    "ctmr_group_create", "ctmr_group_destroy", "ctmr_group_last_error", "ctmr_group_size", "ctmr_group_member",
    "ctmr_group_process_batch", "ctmr_group_issuer_counts", "ctmr_group_set_cardinality", "ctmr_group_status_counters",
    "ctmr_group_table_stats", "ctmr_group_preload_known", "ctmr_group_evict_expired", "ctmr_group_reset",
    "ctmr_group_snapshot_size", "ctmr_group_snapshot_save", "ctmr_group_snapshot_load",
    "ctmr_peer_export", "ctmr_peer_attach", "ctmr_peer_barrier_device", "ctmr_peer_allreduce_histogram_device",
    "ctmr_bind_host_to_device", "ctmr_peer_rounds", "ctmr_peer_round_entries",
    # the sets read back: list, members, canonical export / import
    "ctmr_list_sets", "ctmr_set_members", "ctmr_export_sets", "ctmr_import_sets",
    "ctmr_group_list_sets", "ctmr_group_set_members", "ctmr_group_export_sets", "ctmr_group_import_sets",
]
PEER_HANDLE_BYTES = 256
PEER_ROUNDS = 8   # default; peer_rounds() asks the library (environment override)


def peer_rounds() -> int:
    return int(load().ctmr_peer_rounds())
E_PAIR_TABLE_FULL, E_META_TABLE_FULL, E_PEER_TIMEOUT, E_PEER = -8, -9, -10, -11


class Config(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("device", C.c_int32), ("table_capacity", C.c_uint64),
        ("max_batch_entries", C.c_uint64), ("max_batch_bytes", C.c_uint64), ("max_issuers", C.c_uint32),
        ("pair_capacity_log2", C.c_uint32), ("issuer_cn_filter", C.c_char_p), ("issuer_cn_filter_len", C.c_uint32),
        ("log_expired_entries", C.c_uint32), ("flags", C.c_uint32), ("meta_capacity_log2", C.c_uint32),
        ("max_round_entries", C.c_uint64),
    ]


class Out(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in
                ("status", "sha256", "exp_hour", "serial_off", "serial_len", "was_unknown", "first_issuer_hour",
                 "issuer_name_off", "issuer_name_len", "crldp_off", "crldp_len", "first_issuer_dn", "first_crldp")] + \
               [("pem", C.c_void_p), ("pem_cap", C.c_uint64), ("pem_off", C.c_void_p)]


class DevBatch(C.Structure):
    _fields_ = [
        ("blob", C.c_void_p), ("blob_bytes", C.c_uint64), ("offsets", C.c_void_p), ("n", C.c_uint64),
        ("issuer_idx", C.c_void_p), ("issuer_map", C.c_void_p), ("issuer_map_len", C.c_uint32), ("reserved", C.c_uint32),
        ("first_index", C.c_uint64), ("now_unix_ns", C.c_int64), ("lens", C.c_void_p),
    ]


class DevOut(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in
                ("status", "sha256", "exp_hour", "serial_off", "serial_len", "was_unknown", "first_issuer_hour", "keys",
                 "issuer_name_off", "issuer_name_len", "crldp_off", "crldp_len", "first_issuer_dn", "first_crldp")]


class RawBatch(C.Structure):
    """ctmr_raw_batch (include/ctmr_frontend.h)."""
    _fields_ = [("text", C.c_void_p), ("text_bytes", C.c_uint64), ("leaf_input_off", C.c_void_p), ("leaf_input_len", C.c_void_p),
                ("extra_data_off", C.c_void_p), ("extra_data_len", C.c_void_p), ("n", C.c_uint64), ("now_unix_ns", C.c_int64)]


class RawOut(C.Structure):
    """ctmr_raw_out (include/ctmr_frontend.h)."""
    _fields_ = [("path", Out)] + [(n, C.c_void_p) for n in
                                  ("entry_status", "entry_type", "timestamp_ms", "issuer", "leaf_src", "leaf_off", "leaf_len")]


class SynthCfg(C.Structure):
    """ctmr_synth_cfg (csrc/ctmr_synth.h): the synthetic CT corpus of SURVEY.md §8(d)."""
    _fields_ = [
        ("seed", C.c_uint64), ("n_total", C.c_uint64), ("n_issuers", C.c_uint32), ("len_mode", C.c_uint32),
        ("len_lo", C.c_uint32), ("len_hi", C.c_uint32), ("dup_mode", C.c_uint32), ("reserved", C.c_uint32),
        ("now_sec", C.c_int64),
    ]


class SetInfo(C.Structure):
    """ctmr_set_info (include/ctmr.h)."""
    _fields_ = [("issuer_digest", C.c_uint8 * 32), ("exp_hour", C.c_int64), ("count", C.c_uint64), ("member_off", C.c_uint64)]


SET_INFO_DTYPE = np.dtype([("issuer_digest", "u1", (32,)), ("exp_hour", "<i8"), ("count", "<u8"), ("member_off", "<u8")])
assert SET_INFO_DTYPE.itemsize == 56


class SetExport(C.Structure):
    """ctmr_set_export (include/ctmr.h)."""
    _fields_ = [("next_index", C.c_uint64), ("n_sets", C.c_uint64), ("n_members", C.c_uint64), ("serial_bytes", C.c_uint64),
                ("sets", C.c_void_p), ("sets_cap", C.c_uint64), ("serials", C.c_void_p), ("serials_cap", C.c_uint64),
                ("serial_off", C.c_void_p), ("first_index", C.c_void_p), ("members_cap", C.c_uint64)]


KEY_BYTES = 64
KEY_DTYPE = np.dtype([("index", "<u8"), ("exp_hour", "<i4"), ("issuer", "<u4"), ("serial_len", "u1"),
                      ("serial", "u1", (39,)), ("valid", "<u4"), ("pad", "<u4")])
assert KEY_DTYPE.itemsize == KEY_BYTES

_lib = None


class CtmrError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"ctmr error {code}: {msg}")
        self.code = code


def load():
    """dlopen libctmr.so; fails loudly when the CUDA extension has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: run `python -m ct_mapreduce_b200.build` "
                           "(the CT map/reduce path has no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, u64, u32, i64 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int64
    L.ctmr_abi_version.restype = u32
    L.ctmr_create.argtypes = [C.POINTER(Config), C.POINTER(vp)]
    L.ctmr_destroy.argtypes = [vp]
    L.ctmr_destroy.restype = None
    L.ctmr_last_error.argtypes = [vp]
    L.ctmr_last_error.restype = C.c_char_p
    L.ctmr_host_alloc.argtypes = [C.c_size_t]
    L.ctmr_host_alloc.restype = vp
    L.ctmr_host_free.argtypes = [vp]
    L.ctmr_host_free.restype = None
    L.ctmr_register_issuers.argtypes = [vp, vp, vp, u32, vp]
    L.ctmr_issuer_digest.argtypes = [vp, u32, vp]
    L.ctmr_issuer_count.argtypes = [vp]
    L.ctmr_issuer_count.restype = u32
    L.ctmr_process_batch.argtypes = [vp, vp, vp, u64, vp, vp, u32, vp, i64, C.POINTER(Out)]
    L.ctmr_issuer_counts.argtypes = [vp, vp, vp, C.POINTER(C.c_size_t)]
    L.ctmr_set_cardinality.argtypes = [vp, i64, vp, C.POINTER(u64)]
    L.ctmr_status_counters.argtypes = [vp, vp]
    L.ctmr_table_stats.argtypes = [vp, C.POINTER(u64), C.POINTER(u64)]
    L.ctmr_map_device.argtypes = [vp, C.POINTER(DevBatch), C.POINTER(DevOut), vp]
    L.ctmr_reduce_device.argtypes = [vp, vp, u64, vp, vp, vp]
    L.ctmr_process_device.argtypes = [vp, C.POINTER(DevBatch), C.POINTER(DevOut), vp]
    L.ctmr_read_histogram_device.argtypes = [vp, vp, u32, vp, vp]
    L.ctmr_check_device.argtypes = [vp, vp]
    L.ctmr_reset_device.argtypes = [vp, vp]
    L.ctmr_preload_known.argtypes = [vp, i64, vp, vp, vp, u64]
    L.ctmr_snapshot_size.argtypes = [vp, C.POINTER(u64)]
    L.ctmr_snapshot_save.argtypes = [vp, vp, u64, C.POINTER(u64)]
    L.ctmr_snapshot_load.argtypes = [vp, vp, u64]
    L.ctmr_evict_expired.argtypes = [vp, i64, C.POINTER(u64)]
    L.ctmr_sha256_ceiling_device.argtypes = [vp, u32, u32, u32, C.POINTER(C.c_float), C.POINTER(u64)]
    L.ctmr_profile_last.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_float)]
    L.ctmr_synth_offsets_device.argtypes = [C.POINTER(SynthCfg), u64, u64, vp, C.POINTER(u64), vp]
    L.ctmr_synth_write_device.argtypes = [C.POINTER(SynthCfg), u64, u64, vp, vp, vp, vp]
    L.ctmr_synth_truth_device.argtypes = [C.POINTER(SynthCfg), u64, u64, vp, vp, vp, vp]
    L.ctmr_synth_issuers_host.argtypes = [C.POINTER(SynthCfg), vp, vp, u64]
    L.ctmr_synth_issuers_host.restype = u64
    L.ctmr_synth_raw_pages_host.argtypes = [C.POINTER(SynthCfg), u64, u64, u32, vp, u64, vp, vp, vp, vp]
    L.ctmr_synth_raw_pages_host.restype = u64
    L.ctmr_process_raw.argtypes = [vp, C.POINTER(RawBatch), C.POINTER(RawOut)]
    L.ctmr_group_process_raw.argtypes = [vp, C.POINTER(RawBatch), C.POINTER(RawOut)]
    L.ctmr_frontend_profile_last.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(u64)]
    L.ctmr_group_create.argtypes = [C.POINTER(Config), vp, u32, C.POINTER(vp)]
    L.ctmr_group_destroy.argtypes = [vp]
    L.ctmr_group_destroy.restype = None
    L.ctmr_group_last_error.argtypes = [vp]
    L.ctmr_group_last_error.restype = C.c_char_p
    L.ctmr_group_size.argtypes = [vp]
    L.ctmr_group_size.restype = u32
    L.ctmr_group_member.argtypes = [vp, u32]
    L.ctmr_group_member.restype = vp
    L.ctmr_group_process_batch.argtypes = [vp, vp, vp, u64, vp, vp, u32, vp, i64, C.POINTER(Out)]
    L.ctmr_group_issuer_counts.argtypes = [vp, vp, vp, C.POINTER(C.c_size_t)]
    L.ctmr_group_set_cardinality.argtypes = [vp, i64, vp, C.POINTER(u64)]
    L.ctmr_group_status_counters.argtypes = [vp, vp]
    L.ctmr_group_table_stats.argtypes = [vp, C.POINTER(u64), C.POINTER(u64)]
    L.ctmr_group_preload_known.argtypes = [vp, i64, vp, vp, vp, u64]
    L.ctmr_group_evict_expired.argtypes = [vp, i64, C.POINTER(u64)]
    L.ctmr_group_reset.argtypes = [vp]
    L.ctmr_group_snapshot_size.argtypes = [vp, C.POINTER(u64)]
    L.ctmr_group_snapshot_save.argtypes = [vp, vp, u64, C.POINTER(u64)]
    L.ctmr_group_snapshot_load.argtypes = [vp, vp, u64]
    L.ctmr_peer_export.argtypes = [vp, u32, vp]
    L.ctmr_peer_attach.argtypes = [vp, u32, u32, vp]
    L.ctmr_peer_barrier_device.argtypes = [vp, vp]
    L.ctmr_peer_allreduce_histogram_device.argtypes = [vp, vp, u32, vp, vp]
    L.ctmr_bind_host_to_device.argtypes = [C.c_int32]
    L.ctmr_peer_rounds.restype = u32
    L.ctmr_peer_round_entries.argtypes = [u64]
    L.ctmr_peer_round_entries.restype = u64
    for pre in ("ctmr_", "ctmr_group_"):
        getattr(L, pre + "list_sets").argtypes = [vp, i64, i64, vp, u64, C.POINTER(u64)]
        getattr(L, pre + "set_members").argtypes = [vp, i64, vp, vp, u64, vp, vp, u64, C.POINTER(u64)]
        getattr(L, pre + "export_sets").argtypes = [vp, C.POINTER(SetExport)]
        getattr(L, pre + "import_sets").argtypes = [vp, C.POINTER(SetExport)]
    for name in EXPORTS:
        getattr(L, name)  # every symbol include/ctmr.h declares must resolve
    _lib = L
    return L


def ptr(a):
    """Raw address of a numpy array / torch tensor / int / None."""
    if a is None:
        return None
    if isinstance(a, int):
        return a
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    if hasattr(a, "data_ptr"):
        return a.data_ptr()
    raise TypeError(type(a))


def synth_cfg(n_total, seed=20260922, n_issuers=256, len_mode=0, len_lo=1436, len_hi=1564, dup_mode=0,
              now_sec=1767225600) -> SynthCfg:
    return SynthCfg(seed, n_total, n_issuers, len_mode, len_lo, len_hi, dup_mode, 0, now_sec)


class PinnedBuffer:
    """Page-locked host memory from ctmr_host_alloc, viewed as a numpy array."""

    def __init__(self, nbytes: int):
        self.nbytes = int(nbytes)
        self.addr = load().ctmr_host_alloc(max(1, self.nbytes))
        if not self.addr:
            raise MemoryError(f"ctmr_host_alloc({nbytes}) failed")
        self._raw = (C.c_uint8 * max(1, self.nbytes)).from_address(self.addr)

    def view(self, dtype=np.uint8, count=None, offset=0):
        dt = np.dtype(dtype)
        count = (self.nbytes - offset) // dt.itemsize if count is None else count
        return np.frombuffer(self._raw, dtype=dt, count=count, offset=offset)

    def free(self):
        if self.addr:
            self._raw = None
            load().ctmr_host_free(self.addr)
            self.addr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass
