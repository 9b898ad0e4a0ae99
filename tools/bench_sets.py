"""Cost of reading the known-certificate sets back out of one GPU: list_sets, export_sets and import_sets over a state of
10 M distinct keys (device synthetic corpus, table capacity 2^25).

    python tools/bench_sets.py [--entries N] [--table-log2 K] [--pair-log2 P] [--reps R] [--out FILE]

Prints one JSON line (and writes it to --out): wall time of each call (host clock around a call that ends in a device
synchronise, D2H / H2D included), kernel time of the scans (torch.profiler with CUDA activities, in a pass of its own),
the scans' algorithmic bytes over kernel time, and the HBM bandwidth this GPU reaches on a device-to-device copy, measured
in the same run.  Algorithmic bytes: member scan = 32 B x table slots (first sectors) + 32 B x members (second sectors);
(issuer, hour) scan = 32 B x pair slots per pass.  Needs a CUDA device: there is no CPU fallback.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def device_copy_bandwidth(torch, nbytes=4 << 30, reps=10):
    """bytes read + written per second of a device-to-device copy, best of `reps` (buffers far above the 126 MB L2)."""
    a = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    best = float("inf")
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        e1.synchronize()
        best = min(best, e0.elapsed_time(e1) / 1e3)
    del a, b
    torch.cuda.empty_cache()
    return 2 * nbytes / best


def build_state(torch, capi, engine, n, table_log2, pair_log2):
    cfg = capi.synth_cfg(n, len_mode=1, len_lo=400, len_hi=900, dup_mode=0)
    dev = torch.device("cuda:0")
    iblob, ioffs = engine.synth_issuers(cfg)
    db = engine.GpuCertDatabase(table_capacity=1 << table_log2, issuer_cn_filter=b"", log_expired_entries=True, max_issuers=1024,
                                max_batch_entries=1 << 21, pair_capacity_log2=pair_log2)
    db.register_issuers(iblob, ioffs)
    step = 1 << 21
    wu = torch.empty(step, dtype=torch.uint8, device=dev)
    fi = torch.empty(step, dtype=torch.uint8, device=dev)
    st = torch.empty(step, dtype=torch.uint8, device=dev)
    for first in range(0, n, step):
        m = min(step, n - first)
        blob, offsets, idx, total = engine.synth_corpus_device(cfg, first, m, dev)
        b = capi.DevBatch()
        b.blob, b.blob_bytes, b.offsets, b.n = blob.data_ptr(), total, offsets.data_ptr(), m
        b.issuer_idx, b.issuer_map, b.issuer_map_len = idx.data_ptr(), None, 0
        b.first_index, b.now_unix_ns = first, cfg.now_sec * 10**9
        o = capi.DevOut(st.data_ptr(), None, None, None, None, wu.data_ptr(), fi.data_ptr(), None)
        db.process_device(b, o)
        torch.cuda.synchronize()
        db.check_device()
        del blob, offsets, idx
    return db


def kernel_ms(torch, fn, names):
    """CUDA time per kernel-name substring of one call of fn, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {k: 0.0 for k in names}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = getattr(e, "cuda_time_total", 0.0)
        for k in names:
            if k in e.key:
                out[k] += t / 1e3
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--entries", type=int, default=10_000_000)
    ap.add_argument("--table-log2", type=int, default=25)
    ap.add_argument("--pair-log2", type=int, default=24, help="(issuer, hour) table slots, log2 (the ctx's pair_capacity_log2)")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default="")
    ap.add_argument("--export-only", action="store_true", help="build the state, run one export, exit (for an external profiler)")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_sets.py needs a CUDA device")
    from ct_mapreduce_b200 import capi, engine
    gpu = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        power = "unknown"
    if a.export_only:
        db = build_state(torch, capi, engine, a.entries, a.table_log2, a.pair_log2)
        print(json.dumps({"tool": "bench_sets", "export_only": True, "members": db.export_sets().n_members}))
        db.close()
        return
    hbm = device_copy_bandwidth(torch)
    db = build_state(torch, capi, engine, a.entries, a.table_log2, a.pair_log2)
    used, cap = db.table_stats()
    pair_slots = 1 << a.pair_log2

    def timed(fn):
        best = float("inf")
        for _ in range(a.reps):
            t0 = time.perf_counter()
            r = fn()
            torch.cuda.synchronize()
            best = min(best, time.perf_counter() - t0)
        return best * 1e3, r

    list_ms, sets = timed(db.list_sets)
    export_ms, ex = timed(db.export_sets)
    assert ex.n_members == used, (ex.n_members, used)

    def do_import():
        t = engine.GpuCertDatabase(table_capacity=1 << a.table_log2, max_issuers=1024, pair_capacity_log2=a.pair_log2)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        t.import_sets(ex)
        dt = time.perf_counter() - t0
        t.close()
        return dt
    do_import()   # warm-up
    import_ms = min(do_import() for _ in range(a.reps)) * 1e3

    names = ["set_scan_kernel", "member_scan_kernel", "member_bytes_kernel", "set_prepare_kernel", "member_len_kernel",
             "member_pack_kernel", "set_check_kernel", "DeviceSegmentedSort", "DeviceRadixSort", "DeviceScan"]
    k_export = kernel_ms(torch, db.export_sets, names)
    k_list = kernel_ms(torch, db.list_sets, names)
    member_bytes = 32 * cap + 32 * ex.n_members
    set_bytes = 32 * pair_slots
    scan_ms = k_export["member_scan_kernel"]
    set_scan_ms = k_export["set_scan_kernel"] / 2   # a counting pass and a compaction pass
    d2h_bytes = ex.first_index.nbytes + ex.serial_off.nbytes + ex.serials.nbytes + ex.sets.nbytes
    line = {
        "tool": "bench_sets", "gpu": gpu, "power_limit_and_max_sm_clock": power, "entries": a.entries,
        "table_slots": cap, "pair_slots": pair_slots, "members": ex.n_members, "sets": int(ex.sets.size),
        "serial_bytes": int(ex.serials.size), "export_host_bytes": int(d2h_bytes),
        "wall_ms": {"list_sets": round(list_ms, 3), "export_sets": round(export_ms, 3), "import_sets": round(import_ms, 3)},
        "kernel_ms_export": {k: round(v, 4) for k, v in k_export.items()},
        "kernel_ms_list": {k: round(v, 4) for k, v in k_list.items()},
        "measured_hbm_copy_GBps": round(hbm / 1e9, 1),
        "member_scan_GBps": round(member_bytes / (scan_ms / 1e3) / 1e9, 1) if scan_ms else None,
        "member_scan_share_of_measured_hbm": round(member_bytes / (scan_ms / 1e3) / hbm, 3) if scan_ms else None,
        "set_scan_GBps": round(set_bytes / (set_scan_ms / 1e3) / 1e9, 1) if set_scan_ms else None,
        "set_scan_share_of_measured_hbm": round(set_bytes / (set_scan_ms / 1e3) / hbm, 3) if set_scan_ms else None,
        "export_kernel_ms_total": round(sum(k_export.values()), 3),
    }
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")
    db.close()


if __name__ == "__main__":
    main()
