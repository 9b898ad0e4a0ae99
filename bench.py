#!/usr/bin/env python3
"""bench.py -- CT entries/sec through the B200-native map/reduce hot path.

    python bench.py --gpus N --steps K --warmup W            # this repository's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU algorithm (Go engine if `go` exists, else the oracle port)

A "step" is one pass of the hot path over one batch of synthetic CT entries resident in HBM (BASELINE.json
configs[1] at N=1: 10 M x ~1.5 KB DER, SHA-256 fingerprint + KnownCertificates dedup, per-issuer counts).  At N>1
every rank holds its 10 M-entry shard of ONE corpus in which one entry in 16 repeats a certificate living at a
permuted position -- on another GPU with probability 1-1/N -- and the step runs the exact multi-GPU path: K_map
inserts each key into the table of its set's owner GPU over NVLink, barriers in peer memory, one all-reduce of the
histograms.  `value` is whole-job entries/s (CUDA events, max over ranks); `e2e` is the same metric through the
host-buffer C-ABI call (pinned host memory in, host results out, copies inside the timed region, the same exact
multi-GPU path at N>1).  `secondary` holds BASELINE configs[2..4] as written (streamed chunks, persistent tables,
duplicates straddling chunks and GPUs).  Prints ONE JSON line on rank 0.

    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR

also writes what the timed path returned in its last step to DIR/<name>.npy (rank 0's shard): the per-entry outputs of
a fixed, seeded sample of entries (`entry_index`; all entries when there are at most DUMP_ENTRIES) and the whole
per-issuer / per-status histograms.  The corpus is seeded, so two builds run with the same arguments can be compared
output for output.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import shutil
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NOW_SEC = 1767225600
NOW_NS = NOW_SEC * 10**9
SEED = 20260922
README_FILTER = b"Let's Encrypt, ISRG"
# entries sampled by --dump-outputs: 32 fingerprint bytes as float32 + 5 scalars each, about 20 MB in all
DUMP_ENTRIES = 1 << 17

WORKLOADS = {
    # BASELINE.json configs[1]: SHA-256 fingerprint + KnownCertificates dedup (no CN filter, expired kept)
    "cfg2": dict(desc="configs[1]: 10M synthetic ~1.5KB DER certs per GPU, SHA-256 fingerprint + KnownCertificates dedup",
                 n=10_000_000, synth=dict(len_mode=0, len_lo=1436, len_hi=1564, dup_mode=0), filter=b"", log_expired=True,
                 out_bytes=42),
    # the same shape for N>1: one entry in 16 is a duplicate whose twin sits at a permuted position of the GLOBAL corpus
    "cfg2x": dict(desc="configs[1] shape per GPU (10M x ~1.5KB, SHA-256 + dedup), 1 entry in 16 repeats a certificate at a permuted "
                       "position of the global corpus (cross-GPU twins)",
                  n=10_000_000, synth=dict(len_mode=0, len_lo=1436, len_hi=1564, dup_mode=16), filter=b"", log_expired=True,
                  out_bytes=42),
    # configs[2]: full map incl. issuerCNFilter + expiry, IssuerMetadata reduce
    "cfg3": dict(desc="configs[2]: full map (ASN.1 + issuerCNFilter + expiry) + KnownCertificates / IssuerMetadata reduce",
                 n=10_000_000, synth=dict(len_mode=0, len_lo=1436, len_hi=1564, dup_mode=0), filter=README_FILTER,
                 log_expired=False, out_bytes=54),
    # configs[3]: the 1 B-entry shape, sharded by entry index, histograms merged at chunk end
    "cfg4": dict(desc="configs[3]: entries sharded across the GPUs by index, full map, persistent per-GPU tables, histograms merged at chunk end",
                 n=10_000_000, synth=dict(len_mode=0, len_lo=1436, len_hi=1564, dup_mode=0), filter=README_FILTER,
                 log_expired=False, out_bytes=54),
    # configs[4]: mixed 512 B-8 KB, 50 % duplicates, 256 issuers
    "cfg5": dict(desc="configs[4]: mixed 512B-8KB DER, 50% duplicates (twins straddle chunks and GPUs), 256 issuers",
                 n=5_000_000, synth=dict(len_mode=1, len_lo=512, len_hi=8192, dup_mode=1), filter=README_FILTER,
                 log_expired=False, out_bytes=54),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="", choices=[""] + sorted(WORKLOADS), help="default: cfg2 at N=1, cfg2x at N>1")
    ap.add_argument("--entries", type=int, default=0, help="entries per GPU per step (default: the workload's)")
    ap.add_argument("--no-fingerprint", action="store_true",
                    help="CTMR_F_NO_FINGERPRINT: the reference-faithful path (it never hashes the leaf): parse+filter+dedup+counts")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the BASELINE configs[2..4] streaming runs")
    ap.add_argument("--secondary-entries", type=int, default=0, help="entries per GPU of each streaming run (default: as written)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="entries in the CPU sample (default: auto)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the last timed step's outputs (seeded sample of entries + histograms) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# ---------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md clocks line)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def measured_traffic(kernel, entries_per_launch):
    """dram__bytes_read+write of a kernel from the committed ncu --set full capture (profiles/), scaled from the
    captured launch size to this run's entries per launch; None when no capture is committed."""
    for name in (f"r2_{kernel}_traffic.json", "r1_map_traffic.json" if kernel == "map_stream" else ""):
        p = os.path.join(ROOT, "profiles", name)
        try:
            t = json.load(open(p))
            per_entry = (t["dram_bytes_read"] + t["dram_bytes_write"]) / t["entries"]
            return per_entry * entries_per_launch, t["source"]
        except Exception:
            continue
    return None, None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ---------------------------------------------------------------------------------------------- reference arm
def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def go_probe():
    """BASELINE.md §3 Variant A / SURVEY §8(c): use the Go engine when the box has a Go toolchain AND the reference's
    module dependencies are resolvable offline (reference checkout: $CTMR_REFERENCE_DIR).  Returns (usable, one-line
    description)."""
    go = shutil.which("go")
    if not go:
        return False, "`go version`: command not found on this box"
    try:
        ver = subprocess.run([go, "version"], capture_output=True, text=True, timeout=20).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return False, f"`go version` failed: {e}"
    ref = os.environ.get("CTMR_REFERENCE_DIR", "")
    if not os.path.isdir(ref):
        return False, f"{ver}; no reference checkout (set CTMR_REFERENCE_DIR to one)"
    env = dict(os.environ, GOFLAGS="-mod=mod", GOPROXY="off")
    r = subprocess.run([go, "list", "./storage"], cwd=ref, capture_output=True, text=True, env=env, timeout=120)
    if r.returncode != 0:
        return False, f"{ver}; `go list ./storage` fails offline (certificate-transparency-go v1.1.0 not in the module cache)"
    return True, ver


def cpu_arm(n_sample, workload, steps, warmup, make_sample, map_only_too=False):
    """The reference's CPU algorithm (the oracle port when the Go engine is unavailable) over a bounded sample of
    the same workload, map half on every host thread, reduce half sequential exactly like numThreads=1 over
    MockRemoteCache.  Returns (entries/s, seconds/step, threads, map-only entries/s or None)."""
    from oracle import oracle
    blob, offs, idx, iblob, ioffs = make_sample(n_sample)
    thr = host_threads()
    times = []
    for it in range(warmup + steps):
        db = oracle.DB(workload["filter"], workload["log_expired"])
        t0 = time.perf_counter()
        db.process(blob, offs, iblob, ioffs, idx, NOW_NS, nthreads=thr)
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
        del db
    per = sum(times) / len(times)
    map_rate = None
    if map_only_too:  # the parse + filter + SHA-256 half alone on every thread: the like-for-like of K_map
        t0 = time.perf_counter()
        oracle.map_only(blob, offs, workload["filter"], workload["log_expired"], NOW_NS, thr, want_sha=True)
        map_rate = n_sample / (time.perf_counter() - t0)
    return n_sample / per, per, thr, map_rate


def cpu_sample_maker(workload, n_total, rank_first=0):
    """Sample of the bench corpus for the CPU arm; generated by the CPU generator (no GPU involved)."""
    from oracle import oracle

    def make(n):
        cfg = oracle.synth_cfg(max(n_total, n, 2), seed=SEED, **workload["synth"])
        blob, offs, idx = oracle.synth_corpus(cfg, rank_first, n)
        iblob, ioffs = oracle.synth_issuers(cfg)
        return blob, offs, idx, iblob, ioffs
    return make


def default_workload(args, world):
    return args.workload or ("cfg2" if world == 1 else "cfg2x")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    world = max(1, args.gpus)
    wname = default_workload(args, world)
    wl = WORKLOADS[wname]
    n_sample = args.cpu_sample or 400_000
    go_ok, go_note = go_probe()
    # A Go engine run needs the reference's third-party modules; no box so far carried them (go_note says what was found).
    v, per, thr, map_rate = cpu_arm(n_sample, wl, args.steps, max(args.warmup, 1), cpu_sample_maker(wl, world * wl["n"]), map_only_too=True)
    line = {
        "impl": "reference", "metric": "ct_entries_per_sec", "value": v, "unit": "entries/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": per * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": wl["desc"], "sample_entries_per_step": n_sample},
        "cpu_baseline": {"value": v, "unit": "entries/s", "cores": thr, "kind": "port",
                         "sample": f"{n_sample} entries of the same corpus per step; map half on {thr} threads, reduce half "
                                   "sequential (reference numThreads=1 over MockRemoteCache); C restatement, not the Go engine",
                         "map_only_value": map_rate, "go_probe": go_note},
        "e2e": {"value": v, "unit": "entries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------------------------- our arm
def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist

    from ct_mapreduce_b200 import build, capi, engine, sharded

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # debugging aid: every rank on cuda:0 with gloo plumbing (NCCL refuses two ranks on one device); the data path is the
    # same -- peer tables over CUDA IPC, barriers in peer memory -- only slower (the processes time-slice one GPU)
    same_gpu = os.environ.get("CTMR_BENCH_SAME_GPU", "0") == "1"
    if same_gpu:
        local = 0
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl=ours) needs a CUDA device: the path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    build.build()
    lib = capi.load()
    # pinned buffers allocated from here on are local to the GPU's NUMA node (8 ranks x 56 GB/s of host reads)
    numa_node = lib.ctmr_bind_host_to_device(local) if os.environ.get("CTMR_BENCH_NUMA", "1") == "1" else -2
    if world > 1:
        if same_gpu:
            dist.init_process_group("gloo")
        else:
            dist.init_process_group("nccl", device_id=dev)
    # a CPU-side barrier for the phase in which rank 0 alone drives every GPU (the one-process group form)
    cpu_group = dist.new_group(backend="gloo") if world > 1 else None
    cdev = torch.device("cpu") if same_gpu else dev   # where the bench's own (untimed) reductions live
    wname = default_workload(args, world)
    wl = WORKLOADS[wname]
    n = args.entries or wl["n"]
    K, W = args.steps, args.warmup
    flags = capi.F_NO_FINGERPRINT if args.no_fingerprint else 0
    R = capi.peer_rounds()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def allmax(x):
        t = torch.tensor([x], dtype=torch.float64, device=cdev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allsum(vals):
        t = torch.tensor(vals, dtype=torch.int64, device=cdev)
        if world > 1:
            dist.all_reduce(t)
        return [int(x) for x in t.tolist()]

    def make_db(table_capacity, w, fl, entries_per_call):
        db = engine.GpuCertDatabase(device=local, table_capacity=table_capacity, issuer_cn_filter=w["filter"],
                                    log_expired_entries=w["log_expired"], flags=fl, max_issuers=4096,
                                    max_round_entries=sharded.round_entries(entries_per_call))
        sharded.attach_peers(db)  # N>1: the owners' tables over CUDA IPC; collective calls from here on
        return db

    def pow2(v):
        p = 1
        while p < v:
            p <<= 1
        return p

    # ---- corpus: rank r owns entries [r*n, (r+1)*n) of one global corpus (weak scaling), generated in HBM
    cfg = capi.synth_cfg(world * n, seed=SEED, **wl["synth"])
    blob, offsets, issuer_idx, total_bytes = engine.synth_corpus_device(cfg, rank * n, n, dev)
    iblob, ioffs = engine.synth_issuers(cfg)
    db = make_db(max(1 << 20, 2 * n), wl, flags, n)
    dense = db.register_issuers(iblob, ioffs)
    dense_t = torch.from_numpy(dense.astype(np.int32)).to(dev)
    issuer_dense = dense_t[issuer_idx.long()].contiguous()   # dense registry indices (the registry is shared by the group)

    status = torch.empty(n, dtype=torch.uint8, device=dev)
    sha = torch.empty((n, 32), dtype=torch.uint8, device=dev)
    exp_hour = torch.empty(n, dtype=torch.int64, device=dev)
    was_unknown = torch.empty(n, dtype=torch.uint8, device=dev)
    first = torch.empty(n, dtype=torch.uint8, device=dev)
    hist = torch.zeros(cfg.n_issuers + capi.ST_COUNT, dtype=torch.int64, device=dev)
    stream = torch.cuda.Stream(dev)      # brackets the timed region; the library forks its map / reduce streams off it
    torch.cuda.synchronize(dev)
    torch.cuda.set_stream(stream)
    span = sharded.call_index_span(n, world)
    step_no = [0]

    def dev_batch():
        b = capi.DevBatch()
        b.blob, b.blob_bytes, b.offsets, b.n = blob.data_ptr(), total_bytes, offsets.data_ptr(), n
        b.issuer_idx, b.issuer_map, b.issuer_map_len = issuer_dense.data_ptr(), None, 0
        b.first_index = step_no[0] * span    # round k of rank r: + (k*world + r) * ceil(n/R): rounds in order, ranks inside
        b.now_unix_ns = NOW_NS
        return b

    out = capi.DevOut(status.data_ptr(), None if args.no_fingerprint else sha.data_ptr(), exp_hour.data_ptr(), None, None,
                      was_unknown.data_ptr(), first.data_ptr(), None)

    def step():
        db.reset_device(stream.cuda_stream)               # every step sees an empty known-certificate set (collective at N>1)
        db.process_device(dev_batch(), out, stream.cuda_stream)   # K_map (+ insert at the owners), barriers, resolve, pairs
        if world > 1:   # the chunk-end merge of the per-GPU histograms, over peer memory
            db.peer_allreduce_histogram_device(hist[: cfg.n_issuers], cfg.n_issuers, hist[cfg.n_issuers:], stream.cuda_stream)
        else:
            db.read_histogram_device(hist[: cfg.n_issuers], cfg.n_issuers, hist[cfg.n_issuers:], stream.cuda_stream)
        step_no[0] += 1

    for _ in range(W):
        step()
    db.check_device(stream.cuda_stream)
    barrier()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
    map_ms_acc = 0.0
    t0.record(stream)
    for _ in range(K):
        step()
    t1.record(stream)
    barrier()
    clk = clocks.stop() if rank == 0 else None
    elapsed_ms = allmax(t0.elapsed_time(t1))
    map_ms = allmax(db.profile_last()[0])   # K_map's CUDA-event duration (sum over the step's 4 launches) in the LAST timed step
    db.check_device(stream.cuda_stream)
    counts, stat = hist[: cfg.n_issuers].clone(), hist[cfg.n_issuers:].clone()
    if args.dump_outputs and rank == 0:
        pick = np.sort(np.random.default_rng(SEED).choice(n, min(n, DUMP_ENTRIES), replace=False))
        sel = torch.from_numpy(pick).to(dev)
        dump = {"entry_index": pick.astype(np.float64), "status": status[sel].cpu().numpy().astype(np.float32),
                "exp_hour": exp_hour[sel].cpu().numpy().astype(np.float64),
                "was_unknown": was_unknown[sel].cpu().numpy().astype(np.float32),
                "first_issuer_hour": first[sel].cpu().numpy().astype(np.float32),
                "issuer_counts": counts.cpu().numpy().astype(np.float64), "status_counters": stat.cpu().numpy().astype(np.float64)}
        if not args.no_fingerprint:
            dump["sha256"] = sha[sel].cpu().numpy().astype(np.float32)
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dump.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        del sel

    # ---- the timed result is the real thing: size-independent checks on the LAST timed step's outputs ----------
    truth_id = torch.empty(n, dtype=torch.int64, device=dev)
    truth_na = torch.empty(n, dtype=torch.int64, device=dev)
    truth_bc = torch.empty(n, dtype=torch.uint8, device=dev)
    rc = lib.ctmr_synth_truth_device(C.byref(cfg), rank * n, n, truth_id.data_ptr(), truth_na.data_ptr(), truth_bc.data_ptr(),
                                     stream.cuda_stream)
    assert rc == 0
    torch.cuda.synchronize(dev)
    okm = status == 0
    d = wl["synth"]["dup_mode"]
    paired = (torch.ones_like(okm) if d == 1 else ((truth_id % d) == d - 2)) if d else torch.zeros_like(okm)
    n_ok, n_unknown, n_ok_paired = allsum([int(okm.sum()), int(was_unknown.sum()), int((okm & paired).sum())])
    assert int(counts.sum()) == n_unknown, "per-issuer counts must sum to the number of unknown entries"
    assert int(stat[0]) == n_ok, "status counter OK mismatch"
    # every certificate of the (complete) global corpus is either single or a pair of twins with equal status:
    # distinct kept certificates = kept entries - half of the kept paired entries
    assert n_ok_paired % 2 == 0 and n_unknown == n_ok - n_ok_paired // 2, \
        f"sum(was_unknown)={n_unknown} != distinct kept certificates={n_ok - n_ok_paired // 2}"
    cross_rank_pairs = None
    if d and world > 1:
        # exact cross-GPU semantics on the full data: gather (certificate, global order, bit) of every kept paired entry,
        # sort by certificate, and check that exactly the EARLIER twin is the unknown one
        e_round = sharded.round_entries(n)
        j = torch.arange(n, device=dev, dtype=torch.int64)
        order_pos = ((j // e_round) * world + rank) * e_round + (j % e_round)
        sel = okm & paired
        m_loc = int(sel.sum())
        m_max = int(allmax(m_loc))
        pack = torch.full((m_max, 4), -1, dtype=torch.int64, device=dev)
        pack[:m_loc, 0] = truth_id[sel]
        pack[:m_loc, 1] = order_pos[sel]
        pack[:m_loc, 2] = was_unknown[sel].long()
        pack[:m_loc, 3] = rank
        pack = pack.to(cdev)
        allp = [torch.empty_like(pack) for _ in range(world)]
        dist.all_gather(allp, pack)
        allp = torch.cat(allp).to(dev)
        allp = allp[allp[:, 0] >= 0]
        allp = allp[torch.argsort(allp[:, 1])]
        allp = allp[torch.argsort(allp[:, 0], stable=True)]
        a, b2 = allp[0::2], allp[1::2]
        assert a.shape == b2.shape and bool((a[:, 0] == b2[:, 0]).all()), "twins must pair up"
        assert bool((a[:, 2] == 1).all()) and bool((b2[:, 2] == 0).all()), "the earlier twin is unknown, the later one known"
        cross_rank_pairs = int((a[:, 3] != b2[:, 3]).sum())
        assert cross_rank_pairs > 0
        del allp, a, b2, pack
    # a sampled slice against the oracle (rank 0's first entries = the head of the global order: map outputs bit-exact,
    # membership bits = the oracle's sequential run from an empty set)
    import hashlib
    oracle_sample = 0
    if rank == 0:
        from oracle import oracle
        ns = min(4096, sharded.round_entries(n), n)
        offs_h = offsets[: ns + 1].cpu().numpy().astype(np.uint64)
        blob_h = blob[: int(offs_h[ns])].cpu().numpy()
        want = oracle.DB(wl["filter"], wl["log_expired"]).process(blob_h, offs_h, iblob, ioffs, issuer_idx[:ns].cpu().numpy().astype(np.uint32), NOW_NS)
        assert np.array_equal(status[:ns].cpu().numpy(), want.status), "status differs from the oracle on the sampled slice"
        assert np.array_equal(was_unknown[:ns].cpu().numpy(), want.was_unknown), "membership bits differ from the oracle on the sampled slice"
        assert np.array_equal(first[:ns].cpu().numpy(), want.first_issuer_hour), "first-(issuer,hour) bits differ from the oracle"
        if not args.no_fingerprint:
            assert np.array_equal(sha[:ns].cpu().numpy(), want.sha256), "fingerprints differ from the oracle on the sampled slice"
            for i in range(8):
                assert sha[i].cpu().numpy().tobytes() == hashlib.sha256(blob_h[offs_h[i]:offs_h[i + 1]].tobytes()).digest()
        oracle_sample = ns
    sha_head = sha[:8].cpu().numpy()
    del truth_id, truth_na, truth_bc

    value = world * n * K / (elapsed_ms / 1e3)
    peak, peak_src = measured_peaks()
    alg_bytes = total_bytes + wl["out_bytes"] * n  # SURVEY.md §8(d): sum(L_i) + 42*N (cfg2) / 54*N (cfg3-5), per step
    hbm_achieved = alg_bytes / (map_ms / 1e3) / 1e9
    sha_gbs_kernel = total_bytes / (map_ms / 1e3) / 1e9
    # measured INT-pipe ceiling of the fingerprint on this GPU: register-only SHA-256 at K_map's occupancy
    int_ceiling_gbs = db.sha256_ceiling(iters=2000, rolled=True, ctas_per_sm=2)[0] if not args.no_fingerprint else None
    map_launches = R if world > 1 else (8 if n >= (1 << 21) else (2 if n >= (1 << 18) else 1))
    # per round: len_order (3 kernels) + K_map + resolve + pairs; N>1 adds 2 barrier kernels per round, 2 around the reset,
    # and barrier + sum + barrier for the histogram all-reduce
    launches_per_step = map_launches * 6 + (map_launches * 2 + 2 + 3 if world > 1 else 0)
    kname = "map_light" if args.no_fingerprint else "map_stream"
    traffic, traffic_src = measured_traffic(kname, n / map_launches)

    # ---- e2e through the host-buffer C ABI (pinned host memory -> results on the host); at N>1 the same exact
    # multi-GPU path: a collective ctmr_process_batch per rank, keys inserted at their owners over NVLink
    e2e = None
    if not args.no_e2e:
        ne = n
        hb = capi.PinnedBuffer(total_bytes + 64)
        ho = capi.PinnedBuffer((ne + 1) * 8)
        hi = capi.PinnedBuffer(ne * 4)
        out_bufs = {k: capi.PinnedBuffer(ne * sz) for k, sz in (("status", 1), ("sha256", 32), ("exp_hour", 8),
                                                                   ("was_unknown", 1), ("first", 1))}
        hblob = torch.from_numpy(hb.view(np.uint8, total_bytes))
        hblob.copy_(blob[:total_bytes])
        torch.from_numpy(ho.view(np.int64, ne + 1)).copy_(offsets)
        torch.from_numpy(hi.view(np.int32, ne)).copy_(issuer_idx)
        torch.cuda.synchronize(dev)
        res = engine.BatchResult(out_bufs["status"].view(np.uint8), out_bufs["sha256"].view(np.uint8).reshape(ne, 32),
                                 out_bufs["exp_hour"].view(np.int64), None, None, out_bufs["was_unknown"].view(np.uint8),
                                 out_bufs["first"].view(np.uint8))
        h2d = total_bytes + (ne + 1) * 8 + ne * 4
        d2h = ne * (1 + (0 if args.no_fingerprint else 32) + 8 + 1 + 1)

        def e2e_step():
            db.reset_device(None)
            o = capi.Out(res.status.ctypes.data, None if args.no_fingerprint else res.sha256.ctypes.data, res.exp_hour.ctypes.data,
                         None, None, res.was_unknown.ctypes.data, res.first_issuer_hour.ctypes.data)
            rc = db._lib.ctmr_process_batch(db.handle, hb.addr, ho.addr, ne, iblob.ctypes.data, ioffs.ctypes.data,
                                            cfg.n_issuers, hi.addr, NOW_NS, C.byref(o))
            db._check(rc)

        for _ in range(min(W, 2)):
            e2e_step()
        barrier()
        ts = time.perf_counter()
        for _ in range(K):
            e2e_step()
        torch.cuda.synchronize(dev)
        dt = allmax(time.perf_counter() - ts)
        assert args.no_fingerprint or np.array_equal(res.sha256[:8], sha_head), "e2e fingerprints differ from the device-resident run"
        # the same exactness check as above, on the host-side outputs of the last e2e step
        e_ok, e_unknown = allsum([int((res.status == 0).sum()), int(res.was_unknown.sum())])
        assert e_ok == n_ok and e_unknown == n_unknown, f"e2e: sum(was_unknown)={e_unknown}, kept={e_ok}; expected {n_unknown}, {n_ok}"
        e2e = {"value": world * ne * K / dt, "unit": "entries/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "note": "ctmr_process_batch, pinned host buffers, 3-stage H2D/kernel/D2H pipeline"
                       + ("; collective call per rank, keys inserted at their owner GPU over NVLink (globally exact: "
                          "sum(was_unknown) checked against the distinct kept certificates)" if world > 1 else ""),
               "numa_node": numa_node}
        del hblob, res
        for b_ in [hb, ho, hi] + list(out_bufs.values()):
            b_.free()

    # ---- CPU baseline (rank 0, N=1 only): the oracle port on the box's host cores, bounded sample
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        n_sample = args.cpu_sample or 400_000
        v, per, thr, map_rate = cpu_arm(n_sample, wl, 1, 1, cpu_sample_maker(wl, world * n), map_only_too=True)
        cpu = {"value": v, "unit": "entries/s", "cores": thr, "kind": "port",
               "sample": f"first {n_sample} entries of the same corpus, 1 timed pass ({per:.2f} s); map half on {thr} threads, "
                         "reduce half sequential like the reference's numThreads=1; C restatement, not the Go engine",
               "map_only_value": map_rate,
               "map_only_note": f"parse + filter + SHA-256 alone on {thr} threads (no reducers): the like-for-like of K_map",
               "go_probe": go_probe()[1]}

    # ---- BASELINE configs[2..4] as written: streamed chunks, persistent tables, duplicates across chunks and GPUs ----
    del blob, offsets, issuer_idx, issuer_dense, status, sha, exp_hour, was_unknown, first
    db.close()
    torch.cuda.empty_cache()
    secondary = []
    if not args.no_secondary:
        def stream_run(tag, wname2, per_gpu_entries, fl):
            w2 = WORKLOADS[wname2]
            nc = min(w2["n"], per_gpu_entries)
            chunks = max(1, -(-per_gpu_entries // nc))
            cfg2 = capi.synth_cfg(chunks * world * nc, seed=SEED + 1, **w2["synth"])
            db2 = make_db(pow2(int(1.6 * chunks * nc)), w2, fl, nc)
            try:
                ib2, io2 = engine.synth_issuers(cfg2)
                d2 = torch.from_numpy(db2.register_issuers(ib2, io2).astype(np.int32)).to(dev)
                st = torch.empty(nc, dtype=torch.uint8, device=dev)
                sh = None if (fl & capi.F_NO_FINGERPRINT) else torch.empty((nc, 32), dtype=torch.uint8, device=dev)
                eh = torch.empty(nc, dtype=torch.int64, device=dev)
                wu = torch.empty(nc, dtype=torch.uint8, device=dev)
                fi = torch.empty(nc, dtype=torch.uint8, device=dev)
                tid = torch.empty(nc, dtype=torch.int64, device=dev)
                tna = torch.empty(nc, dtype=torch.int64, device=dev)
                tbc = torch.empty(nc, dtype=torch.uint8, device=dev)
                h2 = torch.zeros(cfg2.n_issuers + capi.ST_COUNT, dtype=torch.int64, device=dev)
                acc = torch.zeros(3, dtype=torch.int64, device=dev)   # kept, unknown, kept & paired
                sp = sharded.call_index_span(nc, world)
                dd = w2["synth"]["dup_mode"]
                tot_ms = tot_map = 0.0
                tot_bytes = 0
                evs = []
                for c in range(chunks):
                    first_entry = (c * world + rank) * nc     # chunk c of the stream: contiguous slices per GPU
                    bl, of, ix, tb = engine.synth_corpus_device(cfg2, first_entry, nc, dev)   # generator: not timed
                    ixd = d2[ix.long()].contiguous()
                    bb = capi.DevBatch()
                    bb.blob, bb.blob_bytes, bb.offsets, bb.n = bl.data_ptr(), tb, of.data_ptr(), nc
                    bb.issuer_idx, bb.issuer_map, bb.issuer_map_len = ixd.data_ptr(), None, 0
                    bb.first_index, bb.now_unix_ns = c * sp, NOW_NS
                    oo = capi.DevOut(st.data_ptr(), sh.data_ptr() if sh is not None else None, eh.data_ptr(), None, None,
                                     wu.data_ptr(), fi.data_ptr(), None)
                    barrier()
                    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    db2.process_device(bb, oo, stream.cuda_stream)          # the table persists: no reset between chunks
                    if world > 1:
                        db2.peer_allreduce_histogram_device(h2[: cfg2.n_issuers], cfg2.n_issuers, h2[cfg2.n_issuers:], stream.cuda_stream)
                    else:
                        db2.read_histogram_device(h2[: cfg2.n_issuers], cfg2.n_issuers, h2[cfg2.n_issuers:], stream.cuda_stream)
                    e1.record(stream)
                    torch.cuda.synchronize(dev)
                    tot_ms += e0.elapsed_time(e1)
                    tot_map += db2.profile_last()[0]
                    tot_bytes += tb
                    assert lib.ctmr_synth_truth_device(C.byref(cfg2), first_entry, nc, tid.data_ptr(), tna.data_ptr(), tbc.data_ptr(),
                                                       stream.cuda_stream) == 0
                    k_ok = st == 0
                    pr = (torch.ones_like(k_ok) if dd == 1 else ((tid % dd) == dd - 2)) if dd else torch.zeros_like(k_ok)
                    acc += torch.stack([k_ok.sum(), wu.sum(), (k_ok & pr).sum()]).long()
                    del bl, of, ix, ixd
                db2.check_device(stream.cuda_stream)
                kept, unk, kept_paired = allsum([int(x) for x in acc.tolist()])
                assert int(h2[: cfg2.n_issuers].sum()) == unk, f"{tag}: histogram sum != unknown entries"
                assert unk == kept - kept_paired // 2, f"{tag}: sum(was_unknown)={unk} != distinct kept certificates={kept - kept_paired // 2}"
                ms, mms = allmax(tot_ms), allmax(tot_map)
                total_entries = world * chunks * nc
                algb = tot_bytes + w2["out_bytes"] * chunks * nc
                nofp = bool(fl & capi.F_NO_FINGERPRINT)
                tr, trs = measured_traffic("map_light" if nofp else "map_stream", nc / R)
                rl = {"bound": "hbm" if nofp else "int_alu", "kernel": "map_light_kernel" if nofp else "map_stream_kernel",
                      "hbm": {"achieved": algb / (mms / 1e3) / 1e9, "peak": peak, "unit": "GB/s", "frac": algb / (mms / 1e3) / 1e9 / peak},
                      "kernel_ms_total": mms, "traffic_per_launch": tr, "traffic_source": trs}
                if not nofp and int_ceiling_gbs:
                    rl.update(achieved=tot_bytes / (mms / 1e3) / 1e9, peak=int_ceiling_gbs, unit="GB/s of message bytes",
                              frac=tot_bytes / (mms / 1e3) / 1e9 / int_ceiling_gbs)
                else:
                    rl.update(achieved=rl["hbm"]["achieved"], peak=peak, unit="GB/s", frac=rl["hbm"]["frac"])
                return {"name": tag, "workload": w2["desc"] + (" [fingerprint OFF: the reference never hashes the leaf]" if nofp else ""),
                        "entries": total_entries, "entries_per_gpu": chunks * nc, "chunks": chunks, "entries_per_chunk_per_gpu": nc,
                        "value": total_entries / (ms / 1e3), "unit": "entries/s", "seconds": ms / 1e3,
                        "kept": kept, "unknown": unk, "duplicates_found": kept - unk,
                        "table": "persistent across chunks (no reset), %d slots per GPU" % pow2(int(1.6 * chunks * nc)),
                        "checks": "sum(was_unknown) == distinct kept certificates (closed form over the complete corpus); histogram sum == unknown",
                        "roofline": rl}
            finally:
                db2.close()
                torch.cuda.empty_cache()

        per_gpu = args.secondary_entries or 125_000_000   # 1 B entries over 8 GPUs (configs[3], configs[4])
        plan = []
        if world == 1:
            plan.append(("configs[2] as written: 100M entries streamed through 1 GPU in 10 chunks", "cfg3", args.secondary_entries or 100_000_000, 0))
            plan.append(("configs[2], fingerprint off (reference-faithful: parse + filter + dedup + IssuerMetadata bits)", "cfg3",
                         args.secondary_entries or 100_000_000, capi.F_NO_FINGERPRINT))
        plan.append((f"configs[3] shape: {per_gpu * world / 1e6:.0f}M entries over {world} GPU(s)", "cfg4", per_gpu, 0))
        plan.append((f"configs[4] shape: {per_gpu * world / 1e6:.0f}M mixed-size entries, 50% duplicates, over {world} GPU(s)", "cfg5", per_gpu, 0))
        def frontend_run(n_raw, devices=None):
            """SURVEY.md §8(f)-2: get-entries response bodies (JSON, base64 leaf_input / extra_data; 2/3 x509 entries, 1/3 precert
            entries) through ctmr_process_raw -- or, with `devices`, through ctmr_group_process_raw on all of them from this one
            process: pinned host text in, host results out, every copy inside the timed calls."""
            from ct_mapreduce_b200 import frontend  # noqa: F401  (span finder; the pages here come with their spans)
            cfgr = capi.synth_cfg(n_raw, seed=SEED + 2)
            need = lib.ctmr_synth_raw_pages_host(C.byref(cfgr), 0, n_raw, 1000, None, 0, None, None, None, None)
            pin = capi.PinnedBuffer(need)
            lo_, ll_ = np.zeros(n_raw, np.uint64), np.zeros(n_raw, np.uint32)
            xo_, xl_ = np.zeros(n_raw, np.uint64), np.zeros(n_raw, np.uint32)
            assert lib.ctmr_synth_raw_pages_host(C.byref(cfgr), 0, n_raw, 1000, pin.addr, need, capi.ptr(lo_), capi.ptr(ll_), capi.ptr(xo_),
                                                 capi.ptr(xl_)) == need
            text = pin.view()
            if devices:
                dbr = engine.GpuCertGroup(devices, log_expired_entries=True, table_capacity=pow2(4 * n_raw // len(devices)), max_issuers=4096)
            else:
                dbr = engine.GpuCertDatabase(device=local, log_expired_entries=True, table_capacity=pow2(4 * n_raw), max_issuers=4096)
            try:
                fe_ms = path_ms = 0.0
                reps = 3
                for it in range(1 + reps):
                    if it == 1:
                        ts_ = time.perf_counter()
                    r_ = dbr.store_raw_entries(text, lo_, ll_, xo_, xl_, NOW_NS)
                    if it >= 1:
                        f_, p_, _ = (dbr.members[0] if devices else dbr).frontend_profile_last()
                        fe_ms += f_
                        path_ms += p_
                dt_ = (time.perf_counter() - ts_) / reps
                assert int((r_.entry_status == 0).sum()) == n_raw, "front end rejected synthetic entries"
                # replays of the same pages: everything is known the second time round
                assert int(r_.path.was_unknown.sum()) == 0
            finally:
                dbr.close()
                pin.free()
            chars = int(ll_.sum()) + int(xl_.sum())
            return {"name": ("get-entries pages through ctmr_group_process_raw on %d GPUs driven by one process (front end on the group path)" % len(devices))
                            if devices else "get-entries pages through ctmr_process_raw (CT wire-format front end, SURVEY 8(f)-2)", "entries": n_raw,
                    "value": n_raw / dt_, "unit": "entries/s", "seconds": dt_, "text_bytes": int(need), "h2d_gbs": need / dt_ / 1e9,
                    "frontend_kernels_ms": fe_ms / reps, "frontend_kernels_entries_per_sec": n_raw / (fe_ms / reps) * 1e3,
                    "frontend_kernels_chars_gbs": chars / (fe_ms / reps) / 1e6, "path_ms": path_ms / reps,
                    "note": "whole calls: pinned host text in (PCIe bound: ~5 KB of base64 per entry), host results out; base64 decode, TLS "
                            "framing, precert TBS check and Chain[0] identification on the GPU"
                            + ("; kernel split = member 0's chunks; the text sits on rank 0's NUMA node" if devices else "")}

        for tag, wn, pe, fl in plan:
            try:
                secondary.append(stream_run(tag, wn, pe, fl))
            except Exception as e:  # noqa: BLE001 -- a secondary must never take the primary line down; all ranks fail alike
                secondary.append({"name": tag, "error": f"{type(e).__name__}: {e}"[:300]})
                try:
                    torch.cuda.synchronize(dev)
                except Exception:
                    break
        n_raw = min(600_000, max(20_000, (args.secondary_entries or 100_000_000) // 100))
        if world == 1:
            try:
                secondary.append(frontend_run(n_raw))
            except Exception as e:  # noqa: BLE001
                secondary.append({"name": "ctmr_process_raw", "error": f"{type(e).__name__}: {e}"[:300]})
        else:
            # the front end on the multi-GPU path: the one-process group form, driven by rank 0 over every GPU of the job
            # while the other ranks wait on a CPU barrier (their GPUs are idle: nothing of theirs is resident any more)
            if rank == 0 and not same_gpu:
                try:
                    secondary.append(frontend_run(min(n_raw * world, 2_400_000), devices=list(range(world))))
                except Exception as e:  # noqa: BLE001
                    secondary.append({"name": "ctmr_group_process_raw", "error": f"{type(e).__name__}: {e}"[:300]})
                torch.cuda.set_device(local)   # the group's calls left another device current on this thread
            dist.barrier(group=cpu_group)

    if rank == 0:
        roofline = {"bound": "int_alu" if not args.no_fingerprint else "hbm",
                    "kernel": "map_light_kernel" if args.no_fingerprint else "map_stream_kernel<8,128,0,1>",
                    "hbm": {"achieved": hbm_achieved, "peak": peak, "unit": "GB/s", "frac": hbm_achieved / peak, "peak_source": peak_src,
                            "algorithmic_bytes_per_step": int(alg_bytes), "algorithmic_bytes_per_launch": int(alg_bytes / map_launches)},
                    "traffic": traffic, "traffic_source": traffic_src,
                    "kernel_ms_per_step": map_ms, "kernel_ms": map_ms / map_launches, "launches_per_step": map_launches}
        if args.no_fingerprint:
            roofline.update(achieved=hbm_achieved, peak=peak, unit="GB/s", frac=hbm_achieved / peak)
        else:
            roofline.update(achieved=sha_gbs_kernel, peak=int_ceiling_gbs, unit="GB/s", frac=sha_gbs_kernel / int_ceiling_gbs,
                            peak_source="register-only SHA-256 microbenchmark (ctmr_sha256_ceiling_device: K_map's own compression function, "
                                        "16 warps/SM, no memory traffic), run in this process",
                            note="whole-certificate SHA-256 is bound by the INT ALU pipe (rotations and boolean ops issue nowhere else), "
                                 "not by HBM: achieved = message bytes / K_map time against the measured ceiling of this instruction mix; "
                                 "`hbm` = the same kernel time against the measured HBM peak (SURVEY.md §8(d) algorithmic bytes)")
        line = {
            "metric": "ct_entries_per_sec", "value": value, "unit": "entries/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": elapsed_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32", "data": "synthetic",
            "config": {"workload": wl["desc"] + (" [fingerprint OFF: reference-faithful path]" if args.no_fingerprint else ""),
                       "entries_per_gpu_per_step": n, "bytes_per_gpu_per_step": int(total_bytes),
                       "issuers": cfg.n_issuers, "l2": "inputs (>=7 GB per step) far exceed the 126 MB L2; no explicit flush",
                       "parallelism": (f"entry-index shards x{world}; every set serials::<expDate>::<issuer> owned by one GPU, K_map inserts "
                                       f"into the owner's table over NVLink (peer atomics), {2 * map_launches} peer-memory barriers + 1 "
                                       "histogram all-reduce per step; no NCCL on the data path") if world > 1 else "single GPU",
                       "exactness": {"kept": n_ok, "unknown": n_unknown, "distinct_kept_expected": n_ok - n_ok_paired // 2,
                                     "cross_gpu_twin_pairs_checked": cross_rank_pairs, "oracle_sample_entries": oracle_sample}},
            "sha256_gbs": total_bytes * world * K / (elapsed_ms / 1e3) / 1e9,
            "roofline": roofline,
            "gpu_launches": launches_per_step * K,
            "clocks": clk,
        }
        if e2e:
            line["e2e"] = e2e
        if cpu:
            line["cpu_baseline"] = cpu
        if secondary:
            line["secondary"] = secondary
        print(json.dumps(line))
    if world > 1:
        try:  # the line is out: nothing below may keep the job from ending
            dist.barrier(group=cpu_group)
            dist.destroy_process_group()
        except Exception:  # noqa: BLE001
            pass
    return 0


if __name__ == "__main__":
    sys.exit(main())
