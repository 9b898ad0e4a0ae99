// ctmr_pipeline.cu -- the host-buffer batch of include/ctmr.h on one GPU, on a group of GPUs driven by one process
// (ctmr_group_*: what a Go host calls), and on one GPU of a multi-process group (ctmr_peer_*: one process per GPU).
//
// One pipeline serves all three.  A batch is cut into ROUNDS; in a round every member GPU takes one slice of at
// most `stage_entries` entries and runs, on the stream of the round's stage (three stages rotate, so H2D, kernels
// and D2H of consecutive rounds overlap):
//
//     H2D slice -> K_map (DER walk + filter + SHA-256 + key routing: a key of a set this GPU owns goes straight into
//                  its table, any other key is appended as a 64-byte record to the OWNER's inbox over NVLink)
//     -- sync 1: every member's appends of this round have landed --
//     owner passes: insert of the inbox records; K_resolve (was_unknown = "mine is the lowest index of the slot",
//                  per-issuer counts, (issuer, hour) first-seen + cardinality) and K_pairs (first_issuer_hour) over
//                  the own entries AND the inbox records, whose bits go to the owner's outbox
//     -- sync 2: every owner's bits of this round are ready --
//     pull of the bits of the entries routed away (contiguous peer reads) [-> string identities: insert, sync 3,
//                  read-back] -> D2H of the requested outputs [-> PEM]
//
// sync = nothing on one GPU; CUDA events recorded on every member's stream and waited for by every member's stream
// in a one-process group; a barrier kernel spinning on flags in peer memory between processes.  Rounds are ordered
// by a per-member chain (resolve of round k waits for resolve of round k-1), which with sync 1 gives the invariant
// the lowest-index-wins rule needs: when an entry is resolved, every entry with a lower global index has been inserted.
#include <sched.h>

#include <fstream>

#include "ctmr_ctx.cuh"

namespace ctmr_host {

// ------------------------------------------------------------------------------------------------ stages
int ensure_stages(ctmr_ctx* c) {
    if (c->stages_ready) return CTMR_OK;
    for (int k = 0; k < kStages; ++k) {
        Stage& s = c->stages[k];
        const uint64_t E = c->stage_entries;
        CU(c, cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
        CU(c, cudaEventCreateWithFlags(&s.mapped, cudaEventDisableTiming));
        CU(c, cudaEventCreateWithFlags(&s.reduced, cudaEventDisableTiming));
        CU(c, cudaEventCreateWithFlags(&s.meta_done, cudaEventDisableTiming));
        CU(c, cudaMalloc(&s.blob, c->stage_bytes + 64));
        // K_map stages records in 16-byte pieces, so its last copy may read up to 15 bytes past the slice's data (inside
        // this allocation, never consumed): written once here so that those bytes are defined (compute-sanitizer initcheck)
        CU(c, cudaMemsetAsync(s.blob, 0, c->stage_bytes + 64, s.stream));
        CU(c, cudaMalloc(&s.offsets, (E + 1) * sizeof(uint64_t)));
        CU(c, cudaMalloc(&s.issuer_idx, E * sizeof(uint32_t)));
        CU(c, cudaMalloc(&s.status, E));
        CU(c, cudaMalloc(&s.sha, E * 32));
        CU(c, cudaMalloc(&s.exp_hour, E * sizeof(int64_t)));
        CU(c, cudaMalloc(&s.serial_off, E * sizeof(uint32_t)));
        CU(c, cudaMalloc(&s.serial_len, E * sizeof(uint32_t)));
        CU(c, cudaMalloc(&s.was_unknown, E));
        CU(c, cudaMalloc(&s.first, E));
        CU(c, cudaMalloc(&s.keys, E * sizeof(ctmr_key)));
        CU(c, cudaMalloc(&s.slot_of, E * sizeof(uint32_t)));
        CU(c, cudaMalloc(&s.pair_slot, E * sizeof(uint32_t)));
        CU(c, cudaMalloc(&s.order, E * sizeof(uint32_t)));
        CU(c, cudaMalloc(&s.len_hist, 256 * sizeof(unsigned int)));
        CU(c, cudaMalloc(&s.spans, 4 * E * sizeof(uint32_t)));
        CU(c, cudaMalloc(&s.meta_slots, 2 * E * sizeof(uint32_t)));
        CU(c, cudaMalloc(&s.first_meta, 2 * E));
    }
    c->stages_ready = true;
    return CTMR_OK;
}

void stages_destroy(ctmr_ctx* c) {
    for (Stage& s : c->stages) {
        cudaFree(s.blob); cudaFree(s.offsets); cudaFree(s.issuer_idx); cudaFree(s.status); cudaFree(s.sha);
        cudaFree(s.exp_hour); cudaFree(s.serial_off); cudaFree(s.serial_len); cudaFree(s.was_unknown); cudaFree(s.first);
        cudaFree(s.keys); cudaFree(s.slot_of); cudaFree(s.pair_slot); cudaFree(s.order); cudaFree(s.len_hist); cudaFree(s.spans);
        cudaFree(s.meta_slots); cudaFree(s.first_meta);
        pem_free(s.pem);
        if (s.mapped) cudaEventDestroy(s.mapped);
        if (s.reduced) cudaEventDestroy(s.reduced);
        if (s.meta_done) cudaEventDestroy(s.meta_done);
        if (s.stream) cudaStreamDestroy(s.stream);
        s = Stage{};
    }
    c->stages_ready = false;
}

// ------------------------------------------------------------------------------------------------ PEM output
void pem_free(PemStage& ps) {
    cudaFree(ps.sizes); cudaFree(ps.off); cudaFree(ps.text); cudaFree(ps.scan_temp);
    ps = PemStage{};
}

int pem_ensure(ctmr_ctx* c, PemStage& ps, uint64_t entries, uint64_t der_bytes) {
    const uint64_t need_bytes = der_bytes / 3 * 4 + der_bytes / 48 + 64 * entries + 256;  // body + newlines + boundary lines
    if (ps.cap_entries >= entries && ps.cap_bytes >= need_bytes) return CTMR_OK;
    CU(c, cudaDeviceSynchronize());
    pem_free(ps);
    CU(c, cudaMalloc(&ps.sizes, (entries + 1) * 8));
    CU(c, cudaMalloc(&ps.off, (entries + 1) * 8));
    CU(c, cudaMalloc(&ps.text, need_bytes));
    ps.scan_temp_bytes = pem_scan_temp_bytes(entries + 1);
    CU(c, cudaMalloc(&ps.scan_temp, ps.scan_temp_bytes ? ps.scan_temp_bytes : 16));
    ps.cap_entries = entries;
    ps.cap_bytes = need_bytes;
    return CTMR_OK;
}

// Encodes the selected certificates of one chunk on `s`, waits for it, and appends the text to the caller's
// buffer at *base (host).  pem_off_out[i] (i < cnt) = absolute start of entry i's text.
int pem_chunk(ctmr_ctx* c, PemStage& ps, const uint8_t* blob, const uint64_t* offsets, const uint32_t* lens, const uint8_t* select,
              uint64_t cnt, const ctmr_out* out, uint64_t first, uint64_t* base, cudaStream_t s) {
    CU(c, launch_pem_encode(blob, offsets, lens, select, cnt, ps.sizes, ps.scan_temp, ps.scan_temp_bytes, ps.off, ps.text, ps.cap_bytes,
                            c->st.error_flag, c->sm_count, s));
    ps.host_off.resize(cnt + 1);
    CU(c, cudaMemcpyAsync(ps.host_off.data(), ps.off, (cnt + 1) * 8, cudaMemcpyDeviceToHost, s));
    CU(c, cudaStreamSynchronize(s));
    const uint64_t total = ps.host_off[cnt];
    if (total > ps.cap_bytes) return fail(c, CTMR_E_BATCH_TOO_LARGE, "PEM staging too small (internal sizing)");
    if (*base + total > out->pem_cap) return fail(c, CTMR_E_BATCH_TOO_LARGE, "ctmr_out.pem_cap too small for the new certificates' PEM");
    if (total) CU(c, cudaMemcpyAsync(out->pem + *base, ps.text, total, cudaMemcpyDeviceToHost, s));
    for (uint64_t i = 0; i < cnt; ++i) out->pem_off[first + i] = *base + ps.host_off[i];
    *base += total;
    return CTMR_OK;
}

}  // namespace ctmr_host

namespace {

struct BatchArgs {
    const uint8_t* blob;
    const uint64_t* offsets;
    uint64_t n;
    const uint32_t* issuer_idx;
    uint32_t n_issuers;
    int64_t now_unix_ns;
    ctmr_out* out;
};

struct Slice {
    uint64_t lo = 0, hi = 0;      // entries of the caller's batch
    uint64_t first_index = 0;     // global index of entry lo
};


// rounds x members.  Every slice respects the entry budget and the byte budget of a stage.
int plan_rounds(ctmr_ctx* c0, uint32_t W, const BatchArgs& a, std::vector<std::vector<Slice>>& plan) {
    const uint64_t E = c0->stage_entries, B = c0->stage_bytes;
    uint64_t pos = 0;
    while (pos < a.n) {
        uint64_t q = std::min<uint64_t>(E, (a.n - pos + W - 1) / W);
        for (;;) {  // shrink until every member's slice fits the byte budget
            bool fits = true;
            for (uint32_t r = 0; r < W && fits; ++r) {
                const uint64_t lo = std::min(a.n, pos + r * q), hi = std::min(a.n, pos + (r + 1) * q);
                fits = a.offsets[hi] - a.offsets[lo] <= B;
            }
            if (fits) break;
            if (q == 1) return fail(c0, CTMR_E_BATCH_TOO_LARGE, "a single entry exceeds the staging budget (config.max_batch_bytes)");
            q = (q + 1) / 2;
        }
        std::vector<Slice> round(W);
        for (uint32_t r = 0; r < W; ++r) {
            round[r].lo = std::min(a.n, pos + r * q);
            round[r].hi = std::min(a.n, pos + (r + 1) * q);
        }
        plan.push_back(std::move(round));
        pos = std::min(a.n, pos + W * q);
    }
    return CTMR_OK;
}

// multi-process group: the ranks agree on the number of rounds of this collective call (the largest any rank needs)
int agree_rounds(ctmr_ctx* c, uint64_t mine, uint64_t* agreed) {
    CU(c, launch_peer_post(c->pf, mine, c->stream));
    int rc = peer_barrier(c, CH_MAILBOX, c->stream);
    if (rc) return rc;
    unsigned long long row[kMaxWorld] = {};
    CU(c, cudaMemcpyAsync(row, c->pf.flags[c->pf.rank] + (size_t)kPeerChannels * kMaxWorld, sizeof row, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    rc = ctmr_check_device(c, nullptr);
    if (rc) return rc;
    uint64_t mx = mine;
    for (uint32_t r = 0; r < c->pf.world; ++r) mx = std::max<uint64_t>(mx, row[r]);
    *agreed = mx ? mx : 1;  // at least one round: its barriers also fence the mailbox against the next call
    return CTMR_OK;
}

int issue_map(ctmr_ctx* c, Stage& s, int sidx, const BatchArgs& a, const Slice& sl, const uint32_t* map_dev, bool want_meta) {
    CU(c, cudaSetDevice(c->device));
    const uint64_t cnt = sl.hi - sl.lo;
    const bool fused = c->fuse_insert || c->px.world > 1;  // a group always fuses: the routing is K_map's epilogue
    int rc = round_begin(c, sidx, s.stream);  // exchange parity = stage
    if (rc) return rc;
    if (cnt) {
        const uint64_t bytes = a.offsets[sl.hi] - a.offsets[sl.lo];
        if (bytes) CU(c, cudaMemcpyAsync(s.blob, a.blob + a.offsets[sl.lo], bytes, cudaMemcpyHostToDevice, s.stream));
        CU(c, cudaMemcpyAsync(s.offsets, a.offsets + sl.lo, (cnt + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, s.stream));
        if (a.issuer_idx) CU(c, cudaMemcpyAsync(s.issuer_idx, a.issuer_idx + sl.lo, cnt * sizeof(uint32_t), cudaMemcpyHostToDevice, s.stream));
        ctmr_dev_batch db{};
        db.blob = s.blob - a.offsets[sl.lo];  // offsets stay absolute
        db.blob_bytes = a.offsets[sl.hi];
        db.offsets = s.offsets;
        db.n = cnt;
        db.issuer_idx = a.issuer_idx ? s.issuer_idx : nullptr;
        db.issuer_map = map_dev;
        db.issuer_map_len = a.n_issuers;
        db.first_index = sl.first_index;
        db.now_unix_ns = a.now_unix_ns;
        ctmr_dev_out dout{};
        dout.status = s.status;
        dout.sha256 = a.out->sha256 ? s.sha : nullptr;
        dout.exp_hour = s.exp_hour;
        dout.serial_off = s.serial_off;
        dout.serial_len = s.serial_len;
        dout.keys = s.keys;
        const uint64_t E = c->stage_entries;
        if (want_meta) {
            dout.issuer_name_off = s.spans;
            dout.issuer_name_len = s.spans + E;
            dout.crldp_off = s.spans + 2 * E;
            dout.crldp_len = s.spans + 3 * E;
        }
        MapParams p;
        fill_map_params(c, &db, &dout, p, sidx, fused ? s.slot_of : nullptr, sidx);
        if (c->bucket_by_length && cnt > 64 && p.sha256) {
            CU(c, launch_len_order(s.offsets, nullptr, cnt, db.blob_bytes, s.len_hist, s.order, s.stream));
            p.order = s.order;
        }
        CU(c, launch_map(p, c->sm_count, s.stream));
        // inserts commute (atomic max on ~index); only RESOLVE must see every earlier entry inserted
        if (!fused) CU(c, launch_insert(c->st, s.keys, cnt, s.slot_of, s.stream));
    }
    rc = round_publish(c, sidx, s.stream);  // how many records this rank left in each owner's inbox
    if (rc) return rc;
    CU(c, cudaEventRecord(s.mapped, s.stream));
    return CTMR_OK;
}

// the owner's work of a round: the records other ranks left in its inbox and its own entries' keys
int issue_owner_insert(ctmr_ctx* c, Stage& s, int sidx) {
    return round_owner_insert(c, sidx, c->stage_entries, s.stream);
}

int issue_resolve(ctmr_ctx* c, Stage& s, int sidx, const Slice& sl) {
    const uint64_t cnt = sl.hi - sl.lo;
    if (cnt) CU(c, launch_resolve(c->st, s.keys, cnt, s.slot_of, s.pair_slot, s.was_unknown, s.stream));
    int rc = round_owner_resolve(c, sidx, c->stage_entries, s.stream);
    if (rc) return rc;
    if (cnt) CU(c, launch_resolve_pairs(c->st, s.keys, cnt, s.pair_slot, s.was_unknown, s.first, s.stream));
    rc = round_owner_pairs(c, sidx, c->stage_entries, s.stream);
    if (rc) return rc;
    CU(c, cudaEventRecord(s.reduced, s.stream));
    return CTMR_OK;
}

// string identities of the new certificates: insert (needs this rank's was_unknown bits, i.e. the pull), then -- after
// every rank's inserts -- the read-back
int issue_meta_insert(ctmr_ctx* c, Stage& s, const BatchArgs& a, const Slice& sl) {
    const uint64_t cnt = sl.hi - sl.lo, E = c->stage_entries;
    if (cnt)
        CU(c, launch_meta_insert(c->st, s.blob - a.offsets[sl.lo], s.offsets, s.keys, cnt, s.was_unknown, s.spans, s.spans + E,
                                 s.spans + 2 * E, s.spans + 3 * E, s.meta_slots, s.stream));
    CU(c, cudaEventRecord(s.meta_done, s.stream));
    return CTMR_OK;
}

int issue_finish(ctmr_ctx* c, Stage& s, const BatchArgs& a, const Slice& sl, bool want_meta, bool want_pem, uint64_t* pem_base) {
    const uint64_t cnt = sl.hi - sl.lo, lo = sl.lo, E = c->stage_entries;
    const ctmr_out* out = a.out;
    if (!cnt) return CTMR_OK;
    if (want_meta) {
        CU(c, launch_meta_resolve(c->st, s.keys, cnt, s.meta_slots, s.first_meta, s.first_meta + E, s.stream));
        if (out->issuer_name_off) CU(c, cudaMemcpyAsync(out->issuer_name_off + lo, s.spans, cnt * 4, cudaMemcpyDeviceToHost, s.stream));
        if (out->issuer_name_len) CU(c, cudaMemcpyAsync(out->issuer_name_len + lo, s.spans + E, cnt * 4, cudaMemcpyDeviceToHost, s.stream));
        if (out->crldp_off) CU(c, cudaMemcpyAsync(out->crldp_off + lo, s.spans + 2 * E, cnt * 4, cudaMemcpyDeviceToHost, s.stream));
        if (out->crldp_len) CU(c, cudaMemcpyAsync(out->crldp_len + lo, s.spans + 3 * E, cnt * 4, cudaMemcpyDeviceToHost, s.stream));
        if (out->first_issuer_dn) CU(c, cudaMemcpyAsync(out->first_issuer_dn + lo, s.first_meta, cnt, cudaMemcpyDeviceToHost, s.stream));
        if (out->first_crldp) CU(c, cudaMemcpyAsync(out->first_crldp + lo, s.first_meta + E, cnt, cudaMemcpyDeviceToHost, s.stream));
    }
    if (out->status) CU(c, cudaMemcpyAsync(out->status + lo, s.status, cnt, cudaMemcpyDeviceToHost, s.stream));
    if (out->sha256) CU(c, cudaMemcpyAsync(out->sha256 + lo * 32, s.sha, cnt * 32, cudaMemcpyDeviceToHost, s.stream));
    if (out->exp_hour) CU(c, cudaMemcpyAsync(out->exp_hour + lo, s.exp_hour, cnt * sizeof(int64_t), cudaMemcpyDeviceToHost, s.stream));
    if (out->serial_off) CU(c, cudaMemcpyAsync(out->serial_off + lo, s.serial_off, cnt * sizeof(uint32_t), cudaMemcpyDeviceToHost, s.stream));
    if (out->serial_len) CU(c, cudaMemcpyAsync(out->serial_len + lo, s.serial_len, cnt * sizeof(uint32_t), cudaMemcpyDeviceToHost, s.stream));
    if (out->was_unknown) CU(c, cudaMemcpyAsync(out->was_unknown + lo, s.was_unknown, cnt, cudaMemcpyDeviceToHost, s.stream));
    if (out->first_issuer_hour) CU(c, cudaMemcpyAsync(out->first_issuer_hour + lo, s.first, cnt, cudaMemcpyDeviceToHost, s.stream));
    if (want_pem) {  // StoreCertificatePEM's argument for this slice's new certificates (the host waits for this slice here)
        int rc = pem_ensure(c, s.pem, c->stage_entries, c->stage_bytes);
        if (rc) return rc;
        rc = pem_chunk(c, s.pem, s.blob - a.offsets[lo], s.offsets, nullptr, s.was_unknown, cnt, out, lo, pem_base, s.stream);
        if (rc) return rc;
    }
    return CTMR_OK;
}

// The pipeline.  m[0..W) = the member GPUs this process drives (W == 1: a plain ctx, or one rank of a multi-process
// group).  `plan` rows beyond a rank's own rounds are empty slices (multi-process: every rank runs the agreed number).
int run_rounds(ctmr_ctx** m, uint32_t W, const BatchArgs& a, const std::vector<std::vector<Slice>>& plan,
               const std::vector<const uint32_t*>& map_dev, ctmr_ctx** failed) {
    const ctmr_out* out = a.out;
    const bool want_meta = out->first_issuer_dn || out->first_crldp || out->issuer_name_off || out->crldp_off;
    const bool want_pem = out->pem != nullptr || out->pem_off != nullptr;
    uint64_t pem_base = 0;
    int rc = CTMR_OK;
#define RR(r, call)                 \
    do {                            \
        rc = (call);                \
        if (rc) {                   \
            *failed = m[r];         \
            return rc;              \
        }                           \
    } while (0)
    for (size_t k = 0; k < plan.size(); ++k) {
        const int sidx = (int)(k % kStages);
        for (uint32_t r = 0; r < W; ++r)  // ---- upload + map + insert at the owners
            RR(r, issue_map(m[r], m[r]->stages[sidx], sidx, a, plan[k][r], map_dev[r], want_meta));
        for (uint32_t r = 0; r < W; ++r) {  // ---- sync 1 (every member's appends have landed), then the owners' passes
            ctmr_ctx* c = m[r];
            Stage& s = c->stages[sidx];
            *failed = c;
            CU(c, cudaSetDevice(c->device));
            for (uint32_t q = 0; q < W; ++q)
                if (q != r) CU(c, cudaStreamWaitEvent(s.stream, m[q]->stages[sidx].mapped, 0));
            RR(r, peer_barrier(c, CH_STAGE_MAP + sidx, s.stream));
            RR(r, issue_owner_insert(c, s, sidx));
            if (k > 0) CU(c, cudaStreamWaitEvent(s.stream, c->stages[(k - 1) % kStages].reduced, 0));  // the chain of rounds
            RR(r, issue_resolve(c, s, sidx, plan[k][r]));
        }
        for (uint32_t r = 0; r < W; ++r) {  // ---- sync 2 (the owners have the bits ready), pull, [string identities]
            ctmr_ctx* c = m[r];
            Stage& s = c->stages[sidx];
            *failed = c;
            CU(c, cudaSetDevice(c->device));
            for (uint32_t q = 0; q < W; ++q)
                if (q != r) CU(c, cudaStreamWaitEvent(s.stream, m[q]->stages[sidx].reduced, 0));
            RR(r, peer_barrier(c, CH_STAGE_RESOLVE + sidx, s.stream));
            RR(r, round_pull(c, sidx, c->stage_entries, s.was_unknown, s.first, s.stream));
            if (want_meta) {
                if (k > 0) CU(c, cudaStreamWaitEvent(s.stream, c->stages[(k - 1) % kStages].meta_done, 0));  // their own chain of rounds
                RR(r, issue_meta_insert(c, s, a, plan[k][r]));
            }
        }
        for (uint32_t r = 0; r < W; ++r) {  // ---- [sync 3: every member's string identities are in], outputs
            ctmr_ctx* c = m[r];
            Stage& s = c->stages[sidx];
            *failed = c;
            CU(c, cudaSetDevice(c->device));
            if (want_meta) {
                for (uint32_t q = 0; q < W; ++q)
                    if (q != r) CU(c, cudaStreamWaitEvent(s.stream, m[q]->stages[sidx].meta_done, 0));
                RR(r, peer_barrier(c, CH_STAGE_META + sidx, s.stream));
            }
            RR(r, issue_finish(c, s, a, plan[k][r], want_meta, want_pem, &pem_base));
        }
    }
#undef RR
    for (uint32_t r = 0; r < W; ++r) {
        *failed = m[r];
        CU(m[r], cudaSetDevice(m[r]->device));
        for (int k = 0; k < kStages; ++k) CU(m[r], cudaStreamSynchronize(m[r]->stages[k].stream));
    }
    if (want_pem) out->pem_off[a.n] = pem_base;
    for (uint32_t r = 0; r < W; ++r) {
        *failed = m[r];
        rc = ctmr_check_device(m[r], nullptr);
        if (rc) return rc;
    }
    *failed = nullptr;
    return CTMR_OK;
}

// no copy from / into the caller's buffers may outlive a failed call
void drain(ctmr_ctx** m, uint32_t W) {
    for (uint32_t r = 0; r < W; ++r) {
        ctmr_ctx* c = m[r];
        if (!c->stages_ready) continue;
        const std::string keep = c->err;
        cudaSetDevice(c->device);
        for (Stage& s : c->stages) cudaStreamSynchronize(s.stream);
        c->err = keep;
    }
}

int process_batch_members(ctmr_ctx** m, uint32_t W, uint64_t* next_index, const uint8_t* blob, const uint64_t* offsets, uint64_t n,
                          const uint8_t* issuer_blob, const uint64_t* issuer_offsets, uint32_t n_issuers, const uint32_t* issuer_idx,
                          int64_t now_unix_ns, ctmr_out* out, ctmr_ctx** failed) {
    ctmr_ctx* c0 = m[0];
    *failed = c0;
    if (!out || (n && (!blob || !offsets))) return fail(c0, CTMR_E_INVALID, "bad argument");
    const bool ipc = c0->peer_mode == PEER_IPC && c0->st.peer.world > 1;
    if (n == 0 && !ipc) {
        *failed = nullptr;
        return CTMR_OK;
    }
    if ((out->pem != nullptr) != (out->pem_off != nullptr)) return fail(c0, CTMR_E_INVALID, "pem and pem_off go together");
    int rc;
    for (uint32_t r = 0; r < W; ++r) {
        *failed = m[r];
        CU(m[r], cudaSetDevice(m[r]->device));
        rc = ensure_stages(m[r]);
        if (rc) return rc;
    }
    *failed = c0;
    // issuers of this batch -> dense indices (GPU work only for certificates never seen before); the registry is
    // shared by the group, so member 0's answer holds for every member
    std::vector<const uint32_t*> map_dev(W, nullptr);
    if (n_issuers) {
        std::vector<uint32_t> dense(n_issuers);
        rc = ctmr_register_issuers(c0, issuer_blob, issuer_offsets, n_issuers, dense.data());
        if (rc) return rc;
        for (uint32_t r = 0; r < W; ++r) {
            *failed = m[r];
            CU(m[r], cudaSetDevice(m[r]->device));
            rc = upload_issuer_map(m[r], dense.data(), n_issuers);
            if (rc) return rc;
            map_dev[r] = m[r]->issuer_map_dev;
        }
        *failed = c0;
    }
    BatchArgs a{blob, offsets, n, issuer_idx, n_issuers, now_unix_ns, out};
    std::vector<std::vector<Slice>> plan;
    rc = plan_rounds(c0, W, a, plan);
    if (rc) return rc;
    uint64_t advance = n;
    if (ipc) {
        // collective call: the agreed number of rounds, each rank's round k at (k * world + rank) * E above the base
        const uint32_t world = c0->st.peer.world, rank = c0->st.peer.rank;
        uint64_t rounds = 0;
        rc = agree_rounds(c0, plan.size(), &rounds);
        if (rc) return rc;
        plan.resize(rounds, std::vector<Slice>(1));
        for (uint64_t k = 0; k < rounds; ++k) {
            if (plan[k][0].hi == plan[k][0].lo) plan[k][0].lo = plan[k][0].hi = n;  // an empty round
            plan[k][0].first_index = *next_index + (k * world + rank) * c0->stage_entries;
        }
        advance = rounds * world * c0->stage_entries;
    } else {
        for (auto& round : plan)
            for (auto& sl : round) sl.first_index = *next_index + sl.lo;  // entry i of the batch = global index base + i
    }
    rc = run_rounds(m, W, a, plan, map_dev, failed);
    // Also after a failure: some rounds may have been inserted, and a retry must not find itself "first" again with
    // the same indices (its entries then read as known, which is what they are).
    *next_index += advance;
    if (rc) drain(m, W);
    return rc;
}

}  // namespace

// =================================================================================================
extern "C" {

int ctmr_process_batch(ctmr_ctx* c, const uint8_t* blob, const uint64_t* offsets, uint64_t n, const uint8_t* issuer_blob,
                       const uint64_t* issuer_offsets, uint32_t n_issuers, const uint32_t* issuer_idx, int64_t now_unix_ns,
                       ctmr_out* out) {
    if (!c) return CTMR_E_INVALID;
    if (c->group) return fail(c, CTMR_E_INVALID, "member of a group: use ctmr_group_process_batch");
    ctmr_ctx* failed = nullptr;
    return process_batch_members(&c, 1, &c->next_index, blob, offsets, n, issuer_blob, issuer_offsets, n_issuers, issuer_idx, now_unix_ns,
                                 out, &failed);
}

// ------------------------------------------------------------------------------------------------ one process, several GPUs
int ctmr_group_create(const ctmr_config* cfg, const int32_t* devices, uint32_t n_devices, ctmr_group** out) {
    if (!cfg || !devices || !out || n_devices == 0 || n_devices > kMaxWorld || cfg->struct_size < sizeof(ctmr_config))
        return fail(nullptr, CTMR_E_INVALID, "bad group configuration (1..8 devices)");
    *out = nullptr;
    ctmr_group* g = new (std::nothrow) ctmr_group();
    if (!g) return fail(nullptr, CTMR_E_NOMEM, "host allocation failed");
    auto bail = [&](int code, const std::string& msg) {
        ctmr_group_destroy(g);
        return fail(nullptr, code, msg);
    };
    for (uint32_t r = 0; r < n_devices; ++r) {
        ctmr_config mc = *cfg;
        mc.device = devices[r];
        ctmr_ctx* c = nullptr;
        const int rc = ctmr_create(&mc, &c);
        if (rc) return bail(rc, ctmr_last_error(nullptr));
        c->group = g;
        g->m.push_back(c);
    }
    // peer access between the distinct devices (NVLink through NVSwitch on a B200 box)
    for (uint32_t r = 0; r < n_devices; ++r)
        for (uint32_t q = 0; q < n_devices; ++q) {
            if (devices[r] == devices[q]) continue;
            int can = 0;
            if (cudaDeviceCanAccessPeer(&can, devices[r], devices[q]) != cudaSuccess || !can)
                return bail(CTMR_E_PEER, "GPUs " + std::to_string(devices[r]) + " and " + std::to_string(devices[q]) + " cannot access each other's memory");
            cudaSetDevice(devices[r]);
            const cudaError_t e = cudaDeviceEnablePeerAccess(devices[q], 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return bail(CTMR_E_PEER, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e));
            (void)cudaGetLastError();
        }
    if (n_devices > 1) {
        uint8_t *bases[kMaxWorld] = {}, *xb[kMaxWorld] = {};
        for (uint32_t r = 0; r < n_devices; ++r) {
            cudaSetDevice(devices[r]);
            const int rc = alloc_exchange(g->m[r], n_devices);
            if (rc) return bail(rc, g->m[r]->err);
            bases[r] = g->m[r]->shared;
            xb[r] = g->m[r]->xchg;
        }
        for (uint32_t r = 0; r < n_devices; ++r) {
            attach_views(g->m[r], bases, n_devices, r);
            attach_exchange(g->m[r], xb, n_devices, r);
            g->m[r]->peer_mode = PEER_GROUP;
        }
    }
    *out = g;
    return CTMR_OK;
}

void ctmr_group_destroy(ctmr_group* g) {
    if (!g) return;
    for (ctmr_ctx* c : g->m) {  // quiesce every member before any shard goes away
        cudaSetDevice(c->device);
        cudaDeviceSynchronize();
    }
    for (ctmr_ctx* c : g->m) ctmr_destroy(c);
    delete g;
}

const char* ctmr_group_last_error(ctmr_group* g) { return g ? g->err.c_str() : g_create_error.c_str(); }
uint32_t ctmr_group_size(ctmr_group* g) { return g ? (uint32_t)g->m.size() : 0; }
ctmr_ctx* ctmr_group_member(ctmr_group* g, uint32_t rank) { return g && rank < g->m.size() ? g->m[rank] : nullptr; }

int ctmr_group_process_batch(ctmr_group* g, const uint8_t* blob, const uint64_t* offsets, uint64_t n, const uint8_t* issuer_blob,
                             const uint64_t* issuer_offsets, uint32_t n_issuers, const uint32_t* issuer_idx, int64_t now_unix_ns,
                             ctmr_out* out) {
    if (!g || g->m.empty()) return CTMR_E_INVALID;
    ctmr_ctx* failed = nullptr;
    const int rc = process_batch_members(g->m.data(), (uint32_t)g->m.size(), &g->next_index, blob, offsets, n, issuer_blob, issuer_offsets,
                                         n_issuers, issuer_idx, now_unix_ns, out, &failed);
    return rc ? group_fail(g, failed ? failed : g->m[0], rc) : rc;
}

int ctmr_group_issuer_counts(ctmr_group* g, uint8_t* digests, uint64_t* counts, size_t* n) {
    if (!g || g->m.empty() || !n) return CTMR_E_INVALID;
    const size_t cap = *n;
    std::vector<uint64_t> part(cap ? cap : 1);
    size_t take = 0;
    for (size_t r = 0; r < g->m.size(); ++r) {
        size_t k = cap;
        const int rc = ctmr_issuer_counts(g->m[r], r == 0 ? digests : nullptr, part.data(), &k);
        if (rc) return group_fail(g, g->m[r], rc);
        if (r == 0) {
            take = k;
            if (counts) std::copy(part.begin(), part.begin() + k, counts);
        } else if (counts) {
            // unsigned wrap-around on purpose: TTL eviction subtracts at the owner what the home rank added
            for (size_t i = 0; i < std::min(k, take); ++i) counts[i] += part[i];
        }
    }
    *n = take;
    return CTMR_OK;
}

int ctmr_group_set_cardinality(ctmr_group* g, int64_t exp_hour, const uint8_t issuer_digest[32], uint64_t* count_out) {
    if (!g || g->m.empty()) return CTMR_E_INVALID;
    const int rc = ctmr_set_cardinality(g->m[0], exp_hour, issuer_digest, count_out);  // probes the owner's slot over peer memory
    return rc ? group_fail(g, g->m[0], rc) : rc;
}

int ctmr_group_status_counters(ctmr_group* g, uint64_t out[CTMR_ST__COUNT]) {
    if (!g || g->m.empty() || !out) return CTMR_E_INVALID;
    uint64_t part[CTMR_ST__COUNT];
    std::fill(out, out + CTMR_ST__COUNT, 0);
    for (ctmr_ctx* c : g->m) {
        const int rc = ctmr_status_counters(c, part);
        if (rc) return group_fail(g, c, rc);
        for (int i = 0; i < CTMR_ST__COUNT; ++i) out[i] += part[i];
    }
    return CTMR_OK;
}

int ctmr_group_table_stats(ctmr_group* g, uint64_t* slots_used, uint64_t* capacity) {
    if (!g || g->m.empty()) return CTMR_E_INVALID;
    uint64_t u = 0, cp = 0;
    for (ctmr_ctx* c : g->m) {
        uint64_t a = 0, b = 0;
        const int rc = ctmr_table_stats(c, &a, &b);
        if (rc) return group_fail(g, c, rc);
        u += a;
        cp += b;
    }
    if (slots_used) *slots_used = u;
    if (capacity) *capacity = cp;
    return CTMR_OK;
}

int ctmr_group_preload_known(ctmr_group* g, int64_t exp_hour, const uint8_t issuer_digest[32], const uint8_t* serial_blob,
                             const uint64_t* serial_offsets, uint64_t n) {
    if (!g || g->m.empty() || !issuer_digest || (n && (!serial_blob || !serial_offsets))) return CTMR_E_INVALID;
    // the set's owner shard receives the serials (every table operation is local to the owner)
    uint32_t issuer = 0;
    bool found = false;
    cudaSetDevice(g->m[0]->device);
    int rc = lookup_digest(g->m[0], issuer_digest, true, &issuer, &found);
    if (rc) return group_fail(g, g->m[0], rc);
    if (exp_hour > INT32_MAX || exp_hour < INT32_MIN) return group_fail(g, g->m[0], fail(g->m[0], CTMR_E_INVALID, "exp_hour out of range"));
    ctmr_ctx* owner = g->m[key_owner((int32_t)exp_hour, issuer, (uint32_t)g->m.size())];
    rc = preload_impl(owner, exp_hour, issuer_digest, serial_blob, serial_offsets, n, g->next_index);
    if (rc) return group_fail(g, owner, rc);
    g->next_index += n;
    return CTMR_OK;
}

int ctmr_group_evict_expired(ctmr_group* g, int64_t now_unix_sec, uint64_t* evicted_out) {
    if (!g || g->m.empty()) return CTMR_E_INVALID;
    uint64_t total = 0;
    for (ctmr_ctx* c : g->m) {  // every shard drops the expired sets it owns
        uint64_t e = 0;
        const int rc = ctmr_evict_expired(c, now_unix_sec, &e);
        if (rc) return group_fail(g, c, rc);
        total += e;
    }
    if (evicted_out) *evicted_out = total;
    return CTMR_OK;
}

// Snapshot of a whole group: every shard's tables and histograms + the one issuer registry + the group's next index.
namespace {
struct GroupSnapHeader {
    char magic[8];  // "CTMRGRP1"
    uint64_t members, shard_bytes, table_slots, max_issuers, n_issuers, next_index;
};
}  // namespace

int ctmr_group_snapshot_size(ctmr_group* g, uint64_t* bytes) {
    if (!g || g->m.empty() || !bytes) return CTMR_E_INVALID;
    ctmr_ctx* c0 = g->m[0];
    cudaSetDevice(c0->device);
    const int rc = refresh_digests(c0);
    if (rc) return group_fail(g, c0, rc);
    *bytes = sizeof(GroupSnapHeader) + g->m.size() * snap_shard_bytes(c0) + c0->digests.size() * 32;
    return CTMR_OK;
}

int ctmr_group_snapshot_save(ctmr_group* g, uint8_t* buf, uint64_t cap, uint64_t* written) {
    uint64_t need = 0;
    int rc = ctmr_group_snapshot_size(g, &need);
    if (rc) return rc;
    ctmr_ctx* c0 = g->m[0];
    if (!buf || cap < need) return group_fail(g, c0, fail(c0, CTMR_E_INVALID, "snapshot buffer too small"));
    GroupSnapHeader h{};
    std::memcpy(h.magic, "CTMRGRP1", 8);
    h.members = g->m.size();
    h.shard_bytes = snap_shard_bytes(c0);
    h.table_slots = c0->st.table_mask + 1;
    h.max_issuers = c0->st.max_issuers;
    h.n_issuers = c0->digests.size();
    h.next_index = g->next_index;
    uint8_t* p = buf;
    std::memcpy(p, &h, sizeof h); p += sizeof h;
    for (ctmr_ctx* c : g->m) {
        rc = snap_shard_save(c, p);
        if (rc) return group_fail(g, c, rc);
        p += h.shard_bytes;
    }
    for (const auto& d : c0->digests) { std::memcpy(p, d.data(), 32); p += 32; }
    if (written) *written = (uint64_t)(p - buf);
    return CTMR_OK;
}

int ctmr_group_snapshot_load(ctmr_group* g, const uint8_t* buf, uint64_t bytes) {
    if (!g || g->m.empty()) return CTMR_E_INVALID;
    ctmr_ctx* c0 = g->m[0];
    GroupSnapHeader h;
    if (!buf || bytes < sizeof h) return group_fail(g, c0, fail(c0, CTMR_E_INVALID, "bad snapshot"));
    std::memcpy(&h, buf, sizeof h);
    if (std::memcmp(h.magic, "CTMRGRP1", 8) != 0) return group_fail(g, c0, fail(c0, CTMR_E_INVALID, "not a ctmr group snapshot"));
    // the owner of a set depends on the group size: a snapshot only fits a group of the same shape
    if (h.members != g->m.size() || h.shard_bytes != snap_shard_bytes(c0) || h.table_slots != c0->st.table_mask + 1 ||
        h.max_issuers != c0->st.max_issuers || h.n_issuers > h.max_issuers)
        return group_fail(g, c0, fail(c0, CTMR_E_INVALID, "snapshot was taken by a group of another size or with other capacities"));
    if (bytes < sizeof h + h.members * h.shard_bytes + h.n_issuers * 32) return group_fail(g, c0, fail(c0, CTMR_E_INVALID, "truncated snapshot"));
    const uint8_t* p = buf + sizeof h;
    for (ctmr_ctx* c : g->m) {
        const int rc = snap_shard_load(c, p);
        if (rc) return group_fail(g, c, rc);
        p += h.shard_bytes;
    }
    const int rc = snap_registry_restore(c0, p, h.n_issuers);
    if (rc) return group_fail(g, c0, rc);
    g->next_index = h.next_index;
    return CTMR_OK;
}

int ctmr_group_reset(ctmr_group* g) {
    if (!g || g->m.empty()) return CTMR_E_INVALID;
    for (ctmr_ctx* c : g->m) {
        cudaSetDevice(c->device);
        cudaDeviceSynchronize();
    }
    for (ctmr_ctx* c : g->m) {
        int rc = ctmr_reset_device(c, nullptr);
        if (rc) return group_fail(g, c, rc);
        if (cudaStreamSynchronize(c->stream) != cudaSuccess) return group_fail(g, c, fail(c, CTMR_E_CUDA, "reset failed"));
    }
    return CTMR_OK;
}

// ------------------------------------------------------------------------------------------------ one process per GPU
namespace {
struct PeerHandle {
    char magic[8];  // "CTMRPEER"
    cudaIpcMemHandle_t mem, xchg;
    uint64_t table_slots, pair_slots, meta_slots, total, X;
    uint32_t max_issuers, world;
};
static_assert(sizeof(PeerHandle) <= CTMR_PEER_HANDLE_BYTES, "peer handle size");
}  // namespace

int ctmr_peer_export(ctmr_ctx* c, uint32_t world, uint8_t handle_out[CTMR_PEER_HANDLE_BYTES]) {
    if (!c || !handle_out || world == 0 || world > kMaxWorld) return fail(c, CTMR_E_INVALID, "bad argument (1..8 ranks)");
    if (c->peer_mode != PEER_NONE || c->group) return fail(c, CTMR_E_INVALID, "ctx already belongs to a group");
    CU(c, cudaSetDevice(c->device));
    PeerHandle h{};
    std::memcpy(h.magic, "CTMRPEER", 8);
    cudaError_t e = cudaIpcGetMemHandle(&h.mem, c->shared);
    if (e != cudaSuccess) return fail(c, CTMR_E_PEER, std::string("cudaIpcGetMemHandle: ") + cudaGetErrorString(e));
    if (world > 1) {
        if (c->xchg && c->exported_world != world) return fail(c, CTMR_E_INVALID, "already exported for a different group size");
        const int rc = alloc_exchange(c, world);
        if (rc) return rc;
        c->exported_world = world;  // the views of the peers' areas are set by ctmr_peer_attach
        e = cudaIpcGetMemHandle(&h.xchg, c->xchg);
        if (e != cudaSuccess) return fail(c, CTMR_E_PEER, std::string("cudaIpcGetMemHandle: ") + cudaGetErrorString(e));
    }
    h.X = c->X;
    h.world = world;
    h.table_slots = c->st.table_mask + 1;
    h.pair_slots = c->st.pair_mask + 1;
    h.meta_slots = c->st.meta_mask + 1;
    h.total = c->lay.total;
    h.max_issuers = c->st.max_issuers;
    std::memset(handle_out, 0, CTMR_PEER_HANDLE_BYTES);
    std::memcpy(handle_out, &h, sizeof h);
    return CTMR_OK;
}

int ctmr_peer_attach(ctmr_ctx* c, uint32_t rank, uint32_t world, const uint8_t* handles) {
    if (!c || !handles || world == 0 || world > kMaxWorld || rank >= world) return fail(c, CTMR_E_INVALID, "bad argument (1..8 ranks)");
    if (c->peer_mode != PEER_NONE || c->group) return fail(c, CTMR_E_INVALID, "ctx already belongs to a group");
    CU(c, cudaSetDevice(c->device));
    if (world == 1) return CTMR_OK;
    if (!c->xchg || c->exported_world != world) return fail(c, CTMR_E_INVALID, "call ctmr_peer_export(ctx, world, ...) with this group size first");
    uint8_t *bases[kMaxWorld] = {}, *xb[kMaxWorld] = {};
    auto close_all = [&]() {
        for (uint32_t q = 0; q < kMaxWorld; ++q) {
            if (c->ipc_base[q]) { cudaIpcCloseMemHandle(c->ipc_base[q]); c->ipc_base[q] = nullptr; }
            if (c->ipc_xchg[q]) { cudaIpcCloseMemHandle(c->ipc_xchg[q]); c->ipc_xchg[q] = nullptr; }
        }
    };
    for (uint32_t r = 0; r < world; ++r) {
        PeerHandle h;
        std::memcpy(&h, handles + (size_t)r * CTMR_PEER_HANDLE_BYTES, sizeof h);
        if (std::memcmp(h.magic, "CTMRPEER", 8) != 0) return fail(c, CTMR_E_INVALID, "not a ctmr peer handle");
        if (h.table_slots != c->st.table_mask + 1 || h.pair_slots != c->st.pair_mask + 1 || h.meta_slots != c->st.meta_mask + 1 ||
            h.max_issuers != c->st.max_issuers || h.total != c->lay.total || h.X != c->X || h.world != world)
            return fail(c, CTMR_E_INVALID, "rank " + std::to_string(r) + " was created with different capacities (or exported for another group size)");
        if (r == rank) {
            bases[r] = c->shared;
            xb[r] = c->xchg;
            continue;
        }
        void *p = nullptr, *x = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&p, h.mem, cudaIpcMemLazyEnablePeerAccess);
        if (e == cudaSuccess) {
            c->ipc_base[r] = p;
            e = cudaIpcOpenMemHandle(&x, h.xchg, cudaIpcMemLazyEnablePeerAccess);
            if (e == cudaSuccess) c->ipc_xchg[r] = x;
        }
        if (e != cudaSuccess) {
            (void)cudaGetLastError();
            close_all();
            return fail(c, CTMR_E_PEER, "cudaIpcOpenMemHandle(rank " + std::to_string(r) + "): " + cudaGetErrorString(e));
        }
        bases[r] = static_cast<uint8_t*>(p);
        xb[r] = static_cast<uint8_t*>(x);
    }
    attach_views(c, bases, world, rank);
    attach_exchange(c, xb, world, rank);
    c->peer_mode = PEER_IPC;
    return CTMR_OK;
}

int ctmr_peer_barrier_device(ctmr_ctx* c, void* stream) {
    if (!c) return CTMR_E_INVALID;
    CU(c, cudaSetDevice(c->device));
    return peer_barrier(c, CH_USER, stream ? (cudaStream_t)stream : c->stream);
}

int ctmr_peer_allreduce_histogram_device(ctmr_ctx* c, uint64_t* counts_dst, uint32_t n_slots, uint64_t* status_dst, void* stream) {
    if (!c || n_slots > c->st.max_issuers) return fail(c, CTMR_E_INVALID, "bad argument");
    CU(c, cudaSetDevice(c->device));
    cudaStream_t s = stream ? (cudaStream_t)stream : c->stream;
    int rc = peer_barrier(c, CH_HIST_A, s);  // every rank's counting kernels have finished
    if (rc) return rc;
    CU(c, launch_hist_sum(c->pf, n_slots, reinterpret_cast<unsigned long long*>(counts_dst), reinterpret_cast<unsigned long long*>(status_dst), s));
    return peer_barrier(c, CH_HIST_B, s);    // nobody resets its histogram while a peer still reads it
}

// ------------------------------------------------------------------------------------------------ host placement
int ctmr_bind_host_to_device(int32_t device) {
    char bus[32] = {};
    if (cudaDeviceGetPCIBusId(bus, sizeof bus, device) != cudaSuccess) {
        (void)cudaGetLastError();
        return -1;
    }
    for (char* p = bus; *p; ++p) *p = (char)tolower(*p);
    int node = -1;
    {
        std::ifstream f(std::string("/sys/bus/pci/devices/") + bus + "/numa_node");
        if (!(f >> node) || node < 0) return -1;
    }
    std::ifstream f("/sys/devices/system/node/node" + std::to_string(node) + "/cpulist");
    std::string list;
    if (!std::getline(f, list) || list.empty()) return -1;
    cpu_set_t allowed, want;
    CPU_ZERO(&want);
    if (sched_getaffinity(0, sizeof allowed, &allowed) != 0) return -1;
    size_t i = 0;
    int picked = 0;
    while (i < list.size()) {  // "0-31,64-95"
        size_t j = list.find(',', i);
        if (j == std::string::npos) j = list.size();
        const std::string tok = list.substr(i, j - i);
        const size_t dash = tok.find('-');
        const int a = atoi(tok.c_str()), b = dash == std::string::npos ? a : atoi(tok.c_str() + dash + 1);
        for (int cpu = a; cpu <= b && cpu < CPU_SETSIZE; ++cpu)
            if (CPU_ISSET(cpu, &allowed)) {
                CPU_SET(cpu, &want);
                ++picked;
            }
        i = j + 1;
    }
    if (!picked || sched_setaffinity(0, sizeof want, &want) != 0) return -1;
    return node;
}

}  // extern "C"
