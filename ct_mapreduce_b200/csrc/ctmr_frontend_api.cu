// ctmr_frontend_api.cu -- the entry points of include/ctmr_frontend.h: get-entries strings -> base64 decode -> TLS framing ->
// Chain[0] identification -> the path (SURVEY.md §8(f)-2), on one GPU (ctmr_process_raw) and on a group of GPUs driven by
// one process (ctmr_group_process_raw).
//
// A call is cut into CHUNKS (entry and character budgets of the front end's buffers).  Per chunk:
//   upload   the chunk's characters and string spans, on a copy stream, into one of two upload stages -- chunk k+1's
//            upload overlaps chunk k's kernels and the host round trips of its issuer identification;
//   front    fe_decode / fe_frame / fe_tbs / fe_issuer: the decoded leaves stay in the arena, the chunk becomes a
//            device-resident batch (ctmr_dev_batch with explicit lengths);
//   path     K_map ... K_pairs over that batch in place -- ctmr_process_device on one GPU; on a group one ROUND of the key
//            exchange (ctmr_pipeline.cu's scheme with device-resident slices): every member maps its chunk, hands
//            foreign keys to their owners over NVLink, the owners reduce, the bits are pulled back;
//   back     x509 leaf failures, PEM of the new certificates, outputs to the host.
// On a group a round takes one chunk per member, cut from ONE contiguous window of the batch, so that entry i keeps
// global index next_index + i and the result equals the single-GPU / sequential run on the same pages.
#include <thread>

#include "ctmr_ctx.cuh"

namespace {

struct RawChunk {
    uint64_t lo = 0, hi = 0;      // entries of the caller's batch
    uint64_t text_bytes = 0;      // characters uploaded for it
    int stage = 0;                // upload stage it sits in
    FeParams p{};
    ctmr_dev_batch db{};
    ctmr_dev_out dout{};
};

// How many entries starting at `lo` fit one chunk (at most max_entries): entry budget and half the character budget
// (the other half belongs to the stage being uploaded next).  Also validates the spans.
int fe_fit(ctmr_ctx* c, const ctmr_raw_batch* b, uint64_t lo, uint64_t max_entries, uint64_t* hi_out) {
    FrontEnd* f = c->fe;
    uint64_t hi = lo, chars = 0;
    while (hi < b->n && hi - lo < max_entries && hi - lo < f->cap_entries) {
        const uint64_t l1 = b->leaf_input_off[hi] + b->leaf_input_len[hi], x1 = b->extra_data_off[hi] + b->extra_data_len[hi];
        if (l1 > b->text_bytes || x1 > b->text_bytes) return fail(c, CTMR_E_INVALID, "string span outside the text buffer");
        const uint64_t add = (uint64_t)b->leaf_input_len[hi] + b->extra_data_len[hi];
        if (chars + add > f->cap_text / 2) break;
        chars += add;
        ++hi;
    }
    *hi_out = hi;
    return CTMR_OK;
}

// Characters and spans of entries [lo, hi) into upload stage `which`, asynchronously on the copy stream.
int fe_upload(ctmr_ctx* c, const ctmr_raw_batch* b, RawChunk& ch) {
    FrontEnd* f = c->fe;
    FeStage& st = f->stage[ch.stage];
    const uint64_t lo = ch.lo, cnt = ch.hi - ch.lo;
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaStreamWaitEvent(f->copy_stream, st.consumed, 0));  // the decode that last read this stage has run
    if (!cnt) {
        ch.text_bytes = 0;
        CU(c, cudaEventRecord(st.uploaded, f->copy_stream));
        return CTMR_OK;
    }
    uint64_t chars = 0, min_off = ~0ull, max_end = 0;
    for (uint64_t i = lo; i < ch.hi; ++i) {
        const uint64_t l0 = b->leaf_input_off[i], l1 = l0 + b->leaf_input_len[i];
        const uint64_t x0 = b->extra_data_off[i], x1 = x0 + b->extra_data_len[i];
        chars += (uint64_t)b->leaf_input_len[i] + b->extra_data_len[i];
        min_off = std::min(min_off, std::min(l0, x0));
        max_end = std::max(max_end, std::max(l1, x1));
    }
    std::memcpy(st.h_leaf_len, b->leaf_input_len + lo, cnt * 4);
    std::memcpy(st.h_extra_len, b->extra_data_len + lo, cnt * 4);
    if (max_end - min_off <= f->cap_text) {  // strings in place inside the response bodies: one copy
        ch.text_bytes = max_end - min_off;
        for (uint64_t i = 0; i < cnt; ++i) {
            st.h_leaf_off[i] = b->leaf_input_off[lo + i] - min_off;
            st.h_extra_off[i] = b->extra_data_off[lo + i] - min_off;
        }
        CU(c, cudaMemcpyAsync(st.text + 16, b->text + min_off, ch.text_bytes, cudaMemcpyHostToDevice, f->copy_stream));
    } else {  // scattered: pack on the host first
        st.pack.resize(chars);
        uint64_t w = 0;
        for (uint64_t i = 0; i < cnt; ++i) {
            st.h_leaf_off[i] = w;
            std::memcpy(st.pack.data() + w, b->text + b->leaf_input_off[lo + i], b->leaf_input_len[lo + i]);
            w += b->leaf_input_len[lo + i];
            st.h_extra_off[i] = w;
            std::memcpy(st.pack.data() + w, b->text + b->extra_data_off[lo + i], b->extra_data_len[lo + i]);
            w += b->extra_data_len[lo + i];
        }
        ch.text_bytes = w;
        CU(c, cudaMemcpyAsync(st.text + 16, st.pack.data(), ch.text_bytes, cudaMemcpyHostToDevice, f->copy_stream));
    }
    CU(c, cudaMemcpyAsync(st.leaf_off, st.h_leaf_off, cnt * 8, cudaMemcpyHostToDevice, f->copy_stream));
    CU(c, cudaMemcpyAsync(st.extra_off, st.h_extra_off, cnt * 8, cudaMemcpyHostToDevice, f->copy_stream));
    CU(c, cudaMemcpyAsync(st.leaf_len, st.h_leaf_len, cnt * 4, cudaMemcpyHostToDevice, f->copy_stream));
    CU(c, cudaMemcpyAsync(st.extra_len, st.h_extra_len, cnt * 4, cudaMemcpyHostToDevice, f->copy_stream));
    CU(c, cudaEventRecord(st.uploaded, f->copy_stream));
    return CTMR_OK;
}

// decode + frame + Chain[0] -> dense index of an uploaded chunk; leaves ch.db / ch.dout describing the device-resident batch
int fe_front(ctmr_ctx* c, const ctmr_raw_batch* b, const ctmr_raw_out* out, RawChunk& ch, uint64_t first_index) {
    FrontEnd* f = c->fe;
    cudaStream_t s = c->stream;
    CU(c, cudaSetDevice(c->device));
    FeStage& st = f->stage[ch.stage];
    const uint64_t cnt = ch.hi - ch.lo, E = f->cap_entries;
    const ctmr_out* po = &out->path;
    const bool want_meta = po->first_issuer_dn || po->first_crldp || po->issuer_name_off || po->crldp_off;
    CU(c, cudaStreamWaitEvent(s, st.uploaded, 0));
    FeParams& p = ch.p;
    p = FeParams{};
    p.text = st.text + 16;
    p.text_bytes = ch.text_bytes;
    p.leaf_off = st.leaf_off; p.leaf_len = st.leaf_len; p.extra_off = st.extra_off; p.extra_len = st.extra_len;
    p.n = cnt;
    p.pad_size = f->pad_size; p.dec_off = f->dec_off; p.dec_len = f->dec_len; p.str_bad = f->str_bad; p.decoded = f->decoded;
    p.entry_status = f->entry_status; p.entry_type = f->entry_type; p.timestamp = f->timestamp; p.leaf_src = f->leaf_src;
    p.leaf_rel = f->leaf_rel; p.leaf_len_out = f->leaf_len_out; p.leaf_abs = f->leaf_abs; p.chain_abs = f->chain_abs;
    p.chain_len = f->chain_len; p.tbs_abs = f->tbs_abs; p.tbs_len = f->tbs_len; p.issuer_idx = f->issuer_idx;
    ch.db = ctmr_dev_batch{};
    ch.dout = ctmr_dev_out{};
    CU(c, cudaEventRecord(f->ev0, s));
    if (cnt) {
        CU(c, launch_fe_decode(p, f->scan_temp, f->scan_temp_bytes, c->sm_count, s));
        CU(c, cudaEventRecord(st.consumed, s));  // text and spans are dead once decoded: the stage may be refilled
        CU(c, launch_fe_frame(p, s));
        f->launches += 5;  // sizes, scan (cub: one kernel visible to us), decode, frame, tbs
        // ---- Chain[0] -> dense index; certificates never seen before go through ctmr_register_issuers once (the registry
        // is the group's: whichever member meets an issuer first, every member gets the same index)
        for (int round = 0;; ++round) {
            if (round > 64) return fail(c, CTMR_E_CUDA, "front end: issuer identification does not converge");
            IssuerCertTable tab{f->slots_dev, f->slot_mask, f->arena};
            CU(c, cudaMemsetAsync(f->pending, 0, (f->pending_mask + 1) * 8, s));
            CU(c, cudaMemsetAsync(f->unknown_count, 0, 4, s));
            CU(c, launch_fe_issuer(p, tab, f->pending, f->pending_mask, f->unknown_list, f->unknown_cap, f->unknown_count, c->sm_count, s));
            ++f->launches;
            unsigned int n_unknown = 0;
            CU(c, cudaMemcpyAsync(&n_unknown, f->unknown_count, 4, cudaMemcpyDeviceToHost, s));
            CU(c, cudaStreamSynchronize(s));
            if (n_unknown == 0) break;
            if (n_unknown > f->unknown_cap) n_unknown = f->unknown_cap;  // the rest shows up again next round
            std::vector<uint32_t> list(n_unknown);
            CU(c, cudaMemcpyAsync(list.data(), f->unknown_list, n_unknown * 4ull, cudaMemcpyDeviceToHost, s));
            CU(c, cudaStreamSynchronize(s));
            std::vector<uint8_t> blob;
            std::vector<uint64_t> offs(1, 0);
            for (uint32_t e : list) {
                uint64_t at = 0;
                uint32_t len = 0;
                CU(c, cudaMemcpyAsync(&at, f->chain_abs + e, 8, cudaMemcpyDeviceToHost, s));
                CU(c, cudaMemcpyAsync(&len, f->chain_len + e, 4, cudaMemcpyDeviceToHost, s));
                CU(c, cudaStreamSynchronize(s));
                const size_t w = blob.size();
                blob.resize(w + len);
                CU(c, cudaMemcpyAsync(blob.data() + w, f->decoded + at, len, cudaMemcpyDeviceToHost, s));
                CU(c, cudaStreamSynchronize(s));
                offs.push_back(blob.size());
            }
            std::vector<uint32_t> dense(n_unknown);
            const uint64_t before = f->slots_used;
            int rc = ctmr_register_issuers(c, blob.data(), offs.data(), n_unknown, dense.data());
            if (rc) return rc;
            if (f->slots_used == before) return fail(c, CTMR_E_CUDA, "front end: unresolved Chain[0] is already registered");
        }
    } else {
        CU(c, cudaEventRecord(st.consumed, s));
    }
    CU(c, cudaEventRecord(f->ev1, s));
    // ---- the path's input: the decoded arena, leaves where the decoder put them
    ctmr_dev_batch& db = ch.db;
    db.blob = f->decoded;
    if (cnt) {
        CU(c, cudaMemcpyAsync(&db.blob_bytes, f->dec_off + 2 * cnt, 8, cudaMemcpyDeviceToHost, s));
        CU(c, cudaStreamSynchronize(s));
    }
    db.offsets = f->leaf_abs;
    db.lens = f->leaf_len_out;
    db.n = cnt;
    db.issuer_idx = f->issuer_idx;
    db.first_index = first_index;
    db.now_unix_ns = b->now_unix_ns;
    ctmr_dev_out& dout = ch.dout;
    dout.status = f->status;
    dout.sha256 = po->sha256 ? f->sha : nullptr;
    dout.exp_hour = f->exp_hour;
    dout.serial_off = f->serial_off;
    dout.serial_len = f->serial_len;
    dout.was_unknown = f->was_unknown;
    dout.first_issuer_hour = f->first;
    if (want_meta) {
        dout.issuer_name_off = f->spans;
        dout.issuer_name_len = f->spans + E;
        dout.crldp_off = f->spans + 2 * E;
        dout.crldp_len = f->spans + 3 * E;
        dout.first_issuer_dn = f->first_meta;
        dout.first_crldp = f->first_meta + E;
    }
    return CTMR_OK;
}

// after the path: x509 leaf failures, PEM, outputs to the host; waits for the chunk
int fe_back(ctmr_ctx* c, const ctmr_raw_out* out, RawChunk& ch, uint64_t* pem_base) {
    FrontEnd* f = c->fe;
    cudaStream_t s = c->stream;
    CU(c, cudaSetDevice(c->device));
    const uint64_t cnt = ch.hi - ch.lo, lo = ch.lo, E = f->cap_entries;
    const ctmr_out* po = &out->path;
    const bool want_meta = po->first_issuer_dn || po->first_crldp || po->issuer_name_off || po->crldp_off;
    const bool want_pem = po->pem != nullptr;
    if (!cnt) {
        CU(c, cudaStreamSynchronize(s));
        return CTMR_OK;
    }
    CU(c, launch_fe_finish(ch.p, f->status, s));
    ++f->launches;
    CU(c, cudaEventRecord(f->ev2, s));
    if (want_pem) {  // the decoded DER exists only on the device: its PEM is how new certificates reach the host
        int rc = pem_ensure(c, f->pem, E, f->cap_decoded);
        if (rc) return rc;
        rc = pem_chunk(c, f->pem, f->decoded, f->leaf_abs, f->leaf_len_out, f->was_unknown, cnt, po, lo, pem_base, s);
        if (rc) return rc;
    }
#define FE_D2H(dst, src, bytes) \
    if (dst) CU(c, cudaMemcpyAsync(reinterpret_cast<uint8_t*>(dst) + lo * ((bytes) / cnt), (src), (bytes), cudaMemcpyDeviceToHost, s))
    FE_D2H(po->status, f->status, cnt);
    FE_D2H(po->sha256, f->sha, cnt * 32);
    FE_D2H(po->exp_hour, f->exp_hour, cnt * 8);
    FE_D2H(po->serial_off, f->serial_off, cnt * 4);
    FE_D2H(po->serial_len, f->serial_len, cnt * 4);
    FE_D2H(po->was_unknown, f->was_unknown, cnt);
    FE_D2H(po->first_issuer_hour, f->first, cnt);
    if (want_meta) {
        FE_D2H(po->issuer_name_off, ch.dout.issuer_name_off, cnt * 4);
        FE_D2H(po->issuer_name_len, ch.dout.issuer_name_len, cnt * 4);
        FE_D2H(po->crldp_off, ch.dout.crldp_off, cnt * 4);
        FE_D2H(po->crldp_len, ch.dout.crldp_len, cnt * 4);
        FE_D2H(po->first_issuer_dn, ch.dout.first_issuer_dn, cnt);
        FE_D2H(po->first_crldp, ch.dout.first_crldp, cnt);
    }
    FE_D2H(out->entry_status, f->entry_status, cnt);
    FE_D2H(out->entry_type, f->entry_type, cnt);
    FE_D2H(out->timestamp_ms, f->timestamp, cnt * 8);
    FE_D2H(out->issuer, f->issuer_idx, cnt * 4);
    FE_D2H(out->leaf_src, f->leaf_src, cnt);
    FE_D2H(out->leaf_off, f->leaf_rel, cnt * 4);
    FE_D2H(out->leaf_len, f->leaf_len_out, cnt * 4);
#undef FE_D2H
    CU(c, cudaStreamSynchronize(s));
    float a = 0.f, d = 0.f;
    CU(c, cudaEventElapsedTime(&a, f->ev0, f->ev1));
    CU(c, cudaEventElapsedTime(&d, f->ev1, f->ev2));
    f->fe_ms += a;
    f->path_ms += d;
    return CTMR_OK;
}

int check_args(ctmr_ctx* c, const ctmr_raw_batch* b, ctmr_raw_out* out) {
    if (!b || !out) return fail(c, CTMR_E_INVALID, "bad argument");
    if (b->n && (!b->text || !b->leaf_input_off || !b->leaf_input_len || !b->extra_data_off || !b->extra_data_len))
        return fail(c, CTMR_E_INVALID, "null batch buffers");
    if ((out->path.pem != nullptr) != (out->path.pem_off != nullptr)) return fail(c, CTMR_E_INVALID, "pem and pem_off go together");
    return CTMR_OK;
}

int process_raw_single(ctmr_ctx* c, const ctmr_raw_batch* b, ctmr_raw_out* out) {
    int rc = check_args(c, b, out);
    if (rc) return rc;
    if (b->n == 0) return CTMR_OK;
    CU(c, cudaSetDevice(c->device));
    rc = frontend_ensure(c);
    if (rc) return rc;
    FrontEnd* f = c->fe;
    f->fe_ms = f->path_ms = 0.f;
    f->launches = 0;
    uint64_t pem_base = 0;
    RawChunk ch[2];
    rc = fe_fit(c, b, 0, ~0ull, &ch[0].hi);
    if (rc) return rc;
    if (ch[0].hi == 0) return fail(c, CTMR_E_BATCH_TOO_LARGE, "a single entry exceeds the front end's character budget");
    rc = fe_upload(c, b, ch[0]);
    if (rc) return rc;
    for (int k = 0;; ++k) {
        RawChunk& cur = ch[k & 1];
        if (cur.hi < b->n) {  // next chunk's upload overlaps this chunk's kernels
            RawChunk& nx = ch[(k + 1) & 1];
            nx = RawChunk{};
            nx.lo = cur.hi;
            nx.stage = (k + 1) & 1;
            rc = fe_fit(c, b, nx.lo, ~0ull, &nx.hi);
            if (rc) return rc;
            if (nx.hi == nx.lo) return fail(c, CTMR_E_BATCH_TOO_LARGE, "a single entry exceeds the front end's character budget");
            rc = fe_upload(c, b, nx);
            if (rc) return rc;
        }
        rc = fe_front(c, b, out, cur, c->next_index + cur.lo);
        if (rc) return rc;
        rc = ctmr_process_device(c, &cur.db, &cur.dout, c->stream);
        if (rc) return rc;
        rc = fe_back(c, out, cur, &pem_base);
        if (rc) return rc;
        if (cur.hi >= b->n) break;
    }
    if (out->path.pem) out->path.pem_off[b->n] = pem_base;
    return ctmr_check_device(c, nullptr);
}

// One round of the path over the members' device-resident chunks: map + route, [events], owner passes, [events], pull,
// [string identities: insert, events, read-back].  Each member works on its own stream; rounds are serialised by the
// callers' fe_back, which is also what orders the rounds for lowest-index-wins.
int group_round(ctmr_group* g, RawChunk* ch, int parity, ctmr_ctx** failed) {
    const uint32_t W = (uint32_t)g->m.size();
    int rc;
    for (uint32_t r = 0; r < W; ++r) {
        ctmr_ctx* c = g->m[r];
        *failed = c;
        CU(c, cudaSetDevice(c->device));
        cudaStream_t s = c->stream;
        const uint64_t cnt = ch[r].hi - ch[r].lo;
        rc = ensure_scratch(c, std::max<uint64_t>(cnt, 1));
        if (rc) return rc;
        for (cudaEvent_t& e : c->ev_g)
            if (!e) CU(c, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        rc = round_begin(c, parity, s);
        if (rc) return rc;
        if (cnt) {
            ch[r].dout.keys = c->keys_scratch;
            MapParams p;
            fill_map_params(c, &ch[r].db, &ch[r].dout, p, 3, c->slot_scratch, parity);
            if (c->bucket_by_length && cnt > 64 && p.sha256) {
                if (cnt > c->order_cap) {
                    CU(c, cudaStreamSynchronize(s));
                    cudaFree(c->order_scratch);
                    c->order_scratch = nullptr;
                    c->order_cap = 0;
                    CU(c, cudaMalloc(&c->order_scratch, cnt * sizeof(uint32_t)));
                    c->order_cap = cnt;
                }
                if (!c->len_hist) CU(c, cudaMalloc(&c->len_hist, 256 * sizeof(unsigned int)));
                CU(c, launch_len_order(ch[r].db.offsets, ch[r].db.lens, cnt, ch[r].db.blob_bytes, c->len_hist, c->order_scratch, s));
                p.order = c->order_scratch;
            }
            CU(c, launch_map(p, c->sm_count, s));
        }
        rc = round_publish(c, parity, s);
        if (rc) return rc;
        CU(c, cudaEventRecord(c->ev_g[0], s));
    }
    const uint64_t maxr = g->m[0]->fe->cap_entries;
    for (uint32_t r = 0; r < W; ++r) {
        ctmr_ctx* c = g->m[r];
        *failed = c;
        CU(c, cudaSetDevice(c->device));
        cudaStream_t s = c->stream;
        const uint64_t cnt = ch[r].hi - ch[r].lo;
        for (uint32_t q = 0; q < W; ++q)
            if (q != r) CU(c, cudaStreamWaitEvent(s, g->m[q]->ev_g[0], 0));
        rc = round_owner_insert(c, parity, maxr, s);
        if (rc) return rc;
        if (cnt) CU(c, launch_resolve(c->st, c->keys_scratch, cnt, c->slot_scratch, c->pair_scratch, ch[r].dout.was_unknown, s));
        rc = round_owner_resolve(c, parity, maxr, s);
        if (rc) return rc;
        if (cnt) CU(c, launch_resolve_pairs(c->st, c->keys_scratch, cnt, c->pair_scratch, ch[r].dout.was_unknown, ch[r].dout.first_issuer_hour, s));
        rc = round_owner_pairs(c, parity, maxr, s);
        if (rc) return rc;
        CU(c, cudaEventRecord(c->ev_g[1], s));
    }
    bool any_meta = false;
    for (uint32_t r = 0; r < W; ++r) {
        ctmr_ctx* c = g->m[r];
        *failed = c;
        CU(c, cudaSetDevice(c->device));
        cudaStream_t s = c->stream;
        const uint64_t cnt = ch[r].hi - ch[r].lo;
        for (uint32_t q = 0; q < W; ++q)
            if (q != r) CU(c, cudaStreamWaitEvent(s, g->m[q]->ev_g[1], 0));
        rc = round_pull(c, parity, maxr, ch[r].dout.was_unknown, ch[r].dout.first_issuer_hour, s);
        if (rc) return rc;
        const bool want_meta = ch[r].dout.first_issuer_dn || ch[r].dout.first_crldp;
        any_meta |= want_meta;
        if (want_meta && cnt)
            CU(c, launch_meta_insert(c->st, ch[r].db.blob, ch[r].db.offsets, c->keys_scratch, cnt, ch[r].dout.was_unknown, ch[r].dout.issuer_name_off,
                                     ch[r].dout.issuer_name_len, ch[r].dout.crldp_off, ch[r].dout.crldp_len, c->meta_scratch, s));
        CU(c, cudaEventRecord(c->ev_g[2], s));
    }
    if (any_meta)
        for (uint32_t r = 0; r < W; ++r) {
            ctmr_ctx* c = g->m[r];
            *failed = c;
            CU(c, cudaSetDevice(c->device));
            cudaStream_t s = c->stream;
            const uint64_t cnt = ch[r].hi - ch[r].lo;
            for (uint32_t q = 0; q < W; ++q)
                if (q != r) CU(c, cudaStreamWaitEvent(s, g->m[q]->ev_g[2], 0));
            if (cnt)
                CU(c, launch_meta_resolve(c->st, c->keys_scratch, cnt, c->meta_scratch, ch[r].dout.first_issuer_dn, ch[r].dout.first_crldp, s));
        }
    *failed = nullptr;
    return CTMR_OK;
}

// cut the next round out of the batch: one chunk per member from ONE contiguous window starting at `pos`
int plan_round(ctmr_group* g, const ctmr_raw_batch* b, uint64_t pos, int stage, std::vector<RawChunk>& ch, ctmr_ctx** failed) {
    const uint32_t W = (uint32_t)g->m.size();
    ctmr_ctx* c0 = g->m[0];
    *failed = c0;
    uint64_t q = std::min<uint64_t>(c0->fe->cap_entries, (b->n - pos + W - 1) / W);
    for (;;) {
        bool fits = true;
        for (uint32_t r = 0; r < W && fits; ++r) {
            const uint64_t lo = std::min(b->n, pos + r * q), want = std::min(b->n, pos + (r + 1) * q);
            uint64_t hi = 0;
            int rc = fe_fit(g->m[r], b, lo, want - lo, &hi);
            if (rc) {
                *failed = g->m[r];
                return rc;
            }
            fits = hi == want;
        }
        if (fits) break;
        if (q == 1) return fail(c0, CTMR_E_BATCH_TOO_LARGE, "a single entry exceeds the front end's character budget");
        q = (q + 1) / 2;
    }
    ch.assign(W, RawChunk{});
    for (uint32_t r = 0; r < W; ++r) {
        ch[r].lo = std::min(b->n, pos + r * q);
        ch[r].hi = std::min(b->n, pos + (r + 1) * q);
        ch[r].stage = stage;
        *failed = g->m[r];
        int rc = fe_upload(g->m[r], b, ch[r]);
        if (rc) return rc;
    }
    *failed = nullptr;
    return CTMR_OK;
}

int process_raw_group(ctmr_group* g, const ctmr_raw_batch* b, ctmr_raw_out* out, ctmr_ctx** failed) {
    const uint32_t W = (uint32_t)g->m.size();
    ctmr_ctx* c0 = g->m[0];
    *failed = c0;
    int rc = check_args(c0, b, out);
    if (rc) return rc;
    if (b->n == 0) return CTMR_OK;
    for (uint32_t r = 0; r < W; ++r) {
        ctmr_ctx* c = g->m[r];
        *failed = c;
        CU(c, cudaSetDevice(c->device));
        rc = frontend_ensure(c);
        if (rc) return rc;
        c->fe->fe_ms = c->fe->path_ms = 0.f;
        c->fe->launches = 0;
    }
    uint64_t pem_base = 0, pos = 0;
    std::vector<RawChunk> cur, nxt;
    rc = plan_round(g, b, 0, 0, cur, failed);
    if (rc) return rc;
    for (int k = 0;; ++k) {
        const uint64_t end = cur[W - 1].hi;
        if (end < b->n) {  // the next round's uploads overlap this round's kernels and host round trips
            rc = plan_round(g, b, end, (k + 1) & 1, nxt, failed);
            if (rc) return rc;
        }
        // The front halves wait on the host (issuer identification round trips, the arena size): one thread per member, so
        // that the members' waits overlap instead of adding up.  Each thread touches its own ctx only; the issuer registry
        // they all resolve against is device memory reached with atomics.
        std::vector<int> rcs;
        for_each_member(W, rcs, [&](uint32_t r) { return fe_front(g->m[r], b, out, cur[r], g->next_index + cur[r].lo); });
        for (uint32_t r = 0; r < W; ++r)
            if (rcs[r]) {
                *failed = g->m[r];
                return rcs[r];
            }
        rc = group_round(g, cur.data(), k % (int)kParities, failed);
        if (rc) return rc;
        if (out->path.pem) {
            for (uint32_t r = 0; r < W; ++r) {  // in entry order: the PEM texts are appended in that order
                *failed = g->m[r];
                rc = fe_back(g->m[r], out, cur[r], &pem_base);
                if (rc) return rc;
            }
        } else {  // disjoint output ranges: the members' copies and waits overlap as well
            for_each_member(W, rcs, [&](uint32_t r) { return fe_back(g->m[r], out, cur[r], &pem_base); });
            for (uint32_t r = 0; r < W; ++r)
                if (rcs[r]) {
                    *failed = g->m[r];
                    return rcs[r];
                }
        }
        pos = end;
        if (end >= b->n) break;
        cur.swap(nxt);
    }
    (void)pos;
    if (out->path.pem) out->path.pem_off[b->n] = pem_base;
    for (uint32_t r = 0; r < W; ++r) {
        *failed = g->m[r];
        rc = ctmr_check_device(g->m[r], nullptr);
        if (rc) return rc;
    }
    *failed = nullptr;
    return CTMR_OK;
}

// an upload of the NEXT chunk may still be reading the caller's text and an output copy may still be writing the caller's
// arrays: neither may outlive a failed call
void drain_frontend(ctmr_ctx* c) {
    if (!c || !c->fe) return;
    const std::string keep = c->err;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->fe->copy_stream);
    cudaStreamSynchronize(c->stream);
    c->err = keep;
}

}  // namespace

extern "C" {

int ctmr_process_raw(ctmr_ctx* c, const ctmr_raw_batch* b, ctmr_raw_out* out) {
    if (!c) return CTMR_E_INVALID;
    if (c->group || c->peer_mode != PEER_NONE) return fail(c, CTMR_E_INVALID, "member of a group: use ctmr_group_process_raw");
    const int rc = process_raw_single(c, b, out);
    if (b) c->next_index += b->n;  // also after a failure: a retry must not reuse the indices
    if (rc != CTMR_OK) drain_frontend(c);
    return rc;
}

int ctmr_group_process_raw(ctmr_group* g, const ctmr_raw_batch* b, ctmr_raw_out* out) {
    if (!g || g->m.empty()) return CTMR_E_INVALID;
    ctmr_ctx* failed = nullptr;
    int rc;
    if (g->m.size() == 1) {  // a group of one is a plain ctx
        ctmr_ctx* c = g->m[0];
        c->next_index = g->next_index;
        rc = process_raw_single(c, b, out);
        failed = c;
    } else {
        rc = process_raw_group(g, b, out, &failed);
    }
    if (b) g->next_index += b->n;  // also after a failure: a retry must not reuse the indices (its entries then read as known)
    if (rc != CTMR_OK) {
        for (ctmr_ctx* c : g->m) drain_frontend(c);
        if (failed) g->err = failed->err;
    }
    return rc;
}

}  // extern "C"
