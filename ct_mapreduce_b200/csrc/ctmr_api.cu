// ctmr_api.cu -- the C ABI of include/ctmr.h: context, issuer registry, host-buffer batch
// pipeline (H2D / kernels / D2H overlapped over three streams) and the device-resident entry points.
// There is deliberately no CPU implementation of the path in this file or anywhere in the library:
// without a CUDA device ctmr_create fails.
#include "ctmr_ctx.cuh"

thread_local std::string ctmr_host::g_create_error;

namespace ctmr_host {

int fail(ctmr_ctx* ctx, int code, const std::string& msg) {
    if (ctx) ctx->err = msg;
    else g_create_error = msg;
    return code;
}

uint64_t pow2_at_least(uint64_t v) {
    uint64_t p = 1;
    while (p < v) p <<= 1;
    return p;
}

}  // namespace ctmr_host

namespace {

void fe_destroy(ctmr_ctx* c);
int fe_add_issuer(ctmr_ctx* c, const std::string& der, uint32_t idx);
int fe_clear_issuers(ctmr_ctx* c);

// strings.Split(*ctconfig.IssuerCNFilter, ",") -- no trimming (ct-fetch.go:58)
int build_filter(const ctmr_config* cfg, FilterCfg& f) {
    std::memset(&f, 0, sizeof f);
    f.filter_nonempty = cfg->issuer_cn_filter_len != 0;
    f.log_expired = cfg->log_expired_entries != 0;
    f.flags = cfg->flags;
    if (!f.filter_nonempty) return 0;
    if (cfg->issuer_cn_filter_len > sizeof f.bytes) return -1;
    uint32_t start = 0, np = 0, used = 0;
    for (uint32_t i = 0; i <= cfg->issuer_cn_filter_len; ++i) {
        if (i == cfg->issuer_cn_filter_len || cfg->issuer_cn_filter[i] == ',') {
            if (np >= 32) return -1;
            f.off[np] = (uint16_t)used;
            std::memcpy(f.bytes + used, cfg->issuer_cn_filter + start, i - start);
            used += i - start;
            ++np;
            f.off[np] = (uint16_t)used;
            start = i + 1;
        }
    }
    f.n_prefix = np;
    return 0;
}

SharedLayout make_layout(uint64_t table_slots, uint64_t pair_slots, uint64_t meta_slots, uint32_t max_issuers) {
    SharedLayout l;
    auto take = [&](size_t bytes) {
        const size_t at = l.total;
        l.total += (bytes + 255) & ~(size_t)255;
        return at;
    };
    l.flags = take((kPeerChannels + 1) * kMaxWorld * sizeof(unsigned long long));
    l.reg_counter = take(sizeof(unsigned long long));
    l.status_counts = take(CTMR_ST__COUNT * sizeof(unsigned long long));
    l.issuer_counts = take((size_t)max_issuers * sizeof(unsigned long long));
    l.reg_digests = take((size_t)max_issuers * 32);
    l.reg_mask = pow2_at_least(2ull * max_issuers) - 1;
    l.reg_slots = take((size_t)(l.reg_mask + 1) * sizeof(IssuerRegSlot));
    l.meta = take((size_t)meta_slots * sizeof(MetaSlot));
    l.pairs = take((size_t)pair_slots * sizeof(PairSlot));
    l.table = take((size_t)table_slots * sizeof(KnownSlot));
    return l;
}

}  // namespace
namespace ctmr_host {
int ensure_scratch(ctmr_ctx* c, uint64_t n) {
    if (n <= c->scratch_cap) return CTMR_OK;
    CU(c, cudaDeviceSynchronize());
    cudaFree(c->keys_scratch); cudaFree(c->slot_scratch); cudaFree(c->pair_scratch); cudaFree(c->bits_scratch);
    cudaFree(c->meta_scratch);
    c->keys_scratch = nullptr; c->slot_scratch = c->pair_scratch = nullptr; c->bits_scratch = nullptr; c->meta_scratch = nullptr;
    c->scratch_cap = 0;
    CU(c, cudaMalloc(&c->keys_scratch, n * sizeof(ctmr_key)));
    CU(c, cudaMalloc(&c->slot_scratch, n * sizeof(uint32_t)));
    CU(c, cudaMalloc(&c->pair_scratch, n * sizeof(uint32_t)));
    CU(c, cudaMalloc(&c->bits_scratch, 2 * n));
    CU(c, cudaMalloc(&c->meta_scratch, 2 * n * sizeof(uint32_t)));
    c->scratch_cap = n;
    return CTMR_OK;
}

void fill_map_params(ctmr_ctx* c, const ctmr_dev_batch* b, const ctmr_dev_out* o, MapParams& p, int counter_slot,
                     uint32_t* fused_slot_of, int parity) {
    std::memset(&p, 0, sizeof p);
    p.blob = b->blob;
    p.blob_bytes = b->blob_bytes;
    p.offsets = b->offsets;
    p.lens = b->lens;
    p.n = b->n;
    p.issuer_idx = b->issuer_idx;
    p.issuer_map = b->issuer_map;
    p.issuer_map_len = b->issuer_map_len;
    p.first_index = b->first_index;
    // NotAfter.Before(now): split now into whole seconds and "has a fractional part"
    int64_t ns = b->now_unix_ns;
    int64_t sec = ns >= 0 ? ns / 1000000000LL : -((-ns + 999999999LL) / 1000000000LL);
    p.now_sec = sec;
    p.now_frac_nonzero = (ns - sec * 1000000000LL) != 0;
    p.one = 1;
    {
        static const bool skip = getenv("CTMR_DEBUG_SKIP_WALK") && atoi(getenv("CTMR_DEBUG_SKIP_WALK"));
        p.debug_skip_walk = skip;
    }
    {
        static const int sh[12] = {2, 13, 22, 6, 11, 25, 7, 18, 3, 17, 19, 10};
        for (int i = 0; i < 12; ++i) p.rot_mul[i] = 1u << (32 - sh[i]);
    }
    p.status = o->status;
    p.sha256 = (c->flags & CTMR_F_NO_FINGERPRINT) ? nullptr : o->sha256;
    p.exp_hour = o->exp_hour;
    p.serial_off = o->serial_off;
    p.serial_len = o->serial_len;
    p.keys = o->keys;
    if (o->issuer_name_off && o->issuer_name_len && o->crldp_off && o->crldp_len) {
        p.issuer_name_off = o->issuer_name_off;
        p.issuer_name_len = o->issuer_name_len;
        p.crldp_off = o->crldp_off;
        p.crldp_len = o->crldp_len;
    }
    {
        static const int lp = env_int("CTMR_LIGHT_PREFETCH", 2);
        p.light_prefetch = (uint32_t)lp;
    }
    p.status_counts = c->st.status_counts;
    p.work_counter = c->small_dev + 84 + counter_slot;  // one per pipeline stage + one for the device entry points
    p.filter = c->filter;
    p.route.world = 1;
    if (fused_slot_of && p.keys) {  // K_insert fused into K_map: own keys into the own table, the others to their owners' inboxes
        p.table = c->st.table;
        const uint32_t W = c->px.world;
        if (W > 1) {
            for (uint32_t r = 0; r < W; ++r) p.route.inbox[r] = c->px.inbox[r] + ((uint64_t)parity * W + c->px.rank) * c->px.X;
            p.route.cursor = c->cursors + (size_t)parity * kMaxWorld;
            p.route.rev = c->rev + (uint64_t)parity * W * c->px.X;
            p.route.X = c->px.X;
            p.route.world = W;
            p.route.rank = c->px.rank;
        }
        p.table_mask = c->st.table_mask;
        p.error_flag = c->st.error_flag;
        p.slot_of = fused_slot_of;
    }
}

// views of every rank's shared region: the tables K_map / K_resolve address, the flags and histograms of the
// cross-process barrier and all-reduce, the issuer registry in rank 0's region
void attach_views(ctmr_ctx* c, uint8_t* const* bases, uint32_t world, uint32_t rank) {
    const SharedLayout& l = c->lay;
    c->st.peer = PeerTables{};
    c->pf = PeerFlags{};
    for (uint32_t r = 0; r < world; ++r) {
        c->st.peer.table[r] = reinterpret_cast<KnownSlot*>(bases[r] + l.table);
        c->st.peer.pairs[r] = reinterpret_cast<PairSlot*>(bases[r] + l.pairs);
        c->st.peer.meta[r] = reinterpret_cast<MetaSlot*>(bases[r] + l.meta);
        c->pf.flags[r] = reinterpret_cast<unsigned long long*>(bases[r] + l.flags);
        c->pf.issuer_counts[r] = reinterpret_cast<unsigned long long*>(bases[r] + l.issuer_counts);
        c->pf.status_counts[r] = reinterpret_cast<unsigned long long*>(bases[r] + l.status_counts);
    }
    c->st.peer.world = c->pf.world = world;
    c->st.peer.rank = c->pf.rank = rank;
    c->pf.timeout_ns = 60000ull * 1000000ull;
    if (const char* ev = getenv("CTMR_PEER_TIMEOUT_MS")) {
        const unsigned long long ms = strtoull(ev, nullptr, 10);
        if (ms) c->pf.timeout_ns = ms * 1000000ull;
    }
    c->reg.slots = reinterpret_cast<IssuerRegSlot*>(bases[0] + l.reg_slots);
    c->reg.mask = l.reg_mask;
    c->reg.counter = reinterpret_cast<unsigned long long*>(bases[0] + l.reg_counter);
    c->reg.by_index = bases[0] + l.reg_digests;
    c->reg.max_issuers = c->st.max_issuers;
}

size_t exchange_bytes(uint32_t world, uint64_t X) {
    return 4096 + (size_t)kParities * world * X * (sizeof(ctmr_key) + 2);
}

// layout of a rank's exchange area: [counts: kParities x world u64, padded to 4 KiB][inbox][out_wu][out_first]
void attach_exchange(ctmr_ctx* c, uint8_t* const* bases, uint32_t world, uint32_t rank) {
    c->px = PeerExchange{};
    const uint64_t per = (uint64_t)kParities * world * c->X;
    for (uint32_t r = 0; r < world; ++r) {
        c->px.counts[r] = reinterpret_cast<unsigned long long*>(bases[r]);
        c->px.inbox[r] = reinterpret_cast<ctmr_key*>(bases[r] + 4096);
        c->px.out_wu[r] = bases[r] + 4096 + per * sizeof(ctmr_key);
        c->px.out_first[r] = c->px.out_wu[r] + per;
    }
    c->px.X = c->X;
    c->px.world = world;
    c->px.rank = rank;
}

int alloc_exchange(ctmr_ctx* c, uint32_t world) {
    if (c->xchg || world <= 1) return CTMR_OK;
    c->X = c->cfg_round_entries ? c->cfg_round_entries : c->stage_entries;
    if (c->X < c->stage_entries) c->X = c->stage_entries;  // the host pipeline maps stage_entries per round
    const size_t per = (size_t)kParities * world * c->X;
    CU(c, cudaMalloc(&c->xchg, exchange_bytes(world, c->X)));
    CU(c, cudaMemsetAsync(c->xchg, 0, 4096, c->stream));
    CU(c, cudaMalloc(&c->cursors, (size_t)kParities * kMaxWorld * sizeof(unsigned long long)));
    CU(c, cudaMemsetAsync(c->cursors, 0, (size_t)kParities * kMaxWorld * sizeof(unsigned long long), c->stream));
    CU(c, cudaMalloc(&c->rev, per * sizeof(uint32_t)));
    CU(c, cudaMalloc(&c->in_slot, per * sizeof(uint32_t)));
    CU(c, cudaMalloc(&c->in_pair, per * sizeof(uint32_t)));
    CU(c, cudaStreamSynchronize(c->stream));
    return CTMR_OK;
}

int round_begin(ctmr_ctx* c, int parity, cudaStream_t s) {
    if (c->px.world <= 1) return CTMR_OK;
    CU(c, cudaMemsetAsync(c->cursors + (size_t)parity * kMaxWorld, 0, kMaxWorld * sizeof(unsigned long long), s));
    return CTMR_OK;
}
int round_publish(ctmr_ctx* c, int parity, cudaStream_t s) {
    if (c->px.world <= 1) return CTMR_OK;
    CU(c, launch_publish_counts(c->px, (uint32_t)parity, c->cursors + (size_t)parity * kMaxWorld, s));
    return CTMR_OK;
}
int round_owner_insert(ctmr_ctx* c, int parity, uint64_t maxr, cudaStream_t s) {
    if (c->px.world <= 1) return CTMR_OK;
    CU(c, launch_inbox_insert(c->st, c->px, (uint32_t)parity, maxr, c->in_slot, s));
    return CTMR_OK;
}
int round_owner_resolve(ctmr_ctx* c, int parity, uint64_t maxr, cudaStream_t s) {
    if (c->px.world <= 1) return CTMR_OK;
    CU(c, launch_inbox_resolve(c->st, c->px, (uint32_t)parity, maxr, c->in_slot, c->in_pair, s));
    return CTMR_OK;
}
int round_owner_pairs(ctmr_ctx* c, int parity, uint64_t maxr, cudaStream_t s) {
    if (c->px.world <= 1) return CTMR_OK;
    CU(c, launch_inbox_pairs(c->st, c->px, (uint32_t)parity, maxr, c->in_pair, s));
    return CTMR_OK;
}
int round_pull(ctmr_ctx* c, int parity, uint64_t maxr, uint8_t* was_unknown, uint8_t* first, cudaStream_t s) {
    if (c->px.world <= 1) return CTMR_OK;
    CU(c, launch_pull_bits(c->px, (uint32_t)parity, c->cursors + (size_t)parity * kMaxWorld,
                           c->rev + (uint64_t)parity * c->px.world * c->px.X, maxr, was_unknown, first, s));
    return CTMR_OK;
}

// Rounds of E entries with a SHORT last round (a quarter of E): what a call exposes at its end is the reduce chain of its
// last round, so that round is kept small; E stays uniform, which is all the global-index formula needs.
uint64_t device_round_entries(uint64_t n, uint32_t rounds) {
    if (rounds >= 4) return (4 * n + 4 * (uint64_t)rounds - 4) / (4 * (uint64_t)rounds - 3);
    return rounds ? (n + rounds - 1) / rounds : n;
}

uint32_t peer_rounds() {
    static const int r = env_int("CTMR_PEER_ROUNDS", (int)CTMR_PEER_ROUNDS);
    return (uint32_t)(r < 1 ? 1 : (r > kMaxRounds ? kMaxRounds : r));
}

int peer_barrier(ctmr_ctx* c, uint32_t channel, cudaStream_t s) {
    if (c->peer_mode != PEER_IPC) return CTMR_OK;
    CU(c, launch_peer_barrier(c->pf, channel, ++c->epoch[channel], c->st.error_flag, s));
    return CTMR_OK;
}
}  // namespace ctmr_host

namespace {
int reduce_on(ctmr_ctx* c, const ctmr_key* keys, uint64_t m, uint32_t* slot_of, uint32_t* pair_slot, uint8_t* was_unknown,
              uint8_t* first, cudaStream_t s, bool already_inserted = false) {
    if (!already_inserted) CU(c, launch_insert(c->st, keys, m, slot_of, s));
    CU(c, launch_resolve(c->st, keys, m, slot_of, pair_slot, was_unknown, s));
    CU(c, launch_resolve_pairs(c->st, keys, m, pair_slot, was_unknown, first, s));
    return CTMR_OK;
}


// ------------------------------------------------------------------------------------------------ front end plumbing
void fe_destroy(ctmr_ctx* c) {
    FrontEnd* f = c->fe;
    if (!f) return;
    for (FeStage& st : f->stage) {
        cudaFree(st.text); cudaFree(st.leaf_off); cudaFree(st.extra_off); cudaFree(st.leaf_len); cudaFree(st.extra_len);
        cudaFreeHost(st.h_leaf_off); cudaFreeHost(st.h_extra_off); cudaFreeHost(st.h_leaf_len); cudaFreeHost(st.h_extra_len);
        if (st.uploaded) cudaEventDestroy(st.uploaded);
        if (st.consumed) cudaEventDestroy(st.consumed);
    }
    if (f->copy_stream) cudaStreamDestroy(f->copy_stream);
    cudaFree(f->pad_size); cudaFree(f->dec_off); cudaFree(f->dec_len); cudaFree(f->str_bad); cudaFree(f->decoded);
    cudaFree(f->scan_temp); cudaFree(f->entry_status); cudaFree(f->entry_type); cudaFree(f->leaf_src); cudaFree(f->timestamp);
    cudaFree(f->leaf_abs); cudaFree(f->chain_abs); cudaFree(f->tbs_abs); cudaFree(f->leaf_rel); cudaFree(f->leaf_len_out);
    cudaFree(f->chain_len); cudaFree(f->tbs_len); cudaFree(f->issuer_idx); cudaFree(f->status); cudaFree(f->sha);
    cudaFree(f->was_unknown); cudaFree(f->first); cudaFree(f->first_meta); cudaFree(f->exp_hour); cudaFree(f->serial_off);
    cudaFree(f->serial_len); cudaFree(f->spans); cudaFree(f->slots_dev); cudaFree(f->arena); cudaFree(f->pending);
    cudaFree(f->unknown_list); cudaFree(f->unknown_count);
    pem_free(f->pem);
    if (f->ev0) cudaEventDestroy(f->ev0);
    if (f->ev1) cudaEventDestroy(f->ev1);
    if (f->ev2) cudaEventDestroy(f->ev2);
    delete f;
    c->fe = nullptr;
}

uint64_t host_issuer_cert_hash(const std::string& der) {
    const uint32_t len = (uint32_t)der.size();
    uint64_t acc = 0;
    for (uint32_t i = 0; 8u * i < len; ++i) {
        uint64_t w = 0;
        const uint32_t rem = len - 8u * i;
        std::memcpy(&w, der.data() + 8u * i, rem < 8u ? rem : 8u);  // little-endian host (x86-64 / aarch64)
        acc += issuer_cert_word(w, i);
    }
    return issuer_cert_finish(acc, len);
}

// one more certificate in the device mirror: bytes into the arena, slot into the probe table
int fe_add_issuer(ctmr_ctx* c, const std::string& der, uint32_t idx) {
    FrontEnd* f = c->fe;
    if (der.empty()) return CTMR_OK;  // the framing never yields an empty Chain[0]
    if (2 * (f->slots_used + 1) > f->slot_mask + 1)
        return fail(c, CTMR_E_TOO_MANY_ISSUERS, "more distinct Chain[0] certificates than the front end's table holds (raise config.max_issuers)");
    const uint64_t padded = (der.size() + 15) & ~15ull;
    if (f->arena_used + padded > f->arena_cap) {
        uint64_t cap = f->arena_cap ? f->arena_cap * 2 : (64ull << 20);
        while (f->arena_used + padded > cap) cap *= 2;
        uint8_t* bigger = nullptr;
        CU(c, cudaDeviceSynchronize());
        CU(c, cudaMalloc(&bigger, cap));
        if (f->arena_used) CU(c, cudaMemcpyAsync(bigger, f->arena, f->arena_used, cudaMemcpyDeviceToDevice, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
        cudaFree(f->arena);
        f->arena = bigger;
        f->arena_cap = cap;
    }
    std::string buf = der;
    buf.resize(padded, '\0');
    CU(c, cudaMemcpyAsync(f->arena + f->arena_used, buf.data(), padded, cudaMemcpyHostToDevice, c->stream));
    IssuerCertSlot sl{};
    sl.h = host_issuer_cert_hash(der);
    sl.len = (uint32_t)der.size();
    sl.idx = idx;
    sl.arena_off = f->arena_used;
    f->arena_used += padded;
    uint64_t slot = sl.h & f->slot_mask;
    while (f->slots_host[slot].h != 0) slot = (slot + 1) & f->slot_mask;
    f->slots_host[slot] = sl;
    ++f->slots_used;
    CU(c, cudaMemcpyAsync(f->slots_dev + slot, &sl, sizeof sl, cudaMemcpyHostToDevice, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));  // both sources are locals
    return CTMR_OK;
}

int fe_clear_issuers(ctmr_ctx* c) {
    FrontEnd* f = c->fe;
    CU(c, cudaDeviceSynchronize());
    std::fill(f->slots_host.begin(), f->slots_host.end(), IssuerCertSlot{});
    f->slots_used = 0;
    f->arena_used = 0;
    CU(c, cudaMemsetAsync(f->slots_dev, 0, (f->slot_mask + 1) * sizeof(IssuerCertSlot), c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    return CTMR_OK;
}

int ensure_frontend(ctmr_ctx* c) {
    if (c->fe) return CTMR_OK;
    FrontEnd* f = new (std::nothrow) FrontEnd();
    if (!f) return fail(c, CTMR_E_NOMEM, "host allocation failed");
    c->fe = f;
    const uint64_t E = c->stage_entries;
    uint64_t T = E * 6144ull < (64ull << 20) ? (64ull << 20) : E * 6144ull;  // leaf_input + extra_data characters per chunk
    if (const char* ev = getenv("CTMR_FE_TEXT_CAP")) {  // tests shrink it to reach the multi-chunk and packing paths
        const uint64_t v = strtoull(ev, nullptr, 10);
        if (v >= (1ull << 16)) T = v;
    }
    f->cap_entries = E;
    f->cap_text = T;
    f->cap_decoded = T / 4 * 3 + 32 * E + 256;
    auto bail = [&](int code) {
        fe_destroy(c);
        return code;
    };
#define FEM(ptr, bytes)                                                                    \
    do {                                                                                   \
        cudaError_t e_ = cudaMalloc(&(ptr), (bytes));                                      \
        if (e_ != cudaSuccess) {                                                           \
            fail(c, e_ == cudaErrorMemoryAllocation ? CTMR_E_NOMEM : CTMR_E_CUDA,           \
                 std::string("front end: cudaMalloc: ") + cudaGetErrorString(e_));         \
            return bail(e_ == cudaErrorMemoryAllocation ? CTMR_E_NOMEM : CTMR_E_CUDA);      \
        }                                                                                  \
    } while (0)
    for (FeStage& st : f->stage) {
        FEM(st.text, 16 + T + 64);
        FEM(st.leaf_off, E * 8); FEM(st.extra_off, E * 8); FEM(st.leaf_len, E * 4); FEM(st.extra_len, E * 4);
        if (cudaMallocHost(&st.h_leaf_off, E * 8) != cudaSuccess || cudaMallocHost(&st.h_extra_off, E * 8) != cudaSuccess ||
            cudaMallocHost(&st.h_leaf_len, E * 4) != cudaSuccess || cudaMallocHost(&st.h_extra_len, E * 4) != cudaSuccess ||
            cudaEventCreateWithFlags(&st.uploaded, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&st.consumed, cudaEventDisableTiming) != cudaSuccess ||
            cudaMemsetAsync(st.text, 0, 16 + T + 64, c->stream) != cudaSuccess) {
            fail(c, CTMR_E_NOMEM, "front end: staging allocation failed");
            return bail(CTMR_E_NOMEM);
        }
    }
    if (cudaStreamCreateWithFlags(&f->copy_stream, cudaStreamNonBlocking) != cudaSuccess) {
        fail(c, CTMR_E_CUDA, "front end: stream creation failed");
        return bail(CTMR_E_CUDA);
    }
    FEM(f->pad_size, (2 * E + 1) * 8); FEM(f->dec_off, (2 * E + 1) * 8); FEM(f->dec_len, 2 * E * 4); FEM(f->str_bad, 2 * E);
    FEM(f->decoded, f->cap_decoded);
    if (cudaMemsetAsync(f->decoded, 0, f->cap_decoded, c->stream) != cudaSuccess) {  // the 16-byte padding between decoded strings is read (never consumed) by K_map's staging
        fail(c, CTMR_E_CUDA, "front end: arena initialisation failed");
        return bail(CTMR_E_CUDA);
    }
    f->scan_temp_bytes = fe_scan_temp_bytes(2 * E + 1);
    FEM(f->scan_temp, f->scan_temp_bytes ? f->scan_temp_bytes : 16);
    FEM(f->entry_status, E); FEM(f->entry_type, E); FEM(f->leaf_src, E); FEM(f->timestamp, E * 8);
    FEM(f->leaf_abs, E * 8); FEM(f->chain_abs, E * 8); FEM(f->tbs_abs, E * 8);
    FEM(f->leaf_rel, E * 4); FEM(f->leaf_len_out, E * 4); FEM(f->chain_len, E * 4); FEM(f->tbs_len, E * 4); FEM(f->issuer_idx, E * 4);
    FEM(f->status, E); FEM(f->sha, E * 32); FEM(f->was_unknown, E); FEM(f->first, E); FEM(f->first_meta, 2 * E);
    FEM(f->exp_hour, E * 8); FEM(f->serial_off, E * 4); FEM(f->serial_len, E * 4); FEM(f->spans, 4 * E * 4);
    f->slot_mask = pow2_at_least(4ull * c->st.max_issuers) - 1;
    FEM(f->slots_dev, (f->slot_mask + 1) * sizeof(IssuerCertSlot));
    f->slots_host.assign(f->slot_mask + 1, IssuerCertSlot{});
    f->pending_mask = (1ull << 16) - 1;
    FEM(f->pending, (f->pending_mask + 1) * 8);
    f->unknown_cap = 1u << 14;
    FEM(f->unknown_list, f->unknown_cap * 4);
    FEM(f->unknown_count, 16);
#undef FEM
    if (cudaMemsetAsync(f->slots_dev, 0, (f->slot_mask + 1) * sizeof(IssuerCertSlot), c->stream) != cudaSuccess ||
        cudaStreamSynchronize(c->stream) != cudaSuccess ||
        cudaEventCreate(&f->ev0) != cudaSuccess ||
        cudaEventCreate(&f->ev1) != cudaSuccess || cudaEventCreate(&f->ev2) != cudaSuccess) {
        fail(c, CTMR_E_CUDA, "front end: initialisation failed");
        return bail(CTMR_E_CUDA);
    }
    for (const auto& kv : c->issuer_by_der) {  // certificates registered before the front end existed
        int rc = fe_add_issuer(c, kv.first, kv.second);
        if (rc) return rc;
    }
    return CTMR_OK;
}

}  // namespace

namespace ctmr_host {
int frontend_ensure(ctmr_ctx* c) { return ensure_frontend(c); }
}  // namespace ctmr_host

// =================================================================================================
extern "C" {

uint32_t ctmr_abi_version(void) { return CTMR_ABI_VERSION; }

const char* ctmr_last_error(ctmr_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

void* ctmr_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) return nullptr;
    return p;
}
void ctmr_host_free(void* p) {
    if (p) cudaFreeHost(p);
}

int ctmr_create(const ctmr_config* cfg, ctmr_ctx** out) {
    if (!cfg || !out || cfg->struct_size < sizeof(ctmr_config)) return fail(nullptr, CTMR_E_INVALID, "bad config");
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || cfg->device < 0 || cfg->device >= ndev) {
        (void)cudaGetLastError();
        return fail(nullptr, CTMR_E_NO_DEVICE, "no usable CUDA device (libctmr has no CPU fallback)");
    }
    ctmr_ctx* c = new (std::nothrow) ctmr_ctx();
    if (!c) return fail(nullptr, CTMR_E_NOMEM, "host allocation failed");
    auto bail = [&](int code) {
        g_create_error = c->err;
        ctmr_destroy(c);
        return code;
    };
    c->device = cfg->device;
    c->flags = cfg->flags;
    if (build_filter(cfg, c->filter)) {
        c->err = "issuerCNFilter too long (max 446 bytes, 32 prefixes)";
        return bail(CTMR_E_INVALID);
    }
#define CUC(call)                                                              \
    do {                                                                       \
        cudaError_t e_ = (call);                                               \
        if (e_ != cudaSuccess) {                                               \
            c->err = std::string(#call) + ": " + cudaGetErrorString(e_);       \
            return bail(e_ == cudaErrorMemoryAllocation ? CTMR_E_NOMEM : CTMR_E_CUDA); \
        }                                                                      \
    } while (0)
    CUC(cudaSetDevice(c->device));
    cudaDeviceProp prop;
    CUC(cudaGetDeviceProperties(&prop, c->device));
    if (prop.major < 10) {
        c->err = "libctmr is built for sm_100a (B200) only";
        return bail(CTMR_E_NO_DEVICE);
    }
    c->sm_count = prop.multiProcessorCount;
    CUC(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    const uint64_t cap = pow2_at_least(cfg->table_capacity ? cfg->table_capacity : (1ull << 20));
    if (cap > (1ull << 32) - 16) {
        c->err = "table_capacity above 2^32 slots";
        return bail(CTMR_E_INVALID);
    }
    c->st.table_mask = cap - 1;
    const uint32_t plog = cfg->pair_capacity_log2 ? cfg->pair_capacity_log2 : 24;
    const uint32_t mlog = cfg->meta_capacity_log2 ? cfg->meta_capacity_log2 : 20;
    if (plog > 32 || mlog > 26) {
        c->err = "pair_capacity_log2 above 32 or meta_capacity_log2 above 26";
        return bail(CTMR_E_INVALID);
    }
    c->st.pair_mask = (1ull << plog) - 1;
    c->st.meta_mask = (1ull << mlog) - 1;  // IssuerMetadata string identities: O(issuers x few)
    c->st.max_issuers = cfg->max_issuers ? cfg->max_issuers : 65536;
    // ONE allocation for everything another rank of a group may address (tables, histograms, barrier flags, issuer
    // registry): one CUDA IPC handle exports it; on a single GPU it is simply this ctx's state
    c->lay = make_layout(cap, c->st.pair_mask + 1, c->st.meta_mask + 1, c->st.max_issuers);
    CUC(cudaMalloc(&c->shared, c->lay.total));
    CUC(cudaMemsetAsync(c->shared, 0, c->lay.total, c->stream));
    c->st.table = reinterpret_cast<KnownSlot*>(c->shared + c->lay.table);
    c->st.pairs = reinterpret_cast<PairSlot*>(c->shared + c->lay.pairs);
    c->st.meta = reinterpret_cast<MetaSlot*>(c->shared + c->lay.meta);
    c->st.issuer_counts = reinterpret_cast<unsigned long long*>(c->shared + c->lay.issuer_counts);
    c->st.status_counts = reinterpret_cast<unsigned long long*>(c->shared + c->lay.status_counts);
    CUC(cudaMalloc(&c->small_dev, 128 * sizeof(unsigned long long)));
    CUC(cudaMemsetAsync(c->small_dev, 0, 128 * sizeof(unsigned long long), c->stream));
    c->st.slots_used = c->small_dev + 72;     // [1]
    c->st.error_flag = reinterpret_cast<int*>(c->small_dev + 73);
    {
        uint8_t* self[1] = {c->shared};
        attach_views(c, self, 1, 0);  // a single GPU is a group of one
    }
    c->stage_entries = cfg->max_batch_entries ? (cfg->max_batch_entries < kStageEntries ? cfg->max_batch_entries : kStageEntries)
                                              : kStageEntries;
    const uint64_t want_bytes = cfg->max_batch_bytes ? cfg->max_batch_bytes : c->stage_entries * 2048ull;
    c->stage_bytes = want_bytes < kStageBytes ? want_bytes : kStageBytes;
    c->cfg_round_entries = cfg->max_round_entries;
    c->px.world = 1;
    if (const char* ev = getenv("CTMR_BUCKET_BY_LENGTH")) c->bucket_by_length = atoi(ev) != 0;
    if (const char* ev = getenv("CTMR_FUSE_INSERT")) c->fuse_insert = atoi(ev) != 0;
    if (const char* ev = getenv("CTMR_MAP_VARIANT")) if (atoi(ev) != 2) c->fuse_insert = false;  // only the streaming kernel fuses
    CUC(cudaStreamSynchronize(c->stream));
#undef CUC
    *out = c;
    return CTMR_OK;
}

void ctmr_destroy(ctmr_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    stages_destroy(c);
    for (uint32_t r = 0; r < kMaxWorld; ++r) {
        if (c->ipc_base[r]) cudaIpcCloseMemHandle(c->ipc_base[r]);
        if (c->ipc_xchg[r]) cudaIpcCloseMemHandle(c->ipc_xchg[r]);
    }
    cudaFree(c->xchg); cudaFree(c->cursors); cudaFree(c->rev); cudaFree(c->in_slot); cudaFree(c->in_pair);
    for (cudaEvent_t e : c->ev_pulled)
        if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : c->ev_g)
        if (e) cudaEventDestroy(e);
    cudaFree(c->shared); cudaFree(c->small_dev);
    cudaFree(c->issuer_map_dev); cudaFree(c->keys_scratch); cudaFree(c->slot_scratch); cudaFree(c->pair_scratch);
    cudaFree(c->bits_scratch); cudaFree(c->meta_scratch); cudaFree(c->order_scratch); cudaFree(c->len_hist);
    for (int k = 0; k < kMaxRounds; ++k) {
        cudaFree(c->len_hist_sub[k]);
        if (c->ev_map0[k]) cudaEventDestroy(c->ev_map0[k]);
        if (c->ev_map1[k]) cudaEventDestroy(c->ev_map1[k]);
        if (c->ev_red1[k]) cudaEventDestroy(c->ev_red1[k]);
        if (c->ev_tok[k]) cudaEventDestroy(c->ev_tok[k]);
    }
    if (c->ev_join_a2) cudaEventDestroy(c->ev_join_a2);
    if (c->stream_a2) cudaStreamDestroy(c->stream_a2);
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    if (c->ev_join_a) cudaEventDestroy(c->ev_join_a);
    if (c->ev_join_b) cudaEventDestroy(c->ev_join_b);
    if (c->stream_a) cudaStreamDestroy(c->stream_a);
    if (c->stream_b) cudaStreamDestroy(c->stream_b);
    if (c->stream) cudaStreamDestroy(c->stream);
    fe_destroy(c);
    delete c;
}

// ------------------------------------------------------------------------------------------------ issuers
// The registry (Issuer.ID digest -> dense index) is a find-or-insert table in the device memory of the group's rank 0,
// reached with system-scope atomics: whichever rank meets an issuer first, every rank gets the same index for it.
// The host keeps memos only (DER -> index, digest -> index, index -> digest), filled from the device.
}  // extern "C"

namespace ctmr_host {

int refresh_digests(ctmr_ctx* c) {
    unsigned long long cnt = 0;
    CU(c, cudaMemcpyAsync(&cnt, c->reg.counter, sizeof cnt, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    if (cnt > c->reg.max_issuers) cnt = c->reg.max_issuers;
    const size_t have = c->digests.size();
    if (cnt <= have) return CTMR_OK;
    std::vector<uint8_t> rows((cnt - have) * 32);
    CU(c, cudaMemcpyAsync(rows.data(), c->reg.by_index + 32 * have, rows.size(), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    for (size_t i = have; i < cnt; ++i) {
        const uint8_t* row = rows.data() + 32 * (i - have);
        bool zero = true;
        for (int k = 0; k < 32; ++k) zero &= row[k] == 0;
        if (zero) break;  // index handed out by another rank's kernel, digest not written yet: next time
        std::array<uint8_t, 32> a;
        std::memcpy(a.data(), row, 32);
        c->digests.push_back(a);
        c->issuer_by_digest.emplace(std::string(reinterpret_cast<const char*>(row), 32), (uint32_t)i);
    }
    return CTMR_OK;
}

// digest -> dense index; `insert` registers an unknown digest (state written by an earlier process, preloads)
int lookup_digest(ctmr_ctx* c, const uint8_t digest[32], bool insert, uint32_t* idx_out, bool* found) {
    const std::string dk(reinterpret_cast<const char*>(digest), 32);
    *found = false;
    auto it = c->issuer_by_digest.find(dk);
    if (it == c->issuer_by_digest.end()) {
        int rc = refresh_digests(c);
        if (rc) return rc;
        it = c->issuer_by_digest.find(dk);
    }
    if (it != c->issuer_by_digest.end()) {
        *idx_out = it->second;
        *found = true;
        return CTMR_OK;
    }
    if (!insert) return CTMR_OK;
    uint8_t* d_dig = reinterpret_cast<uint8_t*>(c->small_dev + 100);  // [4] words = 32 bytes
    uint32_t* d_idx = reinterpret_cast<uint32_t*>(c->small_dev + 104);
    uint32_t idx = CTMR_ISSUER_BAD;
    CU(c, cudaMemcpyAsync(d_dig, digest, 32, cudaMemcpyHostToDevice, c->stream));
    CU(c, launch_issuer_registry(c->reg, d_dig, nullptr, 1, d_idx, c->st.error_flag, c->stream));
    CU(c, cudaMemcpyAsync(&idx, d_idx, 4, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    if (idx == CTMR_ISSUER_BAD) {
        ctmr_check_device(c, nullptr);  // clears the flag
        return fail(c, CTMR_E_TOO_MANY_ISSUERS, "more distinct issuers than config.max_issuers");
    }
    c->issuer_by_digest.emplace(dk, idx);
    *idx_out = idx;
    *found = true;
    return refresh_digests(c);
}

int upload_issuer_map(ctmr_ctx* c, const uint32_t* dense, uint32_t n) {
    if (n > c->issuer_map_cap) {
        cudaFree(c->issuer_map_dev);
        c->issuer_map_dev = nullptr;
        c->issuer_map_cap = 0;
        CU(c, cudaMalloc(&c->issuer_map_dev, (size_t)n * sizeof(uint32_t)));
        c->issuer_map_cap = n;
    }
    CU(c, cudaMemcpyAsync(c->issuer_map_dev, dense, n * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    return CTMR_OK;
}

}  // namespace ctmr_host

extern "C" {

int ctmr_register_issuers(ctmr_ctx* c, const uint8_t* blob, const uint64_t* offsets, uint32_t n, uint32_t* dense_out) {
    if (!c || (n && (!blob || !offsets || !dense_out))) return fail(c, CTMR_E_INVALID, "bad argument");
    CU(c, cudaSetDevice(c->device));
    std::vector<uint32_t> fresh;  // positions whose DER has not been seen before
    std::vector<std::string> ders(n);
    for (uint32_t k = 0; k < n; ++k) {
        if (offsets[k + 1] < offsets[k]) return fail(c, CTMR_E_INVALID, "issuer offsets not monotonic");
        ders[k].assign(reinterpret_cast<const char*>(blob + offsets[k]), (size_t)(offsets[k + 1] - offsets[k]));
        auto it = c->issuer_by_der.find(ders[k]);
        if (it != c->issuer_by_der.end()) {
            dense_out[k] = it->second;
        } else {
            bool dup = false;
            for (uint32_t f : fresh)
                if (ders[f] == ders[k]) { dup = true; break; }
            if (!dup) fresh.push_back(k);
            dense_out[k] = CTMR_ISSUER_NONE;  // patched below
        }
    }
    if (!fresh.empty()) {
        // only never-seen certificates go to the GPU: parse + SHA-256(SPKI) there, then find-or-insert of the digest
        // in the registry (rank 0's memory); indices and digests come back
        std::vector<uint8_t> packed;
        std::vector<uint64_t> poff(1, 0);
        for (uint32_t f : fresh) {
            packed.insert(packed.end(), ders[f].begin(), ders[f].end());
            poff.push_back(packed.size());
        }
        const uint32_t nf = (uint32_t)fresh.size();
        uint8_t *d_blob = nullptr, *d_dig = nullptr, *d_ok = nullptr;
        uint64_t* d_off = nullptr;
        uint32_t* d_idx = nullptr;
        auto release = [&]() { cudaFree(d_blob); cudaFree(d_off); cudaFree(d_dig); cudaFree(d_ok); cudaFree(d_idx); };
        CU(c, cudaMalloc(&d_blob, packed.size() + 64));
        CU(c, cudaMalloc(&d_off, poff.size() * sizeof(uint64_t)));
        CU(c, cudaMalloc(&d_dig, nf * 32));
        CU(c, cudaMalloc(&d_ok, nf));
        CU(c, cudaMalloc(&d_idx, nf * sizeof(uint32_t)));
        CU(c, cudaMemcpyAsync(d_blob, packed.data(), packed.size(), cudaMemcpyHostToDevice, c->stream));
        CU(c, cudaMemcpyAsync(d_off, poff.data(), poff.size() * sizeof(uint64_t), cudaMemcpyHostToDevice, c->stream));
        CU(c, launch_issuer_prepare(d_blob, d_off, nf, d_dig, d_ok, c->stream));
        CU(c, launch_issuer_registry(c->reg, d_dig, d_ok, nf, d_idx, c->st.error_flag, c->stream));
        std::vector<uint8_t> dig(nf * 32), ok(nf);
        std::vector<uint32_t> idx(nf);
        CU(c, cudaMemcpyAsync(dig.data(), d_dig, nf * 32, cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaMemcpyAsync(ok.data(), d_ok, nf, cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaMemcpyAsync(idx.data(), d_idx, nf * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
        release();
        for (uint32_t i = 0; i < nf; ++i) {
            if (ok[i] && idx[i] == CTMR_ISSUER_BAD) {
                ctmr_check_device(c, nullptr);  // clears the flag
                return fail(c, CTMR_E_TOO_MANY_ISSUERS, "more distinct issuers than config.max_issuers");
            }
            if (ok[i]) c->issuer_by_digest.emplace(std::string(reinterpret_cast<const char*>(dig.data() + 32 * i), 32), idx[i]);
            c->issuer_by_der.emplace(ders[fresh[i]], idx[i]);
            if (c->fe) {
                int rc2 = fe_add_issuer(c, ders[fresh[i]], idx[i]);
                if (rc2) return rc2;
            }
        }
        for (uint32_t k = 0; k < n; ++k)
            if (dense_out[k] == CTMR_ISSUER_NONE) dense_out[k] = c->issuer_by_der[ders[k]];
        int rc = refresh_digests(c);
        if (rc) return rc;
    }
    return CTMR_OK;
}

int ctmr_issuer_digest(ctmr_ctx* c, uint32_t idx, uint8_t out[32]) {
    if (!c || !out) return fail(c, CTMR_E_INVALID, "bad argument");
    if (idx >= c->digests.size()) {
        CU(c, cudaSetDevice(c->device));
        int rc = refresh_digests(c);  // another rank of the group may have registered it
        if (rc) return rc;
    }
    if (idx >= c->digests.size()) return fail(c, CTMR_E_INVALID, "no such issuer");
    std::memcpy(out, c->digests[idx].data(), 32);
    return CTMR_OK;
}

uint32_t ctmr_issuer_count(ctmr_ctx* c) {
    if (!c) return 0;
    if (cudaSetDevice(c->device) == cudaSuccess) refresh_digests(c);
    return (uint32_t)c->digests.size();
}

// ------------------------------------------------------------------------------------------------ device entry points
int ctmr_map_device(ctmr_ctx* c, const ctmr_dev_batch* b, const ctmr_dev_out* o, void* stream) {
    if (!c || !b || !o) return fail(c, CTMR_E_INVALID, "bad argument");
    if (b->n && (!b->blob || !b->offsets)) return fail(c, CTMR_E_INVALID, "null batch buffers");
    CU(c, cudaSetDevice(c->device));
    MapParams p;
    fill_map_params(c, b, o, p);
    cudaStream_t s = stream ? (cudaStream_t)stream : c->stream;
    if (c->bucket_by_length && b->n > 64 && p.sha256) {  // the light (no-fingerprint) kernel has no lock-step loop to balance
        if (b->n > c->order_cap) {
            CU(c, cudaDeviceSynchronize());
            cudaFree(c->order_scratch);
            c->order_scratch = nullptr;
            c->order_cap = 0;
            CU(c, cudaMalloc(&c->order_scratch, b->n * sizeof(uint32_t)));
            c->order_cap = b->n;
        }
        if (!c->len_hist) CU(c, cudaMalloc(&c->len_hist, 256 * sizeof(unsigned int)));
        CU(c, launch_len_order(b->offsets, b->lens, b->n, b->blob_bytes, c->len_hist, c->order_scratch, s));
        p.order = c->order_scratch;
    }
    CU(c, launch_map(p, c->sm_count, s));
    return CTMR_OK;
}

int ctmr_reduce_device(ctmr_ctx* c, const ctmr_key* keys, uint64_t m, uint8_t* was_unknown, uint8_t* first, void* stream) {
    if (!c || (m && !keys)) return fail(c, CTMR_E_INVALID, "bad argument");
    CU(c, cudaSetDevice(c->device));
    int rc = ensure_scratch(c, m);
    if (rc) return rc;
    cudaStream_t s = stream ? (cudaStream_t)stream : c->stream;
    return reduce_on(c, keys, m, c->slot_scratch, c->pair_scratch, was_unknown ? was_unknown : c->bits_scratch,
                     first ? first : c->bits_scratch + m, s);
}

int ctmr_process_device(ctmr_ctx* c, const ctmr_dev_batch* b, const ctmr_dev_out* o, void* stream) {
    if (!c || !b || !o) return fail(c, CTMR_E_INVALID, "bad argument");
    if (b->n && (!b->blob || !b->offsets)) return fail(c, CTMR_E_INVALID, "null batch buffers");
    CU(c, cudaSetDevice(c->device));
    int rc = ensure_scratch(c, b->n);
    if (rc) return rc;
    if (c->bucket_by_length && b->n > c->order_cap) {
        CU(c, cudaDeviceSynchronize());
        cudaFree(c->order_scratch);
        c->order_scratch = nullptr;
        c->order_cap = 0;
        CU(c, cudaMalloc(&c->order_scratch, b->n * sizeof(uint32_t)));
        c->order_cap = b->n;
    }
    if (!c->stream_a) {
        CU(c, cudaStreamCreateWithFlags(&c->stream_a, cudaStreamNonBlocking));
        CU(c, cudaStreamCreateWithFlags(&c->stream_a2, cudaStreamNonBlocking));
        CU(c, cudaEventCreateWithFlags(&c->ev_join_a2, cudaEventDisableTiming));
        CU(c, cudaStreamCreateWithFlags(&c->stream_b, cudaStreamNonBlocking));
        CU(c, cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
        CU(c, cudaEventCreateWithFlags(&c->ev_join_a, cudaEventDisableTiming));
        CU(c, cudaEventCreateWithFlags(&c->ev_join_b, cudaEventDisableTiming));
        for (int k = 0; k < kMaxRounds; ++k) {
            CU(c, cudaEventCreate(&c->ev_map0[k]));
            CU(c, cudaEventCreate(&c->ev_map1[k]));
            CU(c, cudaEventCreate(&c->ev_red1[k]));
            CU(c, cudaEventCreateWithFlags(&c->ev_tok[k], cudaEventDisableTiming));
            CU(c, cudaMalloc(&c->len_hist_sub[k], 256 * sizeof(unsigned int)));
        }
        for (cudaEvent_t& e : c->ev_pulled) CU(c, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    const bool want_meta = o->first_issuer_dn || o->first_crldp;
    if (want_meta && !(o->issuer_name_off && o->issuer_name_len && o->crldp_off && o->crldp_len))
        return fail(c, CTMR_E_INVALID, "first_issuer_dn / first_crldp need the four span outputs as well");
    cudaStream_t user = stream ? (cudaStream_t)stream : c->stream;
    // The map half is INT-pipe bound and the reduce half is latency/atomic bound: run sub-batch
    // k+1's K_map (stream A) while sub-batch k's insert/resolve/pairs run (stream B).
    // In a multi-process group the call is collective: every rank runs CTMR_PEER_ROUNDS rounds (empty ones included)
    // and meets the others at two barriers per round; round k of rank r carries the global indices
    // first_index + (k * world + r) * E .. , i.e. the rounds are ordered, and inside a round the ranks.
    const uint32_t world = c->st.peer.world, rank = c->st.peer.rank;
    const bool coll = c->peer_mode == PEER_IPC && world > 1;
    if (c->peer_mode == PEER_GROUP && world > 1)
        return fail(c, CTMR_E_INVALID, "members of an in-process group are driven through ctmr_group_process_batch");
    static const int rounds_env = env_int("CTMR_DEVICE_ROUNDS", 0);   // experiments: rounds of the single-GPU call
    static const int map_streams = env_int("CTMR_MAP_STREAMS", 2);    // K_map launches alternate between two streams
    int nsub = coll ? (int)peer_rounds() : (b->n >= (1u << 21) ? 8 : (b->n >= (1u << 18) ? 2 : 1));
    if (!coll && rounds_env > 0 && b->n >= (1u << 18)) nsub = rounds_env > kMaxRounds ? kMaxRounds : rounds_env;
    const uint64_t per_round = device_round_entries(b->n, (uint32_t)nsub);
    if (coll && per_round > c->px.X)
        return fail(c, CTMR_E_BATCH_TOO_LARGE, "entries per round exceed the key-exchange regions: raise config.max_round_entries to ceil(n / ctmr_peer_rounds())");
    ctmr_key* keys = o->keys ? o->keys : c->keys_scratch;
    uint8_t* wu = o->was_unknown ? o->was_unknown : c->bits_scratch;
    uint8_t* fi = o->first_issuer_hour ? o->first_issuer_hour : c->bits_scratch + b->n;
    CU(c, cudaEventRecord(c->ev_fork, user));
    CU(c, cudaStreamWaitEvent(c->stream_a, c->ev_fork, 0));
    CU(c, cudaStreamWaitEvent(c->stream_a2, c->ev_fork, 0));
    CU(c, cudaStreamWaitEvent(c->stream_b, c->ev_fork, 0));
    for (int k = 0; k < nsub; ++k) {
        uint64_t lo, hi;
        lo = std::min<uint64_t>(b->n, per_round * k);
        hi = std::min<uint64_t>(b->n, per_round * (k + 1));
        const uint64_t cnt = hi - lo;
        ctmr_dev_batch sb = *b;
        sb.offsets = b->offsets + lo;
        sb.lens = b->lens ? b->lens + lo : nullptr;
        sb.n = cnt;
        sb.issuer_idx = b->issuer_idx ? b->issuer_idx + lo : nullptr;
        sb.first_index = coll ? b->first_index + ((uint64_t)k * world + rank) * per_round : b->first_index + lo;
        ctmr_dev_out so{};
        so.status = o->status ? o->status + lo : nullptr;
        so.sha256 = o->sha256 ? o->sha256 + lo * 32 : nullptr;
        so.exp_hour = o->exp_hour ? o->exp_hour + lo : nullptr;
        so.serial_off = o->serial_off ? o->serial_off + lo : nullptr;
        so.serial_len = o->serial_len ? o->serial_len + lo : nullptr;
        so.keys = keys + lo;
        so.issuer_name_off = o->issuer_name_off ? o->issuer_name_off + lo : nullptr;
        so.issuer_name_len = o->issuer_name_len ? o->issuer_name_len + lo : nullptr;
        so.crldp_off = o->crldp_off ? o->crldp_off + lo : nullptr;
        so.crldp_len = o->crldp_len ? o->crldp_len + lo : nullptr;
        const int parity = k % (int)kParities;
        // consecutive K_map launches on alternating streams: the next launch's CTAs fill the SMs the previous one's
        // draining tail leaves idle (a persistent grid ends with its slowest warps)
        cudaStream_t sa = (map_streams > 1 && (k & 1)) ? c->stream_a2 : c->stream_a;
        const bool fused = c->fuse_insert || world > 1;   // a group always fuses: the routing happens in K_map's epilogue
        MapParams p;
        fill_map_params(c, &sb, &so, p, 3, fused ? c->slot_scratch + lo : nullptr, parity);
        if (world > 1 && k >= (int)kParities) CU(c, cudaStreamWaitEvent(sa, c->ev_pulled[parity], 0));  // the parity's regions are free again
        CU(c, cudaEventRecord(c->ev_map0[k], sa));
        rc = round_begin(c, parity, sa);
        if (rc) return rc;
        if (c->bucket_by_length && cnt > 64 && p.sha256) {
            CU(c, launch_len_order(sb.offsets, sb.lens, cnt, sb.blob_bytes, c->len_hist_sub[k], c->order_scratch + lo, sa));
            p.order = c->order_scratch + lo;
        }
        CU(c, launch_map(p, c->sm_count, sa));
        CU(c, cudaEventRecord(c->ev_map1[k], sa));
        rc = round_publish(c, parity, sa);  // region sizes to the owners (outside K_map's timed bracket)
        if (rc) return rc;
        CU(c, cudaEventRecord(c->ev_tok[k], sa));   // ordering token: K_map + the published sizes
        CU(c, cudaStreamWaitEvent(c->stream_b, c->ev_tok[k], 0));
        cudaStream_t sbm = c->stream_b;
        if (!fused) CU(c, launch_insert(c->st, keys + lo, cnt, c->slot_scratch + lo, sbm));
        rc = peer_barrier(c, CH_DEV_MAP, sbm);  // every rank's appends of rounds <= k have landed in the owners' inboxes
        if (rc) return rc;
        rc = round_owner_insert(c, parity, per_round, sbm);
        if (rc) return rc;
        CU(c, launch_resolve(c->st, keys + lo, cnt, c->slot_scratch + lo, c->pair_scratch + lo, wu + lo, sbm));
        rc = round_owner_resolve(c, parity, per_round, sbm);
        if (rc) return rc;
        CU(c, launch_resolve_pairs(c->st, keys + lo, cnt, c->pair_scratch + lo, wu + lo, fi + lo, sbm));
        rc = round_owner_pairs(c, parity, per_round, sbm);
        if (rc) return rc;
        rc = peer_barrier(c, CH_DEV_RESOLVE, sbm);  // every owner has the result bits of this round's records ready
        if (rc) return rc;
        rc = round_pull(c, parity, per_round, wu + lo, fi + lo, sbm);
        if (rc) return rc;
        if (world > 1) CU(c, cudaEventRecord(c->ev_pulled[parity], sbm));
        if (want_meta) {
            if (world > 1) return fail(c, CTMR_E_INVALID, "first_issuer_dn / first_crldp of a group come from the host-buffer call");
            CU(c, launch_meta(c->st, sb.blob, sb.offsets, keys + lo, cnt, wu + lo, so.issuer_name_off, so.issuer_name_len, so.crldp_off,
                              so.crldp_len, c->meta_scratch + 2 * lo, o->first_issuer_dn ? o->first_issuer_dn + lo : nullptr,
                              o->first_crldp ? o->first_crldp + lo : nullptr, sbm));
        }
        CU(c, cudaEventRecord(c->ev_red1[k], c->stream_b));
    }
    c->last_sub = nsub;
    c->last_map_streams = map_streams > 1 ? 2 : 1;
    CU(c, cudaEventRecord(c->ev_join_a2, c->stream_a2));
    CU(c, cudaStreamWaitEvent(user, c->ev_join_a2, 0));
    CU(c, cudaEventRecord(c->ev_join_a, c->stream_a));
    CU(c, cudaEventRecord(c->ev_join_b, c->stream_b));
    CU(c, cudaStreamWaitEvent(user, c->ev_join_a, 0));
    CU(c, cudaStreamWaitEvent(user, c->ev_join_b, 0));
    return CTMR_OK;
}

/* CUDA-event timings of the last ctmr_process_device call (after the caller synchronised):
 * map_ms = sum of the K_map stage durations on their stream, total_ms = first map start -> last reduce end */
uint32_t ctmr_peer_rounds(void) { return peer_rounds(); }
uint64_t ctmr_peer_round_entries(uint64_t n) { return device_round_entries(n, peer_rounds()); }

int ctmr_profile_last(ctmr_ctx* c, float* map_ms, float* total_ms) {
    if (!c || c->last_sub <= 0) return fail(c, CTMR_E_INVALID, "no ctmr_process_device call to report");
    CU(c, cudaSetDevice(c->device));
    float m = 0.f, t = 0.f;
    if (c->last_map_streams > 1) {
        // launches overlap (alternating streams): K_map's time is the span from the first launch's start to the last one's end,
        // during which some K_map CTA is always resident
        float best = 0.f;
        for (int k = 0; k < c->last_sub; ++k) {
            float d = 0.f;
            CU(c, cudaEventElapsedTime(&d, c->ev_map0[0], c->ev_map1[k]));
            best = d > best ? d : best;
        }
        m = best;
    } else {
        for (int k = 0; k < c->last_sub; ++k) {
            float d = 0.f;
            CU(c, cudaEventElapsedTime(&d, c->ev_map0[k], c->ev_map1[k]));
            m += d;
        }
    }
    CU(c, cudaEventElapsedTime(&t, c->ev_map0[0], c->ev_red1[c->last_sub - 1]));
    if (map_ms) *map_ms = m;
    if (total_ms) *total_ms = t;
    return CTMR_OK;
}

int ctmr_read_histogram_device(ctmr_ctx* c, uint64_t* counts_dst, uint32_t n_slots, uint64_t* status_dst, void* stream) {
    if (!c || n_slots > c->st.max_issuers) return fail(c, CTMR_E_INVALID, "bad argument");
    CU(c, cudaSetDevice(c->device));
    cudaStream_t s = stream ? (cudaStream_t)stream : c->stream;
    if (counts_dst && n_slots)
        CU(c, cudaMemcpyAsync(counts_dst, c->st.issuer_counts, n_slots * sizeof(uint64_t), cudaMemcpyDeviceToDevice, s));
    if (status_dst)
        CU(c, cudaMemcpyAsync(status_dst, c->st.status_counts, CTMR_ST__COUNT * sizeof(uint64_t), cudaMemcpyDeviceToDevice, s));
    return CTMR_OK;
}

int ctmr_reset_device(ctmr_ctx* c, void* stream) {
    if (!c) return CTMR_E_INVALID;
    CU(c, cudaSetDevice(c->device));
    cudaStream_t s = stream ? (cudaStream_t)stream : c->stream;
    // multi-process group: collective.  Nobody may still be inserting into this shard when it is cleared, and nobody
    // may insert into it again before it has been cleared.
    int rc = peer_barrier(c, CH_RESET_A, s);
    if (rc) return rc;
    CU(c, cudaMemsetAsync(c->st.table, 0, (c->st.table_mask + 1) * sizeof(KnownSlot), s));
    CU(c, cudaMemsetAsync(c->st.pairs, 0, (c->st.pair_mask + 1) * sizeof(PairSlot), s));
    CU(c, cudaMemsetAsync(c->st.meta, 0, (c->st.meta_mask + 1) * sizeof(MetaSlot), s));
    CU(c, cudaMemsetAsync(c->st.issuer_counts, 0, c->st.max_issuers * sizeof(unsigned long long), s));
    CU(c, cudaMemsetAsync(c->st.status_counts, 0, CTMR_ST__COUNT * sizeof(unsigned long long), s));
    CU(c, cudaMemsetAsync(c->small_dev + 64, 0, 16 * sizeof(unsigned long long), s));
    return peer_barrier(c, CH_RESET_B, s);
}

// Reads AND clears the sticky device-side failure flag: one failed batch does not poison the ctx.
int ctmr_check_device(ctmr_ctx* c, void* stream) {
    if (!c) return CTMR_E_INVALID;
    CU(c, cudaSetDevice(c->device));
    cudaStream_t s = stream ? (cudaStream_t)stream : c->stream;
    int flag = 0;
    CU(c, cudaMemcpyAsync(&flag, c->st.error_flag, sizeof flag, cudaMemcpyDeviceToHost, s));
    CU(c, cudaStreamSynchronize(s));
    if (!flag) return CTMR_OK;
    CU(c, cudaMemsetAsync(c->st.error_flag, 0, sizeof(int), s));
    CU(c, cudaStreamSynchronize(s));
    switch (flag) {
    case CTMR_E_TABLE_FULL: return fail(c, flag, "known-certificate table is full; raise config.table_capacity");
    case CTMR_E_PAIR_TABLE_FULL: return fail(c, flag, "(issuer, expDate) table is full; raise config.pair_capacity_log2");
    case CTMR_E_META_TABLE_FULL: return fail(c, flag, "IssuerMetadata string-identity table is full; raise config.meta_capacity_log2");
    case CTMR_E_TOO_MANY_ISSUERS: return fail(c, flag, "more distinct issuers than config.max_issuers");
    case CTMR_E_PEER_TIMEOUT: return fail(c, flag, "a rank of the group did not reach a barrier in time (peer failed, or the collective calls diverged; CTMR_PEER_TIMEOUT_MS)");
    default: return fail(c, CTMR_E_CUDA, "device-side failure flag set");
    }
}

// ------------------------------------------------------------------------------------------------ warm start / checkpoint
}  // extern "C"

namespace ctmr_host {
// Seeds keys with the indices first_index .. first_index + n - 1 (the caller keeps them below every later batch
// index).  Inserts go to the set's owner, so in a group any member can run it; not collective: the group is quiescent.
int preload_impl(ctmr_ctx* c, int64_t exp_hour, const uint8_t digest[32], const uint8_t* serial_blob, const uint64_t* serial_offsets,
                 uint64_t n, uint64_t first_index) {
    if (exp_hour > INT32_MAX || exp_hour < INT32_MIN) return fail(c, CTMR_E_INVALID, "exp_hour out of range");
    CU(c, cudaSetDevice(c->device));
    uint32_t issuer = 0;
    bool found = false;
    int rc = lookup_digest(c, digest, true, &issuer, &found);  // the issuer may be unknown so far (state written by an earlier process)
    if (rc) return rc;
    if (!n) return CTMR_OK;
    if (c->st.peer.world > 1) {
        const uint32_t owner = key_owner((int32_t)exp_hour, issuer, c->st.peer.world);
        if (owner != c->st.peer.rank)
            return fail(c, CTMR_E_INVALID, "this set is owned by rank " + std::to_string(owner) + " of the group: preload it there");
    }
    std::vector<ctmr_key> keys(n);
    for (uint64_t i = 0; i < n; ++i) {
        const uint64_t len = serial_offsets[i + 1] - serial_offsets[i];
        if (serial_offsets[i + 1] < serial_offsets[i] || len == 0 || len > CTMR_MAX_SERIAL)
            return fail(c, CTMR_E_INVALID, "preloaded serial empty or longer than CTMR_MAX_SERIAL");
        std::memset(&keys[i], 0, sizeof(ctmr_key));
        keys[i].index = first_index + i;
        keys[i].exp_hour = (int32_t)exp_hour;
        keys[i].issuer = issuer;
        keys[i].serial_len = (uint8_t)len;
        std::memcpy(keys[i].serial, serial_blob + serial_offsets[i], len);
        keys[i].valid = 1;
    }
    return reduce_keys_host(c, keys.data(), n);
}

int reduce_keys_host(ctmr_ctx* c, const ctmr_key* keys, uint64_t n) {
    CU(c, cudaSetDevice(c->device));
    // in chunks of the scratch size: a preload's chunks come in index order, an import's keys are distinct, so
    // lowest-index-wins holds across the chunks either way
    constexpr uint64_t kChunk = 1ull << 20;
    int rc = ensure_scratch(c, std::min(n, kChunk));
    if (rc) return rc;
    for (uint64_t lo = 0; lo < n; lo += c->scratch_cap) {
        const uint64_t m = std::min(n - lo, c->scratch_cap);
        CU(c, cudaMemcpyAsync(c->keys_scratch, keys + lo, m * sizeof(ctmr_key), cudaMemcpyHostToDevice, c->stream));
        rc = reduce_on(c, c->keys_scratch, m, c->slot_scratch, c->pair_scratch, c->bits_scratch, c->bits_scratch + m, c->stream);
        if (rc) return rc;
        CU(c, cudaStreamSynchronize(c->stream));
    }
    return ctmr_check_device(c, nullptr);
}
}  // namespace ctmr_host

extern "C" {

int ctmr_preload_known(ctmr_ctx* c, int64_t exp_hour, const uint8_t digest[32], const uint8_t* serial_blob,
                       const uint64_t* serial_offsets, uint64_t n) {
    if (!c || !digest || (n && (!serial_blob || !serial_offsets))) return fail(c, CTMR_E_INVALID, "bad argument");
    if (c->group) return fail(c, CTMR_E_INVALID, "member of a group: use ctmr_group_preload_known");
    // key records with the indices next_index .. BELOW every later batch index: preloaded keys always win "first seen"
    int rc = preload_impl(c, exp_hour, digest, serial_blob, serial_offsets, n, c->next_index);
    if (rc == CTMR_OK) c->next_index += n;
    return rc;
}

}  // extern "C"

namespace ctmr_host {

// one shard's tables and histograms, in a fixed order (device <-> host)
uint64_t snap_shard_bytes(ctmr_ctx* c) {
    return (c->st.table_mask + 1) * sizeof(KnownSlot) + (c->st.pair_mask + 1) * sizeof(PairSlot) + (c->st.meta_mask + 1) * sizeof(MetaSlot) +
           c->st.max_issuers * sizeof(uint64_t) + CTMR_ST__COUNT * sizeof(uint64_t);
}

int snap_shard_save(ctmr_ctx* c, uint8_t* p) {
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaDeviceSynchronize());
    const uint64_t t = (c->st.table_mask + 1) * sizeof(KnownSlot), pr = (c->st.pair_mask + 1) * sizeof(PairSlot),
                   m = (c->st.meta_mask + 1) * sizeof(MetaSlot), ic = c->st.max_issuers * sizeof(uint64_t);
    CU(c, cudaMemcpy(p, c->st.table, t, cudaMemcpyDeviceToHost)); p += t;
    CU(c, cudaMemcpy(p, c->st.pairs, pr, cudaMemcpyDeviceToHost)); p += pr;
    CU(c, cudaMemcpy(p, c->st.meta, m, cudaMemcpyDeviceToHost)); p += m;
    CU(c, cudaMemcpy(p, c->st.issuer_counts, ic, cudaMemcpyDeviceToHost)); p += ic;
    CU(c, cudaMemcpy(p, c->st.status_counts, CTMR_ST__COUNT * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    return CTMR_OK;
}

int snap_shard_load(ctmr_ctx* c, const uint8_t* p) {
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaDeviceSynchronize());
    const uint64_t t = (c->st.table_mask + 1) * sizeof(KnownSlot), pr = (c->st.pair_mask + 1) * sizeof(PairSlot),
                   m = (c->st.meta_mask + 1) * sizeof(MetaSlot), ic = c->st.max_issuers * sizeof(uint64_t);
    CU(c, cudaMemcpy(c->st.table, p, t, cudaMemcpyHostToDevice)); p += t;
    CU(c, cudaMemcpy(c->st.pairs, p, pr, cudaMemcpyHostToDevice)); p += pr;
    CU(c, cudaMemcpy(c->st.meta, p, m, cudaMemcpyHostToDevice)); p += m;
    CU(c, cudaMemcpy(c->st.issuer_counts, p, ic, cudaMemcpyHostToDevice)); p += ic;
    CU(c, cudaMemcpy(c->st.status_counts, p, CTMR_ST__COUNT * sizeof(uint64_t), cudaMemcpyHostToDevice));
    // host memos: the DER memo is rebuilt lazily, the digest memos come back from the device registry
    c->digests.clear();
    c->issuer_by_digest.clear();
    c->issuer_by_der.clear();
    if (c->fe) return fe_clear_issuers(c);
    return CTMR_OK;
}

// the device registry (rank 0's region) again, digest i at index i: cleared, then filled by ONE launch of the
// find-or-insert kernel, which takes a call's digests in order
int snap_registry_restore(ctmr_ctx* c, const uint8_t* digests, uint64_t n) {
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaMemsetAsync(c->reg.slots, 0, (c->reg.mask + 1) * sizeof(IssuerRegSlot), c->stream));
    CU(c, cudaMemsetAsync(c->reg.by_index, 0, (size_t)c->reg.max_issuers * 32, c->stream));
    CU(c, cudaMemsetAsync(c->reg.counter, 0, sizeof(unsigned long long), c->stream));
    if (n) {
        uint8_t* d_dig = nullptr;
        uint32_t* d_idx = nullptr;
        CU(c, cudaMalloc(&d_dig, n * 32));
        CU(c, cudaMalloc(&d_idx, n * sizeof(uint32_t)));
        CU(c, cudaMemcpyAsync(d_dig, digests, n * 32, cudaMemcpyHostToDevice, c->stream));
        CU(c, launch_issuer_registry(c->reg, d_dig, nullptr, (uint32_t)n, d_idx, c->st.error_flag, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
        cudaFree(d_dig);
        cudaFree(d_idx);
    }
    int rc = refresh_digests(c);
    if (rc) return rc;
    if (c->digests.size() != n) return fail(c, CTMR_E_INVALID, "snapshot holds duplicate issuer digests");
    return ctmr_check_device(c, nullptr);
}

}  // namespace ctmr_host

namespace {
struct SnapHeader {
    char magic[8];  // "CTMRSNP3"
    uint64_t table_slots, pair_slots, meta_slots, max_issuers, n_issuers, next_index;
};
}  // namespace

extern "C" {

int ctmr_snapshot_size(ctmr_ctx* c, uint64_t* bytes) {
    if (!c || !bytes) return fail(c, CTMR_E_INVALID, "bad argument");
    if (c->st.peer.world > 1) return fail(c, CTMR_E_INVALID, "member of a group: use ctmr_group_snapshot_* (the shards share one issuer registry)");
    CU(c, cudaSetDevice(c->device));
    int rc = refresh_digests(c);
    if (rc) return rc;
    *bytes = sizeof(SnapHeader) + snap_shard_bytes(c) + c->digests.size() * 32;
    return CTMR_OK;
}

int ctmr_snapshot_save(ctmr_ctx* c, uint8_t* buf, uint64_t cap, uint64_t* written) {
    uint64_t need = 0;
    int rc = ctmr_snapshot_size(c, &need);
    if (rc) return rc;
    if (!buf || cap < need) return fail(c, CTMR_E_INVALID, "snapshot buffer too small");
    SnapHeader h{};
    std::memcpy(h.magic, "CTMRSNP3", 8);
    h.table_slots = c->st.table_mask + 1;
    h.pair_slots = c->st.pair_mask + 1;
    h.meta_slots = c->st.meta_mask + 1;
    h.max_issuers = c->st.max_issuers;
    h.n_issuers = c->digests.size();
    h.next_index = c->next_index;
    uint8_t* p = buf;
    std::memcpy(p, &h, sizeof h); p += sizeof h;
    rc = snap_shard_save(c, p);
    if (rc) return rc;
    p += snap_shard_bytes(c);
    for (const auto& d : c->digests) { std::memcpy(p, d.data(), 32); p += 32; }
    if (written) *written = (uint64_t)(p - buf);
    return CTMR_OK;
}

int ctmr_snapshot_load(ctmr_ctx* c, const uint8_t* buf, uint64_t bytes) {
    if (!c || !buf || bytes < sizeof(SnapHeader)) return fail(c, CTMR_E_INVALID, "bad snapshot");
    SnapHeader h;
    std::memcpy(&h, buf, sizeof h);
    if (std::memcmp(h.magic, "CTMRSNP3", 8) != 0) return fail(c, CTMR_E_INVALID, "not a ctmr snapshot");
    if (h.table_slots != c->st.table_mask + 1 || h.pair_slots != c->st.pair_mask + 1 || h.meta_slots != c->st.meta_mask + 1 ||
        h.max_issuers != c->st.max_issuers)
        return fail(c, CTMR_E_INVALID, "snapshot was taken with different capacities (table / pairs / max_issuers)");
    if (bytes < sizeof h + snap_shard_bytes(c) + h.n_issuers * 32 || h.n_issuers > h.max_issuers) return fail(c, CTMR_E_INVALID, "truncated snapshot");
    if (c->st.peer.world > 1) return fail(c, CTMR_E_INVALID, "member of a group: use ctmr_group_snapshot_*");
    int rc = snap_shard_load(c, buf + sizeof h);
    if (rc) return rc;
    c->next_index = h.next_index;
    return snap_registry_restore(c, buf + sizeof h + snap_shard_bytes(c), h.n_issuers);
}

// ------------------------------------------------------------------------------------------------ tooling
int ctmr_sha256_ceiling_device(ctmr_ctx* c, uint32_t iters, uint32_t rolled, uint32_t ctas_per_sm, float* ms_out,
                               uint64_t* blocks_out) {
    if (!c || !iters || !ctas_per_sm || ctas_per_sm > 8) return fail(c, CTMR_E_INVALID, "bad argument");
    CU(c, cudaSetDevice(c->device));
    cudaEvent_t e0, e1;
    CU(c, cudaEventCreate(&e0));
    CU(c, cudaEventCreate(&e1));
    uint32_t* sink = reinterpret_cast<uint32_t*>(c->small_dev + 90);
    CU(c, launch_sha_ceiling(iters / 8 + 1, (int)rolled, (int)ctas_per_sm, c->sm_count, sink, c->stream));  // warm-up
    CU(c, cudaEventRecord(e0, c->stream));
    CU(c, launch_sha_ceiling(iters, (int)rolled, (int)ctas_per_sm, c->sm_count, sink, c->stream));
    CU(c, cudaEventRecord(e1, c->stream));
    CU(c, cudaEventSynchronize(e1));
    float ms = 0.f;
    CU(c, cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (ms_out) *ms_out = ms;
    if (blocks_out) *blocks_out = (uint64_t)c->sm_count * ctas_per_sm * 256ull * iters;
    return CTMR_OK;
}

// ------------------------------------------------------------------------------------------------ read side
int ctmr_issuer_counts(ctmr_ctx* c, uint8_t* digests, uint64_t* counts, size_t* n) {
    if (!c || !n) return fail(c, CTMR_E_INVALID, "bad argument");
    CU(c, cudaSetDevice(c->device));
    {
        int rc0 = refresh_digests(c);  // issuers another rank of the group registered count too (with 0 here)
        if (rc0) return rc0;
    }
    const size_t have = c->digests.size(), cap = *n;
    const size_t take = have < cap ? have : cap;
    if (take) {
        if (counts) {
            CU(c, cudaMemcpyAsync(counts, c->st.issuer_counts, take * sizeof(uint64_t), cudaMemcpyDeviceToHost, c->stream));
            CU(c, cudaStreamSynchronize(c->stream));
        }
        if (digests)
            for (size_t i = 0; i < take; ++i) std::memcpy(digests + 32 * i, c->digests[i].data(), 32);
    }
    *n = take;
    return CTMR_OK;
}

int ctmr_set_cardinality(ctmr_ctx* c, int64_t exp_hour, const uint8_t digest[32], uint64_t* out) {
    if (!c || !digest || !out) return fail(c, CTMR_E_INVALID, "bad argument");
    CU(c, cudaSetDevice(c->device));
    *out = 0;
    uint32_t issuer = 0;
    bool found = false;
    int rc = lookup_digest(c, digest, false, &issuer, &found);
    if (rc) return rc;
    if (!found || exp_hour > INT32_MAX || exp_hour < INT32_MIN) return CTMR_OK;
    // one probe of the set's (issuer, hour) slot at its owner -- which may be another GPU of the group
    CU(c, launch_cardinality(c->st, (int32_t)exp_hour, issuer, c->small_dev + 80, c->stream));
    unsigned long long v = 0;
    CU(c, cudaMemcpyAsync(&v, c->small_dev + 80, sizeof v, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    *out = v;
    return CTMR_OK;
}

int ctmr_status_counters(ctmr_ctx* c, uint64_t out[CTMR_ST__COUNT]) {
    if (!c || !out) return fail(c, CTMR_E_INVALID, "bad argument");
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaMemcpyAsync(out, c->st.status_counts, CTMR_ST__COUNT * sizeof(uint64_t), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    return CTMR_OK;
}

int ctmr_table_stats(ctmr_ctx* c, uint64_t* used, uint64_t* capacity) {
    if (!c) return CTMR_E_INVALID;
    CU(c, cudaSetDevice(c->device));
    unsigned long long u = 0;
    CU(c, cudaMemsetAsync(c->small_dev + 81, 0, sizeof(unsigned long long), c->stream));
    CU(c, launch_table_count(c->st, c->small_dev + 81, c->stream));
    CU(c, cudaMemcpyAsync(&u, c->small_dev + 81, sizeof u, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    if (used) *used = u;
    if (capacity) *capacity = c->st.table_mask + 1;
    return CTMR_OK;
}

// Redis TTLs firing (SURVEY §8(f)-4): every set "serials::<expDate>::<issuer>" carries EXPIREAT(expDate)
// (storage/knowncertificates.go:44-47,98-104), so at `now` the sets with expDate <= now no longer exist.
int ctmr_evict_expired(ctmr_ctx* c, int64_t now_unix_sec, uint64_t* evicted_out) {
    if (!c) return CTMR_E_INVALID;
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaDeviceSynchronize());
    unsigned long long counters[2] = {0, 0};
    unsigned long long* dev = c->small_dev + 92;  // [92] live, [93] expired, [94] compaction cursor
    CU(c, cudaMemsetAsync(dev, 0, 3 * sizeof(unsigned long long), c->stream));
    CU(c, launch_evict_count(c->st, now_unix_sec, dev, c->stream));
    CU(c, cudaMemcpyAsync(counters, dev, sizeof counters, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    if (evicted_out) *evicted_out = counters[1];
    if (counters[1] == 0) return CTMR_OK;
    CU(c, launch_evict_pairs(c->st, now_unix_sec, c->stream));  // the expired sets' cardinalities are 0 again
    // open addressing with linear probing: taking slots out would cut probe chains, so the survivors are
    // compacted aside, the table is cleared and they are inserted again (first-seen indices preserved)
    KnownSlot* keep = nullptr;
    if (counters[0]) CU(c, cudaMalloc(&keep, counters[0] * sizeof(KnownSlot)));
    if (counters[0]) CU(c, launch_evict_compact(c->st, now_unix_sec, keep, dev + 2, c->stream));
    CU(c, cudaMemsetAsync(c->st.table, 0, (c->st.table_mask + 1) * sizeof(KnownSlot), c->stream));
    CU(c, launch_evict_reinsert(c->st, keep, counters[0], c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    cudaFree(keep);
    return ctmr_check_device(c, nullptr);
}

int ctmr_frontend_profile_last(ctmr_ctx* c, float* frontend_ms, float* path_ms, uint64_t* frontend_launches) {
    if (!c || !c->fe) return fail(c, CTMR_E_INVALID, "no ctmr_process_raw call to report");
    if (frontend_ms) *frontend_ms = c->fe->fe_ms;
    if (path_ms) *path_ms = c->fe->path_ms;
    if (frontend_launches) *frontend_launches = c->fe->launches;
    return CTMR_OK;
}

}  // extern "C"
