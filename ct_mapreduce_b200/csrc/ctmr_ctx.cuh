// ctmr_ctx.cuh -- internal: the context behind the opaque ctmr_ctx of include/ctmr.h, shared by the translation
// units that implement the C ABI (ctmr_api.cu: lifecycle, issuers, device entry points, read side, front end;
// ctmr_pipeline.cu: the host-buffer batch pipeline on one GPU, on a group of GPUs, and across processes).
#pragma once
#include <algorithm>
#include <array>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "ctmr_device.cuh"
#include "ctmr_kernels.cuh"

using namespace ctmr;

namespace ctmr_host {

constexpr int kStages = 3;                      // host-API pipeline depth
constexpr int kMaxRounds = 16;                  // rounds of one ctmr_process_device call
constexpr uint64_t kStageEntries = 1ull << 18;  // entries per pipeline stage
constexpr uint64_t kStageBytes = 768ull << 20;  // leaf bytes per pipeline stage

extern thread_local std::string g_create_error;

inline int env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return v && *v ? atoi(v) : dflt;
}

// device side of the PEM output (ctmr_out.pem): one per host-pipeline stage and one for the front end
struct PemStage {
    uint64_t cap_entries = 0, cap_bytes = 0;
    uint64_t *sizes = nullptr, *off = nullptr;
    uint8_t* text = nullptr;
    void* scan_temp = nullptr;
    size_t scan_temp_bytes = 0;
    std::vector<uint64_t> host_off;
};

struct Stage {
    cudaStream_t stream = nullptr;
    cudaEvent_t mapped = nullptr;   // recorded after this stage's K_map (its inserts have reached the owners' tables)
    cudaEvent_t reduced = nullptr;  // recorded after this stage's owner passes (resolve + pairs of own entries and inbox records)
    cudaEvent_t meta_done = nullptr;  // recorded after this stage's string-identity insert
    uint8_t* blob = nullptr;
    uint64_t* offsets = nullptr;
    uint32_t* issuer_idx = nullptr;
    uint8_t* status = nullptr;
    uint8_t* sha = nullptr;
    int64_t* exp_hour = nullptr;
    uint32_t* serial_off = nullptr;
    uint32_t* serial_len = nullptr;
    uint8_t* was_unknown = nullptr;
    uint8_t* first = nullptr;
    ctmr_key* keys = nullptr;
    uint32_t* slot_of = nullptr;
    uint32_t* pair_slot = nullptr;
    uint32_t* order = nullptr;
    unsigned int* len_hist = nullptr;
    uint32_t* spans = nullptr;       // [4][E]: issuer name off/len, crldp off/len
    uint32_t* meta_slots = nullptr;  // [2*E]
    uint8_t* first_meta = nullptr;   // [2][E]: first_issuer_dn, first_crldp
    PemStage pem;                    // allocated when a caller first asks for PEM output
};

// one upload stage of the front end: a chunk's characters and string spans, device side and pinned host staging
struct FeStage {
    uint8_t* text = nullptr;  // [16 + cap_text + 64]
    uint64_t *leaf_off = nullptr, *extra_off = nullptr, *h_leaf_off = nullptr, *h_extra_off = nullptr;
    uint32_t *leaf_len = nullptr, *extra_len = nullptr, *h_leaf_len = nullptr, *h_extra_len = nullptr;
    cudaEvent_t uploaded = nullptr, consumed = nullptr;
    std::vector<uint8_t> pack;  // host staging of the slow path (strings scattered over more than one chunk of text)
};

// CT wire-format front end (include/ctmr_frontend.h): device buffers of one chunk + the device mirror of
// the issuer registry keyed by certificate bytes
struct FrontEnd {
    uint64_t cap_entries = 0, cap_text = 0, cap_decoded = 0;
    FeStage stage[2];          // upload double buffer
    cudaStream_t copy_stream = nullptr;
    uint64_t *pad_size = nullptr, *dec_off = nullptr;
    uint32_t* dec_len = nullptr;
    uint8_t *str_bad = nullptr, *decoded = nullptr;
    void* scan_temp = nullptr;
    size_t scan_temp_bytes = 0;
    uint8_t *entry_status = nullptr, *entry_type = nullptr, *leaf_src = nullptr;
    uint64_t *timestamp = nullptr, *leaf_abs = nullptr, *chain_abs = nullptr, *tbs_abs = nullptr;
    uint32_t *leaf_rel = nullptr, *leaf_len_out = nullptr, *chain_len = nullptr, *tbs_len = nullptr, *issuer_idx = nullptr;
    // outputs of the path for this chunk
    uint8_t *status = nullptr, *sha = nullptr, *was_unknown = nullptr, *first = nullptr, *first_meta = nullptr;
    int64_t* exp_hour = nullptr;
    uint32_t *serial_off = nullptr, *serial_len = nullptr, *spans = nullptr;
    // issuer certificates by bytes
    IssuerCertSlot* slots_dev = nullptr;
    std::vector<IssuerCertSlot> slots_host;
    uint64_t slot_mask = 0, slots_used = 0;
    uint8_t* arena = nullptr;
    uint64_t arena_cap = 0, arena_used = 0;
    uint64_t* pending = nullptr;
    uint64_t pending_mask = 0;
    uint32_t* unknown_list = nullptr;
    uint32_t unknown_cap = 0;
    unsigned int* unknown_count = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr;
    float fe_ms = 0.f, path_ms = 0.f;
    uint64_t launches = 0;
    PemStage pem;
};

}  // namespace ctmr_host
using namespace ctmr_host;

// offsets inside a rank's SHARED region: the part of its state the other ranks of a group address directly
// (one allocation, so that one CUDA IPC handle exports it).  Identical on every rank: same capacities.
struct SharedLayout {
    size_t flags = 0;          // [kPeerChannels + 1][kMaxWorld] u64: barrier epochs per channel, then the mailbox row
    size_t reg_counter = 0;    // u64 (rank 0's is THE registry)
    size_t status_counts = 0;  // [CTMR_ST__COUNT] u64
    size_t issuer_counts = 0;  // [max_issuers] u64
    size_t reg_digests = 0;    // [max_issuers][32]
    size_t reg_slots = 0;      // [reg_mask + 1] IssuerRegSlot
    size_t meta = 0, pairs = 0, table = 0, total = 0;
    uint64_t reg_mask = 0;
};

enum PeerMode { PEER_NONE = 0, PEER_GROUP = 1 /* one process, ctmr_group */, PEER_IPC = 2 /* one process per GPU */ };

// barrier channels (each is used from ONE stream per rank, so its epochs are stream ordered on every rank)
enum : uint32_t {
    CH_STAGE_MAP = 0,      // + stage index (3): after K_map of a host-pipeline round
    CH_STAGE_RESOLVE = 3,  // + stage index (3): after resolve of a host-pipeline round
    CH_DEV_MAP = 6, CH_DEV_RESOLVE = 7,  // ctmr_process_device
    CH_USER = 8, CH_HIST_A = 9, CH_HIST_B = 10, CH_RESET_A = 11, CH_RESET_B = 12, CH_MAILBOX = 13,
    CH_STAGE_META = 16                   // + stage index (3): after the string-identity insert of a host-pipeline round
};

struct ctmr_ctx {
    int device = 0;
    int sm_count = 148;
    uint32_t flags = 0;
    cudaStream_t stream = nullptr;
    DeviceState st{};
    FilterCfg filter{};
    uint64_t next_index = 0;
    uint64_t stage_entries = 0, stage_bytes = 0;
    bool stages_ready = false;
    Stage stages[kStages];
    // shared region + the views of every rank's region (a single GPU is a group of one)
    uint8_t* shared = nullptr;
    SharedLayout lay{};
    PeerFlags pf{};
    IssuerRegistry reg{};                  // lives in rank 0's region
    int peer_mode = PEER_NONE;
    void* ipc_base[kMaxWorld] = {};        // mappings opened with cudaIpcOpenMemHandle (closed on destroy)
    void* ipc_xchg[kMaxWorld] = {};
    // key exchange of a group: peer-visible area (inboxes, result bits, region sizes) + private bookkeeping
    uint8_t* xchg = nullptr;
    uint64_t X = 0, cfg_round_entries = 0;
    uint32_t exported_world = 0;            // ctmr_peer_export was called for a group of this size (the views follow at attach)
    PeerExchange px{};
    unsigned long long* cursors = nullptr;  // [kParities][kMaxWorld] records appended per owner (local)
    uint32_t* rev = nullptr;                // [kParities][world][X] inbox position -> entry
    uint32_t *in_slot = nullptr, *in_pair = nullptr;  // [kParities][world][X] owner-side scratch of the inbox records
    cudaEvent_t ev_g[3] = {};               // ctmr_group_process_raw: mapped / reduced / string identities inserted
    cudaEvent_t ev_pulled[kParities] = {};  // ctmr_process_device: round k's bits pulled (its exchange parity may be reused)
    unsigned long long epoch[kPeerChannels] = {};
    struct ctmr_group* group = nullptr;    // set when the ctx is a member of an in-process group
    // issuer memo on the host (the registry itself is on the device): DER -> index, digest -> index, index -> digest
    std::unordered_map<std::string, uint32_t> issuer_by_der;
    std::unordered_map<std::string, uint32_t> issuer_by_digest;
    std::vector<std::array<uint8_t, 32>> digests;
    uint32_t* issuer_map_dev = nullptr;
    uint32_t issuer_map_cap = 0;
    // scratch of the device-resident entry points
    ctmr_key* keys_scratch = nullptr;
    uint32_t* slot_scratch = nullptr;
    uint32_t* pair_scratch = nullptr;
    uint8_t* bits_scratch = nullptr;
    uint32_t* meta_scratch = nullptr;  // [2*cap]
    uint64_t scratch_cap = 0;
    uint32_t* order_scratch = nullptr;  // length-bucketed order of the device entry points
    uint64_t order_cap = 0;
    unsigned int* len_hist = nullptr;
    bool bucket_by_length = true;
    bool fuse_insert = true;
    // ctmr_process_device pipelines map (stream A) against reduce (stream B) over kSub sub-batches
    cudaStream_t stream_a = nullptr, stream_a2 = nullptr, stream_b = nullptr;  // K_map alternates between a and a2
    cudaEvent_t ev_fork = nullptr, ev_join_a = nullptr, ev_join_a2 = nullptr, ev_join_b = nullptr;
    cudaEvent_t ev_map0[kMaxRounds] = {}, ev_map1[kMaxRounds] = {}, ev_red1[kMaxRounds] = {}, ev_tok[kMaxRounds] = {};
    int last_sub = 0, last_map_streams = 1;
    unsigned int* len_hist_sub[kMaxRounds] = {};
    unsigned long long* small_dev = nullptr;  // [128] private counters / cursors / results (error flag at +73)
    FrontEnd* fe = nullptr;
    std::string err;
};

struct ctmr_group {
    std::vector<ctmr_ctx*> m;
    uint64_t next_index = 0;
    std::string err;
};

// ---- helpers shared by the ABI translation units --------------------------------------------------------------
namespace ctmr_host {

int fail(ctmr_ctx* ctx, int code, const std::string& msg);

#define CU(ctx, call)                                                                                   \
    do {                                                                                                \
        cudaError_t e_ = (call);                                                                        \
        if (e_ != cudaSuccess) {                                                                        \
            return fail((ctx), e_ == cudaErrorMemoryAllocation ? CTMR_E_NOMEM : CTMR_E_CUDA,             \
                        std::string(#call) + ": " + cudaGetErrorString(e_));                            \
        }                                                                                               \
    } while (0)

uint64_t pow2_at_least(uint64_t v);
void fill_map_params(ctmr_ctx* c, const ctmr_dev_batch* b, const ctmr_dev_out* o, MapParams& p, int counter_slot = 3,
                     uint32_t* fused_slot_of = nullptr, int parity = 0);
// key exchange: allocation for a group of `world` ranks, views of every rank's area
size_t exchange_bytes(uint32_t world, uint64_t X);
int alloc_exchange(ctmr_ctx* c, uint32_t world);
void attach_exchange(ctmr_ctx* c, uint8_t* const* bases, uint32_t world, uint32_t rank);
// one round of the exchange on stream s (no-ops on a single GPU)
int round_begin(ctmr_ctx* c, int parity, cudaStream_t s);                       // before K_map: cursors of this parity to 0
int round_publish(ctmr_ctx* c, int parity, cudaStream_t s);                     // after K_map: region sizes to the owners
int round_owner_insert(ctmr_ctx* c, int parity, uint64_t max_per_region, cudaStream_t s);   // owner: inbox records into the table
int round_owner_resolve(ctmr_ctx* c, int parity, uint64_t max_per_region, cudaStream_t s);  // ... their was_unknown, counts, pair slots
int round_owner_pairs(ctmr_ctx* c, int parity, uint64_t max_per_region, cudaStream_t s);    // ... their first_issuer_hour
int round_pull(ctmr_ctx* c, int parity, uint64_t max_per_region, uint8_t* was_unknown, uint8_t* first, cudaStream_t s);
// views of the shared regions `bases[0..world)` (this rank's own among them) -> st.peer, pf, reg
void attach_views(ctmr_ctx* c, uint8_t* const* bases, uint32_t world, uint32_t rank);
int peer_barrier(ctmr_ctx* c, uint32_t channel, cudaStream_t s);   // PEER_IPC only; no-op otherwise
int refresh_digests(ctmr_ctx* c);                                   // host memo <- device registry
int lookup_digest(ctmr_ctx* c, const uint8_t digest[32], bool insert, uint32_t* idx_out, bool* found);
int upload_issuer_map(ctmr_ctx* c, const uint32_t* dense, uint32_t n);
int preload_impl(ctmr_ctx* c, int64_t exp_hour, const uint8_t digest[32], const uint8_t* serial_blob, const uint64_t* serial_offsets,
                 uint64_t n, uint64_t first_index);
int ensure_stages(ctmr_ctx* c);
// snapshot pieces (ctmr_api.cu): one shard's tables + histograms, and the registry of the group (rank 0's region)
uint64_t snap_shard_bytes(ctmr_ctx* c);
int snap_shard_save(ctmr_ctx* c, uint8_t* p);
int snap_shard_load(ctmr_ctx* c, const uint8_t* p);
int snap_registry_restore(ctmr_ctx* c, const uint8_t* digests, uint64_t n);
int frontend_ensure(ctmr_ctx* c);   // allocates the front end's buffers on first use (ctmr_api.cu)
int ensure_scratch(ctmr_ctx* c, uint64_t n);
uint64_t device_round_entries(uint64_t n, uint32_t rounds);   // E of a ctmr_process_device call cut into `rounds` rounds
uint32_t peer_rounds();   // rounds of the collective ctmr_process_device (CTMR_PEER_ROUNDS, env override for experiments)
void pem_free(PemStage& ps);
void stages_destroy(ctmr_ctx* c);
int pem_ensure(ctmr_ctx* c, PemStage& ps, uint64_t entries, uint64_t der_bytes);
int pem_chunk(ctmr_ctx* c, PemStage& ps, const uint8_t* blob, const uint64_t* offsets, const uint32_t* lens, const uint8_t* select,
              uint64_t cnt, const ctmr_out* out, uint64_t first, uint64_t* base, cudaStream_t s);
// host-built key records through the reduce path of c (insert, resolve, pairs), synchronous; every key must be one c owns
int reduce_keys_host(ctmr_ctx* c, const ctmr_key* keys, uint64_t n);

// a member's error becomes the group's
inline int group_fail(ctmr_group* g, ctmr_ctx* c, int rc) {
    if (g && c) g->err = c->err;
    return rc;
}

// fn(r) for every member, on one thread each (the members' calls wait on the host: issuer round trips, D2H); sequential if
// threads cannot be had.  No exception leaves this function (C ABI).
template <class F>
void for_each_member(uint32_t W, std::vector<int>& rcs, F fn) {
    rcs.assign(W, CTMR_OK);
    std::vector<std::thread> th;
    uint32_t started = 0;
    try {
        for (; started < W; ++started) th.emplace_back([&rcs, &fn, r = started] { rcs[r] = fn(r); });
    } catch (...) {
    }
    for (std::thread& t : th) t.join();
    for (uint32_t r = started; r < W; ++r) rcs[r] = fn(r);
}

}  // namespace ctmr_host
