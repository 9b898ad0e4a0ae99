/*
 * ctmr.h -- C ABI of the B200-native CT-entry map/reduce hot path (libctmr.so).
 *
 * This is the drop-in boundary for ONE path of jcjones/ct-mapreduce (@739eda2): the per-entry
 * worker and its two reducers.  A Go host binds these entry points with cgo (INTEGRATION.md shows
 * the stub) and calls them in place of the loop body of
 *     (*LogSyncEngine).insertCTWorker        cmd/ct-fetch/ct-fetch.go:191-245
 *     certIsFilteredOut                      cmd/ct-fetch/ct-fetch.go:44-70
 *     (*FilesystemDatabase).Store            storage/filesystemdatabase.go:158-211
 *     (*KnownCertificates).WasUnknown/Count  storage/knowncertificates.go:38-63
 *     (*IssuerMetadata).Accumulate (the seenExpDateBefore bit)  storage/issuermetadata.go:92-108
 *     NewIssuer/Issuer.ID, NewSerial, NewExpDateFromTime        storage/types.go:109-130,171-178,339-346
 * while storage.StorageBackend, storage.RemoteCache and storage.CertDatabase
 * (storage/types.go:46-102) stay byte-identical on the Go side.
 *
 * Conventions (SURVEY.md §8(b)):
 *   - plain pointers and sizes only; no C++ or torch types; no exceptions cross the ABI.
 *   - functions return 0 (CTMR_OK) or a negative CTMR_E_* batch-level error; the text is
 *     available from ctmr_last_error(ctx) until the next call on that ctx.
 *   - per-entry problems are never return codes: they are status[i] (CTMR_ST_*), exactly like the
 *     reference's log-and-continue (ct-fetch.go:206-209,223-225,230-232).
 *   - the caller owns every input and output buffer; the library never keeps a caller pointer
 *     past return (cgo rule).  Device state lives in an opaque ctmr_ctx.
 *   - one ctmr_ctx per GPU, calls on a ctx are serialised by the caller; batches are ordered:
 *     every entry of call k precedes every entry of call k+1 for first-seen semantics.
 *   - several GPUs: ctmr_group_* (one process drives the GPUs of the box: what the Go host calls) or
 *     ctmr_peer_* (one process per GPU, tables attached through CUDA IPC).  Either way every set
 *     "serials::<expDate>::<issuer>" has one owner GPU, the map kernels insert straight into the owner's
 *     table over NVLink, and WasUnknown / counts are globally exact -- the fan-out is invisible above the ABI.
 *   - there is no CPU fallback: without a CUDA device ctmr_create fails with CTMR_E_NO_DEVICE.
 */
#ifndef CTMR_H
#define CTMR_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CTMR_ABI_VERSION 3

/* ---- batch-level return codes ------------------------------------------------------------ */
enum {
    CTMR_OK = 0,
    CTMR_E_INVALID = -1,          /* bad argument */
    CTMR_E_CUDA = -2,             /* CUDA runtime error (text in ctmr_last_error) */
    CTMR_E_NOMEM = -3,            /* host or device allocation failed */
    CTMR_E_TABLE_FULL = -4,       /* known-certificate table exhausted (cf. Redis OOM, rediscache.go:61-63) */
    CTMR_E_TOO_MANY_ISSUERS = -5, /* more distinct issuers than config.max_issuers */
    CTMR_E_NO_DEVICE = -6,        /* no usable CUDA device: the product path has no CPU fallback */
    CTMR_E_BATCH_TOO_LARGE = -7,  /* exceeds config.max_batch_* */
    CTMR_E_PAIR_TABLE_FULL = -8,  /* (issuer, expDate) table exhausted: raise config.pair_capacity_log2 */
    CTMR_E_META_TABLE_FULL = -9,  /* IssuerMetadata string-identity table exhausted: raise config.meta_capacity_log2 */
    CTMR_E_PEER_TIMEOUT = -10,    /* a rank of the group did not reach a barrier (a peer failed or the calls diverged) */
    CTMR_E_PEER = -11             /* peer access / CUDA IPC between the GPUs of a group is not available */
};

/* ---- per-entry status -------------------------------------------------------------------- */
enum {
    CTMR_ST_OK = 0,               /* reached Store (counted by insertCTWorker.Inserted, ct-fetch.go:235) */
    CTMR_ST_PARSE_ERR = 1,        /* "Problem decoding certificate", ct-fetch.go:206-209 */
    CTMR_ST_FILTER_CA = 2,        /* certIsFilteredOut.CA, ct-fetch.go:47-50 */
    CTMR_ST_FILTER_EXPIRED = 3,   /* certIsFilteredOut.expired, ct-fetch.go:52-55 */
    CTMR_ST_FILTER_CN = 4,        /* certIsFilteredOut.cn-filtered, ct-fetch.go:57-68 */
    CTMR_ST_NO_ISSUER = 5,        /* len(Chain) < 1, ct-fetch.go:215-219 */
    CTMR_ST_ISSUER_PARSE_ERR = 6, /* "Problem decoding issuing certificate", ct-fetch.go:221-225 */
    CTMR_ST_SERIAL_TOO_LONG = 7,  /* serial INTEGER longer than CTMR_MAX_SERIAL octets (documented limit) */
    CTMR_ST__COUNT = 8
};

#define CTMR_MAX_SERIAL 39u            /* octets of raw serial a key record holds (RFC 5280 allows 20) */
#define CTMR_ISSUER_NONE 0xFFFFFFFFu   /* issuer_idx value for "entry has no chain" */
#define CTMR_ISSUER_BAD 0xFFFFFFFEu    /* dense index of an issuer certificate that failed to parse */

/* config.flags */
#define CTMR_F_NO_FINGERPRINT 1u /* skip SHA-256(leaf DER); the reference itself never computes it (SURVEY §0 M3) */

typedef struct ctmr_ctx ctmr_ctx;

typedef struct ctmr_config {
    uint32_t struct_size;        /* sizeof(ctmr_config), for ABI evolution */
    int32_t device;              /* CUDA device ordinal */
    uint64_t table_capacity;     /* known-certificate slots (64 B each), rounded up to a power of two */
    uint64_t max_batch_entries;  /* ceiling for one ctmr_process_batch call (sizes device staging); 0 = 1<<20 */
    uint64_t max_batch_bytes;    /* ceiling for the leaf blob of one call; 0 = 2 KiB * max_batch_entries */
    uint32_t max_issuers;        /* distinct issuers over the ctx lifetime; 0 = 65536 */
    uint32_t pair_capacity_log2; /* (issuer, exp-hour) first-seen table, log2 slots; 0 = 24 */
    const uint8_t* issuer_cn_filter; /* raw config value issuerCNFilter (config/config.go:193): split on ',' */
    uint32_t issuer_cn_filter_len;   /*   without trimming, HasPrefix on raw CN bytes (ct-fetch.go:57-63)      */
    uint32_t log_expired_entries;    /* config logExpiredEntries (config/config.go:188) */
    uint32_t flags;                  /* CTMR_F_* */
    uint32_t meta_capacity_log2;     /* IssuerMetadata string-identity table (issuer DN / CRL-DP bytes), log2 slots; 0 = 20, max 26 */
    uint64_t max_round_entries;      /* groups only: the most entries one GPU maps per round of ctmr_process_device
                                      * (= ceil(4n / (4R - 3)), R = ctmr_peer_rounds()); sizes the key-exchange regions (78 bytes x
                                      * GPUs x 3 per entry).  0 = the host pipeline's stage size (max_batch_entries) */
} ctmr_config;

/* Caller-allocated per-entry outputs, each [n]; any pointer may be NULL to skip that copy-back. */
typedef struct ctmr_out {
    uint8_t* status;            /* CTMR_ST_* */
    uint8_t* sha256;            /* [n][32] SHA-256 of the leaf DER (crypto/sha256.Sum256(cert.Raw)) */
    int64_t* exp_hour;          /* floor(NotAfter/3600 s): NewExpDateFromTime, storage/types.go:339-346 */
    uint32_t* serial_off;       /* raw serial content octets (NewSerial, storage/types.go:171-178):   */
    uint32_t* serial_len;       /*   offset inside the entry's DER, and length                          */
    uint8_t* was_unknown;       /* KnownCertificates.WasUnknown result, storage/knowncertificates.go:38-55 */
    uint8_t* first_issuer_hour; /* 1 iff Accumulate would return seenExpDateBefore == false (issuermetadata.go:95-108) */
    /* IssuerMetadata's string reducers (SURVEY.md §8(f)-1): spans of the two strings Accumulate looks at, and
     * first-seen bits so that the host only formats / parses them for candidates, not for every new certificate */
    uint32_t* issuer_name_off;  /* issuer Name (full TLV) inside the entry's DER: source of Issuer.String() (issuermetadata.go:94) */
    uint32_t* issuer_name_len;
    uint32_t* crldp_off;        /* cRLDistributionPoints extnValue content (issuermetadata.go:111), len 0 = absent */
    uint32_t* crldp_len;
    uint8_t* first_issuer_dn;   /* 1 iff was_unknown and no earlier new certificate of this issuer had the same Name bytes */
    uint8_t* first_crldp;       /* 1 iff was_unknown, extension present, and its bytes are new for this issuer */
    /* PEM of the NEW certificates, encoded on the device (SURVEY.md §8(f)-3): what Store hands to
     * StorageBackend.StoreCertificatePEM (storage/filesystemdatabase.go:171-175,197-198), i.e.
     * pem.EncodeToMemory(&pem.Block{Type: "CERTIFICATE", Bytes: cert.Raw}).  Optional as a group. */
    uint8_t* pem;               /* [pem_cap] texts of the entries with was_unknown == 1, back to back in entry order */
    uint64_t pem_cap;           /* too small => CTMR_E_BATCH_TOO_LARGE */
    uint64_t* pem_off;          /* [n+1]: entry i's text = pem[pem_off[i] .. pem_off[i+1]), empty unless new */
} ctmr_out;

/* ---- lifecycle ---------------------------------------------------------------------------- */
uint32_t ctmr_abi_version(void);
int ctmr_create(const ctmr_config* cfg, ctmr_ctx** out);      /* replaces GetConfiguredStorage wiring, engine/engine.go:19-48 */
void ctmr_destroy(ctmr_ctx* ctx);
const char* ctmr_last_error(ctmr_ctx* ctx);                   /* ctx may be NULL: error of the last failed ctmr_create */

/* Pinned host memory for batch packing (the Go batcher packs entries straight into it). */
void* ctmr_host_alloc(size_t bytes);
void ctmr_host_free(void* p);

/* ---- issuers ------------------------------------------------------------------------------ */
/* Parses n issuer certificates (x509.ParseCertificate(Chain[0]), ct-fetch.go:221), computes
 * Issuer.ID() digests (SHA-256 of RawSubjectPublicKeyInfo, storage/types.go:124-130,155-159) on the
 * GPU and assigns ctx-lifetime dense indices in order of first appearance.  HOST buffers.
 * dense_idx_out[k] = dense index, or CTMR_ISSUER_BAD when certificate k does not parse. */
int ctmr_register_issuers(ctmr_ctx* ctx, const uint8_t* issuer_blob, const uint64_t* issuer_offsets /* [n+1] */,
                          uint32_t n, uint32_t* dense_idx_out);
/* digest (32 octets) of a dense index; base64url of it is Issuer.ID() */
int ctmr_issuer_digest(ctmr_ctx* ctx, uint32_t dense_idx, uint8_t digest_out[32]);
uint32_t ctmr_issuer_count(ctmr_ctx* ctx);

/* ---- the hot path, HOST buffers (what the Go shim calls) ----------------------------------- */
/* One call = one batch drained from entryChan (ct-fetch.go:132,191).  blob holds the n leaf DERs
 * back to back (entry i = blob[offsets[i] .. offsets[i+1])); issuer_* hold the batch's distinct
 * Chain[0] certificates and issuer_idx[i] selects one (CTMR_ISSUER_NONE = no chain).
 * now_unix_ns replaces time.Now() at ct-fetch.go:52.  Copies host->device, runs the kernels,
 * copies the requested outputs back; synchronous.
 * After a failure (rc != 0) the outputs are undefined and part of the batch may already be in the tables; the
 * call's entry indices are consumed either way, so replaying the batch is safe in the reference's own sense
 * (idempotent replays, SURVEY §5): entries that were inserted read as known, never as unknown twice. */
int ctmr_process_batch(ctmr_ctx* ctx, const uint8_t* blob, const uint64_t* offsets /* [n+1] */, uint64_t n,
                       const uint8_t* issuer_blob, const uint64_t* issuer_offsets /* [n_issuers+1] */,
                       uint32_t n_issuers, const uint32_t* issuer_idx /* [n] */, int64_t now_unix_ns,
                       ctmr_out* out);

/* ---- reducers' read side ------------------------------------------------------------------- */
/* Per-issuer unique-certificate counts = sum over expDates of KnownCertificates.Count()
 * (cmd/storage-statistics/storage-statistics.go:44-53).  *n in: capacity, out: issuers written. */
int ctmr_issuer_counts(ctmr_ctx* ctx, uint8_t* digests /* [cap][32] */, uint64_t* counts /* [cap] */, size_t* n);
/* SetCardinality("serials::<expDate>::<issuer>"), storage/knowncertificates.go:57-63 */
int ctmr_set_cardinality(ctmr_ctx* ctx, int64_t exp_hour, const uint8_t issuer_digest[32], uint64_t* count_out);
/* entries per status since create, indexed by CTMR_ST_* (the certIsFilteredOut.* / Inserted counters) */
int ctmr_status_counters(ctmr_ctx* ctx, uint64_t out[CTMR_ST__COUNT]);
int ctmr_table_stats(ctmr_ctx* ctx, uint64_t* slots_used, uint64_t* capacity);

/* ---- warm start / checkpoint (SURVEY.md §8(f)-4) -------------------------------------------- */
/* Seed the known-certificate table from pre-existing state, e.g. the members of the Redis set
 * "serials::<expDate>::<issuer>" read back with KnownCertificates.Known() (storage/knowncertificates.go:65-96):
 * `n` serials, serial i = serial_blob[serial_offsets[i] .. serial_offsets[i+1]).  Preloaded keys count as
 * seen before every batch: WasUnknown answers false for them, per-issuer counts include them, and the
 * (issuer, expDate) pair counts as already allocated.  HOST buffers. */
int ctmr_preload_known(ctmr_ctx* ctx, int64_t exp_hour, const uint8_t issuer_digest[32], const uint8_t* serial_blob,
                       const uint64_t* serial_offsets /* [n+1] */, uint64_t n);
/* Redis TTLs: WasUnknown puts EXPIREAT(expDate) on every "serials::<expDate>::<issuer>" set
 * (storage/knowncertificates.go:44-47,98-104; expDate = hour-truncated NotAfter, storage/types.go:371-373), so
 * as time passes whole sets vanish from the reference's state.  This call applies that to the device state:
 * every set with expDate <= now is dropped (its serials are unknown again, it stops counting towards
 * ctmr_issuer_counts / ctmr_set_cardinality, its slots are reclaimed).  IssuerMetadata's seenExpDateBefore memo
 * is process memory in the reference and is kept.  Call it between batches, e.g. once per hour. */
int ctmr_evict_expired(ctmr_ctx* ctx, int64_t now_unix_sec, uint64_t* evicted_out);
/* Snapshot of the derived device state (tables, histograms, issuer registry, next entry index) into a
 * caller buffer, and its restoration into a ctx created with the same capacities.  ctmr_snapshot_size
 * gives the bytes needed.  The reference's analogue is the state it keeps in Redis between runs
 * (storage/rediscache.go); its own resume logic is cmd/ct-fetch/ct-fetch.go:288-300. */
int ctmr_snapshot_size(ctmr_ctx* ctx, uint64_t* bytes);
int ctmr_snapshot_save(ctmr_ctx* ctx, uint8_t* buf, uint64_t cap, uint64_t* written);
int ctmr_snapshot_load(ctmr_ctx* ctx, const uint8_t* buf, uint64_t bytes);

/* ---- the sets read back: list, members, canonical export / import ---------------------------- */
/* What the reference reads out of Redis: KnownCertificates.Known() (storage/knowncertificates.go:65-96),
 * GetIssuerAndDatesFromCache (storage/filesystemdatabase.go:59-100, a KEYS serials::* scan) and the walk of
 * cmd/storage-statistics.  Semantics:
 *   - a LIVE set is an (issuer, expDate) whose cardinality is > 0.  Sets emptied by ctmr_evict_expired keep their
 *     first-seen memo on the device but no longer exist in Redis, so they are not listed.
 *   - a MEMBER is a serial in the known-certificate table together with its first-seen global entry index.  Serials
 *     longer than CTMR_MAX_SERIAL never entered the table (CTMR_ST_SERIAL_TOO_LONG), so they never appear.
 *   - CANONICAL ORDER: sets by (issuer digest bytes, exp_hour) ascending, members of a set by first index ascending.
 *     The order depends on the logical state only: a single ctx, a group of any size and the merge of the shards of a
 *     peer group export byte-identical results for the same entries (entry i of a batch keeps global index
 *     next_index + i in every shape).
 *   - an export carries the Redis state (sets, members, cardinalities) and next_index.  It does NOT carry process
 *     memory: the IssuerMetadata string memos (first_issuer_dn / first_crldp) and the first-seen memo of evicted sets.
 *     An imported state therefore behaves like a restarted reference process against the same Redis.
 * Buffers are HOST memory.  A call whose output pointers are NULL only reports the sizes (one (issuer, hour) table
 * scan, plus one counting pass over the known-certificate table for the serial bytes of an export); buffers too small
 * for the result give CTMR_E_BATCH_TOO_LARGE with the sizes reported all the same.
 * On a member of a group (ctmr_group_member, or one rank of a ctmr_peer_* group) list, members and export cover the
 * sets THAT shard owns; they are not collective, and merging the shards' exports in canonical order gives the group's. */
typedef struct ctmr_set_info {
    uint8_t issuer_digest[32];
    int64_t exp_hour;
    uint64_t count;       /* SetCardinality */
    uint64_t member_off;  /* index of the set's first member in the member arrays (= running sum of the counts) */
} ctmr_set_info;

typedef struct ctmr_set_export {
    uint64_t next_index;    /* out on export, in on import: the ctx's (group's) next global entry index (what the host-buffer
                             * calls and preloads have used; callers of the device entry points choose the indices themselves) */
    uint64_t n_sets, n_members, serial_bytes;  /* out on export (also for too-small / NULL buffers), in on import */
    ctmr_set_info* sets;    /* [sets_cap] */
    uint64_t sets_cap;
    uint8_t* serials;       /* [serials_cap]: member k = serials[serial_off[k] .. serial_off[k+1]) */
    uint64_t serials_cap;
    uint64_t* serial_off;   /* [members_cap + 1] */
    uint64_t* first_index;  /* [members_cap] */
    uint64_t members_cap;
} ctmr_set_export;

/* GetIssuerAndDatesFromCache + Count(): the live sets with min_exp_hour <= exp_hour <= max_exp_hour (ListExpirationDates'
 * notBefore is the lower bound), canonical order.  *n = number of sets. */
int ctmr_list_sets(ctmr_ctx* ctx, int64_t min_exp_hour, int64_t max_exp_hour, ctmr_set_info* out, uint64_t cap, uint64_t* n);
/* KnownCertificates.Known() of one set, members by first index; *n = number of members, serial_off [cap + 1].
 * serials_cap >= CTMR_MAX_SERIAL * n always suffices. */
int ctmr_set_members(ctmr_ctx* ctx, int64_t exp_hour, const uint8_t issuer_digest[32], uint8_t* serials, uint64_t serials_cap,
                     uint64_t* serial_off, uint64_t* first_index, uint64_t cap, uint64_t* n);
int ctmr_export_sets(ctmr_ctx* ctx, ctmr_set_export* x);
/* Into an EMPTY ctx only (next_index == 0, no key in the table; else CTMR_E_INVALID), of any capacity: every member keeps
 * its exported first index, next_index becomes the exported one, cardinalities and per-issuer counts follow from the
 * keys, unknown issuer digests are registered (dense indices may differ from the source's; the canonical form does not
 * show them).  Serials empty or longer than CTMR_MAX_SERIAL are CTMR_E_INVALID.  A rank of a ctmr_peer_* group loads
 * the sets it owns only, so every rank can be handed the same full export; a member of an in-process group refuses:
 * use ctmr_group_import_sets. */
int ctmr_import_sets(ctmr_ctx* ctx, const ctmr_set_export* x);

/* ---- device-resident entry points ---------------------------------------------------------- */
/* Same path with every buffer already in HBM on ctx's device (benchmarks, multi-GPU orchestration,
 * hosts that receive entries by GPUDirect).  `stream` is a cudaStream_t passed as void*; NULL =
 * the ctx's own stream.  Asynchronous: the caller synchronises the stream. */

/* 64-byte key record: what WasUnknown is keyed on (SURVEY §0 M4): expDate hour, issuer, raw serial. */
typedef struct ctmr_key {
    uint64_t index;      /* global entry index: lowest index of equal keys wins "was unknown" */
    int32_t exp_hour;
    uint32_t issuer;     /* dense issuer index */
    uint8_t serial_len;
    uint8_t serial[CTMR_MAX_SERIAL]; /* zero padded */
    uint32_t valid;      /* 1 when the entry reached Store (status OK) */
    uint32_t pad;
} ctmr_key;

typedef struct ctmr_dev_batch {
    const uint8_t* blob;        /* device; readable up to blob_bytes rounded up to 16 */
    uint64_t blob_bytes;
    const uint64_t* offsets;    /* device [n+1] */
    uint64_t n;
    const uint32_t* issuer_idx; /* device [n]; NULL = every entry has no chain */
    const uint32_t* issuer_map; /* device [*]: batch-local -> dense index, or NULL when issuer_idx is dense */
    uint32_t issuer_map_len;
    uint32_t reserved;
    uint64_t first_index;       /* global index of entry 0 */
    int64_t now_unix_ns;
    const uint32_t* lens;       /* device [n] or NULL.  When set, entry i = blob[offsets[i] .. offsets[i]+lens[i]):
                                 * records need not be contiguous and offsets needs only n elements (this is how
                                 * the wire-format front end, ctmr_frontend.h, hands over leaves it decoded in place) */
} ctmr_dev_batch;

typedef struct ctmr_dev_out { /* device pointers, each [n]; NULL = not produced */
    uint8_t* status;
    uint8_t* sha256;
    int64_t* exp_hour;
    uint32_t* serial_off;
    uint32_t* serial_len;
    uint8_t* was_unknown;
    uint8_t* first_issuer_hour;
    ctmr_key* keys; /* [n] key records (valid=0 for entries that did not reach Store) */
    uint32_t* issuer_name_off; /* as in ctmr_out; first_* are produced by ctmr_process_device only */
    uint32_t* issuer_name_len;
    uint32_t* crldp_off;
    uint32_t* crldp_len;
    uint8_t* first_issuer_dn;
    uint8_t* first_crldp;
} ctmr_dev_out;

/* map half: DER walk + filter + SHA-256 -> status, exp_hour, serial span, fingerprint, key records */
int ctmr_map_device(ctmr_ctx* ctx, const ctmr_dev_batch* batch, const ctmr_dev_out* out, void* stream);
/* reduce half over m key records in any order WITHIN the call: insert, resolve lowest-index-wins, per-issuer
 * counts.  Across calls the ordering contract of the path holds: every index of a later call must be higher than
 * every index of an earlier call (a lower index arriving later would find itself "first" a second time). */
int ctmr_reduce_device(ctmr_ctx* ctx, const ctmr_key* keys, uint64_t m, uint8_t* was_unknown /* [m] */,
                       uint8_t* first_issuer_hour /* [m] */, void* stream);
/* map + reduce on one GPU */
int ctmr_process_device(ctmr_ctx* ctx, const ctmr_dev_batch* batch, const ctmr_dev_out* out, void* stream);

/* CUDA-event timings of the last ctmr_process_device call, valid once its stream has been synchronised:
 * map_ms = summed duration of the K_map stage (measured on the stream it ran on), total_ms = whole call */
int ctmr_profile_last(ctmr_ctx* ctx, float* map_ms, float* total_ms);

/* copy the per-issuer histogram (uint64 [n_slots], dense index order) and the status counters
 * (uint64 [CTMR_ST__COUNT]) of THIS GPU into device buffers (a group merges them with ctmr_peer_allreduce_histogram_device) */
int ctmr_read_histogram_device(ctmr_ctx* ctx, uint64_t* counts_dst, uint32_t n_slots, uint64_t* status_dst,
                               void* stream);
/* forget everything: known-certificate table, first-seen pairs, per-issuer and status counters
 * (the issuer registry is kept).  The analogue of FLUSHDB on the reference's Redis. */
int ctmr_reset_device(ctmr_ctx* ctx, void* stream);
/* fails with CTMR_E_TABLE_FULL / CTMR_E_CUDA if any asynchronous launch since the last check failed */
int ctmr_check_device(ctmr_ctx* ctx, void* stream);

/* ---- several GPUs, ONE process (what a Go host uses: SURVEY.md §8(b) "fan-out inside the library") ------------ */
/* The worker pool of StartDatabaseThreads (cmd/ct-fetch/ct-fetch.go:140-145) becomes one call per drained batch:
 * the group cuts the batch into rounds of n_devices slices by entry index (entry i keeps global index
 * next_index + i, so the result equals the sequential numThreads=1 run over the batch in its given order), every
 * GPU maps its slice and hands each key to the set's owner GPU over NVLink, events separate the appends from the
 * owners' insert/resolve and that from the pull of the result bits, and the outputs land in the caller's arrays in
 * entry order.  cfg->device is ignored;
 * `devices` may name a device more than once (several shards on one GPU: how the path is tested on a 1-GPU box). */
typedef struct ctmr_group ctmr_group;
int ctmr_group_create(const ctmr_config* cfg, const int32_t* devices, uint32_t n_devices, ctmr_group** out);
void ctmr_group_destroy(ctmr_group* g);
const char* ctmr_group_last_error(ctmr_group* g);
uint32_t ctmr_group_size(ctmr_group* g);
ctmr_ctx* ctmr_group_member(ctmr_group* g, uint32_t rank); /* read-side access to one shard; owned by the group */
/* same arguments and outputs as ctmr_process_batch; globally exact across the GPUs of the group */
int ctmr_group_process_batch(ctmr_group* g, const uint8_t* blob, const uint64_t* offsets, uint64_t n, const uint8_t* issuer_blob,
                             const uint64_t* issuer_offsets, uint32_t n_issuers, const uint32_t* issuer_idx, int64_t now_unix_ns,
                             ctmr_out* out);
int ctmr_group_issuer_counts(ctmr_group* g, uint8_t* digests, uint64_t* counts, size_t* n);   /* summed over the shards */
int ctmr_group_set_cardinality(ctmr_group* g, int64_t exp_hour, const uint8_t issuer_digest[32], uint64_t* count_out);
int ctmr_group_status_counters(ctmr_group* g, uint64_t out[CTMR_ST__COUNT]);
int ctmr_group_table_stats(ctmr_group* g, uint64_t* slots_used, uint64_t* capacity);
int ctmr_group_preload_known(ctmr_group* g, int64_t exp_hour, const uint8_t issuer_digest[32], const uint8_t* serial_blob,
                             const uint64_t* serial_offsets, uint64_t n);
int ctmr_group_evict_expired(ctmr_group* g, int64_t now_unix_sec, uint64_t* evicted_out);
int ctmr_group_reset(ctmr_group* g);
/* snapshot of the whole group (every shard + the one issuer registry); restores into a group of the same size and
 * capacities (a set's owner depends on the group size) */
int ctmr_group_snapshot_size(ctmr_group* g, uint64_t* bytes);
int ctmr_group_snapshot_save(ctmr_group* g, uint8_t* buf, uint64_t cap, uint64_t* written);
int ctmr_group_snapshot_load(ctmr_group* g, const uint8_t* buf, uint64_t bytes);
/* the sets of the whole group (every member scans its own shard on a thread of its own, the host merges the sorted
 * lists); same outputs as the single-ctx calls, byte-identical to a single ctx over the same entries.  Import routes
 * every set to its owner in THIS group, so an export moves between groups of any size and single ctxs. */
int ctmr_group_list_sets(ctmr_group* g, int64_t min_exp_hour, int64_t max_exp_hour, ctmr_set_info* out, uint64_t cap, uint64_t* n);
int ctmr_group_set_members(ctmr_group* g, int64_t exp_hour, const uint8_t issuer_digest[32], uint8_t* serials, uint64_t serials_cap,
                           uint64_t* serial_off, uint64_t* first_index, uint64_t cap, uint64_t* n);
int ctmr_group_export_sets(ctmr_group* g, ctmr_set_export* x);
int ctmr_group_import_sets(ctmr_group* g, const ctmr_set_export* x);

/* ---- several GPUs, one PROCESS PER GPU (torchrun-style launches; SURVEY.md §8(e)) ------------------------------ */
/* Every rank creates its ctx with the same capacities, exports a handle, gathers all handles by whatever means the
 * launcher offers (torch.distributed all_gather in this repository) and attaches them.  From then on
 * ctmr_process_device, ctmr_process_batch, ctmr_reset_device and ctmr_peer_* are COLLECTIVE: every rank must make
 * the same sequence of calls.  Inside them the ranks meet at barriers kept in peer memory (no host round trip, no
 * NCCL on the data path); the global index of entry j of rank r's round k is first_index + (k * world + r) * E + j,
 * i.e. the result equals the sequential run over the rounds in rank order.  E = entries per rank and round: the host
 * pipeline's stage size for ctmr_process_batch; for ctmr_process_device (every rank passes the same n, R =
 * ctmr_peer_rounds() >= 4) E = ceil(4n / (4R - 3)), i.e. R - 1 full rounds and a last one a quarter as long. */
#define CTMR_PEER_HANDLE_BYTES 256u
/* allocates this rank's key-exchange area for a group of `world` ranks and exports it together with the tables */
int ctmr_peer_export(ctmr_ctx* ctx, uint32_t world, uint8_t handle_out[CTMR_PEER_HANDLE_BYTES]);
int ctmr_peer_attach(ctmr_ctx* ctx, uint32_t rank, uint32_t world, const uint8_t* handles /* [world][CTMR_PEER_HANDLE_BYTES] */);
/* barrier over the group on `stream` (device side; returns immediately) */
int ctmr_peer_barrier_device(ctmr_ctx* ctx, void* stream);
/* all-reduce(sum) of [per-issuer unique counts || status counters] over peer memory, bracketed by barriers: the
 * merge of the per-GPU histograms at the end of a chunk.  Device buffers, uint64 [n_slots] and [CTMR_ST__COUNT]. */
int ctmr_peer_allreduce_histogram_device(ctmr_ctx* ctx, uint64_t* counts_dst, uint32_t n_slots, uint64_t* status_dst, void* stream);
/* the collective ctmr_process_device always runs ctmr_peer_rounds() rounds (CTMR_PEER_ROUNDS unless the environment
 * variable of the same name overrides it for experiments; identical on every rank) */
#define CTMR_PEER_ROUNDS 8u
uint32_t ctmr_peer_rounds(void);
/* E of a collective ctmr_process_device call over n entries per rank: what config.max_round_entries must cover and what
 * the global-index formula above uses (R - 1 rounds of E entries and a short last one) */
uint64_t ctmr_peer_round_entries(uint64_t n);

/* ---- host placement -------------------------------------------------------------------------------- */
/* Binds the calling thread to the CPUs of the NUMA node `device` hangs off (sysfs), so that pinned buffers it
 * allocates and first touches afterwards are node-local: with 8 GPUs reading host memory at PCIe rate, remote-node
 * buffers halve the end-to-end rate.  Returns the node, or -1 when the topology cannot be read (no change made). */
int ctmr_bind_host_to_device(int32_t device);

/* ---- measurement tooling -------------------------------------------------------------------- */
/* Register-only SHA-256 microbenchmark: every lane chains `iters` compressions (K_map's own function, no
 * memory traffic) at `ctas_per_sm` x 256 threads per SM.  The measured INT-pipe ceiling of the fingerprint. */
int ctmr_sha256_ceiling_device(ctmr_ctx* ctx, uint32_t iters, uint32_t rolled, uint32_t ctas_per_sm, float* ms_out,
                               uint64_t* blocks_out);

/* ---- synthetic corpus on the device (bench/test tooling; ctmr_synth.h) ---------------------- */
struct ctmr_synth_cfg;
/* pass 1: offsets[0..n] (device) of entries [first, first+n); returns total bytes via *total_bytes */
int ctmr_synth_offsets_device(const struct ctmr_synth_cfg* cfg, uint64_t first, uint64_t n, uint64_t* offsets,
                              uint64_t* total_bytes, void* stream);
/* pass 2: write the DER bytes and (optionally) the issuer index of each entry */
int ctmr_synth_write_device(const struct ctmr_synth_cfg* cfg, uint64_t first, uint64_t n, const uint64_t* offsets,
                            uint8_t* blob, uint32_t* issuer_idx, void* stream);
/* generator-side truth for size-independent checks: cert id, notAfter, basicConstraints mode */
int ctmr_synth_truth_device(const struct ctmr_synth_cfg* cfg, uint64_t first, uint64_t n, uint64_t* cert_id,
                            int64_t* not_after, uint8_t* bc_mode, void* stream);

/* host-side: DER of the n_issuers synthetic CA certificates; returns total bytes, fills
 * offsets[0..n_issuers]; writes bytes when blob != NULL and cap suffices */
uint64_t ctmr_synth_issuers_host(const struct ctmr_synth_cfg* cfg, uint64_t* offsets, uint8_t* blob, uint64_t cap);

/* host-side: RFC 6962 get-entries response bodies (JSON, base64 leaf_input / extra_data; every third entry a
 * precert_entry, chains of one or two certificates) for entries [first, first+n) in pages of `page` entries -- input
 * for ctmr_process_raw (ctmr_frontend.h).  Returns the bytes needed; writes the text and the string spans when
 * text != NULL and cap suffices. */
uint64_t ctmr_synth_raw_pages_host(const struct ctmr_synth_cfg* cfg, uint64_t first, uint64_t n, uint32_t page, uint8_t* text,
                                   uint64_t cap, uint64_t* leaf_off, uint32_t* leaf_len, uint64_t* extra_off, uint32_t* extra_len);

#ifdef __cplusplus
}
#endif
#endif /* CTMR_H */
