// ctmr_sets.cu -- the sets read back out of the device (include/ctmr.h "the sets read back"): the live sets of a shard,
// one set's members, the canonical export of a shard / ctx / group, and its import into an empty ctx or group of any shape.
//
// Export of one shard, on the ctx's stream:
//   1. (issuer, hour) table scan: live slots (count > 0, hour in range) compacted with a warp ballot and one atomic per
//      warp (a counting pass first sizes the compact arrays).
//   2. canonical set order: key = rank of the issuer digest << 32 | biased hour (the host uploads the ranks, O(issuers)),
//      radix sort, exclusive scan of the counts -> each set's first member.  A compact hash map pair key -> set ordinal,
//      sized to the live sets, serves the per-slot lookups of step 3: the pair table is 512 MB at the default 2^24 slots
//      and does not stay in L2, the compact map usually does.
//   3. known-table scan: every thread reads the FIRST 32-byte sector of a slot (inv_first, tag, hour, issuer, serial
//      length, first 7 serial octets); a ready slot of a selected set claims a position in its set with one atomic on the
//      set's cursor and only then reads the second sector; a fixed-width staging record (first index, length, 39 octets)
//      lands at the position.  Every cursor must end at exactly its set's count (cardinality and table agree).
//   4. segmented sort of each set's members by first index, scan of the serial lengths, packing of the serials; one
//      D2H copy per output array.
// Import needs no kernel of its own: host-built key records go through the reduce path (reduce_keys_host), per owner.
#include <cub/cub.cuh>

#include <climits>
#include <numeric>

#include "ctmr_ctx.cuh"

namespace ctmr {

struct SetFilter {
    int64_t lo, hi;               // exp_hour range, inclusive
    unsigned long long only_key;  // one set's pair key, 0 = every set in range
};

struct SetMapSlot {               // compact map of the selected sets: pair key -> ordinal in canonical order
    unsigned long long key;       // 0 = empty
    unsigned long long ord;
};

__device__ __forceinline__ bool set_selected(unsigned long long pk, const SetFilter& f) {
    const int64_t hour = (int32_t)(uint32_t)(pk - 1ull);
    return hour >= f.lo && hour <= f.hi && (f.only_key == 0ull || f.only_key == pk);
}

// step 1.  counters[0] += selected live sets, counters[1] += the sum of their counts; key_out == nullptr: count only
__global__ void __launch_bounds__(256) set_scan_kernel(const PairSlot* __restrict__ pairs, uint64_t pair_mask, SetFilter f,
                                                       const uint32_t* __restrict__ issuer_rank, uint32_t n_rank,
                                                       unsigned long long* __restrict__ key_out, uint32_t* __restrict__ slot_out,
                                                       unsigned long long* counters) {
    const uint32_t lane = threadIdx.x & 31u;
    // warp-uniform trip count: every lane takes part in the ballot
    for (uint64_t base = (uint64_t)blockIdx.x * blockDim.x; base <= pair_mask; base += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t i = base + threadIdx.x;
        bool live = false;
        unsigned long long pk = 0, cnt = 0;
        if (i <= pair_mask) {
            pk = pairs[i].key;
            cnt = pairs[i].count;
            live = pk != 0ull && cnt != 0ull && set_selected(pk, f);
        }
        const uint32_t ballot = __ballot_sync(0xffffffffu, live);
        if (!ballot) continue;
        unsigned long long sum = live ? cnt : 0ull;
        for (int o = 16; o; o >>= 1) sum += __shfl_down_sync(0xffffffffu, sum, o);
        unsigned long long at = 0;
        if (lane == 0) {
            at = atomicAdd(counters, (unsigned long long)__popc(ballot));
            atomicAdd(counters + 1, sum);
        }
        at = __shfl_sync(0xffffffffu, at, 0);
        if (live && key_out) {
            const uint64_t j = at + __popc(ballot & ((1u << lane) - 1u));
            const uint32_t issuer = (uint32_t)((pk - 1ull) >> 32), hour = (uint32_t)(pk - 1ull);
            const uint32_t rank = issuer < n_rank ? issuer_rank[issuer] : 0xFFFFFFFFu;
            key_out[j] = ((unsigned long long)rank << 32) | (hour ^ 0x80000000u);  // biased hour: signed order as unsigned
            slot_out[j] = (uint32_t)i;
        }
    }
}

// step 2, after the sort: counts in canonical order (count[n] = 0 closes the scan) and the compact map
__global__ void __launch_bounds__(256) set_prepare_kernel(const PairSlot* __restrict__ pairs, const uint32_t* __restrict__ sorted_slot,
                                                          uint64_t n, SetMapSlot* map, uint64_t map_mask,
                                                          unsigned long long* __restrict__ count) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j == n) count[n] = 0ull;
    if (j >= n) return;
    const PairSlot& p = pairs[sorted_slot[j]];
    const unsigned long long pk = p.key;
    count[j] = p.count;
    uint64_t pos = mix64(pk) & map_mask;
    while (atomicCAS(&map[pos].key, 0ull, pk) != 0ull) pos = (pos + 1) & map_mask;  // pair keys are distinct
    map[pos].ord = j;
}

__device__ __forceinline__ bool map_find(const SetMapSlot* __restrict__ map, uint64_t mask, unsigned long long pk, uint64_t& ord) {
    uint64_t pos = mix64(pk) & mask;
    for (;;) {  // load factor <= 1/2: an empty slot ends every probe
        const unsigned long long k = map[pos].key;
        if (k == pk) {
            ord = map[pos].ord;
            return true;
        }
        if (k == 0ull) return false;
        pos = (pos + 1) & mask;
    }
}

// serial bytes of the ready slots of selected sets (the sizing pass of an export): first sectors only
__global__ void __launch_bounds__(256) member_bytes_kernel(const KnownSlot* __restrict__ table, uint64_t table_mask, SetFilter f,
                                                           unsigned long long* bytes) {
    unsigned long long local = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= table_mask; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint4* s = reinterpret_cast<const uint4*>(table + i);
        const uint4 a = __ldg(s), b = __ldg(s + 1);
        if ((a.z & 3u) != 2u) continue;
        if (set_selected((((unsigned long long)b.y << 32) | b.x) + 1ull, f)) local += b.z & 0xFFu;
    }
    for (int o = 16; o; o >>= 1) local += __shfl_down_sync(0xffffffffu, local, o);
    if ((threadIdx.x & 31u) == 0 && local) atomicAdd(bytes, local);
}

// step 3.  staging record (48 bytes = 3 x uint4): first index (8), serial length (1), serial (39)
__global__ void __launch_bounds__(256) member_scan_kernel(const KnownSlot* __restrict__ table, uint64_t table_mask, SetFilter f,
                                                          const SetMapSlot* __restrict__ map, uint64_t map_mask,
                                                          const unsigned long long* __restrict__ member_off,
                                                          const unsigned long long* __restrict__ count, unsigned long long* cursor,
                                                          unsigned long long* __restrict__ first_out, uint32_t* __restrict__ pos_out,
                                                          uint4* __restrict__ staging, unsigned long long* mismatch) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= table_mask; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint4* s = reinterpret_cast<const uint4*>(table + i);
        const uint4 a = __ldg(s), b = __ldg(s + 1);  // first sector: inv_first, tag | hour, issuer, length + 7 octets
        if ((a.z & 3u) != 2u) continue;
        const unsigned long long pk = (((unsigned long long)b.y << 32) | b.x) + 1ull;
        if (!set_selected(pk, f)) continue;
        uint64_t ord = 0;
        if (!map_find(map, map_mask, pk, ord)) {  // a key whose set has no live (issuer, hour) slot
            atomicAdd(mismatch, 1ull);
            continue;
        }
        const unsigned long long k = atomicAdd(cursor + ord, 1ull);
        if (k >= count[ord]) {  // more keys than the set's cardinality
            atomicAdd(mismatch, 1ull);
            continue;
        }
        const uint64_t dst = member_off[ord] + k;
        const uint4 c = __ldg(s + 2), d = __ldg(s + 3);  // second sector: the rest of the serial
        const unsigned long long first = ~(((unsigned long long)a.y << 32) | a.x);
        first_out[dst] = first;
        pos_out[dst] = (uint32_t)dst;
        uint4* r = staging + 3 * dst;
        r[0] = make_uint4((uint32_t)first, (uint32_t)(first >> 32), b.z, b.w);
        r[1] = c;
        r[2] = d;
    }
}

// integrity: every set's cursor ends at its count
__global__ void __launch_bounds__(256) set_check_kernel(const unsigned long long* __restrict__ cursor, const unsigned long long* __restrict__ count,
                                                        uint64_t n, unsigned long long* mismatch) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n && cursor[j] != count[j]) atomicAdd(mismatch, 1ull);
}

// step 4: lengths in sorted order (len[n] = 0 closes the scan), then the packing
__global__ void __launch_bounds__(256) member_len_kernel(const uint32_t* __restrict__ pos_sorted, const uint4* __restrict__ staging, uint64_t n,
                                                         unsigned long long* __restrict__ len) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k == n) len[n] = 0ull;
    if (k >= n) return;
    const uint32_t l = staging[3ull * pos_sorted[k]].z & 0xFFu;
    len[k] = l < CTMR_MAX_SERIAL ? l : CTMR_MAX_SERIAL;
}

__global__ void __launch_bounds__(256) member_pack_kernel(const uint32_t* __restrict__ pos_sorted, const uint4* __restrict__ staging, uint64_t n,
                                                          const unsigned long long* __restrict__ soff, uint8_t* __restrict__ blob) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const uint4* r = staging + 3ull * pos_sorted[k];
    const uint4 q0 = r[0], q1 = r[1], q2 = r[2];
    const uint32_t w[12] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w, q2.x, q2.y, q2.z, q2.w};
    const uint8_t* bytes = reinterpret_cast<const uint8_t*>(w);
    const uint64_t o = soff[k], l = soff[k + 1] - o;
    for (uint64_t b = 0; b < l; ++b) blob[o + b] = bytes[9 + b];
}

}  // namespace ctmr

namespace {

inline unsigned grid_over(const ctmr_ctx* c, uint64_t items) {
    const uint64_t want = (items + 255) / 256;
    const uint64_t cap = (uint64_t)c->sm_count * 8;
    return (unsigned)std::max<uint64_t>(1, std::min(want, cap));
}
inline unsigned blocks_of(uint64_t items) { return (unsigned)std::max<uint64_t>(1, (items + 255) / 256); }

// device memory of one call, released on every path (stream ordered)
struct DevMem {
    cudaStream_t s;
    std::vector<void*> ptrs;
    explicit DevMem(cudaStream_t st) : s(st) {}
    ~DevMem() {
        for (void* p : ptrs) cudaFreeAsync(p, s);
    }
    template <class T>
    cudaError_t alloc(T** p, uint64_t count) {
        void* q = nullptr;
        const cudaError_t e = cudaMallocAsync(&q, std::max<uint64_t>(count, 1) * sizeof(T), s);
        if (e == cudaSuccess) ptrs.push_back(q);
        *p = static_cast<T*>(q);
        return e;
    }
};

// one shard's selected sets in canonical order, host side
struct ShardSets {
    std::vector<ctmr_set_info> sets;  // member_off relative to this shard's member arrays
    uint64_t n_members = 0, serial_bytes = 0;
    std::vector<uint64_t> first, soff;  // members, when no caller destination was given
    std::vector<uint8_t> blob;
};

// caller buffers the members go to directly (a single ctx / shard)
struct MemberDest {
    uint8_t* serials;
    uint64_t serials_cap;
    uint64_t* serial_off;
    uint64_t* first_index;
    uint64_t cap;
    uint64_t sets_cap;
};

constexpr SetFilter kAllSets{INT64_MIN, INT64_MAX, 0ull};

unsigned long long pair_key(uint32_t issuer, int32_t hour) { return ((((unsigned long long)issuer) << 32) | (uint32_t)hour) + 1ull; }

// rank of every dense issuer index in digest order (what the canonical order sorts by), and its inverse
int issuer_ranks(ctmr_ctx* c, std::vector<uint32_t>& rank, std::vector<uint32_t>& by_rank) {
    const int rc = refresh_digests(c);
    if (rc) return rc;
    const uint32_t n = (uint32_t)c->digests.size();
    by_rank.resize(n);
    std::iota(by_rank.begin(), by_rank.end(), 0u);
    std::sort(by_rank.begin(), by_rank.end(),
              [&](uint32_t a, uint32_t b) { return std::memcmp(c->digests[a].data(), c->digests[b].data(), 32) < 0; });
    rank.assign(n, 0);
    for (uint32_t k = 0; k < n; ++k) rank[by_rank[k]] = k;
    return CTMR_OK;
}

// sizes only: one (issuer, hour) table scan [+ one first-sector pass over the known table for the serial bytes]
int shard_count(ctmr_ctx* c, const SetFilter& f, bool want_bytes, uint64_t* n_sets, uint64_t* n_members, uint64_t* serial_bytes) {
    CU(c, cudaSetDevice(c->device));
    DevMem mem(c->stream);
    unsigned long long* cnt = nullptr;
    CU(c, mem.alloc(&cnt, 3));
    CU(c, cudaMemsetAsync(cnt, 0, 3 * sizeof(unsigned long long), c->stream));
    set_scan_kernel<<<grid_over(c, c->st.pair_mask + 1), 256, 0, c->stream>>>(c->st.pairs, c->st.pair_mask, f, nullptr, 0, nullptr, nullptr, cnt);
    CU(c, cudaGetLastError());
    if (want_bytes) {
        member_bytes_kernel<<<grid_over(c, c->st.table_mask + 1), 256, 0, c->stream>>>(c->st.table, c->st.table_mask, f, cnt + 2);
        CU(c, cudaGetLastError());
    }
    unsigned long long h[3] = {0, 0, 0};
    CU(c, cudaMemcpyAsync(h, cnt, sizeof h, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    if (n_sets) *n_sets = h[0];
    if (n_members) *n_members = h[1];
    if (serial_bytes) *serial_bytes = h[2];
    return CTMR_OK;
}

bool dest_fits(const MemberDest* d, const ShardSets& o) {
    return d->sets_cap >= o.sets.size() && d->cap >= o.n_members && d->serials_cap >= o.serial_bytes;
}

// Steps 1-4 over this ctx's own shard.  want_members = false: the sets only.  dest != nullptr: the members go straight to
// the caller's buffers (CTMR_E_BATCH_TOO_LARGE when they do not fit; the sizes are in `o` either way).
int shard_scan(ctmr_ctx* c, const SetFilter& f, bool want_members, ShardSets& o, const MemberDest* dest) {
    CU(c, cudaSetDevice(c->device));
    std::vector<uint32_t> rank, by_rank;
    int rc = issuer_ranks(c, rank, by_rank);
    if (rc) return rc;
    cudaStream_t s = c->stream;
    DevMem mem(s);
    unsigned long long* cnt = nullptr;
    CU(c, mem.alloc(&cnt, 5));  // [0,1] counting pass, [2,3] compaction, [4] integrity mismatches
    CU(c, cudaMemsetAsync(cnt, 0, 5 * sizeof(unsigned long long), s));
    const unsigned pair_grid = grid_over(c, c->st.pair_mask + 1);
    set_scan_kernel<<<pair_grid, 256, 0, s>>>(c->st.pairs, c->st.pair_mask, f, nullptr, 0, nullptr, nullptr, cnt);
    CU(c, cudaGetLastError());
    unsigned long long h[2] = {0, 0};
    CU(c, cudaMemcpyAsync(h, cnt, sizeof h, cudaMemcpyDeviceToHost, s));
    CU(c, cudaStreamSynchronize(s));
    const uint64_t n_sets = h[0];
    o.sets.clear();
    o.n_members = h[1];
    o.serial_bytes = 0;
    if (n_sets == 0) {
        o.n_members = 0;
        if (dest && dest->serial_off) dest->serial_off[0] = 0;
        if (!dest) o.soff.assign(1, 0);
        return CTMR_OK;
    }
    if (want_members && o.n_members > (uint64_t)INT_MAX) return fail(c, CTMR_E_INVALID, "more than 2^31 members in one shard");

    // step 1: compaction
    uint32_t* d_rank = nullptr;
    unsigned long long *key_a = nullptr, *key_b = nullptr;
    uint32_t *slot_a = nullptr, *slot_b = nullptr;
    CU(c, mem.alloc(&d_rank, rank.size()));
    CU(c, mem.alloc(&key_a, n_sets));
    CU(c, mem.alloc(&key_b, n_sets));
    CU(c, mem.alloc(&slot_a, n_sets));
    CU(c, mem.alloc(&slot_b, n_sets));
    if (!rank.empty()) CU(c, cudaMemcpyAsync(d_rank, rank.data(), rank.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
    set_scan_kernel<<<pair_grid, 256, 0, s>>>(c->st.pairs, c->st.pair_mask, f, d_rank, (uint32_t)rank.size(), key_a, slot_a, cnt + 2);
    CU(c, cudaGetLastError());

    // step 2: canonical set order, first members, compact map
    size_t tmp_bytes = 0, t = 0;
    CU(c, cub::DeviceRadixSort::SortPairs(nullptr, t, key_a, key_b, slot_a, slot_b, (int)n_sets, 0, 64, s));
    tmp_bytes = std::max(tmp_bytes, t);
    CU(c, cub::DeviceScan::ExclusiveSum(nullptr, t, (unsigned long long*)nullptr, (unsigned long long*)nullptr, (int64_t)o.n_members + 1, s));
    tmp_bytes = std::max(tmp_bytes, t);
    CU(c, cub::DeviceScan::ExclusiveSum(nullptr, t, (unsigned long long*)nullptr, (unsigned long long*)nullptr, (int64_t)n_sets + 1, s));
    tmp_bytes = std::max(tmp_bytes, t);
    if (want_members) {
        CU(c, cub::DeviceSegmentedSort::SortPairs(nullptr, t, (unsigned long long*)nullptr, (unsigned long long*)nullptr, (uint32_t*)nullptr,
                                                  (uint32_t*)nullptr, (int)o.n_members, (int)n_sets, (unsigned long long*)nullptr,
                                                  (unsigned long long*)nullptr, s));
        tmp_bytes = std::max(tmp_bytes, t);
    }
    uint8_t* tmp = nullptr;
    CU(c, mem.alloc(&tmp, tmp_bytes));
    const unsigned long long* key_sorted = key_a;
    const uint32_t* slot_sorted = slot_a;
    if (n_sets > 1) {  // one set (ctmr_set_members) needs no sort
        t = tmp_bytes;
        CU(c, cub::DeviceRadixSort::SortPairs(tmp, t, key_a, key_b, slot_a, slot_b, (int)n_sets, 0, 64, s));
        key_sorted = key_b;
        slot_sorted = slot_b;
    }
    const uint64_t map_slots = pow2_at_least(std::max<uint64_t>(64, 2 * n_sets));
    SetMapSlot* map = nullptr;
    unsigned long long *count = nullptr, *member_off = nullptr;
    CU(c, mem.alloc(&map, map_slots));
    CU(c, mem.alloc(&count, n_sets + 1));
    CU(c, mem.alloc(&member_off, n_sets + 1));
    CU(c, cudaMemsetAsync(map, 0, map_slots * sizeof(SetMapSlot), s));
    set_prepare_kernel<<<blocks_of(n_sets + 1), 256, 0, s>>>(c->st.pairs, slot_sorted, n_sets, map, map_slots - 1, count);
    CU(c, cudaGetLastError());
    t = tmp_bytes;
    CU(c, cub::DeviceScan::ExclusiveSum(tmp, t, count, member_off, (int64_t)n_sets + 1, s));
    std::vector<unsigned long long> hkey(n_sets), hcount(n_sets);
    CU(c, cudaMemcpyAsync(hkey.data(), key_sorted, n_sets * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    CU(c, cudaMemcpyAsync(hcount.data(), count, n_sets * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    CU(c, cudaStreamSynchronize(s));
    o.sets.resize(n_sets);
    uint64_t run = 0;
    for (uint64_t j = 0; j < n_sets; ++j) {
        const uint32_t r = (uint32_t)(hkey[j] >> 32);
        if (r >= by_rank.size()) return fail(c, CTMR_E_INVALID, "a set's issuer is not in the registry yet");
        ctmr_set_info& si = o.sets[j];
        std::memcpy(si.issuer_digest, c->digests[by_rank[r]].data(), 32);
        si.exp_hour = (int32_t)((uint32_t)hkey[j] ^ 0x80000000u);
        si.count = hcount[j];
        si.member_off = run;
        run += hcount[j];
    }
    if (!want_members) return CTMR_OK;

    // step 3: known-table scan into the staging records
    const uint64_t n = o.n_members;
    unsigned long long *cursor = nullptr, *first_a = nullptr, *first_b = nullptr, *len = nullptr, *soff = nullptr;
    uint32_t *pos_a = nullptr, *pos_b = nullptr;
    uint4* staging = nullptr;
    CU(c, mem.alloc(&cursor, n_sets));
    CU(c, mem.alloc(&first_a, n));
    CU(c, mem.alloc(&first_b, n));
    CU(c, mem.alloc(&pos_a, n));
    CU(c, mem.alloc(&pos_b, n));
    CU(c, mem.alloc(&staging, 3 * n));
    CU(c, cudaMemsetAsync(cursor, 0, n_sets * sizeof(unsigned long long), s));
    member_scan_kernel<<<grid_over(c, c->st.table_mask + 1), 256, 0, s>>>(c->st.table, c->st.table_mask, f, map, map_slots - 1, member_off,
                                                                          count, cursor, first_a, pos_a, staging, cnt + 4);
    CU(c, cudaGetLastError());
    set_check_kernel<<<blocks_of(n_sets), 256, 0, s>>>(cursor, count, n_sets, cnt + 4);
    CU(c, cudaGetLastError());
    // a mismatch leaves staging positions unwritten: stop before step 4 reads them
    unsigned long long mismatches = 0;
    CU(c, cudaMemcpyAsync(&mismatches, cnt + 4, sizeof mismatches, cudaMemcpyDeviceToHost, s));
    CU(c, cudaStreamSynchronize(s));
    if (mismatches) return fail(c, CTMR_E_CUDA, "set export: the known-certificate table and the sets' cardinalities disagree (" +
                                                  std::to_string(mismatches) + " keys)");

    // step 4: members by first index within each set, then the packing
    t = tmp_bytes;
    CU(c, cub::DeviceSegmentedSort::SortPairs(tmp, t, first_a, first_b, pos_a, pos_b, (int)n, (int)n_sets, member_off, member_off + 1, s));
    CU(c, mem.alloc(&len, n + 1));
    CU(c, mem.alloc(&soff, n + 1));
    member_len_kernel<<<blocks_of(n + 1), 256, 0, s>>>(pos_b, staging, n, len);
    CU(c, cudaGetLastError());
    t = tmp_bytes;
    CU(c, cub::DeviceScan::ExclusiveSum(tmp, t, len, soff, (int64_t)n + 1, s));
    unsigned long long tail[1] = {0};  // serial bytes
    CU(c, cudaMemcpyAsync(tail, soff + n, sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    CU(c, cudaStreamSynchronize(s));
    o.serial_bytes = tail[0];
    if (dest && !dest_fits(dest, o)) return fail(c, CTMR_E_BATCH_TOO_LARGE, "set export: output buffers too small");
    uint8_t* blob = nullptr;
    CU(c, mem.alloc(&blob, o.serial_bytes));
    member_pack_kernel<<<blocks_of(n), 256, 0, s>>>(pos_b, staging, n, soff, blob);
    CU(c, cudaGetLastError());
    uint64_t *out_first = nullptr, *out_soff = nullptr;
    uint8_t* out_blob = nullptr;
    if (dest) {
        out_first = dest->first_index;
        out_soff = dest->serial_off;
        out_blob = dest->serials;
    } else {
        o.first.resize(n);
        o.soff.resize(n + 1);
        o.blob.resize(o.serial_bytes);
        out_first = o.first.data();
        out_soff = o.soff.data();
        out_blob = o.blob.data();
    }
    CU(c, cudaMemcpyAsync(out_first, first_b, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
    CU(c, cudaMemcpyAsync(out_soff, soff, (n + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
    if (o.serial_bytes) CU(c, cudaMemcpyAsync(out_blob, blob, o.serial_bytes, cudaMemcpyDeviceToHost, s));
    CU(c, cudaStreamSynchronize(s));
    return CTMR_OK;
}

// ---- merge of the shards of a group (their sets are disjoint) ----------------------------------------------------
struct SetRef {
    const ctmr_set_info* s;
    uint32_t shard;
};

std::vector<SetRef> merged_order(const std::vector<ShardSets>& sh) {
    std::vector<SetRef> refs;
    for (uint32_t r = 0; r < sh.size(); ++r)
        for (const ctmr_set_info& si : sh[r].sets) refs.push_back({&si, r});
    std::sort(refs.begin(), refs.end(), [](const SetRef& a, const SetRef& b) {
        const int d = std::memcmp(a.s->issuer_digest, b.s->issuer_digest, 32);
        return d != 0 ? d < 0 : a.s->exp_hour < b.s->exp_hour;
    });
    return refs;
}

// ---- import ------------------------------------------------------------------------------------------------------
int import_validate(ctmr_ctx* c, const ctmr_set_export* x) {
    if (!x) return fail(c, CTMR_E_INVALID, "bad argument");
    if ((x->n_sets && !x->sets) || (x->n_members && (!x->serial_off || !x->first_index || !x->serials)))
        return fail(c, CTMR_E_INVALID, "import: missing arrays");
    for (uint64_t j = 0; j < x->n_sets; ++j) {
        const ctmr_set_info& si = x->sets[j];
        if (si.exp_hour > INT32_MAX || si.exp_hour < INT32_MIN) return fail(c, CTMR_E_INVALID, "import: exp_hour out of range");
        if (si.member_off > x->n_members || si.count > x->n_members - si.member_off)
            return fail(c, CTMR_E_INVALID, "import: a set's members lie outside the member arrays");
    }
    for (uint64_t k = 0; k < x->n_members; ++k) {
        const uint64_t a = x->serial_off[k], b = x->serial_off[k + 1];
        if (b < a || b > x->serial_bytes || b - a == 0 || b - a > CTMR_MAX_SERIAL)
            return fail(c, CTMR_E_INVALID, "import: serial empty or longer than CTMR_MAX_SERIAL");
    }
    return CTMR_OK;
}

int shard_is_empty(ctmr_ctx* c, bool* empty) {
    uint64_t used = 0;
    const int rc = ctmr_table_stats(c, &used, nullptr);
    *empty = used == 0;
    return rc;
}

// key records of the sets, per owner (world 1: all to owner 0); only_rank >= 0 keeps the sets that rank owns.
// `reg` registers unknown digests (the group's registry).
int import_keys(ctmr_ctx* reg, const ctmr_set_export* x, uint32_t world, int only_rank, std::vector<std::vector<ctmr_key>>& keys) {
    keys.assign(world, {});
    for (uint64_t j = 0; j < x->n_sets; ++j) {
        const ctmr_set_info& si = x->sets[j];
        uint32_t issuer = 0;
        bool found = false;
        const int rc = lookup_digest(reg, si.issuer_digest, true, &issuer, &found);
        if (rc) return rc;
        const uint32_t owner = world > 1 ? key_owner((int32_t)si.exp_hour, issuer, world) : 0u;
        if (only_rank >= 0 && owner != (uint32_t)only_rank) continue;
        std::vector<ctmr_key>& dst = keys[owner];
        for (uint64_t k = si.member_off; k < si.member_off + si.count; ++k) {
            ctmr_key key;
            std::memset(&key, 0, sizeof key);
            const uint64_t a = x->serial_off[k], len = x->serial_off[k + 1] - a;
            key.index = x->first_index[k];
            key.exp_hour = (int32_t)si.exp_hour;
            key.issuer = issuer;
            key.serial_len = (uint8_t)len;
            std::memcpy(key.serial, x->serials + a, len);
            key.valid = 1;
            dst.push_back(key);
        }
    }
    return CTMR_OK;
}

void copy_sets(const std::vector<ctmr_set_info>& sets, ctmr_set_info* out) { std::copy(sets.begin(), sets.end(), out); }

}  // namespace

extern "C" {

// ------------------------------------------------------------------------------------------------ one ctx / one shard
int ctmr_list_sets(ctmr_ctx* c, int64_t min_exp_hour, int64_t max_exp_hour, ctmr_set_info* out, uint64_t cap, uint64_t* n) {
    if (!c || !n) return fail(c, CTMR_E_INVALID, "bad argument");
    const SetFilter f{min_exp_hour, max_exp_hour, 0ull};
    if (!out) return shard_count(c, f, false, n, nullptr, nullptr);
    ShardSets sh;
    const int rc = shard_scan(c, f, false, sh, nullptr);
    if (rc) return rc;
    *n = sh.sets.size();
    if (cap < *n) return fail(c, CTMR_E_BATCH_TOO_LARGE, "list_sets: output buffer too small");
    copy_sets(sh.sets, out);
    return CTMR_OK;
}

int ctmr_set_members(ctmr_ctx* c, int64_t exp_hour, const uint8_t digest[32], uint8_t* serials, uint64_t serials_cap, uint64_t* serial_off,
                     uint64_t* first_index, uint64_t cap, uint64_t* n) {
    if (!c || !digest || !n) return fail(c, CTMR_E_INVALID, "bad argument");
    const bool sizing = !serials && !serial_off && !first_index;
    if (!sizing && (!serials || !serial_off || !first_index)) return fail(c, CTMR_E_INVALID, "set_members: give all three output arrays or none");
    CU(c, cudaSetDevice(c->device));
    *n = 0;
    uint32_t issuer = 0;
    bool found = false;
    const int rc = lookup_digest(c, digest, false, &issuer, &found);
    if (rc) return rc;
    if (!found || exp_hour > INT32_MAX || exp_hour < INT32_MIN) {
        if (serial_off) serial_off[0] = 0;
        return CTMR_OK;
    }
    const SetFilter f{exp_hour, exp_hour, pair_key(issuer, (int32_t)exp_hour)};
    if (sizing) return shard_count(c, f, false, nullptr, n, nullptr);
    const MemberDest d{serials, serials_cap, serial_off, first_index, cap, UINT64_MAX};
    ShardSets sh;
    const int rc2 = shard_scan(c, f, true, sh, &d);
    *n = sh.n_members;
    return rc2;
}

int ctmr_export_sets(ctmr_ctx* c, ctmr_set_export* x) {
    if (!c || !x) return fail(c, CTMR_E_INVALID, "bad argument");
    x->next_index = c->group ? c->group->next_index : c->next_index;
    if (!x->sets || !x->serials || !x->serial_off || !x->first_index)
        return shard_count(c, kAllSets, true, &x->n_sets, &x->n_members, &x->serial_bytes);
    const MemberDest d{x->serials, x->serials_cap, x->serial_off, x->first_index, x->members_cap, x->sets_cap};
    ShardSets sh;
    const int rc = shard_scan(c, kAllSets, true, sh, &d);
    x->n_sets = sh.sets.size();
    x->n_members = sh.n_members;
    x->serial_bytes = sh.serial_bytes;
    if (rc) return rc;
    copy_sets(sh.sets, x->sets);
    return CTMR_OK;
}

int ctmr_import_sets(ctmr_ctx* c, const ctmr_set_export* x) {
    if (!c) return CTMR_E_INVALID;
    if (c->group) return fail(c, CTMR_E_INVALID, "member of a group: use ctmr_group_import_sets");
    int rc = import_validate(c, x);
    if (rc) return rc;
    CU(c, cudaSetDevice(c->device));
    bool empty = false;
    rc = shard_is_empty(c, &empty);
    if (rc) return rc;
    if (c->next_index != 0 || !empty) return fail(c, CTMR_E_INVALID, "import_sets needs an empty ctx (no batch, preload or import so far)");
    // a rank of a peer group keeps the sets it owns: every rank can be handed the same full export
    const bool peer = c->st.peer.world > 1;
    std::vector<std::vector<ctmr_key>> keys;
    rc = import_keys(c, x, peer ? c->st.peer.world : 1u, peer ? (int)c->st.peer.rank : -1, keys);
    if (rc) return rc;
    rc = reduce_keys_host(c, keys[peer ? c->st.peer.rank : 0].data(), keys[peer ? c->st.peer.rank : 0].size());
    if (rc) return rc;
    c->next_index = x->next_index;
    return CTMR_OK;
}

// ------------------------------------------------------------------------------------------------ in-process group
int ctmr_group_list_sets(ctmr_group* g, int64_t min_exp_hour, int64_t max_exp_hour, ctmr_set_info* out, uint64_t cap, uint64_t* n) {
    if (!g || g->m.empty() || !n) return CTMR_E_INVALID;
    const uint32_t W = (uint32_t)g->m.size();
    const SetFilter f{min_exp_hour, max_exp_hour, 0ull};
    std::vector<int> rcs;
    if (!out) {
        std::vector<uint64_t> part(W, 0);
        for_each_member(W, rcs, [&](uint32_t r) { return shard_count(g->m[r], f, false, &part[r], nullptr, nullptr); });
        for (uint32_t r = 0; r < W; ++r)
            if (rcs[r]) return group_fail(g, g->m[r], rcs[r]);
        *n = std::accumulate(part.begin(), part.end(), (uint64_t)0);
        return CTMR_OK;
    }
    std::vector<ShardSets> sh(W);
    for_each_member(W, rcs, [&](uint32_t r) { return shard_scan(g->m[r], f, false, sh[r], nullptr); });
    for (uint32_t r = 0; r < W; ++r)
        if (rcs[r]) return group_fail(g, g->m[r], rcs[r]);
    const std::vector<SetRef> refs = merged_order(sh);
    *n = refs.size();
    if (cap < *n) return group_fail(g, g->m[0], fail(g->m[0], CTMR_E_BATCH_TOO_LARGE, "list_sets: output buffer too small"));
    uint64_t run = 0;
    for (uint64_t j = 0; j < refs.size(); ++j) {
        out[j] = *refs[j].s;
        out[j].member_off = run;
        run += out[j].count;
    }
    return CTMR_OK;
}

int ctmr_group_set_members(ctmr_group* g, int64_t exp_hour, const uint8_t digest[32], uint8_t* serials, uint64_t serials_cap,
                           uint64_t* serial_off, uint64_t* first_index, uint64_t cap, uint64_t* n) {
    if (!g || g->m.empty() || !digest || !n) return CTMR_E_INVALID;
    ctmr_ctx* c0 = g->m[0];
    cudaSetDevice(c0->device);
    uint32_t issuer = 0;
    bool found = false;
    int rc = lookup_digest(c0, digest, false, &issuer, &found);
    if (rc) return group_fail(g, c0, rc);
    // the set lives on its owner shard only
    ctmr_ctx* owner = found && exp_hour <= INT32_MAX && exp_hour >= INT32_MIN ? g->m[key_owner((int32_t)exp_hour, issuer, (uint32_t)g->m.size())] : c0;
    rc = ctmr_set_members(owner, exp_hour, digest, serials, serials_cap, serial_off, first_index, cap, n);
    return rc ? group_fail(g, owner, rc) : rc;
}

int ctmr_group_export_sets(ctmr_group* g, ctmr_set_export* x) {
    if (!g || g->m.empty() || !x) return CTMR_E_INVALID;
    const uint32_t W = (uint32_t)g->m.size();
    x->next_index = g->next_index;
    std::vector<int> rcs;
    if (!x->sets || !x->serials || !x->serial_off || !x->first_index) {
        std::vector<uint64_t> s(W, 0), m(W, 0), b(W, 0);
        for_each_member(W, rcs, [&](uint32_t r) { return shard_count(g->m[r], kAllSets, true, &s[r], &m[r], &b[r]); });
        for (uint32_t r = 0; r < W; ++r)
            if (rcs[r]) return group_fail(g, g->m[r], rcs[r]);
        x->n_sets = std::accumulate(s.begin(), s.end(), (uint64_t)0);
        x->n_members = std::accumulate(m.begin(), m.end(), (uint64_t)0);
        x->serial_bytes = std::accumulate(b.begin(), b.end(), (uint64_t)0);
        return CTMR_OK;
    }
    std::vector<ShardSets> sh(W);
    for_each_member(W, rcs, [&](uint32_t r) { return shard_scan(g->m[r], kAllSets, true, sh[r], nullptr); });
    for (uint32_t r = 0; r < W; ++r)
        if (rcs[r]) return group_fail(g, g->m[r], rcs[r]);
    x->n_sets = x->n_members = x->serial_bytes = 0;
    for (const ShardSets& p : sh) {
        x->n_sets += p.sets.size();
        x->n_members += p.n_members;
        x->serial_bytes += p.serial_bytes;
    }
    if (x->sets_cap < x->n_sets || x->members_cap < x->n_members || x->serials_cap < x->serial_bytes)
        return group_fail(g, g->m[0], fail(g->m[0], CTMR_E_BATCH_TOO_LARGE, "set export: output buffers too small"));
    const std::vector<SetRef> refs = merged_order(sh);
    uint64_t mk = 0, bytes = 0;
    for (uint64_t j = 0; j < refs.size(); ++j) {
        const ShardSets& p = sh[refs[j].shard];
        const ctmr_set_info& si = *refs[j].s;
        x->sets[j] = si;
        x->sets[j].member_off = mk;
        for (uint64_t k = si.member_off; k < si.member_off + si.count; ++k, ++mk) {
            const uint64_t a = p.soff[k], len = p.soff[k + 1] - a;
            x->first_index[mk] = p.first[k];
            x->serial_off[mk] = bytes;
            std::memcpy(x->serials + bytes, p.blob.data() + a, len);
            bytes += len;
        }
    }
    x->serial_off[mk] = bytes;
    return CTMR_OK;
}

int ctmr_group_import_sets(ctmr_group* g, const ctmr_set_export* x) {
    if (!g || g->m.empty()) return CTMR_E_INVALID;
    const uint32_t W = (uint32_t)g->m.size();
    ctmr_ctx* c0 = g->m[0];
    int rc = import_validate(c0, x);
    if (rc) return group_fail(g, c0, rc);
    bool all_empty = g->next_index == 0;
    for (ctmr_ctx* c : g->m) {
        bool empty = false;
        rc = shard_is_empty(c, &empty);
        if (rc) return group_fail(g, c, rc);
        all_empty &= empty;
    }
    if (!all_empty) return group_fail(g, c0, fail(c0, CTMR_E_INVALID, "import_sets needs an empty group (no batch, preload or import so far)"));
    std::vector<std::vector<ctmr_key>> keys;
    CU(c0, cudaSetDevice(c0->device));
    rc = import_keys(c0, x, W, -1, keys);  // every set to its owner in THIS group
    if (rc) return group_fail(g, c0, rc);
    std::vector<int> rcs;
    for_each_member(W, rcs, [&](uint32_t r) { return reduce_keys_host(g->m[r], keys[r].data(), keys[r].size()); });
    for (uint32_t r = 0; r < W; ++r)
        if (rcs[r]) return group_fail(g, g->m[r], rcs[r]);
    g->next_index = x->next_index;
    return CTMR_OK;
}

}  // extern "C"
