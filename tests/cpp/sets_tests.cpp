// sets_tests.cpp -- the set read-back of the C++ host mirror (ct_mapreduce_b200/host/ctmr_storage.hpp):
//   sets_tests gpu <dir> <batches> [pipelined] [shards]
// StoreBatch of a corpus on disk into a MockRemoteCache, then RebuildRemoteCache from the device into a fresh mock of the
// same kind: both mocks must hold the same serials:: sets and expiry times; GetIssuerAndDatesFromDevice and
// KnownFromDevice must answer what the first mock holds.
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <iostream>

#include "../../ct_mapreduce_b200/host/ctmr_storage.hpp"

using namespace ctmr_host;

#define CHECK(c)                                                                                              \
    do {                                                                                                      \
        if (!(c)) { std::fprintf(stderr, "FAIL %s:%d: %s\n", __FILE__, __LINE__, #c); std::exit(1); }      \
    } while (0)

template <class T>
static std::vector<T> read_all(const std::string& path) {
    std::ifstream f(path, std::ios::binary);
    if (!f) { std::fprintf(stderr, "cannot open %s\n", path.c_str()); std::exit(2); }
    f.seekg(0, std::ios::end);
    const size_t n = (size_t)f.tellg();
    f.seekg(0);
    std::vector<T> v(n / sizeof(T));
    f.read(reinterpret_cast<char*>(v.data()), (std::streamsize)(v.size() * sizeof(T)));
    return v;
}

static bool is_serials(const std::string& k) { return k.compare(0, 9, "serials::") == 0; }

static int run(const std::string& dir, int batches, bool pipelined, int shards) {
    auto blob = read_all<uint8_t>(dir + "/blob.bin");
    auto offs = read_all<uint64_t>(dir + "/offsets.bin");
    auto iblob = read_all<uint8_t>(dir + "/issuer_blob.bin");
    auto ioffs = read_all<uint64_t>(dir + "/issuer_offsets.bin");
    auto idx = read_all<uint32_t>(dir + "/issuer_idx.bin");
    auto now = read_all<int64_t>(dir + "/now_ns.bin");
    const uint64_t n = offs.size() - 1;
    ctmr_config cfg{};
    cfg.struct_size = sizeof cfg;
    cfg.table_capacity = 1 << 16;
    cfg.log_expired_entries = 1;
    ctmr_ctx* ctx = nullptr;
    ctmr_group* group = nullptr;
    if (shards > 1) {
        std::vector<int32_t> devs((size_t)shards, 0);
        if (ctmr_group_create(&cfg, devs.data(), (uint32_t)shards, &group) != CTMR_OK) {
            std::fprintf(stderr, "ctmr_group_create: %s\n", ctmr_group_last_error(nullptr));
            return 3;
        }
    } else if (ctmr_create(&cfg, &ctx) != CTMR_OK) {
        std::fprintf(stderr, "ctmr_create: %s\n", ctmr_last_error(nullptr));
        return 3;
    }
    MockBatchRemoteCache batch_a, batch_b;
    MockRemoteCache plain_a, plain_b;
    MockRemoteCache& a = pipelined ? static_cast<MockRemoteCache&>(batch_a) : plain_a;
    MockRemoteCache& b = pipelined ? static_cast<MockRemoteCache&>(batch_b) : plain_b;
    MockBackend backend;
    GpuCertDatabase db_single(ctx, &a, &backend), db_group(group, &a, &backend);
    GpuCertDatabase& db = group ? db_group : db_single;
    for (int k = 0; k < batches; ++k) {
        const uint64_t lo = n * k / batches, hi = n * (k + 1) / batches;
        Error e = db.StoreBatch(blob.data(), offs.data() + lo, hi - lo, iblob.data(), ioffs.data(), (uint32_t)ioffs.size() - 1,
                                idx.data() + lo, now[0]);
        if (!ok(e)) { std::fprintf(stderr, "StoreBatch: %s\n", e.c_str()); return 4; }
    }
    Error e = db.RebuildRemoteCache(&b);
    if (!ok(e)) { std::fprintf(stderr, "RebuildRemoteCache: %s\n", e.c_str()); return 5; }
    // the same serials:: sets and expiry times in both caches
    std::map<std::string, std::vector<std::string>> sa, sb;
    std::map<std::string, int64_t> ea, eb;
    uint64_t members = 0;
    for (const auto& kv : a.Data) if (is_serials(kv.first)) { sa[kv.first] = kv.second; members += kv.second.size(); }
    for (const auto& kv : b.Data) if (is_serials(kv.first)) sb[kv.first] = kv.second;
    for (const auto& kv : a.Expirations) if (is_serials(kv.first)) ea[kv.first] = kv.second;
    for (const auto& kv : b.Expirations) if (is_serials(kv.first)) eb[kv.first] = kv.second;
    CHECK(!sa.empty() && members > sa.size());
    CHECK(sa == sb);
    CHECK(ea == eb);
    CHECK(b.Data.size() == sb.size() && b.Expirations.size() == eb.size());  // nothing but the serials:: sets
    if (pipelined) CHECK(batch_b.round_trips == 2);
    else CHECK(b.set_insert_calls == members);
    // the read side from the device answers what the cache holds
    auto listed = db.GetIssuerAndDatesFromDevice();
    CHECK(ok(listed.second) && listed.first.size() == sa.size());
    for (const auto& s : listed.first) {
        KnownCertificates kc(s.expDate, s.issuer, &a);
        const std::string key = kc.serialId();
        CHECK(sa.count(key) && sa[key].size() == s.count);
        auto known = db.KnownFromDevice(s.expDate, s.issuer);
        CHECK(ok(known.second) && known.first.size() == s.count);
        std::vector<std::string> got;
        for (const auto& ser : known.first) got.push_back(ser.BinaryString());
        std::sort(got.begin(), got.end());
        CHECK(got == sa[key]);
    }
    // an hour range keeps the sets inside it
    const int64_t mid = listed.first[listed.first.size() / 2].expDate.hour;
    auto upper = db.GetIssuerAndDatesFromDevice(mid, INT64_MAX);
    size_t want = 0;
    for (const auto& s : listed.first) want += s.expDate.hour >= mid;
    CHECK(ok(upper.second) && upper.first.size() == want);
    std::printf("sets cpp ok: %zu sets, %llu members\n", sa.size(), (unsigned long long)members);
    if (group) ctmr_group_destroy(group);
    else ctmr_destroy(ctx);
    return 0;
}

int main(int argc, char** argv) {
    if (argc >= 4 && std::string(argv[1]) == "gpu")
        return run(argv[2], std::atoi(argv[3]), argc >= 5 && std::string(argv[4]) == "pipelined", argc >= 6 ? std::atoi(argv[5]) : 1);
    std::fprintf(stderr, "usage: sets_tests gpu <dir> <batches> [pipelined|plain] [shards]\n");
    return 64;
}
