// ctmr_storage.hpp -- C++ host side of the drop-in, above the C ABI (include/ctmr.h).
//
// The reference's host language is Go and this image has no Go toolchain, so the host-side mirror of
// the reference's plug-in surface for THIS path is written in C++ (header-only): the same interface
// names, argument meaning and error behaviour as storage/types.go:46-102, the mock implementations
// the reference's own tests use, the two reducers as thin objects over RemoteCache, and
// GpuCertDatabase::StoreBatch -- what replaces N x insertCTWorker -> FilesystemDatabase.Store.
// The GPU decides; every side effect still flows through RemoteCache / StorageBackend, in entry
// order, exactly as the reference would have issued it.
//
//   RemoteCache        storage/types.go:83-102      (18 methods, kept)
//   StorageBackend     storage/types.go:46-68       (12 methods, kept)
//   MockRemoteCache    storage/mockcache.go         (sorted unique string slices)
//   MockBackend        storage/mockbackend.go, NoopBackend storage/noopbackend.go
//   ExpDate/Issuer/Serial  storage/types.go:104-255,333-384 (ID formats)
//   KnownCertificates  storage/knowncertificates.go
//   IssuerMetadata     storage/issuermetadata.go
//   GpuCertDatabase    storage/filesystemdatabase.go:158-240 (Store, GetKnownCertificates, GetIssuerMetadata)
#pragma once
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <functional>
#include <map>
#include <memory>
#include <set>
#include <string>
#include <utility>
#include <vector>

#include "../../include/ctmr.h"

namespace ctmr_host {

// Go's `error`: empty string = nil
using Error = std::string;
inline bool ok(const Error& e) { return e.empty(); }

// ---------------------------------------------------------------------------------- value types
inline std::string Base64URL(const uint8_t* p, size_t n) {  // encoding/base64.URLEncoding (padded)
    static const char A[] = "ABCDEFGHIJKLMNOPQRSTUVWXYZabcdefghijklmnopqrstuvwxyz0123456789-_";
    std::string o;
    size_t i = 0;
    for (; i + 3 <= n; i += 3) {
        uint32_t v = (p[i] << 16) | (p[i + 1] << 8) | p[i + 2];
        o += A[v >> 18]; o += A[(v >> 12) & 63]; o += A[(v >> 6) & 63]; o += A[v & 63];
    }
    if (n - i == 1) { uint32_t v = p[i] << 16; o += A[v >> 18]; o += A[(v >> 12) & 63]; o += "=="; }
    if (n - i == 2) { uint32_t v = (p[i] << 16) | (p[i + 1] << 8); o += A[v >> 18]; o += A[(v >> 12) & 63]; o += A[(v >> 6) & 63]; o += '='; }
    return o;
}

inline void CivilFromDays(int64_t z, int64_t& y, unsigned& m, unsigned& d) {
    z += 719468;
    const int64_t era = (z >= 0 ? z : z - 146096) / 146097;
    const unsigned doe = (unsigned)(z - era * 146097);
    const unsigned yoe = (doe - doe / 1460 + doe / 36524 - doe / 146096) / 365;
    const unsigned doy = doe - (365 * yoe + yoe / 4 - yoe / 100);
    const unsigned mp = (5 * doy + 2) / 153;
    d = doy - (153 * mp + 2) / 5 + 1;
    m = mp < 10 ? mp + 3 : mp - 9;
    y = (int64_t)yoe + era * 400 + (m <= 2);
}

struct ExpDate {  // storage/types.go:333-384, hour resolution
    int64_t hour = 0;  // floor(unix / 3600): NewExpDateFromTime = t.Truncate(time.Hour)
    static ExpDate FromUnix(int64_t s) { return ExpDate{s >= 0 ? s / 3600 : -((-s + 3599) / 3600)}; }
    int64_t ExpireTimeUnix() const { return hour * 3600; }
    std::string ID() const {  // "2006-01-02-15"
        const int64_t days = hour >= 0 ? hour / 24 : -((-hour + 23) / 24);
        int64_t y; unsigned m, d;
        CivilFromDays(days, y, m, d);
        char b[64];
        std::snprintf(b, sizeof b, "%04lld-%02u-%02u-%02u", (long long)y, m, d, (unsigned)(hour - days * 24));
        return b;
    }
    std::string DayID() const {  // kExpirationFormat "2006-01-02" (markDirty, filesystemdatabase.go:140-143)
        return ID().substr(0, 10);
    }
    bool operator<(const ExpDate& o) const { return hour < o.hour; }
};

struct Issuer {  // storage/types.go:104-141: id = base64url(SHA-256(SPKI)); the digest comes from the GPU
    std::string id;
    static Issuer FromDigest(const uint8_t d[32]) { return Issuer{Base64URL(d, 32)}; }
    static Issuer FromString(std::string s) { return Issuer{std::move(s)}; }
    const std::string& ID() const { return id; }
};

struct Serial {  // storage/types.go:161-255: raw INTEGER content octets, leading zeros kept
    std::string bytes;
    static Serial FromBytes(const uint8_t* p, size_t n) { return Serial{std::string((const char*)p, n)}; }
    static Serial FromHex(const std::string& h) {
        Serial s;
        for (size_t i = 0; i + 1 < h.size(); i += 2) s.bytes.push_back((char)std::stoi(h.substr(i, 2), nullptr, 16));
        return s;
    }
    const std::string& BinaryString() const { return bytes; }
    std::string ID() const { return Base64URL((const uint8_t*)bytes.data(), bytes.size()); }
    std::string HexString() const {
        std::string o;
        char b[3];
        for (unsigned char c : bytes) { std::snprintf(b, sizeof b, "%02x", c); o += b; }
        return o;
    }
};

// ---------------------------------------------------------------------------------- plug-in interfaces
struct CertificateLog {  // storage/types.go:25-30
    std::string ShortURL;
    int64_t MaxEntry = 0;
    int64_t LastEntryTime = 0, LastUpdateTime = 0;
};

class RemoteCache {  // storage/types.go:83-102 -- method set unchanged; channels become callbacks
  public:
    virtual ~RemoteCache() = default;
    virtual std::pair<bool, Error> Exists(const std::string& key) = 0;
    virtual std::pair<bool, Error> SetInsert(const std::string& key, const std::string& entry) = 0;  // true iff newly added
    virtual std::pair<bool, Error> SetRemove(const std::string& key, const std::string& entry) = 0;
    virtual std::pair<bool, Error> SetContains(const std::string& key, const std::string& entry) = 0;
    virtual std::pair<std::vector<std::string>, Error> SetList(const std::string& key) = 0;
    virtual Error SetToChan(const std::string& key, const std::function<void(const std::string&)>& c) = 0;
    virtual std::pair<int, Error> SetCardinality(const std::string& key) = 0;
    virtual Error ExpireAt(const std::string& key, int64_t unix_time) = 0;
    virtual Error ExpireIn(const std::string& key, int64_t seconds) = 0;
    virtual std::pair<int64_t, Error> Queue(const std::string& key, const std::string& identifier) = 0;
    virtual std::pair<std::string, Error> Pop(const std::string& key) = 0;
    virtual std::pair<int64_t, Error> QueueLength(const std::string& key) = 0;
    virtual std::pair<std::string, Error> BlockingPopCopy(const std::string& key, const std::string& dest, int64_t timeout_s) = 0;
    virtual Error ListRemove(const std::string& key, const std::string& value) = 0;
    virtual std::pair<std::string, Error> TrySet(const std::string& k, const std::string& v, int64_t life_s) = 0;
    virtual Error KeysToChan(const std::string& pattern, const std::function<void(const std::string&)>& c) = 0;
    virtual Error StoreLogState(const CertificateLog& log) = 0;
    virtual std::pair<CertificateLog, Error> LoadLogState(const std::string& url) = 0;
};

// Optional extension of a RemoteCache (SURVEY §8(f)-3): the SADD / EXPIREAT traffic of one GPU batch in ONE pipelined
// round trip each (go-redis Pipeline over rediscache.go:57-65,116-120) instead of one per new certificate.  The Go
// shim discovers it with a type assertion (`if bc, ok := cache.(BatchRemoteCache); ok { ... }`), this mirror with
// dynamic_cast; a cache without it gets the per-entry calls, so the interface of storage/types.go:83-102 is untouched.
class BatchRemoteCache {
  public:
    virtual ~BatchRemoteCache() = default;
    struct Insert { std::string key, entry; };
    struct Expire { std::string key; int64_t unix_time; };
    // results[i] = what SetInsert(ops[i].key, ops[i].entry) returns when the operations are applied in order
    virtual std::pair<std::vector<bool>, Error> SetInsertBatch(const std::vector<Insert>& ops) = 0;
    virtual Error ExpireAtBatch(const std::vector<Expire>& ops) = 0;
};

class StorageBackend {  // storage/types.go:46-68 -- method set unchanged (context.Context dropped)
  public:
    virtual ~StorageBackend() = default;
    virtual Error MarkDirty(const std::string& id) = 0;
    virtual Error StoreCertificatePEM(const Serial&, const ExpDate&, const Issuer&, const std::string& pem) = 0;
    virtual Error StoreLogState(const CertificateLog&) = 0;
    virtual Error StoreKnownCertificateList(const Issuer&, const std::vector<Serial>&) = 0;
    virtual std::pair<std::string, Error> LoadCertificatePEM(const Serial&, const ExpDate&, const Issuer&) = 0;
    virtual std::pair<CertificateLog, Error> LoadLogState(const std::string& url) = 0;
    virtual Error AllocateExpDateAndIssuer(const ExpDate&, const Issuer&) = 0;
    virtual std::pair<std::vector<ExpDate>, Error> ListExpirationDates(int64_t not_before_unix) = 0;
    virtual std::pair<std::vector<Issuer>, Error> ListIssuersForExpirationDate(const ExpDate&) = 0;
    virtual std::pair<std::vector<Serial>, Error> ListSerialsForExpirationDateAndIssuer(const ExpDate&, const Issuer&) = 0;
    virtual Error StreamSerialsForExpirationDateAndIssuer(const ExpDate&, const Issuer&,
                                                          const std::function<void(const Serial&)>& stream) = 0;
};

// ---------------------------------------------------------------------------------- mocks (the reference's test doubles)
class MockRemoteCache : public RemoteCache {  // storage/mockcache.go
  public:
    std::map<std::string, std::vector<std::string>> Data;  // sorted unique strings per key (mockcache.go:38-61)
    std::map<std::string, int64_t> Expirations;
    uint64_t set_insert_calls = 0;  // for tests: how many round trips a Redis would have seen

    std::pair<bool, Error> Exists(const std::string& key) override { return {Data.count(key) != 0, ""}; }
    std::pair<bool, Error> SetInsert(const std::string& key, const std::string& entry) override {
        ++set_insert_calls;
        auto& v = Data[key];
        auto it = std::lower_bound(v.begin(), v.end(), entry);  // strings.Compare order = bytewise
        if (it != v.end() && *it == entry) return {false, ""};
        v.insert(it, entry);
        return {true, ""};
    }
    std::pair<bool, Error> SetRemove(const std::string& key, const std::string& entry) override {
        auto& v = Data[key];
        auto it = std::lower_bound(v.begin(), v.end(), entry);
        if (it != v.end() && *it == entry) { v.erase(it); return {true, ""}; }
        return {false, ""};
    }
    std::pair<bool, Error> SetContains(const std::string& key, const std::string& entry) override {
        auto& v = Data[key];
        return {std::binary_search(v.begin(), v.end(), entry), ""};
    }
    std::pair<std::vector<std::string>, Error> SetList(const std::string& key) override { return {Data[key], ""}; }
    Error SetToChan(const std::string& key, const std::function<void(const std::string&)>& c) override {
        for (const auto& s : Data[key]) c(s);
        return "";
    }
    std::pair<int, Error> SetCardinality(const std::string& key) override {
        auto it = Data.find(key);
        return {it == Data.end() ? 0 : (int)it->second.size(), ""};
    }
    Error ExpireAt(const std::string& key, int64_t t) override { Expirations[key] = t; return ""; }
    Error ExpireIn(const std::string&, int64_t) override { return "unimplemented"; }
    std::pair<int64_t, Error> Queue(const std::string&, const std::string&) override { return {0, "unimplemented"}; }
    std::pair<std::string, Error> Pop(const std::string&) override { return {"", "unimplemented"}; }
    std::pair<int64_t, Error> QueueLength(const std::string&) override { return {0, "unimplemented"}; }
    std::pair<std::string, Error> BlockingPopCopy(const std::string&, const std::string&, int64_t) override { return {"", "unimplemented"}; }
    Error ListRemove(const std::string&, const std::string&) override { return "unimplemented"; }
    std::pair<std::string, Error> TrySet(const std::string& k, const std::string& v, int64_t) override {
        auto& d = Data[k];
        if (d.empty()) d.push_back(v);
        return {d[0], ""};
    }
    Error KeysToChan(const std::string& pattern, const std::function<void(const std::string&)>& c) override {
        const std::string prefix = pattern.substr(0, pattern.find('*'));  // the path only uses "serials::*"
        for (const auto& kv : Data)
            if (kv.first.compare(0, prefix.size(), prefix) == 0) c(kv.first);
        return "";
    }
    Error StoreLogState(const CertificateLog& l) override { logs_[l.ShortURL] = l; return ""; }
    std::pair<CertificateLog, Error> LoadLogState(const std::string& url) override {
        auto it = logs_.find(url);
        if (it == logs_.end()) return {CertificateLog{url}, ""};
        return {it->second, ""};
    }

  private:
    std::map<std::string, CertificateLog> logs_;
};

// MockRemoteCache that also offers the pipelined extension; round_trips counts what a Redis would have seen
class MockBatchRemoteCache : public MockRemoteCache, public BatchRemoteCache {
  public:
    uint64_t round_trips = 0;
    std::pair<std::vector<bool>, Error> SetInsertBatch(const std::vector<Insert>& ops) override {
        ++round_trips;
        std::vector<bool> r(ops.size());
        for (size_t i = 0; i < ops.size(); ++i) {
            auto one = MockRemoteCache::SetInsert(ops[i].key, ops[i].entry);
            if (!ok(one.second)) return {r, one.second};
            r[i] = one.first;
        }
        return {r, ""};
    }
    Error ExpireAtBatch(const std::vector<Expire>& ops) override {
        ++round_trips;
        for (const auto& o : ops) {
            Error e = MockRemoteCache::ExpireAt(o.key, o.unix_time);
            if (!ok(e)) return e;
        }
        return "";
    }
};

class NoopBackend : public StorageBackend {  // storage/noopbackend.go: stores succeed, loads error
  public:
    Error MarkDirty(const std::string&) override { return ""; }
    Error StoreCertificatePEM(const Serial&, const ExpDate&, const Issuer&, const std::string&) override { return ""; }
    Error StoreLogState(const CertificateLog&) override { return ""; }
    Error StoreKnownCertificateList(const Issuer&, const std::vector<Serial>&) override { return ""; }
    std::pair<std::string, Error> LoadCertificatePEM(const Serial&, const ExpDate&, const Issuer&) override { return {"", "noop"}; }
    std::pair<CertificateLog, Error> LoadLogState(const std::string&) override { return {{}, "noop"}; }
    Error AllocateExpDateAndIssuer(const ExpDate&, const Issuer&) override { return ""; }
    std::pair<std::vector<ExpDate>, Error> ListExpirationDates(int64_t) override { return {{}, "noop"}; }
    std::pair<std::vector<Issuer>, Error> ListIssuersForExpirationDate(const ExpDate&) override { return {{}, "noop"}; }
    std::pair<std::vector<Serial>, Error> ListSerialsForExpirationDateAndIssuer(const ExpDate&, const Issuer&) override { return {{}, "noop"}; }
    Error StreamSerialsForExpirationDateAndIssuer(const ExpDate&, const Issuer&, const std::function<void(const Serial&)>&) override { return "noop"; }
};

class MockBackend : public NoopBackend {  // storage/mockbackend.go: in-memory maps
  public:
    std::map<std::string, std::string> pems;                         // "<exp>/<issuer>/<serialID>" -> PEM
    std::map<std::string, std::set<std::string>> issuers_by_expdate;  // AllocateExpDateAndIssuer
    std::set<std::string> dirty;
    uint64_t mark_dirty_calls = 0;
    Error MarkDirty(const std::string& id) override { ++mark_dirty_calls; dirty.insert(id); return ""; }
    Error StoreCertificatePEM(const Serial& s, const ExpDate& e, const Issuer& i, const std::string& pem) override {
        pems[e.ID() + "/" + i.ID() + "/" + s.ID()] = pem;
        return "";
    }
    Error AllocateExpDateAndIssuer(const ExpDate& e, const Issuer& i) override { issuers_by_expdate[e.ID()].insert(i.ID()); return ""; }
    std::pair<std::string, Error> LoadCertificatePEM(const Serial& s, const ExpDate& e, const Issuer& i) override {
        auto it = pems.find(e.ID() + "/" + i.ID() + "/" + s.ID());
        if (it == pems.end()) return {"", "not found"};
        return {it->second, ""};
    }
};

// ---------------------------------------------------------------------------------- reducers
class KnownCertificates {  // storage/knowncertificates.go
  public:
    KnownCertificates(ExpDate e, Issuer i, RemoteCache* c) : expDate_(e), issuer_(std::move(i)), cache_(c) {}
    std::string serialId() const { return "serials::" + expDate_.ID() + "::" + issuer_.ID(); }  // :28-34
    // :38-55 -- true iff this serial was unknown; first call sets the key's expiry
    std::pair<bool, Error> WasUnknown(const Serial& s) {
        auto r = cache_->SetInsert(serialId(), s.BinaryString());
        if (!ok(r.second)) return {false, r.second};
        if (!expirySet_) { cache_->ExpireAt(serialId(), expDate_.ExpireTimeUnix()); expirySet_ = true; }
        return {r.first, ""};
    }
    int64_t Count() const { return cache_->SetCardinality(serialId()).first; }  // :57-63
    std::vector<Serial> Known() const {                                          // :65-96
        std::set<std::string> u;
        cache_->SetToChan(serialId(), [&](const std::string& s) { u.insert(s); });
        std::vector<Serial> out;
        for (const auto& s : u) out.push_back(Serial{s});
        return out;
    }
    void MarkExpirySet() { expirySet_ = true; }
    bool ExpirySet() const { return expirySet_; }
    int64_t ExpireTimeUnix() const { return expDate_.ExpireTimeUnix(); }

  private:
    ExpDate expDate_;
    Issuer issuer_;
    RemoteCache* cache_;
    bool expirySet_ = false;
};

class IssuerMetadata {  // storage/issuermetadata.go
  public:
    IssuerMetadata(Issuer i, RemoteCache* c) : issuer_(std::move(i)), cache_(c) {}
    std::string crlId() const { return "crl::" + issuer_.ID(); }
    std::string issuersId() const { return "issuer::" + issuer_.ID(); }
    // :48-73 -- trim, parse, drop ldap/ldaps and anything that is not http(s), then SetInsert
    Error addCRL(const std::string& raw) {
        size_t a = 0, b = raw.size();
        while (a < b && std::isspace((unsigned char)raw[a])) ++a;
        while (b > a && std::isspace((unsigned char)raw[b - 1])) --b;
        const std::string u = raw.substr(a, b - a);
        const size_t colon = u.find(':');
        if (colon == std::string::npos) return "";
        std::string scheme = u.substr(0, colon);
        for (auto& ch : scheme) ch = (char)std::tolower((unsigned char)ch);
        if (scheme == "ldap" || scheme == "ldaps") return "";
        if (scheme != "http" && scheme != "https") return "";
        return cache_->SetInsert(crlId(), scheme + u.substr(colon)).second;
    }
    Error addIssuerDN(const std::string& dn) { return cache_->SetInsert(issuersId(), dn).second; }  // :75-90
    // :92-138 -- returns seenExpDateBefore; memoises expDates, CRL-DPs and DNs in-process
    std::pair<bool, Error> Accumulate(const ExpDate& e, const std::string& dn, const std::vector<std::string>& crl_dps) {
        const bool seenExpDate = !knownExpDates_.insert(e.ID()).second;
        for (const auto& dp : crl_dps)
            if (knownCrlDPs_.insert(dp).second) {
                Error err = addCRL(dp);
                if (!ok(err)) return {seenExpDate, err};
            }
        if (knownIssuerDNs_.insert(dn).second) return {seenExpDate, addIssuerDN(dn)};
        return {seenExpDate, ""};
    }
    // the three memo steps of Accumulate, individually (the GPU pre-filters which ones are worth calling)
    bool NoteExpDate(const ExpDate& e) { return !knownExpDates_.insert(e.ID()).second; }
    Error NoteIssuerDN(const std::string& dn) { return knownIssuerDNs_.insert(dn).second ? addIssuerDN(dn) : ""; }
    Error NoteCRL(const std::string& dp) { return knownCrlDPs_.insert(dp).second ? addCRL(dp) : ""; }
    std::vector<std::string> Issuers() const { return cache_->SetList(issuersId()).first; }
    std::vector<std::string> CRLs() const { return cache_->SetList(crlId()).first; }

  private:
    Issuer issuer_;
    RemoteCache* cache_;
    std::set<std::string> knownCrlDPs_, knownIssuerDNs_, knownExpDates_;
};

// ---------------------------------------------------------------------------------- PEM (encoding/pem, no headers)
inline std::string PemEncode(const uint8_t* der, size_t n) {
    static const char A[] = "ABCDEFGHIJKLMNOPQRSTUVWXYZabcdefghijklmnopqrstuvwxyz0123456789+/";
    std::string b64;
    size_t i = 0;
    for (; i + 3 <= n; i += 3) {
        uint32_t v = (der[i] << 16) | (der[i + 1] << 8) | der[i + 2];
        b64 += A[v >> 18]; b64 += A[(v >> 12) & 63]; b64 += A[(v >> 6) & 63]; b64 += A[v & 63];
    }
    if (n - i == 1) { uint32_t v = der[i] << 16; b64 += A[v >> 18]; b64 += A[(v >> 12) & 63]; b64 += "=="; }
    if (n - i == 2) { uint32_t v = (der[i] << 16) | (der[i + 1] << 8); b64 += A[v >> 18]; b64 += A[(v >> 12) & 63]; b64 += A[(v >> 6) & 63]; b64 += '='; }
    std::string out = "-----BEGIN CERTIFICATE-----\n";
    for (size_t p = 0; p < b64.size(); p += 64) out += b64.substr(p, 64) + "\n";
    return out + "-----END CERTIFICATE-----\n";
}

// ---------------------------------------------------------------------------------- strings of IssuerMetadata
// Minimal DER cursor for the two host-side string extractions (only ever applied to spans the GPU
// walker has already validated).
struct DerTlv { uint8_t tag = 0; size_t hdr = 0, len = 0; bool ok = false; };
inline DerTlv DerRead(const uint8_t* d, size_t pos, size_t end) {
    DerTlv t;
    if (pos + 2 > end) return t;
    t.tag = d[pos];
    const uint8_t l = d[pos + 1];
    if (l < 0x80) { t.hdr = 2; t.len = l; }
    else {
        const size_t nb = l & 0x7f;
        if (nb == 0 || nb > 4 || pos + 2 + nb > end) return t;
        for (size_t i = 0; i < nb; ++i) t.len = (t.len << 8) | d[pos + 2 + i];
        t.hdr = 2 + nb;
    }
    t.ok = pos + t.hdr + t.len <= end;
    return t;
}

// pkix.Name.String() (issuermetadata.go:94): FillFromRDNSequence keeps the standard attribute
// types, ToRDNSequence re-emits them grouped by type in the order C, ST, L, STREET, POSTALCODE, O,
// OU, CN, SERIALNUMBER, and String() prints that sequence back to front, values of one type joined
// with '+', RFC 2253 escaping.  Pinned by the reference only for a single CN
// (issuermetadata_test.go:133 "CN=My First Issuer (tm)"); multi-attribute output follows Go's code.
inline std::string FormatIssuerDN(const uint8_t* name, size_t n) {
    static const struct { uint8_t arc; const char* label; } kOrder[] = {
        {6, "C"}, {8, "ST"}, {7, "L"}, {9, "STREET"}, {17, "POSTALCODE"}, {10, "O"}, {11, "OU"}, {3, "CN"}, {5, "SERIALNUMBER"}};
    std::map<uint8_t, std::vector<std::string>> vals;
    DerTlv seq = DerRead(name, 0, n);
    if (!seq.ok || seq.tag != 0x30) return "";
    size_t pos = seq.hdr, end = seq.hdr + seq.len;
    while (pos < end) {
        DerTlv set = DerRead(name, pos, end);
        if (!set.ok) break;
        size_t sp = pos + set.hdr, se = sp + set.len;
        while (sp < se) {
            DerTlv atv = DerRead(name, sp, se);
            if (!atv.ok) break;
            const size_t ap = sp + atv.hdr, ae = ap + atv.len;
            DerTlv oid = DerRead(name, ap, ae);
            if (!oid.ok) break;
            DerTlv val = DerRead(name, ap + oid.hdr + oid.len, ae);
            const uint8_t* o = name + ap + oid.hdr;
            const bool str = val.ok && (val.tag == 0x0c || val.tag == 0x13 || val.tag == 0x16 || val.tag == 0x14 || val.tag == 0x12);
            if (str && oid.len == 3 && o[0] == 0x55 && o[1] == 0x04) {
                const size_t vp = ap + oid.hdr + oid.len + val.hdr;
                if (o[2] == 3) vals[3] = {std::string((const char*)name + vp, val.len)};  // CommonName: the last one wins
                else vals[o[2]].push_back(std::string((const char*)name + vp, val.len));
            }
            sp += atv.hdr + atv.len;
        }
        pos += set.hdr + set.len;
    }
    std::string out;
    for (int k = (int)(sizeof kOrder / sizeof kOrder[0]) - 1; k >= 0; --k) {
        auto it = vals.find(kOrder[k].arc);
        if (it == vals.end() || it->second.empty()) continue;
        if (!out.empty()) out += ",";
        for (size_t j = 0; j < it->second.size(); ++j) {
            if (j) out += "+";
            out += kOrder[k].label;
            out += "=";
            const std::string& v = it->second[j];
            for (size_t c = 0; c < v.size(); ++c) {
                const char ch = v[c];
                bool esc = ch == ',' || ch == '+' || ch == '"' || ch == '\\' || ch == '<' || ch == '>' || ch == ';';
                if (ch == ' ') esc = c == 0 || c + 1 == v.size();
                if (ch == '#') esc = c == 0;
                if (esc) out += '\\';
                out += ch;
            }
        }
    }
    return out;
}

// cert.CRLDistributionPoints (issuermetadata.go:111): the URIs ([6] IA5String) of every
// DistributionPoint.fullName in the extension value.
inline std::vector<std::string> ExtractCrlUris(const uint8_t* v, size_t n) {
    std::vector<std::string> out;
    DerTlv seq = DerRead(v, 0, n);
    if (!seq.ok || seq.tag != 0x30) return out;
    size_t pos = seq.hdr, end = seq.hdr + seq.len;
    while (pos < end) {
        DerTlv dp = DerRead(v, pos, end);
        if (!dp.ok) break;
        size_t p1 = pos + dp.hdr, e1 = p1 + dp.len;
        while (p1 < e1) {
            DerTlv f = DerRead(v, p1, e1);
            if (!f.ok) break;
            if (f.tag == 0xa0) {  // distributionPoint [0]
                size_t p2 = p1 + f.hdr, e2 = p2 + f.len;
                DerTlv fn = DerRead(v, p2, e2);
                if (fn.ok && fn.tag == 0xa0) {  // fullName [0] GeneralNames
                    size_t p3 = p2 + fn.hdr, e3 = p3 + fn.len;
                    while (p3 < e3) {
                        DerTlv gn = DerRead(v, p3, e3);
                        if (!gn.ok) break;
                        if (gn.tag == 0x86) out.emplace_back((const char*)v + p3 + gn.hdr, gn.len);
                        p3 += gn.hdr + gn.len;
                    }
                }
            }
            p1 += f.hdr + f.len;
        }
        pos += dp.hdr + dp.len;
    }
    return out;
}

// ---------------------------------------------------------------------------------- the database facade
struct BatchStats {
    uint64_t entries = 0, stored = 0, unknown = 0, cache_inserts = 0, pem_writes = 0, dn_formats = 0, crl_parses = 0;
    uint64_t status[CTMR_ST__COUNT] = {};
};

// Replaces FilesystemDatabase for the worker path: Store() per entry becomes StoreBatch() per batch.
class GpuCertDatabase {
  public:
    GpuCertDatabase(ctmr_ctx* ctx, RemoteCache* cache, StorageBackend* backend) : ctx_(ctx), cache_(cache), backend_(backend) {}
    // several GPUs behind one handle (ctmr_group_*): the same StoreBatch, the fan-out is inside the library; registry
    // questions (issuer digests) go to member 0, whose registry is the group's
    GpuCertDatabase(ctmr_group* group, RemoteCache* cache, StorageBackend* backend)
        : ctx_(ctmr_group_member(group, 0)), group_(group), cache_(cache), backend_(backend) {}

    // filesystemdatabase.go:213-240 / :40-57 -- objects are created on demand and kept for the process lifetime
    KnownCertificates* GetKnownCertificates(const ExpDate& e, const Issuer& i) {
        auto& p = known_[e.ID() + i.ID()];
        if (!p) p.reset(new KnownCertificates(e, i, cache_));
        return p.get();
    }
    IssuerMetadata* GetIssuerMetadata(const Issuer& i) {
        auto& p = meta_[i.ID()];
        if (!p) p.reset(new IssuerMetadata(i, cache_));
        return p.get();
    }

    // One batch drained from entryChan.  `issuer_dn` / `crl_dps` are optional host-side extractors for
    // the strings of NEW certificates (IssuerMetadata.Accumulate's string sets stay on the host).
    Error StoreBatch(const uint8_t* blob, const uint64_t* offsets, uint64_t n, const uint8_t* issuer_blob,
                     const uint64_t* issuer_offsets, uint32_t n_issuers, const uint32_t* issuer_idx, int64_t now_unix_ns,
                     BatchStats* stats = nullptr,
                     const std::function<std::string(uint64_t)>& issuer_dn = nullptr,
                     const std::function<std::vector<std::string>(uint64_t)>& crl_dps = nullptr) {
        std::vector<uint8_t> status(n), unknown(n), first(n);
        std::vector<int64_t> exp_hour(n);
        std::vector<uint32_t> soff(n), slen(n), noff(n), nlen(n), coff(n), clen(n);
        std::vector<uint8_t> first_dn(n), first_crl(n);
        // PEM of the new certificates comes back encoded by the GPU (SURVEY §8(f)-3); room for "all new"
        const uint64_t der_bytes = n ? offsets[n] - offsets[0] : 0;
        std::vector<uint8_t> pem(der_bytes / 3 * 4 + der_bytes / 48 + 64 * n + 256);
        std::vector<uint64_t> pem_off(n + 1);
        ctmr_out out{status.data(), nullptr, exp_hour.data(), soff.data(), slen.data(), unknown.data(), first.data(),
                     noff.data(), nlen.data(), coff.data(), clen.data(), first_dn.data(), first_crl.data(),
                     pem.data(), pem.size(), pem_off.data()};
        int rc = group_ ? ctmr_group_process_batch(group_, blob, offsets, n, issuer_blob, issuer_offsets, n_issuers, issuer_idx, now_unix_ns, &out)
                        : ctmr_process_batch(ctx_, blob, offsets, n, issuer_blob, issuer_offsets, n_issuers, issuer_idx, now_unix_ns, &out);
        if (rc != CTMR_OK)  // like a Redis outage: the caller stops
            return std::string("ctmr_process_batch: ") + (group_ ? ctmr_group_last_error(group_) : ctmr_last_error(ctx_));
        std::vector<uint32_t> dense(n_issuers);
        if (n_issuers) {
            rc = ctmr_register_issuers(ctx_, issuer_blob, issuer_offsets, n_issuers, dense.data());  // memoised: no GPU work
            if (rc != CTMR_OK) return std::string("ctmr_register_issuers: ") + ctmr_last_error(ctx_);
        }
        std::set<std::string> dirty_days;
        BatchStats st;
        st.entries = n;
        // A cache with the pipelined extension gets this batch's SADDs and EXPIREATs in one round trip each
        BatchRemoteCache* pipelined = dynamic_cast<BatchRemoteCache*>(cache_);
        if (pipelined) {
            std::vector<BatchRemoteCache::Insert> inserts;
            std::vector<BatchRemoteCache::Expire> expires;
            for (uint64_t i = 0; i < n; ++i) {
                if (status[i] != CTMR_ST_OK || !unknown[i]) continue;
                uint8_t dig[32];
                ctmr_issuer_digest(ctx_, dense[issuer_idx[i]], dig);
                KnownCertificates* kc = GetKnownCertificates(ExpDate{exp_hour[i]}, Issuer::FromDigest(dig));
                inserts.push_back({kc->serialId(), Serial::FromBytes(blob + offsets[i] + soff[i], slen[i]).BinaryString()});
                if (!kc->ExpirySet()) {  // knowncertificates.go:44-47: once per KnownCertificates object
                    expires.push_back({kc->serialId(), kc->ExpireTimeUnix()});
                    kc->MarkExpirySet();
                }
            }
            if (!inserts.empty()) {
                auto r = pipelined->SetInsertBatch(inserts);
                if (!ok(r.second)) return r.second;
                st.cache_inserts += inserts.size();
            }
            if (!expires.empty()) {
                Error e = pipelined->ExpireAtBatch(expires);
                if (!ok(e)) return e;
            }
        }
        for (uint64_t i = 0; i < n; ++i) {
            st.status[status[i] < CTMR_ST__COUNT ? status[i] : CTMR_ST_PARSE_ERR]++;
            if (status[i] != CTMR_ST_OK) continue;  // the reference logs and continues (ct-fetch.go:206-232)
            ++st.stored;
            const ExpDate expDate{exp_hour[i]};
            uint8_t dig[32];
            ctmr_issuer_digest(ctx_, dense[issuer_idx[i]], dig);
            const Issuer issuer = Issuer::FromDigest(dig);
            if (unknown[i]) {
                ++st.unknown;
                const Serial serial = Serial::FromBytes(blob + offsets[i] + soff[i], slen[i]);
                if (!pipelined) {
                    KnownCertificates* kc = GetKnownCertificates(expDate, issuer);
                    auto r = kc->WasUnknown(serial);  // SADD only for entries the GPU found new
                    ++st.cache_inserts;
                    if (!ok(r.second)) return r.second;
                }
                // IssuerMetadata.Accumulate: the GPU says which new certificates carry a Name / CRL-DP value not
                // seen before for this issuer; only those are formatted / parsed (its own memo stays authoritative)
                IssuerMetadata* im = GetIssuerMetadata(issuer);
                const uint8_t* der = blob + offsets[i];
                if (first_dn[i] || issuer_dn) {
                    ++st.dn_formats;
                    Error e = im->NoteIssuerDN(issuer_dn ? issuer_dn(i) : FormatIssuerDN(der + noff[i], nlen[i]));
                    if (!ok(e)) return e;
                }
                if (first_crl[i] || crl_dps) {
                    ++st.crl_parses;
                    for (const auto& dp : crl_dps ? crl_dps(i) : ExtractCrlUris(der + coff[i], clen[i])) {
                        Error e = im->NoteCRL(dp);
                        if (!ok(e)) return e;
                    }
                }
                im->NoteExpDate(expDate);
                if (first[i]) {  // !issuerDateSeenBefore (filesystemdatabase.go:189-195)
                    Error e = backend_->AllocateExpDateAndIssuer(expDate, issuer);
                    if (!ok(e)) return e;
                }
                Error e = backend_->StoreCertificatePEM(
                    serial, expDate, issuer,
                    std::string(reinterpret_cast<const char*>(pem.data() + pem_off[i]), (size_t)(pem_off[i + 1] - pem_off[i])));
                if (!ok(e)) return e;
                ++st.pem_writes;
            }
            dirty_days.insert(expDate.DayID());  // markDirty for every stored entry, once per distinct day per batch
        }
        for (const auto& d : dirty_days) {
            Error e = backend_->MarkDirty(d);
            if (!ok(e)) return e;
        }
        if (stats) *stats = st;
        return "";
    }

    // ---- the sets read back out of the device (include/ctmr.h, "the sets read back")
    struct DeviceSet {
        ExpDate expDate;
        Issuer issuer;
        uint8_t digest[32];
        uint64_t count;  // SetCardinality
    };
    // GetIssuerAndDatesFromCache (filesystemdatabase.go:59-100) + Count() per set, answered from HBM instead of a
    // KEYS serials::* scan; [min_hour, max_hour] is ListExpirationDates(notBefore)'s range.  Canonical order.
    std::pair<std::vector<DeviceSet>, Error> GetIssuerAndDatesFromDevice(int64_t min_hour = INT64_MIN, int64_t max_hour = INT64_MAX) {
        std::vector<DeviceSet> out;
        uint64_t n = 0;
        int rc = group_ ? ctmr_group_list_sets(group_, min_hour, max_hour, nullptr, 0, &n) : ctmr_list_sets(ctx_, min_hour, max_hour, nullptr, 0, &n);
        std::vector<ctmr_set_info> raw(n);
        if (rc == CTMR_OK && n)
            rc = group_ ? ctmr_group_list_sets(group_, min_hour, max_hour, raw.data(), n, &n) : ctmr_list_sets(ctx_, min_hour, max_hour, raw.data(), n, &n);
        if (rc != CTMR_OK) return {out, lastError("ctmr_list_sets")};
        for (uint64_t j = 0; j < n; ++j) {
            DeviceSet d{ExpDate{raw[j].exp_hour}, Issuer::FromDigest(raw[j].issuer_digest), {}, raw[j].count};
            std::memcpy(d.digest, raw[j].issuer_digest, 32);
            out.push_back(d);
        }
        return {out, ""};
    }

    // KnownCertificates.Known() (knowncertificates.go:65-96) of one set, from HBM: its serials in first-seen order
    std::pair<std::vector<Serial>, Error> KnownFromDevice(const ExpDate& expDate, const uint8_t issuer_digest[32]) {
        std::vector<Serial> out;
        uint64_t n = 0;
        auto call = [&](uint8_t* ser, uint64_t ser_cap, uint64_t* off, uint64_t* first, uint64_t cap) {
            return group_ ? ctmr_group_set_members(group_, expDate.hour, issuer_digest, ser, ser_cap, off, first, cap, &n)
                          : ctmr_set_members(ctx_, expDate.hour, issuer_digest, ser, ser_cap, off, first, cap, &n);
        };
        int rc = call(nullptr, 0, nullptr, nullptr, 0);
        if (rc != CTMR_OK) return {out, lastError("ctmr_set_members")};
        if (!n) return {out, ""};
        std::vector<uint8_t> blob(n * CTMR_MAX_SERIAL);
        std::vector<uint64_t> off(n + 1), first(n);
        rc = call(blob.data(), blob.size(), off.data(), first.data(), n);
        if (rc != CTMR_OK) return {out, lastError("ctmr_set_members")};
        for (uint64_t k = 0; k < n; ++k) out.push_back(Serial::FromBytes(blob.data() + off[k], off[k + 1] - off[k]));
        return {out, ""};
    }
    std::pair<std::vector<Serial>, Error> KnownFromDevice(const ExpDate& expDate, const Issuer& issuer) {
        uint8_t d[32];
        if (!Base64URLDecode32(issuer.ID(), d)) return {{}, "KnownFromDevice: issuer id is not a base64url SHA-256 digest"};
        return KnownFromDevice(expDate, d);
    }

    // A lost or never-written Redis rebuilt from the device: one SetInsert per member of every live set and one
    // ExpireAt(expDate) per set (knowncertificates.go:44-47), in canonical order.  A cache with the pipelined
    // extension gets all of them in one SetInsertBatch and one ExpireAtBatch.  The IssuerMetadata string sets
    // ("issuer::" / "crl::") are process memory of the device path and are not part of the export.
    Error RebuildRemoteCache(RemoteCache* target) {
        ctmr_set_export x{};
        int rc = exportSets(&x);  // NULL arrays: the sizes
        if (rc != CTMR_OK) return lastError("ctmr_export_sets");
        std::vector<ctmr_set_info> sets(x.n_sets + 1);
        std::vector<uint8_t> serials(x.serial_bytes + 1);
        std::vector<uint64_t> off(x.n_members + 1), first(x.n_members + 1);
        x.sets = sets.data(); x.sets_cap = x.n_sets;
        x.serials = serials.data(); x.serials_cap = x.serial_bytes;
        x.serial_off = off.data(); x.first_index = first.data(); x.members_cap = x.n_members;
        rc = exportSets(&x);
        if (rc != CTMR_OK) return lastError("ctmr_export_sets");
        BatchRemoteCache* pipelined = dynamic_cast<BatchRemoteCache*>(target);
        std::vector<BatchRemoteCache::Insert> inserts;
        std::vector<BatchRemoteCache::Expire> expires;
        for (uint64_t j = 0; j < x.n_sets; ++j) {
            const ExpDate e{sets[j].exp_hour};
            KnownCertificates kc(e, Issuer::FromDigest(sets[j].issuer_digest), target);
            const std::string key = kc.serialId();
            for (uint64_t k = sets[j].member_off; k < sets[j].member_off + sets[j].count; ++k) {
                std::string member(reinterpret_cast<const char*>(serials.data() + off[k]), (size_t)(off[k + 1] - off[k]));
                if (pipelined) {
                    inserts.push_back({key, std::move(member)});
                } else {
                    Error err = target->SetInsert(key, member).second;
                    if (!ok(err)) return err;
                }
            }
            if (pipelined) {
                expires.push_back({key, e.ExpireTimeUnix()});
            } else {
                Error err = target->ExpireAt(key, e.ExpireTimeUnix());
                if (!ok(err)) return err;
            }
        }
        if (pipelined && !inserts.empty()) {
            Error err = pipelined->SetInsertBatch(inserts).second;
            if (!ok(err)) return err;
        }
        if (pipelined && !expires.empty()) return pipelined->ExpireAtBatch(expires);
        return "";
    }

  private:
    int exportSets(ctmr_set_export* x) { return group_ ? ctmr_group_export_sets(group_, x) : ctmr_export_sets(ctx_, x); }
    Error lastError(const char* what) const {
        return std::string(what) + ": " + (group_ ? ctmr_group_last_error(group_) : ctmr_last_error(ctx_));
    }
    // Issuer.ID() back to its digest: base64.URLEncoding of 32 bytes (44 characters, one '=')
    static bool Base64URLDecode32(const std::string& id, uint8_t out[32]) {
        if (id.size() != 44) return false;
        uint32_t acc = 0;
        int bits = 0, n = 0;
        for (char c : id) {
            int v;
            if (c >= 'A' && c <= 'Z') v = c - 'A';
            else if (c >= 'a' && c <= 'z') v = c - 'a' + 26;
            else if (c >= '0' && c <= '9') v = c - '0' + 52;
            else if (c == '-') v = 62;
            else if (c == '_') v = 63;
            else if (c == '=') break;
            else return false;
            acc = (acc << 6) | (uint32_t)v;
            bits += 6;
            if (bits >= 8) {
                bits -= 8;
                if (n == 32) return false;
                out[n++] = (uint8_t)(acc >> bits);
            }
        }
        return n == 32;
    }

    ctmr_ctx* ctx_;
    ctmr_group* group_ = nullptr;
    RemoteCache* cache_;
    StorageBackend* backend_;
    std::map<std::string, std::unique_ptr<KnownCertificates>> known_;
    std::map<std::string, std::unique_ptr<IssuerMetadata>> meta_;
};

}  // namespace ctmr_host
