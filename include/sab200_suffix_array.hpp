// sab200_suffix_array.hpp -- C++ host mirror of the reference's `SuffixArray`
// (/root/reference/src/sa.rs:14-374) over the C ABI of sab200.h.
//
// The reference is a Rust crate and this image has no Rust toolchain, so the compiled-language host
// above the C ABI is C++ (header-only).  Same method names, argument meaning and error behaviour:
//   * construction asserts like saca() (src/saca.rs:10-11) -> std::length_error / std::runtime_error
//   * from_parts returns std::nullopt where the reference returns None (src/sa.rs:57-64)
//   * search_all returns a (pointer, length) view into the suffix array, SA order (src/sa.rs:203)
//   * search_lcp returns the half-open text range (src/sa.rs:207)
// Per-pattern queries go through the batched GPU entry points with a batch of one; the *_batch
// methods are the intended fast path.  No method has a CPU fallback.
#pragma once
#include <cstdint>
#include <fstream>
#include <iterator>
#include <memory>
#include <optional>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "sab200.h"

namespace sab200 {

constexpr std::size_t MAX_LENGTH = SAB200_MAX_LENGTH;  // replaces src/saca.rs:6

struct Slice {
    const std::uint32_t* data;
    std::size_t len;
    const std::uint32_t* begin() const { return data; }
    const std::uint32_t* end() const { return data + len; }
};
struct Range {
    std::size_t start, end;
};

inline void check(std::int32_t rc, const char* what) {
    if (rc != SAB200_OK) throw std::runtime_error(std::string(what) + ": " + sab200_last_error());
}

// src/saca.rs:9-15
inline void saca(const std::uint8_t* s, std::size_t n, std::vector<std::uint32_t>& sa, int ngpus = 1) {
    if (n > MAX_LENGTH) throw std::length_error("text longer than MAX_LENGTH");  // :10
    if (sa.size() != n + 1) throw std::length_error("sa.len() != s.len() + 1");   // :11
    check(sab200_saca(s, n, sa.data(), ngpus), "sab200_saca");
}

// Burrows-Wheeler transform (sab200.h): the n bytes of the last column without the row of '$', and that row's index
// (the primary index).  bwt("banana") = ("annbaa", 4).
inline std::pair<std::vector<std::uint8_t>, std::uint64_t> bwt(const std::uint8_t* s, std::size_t n) {
    if (n > MAX_LENGTH) throw std::length_error("text longer than MAX_LENGTH");
    std::pair<std::vector<std::uint8_t>, std::uint64_t> r(std::vector<std::uint8_t>(n), 0);
    check(sab200_bwt(s, n, r.first.data(), &r.second), "sab200_bwt");
    return r;
}

// The text whose transform is (u, primary); std::invalid_argument when there is none or the primary index is out of
// range.
inline std::vector<std::uint8_t> inverse_bwt(const std::uint8_t* u, std::size_t n, std::uint64_t primary) {
    if (n > MAX_LENGTH) throw std::length_error("transform longer than MAX_LENGTH");
    std::vector<std::uint8_t> s(n);
    const std::int32_t rc = sab200_inverse_bwt(u, n, primary, s.data());
    if (rc == SAB200_ERR_ARGS) throw std::invalid_argument(std::string("sab200_inverse_bwt: ") + sab200_last_error());
    check(rc, "sab200_inverse_bwt");
    return s;
}

// Greedy LZ77 factorization (sab200.h): the z factors (pos[t], len[t]); len = 0 is a literal with pos = the byte,
// otherwise a copy of len bytes from the earlier position pos.  lz77("banana") = (b,0) (a,0) (n,0) (1,3).
inline std::pair<std::vector<std::uint32_t>, std::vector<std::uint32_t>> lz77(const std::uint8_t* s, std::size_t n) {
    if (n > MAX_LENGTH) throw std::length_error("text longer than MAX_LENGTH");
    // cap = n suffices; uninitialised, so only the pages of the z factors are ever touched
    std::unique_ptr<std::uint32_t[]> pos(new std::uint32_t[n ? n : 1]), len(new std::uint32_t[n ? n : 1]);
    std::uint64_t z = 0;
    check(sab200_lz77(s, n, pos.get(), len.get(), n, &z), "sab200_lz77");
    return {std::vector<std::uint32_t>(pos.get(), pos.get() + z), std::vector<std::uint32_t>(len.get(), len.get() + z)};
}

// The n bytes of the parse (pos, len), greedy or not; std::invalid_argument when the factors do not parse n bytes.
inline std::vector<std::uint8_t> lz77_decode(const std::vector<std::uint32_t>& pos, const std::vector<std::uint32_t>& len,
                                             std::size_t n) {
    if (pos.size() != len.size()) throw std::invalid_argument("lz77_decode: pos and len differ in length");
    std::vector<std::uint8_t> s(n);
    const std::int32_t rc = sab200_lz77_decode(pos.data(), len.data(), pos.size(), n, s.data());
    if (rc == SAB200_ERR_ARGS) throw std::invalid_argument(std::string("sab200_lz77_decode: ") + sab200_last_error());
    check(rc, "sab200_lz77_decode");
    return s;
}

class SuffixArray {
  public:
    // src/sa.rs:23-27
    SuffixArray(const std::uint8_t* s, std::size_t n) : s_(s), n_(n), sa_(n + 1, 0) { saca(s_, n_, sa_); }
    static SuffixArray make(const std::uint8_t* s, std::size_t n) { return SuffixArray(s, n); }
    ~SuffixArray() { drop_index(); }
    SuffixArray(SuffixArray&& o) noexcept
        : s_(o.s_), n_(o.n_), sa_(std::move(o.sa_)), bkt_(std::move(o.bkt_)), has_bkt_(o.has_bkt_), ix_(o.ix_) {
        o.ix_ = nullptr;
    }
    SuffixArray(const SuffixArray& o) : s_(o.s_), n_(o.n_), sa_(o.sa_), bkt_(o.bkt_), has_bkt_(o.has_bkt_) {}  // #[derive(Clone)]
    SuffixArray& operator=(const SuffixArray&) = delete;

    // src/sa.rs:30-33, literally: the stored text and the bucket table are NOT replaced (SURVEY.md Q4)
    void set(const std::uint8_t* s, std::size_t n) {
        sa_.resize(n + 1, 0);
        saca(s, n, sa_);
        drop_index();
    }
    void fit() { sa_.shrink_to_fit(); }                 // src/sa.rs:36-38
    std::size_t len() const { return n_; }              // src/sa.rs:41-43
    bool is_empty() const { return n_ == 0; }           // src/sa.rs:46-48
    std::pair<const std::uint8_t*, std::vector<std::uint32_t>> into_parts() && {  // src/sa.rs:51-53
        drop_index();
        return {s_, std::move(sa_)};
    }
    // src/sa.rs:57-64
    static std::optional<SuffixArray> from_parts(const std::uint8_t* s, std::size_t n, std::vector<std::uint32_t> sa) {
        const std::int32_t rc = sab200_check(s, n, sa.data(), sa.size());
        if (rc < 0) check(rc, "sab200_check");
        if (rc != 1) return std::nullopt;
        return SuffixArray(s, n, std::move(sa));
    }
    // src/sa.rs:68-70
    static SuffixArray unchecked_from_parts(const std::uint8_t* s, std::size_t n, std::vector<std::uint32_t> sa) {
        return SuffixArray(s, n, std::move(sa));
    }
    // ---- pack serialisation (feature "pack", src/sa.rs:256-361); io errors -> std::runtime_error
    std::vector<std::uint8_t> dump_bytes() const {  // src/sa.rs:275-278
        std::vector<std::uint8_t> out(sab200_pack_bound(sa_.size()));
        std::uint64_t len = 0;
        check(sab200_pack(sa_.data(), sa_.size(), out.data(), out.size(), &len), "sab200_pack");
        out.resize(len);
        return out;
    }
    void dump(std::ostream& file) const {  // src/sa.rs:257-260
        const auto b = dump_bytes();
        file.write(reinterpret_cast<const char*>(b.data()), (std::streamsize)b.size());
        if (!file) throw std::runtime_error("dump: write failed");
    }
    void dump_file(const std::string& name) const {  // src/sa.rs:264-271
        std::ofstream f(name, std::ios::binary | std::ios::trunc);
        if (!f) throw std::runtime_error("dump_file: cannot create " + name);
        dump(f);
    }
    // src/sa.rs:338-346
    static SuffixArray unchecked_load_bytes(const std::uint8_t* s, std::size_t n, const std::uint8_t* bytes,
                                            std::size_t nbytes) {
        if (nbytes < 16) throw std::runtime_error("load: truncated packed suffix array");
        const std::uint32_t length = (std::uint32_t)bytes[4] | (std::uint32_t)bytes[5] << 8 |
                                     (std::uint32_t)bytes[6] << 16 | (std::uint32_t)bytes[7] << 24;
        std::vector<std::uint32_t> sa(length ? length : 1);
        std::uint64_t len = 0;
        check(sab200_unpack(bytes, nbytes, sa.data(), sa.size(), &len), "sab200_unpack");
        sa.resize(len);
        return SuffixArray(s, n, std::move(sa));
    }
    // src/sa.rs:349-361: InvalidData("inconsistent suffix array") -> std::runtime_error
    static SuffixArray load_bytes(const std::uint8_t* s, std::size_t n, const std::uint8_t* bytes, std::size_t nbytes) {
        SuffixArray t = unchecked_load_bytes(s, n, bytes, nbytes);
        auto ok = from_parts(s, n, std::move(t.sa_));
        if (!ok) throw std::runtime_error("inconsistent suffix array");
        return std::move(*ok);
    }
    static SuffixArray load(const std::uint8_t* s, std::size_t n, std::istream& file) {  // src/sa.rs:293-305
        const std::vector<std::uint8_t> b((std::istreambuf_iterator<char>(file)), std::istreambuf_iterator<char>());
        return load_bytes(s, n, b.data(), b.size());
    }
    static SuffixArray unchecked_load(const std::uint8_t* s, std::size_t n, std::istream& file) {  // src/sa.rs:281-290
        const std::vector<std::uint8_t> b((std::istreambuf_iterator<char>(file)), std::istreambuf_iterator<char>());
        return unchecked_load_bytes(s, n, b.data(), b.size());
    }
    static SuffixArray load_file(const std::uint8_t* s, std::size_t n, const std::string& name) {  // src/sa.rs:323-335
        std::ifstream f(name, std::ios::binary);
        if (!f) throw std::runtime_error("load_file: cannot open " + name);
        return load(s, n, f);
    }
    static SuffixArray unchecked_load_file(const std::uint8_t* s, std::size_t n, const std::string& name) {
        std::ifstream f(name, std::ios::binary);
        if (!f) throw std::runtime_error("load_file: cannot open " + name);
        return unchecked_load(s, n, f);
    }

    // src/sa.rs:89-119
    void enable_buckets() {
        if (has_bkt_) return;
        bkt_.assign(SAB200_BKT_LEN, 0);
        check(sab200_enable_buckets(s_, n_, bkt_.data()), "sab200_enable_buckets");
        has_bkt_ = true;
        drop_index();
    }
    void use_gpus(int ngpus) {
        if (ngpus != ngpus_) {
            drop_index();
            ngpus_ = ngpus;
        }
    }

    // ---- batched queries: pattern q is pats[offs[q] .. offs[q+1])
    void search_all_batch(const std::uint8_t* pats, const std::uint64_t* offs, std::size_t np, std::uint32_t* lo,
                          std::uint32_t* hi) {
        check(sab200_search_all_batch(index(), pats, offs, np, lo, hi), "sab200_search_all_batch");
    }
    void contains_batch(const std::uint8_t* pats, const std::uint64_t* offs, std::size_t np, std::uint8_t* out) {
        check(sab200_contains_batch(index(), pats, offs, np, out), "sab200_contains_batch");
    }
    void search_lcp_batch(const std::uint8_t* pats, const std::uint64_t* offs, std::size_t np, std::uint32_t* start,
                          std::uint32_t* end) {
        check(sab200_search_lcp_batch(index(), pats, offs, np, start, end), "sab200_search_lcp_batch");
    }

    // ---- matching statistics (include/sab200.h): len / lo / hi receive offs[nq] entries each, indexed by the absolute
    // offset in qs; a suffix array that is not the text's throws std::invalid_argument
    void matching_statistics_batch(const std::uint8_t* qs, const std::uint64_t* offs, std::size_t nq, std::uint32_t* len,
                                   std::uint32_t* lo, std::uint32_t* hi) {
        const std::int32_t rc = sab200_matching_statistics_batch(index(), qs, offs, nq, len, lo, hi);
        if (rc == SAB200_ERR_ARGS) throw std::invalid_argument(std::string("sab200_matching_statistics_batch: ") + sab200_last_error());
        check(rc, "sab200_matching_statistics_batch");
    }
    struct MatchingStatistics {
        std::vector<std::uint32_t> len, lo, hi;
    };
    MatchingStatistics matching_statistics(const std::uint8_t* q, std::size_t m) {
        const std::uint64_t offs[2] = {0, m};
        MatchingStatistics r{std::vector<std::uint32_t>(m), std::vector<std::uint32_t>(m), std::vector<std::uint32_t>(m)};
        matching_statistics_batch(q, offs, 1, r.len.data(), r.lo.data(), r.hi.data());
        return r;
    }

    // ---- per-pattern queries (src/sa.rs:164-253)
    bool contains(const std::uint8_t* pat, std::size_t m) {
        const std::uint64_t offs[2] = {0, m};
        std::uint8_t out = 0;
        contains_batch(pat, offs, 1, &out);
        return out != 0;
    }
    Slice search_all(const std::uint8_t* pat, std::size_t m) {
        const std::uint64_t offs[2] = {0, m};
        std::uint32_t lo = 0, hi = 0;
        search_all_batch(pat, offs, 1, &lo, &hi);
        return Slice{sa_.data() + lo, (std::size_t)(hi - lo)};
    }
    Range search_lcp(const std::uint8_t* pat, std::size_t m) {
        const std::uint64_t offs[2] = {0, m};
        std::uint32_t st = 0, en = 0;
        search_lcp_batch(pat, offs, 1, &st, &en);
        return Range{st, en};
    }

    // new() + enable_buckets() (src/sa.rs:23-27, 89-119) in one library call (SURVEY.md 8f N2)
    static SuffixArray with_buckets(const std::uint8_t* s, std::size_t n, int ngpus = 1) {
        std::vector<std::uint32_t> sa(n + 1, 0u);
        std::vector<std::uint32_t> bkt(SAB200_BKT_LEN, 0u);
        if (sab200_saca_buckets(s, n, sa.data(), bkt.data(), ngpus) != 0)
            throw std::runtime_error(std::string("sab200_saca_buckets: ") + sab200_last_error());
        SuffixArray r(s, n, std::move(sa));
        r.bkt_ = std::move(bkt);
        r.has_bkt_ = true;
        return r;
    }

    // LCP array of the suffix array (no reference counterpart; README.md:18-23): lcp[0] = 0, lcp[j] = common prefix
    // of the suffixes sa[j-1] and sa[j]
    std::vector<std::uint32_t> lcp_array() const {
        std::vector<std::uint32_t> out(sa_.size());
        if (sab200_lcp_array(s_, n_, sa_.data(), sa_.size(), out.data()) != 0)
            throw std::runtime_error(std::string("sab200_lcp_array: ") + sab200_last_error());
        return out;
    }

    const std::vector<std::uint32_t>& sa() const { return sa_; }   // From<SuffixArray> for Vec<u32>, src/sa.rs:364-368
    const std::uint8_t* as_ref() const { return s_; }              // AsRef<[u8]>, src/sa.rs:370-374
    const std::vector<std::uint32_t>* buckets() const { return has_bkt_ ? &bkt_ : nullptr; }

  private:
    SuffixArray(const std::uint8_t* s, std::size_t n, std::vector<std::uint32_t> sa) : s_(s), n_(n), sa_(std::move(sa)) {}
    sab200_index* index() {
        if (!ix_) {
            ix_ = sab200_index_create(s_, n_, sa_.data(), sa_.size(), has_bkt_ ? bkt_.data() : nullptr, ngpus_);
            if (!ix_) throw std::runtime_error(std::string("sab200_index_create: ") + sab200_last_error());
        }
        return ix_;
    }
    void drop_index() {
        if (ix_) sab200_index_destroy(ix_);
        ix_ = nullptr;
    }
    const std::uint8_t* s_;
    std::size_t n_;
    std::vector<std::uint32_t> sa_;
    std::vector<std::uint32_t> bkt_;
    bool has_bkt_ = false;
    sab200_index* ix_ = nullptr;
    int ngpus_ = 1;
};

}  // namespace sab200
