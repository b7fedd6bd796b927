// Host-side view of the staged index: key directories (which lists exist, how long they are) and
// the layout of the HBM posting store.  List *contents* live only on the device after staging.
//
// HBM layout (DESIGN.md §2):
//   pool      u32[]   every posting list back to back; a list is either `card` ascending docids (sparse)
//                     or, when card > n_docs/32, a dense bitmap of n_words64 little-endian u64 words
//   lists     ListRef[]  (offset into pool, cardinality, dense flag) indexed by list id
//   pair_keys u64[]   sorted packed keys prox<<42 | w1<<21 | w2 of word_pair_proximity_docids; the i-th key's
//                     list id is pair_list_base + i (so a prefix range of w2 is a contiguous run of lists)
//   dict      bytes + u32 offsets of the sorted dictionary (word id = rank)
//   base_ub   u64[]   documents_ids as a dense bitmap (the initial universe)
#pragma once
#include <cstdint>
#include <cstring>
#include <map>
#include <string>
#include <unordered_map>
#include <vector>

namespace b200 {

struct ListRef {
    uint64_t off;    // u32 index into the pool (even when dense)
    uint32_t card;   // number of docids
    uint32_t dense;  // 1: bitmap words at off
};

struct RawDb {
    uint64_t n = 0;
    std::vector<uint8_t> keys, vals;
    std::vector<uint64_t> koff, voff;
};

struct Settings {
    uint32_t n_fields = 1;
    std::vector<uint16_t> weights{0};
    std::vector<int> criteria{0, 1, 2, 4, 6, 5, 7};
    bool authorize_typos = true;
    uint32_t one_typo = 5, two_typos = 9;
    bool prefix_search = true;
    std::unordered_map<std::string, int> exact_words;
    std::map<std::vector<std::string>, std::vector<std::vector<std::string>>> synonyms;  // pre-tokenised (index `synonyms` db)
    uint16_t max_weight() const {
        uint16_t m = 0;
        for (auto w : weights) m = m > w ? m : w;
        return m;
    }
};

constexpr uint32_t NO_LIST = 0xffffffffu;

struct HostIndex {
    // dictionary
    std::vector<uint8_t> dict_bytes;
    std::vector<uint64_t> dict_off;
    uint64_t n_words = 0;
    // dict_pair_start[b0 << 8 | b1] = first word id whose first two bytes are >= (b0, b1), 65537 entries (the last = n_words).
    // The dictionary is sorted, so the words with first byte c are [start[c << 8], start[(c + 1) << 8]) and those with first
    // bytes (b0, c) are [start[b0 << 8 | c], start[(b0 << 8 | c) + 1]).  A one-byte word counts as second byte 0.
    std::vector<uint32_t> dict_pair_start;
    // universe
    uint32_t n_docs = 0;    // max docid + 1
    uint32_t n_words64 = 0; // ceil(n_docs / 64)
    std::vector<uint64_t> base_ub;
    uint64_t n_documents = 0;
    // posting store
    std::vector<ListRef> lists;
    std::vector<uint32_t> pool;  // host staging copy, released after upload
    // directories
    std::vector<uint32_t> wd_list, ewd_list;  // per word id
    std::vector<uint32_t> wf_off, wf_list, wp_off, wp_list;  // CSR per word id
    std::vector<uint16_t> wf_fid, wp_pos;
    std::vector<std::string> prefixes;  // sorted
    std::vector<uint32_t> pd_list, epd_list;
    std::vector<uint32_t> pf_off, pf_list, pp_off, pp_list;
    std::vector<uint16_t> pf_fid, pp_pos;
    std::vector<uint64_t> pair_keys;
    uint32_t pair_list_base = 0;
    std::map<uint32_t, uint32_t> fwc_list;  // fid<<8|count -> list
    // list id of key i of database db = db_first[db] + i (keys in LMDB order); db_keys[db] = number of staged keys.
    // (word_pair_proximity keys naming unknown words are dropped at staging: for that db the mapping only holds when none was.)
    uint32_t db_first[10] = {0}, db_keys[10] = {0};

    Settings settings;

    const uint8_t *word_ptr(uint64_t i) const { return dict_bytes.data() + dict_off[i]; }
    size_t word_len(uint64_t i) const { return dict_off[i + 1] - dict_off[i]; }
    std::string word(uint64_t i) const { return std::string((const char *)word_ptr(i), word_len(i)); }
    int cmp_word(uint64_t i, const uint8_t *k, size_t kn) const {
        size_t n_i = word_len(i);
        int c = memcmp(word_ptr(i), k, n_i < kn ? n_i : kn);
        if (c) return c;
        return n_i < kn ? -1 : (n_i > kn ? 1 : 0);
    }
    uint64_t lower_bound(const uint8_t *k, size_t kn) const {
        uint64_t lo = 0, hi = n_words;
        while (lo < hi) {
            uint64_t mid = (lo + hi) / 2;
            if (cmp_word(mid, k, kn) < 0)
                lo = mid + 1;
            else
                hi = mid;
        }
        return lo;
    }
    // rank of a word, or -1
    int64_t find_word(const uint8_t *k, size_t kn) const {
        uint64_t i = lower_bound(k, kn);
        return (i < n_words && cmp_word(i, k, kn) == 0) ? (int64_t)i : -1;
    }
    int64_t find_word(const std::string &s) const { return find_word((const uint8_t *)s.data(), s.size()); }
    // [lo, hi) of dictionary words having `p` as a prefix
    void prefix_range(const std::string &p, uint64_t &lo, uint64_t &hi) const {
        lo = lower_bound((const uint8_t *)p.data(), p.size());
        uint64_t a = lo, b = n_words;
        while (a < b) {
            uint64_t mid = (a + b) / 2;
            bool has = word_len(mid) >= p.size() && memcmp(word_ptr(mid), p.data(), p.size()) == 0;
            if (has)
                a = mid + 1;
            else
                b = mid;
        }
        hi = a;
    }
    int32_t find_prefix(const std::string &p) const {
        size_t lo = 0, hi = prefixes.size();
        while (lo < hi) {
            size_t mid = (lo + hi) / 2;
            if (prefixes[mid] < p)
                lo = mid + 1;
            else
                hi = mid;
        }
        return (lo < prefixes.size() && prefixes[lo] == p) ? (int32_t)lo : -1;
    }
    static uint64_t pair_key(uint32_t prox, uint32_t w1, uint32_t w2) { return ((uint64_t)prox << 42) | ((uint64_t)w1 << 21) | w2; }
    // list id of (prox, w1, w2) or NO_LIST
    uint32_t find_pair(uint32_t prox, uint32_t w1, uint32_t w2) const {
        uint64_t k = pair_key(prox, w1, w2);
        size_t lo = 0, hi = pair_keys.size();
        while (lo < hi) {
            size_t mid = (lo + hi) / 2;
            if (pair_keys[mid] < k)
                lo = mid + 1;
            else
                hi = mid;
        }
        return (lo < pair_keys.size() && pair_keys[lo] == k) ? pair_list_base + (uint32_t)lo : NO_LIST;
    }
    uint32_t word_fid_list(uint32_t w, uint16_t fid) const {
        for (uint32_t i = wf_off[w]; i < wf_off[w + 1]; i++)
            if (wf_fid[i] == fid) return wf_list[i];
        return NO_LIST;
    }
    uint32_t word_pos_list(uint32_t w, uint16_t pos) const {
        for (uint32_t i = wp_off[w]; i < wp_off[w + 1]; i++)
            if (wp_pos[i] == pos) return wp_list[i];
        return NO_LIST;
    }
    uint32_t prefix_fid_list(uint32_t p, uint16_t fid) const {
        for (uint32_t i = pf_off[p]; i < pf_off[p + 1]; i++)
            if (pf_fid[i] == fid) return pf_list[i];
        return NO_LIST;
    }
    uint32_t prefix_pos_list(uint32_t p, uint16_t pos) const {
        for (uint32_t i = pp_off[p]; i < pp_off[p + 1]; i++)
            if (pp_pos[i] == pos) return pp_list[i];
        return NO_LIST;
    }
};

// Decode the staged LMDB-format databases into `out` (directories + pool). Throws std::runtime_error.
void build_host_index(const std::vector<uint8_t> &dict_bytes, const std::vector<uint64_t> &dict_off, const RawDb *dbs /*[10]*/,
                      const std::vector<uint8_t> &docids_cbo, HostIndex &out);

}  // namespace b200
