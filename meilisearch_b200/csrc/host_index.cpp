// Staging: decode the LMDB-format databases (keys per heed_codec/*, values per
// CboRoaringBitmapCodec, crates/milli/src/heed_codec/roaring_bitmap/cbo_roaring_bitmap_codec.rs:15-85)
// into the HBM posting-store layout described in host_index.h.
#include "host_index.h"

#include <algorithm>
#include <stdexcept>
#include <thread>

namespace b200 {

namespace {

// Append the docids of one CBO value to `out` (ascending). Returns cardinality.
uint32_t cbo_decode_append(const uint8_t *p, size_t n, std::vector<uint32_t> &out) {
    size_t start = out.size();
    if (n <= 28) {  // raw native-endian u32s (<= THRESHOLD ints)
        for (size_t i = 0; i + 4 <= n; i += 4) {
            uint32_t v;
            memcpy(&v, p + i, 4);
            out.push_back(v);
        }
        return (uint32_t)(out.size() - start);
    }
    uint32_t cookie, nc;
    memcpy(&cookie, p, 4);
    memcpy(&nc, p + 4, 4);
    if (cookie != 12346) throw std::runtime_error("stage: roaring value with run containers / unknown cookie");
    // every length comes from the value itself: check it against the bytes we were given before reading
    if (nc == 0 || nc > 65536 || 8 + 8 * (size_t)nc > n) throw std::runtime_error("stage: malformed roaring value (container count)");
    const uint8_t *desc = p + 8;
    const uint8_t *data = p + 8 + 8 * (size_t)nc;
    const uint8_t *const end = p + n;
    for (uint32_t c = 0; c < nc; c++) {
        uint16_t key, cm1;
        memcpy(&key, desc + 4 * c, 2);
        memcpy(&cm1, desc + 4 * c + 2, 2);
        uint32_t card = (uint32_t)cm1 + 1, hi = (uint32_t)key << 16;
        if ((size_t)(end - data) < (card <= 4096 ? 2 * (size_t)card : (size_t)8192)) throw std::runtime_error("stage: malformed roaring value (truncated container)");
        if (card <= 4096) {
            for (uint32_t i = 0; i < card; i++) {
                uint16_t lo;
                memcpy(&lo, data + 2 * i, 2);
                out.push_back(hi | lo);
            }
            data += 2 * (size_t)card;
        } else {
            for (uint32_t w = 0; w < 1024; w++) {
                uint64_t bits;
                memcpy(&bits, data + 8 * w, 8);
                while (bits) {
                    out.push_back(hi | (w * 64 + (uint32_t)__builtin_ctzll(bits)));
                    bits &= bits - 1;
                }
            }
            data += 8192;
        }
    }
    return (uint32_t)(out.size() - start);
}

struct Builder {
    HostIndex &ix;
    const RawDb *dbs_base = nullptr;
    explicit Builder(HostIndex &i) : ix(i) {}
    // decode values [k0,k1) of a db in parallel, then append to the pool in key order; returns first list id
    uint32_t add_lists(const RawDb &db, const std::vector<uint8_t> &keep /* per key: 1 = stage */) {
        uint64_t n = db.n;
        if (dbs_base && &db >= dbs_base && &db < dbs_base + 10) {
            ix.db_first[&db - dbs_base] = (uint32_t)ix.lists.size();
            ix.db_keys[&db - dbs_base] = (uint32_t)n;
        }
        unsigned nt = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
        std::vector<std::vector<uint32_t>> parts(nt);
        std::vector<std::vector<uint32_t>> cards(nt);
        std::vector<std::thread> th;
        std::vector<std::string> errs(nt);
        for (unsigned t = 0; t < nt; t++) {
            th.emplace_back([&, t]() {
                uint64_t a = n * t / nt, b = n * (t + 1) / nt;
                try {
                    for (uint64_t i = a; i < b; i++) {
                        if (!keep.empty() && !keep[i]) {
                            cards[t].push_back(0xffffffffu);
                            continue;
                        }
                        uint32_t c = cbo_decode_append(db.vals.data() + db.voff[i], db.voff[i + 1] - db.voff[i], parts[t]);
                        cards[t].push_back(c);
                    }
                } catch (const std::exception &e) {
                    errs[t] = e.what();
                }
            });
        }
        for (auto &x : th) x.join();
        for (auto &e : errs)
            if (!e.empty()) throw std::runtime_error(e);
        uint32_t first = (uint32_t)ix.lists.size();
        // A list is stored as a dense bitmap over the docid space when card > n_docs / 128 (B200_DENSE_DIV): a bitmap costs
        // n_docs / 8 bytes, i.e. at most 4x the sorted-docid form at that density, and turns the scatter of the list into a coalesced
        // gather by universe row instead of one random row lookup per docid (DESIGN.md §2).
        uint32_t dense_div = 128;
        if (const char *env = getenv("B200_DENSE_DIV")) dense_div = (uint32_t)std::max(8, atoi(env));
        uint32_t dense_min = ix.n_docs / dense_div;
        for (unsigned t = 0; t < nt; t++) {
            size_t at = 0;
            for (uint32_t c : cards[t]) {
                if (c == 0xffffffffu) {
                    ix.lists.push_back(ListRef{0, 0, 0});
                    continue;
                }
                const uint32_t *src = parts[t].data() + at;
                at += c;
                if (ix.pool.size() & 1) ix.pool.push_back(0);  // keep every list 8-byte aligned
                ListRef r{ix.pool.size(), c, 0};
                if (c > dense_min && c > 64) {
                    r.dense = 1;
                    size_t base = ix.pool.size();
                    ix.pool.resize(base + 2 * (size_t)ix.n_words64, 0);
                    uint64_t *words = reinterpret_cast<uint64_t *>(ix.pool.data() + base);
                    for (uint32_t k = 0; k < c; k++) {
                        uint32_t d = src[k];
                        if (d < ix.n_docs) words[d >> 6] |= 1ull << (d & 63);
                    }
                } else {
                    ix.pool.insert(ix.pool.end(), src, src + c);
                }
                ix.lists.push_back(r);
            }
            std::vector<uint32_t>().swap(parts[t]);
        }
        return first;
    }
};

}  // namespace

void build_host_index(const std::vector<uint8_t> &dict_bytes, const std::vector<uint64_t> &dict_off, const RawDb *dbs,
                      const std::vector<uint8_t> &docids_cbo, HostIndex &ix) {
    ix.dict_bytes = dict_bytes;
    ix.dict_off = dict_off;
    ix.n_words = dict_off.empty() ? 0 : dict_off.size() - 1;
    if (ix.n_words >= (1u << 21)) throw std::runtime_error("stage: dictionary larger than 2^21 words (packed pair keys)");
    // first word id per leading byte pair (the term derivation schedule's word ranges)
    ix.dict_pair_start.assign(65537, 0);
    for (uint64_t i = 0, prev = 0; i < ix.n_words; i++) {
        const size_t n = ix.word_len(i);
        const uint32_t key = n == 0 ? 0u : ((uint32_t)ix.word_ptr(i)[0] << 8) | (n > 1 ? ix.word_ptr(i)[1] : 0u);
        if (key < prev) throw std::runtime_error("stage: dictionary words are not in bytewise order");
        prev = key;
        ix.dict_pair_start[key + 1]++;
    }
    for (uint32_t k = 0; k < 65536; k++) ix.dict_pair_start[k + 1] += ix.dict_pair_start[k];
    // universe
    std::vector<uint32_t> docs;
    cbo_decode_append(docids_cbo.data(), docids_cbo.size(), docs);
    ix.n_documents = docs.size();
    ix.n_docs = docs.empty() ? 0 : docs.back() + 1;
    for (auto d : docs) ix.n_docs = std::max(ix.n_docs, d + 1);
    ix.n_words64 = (ix.n_docs + 63) / 64;
    ix.base_ub.assign(ix.n_words64, 0);
    for (auto d : docs) ix.base_ub[d >> 6] |= 1ull << (d & 63);
    ix.lists.clear();
    ix.pool.clear();
    Builder b(ix);
    b.dbs_base = dbs;
    std::vector<uint8_t> all;

    auto word_of_key = [&](const RawDb &db, uint64_t i, size_t trim) -> int64_t {
        size_t kn = db.koff[i + 1] - db.koff[i];
        if (kn < trim) return -1;
        return ix.find_word(db.keys.data() + db.koff[i], kn - trim);
    };
    // word_docids / exact_word_docids
    for (int which = 0; which < 2; which++) {
        const RawDb &db = dbs[which];
        std::vector<uint32_t> &dir = which == 0 ? ix.wd_list : ix.ewd_list;
        dir.assign(ix.n_words, NO_LIST);
        uint32_t first = b.add_lists(db, all);
        for (uint64_t i = 0; i < db.n; i++) {
            int64_t w = word_of_key(db, i, 0);
            if (w >= 0) dir[w] = first + (uint32_t)i;
        }
    }
    // word_fid / word_position: key = word \0 u16be
    auto csr_u16 = [&](const RawDb &db, std::vector<uint32_t> &off, std::vector<uint16_t> &val, std::vector<uint32_t> &lst) {
        uint32_t first = b.add_lists(db, all);
        off.assign(ix.n_words + 1, 0);
        std::vector<int64_t> wk(db.n);
        for (uint64_t i = 0; i < db.n; i++) {
            wk[i] = word_of_key(db, i, 3);
            if (wk[i] >= 0) off[wk[i] + 1]++;
        }
        for (uint64_t w = 0; w < ix.n_words; w++) off[w + 1] += off[w];
        val.assign(off[ix.n_words], 0);
        lst.assign(off[ix.n_words], NO_LIST);
        std::vector<uint32_t> cur(off.begin(), off.end() - 1);
        for (uint64_t i = 0; i < db.n; i++) {
            if (wk[i] < 0) continue;
            const uint8_t *k = db.keys.data() + db.koff[i + 1] - 2;
            uint32_t at = cur[wk[i]]++;
            val[at] = (uint16_t)((k[0] << 8) | k[1]);
            lst[at] = first + (uint32_t)i;
        }
    };
    csr_u16(dbs[6], ix.wf_off, ix.wf_fid, ix.wf_list);
    csr_u16(dbs[5], ix.wp_off, ix.wp_pos, ix.wp_list);
    // prefixes: union of the keys of the two prefix docids dbs
    {
        std::vector<std::string> ps;
        for (int which : {2, 3})
            for (uint64_t i = 0; i < dbs[which].n; i++)
                ps.emplace_back((const char *)dbs[which].keys.data() + dbs[which].koff[i], dbs[which].koff[i + 1] - dbs[which].koff[i]);
        std::sort(ps.begin(), ps.end());
        ps.erase(std::unique(ps.begin(), ps.end()), ps.end());
        ix.prefixes = ps;
        size_t np = ps.size();
        ix.pd_list.assign(np, NO_LIST);
        ix.epd_list.assign(np, NO_LIST);
        for (int which : {2, 3}) {
            const RawDb &db = dbs[which];
            uint32_t first = b.add_lists(db, all);
            for (uint64_t i = 0; i < db.n; i++) {
                std::string k((const char *)db.keys.data() + db.koff[i], db.koff[i + 1] - db.koff[i]);
                int32_t p = ix.find_prefix(k);
                if (p >= 0) (which == 2 ? ix.pd_list : ix.epd_list)[p] = first + (uint32_t)i;
            }
        }
        auto csr_p = [&](const RawDb &db, std::vector<uint32_t> &off, std::vector<uint16_t> &val, std::vector<uint32_t> &lst) {
            uint32_t first = b.add_lists(db, all);
            off.assign(np + 1, 0);
            std::vector<int32_t> pk(db.n);
            for (uint64_t i = 0; i < db.n; i++) {
                size_t kn = db.koff[i + 1] - db.koff[i];
                pk[i] = kn >= 3 ? ix.find_prefix(std::string((const char *)db.keys.data() + db.koff[i], kn - 3)) : -1;
                if (pk[i] >= 0) off[pk[i] + 1]++;
            }
            for (size_t p = 0; p < np; p++) off[p + 1] += off[p];
            val.assign(off[np], 0);
            lst.assign(off[np], NO_LIST);
            std::vector<uint32_t> cur(off.begin(), off.end() - 1);
            for (uint64_t i = 0; i < db.n; i++) {
                if (pk[i] < 0) continue;
                const uint8_t *k = db.keys.data() + db.koff[i + 1] - 2;
                uint32_t at = cur[pk[i]]++;
                val[at] = (uint16_t)((k[0] << 8) | k[1]);
                lst[at] = first + (uint32_t)i;
            }
        };
        csr_p(dbs[8], ix.pf_off, ix.pf_fid, ix.pf_list);
        csr_p(dbs[7], ix.pp_off, ix.pp_pos, ix.pp_list);
    }
    // field_id_word_count: key = u16be fid | u8 count
    {
        const RawDb &db = dbs[9];
        uint32_t first = b.add_lists(db, all);
        for (uint64_t i = 0; i < db.n; i++) {
            const uint8_t *k = db.keys.data() + db.koff[i];
            if (db.koff[i + 1] - db.koff[i] != 3) continue;
            uint32_t fid = (k[0] << 8) | k[1];
            ix.fwc_list[(fid << 8) | k[2]] = first + (uint32_t)i;
        }
    }
    // word pair proximity: key = prox | w1 | 0 | w2, already sorted by (prox, w1, w2) == packed key order
    {
        const RawDb &db = dbs[4];
        std::vector<uint64_t> keys(db.n, ~0ull);
        std::vector<uint8_t> keep(db.n, 0);
        unsigned nt = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
        std::vector<std::thread> th;
        for (unsigned t = 0; t < nt; t++)
            th.emplace_back([&, t]() {
                uint64_t a = db.n * t / nt, e = db.n * (t + 1) / nt;
                std::string last_w1;
                int64_t last_r1 = -1;
                for (uint64_t i = a; i < e; i++) {
                    const uint8_t *k = db.keys.data() + db.koff[i];
                    size_t kn = db.koff[i + 1] - db.koff[i];
                    if (kn < 3) continue;
                    const uint8_t *z = (const uint8_t *)memchr(k + 1, 0, kn - 1);
                    if (!z) continue;
                    size_t l1 = z - (k + 1);
                    int64_t r1;
                    if (last_r1 >= 0 && last_w1.size() == l1 && memcmp(last_w1.data(), k + 1, l1) == 0)
                        r1 = last_r1;
                    else {
                        r1 = ix.find_word(k + 1, l1);
                        last_w1.assign((const char *)k + 1, l1);
                        last_r1 = r1;
                    }
                    int64_t r2 = ix.find_word(z + 1, kn - 2 - l1);
                    if (r1 < 0 || r2 < 0) continue;
                    keys[i] = HostIndex::pair_key(k[0], (uint32_t)r1, (uint32_t)r2);
                    keep[i] = 1;
                }
            });
        for (auto &x : th) x.join();
        // keys whose words are unknown are dropped; the rest must be strictly ascending
        bool all_kept = true;
        for (auto kflag : keep) all_kept = all_kept && kflag;
        uint32_t first = b.add_lists(db, keep);
        ix.pair_list_base = first;
        if (all_kept) {
            ix.pair_keys = std::move(keys);
        } else {
            // compact: list ids must stay contiguous with the keys, so rebuild the list table slice
            std::vector<ListRef> kept;
            for (uint64_t i = 0; i < db.n; i++)
                if (keep[i]) {
                    ix.pair_keys.push_back(keys[i]);
                    kept.push_back(ix.lists[first + i]);
                }
            ix.lists.resize(first);
            ix.lists.insert(ix.lists.end(), kept.begin(), kept.end());
        }
        for (size_t i = 1; i < ix.pair_keys.size(); i++)
            if (ix.pair_keys[i - 1] >= ix.pair_keys[i]) throw std::runtime_error("stage: word_pair_proximity_docids keys not in LMDB order");
    }
}

}  // namespace b200
