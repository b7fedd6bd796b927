// Staging to HBM, term derivation (S3) and the vector store (S4).
#include <cuda_fp16.h>
#include <dlfcn.h>

#include <algorithm>
#include <cctype>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <stdexcept>

#include "engine.h"
#include "kernels.h"

namespace b200 {

void HostAffinity::detect(int device) {
    valid = false;
    if (const char *env = getenv("B200_PIN"))
        if (atoi(env) == 0) return;
    char bus[32] = {};
    if (cudaDeviceGetPCIBusId(bus, sizeof bus, device) != cudaSuccess) return;
    for (char *c = bus; *c; c++) *c = (char)tolower((unsigned char)*c);
    int node = -1;
    {
        std::string path = std::string("/sys/bus/pci/devices/") + bus + "/numa_node";
        FILE *f = fopen(path.c_str(), "r");
        if (!f) return;
        if (fscanf(f, "%d", &node) != 1) node = -1;
        fclose(f);
    }
    if (node < 0) return;
    char list[4096] = {};
    {
        std::string path = "/sys/devices/system/node/node" + std::to_string(node) + "/cpulist";
        FILE *f = fopen(path.c_str(), "r");
        if (!f) return;
        if (!fgets(list, sizeof list, f)) list[0] = 0;
        fclose(f);
    }
    cpu_set_t allowed, want;
    if (sched_getaffinity(0, sizeof allowed, &allowed) != 0) return;
    CPU_ZERO(&want);
    int n = 0, n_allowed = CPU_COUNT(&allowed);
    for (const char *c = list; *c;) {  // "0-31,64-95"
        if (*c < '0' || *c > '9') {
            c++;
            continue;
        }
        char *end;
        long a = strtol(c, &end, 10), b2 = a;
        if (*end == '-') b2 = strtol(end + 1, &end, 10);
        for (long k = a; k <= b2 && k < CPU_SETSIZE; k++)
            if (CPU_ISSET((int)k, &allowed)) {
                CPU_SET((int)k, &want);
                n++;
            }
        c = end;
    }
    if (n < 4 || n == n_allowed) return;  // nothing to narrow, or too little left to work with
    cpus = want;
    valid = true;
}


#define CU(call, what)                         \
    do {                                       \
        cudaError_t e_ = (call);               \
        if (e_ != cudaSuccess) return cuda_fail(e_, what); \
    } while (0)

template <class T>
static cudaError_t upload(T **dst, const T *src, size_t n) {
    *dst = nullptr;
    if (n == 0) n = 1;
    cudaError_t e = cudaMalloc((void **)dst, n * sizeof(T));
    if (e != cudaSuccess) return e;
    if (src) return cudaMemcpy(*dst, src, n * sizeof(T), cudaMemcpyHostToDevice);
    return cudaMemset(*dst, 0, n * sizeof(T));
}

Engine::~Engine() {
    for (auto &t : reapers)
        if (t.joinable()) t.join();
    reapers.clear();
    cudaSetDevice(device);
    for (void *p : {(void *)dix.dict_bytes, (void *)dix.dict_off, (void *)dix.pool, (void *)dix.lists, (void *)dix.pair_keys, (void *)dix.base_ub,
                    (void *)dix.emb, (void *)dix.emb_inv_norm, (void *)dix.emb_docids, (void *)arena, (void *)scratch})
        if (p) cudaFree(p);
    for (auto &ln : lanes) ln.release();
    d_step.release();
    d_results.release();
    d_queue.release();
    d_qcount.release();
    d_pathbuf.release();
    d_docids_out.release();
    d_lev_terms.release();
    d_lev_recs.release();
    d_lev_u32.release();
    d_lev_sched.release();
    d_vq.release();
    d_vdist.release();
    d_vsel_dist.release();
    d_vsel_ids.release();
    d_vsel_n.release();
    d_cand.release();
    if (h_step) cudaFreeHost(h_step);
    if (h_results) cudaFreeHost(h_results);
    for (auto e : ev_pool) cudaEventDestroy(e);
    if (sc.comm && sc.comm_destroy) sc.comm_destroy(sc.comm);
    d_gather_ids.release();
    d_gather_dist.release();
    d_gather_n.release();
    for (auto e : vt.ev_pool) cudaEventDestroy(e);
    if (vt.stream) cudaStreamDestroy(vt.stream);
    if (ev0) cudaEventDestroy(ev0);
    if (ev1) cudaEventDestroy(ev1);
    if (stream) cudaStreamDestroy(stream);
}

size_t Engine::mark() {
    if (ev_used == ev_pool.size()) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        ev_pool.push_back(e);
    }
    cudaEventRecord(ev_pool[ev_used], stream);
    return ev_used++;
}
void Engine::resolve_timers() {
    for (auto &t : timed) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, ev_pool[t.a], ev_pool[t.b]) == cudaSuccess) stats.kernel_ms[t.cls] += ms;
    }
    timed.clear();
    ev_used = 0;
}

int Engine::stage_finish() {
    CU(cudaSetDevice(device), "cudaSetDevice");
    try {
        build_host_index(raw_dict_bytes, raw_dict_off, raw_dbs, raw_docids, hix);
    } catch (const std::exception &e) {
        return fail(B200_ERR_INVALID, e.what());
    }
    Settings keep = hix.settings;
    (void)keep;
    // dictionary
    std::vector<uint32_t> off32(hix.dict_off.size());
    for (size_t i = 0; i < off32.size(); i++) off32[i] = (uint32_t)hix.dict_off[i];
    if (off32.empty()) off32.push_back(0);
    CU(upload(&dix.dict_bytes, hix.dict_bytes.data(), hix.dict_bytes.size()), "upload dictionary");
    CU(upload(&dix.dict_off, off32.data(), off32.size()), "upload dictionary offsets");
    // posting store
    CU(upload(&dix.pool, hix.pool.data(), hix.pool.size()), "upload posting pool");
    static_assert(sizeof(ListRef) == sizeof(DListRef), "ListRef layout");
    CU(upload(&dix.lists, reinterpret_cast<const DListRef *>(hix.lists.data()), hix.lists.size()), "upload list table");
    CU(upload(&dix.pair_keys, reinterpret_cast<const unsigned long long *>(hix.pair_keys.data()), hix.pair_keys.size()), "upload pair keys");
    CU(upload(&dix.base_ub, reinterpret_cast<const unsigned long long *>(hix.base_ub.data()), hix.base_ub.size()), "upload universe");
    stats.hbm_bytes_staged = hix.dict_bytes.size() + off32.size() * 4 + hix.pool.size() * 4 + hix.lists.size() * sizeof(ListRef) +
                             hix.pair_keys.size() * 8 + hix.base_ub.size() * 8;
    std::vector<uint32_t>().swap(hix.pool);
    // release the raw staging copies
    for (auto &db : raw_dbs) {
        std::vector<uint8_t>().swap(db.keys);
        std::vector<uint8_t>().swap(db.vals);
        std::vector<uint64_t>().swap(db.koff);
        std::vector<uint64_t>().swap(db.voff);
    }
    // work pools
    size_t free_b = 0, total_b = 0;
    CU(cudaMemGetInfo(&free_b, &total_b), "cudaMemGetInfo");
    auto env_mb = [](const char *name, size_t dflt) {
        const char *v = getenv(name);
        return v ? (size_t)atoll(v) << 20 : dflt;
    };
    // sized for 180 GB of HBM: a sixth of what is free each (capped; two handles can coexist), the rest stays for the embeddings staged afterwards and
    // the row lookup tables; a 10 M-document index at batch 256 needs ~ 30 GB of scratch for its widest rule step
    arena_bytes = env_mb("B200_ARENA_MB", std::min<size_t>(free_b / 6, (size_t)32 << 30));
    scratch_bytes = env_mb("B200_SCRATCH_MB", std::min<size_t>(free_b / 6, (size_t)40 << 30));
    CU(cudaMalloc((void **)&arena, arena_bytes), "alloc arena");
    CU(cudaMalloc((void **)&scratch, scratch_bytes), "alloc scratch");
    staged = true;
    return B200_OK;
}

// The vector store: fp16 rows + f32 inverse norms + docids.  f32 input (what arroy/hannoy item nodes hold) is converted on the
// device, chunk by chunk; `half_rows` non-null = the caller already holds IEEE binary16 rows.
int Engine::stage_embeddings(const float *vectors, const uint16_t *half_rows, uint64_t n, uint32_t d, const uint32_t *docids) {
    CU(cudaSetDevice(device), "cudaSetDevice");
    if (d == 0) return fail(B200_ERR_INVALID, "embedding dimension must be positive");
    if (!vectors && !half_rows && n) return fail(B200_ERR_INVALID, "embeddings: null matrix");
    if (d % 8 != 0) {
        // the kernels read rows in 128-bit pieces: pad every row with zeros up to a multiple of 8 (cosine does not change)
        const uint32_t dp = (d + 7) & ~7u;
        std::vector<float> padded((size_t)n * dp, 0.f);
        for (uint64_t r = 0; r < n; r++)
            for (uint32_t i = 0; i < d; i++)
                padded[r * dp + i] = vectors ? vectors[r * d + i] : __half2float(reinterpret_cast<const __half *>(half_rows)[r * d + i]);
        int rc = stage_embeddings(padded.data(), nullptr, n, dp, docids);
        if (rc == B200_OK) emb_d_user = d;
        return rc;
    }
    emb_d_user = d;
    for (void *p : {(void *)dix.emb, (void *)dix.emb_inv_norm, (void *)dix.emb_docids})
        if (p) cudaFree(p);
    dix.emb = nullptr;
    dix.emb_inv_norm = nullptr;
    dix.emb_docids = nullptr;
    dix.emb_n = 0;
    const size_t rows_alloc = std::max<uint64_t>(n, 1);
    CU(cudaMalloc(&dix.emb, rows_alloc * d * 2), "alloc embeddings");
    CU(cudaMalloc((void **)&dix.emb_inv_norm, rows_alloc * 4), "alloc norms");
    CU(cudaMalloc((void **)&dix.emb_docids, rows_alloc * 4), "alloc embedding docids");
    uint8_t *dm = reinterpret_cast<uint8_t *>(dix.emb);
    const uint64_t chunk = std::max<uint64_t>(1, ((uint64_t)256 << 20) / ((uint64_t)d * 4));  // rows per 256 MB of f32
    if (half_rows) {
        for (uint64_t r0 = 0; r0 < n; r0 += chunk * 2) {
            const uint64_t nr = std::min<uint64_t>(chunk * 2, n - r0);
            CU(cudaMemcpyAsync(dm + r0 * d * 2, half_rows + r0 * d, nr * d * 2, cudaMemcpyHostToDevice, stream), "H2D embeddings");
        }
        CU(launch_emb_norm_f16(stream, dix.emb, dix.emb_inv_norm, n, d), "embedding norms");
    } else {
        float *stage = nullptr;
        CU(cudaMalloc((void **)&stage, std::min<uint64_t>(chunk, rows_alloc) * d * 4), "alloc embedding staging");
        for (uint64_t r0 = 0; r0 < n; r0 += chunk) {
            const uint64_t nr = std::min<uint64_t>(chunk, n - r0);
            cudaError_t e = cudaMemcpyAsync(stage, vectors + r0 * d, nr * d * 4, cudaMemcpyHostToDevice, stream);
            if (e == cudaSuccess) e = launch_emb_from_f32(stream, stage, dm + r0 * d * 2, dix.emb_inv_norm + r0, nr, d);
            if (e != cudaSuccess) {
                cudaFree(stage);
                return cuda_fail(e, "convert embeddings");
            }
        }
        cudaStreamSynchronize(stream);
        cudaFree(stage);
    }
    if (docids)
        CU(cudaMemcpyAsync(dix.emb_docids, docids, n * 4, cudaMemcpyHostToDevice, stream), "H2D embedding docids");
    else {
        std::vector<uint32_t> ids(n);
        for (uint64_t r = 0; r < n; r++) ids[r] = (uint32_t)r;
        CU(cudaMemcpy(dix.emb_docids, ids.data(), n * 4, cudaMemcpyHostToDevice), "H2D embedding docids");
    }
    CU(cudaStreamSynchronize(stream), "sync");
    // which documents own an embedding (VectorSort returns the others as its last bucket, vector_sort.rs:128-160)
    emb_bitmap.assign(hix.n_words64, 0);
    for (uint64_t r = 0; r < n; r++) {
        const uint32_t doc = docids ? docids[r] : (uint32_t)r;
        if ((doc >> 6) < emb_bitmap.size()) emb_bitmap[doc >> 6] |= 1ull << (doc & 63);
    }
    dix.emb_n = n;
    dix.emb_d = d;
    stats.hbm_bytes_staged += n * d * 2 + n * 8;
    return B200_OK;
}

// The derivation schedule: which (chunk of terms, 256-word tile) pairs lev_match_kernel visits, one CTA each.
//
// Why it is exact.  The kernel's filter lets a (term, word) pair through only when
//   w[0] == q[0] (budget k_same), or
//   w[0] != q[0], k_diff >= 0 and (m < 2 or w[1] == q[1] or w[1] == q[0] or w[0] == q[1]),
// and it rejects every word of a term with k_same < 0 (its first test, popcount > k_same, always holds).  For every term those
// words are the disjoint union of its groups (device_types.h):
//   k_same < 0                      none
//   k_diff < 0                      F(q0)
//   k_diff >= 0, m < 2              ALL
//   k_diff >= 0, m >= 2             F(q0), S(q0), and when q1 != q0 also F(q1), S(q1)
// since F(q1) holds the words with w[0] == q1 != q0, and S(q0) ∪ S(q1) those with w[0] not in {q0, q1} and w[1] in {q0, q1}.
// A group's tiles cover all of its words, and inside an item the kernel tests a pair only when the word lies in the item's group
// for that term.  So every pair that a full (tile x term) sweep could pass through the first-byte rule is tested exactly once,
// by the same filter and DP, and no other pair is.  The records of one 32-word group that two items produce hold disjoint words;
// lev_finalize_kernel ORs them after sorting by word id, so it replays the 150 / 50 caps over the same codes in the same word-id
// order and keeps the same words.
namespace {
struct LevSchedule {
    std::vector<LevItem> items;
    std::vector<LevChunk> chunks;
    std::vector<uint32_t> term_idx;  // the members of every group, group by group
    uint64_t bytes = 0;              // dictionary bytes + offsets of the tiles the items stage
};
void build_lev_schedule(const HostIndex &ix, const std::vector<LevTerm> &terms, LevSchedule &s) {
    constexpr uint32_t G_S = 256, G_ALL = 512, N_GROUPS = 513;  // group ids: F(c) = c, S(c) = 256 + c, ALL = 512
    auto groups_of = [](const LevTerm &t, auto &&add) {
        if (t.k_same < 0) return;
        const uint8_t q0 = t.q[0], q1 = t.q[1];
        if (t.k_diff < 0) {
            add(q0);
        } else if (t.len < 2) {
            add(G_ALL);
        } else {
            add(q0);
            add(G_S + q0);
            if (q1 != q0) {
                add(q1);
                add(G_S + q1);
            }
        }
    };
    std::vector<uint32_t> first(N_GROUPS + 1, 0);
    for (const LevTerm &t : terms) groups_of(t, [&](uint32_t g) { first[g + 1]++; });
    for (uint32_t g = 0; g < N_GROUPS; g++) first[g + 1] += first[g];
    s.term_idx.resize(first[N_GROUPS]);
    std::vector<uint32_t> fill(first.begin(), first.end() - 1);
    for (uint32_t i = 0; i < (uint32_t)terms.size(); i++) groups_of(terms[i], [&](uint32_t g) { s.term_idx[fill[g]++] = i; });

    const uint32_t n_words = (uint32_t)ix.n_words;
    const std::vector<uint32_t> &start = ix.dict_pair_start;
    std::vector<uint32_t> tiles;
    auto add_words = [&](uint32_t lo, uint32_t hi) {  // the tiles of words [lo, hi); ranges come in increasing order
        if (lo >= hi) return;
        uint32_t t = lo / 256;
        if (!tiles.empty() && tiles.back() >= t) t = tiles.back() + 1;
        for (; t <= (hi - 1) / 256; t++) tiles.push_back(t);
    };
    for (uint32_t g = 0; g < N_GROUPS; g++) {
        if (first[g] == first[g + 1]) continue;
        tiles.clear();
        if (g < G_S) {
            add_words(start[g << 8], start[(g + 1) << 8]);
        } else if (g < G_ALL) {
            for (uint32_t b0 = 0; b0 < 256; b0++) add_words(start[b0 << 8 | (g - G_S)], start[(b0 << 8 | (g - G_S)) + 1]);
        } else {
            add_words(0, n_words);
        }
        uint64_t tile_bytes = 0;
        for (uint32_t t : tiles) {
            const uint32_t w0 = t * 256, w1 = std::min(n_words, w0 + 256);
            tile_bytes += ix.dict_off[w1] - ix.dict_off[w0] + 4ull * (w1 - w0);
        }
        const uint8_t kind = g < G_S ? LEV_GROUP_F : (g < G_ALL ? LEV_GROUP_S : LEV_GROUP_ALL);
        for (uint32_t c0 = first[g]; c0 < first[g + 1]; c0 += LEV_TERMS_PER_CTA) {
            const uint32_t chunk = (uint32_t)s.chunks.size();
            s.chunks.push_back(LevChunk{c0, (uint8_t)std::min<uint32_t>(LEV_TERMS_PER_CTA, first[g + 1] - c0), kind, (uint8_t)(g & 255), 0});
            for (uint32_t t : tiles) s.items.push_back(LevItem{t, chunk});
            s.bytes += tile_bytes;
        }
    }
}
}  // namespace

int Engine::derive_batch(uint32_t n, const char *words, const uint32_t *off, const uint8_t *max_typo, const uint8_t *is_prefix,
                         uint32_t *one_out, uint32_t *n_one, uint32_t *two_out, uint32_t *n_two) {
    if (!staged) return fail(B200_ERR_STATE, "derive before b200_stage_finish");
    CU(cudaSetDevice(device), "cudaSetDevice");
    if (n == 0) return B200_OK;
    std::vector<LevTerm> terms(n);
    for (uint32_t i = 0; i < n; i++) {
        uint32_t len = off[i + 1] - off[i];
        if (len == 0 || len > LEV_MAX_Q) return fail(B200_ERR_UNSUPPORTED, "derive: word longer than 64 bytes (or empty)");
        LevTerm &t = terms[i];
        memset(&t, 0, sizeof t);
        memcpy(t.q, words + off[i], len);
        t.len = (uint8_t)len;
        t.k_same = max_typo[i] >= 2 ? 2 : 1;
        t.k_diff = max_typo[i] >= 2 ? 1 : -1;
        t.prefix = is_prefix[i] ? 1 : 0;
        if (max_typo[i] == 0) t.k_same = -1;
    }
    CU(d_lev_terms.reserve(n), "alloc lev terms");
    CU(d_lev_recs.reserve((size_t)n * LEV_REC_CAP), "alloc lev records");
    size_t per = 1 + 150 + 1 + 50 + 1 + 1;
    CU(d_lev_u32.reserve((size_t)n * per), "alloc lev outputs");
    uint32_t *rec_count = d_lev_u32.p, *d_one = rec_count + n, *d_n_one = d_one + (size_t)n * 150, *d_two = d_n_one + n,
             *d_n_two = d_two + (size_t)n * 50;
    int32_t *d_status = reinterpret_cast<int32_t *>(d_n_two + n);
    LevSchedule sched;
    build_lev_schedule(hix, terms, sched);
    static_assert(sizeof(LevItem) % 4 == 0 && sizeof(LevChunk) % 4 == 0, "schedule layout");
    const size_t items_u32 = sched.items.size() * sizeof(LevItem) / 4, chunks_u32 = sched.chunks.size() * sizeof(LevChunk) / 4;
    CU(d_lev_sched.reserve(items_u32 + chunks_u32 + sched.term_idx.size()), "alloc lev schedule");
    const LevItem *d_items = reinterpret_cast<const LevItem *>(d_lev_sched.p);
    const LevChunk *d_chunks = reinterpret_cast<const LevChunk *>(d_lev_sched.p + items_u32);
    const uint32_t *d_term_idx = d_lev_sched.p + items_u32 + chunks_u32;
    CU(cudaMemcpyAsync(d_lev_terms.p, terms.data(), n * sizeof(LevTerm), cudaMemcpyHostToDevice, stream), "H2D lev terms");
    CU(cudaMemcpyAsync((void *)d_items, sched.items.data(), items_u32 * 4, cudaMemcpyHostToDevice, stream), "H2D lev schedule");
    CU(cudaMemcpyAsync((void *)d_chunks, sched.chunks.data(), chunks_u32 * 4, cudaMemcpyHostToDevice, stream), "H2D lev schedule");
    CU(cudaMemcpyAsync((void *)d_term_idx, sched.term_idx.data(), sched.term_idx.size() * 4, cudaMemcpyHostToDevice, stream), "H2D lev schedule");
    stats.h2d_bytes += n * sizeof(LevTerm) + (items_u32 + chunks_u32 + sched.term_idx.size()) * 4;
    stats.d2h_bytes += (size_t)n * (150 + 50 + 3) * 4;
    size_t m0 = mark();
    CU(launch_lev(stream, dix.dict_bytes, dix.dict_off, (uint32_t)hix.n_words, d_lev_terms.p, n, d_term_idx, d_chunks, d_items,
                  (uint32_t)sched.items.size(), d_lev_recs.p, rec_count, d_one, d_n_one, d_two, d_n_two, d_status),
       "lev kernels");
    size_t m1 = mark();
    time_kernel(B200_K_LEV, m0, m1, sched.bytes);
    stats.kernel_launches += 1;
    stats.dictionary_bytes += sched.bytes;
    std::vector<int32_t> status(n);
    CU(cudaMemcpyAsync(one_out, d_one, (size_t)n * 150 * 4, cudaMemcpyDeviceToHost, stream), "D2H");
    CU(cudaMemcpyAsync(n_one, d_n_one, (size_t)n * 4, cudaMemcpyDeviceToHost, stream), "D2H");
    CU(cudaMemcpyAsync(two_out, d_two, (size_t)n * 50 * 4, cudaMemcpyDeviceToHost, stream), "D2H");
    CU(cudaMemcpyAsync(n_two, d_n_two, (size_t)n * 4, cudaMemcpyDeviceToHost, stream), "D2H");
    CU(cudaMemcpyAsync(status.data(), d_status, (size_t)n * 4, cudaMemcpyDeviceToHost, stream), "D2H");
    CU(cudaStreamSynchronize(stream), "sync");
    resolve_timers();
    for (uint32_t i = 0; i < n; i++)
        if (status[i] != 0) return fail(B200_ERR_CAPACITY, "derive: match-record capacity exceeded for a term");
    return B200_OK;
}

int Engine::comm_load() {
    if (sc.lib) return B200_OK;
    void *lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);  // the copy this process already has (torch's), if any
    if (!lib) lib = dlopen("libnccl.so.2", RTLD_NOW);
    if (!lib) return fail(B200_ERR_STATE, std::string("cannot load libnccl.so.2: ") + dlerror());
    sc.get_unique_id = reinterpret_cast<int (*)(void *)>(dlsym(lib, "ncclGetUniqueId"));
    sc.comm_init_rank = reinterpret_cast<int (*)(void **, int, NcclId, int)>(dlsym(lib, "ncclCommInitRank"));
    sc.all_gather = reinterpret_cast<int (*)(const void *, void *, size_t, int, void *, cudaStream_t)>(dlsym(lib, "ncclAllGather"));
    sc.group_start = reinterpret_cast<int (*)()>(dlsym(lib, "ncclGroupStart"));
    sc.group_end = reinterpret_cast<int (*)()>(dlsym(lib, "ncclGroupEnd"));
    sc.comm_destroy = reinterpret_cast<int (*)(void *)>(dlsym(lib, "ncclCommDestroy"));
    sc.get_error_string = reinterpret_cast<const char *(*)(int)>(dlsym(lib, "ncclGetErrorString"));
    if (!sc.get_unique_id || !sc.comm_init_rank || !sc.all_gather || !sc.group_start || !sc.group_end || !sc.comm_destroy)
        return fail(B200_ERR_STATE, "libnccl.so.2 lacks an expected symbol");
    sc.lib = lib;
    return B200_OK;
}
int Engine::comm_init(int rank, int world, const uint8_t *unique_id) {
    int rc = comm_load();
    if (rc != B200_OK) return rc;
    if (world < 1 || rank < 0 || rank >= world) return fail(B200_ERR_INVALID, "comm_init: bad rank / world");
    CU(cudaSetDevice(device), "cudaSetDevice");
    if (sc.comm) {
        sc.comm_destroy(sc.comm);
        sc.comm = nullptr;
    }
    NcclId id;
    memcpy(id.internal, unique_id, 128);
    int e = sc.comm_init_rank(&sc.comm, world, id, rank);
    if (e != 0) return fail(B200_ERR_CUDA, std::string("ncclCommInitRank: ") + (sc.get_error_string ? sc.get_error_string(e) : "error"));
    sc.rank = rank;
    sc.world = world;
    return B200_OK;
}

int Engine::nns_batch(const float *queries, uint32_t n_q, uint32_t d, uint32_t limit, const uint64_t *cand, uint64_t n_cand_words,
                      uint32_t *ids_out, float *dist_out, uint32_t *n_out, bool sharded) {
    if (sharded && (!sc.comm || sc.world < 1)) return fail(B200_ERR_STATE, "sharded nns before b200_comm_init");
    CU(cudaSetDevice(device), "cudaSetDevice");
    if (!dix.emb) return fail(B200_ERR_STATE, "nns before b200_stage_embeddings");
    if (d != emb_d_user && d != dix.emb_d) return fail(B200_ERR_INVALID, "nns: query dimension differs from the staged embeddings");
    if (d != dix.emb_d) {  // rows were zero-padded at staging: pad the queries the same way
        std::vector<float> padded((size_t)n_q * dix.emb_d, 0.f);
        for (uint32_t q = 0; q < n_q; q++) memcpy(padded.data() + (size_t)q * dix.emb_d, queries + (size_t)q * d, (size_t)d * 4);
        return nns_batch(padded.data(), n_q, dix.emb_d, limit, cand, n_cand_words, ids_out, dist_out, n_out, sharded);
    }
    if (n_q == 0) return B200_OK;
    const uint64_t N = dix.emb_n;
    const uint32_t tie_cap = 1024;
    const uint32_t QT = 8;  // queries per scan pass
    uint32_t chunk = std::min<uint32_t>(n_q, 64);  // queries whose distance rows are resident at once
    CU(d_vq.reserve((size_t)chunk * d + chunk), "alloc queries");
    CU(d_vdist.reserve((size_t)chunk * N), "alloc distances");
    CU(d_vsel_dist.reserve((size_t)chunk * (limit + tie_cap)), "alloc selection");
    CU(d_vsel_ids.reserve((size_t)chunk * (limit + tie_cap)), "alloc selection");
    CU(d_vsel_n.reserve((size_t)chunk * 2), "alloc selection");
    const unsigned long long *d_c = nullptr;
    if (cand) {
        CU(d_cand.reserve(n_cand_words), "alloc candidates");
        CU(cudaMemcpyAsync(d_cand.p, cand, n_cand_words * 8, cudaMemcpyHostToDevice, vt.stream), "H2D candidates");
        d_c = d_cand.p;
    }
    // ---- batched path: tcgen05 GEMM with the top-k fused into its epilogue (vec_gemm.cu)
    {
        const char *force = getenv("B200_VEC_GEMM");
        bool want = force ? atoi(force) != 0 : n_q >= 16;
        if (sharded) {
            want = true;  // the exchange works on the device-resident top-k lists of the batched path
            if (!vec_gemm_supported(d, limit)) return fail(B200_ERR_UNSUPPORTED, "sharded nns: dimension / limit outside the batched kernel's range");
        }
        if (want && vec_gemm_supported(d, limit)) {
            const uint32_t vec_sms = getenv("B200_VEC_SMS") ? (uint32_t)std::max(8, std::min(sm_count, atoi(getenv("B200_VEC_SMS")))) : (uint32_t)sm_count;
            const uint32_t tiles_per_pass = vec_sms;  // query tiles resident in one launch
            std::vector<uint32_t> h_ids, h_n;
            std::vector<float> h_dist;
            for (uint32_t q0 = 0; q0 < n_q; q0 += tiles_per_pass * 128) {
                uint32_t nq = std::min<uint32_t>(n_q - q0, tiles_per_pass * 128);
                uint32_t n_qtiles = (nq + 127) / 128, n_pad = n_qtiles * 128;
                uint64_t n_row_tiles = (N + 63) / 64;
                uint32_t n_groups = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)vec_sms / n_qtiles, n_row_tiles));
                CU(d_vq.reserve((size_t)nq * d + n_pad), "alloc queries");
                CU(d_vq16.reserve((size_t)n_pad * d), "alloc fp16 queries");
                CU(d_vruns.reserve((size_t)n_qtiles * n_groups * 128 * VEC_GEMM_CAND_CAP + (size_t)n_pad * n_groups), "alloc candidate runs");
                CU(d_vpartial.reserve((size_t)n_pad * n_groups * VEC_GEMM_KMAX), "alloc partial top-k");
                CU(d_vsel_dist.reserve((size_t)n_pad * limit), "alloc selection");
                CU(d_vsel_ids.reserve((size_t)n_pad * limit), "alloc selection");
                CU(d_vsel_n.reserve(n_pad), "alloc selection");
                float *d_qinv = d_vq.p + (size_t)nq * d;
                CU(cudaMemcpyAsync(d_vq.p, queries + (size_t)q0 * d, (size_t)nq * d * 4, cudaMemcpyHostToDevice, vt.stream), "H2D queries");
                vstats.h2d_bytes += (size_t)nq * d * 4;
                CU(launch_vec_prep_queries(vt.stream, d_vq.p, nq, n_pad, d, d_vq16.p, d_qinv), "vec_prep_queries");
                vstats.kernel_launches++;
                size_t m0 = vt.mark();
                CU(launch_vec_gemm_topk(vt.stream, vec_sms, dix.emb, dix.emb_inv_norm, dix.emb_docids, N, d, d_vq16.p, d_qinv, n_qtiles, n_groups,
                                        d_c, n_cand_words, limit, d_vruns.p + (size_t)n_qtiles * n_groups * 128 * VEC_GEMM_CAND_CAP, d_vruns.p, d_vpartial.p, d_vsel_ids.p, d_vsel_dist.p, d_vsel_n.p, nq),
                   "vec_gemm_topk");
                if (sharded && sc.world > 1) {
                    // one all-gather of the per-shard top-k (ids, distances, counts) on the vector stream, then the merge: the lists
                    // never leave the device between the scan and the merged result
                    const uint32_t Wd = (uint32_t)sc.world;
                    CU(d_gather_ids.reserve((size_t)Wd * nq * limit), "alloc gather");
                    CU(d_gather_dist.reserve((size_t)Wd * nq * limit), "alloc gather");
                    CU(d_gather_n.reserve((size_t)Wd * nq), "alloc gather");
                    int e = sc.group_start();
                    if (!e) e = sc.all_gather(d_vsel_ids.p, d_gather_ids.p, (size_t)nq * limit * 4, 1 /* ncclUint8 */, sc.comm, vt.stream);
                    if (!e) e = sc.all_gather(d_vsel_dist.p, d_gather_dist.p, (size_t)nq * limit * 4, 1, sc.comm, vt.stream);
                    if (!e) e = sc.all_gather(d_vsel_n.p, d_gather_n.p, (size_t)nq * 4, 1, sc.comm, vt.stream);
                    int e2 = sc.group_end();
                    if (e || e2) return fail(B200_ERR_CUDA, std::string("ncclAllGather: ") + (sc.get_error_string ? sc.get_error_string(e ? e : e2) : "error"));
                    CU(launch_shard_merge(vt.stream, d_gather_ids.p, d_gather_dist.p, d_gather_n.p, Wd, nq, limit, d_vsel_ids.p, d_vsel_dist.p, d_vsel_n.p),
                       "shard merge");
                    vstats.kernel_launches++;
                }
                size_t m1 = vt.mark();
                // algorithmic bytes: every query tile streams the matrix once (L2 absorbs the re-reads across tiles of the same rows)
                vt.time_kernel(vstats, B200_K_VEC_GEMM, m0, m1, (uint64_t)N * d * 2 + N * 8 + (uint64_t)n_pad * d * 2);
                vstats.kernel_launches++;  // merge kernel
                vstats.vector_bytes += (uint64_t)N * d * 2;
                h_ids.resize((size_t)nq * limit);
                h_dist.resize((size_t)nq * limit);
                h_n.resize(nq);
                CU(cudaMemcpyAsync(h_ids.data(), d_vsel_ids.p, (size_t)nq * limit * 4, cudaMemcpyDeviceToHost, vt.stream), "D2H");
                CU(cudaMemcpyAsync(h_dist.data(), d_vsel_dist.p, (size_t)nq * limit * 4, cudaMemcpyDeviceToHost, vt.stream), "D2H");
                CU(cudaMemcpyAsync(h_n.data(), d_vsel_n.p, (size_t)nq * 4, cudaMemcpyDeviceToHost, vt.stream), "D2H");
                vstats.d2h_bytes += (size_t)nq * limit * 8 + nq * 4;
                CU(cudaStreamSynchronize(vt.stream), "sync");
                vt.resolve(vstats);
                for (uint32_t q = 0; q < nq; q++) {
                    uint32_t n = std::min(h_n[q], limit);
                    n_out[q0 + q] = n;
                    memcpy(ids_out + (size_t)(q0 + q) * limit, h_ids.data() + (size_t)q * limit, (size_t)n * 4);
                    memcpy(dist_out + (size_t)(q0 + q) * limit, h_dist.data() + (size_t)q * limit, (size_t)n * 4);
                }
            }
            return B200_OK;
        }
    }
    std::vector<float> qinv(chunk);
    std::vector<float> sel_d((size_t)chunk * (limit + tie_cap));
    std::vector<uint32_t> sel_i((size_t)chunk * (limit + tie_cap)), sel_n((size_t)chunk * 2);
    float total_ms = 0;
    for (uint32_t q0 = 0; q0 < n_q; q0 += chunk) {
        uint32_t nq = std::min(chunk, n_q - q0);
        for (uint32_t q = 0; q < nq; q++) {
            double s = 0;
            const float *v = queries + (size_t)(q0 + q) * d;
            for (uint32_t i = 0; i < d; i++) s += (double)v[i] * v[i];
            float nrm = (float)std::sqrt(s);
            qinv[q] = nrm > 0.f ? 1.0f / nrm : 0.f;
        }
        float *d_qinv = d_vq.p + (size_t)chunk * d;
        CU(cudaMemcpyAsync(d_vq.p, queries + (size_t)q0 * d, (size_t)nq * d * 4, cudaMemcpyHostToDevice, vt.stream), "H2D queries");
        vstats.h2d_bytes += (size_t)nq * d * 4 + nq * 4;
        vstats.d2h_bytes += (size_t)nq * (limit + tie_cap) * 8 + nq * 8;
        CU(cudaMemcpyAsync(d_qinv, qinv.data(), nq * 4, cudaMemcpyHostToDevice, vt.stream), "H2D query norms");
        for (uint32_t t = 0; t < nq;) {
            uint32_t left = nq - t;
            int qt = left >= 8 ? 8 : (left >= 4 ? 4 : (left >= 2 ? 2 : 1));
            (void)QT;
            size_t m0 = vt.mark();
            CU(launch_vec_dist(vt.stream, sm_count * 6, qt, dix.emb, dix.emb_inv_norm, dix.emb_docids, N, d, d_vq.p + (size_t)t * d, d_qinv + t, d_c,
                               n_cand_words, d_vdist.p + (size_t)t * N),
               "vec_dist");
            size_t m1 = vt.mark();
            uint64_t vb = N * d * 2 + N * 4 + (d_c ? N / 8 : 0) + (uint64_t)qt * d * 4 + (uint64_t)qt * N * 4;
            vt.time_kernel(vstats, B200_K_VEC_DIST, m0, m1, vb);
            vstats.vector_bytes += vb;
            t += qt;
        }
        size_t k0 = vt.mark();
        // long rows are selected in pieces side by side (one CTA per >= 16 k distances, about two waves of CTAs per query batch)
        const uint32_t n_slices = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(std::min<uint64_t>(128, (uint64_t)sm_count * 4 / std::max(1u, nq)), N / 16384));
        if (n_slices > 1) {
            CU(d_vpart_dist.reserve((size_t)nq * n_slices * (limit + tie_cap)), "alloc partial selection");
            CU(d_vpart_ids.reserve((size_t)nq * n_slices * (limit + tie_cap)), "alloc partial selection");
            CU(d_vpart_n.reserve((size_t)nq * n_slices * 2), "alloc partial selection");
        }
        CU(launch_topk(vt.stream, nq, d_vdist.p, dix.emb_docids, N, limit, tie_cap, n_slices, d_vpart_dist.p, d_vpart_ids.p, d_vpart_n.p, d_vsel_dist.p,
                       d_vsel_ids.p, d_vsel_n.p),
           "topk");
        size_t k1 = vt.mark();
        vt.time_kernel(vstats, B200_K_TOPK, k0, k1, (uint64_t)nq * N * 4 * 4);
        CU(cudaMemcpyAsync(sel_d.data(), d_vsel_dist.p, (size_t)nq * (limit + tie_cap) * 4, cudaMemcpyDeviceToHost, vt.stream), "D2H");
        CU(cudaMemcpyAsync(sel_i.data(), d_vsel_ids.p, (size_t)nq * (limit + tie_cap) * 4, cudaMemcpyDeviceToHost, vt.stream), "D2H");
        CU(cudaMemcpyAsync(sel_n.data(), d_vsel_n.p, (size_t)nq * 2 * 4, cudaMemcpyDeviceToHost, vt.stream), "D2H");
        CU(cudaStreamSynchronize(vt.stream), "sync");
        vt.resolve(vstats);
        for (uint32_t q = 0; q < nq; q++) {
            std::vector<std::pair<float, uint32_t>> c;
            const float *sd = sel_d.data() + (size_t)q * (limit + tie_cap);
            const uint32_t *si = sel_i.data() + (size_t)q * (limit + tie_cap);
            for (uint32_t i = 0; i < sel_n[2 * q]; i++) c.push_back({sd[i], si[i]});
            for (uint32_t i = 0; i < sel_n[2 * q + 1]; i++) c.push_back({sd[limit + i], si[limit + i]});
            std::sort(c.begin(), c.end());
            uint32_t n = (uint32_t)std::min<size_t>(c.size(), limit);
            n_out[q0 + q] = n;
            for (uint32_t i = 0; i < n; i++) {
                ids_out[(size_t)(q0 + q) * limit + i] = c[i].second;
                dist_out[(size_t)(q0 + q) * limit + i] = c[i].first;
            }
        }
    }
    (void)total_ms;
    return B200_OK;
}

// S2: OR of posting lists, restricted to a universe — what ConditionDocIdsCache::get_computed_condition
// (crates/milli/src/search/new/ranking_rule_graph/condition_docids_cache.rs:34-57) obtains from G::resolve_condition for the
// union-shaped conditions (compute_query_term_subset_docids, resolve_query_graph.rs:33-59: `docids |= list` for every derivation,
// then `& universe`).  One scatter_kernel launch over the dense universe.
int Engine::union_postings(int db, const uint32_t *key_index, uint32_t n_keys, const uint64_t *universe, uint64_t n_universe_words, uint64_t *out) {
    if (!staged) return fail(B200_ERR_STATE, "union_postings before b200_stage_finish");
    if (db < 0 || db >= 10) return fail(B200_ERR_INVALID, "union_postings: unknown database id");
    if (db == 4 && hix.pair_keys.size() != hix.db_keys[4])
        return fail(B200_ERR_UNSUPPORTED, "union_postings: word_pair_proximity keys were dropped at staging, key indices are not stable");
    CU(cudaSetDevice(device), "cudaSetDevice");
    const uint64_t W = hix.n_words64;
    if (universe && n_universe_words < W) return fail(B200_ERR_INVALID, "union_postings: universe bitmap shorter than the document range");
    std::vector<Job> jobs;
    for (uint32_t i = 0; i < n_keys; i++) {
        if (key_index[i] >= hix.db_keys[db]) return fail(B200_ERR_INVALID, "union_postings: key index out of range");
        const uint32_t list = hix.db_first[db] + key_index[i];
        const ListRef &lr = hix.lists[list];
        if (!lr.card) continue;
        const uint64_t units = lr.dense ? W : lr.card;
        for (uint32_t k = 0; k < (units + JOB_CHUNK - 1) / JOB_CHUNK; k++) jobs.push_back(Job{0, 0, list, k});
    }
    const size_t o_ub = 0, o_col = o_ub + W * 8, o_act = (o_col + W * 8 + 255) & ~(size_t)255, o_res = o_act + ((sizeof(ActDesc) + 255) & ~(size_t)255),
                 o_jobs = o_res + 256, o_bigq = (o_jobs + std::max<size_t>(1, jobs.size()) * sizeof(Job) + 255) & ~(size_t)255,
                 total = o_bigq + std::max<size_t>(1, jobs.size()) * 4;
    CU(d_s2.reserve(total), "alloc S2 scratch");
    uint8_t *base = d_s2.p;
    if (universe)
        CU(cudaMemcpyAsync(base + o_ub, universe, W * 8, cudaMemcpyHostToDevice, stream), "H2D universe");
    else
        CU(cudaMemcpyAsync(base + o_ub, dix.base_ub, W * 8, cudaMemcpyDeviceToDevice, stream), "universe");
    CU(cudaMemsetAsync(base + o_col, 0, W * 8, stream), "zero column");
    ActDesc a;
    memset(&a, 0, sizeof a);
    a.ub = reinterpret_cast<unsigned long long *>(base + o_ub);
    a.C = reinterpret_cast<unsigned long long *>(base + o_col);
    a.ld = (uint32_t)W;
    a.n_cols = 1;
    a.res_off = 0;
    uint32_t counters[4] = {(uint32_t)W, 0, 0, 0};      // results[0] = rows
    uint32_t qcount[8] = {(uint32_t)jobs.size(), 0, 0, 0, 0, 0, 0, 0};
    CU(cudaMemcpyAsync(base + o_act, &a, sizeof a, cudaMemcpyHostToDevice, stream), "H2D activation");
    CU(cudaMemcpyAsync(base + o_res, counters, sizeof counters, cudaMemcpyHostToDevice, stream), "H2D rows");
    CU(cudaMemcpyAsync(base + o_res + 64, qcount, sizeof qcount, cudaMemcpyHostToDevice, stream), "H2D job count");
    if (!jobs.empty()) {
        CU(cudaMemcpyAsync(base + o_jobs, jobs.data(), jobs.size() * sizeof(Job), cudaMemcpyHostToDevice, stream), "H2D jobs");
        size_t m0 = mark();
        CU(launch_scatter(stream, (uint32_t)sm_count * 5, reinterpret_cast<const Job *>(base + o_jobs), reinterpret_cast<uint32_t *>(base + o_res + 64),
                          (uint32_t)jobs.size(), reinterpret_cast<const ActDesc *>(base + o_act), reinterpret_cast<const uint32_t *>(base + o_res),
                          dix.lists, dix.pool, reinterpret_cast<uint32_t *>(base + o_bigq)),
           "scatter");
        uint64_t bytes = 0;
        for (auto &j : jobs) bytes += hix.lists[j.list].dense ? (uint64_t)JOB_CHUNK * 8 : (uint64_t)std::min<uint32_t>(JOB_CHUNK, hix.lists[j.list].card) * 4;
        time_kernel(B200_K_SCATTER, m0, mark(), bytes);
    }
    CU(cudaMemcpyAsync(out, base + o_col, W * 8, cudaMemcpyDeviceToHost, stream), "D2H column");
    CU(cudaStreamSynchronize(stream), "sync");
    resolve_timers();
    // scatter_kernel does not consult the universe for sparse lists (inside the engine the DP masks with it): apply it here
    for (uint64_t w = 0; w < W; w++) out[w] &= universe ? universe[w] : hix.base_ub[w];
    stats.h2d_bytes += (universe ? W * 8 : 0) + jobs.size() * sizeof(Job) + sizeof a;
    stats.d2h_bytes += W * 8;
    return B200_OK;
}

// S2 for proximity conditions: what ProximityGraph::resolve_condition (ranking_rule_graph/proximity/compute_docids.rs:15-108)
// unions for one edge — every (l, r) of two word sets looked up forwards at proximity `fwd_prox` and backwards (r, l) at
// `bwd_prox` (0 = no lookup in that direction) in word_pair_proximity_docids — restricted to a universe.  pair_probe_kernel
// resolves the key probes against the staged key directory, scatter_kernel ORs the lists it found.
int Engine::proximity_pairs(const uint32_t *left, uint32_t n_left, const uint32_t *right, uint32_t n_right, uint32_t fwd_prox, uint32_t bwd_prox,
                            const uint64_t *universe, uint64_t n_universe_words, uint64_t *out) {
    if (!staged) return fail(B200_ERR_STATE, "proximity_pairs before b200_stage_finish");
    if (fwd_prox > 3 || bwd_prox > 3) return fail(B200_ERR_INVALID, "proximity_pairs: proximities are 0 (none) .. 3");
    CU(cudaSetDevice(device), "cudaSetDevice");
    const uint64_t W = hix.n_words64;
    if (universe && n_universe_words < W) return fail(B200_ERR_INVALID, "proximity_pairs: universe bitmap shorter than the document range");
    for (uint32_t i = 0; i < n_left; i++)
        if (left[i] >= hix.n_words) return fail(B200_ERR_INVALID, "proximity_pairs: word id out of range");
    for (uint32_t i = 0; i < n_right; i++)
        if (right[i] >= hix.n_words) return fail(B200_ERR_INVALID, "proximity_pairs: word id out of range");
    const uint64_t n_probes = (uint64_t)n_left * n_right;
    if (n_probes == 0 || (fwd_prox == 0 && bwd_prox == 0)) {
        memset(out, 0, W * 8);
        return B200_OK;
    }
    if (n_probes > (1u << 26)) return fail(B200_ERR_CAPACITY, "proximity_pairs: more than 2^26 word pairs in one call");
    const size_t qcap = std::max<size_t>((size_t)1 << 16, (size_t)n_probes * 4);
    const size_t o_ub = 0, o_col = o_ub + W * 8, o_act = (o_col + W * 8 + 255) & ~(size_t)255, o_res = o_act + ((sizeof(ActDesc) + 255) & ~(size_t)255),
                 o_set = o_res + 256, o_words = o_set + 256, o_queue = (o_words + ((size_t)n_left + n_right) * 4 + 255) & ~(size_t)255,
                 o_bigq = o_queue + qcap * sizeof(Job), total = o_bigq + qcap * 4;
    CU(d_s2.reserve(total), "alloc S2 scratch");
    uint8_t *base = d_s2.p;
    if (universe)
        CU(cudaMemcpyAsync(base + o_ub, universe, W * 8, cudaMemcpyHostToDevice, stream), "H2D universe");
    else
        CU(cudaMemcpyAsync(base + o_ub, dix.base_ub, W * 8, cudaMemcpyDeviceToDevice, stream), "universe");
    CU(cudaMemsetAsync(base + o_col, 0, W * 8, stream), "zero column");
    ActDesc a;
    memset(&a, 0, sizeof a);
    a.ub = reinterpret_cast<unsigned long long *>(base + o_ub);
    a.C = reinterpret_cast<unsigned long long *>(base + o_col);
    a.ld = (uint32_t)W;
    a.n_cols = 1;
    uint32_t counters[16] = {(uint32_t)W};  // results[0] = rows | qcount at +16: [0] jobs, [2] scatter cursor
    PairSet ps{};
    ps.left_off = 0;
    ps.n_left = n_left;
    ps.right_off = n_left;
    ps.n_right = n_right;
    ps.fwd_prox = (uint8_t)fwd_prox;
    ps.bwd_prox = (uint8_t)bwd_prox;
    CU(cudaMemcpyAsync(base + o_act, &a, sizeof a, cudaMemcpyHostToDevice, stream), "H2D activation");
    CU(cudaMemcpyAsync(base + o_res, counters, sizeof counters, cudaMemcpyHostToDevice, stream), "H2D counters");
    CU(cudaMemcpyAsync(base + o_set, &ps, sizeof ps, cudaMemcpyHostToDevice, stream), "H2D pair set");
    CU(cudaMemcpyAsync(base + o_words, left, (size_t)n_left * 4, cudaMemcpyHostToDevice, stream), "H2D words");
    CU(cudaMemcpyAsync(base + o_words + (size_t)n_left * 4, right, (size_t)n_right * 4, cudaMemcpyHostToDevice, stream), "H2D words");
    uint32_t *d_res = reinterpret_cast<uint32_t *>(base + o_res), *d_qcount = d_res + 4;
    size_t m0 = mark();
    CU(launch_pair_probe(stream, reinterpret_cast<const PairSet *>(base + o_set), 1, (uint32_t)n_probes, reinterpret_cast<const uint32_t *>(base + o_words),
                         dix.pair_keys, hix.pair_keys.size(), hix.pair_list_base, dix.lists, reinterpret_cast<const ActDesc *>(base + o_act), d_res,
                         reinterpret_cast<Job *>(base + o_queue), d_qcount, (uint32_t)qcap),
       "pair probe");
    size_t m1 = mark();
    time_kernel(B200_K_PAIR_PROBE, m0, m1, n_probes * 8 * 23);
    CU(launch_scatter(stream, (uint32_t)sm_count * 5, reinterpret_cast<const Job *>(base + o_queue), d_qcount, (uint32_t)qcap,
                      reinterpret_cast<const ActDesc *>(base + o_act), d_res, dix.lists, dix.pool, reinterpret_cast<uint32_t *>(base + o_bigq)),
       "scatter");
    time_kernel(B200_K_SCATTER, m1, mark(), 0);
    uint32_t h_counts[8];
    CU(cudaMemcpyAsync(h_counts, d_res, sizeof h_counts, cudaMemcpyDeviceToHost, stream), "D2H counters");
    CU(cudaMemcpyAsync(out, base + o_col, W * 8, cudaMemcpyDeviceToHost, stream), "D2H column");
    CU(cudaStreamSynchronize(stream), "sync");
    resolve_timers();
    if (h_counts[4] > qcap) return fail(B200_ERR_CAPACITY, "proximity_pairs: job queue overflow");
    for (uint64_t w = 0; w < W; w++) out[w] &= universe ? universe[w] : hix.base_ub[w];
    stats.h2d_bytes += (universe ? W * 8 : 0) + ((size_t)n_left + n_right) * 4 + sizeof a;
    stats.d2h_bytes += W * 8;
    return B200_OK;
}

}  // namespace b200
