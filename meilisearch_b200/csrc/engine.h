// The engine behind the C ABI: staged index in HBM + batched search.
#pragma once
#include <cuda_runtime.h>

#include <chrono>
#include <condition_variable>
#include <functional>
#include <map>
#include <mutex>
#include <thread>
#include <atomic>
#include <memory>
#include <string>
#include <vector>

#include <sched.h>

#include "../../include/b200milli.h"
#include "device_types.h"
#include "host_index.h"
#include "query_model.h"

namespace b200 {

struct DeviceIndex {
    uint8_t *dict_bytes = nullptr;
    uint32_t *dict_off = nullptr;
    uint32_t *pool = nullptr;
    DListRef *lists = nullptr;
    unsigned long long *pair_keys = nullptr;
    unsigned long long *base_ub = nullptr;
    // embeddings
    void *emb = nullptr;  // __half[n][d]
    float *emb_inv_norm = nullptr;
    uint32_t *emb_docids = nullptr;
    uint64_t emb_n = 0;
    uint32_t emb_d = 0;
};

template <class T>
struct DevBuf {  // grow-only device buffer
    T *p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = n + n / 4 + 64;
        cudaError_t e = cudaMalloc((void **)&p, want * sizeof(T));
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

// Persistent worker pool: the per-step host work (one bucket-sort advance per query) is a parallel-for.  Steps arrive every
// few hundred microseconds, so idle workers spin briefly on the generation counter before they block.
struct WorkerPool {
    std::vector<std::thread> threads;
    std::mutex mu;
    std::condition_variable cv_work;
    std::function<void(size_t)> fn;
    // run(): announce (generation++), wait until no worker is still inside the previous job (entered == left), publish the job,
    // set ready = generation.  A worker touches fn/n/next only between entered++ and left++ and only after re-checking that no
    // newer job has been announced, so a late waker can never claim an index of a job it did not observe.
    std::atomic<size_t> next{0}, generation{0}, ready{0}, remaining{0}, entered{0}, left{0};
    size_t n = 0;
    std::atomic<bool> stop{false};
    // how long an idle worker spins before it blocks (B200_POOL_SPIN_US; several ranks sharing one host want it short)
    long spin_us = getenv("B200_POOL_SPIN_US") ? std::max(0, atoi(getenv("B200_POOL_SPIN_US"))) : 300;
    explicit WorkerPool(unsigned nt) {
        for (unsigned t = 0; t < nt; t++)
            threads.emplace_back([this]() {
                size_t seen = 0;
                for (;;) {
                    // spin ~300 us, then sleep
                    bool got = false;
                    auto t0 = std::chrono::steady_clock::now();
                    for (int spin = 0;; spin++) {
                        if (stop.load(std::memory_order_acquire)) return;
                        if (ready.load(std::memory_order_acquire) != seen) {
                            got = true;
                            break;
                        }
                        if ((spin & 63) == 63 && std::chrono::steady_clock::now() - t0 > std::chrono::microseconds(spin_us)) break;
#if defined(__x86_64__)
                        __builtin_ia32_pause();
#endif
                    }
                    if (!got) {
                        std::unique_lock<std::mutex> lk(mu);
                        cv_work.wait(lk, [&] { return stop.load() || ready.load() != seen; });
                        if (stop.load()) return;
                    }
                    const size_t g = ready.load(std::memory_order_acquire);
                    entered.fetch_add(1, std::memory_order_acq_rel);
                    if (generation.load(std::memory_order_acquire) == g) {
                        for (;;) {
                            size_t i = next.fetch_add(1);
                            if (i >= n) break;
                            fn(i);
                            remaining.fetch_sub(1, std::memory_order_acq_rel);
                        }
                    }
                    left.fetch_add(1, std::memory_order_acq_rel);
                    seen = g;
                }
            });
    }
    void run(size_t count, std::function<void(size_t)> f) {
        if (count == 0) return;
        if (threads.empty() || count < 4) {
            for (size_t i = 0; i < count; i++) f(i);
            return;
        }
        const size_t g = generation.fetch_add(1, std::memory_order_acq_rel) + 1;
        while (entered.load(std::memory_order_acquire) != left.load(std::memory_order_acquire)) {
#if defined(__x86_64__)
            __builtin_ia32_pause();
#endif
        }
        {
            std::lock_guard<std::mutex> lk(mu);
            fn = std::move(f);
            n = count;
            next.store(0);
            remaining.store(count);
            ready.store(g, std::memory_order_release);
        }
        cv_work.notify_all();
        // the caller works too
        for (;;) {
            size_t i = next.fetch_add(1);
            if (i >= count) break;
            fn(i);
            remaining.fetch_sub(1, std::memory_order_acq_rel);
        }
        while (remaining.load(std::memory_order_acquire) != 0) {
#if defined(__x86_64__)
            __builtin_ia32_pause();
#endif
        }
    }
    ~WorkerPool() {
        {
            std::lock_guard<std::mutex> lk(mu);
            stop.store(true);
        }
        cv_work.notify_all();
        for (auto &t : threads) t.join();
    }
};

// Host-side first-fit allocator over a lane's slice of the device arena.  Blocks are the persistent buffers of one ranking-rule
// level (universe rows + bucket columns); they are returned when bucket_sort leaves the level, so the live set follows the
// depth-first descent of the queries instead of growing for the whole batch.
struct ArenaAlloc {
    std::map<size_t, size_t> free_;  // offset -> length, non-adjacent
    size_t total = 0, used = 0, peak = 0;
    void reset(size_t bytes) {
        free_.clear();
        total = bytes;
        used = peak = 0;
        if (bytes) free_[0] = bytes;
    }
    size_t take(size_t bytes) {  // SIZE_MAX when nothing fits
        bytes = (bytes + 255) & ~(size_t)255;
        for (auto it = free_.begin(); it != free_.end(); ++it)
            if (it->second >= bytes) {
                size_t off = it->first, rest = it->second - bytes;
                free_.erase(it);
                if (rest) free_[off + bytes] = rest;
                used += bytes;
                peak = std::max(peak, used);
                return off;
            }
        return SIZE_MAX;
    }
    void give(size_t off, size_t bytes) {
        bytes = (bytes + 255) & ~(size_t)255;
        used -= bytes;
        auto nx = free_.lower_bound(off);
        if (nx != free_.end() && off + bytes == nx->first) {
            bytes += nx->second;
            nx = free_.erase(nx);
        }
        if (nx != free_.begin()) {
            auto pv = std::prev(nx);
            if (pv->first + pv->second == off) {
                pv->second += bytes;
                return;
            }
        }
        free_[off] = bytes;
    }
};

// One software-pipeline lane of the step loop: own stream, step buffers, scratch slice and kernel timers.
struct Lane {
    cudaStream_t stream = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    cudaStream_t cls_stream[EVAL_CLASSES + 1] = {};  // eval_dp classes 1.. run beside class 0 (forked from / joined into `stream`)
    cudaEvent_t ev_fork = nullptr, ev_join[EVAL_CLASSES + 1] = {};
    DevBuf<uint8_t> d_step;
    DevBuf<uint32_t> d_results, d_qcount, d_segcount;
    DevBuf<Job> d_queue;
    DevBuf<uint32_t> d_bigq;  // indices of the step's big scatter jobs (scatter_kernel -> scatter_big_kernel)
    DevBuf<PathOut> d_pathbuf;
    DevBuf<unsigned long long> d_tile_summary;  // 2 u64 per eval tile: its non-empty buckets (eval_dp_kernel -> walk_kernel)
    uint8_t *h_step = nullptr;
    size_t h_step_cap = 0;
    uint32_t *h_results = nullptr;
    size_t h_results_cap = 0;
    uint8_t *scratch = nullptr;
    size_t scratch_bytes = 0;
    std::vector<uint32_t> members, act_q;
    // a lane is driven by its own host thread with its own slice of the workers, of the arena and of the statistics
    WorkerPool *pool = nullptr;  // the pool of the lane's driver (shared by the lanes that driver alternates between)
    uint8_t *arena = nullptr;
    size_t arena_bytes = 0;
    ArenaAlloc alloc;
    b200_stats lst{};
    int rc = 0;
    std::string error;
    uint32_t res_words = 0;
    size_t qcap = 0;
    bool inflight = false;
    struct Timed {
        int cls;
        size_t a, b;
    };
    std::vector<cudaEvent_t> ev_pool;
    std::vector<Timed> timed;
    size_t ev_used = 0;
    bool timing = true;  // per-kernel CUDA-event timing (B200_KERNEL_TIMERS=0 turns the ~10 event records per step off)
    size_t mark() {
        if (!timing) return 0;
        if (ev_used == ev_pool.size()) {
            cudaEvent_t e;
            cudaEventCreate(&e);
            ev_pool.push_back(e);
        }
        cudaEventRecord(ev_pool[ev_used], stream);
        return ev_used++;
    }
    void time_kernel(b200_stats &st, int cls, size_t a, size_t b, uint64_t bytes) {
        if (timing) timed.push_back(Timed{cls, a, b});
        st.kernel_count[cls]++;
        st.kernel_bytes[cls] += bytes;
        st.kernel_launches++;
    }
    void resolve_timers(b200_stats &st) {
        for (auto &t : timed) {
            float ms = 0;
            if (cudaEventElapsedTime(&ms, ev_pool[t.a], ev_pool[t.b]) == cudaSuccess) st.kernel_ms[t.cls] += ms;
        }
        timed.clear();
        ev_used = 0;
    }
    void release() {
        d_step.release();
        d_results.release();
        d_qcount.release();
        d_queue.release();
        d_segcount.release();
        d_pathbuf.release();
        d_tile_summary.release();
        d_bigq.release();
        if (h_step) cudaFreeHost(h_step);
        if (h_results) cudaFreeHost(h_results);
        for (auto e : ev_pool) cudaEventDestroy(e);
        if (e0) cudaEventDestroy(e0);
        if (e1) cudaEventDestroy(e1);
        if (ev_fork) cudaEventDestroy(ev_fork);
        for (auto e : ev_join)
            if (e) cudaEventDestroy(e);
        for (auto cs : cls_stream)
            if (cs) cudaStreamDestroy(cs);
        if (stream) cudaStreamDestroy(stream);
    }
};

// a stream with its own pool of timing events (the vector stage runs beside the keyword stage in hybrid searches)
struct TimerSet {
    cudaStream_t stream = nullptr;
    std::vector<cudaEvent_t> ev_pool;
    struct Timed {
        int cls;
        size_t a, b;
    };
    std::vector<Timed> timed;
    size_t ev_used = 0;
    size_t mark() {
        if (ev_used == ev_pool.size()) {
            cudaEvent_t e;
            cudaEventCreate(&e);
            ev_pool.push_back(e);
        }
        cudaEventRecord(ev_pool[ev_used], stream);
        return ev_used++;
    }
    void time_kernel(b200_stats &st, int cls, size_t a, size_t b, uint64_t bytes) {
        timed.push_back(Timed{cls, a, b});
        st.kernel_count[cls]++;
        st.kernel_bytes[cls] += bytes;
        st.kernel_launches++;
    }
    void resolve(b200_stats &st) {
        for (auto &t : timed) {
            float ms = 0;
            if (cudaEventElapsedTime(&ms, ev_pool[t.a], ev_pool[t.b]) == cudaSuccess) st.kernel_ms[t.cls] += ms;
        }
        timed.clear();
        ev_used = 0;
    }
};

// NCCL, bound at run time (dlopen of libnccl.so.2: inside a torch process that is the copy torch already loaded): the library only
// needs it when the corpus is partitioned across GPUs (SURVEY §8(e): one all-gather of the per-shard top-k)
struct ShardComm {
    void *lib = nullptr;
    void *comm = nullptr;  // ncclComm_t
    int rank = 0, world = 1;
    int (*get_unique_id)(void *) = nullptr;
    int (*comm_init_rank)(void **, int, struct NcclId, int) = nullptr;
    int (*all_gather)(const void *, void *, size_t, int, void *, cudaStream_t) = nullptr;
    int (*group_start)() = nullptr;
    int (*group_end)() = nullptr;
    int (*comm_destroy)(void *) = nullptr;
    const char *(*get_error_string)(int) = nullptr;
};
struct NcclId {
    char internal[128];
};

struct GraphObj;  // S1: opaque query graph (engine_search.cpp)
struct S1Job;
void free_graph(GraphObj *);

// The host side of a search is a few dozen threads working on the same per-query state.  On a two-socket host it is ~13 % faster
// (cfg 3, measured) when all of them sit on the socket the GPU hangs off, so a search call narrows the calling thread's affinity to
// that NUMA node for its duration — the threads it creates inherit it — and restores it on return.  B200_PIN=0 turns this off;
// nothing happens either when sysfs does not name a node for the device or the process is not allowed on any of its CPUs.
struct HostAffinity {
    cpu_set_t cpus;
    bool valid = false;
    void detect(int device);
};
struct AffinityScope {
    cpu_set_t old;
    bool active = false;
    explicit AffinityScope(const HostAffinity &a) {
        if (!a.valid || sched_getaffinity(0, sizeof old, &old) != 0) return;
        active = sched_setaffinity(0, sizeof a.cpus, &a.cpus) == 0;
    }
    ~AffinityScope() {
        if (active) sched_setaffinity(0, sizeof old, &old);
    }
    AffinityScope(const AffinityScope &) = delete;
    AffinityScope &operator=(const AffinityScope &) = delete;
};

struct Engine {
    std::unique_ptr<WorkerPool> pool;
    std::vector<std::thread> reapers;  // free the previous batch's per-query state in the background (several: one thread cannot
                                       // free a batch's worth of small allocations within the next batch's time)
    static constexpr unsigned MAX_LANES = 8, MAX_DRIVERS = 4;
    Lane lanes[MAX_LANES];
    std::unique_ptr<WorkerPool> driver_pools[MAX_DRIVERS];
    int device = 0;
    HostAffinity affinity;
    cudaStream_t stream = nullptr;
    std::mutex mu;
    std::string last_error;
    // staging inputs
    std::vector<uint8_t> raw_dict_bytes;
    std::vector<uint64_t> raw_dict_off;
    RawDb raw_dbs[10];
    std::vector<uint8_t> raw_docids;
    bool staged = false;
    HostIndex hix;
    DeviceIndex dix;
    std::vector<uint64_t> emb_bitmap;  // documents owning at least one embedding
    uint32_t emb_d_user = 0;           // the caller's embedding dimension (rows are zero-padded to a multiple of 8 on the device)
    bool has_distribution = false;
    float dist_mean = 0, dist_sigma = 0;
    b200_stats stats{};
    // hybrid: derivation waves the keyword stage has finished (KW_DERIVED_ALL after the last one); the vector stage waits for
    // VEC_START_DEFAULT of them
    static constexpr int KW_DERIVED_ALL = 1 << 20, VEC_START_DEFAULT = 1;
    std::atomic<int> kw_derived{0};
    TimerSet vt;          // vector stage: own stream and timers
    b200_stats vstats{};  // what the vector stage accumulated since it was last folded into `stats`
    void fold_vector_stats() {
        stats.kernel_launches += vstats.kernel_launches;
        stats.vector_bytes += vstats.vector_bytes;
        stats.h2d_bytes += vstats.h2d_bytes;
        stats.d2h_bytes += vstats.d2h_bytes;
        for (int k = 0; k < B200_K_COUNT; k++) {
            stats.kernel_ms[k] += vstats.kernel_ms[k];
            stats.kernel_count[k] += vstats.kernel_count[k];
            stats.kernel_bytes[k] += vstats.kernel_bytes[k];
        }
        vstats = b200_stats{};
    }
    int sm_count = 148;
    // pools
    uint8_t *arena = nullptr;
    size_t arena_bytes = 0;
    uint8_t *scratch = nullptr;
    size_t scratch_bytes = 0;
    DevBuf<uint8_t> d_step;     // per-step input blob
    DevBuf<uint32_t> d_results; // per-step results
    DevBuf<Job> d_queue;
    DevBuf<uint32_t> d_qcount;   // [0] scatter jobs, [1] surviving paths
    DevBuf<PathOut> d_pathbuf;
    DevBuf<uint32_t> d_docids_out;  // n_queries x limit
    DevBuf<unsigned long long> d_universes;  // the batch's distinct filtered universes (documents_ids & filter), n_words64 words each
    DevBuf<uint32_t> d_rowtab;      // n_queries x n_words64: word -> (tag, row) of the query's current activation (ActDesc::row_tab)
    uint8_t *h_step = nullptr;      // pinned
    size_t h_step_cap = 0;
    uint32_t *h_results = nullptr;  // pinned
    size_t h_results_cap = 0;
    // lev buffers
    DevBuf<LevTerm> d_lev_terms;
    DevBuf<LevRec> d_lev_recs;
    DevBuf<uint32_t> d_lev_u32;  // rec_count | one_out | n_one | two_out | n_two | status
    DevBuf<uint32_t> d_lev_sched;  // derivation schedule: LevItem[] | LevChunk[] | term indices
    // vector buffers
    DevBuf<float> d_vq, d_vdist, d_vsel_dist;
    DevBuf<uint32_t> d_vsel_ids, d_vsel_n;
    DevBuf<unsigned long long> d_cand, d_vruns, d_vpartial;
    DevBuf<uint16_t> d_vq16;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::vector<cudaEvent_t> ev_pool;  // pairs recorded around kernels, resolved after the step's sync
    struct Timed { int cls; size_t a, b; };
    std::vector<Timed> timed;
    size_t ev_used = 0;
    // record an event (from the pool) on the stream; returns its index
    size_t mark();
    void time_kernel(int cls, size_t a, size_t b, uint64_t bytes) {
        timed.push_back(Timed{cls, a, b});
        stats.kernel_count[cls]++;
        stats.kernel_bytes[cls] += bytes;
        stats.kernel_launches++;
    }
    void resolve_timers();  // after a stream sync

    std::mutex err_mu;  // lanes report errors from their own threads
    int fail(int code, const std::string &msg) {
        std::lock_guard<std::mutex> g(err_mu);
        last_error = msg;
        return code;
    }
    int cuda_fail(cudaError_t e, const char *what) { return fail(B200_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e)); }

    int stage_finish();
    int stage_embeddings(const float *vectors, const uint16_t *half_rows, uint64_t n, uint32_t d, const uint32_t *docids);
    int derive_batch(uint32_t n, const char *words, const uint32_t *off, const uint8_t *max_typo, const uint8_t *is_prefix, uint32_t *one_out,
                     uint32_t *n_one, uint32_t *two_out, uint32_t *n_two);
    // sharded: every rank passes the same queries and scans its own rows; the per-shard top-k lists are all-gathered (NCCL, on the
    // vector stream) and merged on the device; every rank returns the merged result
    int nns_batch(const float *queries, uint32_t n_q, uint32_t d, uint32_t limit, const uint64_t *cand, uint64_t n_cand_words, uint32_t *ids_out,
                  float *dist_out, uint32_t *n_out, bool sharded = false);
    ShardComm sc;
    DevBuf<float> d_vpart_dist;  // sliced top-k selection: per-slice candidates
    DevBuf<uint32_t> d_vpart_ids, d_vpart_n;
    DevBuf<uint32_t> d_gather_ids, d_gather_n;
    DevBuf<float> d_gather_dist;
    int comm_load();
    int comm_init(int rank, int world, const uint8_t *unique_id);
    int search_batch(const b200_query_batch *b, b200_results *r);
    int union_postings(int db, const uint32_t *key_index, uint32_t n_keys, const uint64_t *universe, uint64_t n_universe_words, uint64_t *out);
    DevBuf<uint8_t> d_s2;  // S2 scratch: universe | column | ActDesc | jobs | counters
    int keyword_batch(const b200_query_batch *b, b200_results *r, uint32_t offset, uint32_t limit, int scoring, S1Job *s1 = nullptr);
    // S1 (RankingRule seam): see include/b200milli.h
    int graph_from_tokens(const b200_query_batch *one_query, GraphObj **out);
    struct RuleRun;
    int rule_start(int rule_kind, int tms, const GraphObj *query, const uint64_t *universe, uint64_t n_universe_words, RuleRun **out);
    // S2 for proximity conditions
    int proximity_pairs(const uint32_t *left, uint32_t n_left, const uint32_t *right, uint32_t n_right, uint32_t fwd_prox, uint32_t bwd_prox,
                        const uint64_t *universe, uint64_t n_universe_words, uint64_t *out);
    int semantic_batch(const b200_query_batch *b, b200_results *r, uint32_t offset, uint32_t limit);
    ~Engine();
};

}  // namespace b200
