// CUDA kernels for sm_100a.  HBM/L2-bound integer work: 128-bit coalesced loads where rows are streamed,
// warp shuffles/ballots for reductions and ordered compaction, no tensor cores (DESIGN.md §4).
//
//   lev_match_kernel / lev_finalize_kernel   term derivation: Levenshtein(<=2, transposition) x dictionary
//   act_compact_kernel                       child universe = non-zero words of a parent bucket
//   pair_probe_kernel                        (prox,w1,w2) directory probes -> scatter jobs
//   scatter_kernel                           posting lists -> condition bit-matrix columns
//   eval_dp_kernel                           column program + bit-sliced DP over the rule graph -> buckets + surviving paths
//   emit_kernel                              bucket -> first-k docids, ascending
//   vec_dist_kernel / topk_*                 cosine distance scan + exact top-k
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <cstdint>

#include "device_types.h"
#include "kernels.h"

#include <algorithm>

namespace b200 {

// ======================================================================================== lev
// Banded restricted Damerau-Levenshtein: returns min(distance, k+1).  prefix: min over prefixes of w.
__device__ __forceinline__ int banded_osa(const uint8_t *q, int m, const uint8_t *w, int n, int k, bool prefix) {
    const int INF = k + 1;
    // column j holds D[i][j] for i = j + b - k, b in [0, 2k]
    int c2[5], c1[5], c0[5];
#pragma unroll
    for (int b = 0; b < 5; b++) {
        int i = b - k;
        c1[b] = (b <= 2 * k && i >= 0 && i <= m) ? (i < INF ? i : INF) : INF;
        c2[b] = INF;
    }
    int best = INF;
    if (prefix && m <= k) best = m;  // empty prefix (never happens for words long enough to have typos)
    int jmax = n;
    if (jmax > m + k) jmax = m + k;
    if (!prefix && (n > m + k || n < m - k)) return INF;
    if (prefix && n < m - k) return INF;
    for (int j = 1; j <= jmax; j++) {
        uint8_t wc = w[j - 1];
        uint8_t wp = j > 1 ? w[j - 2] : 0;
        int rowmin = INF;
#pragma unroll
        for (int b = 0; b < 5; b++) {
            int v = INF;
            if (b <= 2 * k) {
                int i = j + b - k;
                if (i >= 0 && i <= m) {
                    if (i == 0)
                        v = j;
                    else {
                        int del = (b > 0) ? c0[b - 1] + 1 : INF;              // D[i-1][j] + 1
                        int ins = (b < 2 * k) ? c1[b + 1] + 1 : INF;          // D[i][j-1] + 1
                        int sub = c1[b] + (q[i - 1] != wc ? 1 : 0);           // D[i-1][j-1] + cost
                        v = min(del, min(ins, sub));
                        if (i > 1 && j > 1 && q[i - 1] == wp && q[i - 2] == wc) v = min(v, c2[b] + 1);  // D[i-2][j-2] + 1
                    }
                    if (v > INF) v = INF;
                }
            }
            c0[b] = v;
            rowmin = min(rowmin, v);
        }
        if (prefix) {
            int b = m - j + k;
            if (b >= 0 && b <= 2 * k) best = min(best, c0[b]);
        }
#pragma unroll
        for (int b = 0; b < 5; b++) {
            c2[b] = c1[b];
            c1[b] = c0[b];
        }
        if (rowmin >= INF && !prefix) {
            // both this and (via c2) an earlier column may still matter for a transposition; stop only when two columns are dead
            int m2 = INF;
#pragma unroll
            for (int b = 0; b < 5; b++) m2 = min(m2, c2[b]);
            if (m2 >= INF) return INF;
        }
    }
    if (prefix) return best;
    int b = m - n + k;
    return (b >= 0 && b <= 2 * k) ? c1[b] : INF;
}

// Character-class signature: bit (c & 31) for every byte.  If OSA(q, w) <= k then at most k classes of q are missing from w
// (every edit removes at most one class; a transposition none), and — outside prefix mode — vice versa.  Sound with collisions.
__device__ __forceinline__ uint32_t char_signature(const uint8_t *s, int n) {
    uint32_t m = 0;
    for (int i = 0; i < n; i++) m |= 1u << (s[i] & 31);
    return m;
}

// One CTA per schedule item = (chunk of <= LEV_TERMS_PER_CTA terms of one group, one 256-word tile of the dictionary).
// Words of the tile outside the group's word set (device_types.h) are skipped before any test; the rest go through the full
// filter, first-letter rule included.  Two phases per group of 8 terms: (1) every thread filters its word against the 8 terms (length,
// first-letter rule, signature) and queues the surviving (term, word) pairs in shared memory; (2) the queue is processed densely,
// one banded DP per thread — the DP, which is the expensive part, runs on a few percent of the pairs and without divergence
// between matching and non-matching lanes.  Match codes are collected per (term, 32-word group) and reported as ballot records.
constexpr int LEV_TERM_GROUP = 8;
__global__ void __launch_bounds__(256) lev_match_kernel(const uint8_t *__restrict__ dict_bytes, const uint32_t *__restrict__ dict_off,
                                                        uint32_t n_words, const LevTerm *__restrict__ terms,
                                                        const uint32_t *__restrict__ term_idx, const LevChunk *__restrict__ chunks,
                                                        const LevItem *__restrict__ items, LevRec *__restrict__ recs,
                                                        uint32_t *__restrict__ rec_count) {
    __shared__ LevTerm sterms[LEV_TERMS_PER_CTA];
    __shared__ uint32_t sterm_sig[LEV_TERMS_PER_CTA], sterm_meta[LEV_TERMS_PER_CTA], sterm_id[LEV_TERMS_PER_CTA];
    __shared__ uint8_t sbytes[8192];
    __shared__ uint16_t s_woff[257];
    __shared__ uint32_t s_queue[LEV_TERM_GROUP * 256];  // (term << 16) | word-in-tile | (same-first << 31)
    __shared__ uint32_t s_qn;
    __shared__ unsigned long long s_codes[LEV_TERM_GROUP][8];
    const LevItem item = items[blockIdx.x];
    const LevChunk ch = chunks[item.chunk];
    const uint32_t nt = ch.n;
    uint32_t w0 = item.tile * 256;
    uint32_t wn = min(256u, n_words - w0);
    uint32_t byte0 = dict_off[w0], byte1 = dict_off[w0 + wn];
    bool in_smem = (byte1 - byte0) <= sizeof(sbytes);
    if (in_smem) {
        for (uint32_t i = threadIdx.x; i < byte1 - byte0; i += blockDim.x) sbytes[i] = dict_bytes[byte0 + i];
        for (uint32_t i = threadIdx.x; i <= wn; i += blockDim.x) s_woff[i] = (uint16_t)(dict_off[w0 + i] - byte0);
    }
    if (threadIdx.x < nt) sterm_id[threadIdx.x] = term_idx[ch.first + threadIdx.x];
    __syncthreads();
    {
        constexpr uint32_t WORDS = sizeof(LevTerm) / 4;
        uint32_t *dst = reinterpret_cast<uint32_t *>(sterms);
        for (uint32_t i = threadIdx.x; i < nt * WORDS; i += blockDim.x)
            dst[i] = reinterpret_cast<const uint32_t *>(terms + sterm_id[i / WORDS])[i % WORDS];
    }
    uint32_t wid = w0 + threadIdx.x;
    bool valid = threadIdx.x < wn;
    uint32_t off = valid ? dict_off[wid] : byte0;
    int n = valid ? (int)(dict_off[wid + 1] - off) : 0;
    const uint8_t *w = in_smem ? (sbytes + (off - byte0)) : (dict_bytes + off);
    uint8_t w0c = n > 0 ? w[0] : 0, w1c = n > 1 ? w[1] : 0;
    // the part of the group's word set that is the same for every term of the chunk
    if (ch.kind == LEV_GROUP_F) valid = valid && w0c == ch.c;
    if (ch.kind == LEV_GROUP_S) valid = valid && w1c == ch.c;
    const uint32_t wsig = char_signature(w, n);
    __syncthreads();
    if (threadIdx.x < nt) {
        const LevTerm &T = sterms[threadIdx.x];
        sterm_sig[threadIdx.x] = char_signature(T.q, T.len);
        sterm_meta[threadIdx.x] = (uint32_t)T.len | ((uint32_t)(T.k_same + 1) << 8) | ((uint32_t)(T.k_diff + 1) << 12) |
                                  ((uint32_t)(T.prefix ? 1 : 0) << 16) | ((uint32_t)T.q[0] << 24);
    }
    for (uint32_t tg = 0; tg < nt; tg += LEV_TERM_GROUP) {
        const uint32_t ng = min((uint32_t)LEV_TERM_GROUP, nt - tg);
        if (threadIdx.x == 0) s_qn = 0;
        if (threadIdx.x < LEV_TERM_GROUP * 8) s_codes[threadIdx.x >> 3][threadIdx.x & 7] = 0;
        __syncthreads();
        // phase 1: filter, most selective test first (the signature rejects ~95 % of the pairs with two shared-memory loads)
        if (valid && n > 0) {
            for (uint32_t t = 0; t < ng; t++) {
                // S(c): the words whose first byte is q[0] or q[1] of this term belong to its F groups
                if (ch.kind == LEV_GROUP_S && (w0c == sterms[tg + t].q[0] || w0c == sterms[tg + t].q[1])) continue;
                const uint32_t tsig = sterm_sig[tg + t];
                const uint32_t meta = sterm_meta[tg + t];  // len | (k_same+1) << 8 | (k_diff+1) << 12 | prefix << 16 | q0 << 24
                const int kmax = (int)((meta >> 8) & 15) - 1;
                if (__popc(tsig & ~wsig) > kmax) continue;
                const bool prefix = (meta >> 16) & 1;
                const bool sf = (uint8_t)(meta >> 24) == w0c;
                const int k = sf ? kmax : (int)((meta >> 12) & 15) - 1;
                if (k < 0) continue;
                const int m = (int)(meta & 255);
                bool ok = prefix ? (n >= m - k) : (n >= m - k && n <= m + k);
                ok = ok && __popc(tsig & ~wsig) <= k && (prefix || __popc(wsig & ~tsig) <= k);
                // different first char at distance <= 1: the single edit sits on the first position
                if (ok && !sf && m >= 2) {
                    const LevTerm &T = sterms[tg + t];
                    ok = (w1c == T.q[1]) || (w1c == T.q[0]) || (w0c == T.q[1]);
                }
                if (ok) s_queue[atomicAdd(&s_qn, 1u)] = (t << 16) | threadIdx.x | (sf ? 0x80000000u : 0u);
            }
        }
        __syncthreads();
        // phase 2: dense DP over the queue
        const uint32_t qn = s_qn;
        for (uint32_t i = threadIdx.x; i < qn; i += blockDim.x) {
            const uint32_t e = s_queue[i];
            const uint32_t t = (e >> 16) & 0x7fff, wi = e & 0xffff;
            const bool sf = (e >> 31) != 0;
            const LevTerm &T = sterms[tg + t];
            const int k = sf ? T.k_same : T.k_diff;
            const uint8_t *ww;
            int wl;
            if (in_smem) {
                ww = sbytes + s_woff[wi];
                wl = (int)s_woff[wi + 1] - (int)s_woff[wi];
            } else {
                uint32_t o = dict_off[w0 + wi];
                ww = dict_bytes + o;
                wl = (int)(dict_off[w0 + wi + 1] - o);
            }
            int d = banded_osa(T.q, T.len, ww, wl, k, T.prefix != 0);
            if (d <= k && d > 0) {
                unsigned long long code = sf ? (unsigned long long)d : 3ull;
                atomicOr(&s_codes[t][wi >> 5], code << (2 * (wi & 31)));
            }
        }
        __syncthreads();
        // report: one record per (term, 32-word group) holding at least one match; another item of the same term may report
        // other words of the same 32-word group (lev_finalize_kernel merges them)
        if (threadIdx.x < ng * 8) {
            const uint32_t t = threadIdx.x >> 3, g = threadIdx.x & 7;
            const unsigned long long codes = s_codes[t][g];
            if (codes) {
                const uint32_t term = sterm_id[tg + t];
                uint32_t slot = atomicAdd(&rec_count[term], 1u);
                if (slot < LEV_REC_CAP) {
                    LevRec r;
                    r.base = w0 + g * 32;
                    r.pad = 0;
                    r.codes = codes;
                    recs[(size_t)term * LEV_REC_CAP + slot] = r;
                }
            }
        }
        __syncthreads();
    }
}

// One thread per term: order the records by word id and replay the reference's capped, order-dependent
// classification (compute_derivations.rs:89-105, 128-166).
__global__ void lev_finalize_kernel(LevRec *__restrict__ recs, const uint32_t *__restrict__ rec_count, const LevTerm *__restrict__ terms,
                                    uint32_t n_terms, uint32_t *__restrict__ one_out, uint32_t *__restrict__ n_one,
                                    uint32_t *__restrict__ two_out, uint32_t *__restrict__ n_two, int32_t *__restrict__ status) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_terms) return;
    uint32_t cnt = rec_count[t];
    if (cnt > LEV_REC_CAP) {
        status[t] = -5;
        cnt = LEV_REC_CAP;
    } else
        status[t] = 0;
    LevRec *r = recs + (size_t)t * LEV_REC_CAP;
    for (uint32_t i = 1; i < cnt; i++) {  // insertion sort by base
        LevRec x = r[i];
        uint32_t j = i;
        while (j > 0 && r[j - 1].base > x.base) {
            r[j] = r[j - 1];
            j--;
        }
        r[j] = x;
    }
    // records of one 32-word group from different items hold disjoint words: one record per group again
    uint32_t u = 0;
    for (uint32_t i = 0; i < cnt; i++) {
        if (u > 0 && r[u - 1].base == r[i].base)
            r[u - 1].codes |= r[i].codes;
        else
            r[u++] = r[i];
    }
    cnt = u;
    bool two_budget = terms[t].k_same >= 2;
    uint32_t c1 = 0, c2 = 0;
    uint32_t *o1 = one_out + (size_t)t * 150, *o2 = two_out + (size_t)t * 50;
    for (uint32_t i = 0; i < cnt; i++) {
        unsigned long long codes = r[i].codes;
        for (int l = 0; l < 32 && codes; l++, codes >>= 2) {
            int code = (int)(codes & 3);
            if (!code) continue;
            uint32_t wid = r[i].base + l;
            if (!two_budget) {  // find_one_typo_derivations: same first char, d == 1, cap 150
                if (code == 1 && c1 < 150) o1[c1++] = wid;
                continue;
            }
            bool fin1 = c1 >= 150, fin2 = c2 >= 50;
            if (fin1 && fin2) break;
            if (code == 3 && !fin2) {
                o2[c2++] = wid;
                continue;
            }
            int d = (code == 2) ? 2 : 1;  // second_dfa.distance: 1 for a different first char
            if (d == 1) {
                if (!fin1) o1[c1++] = wid;
            } else if (!fin2)
                o2[c2++] = wid;
        }
        if (c1 >= 150 && (c2 >= 50 || !two_budget)) break;
    }
    n_one[t] = c1;
    n_two[t] = c2;
}

// ======================================================================================== activations
// row of 64-document word `w` in an activation's universe, or -1
__device__ __forceinline__ int find_row(const uint32_t *uw, uint32_t rows, uint32_t w);
__device__ __forceinline__ int act_row(const ActDesc &a, uint32_t rows, uint32_t w) {
    if (!a.uw) return w < rows ? (int)w : -1;
    if (a.row_tab) {
        uint32_t e = a.row_tab[w];
        return (e >> 20) == a.row_tag ? (int)(e & 0xfffffu) : -1;
    }
    return find_row(a.uw, rows, w);
}
__device__ __forceinline__ int find_row(const uint32_t *uw, uint32_t rows, uint32_t w) {
    uint32_t lo = 0, hi = rows;
    while (lo < hi) {
        uint32_t mid = (lo + hi) >> 1;
        if (uw[mid] < w)
            lo = mid + 1;
        else
            hi = mid;
    }
    return (lo < rows && uw[lo] == w) ? (int)lo : -1;
}

// Ordered compaction of the parent's non-zero bucket words, split into segments of COMPACT_SEG parent rows (one CTA each) so that a
// 150 k-row parent is compacted by 19 CTAs instead of one.  Pass 1 (act_count_kernel) counts the surviving rows of every segment;
// pass 2 starts each segment at the sum of the earlier segments' counts and compacts it in rounds of 2048 rows (4 per thread, loads
// issued together).
constexpr int COMPACT_THREADS = 512, COMPACT_PER_THREAD = 4;
__device__ __forceinline__ unsigned long long compact_row_value(const ActDesc &a, uint32_t j) {
    if (!a.p_out) return a.p_ub[j];
    unsigned long long v = 0;
    for (uint32_t c = a.p_col_lo; c < a.p_col_hi; c++) v |= a.p_out[(size_t)c * a.p_ld + j];
    return v;
}
__global__ void __launch_bounds__(COMPACT_THREADS) act_count_kernel(const CompactTile *__restrict__ tiles, const ActDesc *__restrict__ acts,
                                                                    uint32_t *__restrict__ seg_count) {
    const CompactTile t = tiles[blockIdx.x];
    const ActDesc &a = acts[t.act];
    if (t.n_seg <= 1) return;  // single segment: pass 2 needs no base
    __shared__ uint32_t warp_sums[COMPACT_THREADS / 32];
    const uint32_t r0 = t.seg * COMPACT_SEG, r1 = min(a.p_rows, r0 + COMPACT_SEG);
    uint32_t c = 0;
    for (uint32_t j0 = r0; j0 < r1; j0 += COMPACT_THREADS * COMPACT_PER_THREAD) {
        unsigned long long v[COMPACT_PER_THREAD];
#pragma unroll
        for (int i = 0; i < COMPACT_PER_THREAD; i++) {
            uint32_t j = j0 + (uint32_t)i * COMPACT_THREADS + threadIdx.x;
            v[i] = j < r1 ? compact_row_value(a, j) : 0ull;
        }
#pragma unroll
        for (int i = 0; i < COMPACT_PER_THREAD; i++) c += v[i] != 0 ? 1u : 0u;
    }
#pragma unroll
    for (int sft = 16; sft > 0; sft >>= 1) c += __shfl_xor_sync(0xffffffffu, c, sft);
    if ((threadIdx.x & 31) == 0) warp_sums[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t tot = 0;
        for (int k = 0; k < COMPACT_THREADS / 32; k++) tot += warp_sums[k];
        seg_count[blockIdx.x] = tot;
    }
}
__global__ void __launch_bounds__(COMPACT_THREADS) act_compact_kernel(const CompactTile *__restrict__ tiles, const ActDesc *__restrict__ acts,
                                                                      const uint32_t *__restrict__ seg_count, uint32_t *__restrict__ results) {
    const CompactTile t = tiles[blockIdx.x];
    const ActDesc a = acts[t.act];
    if (!a.uw) {  // the activation works directly on the dense base universe (row j == word j): nothing to compact
        if (threadIdx.x == 0 && t.seg == 0) results[a.res_off] = a.p_rows;
        return;
    }
    constexpr int NW = COMPACT_THREADS / 32;
    __shared__ uint32_t warp_sums[COMPACT_PER_THREAD][NW];
    __shared__ uint32_t s_before[COMPACT_PER_THREAD][NW];
    __shared__ uint32_t s_total;
    const uint32_t lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
    uint32_t base = 0;
    for (uint32_t sg = 0; sg < t.seg; sg++) base += seg_count[t.first_tile + sg];  // <= a few dozen
    const uint32_t r0 = t.seg * COMPACT_SEG, r1 = min(a.p_rows, r0 + COMPACT_SEG);
    for (uint32_t j0 = r0; j0 < r1; j0 += COMPACT_THREADS * COMPACT_PER_THREAD) {
        unsigned long long v[COMPACT_PER_THREAD];
        uint32_t src[COMPACT_PER_THREAD];
#pragma unroll
        for (int i = 0; i < COMPACT_PER_THREAD; i++) {  // sub-chunk i holds rows j0 + i*512 + tid: ordered by (i, warp, lane)
            uint32_t j = j0 + (uint32_t)i * COMPACT_THREADS + threadIdx.x;
            v[i] = 0;
            src[i] = j;
            if (j < r1) {
                v[i] = compact_row_value(a, j);
                if (a.p_uw) src[i] = a.p_uw[j];
            }
        }
        uint32_t wpre[COMPACT_PER_THREAD];
#pragma unroll
        for (int i = 0; i < COMPACT_PER_THREAD; i++) {
            unsigned m = __ballot_sync(0xffffffffu, v[i] != 0);
            wpre[i] = __popc(m & ((1u << lane) - 1));
            if (lane == 0) warp_sums[i][wrp] = __popc(m);
        }
        __syncthreads();
        if (wrp == 0) {  // exclusive scan of the 64 warp counts in (i, warp) order
            uint32_t x0 = warp_sums[lane / NW][lane % NW], x1 = warp_sums[(lane + 32) / NW][(lane + 32) % NW];
            uint32_t p0 = x0, p1 = x1;
#pragma unroll
            for (int sft = 1; sft < 32; sft <<= 1) {
                uint32_t t0 = __shfl_up_sync(0xffffffffu, p0, sft), t1 = __shfl_up_sync(0xffffffffu, p1, sft);
                if (lane >= (uint32_t)sft) {
                    p0 += t0;
                    p1 += t1;
                }
            }
            uint32_t tot0 = __shfl_sync(0xffffffffu, p0, 31);
            s_before[lane / NW][lane % NW] = p0 - x0;
            s_before[(lane + 32) / NW][(lane + 32) % NW] = tot0 + p1 - x1;
            if (lane == 31) s_total = tot0 + p1;
        }
        __syncthreads();
#pragma unroll
        for (int i = 0; i < COMPACT_PER_THREAD; i++)
            if (v[i] != 0) {
                uint32_t at = base + s_before[i][wrp] + wpre[i];
                if (at < a.ld) {
                    a.uw[at] = src[i];
                    a.ub[at] = v[i];
                    if (a.row_tab) a.row_tab[src[i]] = (a.row_tag << 20) | at;
                }
            }
        base += s_total;
        __syncthreads();
    }
    if (threadIdx.x == 0 && t.seg + 1 == t.n_seg) results[a.res_off] = min(base, a.ld);
}

__device__ __forceinline__ int64_t pair_lower_bound(const unsigned long long *keys, uint64_t n, unsigned long long k) {
    uint64_t lo = 0, hi = n;
    while (lo < hi) {
        uint64_t mid = (lo + hi) >> 1;
        if (keys[mid] < k)
            lo = mid + 1;
        else
            hi = mid;
    }
    return (int64_t)lo;
}

__device__ __forceinline__ void push_list_jobs(Job *queue, uint32_t *qcount, uint32_t qcap, uint32_t act, uint32_t col, uint32_t list,
                                               const DListRef &lr, uint32_t rows_hint) {
    uint32_t units = lr.dense ? rows_hint : lr.card;
    uint32_t nchunks = (units + JOB_CHUNK - 1) / JOB_CHUNK;
    if (nchunks == 0) return;
    uint32_t at = atomicAdd(qcount, nchunks);
    for (uint32_t c = 0; c < nchunks; c++)
        if (at + c < qcap) queue[at + c] = Job{act, col, list, c};
}

// one thread per probe: (pairset, l, r); each probe may look up the forward and the backward key
__global__ void __launch_bounds__(256) pair_probe_kernel(const PairSet *__restrict__ sets, uint32_t n_sets, uint32_t n_probes,
                                                         const uint32_t *__restrict__ wordpool, const unsigned long long *__restrict__ pair_keys,
                                                         uint64_t n_pairs, uint32_t pair_list_base, const DListRef *__restrict__ lists,
                                                         const ActDesc *__restrict__ acts, const uint32_t *__restrict__ results,
                                                         Job *__restrict__ queue, uint32_t *__restrict__ qcount, uint32_t qcap) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_probes) return;
    // find the set: last s with probe_base <= p
    uint32_t lo = 0, hi = n_sets;
    while (hi - lo > 1) {
        uint32_t mid = (lo + hi) >> 1;
        if (sets[mid].probe_base <= p)
            lo = mid;
        else
            hi = mid;
    }
    const PairSet s = sets[lo];
    uint32_t idx = p - s.probe_base;
    uint32_t rows = results[acts[s.act].res_off];
    if (rows == 0) return;
    uint32_t li = idx / s.n_right, ri = idx % s.n_right;
    uint32_t w1 = wordpool[s.left_off + li];
    if (s.right_is_range) {
        uint32_t rlo = wordpool[s.right_off + 2 * ri], rhi = wordpool[s.right_off + 2 * ri + 1];
        if (s.fwd_prox) {
            unsigned long long k0 = ((unsigned long long)s.fwd_prox << 42) | ((unsigned long long)w1 << 21) | rlo;
            unsigned long long k1 = ((unsigned long long)s.fwd_prox << 42) | ((unsigned long long)w1 << 21) | rhi;
            int64_t a = pair_lower_bound(pair_keys, n_pairs, k0), b = pair_lower_bound(pair_keys, n_pairs, k1);
            for (int64_t i = a; i < b; i++) {
                uint32_t list = pair_list_base + (uint32_t)i;
                push_list_jobs(queue, qcount, qcap, s.act, s.col, list, lists[list], rows);
            }
        }
        return;
    }
    uint32_t w2 = wordpool[s.right_off + ri];
    if (s.fwd_prox) {
        unsigned long long k = ((unsigned long long)s.fwd_prox << 42) | ((unsigned long long)w1 << 21) | w2;
        int64_t i = pair_lower_bound(pair_keys, n_pairs, k);
        if ((uint64_t)i < n_pairs && pair_keys[i] == k) {
            uint32_t list = pair_list_base + (uint32_t)i;
            push_list_jobs(queue, qcount, qcap, s.act, s.col, list, lists[list], rows);
        }
    }
    if (s.bwd_prox) {
        unsigned long long k = ((unsigned long long)s.bwd_prox << 42) | ((unsigned long long)w2 << 21) | w1;
        int64_t i = pair_lower_bound(pair_keys, n_pairs, k);
        if ((uint64_t)i < n_pairs && pair_keys[i] == k) {
            uint32_t list = pair_list_base + (uint32_t)i;
            push_list_jobs(queue, qcount, qcap, s.act, s.col, list, lists[list], rows);
        }
    }
}

// Each warp takes 32 jobs at a time: tiny lists (the common case for word-pair lists) are handled one per lane,
// the others cooperatively by the whole warp, one after the other.
__device__ __forceinline__ void scatter_job_coop(const Job job, const ActDesc &a, uint32_t rows, const DListRef lr,
                                                 const uint32_t *__restrict__ pool, uint32_t lane) {
    unsigned long long *col = a.C + (size_t)job.col * a.ld;
    if (lr.dense) {
        const unsigned long long *words = reinterpret_cast<const unsigned long long *>(pool + lr.off);
        uint32_t r0 = job.chunk * JOB_CHUNK, r1 = min(rows, r0 + JOB_CHUNK);
        // four rows per lane and round: the three dependent loads (row -> word index -> list word, universe word) of the four rows
        // are in flight together
        for (uint32_t j0 = r0 + lane; j0 < r1; j0 += 128) {
            uint32_t wi[4];
            unsigned long long ubv[4], lw[4];
#pragma unroll
            for (int x = 0; x < 4; x++) {
                const uint32_t j = j0 + 32 * x;
                wi[x] = j < r1 ? (a.uw ? a.uw[j] : j) : 0;
                ubv[x] = j < r1 ? a.ub[j] : 0ull;
            }
#pragma unroll
            for (int x = 0; x < 4; x++) lw[x] = ubv[x] ? words[wi[x]] : 0ull;
#pragma unroll
            for (int x = 0; x < 4; x++) {
                const unsigned long long v = lw[x] & ubv[x];
                if (v) atomicOr(&col[j0 + 32 * x], v);
            }
        }
        return;
    }
    const uint32_t *ids = pool + lr.off;
    if (a.uw && (unsigned long long)rows * 16ull < lr.card) {
        // universe much smaller than the list: walk the rows and binary-search the list; the rows are dealt round-robin to the
        // list's chunks (every chunk of the list has a job), so a 100-chunk list searches with 100 warps
        const uint32_t n_chunks = (lr.card + JOB_CHUNK - 1) / JOB_CHUNK;
        for (uint32_t j = job.chunk * 32 + lane; j < rows; j += 32 * n_chunks) {
            uint32_t w = a.uw[j];
            uint32_t lo = 0, hi = lr.card, key = w << 6;
            while (lo < hi) {
                uint32_t mid = (lo + hi) >> 1;
                if (ids[mid] < key)
                    lo = mid + 1;
                else
                    hi = mid;
            }
            unsigned long long v = 0;
            while (lo < lr.card && (ids[lo] >> 6) == w) {
                v |= 1ull << (ids[lo] & 63);
                lo++;
            }
            v &= a.ub[j];
            if (v) atomicOr(&col[j], v);
        }
        return;
    }
    uint32_t e0 = job.chunk * JOB_CHUNK, e1 = min(lr.card, e0 + JOB_CHUNK);
    // Eight docids per lane and round, their row lookups in flight together.  The universe word is NOT consulted here: a document
    // outside the universe can never leave the DP (S[END] = universe word and every S value is an AND chain down to it), so stray
    // bits in a condition column are harmless and the dependent chain is docid -> row -> fire-and-forget reduction.
    for (uint32_t eb = e0 + lane; eb < e1; eb += 256) {
        uint32_t d[8];
        int jr[8];
#pragma unroll
        for (int x = 0; x < 8; x++) d[x] = eb + 32 * x < e1 ? ids[eb + 32 * x] : 0xffffffffu;
#pragma unroll
        for (int x = 0; x < 8; x++) jr[x] = d[x] != 0xffffffffu ? act_row(a, rows, d[x] >> 6) : -1;
#pragma unroll
        for (int x = 0; x < 8; x++)
            if (jr[x] >= 0) atomicOr(&col[jr[x]], 1ull << (d[x] & 63));
    }
}

// Two launches per step.  scatter_kernel takes the jobs 32 at a time: tiny lists (the common case for word-pair lists) are handled
// one per lane, the others are only *noted* in a second queue (bigq).  scatter_big_kernel then gives every noted job to a whole
// warp.  Handling the big jobs inside the first kernel made a warp that drew 20 of them work through 20 x 2048 elements alone
// while the rest of the GPU idled (measured: every launch took ~300 us whatever its size).
__global__ void __launch_bounds__(256) scatter_kernel(const Job *__restrict__ queue, uint32_t *__restrict__ qcount, uint32_t qcap,
                                                      const ActDesc *__restrict__ acts, const uint32_t *__restrict__ results,
                                                      const DListRef *__restrict__ lists, const uint32_t *__restrict__ pool,
                                                      uint32_t *__restrict__ bigq) {
    const uint32_t n_jobs = min(qcount[0], qcap);
    const uint32_t lane = threadIdx.x & 31;
    // Persistent warps pull 32 jobs at a time from a shared cursor (qcount[2], zeroed by the host): the cost of a job ranges from
    // one docid to a 2048-element chunk, so a static split leaves most warps idle behind the few that drew long lists.
    // A grab g covers the jobs g, g + n_grabs, g + 2 n_grabs, ...: neighbouring jobs (the chunks of one long list) go to different
    // warps, and the 32 jobs of one grab come from all over the step.
    const uint32_t n_grabs = (n_jobs + 31) / 32;
    for (;;) {
        uint32_t g = 0;
        if (lane == 0) g = atomicAdd(&qcount[2], 1u);
        g = __shfl_sync(0xffffffffu, g, 0);
        if (g >= n_grabs) break;
        const uint32_t jb = lane * n_grabs + g;
        const bool have = jb < n_jobs;
        Job job{0, 0, 0, 0};
        DListRef lr{0, 0, 0};
        uint32_t rows = 0;
        if (have) {
            job = queue[jb];
            rows = results[acts[job.act].res_off];
            lr = lists[job.list];
        }
        bool live = have && rows > 0 && lr.card > 0;
        bool small = live && !lr.dense && lr.card <= 16;
        if (small) {
            const ActDesc &a = acts[job.act];
            unsigned long long *col = a.C + (size_t)job.col * a.ld;
            const uint32_t *ids = pool + lr.off;
            for (uint32_t e0 = 0; e0 < lr.card; e0 += 4) {  // lookups of four docids in flight together; no universe check (see below)
                uint32_t d[4];
                int j[4];
#pragma unroll
                for (int x = 0; x < 4; x++) d[x] = e0 + x < lr.card ? ids[e0 + x] : 0xffffffffu;
#pragma unroll
                for (int x = 0; x < 4; x++) j[x] = d[x] != 0xffffffffu ? act_row(a, rows, d[x] >> 6) : -1;
#pragma unroll
                for (int x = 0; x < 4; x++)
                    if (j[x] >= 0) atomicOr(&col[j[x]], 1ull << (d[x] & 63));
            }
        }
        const bool is_big = live && !small;
        const unsigned big = __ballot_sync(0xffffffffu, is_big);
        if (big) {  // note the big jobs for scatter_big_kernel: qcount[3] = number noted
            uint32_t at = 0;
            if (lane == 0) at = atomicAdd(&qcount[3], (uint32_t)__popc(big));
            at = __shfl_sync(0xffffffffu, at, 0);
            if (is_big) bigq[at + __popc(big & ((1u << lane) - 1))] = jb;
        }
    }
}
__global__ void __launch_bounds__(256) scatter_big_kernel(const Job *__restrict__ queue, uint32_t *__restrict__ qcount,
                                                          const ActDesc *__restrict__ acts, const uint32_t *__restrict__ results,
                                                          const DListRef *__restrict__ lists, const uint32_t *__restrict__ pool,
                                                          const uint32_t *__restrict__ bigq) {
    const uint32_t n_big = qcount[3];
    const uint32_t lane = threadIdx.x & 31;
    // up to eight jobs per draw: lanes 0..7 fetch the descriptors of their job side by side (five dependent loads each), then the warp
    // works through the eight one after the other
    // (fewer per draw when the step has few big jobs: then the length of the longest warp's chain is what the launch costs)
    const uint32_t GRAB = min(8u, max(1u, n_big / (2u * ((gridDim.x * blockDim.x) >> 5))));
    for (;;) {
        uint32_t k0 = 0;
        if (lane == 0) k0 = atomicAdd(&qcount[4], GRAB);
        k0 = __shfl_sync(0xffffffffu, k0, 0);
        if (k0 >= n_big) break;
        Job job{0, 0, 0, 0};
        uint32_t rows = 0;
        const bool have = lane < GRAB && k0 + lane < n_big;
        if (have) {
            job = queue[bigq[k0 + lane]];
            rows = results[acts[job.act].res_off];
        }
        unsigned todo = __ballot_sync(0xffffffffu, have);
        while (todo) {
            const int src = __ffs(todo) - 1;
            todo &= todo - 1;
            Job bj;
            bj.act = __shfl_sync(0xffffffffu, job.act, src);
            bj.col = __shfl_sync(0xffffffffu, job.col, src);
            bj.list = __shfl_sync(0xffffffffu, job.list, src);
            bj.chunk = __shfl_sync(0xffffffffu, job.chunk, src);
            const uint32_t brows = __shfl_sync(0xffffffffu, rows, src);
            scatter_job_coop(bj, acts[bj.act], brows, lists[bj.list], pool, lane);
        }
    }
}

__device__ __forceinline__ unsigned long long mix64(unsigned long long x) {
    x ^= x >> 33;
    x *= 0xff51afd7ed558ccdull;
    x ^= x >> 33;
    x *= 0xc4ceb9fe1a85ec53ull;
    x ^= x >> 33;
    return x;
}

// ---- evaluation of an activation: column program, backward DP over the state graph, buckets, counts, surviving paths.
// Thread per row (64 documents).  Every thread owns `n_cols + n_pairs + 2` 64-bit *slots*: the condition columns of its row, the
// DP table S[(state, cost) pair], and the constants ZERO / ONES.  SMEM = true keeps the slots in shared memory, [slot][thread]
// (thread-private, conflict-free, no barriers): the thread first loads all its condition words from global memory (independent,
// coalesced loads: one round of latency), runs the column program on them, and from then on the DP, the buckets and the walk
// touch shared memory only.  Global traffic = condition columns in + universe word in + bucket columns out, i.e. the algorithmic
// bytes.  The host bins the tiles of a step by slot count (EVAL_CLASS_SLOTS) and launches one grid per class with that much
// dynamic shared memory; SMEM = false (more slots than fit) works on the global matrices C and S directly.
//
// The DP is a straight-line program built by the host once per activation (emit_activation_work): one 32-bit op per
// (pair, feasible edge) in processing order (pairs descending = states in reverse topological order):
// {src slot : 15 | last-of-pair : 1 | condition slot : 16}; acc |= slot[src] & slot[cond]; on `last` the accumulator is stored to
// the current destination pair, which then steps down.  Ops are consumed four at a time.
//
// Surviving paths (graph_based_ranking_rule.rs:340-353: the host rebuilds the next query graph from the paths that took at
// least one document) are the business of walk_kernel, which runs after this kernel over the same tiles: this kernel leaves, per
// tile, the set of its non-empty buckets (tile_summary), so that whole tiles are skipped there.
constexpr int WALK_CLASSES = 8;  // distinct signatures tracked per row (more: every needed document of the row walks)
__device__ __forceinline__ void load_act(ActDesc *dst, const ActDesc *src) {
    static_assert(sizeof(ActDesc) % 4 == 0, "ActDesc is copied word by word");
    const uint32_t *s = reinterpret_cast<const uint32_t *>(src);
    uint32_t *d = reinterpret_cast<uint32_t *>(dst);
    for (uint32_t i = threadIdx.x; i < sizeof(ActDesc) / 4; i += blockDim.x) d[i] = s[i];
}
// insert h into the activation's global table; 1 new, 0 known, -1 table full
__device__ __forceinline__ int tab_insert(const ActDesc &a, unsigned long long h) {
    uint32_t slot = (uint32_t)(h % a.tab_size);
    for (uint32_t probe = 0; probe < a.tab_size; probe++) {
        unsigned long long prev = atomicCAS(&a.tab[slot], 0ull, h);
        if (prev == 0ull) return 1;
        if (prev == h) return 0;
        slot = slot + 1 == a.tab_size ? 0 : slot + 1;
    }
    return -1;
}
// The walk of one row: `slot(k)` reads the row's slot k (condition columns after the column program, then the DP table).
template <class SlotFn>
__device__ __forceinline__ void walk_row(const ActDesc &a, uint32_t act_i, uint32_t last_bucket, unsigned long long only, const DpState *st,
                                         const DpEdge *ed, const uint16_t *cost_vals, size_t j, SlotFn slot, unsigned long long *s_seen /* 64 */, uint32_t *results, PathOut *pathbuf,
                                         uint32_t *path_count, uint32_t path_cap) {
    const uint32_t END = a.n_states - 1, n_cols = a.n_cols;
    for (uint32_t ci = 0; ci <= last_bucket && ci < a.n_costs; ci++) {
        const unsigned long long b = a.out[(size_t)ci * a.ld + j] & only;
        if (!b) continue;
        struct Frame {
            unsigned long long mask;
            uint16_t state, e, r;
        } stack[MAX_WALK];
        uint16_t pedges[MAX_WALK];
        int d = 0;
        stack[0].mask = b;
        stack[0].state = 0;
        stack[0].e = 0;
        stack[0].r = cost_vals[ci];
        while (d >= 0) {
            Frame &f = stack[d];
            const DpState fs = st[f.state];
            if (f.mask == 0 || f.e >= fs.n_edges) {
                d--;
                continue;
            }
            uint32_t eidx = fs.edge_begin + f.e;
            const DpEdge ee = ed[eidx];
            f.e++;
            if (ee.cost > f.r) continue;
            uint32_t rr = f.r - ee.cost;
            const DpState ds = st[ee.dst];
            if (rr < ds.rmin || rr >= (uint32_t)ds.rmin + ds.rcount) continue;
            unsigned long long take = f.mask & slot(n_cols + ds.pair_off + rr - ds.rmin);
            if (take && ee.col != 0xffff) take &= slot(ee.col);
            if (!take) continue;
            f.mask &= ~take;
            pedges[d] = (uint16_t)eidx;
            if (ee.dst == END) {
                // a complete path: report it once per activation
                unsigned long long h = mix64(0x9e3779b97f4a7c15ull * (ci + 1));
                for (int k = 0; k <= d; k++) h = mix64(h + 0xd6e8feb86659fd93ull * (unsigned long long)(pedges[k] + 1));
                h = (h & ~2ull) | 1ull;  // bit 1 clear: a path (signatures have it set)
                bool known = false;
                {
                    // the local filter may be shared by rows of different activations (walk_kernel): its key carries the activation
                    const unsigned long long hl = (h ^ (0x9e3779b97f4a7c15ull * (unsigned long long)(act_i + 1))) | 1ull;
                    uint32_t sl = (uint32_t)(hl >> 20) & 63u;
                    for (int probe = 0; probe < 8; probe++) {
                        unsigned long long prev = atomicCAS(&s_seen[sl], 0ull, hl);
                        if (prev == hl) {
                            known = true;
                            break;
                        }
                        if (prev == 0ull) break;  // we claimed it: go on to the global table
                        sl = (sl + 1) & 63u;
                    }
                }
                if (known) continue;
                const int fresh = tab_insert(a, h);
                if (fresh < 0) atomicOr(&results[a.res_off + 1 + a.n_costs + 1], 1u);  // table saturated: the host reruns the step
                if (fresh > 0) {
                    uint32_t at = atomicAdd(path_count, 1u);
                    if (at < path_cap) {
                        PathOut po;
                        po.act = act_i;
                        po.cost_idx = (uint16_t)ci;
                        po.len = (uint16_t)(d + 1);
                        for (int k = 0; k < (int)MAX_WALK; k++) po.edges[k] = k <= d ? pedges[k] : 0;
                        pathbuf[at] = po;
                    }
                }
                continue;
            }
            if (d + 1 >= (int)MAX_WALK) continue;  // host guarantees path length <= MAX_WALK
            d++;
            stack[d].mask = take;
            stack[d].state = ee.dst;
            stack[d].e = 0;
            stack[d].r = (uint16_t)rr;
        }
    }
}

template <bool SMEM>
__global__ void __launch_bounds__(128, 8) eval_dp_kernel(const TileDesc *__restrict__ tiles, const ActDesc *__restrict__ acts,
                                                      uint32_t *__restrict__ results, const ColOp *__restrict__ colprog,
                                                      const uint16_t *__restrict__ costpool, const uint32_t *__restrict__ progpool,
                                                      unsigned long long *__restrict__ tile_summary) {
    extern __shared__ unsigned long long s_slot[];  // SMEM: [n_cols + n_pairs + 2][128]
    const TileDesc tile = tiles[blockIdx.x];
    __shared__ ActDesc a;
    __shared__ uint32_t counts[MAX_COSTS + 1];
    load_act(&a, &acts[tile.act]);
    for (uint32_t i = threadIdx.x; i <= MAX_COSTS; i += blockDim.x) counts[i] = 0;
    __syncthreads();
    const uint32_t rows = results[a.res_off];
    if (tile.row_begin >= rows) {
        if (threadIdx.x < 2) tile_summary[2 * (size_t)blockIdx.x + threadIdx.x] = 0ull;
        return;
    }
    const uint32_t n_cols = a.n_cols, n_pairs = a.n_pairs, n_costs = a.n_costs;
    const uint32_t ZERO_SLOT = n_cols + n_pairs, ONES_SLOT = n_cols + n_pairs + 1;
    const size_t ld = a.ld;
    unsigned long long *const C = a.C;
    unsigned long long *const Sg = a.S;
    unsigned long long *const out = a.out;
    const uint32_t *const prog = progpool + a.prog_off;
    const uint16_t *const cost_vals = costpool + a.cost_off;
    const uint32_t lane = threadIdx.x & 31;
    if (SMEM) {
        s_slot[(size_t)ZERO_SLOT * 128 + threadIdx.x] = 0ull;
        s_slot[(size_t)ONES_SLOT * 128 + threadIdx.x] = ~0ull;
    }
    for (uint32_t rr_ = 0; rr_ < tile.rows_per_thread; rr_++) {
        const uint32_t j = tile.row_begin + rr_ * 128 + threadIdx.x;
        if (tile.row_begin + rr_ * 128 >= rows) break;  // uniform
        const bool active = j < rows;
        unsigned long long g_const[2] = {0ull, ~0ull};
#define SLOT(k) (*(SMEM ? &s_slot[(size_t)(k) * 128 + threadIdx.x] : ((k) < n_cols ? &C[(size_t)(k) * ld + j] : ((k) < ZERO_SLOT ? &Sg[(size_t)((k) - n_cols) * ld + j] : &g_const[(k) - ZERO_SLOT]))))
        const unsigned long long u = active ? a.ub[j] : 0ull;
        bool run = active;
        if (SMEM && active) {
            unsigned long long any = 0;
            uint32_t c = 0;
            for (; c + 8 <= n_cols; c += 8) {
                unsigned long long v[8];
#pragma unroll
                for (int x = 0; x < 8; x++) v[x] = C[(size_t)(c + x) * ld + j];
#pragma unroll
                for (int x = 0; x < 8; x++) {
                    s_slot[(size_t)(c + x) * 128 + threadIdx.x] = v[x];
                    any |= v[x];
                }
            }
            for (; c < n_cols; c++) {
                const unsigned long long v = C[(size_t)c * ld + j];
                s_slot[(size_t)c * 128 + threadIdx.x] = v;
                any |= v;
            }
            // a row that satisfies no condition at all cannot be on any path: it only contributes to the "rest" column
            if (a.all_conditional && !(any & u)) run = false;
        }
        if (run) {
            for (uint32_t i = 0; i < a.colprog_len; i++) {
                const ColOp op = colprog[a.colprog_off + i];
                unsigned long long x = SLOT(op.a), r;
                if (op.op == 3)
                    r = x;
                else {
                    unsigned long long y = SLOT(op.b);
                    r = op.op == 0 ? (x & y) : (op.op == 1 ? (x | y) : (x & ~y));
                }
                SLOT(op.dst) = r;
            }
            if (!SMEM && a.all_conditional) {
                unsigned long long any = 0;
#pragma unroll 4
                for (uint32_t c = 0; c < n_cols; c++) any |= C[(size_t)c * ld + j];
                if (!(any & u)) run = false;
            }
        }
        if (run) {
            SLOT(n_cols + n_pairs - 1) = u;  // END has the single pair (cost 0), the last one
            const uint32_t plen = a.prog_len;  // multiple of 4 (padded with no-ops)
            uint32_t dst = n_cols + n_pairs - 2;
            unsigned long long acc = 0;
            for (uint32_t i = 0; i < plen; i += 4) {
                const uint4 o4 = __ldg(reinterpret_cast<const uint4 *>(prog + i));
                const uint32_t op[4] = {o4.x, o4.y, o4.z, o4.w};
                unsigned long long cc[4];
#pragma unroll
                for (int x = 0; x < 4; x++) cc[x] = SLOT(op[x] >> 16);  // a condition slot, or the constant ZERO / ONES slot
                // sources written inside this group of four are re-read after the store (in-order per thread): read them one by one
#pragma unroll
                for (int x = 0; x < 4; x++) {
                    acc |= SLOT(op[x] & 0x7fffu) & cc[x];
                    if (op[x] & 0x8000u) {
                        SLOT(dst) = acc;
                        acc = 0;
                        dst--;
                    }
                }
            }
        }
        // buckets, cheapest cost first; the counters are aggregated per warp before they touch shared memory
        unsigned long long taken = 0;
        for (uint32_t ci = 0; ci < n_costs; ci++) {
            const uint32_t r = cost_vals[ci];
            unsigned long long b = 0;
            if (run && r >= a.root_rmin && r < a.root_rmin + a.root_rcount) b = SLOT(n_cols + r - a.root_rmin) & ~taken;  // START's pairs come first
            if (active) out[(size_t)ci * ld + j] = b;
            taken |= b;
            const uint32_t pc = __reduce_add_sync(0xffffffffu, (uint32_t)__popcll(b));
            if (lane == 0 && pc) atomicAdd(&counts[ci], pc);
        }
        const unsigned long long rest = u & ~taken;
        if (active) out[(size_t)n_costs * ld + j] = rest;
        {
            const uint32_t pc = __reduce_add_sync(0xffffffffu, (uint32_t)__popcll(rest));
            if (lane == 0 && pc) atomicAdd(&counts[n_costs], pc);
        }
#undef SLOT
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i <= n_costs; i += blockDim.x)
        if (counts[i]) atomicAdd(&results[a.res_off + 1 + i], counts[i]);
    if (threadIdx.x < 2) {  // non-empty buckets of this tile, 64 per word (walk_kernel skips whole tiles with it)
        unsigned long long m = 0;
        for (uint32_t i = 0; i < 64; i++) {
            const uint32_t ci = threadIdx.x * 64 + i;
            if (ci < n_costs && counts[ci]) m |= 1ull << i;
        }
        tile_summary[2 * (size_t)blockIdx.x + threadIdx.x] = m;
    }
}

// Pass 2 over the same tiles (same grid, same shared-memory class): which paths produced the buckets the query can still need.
// bucket_sort only descends into the cheapest buckets that together hold `need` documents (the hits it still has to return
// plus the offset it still has to skip; every document of a bucket it enters is eventually returned or skipped), so only rows
// holding documents of those buckets are re-evaluated: DP as in eval_dp_kernel, then every document *walks* the graph taking, at
// each state, the first edge (in order) whose condition it satisfies and from which it can still finish with its remaining
// budget.  Distinct walked paths are de-duplicated (per CTA in shared memory, then per activation in a global hash table) and
// reported.  The path a document takes is a function of its condition bits alone, and a large bucket holds few distinct bit
// patterns: with at most 64 condition columns, the needed documents of a row are first split into classes of identical bits
// (their *signatures*), every class is looked up in the same tables, and only documents of classes nobody has met walk —
// somebody else walks (or walked) a document with the same pattern.
template <bool SMEM>
__global__ void __launch_bounds__(128, 8) walk_kernel(const TileDesc *__restrict__ tiles, const ActDesc *__restrict__ acts,
                                                      uint32_t *__restrict__ results, const ColOp *__restrict__ colprog,
                                                      const DpState *__restrict__ states, const DpEdge *__restrict__ edges,
                                                      const uint16_t *__restrict__ costpool, const uint32_t *__restrict__ progpool,
                                                      const unsigned long long *__restrict__ tile_summary, PathOut *__restrict__ pathbuf,
                                                      uint32_t *__restrict__ path_count, uint32_t path_cap) {
    extern __shared__ unsigned long long s_slot[];  // SMEM: [n_cols + n_pairs + 2][128]
    const TileDesc tile = tiles[blockIdx.x];
    if (!acts[tile.act].want_paths) return;
    __shared__ ActDesc a;
    __shared__ unsigned long long s_seen[64];   // path reports already made by this CTA (hashes)
    __shared__ unsigned long long s_sig[128];   // document signatures this CTA already met
    __shared__ uint32_t s_m;
    load_act(&a, &acts[tile.act]);
    if (threadIdx.x < 64) s_seen[threadIdx.x] = 0;
    s_sig[threadIdx.x] = 0;
    __syncthreads();
    if (threadIdx.x == 0) {
        // last needed bucket: the first one at which the cumulative count reaches `need`
        const uint32_t *cnt = results + a.res_off + 1;
        unsigned long long cum = 0;
        uint32_t m = 0;
        for (; m < a.n_costs; m++) {
            cum += cnt[m];
            if (cum >= a.need) break;
        }
        if (m >= a.n_costs) m = a.n_costs ? a.n_costs - 1 : 0;
        s_m = m;
        if (tile.row_begin == 0) results[a.res_off + 1 + a.n_costs + 2] = m;  // the host checks it before it descends
    }
    __syncthreads();
    const uint32_t m = s_m;
    {
        const unsigned long long s0 = tile_summary[2 * (size_t)blockIdx.x], s1 = tile_summary[2 * (size_t)blockIdx.x + 1];
        const unsigned long long k0 = m >= 63 ? ~0ull : ((2ull << m) - 1), k1 = m < 64 ? 0ull : (m >= 127 ? ~0ull : ((2ull << (m - 64)) - 1));
        if (((s0 & k0) | (s1 & k1)) == 0) return;
    }
    const uint32_t rows = results[a.res_off];
    const uint32_t n_cols = a.n_cols, n_pairs = a.n_pairs;
    const uint32_t ZERO_SLOT = n_cols + n_pairs, ONES_SLOT = n_cols + n_pairs + 1;
    const size_t ld = a.ld;
    unsigned long long *const C = a.C;
    unsigned long long *const Sg = a.S;
    const uint32_t *const prog = progpool + a.prog_off;
    const uint16_t *const cost_vals = costpool + a.cost_off;
    if (SMEM) {
        s_slot[(size_t)ZERO_SLOT * 128 + threadIdx.x] = 0ull;
        s_slot[(size_t)ONES_SLOT * 128 + threadIdx.x] = ~0ull;
    }
    for (uint32_t rr_ = 0; rr_ < tile.rows_per_thread; rr_++) {
        const uint32_t j = tile.row_begin + rr_ * 128 + threadIdx.x;
        if (j >= rows) break;
        unsigned long long needed = 0;
        for (uint32_t ci = 0; ci <= m; ci++) needed |= a.out[(size_t)ci * ld + j];
        if (!needed) continue;
        unsigned long long g_const[2] = {0ull, ~0ull};
#define SLOT(k) (*(SMEM ? &s_slot[(size_t)(k) * 128 + threadIdx.x] : ((k) < n_cols ? &C[(size_t)(k) * ld + j] : ((k) < ZERO_SLOT ? &Sg[(size_t)((k) - n_cols) * ld + j] : &g_const[(k) - ZERO_SLOT]))))
        if (SMEM) {
            uint32_t c = 0;
            for (; c + 8 <= n_cols; c += 8) {
                unsigned long long v[8];
#pragma unroll
                for (int x = 0; x < 8; x++) v[x] = C[(size_t)(c + x) * ld + j];
#pragma unroll
                for (int x = 0; x < 8; x++) s_slot[(size_t)(c + x) * 128 + threadIdx.x] = v[x];
            }
            for (; c < n_cols; c++) s_slot[(size_t)c * 128 + threadIdx.x] = C[(size_t)c * ld + j];
        }
        unsigned long long walk_mask = needed;  // the documents that have to walk
        if (n_cols <= 64) {
            // Partition refinement, bit-sliced: split the needed documents of the row into classes of identical condition bits
            // (column after column, every class is cut in two by the column's word) — the classes are the row's distinct
            // signatures.  A class somebody already met is dropped; only documents of new classes walk.
            unsigned long long cm[WALK_CLASSES], cp[WALK_CLASSES];
            int nc = 1;
            bool overflow = false;
            cm[0] = needed;
            cp[0] = 0;
            for (uint32_t c = 0; c < n_cols && !overflow; c++) {
                const unsigned long long v = SLOT(c);
                if (!(v & needed)) continue;
                const int n0 = nc;
                for (int k = 0; k < n0; k++) {
                    const unsigned long long m1 = cm[k] & v;
                    if (!m1) continue;
                    if (m1 == cm[k])
                        cp[k] |= 1ull << c;
                    else if (nc == WALK_CLASSES) {
                        overflow = true;
                        break;
                    } else {
                        cm[nc] = m1;
                        cp[nc] = cp[k] | (1ull << c);
                        cm[k] &= ~v;
                        nc++;
                    }
                }
            }
            if (!overflow) {
                walk_mask = 0;
                for (int k = 0; k < nc; k++) {
                    const unsigned long long h = mix64(cp[k] ^ ((unsigned long long)n_cols << 56) ^ 0x51ed270b1ull) | 3ull;  // bit 1 set: a signature
                    bool known = false;
                    uint32_t sl = (uint32_t)(h >> 20) & 127u;
                    for (int probe = 0; probe < 8; probe++) {
                        unsigned long long prev = atomicCAS(&s_sig[sl], 0ull, h);
                        if (prev == h) {
                            known = true;
                            break;
                        }
                        if (prev == 0ull) break;
                        sl = (sl + 1) & 127u;
                    }
                    if (known) continue;
                    if (tab_insert(a, h) != 0) walk_mask |= cm[k];  // new for the activation, or the table is full (then walk: the walk reports the overflow)
                }
                if (!walk_mask) continue;
            }
        }
        if (SMEM) {  // (the global variant already holds the column program's results in C and the DP table in S)
            for (uint32_t i = 0; i < a.colprog_len; i++) {
                const ColOp op = colprog[a.colprog_off + i];
                unsigned long long x = SLOT(op.a), r;
                if (op.op == 3)
                    r = x;
                else {
                    unsigned long long y = SLOT(op.b);
                    r = op.op == 0 ? (x & y) : (op.op == 1 ? (x | y) : (x & ~y));
                }
                SLOT(op.dst) = r;
            }
            SLOT(n_cols + n_pairs - 1) = a.ub[j];
            const uint32_t plen = a.prog_len;
            uint32_t dst = n_cols + n_pairs - 2;
            unsigned long long acc = 0;
            for (uint32_t i = 0; i < plen; i += 4) {
                const uint4 o4 = __ldg(reinterpret_cast<const uint4 *>(prog + i));
                const uint32_t op[4] = {o4.x, o4.y, o4.z, o4.w};
#pragma unroll
                for (int x = 0; x < 4; x++) {
                    acc |= SLOT(op[x] & 0x7fffu) & SLOT(op[x] >> 16);
                    if (op[x] & 0x8000u) {
                        SLOT(dst) = acc;
                        acc = 0;
                        dst--;
                    }
                }
            }
        }
        walk_row(a, tile.act, m, walk_mask, states + a.state_off, edges + a.edge_off, cost_vals, j, [&](uint32_t k) { return SLOT(k); }, s_seen, results,
                 pathbuf, path_count, path_cap);
#undef SLOT
    }
}

// one CTA per emission: ascending docids of OR(out[col_lo..col_hi)), skipping `skip`, taking `take`.
// 2048 rows per round — 8 consecutive rows per thread, loads issued together — because a sparse bucket of a large universe is a long
// scan (a 20-document bucket of a 150 k-row universe) whose cost is the number of dependent global-memory round trips.
constexpr int EMIT_ROWS_PER_LANE = 8, EMIT_THREADS = 256;
__global__ void __launch_bounds__(EMIT_THREADS) emit_kernel(const EmitDesc *__restrict__ emits, uint32_t n_emits) {
    const uint32_t e = blockIdx.x;
    if (e >= n_emits) return;
    const EmitDesc d = emits[e];
    __shared__ uint32_t warp_tot[EMIT_THREADS / 32];
    const uint32_t lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
    uint32_t seen = 0;  // documents of the bucket in the rows before this round
    for (uint32_t j0 = 0; j0 < d.rows && seen < d.skip + d.take; j0 += EMIT_THREADS * EMIT_ROWS_PER_LANE) {
        const uint32_t jb = j0 + threadIdx.x * EMIT_ROWS_PER_LANE;
        unsigned long long v[EMIT_ROWS_PER_LANE];
#pragma unroll
        for (int i = 0; i < EMIT_ROWS_PER_LANE; i++) {
            const uint32_t j = jb + i;
            v[i] = 0;
            if (j < d.rows) {
                if (d.out) {
                    for (uint32_t c = d.col_lo; c < d.col_hi; c++) v[i] |= d.out[(size_t)c * d.ld + j];
                } else
                    v[i] = d.ub[j];
            }
        }
        uint32_t pc = 0;
#pragma unroll
        for (int i = 0; i < EMIT_ROWS_PER_LANE; i++) pc += (uint32_t)__popcll(v[i]);
        uint32_t pre = pc;
#pragma unroll
        for (int s = 1; s < 32; s <<= 1) {
            uint32_t t = __shfl_up_sync(0xffffffffu, pre, s);
            if (lane >= (uint32_t)s) pre += t;
        }
        if (lane == 31) warp_tot[wrp] = pre;
        __syncthreads();
        uint32_t before = 0, total = 0;
#pragma unroll
        for (int w = 0; w < EMIT_THREADS / 32; w++) {
            const uint32_t t = warp_tot[w];
            before += (uint32_t)w < wrp ? t : 0u;
            total += t;
        }
        uint32_t rk = seen + before + pre - pc;  // rank of this thread's first document within the bucket
        if (pc && rk < d.skip + d.take && rk + pc > d.skip) {
#pragma unroll
            for (int i = 0; i < EMIT_ROWS_PER_LANE; i++) {
                unsigned long long x = v[i];
                if (!x) continue;
                const uint32_t base = d.uw ? d.uw[jb + i] : jb + i;
                while (x) {
                    uint32_t bit = (uint32_t)__ffsll((long long)x) - 1;
                    x &= x - 1;
                    if (rk >= d.skip) {
                        uint32_t o = rk - d.skip;
                        if (o < d.take) d.dst[o] = base * 64 + bit;
                    }
                    rk++;
                }
            }
        }
        seen += total;
        __syncthreads();
    }
}

// ======================================================================================== vector stage
// distance = (1 - cos)/2, cos = q.v / (|q||v|): arroy/hannoy `Cosine` (SURVEY §A.6).  One warp per row,
// 3 x 128-bit loads per lane per 768-d fp16 row; QT query vectors are held in shared memory as fp32.
template <int QT>
__global__ void __launch_bounds__(256) vec_dist_kernel(const __half *__restrict__ mat, const float *__restrict__ inv_norm,
                                                       const uint32_t *__restrict__ docids, uint64_t n_rows, uint32_t d,
                                                       const float *__restrict__ queries /* QT x d */, const float *__restrict__ q_inv_norm,
                                                       const unsigned long long *__restrict__ cand, uint64_t n_cand_words,
                                                       float *__restrict__ dist /* QT x n_rows */) {
    extern __shared__ float sq[];  // QT * d
    const uint32_t vpr = d / 8;  // 128-bit vectors per row
    for (uint32_t i = threadIdx.x; i < QT * d; i += blockDim.x) {
        uint32_t q = i / d, e = i % d;
        sq[q * d + (e & 7) * vpr + (e >> 3)] = queries[i];  // [q][k][v]: lanes read consecutive banks
    }
    __syncthreads();
    uint32_t lane = threadIdx.x & 31;
    uint64_t warp = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
    uint64_t n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    uint32_t vec_per_row = d / 8;  // uint4 = 8 halfs
    for (uint64_t r = warp; r < n_rows; r += n_warps) {
        bool ok = true;
        if (cand) {
            uint32_t doc = docids[r];
            ok = (doc >> 6) < n_cand_words && ((cand[doc >> 6] >> (doc & 63)) & 1);
        }
        if (!ok) {
            if (lane < QT) dist[(uint64_t)lane * n_rows + r] = 3.0f;  // > any distance: never selected
            continue;
        }
        const uint4 *row = reinterpret_cast<const uint4 *>(mat + r * d);
        float acc[QT];
#pragma unroll
        for (int q = 0; q < QT; q++) acc[q] = 0.f;
#pragma unroll 3
        for (uint32_t v = lane; v < vec_per_row; v += 32) {
            uint4 x = __ldg(row + v);
            const __half2 *h = reinterpret_cast<const __half2 *>(&x);
            float f[8];
#pragma unroll
            for (int k = 0; k < 4; k++) {
                float2 t = __half22float2(h[k]);
                f[2 * k] = t.x;
                f[2 * k + 1] = t.y;
            }
#pragma unroll
            for (int q = 0; q < QT; q++) {
                const float *qq = sq + q * d + v;
#pragma unroll
                for (int k = 0; k < 8; k++) acc[q] = fmaf(f[k], qq[k * vpr], acc[q]);
            }
        }
#pragma unroll
        for (int q = 0; q < QT; q++) {
#pragma unroll
            for (int s = 16; s > 0; s >>= 1) acc[q] += __shfl_xor_sync(0xffffffffu, acc[q], s);
        }
        if (lane == 0) {
            float vn = inv_norm[r];
#pragma unroll
            for (int q = 0; q < QT; q++) {
                float dd = 0.f;
                float pn = vn * q_inv_norm[q];
                if (pn > 0.f && isfinite(pn)) {
                    float cs = acc[q] * pn;
                    cs = fminf(1.f, fmaxf(-1.f, cs));
                    dd = (1.f - cs) * 0.5f;
                }
                dist[(uint64_t)q * n_rows + r] = dd;
            }
        }
    }
}

// exact top-k by radix select (4 x 8 bits) on the (non-negative) float bit patterns.  One CTA per (query, slice): a query's
// distance row is cut into n_slices pieces that are selected side by side (a single CTA walking 10^7 distances four times was 80 %
// of a B = 1 query); the slices' outputs (k + tie_cap slots each, unused ones set to 3.0 = "no candidate") are then selected once
// more by the same kernel with n_slices = 1 and per-query id arrays (ids_stride != 0).
__global__ void __launch_bounds__(1024) topk_select_kernel(const float *__restrict__ dist, uint64_t dist_stride, const uint32_t *__restrict__ docids,
                                                           uint64_t ids_stride, uint64_t n_rows_total, uint32_t n_slices, uint32_t k,
                                                           uint32_t tie_cap, float *__restrict__ out_dist, uint32_t *__restrict__ out_ids,
                                                           uint32_t *__restrict__ out_n /* 2 per (query, slice) */) {
    __shared__ uint32_t hist[256];
    __shared__ uint32_t s_prefix, s_remaining, s_count_lt, s_count_eq;
    const uint32_t qi = blockIdx.x / n_slices, sl = blockIdx.x % n_slices;
    const uint64_t slice_len = (n_rows_total + n_slices - 1) / n_slices, r_begin = (uint64_t)sl * slice_len;
    const uint64_t n_rows = r_begin < n_rows_total ? min(slice_len, n_rows_total - r_begin) : 0;
    const float *dq = dist + (uint64_t)qi * dist_stride + r_begin;
    docids += (uint64_t)qi * ids_stride + r_begin;
    float *od = out_dist + (uint64_t)blockIdx.x * (k + tie_cap);
    uint32_t *oi = out_ids + (uint64_t)blockIdx.x * (k + tie_cap);
    // number of selectable rows (distance <= 1.0)
    uint32_t prefix = 0, remaining = k;
    // four passes of 8 bits, most significant first (256 bins: the serial scan of the histogram by one thread stays short; with
    // 4096 bins it was the longest part of a pass)
    const int shifts[4] = {24, 16, 8, 0};
    const int bits[4] = {8, 8, 8, 8};
    uint32_t mask_hi = 0;
    for (int pass = 0; pass < 4; pass++) {
        for (uint32_t i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0;
        __syncthreads();
        for (uint64_t r = threadIdx.x; r < n_rows; r += blockDim.x) {
            float v = dq[r];
            if (v > 1.5f) continue;
            uint32_t b = __float_as_uint(v);
            if ((b & mask_hi) == prefix) {
                // distances cluster (cosine of random directions: nearly all share their top byte): count per warp first
                const uint32_t bin = (b >> shifts[pass]) & ((1u << bits[pass]) - 1);
                const unsigned peers = __match_any_sync(__activemask(), bin);
                if ((threadIdx.x & 31) == (uint32_t)(__ffs(peers) - 1)) atomicAdd(&hist[bin], (uint32_t)__popc(peers));
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t acc = 0, nb = 1u << bits[pass], sel = nb - 1;
            bool found = false;
            for (uint32_t i = 0; i < nb; i++) {
                if (acc + hist[i] >= remaining) {
                    sel = i;
                    found = true;
                    break;
                }
                acc += hist[i];
            }
            if (!found) {  // fewer than k selectable rows: everything qualifies
                s_prefix = 0xffffffffu;
                s_remaining = 0;
            } else {
                s_prefix = prefix | (sel << shifts[pass]);
                s_remaining = remaining - acc;
            }
        }
        __syncthreads();
        if (s_prefix == 0xffffffffu) {
            prefix = 0xffffffffu;
            break;
        }
        prefix = s_prefix;
        remaining = s_remaining;
        mask_hi |= ((1u << bits[pass]) - 1) << shifts[pass];
        __syncthreads();
    }
    // prefix == bit pattern of the k-th smallest distance (or 0xffffffff: take all)
    if (threadIdx.x == 0) {
        s_count_lt = 0;
        s_count_eq = 0;
    }
    __syncthreads();
    for (uint64_t r = threadIdx.x; r < n_rows; r += blockDim.x) {
        float v = dq[r];
        if (v > 1.5f) continue;
        uint32_t b = __float_as_uint(v);
        if (prefix == 0xffffffffu || b < prefix) {
            uint32_t at = atomicAdd(&s_count_lt, 1u);
            if (at < k) {
                od[at] = v;
                oi[at] = docids[r];
            }
        } else if (b == prefix) {
            uint32_t at = atomicAdd(&s_count_eq, 1u);
            if (at < tie_cap) {
                od[k + at] = v;
                oi[k + at] = docids[r];
            }
        }
    }
    __syncthreads();
    const uint32_t n_lt = min(s_count_lt, k), n_eq = min(s_count_eq, tie_cap);
    for (uint32_t i = n_lt + threadIdx.x; i < k; i += blockDim.x) od[i] = 3.0f;           // unused slots: "no candidate"
    for (uint32_t i = n_eq + threadIdx.x; i < tie_cap; i += blockDim.x) od[k + i] = 3.0f;
    if (threadIdx.x == 0) {
        out_n[2 * blockIdx.x] = n_lt;
        out_n[2 * blockIdx.x + 1] = n_eq;
    }
}

// ---- staging of the vector store: fp16 rows + f32 inverse norms, one warp per row
__global__ void __launch_bounds__(256) emb_from_f32_kernel(const float *__restrict__ in, __half *__restrict__ out, float *__restrict__ inv_norm,
                                                           uint64_t n, uint32_t d) {
    const uint64_t r = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
    if (r >= n) return;
    const uint32_t lane = threadIdx.x & 31;
    float ss = 0.f;
    for (uint32_t i = lane; i < d; i += 32) {
        const float v = in[r * d + i];
        ss = fmaf(v, v, ss);
        out[r * d + i] = __float2half_rn(v);
    }
#pragma unroll
    for (int sft = 16; sft > 0; sft >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, sft);
    if (lane == 0) {
        const float nrm = sqrtf(ss);
        inv_norm[r] = nrm > 0.f ? 1.0f / nrm : 0.f;
    }
}
__global__ void __launch_bounds__(256) emb_norm_f16_kernel(const __half *__restrict__ rows, float *__restrict__ inv_norm, uint64_t n, uint32_t d) {
    const uint64_t r = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
    if (r >= n) return;
    const uint32_t lane = threadIdx.x & 31;
    float ss = 0.f;
    for (uint32_t i = lane; i < d; i += 32) {
        const float v = __half2float(rows[r * d + i]);
        ss = fmaf(v, v, ss);
    }
#pragma unroll
    for (int sft = 16; sft > 0; sft >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, sft);
    if (lane == 0) {
        const float nrm = sqrtf(ss);
        inv_norm[r] = nrm > 0.f ? 1.0f / nrm : 0.f;
    }
}
cudaError_t launch_emb_from_f32(cudaStream_t s, const float *in, void *out_fp16, float *inv_norm, uint64_t n, uint32_t d) {
    if (!n) return cudaSuccess;
    emb_from_f32_kernel<<<(unsigned)((n * 32 + 255) / 256), 256, 0, s>>>(in, reinterpret_cast<__half *>(out_fp16), inv_norm, n, d);
    return cudaGetLastError();
}
cudaError_t launch_emb_norm_f16(cudaStream_t s, const void *rows_fp16, float *inv_norm, uint64_t n, uint32_t d) {
    if (!n) return cudaSuccess;
    emb_norm_f16_kernel<<<(unsigned)((n * 32 + 255) / 256), 256, 0, s>>>(reinterpret_cast<const __half *>(rows_fp16), inv_norm, n, d);
    return cudaGetLastError();
}

// ---- corpus-sharded vector stage: merge of the per-shard top-k lists after the all-gather
// One CTA per query: the shards' runs (ascending (distance, docid), n valid entries each) become 64-bit keys
// distance-bits << 32 | docid, are sorted by a bitonic network in shared memory, and the first `k` are written back.
__global__ void __launch_bounds__(256) shard_merge_kernel(const uint32_t *__restrict__ g_ids, const float *__restrict__ g_dist,
                                                          const uint32_t *__restrict__ g_n, uint32_t world, uint32_t n_q, uint32_t k,
                                                          uint32_t cap /* power of two >= world * k */, uint32_t *__restrict__ out_ids,
                                                          float *__restrict__ out_dist, uint32_t *__restrict__ out_n) {
    extern __shared__ unsigned long long s_keys[];
    const uint32_t q = blockIdx.x;
    uint32_t total = 0;
    for (uint32_t i = threadIdx.x; i < cap; i += blockDim.x) {
        unsigned long long key = ~0ull;
        if (i < world * k) {
            const uint32_t sh = i / k, j = i % k;
            const uint32_t n = min(g_n[(size_t)sh * n_q + q], k);
            if (j < n) {
                const size_t at = ((size_t)sh * n_q + q) * k + j;
                key = ((unsigned long long)__float_as_uint(g_dist[at]) << 32) | g_ids[at];
            }
        }
        s_keys[i] = key;
    }
    for (uint32_t sh = 0; sh < world; sh++) total += min(g_n[(size_t)sh * n_q + q], k);
    __syncthreads();
    for (uint32_t size = 2; size <= cap; size <<= 1)
        for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
            for (uint32_t i = threadIdx.x; i < cap; i += blockDim.x) {
                const uint32_t j = i ^ stride;
                if (j > i) {
                    const bool up = (i & size) == 0;
                    const unsigned long long a = s_keys[i], b = s_keys[j];
                    if ((a > b) == up) {
                        s_keys[i] = b;
                        s_keys[j] = a;
                    }
                }
            }
            __syncthreads();
        }
    const uint32_t n_out = min(total, k);
    for (uint32_t i = threadIdx.x; i < n_out; i += blockDim.x) {
        out_ids[(size_t)q * k + i] = (uint32_t)s_keys[i];
        out_dist[(size_t)q * k + i] = __uint_as_float((uint32_t)(s_keys[i] >> 32));
    }
    if (threadIdx.x == 0) out_n[q] = n_out;
}
cudaError_t launch_shard_merge(cudaStream_t s, const uint32_t *g_ids, const float *g_dist, const uint32_t *g_n, uint32_t world, uint32_t n_q,
                               uint32_t k, uint32_t *out_ids, float *out_dist, uint32_t *out_n) {
    if (!n_q) return cudaSuccess;
    uint32_t cap = 1;
    while (cap < world * k) cap <<= 1;
    const size_t smem = (size_t)cap * 8;
    if (smem > 200 * 1024) return cudaErrorInvalidValue;
    static bool attr_done = false;
    if (!attr_done) {
        cudaError_t e = cudaFuncSetAttribute(shard_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return e;
        attr_done = true;
    }
    shard_merge_kernel<<<n_q, 256, smem, s>>>(g_ids, g_dist, g_n, world, n_q, k, cap, out_ids, out_dist, out_n);
    return cudaGetLastError();
}

// ======================================================================================== launch wrappers
#define CK(x)                          \
    do {                               \
        cudaError_t e_ = (x);          \
        if (e_ != cudaSuccess) return e_; \
    } while (0)

cudaError_t launch_lev(cudaStream_t s, const uint8_t *dict_bytes, const uint32_t *dict_off, uint32_t n_words, const LevTerm *terms,
                       uint32_t n_terms, const uint32_t *term_idx, const LevChunk *chunks, const LevItem *items, uint32_t n_items,
                       LevRec *recs, uint32_t *rec_count, uint32_t *one_out, uint32_t *n_one, uint32_t *two_out, uint32_t *n_two,
                       int32_t *status) {
    if (n_terms == 0) return cudaSuccess;
    CK(cudaMemsetAsync(rec_count, 0, sizeof(uint32_t) * n_terms, s));
    if (n_items) lev_match_kernel<<<n_items, 256, 0, s>>>(dict_bytes, dict_off, n_words, terms, term_idx, chunks, items, recs, rec_count);
    lev_finalize_kernel<<<(n_terms + 63) / 64, 64, 0, s>>>(recs, rec_count, terms, n_terms, one_out, n_one, two_out, n_two, status);
    return cudaGetLastError();
}

cudaError_t launch_compact(cudaStream_t s, const CompactTile *tiles, uint32_t n_tiles, bool multi_segment, const ActDesc *acts,
                           uint32_t *seg_count, uint32_t *results) {
    if (!n_tiles) return cudaSuccess;
    if (multi_segment) act_count_kernel<<<n_tiles, COMPACT_THREADS, 0, s>>>(tiles, acts, seg_count);
    act_compact_kernel<<<n_tiles, COMPACT_THREADS, 0, s>>>(tiles, acts, seg_count, results);
    return cudaGetLastError();
}
cudaError_t launch_pair_probe(cudaStream_t s, const PairSet *sets, uint32_t n_sets, uint32_t n_probes, const uint32_t *wordpool,
                              const unsigned long long *pair_keys, uint64_t n_pairs, uint32_t pair_list_base, const DListRef *lists,
                              const ActDesc *acts, const uint32_t *results, Job *queue, uint32_t *qcount, uint32_t qcap) {
    if (!n_probes) return cudaSuccess;
    pair_probe_kernel<<<(n_probes + 255) / 256, 256, 0, s>>>(sets, n_sets, n_probes, wordpool, pair_keys, n_pairs, pair_list_base, lists, acts,
                                                             results, queue, qcount, qcap);
    return cudaGetLastError();
}
cudaError_t launch_scatter(cudaStream_t s, uint32_t n_ctas, const Job *queue, uint32_t *qcount, uint32_t qcap, const ActDesc *acts,
                           const uint32_t *results, const DListRef *lists, const uint32_t *pool, uint32_t *bigq) {
    scatter_kernel<<<n_ctas, 256, 0, s>>>(queue, qcount, qcap, acts, results, lists, pool, bigq);
    scatter_big_kernel<<<n_ctas, 256, 0, s>>>(queue, qcount, acts, results, lists, pool, bigq);
    return cudaGetLastError();
}
cudaError_t launch_eval(cudaStream_t s, int cls, const TileDesc *tiles, uint32_t n_tiles, const ActDesc *acts, uint32_t *results,
                        const ColOp *colprog, const uint16_t *costpool, const uint32_t *progpool, unsigned long long *tile_summary) {
    if (!n_tiles) return cudaSuccess;
    if (cls >= (int)EVAL_CLASSES) {
        eval_dp_kernel<false><<<n_tiles, 128, 0, s>>>(tiles, acts, results, colprog, costpool, progpool, tile_summary);
        return cudaGetLastError();
    }
    static bool attr_done = false;
    if (!attr_done) {
        CK(cudaFuncSetAttribute(eval_dp_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(EVAL_CLASS_SLOTS[EVAL_CLASSES - 1] * 1024)));
        attr_done = true;
    }
    eval_dp_kernel<true><<<n_tiles, 128, (size_t)EVAL_CLASS_SLOTS[cls] * 1024, s>>>(tiles, acts, results, colprog, costpool, progpool, tile_summary);
    return cudaGetLastError();
}
cudaError_t launch_walk(cudaStream_t s, int cls, const TileDesc *tiles, uint32_t n_tiles, const ActDesc *acts, uint32_t *results,
                        const ColOp *colprog, const DpState *states, const DpEdge *edges, const uint16_t *costpool, const uint32_t *progpool,
                        const unsigned long long *tile_summary, PathOut *pathbuf, uint32_t *path_count, uint32_t path_cap) {
    if (!n_tiles) return cudaSuccess;
    if (cls >= (int)EVAL_CLASSES) {
        walk_kernel<false><<<n_tiles, 128, 0, s>>>(tiles, acts, results, colprog, states, edges, costpool, progpool, tile_summary, pathbuf, path_count,
                                                   path_cap);
        return cudaGetLastError();
    }
    static bool attr_done = false;
    if (!attr_done) {
        CK(cudaFuncSetAttribute(walk_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(EVAL_CLASS_SLOTS[EVAL_CLASSES - 1] * 1024)));
        attr_done = true;
    }
    walk_kernel<true><<<n_tiles, 128, (size_t)EVAL_CLASS_SLOTS[cls] * 1024, s>>>(tiles, acts, results, colprog, states, edges, costpool, progpool,
                                                                             tile_summary, pathbuf, path_count, path_cap);
    return cudaGetLastError();
}
cudaError_t launch_emit(cudaStream_t s, const EmitDesc *emits, uint32_t n_emits) {
    if (!n_emits) return cudaSuccess;
    emit_kernel<<<n_emits, EMIT_THREADS, 0, s>>>(emits, n_emits);
    return cudaGetLastError();
}

cudaError_t launch_vec_dist(cudaStream_t s, int n_ctas, int qt, const void *mat, const float *inv_norm, const uint32_t *docids, uint64_t n_rows,
                            uint32_t d, const float *queries, const float *q_inv_norm, const unsigned long long *cand, uint64_t n_cand_words,
                            float *dist) {
    size_t smem = (size_t)qt * d * sizeof(float);
    const __half *m = reinterpret_cast<const __half *>(mat);
#define VD(QT)                                                                                                           \
    case QT:                                                                                                             \
        CK(cudaFuncSetAttribute(vec_dist_kernel<QT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));           \
        vec_dist_kernel<QT><<<n_ctas, 256, smem, s>>>(m, inv_norm, docids, n_rows, d, queries, q_inv_norm, cand, n_cand_words, dist); \
        break;
    switch (qt) {
        VD(1)
        VD(2)
        VD(4)
        VD(8)
        default: return cudaErrorInvalidValue;
    }
#undef VD
    return cudaGetLastError();
}
cudaError_t launch_topk(cudaStream_t s, uint32_t n_q, const float *dist, const uint32_t *docids, uint64_t n_rows, uint32_t k, uint32_t tie_cap,
                        uint32_t n_slices, float *part_dist, uint32_t *part_ids, uint32_t *part_n, float *out_dist, uint32_t *out_ids,
                        uint32_t *out_n) {
    if (!n_q) return cudaSuccess;
    if (n_slices <= 1) {
        topk_select_kernel<<<n_q, 1024, 0, s>>>(dist, n_rows, docids, 0, n_rows, 1, k, tie_cap, out_dist, out_ids, out_n);
        return cudaGetLastError();
    }
    const uint64_t part_len = (uint64_t)n_slices * (k + tie_cap);
    topk_select_kernel<<<n_q * n_slices, 1024, 0, s>>>(dist, n_rows, docids, 0, n_rows, n_slices, k, tie_cap, part_dist, part_ids, part_n);
    topk_select_kernel<<<n_q, 1024, 0, s>>>(part_dist, part_len, part_ids, part_len, part_len, 1, k, tie_cap, out_dist, out_ids, out_n);
    return cudaGetLastError();
}

}  // namespace b200
