// Launch wrappers of kernels.cu (host-callable; keep CUDA types out of the engine's headers).
#pragma once
#include <cuda_runtime.h>

#include "device_types.h"

namespace b200 {
// items / chunks / term_idx: the pruned schedule of Engine::derive_batch (one CTA per item)
cudaError_t launch_lev(cudaStream_t s, const uint8_t *dict_bytes, const uint32_t *dict_off, uint32_t n_words, const LevTerm *terms,
                       uint32_t n_terms, const uint32_t *term_idx, const LevChunk *chunks, const LevItem *items, uint32_t n_items,
                       LevRec *recs, uint32_t *rec_count, uint32_t *one_out, uint32_t *n_one, uint32_t *two_out, uint32_t *n_two,
                       int32_t *status);
// tiles: one per COMPACT_SEG parent rows of every activation; seg_count: n_tiles u32 scratch; multi_segment: some activation has > 1 segment
cudaError_t launch_compact(cudaStream_t s, const CompactTile *tiles, uint32_t n_tiles, bool multi_segment, const ActDesc *acts,
                           uint32_t *seg_count, uint32_t *results);
cudaError_t launch_pair_probe(cudaStream_t s, const PairSet *sets, uint32_t n_sets, uint32_t n_probes, const uint32_t *wordpool,
                              const unsigned long long *pair_keys, uint64_t n_pairs, uint32_t pair_list_base, const DListRef *lists,
                              const ActDesc *acts, const uint32_t *results, Job *queue, uint32_t *qcount, uint32_t qcap);
// qcount: [0] number of jobs (host + pair_probe), [2] work cursor, [3] big jobs noted, [4] big-job cursor ([2..4] must be 0 at
// launch); bigq: qcap u32 of scratch
cudaError_t launch_scatter(cudaStream_t s, uint32_t n_ctas, const Job *queue, uint32_t *qcount, uint32_t qcap, const ActDesc *acts,
                           const uint32_t *results, const DListRef *lists, const uint32_t *pool, uint32_t *bigq);
// evaluation of the activations' tiles, pass 1 (DP, buckets, counts); cls: eval_class() of the tiles' activations (EVAL_CLASSES =
// slots in global scratch); tile_summary: 2 u64 per tile (its non-empty buckets), indexed like `tiles`
cudaError_t launch_eval(cudaStream_t s, int cls, const TileDesc *tiles, uint32_t n_tiles, const ActDesc *acts, uint32_t *results,
                        const ColOp *colprog, const uint16_t *costpool, const uint32_t *progpool, unsigned long long *tile_summary);
// pass 2 over the same tiles: surviving paths of the buckets a query can still need (ActDesc::need)
cudaError_t launch_walk(cudaStream_t s, int cls, const TileDesc *tiles, uint32_t n_tiles, const ActDesc *acts, uint32_t *results,
                        const ColOp *colprog, const DpState *states, const DpEdge *edges, const uint16_t *costpool, const uint32_t *progpool,
                        const unsigned long long *tile_summary, PathOut *pathbuf, uint32_t *path_count, uint32_t path_cap);
cudaError_t launch_emit(cudaStream_t s, const EmitDesc *emits, uint32_t n_emits);
cudaError_t launch_vec_dist(cudaStream_t s, int n_ctas, int qt, const void *mat_fp16, const float *inv_norm, const uint32_t *docids,
                            uint64_t n_rows, uint32_t d, const float *queries, const float *q_inv_norm, const unsigned long long *cand,
                            uint64_t n_cand_words, float *dist);
// n_slices > 1: every query's distance row is selected in n_slices pieces side by side (part_*: n_q * n_slices * (k + tie_cap) slots
// and 2 counters per piece), then the pieces' candidates once more
cudaError_t launch_topk(cudaStream_t s, uint32_t n_q, const float *dist, const uint32_t *docids, uint64_t n_rows, uint32_t k, uint32_t tie_cap,
                        uint32_t n_slices, float *part_dist, uint32_t *part_ids, uint32_t *part_n, float *out_dist, uint32_t *out_ids,
                        uint32_t *out_n);

// staging of the vector store: f32 rows -> fp16 rows + inverse norms; inverse norms of fp16 rows
cudaError_t launch_emb_from_f32(cudaStream_t s, const float *in, void *out_fp16, float *inv_norm, uint64_t n, uint32_t d);
cudaError_t launch_emb_norm_f16(cudaStream_t s, const void *rows_fp16, float *inv_norm, uint64_t n, uint32_t d);

// corpus-sharded vector stage: merge `world` gathered per-shard top-k lists ([shard][query][k] + [shard][query] counts) per query
cudaError_t launch_shard_merge(cudaStream_t s, const uint32_t *g_ids, const float *g_dist, const uint32_t *g_n, uint32_t world, uint32_t n_q,
                               uint32_t k, uint32_t *out_ids, float *out_dist, uint32_t *out_n);

// ---- vec_gemm.cu: batched vector stage on tcgen05 (queries x matrix^T with the top-k fused into the epilogue)
#define VEC_GEMM_CAND_CAP 256
#define VEC_GEMM_KMAX 128
bool vec_gemm_supported(uint32_t d, uint32_t limit);
size_t vec_gemm_smem_bytes(uint32_t d, bool ts);
cudaError_t launch_vec_prep_queries(cudaStream_t s, const float *q, uint32_t n_q, uint32_t n_pad, uint32_t d, void *out_fp16, float *inv);
// runs: n_qtiles*n_groups*128*VEC_GEMM_CAND_CAP u64 scratch; partial: n_qtiles*128*n_groups*VEC_GEMM_KMAX u64
cudaError_t launch_vec_gemm_topk(cudaStream_t s, uint32_t sm_count, const void *mat_fp16, const float *inv_norm, const uint32_t *docids,
                                 uint64_t n_rows, uint32_t d, const void *q_fp16, const float *q_inv_norm, uint32_t n_qtiles, uint32_t n_groups,
                                 const unsigned long long *cand, uint64_t n_cand_words, uint32_t k, unsigned long long *gthr /* n_qtiles*128*n_groups u64 */,
                                 unsigned long long *runs,
                                 unsigned long long *partial, uint32_t *out_ids, float *out_dist, uint32_t *out_n, uint32_t n_q);
}  // namespace b200
