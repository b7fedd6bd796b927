// POD structures shared by the host engine and the CUDA kernels.
#pragma once
#include <cstdint>

namespace b200 {

struct DListRef {  // mirrors host ListRef
    unsigned long long off;
    uint32_t card;
    uint32_t dense;
};

// ---- term derivation (lev kernel) ----
constexpr int LEV_MAX_Q = 64;        // longest query word handled on device (bytes)
constexpr int LEV_TERMS_PER_CTA = 32;
constexpr int LEV_REC_CAP = 2048;    // match records (32 words each) per term
struct LevTerm {
    uint8_t q[LEV_MAX_Q];
    uint8_t len;
    int8_t k_same;    // budget when first chars are equal
    int8_t k_diff;    // budget when they differ (-1: excluded)
    uint8_t prefix;   // prefix automaton
};
struct LevRec {
    uint32_t base;              // first word id of the 32-word group
    uint32_t pad;
    unsigned long long codes;   // 2 bits per lane: 0 none, 1 same-first d=1, 2 same-first d=2, 3 different-first (d=1)
};
// Pruned derivation schedule (built by Engine::derive_batch): a term is only swept over the dictionary words whose first two
// bytes can pass the first-letter rule.  Those words form groups, each a union of id ranges of the sorted dictionary:
//   LEV_GROUP_F  (c): words with w[0] == c
//   LEV_GROUP_S  (c): words with w[1] == c (a one-byte word counts as w[1] == 0), minus those with w[0] in {q[0], q[1]} of the term
//   LEV_GROUP_ALL   : every word
constexpr uint8_t LEV_GROUP_F = 0, LEV_GROUP_S = 1, LEV_GROUP_ALL = 2;
struct LevChunk {     // up to LEV_TERMS_PER_CTA terms of one group
    uint32_t first;   // into the term index list
    uint8_t n, kind, c, pad;
};
struct LevItem {      // one CTA: one chunk against one 256-word tile that overlaps the chunk's group
    uint32_t tile, chunk;
};

// ---- rule activations ----
constexpr uint32_t MAX_COSTS = 128;
constexpr uint32_t JOB_CHUNK = 2048;  // elements (sparse) or rows (dense) per scatter job

// An activation evaluates a small DAG ("state graph") over the activation's universe, 64 documents per thread:
//   S[state][r] = documents that can go from `state` to END spending exactly r        (backward min-plus DP, bit-sliced)
//   bucket[ci]  = S[ROOT][cost_vals[ci]] minus the cheaper buckets                    (= the rule's buckets, all at once)
//   walk        = per document the first START->END path in edge order among its cheapest ones; distinct paths are
//                 reported to the host, which rebuilds the next query graph from them (graph_based_ranking_rule.rs:340-353)
struct DpState {
    uint32_t edge_begin;  // into DpEdge[], edges in visiting (DFS) order
    uint32_t pair_off;    // first S column of this state
    uint16_t n_edges;
    uint16_t rmin, rcount;  // S columns cover costs [rmin, rmin + rcount)
    uint16_t pad;
};
struct DpEdge {
    uint16_t dst;   // state index (always greater than the source: states are in topological order)
    uint16_t cost;
    uint16_t col;   // condition column, 0xffff = unconditional
    uint16_t pad;
};
constexpr uint32_t MAX_WALK = 14;  // edges on a START->END path (10 words + END, with slack)
struct PathOut {     // one distinct first-match path
    uint32_t act;
    uint16_t cost_idx;
    uint16_t len;
    uint16_t edges[MAX_WALK];  // activation-local DpEdge indices
};

struct ActDesc {
    // parent universe: rows (p_uw,p_ub); child = rows where OR(p_out[col_lo..col_hi)) != 0. p_out==0: take p_ub as is.
    const uint32_t *p_uw;            // nullptr => identity (row j is word j)
    const unsigned long long *p_ub;
    const unsigned long long *p_out; // column-major, leading dimension p_ld
    uint32_t p_rows, p_ld, p_col_lo, p_col_hi;
    // this activation
    uint32_t *uw;
    unsigned long long *ub;
    unsigned long long *C;    // column-major [n_cols][ld], scratch for this step
    unsigned long long *S;    // column-major [n_pairs][ld], scratch
    unsigned long long *out;  // column-major [n_costs+1][ld]; last column = matched by no path
    unsigned long long *tab;  // path dedup table (tab_size slots, zeroed), scratch
    uint32_t ld, n_cols, n_costs, n_states;
    uint32_t state_off, edge_off, cost_off;  // into DpState[], DpEdge[], u16 cost_vals[]
    uint32_t colprog_off, colprog_len;
    uint32_t prog_off, prog_len;  // DP program, u32 ops in the step's program pool; prog_len is a multiple of 4
    uint32_t n_pairs;             // (state, cost) pairs of the DP table; START's pairs come first, END's single pair last
    uint32_t root_rmin, root_rcount;  // START's cost range
    uint32_t need;                // documents bucket_sort can still use from this activation (hits left + offset left), saturating
    uint32_t tab_size, want_paths;
    uint32_t res_off;         // into results u32[]: [0] rows, [1..n_costs+1] counts, then: path-table saturation flag, last walked bucket
    uint32_t all_conditional; // every START->END path has at least one condition: rows whose columns are all zero match nothing
    // per-query lookup table word index -> (tag << 20 | row), written by act_compact, read by scatter instead of a binary search in
    // uw; nullptr = not available (then uw is searched).  Entries of other activations carry other tags.
    uint32_t *row_tab;
    uint32_t row_tag, pad_;
};

struct ColOp {  // executed per row before the paths
    uint16_t op;  // 0 AND dst=a&b, 1 OR dst=a|b, 2 ANDNOT dst=a&~b, 3 COPY dst=a
    uint16_t dst, a, b;
};

struct Job {  // scatter one chunk of one posting list into column `col` of activation `act`
    uint32_t act, col, list, chunk;
};

struct PairSet {  // expanded on device into Jobs: all (l, r) pairs of two word sets
    uint32_t act, col;
    uint32_t left_off, n_left, right_off, n_right;  // into the step's u32 word pool
    uint8_t fwd_prox, bwd_prox;  // 0 = no lookup in that direction
    uint8_t right_is_range;      // right entries are [lo,hi) dictionary ranges (prefix db): n_right pairs of u32
    uint8_t pad;
    uint32_t probe_base;         // first global probe index of this set
};

struct EmitDesc {  // append the first docids of OR(out[col_lo..col_hi)) to a result buffer
    const uint32_t *uw;
    const unsigned long long *ub;
    const unsigned long long *out;  // nullptr: emit ub itself
    uint32_t rows, ld, col_lo, col_hi;
    uint32_t skip, take;
    uint32_t *dst;
};

struct TileDesc {
    uint32_t act, row_begin;
    uint32_t rows_per_thread, pad;  // the tile covers 128 * rows_per_thread rows
};
// eval_dp_kernel keeps a row's condition words and DP table in thread-private shared-memory slots ([slot][128 rows] u64 = 1 KB per
// slot and CTA); a step's tiles are binned by the slot count (n_cols + n_pairs) of their activation, one launch per class; wider
// activations use the global-memory variant.
constexpr uint32_t EVAL_CLASSES = 8;
constexpr uint32_t EVAL_CLASS_SLOTS[EVAL_CLASSES] = {16, 24, 40, 56, 80, 112, 160, 216};
inline uint32_t eval_class(uint32_t slots) {
    for (uint32_t c = 0; c < EVAL_CLASSES; c++)
        if (slots <= EVAL_CLASS_SLOTS[c]) return c;
    return EVAL_CLASSES;
}
// DP program ops (built by the host, emit_activation_work): src slot | last-of-pair << 15 | condition slot << 16.  Slots of a row:
// [0, n_cols) condition columns, [n_cols, n_cols + n_pairs) DP table, then the constants ZERO and ONES.
constexpr uint32_t EVAL_EXTRA_SLOTS = 2;

// one segment of COMPACT_SEG parent rows of an activation's compaction (act_count_kernel / act_compact_kernel)
constexpr uint32_t COMPACT_SEG = 8192;
struct CompactTile {
    uint32_t act, seg;
    uint32_t first_tile;  // index of the activation's segment 0 in the tile list (segment counts are stored per tile)
    uint32_t n_seg;
};

}  // namespace b200
