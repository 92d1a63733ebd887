// device_types.h — structures shared by the host engine (engine.cu host half) and the kernels.
#pragma once
#include <stddef.h>
#include <stdint.h>

#include "../../include/qwgpu_format.h"

#ifndef QW_THREADS
#define QW_THREADS 512
#endif
#ifndef QW_MIN_BLOCKS_PER_SM
#define QW_MIN_BLOCKS_PER_SM 2
#endif
#define QW_WARPS (QW_THREADS / 32)
#define QW_MAX_INSTR 96
#define QW_MAX_DCOLS 16
#define QW_MAX_DAGGS 8
#define QW_MAX_LEVELS QW_MAX_PLAN_DEPTH
#define QW_MAX_TERMS 64      /* TERM instructions per plan */
#define QW_BLK_TAB 160       /* staged blocks per (term, window) before falling back to direct mode */
#define QW_MAX_WBLK 512      /* staged blocks per window over all terms */
#define QW_HIST_BINS 2048    /* 11-bit radix digits */
#define QW_DIGIT_BITS 11
#define QW_KEY_BITS 192
#define QW_CAND_CAP 8192     /* candidates kept per split before the final sort */
#define QW_MAX_TOPK 4096
#define QW_SMEM_AGG_CELLS 4096

enum { OP_TERM = 1, OP_RANGE = 2, OP_EXISTS = 3, OP_ALL = 4, OP_BOOL_BEGIN = 5, OP_BOOL_END = 6, OP_PHRASE = 7 };
enum { IF_SCORED = 1u, IF_HAS_TF = 2u, IF_HAS_FN = 4u, IF_BITS_FROM_SCORE = 8u };
#define QW_TFF_ROWS 16 /* tf-factor table: tff[tf][fieldnorm_id] = tf / (tf + norm[id]) for tf < 16 */

struct DInstr {  // 64 bytes
  uint32_t op, level, occur, flags;
  uint64_t a, b, c;  // TERM: data_off, widx_off, skip_off | RANGE: lo, hi | PHRASE: a = VBlk[] (device address), c = driver skip_off
  uint32_t n;        // TERM: num_blocks   | BOOL_END: n_req
  uint32_t m;        // TERM: win_shift    | BOOL_END: n_should
  uint32_t r;        // TERM: fn slot      | RANGE/EXISTS: column | BOOL_END: required_should
  float f;           // TERM: bm25 weight  | const-score leaves: boost
  uint32_t t;        // TERM: term slot (index among the plan's TERM instructions)
  uint32_t pad;
};

// A phrase evaluated by the pre-pass (phrase_kernel.cuh): one uncompressed posting block per 128-posting block of
// the phrase's driver term — doc = 0xFFFFFFFF where the driver posting's doc does not hold the phrase.
struct VBlk {
  uint32_t doc[QW_BLOCK_LEN];
  float val[QW_BLOCK_LEN];  // score contribution (0 when the phrase is not scored)
};
struct DPhraseTerm {
  uint64_t data_off, skip_off, pos_off, pidx_off;  // data-relative (QwImgTerm)
  uint32_t nblk, offset;                           // offset = position of the term inside the phrase
};
struct DPhrase {
  uint64_t data_base;  // the split's data region (device address)
  uint64_t out;        // VBlk[driver blocks] (device address)
  uint64_t fn_off;     // per-document fieldnorm ids, data-relative; ~0 = the field keeps none (constant id 1)
  uint64_t tab;        // the field's BM25 tables (device address): float[256] norms, then tff[16][256]
  float weight;        // (sum of the terms' idf) * (1 + K1) * boost
  uint32_t n_terms, driver, scored;
  uint32_t first_work, pad[3];  // prefix of driver blocks over the batch's phrases
  DPhraseTerm t[QW_MAX_PHRASE_TERMS];
};

struct DCol {  // 48 bytes
  uint64_t values_off, index_off, min_value, gcd;
  uint32_t bits, card, type, nwords64;
};

struct DAgg {
  uint32_t kind, parent, first_child, num_children;
  uint32_t col, num_buckets, has_bounds, num_ranges;
  uint32_t has_missing, cell_base;
  uint32_t is_f64;  // STATS: 1 = the cell sums f64 values, 0 = exact u64 sum of raws (qw_col_sum_exact on the host)
  uint32_t pad;
  double interval, offset, bound_min, bound_max;
  int64_t base_pos;
  // fast path (flat bucket aggregations over single-valued columns, see lower_plan): histogram
  // buckets are found in RAW space — bounds[k] = smallest bit-packed raw value that falls into
  // bucket >= k (k = 0..num_buckets), computed on the host with the reference f64 formula, so the
  // device needs no f64 arithmetic and stays bit-exact
  uint64_t bounds;       // device address of uint64[num_buckets + 1] (HISTOGRAM only)
  float inv_step;        // ~ num_buckets / (bounds[nb] - bounds[0]): first guess of the bucket
  uint32_t stat_base;    // STATS on the fast path: first of this node's {sum, ~min, max} triples in shared memory
  uint32_t pad3[2];      // keeps sizeof(DAgg) a multiple of 16 (copied to shared memory as uint4)
  uint64_t range_from[QW_MAX_AGG_RANGES], range_to[QW_MAX_AGG_RANGES];
};
static_assert(sizeof(DInstr) % 16 == 0 && sizeof(DCol) % 16 == 0 && sizeof(DAgg) % 16 == 0, "uint4-copied structs");

// Composite sort key: a big-endian bit string of at most 192 bits, greater = better, packed from the
// most significant bit with no padding between fields:
//   [has1:1][r1:rbits0] [has2:1][r2:rbits1] [doc':doc_bits]
// r_i is the RANK of sort value i: the column's bit-packed raw value (raw_max - raw for ascending
// order), or for _score a value-linear 10-bit bucket followed by the order-preserving f32 bits (42
// bits as first key, 32 as second). A field that cannot discriminate (doc-id sort, column absent from
// the split) contributes no bits at all. doc' is the doc id (complemented within doc_bits when the
// first order is ascending). This is exactly the total order of SegmentPartialHitSortingKey
// (quickwit-search/src/collector.rs:1082-1112), None last; because the fields are only as wide as
// the split's data needs, every 11-bit radix digit of the key discriminates.
struct alignas(16) DKeySpec {
  uint32_t kind[2], order[2], col[2];
  uint32_t rbits[2];     // width of r_i
  uint32_t hasbit[2];    // 1: a has-value bit precedes r_i
  uint32_t doc_bits, total_bits;
  uint32_t top_mode;     // how the first 11 key bits are derived cheaply (QW_TOP_*)
  float score_scale;     // SCORE: lin = min(1023, (uint)(score * scale))
  uint64_t raw_max[2];   // r_i = order == DESC ? raw : raw_max - raw
  // total_bits <= 64 (the usual case): the key is w0 = OR of (field << shift), shifts precomputed
  uint32_t narrow, sh_has[2], sh_r[2], sh_doc;
};
static_assert(sizeof(DKeySpec) % 16 == 0, "uint4-copied struct");
enum { QW_TOP_FULL = 0, QW_TOP_SCORE = 1, QW_TOP_COLUMN = 2, QW_TOP_DOC = 3 };

struct DThresh {  // per split, device-resident, written by k_pick
  uint64_t key[3];       // candidates are docs with composite key >= key
  uint32_t prefix_bits;  // number of leading bits of `key` that are fixed so far
  uint32_t above;        // docs strictly above the prefix (exact path bookkeeping)
  uint32_t done;         // 1 when the candidate set fits QW_CAND_CAP
  uint32_t matched;      // docs matching the prefix at the last level
};

struct DSplitPlan {
  uint64_t data_base;  // device address of the split's data region
  uint32_t num_docs, num_windows;
  uint32_t n_instr, instr_base;
  uint32_t n_cols, col_base;
  uint32_t n_aggs, agg_base;
  uint32_t n_terms, n_levels;
  uint32_t max_hits, scoring;
  uint32_t n_fn_slots, n_cells;
  uint32_t fused_score_root;  // root bool is a pure OR of positive-weight scored terms
  uint32_t fast_aggs;         // every aggregation is a bucket aggregation (optionally with stats children)
                              // or a stats node over always-present single-valued columns
  uint32_t n_stat_cells, pad1;  // fast path: number of privatised stats cells
  uint64_t fn_off[2];      // data-relative fieldnorm arrays staged per window
  uint64_t bm25_tab[2];    // device addresses of float[256] BM25 norm tables, followed by the
                           // float[QW_TFF_ROWS][256] tf-factor table of the same field
  DKeySpec key;
  QwSearchAfter sa;
  uint64_t out_num_hits;   // device address of a uint64 counter
  uint64_t out_hist;       // device address of uint32[QW_HIST_BINS]
  uint64_t out_cand_count; // device address of a uint32 counter
  uint64_t out_cands;      // device address of uint64[3 * QW_CAND_CAP]
  uint64_t out_cells;      // device address of QwAggCell[n_cells]
  uint64_t out_hits;       // device address of QwHit[max_hits]
  uint64_t out_nhits;      // device address of uint32 (hits written by k_select)
};

static_assert(offsetof(DSplitPlan, key) % 16 == 0 && sizeof(DSplitPlan) % 16 == 0, "DKeySpec is read as uint4");

struct SmemLevel {
  uint32_t req, shd, nt, cnt, msum, ssum;  // byte offsets; 0xFFFFFFFF = not allocated
  uint32_t rsc, pad;                       // result score array of the level (msum, else ssum)
};
struct SmemLayout {
  uint32_t instr, cols, aggs, key, hitq;  // hitq: per-warp compacted hit queues of the generic collect
  uint32_t rangeq;  // per-warp queues of required RANGE / EXISTS clauses (0xFFFFFFFF: probe per bitmap word)
  SmemLevel lvl[QW_MAX_LEVELS];
  uint32_t tmp, fn[2];          // scratch bitmap; staged fieldnorm bytes per scored field
  uint32_t rng, blkrec, termblk, stage, hist, misc;  // hist aliases stage (dead by collect time)
  uint32_t l0hist;  // COLLECT pass: exact level-0 digit histogram of the window's matches (0xFFFFFFFF: not recorded)
  uint32_t total;
};

struct KParams {
  const DSplitPlan* plans;
  const DInstr* instrs;
  const DCol* cols;
  const DAgg* aggs;
  DThresh* thresh;
  const uint32_t* first_work;  // prefix over splits of (sampled) window counts; [n_splits + 1]
  uint32_t n_splits;
  uint32_t total_work;
  uint32_t stride;   // sampling stride over windows (1 = all)
  uint32_t W;        // window size in docs (power of two, <= 8192)
  uint32_t level;    // MODE_HIST: radix level being histogrammed
  uint32_t use_prefix;  // MODE_HIST: restrict to docs whose key matches thresh prefix
  uint32_t smem_aggs;   // 1: aggregation counts privatised in shared memory
  uint32_t stage_bytes; // capacity of the posting staging area
  // second-chance top-K (engine.cu): a COLLECT pass may record the exact level-0 histogram and each
  // window's best level-0 digit; refinement passes then skip verified splits and windows that cannot
  // hold a candidate, and only emit candidates (hit counts / aggregations are already final)
  uint32_t rec_l0;        // COLLECT: record out_hist + wmax
  uint32_t refine;        // 1: skip splits with split_state == 0 and windows with wmax < threshold digit
  uint32_t cands_only;    // COLLECT: emit candidates only
  uint16_t* wmax;         // per flat window: 1 + best level-0 digit among its matches (0: no match)
  const uint32_t* split_state;  // per split: 1 = needs refinement
  const uint32_t* sample_win;   // sampled passes: per work item, window | edge << 31 (null: strided formula)
  SmemLayout sm;
};
