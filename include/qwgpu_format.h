/*
 * qwgpu_format.h — plain-old-data layouts shared across the C ABI of libqwgpu:
 *   (1) the split IMAGE (what a registered split looks like in host memory / HBM),
 *   (2) the per-split search PLAN (seam C of SURVEY.md §3.4: what replaces
 *       `searcher.search(&query, &collector)` at quickwit-search/src/leaf.rs:637),
 *   (3) the per-split RESULT (the fields of `LeafSearchResponse` produced by
 *       `QuickwitSegmentCollector::harvest`, quickwit-search/src/collector.rs:564-594).
 *
 * Everything is little-endian, naturally aligned, no pointers — only byte offsets — so the same
 * bytes can be mmapped, sent over FFI from Rust (`#[repr(C)]`), or copied to the device verbatim.
 *
 * The image follows the SHAPES of a tantivy segment (SURVEY.md Appendix A: 128-doc bit-packed
 * posting blocks with 4-lane interleave + skip entries, 1-byte fieldnorm ids, bit-packed columns
 * with min/gcd header, dictionary-encoded string columns), but it is OUR format: tantivy's byte
 * layout is not pinned by anything in /root/reference (SURVEY.md §8c "NOT pinned").
 */
#ifndef QWGPU_FORMAT_H
#define QWGPU_FORMAT_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QW_IMG_MAGIC 0x31474D4947575151ull /* "QQWGIMG1" */
#define QW_IMG_VERSION 3u
#define QW_BLOCK_LEN 128u                  /* tantivy COMPRESSION_BLOCK_SIZE */
#define QW_TERMINATED 0x7FFFFFFFu          /* tantivy TERMINATED sentinel (i32::MAX as u32) */
#define QW_NO_PREV_DOC 0xFFFFFFFFu
#define QW_MIN_WIN_SHIFT 12u /* index windows are >= 4096 docs; an evaluation window (<= 8192 docs) spans <= 2 entries */

/* ---------------------------------------------------------------- image ---------------------- */

typedef struct QwImgHeader {
  uint64_t magic;
  uint32_t version;
  uint32_t num_docs;
  uint32_t num_fields;  /* inverted (text) fields */
  uint32_t num_terms;   /* dictionary entries over all fields, sorted by (field_id, bytes) */
  uint32_t num_columns; /* fast fields */
  uint32_t reserved0;
  uint64_t fields_off;     /* QwImgField[num_fields] */
  uint64_t terms_off;      /* QwImgTerm[num_terms]   */
  uint64_t term_bytes_off; /* concatenated term bytes */
  uint64_t term_bytes_len;
  uint64_t columns_off; /* QwImgColumn[num_columns] */
  uint64_t strings_off; /* names + column dictionaries (host-only blob) */
  uint64_t strings_len;
  uint64_t data_off; /* device-resident region: postings, skip lists, fieldnorms, column data */
  uint64_t data_len; /* multiple of 16 */
  uint64_t total_len;
  uint64_t reserved1[3];
} QwImgHeader; /* 128 bytes */

enum { QW_FIELD_HAS_FREQS = 1u, QW_FIELD_HAS_FIELDNORMS = 2u, QW_FIELD_HAS_POSITIONS = 4u };
enum { QW_TOK_RAW = 0u, QW_TOK_DEFAULT = 1u };

typedef struct QwImgField {
  uint32_t name_off, name_len; /* into strings blob */
  uint32_t flags;              /* QW_FIELD_* */
  uint32_t tokenizer;          /* QW_TOK_* */
  uint64_t total_num_tokens;   /* Σ field lengths; average_fieldnorm = total / num_docs */
  uint64_t fieldnorm_off;      /* data-relative; num_docs bytes (fieldnorm ids); valid iff HAS_FIELDNORMS */
  uint32_t first_term, num_terms;
  uint64_t reserved;
} QwImgField; /* 48 bytes */

typedef struct QwImgTerm {
  uint32_t field_id;
  uint32_t bytes_off, bytes_len; /* into term bytes blob */
  uint32_t doc_freq;
  uint32_t num_blocks; /* ceil(doc_freq / 128) */
  uint32_t win_shift;  /* window index granularity: one entry per 2^win_shift docs (>= 12) */
  uint64_t skip_off; /* data-relative: QwSkip[num_blocks] (CPU-style seek structure) */
  uint64_t data_off; /* data-relative: blocks, each [QwSkip header][packed docs][packed tfs][fieldnorm ids] */
  uint64_t data_len;
  uint64_t widx_off; /* data-relative: QwWinIdx[ceil(num_docs / 2^win_shift)] */
  uint64_t tf_len;   /* bytes of data_len that are packed term frequencies (roofline accounting) */
  uint64_t fn_len;   /* bytes of data_len that are per-posting fieldnorm ids (128 per block, see QwSkip) */
  uint64_t sub_off;  /* data-relative: QwSubIdx[num_blocks] (doc-id checkpoints inside each block) */
  /* positions (fields indexed with `record: position`, QW_FIELD_HAS_POSITIONS; both 0 otherwise): the token
   * positions of every posting, in posting order — posting i owns tf[i] consecutive entries, ascending
   * (tantivy's .pos stream keeps them delta-bit-packed per 128 positions; here they are plain uint32) */
  uint64_t pos_off;  /* data-relative: uint32 positions[sum of tf] */
  uint64_t pidx_off; /* data-relative: uint32 first_pos[num_blocks + 1] — index into positions[] of the first
                        position of each block; [num_blocks] = sum of tf */
} QwImgTerm; /* 96 bytes */

/* Window index: for index-window j (docs [j<<win_shift, (j+1)<<win_shift)) the byte range
 * [start, end) of QwImgTerm data holding every block that overlaps it (start == end if none).
 * This is what lets a GPU thread block that owns a doc-id window fetch exactly the posting bytes
 * it needs with ONE dependent load instead of a binary search over the skip list. */
typedef struct QwWinIdx {
  uint32_t start, end;             /* byte range inside QwImgTerm data */
  uint32_t first_block, end_block; /* the same blocks as ordinals into the skip list */
} QwWinIdx;

/* One skip entry per posting block; 16 bytes = one coalesced 128-bit load.
 * A block holds `count` (1..128) postings. Doc ids are stored as strictly-sorted deltas:
 *   v[i] = doc[i] - doc[i-1] - 1, with doc[-1] := prev_last_doc (0xFFFFFFFF for the first block,
 *   arithmetic mod 2^32), bit-packed at `doc_bits` bits with the BitPacker4x interleave
 *   (value i lives in lane i%4 at position i/4; 128-bit word w holds 32-bit word w of the four
 *   lanes) => 16*doc_bits bytes. Term frequencies follow, raw, at `tf_bits` bits => 16*tf_bits
 *   bytes (tf_bits == 0 when the field is indexed `record: basic`; tf := 1).
 * When the field has fieldnorms, 128 bytes follow: the fieldnorm id of each posting's document
 * (byte i = fieldnorm id of doc[i], zero padded). tantivy keeps fieldnorms per document only; the
 * image ALSO keeps that array (QwImgField.fieldnorm_off) but denormalises the id next to every
 * posting so that BM25 scoring reads one contiguous byte stream per block instead of a random
 * 1-byte gather per posting (the bytes read equal SURVEY.md 8d's "1 B per scored posting").
 * The trailing partial block uses the same layout, zero padded (tantivy VInt-encodes it; a
 * real-split ingester transcodes, SURVEY.md §8f-2). */
typedef struct QwSkip {
  uint32_t last_doc;
  uint32_t prev_last_doc;
  uint32_t byte_off; /* of this block's inline header, relative to QwImgTerm.data_off */
  uint8_t doc_bits;
  uint8_t tf_bits;
  uint16_t count;
} QwSkip;

/* Checkpoints inside a posting block: the doc id reached after 32, 64 and 96 postings, relative to
 * prev_last_doc (mod 2^32), and the block's whole span. A reader that only needs the postings of a
 * doc-id sub-range can start decoding at any 32-posting boundary (sub-block s starts from
 * prev_last_doc + ck[s-1]) instead of prefix-summing the block from its beginning — the GPU union
 * kernel gives every warp its own doc-id range of a window and decodes only the sub-blocks that
 * overlap it. Sub-blocks past `count` are empty and repeat `span`. */
typedef struct QwSubIdx {
  uint32_t ck[3]; /* doc[32k - 1] - prev_last_doc for k = 1..3 (span when 32k > count) */
  uint32_t span;  /* last_doc - prev_last_doc */
} QwSubIdx;

enum {
  QW_COL_U64 = 0,
  QW_COL_I64 = 1,
  QW_COL_F64 = 2,
  QW_COL_BOOL = 3,
  QW_COL_DATETIME = 4, /* i64 nanoseconds, truncated to fast_precision at build time */
  QW_COL_STR = 5       /* term ordinals into a sorted dictionary */
};
enum { QW_CARD_FULL = 0, QW_CARD_OPTIONAL = 1, QW_CARD_MULTI = 2 };

/* Column values are stored in tantivy's order-preserving u64 mapping
 * (MonotonicallyMappableToU64: i64 -> x ^ 1<<63, f64 -> sign-flip trick, bool -> 0/1,
 * DateTime -> i64 nanos, Str -> ordinal) as raw = (mapped - min_value) / gcd, bit-packed
 * little-endian at `bits` bits per value (value i occupies bits [i*bits, (i+1)*bits)).
 * index (data-relative):
 *   FULL:     none; value index == doc id.
 *   OPTIONAL: uint64 present[ceil(num_docs/64)] then uint32 rank[ceil(num_docs/64)+1]
 *             (rank[w] = number of set bits before word w); value index = rank + popc(below).
 *   MULTI:    uint32 start[num_docs+1]; values of doc d are [start[d], start[d+1]). */
typedef struct QwImgColumn {
  uint32_t name_off, name_len;
  uint32_t type;        /* QW_COL_* */
  uint32_t cardinality; /* QW_CARD_* */
  uint64_t min_value, max_value, gcd;
  uint64_t num_vals;
  uint32_t bits;
  uint32_t dict_num_terms; /* STR only */
  uint64_t values_off, values_len; /* data-relative; padded with 16 zero bytes */
  uint64_t index_off, index_len;   /* data-relative */
  uint64_t dict_off, dict_len;     /* strings-blob relative: uint32 offs[n+1] then bytes */
  uint64_t reserved;
} QwImgColumn; /* 112 bytes */

/* ---------------------------------------------------------------- plan ----------------------- */

#define QW_PLAN_MAGIC 0x4E4C5051u /* "QPLN" */
#define QW_MAX_PLAN_DEPTH 4
#define QW_MAX_PHRASE_TERMS 8

enum {
  QW_NODE_TERM = 1,   /* tantivy TermQuery */
  QW_NODE_RANGE = 2,  /* tantivy FastFieldRangeQuery; const score 1 */
  QW_NODE_BOOL = 3,   /* tantivy BooleanQuery */
  QW_NODE_ALL = 4,    /* AllQuery; score 1 */
  QW_NODE_NONE = 5,   /* EmptyQuery */
  QW_NODE_EXISTS = 6, /* ExistsQuery on a column; const score 1 */
  QW_NODE_PHRASE = 7  /* tantivy PhraseQuery, slop 0: children = its TERM nodes in phrase order, all of one field
                         with positions; child k's `lo` = position offset of the term inside the phrase. A doc
                         matches when some base position b has term k at b + lo_k for every k; phrase_count =
                         number of such b. Score = bm25_weight * tf-factor(phrase_count, fieldnorm) with
                         bm25_weight = (sum of the terms' idf, duplicates included) * (1 + K1) * boost
                         (Bm25Weight::for_terms). */
};
enum { QW_OCCUR_MUST = 0, QW_OCCUR_SHOULD = 1, QW_OCCUR_MUST_NOT = 2, QW_OCCUR_FILTER = 3 };

/* Children of a BOOL node are the nodes [first_child, first_child + num_children) in the node
 * array, each tagged with its `occur`. FILTER = Must(ConstScoreQuery(q, 0.0))
 * (quickwit-query/src/query_ast/tantivy_query_ast.rs:345-377). */
typedef struct QwPlanNode {
  uint32_t kind;
  uint32_t occur; /* role in the parent BOOL (ignored for the root) */
  float boost;    /* multiplies the node's score (QueryAst::Boost); 1.0 by default */
  uint32_t first_child, num_children;
  uint32_t min_should_match; /* BOOL; 0xFFFFFFFF = unset */
  /* TERM */
  uint32_t term_ord;  /* index into QwImgTerm[]; 0xFFFFFFFF = term absent from the split */
  uint32_t field_id;
  float bm25_weight;  /* idf * (1 + K1), already including boost; host-computed (f32) */
  /* RANGE / EXISTS */
  uint32_t column;  /* index into QwImgColumn[]; 0xFFFFFFFF = column absent */
  uint64_t lo, hi;  /* inclusive bounds in the column's mapped-u64 space */
} QwPlanNode; /* 56 bytes */

enum { QW_SORT_NONE = 0, QW_SORT_DOCID = 1, QW_SORT_SCORE = 2, QW_SORT_COLUMN = 3 };
enum { QW_ORDER_ASC = 0, QW_ORDER_DESC = 1 }; /* quickwit SortOrder: ASC=0, DESC=1 */

typedef struct QwSortSpec {
  uint32_t kind;   /* QW_SORT_* (QW_SORT_NONE only valid for the second key) */
  uint32_t order;  /* QW_ORDER_* */
  uint32_t column; /* QW_SORT_COLUMN: column index, 0xFFFFFFFF = missing (all None) */
  uint32_t reserved;
} QwSortSpec;

/* search_after, already converted to the u64 fast-field space
 * (SearchAfterSegment::new, quickwit-search/src/top_k_collector.rs:829-872). */
typedef struct QwSearchAfter {
  uint32_t present;
  uint32_t has_v1, has_v2;
  uint32_t compare_on_equal; /* !search_after.split_id.is_empty() */
  int32_t precomp_order;     /* order1.compare(split_id, sa.split_id).then(segment_ord): -1/0/1 */
  uint32_t doc_id;
  uint64_t v1, v2;
} QwSearchAfter;

enum {
  QW_AGG_TERMS = 1,
  QW_AGG_HISTOGRAM = 2,      /* also date_histogram (interval/offset pre-scaled to column units) */
  QW_AGG_RANGE = 3,
  QW_AGG_STATS = 4           /* stats / avg / sum / min / max / value_count share one collector */
};

#define QW_MAX_AGG_RANGES 16

/* One aggregation node. Bucket aggregations may have children (sub-aggregations):
 * nodes [first_child, first_child+num_children). Top-level aggs have parent == 0xFFFFFFFF. */
typedef struct QwAggNode {
  uint32_t kind;
  uint32_t parent;
  uint32_t first_child, num_children;
  uint32_t column;      /* 0xFFFFFFFF = column absent in this split */
  uint32_t num_buckets; /* dense bucket space of this node in this split (host-computed) */
  /* HISTOGRAM: bucket_pos = floor((val_f64 - offset) / interval) (all in column units, f64);
   * dense index = bucket_pos - base_pos. */
  double interval, offset;
  int64_t base_pos;
  /* hard_bounds (inclusive, f64 in column units); has_bounds=0 when absent */
  uint32_t has_bounds;
  uint32_t num_ranges;
  double bound_min, bound_max;
  /* RANGE: bucket i = [range_from[i], range_to[i]) in mapped-u64 space */
  uint64_t range_from[QW_MAX_AGG_RANGES], range_to[QW_MAX_AGG_RANGES];
  /* TERMS on numeric columns: dense index = raw value; on STR: ordinal */
  uint32_t has_missing;  /* `missing` parameter present */
  uint32_t reserved;
  uint64_t missing_value; /* mapped-u64 (numeric) or ordinal==dict_num_terms for "new key" */
} QwAggNode;

typedef struct QwPlanHeader {
  uint32_t magic;
  uint32_t version;
  uint32_t num_nodes; /* query nodes; node 0 is the root */
  uint32_t num_aggs;  /* QwAggNode count */
  uint32_t max_hits;  /* leaf_max_hits = max_hits + start_offset (collector.rs:772-774) */
  uint32_t scoring;   /* QuickwitCollector::requires_scoring (collector.rs:819-830) */
  uint32_t count_only; /* max_hits == 0 && no aggregation (collector.rs:723-725) */
  uint32_t reserved;
  QwSortSpec sort[2];
  QwSearchAfter search_after;
  /* followed by QwPlanNode[num_nodes], then QwAggNode[num_aggs] */
} QwPlanHeader;

/* ---------------------------------------------------------------- result --------------------- */

/* One hit of the per-split top-K, best first. v1/v2 are the u64 fast-field representations
 * (SegmentPartialHit, collector.rs:484-491); for QW_SORT_SCORE v1 = f64_to_u64(score as f64)
 * (collector.rs:180) and `score` carries the raw f32. */
typedef struct QwHit {
  uint64_t v1, v2;
  uint32_t doc_id;
  uint32_t flags; /* bit0: v1 is Some, bit1: v2 is Some */
  float score;
  uint32_t reserved;
} QwHit;

/* Dense aggregation result. Every QwAggNode owns `cells(node)` = Π num_buckets over its ancestor
 * chain (itself included; metric nodes count 1) cells, laid out row-major (outermost ancestor
 * slowest). Bucket nodes use only `count` (doc_count). Metric nodes (QW_AGG_STATS) use all four:
 * `sum_bits`: for columns where qw_col_sum_exact() holds, the exact integer sum of the RAW offsets
 * (value = min_value + gcd * raw in the mapped space) — the host rebuilds count * min + gcd * sum in
 * 128-bit arithmetic, so e.g. an avg over nanosecond timestamps cannot overflow; for every other
 * column, the bit pattern of an f64 sum of the typed values (what tantivy accumulates). min/max are
 * in the column's mapped-u64 space (initialised to UINT64_MAX / 0). The host converts to f64 when it
 * builds the intermediate aggregation result. */
#define QW_SUM_EXACT_BITS 40u /* widest raw that may take the exact integer sum (see qw_col_sum_exact) */

/* How a stats cell sums a column: 1 = exact uint64 sum of the raw offsets, 0 = f64 sum of the typed values.
 * Exact only for integer-typed columns whose raws are at most QW_SUM_EXACT_BITS wide AND whose raws cannot
 * wrap a uint64 when all of them are added: num_vals * (2^bits - 1) < 2^64. A cell sums a subset of the
 * column's values, so the bound holds for every cell. The width alone is not enough: a multi-valued column
 * holds more values than docs, and 2^24 values of 40 bits already reach 2^64. The oracle, the kernels (through
 * DAgg::is_f64) and the host finalisation all decide with this one predicate. */
static inline int qw_col_sum_exact(const QwImgColumn* c) {
  if (c->type == QW_COL_F64 || c->bits > QW_SUM_EXACT_BITS) return 0;
  return c->bits == 0 || c->num_vals <= UINT64_MAX / ((1ull << c->bits) - 1);
}
typedef struct QwAggCell {
  uint64_t count;
  uint64_t sum_bits;
  uint64_t min_mapped;
  uint64_t max_mapped;
} QwAggCell;

#ifdef __cplusplus
}
#endif
#endif /* QWGPU_FORMAT_H */
