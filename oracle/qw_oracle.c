/*
 * qw_oracle.c — CPU ORACLE for the per-split leaf-search hot path.  TEST INFRASTRUCTURE ONLY.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
 * load this. The product (libqwgpu.so) never links, calls or falls back to anything in here.
 *
 * PARITY STATUS: "semantics pinned, byte format unpinned". The arithmetic of this path lives in
 * tantivy 0.26.0 @ edfb02b (+ tantivy-columnar 0.7.0, tantivy-bitpacker 0.10.0, bitpacking 0.9.3),
 * an un-vendored git dependency absent from /root/reference (quickwit/Cargo.toml:385-391), and no
 * Rust toolchain exists here, so oracle/_ref cannot be built. This file restates the published
 * algorithms (SURVEY.md Appendix A) doc-at-a-time, the way tantivy drives a SegmentCollector, and
 * is pinned against every golden vector the reference's own tests hold for this path
 * (tests/test_oracle_goldens.py; SURVEY.md §8c). The split bytes it reads are OUR image format
 * (include/qwgpu_format.h), decoded here by an independent scalar reader.
 *
 * Each function cites the reference file:line whose behaviour it follows (paths relative to
 * /root/reference/quickwit/).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "../include/qwgpu_format.h"

/* ------------------------------------------------------------------ image reader ------------- */
typedef struct {
  const uint8_t* base;
  const QwImgHeader* hdr;
  const QwImgField* fields;
  const QwImgTerm* terms;
  const QwImgColumn* cols;
  const uint8_t* data;
} OImg;

static int oimg_open(OImg* im, const uint8_t* p, uint64_t n) {
  if (n < sizeof(QwImgHeader)) return -1;
  im->base = p;
  im->hdr = (const QwImgHeader*)p;
  if (im->hdr->magic != QW_IMG_MAGIC || im->hdr->total_len > n) return -1;
  im->fields = (const QwImgField*)(p + im->hdr->fields_off);
  im->terms = (const QwImgTerm*)(p + im->hdr->terms_off);
  im->cols = (const QwImgColumn*)(p + im->hdr->columns_off);
  im->data = p + im->hdr->data_off;
  return 0;
}

/* tantivy FIELD_NORMS_TABLE (Lucene SmallFloat byte4ToInt), SURVEY.md Appendix A.3. */
static uint32_t o_id_to_fieldnorm(uint32_t id) {
  if (id < 24) return id;
  uint32_t i = id - 24, bits = i & 7, shift = i >> 3;
  return 24 + (shift == 0 ? bits : ((bits | 8) << (shift - 1)));
}

/* Scalar unpack of one 4-lane-interleaved block (bitpacking::BitPacker4x layout, App. A.2):
 * value i sits in lane i%4 at position i/4; 128-bit word w = word w of lanes 0..3. */
static void o_unpack_4x(const uint8_t* p, uint32_t bits, uint32_t* out) {
  if (bits == 0) { memset(out, 0, 4 * QW_BLOCK_LEN); return; }
  const uint32_t* w = (const uint32_t*)p;
  uint64_t mask = bits == 32 ? 0xFFFFFFFFull : ((1ull << bits) - 1);
  for (uint32_t i = 0; i < QW_BLOCK_LEN; i++) {
    uint32_t lane = i & 3, k = i >> 2;
    uint64_t bitpos = (uint64_t)k * bits;
    uint32_t wi = (uint32_t)(bitpos >> 5), sh = (uint32_t)(bitpos & 31);
    uint64_t lo = w[4 * wi + lane];
    uint64_t hi = (sh + bits > 32) ? w[4 * (wi + 1) + lane] : 0;
    out[i] = (uint32_t)(((lo | (hi << 32)) >> sh) & mask);
  }
}

/* tantivy-bitpacker BitUnpacker::get: value idx at bit offset idx*bits, little endian. */
static uint64_t o_col_raw(const OImg* im, const QwImgColumn* c, uint64_t idx) {
  if (c->bits == 0) return 0;
  const uint8_t* v = im->data + c->values_off;
  uint64_t bitpos = idx * c->bits, byte = bitpos >> 3;
  uint32_t sh = (uint32_t)(bitpos & 7);
  uint64_t lo;
  memcpy(&lo, v + byte, 8);
  uint64_t val = lo >> sh;
  if (sh + c->bits > 64) { uint64_t hi = v[byte + 8]; val |= hi << (64 - sh); }
  return c->bits == 64 ? val : (val & ((1ull << c->bits) - 1));
}
static uint64_t o_col_mapped(const OImg* im, const QwImgColumn* c, uint64_t idx) {
  return c->min_value + c->gcd * o_col_raw(im, c, idx);
}
/* value index range [*a, *b) of doc d (Column::values_for_doc) */
static void o_col_range(const OImg* im, const QwImgColumn* c, uint32_t d, uint64_t* a, uint64_t* b) {
  if (c->cardinality == QW_CARD_FULL) { *a = d; *b = (uint64_t)d + 1; return; }
  const uint8_t* ix = im->data + c->index_off;
  if (c->cardinality == QW_CARD_OPTIONAL) {
    uint32_t nw = (im->hdr->num_docs + 63) / 64;
    const uint64_t* present = (const uint64_t*)ix;
    const uint32_t* rank = (const uint32_t*)(ix + 8ull * nw);
    uint64_t word = present[d >> 6];
    if (!((word >> (d & 63)) & 1)) { *a = *b = 0; return; }
    uint64_t below = word & ((1ull << (d & 63)) - 1);
    *a = rank[d >> 6] + (uint64_t)__builtin_popcountll(below);
    *b = *a + 1;
    return;
  }
  const uint32_t* start = (const uint32_t*)ix;
  *a = start[d]; *b = start[d + 1];
}
/* Column::first(doc) -> Option<u64> (quickwit-search/src/collector.rs:177-179) */
static int o_col_first(const OImg* im, const QwImgColumn* c, uint32_t d, uint64_t* out) {
  uint64_t a, b;
  o_col_range(im, c, d, &a, &b);
  if (a == b) return 0;
  *out = o_col_mapped(im, c, a);
  return 1;
}

static double o_mapped_to_f64(uint32_t type, uint64_t m) {
  switch (type) {
    case QW_COL_U64: case QW_COL_BOOL: case QW_COL_STR: return (double)m;
    case QW_COL_I64: case QW_COL_DATETIME: return (double)(int64_t)(m ^ (1ull << 63));
    default: {
      uint64_t bits = (m & (1ull << 63)) ? (m ^ (1ull << 63)) : ~m;
      double d; memcpy(&d, &bits, 8); return d;
    }
  }
}
static uint64_t o_f64_to_u64(double d) {
  uint64_t bits; memcpy(&bits, &d, 8);
  return (bits & (1ull << 63)) ? ~bits : (bits ^ (1ull << 63));
}

/* ------------------------------------------------------------------ docsets ------------------ */
/* tantivy DocSet/Scorer contract: doc(), advance(), seek(target >= doc), score(); TERMINATED when
 * exhausted (in-reference example of the contract: quickwit-query/src/query_ast/cache_node.rs:153-306). */
typedef struct DocSet DocSet;
struct DocSet {
  int kind;
  uint32_t doc;
  float boost;
  uint32_t occur;
  /* TERM: BlockSegmentPostings + Bm25Weight */
  const QwSkip* skips; const uint8_t* tdata;
  uint32_t nblocks, blk, cnt, pos, has_tf;
  uint32_t docs[QW_BLOCK_LEN], tfs[QW_BLOCK_LEN];
  float weight; const float* cache; const uint8_t* fieldnorms;
  uint64_t* visited;
  /* RANGE / EXISTS / ALL */
  const OImg* im; const QwImgColumn* col; uint64_t lo, hi; uint32_t max_doc;
  /* BOOL */
  DocSet** kids; uint32_t nkids; uint32_t n_req, n_should, n_not, required_should;
  int scoring;
  /* PHRASE (kids = its terms; a TERM kid of a phrase also carries its positions) */
  const uint32_t* positions; const uint32_t* first_pos; uint32_t pos_offset; uint32_t phrase_count;
};

static void term_load_block(DocSet* s) {
  const QwSkip* sk = &s->skips[s->blk];
  uint32_t deltas[QW_BLOCK_LEN];
  o_unpack_4x(s->tdata + sk->byte_off + 16u, sk->doc_bits, deltas);
  uint32_t prev = sk->prev_last_doc;
  for (uint32_t i = 0; i < sk->count; i++) { prev = prev + deltas[i] + 1; s->docs[i] = prev; }
  if (s->has_tf && s->scoring) o_unpack_4x(s->tdata + sk->byte_off + 16u + 16u * sk->doc_bits, sk->tf_bits, s->tfs);
  s->cnt = sk->count; s->pos = 0;
  if (s->visited) *s->visited += sk->count;
}
static uint32_t ds_advance(DocSet* s);
static uint32_t ds_seek(DocSet* s, uint32_t target);
static float ds_score(DocSet* s);

static uint32_t term_advance(DocSet* s) {
  if (s->doc == QW_TERMINATED) return s->doc;
  s->pos++;
  if (s->pos >= s->cnt) {
    s->blk++;
    if (s->blk >= s->nblocks) return s->doc = QW_TERMINATED;
    term_load_block(s);
  }
  return s->doc = s->docs[s->pos];
}
static uint32_t term_seek(DocSet* s, uint32_t target) {
  if (s->doc >= target) return s->doc;
  /* SkipReader::seek: skip whole blocks whose last_doc < target */
  if (s->skips[s->blk].last_doc < target) {
    uint32_t b = s->blk + 1;
    while (b < s->nblocks && s->skips[b].last_doc < target) b++;
    if (b >= s->nblocks) return s->doc = QW_TERMINATED;
    s->blk = b;
    term_load_block(s);
  }
  while (s->docs[s->pos] < target) s->pos++;
  return s->doc = s->docs[s->pos];
}
/* Bm25Weight::score (App. A.3): weight * tf / (tf + cache[fieldnorm_id]), f32 */
static float term_score(DocSet* s) {
  if (!s->scoring) return 0.0f;
  float tf = s->has_tf ? (float)s->tfs[s->pos] : 1.0f;
  uint32_t fid = s->fieldnorms ? s->fieldnorms[s->doc] : 0;
  float norm = s->cache[fid];
  return s->weight * (tf / (tf + norm));
}

/* PhraseScorer, slop 0 (tantivy phrase_scorer.rs; recalled, SURVEY.md Appendix A): intersection of the terms'
 * docsets, then of their position lists shifted by the terms' offsets; phrase_count = size of that intersection. */
static void term_positions(DocSet* t, const uint32_t** p, uint32_t* n) {
  uint32_t at = t->first_pos[t->blk];
  for (uint32_t i = 0; i < t->pos; i++) at += t->tfs[i];
  *p = t->positions + at;
  *n = t->tfs[t->pos];
}
static uint32_t phrase_count_here(DocSet* s) {
  uint32_t max_off = 0;
  for (uint32_t k = 0; k < s->nkids; k++) if (s->kids[k]->pos_offset > max_off) max_off = s->kids[k]->pos_offset;
  const uint32_t* p0; uint32_t n0;
  term_positions(s->kids[0], &p0, &n0);
  uint32_t count = 0;
  for (uint32_t i = 0; i < n0; i++) {
    const uint32_t shifted = p0[i] + (max_off - s->kids[0]->pos_offset);  /* = base + max_off */
    int all = 1;
    for (uint32_t k = 1; k < s->nkids && all; k++) {
      const uint32_t* pk; uint32_t nk;
      term_positions(s->kids[k], &pk, &nk);
      const uint32_t add = max_off - s->kids[k]->pos_offset;
      int found = 0;
      for (uint32_t j = 0; j < nk; j++) if (pk[j] + add == shifted) { found = 1; break; }
      all = found;
    }
    count += (uint32_t)all;
  }
  return count;
}
static uint32_t phrase_next(DocSet* s, uint32_t from) {
  uint32_t cand = from;
  for (;;) {
    if (cand >= QW_TERMINATED) return s->doc = QW_TERMINATED;
    uint32_t i = 0, agreed = 0;
    while (agreed < s->nkids) {
      uint32_t d = ds_seek(s->kids[i], cand);
      if (d == QW_TERMINATED) return s->doc = QW_TERMINATED;
      if (d > cand) { cand = d; agreed = 1; } else agreed++;
      i = (i + 1) % s->nkids;
    }
    s->phrase_count = phrase_count_here(s);
    if (s->phrase_count) return s->doc = cand;
    cand++;
  }
}
static float phrase_score(DocSet* s) {
  if (!s->scoring) return 0.0f;
  float tf = (float)s->phrase_count;
  uint32_t fid = s->fieldnorms ? s->fieldnorms[s->doc] : 0;
  return s->weight * (tf / (tf + s->cache[fid]));
}

static int range_match(DocSet* s, uint32_t d) {
  uint64_t a, b;
  o_col_range(s->im, s->col, d, &a, &b);
  for (uint64_t i = a; i < b; i++) {
    if (s->kind == QW_NODE_EXISTS) return 1;
    uint64_t m = o_col_mapped(s->im, s->col, i);
    if (m >= s->lo && m <= s->hi) return 1;
  }
  return 0;
}
static uint32_t scan_from(DocSet* s, uint32_t d) {
  for (; d < s->max_doc; d++) {
    if (s->kind == QW_NODE_ALL || range_match(s, d)) return s->doc = d;
  }
  return s->doc = QW_TERMINATED;
}

/* BooleanQuery semantics (tantivy BooleanWeight; lowering at
 * quickwit-query/src/query_ast/tantivy_query_ast.rs:345-377):
 * kids are ordered [required (must, filter) | should | must_not]. */
static int bool_check(DocSet* s, uint32_t cand) {
  for (uint32_t i = s->n_req + s->n_should; i < s->nkids; i++)
    if (ds_seek(s->kids[i], cand) == cand) return 0;
  if (s->n_req > 0) {
    if (s->required_should == 0) return 1;
    uint32_t c = 0;
    for (uint32_t i = s->n_req; i < s->n_req + s->n_should; i++)
      if (ds_seek(s->kids[i], cand) == cand) c++;
    return c >= s->required_should;
  }
  uint32_t c = 0;
  for (uint32_t i = 0; i < s->n_should; i++)
    if (s->kids[i]->doc == cand) c++;
  return c >= s->required_should;
}
static uint32_t bool_next(DocSet* s, uint32_t from) { /* first matching doc >= from */
  if (s->n_req == 0 && (s->n_should == 0 || s->required_should > s->n_should)) return s->doc = QW_TERMINATED;
  uint32_t cand = from;
  for (;;) {
    if (cand >= QW_TERMINATED) return s->doc = QW_TERMINATED;
    if (s->n_req > 0) {
      /* Intersection: leap-frog */
      uint32_t i = 0, agreed = 0;
      while (agreed < s->n_req) {
        uint32_t d = ds_seek(s->kids[i], cand);
        if (d == QW_TERMINATED) return s->doc = QW_TERMINATED;
        if (d > cand) { cand = d; agreed = 1; } else agreed++;
        i = (i + 1) % s->n_req;
      }
    } else {
      /* Union: smallest doc >= cand among should kids */
      uint32_t m = QW_TERMINATED;
      for (uint32_t i = 0; i < s->n_should; i++) {
        uint32_t d = ds_seek(s->kids[i], cand);
        if (d < m) m = d;
      }
      if (m == QW_TERMINATED) return s->doc = QW_TERMINATED;
      cand = m;
    }
    if (bool_check(s, cand)) return s->doc = cand;
    cand++;
  }
}
/* score = (Σ must scores, clause order) + (Σ matching should scores, clause order); filter = 0 */
static float bool_score(DocSet* s) {
  float must_sum = 0.0f, should_sum = 0.0f;
  for (uint32_t i = 0; i < s->n_req; i++)
    if (s->kids[i]->occur == QW_OCCUR_MUST) must_sum += ds_score(s->kids[i]);
  for (uint32_t i = s->n_req; i < s->n_req + s->n_should; i++)
    if (ds_seek(s->kids[i], s->doc) == s->doc) should_sum += ds_score(s->kids[i]);
  return must_sum + should_sum;
}

static uint32_t ds_advance(DocSet* s) {
  switch (s->kind) {
    case QW_NODE_TERM: return term_advance(s);
    case QW_NODE_NONE: return s->doc = QW_TERMINATED;
    case QW_NODE_BOOL: return s->doc == QW_TERMINATED ? s->doc : bool_next(s, s->doc + 1);
    case QW_NODE_PHRASE: return s->doc == QW_TERMINATED ? s->doc : phrase_next(s, s->doc + 1);
    default: return s->doc == QW_TERMINATED ? s->doc : scan_from(s, s->doc + 1);
  }
}
static uint32_t ds_seek(DocSet* s, uint32_t target) {
  if (s->doc >= target) return s->doc;
  switch (s->kind) {
    case QW_NODE_TERM: return term_seek(s, target);
    case QW_NODE_NONE: return s->doc = QW_TERMINATED;
    case QW_NODE_BOOL: return bool_next(s, target);
    case QW_NODE_PHRASE: return phrase_next(s, target);
    default: return scan_from(s, target);
  }
}
static float ds_score(DocSet* s) {
  switch (s->kind) {
    case QW_NODE_TERM: return term_score(s);
    case QW_NODE_BOOL: return bool_score(s);
    case QW_NODE_PHRASE: return phrase_score(s);
    case QW_NODE_NONE: return 0.0f;
    default: return s->scoring ? s->boost : 0.0f; /* ConstScorer(1.0 * boost) */
  }
}

typedef struct { DocSet** all; uint32_t n, cap; float** caches; uint32_t ncaches; } Arena;
static DocSet* arena_new(Arena* a) {
  if (a->n == a->cap) { a->cap = a->cap ? a->cap * 2 : 16; a->all = (DocSet**)realloc(a->all, a->cap * sizeof(DocSet*)); }
  DocSet* s = (DocSet*)calloc(1, sizeof(DocSet));
  a->all[a->n++] = s;
  return s;
}
static void arena_free(Arena* a) {
  for (uint32_t i = 0; i < a->n; i++) { free(a->all[i]->kids); free(a->all[i]); }
  for (uint32_t i = 0; i < a->ncaches; i++) free(a->caches[i]);
  free(a->all); free(a->caches);
}

/* Bm25Weight cache (App. A.3): cache[id] = K1 * (1 - B + B * fieldnorm(id) / average_fieldnorm) */
static float* bm25_cache(Arena* a, const OImg* im, const QwImgField* f) {
  float* c = (float*)malloc(256 * sizeof(float));
  a->caches = (float**)realloc(a->caches, (a->ncaches + 1) * sizeof(float*));
  a->caches[a->ncaches++] = c;
  float avg = (float)f->total_num_tokens / (float)im->hdr->num_docs;
  for (uint32_t id = 0; id < 256; id++)
    c[id] = 1.2f * (1.0f - 0.75f + 0.75f * (float)o_id_to_fieldnorm(id) / avg);
  return c;
}

static DocSet* build(Arena* a, const OImg* im, const QwPlanNode* nodes, uint32_t idx, int scoring, uint64_t* visited) {
  const QwPlanNode* n = &nodes[idx];
  DocSet* s = arena_new(a);
  s->kind = (int)n->kind; s->boost = n->boost; s->occur = n->occur; s->scoring = scoring;
  s->im = im; s->max_doc = im->hdr->num_docs; s->visited = visited;
  switch (n->kind) {
    case QW_NODE_TERM: {
      if (n->term_ord == 0xFFFFFFFFu) { s->kind = QW_NODE_NONE; s->doc = QW_TERMINATED; break; }
      const QwImgTerm* t = &im->terms[n->term_ord];
      const QwImgField* f = &im->fields[t->field_id];
      s->skips = (const QwSkip*)(im->data + t->skip_off);
      s->tdata = im->data + t->data_off;
      s->nblocks = t->num_blocks;
      s->has_tf = (f->flags & QW_FIELD_HAS_FREQS) != 0;
      /* Bm25Weight::for_one_term + boost_by (tantivy, SURVEY.md Appendix A.3 / B.1), computed HERE from the
       * split's own statistics, not read from the plan: idf = ln(1 + (N - n + 0.5) / (n + 0.5)), weight =
       * idf * (1 + K1) * boost, all f32. (The plan's bm25_weight field is the product's; a mismatch shows
       * up as a score difference in every parity test.) */
      {
        float nn = (float)t->doc_freq, N = (float)im->hdr->num_docs;
        float idf = logf(1.0f + ((N - nn) + 0.5f) / (nn + 0.5f));
        s->weight = idf * (1.0f + 1.2f) * n->boost;
      }
      s->fieldnorms = (f->flags & QW_FIELD_HAS_FIELDNORMS) ? im->data + f->fieldnorm_off : NULL;
      s->cache = bm25_cache(a, im, f);
      if (!s->fieldnorms) {
        /* fieldnorms: false => constant fieldnorm 1 for every doc (tantivy FieldNormReader::constant) */
        float avg = (float)f->total_num_tokens / (float)im->hdr->num_docs;
        ((float*)s->cache)[0] = 1.2f * (1.0f - 0.75f + 0.75f * 1.0f / avg);
      }
      s->blk = 0; term_load_block(s); s->doc = s->docs[0];
      break;
    }
    case QW_NODE_RANGE: case QW_NODE_EXISTS:
      if (n->column == 0xFFFFFFFFu) { s->kind = QW_NODE_NONE; s->doc = QW_TERMINATED; break; }
      s->col = &im->cols[n->column]; s->lo = n->lo; s->hi = n->hi;
      scan_from(s, 0);
      break;
    case QW_NODE_ALL: scan_from(s, 0); break;
    case QW_NODE_NONE: s->doc = QW_TERMINATED; break;
    case QW_NODE_BOOL: {
      s->nkids = n->num_children;
      s->kids = (DocSet**)calloc(n->num_children ? n->num_children : 1, sizeof(DocSet*));
      uint32_t k = 0;
      for (int pass = 0; pass < 3; pass++)
        for (uint32_t c = 0; c < n->num_children; c++) {
          const QwPlanNode* cn = &nodes[n->first_child + c];
          int grp = (cn->occur == QW_OCCUR_MUST || cn->occur == QW_OCCUR_FILTER) ? 0 : (cn->occur == QW_OCCUR_SHOULD ? 1 : 2);
          if (grp != pass) continue;
          int child_scoring = scoring && (cn->occur == QW_OCCUR_MUST || cn->occur == QW_OCCUR_SHOULD);
          s->kids[k++] = build(a, im, nodes, n->first_child + c, child_scoring, visited);
          if (pass == 0) s->n_req++; else if (pass == 1) s->n_should++; else s->n_not++;
        }
      uint32_t msm = n->min_should_match == 0xFFFFFFFFu ? 0 : n->min_should_match;
      s->required_should = msm > 0 ? msm : (s->n_req == 0 ? 1 : 0);
      bool_next(s, 0);
      break;
    }
    case QW_NODE_PHRASE: {
      /* PhraseWeight: any term missing from the split -> no scorer; Bm25Weight::for_terms = summed idf */
      int ok = n->num_children >= 2;
      for (uint32_t c = 0; c < n->num_children && ok; c++) {
        const QwPlanNode* cn = &nodes[n->first_child + c];
        if (cn->kind != QW_NODE_TERM || cn->term_ord == 0xFFFFFFFFu || im->terms[cn->term_ord].pidx_off == 0) ok = 0;
      }
      if (!ok) { s->kind = QW_NODE_NONE; s->doc = QW_TERMINATED; break; }
      s->nkids = n->num_children;
      s->kids = (DocSet**)calloc(n->num_children, sizeof(DocSet*));
      float idf_sum = 0.0f;
      const QwImgField* f = NULL;
      for (uint32_t c = 0; c < n->num_children; c++) {
        const QwPlanNode* cn = &nodes[n->first_child + c];
        const QwImgTerm* t = &im->terms[cn->term_ord];
        DocSet* k = build(a, im, nodes, n->first_child + c, /*scoring: the tfs locate the positions*/ 1, visited);
        k->positions = (const uint32_t*)(im->data + t->pos_off);
        k->first_pos = (const uint32_t*)(im->data + t->pidx_off);
        k->pos_offset = (uint32_t)cn->lo;
        s->kids[c] = k;
        f = &im->fields[t->field_id];
        float nn = (float)t->doc_freq, N = (float)im->hdr->num_docs;
        idf_sum += logf(1.0f + ((N - nn) + 0.5f) / (nn + 0.5f));
      }
      s->weight = idf_sum * (1.0f + 1.2f) * n->boost;
      s->fieldnorms = (f->flags & QW_FIELD_HAS_FIELDNORMS) ? im->data + f->fieldnorm_off : NULL;
      s->cache = bm25_cache(a, im, f);
      if (!s->fieldnorms) {
        float avg = (float)f->total_num_tokens / (float)im->hdr->num_docs;
        ((float*)s->cache)[0] = 1.2f * (1.0f - 0.75f + 0.75f * 1.0f / avg);
      }
      phrase_next(s, 0);
      break;
    }
    default: s->kind = QW_NODE_NONE; s->doc = QW_TERMINATED;
  }
  return s;
}

/* ------------------------------------------------------------------ top-K collectors --------- */
typedef struct { uint64_t v1, v2; uint32_t doc, flags; float score; } OHit;

/* SortOrder::compare_opt / compare (quickwit-proto/src/lib.rs:122-140): Some > None always;
 * Desc = natural order, Asc = reversed. Returns -1/0/1. */
static int cmp_u64(uint64_t a, uint64_t b) { return a < b ? -1 : (a > b ? 1 : 0); }
static int order_cmp(uint32_t order, uint64_t a, uint64_t b) { return order == QW_ORDER_DESC ? cmp_u64(a, b) : cmp_u64(b, a); }
static int order_cmp_opt(uint32_t order, int ha, uint64_t a, int hb, uint64_t b) {
  if (ha && hb) return order_cmp(order, a, b);
  if (ha) return 1;
  if (hb) return -1;
  return 0;
}
/* SegmentPartialHitSortingKey::cmp (quickwit-search/src/collector.rs:1082-1112) ==
 * Hit<V1,V2,REVERSE_DOCID>::cmp (top_k_collector.rs:137-158): greater = better. */
typedef struct { uint32_t order1, order2; } Orders;
static int hit_cmp(const Orders* o, const OHit* a, const OHit* b) {
  int c = order_cmp_opt(o->order1, a->flags & 1, a->v1, b->flags & 1, b->v1);
  if (c) return c;
  c = order_cmp_opt(o->order2, (a->flags >> 1) & 1, a->v2, (b->flags >> 1) & 1, b->v2);
  if (c) return c;
  return order_cmp(o->order1, a->doc, b->doc);
}

/* quickwit_common::binary_heap::TopK (quickwit-common/src/binary_heap.rs:125-194): min-heap of
 * K; once full, replace the head iff head.order < order (strict). */
typedef struct { OHit* h; uint32_t n, k; Orders o; } Heap;
static void heap_sift_down(Heap* hp, uint32_t i) {
  for (;;) {
    uint32_t l = 2 * i + 1, r = l + 1, m = i;
    if (l < hp->n && hit_cmp(&hp->o, &hp->h[l], &hp->h[m]) < 0) m = l;
    if (r < hp->n && hit_cmp(&hp->o, &hp->h[r], &hp->h[m]) < 0) m = r;
    if (m == i) return;
    OHit t = hp->h[i]; hp->h[i] = hp->h[m]; hp->h[m] = t; i = m;
  }
}
static void heap_add(Heap* hp, const OHit* x) {
  if (hp->k == 0) return;
  if (hp->n < hp->k) {
    uint32_t i = hp->n++;
    hp->h[i] = *x;
    while (i > 0) {
      uint32_t p = (i - 1) / 2;
      if (hit_cmp(&hp->o, &hp->h[i], &hp->h[p]) < 0) { OHit t = hp->h[i]; hp->h[i] = hp->h[p]; hp->h[p] = t; i = p; } else break;
    }
    return;
  }
  if (hit_cmp(&hp->o, &hp->h[0], x) < 0) { hp->h[0] = *x; heap_sift_down(hp, 0); }
}

static __thread const Orders* t_orders;
static int qsort_desc(const void* a, const void* b) { return hit_cmp(t_orders, (const OHit*)b, (const OHit*)a); }

/* TopKComputer (quickwit-search/src/top_k_collector.rs:331-422): buffer of capacity 10*K;
 * reject below threshold; when full, keep the top K and set threshold to the K-th. */
typedef struct { OHit* buf; uint32_t n, cap, k; OHit thr; int has_thr; Orders o; } TopKC;
static OHit topkc_truncate(TopKC* t) {
  t_orders = &t->o;
  qsort(t->buf, t->n, sizeof(OHit), qsort_desc); /* select_nth_unstable(top_n) + truncate */
  OHit median = t->buf[t->k]; /* element at index top_n in descending order */
  t->n = t->k;
  return median;
}
static void topkc_push(TopKC* t, const OHit* x) {
  if (t->has_thr && hit_cmp(&t->o, x, &t->thr) < 0) return;
  if (t->n == t->cap) { t->thr = topkc_truncate(t); t->has_thr = 1; }
  t->buf[t->n++] = *x;
}

/* ------------------------------------------------------------------ aggregations ------------- */
/* Dense-cell restatement of tantivy's segment aggregation collectors for the shapes the plan
 * supports (terms / histogram / date_histogram / range buckets, stats-family metrics; semantics
 * per docs/reference/aggregation.md:140-560 and SURVEY.md Appendix A.6). */
typedef struct { const QwAggNode* nodes; uint32_t n; uint64_t* cell_off; QwAggCell* cells; const OImg* im; uint64_t geometry_errors; } Aggs;

static void agg_collect(Aggs* A, uint32_t ni, uint32_t doc, uint64_t parent_cell) {
  const QwAggNode* g = &A->nodes[ni];
  QwAggCell* base = A->cells + A->cell_off[ni];
  if (g->column == 0xFFFFFFFFu) {
    if (g->kind == QW_AGG_TERMS && g->has_missing) {
      uint64_t cell = parent_cell * g->num_buckets + (g->num_buckets - 1);
      base[cell].count++;
      for (uint32_t c = 0; c < g->num_children; c++) agg_collect(A, g->first_child + c, doc, cell);
    }
    return;
  }
  const QwImgColumn* col = &A->im->cols[g->column];
  uint64_t a, b;
  o_col_range(A->im, col, doc, &a, &b);
  if (g->kind == QW_AGG_STATS) {
    QwAggCell* c = &base[parent_cell];
    for (uint64_t i = a; i < b; i++) {
      uint64_t m = o_col_mapped(A->im, col, i);
      c->count++;
      if (!qw_col_sum_exact(col)) {
        /* tantivy: sum += value as f64, in doc order */
        double s; memcpy(&s, &c->sum_bits, 8); s += o_mapped_to_f64(col->type, m); memcpy(&c->sum_bits, &s, 8);
      } else {
        /* integer-typed columns: exact integer sum of the raw offsets (QwAggCell contract: the host
         * rebuilds count * min + gcd * sum in 128 bits; no overflow for nanosecond timestamps) */
        c->sum_bits += o_col_raw(A->im, col, i);
      }
      if (m < c->min_mapped) c->min_mapped = m;
      if (m > c->max_mapped) c->max_mapped = m;
    }
    return;
  }
  if (a == b && g->kind == QW_AGG_TERMS && g->has_missing) {
    uint64_t cell = parent_cell * g->num_buckets + (g->num_buckets - 1);
    base[cell].count++;
    for (uint32_t c = 0; c < g->num_children; c++) agg_collect(A, g->first_child + c, doc, cell);
    return;
  }
  for (uint64_t i = a; i < b; i++) {
    uint64_t raw = o_col_raw(A->im, col, i);
    uint64_t m = col->min_value + col->gcd * raw;
    if (g->kind == QW_AGG_TERMS) {
      if (raw >= g->num_buckets - (g->has_missing ? 1u : 0u)) { A->geometry_errors++; continue; }
      uint64_t cell = parent_cell * g->num_buckets + raw;
      base[cell].count++;
      for (uint32_t c = 0; c < g->num_children; c++) agg_collect(A, g->first_child + c, doc, cell);
    } else if (g->kind == QW_AGG_HISTOGRAM) {
      double val = o_mapped_to_f64(col->type, m);
      if (g->has_bounds && !(val >= g->bound_min && val <= g->bound_max)) continue;
      double pos = floor((val - g->offset) / g->interval);
      int64_t idx = (int64_t)pos - g->base_pos;
      /* the dense bucket range [base_pos, base_pos + num_buckets) is the product's cell LAYOUT; a value
       * inside the hard bounds that falls outside it means the layout is wrong: reported as an error */
      if (idx < 0 || idx >= (int64_t)g->num_buckets) { A->geometry_errors++; continue; }
      uint64_t cell = parent_cell * g->num_buckets + (uint64_t)idx;
      base[cell].count++;
      for (uint32_t c = 0; c < g->num_children; c++) agg_collect(A, g->first_child + c, doc, cell);
    } else if (g->kind == QW_AGG_RANGE) {
      for (uint32_t r = 0; r < g->num_ranges; r++) {
        if (m >= g->range_from[r] && m < g->range_to[r]) {
          uint64_t cell = parent_cell * g->num_buckets + r;
          base[cell].count++;
          for (uint32_t c = 0; c < g->num_children; c++) agg_collect(A, g->first_child + c, doc, cell);
        }
      }
    }
  }
}

uint64_t qwo_agg_num_cells(const QwAggNode* nodes, uint32_t n, uint64_t* cell_off) {
  uint64_t total = 0;
  for (uint32_t i = 0; i < n; i++) {
    uint64_t cells = nodes[i].kind == QW_AGG_STATS ? 1 : nodes[i].num_buckets;
    uint32_t p = nodes[i].parent;
    while (p != 0xFFFFFFFFu) { cells *= nodes[p].num_buckets; p = nodes[p].parent; }
    if (cell_off) cell_off[i] = total;
    total += cells;
  }
  return total;
}

/* ------------------------------------------------------------------ entry point -------------- */
/* Restates searcher.search(&query, &collector) for one split (quickwit-search/src/leaf.rs:637):
 * weight.for_each / for_each_no_score feeding QuickwitSegmentCollector::{collect,collect_block}
 * (collector.rs:523-562), then harvest (collector.rs:564-594). Returns 0 or a negative error. */
int qwo_split_search(const uint8_t* img, uint64_t img_len, const uint8_t* plan, uint64_t plan_len,
                     QwHit* hits_out, uint32_t* n_hits_out, uint64_t* num_hits_out,
                     QwAggCell* cells_out, uint64_t cells_cap, uint64_t* postings_visited) {
  OImg im;
  if (oimg_open(&im, img, img_len)) return -1;
  if (plan_len < sizeof(QwPlanHeader)) return -2;
  const QwPlanHeader* ph = (const QwPlanHeader*)plan;
  if (ph->magic != QW_PLAN_MAGIC) return -2;
  const QwPlanNode* nodes = (const QwPlanNode*)(plan + sizeof(QwPlanHeader));
  const QwAggNode* aggs = (const QwAggNode*)(plan + sizeof(QwPlanHeader) + (uint64_t)ph->num_nodes * sizeof(QwPlanNode));
  uint64_t visited = 0;
  Arena arena; memset(&arena, 0, sizeof arena);
  DocSet* root = build(&arena, &im, nodes, 0, (int)ph->scoring, &visited);

  Orders ord = { ph->sort[0].order, ph->sort[1].kind == QW_SORT_NONE ? QW_ORDER_DESC : ph->sort[1].order };
  uint32_t K = ph->max_hits;
  /* specialized_top_k_segment_collector dispatch (top_k_collector.rs:190-206) */
  int generic = ph->search_after.present || ph->scoring;
  Heap heap; memset(&heap, 0, sizeof heap);
  TopKC tk; memset(&tk, 0, sizeof tk);
  if (K > 0) {
    if (generic) { heap.h = (OHit*)malloc((size_t)K * sizeof(OHit)); heap.k = K; heap.o = ord; }
    else { tk.k = K; tk.cap = (K > 1 ? K : 1) * 10; tk.buf = (OHit*)malloc((size_t)tk.cap * sizeof(OHit)); tk.o = ord; }
  }
  Aggs A; memset(&A, 0, sizeof A);
  uint64_t ncells = 0;
  if (ph->num_aggs) {
    A.nodes = aggs; A.n = ph->num_aggs; A.im = &im;
    A.cell_off = (uint64_t*)malloc(ph->num_aggs * sizeof(uint64_t));
    ncells = qwo_agg_num_cells(aggs, ph->num_aggs, A.cell_off);
    if (ncells > cells_cap) { free(A.cell_off); arena_free(&arena); free(heap.h); free(tk.buf); return -3; }
    A.cells = cells_out;
    for (uint64_t i = 0; i < ncells; i++) { cells_out[i].count = 0; cells_out[i].sum_bits = 0; cells_out[i].min_mapped = ~0ull; cells_out[i].max_mapped = 0; }
  }
  const QwImgColumn* c1 = (ph->sort[0].kind == QW_SORT_COLUMN && ph->sort[0].column != 0xFFFFFFFFu) ? &im.cols[ph->sort[0].column] : NULL;
  const QwImgColumn* c2 = (ph->sort[1].kind == QW_SORT_COLUMN && ph->sort[1].column != 0xFFFFFFFFu) ? &im.cols[ph->sort[1].column] : NULL;
  const QwSearchAfter* sa = &ph->search_after;
  uint64_t num_hits = 0;
  for (uint32_t doc = root->doc; doc != QW_TERMINATED; doc = ds_advance(root)) {
    num_hits++;
    if (K > 0) {
      OHit h; memset(&h, 0, sizeof h);
      h.doc = doc;
      /* SortingFieldExtractorComponent::extract_typed_sort_value_opt (collector.rs:171-182) */
      if (ph->sort[0].kind == QW_SORT_SCORE) { h.score = ds_score(root); h.v1 = o_f64_to_u64((double)h.score); h.flags |= 1; }
      else if (c1) { if (o_col_first(&im, c1, doc, &h.v1)) h.flags |= 1; }
      if (ph->sort[1].kind == QW_SORT_SCORE) { h.score = ds_score(root); h.v2 = o_f64_to_u64((double)h.score); h.flags |= 2; }
      else if (c2) { if (o_col_first(&im, c2, doc, &h.v2)) h.flags |= 2; }
      if (generic) {
        int keep = 1;
        if (sa->present) { /* collect_top_k_vals (top_k_collector.rs:663-699) */
          int c = order_cmp_opt(ord.order1, h.flags & 1, h.v1, (int)sa->has_v1, sa->v1);
          if (!c) c = order_cmp_opt(ord.order2, (h.flags >> 1) & 1, h.v2, (int)sa->has_v2, sa->v2);
          if (sa->compare_on_equal) {
            if (!c) c = sa->precomp_order;
            if (!c) c = order_cmp(ord.order1, doc, sa->doc_id);
          }
          if (c >= 0) keep = 0;
        }
        if (keep) heap_add(&heap, &h);
      } else {
        topkc_push(&tk, &h);
      }
    }
    for (uint32_t a = 0; a < ph->num_aggs; a++)
      if (aggs[a].parent == 0xFFFFFFFFu) agg_collect(&A, a, doc, 0);
  }
  /* harvest: sorted best-first (binary_heap.rs:187-193; top_k_collector.rs:404-410) */
  uint32_t n = 0;
  if (K > 0) {
    OHit* src; uint32_t cnt;
    if (generic) { src = heap.h; cnt = heap.n; }
    else { if (tk.n > tk.k) topkc_truncate(&tk); src = tk.buf; cnt = tk.n; }
    t_orders = &ord;
    qsort(src, cnt, sizeof(OHit), qsort_desc);
    for (uint32_t i = 0; i < cnt; i++) {
      hits_out[i].v1 = src[i].v1; hits_out[i].v2 = src[i].v2; hits_out[i].doc_id = src[i].doc;
      hits_out[i].flags = src[i].flags; hits_out[i].score = src[i].score; hits_out[i].reserved = 0;
    }
    n = cnt;
  }
  *n_hits_out = n;
  *num_hits_out = num_hits;
  if (postings_visited) *postings_visited = visited;
  free(heap.h); free(tk.buf); free(A.cell_off);
  arena_free(&arena);
  return A.geometry_errors ? -4 : 0;  /* -4: a value fell outside the plan's dense bucket layout */
}

/* ------------------------------------------------------------------ CPU baseline fast path ---- */
/* What bench.py times as the reference's CPU algorithm for the BM25-union shape: the same arithmetic
 * as qwo_split_search, organised the way tantivy runs it — BitPacker4x blocks unpacked four lanes at a
 * time (SSE2 through GCC vector types) and a BufferedUnionScorer-style 4096-doc horizon (bitset + f32
 * accumulator, scorers folded in clause order, matches swept in doc order) feeding the binary-heap TopK —
 * instead of the doc-at-a-time min-scan above. tests/test_oracle_goldens.py checks that both paths
 * return identical hits, scores and counts. Plans that are not a pure OR of scored terms ranked by
 * _score (no search_after, no aggregations) fall back to qwo_split_search. */
typedef uint32_t v4u __attribute__((vector_size(16)));
static void o_unpack_4x_simd(const uint8_t* p, uint32_t bits, uint32_t* out) {
  if (bits == 0) { memset(out, 0, 4 * QW_BLOCK_LEN); return; }
  const uint32_t m = bits == 32 ? 0xFFFFFFFFu : ((1u << bits) - 1u);
  const v4u mask = {m, m, m, m};
  for (uint32_t k = 0; k < 32; k++) {
    const uint32_t bitpos = k * bits, wi = bitpos >> 5, sh = bitpos & 31;
    v4u lo, hi;
    memcpy(&lo, p + 16u * wi, 16);
    v4u v = lo >> sh;
    if (sh + bits > 32) { memcpy(&hi, p + 16u * (wi + 1), 16); v |= hi << (32 - sh); }
    v &= mask;
    memcpy(out + 4 * k, &v, 16);
  }
}
typedef struct {
  const QwSkip* skips; const uint8_t* tdata; const uint8_t* fieldnorms;
  uint32_t nblocks, blk, pos, cnt, has_tf, doc;
  float weight, cache[256];
  uint32_t docs[QW_BLOCK_LEN], tfs[QW_BLOCK_LEN];
} FTerm;
static void fterm_load(FTerm* t, uint64_t* visited) {
  const QwSkip* sk = &t->skips[t->blk];
  uint32_t deltas[QW_BLOCK_LEN];
  o_unpack_4x_simd(t->tdata + sk->byte_off + 16u, sk->doc_bits, deltas);
  uint32_t prev = sk->prev_last_doc;
  for (uint32_t i = 0; i < sk->count; i++) { prev = prev + deltas[i] + 1; t->docs[i] = prev; }
  if (t->has_tf) o_unpack_4x_simd(t->tdata + sk->byte_off + 16u + 16u * sk->doc_bits, sk->tf_bits, t->tfs);
  t->cnt = sk->count; t->pos = 0; t->doc = t->docs[0];
  *visited += sk->count;
}
#define QWO_HORIZON 4096u /* tantivy BufferedUnionScorer: 64 words of 64 docs */
static int fast_union_eligible(const QwPlanHeader* ph, const QwPlanNode* nodes) {
  if (!ph->scoring || ph->max_hits == 0 || ph->num_aggs || ph->search_after.present) return 0;
  if (ph->sort[0].kind != QW_SORT_SCORE || ph->sort[0].order != QW_ORDER_DESC || ph->sort[1].kind != QW_SORT_NONE) return 0;
  if (nodes[0].kind != QW_NODE_BOOL || nodes[0].num_children == 0 || nodes[0].num_children > 64) return 0;
  if (nodes[0].min_should_match != 0xFFFFFFFFu && nodes[0].min_should_match > 1) return 0;
  for (uint32_t c = 0; c < nodes[0].num_children; c++) {
    const QwPlanNode* n = &nodes[nodes[0].first_child + c];
    if (n->kind != QW_NODE_TERM || n->occur != QW_OCCUR_SHOULD) return 0;
  }
  return 1;
}
int qwo_split_search_fast(const uint8_t* img, uint64_t img_len, const uint8_t* plan, uint64_t plan_len,
                          QwHit* hits_out, uint32_t* n_hits_out, uint64_t* num_hits_out,
                          QwAggCell* cells_out, uint64_t cells_cap, uint64_t* postings_visited) {
  OImg im;
  if (oimg_open(&im, img, img_len)) return -1;
  if (plan_len < sizeof(QwPlanHeader)) return -2;
  const QwPlanHeader* ph = (const QwPlanHeader*)plan;
  if (ph->magic != QW_PLAN_MAGIC) return -2;
  const QwPlanNode* nodes = (const QwPlanNode*)(plan + sizeof(QwPlanHeader));
  if (!fast_union_eligible(ph, nodes))
    return qwo_split_search(img, img_len, plan, plan_len, hits_out, n_hits_out, num_hits_out, cells_out, cells_cap, postings_visited);
  const uint32_t nt = nodes[0].num_children, N = im.hdr->num_docs, K = ph->max_hits;
  FTerm* T = (FTerm*)calloc(nt, sizeof(FTerm));
  uint64_t visited = 0;
  uint32_t live = 0;
  for (uint32_t c = 0; c < nt; c++) {
    const QwPlanNode* n = &nodes[nodes[0].first_child + c];
    FTerm* t = &T[c];
    t->doc = QW_TERMINATED;
    if (n->term_ord == 0xFFFFFFFFu) continue;
    const QwImgTerm* it = &im.terms[n->term_ord];
    const QwImgField* f = &im.fields[it->field_id];
    t->skips = (const QwSkip*)(im.data + it->skip_off);
    t->tdata = im.data + it->data_off;
    t->nblocks = it->num_blocks;
    t->has_tf = (f->flags & QW_FIELD_HAS_FREQS) != 0;
    t->fieldnorms = (f->flags & QW_FIELD_HAS_FIELDNORMS) ? im.data + f->fieldnorm_off : NULL;
    float nn = (float)it->doc_freq, Nf = (float)N;
    t->weight = logf(1.0f + ((Nf - nn) + 0.5f) / (nn + 0.5f)) * (1.0f + 1.2f) * n->boost;
    float avg = (float)f->total_num_tokens / (float)N;
    for (uint32_t id = 0; id < 256; id++) t->cache[id] = 1.2f * (1.0f - 0.75f + 0.75f * (float)o_id_to_fieldnorm(id) / avg);
    if (!t->fieldnorms) t->cache[0] = 1.2f * (1.0f - 0.75f + 0.75f * 1.0f / avg);
    if (t->nblocks) { fterm_load(t, &visited); live++; }
  }
  Heap heap; memset(&heap, 0, sizeof heap);
  heap.h = (OHit*)malloc((size_t)K * sizeof(OHit)); heap.k = K;
  Orders ord = { QW_ORDER_DESC, QW_ORDER_DESC };
  heap.o = ord;
  float* acc = (float*)calloc(QWO_HORIZON, sizeof(float));
  uint64_t bits[QWO_HORIZON / 64];
  uint64_t num_hits = 0;
  while (live) {
    uint32_t base = QW_TERMINATED;
    for (uint32_t c = 0; c < nt; c++) if (T[c].doc < base) base = T[c].doc;
    if (base == QW_TERMINATED) break;
    memset(bits, 0, sizeof bits);
    const uint32_t end = base + QWO_HORIZON;  /* (docs < 2^31: no wrap) */
    for (uint32_t c = 0; c < nt; c++) {  /* clause order = the order of the f32 sums */
      FTerm* t = &T[c];
      while (t->doc < end) {
        const uint32_t i = t->doc - base;
        const float tf = t->has_tf ? (float)t->tfs[t->pos] : 1.0f;
        const float norm = t->cache[t->fieldnorms ? t->fieldnorms[t->doc] : 0];
        acc[i] += t->weight * (tf / (tf + norm));
        bits[i >> 6] |= 1ull << (i & 63);
        if (++t->pos >= t->cnt) {
          if (++t->blk >= t->nblocks) { t->doc = QW_TERMINATED; live--; break; }
          fterm_load(t, &visited);
        } else t->doc = t->docs[t->pos];
      }
    }
    for (uint32_t w = 0; w < QWO_HORIZON / 64; w++) {
      uint64_t m = bits[w];
      while (m) {
        const uint32_t i = 64 * w + (uint32_t)__builtin_ctzll(m);
        m &= m - 1;
        OHit h; memset(&h, 0, sizeof h);
        h.doc = base + i; h.score = acc[i]; h.v1 = o_f64_to_u64((double)h.score); h.flags = 1;
        acc[i] = 0.0f;
        num_hits++;
        heap_add(&heap, &h);
      }
    }
  }
  t_orders = &ord;
  qsort(heap.h, heap.n, sizeof(OHit), qsort_desc);
  for (uint32_t i = 0; i < heap.n; i++) {
    hits_out[i].v1 = heap.h[i].v1; hits_out[i].v2 = 0; hits_out[i].doc_id = heap.h[i].doc;
    hits_out[i].flags = heap.h[i].flags; hits_out[i].score = heap.h[i].score; hits_out[i].reserved = 0;
  }
  *n_hits_out = heap.n;
  *num_hits_out = num_hits;
  if (postings_visited) *postings_visited = visited;
  free(heap.h); free(acc); free(T);
  return 0;
}

/* The same search over many (split, plan) pairs from a pool of C threads (one pair at a time per thread):
 * the CPU reference arm of bench.py. Returns 0, or the first error; sums in totals[0..1] = hits, postings. */
#include <pthread.h>
typedef struct {
  const uint8_t* const* imgs; const uint64_t* img_lens; const uint8_t* const* plans; const uint64_t* plan_lens;
  uint32_t n, next, fast; int err; uint64_t hits, postings; pthread_mutex_t mu;
} ManyCtx;
static void* many_worker(void* arg) {
  ManyCtx* c = (ManyCtx*)arg;
  QwHit* hits = NULL; uint32_t cap = 0;
  for (;;) {
    pthread_mutex_lock(&c->mu);
    uint32_t i = c->next < c->n ? c->next++ : 0xFFFFFFFFu;
    pthread_mutex_unlock(&c->mu);
    if (i == 0xFFFFFFFFu) break;
    const QwPlanHeader* ph = (const QwPlanHeader*)c->plans[i];
    uint32_t k = ph->max_hits ? ph->max_hits : 1;
    if (k > cap) { free(hits); hits = (QwHit*)malloc((size_t)k * sizeof(QwHit)); cap = k; }
    uint32_t nh = 0; uint64_t total = 0, vis = 0;
    QwAggCell dummy;
    int rc = (c->fast ? qwo_split_search_fast : qwo_split_search)(c->imgs[i], c->img_lens[i], c->plans[i], c->plan_lens[i], hits, &nh, &total, &dummy, 0, &vis);
    pthread_mutex_lock(&c->mu);
    if (rc && !c->err) c->err = rc;
    c->hits += total; c->postings += vis;
    pthread_mutex_unlock(&c->mu);
  }
  free(hits);
  return NULL;
}
int qwo_search_many(const uint8_t* const* imgs, const uint64_t* img_lens, const uint8_t* const* plans, const uint64_t* plan_lens,
                    uint32_t n, uint32_t threads, uint32_t fast, uint64_t* totals) {
  ManyCtx c; memset(&c, 0, sizeof c);
  c.imgs = imgs; c.img_lens = img_lens; c.plans = plans; c.plan_lens = plan_lens; c.n = n; c.fast = fast;
  pthread_mutex_init(&c.mu, NULL);
  if (threads == 0) threads = 1;
  if (threads > 256) threads = 256;
  pthread_t th[256];
  for (uint32_t t = 0; t < threads; t++) pthread_create(&th[t], NULL, many_worker, &c);
  for (uint32_t t = 0; t < threads; t++) pthread_join(th[t], NULL);
  pthread_mutex_destroy(&c.mu);
  if (totals) { totals[0] = c.hits; totals[1] = c.postings; }
  return c.err;
}

/* Posting-list decode only (for format round-trip tests): writes up to cap (doc, tf) pairs. */
int qwo_decode_postings(const uint8_t* img, uint64_t img_len, uint32_t term_ord, uint32_t* docs, uint32_t* tfs, uint32_t cap) {
  OImg im;
  if (oimg_open(&im, img, img_len) || term_ord >= im.hdr->num_terms) return -1;
  const QwImgTerm* t = &im.terms[term_ord];
  const QwSkip* sk = (const QwSkip*)(im.data + t->skip_off);
  uint32_t n = 0, d[QW_BLOCK_LEN], f[QW_BLOCK_LEN];
  for (uint32_t b = 0; b < t->num_blocks; b++) {
    o_unpack_4x(im.data + t->data_off + sk[b].byte_off + 16u, sk[b].doc_bits, d);
    o_unpack_4x(im.data + t->data_off + sk[b].byte_off + 16u + 16u * sk[b].doc_bits, sk[b].tf_bits, f);
    uint32_t prev = sk[b].prev_last_doc;
    for (uint32_t i = 0; i < sk[b].count && n < cap; i++, n++) { prev = prev + d[i] + 1; docs[n] = prev; tfs[n] = sk[b].tf_bits ? f[i] : 1; }
  }
  return (int)n;
}

/* Column read (for format round-trip tests): Column::first for every doc. */
int qwo_column_first(const uint8_t* img, uint64_t img_len, uint32_t col, uint64_t* vals, uint8_t* present) {
  OImg im;
  if (oimg_open(&im, img, img_len) || col >= im.hdr->num_columns) return -1;
  for (uint32_t d = 0; d < im.hdr->num_docs; d++) { uint64_t v = 0; present[d] = (uint8_t)o_col_first(&im, &im.cols[col], d, &v); vals[d] = v; }
  return 0;
}
