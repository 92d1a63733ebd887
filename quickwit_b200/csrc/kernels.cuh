// kernels.cuh — sm_100a kernels of the per-split leaf search hot path.
//
// Execution model ("window engine"): a 512-thread block owns one doc-id WINDOW (16384 docs when shared
// memory allows; 32768 for unscored plans) of one split and evaluates the whole boolean query over it
// in shared memory; the grid is persistent (2 blocks per SM) and walks a static partition of the flat
// (split, window) list of the request, so one launch covers every split:
//   1. one load per query term fetches the window-index entry (QwWinIdx) = the exact byte range and
//      block ordinals of the posting blocks overlapping the window; fieldnorm bytes of the window are
//      staged with 16-byte cp.async copies at the same time;
//   2. the packed posting bytes of ALL terms are staged with cp.async (16-byte, coalesced) while the
//      same load round turns the terms' skip-list entries into the window's block table;
//   3. terms are decoded block-per-warp (4-lane-interleaved bit-unpack -> warp-shuffle prefix scan ->
//      doc ids), BM25 is applied in f32 and accumulated into per-window score arrays in the
//      reference's clause order (bit-reproducible sums) — with a barrier per clause in the generic
//      program, with a ticket counter and no barrier in the BM25-union instantiation (UNION) — and
//      match sets are shared-memory bitmaps combined with AND / OR / AND-NOT exactly like tantivy's
//      BooleanWeight;
//   4. the matched docs of the window are counted, aggregated (bucket counts privatised in shared
//      memory) and filtered against a per-split top-K threshold over compacted hits (full warps);
//      survivors go to a candidate list that k_select reduces with the reference's total order.
// This replaces tantivy's doc-at-a-time Scorer/Collector loop (SURVEY.md §3.3 step 10c, §8a rows
// a3-a12). No tensor cores: the work is integer decode / compare plus one f32 multiply-add per
// posting; the binding resource measured on B200 is instruction issue, well before HBM bandwidth
// (DESIGN.md §5, profiles/r1_summary.md).
#pragma once
#include <cuda_runtime.h>

#include "device_types.h"

namespace qwk {

// The one dynamic shared-memory arena of every kernel in this file. Device functions address it as
// `qw_smem + offset`, so the compiler emits LDS/STS/ATOMS (32-bit shared addressing) instead of
// generic loads with 64-bit address arithmetic.
extern __shared__ __align__(16) uint8_t qw_smem[];

struct Key {
  uint64_t w0, w1, w2;
};

__device__ __forceinline__ bool key_ge(const Key& a, const Key& b) {
  if (a.w0 != b.w0) return a.w0 > b.w0;
  if (a.w1 != b.w1) return a.w1 > b.w1;
  return a.w2 >= b.w2;
}
__device__ __forceinline__ bool key_lt(const Key& a, const Key& b) { return !key_ge(a, b); }

// ORs the low `nbits` bits of v (v < 2^nbits) into the key at bit position `pos`, counted from the
// most significant bit of the 192-bit string
__device__ __forceinline__ void key_put(Key& k, uint32_t pos, uint64_t v, uint32_t nbits) {
  if (nbits == 0) return;
  const uint32_t sh = 192u - pos - nbits, w = sh >> 6, s = sh & 63u;
  const uint64_t lo = v << s, hi = s ? v >> (64u - s) : 0ull;
  if (w == 0) { k.w2 |= lo; k.w1 |= hi; }
  else if (w == 1) { k.w1 |= lo; k.w0 |= hi; }
  else k.w0 |= lo;
}
__device__ __forceinline__ uint64_t key_get(const Key& k, uint32_t pos, uint32_t nbits) {
  if (nbits == 0) return 0;
  const uint32_t sh = 192u - pos - nbits, w = sh >> 6, s = sh & 63u;
  const uint64_t lo = w == 0 ? k.w2 : (w == 1 ? k.w1 : k.w0);
  const uint64_t hi = w == 0 ? k.w1 : (w == 1 ? k.w0 : 0ull);
  const uint64_t v = s ? ((lo >> s) | (hi << (64u - s))) : lo;
  return nbits >= 64 ? v : (v & ((1ull << nbits) - 1));
}
// 11-bit digit number `level` counted from the most significant bit of the 192-bit key
__device__ __forceinline__ uint32_t key_digit(const Key& k, uint32_t level) {
  uint32_t o = level * QW_DIGIT_BITS, word = o >> 6, sh = o & 63;
  uint64_t hi = word == 0 ? k.w0 : (word == 1 ? k.w1 : k.w2);
  uint64_t lo = word == 0 ? k.w1 : (word == 1 ? k.w2 : 0ull);
  uint64_t v = sh ? ((hi << sh) | (lo >> (64 - sh))) : hi;
  return (uint32_t)(v >> (64 - QW_DIGIT_BITS));
}
// do the first `bits` bits of a and b agree?
__device__ __forceinline__ bool key_prefix_eq(const Key& a, const uint64_t* t, uint32_t bits) {
  if (bits == 0) return true;
  uint64_t x0 = a.w0 ^ t[0], x1 = a.w1 ^ t[1], x2 = a.w2 ^ t[2];
  if (bits <= 64) return (x0 >> (64 - bits)) == 0;
  if (x0) return false;
  if (bits <= 128) return (x1 >> (128 - bits)) == 0;
  if (x1) return false;
  return (x2 >> (192 - bits)) == 0;
}

__device__ __forceinline__ uint32_t f32_ordered(float f) {
  uint32_t b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ uint64_t f64_to_u64_dev(double d) {
  uint64_t b = (uint64_t)__double_as_longlong(d);
  return (b & (1ull << 63)) ? ~b : (b ^ (1ull << 63));
}
__device__ __forceinline__ double mapped_to_f64(uint32_t type, uint64_t m) {
  switch (type) {
    case QW_COL_U64: case QW_COL_BOOL: case QW_COL_STR: return (double)m;
    case QW_COL_I64: case QW_COL_DATETIME: return (double)(long long)(m ^ (1ull << 63));
    default: {
      uint64_t bits = (m & (1ull << 63)) ? (m ^ (1ull << 63)) : ~m;
      return __longlong_as_double((long long)bits);
    }
  }
}

// ---- columnar reads (tantivy-bitpacker BitUnpacker::get semantics, aligned 64-bit loads) ---------
__device__ __forceinline__ uint64_t col_raw(const uint8_t* base, const DCol& c, uint64_t idx) {
  if (c.bits == 0) return 0;
  const uint64_t* w = (const uint64_t*)(base + c.values_off);
  uint64_t bitpos = idx * c.bits, wi = bitpos >> 6;
  uint32_t sh = (uint32_t)(bitpos & 63);
  uint64_t v = __ldg(w + wi) >> sh;
  if (sh + c.bits > 64) v |= __ldg(w + wi + 1) << (64 - sh);
  return c.bits == 64 ? v : (v & ((1ull << c.bits) - 1));
}
__device__ __forceinline__ void col_range(const uint8_t* base, const DCol& c, uint32_t d, uint64_t& a, uint64_t& b) {
  if (c.card == QW_CARD_FULL) { a = d; b = (uint64_t)d + 1; return; }
  const uint8_t* ix = base + c.index_off;
  if (c.card == QW_CARD_OPTIONAL) {
    const uint64_t* present = (const uint64_t*)ix;
    const uint32_t* rank = (const uint32_t*)(ix + 8ull * c.nwords64);
    uint64_t word = __ldg(present + (d >> 6));
    if (!((word >> (d & 63)) & 1)) { a = b = 0; return; }
    a = __ldg(rank + (d >> 6)) + __popcll(word & ((1ull << (d & 63)) - 1));
    b = a + 1;
    return;
  }
  const uint32_t* start = (const uint32_t*)ix;
  a = __ldg(start + d);
  b = __ldg(start + d + 1);
}

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  uint32_t s = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gsrc));
}
__device__ __forceinline__ void cp_async_wait_all() {
  asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;\n" ::: "memory");
}

// SortOrder::compare_opt (quickwit-proto/src/lib.rs:122-140)
__device__ __forceinline__ int order_cmp(uint32_t order, uint64_t a, uint64_t b) {
  int c = a < b ? -1 : (a > b ? 1 : 0);
  return order == QW_ORDER_DESC ? c : -c;
}
__device__ __forceinline__ int order_cmp_opt(uint32_t order, bool ha, uint64_t a, bool hb, uint64_t b) {
  if (ha && hb) return order_cmp(order, a, b);
  if (ha) return 1;
  if (hb) return -1;
  return 0;
}

// Per-CTA view of the shared-memory arena
struct Sm {
  const SmemLayout* L;
  __device__ __forceinline__ uint32_t* u32(uint32_t off) const { return (uint32_t*)(qw_smem + off); }
  __device__ __forceinline__ float* f32(uint32_t off) const { return (float*)(qw_smem + off); }
  __device__ __forceinline__ uint8_t* u8(uint32_t off) const { return qw_smem + off; }
};

struct TermTarget {
  uint32_t bits;   // shared-memory byte offsets (0xFFFFFFFF = absent)
  uint32_t cnt;
  uint32_t score;
  uint32_t fn;     // staged fieldnorm ids of the window (absent: constant fieldnorm id 1)
  const float* gtab;  // global: float[256] BM25 norms then float[QW_TFF_ROWS][256] tf factors (read via L1)
  float weight;
  bool has_tf;
};

// Decode one posting block (header + 4-lane-interleaved bit-packed doc deltas + tfs) with one warp
// and fold the postings that fall into [ws, we) into the target (all targets live in shared
// memory). STAGED: the block bytes are in shared memory at qw_smem + blk_off; otherwise `gblk`
// points to global memory.
template <bool SCORED, bool CNT, bool STAGED, bool BITS = true>
__device__ __forceinline__ void fold_block(uint32_t blk_off, const uint8_t* gblk, uint32_t ws, uint32_t rlo, uint32_t rlen, const TermTarget& tg, uint32_t lane) {
  const uint8_t* blk = STAGED ? (qw_smem + blk_off) : gblk;
  const uint4 h = *reinterpret_cast<const uint4*>(blk);  // QwSkip: last_doc, prev_last_doc, byte_off, bits/count
  const uint32_t last_doc = h.x, prev = h.y;
  const uint32_t doc_bits = h.w & 0xFF, tf_bits = (h.w >> 8) & 0xFF, count = h.w >> 16;
  // accepted docs: ws + rlo <= doc < ws + rlo + rlen (targets are indexed by doc - ws)
  if (last_doc < ws + rlo) return;
  if (prev != QW_NO_PREV_DOC && prev + 1 >= ws + rlo + rlen) return;
  const uint4* dp = reinterpret_cast<const uint4*>(blk + 16);
  uint32_t v0 = 0, v1 = 0, v2 = 0, v3 = 0;
  if (doc_bits) {
    uint32_t bitpos = lane * doc_bits, wi = bitpos >> 5, sh = bitpos & 31;
    uint4 A = dp[wi];
    uint4 B = (sh + doc_bits > 32) ? dp[wi + 1] : make_uint4(0, 0, 0, 0);
    uint32_t mask = 0xFFFFFFFFu >> (32 - doc_bits);
    v0 = __funnelshift_r(A.x, B.x, sh) & mask;
    v1 = __funnelshift_r(A.y, B.y, sh) & mask;
    v2 = __funnelshift_r(A.z, B.z, sh) & mask;
    v3 = __funnelshift_r(A.w, B.w, sh) & mask;
  }
  // strictly-sorted deltas: doc[i] = doc[i-1] + v[i] + 1
  uint32_t d0 = v0 + 1, d1 = d0 + v1 + 1, d2 = d1 + v2 + 1, d3 = d2 + v3 + 1;
  uint32_t incl = d3;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    uint32_t n = __shfl_up_sync(0xFFFFFFFFu, incl, o);
    if ((int)lane >= o) incl += n;
  }
  const uint32_t basev = prev + (incl - d3) - ws;  // mod 2^32; window-relative
  uint32_t rel[4] = {basev + d0, basev + d1, basev + d2, basev + d3};
  const uint32_t nvalid = count > lane * 4 ? count - lane * 4 : 0;  // postings of this lane that exist
  uint32_t tf[4] = {1, 1, 1, 1};
  if (SCORED && tg.has_tf && tf_bits) {
    const uint4* tp = dp + doc_bits;
    uint32_t bitpos = lane * tf_bits, wi = bitpos >> 5, sh = bitpos & 31;
    uint4 A = tp[wi];
    uint4 B = (sh + tf_bits > 32) ? tp[wi + 1] : make_uint4(0, 0, 0, 0);
    uint32_t mask = 0xFFFFFFFFu >> (32 - tf_bits);
    tf[0] = __funnelshift_r(A.x, B.x, sh) & mask;
    tf[1] = __funnelshift_r(A.y, B.y, sh) & mask;
    tf[2] = __funnelshift_r(A.z, B.z, sh) & mask;
    tf[3] = __funnelshift_r(A.w, B.w, sh) & mask;
  }
  uint32_t* bits = reinterpret_cast<uint32_t*>(qw_smem + tg.bits);
  float* score = reinterpret_cast<float*>(qw_smem + tg.score);
  const float* tab = tg.gtab;
  const uint8_t* fn = qw_smem + tg.fn;
  uint8_t* cnt = qw_smem + tg.cnt;
  const bool has_fn = tg.fn != 0xFFFFFFFFu;
  // The 4 postings of a lane are independent (distinct docs): issue all loads of a stage before
  // consuming them so the shared-memory latencies overlap (fieldnorm -> table -> score RMW).
  bool in[4];
  uint32_t f[4];
#pragma unroll
  for (int j = 0; j < 4; j++) {
    in[j] = (uint32_t)j < nvalid && rel[j] - rlo < rlen;  // rel = doc - ws (unsigned wrap before the window)
    f[j] = (SCORED && has_fn && in[j]) ? fn[rel[j]] : 1u;
  }
  if (SCORED) {
    float tfn[4], old[4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
      // Bm25Weight::score: weight * (tf / (tf + cache[fieldnorm_id])), f32 round-to-nearest; the
      // quotient comes from a table built with the same IEEE ops for tf < 16
      const uint32_t t = tf[j];
      tfn[j] = 0.0f;
      old[j] = 0.0f;
      if (in[j]) {
        if (t < QW_TFF_ROWS) tfn[j] = __ldg(tab + 256 + t * 256 + f[j]);
        else { float tff = (float)t; tfn[j] = __fdiv_rn(tff, __fadd_rn(tff, __ldg(tab + f[j]))); }
        old[j] = score[rel[j]];
      }
    }
#pragma unroll
    for (int j = 0; j < 4; j++)
      if (in[j]) score[rel[j]] = __fadd_rn(old[j], __fmul_rn(tg.weight, tfn[j]));
  }
  if (CNT) {
#pragma unroll
    for (int j = 0; j < 4; j++) if (in[j]) cnt[rel[j]] = (uint8_t)(cnt[rel[j]] + 1);
  }
  if (BITS) {
    uint32_t cur_word = 0xFFFFFFFFu, cur_mask = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      if (!in[j]) continue;
      const uint32_t w = rel[j] >> 5;
      if (w != cur_word) {
        if (cur_mask) atomicOr(&bits[cur_word], cur_mask);
        cur_word = w;
        cur_mask = 0;
      }
      cur_mask |= 1u << (rel[j] & 31);
    }
    if (cur_mask) atomicOr(&bits[cur_word], cur_mask);
  }
}

template <bool STAGED>
__device__ __forceinline__ void fold_block_dyn(uint32_t blk_off, const uint8_t* gblk, uint32_t ws, uint32_t rlo, uint32_t rlen, const TermTarget& tg, uint32_t lane) {
  const bool sc = tg.score != 0xFFFFFFFFu, cn = tg.cnt != 0xFFFFFFFFu;
  if (sc) { if (cn) fold_block<true, true, STAGED>(blk_off, gblk, ws, rlo, rlen, tg, lane); else fold_block<true, false, STAGED>(blk_off, gblk, ws, rlo, rlen, tg, lane); }
  else { if (cn) fold_block<false, true, STAGED>(blk_off, gblk, ws, rlo, rlen, tg, lane); else fold_block<false, false, STAGED>(blk_off, gblk, ws, rlo, rlen, tg, lane); }
}

// A phrase's pre-computed posting block (phrase_kernel.cuh): doc ids and score contributions are already
// decoded, 4 entries per lane; same targets as fold_block (score add in clause order, should counter, bitmap).
__device__ __forceinline__ void fold_vblock(const VBlk* vb, uint32_t ws, uint32_t rlen, const TermTarget& tg, uint32_t lane) {
  const uint4 d = __ldg(reinterpret_cast<const uint4*>(&vb->doc[lane * 4]));
  const float4 v = __ldg(reinterpret_cast<const float4*>(&vb->val[lane * 4]));
  const uint32_t doc[4] = {d.x, d.y, d.z, d.w};
  const float val[4] = {v.x, v.y, v.z, v.w};
  uint32_t* bits = reinterpret_cast<uint32_t*>(qw_smem + tg.bits);
  float* score = reinterpret_cast<float*>(qw_smem + tg.score);
  uint8_t* cnt = qw_smem + tg.cnt;
  const bool sc = tg.score != 0xFFFFFFFFu, cn = tg.cnt != 0xFFFFFFFFu;
#pragma unroll
  for (int j = 0; j < 4; j++) {
    const uint32_t rel = doc[j] - ws;  // (0xFFFFFFFF = no phrase match at this driver posting: never inside a window)
    if (doc[j] == 0xFFFFFFFFu || rel >= rlen) continue;
    if (sc) score[rel] = __fadd_rn(score[rel], val[j]);
    if (cn) cnt[rel] = (uint8_t)(cnt[rel] + 1);
    atomicOr(&bits[rel >> 5], 1u << (rel & 31));
  }
}

// BM25-union pipeline, first half: decode a STAGED posting block and compute the score contribution
// of each of the lane's 4 postings (weight * tf-factor) WITHOUT touching the accumulator, so that it
// can run ahead of the clause order; `inmask` bit j = posting j exists and lies inside the window.
__device__ __forceinline__ void union_decode(uint32_t blk_off, uint32_t ws, uint32_t wlen, const TermTarget& tg, uint32_t lane,
                                             uint32_t (&rel)[4], float (&contrib)[4], uint32_t& inmask) {
  const uint8_t* blk = qw_smem + blk_off;
  const uint4 h = *reinterpret_cast<const uint4*>(blk);  // QwSkip: last_doc, prev_last_doc, byte_off, bits/count
  const uint32_t last_doc = h.x, prev = h.y;
  const uint32_t doc_bits = h.w & 0xFF, tf_bits = (h.w >> 8) & 0xFF, count = h.w >> 16;
  inmask = 0;
  if (last_doc < ws) return;
  if (prev != QW_NO_PREV_DOC && prev + 1 >= ws + wlen) return;
  const uint4* dp = reinterpret_cast<const uint4*>(blk + 16);
  uint32_t v0 = 0, v1 = 0, v2 = 0, v3 = 0;
  if (doc_bits) {
    uint32_t bitpos = lane * doc_bits, wi = bitpos >> 5, sh = bitpos & 31;
    uint4 A = dp[wi];
    uint4 B = (sh + doc_bits > 32) ? dp[wi + 1] : make_uint4(0, 0, 0, 0);
    uint32_t mask = 0xFFFFFFFFu >> (32 - doc_bits);
    v0 = __funnelshift_r(A.x, B.x, sh) & mask;
    v1 = __funnelshift_r(A.y, B.y, sh) & mask;
    v2 = __funnelshift_r(A.z, B.z, sh) & mask;
    v3 = __funnelshift_r(A.w, B.w, sh) & mask;
  }
  uint32_t d0 = v0 + 1, d1 = d0 + v1 + 1, d2 = d1 + v2 + 1, d3 = d2 + v3 + 1;
  uint32_t incl = d3;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    uint32_t n = __shfl_up_sync(0xFFFFFFFFu, incl, o);
    if ((int)lane >= o) incl += n;
  }
  const uint32_t basev = prev + (incl - d3) - ws;  // mod 2^32; window-relative
  rel[0] = basev + d0; rel[1] = basev + d1; rel[2] = basev + d2; rel[3] = basev + d3;
  const uint32_t nvalid = count > lane * 4 ? count - lane * 4 : 0;
  uint32_t tf[4] = {1, 1, 1, 1};
  if (tg.has_tf && tf_bits) {
    const uint4* tp = dp + doc_bits;
    uint32_t bitpos = lane * tf_bits, wi = bitpos >> 5, sh = bitpos & 31;
    uint4 A = tp[wi];
    uint4 B = (sh + tf_bits > 32) ? tp[wi + 1] : make_uint4(0, 0, 0, 0);
    uint32_t mask = 0xFFFFFFFFu >> (32 - tf_bits);
    tf[0] = __funnelshift_r(A.x, B.x, sh) & mask;
    tf[1] = __funnelshift_r(A.y, B.y, sh) & mask;
    tf[2] = __funnelshift_r(A.z, B.z, sh) & mask;
    tf[3] = __funnelshift_r(A.w, B.w, sh) & mask;
  }
  const float* tab = tg.gtab;
  const uint8_t* fn = qw_smem + tg.fn;
  const bool has_fn = tg.fn != 0xFFFFFFFFu;
  uint32_t f[4];
#pragma unroll
  for (int j = 0; j < 4; j++) {
    const bool in = (uint32_t)j < nvalid && rel[j] < wlen;  // rel = doc - ws (unsigned wrap before the window)
    inmask |= (in ? 1u : 0u) << j;
    f[j] = (has_fn && in) ? fn[rel[j]] : 1u;
  }
#pragma unroll
  for (int j = 0; j < 4; j++) {
    // Bm25Weight::score: weight * (tf / (tf + cache[fieldnorm_id])), f32 round-to-nearest
    const uint32_t t = tf[j];
    float tfn = 0.0f;
    if ((inmask >> j) & 1) {
      if (t < QW_TFF_ROWS) tfn = __ldg(tab + 256 + t * 256 + f[j]);
      else { float tff = (float)t; tfn = __fdiv_rn(tff, __fadd_rn(tff, __ldg(tab + f[j]))); }
    }
    contrib[j] = __fmul_rn(tg.weight, tfn);
  }
}

// Composite key + eligibility of one matched doc (sort-value extraction:
// SortingFieldExtractorComponent, quickwit-search/src/collector.rs:139-205)
struct DocKey {
  Key key;
  bool eligible;
};
__device__ __forceinline__ uint32_t score_lin(const DKeySpec& ks, float score, bool desc) {
  const float x = __fmul_rn(score, ks.score_scale);
  const uint32_t l = x >= 1023.0f ? 1023u : (x > 0.0f ? (uint32_t)x : 0u);
  return desc ? l : 1023u - l;
}
__device__ __forceinline__ DocKey doc_key(const DSplitPlan& P, const DKeySpec& ks, const DCol* cols, const uint8_t* base, uint32_t doc, float score) {
  uint32_t has[2] = {0, 0};
  uint64_t v[2] = {0, 0}, r[2] = {0, 0};
#pragma unroll
  for (int i = 0; i < 2; i++) {
    const bool desc = ks.order[i] == QW_ORDER_DESC;
    if (ks.kind[i] == QW_SORT_SCORE) {
      has[i] = 1;
      v[i] = f64_to_u64_dev((double)score);
      const uint32_t o = f32_ordered(score);
      r[i] = desc ? o : ~o;
      if (i == 0) r[i] |= (uint64_t)score_lin(ks, score, desc) << 32;
    } else if (ks.kind[i] == QW_SORT_COLUMN && ks.col[i] != 0xFFFFFFFFu) {
      const DCol& c = cols[ks.col[i]];
      uint64_t a, b;
      col_range(base, c, doc, a, b);
      if (a != b) {
        has[i] = 1;
        const uint64_t raw = col_raw(base, c, a);
        v[i] = c.min_value + c.gcd * raw;
        r[i] = desc ? raw : ks.raw_max[i] - raw;
      }
    }  // doc-id order / column absent from the split: the field contributes no key bits
  }
  const bool desc1 = ks.order[0] == QW_ORDER_DESC;
  const uint32_t docmask = ks.doc_bits >= 32 ? 0xFFFFFFFFu : ((1u << ks.doc_bits) - 1);
  DocKey out;
  out.key = Key{0, 0, 0};
  const uint32_t docr = desc1 ? doc : docmask - doc;
  if (ks.narrow) {
    // fields that are absent have width 0 and value 0, so their (zero) shift is harmless
    out.key.w0 = ((uint64_t)(has[0] & ks.hasbit[0]) << ks.sh_has[0]) | (r[0] << ks.sh_r[0]) |
                 ((uint64_t)(has[1] & ks.hasbit[1]) << ks.sh_has[1]) | (r[1] << ks.sh_r[1]) |
                 ((uint64_t)(ks.doc_bits ? docr : 0u) << ks.sh_doc);
  } else {
    uint32_t pos = 0;
#pragma unroll
    for (int i = 0; i < 2; i++) {
      if (ks.hasbit[i]) { key_put(out.key, pos, has[i], 1); pos++; }
      key_put(out.key, pos, r[i], ks.rbits[i]);
      pos += ks.rbits[i];
    }
    key_put(out.key, pos, docr, ks.doc_bits);
  }
  out.eligible = true;
  if (P.sa.present) {
    // GenericQuickwitSegmentTopKCollector::collect_top_k_vals (top_k_collector.rs:663-699)
    int c = order_cmp_opt(ks.order[0], has[0], v[0], P.sa.has_v1, P.sa.v1);
    if (!c) c = order_cmp_opt(ks.order[1], has[1], v[1], P.sa.has_v2, P.sa.v2);
    if (P.sa.compare_on_equal) {
      if (!c) c = P.sa.precomp_order;
      if (!c) c = order_cmp(ks.order[0], doc, P.sa.doc_id);
    }
    out.eligible = c < 0;
  }
  return out;
}

// The 11 most significant bits of the composite key — the level-0 radix digit and the cheap
// threshold pre-filter — without building the whole key when the first field is wide enough.
__device__ __forceinline__ uint32_t key_top11(const DSplitPlan& P, const DKeySpec& ks, const DCol* cols, const uint8_t* base, uint32_t doc, float score) {
  const bool desc1 = ks.order[0] == QW_ORDER_DESC;
  if (ks.top_mode == QW_TOP_SCORE) return 1024u | score_lin(ks, score, desc1);
  if (ks.top_mode == QW_TOP_COLUMN) {
    const DCol& c = cols[ks.col[0]];
    uint64_t a, b;
    col_range(base, c, doc, a, b);
    if (a == b) return 0;
    const uint64_t raw = col_raw(base, c, a);
    return 1024u | (uint32_t)((desc1 ? raw : ks.raw_max[0] - raw) >> (ks.rbits[0] - 10));
  }
  if (ks.top_mode == QW_TOP_DOC) {
    const uint32_t docmask = ks.doc_bits >= 32 ? 0xFFFFFFFFu : ((1u << ks.doc_bits) - 1);
    return (desc1 ? doc : docmask - doc) >> (ks.doc_bits - 11);
  }
  return (uint32_t)(doc_key(P, ks, cols, base, doc, score).key.w0 >> 53);
}

// ---- aggregation collection (dense cells; mirrors oracle agg_collect) -------------------------------
// All 32 lanes of a warp call these together (`on` = this lane holds a matched doc): lanes that hit
// the same cell are combined before touching the counter, because time-ordered log data sends whole
// warps to the same histogram / terms bucket and same-address atomics serialise.
#define QW_FULL 0xFFFFFFFFu
// Counters whose lanes usually agree (histogram digits / buckets of time-ordered keys): one broadcast
// + ballot decides between a single aggregated atomic and plain per-lane atomics.
__device__ __forceinline__ void warp_count_uniform(uint32_t* ctr, uint32_t idx, bool on, uint32_t lane) {
  const uint32_t m = __ballot_sync(QW_FULL, on);
  if (m == 0) return;
  const uint32_t lead = __ffs(m) - 1;
  const uint32_t lead_idx = __shfl_sync(QW_FULL, idx, lead);  // (outside the &&: every lane must take part)
  const uint32_t same = __ballot_sync(QW_FULL, on && idx == lead_idx);
  if (same == m) { if (lane == lead) atomicAdd(&ctr[idx], (uint32_t)__popc(m)); }
  else if (on) atomicAdd(&ctr[idx], 1u);
}
// Same contract for counters with a handful of distinct targets per warp (terms buckets of a
// low-cardinality column): up to four leader-broadcast rounds, stragglers fall back to plain atomics.
__device__ __forceinline__ void warp_count_few(uint32_t* ctr, uint32_t idx, bool on, uint32_t lane) {
  uint32_t rem = __ballot_sync(QW_FULL, on);
#pragma unroll 1
  for (int r = 0; r < 4 && rem; r++) {
    const uint32_t lead = __ffs(rem) - 1;
    const uint32_t lead_idx = __shfl_sync(QW_FULL, idx, lead);
    const uint32_t same = __ballot_sync(QW_FULL, on && idx == lead_idx) & rem;
    if (lane == lead) atomicAdd(&ctr[lead_idx], (uint32_t)__popc(same));
    rem &= ~same;
  }
  if ((rem >> lane) & 1) atomicAdd(&ctr[idx], 1u);
}
// Fast aggregation path (DSplitPlan::fast_aggs): flat TERMS / HISTOGRAM nodes over single-valued
// columns, counts privatised in shared memory. A histogram bucket is found in raw space through the
// host-built boundary table (DAgg::bounds) — no f64 arithmetic, bit-exact by construction.
// Bit-unpack for the fast aggregation path: single-valued column, index = doc. Columns whose packed
// array is addressable with 32-bit bit positions and whose width is <= 32 use two 32-bit loads and
// a funnel shift (the array is padded with 16 zero bytes, so the second word always exists).
__device__ __forceinline__ uint64_t col_raw_doc(const uint8_t* base, const DCol& c, uint32_t doc, uint32_t num_docs) {
  if (c.bits <= 32 && (uint64_t)num_docs * c.bits < (1ull << 32)) {
    if (c.bits == 0) return 0;
    const uint32_t* w = (const uint32_t*)(base + c.values_off);
    const uint32_t bitpos = doc * c.bits, wi = bitpos >> 5, sh = bitpos & 31;
    const uint32_t v = __funnelshift_r(__ldg(w + wi), __ldg(w + wi + 1), sh);
    return c.bits == 32 ? v : (v & ((1u << c.bits) - 1));
  }
  return col_raw(base, c, doc);
}
// Privatised stats cell of the fast path: {sum (u64 wrapping, or f64 bits), max(~mapped) = min, max(mapped)}.
// When the whole warp feeds one cell the three values are butterfly-reduced first.
__device__ __forceinline__ void stat_update(unsigned long long* st, const DAgg& g, const DCol& c, const uint8_t* base, uint32_t cell, uint32_t doc, uint32_t num_docs, bool ok, uint32_t lane) {
  const uint32_t okmask = __ballot_sync(QW_FULL, ok);
  if (okmask == 0) return;
  const uint64_t raw = ok ? col_raw_doc(base, c, doc, num_docs) : 0ull;
  const uint64_t m = ok ? c.min_value + c.gcd * raw : 0ull;
  // sums: exact integer sum of the RAW offsets (the host rebuilds count * min + gcd * sum in 128 bits, so
  // nanosecond timestamps cannot overflow); other columns add doubles (qw_col_sum_exact, decided on the host)
  const bool is_f64 = g.is_f64;
  unsigned long long isum = ok ? raw : 0ull;
  double dsum = (ok && is_f64) ? mapped_to_f64(c.type, m) : 0.0;
  unsigned long long nmin = ok ? ~m : 0ull, vmax = ok ? m : 0ull;
  const uint32_t lead = __ffs(okmask) - 1;
  const uint32_t lead_cell = __shfl_sync(QW_FULL, cell, lead);
  const bool one = __ballot_sync(QW_FULL, ok && cell != lead_cell) == 0;
  if (one) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      isum += __shfl_xor_sync(QW_FULL, isum, o);
      if (is_f64) dsum += __shfl_xor_sync(QW_FULL, dsum, o);
      const unsigned long long x = __shfl_xor_sync(QW_FULL, nmin, o), y = __shfl_xor_sync(QW_FULL, vmax, o);
      nmin = x > nmin ? x : nmin;
      vmax = y > vmax ? y : vmax;
    }
  }
  if (one ? lane == lead : ok) {
    unsigned long long* t = st + 3ull * cell;
    if (is_f64) atomicAdd((double*)t, dsum); else atomicAdd(t, isum);
    atomicMax(t + 1, nmin);
    atomicMax(t + 2, vmax);
  }
}
__device__ __forceinline__ void agg_collect_fast(const Sm& sm, const DSplitPlan& P, const DAgg* aggs, const DCol* cols,
                                                 const uint8_t* base, uint32_t doc, bool on, uint32_t lane) {
  uint32_t* ctr = sm.u32(sm.L->hist);
  unsigned long long* st = (unsigned long long*)(sm.u8(sm.L->hist) + ((P.n_cells * 4u + 7u) & ~7u));
  for (uint32_t gi = 0; gi < P.n_aggs; gi++) {
    const DAgg& g = aggs[gi];
    if (g.parent != 0xFFFFFFFFu) continue;  // children are visited under their parent
    if (g.kind == QW_AGG_STATS) {
      stat_update(st, g, cols[g.col], base, g.stat_base, doc, P.num_docs, on, lane);
      continue;
    }
    const uint64_t raw = on ? col_raw_doc(base, cols[g.col], doc, P.num_docs) : 0ull;
    bool ok = on;
    uint32_t bk = (uint32_t)raw;
    if (g.kind == QW_AGG_HISTOGRAM) {
      const uint64_t* B = (const uint64_t*)g.bounds;
      const uint32_t nb = g.num_buckets;
      const uint64_t b0 = __ldg(B), bn = __ldg(B + nb);
      ok = on && raw >= b0 && raw < bn;
      bk = 0;
      if (ok) {
        const float f = __fmul_rn((float)(raw - b0), g.inv_step);
        bk = f >= (float)(nb - 1) ? nb - 1 : (uint32_t)f;
        while (raw < __ldg(B + bk)) bk--;
        while (raw >= __ldg(B + bk + 1)) bk++;
      }
    }
    // histogram buckets of (time-)ordered data are usually warp-uniform; terms buckets of a
    // low-cardinality column take a few leader rounds
    if (g.kind == QW_AGG_HISTOGRAM) warp_count_uniform(ctr, g.cell_base + bk, ok, lane);
    else warp_count_few(ctr, g.cell_base + bk, ok, lane);
    for (uint32_t ci = 0; ci < g.num_children; ci++) {
      const DAgg& ch = aggs[g.first_child + ci];  // STATS over an always-present column
      stat_update(st, ch, cols[ch.col], base, ch.stat_base + bk, doc, P.num_docs, ok, lane);
    }
  }
}
__device__ __forceinline__ void agg_count(const KParams& p, const Sm& sm, QwAggCell* cells, uint32_t cell, bool on, uint32_t lane) {
  const uint32_t peers = __match_any_sync(QW_FULL, on ? cell : 0xFFFFFFFFu);
  if (on && (uint32_t)(__ffs(peers) - 1) == lane) {
    if (p.smem_aggs) atomicAdd(&sm.u32(sm.L->hist)[cell], (uint32_t)__popc(peers));
    else atomicAdd((unsigned long long*)&cells[cell].count, (unsigned long long)__popc(peers));
  }
}
__device__ __forceinline__ void agg_stats(const DAgg& g, const DCol& c, const uint8_t* base, QwAggCell* cells, uint32_t cell, uint32_t doc, bool on, uint32_t lane) {
  uint64_t a = 0, b = 0;
  if (on) col_range(base, c, doc, a, b);
  const uint32_t nv = (uint32_t)(b - a);
  const uint32_t maxv = __reduce_max_sync(QW_FULL, nv);
  const bool is_f64 = g.is_f64;
  for (uint32_t k = 0; k < maxv; k++) {
    const bool ok = k < nv;
    const uint32_t okmask = __ballot_sync(QW_FULL, ok);
    uint64_t m = 0, raw = 0;
    if (ok) { raw = col_raw(base, c, a + k); m = c.min_value + c.gcd * raw; }
    const uint32_t peers = __match_any_sync(QW_FULL, ok ? cell : 0xFFFFFFFFu);
    QwAggCell* out = &cells[g.cell_base + cell];
    if (__all_sync(QW_FULL, !ok || peers == okmask)) {
      // the whole warp feeds one cell: butterfly-reduce, one lane issues the four atomics
      unsigned long long isum = ok ? raw : 0ull;
      double dsum = (ok && is_f64) ? mapped_to_f64(c.type, m) : 0.0;
      unsigned long long nmin = ok ? ~m : 0ull, vmax = ok ? m : 0ull;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        isum += __shfl_xor_sync(QW_FULL, isum, o);
        if (is_f64) dsum += __shfl_xor_sync(QW_FULL, dsum, o);
        const unsigned long long x = __shfl_xor_sync(QW_FULL, nmin, o), y = __shfl_xor_sync(QW_FULL, vmax, o);
        nmin = x > nmin ? x : nmin;
        vmax = y > vmax ? y : vmax;
      }
      if (ok && (uint32_t)(__ffs(okmask) - 1) == lane) {
        atomicAdd((unsigned long long*)&out->count, (unsigned long long)__popc(okmask));
        if (is_f64) atomicAdd((double*)&out->sum_bits, dsum);
        else atomicAdd((unsigned long long*)&out->sum_bits, isum);
        atomicMax((unsigned long long*)&out->min_mapped, nmin);  // min kept as max(~m): zero-initialisable
        atomicMax((unsigned long long*)&out->max_mapped, vmax);
      }
    } else if (ok) {
      atomicAdd((unsigned long long*)&out->count, 1ull);
      if (is_f64) atomicAdd((double*)&out->sum_bits, mapped_to_f64(c.type, m));
      else atomicAdd((unsigned long long*)&out->sum_bits, (unsigned long long)raw);
      atomicMax((unsigned long long*)&out->min_mapped, (unsigned long long)~m);
      atomicMax((unsigned long long*)&out->max_mapped, (unsigned long long)m);
    }
  }
}
// bucket index of value index i for bucket aggregation g; returns false when the value falls in no bucket
__device__ __forceinline__ bool agg_bucket(const DAgg& g, const DCol& c, const uint8_t* base, uint64_t i, uint32_t r, uint32_t& bucket) {
  uint64_t raw = col_raw(base, c, i);
  if (g.kind == QW_AGG_TERMS) { bucket = (uint32_t)raw; return r == 0; }
  uint64_t m = c.min_value + c.gcd * raw;
  if (g.kind == QW_AGG_HISTOGRAM) {
    if (r != 0) return false;
    double val = mapped_to_f64(c.type, m);
    if (g.has_bounds && !(val >= g.bound_min && val <= g.bound_max)) return false;
    double pos = floor(__ddiv_rn(__dsub_rn(val, g.offset), g.interval));
    long long idx = (long long)pos - g.base_pos;
    if (idx < 0 || idx >= (long long)g.num_buckets) return false;
    bucket = (uint32_t)idx;
    return true;
  }
  // RANGE: bucket r = [from, to)
  bucket = r;
  return m >= g.range_from[r] && m < g.range_to[r];
}
// value-index range of `doc` in bucket aggregation g's column (one pseudo value for a `missing` bucket)
__device__ __forceinline__ uint32_t agg_values(const DAgg& g, const DCol* cols, const uint8_t* base, uint32_t doc, bool on, uint64_t& a, bool& missing) {
  uint64_t b = 0;
  a = 0;
  if (on && g.col != 0xFFFFFFFFu) col_range(base, cols[g.col], doc, a, b);
  missing = on && (a == b) && g.kind == QW_AGG_TERMS && g.has_missing;
  return on ? (missing ? 1u : (uint32_t)(b - a)) : 0u;
}
__device__ void agg_collect_doc(const KParams& p, const Sm& sm, const DSplitPlan& P, const DAgg* aggs, const DCol* cols,
                                const uint8_t* base, QwAggCell* cells, uint32_t doc, bool on, uint32_t lane) {
  for (uint32_t gi = 0; gi < P.n_aggs; gi++) {
    const DAgg& g = aggs[gi];
    if (g.parent != 0xFFFFFFFFu) continue;
    if (g.kind == QW_AGG_STATS) {
      if (g.col != 0xFFFFFFFFu) agg_stats(g, cols[g.col], base, cells, 0, doc, on, lane);
      continue;
    }
    uint64_t a;
    bool missing;
    const uint32_t nv = agg_values(g, cols, base, doc, on, a, missing);
    const uint32_t maxv = __reduce_max_sync(QW_FULL, nv);
    const uint32_t nrep = g.kind == QW_AGG_RANGE ? g.num_ranges : 1;
    for (uint32_t k = 0; k < maxv; k++) {
      for (uint32_t r = 0; r < nrep; r++) {
        bool ok = k < nv;
        uint32_t bk = 0;
        if (ok) {
          if (missing) bk = g.num_buckets - 1;
          else ok = agg_bucket(g, cols[g.col], base, a + k, r, bk);
        }
        agg_count(p, sm, cells, g.cell_base + bk, ok, lane);
        for (uint32_t ci = 0; ci < g.num_children; ci++) {
          const DAgg& ch = aggs[g.first_child + ci];
          if (ch.kind == QW_AGG_STATS) {
            if (ch.col != 0xFFFFFFFFu) agg_stats(ch, cols[ch.col], base, cells, bk, doc, ok, lane);
            continue;
          }
          uint64_t a2;
          bool missing2;
          const uint32_t nv2 = agg_values(ch, cols, base, doc, ok, a2, missing2);
          const uint32_t maxv2 = __reduce_max_sync(QW_FULL, nv2);
          const uint32_t nrep2 = ch.kind == QW_AGG_RANGE ? ch.num_ranges : 1;
          for (uint32_t k2 = 0; k2 < maxv2; k2++) {
            for (uint32_t r2 = 0; r2 < nrep2; r2++) {
              bool ok2 = k2 < nv2;
              uint32_t bk2 = 0;
              if (ok2) {
                if (missing2) bk2 = ch.num_buckets - 1;
                else ok2 = agg_bucket(ch, cols[ch.col], base, a2 + k2, r2, bk2);
              }
              const uint32_t cell2 = bk * ch.num_buckets + bk2;
              agg_count(p, sm, cells, ch.cell_base + cell2, ok2, lane);
              for (uint32_t gc = 0; gc < ch.num_children; gc++) {
                const DAgg& g3 = aggs[ch.first_child + gc];
                if (g3.kind == QW_AGG_STATS && g3.col != 0xFFFFFFFFu) agg_stats(g3, cols[g3.col], base, cells, cell2, doc, ok2, lane);
              }
            }
          }
        }
      }
    }
  }
}

enum { MODE_HIST = 0, MODE_COLLECT = 1 };

// ---- warp-private helpers (each warp owns the doc sub-range [lo, lo + S) of the window) ------------
__device__ __forceinline__ void wzero_u32(uint32_t* p, uint32_t first, uint32_t n, uint32_t lane) {
  for (uint32_t i = lane; i < n; i += 32) p[first + i] = 0;
}

__device__ __forceinline__ void zero_f4(float* p, uint32_t n, uint32_t tid) {
  float4* q = reinterpret_cast<float4*>(p);
  const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
  for (uint32_t i = tid; i < (n >> 2); i += QW_THREADS) q[i] = z;
}

// Runs body(i, on) over the set bits of a window bitmap with FULL warps: each warp compacts the hits of
// its share of the bitmap (8 words = 256 docs per step) into a small shared-memory queue and calls the
// body on 32 hits at a time — sparse result sets (a few hits per 32-doc word) would otherwise spend a
// whole warp iteration per word with one or two active lanes. The body always runs converged (all 32
// lanes, `on` false for padding lanes), so it may use warp collectives.
// The queues alias the per-window term tables (rng / blkrec / termblk), which are dead once the
// program has run.
#define QW_HITQ_WORDS 4
#define QW_HITQ_CAP (32 + 32 * QW_HITQ_WORDS)
static_assert(QW_WARPS * QW_HITQ_CAP * 2 <= QW_MAX_TERMS * 16 + QW_MAX_WBLK * 8 + QW_MAX_TERMS * 8, "hit queues must fit the aliased term tables");
static_assert(QW_MAX_INSTR <= 255, "s_tinstr holds instruction indices as bytes");
template <class F>
__device__ __forceinline__ void warp_for_hits(const uint32_t* res, uint32_t NW, uint32_t warp, uint32_t lane, uint16_t* q, F&& body) {
  uint32_t cnt = 0;  // queued hits (warp-uniform, < 32 between steps)
  // drain full batches of 32 from the queue, move the remainder to the front
  auto drain = [&]() {
    uint32_t done = 0;
    while (cnt - done >= 32) {
      body((uint32_t)q[done + lane], true);
      done += 32;
    }
    if (done) {
      const uint32_t rem = cnt - done;
      const uint16_t v = lane < rem ? q[done + lane] : (uint16_t)0;
      __syncwarp();
      if (lane < rem) q[lane] = v;
      cnt = rem;
    }
    __syncwarp();
  };
  // a super-step covers 32 bitmap words (1024 docs), one word per lane
  for (uint32_t s0 = warp * 32; s0 < NW; s0 += QW_WARPS * 32) {
    uint32_t word = s0 + lane < NW ? res[s0 + lane] : 0u;
    const uint32_t c = __popc(word);
    uint32_t incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
      if ((int)lane >= o) incl += t;
    }
    const uint32_t total = __shfl_sync(0xFFFFFFFFu, incl, 31);
    if (total == 0) continue;
    if (total <= 32 * QW_HITQ_WORDS) {
      // sparse: every lane extracts the hits of its own word; the queue has room for all of them
      uint32_t off = cnt + incl - c;
      const uint32_t first = (s0 + lane) * 32;
      while (word) {
        q[off++] = (uint16_t)(first + __ffs(word) - 1);
        word &= word - 1;
      }
      __syncwarp();
      cnt += total;
      drain();
      continue;
    }
    // denser: QW_HITQ_WORDS words at a time
    for (uint32_t g = 0; g < 32; g += QW_HITQ_WORDS) {
      uint32_t wg = __shfl_sync(0xFFFFFFFFu, word, g + (lane & (QW_HITQ_WORDS - 1)));
      if (lane >= QW_HITQ_WORDS) wg = 0;
      const uint32_t cg = __popc(wg);
      uint32_t ig = cg;
#pragma unroll
      for (int o = 1; o < QW_HITQ_WORDS; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, ig, o);
        if ((int)lane >= o) ig += t;
      }
      const uint32_t tg = __shfl_sync(0xFFFFFFFFu, ig, QW_HITQ_WORDS - 1);
      if (tg == 0) continue;
      if (tg >= 24 * QW_HITQ_WORDS) {
        // dense stretch: lanes map straight to docs, no compaction
#pragma unroll
        for (int k = 0; k < QW_HITQ_WORDS; k++) {
          const uint32_t wk = __shfl_sync(0xFFFFFFFFu, wg, k);
          if (wk) body((s0 + g + k) * 32 + lane, (wk >> lane) & 1);
        }
        continue;
      }
      uint32_t off = cnt + ig - cg;
      const uint32_t first = (s0 + g + lane) * 32;
      while (wg) {
        q[off++] = (uint16_t)(first + __ffs(wg) - 1);
        wg &= wg - 1;
      }
      __syncwarp();
      cnt += tg;
      drain();
    }
  }
  if (cnt) body(lane < cnt ? (uint32_t)q[lane] : 0u, lane < cnt);
}

// Warp-cooperative 32-ary search of a term's skip list: ordinal of the first block whose last doc
// is >= ws (nblk when there is none). All lanes return the same value.
__device__ __forceinline__ uint32_t first_block_ge(const QwSkip* skips, uint32_t nblk, uint32_t ws, uint32_t lane) {
  uint32_t a = 0, b = nblk;
  while (b - a > 32) {
    uint32_t step = (b - a + 31) >> 5;
    uint32_t idx = a + lane * step;
    bool ok = idx < b && __ldg(&skips[idx].last_doc) >= ws;
    uint32_t m = __ballot_sync(0xFFFFFFFFu, ok);
    if (m == 0) a = a + ((b - 1 - a) / step) * step + 1;
    else { uint32_t f = __ffs(m) - 1; b = a + f * step + 1; if (f > 0) a = a + (f - 1) * step + 1; }
  }
  uint32_t idx = a + lane;
  bool ok = idx < b && __ldg(&skips[idx].last_doc) >= ws;
  uint32_t m = __ballot_sync(0xFFFFFFFFu, ok);
  return m ? a + (__ffs(m) - 1) : nblk;
}

struct BlkRec {  // one staged posting block of the window
  uint16_t soff;  // byte offset of the block inside the stage area
  uint16_t lo;    // lower bound of its first doc, window-relative, clamped to [0, W]
  uint16_t hi;    // last doc, window-relative, clamped to [0, W-1] (0xFFFF: entirely before the window)
  uint8_t slot;   // term slot
  uint8_t pad;
};

// The window engine (see the file header): phases 1-3 stage the window's bytes and build the block
// table, then the boolean program runs block-wide, then the matches are collected.
//
// UNION = true is the specialised instantiation for the BM25 top-K shape (every plan of the batch is
// a pure OR of positive-weight scored terms ranked by _score desc, no search_after, no aggregations;
// see lower_plan): the program degenerates to "zero the accumulator, fold every term", matches and
// the hit count come from the score array in the fused collect sweep, and none of the bitmap
// machinery is compiled in. The host launches it only when the whole batch qualifies.
template <int MODE, bool UNION>
__global__ void __launch_bounds__(QW_THREADS, QW_MIN_BLOCKS_PER_SM) k_window(const KParams p) {
  Sm sm{&p.sm};
  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t W = p.W, NW = W >> 5;
  const uint32_t S = W / QW_WARPS, SW = S >> 5;      // docs / bitmap words per warp
  const uint32_t lo = warp * S, wlo = warp * SW;      // this warp's sub-range (window-relative)
  DInstr* s_instr = (DInstr*)sm.u8(p.sm.instr);
  DCol* s_cols = (DCol*)sm.u8(p.sm.cols);
  DAgg* s_aggs = (DAgg*)sm.u8(p.sm.aggs);
  const DKeySpec& ks = *(const DKeySpec*)sm.u8(p.sm.key);  // the current split's key spec (shared-memory copy)
  uint16_t* s_hitq = (uint16_t*)sm.u8(p.sm.hitq) + (threadIdx.x >> 5) * QW_HITQ_CAP;  // this warp's hit queue
  uint32_t* s_misc = sm.u32(p.sm.misc);  // [0] total staged blocks, [2] hits, [3] eligible
  uint32_t* s_rng = sm.u32(p.sm.rng);    // per term slot: start, len, stage_off (per window)
  uint8_t* s_tinstr = sm.u8(p.sm.misc) + 32 + 4 * QW_MAX_TERMS;  // per term slot: its TERM instruction (per split)
  BlkRec* s_blk = (BlkRec*)sm.u8(p.sm.blkrec);
  uint32_t* s_tblk = sm.u32(p.sm.termblk);  // per term slot: first global block, block count
  uint32_t* s_hist = sm.u32(p.sm.hist);
  uint8_t* s_stage = sm.u8(p.sm.stage);
  uint32_t loaded_split = 0xFFFFFFFFu;
  bool ssum_clean = false;  // level-0 should-score array is all zero (left so by a fused collect)

  const uint32_t per = (p.total_work + gridDim.x - 1) / gridDim.x;
  const uint32_t w_begin = blockIdx.x * per;
  const uint32_t w_end = min(w_begin + per, p.total_work);
  uint32_t split = 0;
  if (w_begin < w_end) {
    uint32_t a = 0, b = p.n_splits;
    while (b - a > 1) {
      uint32_t mid = (a + b) >> 1;
      if (__ldg(p.first_work + mid) <= w_begin) a = mid; else b = mid;
    }
    split = a;
  }

  for (uint32_t work = w_begin; work < w_end; work++) {
    while (__ldg(p.first_work + split + 1) <= work) split++;
    // sampled passes with an explicit window list: the strided sample plus the first and last window of every
    // split (keys that follow doc order — doc id, timestamps of time-ordered logs — have their best K there);
    // a strided window stands for `stride` windows in the histogram, an edge window for itself
    uint32_t window, hist_weight = 1;
    if (p.sample_win) {
      const uint32_t e = __ldg(p.sample_win + work);
      window = e & 0x7FFFFFFFu;
      hist_weight = (e >> 31) ? 1u : p.stride;
    } else window = (work - __ldg(p.first_work + split)) * p.stride + (p.stride > 1 ? split % p.stride : 0);
    if (p.refine) {
      // second-chance passes: verified splits are final, and a window whose best level-0 digit is
      // below the threshold digit cannot hold a candidate (block-uniform tests)
      if (__ldg(p.split_state + split) == 0) continue;
      if ((uint32_t)p.wmax[work] < (uint32_t)(p.thresh[split].key[0] >> 53) + 1u) continue;
    }
    const DSplitPlan& P = p.plans[split];
    __syncthreads();  // previous window fully finished (stage / entries / program are reused)
    if (split != loaded_split) {
      const uint4* src = (const uint4*)(p.instrs + P.instr_base);
      for (uint32_t i = tid; i < P.n_instr * (sizeof(DInstr) / 16); i += QW_THREADS) ((uint4*)s_instr)[i] = __ldg(src + i);
      src = (const uint4*)(p.cols + P.col_base);
      for (uint32_t i = tid; i < P.n_cols * (sizeof(DCol) / 16); i += QW_THREADS) ((uint4*)s_cols)[i] = __ldg(src + i);
      src = (const uint4*)(p.aggs + P.agg_base);
      for (uint32_t i = tid; i < P.n_aggs * (sizeof(DAgg) / 16); i += QW_THREADS) ((uint4*)s_aggs)[i] = __ldg(src + i);
      src = (const uint4*)&P.key;
      if (tid < sizeof(DKeySpec) / 16) ((uint4*)sm.u8(p.sm.key))[tid] = __ldg(src + tid);
      loaded_split = split;
      ssum_clean = false;
      __syncthreads();
      if (tid < P.n_instr && s_instr[tid].op == OP_TERM) s_tinstr[s_instr[tid].t] = (uint8_t)tid;  // term slot -> instruction (kept per split)
      __syncthreads();
    }
    const uint8_t* base = (const uint8_t*)P.data_base;
    const uint32_t ws = window * W;
    const uint32_t we = min(ws + W, P.num_docs);
    const uint32_t wlen = we - ws;
    const uint32_t n_terms = P.n_terms, n_instr = P.n_instr, n_fn = P.n_fn_slots;

    // ---- phase 1: window-index entries + fieldnorm staging (one round of independent loads) --------
    if (tid < n_terms) {
      const DInstr& in = s_instr[s_tinstr[tid]];
      uint32_t start = 0, len = 0, fb = 0, nb = 0;
      if (in.n) {
        const uint4* wi = (const uint4*)(base + in.b);
        const uint32_t e0 = ws >> in.m, e1 = (we - 1) >> in.m;
        uint4 a = __ldg(wi + e0);
        uint4 b = e1 != e0 ? __ldg(wi + e1) : a;
        start = a.x;
        len = b.y > a.x ? b.y - a.x : 0;
        fb = a.z;
        nb = (len && b.w > a.z) ? b.w - a.z : 0;
      }
      s_rng[4 * tid + 0] = start;
      s_rng[4 * tid + 1] = len;
      s_tblk[2 * tid] = fb;        // first block ordinal (rewritten to the global block base below)
      s_tblk[2 * tid + 1] = nb;
    }
    if (tid == 0) { s_misc[2] = 0; s_misc[3] = 0; }
    for (uint32_t s = 0; s < n_fn; s++) {
      if (P.fn_off[s] == ~0ull) continue;
      const uint8_t* src = base + P.fn_off[s] + ws;
      uint8_t* dst = sm.u8(p.sm.fn[s]);
      const uint32_t n16 = min(W, (wlen + 15u) & ~15u) >> 4;  // the array is padded by 16 bytes only
      for (uint32_t i = tid; i < n16; i += QW_THREADS) cp_async16(dst + 16 * i, src + 16 * i);
    }
    __syncthreads();
    // ---- phase 2: stage offsets + global block numbering (one thread), then, in ONE round of loads,
    // cp.async the packed posting bytes and read the skip entries that describe each staged block ------
    if (tid == 0) {
      uint32_t off = 0, g = 0, n_direct = 0;
      for (uint32_t t = 0; t < n_terms; t++) {
        const uint32_t len = s_rng[4 * t + 1], nb = s_tblk[2 * t + 1];
        if (len && off + len <= p.stage_bytes && nb <= QW_BLK_TAB && g + nb <= QW_MAX_WBLK) {
          s_rng[4 * t + 2] = off;
          off += len;
          s_misc[8 + t] = g;  // global block base of term slot t
          g += nb;
        } else {
          s_rng[4 * t + 2] = 0xFFFFFFFFu;  // direct mode (or nothing to do)
          s_misc[8 + t] = g;
          if (len) n_direct++;
        }
      }
      s_misc[0] = g;
      s_misc[6] = n_direct;  // terms of this window that are decoded from global memory
    }
    __syncthreads();
    for (uint32_t t = warp; t < n_terms; t += QW_WARPS) {
      const uint32_t so = s_rng[4 * t + 2];
      if (so == 0xFFFFFFFFu) continue;
      const DInstr& in = s_instr[s_tinstr[t]];
      const uint32_t start = s_rng[4 * t + 0];
      const uint8_t* src = base + in.a + start;
      const uint32_t n16 = s_rng[4 * t + 1] >> 4;
      for (uint32_t i = lane; i < n16; i += 32) cp_async16(s_stage + so + 16 * i, src + 16 * i);
      // block records straight from the skip list (coalesced 16-byte entries)
      const uint4* skips = (const uint4*)(base + in.c) + s_tblk[2 * t];
      const uint32_t nb = s_tblk[2 * t + 1], g0 = s_misc[8 + t];
      for (uint32_t k = lane; k < nb; k += 32) {
        const uint4 h = __ldg(skips + k);  // last_doc, prev_last_doc, byte_off, widths/count
        BlkRec r;
        r.soff = (uint16_t)(so + (h.z - start));
        r.slot = (uint8_t)t;
        r.pad = 0;
        const uint32_t first_lb = h.y + 1;  // lower bound of the first doc (0 when h.y == 0xFFFFFFFF)
        r.lo = (uint16_t)(first_lb <= ws ? 0u : min(first_lb - ws, W));
        r.hi = (uint16_t)(h.x < ws ? 0xFFFFu : min(h.x - ws, W - 1));
        if (h.x < ws || first_lb >= we) { r.lo = (uint16_t)W; r.hi = 0; }  // no overlap: lo > hi
        s_blk[g0 + k] = r;
      }
    }
    cp_async_wait_all();
    __syncthreads();
    if (tid < n_terms) s_tblk[2 * tid] = s_misc[8 + tid];  // from here on: global block base
    __syncthreads();

    // ---- execute the boolean program (block-wide; one barrier per clause keeps the f32 order fixed) ----
    // A TERM clause folds its staged posting blocks directly into the level's bitmaps / score array,
    // one block per warp per step (fold_block); clauses whose range was not staged decode from global
    // memory (direct mode).
    uint32_t ip = 0;
    uint32_t req_init = 0;  // bit per level, uniform across the block
    // fused BM25 shape (COLLECT pass only): matches / hit count come from the score array, which the
    // collect loop also re-zeroes for the next window of the same split plan
    constexpr bool fused = UNION;
    {
      while (ip < n_instr) {
        const DInstr& in = s_instr[ip];
        const uint32_t op = in.op, level = in.level, occur = in.occur;
        const SmemLevel& LV = p.sm.lvl[level];
        const bool scored = (in.flags & IF_SCORED) != 0;
        if (UNION && op == OP_BOOL_BEGIN) {
          if (!ssum_clean) zero_f4(sm.f32(LV.ssum), W, tid);
          if (tid == 0) s_misc[5] = 0;  // ticket: posting blocks applied so far
          __syncthreads();
          ip++;
          if (s_misc[6] == 0) {
            // Every term of the window is staged: run the whole union as ONE pipelined pass over the
            // flat block table (blocks are numbered in clause order). A warp decodes its next block
            // right away and only the read-modify-write of the accumulator waits until every block of
            // the EARLIER clauses has been applied (ticket counter) — the f32 sums keep the reference's
            // clause order, but there is no block-wide barrier per clause and no warp idles while a
            // short clause finishes. Blocks of one clause touch distinct docs, so they commute.
            const uint32_t G = s_misc[0];
            // (measured and rejected: a spare warp prefetching the next window's bytes into L2 made the
            // kernel 4-5 % slower — the staging phases are not DRAM-latency bound enough to pay for it)
            volatile uint32_t* ticket = (volatile uint32_t*)&s_misc[5];
            float* score = sm.f32(LV.ssum);
            // (static round-robin assignment; handing blocks out from a shared counter measured slower)
            for (uint32_t g = warp; g < G; g += QW_WARPS) {
              const BlkRec r = s_blk[g];
              const DInstr& ti = s_instr[s_tinstr[r.slot]];
              TermTarget tg;
              tg.bits = 0xFFFFFFFFu;
              tg.cnt = 0xFFFFFFFFu;
              tg.score = LV.ssum;
              tg.weight = ti.f;
              tg.has_tf = (ti.flags & IF_HAS_TF) != 0;
              tg.fn = (ti.flags & IF_HAS_FN) ? p.sm.fn[ti.r] : 0xFFFFFFFFu;
              tg.gtab = (const float*)P.bm25_tab[ti.r];
              uint32_t rel[4], inmask;
              float contrib[4];
              union_decode(p.sm.stage + r.soff, ws, wlen, tg, lane, rel, contrib, inmask);
              const uint32_t need = s_tblk[2 * r.slot];  // first block of this clause = blocks of earlier clauses
              if (need) {
                if (lane == 0) {
                  while (*ticket < need) __nanosleep(20);
                  __threadfence_block();
                }
                __syncwarp();
              }
              float old[4];
#pragma unroll
              for (int j = 0; j < 4; j++) old[j] = ((inmask >> j) & 1) ? score[rel[j]] : 0.0f;
#pragma unroll
              for (int j = 0; j < 4; j++) if ((inmask >> j) & 1) score[rel[j]] = __fadd_rn(old[j], contrib[j]);
              __syncwarp();
              if (lane == 0) {
                __threadfence_block();
                atomicAdd(&s_misc[5], 1u);
              }
            }
            __syncthreads();
            ip = n_instr;  // the TERM / BOOL_END instructions are done
          }
        } else if (UNION && op == OP_BOOL_END) {
          ip++;
        } else if (UNION) {  // OP_TERM, should + scored, bitmap implied by the score
          const uint32_t slot = in.t;
          TermTarget tg;
          tg.bits = 0xFFFFFFFFu;
          tg.cnt = 0xFFFFFFFFu;
          tg.score = LV.ssum;
          tg.weight = in.f;
          tg.has_tf = (in.flags & IF_HAS_TF) != 0;
          tg.fn = (in.flags & IF_HAS_FN) ? p.sm.fn[in.r] : 0xFFFFFFFFu;
          tg.gtab = (const float*)P.bm25_tab[in.r];
          if (s_rng[4 * slot + 2] != 0xFFFFFFFFu) {
            const uint32_t g0 = s_tblk[2 * slot], nb = s_tblk[2 * slot + 1];
            for (uint32_t k = warp; k < nb; k += QW_WARPS) fold_block<true, false, true, false>(p.sm.stage + s_blk[g0 + k].soff, nullptr, ws, 0, wlen, tg, lane);
          } else if (s_rng[4 * slot + 1]) {
            const QwSkip* skips = (const QwSkip*)(base + in.c);
            const uint32_t bfirst = first_block_ge(skips, in.n, ws, lane);
            const uint8_t* tdata = base + in.a;
            for (uint32_t bb = bfirst + warp; bb < in.n; bb += QW_WARPS) {
              uint4 h = __ldg((const uint4*)&skips[bb]);
              if (h.y != QW_NO_PREV_DOC && h.y + 1 >= we) break;
              fold_block<true, false, false, false>(0, tdata + h.z, ws, 0, wlen, tg, lane);
            }
          }
          __syncthreads();
          ip++;
        } else if (op == OP_BOOL_BEGIN) {
          zero_f4((float*)sm.u32(LV.shd), NW, tid);
          zero_f4((float*)sm.u32(LV.nt), NW, tid);
          if (LV.cnt != 0xFFFFFFFFu) zero_f4((float*)sm.u32(LV.cnt), W >> 2, tid);
          if (LV.msum != 0xFFFFFFFFu) zero_f4(sm.f32(LV.msum), W, tid);
          if (LV.ssum != 0xFFFFFFFFu && !(fused && level == 0 && ssum_clean)) zero_f4(sm.f32(LV.ssum), W, tid);
          req_init &= ~(1u << level);
          __syncthreads();
          ip++;
        } else if (op == OP_TERM || op == OP_PHRASE) {
          const bool required = occur == QW_OCCUR_MUST || occur == QW_OCCUR_FILTER;
          const uint32_t slot = in.t;
          const bool from_score = (in.flags & IF_BITS_FROM_SCORE) != 0;  // bitmap derived at BOOL_END
          TermTarget tg;
          tg.cnt = 0xFFFFFFFFu;
          tg.score = 0xFFFFFFFFu;
          if (required) {
            tg.bits = p.sm.tmp;
            zero_f4((float*)sm.u32(p.sm.tmp), NW, tid);
            if (scored) tg.score = LV.msum;
            __syncthreads();
          } else if (occur == QW_OCCUR_SHOULD) {
            tg.bits = LV.shd;
            tg.cnt = LV.cnt;
            if (scored) tg.score = LV.ssum;
          } else tg.bits = LV.nt;
          tg.weight = in.f;
          tg.has_tf = (in.flags & IF_HAS_TF) != 0;
          tg.fn = (scored && (in.flags & IF_HAS_FN)) ? p.sm.fn[in.r] : 0xFFFFFFFFu;
          tg.gtab = scored ? (const float*)P.bm25_tab[in.r] : nullptr;
          if (op == OP_PHRASE) {
            // blocks of the phrase's posting list = blocks of its driver term: found through that term's skip list
            const QwSkip* skips = (const QwSkip*)(base + in.c);
            const VBlk* vblks = (const VBlk*)in.a;
            const uint32_t nblk = in.n;
            const uint32_t bfirst = first_block_ge(skips, nblk, ws, lane);
            for (uint32_t bb = bfirst + warp; bb < nblk; bb += QW_WARPS) {
              const uint32_t prev = __ldg(&skips[bb].prev_last_doc);
              if (prev != QW_NO_PREV_DOC && prev + 1 >= we) break;
              fold_vblock(vblks + bb, ws, wlen, tg, lane);
            }
          } else if (s_rng[4 * slot + 2] != 0xFFFFFFFFu) {
            const uint32_t g0 = s_tblk[2 * slot], nb = s_tblk[2 * slot + 1];
            const bool sc = tg.score != 0xFFFFFFFFu, cn = tg.cnt != 0xFFFFFFFFu;
            if (sc && !cn && from_score) { for (uint32_t k = warp; k < nb; k += QW_WARPS) fold_block<true, false, true, false>(p.sm.stage + s_blk[g0 + k].soff, nullptr, ws, 0, wlen, tg, lane); }
            else if (sc && !cn) { for (uint32_t k = warp; k < nb; k += QW_WARPS) fold_block<true, false, true, true>(p.sm.stage + s_blk[g0 + k].soff, nullptr, ws, 0, wlen, tg, lane); }
            else if (!sc && !cn) { for (uint32_t k = warp; k < nb; k += QW_WARPS) fold_block<false, false, true, true>(p.sm.stage + s_blk[g0 + k].soff, nullptr, ws, 0, wlen, tg, lane); }
            else { for (uint32_t k = warp; k < nb; k += QW_WARPS) fold_block_dyn<true>(p.sm.stage + s_blk[g0 + k].soff, nullptr, ws, 0, wlen, tg, lane); }
          } else if (s_rng[4 * slot + 1]) {
            // direct mode (range not staged): warps decode whole blocks straight from global memory
            const QwSkip* skips = (const QwSkip*)(base + in.c);
            const uint32_t nblk = in.n;
            const uint32_t bfirst = first_block_ge(skips, nblk, ws, lane);
            const uint8_t* tdata = base + in.a;
            for (uint32_t bb = bfirst + warp; bb < nblk; bb += QW_WARPS) {
              uint4 h = __ldg((const uint4*)&skips[bb]);
              if (h.y != QW_NO_PREV_DOC && h.y + 1 >= we) break;
              fold_block_dyn<false>(0, tdata + h.z, ws, 0, wlen, tg, lane);
            }
          }
          __syncthreads();
          if (required) {
            uint32_t* req = sm.u32(LV.req);
            const uint32_t* tmp = sm.u32(p.sm.tmp);
            const bool init = (req_init >> level) & 1;
            for (uint32_t i = tid; i < NW; i += QW_THREADS) req[i] = init ? (req[i] & tmp[i]) : tmp[i];
            req_init |= 1u << level;
            __syncthreads();
          }
          ip++;
      } else if (op == OP_RANGE || op == OP_EXISTS || op == OP_ALL) {
        const bool required = occur == QW_OCCUR_MUST || occur == QW_OCCUR_FILTER;
        const bool init = (req_init >> level) & 1;
        const bool gather = required && init;
        uint32_t* req = sm.u32(LV.req);
        const uint32_t col = in.r;
        const bool has_col = op == OP_ALL || col != 0xFFFFFFFFu;
        const uint64_t lo = in.a, hi = in.b;
        const float boost = in.f;
        if (gather && op != OP_ALL && p.sm.rangeq != 0xFFFFFFFFu) {
          // required clause over an already narrowed candidate set: probe only the surviving docs,
          // 32 per warp step (compacted), and clear the bits of those that fail
          uint16_t* rq = (uint16_t*)sm.u8(p.sm.rangeq) + warp * QW_HITQ_CAP;
          warp_for_hits(req, NW, warp, lane, rq, [&](uint32_t i, bool on) {
            bool hit = false;
            if (on && has_col) {
              const DCol& c = s_cols[col];
              uint64_t a, b;
              col_range(base, c, ws + i, a, b);
              if (op == OP_EXISTS) hit = a != b;
              else for (uint64_t k = a; k < b && !hit; k++) {
                uint64_t mv = c.min_value + c.gcd * col_raw(base, c, k);
                hit = mv >= lo && mv <= hi;
              }
            }
            if (on && !hit) atomicAnd(&req[i >> 5], ~(1u << (i & 31)));
            if (hit && scored) sm.f32(LV.msum)[i] = __fadd_rn(sm.f32(LV.msum)[i], boost);
          });
        } else
        for (uint32_t wd = warp; wd < NW; wd += QW_WARPS) {
          const uint32_t d = ws + wd * 32 + lane;
          bool cand = d < we && has_col;
          if (gather) {
            const uint32_t rw = req[wd];
            if (rw == 0) continue;  // warp-uniform
            cand = cand && ((rw >> lane) & 1);
          }
          bool hit = false;
          if (cand) {
            if (op == OP_ALL) hit = true;
            else {
              const DCol& c = s_cols[col];
              uint64_t a, b;
              col_range(base, c, d, a, b);
              if (op == OP_EXISTS) hit = a != b;
              else for (uint64_t i = a; i < b && !hit; i++) {
                uint64_t mv = c.min_value + c.gcd * col_raw(base, c, i);
                hit = mv >= lo && mv <= hi;
              }
            }
          }
          const uint32_t word = __ballot_sync(0xFFFFFFFFu, hit);
          const uint32_t di = wd * 32 + lane;
          if (required) {
            if (lane == 0) req[wd] = init ? (req[wd] & word) : word;
            if (hit && scored) sm.f32(LV.msum)[di] = __fadd_rn(sm.f32(LV.msum)[di], boost);
          } else if (occur == QW_OCCUR_SHOULD) {
            if (lane == 0) sm.u32(LV.shd)[wd] |= word;
            if (hit && LV.cnt != 0xFFFFFFFFu) sm.u8(LV.cnt)[di]++;
            if (hit && scored) sm.f32(LV.ssum)[di] = __fadd_rn(sm.f32(LV.ssum)[di], boost);
          } else {
            if (lane == 0) sm.u32(LV.nt)[wd] |= word;
          }
        }
        if (required) req_init |= 1u << level;
        __syncthreads();
        ip++;
      } else if (op == OP_BOOL_END) {
        // BooleanWeight combination: all required AND NOT any excluded AND >= r should clauses
        uint32_t* req = sm.u32(LV.req);
        const uint32_t need = in.r, n_req = in.n;
        if ((in.flags & IF_BITS_FROM_SCORE) && !(fused && level == 0)) {
          // every contribution of the flagged should-terms is > 0, so "matched some of them" == (ssum > 0)
          const float* ss = sm.f32(LV.ssum);
          uint32_t* shd = sm.u32(LV.shd);
          for (uint32_t wd = warp; wd < NW; wd += QW_WARPS) {
            const uint32_t m = __ballot_sync(0xFFFFFFFFu, ss[wd * 32 + lane] > 0.0f);
            if (lane == 0) shd[wd] |= m;
          }
          __syncthreads();
        }
        for (uint32_t wd = tid; wd < NW; wd += QW_THREADS) {
          const uint32_t d0 = ws + wd * 32;
          uint32_t valid = d0 >= we ? 0u : (we - d0 >= 32 ? 0xFFFFFFFFu : ((1u << (we - d0)) - 1));
          uint32_t r = n_req ? (((req_init >> level) & 1) ? req[wd] : 0u) : 0xFFFFFFFFu;
          uint32_t so;
          if (need == 0) so = 0xFFFFFFFFu;
          else if (need == 1) so = sm.u32(LV.shd)[wd];
          else {
            so = 0;
            const uint8_t* cnt = sm.u8(LV.cnt) + wd * 32;
            for (uint32_t b = 0; b < 32; b++) so |= (cnt[b] >= need ? 1u : 0u) << b;
          }
          req[wd] = r & so & ~sm.u32(LV.nt)[wd] & valid;
        }
        if (LV.msum != 0xFFFFFFFFu && LV.ssum != 0xFFFFFFFFu) {
          float4* ms = (float4*)sm.f32(LV.msum);
          const float4* ss = (const float4*)sm.f32(LV.ssum);
          for (uint32_t i = tid; i < (W >> 2); i += QW_THREADS) {
            float4 a = ms[i], b = ss[i];
            a.x = __fadd_rn(a.x, b.x); a.y = __fadd_rn(a.y, b.y); a.z = __fadd_rn(a.z, b.z); a.w = __fadd_rn(a.w, b.w);
            ms[i] = a;
          }
        }
        __syncthreads();
        if (level > 0) {
          // fold this bool's (bits, score) into the parent level as one clause
          const SmemLevel& PL = p.sm.lvl[level - 1];
          const uint32_t plevel = level - 1;
          const bool required = occur == QW_OCCUR_MUST || occur == QW_OCCUR_FILTER;
          const bool pinit = (req_init >> plevel) & 1;
          const float* csc = LV.rsc != 0xFFFFFFFFu ? sm.f32(LV.rsc) : nullptr;
          for (uint32_t wd = tid; wd < NW; wd += QW_THREADS) {
            uint32_t m = req[wd];
            if (required) sm.u32(PL.req)[wd] = pinit ? (sm.u32(PL.req)[wd] & m) : m;
            else if (occur == QW_OCCUR_SHOULD) sm.u32(PL.shd)[wd] |= m;
            else sm.u32(PL.nt)[wd] |= m;
          }
          if (occur == QW_OCCUR_SHOULD && (PL.cnt != 0xFFFFFFFFu || (scored && csc))) {
            for (uint32_t i = tid; i < W; i += QW_THREADS) {
              if ((req[i >> 5] >> (i & 31)) & 1) {
                if (PL.cnt != 0xFFFFFFFFu) sm.u8(PL.cnt)[i]++;
                if (scored && csc) sm.f32(PL.ssum)[i] = __fadd_rn(sm.f32(PL.ssum)[i], csc[i]);
              }
            }
          } else if (occur == QW_OCCUR_MUST && scored && csc) {
            for (uint32_t i = tid; i < W; i += QW_THREADS) sm.f32(PL.msum)[i] = __fadd_rn(sm.f32(PL.msum)[i], csc[i]);
          }
          if (required) req_init |= 1u << plevel;
          __syncthreads();
        }
        ip++;
      }
      }  // while ip
    }


    // ---- collect the window's matches ---------------------------------------------------------------
    const uint32_t* res = sm.u32(p.sm.lvl[0].req);
    const float* rscore = p.sm.lvl[0].rsc != 0xFFFFFFFFu ? sm.f32(p.sm.lvl[0].rsc) : nullptr;
    const DThresh& T = p.thresh[split];
    const uint32_t max_hits = P.max_hits, sa_present = P.sa.present;
    const uint32_t n_aggs = (MODE == MODE_COLLECT && p.cands_only) ? 0u : P.n_aggs;
    QwAggCell* cells = (QwAggCell*)P.out_cells;
    const bool rec = MODE == MODE_COLLECT && p.rec_l0 && max_hits && !fused;
    const bool fast_aggs = P.fast_aggs && p.smem_aggs;
    uint32_t* s_l0 = sm.u32(p.sm.l0hist);
    if (MODE == MODE_HIST || (p.smem_aggs && n_aggs) || rec) {
      // the histogram / privatised aggregation counters alias the (now dead) staging area
      for (uint32_t i = tid; i < (MODE == MODE_HIST ? (uint32_t)QW_HIST_BINS : P.n_cells); i += QW_THREADS) s_hist[i] = 0;
      if (rec) for (uint32_t i = tid; i < QW_HIST_BINS; i += QW_THREADS) s_l0[i] = 0;
      if (fast_aggs && n_aggs && P.n_stat_cells) {
        unsigned long long* st = (unsigned long long*)(sm.u8(p.sm.hist) + ((P.n_cells * 4u + 7u) & ~7u));
        for (uint32_t i = tid; i < 3 * P.n_stat_cells; i += QW_THREADS) st[i] = 0ull;
      }
      if (tid == 0) s_misc[4] = 0;
      __syncthreads();
    }
    if (MODE == MODE_COLLECT) {
      const Key thr{T.key[0], T.key[1], T.key[2]};
      const uint32_t thr_top = (uint32_t)(thr.w0 >> 53);
      uint32_t my_hits = 0, my_elig = 0, my_top = 0;
      // hit count: one popc per bitmap word
      if (!fused && !p.cands_only) for (uint32_t wd = tid; wd < NW; wd += QW_THREADS) my_hits += __popc(res[wd]);
      auto emit = [&](const Key& k) {
        const uint32_t pos = atomicAdd((uint32_t*)P.out_cand_count, 1u);
        if (pos < QW_CAND_CAP) {
          uint64_t* c = (uint64_t*)P.out_cands + 3ull * pos;
          c[0] = k.w0; c[1] = k.w1; c[2] = k.w2;
        }
      };
      auto slow_path = [&](uint32_t i, float sc) {
        DocKey dk = doc_key(P, ks, s_cols, base, ws + i, sc);
        if (dk.eligible) {
          my_elig++;
          if (key_ge(dk.key, thr)) emit(dk.key);
        }
      };
      if (fused) {
        // fused BM25 pass: one sweep over the score array counts the matches (score > 0), filters them
        // against the float lower bound of the threshold bucket and clears the array for the next window
        float s_lo = -1.0f;
        if (thr_top >= 1024u) s_lo = __fmul_rn(__fdiv_rn((float)(thr_top & 1023u), ks.score_scale), 0.999999f);
        float4* sc4 = reinterpret_cast<float4*>(sm.f32(p.sm.lvl[0].ssum));
        my_hits = 0;
        for (uint32_t q = tid; q < (W >> 2); q += QW_THREADS) {
          const float4 v = sc4[q];
          sc4[q] = make_float4(0.f, 0.f, 0.f, 0.f);
          my_hits += (v.x > 0.0f) + (v.y > 0.0f) + (v.z > 0.0f) + (v.w > 0.0f);
          if (v.x > 0.0f && v.x >= s_lo) slow_path(4 * q + 0, v.x);
          if (v.y > 0.0f && v.y >= s_lo) slow_path(4 * q + 1, v.y);
          if (v.z > 0.0f && v.z >= s_lo) slow_path(4 * q + 2, v.z);
          if (v.w > 0.0f && v.w >= s_lo) slow_path(4 * q + 3, v.w);
        }
        if (p.cands_only) my_hits = 0;
        ssum_clean = true;
      } else if (max_hits && ks.kind[0] == QW_SORT_SCORE && ks.order[0] == QW_ORDER_DESC && !sa_present && rscore && !n_aggs && !rec) {
        // fast path (BM25 top-K): a float lower bound of the threshold bucket filters 4 docs per lane
        // per step; only survivors build the composite key. s_lo is conservative (one part in 2^20).
        float s_lo = -1.0f;
        if (thr_top >= 1024u) s_lo = __fmul_rn(__fdiv_rn((float)(thr_top & 1023u), ks.score_scale), 0.999999f);
        const float4* sc4 = reinterpret_cast<const float4*>(rscore);
        for (uint32_t q = tid; q < (W >> 2); q += QW_THREADS) {
          const uint32_t nib = (res[q >> 3] >> ((q & 7) * 4)) & 0xFu;
          if (!nib) continue;
          const float4 v = sc4[q];
          if ((nib & 1u) && v.x >= s_lo) slow_path(4 * q + 0, v.x);
          if ((nib & 2u) && v.y >= s_lo) slow_path(4 * q + 1, v.y);
          if ((nib & 4u) && v.z >= s_lo) slow_path(4 * q + 2, v.z);
          if ((nib & 8u) && v.w >= s_lo) slow_path(4 * q + 3, v.w);
        }
      } else if (max_hits || n_aggs) {
        // generic path, warp-converged over compacted hits: lane = one matched doc
        warp_for_hits(res, NW, warp, lane, s_hitq, [&](uint32_t i, bool on) {
          const uint32_t doc = ws + i;
          if (max_hits) {
            const float sc = (on && rscore) ? rscore[i] : 0.0f;
            uint32_t top = 0;
            bool ranked = false;  // eligible for the top-K (search_after may exclude matches)
            if (on) {
              if (sa_present) {
                const DocKey dk = doc_key(P, ks, s_cols, base, doc, sc);
                if (dk.eligible) {
                  ranked = true;
                  my_elig++;
                  top = (uint32_t)(dk.key.w0 >> 53);
                  if (key_ge(dk.key, thr)) emit(dk.key);
                }
              } else {
                // cheap pre-filter on the key's first 11 bits; the composite key is only built for docs
                // that can reach the threshold
                ranked = true;
                top = key_top11(P, ks, s_cols, base, doc, sc);
                if (top >= thr_top) {
                  const DocKey dk = doc_key(P, ks, s_cols, base, doc, sc);
                  if (key_ge(dk.key, thr)) emit(dk.key);
                }
              }
            }
            if (rec) {
              warp_count_uniform(s_l0, top, ranked, lane);
              if (ranked) my_top = max(my_top, top + 1);
            }
          }
          if (n_aggs) {
            if (fast_aggs) agg_collect_fast(sm, P, s_aggs, s_cols, base, doc, on, lane);
            else agg_collect_doc(p, sm, P, s_aggs, s_cols, base, cells, doc, on, lane);
          }
        });
        if (!sa_present) my_elig = 0;
      }
      // block-reduce the counters, one global atomic per window
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        my_elig += __shfl_down_sync(0xFFFFFFFFu, my_elig, o);
        my_hits += __shfl_down_sync(0xFFFFFFFFu, my_hits, o);
      }
      if (rec) my_top = __reduce_max_sync(0xFFFFFFFFu, my_top);
      if (lane == 0) {
        if (my_hits) atomicAdd(&s_misc[2], my_hits);
        if (my_elig) atomicAdd(&s_misc[3], my_elig);
        if (rec && my_top) atomicMax(&s_misc[4], my_top);
      }
      __syncthreads();
      if (tid == 0 && !p.cands_only) {
        const uint32_t hits = s_misc[2];
        if (hits) atomicAdd((unsigned long long*)P.out_num_hits, (unsigned long long)hits);
        // without search_after every hit is eligible
        const uint32_t elig = sa_present ? s_misc[3] : (max_hits ? hits : 0);
        if (elig) atomicAdd((unsigned long long*)P.out_num_hits + 1, (unsigned long long)elig);
        if (rec) p.wmax[work] = (uint16_t)s_misc[4];
      }
      if (fast_aggs && n_aggs && P.n_stat_cells) {
        // privatised stats: one set of global atomics per touched cell and window; the cell's value
        // count is its bucket's doc count (the column is single-valued and always present)
        const unsigned long long* st = (const unsigned long long*)(sm.u8(p.sm.hist) + ((P.n_cells * 4u + 7u) & ~7u));
        for (uint32_t gi = 0; gi < P.n_aggs; gi++) {
          const DAgg& g = s_aggs[gi];
          if (g.kind != QW_AGG_STATS) continue;
          const bool top = g.parent == 0xFFFFFFFFu;
          const uint32_t nc = top ? 1u : s_aggs[g.parent].num_buckets;
          const bool is_f64 = g.is_f64;
          for (uint32_t c = tid; c < nc; c += QW_THREADS) {
            const uint32_t cnt = top ? s_misc[2] : s_hist[s_aggs[g.parent].cell_base + c];
            if (!cnt) continue;
            const unsigned long long* t = st + 3ull * (g.stat_base + c);
            QwAggCell* out = &cells[g.cell_base + c];
            atomicAdd((unsigned long long*)&out->count, (unsigned long long)cnt);
            if (is_f64) atomicAdd((double*)&out->sum_bits, __longlong_as_double((long long)t[0]));
            else atomicAdd((unsigned long long*)&out->sum_bits, t[0]);
            atomicMax((unsigned long long*)&out->min_mapped, t[1]);
            atomicMax((unsigned long long*)&out->max_mapped, t[2]);
          }
        }
        __syncthreads();  // the bucket counts read above are cleared below
      }
      if (p.smem_aggs && n_aggs) {
        for (uint32_t i = tid; i < P.n_cells; i += QW_THREADS) {
          uint32_t v = s_hist[i];
          if (v) { atomicAdd((unsigned long long*)&cells[i].count, (unsigned long long)v); s_hist[i] = 0; }
        }
      }
      if (rec) {
        uint32_t* gh = (uint32_t*)P.out_hist;
        for (uint32_t i = tid; i < QW_HIST_BINS; i += QW_THREADS) {
          const uint32_t v = s_l0[i];
          if (v) atomicAdd(&gh[i], v);
        }
      }
    } else {
      if (UNION) {
        // level-0 histogram of a BM25 union straight from the score array (digit = [1 | lin:10]);
        // the sweep also clears the array for the next window
        float4* sc4 = reinterpret_cast<float4*>(sm.f32(p.sm.lvl[0].ssum));
        for (uint32_t q = tid; q < (W >> 2); q += QW_THREADS) {
          const float4 v = sc4[q];
          sc4[q] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (v.x > 0.0f) atomicAdd(&s_hist[1024u | score_lin(ks, v.x, true)], 1u);
          if (v.y > 0.0f) atomicAdd(&s_hist[1024u | score_lin(ks, v.y, true)], 1u);
          if (v.z > 0.0f) atomicAdd(&s_hist[1024u | score_lin(ks, v.z, true)], 1u);
          if (v.w > 0.0f) atomicAdd(&s_hist[1024u | score_lin(ks, v.w, true)], 1u);
        }
        ssum_clean = true;
      } else if (max_hits) {
        warp_for_hits(res, NW, warp, lane, s_hitq, [&](uint32_t i, bool on) {
          const uint32_t doc = ws + i;
          const float sc = (on && rscore) ? rscore[i] : 0.0f;
          uint32_t digit = 0;
          bool ranked = false;
          if (on) {
            if (p.level == 0 && !sa_present) {
              digit = key_top11(P, ks, s_cols, base, doc, sc);
              ranked = true;
            } else {
              const DocKey dk = doc_key(P, ks, s_cols, base, doc, sc);
              ranked = dk.eligible && (!p.use_prefix || key_prefix_eq(dk.key, T.key, T.prefix_bits));
              digit = key_digit(dk.key, p.level);
            }
          }
          warp_count_uniform(s_hist, digit, ranked, lane);
        });
      }
      __syncthreads();
      uint32_t* gh = (uint32_t*)P.out_hist;
      for (uint32_t i = tid; i < QW_HIST_BINS; i += QW_THREADS) {
        uint32_t v = s_hist[i];
        if (v) { atomicAdd(&gh[i], v * hist_weight); s_hist[i] = 0; }
      }
    }
  }
}

// Picks the radix digit of the top-K threshold from a split's histogram.
//   sampled != 0: histogram comes from every `stride`-th window; pick the digit at a conservative
//                 sample rank `k_sample` (verified afterwards against the true candidate count).
//   sampled == 0: exact radix-select step at `level` (prefix / above bookkeeping in DThresh).
//   split_state != null: only splits flagged for refinement are touched, and their candidate
//                 counters are reset for the candidates-only collect pass that follows.
__global__ void __launch_bounds__(256) k_pick(const DSplitPlan* plans, DThresh* thresh, uint32_t level, uint32_t sampled, uint32_t stride,
                                              const uint32_t* split_state) {
  __shared__ uint32_t s_part[256];
  __shared__ uint32_t s_sel[2];
  const uint32_t split = blockIdx.x, tid = threadIdx.x;
  const DSplitPlan& P = plans[split];
  DThresh& T = thresh[split];
  if (P.max_hits == 0 || (split_state && split_state[split] == 0)) return;
  if (split_state && tid == 0) *(uint32_t*)P.out_cand_count = 0;
  if (!sampled && level > 0 && T.done) return;
  const uint32_t* h = (const uint32_t*)P.out_hist;
  // thread t owns the 8 bins [2048 - 8(t+1), 2048 - 8t), i.e. thread 0 owns the top bins
  const uint32_t hi = QW_HIST_BINS - 8 * tid;
  uint32_t loc[8], sum = 0;
#pragma unroll
  for (int j = 0; j < 8; j++) { loc[j] = h[hi - 1 - j]; sum += loc[j]; }
  // exclusive prefix over threads (bins above mine): warp scan + the totals of the warps before mine
  uint32_t incl = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, o); if ((int)(tid & 31) >= o) incl += t; }
  if ((tid & 31) == 31) s_part[tid >> 5] = incl;
  if (tid == 0) { s_sel[0] = 0xFFFFFFFFu; s_sel[1] = 0; }
  __syncthreads();
  uint32_t above_me = incl - sum, total_all = 0;
#pragma unroll
  for (uint32_t w = 0; w < 8; w++) { const uint32_t t = s_part[w]; total_all += t; if (w < (tid >> 5)) above_me += t; }
  uint32_t K = P.max_hits;
  uint32_t target, base_above = 0;
  if (sampled == 2) {
    // weighted sample (counts are estimates of the true counts): twice K plus the same slack in windows
    target = 2 * K + 24 * stride;
  } else if (sampled) {
    // conservative sample rank: 2x the expected sample share of K plus slack
    target = (2 * K + stride - 1) / stride + 24;
  } else {
    base_above = level == 0 ? 0u : T.above;
    target = K > base_above ? K - base_above : 1;
  }
  // find the largest digit t with suffix(t) >= target
  uint32_t run = above_me;
#pragma unroll
  for (int j = 0; j < 8; j++) {
    uint32_t before = run;
    run += loc[j];
    if (before < target && run >= target) { s_sel[0] = hi - 1 - j; s_sel[1] = before; }
  }
  __syncthreads();
  if (tid == 0) {
    uint32_t digit = s_sel[0];
    const uint32_t total = total_all;
    if (digit == 0xFFFFFFFFu) {
      // fewer than `target` ranked docs: keep everything that matches the current prefix
      T.done = 1;
      T.matched = total;
      if (sampled || level == 0) { T.key[0] = T.key[1] = T.key[2] = 0; T.prefix_bits = 0; T.above = 0; }
      return;
    }
    uint32_t o = level * QW_DIGIT_BITS, word = o >> 6, sh = o & 63;
    uint64_t d = (uint64_t)digit << (64 - QW_DIGIT_BITS);
    if (sampled || level == 0) { T.key[0] = T.key[1] = T.key[2] = 0; }
    T.key[word] |= d >> sh;
    if (sh + QW_DIGIT_BITS > 64 && word < 2) T.key[word + 1] |= d << (64 - sh);
    T.prefix_bits = o + QW_DIGIT_BITS;
    if (sampled) { T.above = 0; T.matched = 0; T.done = 1; }
    else {
      T.above = base_above + s_sel[1];
      T.matched = h[digit];
      T.done = (T.above + T.matched <= QW_CAND_CAP) ? 1 : 0;
    }
  }
}

// Harvest (quickwit-search/src/top_k_collector.rs:404-410, binary_heap.rs:187-193): the best
// min(K, n) candidates of a split, best first, decoded back to QwHit.
//   1. exact radix select (8-bit digits, MSB first) of the K-th largest first key word;
//   2. compaction of the candidates >= that word (all ties kept) — normally ~K of the ~2-3K candidates;
//   3. bitonic sort of the survivors with the full 192-bit comparison (the reference total order).
#define QW_SEL_MAX 2048  /* survivors sorted in shared memory; more ties than this => sort everything */
__global__ void __launch_bounds__(1024) k_select(const DSplitPlan* plans, const DCol* all_cols) {
  const DSplitPlan& P = plans[blockIdx.x];
  const uint32_t tid = threadIdx.x;
  if (P.max_hits == 0) { if (tid == 0) *(uint32_t*)P.out_nhits = 0; return; }
  uint32_t n = *(const uint32_t*)P.out_cand_count;
  if (n > QW_CAND_CAP) n = QW_CAND_CAP;  // overflow is detected by the host (cand_count > cap)
  const uint32_t K = P.max_hits;
  const uint64_t* src = (const uint64_t*)P.out_cands;
  // shared memory: all first words [QW_CAND_CAP], then the compacted survivors (3 x sort capacity)
  uint64_t* a0 = (uint64_t*)qw_smem;
  __shared__ uint32_t s_hist[256];
  __shared__ uint32_t s_sel[4];  // [0] digit, [1] count above digit, [2] survivor counter, [3] count in the digit's bin
  for (uint32_t i = tid; i < n; i += 1024) a0[i] = src[3ull * i];
  if (tid == 0) s_sel[2] = 0;
  __syncthreads();
  uint64_t thr = 0;  // keep candidates with w0 >= thr
  if (n > K) {
    uint64_t prefix = 0;
    uint32_t need = K;  // rank of the wanted element among those matching the prefix
    // the sort below pads to a power of two anyway: once the candidates above the current bin plus the bin itself
    // fit that size, the remaining digits need not be resolved (the whole bin is kept)
    uint32_t cap = 32;
    while (cap < K) cap <<= 1;
    for (int shift = 56; shift >= 0; shift -= 8) {
      if (tid < 256) s_hist[tid] = 0;
      __syncthreads();
      const uint64_t himask = shift == 56 ? 0ull : (~0ull << (shift + 8));
      for (uint32_t base = 0; base < n; base += 1024) {
        const uint32_t i = base + tid;
        const uint64_t v = i < n ? a0[i] : 0ull;
        const bool in = i < n && (v & himask) == prefix;
        const uint32_t bin = (uint32_t)(v >> shift) & 255u;
        // candidates near the threshold share their leading digits: one atomic per distinct bin of the warp
        const uint32_t act = __ballot_sync(0xFFFFFFFFu, in);
        if (in) {
          const uint32_t peers = __match_any_sync(act, bin);
          if ((tid & 31) == (uint32_t)__ffs(peers) - 1u) atomicAdd(&s_hist[bin], (uint32_t)__popc(peers));
        }
      }
      __syncthreads();
      if (tid < 32) {
        // lane owns 8 bins, top bins first: lane 0 -> bins 255..248
        uint32_t loc[8], sum = 0;
#pragma unroll
        for (int j = 0; j < 8; j++) { loc[j] = s_hist[255 - (tid * 8 + j)]; sum += loc[j]; }
        uint32_t incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, o); if ((int)tid >= o) incl += t; }
        uint32_t run = incl - sum;
#pragma unroll
        for (int j = 0; j < 8; j++) {
          const uint32_t before = run;
          run += loc[j];
          if (before < need && run >= need) { s_sel[0] = 255 - (tid * 8 + j); s_sel[1] = before; s_sel[3] = loc[j]; }
        }
      }
      __syncthreads();
      prefix |= (uint64_t)s_sel[0] << shift;
      need -= s_sel[1];
      const uint32_t in_bin = s_sel[3];
      __syncthreads();
      if ((K - need) + in_bin <= cap) break;  // (block-uniform: every operand comes from shared memory)
    }
    thr = prefix;  // K-th largest first word with its unresolved low digits cleared: everything >= thr is kept
  }
  // count survivors; too many ties on the first word => sort every candidate instead
  uint32_t mine = 0;
  for (uint32_t i = tid; i < n; i += 1024) mine += a0[i] >= thr;
  for (int o = 16; o > 0; o >>= 1) mine += __shfl_down_sync(0xFFFFFFFFu, mine, o);
  if ((tid & 31) == 0 && mine) atomicAdd(&s_sel[2], mine);
  __syncthreads();
  uint32_t m = s_sel[2];
  const bool all = m > QW_SEL_MAX;
  __syncthreads();
  uint64_t *k0, *k1, *k2;
  uint32_t N = 32;
  if (all) {
    // degenerate: keys live interleaved [w0 | w1 | w2] over the whole candidate set
    m = n;
    while (N < m) N <<= 1;
    k0 = a0; k1 = k0 + N; k2 = k1 + N;
    for (uint32_t i = tid; i < N; i += 1024) {
      if (i < n) { k0[i] = src[3ull * i]; k1[i] = src[3ull * i + 1]; k2[i] = src[3ull * i + 2]; }
      else { k0[i] = 0; k1[i] = 0; k2[i] = 0; }
    }
  } else {
    while (N < m) N <<= 1;
    k0 = a0 + QW_CAND_CAP; k1 = k0 + QW_SEL_MAX; k2 = k1 + QW_SEL_MAX;
    if (tid == 0) s_sel[2] = 0;
    __syncthreads();
    for (uint32_t base = 0; base < n; base += 1024) {
      const uint32_t i = base + tid;
      const uint64_t v = i < n ? a0[i] : 0ull;
      const bool keep = i < n && v >= thr;
      const uint32_t km = __ballot_sync(0xFFFFFFFFu, keep);  // one atomic per warp
      uint32_t wpos = 0;
      if ((tid & 31) == 0 && km) wpos = atomicAdd(&s_sel[2], (uint32_t)__popc(km));
      wpos = __shfl_sync(0xFFFFFFFFu, wpos, 0);
      if (keep) {
        const uint32_t pos = wpos + __popc(km & ((1u << (tid & 31)) - 1u));
        k0[pos] = v; k1[pos] = src[3ull * i + 1]; k2[pos] = src[3ull * i + 2];
      }
    }
    for (uint32_t i = m + tid; i < N; i += 1024) { k0[i] = 0; k1[i] = 0; k2[i] = 0; }
  }
  __syncthreads();
  if (N <= 1024 && !all) {
    // One key per thread, in registers: the compare-exchange partner of thread i at distance `stride` is thread
    // i ^ stride, reached with warp shuffles below 32 and through shared memory (two buffers in turn: one barrier
    // per exchange) from 32 up — 15 barriers for 1024 keys instead of the 55 of the generic network below.
    const bool act = tid < N;
    Key mine{0, 0, 0};
    if (act) mine = Key{k0[tid], k1[tid], k2[tid]};
    uint32_t pb = 1;  // exchange buffer: 1 = the first-word array (dead by now), 0 = the survivor arrays
    __syncthreads();
    for (uint32_t size = 2; size <= N; size <<= 1) {
      for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
        Key other{0, 0, 0};
        if (stride >= 32) {
          uint64_t *b0 = pb ? a0 : k0, *b1 = pb ? a0 + 1024 : k1, *b2 = pb ? a0 + 2048 : k2;
          if (act) { b0[tid] = mine.w0; b1[tid] = mine.w1; b2[tid] = mine.w2; }
          __syncthreads();
          if (act) other = Key{b0[tid ^ stride], b1[tid ^ stride], b2[tid ^ stride]};
          pb ^= 1;
        } else if (act) {
          other.w0 = __shfl_xor_sync(0xFFFFFFFFu, mine.w0, stride);
          other.w1 = __shfl_xor_sync(0xFFFFFFFFu, mine.w1, stride);
          other.w2 = __shfl_xor_sync(0xFFFFFFFFu, mine.w2, stride);
        }
        // descending runs where (i & size) == 0; the lower index of a pair keeps the larger key there
        const bool want_larger = ((tid & stride) == 0) == ((tid & size) == 0);
        if (act && want_larger == key_lt(mine, other)) mine = other;
      }
    }
    __syncthreads();
    if (act) { k0[tid] = mine.w0; k1[tid] = mine.w1; k2[tid] = mine.w2; }
    __syncthreads();
  } else
  for (uint32_t size = 2; size <= N; size <<= 1) {
    for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
      for (uint32_t i = tid; i < (N >> 1); i += 1024) {
        uint32_t pos = 2 * i - (i & (stride - 1));
        uint32_t q = pos + stride;
        bool desc = (pos & size) == 0;
        Key a{k0[pos], k1[pos], k2[pos]}, b{k0[q], k1[q], k2[q]};
        bool a_lt_b = key_lt(a, b);
        bool b_lt_a = key_lt(b, a);
        if (desc ? a_lt_b : b_lt_a) {
          k0[pos] = b.w0; k1[pos] = b.w1; k2[pos] = b.w2;
          k0[q] = a.w0; k1[q] = a.w1; k2[q] = a.w2;
        }
      }
      __syncthreads();
    }
  }
  const uint32_t out_n = m < K ? m : K;
  QwHit* hits = (QwHit*)P.out_hits;
  const DKeySpec& ks = P.key;
  const DCol* cols = all_cols + P.col_base;
  const uint32_t docmask = ks.doc_bits >= 32 ? 0xFFFFFFFFu : ((1u << ks.doc_bits) - 1);
  for (uint32_t i = tid; i < out_n; i += 1024) {
    const Key k{k0[i], k1[i], k2[i]};
    uint32_t pos = 0, has[2];
    uint64_t r[2];
#pragma unroll
    for (int f = 0; f < 2; f++) {
      has[f] = ks.hasbit[f] ? (uint32_t)key_get(k, pos, 1) : 0u;
      pos += ks.hasbit[f];
      r[f] = key_get(k, pos, ks.rbits[f]);
      pos += ks.rbits[f];
    }
    const uint32_t docr = (uint32_t)key_get(k, pos, ks.doc_bits);
    QwHit hh;
    hh.doc_id = ks.order[0] == QW_ORDER_DESC ? docr : docmask - docr;
    hh.flags = has[0] | (has[1] << 1);
    hh.score = 0.0f;
    hh.reserved = 0;
    uint64_t v[2] = {0, 0};
#pragma unroll
    for (int f = 0; f < 2; f++) {
      if (!has[f]) continue;
      const bool desc = ks.order[f] == QW_ORDER_DESC;
      if (ks.kind[f] == QW_SORT_SCORE) {
        uint32_t o = (uint32_t)r[f];
        if (!desc) o = ~o;
        const uint32_t bits = (o & 0x80000000u) ? (o & 0x7FFFFFFFu) : ~o;
        hh.score = __uint_as_float(bits);
        v[f] = f64_to_u64_dev((double)hh.score);
      } else {
        const DCol& c = cols[ks.col[f]];
        v[f] = c.min_value + c.gcd * (desc ? r[f] : ks.raw_max[f] - r[f]);
      }
    }
    hh.v1 = v[0];
    hh.v2 = v[1];
    hits[i] = hh;
  }
  if (tid == 0) *(uint32_t*)P.out_nhits = out_n;
}


// Leaf-level merge on the device (IncrementalCollector / top_k_partial_hits, quickwit-search/src/
// collector.rs:1195-1313, 980-992): the per-split lists written by k_select are sorted best-first; a hit's
// position in the merged order is the number of hits of ALL lists that beat it — its own index plus one
// binary search per other list — so every hit finds its slot independently and the best K land in
// out[0..K) already sorted. Order = PartialHitSortingKey: (sort value 1, sort value 2) in the request's
// directions with None last, then (split id rank, doc id) in the direction of the first key
// (collector.rs:1120-1153); keys are unique, so the ranks are a permutation.
struct MKey {
  uint64_t v1, v2, tie;
  uint32_t has;  // has1 << 1 | has2 (None is last in both directions)
};
__device__ __forceinline__ MKey merge_key(const QwHit& h, uint32_t rank, uint32_t o1, uint32_t o2) {
  MKey k;
  const uint32_t has1 = h.flags & 1u, has2 = (h.flags >> 1) & 1u;
  k.has = has1 << 1 | has2;
  k.v1 = has1 ? (o1 == QW_ORDER_DESC ? h.v1 : ~h.v1) : 0ull;
  k.v2 = has2 ? (o2 == QW_ORDER_DESC ? h.v2 : ~h.v2) : 0ull;
  const uint64_t t = ((uint64_t)rank << 32) | h.doc_id;
  k.tie = o1 == QW_ORDER_DESC ? t : ~t;
  return k;
}
__device__ __forceinline__ bool mkey_gt(const MKey& a, const MKey& b) {  // a beats b
  const uint32_t a1 = a.has >> 1, b1 = b.has >> 1;
  if (a1 != b1) return a1 > b1;
  if (a.v1 != b.v1) return a.v1 > b.v1;
  const uint32_t a2 = a.has & 1u, b2 = b.has & 1u;
  if (a2 != b2) return a2 > b2;
  if (a.v2 != b.v2) return a.v2 > b.v2;
  return a.tie > b.tie;
}
struct DMergedHit {
  QwHit hit;
  uint32_t split, pad;
};
// The lists a merge reads: the per-split lists of one batch (k_select output, tie-break rank per list), or
// the per-rank merged lists gathered over NCCL (DMergedHit records that carry the global split rank).
struct SrcSplits {
  const DSplitPlan* plans;
  const uint32_t* rank;
  uint32_t tag_rank;  // 1: output hits are tagged with the list's (global) rank instead of its index
  __device__ __forceinline__ uint32_t count(uint32_t s) const { return *(const uint32_t*)plans[s].out_nhits; }
  __device__ __forceinline__ QwHit hit(uint32_t s, uint32_t i, uint32_t& rk) const { rk = __ldg(rank + s); return ((const QwHit*)plans[s].out_hits)[i]; }
  __device__ __forceinline__ uint32_t tag(uint32_t s, uint32_t rk) const { return tag_rank ? rk : s; }  // DMergedHit.split of an output hit
};
struct SrcGathered {
  const uint8_t* base;   // rank r: [uint32 n_hits ... header of hdr_bytes][DMergedHit x K]
  uint32_t rec_bytes, hdr_bytes;
  __device__ __forceinline__ uint32_t count(uint32_t s) const { return *(const uint32_t*)(base + (size_t)s * rec_bytes); }
  __device__ __forceinline__ QwHit hit(uint32_t s, uint32_t i, uint32_t& rk) const {
    const DMergedHit* m = (const DMergedHit*)(base + (size_t)s * rec_bytes + hdr_bytes) + i;
    rk = m->split;
    return m->hit;
  }
  __device__ __forceinline__ uint32_t tag(uint32_t, uint32_t rk) const { return rk; }
};

// Pruning before the merge: with m = ceil(K / #lists), every list holds min(m, len) hits that are at least as
// good as its own m-th hit, so if those add up to K the K-th best hit overall is at least as good as the WORST of
// the lists' m-th hits (tau) and only hits >= tau can reach the merged top-K. cut[s] = number of such hits in
// list s (all of the list when the short lists leave fewer than K guaranteed hits). One block, warp = list.
template <class Src>
__global__ void __launch_bounds__(1024) k_merge_prep(const Src src, uint32_t n_lists, uint32_t K, uint32_t o1, uint32_t o2, uint32_t* cut) {
  __shared__ MKey s_key[64];
  __shared__ MKey s_keyK[64];
  __shared__ uint32_t s_have[64], s_full[64];
  __shared__ MKey s_tau;
  __shared__ uint32_t s_prune;
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  if (n_lists > 64) {  // more lists than the shared tables hold: no pruning
    for (uint32_t s = threadIdx.x; s < n_lists; s += blockDim.x) cut[s] = min(src.count(s), K);
    return;
  }
  uint32_t nonempty = 0;
  for (uint32_t s = lane; s < n_lists; s += 32) nonempty += src.count(s) ? 1u : 0u;  // (one round of loads per warp)
  nonempty = __reduce_add_sync(0xFFFFFFFFu, nonempty);
  const uint32_t m = nonempty ? (K + nonempty - 1) / nonempty : 0;
  for (uint32_t s = warp; s < n_lists; s += nw) {
    if (lane == 0) {
      const uint32_t nh = min(src.count(s), K), ms = min(m, nh);
      s_have[s] = ms;
      if (ms) { uint32_t rk; const QwHit h = src.hit(s, ms - 1, rk); s_key[s] = merge_key(h, rk, o1, o2); }
      // a list that holds K hits by itself: its own K-th hit bounds the merged K-th hit as well (the bound that
      // bites when the lists are skewed — time-sorted hits of time-partitioned splits all come from one split)
      s_full[s] = (K > 0 && nh >= K) ? 1u : 0u;
      if (s_full[s]) { uint32_t rk; const QwHit h = src.hit(s, K - 1, rk); s_keyK[s] = merge_key(h, rk, o1, o2); }
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t have = 0, first = 1;
    MKey tau;
    tau.v1 = tau.v2 = tau.tie = 0; tau.has = 0;
    for (uint32_t s = 0; s < n_lists; s++) {
      have += s_have[s];
      if (s_have[s] && (first || mkey_gt(tau, s_key[s]))) { tau = s_key[s]; first = 0; }
    }
    uint32_t prune = have >= K ? 1u : 0u;
    for (uint32_t s = 0; s < n_lists; s++)
      if (s_full[s] && (!prune || mkey_gt(s_keyK[s], tau))) { tau = s_keyK[s]; prune = 1; }  // the tighter of the valid bounds
    s_tau = tau;
    s_prune = prune;
  }
  __syncthreads();
  const MKey tau = s_tau;
  for (uint32_t s = warp; s < n_lists; s += nw) {
    const uint32_t nh = min(src.count(s), K);
    uint32_t lo = 0, hi = nh;  // first index whose hit is worse than tau
    if (s_prune) {
      // 32-ary search: the lanes probe evenly spaced hits of [lo, hi) at once (the list is sorted best-first, so the
      // hits that are not worse than tau form a prefix of the probes): two or three rounds of loads for 1000 hits
      while (lo < hi) {
        const uint32_t step = (hi - lo + 31) / 32, idx = lo + lane * step;
        bool keep = false;
        if (idx < hi) {
          uint32_t rk;
          const QwHit h = src.hit(s, idx, rk);
          keep = !mkey_gt(tau, merge_key(h, rk, o1, o2));
        }
        const uint32_t c = (uint32_t)__popc(__ballot_sync(0xFFFFFFFFu, keep));
        if (c == 0) { hi = lo; break; }
        hi = min(hi, lo + c * step);
        lo = lo + (c - 1) * step + 1;
      }
    } else lo = nh;
    if (lane == 0) cut[s] = lo;
  }
}
template <class Src>
__global__ void __launch_bounds__(256) k_merge(const Src src, const uint32_t* cut, uint32_t n_lists, uint32_t kmax, uint32_t K, uint32_t o1, uint32_t o2,
                                               DMergedHit* out, uint32_t* out_n) {
  // one warp per surviving hit; lane = one of the other lists (the binary searches of a hit run side by side)
  const uint32_t lane = threadIdx.x & 31, e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (e == 0 && lane == 0) {
    uint64_t total = 0;
    for (uint32_t s = 0; s < n_lists; s++) total += src.count(s);
    *out_n = (uint32_t)(total < K ? total : K);
  }
  const uint32_t s = e / kmax, i = e % kmax;
  if (s >= n_lists || i >= __ldg(cut + s)) return;
  uint32_t my_rk;
  const QwHit mine = src.hit(s, i, my_rk);
  const MKey key = merge_key(mine, my_rk, o1, o2);
  uint32_t r = 0;
  for (uint32_t s2 = lane; s2 < n_lists; s2 += 32) {
    if (s2 == s) continue;
    uint32_t lo = 0, hi = __ldg(cut + s2);  // first index whose hit does not beat `key` (hits past the cut never do)
    while (lo < hi) {
      const uint32_t mid = (lo + hi) >> 1;
      uint32_t rk;
      const QwHit h = src.hit(s2, mid, rk);
      if (mkey_gt(merge_key(h, rk, o1, o2), key)) lo = mid + 1; else hi = mid;
    }
    r += lo;
  }
  r = __reduce_add_sync(0xFFFFFFFFu, r) + i;
  if (lane == 0 && r < K) { DMergedHit m; m.hit = mine; m.split = src.tag(s, my_rk); m.pad = 0; out[r] = m; }
}

// Header of a rank's gather record: its hit count (already written by k_merge at offset 0) plus the sums the
// root merge adds up (collector.rs:914-974): num_hits over the batch's splits, split accounting from the host.
struct DRankHeader {
  uint32_t n_hits, pad;
  uint64_t num_hits, attempted, successful, n_failed, reserved[3];
};
__global__ void k_rank_header(const DSplitPlan* plans, uint32_t n_splits, DRankHeader* h, uint64_t attempted, uint64_t successful, uint64_t n_failed) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    uint64_t nh = 0;
    for (uint32_t s = 0; s < n_splits; s++) nh += *(const uint64_t*)plans[s].out_num_hits;
    h->pad = 0; h->num_hits = nh; h->attempted = attempted; h->successful = successful; h->n_failed = n_failed;
    h->reserved[0] = h->reserved[1] = h->reserved[2] = 0;
  }
}

}  // namespace qwk
