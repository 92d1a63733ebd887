// aggs.cpp — aggregation request parsing, lowering to dense GPU bucket spaces, intermediate
// results (build / merge / serialise) and finalisation.
//
// Reference behaviour restated (the engine itself is tantivy::aggregation, external):
//   * request shape + parameters: docs/reference/aggregation.md:40-700
//   * leaf: AggregationSegmentCollector::harvest -> IntermediateAggregationResults, cut to
//     `segment_size` per split with sum_other_doc_count / doc_count_error_upper_bound
//     (quickwit-search/src/collector.rs:577-581; aggregation.md:500-560)
//   * merge: IntermediateAggregationResults::merge_fruits (collector.rs:870-911)
//   * final: into_final_result (quickwit-search/src/root.rs:1105-1135): buckets cut to `size`,
//     histogram gaps filled when min_doc_count == 0, extended_bounds, key_as_string.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <map>
#include <memory>

#include "compile.h"

namespace qw {

// ---- request parsing -----------------------------------------------------------------------------------
static double parse_duration_ms(const std::string& s, bool allow_negative) {
  // fixed_interval / offset syntax: <int><unit>, unit in ms|s|m|h|d (aggregation.md:300-320)
  size_t i = 0;
  bool neg = false;
  if (i < s.size() && (s[i] == '-' || s[i] == '+')) { neg = s[i] == '-'; i++; }
  if (neg && !allow_negative) fail(QWGPU_EINVALID_AGG, "negative duration `%s`", s.c_str());
  size_t j = i;
  while (j < s.size() && isdigit((unsigned char)s[j])) j++;
  if (j == i) fail(QWGPU_EINVALID_AGG, "invalid duration `%s`", s.c_str());
  double n = strtod(s.substr(i, j - i).c_str(), nullptr);
  std::string unit = s.substr(j);
  double mult;
  if (unit == "ms") mult = 1;
  else if (unit == "s") mult = 1000;
  else if (unit == "m") mult = 60000;
  else if (unit == "h") mult = 3600000;
  else if (unit == "d") mult = 86400000;
  else fail(QWGPU_EINVALID_AGG, "unsupported duration unit in `%s` (only fixed intervals ms|s|m|h|d)", s.c_str());
  return (neg ? -1 : 1) * n * mult;
}

static double num_or(const Json& j, const char* k, double d) {
  const Json* v = j.get(k);
  if (!v) return d;
  if (v->is_num()) return v->as_f64();
  if (v->is_str()) return strtod(v->s.c_str(), nullptr);
  return d;
}

static void parse_agg_map(const Json& j, std::vector<AggReq>& out, int depth) {
  if (!j.is_obj()) fail(QWGPU_EINVALID_AGG, "aggregation request must be a JSON object");
  if (depth > 8) fail(QWGPU_EINVALID_AGG, "aggregation nesting too deep");
  for (auto& kv : j.obj) {
    AggReq a;
    a.name = kv.first;
    const Json& body = kv.second;
    bool found = false;
    for (auto& p : body.obj) {
      const std::string& t = p.first;
      const Json& spec = p.second;
      if (t == "aggs" || t == "aggregations") { parse_agg_map(spec, a.children, depth + 1); continue; }
      if (found) fail(QWGPU_EINVALID_AGG, "aggregation `%s` has more than one type", a.name.c_str());
      found = true;
      a.field = spec.str_or("field", "");
      if (t == "terms") {
        a.kind = AggReq::Terms;
        a.size = (uint32_t)num_or(spec, "size", 10);
        double ss = -1;
        for (const char* k : {"split_size", "segment_size", "shard_size"}) if (spec.get(k)) ss = num_or(spec, k, -1);
        a.segment_size = ss >= 0 ? (uint32_t)ss : a.size * 10;
        a.segment_size = std::max(a.segment_size, a.size);
        a.min_doc_count = (uint64_t)num_or(spec, "min_doc_count", 1);
        if (const Json* m = spec.get("missing")) { a.has_missing = true; a.missing = *m; }
        if (const Json* o = spec.get("order")) {
          if (!o->is_obj() || o->obj.size() != 1) fail(QWGPU_EINVALID_AGG, "terms `order` must be an object with one property");
          a.order_target = o->obj[0].first;
          a.order_desc = o->obj[0].second.is_str() && o->obj[0].second.s == "desc";
        }
      } else if (t == "histogram" || t == "date_histogram") {
        a.kind = t == "histogram" ? AggReq::Histogram : AggReq::DateHistogram;
        if (a.kind == AggReq::DateHistogram) {
          if (spec.get("interval") || spec.get("calendar_interval")) fail(QWGPU_EINVALID_AGG, "date_histogram only supports `fixed_interval`");
          const Json* fi = spec.get("fixed_interval");
          if (!fi || !fi->is_str()) fail(QWGPU_EINVALID_AGG, "date_histogram requires `fixed_interval`");
          a.interval = parse_duration_ms(fi->s, false);
          if (const Json* off = spec.get("offset")) a.offset = off->is_str() ? parse_duration_ms(off->s, true) : off->as_f64();
        } else {
          a.interval = num_or(spec, "interval", 0);
          a.offset = num_or(spec, "offset", 0);
        }
        if (!(a.interval > 0)) fail(QWGPU_EINVALID_AGG, "histogram interval must be larger than 0");
        a.min_doc_count = (uint64_t)num_or(spec, "min_doc_count", 0);
        a.keyed = spec.bool_or("keyed", false);
        if (const Json* b = spec.get("hard_bounds")) { a.has_hard_bounds = true; a.hard_min = num_or(*b, "min", -INFINITY); a.hard_max = num_or(*b, "max", INFINITY); }
        if (const Json* b = spec.get("extended_bounds")) {
          a.has_extended_bounds = true; a.ext_min = num_or(*b, "min", INFINITY); a.ext_max = num_or(*b, "max", -INFINITY);
          if (a.min_doc_count > 0) fail(QWGPU_EINVALID_AGG, "Cannot set min_doc_count and extended_bounds at the same time");
        }
      } else if (t == "range") {
        a.kind = AggReq::Range;
        const Json* rs = spec.get("ranges");
        if (!rs || !rs->is_arr()) fail(QWGPU_EINVALID_AGG, "range aggregation requires `ranges`");
        for (auto& r : rs->arr) {
          AggReq::R x;
          if (const Json* f = r.get("from")) if (f->is_num()) { x.has_from = true; x.from = f->as_f64(); }
          if (const Json* f = r.get("to")) if (f->is_num()) { x.has_to = true; x.to = f->as_f64(); }
          x.key = r.str_or("key", "");
          a.ranges.push_back(x);
        }
        a.keyed = spec.bool_or("keyed", false);
      } else if (t == "stats") a.kind = AggReq::Stats;
      else if (t == "avg") a.kind = AggReq::Avg;
      else if (t == "sum") a.kind = AggReq::Sum;
      else if (t == "min") a.kind = AggReq::Min;
      else if (t == "max") a.kind = AggReq::Max;
      else if (t == "value_count" || t == "count") a.kind = AggReq::Count;
      else if (t == "percentiles" || t == "cardinality" || t == "extended_stats" || t == "composite" || t == "top_hits" || t == "filter")
        fail(QWGPU_EUNSUPPORTED, "`%s` aggregations are not implemented on the GPU path yet", t.c_str());
      else fail(QWGPU_EINVALID_AGG, "unknown aggregation type `%s`", t.c_str());
    }
    if (!found) fail(QWGPU_EINVALID_AGG, "aggregation `%s` has no type", a.name.c_str());
    if (a.is_metric() && !a.children.empty()) fail(QWGPU_EINVALID_AGG, "metric aggregation `%s` cannot have sub-aggregations", a.name.c_str());
    out.push_back(std::move(a));
  }
}

std::vector<AggReq> parse_agg_request(const std::string& json) {
  std::vector<AggReq> out;
  parse_agg_map(parse_json(json, QWGPU_EINVALID_AGG), out, 0);
  return out;
}

// ---- lowering ------------------------------------------------------------------------------------------
static double mapped_to_f64(uint32_t type, uint64_t m) {
  switch (type) {
    case QW_COL_U64: case QW_COL_BOOL: case QW_COL_STR: return (double)m;
    case QW_COL_I64: case QW_COL_DATETIME: return (double)u64_to_i64(m);
    default: return u64_to_f64(m);
  }
}
static uint64_t f64_bound_to_mapped(uint32_t type, double v) {  // smallest mapped value whose f64 is >= v
  switch (type) {
    case QW_COL_F64: return f64_to_u64(v);
    case QW_COL_U64: case QW_COL_BOOL: return v <= 0 ? 0 : (v >= 18446744073709551615.0 ? ~0ull : (uint64_t)std::ceil(v));
    default: {
      double c = std::ceil(v);
      int64_t i = c <= -9223372036854775808.0 ? INT64_MIN : (c >= 9223372036854775807.0 ? INT64_MAX : (int64_t)c);
      return i64_to_u64(i);
    }
  }
}

static QwAggNode lower_one(const AggReq& a, const ImageView& img, AggBinding& b) {
  QwAggNode n;
  memset(&n, 0, sizeof n);
  n.parent = 0xFFFFFFFFu;
  n.column = 0xFFFFFFFFu;
  b.req = &a;
  int c = img.find_column(a.field);
  b.column = c;
  const QwImgColumn* col = c >= 0 ? &img.columns[c] : nullptr;
  if (col) { n.column = (uint32_t)c; b.col_type = col->type; }
  switch (a.kind) {
    case AggReq::Terms: {
      n.kind = QW_AGG_TERMS;
      uint64_t nb = col ? (col->max_value - col->min_value) / col->gcd + 1 : 0;
      if (col && col->num_vals == 0) nb = 0;
      if (nb > (1u << 24)) fail(QWGPU_EUNSUPPORTED, "terms aggregation over %llu distinct dense slots is not supported on the GPU path", (unsigned long long)nb);
      n.num_buckets = (uint32_t)nb + (a.has_missing ? 1 : 0);
      n.has_missing = a.has_missing;
      break;
    }
    case AggReq::Histogram: case AggReq::DateHistogram: {
      n.kind = QW_AGG_HISTOGRAM;
      if (col && col->type == QW_COL_STR) fail(QWGPU_EINVALID_AGG, "histogram on text field `%s`", a.field.c_str());
      if (a.kind == AggReq::DateHistogram && col && col->type != QW_COL_DATETIME)
        fail(QWGPU_EINVALID_AGG, "date_histogram requires a datetime field, `%s` is not", a.field.c_str());
      // DateTime columns hold nanoseconds: request values are milliseconds (aggregation.md:150-160)
      double scale = (col && col->type == QW_COL_DATETIME) ? 1e6 : 1.0;
      n.interval = a.interval * scale;
      n.offset = a.offset * scale;
      if (a.has_hard_bounds) { n.has_bounds = 1; n.bound_min = a.hard_min * scale; n.bound_max = a.hard_max * scale; }
      if (col && col->num_vals) {
        double lo = mapped_to_f64(col->type, col->min_value), hi = mapped_to_f64(col->type, col->max_value);
        if (n.has_bounds) { lo = std::max(lo, n.bound_min); hi = std::min(hi, n.bound_max); }
        if (lo <= hi) {
          double p0 = std::floor((lo - n.offset) / n.interval), p1 = std::floor((hi - n.offset) / n.interval);
          if (p1 - p0 + 1 > 65000.0 * 16) fail(QWGPU_EINVALID_AGG, "histogram would create too many buckets (%g)", p1 - p0 + 1);
          n.base_pos = (int64_t)p0;
          n.num_buckets = (uint32_t)(p1 - p0 + 1);
        }
      }
      break;
    }
    case AggReq::Range: {
      n.kind = QW_AGG_RANGE;
      if (a.ranges.size() > QW_MAX_AGG_RANGES) fail(QWGPU_EUNSUPPORTED, "more than %d ranges", QW_MAX_AGG_RANGES);
      n.num_ranges = n.num_buckets = (uint32_t)a.ranges.size();
      uint32_t t = col ? col->type : (uint32_t)QW_COL_F64;
      for (size_t i = 0; i < a.ranges.size(); i++) {
        n.range_from[i] = a.ranges[i].has_from ? f64_bound_to_mapped(t, a.ranges[i].from) : 0;
        n.range_to[i] = a.ranges[i].has_to ? f64_bound_to_mapped(t, a.ranges[i].to) : ~0ull;
      }
      break;
    }
    default: n.kind = QW_AGG_STATS; n.num_buckets = 1; break;
  }
  return n;
}

std::vector<QwAggNode> lower_aggs(const std::vector<AggReq>& reqs, const ImageView& img, std::vector<AggBinding>& bindings) {
  std::vector<QwAggNode> out;
  bindings.clear();
  struct Pending { const AggReq* a; uint32_t idx; };
  std::vector<Pending> queue;
  for (auto& a : reqs) {
    AggBinding b;
    out.push_back(lower_one(a, img, b));
    bindings.push_back(b);
    queue.push_back({&a, (uint32_t)out.size() - 1});
  }
  for (size_t qi = 0; qi < queue.size(); qi++) {
    Pending p = queue[qi];
    if (p.a->children.empty()) continue;
    out[p.idx].first_child = (uint32_t)out.size();
    out[p.idx].num_children = (uint32_t)p.a->children.size();
    for (auto& c : p.a->children) {
      AggBinding b;
      QwAggNode n = lower_one(c, img, b);
      n.parent = p.idx;
      out.push_back(n);
      bindings.push_back(b);
      queue.push_back({&c, (uint32_t)out.size() - 1});
    }
  }
  return out;
}

// ---- intermediate model --------------------------------------------------------------------------------
struct IKey {
  enum K : uint8_t { Str = 0, F64 = 1, I64 = 2, U64 = 3 } kind = Str;
  std::string s;
  double f = 0;
  int64_t i = 0;
  uint64_t u = 0;
  bool operator<(const IKey& o) const {
    if (kind != o.kind) {
      if (kind != Str && o.kind != Str) return num() < o.num();
      return kind < o.kind;
    }
    switch (kind) { case Str: return s < o.s; case F64: return f < o.f; case I64: return i < o.i; default: return u < o.u; }
  }
  bool operator==(const IKey& o) const { return !(*this < o) && !(o < *this); }
  double num() const { return kind == F64 ? f : (kind == I64 ? (double)i : (double)u); }
};
struct IAgg;
struct IBucket {
  IKey key;        // terms
  double hkey = 0;  // histogram (column units) / range index
  uint64_t count = 0;
  std::vector<IAgg> subs;
};
struct IAgg {
  uint8_t kind = 0;  // AggReq::Kind
  std::vector<IBucket> buckets;
  uint64_t sum_other = 0, error_bound = 0;
  uint8_t is_date = 0;
  // metric
  uint64_t m_count = 0;
  double m_sum = 0, m_min = INFINITY, m_max = -INFINITY;
  // key -> position in `buckets`, built on the first merge into this node and kept up to date, so that
  // folding n responses costs O(total buckets · log) instead of re-indexing the accumulator n times
  struct Index {
    std::map<IKey, size_t> terms;
    std::map<double, size_t> hist;
  };
  std::shared_ptr<Index> index;  // allocated on the first merge into this node (accumulators only)
};

struct BW {
  std::string out;
  void varint(uint64_t v) { while (v >= 0x80) { out += (char)(v | 0x80); v >>= 7; } out += (char)v; }
  void f64(double d) { out.append((const char*)&d, 8); }
  void str(const std::string& s) { varint(s.size()); out += s; }
};
struct BR {
  const uint8_t *p, *e;
  uint64_t varint() {
    uint64_t v = 0; int sh = 0;
    while (p < e) { uint8_t c = *p++; v |= (uint64_t)(c & 0x7F) << sh; if (!(c & 0x80)) return v; sh += 7; }
    fail(QWGPU_EINTERNAL, "failed to merge intermediate aggregation results: truncated buffer");
  }
  double f64() { if (e - p < 8) fail(QWGPU_EINTERNAL, "failed to merge intermediate aggregation results: truncated buffer"); double d; memcpy(&d, p, 8); p += 8; return d; }
  std::string str() { uint64_t n = varint(); if ((uint64_t)(e - p) < n) fail(QWGPU_EINTERNAL, "failed to merge intermediate aggregation results: truncated buffer"); std::string s((const char*)p, n); p += n; return s; }
};

static void ser_aggs(BW& w, const std::vector<IAgg>& v);
static void ser_agg(BW& w, const IAgg& a) {
  w.varint(a.kind);
  if (a.kind >= AggReq::Stats) { w.varint(a.m_count); w.f64(a.m_sum); w.f64(a.m_min); w.f64(a.m_max); return; }
  w.varint(a.is_date);
  w.varint(a.sum_other);
  w.varint(a.error_bound);
  w.varint(a.buckets.size());
  for (auto& b : a.buckets) {
    if (a.kind == AggReq::Terms) {
      w.varint(b.key.kind);
      switch (b.key.kind) { case IKey::Str: w.str(b.key.s); break; case IKey::F64: w.f64(b.key.f); break; case IKey::I64: w.varint((uint64_t)b.key.i); break; default: w.varint(b.key.u); }
    } else w.f64(b.hkey);
    w.varint(b.count);
    ser_aggs(w, b.subs);
  }
}
static void ser_aggs(BW& w, const std::vector<IAgg>& v) {
  w.varint(v.size());
  for (auto& a : v) ser_agg(w, a);
}
static std::vector<IAgg> de_aggs(BR& r);
static IAgg de_agg(BR& r) {
  IAgg a;
  a.kind = (uint8_t)r.varint();
  if (a.kind >= AggReq::Stats) { a.m_count = r.varint(); a.m_sum = r.f64(); a.m_min = r.f64(); a.m_max = r.f64(); return a; }
  a.is_date = (uint8_t)r.varint();
  a.sum_other = r.varint();
  a.error_bound = r.varint();
  uint64_t n = r.varint();
  for (uint64_t i = 0; i < n; i++) {
    IBucket b;
    if (a.kind == AggReq::Terms) {
      b.key.kind = (IKey::K)r.varint();
      switch (b.key.kind) { case IKey::Str: b.key.s = r.str(); break; case IKey::F64: b.key.f = r.f64(); break; case IKey::I64: b.key.i = (int64_t)r.varint(); break; default: b.key.u = r.varint(); }
    } else b.hkey = r.f64();
    b.count = r.varint();
    b.subs = de_aggs(r);
    a.buckets.push_back(std::move(b));
  }
  return a;
}
static std::vector<IAgg> de_aggs(BR& r) {
  uint64_t n = r.varint();
  std::vector<IAgg> v;
  for (uint64_t i = 0; i < n; i++) v.push_back(de_agg(r));
  return v;
}
static const char kMagic[4] = {'Q', 'W', 'I', 'A'};
static std::string ser_top(const std::vector<IAgg>& v) {
  BW w;
  w.out.append(kMagic, 4);
  ser_aggs(w, v);
  return w.out;
}
static std::vector<IAgg> de_top(const std::string& s) {
  if (s.size() < 4 || memcmp(s.data(), kMagic, 4) != 0) fail(QWGPU_EINTERNAL, "failed to merge intermediate aggregation results: bad header");
  BR r{(const uint8_t*)s.data() + 4, (const uint8_t*)s.data() + s.size()};
  return de_aggs(r);
}

// ---- build from dense cells ----------------------------------------------------------------------------
struct BuildCtx {
  const CompiledPlan& cp;
  const ImageView& img;
  const QwAggNode* nodes;
  const QwAggCell* cells;
  std::vector<uint32_t> bases;
};

static IAgg build_node(const BuildCtx& c, uint32_t ni, uint64_t parent_cell);

static std::vector<IAgg> build_children(const BuildCtx& c, uint32_t ni, uint64_t cell) {
  std::vector<IAgg> out;
  const QwAggNode& n = c.nodes[ni];
  for (uint32_t k = 0; k < n.num_children; k++) out.push_back(build_node(c, n.first_child + k, cell));
  return out;
}

static IKey term_key(const BuildCtx& c, const AggBinding& b, const QwAggNode& n, uint32_t bucket) {
  IKey k;
  if (n.has_missing && bucket == n.num_buckets - 1) {
    const Json& m = b.req->missing;
    if (m.type == Json::Str) { k.kind = IKey::Str; k.s = m.s; }
    else if (m.type == Json::U64) { k.kind = IKey::U64; k.u = m.u; }
    else if (m.type == Json::I64) { k.kind = IKey::I64; k.i = m.i; }
    else { k.kind = IKey::F64; k.f = m.as_f64(); }
    return k;
  }
  const QwImgColumn& col = c.img.columns[b.column];
  uint64_t mapped = col.min_value + col.gcd * (uint64_t)bucket;
  switch (col.type) {
    case QW_COL_STR: { const uint8_t* p; uint32_t len; c.img.dict_term(col, (uint32_t)mapped, &p, &len); k.kind = IKey::Str; k.s.assign((const char*)p, len); break; }
    case QW_COL_F64: k.kind = IKey::F64; k.f = u64_to_f64(mapped); break;
    case QW_COL_I64: case QW_COL_DATETIME: k.kind = IKey::I64; k.i = u64_to_i64(mapped); break;
    default: k.kind = IKey::U64; k.u = mapped; break;
  }
  if (k.kind == IKey::U64 && k.u <= (uint64_t)INT64_MAX) { k.kind = IKey::I64; k.i = (int64_t)k.u; }
  return k;
}

static double metric_of(const IAgg& a, const std::string& prop) {
  if (a.kind < AggReq::Stats) return 0;
  std::string p = prop;
  if (p.empty()) p = a.kind == AggReq::Avg ? "avg" : a.kind == AggReq::Sum ? "sum" : a.kind == AggReq::Min ? "min" : a.kind == AggReq::Max ? "max" : a.kind == AggReq::Count ? "count" : "avg";
  if (p == "avg") return a.m_count ? a.m_sum / (double)a.m_count : 0;
  if (p == "sum") return a.m_sum;
  if (p == "min") return a.m_min;
  if (p == "max") return a.m_max;
  return (double)a.m_count;
}

// sorts term buckets in the requested order (ties: key ascending, for determinism)
static void sort_term_buckets(const AggReq& req, std::vector<IBucket>& bs) {
  if (req.order_target == "_key") {
    std::sort(bs.begin(), bs.end(), [&](const IBucket& a, const IBucket& b) { return req.order_desc ? b.key < a.key : a.key < b.key; });
    return;
  }
  if (req.order_target == "_count") {
    std::sort(bs.begin(), bs.end(), [&](const IBucket& a, const IBucket& b) {
      if (a.count != b.count) return req.order_desc ? a.count > b.count : a.count < b.count;
      return a.key < b.key;
    });
    return;
  }
  std::string name = req.order_target, prop;
  size_t dot = name.find('.');
  if (dot != std::string::npos) { prop = name.substr(dot + 1); name = name.substr(0, dot); }
  int ci = -1;
  for (size_t i = 0; i < req.children.size(); i++) if (req.children[i].name == name) ci = (int)i;
  if (ci < 0) fail(QWGPU_EINVALID_AGG, "could not find aggregation with name `%s` in metric sub_aggregations", name.c_str());
  std::sort(bs.begin(), bs.end(), [&](const IBucket& a, const IBucket& b) {
    double x = metric_of(a.subs[ci], prop), y = metric_of(b.subs[ci], prop);
    if (x != y) return req.order_desc ? x > y : x < y;
    return a.key < b.key;
  });
}

static IAgg build_node(const BuildCtx& c, uint32_t ni, uint64_t parent_cell) {
  const QwAggNode& n = c.nodes[ni];
  const AggBinding& b = c.cp.agg_bindings[ni];
  const AggReq& req = *b.req;
  const QwAggCell* base = c.cells + c.bases[ni];
  IAgg a;
  a.kind = (uint8_t)req.kind;
  if (req.is_metric()) {
    const QwAggCell& cell = base[parent_cell];
    a.m_count = cell.count;
    if (cell.count && b.column >= 0) {
      uint32_t t = b.col_type;
      const QwImgColumn& col = c.img.columns[b.column];
      if (!qw_col_sum_exact(&col)) memcpy(&a.m_sum, &cell.sum_bits, 8);
      else {
        // exact: sum of the typed values = count * min + gcd * (sum of raw offsets); the mapped u64 of an
        // i64 / datetime is value + 2^63
        __int128 sum = (__int128)(unsigned __int128)col.min_value * (__int128)cell.count + (__int128)((unsigned __int128)col.gcd * cell.sum_bits);
        if (!(t == QW_COL_U64 || t == QW_COL_BOOL)) sum -= ((__int128)1 << 63) * (__int128)cell.count;
        a.m_sum = (double)sum;
      }
      a.m_min = mapped_to_f64(t, cell.min_mapped);
      a.m_max = mapped_to_f64(t, cell.max_mapped);
    }
    return a;
  }
  a.is_date = req.kind == AggReq::DateHistogram;
  for (uint32_t k = 0; k < n.num_buckets; k++) {
    uint64_t cell = parent_cell * n.num_buckets + k;
    uint64_t cnt = base[cell].count;
    if (cnt == 0 && req.kind != AggReq::Range) continue;
    IBucket bk;
    bk.count = cnt;
    if (req.kind == AggReq::Terms) bk.key = term_key(c, b, n, k);
    else if (req.kind == AggReq::Range) bk.hkey = (double)k;
    else bk.hkey = (double)(n.base_pos + (int64_t)k) * n.interval + n.offset;
    bk.subs = build_children(c, ni, cell);
    a.buckets.push_back(std::move(bk));
  }
  if (req.kind == AggReq::Terms && req.order_target.find('.') == std::string::npos &&
      (req.order_target == "_count" || req.order_target == "_key")) {
    // per-split cut to segment_size (cut_off_buckets): error bound = doc count of the first dropped
    // bucket, sum_other = sum of dropped doc counts
    sort_term_buckets(req, a.buckets);
    if (a.buckets.size() > req.segment_size) {
      if (req.order_target == "_count" && req.order_desc) a.error_bound = a.buckets[req.segment_size].count;
      for (size_t i = req.segment_size; i < a.buckets.size(); i++) a.sum_other += a.buckets[i].count;
      a.buckets.resize(req.segment_size);
    }
  }
  return a;
}

static std::vector<IAgg> build_top(const CompiledPlan& cp, const ImageView& img, const QwAggCell* cells, size_t ncells);
std::string build_intermediate_aggs(const CompiledPlan& cp, const ImageView& img, const QwAggCell* cells, size_t ncells) {
  return ser_top(build_top(cp, img, cells, ncells));
}
static std::vector<IAgg> build_top(const CompiledPlan& cp, const ImageView& img, const QwAggCell* cells, size_t ncells) {
  const QwPlanHeader& h = cp.header;
  const QwAggNode* nodes = (const QwAggNode*)(cp.bytes.data() + sizeof(QwPlanHeader) + (size_t)h.num_nodes * sizeof(QwPlanNode));
  BuildCtx c{cp, img, nodes, cells, {}};
  uint64_t total = 0;
  c.bases.resize(h.num_aggs);
  for (uint32_t i = 0; i < h.num_aggs; i++) {
    uint64_t cnt = nodes[i].kind == QW_AGG_STATS ? 1 : nodes[i].num_buckets;
    uint32_t p = nodes[i].parent;
    while (p != 0xFFFFFFFFu) { cnt *= nodes[p].num_buckets; p = nodes[p].parent; }
    c.bases[i] = (uint32_t)total;
    total += cnt;
  }
  if (total != ncells) fail(QWGPU_EINTERNAL, "aggregation cell count mismatch (%llu vs %zu)", (unsigned long long)total, ncells);
  std::vector<IAgg> top;
  for (uint32_t i = 0; i < h.num_aggs; i++) if (nodes[i].parent == 0xFFFFFFFFu) top.push_back(build_node(c, i, 0));
  return top;
}

// ---- merge ------------------------------------------------------------------------------------------------
static void merge_into(const AggReq& req, IAgg& acc, IAgg&& other);
static void merge_lists(const std::vector<AggReq>& reqs, std::vector<IAgg>& acc, std::vector<IAgg>&& other) {
  if (acc.empty()) { acc = std::move(other); return; }
  if (other.empty()) return;
  if (acc.size() != other.size() || acc.size() != reqs.size()) fail(QWGPU_EINTERNAL, "failed to merge intermediate aggregation results: shape mismatch");
  for (size_t i = 0; i < acc.size(); i++) merge_into(reqs[i], acc[i], std::move(other[i]));
}
static void merge_into(const AggReq& req, IAgg& acc, IAgg&& other) {
  if (acc.kind != other.kind) fail(QWGPU_EINTERNAL, "failed to merge intermediate aggregation results: kind mismatch");
  if (acc.kind >= AggReq::Stats) {
    acc.m_count += other.m_count;
    acc.m_sum += other.m_sum;
    acc.m_min = std::min(acc.m_min, other.m_min);
    acc.m_max = std::max(acc.m_max, other.m_max);
    return;
  }
  acc.sum_other += other.sum_other;
  acc.error_bound += other.error_bound;
  if (acc.kind == AggReq::Terms) {
    if (!acc.index) { acc.index = std::make_shared<IAgg::Index>(); for (size_t i = 0; i < acc.buckets.size(); i++) acc.index->terms[acc.buckets[i].key] = i; }
    auto& index = acc.index->terms;
    for (auto& b : other.buckets) {
      auto it = index.find(b.key);
      if (it == index.end()) { index[b.key] = acc.buckets.size(); acc.buckets.push_back(std::move(b)); }
      else { IBucket& t = acc.buckets[it->second]; t.count += b.count; merge_lists(req.children, t.subs, std::move(b.subs)); }
    }
  } else {
    if (!acc.index) { acc.index = std::make_shared<IAgg::Index>(); for (size_t i = 0; i < acc.buckets.size(); i++) acc.index->hist[acc.buckets[i].hkey] = i; }
    auto& index = acc.index->hist;
    for (auto& b : other.buckets) {
      auto it = index.find(b.hkey);
      if (it == index.end()) { index[b.hkey] = acc.buckets.size(); acc.buckets.push_back(std::move(b)); }
      else { IBucket& t = acc.buckets[it->second]; t.count += b.count; merge_lists(req.children, t.subs, std::move(b.subs)); }
    }
  }
}

// Leaf-level merge of the splits of one request straight from their dense cells: what
// merge_intermediate_aggs(build_intermediate_aggs(split) ...) yields, without serialising every split's
// result only to parse it again.
std::string build_and_merge_intermediate_aggs(const std::vector<AggReq>& reqs, const std::vector<SplitAggCells>& splits) {
  std::vector<IAgg> acc;
  for (const SplitAggCells& sp : splits) {
    std::vector<IAgg> top = build_top(*sp.plan, *sp.img, sp.cells, sp.ncells);
    if (acc.empty() && !top.empty()) {
      // same normalisation as a serialise / parse round trip would apply: none needed — the first
      // split's tree becomes the accumulator
      acc = std::move(top);
      continue;
    }
    merge_lists(reqs, acc, std::move(top));
  }
  return ser_top(acc);
}

std::string merge_intermediate_aggs(const std::vector<AggReq>& reqs, const std::vector<std::string>& parts) {
  std::vector<IAgg> acc;
  static const bool trace = getenv("QWGPU_TRACE_AGG") != nullptr;
  if (!trace) {
    for (auto& p : parts) merge_lists(reqs, acc, de_top(p));
    return ser_top(acc);
  }
  using clk = std::chrono::steady_clock;
  long de = 0, mg = 0;
  for (auto& p : parts) {
    auto t0 = clk::now();
    std::vector<IAgg> d = de_top(p);
    auto t1 = clk::now();
    merge_lists(reqs, acc, std::move(d));
    auto t2 = clk::now();
    de += std::chrono::duration_cast<std::chrono::nanoseconds>(t1 - t0).count();
    mg += std::chrono::duration_cast<std::chrono::nanoseconds>(t2 - t1).count();
  }
  auto t0 = clk::now();
  std::string out = ser_top(acc);
  long se = std::chrono::duration_cast<std::chrono::nanoseconds>(clk::now() - t0).count();
  fprintf(stderr, "[qwgpu] merge_intermediate_aggs: %zu parts, decode %ld us, merge %ld us, encode %ld us\n", parts.size(), de / 1000, mg / 1000, se / 1000);
  return out;
}

// ---- finalize -----------------------------------------------------------------------------------------------
static void civil_from_days(int64_t z, int64_t* y, unsigned* m, unsigned* d) {
  z += 719468;
  const int64_t era = (z >= 0 ? z : z - 146096) / 146097;
  const unsigned doe = (unsigned)(z - era * 146097);
  const unsigned yoe = (doe - doe / 1460 + doe / 36524 - doe / 146096) / 365;
  *y = (int64_t)yoe + era * 400;
  const unsigned doy = doe - (365 * yoe + yoe / 4 - yoe / 100);
  const unsigned mp = (5 * doy + 2) / 153;
  *d = doy - (153 * mp + 2) / 5 + 1;
  *m = mp < 10 ? mp + 3 : mp - 9;
  *y += *m <= 2;
}
static std::string rfc3339_from_ms(double ms) {
  int64_t total_ms = (int64_t)std::floor(ms);
  int64_t secs = total_ms / 1000, rem = total_ms % 1000;
  if (rem < 0) { rem += 1000; secs -= 1; }
  int64_t days = secs / 86400, sod = secs % 86400;
  if (sod < 0) { sod += 86400; days -= 1; }
  int64_t y; unsigned m, d;
  civil_from_days(days, &y, &m, &d);
  char b[64];
  if (rem) snprintf(b, sizeof b, "%04lld-%02u-%02uT%02lld:%02lld:%02lld.%03lldZ", (long long)y, m, d, (long long)(sod / 3600), (long long)(sod % 3600 / 60), (long long)(sod % 60), (long long)rem);
  else snprintf(b, sizeof b, "%04lld-%02u-%02uT%02lld:%02lld:%02lldZ", (long long)y, m, d, (long long)(sod / 3600), (long long)(sod % 3600 / 60), (long long)(sod % 60));
  return b;
}

static void fin_aggs(const std::vector<AggReq>& reqs, const std::vector<IAgg>* aggs, std::string& out);

static void fin_key(const IKey& k, std::string& out) {
  switch (k.kind) {
    case IKey::Str: json_escape(k.s, out); break;
    case IKey::F64: json_f64(k.f, out); break;
    case IKey::I64: out += std::to_string(k.i); break;
    default: out += std::to_string(k.u);
  }
}
static void opt_f64(bool some, double v, std::string& out) { if (some) json_f64(v, out); else out += "null"; }
static std::string range_num(double v) {
  std::string s;
  if (v == std::floor(v) && std::fabs(v) < 1e15) { char b[32]; snprintf(b, sizeof b, "%.0f", v); s = b; }
  else json_f64(v, s);
  return s;
}

static void fin_agg(const AggReq& req, const IAgg* a, std::string& out) {
  IAgg empty;
  empty.kind = (uint8_t)req.kind;
  if (!a) a = &empty;
  if (req.is_metric()) {
    bool some = a->m_count > 0;
    double avg = some ? a->m_sum / (double)a->m_count : 0;
    switch (req.kind) {
      case AggReq::Stats:
        out += "{\"avg\":"; opt_f64(some, avg, out);
        out += ",\"count\":" + std::to_string(a->m_count);
        out += ",\"max\":"; opt_f64(some, a->m_max, out);
        out += ",\"min\":"; opt_f64(some, a->m_min, out);
        out += ",\"sum\":"; json_f64(a->m_sum, out);
        out += "}";
        break;
      case AggReq::Avg: out += "{\"value\":"; opt_f64(some, avg, out); out += "}"; break;
      case AggReq::Sum: out += "{\"value\":"; json_f64(a->m_sum, out); out += "}"; break;
      case AggReq::Min: out += "{\"value\":"; opt_f64(some, a->m_min, out); out += "}"; break;
      case AggReq::Max: out += "{\"value\":"; opt_f64(some, a->m_max, out); out += "}"; break;
      default: out += "{\"value\":"; json_f64((double)a->m_count, out); out += "}"; break;
    }
    return;
  }
  auto subs = [&](const IBucket* b) {
    if (req.children.empty()) return;
    out += ",";
    std::string inner;
    fin_aggs(req.children, b ? &b->subs : nullptr, inner);
    out += inner.substr(1, inner.size() - 2);  // splice the members of {...}
  };
  if (req.kind == AggReq::Terms) {
    std::vector<IBucket> bs = a->buckets;
    sort_term_buckets(req, bs);
    uint64_t sum_other = a->sum_other;
    std::vector<const IBucket*> kept;
    for (auto& b : bs) {
      if (b.count < req.min_doc_count) continue;
      if (kept.size() < req.size) kept.push_back(&b);
      else sum_other += b.count;
    }
    out += "{\"buckets\":[";
    for (size_t i = 0; i < kept.size(); i++) {
      if (i) out += ",";
      out += "{\"doc_count\":" + std::to_string(kept[i]->count) + ",\"key\":";
      fin_key(kept[i]->key, out);
      subs(kept[i]);
      out += "}";
    }
    out += "],\"doc_count_error_upper_bound\":" + std::to_string(a->error_bound) + ",\"sum_other_doc_count\":" + std::to_string(sum_other) + "}";
    return;
  }
  if (req.kind == AggReq::Range) {
    // buckets in request order, plus the open-ended buckets needed to cover the whole axis
    struct RB { bool has_from, has_to; double from, to; std::string key; const IBucket* b; };
    std::vector<RB> rbs;
    for (size_t i = 0; i < req.ranges.size(); i++) {
      const IBucket* b = nullptr;
      for (auto& x : a->buckets) if ((size_t)x.hkey == i) b = &x;
      rbs.push_back({req.ranges[i].has_from, req.ranges[i].has_to, req.ranges[i].from, req.ranges[i].to, req.ranges[i].key, b});
    }
    out += "{\"buckets\":[";
    for (size_t i = 0; i < rbs.size(); i++) {
      if (i) out += ",";
      std::string key = rbs[i].key;
      if (key.empty()) key = (rbs[i].has_from ? range_num(rbs[i].from) : "*") + "-" + (rbs[i].has_to ? range_num(rbs[i].to) : "*");
      out += "{\"doc_count\":" + std::to_string(rbs[i].b ? rbs[i].b->count : 0);
      if (rbs[i].has_from) { out += ",\"from\":"; json_f64(rbs[i].from, out); }
      out += ",\"key\":";
      json_escape(key, out);
      if (rbs[i].has_to) { out += ",\"to\":"; json_f64(rbs[i].to, out); }
      subs(rbs[i].b);
      out += "}";
    }
    out += "]}";
    return;
  }
  // histogram / date_histogram: keys are in column units (ns for dates); output keys in request
  // units (ms for dates), gaps filled when min_doc_count == 0
  const double unit = a->is_date || req.kind == AggReq::DateHistogram ? 1e6 : 1.0;
  const double interval = req.interval * unit, offset = req.offset * unit;
  std::map<int64_t, const IBucket*> by_pos;
  for (auto& b : a->buckets) by_pos[(int64_t)std::llround((b.hkey - offset) / interval)] = &b;
  std::vector<std::pair<int64_t, const IBucket*>> seq;
  if (req.min_doc_count == 0) {
    bool any = !by_pos.empty();
    int64_t lo = any ? by_pos.begin()->first : 0, hi = any ? by_pos.rbegin()->first : -1;
    if (req.has_extended_bounds) {
      int64_t elo = (int64_t)std::floor((req.ext_min * unit - offset) / interval), ehi = (int64_t)std::floor((req.ext_max * unit - offset) / interval);
      if (elo <= ehi) {
        if (!any) { lo = elo; hi = ehi; any = true; }
        else { lo = std::min(lo, elo); hi = std::max(hi, ehi); }
      }
    }
    if (any) {
      if (hi - lo > 65000) fail(QWGPU_EINVALID_AGG, "aborting aggregation: too many histogram buckets (%lld)", (long long)(hi - lo + 1));
      for (int64_t p = lo; p <= hi; p++) {
        auto it = by_pos.find(p);
        seq.push_back({p, it == by_pos.end() ? nullptr : it->second});
      }
    }
  } else {
    for (auto& kv : by_pos) if (kv.second->count >= req.min_doc_count) seq.push_back(kv);
  }
  out += "{\"buckets\":[";
  bool first = true;
  for (auto& kv : seq) {
    double key = ((double)kv.first * interval + offset) / unit;
    if (req.has_hard_bounds && (key < req.hard_min || key > req.hard_max) && !kv.second) continue;
    if (!first) out += ",";
    first = false;
    out += "{\"doc_count\":" + std::to_string(kv.second ? kv.second->count : 0) + ",\"key\":";
    json_f64(key, out);
    if (req.kind == AggReq::DateHistogram) { out += ",\"key_as_string\":"; json_escape(rfc3339_from_ms(key), out); }
    subs(kv.second);
    out += "}";
  }
  out += "]}";
}

static void fin_aggs(const std::vector<AggReq>& reqs, const std::vector<IAgg>* aggs, std::string& out) {
  out += "{";
  for (size_t i = 0; i < reqs.size(); i++) {
    if (i) out += ",";
    json_escape(reqs[i].name, out);
    out += ":";
    fin_agg(reqs[i], aggs && i < aggs->size() ? &(*aggs)[i] : nullptr, out);
  }
  out += "}";
}

std::string finalize_aggs_json(const std::vector<AggReq>& reqs, const std::string& intermediate) {
  std::vector<IAgg> top;
  if (!intermediate.empty()) top = de_top(intermediate);
  if (!top.empty() && top.size() != reqs.size()) fail(QWGPU_EINTERNAL, "intermediate aggregation result does not match the request");
  std::string out;
  fin_aggs(reqs, top.empty() ? nullptr : &top, out);
  return out;
}

}  // namespace qw
