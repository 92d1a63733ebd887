// engine.cu — host engine: HBM residency of split images, lowering of seam-C plans into the
// window-engine program, batched launches (one launch sequence covers every split of a request),
// top-K threshold selection (sampled fast path + exact radix-select fallback) and result readback.
//
// Replaces, for one leaf request: open_index_with_caches + warmup (quickwit-search/src/leaf.rs:
// 210-251,269-472) at register time, and searcher.search(&query,&collector) (leaf.rs:637) per call.
#include <algorithm>
#include <chrono>
#include <cmath>

#include "engine.h"
#include "kernels.cuh"
#include "union_kernel.cuh"
#include "phrase_kernel.cuh"
#include "driver_kernel.cuh"
#include "agg_kernel.cuh"

namespace qw {

#define CUDA_CHECK(expr)                                                                          \
  do {                                                                                            \
    cudaError_t _e = (expr);                                                                      \
    if (_e != cudaSuccess)                                                                        \
      fail((_e == cudaErrorNoDevice || _e == cudaErrorInsufficientDriver) ? QWGPU_ENODEVICE       \
                                                                           : QWGPU_EINTERNAL,     \
           "CUDA error %s at %s:%d: %s", cudaGetErrorName(_e), __FILE__, __LINE__,               \
           cudaGetErrorString(_e));                                                               \
  } while (0)

uint32_t id_to_fieldnorm(uint8_t id);  // image_builder.cpp

SplitDev::~SplitDev() {
  if (d_data) cudaFree(d_data);
  if (d_tabs) cudaFree(d_tabs);
}

struct CallSlot {
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr, ev3 = nullptr;
  cudaEvent_t ev_block = nullptr;  // cudaEventBlockingSync: waits that yield the CPU (many calls in flight)
  uint8_t *d_blob = nullptr, *h_blob = nullptr;
  size_t blob_cap = 0;
  uint8_t* d_scratch = nullptr;
  size_t scratch_cap = 0;
  uint8_t *d_out = nullptr, *h_out = nullptr;
  size_t out_cap = 0;
  void ensure(size_t blob, size_t scratch, size_t out) {
    if (blob > blob_cap) {
      if (d_blob) cudaFree(d_blob);
      if (h_blob) cudaFreeHost(h_blob);
      blob_cap = blob * 2;
      CUDA_CHECK(cudaMalloc(&d_blob, blob_cap));
      CUDA_CHECK(cudaMallocHost(&h_blob, blob_cap));
    }
    if (scratch > scratch_cap) {
      if (d_scratch) cudaFree(d_scratch);
      scratch_cap = scratch * 2;
      CUDA_CHECK(cudaMalloc(&d_scratch, scratch_cap));
    }
    if (out > out_cap) {
      if (d_out) cudaFree(d_out);
      if (h_out) cudaFreeHost(h_out);
      out_cap = out * 2;
      CUDA_CHECK(cudaMalloc(&d_out, out_cap));
      CUDA_CHECK(cudaMallocHost(&h_out, out_cap));
    }
  }
  ~CallSlot() {
    if (d_blob) cudaFree(d_blob);
    if (h_blob) cudaFreeHost(h_blob);
    if (d_scratch) cudaFree(d_scratch);
    if (d_out) cudaFree(d_out);
    if (h_out) cudaFreeHost(h_out);
    if (ev0) cudaEventDestroy(ev0);
    if (ev_block) cudaEventDestroy(ev_block);
    if (ev1) cudaEventDestroy(ev1);
    if (ev2) cudaEventDestroy(ev2);
    if (ev3) cudaEventDestroy(ev3);
    if (stream) cudaStreamDestroy(stream);
  }
};

Engine::Engine(int dev) : device(dev) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0)
    fail(QWGPU_ENODEVICE, "no CUDA device available (%s); the qwgpu search path has no CPU fallback",
         e == cudaSuccess ? "0 devices" : cudaGetErrorString(e));
  if (dev >= n) fail(QWGPU_EINVALID_ARG, "device %d out of range (%d devices)", dev, n);
  CUDA_CHECK(cudaSetDevice(dev));
  cudaDeviceProp prop;
  CUDA_CHECK(cudaGetDeviceProperties(&prop, dev));
  sm_count = prop.multiProcessorCount;
  max_smem_optin = (int)prop.sharedMemPerBlockOptin;
  CUDA_CHECK(cudaFuncSetAttribute(qwk::k_window<qwk::MODE_HIST, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem_optin));
  CUDA_CHECK(cudaFuncSetAttribute(qwk::k_window<qwk::MODE_COLLECT, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem_optin));
  CUDA_CHECK(cudaFuncSetAttribute(qwk::k_window<qwk::MODE_COLLECT, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem_optin));
  CUDA_CHECK(cudaFuncSetAttribute(qwk::k_window<qwk::MODE_HIST, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem_optin));
  CUDA_CHECK(cudaFuncSetAttribute(qwk::k_union<qwk::MODE_HIST>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem_optin));
  CUDA_CHECK(cudaFuncSetAttribute(qwk::k_union<qwk::MODE_COLLECT>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem_optin));
  CUDA_CHECK(cudaFuncSetAttribute(qwk::k_aggscan, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem_optin));
  CUDA_CHECK(cudaFuncSetAttribute(qwk::k_select, cudaFuncAttributeMaxDynamicSharedMemorySize, 3 * 8 * QW_CAND_CAP));
}

Engine::~Engine() {
  for (Loader& l : loaders) if (l.t.joinable()) l.t.join();
  cudaSetDevice(device);
  for (CallSlot* s : free_slots) delete s;
  splits.clear();
}

// host half of a registration: directory copy + views (no device work)
static std::shared_ptr<SplitDev> open_split(const char* id, const uint8_t* img, uint64_t len, ImageView* full_out) {
  ImageView full;
  full.open(img, len);
  auto sp = std::make_shared<SplitDev>();
  sp->id = id;
  sp->dir.assign(img, img + full.hdr->data_off);
  // the directory-only view: relax the length check by opening over the original then rebasing
  sp->view = full;
  sp->view.base = sp->dir.data();
  sp->view.hdr = (const QwImgHeader*)sp->dir.data();
  sp->view.fields = (const QwImgField*)(sp->dir.data() + full.hdr->fields_off);
  sp->view.terms = (const QwImgTerm*)(sp->dir.data() + full.hdr->terms_off);
  sp->view.columns = (const QwImgColumn*)(sp->dir.data() + full.hdr->columns_off);
  sp->view.term_bytes = sp->dir.data() + full.hdr->term_bytes_off;
  sp->view.strings = sp->dir.data() + full.hdr->strings_off;
  sp->view.data = nullptr;
  sp->data_len = full.hdr->data_len;
  *full_out = full;
  return sp;
}

// Bm25Weight cache per field (SURVEY.md Appendix A.3): K1 * (1 - B + B * fieldnorm(id) / avg), followed, per field,
// by the tf-factor table tff[tf][id] = tf / (tf + norm[id]) (tf < 16), built with the same IEEE f32 ops the kernel
// would use, so table lookups are bit-identical to dividing
static std::vector<float> bm25_tables(const ImageView& full) {
  const uint32_t nf = full.hdr->num_fields;
  const size_t kTab = 256 + QW_TFF_ROWS * 256;
  std::vector<float> tabs((size_t)std::max(nf, 1u) * kTab);
  for (uint32_t f = 0; f < nf; f++) {
    // an empty split scores nothing; keep its tables finite
    float avg = full.hdr->num_docs ? (float)full.fields[f].total_num_tokens / (float)full.hdr->num_docs : 1.0f;
    float* t = tabs.data() + f * kTab;
    for (uint32_t i = 0; i < 256; i++)
      t[i] = BM25_K1 * (1.0f - BM25_B + BM25_B * (float)id_to_fieldnorm((uint8_t)i) / avg);
    for (uint32_t tf = 0; tf < QW_TFF_ROWS; tf++)
      for (uint32_t i = 0; i < 256; i++) {
        volatile float num = (float)tf, den = (float)tf + t[i];
        t[256 + tf * 256 + i] = num / den;
      }
  }
  return tabs;
}

// Makes room for `need` more bytes under the budget: drops the least recently searched splits that nothing but
// the table references (a split in use by a running call, or still loading, stays). Caller holds `mu`.
static void evict_for(Engine& e, uint64_t need, const std::string& keep) {
  if (!e.budget) return;
  while (e.resident + need > e.budget) {
    auto victim = e.splits.end();
    for (auto it = e.splits.begin(); it != e.splits.end(); ++it) {
      if (it->first == keep || it->second.use_count() > 1 || it->second->state == 0) continue;
      if (victim == e.splits.end() || it->second->last_use < victim->second->last_use) victim = it;
    }
    if (victim == e.splits.end()) break;  // everything left is in use: over budget until those calls end
    e.resident -= victim->second->data_len;
    e.splits.erase(victim);
    e.evictions++;
  }
}

static void publish(Engine& e, const std::shared_ptr<SplitDev>& sp) {
  auto it = e.splits.find(sp->id);
  if (it != e.splits.end()) e.resident -= it->second->data_len;
  sp->last_use = ++e.tick;
  e.splits[sp->id] = sp;
  e.resident += sp->data_len;
}

void Engine::register_split(const char* id, const uint8_t* img, uint64_t len) {
  ImageView full;
  auto sp = open_split(id, img, len, &full);
  {
    std::lock_guard<std::mutex> g(mu);
    if (budget && sp->data_len > budget) fail(QWGPU_EINVALID_ARG, "split `%s` needs %llu bytes, the residency budget is %llu", id, (unsigned long long)sp->data_len, (unsigned long long)budget);
    evict_for(*this, sp->data_len, sp->id);
  }
  CUDA_CHECK(cudaSetDevice(device));
  CUDA_CHECK(cudaMalloc(&sp->d_data, std::max<uint64_t>(sp->data_len, 16)));
  CUDA_CHECK(cudaMemcpy(sp->d_data, full.data, sp->data_len, cudaMemcpyHostToDevice));
  std::vector<float> tabs = bm25_tables(full);
  CUDA_CHECK(cudaMalloc(&sp->d_tabs, tabs.size() * sizeof(float)));
  CUDA_CHECK(cudaMemcpy(sp->d_tabs, tabs.data(), tabs.size() * sizeof(float), cudaMemcpyHostToDevice));
  std::lock_guard<std::mutex> g(mu);
  publish(*this, sp);
}

// Background upload: the split is visible (loading) at once; a loader thread stages the data region through two
// pinned buffers (pageable -> pinned memcpy of chunk i+1 overlaps the DMA of chunk i) on its own stream, so
// searches on other splits keep the GPU while a cold split comes in (leaf.rs:269-472 warmup runs beside searches).
void Engine::register_split_async(const char* id, const uint8_t* img, uint64_t len) {
  ImageView full;
  auto sp = open_split(id, img, len, &full);
  sp->state = 0;
  {
    std::lock_guard<std::mutex> g(mu);
    if (budget && sp->data_len > budget) fail(QWGPU_EINVALID_ARG, "split `%s` needs %llu bytes, the residency budget is %llu", id, (unsigned long long)sp->data_len, (unsigned long long)budget);
    evict_for(*this, sp->data_len, sp->id);
  }
  CUDA_CHECK(cudaSetDevice(device));
  CUDA_CHECK(cudaMalloc(&sp->d_data, std::max<uint64_t>(sp->data_len, 16)));
  std::vector<float> tabs = bm25_tables(full);
  CUDA_CHECK(cudaMalloc(&sp->d_tabs, tabs.size() * sizeof(float)));
  std::lock_guard<std::mutex> g(mu);
  publish(*this, sp);
  // loaders that have finished (state set, lock released) are reaped here
  for (size_t i = 0; i < loaders.size();) {
    if (loaders[i].sp->state != 0) { loaders[i].t.join(); loaders[i] = std::move(loaders.back()); loaders.pop_back(); }
    else i++;
  }
  loaders.push_back(Loader{std::thread(), sp});
  loaders.back().t = std::thread([this, sp, full, tabs]() {
    std::string err;
    cudaStream_t st = nullptr;
    uint8_t* pin[2] = {nullptr, nullptr};
    cudaEvent_t ev[2] = {nullptr, nullptr};
    const size_t kChunk = 8u << 20;
    auto ok = [&](cudaError_t e, const char* what) { if (e != cudaSuccess && err.empty()) err = std::string(what) + ": " + cudaGetErrorString(e); return e == cudaSuccess; };
    if (ok(cudaSetDevice(device), "cudaSetDevice") && ok(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking), "cudaStreamCreate")) {
      for (int i = 0; i < 2; i++) { ok(cudaMallocHost(&pin[i], kChunk), "cudaMallocHost"); ok(cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming), "cudaEventCreate"); }
      uint64_t off = 0;
      for (int k = 0; err.empty() && off < sp->data_len; k ^= 1) {
        const size_t nb = (size_t)std::min<uint64_t>(kChunk, sp->data_len - off);
        ok(cudaEventSynchronize(ev[k]), "upload event");  // the DMA that last used this buffer is done
        memcpy(pin[k], full.data + off, nb);
        ok(cudaMemcpyAsync(sp->d_data + off, pin[k], nb, cudaMemcpyHostToDevice, st), "H2D of the split data");
        ok(cudaEventRecord(ev[k], st), "upload event");
        off += nb;
      }
      ok(cudaMemcpyAsync(sp->d_tabs, tabs.data(), tabs.size() * sizeof(float), cudaMemcpyHostToDevice, st), "H2D of the BM25 tables");
      ok(cudaStreamSynchronize(st), "upload stream");
    }
    for (int i = 0; i < 2; i++) { if (pin[i]) cudaFreeHost(pin[i]); if (ev[i]) cudaEventDestroy(ev[i]); }
    if (st) cudaStreamDestroy(st);
    {
      std::lock_guard<std::mutex> g2(mu);
      sp->load_error = err;
      sp->state = err.empty() ? 1 : 2;
    }
    loaded_cv.notify_all();
  });
}

void Engine::wait_split(const char* id) {
  std::unique_lock<std::mutex> g(mu);
  auto it = splits.find(id);
  if (it == splits.end()) fail(QWGPU_ENOTFOUND, "split '%s' is not registered", id);
  std::shared_ptr<SplitDev> sp = it->second;
  loaded_cv.wait(g, [&] { return sp->state != 0; });
  if (sp->state == 2) fail(QWGPU_EINTERNAL, "upload of split '%s' failed: %s", id, sp->load_error.c_str());
}

void Engine::set_budget(uint64_t bytes) {
  std::lock_guard<std::mutex> g(mu);
  budget = bytes;
  evict_for(*this, 0, "");
}

void Engine::unregister_split(const char* id) {
  std::unique_lock<std::mutex> g(mu);
  auto it = splits.find(id);
  if (it == splits.end()) fail(QWGPU_ENOTFOUND, "split '%s' is not registered", id);
  std::shared_ptr<SplitDev> sp = it->second;
  loaded_cv.wait(g, [&] { return sp->state != 0; });  // (its loader still writes the device buffer)
  it = splits.find(id);
  if (it != splits.end() && it->second == sp) { resident -= sp->data_len; splits.erase(it); }
}

// A search takes the split in use: recency for the LRU; a split that is still loading is waited for.
std::shared_ptr<SplitDev> Engine::find(const std::string& id) {
  std::unique_lock<std::mutex> g(mu);
  auto it = splits.find(id);
  if (it == splits.end()) return nullptr;
  std::shared_ptr<SplitDev> sp = it->second;
  loaded_cv.wait(g, [&] { return sp->state != 0; });
  if (sp->state == 2) return nullptr;
  sp->last_use = ++tick;
  return sp;
}

uint64_t agg_cell_layout(const QwAggNode* aggs, uint32_t n, std::vector<uint32_t>* bases) {
  uint64_t total = 0;
  if (bases) bases->resize(n);
  for (uint32_t i = 0; i < n; i++) {
    uint64_t cells = aggs[i].kind == QW_AGG_STATS ? 1 : aggs[i].num_buckets;
    uint32_t p = aggs[i].parent;
    while (p != 0xFFFFFFFFu) { cells *= aggs[p].num_buckets; p = aggs[p].parent; }
    if (bases) (*bases)[i] = (uint32_t)total;
    total += cells;
    if (total > (1ull << 26)) fail(QWGPU_EINVALID_AGG, "aggregation bucket space too large (%llu cells)", (unsigned long long)total);
  }
  return total;
}

// ---- lowering: QwPlan tree -> window-engine program ----------------------------------------------
// kernels.cuh mapped_to_f64 on the host (tantivy MonotonicallyMappableToU64 inverses, as f64)
static double mapped_to_f64_host(uint32_t type, uint64_t m) {
  switch (type) {
    case QW_COL_U64: case QW_COL_BOOL: case QW_COL_STR: return (double)m;
    case QW_COL_I64: case QW_COL_DATETIME: return (double)(int64_t)(m ^ (1ull << 63));
    default: return u64_to_f64(m);
  }
}

struct Lowered {
  DSplitPlan P;
  std::vector<DInstr> instrs;
  std::vector<DCol> cols;
  std::vector<uint64_t> bounds;  // raw-space histogram boundary tables of the fast aggregation path
  uint32_t bounds_base = 0;      // position of `bounds` in the batch's table region
  std::vector<uint64_t> col_max_raw;  // parallel to cols: largest bit-packed raw value present in the column
  std::vector<DAgg> aggs;
  std::vector<int> col_map;  // image column -> DCol index
  uint32_t need_cnt = 0, need_ssum = 0, need_msum = 0, levels = 0;  // bit per level
  float score_max = 0.f;
  int fn_field[2] = {-1, -1};
  uint64_t postings = 0, alg_bytes = 0, min_required_df = ~0ull;
  std::vector<std::pair<uint32_t, uint64_t>> range_cols;  // (col, driver df) for roofline accounting
  bool empty = false;                   // a required clause of the root cannot match in this split: no work at all
  std::vector<DPhrase> phrases;         // phrase pre-pass descriptors (out / first_work filled per batch)
  std::vector<uint32_t> phrase_instr;   // instruction that consumes phrases[i]
};

static uint32_t use_col(Lowered& L, const SplitDev& sp, uint32_t c) {
  if (c == 0xFFFFFFFFu) return c;
  if (c >= sp.view.hdr->num_columns) fail(QWGPU_EINVALID_ARG, "plan references column %u (split has %u)", c, sp.view.hdr->num_columns);
  if (L.col_map[c] >= 0) return (uint32_t)L.col_map[c];
  if (L.cols.size() >= QW_MAX_DCOLS) fail(QWGPU_EUNSUPPORTED, "plan uses more than %d columns", QW_MAX_DCOLS);
  const QwImgColumn& ic = sp.view.columns[c];
  DCol d;
  d.values_off = ic.values_off; d.index_off = ic.index_off; d.min_value = ic.min_value; d.gcd = ic.gcd;
  d.bits = ic.bits; d.card = ic.cardinality; d.type = ic.type; d.nwords64 = (sp.view.hdr->num_docs + 63) / 64;
  L.col_map[c] = (int)L.cols.size();
  L.cols.push_back(d);
  L.col_max_raw.push_back(ic.gcd ? (ic.max_value - ic.min_value) / ic.gcd : 0);
  return (uint32_t)L.col_map[c];
}

static void lower_node(Lowered& L, const SplitDev& sp, const QwPlanNode* nodes, uint32_t nn, uint32_t idx,
                       uint32_t level, uint32_t occur, bool scored_ctx) {
  if (idx >= nn) fail(QWGPU_EINVALID_ARG, "plan node index out of range");
  const QwPlanNode& n = nodes[idx];
  const bool scored = scored_ctx && (occur == QW_OCCUR_MUST || occur == QW_OCCUR_SHOULD);
  DInstr in;
  memset(&in, 0, sizeof in);
  in.level = level;
  in.occur = occur;
  in.flags = scored ? IF_SCORED : 0;
  switch (n.kind) {
    case QW_NODE_TERM: {
      in.op = OP_TERM;
      if (n.term_ord == 0xFFFFFFFFu && level == 0 && (occur == QW_OCCUR_MUST || occur == QW_OCCUR_FILTER)) L.empty = true;
      in.t = L.P.n_terms++;
      if (L.P.n_terms > QW_MAX_TERMS) fail(QWGPU_EUNSUPPORTED, "more than %d term clauses", QW_MAX_TERMS);
      in.r = 0;
      if (n.term_ord != 0xFFFFFFFFu) {
        if (n.term_ord >= sp.view.hdr->num_terms) fail(QWGPU_EINVALID_ARG, "plan term ord out of range");
        const QwImgTerm& t = sp.view.terms[n.term_ord];
        const QwImgField& f = sp.view.fields[t.field_id];
        in.a = t.data_off; in.b = t.widx_off; in.c = t.skip_off;
        in.n = t.num_blocks; in.m = t.win_shift; in.f = n.bm25_weight;
        in.pad = (uint32_t)((t.sub_off - t.skip_off) >> 4);  // QwSubIdx[] relative to QwSkip[], in 16-byte units
        if (f.flags & QW_FIELD_HAS_FREQS) in.flags |= IF_HAS_TF;
        if (f.flags & QW_FIELD_HAS_FIELDNORMS) in.flags |= IF_HAS_FN;
        L.postings += t.doc_freq;
        L.alg_bytes += t.data_len - t.fn_len - (scored ? 0 : t.tf_len);  // fieldnorm bytes are counted once per plan below
        if (occur == QW_OCCUR_MUST || occur == QW_OCCUR_FILTER) L.min_required_df = std::min<uint64_t>(L.min_required_df, t.doc_freq);
        if (scored) {
          int slot = -1;
          for (int s = 0; s < 2; s++) if (L.fn_field[s] == (int)t.field_id) slot = s;
          if (slot < 0) {
            for (int s = 0; s < 2 && slot < 0; s++) if (L.fn_field[s] < 0) { L.fn_field[s] = (int)t.field_id; slot = s; }
            if (slot < 0) fail(QWGPU_EUNSUPPORTED, "scoring over more than 2 distinct text fields");
          }
          in.r = (uint32_t)slot;
          L.score_max += n.bm25_weight > 0 ? n.bm25_weight : 0.f;
        }
      }
      L.instrs.push_back(in);
      break;
    }
    case QW_NODE_RANGE: case QW_NODE_EXISTS: case QW_NODE_ALL: case QW_NODE_NONE: {
      if (n.kind == QW_NODE_NONE) { in.op = OP_EXISTS; in.r = 0xFFFFFFFFu; }  // matches nothing
      else if (n.kind == QW_NODE_ALL) in.op = OP_ALL;
      else {
        in.op = n.kind == QW_NODE_RANGE ? OP_RANGE : OP_EXISTS;
        in.r = use_col(L, sp, n.column);
        in.a = n.lo; in.b = n.hi;
        if (n.column != 0xFFFFFFFFu) L.range_cols.push_back({n.column, 0});
        // a range that misses the column's [min, max] (the split's own value range) matches nothing
        if (n.kind == QW_NODE_RANGE && n.column != 0xFFFFFFFFu) {
          const QwImgColumn& ic = sp.view.columns[n.column];
          if (ic.num_vals == 0 || n.hi < ic.min_value || n.lo > ic.max_value) in.r = 0xFFFFFFFFu;
        }
      }
      // a required clause at the root that cannot match: the split has no hits (its windows are skipped)
      if (in.r == 0xFFFFFFFFu && in.op != OP_ALL && level == 0 && (occur == QW_OCCUR_MUST || occur == QW_OCCUR_FILTER)) L.empty = true;
      in.f = n.boost;
      if (scored) L.score_max += n.boost > 0 ? n.boost : 0.f;
      L.instrs.push_back(in);
      break;
    }
    case QW_NODE_BOOL: {
      if (level + 1 > QW_MAX_LEVELS) fail(QWGPU_EUNSUPPORTED, "boolean query nested deeper than %d levels", QW_MAX_LEVELS);
      // the bool's own accumulators live at `level`; when it is a child, the caller passed level+1
      DInstr bg;
      memset(&bg, 0, sizeof bg);
      bg.op = OP_BOOL_BEGIN; bg.level = level;
      L.instrs.push_back(bg);
      const size_t first_instr = L.instrs.size();
      L.levels |= 1u << level;
      uint32_t n_req = 0, n_should = 0;
      if (n.first_child + n.num_children > nn) fail(QWGPU_EINVALID_ARG, "plan children out of range");
      // required group: scored MUST clauses in plan order first (fixes the f32 summation order),
      // then unscored required clauses, posting lists before column predicates (so range filters
      // only probe surviving candidates)
      std::vector<uint32_t> order;
      auto child = [&](uint32_t c) -> const QwPlanNode& { return nodes[n.first_child + c]; };
      auto is_req = [&](uint32_t c) { return child(c).occur == QW_OCCUR_MUST || child(c).occur == QW_OCCUR_FILTER; };
      auto is_colpred = [&](uint32_t c) { return child(c).kind == QW_NODE_RANGE || child(c).kind == QW_NODE_EXISTS || child(c).kind == QW_NODE_ALL; };
      const bool child_scored_ctx = scored_ctx;
      for (uint32_t c = 0; c < n.num_children; c++) if (is_req(c) && child_scored_ctx && child(c).occur == QW_OCCUR_MUST) order.push_back(c);
      for (int pass = 0; pass < 2; pass++)
        for (uint32_t c = 0; c < n.num_children; c++)
          if (is_req(c) && !(child_scored_ctx && child(c).occur == QW_OCCUR_MUST) && (is_colpred(c) ? pass == 1 : pass == 0)) order.push_back(c);
      if (child_scored_ctx) {
        // scored column predicates must also come after posting lists only when that keeps order;
        // scored clauses keep plan order, so nothing to do here
      }
      n_req = (uint32_t)order.size();
      for (uint32_t c = 0; c < n.num_children; c++) if (child(c).occur == QW_OCCUR_SHOULD) { order.push_back(c); n_should++; }
      for (uint32_t c = 0; c < n.num_children; c++) if (child(c).occur == QW_OCCUR_MUST_NOT) order.push_back(c);
      for (uint32_t c : order) {
        const QwPlanNode& cn = child(c);
        uint32_t child_level = cn.kind == QW_NODE_BOOL ? level + 1 : level;
        if (scored && cn.occur == QW_OCCUR_MUST) L.need_msum |= 1u << level;
        if (scored && cn.occur == QW_OCCUR_SHOULD) L.need_ssum |= 1u << level;
        lower_node(L, sp, nodes, nn, n.first_child + c, child_level, cn.occur, scored);
      }
      uint32_t msm = n.min_should_match == 0xFFFFFFFFu ? 0 : n.min_should_match;
      uint32_t need = msm > 0 ? msm : (n_req == 0 ? 1 : 0);
      if (need >= 2) L.need_cnt |= 1u << level;
      // Scored should-TERMs with a strictly positive weight contribute > 0 to ssum for every matching
      // doc, so their bitmap is (ssum > 0): skip the per-posting bit set and rebuild it at BOOL_END.
      bool any_from_score = false;
      if (need < 2 && scored) {
        for (size_t ii = first_instr; ii < L.instrs.size(); ii++) {
          DInstr& ci = L.instrs[ii];
          if (ci.op == OP_TERM && ci.level == level && ci.occur == QW_OCCUR_SHOULD && (ci.flags & IF_SCORED) && ci.f >= 1e-20f && ci.f < 1e30f) {
            ci.flags |= IF_BITS_FROM_SCORE;
            any_from_score = true;
          }
        }
      }
      DInstr en;
      memset(&en, 0, sizeof en);
      en.op = OP_BOOL_END; en.level = level; en.occur = occur; en.flags = (scored ? IF_SCORED : 0) | (any_from_score ? IF_BITS_FROM_SCORE : 0);
      en.n = n_req; en.m = n_should; en.r = need;
      L.instrs.push_back(en);
      break;
    }
    case QW_NODE_PHRASE: {
      // evaluated by the pre-pass (phrase_kernel.cuh) into one uncompressed posting block per block of its
      // rarest term; the window program consumes those blocks (OP_PHRASE)
      if (n.num_children < 2 || n.num_children > QW_MAX_PHRASE_TERMS || n.first_child + n.num_children > nn)
        fail(QWGPU_EINVALID_ARG, "phrase node with %u terms", n.num_children);
      DPhrase ph;
      memset(&ph, 0, sizeof ph);
      ph.data_base = (uint64_t)sp.d_data;
      ph.n_terms = n.num_children;
      ph.weight = n.bm25_weight;
      ph.scored = scored ? 1 : 0;
      uint64_t best_df = ~0ull;
      const QwImgField* fld = nullptr;
      uint32_t field_id = 0;
      for (uint32_t k = 0; k < n.num_children; k++) {
        const QwPlanNode& c = nodes[n.first_child + k];
        if (c.kind != QW_NODE_TERM || c.term_ord >= sp.view.hdr->num_terms) fail(QWGPU_EINVALID_ARG, "phrase term %u is not a term of this split", k);
        const QwImgTerm& t = sp.view.terms[c.term_ord];
        if (!t.pidx_off) fail(QWGPU_EINVALID_ARG, "phrase over a field without positions");
        if (k && t.field_id != field_id) fail(QWGPU_EINVALID_ARG, "phrase terms of different fields");
        field_id = t.field_id;
        fld = &sp.view.fields[t.field_id];
        ph.t[k].data_off = t.data_off; ph.t[k].skip_off = t.skip_off; ph.t[k].pos_off = t.pos_off; ph.t[k].pidx_off = t.pidx_off;
        ph.t[k].nblk = t.num_blocks; ph.t[k].offset = (uint32_t)c.lo;
        if (t.doc_freq < best_df) { best_df = t.doc_freq; ph.driver = k; }
        L.alg_bytes += t.data_len - t.fn_len;
      }
      const QwImgTerm& drv = sp.view.terms[nodes[n.first_child + ph.driver].term_ord];
      L.postings += drv.doc_freq;
      L.alg_bytes += (uint64_t)drv.doc_freq * 4 * n.num_children;  // positions probed per candidate (lower bound)
      if (occur == QW_OCCUR_MUST || occur == QW_OCCUR_FILTER) L.min_required_df = std::min<uint64_t>(L.min_required_df, drv.doc_freq);
      ph.fn_off = (fld->flags & QW_FIELD_HAS_FIELDNORMS) ? fld->fieldnorm_off : ~0ull;
      ph.tab = (uint64_t)(sp.d_tabs + (size_t)(256 + QW_TFF_ROWS * 256) * field_id);
      in.op = OP_PHRASE;
      in.c = drv.skip_off;
      in.n = drv.num_blocks;
      in.f = n.bm25_weight;
      if (scored) L.score_max += n.bm25_weight > 0 ? n.bm25_weight : 0.f;
      L.phrase_instr.push_back((uint32_t)L.instrs.size());
      L.phrases.push_back(ph);
      L.instrs.push_back(in);
      break;
    }
    default: fail(QWGPU_EINVALID_ARG, "unknown plan node kind %u", n.kind);
  }
}

static inline uint32_t bits_needed64(uint64_t v) { return v == 0 ? 0 : 64 - __builtin_clzll(v); }

static void lower_plan(Lowered& L, const SplitDev& sp, const uint8_t* plan, size_t plan_len) {
  if (plan_len < sizeof(QwPlanHeader)) fail(QWGPU_EINVALID_ARG, "plan too short");
  const QwPlanHeader* ph = (const QwPlanHeader*)plan;
  if (ph->magic != QW_PLAN_MAGIC) fail(QWGPU_EINVALID_ARG, "bad plan magic");
  size_t need = sizeof(QwPlanHeader) + (size_t)ph->num_nodes * sizeof(QwPlanNode) + (size_t)ph->num_aggs * sizeof(QwAggNode);
  if (plan_len < need || ph->num_nodes == 0) fail(QWGPU_EINVALID_ARG, "plan truncated");
  if (ph->max_hits > QW_MAX_TOPK) fail(QWGPU_EUNSUPPORTED, "max_hits + start_offset = %u exceeds the GPU top-K limit %d", ph->max_hits, QW_MAX_TOPK);
  const QwPlanNode* nodes = (const QwPlanNode*)(plan + sizeof(QwPlanHeader));
  const QwAggNode* aggs = (const QwAggNode*)(nodes + ph->num_nodes);
  memset(&L.P, 0, sizeof L.P);
  L.col_map.assign(sp.view.hdr->num_columns, -1);
  DSplitPlan& P = L.P;
  P.data_base = (uint64_t)sp.d_data;
  P.num_docs = sp.view.hdr->num_docs;
  P.max_hits = ph->max_hits;
  P.scoring = ph->scoring;
  P.sa = ph->search_after;
  const bool scoring = ph->scoring != 0;
  if (nodes[0].kind == QW_NODE_BOOL) {
    lower_node(L, sp, nodes, ph->num_nodes, 0, 0, QW_OCCUR_MUST, scoring);
  } else if (nodes[0].kind == QW_NODE_TERM && scoring) {
    // a scored single-term query is the one-clause case of the BM25 union: lower it as
    // bool{should: [term]} so that it takes the UNION kernels (same matches, same f32 score)
    QwPlanNode wrap[2];
    memset(wrap, 0, sizeof wrap);
    wrap[0].kind = QW_NODE_BOOL; wrap[0].occur = QW_OCCUR_MUST; wrap[0].boost = 1.0f;
    wrap[0].first_child = 1; wrap[0].num_children = 1; wrap[0].min_should_match = 0xFFFFFFFFu;
    wrap[1] = nodes[0];
    wrap[1].occur = QW_OCCUR_SHOULD;
    lower_node(L, sp, wrap, 2, 0, 0, QW_OCCUR_MUST, scoring);
  } else {
    DInstr bg; memset(&bg, 0, sizeof bg); bg.op = OP_BOOL_BEGIN; L.instrs.push_back(bg);
    L.levels |= 1;
    if (scoring) L.need_msum |= 1;
    lower_node(L, sp, nodes, ph->num_nodes, 0, 0, QW_OCCUR_MUST, scoring);
    DInstr en; memset(&en, 0, sizeof en); en.op = OP_BOOL_END; en.n = 1; en.flags = scoring ? IF_SCORED : 0; L.instrs.push_back(en);
  }
  {
    // root bool == pure OR of positive-weight scored terms (the BM25 top-K shape): the collect pass can
    // take matches, hit count and the next window's zeroed accumulator straight from the score array
    const DInstr& last = L.instrs.back();
    bool pure = last.op == OP_BOOL_END && last.level == 0 && (last.flags & IF_BITS_FROM_SCORE) && last.n == 0 && last.r == 1;
    for (const DInstr& in : L.instrs) {
      if (in.op == OP_BOOL_BEGIN || in.op == OP_BOOL_END) { if (in.level != 0) pure = false; continue; }
      if (!(in.op == OP_TERM && in.occur == QW_OCCUR_SHOULD && (in.flags & IF_BITS_FROM_SCORE))) pure = false;
    }
    L.P.fused_score_root = pure ? 1 : 0;
  }
  if (L.instrs.size() > QW_MAX_INSTR) fail(QWGPU_EUNSUPPORTED, "query too large for the GPU program (%zu > %d instructions)", L.instrs.size(), QW_MAX_INSTR);
  P.n_instr = (uint32_t)L.instrs.size();
  uint32_t nl = 0;
  while (L.levels >> nl) nl++;
  P.n_levels = nl;
  // fieldnorm / BM25 slots
  for (int s = 0; s < 2; s++) {
    P.fn_off[s] = ~0ull;
    if (L.fn_field[s] >= 0) {
      const QwImgField& f = sp.view.fields[L.fn_field[s]];
      P.n_fn_slots = s + 1;
      P.bm25_tab[s] = (uint64_t)(sp.d_tabs + (size_t)(256 + QW_TFF_ROWS * 256) * L.fn_field[s]);
      if (f.flags & QW_FIELD_HAS_FIELDNORMS) {
        P.fn_off[s] = f.fieldnorm_off;
        L.alg_bytes += std::min<uint64_t>(L.postings, P.num_docs);
      }
    }
  }
  // sort / key spec (sort_by_from_request, quickwit-search/src/collector.rs:994-1030)
  DKeySpec& ks = P.key;
  for (int i = 0; i < 2; i++) {
    ks.kind[i] = ph->sort[i].kind; ks.order[i] = ph->sort[i].order; ks.col[i] = 0xFFFFFFFFu;
    if (ph->sort[i].kind == QW_SORT_COLUMN) {
      if (ph->sort[i].column == 0xFFFFFFFFu) ks.kind[i] = i == 0 ? (uint32_t)QW_SORT_DOCID : (uint32_t)QW_SORT_NONE;  // all None
      else {
        uint32_t t = sp.view.columns[ph->sort[i].column].type;
        if (t == QW_COL_STR) fail(QWGPU_EINVALID_ARG, "Unsupported sort field type `Str`.");
        ks.col[i] = use_col(L, sp, ph->sort[i].column);
      }
    }
  }
  if (ks.kind[1] == QW_SORT_DOCID) ks.kind[1] = QW_SORT_NONE;  // _doc as 2nd key extracts None
  if (ks.kind[0] == QW_SORT_NONE) ks.kind[0] = QW_SORT_DOCID;
  if (ks.kind[1] == QW_SORT_NONE) ks.order[1] = QW_ORDER_DESC;  // SortByPair::sort_orders default
  ks.score_scale = 0.f;
  ks.doc_bits = bits_needed64(P.num_docs ? P.num_docs - 1 : 0);
  ks.total_bits = ks.doc_bits;
  for (int i = 0; i < 2; i++) {
    ks.rbits[i] = 0; ks.hasbit[i] = 0; ks.raw_max[i] = 0;
    if (ks.kind[i] == QW_SORT_SCORE) {
      ks.hasbit[i] = 1;
      ks.rbits[i] = i == 0 ? 42 : 32;  // [lin:10 |] order-preserving f32 bits
    } else if (ks.kind[i] == QW_SORT_COLUMN) {
      const uint32_t bits = L.cols[ks.col[i]].bits;
      ks.hasbit[i] = 1;
      ks.rbits[i] = bits;
      ks.raw_max[i] = bits == 64 ? ~0ull : ((1ull << bits) - 1);
    }
    ks.total_bits += ks.hasbit[i] + ks.rbits[i];
  }
  ks.narrow = ks.total_bits <= 64 ? 1 : 0;
  {
    uint32_t pos = 0;
    for (int i = 0; i < 2; i++) {
      ks.sh_has[i] = ks.hasbit[i] ? 64 - pos - 1 : 0;
      pos += ks.hasbit[i];
      ks.sh_r[i] = (ks.narrow && ks.rbits[i]) ? 64 - pos - ks.rbits[i] : 0;
      pos += ks.rbits[i];
    }
    ks.sh_doc = (ks.narrow && ks.doc_bits) ? 64 - pos - ks.doc_bits : 0;
    if (!ks.narrow) ks.sh_has[0] = ks.sh_has[1] = 0;
  }
  if (ks.kind[0] == QW_SORT_SCORE) {
    float smax = L.score_max > 1e-30f ? L.score_max : 1.0f;
    ks.score_scale = 1024.0f / smax;
    ks.top_mode = QW_TOP_SCORE;
  } else if (ks.kind[0] == QW_SORT_COLUMN && ks.rbits[0] >= 10) ks.top_mode = QW_TOP_COLUMN;
  else if (ks.kind[0] == QW_SORT_DOCID && ks.kind[1] == QW_SORT_NONE && ks.doc_bits >= 11) ks.top_mode = QW_TOP_DOC;
  else ks.top_mode = QW_TOP_FULL;
  // aggregations
  if (ph->num_aggs > QW_MAX_DAGGS) fail(QWGPU_EUNSUPPORTED, "more than %d aggregation nodes", QW_MAX_DAGGS);
  std::vector<uint32_t> bases;
  uint64_t ncells = agg_cell_layout(aggs, ph->num_aggs, &bases);
  P.n_cells = (uint32_t)ncells;
  for (uint32_t i = 0; i < ph->num_aggs; i++) {
    const QwAggNode& a = aggs[i];
    DAgg d;
    memset(&d, 0, sizeof d);
    d.kind = a.kind; d.parent = a.parent; d.first_child = a.first_child; d.num_children = a.num_children;
    d.col = use_col(L, sp, a.column); d.num_buckets = a.num_buckets; d.has_bounds = a.has_bounds;
    d.num_ranges = a.num_ranges; d.has_missing = a.has_missing; d.cell_base = bases[i];
    d.is_f64 = a.kind == QW_AGG_STATS && d.col != 0xFFFFFFFFu && !qw_col_sum_exact(&sp.view.columns[a.column]);
    d.interval = a.interval; d.offset = a.offset; d.bound_min = a.bound_min; d.bound_max = a.bound_max;
    d.base_pos = a.base_pos;
    memcpy(d.range_from, a.range_from, sizeof d.range_from);
    memcpy(d.range_to, a.range_to, sizeof d.range_to);
    if (a.parent != 0xFFFFFFFFu) {
      if (a.parent >= ph->num_aggs) fail(QWGPU_EINVALID_ARG, "aggregation parent out of range");
      uint32_t depth = 1, p = a.parent;
      while (aggs[p].parent != 0xFFFFFFFFu) { depth++; p = aggs[p].parent; }
      if (depth > 2 || (depth == 2 && a.kind != QW_AGG_STATS)) fail(QWGPU_EUNSUPPORTED, "aggregation nesting deeper than bucket -> bucket -> metric");
      if (aggs[a.parent].kind == QW_AGG_STATS) fail(QWGPU_EINVALID_AGG, "metric aggregations cannot have sub-aggregations");
    }
    if (a.kind == QW_AGG_RANGE && a.num_ranges > QW_MAX_AGG_RANGES) fail(QWGPU_EUNSUPPORTED, "more than %d ranges", QW_MAX_AGG_RANGES);
    L.aggs.push_back(d);
  }
  P.n_aggs = ph->num_aggs;
  P.n_cols = (uint32_t)L.cols.size();
  // fast aggregation path: flat (no nesting) TERMS / HISTOGRAM nodes over always-present single-valued
  // columns. Histogram buckets are located through a raw-space boundary table built here with the
  // reference formula (agg_bucket in kernels.cuh == tantivy's ((val - offset) / interval).floor()),
  // which is monotone in the raw value.
  bool fast = ph->num_aggs > 0;
  P.n_stat_cells = 0;
  for (DAgg& d : L.aggs) {
    const bool full_col = d.col != 0xFFFFFFFFu && L.cols[d.col].card == QW_CARD_FULL;
    if (d.kind == QW_AGG_STATS) {
      // stats: top-level, or directly under a top-level bucket node; one {sum, min, max} triple per cell
      if (!full_col || d.num_children || (d.parent != 0xFFFFFFFFu && L.aggs[d.parent].parent != 0xFFFFFFFFu)) fast = false;
      d.stat_base = P.n_stat_cells;
      P.n_stat_cells += d.parent == 0xFFFFFFFFu ? 1u : L.aggs[d.parent].num_buckets;
    } else {
      // a histogram's raw-space boundary table ends one past the largest raw; a column whose raws reach
      // 2^64 - 1 has no such uint64 bound (its top value would fall outside the last bucket)
      if (d.parent != 0xFFFFFFFFu || (d.kind != QW_AGG_TERMS && d.kind != QW_AGG_HISTOGRAM) || !full_col ||
          d.num_buckets > QW_SMEM_AGG_CELLS || d.num_buckets == 0 ||
          (d.kind == QW_AGG_HISTOGRAM && L.col_max_raw[d.col] == ~0ull))
        fast = false;
    }
  }
  if (!fast) P.n_stat_cells = 0;
  if (fast) {
    for (DAgg& d : L.aggs) {
      if (d.kind != QW_AGG_HISTOGRAM) continue;
      const DCol& c = L.cols[d.col];
      // raws present in the column are < raw_end; searching beyond would leave the value domain
      // (f64 columns: bit patterns past the maximum are NaNs and break monotonicity)
      const uint64_t raw_end = L.col_max_raw[d.col] + 1;  // < 2^64: checked above
      const uint32_t nb = d.num_buckets;
      // g(raw): bucket index clamped to [-1, nb]; monotone non-decreasing in raw
      auto g = [&](uint64_t raw) -> int64_t {
        const unsigned __int128 wide = (unsigned __int128)c.gcd * raw + c.min_value;  // saturate beyond the column's range
        const double val = mapped_to_f64_host(c.type, wide > (unsigned __int128)~0ull ? ~0ull : (uint64_t)wide);
        if (d.has_bounds) {
          if (!(val >= d.bound_min)) return -1;
          if (!(val <= d.bound_max)) return (int64_t)nb;
        }
        const double pos = std::floor((val - d.offset) / d.interval);
        if (!(pos >= -9.0e18)) return -1;
        if (!(pos <= 9.0e18)) return (int64_t)nb;
        const int64_t idx = (int64_t)pos - d.base_pos;
        return idx < 0 ? -1 : (idx >= (int64_t)nb ? (int64_t)nb : idx);
      };
      d.bounds = L.bounds.size();  // index for now; turned into a device address when the blob is laid out
      uint64_t lo = 0;
      for (uint32_t k = 0; k <= nb; k++) {
        // smallest raw in [lo, raw_end] with g(raw) >= k (raw_end when there is none)
        uint64_t a = lo, b = raw_end;
        while (a < b) {
          const uint64_t mid = a + (b - a) / 2;
          if (g(mid) >= (int64_t)k) b = mid; else a = mid + 1;
        }
        L.bounds.push_back(a);
        lo = a;
      }
      const uint64_t b0 = L.bounds[d.bounds], bn = L.bounds[d.bounds + nb];
      d.inv_step = bn > b0 ? (float)((double)nb / (double)(bn - b0)) : 0.0f;
    }
  }
  P.fast_aggs = fast ? 1 : 0;
}

// shared-memory arena for a batch (max over the batch's plans)
static uint32_t stage_bytes_for(uint32_t W) {
  if (const char* e = getenv("QWGPU_STAGE")) return (uint32_t)atoi(e) & ~15u;
  return std::min<uint32_t>(std::max<uint32_t>(W, 8192), 24576);
}

static SmemLayout make_layout(uint32_t W, uint32_t n_levels, uint32_t need_cnt, uint32_t need_msum, uint32_t need_ssum,
                              uint32_t max_instr, uint32_t max_cols, uint32_t max_aggs, uint32_t n_fn, bool rec_l0, bool rangeq) {
  SmemLayout L;
  memset(&L, 0xFF, sizeof L);
  uint32_t off = 0;
  auto take = [&](uint32_t bytes) { uint32_t o = off; off = (off + bytes + 15) & ~15u; return o; };
  L.misc = take(32 + 4 * QW_MAX_TERMS + QW_MAX_TERMS);  // counters, per-term block bases, per-term instruction index
  L.instr = take(std::max(max_instr, 1u) * sizeof(DInstr));
  L.cols = take(std::max(max_cols, 1u) * sizeof(DCol));
  L.aggs = take(std::max(max_aggs, 1u) * sizeof(DAgg));
  L.key = take(sizeof(DKeySpec));

  for (uint32_t l = 0; l < n_levels; l++) {
    L.lvl[l].req = take(W / 8);
    L.lvl[l].shd = take(W / 8);
    L.lvl[l].nt = take(W / 8);
    if ((need_cnt >> l) & 1) L.lvl[l].cnt = take(W);
    if ((need_msum >> l) & 1) L.lvl[l].msum = take(W * 4);
    if ((need_ssum >> l) & 1) L.lvl[l].ssum = take(W * 4);
    L.lvl[l].rsc = L.lvl[l].msum != 0xFFFFFFFFu ? L.lvl[l].msum : L.lvl[l].ssum;
  }
  L.tmp = take(W / 8);
  for (uint32_t s = 0; s < n_fn; s++) L.fn[s] = take(W);  // BM25 tables stay in global memory (L1-resident)
  L.rng = take(QW_MAX_TERMS * 16);
  L.hitq = L.rng;  // the collect-time hit queues alias rng / blkrec / termblk (contiguous, dead after the program)
  L.blkrec = take(QW_MAX_WBLK * 8);
  L.termblk = take(QW_MAX_TERMS * 8);
  L.stage = take(stage_bytes_for(W));
  L.hist = L.stage;  // histogram / privatised aggregation counters reuse the staging area at collect time
  if (rec_l0) L.l0hist = take(QW_HIST_BINS * 4);
  if (rangeq) L.rangeq = take(QW_WARPS * (32 + 32 * 4) * 2);  // QW_WARPS x QW_HITQ_CAP uint16 (kernels.cuh)
  L.total = off;
  return L;
}

// shared-memory arena of the BM25-union pipeline (union_kernel.cuh): score array, QU_SLOTS staging slots
// (block payload + records + per-term table + header), mbarriers, MODE_HIST histogram
static qwk::USmem make_union_layout(uint32_t W, bool hist, uint32_t budget) {
  qwk::USmem L;
  memset(&L, 0, sizeof L);
  uint32_t off = 0;
  auto take = [&](uint32_t bytes) { uint32_t o = off; off = (off + bytes + 15) & ~15u; return o; };
  L.score = take(W * 4);
  L.bars = take(8 * (2 * QU_SLOTS + QU_CHAIN));
  if (hist) L.hist = take(QW_HIST_BINS * 4);
  L.cands = take(QU_NCW * QU_CANDS * 8 + QU_NCW * 4);
  const uint32_t fixed = QU_MAXBLK * 16 + QU_MAX_TERMS * 16 + 32 + QU_PAD;
  uint32_t cap = budget > off + QU_SLOTS * (fixed + 2048) ? ((budget - off) / QU_SLOTS - fixed) & ~15u : 2048;
  if (const char* e = getenv("QWGPU_UCAP")) cap = (uint32_t)atoi(e) & ~15u;
  L.cap = cap;
  L.payload = 0;
  L.recs = cap + QU_PAD;
  L.ttab = L.recs + QU_MAXBLK * 16;
  L.hdr = L.ttab + QU_MAX_TERMS * 16;
  L.slot_stride = L.hdr + 48;  // header (32 B) + block hand-out counter
  L.slot0 = take(QU_SLOTS * L.slot_stride);
  L.total = off;
  return L;
}

void Engine::search(const std::vector<std::shared_ptr<SplitDev>>& sp, const std::vector<const uint8_t*>& plans,
                    const std::vector<size_t>& plan_lens, std::vector<SplitOutput>& outs, BatchStats& stats,
                    const MergeSpec* merge, std::vector<MergedHit>* merged, const GatherSpec* gather, std::vector<RankHeader>* rank_headers) {
  const uint32_t n_in = (uint32_t)sp.size();
  outs.assign(n_in, SplitOutput());
  static const bool trace = getenv("QWGPU_TRACE") != nullptr;  // host phase timings on stderr
  using tclock = std::chrono::steady_clock;
  const auto t_begin = tclock::now();
  CUDA_CHECK(cudaSetDevice(device));
  // ---- lower every plan; splits whose plan cannot be lowered fail individually ----------------------
  std::vector<Lowered> low;
  std::vector<uint32_t> idx;  // position in the caller's arrays
  low.reserve(n_in);
  for (uint32_t i = 0; i < n_in; i++) {
    try {
      if (!sp[i]) fail(QWGPU_ENOTFOUND, "split not registered");
      Lowered L;
      lower_plan(L, *sp[i], plans[i], plan_lens[i]);
      low.push_back(std::move(L));
      idx.push_back(i);
    } catch (const Error& e) {
      outs[i].status = e.code;
      outs[i].error = e.what();
    }
  }
  const uint32_t n = (uint32_t)low.size();
  if (n == 0) {
    // no searchable split on this rank: it still takes part in the collective with an empty record
    if (merge && merged && gather && gather->allgather && gather->world > 1 && rank_headers && merge->k) {
      const size_t rec = 64 + (size_t)merge->k * sizeof(qwk::DMergedHit), W8 = (size_t)gather->world;
      uint8_t *d = nullptr;
      const size_t o_recv = 256 * ((rec + 255) / 256), o_fin = o_recv + 256 * ((W8 * rec + 255) / 256), o_cut = o_fin + 256 * ((16 + rec + 255) / 256), o_hd = o_cut + 1024, total = o_hd + W8 * 64;
      CUDA_CHECK(cudaMalloc(&d, total));
      cudaStream_t st0 = nullptr;
      CUDA_CHECK(cudaStreamCreateWithFlags(&st0, cudaStreamNonBlocking));
      CUDA_CHECK(cudaMemsetAsync(d, 0, total, st0));
      qwk::DRankHeader h;
      memset(&h, 0, sizeof h);
      h.attempted = gather->attempted; h.successful = gather->successful; h.n_failed = gather->n_failed;
      CUDA_CHECK(cudaMemcpyAsync(d, &h, sizeof h, cudaMemcpyHostToDevice, st0));
      if (gather->allgather(gather->comm, d, d + o_recv, rec, (void*)st0)) fail(QWGPU_EINTERNAL, "ncclAllGather failed");
      const qwk::SrcGathered gsrc{d + o_recv, (uint32_t)rec, 64u};
      qwk::k_merge_prep<qwk::SrcGathered><<<1, 1024, 0, st0>>>(gsrc, (uint32_t)gather->world, merge->k, merge->order1, merge->order2, (uint32_t*)(d + o_cut));
      const uint64_t gthreads = (uint64_t)gather->world * merge->k * 32;
      qwk::k_merge<qwk::SrcGathered><<<(uint32_t)((gthreads + 255) / 256), 256, 0, st0>>>(gsrc, (uint32_t*)(d + o_cut), (uint32_t)gather->world, merge->k, merge->k, merge->order1, merge->order2,
                                                                                       (qwk::DMergedHit*)(d + o_fin + 16), (uint32_t*)(d + o_fin));
      CUDA_CHECK(cudaMemcpy2DAsync(d + o_hd, 64, d + o_recv, rec, 64, W8, cudaMemcpyDeviceToDevice, st0));
      std::vector<uint8_t> host(16 + (size_t)merge->k * sizeof(qwk::DMergedHit));
      rank_headers->resize(gather->world);
      CUDA_CHECK(cudaMemcpyAsync(host.data(), d + o_fin, host.size(), cudaMemcpyDeviceToHost, st0));
      CUDA_CHECK(cudaMemcpyAsync(rank_headers->data(), d + o_hd, W8 * 64, cudaMemcpyDeviceToHost, st0));
      CUDA_CHECK(cudaStreamSynchronize(st0));
      const uint32_t nm = *(const uint32_t*)host.data();
      const qwk::DMergedHit* mh = (const qwk::DMergedHit*)(host.data() + 16);
      merged->resize(nm);
      for (uint32_t j = 0; j < nm; j++) { (*merged)[j].hit = mh[j].hit; (*merged)[j].split = mh[j].split; (*merged)[j].pad = 0; }
      cudaStreamDestroy(st0);
      cudaFree(d);
    }
    return;
  }
  const auto t_lowered = tclock::now();

  // ---- batch-wide parameters --------------------------------------------------------------------------
  uint32_t n_levels = 1, need_cnt = 0, need_ssum = 0, need_msum = 0, max_instr = 0, max_cols = 0, max_aggs = 0, n_fn = 0;
  bool scoring = false, any_topk = false, any_aggs = false, smem_aggs = true;
  uint32_t max_cells = 0, max_key_bits = 0;
  uint32_t tot_instr = 0, tot_cols = 0, tot_aggs = 0, tot_bounds = 0;
  // second-chance top-K: when no plan ranks by _score first, the collect pass also records the exact
  // level-0 histogram and every window's best digit, so that a failed sampled threshold is repaired
  // by a candidates-only pass over the few windows that can hold candidates
  bool rec_l0 = true, rangeq = false;
  // every plan has the BM25 top-K shape => the specialised UNION instantiation of the collect kernel
  bool all_union = true, all_driver = true;
  for (auto& L : low) {
    if (!(L.P.fused_score_root && L.P.max_hits && !L.P.sa.present && !L.P.n_aggs && L.P.key.kind[0] == QW_SORT_SCORE &&
          L.P.key.order[0] == QW_ORDER_DESC))
      all_union = false;
    if (L.P.n_terms > QU_MAX_TERMS || L.P.n_instr != L.P.n_terms + 2) all_union = false;  // [BOOL_BEGIN, TERM x n, BOOL_END]
    {
      // one driving posting list + required column filters, no aggregations: the posting-driven kernel
      // (driver_kernel.cuh). [BOOL_BEGIN, TERM, (RANGE | EXISTS) x 0..4, BOOL_END] at level 0.
      const std::vector<DInstr>& I = L.instrs;
      bool d = L.P.n_aggs == 0 && I.size() >= 3 && I.size() <= 3 + QD_MAX_FILTERS && I[0].op == OP_BOOL_BEGIN && I[1].op == OP_TERM &&
               I.back().op == OP_BOOL_END && I.back().level == 0;
      if (d) {
        const bool req = I[1].occur == QW_OCCUR_MUST || I[1].occur == QW_OCCUR_FILTER;
        if (!req && !(I[1].occur == QW_OCCUR_SHOULD && I.size() == 3 && I.back().r == 1 && I.back().n == 0)) d = false;
        for (size_t k = 2; k + 1 < I.size() && d; k++) {
          const bool colpred = I[k].op == OP_RANGE || I[k].op == OP_EXISTS;
          const bool unscored_req = I[k].occur == QW_OCCUR_FILTER || (I[k].occur == QW_OCCUR_MUST && !(I[k].flags & IF_SCORED));
          if (!colpred || !unscored_req || I[k].level != 0) d = false;
        }
      }
      if (!d) all_driver = false;
    }
    if (L.P.max_hits && L.P.key.kind[0] == QW_SORT_SCORE) rec_l0 = false;
    max_key_bits = std::max(max_key_bits, L.P.key.total_bits);
    for (const DInstr& in : L.instrs)
      if ((in.op == OP_RANGE || in.op == OP_EXISTS) && (in.occur == QW_OCCUR_MUST || in.occur == QW_OCCUR_FILTER)) rangeq = true;
    n_levels = std::max(n_levels, L.P.n_levels);
    need_cnt |= L.need_cnt; need_ssum |= L.need_ssum; need_msum |= L.need_msum;
    max_instr = std::max(max_instr, L.P.n_instr); max_cols = std::max(max_cols, L.P.n_cols); max_aggs = std::max(max_aggs, L.P.n_aggs);
    n_fn = std::max(n_fn, L.P.n_fn_slots);
    scoring |= L.P.scoring != 0; any_topk |= L.P.max_hits > 0; any_aggs |= L.P.n_aggs > 0;
    max_cells = std::max(max_cells, L.P.n_cells);
    L.P.instr_base = tot_instr; L.P.col_base = tot_cols; L.P.agg_base = tot_aggs;
    L.bounds_base = tot_bounds;
    tot_instr += L.P.n_instr; tot_cols += L.P.n_cols; tot_aggs += L.P.n_aggs; tot_bounds += (uint32_t)L.bounds.size();
  }
  rec_l0 = rec_l0 && any_topk;
  // window size: as large as shared memory allows for the configured blocks/SM (per-window fixed
  // costs — staging, program interpretation, barriers — amortise over more postings)
  uint32_t W = 32768;
  if (const char* e = getenv("QWGPU_W")) W = (uint32_t)atoi(e);
  // BM25-union batches run the TMA + mbarrier pipeline (union_kernel.cuh): fixed 16384-doc windows,
  // two blocks per SM; QWGPU_OLD_UNION=1 keeps the round-1 window kernel for A/B runs
  static const bool old_union = getenv("QWGPU_OLD_UNION") != nullptr;
  // (QWGPU_NO_DRIVER=1 keeps the window engine for these shapes: A/B runs)
  static const bool driver_on = getenv("QWGPU_NO_DRIVER") == nullptr;
  const bool use_driver = all_driver && driver_on;
  if (use_driver) rec_l0 = false;
  const bool use_union = all_union && !old_union && !use_driver;
  const uint32_t u_budget = (uint32_t)(max_smem_optin + 1024) / QU_MINB - 1024 - 64;
  // match_all + flat terms / histogram aggregations, no hits: the streaming column kernel (agg_kernel.cuh)
  static const bool old_aggs = getenv("QWGPU_OLD_AGGS") != nullptr;
  bool use_aggscan = !old_aggs;
  qwk::ASmem alay;
  memset(&alay, 0, sizeof alay);
  {
    uint32_t maxbits[QW_MAX_DAGGS] = {0};
    for (auto& L : low) {
      if (!(L.P.n_instr == 3 && L.instrs[1].op == OP_ALL && L.P.max_hits == 0 && L.P.n_aggs > 0 && L.P.n_cells <= QA_MAX_CELLS)) { use_aggscan = false; break; }
      for (uint32_t gi = 0; gi < L.P.n_aggs; gi++) {
        const DAgg& d = L.aggs[gi];
        const bool flat = d.parent == 0xFFFFFFFFu && d.num_children == 0 && (d.kind == QW_AGG_TERMS || d.kind == QW_AGG_HISTOGRAM) && !d.has_missing;
        if (!flat || !L.P.fast_aggs || d.col == 0xFFFFFFFFu || L.cols[d.col].card != QW_CARD_FULL || L.cols[d.col].bits > 32) { use_aggscan = false; break; }
        maxbits[gi] = std::max(maxbits[gi], L.cols[d.col].bits);
      }
      if (!use_aggscan) break;
    }
    if (use_aggscan) {
      uint32_t off = 0;
      auto take = [&](uint32_t bytes) { uint32_t o = off; off = (off + bytes + 15) & ~15u; return o; };
      for (uint32_t gi = 0; gi < QW_MAX_DAGGS; gi++) alay.col_off[gi] = take(maxbits[gi] ? QA_CHUNK / 8 * maxbits[gi] + 16 : 0);
      alay.hdr = take(16);
      alay.slot_stride = off;
      off = 0;
      uint32_t a_cells = 1;
      for (auto& L : low) a_cells = std::max(a_cells, L.P.n_cells);
      alay.bars = take(8 * 2 * QA_SLOTS);
      alay.atab = take(QW_MAX_DAGGS * sizeof(qwk::AggRow));
      alay.bcache = take(QA_CW * QW_MAX_DAGGS * 16);
      alay.cells = take(a_cells * 4);
      alay.slot0 = take(QA_SLOTS * alay.slot_stride);
      alay.total = off;
      if ((int)alay.total + 1024 > max_smem_optin) use_aggscan = false;
    }
  }
  if (use_aggscan) W = QA_CHUNK;  // the flat work list is the list of 8192-doc chunks
  qwk::USmem ulay_c, ulay_h;
  if (use_union && !getenv("QWGPU_W"))
    W = getenv("QWGPU_UW") ? (uint32_t)atoi(getenv("QWGPU_UW")) : 15360u * 2 / QU_MINB;
  SmemLayout lay;
  for (;;) {
    lay = make_layout(W, n_levels, need_cnt, need_msum, need_ssum, max_instr, max_cols, max_aggs, n_fn, rec_l0, rangeq);
    if ((int)lay.total + 1024 <= max_smem_optin / (use_union ? 1 : QW_MIN_BLOCKS_PER_SM) || W == 1024) break;  // (union batches: k_window is only the rare exact-radix fallback)
    W >>= 1;
  }
  (void)scoring;
  if (use_aggscan && W != QA_CHUNK) use_aggscan = false;
  if (use_union) {
    // (the generic layout above stays valid for the same W: exact radix passes below level 0 use k_window)
    ulay_c = make_union_layout(W, false, u_budget);
    ulay_h = make_union_layout(W, true, u_budget);
  }
  if ((int)lay.total > max_smem_optin) fail(QWGPU_EUNSUPPORTED, "query needs %u bytes of shared memory per block", lay.total);

  // ---- device blob: plans, programs, work maps ----------------------------------------------------------
  std::vector<uint32_t> fw_all(n + 1), fw_smp(n + 1);
  uint32_t max_windows = 0;
  for (uint32_t i = 0; i < n; i++) {
    low[i].P.num_windows = low[i].empty ? 0 : (low[i].P.num_docs + W - 1) / W;
    max_windows = std::max(max_windows, low[i].P.num_windows);
  }
  // sampling stride of the threshold-estimation pass: 1/16 of the windows (24 or 32 save ~15 us in the
  // histogram pass but the looser threshold costs about as much in the collect pass)
  static const uint32_t stride_cap = getenv("QWGPU_STRIDE_CAP") ? (uint32_t)atoi(getenv("QWGPU_STRIDE_CAP")) : 16u;
  uint32_t stride = std::min(std::max(stride_cap, 1u), std::max(1u, max_windows / 8));
  // BM25-union batches can sample the threshold over finer windows (W / QWGPU_HDIV: the same fraction of the docs in
  // more work items). Measured on the bench workload: 1 and 2 are equal (1.22 ms per 4-query step), 4 and 8 are slower
  // (1.28 / 1.48 ms: the per-window clause chain does not shrink with the window), so the default stays 1.
  static const uint32_t hdiv = getenv("QWGPU_HDIV") ? std::max(1u, (uint32_t)atoi(getenv("QWGPU_HDIV"))) : 1u;
  const uint32_t W_h = use_union ? std::max(1024u, (W / hdiv) & ~1023u) : W;
  if (use_union) {
    uint32_t mw = 0, tw = 0;
    for (uint32_t i = 0; i < n; i++) {
      const uint32_t nw = low[i].empty ? 0u : (low[i].P.num_docs + W_h - 1) / W_h;
      mw = std::max(mw, nw);
      tw += nw;
    }
    stride = std::min(std::max(stride_cap, 1u), std::max(1u, mw / 8));
    // Large requests: at most ONE sampled window per resident block (the sampled pass is latency bound — a block
    // that gets two windows doubles its duration), up to a stride of 32. Bench workload (6528 windows, 296 blocks):
    // stride 23 instead of 16, 1.146 against 1.186 ms per 4-query step (32: 1.169 — the looser threshold then costs
    // more candidates in the collect pass than the sampled pass saves).
    if (!getenv("QWGPU_STRIDE_CAP")) {
      const uint32_t per_block = (tw + (uint32_t)(sm_count * QU_MINB) - 1) / (uint32_t)(sm_count * QU_MINB);
      stride = std::max(stride, std::min({per_block, 32u, std::max(1u, mw / 8)}));
    }
  }
  // posting-driven kernel: the work list is the driving term's posting blocks; the threshold sample takes every
  // stride-th BLOCK (128 postings, fine enough for keys that follow doc order: what lies between two sampled
  // blocks is < 2K postings)
  std::vector<uint32_t> fw_drv(n + 1, 0), fw_dsm(n + 1, 0);
  if (use_driver) {
    uint32_t max_blocks = 0;
    for (uint32_t i = 0; i < n; i++) max_blocks = std::max(max_blocks, low[i].empty ? 0u : low[i].instrs[1].n);
    stride = std::min(std::max(stride_cap, 1u), std::max(1u, max_blocks / 64));
    for (uint32_t i = 0; i < n; i++) {
      const uint32_t nb = low[i].empty ? 0u : low[i].instrs[1].n, phase = stride > 1 ? i % stride : 0;
      fw_drv[i + 1] = fw_drv[i] + nb;
      fw_dsm[i + 1] = fw_dsm[i] + (nb > phase ? (nb - phase + stride - 1) / stride : 0);
    }
  }
  // the generic kernels sample an explicit window list: strided windows + the first and last window of each
  // split (weight 1 in the histogram); the union pipeline keeps the plain strided sample (scores do not
  // follow doc order)
  const bool edge_sample = !use_union && !use_driver && stride > 1;
  std::vector<uint32_t> sample_win;
  fw_all[0] = fw_smp[0] = 0;
  for (uint32_t i = 0; i < n; i++) {
    uint32_t nw = low[i].P.num_windows, phase = stride > 1 ? i % stride : 0;
    fw_all[i + 1] = fw_all[i] + nw;
    if (use_union) nw = low[i].empty ? 0 : (low[i].P.num_docs + W_h - 1) / W_h;  // (the sampled pass has its own window size)
    if (edge_sample) {
      uint32_t cnt = 0;
      for (uint32_t w = 0; w < nw; w++) {
        const bool edge = w == 0 || w + 1 == nw, strided = w % stride == phase;
        if (edge || strided) { sample_win.push_back(w | (edge ? 0x80000000u : 0u)); cnt++; }
      }
      fw_smp[i + 1] = fw_smp[i] + cnt;
    } else fw_smp[i + 1] = fw_smp[i] + (nw > phase ? (nw - phase + stride - 1) / stride : 0);
  }
  // phrases: one uncompressed posting block per block of each phrase's driver term (phrase_kernel.cuh)
  uint32_t n_phrases = 0, phrase_blocks = 0;
  for (auto& L : low)
    for (size_t k = 0; k < L.phrases.size(); k++) { n_phrases++; phrase_blocks += L.instrs[L.phrase_instr[k]].n; }
  auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
  size_t o_plans = 0, o_instr = al(o_plans + n * sizeof(DSplitPlan)), o_cols = al(o_instr + tot_instr * sizeof(DInstr)),
         o_aggs = al(o_cols + std::max(tot_cols, 1u) * sizeof(DCol)), o_fwa = al(o_aggs + std::max(tot_aggs, 1u) * sizeof(DAgg)),
         o_fws = al(o_fwa + (n + 1) * 4), o_bounds = al(o_fws + (n + 1) * 4), o_rank = al(o_bounds + (size_t)tot_bounds * 8),
         o_smp = al(o_rank + (size_t)n * 4), o_phr = al(o_smp + sample_win.size() * 4), o_fwd = al(o_phr + (size_t)n_phrases * sizeof(DPhrase)),
         o_fwds = al(o_fwd + (use_driver ? (size_t)(n + 1) * 4 : 0)), blob_bytes = al(o_fwds + (use_driver ? (size_t)(n + 1) * 4 : 0));
  // device-side cross-split merge: the per-split hit lists stay in scratch, only the merged top-K comes back
  const bool do_merge = merge && merged && merge->k > 0 && any_topk && merge->rank.size() == n_in;
  uint32_t kmax = 1;
  for (auto& L : low) kmax = std::max(kmax, L.P.max_hits);
  // scratch: thresholds, histograms, candidates
  size_t s_thr = 0, s_hist = al(s_thr + n * sizeof(DThresh)), s_state = al(s_hist + (size_t)n * QW_HIST_BINS * 4),
         s_ctr = al(s_state + (size_t)n * 4), s_wmax = al(s_ctr + 64 * 4), s_cand = al(s_wmax + (rec_l0 ? (size_t)fw_all[n] * 2 : 0)),
         s_hits = al(s_cand + (any_topk ? (size_t)n * QW_CAND_CAP * 24 : 0)),
         s_cut = al(s_hits + (do_merge ? (size_t)n * kmax * sizeof(QwHit) : 0)),
         s_grecv = al(s_cut + (size_t)std::max<uint32_t>(n, 64) * 4 + 1024),
         s_vblk = al(s_grecv + (gather && gather->world > 1 && do_merge ? (size_t)gather->world * (64 + (size_t)merge->k * sizeof(qwk::DMergedHit)) : 0)),
         scratch_bytes = al(s_vblk + (size_t)phrase_blocks * sizeof(VBlk));
  // out: per split [hdr 32B][hits][cells]
  std::vector<size_t> out_off(n + 1);
  out_off[0] = 0;
  for (uint32_t i = 0; i < n; i++)
    out_off[i + 1] = al(out_off[i] + 32 + (do_merge ? 0 : (size_t)low[i].P.max_hits * sizeof(QwHit)) + (size_t)low[i].P.n_cells * sizeof(QwAggCell));
  // [RankHeader 64 B (n_hits first)][DMergedHit x k]: the batch's merged top-k = this rank's gather record
  const size_t o_merged = out_off[n];
  const size_t rec_bytes = do_merge ? 64 + (size_t)merge->k * sizeof(qwk::DMergedHit) : 0;
  const bool do_gather = do_merge && gather && gather->allgather && gather->world > 1 && rank_headers;
  // gathered: [world x RankHeader (compacted copy)][final count 16 B][final DMergedHit x k]
  const size_t o_ghdr = al(o_merged + rec_bytes), o_final = al(o_ghdr + (do_gather ? (size_t)gather->world * 64 : 0));
  size_t out_bytes = do_merge ? (do_gather ? al(o_final + 16 + (size_t)merge->k * sizeof(qwk::DMergedHit)) : al(o_merged + rec_bytes)) : out_off[n];

  // Admission: at most QWGPU_MAX_IN_FLIGHT (default 16) searches drive the device at once; further callers wait here
  // on a condition variable (no CUDA calls, no spinning). Measured on the mixed config-5 query set: 16 host threads
  // sustain 1860 queries/s, 64 unthrottled threads 920 — beyond a dozen or so submitters the driver's per-context
  // lock and 64 interleaved streams cost more than the extra overlap brings.
  static const int max_in_flight = getenv("QWGPU_MAX_IN_FLIGHT") ? std::max(1, atoi(getenv("QWGPU_MAX_IN_FLIGHT"))) : 16;
  CallSlot* slot = nullptr;
  {
    std::unique_lock<std::mutex> g(mu);
    cv_admit.wait(g, [&] { return admitted < max_in_flight; });
    admitted++;
    if (!free_slots.empty()) { slot = free_slots.back(); free_slots.pop_back(); }
  }
  struct Admit {  // (released on every path, including a throw before the slot guard below exists)
    Engine* e;
    ~Admit() {
      { std::lock_guard<std::mutex> g(e->mu); e->admitted--; }
      e->cv_admit.notify_one();
    }
  } admit{this};
  if (!slot) {
    slot = new CallSlot();
    CUDA_CHECK(cudaStreamCreateWithFlags(&slot->stream, cudaStreamNonBlocking));
    CUDA_CHECK(cudaEventCreate(&slot->ev0));
    CUDA_CHECK(cudaEventCreate(&slot->ev1));
    CUDA_CHECK(cudaEventCreate(&slot->ev2));
    CUDA_CHECK(cudaEventCreate(&slot->ev3));
    CUDA_CHECK(cudaEventCreateWithFlags(&slot->ev_block, cudaEventBlockingSync | cudaEventDisableTiming));
  }
  // the slot goes back to the pool only once its stream is idle: on an error path copies / kernels of this
  // call may still be in flight, and the next call would reuse the pinned buffers under them
  struct Release {
    Engine* e; CallSlot* s;
    ~Release() {
      cudaStreamSynchronize(s->stream);
      e->in_flight.fetch_sub(1);
      std::lock_guard<std::mutex> g(e->mu);
      e->free_slots.push_back(s);
    }
  } rel{this, slot};
  in_flight.fetch_add(1);
  // Waiting for the call's stream: cudaStreamSynchronize spins on a CPU core, which is the fastest wake-up while a
  // few calls are in flight (single-query latency) and a disaster when more host threads wait than there are cores
  // to spare — the spinners starve the threads that still have plans to compile. Beyond a quarter of the cores the
  // wait goes through a blocking event instead (the thread sleeps until the driver's interrupt).
  static const uint32_t spin_limit = getenv("QWGPU_SPIN_LIMIT") ? (uint32_t)atoi(getenv("QWGPU_SPIN_LIMIT")) : std::max(2u, std::thread::hardware_concurrency() / 4);
  auto wait_stream = [&]() {
    if (in_flight.load(std::memory_order_relaxed) > (int)spin_limit) {
      CUDA_CHECK(cudaEventRecord(slot->ev_block, slot->stream));
      CUDA_CHECK(cudaEventSynchronize(slot->ev_block));
    } else CUDA_CHECK(cudaStreamSynchronize(slot->stream));
  };
  size_t want_blob, want_scratch, want_out;
  {
    // slots are sized to the largest request the context has seen: a slot that meets a bigger request later would
    // have to cudaFree / cudaMalloc (device-synchronising) in the middle of concurrent searches
    std::lock_guard<std::mutex> g(mu);
    hw_blob = std::max(hw_blob, blob_bytes); hw_scratch = std::max(hw_scratch, scratch_bytes); hw_out = std::max(hw_out, out_bytes);
    // (only while the marks stay moderate: one huge aggregation request must not size every slot after itself)
    auto sized = [](size_t hw, size_t need) { return hw <= ((size_t)64 << 20) ? hw : need; };
    want_blob = sized(hw_blob, blob_bytes); want_scratch = sized(hw_scratch, scratch_bytes); want_out = sized(hw_out, out_bytes);
  }
  slot->ensure(want_blob, want_scratch, want_out);
  cudaStream_t st = slot->stream;

  uint32_t phr_done = 0, phr_blocks_done = 0;
  for (uint32_t i = 0; i < n; i++) {
    DSplitPlan& P = low[i].P;
    // privatised counters + stats triples must fit the (dead at collect time) staging area
    if (P.fast_aggs && (((size_t)P.n_cells * 4 + 7) & ~(size_t)7) + (size_t)P.n_stat_cells * 24 > stage_bytes_for(W)) P.fast_aggs = 0;
    uint8_t* ob = slot->d_out + out_off[i];
    P.out_num_hits = (uint64_t)ob;            // [0] hits, [1] eligible
    P.out_nhits = (uint64_t)(ob + 16);
    P.out_cand_count = (uint64_t)(ob + 20);
    P.out_hits = do_merge ? (uint64_t)(slot->d_scratch + s_hits + (size_t)i * kmax * sizeof(QwHit)) : (uint64_t)(ob + 32);
    P.out_cells = (uint64_t)(ob + 32 + (do_merge ? 0 : (size_t)P.max_hits * sizeof(QwHit)));
    P.out_hist = (uint64_t)(slot->d_scratch + s_hist + (size_t)i * QW_HIST_BINS * 4);
    P.out_cands = (uint64_t)(slot->d_scratch + s_cand + (size_t)i * QW_CAND_CAP * 24);
    for (size_t k = 0; k < low[i].phrases.size(); k++) {
      DPhrase& ph = low[i].phrases[k];
      DInstr& pin = low[i].instrs[low[i].phrase_instr[k]];
      ph.first_work = phr_blocks_done;
      ph.out = (uint64_t)(slot->d_scratch + s_vblk + (size_t)phr_blocks_done * sizeof(VBlk));
      pin.a = ph.out;
      phr_blocks_done += pin.n;
      memcpy(slot->h_blob + o_phr + (size_t)phr_done++ * sizeof(DPhrase), &ph, sizeof ph);
    }
    memcpy(slot->h_blob + o_plans + i * sizeof(DSplitPlan), &P, sizeof P);
    memcpy(slot->h_blob + o_instr + P.instr_base * sizeof(DInstr), low[i].instrs.data(), P.n_instr * sizeof(DInstr));
    if (P.n_cols) memcpy(slot->h_blob + o_cols + P.col_base * sizeof(DCol), low[i].cols.data(), P.n_cols * sizeof(DCol));
    if (P.fast_aggs)
      for (DAgg& d : low[i].aggs)
        if (d.kind == QW_AGG_HISTOGRAM) d.bounds = (uint64_t)(slot->d_blob + o_bounds) + (low[i].bounds_base + d.bounds) * 8;
    if (P.n_aggs) memcpy(slot->h_blob + o_aggs + P.agg_base * sizeof(DAgg), low[i].aggs.data(), P.n_aggs * sizeof(DAgg));
    if (!low[i].bounds.empty()) memcpy(slot->h_blob + o_bounds + (size_t)low[i].bounds_base * 8, low[i].bounds.data(), low[i].bounds.size() * 8);
  }
  if (do_merge) for (uint32_t i = 0; i < n; i++) ((uint32_t*)(slot->h_blob + o_rank))[i] = merge->rank[idx[i]];
  if (!sample_win.empty()) memcpy(slot->h_blob + o_smp, sample_win.data(), sample_win.size() * 4);
  if (use_driver) { memcpy(slot->h_blob + o_fwd, fw_drv.data(), (n + 1) * 4); memcpy(slot->h_blob + o_fwds, fw_dsm.data(), (n + 1) * 4); }
  memcpy(slot->h_blob + o_fwa, fw_all.data(), (n + 1) * 4);
  memcpy(slot->h_blob + o_fws, fw_smp.data(), (n + 1) * 4);
  CUDA_CHECK(cudaMemcpyAsync(slot->d_blob, slot->h_blob, blob_bytes, cudaMemcpyHostToDevice, st));
  stats.h2d_bytes += blob_bytes;

  KParams kp;
  memset(&kp, 0, sizeof kp);
  kp.plans = (const DSplitPlan*)(slot->d_blob + o_plans);
  kp.instrs = (const DInstr*)(slot->d_blob + o_instr);
  kp.cols = (const DCol*)(slot->d_blob + o_cols);
  kp.aggs = (const DAgg*)(slot->d_blob + o_aggs);
  kp.thresh = (DThresh*)(slot->d_scratch + s_thr);
  kp.n_splits = n;
  kp.W = W;
  kp.stage_bytes = stage_bytes_for(W);
  // privatised aggregation counters (and the radix histogram, 8 KB) live in the staging area
  if (max_cells * 4 > kp.stage_bytes || max_cells > QW_SMEM_AGG_CELLS) smem_aggs = false;
  kp.smem_aggs = (any_aggs && smem_aggs) ? 1 : 0;
  kp.sm = lay;
  kp.wmax = (uint16_t*)(slot->d_scratch + s_wmax);
  kp.split_state = (const uint32_t*)(slot->d_scratch + s_state);
  int occ = 1;
  CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, qwk::k_window<qwk::MODE_COLLECT, false>, QW_THREADS, lay.total));
  occ = std::max(occ, 1);
  enum { F_REC = 1, F_REFINE = 2, F_CANDS_ONLY = 4 };
  uint32_t n_ctr = 0;  // work counters handed to k_union launches (zeroed with the scratch region)
  auto launch_window = [&](int mode, bool sampled, uint32_t level, uint32_t use_prefix, uint32_t flags) {
    KParams q = kp;
    q.first_work = (const uint32_t*)(slot->d_blob + (sampled ? o_fws : o_fwa));
    q.total_work = sampled ? fw_smp[n] : fw_all[n];
    q.stride = sampled ? stride : 1;
    q.sample_win = (sampled && edge_sample) ? (const uint32_t*)(slot->d_blob + o_smp) : nullptr;
    q.level = level;
    q.use_prefix = use_prefix;
    q.rec_l0 = (flags & F_REC) ? 1 : 0;
    q.refine = (flags & F_REFINE) ? 1 : 0;
    q.cands_only = (flags & F_CANDS_ONLY) ? 1 : 0;
    if (use_driver && flags == 0) {
      qwk::DrvParams d;
      memset(&d, 0, sizeof d);
      d.plans = kp.plans; d.instrs = kp.instrs; d.cols = kp.cols; d.thresh = kp.thresh;
      d.first_work = (const uint32_t*)(slot->d_blob + (sampled ? o_fwds : o_fwd)); d.n_splits = n; d.total_work = sampled ? fw_dsm[n] : fw_drv[n];
      d.level = level; d.use_prefix = use_prefix; d.stride = sampled ? stride : 1;
      if (d.total_work == 0) return;
      const uint32_t dgrid = std::min<uint32_t>((d.total_work + QD_WARPS - 1) / QD_WARPS, (uint32_t)(sm_count * 4));
      if (mode == qwk::MODE_HIST) qwk::k_driver<qwk::MODE_HIST><<<dgrid, QD_WARPS * 32, 0, st>>>(d);
      else qwk::k_driver<qwk::MODE_COLLECT><<<dgrid, QD_WARPS * 32, 0, st>>>(d);
      stats.launches++;
      return;
    }
    if (q.total_work == 0) return;
    if (use_aggscan && mode == qwk::MODE_COLLECT && flags == 0) {
      qwk::AParams a;
      memset(&a, 0, sizeof a);
      a.plans = kp.plans; a.cols = kp.cols; a.aggs = kp.aggs;
      a.first_work = q.first_work; a.n_splits = n; a.total_work = q.total_work;
      a.sm = alay;
      int aocc = 1;
      CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&aocc, qwk::k_aggscan, QA_THREADS, alay.total));
      const uint32_t agrid = std::min<uint32_t>(q.total_work, (uint32_t)(sm_count * std::max(aocc, 1)));
      qwk::k_aggscan<<<agrid, QA_THREADS, alay.total, st>>>(a);
      stats.launches++;
      return;
    }
    if (use_union && flags == 0 && (mode == qwk::MODE_COLLECT || (level == 0 && !use_prefix))) {
      qwk::UParams u;
      memset(&u, 0, sizeof u);
      u.plans = kp.plans; u.instrs = kp.instrs; u.cols = kp.cols; u.thresh = kp.thresh;
      u.first_work = q.first_work; u.n_splits = n; u.total_work = q.total_work; u.stride = q.stride; u.W = sampled ? W_h : W;
      u.sm = mode == qwk::MODE_HIST ? ulay_h : ulay_c;
      // QWGPU_DYNAMIC_WORK=1: windows handed out one at a time from a counter instead of a static chunk per block.
      // Measured on the bench workload (uniform splits): 207 us against 194 us per launch — consecutive windows of a
      // block then belong to different splits, and the per-window plan switch sits on the producer's critical path —
      // with no gain for concurrent calls, so static chunks stay the default; the counter road is kept for skewed
      // corpora (validated: the full GPU suite passes in both modes).
      static const bool dynamic_work = getenv("QWGPU_DYNAMIC_WORK") != nullptr;
      if (dynamic_work && n_ctr < 64) u.work_ctr = (uint32_t*)(slot->d_scratch + s_ctr) + n_ctr++;
#ifdef QU_PROFILE
      static unsigned long long* d_prof = nullptr;
      if (!d_prof) CUDA_CHECK(cudaMalloc(&d_prof, 16 * 8));
      if (mode == qwk::MODE_COLLECT) { CUDA_CHECK(cudaMemsetAsync(d_prof, 0, 16 * 8, st)); u.prof = d_prof; }
#endif
      // cross-rank calls leave a few block slots free: the persistent grid would otherwise hold every SM's shared
      // memory, a concurrent call's NCCL kernel would take the place of one of its blocks, and that block — with its
      // static share of the windows — would only start when another one has finished (twice the kernel time)
      const uint32_t ugrid = std::min<uint32_t>(q.total_work, (uint32_t)(sm_count * QU_MINB) - (do_gather ? 4u : 0u));
      if (mode == qwk::MODE_HIST) qwk::k_union<qwk::MODE_HIST><<<ugrid, QU_THREADS, u.sm.total, st>>>(u);
      else qwk::k_union<qwk::MODE_COLLECT><<<ugrid, QU_THREADS, u.sm.total, st>>>(u);
#ifdef QU_PROFILE
      if (u.prof && getenv("QWGPU_UPROF")) {
        unsigned long long h[16];
        CUDA_CHECK(cudaMemcpyAsync(h, d_prof, sizeof h, cudaMemcpyDeviceToHost, st));
        wait_stream();
        const double np = (double)ugrid, nc = (double)h[15];
        fprintf(stderr, "[uprof] producer/CTA: total %.0f cyc, empty-wait %.0f, phaseA %.0f, window(A+B) %.0f, windows %.1f, slots %.1f | consumer/warp: total %.0f, full-wait %.0f, chain-wait %.0f (end-of-window %.0f), sweep %.0f, block-loop %.0f, blocks %.1f\n",
                h[0] / np, h[1] / np, h[2] / np, h[3] / np, h[4] / np, h[5] / np, h[8] / nc, h[9] / nc, h[10] / nc, h[11] / nc, h[12] / nc, h[13] / nc, h[14] / nc);
      }
#endif
      stats.launches++;
      return;
    }
    uint32_t grid = std::min<uint32_t>(q.total_work, (uint32_t)(sm_count * occ));
    if (mode == qwk::MODE_HIST && all_union && old_union && level == 0 && !use_prefix) qwk::k_window<qwk::MODE_HIST, true><<<grid, QW_THREADS, lay.total, st>>>(q);
    else if (mode == qwk::MODE_HIST) qwk::k_window<qwk::MODE_HIST, false><<<grid, QW_THREADS, lay.total, st>>>(q);
    else if (all_union && old_union) qwk::k_window<qwk::MODE_COLLECT, true><<<grid, QW_THREADS, lay.total, st>>>(q);
    else qwk::k_window<qwk::MODE_COLLECT, false><<<grid, QW_THREADS, lay.total, st>>>(q);
    stats.launches++;
  };
  const uint32_t sel_smem = 3 * 8 * QW_CAND_CAP;  // [all first words | 3 x QW_SEL_MAX survivors] or 3 x all (degenerate ties)
  auto run_collect = [&](uint32_t flags) {
    if (!(flags & F_CANDS_ONLY)) CUDA_CHECK(cudaMemsetAsync(slot->d_out, 0, out_bytes, st));
    CUDA_CHECK(cudaEventRecord(slot->ev2, st));
    launch_window(qwk::MODE_COLLECT, false, 0, 0, flags);
    CUDA_CHECK(cudaEventRecord(slot->ev3, st));
    if (any_topk) { qwk::k_select<<<n, 1024, sel_smem, st>>>(kp.plans, kp.cols); stats.launches++; }
    if (do_merge) {
      uint32_t* d_cut = (uint32_t*)(slot->d_scratch + s_cut);
      const qwk::SrcSplits src{kp.plans, (const uint32_t*)(slot->d_blob + o_rank), do_gather ? 1u : 0u};
      qwk::k_merge_prep<qwk::SrcSplits><<<1, 1024, 0, st>>>(src, n, merge->k, merge->order1, merge->order2, d_cut);
      const uint64_t threads = (uint64_t)n * kmax * 32;  // one warp per hit (warps of pruned hits leave at once)
      qwk::k_merge<qwk::SrcSplits><<<(uint32_t)((threads + 255) / 256), 256, 0, st>>>(src, d_cut, n, kmax, merge->k, merge->order1, merge->order2,
                                                          (qwk::DMergedHit*)(slot->d_out + o_merged + 64), (uint32_t*)(slot->d_out + o_merged));
      stats.launches += 2;
    }
    const size_t back = do_gather ? o_ghdr : out_bytes;  // (gathering: the final hits follow in the cross-rank phase)
    CUDA_CHECK(cudaMemcpyAsync(slot->h_out, slot->d_out, back, cudaMemcpyDeviceToHost, st));
    stats.d2h_bytes += back;
  };
  // a split's candidate set is good when it holds at least min(K, eligible) and did not overflow
  std::vector<uint32_t> state(n, 0);
  auto verify = [&]() -> bool {
    bool all = true;
    for (uint32_t i = 0; i < n; i++) {
      state[i] = 0;
      if (low[i].P.max_hits == 0) continue;
      const uint8_t* ob = slot->h_out + out_off[i];
      uint64_t eligible = ((const uint64_t*)ob)[1];
      uint32_t cand = *(const uint32_t*)(ob + 20);
      if (cand > QW_CAND_CAP || cand < std::min<uint64_t>(low[i].P.max_hits, eligible)) { state[i] = 1; all = false; }
    }
    return all;
  };

  const auto t_staged = tclock::now();
  CUDA_CHECK(cudaEventRecord(slot->ev0, st));
  CUDA_CHECK(cudaMemsetAsync(slot->d_scratch, 0, s_cand, st));  // thresholds, histograms, refinement state
  if (phrase_blocks) {
    // phrase pre-pass (inside the timed device region): every phrase of the batch becomes a posting list in
    // scratch (beyond s_cand: never cleared), read by every later pass
    uint32_t max_terms = 1;
    for (auto& L : low) for (auto& ph : L.phrases) max_terms = std::max(max_terms, ph.n_terms);
    const size_t psm = (size_t)QP_WARPS * QP_SMEM_WORDS(max_terms) * 4;
    qwk::k_phrase<<<(phrase_blocks + QP_WARPS - 1) / QP_WARPS, QP_WARPS * 32, psm, st>>>((const DPhrase*)(slot->d_blob + o_phr), n_phrases, phrase_blocks, max_terms);
    stats.launches++;
  }
  bool ok = true;
  float main_ms = 0;
  auto add_main = [&]() { float ms = 0; cudaEventElapsedTime(&ms, slot->ev2, slot->ev3); main_ms += ms; };
  if (any_topk && stride > 1) {
    // fast path: threshold from a 1/stride sample of the windows, verified after the collect pass
    launch_window(qwk::MODE_HIST, true, 0, 0, 0);
    qwk::k_pick<<<n, 256, 0, st>>>(kp.plans, kp.thresh, 0, edge_sample ? 2 : 1, stride, nullptr);
    stats.launches++;
    if (rec_l0) CUDA_CHECK(cudaMemsetAsync(slot->d_scratch + s_hist, 0, (size_t)n * QW_HIST_BINS * 4, st));
    run_collect(rec_l0 ? F_REC : 0);
    CUDA_CHECK(cudaEventRecord(slot->ev1, st));
    wait_stream();
    ok = verify();
    if (!ok) {
      float ms = 0;
      cudaEventElapsedTime(&ms, slot->ev0, slot->ev1);
      stats.gpu_time_us += ms * 1000.f;
      add_main();
      stats.exact_fallbacks++;
      CUDA_CHECK(cudaEventRecord(slot->ev0, st));
    }
  }
  if (!any_topk) {
    run_collect(0);
    CUDA_CHECK(cudaEventRecord(slot->ev1, st));
    wait_stream();
  } else if (stride == 1 || !ok) {
    // exact radix select over the composite key: one histogram pass per 11-bit digit until the
    // candidate set of every split fits QW_CAND_CAP. After a failed sampled threshold with the
    // level-0 histogram on record (refine), level 0 needs no pass at all, only the failing splits are
    // revisited, and windows whose best digit is below the threshold digit are skipped.
    const bool refine = !ok && rec_l0;
    const uint32_t* d_state = refine ? kp.split_state : nullptr;
    std::vector<DThresh> th(n);
    auto all_done = [&]() {
      for (uint32_t i = 0; i < n; i++) if (low[i].P.max_hits && (!refine || state[i]) && !th[i].done) return false;
      return true;
    };
    uint32_t level = 0;
    bool done = false;
    if (refine) {
      CUDA_CHECK(cudaMemcpyAsync(slot->d_scratch + s_state, state.data(), n * 4, cudaMemcpyHostToDevice, st));
      qwk::k_pick<<<n, 256, 0, st>>>(kp.plans, kp.thresh, 0, 0, 1, d_state);
      stats.launches++;
      CUDA_CHECK(cudaMemcpyAsync(th.data(), slot->d_scratch + s_thr, n * sizeof(DThresh), cudaMemcpyDeviceToHost, st));
      wait_stream();
      done = all_done();
      level = 1;
    } else {
      CUDA_CHECK(cudaMemsetAsync(slot->d_scratch, 0, s_cand, st));
    }
    for (; !done && level * QW_DIGIT_BITS < std::max(max_key_bits, 1u); level++) {
      CUDA_CHECK(cudaMemsetAsync(slot->d_scratch + s_hist, 0, (size_t)n * QW_HIST_BINS * 4, st));
      launch_window(qwk::MODE_HIST, false, level, level > 0 ? 1 : 0, refine ? F_REFINE : 0);
      qwk::k_pick<<<n, 256, 0, st>>>(kp.plans, kp.thresh, level, 0, 1, d_state);
      stats.launches++;
      CUDA_CHECK(cudaMemcpyAsync(th.data(), slot->d_scratch + s_thr, n * sizeof(DThresh), cudaMemcpyDeviceToHost, st));
      wait_stream();
      done = all_done();
    }
    run_collect(refine ? (F_REFINE | F_CANDS_ONLY) : 0);
    CUDA_CHECK(cudaEventRecord(slot->ev1, st));
    wait_stream();
    if (!verify()) fail(QWGPU_EINTERNAL, "top-K candidate selection failed verification");
  }
  if (do_gather) {
    // Cross-rank phase, after this rank's result is final (a verification fallback above must not repeat a
    // collective the other ranks run once): the rank's record -> every rank (one NCCL all-gather on this
    // call's stream) -> merged again on the device -> one more small copy back.
    uint32_t* d_cut = (uint32_t*)(slot->d_scratch + s_cut);
    qwk::k_rank_header<<<1, 32, 0, st>>>(kp.plans, n, (qwk::DRankHeader*)(slot->d_out + o_merged), gather->attempted, gather->successful, gather->n_failed);
    uint8_t* g_recv = slot->d_scratch + s_grecv;
    if (gather->allgather(gather->comm, slot->d_out + o_merged, g_recv, rec_bytes, (void*)st)) fail(QWGPU_EINTERNAL, "ncclAllGather failed");
    const qwk::SrcGathered gsrc{g_recv, (uint32_t)rec_bytes, 64u};
    uint32_t* g_cut = d_cut + std::max<uint32_t>(n, 64);
    qwk::k_merge_prep<qwk::SrcGathered><<<1, 1024, 0, st>>>(gsrc, (uint32_t)gather->world, merge->k, merge->order1, merge->order2, g_cut);
    const uint64_t gthreads = (uint64_t)gather->world * merge->k * 32;
    qwk::k_merge<qwk::SrcGathered><<<(uint32_t)((gthreads + 255) / 256), 256, 0, st>>>(gsrc, g_cut, (uint32_t)gather->world, merge->k, merge->k, merge->order1, merge->order2,
                                                                                    (qwk::DMergedHit*)(slot->d_out + o_final + 16), (uint32_t*)(slot->d_out + o_final));
    CUDA_CHECK(cudaMemcpy2DAsync(slot->d_out + o_ghdr, 64, g_recv, rec_bytes, 64, (size_t)gather->world, cudaMemcpyDeviceToDevice, st));
    CUDA_CHECK(cudaMemcpyAsync(slot->h_out + o_ghdr, slot->d_out + o_ghdr, out_bytes - o_ghdr, cudaMemcpyDeviceToHost, st));
    CUDA_CHECK(cudaEventRecord(slot->ev1, st));
    wait_stream();
    stats.launches += 4;
    stats.d2h_bytes += out_bytes - o_ghdr;
  }
  CUDA_CHECK(cudaGetLastError());
  {
    float ms = 0;
    cudaEventElapsedTime(&ms, slot->ev0, slot->ev1);
    stats.gpu_time_us += ms * 1000.f;
    add_main();
    stats.main_kernel_us = main_ms * 1000.f;
  }

  const auto t_searched = tclock::now();
  // ---- unpack ---------------------------------------------------------------------------------------
  for (uint32_t i = 0; i < n; i++) {
    SplitOutput& o = outs[idx[i]];
    const DSplitPlan& P = low[i].P;
    const uint8_t* ob = slot->h_out + out_off[i];
    o.num_hits = ((const uint64_t*)ob)[0];
    uint32_t nh = *(const uint32_t*)(ob + 16);
    if (!do_merge) {
      o.hits.assign((const QwHit*)(ob + 32), (const QwHit*)(ob + 32) + nh);
      if (P.key.kind[0] == QW_SORT_DOCID) for (auto& h : o.hits) { h.flags &= ~1u; h.v1 = 0; }
    }
    const QwAggCell* c = (const QwAggCell*)(ob + 32 + (do_merge ? 0 : (size_t)P.max_hits * sizeof(QwHit)));
    o.cells.assign(c, c + P.n_cells);
    for (auto& cell : o.cells) cell.min_mapped = ~cell.min_mapped;  // device keeps max(~m); see agg_stats
    o.postings_scored = low[i].postings;
    // SURVEY.md §8d algorithmic bytes: postings (+ fieldnorms, added at lowering) + column probes
    uint64_t bytes = low[i].alg_bytes;
    const SplitDev& s = *sp[idx[i]];
    auto col_bytes = [&](uint32_t c, uint64_t probes) {
      const QwImgColumn& ic = s.view.columns[c];
      uint64_t full = ((uint64_t)ic.num_vals * ic.bits + 7) / 8;
      return std::min<uint64_t>(probes * ((ic.bits + 7) / 8), full);
    };
    uint64_t driver = low[i].min_required_df == ~0ull ? P.num_docs : low[i].min_required_df;
    for (auto& rc : low[i].range_cols) bytes += col_bytes(rc.first, driver);
    const QwPlanHeader* ph = (const QwPlanHeader*)plans[idx[i]];
    for (int k = 0; k < 2; k++)
      if (ph->sort[k].kind == QW_SORT_COLUMN && ph->sort[k].column != 0xFFFFFFFFu && P.max_hits) bytes += col_bytes(ph->sort[k].column, o.num_hits);
    const QwAggNode* an = (const QwAggNode*)(plans[idx[i]] + sizeof(QwPlanHeader) + (size_t)ph->num_nodes * sizeof(QwPlanNode));
    for (uint32_t a = 0; a < ph->num_aggs; a++) if (an[a].column != 0xFFFFFFFFu) bytes += col_bytes(an[a].column, o.num_hits);
    o.algorithmic_bytes = bytes;
  }
  if (do_gather) {
    // the cross-rank result: hits carry GLOBAL split ranks (the caller owns the rank -> split id table)
    const uint32_t nm = *(const uint32_t*)(slot->h_out + o_final);
    const qwk::DMergedHit* mh = (const qwk::DMergedHit*)(slot->h_out + o_final + 16);
    merged->resize(nm);
    const bool by_doc = low[0].P.key.kind[0] == QW_SORT_DOCID;
    for (uint32_t j = 0; j < nm; j++) {
      MergedHit& m = (*merged)[j];
      m.hit = mh[j].hit; m.split = mh[j].split; m.pad = 0;
      if (by_doc) { m.hit.flags &= ~1u; m.hit.v1 = 0; }
    }
    rank_headers->resize(gather->world);
    memcpy(rank_headers->data(), slot->h_out + o_ghdr, (size_t)gather->world * 64);
  } else if (do_merge) {
    const uint32_t nm = *(const uint32_t*)(slot->h_out + o_merged);
    const qwk::DMergedHit* mh = (const qwk::DMergedHit*)(slot->h_out + o_merged + 64);
    merged->resize(nm);
    for (uint32_t j = 0; j < nm; j++) {
      MergedHit& m = (*merged)[j];
      m.hit = mh[j].hit;
      m.split = idx[mh[j].split];
      m.pad = 0;
      if (low[mh[j].split].P.key.kind[0] == QW_SORT_DOCID) { m.hit.flags &= ~1u; m.hit.v1 = 0; }
    }
  }
  if (trace) {
    auto us = [](tclock::time_point a, tclock::time_point b) { return (long)std::chrono::duration_cast<std::chrono::microseconds>(b - a).count(); };
    fprintf(stderr, "[qwgpu] search: lower %ld us, stage %ld us, launch+wait %ld us (device %.0f us), unpack %ld us\n", us(t_begin, t_lowered),
            us(t_lowered, t_staged), us(t_staged, t_searched), stats.gpu_time_us, us(t_searched, tclock::now()));
  }
}

}  // namespace qw
