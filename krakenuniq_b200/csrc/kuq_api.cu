// kuq_api.cu — host side of libkuq.so: the C ABI declared in include/kuq.h.
//
// Owns HBM (database range, taxonomy arrays, per-taxon state), the batch slots (stream + device and pinned
// host staging) and the host-side pieces of the path that are not data parallel: database header validation
// (krakendb.cpp:60-78,534-544), dense taxon numbering, work-unit cutting (classify.cpp:514-520) and the
// double-precision Ertl estimator (hyperloglogplus.cpp:722-753).  There is no CPU classification path: without
// an sm_100 device kuq_create fails with KUQ_E_NO_DEVICE.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "../../include/kuq.h"
#include "kuq_kernels.cuh"

using namespace kuq;

namespace {

constexpr uint64_t INDEX2_XOR_MASK = 0xe37e28c4271b5a2dULL;   // krakendb.cpp:45
constexpr uint32_t SLACK = 64;                                // bytes readable past the end of a bases buffer
constexpr uint32_t UMAP_CAP = 1u << 21;                       // (unit, taxon) pairs per batch
constexpr uint32_t USET_CAP = 1u << 22;                       // distinct (pair, code) entries per batch

struct Slot {
  cudaStream_t stream = nullptr;
  cudaEvent_t ev_k0 = nullptr, ev_k1 = nullptr, ev_stage[2] = {nullptr, nullptr}, ev_sync = nullptr;
  // device
  char *d_bases = nullptr, *d_clean = nullptr;
  uint64_t *d_offsets = nullptr;
  uint32_t *d_unit = nullptr, *d_call = nullptr, *d_nwin = nullptr, *d_codes = nullptr;
  // HLL mode rule bookkeeping (KUQ_HLL_PRELOAD), allocated on first use
  unsigned long long *u_keys = nullptr, *u_last = nullptr, *u_set_keys = nullptr;
  uint32_t *u_inserts = nullptr, *u_distinct = nullptr, *u_set_count = nullptr, *u_ncand = nullptr, *u_direct = nullptr;
  uint32_t u_direct_rows = 0;
  uint8_t *u_cand = nullptr, *u_taxon_cand = nullptr;
  uint64_t *d_canon = nullptr;                 // scratch between the stages
  uint32_t *d_bins = nullptr, *d_dense = nullptr, *d_codes_in = nullptr;
  unsigned long long *d_ovf = nullptr;          // hit-table pool for reads with > 32 distinct taxa
  uint64_t ovf_entries = 0;
  uint32_t *d_run_start = nullptr, *d_run_count = nullptr;
  uint2 *d_runs = nullptr;
  uint64_t runs_cap = 0;
  unsigned long long *d_scalars = nullptr;   // [0] run cursor, [1] n_classified, [2] chunk counter(u32) [3] error(u32)
  // pinned host
  uint32_t *h_call = nullptr, *h_nwin = nullptr, *h_run_start = nullptr, *h_run_count = nullptr, *h_codes = nullptr;
  uint32_t *h_unit = nullptr;
  kuq_run *h_runs = nullptr;
  uint64_t h_runs_cap = 0;
  unsigned long long *h_scalars = nullptr;
  // in-flight batch
  bool busy = false;
  bool timed = false;      // the timing events of this slot have been recorded at least once
  uint32_t n_reads = 0, flags = 0;
  uint64_t total_bases = 0;
  double kernel_ms = 0;
};

}  // namespace

struct CountsHost {
  std::vector<unsigned long long> n_kmers, n_reads;
  std::vector<uint32_t> hist;      // [n_sketch][64]
  std::vector<uint8_t> dense_flag;
  std::vector<uint32_t> distinct;
  std::vector<uint32_t> sparse_hist;   // [n_sketch][64] rank histogram of the sparse tier
  std::vector<unsigned long long> exact;   // KUQ_HLL_EXACT: [n_sketch] distinct k-mers per taxon
};

struct kuq_ctx {
  kuq_config cfg;
  CountsHost snap;                 // host copy of the per-taxon state, valid until the next batch
  bool snap_valid = false;
  int device = 0;
  int n_sm = 148;
  std::string err;
  std::vector<Slot> slots;
  uint64_t launches = 0;
  cudaStream_t aux = nullptr;

  // database
  bool db_owned = false;
  uint8_t *d_pairs = nullptr;
  uint64_t *d_offsets_owned = nullptr;
  const uint64_t *d_offsets = nullptr;
  uint64_t key_ct = 0, rec_base = 0;
  uint32_t k = 0, nt = 0, idx_type = 0;
  uint64_t bin_lo = 0, bin_hi = 0;
  bool db_staged = false, db_remapped = false;
  std::vector<uint32_t> db_taxids;        // distinct taxids of the staged records (ascending)
  std::vector<uint64_t> db_taxid_counts;
  std::vector<uint32_t> universe;         // taxids of all records of the database (optional)
  // device hash of the staged taxids (keys = taxid + 1)
  uint32_t *d_tx_keys = nullptr, *d_tx_dense = nullptr;
  unsigned long long *d_tx_counts = nullptr;
  uint32_t tx_cap = 0;

  // taxonomy
  bool tax_set = false, finalized = false;
  uint32_t quick_min = 0;                 // kuq_set_quick_mode: classify -q -m quick_min (0 = off)
  bool quick_stop = false;                // reads end at their quick_min-th hit (preloaded path) or not (-x path)
  bool mark_zero_hits = false;            // kuq_mark_zero_hits: lookups report stored taxon 0 as KUQ_CODE_FOUND_ZERO
  std::vector<uint32_t> tax_ids, tax_parents;
  std::vector<uint32_t> raw_of_dense;
  std::vector<uint32_t> parent_dense;     // host copy of d_parent (dense id of the parent, 0 = none)
  std::unordered_map<uint32_t, uint32_t> dense_of_raw;
  uint32_t n_taxa = 0, n_sketch = 0;
  uint32_t *d_parent = nullptr, *d_raw = nullptr;
  uint16_t *d_depth = nullptr;

  // per-taxon state
  uint8_t *d_regs = nullptr, *d_dense_flag = nullptr;
  unsigned long long *d_n_kmers = nullptr, *d_n_reads = nullptr;
  unsigned long long *d_sparse_slots = nullptr, *d_sparse_used = nullptr;
  uint32_t *d_sparse_distinct = nullptr;
  uint64_t sparse_cap = 0;
  ExactPair *d_exact = nullptr;           // KUQ_HLL_EXACT: the (taxon, k-mer) table and the per-taxon set sizes
  unsigned long long *d_exact_count = nullptr;
  uint64_t exact_cap = 0;

  // database streamed through HBM range by range (kuq_stream_*): two device buffers, one copy stream
  struct StreamBuf {
    uint8_t *d_pairs = nullptr;
    uint64_t *d_offsets = nullptr;
    cudaEvent_t ready = nullptr;
    uint64_t key_ct = 0, rec_base = 0, bin_lo = 0, bin_hi = 0;
    bool loaded = false;
  } sbuf[2];
  bool stream_open = false;
  uint64_t stream_cap_records = 0, stream_cap_bins = 0;
  cudaStream_t copy_stream = nullptr;
  uint32_t *d_stream_missing = nullptr;
  bool shard_counting = false;            // kuq_set_shard_counting: hits are counted by the GPU that finds them
  uint32_t extra_flags = 0;               // kuq_set_stats: KUQ_F_STATS for calls that take no flags
  uint32_t *d_sync_err = nullptr;         // set by a kuq_wait_flags that timed out
  bool merged_summary = false;            // kuq_set_sparse_summary: snap.sparse_hist / distinct hold cross-GPU sums
  std::vector<uint32_t> merged_hist, merged_distinct;
  uint64_t direct_upper = 0;              // upper bound of the keys in the sparse-tier set (reserve_direct_inserts)
  bool seen_dirty = false;                // counted hits flagged records since the last harvest (SEEN_BIT)
  uint64_t sparse_grown = 0;              // times the sparse-tier set was re-allocated at a harvest
  double harvest_ms = 0;                  // device time of the last harvest
  bool lca_mode = false;                  // kuq_set_lcas_batch ran: record values are LCA results, not classifiable
  // work-unit cutting across batches (classify.cpp:506-521)
  uint64_t unit_nt = 0;
  uint32_t unit_next = 0;
};

namespace {

void stream_close(kuq_ctx *ctx);

int fail(kuq_ctx *c, int code, const char *fmt, ...) {
  if (c) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    c->err = buf;
  }
  return code;
}

#define CU(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e__ = (call);                                                                      \
    if (e__ != cudaSuccess)                                                                        \
      return fail(ctx, KUQ_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)

template <typename T>
cudaError_t dmalloc(T **p, uint64_t n) { return cudaMalloc((void **)p, n * sizeof(T)); }
template <typename T>
cudaError_t hmalloc(T **p, uint64_t n) { return cudaMallocHost((void **)p, n * sizeof(T)); }

void free_slot(Slot &s) {
  cudaFree(s.d_bases); cudaFree(s.d_clean); cudaFree(s.d_offsets); cudaFree(s.d_unit); cudaFree(s.d_call);
  cudaFree(s.d_nwin); cudaFree(s.d_codes); cudaFree(s.d_run_start); cudaFree(s.d_run_count); cudaFree(s.d_runs);
  cudaFree(s.d_scalars); cudaFree(s.d_canon); cudaFree(s.d_bins); cudaFree(s.d_dense); cudaFree(s.d_codes_in); cudaFree(s.d_ovf);
  cudaFree(s.u_keys); cudaFree(s.u_last); cudaFree(s.u_set_keys); cudaFree(s.u_inserts); cudaFree(s.u_distinct);
  cudaFree(s.u_set_count); cudaFree(s.u_ncand); cudaFree(s.u_cand); cudaFree(s.u_taxon_cand); cudaFree(s.u_direct);
  cudaFreeHost(s.h_call); cudaFreeHost(s.h_nwin); cudaFreeHost(s.h_run_start); cudaFreeHost(s.h_run_count);
  cudaFreeHost(s.h_codes); cudaFreeHost(s.h_runs); cudaFreeHost(s.h_scalars); cudaFreeHost(s.h_unit);
  if (s.ev_k0) cudaEventDestroy(s.ev_k0);
  if (s.ev_k1) cudaEventDestroy(s.ev_k1);
  if (s.ev_stage[0]) cudaEventDestroy(s.ev_stage[0]);
  if (s.ev_stage[1]) cudaEventDestroy(s.ev_stage[1]);
  if (s.ev_sync) cudaEventDestroy(s.ev_sync);
  if (s.stream) cudaStreamDestroy(s.stream);
  s = Slot();
}

void free_db(kuq_ctx *ctx) {
  if (ctx->db_owned) { cudaFree(ctx->d_pairs); cudaFree(ctx->d_offsets_owned); }
  ctx->d_pairs = nullptr; ctx->d_offsets_owned = nullptr; ctx->d_offsets = nullptr;
  cudaFree(ctx->d_tx_keys); cudaFree(ctx->d_tx_dense); cudaFree(ctx->d_tx_counts);
  ctx->d_tx_keys = ctx->d_tx_dense = nullptr; ctx->d_tx_counts = nullptr;
  ctx->db_staged = false; ctx->db_remapped = false;
}

void free_tax_state(kuq_ctx *ctx) {
  cudaFree(ctx->d_parent); cudaFree(ctx->d_raw); cudaFree(ctx->d_depth);
  cudaFree(ctx->d_regs); cudaFree(ctx->d_dense_flag); cudaFree(ctx->d_n_kmers); cudaFree(ctx->d_n_reads);
  cudaFree(ctx->d_sparse_slots); cudaFree(ctx->d_sparse_used); cudaFree(ctx->d_sparse_distinct);
  cudaFree(ctx->d_exact); cudaFree(ctx->d_exact_count);
  ctx->d_exact = nullptr; ctx->d_exact_count = nullptr;
  ctx->d_parent = ctx->d_raw = nullptr; ctx->d_depth = nullptr; ctx->d_regs = ctx->d_dense_flag = nullptr;
  ctx->d_n_kmers = ctx->d_n_reads = nullptr; ctx->d_sparse_slots = ctx->d_sparse_used = nullptr;
  ctx->d_sparse_distinct = nullptr;
  ctx->finalized = false;
}

// ---- Ertl estimator (hyperloglogplus.cpp:373-422,738-752), same operation order as the reference ----------
double ertl_sigma(double x) {
  if (x == 1.0) return INFINITY;
  double prev, sigma_x = x, y = 1.0;
  do { prev = sigma_x; x *= x; sigma_x += x * y; y += y; } while (sigma_x != prev);
  return sigma_x;
}
double ertl_tau(double x) {
  if (x == 0.0 || x == 1.0) return 0.0;
  double prev, y = 1.0, tau_x = 1 - x;
  do { prev = tau_x; x = std::sqrt(x); y /= 2.0; tau_x -= std::pow(1 - x, 2) * y; } while (tau_x != prev);
  return tau_x / 3.0;
}
uint64_t ertl_from_hist(const int *C, size_t q, size_t m, uint64_t n_observed) {
  double est_denominator = m * ertl_tau(1.0 - double(C[q + 1]) / double(m));
  for (int k = (int)q; k >= 1; --k) { est_denominator += C[k]; est_denominator *= 0.5; }
  est_denominator += m * ertl_sigma(double(C[0]) / double(m));
  double m_sq_alpha_inf = (m / (2.0 * std::log(2))) * m;
  double est = m_sq_alpha_inf / est_denominator;
  return (double(n_observed) < est) ? n_observed : (uint64_t)std::round(est);
}
uint64_t ertl_dense_hist(const uint32_t *hist64, uint64_t n_observed) {
  int C[66];
  for (int i = 0; i < 64; i++) C[i] = (int)hist64[i];
  C[64] = C[65] = 0;
  return ertl_from_hist(C, 64 - HLL_P, HLL_M, n_observed);
}
// ertlCardinality of a sparse sketch (hyperloglogplus.cpp:726-729): q = 64 - 25, m = 2^25, C from
// sparseRegisterHistogram (:356-366): hist64[r] = distinct codes of encoded rank r, C[0] = m - |S|.
uint64_t ertl_sparse_hist(const uint32_t *hist64, uint64_t n_codes, uint64_t n_observed) {
  int C[66];
  memset(C, 0, sizeof C);
  for (int i = 1; i <= 40; i++) C[i] = (int)hist64[i];
  const size_t m = 1u << 25;
  C[0] = (int)(m - n_codes);
  return ertl_from_hist(C, 64 - 25, m, n_observed);
}

int alloc_slot(kuq_ctx *ctx, Slot &s) {
  const uint64_t mr = ctx->cfg.max_reads_per_batch, mb = ctx->cfg.max_bases_per_batch;
  CU(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
  CU(cudaEventCreate(&s.ev_k0));
  CU(cudaEventCreate(&s.ev_k1));
  CU(cudaEventCreate(&s.ev_stage[0]));
  CU(cudaEventCreate(&s.ev_stage[1]));
  CU(cudaEventCreateWithFlags(&s.ev_sync, cudaEventDisableTiming));
  CU(dmalloc(&s.d_bases, mb + SLACK));
  CU(dmalloc(&s.d_clean, mb + SLACK));
  CU(dmalloc(&s.d_offsets, mr + 4));   // + slack: offsets slices are bulk-copied in 16-byte units
  CU(dmalloc(&s.d_unit, mr));
  CU(dmalloc(&s.d_call, mr));
  CU(dmalloc(&s.d_nwin, mr));
  CU(dmalloc(&s.d_codes, mb + SLACK));
  CU(dmalloc(&s.d_canon, mb + SLACK));
  CU(dmalloc(&s.d_bins, mb + SLACK));
  CU(dmalloc(&s.d_dense, mb + SLACK));
  // worst case one table of < 4 * windows entries per read: 4 entries (64 B) per base always suffices, but reads that
  // need it are rare: a pool of max(bases / 4, 1 Mi) entries + the largest single table
  s.ovf_entries = std::max<uint64_t>(mb / 4, 1ull << 20);
  CU(dmalloc(&s.d_ovf, 2 * s.ovf_entries));
  CU(dmalloc(&s.d_run_start, mr));
  CU(dmalloc(&s.d_run_count, mr));
  // every resolving warp may leave one partly used block of 256 run slots behind (k_resolve)
  s.runs_cap = mb + SLACK + 256ull * (uint64_t)ctx->n_sm * 64;
  if (s.runs_cap > 0xFFFFFF00ull) s.runs_cap = 0xFFFFFF00ull;   // run indices are 32-bit
  CU(dmalloc(&s.d_runs, s.runs_cap));
  CU(dmalloc(&s.d_scalars, 8));
  CU(cudaMemset(s.d_scalars, 0, 8 * 8));           // kuq_sync_slot reads the error word even before the first batch
  CU(hmalloc(&s.h_call, mr));
  CU(hmalloc(&s.h_nwin, mr));
  CU(hmalloc(&s.h_run_start, mr));
  CU(hmalloc(&s.h_run_count, mr));
  CU(hmalloc(&s.h_unit, mr));
  CU(hmalloc(&s.h_scalars, 8));
  s.h_runs_cap = std::max<uint64_t>(mr * 8, 1024);
  CU(hmalloc(&s.h_runs, s.h_runs_cap));
  return KUQ_OK;
}

int check_slot(kuq_ctx *ctx, uint32_t slot) {
  if (!ctx) return KUQ_E_INVALID_ARG;
  if (slot >= ctx->slots.size()) return fail(ctx, KUQ_E_INVALID_ARG, "slot %u out of range (%zu slots)", slot, ctx->slots.size());
  return KUQ_OK;
}

// Scan the staged records for their distinct taxids (+counts): count_taxons (krakendb.cpp:90-113) on the GPU.
int collect_taxids(kuq_ctx *ctx) {
  uint32_t cap = 1u << 16;
  for (;;) {
    cudaFree(ctx->d_tx_keys); cudaFree(ctx->d_tx_counts); cudaFree(ctx->d_tx_dense);
    ctx->d_tx_keys = ctx->d_tx_dense = nullptr; ctx->d_tx_counts = nullptr;
    CU(dmalloc(&ctx->d_tx_keys, cap));
    CU(dmalloc(&ctx->d_tx_counts, cap));
    CU(dmalloc(&ctx->d_tx_dense, cap));
    CU(cudaMemsetAsync(ctx->d_tx_keys, 0, cap * 4ull, ctx->aux));
    CU(cudaMemsetAsync(ctx->d_tx_counts, 0, cap * 8ull, ctx->aux));
    uint32_t *d_over;
    CU(dmalloc(&d_over, 1));
    CU(cudaMemsetAsync(d_over, 0, 4, ctx->aux));
    launch_collect_taxids(ctx->d_pairs, ctx->key_ct, ctx->d_tx_keys, ctx->d_tx_counts, cap - 1, d_over, ctx->aux);
    ctx->launches++;
    uint32_t over = 0;
    CU(cudaMemcpyAsync(&over, d_over, 4, cudaMemcpyDeviceToHost, ctx->aux));
    CU(cudaStreamSynchronize(ctx->aux));
    cudaFree(d_over);
    if (over == 2) return fail(ctx, KUQ_E_DB_FORMAT, "taxid 0xFFFFFFFF is reserved");
    std::vector<uint32_t> keys(cap);
    std::vector<unsigned long long> counts(cap);
    CU(cudaMemcpy(keys.data(), ctx->d_tx_keys, cap * 4ull, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(counts.data(), ctx->d_tx_counts, cap * 8ull, cudaMemcpyDeviceToHost));
    uint64_t used = 0;
    for (uint32_t i = 0; i < cap; i++) used += keys[i] != 0;
    if (over == 1 || used * 2 > cap) {            // too full: the probe chains got long or overflowed
      if (cap >= (1u << 28)) return fail(ctx, KUQ_E_CAPACITY, "more than 2^27 distinct taxids in the database");
      cap <<= 2;
      continue;
    }
    std::vector<std::pair<uint32_t, uint64_t>> v;
    v.reserve(used);
    for (uint32_t i = 0; i < cap; i++) if (keys[i]) v.emplace_back(keys[i] - 1, counts[i]);
    std::sort(v.begin(), v.end());
    ctx->db_taxids.clear(); ctx->db_taxid_counts.clear();
    for (auto &pr : v) { ctx->db_taxids.push_back(pr.first); ctx->db_taxid_counts.push_back(pr.second); }
    ctx->tx_cap = cap;
    return KUQ_OK;
  }
}

// Dense numbering: 0 = "no taxon", 1 = taxid 1 (the reference's hard-wired root, krakenutil.cpp:96,106), then every
// taxid stored in database records (these own HLL sketches), then the remaining taxonomy nodes; each group
// ascending by taxid.  Builds the flattened Parent_map and uploads everything.
int finalize(kuq_ctx *ctx) {
  if (ctx->finalized) return KUQ_OK;
  if (!ctx->db_staged) return fail(ctx, KUQ_E_STATE, "no database staged");
  if (!ctx->tax_set) return fail(ctx, KUQ_E_STATE, "no taxonomy set");
  std::vector<uint32_t> dbt = ctx->universe.empty() ? ctx->db_taxids : ctx->universe;
  std::sort(dbt.begin(), dbt.end());
  dbt.erase(std::unique(dbt.begin(), dbt.end()), dbt.end());
  std::vector<uint32_t> &raw = ctx->raw_of_dense;
  raw.clear();
  ctx->dense_of_raw.clear();
  raw.push_back(0);
  raw.push_back(1);
  for (uint32_t t : dbt) if (t > 1) raw.push_back(t);
  ctx->n_sketch = (uint32_t)raw.size();
  for (uint32_t i = 0; i < raw.size(); i++) ctx->dense_of_raw[raw[i]] = i;
  std::vector<uint32_t> rest;
  for (uint32_t t : ctx->tax_ids) if (!ctx->dense_of_raw.count(t)) rest.push_back(t);
  for (uint32_t t : ctx->tax_parents) if (t && !ctx->dense_of_raw.count(t)) rest.push_back(t);   // parents without a row
  std::sort(rest.begin(), rest.end());
  rest.erase(std::unique(rest.begin(), rest.end()), rest.end());
  for (uint32_t t : rest) { ctx->dense_of_raw[t] = (uint32_t)raw.size(); raw.push_back(t); }
  ctx->n_taxa = (uint32_t)raw.size();
  // staged taxids must all be numbered
  for (uint32_t t : ctx->db_taxids)
    if (!ctx->dense_of_raw.count(t) || ctx->dense_of_raw[t] >= ctx->n_sketch)
      return fail(ctx, KUQ_E_STATE, "staged records hold taxid %u that is not in the declared taxid universe", t);

  // Parent_map (taxdb.hpp:383-398): every taxonomy row has an entry; rows whose parent is themselves / 0 map to
  // 0.  A parent id WITHOUT a row of its own is still walked to by resolve_tree/lca (then the walk stops:
  // "No parent for ..." krakenutil.cpp:166-169), so such ids got a dense id above with parent 0.
  std::vector<uint32_t> parent(ctx->n_taxa, 0);
  for (size_t i = 0; i < ctx->tax_ids.size(); i++) {
    uint32_t t = ctx->tax_ids[i], p = ctx->tax_parents[i];
    if (t == 0) continue;
    parent[ctx->dense_of_raw[t]] = (p == t || p == 0) ? 0 : ctx->dense_of_raw[p];
  }
  // depth = steps until the chain ends at 0 or at dense 1 (lca() stops at taxid 1, krakenutil.cpp:96,106)
  std::vector<uint16_t> depth(ctx->n_taxa, 0);
  std::vector<uint8_t> state(ctx->n_taxa, 0);   // 0 new, 1 on stack, 2 done
  state[0] = state[1] = 2;
  std::vector<uint32_t> stack;
  for (uint32_t i = 2; i < ctx->n_taxa; i++) {
    if (state[i]) continue;
    uint32_t x = i;
    stack.clear();
    while (state[x] == 0) { state[x] = 1; stack.push_back(x); x = parent[x]; }
    if (state[x] == 1) return fail(ctx, KUQ_E_TAXONOMY, "cycle in the taxonomy at taxid %u", raw[x]);
    uint32_t d = depth[x];
    while (!stack.empty()) {
      uint32_t y = stack.back(); stack.pop_back();
      d++;
      if (d > 65000) return fail(ctx, KUQ_E_TAXONOMY, "taxonomy deeper than 65000 levels");
      depth[y] = (uint16_t)d; state[y] = 2;
    }
  }
  free_tax_state(ctx);
  ctx->parent_dense = parent;
  CU(dmalloc(&ctx->d_parent, ctx->n_taxa));
  CU(dmalloc(&ctx->d_raw, ctx->n_taxa));
  CU(dmalloc(&ctx->d_depth, ctx->n_taxa));
  CU(cudaMemcpy(ctx->d_parent, parent.data(), ctx->n_taxa * 4ull, cudaMemcpyHostToDevice));
  CU(cudaMemcpy(ctx->d_raw, raw.data(), ctx->n_taxa * 4ull, cudaMemcpyHostToDevice));
  CU(cudaMemcpy(ctx->d_depth, depth.data(), ctx->n_taxa * 2ull, cudaMemcpyHostToDevice));
  CU(dmalloc(&ctx->d_regs, (uint64_t)ctx->n_sketch * HLL_M));
  CU(dmalloc(&ctx->d_dense_flag, ctx->n_sketch));
  CU(dmalloc(&ctx->d_n_kmers, ctx->n_sketch));
  CU(dmalloc(&ctx->d_n_reads, ctx->n_taxa));
  CU(cudaMemset(ctx->d_regs, 0, (uint64_t)ctx->n_sketch * HLL_M));
  CU(cudaMemset(ctx->d_dense_flag, 0, ctx->n_sketch));
  CU(cudaMemset(ctx->d_n_kmers, 0, ctx->n_sketch * 8ull));
  CU(cudaMemset(ctx->d_n_reads, 0, ctx->n_taxa * 8ull));
  if (ctx->cfg.hll_mode == KUQ_HLL_EXACT) {
    ctx->exact_cap = ctx->cfg.sparse_set_slots;            // entries of 16 B
    CU(dmalloc(&ctx->d_exact, ctx->exact_cap));
    CU(dmalloc(&ctx->d_exact_count, ctx->n_sketch));
    CU(cudaMemset(ctx->d_exact, 0, ctx->exact_cap * 16ull));
    CU(cudaMemset(ctx->d_exact_count, 0, ctx->n_sketch * 8ull));
  } else if (ctx->cfg.hll_mode != KUQ_HLL_DENSE_ONLY) {
    ctx->sparse_cap = ctx->cfg.sparse_set_slots;
    CU(dmalloc(&ctx->d_sparse_slots, ctx->sparse_cap));
    CU(dmalloc(&ctx->d_sparse_used, 1));
    CU(dmalloc(&ctx->d_sparse_distinct, ctx->n_sketch));
    CU(cudaMemset(ctx->d_sparse_slots, 0, ctx->sparse_cap * 8ull));
    CU(cudaMemset(ctx->d_sparse_used, 0, 8));
    CU(cudaMemset(ctx->d_sparse_distinct, 0, ctx->n_sketch * 4ull));
  }
  ctx->finalized = true;
  return KUQ_OK;
}

// rewrite the staged record values taxid → dense id (once per staged range)
int remap_db(kuq_ctx *ctx) {
  if (ctx->db_remapped) return KUQ_OK;
  std::vector<uint32_t> keys(ctx->tx_cap), dense(ctx->tx_cap, 0);
  CU(cudaMemcpy(keys.data(), ctx->d_tx_keys, ctx->tx_cap * 4ull, cudaMemcpyDeviceToHost));
  for (uint32_t i = 0; i < ctx->tx_cap; i++)
    if (keys[i]) {
      auto it = ctx->dense_of_raw.find(keys[i] - 1);
      if (it == ctx->dense_of_raw.end() || it->second >= ctx->n_sketch)
        return fail(ctx, KUQ_E_STATE, "staged records hold taxid %u outside the numbered universe", keys[i] - 1);
      dense[i] = it->second;
    }
  CU(cudaMemcpy(ctx->d_tx_dense, dense.data(), ctx->tx_cap * 4ull, cudaMemcpyHostToDevice));
  uint32_t *d_missing;
  CU(dmalloc(&d_missing, 1));
  CU(cudaMemset(d_missing, 0, 4));
  launch_remap_values(ctx->d_pairs, ctx->key_ct, ctx->d_tx_keys, ctx->d_tx_dense, ctx->tx_cap - 1, d_missing,
                      ctx->k >= 32 ? ~0ull : ((1ull << (2 * ctx->k)) - 1), ctx->aux);
  ctx->launches++;
  uint32_t missing = 0;
  CU(cudaMemcpyAsync(&missing, d_missing, 4, cudaMemcpyDeviceToHost, ctx->aux));
  CU(cudaStreamSynchronize(ctx->aux));
  cudaFree(d_missing);
  if (missing) return fail(ctx, KUQ_E_STATE, "internal: a record value was missing from the taxid table");
  ctx->db_remapped = true;
  return KUQ_OK;
}

// Sparse HLL tier of the hits: the fused lookup only flags the records it counted (SEEN_BIT); here the flagged
// records of the staged range become (taxon, encoded hash) keys of the device set — the union the reference builds
// with `taxon_counts[t] += ...` over sparse sketches (hyperloglogplus.cpp:600-603) — and the flags are cleared.
// The number of keys is known before they are inserted, so the set grows here instead of failing mid-batch.
// Re-allocate the sparse-tier set with `cap` slots and re-insert its keys.  All slots must be idle.
int grow_sparse_set(kuq_ctx *ctx, uint64_t cap) {
  unsigned long long *bigger = nullptr;
  uint32_t *d_err = nullptr;
  if (dmalloc(&bigger, cap) != cudaSuccess) {
    (void)cudaGetLastError();
    return fail(ctx, KUQ_E_NOMEM, "sparse-tier set: no room to grow from %llu to %llu slots", (unsigned long long)ctx->sparse_cap, (unsigned long long)cap);
  }
  CU(dmalloc(&d_err, 1));
  CU(cudaMemsetAsync(d_err, 0, 4, ctx->aux));
  CU(cudaMemsetAsync(bigger, 0, cap * 8ull, ctx->aux));
  SparseSet nb;
  nb.slots = bigger; nb.mask = cap - 1; nb.n_used = ctx->d_sparse_used; nb.distinct = ctx->d_sparse_distinct;
  launch_sparse_rehash(ctx->d_sparse_slots, ctx->sparse_cap, nb, d_err, ctx->aux);
  ctx->launches++;
  CU(cudaStreamSynchronize(ctx->aux));
  cudaFree(d_err);
  cudaFree(ctx->d_sparse_slots);
  ctx->d_sparse_slots = bigger;
  ctx->sparse_cap = cap;
  ctx->sparse_grown++;
  return KUQ_OK;
}

// The resolve half inserts (taxon, code) pairs straight into the set — at most one per window of the batch.  Make room
// BEFORE the batch instead of failing in the middle of it: `direct_upper` bounds the keys inserted that way since the
// last exact count; when the bound says the set could pass a load factor of 0.8 the exact fill is read back, and only
// if that still does not fit the set doubles (all slots drained first).
int reserve_direct_inserts(kuq_ctx *ctx, uint64_t windows) {
  if (!ctx->d_sparse_slots) return KUQ_OK;
  if ((ctx->direct_upper + windows) * 10 <= ctx->sparse_cap * 8) { ctx->direct_upper += windows; return KUQ_OK; }
  for (auto &s : ctx->slots) CU(cudaStreamSynchronize(s.stream));
  std::vector<uint32_t> distinct(ctx->n_sketch);
  CU(cudaMemcpy(distinct.data(), ctx->d_sparse_distinct, ctx->n_sketch * 4ull, cudaMemcpyDeviceToHost));
  uint64_t used = 0;
  for (uint32_t v : distinct) used += v;
  ctx->direct_upper = used;
  if ((used + windows) * 10 > ctx->sparse_cap * 8) {
    uint64_t cap = ctx->sparse_cap;
    while ((used + windows) * 10 > cap * 6) cap <<= 1;
    int rc = grow_sparse_set(ctx, cap);
    if (rc) return rc;
  }
  ctx->direct_upper += windows;
  return KUQ_OK;
}

int harvest_seen(kuq_ctx *ctx, bool discard) {
  if (!ctx->seen_dirty) return KUQ_OK;
  CU(cudaSetDevice(ctx->device));
  for (auto &s : ctx->slots) CU(cudaStreamSynchronize(s.stream));
  ctx->seen_dirty = false;
  if (!ctx->d_pairs || !ctx->key_ct) return KUQ_OK;
  const uint64_t key_mask = ctx->k >= 32 ? ~0ull : ((1ull << (2 * ctx->k)) - 1);
  SparseSet ss;
  ss.slots = ctx->d_sparse_slots; ss.mask = ctx->sparse_cap ? ctx->sparse_cap - 1 : 0; ss.n_used = ctx->d_sparse_used;
  ss.distinct = ctx->d_sparse_distinct;
  unsigned long long *d_stat;
  CU(dmalloc(&d_stat, 2));
  CU(cudaMemsetAsync(d_stat, 0, 16, ctx->aux));
  cudaEvent_t e0, e1;
  CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
  CU(cudaEventRecord(e0, ctx->aux));
  if (discard || !ctx->d_sparse_slots) {
    launch_harvest_seen(ctx->d_pairs, ctx->key_ct, key_mask, ctx->d_dense_flag, ss, d_stat, reinterpret_cast<uint32_t *>(d_stat + 1), 2, ctx->aux);
    ctx->launches++;
  } else {
    launch_harvest_seen(ctx->d_pairs, ctx->key_ct, key_mask, ctx->d_dense_flag, ss, d_stat, reinterpret_cast<uint32_t *>(d_stat + 1), 0, ctx->aux);
    ctx->launches++;
    unsigned long long n_new = 0;
    CU(cudaMemcpyAsync(&n_new, d_stat, 8, cudaMemcpyDeviceToHost, ctx->aux));
    std::vector<uint32_t> distinct(ctx->n_sketch);
    CU(cudaMemcpyAsync(distinct.data(), ctx->d_sparse_distinct, ctx->n_sketch * 4ull, cudaMemcpyDeviceToHost, ctx->aux));
    CU(cudaStreamSynchronize(ctx->aux));
    uint64_t used = 0;
    for (uint32_t v : distinct) used += v;
    if ((used + n_new) * 10 > ctx->sparse_cap * 8) {             // keep the load factor below 0.8
      uint64_t cap = ctx->sparse_cap;
      while ((used + n_new) * 10 > cap * 6) cap <<= 1;
      int grc = grow_sparse_set(ctx, cap);
      if (grc) { cudaFree(d_stat); return grc; }
      ss.slots = ctx->d_sparse_slots; ss.mask = ctx->sparse_cap - 1;
    }
    ctx->direct_upper = used + n_new;
    // Insert in record order.  (Round 2 also tried staging the keys by table slice so that the inserts of a slice are
    // L2-resident — profiles/README.md: read-only probes got 3x faster, but NEW keys did not (each one still costs a
    // DRAM sector fetch and a dirty sector write-back), and new keys are what a harvest mostly sees.)
    launch_harvest_seen(ctx->d_pairs, ctx->key_ct, key_mask, ctx->d_dense_flag, ss, d_stat, reinterpret_cast<uint32_t *>(d_stat + 1), 1, ctx->aux);
    ctx->launches++;
    CU(cudaStreamSynchronize(ctx->aux));
    if (getenv("KUQ_TIMING")) fprintf(stderr, "[timing] harvest: %llu flagged records, %llu slots\n", n_new, (unsigned long long)ctx->sparse_cap);
  }
  CU(cudaEventRecord(e1, ctx->aux));
  unsigned long long st[2] = {0, 0};
  CU(cudaMemcpyAsync(st, d_stat, 16, cudaMemcpyDeviceToHost, ctx->aux));
  CU(cudaStreamSynchronize(ctx->aux));
  float ms = 0;
  cudaEventElapsedTime(&ms, e0, e1);
  ctx->harvest_ms = ms;
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaFree(d_stat);
  ctx->snap_valid = false;
  if ((uint32_t)st[1]) return fail(ctx, KUQ_E_CAPACITY, "sparse-tier set saturated during the harvest (%llu slots)", (unsigned long long)ctx->sparse_cap);
  return KUQ_OK;
}

int ensure_ready(kuq_ctx *ctx) {
  int rc = finalize(ctx);
  if (rc) return rc;
  return remap_db(ctx);
}

void set_unit_ptrs(Params &p, Slot &s);
int prepare_unit_map(kuq_ctx *ctx, Slot &s) {
  if (ctx->cfg.hll_mode != KUQ_HLL_PRELOAD) return KUQ_OK;
  if (!s.u_keys) {
    CU(dmalloc(&s.u_keys, UMAP_CAP));
    CU(dmalloc(&s.u_last, UMAP_CAP));
    CU(dmalloc(&s.u_inserts, UMAP_CAP));
    CU(dmalloc(&s.u_distinct, UMAP_CAP));
    CU(dmalloc(&s.u_cand, UMAP_CAP));
    CU(dmalloc(&s.u_taxon_cand, ctx->n_sketch));
    CU(dmalloc(&s.u_ncand, 1));
    CU(dmalloc(&s.u_set_keys, USET_CAP));
    CU(dmalloc(&s.u_set_count, USET_CAP));
    // dense (unit, taxon) table: the units a batch can hold when the library cuts them, at most 64 Mi counters
    uint64_t rows = ctx->cfg.max_bases_per_batch / std::max<uint64_t>(ctx->cfg.work_unit_size, 1) + 8;
    rows = std::min<uint64_t>(rows, (64ull << 20) / std::max<uint32_t>(ctx->n_sketch, 1));
    s.u_direct_rows = (uint32_t)rows;
    if (rows) CU(dmalloc(&s.u_direct, rows * ctx->n_sketch));
  }
  Params tmp;
  set_unit_ptrs(tmp, s);
  launch_unit_clear(tmp.units, ctx->n_sketch, ctx->n_sm, s.stream);
  ctx->launches++;
  return KUQ_OK;
}

// process_file's unit cutting (classify.cpp:506-521): reads join the open unit until its length reaches -u.
void cut_units(kuq_ctx *ctx, const uint64_t *offsets, uint32_t n, uint32_t *unit) {
  const uint64_t wus = ctx->cfg.work_unit_size;
  for (uint32_t i = 0; i < n; i++) {
    unit[i] = ctx->unit_next;
    ctx->unit_nt += offsets[i + 1] - offsets[i];
    if (ctx->unit_nt >= wus) { ctx->unit_next++; ctx->unit_nt = 0; }
  }
}

void set_unit_ptrs(Params &p, Slot &s) {
  p.units.keys = s.u_keys;
  p.units.inserts = s.u_inserts;
  p.units.distinct = s.u_distinct;
  p.units.last = s.u_last;
  p.units.cand = s.u_cand;
  p.units.mask = UMAP_CAP - 1;
  p.units.taxon_cand = s.u_taxon_cand;
  p.units.n_cand = s.u_ncand;
  p.units.set_keys = s.u_set_keys;
  p.units.set_count = s.u_set_count;
  p.units.set_mask = USET_CAP - 1;
  p.units.direct = s.u_direct;
  p.units.direct_rows = s.u_direct_rows;
}

void fill_params(kuq_ctx *ctx, Slot &s, Params &p, const char *d_bases, const uint64_t *d_offsets,
                 const uint32_t *d_unit, uint32_t n_reads, uint32_t flags) {
  memset(&p, 0, sizeof p);
  p.db.pairs = ctx->d_pairs;
  p.db.offsets = ctx->d_offsets;
  p.db.rec_base = ctx->rec_base;
  p.db.key_mask = ctx->k >= 32 ? ~0ull : ((1ull << (2 * ctx->k)) - 1);
  p.db.bin_lo = (uint32_t)ctx->bin_lo;
  p.db.bin_hi = (uint32_t)ctx->bin_hi;
  p.db.k = ctx->k;
  p.db.nt = ctx->nt;
  p.db.xor_mask = (uint32_t)((ctx->idx_type == 1 ? 0ull : INDEX2_XOR_MASK) & ((1ull << (2 * ctx->nt)) - 1));
  p.db.n_mini = ctx->k - ctx->nt + 1;
  p.tax.parent = ctx->d_parent;
  p.tax.depth = ctx->d_depth;
  p.tax.raw = ctx->d_raw;
  p.tax.n_taxa = ctx->n_taxa;
  p.tax.n_sketch = ctx->n_sketch;
  p.bases = d_bases;
  p.offsets = d_offsets;
  p.unit_id = d_unit;
  p.clean = s.d_clean;
  p.n_reads = n_reads;
  p.n_chunks = (n_reads + CHUNK_READS - 1) / CHUNK_READS;
  p.flags = flags;
  p.hll_mode = ctx->cfg.hll_mode;
  p.call = s.d_call;
  p.n_windows = s.d_nwin;
  p.codes = s.d_codes;
  p.total_bases = s.total_bases;
  p.canon = s.d_canon;
  p.bins = s.d_bins;
  p.codes_dense = s.d_dense;
  p.run_start = s.d_run_start;
  p.run_count = s.d_run_count;
  p.runs = s.d_runs;
  p.run_cursor = s.d_scalars;
  p.runs_capacity = s.runs_cap;
  p.n_classified = s.d_scalars + 1;
  p.chunk_counter = reinterpret_cast<uint32_t *>(s.d_scalars + 2);
  p.error_flag = reinterpret_cast<uint32_t *>(s.d_scalars + 3);
  p.stats = s.d_scalars + 4;
  p.ovf_mem = s.d_ovf;
  p.ovf_cursor = s.d_scalars + 6;
  p.ovf_capacity = s.ovf_entries;
  p.regs = ctx->d_regs;
  p.n_kmers = ctx->d_n_kmers;
  p.n_reads_ctr = ctx->d_n_reads;
  p.dense_flag = ctx->d_dense_flag;
  p.sparse.slots = ctx->d_sparse_slots;
  p.sparse.mask = ctx->sparse_cap ? ctx->sparse_cap - 1 : 0;
  p.sparse.n_used = ctx->d_sparse_used;
  p.sparse.distinct = ctx->d_sparse_distinct;
  p.exact.slots = ctx->d_exact;
  p.exact.mask = ctx->exact_cap ? ctx->exact_cap - 1 : 0;
  p.exact.count = ctx->d_exact_count;
  set_unit_ptrs(p, s);
}

int launch_on_slot(kuq_ctx *ctx, Slot &s, int mode, Params &p) {
  if (ctx->lca_mode) return fail(ctx, KUQ_E_STATE, "this context built a database (kuq_set_lcas_batch): stage it anew to classify");
  ctx->snap_valid = false;
  p.flags |= ctx->extra_flags;
  if (mode == MODE_LOOKUP && ctx->mark_zero_hits) p.flags |= F_FOUND_ZERO;
  if (ctx->shard_counting && mode != MODE_FUSED && !ctx->mark_zero_hits && !ctx->quick_min &&
      ctx->cfg.hll_mode != KUQ_HLL_EXACT) {
    p.flags |= F_SHARD_COUNTING;
    if (mode == MODE_LOOKUP && p.n_reads && ctx->cfg.hll_mode <= KUQ_HLL_CHUNKED) ctx->seen_dirty = true;
  }
  ctx->merged_summary = false;
  if (mode != MODE_LOOKUP && ctx->quick_min) {           // "Q:hits" replaces the hit list (classify.cpp:989-990)
    p.quick_min = ctx->quick_min;
    p.quick_stop = ctx->quick_stop;
    p.flags |= KUQ_F_NO_RUNS;
    s.flags |= KUQ_F_NO_RUNS;
  }
  if (mode == MODE_RESOLVE && !(p.flags & KUQ_F_NO_COUNTS) && ctx->cfg.hll_mode <= KUQ_HLL_CHUNKED && p.n_reads) {
    int rrc = reserve_direct_inserts(ctx, s.total_bases);
    if (rrc) return rrc;
    // the set may have moved
    p.sparse.slots = ctx->d_sparse_slots;
    p.sparse.mask = ctx->sparse_cap ? ctx->sparse_cap - 1 : 0;
  }
  const bool units = mode != MODE_LOOKUP && ctx->cfg.hll_mode == KUQ_HLL_PRELOAD && p.unit_id && !(p.flags & KUQ_F_NO_COUNTS);
  if (units) {
    int rc = prepare_unit_map(ctx, s);
    if (rc) return rc;
    set_unit_ptrs(p, s);                 // the map is allocated on first use
  } else if (ctx->cfg.hll_mode == KUQ_HLL_PRELOAD) {
    p.unit_id = nullptr;                 // no per-unit bookkeeping for this call
  }
  CU(cudaMemsetAsync(s.d_scalars, 0, 8 * 8, s.stream));
  CU(cudaEventRecord(s.ev_k0, s.stream));
  CU(cudaEventRecord(s.ev_stage[0], s.stream));
  CU(cudaEventRecord(s.ev_stage[1], s.stream));
  if (p.n_reads) ctx->launches += launch_classify(mode, p, ctx->n_sm, s.stream, s.ev_stage);
  // the fused path flags the records of its counted hits (k_lookup); quick / exact runs go through the other halves
  if (p.n_reads && mode == MODE_FUSED && !(p.flags & KUQ_F_NO_COUNTS) && ctx->cfg.hll_mode <= KUQ_HLL_CHUNKED &&
      !(ctx->quick_min && ctx->quick_stop))
    ctx->seen_dirty = true;
  CU(cudaEventRecord(s.ev_k1, s.stream));
  s.timed = true;
  // HLL mode rule: which taxa have a sketch that converted to dense (SURVEY.md App. C)
  if (p.n_reads && mode != MODE_LOOKUP && !(p.flags & KUQ_F_NO_COUNTS)) {
    if (units) ctx->launches += launch_unit_accounting(p, ctx->n_sm, s.stream);
    else if (ctx->cfg.hll_mode == KUQ_HLL_CHUNKED) {
      launch_flag_dense_global(ctx->d_sparse_distinct, ctx->d_dense_flag, ctx->n_sketch, s.stream);
      ctx->launches++;
    }
  }
  CU(cudaGetLastError());
  return KUQ_OK;
}

}  // namespace

// ===========================================================================================================
extern "C" {

const char *kuq_version(void) { return "libkuq 0.2.0 sm_100a"; }

int kuq_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { (void)cudaGetLastError(); return 0; }
  int usable = 0;
  for (int d = 0; d < n; d++) {
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, d) == cudaSuccess && prop.major >= 10) usable = d + 1;
  }
  return usable;
}

const char *kuq_strerror(int code) {
  switch (code) {
    case KUQ_OK: return "ok";
    case KUQ_E_INVALID_ARG: return "invalid argument";
    case KUQ_E_CUDA: return "CUDA error";
    case KUQ_E_NO_DEVICE: return "no sm_100 CUDA device (libkuq has no CPU path)";
    case KUQ_E_DB_FORMAT: return "database in improper format";
    case KUQ_E_UNSUPPORTED_K: return "unsupported k (only 8-byte keys: k = 29..31)";
    case KUQ_E_STATE: return "call order / state error";
    case KUQ_E_CAPACITY: return "capacity exceeded";
    case KUQ_E_NOMEM: return "out of memory";
    case KUQ_E_TAXA_OVERFLOW: return "hit-table pool exhausted (too many reads with more than 32 distinct taxa in one batch)";
    case KUQ_E_TAXONOMY: return "malformed taxonomy";
    default: return "unknown error";
  }
}

const char *kuq_last_error(const kuq_ctx *ctx) { return ctx ? ctx->err.c_str() : ""; }

void kuq_config_default(kuq_config *cfg) {
  if (!cfg) return;
  memset(cfg, 0, sizeof *cfg);
  cfg->device = 0;
  cfg->n_slots = 2;
  cfg->max_reads_per_batch = 1u << 20;
  cfg->max_bases_per_batch = 160ull << 20;
  cfg->work_unit_size = 500000;           // DEF_WORK_UNIT_SIZE, classify.cpp:38
  cfg->hll_mode = KUQ_HLL_PRELOAD;
  cfg->sparse_set_slots = 1ull << 26;
}

int kuq_create(const kuq_config *cfg_in, kuq_ctx **out) {
  if (!out) return KUQ_E_INVALID_ARG;
  *out = nullptr;
  kuq_config cfg;
  kuq_config_default(&cfg);
  if (cfg_in) {
    cfg = *cfg_in;
    kuq_config d;
    kuq_config_default(&d);
    if (!cfg.n_slots) cfg.n_slots = d.n_slots;
    if (!cfg.max_reads_per_batch) cfg.max_reads_per_batch = d.max_reads_per_batch;
    if (!cfg.max_bases_per_batch) cfg.max_bases_per_batch = d.max_bases_per_batch;
    if (!cfg.work_unit_size) cfg.work_unit_size = d.work_unit_size;
    if (!cfg.sparse_set_slots) cfg.sparse_set_slots = d.sparse_set_slots;
  }
  if (cfg.hll_mode > KUQ_HLL_EXACT || cfg.n_slots > 16) return KUQ_E_INVALID_ARG;
  // round the sparse set to a power of two
  uint64_t sc = 1024;
  while (sc < cfg.sparse_set_slots) sc <<= 1;
  cfg.sparse_set_slots = sc;
  int n_dev = 0;
  if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev <= cfg.device || cfg.device < 0) return KUQ_E_NO_DEVICE;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, cfg.device) != cudaSuccess) return KUQ_E_NO_DEVICE;
  if (prop.major < 10) return KUQ_E_NO_DEVICE;     // kernels are built for sm_100a only
  if (cudaSetDevice(cfg.device) != cudaSuccess) return KUQ_E_NO_DEVICE;
  kuq_ctx *ctx = new kuq_ctx();
  ctx->cfg = cfg;
  ctx->device = cfg.device;
  ctx->n_sm = prop.multiProcessorCount;
  if (cudaStreamCreateWithFlags(&ctx->aux, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return KUQ_E_CUDA; }
  ctx->slots.resize(cfg.n_slots);
  for (auto &s : ctx->slots) {
    int rc = alloc_slot(ctx, s);
    if (rc) {
      fprintf(stderr, "libkuq: %s\n", ctx->err.c_str());
      kuq_destroy(ctx);
      return rc == KUQ_E_CUDA ? KUQ_E_NOMEM : rc;
    }
  }
  *out = ctx;
  return KUQ_OK;
}

void kuq_destroy(kuq_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  for (auto &s : ctx->slots) free_slot(s);
  stream_close(ctx);
  free_db(ctx);
  free_tax_state(ctx);
  cudaFree(ctx->d_sync_err);
  if (ctx->aux) cudaStreamDestroy(ctx->aux);
  delete ctx;
}

void *kuq_host_alloc(uint64_t bytes) {
  void *p = nullptr;
  // portable: pinned for every CUDA context of the process, whichever thread / device it was allocated from (a buffer
  // that the copying context does not know as pinned silently takes the pageable path: 6 GB/s instead of 50)
  if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) { (void)cudaGetLastError(); return nullptr; }
  return p;
}
void kuq_host_free(void *p) { if (p) cudaFreeHost(p); }

// ---- database -------------------------------------------------------------------------------------------------
int kuq_stage_db(kuq_ctx *ctx, const void *kdb_image, uint64_t kdb_bytes, const void *idx_image, uint64_t idx_bytes,
                 uint64_t bin_lo, uint64_t bin_hi) {
  if (!ctx || !kdb_image || !idx_image) return KUQ_E_INVALID_ARG;
  CU(cudaSetDevice(ctx->device));
  const uint8_t *p = (const uint8_t *)kdb_image;
  if (kdb_bytes < 56 || memcmp(p, "JFLISTDN", 8) != 0)                     // krakendb.cpp:32,67-68
    return fail(ctx, KUQ_E_DB_FORMAT, "database in improper format");
  uint64_t key_bits, val_len, key_ct;
  memcpy(&key_bits, p + 8, 8);
  memcpy(&val_len, p + 16, 8);
  memcpy(&key_ct, p + 48, 8);
  if (val_len != 4) return fail(ctx, KUQ_E_DB_FORMAT, "can only handle 4 byte DB values");   // :73-74
  uint32_t k = (uint32_t)(key_bits / 2);
  uint64_t key_len = key_bits / 8 + !!(key_bits % 8);
  if (key_len != 8 || k > 31)
    return fail(ctx, KUQ_E_UNSUPPORTED_K, "k = %u (key_len %llu): only 8-byte keys (k = 29..31) are supported", k,
                (unsigned long long)key_len);
  uint64_t header = 72 + 2 * (4 + 8 * key_bits);                           // :177
  if (kdb_bytes < header + key_ct * 12) return fail(ctx, KUQ_E_DB_FORMAT, "database file truncated");
  const uint8_t *q = (const uint8_t *)idx_image;
  uint32_t idx_type;
  if (idx_bytes < 8) return fail(ctx, KUQ_E_DB_FORMAT, "illegal Kraken DB index format");
  if (memcmp(q, "KRAKIDX", 7) == 0) idx_type = 1;
  else if (memcmp(q, "KRAKIX2", 7) == 0) idx_type = 2;
  else return fail(ctx, KUQ_E_DB_FORMAT, "illegal Kraken DB index format");  // :541
  uint32_t nt = q[7];
  if (nt < 1 || nt > 15 || nt > k) return fail(ctx, KUQ_E_DB_FORMAT, "index minimizer length %u out of range", nt);
  uint64_t n_bins = 1ull << (2 * nt);
  if (idx_bytes < 8 + 8 * (n_bins + 1)) return fail(ctx, KUQ_E_DB_FORMAT, "index file truncated");
  const uint64_t *offsets = (const uint64_t *)(q + 8);
  if (bin_hi == 0 || bin_hi > n_bins) bin_hi = n_bins;
  if (bin_lo >= bin_hi) return fail(ctx, KUQ_E_INVALID_ARG, "empty minimizer range");
  uint64_t rec_lo = offsets[bin_lo], rec_hi = offsets[bin_hi];
  if (rec_hi < rec_lo || rec_hi > key_ct) return fail(ctx, KUQ_E_DB_FORMAT, "index offsets inconsistent with key count");
  // taxonomy numbering survives a re-stage (chunked mode) as long as the new range only holds numbered taxids
  { int hrc = harvest_seen(ctx, false); if (hrc) return hrc; }
  stream_close(ctx);
  free_db(ctx);
  ctx->k = k; ctx->nt = nt; ctx->idx_type = idx_type;
  ctx->bin_lo = bin_lo; ctx->bin_hi = bin_hi;
  ctx->rec_base = rec_lo;
  ctx->key_ct = rec_hi - rec_lo;
  ctx->db_owned = true;
  CU(cudaMalloc((void **)&ctx->d_pairs, ctx->key_ct * 12 + SLACK));
  CU(dmalloc(&ctx->d_offsets_owned, bin_hi - bin_lo + 1));
  ctx->d_offsets = ctx->d_offsets_owned;
  // bulk H2D.  The images are usually mmap'ed files: a plain cudaMemcpy from pageable memory goes through the driver's
  // single-threaded staging (~7 GB/s, page faults included).  Instead a few threads fault the pages in and copy 64 MB
  // pieces into two pinned bounce buffers while the previous piece travels (cudaMemcpyAsync on the aux stream).
  {
    const uint64_t CH = 64ull << 20;
    const int NT = 8;
    uint8_t *bounce[2] = {nullptr, nullptr};
    cudaEvent_t ev[2];
    bool ok = cudaHostAlloc((void **)&bounce[0], CH, cudaHostAllocPortable) == cudaSuccess &&
              cudaHostAlloc((void **)&bounce[1], CH, cudaHostAllocPortable) == cudaSuccess;
    if (!ok) (void)cudaGetLastError();
    for (int b = 0; b < 2; b++) CU(cudaEventCreateWithFlags(&ev[b], cudaEventDisableTiming));
    auto piece_copy = [&](uint8_t *d_dst, const uint8_t *h_src, uint64_t bytes) -> int {
      if (!ok) { CU(cudaMemcpy(d_dst, h_src, bytes, cudaMemcpyHostToDevice)); return KUQ_OK; }
      uint64_t i = 0;
      for (uint64_t off = 0; off < bytes; off += CH, i++) {
        const uint64_t n = std::min(CH, bytes - off);
        const int b = (int)(i & 1);
        CU(cudaEventSynchronize(ev[b]));                       // the bounce buffer's previous piece has left
        std::vector<std::thread> th;
        const uint64_t per = (n + NT - 1) / NT;
        for (int t = 0; t < NT; t++) {
          const uint64_t a = std::min(n, per * t), e = std::min(n, per * (t + 1));
          if (e > a) th.emplace_back([=] { memcpy(bounce[b] + a, h_src + off + a, e - a); });
        }
        for (auto &x : th) x.join();
        CU(cudaMemcpyAsync(d_dst + off, bounce[b], n, cudaMemcpyHostToDevice, ctx->aux));
        CU(cudaEventRecord(ev[b], ctx->aux));
      }
      CU(cudaStreamSynchronize(ctx->aux));
      return KUQ_OK;
    };
    const uint8_t *src = p + header + rec_lo * 12;
    int crc = piece_copy(ctx->d_pairs, src, ctx->key_ct * 12);
    if (!crc) crc = piece_copy(reinterpret_cast<uint8_t *>(ctx->d_offsets_owned), reinterpret_cast<const uint8_t *>(offsets + bin_lo),
                               (bin_hi - bin_lo + 1) * 8);
    for (int b = 0; b < 2; b++) { cudaEventDestroy(ev[b]); if (bounce[b]) cudaFreeHost(bounce[b]); }
    if (crc) return crc;
  }
  ctx->db_staged = true;
  int rc = collect_taxids(ctx);
  if (rc) return rc;
  if (ctx->finalized) return remap_db(ctx);
  return KUQ_OK;
}

int kuq_attach_db_device(kuq_ctx *ctx, void *d_pairs, uint64_t key_ct, const uint64_t *d_offsets, uint32_t k,
                         uint32_t nt, uint32_t idx_type, uint64_t bin_lo, uint64_t bin_hi) {
  if (!ctx || !d_pairs || !d_offsets) return KUQ_E_INVALID_ARG;
  if (k < 29 || k > 31) return fail(ctx, KUQ_E_UNSUPPORTED_K, "k = %u: only 8-byte keys (k = 29..31)", k);
  if (nt < 1 || nt > 15 || (idx_type != 1 && idx_type != 2)) return fail(ctx, KUQ_E_INVALID_ARG, "bad index parameters");
  CU(cudaSetDevice(ctx->device));
  uint64_t n_bins = 1ull << (2 * nt);
  if (bin_hi == 0 || bin_hi > n_bins) bin_hi = n_bins;
  if (bin_lo >= bin_hi) return fail(ctx, KUQ_E_INVALID_ARG, "empty minimizer range");
  { int hrc = harvest_seen(ctx, false); if (hrc) return hrc; }
  free_db(ctx);
  ctx->k = k; ctx->nt = nt; ctx->idx_type = idx_type;
  ctx->bin_lo = bin_lo; ctx->bin_hi = bin_hi;
  ctx->db_owned = false;
  ctx->d_pairs = (uint8_t *)d_pairs;
  ctx->d_offsets = d_offsets;
  uint64_t first = 0;
  CU(cudaMemcpy(&first, d_offsets, 8, cudaMemcpyDeviceToHost));
  ctx->rec_base = first;
  ctx->key_ct = key_ct;
  ctx->db_staged = true;
  int rc = collect_taxids(ctx);
  if (rc) return rc;
  if (ctx->finalized) return remap_db(ctx);
  return KUQ_OK;
}

int kuq_db_taxids(kuq_ctx *ctx, uint32_t *taxid, uint64_t *count, uint32_t cap, uint32_t *n) {
  if (!ctx || !n) return KUQ_E_INVALID_ARG;
  if (!ctx->db_staged) return fail(ctx, KUQ_E_STATE, "no database staged");
  *n = (uint32_t)ctx->db_taxids.size();
  if (cap == 0) return KUQ_OK;
  if (cap < *n) return fail(ctx, KUQ_E_CAPACITY, "need room for %u taxids", *n);
  for (uint32_t i = 0; i < *n; i++) {
    if (taxid) taxid[i] = ctx->db_taxids[i];
    if (count) count[i] = ctx->db_taxid_counts[i];
  }
  return KUQ_OK;
}

int kuq_set_db_taxid_universe(kuq_ctx *ctx, const uint32_t *taxid, uint32_t n) {
  if (!ctx || (!taxid && n)) return KUQ_E_INVALID_ARG;
  if (ctx->finalized) return fail(ctx, KUQ_E_STATE, "taxid universe must be declared before the first classification");
  ctx->universe.assign(taxid, taxid + n);
  return KUQ_OK;
}

int kuq_set_quick_mode(kuq_ctx *ctx, uint32_t min_hits, int stop_at_last_hit) {
  if (!ctx) return KUQ_E_INVALID_ARG;
  for (auto &s : ctx->slots)
    if (s.busy) return fail(ctx, KUQ_E_STATE, "quick mode cannot change while a batch is in flight");
  if (min_hits && ctx->cfg.hll_mode == KUQ_HLL_EXACT) return fail(ctx, KUQ_E_INVALID_ARG, "quick mode is not available with KUQ_HLL_EXACT");
  ctx->quick_min = min_hits;
  ctx->quick_stop = min_hits && stop_at_last_hit;
  return KUQ_OK;
}

int kuq_mark_zero_hits(kuq_ctx *ctx, int on) {
  if (!ctx) return KUQ_E_INVALID_ARG;
  ctx->mark_zero_hits = on != 0;
  return KUQ_OK;
}

int kuq_set_taxonomy(kuq_ctx *ctx, const uint32_t *taxid, const uint32_t *parent, uint32_t n) {
  if (!ctx || ((!taxid || !parent) && n)) return KUQ_E_INVALID_ARG;
  if (ctx->finalized) return fail(ctx, KUQ_E_STATE, "taxonomy already in use; create a new context to change it");
  // later rows overwrite earlier ones, like Parent_map[taxid] = parent
  std::unordered_map<uint32_t, uint32_t> m;
  for (uint32_t i = 0; i < n; i++) m[taxid[i]] = parent[i];
  ctx->tax_ids.clear(); ctx->tax_parents.clear();
  for (auto &kv : m) { ctx->tax_ids.push_back(kv.first); ctx->tax_parents.push_back(kv.second); }
  ctx->tax_set = true;
  return KUQ_OK;
}

// ---- classification -------------------------------------------------------------------------------------------
namespace {
// What every batch call checks before it touches slot `slot`; then the slot records the batch.  A slot with an unread
// batch refuses every call until kuq_wait_batch: a new launch would overwrite the results it has not copied yet.
// Device inputs must also be non-NULL and 16-byte aligned (TMA bulk loads); the callers check host inputs.
int begin_batch(kuq_ctx *ctx, uint32_t slot, uint32_t n_reads, uint64_t total_bases, uint32_t flags, bool device_inputs,
                const char *d_bases = nullptr, const uint64_t *d_offsets = nullptr) {
  int rc = check_slot(ctx, slot);
  if (rc) return rc;
  if (device_inputs) {
    if (n_reads && (!d_bases || !d_offsets)) return fail(ctx, KUQ_E_INVALID_ARG, "NULL device buffers");
    if ((uintptr_t)d_bases & 15) return fail(ctx, KUQ_E_INVALID_ARG, "d_bases must be 16-byte aligned");
  }
  CU(cudaSetDevice(ctx->device));
  Slot &s = ctx->slots[slot];
  if (s.busy) return fail(ctx, KUQ_E_STATE, "slot %u still has an unread batch: call kuq_wait_batch first", slot);
  if (n_reads > ctx->cfg.max_reads_per_batch) return fail(ctx, KUQ_E_CAPACITY, "%u reads > slot capacity %u", n_reads, ctx->cfg.max_reads_per_batch);
  if (total_bases > ctx->cfg.max_bases_per_batch) return fail(ctx, KUQ_E_CAPACITY, "%llu bases > slot capacity %llu", (unsigned long long)total_bases, (unsigned long long)ctx->cfg.max_bases_per_batch);
  if (total_bases >= (1ull << 32)) return fail(ctx, KUQ_E_CAPACITY, "batches are limited to 4 Gbases");
  s.n_reads = n_reads; s.flags = flags; s.total_bases = total_bases;
  return KUQ_OK;
}

uint64_t host_bases(const uint64_t *read_offsets, uint32_t n_reads) { return n_reads ? read_offsets[n_reads] - read_offsets[0] : 0; }

// copy the batch begin_batch recorded (reads on the host) into the slot's device buffers
int upload_reads(kuq_ctx *ctx, Slot &s, const char *bases, const uint64_t *read_offsets) {
  const uint32_t n_reads = s.n_reads;
  if (!n_reads) return KUQ_OK;
  const uint64_t base0 = read_offsets[0], total = s.total_bases;
  CU(cudaMemcpyAsync(s.d_bases, bases + base0, total, cudaMemcpyHostToDevice, s.stream));
  CU(cudaMemsetAsync(s.d_bases + total, 'N', SLACK, s.stream));
  if (base0 == 0) {
    CU(cudaMemcpyAsync(s.d_offsets, read_offsets, (n_reads + 1ull) * 8, cudaMemcpyHostToDevice, s.stream));
  } else {
    std::vector<uint64_t> tmp(n_reads + 1);
    for (uint32_t i = 0; i <= n_reads; i++) tmp[i] = read_offsets[i] - base0;
    CU(cudaMemcpy(s.d_offsets, tmp.data(), (n_reads + 1ull) * 8, cudaMemcpyHostToDevice));
  }
  return KUQ_OK;
}

// Work-unit id of every read for the KUQ_HLL_PRELOAD rule, on the device: the caller's, or cut like process_file does.
// *d_unit stays nullptr when the rule needs none.
int upload_units(kuq_ctx *ctx, Slot &s, const uint64_t *read_offsets, const uint32_t *unit_id, const uint32_t **d_unit) {
  *d_unit = nullptr;
  if (ctx->cfg.hll_mode != KUQ_HLL_PRELOAD || !s.n_reads) return KUQ_OK;
  if (unit_id) memcpy(s.h_unit, unit_id, s.n_reads * 4ull);
  else cut_units(ctx, read_offsets, s.n_reads, s.h_unit);
  CU(cudaMemcpyAsync(s.d_unit, s.h_unit, s.n_reads * 4ull, cudaMemcpyHostToDevice, s.stream));
  *d_unit = s.d_unit;
  return KUQ_OK;
}

// Host inputs: begin_batch, a staged database, the reads (and for the counting modes the work-unit ids) copied into the
// slot, and `p` filled over those copies; the caller adds the fields of `mode` and launches.
int host_call(kuq_ctx *ctx, uint32_t slot, int mode, const char *bases, const uint64_t *read_offsets, uint32_t n_reads,
              const uint32_t *unit_id, uint32_t flags, Params &p) {
  int rc = begin_batch(ctx, slot, n_reads, host_bases(read_offsets, n_reads), flags, false);
  if (!rc) rc = ensure_ready(ctx);
  if (rc) return rc;
  Slot &s = ctx->slots[slot];
  const uint32_t *d_unit = nullptr;
  rc = upload_reads(ctx, s, bases, read_offsets);
  if (!rc && mode != MODE_LOOKUP) rc = upload_units(ctx, s, read_offsets, unit_id, &d_unit);
  if (rc) return rc;
  fill_params(ctx, s, p, s.d_bases, s.d_offsets, d_unit, n_reads, flags);
  return KUQ_OK;
}

// Device inputs: begin_batch, a staged database, and `p` filled over the caller's buffers; the caller adds the fields of
// `mode` and launches.
int device_call(kuq_ctx *ctx, uint32_t slot, int mode, const char *d_bases, const uint64_t *d_offsets, uint32_t n_reads,
                uint64_t total_bases, const uint32_t *d_unit, uint32_t flags, Params &p) {
  int rc = begin_batch(ctx, slot, n_reads, total_bases, flags, true, d_bases, d_offsets);
  if (!rc) rc = ensure_ready(ctx);
  if (rc) return rc;
  if (mode != MODE_LOOKUP && ctx->cfg.hll_mode == KUQ_HLL_PRELOAD && !d_unit && !(flags & KUQ_F_NO_COUNTS) && n_reads)
    return fail(ctx, KUQ_E_INVALID_ARG, "KUQ_HLL_PRELOAD needs the work-unit id of every read (d_unit_id) to "
                "reproduce the per-unit sketches; pass it, or create the context with KUQ_HLL_CHUNKED / KUQ_HLL_DENSE_ONLY");
  fill_params(ctx, ctx->slots[slot], p, d_bases, d_offsets, d_unit, n_reads, flags);
  return KUQ_OK;
}

// D2H of the batch's fixed-size results into the slot's pinned buffers; the variable-size hit lists follow in
// kuq_wait_batch, which the slot now waits for
int copy_results(kuq_ctx *ctx, Slot &s) {
  if (s.n_reads) {
    CU(cudaMemcpyAsync(s.h_call, s.d_call, s.n_reads * 4ull, cudaMemcpyDeviceToHost, s.stream));
    CU(cudaMemcpyAsync(s.h_nwin, s.d_nwin, s.n_reads * 4ull, cudaMemcpyDeviceToHost, s.stream));
    if (!(s.flags & KUQ_F_NO_RUNS) || ctx->quick_min) {
      CU(cudaMemcpyAsync(s.h_run_start, s.d_run_start, s.n_reads * 4ull, cudaMemcpyDeviceToHost, s.stream));
      CU(cudaMemcpyAsync(s.h_run_count, s.d_run_count, s.n_reads * 4ull, cudaMemcpyDeviceToHost, s.stream));
    }
  }
  CU(cudaMemcpyAsync(s.h_scalars, s.d_scalars, 8 * 8, cudaMemcpyDeviceToHost, s.stream));
  s.busy = true;
  return KUQ_OK;
}

// the error word the kernels of the slot's last batch left (Params::error_flag) as a libkuq error code
int batch_error(kuq_ctx *ctx, const Slot &s, uint32_t err) {
  if (err == 1) return fail(ctx, KUQ_E_TAXA_OVERFLOW, "the batch exhausted the hit-table pool for reads with more than 32 distinct taxa: use smaller batches");
  if (err == 4) return fail(ctx, KUQ_E_CAPACITY, "sparse-tier set saturated: raise kuq_config.sparse_set_slots (now %llu)", (unsigned long long)ctx->sparse_cap);
  if (err == 5) return fail(ctx, KUQ_E_CAPACITY, "the hit lists of the batch need more run slots than the slot holds (%llu): use smaller batches", (unsigned long long)s.runs_cap);
  if (err) return fail(ctx, KUQ_E_CAPACITY, "per-batch work-unit bookkeeping overflowed (code %u): use smaller batches", err);
  return KUQ_OK;
}
}  // namespace

int kuq_lookup_batch(kuq_ctx *ctx, const char *bases, const uint64_t *read_offsets, uint32_t n_reads,
                     uint32_t *codes_out, uint32_t *n_windows_out) {
  if (n_reads && (!bases || !read_offsets || !codes_out)) return fail(ctx, KUQ_E_INVALID_ARG, "NULL batch buffers");
  Params p;
  int rc = host_call(ctx, 0, MODE_LOOKUP, bases, read_offsets, n_reads, nullptr, 0, p);
  if (rc) return rc;
  Slot &s = ctx->slots[0];
  // positions without a window are not written by the kernels: give the caller zeros there
  CU(cudaMemsetAsync(s.d_dense, 0, s.total_bases * 4, s.stream));
  rc = launch_on_slot(ctx, s, MODE_LOOKUP, p);
  if (rc) return rc;
  if (n_reads) {
    CU(cudaMemcpyAsync(codes_out, s.d_dense, s.total_bases * 4, cudaMemcpyDeviceToHost, s.stream));
    if (n_windows_out) CU(cudaMemcpyAsync(n_windows_out, s.d_nwin, n_reads * 4ull, cudaMemcpyDeviceToHost, s.stream));
  }
  CU(cudaStreamSynchronize(s.stream));
  return KUQ_OK;
}

int kuq_resolve_batch(kuq_ctx *ctx, const char *bases, const uint64_t *read_offsets, uint32_t n_reads,
                      const uint32_t *codes_in, const uint32_t *unit_id, uint32_t flags, kuq_batch_result *out) {
  if (!out || (n_reads && (!bases || !read_offsets || !codes_in))) return fail(ctx, KUQ_E_INVALID_ARG, "NULL batch buffers");
  Params p;
  int rc = host_call(ctx, 0, MODE_RESOLVE, bases, read_offsets, n_reads, unit_id, flags, p);
  if (rc) return rc;
  Slot &s = ctx->slots[0];
  if (!s.d_codes_in) CU(dmalloc(&s.d_codes_in, ctx->cfg.max_bases_per_batch + SLACK));
  if (n_reads) CU(cudaMemcpyAsync(s.d_codes_in, codes_in, s.total_bases * 4, cudaMemcpyHostToDevice, s.stream));
  p.codes_in = s.d_codes_in;
  rc = launch_on_slot(ctx, s, MODE_RESOLVE, p);
  return rc ? rc : kuq_collect_device_batch(ctx, 0, out);
}

int kuq_submit_batch(kuq_ctx *ctx, uint32_t slot, const char *bases, const uint64_t *read_offsets, uint32_t n_reads,
                     const uint32_t *unit_id, uint32_t flags) {
  if (n_reads && (!bases || !read_offsets)) return fail(ctx, KUQ_E_INVALID_ARG, "NULL batch buffers");
  Params p;
  int rc = host_call(ctx, slot, MODE_FUSED, bases, read_offsets, n_reads, unit_id, flags, p);
  if (!rc) rc = launch_on_slot(ctx, ctx->slots[slot], MODE_FUSED, p);
  return rc ? rc : copy_results(ctx, ctx->slots[slot]);
}

int kuq_wait_batch(kuq_ctx *ctx, uint32_t slot, kuq_batch_result *out) {
  int rc = check_slot(ctx, slot);
  if (rc) return rc;
  if (!out) return KUQ_E_INVALID_ARG;
  CU(cudaSetDevice(ctx->device));
  Slot &s = ctx->slots[slot];
  if (!s.busy) return fail(ctx, KUQ_E_STATE, "slot %u has no batch in flight", slot);
  CU(cudaStreamSynchronize(s.stream));
  s.busy = false;
  float ms = 0;
  if (s.timed) cudaEventElapsedTime(&ms, s.ev_k0, s.ev_k1);
  (void)cudaGetLastError();
  s.kernel_ms = ms;
  rc = batch_error(ctx, s, (uint32_t)(s.h_scalars[3] & 0xFFFFFFFFu));
  if (rc) return rc;
  const uint64_t n_runs = (s.flags & KUQ_F_NO_RUNS) ? 0 : s.h_scalars[0];
  if (n_runs) {
    if (n_runs > s.h_runs_cap) {
      cudaFreeHost(s.h_runs);
      s.h_runs = nullptr;
      s.h_runs_cap = n_runs + n_runs / 2;
      CU(hmalloc(&s.h_runs, s.h_runs_cap));
    }
    CU(cudaMemcpyAsync(s.h_runs, s.d_runs, n_runs * 8, cudaMemcpyDeviceToHost, s.stream));
  }
  if ((s.flags & KUQ_F_WANT_CODES) && s.total_bases) {
    if (!s.h_codes) CU(hmalloc(&s.h_codes, ctx->cfg.max_bases_per_batch));
    CU(cudaMemcpyAsync(s.h_codes, s.d_codes, s.total_bases * 4, cudaMemcpyDeviceToHost, s.stream));
  }
  CU(cudaStreamSynchronize(s.stream));
  memset(out, 0, sizeof *out);
  out->n_reads = s.n_reads;
  out->call = s.h_call;
  out->n_windows = s.h_nwin;
  out->run_start = s.h_run_start;
  out->run_count = s.h_run_count;
  out->runs = s.h_runs;
  out->n_runs = n_runs;
  out->codes = (s.flags & KUQ_F_WANT_CODES) ? s.h_codes : nullptr;
  out->n_classified = s.h_scalars[1];
  out->kernel_ms = s.kernel_ms;
  return KUQ_OK;
}

int kuq_classify_batch(kuq_ctx *ctx, const char *bases, const uint64_t *read_offsets, uint32_t n_reads,
                       const uint32_t *unit_id, uint32_t flags, kuq_batch_result *out) {
  int rc = kuq_submit_batch(ctx, 0, bases, read_offsets, n_reads, unit_id, flags);
  if (rc) return rc;
  return kuq_wait_batch(ctx, 0, out);
}

int kuq_classify_device(kuq_ctx *ctx, uint32_t slot, const char *d_bases, const uint64_t *d_read_offsets,
                        uint32_t n_reads, uint64_t total_bases, const uint32_t *d_unit_id, uint32_t flags) {
  Params p;
  int rc = device_call(ctx, slot, MODE_FUSED, d_bases, d_read_offsets, n_reads, total_bases, d_unit_id, flags, p);
  return rc ? rc : launch_on_slot(ctx, ctx->slots[slot], MODE_FUSED, p);
}
int kuq_lookup_device(kuq_ctx *ctx, uint32_t slot, const char *d_bases, const uint64_t *d_read_offsets,
                      uint32_t n_reads, uint64_t total_bases, uint32_t *d_codes_out, uint32_t only_hits) {
  if (!d_codes_out) return KUQ_E_INVALID_ARG;
  Params p;
  int rc = device_call(ctx, slot, MODE_LOOKUP, d_bases, d_read_offsets, n_reads, total_bases, nullptr, 0, p);
  if (rc) return rc;
  p.codes_dense = d_codes_out;
  p.only_hits = only_hits;
  return launch_on_slot(ctx, ctx->slots[slot], MODE_LOOKUP, p);
}
int kuq_resolve_device(kuq_ctx *ctx, uint32_t slot, const char *d_bases, const uint64_t *d_read_offsets,
                       uint32_t n_reads, uint64_t total_bases, const uint32_t *d_codes_in, const uint32_t *d_unit_id,
                       uint32_t flags) {
  if (!d_codes_in) return KUQ_E_INVALID_ARG;
  Params p;
  int rc = device_call(ctx, slot, MODE_RESOLVE, d_bases, d_read_offsets, n_reads, total_bases, d_unit_id, flags, p);
  if (rc) return rc;
  p.codes_in = d_codes_in;
  return launch_on_slot(ctx, ctx->slots[slot], MODE_RESOLVE, p);
}

int kuq_lookup_device_peers(kuq_ctx *ctx, uint32_t slot, const char *d_bases, const uint64_t *d_read_offsets,
                            uint32_t n_reads, uint64_t total_bases, uint32_t *const *d_codes_peers,
                            const uint64_t *base_bounds, uint32_t n_peers) {
  if (!d_codes_peers || !base_bounds || n_peers == 0 || n_peers > 8) return KUQ_E_INVALID_ARG;
  Params p;
  int rc = device_call(ctx, slot, MODE_LOOKUP, d_bases, d_read_offsets, n_reads, total_bases, nullptr, 0, p);
  if (rc) return rc;
  p.only_hits = 1;
  p.n_peers = n_peers;
  for (uint32_t j = 0; j < n_peers; j++) { p.peer_codes[j] = d_codes_peers[j]; p.peer_bounds[j] = base_bounds[j]; }
  p.peer_bounds[n_peers] = base_bounds[n_peers];
  return launch_on_slot(ctx, ctx->slots[slot], MODE_LOOKUP, p);
}

// ---- device memory that can be shared with the other ranks of a node (CUDA IPC) --------------------------------
void *kuq_device_alloc(kuq_ctx *ctx, uint64_t bytes) {
  if (!ctx) return nullptr;
  if (cudaSetDevice(ctx->device) != cudaSuccess) return nullptr;
  void *p = nullptr;
  if (cudaMalloc(&p, bytes ? bytes : 1) != cudaSuccess) return nullptr;
  return p;
}
void kuq_device_free(kuq_ctx *ctx, void *p) {
  if (ctx) cudaSetDevice(ctx->device);
  if (p) cudaFree(p);
}
int kuq_device_memset(kuq_ctx *ctx, uint32_t slot, void *p, int value, uint64_t bytes) {
  int rc = check_slot(ctx, slot);
  if (rc) return rc;
  CU(cudaSetDevice(ctx->device));
  CU(cudaMemsetAsync(p, value, bytes, ctx->slots[slot].stream));
  return KUQ_OK;
}
int kuq_ipc_export(kuq_ctx *ctx, void *d_ptr, uint8_t handle64[64]) {
  if (!ctx || !d_ptr || !handle64) return KUQ_E_INVALID_ARG;
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  CU(cudaSetDevice(ctx->device));
  cudaIpcMemHandle_t h;
  CU(cudaIpcGetMemHandle(&h, d_ptr));
  memcpy(handle64, &h, 64);
  return KUQ_OK;
}
int kuq_ipc_open(kuq_ctx *ctx, const uint8_t handle64[64], void **d_ptr_out) {
  if (!ctx || !handle64 || !d_ptr_out) return KUQ_E_INVALID_ARG;
  CU(cudaSetDevice(ctx->device));
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  CU(cudaIpcOpenMemHandle(d_ptr_out, h, cudaIpcMemLazyEnablePeerAccess));
  return KUQ_OK;
}
int kuq_ipc_close(kuq_ctx *ctx, void *d_ptr) {
  if (!ctx || !d_ptr) return KUQ_E_INVALID_ARG;
  CU(cudaSetDevice(ctx->device));
  CU(cudaIpcCloseMemHandle(d_ptr));
  return KUQ_OK;
}

int kuq_copy_to_device(kuq_ctx *ctx, uint32_t slot, void *d_dst, const void *h_src, uint64_t bytes) {
  int rc = check_slot(ctx, slot);
  if (rc) return rc;
  if (!bytes) return KUQ_OK;
  if (!d_dst || !h_src) return KUQ_E_INVALID_ARG;
  CU(cudaSetDevice(ctx->device));
  CU(cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, ctx->slots[slot].stream));
  return KUQ_OK;
}

uint64_t kuq_device_free_bytes(kuq_ctx *ctx) {
  if (!ctx || cudaSetDevice(ctx->device) != cudaSuccess) return 0;
  size_t fr = 0, tot = 0;
  if (cudaMemGetInfo(&fr, &tot) != cudaSuccess) { (void)cudaGetLastError(); return 0; }
  return fr;
}

// after kuq_classify_device / kuq_resolve_device on `slot`: bring the batch's results to the slot's pinned host
// buffers and wait — the device-input counterpart of kuq_classify_batch's second half
int kuq_collect_device_batch(kuq_ctx *ctx, uint32_t slot, kuq_batch_result *out) {
  int rc = check_slot(ctx, slot);
  if (rc) return rc;
  if (!out) return KUQ_E_INVALID_ARG;
  CU(cudaSetDevice(ctx->device));
  Slot &s = ctx->slots[slot];
  if (s.busy) return fail(ctx, KUQ_E_STATE, "slot %u still has an unread batch", slot);
  rc = copy_results(ctx, s);
  return rc ? rc : kuq_wait_batch(ctx, slot, out);
}

int kuq_sync_slot(kuq_ctx *ctx, uint32_t slot) {
  int rc = check_slot(ctx, slot);
  if (rc) return rc;
  Slot &s = ctx->slots[slot];
  CU(cudaStreamSynchronize(s.stream));
  float ms = 0;
  if (s.timed && cudaEventElapsedTime(&ms, s.ev_k0, s.ev_k1) == cudaSuccess) s.kernel_ms = ms;
  (void)cudaGetLastError();      // never leave a stale error code behind for the next CUDA user of this process
  uint32_t err = 0;
  if (ctx->d_sync_err) {
    CU(cudaMemcpy(&err, ctx->d_sync_err, 4, cudaMemcpyDeviceToHost));
    if (err) return fail(ctx, KUQ_E_STATE, "kuq_wait_flags timed out: a peer GPU never signalled (code %u)", err);
  }
  CU(cudaMemcpy(&err, reinterpret_cast<uint32_t *>(s.d_scalars + 3), 4, cudaMemcpyDeviceToHost));
  return batch_error(ctx, s, err);
}

int kuq_slot_device_result(kuq_ctx *ctx, uint32_t slot, kuq_device_result *out) {
  int rc = check_slot(ctx, slot);
  if (rc) return rc;
  if (!out) return KUQ_E_INVALID_ARG;
  Slot &s = ctx->slots[slot];
  out->d_call = s.d_call;
  out->d_n_windows = s.d_nwin;
  out->d_codes = s.d_codes;
  out->d_run_start = s.d_run_start;
  out->d_run_count = s.d_run_count;
  out->d_runs = reinterpret_cast<const kuq_run *>(s.d_runs);
  out->d_n_runs = reinterpret_cast<const uint64_t *>(s.d_scalars);
  return KUQ_OK;
}

int kuq_slot_stats(kuq_ctx *ctx, uint32_t slot, uint64_t *n_lookups, uint64_t *sum_probes) {
  int rc = check_slot(ctx, slot);
  if (rc) return rc;
  Slot &s = ctx->slots[slot];
  CU(cudaStreamSynchronize(s.stream));
  unsigned long long v[2];
  CU(cudaMemcpy(v, s.d_scalars + 4, 16, cudaMemcpyDeviceToHost));
  if (n_lookups) *n_lookups = v[0];
  if (sum_probes) *sum_probes = v[1];
  return KUQ_OK;
}

void *kuq_slot_stream(kuq_ctx *ctx, uint32_t slot) {
  if (!ctx || slot >= ctx->slots.size()) return nullptr;
  return (void *)ctx->slots[slot].stream;
}
uint64_t kuq_launch_count(const kuq_ctx *ctx) { return ctx ? ctx->launches : 0; }
double kuq_last_kernel_ms(kuq_ctx *ctx, uint32_t slot) {
  if (!ctx || slot >= ctx->slots.size()) return -1;
  return ctx->slots[slot].kernel_ms;
}
int kuq_last_stage_ms(kuq_ctx *ctx, uint32_t slot, double *ms3) {
  int rc = check_slot(ctx, slot);
  if (rc) return rc;
  if (!ms3) return KUQ_E_INVALID_ARG;
  Slot &s = ctx->slots[slot];
  CU(cudaStreamSynchronize(s.stream));
  float a = 0, b = 0, c = 0;
  if (s.timed) {
    cudaEventElapsedTime(&a, s.ev_k0, s.ev_stage[0]);
    cudaEventElapsedTime(&b, s.ev_stage[0], s.ev_stage[1]);
    cudaEventElapsedTime(&c, s.ev_stage[1], s.ev_k1);
  }
  (void)cudaGetLastError();
  ms3[0] = a; ms3[1] = b; ms3[2] = c;
  return KUQ_OK;
}

// ---- per-taxon results ------------------------------------------------------------------------------------------
int kuq_finish(kuq_ctx *ctx) {
  if (!ctx) return KUQ_E_INVALID_ARG;
  CU(cudaSetDevice(ctx->device));
  for (auto &s : ctx->slots) CU(cudaStreamSynchronize(s.stream));
  ctx->unit_nt = 0;
  ctx->unit_next++;
  return harvest_seen(ctx, false);
}

namespace {
int fetch_counts(kuq_ctx *ctx, CountsHost &h) {
  if (!ctx->finalized) return fail(ctx, KUQ_E_STATE, "nothing classified yet");
  CU(cudaSetDevice(ctx->device));
  for (auto &s : ctx->slots) CU(cudaStreamSynchronize(s.stream));
  { int hrc = harvest_seen(ctx, false); if (hrc) return hrc; }
  ctx->snap_valid = false;
  h.n_kmers.resize(ctx->n_sketch);
  h.n_reads.resize(ctx->n_taxa);
  h.hist.resize((size_t)ctx->n_sketch * 64);
  h.dense_flag.assign(ctx->n_sketch, 1);
  h.distinct.assign(ctx->n_sketch, 0);
  CU(cudaMemcpy(h.n_kmers.data(), ctx->d_n_kmers, ctx->n_sketch * 8ull, cudaMemcpyDeviceToHost));
  CU(cudaMemcpy(h.n_reads.data(), ctx->d_n_reads, ctx->n_taxa * 8ull, cudaMemcpyDeviceToHost));
  uint32_t *d_hist;
  CU(dmalloc(&d_hist, (uint64_t)ctx->n_sketch * 64));
  launch_register_histograms(ctx->d_regs, ctx->n_sketch, d_hist, ctx->aux);
  ctx->launches++;
  CU(cudaMemcpyAsync(h.hist.data(), d_hist, (uint64_t)ctx->n_sketch * 64 * 4, cudaMemcpyDeviceToHost, ctx->aux));
  CU(cudaStreamSynchronize(ctx->aux));
  cudaFree(d_hist);
  if (ctx->cfg.hll_mode == KUQ_HLL_EXACT) {
    h.exact.resize(ctx->n_sketch);
    CU(cudaMemcpy(h.exact.data(), ctx->d_exact_count, ctx->n_sketch * 8ull, cudaMemcpyDeviceToHost));
  } else if (ctx->cfg.hll_mode != KUQ_HLL_DENSE_ONLY) {
    if (ctx->cfg.hll_mode == KUQ_HLL_CHUNKED) {
      launch_flag_dense_global(ctx->d_sparse_distinct, ctx->d_dense_flag, ctx->n_sketch, ctx->aux);
      ctx->launches++;
    }
    uint32_t *d_sh;
    CU(dmalloc(&d_sh, (uint64_t)ctx->n_sketch * 64));
    CU(cudaMemsetAsync(d_sh, 0, (uint64_t)ctx->n_sketch * 64 * 4, ctx->aux));
    launch_sparse_histograms(ctx->d_sparse_slots, ctx->sparse_cap, ctx->d_dense_flag, d_sh, ctx->aux);
    ctx->launches++;
    h.sparse_hist.resize((size_t)ctx->n_sketch * 64);
    CU(cudaMemcpyAsync(h.sparse_hist.data(), d_sh, (uint64_t)ctx->n_sketch * 64 * 4, cudaMemcpyDeviceToHost, ctx->aux));
    CU(cudaMemcpyAsync(h.dense_flag.data(), ctx->d_dense_flag, ctx->n_sketch, cudaMemcpyDeviceToHost, ctx->aux));
    CU(cudaMemcpyAsync(h.distinct.data(), ctx->d_sparse_distinct, ctx->n_sketch * 4ull, cudaMemcpyDeviceToHost, ctx->aux));
    CU(cudaStreamSynchronize(ctx->aux));
    cudaFree(d_sh);
    if (ctx->merged_summary) {             // sums over the code partitions of all GPUs (kuq_set_sparse_summary)
      h.sparse_hist = ctx->merged_hist;
      h.distinct = ctx->merged_distinct;
    }
  }
  if (&h == &ctx->snap) ctx->snap_valid = true;
  return KUQ_OK;
}
}  // namespace

namespace {
// Histogram of the merged sketch of the member taxa (dense ids with k-mers): register-value histogram of the
// register-wise max when any member is dense, else rank histogram of the union of the members' sparse code sets.
// With a cross-GPU summary installed (kuq_set_sparse_summary) the local set is one code partition: the union
// histogram of several sparse members is then a PARTIAL result the caller sums over GPUs (allow_partial).
int clade_hist(kuq_ctx *ctx, const std::vector<uint32_t> &members, uint32_t *hist64, int *is_dense, bool allow_partial) {
  const CountsHost &h = ctx->snap;
  memset(hist64, 0, 64 * sizeof(uint32_t));
  bool any_dense = ctx->cfg.hll_mode == KUQ_HLL_DENSE_ONLY;
  uint64_t sum_distinct = 0;
  for (uint32_t d : members) { any_dense |= h.dense_flag[d] != 0; sum_distinct += h.distinct[d]; }
  *is_dense = any_dense ? 1 : 0;
  if (members.empty()) return KUQ_OK;
  if (members.size() == 1 && !(allow_partial && ctx->merged_summary && !any_dense)) {
    // a clade with a single contributing taxon has that taxon's sketch
    const uint32_t d = members[0];
    memcpy(hist64, any_dense ? &h.hist[(size_t)d * 64] : &h.sparse_hist[(size_t)d * 64], 64 * sizeof(uint32_t));
    return KUQ_OK;
  }
  if (!any_dense) {
    if (ctx->merged_summary && !allow_partial)
      return fail(ctx, KUQ_E_STATE, "the sparse tier is partitioned over GPUs: sum kuq_clade_partial over the GPUs instead");
    std::vector<uint8_t> member(ctx->n_sketch, 0);
    for (uint32_t d : members) member[d] = 1;
    uint64_t cap = 1024;
    while (cap < 2 * sum_distinct + 16) cap <<= 1;
    uint8_t *d_member; unsigned long long *d_set; uint32_t *d_hist;
    CU(dmalloc(&d_member, ctx->n_sketch));
    CU(dmalloc(&d_set, cap));
    CU(dmalloc(&d_hist, 65));
    CU(cudaMemcpyAsync(d_member, member.data(), ctx->n_sketch, cudaMemcpyHostToDevice, ctx->aux));
    CU(cudaMemsetAsync(d_set, 0, cap * 8, ctx->aux));
    CU(cudaMemsetAsync(d_hist, 0, 65 * 4, ctx->aux));
    launch_sparse_union(ctx->d_sparse_slots, ctx->sparse_cap, d_member, d_set, cap - 1, d_hist, d_hist + 64, ctx->aux);
    ctx->launches++;
    uint32_t hist[65];
    CU(cudaMemcpyAsync(hist, d_hist, sizeof hist, cudaMemcpyDeviceToHost, ctx->aux));
    CU(cudaStreamSynchronize(ctx->aux));
    cudaFree(d_member); cudaFree(d_set); cudaFree(d_hist);
    if (hist[64]) return fail(ctx, KUQ_E_CAPACITY, "internal: clade union scratch overflow");
    memcpy(hist64, hist, 64 * sizeof(uint32_t));
    return KUQ_OK;
  }
  uint32_t *d_members; uint8_t *d_out; uint32_t *d_hist;
  CU(dmalloc(&d_members, members.size()));
  CU(dmalloc(&d_out, HLL_M));
  CU(dmalloc(&d_hist, 64));
  CU(cudaMemcpyAsync(d_members, members.data(), members.size() * 4, cudaMemcpyHostToDevice, ctx->aux));
  launch_clade_max(ctx->d_regs, d_members, (uint32_t)members.size(), d_out, ctx->aux);
  launch_register_histograms(d_out, 1, d_hist, ctx->aux);
  ctx->launches += 2;
  CU(cudaMemcpyAsync(hist64, d_hist, 64 * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->aux));
  CU(cudaStreamSynchronize(ctx->aux));
  cudaFree(d_members); cudaFree(d_out); cudaFree(d_hist);
  return KUQ_OK;
}
}  // namespace

uint64_t kuq_ertl_sparse(const uint32_t *hist64, uint64_t n_observed);

int kuq_counts_size(kuq_ctx *ctx, uint32_t *n) {
  if (!ctx || !n) return KUQ_E_INVALID_ARG;
  CountsHost &h = ctx->snap;
  int rc = ctx->snap_valid ? KUQ_OK : fetch_counts(ctx, h);
  if (rc) return rc;
  uint32_t c = 0;
  for (uint32_t d = 0; d < ctx->n_taxa; d++)
    if (h.n_reads[d] || (d < ctx->n_sketch && h.n_kmers[d])) c++;
  *n = c;
  return KUQ_OK;
}

int kuq_read_counts(kuq_ctx *ctx, uint32_t *taxid, uint64_t *n_reads, uint64_t *n_kmers, uint64_t *unique,
                    uint8_t *is_sparse, uint32_t cap) {
  if (!ctx) return KUQ_E_INVALID_ARG;
  CountsHost &h = ctx->snap;
  int rc = ctx->snap_valid ? KUQ_OK : fetch_counts(ctx, h);
  if (rc) return rc;
  std::vector<std::pair<uint32_t, uint32_t>> rows;   // (taxid, dense)
  for (uint32_t d = 0; d < ctx->n_taxa; d++)
    if (h.n_reads[d] || (d < ctx->n_sketch && h.n_kmers[d])) rows.emplace_back(ctx->raw_of_dense[d], d);
  std::sort(rows.begin(), rows.end());
  if (rows.size() > cap) return fail(ctx, KUQ_E_CAPACITY, "need room for %zu rows", rows.size());
  for (size_t i = 0; i < rows.size(); i++) {
    uint32_t d = rows[i].second;
    uint64_t nk = d < ctx->n_sketch ? h.n_kmers[d] : 0;
    if (taxid) taxid[i] = rows[i].first;
    if (n_reads) n_reads[i] = h.n_reads[d];
    if (n_kmers) n_kmers[i] = nk;
    // the sketch the reference would hold: dense registers if some per-unit (or the global) sketch converted,
    // else the union of the encoded hashes (sparse tier)
    const bool exact = ctx->cfg.hll_mode == KUQ_HLL_EXACT;
    const bool sparse = d < ctx->n_sketch && !exact && ctx->cfg.hll_mode != KUQ_HLL_DENSE_ONLY && !h.dense_flag[d];
    uint64_t u = 0;
    if (exact) u = d < ctx->n_sketch ? h.exact[d] : 0;     // khset size, readcounts.hpp:127-130
    else if (d < ctx->n_sketch && nk)
      u = sparse ? ertl_sparse_hist(&h.sparse_hist[(size_t)d * 64], h.distinct[d], nk)
                 : ertl_dense_hist(&h.hist[(size_t)d * 64], nk);
    if (unique) unique[i] = u;
    if (is_sparse) is_sparse[i] = sparse ? 1 : 0;
  }
  return KUQ_OK;
}

int kuq_clade_counts(kuq_ctx *ctx, const uint32_t *taxids, uint32_t n, uint64_t *n_reads, uint64_t *n_kmers,
                     uint64_t *unique) {
  if (!ctx || (!taxids && n)) return KUQ_E_INVALID_ARG;
  if (!ctx->finalized) return fail(ctx, KUQ_E_STATE, "nothing classified yet");
  CU(cudaSetDevice(ctx->device));
  for (auto &s : ctx->slots) CU(cudaStreamSynchronize(s.stream));
  if (!ctx->snap_valid) {
    int rc = fetch_counts(ctx, ctx->snap);
    if (rc) return rc;
  }
  const CountsHost &h = ctx->snap;
  std::vector<uint32_t> members;
  uint64_t reads = 0, kmers = 0;
  for (uint32_t i = 0; i < n; i++) {
    auto it = ctx->dense_of_raw.find(taxids[i]);
    if (it == ctx->dense_of_raw.end()) continue;
    const uint32_t d = it->second;
    reads += h.n_reads[d];
    if (d < ctx->n_sketch && h.n_kmers[d]) { kmers += h.n_kmers[d]; members.push_back(d); }
  }
  uint64_t u = 0;
  if (ctx->cfg.hll_mode == KUQ_HLL_EXACT) {
    // the clade's container is the union of the members' k-mer sets (readcounts.hpp:76-81)
    uint64_t sum = 0;
    for (uint32_t d : members) sum += h.exact[d];
    if (members.size() == 1) {
      u = sum;
    } else if (!members.empty()) {
      std::vector<uint8_t> member(ctx->n_sketch, 0);
      for (uint32_t d : members) member[d] = 1;
      uint64_t cap = 1024;
      while (cap < 2 * sum + 16) cap <<= 1;
      uint8_t *d_member; unsigned long long *d_set; unsigned long long *d_cnt;
      CU(dmalloc(&d_member, ctx->n_sketch));
      CU(dmalloc(&d_set, cap));
      CU(dmalloc(&d_cnt, 2));
      CU(cudaMemcpyAsync(d_member, member.data(), ctx->n_sketch, cudaMemcpyHostToDevice, ctx->aux));
      CU(cudaMemsetAsync(d_set, 0, cap * 8, ctx->aux));
      CU(cudaMemsetAsync(d_cnt, 0, 16, ctx->aux));
      ExactSet es{ctx->d_exact, ctx->exact_cap - 1, ctx->d_exact_count};
      launch_exact_union(es, d_member, d_set, cap - 1, d_cnt, reinterpret_cast<uint32_t *>(d_cnt + 1), ctx->aux);
      ctx->launches++;
      unsigned long long out[2];
      CU(cudaMemcpyAsync(out, d_cnt, 16, cudaMemcpyDeviceToHost, ctx->aux));
      CU(cudaStreamSynchronize(ctx->aux));
      cudaFree(d_member); cudaFree(d_set); cudaFree(d_cnt);
      if (out[1]) return fail(ctx, KUQ_E_CAPACITY, "internal: clade union scratch overflow");
      u = out[0];
    }
    if (n_reads) *n_reads = reads;
    if (n_kmers) *n_kmers = kmers;
    if (unique) *unique = u;
    return KUQ_OK;
  }
  // clade sketch = merge of the members' sketches: dense as soon as one member is dense
  // (hyperloglogplus.cpp:604-621), else the union of the sparse sets (:600-603)
  uint32_t hist[64];
  int is_dense = 0;
  int rc = clade_hist(ctx, members, hist, &is_dense, /*allow_partial=*/false);
  if (rc) return rc;
  if (!members.empty()) u = is_dense ? ertl_dense_hist(hist, kmers) : kuq_ertl_sparse(hist, kmers);
  if (n_reads) *n_reads = reads;
  if (n_kmers) *n_kmers = kmers;
  if (unique) *unique = u;
  return KUQ_OK;
}

int kuq_clade_partial(kuq_ctx *ctx, const uint32_t *taxids, uint32_t n, uint64_t *n_reads, uint64_t *n_kmers, int *is_dense,
                      uint32_t *hist64) {
  if (!ctx || (!taxids && n) || !hist64 || !is_dense) return KUQ_E_INVALID_ARG;
  if (!ctx->finalized) return fail(ctx, KUQ_E_STATE, "nothing classified yet");
  if (ctx->cfg.hll_mode == KUQ_HLL_EXACT) return fail(ctx, KUQ_E_STATE, "kuq_clade_partial is about sketches (not KUQ_HLL_EXACT)");
  CU(cudaSetDevice(ctx->device));
  for (auto &s : ctx->slots) CU(cudaStreamSynchronize(s.stream));
  if (!ctx->snap_valid) {
    int rc = fetch_counts(ctx, ctx->snap);
    if (rc) return rc;
  }
  const CountsHost &h = ctx->snap;
  std::vector<uint32_t> members;
  uint64_t reads = 0, kmers = 0;
  for (uint32_t i = 0; i < n; i++) {
    auto it = ctx->dense_of_raw.find(taxids[i]);
    if (it == ctx->dense_of_raw.end()) continue;
    const uint32_t d = it->second;
    reads += h.n_reads[d];
    if (d < ctx->n_sketch && h.n_kmers[d]) { kmers += h.n_kmers[d]; members.push_back(d); }
  }
  if (n_reads) *n_reads = reads;
  if (n_kmers) *n_kmers = kmers;
  return clade_hist(ctx, members, hist64, is_dense, /*allow_partial=*/true);
}

// All clades at once (kuq.h).  Host: one pass up the tree for the counters and for which clades are dense / sparse /
// carried by a single taxon; device: kuq_clades.cu.
int kuq_clade_counts_tree(kuq_ctx *ctx, const uint32_t *taxids, uint32_t n, uint64_t *n_reads, uint64_t *n_kmers,
                          uint64_t *unique) {
  if (!ctx || (!taxids && n)) return KUQ_E_INVALID_ARG;
  if (!ctx->finalized) return fail(ctx, KUQ_E_STATE, "nothing classified yet");
  CU(cudaSetDevice(ctx->device));
  for (auto &s : ctx->slots) CU(cudaStreamSynchronize(s.stream));
  if (!ctx->snap_valid) {
    int rc = fetch_counts(ctx, ctx->snap);
    if (rc) return rc;
  }
  const CountsHost &h = ctx->snap;
  const uint32_t NT = ctx->n_taxa, NS = ctx->n_sketch;
  const std::vector<uint32_t> &par = ctx->parent_dense;
  const uint32_t NONE = 0xFFFFFFFFu;
  auto has_kmers = [&](uint32_t d) { return d < NS && h.n_kmers[d] != 0; };
  // ---- the nodes on a path from a counted taxon to its root, children before parents ----------------------------
  std::vector<uint32_t> cid(NT, NONE), nodes;
  for (uint32_t d = 0; d < NT; d++) {
    if (!(h.n_reads[d] || has_kmers(d))) continue;
    for (uint32_t x = d; cid[x] == NONE;) {
      cid[x] = (uint32_t)nodes.size();
      nodes.push_back(x);
      if (x == 0 || par[x] == 0) break;
      x = par[x];
    }
  }
  const uint32_t NC = (uint32_t)nodes.size();
  std::vector<uint32_t> parent_c(NC, NONE), depth_c(NC, 0), order(NC);
  for (uint32_t c = 0; c < NC; c++) {
    const uint32_t x = nodes[c];
    if (x != 0 && par[x] != 0) parent_c[c] = cid[par[x]];
  }
  {  // depth in the compact forest (roots 0); a node's chain was appended root-last, so walk it explicitly
    std::vector<uint32_t> chain;
    std::vector<uint8_t> done(NC, 0);
    for (uint32_t c = 0; c < NC; c++) {
      chain.clear();
      uint32_t x = c;
      while (x != NONE && !done[x]) { chain.push_back(x); x = parent_c[x]; }
      uint32_t d = x == NONE ? 0 : depth_c[x] + 1;
      for (size_t i = chain.size(); i-- > 0;) { depth_c[chain[i]] = d++; done[chain[i]] = 1; }
    }
    for (uint32_t c = 0; c < NC; c++) order[c] = c;
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return depth_c[a] > depth_c[b]; });
  }
  const bool all_dense = ctx->cfg.hll_mode == KUQ_HLL_DENSE_ONLY;
  std::vector<uint64_t> c_reads(NC, 0), c_kmers(NC, 0);
  std::vector<uint32_t> c_members(NC, 0), c_single(NC, NONE);
  std::vector<uint8_t> c_dense(NC, 0);
  for (uint32_t c = 0; c < NC; c++) {
    const uint32_t d = nodes[c];
    c_reads[c] = h.n_reads[d];
    if (has_kmers(d)) { c_kmers[c] = h.n_kmers[d]; c_members[c] = 1; c_single[c] = d; c_dense[c] = all_dense || h.dense_flag[d]; }
  }
  for (uint32_t c : order) {
    const uint32_t q = parent_c[c];
    if (q == NONE) continue;
    c_reads[q] += c_reads[c];
    c_kmers[q] += c_kmers[c];
    if (c_members[c]) {
      if (c_members[q] == 0) c_single[q] = c_single[c];
      c_members[q] += c_members[c];
      c_dense[q] |= c_dense[c];
    }
  }
  // ---- what was asked for ---------------------------------------------------------------------------------------
  std::vector<uint32_t> req(n, NONE);
  std::vector<uint8_t> wanted(NC, 0);
  for (uint32_t i = 0; i < n; i++) {
    auto it = ctx->dense_of_raw.find(taxids[i]);
    if (it != ctx->dense_of_raw.end() && cid[it->second] != NONE) { req[i] = cid[it->second]; wanted[req[i]] = 1; }
  }
  std::vector<uint64_t> c_unique(NC, 0);
  const bool per_clade = ctx->cfg.hll_mode == KUQ_HLL_EXACT || ctx->merged_summary;
  bool sparse_fallback = false;
  std::vector<uint32_t> dense_list, sparse_multi;          // compact ids
  if (!per_clade) {
    for (uint32_t c = 0; c < NC; c++) {
      if (c_members[c] == 0) continue;
      if (c_members[c] == 1) {
        if (!wanted[c]) continue;
        const uint32_t d = c_single[c];
        c_unique[c] = c_dense[c] ? ertl_dense_hist(&h.hist[(size_t)d * 64], c_kmers[c]) : kuq_ertl_sparse(&h.sparse_hist[(size_t)d * 64], c_kmers[c]);
      } else if (c_dense[c]) {
        if (wanted[c]) dense_list.push_back(c);
      } else {
        sparse_multi.push_back(c);                          // needed for the sums up the tree whether asked for or not
      }
    }
  }
  // ---- dense clades: register-wise max of the members, in chunks ---------------------------------------------------
  if (!dense_list.empty()) {
    std::vector<uint32_t> dix(NC, NONE);
    for (uint32_t i = 0; i < dense_list.size(); i++) dix[dense_list[i]] = i;
    std::vector<uint32_t> offs(dense_list.size() + 1, 0), mem;
    for (int pass = 0; pass < 2; pass++) {
      std::vector<uint32_t> fill(offs.begin(), offs.end() - 1);
      for (uint32_t c = 0; c < NC; c++) {
        if (!has_kmers(nodes[c])) continue;
        for (uint32_t x = c; x != NONE; x = parent_c[x])
          if (dix[x] != NONE) { if (pass == 0) offs[dix[x] + 1]++; else mem[fill[dix[x]]++] = nodes[c]; }
      }
      if (pass == 0) { for (size_t i = 1; i < offs.size(); i++) offs[i] += offs[i - 1]; mem.resize(offs.back()); }
    }
    const uint32_t CH = 8192;                                // clades per launch: 32 MB of folded registers
    uint32_t *d_offs = nullptr, *d_mem = nullptr, *d_hist = nullptr;
    uint8_t *d_out = nullptr;
    std::vector<uint32_t> hist((size_t)CH * 64), loc;
    CU(dmalloc(&d_offs, CH + 1));
    CU(dmalloc(&d_mem, std::max<size_t>(mem.size(), 1)));
    CU(dmalloc(&d_out, (uint64_t)CH * HLL_M));
    CU(dmalloc(&d_hist, (uint64_t)CH * 64));
    CU(cudaMemcpyAsync(d_mem, mem.data(), mem.size() * 4, cudaMemcpyHostToDevice, ctx->aux));
    for (uint32_t a = 0; a < dense_list.size(); a += CH) {
      const uint32_t m = std::min<uint32_t>(CH, (uint32_t)dense_list.size() - a);
      loc.assign(offs.begin() + a, offs.begin() + a + m + 1);           // absolute offsets into d_mem
      CU(cudaMemcpyAsync(d_offs, loc.data(), (m + 1) * 4ull, cudaMemcpyHostToDevice, ctx->aux));
      launch_clade_max_batch(ctx->d_regs, d_offs, d_mem, m, d_out, ctx->aux);
      launch_register_histograms(d_out, m, d_hist, ctx->aux);
      ctx->launches += 2;
      CU(cudaMemcpyAsync(hist.data(), d_hist, (uint64_t)m * 64 * 4, cudaMemcpyDeviceToHost, ctx->aux));
      CU(cudaStreamSynchronize(ctx->aux));
      for (uint32_t i = 0; i < m; i++) {
        const uint32_t c = dense_list[a + i];
        c_unique[c] = ertl_dense_hist(&hist[(size_t)i * 64], c_kmers[c]);
      }
    }
    cudaFree(d_offs); cudaFree(d_mem); cudaFree(d_out); cudaFree(d_hist);
  }
  // ---- sparse clades with several members: distinct codes of every subtree from one sort ------------------------------
  if (!sparse_multi.empty()) {
    std::vector<int32_t> sid(NC, -1);
    for (uint32_t i = 0; i < sparse_multi.size(); i++) sid[sparse_multi[i]] = (int32_t)i;
    // preorder numbers: children lists from the parent pointers, explicit stack
    std::vector<uint32_t> first_child(NC + 1, 0), child(NC), pre(NC, NONE), node_of_pre(NC, 0);
    for (uint32_t c = 0; c < NC; c++) if (parent_c[c] != NONE) first_child[parent_c[c] + 1]++;
    for (uint32_t c = 0; c < NC; c++) first_child[c + 1] += first_child[c];
    {
      std::vector<uint32_t> fill(first_child.begin(), first_child.end() - 1);
      for (uint32_t c = 0; c < NC; c++) if (parent_c[c] != NONE) child[fill[parent_c[c]]++] = c;
      std::vector<uint32_t> stack;
      uint32_t counter = 0;
      for (uint32_t r = 0; r < NC; r++) {
        if (parent_c[r] != NONE) continue;
        stack.push_back(r);
        while (!stack.empty()) {
          const uint32_t x = stack.back();
          stack.pop_back();
          pre[x] = counter;
          node_of_pre[counter++] = x;
          for (uint32_t i = first_child[x]; i < first_child[x + 1]; i++) stack.push_back(child[i]);
        }
      }
    }
    std::vector<uint32_t> pre_of_taxon(NS, NONE);
    uint64_t n_keys = 0;
    for (uint32_t c = 0; c < NC; c++) {
      const uint32_t d = nodes[c];
      if (d < NS) { pre_of_taxon[d] = pre[c]; if (has_kmers(d) && !h.dense_flag[d]) n_keys += h.distinct[d]; }
    }
    uint32_t *d_pre = nullptr, *d_nop = nullptr, *d_par = nullptr, *d_dep = nullptr, *d_dup = nullptr;
    int32_t *d_sid = nullptr;
    CU(dmalloc(&d_pre, NS)); CU(dmalloc(&d_nop, NC)); CU(dmalloc(&d_par, NC)); CU(dmalloc(&d_dep, NC)); CU(dmalloc(&d_sid, NC));
    CU(dmalloc(&d_dup, sparse_multi.size() * 64));
    CU(cudaMemcpyAsync(d_pre, pre_of_taxon.data(), NS * 4ull, cudaMemcpyHostToDevice, ctx->aux));
    CU(cudaMemcpyAsync(d_nop, node_of_pre.data(), NC * 4ull, cudaMemcpyHostToDevice, ctx->aux));
    CU(cudaMemcpyAsync(d_par, parent_c.data(), NC * 4ull, cudaMemcpyHostToDevice, ctx->aux));
    CU(cudaMemcpyAsync(d_dep, depth_c.data(), NC * 4ull, cudaMemcpyHostToDevice, ctx->aux));
    CU(cudaMemcpyAsync(d_sid, sid.data(), NC * 4ull, cudaMemcpyHostToDevice, ctx->aux));
    CU(cudaMemsetAsync(d_dup, 0, sparse_multi.size() * 64 * 4ull, ctx->aux));
    const int src = sparse_clade_dups(ctx->d_sparse_slots, ctx->sparse_cap, ctx->d_dense_flag, n_keys, d_pre, d_nop, d_par, d_dep,
                                      d_sid, d_dup, ctx->n_sm, ctx->aux);
    ctx->launches += 3;
    std::vector<uint32_t> dup(sparse_multi.size() * 64, 0);
    cudaError_t ce = cudaSuccess;
    if (src == 0) {
      ce = cudaMemcpyAsync(dup.data(), d_dup, dup.size() * 4, cudaMemcpyDeviceToHost, ctx->aux);
      if (ce == cudaSuccess) ce = cudaStreamSynchronize(ctx->aux);
    }
    cudaFree(d_pre); cudaFree(d_nop); cudaFree(d_par); cudaFree(d_dep); cudaFree(d_sid); cudaFree(d_dup);
    if (src == 2 || ce != cudaSuccess) return fail(ctx, KUQ_E_CUDA, "clade roll-up (sparse tier) failed: %s", cudaGetErrorString(cudaGetLastError()));
    if (src == 1) {
      sparse_fallback = true;                                // no room for the sort: one union per clade instead
    } else {
      // rank histogram of every sparse subtree: own codes + children's − the pairs booked at the node
      std::vector<std::vector<uint32_t>> H(NC);
      for (uint32_t c : order) {
        if (c_members[c] == 0 || c_dense[c]) continue;
        std::vector<uint32_t> &hc = H[c];
        if (hc.empty()) hc.assign(64, 0);
        const uint32_t d = nodes[c];
        if (has_kmers(d)) for (int r = 0; r < 64; r++) hc[r] += h.sparse_hist[(size_t)d * 64 + r];
        if (sid[c] >= 0) for (int r = 0; r < 64; r++) hc[r] -= dup[(size_t)sid[c] * 64 + r];
        if (wanted[c] && c_members[c] > 1) c_unique[c] = kuq_ertl_sparse(hc.data(), c_kmers[c]);
        const uint32_t q = parent_c[c];
        if (q != NONE && !c_dense[q]) {
          std::vector<uint32_t> &hq = H[q];
          if (hq.empty()) hq.assign(64, 0);
          for (int r = 0; r < 64; r++) hq[r] += hc[r];
        }
        std::vector<uint32_t>().swap(hc);
      }
    }
  }
  // ---- exact counting / partitioned sparse tier / no memory for the sort: one merge per clade ------------------------
  if (per_clade || sparse_fallback) {
    std::vector<std::vector<uint32_t>> lists(NC);
    for (uint32_t c = 0; c < NC; c++) {
      if (!(h.n_reads[nodes[c]] || has_kmers(nodes[c]))) continue;
      for (uint32_t x = c; x != NONE; x = parent_c[x])
        if (wanted[x] && (per_clade || (c_members[x] > 1 && !c_dense[x]))) lists[x].push_back(ctx->raw_of_dense[nodes[c]]);
    }
    for (uint32_t c = 0; c < NC; c++) {
      if (lists[c].empty()) continue;
      uint64_t r = 0, k = 0, u = 0;
      int rc = kuq_clade_counts(ctx, lists[c].data(), (uint32_t)lists[c].size(), &r, &k, &u);
      if (rc) return rc;
      c_unique[c] = u;
    }
  }
  for (uint32_t i = 0; i < n; i++) {
    const uint32_t c = req[i];
    if (n_reads) n_reads[i] = c == NONE ? 0 : c_reads[c];
    if (n_kmers) n_kmers[i] = c == NONE ? 0 : c_kmers[c];
    if (unique) unique[i] = c == NONE ? 0 : c_unique[c];
  }
  return KUQ_OK;
}

uint64_t kuq_ertl_dense_hist(const uint32_t *hist64, uint64_t n_observed) { return ertl_dense_hist(hist64, n_observed); }

int kuq_get_registers(kuq_ctx *ctx, uint32_t taxid, uint8_t *regs) {
  if (!ctx || !regs) return KUQ_E_INVALID_ARG;
  if (!ctx->finalized) return fail(ctx, KUQ_E_STATE, "nothing classified yet");
  CU(cudaSetDevice(ctx->device));
  for (auto &s : ctx->slots) CU(cudaStreamSynchronize(s.stream));
  memset(regs, 0, HLL_M);
  auto it = ctx->dense_of_raw.find(taxid);
  if (it == ctx->dense_of_raw.end() || it->second >= ctx->n_sketch) return KUQ_OK;
  CU(cudaMemcpy(regs, ctx->d_regs + (size_t)it->second * HLL_M, HLL_M, cudaMemcpyDeviceToHost));
  return KUQ_OK;
}

int kuq_state_ptrs_get(kuq_ctx *ctx, kuq_state_ptrs *out) {
  if (!ctx || !out) return KUQ_E_INVALID_ARG;
  int rc = ensure_ready(ctx);
  if (rc) return rc;
  out->d_regs = ctx->d_regs;
  out->regs_bytes = (uint64_t)ctx->n_sketch * HLL_M;
  out->d_n_kmers = reinterpret_cast<uint64_t *>(ctx->d_n_kmers);
  out->d_n_reads = reinterpret_cast<uint64_t *>(ctx->d_n_reads);
  out->d_dense_flag = ctx->d_dense_flag;
  out->n_sketch = ctx->n_sketch;
  out->n_taxa = ctx->n_taxa;
  return KUQ_OK;
}

int kuq_sparse_export(kuq_ctx *ctx, uint64_t *d_keys_out, uint64_t cap, uint64_t *n) {
  if (!ctx || !n) return KUQ_E_INVALID_ARG;
  int rc = ensure_ready(ctx);
  if (rc) return rc;
  *n = 0;
  if (!ctx->d_sparse_slots) return KUQ_OK;                    // KUQ_HLL_DENSE_ONLY: no sparse tier
  CU(cudaSetDevice(ctx->device));
  for (auto &s : ctx->slots) CU(cudaStreamSynchronize(s.stream));
  rc = harvest_seen(ctx, false);
  if (rc) return rc;
  unsigned long long *d_n;
  CU(dmalloc(&d_n, 1));
  CU(cudaMemsetAsync(d_n, 0, 8, ctx->aux));
  launch_sparse_export(ctx->d_sparse_slots, ctx->sparse_cap, ctx->d_dense_flag,
                       reinterpret_cast<unsigned long long *>(d_keys_out), d_keys_out ? cap : 0, d_n, ctx->aux);
  ctx->launches++;
  unsigned long long cnt = 0;
  CU(cudaMemcpyAsync(&cnt, d_n, 8, cudaMemcpyDeviceToHost, ctx->aux));
  CU(cudaStreamSynchronize(ctx->aux));
  cudaFree(d_n);
  *n = cnt;
  if (d_keys_out && cnt > cap) return fail(ctx, KUQ_E_CAPACITY, "need room for %llu keys", cnt);
  return KUQ_OK;
}

// ---- database sharded over GPUs: who counts, step flags, partitioned merge of the sparse tier ---------------------
int kuq_set_shard_counting(kuq_ctx *ctx, int on) {
  if (!ctx) return KUQ_E_INVALID_ARG;
  for (auto &s : ctx->slots)
    if (s.busy) return fail(ctx, KUQ_E_STATE, "cannot change while a batch is in flight");
  ctx->shard_counting = on != 0;
  return KUQ_OK;
}

// ---- a database larger than HBM: ranges streamed from pinned host memory, copy overlapped with the lookups -------------
extern "C++" {
namespace {
uint32_t host_hash_u32(uint32_t x) {                        // == hash_u32 of kuq_kernels.cu
  x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16;
  return x;
}
void stream_close(kuq_ctx *ctx) {
  for (auto &b : ctx->sbuf) {
    cudaFree(b.d_pairs); cudaFree(b.d_offsets);
    if (b.ready) cudaEventDestroy(b.ready);
    b = kuq_ctx::StreamBuf();
  }
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  ctx->copy_stream = nullptr;
  cudaFree(ctx->d_stream_missing);
  ctx->d_stream_missing = nullptr;
  if (ctx->stream_open) { ctx->d_pairs = nullptr; ctx->d_offsets = nullptr; ctx->db_staged = false; }
  ctx->stream_open = false;
}
}  // namespace
}  // extern "C++"

int kuq_stream_open(kuq_ctx *ctx, uint32_t k, uint32_t nt, uint32_t idx_type, uint64_t max_records, uint64_t max_bins) {
  if (!ctx || !max_records || !max_bins) return KUQ_E_INVALID_ARG;
  if (k < 29 || k > 31) return fail(ctx, KUQ_E_UNSUPPORTED_K, "k = %u: only 8-byte keys (k = 29..31)", k);
  if (nt < 1 || nt > 15 || (idx_type != 1 && idx_type != 2)) return fail(ctx, KUQ_E_INVALID_ARG, "bad index parameters");
  if (ctx->universe.empty()) return fail(ctx, KUQ_E_STATE, "declare the taxids of the whole database first (kuq_set_db_taxid_universe)");
  if (!ctx->tax_set) return fail(ctx, KUQ_E_STATE, "no taxonomy set");
  CU(cudaSetDevice(ctx->device));
  { int hrc = harvest_seen(ctx, false); if (hrc) return hrc; }
  free_db(ctx);
  stream_close(ctx);
  ctx->k = k; ctx->nt = nt; ctx->idx_type = idx_type;
  ctx->db_owned = false;
  ctx->db_taxids = ctx->universe;
  std::sort(ctx->db_taxids.begin(), ctx->db_taxids.end());
  ctx->db_taxids.erase(std::unique(ctx->db_taxids.begin(), ctx->db_taxids.end()), ctx->db_taxids.end());
  ctx->db_taxid_counts.assign(ctx->db_taxids.size(), 0);
  ctx->db_staged = true;
  int rc = finalize(ctx);
  if (rc) { ctx->db_staged = false; return rc; }
  // device table taxid → dense id over the whole universe (what collect_taxids builds per staged range otherwise)
  uint32_t cap = 1u << 16;
  while ((uint64_t)cap < 4ull * ctx->db_taxids.size()) cap <<= 1;
  std::vector<uint32_t> keys(cap, 0), dense(cap, 0);
  for (uint32_t t : ctx->db_taxids) {
    uint32_t slot = host_hash_u32(t) & (cap - 1);
    while (keys[slot]) slot = (slot + 1) & (cap - 1);
    keys[slot] = t + 1;
    dense[slot] = ctx->dense_of_raw[t];
  }
  CU(dmalloc(&ctx->d_tx_keys, cap));
  CU(dmalloc(&ctx->d_tx_dense, cap));
  CU(cudaMemcpy(ctx->d_tx_keys, keys.data(), cap * 4ull, cudaMemcpyHostToDevice));
  CU(cudaMemcpy(ctx->d_tx_dense, dense.data(), cap * 4ull, cudaMemcpyHostToDevice));
  ctx->tx_cap = cap;
  ctx->db_remapped = true;                       // each range is remapped as it arrives
  CU(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
  CU(dmalloc(&ctx->d_stream_missing, 1));
  CU(cudaMemset(ctx->d_stream_missing, 0, 4));
  for (auto &b : ctx->sbuf) {
    CU(cudaMalloc((void **)&b.d_pairs, max_records * 12 + SLACK));
    CU(dmalloc(&b.d_offsets, max_bins + 1));
    CU(cudaEventCreateWithFlags(&b.ready, cudaEventDisableTiming));
  }
  ctx->stream_cap_records = max_records;
  ctx->stream_cap_bins = max_bins;
  ctx->stream_open = true;
  ctx->key_ct = 0;
  return KUQ_OK;
}

int kuq_stream_load(kuq_ctx *ctx, uint32_t buf, const void *host_records, uint64_t n_records, const uint64_t *host_offsets,
                    uint64_t bin_lo, uint64_t bin_hi) {
  if (!ctx || buf > 1 || !host_offsets || (!host_records && n_records)) return KUQ_E_INVALID_ARG;
  if (!ctx->stream_open) return fail(ctx, KUQ_E_STATE, "kuq_stream_open first");
  if (bin_lo >= bin_hi || bin_hi - bin_lo > ctx->stream_cap_bins || n_records > ctx->stream_cap_records)
    return fail(ctx, KUQ_E_CAPACITY, "range of %llu records / %llu bins exceeds the stream buffers", (unsigned long long)n_records,
                (unsigned long long)(bin_hi - bin_lo));
  CU(cudaSetDevice(ctx->device));
  kuq_ctx::StreamBuf &b = ctx->sbuf[buf];
  // whoever still reads this buffer was queued before this call: the copy waits for the slots' streams as they stand
  if (ctx->seen_dirty) { int hrc = harvest_seen(ctx, false); if (hrc) return hrc; }
  for (auto &s : ctx->slots) {
    CU(cudaEventRecord(s.ev_sync, s.stream));
    CU(cudaStreamWaitEvent(ctx->copy_stream, s.ev_sync, 0));
  }
  if (n_records) CU(cudaMemcpyAsync(b.d_pairs, host_records, n_records * 12, cudaMemcpyHostToDevice, ctx->copy_stream));
  CU(cudaMemcpyAsync(b.d_offsets, host_offsets, (bin_hi - bin_lo + 1) * 8, cudaMemcpyHostToDevice, ctx->copy_stream));
  launch_remap_values(b.d_pairs, n_records, ctx->d_tx_keys, ctx->d_tx_dense, ctx->tx_cap - 1, ctx->d_stream_missing,
                      ctx->k >= 32 ? ~0ull : ((1ull << (2 * ctx->k)) - 1), ctx->copy_stream);
  ctx->launches++;
  CU(cudaEventRecord(b.ready, ctx->copy_stream));
  b.key_ct = n_records; b.rec_base = host_offsets[0]; b.bin_lo = bin_lo; b.bin_hi = bin_hi; b.loaded = true;
  return KUQ_OK;
}

int kuq_stream_use(kuq_ctx *ctx, uint32_t buf) {
  if (!ctx || buf > 1) return KUQ_E_INVALID_ARG;
  if (!ctx->stream_open || !ctx->sbuf[buf].loaded) return fail(ctx, KUQ_E_STATE, "stream buffer %u holds no range", buf);
  CU(cudaSetDevice(ctx->device));
  if (ctx->seen_dirty) { int hrc = harvest_seen(ctx, false); if (hrc) return hrc; }
  kuq_ctx::StreamBuf &b = ctx->sbuf[buf];
  for (auto &s : ctx->slots) CU(cudaStreamWaitEvent(s.stream, b.ready, 0));
  ctx->d_pairs = b.d_pairs; ctx->d_offsets = b.d_offsets;
  ctx->key_ct = b.key_ct; ctx->rec_base = b.rec_base; ctx->bin_lo = b.bin_lo; ctx->bin_hi = b.bin_hi;
  return KUQ_OK;
}

int kuq_stream_check(kuq_ctx *ctx) {
  if (!ctx) return KUQ_E_INVALID_ARG;
  if (!ctx->stream_open) return KUQ_OK;
  CU(cudaSetDevice(ctx->device));
  CU(cudaStreamSynchronize(ctx->copy_stream));
  uint32_t missing = 0;
  CU(cudaMemcpy(&missing, ctx->d_stream_missing, 4, cudaMemcpyDeviceToHost));
  if (missing) return fail(ctx, KUQ_E_STATE, "a streamed range holds a taxid outside the declared universe");
  return KUQ_OK;
}

int kuq_host_register(void *p, uint64_t bytes) {
  if (!p || !bytes) return KUQ_E_INVALID_ARG;
  if (cudaHostRegister(p, bytes, cudaHostRegisterDefault) == cudaSuccess) return KUQ_OK;
  (void)cudaGetLastError();
  // a read-only mapping (mmap PROT_READ of database.kdb) can only be pinned read-only
  if (cudaHostRegister(p, bytes, cudaHostRegisterReadOnly) == cudaSuccess) return KUQ_OK;
  (void)cudaGetLastError();
  return KUQ_E_CUDA;
}
int kuq_host_unregister(void *p) {
  if (!p) return KUQ_E_INVALID_ARG;
  if (cudaHostUnregister(p) != cudaSuccess) { (void)cudaGetLastError(); return KUQ_E_CUDA; }
  return KUQ_OK;
}

// Several GPUs in ONE process (the drop-in `classify` with replicas): fold the per-taxon state of `src` into `dst`.
int kuq_merge_into(kuq_ctx *dst, kuq_ctx *src) {
  kuq_ctx *ctx = dst;
  if (!dst || !src || dst == src) return KUQ_E_INVALID_ARG;
  if (!src->finalized) return KUQ_OK;                       // src never classified anything: nothing to add
  if (!dst->finalized) return fail(ctx, KUQ_E_STATE, "the destination context has not classified anything yet");
  if (dst->n_taxa != src->n_taxa || dst->n_sketch != src->n_sketch || dst->raw_of_dense != src->raw_of_dense ||
      dst->cfg.hll_mode != src->cfg.hll_mode)
    return fail(ctx, KUQ_E_STATE, "the contexts number their taxa differently (different database / taxonomy / HLL mode)");
  if (dst->cfg.hll_mode == KUQ_HLL_EXACT) return fail(ctx, KUQ_E_STATE, "kuq_merge_into does not merge exact k-mer sets");
  // src: flagged records → its set (skipping what dst already knows to be dense is a refinement left out)
  CU(cudaSetDevice(src->device));
  for (auto &s : src->slots) CU(cudaStreamSynchronize(s.stream));
  { int rc = harvest_seen(src, false); if (rc) { dst->err = src->err; return rc; } }
  uint64_t n_keys = 0;
  uint64_t *d_keys_src = nullptr;
  if (src->d_sparse_slots) {
    int rc = kuq_sparse_export(src, nullptr, 0, &n_keys);
    if (rc) { dst->err = src->err; return rc; }
    if (n_keys) {
      if (cudaMalloc((void **)&d_keys_src, n_keys * 8) != cudaSuccess) { (void)cudaGetLastError(); return fail(ctx, KUQ_E_NOMEM, "no room for %llu keys", (unsigned long long)n_keys); }
      uint64_t n2 = 0;
      rc = kuq_sparse_export(src, d_keys_src, n_keys, &n2);
      if (rc) { cudaFree(d_keys_src); dst->err = src->err; return rc; }
      n_keys = n2;
    }
  }
  CU(cudaSetDevice(dst->device));
  for (auto &s : dst->slots) CU(cudaStreamSynchronize(s.stream));
  { int rc = harvest_seen(dst, false); if (rc) return rc; }
  dst->snap_valid = false;
  dst->merged_summary = false;
  uint8_t *t_regs, *t_dense; unsigned long long *t_nk, *t_nr;
  const uint64_t reg_bytes = (uint64_t)dst->n_sketch * HLL_M;
  CU(cudaMalloc((void **)&t_regs, reg_bytes));
  CU(dmalloc(&t_dense, dst->n_sketch));
  CU(dmalloc(&t_nk, dst->n_sketch));
  CU(dmalloc(&t_nr, dst->n_taxa));
  CU(cudaMemcpyPeer(t_regs, dst->device, src->d_regs, src->device, reg_bytes));
  CU(cudaMemcpyPeer(t_dense, dst->device, src->d_dense_flag, src->device, dst->n_sketch));
  CU(cudaMemcpyPeer(t_nk, dst->device, src->d_n_kmers, src->device, dst->n_sketch * 8ull));
  CU(cudaMemcpyPeer(t_nr, dst->device, src->d_n_reads, src->device, dst->n_taxa * 8ull));
  launch_merge_state(dst->d_regs, t_regs, dst->d_n_kmers, t_nk, dst->n_sketch, dst->d_n_reads, t_nr, dst->n_taxa, dst->d_dense_flag,
                     t_dense, dst->aux);
  dst->launches++;
  CU(cudaStreamSynchronize(dst->aux));
  cudaFree(t_regs); cudaFree(t_dense); cudaFree(t_nk); cudaFree(t_nr);
  int rc = KUQ_OK;
  if (n_keys && dst->d_sparse_slots) {
    uint64_t *d_keys_dst = nullptr;
    if (cudaMalloc((void **)&d_keys_dst, n_keys * 8) != cudaSuccess) { (void)cudaGetLastError(); cudaSetDevice(src->device); cudaFree(d_keys_src); return fail(ctx, KUQ_E_NOMEM, "no room for %llu keys", (unsigned long long)n_keys); }
    CU(cudaMemcpyPeer(d_keys_dst, dst->device, d_keys_src, src->device, n_keys * 8));
    // make room first: the import itself cannot grow the set
    std::vector<uint32_t> distinct(dst->n_sketch);
    CU(cudaMemcpy(distinct.data(), dst->d_sparse_distinct, dst->n_sketch * 4ull, cudaMemcpyDeviceToHost));
    uint64_t used = 0;
    for (uint32_t v : distinct) used += v;
    if ((used + n_keys) * 10 > dst->sparse_cap * 8) {
      uint64_t cap = dst->sparse_cap;
      while ((used + n_keys) * 10 > cap * 6) cap <<= 1;
      int grc = grow_sparse_set(dst, cap);
      if (grc) { cudaFree(d_keys_dst); return grc; }
    }
    dst->direct_upper = used + n_keys;
    rc = kuq_sparse_import(dst, d_keys_dst, n_keys);
    cudaFree(d_keys_dst);
  }
  if (d_keys_src) { cudaSetDevice(src->device); cudaFree(d_keys_src); cudaSetDevice(dst->device); }
  return rc;
}

int kuq_enable_peer_access(kuq_ctx *ctx, kuq_ctx *peer) {
  if (!ctx || !peer) return KUQ_E_INVALID_ARG;
  if (ctx->device == peer->device) return KUQ_OK;
  CU(cudaSetDevice(ctx->device));
  int can = 0;
  CU(cudaDeviceCanAccessPeer(&can, ctx->device, peer->device));
  if (!can) return fail(ctx, KUQ_E_STATE, "device %d cannot map the memory of device %d", ctx->device, peer->device);
  cudaError_t e = cudaDeviceEnablePeerAccess(peer->device, 0);
  if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return fail(ctx, KUQ_E_CUDA, "cudaDeviceEnablePeerAccess: %s", cudaGetErrorString(e));
  (void)cudaGetLastError();
  return KUQ_OK;
}

int kuq_set_stats(kuq_ctx *ctx, int on) {
  if (!ctx) return KUQ_E_INVALID_ARG;
  ctx->extra_flags = on ? KUQ_F_STATS : 0u;
  return KUQ_OK;
}

int kuq_signal_peers(kuq_ctx *ctx, uint32_t slot, uint64_t *const *d_flag_peers, uint32_t n_peers, uint32_t my_index,
                     uint64_t value) {
  int rc = check_slot(ctx, slot);
  if (rc) return rc;
  if (!d_flag_peers || n_peers == 0 || n_peers > 8 || my_index >= 8) return fail(ctx, KUQ_E_INVALID_ARG, "1..8 peers");
  CU(cudaSetDevice(ctx->device));
  launch_signal_peers(reinterpret_cast<unsigned long long *const *>(d_flag_peers), n_peers, my_index, value, ctx->slots[slot].stream);
  ctx->launches++;
  CU(cudaGetLastError());
  return KUQ_OK;
}

int kuq_wait_flags(kuq_ctx *ctx, uint32_t slot, const uint64_t *d_flags, uint32_t n, uint64_t value, uint32_t timeout_ms) {
  int rc = check_slot(ctx, slot);
  if (rc) return rc;
  if (!d_flags || n == 0 || n > 32) return fail(ctx, KUQ_E_INVALID_ARG, "1..32 flags");
  CU(cudaSetDevice(ctx->device));
  if (!ctx->d_sync_err) {
    CU(dmalloc(&ctx->d_sync_err, 1));
    CU(cudaMemset(ctx->d_sync_err, 0, 4));
  }
  launch_wait_flags(reinterpret_cast<const unsigned long long *>(d_flags), n, value, (unsigned long long)(timeout_ms ? timeout_ms : 20000) * 1000000ull,
                    ctx->d_sync_err, ctx->slots[slot].stream);
  ctx->launches++;
  CU(cudaGetLastError());
  return KUQ_OK;
}

static int export_partitioned(kuq_ctx *ctx, uint32_t n_parts, uint64_t *d_keys_out, uint64_t cap, uint64_t *counts, uint64_t **alloc_out);

int kuq_sparse_export_partitioned(kuq_ctx *ctx, uint32_t n_parts, uint64_t *d_keys_out, uint64_t cap, uint64_t *counts) {
  return export_partitioned(ctx, n_parts, d_keys_out, cap, counts, nullptr);
}
int kuq_sparse_export_partitioned_alloc(kuq_ctx *ctx, uint32_t n_parts, uint64_t **d_keys_out, uint64_t *counts) {
  if (!d_keys_out) return KUQ_E_INVALID_ARG;
  *d_keys_out = nullptr;
  return export_partitioned(ctx, n_parts, nullptr, 0, counts, d_keys_out);
}

static int export_partitioned(kuq_ctx *ctx, uint32_t n_parts, uint64_t *d_keys_out, uint64_t cap, uint64_t *counts, uint64_t **alloc_out) {
  if (!ctx || !counts || n_parts == 0 || n_parts > 8) return KUQ_E_INVALID_ARG;
  int rc = ensure_ready(ctx);
  if (rc) return rc;
  for (uint32_t j = 0; j < n_parts; j++) counts[j] = 0;
  if (!ctx->d_sparse_slots) return KUQ_OK;
  CU(cudaSetDevice(ctx->device));
  for (auto &s : ctx->slots) CU(cudaStreamSynchronize(s.stream));
  // Two sources: the keys already in the local set (misses, resolve-half inserts, earlier harvests) and the records
  // flagged since the last harvest.  The flagged records are NOT inserted locally first: their keys go straight into
  // the export buffer (and the flags are cleared) — after the exchange every key is inserted exactly once, by its owner.
  const uint64_t key_mask = ctx->k >= 32 ? ~0ull : ((1ull << (2 * ctx->k)) - 1);
  const bool records = ctx->seen_dirty && ctx->d_pairs && ctx->key_ct;
  unsigned long long *d_cnt;
  CU(dmalloc(&d_cnt, 24));                       // [0:8) counts / cursors, [8:16) part ends, [16] error word
  CU(cudaMemsetAsync(d_cnt, 0, 24 * 8, ctx->aux));
  uint32_t *d_err = reinterpret_cast<uint32_t *>(d_cnt + 16);
  launch_keys_parts(0, ctx->d_sparse_slots, nullptr, ctx->sparse_cap, key_mask, ctx->d_dense_flag, n_parts, d_cnt, nullptr, nullptr, d_err, 0, ctx->aux);
  ctx->launches++;
  if (records) {
    launch_keys_parts(1, nullptr, ctx->d_pairs, ctx->key_ct, key_mask, ctx->d_dense_flag, n_parts, d_cnt, nullptr, nullptr, d_err, 0, ctx->aux);
    ctx->launches++;
  }
  unsigned long long h[8];
  CU(cudaMemcpyAsync(h, d_cnt, 64, cudaMemcpyDeviceToHost, ctx->aux));
  CU(cudaStreamSynchronize(ctx->aux));
  uint64_t total = 0;
  for (uint32_t j = 0; j < n_parts; j++) { counts[j] = h[j]; total += h[j]; }
  if (alloc_out) {                                         // the library sizes the buffer (one counting pass instead of two)
    if (cudaMalloc((void **)&d_keys_out, (total ? total : 1) * 8) != cudaSuccess) {
      (void)cudaGetLastError();
      cudaFree(d_cnt);
      return fail(ctx, KUQ_E_NOMEM, "no room for %llu exported keys", (unsigned long long)total);
    }
    *alloc_out = d_keys_out;
    cap = total;
  }
  if (!d_keys_out) { cudaFree(d_cnt); return KUQ_OK; }     // counts only: nothing was consumed
  if (total > cap) { cudaFree(d_cnt); return fail(ctx, KUQ_E_CAPACITY, "need room for %llu keys", (unsigned long long)total); }
  unsigned long long lay[16];
  lay[0] = 0;
  for (uint32_t j = 1; j < 8; j++) lay[j] = lay[j - 1] + (j - 1 < n_parts ? h[j - 1] : 0);
  for (uint32_t j = 0; j < 8; j++) lay[8 + j] = lay[j] + (j < n_parts ? h[j] : 0);
  CU(cudaMemcpyAsync(d_cnt, lay, 128, cudaMemcpyHostToDevice, ctx->aux));
  launch_keys_parts(0, ctx->d_sparse_slots, nullptr, ctx->sparse_cap, key_mask, ctx->d_dense_flag, n_parts, d_cnt,
                    reinterpret_cast<unsigned long long *>(d_keys_out), d_cnt + 8, d_err, 1, ctx->aux);
  ctx->launches++;
  if (records) {
    launch_keys_parts(1, nullptr, ctx->d_pairs, ctx->key_ct, key_mask, ctx->d_dense_flag, n_parts, d_cnt,
                      reinterpret_cast<unsigned long long *>(d_keys_out), d_cnt + 8, d_err, 1, ctx->aux);
    ctx->launches++;
    ctx->seen_dirty = false;                     // the flags are gone: their keys live in the export buffer now
  }
  uint32_t err = 0;
  CU(cudaMemcpyAsync(&err, d_err, 4, cudaMemcpyDeviceToHost, ctx->aux));
  CU(cudaStreamSynchronize(ctx->aux));
  cudaFree(d_cnt);
  if (err) return fail(ctx, KUQ_E_CAPACITY, "internal: partitioned export overran a segment");
  return KUQ_OK;
}

int kuq_sparse_replace(kuq_ctx *ctx, const uint64_t *d_keys, uint64_t n) {
  if (!ctx || (!d_keys && n)) return KUQ_E_INVALID_ARG;
  int rc = ensure_ready(ctx);
  if (rc) return rc;
  if (!ctx->d_sparse_slots) return KUQ_OK;
  CU(cudaSetDevice(ctx->device));
  for (auto &s : ctx->slots) CU(cudaStreamSynchronize(s.stream));
  rc = harvest_seen(ctx, true);                  // anything still flagged was exported before; drop the flags
  if (rc) return rc;
  ctx->snap_valid = false;
  uint64_t cap = ctx->sparse_cap;
  while (n * 10 > cap * 7) cap <<= 1;
  if (cap != ctx->sparse_cap) {
    cudaFree(ctx->d_sparse_slots);
    ctx->d_sparse_slots = nullptr;
    if (dmalloc(&ctx->d_sparse_slots, cap) != cudaSuccess) {
      (void)cudaGetLastError();
      ctx->sparse_cap = 0;
      return fail(ctx, KUQ_E_NOMEM, "sparse-tier set: no room for %llu slots", (unsigned long long)cap);
    }
    ctx->sparse_cap = cap;
    ctx->sparse_grown++;
  }
  CU(cudaMemsetAsync(ctx->d_sparse_slots, 0, ctx->sparse_cap * 8ull, ctx->aux));
  CU(cudaMemsetAsync(ctx->d_sparse_distinct, 0, ctx->n_sketch * 4ull, ctx->aux));
  CU(cudaStreamSynchronize(ctx->aux));
  ctx->direct_upper = n;
  return kuq_sparse_import(ctx, d_keys, n);
}

int kuq_sparse_summary(kuq_ctx *ctx, uint32_t *d_hist_out, uint32_t *d_distinct_out) {
  if (!ctx || !d_hist_out || !d_distinct_out) return KUQ_E_INVALID_ARG;
  int rc = ensure_ready(ctx);
  if (rc) return rc;
  CU(cudaSetDevice(ctx->device));
  for (auto &s : ctx->slots) CU(cudaStreamSynchronize(s.stream));
  rc = harvest_seen(ctx, false);
  if (rc) return rc;
  CU(cudaMemsetAsync(d_hist_out, 0, (uint64_t)ctx->n_sketch * 64 * 4, ctx->aux));
  if (ctx->d_sparse_slots) {
    launch_sparse_histograms(ctx->d_sparse_slots, ctx->sparse_cap, ctx->d_dense_flag, d_hist_out, ctx->aux);
    ctx->launches++;
    CU(cudaMemcpyAsync(d_distinct_out, ctx->d_sparse_distinct, ctx->n_sketch * 4ull, cudaMemcpyDeviceToDevice, ctx->aux));
  } else {
    CU(cudaMemsetAsync(d_distinct_out, 0, ctx->n_sketch * 4ull, ctx->aux));
  }
  CU(cudaStreamSynchronize(ctx->aux));
  return KUQ_OK;
}

int kuq_set_sparse_summary(kuq_ctx *ctx, const uint32_t *d_hist, const uint32_t *d_distinct) {
  if (!ctx || !d_hist || !d_distinct) return KUQ_E_INVALID_ARG;
  int rc = ensure_ready(ctx);
  if (rc) return rc;
  CU(cudaSetDevice(ctx->device));
  ctx->merged_hist.resize((size_t)ctx->n_sketch * 64);
  ctx->merged_distinct.resize(ctx->n_sketch);
  CU(cudaMemcpy(ctx->merged_hist.data(), d_hist, (uint64_t)ctx->n_sketch * 64 * 4, cudaMemcpyDeviceToHost));
  CU(cudaMemcpy(ctx->merged_distinct.data(), d_distinct, ctx->n_sketch * 4ull, cudaMemcpyDeviceToHost));
  ctx->merged_summary = true;
  ctx->snap_valid = false;
  return KUQ_OK;
}

uint64_t kuq_ertl_sparse(const uint32_t *hist64, uint64_t n_observed) {
  uint64_t n_codes = 0;
  for (int i = 0; i < 64; i++) n_codes += hist64[i];
  return ertl_sparse_hist(hist64, n_codes, n_observed);
}

int kuq_scan_device(kuq_ctx *ctx, uint32_t slot, uint32_t k, uint32_t nt, uint32_t idx_type, const char *d_bases,
                    const uint64_t *d_read_offsets, uint32_t n_reads, uint64_t total_bases, uint64_t *d_canon_out,
                    uint32_t *d_bins_out) {
  if (!d_bases || !d_read_offsets || !d_canon_out || !d_bins_out) return fail(ctx, KUQ_E_INVALID_ARG, "NULL device buffers");
  if (k < 2 || k > 31 || nt < 1 || nt > 15 || nt > k || (idx_type != 1 && idx_type != 2)) return fail(ctx, KUQ_E_INVALID_ARG, "bad k / minimizer length / index type");
  int rc = begin_batch(ctx, slot, n_reads, total_bases, 0, true, d_bases, d_read_offsets);
  if (rc) return rc;
  Slot &s = ctx->slots[slot];
  Params p;
  memset(&p, 0, sizeof p);
  p.db.k = k; p.db.nt = nt;
  p.db.key_mask = (1ull << (2 * k)) - 1;
  p.db.xor_mask = (uint32_t)((idx_type == 1 ? 0ull : INDEX2_XOR_MASK) & ((1ull << (2 * nt)) - 1));
  p.db.n_mini = k - nt + 1;
  p.bases = d_bases; p.offsets = d_read_offsets; p.clean = s.d_clean;
  p.n_reads = n_reads; p.n_chunks = (n_reads + CHUNK_READS - 1) / CHUNK_READS;
  p.total_bases = total_bases;
  p.n_windows = s.d_nwin; p.canon = d_canon_out; p.bins = d_bins_out;
  p.chunk_counter = reinterpret_cast<uint32_t *>(s.d_scalars + 2);
  p.error_flag = reinterpret_cast<uint32_t *>(s.d_scalars + 3);
  CU(cudaMemsetAsync(s.d_scalars, 0, 8 * 8, s.stream));
  ctx->launches += launch_scan_only(p, ctx->n_sm, s.stream);
  CU(cudaGetLastError());
  return KUQ_OK;
}

int kuq_layout_experiment(kuq_ctx *ctx, uint32_t slot, uint64_t n_positions, uint32_t reps, kuq_layout_result *out) {
  int rc = check_slot(ctx, slot);
  if (rc) return rc;
  if (!out) return fail(ctx, KUQ_E_INVALID_ARG, "NULL result");
  CU(cudaSetDevice(ctx->device));
  rc = ensure_ready(ctx);
  if (rc) return rc;
  if (!ctx->db_staged || ctx->stream_open || !ctx->d_pairs) return fail(ctx, KUQ_E_STATE, "the experiment needs a staged (not streamed) database");
  if (ctx->k != 31 || ctx->nt != 15) return fail(ctx, KUQ_E_INVALID_ARG, "the 8-byte record code is defined for k = 31, m = 15");
  Slot &s = ctx->slots[slot];
  if (!s.timed || n_positions == 0 || n_positions > s.total_bases)
    return fail(ctx, KUQ_E_STATE, "run a batch on the slot first; n_positions must not exceed its text length");
  Params p;
  fill_params(ctx, s, p, nullptr, nullptr, nullptr, 0, 0);
  const int erc = layout_experiment(p, ctx->key_ct, s.d_canon, s.d_bins, s.d_dense, n_positions, ctx->n_sm, s.stream, reps,
                                    ctx->cfg.hll_mode == KUQ_HLL_DENSE_ONLY, out);
  ctx->snap_valid = false;
  ctx->launches += 2 + (uint64_t)KUQ_LAYOUT_VARIANTS * (reps + 2ull);
  if (erc == 1) return fail(ctx, KUQ_E_NOMEM, "not enough free device memory for the transcoded records");
  if (erc == 3) return fail(ctx, KUQ_E_CAPACITY, "dense taxon ids need more than 24 bits");
  if (erc) return fail(ctx, KUQ_E_CUDA, "layout experiment: %s", cudaGetErrorString(cudaGetLastError()));
  return KUQ_OK;
}

int kuq_sparse_tier_info(kuq_ctx *ctx, uint64_t *slots, uint64_t *keys, uint64_t *times_grown, double *last_harvest_ms) {
  if (!ctx) return KUQ_E_INVALID_ARG;
  int rc = ensure_ready(ctx);
  if (rc) return rc;
  if (slots) *slots = ctx->sparse_cap;
  if (times_grown) *times_grown = ctx->sparse_grown;
  if (last_harvest_ms) *last_harvest_ms = ctx->harvest_ms;
  if (keys) {
    *keys = 0;
    if (ctx->d_sparse_distinct) {
      CU(cudaSetDevice(ctx->device));
      for (auto &s : ctx->slots) CU(cudaStreamSynchronize(s.stream));
      std::vector<uint32_t> d(ctx->n_sketch);
      CU(cudaMemcpy(d.data(), ctx->d_sparse_distinct, ctx->n_sketch * 4ull, cudaMemcpyDeviceToHost));
      for (uint32_t v : d) *keys += v;
    }
  }
  return KUQ_OK;
}

int kuq_sparse_import(kuq_ctx *ctx, const uint64_t *d_keys, uint64_t n) {
  if (!ctx || (!d_keys && n)) return KUQ_E_INVALID_ARG;
  int rc = ensure_ready(ctx);
  if (rc) return rc;
  if (!ctx->d_sparse_slots || !n) return KUQ_OK;
  ctx->snap_valid = false;
  CU(cudaSetDevice(ctx->device));
  for (auto &s : ctx->slots) CU(cudaStreamSynchronize(s.stream));
  SparseSet ss;
  ss.slots = ctx->d_sparse_slots; ss.mask = ctx->sparse_cap - 1; ss.n_used = ctx->d_sparse_used;
  ss.distinct = ctx->d_sparse_distinct;
  uint32_t *d_err;
  CU(dmalloc(&d_err, 1));
  CU(cudaMemsetAsync(d_err, 0, 4, ctx->aux));
  launch_sparse_import(reinterpret_cast<const unsigned long long *>(d_keys), n, ss, ctx->d_dense_flag, d_err, ctx->aux);
  ctx->launches++;
  uint32_t err = 0;
  CU(cudaMemcpyAsync(&err, d_err, 4, cudaMemcpyDeviceToHost, ctx->aux));
  CU(cudaStreamSynchronize(ctx->aux));
  cudaFree(d_err);
  if (err) return fail(ctx, KUQ_E_CAPACITY, "sparse-tier set saturated while importing");
  return KUQ_OK;
}

int kuq_dense_taxids(kuq_ctx *ctx, uint32_t *taxid_of_dense, uint32_t cap, uint32_t *n) {
  if (!ctx || !n) return KUQ_E_INVALID_ARG;
  int rc = ensure_ready(ctx);
  if (rc) return rc;
  *n = ctx->n_taxa;
  if (cap == 0) return KUQ_OK;
  if (cap < ctx->n_taxa) return fail(ctx, KUQ_E_CAPACITY, "need room for %u ids", ctx->n_taxa);
  memcpy(taxid_of_dense, ctx->raw_of_dense.data(), ctx->n_taxa * 4ull);
  return KUQ_OK;
}

int kuq_reset_counts(kuq_ctx *ctx) {
  if (!ctx) return KUQ_E_INVALID_ARG;
  ctx->snap_valid = false;
  if (!ctx->finalized) return KUQ_OK;
  CU(cudaSetDevice(ctx->device));
  for (auto &s : ctx->slots) CU(cudaStreamSynchronize(s.stream));
  { int hrc = harvest_seen(ctx, true); if (hrc) return hrc; }
  CU(cudaMemset(ctx->d_regs, 0, (uint64_t)ctx->n_sketch * HLL_M));
  CU(cudaMemset(ctx->d_dense_flag, 0, ctx->n_sketch));
  CU(cudaMemset(ctx->d_n_kmers, 0, ctx->n_sketch * 8ull));
  CU(cudaMemset(ctx->d_n_reads, 0, ctx->n_taxa * 8ull));
  if (ctx->d_sparse_slots) {
    CU(cudaMemset(ctx->d_sparse_slots, 0, ctx->sparse_cap * 8ull));
    CU(cudaMemset(ctx->d_sparse_used, 0, 8));
    CU(cudaMemset(ctx->d_sparse_distinct, 0, ctx->n_sketch * 4ull));
    ctx->direct_upper = 0;
  }
  if (ctx->d_exact) {
    CU(cudaMemset(ctx->d_exact, 0, ctx->exact_cap * 16ull));
    CU(cudaMemset(ctx->d_exact_count, 0, ctx->n_sketch * 8ull));
  }
  ctx->unit_nt = 0;
  ctx->unit_next = 0;
  return KUQ_OK;
}

uint64_t kuq_ertl_dense(const uint8_t *regs, uint64_t n_observed) {
  int C[66];
  memset(C, 0, sizeof C);
  for (uint32_t i = 0; i < HLL_M; i++) C[regs[i] > 65 ? 65 : regs[i]]++;
  return ertl_from_hist(C, 64 - HLL_P, HLL_M, n_observed);
}

// ---- database build (SURVEY.md §8 f4; ROUND 1: compiled, not yet run on hardware) ---------------------------------
int kuq_db_sort(int device, const void *jdb_image, uint64_t jdb_bytes, uint32_t nt, int zero_vals, void *kdb_out,
                void *idx_out, char *err, uint64_t err_cap) {
  int n_dev = 0;
  if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) {
    if (err && err_cap) snprintf(err, err_cap, "db_sort: no CUDA device (there is no CPU path)");
    (void)cudaGetLastError();
    return KUQ_E_NO_DEVICE;
  }
  if (device < 0 || device >= n_dev || cudaSetDevice(device) != cudaSuccess) return KUQ_E_INVALID_ARG;
  int rc = dbsort_device((const uint8_t *)jdb_image, jdb_bytes, nt, zero_vals, (uint8_t *)kdb_out, (uint8_t *)idx_out, err, err_cap);
  return rc ? KUQ_E_DB_FORMAT : KUQ_OK;
}

int kuq_set_lcas_batch(kuq_ctx *ctx, const char *bases, const uint64_t *piece_offsets, uint32_t n_pieces,
                       const uint32_t *taxid, uint32_t flags, uint64_t *n_missing) {
  if (n_pieces && (!bases || !piece_offsets || !taxid)) return fail(ctx, KUQ_E_INVALID_ARG, "NULL batch buffers");
  int rc = begin_batch(ctx, 0, n_pieces, host_bases(piece_offsets, n_pieces), 0, false);
  if (!rc) rc = ensure_ready(ctx);
  if (rc) return rc;
  Slot &s = ctx->slots[0];
  if (ctx->bin_lo != 0 || ctx->rec_base != 0) return fail(ctx, KUQ_E_STATE, "set_lcas needs the whole database staged");
  for (uint32_t i = 0; i < n_pieces; i++) {
    // the reference skips sequences whose taxid the taxonomy does not hold (set_lcas.cpp:336-341): the caller's job
    auto it = ctx->dense_of_raw.find(taxid[i]);
    if (taxid[i] == 0 || it == ctx->dense_of_raw.end())
      return fail(ctx, KUQ_E_INVALID_ARG, "piece %u: taxid %u is not in the taxonomy", i, taxid[i]);
    s.h_unit[i] = it->second;
  }
  if (flags & KUQ_LCA_FORCE_CONTAMINANT) {
    // first-come-first-kept between the two contaminant taxids is the one order dependence of -T: one kind per batch
    bool c1 = false, c2 = false;
    for (uint32_t i = 0; i < n_pieces; i++) { c1 |= taxid[i] == 32630u; c2 |= taxid[i] == 81077u; }
    if (c1 && c2) return fail(ctx, KUQ_E_INVALID_ARG, "with KUQ_LCA_FORCE_CONTAMINANT a batch may hold pieces of taxid 32630 or of 81077, not both");
  }
  rc = upload_reads(ctx, s, bases, piece_offsets);
  if (rc) return rc;
  if (n_pieces) CU(cudaMemcpyAsync(s.d_unit, s.h_unit, n_pieces * 4ull, cudaMemcpyHostToDevice, s.stream));
  Params p;
  fill_params(ctx, s, p, s.d_bases, s.d_offsets, s.d_unit, n_pieces, 0);
  p.lca_flags = flags & (KUQ_LCA_FORCE_CONTAMINANT | KUQ_LCA_RESET);
  {
    auto c1 = ctx->dense_of_raw.find(32630u), c2 = ctx->dense_of_raw.find(81077u);   // set_lcas.cpp:88-89
    p.lca_keep[0] = c1 == ctx->dense_of_raw.end() ? 0 : c1->second;
    p.lca_keep[1] = c2 == ctx->dense_of_raw.end() ? 0 : c2->second;
  }
  CU(cudaMemsetAsync(s.d_scalars, 0, 8 * 8, s.stream));
  ctx->lca_mode = true;
  ctx->snap_valid = false;
  ctx->launches += launch_set_lcas(p, ctx->n_sm, s.stream);
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(s.h_scalars, s.d_scalars, 8 * 8, cudaMemcpyDeviceToHost, s.stream));
  CU(cudaStreamSynchronize(s.stream));
  if (n_missing) *n_missing = s.h_scalars[4];
  return KUQ_OK;
}

int kuq_export_db_values(kuq_ctx *ctx, void *kdb_image, uint64_t kdb_bytes) {
  if (!ctx || !kdb_image) return KUQ_E_INVALID_ARG;
  if (!ctx->db_staged || !ctx->db_owned) return fail(ctx, KUQ_E_STATE, "no database staged from a host image");
  if (ctx->bin_lo != 0 || ctx->rec_base != 0) return fail(ctx, KUQ_E_STATE, "only a fully staged database can be exported");
  CU(cudaSetDevice(ctx->device));
  for (auto &s : ctx->slots) CU(cudaStreamSynchronize(s.stream));
  const uint64_t key_bits = 2ull * ctx->k, header = 72 + 2 * (4 + 8 * key_bits);
  if (kdb_bytes < header + ctx->key_ct * 12) return fail(ctx, KUQ_E_INVALID_ARG, "image too small for %llu records", (unsigned long long)ctx->key_ct);
  std::vector<uint8_t> rec(ctx->key_ct * 12);
  CU(cudaMemcpy(rec.data(), ctx->d_pairs, rec.size(), cudaMemcpyDeviceToHost));
  uint8_t *out = (uint8_t *)kdb_image + header;
  for (uint64_t i = 0; i < ctx->key_ct; i++) {
    uint32_t v;
    memcpy(&v, rec.data() + i * 12 + 8, 4);
    if (ctx->db_remapped) {                                 // dense id → taxid
      if (v >= ctx->n_taxa) return fail(ctx, KUQ_E_STATE, "record %llu holds an unknown dense id %u", (unsigned long long)i, v);
      v = ctx->raw_of_dense[v];
    }
    memcpy(out + i * 12 + 8, &v, 4);
  }
  return KUQ_OK;
}

}  // extern "C"
