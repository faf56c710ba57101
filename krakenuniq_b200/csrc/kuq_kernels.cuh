// kuq_kernels.cuh — sm_100a kernels of the KrakenUniq classification hot path (device side of libkuq.so).
//
// The per-read path of the reference's classify_sequence() (src/classify.cpp:897-1012) as three kernels:
//
//  k_scan     read blocks --TMA bulk copy--> shared memory    (cp.async.bulk + mbarrier, double buffered)
//   (warp     2-bit packing + ambiguity mask   KmerScanner::next_kmer   src/krakenutil.cpp:239-282
//    per      canonical k-mer                  canonical_representation src/krakendb.cpp:238-246
//    read)    rolling minimizer                bin_key                  src/krakendb.cpp:200-215
//             → scratch: canonical k-mer + bin per window (12 B, coalesced)
//  k_lookup   index fetch + bin search         kmer_query               src/krakendb.cpp:250-321, :586-593
//   (thread   HLL register update              ReadCounts::add_kmer     src/readcounts.hpp:71-74,
//    per                                                                 hyperloglogplus.cpp:485-523
//    window)  → scratch: dense taxon id per window
//  k_resolve  hit aggregation + tree resolve   resolve_tree / lca       src/krakenutil.cpp:90-118,149-200
//   (warp     per-taxon counters               classify.cpp:939,968
//    per      run-length hit list              hitlist_string           src/classify.cpp:826-861
//    read)
//
// k_scan is ALU/shuffle work with no dependent memory access; k_lookup is the random-HBM stage and is written
// thread-per-window with a small register footprint so that ~48 warps per SM keep enough probes in flight;
// consecutive threads hold consecutive windows of a read, so windows sharing a minimizer touch the same index
// sector and the same pivots (coalesced by the load unit).  No tensor cores: the path is integer compares on
// randomly addressed HBM (SURVEY.md §8(d)).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/kuq.h"

namespace kuq {

// Params::flags holds the public KUQ_F_* bits of kuq.h and two internal bits the library sets above them:
constexpr uint32_t F_FOUND_ZERO = 16u;        // MODE_LOOKUP reports a stored taxon 0 as FOUND_ZERO (kuq_mark_zero_hits)
constexpr uint32_t F_SHARD_COUNTING = 32u;    // the lookup half does the sketch work of its hits (kuq_set_shard_counting)
static_assert(F_FOUND_ZERO > (KUQ_F_WANT_CODES | KUQ_F_NO_RUNS | KUQ_F_NO_COUNTS | KUQ_F_STATS),
              "the internal launch flags must not overlap the public KUQ_F_* bits");

constexpr uint32_t AMBIG = 0xFFFFFFFFu;
// MODE_LOOKUP with F_FOUND_ZERO: the key IS in the database but stores taxon 0 (an un-LCA'd record).  With several
// databases that still ends the search (classify.cpp:928-936), so the lookup has to tell it from a miss.
constexpr uint32_t FOUND_ZERO = 0xFFFFFFFDu;
constexpr int CTA_THREADS = 256;
constexpr int CTA_WARPS = CTA_THREADS / 32;
constexpr int CHUNK_READS = 64;            // reads per CTA work item
constexpr int STAGE_BYTES = 24 * 1024;     // bytes of read text per shared-memory stage
constexpr int N_STAGES = 2;
constexpr uint32_t HLL_P = 12;
constexpr uint32_t HLL_M = 4096;
// Record flag in the key word's free top bit (keys hold 2k <= 62 bits; the reference masks the rest away,
// krakendb.cpp:283-284): "a counted hit has seen this record since the last harvest" — the sparse HLL tier of hits.
constexpr uint32_t SEEN_BIT = 0x80000000u;
constexpr int SEARCH_WINDOW = 8;           // records scanned linearly once the bisection window is this small

enum Mode { MODE_FUSED = 0, MODE_LOOKUP = 1, MODE_RESOLVE = 2 };

struct DbView {
  const uint8_t *pairs;      // records of the staged range, on-disk layout: {u64 key, u32 value} packed to 12 B
  const uint64_t *offsets;   // offsets[b - bin_lo] = absolute record index of the first record of bin b
  uint64_t rec_base;         // absolute record index of pairs[0]
  uint64_t key_mask;         // (1 << 2k) - 1
  uint32_t bin_lo, bin_hi;   // staged minimizer range [bin_lo, bin_hi)
  uint32_t k, nt;
  uint32_t xor_mask;         // INDEX2_XOR_MASK & (4^nt - 1) for KRAKIX2, 0 for KRAKIDX (krakendb.cpp:45,203-206)
  uint32_t n_mini;           // k - nt + 1 minimizer candidates per k-mer (krakendb.cpp:208)
};

struct TaxView {
  const uint32_t *parent;    // dense id → dense id of the parent (0 = none), Parent_map of taxdb.hpp:383-398
  const uint16_t *depth;     // dense id → steps to the end of its parent chain (0 or the node of taxid 1)
  const uint32_t *raw;       // dense id → taxid
  uint32_t n_taxa;
  uint32_t n_sketch;         // dense ids < n_sketch own HLL registers / k-mer counters
};

struct SparseSet {           // device set of (dense taxon, encoded hash) pairs: the sparse HLL tier
  unsigned long long *slots; // 0 = empty; key = (taxon + 1) << 32 | code
  uint64_t mask;             // capacity - 1 (power of two)
  unsigned long long *n_used;
  uint32_t *distinct;        // [n_sketch] distinct codes inserted per taxon
};

// Per-batch bookkeeping of the reference's per-work-unit sketches (classify.cpp:525: one ReadCounts map per work
// unit).  A (unit, taxon) sketch converts from sparse to dense iff an insert finds >= 1024 distinct encoded hashes
// already stored (hyperloglogplus.cpp:496-498), so only pairs with > 1024 inserts need their distinct count.
struct UnitMap {
  unsigned long long *keys;   // 0 = empty; (unit + 1) << 32 | taxon   (open addressing, per batch)
  uint32_t *inserts;          // N(unit, taxon): add_kmer calls
  uint32_t *distinct;         // D(unit, taxon): distinct encoded hashes (only counted for candidates, saturating)
  unsigned long long *last;   // (read << 32 | window) of the last insert of the pair
  uint8_t *cand;              // 1 = candidate (N >= 1025 and the taxon is not already known dense)
  uint32_t mask;              // capacity - 1
  uint8_t *taxon_cand;        // [n_sketch] some unit of this batch makes the taxon a candidate
  uint32_t *n_cand;           // number of candidate pairs of the batch
  unsigned long long *set_keys;  // distinct (pair slot, code): 0 = empty; (slot + 1) << 32 | code
  uint32_t *set_count;           // occurrences of the key
  uint32_t set_mask;
  // fast path for the insert counts: units of a batch are (nearly always) consecutive ids, so N(unit, taxon) lives in a
  // dense table direct[(unit - unit_id[0]) * n_sketch + taxon] — one fire-and-forget atomic per (read, taxon), no probe.
  // Pairs outside the table (rows >= direct_rows) use the hash map above; k_unit_mark moves the candidates there.
  uint32_t *direct;
  uint32_t direct_rows;
};

// classifyExact (EXACT_COUNTING, classify.cpp:46-49): the per-taxon container is a set of canonical k-mers.  All
// sets of a run share one open-addressing table of 16-byte entries, filled with 128-bit compare-and-swap.
struct alignas(16) ExactPair {
  unsigned long long kmer1;    // canonical k-mer + 1 (0 = empty slot)
  unsigned long long taxon1;   // dense taxon id + 1
};
struct ExactSet {
  ExactPair *slots;
  uint64_t mask;               // capacity - 1 (power of two)
  unsigned long long *count;   // [n_sketch] distinct k-mers per taxon == khset size (readcounts.hpp:127-130)
};

struct Params {
  DbView db;
  TaxView tax;
  // batch
  const char *bases;            // 16-byte aligned, >= 32 bytes of slack after the last base
  const uint64_t *offsets;      // [n_reads + 1], relative to bases
  const uint32_t *unit_id;      // [n_reads] or nullptr
  char *clean;                  // scratch of the same size as bases for reads containing '\n' / '\r'
  uint32_t n_reads;
  uint32_t n_chunks;
  uint32_t flags;
  uint32_t hll_mode;
  // outputs
  uint32_t *call;               // [n_reads] taxid
  uint32_t *n_windows;          // [n_reads]
  uint32_t *codes;              // per window, indexed like bases (taxids; only with KUQ_F_WANT_CODES)
  uint64_t total_bases;
  // scratch between the stages (indexed like bases)
  uint64_t *canon;              // canonical k-mer of the window
  uint32_t *bins;               // minimizer bin, or BIN_AMBIG / BIN_NONE
  uint32_t *codes_dense;        // dense taxon id of the window (0 = miss) or AMBIG
  const uint32_t *codes_in;     // MODE_RESOLVE: merged dense ids
  uint32_t *run_start;
  uint32_t *run_count;
  uint2 *runs;
  unsigned long long *run_cursor;
  uint64_t runs_capacity;       // entries of runs[]
  unsigned long long *n_classified;
  uint32_t *chunk_counter;      // dynamic chunk scheduler
  uint32_t *error_flag;
  uint32_t only_hits;           // MODE_LOOKUP: write hits only (peer-memory merge)
  // MODE_LOOKUP over NVLink: text positions [peer_bounds[j], peer_bounds[j+1]) belong to the reads GPU j resolves;
  // their hits are stored straight into that GPU's buffer (peer memory mapped through CUDA IPC)
  uint32_t n_peers;
  uint32_t *peer_codes[8];
  uint64_t peer_bounds[9];
  unsigned long long *stats;    // KUQ_F_STATS: [0] += looked-up windows, [1] += sum of ceil(log2(bin size + 1))
  // per-taxon state
  uint8_t *regs;                // [n_sketch][4096]
  unsigned long long *n_kmers;  // [n_sketch]
  unsigned long long *n_reads_ctr; // [n_taxa]
  uint8_t *dense_flag;          // [n_sketch]
  SparseSet sparse;
  UnitMap units;
  // pool for the hit tables of reads with more than 32 distinct taxa (2 u64 per entry)
  unsigned long long *ovf_mem;
  unsigned long long *ovf_cursor;
  uint64_t ovf_capacity;
  // quick mode (classify -q -m quick_min; 0 = off).  quick_stop: the read ends at its quick_min-th hit
  // (classify.cpp:943-944); otherwise every k-mer counts and only the call rule changes (the -x path, :701-738)
  uint32_t quick_min;
  uint32_t quick_stop;
  ExactSet exact;               // hll_mode 3 (KUQ_HLL_EXACT)
  // set_lcas: 1 = -T (values lca_keep[] stick, pieces with such a taxid overwrite), 2 = -R (values become 0)
  uint32_t lca_flags;
  uint32_t lca_keep[2];         // dense ids of taxids 32630 / 81077 (0 = not in the taxonomy)
};

// returns #kernels launched; stage_events[0] / [1] (optional) are recorded after k_scan / k_lookup
int launch_classify(int mode, const Params &p, int n_sm, cudaStream_t stream, cudaEvent_t *stage_events);
int classify_smem_bytes();
// set_lcas: k_scan + k_set_lcas over library pieces (p.unit_id = dense taxid per piece, p.stats[0] += k-mers not found)
int launch_set_lcas(const Params &p, int n_sm, cudaStream_t stream);
int launch_scan_only(const Params &p, int n_sm, cudaStream_t stream);
int launch_lookup_only(const Params &p, int n_sm, cudaStream_t stream, int fused, int lean);
// db_sort on the device (kuq_dbbuild.cu)
int dbsort_device(const uint8_t *jdb_image, uint64_t jdb_bytes, uint32_t nt, int zero_vals, uint8_t *kdb_out,
                  uint8_t *idx_out, char *err, size_t err_cap);

// database staging helpers
void launch_collect_taxids(const uint8_t *pairs, uint64_t n_rec, uint32_t *keys, unsigned long long *counts,
                           uint32_t cap_mask, uint32_t *overflow, cudaStream_t stream);
void launch_remap_values(uint8_t *pairs, uint64_t n_rec, const uint32_t *keys, const uint32_t *dense,
                         uint32_t cap_mask, uint32_t *missing, uint64_t key_mask, cudaStream_t stream);
// flagged records → sparse-tier keys: mode 0 count (stats[0]), 1 insert + clear, 2 clear only
void launch_harvest_seen(uint8_t *pairs, uint64_t n_rec, uint64_t key_mask, const uint8_t *dense_flag, const SparseSet &set,
                         unsigned long long *stats, uint32_t *error_flag, int mode, cudaStream_t stream);
void launch_sparse_rehash(const unsigned long long *old_slots, uint64_t old_cap, const SparseSet &s, uint32_t *error_flag,
                          cudaStream_t stream);
void launch_register_histograms(const uint8_t *regs, uint32_t n_sketch, uint32_t *hist /*[n_sketch][64]*/,
                                cudaStream_t stream);
void launch_clade_max(const uint8_t *regs, const uint32_t *members, uint32_t n_members, uint8_t *out4096,
                      cudaStream_t stream);
void launch_fill_u32(uint32_t *p, uint64_t n, uint32_t v, cudaStream_t stream);
// HLL mode rule, per batch: mark candidate (unit, taxon) pairs, count their distinct codes, flag dense taxa
int launch_unit_accounting(const Params &p, int n_sm, cudaStream_t stream);
void launch_unit_clear(const UnitMap &u, uint32_t n_sketch, int n_sm, cudaStream_t stream);
// chunked rule: one global sketch per taxon converts once it holds >= 1025 distinct codes
void launch_flag_dense_global(const uint32_t *distinct, uint8_t *dense_flag, uint32_t n_sketch, cudaStream_t stream);
// histogram of encoded ranks over the sparse set, per taxon: hist[t][64] (+ hist[t][63] unused)
void launch_sparse_histograms(const unsigned long long *slots, uint64_t cap, const uint8_t *dense_flag,
                              uint32_t *hist, cudaStream_t stream);
// distinct codes of the union of the member taxa (member[t] != 0): rank histogram hist64 via a scratch set
// exact mode: distinct k-mers over the member taxa (set union of ReadCounts::operator+=, readcounts.hpp:76-81)
void launch_exact_union(const ExactSet &e, const uint8_t *member, unsigned long long *scratch_set, uint64_t scratch_mask,
                        unsigned long long *n_distinct, uint32_t *overflow, cudaStream_t stream);
void launch_sparse_union(const unsigned long long *slots, uint64_t cap, const uint8_t *member,
                         unsigned long long *scratch_set, uint64_t scratch_mask, uint32_t *hist64, uint32_t *overflow,
                         cudaStream_t stream);

void launch_sparse_export(const unsigned long long *slots, uint64_t cap, const uint8_t *dense_flag,
                          unsigned long long *out, uint64_t out_cap, unsigned long long *n_out, cudaStream_t stream);
void launch_sparse_import(const unsigned long long *keys, uint64_t n, const SparseSet &s, const uint8_t *dense_flag,
                          uint32_t *error_flag, cudaStream_t stream);

void launch_merge_state(uint8_t *regs, const uint8_t *regs2, unsigned long long *n_kmers, const unsigned long long *n_kmers2,
                        uint32_t n_sketch, unsigned long long *n_reads, const unsigned long long *n_reads2, uint32_t n_taxa,
                        uint8_t *dense, const uint8_t *dense2, cudaStream_t stream);
// cross-GPU flags (kuq_signal_peers / kuq_wait_flags) and the partitioned export of the sparse tier
void launch_signal_peers(unsigned long long *const *flag_ptrs, uint32_t n, uint32_t my_index, unsigned long long value,
                         cudaStream_t stream);
void launch_wait_flags(const unsigned long long *flags, uint32_t n, unsigned long long value, unsigned long long timeout_ns,
                       uint32_t *error_flag, cudaStream_t stream);
// keys of the still-sparse taxa grouped by owner part: src 0 = slots of the local set, src 1 = flagged records (pass 1
// clears the flags); pass 0 counts into counters[part], pass 1 scatters through counters[part] (cursors), bounded by part_end
void launch_keys_parts(int src, const unsigned long long *slots, uint8_t *pairs, uint64_t n_items, uint64_t key_mask,
                       const uint8_t *dense_flag, uint32_t n_parts, unsigned long long *counters, unsigned long long *out,
                       const unsigned long long *part_end, uint32_t *error_flag, int pass, cudaStream_t stream);

// kuq_clades.cu: all clades of the report at once
void launch_clade_max_batch(const uint8_t *regs, const uint32_t *d_offs, const uint32_t *d_members, uint32_t n_clades,
                            uint8_t *d_out, cudaStream_t stream);
int sparse_clade_dups(const unsigned long long *slots, uint64_t cap, const uint8_t *dense_flag, uint64_t n_keys_upper,
                      const uint32_t *d_pre_of_taxon, const uint32_t *d_node_of_pre, const uint32_t *d_parent_c,
                      const uint32_t *d_depth_c, const int32_t *d_sid_of_node, uint32_t *d_dup, int n_sm, cudaStream_t stream);
// kuq_layout_exp.cu: record-layout / search-shape experiment (0 ok, 1 no memory, 2 CUDA error, 3 taxon ids > 24 bits);
// `product` = parameters of a k_lookup<MODE_LOOKUP> launch on the same database (scratch / output pointers are set there)
int layout_experiment(const Params &product, uint64_t n_records, const uint64_t *canon, const uint32_t *bins, const uint32_t *ref,
                      uint64_t n_pos, int n_sm, cudaStream_t st, uint32_t reps, int allow_fused, ::kuq_layout_result *res);

}  // namespace kuq
