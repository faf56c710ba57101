/* include/kuq.h — C ABI of libkuq.so: KrakenUniq's per-read classification hot path on one NVIDIA B200 (sm_100a).
 *
 * The reference (fbreitwieser/krakenuniq v1.0.4) has no plugin / FFI interface; its drop-in surface is the
 * `classify` executable and the on-disk formats (SURVEY.md §8(b)).  Inside that executable the hot path is one
 * function, `classify_sequence()` (src/classify.cpp:897-1012), called per read from the work-unit loop of
 * `process_file()` (src/classify.cpp:487-564) with the global state `KrakenDatabases`, `Parent_map` and
 * `taxon_counts` (src/classify.cpp:78,109,113).  This header is the boundary a maintainer binds instead of that
 * loop body: plain pointers and sizes in, plain arrays out, int error codes, no C++ or torch types.
 * Citations are file:line under the reference's src/.
 *
 *   reference object / call                              → entry point here
 *   ---------------------------------------------------------------------------------------------------------
 *   QuickFile::open_file + load_file (-M), KrakenDB(ptr),   kuq_stage_db            (HBM takes the place of the
 *     KrakenDBIndex(ptr)   classify.cpp:176-200,             page cache; krakendb.cpp:60-78,534-544 validation)
 *   KrakenDB::prepare_chunking / load_chunk (-x)            kuq_stage_db with a minimizer range [bin_lo,bin_hi)
 *     krakendb.cpp:411-522
 *   KrakenDB::count_taxons  krakendb.cpp:90-113             kuq_db_taxids           (by-product of staging)
 *   TaxonomyDB::getParentMap → Parent_map                   kuq_set_taxonomy
 *     taxdb.hpp:383-398, classify.cpp:217-219
 *   process_file work-unit loop + classify_sequence         kuq_classify_batch / kuq_submit_batch+kuq_wait_batch
 *     classify.cpp:506-559, 897-1012                          (host buffers) and kuq_classify_device (HBM buffers)
 *   classify_sequence_with_db_chunk (per-chunk lookups)     kuq_lookup_device   (per-window taxa of one DB range)
 *     classify.cpp:1014-1056
 *   merge + final pass of the chunked mode                  kuq_resolve_device  (calls + counters from merged taxa)
 *     classify.cpp:390-485, 663-791
 *   taxon_counts (ReadCounts<HyperLogLogPlusMinus>)         kuq_read_counts / kuq_get_registers / kuq_state_ptrs
 *     classify.cpp:78, readcounts.hpp:32-129
 *
 * Threading: a context is bound to one CUDA device and is thread-compatible (one caller at a time).  Each of
 * its `n_slots` batch slots owns a CUDA stream plus device and pinned-host staging, so H2D copy, kernels and D2H
 * copy of consecutive batches overlap when the caller alternates slots.
 */
#ifndef KUQ_H
#define KUQ_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

/* ---- error codes (0 = success).  The reference calls errx()/exit() in these situations. ---------------- */
#define KUQ_OK 0
#define KUQ_E_INVALID_ARG (-1)    /* NULL pointer, zero size, bad slot ... */
#define KUQ_E_CUDA (-2)           /* a CUDA runtime call failed (kuq_last_error has the text) */
#define KUQ_E_NO_DEVICE (-3)      /* no usable sm_100 device: there is no CPU fallback */
#define KUQ_E_DB_FORMAT (-4)      /* krakendb.cpp:64-74: not JFLISTDN / val_len != 4; :541: bad index magic */
#define KUQ_E_UNSUPPORTED_K (-5)  /* only 8-byte keys (k = 29..31; every published KrakenUniq DB is k=31) */
#define KUQ_E_STATE (-6)          /* call order: DB and taxonomy must be set before classifying, ... */
#define KUQ_E_CAPACITY (-7)       /* batch larger than the configured slot capacity */
#define KUQ_E_NOMEM (-8)          /* host or device allocation failed */
#define KUQ_E_TAXA_OVERFLOW (-9)  /* pool for the hit tables of reads with > 32 distinct taxa exhausted */
#define KUQ_E_TAXONOMY (-10)      /* cyclic parent chain in the taxonomy */

/* per-window code for an ambiguous k-mer ("A:" in the Kraken hit list, classify.cpp:846-848) */
#define KUQ_CODE_AMBIG 0xFFFFFFFFu

/* HLL mode rule to reproduce (SURVEY.md §7.3 item 1, App. C) */
#define KUQ_HLL_PRELOAD 0   /* per-work-unit sketches merged into the global map (classify.cpp:525,542-544) */
#define KUQ_HLL_CHUNKED 1   /* one global sketch per taxon (classify.cpp:719) — the `-x` path */
#define KUQ_HLL_DENSE_ONLY 2 /* p=12 registers only, no sparse-tier emulation (fastest; estimates = dense Ertl) */
#define KUQ_HLL_EXACT 3     /* classifyExact (EXACT_COUNTING, classify.cpp:46-49): sets of k-mers instead of sketches;
                               `unique` of kuq_read_counts / kuq_clade_counts is the exact set / union size.  The
                               (taxon, k-mer) table takes kuq_config.sparse_set_slots entries of 16 bytes. */

/* flags of the classify calls */
#define KUQ_F_WANT_CODES 1u     /* also return the per-window codes (4 B per base position) */
#define KUQ_F_NO_RUNS 2u        /* skip the run-length-encoded hit lists */
#define KUQ_F_NO_COUNTS 4u      /* do not touch the per-taxon counters / sketches (pure lookups) */
#define KUQ_F_STATS 8u          /* measurement aid: accumulate the algorithmic probe counts (kuq_slot_stats) */

typedef struct kuq_ctx kuq_ctx;

typedef struct kuq_config {
  int32_t device;                /* CUDA device ordinal */
  uint32_t n_slots;              /* batch slots (streams) for copy/compute overlap; 0 → 2 */
  uint32_t max_reads_per_batch;  /* slot capacity in reads; 0 → 1<<20 */
  uint64_t max_bases_per_batch;  /* slot capacity in bases (bytes of sequence); 0 → 160 MiB */
  uint64_t work_unit_size;       /* classify -u (classify.cpp:38,1106); 0 → 500000 */
  uint32_t hll_mode;             /* KUQ_HLL_* */
  uint32_t reserved0;
  uint64_t sparse_set_slots;     /* capacity (slots of 8 B) of the device set that backs the sparse HLL tier;
                                    0 → 1<<26 */
} kuq_config;

/* One run of the Kraken hit list: `code:count` (classify.cpp:826-861). code = taxid, 0 (miss) or KUQ_CODE_AMBIG */
typedef struct kuq_run {
  uint32_t code;
  uint32_t count;
} kuq_run;

/* Result of one batch; every pointer refers to pinned host memory owned by the slot and stays valid until the
 * slot is submitted again. */
typedef struct kuq_batch_result {
  uint32_t n_reads;
  uint32_t reserved0;
  const uint32_t *call;        /* [n_reads] taxon call (classify.cpp:965; 0 = unclassified) */
  const uint32_t *n_windows;   /* [n_reads] k-mer windows scanned (0 when the read is shorter than k, :913) */
  const uint32_t *run_start;   /* [n_reads] first run of the read in `runs` (undefined with KUQ_F_NO_RUNS) */
  const uint32_t *run_count;   /* [n_reads] number of runs (0 → the reference prints "0:0", :994-995) */
  const kuq_run *runs;         /* [n_runs] */
  uint64_t n_runs;
  const uint32_t *codes;       /* KUQ_F_WANT_CODES: code of window i of read r at codes[read_offsets[r] -
                                  read_offsets[0] + i]; NULL otherwise */
  uint64_t n_classified;       /* reads with call != 0 (total_classified, classify.cpp:541) */
  double kernel_ms;            /* device time of the batch's kernels (CUDA events on the slot's stream) */
} kuq_batch_result;

/* Device-side view of a slot's outputs after kuq_classify_device / kuq_resolve_device (HBM pointers). */
typedef struct kuq_device_result {
  const uint32_t *d_call;      /* [n_reads] raw taxids */
  const uint32_t *d_n_windows; /* [n_reads] */
  const uint32_t *d_codes;     /* per window, indexed like the bases; taxids / KUQ_CODE_AMBIG (KUQ_F_WANT_CODES) */
  const uint32_t *d_run_start;
  const uint32_t *d_run_count;
  const kuq_run *d_runs;
  const uint64_t *d_n_runs;    /* device scalar */
} kuq_device_result;

/* Raw device pointers to the per-taxon state, for the cross-GPU merge the caller performs with NCCL
 * (allreduce MAX over regs, SUM over the counters) when reads or DB ranges are spread over GPUs (SURVEY §8(e)). */
typedef struct kuq_state_ptrs {
  uint8_t *d_regs;             /* [n_sketch][4096] HLL registers, p = 12 (readcounts.hpp:40) */
  uint64_t regs_bytes;
  uint64_t *d_n_kmers;         /* [n_sketch] add_kmer count per taxon (readcounts.hpp:71-74) */
  uint64_t *d_n_reads;         /* [n_taxa]   incrementReadCount per taxon (readcounts.hpp:36) */
  uint8_t *d_dense_flag;       /* [n_sketch] 1 = some sketch of the taxon converted to dense (mode emulation) */
  uint32_t n_sketch;
  uint32_t n_taxa;
} kuq_state_ptrs;

void kuq_config_default(kuq_config *cfg);
int kuq_create(const kuq_config *cfg, kuq_ctx **ctx_out);
void kuq_destroy(kuq_ctx *ctx);
const char *kuq_strerror(int code);
const char *kuq_last_error(const kuq_ctx *ctx);
/* Build identification: "libkuq <version> sm_100a" */
const char *kuq_version(void);
/* Number of device ordinals [0, n) among which sm_100 devices were found (0 without a usable GPU). */
int kuq_device_count(void);

/* ---- database -------------------------------------------------------------------------------------------- */
/* Stage (a minimizer range of) the database into HBM.  kdb_image / idx_image are the bytes of database.kdb and
 * database.idx (mmap'ed files are fine).  Bins [bin_lo, bin_hi) are copied; bin_hi = 0 means "to the end".
 * Replaces a previously staged range (the `load_chunk` step of the chunked mode, krakendb.cpp:411-425). */
int kuq_stage_db(kuq_ctx *ctx, const void *kdb_image, uint64_t kdb_bytes, const void *idx_image,
                 uint64_t idx_bytes, uint64_t bin_lo, uint64_t bin_hi);
/* Adopt a database that already lives in HBM (records in on-disk layout, values still raw taxids; offsets =
 * the full 4^nt+1 table or, with bin_lo>0, the slice starting at bin_lo).  The buffers stay owned by the caller
 * but the record values are rewritten in place (taxid → dense id). */
int kuq_attach_db_device(kuq_ctx *ctx, void *d_pairs, uint64_t key_ct, const uint64_t *d_offsets, uint32_t k,
                         uint32_t nt, uint32_t idx_type, uint64_t bin_lo, uint64_t bin_hi);
/* Distinct taxids stored in the staged records with their record counts — what KrakenDB::count_taxons()
 * (krakendb.cpp:90-113) computes for database.kdb.counts.  Pass cap = 0 to query *n only. */
int kuq_db_taxids(kuq_ctx *ctx, uint32_t *taxid, uint64_t *count, uint32_t cap, uint32_t *n);
/* Optional: the taxids of ALL database records when only a range is staged (other chunks / other GPUs), so that
 * every participant numbers taxa identically.  Must precede the first classify/lookup call. */
int kuq_set_db_taxid_universe(kuq_ctx *ctx, const uint32_t *taxid, uint32_t n);
/* Several databases (`classify -d a -d b`): every k-mer takes the value of the FIRST database that holds the key,
 * even when that value is taxon 0 (classify.cpp:928-936).  With on != 0 the lookup calls report such a stored zero
 * as KUQ_CODE_FOUND_ZERO instead of 0, so that the caller's merge over databases can stop at it; the resolve calls
 * read KUQ_CODE_FOUND_ZERO as 0 in any case.  The caller stages the databases one after the other, runs
 * kuq_lookup_* against each, keeps the first non-zero code per position and hands the result to kuq_resolve_*. */
#define KUQ_CODE_FOUND_ZERO 0xFFFFFFFDu
int kuq_mark_zero_hits(kuq_ctx *ctx, int on);
/* Quick mode, `classify -q [-m min_hits]` (Quick_mode / Minimum_hit_count, classify.cpp:44-45; min_hits = 0 turns it
 * off).  Classification and resolve calls then skip resolve_tree: a read is called as soon as it has min_hits hits.
 *   stop_at_last_hit != 0 — the preloaded path (:943-944,963-964): the read ends at its min_hits-th hit; later
 *     k-mers are neither looked at nor counted; the call is that hit's taxon.  n_windows = windows visited.
 *   stop_at_last_hit == 0 — the -x path (:701-702,705-721,737-738): every k-mer is counted, hits stop counting at
 *     min_hits and the call is the taxon of the read's last unambiguous k-mer (0 if that one missed).
 * Either way run_count[r] (d_run_count) carries the "Q:<hits>" value of the Kraken line (:989-990), no runs are
 * produced (as with KUQ_F_NO_RUNS) and a read with fewer than min_hits hits stays unclassified. */
int kuq_set_quick_mode(kuq_ctx *ctx, uint32_t min_hits, int stop_at_last_hit);

/* ---- taxonomy: Parent_map (taxdb.hpp:383-398): taxid → parent taxid, 0 for the root / unknown parent --------- */
int kuq_set_taxonomy(kuq_ctx *ctx, const uint32_t *taxid, const uint32_t *parent_taxid, uint32_t n);

/* ---- classification, host buffers (the call a user makes) ----------------------------------------------- */
/* bases: concatenated sequences exactly as DNASequence::seq holds them (seqreader.hpp:27-32), read r =
 * bases[read_offsets[r] .. read_offsets[r+1]).  unit_id: work-unit id per read for the HLL mode rule, or NULL to
 * let the library cut units like process_file does (classify.cpp:514-520, continuing across batches).
 * kuq_classify_batch = submit + wait on slot 0.  A slot with an unread batch (kuq_submit_batch without its
 * kuq_wait_batch yet) refuses every batch call, host or device inputs, with KUQ_E_STATE until kuq_wait_batch. */
int kuq_classify_batch(kuq_ctx *ctx, const char *bases, const uint64_t *read_offsets, uint32_t n_reads,
                       const uint32_t *unit_id, uint32_t flags, kuq_batch_result *out);
int kuq_submit_batch(kuq_ctx *ctx, uint32_t slot, const char *bases, const uint64_t *read_offsets,
                     uint32_t n_reads, const uint32_t *unit_id, uint32_t flags);
int kuq_wait_batch(kuq_ctx *ctx, uint32_t slot, kuq_batch_result *out);
/* The two halves with host buffers, for databases staged range by range (classify -x, classify.cpp:566-791):
 * kuq_lookup_batch    = classify_sequence_with_db_chunk (:1014-1056): per-window DENSE taxon ids of the staged range
 *                       into codes_out (host; indexed like the bases; 0 = no hit in this range, KUQ_CODE_AMBIG for
 *                       ambiguous windows, 0 at positions without a window).  Ranges are merged by the caller with
 *                       an element-wise max (a key hits in at most one range, :447).
 * kuq_resolve_batch   = the final pass (:663-791): calls, hit lists and counters from the merged ids. */
int kuq_lookup_batch(kuq_ctx *ctx, const char *bases, const uint64_t *read_offsets, uint32_t n_reads,
                     uint32_t *codes_out, uint32_t *n_windows_out);
int kuq_resolve_batch(kuq_ctx *ctx, const char *bases, const uint64_t *read_offsets, uint32_t n_reads,
                      const uint32_t *codes_in, const uint32_t *unit_id, uint32_t flags, kuq_batch_result *out);
/* Pinned host memory for callers that want zero-copy staging of their batches. */
void *kuq_host_alloc(uint64_t bytes);
void kuq_host_free(void *p);

/* ---- classification, device buffers (inputs already in HBM) ---------------------------------------------- */
/* d_bases must be 16-byte aligned with 32 readable bytes of slack after the last base (TMA bulk loads fetch
 * whole 16-byte blocks); d_read_offsets (16-byte aligned, n_reads + 2 entries readable) are relative to d_bases.  Asynchronous on the slot's stream;
 * kuq_sync_slot() waits.  d_unit_id: work-unit id of every read (device array) — required with KUQ_HLL_PRELOAD
 * (the per-unit sketches of classify.cpp:525 are what the mode rule is about), NULL otherwise. */
int kuq_classify_device(kuq_ctx *ctx, uint32_t slot, const char *d_bases, const uint64_t *d_read_offsets,
                        uint32_t n_reads, uint64_t total_bases, const uint32_t *d_unit_id, uint32_t flags);
/* Stage 1 only (classify_sequence_with_db_chunk): per-window DENSE taxon ids of the staged DB range into
 * d_codes_out (indexed like the bases; 0 where the range has no hit; KUQ_CODE_AMBIG for ambiguous windows).
 * d_codes_out may be peer memory of another GPU (NVLink P2P stores) when only_hits != 0: then only hits are
 * written, so several ranges can be merged into one zero-initialised buffer without a reduction. */
int kuq_lookup_device(kuq_ctx *ctx, uint32_t slot, const char *d_bases, const uint64_t *d_read_offsets,
                      uint32_t n_reads, uint64_t total_bases, uint32_t *d_codes_out, uint32_t only_hits);
/* Stage 2 only: calls, hit lists and counters from merged per-window dense ids (the final pass of the chunked
 * mode, classify.cpp:663-791). */
int kuq_resolve_device(kuq_ctx *ctx, uint32_t slot, const char *d_bases, const uint64_t *d_read_offsets,
                       uint32_t n_reads, uint64_t total_bases, const uint32_t *d_codes_in,
                       const uint32_t *d_unit_id, uint32_t flags);
/* Fused lookup + scatter for a database sharded by minimizer range over the GPUs of one node: text positions
 * [base_bounds[j], base_bounds[j+1]) belong to the reads GPU j resolves; every hit of the staged range is stored
 * straight into d_codes_peers[j] (that GPU's zero-initialised buffer, mapped with kuq_ipc_open) over NVLink, so no
 * reduction is needed afterwards.  Synchronise the ranks (e.g. a barrier) before the owners call
 * kuq_resolve_device on their buffer. */
int kuq_lookup_device_peers(kuq_ctx *ctx, uint32_t slot, const char *d_bases, const uint64_t *d_read_offsets,
                            uint32_t n_reads, uint64_t total_bases, uint32_t *const *d_codes_peers,
                            const uint64_t *base_bounds, uint32_t n_peers);
/* Device memory that other ranks can map (cudaMalloc + CUDA IPC); handles are 64 opaque bytes. */
void *kuq_device_alloc(kuq_ctx *ctx, uint64_t bytes);
void kuq_device_free(kuq_ctx *ctx, void *p);
int kuq_device_memset(kuq_ctx *ctx, uint32_t slot, void *p, int value, uint64_t bytes);   /* async on the slot's stream */
int kuq_ipc_export(kuq_ctx *ctx, void *d_ptr, uint8_t handle64[64]);
int kuq_ipc_open(kuq_ctx *ctx, const uint8_t handle64[64], void **d_ptr_out);
int kuq_ipc_close(kuq_ctx *ctx, void *d_ptr);
int kuq_sync_slot(kuq_ctx *ctx, uint32_t slot);
/* Helpers for callers that keep their batches in HBM across several passes (a database streamed in ranges): an
 * asynchronous host → device copy on the slot's stream (pageable memory is fine), the free device memory, and the
 * second half of kuq_classify_batch for device inputs: after kuq_classify_device / kuq_resolve_device on `slot`,
 * kuq_collect_device_batch copies the batch's calls / window counts / hit lists to the slot's pinned host buffers,
 * waits, and fills `out` exactly like kuq_wait_batch. */
int kuq_copy_to_device(kuq_ctx *ctx, uint32_t slot, void *d_dst, const void *h_src, uint64_t bytes);
uint64_t kuq_device_free_bytes(kuq_ctx *ctx);
int kuq_collect_device_batch(kuq_ctx *ctx, uint32_t slot, kuq_batch_result *out);
int kuq_slot_device_result(kuq_ctx *ctx, uint32_t slot, kuq_device_result *out);
/* With KUQ_F_STATS: number of non-ambiguous windows looked up by the slot's last batch and the sum over them of
 * ceil(log2(bin size + 1)) — the textbook probe count SURVEY.md §8(d) defines the algorithmic bytes with. */
int kuq_slot_stats(kuq_ctx *ctx, uint32_t slot, uint64_t *n_lookups, uint64_t *sum_probes);
/* Turn KUQ_F_STATS on / off for every later call, including those that take no flags (kuq_lookup_device_peers). */
int kuq_set_stats(kuq_ctx *ctx, int on);
/* CUDA stream (cudaStream_t) of a slot, so callers can order their own work (e.g. NCCL) against it. */
void *kuq_slot_stream(kuq_ctx *ctx, uint32_t slot);
/* Number of kernels this context has launched so far (for bench.py's gpu_launches). */
uint64_t kuq_launch_count(const kuq_ctx *ctx);
/* Device time in ms of the most recent batch's kernels on `slot` (all stages). */
double kuq_last_kernel_ms(kuq_ctx *ctx, uint32_t slot);
/* Device time in ms of the three stages of the slot's last batch: ms3[0] k_scan (k-mers + minimizers),
 * ms3[1] k_lookup (index + bin search + HLL), ms3[2] k_resolve (hit lists, tree resolution, counters). */
int kuq_last_stage_ms(kuq_ctx *ctx, uint32_t slot, double *ms3);

/* ---- per-taxon results --------------------------------------------------------------------------------- */
/* End of input: closes the open work unit (the flush the reference performs when the reader runs dry). */
int kuq_finish(kuq_ctx *ctx);
/* Number of taxa with a non-zero counter, then their rows sorted by taxid: reads (readCount), kmers (kmerCount)
 * and unique (uniqueKmerCount = ertlCardinality under the configured mode rule, hyperloglogplus.cpp:722-753). */
int kuq_counts_size(kuq_ctx *ctx, uint32_t *n);
int kuq_read_counts(kuq_ctx *ctx, uint32_t *taxid, uint64_t *n_reads, uint64_t *n_kmers, uint64_t *unique,
                    uint8_t *is_sparse, uint32_t cap);
/* Clade roll-up of the report (TaxReport ctor, taxdb.hpp:956-973): sums the counters and merges the sketches
 * of the listed taxa; returns reads / kmers / unique of the union. */
int kuq_clade_counts(kuq_ctx *ctx, const uint32_t *taxids, uint32_t n, uint64_t *n_reads, uint64_t *n_kmers,
                     uint64_t *unique);
/* The same roll-up for many clades in one call: clade(taxids[i]) = that taxon and all its descendants in the taxonomy
 * given to kuq_set_taxonomy (what the TaxReport constructor builds for every node, taxdb.hpp:928-982).  Counters by
 * one pass up the tree; dense clades (a member's sketch is dense: register-wise max, hyperloglogplus.cpp:604-621) by
 * one launch per 8192 clades; sparse clades (union of the members' code sets, :600-603) from ONE sort of the sparse
 * tier's keys by (code, preorder of the taxon) — a subtree is a preorder interval, so its distinct codes are its
 * keys minus the adjacent equal-code pairs whose lowest common ancestor lies inside it.  Results equal
 * kuq_clade_counts() of the member list, clade by clade.  Unknown taxids and taxa without counted descendants give 0. */
int kuq_clade_counts_tree(kuq_ctx *ctx, const uint32_t *taxids, uint32_t n, uint64_t *n_reads, uint64_t *n_kmers,
                          uint64_t *unique);
/* The 4096 p=12 registers of one taxon (all zero if it received no k-mer). */
int kuq_get_registers(kuq_ctx *ctx, uint32_t taxid, uint8_t *regs4096);
int kuq_state_ptrs_get(kuq_ctx *ctx, kuq_state_ptrs *out);
/* Sparse tier across GPUs (replicas / shards with the exact HLL rule): export the (taxon, encoded hash) keys of the
 * taxa that are still sparse into d_keys_out (HBM; pass NULL / cap 0 to query *n), all-gather them, and import the
 * peers' keys; together with allreduce(MAX) on d_dense_flag / d_regs and SUM on the counters this is the merge
 * `taxon_counts[t] += ...` of classify.cpp:542-544 across processes. */
int kuq_sparse_export(kuq_ctx *ctx, uint64_t *d_keys_out, uint64_t cap, uint64_t *n);
/* The sparse tier's device set: capacity in slots, keys held, how often a harvest re-allocated it, and the device time
 * of the last harvest.  Hits reach the set lazily: the fused lookup only flags the database records it counted (the
 * free top bit of the key word) and kuq_finish / kuq_read_counts / kuq_sparse_export / a re-stage turn the flagged
 * records into (taxon, encoded hash) keys, growing the set first when it would pass a load factor of 0.7. */
int kuq_sparse_tier_info(kuq_ctx *ctx, uint64_t *slots, uint64_t *keys, uint64_t *times_grown, double *last_harvest_ms);
int kuq_sparse_import(kuq_ctx *ctx, const uint64_t *d_keys, uint64_t n);
/* ---- database sharded by minimizer range over the GPUs of a node (SURVEY.md §8(e).2) ------------------------------
 * Who counts: with kuq_set_shard_counting(on) the GPU that FINDS a hit does that hit's sketch work inside the lookup
 * half (kuq_lookup_device / kuq_lookup_device_peers): HLL register update and the record flag behind the sparse tier;
 * the resolve half on the GPU that owns the read then only adds the misses (taxon 0), the counters and the per-unit
 * bookkeeping.  Only valid when every looked-up window is counted exactly once (one database, no quick mode). */
int kuq_set_shard_counting(kuq_ctx *ctx, int on);
/* Step flags instead of host barriers.  A flag array is device memory of 8-byte counters that every peer has mapped
 * (kuq_device_alloc + kuq_ipc_export/open).  kuq_signal_peers: in stream order on the slot — i.e. after everything
 * queued before it, peer stores included, is complete — store `value` into d_flag_peers[j][my_index] for every
 * peer j (system-scope fence first).  kuq_wait_flags: in stream order, spin until d_flags[0..n) >= value; after
 * timeout_ms (0 → 20 s) it gives up and the next kuq_sync_slot returns KUQ_E_STATE instead of hanging the GPU. */
int kuq_signal_peers(kuq_ctx *ctx, uint32_t slot, uint64_t *const *d_flag_peers, uint32_t n_peers, uint32_t my_index,
                     uint64_t value);
int kuq_wait_flags(kuq_ctx *ctx, uint32_t slot, const uint64_t *d_flags, uint32_t n, uint64_t value, uint32_t timeout_ms);
/* End-of-run merge of the sparse tier across GPUs in O(keys / GPUs) per GPU (replicas or shards): the keys of the
 * still-sparse taxa are grouped by the GPU that owns their CODE (hash(code) % n_parts; counts[j] keys for part j,
 * parts stored back to back in d_keys_out; pass d_keys_out = NULL to get the counts only), exchanged with one
 * all-to-all, and kuq_sparse_replace makes the received keys this GPU's set (duplicates collapse there).  The export
 * covers the local set and the database records flagged since the last harvest; with a buffer it CONSUMES those
 * flags (their keys exist only in the buffer afterwards), so it must be followed by kuq_sparse_replace.  Every key
 * that can duplicate another — the same (taxon, code) from two GPUs, the same code under two taxa of a clade — lands
 * on one GPU, so global per-taxon numbers are SUMS: kuq_sparse_summary writes this GPU's rank histograms
 * ([n_sketch][64] uint32) and distinct counts ([n_sketch] uint32) to device buffers for an all-reduce(SUM), and
 * kuq_set_sparse_summary installs the sums, which kuq_read_counts then reports (until the next batch).  Clade
 * unions of several sparse taxa: sum kuq_clade_partial's hist64 over the GPUs and evaluate kuq_ertl_sparse /
 * kuq_ertl_dense_hist (is_dense is the same on every GPU once dense flags and registers were all-reduced). */
int kuq_sparse_export_partitioned(kuq_ctx *ctx, uint32_t n_parts, uint64_t *d_keys_out, uint64_t cap, uint64_t *counts);
/* the same with the buffer sized and allocated by the library after its counting pass (release with kuq_device_free) */
int kuq_sparse_export_partitioned_alloc(kuq_ctx *ctx, uint32_t n_parts, uint64_t **d_keys_out, uint64_t *counts);
int kuq_sparse_replace(kuq_ctx *ctx, const uint64_t *d_keys, uint64_t n);
int kuq_sparse_summary(kuq_ctx *ctx, uint32_t *d_hist_out, uint32_t *d_distinct_out);
int kuq_set_sparse_summary(kuq_ctx *ctx, const uint32_t *d_hist, const uint32_t *d_distinct);
int kuq_clade_partial(kuq_ctx *ctx, const uint32_t *taxids, uint32_t n, uint64_t *n_reads, uint64_t *n_kmers, int *is_dense,
                      uint32_t *hist64);
uint64_t kuq_ertl_sparse(const uint32_t *hist64, uint64_t n_observed);
uint64_t kuq_ertl_dense_hist(const uint32_t *hist64, uint64_t n_observed);
/* Stage 1 alone (KmerScanner + canonical_representation + bin_key, krakenutil.cpp:239-282, krakendb.cpp:200-246) on
 * device buffers: canonical k-mer and minimizer bin of every window, indexed like the bases (window i of read r at
 * d_read_offsets[r] + i; bins: 0xFFFFFFFE = ambiguous window, 0xFFFFFFFF = no window at this position).  Needs no
 * staged database; used by the database-build tools and the synthetic-workload generator. */
int kuq_scan_device(kuq_ctx *ctx, uint32_t slot, uint32_t k, uint32_t nt, uint32_t idx_type, const char *d_bases,
                    const uint64_t *d_read_offsets, uint32_t n_reads, uint64_t total_bases, uint64_t *d_canon_out,
                    uint32_t *d_bins_out);

/* ---- a database larger than HBM, streamed range by range (classify -x / --preload-size, krakendb.cpp:411-526) ------
 * kuq_stage_db replaces the staged range synchronously.  The stream calls keep TWO device buffers and a copy stream, so
 * the next minimizer range travels over PCIe while the lookups of the current one run:
 *     kuq_set_db_taxid_universe(all taxids of the database); kuq_set_taxonomy(...);
 *     kuq_stream_open(k, nt, idx_type, max records / bins of a range)
 *     kuq_stream_load(0, range 0)
 *     for r in ranges:  kuq_stream_use(r & 1);  kuq_stream_load((r + 1) & 1, range r + 1);      // order matters
 *                       kuq_lookup_device(... only_hits = 1 ...) for every batch, ids merged in the caller's buffers
 *     kuq_resolve_device(...) for every batch                                  // the final pass (classify.cpp:663-791)
 * host_records = the range's records (12 bytes each, raw taxids, as in database.kdb), host_offsets = the bin_hi -
 * bin_lo + 1 cumulative ABSOLUTE record offsets of its bins (a slice of database.idx); both should be pinned
 * (kuq_host_alloc / kuq_host_register) or the copy will not overlap.  kuq_stream_load waits, on the device, for the
 * work queued on the slots so far (the users of the buffer it overwrites), never for the host.  Record values are
 * rewritten to dense ids on arrival; kuq_stream_check reports a taxid outside the declared universe. */
int kuq_stream_open(kuq_ctx *ctx, uint32_t k, uint32_t nt, uint32_t idx_type, uint64_t max_records, uint64_t max_bins);
int kuq_stream_load(kuq_ctx *ctx, uint32_t buf, const void *host_records, uint64_t n_records, const uint64_t *host_offsets,
                    uint64_t bin_lo, uint64_t bin_hi);
int kuq_stream_use(kuq_ctx *ctx, uint32_t buf);
int kuq_stream_check(kuq_ctx *ctx);
/* Pin / unpin caller memory (e.g. an mmap'ed database.kdb) for asynchronous copies. */
int kuq_host_register(void *p, uint64_t bytes);
int kuq_host_unregister(void *p);

/* Several GPUs in one process (what the drop-in `classify` does when it sees more than one device: every GPU holds the
 * database, batches go round-robin): fold the per-taxon state of `src` into `dst` — counters add, registers max, dense
 * anywhere = dense, sparse-tier keys united (classify.cpp:542-544 across devices; cudaMemcpyPeer, no NCCL).  Both
 * contexts must have been given the same database and taxonomy.  `src` keeps its state. */
int kuq_merge_into(kuq_ctx *dst, kuq_ctx *src);
/* In one process the GPUs of a sharded database need no CUDA IPC: after kuq_enable_peer_access(ctx, peer) the device
 * pointers of `peer` (kuq_device_alloc) can be handed to kuq_lookup_device_peers / kuq_signal_peers of `ctx` as they are. */
int kuq_enable_peer_access(kuq_ctx *ctx, kuq_ctx *peer);

/* Dense id ↔ taxid tables (n_taxa entries) for callers that exchange dense ids between GPUs. */
int kuq_dense_taxids(kuq_ctx *ctx, uint32_t *taxid_of_dense, uint32_t cap, uint32_t *n);
int kuq_reset_counts(kuq_ctx *ctx);

/* Host-side estimator (no device needed): ertlCardinality over 4096 dense registers (hyperloglogplus.cpp:
 * 730-752) — exported so bindings and tests can call the exact code the report path uses. */
uint64_t kuq_ertl_dense(const uint8_t *regs4096, uint64_t n_observed);

/* ---- measurement aid: the random-access roofline of SURVEY.md §8(d) ------------------------------------------- */
/* Random 32-byte-sector gather ceiling of the device's HBM: a kernel with k_lookup's launch shape (256 threads,
 * 8 CTAs per SM) issues independent loads at hashed sector addresses of a freshly allocated buffer of buffer_bytes
 * (use several GB: far beyond L2) until n_sectors_to_read sectors were touched; bytes_per_access = 32 (whole
 * sector) or 8 (one word of it — the sector is still what HBM moves).  Best of three timed launches after one
 * warm-up, CUDA events.  Returns sectors/s (in 1e9) and the same as GB/s of 32-byte sectors.  Needs no context. */
int kuq_random_gather_peak(int device, uint64_t buffer_bytes, uint64_t n_sectors_to_read, uint32_t bytes_per_access,
                           double *gsectors_per_s, double *gbytes_per_s, double *kernel_ms);

/* Record-layout / search-shape experiment for the bin search (kmer_query, krakendb.cpp:250-321) — measurement aid.
 * Transcodes the staged 12-byte records once into 8-byte minimizer-relative records (the 16 bases outside the bin's
 * minimizer + minimizer position / orientation + 24-bit dense taxon; k = 31, m = 15 only) and times a lookup-only
 * kernel over the windows the LAST batch of `slot` left in the slot's scratch (text positions [0, n_positions), i.e.
 * a batch whose first read starts at offset 0), for both layouts x {4, 8, 16}-ary narrowing x final scans of <= 8 /
 * <= 16 records.  Every variant's per-window dense ids are compared with the ids the product's k_lookup wrote for
 * that batch (mismatches[] must be 0).  On the product's layout and search it also times other launch SHAPES:
 * shape 0 = thread per window with the next window's scratch prefetched (the product's), 1 = the product's own
 * k_lookup<MODE_LOOKUP> in the same harness, 2 / 3 = the next window's index entry prefetched too (8 / 6 CTAs per SM),
 * 4 / 5 / 6 = two windows per thread in lock step (8 / 6 / 4 CTAs per SM), 7 = four windows per thread (4 CTAs),
 * 8 = the product's k_lookup<MODE_LOOKUP> with its launch-uniform switches compiled out, 9 / 10 = the product's
 * k_lookup<MODE_FUSED> (search + register update) with / without those switches — these two run only on a
 * KUQ_HLL_DENSE_ONLY context (they count the batch's windows into its sketches once per launch; use a throwaway
 * context) and are reported as 0 ms otherwise; 11 = shape 0 with the narrowing step as an if / else-if chain instead
 * of a count of the pivots <= key, 12 = shape 0 fed through the product's parameter block.
 * Needs 8 bytes per record + 4 bytes per position of free device memory.
 * Times: CUDA events on the slot's stream, one warm-up launch then `reps` timed ones per variant. */
#define KUQ_LAYOUT_VARIANTS 22
typedef struct kuq_layout_result {
  uint64_t n_records, n_positions;
  uint64_t n_windows;                         /* windows looked up in the staged range */
  uint64_t sum_probes;                        /* sum of ceil(log2(bin size + 1)) over them (SURVEY.md §8(d)'s P) */
  uint64_t bin_class[6];                      /* windows whose bin holds <= 8, <= 16, <= 64, <= 256, <= 1024, more records */
  double transcode_ms;
  uint32_t n_variants;
  uint32_t rec_bytes[KUQ_LAYOUT_VARIANTS], arity[KUQ_LAYOUT_VARIANTS], window[KUQ_LAYOUT_VARIANTS];
  uint32_t shape[KUQ_LAYOUT_VARIANTS];        /* see below */
  double best_ms[KUQ_LAYOUT_VARIANTS], mean_ms[KUQ_LAYOUT_VARIANTS];
  uint64_t mismatches[KUQ_LAYOUT_VARIANTS];
} kuq_layout_result;
int kuq_layout_experiment(kuq_ctx *ctx, uint32_t slot, uint64_t n_positions, uint32_t reps, kuq_layout_result *out);

/* ---- database build (SURVEY.md §8 f4) ---------------------------------------------------------------------- */
/* db_sort [-z] -n nt (db_sort.cpp:41-116 + KrakenDB::make_index, krakendb.cpp:118-148): unsorted Jellyfish-style
 * image → database.kdb image (kdb_out: header + key_ct * (key_len + 4) bytes) and KRAKIX2 index image (idx_out:
 * 8 + 8 * (4^nt + 1) bytes).  Needs no context.  err (optional) receives a message on failure. */
int kuq_db_sort(int device, const void *jdb_image, uint64_t jdb_bytes, uint32_t nt, int zero_vals, void *kdb_out,
                void *idx_out, char *err, uint64_t err_cap);
/* set_lcas (set_lcas.cpp:429-476): for every k-mer of the library pieces that the staged database holds,
 * value = lca(taxid of the piece, value).  A piece is a stretch of one library sequence; consecutive pieces of a
 * sequence overlap by k-1 bases (the reference's SKIP_LEN pieces, :363-364).  The context needs the database
 * (kuq_stage_db, whole) and the taxonomy (kuq_set_taxonomy); every taxid must be in the taxonomy — the reference
 * skips other sequences (:336-341) and so must the caller.  *n_missing = k-mers of this batch the database lacks (set_lcas
 * without -x stops there, :441-443).  After the first call the context cannot classify any more.
 * flags: KUQ_LCA_FORCE_CONTAMINANT = set_lcas -T (what build_db.sh always passes: a value of 32630 'synthetic
 * construct' / 81077 'artificial sequences' sticks and a piece with such a taxid overwrites instead of taking the LCA,
 * :462-474; between those two taxids the first to arrive wins, so one batch may hold pieces of only one of them),
 * KUQ_LCA_RESET = -R (the value becomes 0, :458-459). */
#define KUQ_LCA_FORCE_CONTAMINANT 1u
#define KUQ_LCA_RESET 2u
int kuq_set_lcas_batch(kuq_ctx *ctx, const char *bases, const uint64_t *piece_offsets, uint32_t n_pieces,
                       const uint32_t *taxid, uint32_t flags, uint64_t *n_missing);
/* Copy the record values of the staged database (as taxids) into the value fields of a host database.kdb image
 * with the same records — what set_lcas leaves in the memory-mapped file. */
int kuq_export_db_values(kuq_ctx *ctx, void *kdb_image, uint64_t kdb_bytes);

#ifdef __cplusplus
}
#endif
#endif /* KUQ_H */
