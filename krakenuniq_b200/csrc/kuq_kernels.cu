// kuq_kernels.cu — see kuq_kernels.cuh for the map from kernel stages to reference functions.
// Design history: round 1 first fused all stages into one persistent warp-per-read kernel; at 128 registers it ran
// at 25 % occupancy and was bound by exposed latency (profiles/README.md), so the path is now three kernels that
// each keep a small register footprint and hand windows over through HBM scratch (12 B per window, streamed).
#include "kuq_kernels.cuh"

namespace kuq {

// ------------------------------------------------------------------------------------------------------
// small PTX wrappers: mbarrier + 1-D TMA bulk copy (global → shared), sm_90+/sm_100a
// ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
// cp.async.bulk: one thread moves `bytes` (multiple of 16, 16-byte aligned on both sides) and signals `bar`.
__device__ __forceinline__ void tma_load_1d(void *smem_dst, const void *gmem_src, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// ------------------------------------------------------------------------------------------------------
// bit arithmetic
// ------------------------------------------------------------------------------------------------------
// KrakenDB::reverse_complement (krakendb.cpp:218-225): reverse the 2-bit groups, complement, shift down.
__device__ __forceinline__ uint64_t revcomp64(uint64_t x, uint32_t n) {
  x = __brevll(x);                                                              // reverses bits inside groups too
  x = ((x >> 1) & 0x5555555555555555ull) | ((x & 0x5555555555555555ull) << 1);  // ... so swap them back
  return (~x) >> (64 - 2 * n);
}
__device__ __forceinline__ uint32_t revcomp32(uint32_t x, uint32_t n) {   // n <= 15
  x = __brev(x);
  x = ((x >> 1) & 0x55555555u) | ((x & 0x55555555u) << 1);
  return (~x) >> (32 - 2 * n);
}
// murmurhash3_finalizer (hyperloglogplus.cpp:830-838)
__device__ __forceinline__ uint64_t fmix64(uint64_t key) {
  key += 1;
  key ^= key >> 33;
  key *= 0xff51afd7ed558ccdull;
  key ^= key >> 33;
  key *= 0xc4ceb9fe1a85ec53ull;
  key ^= key >> 33;
  return key;
}

// 12-byte records are only 4-byte aligned: a key is two 32-bit loads.
__device__ __forceinline__ uint64_t load_key(const uint8_t *pairs, uint64_t pos, uint64_t key_mask) {
  const uint32_t *p = reinterpret_cast<const uint32_t *>(pairs + pos * 12);
  uint32_t lo = __ldg(p), hi = __ldg(p + 1);
  return (((uint64_t)hi << 32) | lo) & key_mask;                                // krakendb.cpp:283-284
}
__device__ __forceinline__ uint32_t load_val(const uint8_t *pairs, uint64_t pos) {
  return __ldg(reinterpret_cast<const uint32_t *>(pairs + pos * 12) + 2);
}

// HyperLogLogPlusMinus::insert, dense branch (hyperloglogplus.cpp:514-521): M[idx] = max(M[idx], rank).
// Registers are bytes; a byte-wide max is a CAS on the enclosing word, reached only when the plain load says the
// register would grow (after warm-up almost never: P[grow] ~ 1/n).  A stale load can only be too small, which
// costs a redundant CAS, never a lost update.
__device__ __forceinline__ void hll_update(uint8_t *regs, uint32_t taxon, uint64_t hash) {
  uint32_t idx = (uint32_t)(hash >> (64 - HLL_P));
  uint64_t rest = hash << HLL_P;
  uint32_t rank = rest ? (uint32_t)__clzll((long long)rest) + 1 : (64 - HLL_P + 1);   // getRank, :140-147
  uint8_t *reg = regs + (size_t)taxon * HLL_M + idx;
  if (*reinterpret_cast<volatile uint8_t *>(reg) >= rank) return;
  uint32_t *word = reinterpret_cast<uint32_t *>(reinterpret_cast<uintptr_t>(reg) & ~(uintptr_t)3);
  uint32_t shift = (uint32_t)(reinterpret_cast<uintptr_t>(reg) & 3) * 8;
  uint32_t old = *reinterpret_cast<volatile uint32_t *>(word);
  while (((old >> shift) & 0xFF) < rank) {
    uint32_t upd = (old & ~(0xFFu << shift)) | (rank << shift);
    uint32_t prev = atomicCAS(word, old, upd);
    if (prev == old) break;
    old = prev;
  }
}

// encodeHashIn32Bit(h, pPrime=25, p=12), hyperloglogplus.cpp:181-204
__device__ __forceinline__ uint32_t encode_hash32(uint64_t hash) {
  uint32_t idx = (uint32_t)((hash >> 39) << 7);
  if ((idx << 12) == 0) {
    uint64_t rest = hash << 25;
    uint32_t add_rank = rest ? (uint32_t)__clzll((long long)rest) + 1 : 40;
    return idx | (add_rank << 1) | 1;
  }
  return idx;
}

__device__ __forceinline__ uint64_t mix64(uint64_t x) {   // table hash for the device sets (not reference arithmetic)
  x ^= x >> 31;
  x *= 0x7fb5d329728ea185ull;
  x ^= x >> 27;
  x *= 0x81dadef4bc2dd44dull;
  x ^= x >> 33;
  return x;
}

// Insert into the (taxon, code) set behind the sparse HLL tier.  Returns 1 when the key is new, 0 when it was
// there already, -1 when the table is saturated (the host turns that into KUQ_E_CAPACITY).
__device__ __forceinline__ int sparse_insert(const SparseSet &s, uint32_t taxon, uint32_t code) {
  unsigned long long key = ((unsigned long long)(taxon + 1) << 32) | code;
  uint64_t slot = mix64(key) & s.mask;
  for (uint32_t probe = 0; probe < 512; probe++) {
    unsigned long long cur = __ldcg(s.slots + slot);          // L2 is where the CAS of other threads lands
    if (cur == key) return 0;
    if (cur == 0) {
      unsigned long long prev = atomicCAS(s.slots + slot, 0ull, key);
      if (prev == 0) return 1;
      if (prev == key) return 0;
    }
    slot = (slot + 1) & s.mask;
  }
  return -1;
}

// ------------------------------------------------------------------------------------------------------
// taxonomy walks on the flattened parent array
// ------------------------------------------------------------------------------------------------------
// lca(), krakenutil.cpp:90-118, in dense ids.  Dense id 1 is ALWAYS the node of taxid 1 (the reference's
// hard-wired root: loops run `while (a > 1)`), dense id 0 is "no taxon".  depth[] counts the steps of a node's
// parent chain until it ends (at 0, or at node 1), so both chains can be levelled first.
__device__ uint32_t lca_dense(const TaxView &t, uint32_t a, uint32_t b) {
  if (a == 0 || b == 0) return a ? a : b;
  uint32_t da = a <= 1 ? 0 : t.depth[a], db = b <= 1 ? 0 : t.depth[b];
  while (da > db) { a = t.parent[a]; da--; }
  while (db > da) { b = t.parent[b]; db--; }
  while (a != b && a > 1 && b > 1) {
    a = t.parent[a];
    b = t.parent[b];
  }
  return (a == b && a > 1) ? a : 1u;
}

// ------------------------------------------------------------------------------------------------------
// one read, one warp
// ------------------------------------------------------------------------------------------------------
struct Block64 {         // 32 bases: 2-bit codes, first base in bits 63:62; amb bit l = base l is not ACGT
  uint64_t codes;
  uint32_t amb;
  uint32_t mark;         // bit l = a window ENDS at base l (only for cleaned reads, see clean_read)
  bool skip;             // the block holds a '\n' / '\r' (not set for cleaned reads)
};

// Convert 32 characters (lane = position) — krakenutil.cpp:253-273.  Positions >= len read as ambiguous.
__device__ __forceinline__ Block64 load_block(const char *seq, uint32_t len, uint32_t blk, uint32_t lane, bool marks) {
  uint32_t pos = blk * 32 + lane;
  uint32_t c = pos < len ? (uint32_t)(uint8_t)seq[pos] : (uint32_t)'N';
  uint32_t mk = 0;
  if (marks) { mk = c >> 7; c &= 0x7Fu; }
  uint32_t uc = c & 0xDFu;                                  // case-insensitive, :254-264
  bool ok = (uc == 'A') | (uc == 'C') | (uc == 'G') | (uc == 'T');
  uint32_t code = ok ? (((c >> 1) ^ (c >> 2)) & 3u) : 0u;   // A=0 C=1 G=2 T=3
  uint32_t sh = 2 * (15 - (lane & 15));
  uint32_t hi = __reduce_or_sync(0xFFFFFFFFu, lane < 16 ? code << sh : 0u);
  uint32_t lo = __reduce_or_sync(0xFFFFFFFFu, lane >= 16 ? code << sh : 0u);
  Block64 b;
  b.codes = ((uint64_t)hi << 32) | lo;
  b.amb = __ballot_sync(0xFFFFFFFFu, !ok);
  b.mark = marks ? __ballot_sync(0xFFFFFFFFu, mk != 0) : 0u;
  // a skipped character is first of all a non-ACGT one: blocks without any (the common case) need no second vote
  b.skip = !marks && b.amb != 0 && __any_sync(0xFFFFFFFFu, !ok && (c == '\n' || c == '\r'));
  return b;
}

constexpr uint32_t BIN_NONE = 0xFFFFFFFFu;    // scratch marker: no window at this position
constexpr uint32_t BIN_AMBIG = 0xFFFFFFFEu;   // scratch marker: window with a non-ACGT base

// Stage 1 for one read (one warp, one slot of 32 windows at a time): canonical k-mer and minimizer bin of every
// window → scratch.  Pure ALU + shuffles, no dependent memory access.
// FAST = the (k, m) = (31, 15) of every published KrakenUniq database, with the window arithmetic as constants.
// Returns false (having possibly written a prefix of the read's windows, all of which the caller rewrites) when it
// meets a skipped character: the read then goes through clean_read.
template <bool FAST>
__device__ bool scan_read(const Params &p, uint32_t r, const char *seq, uint32_t len, uint32_t raw_len,
                          uint64_t out_base, uint32_t lane, bool marks) {
  const DbView &db = p.db;
  const uint32_t k = FAST ? 31u : db.k, nt = FAST ? 15u : db.nt;
  const uint32_t n_mini = FAST ? 17u : db.n_mini;
  // candidate windows; every one of them is a scanner window unless the read was cleaned (marks), in which case
  // only the marked ones are (the scanner drops a window per skipped character, see clean_read)
  const uint32_t nwin = len >= k ? len - k + 1 : 0;           // classify.cpp:913-914
  uint32_t n_out = 0;                                         // windows emitted so far
  if (nwin > 0) {
    Block64 A = load_block(seq, len, 0, lane, marks);
    if (A.skip) return false;
    const uint32_t nslots = (nwin + 31) / 32;
    for (uint32_t s = 0; s < nslots; s++) {
      Block64 B = load_block(seq, len, s + 1, lane, marks);
      if (B.skip) return false;
      const uint32_t i = s * 32 + lane;
      bool valid = i < nwin;
      if (marks) valid = valid && (((((uint64_t)B.mark << 32) | A.mark) >> (lane + k - 1)) & 1);
      const uint32_t vmask = __ballot_sync(0xFFFFFFFFu, valid);
      const uint32_t oi = n_out + __popc(vmask & ((1u << lane) - 1));   // output slot of this window
      n_out += __popc(vmask);
      // k-mer of window i: bases [i, i+k) of the 128-bit string A:B
      uint64_t hi = lane ? (A.codes << (2 * lane)) | (B.codes >> (64 - 2 * lane)) : A.codes;
      uint64_t kmer = hi >> (64 - 2 * k);
      uint64_t amb64 = ((uint64_t)B.amb << 32) | A.amb;
      bool amb = ((amb64 >> lane) & ((1ull << k) - 1)) != 0;  // any non-ACGT base in the window, :275,280-282
      uint64_t rc = revcomp64(kmer, k);                       // canonical k-mer (krakendb.cpp:238-246)
      uint64_t canon = kmer < rc ? kmer : rc;
      // minimizer = min over the k-nt+1 nt-mers of (xor_mask ^ canonical(nt-mer)) (krakendb.cpp:200-215).
      // Candidate of position q (0..63 relative to the slot): lane holds q = lane (m0) and q = 32+lane (m1).
      uint32_t f0 = (uint32_t)(hi >> (64 - 2 * nt));
      uint32_t r0 = revcomp32(f0, nt);
      uint32_t m0 = db.xor_mask ^ (f0 < r0 ? f0 : r0);
      uint32_t f1 = (uint32_t)((B.codes << (2 * lane)) >> (64 - 2 * nt));
      uint32_t r1 = revcomp32(f1, nt);
      uint32_t m1 = db.xor_mask ^ (f1 < r1 ? f1 : r1);
      // sliding-window minimum of width n_mini by doubling: after the loop m0 holds min over [q, q+n_mini)
      uint32_t w = 1;
#pragma unroll
      for (int step = 0; step < 5; step++) {                  // n_mini <= 31 → at most 4 doublings
        if (2 * w > n_mini) break;
        uint32_t src = (lane + w) & 31;
        uint32_t x0 = __shfl_sync(0xFFFFFFFFu, m0, src), x1 = __shfl_sync(0xFFFFFFFFu, m1, src);
        bool wrap = lane + w >= 32;
        m0 = min(m0, wrap ? x1 : x0);
        m1 = min(m1, wrap ? 0xFFFFFFFFu : x1);
        w *= 2;
      }
      if (w < n_mini) {                                       // [q, q+n_mini) = [q, q+w) U [q+n_mini-w, q+n_mini)
        uint32_t d = n_mini - w;
        uint32_t src = (lane + d) & 31;
        uint32_t x0 = __shfl_sync(0xFFFFFFFFu, m0, src), x1 = __shfl_sync(0xFFFFFFFFu, m1, src);
        m0 = min(m0, lane + d >= 32 ? x1 : x0);
      }
      if (valid) {
        p.bins[out_base + oi] = amb ? BIN_AMBIG : m0;
        p.canon[out_base + oi] = canon;
      }
      A = B;
    }
  }
  // positions of the read's text that carry no window
  for (uint32_t q = n_out + lane; q < raw_len; q += 32) p.bins[out_base + q] = BIN_NONE;
  if (lane == 0) p.n_windows[r] = n_out;
  return true;
}

// A read that contains '\n' / '\r' (CRLF input, SURVEY App. A9).  KmerScanner::next_kmer (krakenutil.cpp:239-278)
// "skips" such a character by undoing the loaded_nt increment (:265-269), but the base that follows a skipped
// character is then loaded WITHOUT being counted (skip_pos, :246-247), and every further skipped character of a
// run decrements loaded_nt once more.  Net effect: each skipped character makes the scanner swallow one extra
// base, i.e. one k-mer window is never produced.  If the text ends while a call is still loading, the scanner
// reads the string terminator as an ambiguous base and produces one last (ambiguous) window.
// The warp's lane 0 replays that automaton once (rare path) and writes the cleaned bases to scratch, setting bit 7
// of the base each produced window ENDS at; process_read then only keeps the marked windows.
__device__ uint32_t clean_read(const char *seq, uint32_t len, char *dst, uint32_t k, uint32_t lane) {
  uint32_t n = 0;
  if (lane == 0) {
    int loaded = 0;
    bool skipflag = false;
    int64_t last_emit = -1;
    for (uint32_t i = 0; i < len; i++) {
      char c = seq[i];
      if (c == '\n' || c == '\r') {
        if (skipflag) loaded--;
        skipflag = true;
      } else {
        uint8_t o = ((uint8_t)c & 0x80) ? (uint8_t)'N' : (uint8_t)c;   // bit 7 is the window mark
        if (!skipflag) {
          loaded++;
          if (loaded == (int)k) { o |= 0x80; loaded = (int)k - 1; last_emit = i; }
        }
        skipflag = false;
        dst[n++] = (char)o;
      }
    }
    if (len >= k && last_emit + 1 < (int64_t)len) {     // a call is still loading: one last, ambiguous window
      uint32_t target = n + 1 > k ? n + 1 : k;          // <= len because at least one character was skipped
      while (n < target) dst[n++] = 'N';
      dst[n - 1] = (char)((uint8_t)'N' | 0x80);
    }
  }
  n = __shfl_sync(0xFFFFFFFFu, n, 0);
  __syncwarp();
  return n;
}

// ------------------------------------------------------------------------------------------------------
// the persistent kernel
// ------------------------------------------------------------------------------------------------------
struct __align__(16) SharedState {
  uint64_t off[N_STAGES][CHUNK_READS + 2];   // read offsets of the chunk (bulk-copied with the bases)
  uint64_t bar[N_STAGES];
  uint64_t a0[N_STAGES];                     // global byte offset the stage's text starts at
  uint32_t chunk[N_STAGES];
  uint32_t staged[N_STAGES];
  uint32_t next_read[N_STAGES];              // warps take the reads of a chunk from this counter
};

// Stage 1: persistent CTAs; one thread pulls the next chunk of reads (offsets slice + text) into shared memory
// with TMA bulk copies while the warps still scan the previous chunk.
__global__ void __launch_bounds__(CTA_THREADS, 4) k_scan(const __grid_constant__ Params p) {
  extern __shared__ __align__(128) uint8_t smem[];
  uint8_t *stage_buf = smem;                                                   // N_STAGES x STAGE_BYTES
  SharedState *ss = reinterpret_cast<SharedState *>(smem + N_STAGES * STAGE_BYTES);
  const uint32_t tid = threadIdx.x, lane = tid & 31;

  auto fetch = [&](uint32_t st) {
    uint32_t c = atomicAdd(p.chunk_counter, 1u);
    ss->chunk[st] = c;
    ss->staged[st] = 0;
    ss->next_read[st] = 0;
    if (c < p.n_chunks) {
      const uint32_t r0 = c * CHUNK_READS, r1 = min(r0 + CHUNK_READS, p.n_reads);
      const uint32_t n_off = (r1 - r0 + 2) & ~1u;                  // even count → multiple of 16 bytes
      const uint64_t b0 = p.offsets[r0], b1 = p.offsets[r1];
      const uint64_t a0 = b0 & ~15ull, a1 = (b1 + 15) & ~15ull;
      ss->a0[st] = a0;
      uint32_t bytes = n_off * 8;
      const bool text = a1 - a0 <= (uint64_t)STAGE_BYTES && a1 > a0;
      if (text) bytes += (uint32_t)(a1 - a0);
      mbar_expect_tx(&ss->bar[st], bytes);
      tma_load_1d(&ss->off[st][0], p.offsets + r0, n_off * 8, &ss->bar[st]);
      if (text) {
        tma_load_1d(stage_buf + st * STAGE_BYTES, p.bases + a0, (uint32_t)(a1 - a0), &ss->bar[st]);
        ss->staged[st] = 1;
      }
    }
  };

  if (tid == 0) {
    for (int s = 0; s < N_STAGES; s++) mbar_init(&ss->bar[s], 1);
    mbar_fence_init();
    fetch(0);
  }
  __syncthreads();
  uint32_t phase[N_STAGES] = {0, 0};
  const bool fast = p.db.k == 31 && p.db.nt == 15;
  for (uint32_t it = 0;; it++) {
    const uint32_t st = it & 1;
    const uint32_t c = ss->chunk[st];
    if (c >= p.n_chunks) break;
    if (tid == 0) fetch(st ^ 1);        // the other stage was released by the barrier that ended the last round
    const bool staged = ss->staged[st] != 0;
    const uint64_t a0 = ss->a0[st];
    mbar_wait(&ss->bar[st], phase[st]);
    phase[st] ^= 1;
    const uint32_t r0 = c * CHUNK_READS, r1 = min(r0 + CHUNK_READS, p.n_reads);
    for (;;) {
      uint32_t q = 0;
      if (lane == 0) q = atomicAdd(&ss->next_read[st], 1u);
      q = __shfl_sync(0xFFFFFFFFu, q, 0);
      const uint32_t r = r0 + q;
      if (r >= r1) break;
      const uint64_t b0 = ss->off[st][q], b1 = ss->off[st][q + 1];
      const uint32_t raw_len = (uint32_t)(b1 - b0);
      uint32_t len = raw_len;
      const char *seq = staged ? reinterpret_cast<const char *>(stage_buf + st * STAGE_BYTES + (b0 - a0))
                               : p.bases + b0;
      const bool done = fast ? scan_read<true>(p, r, seq, len, raw_len, b0, lane, false)
                             : scan_read<false>(p, r, seq, len, raw_len, b0, lane, false);
      if (!done) {   // the read holds '\n' / '\r' (rare: CRLF input): replay the scanner, then rescan the cleaned copy
        len = clean_read(seq, len, p.clean + b0, p.db.k, lane);
        scan_read<false>(p, r, p.clean + b0, len, raw_len, b0, lane, true);
      }
    }
    __syncthreads();
  }
}

// Stage 2: one thread per text position.  Index fetch (KrakenDBIndex::at, krakendb.cpp:586-593), bin search
// (kmer_query, :280-299: 4-ary narrowing while the bin is large, then a scan of <= 8 records) and — unless the
// lookups belong to one range of a sharded database — the HLL insert of ReadCounts::add_kmer (classify.cpp:939).
// Threads of a warp hold consecutive windows of a read: windows that share a minimizer read the same index
// sector and the same pivots, which the load unit coalesces.
// LEAN = the launch uses none of: probe statistics (KUQ_F_STATS), F_FOUND_ZERO, F_SHARD_COUNTING, hits-only
// output, peer buffers.  Those are launch-uniform run-time switches; compiled out, the common path of the fused kernel
// is a third shorter and measurably faster (profiles/layout_probe_r02.log: the search alone 1.87 -> 1.62 ms).
template <int MODE, bool LEAN>
__global__ void __launch_bounds__(256, 8) k_lookup(const __grid_constant__ Params p) {
  const DbView &db = p.db;
  const uint32_t flags = LEAN ? (p.flags & KUQ_F_NO_COUNTS) : p.flags;
  const uint32_t only_hits = LEAN ? 0u : p.only_hits;
  const uint32_t n_peers = LEAN ? 0u : p.n_peers;
  const uint32_t hi_mask = (uint32_t)(db.key_mask >> 32);
  const bool counting = (MODE == MODE_FUSED) && !(flags & KUQ_F_NO_COUNTS);
  // hits of the fused path reach the sparse tier through the record flag (see below); dense-only / exact runs have
  // no sparse tier
  // F_SHARD_COUNTING (database sharded over GPUs, one database): the GPU that FINDS a hit owns its sketch work —
  // register update and record flag happen in the lookup half, and the resolve half (on the GPU that owns the read)
  // only adds the misses (taxon 0).  Valid because every looked-up window is counted exactly once in that layout.
  const bool shard_counting = (flags & F_SHARD_COUNTING) != 0;
  const bool mark_seen = (counting || (MODE == MODE_LOOKUP && shard_counting)) && p.hll_mode <= KUQ_HLL_CHUNKED;
  // only the text of this call's reads (the scratch beyond it may hold windows of an earlier call on the slot)
  const uint64_t g_begin = p.offsets[0], g_end = p.offsets[p.n_reads];
  // the scratch of the NEXT position of this thread is fetched while the current window is searched: the grid-stride
  // loop would otherwise start every window with an exposed (streaming, but still ~1 us) load
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  uint64_t g = g_begin + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t bin_n = g < g_end ? __ldg(p.bins + g) : BIN_NONE;
  uint64_t canon_n = g < g_end ? __ldg(p.canon + g) : 0ull;
  for (; g < g_end; g += stride) {
    const uint32_t bin = bin_n;
    const uint64_t canon = canon_n;
    if (g + stride < g_end) { bin_n = __ldg(p.bins + g + stride); canon_n = __ldg(p.canon + g + stride); }
    if (bin == BIN_NONE) continue;
    if (bin == BIN_AMBIG) {
      if (!only_hits && !(MODE == MODE_LOOKUP && n_peers)) p.codes_dense[g] = AMBIG;
      continue;
    }
    uint32_t taxon = 0;
    if (MODE == MODE_RESOLVE) {
      taxon = p.codes_in[g];                                 // merged dense ids of all database ranges
      if (taxon == FOUND_ZERO) taxon = 0;                    // a stored taxon 0 counts like a miss from here on
    } else if (bin >= db.bin_lo && bin < db.bin_hi) {
      const uint64_t *o = db.offsets + (bin - db.bin_lo);
      const uint64_t o0 = __ldg(o), o1 = __ldg(o + 1);
      uint64_t lo = o0 - db.rec_base;
      uint32_t n = (uint32_t)(o1 - o0);
      if (flags & KUQ_F_STATS) {   // measurement aid: algorithmic probe count of SURVEY.md §8(d)
        atomicAdd(p.stats, 1ull);
        atomicAdd(p.stats + 1, (unsigned long long)(n ? 32 - __clz(n) : 0));
      }
      while (n > (uint32_t)SEARCH_WINDOW) {
        const uint32_t q = n >> 2;
        const uint64_t k1 = load_key(db.pairs, lo + q, db.key_mask);
        const uint64_t k2 = load_key(db.pairs, lo + 2 * q, db.key_mask);
        const uint64_t k3 = load_key(db.pairs, lo + 3 * q, db.key_mask);
        // pivots <= the key: the quarter that can hold it (branch-free; the lanes of a warp disagree here all the time)
        const uint32_t c = (canon >= k1 ? 1u : 0u) + (canon >= k2 ? 1u : 0u) + (canon >= k3 ? 1u : 0u);
        lo += (uint64_t)c * q;
        n = (c == 3u) ? n - 3 * q : q;
      }
      if (n) {
        // compare the low key words of the window first, confirm the (rare) matches on the high word
        const uint32_t *b = reinterpret_cast<const uint32_t *>(db.pairs + lo * 12);
        const uint32_t clo = (uint32_t)canon, chi = (uint32_t)(canon >> 32);
        uint32_t lw[SEARCH_WINDOW];
#pragma unroll
        for (int t = 0; t < SEARCH_WINDOW; t++) lw[t] = ((uint32_t)t < n) ? __ldg(b + 3 * t) : 0;
        uint32_t m = 0;
#pragma unroll
        for (int t = 0; t < SEARCH_WINDOW; t++) m |= ((uint32_t)t < n && lw[t] == clo) ? (1u << t) : 0u;
        while (m) {
          const int t = __ffs(m) - 1;
          m &= m - 1;
          const uint32_t hiw = __ldg(b + 3 * t + 1);
          if ((hiw & hi_mask) == chi) {
            taxon = __ldg(b + 3 * t + 2);                        // value = dense id
            if (MODE == MODE_LOOKUP && taxon == 0 && (flags & F_FOUND_ZERO)) taxon = FOUND_ZERO;
            // Sparse HLL tier of a hit (hyperloglogplus.cpp:499-512): the (taxon, encoded hash) pair is a function
            // of the RECORD, so instead of probing a hash set per window the record itself is flagged in the free
            // top bit of its key word — the sector is in L1/L2 already, the flag costs no DRAM read, and only the
            // first sighting of a record issues the atomic.  k_harvest_seen turns flagged records into set keys
            // once per run.  A stale (non-coherent) load can only miss a flag another thread just set: the
            // atomicOr is then redundant, never wrong.
            if (mark_seen && taxon != 0 && taxon != FOUND_ZERO && !(hiw & SEEN_BIT))
              atomicOr(const_cast<uint32_t *>(b + 3 * t + 1), SEEN_BIT);
            m = 0;
          }
        }
      }
    } else if (flags & KUQ_F_STATS) {
      atomicAdd(p.stats + 3, 1ull);                          // a window of another range: nothing fetched here
    }
    // only_hits: several DB ranges (GPUs) write their hits into one zero-initialised buffer, possibly over
    // NVLink; a key lives in exactly one range (classify.cpp:447), so no two writers touch the same word.
    if (MODE == MODE_LOOKUP && n_peers) {
      // fused lookup + scatter: the hit goes to the GPU that resolves this read, as a peer store over NVLink
      if (taxon != 0) {
        uint32_t j = 0;
        while (j + 1 < n_peers && g >= p.peer_bounds[j + 1]) j++;
        p.peer_codes[j][g] = taxon;
      }
    } else if (MODE == MODE_RESOLVE || !only_hits || taxon != 0) {
      p.codes_dense[g] = taxon;
    }
    if (MODE == MODE_LOOKUP && shard_counting) {
      if (taxon != 0 && taxon != FOUND_ZERO) hll_update(p.regs, taxon, fmix64(canon));
    } else if ((counting || (MODE == MODE_RESOLVE && !(flags & KUQ_F_NO_COUNTS))) && !(MODE == MODE_RESOLVE && shard_counting && taxon != 0)) {
      const uint64_t h = fmix64(canon);
      hll_update(p.regs, taxon, h);
      // direct set insert: misses (taxon 0 has no record to flag) and the resolve half, which only sees merged ids
      if (p.hll_mode != KUQ_HLL_DENSE_ONLY && !(mark_seen && taxon != 0) && !p.dense_flag[taxon]) {
        const int ins = sparse_insert(p.sparse, taxon, encode_hash32(h));
        if (ins > 0) atomicAdd(p.sparse.distinct + taxon, 1u);
        else if (ins < 0) atomicExch(p.error_flag, 4u);       // set saturated
      }
    }
  }
}

// ---- per-batch (unit, taxon) map ----------------------------------------------------------------------------
__device__ __forceinline__ uint32_t umap_slot(const UnitMap &u, uint32_t unit, uint32_t taxon, bool insert) {
  const unsigned long long key = ((unsigned long long)(unit + 1) << 32) | taxon;
  uint32_t slot = (uint32_t)mix64(key) & u.mask;
  for (uint32_t probe = 0; probe <= u.mask; probe++) {
    unsigned long long cur = *reinterpret_cast<volatile unsigned long long *>(u.keys + slot);
    if (cur == key) return slot;
    if (cur == 0) {
      if (!insert) return 0xFFFFFFFFu;
      unsigned long long prev = atomicCAS(u.keys + slot, 0ull, key);
      if (prev == 0 || prev == key) return slot;
    }
    slot = (slot + 1) & u.mask;
  }
  return 0xFFFFFFFFu;
}

// Reads that hit more than 32 distinct taxa (long reads, contigs): the hit list moves to a hash table in HBM taken from
// a per-batch pool ({taxon+1 << 32 | count, score} per entry).  Same arithmetic as the register path, just slower.
struct OverflowPool {
  unsigned long long *mem;        // 2 words per entry
  unsigned long long *cursor;     // entries handed out
  uint64_t capacity;              // entries
};

__device__ uint32_t resolve_overflow(const Params &p, const OverflowPool &pool, const uint32_t *codes_src, uint64_t out_base,
                                     uint32_t nwin, uint32_t unit, bool counting, bool units, uint32_t lane) {
  // capacity: next power of two >= 2 * (upper bound of distinct taxa); distinct taxa <= windows
  // (and <= taxa that own a sketch: only database values can be hits)
  const uint32_t most = min(nwin, p.tax.n_sketch);
  uint32_t cap = 64;
  while (cap < 2 * most) cap <<= 1;
  unsigned long long start = 0;
  if (lane == 0) start = atomicAdd(pool.cursor, (unsigned long long)cap);
  start = __shfl_sync(0xFFFFFFFFu, start, 0);
  if (start + cap > pool.capacity) {
    if (lane == 0) atomicExch(p.error_flag, 1u);
    return 0;
  }
  unsigned long long *tab = pool.mem + 2 * start;
  for (uint32_t i = lane; i < cap; i += 32) { tab[2 * i] = 0; tab[2 * i + 1] = 0; }
  __syncwarp();
  auto find = [&](uint32_t t) -> int {              // slot of taxon t or -1
    uint32_t s = (uint32_t)mix64(t) & (cap - 1);
    for (uint32_t probe = 0; probe < cap; probe++) {
      const unsigned long long e = *reinterpret_cast<volatile unsigned long long *>(tab + 2 * s);
      if (e == 0) return -1;
      if ((uint32_t)(e >> 32) == t + 1) return (int)s;
      s = (s + 1) & (cap - 1);
    }
    return -1;
  };
  // hit_counts[taxon]++ over all windows
  for (uint32_t i = lane; i < nwin; i += 32) {
    const uint32_t t = codes_src[out_base + i];
    if (t == AMBIG || t == 0) continue;
    uint32_t s = (uint32_t)mix64(t) & (cap - 1);
    for (;;) {
      unsigned long long e = *reinterpret_cast<volatile unsigned long long *>(tab + 2 * s);
      if (e == 0) {
        e = atomicCAS(tab + 2 * s, 0ull, ((unsigned long long)(t + 1) << 32) | 1ull);
        if (e == 0) break;
      }
      if ((uint32_t)(e >> 32) == t + 1) { atomicAdd(tab + 2 * s, 1ull); break; }
      s = (s + 1) & (cap - 1);
    }
  }
  __syncwarp();
  // score(t) = sum of hit counts along t's root path (krakenutil.cpp:156-177)
  uint32_t best = 0;
  for (uint32_t s = lane; s < cap; s += 32) {
    const unsigned long long e = tab[2 * s];
    if (!e) continue;
    const uint32_t t = (uint32_t)(e >> 32) - 1, c = (uint32_t)e;
    if (counting) {
      atomicAdd(p.n_kmers + t, (unsigned long long)c);
      if (units) {
        const uint32_t row = unit - p.unit_id[0];
        if (row < p.units.direct_rows) {
          atomicAdd(p.units.direct + (size_t)row * p.tax.n_sketch + t, c);
        } else {
          uint32_t sl = umap_slot(p.units, unit, t, true);
          if (sl == 0xFFFFFFFFu) atomicExch(p.error_flag, 2u);
          else atomicAdd(p.units.inserts + sl, c);
        }
      }
    }
    uint32_t score = 0;
    for (uint32_t node = t; node; node = __ldg(p.tax.parent + node)) {
      int q = find(node);
      if (q >= 0) score += (uint32_t)tab[2 * q];
    }
    tab[2 * s + 1] = score;
    best = max(best, score);
  }
  best = __reduce_max_sync(0xFFFFFFFFu, best);
  __syncwarp();
  if (best == 0) return 0;
  // ties → LCA of all tied taxa, folded in ascending taxid order (std::set iteration, krakenutil.cpp:190-196)
  uint32_t acc = 0;
  unsigned long long last = 0;          // raw taxid + 1 of the last folded taxon
  for (;;) {
    unsigned long long mn = ~0ull;      // smallest (raw+1) << 32 | dense among the tied entries above `last`
    for (uint32_t s = lane; s < cap; s += 32) {
      const unsigned long long e = tab[2 * s];
      if (!e || (uint32_t)tab[2 * s + 1] != best) continue;
      const uint32_t t = (uint32_t)(e >> 32) - 1;
      const unsigned long long r1 = (unsigned long long)__ldg(p.tax.raw + t) + 1;
      if (r1 > last) mn = min(mn, (r1 << 32) | t);
    }
    for (int o = 16; o; o >>= 1) mn = min(mn, __shfl_xor_sync(0xFFFFFFFFu, mn, o));
    if (mn == ~0ull) break;
    const uint32_t t = (uint32_t)mn;
    acc = acc ? lca_dense(p.tax, acc, t) : t;
    last = mn >> 32;
  }
  return acc;
}

// Stage 3: one warp per read.  hit_counts (classify.cpp:941-942), resolve_tree / lca (krakenutil.cpp:90-118,
// 149-200), the per-taxon counters (classify.cpp:939,968) and the run-length encoded hit list (:826-861).
constexpr int RUN_BUF = 96;      // runs buffered per warp before they are flushed to global memory
constexpr uint32_t RUN_BLOCK = 256;   // run slots a warp takes from the global cursor at a time

// QUICK (classify -q): no resolve_tree; hits = min(#hits, quick_min) goes to run_count[] ("Q:hits", :989-990) and the
// call is the taxon of the last unambiguous window once quick_min hits were seen (:963-964 after k_quick_cut ended
// the read at that hit; :705-721,737-738 on the -x path, where the last window of the whole read decides).
template <bool QUICK>
__global__ void __launch_bounds__(256, 4) k_resolve(const __grid_constant__ Params p) {
  __shared__ uint2 s_runs[CTA_WARPS][RUN_BUF];
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t warps_total = gridDim.x * CTA_WARPS;
  const bool counting = !(p.flags & KUQ_F_NO_COUNTS);
  const bool want_runs = !(p.flags & KUQ_F_NO_RUNS);
  const uint32_t *codes_src = p.codes_dense;
  // Same-address atomics serialise in L2 (about one per few cycles): a million reads per batch must not each hit
  // the run cursor, n_kmers[0] and n_reads[0].  Each warp therefore allocates run slots in blocks of RUN_BLOCK
  // and keeps the hot counters in registers until it is done.
  uint32_t blk_next = 0, blk_end = 0;                           // this warp's block of run slots
  uint32_t acc_miss = 0, acc_unclassified = 0, acc_classified = 0;
  uint32_t unit_cur = 0xFFFFFFFFu, unit_miss = 0;               // misses of the current work unit, not yet booked
  const bool units = counting && p.hll_mode == KUQ_HLL_PRELOAD && p.unit_id;
  const uint32_t unit_row0 = units ? p.unit_id[0] : 0u;
  auto book_unit = [&](uint32_t unit, uint32_t taxon, uint32_t cnt) {          // N(unit, taxon) += cnt
    const uint32_t row = unit - unit_row0;
    if (row < p.units.direct_rows) {
      atomicAdd(p.units.direct + (size_t)row * p.tax.n_sketch + taxon, cnt);
    } else {
      const uint32_t sl = umap_slot(p.units, unit, taxon, true);
      if (sl == 0xFFFFFFFFu) atomicExch(p.error_flag, 2u);
      else atomicAdd(p.units.inserts + sl, cnt);
    }
  };
  auto flush_unit = [&]() {
    if (lane == 0 && unit_miss) book_unit(unit_cur, 0, unit_miss);
    unit_miss = 0;
  };
  // each warp takes a contiguous range of reads: consecutive reads share their work unit and their run block
  const uint32_t per_warp = (p.n_reads + warps_total - 1) / warps_total;
  const uint32_t r_begin = (blockIdx.x * CTA_WARPS + warp) * per_warp;
  const uint32_t r_end = min(r_begin + per_warp, p.n_reads);
  // A warp works through its reads one after the other and every read is a chain of dependent loads (offset →
  // codes → taxonomy → counters), so the kernel is latency bound (round 1: 36 % warps active, 6 % DRAM).  The loads
  // that do not depend on the read's outcome are therefore issued one read ahead: while read r is resolved, the
  // codes of read r+1 (first PRE_SLOTS x 32 windows) and the offset / window count / unit of read r+2 are in flight.
  constexpr int PRE_SLOTS = 4;
  const bool want_codes = (p.flags & KUQ_F_WANT_CODES) != 0;
  uint64_t base_a = 0, base_b = 0;                              // read r, read r+1
  uint32_t nwin_a = 0, nwin_b = 0, unit_a = 0, unit_b = 0;
  uint32_t pre[PRE_SLOTS];
#pragma unroll
  for (int j = 0; j < PRE_SLOTS; j++) pre[j] = 0;
  if (r_begin < r_end) {
    base_a = p.offsets[r_begin]; nwin_a = p.n_windows[r_begin];
    if (units) unit_a = p.unit_id[r_begin];
#pragma unroll
    for (int j = 0; j < PRE_SLOTS; j++) { const uint32_t i = j * 32 + lane; pre[j] = i < nwin_a ? codes_src[base_a + i] : 0u; }
  }
  if (r_begin + 1 < r_end) {
    base_b = p.offsets[r_begin + 1]; nwin_b = p.n_windows[r_begin + 1];
    if (units) unit_b = p.unit_id[r_begin + 1];
  }
  for (uint32_t r = r_begin; r < r_end; r++) {
    const uint64_t out_base = base_a;
    const uint32_t nwin = nwin_a;
    const uint32_t unit = unit_a;
    uint32_t cur[PRE_SLOTS];
#pragma unroll
    for (int j = 0; j < PRE_SLOTS; j++) cur[j] = pre[j];
    base_a = base_b; nwin_a = nwin_b; unit_a = unit_b;
    if (r + 1 < r_end) {
#pragma unroll
      for (int j = 0; j < PRE_SLOTS; j++) { const uint32_t i = j * 32 + lane; pre[j] = i < nwin_a ? codes_src[base_a + i] : 0u; }
    }
    if (r + 2 < r_end) {
      base_b = p.offsets[r + 2]; nwin_b = p.n_windows[r + 2];
      if (units) unit_b = p.unit_id[r + 2];
    }
    uint32_t my_t = 0, my_c = 0;                                // hit list: lane j holds entry j (dense id, count)
    uint32_t n_hits = 0, n_miss = 0, n_runs = 0;
    uint32_t carry_code = 0;
    bool overflow = false;
    uint32_t q_hits = 0, q_last = 0;                            // QUICK: hits seen, taxon of the last unambiguous window
    const uint32_t nslots = (nwin + 31) / 32;
    // one slot of 32 windows; c = dense id of the lane's window, 0 = miss, AMBIG.  Runs of the hit list break where
    // the DENSE code changes (dense id <-> taxid is one to one); taxids are looked up per run when the list is flushed
    auto do_slot = [&](uint32_t s, uint32_t c) {
      const uint32_t i = s * 32 + lane;
      const bool valid = i < nwin;
      const bool amb = valid && c == AMBIG;
      const bool look = valid && !amb;
      const uint32_t taxon = look ? c : 0;
      const uint32_t out_code = amb ? AMBIG : taxon;
      if (want_codes && valid) p.codes[out_base + i] = amb ? AMBIG : (taxon ? __ldg(p.tax.raw + taxon) : 0u);
      // runs of the hit list
      uint32_t prev = __shfl_up_sync(0xFFFFFFFFu, out_code, 1);
      if (lane == 0) prev = carry_code;
      const bool brk = valid && (i == 0 || out_code != prev);
      const uint32_t bm = __ballot_sync(0xFFFFFFFFu, brk);
      if (want_runs && brk) {
        const uint32_t idx = n_runs + __popc(bm & ((1u << lane) - 1));
        if (idx < RUN_BUF) s_runs[warp][idx] = make_uint2(out_code, i);   // (dense code, start); lengths at flush
      }
      n_runs += __popc(bm);
      carry_code = __shfl_sync(0xFFFFFFFFu, out_code, 31);
      // hit_counts[taxon]++, aggregated per distinct taxon of the slot
      n_miss += __popc(__ballot_sync(0xFFFFFFFFu, look && taxon == 0));
      uint32_t rem = __ballot_sync(0xFFFFFFFFu, look && taxon != 0);
      if (QUICK) {
        q_hits += __popc(rem);
        const uint32_t lm = __ballot_sync(0xFFFFFFFFu, look);
        if (lm) q_last = __shfl_sync(0xFFFFFFFFu, taxon, 31 - __clz(lm));
      }
      while (rem) {
        const int ldr = __ffs(rem) - 1;
        const uint32_t t = __shfl_sync(0xFFFFFFFFu, taxon, ldr);
        const uint32_t same = __ballot_sync(0xFFFFFFFFu, look && taxon == t) & rem;
        const uint32_t cnt = __popc(same);
        rem &= ~same;
        const uint32_t pos = __ballot_sync(0xFFFFFFFFu, lane < n_hits && my_t == t);
        if (pos) {
          if (lane == (uint32_t)(__ffs(pos) - 1)) my_c += cnt;
        } else if (n_hits < 32) {
          if (lane == n_hits) { my_t = t; my_c = cnt; }
          n_hits++;
        } else {
          overflow = true;
        }
      }
    };
#pragma unroll
    for (int j = 0; j < PRE_SLOTS; j++)
      if ((uint32_t)j < nslots) do_slot((uint32_t)j, cur[j]);
    for (uint32_t s = PRE_SLOTS; s < nslots; s++) {
      const uint32_t i = s * 32 + lane;
      do_slot(s, i < nwin ? codes_src[out_base + i] : 0u);
    }

    // ---- resolve_tree (krakenutil.cpp:149-200) ------------------------------------------------------------
    uint32_t call = 0;
    if (overflow) {
      OverflowPool pool{p.ovf_mem, p.ovf_cursor, p.ovf_capacity};
      call = resolve_overflow(p, pool, codes_src, out_base, nwin, unit, counting, units, lane);
      n_hits = 0;                                               // counters were booked from the table
    } else if (!QUICK && n_hits == 1) {
      call = __shfl_sync(0xFFFFFFFFu, my_t, 0);                 // a single hit taxon is its own best path
    } else if (!QUICK && n_hits > 1) {
      // score(t) = sum of hit counts along t's root path (:156-177); lane j walks entry j
      uint32_t node = lane < n_hits ? my_t : 0;
      uint32_t score = 0;
      while (__any_sync(0xFFFFFFFFu, node != 0)) {
        for (uint32_t q = 0; q < n_hits; q++) {
          uint32_t tq = __shfl_sync(0xFFFFFFFFu, my_t, q);
          uint32_t cq = __shfl_sync(0xFFFFFFFFu, my_c, q);
          if (node == tq) score += cq;
        }
        if (node) node = __ldg(p.tax.parent + node);
      }
      uint32_t best = __reduce_max_sync(0xFFFFFFFFu, score);
      uint32_t tied = __ballot_sync(0xFFFFFFFFu, lane < n_hits && score == best);
      if (__popc(tied) == 1) {
        call = __shfl_sync(0xFFFFFFFFu, my_t, __ffs(tied) - 1);
      } else {
        // ties → LCA of all tied taxa, folded in ascending taxid order (std::set iteration, :190-196)
        uint32_t raw = (tied >> lane) & 1 ? __ldg(p.tax.raw + my_t) : 0xFFFFFFFFu;
        uint32_t acc = 0;
        uint32_t left = tied;
        while (left) {
          uint32_t cand = (left >> lane) & 1 ? raw : 0xFFFFFFFFu;
          uint32_t mn = __reduce_min_sync(0xFFFFFFFFu, cand);
          uint32_t who = __ballot_sync(0xFFFFFFFFu, cand == mn && ((left >> lane) & 1));
          int src = __ffs(who) - 1;
          uint32_t t = __shfl_sync(0xFFFFFFFFu, my_t, src);
          acc = acc ? lca_dense(p.tax, acc, t) : t;             // all lanes compute the same walk
          left &= ~(1u << src);
        }
        call = acc;
      }
    }
    if (QUICK) {
      const uint32_t hits = min(q_hits, p.quick_min);
      call = hits >= p.quick_min ? q_last : 0;
      if (lane == 0) p.run_count[r] = hits;
    }
    const uint32_t call_raw = call ? __ldg(p.tax.raw + call) : 0;
    if (lane == 0) p.call[r] = call_raw;
    // ---- counters: n_kmers per hit taxon (+ misses on taxon 0), n_reads of the call (classify.cpp:939,968) ---
    if (units) {
      // inserts per (work unit, taxon): the necessary condition for a per-unit sketch to convert
      if (unit != unit_cur) { flush_unit(); unit_cur = unit; }
      unit_miss += n_miss;
      if (lane < n_hits) book_unit(unit, my_t, my_c);
    }
    if (counting) {
      if (lane < n_hits) atomicAdd(p.n_kmers + my_t, (unsigned long long)my_c);
      acc_miss += n_miss;
      if (call) {
        acc_classified++;
        if (lane == 0) atomicAdd(p.n_reads_ctr + call, 1ull);
      } else {
        acc_unclassified++;
      }
    }
    // ---- run-length encoded hit list ----------------------------------------------------------------------
    if (want_runs) {
      uint32_t start = 0;
      if (lane == 0) {
        if (n_runs > blk_end - blk_next) {                      // take a fresh block (the old tail stays a hole)
          const uint32_t take = n_runs > RUN_BLOCK ? n_runs : RUN_BLOCK;
          const unsigned long long got = atomicAdd(p.run_cursor, (unsigned long long)take);
          if (got + take > p.runs_capacity) {                   // run buffer exhausted: report, write nothing more
            atomicExch(p.error_flag, 5u);
            blk_next = blk_end = 0xFFFFFFFFu;
          } else {
            blk_next = (uint32_t)got;
            blk_end = blk_next + take;
          }
        }
        start = blk_next;
        if (blk_next != 0xFFFFFFFFu) blk_next += n_runs;
        p.run_start[r] = start;
        p.run_count[r] = n_runs;
      }
      start = __shfl_sync(0xFFFFFFFFu, start, 0);
      __syncwarp();
      if (start == 0xFFFFFFFFu) {
        // no room (KUQ_E_CAPACITY on the host side)
      } else if (n_runs <= RUN_BUF) {
        for (uint32_t j = lane; j < n_runs; j += 32) {
          const uint2 a = s_runs[warp][j];
          const uint32_t end = j + 1 < n_runs ? s_runs[warp][j + 1].y : nwin;
          const uint32_t code = (a.x == AMBIG || a.x == 0) ? a.x : __ldg(p.tax.raw + a.x);
          p.runs[start + j] = make_uint2(code, end - a.y);
        }
      } else {
        // long hit list (long read): recompute from the codes, walking the slots backwards so that each run
        // knows where the next one starts
        uint32_t next_start = nwin, later = 0;
        for (int s = (int)nslots - 1; s >= 0; s--) {
          uint32_t i = (uint32_t)s * 32 + lane;
          bool valid = i < nwin;
          auto code_at = [&](uint32_t w) {
            uint32_t c = codes_src[out_base + w];
            return c == AMBIG ? AMBIG : (c ? __ldg(p.tax.raw + c) : 0u);
          };
          uint32_t c = valid ? code_at(i) : 0;
          uint32_t prev = __shfl_up_sync(0xFFFFFFFFu, c, 1);
          if (lane == 0) prev = (s > 0) ? code_at(i - 1) : 0;
          bool brk = valid && (i == 0 || c != prev);
          uint32_t bm = __ballot_sync(0xFFFFFFFFu, brk);
          if (brk) {
            uint32_t after = lane == 31 ? 0u : (bm >> (lane + 1));
            uint32_t end = after ? (uint32_t)s * 32 + lane + (uint32_t)__ffs(after) : next_start;
            uint32_t idx = n_runs - later - (uint32_t)__popc(bm >> lane);
            p.runs[start + idx] = make_uint2(c, end - i);
          }
          if (bm) next_start = (uint32_t)s * 32 + (uint32_t)__ffs(bm) - 1;
          later += __popc(bm);
        }
      }
      __syncwarp();
    }
  }
  if (units) flush_unit();
  if (counting && lane == 0) {
    if (acc_miss) atomicAdd(p.n_kmers, (unsigned long long)acc_miss);
    if (acc_unclassified) atomicAdd(p.n_reads_ctr, (unsigned long long)acc_unclassified);
    if (acc_classified) atomicAdd(p.n_classified, (unsigned long long)acc_classified);
  }
}

// ---- HLL mode rule (SURVEY.md App. C) ------------------------------------------------------------------------
__global__ void k_unit_mark(const __grid_constant__ Params p) {
  const UnitMap &u = p.units;
  // dense table first: a pair with >= 1025 inserts moves to the hash map, where the candidate bookkeeping lives
  if (u.direct_rows) {
    const uint32_t row0 = p.unit_id[0];
    const uint64_t n = (uint64_t)u.direct_rows * p.tax.n_sketch;
    for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (uint64_t)gridDim.x * blockDim.x) {
      const uint32_t cnt = u.direct[e];
      if (cnt < 1025u) continue;
      const uint32_t taxon = (uint32_t)(e % p.tax.n_sketch), row = (uint32_t)(e / p.tax.n_sketch);
      if (p.dense_flag[taxon]) continue;
      const uint32_t sl = umap_slot(u, row0 + row, taxon, true);
      if (sl == 0xFFFFFFFFu) { atomicExch(p.error_flag, 2u); continue; }
      u.inserts[sl] = cnt;
      u.cand[sl] = 1;
      u.taxon_cand[taxon] = 1;
      atomicAdd(u.n_cand, 1u);
    }
  }
  for (uint32_t s = blockIdx.x * blockDim.x + threadIdx.x; s <= u.mask; s += gridDim.x * blockDim.x) {
    const unsigned long long key = u.keys[s];
    if (!key) continue;
    const uint32_t taxon = (uint32_t)key;
    if (u.inserts[s] >= 1025u && !p.dense_flag[taxon] && !u.cand[s]) {
      u.cand[s] = 1;
      u.taxon_cand[taxon] = 1;
      atomicAdd(u.n_cand, 1u);
    }
  }
}

// warp per read; only windows of candidate (unit, taxon) pairs do any work
__global__ void __launch_bounds__(256) k_unit_distinct(const __grid_constant__ Params p) {
  const UnitMap &u = p.units;
  if (*reinterpret_cast<volatile uint32_t *>(u.n_cand) == 0) return;
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t warps_total = gridDim.x * (blockDim.x >> 5);
  for (uint32_t r = blockIdx.x * (blockDim.x >> 5) + warp; r < p.n_reads; r += warps_total) {
    const uint64_t base = p.offsets[r];
    const uint32_t nwin = p.n_windows[r];
    const uint32_t unit = p.unit_id[r];
    for (uint32_t i = lane; i < nwin; i += 32) {
      const uint32_t t = p.codes_dense[base + i];
      if (t == AMBIG || !u.taxon_cand[t]) continue;
      const uint32_t sl = umap_slot(u, unit, t, false);
      if (sl == 0xFFFFFFFFu || !u.cand[sl]) continue;
      atomicMax(u.last + sl, ((unsigned long long)r << 32) | i);
      if (*reinterpret_cast<volatile uint32_t *>(u.distinct + sl) >= 1025u) continue;   // decided already
      const uint32_t code = encode_hash32(fmix64(p.canon[base + i]));
      const unsigned long long key = ((unsigned long long)(sl + 1) << 32) | code;
      uint32_t q = (uint32_t)mix64(key) & u.set_mask;
      for (uint32_t probe = 0; probe <= u.set_mask; probe++) {
        unsigned long long cur = *reinterpret_cast<volatile unsigned long long *>(u.set_keys + q);
        if (cur == 0) {
          cur = atomicCAS(u.set_keys + q, 0ull, key);
          if (cur == 0) { atomicAdd(u.distinct + sl, 1u); cur = key; }
        }
        if (cur == key) { atomicAdd(u.set_count + q, 1u); break; }
        q = (q + 1) & u.set_mask;
        if (probe == u.set_mask) atomicExch(p.error_flag, 3u);
      }
    }
  }
}

// A (unit, taxon) sketch receiving inserts x_1..x_N converts iff D >= 1025, or D == 1024 and the 1024th distinct
// code arrives before the last insert (SURVEY.md §7.3): i.e. the last insert repeats a code seen earlier.
__global__ void k_unit_apply(const __grid_constant__ Params p) {
  const UnitMap &u = p.units;
  if (*reinterpret_cast<volatile uint32_t *>(u.n_cand) == 0) return;
  for (uint32_t s = blockIdx.x * blockDim.x + threadIdx.x; s <= u.mask; s += gridDim.x * blockDim.x) {
    if (!u.cand[s]) continue;
    const uint32_t taxon = (uint32_t)u.keys[s];
    const uint32_t d = u.distinct[s];
    bool conv = d >= 1025u;
    if (!conv && d == 1024u) {
      const unsigned long long lp = u.last[s];
      const uint32_t r = (uint32_t)(lp >> 32), i = (uint32_t)lp;
      const uint32_t code = encode_hash32(fmix64(p.canon[p.offsets[r] + i]));
      const unsigned long long key = ((unsigned long long)(s + 1) << 32) | code;
      uint32_t q = (uint32_t)mix64(key) & u.set_mask;
      for (uint32_t probe = 0; probe <= u.set_mask; probe++) {
        unsigned long long cur = u.set_keys[q];
        if (cur == key) { conv = u.set_count[q] >= 2u; break; }
        if (cur == 0) break;
        q = (q + 1) & u.set_mask;
      }
    }
    if (conv) p.dense_flag[taxon] = 1;
  }
}

// one launch instead of nine memsets: empty the per-batch (unit, taxon) map and its distinct-code set
__global__ void __launch_bounds__(256) k_unit_clear(UnitMap u, uint32_t n_sketch) {
  const uint64_t tid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (uint64_t)gridDim.x * blockDim.x;
  const uint4 z = make_uint4(0, 0, 0, 0);
  const uint64_t cap = (uint64_t)u.mask + 1, scap = (uint64_t)u.set_mask + 1;     // powers of two >= 1024
  for (uint64_t i = tid; i < cap / 2; i += nth) {
    reinterpret_cast<uint4 *>(u.keys)[i] = z;
    reinterpret_cast<uint4 *>(u.last)[i] = z;
  }
  for (uint64_t i = tid; i < cap / 4; i += nth) {
    reinterpret_cast<uint4 *>(u.inserts)[i] = z;
    reinterpret_cast<uint4 *>(u.distinct)[i] = z;
  }
  for (uint64_t i = tid; i < cap / 16; i += nth) reinterpret_cast<uint4 *>(u.cand)[i] = z;
  for (uint64_t i = tid; i < scap / 2; i += nth) reinterpret_cast<uint4 *>(u.set_keys)[i] = z;
  for (uint64_t i = tid; i < scap / 4; i += nth) reinterpret_cast<uint4 *>(u.set_count)[i] = z;
  for (uint64_t i = tid; i < n_sketch; i += nth) u.taxon_cand[i] = 0;
  const uint64_t nd = (uint64_t)u.direct_rows * n_sketch;
  for (uint64_t i = tid; i < nd; i += nth) u.direct[i] = 0;
  if (tid == 0) *u.n_cand = 0;
}
void launch_unit_clear(const UnitMap &u, uint32_t n_sketch, int n_sm, cudaStream_t stream) {
  k_unit_clear<<<n_sm * 8, 256, 0, stream>>>(u, n_sketch);
}

int launch_unit_accounting(const Params &p, int n_sm, cudaStream_t stream) {
  if (p.n_reads == 0) return 0;
  k_unit_mark<<<n_sm * 4, 256, 0, stream>>>(p);
  const int rgrid = (int)min((uint32_t)n_sm * 8, (p.n_reads + 7) / 8);
  k_unit_distinct<<<rgrid, 256, 0, stream>>>(p);
  k_unit_apply<<<n_sm * 4, 256, 0, stream>>>(p);
  return 3;
}

__global__ void k_flag_dense_global(const uint32_t *distinct, uint8_t *dense_flag, uint32_t n_sketch) {
  uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n_sketch && distinct[t] >= 1025u) dense_flag[t] = 1;
}
void launch_flag_dense_global(const uint32_t *distinct, uint8_t *dense_flag, uint32_t n_sketch, cudaStream_t stream) {
  if (n_sketch) k_flag_dense_global<<<(n_sketch + 255) / 256, 256, 0, stream>>>(distinct, dense_flag, n_sketch);
}

// getEncodedRank(enc, 25, 12), hyperloglogplus.cpp:152-161
__device__ __forceinline__ uint32_t encoded_rank_dev(uint32_t e) {
  if (e & 1) return 13 + ((e >> 1) & 0x3F);
  uint32_t r = e << 12;
  return (r ? (uint32_t)__clz(r) : 20u) + 1;
}

// sparseRegisterHistogram (hyperloglogplus.cpp:356-366) for every taxon that stayed sparse: C[t][rank]++ over the
// distinct codes of t (the host derives C[0] = 2^25 - |S_t|)
__global__ void k_sparse_histograms(const unsigned long long *slots, uint64_t cap, const uint8_t *dense_flag,
                                    uint32_t *hist) {
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < cap; i += (uint64_t)gridDim.x * blockDim.x) {
    const unsigned long long key = slots[i];
    if (!key) continue;
    const uint32_t taxon = (uint32_t)(key >> 32) - 1;
    if (dense_flag[taxon]) continue;
    atomicAdd(hist + (size_t)taxon * 64 + min(encoded_rank_dev((uint32_t)key), 63u), 1u);
  }
}
void launch_sparse_histograms(const unsigned long long *slots, uint64_t cap, const uint8_t *dense_flag,
                              uint32_t *hist, cudaStream_t stream) {
  if (cap) k_sparse_histograms<<<148 * 16, 256, 0, stream>>>(slots, cap, dense_flag, hist);
}

// union of the sparse code sets of the member taxa (sparse ∪ sparse merge, hyperloglogplus.cpp:600-603)
__global__ void k_sparse_union(const unsigned long long *slots, uint64_t cap, const uint8_t *member,
                               unsigned long long *scratch, uint64_t smask, uint32_t *hist64, uint32_t *overflow) {
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < cap; i += (uint64_t)gridDim.x * blockDim.x) {
    const unsigned long long key = slots[i];
    if (!key) continue;
    const uint32_t taxon = (uint32_t)(key >> 32) - 1;
    if (!member[taxon]) continue;
    const uint32_t code = (uint32_t)key;
    const unsigned long long k2 = (1ull << 32) | code;
    uint64_t q = mix64(k2) & smask;
    for (uint64_t probe = 0; probe <= smask; probe++) {
      unsigned long long cur = *reinterpret_cast<volatile unsigned long long *>(scratch + q);
      if (cur == k2) break;
      if (cur == 0) {
        cur = atomicCAS(scratch + q, 0ull, k2);
        if (cur == 0) { atomicAdd(hist64 + min(encoded_rank_dev(code), 63u), 1u); break; }
        if (cur == k2) break;
      }
      q = (q + 1) & smask;
      if (probe == smask) atomicExch(overflow, 1u);
    }
  }
}
void launch_sparse_union(const unsigned long long *slots, uint64_t cap, const uint8_t *member,
                         unsigned long long *scratch_set, uint64_t scratch_mask, uint32_t *hist64, uint32_t *overflow,
                         cudaStream_t stream) {
  if (cap) k_sparse_union<<<148 * 16, 256, 0, stream>>>(slots, cap, member, scratch_set, scratch_mask, hist64, overflow);
}

// export / import of the sparse tier (cross-GPU union of the (taxon, code) sets)
__global__ void k_sparse_export(const unsigned long long *slots, uint64_t cap, const uint8_t *dense_flag,
                                unsigned long long *out, uint64_t out_cap, unsigned long long *n_out) {
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < cap; i += (uint64_t)gridDim.x * blockDim.x) {
    const unsigned long long key = slots[i];
    const bool keep = key && !dense_flag[(uint32_t)(key >> 32) - 1];
    const uint32_t m = __ballot_sync(__activemask(), keep);
    if (!keep) continue;
    const uint32_t lane = threadIdx.x & 31;
    unsigned long long base = 0;
    const int leader = __ffs(m) - 1;
    if ((int)lane == leader) base = atomicAdd(n_out, (unsigned long long)__popc(m));
    base = __shfl_sync(m, base, leader);
    const unsigned long long pos = base + __popc(m & ((1u << lane) - 1));
    if (pos < out_cap) out[pos] = key;
  }
}
__global__ void k_sparse_import(const unsigned long long *keys, uint64_t n, SparseSet s, const uint8_t *dense_flag,
                                uint32_t *error_flag) {
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    const unsigned long long key = keys[i];
    if (!key) continue;
    const uint32_t taxon = (uint32_t)(key >> 32) - 1;
    if (dense_flag[taxon]) continue;
    const int ins = sparse_insert(s, taxon, (uint32_t)key);
    if (ins > 0) atomicAdd(s.distinct + taxon, 1u);
    else if (ins < 0) atomicExch(error_flag, 4u);
  }
}
void launch_sparse_export(const unsigned long long *slots, uint64_t cap, const uint8_t *dense_flag,
                          unsigned long long *out, uint64_t out_cap, unsigned long long *n_out, cudaStream_t stream) {
  if (cap) k_sparse_export<<<148 * 16, 256, 0, stream>>>(slots, cap, dense_flag, out, out_cap, n_out);
}
void launch_sparse_import(const unsigned long long *keys, uint64_t n, const SparseSet &s, const uint8_t *dense_flag,
                          uint32_t *error_flag, cudaStream_t stream) {
  if (n) k_sparse_import<<<(int)min((uint64_t)148 * 16, (n + 255) / 256), 256, 0, stream>>>(keys, n, s, dense_flag, error_flag);
}

// ---- exact counting (classifyExact) ---------------------------------------------------------------------------
// 1 = new pair, 0 = already there, -1 = table full.  Entries go 0 → final in one 128-bit CAS and never change again.
__device__ __forceinline__ int exact_insert(const ExactSet &e, uint32_t taxon, uint64_t canon) {
  const ExactPair want{canon + 1ull, (unsigned long long)taxon + 1ull};
  const ExactPair empty{0ull, 0ull};
  uint64_t s = mix64(canon * 0x9E3779B97F4A7C15ull + taxon) & e.mask;
  for (uint64_t probe = 0; probe <= e.mask; probe++) {
    const ulonglong2 seen = __ldcg(reinterpret_cast<const ulonglong2 *>(e.slots + s));    // one 16-byte load
    ExactPair cur{seen.x, seen.y};
    if (cur.kmer1 == 0 || cur.taxon1 == 0) {                // empty (or a load that raced with the writer): ask atomically
      cur = atomicCAS(e.slots + s, empty, want);
      if (cur.kmer1 == 0 && cur.taxon1 == 0) return 1;
    }
    if (cur.kmer1 == want.kmer1 && cur.taxon1 == want.taxon1) return 0;
    s = (s + 1) & e.mask;
  }
  return -1;
}

// add_kmer of the exact container (readcounts.hpp:71-74 with khset64_t): thread per text position, after the lookup
// wrote the window's dense taxon (0 for a miss) to codes_dense
__global__ void __launch_bounds__(256) k_exact_insert(const __grid_constant__ Params p) {
  const uint64_t g_begin = p.offsets[0], g_end = p.offsets[p.n_reads];
  for (uint64_t g = g_begin + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; g < g_end;
       g += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t bin = __ldg(p.bins + g);
    if (bin == BIN_NONE || bin == BIN_AMBIG) continue;
    const uint32_t taxon = p.codes_dense[g];
    const int ins = exact_insert(p.exact, taxon, __ldg(p.canon + g));
    if (ins > 0) atomicAdd(p.exact.count + taxon, 1ull);
    else if (ins < 0) atomicExch(p.error_flag, 4u);
  }
}

// distinct k-mers among the pairs whose taxon is a clade member
__global__ void k_exact_union(ExactSet e, const uint8_t *member, unsigned long long *scratch, uint64_t smask,
                              unsigned long long *n_distinct, uint32_t *overflow) {
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= e.mask; i += (uint64_t)gridDim.x * blockDim.x) {
    const ExactPair pr = e.slots[i];
    if (!pr.kmer1 || !member[pr.taxon1 - 1]) continue;
    uint64_t q = mix64(pr.kmer1) & smask;
    for (uint64_t probe = 0; probe <= smask; probe++) {
      unsigned long long cur = *reinterpret_cast<volatile unsigned long long *>(scratch + q);
      if (cur == pr.kmer1) break;
      if (cur == 0) {
        cur = atomicCAS(scratch + q, 0ull, pr.kmer1);
        if (cur == 0) { atomicAdd(n_distinct, 1ull); break; }
        if (cur == pr.kmer1) break;
      }
      q = (q + 1) & smask;
      if (probe == smask) atomicExch(overflow, 1u);
    }
  }
}
void launch_exact_union(const ExactSet &e, const uint8_t *member, unsigned long long *scratch_set, uint64_t scratch_mask,
                        unsigned long long *n_distinct, uint32_t *overflow, cudaStream_t stream) {
  if (e.slots) k_exact_union<<<148 * 16, 256, 0, stream>>>(e, member, scratch_set, scratch_mask, n_distinct, overflow);
}

// Quick mode, preloaded path: the k-mer loop of classify_sequence leaves at the quick_min-th hit (classify.cpp:943-944),
// so the windows behind it are never looked at — no add_kmer, no hit.  One warp per read finds that window in the
// looked-up codes, shortens the read to it and wipes the later windows from the scan scratch; the counting pass
// (k_lookup<MODE_RESOLVE>), the per-unit accounting and k_resolve<true> then see the read the reference saw.
__global__ void __launch_bounds__(256) k_quick_cut(const __grid_constant__ Params p, const uint32_t *codes) {
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t warps_total = gridDim.x * (blockDim.x >> 5);
  for (uint32_t r = blockIdx.x * (blockDim.x >> 5) + warp; r < p.n_reads; r += warps_total) {
    const uint64_t base = p.offsets[r];
    const uint32_t nwin = p.n_windows[r];
    uint32_t seen = 0, cutoff = nwin;
    for (uint32_t s = 0; s * 32 < nwin; s++) {
      const uint32_t i = s * 32 + lane;
      const uint32_t c = i < nwin ? codes[base + i] : 0;
      const uint32_t bm = __ballot_sync(0xFFFFFFFFu, c != 0 && c != AMBIG && c != FOUND_ZERO);
      const uint32_t cnt = __popc(bm);
      if (seen + cnt >= p.quick_min) {
        uint32_t m = bm;
        for (uint32_t j = seen + 1; j < p.quick_min; j++) m &= m - 1;   // drop the hits before the quick_min-th
        cutoff = s * 32 + (uint32_t)__ffs(m) - 1;
        break;
      }
      seen += cnt;
    }
    if (cutoff < nwin) {
      for (uint32_t i = cutoff + 1 + lane; i < nwin; i += 32) p.bins[base + i] = BIN_NONE;
      if (lane == 0) p.n_windows[r] = cutoff + 1;
    }
  }
}

int classify_smem_bytes() { return N_STAGES * STAGE_BYTES + (int)sizeof(SharedState); }

// mode MODE_FUSED : scan → lookup (+HLL) → resolve            (whole database on this GPU)
//      MODE_LOOKUP: scan → lookup into p.codes_dense            (one range of a sharded / chunked database)
//      MODE_RESOLVE: scan → HLL from merged codes → resolve    (owner of the reads after the merge)
// picks the lean instantiation when the launch uses none of the rare switches (see k_lookup)
template <int MODE>
static void launch_lookup(const Params &q, int lgrid, cudaStream_t stream) {
  const bool lean = !(q.flags & (KUQ_F_STATS | F_FOUND_ZERO | F_SHARD_COUNTING)) && !q.only_hits && !q.n_peers;
  if (lean) k_lookup<MODE, true><<<lgrid, 256, 0, stream>>>(q);
  else k_lookup<MODE, false><<<lgrid, 256, 0, stream>>>(q);
}

int launch_classify(int mode, const Params &p, int n_sm, cudaStream_t stream, cudaEvent_t *stage_events) {
  const int smem = classify_smem_bytes();
  // per device (function attributes belong to the current context): cheap enough to set on every call
  cudaFuncSetAttribute(k_scan, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  int launches = 0;
  if (p.n_reads == 0) return 0;
  int grid = n_sm * 4;
  if ((uint32_t)grid > p.n_chunks) grid = (int)p.n_chunks;
  k_scan<<<grid, CTA_THREADS, smem, stream>>>(p);
  launches++;
  if (stage_events) cudaEventRecord(stage_events[0], stream);
  const int lgrid = (int)min((uint64_t)n_sm * 8 * 8, (p.total_bases + 255) / 256);
  const bool quick = p.quick_min != 0 && mode != MODE_LOOKUP;
  const bool exact = p.hll_mode == KUQ_HLL_EXACT && mode != MODE_LOOKUP;
  if (exact) {
    // classifyExact: plain lookup (no sketch work), then the k-mer sets, then the usual resolve
    Params q = p;
    if (mode == MODE_FUSED) {
      q.only_hits = 0; q.n_peers = 0; q.flags &= ~F_FOUND_ZERO;
      launch_lookup<MODE_LOOKUP>(q, lgrid, stream);
    } else {
      q.flags |= KUQ_F_NO_COUNTS;                                     // merged codes → codes_dense, no sketches
      launch_lookup<MODE_RESOLVE>(q, lgrid, stream);
    }
    if (!(p.flags & KUQ_F_NO_COUNTS)) { k_exact_insert<<<lgrid, 256, 0, stream>>>(p); launches++; }
  } else if (quick && p.quick_stop) {
    // lookup first, end every read at its quick_min-th hit, then count what is left
    Params q = p;
    if (mode == MODE_FUSED) {
      q.only_hits = 0; q.n_peers = 0; q.flags &= ~F_FOUND_ZERO;
      launch_lookup<MODE_LOOKUP>(q, lgrid, stream);
      launches++;
      q.codes_in = p.codes_dense;
    }
    const int cgrid = (int)min((uint32_t)n_sm * 8, (p.n_reads + 7) / 8);
    k_quick_cut<<<cgrid, 256, 0, stream>>>(p, q.codes_in);
    q.flags = p.flags;
    launch_lookup<MODE_RESOLVE>(q, lgrid, stream);
    launches += 2;
  } else if (mode == MODE_FUSED) launch_lookup<MODE_FUSED>(p, lgrid, stream);
  else if (mode == MODE_LOOKUP) launch_lookup<MODE_LOOKUP>(p, lgrid, stream);
  else launch_lookup<MODE_RESOLVE>(p, lgrid, stream);
  if (exact || !(quick && p.quick_stop)) launches++;
  if (stage_events) cudaEventRecord(stage_events[1], stream);
  if (mode != MODE_LOOKUP) {
    const int rgrid = (int)min((uint32_t)n_sm * 4 * 2, (p.n_reads + CTA_WARPS - 1) / CTA_WARPS);
    if (quick) k_resolve<true><<<rgrid, 256, 0, stream>>>(p);
    else k_resolve<false><<<rgrid, 256, 0, stream>>>(p);
    launches++;
  }
  return launches;
}

// ------------------------------------------------------------------------------------------------------
// set_lcas (set_lcas.cpp:429-476), SURVEY.md §8 f4.  ROUND 1: compiled, not yet run on hardware.
// Library sequences arrive cut into pieces (the reference's SKIP_LEN pieces, :363-364); unit_id[r] carries the dense
// taxid of piece r.  One warp per piece, lane = window: find the record of the canonical k-mer and fold the
// sequence's taxid into its value with lca() through a CAS loop.  lca over taxa of one tree is associative,
// commutative and idempotent (default ancestor 1), so the order in which pieces and sequences land does not matter.
// Under -T a contaminant taxid beats everything and sticks; with at most ONE of the two contaminant taxids per batch
// (the host side sees to that) the outcome is again independent of the order inside the batch.
// ------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_set_lcas(const __grid_constant__ Params p) {
  const DbView &db = p.db;
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t warps_total = gridDim.x * (blockDim.x >> 5);
  uint8_t *pairs = const_cast<uint8_t *>(db.pairs);
  for (uint32_t r = blockIdx.x * (blockDim.x >> 5) + warp; r < p.n_reads; r += warps_total) {
    const uint64_t base = p.offsets[r];
    const uint32_t nwin = p.n_windows[r];
    const uint32_t t = p.unit_id[r];
    for (uint32_t i = lane; i < nwin; i += 32) {
      const uint32_t bin = __ldg(p.bins + base + i);
      if (bin == BIN_NONE || bin == BIN_AMBIG) continue;                  // :434-435
      if (bin < db.bin_lo || bin >= db.bin_hi) continue;                  // another range of the database
      const uint64_t canon = __ldg(p.canon + base + i);
      const uint64_t *o = db.offsets + (bin - db.bin_lo);
      uint64_t lo = __ldg(o) - db.rec_base, hi = __ldg(o + 1) - db.rec_base;
      bool found = false;
      while (lo < hi) {
        const uint64_t mid = lo + ((hi - lo) >> 1);
        const uint64_t key = load_key(db.pairs, mid, db.key_mask);
        if (key < canon) lo = mid + 1;
        else if (key > canon) hi = mid;
        else { lo = mid; found = true; break; }
      }
      if (!found) { atomicAdd(p.stats, 1ull); continue; }                 // "kmer found in sequence that is not in database"
      uint32_t *val = reinterpret_cast<uint32_t *>(pairs + lo * 12) + 2;
      uint32_t old = *reinterpret_cast<volatile uint32_t *>(val);
      for (;;) {
        uint32_t nw;
        if (p.lca_flags & KUQ_LCA_RESET) nw = 0;                                           // -R, :458-459
        else if (!(p.lca_flags & KUQ_LCA_FORCE_CONTAMINANT)) nw = lca_dense(p.tax, t, old);  // :461
        else if (old != 0 && (old == p.lca_keep[0] || old == p.lca_keep[1])) nw = old;   // -T: contaminants stick, :465-466
        else if (t == p.lca_keep[0] || t == p.lca_keep[1]) nw = t;        // :467-470
        else nw = lca_dense(p.tax, t, old);                               // :472
        if (nw == old) break;
        const uint32_t prev = atomicCAS(val, old, nw);
        if (prev == old) break;
        old = prev;
      }
    }
  }
}

// stage 1 alone: canonical k-mer + minimizer bin of every window into p.canon / p.bins (database build, workload tools)
int launch_scan_only(const Params &p, int n_sm, cudaStream_t stream) {
  if (p.n_reads == 0) return 0;
  const int smem = classify_smem_bytes();
  cudaFuncSetAttribute(k_scan, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  int grid = n_sm * 4;
  if ((uint32_t)grid > p.n_chunks) grid = (int)p.n_chunks;
  k_scan<<<grid, CTA_THREADS, smem, stream>>>(p);
  return 1;
}

// stage 2 alone over scratch that is already there (kuq_layout_exp.cu times the product's kernel next to its variants):
// p.offsets = {first, last + 1} text positions with p.n_reads = 1
// fused = 1: k_lookup<MODE_FUSED> (counts into the sketches of p); lean: see k_lookup (the caller vouches for the flags)
int launch_lookup_only(const Params &p, int n_sm, cudaStream_t stream, int fused, int lean) {
  const int lgrid = (int)max((uint64_t)1, min((uint64_t)n_sm * 8 * 8, (p.total_bases + 255) / 256));
  if (fused) {
    if (lean) k_lookup<MODE_FUSED, true><<<lgrid, 256, 0, stream>>>(p);
    else k_lookup<MODE_FUSED, false><<<lgrid, 256, 0, stream>>>(p);
  } else {
    if (lean) k_lookup<MODE_LOOKUP, true><<<lgrid, 256, 0, stream>>>(p);
    else k_lookup<MODE_LOOKUP, false><<<lgrid, 256, 0, stream>>>(p);
  }
  return 1;
}

// scan the pieces, then fold their taxids into the record values; returns #kernels launched
int launch_set_lcas(const Params &p, int n_sm, cudaStream_t stream) {
  if (p.n_reads == 0) return 0;
  const int smem = classify_smem_bytes();
  cudaFuncSetAttribute(k_scan, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  int grid = n_sm * 4;
  if ((uint32_t)grid > p.n_chunks) grid = (int)p.n_chunks;
  k_scan<<<grid, CTA_THREADS, smem, stream>>>(p);
  const int rgrid = (int)min((uint32_t)n_sm * 8, (p.n_reads + 7) / 8);
  k_set_lcas<<<rgrid, 256, 0, stream>>>(p);
  return 2;
}

// ------------------------------------------------------------------------------------------------------
// database staging: distinct taxids + record counts (KrakenDB::count_taxons, krakendb.cpp:90-113) and the
// in-place rewrite taxid → dense id
// ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t hash_u32(uint32_t x) {
  x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16;
  return x;
}

// keys[] holds taxid + 1 (0 = empty)
__global__ void k_collect_taxids(const uint8_t *pairs, uint64_t n_rec, uint32_t *keys, unsigned long long *counts,
                                 uint32_t cap_mask, uint32_t *overflow) {
  const uint32_t lane = threadIdx.x & 31;
  for (uint64_t base = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) - lane; base < n_rec;
       base += (uint64_t)gridDim.x * blockDim.x) {
    uint64_t i = base + lane;
    bool in = i < n_rec;
    uint32_t v = in ? load_val(pairs, i) : 0;
    uint32_t active = __ballot_sync(0xFFFFFFFFu, in);
    if (!in) continue;
    uint32_t same = __match_any_sync(active, v);
    if (lane != (uint32_t)(__ffs(same) - 1)) continue;      // one lane per distinct value
    uint32_t key = v + 1;
    if (key == 0) { atomicExch(overflow, 2u); continue; }   // taxid 0xFFFFFFFF is reserved
    uint32_t slot = hash_u32(v) & cap_mask;
    for (uint32_t probe = 0; probe <= cap_mask; probe++) {
      uint32_t cur = keys[slot];
      if (cur == 0) cur = atomicCAS(keys + slot, 0u, key), cur = cur ? cur : key;
      if (cur == key) { atomicAdd(counts + slot, (unsigned long long)__popc(same)); break; }
      slot = (slot + 1) & cap_mask;
      if (probe == cap_mask) atomicExch(overflow, 1u);
    }
  }
}

__global__ void k_remap_values(uint8_t *pairs, uint64_t n_rec, const uint32_t *keys, const uint32_t *dense,
                               uint32_t cap_mask, uint32_t *missing, uint32_t hi_mask) {
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_rec; i += (uint64_t)gridDim.x * blockDim.x) {
    uint32_t *vp = reinterpret_cast<uint32_t *>(pairs + i * 12) + 2;
    uint32_t v = *vp;
    uint32_t key = v + 1, slot = hash_u32(v) & cap_mask, d = 0xFFFFFFFFu;
    for (uint32_t probe = 0; probe <= cap_mask; probe++) {
      uint32_t cur = keys[slot];
      if (cur == key) { d = dense[slot]; break; }
      if (cur == 0) break;
      slot = (slot + 1) & cap_mask;
    }
    if (d == 0xFFFFFFFFu) { atomicExch(missing, 1u); d = 0; }
    *vp = d;
    // bits of the key word above 2k are ignored by the reference (krakendb.cpp:283-284) and serve as record flags
    // here (SEEN_BIT): start from zero
    if ((vp[-1] & ~hi_mask) != 0) vp[-1] &= hi_mask;
  }
}

// Flagged records → sparse-tier keys (once per run / before a range leaves HBM): for every record a counted hit
// flagged, insert (taxon, encodeHashIn32Bit(hash(k-mer))) into the set unless the taxon went dense, and clear the
// flag.  mode 0 = count the flagged records of taxa that are not dense (stats[0]), 1 = insert + clear, 2 = clear only.
__global__ void __launch_bounds__(256) k_harvest_seen(uint8_t *pairs, uint64_t n_rec, uint32_t hi_mask, const uint8_t *dense_flag,
                                                      SparseSet set, unsigned long long *stats, uint32_t *error_flag, int mode) {
  unsigned long long n_local = 0;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_rec; i += (uint64_t)gridDim.x * blockDim.x) {
    uint32_t *w = reinterpret_cast<uint32_t *>(pairs + i * 12);
    const uint32_t hiw = w[1];
    if (!(hiw & SEEN_BIT)) continue;
    const uint32_t taxon = w[2];
    if (mode == 0) { n_local += dense_flag[taxon] ? 0 : 1; continue; }
    w[1] = hiw & ~SEEN_BIT;
    if (mode == 2 || dense_flag[taxon]) continue;
    const uint64_t key = ((uint64_t)(hiw & hi_mask) << 32) | w[0];
    const int ins = sparse_insert(set, taxon, encode_hash32(fmix64(key)));
    if (ins > 0) atomicAdd(set.distinct + taxon, 1u);
    else if (ins < 0) atomicExch(error_flag, 4u);
  }
  if (mode == 0) {
    for (int o = 16; o; o >>= 1) n_local += __shfl_xor_sync(0xFFFFFFFFu, n_local, o);
    if ((threadIdx.x & 31) == 0 && n_local) atomicAdd(stats, n_local);
  }
}
void launch_harvest_seen(uint8_t *pairs, uint64_t n_rec, uint64_t key_mask, const uint8_t *dense_flag, const SparseSet &set,
                         unsigned long long *stats, uint32_t *error_flag, int mode, cudaStream_t stream) {
  if (!n_rec) return;
  const int grid = (int)min((uint64_t)148 * 16, (n_rec + 255) / 256);
  k_harvest_seen<<<grid, 256, 0, stream>>>(pairs, n_rec, (uint32_t)(key_mask >> 32), dense_flag, set, stats, error_flag, mode);
}

// re-insert the keys of an outgrown table into its successor (no per-taxon counting: the keys were counted before)
__global__ void k_sparse_rehash(const unsigned long long *old_slots, uint64_t old_cap, SparseSet s, uint32_t *error_flag) {
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < old_cap; i += (uint64_t)gridDim.x * blockDim.x) {
    const unsigned long long key = old_slots[i];
    if (!key) continue;
    if (sparse_insert(s, (uint32_t)(key >> 32) - 1, (uint32_t)key) < 0) atomicExch(error_flag, 4u);
  }
}
void launch_sparse_rehash(const unsigned long long *old_slots, uint64_t old_cap, const SparseSet &s, uint32_t *error_flag,
                          cudaStream_t stream) {
  if (old_cap) k_sparse_rehash<<<148 * 16, 256, 0, stream>>>(old_slots, old_cap, s, error_flag);
}

// C[taxon][v] = number of registers of the taxon holding v (registerHistogram, hyperloglogplus.cpp:337-354);
// the double-precision Ertl sum over it runs on the host.
__global__ void k_register_histograms(const uint8_t *regs, uint32_t n_sketch, uint32_t *hist) {
  __shared__ uint32_t h[64];
  for (uint32_t t = blockIdx.x; t < n_sketch; t += gridDim.x) {
    if (threadIdx.x < 64) h[threadIdx.x] = 0;
    __syncthreads();
    const uint32_t *w = reinterpret_cast<const uint32_t *>(regs + (size_t)t * HLL_M);
    for (uint32_t i = threadIdx.x; i < HLL_M / 4; i += blockDim.x) {
      uint32_t x = w[i];
      atomicAdd(&h[x & 63], 1u);
      atomicAdd(&h[(x >> 8) & 63], 1u);
      atomicAdd(&h[(x >> 16) & 63], 1u);
      atomicAdd(&h[(x >> 24) & 63], 1u);
    }
    __syncthreads();
    if (threadIdx.x < 64) hist[(size_t)t * 64 + threadIdx.x] = h[threadIdx.x];
    __syncthreads();
  }
}

// register-wise max over the sketches of the listed dense ids: the dense∪dense merge of the clade roll-up
// (hyperloglogplus.cpp:614-620)
__global__ void k_clade_max(const uint8_t *regs, const uint32_t *members, uint32_t n_members, uint8_t *out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;     // word index 0..1023
  if (i >= HLL_M / 4) return;
  uint32_t acc = 0;
  for (uint32_t m = 0; m < n_members; m++) {
    uint32_t x = reinterpret_cast<const uint32_t *>(regs + (size_t)members[m] * HLL_M)[i];
    acc = __vmaxu4(acc, x);
  }
  reinterpret_cast<uint32_t *>(out)[i] = acc;
}

__global__ void k_fill_u32(uint32_t *p, uint64_t n, uint32_t v) {
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) p[i] = v;
}

void launch_collect_taxids(const uint8_t *pairs, uint64_t n_rec, uint32_t *keys, unsigned long long *counts,
                           uint32_t cap_mask, uint32_t *overflow, cudaStream_t stream) {
  if (!n_rec) return;
  int grid = (int)min((uint64_t)148 * 8, (n_rec + 255) / 256);
  k_collect_taxids<<<grid, 256, 0, stream>>>(pairs, n_rec, keys, counts, cap_mask, overflow);
}
void launch_remap_values(uint8_t *pairs, uint64_t n_rec, const uint32_t *keys, const uint32_t *dense,
                         uint32_t cap_mask, uint32_t *missing, uint64_t key_mask, cudaStream_t stream) {
  if (!n_rec) return;
  int grid = (int)min((uint64_t)148 * 8, (n_rec + 255) / 256);
  k_remap_values<<<grid, 256, 0, stream>>>(pairs, n_rec, keys, dense, cap_mask, missing, (uint32_t)(key_mask >> 32));
}
void launch_register_histograms(const uint8_t *regs, uint32_t n_sketch, uint32_t *hist, cudaStream_t stream) {
  if (!n_sketch) return;
  k_register_histograms<<<min(n_sketch, 148u * 16), 256, 0, stream>>>(regs, n_sketch, hist);
}
void launch_clade_max(const uint8_t *regs, const uint32_t *members, uint32_t n_members, uint8_t *out4096,
                      cudaStream_t stream) {
  k_clade_max<<<4, 256, 0, stream>>>(regs, members, n_members, out4096);
}
void launch_fill_u32(uint32_t *p, uint64_t n, uint32_t v, cudaStream_t stream) {
  if (!n) return;
  k_fill_u32<<<(int)min((uint64_t)148 * 8, (n + 255) / 256), 256, 0, stream>>>(p, n, v);
}

// `taxon_counts[t] += other[t]` (classify.cpp:542-544) for the state of another context copied next to ours:
// registers max (hyperloglogplus.cpp:614-620), counters add (readcounts.hpp:76-88), dense anywhere = dense (:604-612)
__global__ void k_merge_state(uint32_t *regs, const uint32_t *regs2, uint64_t n_words, unsigned long long *n_kmers,
                              const unsigned long long *n_kmers2, uint32_t n_sketch, unsigned long long *n_reads,
                              const unsigned long long *n_reads2, uint32_t n_taxa, uint8_t *dense, const uint8_t *dense2) {
  const uint64_t tid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t i = tid; i < n_words; i += nth) regs[i] = __vmaxu4(regs[i], regs2[i]);
  for (uint64_t i = tid; i < n_sketch; i += nth) { n_kmers[i] += n_kmers2[i]; dense[i] |= dense2[i]; }
  for (uint64_t i = tid; i < n_taxa; i += nth) n_reads[i] += n_reads2[i];
}
void launch_merge_state(uint8_t *regs, const uint8_t *regs2, unsigned long long *n_kmers, const unsigned long long *n_kmers2,
                        uint32_t n_sketch, unsigned long long *n_reads, const unsigned long long *n_reads2, uint32_t n_taxa,
                        uint8_t *dense, const uint8_t *dense2, cudaStream_t stream) {
  k_merge_state<<<148 * 4, 256, 0, stream>>>(reinterpret_cast<uint32_t *>(regs), reinterpret_cast<const uint32_t *>(regs2),
                                             (uint64_t)n_sketch * (HLL_M / 4), n_kmers, n_kmers2, n_sketch, n_reads, n_reads2, n_taxa,
                                             dense, dense2);
}

// ------------------------------------------------------------------------------------------------------
// Cross-GPU step synchronisation without the host (database sharded by minimizer range, SURVEY.md §8(e).2).
// Flags are 64-bit counters in device memory every peer has mapped (CUDA IPC or peer access).  k_signal_peers runs
// in stream order after the work it announces: the kernel boundary has made that work's peer stores visible at
// system scope, the fence orders them before the flag stores.  k_wait_flags spins (one lane per flag) until every
// flag has reached `value`; a peer that died shows up as a timeout (error code 6), not as a hung GPU.
// ------------------------------------------------------------------------------------------------------
struct PeerFlags { unsigned long long *ptr[8]; };
__global__ void k_signal_peers(PeerFlags f, uint32_t n, uint32_t my_index, unsigned long long value) {
  if (threadIdx.x < n) {
    __threadfence_system();
    *reinterpret_cast<volatile unsigned long long *>(f.ptr[threadIdx.x] + my_index) = value;
    __threadfence_system();
  }
}
__global__ void k_wait_flags(const unsigned long long *flags, uint32_t n, unsigned long long value, unsigned long long timeout_ns,
                             uint32_t *error_flag) {
  if (threadIdx.x >= n) return;
  unsigned long long t0;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  const volatile unsigned long long *f = flags + threadIdx.x;
  while (*f < value) {
    unsigned long long t1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
    if (t1 - t0 > timeout_ns) { atomicExch(error_flag, 6u); break; }
    __nanosleep(200);
  }
  __threadfence_system();
}
void launch_signal_peers(unsigned long long *const *flag_ptrs, uint32_t n, uint32_t my_index, unsigned long long value,
                         cudaStream_t stream) {
  PeerFlags f;
  for (uint32_t j = 0; j < 8; j++) f.ptr[j] = j < n ? flag_ptrs[j] : nullptr;
  k_signal_peers<<<1, 32, 0, stream>>>(f, n, my_index, value);
}
void launch_wait_flags(const unsigned long long *flags, uint32_t n, unsigned long long value, unsigned long long timeout_ns,
                       uint32_t *error_flag, cudaStream_t stream) {
  k_wait_flags<<<1, 32, 0, stream>>>(flags, n, value, timeout_ns, error_flag);
}

// Sparse-tier keys of the taxa that are still sparse, grouped by the rank that owns their CODE
// (part = hash(code) % n_parts): all keys that can ever be duplicates of each other — the same (taxon, code) seen on
// several GPUs, or the same code under two taxa of one clade — meet on one rank, so per-taxon distinct counts and
// clade unions are sums of per-rank results.  pass 0 counts (counts[part]), pass 1 scatters through cursors[part].
__device__ __forceinline__ uint32_t key_part(unsigned long long key, uint32_t n_parts) {
  return (uint32_t)((mix64((uint32_t)key) >> 33) % n_parts);
}
// One kernel for both sources of keys — SRC 0: the slots of the local set, SRC 1: the records a counted hit flagged
// (pass 1 clears the flag: the key leaves this GPU instead of entering its set).  pass 0 counts per part, pass 1
// scatters through the per-part cursors.  Same-address atomics would serialise hundreds of millions of keys on
// n_parts counters, so keys are counted / ranked on shared-memory counters (only real keys touch them — most slots are
// empty and most records unflagged, and a per-part warp vote for every item made the kernel instruction bound), and
// only one thread per part and CTA touches the global cursor per tile.
constexpr int KP_E = 8;      // keys per thread and tile: four block-wide barriers per 2048 items instead of per 256
template <int SRC>
__global__ void __launch_bounds__(256) k_keys_parts(const unsigned long long *slots, uint8_t *pairs, uint64_t n_items, uint32_t hi_mask,
                                                    const uint8_t *dense_flag, uint32_t n_parts, unsigned long long *counters,
                                                    unsigned long long *out, const unsigned long long *part_end, uint32_t *error_flag,
                                                    int pass) {
  __shared__ uint32_t s_total32[8];              // pass 0: the CTA's counts (a CTA sees far fewer than 2^32 items)
  __shared__ uint32_t s_cnt[8];                  // pass 1: keys of the tile per part
  __shared__ unsigned long long s_base[8];
  const uint32_t tid = threadIdx.x;
  if (tid < 8) { s_total32[tid] = 0; s_cnt[tid] = 0; }
  __syncthreads();
  const uint64_t tile = (uint64_t)blockDim.x * KP_E;
  for (uint64_t base = (uint64_t)blockIdx.x * tile; base < n_items; base += (uint64_t)gridDim.x * tile) {
    unsigned long long key[KP_E];
    uint32_t where[KP_E];                        // part << 28 | rank inside the tile's group of that part
    // all loads of the tile first (KP_E independent requests per thread in flight: the scan is bandwidth work), then
    // the per-key arithmetic
    uint32_t hiws[KP_E];
#pragma unroll
    for (int j = 0; j < KP_E; j++) {
      const uint64_t i = base + (uint64_t)j * blockDim.x + tid;
      key[j] = 0; hiws[j] = 0;
      if (i < n_items) {
        if (SRC == 0) key[j] = __ldg(slots + i);
        else hiws[j] = __ldg(reinterpret_cast<const uint32_t *>(pairs + i * 12) + 1);
      }
    }
#pragma unroll
    for (int j = 0; j < KP_E; j++) {
      const uint64_t i = base + (uint64_t)j * blockDim.x + tid;
      unsigned long long k = 0;
      if (i < n_items) {
        if (SRC == 0) {
          k = key[j];
          if (k && dense_flag[(uint32_t)(k >> 32) - 1]) k = 0;
        } else {
          uint32_t *w = reinterpret_cast<uint32_t *>(pairs + i * 12);
          const uint32_t hiw = hiws[j];
          if (hiw & SEEN_BIT) {
            if (pass == 1) w[1] = hiw & ~SEEN_BIT;
            const uint32_t taxon = w[2];
            if (!dense_flag[taxon]) {
              const uint64_t kmer = ((uint64_t)(hiw & hi_mask) << 32) | w[0];
              k = ((unsigned long long)(taxon + 1) << 32) | encode_hash32(fmix64(kmer));
            }
          }
        }
      }
      key[j] = k;
      where[j] = 0;
      if (k) {                                   // only real keys cost anything: one shared-memory atomic on the part's counter
        const uint32_t part = key_part(k, n_parts);
        if (pass == 0) atomicAdd(&s_total32[part], 1u);
        else where[j] = (part << 28) | atomicAdd(&s_cnt[part], 1u);
      }
    }
    if (pass == 1) {
      __syncthreads();
      if (tid < n_parts && s_cnt[tid]) s_base[tid] = atomicAdd(counters + tid, (unsigned long long)s_cnt[tid]);
      __syncthreads();
#pragma unroll
      for (int j = 0; j < KP_E; j++) {
        if (!key[j]) continue;
        const uint32_t part = where[j] >> 28;
        const unsigned long long at = s_base[part] + (where[j] & 0x0FFFFFFFu);
        if (at < part_end[part]) out[at] = key[j]; else atomicExch(error_flag, 7u);
      }
      __syncthreads();
      if (tid < 8) s_cnt[tid] = 0;
      __syncthreads();
    }
  }
  if (pass == 0) {
    __syncthreads();
    if (tid < n_parts && s_total32[tid]) atomicAdd(counters + tid, (unsigned long long)s_total32[tid]);
  }
}
void launch_keys_parts(int src, const unsigned long long *slots, uint8_t *pairs, uint64_t n_items, uint64_t key_mask,
                       const uint8_t *dense_flag, uint32_t n_parts, unsigned long long *counters, unsigned long long *out,
                       const unsigned long long *part_end, uint32_t *error_flag, int pass, cudaStream_t stream) {
  if (!n_items) return;
  const int grid = (int)min((uint64_t)148 * 8, (n_items + 256 * KP_E - 1) / (256 * KP_E));
  if (src == 0) k_keys_parts<0><<<grid, 256, 0, stream>>>(slots, pairs, n_items, (uint32_t)(key_mask >> 32), dense_flag, n_parts, counters, out, part_end, error_flag, pass);
  else k_keys_parts<1><<<grid, 256, 0, stream>>>(slots, pairs, n_items, (uint32_t)(key_mask >> 32), dense_flag, n_parts, counters, out, part_end, error_flag, pass);
}

}  // namespace kuq
