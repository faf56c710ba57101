#!/usr/bin/env python
"""bench.py — KrakenUniq classification hot path on B200: Mreads/s on 150 bp reads (BASELINE.json metric).

  python bench.py --gpus 1 --steps 10 --warmup 3            # our arm (libkuq.so)
  python bench.py --impl reference --gpus 1 --steps 3 --warmup 1   # the unmodified reference on the host cores
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...   # one rank per GPU (replicas)

Workload (config.workload): BASELINE.json configs[1] — an "8 GB" synthetic KrakenDB (k=31, m=15: 666 M records
→ 8.0 GB database.kdb + 8.6 GB database.idx, all of it resident in HBM) and 10 M synthetic 150 bp reads,
generated on the GPU from fixed seeds (krakenuniq_b200/synth_gpu.py).  One step = one pass of the hot path
over one batch of 1 M reads (150 MB of read text, > L2; the lookups touch the 16.6 GB database at random).

`value`  : device-resident inputs, CUDA events on the launching stream (the slot's stream), max over ranks.
`e2e`    : the same metric through the C ABI with HOST buffers: pinned reads → H2D → kernel → D2H of calls and
           run-length hit lists every step, pipelined over the context's batch slots.
`--mode shards` (SURVEY.md §8(e).2, BASELINE configs[3]): the database is cut into one minimizer range per GPU
(each rank builds only its range), every GPU scans every batch, hits go to the owner GPU over NVLink
(`--merge p2p`, fused lookup + peer scatter) or through an NCCL all-reduce (`--merge nccl`).
Multi-GPU default (SURVEY.md §8(e).1): the database fits one card, so ranks are replicas; reads are partitioned across
ranks (weak scaling: 1 M reads per rank per step); the only collective is the once-per-run merge of the per-taxon
state (allreduce MAX over HLL registers, SUM over counters, all-gather of the sparse-tier keys); it is not part of a
step and is reported separately as config.end_of_run_merge_ms.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import re
import shutil
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "Mreads/s (150 bp)"
READ_LEN = 150
K, NT = 31, 15


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--db-records", type=int, default=0,
                    help="records of the synthetic database (0 = 666 M for replicas / the configs[3] size for shards)")
    ap.add_argument("--db-passes", type=int, default=0, help="build the synthetic DB in this many minimizer ranges (0 = auto)")
    ap.add_argument("--genomes", type=int, default=2000)
    ap.add_argument("--reads", type=int, default=10_000_000, help="reads in the pool")
    ap.add_argument("--batch-reads", type=int, default=1_000_000, help="reads per step")
    ap.add_argument("--cpu-sample-reads", type=int, default=250_000, help="reads per CPU-reference step")
    ap.add_argument("--cpu-threads", type=int, default=0, help="threads for the reference (0 = all host cores)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--hll-mode", type=int, default=0, help="0 preload rule (reference default), 1 chunked, 2 dense only")
    ap.add_argument("--cache-dir", default=os.environ.get("KUQ_BENCH_CACHE", "/dev/shm"))
    ap.add_argument("--range-gb", type=float, default=0.0, help="stream mode: GB of records per streamed range (0 = 24, paired 32)")
    ap.add_argument("--paired", action="store_true", help="stream mode: configs[4], 2 x 150 bp mates merged with N")
    ap.add_argument("--stream-both", action="store_true", help="stream mode: configs[2] and configs[4] against one generated database")
    ap.add_argument("--mode", default="auto", choices=["auto", "replicas", "shards", "stream"],
                    help="multi-GPU layout: replicas (DB on every GPU, reads partitioned) or minimizer-range shards; "
                         "auto = replicas on one GPU, on several GPUs the sharded configs[3] line with the replicas "
                         "numbers under the key 'replicas'")
    ap.add_argument("--merge", default="p2p", choices=["p2p", "nccl"],
                    help="shards: hits stored into the owner's buffer over NVLink (p2p) or ids all-reduced (nccl)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="replicas layout: after the timed steps, write what the last timed step returned (calls, window "
                         "counts, hit lists of a seeded sample of reads) and the run's per-taxon counters as DIR/<name>.npy, "
                         "so that two builds can be compared output for output")
    return ap.parse_args()


# ------------------------------------------------------------------------------------------------------------
# clocks: sample nvidia-smi DURING the timed regions
# ------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.idx = [], None, gpu_index
        self.marks = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def mark(self, t0, t1):
        self.marks.append((t0, t1))

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ts, line in self.rows:
            if not any(a <= ts <= b for a, b in self.marks):
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------
# workload
# ------------------------------------------------------------------------------------------------------------
def cache_dir(args):
    return os.path.join(args.cache_dir, f"kuq_bench_r{args.db_records or 666_000_000}_g{args.genomes}_k{K}m{NT}")


def write_fastq(path, bases: np.ndarray, n_reads: int):
    """n_reads x 150 ASCII bases → FASTQ with fixed-width records (vectorised)."""
    width = 10
    hdr = np.char.zfill(np.arange(n_reads).astype("U"), width)
    rec_len = 1 + 1 + width + 1 + READ_LEN + 1 + 2 + READ_LEN + 1
    out = np.empty((n_reads, rec_len), np.uint8)
    out[:, 0] = ord("@"); out[:, 1] = ord("r")
    out[:, 2:2 + width] = np.frombuffer("".join(hdr.tolist()).encode(), np.uint8).reshape(n_reads, width)
    p = 2 + width
    out[:, p] = ord("\n"); p += 1
    out[:, p:p + READ_LEN] = bases[:n_reads * READ_LEN].reshape(n_reads, READ_LEN); p += READ_LEN
    out[:, p] = ord("\n"); out[:, p + 1] = ord("+"); out[:, p + 2] = ord("\n"); p += 3
    out[:, p:p + READ_LEN] = ord("I"); p += READ_LEN
    out[:, p] = ord("\n")
    out.tofile(path)


def ensure_files(args, db, sample_bases_host):
    """database.kdb / database.idx / taxDB / sample FASTQ for the reference binary, cached in tmpfs."""
    d = cache_dir(args)
    done = os.path.join(d, "COMPLETE")
    fq = os.path.join(d, f"sample_{args.cpu_sample_reads}.fq")
    if not os.path.exists(done):
        os.makedirs(d, exist_ok=True)
        db.write_files(os.path.join(d, "database.kdb"), os.path.join(d, "database.idx"))
        db.write_taxdb(os.path.join(d, "taxDB"))
        open(done, "w").write("ok\n")
    if not os.path.exists(fq):
        write_fastq(fq, sample_bases_host, args.cpu_sample_reads)
    return d, fq


def run_reference_classify(d, fq_files, threads):
    """Run the UNMODIFIED reference (oracle/_ref/classify -M) and parse its own stats line
    (classify.cpp:361-375): returns (n_sequences, seconds)."""
    exe = os.path.join(ROOT, "oracle", "_ref", "classify")
    cmd = [exe, "-d", os.path.join(d, "database.kdb"), "-i", os.path.join(d, "database.idx"), "-a",
           os.path.join(d, "taxDB"), "-M", "-t", str(threads), "-o", "/dev/null"] + list(fq_files)
    env = dict(os.environ, OMP_NUM_THREADS=str(threads))
    r = subprocess.run(cmd, capture_output=True, text=True, env=env)
    m = re.search(r"(\d+) sequences \(([\d.]+) Mbp\) processed in ([\d.]+)s", r.stderr)
    if r.returncode != 0 or not m:
        raise RuntimeError(f"reference classify failed ({r.returncode}): {r.stderr[-1500:]}")
    return int(m.group(1)), float(m.group(3))


def host_threads(args=None):
    if args is not None and getattr(args, "cpu_threads", 0) > 0:
        return args.cpu_threads
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


# ------------------------------------------------------------------------------------------------------------
def warm_collectives(dist, dev, world):
    """NCCL builds its all-to-all / all-reduce channels on first use: do that before anything is timed"""
    import torch
    wa = torch.zeros(world * 1024, dtype=torch.int64, device=dev)
    wb = torch.empty_like(wa)
    dist.all_to_all_single(wb, wa)
    for dt in (torch.uint8, torch.int32, torch.int64):
        t_ = torch.zeros(1024, dtype=dt, device=dev)
        dist.all_reduce(t_, op=dist.ReduceOp.MAX)
        dist.all_reduce(t_, op=dist.ReduceOp.SUM)
    torch.cuda.synchronize()


def resolve_mode(args, world):
    if args.mode != "auto":
        return args.mode
    return "shards" if world > 1 else "replicas"


def shard_db_records(args, world):
    """BASELINE configs[3]: a 300 GB database (25.0 G records) sharded by minimizer range.  Every card holds at most
    75 GB of records here (the generator sorts a range next to the finished records), so 2 cards run a 150 GB database;
    4 and 8 cards run the 300 GB one (75 / 37.5 GB per card)."""
    if args.db_records:
        return args.db_records
    return min(25_000_000_000, world * 6_250_000_000)


class Workload:
    pass


def build_workload(args, mode, rank, world, dev, dist, n_steps):
    import torch
    from krakenuniq_b200 import synth_gpu
    w = Workload()
    t_gen = time.time()
    sharded = mode == "shards" and world > 1
    records = shard_db_records(args, world) if sharded else (args.db_records or 666_000_000)
    passes = args.db_passes or (max(1, -(-records // world // 600_000_000)) if sharded else max(1, records // 1_500_000_000))
    torch.cuda.reset_peak_memory_stats()
    w.db = synth_gpu.GpuDatabase(records, n_genomes=args.genomes, k=K, nt=NT, seed=2, device=dev, passes=passes,
                                 shard=(rank, world) if sharded else None)
    # every step classifies reads no earlier step has seen (a re-classified read finds its records already flagged /
    # its sparse-tier keys already stored and would be cheaper): the pool covers all steps of the run
    w.n_pool = max(args.reads, args.batch_reads * n_steps)
    # replicas: every rank draws its own reads (seed + rank), reads are partitioned across GPUs;
    # shards: every GPU scans the same reads
    w.pool_bases, _ = w.db.sample_reads(w.n_pool, READ_LEN, seed=3 + (0 if sharded else 1000 * rank))
    torch.cuda.synchronize()
    w.gen_s = time.time() - t_gen
    w.gen_peak_gb = torch.cuda.max_memory_allocated() / 1e9
    total_records = w.db.key_ct
    if sharded:
        t = torch.tensor([w.db.key_ct], device=dev, dtype=torch.int64)
        dist.all_reduce(t)
        total_records = int(t.item())
    tag = "configs[1]" if records == 666_000_000 and not sharded else ("configs[3]" if sharded and records == 25_000_000_000 else
                                                                       ("scaled configs[3]" if sharded else "scaled configs[1]"))
    w.workload = (f"{tag}: {total_records * 12 / 1e9:.1f} GB synthetic KrakenDB (k={K}, m={NT}, {total_records} records) "
                  f"+ {8 * ((1 << (2 * NT)) + 1) / 1e9:.1f} GB index in HBM, {w.n_pool} x {READ_LEN} bp reads, "
                  f"{args.batch_reads} reads per step")
    w.records = records
    return w


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference" and rank != 0:
        return 0                                              # rank 0 alone runs the CPU reference
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU (workload generation and the product path are CUDA only)")
    torch.cuda.set_device(local_rank)
    dev = f"cuda:{local_rank}"
    dist = None
    if world > 1 and args.impl == "ours":
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group("nccl", device_id=torch.device(dev))
    mode = resolve_mode(args, world if args.impl == "ours" else 1)
    if args.dump_outputs and (args.impl != "ours" or mode != "replicas"):
        raise SystemExit("--dump-outputs writes the outputs of our replicas layout (--impl ours, one GPU or --mode replicas)")
    B = args.batch_reads
    steps_rep = (args.warmup + args.steps) + 5 + (max(args.warmup, 3) + args.steps)

    # ---------------- reference arm: the unmodified reference on the host cores ------------------------------
    if args.impl == "reference":
        w = build_workload(args, "replicas", 0, 1, dev, None, 1)
        db, pool_bases, workload = w.db, w.pool_bases, w.workload
        threads = host_threads(args)
        sample = pool_bases[:args.cpu_sample_reads * READ_LEN].cpu().numpy()
        d, fq = ensure_files(args, db, sample)
        del db, pool_bases
        torch.cuda.empty_cache()
        if args.warmup > 0:
            run_reference_classify(d, [fq] * min(args.warmup, 1), threads)      # warms the page cache (run-fq.sh:19)
        n_seq, secs = run_reference_classify(d, [fq] * args.steps, threads)
        v = n_seq / secs / 1e6
        line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "Mreads/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": secs / args.steps * 1e3,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
                "config": {"workload": workload, "sample": f"{args.cpu_sample_reads} reads per step (FASTQ in tmpfs)"},
                "cpu_baseline": {"value": v, "unit": "Mreads/s", "cores": threads, "kind": "reference",
                                 "sample": f"oracle/_ref/classify -M -t {threads} -o /dev/null, {args.steps} x "
                                           f"{args.cpu_sample_reads} reads, time from its own stats line "
                                           "(DB load excluded, FASTQ parsing + Kraken output formatting included)"},
                "e2e": {"value": v, "unit": "Mreads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    # ---------------- our arm ----------------------------------------------------------------------------------
    if mode == "stream":
        if world > 1:
            raise SystemExit("--mode stream is the one-GPU layout (a database larger than HBM); several GPUs shard it instead")
        return run_stream(args, local_rank, dev)
    line, rep_line, cpu_baseline = None, None, None
    if mode == "replicas" or (args.mode == "auto" and world > 1):
        w = build_workload(args, "replicas", rank, world, dev, dist, steps_rep)
        cpu_baseline = measure_cpu_baseline(args, w, rank)
        rep_line = run_replicas(args, w, rank, world, local_rank, dev, dist, cpu_baseline)
        del w
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        line = rep_line
    if mode == "shards":
        w = build_workload(args, "shards", rank, world, dev, dist, 2 * (args.warmup + args.steps) + 6)
        extra = None
        if rep_line is not None:
            keep = ("value", "ms_per_step", "scaling", "e2e", "gpu_launches")
            extra = {"replicas": dict({k: rep_line[k] for k in keep}, workload=rep_line["config"]["workload"],
                                      end_of_run_merge_ms=rep_line["config"]["end_of_run_merge_ms"],
                                      note="second layout, same run: the configs[1] database replicated on every GPU, reads "
                                           "partitioned (weak scaling); merge of the per-taxon state timed separately")}
        line = run_shards(args, w.db, w.pool_bases, rank, world, local_rank, dev, dist, w.workload, w.gen_s, cpu_baseline, extra)
        if line is not None:
            line["config"]["workload_gen_peak_gb"] = w.gen_peak_gb
    if rank == 0 and line is not None:
        print(json.dumps(line))
    if dist:
        dist.destroy_process_group()
    return 0


def measure_cpu_baseline(args, w, rank):
    """the unmodified reference on the host cores, rank 0 only, on a bounded sample of the configs[1] workload"""
    db, pool_bases = w.db, w.pool_bases
    cpu_baseline = None
    if rank == 0 and not args.no_cpu_baseline and os.path.exists(os.path.join(ROOT, "oracle", "_ref", "classify")):
        try:
            threads = host_threads(args)
            sample = pool_bases[:args.cpu_sample_reads * READ_LEN].cpu().numpy()
            d, fq = ensure_files(args, db, sample)                 # must precede attach (values still raw taxids)
            run_reference_classify(d, [fq], threads)               # warm-up (page cache, run-fq.sh:19)
            n_files = 4                                            # same protocol as the reference arm: several files per run
            n_seq, secs = run_reference_classify(d, [fq] * n_files, threads)
            cpu_baseline = {"value": n_seq / secs / 1e6, "unit": "Mreads/s", "cores": threads, "kind": "reference",
                            "sample": f"oracle/_ref/classify -M -t {threads} -o /dev/null on {n_files} x {args.cpu_sample_reads} "
                                      "reads of the same workload (FASTQ in tmpfs), after one warm-up run; time from its own "
                                      "stats line (DB load excluded, FASTQ parsing + Kraken formatting included) — the "
                                      "reference arm's protocol"}
        except Exception as e:  # noqa: BLE001
            cpu_baseline = {"value": None, "unit": "Mreads/s", "cores": host_threads(), "kind": "reference",
                            "sample": f"failed: {e}"[:300]}

    return cpu_baseline


DUMP_READS = 1 << 20          # per-read outputs of every read of the step, or of a seeded sample of this many
DUMP_HIT_READS = 1 << 16      # hit lists of a seeded sample of this many of those reads


def dump_outputs(out_dir, clf, n_reads, offsets):
    """What the caller of the timed path receives from its last step — per-read calls (taxids), window counts and
    run-length hit lists of the batch in slot 0 (kuq_collect_device_batch) — and the per-taxon counters of the run
    (kuq_read_counts), as float64 / float32 .npy files in out_dir, 64 MB at most."""
    from krakenuniq_b200 import binding
    res = binding.BatchResult()
    clf._ck(clf.L.kuq_collect_device_batch(clf.h, 0, ctypes.byref(res)))
    r = clf._result(res, offsets)
    rng = np.random.default_rng(0)
    reads = np.arange(n_reads) if n_reads <= DUMP_READS else np.sort(rng.choice(n_reads, DUMP_READS, replace=False))
    hit_reads = np.sort(rng.choice(reads, min(len(reads), DUMP_HIT_READS), replace=False))
    start = r["run_start"][hit_reads].astype(np.int64)
    count = r["run_count"][hit_reads].astype(np.int64)
    runs = np.repeat(start - (np.cumsum(count) - count), count) + np.arange(int(count.sum()))
    cnt = clf.counts()
    arrays = {"read_index": reads.astype(np.float64), "call": r["call"][reads].astype(np.float64),
              "n_windows": r["n_windows"][reads].astype(np.float32),
              "hit_read_index": hit_reads.astype(np.float64), "hit_run_count": count.astype(np.float64),
              # one row per run: (taxid, or 0xFFFFFFFF for ambiguous windows; number of windows)
              "hit_runs": r["runs"][runs].astype(np.float64)}
    arrays.update({f"taxon_{k}": cnt[k].astype(np.float64) for k in ("taxid", "n_reads", "n_kmers", "unique")})
    total = sum(a.nbytes for a in arrays.values())
    if total > 64 << 20:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the 64 MB budget")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_replicas(args, w, rank, world, local_rank, dev, dist, cpu_baseline):
    """SURVEY §8(e).1: the database fits one card — every GPU holds it, reads are partitioned (weak scaling)."""
    import torch
    from krakenuniq_b200 import binding
    db, pool_bases, n_pool, workload, gen_s = w.db, w.pool_bases, w.n_pool, w.workload, w.gen_s
    B = args.batch_reads
    n_batches = n_pool // B
    # sparse-tier set sized for the worst case of this workload (no taxon ever converts: one key per database record)
    clf = binding.Classifier(device=local_rank, n_slots=3, max_reads=B, max_bases=B * READ_LEN + 4096,
                             hll_mode=args.hll_mode, sparse_set_slots=1 << 31)
    clf.attach_db_device(db.records.data_ptr(), db.key_ct, db.offsets.data_ptr(), K, NT, 2)
    clf.set_taxonomy(*db.parent_map())

    d_offsets = (torch.arange(B + 2, dtype=torch.int64, device=dev) * READ_LEN)   # +1: slices are copied in 16-byte units
    # work units as process_file cuts them (classify.cpp:514-520): reads join a unit until it holds >= 500000 nt;
    # every batch starts a fresh unit (a batch = one input file of the reference)
    per_unit = -(-500000 // READ_LEN)
    units_per_batch = -(-B // per_unit)
    unit_local = (torch.arange(B, dtype=torch.int64, device=dev) // per_unit).to(torch.int32)
    host_unit_local = (np.arange(B, dtype=np.int64) // per_unit).astype(np.uint32)
    unit_bufs = {}

    def d_units(step_idx):
        if args.hll_mode != 0:
            return None
        t = unit_local + step_idx * units_per_batch
        unit_bufs[step_idx % 8] = t              # keep alive until the kernels have run
        return t.data_ptr()

    def h_units(step_idx):
        return (host_unit_local + np.uint32(step_idx * units_per_batch)) if args.hll_mode == 0 else None
    host_offsets = (np.arange(B + 1, dtype=np.uint64) * READ_LEN)

    def batch_ptr(i):
        return pool_bases.data_ptr() + (i % n_batches) * B * READ_LEN        # 16-byte aligned: B*150 % 16 == 0

    assert (B * READ_LEN) % 16 == 0 or n_batches == 1
    stream = torch.cuda.ExternalStream(clf.slot_stream(0), device=dev)
    sampler = ClockSampler(local_rank)
    sampler.start()

    def barrier():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    if dist:
        warm_collectives(dist, dev, world)

    def merge_state():
        """end-of-run merge across replicas (SURVEY §8(e).1): NCCL allreduce MAX/SUM + sparse-tier union"""
        if dist:
            from krakenuniq_b200 import dist as kdist
            kdist.merge_classifier_state_partitioned(clf, dev)

    # ---- value: device-resident inputs ----------------------------------------------------------------------------
    # one slot (stream): alternating the batches over two slots was measured 25 % SLOWER per step (4.67 vs 3.70 ms) —
    # the lookups of one batch and the scan / resolve of its neighbours evict each other's sectors from L2
    step = 0
    for _ in range(args.warmup):
        clf.classify_device(0, batch_ptr(step), d_offsets.data_ptr(), B, B * READ_LEN, d_units(step)); step += 1
    clf.sync(0)
    clf.finish()                                  # the warm-up's flagged records are harvested outside the timed region
    if dist:                                      # rehearsal of the cross-rank merge (first-use costs of NCCL / allocators)
        merge_state()
        clf.reset_counts()
        # one more untimed step: like at N = 1, the timed steps start with the run's start-up behind them (the misses'
        # taxon converts to dense in the first batch of any run)
        clf.classify_device(0, batch_ptr(step), d_offsets.data_ptr(), B, B * READ_LEN, d_units(step)); step += 1
        clf.sync(0)
        clf.finish()
    barrier()
    launches0 = clf.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kernel_ms = []
    t0 = time.time()
    with torch.cuda.stream(stream):
        ev0.record(stream)
    for _ in range(args.steps):
        clf.classify_device(0, batch_ptr(step), d_offsets.data_ptr(), B, B * READ_LEN, d_units(step)); step += 1
    # end of the run: the records flagged by the K steps become sparse-tier keys (kuq_finish) — part of the job, so
    # inside the timed region
    clf.finish()
    with torch.cuda.stream(stream):
        ev1.record(stream)
    clf.sync(0)
    barrier()
    harvest_ms_value = clf.sparse_tier_info()["last_harvest_ms"]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, clf, B, host_offsets)
    sampler.mark(t0, time.time())
    launches = clf.launch_count() - launches0
    dev_ms = ev0.elapsed_time(ev1)
    if dist:
        t = torch.tensor([dev_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms = float(t.item())
    value = world * B * args.steps / (dev_ms / 1e3) / 1e6

    # per-launch duration of the dominant kernel + algorithmic bytes (one extra, untimed, instrumented step)
    clf.classify_device(0, batch_ptr(step), d_offsets.data_ptr(), B, B * READ_LEN, d_units(step), flags=binding.F_STATS); step += 1
    clf.sync(0)
    n_lookups, sum_probes = clf.slot_stats(0)
    # SURVEY §8(d): B_kmer = 16 + 12*P(n_b) + 1 per non-ambiguous k-mer, B_read = L + 4 + 4*(L-30) per read
    algo_bytes = 17 * n_lookups + 12 * sum_probes + B * (READ_LEN + 4 + 4 * (READ_LEN - 30))
    k_ms, st_ms = [], []
    for _ in range(3):
        clf.classify_device(0, batch_ptr(step), d_offsets.data_ptr(), B, B * READ_LEN, d_units(step)); step += 1
        clf.sync(0)
        k_ms.append(clf.last_kernel_ms(0))
        st_ms.append(clf.last_stage_ms(0))
    st_ms = np.mean(np.array(st_ms), axis=0)
    kern_ms = float(st_ms[1])            # k_lookup: the random-HBM stage dominates the step
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = algo_bytes / (kern_ms / 1e3) / 1e9
    traffic, traffic_src = None, None
    try:    # DRAM bytes per launch of the same kernel on the same workload, from the committed ncu capture of THIS build
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic_r02.json")))
        if w.records == 666_000_000 and B == 1_000_000:
            e = tj["k_lookup_dense_only" if args.hll_mode == 2 else "k_lookup_exact_hll"]
            traffic = e["dram_bytes"]
            traffic_src = {"capture": e["capture"], "kernel_ms_in_capture": e["kernel_ms"], "build": tj.get("build")}
    except Exception:
        pass
    # second roofline (SURVEY.md §8(d)): random 32-byte-sector gathers, measured here with k_lookup's launch shape
    gather = None
    try:
        gs, gb, gms = binding.random_gather_peak(local_rank, 16 << 30, 1 << 29, 32)
        sectors = n_lookups + sum_probes                       # 32*(1+P) bytes per looked-up k-mer
        gather = {"random_gather_peak": gb, "unit": "GB/s of 32 B sectors", "gsectors_per_s": gs,
                  "algorithmic_sectors_per_launch": int(sectors),
                  "frac_random": 32.0 * sectors / (kern_ms / 1e3) / 1e9 / gb,
                  "how": "kuq_random_gather_peak: independent loads at hashed sector addresses of a 16 GB buffer, 256 threads x "
                         "8 CTAs/SM, best of 3; frac_random = 32*(1+P)*lookups / kernel time / this peak.  It exceeds 1 when "
                         "consecutive windows share a minimizer bin (their sectors come from L1/L2, not DRAM)"}
    except Exception as e:  # noqa: BLE001
        gather = {"random_gather_peak": None, "error": str(e)[:200]}
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src, "kernel": "k_lookup<MODE_FUSED>", "kernel_ms": kern_ms,
                "stage_ms": {"k_scan": float(st_ms[0]), "k_lookup": float(st_ms[1]), "k_resolve": float(st_ms[2])},
                "algorithmic_bytes_per_launch": algo_bytes, "bytes_per_read": algo_bytes / B,
                "random": gather,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (copy bandwidth, of measured)" if peaks else "fallback 6650 GB/s"}

    # ---- e2e: host buffers through the C ABI, H2D + D2H inside the timed region ------------------------------------
    # pinned host copies of the batches the e2e steps will classify (each batch once: no step re-sees reads)
    n_e2e = max(args.warmup, 3) + args.steps
    first = step % n_batches
    n_host = min(n_batches, n_e2e)
    host_bufs = []
    for i in range(n_host):
        p = clf.L.kuq_host_alloc(B * READ_LEN + 64)
        hb = np.ctypeslib.as_array(ctypes.cast(p, ctypes.POINTER(ctypes.c_uint8)), shape=(B * READ_LEN + 64,))
        b = (first + i) % n_batches
        hb[:B * READ_LEN] = pool_bases[b * B * READ_LEN:(b + 1) * B * READ_LEN].cpu().numpy()
        host_bufs.append((p, hb))
    n_slots = 3
    d2h_bytes = [0]
    sanity = {"reads": 0, "classified": 0}
    e2e_step = [step]

    e2e_buf = [0]

    def run_e2e(n_steps):
        inflight = []
        for s in range(n_steps):
            slot = s % n_slots
            if len(inflight) == n_slots:
                res = clf.wait(inflight.pop(0))
                d2h_bytes[0] = 4 * B * 4 + 8 * res["n_runs"] + 64
                sanity["reads"] += B; sanity["classified"] += res["n_classified"]
            clf.submit(slot, host_bufs[e2e_buf[0] % n_host][0], host_offsets, h_units(e2e_step[0])); e2e_step[0] += 1
            e2e_buf[0] += 1
            inflight.append(slot)
        for slot in inflight:
            res = clf.wait(slot)
            d2h_bytes[0] = 4 * B * 4 + 8 * res["n_runs"] + 64
            sanity["reads"] += B; sanity["classified"] += res["n_classified"]

    run_e2e(max(args.warmup, 3))
    clf.finish()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    e0.record()
    run_e2e(args.steps)
    clf.finish()                                  # harvest of the run's flagged records: part of the job
    torch.cuda.synchronize()
    e1.record()
    torch.cuda.synchronize()
    e2e_ms = e0.elapsed_time(e1)
    barrier()
    sampler.mark(t0, time.time())
    if dist:
        t = torch.tensor([e2e_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    e2e_value = world * B * args.steps / (e2e_ms / 1e3) / 1e6
    # end-of-run merge of the per-taxon state across ranks: once per run, not per step — timed on its own
    merge_ms = 0.0
    if dist:
        barrier()
        tm0 = torch.cuda.Event(enable_timing=True); tm1 = torch.cuda.Event(enable_timing=True)
        tm0.record(); merge_state(); tm1.record(); torch.cuda.synchronize()
        t = torch.tensor([tm0.elapsed_time(tm1)], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        merge_ms = float(t.item())
    clocks = sampler.stop()
    for p, _ in host_bufs:
        clf.L.kuq_host_free(p)

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "Mreads/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u64", "data": "synthetic",
                "config": {"workload": workload, "parallelism": f"replicas x{world} (reads partitioned, DB replicated)",
                           "l2": "inputs larger than L2: 150 MB of reads per step, 16.6 GB database probed at random",
                           "hll_mode": ["preload rule", "chunked rule", "dense only"][args.hll_mode],
                           "timing": "CUDA events on the slot stream around K steps + the end-of-run harvest (kuq_finish), max over "
                                     "ranks; the once-per-run NCCL merge of the per-taxon state across ranks is timed separately",
                           "end_of_run_merge_ms": merge_ms,
                           "value_including_merge": world * B * args.steps / ((dev_ms + merge_ms) / 1e3) / 1e6,
                           "steps_only_mreads_s": world * B * args.steps / (max(dev_ms - harvest_ms_value, 1e-3) / 1e3) / 1e6,
                           "harvest_ms_in_timed_region": harvest_ms_value,
                           "read_pool": f"{n_pool} reads: every step of the run classifies reads no earlier step saw",
                           "sparse_tier": clf.sparse_tier_info(),
                           "workload_gen_s": gen_s},
                "roofline": roofline,
                "cpu_baseline": cpu_baseline,
                "e2e": {"value": e2e_value, "unit": "Mreads/s", "h2d_bytes_per_step": B * READ_LEN + 8 * (B + 1),
                        "d2h_bytes_per_step": int(d2h_bytes[0]), "ms_per_step": e2e_ms / args.steps,
                        "how": "kuq_submit_batch/kuq_wait_batch over 3 slots, pinned host reads, results = calls + "
                               "window counts + RLE hit lists"},
                "gpu_launches": int(launches),
                "sanity": {"classified_fraction": sanity["classified"] / max(sanity["reads"], 1),
                           "expected": "about 0.80: 80 % of the reads are sampled from the database genomes (1 % substitutions)"},
                "clocks": clocks}
        return line
    return None


def run_shards(args, db, pool_bases, rank, world, local_rank, dev, dist, workload, gen_s, cpu_baseline=None, extra=None):
    """SURVEY §8(e).2 / BASELINE configs[3]: the database is split into `world` minimizer ranges (balanced by records,
    like prepare_chunking); every GPU scans the SAME batch and looks up the k-mers whose minimizer it owns; read r is
    resolved by one owner GPU.  Per step, all in stream order on each GPU — no host barrier inside the loop:
        wait(ready)  → fused lookup + NVLink peer scatter of the hits (the finder also does the hit's sketch work)
        signal(done) → wait(done) → resolve own share from the merged ids → zero own buffer → signal(ready)
    `--merge nccl` replaces the peer scatter by a MAX all-reduce of the id buffers (stream-ordered NCCL).
    End of run: code-partitioned merge of the per-taxon state (dist.merge_classifier_state_partitioned).
    value = reads of the job / (time of the K steps + the end-of-run merge)."""
    import torch
    from krakenuniq_b200 import binding
    from krakenuniq_b200 import dist as kdist
    B = args.batch_reads
    n_pool = pool_bases.numel() // READ_LEN if pool_bases.numel() % READ_LEN == 0 else (pool_bases.numel() - 64) // READ_LEN
    n_batches = n_pool // B
    lo_bin, hi_bin = db.bin_lo, db.bin_hi
    # the owner of a code keeps its keys after the merge: at most one per record of the whole database / world
    want_slots = 1 << 26
    while want_slots < (1 << 31) and want_slots < 2.5 * min(db.key_ct, (args.warmup + args.steps) * B * 100 / world):
        want_slots <<= 1
    clf = binding.Classifier(device=local_rank, n_slots=2, max_reads=B, max_bases=B * READ_LEN + 4096,
                             hll_mode=args.hll_mode, sparse_set_slots=want_slots)
    clf.set_db_taxid_universe(np.array(db.species, np.uint32))
    clf.attach_db_device(db.records.data_ptr(), db.key_ct, db.offsets.data_ptr(), K, NT, 2, lo_bin, hi_bin)
    clf.set_taxonomy(*db.parent_map())
    clf.set_shard_counting(args.merge == "p2p")
    per_unit = -(-500000 // READ_LEN)
    n_units = -(-B // per_unit)                                  # owner shares: whole work units, contiguous
    share_units = [kdist.partition(n_units, world, r) for r in range(world)]
    shares = [(min(a * per_unit, B), min(b * per_unit, B)) for a, b in share_units]
    lo, hi = shares[rank]
    assert lo % 2 == 0
    d_offsets = (torch.arange(B + 2, dtype=torch.int64, device=dev) * READ_LEN)
    unit_local = (torch.arange(B, dtype=torch.int64, device=dev) // per_unit).to(torch.int32)
    total = B * READ_LEN
    nbytes = (total + 64) * 4
    bounds = np.array([s_[0] * READ_LEN for s_ in shares] + [total], np.uint64)
    bounds[0] = 0
    own_off, own_len = int(bounds[rank]) * 4, (int(bounds[rank + 1]) - int(bounds[rank])) * 4
    bufs = [clf.device_alloc(nbytes) for _ in range(2)]           # double buffered by step parity
    flags = clf.device_alloc(256)                                 # [0:8) done counters, [16:24) ready counters (u64)
    flags_t = kdist.device_view(flags, 256, torch.int64, dev)
    flags_t.zero_()
    flags_t[16:24] = 2                                            # both buffers are clean for steps 0 and 1
    for b_ in bufs:
        clf.device_memset(0, b_, 0, nbytes)
    clf.sync(0)
    torch.cuda.synchronize()
    peers_buf, peers_done, peers_ready, opened = [bufs, bufs], None, None, []
    if args.merge == "p2p":
        handles = [None] * world
        dist.all_gather_object(handles, (clf.ipc_export(bufs[0]), clf.ipc_export(bufs[1]), clf.ipc_export(flags)))
        pb0, pb1, pf = [], [], []
        for r in range(world):
            if r == rank:
                pb0.append(bufs[0]); pb1.append(bufs[1]); pf.append(flags)
            else:
                m = [clf.ipc_open(h) for h in handles[r]]
                opened += m
                pb0.append(m[0]); pb1.append(m[1]); pf.append(m[2])
        peers_buf = [pb0, pb1]
        peers_done = pf                                           # flag arrays start with the done counters
        peers_ready = [p + 128 for p in pf]
    bufs_t = [kdist.device_view(b_, nbytes, torch.int32, dev) for b_ in bufs]
    stream = torch.cuda.ExternalStream(clf.slot_stream(0), device=dev)
    dist.barrier()                                                # once: every rank's buffers and flags exist
    warm_collectives(dist, dev, world)
    # merge buffers, allocated once: a rank exports at most one key per hit it found (+ its misses' keys), and receives
    # about as many
    n_run_steps = args.warmup + args.steps
    key_bound = int(min(db.key_ct + (1 << 26), 1.3 * n_run_steps * B * 100 / world + (1 << 26)))
    merge_bufs = (torch.empty(key_bound, dtype=torch.int64, device=dev), torch.empty(key_bound, dtype=torch.int64, device=dev))
    keep = {}

    def step(i, bptr=None):
        if bptr is None:
            bptr = pool_bases.data_ptr() + (i % n_batches) * B * READ_LEN
        par = i & 1
        if args.merge == "p2p":
            clf.wait_flags(0, flags + 128, world, i + 1)          # every owner has zeroed its buffer of this parity
            clf.lookup_device_peers(0, bptr, d_offsets.data_ptr(), B, total, peers_buf[par], bounds)
            clf.signal_peers(0, peers_done, rank, i + 1)
            clf.wait_flags(0, flags, world, i + 1)                # every GPU's hits for my reads have landed
        else:
            clf.lookup_device(0, bptr, d_offsets.data_ptr(), B, total, bufs[par], only_hits=1)
            with torch.cuda.stream(stream):
                dist.all_reduce(bufs_t[par], op=dist.ReduceOp.MAX)
        if hi > lo:
            u = unit_local[lo:hi] + i * n_units
            keep[i % 4] = u
            clf.resolve_device(0, bptr, d_offsets.data_ptr() + lo * 8, hi - lo, total, bufs[par],
                               u.data_ptr() if args.hll_mode == 0 else None)
        if args.merge == "p2p":
            clf.device_memset(0, bufs[par] + own_off, 0, own_len)
            clf.signal_peers(0, peers_ready, rank, i + 3)
        else:
            clf.device_memset(0, bufs[par], 0, nbytes)

    sampler = ClockSampler(local_rank)
    sampler.start()
    s = 0
    for _ in range(args.warmup):
        step(s); s += 1
    clf.sync(0); torch.cuda.synchronize(); dist.barrier()
    # dress rehearsal of the end-of-run merge on the warm-up's state: NCCL sets up its all-to-all channels for real message
    # sizes and the allocators see the big buffers once (both are first-use costs of a process, not of a run); then the
    # state is wiped — the timed run starts like a fresh run
    kdist.merge_classifier_state_partitioned(clf, dev, buffers=merge_bufs)
    clf.reset_counts()
    step(s); s += 1                               # one more untimed step: the run's start-up (the misses' taxon converts to
    clf.sync(0)                                   # dense in the first batch of any run) stays outside, as at N = 1
    torch.cuda.synchronize(); dist.barrier()
    ev0, ev1, ev2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    t0 = time.time()
    launches0 = clf.launch_count()
    with torch.cuda.stream(stream):
        ev0.record(stream)
    for _ in range(args.steps):
        step(s); s += 1
    with torch.cuda.stream(stream):
        ev1.record(stream)
    clf.sync(0)
    tm = {}
    kdist.merge_classifier_state_partitioned(clf, dev, timings=tm, buffers=merge_bufs)
    with torch.cuda.stream(stream):
        ev2.record(stream)
    clf.sync(0); torch.cuda.synchronize(); dist.barrier()
    sampler.mark(t0, time.time())
    ms = torch.tensor([ev0.elapsed_time(ev1), ev0.elapsed_time(ev2)], device=dev, dtype=torch.float64)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    steps_ms, run_ms = float(ms[0].item()), float(ms[1].item())
    launches = clf.launch_count() - launches0
    st = clf.last_stage_ms(0)
    cnt = clf.counts()

    # ---- e2e: the same steps with HOST buffers — every GPU copies the batch from pinned host memory (copy stream,
    # double buffered against the step before) and reads its share's calls / window counts / hit lists back ----------
    dres = clf.device_result(0)
    n_own = hi - lo
    copy_stream = torch.cuda.Stream(device=dev)
    n_e2e = args.warmup + args.steps + 1
    h_in = [torch.empty(total + 64, dtype=torch.uint8).pin_memory() for _ in range(min(n_e2e, n_batches))]
    first_b = s % n_batches
    for j, hb in enumerate(h_in):
        b_ = (first_b + j) % n_batches
        hb[:total].copy_(pool_bases[b_ * total:(b_ + 1) * total])
        hb[total:] = ord("N")
    d_in = [torch.empty(total + 64, dtype=torch.uint8, device=dev) for _ in range(2)]
    ev_copied = [torch.cuda.Event() for _ in range(2)]
    ev_free = [torch.cuda.Event() for _ in range(2)]
    h_out = torch.empty(4 * max(n_own, 1) + 2, dtype=torch.int32).pin_memory()
    h_runs = torch.empty((total // 2 + 64, 2), dtype=torch.int32).pin_memory()
    views = None
    if n_own:
        views = [kdist.device_view(dres.d_call, n_own * 4, torch.int32, dev), kdist.device_view(dres.d_n_windows, n_own * 4, torch.int32, dev),
                 kdist.device_view(dres.d_run_start, n_own * 4, torch.int32, dev), kdist.device_view(dres.d_run_count, n_own * 4, torch.int32, dev)]
        runs_v = kdist.device_view(dres.d_runs, (total // 2 + 64) * 8, torch.int32, dev).view(-1, 2)
        nruns_v = kdist.device_view(dres.d_n_runs, 8, torch.int64, dev)
    d2h = [0]
    est_runs = [min(8 * n_own + 64, total // 2)]

    def step_e2e(i, j):
        par = j & 1
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(ev_free[par])
            d_in[par].copy_(h_in[j % len(h_in)], non_blocking=True)
            ev_copied[par].record(copy_stream)
        stream.wait_event(ev_copied[par])
        step(i, d_in[par].data_ptr())
        with torch.cuda.stream(stream):
            ev_free[par].record(stream)
            if n_own:
                for q_, v in enumerate(views):
                    h_out[q_ * n_own:(q_ + 1) * n_own].copy_(v, non_blocking=True)
                h_runs[:est_runs[0]].copy_(runs_v[:est_runs[0]], non_blocking=True)
        d2h[0] = 16 * n_own + 8 * est_runs[0]

    for ev in ev_free:
        ev.record(stream)
    j = 0
    for _ in range(args.warmup):
        step_e2e(s, j); s += 1; j += 1
    clf.sync(0); torch.cuda.synchronize()
    if n_own:
        est_runs[0] = min(int(nruns_v.item()) + 4096, total // 2)      # hit-list volume of a step (same workload every step)
    clf.reset_counts()
    step_e2e(s, j); s += 1; j += 1                # start-up step of the fresh state, untimed (see above)
    clf.sync(0)
    torch.cuda.synchronize(); dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t1 = time.time()
    with torch.cuda.stream(stream):
        e0.record(stream)
    for _ in range(args.steps):
        step_e2e(s, j); s += 1; j += 1
    clf.sync(0)
    kdist.merge_classifier_state_partitioned(clf, dev, buffers=merge_bufs)
    with torch.cuda.stream(stream):
        e1.record(stream)
    clf.sync(0); torch.cuda.synchronize(); dist.barrier()
    sampler.mark(t1, time.time())
    t_e2e = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    e2e_ms = float(t_e2e.item())
    d2h_t = torch.tensor([d2h[0]], device=dev, dtype=torch.int64)
    dist.all_reduce(d2h_t)

    # ---- roofline of the dominant kernel (k_lookup<MODE_LOOKUP> with peer scatter) on rank 0's range: one instrumented
    # step for the algorithmic bytes, one plain step with a sync after the lookup for its duration -------------------
    roofline = None
    if args.merge == "p2p":
        clf.set_stats(True)
        bptr = pool_bases.data_ptr() + (s % n_batches) * B * READ_LEN
        clf.wait_flags(0, flags + 128, world, s + 1)
        clf.lookup_device_peers(0, bptr, d_offsets.data_ptr(), B, total, peers_buf[s & 1], bounds)
        clf.sync(0)
        n_lookups, sum_probes = clf.slot_stats(0)
        clf.set_stats(False)
        lk_ms = clf.last_stage_ms(0)
        clf.signal_peers(0, peers_done, rank, s + 1)
        clf.wait_flags(0, flags, world, s + 1)
        clf.device_memset(0, bufs[s & 1] + own_off, 0, own_len)
        clf.signal_peers(0, peers_ready, rank, s + 3)
        s += 1
        k_ms = []
        for _ in range(2):
            bptr = pool_bases.data_ptr() + (s % n_batches) * B * READ_LEN
            clf.wait_flags(0, flags + 128, world, s + 1)
            clf.lookup_device_peers(0, bptr, d_offsets.data_ptr(), B, total, peers_buf[s & 1], bounds)
            clf.sync(0)
            k_ms.append(clf.last_stage_ms(0)[1])
            clf.signal_peers(0, peers_done, rank, s + 1)
            clf.wait_flags(0, flags, world, s + 1)
            clf.device_memset(0, bufs[s & 1] + own_off, 0, own_len)
            clf.signal_peers(0, peers_ready, rank, s + 3)
            s += 1
        clf.sync(0); torch.cuda.synchronize(); dist.barrier()
        kern_ms = float(np.mean(k_ms))
        # SURVEY §8(d) for this GPU's range: 17 B per looked-up window of the range + 12 B per probe + the windows' scratch
        # (12 B canonical k-mer + bin in) and 4 B out per hit are not counted: bin fetch + probes only, plus the read text share
        algo_bytes = 17 * n_lookups + 12 * sum_probes + (B * (READ_LEN + 4 + 4 * (READ_LEN - 30))) // world
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        roofline = {"bound": "hbm", "achieved": algo_bytes / (kern_ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                    "frac": algo_bytes / (kern_ms / 1e3) / 1e9 / peak, "traffic": None,
                    "kernel": "k_lookup<MODE_LOOKUP> (rank 0's minimizer range, hits stored over NVLink)", "kernel_ms": kern_ms,
                    "algorithmic_bytes_per_launch": int(algo_bytes), "lookups_in_range": int(n_lookups), "sum_probes": int(sum_probes),
                    "how": "SURVEY §8(d) per-unit bytes x the units of this GPU's range (17 B per window of the range + 12 B per "
                           "bisection probe + 1/world of the per-read bytes), kernel duration from CUDA events on the slot stream",
                    "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s"}
    clocks = sampler.stop()
    tot_reads = int(cnt["n_reads"].sum())
    unclassified = int(cnt["n_reads"][cnt["taxid"] == 0].sum())
    info = clf.sparse_tier_info()
    line = None
    if rank == 0:
        value = B * args.steps / (run_ms / 1e3) / 1e6
        line = {
            "metric": METRIC, "value": value, "unit": "Mreads/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": run_ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {"workload": workload, "parallelism": f"database sharded by minimizer range over {world} GPUs "
                       f"({db.key_ct * 12 / 1e9:.1f} GB of records on rank 0), every GPU scans every batch, the finder of a hit "
                       f"does its sketch work, id merge = {args.merge}",
                       "hll_mode": ["preload rule", "chunked rule", "dense only"][args.hll_mode],
                       "timing": "CUDA events on the slot stream around the K steps AND the end-of-run merge of the per-taxon "
                                 "state (run_ms); no host barrier inside the step loop (device flags over NVLink); max over ranks",
                       "l2": "inputs larger than L2: 150 MB of reads per step, the database ranges are probed at random",
                       "steps_ms": steps_ms, "run_ms": run_ms, "end_of_run_merge_ms": run_ms - steps_ms,
                       "steps_only_mreads_s": B * args.steps / (steps_ms / 1e3) / 1e6,
                       "merge": tm, "sparse_tier": info, "workload_gen_s": gen_s,
                       "owner_stage_ms_last_step": {"k_scan": st[0], "k_lookup(misses + merged ids)": st[1], "k_resolve": st[2]}},
            "roofline": roofline,
            "cpu_baseline": cpu_baseline,
            "e2e": {"value": B * args.steps / (e2e_ms / 1e3) / 1e6, "unit": "Mreads/s", "ms_per_step": e2e_ms / args.steps,
                    "h2d_bytes_per_step": world * (total + 64), "d2h_bytes_per_step": int(d2h_t.item()),
                    "how": "every GPU copies the whole batch from pinned host memory (copy stream, double buffered), runs the "
                           "sharded step through the C ABI, and copies its share's calls / window counts / RLE hit lists to pinned "
                           "host memory; the end-of-run merge is inside the timed region; max over ranks"},
            "sanity": {"reads_counted": tot_reads, "classified_fraction": 1.0 - unclassified / max(tot_reads, 1),
                       "expected": "about 0.80 (80 % of the reads come from the database genomes)"},
            "gpu_launches": int(launches), "clocks": clocks}
        if extra:
            line.update(extra)
    dist.barrier()
    for p_ in opened:
        clf.ipc_close(p_)
    dist.barrier()
    return line


def run_stream(args, local_rank, dev):
    """BASELINE configs[2] / configs[4]: a database larger than HBM on ONE GPU.  The records live in pinned host memory
    and travel over PCIe one minimizer range at a time into two device buffers (kuq_stream_*), the next range's copy
    overlapping the current range's lookups; per-window ids are merged on the device (hits only); the final pass
    resolves every batch.  The whole job is the timed region (DB traffic over PCIe included: it IS the hot path here);
    a 'step' is one batch of reads carried through all ranges and the final pass.  `--paired` = configs[4]: 2 x 150 bp
    mates merged `mate1 + N + mate2` (scripts/read_merger.pl:187-191); `--stream-both` runs configs[2] and configs[4]
    against one generated database.  HLL: the chunked rule, as the reference's -x path (classify.cpp:719)."""
    import torch
    from krakenuniq_b200 import binding, synth_gpu
    from krakenuniq_b200 import dist as kdist
    # The configurations are quoted on a 300 GB database (25 G records).  The whole database has to sit in pinned host
    # memory here, and this pool's boxes give a container 200 GiB of host memory (cgroup memory.max) — a 300 GB run
    # takes the box down.  Default = what is safe there: 60 GB of records in ranges of 6 GB (the behaviour is the same,
    # PCIe-bound: one pass moves the database once); --db-records 25000000000 --range-gb 24 is the real thing on a
    # host that has the memory, and the guard below refuses sizes the container cannot hold.
    records = args.db_records or 5_000_000_000
    range_gb = args.range_gb or (24.0 if records >= 20_000_000_000 else 6.0)
    need_host = records * 12 * 1.10 + (1 << (2 * NT)) * 8 + 2 * args.steps * args.batch_reads * READ_LEN * (2 if args.stream_both else 1) + (8 << 30)
    try:
        lim = open("/sys/fs/cgroup/memory.max").read().strip()
        lim = int(lim) if lim != "max" else None
    except Exception:
        lim = None
    if lim is not None and need_host > 0.7 * lim:
        raise SystemExit(f"bench.py --mode stream: about {need_host / 2**30:.0f} GiB of pinned host memory needed, the container "
                         f"allows {lim / 2**30:.0f} GiB: use a smaller --db-records / fewer --steps")
    # the generator builds the database in passes of <= ~0.9 G records (its sorts stay below 2^31 elements); a streamed
    # range is a run of consecutive passes
    passes = max(2, int(np.ceil(records / 0.9e9)))
    ppr = max(1, int((range_gb * 1e9 / 12) // (records / passes)))          # passes per streamed range
    variants = [False, True] if args.stream_both else [bool(args.paired)]
    n_batches = args.steps
    hll_mode = 2 if args.hll_mode == 2 else 1
    t_gen = time.time()
    db = synth_gpu.GpuDatabase(records, n_genomes=args.genomes, k=K, nt=NT, seed=2, device=dev, passes=passes, defer_build=True)
    host_pools = {}
    for paired in variants:                                 # reads first (they need the genome), parked in pinned host memory
        L = 2 * READ_LEN + 1 if paired else READ_LEN
        B = args.batch_reads // 2 if paired else args.batch_reads
        n_reads = n_batches * B
        if paired:
            mates, _ = db.sample_reads(2 * n_reads, READ_LEN, seed=5)
            pool = torch.full((n_reads * L + 64,), ord("N"), dtype=torch.uint8, device=dev)
            pv = pool[:n_reads * L].view(n_reads, L)
            mv = mates[:2 * n_reads * READ_LEN].view(n_reads, 2, READ_LEN)
            pv[:, :READ_LEN] = mv[:, 0]
            pv[:, READ_LEN + 1:] = mv[:, 1]
            del mates, mv, pv
        else:
            pool, _ = db.sample_reads(n_reads, READ_LEN, seed=3)
        hp = torch.empty(n_reads * L + 64, dtype=torch.uint8).pin_memory()
        hp.copy_(pool)
        host_pools[paired] = hp
        del pool
        torch.cuda.empty_cache()
    # the database: generated range by range on the GPU, parked in pinned host memory (where a real run mmaps the file)
    h_rec, h_off, meta = [], [], []
    cap_rows = int(records / passes * ppr * 1.08) + (1 << 20)
    pi = 0
    for lo, hi, rec, off in db.stream_ranges():
        if pi % ppr == 0:
            h_rec.append(torch.empty((cap_rows, 3), dtype=torch.int32).pin_memory())
            h_off.append([])
            meta.append([lo, hi, 0])
        m = meta[-1]
        assert m[2] + rec.shape[0] <= cap_rows, "range buffer too small"
        h_rec[-1][m[2]:m[2] + rec.shape[0]].copy_(rec)
        h_off[-1].append(off.cpu() if not h_off[-1] else off[1:].cpu())
        m[1] = hi
        m[2] += rec.shape[0]
        pi += 1
        del rec, off
    h_off = [torch.cat(o).pin_memory() for o in h_off]
    key_ct = db.key_ct
    species = np.array(db.species, np.uint32)
    pmap = db.parent_map()
    del db.genome
    torch.cuda.empty_cache()
    gen_s = time.time() - t_gen
    for paired in variants:
        _stream_job(args, local_rank, dev, paired, [host_pools.pop(paired)], h_rec, h_off, meta, key_ct, species, pmap, records, range_gb,
                    hll_mode, gen_s)
        torch.cuda.empty_cache()
    return 0


def _stream_job(args, local_rank, dev, paired, host_pool_box, h_rec, h_off, meta, key_ct, species, pmap, records, range_gb, hll_mode, gen_s):
    import torch
    host_pool = host_pool_box.pop()              # owned here: it is freed below, while the slots' streams still exist
    from krakenuniq_b200 import binding
    from krakenuniq_b200 import dist as kdist
    L = 2 * READ_LEN + 1 if paired else READ_LEN
    B = args.batch_reads // 2 if paired else args.batch_reads
    n_batches = args.steps
    n_reads = n_batches * B
    total_b = B * L
    pool = torch.empty(n_reads * L + 64, dtype=torch.uint8, device=dev)
    pool.copy_(host_pool)
    clf = binding.Classifier(device=local_rank, n_slots=2, max_reads=B, max_bases=total_b + 4096, hll_mode=hll_mode,
                             sparse_set_slots=1 << 27)
    clf.set_db_taxid_universe(species)
    clf.set_taxonomy(*pmap)
    clf.stream_open(K, NT, 2, max(m[2] for m in meta), max(m[1] - m[0] for m in meta))
    d_offsets = torch.arange(B + 2, dtype=torch.int64, device=dev) * L
    merged = torch.zeros(n_reads * L + 64, dtype=torch.int32, device=dev)
    streams = [torch.cuda.ExternalStream(clf.slot_stream(i), device=dev) for i in range(2)]
    h_call = torch.empty(n_reads, dtype=torch.int32).pin_memory()

    def load(buf, r):
        clf.stream_load(buf, h_rec[r].data_ptr(), meta[r][2], h_off[r].data_ptr(), meta[r][0], meta[r][1])

    def job(from_host):
        """the whole job; with from_host the reads are copied from pinned host memory as the first range reaches them"""
        merged.zero_()
        torch.cuda.synchronize()
        load(0, 0)
        for r in range(len(meta)):
            clf.stream_use(r & 1)
            if r + 1 < len(meta):
                load((r + 1) & 1, r + 1)
            for bi in range(n_batches):
                sl = bi & 1
                if from_host and r == 0:
                    with torch.cuda.stream(streams[sl]):
                        pool[bi * total_b:(bi + 1) * total_b].copy_(host_pool[bi * total_b:(bi + 1) * total_b], non_blocking=True)
                clf.lookup_device(sl, pool.data_ptr() + bi * total_b, d_offsets.data_ptr(), B, total_b,
                                  merged.data_ptr() + 4 * bi * total_b, only_hits=1)
        for bi in range(n_batches):
            sl = bi & 1
            clf.resolve_device(sl, pool.data_ptr() + bi * total_b, d_offsets.data_ptr(), B, total_b,
                               merged.data_ptr() + 4 * bi * total_b, None)
            if from_host:                                      # D2H of the calls of the batch
                r_ = clf.device_result(sl)
                with torch.cuda.stream(streams[sl]):
                    h_call[bi * B:(bi + 1) * B].copy_(kdist.device_view(r_.d_call, B * 4, torch.int32, dev), non_blocking=True)
        clf.sync(0); clf.sync(1)
        clf.finish()
        clf.stream_check()

    sampler = ClockSampler(local_rank)
    sampler.start()
    # warm-up: a few batches against the first range (kernels, clocks), state wiped afterwards
    load(0, 0); clf.stream_use(0)
    for bi in range(min(args.warmup, n_batches)):
        clf.lookup_device(bi & 1, pool.data_ptr() + bi * total_b, d_offsets.data_ptr(), B, total_b, merged.data_ptr() + 4 * bi * total_b, only_hits=1)
    clf.sync(0); clf.sync(1)
    res = {}
    for name, from_host in (("value", False), ("e2e", True)):
        clf.reset_counts()
        launches0 = clf.launch_count()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        with torch.cuda.stream(streams[0]):
            e0.record(streams[0])
        job(from_host)
        with torch.cuda.stream(streams[0]):
            e1.record(streams[0])
        torch.cuda.synchronize()
        sampler.mark(t0, time.time())
        res[name] = (e0.elapsed_time(e1), clf.launch_count() - launches0)
    clocks = sampler.stop()
    cnt = clf.counts()
    tot = int(cnt["n_reads"].sum())
    uncl = int(cnt["n_reads"][cnt["taxid"] == 0].sum())
    ms, launches = res["value"]
    db_bytes = key_ct * 12 + 8 * ((1 << (2 * NT)) + 1)
    unit_name = "pairs" if paired else "reads"
    unit = "Mreads/s" if not paired else "Mpairs/s"
    line = {"metric": METRIC if not paired else "Mpairs/s (2 x 150 bp)", "value": n_reads / (ms / 1e3) / 1e6,
            "unit": unit, "n_gpus": 1, "steps": n_batches, "warmup": args.warmup,
            "ms_per_step": ms / n_batches, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
            "data": "synthetic",
            "config": {"workload": f"{'configs[4]' if paired else 'configs[2]'}{'' if records == 25_000_000_000 else ' (scaled)'}: "
                                   f"{key_ct * 12 / 1e9:.1f} GB synthetic KrakenDB ({key_ct} records) + 8.6 GB index in PINNED HOST memory, streamed "
                                   f"through one GPU in {len(meta)} minimizer ranges of <= {range_gb:.0f} GB, {n_reads} {unit_name} "
                                   f"({L} chars each), {B} per step",
                       "parallelism": "1 GPU, two range buffers, copy stream overlapping the lookups",
                       "hll_mode": ["preload rule", "chunked rule", "dense only"][hll_mode],
                       "timing": "CUDA events around the whole job: every range H2D + all lookups + the final resolve pass + harvest; "
                                 "reads resident in HBM for `value`, copied from pinned host memory once for `e2e`",
                       "pcie_bound": {"db_bytes_over_pcie": db_bytes, "gbs_achieved_value": db_bytes / (ms / 1e3) / 1e9,
                                      "note": "every pass moves the whole database over PCIe: throughput = reads / (DB bytes / PCIe "
                                              "bandwidth) once the lookups hide behind the copy"},
                       "l2": "inputs larger than L2", "workload_gen_s": gen_s},
            "roofline": {"bound": "hbm", "achieved": None, "peak": None, "unit": "GB/s", "frac": None, "traffic": None,
                         "note": "PCIe-bound configuration: see config.pcie_bound; the kernels are those of the configs[1] line"},
            "cpu_baseline": {"value": None, "unit": unit, "cores": host_threads(), "kind": "reference",
                             "sample": "not run: the reference needs the 309 GB of database files in tmpfs plus the same again for -M"},
            "e2e": {"value": n_reads / (res["e2e"][0] / 1e3) / 1e6, "unit": unit,
                    "h2d_bytes_per_step": int(total_b + db_bytes / n_batches), "d2h_bytes_per_step": 4 * B,
                    "ms_per_step": res["e2e"][0] / n_batches,
                    "how": "reads copied from pinned host memory as the first range reaches them, calls copied back after the final pass"},
            "gpu_launches": int(launches),
            "sanity": {"reads_counted": tot, "classified_fraction": 1.0 - uncl / max(tot, 1),
                       "expected": "about 0.80" if not paired else "about 0.96 (a pair is classified if either mate is)"},
            "clocks": clocks}
    print(json.dumps(line), flush=True)
    # tensors that were used on the slots' streams go first: torch's allocator records an event on those streams when
    # it frees them, and kuq_destroy takes the streams away
    del pool, merged, h_call, d_offsets, host_pool
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    clf.close()


if __name__ == "__main__":
    sys.exit(main())
