"""BASELINE configs[1] through the drop-in executable: 8 GB synthetic KrakenDB (666 M records, k=31, m=15), reads of
the bench workload, our `classify` against the UNMODIFIED reference (`classify -M`) — Kraken lines equal (as sorted
multisets: the reference runs multi-threaded, SURVEY §8(c)) and every report row equal, `kmers` included.  The
reference's outputs on this seeded workload are pinned by their sha256 in tests/golden/reference/configs1_cli.json
(written by tests/golden/make_golden_configs1.py on a GPU machine: the database is generated on the device).
Also times the whole command on a larger FASTQ (tmpfs → Kraken file + report, the reference's own stats-line
convention) and leaves the numbers in gpurun_out/cli_speed.json for bench.py / DESIGN.md."""
import json
import os
import re
import subprocess
import time

import numpy as np
import pytest

from krakenuniq_b200 import build
from tests import util

pytestmark = pytest.mark.gpu

N_PARITY = 250_000                       # the reads the golden digests were taken on
N_SPEED = int(os.environ.get("KUQ_LARGE_SPEED_READS", 8_000_000))


def _rows(path):
    rows = {}
    for line in open(path):
        if line.startswith("#") or line.startswith("%"):
            continue
        f = line.rstrip("\n").split("\t")
        rows[f[6]] = f
    return rows


def kraken_digest(path):
    """sha256 of the Kraken lines as a sorted multiset"""
    return util.digest(b"\n".join(sorted(open(path, "rb").read().splitlines())))


def report_digest(rows):
    return util.digest(json.dumps(sorted(rows.items())))


def make_workload():
    """database files, taxDB and the parity / speed FASTQs of the bench workload in tmpfs: (dir, parity fq, speed fq)"""
    import torch
    import bench
    from krakenuniq_b200 import synth_gpu

    class A:
        cache_dir, db_records, genomes, cpu_sample_reads = "/dev/shm", 666_000_000, 2000, N_PARITY
    db = synth_gpu.GpuDatabase(A.db_records, n_genomes=A.genomes, k=31, nt=15, seed=2, device="cuda:0")
    n = max(N_PARITY, N_SPEED)
    pool, _ = db.sample_reads(n, 150, seed=3)
    host = pool[:n * 150].cpu().numpy()
    d, fq_par = bench.ensure_files(A, db, host)
    fq_speed = os.path.join(d, f"sample_{N_SPEED}.fq")
    if not os.path.exists(fq_speed):
        bench.write_fastq(fq_speed, host, N_SPEED)
    del db, pool
    torch.cuda.empty_cache()
    return d, fq_par, fq_speed


@pytest.fixture(scope="module")
def workload():
    free = os.statvfs("/dev/shm")
    if free.f_bavail * free.f_frsize < 24 << 30:
        pytest.skip("needs 24 GB of tmpfs for the database files")
    return make_workload()


def test_configs1_cli_parity_with_the_reference(workload, tmp_path):
    d, fq_par, _ = workload
    dbargs = ["-d", f"{d}/database.kdb", "-i", f"{d}/database.idx", "-a", f"{d}/taxDB"]
    threads = str(min(16, os.cpu_count() or 1))
    exe = build.build_classify()
    r2 = subprocess.run([exe] + dbargs + ["-M", "-t", threads, "-o", str(tmp_path / "our.kraken"), "-r", str(tmp_path / "our.report"), fq_par],
                        capture_output=True, text=True, env=dict(os.environ, KUQ_SPARSE_SLOTS=str(1 << 28)))
    assert r2.returncode == 0, r2.stderr[-1500:]
    ref = util.reference_json("configs1_cli.json")
    assert ref["reads"] == N_PARITY and ref["report_rows"] > 2000     # 2000 species + genera + families + root + unclassified
    assert len(open(tmp_path / "our.kraken", "rb").read().splitlines()) == N_PARITY
    assert kraken_digest(tmp_path / "our.kraken") == ref["kraken_sorted_sha256"]
    b = _rows(tmp_path / "our.report")
    assert len(b) == ref["report_rows"] and report_digest(b) == ref["report_rows_sha256"]


def test_configs1_cli_throughput(workload, tmp_path):
    """file → file: FASTQ in tmpfs → Kraken file + report; numbers go to gpurun_out/cli_speed.json (no assertion on speed)"""
    d, _, fq_speed = workload
    dbargs = ["-d", f"{d}/database.kdb", "-i", f"{d}/database.idx", "-a", f"{d}/taxDB"]
    exe = build.build_classify()
    threads = str(min(64, os.cpu_count() or 1))
    out = {}
    for tag, extra in (("kraken_file", ["-o", f"{d}/speed.kraken"]), ("no_kraken_output", ["-o", "off"])):
        t0 = time.time()
        r = subprocess.run([exe] + dbargs + ["-M", "-t", threads, "-r", str(tmp_path / "speed.report")] + extra + [fq_speed],
                           capture_output=True, text=True, env=dict(os.environ, KUQ_SPARSE_SLOTS=str(1 << 30), KUQ_TIMING="1"))
        wall = time.time() - t0
        assert r.returncode == 0, r.stderr[-1500:]
        m = re.search(r"(\d+) sequences \(([\d.]+) Mbp\) processed in ([\d.]+)s", r.stderr)
        n, secs = int(m.group(1)), float(m.group(3))
        assert n == N_SPEED
        out[tag] = {"reads": n, "classification_s": secs, "mreads_per_s": n / secs / 1e6, "whole_command_s": wall, "threads": int(threads),
                    "timing": [line for line in r.stderr.splitlines() if "[timing]" in line]}
    os.makedirs(os.path.join(util.ROOT, "gpurun_out"), exist_ok=True)
    json.dump(out, open(os.path.join(util.ROOT, "gpurun_out", "cli_speed.json"), "w"), indent=1)
    if os.path.exists(f"{d}/speed.kraken"):
        os.remove(f"{d}/speed.kraken")
