"""Digests of the UNMODIFIED reference `classify -M` on the configs[1] workload of tests/test_large_cli_gpu.py (the 8 GB
synthetic database and 250 000 reads, generated on the GPU from fixed seeds).  Needs a GPU, 24 GB of tmpfs and
oracle/_ref (oracle/build_ref.sh):
    python tests/golden/make_golden_configs1.py [--out tests/golden/reference/configs1_cli.json]"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from tests import test_large_cli_gpu as T  # noqa: E402
from tests import util  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(util.REFERENCE, "configs1_cli.json"))
    args = ap.parse_args()
    exe = os.path.join(ROOT, "oracle", "_ref", "classify")
    if not os.path.exists(exe):
        raise SystemExit("oracle/_ref/classify is missing: build it with oracle/build_ref.sh")
    d, fq_par, _ = T.make_workload()
    threads = str(min(16, os.cpu_count() or 1))
    with tempfile.TemporaryDirectory() as tmp:
        kraken, report = os.path.join(tmp, "ref.kraken"), os.path.join(tmp, "ref.report")
        r = subprocess.run([exe, "-d", f"{d}/database.kdb", "-i", f"{d}/database.idx", "-a", f"{d}/taxDB", "-M", "-t", threads,
                            "-o", kraken, "-r", report, fq_par], capture_output=True, text=True,
                           env=dict(os.environ, OMP_NUM_THREADS=threads))
        if r.returncode != 0:
            raise SystemExit(r.stderr[-2000:])
        rows = T._rows(report)
        out = {"reads": len(open(kraken, "rb").read().splitlines()), "kraken_sorted_sha256": T.kraken_digest(kraken),
               "report_rows": len(rows), "report_rows_sha256": T.report_digest(rows)}
    assert out["reads"] == T.N_PARITY
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print(json.dumps(out))


if __name__ == "__main__":
    main()
