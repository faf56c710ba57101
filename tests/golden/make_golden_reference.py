"""Answers of the UNMODIFIED reference on the seeded inputs of the tests that compare the oracle with it:
tests/test_oracle_vs_reference.py (its classes, through oracle/_ref/libkuref.so), tests/test_oracle_live_reference.py
(`classify` / `classifyExact` on fresh databases), tests/test_oracle_db_build.py and tests/test_synth_gpu.py
(`db_sort` / `set_lcas`).  Needs oracle/_ref (oracle/build_ref.sh):  python tests/golden/make_golden_reference.py
Writes tests/golden/reference/{functions.npz, fresh.json, dbtools.json}."""
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from krakenuniq_b200 import synth  # noqa: E402
from oracle import oracle_py  # noqa: E402
from oracle.oracle_py import Oracle, RefHLL, RefShim  # noqa: E402
from tests import test_oracle_db_build as T_db  # noqa: E402
from tests import test_oracle_live_reference as T_live  # noqa: E402
from tests import test_oracle_vs_reference as T_fn  # noqa: E402
from tests import test_synth_gpu as T_synth  # noqa: E402
from tests import util  # noqa: E402

K = 31


def run_ref(tool, cwd, args):
    r = oracle_py.run_ref_tool(tool, args, cwd=cwd)
    assert r.returncode == 0, (tool, args, r.stderr[-2000:])
    return r


def functions(ref):
    out = {}
    out["fmix_kats"] = np.array([ref.L.kuref_murmur_fmix(x) for x in T_fn.FMIX_KATS], np.uint64)
    assert out["fmix_kats"].tolist() == list(T_fn.FMIX_KATS.values())
    out["fmix"] = np.array([ref.L.kuref_murmur_fmix(x) for x in T_fn.fmix_inputs().tolist()], np.uint64)

    for idx_type, nt in T_fn.BITS_CASES:
        _, _, _, kdb, idx, probe = T_fn.bits_inputs(idx_type, nt)
        rdb = ref.open_db(kdb, idx)
        key = f"bits_{idx_type}_{nt}"
        out[key + "_header"] = np.array([ref.L.kuref_db_k(rdb.h), ref.L.kuref_db_index_nt(rdb.h),
                                         ref.L.kuref_db_index_type(rdb.h)], np.uint32)
        arrays = T_fn.bits_outputs(rdb.canonical, rdb.revcomp, rdb.bin_key, lambda x: rdb.bin_key_nt(x, nt), rdb.query, probe)
        for name, arr in arrays.items():
            out[f"{key}_{name}"] = np.array(util.digest(arr))

    kdb, idx, per_read = T_fn.stateful_inputs(Oracle())
    rdb = ref.open_db(kdb, idx)
    out["stateful"] = np.concatenate([rdb.query_stateful(c) for c in per_read]).astype(np.uint32)

    out["scan"] = np.array([T_fn.scan_digest(*ref.scan(seq, K)) for seq in T_fn.scanner_cases()])

    for with_one in (True, False):
        ids, parent, pairs, hit_maps = T_fn.lca_inputs(with_one)
        rpm = ref.parent_map(ids, parent)
        out[f"lca_{int(with_one)}"] = np.array([rpm.lca(a, b) for a, b in pairs], np.uint32)
        out[f"resolve_{int(with_one)}"] = np.array([rpm.resolve_tree(h) for h in hit_maps], np.uint32)

    kats = []
    for n, want in T_fn.HLL_KATS:
        r = RefHLL(ref); r.insert(T_fn.hll_seq(n))
        kats.append((r.cardinality(), r.n_observed()))
    out["hll_kats"] = np.array(kats, np.uint64)
    dense = []
    for n, want in T_fn.HLL_DENSE12_KATS:
        r = RefHLL(ref, dense_p=12); r.insert(T_fn.hll_seq(n))
        dense.append(r.cardinality())
    out["hll_dense12"] = np.array(dense, np.uint64)
    rg = RefHLL(ref)
    for i in range(10):
        r = RefHLL(ref); r.insert(T_fn.hll_seq(1000, off=1000 * i)); rg.merge(r, move=bool(i & 1))
    out["hll_merged10"] = np.array(rg.cardinality(), np.uint64)
    seq = []
    for parts in T_fn.hll_merge_sequences():
        rg = RefHLL(ref)
        for items, move in parts:
            r = RefHLL(ref); r.insert(items)
            card = r.cardinality()
            rg.merge(r, move=move)
            seq.append((card, rg.cardinality(), rg.n_observed()))
    out["hll_merge"] = np.array(seq, np.uint64)
    return out


def _classify(tool, d, db_args, flags):
    run_ref(tool, d, db_args + ["-a", "taxDB", "-t", 1, "-r", "ref.report", "-o", "ref.kraken"] + flags + ["reads.fa"])
    return {"kraken_sha256": util.digest(open(os.path.join(d, "ref.kraken"), "rb").read()),
            "report": open(os.path.join(d, "ref.report")).read()}


def fresh():
    one = ["-d", "database.kdb", "-i", "database.idx"]
    out = {}
    for tag, k, nt, idx_type, n_sp, glen, n_reads, flags, _ in T_live.CASES:
        with tempfile.TemporaryDirectory() as d:
            T_live.case_inputs(tag, k, nt, idx_type, n_sp, glen, n_reads, out_dir=d)
            out[f"live/{tag}"] = _classify("classify", d, one, flags)
    for order in ("ab", "ba"):
        with tempfile.TemporaryDirectory() as d:
            T_live.two_db_inputs(out_dir=d)
            first, second = order
            out[f"two_db/{order}"] = _classify("classify", d, ["-d", f"{first}.kdb", "-i", f"{first}.idx", "-d", f"{second}.kdb",
                                                               "-i", f"{second}.idx"], ["-M", "-u", "20000"])
    for min_hits, flags, _ in T_live.QUICK_CASES:
        with tempfile.TemporaryDirectory() as d:
            T_live.single_db_inputs(50 + min_hits, 7, 6, out_dir=d)
            out[f"quick/{min_hits}"] = _classify("classify", d, one, ["-q", "-m", min_hits] + flags)
    with tempfile.TemporaryDirectory() as d:
        T_live.single_db_inputs(77, 9, 7, out_dir=d)
        out["exact"] = _classify("classifyExact", d, one, ["-M"])
    return out


def _file_digest(path):
    return util.digest(np.fromfile(path, np.uint8))


def _write_library(d, tax, names, seqs, taxids, allk, width=None, strip_version=False, header_suffix=b""):
    with open(os.path.join(d, "lib.fa"), "wb") as f:
        for n, s in zip(names, seqs):
            f.write(b">" + n.encode() + header_suffix + b"\n")
            for i in range(0, len(s), width or max(len(s), 1)):
                f.write(s[i:i + (width or max(len(s), 1))] + b"\n")
    with open(os.path.join(d, "seqid2taxid.map"), "w") as f:
        for n, t in zip(names, taxids):
            f.write(f"{n[:-2] if strip_version and n.endswith('.2') else n}\t{t}\n")
    tax.write(os.path.join(d, "taxDB"))
    synth.unsorted_jdb_image(allk, K).tofile(os.path.join(d, "database.jdb"))
    run_ref("db_sort", d, ["-z", "-n", 6, "-d", "database.jdb", "-o", "database0.kdb", "-i", "database.idx"])
    return {"db_sort_kdb": _file_digest(os.path.join(d, "database0.kdb")),
            "db_sort_idx": _file_digest(os.path.join(d, "database.idx"))}


def _set_lcas(d, fa, flags=()):
    run_ref("set_lcas", d, ["-x", "-d", "database0.kdb", "-i", "database.idx", "-b", "taxDB", "-m", "seqid2taxid.map",
                            "-F", fa] + list(flags))
    return _file_digest(os.path.join(d, "database0.kdb"))        # without -M the mmap'ed input is rewritten in place


def dbtools():
    out = {}
    for nt, zero in T_db.DB_SORT_CASES:
        with tempfile.TemporaryDirectory() as d:
            _, jdb = T_db.db_sort_input(nt)
            jdb.tofile(os.path.join(d, "in.jdb"))
            run_ref("db_sort", d, (["-z"] if zero else []) + ["-n", nt, "-d", "in.jdb", "-o", "out.kdb", "-i", "out.idx"])
            out[f"db_sort/{nt}"] = {"kdb": _file_digest(os.path.join(d, "out.kdb")), "idx": _file_digest(os.path.join(d, "out.idx"))}

    with tempfile.TemporaryDirectory() as d:
        tax, sp, genomes, allk, names, seqs, taxids = T_db.set_lcas_inputs()
        e = _write_library(d, tax, names, seqs, taxids, allk, width=61, strip_version=True, header_suffix=b" some description")
        e["kdb"] = _set_lcas(d, "lib.fa")
        out["set_lcas"] = e

    with tempfile.TemporaryDirectory() as d:
        tax, g, allk2, names, seqs, taxids = T_db.contaminant_inputs()
        e = _write_library(d, tax, names, seqs, taxids, allk2)
        e["kdb"] = []
        for flag, part, _ in T_db.CONTAMINANT_RUNS:
            fa = "lib.fa"
            if part != slice(None):
                fa = "sub.fa"
                T_live.write_fasta(os.path.join(d, fa), names[part], seqs[part])
            e["kdb"].append(_set_lcas(d, fa, [flag]))
        out["contaminant"] = e

    with tempfile.TemporaryDirectory() as d:
        T_synth.shuffled_records(T_synth._small().images()[0]).tofile(os.path.join(d, "in.jdb"))
        run_ref("db_sort", d, ["-n", 7, "-d", "in.jdb", "-o", "out.kdb", "-i", "out.idx"])
        out["synth_gpu_db_sort"] = {"kdb": _file_digest(os.path.join(d, "out.kdb")), "idx": _file_digest(os.path.join(d, "out.idx"))}
    return out


def main():
    if not oracle_py.have_reference():
        raise SystemExit("oracle/_ref is missing: build it with oracle/build_ref.sh")
    os.makedirs(util.REFERENCE, exist_ok=True)
    np.savez_compressed(os.path.join(util.REFERENCE, "functions.npz"), **functions(RefShim()))
    for name, data in (("fresh.json", fresh()), ("dbtools.json", dbtools())):
        with open(os.path.join(util.REFERENCE, name), "w") as f:
            json.dump(data, f, indent=1, sort_keys=True)
            f.write("\n")
    for name in sorted(os.listdir(util.REFERENCE)):
        print(name, os.path.getsize(os.path.join(util.REFERENCE, name)))


if __name__ == "__main__":
    main()
