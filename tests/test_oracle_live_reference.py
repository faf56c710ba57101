"""The oracle against the UNMODIFIED reference `classify` on freshly generated databases — other k, minimizer lengths,
index flavours, work-unit sizes and taxonomies than the committed golden set holds (k = 29..31: the 12-byte records of
every published database).  Kraken lines byte for byte (pinned by their sha256), report rows exactly.
tests/golden/make_golden_reference.py ran the reference on the same seeded inputs; its answers are in
tests/golden/reference/fresh.json."""
import os

import numpy as np
import pytest

from krakenuniq_b200 import synth
from tests import util


@pytest.fixture(scope="module")
def ref():
    return util.reference_json("fresh.json")


def write_fasta(path, names, seqs):
    with open(path, "wb") as f:
        for n, s in zip(names, seqs):
            f.write(b">" + n.encode() + b"\n" + s + b"\n")


def _write_db(out_dir, kdb, idx, tax=None, name="database"):
    kdb.tofile(os.path.join(out_dir, f"{name}.kdb"))
    idx.tofile(os.path.join(out_dir, f"{name}.idx"))
    if tax is not None:
        tax.write(os.path.join(out_dir, "taxDB"))


def _expect(ref, key, tmp_path, ids, seqs, calls, codes, code_off):
    """Kraken lines against the reference's digest; the reference's report is written to tmp_path for _report_equals"""
    want = ref[key]
    assert util.digest(util.kraken_lines(ids, seqs, calls, codes, code_off)) == want["kraken_sha256"]
    (tmp_path / "ref.report").write_text(want["report"])
    return tmp_path / "ref.report"


CASES = [
    # tag, k, nt, idx_type, n_species, genome length, reads, classify flags, oracle (unit, mode)
    ("k31_nt8", 31, 8, 2, 9, 2500, 1200, ["-M"], (500000, 0)),
    ("k31_nt11_small_units", 31, 11, 2, 5, 4000, 1500, ["-M", "-u", "3000"], (3000, 0)),
    ("k31_krakidx", 31, 6, 1, 6, 2000, 800, ["-M"], (500000, 0)),
    ("k30_nt9", 30, 9, 2, 7, 2200, 1000, ["-M", "-u", "20000"], (20000, 0)),
    ("k29_nt5_chunked", 29, 5, 2, 4, 1800, 700, ["-x", "30K"], (500000, 1)),
]


def case_inputs(tag, k, nt, idx_type, n_sp, glen, n_reads, out_dir=None):
    """database, taxonomy and reads of one CASES row; with out_dir, also the files the reference reads"""
    import zlib
    rng = np.random.default_rng(zlib.crc32(tag.encode()))
    tax = synth.make_taxonomy(n_sp, max(2, n_sp // 2), 2)
    genomes = synth.random_genomes(rng, n_sp, glen, shared_frac=0.25)
    km, tx = synth.label_kmers(genomes, synth.species_ids(tax), tax, k)
    kdb, idx = synth.build_db_images(km, tx, k, nt, idx_type)
    bases, offs = synth.sample_reads(rng, genomes, n_reads, 150, 0.01, 0.15, 0.15)
    seqs = [bases[int(offs[i]):int(offs[i + 1])].tobytes() for i in range(n_reads)]
    g0 = synth.decode(genomes[0]).tobytes()
    seqs += [b"", b"ACG", g0[:k - 1], g0[:k], g0[5:5 + k] + b"N" + g0[400:400 + k + 3], b"N" * 90, g0[100:460]]
    ids = [f"r{i}" for i in range(len(seqs))]
    if out_dir:
        _write_db(out_dir, kdb, idx, tax)
        write_fasta(os.path.join(out_dir, "reads.fa"), ids, seqs)
    return tax, kdb, idx, ids, seqs


@pytest.mark.parametrize("tag,k,nt,idx_type,n_sp,glen,n_reads,flags,omode", CASES, ids=[c[0] for c in CASES])
def test_oracle_equals_live_reference(oracle, ref, tmp_path, tag, k, nt, idx_type, n_sp, glen, n_reads, flags, omode):
    tax, kdb, idx, ids, seqs = case_inputs(tag, k, nt, idx_type, n_sp, glen, n_reads)
    db = oracle.open_db(kdb, idx)
    pm = oracle.parent_map(*tax.parent_map())
    run = oracle.run(db, pm, *omode)
    b2, o2 = synth.pack_reads(seqs)
    calls, codes, code_off = run.classify(b2, o2)
    run.finish()
    report = _expect(ref, f"live/{tag}", tmp_path, ids, seqs, calls, codes, code_off)
    cnt = run.counts()
    rep = util.parse_report(str(report))
    by_tax = {int(t): i for i, t in enumerate(cnt["taxid"])}
    members = util.clade_members(tax.rows, cnt["taxid"])
    assert len(rep) >= 4
    for taxid, row in rep.items():
        i = by_tax.get(taxid)
        assert row["taxReads"] == (int(cnt["n_reads"][i]) if i is not None else 0)
        u, rd, kk = run.clade(members[taxid])
        assert (row["reads"], row["kmers"]) == (rd, u), (tag, taxid, row, rd, u)


def fresh_inputs(seed, k=31, nt=8, idx_type=2, n_sp=8, glen=2400, n_reads=1000, out_dir=None, name="database"):
    rng = np.random.default_rng(seed)
    tax = synth.make_taxonomy(n_sp, max(2, n_sp // 2), 2)
    genomes = synth.random_genomes(rng, n_sp, glen, shared_frac=0.25)
    km, tx = synth.label_kmers(genomes, synth.species_ids(tax)[:len(genomes)], tax, k)
    kdb, idx = synth.build_db_images(km, tx, k, nt, idx_type)
    if out_dir:
        _write_db(out_dir, kdb, idx, tax, name)
    bases, offs = synth.sample_reads(rng, genomes, n_reads, 150, 0.01, 0.15, 0.15)
    seqs = [bases[int(offs[i]):int(offs[i + 1])].tobytes() for i in range(n_reads)]
    return tax, genomes, kdb, idx, seqs


def _report_equals(run, tax, report_path):
    cnt = run.counts()
    rep = util.parse_report(str(report_path))
    by_tax = {int(t): i for i, t in enumerate(cnt["taxid"])}
    members = util.clade_members(tax.rows, cnt["taxid"])
    assert len(rep) >= 4
    for taxid, row in rep.items():
        i = by_tax.get(taxid)
        assert row["taxReads"] == (int(cnt["n_reads"][i]) if i is not None else 0)
        u, rd, kk = run.clade(members[taxid])
        assert (row["reads"], row["kmers"]) == (rd, u), (taxid, row, rd, u)


def two_db_inputs(out_dir=None):
    """databases a and b that label shared k-mers differently, minimizer lengths differ; files a.* / b.* / taxDB / reads.fa"""
    tax, genomes, kdb_a, idx_a, seqs = fresh_inputs(41, nt=8, n_sp=8, out_dir=out_dir, name="a")
    # B: the first five genomes again, labelled with the NEXT species (so the same k-mer has another taxon there), plus
    # one genome only B knows
    rng = np.random.default_rng(42)
    sp = synth.species_ids(tax)
    gb = genomes[:5] + [rng.integers(0, 4, 2400, dtype=np.uint8)]
    km, tx = synth.label_kmers(gb, sp[1:6] + [sp[7]], tax, 31)
    kdb_b, idx_b = synth.build_db_images(km, tx, 31, 10, 2)
    extra, _ = synth.sample_reads(rng, gb, 300, 150, 0.01, 0.1, 0.1)
    seqs = seqs + [extra[i * 150:(i + 1) * 150].tobytes() for i in range(300)]
    ids = [f"r{i}" for i in range(len(seqs))]
    if out_dir:
        _write_db(out_dir, kdb_b, idx_b, name="b")
        write_fasta(os.path.join(out_dir, "reads.fa"), ids, seqs)
    return tax, {"a": (kdb_a, idx_a), "b": (kdb_b, idx_b)}, ids, seqs


@pytest.mark.parametrize("order", ["ab", "ba"])
def test_two_fresh_databases_first_hit(oracle, ref, tmp_path, order):
    """-d A -d B with databases that label shared k-mers differently (classify.cpp:928-936), minimizer lengths differ"""
    tax, images, ids, seqs = two_db_inputs()
    first, second = order
    dbs = {n: oracle.open_db(*images[n]) for n in images}
    run = oracle.run(dbs[first], oracle.parent_map(*tax.parent_map()), 20000, 0)
    run.add_db(dbs[second])
    bases, offs = synth.pack_reads(seqs)
    calls, codes, code_off = run.classify(bases, offs)
    run.finish()
    _report_equals(run, tax, _expect(ref, f"two_db/{order}", tmp_path, ids, seqs, calls, codes, code_off))


QUICK_CASES = [(2, ["-M"], (500000, 0)), (5, ["-M", "-u", "20000"], (20000, 0)), (3, ["-x", "40K"], (500000, 1))]


def single_db_inputs(seed, nt, n_sp, out_dir=None):
    tax, genomes, kdb, idx, seqs = fresh_inputs(seed, nt=nt, n_sp=n_sp, out_dir=out_dir)
    ids = [f"r{i}" for i in range(len(seqs))]
    if out_dir:
        write_fasta(os.path.join(out_dir, "reads.fa"), ids, seqs)
    return tax, kdb, idx, ids, seqs


@pytest.mark.parametrize("min_hits,flags,omode", QUICK_CASES)
def test_quick_mode_on_a_fresh_database(oracle, ref, tmp_path, min_hits, flags, omode):
    tax, kdb, idx, ids, seqs = single_db_inputs(50 + min_hits, 7, 6)
    run = oracle.run(oracle.open_db(kdb, idx), oracle.parent_map(*tax.parent_map()), *omode)
    run.set_quick(min_hits)
    bases, offs = synth.pack_reads(seqs)
    calls, codes, code_off = run.classify(bases, offs)
    run.finish()
    lines = []
    for i, (rid, s) in enumerate(zip(ids, seqs)):
        c = codes[int(code_off[i]):int(code_off[i + 1])]
        hits = min(int(((c != 0) & (c != 0xFFFFFFFF)).sum()), min_hits)
        lines.append(f"{'C' if calls[i] else 'U'}\t{rid}\t{int(calls[i])}\t{len(s)}\tQ:{hits}\n")
    want = ref[f"quick/{min_hits}"]
    assert util.digest("".join(lines)) == want["kraken_sha256"]
    (tmp_path / "ref.report").write_text(want["report"])
    _report_equals(run, tax, tmp_path / "ref.report")


def test_exact_counting_on_a_fresh_database(oracle, ref, tmp_path):
    tax, kdb, idx, ids, seqs = single_db_inputs(77, 9, 7)
    run = oracle.run(oracle.open_db(kdb, idx), oracle.parent_map(*tax.parent_map()), 500000, 0)
    run.set_exact()
    bases, offs = synth.pack_reads(seqs)
    calls, codes, code_off = run.classify(bases, offs)
    run.finish()
    _report_equals(run, tax, _expect(ref, "exact", tmp_path, ids, seqs, calls, codes, code_off))
