"""Database build tools (SURVEY.md §8 f4): the oracle's db_sort and set_lcas against the unmodified reference
executables (oracle/_ref/db_sort, oracle/_ref/set_lcas) on the same inputs, byte for byte.  The reference ran on these
seeded inputs in tests/golden/make_golden_reference.py; tests/golden/reference/dbtools.json holds the sha256 of every
image it wrote."""
import os

import numpy as np
import pytest

from krakenuniq_b200 import synth
from tests import util

K = 31


@pytest.fixture(scope="module")
def ref():
    return util.reference_json("dbtools.json")


def _library(seed, n_genomes=6, glen=1500):
    rng = np.random.default_rng(seed)
    tax = synth.make_taxonomy(n_genomes, 3, 2, first_id=100)
    sp = synth.species_ids(tax)
    genomes = synth.random_genomes(rng, n_genomes, glen, shared_frac=0.3)
    ks = []
    for g in genomes:
        km, ok = synth.forward_kmers(g, K)
        ks.append(synth.canonical(km[ok], K))
    allk = np.unique(np.concatenate(ks))
    rng.shuffle(allk)
    return rng, tax, sp, genomes, allk


DB_SORT_CASES = [(5, True), (7, False), (9, True)]


def db_sort_input(nt):
    """unsorted Jellyfish-style image with random values; header bytes the tools ignore must be copied through"""
    rng, tax, sp, genomes, allk = _library(nt)
    rec = np.zeros(len(allk), synth._REC)
    rec["key"] = allk
    rec["taxon"] = rng.integers(0, 1 << 20, len(allk))
    jdb = np.concatenate([synth.kdb_header(K, len(allk)), rec.view(np.uint8)])
    jdb[100:140] = rng.integers(0, 255, 40)
    return allk, jdb


def _sorted_library(oracle, ref, allk, key):
    """db_sort -z -n 6 of the library's k-mers, checked against the reference's images (the input of set_lcas)"""
    kdb0, idx = oracle.db_sort(synth.unsorted_jdb_image(allk, K), 6, True)
    assert util.digest(kdb0) == ref[key]["db_sort_kdb"] and util.digest(idx) == ref[key]["db_sort_idx"]
    return kdb0, idx


@pytest.mark.parametrize("nt,zero", DB_SORT_CASES)
def test_db_sort_matches_reference(oracle, ref, nt, zero):
    allk, jdb = db_sort_input(nt)
    kdb, idx = oracle.db_sort(jdb, nt, zero)
    want = ref[f"db_sort/{nt}"]
    assert util.digest(kdb) == want["kdb"]
    assert util.digest(idx) == want["idx"]
    # and the numpy builder used for the synthetic databases agrees (zeroed values / kept values)
    _, keys, vals = synth.parse_kdb(kdb)
    assert set(keys.tolist()) == set(allk.tolist())
    if zero:
        assert not vals.any()


def set_lcas_inputs():
    """library, taxa and k-mers: two extra library sequences, one whose taxid the taxonomy does not know (skipped,
    set_lcas.cpp:336-341) and one that holds k-mers the database lacks (-x: ignored, :439-447); one id only matches
    without its ".2" suffix"""
    rng, tax, sp, genomes, allk = _library(21)
    extra = rng.integers(0, 4, 700, dtype=np.uint8)
    names = [f"seq{i}" for i in range(len(genomes))] + ["unknown_tax", "novel.2"]
    seqs = [synth.decode(g).tobytes() for g in genomes] + [synth.decode(genomes[0][:400]).tobytes(),
                                                           synth.decode(genomes[1][:300]).tobytes() + b"N" + synth.decode(extra).tobytes()]
    taxids = list(sp) + [4242, sp[3]]
    return tax, sp, genomes, allk, names, seqs, taxids


def test_set_lcas_matches_reference(oracle, ref):
    tax, sp, genomes, allk, names, seqs, taxids = set_lcas_inputs()
    kdb0, idx = _sorted_library(oracle, ref, allk, "set_lcas")
    want = ref["set_lcas"]["kdb"]                 # without -M the reference rewrites its mmap'ed input in place
    assert want != util.digest(kdb0)

    ids, parents = tax.parent_map()
    known = set(int(t) for t in ids)
    pm = oracle.parent_map(ids, parents)
    db = oracle.open_db(kdb0.copy(), idx)
    missing = 0
    for s, t in zip(seqs, taxids):
        if t not in known:
            continue
        missing += oracle.set_lcas_sequence(db, pm, s, t)
    assert missing > 0
    assert util.digest(db.kdb) == want
    # the values are the LCA of the owners, as the numpy labeller computes them
    km, tx = synth.label_kmers(genomes + [np.concatenate([genomes[1][:300]])], list(sp) + [sp[3]], tax, K)
    _, keys, vals = synth.parse_kdb(db.kdb)
    got = dict(zip(keys.tolist(), vals.tolist()))
    for kk, t in zip(km.tolist(), tx.tolist()):
        assert got[kk] == t


def contaminant_inputs():
    """a library with two contaminant sequences ('synthetic construct' 32630 / 'artificial sequences' 81077)"""
    rng, tax, sp, genomes, allk = _library(33)
    tax = synth.Taxonomy(tax.rows + [(32630, 1, "synthetic construct", "species"), (81077, 1, "artificial sequences", "species")])
    g = [synth.decode(x).tobytes() for x in genomes]
    novel1 = synth.decode(rng.integers(0, 4, 300, dtype=np.uint8)).tobytes()
    vec1 = g[2][200:500] + novel1 + g[0][900:1100]           # contaminant 1: parts of genomes 2 and 0
    vec2 = g[2][350:650] + g[4][100:400]                     # contaminant 2: overlaps vec1 on genome 2, plus genome 4
    names = ["seq0", "seq1", "seq2", "vec1", "seq3", "vec2", "seq4", "seq5"]
    seqs = [g[0], g[1], g[2], vec1, g[3], vec2, g[4], g[5]]
    taxids = [sp[0], sp[1], sp[2], 32630, sp[3], 81077, sp[4], sp[5]]
    ks = [allk]
    for s in (vec1,):
        km, ok = synth.forward_kmers(synth.encode(s), K)
        ks.append(synth.canonical(km[ok], K))
    allk2 = np.unique(np.concatenate(ks))
    rng.shuffle(allk2)
    return tax, g, allk2, names, seqs, taxids


# the runs of set_lcas on one image, in order: -T over the library, then the hierarchical re-labelling of
# build_db.sh:286-296 — -TR on a sub-library (sequences 2..4), then -T on it
CONTAMINANT_RUNS = [("-T", slice(None), 1), ("-TR", slice(2, 5), 3), ("-T", slice(2, 5), 1)]


def test_set_lcas_contaminant_and_reset_flags_match_reference(oracle, ref):
    """set_lcas -T (what build_db.sh always passes: 'synthetic construct' 32630 / 'artificial sequences' 81077 stick,
    set_lcas.cpp:462-474) and -TR (values of the library's k-mers reset to 0, :458-459)"""
    tax, g, allk2, names, seqs, taxids = contaminant_inputs()
    kdb0, idx = _sorted_library(oracle, ref, allk2, "contaminant")
    ids, parents = tax.parent_map()
    pm = oracle.parent_map(ids, parents)
    db = oracle.open_db(kdb0.copy(), idx)
    wants = ref["contaminant"]["kdb"]
    assert len(wants) == len(CONTAMINANT_RUNS)
    for i, ((_, part, flags), want) in enumerate(zip(CONTAMINANT_RUNS, wants)):
        for s, t in list(zip(seqs, taxids))[part]:
            oracle.set_lcas_sequence(db, pm, s, t, flags=flags)
        assert util.digest(db.kdb) == want, CONTAMINANT_RUNS[i]
        if i == 0:
            _, keys, vals = synth.parse_kdb(db.kdb)
            got = dict(zip(keys.tolist(), vals.tolist()))
            km, ok = synth.forward_kmers(synth.encode(g[2][350:500]), K)      # shared by both contaminants: the first one wins
            assert {got[int(c)] for c in synth.canonical(km[ok], K).tolist()} == {32630}
            km, ok = synth.forward_kmers(synth.encode(g[4][100:400]), K)      # contaminant 2 before its genome in the file
            assert {got[int(c)] for c in synth.canonical(km[ok], K).tolist()} == {81077}
