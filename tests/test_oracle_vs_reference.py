"""Pin the C restatement (oracle/kuq_oracle.c) against the UNMODIFIED reference classes, function by function, plus the
known answers SURVEY.md §8(c) extracted from the compiled reference.  The reference's answers on these seeded inputs
(oracle/_ref/libkuref.so) are stored in tests/golden/reference/functions.npz by tests/golden/make_golden_reference.py;
outputs too large to store are pinned by their sha256."""
import os

import numpy as np
import pytest

from krakenuniq_b200 import synth
from tests import util

K = 31
FMIX_KATS = {0: 0xb456bcfc34c2cb2c, 1: 0x3abf2a20650683e7, 2: 0x0b5181c509f8d8ce,
             0x0123456789abcdef: 0x6573ed81fcdd91d5, (1 << 62) - 1: 0x6554a70955a989a0}
BITS_CASES = [(2, 8), (1, 6), (2, 11)]
# SURVEY §8(c) known answers of the compiled reference: n items → cardinality, default sketch / forced dense p=12
HLL_KATS = [(1000, 1000), (1024, 1024), (1025, 1017), (2000, 2000), (10000, 9965), (100000, 100000)]
HLL_DENSE12_KATS = [(1000, 994), (1024, 1015)]


@pytest.fixture(scope="module")
def ref():
    return np.load(os.path.join(util.REFERENCE, "functions.npz"))


def _mini_db(rng, nt=8, idx_type=2, n_genomes=4, glen=1500):
    tax = synth.make_taxonomy(n_genomes)
    sp = synth.species_ids(tax)
    genomes = synth.random_genomes(rng, n_genomes, glen)
    km, tx = synth.label_kmers(genomes, sp, tax, K)
    kdb, idx = synth.build_db_images(km, tx, K, nt, idx_type)
    return tax, genomes, km, tx, kdb, idx


def fmix_inputs():
    return np.random.default_rng(1).integers(0, 1 << 63, 2000, dtype=np.uint64)


def test_fmix_kats(oracle, ref):
    for x, h in FMIX_KATS.items():
        assert oracle.fmix64(x) == h
    assert ref["fmix_kats"].tolist() == list(FMIX_KATS.values())
    got = np.array([oracle.fmix64(x) for x in fmix_inputs().tolist()], np.uint64)
    assert np.array_equal(got, ref["fmix"])


def test_kmer_kat_from_survey(oracle):
    # SURVEY §8(c): read ACGTACGTTAGCTAGCTAGGATCGATCGATTAGC..., window 0
    seq = b"ACGTACGTTAGCTAGCTAGGATCGATCGATTAGC"
    kmers, amb = oracle.scan(seq, K)
    assert kmers[0] == 0x06c6f272728d8d8f and amb[0] == 0
    canon = oracle.canonical(int(kmers[0]), K)
    assert canon == 0x0363635c9c9c1b1b
    assert oracle.bin_key(canon, K, 15, 2) == 3375861
    assert oracle.bin_key(canon, K, 8, 2) == 1713


def bits_inputs(idx_type, nt):
    rng = np.random.default_rng(10 + nt)
    tax, genomes, km, tx, kdb, idx = _mini_db(rng, nt, idx_type)
    probe = np.concatenate([km[rng.integers(0, len(km), 1500)],
                            synth.canonical(rng.integers(0, 1 << 62, 1500, dtype=np.uint64), K)])
    return rng, km, tx, kdb, idx, probe


def bits_outputs(canonical, revcomp, bin_key, bin_key_nt, query, probe):
    """The per-probe answers of one implementation, as the arrays whose sha256 the golden file holds."""
    xs = probe.tolist()
    low = [x & ((1 << 30) - 1) for x in xs]
    return {"canonical": np.array([canonical(x) for x in xs], np.uint64),
            "revcomp": np.array([revcomp(x, K) for x in xs], np.uint64),
            "revcomp15": np.array([revcomp(x, 15) for x in low], np.uint64),
            "bin_key": np.array([bin_key(x) for x in xs], np.uint64),
            "bin_key_nt": np.array([bin_key_nt(x) for x in xs], np.uint64),
            "query": np.array([query(x) for x in xs], np.uint64)}


@pytest.mark.parametrize("idx_type,nt", BITS_CASES)
def test_bits_and_lookup_match_reference(oracle, ref, idx_type, nt):
    rng, km, tx, kdb, idx, probe = bits_inputs(idx_type, nt)
    odb = oracle.open_db(kdb, idx)
    key = f"bits_{idx_type}_{nt}"
    assert ref[key + "_header"].tolist() == [K, nt, idx_type]
    assert [odb.k, odb.nt, odb.idx_type] == [K, nt, idx_type]
    got = bits_outputs(lambda x: oracle.canonical(x, K), oracle.revcomp, lambda x: oracle.bin_key(x, K, nt, idx_type),
                       lambda x: oracle.bin_key(x, K, nt, 2), odb.query, probe)
    for name, arr in got.items():
        assert util.digest(arr) == str(ref[f"{key}_{name}"]), name
    # numpy generator agrees too (it builds the fixtures)
    assert util.digest(synth.bin_key(probe, K, nt, idx_type).astype(np.uint64)) == str(ref[key + "_bin_key"])
    # every stored key is found with its taxon; stateful (cached-range) lookups agree with stateless ones
    sel = rng.integers(0, len(km), 500)
    for x, t in zip(km[sel].tolist(), tx[sel].tolist()):
        assert odb.query(x) == (True, t)


def stateful_inputs(oracle):
    """canonical k-mers of 200 reads, one array per read"""
    rng = np.random.default_rng(3)
    tax, genomes, km, tx, kdb, idx = _mini_db(rng, 8, 2)
    reads, offs = synth.sample_reads(rng, genomes, 200, 150, 0.02, 0.0, 0.3)
    per_read = []
    for i in range(200):
        kmers, amb = oracle.scan(reads[int(offs[i]):int(offs[i + 1])].tobytes(), K)
        per_read.append(synth.canonical(kmers[amb == 0], K))
    return kdb, idx, per_read


def test_stateful_query_equals_stateless(oracle, ref):
    """the reference's stateful (cached-range) lookups over each read's k-mers equal the oracle's stateless ones"""
    kdb, idx, per_read = stateful_inputs(oracle)
    odb = oracle.open_db(kdb, idx)
    want = np.split(ref["stateful"], np.cumsum([len(c) for c in per_read])[:-1])
    for canon, w in zip(per_read, want):
        assert np.array_equal(np.array([odb.query(x)[1] for x in canon.tolist()], np.uint32), w)


def scanner_cases():
    rng = np.random.default_rng(5)
    cases = [b"", b"ACGT", b"A" * 30, b"A" * 31, b"ACGTN" * 20, b"acgtacgtacgtacgtacgtacgtacgtacgtacgt",
             b"ACGT" * 10 + b"\r", b"ACGTAC" * 10 + b"\r", b"ACGTACGTAC" * 6 + b"\r" + b"GATTACA" * 8 + b"\r",
             b"N" * 40, b"ACGT" * 8 + b"R" + b"TGCA" * 9, b"ACGU" * 12, b"ACGT" * 8 + b"\n" + b"TTGA" * 9]
    for _ in range(200):
        n = int(rng.integers(0, 200))
        alphabet = np.frombuffer(b"ACGTACGTACGTacgtNnRY", np.uint8)
        cases.append(alphabet[rng.integers(0, len(alphabet), n)].tobytes())
    return cases


def scan_digest(kmers, amb):
    """window count, ambiguity flags and the k-mers of the unambiguous windows (the others are unspecified)"""
    return util.digest(np.array([len(kmers)], np.uint64), amb.astype(np.uint8), kmers[amb == 0].astype(np.uint64))


def test_scanner_matches_reference(oracle, ref):
    cases = scanner_cases()
    assert len(ref["scan"]) == len(cases)
    for seq, want in zip(cases, ref["scan"]):
        assert scan_digest(*oracle.scan(seq, K)) == str(want), seq


def _random_forest(rng, n, with_one=True):
    ids = np.unique(rng.integers(2, 5000, n)).astype(np.uint32)
    parent = np.zeros(len(ids), np.uint32)
    for i in range(len(ids)):
        r = rng.random()
        if i == 0 or r < 0.05:
            parent[i] = 1 if with_one else 0
        elif r < 0.08:
            parent[i] = 0                      # a second root (parent NULL → 0, taxdb.hpp:389-391)
        elif r < 0.10:
            parent[i] = 77777                  # parent id that has no entry of its own
        else:
            parent[i] = ids[int(rng.integers(0, i))]
    if with_one:
        ids = np.concatenate([[1], ids]).astype(np.uint32)
        parent = np.concatenate([[0], parent]).astype(np.uint32)
    return ids, parent


def lca_inputs(with_one):
    """a random forest, 3000 taxon pairs and 1500 hit maps"""
    rng = np.random.default_rng(7 + with_one)
    ids, parent = _random_forest(rng, 300, with_one)
    pool = np.concatenate([ids, [0, 1, 99999]]).astype(np.uint32)
    pairs = [tuple(int(x) for x in pool[rng.integers(0, len(pool), 2)]) for _ in range(3000)]
    hit_maps = []
    for _ in range(1500):
        n = int(rng.integers(0, 7))
        nz = pool[pool != 0]
        taxa = np.unique(nz[rng.integers(0, len(nz), n)]) if n else np.zeros(0, np.uint32)
        hit_maps.append({int(t): int(rng.integers(1, 4)) for t in taxa})
    return ids, parent, pairs, hit_maps


@pytest.mark.parametrize("with_one", [True, False])
def test_lca_and_resolve_tree_match_reference(oracle, ref, with_one):
    ids, parent, pairs, hit_maps = lca_inputs(with_one)
    opm = oracle.parent_map(ids, parent)
    for (a, b), want in zip(pairs, ref[f"lca_{int(with_one)}"].tolist()):
        assert opm.lca(a, b) == want, (a, b)
    for hits, want in zip(hit_maps, ref[f"resolve_{int(with_one)}"].tolist()):
        assert opm.resolve_tree(hits) == want, hits


def hll_seq(n, mul=0x9E3779B97F4A7C15, off=0):
    return ((np.arange(off, off + n, dtype=np.uint64)) * np.uint64(mul))


def test_hll_kats_and_state_machine(oracle, ref):
    for (n, want), (r_card, r_obs) in zip(HLL_KATS, ref["hll_kats"].tolist()):
        o = oracle.hll(); o.insert(hll_seq(n))
        assert r_card == want
        assert o.cardinality() == want
        assert o.n_observed() == r_obs == n
        assert o.is_sparse() == (n <= 1024)
    # forced dense p=12 via the registers-only estimator
    for (n, want), r_card in zip(HLL_DENSE12_KATS, ref["hll_dense12"].tolist()):
        assert r_card == want
        o = oracle.hll(); o.insert(hll_seq(n))
        assert oracle.ertl_dense(o.registers(), n) == want
    # ten sparse sketches of 1000 merged stay sparse and near exact
    og = oracle.hll()
    for i in range(10):
        o = oracle.hll(); o.insert(hll_seq(1000, off=1000 * i)); og.merge(o)
    assert og.is_sparse() and og.cardinality() == int(ref["hll_merged10"]) == 10000


def hll_merge_sequences():
    """12 trials of (items, merge by move) parts, duplicates on purpose: items are drawn from a pool about as large as n"""
    rng = np.random.default_rng(11)
    trials = []
    for trial in range(12):
        parts = []
        for part in range(int(rng.integers(1, 8))):
            n = int(rng.choice([0, 3, 200, 1023, 1024, 1025, 1500, 5000]))
            parts.append((rng.integers(0, max(n, 1) * int(rng.choice([1, 4, 1000])), n, dtype=np.uint64), bool(part & 1)))
        trials.append(parts)
    return trials


def test_hll_random_merge_sequences(oracle, ref):
    """per part: (cardinality of the part, cardinality and items observed of the running merge)"""
    got = []
    for parts in hll_merge_sequences():
        og = oracle.hll()
        for items, _ in parts:
            o = oracle.hll(); o.insert(items)
            og.merge(o)
            got.append((o.cardinality(), og.cardinality(), og.n_observed()))
    assert np.array_equal(np.array(got, np.uint64), ref["hll_merge"])
