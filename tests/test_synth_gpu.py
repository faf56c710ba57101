"""The torch workload generator (krakenuniq_b200/synth_gpu.py) writes the reference's on-disk layout: checked on
CPU tensors against the numpy generator and byte-for-byte against what the reference's own db_sort made of the same
records (its sha256 in tests/golden/reference/dbtools.json, written by tests/golden/make_golden_reference.py)."""
import numpy as np
import pytest

from krakenuniq_b200 import synth, synth_gpu
from tests import util


def _small(device="cpu", nt=7, idx_type=2):
    return synth_gpu.GpuDatabase(20000, n_genomes=10, k=31, nt=nt, idx_type=idx_type, seed=5, device=device, chunk=7000)


@pytest.mark.parametrize("nt,idx_type", [(7, 2), (5, 1)])
def test_layout_matches_numpy_generator(nt, idx_type):
    db = _small(nt=nt, idx_type=idx_type)
    kdb, idx = db.images()
    k, keys, taxa = synth.parse_kdb(kdb)
    assert k == 31 and len(keys) == db.key_ct
    kdb2, idx2 = synth.build_db_images(keys, taxa, 31, nt, idx_type)
    assert np.array_equal(kdb, kdb2) and np.array_equal(idx, idx2)
    # keys are the canonical k-mers of the genome, labelled by owner
    g = db.genome.numpy()
    km, ok = synth.forward_kmers(g, 31)
    canon = synth.canonical(km, 31)
    assert set(np.unique(canon).tolist()) == set(keys.tolist())
    pos = {int(c): i for i, c in reversed(list(enumerate(canon.tolist())))}
    sel = np.random.default_rng(0).integers(0, len(keys), 300)
    for kk, t in zip(keys[sel].tolist(), taxa[sel].tolist()):
        assert t == db.species[pos[kk] // db.genome_len]


def shuffled_records(kdb):
    """the records of a database image in a seeded random order, as db_sort's unsorted input"""
    k, keys, taxa = synth.parse_kdb(kdb)
    perm = np.random.default_rng(1).permutation(len(keys))
    rec = np.zeros(len(keys), synth._REC)
    rec["key"], rec["taxon"] = keys[perm], taxa[perm]
    return np.concatenate([synth.kdb_header(31, len(keys)), rec.view(np.uint8)])


def test_matches_reference_db_sort():
    """the reference's `db_sort -n 7` of the generator's records, shuffled, gives back the generator's images"""
    kdb, idx = _small().images()
    want = util.reference_json("dbtools.json")["synth_gpu_db_sort"]
    assert util.digest(kdb) == want["kdb"]
    assert util.digest(idx) == want["idx"]


def test_reads_shape_and_content():
    db = _small()
    bases, offs = db.sample_reads(500, 150, seed=9, chunk=128)
    b = bases.numpy()
    assert b.size == 500 * 150 + 64 and offs[-1].item() == 500 * 150
    assert set(np.unique(b[:500 * 150]).tolist()) <= set(b"ACGT")
    # most non-random reads share k-mers with the database
    kdb, idx = db.images()
    _, keys, _ = synth.parse_kdb(kdb)
    keyset = set(keys.tolist())
    hits = 0
    for i in range(100):
        km, ok = synth.forward_kmers(synth.encode(b[i * 150:(i + 1) * 150]), 31)
        hits += any(int(c) in keyset for c in synth.canonical(km, 31).tolist())
    assert hits > 60


def test_multi_pass_generation_equals_single_pass():
    a = synth_gpu.GpuDatabase(30000, n_genomes=7, k=31, nt=7, seed=11, device="cpu", chunk=9000)
    b = synth_gpu.GpuDatabase(30000, n_genomes=7, k=31, nt=7, seed=11, device="cpu", chunk=9000, passes=3)
    assert a.key_ct == b.key_ct
    assert np.array_equal(a.records.numpy(), b.records.numpy())
    assert np.array_equal(a.offsets.numpy(), b.offsets.numpy())


def test_sharded_generation_partitions_the_database():
    full = synth_gpu.GpuDatabase(30000, n_genomes=7, k=31, nt=7, seed=11, device="cpu", chunk=9000)
    recs, n = [], 0
    for r in range(3):
        sh = synth_gpu.GpuDatabase(30000, n_genomes=7, k=31, nt=7, seed=11, device="cpu", chunk=9000, passes=2,
                                   shard=(r, 3))
        lo, hi = sh.bin_lo, sh.bin_hi
        want_off = full.offsets[lo:hi + 1] - full.offsets[lo]
        assert np.array_equal(sh.offsets.numpy(), want_off.numpy())
        a, b = int(full.offsets[lo]), int(full.offsets[hi])
        assert np.array_equal(sh.records.numpy(), full.records[a:b].numpy())
        n += sh.key_ct
    assert n == full.key_ct


@pytest.mark.gpu
@pytest.mark.parametrize("shard", [None, (1, 3)])
def test_kernel_scan_generator_equals_torch_generator(shard):
    """On a GPU the generator takes k-mers and minimizer bins from the product's scan stage (kuq_scan_device):
    same database as the elementwise torch path that the CPU tests pin against the reference's db_sort."""
    kw = dict(n_genomes=9, k=31, nt=7, seed=13, device="cuda:0", chunk=10000, passes=2, shard=shard)
    a = synth_gpu.GpuDatabase(40000, use_kernel_scan=True, **kw)
    b = synth_gpu.GpuDatabase(40000, use_kernel_scan=False, **kw)
    assert a.key_ct == b.key_ct and (a.bin_lo, a.bin_hi) == (b.bin_lo, b.bin_hi)
    assert np.array_equal(a.records.cpu().numpy(), b.records.cpu().numpy())
    assert np.array_equal(a.offsets.cpu().numpy(), b.offsets.cpu().numpy())


def test_streamed_ranges_concatenate_to_the_database():
    full = synth_gpu.GpuDatabase(30000, n_genomes=7, k=31, nt=7, seed=11, device="cpu", chunk=9000)
    st = synth_gpu.GpuDatabase(30000, n_genomes=7, k=31, nt=7, seed=11, device="cpu", chunk=9000, passes=4, defer_build=True)
    recs, prev_hi = [], 0
    for lo, hi, rec, off in st.stream_ranges():
        assert lo == prev_hi
        prev_hi = hi
        assert np.array_equal(off.numpy(), full.offsets[lo:hi + 1].numpy())
        recs.append(rec.numpy().copy())
    assert prev_hi == 1 << 14 and st.key_ct == full.key_ct
    assert np.array_equal(np.concatenate(recs), full.records.numpy())
