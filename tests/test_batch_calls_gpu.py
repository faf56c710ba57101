"""Checks every batch entry point of libkuq (include/kuq.h) makes before it launches anything: a slot out of range, NULL
or misaligned buffers, a batch above the slot capacity and a preload-rule device call without work-unit ids are
refused on the host, and a slot with an unread batch refuses every batch call until kuq_wait_batch, which then returns
that batch unchanged.  Every buffer handed over is a valid allocation large enough for its batch, so a check that
stopped refusing would show as a wrong return code, not as a kernel reading through a bad pointer."""
import ctypes as C

import numpy as np
import pytest

from krakenuniq_b200 import binding, synth

pytestmark = pytest.mark.gpu
K, NT, IDX_TYPE = 31, 8, 2
E_INVALID_ARG, E_STATE, E_CAPACITY = -1, -6, -7
MAX_READS, MAX_BASES = 512, 1 << 17
N_POOL, READ_LEN = 1000, 150            # 150000 bases: one read can span more than MAX_BASES
DEV = "cuda:0"


@pytest.fixture(scope="module")
def synthetic():
    rng = np.random.default_rng(41)
    tax = synth.make_taxonomy(4)
    genomes = synth.random_genomes(rng, 4, 2500, shared_frac=0.25)
    km, tx = synth.label_kmers(genomes, synth.species_ids(tax), tax, K)
    kdb, idx = synth.build_db_images(km, tx, K, NT, IDX_TYPE)
    bases, offs = synth.sample_reads(rng, genomes, N_POOL, READ_LEN, 0.01, 0.2, 0.2)
    return tax, kdb, idx, bases, offs


def _classifier(synthetic):
    tax, kdb, idx, _, _ = synthetic
    clf = binding.Classifier(n_slots=2, max_reads=MAX_READS, max_bases=MAX_BASES, sparse_set_slots=1 << 20)
    clf.stage_db(kdb, idx)
    clf.set_taxonomy(*tax.parent_map())
    return clf


class Batch:
    """The reads of the pool that `offs` delimits, with host and device copies of everything the entry points take;
    device buffers cover the whole pool plus slack, and the device bases are 16-byte aligned."""

    def __init__(self, synthetic, offs):
        import torch
        tax, _, _, bases, _ = synthetic
        self.offs = np.ascontiguousarray(offs, np.uint64)
        self.n, self.total = len(offs) - 1, int(offs[-1] - offs[0])
        self.h_bases, self.h_offs = bases.ctypes.data, self.offs.ctypes.data_as(binding.u64p)
        self.h_codes = np.zeros(bases.size, np.uint32)          # lookup output / resolve input
        self.h_nwin = np.zeros(N_POOL, np.uint32)
        self.taxid = np.full(N_POOL, synth.species_ids(tax)[0], np.uint32)
        self._keep = [bases, torch.from_numpy(np.concatenate([bases, np.full(64, ord("N"), np.uint8)])).to(DEV),
                      torch.from_numpy(np.concatenate([self.offs, self.offs[-1:]]).astype(np.int64)).to(DEV),
                      torch.zeros(N_POOL, dtype=torch.int32, device=DEV),             # work-unit ids
                      torch.zeros(bases.size + 64, dtype=torch.int32, device=DEV),    # per-window ids
                      torch.zeros(bases.size + 64, dtype=torch.int64, device=DEV),    # scan: canonical k-mers
                      torch.zeros(bases.size + 64, dtype=torch.int32, device=DEV)]    # scan: bins
        self.d_bases, self.d_offs, self.d_unit, self.d_codes, self.d_canon, self.d_bins = \
            (t.data_ptr() for t in self._keep[1:])


def _entry_points(clf, slot, b):
    """Every batch entry point of kuq.h over batch b, on `slot` where the call takes one: name → call → return code."""
    L, h, u32p = clf.L, clf.h, binding.u32p
    res, missing = binding.BatchResult(), C.c_uint64()
    peers = (C.c_void_p * 1)(b.d_codes)
    bounds = np.array([0, b.total], np.uint64)
    calls = {
        "kuq_submit_batch": lambda: L.kuq_submit_batch(h, slot, b.h_bases, b.h_offs, b.n, None, 0),
        "kuq_classify_device": lambda: L.kuq_classify_device(h, slot, b.d_bases, b.d_offs, b.n, b.total, b.d_unit, 0),
        "kuq_lookup_device": lambda: L.kuq_lookup_device(h, slot, b.d_bases, b.d_offs, b.n, b.total, b.d_codes, 0),
        "kuq_resolve_device": lambda: L.kuq_resolve_device(h, slot, b.d_bases, b.d_offs, b.n, b.total, b.d_codes,
                                                           b.d_unit, 0),
        "kuq_lookup_device_peers": lambda: L.kuq_lookup_device_peers(h, slot, b.d_bases, b.d_offs, b.n, b.total, peers,
                                                                     bounds.ctypes.data_as(binding.u64p), 1),
        "kuq_scan_device": lambda: L.kuq_scan_device(h, slot, K, NT, IDX_TYPE, b.d_bases, b.d_offs, b.n, b.total,
                                                     b.d_canon, b.d_bins),
    }
    if slot == 0:                       # these always use slot 0
        calls.update({
            "kuq_classify_batch": lambda: L.kuq_classify_batch(h, b.h_bases, b.h_offs, b.n, None, 0, C.byref(res)),
            "kuq_lookup_batch": lambda: L.kuq_lookup_batch(h, b.h_bases, b.h_offs, b.n, b.h_codes.ctypes.data_as(u32p),
                                                           b.h_nwin.ctypes.data_as(u32p)),
            "kuq_resolve_batch": lambda: L.kuq_resolve_batch(h, b.h_bases, b.h_offs, b.n, b.h_codes.ctypes.data_as(u32p),
                                                             None, 0, C.byref(res)),
            "kuq_set_lcas_batch": lambda: L.kuq_set_lcas_batch(h, b.h_bases, b.h_offs, b.n, b.taxid.ctypes.data_as(u32p),
                                                               0, C.byref(missing)),
        })
    return calls


def _device_calls(calls):
    return {name: call for name, call in calls.items() if "_device" in name}


def test_slot_out_of_range(synthetic):
    clf = _classifier(synthetic)
    calls = _entry_points(clf, 2, Batch(synthetic, synthetic[4][:301]))     # the context has slots 0 and 1
    assert {name: call() for name, call in calls.items()} == dict.fromkeys(calls, E_INVALID_ARG)


@pytest.mark.parametrize("missing", ["bases", "offsets"])
def test_null_batch_buffers(synthetic, missing):
    clf = _classifier(synthetic)
    b = Batch(synthetic, synthetic[4][:301])
    if missing == "bases":
        b.h_bases = b.d_bases = None
    else:
        b.h_offs = b.d_offs = None
    calls = _entry_points(clf, 0, b)
    assert {name: call() for name, call in calls.items()} == dict.fromkeys(calls, E_INVALID_ARG)


def test_misaligned_device_bases(synthetic):
    clf = _classifier(synthetic)
    b = Batch(synthetic, synthetic[4][:301])
    b.d_bases += 1
    calls = _device_calls(_entry_points(clf, 0, b))
    assert {name: call() for name, call in calls.items()} == dict.fromkeys(calls, E_INVALID_ARG)


@pytest.mark.parametrize("over", ["reads", "bases"])
def test_batch_above_slot_capacity(synthetic, over):
    clf = _classifier(synthetic)
    # MAX_READS + 1 reads of 150 bases, or one read one base longer than a slot holds
    offs = synthetic[4][:MAX_READS + 2] if over == "reads" else np.array([0, MAX_BASES + 1], np.uint64)
    calls = _entry_points(clf, 0, Batch(synthetic, offs))
    assert {name: call() for name, call in calls.items()} == dict.fromkeys(calls, E_CAPACITY)


def test_preload_rule_device_calls_need_unit_ids(synthetic):
    clf = _classifier(synthetic)                # KUQ_HLL_PRELOAD: the sketches are per work unit
    b = Batch(synthetic, synthetic[4][:301])
    b.d_unit = None
    calls = _entry_points(clf, 0, b)
    calls = {name: calls[name] for name in ("kuq_classify_device", "kuq_resolve_device")}
    assert {name: call() for name, call in calls.items()} == dict.fromkeys(calls, E_INVALID_ARG)


def test_unread_batch_refuses_every_batch_call(synthetic):
    """After kuq_submit_batch on a slot, no batch call may launch on it before kuq_wait_batch has read the batch back:
    the wait returns what the same batch gives on a fresh context, and so do the per-taxon counters."""
    b = Batch(synthetic, synthetic[4][:301])
    clf = _classifier(synthetic)
    calls = _entry_points(clf, 0, b)
    clf._ck(calls["kuq_submit_batch"]())
    assert {name: call() for name, call in calls.items()} == dict.fromkeys(calls, E_STATE)
    got = clf.wait(0, b.offs, copy=True)
    clf.finish()
    fresh = _classifier(synthetic)
    want = fresh.classify(synthetic[3], b.offs)
    fresh.finish()
    for key in ("call", "n_windows", "n_classified"):
        assert np.array_equal(got[key], want[key]), key
    for i in range(b.n):
        assert binding.decode_runs(got, i) == binding.decode_runs(want, i), f"hit list of read {i}"
    got_counts, want_counts = clf.counts(), fresh.counts()
    for key in ("taxid", "n_reads", "n_kmers", "unique"):
        assert np.array_equal(got_counts[key], want_counts[key]), key
