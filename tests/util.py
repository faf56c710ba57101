"""Shared helpers for the parity tests (host-side only; no product logic)."""
import hashlib
import json
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "mini")
# answers of the unmodified reference on the tests' seeded inputs (tests/golden/make_golden_reference.py)
REFERENCE = os.path.join(ROOT, "tests", "golden", "reference")
AMBIG = 0xFFFFFFFF


def digest(*parts):
    """sha256 over arrays / bytes / str in order: pins a reference output too large to store in full."""
    h = hashlib.sha256()
    for p in parts:
        if isinstance(p, str):
            p = p.encode()
        elif isinstance(p, np.ndarray):
            p = np.ascontiguousarray(p).tobytes()
        h.update(p)
    return h.hexdigest()


def reference_json(name):
    with open(os.path.join(REFERENCE, name)) as f:
        return json.load(f)


def read_fasta(path):
    """FastaReader::next_sequence (seqreader.cpp:34-79): id = first whitespace token of the header, sequence
    lines concatenated (a trailing '\\r' of CRLF files stays in the sequence)."""
    ids, seqs = [], []
    cur = None
    with open(path, "rb") as f:
        for line in f.read().split(b"\n"):
            if line.startswith(b">"):
                if cur is not None:
                    seqs.append(b"".join(cur))
                hdr = line[1:].split()
                ids.append(hdr[0].decode() if hdr else "")
                cur = []
            elif cur is not None:
                cur.append(line)
    if cur is not None:
        seqs.append(b"".join(cur))
    return ids, seqs


def read_fastq(path):
    """FastqReader::next_sequence (seqreader.cpp:93-129)."""
    ids, seqs = [], []
    with open(path, "rb") as f:
        lines = f.read().split(b"\n")
    i = 0
    while i + 3 < len(lines) and lines[i].startswith(b"@"):
        ids.append(lines[i][1:].split()[0].decode())
        seqs.append(lines[i + 1])
        i += 4
    return ids, seqs


def hitlist(codes):
    """hitlist_string (classify.cpp:826-861) from per-window codes (AMBIG = ambiguous)."""
    if len(codes) == 0:
        return "0:0"
    codes = np.asarray(codes, np.uint32)
    brk = np.nonzero(np.diff(codes.astype(np.int64)) != 0)[0] + 1
    starts = np.concatenate([[0], brk])
    ends = np.concatenate([brk, [len(codes)]])
    return " ".join(("A" if codes[s] == AMBIG else str(int(codes[s]))) + ":" + str(int(e - s))
                    for s, e in zip(starts, ends))


def kraken_lines(ids, seqs, calls, codes, code_off):
    """Kraken output lines (classify.cpp:980-1010), default flags."""
    out = []
    for i, (rid, s) in enumerate(zip(ids, seqs)):
        c = codes[int(code_off[i]):int(code_off[i + 1])]
        out.append(f"{'C' if calls[i] else 'U'}\t{rid}\t{int(calls[i])}\t{len(s)}\t{hitlist(c)}\n")
    return "".join(out)


def parse_report(path):
    """report.tsv → {taxID: dict(pct, reads, taxReads, kmers, dup, cov, rank, name)} (taxdb.hpp:1078-1123)."""
    rows = {}
    with open(path) as f:
        hdr = None
        for line in f:
            if line.startswith("#"):
                continue
            parts = line.rstrip("\n").split("\t")
            if hdr is None:
                hdr = parts
                continue
            d = dict(zip(hdr, parts))
            rows[int(d["taxID"])] = dict(pct=d["%"], reads=int(d["reads"]), taxReads=int(d["taxReads"]),
                                         kmers=int(d["kmers"]), dup=d["dup"], cov=d["cov"], rank=d["rank"],
                                         name=d["taxName"])
    return rows


def clade_members(tax_rows, counted_taxids):
    """TaxReport ctor (taxdb.hpp:935-951): for every counted taxon that has a taxDB entry, it is a member of the
    clade of each of its ancestors (walk parent pointers; parent is NULL for the root / unknown parents).
    Taxon 0 always has an entry ("unclassified", taxdb.hpp:596)."""
    parent = {t: p for t, p, _, _ in tax_rows}
    ids = set(parent) | {0}
    members = {}
    for t in counted_taxids:
        t = int(t)
        if t not in ids:
            continue
        node, seen = t, set()
        while node is not None and node not in seen:
            seen.add(node)
            members.setdefault(node, []).append(t)
            p = parent.get(node)
            node = p if (p is not None and p != node and p in ids and node != 0) else None
    return members
