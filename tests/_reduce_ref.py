"""Rows a11-a14 of `mash screen` restated in NumPy, for databases too large for the C oracle's
per-reference loops.

TEST INFRASTRUCTURE.  Counts per stored hash come from the C oracle's hash function (canonical,
N-aware) and np.unique, independently of the GPU; everything after that is vectorised array work,
so that 3 * 10^7 entries take seconds.  Identity, p-value and set size are the oracle's own
functions (orc_identity, orc_pvalue, orc_set_size), called once per reference with hits.

The rules restated here, with the labels the oracle uses:
  S8   a count is kept mod 2^32 (the oracle's and the GPU's counters are uint32)
  S11  shared = the reference's entries whose count is non-zero
  S12  median = element shared // 2 of the reference's sorted non-zero counts
  S17  -w, per source file: each present key goes to one holder, the best by (identity, length, index)
  S10  set size from the s smallest distinct query hashes
  S13/S14 identity and p-value
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np

from tests import _oracle as orc

WRAP = np.uint64(1 << 32)


def query_hashes(records: Sequence[bytes], k: int, seed: int = 42):
    """Distinct canonical hashes of all valid k-mers of the records (ascending) and how often each occurs.
    k-mers never span two records."""
    parts = []
    for r in records:
        h, v = orc.hash_sequence(r, k, seed)
        parts.append(h[v])
    allh = np.concatenate(parts) if parts else np.zeros(0, np.uint64)
    keys, counts = np.unique(allh, return_counts=True)
    return keys, counts.astype(np.uint64)


def fasta_records(text: bytes):
    """Sequences of a FASTA text, one bytes object per record, upper-cased (the oracle's parser does the same)."""
    out = []
    for rec in text.split(b">")[1:]:
        nl = rec.find(b"\n")
        body = rec[nl + 1:] if nl >= 0 else b""
        out.append(body.replace(b"\n", b"").replace(b"\r", b"").upper())
    return out


def tandem_counts(unit: bytes, copies: int, k: int, seed: int = 42):
    """Closed form of query_hashes([unit * copies]) for k <= len(unit): the k-mer at cyclic offset o
    occurs `copies` times when o <= len(unit) - k and `copies` - 1 times otherwise."""
    u = len(unit)
    assert k <= u and copies >= 1
    h, v = orc.hash_sequence(unit + unit[:k - 1], k, seed)
    mult = np.where(np.arange(u) <= u - k, copies, copies - 1).astype(np.uint64)
    h, mult = h[v], mult[v]
    keys, inv = np.unique(h, return_inverse=True)
    counts = np.zeros(len(keys), np.uint64)
    np.add.at(counts, inv, mult)
    keep = counts > 0
    return keys[keep], counts[keep]


def merge_counts(*pairs):
    """Sum several (keys, counts) pairs key by key."""
    keys = np.concatenate([p[0] for p in pairs])
    cnts = np.concatenate([p[1] for p in pairs])
    u, inv = np.unique(keys, return_inverse=True)
    out = np.zeros(len(u), np.uint64)
    np.add.at(out, inv, cnts)
    return u, out


def entry_counts(hashes: np.ndarray, keys: np.ndarray, counts: np.ndarray) -> np.ndarray:
    """Count of every stored hash (uint64, not yet reduced mod 2^32); 0 for hashes the query lacks."""
    hashes = np.asarray(hashes, np.uint64)
    out = np.zeros(len(hashes), np.uint64)
    if len(keys) and len(hashes):
        pos = np.minimum(np.searchsorted(keys, hashes), len(keys) - 1)
        hit = keys[pos] == hashes
        out[hit] = counts[pos[hit]]
    return out


def set_size(mixture: np.ndarray, use64: bool, s_limit: Optional[int] = None) -> int:
    m = np.ascontiguousarray(mixture[:s_limit] if s_limit is not None else mixture, np.uint64)
    return int(orc.lib().orc_set_size(orc._p(m, orc.C.c_uint64), len(m), int(use64)))


@dataclass
class Reduced:
    shared: np.ndarray     # uint64 [N]
    median: np.ndarray     # uint32 [N]
    identity: np.ndarray   # float64 [N]
    pvalue: np.ndarray     # float64 [N]
    set_sizes: list        # per source file


def _upper_median(ref: np.ndarray, cnt: np.ndarray, shared: np.ndarray) -> np.ndarray:
    """S12 for every reference at once: sort the (reference, count) pairs and take element shared // 2."""
    N = len(shared)
    median = np.zeros(N, np.uint32)
    if not len(ref):
        return median
    order = np.lexsort((cnt, ref))
    r_s, c_s = ref[order], cnt[order]
    refs = np.nonzero(shared)[0]
    first = np.searchsorted(r_s, refs)
    median[refs] = c_s[first + shared[refs].astype(np.int64) // 2]
    return median


def reduce(offsets, lengths, hashes, counts, k: int, set_sizes: Sequence[int], seg_begin=None,
           wta: bool = False) -> Reduced:
    """shared, median, identity and p-value of every reference from the count of every stored hash.

    offsets [N+1], lengths [N], hashes [E] (identify keys for -w), counts [E] (any width: reduced mod 2^32
    here), seg_begin [F+1] (first reference of each source file; default one file), set_sizes [F]."""
    offsets = np.asarray(offsets, np.uint64).astype(np.int64)
    lengths = np.asarray(lengths, np.uint64)
    hashes = np.asarray(hashes, np.uint64)
    N, E = len(offsets) - 1, int(offsets[-1])
    seg_begin = [0, N] if seg_begin is None else [int(x) for x in seg_begin]
    assert len(set_sizes) == len(seg_begin) - 1
    c32 = (np.asarray(counts, np.uint64) % WRAP).astype(np.uint32)
    sizes = np.diff(offsets)
    ref = np.repeat(np.arange(N, dtype=np.int64), sizes)
    assert len(ref) == E == len(c32)
    keep = c32 != 0
    shared = np.bincount(ref[keep], minlength=N).astype(np.uint64)
    if wta:
        score = np.array([identity_of(int(shared[i]), int(sizes[i]), k) for i in range(N)])
        win = np.zeros(E, bool)
        for j in range(len(seg_begin) - 1):
            lo, hi = offsets[seg_begin[j]], offsets[seg_begin[j + 1]]
            idx = lo + np.nonzero(keep[lo:hi])[0]
            if not len(idx):
                continue
            r = ref[idx]
            order = np.lexsort((r, lengths[r], score[r], hashes[idx]))    # last key is the primary one
            hk = hashes[idx][order]
            last = np.ones(len(order), bool)
            last[:-1] = hk[1:] != hk[:-1]                                  # the best holder of each key
            win[idx[order[last]]] = True
        keep = win
        shared = np.bincount(ref[keep], minlength=N).astype(np.uint64)
    median = _upper_median(ref[keep], c32[keep], shared)
    identity = np.where(sizes == 0, 1.0, 0.0)      # shared == size == 0 is identity 1 (orc_identity)
    pvalue = np.ones(N, np.float64)
    kmer_space = 4.0 ** k
    for j in range(len(seg_begin) - 1):
        for i in np.nonzero(shared[seg_begin[j]:seg_begin[j + 1]])[0] + seg_begin[j]:
            x, sz = int(shared[i]), int(sizes[i])
            identity[i] = orc.lib().orc_identity(x, sz, k)
            pvalue[i] = orc.lib().orc_pvalue(x, int(set_sizes[j]), kmer_space, sz)
    return Reduced(shared, median, identity, pvalue, list(set_sizes))


def identity_of(shared: int, size: int, k: int) -> float:
    return float(orc.lib().orc_identity(shared, size, k))
