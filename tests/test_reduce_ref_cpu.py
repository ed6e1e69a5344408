"""The NumPy restatement of rows a11-a14 (tests/_reduce_ref.py) against the C oracle, field for field.
Runs without a GPU: it pins the reference that tests/test_gpu_reduce_scale.py holds the kernels to."""
import json
import os

import numpy as np
import pytest

from hymet_b200 import synth
from tests import _oracle as orc
from tests import _reduce_ref as rr

K = 21


def oracle_db_arrays(genomes, k, s):
    hs_list, lens = [], []
    for g in genomes:
        h, ln = orc.sketch_text(synth.to_fasta([g], "g"), k, s)
        hs_list.append(h); lens.append(ln)
    offsets = np.concatenate([[0], np.cumsum([len(h) for h in hs_list])]).astype(np.uint64)
    return offsets, np.concatenate(hs_list), np.array(lens, np.uint64)


def restate(offsets, hashes, lengths, fasta, k, s, wta, seg=None):
    keys, counts = rr.query_hashes(rr.fasta_records(fasta), k)
    mix = keys[:s]
    seg_s = [s] if seg is None else [ss for _, ss in seg]
    seg_begin = None if seg is None else [0] + list(np.cumsum([n for n, _ in seg]))
    sizes = [rr.set_size(mix, orc.lib().orc_use64(k), ss) for ss in seg_s]
    ec = rr.entry_counts(hashes, keys, counts)
    return rr.reduce(offsets, lengths, hashes, ec, k, sizes, seg_begin, wta), mix, ec


def assert_same(got, want, lo=0, hi=None):
    hi = len(want.shared) + lo if hi is None else hi
    assert got.shared[lo:hi].tolist() == want.shared.tolist()
    assert got.median[lo:hi].tolist() == want.median.tolist()
    assert got.identity[lo:hi].tolist() == want.identity.tolist()
    assert got.pvalue[lo:hi].tolist() == want.pvalue.tolist()


@pytest.mark.parametrize("wta", [False, True])
def test_small_golden_case(golden_dir, wta):
    g = json.load(open(os.path.join(golden_dir, "screen_small.json")))
    hsl = [np.array([int(h) for h in r["hashes"]], np.uint64) for r in g["db"]]
    offsets = np.concatenate([[0], np.cumsum([len(h) for h in hsl])]).astype(np.uint64)
    hashes = np.concatenate(hsl)
    lengths = np.array([r["length"] for r in g["db"]], np.uint64)
    fasta = g["fasta"].encode()
    want = orc.OracleDB.from_arrays(g["k"], g["s"], g["seed"], offsets, hashes, lengths).screen_text(fasta, wta=wta)
    got, mix, ec = restate(offsets, hashes, lengths, fasta, g["k"], g["s"], wta)
    assert_same(got, want)
    assert got.set_sizes == [want.set_size]
    assert mix.tolist() == want.mixture.tolist()
    assert ec.tolist() == want.counts_per_entry.tolist()
    assert int(want.shared.sum()) > 0


@pytest.fixture(scope="module")
def cluster_db():
    """cluster_case's shape at a third of its size: relatives, length-perturbed members, exact duplicates
    (full -w ties), unrelated genomes."""
    rng = np.random.default_rng(11)
    genomes = []
    for c in range(4):
        anc = synth.random_genome(rng, 30_000)
        for m in range(5):
            g = synth.mutate(anc, float(rng.uniform(0.01, 0.05)), rng)
            genomes.append(g if m < 2 else g[:30_000 - int(rng.integers(1, 999))])
        genomes.append(genomes[-1].copy())
    genomes += [synth.random_genome(rng, 30_000) for _ in range(10)]
    offsets, hashes, lengths = oracle_db_arrays(genomes, K, 1000)
    fasta = synth.to_fasta(synth.cut_contigs(rng, genomes[::5] + genomes[24:28], 300_000, 0.005, median=5000.0),
                           "c", lower_frac=0.05, rng=rng)
    return genomes, offsets, hashes, lengths, fasta


@pytest.mark.parametrize("wta", [False, True])
def test_cluster_case(cluster_db, wta):
    _, offsets, hashes, lengths, fasta = cluster_db
    want = orc.OracleDB.from_arrays(K, 1000, 42, offsets, hashes, lengths).screen_text(fasta, threads=2, wta=wta)
    got, mix, ec = restate(offsets, hashes, lengths, fasta, K, 1000, wta)
    assert_same(got, want)
    assert got.set_sizes == [want.set_size] and mix.tolist() == want.mixture.tolist()
    assert int((want.shared > 0).sum()) > 10 and int(np.diff(want.shared.astype(np.int64)).max()) > 0
    assert int((want.shared % 2 == 0)[want.shared > 0].sum()) > 0     # even shared: the upper median matters


@pytest.mark.parametrize("wta", [False, True])
def test_three_files_with_different_sketch_sizes(cluster_db, wta):
    """-w per source file: one concatenated database, each file's slice equals the oracle on that file alone."""
    genomes, _, _, _, fasta = cluster_db
    files = [(list(range(0, 14)), 1000), (list(range(6, 24)) + [0], 1000), (list(range(18, 34)) + [3, 9], 400)]
    arrays = [oracle_db_arrays([genomes[i] for i in idx], K, s) for idx, s in files]
    offsets = np.concatenate([[0]] + [a[0][1:] + sum(int(b[0][-1]) for b in arrays[:j]) for j, a in enumerate(arrays)])
    hashes = np.concatenate([a[1] for a in arrays])
    lengths = np.concatenate([a[2] - np.arange(len(a[2]), dtype=np.uint64) % np.uint64(3) for a in arrays])
    got, mix, _ = restate(offsets.astype(np.uint64), hashes, lengths, fasta, K, 1000, wta,
                          seg=[(len(idx), s) for idx, s in files])
    b = 0
    for j, (idx, s) in enumerate(files):
        n = len(idx)
        want = orc.OracleDB.from_arrays(K, s, 42, arrays[j][0], arrays[j][1], lengths[b:b + n]).screen_text(
            fasta, threads=2, wta=wta)
        assert_same(got, want, b, b + n)
        assert got.set_sizes[j] == want.set_size and mix[:s].tolist() == want.mixture.tolist()
        b += n


def test_tandem_closed_form_equals_hashing():
    rng = np.random.default_rng(3)
    for u in (21, 32, 57):
        unit = synth.ASCII[synth.random_genome(rng, u)].tobytes()
        for copies in (1, 2, 5, 13):
            assert [x.tolist() for x in rr.tandem_counts(unit, copies, K)] == \
                   [x.tolist() for x in rr.query_hashes([unit * copies], K)]
    # poly-A: one canonical key, n - k + 1 occurrences
    keys, counts = rr.tandem_counts(b"A" * 32, 1000, K)
    assert len(keys) == 1 and int(counts[0]) == 32 * 1000 - K + 1


def test_counts_at_the_32bit_edge():
    """S8 by hand: a count of 2^32 - 1 is the median; 2^32 wraps to 0 (no hit); 2^32 + 5 wraps to 5."""
    offsets = np.array([0, 1, 3, 6, 7], np.uint64)
    hashes = np.array([10, 10, 20, 10, 20, 30, 20], np.uint64)
    lengths = np.array([100, 100, 100, 100], np.uint64)
    top = (1 << 32) - 1
    for c10, shared, median in ((top, [1, 2, 3, 1], [top, top, 9, 7]),
                                (1 << 32, [0, 1, 2, 1], [0, 7, 9, 7]),
                                ((1 << 32) + 5, [1, 2, 3, 1], [5, 7, 7, 7])):
        keys = np.array([10, 20, 30], np.uint64)
        counts = np.array([c10, 7, 9], np.uint64)
        ec = rr.entry_counts(hashes, keys, counts)
        got = rr.reduce(offsets, lengths, hashes, ec, K, [10 ** 6])
        assert got.shared.tolist() == shared and got.median.tolist() == median, c10
        assert got.pvalue[np.array(shared) == 0].tolist() == [1.0] * shared.count(0)
        w = rr.reduce(offsets, lengths, hashes, ec, K, [10 ** 6], wta=True)
        assert int(w.shared.sum()) == len(set(keys[rr.entry_counts(keys, keys, counts) % rr.WRAP != 0].tolist()))


def test_empty_sketches_and_identity_rule():
    """Empty sketches: shared 0, identity 1 (orc_identity(0, 0)), p-value 1 -- what the oracle prints."""
    offsets = np.array([0, 0, 2, 2, 3, 3], np.uint64)
    hashes = np.array([5, 6, 5], np.uint64)
    lengths = np.array([0, 50, 0, 40, 0], np.uint64)
    want = orc.OracleDB.from_arrays(K, 10, 42, offsets, hashes, lengths)
    assert want.n_refs == 5
    got = rr.reduce(offsets, lengths, hashes, np.array([3, 0, 3], np.uint64), K, [1000])
    assert got.shared.tolist() == [0, 1, 0, 1, 0] and got.identity.tolist()[0::2] == [1.0, 1.0, 1.0]
    assert got.median.tolist() == [0, 3, 0, 3, 0] and got.pvalue[0] == 1.0
