"""The post-stream reduction (rows a11-a14: k_sparse_walk / k_sparse_alloc / k_sparse_median, the dense
k_sketch_reduce / k_winner fallback, k_stats / k_stats_hits) at database scale, against the NumPy
restatement in tests/_reduce_ref.py (needs a B200: `pytest -m gpu`).

The databases are built at hash level: every sketch is a sorted, distinct set of the query's own hashes
plus hashes the query lacks, all below 2^62 (so the table's keys fill the low quarter of the range and
the filtered stream route is the default one).  That puts any number of references, chain lengths and
multiplicities in front of the kernels with a query of a few Mbp.  Each shape asserts the regime it is
there for, so that it cannot shrink into one the small-database tests already cover."""
import numpy as np
import pytest

from hymet_b200 import msh as mshfmt
from hymet_b200 import screen as hs
from hymet_b200 import synth
from tests import _oracle as orc
from tests import _reduce_ref as rr

pytestmark = pytest.mark.gpu
K, S, LOW = 21, 1000, np.uint64(1 << 62)
RTOL = 1e-12
WALK_THREADS, AGG_SLOTS = 256, 2048       # k_sparse_walk's block size and per-CTA table (screen_kernels.cu)


def check(res, want, lo=0, hi=None):
    hi = len(res.shared) if hi is None else hi
    assert res.shared[lo:hi].tolist() == want.shared[lo:hi].tolist()
    assert res.median[lo:hi].tolist() == want.median[lo:hi].tolist()
    wi, gi = want.identity[lo:hi], res.identity[lo:hi]
    assert np.all(np.abs(gi - wi) <= RTOL * wi)
    wp, gp = want.pvalue[lo:hi], res.pvalue[lo:hi]
    tiny = wp < 1e-300
    assert np.all(gp[tiny] < 1e-299)
    assert np.all(np.abs(gp[~tiny] - wp[~tiny]) <= RTOL * wp[~tiny])


def check_hits(hits, dense):
    """finish_hits rows == the finish columns of the references with hits."""
    sel = dense.shared > 0
    assert hits.ref.tolist() == np.nonzero(sel)[0].tolist()
    assert hits.shared.tolist() == dense.shared[sel].tolist() and hits.median.tolist() == dense.median[sel].tolist()
    assert hits.identity.tolist() == dense.identity[sel].tolist() and hits.pvalue.tolist() == dense.pvalue[sel].tolist()
    assert hits.set_size == dense.set_size


def sketches(rng, sizes, present, absent, frac):
    """Per reference: round(size * frac) distinct hashes of `present`, the rest distinct hashes of `absent`
    (windows of random permutations), sorted.  -> offsets, hashes."""
    sizes = np.asarray(sizes, np.int64)
    n_p = np.minimum(np.rint(sizes * frac).astype(np.int64), len(present))
    n_a = sizes - n_p
    pp, pa = rng.permutation(present), rng.permutation(absent)
    rows = []
    for i, (a, b) in enumerate(zip(n_p, n_a)):
        s0, s1 = int(rng.integers(0, len(pp) - a + 1)), int(rng.integers(0, len(pa) - b + 1))
        rows.append(np.sort(np.concatenate([pp[s0:s0 + a], pa[s1:s1 + b]])))
    offsets = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    return offsets, (np.concatenate(rows) if rows else np.zeros(0, np.uint64)).astype(np.uint64)


def absent_hashes(rng, n, avoid):
    x = np.unique(rng.integers(1, 1 << 62, size=int(n * 1.1) + 16, dtype=np.uint64))
    x = np.setdiff1d(x, avoid, assume_unique=True)
    return rng.permutation(x)[:n]


@pytest.fixture(scope="module")
def query():
    """6 Mbp of random sequence in 100 kb contigs, some of them repeated (counts 1-6): ~1.5 M distinct
    hashes below 2^62."""
    rng = np.random.default_rng(2024)
    contigs = [synth.random_genome(rng, 100_000) for _ in range(60)]
    recs = contigs + [contigs[i] for i in rng.integers(0, 60, size=40)]
    text = synth.to_fasta(recs, "q")
    keys, counts = rr.query_hashes([synth.ASCII[r].tobytes() for r in recs], K)
    return text, keys, counts, keys[keys < LOW]


def reference(offsets, lengths, hashes, keys, counts, wta=False, seg_begin=None, seg_s=(S,), s=S):
    mix = keys[:s]
    sizes = [rr.set_size(mix, True, ss) for ss in seg_s]
    ec = rr.entry_counts(hashes, keys, counts)
    return rr.reduce(offsets, lengths, hashes, ec, K, sizes, seg_begin, wta), mix


def run(db, text, wta, **opts):
    scr = hs.Screen(db)
    for k_, v in opts.items():
        scr.set_option(k_, v)
    scr.reset()
    scr.feed_text(text, 4)
    r = scr.finish(wta)
    m = scr.mixture()
    scr.close()
    return r, m


def cta_distinct_refs(offsets, hashes, present_keys, n_touched, grid, rng):
    """k_sparse_walk's thread -> key assignment: thread t of the grid takes touched[t], touched[t + grid * 256],
    ...  The order of touched[] is the order of first increments, so it is modelled as a random permutation.
    -> the number of distinct references each CTA's walk sees."""
    N = len(offsets) - 1
    ref = np.repeat(np.arange(N, dtype=np.int64), np.diff(offsets.astype(np.int64)))
    held = np.isin(hashes, present_keys)
    key_rank = np.searchsorted(present_keys, hashes[held])
    pos = rng.permutation(len(present_keys))[key_rank]            # position of each holder's key in touched[]
    cta = (pos % (grid * WALK_THREADS)) // WALK_THREADS
    pairs = np.unique(cta * N + ref[held])
    return np.bincount(pairs // N, minlength=grid)


def test_a_wide_uneven_sketches(query):
    """30 000 references of very uneven sizes, empty sketches first, in the middle and last: every CTA of the
    walk sees more than 2048 distinct references (the per-CTA table overflows to global atomics and to
    seg_fill), and e * N / E is a poor guess of the owning reference."""
    import torch
    text, keys, counts, present = query
    rng = np.random.default_rng(7)
    N = 30_000
    sizes = rng.choice([0, 1, 2, 17, 300, 1000, 4000], size=N, p=[0.03, 0.10, 0.12, 0.20, 0.30, 0.20, 0.05])
    sizes[[0, N // 2, N - 1]] = 0
    absent = absent_hashes(rng, 4_000_000, keys)
    offsets, hashes = sketches(rng, sizes, present, absent, np.where(sizes < 300, 0.9, 0.4))
    lengths = rng.integers(10_000, 5_000_000, size=N).astype(np.uint64)
    E = len(hashes)
    db = hs.Database.from_arrays(K, S, 42, offsets, hashes, lengths)
    assert db.info.max_key < LOW
    # entries whose e * N / E guess (ref_of_entry) is more than one reference away
    guess = np.minimum((np.arange(E, dtype=np.float64) * (N / (E + 1))).astype(np.int64), N - 1)
    owner = np.repeat(np.arange(N), sizes)
    assert np.mean(np.abs(guess - owner) > 1) > 0.10
    for wta in (False, True):
        want, mix = reference(offsets, lengths, hashes, keys, counts, wta)
        res, m = run(db, text, wta)
        assert res.stats["reduce_path"] == 0
        check(res, want)
        assert m.tolist() == mix.tolist() and res.set_size == want.set_sizes[0]
        if not wta:
            assert int(want.shared.sum()) < 1 << 23      # the pairs fit the default depths buffer: no fallback
            assert res.stats["n_hit_refs"] == int((want.shared > 0).sum()) > 0.9 * N
            per_cta = cta_distinct_refs(offsets, hashes, present[np.isin(present, hashes)], res.stats["n_touched"],
                                        4 * torch.cuda.get_device_properties(0).multi_processor_count, rng)
            assert per_cta.min() > AGG_SLOTS, per_cta.min()
            res0, _ = run(db, text, False, filter=0)          # the probe-everything stream feeds the same reduction
            check(res0, want)
            assert res0.stats["n_probes"] == res0.stats["n_valid_kmers"]
    db.close()


def test_a_more_references_than_entries(query):
    """N > E (mostly empty sketches): ref_of_entry has no scale and binary-searches every entry."""
    text, keys, counts, present = query
    rng = np.random.default_rng(8)
    N = 50_000
    sizes = np.zeros(N, np.int64)
    full = rng.choice(N - 2, size=4_000, replace=False) + 1
    sizes[full] = rng.choice([1, 2, 17], size=len(full))
    sizes[full[:10]] = 300
    absent = absent_hashes(rng, 200_000, keys)
    offsets, hashes = sketches(rng, sizes, present, absent, 0.7)
    lengths = rng.integers(1_000, 100_000, size=N).astype(np.uint64)
    assert len(hashes) < N
    db = hs.Database.from_arrays(K, S, 42, offsets, hashes, lengths)
    for wta in (False, True):
        want, mix = reference(offsets, lengths, hashes, keys, counts, wta)
        res, m = run(db, text, wta)
        assert res.stats["reduce_path"] == 0 and int((want.shared > 0).sum()) > 2_000
        check(res, want)
        assert m.tolist() == mix.tolist() and res.set_size == want.set_sizes[0]
    db.close()


def test_b_hot_keys_eight_files_wta(query, tmp_path):
    """8 sketch files of 2 000 references with different s; 200 hot keys held by every reference (chains of
    16 000 entries, walked once per file by chain_winner); exact duplicates with equal lengths (full ties:
    the higher index wins) and with different lengths; relatives that lost some keys."""
    text, keys, counts, present = query
    rng = np.random.default_rng(9)
    seg_s = [1000, 400, 700, 250, 1000, 550, 850, 300]
    n_per = 2_000
    hot = rng.choice(present, size=200, replace=False)
    rest = np.setdiff1d(present, hot)
    absent = absent_hashes(rng, 3_000_000, keys)
    paths, all_off, all_h, all_len = [], [0], [], []
    for j, s in enumerate(seg_s):
        sizes = np.full(n_per, s - 200)
        sizes[rng.random(n_per) < 0.2] //= 3
        frac = rng.uniform(0.2, 0.9, size=n_per)
        o, h = sketches(rng, sizes, rest, absent, frac)
        rows = [np.sort(np.concatenate([r, hot])) for r in np.split(h, o[1:-1].astype(np.int64))]
        lengths = rng.integers(1_000_000, 1_000_050, size=n_per).astype(np.uint64)   # many equal lengths
        for i in range(1, n_per):
            u = rng.random()
            src = int(rng.integers(0, i))
            if u < 0.15:      # exact duplicate; equal length two times in three
                rows[i] = rows[src].copy()
                if rng.random() < 0.67:
                    lengths[i] = lengths[src]
            elif u < 0.25:    # relative: some of the source's hashes replaced by absent ones
                r = rows[src].copy()
                drop = rng.random(len(r)) < 0.05
                drop &= ~np.isin(r, hot)
                r[drop] = rng.choice(absent, size=int(drop.sum()))
                rows[i] = np.unique(r)
                if rng.random() < 0.5:
                    lengths[i] = lengths[src]
        off = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.uint64)
        h = np.concatenate(rows)
        db_j = mshfmt.SketchDB(k=K, s=s, names=["f%d_r%d" % (j, i) for i in range(n_per)], comments=[""] * n_per,
                               lengths=lengths, offsets=off, hashes=h)
        p = str(tmp_path / ("part%d.msh" % j))
        mshfmt.write_msh(p, db_j)
        paths.append(p)
        all_off.extend((off[1:] + np.uint64(all_off[-1])).tolist()); all_h.append(h); all_len.append(lengths)
    offsets = np.array(all_off, np.uint64)
    hashes = np.concatenate(all_h); lengths = np.concatenate(all_len)
    _, holders = np.unique(hashes, return_counts=True)
    assert holders.max() >= 8 * n_per                      # the longest chain in next[]
    db = hs.Database.load_msh_multi(paths)
    segs = db.segments
    assert db.segment_s == seg_s and len(segs) == 8 and db.s == max(seg_s)
    seg_begin = [b for b, _ in segs] + [segs[-1][1]]
    for wta in (False, True):
        want, mix = reference(offsets, lengths, hashes, keys, counts, wta, seg_begin, seg_s, db.s)
        scr = hs.Screen(db)
        scr.feed_text(text, 4)
        res = scr.finish(wta)
        assert res.stats["reduce_path"] == 0
        check(res, want)
        assert scr.mixture().tolist() == mix.tolist()
        for j in range(8):
            assert scr.segment_set_size(j) == want.set_sizes[j]
        scr.close()
        if wta:   # every file hands each hot key to exactly one of its references
            assert int(want.shared.sum()) < int(plain_sum)
        plain_sum = want.shared.sum()
    db.close()


def tandem_query(rng, n_units, unit_len):
    """Tandem repeats of random units, one record each, at copy numbers from 1 to 10^6 (log-uniform):
    counts per key span 20 bits."""
    copies = np.rint(10.0 ** rng.uniform(0, 6, size=n_units)).astype(np.int64)
    copies[:2] = (1, 10 ** 6)
    units = [synth.ASCII[synth.random_genome(rng, unit_len)].tobytes() for _ in range(n_units)]
    text = b"".join(b">t%d\n" % i + u * int(c) + b"\n" for i, (u, c) in enumerate(zip(units, copies)))
    keys, counts = rr.merge_counts(*[rr.tandem_counts(u, int(c), K) for u, c in zip(units, copies)])
    return text, keys, counts


def test_c_deep_multiplicities():
    """Counts up to ~10^6 on every key, many even `shared`: sparse and dense paths, columns and hit rows, and
    the probe-everything stream, all equal the restatement."""
    rng = np.random.default_rng(10)
    text, keys, counts = tandem_query(rng, 120, 40)
    present = keys[keys < LOW]
    assert int(counts.max()) >= 10 ** 6 - 1 and int(counts.min()) <= 1
    N = 3_000
    sizes = rng.integers(2, 400, size=N)
    absent = absent_hashes(rng, 500_000, keys)
    offsets, hashes = sketches(rng, sizes, present, absent, 0.5)
    lengths = rng.integers(1_000, 1_010, size=N).astype(np.uint64)
    db = hs.Database.from_arrays(K, S, 42, offsets, hashes, lengths)
    for wta in (False, True):
        want, mix = reference(offsets, lengths, hashes, keys, counts, wta)
        if not wta:
            assert int((want.shared % 2 == 0)[want.shared > 0].sum()) > 200
        for sparse in (1, 0):
            scr = hs.Screen(db)
            scr.set_option("sparse", sparse)
            scr.reset()
            scr.feed_text(text, 4)
            hits = scr.finish_hits(wta)
            res = scr.finish(wta)
            assert res.stats["reduce_path"] == (0 if sparse else 1) == hits.stats["reduce_path"]
            check(res, want)
            check_hits(hits, res)
            assert scr.mixture().tolist() == mix.tolist() and res.set_size == want.set_sizes[0]
            scr.close()
    res0, _ = run(db, text, False, filter=0)
    check(res0, reference(offsets, lengths, hashes, keys, counts)[0])
    db.close()


def test_d_counts_at_the_32bit_edge():
    """One key (poly-A) counted 2^32 - 1, 2^32 and 2^32 + 5 times: device-resident packed words fed again and
    again.  Each hs_screen_feed_packed_device call is its own chunk (launch_chunk streams positions
    [0, n_bases) of it alone), so k-mers never span two feeds and a feed of n bases adds n - k + 1.
    2^32 - 1 stays on the O(present) path; a count that wraps sends the screen to the dense kernels,
    which see it mod 2^32 (0: no hit; 5)."""
    import torch
    rng = np.random.default_rng(12)
    M = 1 << 30
    seq = torch.zeros((M + 128) // 32, dtype=torch.int64, device="cuda")       # poly-A: code 0, all valid
    inv = torch.zeros((M + 128) // 32, dtype=torch.int32, device="cuda")
    unit = synth.ASCII[synth.random_genome(rng, 37)].tobytes()
    u_text = b">u\n" + unit * 3000 + b"\n"
    s2, i2, n2, _ = hs.pack_text(u_text)
    seq2 = torch.from_numpy(s2.view(np.int64).copy()).cuda(); inv2 = torch.from_numpy(i2.view(np.int32).copy()).cuda()
    polya = rr.tandem_counts(b"A" * 32, 1, K)[0]
    ukeys, ucounts = rr.tandem_counts(unit, 3000, K)
    assert len(polya) == 1 and polya[0] not in ukeys
    pa = polya[0]
    absent = absent_hashes(rng, 10_000, np.concatenate([polya, ukeys]))
    refs = [[pa], [pa] + list(ukeys[:3]), list(ukeys) + list(absent[:50]), [], list(absent[50:90]),
            [pa] + list(ukeys[3:5]) + list(absent[90:95])]
    rows = [np.unique(np.array(r, np.uint64)) for r in refs]
    offsets = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.uint64)
    hashes = np.concatenate(rows); lengths = np.array([500, 600, 700, 0, 800, 900], np.uint64)
    N = len(rows)
    db = hs.Database.from_arrays(K, S, 42, offsets, hashes, lengths)
    scr = hs.Screen(db)
    for tail, path in ((99, 0), (100, 1), (105, 1)):
        total = 4 * (M - K + 1) + tail - K + 1
        scr.reset()
        for _ in range(4):
            scr.feed_packed_device(seq.data_ptr(), inv.data_ptr(), M)
        scr.feed_packed_device(seq.data_ptr(), inv.data_ptr(), tail)
        scr.feed_packed_device(seq2.data_ptr(), inv2.data_ptr(), n2)
        keys, counts = rr.merge_counts((polya, np.array([total], np.uint64)), (ukeys, ucounts))
        want, mix = reference(offsets, lengths, hashes, keys, counts, s=S)
        hits = scr.finish_hits(False)
        res = scr.finish(False)
        assert res.stats["n_valid_kmers"] == total + int(ucounts.sum())
        assert res.stats["reduce_path"] == path == hits.stats["reduce_path"], (tail, res.stats)
        check(res, want)
        check_hits(hits, res)
        assert scr.mixture().tolist() == mix.tolist() and res.set_size == want.set_sizes[0]
        assert res.median[0] == (4294967295 if tail == 99 else 0 if tail == 100 else 5)
        for wta in (True,):
            w, _ = reference(offsets, lengths, hashes, keys, counts, wta)
            scr.reset()
            for _ in range(4):
                scr.feed_packed_device(seq.data_ptr(), inv.data_ptr(), M)
            scr.feed_packed_device(seq.data_ptr(), inv.data_ptr(), tail)
            scr.feed_packed_device(seq2.data_ptr(), inv2.data_ptr(), n2)
            check(scr.finish(True), w)
    # the handle is clean afterwards: an ordinary query on it equals the restatement
    scr.reset()
    scr.feed_text(u_text, 2)
    res = scr.finish(False)
    want, _ = reference(offsets, lengths, hashes, ukeys, ucounts)
    assert res.stats["reduce_path"] == 0
    check(res, want)
    scr.close(); db.close()
    del seq, inv, seq2, inv2
    torch.cuda.empty_cache()
    assert N == 6


def test_e_default_caps_fall_back_to_dense(query):
    """E > 2^25 and more present (key, reference) pairs than the default pair_cap (E / 4): the depths buffer
    cannot hold them, the dense kernels answer, with no environment override.  A small query on the same
    handle afterwards is back on the O(present) path."""
    text, keys, counts, present = query
    rng = np.random.default_rng(13)
    N, size = 34_000, 1000
    assert N * size > 1 << 25
    absent = absent_hashes(rng, 4_000_000, keys)
    offsets, hashes = sketches(rng, np.full(N, size), present, absent, 0.3)
    lengths = rng.integers(1_000_000, 2_000_000, size=N).astype(np.uint64)
    E = len(hashes)
    want, mix = reference(offsets, lengths, hashes, keys, counts)
    assert int(want.shared.sum()) > E // 4 and len(present) < E // 8
    db = hs.Database.from_arrays(K, S, 42, offsets, hashes, lengths)
    scr = hs.Screen(db)
    scr.feed_text(text, 4)
    res = scr.finish(False)
    assert res.stats["reduce_path"] == 1
    check(res, want)
    assert scr.mixture().tolist() == mix.tolist()
    small = text[:text.index(b">", 300_000)]
    k2, c2 = rr.query_hashes(rr.fasta_records(small), K)
    scr.reset()
    scr.feed_text(small, 2)
    res = scr.finish(False)
    assert res.stats["reduce_path"] == 0
    check(res, reference(offsets, lengths, hashes, k2, c2)[0])
    scr.close(); db.close()
