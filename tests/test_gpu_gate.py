"""The stream kernel's range gate on the hash's high word, on the GPU (needs a B200: `pytest -m gpu`).

For 64-bit hashes the screen kernel decides `h <= gate` from the high words of the two MurmurHash3
finalizer outputs, whose sum is the hash's high word or one less (the carry out of the low words), and
finishes the hash only for the k-mers that pass (kmer_core.cuh: murmur_finish_hi_floor).  Here the
largest key of the database is placed exactly on a query k-mer's hash, once where that k-mer's low-word
add carries and once where it does not, and one below it.  Shared counts and medians must equal the
oracle's and those of the probe-everything kernel, which has no gate.

The kernel's gate is max(max_key, mixture threshold).  The mixture threshold of a launch that starts an
empty mixture is a cap that falls with the launch's length, so the query is one packed feed (one launch)
long enough for that cap to lie below max_key -- which the test checks from the launch's own count of
mixture offers -- and the database's keys stay below 1 % of the hash range, so it has no Bloom tier.
"""
import numpy as np
import pytest

from hymet_b200 import screen as hs
from hymet_b200 import synth
from tests import _oracle as orc

pytestmark = pytest.mark.gpu
M64 = (1 << 64) - 1
S = 1000


def canonical(kmer: bytes) -> bytes:
    rc = kmer[::-1].translate(bytes.maketrans(b"ACGT", b"TGCA"))
    return min(kmer, rc)


def carries(kmer: bytes) -> bool:
    """h1 = A + B and h2 = h1 + B (A, B: the fmix64 outputs): does the low-word add of A + B carry?"""
    h1, h2 = orc.murmur(kmer, 42)
    b = (h2 - h1) & M64
    a = (h1 - b) & M64
    return (a & 0xFFFFFFFF) + (b & 0xFFFFFFFF) > 0xFFFFFFFF


ACGT = np.frombuffer(b"ACGT", np.uint8)


@pytest.fixture(scope="module")
def gate_case():
    rng = np.random.default_rng(2121)
    # 1000-hash sketches of 125 kbp genomes keep their largest keys near 0.8 % of the range: above the
    # mixture cap of a 20 Mbp launch, below the 1 % from which the build adds a Bloom tier
    genomes = [synth.random_genome(rng, 125_000) for _ in range(12)]
    contigs = synth.cut_contigs(rng, genomes[:6], 20_000_000, 0.01, median=4000.0, lo=500)
    fasta = synth.to_fasta(contigs, "c")
    seqs = [ACGT[c].tobytes() for c in contigs]
    return genomes, seqs, fasta, {}


def query_hashes(seqs, k, cache):
    """(hash, k-mer) of every valid query k-mer position, in stream order."""
    if k not in cache:
        hs_, pos = [], []
        for i, seq in enumerate(seqs):
            h, v = orc.hash_sequence(seq, k)
            keep = np.flatnonzero(v.astype(bool))
            hs_.append(h[keep]); pos.append(np.stack([np.full(len(keep), i), keep], 1))
        cache[k] = (np.concatenate(hs_), np.concatenate(pos))
    return cache[k]


def place_key(k, genomes, seqs, cache, want_carry):
    """Sketches of the genomes plus one extra reference whose largest key is the hash H of a query
    k-mer just above every other key, with the wanted carry."""
    sk = [orc.sketch_text(synth.to_fasta([g], "g"), k, S)[0] for g in genomes]
    top = max(int(h.max()) for h in sk)
    qh, qpos = query_hashes(seqs, k, cache)
    sel = np.flatnonzero((qh > np.uint64(top)) & (qh < np.uint64(top + (top >> 4))))
    for i in sel[np.argsort(qh[sel], kind="stable")]:
        H = int(qh[i]); r, p = (int(x) for x in qpos[i])
        canon = canonical(seqs[r][p:p + k])
        assert orc.murmur(canon, 42)[0] == H
        if carries(canon) == want_carry:
            below = sorted({int(x) for x in np.concatenate(sk)})[:: len(genomes)][: S - 1]
            return sk, H, below, qh
    raise AssertionError("no query k-mer with the wanted carry above the sketches")


@pytest.mark.parametrize("k", [21, 31])
@pytest.mark.parametrize("want_carry", [True, False])
def test_max_key_on_a_query_hash(gate_case, k, want_carry):
    genomes, seqs, fasta, cache = gate_case
    sk, H, below, qh = place_key(k, genomes, seqs, cache, want_carry)
    seq2, inv, n_pos, _ = hs.pack_text(fasta)
    assert n_pos <= 32 << 20                     # one piece of a packed feed: one stream launch
    for delta in (0, 1):
        extra = np.array(below + [H - delta], np.uint64)
        refs = sk + [extra]
        offsets = np.concatenate([[0], np.cumsum([len(h) for h in refs])]).astype(np.uint64)
        hashes = np.concatenate(refs)
        lengths = np.array([len(g) for g in genomes] + [125_000], np.uint64)
        db = hs.Database.from_arrays(k, S, 42, offsets, hashes, lengths)
        assert db.info.max_key == H - delta
        assert db.info.bloom_bytes == 0          # the plain range gate, not the Bloom tier
        want = orc.OracleDB.from_arrays(k, S, 42, offsets, hashes, lengths).screen_text(fasta, threads=4)
        out = {}
        for name, probe_filter in (("gate", True), ("probe_all", False)):
            scr = hs.Screen(db, probe_filter=probe_filter)
            scr.feed_packed(seq2, inv, n_pos)
            out[name] = scr.finish(False)
            scr.close()
            assert out[name].shared.tolist() == want.shared.tolist(), (name, delta)
            assert out[name].median.tolist() == want.median.tolist(), (name, delta)
            assert out[name].set_size == want.set_size
        # The launch offered the mixture every k-mer at or below its threshold.  Fewer offers than k-mers at
        # or below max_key mean the threshold was below max_key: the kernel's gate was max_key itself.
        assert out["gate"].stats["n_mix_inserts"] < int(np.count_nonzero(qh <= np.uint64(H - delta)))
        assert out["gate"].stats["n_valid_kmers"] == len(qh)
        assert out["gate"].stats["n_hits"] == out["probe_all"].stats["n_hits"]
        assert out["gate"].stats["n_probes"] < out["probe_all"].stats["n_probes"]
        assert int(out["gate"].shared[-1]) >= 1   # the extra reference shares hashes with the query
