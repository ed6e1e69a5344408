"""Every handle and single-stage call gives back every CUDA resource it took.

A child process runs with an LD_PRELOAD interposer (tests/host_emul/cuda_count.cpp) that counts live
device buffers, pinned buffers, events and streams and forwards each call unchanged to the CUDA runtime
(libhymet_screen.so links it shared).  The child drives databases, screens on every feed path, the
reductions, the in-process exchange, the sketcher, the single stages and a refused call, frees each,
and checks after every free that the four counts are back where they were before the first handle.
The child does not import torch, whose caching allocator would hold memory of its own.
"""
import ctypes as C
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KINDS = ("device buffers", "pinned buffers", "events", "streams")


@pytest.mark.gpu
def test_every_free_returns_every_resource(tmp_path):
    so = str(tmp_path / "libcuda_count.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC",
                    "-I" + os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include"), "-o", so,
                    os.path.join(ROOT, "tests", "host_emul", "cuda_count.cpp"), "-ldl"], check=True)
    env = dict(os.environ, LD_PRELOAD=so, PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), so, str(tmp_path)], env=env, capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "lifecycle ok" in r.stdout


def _child(so, tmp):
    import gzip

    import numpy as np

    from hymet_b200 import _abi, _lite, msh as mshfmt, screen as hs, synth

    count = C.CDLL(so).cuda_count_live
    live = lambda: tuple(count(k) for k in range(4))  # noqa: E731
    _abi.init(0)
    rng = np.random.default_rng(7)
    k, s = 21, 1000
    genomes = [synth.random_genome(rng, 30_000) for _ in range(12)]
    fastas = [synth.to_fasta([g], "g") for g in genomes]
    base = live()

    def settled(what, want=None):
        want, now = want or base, live()
        bad = ["%s %d -> %d" % (KINDS[i], want[i], now[i]) for i in range(4) if now[i] != want[i]]
        assert not bad, "%s leaves resources behind: %s" % (what, ", ".join(bad))
        print("ok:", what, flush=True)

    sk = [hs.sketch_text(f, k, s)[0] for f in fastas]
    settled("sketch_text")
    paths = []
    for j, f in enumerate(fastas):
        paths.append(os.path.join(tmp, "g%d.fna" % j))
        open(paths[-1], "wb").write(f)
    with pytest.raises(hs.HsError) as ei:
        hs.sketch_files(paths[:2] + [os.path.join(tmp, "missing.fna")], k, s, threads=2)
    assert ei.value.code == -4   # HS_EIO
    settled("sketch_files with a missing path")
    got, _ = hs.sketch_files(paths, k, s, threads=2)
    assert [g.hashes.tolist() for g in got] == [h.tolist() for h in sk]
    settled("sketch_files")

    offsets = np.concatenate([[0], np.cumsum([len(h) for h in sk])]).astype(np.uint64)
    hashes = np.concatenate(sk)
    lengths = np.array([len(g) for g in genomes], np.uint64)
    msh = []
    for j in range(2):
        part = slice(6 * j, 6 * j + 6)
        o = np.concatenate([[0], np.cumsum([len(h) for h in sk[part]])]).astype(np.uint64)
        msh.append(os.path.join(tmp, "db%d.msh" % j))
        mshfmt.write_msh(msh[-1], mshfmt.SketchDB(k=k, s=s, names=[synth.gcf_name(6 * j + i) for i in range(6)],
                                                   comments=[""] * 6, lengths=lengths[part], offsets=o,
                                                   hashes=np.concatenate(sk[part])))
    query = synth.to_fasta(synth.cut_contigs(rng, genomes[:5], 200_000, 0.01, median=4000.0), "c")
    qpath = os.path.join(tmp, "q.fna")
    open(qpath, "wb").write(query)
    gzpath = qpath + ".gz"
    with gzip.open(gzpath, "wb") as fh:
        fh.write(query)

    for name, make in (("database from one .msh", lambda: hs.Database.load_msh(msh[0])),
                       ("database from several .msh", lambda: hs.Database.load_msh_multi(msh)),
                       ("database from arrays", lambda: hs.Database.from_arrays(k, s, 42, offsets, hashes, lengths))):
        db = make()
        assert db.probe(hashes[:100]).size == 100
        db.close()
        settled(name + " + probe")

    db = hs.Database.from_arrays(k, s, 42, offsets, hashes, lengths)
    with_db = live()   # what the screens below must come back to
    seq, inv, n_pos, _ = hs.pack_text(query)

    def screen(feed, finish, **opts):
        scr = hs.Screen(db)
        for key, v in opts.items():
            scr.set_option(key, v)
        feed(scr)
        res = finish(scr)
        scr.close()
        return res

    want = screen(lambda x: x.feed_text(query, 2), lambda x: x.finish().shared.tolist())
    settled("screen fed text, finish", with_db)
    feeds = (("file_mode 0", lambda x: x.feed_fasta(qpath, 2), {"file_mode": 0}),
             ("file_mode 1", lambda x: x.feed_fasta(qpath, 4), {"file_mode": 1}),
             ("a gzip file", lambda x: x.feed_fasta(gzpath, 2), {}),
             ("packed words", lambda x: x.feed_packed(seq, inv, n_pos), {}))
    for name, feed, opts in feeds:
        got = screen(feed, lambda x: x.finish().shared.tolist(), **opts)
        assert got == want, "%s: shared %s, fed as text %s" % (name, got, want)
        settled("screen fed " + name + ", finish", with_db)
    hits = screen(lambda x: x.feed_text(query, 2), lambda x: x.finish_hits())
    assert sorted(hits.ref.tolist()) == [i for i, v in enumerate(want) if v]
    settled("screen, finish_hits", with_db)
    screen(lambda x: x.feed_text(query, 2), lambda x: x.finish(wta=True), sparse=0)
    settled("screen on the dense path with -w", with_db)

    # a record of the screen's own mixture, merged back on the device
    cudart = C.CDLL("libcudart.so.12")   # already loaded by the library: its calls do not pass the interposer
    rec = C.c_void_p()
    assert cudart.cudaMalloc(C.byref(rec), C.c_size_t((s + 1) * 8)) == 0
    scr = hs.Screen(db)
    scr.feed_text(query, 2)
    scr.flush()
    scr.mixture_record(rec.value)
    scr.mixture_merge_device(rec.value, 1)
    assert scr.finish().shared.tolist() == want
    scr.close()
    assert cudart.cudaFree(rec) == 0
    settled("mixture_merge_device", with_db)

    scr = hs.Screen(db)
    scr.feed_text(query, 2)
    scr.flush()
    with pytest.raises(hs.HsError) as ei:
        scr.feed_text(query, 2)
    assert ei.value.code == -9   # HS_ESTATE
    scr.close()
    settled("a feed refused after flush", with_db)
    db.close()
    settled("database freed after its screens")

    ldb = _lite.LiteDb(msh[0], 0)
    size = os.path.getsize(qpath)
    scrs = [_lite.LiteScreen(ldb) for _ in range(2)]
    for i, x in enumerate(scrs):
        x.feed_fasta_range(qpath, size * i // 2, size * (i + 1) // 2, 2)
        x.flush()
    scrs[0].absorb([scrs[1]])
    assert "".join(scrs[0].finish_lines(False, 0.0, 1.0))
    for x in scrs:
        x.close()
    ldb.close()
    settled("absorb_screens of two screens on one GPU")

    h, v = hs.hash_packed(k, 42, seq, inv, n_pos)
    assert v.any()
    settled("hash_packed")
    dseq, dinv, dn, _ = hs.pack_text_device(query)
    assert dn == n_pos and np.array_equal(dseq, seq)
    settled("pack_text_device")
    ident, _ = hs.stat_batch(k, 10 ** 6, np.array([10, 20], np.uint64), np.array([s, s], np.uint64))
    assert ident.size == 2
    settled("stat_batch")
    assert "torch" not in sys.modules
    print("lifecycle ok", flush=True)


if __name__ == "__main__":
    sys.path.insert(0, ROOT)
    _child(sys.argv[1], sys.argv[2])
