"""C-ABI surface on a box without a GPU: the library loads, exports every symbol the
header declares, refuses to run without a B200 (no CPU fallback), and its host-only
entry points (FASTA packer, .msh parser) work."""
import ctypes as C
import os
import sys
import re

import numpy as np
import pytest

from hymet_b200 import _abi
from hymet_b200 import msh as mshfmt
from hymet_b200 import screen as hs
from hymet_b200 import synth
from tests import _oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    text = open(os.path.join(ROOT, "include", "hymet_screen.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(hs_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = _abi.load()
    syms = header_symbols()
    assert len(syms) >= 35
    for s in syms:
        assert hasattr(lib, s), "libhymet_screen.so lacks " + s
        assert s in _abi.SIGNATURES, "ctypes table lacks " + s
    assert sorted(_abi.SIGNATURES) == syms
    assert b"sm_100a" in lib.hs_version()


def test_no_gpu_means_error_not_fallback():
    """Run in a child process that sees no device (CUDA_VISIBLE_DEVICES empty), so that the check also
    holds on a box with a B200."""
    import subprocess
    code = r'''
import ctypes as C, sys
sys.path.insert(0, %r)
import numpy as np
import pytest
from hymet_b200 import _abi
from hymet_b200 import screen as hs
lib = _abi.load()
assert lib.hs_init(0) == -2  # HS_ENODEV
assert b"no CPU fallback" in lib.hs_last_error()
h = C.c_void_p()
off = np.array([0, 1], np.uint64); hh = np.array([5], np.uint64)
rc = lib.hs_db_from_arrays(21, 1000, 42, 1, off.ctypes.data_as(_abi.u64p), hh.ctypes.data_as(_abi.u64p), None,
                           C.byref(h))
assert rc == -2 and not h.value
with pytest.raises(_abi.HsError):
    hs.hash_packed(21, 42, np.zeros(256, np.uint64), np.zeros(256, np.uint32), 100)
with pytest.raises(_abi.HsError):
    hs.Database.from_arrays(21, 1000, 42, off, hh)
print("ok")
''' % ROOT
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0 and r.stdout.strip() == "ok", (r.returncode, r.stdout, r.stderr[-2000:])


def test_host_packer_layout():
    text = b">r1 x\nACGTN\nacgt\n>r2\n\nTT\n"
    seq, inv, n, st = hs.pack_text(text)
    # positions: sep A C G T N a c g t sep T T
    assert n == 13 and st["n_records"] == 2 and st["n_bases"] == 11
    codes = [(int(seq[0]) >> (62 - 2 * j)) & 3 for j in range(13)]
    bad = [(int(inv[0]) >> (31 - j)) & 1 for j in range(32)]
    assert codes[1:5] == [0, 1, 2, 3] and codes[6:10] == [0, 1, 2, 3] and codes[11:13] == [3, 3]
    assert bad[:13] == [1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0] and all(bad[13:])
    assert hs.packed_words(1) == 256 and hs.packed_words(8192) == 256 and hs.packed_words(8193) == 512
    # invalid positions carry code 0 whatever the byte was (vector and scalar paths agree bit for bit)
    line = (b"ACGT\rN-*xyz" * 30)[:300]
    seq, inv, n, _ = hs.pack_text(b">v\n" + line + b"\n")
    for pos, ch in enumerate(b"!" + line):
        code = (int(seq[pos // 32]) >> (62 - 2 * (pos % 32))) & 3
        bad = (int(inv[pos // 32]) >> (31 - pos % 32)) & 1
        want = b"ACGT".find(bytes([ch]).upper())
        assert (code, bad) == ((want, 0) if want >= 0 else (0, 1)), (pos, ch)


def _toy_db(rng, n=7, s=50, k=21, bits=64):
    hs_list = [np.unique(rng.integers(0, 2 ** bits - 1, size=s, dtype=np.uint64)) for _ in range(n)]
    hs_list[2] = np.zeros(0, np.uint64)   # a reference without hashes
    offsets = np.concatenate([[0], np.cumsum([len(h) for h in hs_list])]).astype(np.uint64)
    return mshfmt.SketchDB(k=k, s=s, names=[synth.gcf_name(i) for i in range(n)],
                           comments=["[3 seqs] NZ_%d some plasmid [...]" % i if i % 2 else "" for i in range(n)],
                           lengths=np.array([10 ** 6 + i for i in range(n - 1)] + [2 ** 33 + 5], np.uint64),
                           offsets=offsets, hashes=np.concatenate(hs_list))


@pytest.mark.parametrize("variant", ["single", "multi", "double_far", "old_list", "no_alphabet", "k16"])
def test_msh_three_readers_agree(tmp_path, variant):
    rng = np.random.default_rng(3)
    db = _toy_db(rng, k=16 if variant == "k16" else 21, bits=32 if variant == "k16" else 64)
    kw = {}
    if variant == "multi":
        kw = dict(seg_cap_words=64)
    elif variant == "double_far":
        kw = dict(seg_cap_words=128, double_far_refs=[0, 4])
    elif variant == "old_list":
        kw = dict(use_old_list=True)
    elif variant == "no_alphabet":
        kw = dict(write_alphabet=False)
    p = str(tmp_path / "t.msh")
    mshfmt.write_msh(p, db, **kw)
    if variant in ("multi", "double_far"):
        import struct
        assert struct.unpack("<I", open(p, "rb").read(4))[0] + 1 > 3   # really multi-segment
    py = mshfmt.read_msh(p)                 # NumPy reader
    cc = hs.read_msh_host(p)                # product C++ reader (host only)
    oc = orc.OracleDB.load_msh(p)           # oracle C reader
    assert py._root_shape == (3, 4)
    for got in (py.__dict__, cc):
        assert got["k"] == db.k and got["s"] == db.s and got["seed"] == 42
        assert list(got["names"]) == db.names and list(got["comments"]) == db.comments
        assert np.array_equal(got["lengths"], db.lengths)
        assert np.array_equal(got["offsets"], db.offsets)
        assert np.array_equal(got["hashes"], db.hashes)
    assert (oc.k, oc.s, oc.seed, oc.n_refs) == (db.k, db.s, 42, db.n_refs)
    for i in range(db.n_refs):
        assert oc.name(i) == db.names[i] and oc.comment(i) == db.comments[i]
        assert oc.length(i) == int(db.lengths[i])
        assert np.array_equal(oc.hashes(i), db.ref_hashes(i))


def test_msh_rejects_what_it_cannot_screen(tmp_path):
    rng = np.random.default_rng(4)
    lib = _abi.load()
    for kw, code in ((dict(noncanonical=True), -7), (dict(preserve_case=True), -7), (dict(alphabet="ACDEFGHIKLMNPQRSTVWY"), -7)):
        db = _toy_db(rng)
        for a, v in kw.items():
            setattr(db, a, v)
        p = str(tmp_path / "bad.msh")
        mshfmt.write_msh(p, db)
        h = C.c_void_p()
        assert lib.hs_msh_open(p.encode(), C.byref(h)) == code
    p = str(tmp_path / "trunc.msh")
    good = str(tmp_path / "good.msh")
    mshfmt.write_msh(good, _toy_db(rng))
    open(p, "wb").write(open(good, "rb").read()[:200])
    h = C.c_void_p()
    assert lib.hs_msh_open(p.encode(), C.byref(h)) == -5
    assert lib.hs_msh_open(str(tmp_path / "missing.msh").encode(), C.byref(h)) == -4
    open(p, "wb").write(b"\x00" * 4096)   # all-zero file: null root
    assert lib.hs_msh_open(p.encode(), C.byref(h)) == -5


def test_header_is_plain_c_and_links_from_a_c_program(tmp_path):
    """The boundary is a C ABI: include/hymet_screen.h must compile as C99 (no C++ types) and a C
    program must link against libhymet_screen.so and call it (host-only entry points here)."""
    import subprocess
    from hymet_b200 import build as b
    lib = b.build()
    src = tmp_path / "abi_demo.c"
    src.write_text(r'''
#include <stdio.h>
#include <string.h>
#include "hymet_screen.h"
int main(void) {
    hs_db_info_t info; hs_stats_t st; uint64_t seq[16]; uint32_t inv[16]; uint64_t n = 0;
    const char *fa = ">r\nACGTNACGT\n";
    memset(&info, 0, sizeof info);
    if (!hs_version() || !hs_last_error()) return 2;
    if (hs_packed_words(1) < 1) return 3;
    if (hs_pack_text(fa, strlen(fa), seq, inv, 16, &n, &st) != 0) return 4;
    if (n != 10 || st.n_records != 1) return 5;            /* separator + 9 bases */
    if (hs_init(0) == 0) return 0;                          /* a B200 is present: fine */
    printf("%s\n", hs_last_error());
    return hs_db_load_msh("nonexistent.msh", (hs_db **)&info) == 0 ? 6 : 0;   /* no device: an error, never a result */
}
''')
    exe = tmp_path / "abi_demo"
    inc = os.path.join(ROOT, "include")
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-I", inc, str(src), "-o", str(exe),
                        "-L", os.path.dirname(lib), "-l:libhymet_screen.so", "-Wl,-rpath," + os.path.dirname(lib)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)


def test_msh_reader_survives_corrupted_files(tmp_path, golden_dir):
    """.msh files come from outside: truncated or bit-flipped input must end in an error code (or a
    clean parse), never in a crash or an out-of-bounds read.  Run in a child process so that a crash
    would be seen as a non-zero exit status."""
    import subprocess
    script = tmp_path / "fuzz.py"
    script.write_text(r'''
import ctypes as C, os, random, sys
sys.path.insert(0, %r)
from hymet_b200 import _abi
L = _abi.load()
data = bytearray(open(%r, "rb").read())
rng = random.Random(7)
out = os.path.join(%r, "m.msh")
ok = bad = 0
for t in range(400):
    d = bytearray(data)
    kind = t %% 4
    if kind == 0:
        d = d[:rng.randrange(0, len(d))]                                   # truncation
    elif kind == 1:
        for _ in range(rng.randrange(1, 8)):
            d[rng.randrange(0, min(len(d), 4096))] = rng.randrange(256)    # header / pointer area
    elif kind == 2:
        for _ in range(rng.randrange(1, 64)):
            d[rng.randrange(0, len(d))] ^= 1 << rng.randrange(8)           # anywhere
    else:
        p = rng.randrange(0, len(d) - 8) & ~7                              # a whole word: far pointers, list sizes
        d[p:p + 8] = rng.getrandbits(64).to_bytes(8, "little")
    open(out, "wb").write(d)
    m = C.c_void_p()
    rc = L.hs_msh_open(out.encode(), C.byref(m))
    if rc == 0:
        info = _abi.DbInfo()
        L.hs_msh_info(m, C.byref(info))
        L.hs_msh_free(m)
        ok += 1
    else:
        assert L.hs_last_error(), "error code without a message"
        bad += 1
print(ok, bad)
''' % (ROOT, os.path.join(golden_dir, "zymo25.msh"), str(tmp_path)))
    r = subprocess.run([sys.executable, str(script)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, (r.returncode, r.stderr[-2000:])
    ok, bad = map(int, r.stdout.split())
    assert ok + bad == 400 and bad > 100


def test_host_parsers_under_address_sanitizer(tmp_path, golden_dir):
    """The .msh reader on 600 corrupted copies of a real sketch file and the FASTA packer / splitter on
    10 000 random texts, compiled with -fsanitize=address,undefined (tests/host_emul/fuzz_asan.cpp)."""
    import random
    import subprocess
    exe = str(tmp_path / "fuzz_asan")
    csrc = os.path.join(ROOT, "hymet_b200", "csrc")
    r = subprocess.run(["g++", "-O1", "-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined", "-std=c++17",
                        os.path.join(ROOT, "tests", "host_emul", "fuzz_asan.cpp"), os.path.join(csrc, "msh_capnp.cpp"),
                        os.path.join(csrc, "fasta_pack.cpp"), "-lz", "-o", exe], capture_output=True, text=True)
    if r.returncode != 0 and "asan" in r.stderr.lower():
        pytest.skip("no sanitizer runtime in this image")
    assert r.returncode == 0, r.stderr[-2000:]
    data = bytearray(open(os.path.join(golden_dir, "zymo25.msh"), "rb").read())
    rng = random.Random(11)
    files = []
    for t in range(600):
        d = bytearray(data)
        kind = t % 5
        if kind == 0:
            d = d[:rng.randrange(0, len(d))]
        elif kind == 1:
            for _ in range(rng.randrange(1, 8)):
                d[rng.randrange(0, min(len(d), 4096))] = rng.randrange(256)
        elif kind == 2:
            for _ in range(rng.randrange(1, 64)):
                d[rng.randrange(0, len(d))] ^= 1 << rng.randrange(8)
        elif kind == 3:
            p = rng.randrange(0, len(d) - 8) & ~7
            d[p:p + 8] = rng.getrandbits(64).to_bytes(8, "little")
        else:
            p = rng.randrange(0, min(len(d) - 8, 2048)) & ~7
            d[p:p + 8] = rng.choice([0, 2 ** 64 - 1, 2 ** 63, 2 ** 32, 2 ** 31, 1, 2, 3, 4]).to_bytes(8, "little")
        f = str(tmp_path / ("m%d.msh" % t))
        open(f, "wb").write(d)
        files.append(f)
    env = dict(os.environ, ASAN_OPTIONS="detect_leaks=0")
    r = subprocess.run([exe, "msh"] + files, capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    ok, bad = map(int, r.stdout.split())
    assert ok + bad == 600 and bad > 100
    r = subprocess.run([exe, "pack", "10000"], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0 and r.stdout.startswith("ok "), (r.stdout, r.stderr[-3000:])
