"""Shared-memory bank model of the stream kernel's table reads.

k_stream hashes every k-mer with 64-bit reads of two premultiplied tables (full words), 32-bit reads of
their low words and, at k = 21, one 64-bit read of the tail-term table.  Each read starts a dependency
chain, so a bank conflict is exposed latency.  These tests take the lane addresses from the header
functions the kernel uses (kmer_core.cuh: SmemLayout, through tests/host_emul/bank_emul.cpp) and count
wavefronts with 32 banks of 4 bytes:
  - a 64-bit read is served per half-warp; a half-warp costs as many wavefronts as the most distinct
    8-byte words that fall on one bank pair;
  - a 32-bit read costs as many wavefronts as the most distinct 4-byte words that fall on one bank.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LUT = 0x8000          # a table window at a 32 KB boundary, as the kernel aligns it
TRIALS = 4000


@pytest.fixture(scope="module")
def lib():
    out = os.path.join(ROOT, "tests", "host_emul", "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libbankemul.so")
    src = os.path.join(ROOT, "tests", "host_emul", "bank_emul.cpp")
    deps = [src, os.path.join(ROOT, "hymet_b200", "csrc", "kmer_core.cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(so) < os.path.getmtime(d) for d in deps):
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so, src], check=True)
    L = C.CDLL(so)
    L.lane_addrs.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_uint64), C.c_int, C.c_uint32, C.POINTER(C.c_uint32)]
    L.lane_addrs.restype = C.c_int
    L.table_bytes.argtypes = [C.c_int]; L.table_bytes.restype = C.c_uint32
    L.word_index.argtypes = [C.c_uint64, C.c_int, C.c_int]; L.word_index.restype = C.c_uint32
    return L


def lane_addrs(L, copies, k, ct, word):
    ct = np.ascontiguousarray(ct, np.uint64)
    out = np.zeros(32, np.uint32)
    assert L.lane_addrs(copies, k, ct.ctypes.data_as(C.POINTER(C.c_uint64)), word, LUT,
                        out.ctypes.data_as(C.POINTER(C.c_uint32))) == 0
    return [int(a) for a in out]


def half_wavefronts64(half):
    per_pair = {}
    for a in set(a >> 3 for a in half):
        per_pair.setdefault(a % 16, set()).add(a)
    return max(len(v) for v in per_pair.values())


def wavefronts64(addrs):
    return half_wavefronts64(addrs[:16]) + half_wavefronts64(addrs[16:])


def wavefronts32(addrs):
    per_bank = {}
    for a in set(a >> 2 for a in addrs):
        per_bank.setdefault(a % 32, set()).add(a)
    return max(len(v) for v in per_bank.values())


def reads(k):
    """(word, 64-bit?) of every premultiplied-table read of one k-mer (kmer_core.cuh: murmur_state_premul)"""
    tail_lane = 2 * (k >> 4) if 1 <= (k & 15) <= 5 else -1
    out = []
    for lane in range(4):
        nb = k - 8 * lane
        if nb > 0 and lane != tail_lane:
            out.append((2 * lane, True))
            if nb > 4:
                out.append((2 * lane + 1, False))
    return out


def kmers(rng):
    return rng.integers(0, 2**64, size=32, dtype=np.uint64)


@pytest.mark.parametrize("k", [21, 31])
def test_addresses_select_the_right_entry(lib, k):
    rng = np.random.default_rng(k)
    tb = lib.table_bytes(16)
    for _ in range(200):
        ct = kmers(rng)
        for word, _wide in reads(k):
            addrs = lane_addrs(lib, 16, k, ct, word)
            for lane, a in enumerate(addrs):
                assert a % 8 == 0 and LUT <= a < LUT + tb
                assert (a - LUT) % 128 == 8 * (lane % 16)
                assert (a - LUT) // 128 == lib.word_index(int(ct[lane]), word, k)


@pytest.mark.parametrize("k", [21, 31])
def test_premultiplied_reads_are_conflict_free(lib, k):
    rng = np.random.default_rng(100 + k)
    for _ in range(TRIALS):
        ct = kmers(rng)
        for word, wide in reads(k):
            addrs = lane_addrs(lib, 16, k, ct, word)
            if wide:
                for half in (addrs[:16], addrs[16:]):   # every lane of a half-warp on its own bank pair
                    assert len({(a >> 3) % 16 for a in half}) == 16
                assert wavefronts64(addrs) == 2
            else:
                assert wavefronts32(addrs) <= 2


def test_eight_copies_conflict(lib):
    """The model tells the layouts apart: 8 lane copies (two lanes of a half-warp per copy) conflict."""
    rng = np.random.default_rng(7)
    w64 = w32 = 0
    for _ in range(TRIALS):
        ct = kmers(rng)
        w64 += wavefronts64(lane_addrs(lib, 8, 21, ct, 0))
        w32 += wavefronts32(lane_addrs(lib, 8, 21, ct, 1))
    assert w64 / TRIALS > 3.5 and w32 / TRIALS > 3.0


def test_tail_reads(lib):
    """k = 21: two interleaved tail-table copies on disjoint bank pairs.  A half-warp's 16 lanes split
    8 + 8 over the two copies, so a read takes at most 8 wavefronts per half-warp (one copy: 16), and
    fewer than with one copy on average."""
    rng = np.random.default_rng(21)
    tb = lib.table_bytes(16)
    w2 = w1 = 0
    for _ in range(TRIALS):
        ct = kmers(rng)
        addrs = lane_addrs(lib, 16, 21, ct, -1)
        for lane, a in enumerate(addrs):
            entry = (int(ct[lane]) & 0xFFFFFFFF) >> 22   # the 5 tail letters: top 10 bits of the low half
            assert a == LUT + 2 * tb + 16 * entry + 8 * (lane & 1)
        for half in (addrs[:16], addrs[16:]):
            pairs = [{(a >> 3) % 16 for a in half[c::2]} for c in (0, 1)]
            assert not pairs[0] & pairs[1]
            assert half_wavefronts64(half) <= 8
        w2 += wavefronts64(addrs)
        w1 += wavefronts64(lane_addrs(lib, 8, 21, ct, -1))
    assert w2 < w1
