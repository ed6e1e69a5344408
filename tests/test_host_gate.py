"""The stream kernel's range gate on the hash's high word, emulated on the CPU.

k_stream (screen, 64-bit hashes) decides `h <= gate` from s = fmix64_hi(x) + fmix64_hi(y), the high
words of the two finalizer outputs, and finishes the hash only for the k-mers that pass
(kmer_core.cuh: murmur_finish_hi_floor, hi_gate_may_pass).  The true high word of h is s or s + 1;
these tests check that the test built on that bound never turns away a k-mer with h <= gate, and that
every k-mer it lets through beyond a plain high-word compare is one the carry bound allows.
"""
import ctypes as C
import os
import random
import subprocess

import numpy as np
import pytest

from tests import _oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
M64 = (1 << 64) - 1
N_KMERS = 10_000_000


@pytest.fixture(scope="module")
def gate_lib():
    out = os.path.join(ROOT, "tests", "host_emul", "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libgateemul.so")
    src = os.path.join(ROOT, "tests", "host_emul", "gate_emul.cpp")
    deps = [src, os.path.join(ROOT, "hymet_b200", "csrc", "kmer_core.cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(so) < os.path.getmtime(d) for d in deps):
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so, src], check=True)
    L = C.CDLL(so)
    u64p = C.POINTER(C.c_uint64)
    L.gate_scan.argtypes = [C.c_int, C.c_uint32, C.c_uint64, C.c_uint64, u64p, C.c_int, u64p, u64p]
    L.gate_scan.restype = None
    L.find_hashes.argtypes = [C.c_int, C.c_uint32, C.c_uint64, C.c_int, u64p, C.c_uint64]
    L.find_hashes.restype = C.c_uint64
    L.state_for.argtypes = [C.c_uint64, C.c_uint64, u64p]
    L.state_for.restype = None
    L.emul_finish.argtypes = [C.c_uint64, C.c_uint64]; L.emul_finish.restype = C.c_uint64
    L.emul_finish_hi_floor.argtypes = [C.c_uint64, C.c_uint64]; L.emul_finish_hi_floor.restype = C.c_uint32
    L.emul_hi_gate_may_pass.argtypes = [C.c_uint32, C.c_uint64]; L.emul_hi_gate_may_pass.restype = C.c_int
    return L


def _ptr(a):
    return a.ctypes.data_as(C.POINTER(C.c_uint64))


def find_hashes(L, k, rng_seed, carry, n):
    out = np.zeros(n, np.uint64)
    got = L.find_hashes(k, 42, rng_seed, int(carry), _ptr(out), n)
    assert got == n
    return [int(x) for x in out]


@pytest.mark.parametrize("k", [21, 31])
def test_high_word_gate_has_no_false_negatives(gate_lib, k):
    rng = random.Random(k)
    # the first k-mers of the scan's own stream whose low-word add carries, and two whose add does not
    carried = find_hashes(gate_lib, k, 77 + k, True, 4)
    plain = find_hashes(gate_lib, k, 77 + k, False, 2)
    gates = [0, 0xFFFFFFFF,                                  # gate_hi = 0
             0xFFFFFFFE_FFFFFFFF, 0xFFFFFFFE_00000000,         # gate_hi = 0xFFFFFFFE: the largest the bound covers
             M64,                                              # gate_hi = 0xFFFFFFFF: everything passes
             (1 << 64) // 1400, (1 << 62) - 1]                 # about the screen's pass rate; the largest MODE 0 key
    gates += [rng.getrandbits(64) for _ in range(4)] + [rng.getrandbits(rng.randrange(33, 64)) for _ in range(4)]
    # gates exactly at (and one below) hashes whose low-word add carries, and at hashes where it does not
    gates += carried + [h - 1 for h in carried] + plain + [h - 1 for h in plain]
    g = np.array(gates, np.uint64)
    out = np.zeros(5 * len(g), np.uint64)
    n_carry = np.zeros(1, np.uint64)
    gate_lib.gate_scan(k, 42, N_KMERS, 77 + k, _ptr(g), len(g), _ptr(out), _ptr(n_carry))
    out = out.reshape(-1, 5)
    # about half of all finalizer low-word adds carry: the bound is exercised, not skirted
    assert 0.45 * N_KMERS < int(n_carry[0]) < 0.55 * N_KMERS
    for gate, (n_exact, n_pass, n_fn, n_fp_bound, n_unexplained) in zip(gates, out.tolist()):
        assert n_fn == 0, hex(gate)
        assert n_pass >= n_exact
        assert n_unexplained == 0, hex(gate)
        # the bound's own false positives need s on one of two values out of 2^32
        assert n_fp_bound <= 8, (hex(gate), n_fp_bound)
        if gate == M64:
            assert n_pass == n_exact == N_KMERS
    for h in carried + plain:     # the k-mer the gate sits on is inside it
        assert int(out[gates.index(h)][0]) >= 1


def test_high_word_gate_at_the_wrap(gate_lib):
    """Finalizer outputs placed by hand: s = 0xFFFFFFFF whose carry wraps the high word to 0, the same s
    without a carry, a carry into gate_hi + 1, and random words against gates at and around the hash."""
    xy = (C.c_uint64 * 2)()
    rng = random.Random(3)
    cases = [(0xFFFFFFFF_80000000, 0x00000000_80000000), (0xFFFFFFFF_00000000, 0),
             (0x12345678_FFFFFFFF, 0x00000000_00000001), (0x7FFFFFFF_FFFFFFFF, 0x80000000_00000000)]
    cases += [(rng.getrandbits(64), rng.getrandbits(64)) for _ in range(2000)]
    for a, b in cases:
        gate_lib.state_for(a, b, xy)
        h = gate_lib.emul_finish(xy[0], xy[1])
        assert h == (a + b) & M64
        s = gate_lib.emul_finish_hi_floor(xy[0], xy[1])
        assert s == ((a >> 32) + (b >> 32)) & 0xFFFFFFFF
        assert (h >> 32) in (s, (s + 1) & 0xFFFFFFFF)
        for gate in (h, h - 1 if h else 0, h + 1, h | 0xFFFFFFFF, h & ~0xFFFFFFFF, 0, 0xFFFFFFFE_FFFFFFFF, M64):
            gate &= M64
            if h <= gate:
                assert gate_lib.emul_hi_gate_may_pass(s, gate), (hex(a), hex(b), hex(gate))


@pytest.mark.parametrize("k", [21, 31])
def test_finalizer_state_matches_murmur(gate_lib, k):
    """MurmurHash3_x64_128 ends with h1 = A + B and h2 = h1 + B (A, B: the two fmix64 outputs), so the
    oracle's (h1, h2) give back A and B: the state built from them finishes to the oracle's h1, about
    half of them carry, and the high-word test lets h1 through a gate at h1."""
    rng = random.Random(k)
    xy = (C.c_uint64 * 2)()
    carries = set()
    for _ in range(400):
        kmer = bytes(rng.choice(b"ACGT") for _ in range(k))
        h1, h2 = orc.murmur(kmer, 42)
        b = (h2 - h1) & M64
        a = (h1 - b) & M64
        carries.add(((a & 0xFFFFFFFF) + (b & 0xFFFFFFFF)) >> 32)
        gate_lib.state_for(a, b, xy)
        assert gate_lib.emul_finish(xy[0], xy[1]) == h1
        assert gate_lib.emul_hi_gate_may_pass(gate_lib.emul_finish_hi_floor(xy[0], xy[1]), h1)
    assert carries == {0, 1}
