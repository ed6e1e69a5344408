// The stream kernel's range gate on the hash's high word (kmer_core.cuh: murmur_finish_hi_floor,
// hi_gate_may_pass), run on the CPU over random canonical k-mers cut from random windows the way one
// CUDA thread cuts them (win_init_top + canonical_top, pre-multiplied tables, tail-term table).
// Built with g++ by tests/test_host_gate.py.
#include <stdint.h>

#include "../../hymet_b200/csrc/kmer_core.cuh"

namespace {

uint64_t splitmix(uint64_t &s)
{
    uint64_t z = (s += 0x9E3779B97F4A7C15ull);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

uint64_t inverse_odd(uint64_t c)  // c * inverse_odd(c) == 1 (mod 2^64)
{
    uint64_t x = c;
    for (int i = 0; i < 6; i++) x *= 2 - c * x;
    return x;
}

}  // namespace

extern "C" {

// For n random k-mers and every gate g[0..n_gates): out[5*i + ...] =
//   0: k-mers with h <= gate              1: k-mers the high-word test lets through
//   2: false negatives (h <= gate, turned away)
//   3: false positives whose high word is above gate_hi (the carry bound's own)
//   4: false positives the carry bound does not explain (neither s == gate_hi carrying into gate_hi + 1
//      nor s == 0xFFFFFFFF without a carry)
// and carry[0]: k-mers whose finalizer low-word add carried.
void gate_scan(int k, uint32_t seed, uint64_t n, uint64_t rng, const uint64_t *gates, int n_gates, uint64_t *out,
               uint64_t *carry)
{
    const hs::PremulArithMsb pre{};
    for (int i = 0; i < 5 * n_gates; i++) out[i] = 0;
    carry[0] = 0;
    uint32_t bound[64];
    for (int g = 0; g < n_gates && g < 64; g++) bound[g] = hs::hi_gate_bound(gates[g]);
    for (uint64_t t = 0; t < n; t++) {
        const uint64_t prev = splitmix(rng), cur = splitmix(rng);
        const hs::Win w = hs::win_init_top(prev, cur, k);
        const uint64_t ct = hs::canonical_top(w, (int)(t & 31));
        const hs::MurmurState st = hs::murmur_state_premul_top(ct, k, seed, pre);
        const uint64_t h = hs::hash_canonical_premul_top(ct, k, seed, true, pre);
        const uint32_t s = hs::murmur_finish_hi_floor(st), hh = (uint32_t)(h >> 32);
        carry[0] += hh != s;
        for (int g = 0; g < n_gates && g < 64; g++) {
            const uint32_t gate_hi = (uint32_t)(gates[g] >> 32);
            const bool exact = h <= gates[g], pass = hs::hi_gate_may_pass(s, bound[g]);
            uint64_t *o = out + 5 * g;
            o[0] += exact;
            o[1] += pass;
            o[2] += exact && !pass;
            if (pass && !exact && hh > gate_hi) {
                o[3]++;
                const bool explained = (s == gate_hi && hh == gate_hi + 1u) || (s == 0xFFFFFFFFu && hh == 0xFFFFFFFFu);
                o[4] += !explained;
            }
        }
    }
}

// Up to cap hashes of random k-mers whose finalizer low-word add carries (want_carry) or does not.
uint64_t find_hashes(int k, uint32_t seed, uint64_t rng, int want_carry, uint64_t *out, uint64_t cap)
{
    const hs::PremulArithMsb pre{};
    uint64_t n = 0;
    for (uint64_t t = 0; n < cap && t < (cap << 8); t++) {
        const uint64_t prev = splitmix(rng), cur = splitmix(rng);
        const hs::Win w = hs::win_init_top(prev, cur, k);
        const uint64_t ct = hs::canonical_top(w, (int)(t & 31));
        const uint64_t h = hs::hash_canonical_premul_top(ct, k, seed, true, pre);
        const bool carried = (uint32_t)(h >> 32) != hs::murmur_finish_hi_floor(hs::murmur_state_premul_top(ct, k, seed, pre));
        if (carried == (want_carry != 0)) out[n++] = h;
    }
    return n;
}

// The finalizer state whose two fmix64 outputs are a and b (fmix64 is a bijection), so that a test can
// place the two words anywhere, e.g. s = 0xFFFFFFFF with and without the carry.
void state_for(uint64_t a, uint64_t b, uint64_t *xy)
{
    const uint64_t i1 = inverse_odd(0xff51afd7ed558ccdull), i2 = inverse_odd(0xc4ceb9fe1a85ec53ull);
    const uint64_t v[2] = {a, b};
    for (int i = 0; i < 2; i++) {
        uint64_t x = v[i];
        x ^= x >> 33; x *= i2;   // x ^ (x >> 33) is its own inverse
        x ^= x >> 33; x *= i1;
        x ^= x >> 33;
        xy[i] = x;
    }
}

uint64_t emul_finish(uint64_t x, uint64_t y) { return hs::murmur_finish(hs::MurmurState{x, y}); }
uint32_t emul_finish_hi_floor(uint64_t x, uint64_t y) { return hs::murmur_finish_hi_floor(hs::MurmurState{x, y}); }
int emul_hi_gate_may_pass(uint32_t s, uint64_t gate) { return hs::hi_gate_may_pass(s, hs::hi_gate_bound(gate)); }

}
