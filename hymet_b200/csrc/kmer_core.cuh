// kmer_core.cuh -- arithmetic shared by every kernel on the screen hot path.
//
// Restates, for 2-bit packed sequence, what `mash screen` does per k-mer
// (the binary HYMET runs at /root/reference/scripts/mash.sh:14; rules S1-S5 of
// SURVEY.md Appendix A): canonical k-mer = min(fwd, revcomp) byte-wise,
// hash = MurmurHash3_x64_128(ASCII k-mer, seed)[h1], low 32 bits when 4^k <= 2^32.
//
// Everything here is `HS_HD` (host+device) on purpose: tests/ compiles this
// header with g++ and checks each function against the CPU oracle before any
// GPU time is spent.  The product only ever calls it from CUDA kernels.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define HS_HD __host__ __device__ __forceinline__
#define HS_HDC __host__ __device__ constexpr
#else
#define HS_HD inline
#define HS_HDC constexpr
#endif

namespace hs {

// ---- packed query layout --------------------------------------------------
// seq word w holds bases 32w..32w+31, base j at bits [62-2j, 63-2j] (first base
// most significant), codes A=0 C=1 G=2 T=3.  inv word w: bit (31-j) set when
// base j is not A/C/G/T (N, IUPAC, record separator, padding).
constexpr int kBasesPerWord = 32;

HS_HD uint64_t kmer_mask(int k) { return k >= 32 ? ~0ull : ((1ull << (2 * k)) - 1ull); }

// Reverse the order of the 32 two-bit groups of x.
HS_HD uint64_t pair_reverse64(uint64_t x)
{
#if defined(__CUDA_ARCH__)
    x = __brevll(x);
#else
    x = ((x >> 1) & 0x5555555555555555ull) | ((x & 0x5555555555555555ull) << 1);
    x = ((x >> 2) & 0x3333333333333333ull) | ((x & 0x3333333333333333ull) << 2);
    x = ((x >> 4) & 0x0F0F0F0F0F0F0F0Full) | ((x & 0x0F0F0F0F0F0F0F0Full) << 4);
    x = ((x >> 8) & 0x00FF00FF00FF00FFull) | ((x & 0x00FF00FF00FF00FFull) << 8);
    x = ((x >> 16) & 0x0000FFFF0000FFFFull) | ((x & 0x0000FFFF0000FFFFull) << 16);
    x = (x >> 32) | (x << 32);
#endif
    // full bit reversal also swapped the two bits inside every pair: swap back
    return ((x >> 1) & 0x5555555555555555ull) | ((x & 0x5555555555555555ull) << 1);
}

// For the 64 bases (prev word, cur word): bit (31-j) of the result is set when
// the k-mer ENDING at base j of the current word covers an invalid base.
HS_HD uint32_t invalid_kmer_ends(uint32_t inv_prev, uint32_t inv_cur, int k)
{
    uint64_t acc = ((uint64_t)inv_prev << 32) | inv_cur;
    int w = 1;
    while (2 * w <= k) { acc |= acc >> w; w *= 2; }  // bit p = OR of V[p .. p+w-1]
    if (w < k) acc |= acc >> (k - w);                // ... V[p .. p+k-1]
    return (uint32_t)acc;
}

// Rolling state of one thread: the k-mer ending at the most recent base.
//   fm  : forward k-mer, first base most significant, right aligned, masked
//   flp : forward k-mer, first base LEAST significant, LEFT aligned in 64 bits
//         (bits below 64-2k hold older bases and are ignored)
struct Roll { uint64_t fm, flp; };

HS_HD Roll roll_init(uint64_t prev_word, int k)
{
    Roll r;
    r.fm = prev_word & kmer_mask(k);     // k-mer ending at base 31 of the previous word
    r.flp = pair_reverse64(r.fm);
    return r;
}

HS_HD void roll_push(Roll &r, uint32_t code, int k)
{
    r.fm = ((r.fm << 2) | code) & kmer_mask(k);
    r.flp = (r.flp >> 2) | ((uint64_t)code << 62);
}

// S5: canonical k-mer, returned first-base-least-significant (byte order of the
// ASCII string murmur will read).  fwd <= rc compared first-base-most-significant
// == memcmp of the ASCII strings because 'A'<'C'<'G'<'T' and codes are 0..3.
HS_HD uint64_t canonical_lsb(const Roll &r, int k)
{
    const uint64_t mask = kmer_mask(k);
    const uint64_t fl = r.flp >> (64 - 2 * k);  // forward, LSB-first
    const uint64_t rm = (~fl) & mask;           // reverse complement, MSB-first
    return (r.fm <= rm) ? fl : ((~r.fm) & mask);
}

// ---- 2-bit -> ASCII expansion ---------------------------------------------
// ascii4(b): the four ASCII letters of the 4 bases in byte b (base i at bits
// [2i,2i+1]), first base in the low byte: what a little-endian load of the
// k-mer string would see.
HS_HD uint32_t ascii4(uint32_t b)
{
    const uint32_t lut = 0x54474341u;  // 'A','C','G','T' for codes 0..3
    return ((lut >> (8 * (b & 3))) & 0xFFu) | (((lut >> (8 * ((b >> 2) & 3))) & 0xFFu) << 8) |
           (((lut >> (8 * ((b >> 4) & 3))) & 0xFFu) << 16) | (((lut >> (8 * ((b >> 6) & 3))) & 0xFFu) << 24);
}

// ---- MurmurHash3_x64_128 ----------------------------------------------------
HS_HD uint64_t rotl64(uint64_t x, int r)
{
#if defined(__CUDA_ARCH__)
    // two funnel shifts; written out because the compiler otherwise builds the low word from a
    // multiply, a shift and an OR (the kernel is bound by integer issue slots)
    const uint32_t lo = (uint32_t)x, hi = (uint32_t)(x >> 32);
    const uint32_t a = r < 32 ? lo : hi, b = r < 32 ? hi : lo;   // rotate by r mod 32 after an optional swap
    const uint32_t nh = __funnelshift_l(a, b, (uint32_t)r), nl = __funnelshift_l(b, a, (uint32_t)r);
    return ((uint64_t)nh << 32) | nl;
#else
    return (x << r) | (x >> (64 - r));
#endif
}
// (Tried on B200 and dropped: x >> 1 as mul.hi by 2^31 and 64-bit adds as mad.wide by one, to move work
// from the busy ALU pipe to the multiply pipe -- 11 % slower, those forms do not issue at the plain
// multiply-add rate.)
HS_HD uint64_t xorshift33(uint64_t k)  // k ^ (k >> 33): only the low word changes
{
    const uint32_t hi = (uint32_t)(k >> 32);
    return ((uint64_t)hi << 32) | ((uint32_t)k ^ (hi >> 1));
}
HS_HD uint64_t fmix64(uint64_t k)
{
    k = xorshift33(k); k *= 0xff51afd7ed558ccdull;
    k = xorshift33(k); k *= 0xc4ceb9fe1a85ec53ull;
    k = xorshift33(k);
    return k;
}

// High word of fmix64(k).  Its last xorshift33 changes only the low word, and the high word of the
// last product is mul.hi(lo, c_lo) + lo * c_hi + hi * c_lo: three multiply-adds, no low-word product.
HS_HD uint32_t fmix64_hi(uint64_t k)
{
    k = xorshift33(k); k *= 0xff51afd7ed558ccdull;
    k = xorshift33(k);
    const uint32_t lo = (uint32_t)k, hi = (uint32_t)(k >> 32);
    const uint32_t c_lo = 0x1a85ec53u, c_hi = 0xc4ceb9feu;
#if defined(__CUDA_ARCH__)
    const uint32_t mh = __umulhi(lo, c_lo);
#else
    const uint32_t mh = (uint32_t)(((uint64_t)lo * c_lo) >> 32);
#endif
    return mh + lo * c_hi + hi * c_lo;
}

HS_HD uint64_t mul5_add(uint64_t h, uint32_t c)  // h * 5 + c
{
#if defined(__CUDA_ARCH__)
    const uint64_t t = (uint64_t)(uint32_t)h * 5u + c;                       // one wide multiply-add
    const uint32_t hi = (uint32_t)(h >> 32) * 5u + (uint32_t)(t >> 32);      // one multiply-add
    return ((uint64_t)hi << 32) | (uint32_t)t;
#else
    return h * 5 + c;
#endif
}

// h1 of MurmurHash3_x64_128 over the k (<= 32) ASCII bytes given as eight
// little-endian 32-bit words w[0..7]; bytes at index >= k MUST be zero.
HS_HD uint64_t murmur3_h1_words(const uint32_t w[8], int k, uint32_t seed)
{
    const uint64_t c1 = 0x87c37b91114253d5ull, c2 = 0x4cf5ad432745937full;
    uint64_t h1 = seed, h2 = seed;
    const int nblocks = k >> 4;
    int base = 0;
    for (int b = 0; b < 2; b++) {
        if (b < nblocks) {
            uint64_t k1 = (uint64_t)w[base] | ((uint64_t)w[base + 1] << 32);
            uint64_t k2 = (uint64_t)w[base + 2] | ((uint64_t)w[base + 3] << 32);
            k1 *= c1; k1 = rotl64(k1, 31); k1 *= c2; h1 ^= k1;
            h1 = rotl64(h1, 27); h1 += h2; h1 = h1 * 5 + 0x52dce729;
            k2 *= c2; k2 = rotl64(k2, 33); k2 *= c1; h2 ^= k2;
            h2 = rotl64(h2, 31); h2 += h1; h2 = h2 * 5 + 0x38495ab5;
            base += 4;
        }
    }
    if (k & 15) {
        // tail: zero padding makes the unconditional k2 step a no-op when <= 8 bytes remain
        uint64_t k1 = (uint64_t)w[base & 7] | ((uint64_t)w[(base + 1) & 7] << 32);
        uint64_t k2 = ((k & 15) > 8) ? ((uint64_t)w[(base + 2) & 7] | ((uint64_t)w[(base + 3) & 7] << 32)) : 0ull;
        k2 *= c2; k2 = rotl64(k2, 33); k2 *= c1; h2 ^= k2;
        k1 *= c1; k1 = rotl64(k1, 31); k1 *= c2; h1 ^= k1;
    }
    h1 ^= (uint64_t)k; h2 ^= (uint64_t)k;
    h1 += h2; h2 += h1;
    h1 = fmix64(h1); h2 = fmix64(h2);
    h1 += h2;
    return h1;
}

// Expand a canonical LSB-first k-mer and hash it.  `Lut(cl, i)` returns the 4 ASCII
// letters of byte i of cl: a shared-memory table on the device, plain arithmetic on the host.
template <class Lut>
HS_HD uint64_t hash_canonical(uint64_t cl, int k, uint32_t seed, bool use64, const Lut &lut)
{
    uint32_t w[8];
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const int nb = k - 4 * i;  // bases available for this word
        uint32_t v = 0;
        if (nb > 0) {
            v = lut(cl, i);  // letters of bases 4i..4i+3
            if (nb < 4) v &= (1u << (8 * nb)) - 1u;
        }
        w[i] = v;
    }
    const uint64_t h = murmur3_h1_words(w, k, seed);
    return use64 ? h : (h & 0xFFFFFFFFull);
}

// ---- the same hash from PRE-MULTIPLIED table entries ---------------------------------
// Murmur reads the k-mer string as 64-bit lanes: lane 0 = bytes 0-7 and lane 2 = bytes 16-23 are
// multiplied by c1 first, lanes 1 and 3 by c2.  A lane is (lo word) + (hi word << 32), so modulo
// 2^64   lane * c = (u64)lo * c  +  ((u32)(hi * c) << 32):
// a table of the 64-bit products of all 256 four-letter words (one per constant) turns the first
// multiply of every lane -- 3 of the 10 64-bit multiplies at k=21, 4 of 12 at k=31 -- into one
// 64-bit and one 32-bit load plus one add.  Table entries exist for whole words only; a lane
// that ends inside a word sees 'A' (code 0) in the unused byte positions, whose known product
// is subtracted.
constexpr uint64_t kMurmurC1 = 0x87c37b91114253d5ull, kMurmurC2 = 0x4cf5ad432745937full;

HS_HD uint64_t premul_entry(uint32_t b, bool second) { return (uint64_t)ascii4(b) * (second ? kMurmurC2 : kMurmurC1); }

// product of the filler letters of a lane holding nb (1..8) real bytes
HS_HD uint64_t premul_filler(int nb, bool second)
{
    const uint64_t c = second ? kMurmurC2 : kMurmurC1;
    if (nb >= 8 || nb == 4) return 0;
    if (nb > 4) return ((uint64_t)(0x41414141u & ~((1u << (8 * (nb - 4))) - 1u)) << 32) * c;
    return (uint64_t)(0x41414141u & ~((1u << (8 * nb)) - 1u)) * c;
}

// A tail of 1..5 letters (k mod 16, e.g. k = 21: the HYMET default) is one lane of at most ten bits:
// its whole contribution  rotl64(lane * c1, 31) * c2  -- two table reads, an add, a rotate and a 64-bit
// multiply, about a tenth of the loop -- fits a table of 4^r 64-bit entries (8 KB at r = 5).
// x holds the r letters, first letter most significant, in its low 2r bits.
HS_HD bool tail_table_applies(int k) { return (k & 15) >= 1 && (k & 15) <= 5; }
HS_HD uint64_t tail_entry(uint32_t x, int r)
{
    uint64_t lane = 0;
    for (int i = 0; i < r; i++) lane |= (uint64_t)((0x54474341u >> (8 * ((x >> (2 * (r - 1 - i))) & 3u))) & 0xFFu) << (8 * i);
    uint64_t k1 = lane * kMurmurC1;
    k1 = (k1 << 31) | (k1 >> 33);
    return k1 * kMurmurC2;
}

// h1 and h2 of MurmurHash3_x64_128 right before the finalizer: h1 of the hash is fmix64(x) + fmix64(y).
struct MurmurState { uint64_t x, y; };

HS_HD uint64_t murmur_finish(const MurmurState &s) { return fmix64(s.x) + fmix64(s.y); }

// ---- range gate on the high word ---------------------------------------------------------------
// The kernels' pre-filter keeps a 64-bit hash h only when h <= gate, and turns away all but a few
// k-mers in a thousand.  Deciding that from the high words alone saves most of the finalizer:
// with  s = fmix64_hi(x) + fmix64_hi(y)  (mod 2^32), the true high word of h is s or s + 1, the
// carry out of the low-word add.  The test  (u32)(s + 1) <= gate_hi + 1  accepts every s in
// [0, gate_hi] and also s = 0xFFFFFFFF (whose carry wraps the high word to 0), so it accepts every
// h <= gate: no false negatives.  It also accepts h > gate when hi32(h) == gate_hi (as a compare of
// high words would), when s == gate_hi carried into gate_hi + 1, and when s == 0xFFFFFFFF did not
// carry -- a few in 2^32 beyond that.  Callers finish the hash exactly for the k-mers that pass and
// repeat the exact 64-bit test.  gate_hi + 1 must not wrap: for gate_hi == 0xFFFFFFFF the bound
// saturates and every k-mer takes the exact test (then every k-mer is let through by the gate
// anyway).
HS_HD uint32_t murmur_finish_hi_floor(const MurmurState &s) { return fmix64_hi(s.x) + fmix64_hi(s.y); }
HS_HD uint32_t hi_gate_bound(uint64_t gate)
{
    const uint32_t gate_hi = (uint32_t)(gate >> 32);
    return gate_hi == 0xFFFFFFFFu ? gate_hi : gate_hi + 1u;
}
HS_HD bool hi_gate_may_pass(uint32_t s_hi, uint32_t bound) { return (uint32_t)(s_hi + 1u) <= bound; }

// `Pre::full(cl, i, second)`: 64-bit product of word i's letters; `Pre::low`: its low 32 bits;
// `Pre::kTail` / `Pre::tail(cl, k)`: the finished tail term when a table of it exists.
template <class Pre>
HS_HD MurmurState murmur_state_premul(uint64_t cl, int k, uint32_t seed, const Pre &pre)
{
    const bool tail_tab = Pre::kTail && tail_table_applies(k);
    uint64_t m[4];
#pragma unroll
    for (int l = 0; l < 4; l++) {
        const int nb = k - 8 * l;
        uint64_t p = 0;
        if (nb > 0 && !(tail_tab && l == 2 * (k >> 4))) {
            p = pre.full(cl, 2 * l, (l & 1) != 0);
            if (nb > 4) {   // only the high word changes: one 32-bit add (filler folded in), no carry chain
                const uint32_t hi = (uint32_t)(p >> 32) + pre.low(cl, 2 * l + 1, (l & 1) != 0) -
                                    (uint32_t)(premul_filler(nb, (l & 1) != 0) >> 32);
                p = ((uint64_t)hi << 32) | (uint32_t)p;
            } else {
                p -= premul_filler(nb, (l & 1) != 0);
            }
        }
        m[l] = p;
    }
    const uint64_t c1 = kMurmurC1, c2 = kMurmurC2;
    uint64_t h1 = seed, h2 = seed;
    const int t = 2 * (k >> 4);  // first lane of the tail
#pragma unroll
    for (int b = 0; b < 2; b++) {
        if (b < (k >> 4)) {
            uint64_t k1 = m[2 * b], k2 = m[2 * b + 1];
            k1 = rotl64(k1, 31); k1 *= c2; h1 ^= k1;
            h1 = rotl64(h1, 27); h1 += h2; h1 = mul5_add(h1, 0x52dce729u);
            k2 = rotl64(k2, 33); k2 *= c1; h2 ^= k2;
            h2 = rotl64(h2, 31); h2 += h1; h2 = mul5_add(h2, 0x38495ab5u);
        }
    }
    if (k & 15) {
        if ((k & 15) > 8) { uint64_t k2 = m[(t + 1) & 3]; k2 = rotl64(k2, 33); k2 *= c1; h2 ^= k2; }
        uint64_t k1;
        if (tail_tab) { k1 = pre.tail(cl, k); }
        else { k1 = m[t & 3]; k1 = rotl64(k1, 31); k1 *= c2; }
        h1 ^= k1;
    }
    h1 ^= (uint64_t)k; h2 ^= (uint64_t)k;
    h1 += h2; h2 += h1;
    return MurmurState{h1, h2};
}

template <class Pre>
HS_HD uint64_t hash_canonical_premul(uint64_t cl, int k, uint32_t seed, bool use64, const Pre &pre)
{
    const uint64_t h = murmur_finish(murmur_state_premul(cl, k, seed, pre));
    return use64 ? h : (h & 0xFFFFFFFFull);
}

struct PremulArith {  // host-side stand-in for the shared-memory tables (tests)
    static constexpr bool kTail = false;
    HS_HD uint64_t tail(uint64_t, int) const { return 0; }
    HS_HD uint64_t full(uint64_t cl, int i, bool second) const { return premul_entry((uint32_t)(cl >> (8 * i)) & 0xFFu, second); }
    HS_HD uint32_t low(uint64_t cl, int i, bool second) const { return (uint32_t)full(cl, i, second); }
};

// ---- windowed canonical k-mers ------------------------------------------------------------
// One thread owns the 64 bases (prev word, cur word).  Instead of rolling two k-mers base by base,
// keep the 128-bit window W = prev:cur and its reverse complement in eight 32-bit registers and cut
// every k-mer out of them with funnel shifts (below: TOP-aligned).
struct Win { uint32_t f0, f1, f2, f3, r0, r1, r2, r3; };  // word 0 least significant

HS_HD uint32_t funnel_r(uint32_t lo, uint32_t hi, int s)  // low 32 bits of (hi:lo) >> s, 0 <= s <= 31
{
#if defined(__CUDA_ARCH__)
    return __funnelshift_r(lo, hi, (uint32_t)s);
#else
    return (uint32_t)((((uint64_t)hi << 32) | lo) >> s);
#endif
}

// Table entries for k-mers whose first base is MOST significant: the index byte holds a word's first
// letter in its top two bits.
HS_HD uint32_t pair_reverse8(uint32_t b) { return ((b & 3u) << 6) | ((b & 0xCu) << 2) | ((b >> 2) & 0xCu) | ((b >> 6) & 3u); }
HS_HD uint64_t premul_entry_msb(uint32_t b, bool second) { return premul_entry(pair_reverse8(b), second); }

// ---- TOP-aligned: k-mers sit in the most significant 2k bits of 64 ------------------------------
// With F'' = W << (66-2k) and R'' = revcomp(W) >> 2, the forward k-mer ending at base j is the top
// of F'' << 2j and its reverse complement the bottom 64 bits of R'' >> 2j.  Whatever lies below the
// 2k bits (later bases) only matters when forward == reverse complement, and then either choice is
// the same k-mer: no masks before the compare.  String word i is byte (7-i) of the value for
// every k, so index shifts never straddle a register; a last word with fewer than four bases drops
// the bases that are not its own through the mask of the address computation.
HS_HD uint32_t funnel_l(uint32_t lo, uint32_t hi, int s)  // high 32 bits of (hi:lo) << s, 0 <= s <= 31
{
#if defined(__CUDA_ARCH__)
    return __funnelshift_l(lo, hi, (uint32_t)s);
#else
    return (uint32_t)(((((uint64_t)hi << 32) | lo) << s) >> 32);
#endif
}

HS_HD Win win_init_top(uint64_t prev, uint64_t cur, int k)
{
    Win w;
    const int c = 66 - 2 * k;   // 2..64
    const uint64_t fh = c >= 64 ? cur : ((prev << c) | (cur >> (64 - c)));
    const uint64_t fl = c >= 64 ? 0ull : (cur << c);
    w.f0 = (uint32_t)fl; w.f1 = (uint32_t)(fl >> 32); w.f2 = (uint32_t)fh; w.f3 = (uint32_t)(fh >> 32);
    const uint64_t rh = pair_reverse64(~cur), rl = pair_reverse64(~prev);  // revcomp(W) = rh:rl
    const uint64_t lo = (rl >> 2) | (rh << 62), hi = rh >> 2;
    w.r0 = (uint32_t)lo; w.r1 = (uint32_t)(lo >> 32); w.r2 = (uint32_t)hi; w.r3 = (uint32_t)(hi >> 32);
    return w;
}

// q = j mod 16; forward words (fa, fb, fc) = (f1, f2, f3) for j < 16 else (f0, f1, f2); reverse words
// (ra, rb, rc) = (r0, r1, r2) for j < 16 else (r1, r2, r3)
HS_HD uint64_t canonical_top_half(uint32_t fa, uint32_t fb, uint32_t fc, uint32_t ra, uint32_t rb, uint32_t rc, int q)
{
    const uint32_t flo = funnel_l(fa, fb, 2 * q), fhi = funnel_l(fb, fc, 2 * q);
    const uint32_t rlo = funnel_r(ra, rb, 2 * q), rhi = funnel_r(rb, rc, 2 * q);
    const uint64_t fm = ((uint64_t)fhi << 32) | flo, rm = ((uint64_t)rhi << 32) | rlo;
    return fm <= rm ? fm : rm;
}

HS_HD uint64_t canonical_top(const Win &w, int j)
{
    return j < 16 ? canonical_top_half(w.f1, w.f2, w.f3, w.r0, w.r1, w.r2, j)
                  : canonical_top_half(w.f0, w.f1, w.f2, w.r1, w.r2, w.r3, j - 16);
}

// index byte of word i, times 2^lg (the table's entry stride)
HS_HD uint32_t top_word_index(uint64_t ct, int i, int k, int lg)
{
    const uint32_t w = i < 4 ? (uint32_t)(ct >> 32) : (uint32_t)ct;
    const int sh = 24 - lg - 8 * (i & 3);
    const uint32_t x = sh >= 0 ? (w >> sh) : (w << (-sh));
    const int nb = k - 4 * i;   // bases of this word that belong to the k-mer
    const uint32_t keep = (nb >= 4 ? 0xFFu : ((0xFFu << (8 - 2 * nb)) & 0xFFu)) << lg;
    return x & keep;
}

// ---- shared-memory layout of the stream kernel's tables (screen_kernels.cu: SmemPremul) -------------
// The host tests model the 32 banks with these same functions.
//   Premultiplied tables: 256 entries, COPIES lane copies each; entry b, copy c at b * 8 * COPIES + c * 8.
//     Lane l reads copy l mod COPIES.  With 16 copies the entry stride is 128 B, so the 16 lanes of a
//     half-warp read 16 different bank pairs whatever their entries: a 64-bit read takes 2 wavefronts, a
//     32-bit read (the low word) 2.  The second table lies kBytes further on, reached through the
//     load's immediate offset; the base is kBytes-aligned, so lane term and index combine with one OR.
//   Tail-term table: 4^r entries, TCOPIES interleaved copies; entry e, copy c at (e * TCOPIES + c) * 8.
//     Lane l reads copy l mod TCOPIES, so the lanes of different copies read disjoint sets of bank pairs.
//     The table lies 2 * kBytes above the same base.
template <int COPIES, int TCOPIES>
struct SmemLayout {
    static constexpr uint32_t kStride = 8u * COPIES, kBytes = 256u * kStride;
    static constexpr int kStrideLog2 = COPIES == 16 ? 7 : COPIES == 8 ? 6 : -1;
    static constexpr int kTailLog2 = TCOPIES == 2 ? 4 : TCOPIES == 1 ? 3 : -1;
    static_assert(kStrideLog2 > 0 && kTailLog2 > 0, "layouts with 8 or 16 copies, 1 or 2 tail copies");
    HS_HDC static uint32_t tail_bytes(int r) { return (8u * TCOPIES) << (2 * r); }
    HS_HD static uint32_t lane_base(uint32_t lut, uint32_t lane) { return lut | ((lane & (COPIES - 1u)) << 3); }
    HS_HD static uint32_t tail_base(uint32_t lut, uint32_t lane) { return lut | ((lane & (TCOPIES - 1u)) << 3); }
    // Word i's entry (add kBytes for the second table).  A whole word's index byte sits on a byte boundary
    // of the top-aligned k-mer: ONE byte permute (ALU pipe) and ONE multiply-add (FMA pipe) by `stride`
    // (== kStride; the kernel passes it in a register the compiler cannot see through, or ptxas would
    // strength-reduce the multiply back to a shift and a three-input logic op, two ALU-pipe instructions,
    // and the kernel is bound by the half-rate ALU pipe).  A partial last word keeps the masked form.
    HS_HD static uint32_t word_addr(uint64_t ct, int i, int k, uint32_t base, uint32_t stride)
    {
        if (k - 4 * i >= 4) {
            const uint32_t w = i < 4 ? (uint32_t)(ct >> 32) : (uint32_t)ct;
#if defined(__CUDA_ARCH__)
            const uint32_t byte = __byte_perm(w, 0u, 0x4440u + (uint32_t)(3 - (i & 3)));
            uint32_t addr;
            asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(addr) : "r"(byte), "r"(stride), "r"(base));
            return addr;
#else
            return ((w >> (8 * (3 - (i & 3)))) & 0xFFu) * stride + base;
#endif
        }
        return top_word_index(ct, i, k, kStrideLog2) | base;
    }
    // the tail's entry (add 2 * kBytes): its letters start at the top of one 32-bit half of the k-mer
    // (top_tail_index), so one shift and one AND-OR
    HS_HD static uint32_t tail_addr(uint64_t ct, int k, uint32_t tbase)
    {
        const int r = k & 15;
        const uint32_t w = (k >> 4) ? (uint32_t)ct : (uint32_t)(ct >> 32);
        return ((w >> (32 - 2 * r - kTailLog2)) & (((1u << (2 * r)) - 1u) << kTailLog2)) | tbase;
    }
};

template <class Pre>
struct TopAdapter {   // `where` turns (k-mer, word number) into whatever the table accessor addresses by
    static constexpr bool kTail = Pre::kTail;
    const Pre &p; int k;
    HS_HD uint64_t full(uint64_t c, int i, bool second) const { return p.full(p.where(c, i, k), second); }
    HS_HD uint32_t low(uint64_t c, int i, bool second) const { return p.low(p.where(c, i, k), second); }
    HS_HD uint64_t tail(uint64_t c, int kk) const { return p.tail(c, kk); }
};

template <class Pre>
HS_HD uint64_t hash_canonical_premul_top(uint64_t ct, int k, uint32_t seed, bool use64, const Pre &pre)
{
    return hash_canonical_premul(ct, k, seed, use64, TopAdapter<Pre>{pre, k});
}

template <class Pre>
HS_HD MurmurState murmur_state_premul_top(uint64_t ct, int k, uint32_t seed, const Pre &pre)
{
    return murmur_state_premul(ct, k, seed, TopAdapter<Pre>{pre, k});
}

// the tail's letters inside a TOP-aligned k-mer: letters 16*(k>>4) .. k-1 end at bit 64-2k, and start at
// the top of one of the two 32-bit halves (letter 0 or letter 16), so the index is one right shift
HS_HD uint32_t top_tail_index(uint64_t ct, int k)
{
    const int r = k & 15;
    const uint32_t w = (k >> 4) ? (uint32_t)ct : (uint32_t)(ct >> 32);
    return w >> (32 - 2 * r);
}

struct PremulArithMsb {  // host-side stand-in for the shared-memory tables (tests)
    static constexpr bool kTail = true;
    HS_HD uint64_t tail(uint64_t ct, int k) const { return tail_entry(top_tail_index(ct, k), k & 15); }
    HS_HD uint32_t where(uint64_t ct, int i, int k) const { return top_word_index(ct, i, k, 6); }
    HS_HD uint64_t full(uint32_t index64, bool second) const { return premul_entry_msb(index64 >> 6, second); }
    HS_HD uint32_t low(uint32_t index64, bool second) const { return (uint32_t)full(index64, second); }
};

struct AsciiArith {
    HS_HD uint32_t operator()(uint64_t cl, int i) const { return ascii4((uint32_t)(cl >> (8 * i)) & 0xFFu); }
};

// One thread's unit of work: the 32 k-mers that END inside word `cur` (their
// first bases may lie in `prev`; k <= 32 so never further back).  sink(j, hash)
// is called for every valid k-mer ending at base j of `cur`, in order.
template <class Lut, class Sink>
HS_HD void for_each_kmer_in_word(uint64_t prev, uint64_t cur, uint32_t inv_prev, uint32_t inv_cur, int k,
                                 uint32_t seed, bool use64, const Lut &lut, Sink &&sink)
{
    const uint32_t bad = invalid_kmer_ends(inv_prev, inv_cur, k);
    Roll r = roll_init(prev, k);
#pragma unroll 4
    for (int j = 0; j < kBasesPerWord; j++) {
        roll_push(r, (uint32_t)(cur >> (62 - 2 * j)) & 3u, k);
        if (!((bad >> (31 - j)) & 1u)) sink(j, hash_canonical(canonical_lsb(r, k), k, seed, use64, lut));
    }
}

// ---- sketch hash table ------------------------------------------------------
// One bucket = one 128-byte line, the unit B200 moves between HBM and L2 whatever the
// request size (round 1, ncu: 3.8 DRAM sectors per 32-byte bucket read):
//   u64 word  0..9   keys (kEmptyKey = free)
//   u32 word 20..29  canonical entry id of the key in the same slot
//   u32 word 30      overflow flag: a key whose probe sequence passed this bucket lives further on
//   u32 word 31      unused
// so a probe is ONE line whether it hits or misses (round 1 kept the ids in a second array: a
// second DRAM fetch per hit), a miss ends at the first bucket whose flag is clear, and ten slots
// per bucket let the load factor be 0.5 (26 B per key; round 1: four slots at 1/3 = 36 B).
// Reference hashes are bottom-s values (numerically small) so the bucket index re-mixes both
// halves before the multiply-high range reduction.
constexpr uint64_t kEmptyKey = ~0ull;
constexpr int kBucketSlots = 10;
constexpr int kBucketWords = 16;          // 64-bit words per bucket
constexpr int kBucketValWord32 = 20;      // first id, as a 32-bit word index inside the bucket
constexpr int kBucketOverWord32 = 30;

HS_HD uint32_t bucket_of(uint64_t h, uint32_t n_buckets)
{
    uint32_t m = (uint32_t)h ^ ((uint32_t)(h >> 32) * 0x9E3779B1u);
    m *= 0x85EBCA77u;
    m ^= m >> 15;
    m *= 0xC2B2AE3Du;
#if defined(__CUDA_ARCH__)
    return __umulhi(m, n_buckets);
#else
    return (uint32_t)(((uint64_t)m * n_buckets) >> 32);
#endif
}

// Blocked Bloom filter over the keys ABOVE the dense range (see TableView): which 32-bit word, and
// which 3 bits inside it, belong to hash h.  A 64-bit MurmurHash3 value is already mixed, so its
// bits are used as they are (18 position bits, then the word index); 32-bit hashes (k <= 16) are
// re-mixed first.
HS_HD void bloom_slot(uint64_t h, uint32_t word_mask, bool use64, uint32_t &word, uint32_t &bits)
{
    const uint64_t g = use64 ? h : h * 0x9E3779B97F4A7C15ull;
    const uint32_t lo = use64 ? (uint32_t)g : (uint32_t)(g >> 32);
    word = (uint32_t)(g >> (use64 ? 15 : 8)) & word_mask;
    bits = (1u << (lo & 31u)) | (1u << ((lo >> 5) & 31u)) | (1u << ((lo >> 10) & 31u));
}

HS_HD uint32_t mixset_slot(uint64_t h, uint32_t mask)
{
    uint64_t x = h * 0x9E3779B97F4A7C15ull;
    return (uint32_t)(x >> 40) & mask;
}

}  // namespace hs
