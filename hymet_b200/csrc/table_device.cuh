// table_device.cuh -- device functions shared by the screen kernels (screen_kernels.cu) and the
// distance kernels (distance_kernels.cu): the key-table probe, the entry -> reference lookup of the
// hash -> references chains, and the binomial upper tail of the p-values.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "kmer_core.cuh"
#include "screen_kernels.h"

namespace hs {

// ---------------------------------------------------------------------------
// table lookup, one thread per probe (k_stream's rare path, k_table_canon)
// ---------------------------------------------------------------------------
// LEAN: one 16-byte load at a time (two live registers instead of twenty) -- k_stream probes for
// ~0.07 % of its k-mers and must not pay for the probe's registers in its hot loop; the later
// loads of a bucket hit the line the first one brought in.  !LEAN: all six loads of a bucket in flight.
template <bool LEAN>
__device__ __forceinline__ uint32_t table_find_from(const TableView &t, uint64_t h, uint32_t b, uint32_t &n_reads)
{
    for (uint32_t tries = 0; tries < t.n_buckets; tries++) {
        const ulonglong2 *p = reinterpret_cast<const ulonglong2 *>(t.buckets + (size_t)b * kBucketWords);
        const uint32_t *p32 = reinterpret_cast<const uint32_t *>(p);
        n_reads++;
        int slot = -1;
        if (LEAN) {
#pragma unroll 1
            for (int i = 0; i < kBucketSlots / 2; i++) {
                const ulonglong2 k = __ldg(p + i);
                if (k.x == h) { slot = 2 * i; break; }
                if (k.y == h) { slot = 2 * i + 1; break; }
            }
        } else {
            ulonglong2 k[kBucketSlots / 2];
#pragma unroll
            for (int i = 0; i < kBucketSlots / 2; i++) k[i] = __ldg(p + i);
#pragma unroll
            for (int i = 0; i < kBucketSlots / 2; i++) {
                if (k[i].x == h) slot = 2 * i;
                if (k[i].y == h) slot = 2 * i + 1;
            }
        }
        if (slot >= 0) return __ldg(p32 + kBucketValWord32 + slot);
        if (!__ldg(p32 + kBucketOverWord32)) return kNoEntry;   // nothing that hashed here went further
        b = (b + 1 == t.n_buckets) ? 0u : b + 1;
    }
    return kNoEntry;
}

template <bool LEAN>
__device__ __forceinline__ uint32_t table_find(const TableView &t, uint64_t h, uint32_t &n_reads)
{
    if (h == kEmptyKey) return t.special;
    return table_find_from<LEAN>(t, h, bucket_of(h, t.n_buckets), n_reads);
}

// reference that owns entry e: the largest i with offsets[i] <= e (offsets[0] = 0 <= e < offsets[n_refs]).
// Sketches of one database nearly all hold s hashes, so e * n_refs / E is the answer or next to it: two
// loads instead of the ~18 dependent ones of a binary search over 300 000 offsets (the search stays as
// the fallback for databases with uneven sketch sizes).
__device__ __forceinline__ uint32_t ref_of_entry(const uint64_t *offsets, uint32_t n_refs, uint64_t e, uint64_t scale = 0)
{
    if (scale) {
        uint32_t g = (uint32_t)__umul64hi(e, scale);
        if (g >= n_refs) g = n_refs - 1;
        const uint64_t a = __ldg(offsets + g), b = __ldg(offsets + g + 1);
        if (a <= e && e < b) return g;
        if (e >= b && g + 2 <= n_refs && e < __ldg(offsets + g + 2)) return g + 1;
        if (e < a && g > 0 && __ldg(offsets + g - 1) <= e) return g - 1;
    }
    uint32_t lo = 0, hi = n_refs;
    while (hi - lo > 1u) {
        const uint32_t mid = (lo + hi) >> 1;
        if (__ldg(offsets + mid) <= e) lo = mid; else hi = mid;
    }
    return lo;
}

// ---------------------------------------------------------------------------
// binomial upper tail (K6 and the distance p-values)
// ---------------------------------------------------------------------------
// P[Binomial(n, r) >= x], summed term by term from the term at x.  The leading term
// C(n,x) r^x (1-r)^(n-x) is built as a running product with an explicit binary
// exponent, so nothing large is ever exponentiated: relative error ~ sqrt(x) ulp.
// One WARP per sketch: the lanes split the factors of the leading term between them (a sketch with
// 10 000 shared hashes has a 10 000-factor product, and the few hundred sketches with hits used to
// be the whole run time of the kernel as 16 fully divergent warps), combine the partial products
// in a butterfly (multiplication commutes, so every lane ends with the same bits) and then all
// evaluate the short geometric-like tail redundantly.
__device__ inline double binom_upper_tail_warp(uint64_t x, uint64_t n, double r, uint32_t lane)
{
    if (x == 0) return 1.0;
    if (x > n) return 0.0;
    if (!(r > 0.0)) return 0.0;
    if (r >= 1.0) return 1.0;
    const double q = 1.0 - r;
    const bool upper = (double)x > (double)n * r;  // sum the smaller side
    const uint64_t j0 = upper ? x : x - 1;         // first term of the side we sum
    // t(j0) = prod_{i=1..j0} ((n-j0+i)/i * r) * q^(n-j0): numerator and denominator as separate
    // running products (one division at the end: FP64 division is slow), renormalised every four
    // factors -- four factors cannot move a value normalised into [0.5, 1) out of range (5e-20 .. 1e7)
    double num = 1.0, den = 1.0;
    long long ex = 0;
    uint32_t since = 0;
    for (uint64_t i = 1 + lane; i <= j0; i += 32) {
        num *= (double)(n - j0 + i) * r;
        den *= (double)i;
        if (++since == 4) {
            int e2;
            num = frexp(num, &e2); ex += e2;
            den = frexp(den, &e2); ex -= e2;
            since = 0;
        }
    }
    {
        int e2;
        num = frexp(num, &e2); ex += e2;
        den = frexp(den, &e2); ex -= e2;
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        num *= __shfl_xor_sync(0xffffffffu, num, o);
        den *= __shfl_xor_sync(0xffffffffu, den, o);
        ex += __shfl_xor_sync(0xffffffffu, ex, o);
        int e2;
        num = frexp(num, &e2); ex += e2;
        den = frexp(den, &e2); ex -= e2;
    }
    double mant = num / den;
    {
        const double e2 = (double)(n - j0) * log2(q);
        const double fl = floor(e2);
        mant *= exp2(e2 - fl);
        ex += (long long)fl;
    }
    // geometric-like continuation
    double sum = 1.0, term = 1.0;
    if (upper) {
        const double rq = r / q;
        for (uint64_t j = j0; j < n; j++) {
            term *= ((double)(n - j) / (double)(j + 1)) * rq;
            sum += term;
            if (term < sum * 1e-18) break;
        }
    } else {
        const double qr = q / r;
        for (uint64_t j = j0; j > 0; j--) {
            term *= ((double)j / (double)(n - j + 1)) * qr;
            sum += term;
            if (term < sum * 1e-18) break;
        }
    }
    int e2;
    mant = frexp(mant * sum, &e2);
    ex += e2;
    const double side = ex < -1100 ? 0.0 : ldexp(mant, (int)ex);
    return upper ? side : 1.0 - side;
}

}  // namespace hs
