// distance_kernels.cu -- hand-written sm_100a kernels of `mash dist` (DESIGN.md §5 "mash dist").
//
// A block of query sketches against every reference sketch of one .msh, exactly:
//   k_dist_mark     probe every query hash in the references' key table and walk the chain of the
//                   references that hold it: bit r of the query's bitmap row = "shares a hash with r".
//                   Pairs that share nothing never leave the device (the host writes them implicitly).
//   k_dist_count / k_dist_scan / k_dist_compact
//                   popcount of every row, one scan, and the set bits as (q, r) rows in (q, r) order:
//                   output slots come from the scan, so line order does not depend on scheduling.
//   k_dist_merge    one warp per candidate pair: Mash's truncated merge of the two sorted sketches,
//                   32 union elements per step (merge-path windows), then the binomial p-value.
#include <cuda_runtime.h>
#include <stdint.h>

#include "distance_kernels.h"
#include "kmer_core.cuh"
#include "table_device.cuh"

namespace hs {

namespace {

constexpr uint32_t kFull = 0xffffffffu;

__device__ __forceinline__ uint32_t warp_inclusive_sum(uint32_t v, uint32_t lane)
{
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t u = __shfl_up_sync(kFull, v, o);
        if (lane >= (uint32_t)o) v += u;
    }
    return v;
}

// one warp per query row; lanes stride over the query's hashes
__global__ void __launch_bounds__(256) k_dist_mark(const DistArgs a)
{
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t row = warp; row < a.n_q; row += n_warps) {
        const uint32_t q = a.q0 + row;
        const uint64_t b = __ldg(a.q_off + q), e = __ldg(a.q_off + q + 1);
        uint32_t *bits = a.bitmap + (size_t)row * a.words;
        for (uint64_t x = b + lane; x < e; x += 32) {
            const uint64_t h = __ldg(a.q_hashes + x);
            if (h > a.tab.max_key) continue;          // above every stored hash: shared with nobody
            uint32_t reads = 0;
            for (uint32_t id = table_find<true>(a.tab, h, reads); id != kNoEntry; id = __ldg(a.next + id)) {
                const uint32_t r = ref_of_entry(a.ref_off, a.n_refs, id, a.ref_scale);
                atomicOr(bits + (r >> 5), 1u << (r & 31u));
            }
        }
    }
}

__global__ void __launch_bounds__(256) k_dist_count(const DistArgs a)
{
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t row = warp; row < a.n_q; row += n_warps) {
        const uint32_t *bits = a.bitmap + (size_t)row * a.words;
        uint32_t n = 0;
        for (uint32_t w = lane; w < a.words; w += 32) n += __popc(__ldcg(bits + w));
#pragma unroll
        for (int o = 16; o; o >>= 1) n += __shfl_xor_sync(kFull, n, o);
        if (lane == 0) a.row_start[row] = n;
    }
}

// exclusive scan of row_start[0, n_q) in place, total in row_start[n_q]; one CTA of 1024 threads
__global__ void __launch_bounds__(1024) k_dist_scan(const DistArgs a)
{
    __shared__ unsigned long long warp_tot[32];
    __shared__ unsigned long long carry;
    const uint32_t lane = threadIdx.x & 31u, wid = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < a.n_q; base += 1024) {
        const uint32_t i = base + threadIdx.x;
        const unsigned long long v = i < a.n_q ? a.row_start[i] : 0;
        unsigned long long incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long u = __shfl_up_sync(kFull, incl, o);
            if (lane >= (uint32_t)o) incl += u;
        }
        if (lane == 31) warp_tot[wid] = incl;
        __syncthreads();
        if (wid == 0) {
            unsigned long long t = warp_tot[lane], ti = t;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned long long u = __shfl_up_sync(kFull, ti, o);
                if (lane >= (uint32_t)o) ti += u;
            }
            warp_tot[lane] = ti - t;   // exclusive over warps
        }
        __syncthreads();
        const unsigned long long c0 = carry;
        if (i < a.n_q) a.row_start[i] = c0 + warp_tot[wid] + incl - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry = c0 + warp_tot[31] + incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) a.row_start[a.n_q] = carry;
}

// one warp per row: its set bits, in reference order, to rows[row_start[row] ...]; the row is cleared
// on the way (the next block needs a zero bitmap)
__global__ void __launch_bounds__(256) k_dist_compact(const DistArgs a)
{
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t row = warp; row < a.n_q; row += n_warps) {
        uint32_t *bits = a.bitmap + (size_t)row * a.words;
        unsigned long long out = a.row_start[row];
        for (uint32_t w0 = 0; w0 < a.words; w0 += 32) {
            const uint32_t w = w0 + lane;
            uint32_t m = 0;
            if (w < a.words) {
                m = __ldcg(bits + w);
                if (m) bits[w] = 0;
            }
            const uint32_t n = __popc(m), incl = warp_inclusive_sum(n, lane);
            unsigned long long o = out + incl - n;
            while (m) {
                const uint32_t bit = __ffs(m) - 1;
                m &= m - 1;
                if (o < a.cap) {
                    DistRow *d = a.rows + o;
                    d->q = a.q0 + row;
                    d->r = w * 32 + bit;
                }
                o++;
            }
            out += __shfl_sync(kFull, incl, 31);
        }
    }
}

// D1 for one pair, the whole warp cooperating: Mash's loop
//     while (denom < s && i < |A| && j < |B|) { if A[i] < B[j] i++; else if A[i] > B[j] j++; else { i++; j++; common++; } denom++; }
//     then the rest of the longer list, denom capped at s
// consumes the union of A and B in ascending order.  Here each step takes the next 32 hashes of each
// list; every element <= m (the smaller of the two windows' last elements, when a window is full) has
// all its smaller elements of the other list inside that list's window, so its union rank is known:
// a shared hash at A[ia] == B[jb] with c shared hashes before it has rank ia + jb - c + 1, and the
// loop counts it iff that rank is <= s.  A full window is consumed whole, so each step takes >= 32.
__device__ __forceinline__ void dist_merge_warp(const uint64_t *A, uint32_t na, const uint64_t *B, uint32_t nb, uint32_t sp,
                                                uint32_t lane, uint32_t &common, uint32_t &denom)
{
    const uint32_t lt = (1u << lane) - 1u;
    uint32_t i = 0, j = 0, c = 0, cm = 0;
    while (i + j - c < sp && i < na && j < nb) {
        const bool va = i + lane < na, vb = j + lane < nb;
        const uint64_t a = va ? __ldg(A + i + lane) : 0, b = vb ? __ldg(B + j + lane) : 0;
        const bool full_a = i + 32 <= na, full_b = j + 32 <= nb;
        const uint64_t last_a = __shfl_sync(kFull, a, 31), last_b = __shfl_sync(kFull, b, 31);
        const bool bounded = full_a || full_b;
        const uint64_t m = full_a ? (full_b ? min(last_a, last_b) : last_a) : last_b;
        const bool ca = va && (!bounded || a <= m), cb = vb && (!bounded || b <= m);
        uint32_t n_lt = 0;
        bool eq = false;
        const uint32_t nvb = min(nb - j, 32u);
#pragma unroll 8
        for (uint32_t t = 0; t < 32; t++) {
            const uint64_t bt = __shfl_sync(kFull, b, t);
            const bool vt = t < nvb;
            n_lt += (vt && bt < a);
            eq |= (vt && bt == a);
        }
        const bool shared = ca && eq;
        const uint32_t S = __ballot_sync(kFull, shared);
        const uint32_t before = c + __popc(S & lt);
        const bool counted = shared && (i + lane) + (j + n_lt) - before + 1u <= sp;
        cm += __popc(__ballot_sync(kFull, counted));
        i += __popc(__ballot_sync(kFull, ca));
        j += __popc(__ballot_sync(kFull, cb));
        c += __popc(S);
    }
    uint64_t u = (uint64_t)i + j - c;
    if (u < sp) u += (uint64_t)(na - i) + (nb - j);   // one list is exhausted: the rest of the other shares nothing
    denom = (uint32_t)(u < sp ? u : sp);
    common = cm;
}

__global__ void __launch_bounds__(256) k_dist_merge(const DistArgs a)
{
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    const unsigned long long total = __ldcg(a.row_start + a.n_q);
    const uint32_t n = (uint32_t)(total < a.cap ? total : a.cap);
    const double kmer_space = ldexp(1.0, 2 * (int)a.k);  // 4^k
    for (uint32_t x = warp; x < n; x += n_warps) {
        DistRow *row = a.rows + x;
        const uint32_t q = row->q, r = row->r;
        const uint64_t ra = __ldg(a.ref_off + r), qa = __ldg(a.q_off + q);
        uint32_t common, denom;
        dist_merge_warp(a.ref_hashes + ra, (uint32_t)(__ldg(a.ref_off + r + 1) - ra), a.q_hashes + qa,
                        (uint32_t)(__ldg(a.q_off + q + 1) - qa), __ldg(a.q_sp + q), lane, common, denom);
        // D2 on the device only to skip p-values: the host decides -d from the exact integers, so a
        // pair is skipped only when it is farther than -d by a margin no rounding difference can cross
        double dist;
        if (common == denom) dist = 0.0;
        else if (common == 0) dist = 1.0;
        else {
            const double jac = (double)common / (double)denom;
            dist = fmin(-log(2.0 * jac / (1.0 + jac)) / (double)a.k, 1.0);
        }
        double p = 1.0;
        if (common != 0) {
            if (dist > a.max_d * (1.0 + 1e-9)) {
                p = -1.0;
            } else {
                // D3, without contractions: the same roundings as Mash's double expression
                const double px = __drcp_rn(__dadd_rn(1.0, kmer_space / (double)__ldg(a.ref_len + r)));
                const double py = __drcp_rn(__dadd_rn(1.0, kmer_space / (double)__ldg(a.q_len + q)));
                const double pxy = __dmul_rn(px, py);
                const double rr = pxy / __dsub_rn(__dadd_rn(px, py), pxy);
                p = binom_upper_tail_warp(common, denom, rr, lane);
            }
        }
        if (lane == 0) {
            row->common = common;
            row->denom = denom;
            row->p = p;
        }
    }
}

uint32_t warp_grid(uint64_t n_warps, int sm_count)
{
    const uint64_t blocks = (n_warps + 7) / 8, cap = (uint64_t)sm_count * 32;
    return (uint32_t)(blocks < 1 ? 1 : blocks > cap ? cap : blocks);
}

}  // namespace

cudaError_t launch_dist_candidates(const DistArgs &a, int sm_count, cudaEvent_t ev_mid, cudaStream_t st)
{
    if (!a.n_q) return cudaSuccess;
    const uint32_t g = warp_grid(a.n_q, sm_count);
    k_dist_mark<<<g, 256, 0, st>>>(a);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    if (ev_mid && (e = cudaEventRecord(ev_mid, st)) != cudaSuccess) return e;
    k_dist_count<<<g, 256, 0, st>>>(a);
    k_dist_scan<<<1, 1024, 0, st>>>(a);
    k_dist_compact<<<g, 256, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_dist_merge(const DistArgs &a, int sm_count, cudaStream_t st)
{
    if (!a.n_q) return cudaSuccess;
    k_dist_merge<<<(uint32_t)sm_count * 16, 256, 0, st>>>(a);
    return cudaGetLastError();
}

}  // namespace hs
