// screen_kernels.cu -- hand-written sm_100a kernels for the `mash screen` hot path.
//
// Path replaced: the streaming loop of `mash screen` (hashSequence + getHash +
// MinHashHeap::tryInsert + hashCounts[key]++), its "Summing shared" / "-w" /
// median / identity / p-value stages, and the hash-table build, i.e. SURVEY.md 8a
// rows a5, a7-a15, for the invocation at /root/reference/scripts/mash.sh:14.
//
//   k_stream        K1+K2(+K3 insert): rolling canonical k-mer -> MurmurHash3 ->
//                   range pre-filter -> 32-byte bucket probe -> warp-aggregated count.
//                   Persistent CTAs; packed tiles arrive through the TMA engine
//                   (1-D cp.async.bulk + mbarrier, double buffered).
//   k_table_insert / k_table_canon   GPU build of the key table (row a5)
//   k_probe         K2 alone (parity + HBM roofline of the random probes)
//   k_mix_*         K3: mixture bottom-s set maintenance
//   k_sort_unique   K3: final ordering of the <= few-thousand candidates
//   k_sketch_reduce K4: shared count + median multiplicity per sketch
//   k_winner        K5: -w reassignment
//   k_stats         K6: identity + binomial upper tail
#include <cuda_runtime.h>
#include <stdint.h>

#include <mutex>
#include <type_traits>

#include "kmer_core.cuh"
#include "screen_kernels.h"

namespace hs {

constexpr int kMaxDevices = 64;

// ---------------------------------------------------------------------------
// PTX: mbarrier + bulk async copy global -> shared (TMA engine; SASS UBLKCP)
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(__cvta_generic_to_global(src)), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
constexpr unsigned kWaitSleepNs = 100;   // between tries of a warp that is ahead of its CTA
__device__ __forceinline__ bool mbar_try(uint64_t *bar, uint32_t phase)
{
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(phase)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t phase)
{
    if (mbar_try(bar, phase)) return;   // the usual case: the tile landed long ago
    // A warp that waits here has run ahead of the slowest warp of its CTA by the whole ring (the tile it wants
    // cannot be issued before its stage is released), so it should get out of the way: spinning on try_wait
    // with a clock read per trip was 3.9 % of all issued warp instructions of the kernel (ncu r02, 13 trips per
    // wait), taken from the issue slots of the very warps it was waiting for.
    for (uint32_t spins = 1;; spins++) {
        __nanosleep(kWaitSleepNs);
        if (mbar_try(bar, phase)) return;
        // a tile that never lands means a broken launch contract: fail loudly, never hang the GPU
        if (spins > (1u << 24)) __trap();
    }
}

__device__ __forceinline__ uint32_t warp_sum(uint32_t v)
{
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

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

// a count left zero: remember which one (SparseState), or note that it wrapped (S8)
__device__ __forceinline__ void count_add(const SparseView &sp, uint32_t *counts, uint32_t id, uint32_t add)
{
    const uint32_t old = atomicAdd(counts + id, add);
    if (sp.touched) {
        if (old == 0u) {
            const uint32_t p = atomicAdd(&sp.st->n_touched, 1u);
            if (p < sp.cap) sp.touched[p] = id;
        } else if (old + add < old) {
            atomicExch(&sp.st->wrapped, 1u);
        }
    }
}

// Warp-cooperative table lookup of NH HASHES PER LANE (K2's "warp-cooperative bucket probe").
// Eight lanes read one 128-byte bucket with one 16-byte load each -- a single coalesced line per
// probe, one L1 wavefront instead of the 32 a per-thread load of a random line costs -- so a warp
// works on four probes per round and needs 8 * NH rounds for its 32 * NH hashes.  ALL rounds' loads
// are issued before the first compare (the kernel waits on HBM latency: lines in flight are what
// counts), and only the LOW WORDS of what came back are kept -- two registers per round -- which is
// all the common case needs: lanes 0-4 of a group hold the ten keys, lane 7 the overflow flag, and a
// round in which no low word matches and no flag is set (nearly all of them) is one vote.  Possible
// matches and overflowed buckets re-read their line (L1/L2 hit) in a warp-uniform slow path that
// compares whole keys and fetches the id from lanes 5-7; a probe whose home bucket overflowed (1.4 %
// at load 0.5) is not chased on the spot by one lane while 31 wait for a DRAM round trip: the warp
// follows all such chains together, four at a time, after the main rounds.
// Must be called by all 32 lanes (convergent).  out[i] = canonical entry id of mine[i] (kNoEntry:
// absent, or want[i] == false); `reads` counts bucket lines read for wanted probes (lane 0 / leaders).
template <int NH>
__device__ __forceinline__ void coop_probe(const TableView &t, const uint64_t (&mine)[NH], const bool (&want)[NH],
                                           uint32_t (&out)[NH], uint32_t &reads)
{
    static_assert(NH >= 1 && NH <= 4, "up to 32 rounds: one bit each in the pending mask");
    constexpr int R = 8 * NH;
    const uint32_t lane = threadIdx.x & 31u, g = lane & 7u, G = lane >> 3, full = 0xffffffffu;
    bool special[NH];
    uint32_t wants[NH], myb[NH], any_want = 0;
#pragma unroll
    for (int i = 0; i < NH; i++) {
        special[i] = want[i] && mine[i] == kEmptyKey;          // never stored in a bucket: answered from the view
        wants[i] = __ballot_sync(full, want[i] && !special[i]);
        any_want |= wants[i];
        out[i] = special[i] ? t.special : kNoEntry;
    }
    if (!any_want) return;                                     // warp-uniform
    // A lane that wants nothing is probed all the same (its bucket index is a valid address whatever its
    // hash holds) and its answer dropped at the end: the rounds below carry no per-lane liveness logic.
#pragma unroll
    for (int i = 0; i < NH; i++) {
        myb[i] = bucket_of(mine[i], t.n_buckets);
        if (lane == 0) reads += (uint32_t)__popc(wants[i]);
    }
    const ulonglong2 *line0 = reinterpret_cast<const ulonglong2 *>(t.buckets) + g;   // this lane's 16 bytes of bucket 0

    uint2 klo[R];                                              // the only per-round state: two registers
#pragma unroll
    for (int r = 0; r < R; r++) {
        const uint32_t b = __shfl_sync(full, myb[r >> 3], (r & 7) * 4 + (int)G);
        const ulonglong2 v = __ldg(line0 + (size_t)b * (kBucketWords / 2));
        klo[r] = make_uint2((uint32_t)v.x, (uint32_t)v.y);
    }

    uint32_t pend = 0;                                         // rounds whose chain goes on (group-uniform)
    // slow path: the whole line of bucket b for the group's probe of hash h -- id if a key matches, overflow flag
    auto resolve = [&](uint32_t b, uint64_t h, bool lv, bool &found, bool &over) -> uint32_t {
        const ulonglong2 v = __ldg(line0 + (size_t)b * (kBucketWords / 2));
        int slot = -1;
        if (lv && g < 5u) {
            if (v.x == h) slot = 2 * (int)g;
            else if (v.y == h) slot = 2 * (int)g + 1;
        }
        const uint32_t m = (__ballot_sync(full, slot >= 0) >> (G * 8u)) & 0xFFu;
        const int kl = m ? __ffs(m) - 1 : 0;
        const uint32_t w32 = (uint32_t)kBucketValWord32 + (uint32_t)__shfl_sync(full, slot, (int)(G * 8u) + kl);
        const uint32_t comp = w32 & 3u;
        const uint32_t pick = comp == 0 ? (uint32_t)v.x : comp == 1 ? (uint32_t)(v.x >> 32)
                            : comp == 2 ? (uint32_t)v.y : (uint32_t)(v.y >> 32);
        const uint32_t id = __shfl_sync(full, pick, (int)(G * 8u + ((w32 >> 2) & 7u)));
        const uint32_t flag = __shfl_sync(full, (uint32_t)v.y, (int)(G * 8u) + 7);   // 32-bit word 30 of the bucket
        over = lv && flag != 0u;               // (the shuffle is unconditional: every lane takes part in it)
        found = m != 0u;
        return id;
    };
    // a group found the id of the probe it handled in round r (r may differ between groups): hand it to the
    // lane that owns the hash -- lane (r & 7) * 4 + G, hash r >> 3 -- right away; nothing is kept per round
    auto deliver = [&](int r, bool found, uint32_t id) {
        const int from = (int)((lane & 3u) * 8u);              // a lane of the group that probed for this lane
        const int fr = __shfl_sync(full, found ? r : -1, from);
        const uint32_t fid = __shfl_sync(full, id, from);
        if (fr >= 0 && (fr & 7) == (int)(lane >> 2)) {
#pragma unroll
            for (int i = 0; i < NH; i++)
                if ((fr >> 3) == i && want[i] && !special[i]) out[i] = fid;
        }
    };

    const bool key_lane = g < 5u, flag_lane = g == 7u;
#pragma unroll
    for (int r = 0; r < R; r++) {
        const int src = (r & 7) * 4 + (int)G;
        const uint32_t hlo = __shfl_sync(full, (uint32_t)mine[r >> 3], src);
        const bool maybe = key_lane ? (klo[r].x == hlo || klo[r].y == hlo) : (flag_lane && klo[r].y != 0u);
        if (__any_sync(full, maybe)) {                          // rare: a key may match, or a bucket overflowed
            const uint64_t h = __shfl_sync(full, mine[r >> 3], src);
            const uint32_t b = __shfl_sync(full, myb[r >> 3], src);
            const bool lv = (wants[r >> 3] >> src) & 1u;
            bool found, over;
            const uint32_t id = resolve(b, h, lv, found, over);
            if (__any_sync(full, found)) deliver(r, found, id);
            if (!found && over) pend |= 1u << r;
        }
    }
    // chains: every group follows its own pending probes, one bucket per trip, all groups in step
    if (__ballot_sync(full, pend != 0u)) {
        int cr = -1;                                           // round being followed by this group (group-uniform)
        uint32_t cstep = 0;                                    // buckets past the home bucket
        for (;;) {
            if (cr < 0 && pend) {
                cr = __ffs(pend) - 1;
                pend &= pend - 1;
                cstep = 1;
            }
            if (!__any_sync(full, cr >= 0)) break;
            const int rr = cr < 0 ? 0 : cr;
            const int src = (rr & 7) * 4 + (int)G;
            uint64_t hh = 0;
            uint32_t hb = 0;
#pragma unroll
            for (int i = 0; i < NH; i++) {                     // (rr >> 3 differs between groups: every lane shuffles every hash)
                const uint64_t x = __shfl_sync(full, mine[i], src);
                const uint32_t y = __shfl_sync(full, myb[i], src);
                if ((rr >> 3) == i) { hh = x; hb = y; }
            }
            uint64_t cb = (uint64_t)hb + cstep;
            if (cb >= t.n_buckets) cb -= t.n_buckets;
            bool found, over;
            const uint32_t id = resolve((uint32_t)cb, hh, cr >= 0, found, over);
            const bool was = cr >= 0;
            if (was && g == 0u) reads++;
            if (__any_sync(full, was && found)) deliver(rr, was && found, id);
            if (was) {
                if (found || !over || cstep + 1 >= t.n_buckets) cr = -1;
                else cstep++;
            }
        }
    }
}

__device__ __forceinline__ void mix_insert(const MixView &m, uint64_t *set, uint64_t h)
{
    if (h == kEmptyKey) { atomicExch(&m.st->has_max, 1u); return; }
    uint32_t slot = mixset_slot(h, m.mask);
    for (uint32_t tries = 0; tries <= m.mask; tries++) {
        unsigned long long cur = __ldcg(reinterpret_cast<const unsigned long long *>(set + slot));
        if (cur == h) return;
        if (cur == kEmptyKey) {
            if (__ldcg(&m.st->count) >= m.limit) { atomicExch(&m.st->overflow, 1u); return; }
            cur = atomicCAS(reinterpret_cast<unsigned long long *>(set + slot), (unsigned long long)kEmptyKey,
                            (unsigned long long)h);
            if (cur == kEmptyKey) { atomicAdd(&m.st->count, 1u); return; }
            if (cur == h) return;
        }
        slot = (slot + 1) & m.mask;
    }
    atomicExch(&m.st->overflow, 1u);
}

// ---------------------------------------------------------------------------
// K1 + K2 (+ K3 insert): the streaming kernel
// ---------------------------------------------------------------------------
struct __align__(16) TileBuf {
    uint64_t seq[kTileWords + 2];  // [1] = halo word, [2..] = the tile
    uint32_t inv[kTileWords + 4];  // [3] = halo word, [4..] = the tile
};
static_assert(sizeof(TileBuf) % 16 == 0, "tile buffers must keep 16-byte alignment");

// Pre-multiplied murmur tables (kmer_core.cuh: hash_canonical_premul): (u64)letters*c1 and
// (u64)letters*c2 for all 256 four-letter words, 8 lane copies each (entry b, copy c at
// b*64 + c*8 bytes) = 16 KB per table, adjacent, at a 16 KB-ALIGNED shared address, so that the
// address of a lookup is
//     (index byte << 6, taken from the k-mer with one shift and the AND below) | (table base | (lane & 7) * 8)
// i.e. one shift + one LOP3 instead of shift/and/or/lea -- the kernel is ALU-pipe bound (ncu).  A
// half-warp's 64-bit loads touch each bank pair once per copy; two lanes share a copy (2-way conflict
// when their entries differ in parity).  The second table is reached through the load's immediate
// offset.  (First version: a 16-copy table of the ASCII letters and the multiply done in registers.)
constexpr uint32_t kLutBytes = 16384;   // alignment and size of one table
constexpr uint32_t kPreBytes = 256 * 8 * 8;
static_assert(kPreBytes == 16384 && kPreBytes == kLutBytes, "SmemPremul's loads carry this offset as an immediate");
constexpr uint32_t kTailBytes = 8192;   // 4^5 finished tail terms (kmer_core.cuh: tail_entry), right behind the two tables
template <bool TAIL>
struct SmemPremul {
    static constexpr bool kTail = TAIL;
    uint32_t base;  // table address | (lane & 7) * 8
    uint32_t k64;   // the constant 64 in a register the compiler cannot see through (below)
    uint32_t lut;   // table address alone (16 KB aligned): the tail table has no lane copies
    // finished tail term of a top-aligned k-mer: one shift, one AND-OR, one 64-bit load
    __device__ __forceinline__ uint64_t tail(uint64_t ct, int k) const
    {
        const int r = k & 15;
        const uint32_t w = (k >> 4) ? (uint32_t)ct : (uint32_t)(ct >> 32);
        const uint32_t addr = ((w >> (29 - 2 * r)) & (((1u << (2 * r)) - 1u) << 3)) | lut;
        uint64_t v;
        asm("ld.shared.u64 %0, [%1+32768];" : "=l"(v) : "r"(addr));
        return v;
    }
    // Address of word i's entry.  The index byte sits on a byte boundary of the top-aligned k-mer, so it
    // is ONE byte permute (ALU pipe) and ONE multiply-add by 64 (FMA pipe) instead of a shift and a
    // three-input logic op (two ALU-pipe instructions): the kernel is bound by the half-rate ALU pipe
    // (ncu: 74 % busy) while the FMA pipe idles at 26 %.  A multiplier the compiler could see would be
    // strength-reduced back to a shift/LEA on the ALU pipe.  Partial last words keep the masked form.
    __device__ __forceinline__ uint32_t where(uint64_t ct, int i, int k) const
    {
        if (k - 4 * i >= 4) {
            const uint32_t w = i < 4 ? (uint32_t)(ct >> 32) : (uint32_t)ct;
            const uint32_t byte = __byte_perm(w, 0u, 0x4440u + (uint32_t)(3 - (i & 3)));
            uint32_t addr;
            asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(addr) : "r"(byte), "r"(k64), "r"(base));
            return addr;
        }
        return top_word_index64(ct, i, k) | base;
    }
    __device__ __forceinline__ uint64_t full(uint32_t addr, bool second) const
    {
        uint64_t v;
        if (second) asm("ld.shared.u64 %0, [%1+16384];" : "=l"(v) : "r"(addr));
        else asm("ld.shared.u64 %0, [%1];" : "=l"(v) : "r"(addr));
        return v;
    }
    __device__ __forceinline__ uint32_t low(uint32_t addr, bool second) const
    {
        uint32_t v;
        if (second) asm("ld.shared.u32 %0, [%1+16384];" : "=r"(v) : "r"(addr));
        else asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
        return v;
    }
};

constexpr int kMinCtas = 4;   // 48 KB of shared memory per CTA
// compile-time k with a 1..5 letter tail (k = 21): the tail term comes from its own table.  It takes 8 KB
// from the L1 of every CTA, so the probe-everything kernel (MODE 3), which lives on L1/L2 traffic, goes without
__host__ __device__ constexpr bool stream_tail_table(int kt, int mode)
{
    return mode != 3 && kt > 0 && (kt & 15) >= 1 && (kt & 15) <= 5;
}
constexpr int kIlp = 4;   // k-mers hashed side by side per thread (measured, ms per Gbp: 1: 5.33, 2: 5.02, 4: 4.83, 8: 6.47)

// MODE: 0 = screen, 1 = K1 parity (emit every hash), 2 = screen with the Bloom reads of a group of
// kIlp k-mers issued together (databases with keys above the dense range), 3 = screen that probes for
// (nearly) every k-mer: the warp looks its hashes up cooperatively (coop_probe), control flow stays
// warp-uniform and the CTA may use twice the registers (the kernel waits on HBM, not on issue slots)
template <int KT, int MODE>
__global__ void __launch_bounds__(kCtaThreads, MODE == 3 ? 3 : kMinCtas) k_stream(const StreamArgs a)
{
    constexpr bool EMIT = MODE == 1, BLOOMB = MODE == 2, COOP = MODE == 3;
    constexpr bool kTailTab = stream_tail_table(KT, MODE);
    // kStages tile buffers, filled kPrefetch tiles ahead through the TMA engine.
    // full[s]: the bytes of stage s have landed; empty[s]: all 8 warps copied their words of
    // stage s to registers.  No CTA-wide barrier in the loop: warps drift up to two tiles
    // apart (ncu r01: 12 % of warp time sat in __syncthreads with the 2-stage version).
    // WHO issues a tile: whichever warp gets to an iteration first claims the outstanding tile
    // ordinals (issue_next, compare-and-swap) and issues them.  Round 1 left that to thread 0 with one
    // tile of look-ahead; warp 0 also does its share of the hashing, so it was usually BEHIND the others,
    // which then spun on `full` for a tile nobody had asked for yet -- 7 % of all issued instructions
    // were that spin (ncu r02: 35 try_wait per wait).
    // (Measured alternative: a ring PER WARP -- every warp streams its own 32-word slices and refills them itself,
    // nothing shared, no warp ever waits for another.  With the shared ring the leading warps sleep 15 % of their
    // time at the ring's end (32 sleep-and-retry trips per tile wait); with private rings nobody waits -- and the
    // kernel is no faster: 4.43 vs 4.40 ms per Gbp, 6.22 vs 6.18 on the Bloom tier, 5.24 vs 5.21 at k = 31.  The
    // other three CTAs of the SM fill the sleepers' issue slots; the limit is the ALU pipe, not the number of
    // warps awake.)
    constexpr uint32_t kStages = 4, kPrefetch = 2;
    __shared__ TileBuf buf[kStages];
    __shared__ __align__(8) uint64_t full[kStages], empty[kStages];
    __shared__ uint32_t issue_next;   // ordinal (iteration index of this CTA) of the next tile nobody has issued
    extern __shared__ __align__(16) uint8_t dyn_smem[];  // 2 * kLutBytes: room to align the table to 16 KB

    const int k = KT ? KT : a.k;
    const bool use64 = KT ? (KT > 16) : (a.use64 != 0);
    const uint32_t tid = threadIdx.x, lane = tid & 31;

    if (tid == 0) {
        for (uint32_t i = 0; i < kStages; i++) {
            mbar_init(&full[i], 1);
            mbar_init(&empty[i], kCtaThreads / 32);
        }
        issue_next = kPrefetch;   // the prologue below issues ordinals 0 .. kPrefetch-1
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    const uint32_t dyn_addr = smem_u32(dyn_smem);
    const uint32_t lut_addr = (dyn_addr + (kLutBytes - 1)) & ~(kLutBytes - 1);
    {
        uint32_t dyn_size;
        asm("mov.u32 %0, %%dynamic_smem_size;" : "=r"(dyn_size));
        if (lut_addr + 2 * kPreBytes + (kTailTab ? kTailBytes : 0u) > dyn_addr + dyn_size) __trap();  // launch did not leave room for the aligned tables
        uint64_t *t = reinterpret_cast<uint64_t *>(dyn_smem + (lut_addr - dyn_addr));
        for (uint32_t i = tid; i < 2 * 256 * 8; i += kCtaThreads) t[i] = premul_entry_msb((i >> 3) & 255u, i >= 256 * 8);
        if (kTailTab)
            for (uint32_t i = tid; i < (1u << (2 * (KT & 15))); i += kCtaThreads) t[2 * 256 * 8 + i] = tail_entry(i, KT & 15);
    }
    __syncthreads();
    uint32_t lut_lane = lut_addr | ((lane & 7u) << 3);
    asm volatile("mov.u32 %0, %0;" : "+r"(lut_lane));  // one opaque per-thread register: keeps ptxas from
                                                        // splitting it back into uniform base + lane term
    uint32_t k64 = 64u;
    asm volatile("mov.u32 %0, %0;" : "+r"(k64));
    const SmemPremul<kTailTab> L{lut_lane, k64, lut_addr};

    auto issue = [&](uint32_t tile, uint32_t b) {
        // tile 0 has no halo (positions before the chunk do not exist)
        const uint32_t sw = tile ? 2u : 0u, iw = tile ? 4u : 0u;
        const uint32_t sbytes = (kTileWords + sw) * 8u, ibytes = (kTileWords + iw) * 4u;
        mbar_expect_tx(&full[b], sbytes + ibytes);
        bulk_g2s(&buf[b].seq[2 - sw], a.seq + (size_t)tile * kTileWords - sw, sbytes, &full[b]);
        bulk_g2s(&buf[b].inv[4 - iw], a.inv + (size_t)tile * kTileWords - iw, ibytes, &full[b]);
    };

    // mixture threshold and live set come from device state (maintained between launches)
    uint64_t mix_tau = 0;
    uint64_t *mix_set = nullptr;
    if (a.do_mix) {
        const unsigned long long t = __ldcg(&a.mix.st->tau);
        mix_tau = t < a.mix.tau_cap ? t : a.mix.tau_cap;
        mix_set = a.mix.sets[__ldcg(&a.mix.st->cur) & 1u];
    }

    const uint64_t n_bases = a.n_bases_dev ? (uint64_t)__ldcg(a.n_bases_dev) : a.n_bases;
    // one compare per k-mer decides whether anything at all has to happen with its hash
    uint64_t gate = a.do_mix ? mix_tau : 0;
    if (a.do_count) gate = a.do_filter ? (a.tab.max_key > gate ? a.tab.max_key : gate) : ~0ull;
    if (EMIT) gate = ~0ull;   // K1 parity runs want every hash
    const uint32_t gate_hi = (uint32_t)(gate >> 32);
    // Bloom-tier instantiation: hashes <= lowgate are handled without the filter (direct probe, mixture insert)
    const uint64_t lowgate = a.do_mix ? (mix_tau > a.tab.dense_max ? mix_tau : a.tab.dense_max) : a.tab.dense_max;
    [[maybe_unused]] const uint32_t lowgate_hi = (uint32_t)(lowgate >> 32), max_hi = (uint32_t)(a.tab.max_key >> 32);
    uint32_t n_valid = 0, n_probe = 0, n_reads = 0, n_hits = 0, n_mix = 0;
    uint32_t tile = a.tile_begin + blockIdx.x, it = 0;
    if (tid == 0)
        for (uint32_t p = 0; p < kPrefetch; p++)
            if ((uint64_t)tile + (uint64_t)p * gridDim.x < a.n_tiles) issue(tile + p * gridDim.x, p);

    for (; tile < a.n_tiles; tile += gridDim.x, it++) {
        if (lane == 0) {
            // Ordinals up to it + kPrefetch should be on their way; claim the ones that are not.  The tile this
            // warp is about to wait for (ordinal it) MUST be issued, so for it the stage's release is waited
            // for; look-ahead tiles are only taken when their stage is already free -- otherwise the warp goes
            // on hashing and whoever comes by next tries again (round 2, first form: the fastest warp span
            // here for the slowest one, 4 % of all issued instructions).
            for (;;) {
                const uint32_t nt = *reinterpret_cast<volatile uint32_t *>(&issue_next);
                const uint64_t ntile = (uint64_t)a.tile_begin + blockIdx.x + (uint64_t)nt * gridDim.x;
                if (nt > it + kPrefetch || ntile >= a.n_tiles) break;
                const uint32_t sb = nt % kStages;
                const uint32_t par = ((nt / kStages) - 1u) & 1u;   // parity of the phase that frees the stage (ordinal nt - kStages consumed by all)
                if (nt > it && nt >= kStages && !mbar_try(&empty[sb], par)) break;
                if (atomicCAS(&issue_next, nt, nt + 1u) != nt) continue;      // another warp took it
                if (nt >= kStages) mbar_wait(&empty[sb], par);
                issue((uint32_t)ntile, sb);
            }
        }
        const uint32_t b = it % kStages;
        mbar_wait(&full[b], (it / kStages) & 1u);
        uint64_t cur = buf[b].seq[tid + 2], prev = buf[b].seq[tid + 1];
        uint32_t icur = buf[b].inv[tid + 4], iprev = buf[b].inv[tid + 3];
        // Handing the stage back is a write-after-read hazard ACROSS PROXIES: these were generic-proxy
        // reads (LDS), the refill is an async-proxy write (TMA).  The mbarrier arrive alone does not
        // order the two: with the load/store pipe backed up by table probes, about one word per 1e9
        // was read after the TMA engine had refilled the stage (found as +-1 differences in per-hash
        // counts between filter modes; 10/10 runs deterministic with the proxy fence, 9/10 with a
        // CTA memory fence only).  So: retire the loads, fence the proxies, then release.
        __threadfence_block();
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[b]);  // this warp holds its words: the stage may be refilled

        if (tile == 0 && tid == 0) { prev = 0; iprev = ~0u; }
        const uint64_t pos0 = ((uint64_t)tile * kTileWords + tid) * kBasesPerWord;
        if (pos0 + kBasesPerWord > n_bases) {
            const uint32_t nv = pos0 >= n_bases ? 0u : (uint32_t)(n_bases - pos0);
            icur |= nv ? ((1u << (32 - nv)) - 1u) : ~0u;
        }
        if (!COOP && icur == ~0u) continue;  // padding / all-N word: no k-mer ends here (COOP: every lane stays for the warp's lookups)

        auto sink = [&](int j, uint64_t h, uint32_t bloom_word) {
            if (EMIT) {
                a.emit_hash[pos0 + j] = h;
                a.emit_valid[pos0 + j] = 1;
            }
            if (a.do_mix && h <= mix_tau) {
                n_mix++;
                mix_insert(a.mix, mix_set, h);
            }
            if (a.do_count && (!a.do_filter || h <= a.tab.max_key)) {
                // second tier (exact: no false negatives); only MODE 2 runs with one, its words read in word()
                if (BLOOMB && a.do_filter && a.tab.bloom && h > a.tab.dense_max) {
                    uint32_t bw, bb;
                    bloom_slot(h, a.tab.bloom_mask, use64, bw, bb);
                    if ((bloom_word & bb) != bb) return;
                }
                n_probe++;
                const uint32_t id = table_find<true>(a.tab, h, n_reads);
                if (id != kNoEntry) {
                    // warp-aggregated count: lanes that hit the same key add once
                    const uint32_t peers = __match_any_sync(__activemask(), id);
                    if ((uint32_t)(__ffs(peers) - 1) == lane) count_add(a.sparse, a.counts, id, (uint32_t)__popc(peers));
                    n_hits++;
                }
            }
        };
        // kIlp k-mers per trip: their hashes are computed unconditionally (invalid k-mers are rare) and
        // independently, so the scheduler can interleave the multiply chains; validity and the gate
        // are looked at afterwards.
        const uint32_t ok = ~invalid_kmer_ends(iprev, icur, k);
        n_valid += (uint32_t)__popc(ok);
        const Win w = win_init_top(prev, cur, k);
        // words whose 32 k-mers are all valid (nearly all of them) run a copy of the loop that never
        // looks at the validity mask
        // (measured dead ends, ms per Gbp at kIlp = 4: compile-time halves + a one-word gate pre-compare
        // 6.22, the rare path as a __noinline__ function 5.08, this form 4.83 -- more copies of the
        // loop and call conventions cost more than the few selects they remove)
        auto word = [&](auto check) {
#pragma unroll 1
            for (int half = 0; half < 2; half++) {
                const uint32_t fa = half ? w.f0 : w.f1, fb = half ? w.f1 : w.f2, fc = half ? w.f2 : w.f3;
                const uint32_t ra = half ? w.r1 : w.r0, rb = half ? w.r2 : w.r1, rc = half ? w.r3 : w.r2;
#pragma unroll 1
                for (int q = 0; q < 16; q += kIlp) {
                    uint64_t h[kIlp];
#pragma unroll
                    for (int u = 0; u < kIlp; u++)
                        h[u] = hash_canonical_premul_top(canonical_top_half(fa, fb, fc, ra, rb, rc, q + u), k, a.seed, use64, L);
                    uint32_t pre[kIlp], bbits[kIlp];
#pragma unroll
                    for (int u = 0; u < kIlp; u++) {
                        pre[u] = ~0u; bbits[u] = 0u;
                        if (BLOOMB) {   // all kIlp reads are issued before the first one is looked at
                            uint32_t bw;
                            bloom_slot(h[u], a.tab.bloom_mask, use64, bw, bbits[u]);
                            pre[u] = 0u;                               // fails the test below: bbits is never 0
                            // (high words only: a superset of h <= max_key, and the word index is masked into range).
                            // Read through L2 only: with the filter words out of L1 the tail-term table pays in
                            // this instantiation too (tiny-genome DB: 6.30 -> 6.18 ms; with __ldg 6.50)
                            if ((uint32_t)(h[u] >> 32) <= max_hi) pre[u] = __ldcg(a.tab.bloom + bw);
                        }
                    }
                    if (COOP) {
                        bool valid[kIlp];
#pragma unroll
                        for (int u = 0; u < kIlp; u++) {
                            const int j = half * 16 + q + u;
                            valid[u] = (ok >> (31 - j)) & 1u;
                            if (valid[u] && a.do_mix && h[u] <= mix_tau) {
                                n_mix++;
                                mix_insert(a.mix, mix_set, h[u]);
                            }
                        }
                        static_assert(kIlp % 2 == 0, "the cooperative lookup takes the k-mers two at a time");
                        // (Measured dead end: requesting all 128 home buckets of the trip with prefetch.global.L2 before
                        // the first cooperative round -- no registers, the second pair of lookups would find its lines in
                        // L2 -- made the kernel 1.5x SLOWER, 37.8 -> 55.8 ms per Gbp.  So did software pipelining --
                        // request a pair's lines, hash the next pair, then look: the flight's state (16 x 2 registers
                        // + hashes + buckets) went to local memory at 120 registers, 2 CTAs per SM: 81 ms.)
#pragma unroll
                        for (int u = 0; u < kIlp; u += 2) {     // all 32 lanes, every trip: 64 probes, 16 lines in flight per lane
                            const uint64_t hh[2] = {h[u], h[u + 1]};
                            const bool want[2] = {valid[u] && a.do_count && (!a.do_filter || h[u] <= a.tab.max_key),
                                                  valid[u + 1] && a.do_count && (!a.do_filter || h[u + 1] <= a.tab.max_key)};
                            uint32_t id[2];
                            n_probe += (uint32_t)want[0] + (uint32_t)want[1];
                            coop_probe<2>(a.tab, hh, want, id, n_reads);
#pragma unroll
                            for (int w2 = 0; w2 < 2; w2++)
                                if (id[w2] != kNoEntry) {
                                    const uint32_t peers = __match_any_sync(__activemask(), id[w2]);
                                    if ((uint32_t)(__ffs(peers) - 1) == lane) count_add(a.sparse, a.counts, id[w2], (uint32_t)__popc(peers));
                                    n_hits++;
                                }
                        }
                    } else if (BLOOMB) {
                        // Most k-mers of a run against such a database lie in the Bloom tier's range and are
                        // turned away by it: that decision must cost a handful of instructions, so the sink
                        // (mixture insert, direct probe, the tier's own re-check) is entered only below the
                        // low gate or when the filter word really has the three bits.
#pragma unroll
                        for (int u = 0; u < kIlp; u++) {
                            const int j = half * 16 + q + u;
                            // (high word of the low gate: a superset; the sink repeats every test exactly)
                            const bool enter = (uint32_t)(h[u] >> 32) <= lowgate_hi || (pre[u] & bbits[u]) == bbits[u];
                            if (enter && (!decltype(check)::value || ((ok >> (31 - j)) & 1u))) sink(j, h[u], pre[u]);
                        }
                    } else {
#pragma unroll
                        for (int u = 0; u < kIlp; u++) {
                            const int j = half * 16 + q + u;
                            // high words first: one compare turns away all but ~1 k-mer in a thousand
                            if ((uint32_t)(h[u] >> 32) <= gate_hi)
                                if (h[u] <= gate && (!decltype(check)::value || ((ok >> (31 - j)) & 1u))) sink(j, h[u], pre[u]);
                        }
                    }
                }
            }
        };
        if (!COOP && ok == ~0u) word(std::false_type{}); else word(std::true_type{});
    }

    n_valid = warp_sum(n_valid); n_probe = warp_sum(n_probe); n_reads = warp_sum(n_reads);
    n_hits = warp_sum(n_hits); n_mix = warp_sum(n_mix);
    if (lane == 0) {
        if (n_valid) atomicAdd(a.stats + ST_VALID, (unsigned long long)n_valid);
        if (n_probe) atomicAdd(a.stats + ST_PROBES, (unsigned long long)n_probe);
        if (n_reads) atomicAdd(a.stats + ST_BUCKETS, (unsigned long long)n_reads);
        if (n_hits) atomicAdd(a.stats + ST_HITS, (unsigned long long)n_hits);
        if (n_mix) atomicAdd(a.stats + ST_MIXINS, (unsigned long long)n_mix);
    }
}

template <int KT, int MODE>
static cudaError_t launch_stream_t(const StreamArgs &a, int sm_count, cudaStream_t st)
{
    // per device: function attributes belong to the context, and one process may drive several GPUs
    static std::mutex mu;
    static int occ_dev[kMaxDevices] = {0};
    static uint32_t dyn_dev[kMaxDevices] = {0};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= kMaxDevices) return cudaErrorInvalidDevice;
    int occ;
    uint32_t dyn;
    {
        std::lock_guard<std::mutex> lk(mu);
        if (!occ_dev[dev]) {
            // the tables need a 16 KB-aligned 32 KB window.  Dynamic shared memory starts right after the
            // 1 KB the system reserves per CTA and the kernel's static buffers, so ask for exactly the
            // distance to the next 16 KB boundary plus the tables (the kernel traps if that ever stops
            // being true): 4 CTAs of 48 KB per SM instead of 3 with a full 16 KB of slack.
            cudaFuncAttributes fa;
            if ((e = cudaFuncGetAttributes(&fa, k_stream<KT, MODE>)) != cudaSuccess) return e;
            const uint32_t start = 1024u + (((uint32_t)fa.sharedSizeBytes + 15u) & ~15u);
            const uint32_t d = (((start + kLutBytes - 1) & ~(kLutBytes - 1)) - start) + 2 * kPreBytes +
                               (stream_tail_table(KT, MODE) ? kTailBytes : 0u);
            if ((e = cudaFuncSetAttribute(k_stream<KT, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)d)) != cudaSuccess) return e;
            int o = 0;
            e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, k_stream<KT, MODE>, kCtaThreads, d);
            if (e != cudaSuccess) return e;
            dyn_dev[dev] = d;
            occ_dev[dev] = o < 1 ? 1 : o;
        }
        occ = occ_dev[dev];
        dyn = dyn_dev[dev];
    }
    uint32_t grid = (uint32_t)sm_count * (uint32_t)occ;
    if (grid > a.n_tiles - a.tile_begin) grid = a.n_tiles - a.tile_begin;
    if (!grid) return cudaSuccess;
    k_stream<KT, MODE><<<grid, kCtaThreads, dyn, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_stream(const StreamArgs &a, int sm_count, cudaStream_t st)
{
    if (a.emit_hash) return launch_stream_t<0, 1>(a, sm_count, st);   // parity runs: generic-k instantiation
    if (a.probe_all && a.do_count) {
        switch (a.k) {
        case 21: return launch_stream_t<21, 3>(a, sm_count, st);
        case 31: return launch_stream_t<31, 3>(a, sm_count, st);
        default: return launch_stream_t<0, 3>(a, sm_count, st);
        }
    }
    if (a.do_count && a.do_filter && a.tab.bloom) {
        switch (a.k) {
        case 21: return launch_stream_t<21, 2>(a, sm_count, st);
        case 31: return launch_stream_t<31, 2>(a, sm_count, st);
        default: return launch_stream_t<0, 2>(a, sm_count, st);
        }
    }
    switch (a.k) {
    case 21: return launch_stream_t<21, 0>(a, sm_count, st);
    case 31: return launch_stream_t<31, 0>(a, sm_count, st);
    case 16: return launch_stream_t<16, 0>(a, sm_count, st);
    default: return launch_stream_t<0, 0>(a, sm_count, st);
    }
}

// ---------------------------------------------------------------------------
// Table build (row a5) and standalone probe (K2)
// ---------------------------------------------------------------------------
__global__ void k_table_init(uint64_t *buckets, uint64_t n_words)
{   // keys and ids all-ones (free slot / identity of atomicMin), overflow flag + pad zero
    for (uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; w < n_words; w += (uint64_t)gridDim.x * blockDim.x)
        buckets[w] = (w & (kBucketWords - 1)) == kBucketWords - 1 ? 0ull : ~0ull;
}

__global__ void k_table_insert(uint64_t *buckets, uint32_t n_buckets, const uint64_t *hashes, uint64_t n,
                               uint32_t *special, uint32_t *fail)
{
    for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t h = hashes[e];
        if (h == kEmptyKey) { atomicMin(special, (uint32_t)e); continue; }
        uint32_t b = bucket_of(h, n_buckets);
        bool done = false;
        for (uint32_t tries = 0; tries < n_buckets && !done; tries++) {
            uint64_t *kb = buckets + (size_t)b * kBucketWords;
            uint32_t *b32 = reinterpret_cast<uint32_t *>(kb);
#pragma unroll 1
            for (int s = 0; s < kBucketSlots && !done; s++) {
                unsigned long long cur = __ldcg(reinterpret_cast<const unsigned long long *>(kb + s));
                if (cur == kEmptyKey) {
                    cur = atomicCAS(reinterpret_cast<unsigned long long *>(kb + s), (unsigned long long)kEmptyKey,
                                    (unsigned long long)h);
                    if (cur == kEmptyKey) cur = h;
                }
                if (cur == h) {
                    // canonical id of a key = smallest entry index holding it: identical on
                    // every GPU whatever the insertion order, so counts[] all-reduce cleanly
                    atomicMin(b32 + kBucketValWord32 + s, (uint32_t)e);
                    done = true;
                }
            }
            if (!done) {   // full of other keys: this key moves on, and lookups must follow
                atomicExch(b32 + kBucketOverWord32, 1u);
                b = (b + 1 == n_buckets) ? 0u : b + 1;
            }
        }
        if (!done) atomicExch(fail, 1u);
    }
}

__global__ void k_bloom_build(uint32_t *bloom, uint32_t bloom_mask, uint64_t dense_max, bool use64,
                              const uint64_t *hashes, uint64_t n)
{
    for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t h = hashes[e];
        if (h <= dense_max) continue;   // probed directly
        uint32_t w, b;
        bloom_slot(h, bloom_mask, use64, w, b);
        atomicOr(bloom + w, b);
    }
}

__global__ void k_table_canon(const TableView t, const uint64_t *hashes, uint64_t n, uint32_t *canon, uint32_t *next,
                              unsigned long long *n_distinct)
{
    uint32_t local = 0, dummy = 0;
    for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t id = table_find<false>(t, hashes[e], dummy);
        canon[e] = id;
        // the inverted index (hash -> references that hold it, SURVEY.md 7.2) as a chain through the
        // entries: the canonical entry is the head, every other holder pushes itself behind it
        if (id != (uint32_t)e) next[e] = atomicExch(next + id, (uint32_t)e);
        local += id == (uint32_t)e;
    }
    local = warp_sum(local);
    if ((threadIdx.x & 31) == 0 && local) atomicAdd(n_distinct, (unsigned long long)local);
}

// K2 alone: two hashes per lane (64 probes per warp and trip, 16 lines in flight per lane).
constexpr int kProbeNH = 2;
__global__ void __launch_bounds__(128, 6) k_probe(const TableView t, const uint64_t *hashes, uint64_t n,
                                                  uint32_t *out_entry, unsigned long long *stats)
{
    const uint32_t lane = threadIdx.x & 31u;
    uint32_t hits = 0, reads = 0;
    const uint64_t warp = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint64_t n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t base = warp * (32 * kProbeNH); base < n; base += n_warps * (32 * kProbeNH)) {
        uint64_t mine[kProbeNH];
        bool have[kProbeNH];
        uint32_t id[kProbeNH];
#pragma unroll
        for (int i = 0; i < kProbeNH; i++) {
            have[i] = base + 32 * i + lane < n;
            mine[i] = have[i] ? __ldg(hashes + base + 32 * i + lane) : 0ull;
        }
        coop_probe<kProbeNH>(t, mine, have, id, reads);
#pragma unroll
        for (int i = 0; i < kProbeNH; i++)
            if (have[i]) {
                if (out_entry) out_entry[base + 32 * i + lane] = id[i];
                hits += id[i] != kNoEntry;
            }
    }
    hits = warp_sum(hits); reads = warp_sum(reads);
    if (lane == 0) {
        if (hits) atomicAdd(stats + 0, (unsigned long long)hits);
        if (reads) atomicAdd(stats + 1, (unsigned long long)reads);
    }
}

// Reference point for K2: the rate at which this GPU serves independent random 32-byte
// sector reads from a buffer far larger than L2 (no hashing, no compares, 8 loads in flight
// per thread).  k_probe is reported against this as well as against the streaming peak.
__global__ void __launch_bounds__(256) k_gather_bench(const ulonglong2 *buf, uint64_t n_sectors, uint64_t per_thread,
                                                      unsigned long long *sink)
{
    uint64_t x = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) * 0x9E3779B97F4A7C15ull + 0x1234567ull;
    unsigned long long acc = 0;
    for (uint64_t i = 0; i < per_thread; i += 8) {
        ulonglong2 v[16];
#pragma unroll
        for (int u = 0; u < 8; u++) {
            x = x * 6364136223846793005ull + 1442695040888963407ull;
            const uint64_t sct = (uint64_t)(((unsigned __int128)(x >> 11) * n_sectors) >> 53);
            v[2 * u] = __ldg(buf + 2 * sct); v[2 * u + 1] = __ldg(buf + 2 * sct + 1);
        }
#pragma unroll
        for (int u = 0; u < 16; u++) acc += v[u].x ^ v[u].y;
    }
    if (acc == 0x0123456789ABCDEFull) *sink = acc;  // keeps the loads alive
}

cudaError_t launch_gather_bench(const void *buf, uint64_t bytes, uint64_t total_reads, int sm_count, cudaStream_t st)
{
    const uint32_t grid = (uint32_t)sm_count * 8u;
    const uint64_t per_thread = (total_reads / ((uint64_t)grid * 256) + 7) / 8 * 8;
    static unsigned long long *sink = nullptr;
    if (!sink) { cudaError_t e = cudaMalloc((void **)&sink, 8); if (e != cudaSuccess) return e; }
    k_gather_bench<<<grid, 256, 0, st>>>((const ulonglong2 *)buf, bytes / 32, per_thread, sink);
    return cudaGetLastError();
}

static inline uint32_t grid_for(uint64_t n, int threads, uint32_t cap)
{
    uint64_t g = (n + threads - 1) / threads;
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (uint32_t)g;
}

cudaError_t launch_table_insert(uint64_t *buckets, uint32_t n_buckets, const uint64_t *hashes, uint64_t n_entries,
                                uint32_t *special, uint32_t *fail, cudaStream_t st)
{
    const uint64_t words = (uint64_t)n_buckets * kBucketWords;
    k_table_init<<<grid_for(words, 256, 148 * 32), 256, 0, st>>>(buckets, words);
    if (!n_entries) return cudaGetLastError();
    k_table_insert<<<grid_for(n_entries, 256, 148 * 32), 256, 0, st>>>(buckets, n_buckets, hashes, n_entries, special, fail);
    return cudaGetLastError();
}

cudaError_t launch_bloom_build(uint32_t *bloom, uint32_t bloom_mask, uint64_t dense_max, bool use64,
                               const uint64_t *hashes, uint64_t n, cudaStream_t st)
{
    if (!n) return cudaSuccess;
    k_bloom_build<<<grid_for(n, 256, 148 * 32), 256, 0, st>>>(bloom, bloom_mask, dense_max, use64, hashes, n);
    return cudaGetLastError();
}

cudaError_t launch_table_canon(const TableView &t, const uint64_t *hashes, uint64_t n_entries, uint32_t *canon,
                               uint32_t *next, unsigned long long *n_distinct, cudaStream_t st)
{
    if (!n_entries) return cudaSuccess;
    k_table_canon<<<grid_for(n_entries, 256, 148 * 32), 256, 0, st>>>(t, hashes, n_entries, canon, next, n_distinct);
    return cudaGetLastError();
}

cudaError_t launch_probe(const TableView &t, const uint64_t *hashes, uint64_t n, uint32_t *out_entry,
                         unsigned long long *stats, int sm_count, cudaStream_t st)
{
    if (!n) return cudaSuccess;
    k_probe<<<grid_for((n + kProbeNH - 1) / kProbeNH, 128, (uint32_t)sm_count * 24u), 128, 0, st>>>(t, hashes, n, out_entry, stats);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// K3: mixture bottom-s set
// ---------------------------------------------------------------------------
__global__ void k_mix_collect(const uint64_t *set, uint32_t cap, uint64_t thr, uint64_t *out, uint32_t out_cap,
                              uint32_t *n_out)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < cap; i += gridDim.x * blockDim.x) {
        const uint64_t v = set[i];
        if (v != kEmptyKey && v <= thr) {
            const uint32_t p = atomicAdd(n_out, 1u);
            if (p < out_cap) out[p] = v;
        }
    }
}

// ---- maintenance after every streaming launch (no host involvement) ----------
__device__ __forceinline__ bool mix_needs_shrink(const MixView &v, unsigned long long &t)
{
    const MixState *st = v.st;
    t = st->tau < v.tau_cap ? st->tau : v.tau_cap;
    return !st->overflow && st->count > (v.mask + 1u) / 4u && (t >> 2) > 0;
}

__global__ void k_mix_clear_cond(const MixView v)
{
    unsigned long long t;
    if (!mix_needs_shrink(v, t)) return;
    uint64_t *dst = v.sets[(v.st->cur & 1u) ^ 1u];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i <= v.mask; i += gridDim.x * blockDim.x) dst[i] = kEmptyKey;
}

__global__ void k_mix_rebuild_cond(const MixView v)
{
    unsigned long long t;
    if (!mix_needs_shrink(v, t)) return;
    const uint64_t thr = t >> 2;
    const uint64_t *src = v.sets[v.st->cur & 1u];
    uint64_t *dst = v.sets[(v.st->cur & 1u) ^ 1u];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i <= v.mask; i += gridDim.x * blockDim.x) {
        const uint64_t x = src[i];
        if (x == kEmptyKey || x > thr) continue;
        uint32_t slot = mixset_slot(x, v.mask);
        for (;;) {
            const unsigned long long cur = atomicCAS(reinterpret_cast<unsigned long long *>(dst + slot),
                                                     (unsigned long long)kEmptyKey, (unsigned long long)x);
            if (cur == kEmptyKey) { atomicAdd(&v.st->new_count, 1u); break; }
            slot = (slot + 1) & v.mask;
        }
    }
}

__global__ void k_mix_apply(const MixView v)
{
    unsigned long long t;
    const bool shrink = mix_needs_shrink(v, t);
    MixState *st = v.st;
    if (shrink) {
        st->tau = t >> 2;
        st->cur = (st->cur & 1u) ^ 1u;
        st->count = st->new_count;
        st->rebuilds++;
    } else {
        st->tau = t;
    }
    st->new_count = 0;
}

__global__ void k_mix_state_init(MixState *st, unsigned long long tau)
{
    MixState z;
    memset(&z, 0, sizeof z);
    z.tau = tau;
    *st = z;
}
cudaError_t launch_mix_state_init(MixState *st, uint64_t tau, cudaStream_t stm)
{
    k_mix_state_init<<<1, 1, 0, stm>>>(st, (unsigned long long)tau);
    return cudaGetLastError();
}

cudaError_t launch_mix_collect(const uint64_t *set, uint32_t cap, uint64_t thr, uint64_t *out, uint32_t out_cap,
                               uint32_t *n_out, cudaStream_t st)
{
    k_mix_collect<<<grid_for(cap, 256, 148 * 8), 256, 0, st>>>(set, cap, thr, out, out_cap, n_out);
    return cudaGetLastError();
}
cudaError_t launch_mix_maintain(const MixView &v, cudaStream_t st)
{
    const uint32_t cap = v.mask + 1u;
    k_mix_clear_cond<<<grid_for(cap, 256, 148 * 4), 256, 0, st>>>(v);
    k_mix_rebuild_cond<<<grid_for(cap, 256, 148 * 4), 256, 0, st>>>(v);
    k_mix_apply<<<1, 1, 0, st>>>(v);
    return cudaGetLastError();
}

// Single-CTA bitonic sort + unique.  work = shared memory (n_pad <= kSortSmemMax) or a
// global scratch buffer.  Padding value kEmptyKey sorts last and is never a real key.
constexpr uint32_t kSortSmemMax = 16384;   // 128 KB of the 227 KB a CTA may have: covers sketch sizes up to ~10 000

__device__ void bitonic_sort_block(uint64_t *w, uint32_t n_pad)
{
    for (uint32_t kk = 2; kk <= n_pad; kk <<= 1) {
        for (uint32_t j = kk >> 1; j > 0; j >>= 1) {
            for (uint32_t i = threadIdx.x; i < n_pad; i += blockDim.x) {
                const uint32_t p = i ^ j;
                if (p > i) {
                    const uint64_t x = w[i], y = w[p];
                    const bool up = (i & kk) == 0;
                    if ((x > y) == up) { w[i] = y; w[p] = x; }
                }
            }
            __syncthreads();
        }
    }
}

__global__ void __launch_bounds__(1024) k_sort_unique(uint64_t *data, uint32_t n, const uint32_t *n_dev, uint32_t n_pad,
                                                      uint64_t *scratch, uint32_t *n_unique)
{
    extern __shared__ uint64_t sm[];
    __shared__ uint32_t warp_tot[32];
    uint64_t *w = scratch ? scratch : sm;
    if (n_dev) n = min(__ldcg(n_dev), n_pad);
    for (uint32_t i = threadIdx.x; i < n_pad; i += blockDim.x) w[i] = i < n ? data[i] : kEmptyKey;
    __syncthreads();
    bitonic_sort_block(w, n_pad);
    // unique: each thread owns a contiguous run of the sorted array
    const uint32_t per = (n_pad + blockDim.x - 1) / blockDim.x;
    const uint32_t beg = threadIdx.x * per, end = min(beg + per, n_pad);
    uint32_t cnt = 0;
    for (uint32_t i = beg; i < end; i++) cnt += (w[i] != kEmptyKey) && (i == 0 || w[i] != w[i - 1]);
    // exclusive scan of cnt over the block
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t inc = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (uint32_t)o) inc += t;
    }
    if (lane == 31) warp_tot[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        uint32_t v = lane < (blockDim.x >> 5) ? warp_tot[lane] : 0u, s = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= (uint32_t)o) s += t;
        }
        warp_tot[lane] = s - v;  // exclusive
        if (lane == 31) *n_unique = s;
    }
    __syncthreads();
    uint32_t pos = warp_tot[wid] + inc - cnt;
    for (uint32_t i = beg; i < end; i++)
        if ((w[i] != kEmptyKey) && (i == 0 || w[i] != w[i - 1])) data[pos++] = w[i];
}

cudaError_t launch_sort_unique(uint64_t *data, uint32_t n, uint64_t *scratch, uint32_t *n_unique, cudaStream_t st)
{
    uint32_t n_pad = 2;
    while (n_pad < n) n_pad <<= 1;
    static bool attr = false;
    if (!attr) {
        cudaError_t e = cudaFuncSetAttribute(k_sort_unique, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)(kSortSmemMax * sizeof(uint64_t)));
        if (e != cudaSuccess) return e;
        attr = true;
    }
    const bool in_smem = n_pad <= kSortSmemMax;
    k_sort_unique<<<1, 1024, in_smem ? n_pad * sizeof(uint64_t) : 0, st>>>(data, n, nullptr, n_pad, in_smem ? nullptr : scratch,
                                                                          n_unique);
    return cudaGetLastError();
}

// ---- device-side selection of the s smallest (no host round trip) -----------------
constexpr uint32_t kSelBins = 2048;
__device__ __forceinline__ unsigned long long sel_width(const MixState *st, bool use64)
{
    const unsigned long long tau = use64 ? st->tau : min(st->tau, 0xFFFFFFFFull);
    return tau / kSelBins + 1ull;
}

__global__ void __launch_bounds__(256) k_mix_hist(const MixView v, int use64, uint32_t *hist)
{
    __shared__ uint32_t sh[kSelBins];
    for (uint32_t i = threadIdx.x; i < kSelBins; i += blockDim.x) sh[i] = 0;
    __syncthreads();
    const unsigned long long tau = v.st->tau, width = sel_width(v.st, use64 != 0);
    const uint64_t *set = v.sets[v.st->cur & 1u];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i <= v.mask; i += gridDim.x * blockDim.x) {
        const uint64_t x = set[i];
        if (x == kEmptyKey || x > tau) continue;   // older, larger values may linger from before tau dropped
        const unsigned long long b = x / width;
        atomicAdd(&sh[b < kSelBins ? (uint32_t)b : kSelBins - 1], 1u);
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < kSelBins; i += blockDim.x)
        if (sh[i]) atomicAdd(hist + i, sh[i]);
}

// hist[0..2047] = bin counts (in), fill counters (out: zeroed); hist[2048 + b] = where bin b starts in the
// output (exclusive prefix sums), hist[2048 + 2048] = index of the last bin collected
constexpr uint32_t kSelStart = kSelBins, kSelFirst = 2 * kSelBins;
__global__ void __launch_bounds__(1024) k_mix_pick(const MixView v, int use64, uint32_t s, uint32_t *hist, uint32_t out_cap)
{
    __shared__ uint32_t tot[32];
    __shared__ uint32_t first;
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    // inclusive prefix sums of the 2048 bins, two per thread
    const uint32_t a = hist[2 * threadIdx.x], b = hist[2 * threadIdx.x + 1];
    uint32_t inc = a + b;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (uint32_t)o) inc += t;
    }
    if (lane == 31) tot[wid] = inc;
    if (threadIdx.x == 0) first = kSelBins;
    __syncthreads();
    uint32_t before = 0;
    for (uint32_t w = 0; w < wid; w++) before += tot[w];
    const uint32_t cum1 = before + inc, cum0 = cum1 - b;        // through bins 2t+1 and 2t
    if (cum0 >= s) atomicMin(&first, 2 * threadIdx.x);
    else if (cum1 >= s) atomicMin(&first, 2 * threadIdx.x + 1);
    hist[kSelStart + 2 * threadIdx.x] = cum0 - a;               // the collect pass is a counting sort by bin
    hist[kSelStart + 2 * threadIdx.x + 1] = cum0;
    hist[2 * threadIdx.x] = 0; hist[2 * threadIdx.x + 1] = 0;   // ... with these as its fill counters
    __syncthreads();
    const uint32_t f = first < kSelBins ? first : kSelBins - 1; // fewer than s values in all: take every bin
    if (threadIdx.x == f / 2) {
        MixState *st = v.st;
        const uint32_t n = (f & 1u) ? cum1 : cum0;
        st->n_out = n;
        st->n_unique = n;                                       // the live set holds every value once
        st->sel_too_many = n > out_cap ? 1u : 0u;
        hist[kSelFirst] = f;
    }
    if (threadIdx.x == 0) {
        MixState *st = v.st;
        const unsigned long long width = sel_width(st, use64 != 0);
        unsigned long long thr = st->tau;
        if (first + 1 < kSelBins) {
            const unsigned long long t = (unsigned long long)(first + 1) * width - 1ull;
            if (t < thr) thr = t;
        }
        st->sel_thr = thr;
    }
}

// counting sort by bin: the bins are value ranges in ascending order, so after this pass the output is sorted
// up to the order inside each bin
__global__ void __launch_bounds__(256) k_mix_collect_sel(const MixView v, int use64, uint32_t *hist, uint64_t *out, uint32_t out_cap)
{
    const unsigned long long tau = v.st->tau, width = sel_width(v.st, use64 != 0);
    const uint32_t last = hist[kSelFirst];
    const uint64_t *set = v.sets[v.st->cur & 1u];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i <= v.mask; i += gridDim.x * blockDim.x) {
        const uint64_t x = set[i];
        if (x == kEmptyKey || x > tau) continue;
        const unsigned long long bb = x / width;
        const uint32_t b = bb < kSelBins ? (uint32_t)bb : kSelBins - 1;
        if (b > last) continue;
        const uint32_t p = hist[kSelStart + b] + atomicAdd(&hist[b], 1u);
        if (p < out_cap) out[p] = x;
    }
}

// ... which one warp per bin then establishes (bitonic network in shared memory, <= 512 values per bin: a bin
// holds ~130 of a quarter-full set; a crowded one sends the host to the iterative path).  The single-CTA sort
// of all s + slack candidates this replaces was 0.25 ms at s = 10 000 -- the largest kernel after the stream.
constexpr uint32_t kBinSortMax = 512;
__global__ void __launch_bounds__(256) k_mix_binsort(const MixView v, const uint32_t *hist, uint64_t *out, uint32_t out_cap)
{
    __shared__ uint64_t sm[8][kBinSortMax];
    const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
    const uint32_t bin = blockIdx.x * 8u + w;
    if (bin > hist[kSelFirst] || v.st->sel_too_many) return;
    const uint32_t beg = hist[kSelStart + bin];
    const uint32_t end = bin + 1 < kSelBins ? hist[kSelStart + bin + 1] : v.st->n_out;
    const uint32_t L = end - beg;
    if (L < 2 || end > out_cap) return;
    if (L > kBinSortMax) { if (lane == 0) v.st->sel_too_many = 1u; return; }
    uint32_t n_pad = 32;
    while (n_pad < L) n_pad <<= 1;
    uint64_t *a = sm[w];
    for (uint32_t i = lane; i < n_pad; i += 32) a[i] = i < L ? out[beg + i] : kEmptyKey;
    __syncwarp();
    for (uint32_t kk = 2; kk <= n_pad; kk <<= 1)
        for (uint32_t j = kk >> 1; j > 0; j >>= 1) {
            for (uint32_t i = lane; i < n_pad; i += 32) {
                const uint32_t p = i ^ j;
                if (p > i) {
                    const uint64_t x = a[i], y = a[p];
                    if ((x > y) == ((i & kk) == 0)) { a[i] = y; a[p] = x; }
                }
            }
            __syncwarp();
        }
    for (uint32_t i = lane; i < L; i += 32) out[beg + i] = a[i];
}

cudaError_t launch_mix_select(const MixView &v, uint32_t s, bool use64, uint32_t *hist, uint64_t *out, uint32_t n_pad,
                              uint64_t *scratch, cudaStream_t st)
{
    (void)scratch;
    cudaError_t e = cudaMemsetAsync(hist, 0, kSelBins * sizeof(uint32_t), st);
    if (e != cudaSuccess) return e;
    const uint32_t cap = v.mask + 1u;
    k_mix_hist<<<grid_for(cap, 256, 148 * 2), 256, 0, st>>>(v, use64 ? 1 : 0, hist);
    k_mix_pick<<<1, 1024, 0, st>>>(v, use64 ? 1 : 0, s, hist, n_pad);
    k_mix_collect_sel<<<grid_for(cap, 256, 148 * 8), 256, 0, st>>>(v, use64 ? 1 : 0, hist, out, n_pad);
    k_mix_binsort<<<kSelBins / 8, 256, 0, st>>>(v, hist, out, n_pad);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// K4: per-sketch shared count + median multiplicity (rows a11, a13)
// ---------------------------------------------------------------------------
constexpr int kReduceThreads = 128;
// One WARP per sketch, no block barriers: 50 000 sketches of 1000 hashes are 50 000 small
// independent reductions, and almost all of them end after the first pass (no hash present).
// The first version used a CTA per sketch with two __syncthreads per block sum: latency bound at
// 1.4 TB/s of a stream that is mostly sequential (canon[e] == e for keys stored once).
__global__ void __launch_bounds__(256) k_sketch_reduce(const uint64_t *offsets, uint64_t n_refs,
                                                       const uint32_t *canon, const uint32_t *counts,
                                                       const uint32_t *winner, uint32_t *shared_out,
                                                       uint32_t *median_out)
{
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t warp = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint64_t n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t i = warp; i < n_refs; i += n_warps) {
        const uint64_t beg = offsets[i], end = offsets[i + 1];
        auto value = [&](uint64_t e) -> uint32_t {
            const uint32_t id = __ldg(canon + e);
            uint32_t c = __ldcg(counts + id);
            if (winner && c && winner[id] != (uint32_t)i) c = 0;
            return c;
        };
        uint32_t cnt = 0, mx = 0;
        auto take = [&](uint32_t id) {
            // through L1: a lane's four ids are usually consecutive (keys stored once have canon[e] == e),
            // so the four gathers of a 128-bit id load fall into the same sectors
            uint32_t c = __ldg(counts + id);
            if (winner && c && winner[id] != (uint32_t)i) c = 0;
            cnt += c != 0;
            mx = max(mx, c);
        };
        // head up to a 16-byte boundary of canon[], then 256 entries per trip: every lane holds two
        // 128-bit loads of ids and turns them into eight independent count gathers
        uint64_t e = beg;
        const uint64_t head = min(end, (beg + 3) & ~(uint64_t)3);
        if (e + lane < head) take(__ldg(canon + e + lane));
        e = head;
        for (; e + 256 <= end; e += 256) {
            const uint4 a = __ldg(reinterpret_cast<const uint4 *>(canon + e) + lane);
            const uint4 b = __ldg(reinterpret_cast<const uint4 *>(canon + e + 128) + lane);
            take(a.x); take(a.y); take(a.z); take(a.w);
            take(b.x); take(b.y); take(b.z); take(b.w);
        }
        for (uint64_t q = e + lane; q < end; q += 32) take(__ldg(canon + q));
        const uint32_t S = warp_sum(cnt);
        if (S == 0) {
            if (lane == 0) { shared_out[i] = 0; median_out[i] = 0; }
            continue;
        }
#pragma unroll
        for (int o = 16; o; o >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        // S12: sorted_depths[S/2] by MSB-first radix selection over the non-zero counts (re-read: L2 hot)
        uint32_t kk = S / 2, prefix = 0;
        for (int bit = 31 - __clz(mx); bit >= 0; bit--) {
            const uint32_t himask = ~((2u << bit) - 1u);
            uint32_t z = 0;
            auto below = [&](uint32_t c) { z += (c != 0) && ((c & himask) == prefix) && !((c >> bit) & 1u); };
            uint64_t q = beg + lane;
            for (; q + 7 * 32 < end; q += 8 * 32) {   // eight dependent-load chains in flight: only the few
                uint32_t c[8];                         // sketches with hits get here, and they are the tail
#pragma unroll
                for (int u = 0; u < 8; u++) c[u] = value(q + 32 * u);
#pragma unroll
                for (int u = 0; u < 8; u++) below(c[u]);
            }
            for (; q < end; q += 32) below(value(q));
            z = warp_sum(z);
            if (kk >= z) { kk -= z; prefix |= 1u << bit; }
        }
        if (lane == 0) { shared_out[i] = S; median_out[i] = prefix; }
    }
}

cudaError_t launch_sketch_reduce(const uint64_t *offsets, uint64_t n_refs, const uint32_t *canon,
                                 const uint32_t *counts, const uint32_t *winner, uint32_t *shared, uint32_t *median,
                                 int sm_count, cudaStream_t st)
{
    if (!n_refs) return cudaSuccess;
    const uint64_t want = (n_refs + 7) / 8;   // 8 warps per CTA
    const uint32_t grid = (uint32_t)(want < (uint64_t)sm_count * 8 ? want : (uint64_t)sm_count * 8);
    k_sketch_reduce<<<grid, 256, 0, st>>>(offsets, n_refs, canon, counts, winner, shared, median);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// K5: winner-take-all (S17)
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(kReduceThreads) k_winner(const uint64_t *offsets, uint64_t n_refs,
                                                           const uint32_t *canon, const uint32_t *counts,
                                                           const uint32_t *shared, const uint64_t *lengths,
                                                           unsigned long long *best_score,
                                                           unsigned long long *best_len, uint32_t *winner, int pass)
{
    for (uint64_t i = blockIdx.x; i < n_refs; i += gridDim.x) {
        const uint64_t beg = offsets[i], end = offsets[i + 1];
        const uint32_t sh = shared[i];
        if (!sh) continue;  // no present key can belong to a sketch without hits
        const uint64_t size = end - beg;
        // score order == identity order (S13): identity is monotone in shared/size
        const double jac = sh == size ? 1.0 : (double)sh / (double)size;
        const unsigned long long sbits = (unsigned long long)__double_as_longlong(jac);
        const unsigned long long len = lengths[i];
        for (uint64_t e = beg + threadIdx.x; e < end; e += kReduceThreads) {
            const uint32_t id = canon[e];
            if (!counts[id]) continue;
            if (pass < 0) {   // clear only what the later passes will touch (E x 20 bytes of memset otherwise)
                best_score[id] = 0; best_len[id] = 0; winner[id] = 0;
            } else if (pass == 0) {
                atomicMax(best_score + id, sbits);
            } else if (pass == 1) {
                if (best_score[id] == sbits) atomicMax(best_len + id, len);
            } else {
                if (best_score[id] == sbits && best_len[id] == len) atomicMax(winner + id, (uint32_t)i);
            }
        }
    }
}

cudaError_t launch_winner(const uint64_t *offsets, uint64_t n_refs, const uint32_t *canon, const uint32_t *counts,
                          const uint32_t *shared, const uint64_t *lengths, unsigned long long *best_score,
                          unsigned long long *best_len, uint32_t *winner, uint64_t n_entries, int sm_count,
                          cudaStream_t st)
{
    if (!n_refs) return cudaSuccess;
    cudaError_t e;
    (void)n_entries;
    const uint32_t grid = (uint32_t)((n_refs < (uint64_t)sm_count * 16) ? n_refs : (uint64_t)sm_count * 16);
    for (int pass = -1; pass < 3; pass++) {
        k_winner<<<grid, kReduceThreads, 0, st>>>(offsets, n_refs, canon, counts, shared, lengths, best_score,
                                                  best_len, winner, pass);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    return cudaSuccess;
}

// ---------------------------------------------------------------------------
// K6: identity (S13) and p-value (S14) in double precision
// ---------------------------------------------------------------------------
// P[Binomial(n, r) >= x], summed term by term from the term at x.  The leading term
// C(n,x) r^x (1-r)^(n-x) is built as a running product with an explicit binary
// exponent, so nothing large is ever exponentiated: relative error ~ sqrt(x) ulp.
// One WARP per sketch: the lanes split the factors of the leading term between them (a sketch with
// 10 000 shared hashes has a 10 000-factor product, and the few hundred sketches with hits used to
// be the whole run time of the kernel as 16 fully divergent warps), combine the partial products
// in a butterfly (multiplication commutes, so every lane ends with the same bits) and then all
// evaluate the short geometric-like tail redundantly.
__device__ double binom_upper_tail_warp(uint64_t x, uint64_t n, double r, uint32_t lane)
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

__global__ void __launch_bounds__(256) k_stats(uint32_t k, uint64_t set_size, const unsigned long long *set_size_dev,
                                               uint64_t n, const uint32_t *shared32, const uint64_t *shared64,
                                               const uint64_t *offsets, const uint64_t *sizes, double *identity,
                                               double *pvalue)
{
    const uint32_t lane = threadIdx.x & 31u;
    if (set_size_dev) set_size = __ldcg(set_size_dev);
    const uint64_t n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const double kmer_space = ldexp(1.0, 2 * (int)k);  // 4^k
    const double r = 1.0 / (1.0 + kmer_space / (double)set_size);
    for (uint64_t i = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += n_warps) {
        const uint64_t x = shared32 ? (uint64_t)shared32[i] : shared64[i];
        const uint64_t size = offsets ? offsets[i + 1] - offsets[i] : sizes[i];
        const double p = binom_upper_tail_warp(x, size, r, lane);
        if (lane == 0) {
            double id;
            if (x == size) id = 1.0;
            else if (x == 0) id = 0.0;
            else id = pow((double)x / (double)size, 1.0 / (double)k);
            identity[i] = id;
            pvalue[i] = p;
        }
    }
}

// Rows a14-a16 in O(references with hits): identity + p-value only where shared > 0 -- everything
// else is "not reported" (S15) -- written straight into host-mapped rows, so that the trip home is the
// hits, not N x 24 bytes of mostly zeros (300 000 sketches: 7 MB per screen).
__global__ void __launch_bounds__(256) k_stats_hits(const StatsHitArgs a)
{
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    const uint32_t nh = min(__ldcg(a.n_hit), a.rows.cap);
    const double kmer_space = ldexp(1.0, 2 * (int)a.k);  // 4^k
    for (uint32_t q = warp; q < nh; q += n_warps) {
        const uint32_t i = a.hit[q];
        uint32_t j = 0;
        while (j + 1 < a.n_seg && (uint64_t)i >= a.seg_begin[j + 1]) j++;
        const unsigned long long set_size = a.set_size_dev ? __ldcg(a.set_size_dev + j) : a.set_size[j];
        const double r = 1.0 / (1.0 + kmer_space / (double)set_size);
        const uint64_t x = a.shared[i], size = a.offsets[i + 1] - a.offsets[i];
        const double p = binom_upper_tail_warp(x, size, r, lane);
        if (lane == 0) {
            double id;
            if (x == size) id = 1.0;
            else if (x == 0) id = 0.0;
            else id = pow((double)x / (double)size, 1.0 / (double)a.k);
            a.rows.ref[q] = i; a.rows.shared[q] = (uint32_t)x; a.rows.median[q] = a.median[i];
            a.rows.identity[q] = id; a.rows.pvalue[q] = p;
        }
    }
}

// dense reduction ran: the references with hits are found by looking at all of them
__global__ void __launch_bounds__(256) k_hits_from_dense(const uint32_t *shared, uint32_t n_refs, uint32_t *hit, uint32_t *n_hit)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_refs; i += gridDim.x * blockDim.x)
        if (shared[i]) hit[atomicAdd(n_hit, 1u)] = i;
}

cudaError_t launch_stats_hits(const StatsHitArgs &a, bool from_dense, uint32_t n_refs, uint32_t *hit, uint32_t *n_hit,
                              int sm_count, cudaStream_t st)
{
    if (!n_refs) return cudaSuccess;
    if (from_dense) {
        cudaError_t e = cudaMemsetAsync(n_hit, 0, sizeof(uint32_t), st);
        if (e != cudaSuccess) return e;
        k_hits_from_dense<<<grid_for(n_refs, 256, 148 * 4), 256, 0, st>>>(a.shared, n_refs, hit, n_hit);
    }
    k_stats_hits<<<(uint32_t)sm_count * 4u, 256, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_stats(uint32_t k, uint64_t set_size, const unsigned long long *set_size_dev, uint64_t n,
                         const uint32_t *shared32, const uint64_t *shared64, const uint64_t *offsets,
                         const uint64_t *sizes, double *identity, double *pvalue, cudaStream_t st)
{
    if (!n) return cudaSuccess;
    const uint64_t want = (n + 7) / 8;   // 8 warps per CTA, one sketch per warp and trip
    k_stats<<<(uint32_t)(want < 148 * 32 ? want : 148 * 32), 256, 0, st>>>(k, set_size, set_size_dev, n, shared32, shared64,
                                                                          offsets, sizes, identity, pvalue);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// Device-side packer: one thread builds one 64-bit word from 32 base codes
// (two 128-bit loads), flags codes > 3 and everything past n as invalid.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_pack_codes(const uint8_t *codes, uint64_t n, uint64_t *seq, uint32_t *inv,
                                                    uint64_t n_words)
{
    for (uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; w < n_words;
         w += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t p0 = w * 32;
        uint64_t acc = 0;
        uint32_t bad = 0;
        if (p0 + 32 <= n && ((uintptr_t)(codes + p0) & 15) == 0) {
            const uint4 a = __ldg(reinterpret_cast<const uint4 *>(codes + p0));
            const uint4 b = __ldg(reinterpret_cast<const uint4 *>(codes + p0) + 1);
            const uint32_t v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 8; i++) {
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    const uint32_t c = (v[i] >> (8 * j)) & 0xFFu;
                    acc = (acc << 2) | (c & 3u);
                    bad = (bad << 1) | (c > 3u);
                }
            }
        } else {
            for (int j = 0; j < 32; j++) {
                const uint64_t p = p0 + j;
                const uint32_t c = p < n ? codes[p] : 4u;
                acc = (acc << 2) | (c & 3u);
                bad = (bad << 1) | (c > 3u);
            }
        }
        seq[w] = acc;
        inv[w] = bad;
    }
}

cudaError_t launch_pack_codes(const uint8_t *codes, uint64_t n, uint64_t *seq, uint32_t *inv, uint64_t n_words_alloc,
                              cudaStream_t st)
{
    if (!n_words_alloc) return cudaSuccess;
    k_pack_codes<<<grid_for(n_words_alloc, 256, 148 * 16), 256, 0, st>>>(codes, n, seq, inv, n_words_alloc);
    return cudaGetLastError();
}

__global__ void __launch_bounds__(256) k_pack_codes_dyn(const uint8_t *codes, const unsigned long long *n_dev,
                                                        uint64_t *seq, uint32_t *inv, uint64_t n_words)
{
    const uint64_t n = __ldcg(n_dev);
    for (uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; w < n_words;
         w += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t p0 = w * 32;
        uint64_t acc = 0;
        uint32_t bad = 0;
        if (p0 + 32 <= n) {
            const uint4 a = __ldg(reinterpret_cast<const uint4 *>(codes + p0));
            const uint4 b = __ldg(reinterpret_cast<const uint4 *>(codes + p0) + 1);
            const uint32_t v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 8; i++) {
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    const uint32_t c = (v[i] >> (8 * j)) & 0xFFu;
                    acc = (acc << 2) | (c & 3u);
                    bad = (bad << 1) | (c > 3u);
                }
            }
        } else if (p0 < n) {
            for (int j = 0; j < 32; j++) {
                const uint64_t p = p0 + j;
                const uint32_t c = p < n ? codes[p] : 4u;
                acc = (acc << 2) | (c & 3u);
                bad = (bad << 1) | (c > 3u);
            }
        } else {
            bad = ~0u;
        }
        seq[w] = acc;
        inv[w] = bad;
    }
}

cudaError_t launch_pack_codes_dyn(const uint8_t *codes, const unsigned long long *n_dev, uint64_t *seq, uint32_t *inv,
                                  uint64_t n_words_alloc, cudaStream_t st)
{
    if (!n_words_alloc) return cudaSuccess;
    k_pack_codes_dyn<<<grid_for(n_words_alloc, 256, 148 * 16), 256, 0, st>>>(codes, n_dev, seq, inv, n_words_alloc);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// Device-side FASTA ingest (row a6 on the GPU).
//
// "Events" change the parser state: a newline, a header start ('>' as first byte of a
// line) and a '+' line start.  Two "latest event wins" streams,
//   A: newline (even code) / header start (odd)        -> in a header line iff latest A is odd
//   B: header start (even) / '+' line start (odd)      -> skipping to the next header iff
//      latest B is odd (B is seeded odd: everything before the first header is skipped, like
//      the host packer's SEEK_HDR state; a '+' line ends a record's sequence, kseq's rule),
// make the state a prefix MAX of event codes and output positions a prefix SUM; each scan is
// tile aggregate -> single-CTA scan -> tile re-walk.  Bytes are turned into 32-bit masks
// ONCE (k_fa_masks, SIMD-in-register compares); the later passes work on masks.
// Same output as fasta_pack.cpp: header => one invalid position, CR before LF dropped,
// every other byte of a sequence line kept (non-ACGT => code 4).
// ---------------------------------------------------------------------------
// 4-bit mask (bit b = byte b) of the bytes of w equal to the byte replicated in pat
__device__ __forceinline__ uint32_t eq_mask4(uint32_t w, uint32_t pat)
{
    const uint32_t x = w ^ pat;
    const uint32_t t = ((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x;  // bit 7 of a byte set iff that byte != 0
    const uint32_t z = (~t & 0x80808080u) >> 7;               // 0x01 per equal byte
    return (z * 0x01020408u) >> 24;                           // gather the four flags (no carries collide)
}

struct FaMasks { uint32_t nl, hs, pl, crdrop; };

__device__ __forceinline__ void fa_load_words(const uint8_t *text, uint32_t n, uint32_t i0, uint32_t w[8], uint32_t &n_here,
                                              uint32_t &prev, uint32_t &next)
{
    n_here = i0 >= n ? 0u : min(32u, n - i0);
    if (n_here == 32 && ((uintptr_t)(text + i0) & 15) == 0) {
        const uint4 a = __ldg(reinterpret_cast<const uint4 *>(text + i0));
        const uint4 c = __ldg(reinterpret_cast<const uint4 *>(text + i0) + 1);
        w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w; w[4] = c.x; w[5] = c.y; w[6] = c.z; w[7] = c.w;
    } else {
#pragma unroll
        for (int q = 0; q < 8; q++) {
            uint32_t v = 0;
#pragma unroll
            for (int b = 0; b < 4; b++) {
                const uint32_t i = q * 4 + b;
                v |= (uint32_t)(i < n_here ? text[i0 + i] : (uint8_t)'\n') << (8 * b);
            }
            w[q] = v;
        }
    }
    prev = (i0 == 0 || i0 > n) ? (uint32_t)'\n' : (uint32_t)text[i0 - 1];
    next = i0 + 32 < n ? (uint32_t)text[i0 + 32] : (uint32_t)'\n';
}

__device__ __forceinline__ void fa_event_codes(const FaMasks &m, uint32_t i0, uint32_t &eva, uint32_t &evb)
{
    eva = 0; evb = 0;
    const uint32_t a = m.nl | m.hs, b = m.hs | m.pl;
    if (a) { const uint32_t top = 31 - __clz(a); eva = 2u * (i0 + top) + 2u + ((m.hs >> top) & 1u); }
    if (b) { const uint32_t top = 31 - __clz(b); evb = 2u * (i0 + top) + 2u + ((m.pl >> top) & 1u); }
}

__device__ __forceinline__ uint32_t block_excl_max(uint32_t v, uint32_t *warp_buf, uint32_t &total)
{
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (uint32_t)o) inc = max(inc, t);
    }
    uint32_t excl = __shfl_up_sync(0xffffffffu, inc, 1);
    if (lane == 0) excl = 0;
    __syncthreads();
    if (lane == 31) warp_buf[wid] = inc;
    __syncthreads();
    uint32_t before = 0, tot = 0;
    for (uint32_t w = 0; w < blockDim.x / 32; w++) {
        const uint32_t x = warp_buf[w];
        if (w < wid) before = max(before, x);
        tot = max(tot, x);
    }
    total = tot;
    return max(before, excl);
}

__device__ __forceinline__ uint32_t block_excl_sum(uint32_t v, uint32_t *warp_buf, uint32_t &total)
{
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (uint32_t)o) inc += t;
    }
    __syncthreads();
    if (lane == 31) warp_buf[wid] = inc;
    __syncthreads();
    uint32_t before = 0, tot = 0;
    for (uint32_t w = 0; w < blockDim.x / 32; w++) {
        const uint32_t x = warp_buf[w];
        if (w < wid) before += x;
        tot += x;
    }
    total = tot;
    return before + inc - v;
}

// pass 1: bytes -> per-thread masks (stored) + per-tile last events
__global__ void __launch_bounds__(256) k_fa_masks(const uint8_t *text, uint32_t n, uint4 *masks, uint32_t *tile_event_a,
                                                  uint32_t *tile_event_b)
{
    __shared__ uint32_t wb[8];
    const uint32_t i0 = blockIdx.x * kFaTileBytes + threadIdx.x * 32;
    uint32_t w[8], n_here, prev, next;
    fa_load_words(text, n, i0, w, n_here, prev, next);
    uint32_t nl = 0, gt = 0, plus = 0, cr = 0;
#pragma unroll
    for (int q = 0; q < 8; q++) {
        nl |= eq_mask4(w[q], 0x0A0A0A0Au) << (4 * q);
        gt |= eq_mask4(w[q], 0x3E3E3E3Eu) << (4 * q);
        plus |= eq_mask4(w[q], 0x2B2B2B2Bu) << (4 * q);
        cr |= eq_mask4(w[q], 0x0D0D0D0Du) << (4 * q);
    }
    const uint32_t here = n_here >= 32 ? ~0u : ((1u << n_here) - 1u);
    const uint32_t nl_real = nl & here;                 // bytes past the text were loaded as '\n'
    const uint32_t line_start = (nl << 1) | (prev == '\n');
    FaMasks m;
    m.nl = nl_real;
    m.hs = gt & line_start & here;
    m.pl = plus & line_start & here;
    m.crdrop = cr & ((nl >> 1) | ((next == '\n') ? 0x80000000u : 0u)) & here;
    masks[blockIdx.x * 256 + threadIdx.x] = make_uint4(m.nl, m.hs, m.pl, m.crdrop);
    uint32_t ea, eb, ta, tb;
    fa_event_codes(m, i0, ea, eb);
    block_excl_max(ea, wb, ta);
    block_excl_max(eb, wb, tb);
    if (threadIdx.x == 0) { tile_event_a[blockIdx.x] = ta; tile_event_b[blockIdx.x] = tb; }
}

// single CTA: exclusive prefix max (out_max) or exclusive prefix sum (out_sum) over the tiles
__global__ void __launch_bounds__(1024) k_tile_scan(const uint32_t *in, uint32_t n, uint32_t *out_max, uint64_t *out_sum,
                                                    unsigned long long *total_out, uint32_t init)
{
    __shared__ unsigned long long wsum[32];
    __shared__ unsigned long long carry_s;
    if (threadIdx.x == 0) carry_s = init;
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (uint32_t base = 0; base < n; base += 1024) {
        const uint32_t i = base + threadIdx.x;
        const unsigned long long v = i < n ? in[i] : 0ull;
        unsigned long long inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= (uint32_t)o) inc = out_max ? max(inc, t) : inc + t;
        }
        if (lane == 31) wsum[wid] = inc;
        __syncthreads();
        unsigned long long before = carry_s;
        for (uint32_t w = 0; w < wid; w++) before = out_max ? max(before, wsum[w]) : before + wsum[w];
        unsigned long long excl = __shfl_up_sync(0xffffffffu, inc, 1);
        if (lane == 0) excl = 0;
        const unsigned long long e = out_max ? max(before, excl) : before + excl;
        if (i < n) {
            if (out_max) out_max[i] = (uint32_t)e; else out_sum[i] = e;
        }
        __syncthreads();
        if (threadIdx.x == 1023) carry_s = out_max ? max(e, v) : e + v;
        __syncthreads();
    }
    if (threadIdx.x == 0 && total_out) *total_out = carry_s;
}

// pass 2: masks + carried state -> which bytes are emitted; per-tile counts
__global__ void __launch_bounds__(256) k_fa_state(uint32_t n, const uint4 *masks, const uint32_t *tile_carry_a,
                                                  const uint32_t *tile_carry_b, uint2 *emit, uint32_t *tile_count,
                                                  unsigned long long *totals)
{
    __shared__ uint32_t wb[8];
    const uint32_t i0 = blockIdx.x * kFaTileBytes + threadIdx.x * 32;
    const uint4 mm = masks[blockIdx.x * 256 + threadIdx.x];
    const FaMasks m{mm.x, mm.y, mm.z, mm.w};
    uint32_t ea, eb, tot_ev;
    fa_event_codes(m, i0, ea, eb);
    const uint32_t carry_a = max(tile_carry_a[blockIdx.x], block_excl_max(ea, wb, tot_ev));
    const uint32_t carry_b = max(tile_carry_b[blockIdx.x], block_excl_max(eb, wb, tot_ev));
    bool in_header = (carry_a & 1u) != 0, in_skip = (carry_b & 1u) != 0;
    const uint32_t n_here = i0 >= n ? 0u : min(32u, n - i0);
    const uint32_t here = n_here >= 32 ? ~0u : ((1u << n_here) - 1u);
    uint32_t keep = 0, pos = 0, ev = m.nl | m.hs | m.pl;
    while (ev) {  // one iteration per event (about one per 80 bytes of wrapped FASTA)
        const uint32_t e = __ffs(ev) - 1;
        if (!in_header && !in_skip && e > pos) keep |= ((1u << e) - 1u) & ~((1u << pos) - 1u);
        const uint32_t bit = 1u << e;
        if (m.nl & bit) in_header = false;
        else if (m.hs & bit) { in_header = true; in_skip = false; }
        else in_skip = true;
        pos = e + 1;
        ev &= ev - 1;
    }
    if (!in_header && !in_skip && pos < 32) keep |= ~((1u << pos) - 1u);
    keep &= here & ~m.crdrop;
    const uint32_t em = keep | m.hs;  // a header start emits the record separator (S6)
    emit[blockIdx.x * 256 + threadIdx.x] = make_uint2(em, m.hs);
    uint32_t tile_total;
    block_excl_sum(__popc(em), wb, tile_total);
    if (threadIdx.x == 0) tile_count[blockIdx.x] = tile_total;
    uint32_t bases = warp_sum((uint32_t)__popc(keep)), recs = warp_sum((uint32_t)__popc(m.hs));
    if ((threadIdx.x & 31) == 0) {
        if (bases) atomicAdd(totals + 1, (unsigned long long)bases);
        if (recs) atomicAdd(totals + 2, (unsigned long long)recs);
    }
}

// pass 3: emitted bytes -> base codes, compacted through shared memory, written coalesced
__global__ void __launch_bounds__(256) k_fa_emit(const uint8_t *text, uint32_t n, const uint2 *emit,
                                                 const uint64_t *tile_offset, uint8_t *codes)
{
    __shared__ uint32_t wb[8];
    __shared__ __align__(16) uint8_t out[kFaTileBytes];
    const uint32_t i0 = blockIdx.x * kFaTileBytes + threadIdx.x * 32;
    const uint2 e = emit[blockIdx.x * 256 + threadIdx.x];
    uint32_t tile_total;
    uint32_t local = block_excl_sum(__popc(e.x), wb, tile_total);
    if (e.x) {
        uint32_t w[8], n_here, prev, next;
        fa_load_words(text, n, i0, w, n_here, prev, next);
#pragma unroll
        for (int q = 0; q < 8; q++) {
            // SIMD-in-register: fold case, (c>>1)&3 gives A0 C1 T2 G3, xor with its own high bit -> A0 C1 G2 T3
            const uint32_t up = w[q] & 0xDFDFDFDFu;
            const uint32_t c1 = (up >> 1) & 0x03030303u;
            uint32_t code = c1 ^ ((c1 >> 1) & 0x01010101u);
            const uint32_t ok = eq_mask4(up, 0x41414141u) | eq_mask4(up, 0x43434343u) | eq_mask4(up, 0x47474747u) |
                                eq_mask4(up, 0x54545454u);
#pragma unroll
            for (int b = 0; b < 4; b++) {
                const uint32_t bit = 1u << (q * 4 + b);
                if (e.x & bit) {
                    uint32_t c = (code >> (8 * b)) & 3u;
                    if (!((ok >> b) & 1u) || (e.y & bit)) c = 4u;  // not A/C/G/T, or the record separator
                    out[local++] = (uint8_t)c;
                }
            }
        }
    }
    __syncthreads();
    uint8_t *dst = codes + tile_offset[blockIdx.x];
    for (uint32_t i = threadIdx.x; i < tile_total; i += 256) dst[i] = out[i];
}

__global__ void k_fa_totals(const unsigned long long *chunk_positions, unsigned long long *totals)
{
    totals[0] += *chunk_positions;
}

cudaError_t launch_fasta_to_codes(const uint8_t *text, uint32_t n, uint8_t *codes, const FaScratch &sc, cudaStream_t st)
{
    if (!n) return cudaMemsetAsync(sc.chunk_positions, 0, sizeof(unsigned long long), st);
    const uint32_t tiles = (n + kFaTileBytes - 1) / kFaTileBytes;
    k_fa_masks<<<tiles, 256, 0, st>>>(text, n, sc.masks, sc.tile_event, sc.tile_event_b);
    k_tile_scan<<<1, 1024, 0, st>>>(sc.tile_event, tiles, sc.tile_carry, nullptr, nullptr, 0u);
    k_tile_scan<<<1, 1024, 0, st>>>(sc.tile_event_b, tiles, sc.tile_carry_b, nullptr, nullptr, 1u);
    k_fa_state<<<tiles, 256, 0, st>>>(n, sc.masks, sc.tile_carry, sc.tile_carry_b, sc.emit, sc.tile_count, sc.totals);
    k_tile_scan<<<1, 1024, 0, st>>>(sc.tile_count, tiles, nullptr, sc.tile_offset, sc.chunk_positions, 0u);
    k_fa_emit<<<tiles, 256, 0, st>>>(text, n, sc.emit, sc.tile_offset, codes);
    k_fa_totals<<<1, 1, 0, st>>>(sc.chunk_positions, sc.totals);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// O(present hashes) reduction: rows a11 ("Summing shared"), a12 (-w), a13 (medians)
//
// k_stream left the ids of the non-zero counts in touched[].  Per present key the chain
// next[] lists the entries (hence references) that hold it.  Four small passes:
//   count    shared[ref]++ per (key, holder)            (-w: only for the key's winner, S17)
//   alloc    hand every reference with hits a segment of depths[]
//   scatter  the same walk again, writing each key's count into its reference's segment
//   median   one warp per reference with hits: radix selection of element shared/2 (S12)
// Every kernel returns at once when the list is incomplete (overflow) or a count wrapped; the
// host then reruns the dense O(stored hashes) kernels above.
// ---------------------------------------------------------------------------
__device__ __forceinline__ bool sparse_list(const SparseView &sp, uint32_t &n)
{
    n = __ldcg(&sp.st->n_touched);
    return n <= sp.cap;
}
__device__ __forceinline__ bool sparse_ok(const SparseView &sp, uint32_t &n)
{
    return sparse_list(sp, n) && !__ldcg(&sp.st->wrapped);
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

// S17: among the holders of key t inside source file j, the one with the best (score, length, index);
// score order == identity order (S13): identity is monotone in shared/size, and equal rationals give
// equal doubles.  kNoEntry when file j does not hold the key.
__device__ __forceinline__ uint32_t chain_winner(const SparseReduceArgs &a, uint32_t t, uint32_t j)
{
    const uint64_t lo = a.seg_begin[j], hi = a.seg_begin[j + 1];
    unsigned long long best_s = 0, best_l = 0;
    uint32_t best_i = kNoEntry;
    for (uint32_t e = t; e != kNoEntry; e = __ldg(a.next + e)) {
        const uint32_t i = ref_of_entry(a.offsets, a.n_refs, e, a.ref_scale);
        if (i < lo || i >= hi) continue;
        const uint32_t sh = a.plain[i];
        const uint64_t size = a.offsets[i + 1] - a.offsets[i];
        const double jac = sh == size ? 1.0 : (double)sh / (double)size;
        const unsigned long long sb = (unsigned long long)__double_as_longlong(jac), len = a.lengths[i];
        if (best_i == kNoEntry || sb > best_s || (sb == best_s && (len > best_l || (len == best_l && i > best_i)))) {
            best_s = sb; best_l = len; best_i = i;
        }
    }
    return best_i;
}

// Per-CTA aggregation of the walk's updates.  The references with hits are few (hundreds) and often adjacent
// (strains of one species sit next to each other in a RefSeq-ordered sketch file), so millions of
// atomicAdd(shared + ref) land on a handful of cache lines: at s = 10 000 (2.76 M present hashes, 500
// references with hits, all in 16 lines) the two walks took 0.41 ms each.  Each CTA first counts per reference
// in a small shared-memory table and then touches global memory once per (CTA, reference).
constexpr uint32_t kAggSlots = 2048, kAggEmpty = 0xFFFFFFFFu;
struct CtaAgg { uint32_t key[kAggSlots], val[kAggSlots], cur[kAggSlots]; };   // 24 KB

__device__ __forceinline__ int agg_insert(CtaAgg &g, uint32_t i)   // slot of reference i, claimed if new; -1: no room nearby
{
    uint32_t h = (i * 2654435761u) >> 21;
    for (int tries = 0; tries < 32; tries++) {
        const uint32_t old = atomicCAS(&g.key[h], kAggEmpty, i);
        if (old == kAggEmpty || old == i) return (int)h;
        h = (h + 1) & (kAggSlots - 1);
    }
    return -1;
}
__device__ __forceinline__ int agg_find(const CtaAgg &g, uint32_t i)   // after all inserts: same probe path, no claims
{
    uint32_t h = (i * 2654435761u) >> 21;
    for (int tries = 0; tries < 32; tries++) {
        const uint32_t k = g.key[h];
        if (k == i) return (int)h;
        if (k == kAggEmpty) return -1;
        h = (h + 1) & (kAggSlots - 1);
    }
    return -1;
}

template <bool WTA, bool SCATTER>
__global__ void __launch_bounds__(256) k_sparse_walk(const SparseReduceArgs a)
{
    __shared__ CtaAgg g;
    uint32_t n;
    if (!sparse_ok(a.sp, n)) return;                       // (the same answer in every thread of every CTA)
    for (uint32_t q = threadIdx.x; q < kAggSlots; q += blockDim.x) { g.key[q] = kAggEmpty; g.val[q] = 0; g.cur[q] = 0; }
    __syncthreads();
    // the (reference, count) pairs of this thread's present hashes, in a fixed order: f(reference, count) for each
    auto walk = [&](auto &&f) {
        for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < n; p += gridDim.x * blockDim.x) {
            const uint32_t t = a.sp.touched[p];
            const uint32_t c = __ldcg(a.counts + t);
            if (!c) continue;
            if (!WTA) {
                for (uint32_t e = t; e != kNoEntry; e = __ldg(a.next + e)) f(ref_of_entry(a.offsets, a.n_refs, e, a.ref_scale), c);
            } else {
                for (uint32_t j = 0; j < a.n_seg; j++) {
                    const uint32_t w = chain_winner(a, t, j);
                    if (w != kNoEntry) f(w, c);
                }
            }
        }
    };
    auto count_global = [&](uint32_t i, uint32_t add) {
        const uint32_t old = atomicAdd(a.shared + i, add);
        if (!WTA && old == 0u) a.hit[atomicAdd(&a.sp.st->n_hit, 1u)] = i;   // at most n_refs appends
    };
    // pass A: per-CTA counts (a reference that finds no slot nearby goes straight to global memory)
    walk([&](uint32_t i, uint32_t) {
        const int sl = agg_insert(g, i);
        if (sl >= 0) atomicAdd(&g.val[sl], 1u);
        else if (!SCATTER) count_global(i, 1u);
    });
    __syncthreads();
    if constexpr (!SCATTER) {
        for (uint32_t q = threadIdx.x; q < kAggSlots; q += blockDim.x)
            if (g.key[q] != kAggEmpty) count_global(g.key[q], g.val[q]);
    } else {
        // scatter: reserve this CTA's stretch of every reference's segment, then hand the slots out locally
        for (uint32_t q = threadIdx.x; q < kAggSlots; q += blockDim.x)
            if (g.key[q] != kAggEmpty) g.val[q] = atomicAdd(a.seg_fill + g.key[q], g.val[q]);
        __syncthreads();
        walk([&](uint32_t i, uint32_t c) {
            const int sl = agg_find(g, i);
            const uint32_t off = sl >= 0 ? g.val[sl] + atomicAdd(&g.cur[sl], 1u) : atomicAdd(a.seg_fill + i, 1u);
            const uint32_t pos = a.seg_start[i] + off;
            if (pos < a.pair_cap) a.depths[pos] = c;
        });
    }
}

__global__ void __launch_bounds__(256) k_sparse_zero_hit(const SparseReduceArgs a)
{
    uint32_t n;
    if (!sparse_ok(a.sp, n)) return;
    const uint32_t nh = __ldcg(&a.sp.st->n_hit);
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < nh; q += gridDim.x * blockDim.x) a.shared[a.hit[q]] = 0;
}

__global__ void __launch_bounds__(256) k_sparse_alloc(const SparseReduceArgs a)
{
    uint32_t n;
    if (!sparse_ok(a.sp, n)) return;
    const uint32_t nh = __ldcg(&a.sp.st->n_hit);
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < nh; q += gridDim.x * blockDim.x) {
        const uint32_t i = a.hit[q], sh = a.shared[i];
        const uint32_t start = atomicAdd(&a.sp.st->n_pairs, sh);   // sum of shared <= stored hashes < 2^32
        a.seg_start[i] = start;
        a.seg_fill[i] = 0;
        if (start + sh > a.pair_cap) atomicExch(&a.sp.st->overflow, 1u);
    }
}

__global__ void __launch_bounds__(256) k_sparse_median(const SparseReduceArgs a)
{
    uint32_t n;
    if (!sparse_ok(a.sp, n) || __ldcg(&a.sp.st->overflow)) return;
    const uint32_t nh = __ldcg(&a.sp.st->n_hit), lane = threadIdx.x & 31u;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t q = warp; q < nh; q += n_warps) {
        const uint32_t i = a.hit[q], S = a.shared[i];
        if (!S) continue;   // lost every key to a better reference (-w): median stays 0
        const uint32_t *d = a.depths + a.seg_start[i];
        uint32_t mx = 0;
        for (uint32_t x = lane; x < S; x += 32) mx = max(mx, __ldcg(d + x));
#pragma unroll
        for (int o = 16; o; o >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        // S12: sorted_depths[S/2] by MSB-first radix selection (depths are the non-zero counts)
        uint32_t kk = S / 2, prefix = 0;
        for (int bit = 31 - __clz(mx); bit >= 0; bit--) {
            const uint32_t himask = ~((2u << bit) - 1u);
            uint32_t z = 0;
            for (uint32_t x = lane; x < S; x += 32) {
                const uint32_t c = __ldcg(d + x);
                z += ((c & himask) == prefix) && !((c >> bit) & 1u);
            }
            z = warp_sum(z);
            if (kk >= z) { kk -= z; prefix |= 1u << bit; }
        }
        if (lane == 0) a.median[i] = prefix;
    }
}

cudaError_t launch_sparse_reduce(const SparseReduceArgs &a, bool wta, int sm_count, cudaStream_t st)
{
    if (!a.n_refs || !a.sp.touched) return cudaSuccess;
    const uint32_t grid = (uint32_t)sm_count * 4u;
    k_sparse_walk<false, false><<<grid, 256, 0, st>>>(a);
    if (wta) {
        cudaError_t e = cudaMemcpyAsync(a.plain, a.shared, (size_t)a.n_refs * 4, cudaMemcpyDeviceToDevice, st);
        if (e != cudaSuccess) return e;
        k_sparse_zero_hit<<<grid, 256, 0, st>>>(a);
        k_sparse_walk<true, false><<<grid, 256, 0, st>>>(a);
    }
    k_sparse_alloc<<<grid, 256, 0, st>>>(a);
    if (wta) k_sparse_walk<true, true><<<grid, 256, 0, st>>>(a);
    else k_sparse_walk<false, true><<<grid, 256, 0, st>>>(a);
    k_sparse_median<<<grid, 256, 0, st>>>(a);
    return cudaGetLastError();
}

// counts[] back to zero in O(touched): only the recorded ids were ever non-zero
__global__ void __launch_bounds__(256) k_sparse_reset(const SparseView sp, uint32_t *counts)
{
    uint32_t n;
    if (!sparse_list(sp, n)) return;
    for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < n; p += gridDim.x * blockDim.x) counts[sp.touched[p]] = 0;
}

// ... unless the list is incomplete: then every count is cleared
__global__ void __launch_bounds__(256) k_counts_clear_if_overflow(const SparseView sp, uint4 *counts16, uint64_t n16)
{
    uint32_t n;
    if (sparse_list(sp, n)) return;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (uint64_t)gridDim.x * blockDim.x)
        counts16[i] = make_uint4(0, 0, 0, 0);
}

cudaError_t launch_counts_clear_if_overflow(const SparseView &sp, uint32_t *counts, uint64_t n, cudaStream_t st)
{
    if (!n) return cudaSuccess;
    // counts[] is a cudaMalloc allocation (256-byte aligned) padded to a multiple of four entries
    const uint64_t n16 = (n + 3) / 4;
    k_counts_clear_if_overflow<<<grid_for(n16, 256, 148 * 8), 256, 0, st>>>(sp, reinterpret_cast<uint4 *>(counts), n16);
    return cudaGetLastError();
}

cudaError_t launch_sparse_reset(const SparseView &sp, uint32_t *counts, int sm_count, cudaStream_t st)
{
    k_sparse_reset<<<(uint32_t)sm_count * 4u, 256, 0, st>>>(sp, counts);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// Multi-GPU count exchange: ranks trade (entry id, count) pairs of the hashes that occurred in
// their shard instead of the dense vector.  Integer adds: order independent, exact.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_touched_pairs(const SparseView sp, const uint32_t *counts,
                                                       unsigned long long *pairs, uint32_t cap, uint32_t *n_out)
{
    uint32_t n;
    if (!sparse_list(sp, n)) return;
    if (blockIdx.x == 0 && threadIdx.x == 0) *n_out = n;
    for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < n && p < cap; p += gridDim.x * blockDim.x) {
        const uint32_t t = sp.touched[p];
        pairs[p] = ((unsigned long long)t << 32) | __ldcg(counts + t);
    }
}

// the touched list is missing or incomplete: scan every count
__global__ void __launch_bounds__(256) k_counts_compact(const SparseView sp, const uint32_t *counts, uint64_t n,
                                                        unsigned long long *pairs, uint32_t cap, uint32_t *n_out)
{
    uint32_t nt;
    if (sp.touched && sparse_list(sp, nt)) return;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t c = counts[i];
        if (c) {
            const uint32_t p = atomicAdd(n_out, 1u);
            if (p < cap) pairs[p] = ((unsigned long long)i << 32) | c;
        }
    }
}

__device__ __forceinline__ void add_pair(const SparseView &sp, uint32_t *counts, uint64_t n_counts, unsigned long long p)
{
    const uint64_t id = p >> 32;
    const uint32_t c = (uint32_t)p;
    if (id < n_counts && c) count_add(sp, counts, (uint32_t)id, c);   // padding carries id 0xFFFFFFFF
}

__global__ void __launch_bounds__(256) k_counts_scatter_add(const SparseView sp, uint32_t *counts, uint64_t n_counts,
                                                            const unsigned long long *pairs, uint64_t n_pairs)
{
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_pairs; i += (uint64_t)gridDim.x * blockDim.x)
        add_pair(sp, counts, n_counts, pairs[i]);
}

__global__ void __launch_bounds__(256) k_counts_absorb(const SparseView sp, uint32_t *counts, uint64_t n_counts,
                                                       const unsigned long long *rows, uint32_t n_rows, uint32_t cap,
                                                       uint32_t skip)
{
    const size_t stride = (size_t)cap + 1;
    uint32_t most = 0;
    for (uint32_t r = 0; r < n_rows; r++) most = max(most, (uint32_t)__ldcg(rows + r * stride));
    if (blockIdx.x == 0 && threadIdx.x == 0) sp.st->xchg_max = most;
    if (most > cap) {   // some rank's record is incomplete: add nothing
        if (blockIdx.x == 0 && threadIdx.x == 0) sp.st->xchg_overflow = 1u;
        return;
    }
    const uint64_t total = (uint64_t)n_rows * cap;
    for (uint64_t x = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; x < total; x += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t r = (uint32_t)(x / cap), i = (uint32_t)(x % cap);
        if (r == skip || i >= (uint32_t)__ldcg(rows + r * stride)) continue;
        add_pair(sp, counts, n_counts, __ldcg(rows + r * stride + 1 + i));
    }
}

cudaError_t launch_counts_compact(const SparseView &sp, const uint32_t *counts, uint64_t n, unsigned long long *pairs,
                                  uint32_t cap, uint32_t *n_out, cudaStream_t st)
{
    if (!n) return cudaSuccess;
    if (sp.touched) k_touched_pairs<<<148 * 4, 256, 0, st>>>(sp, counts, pairs, cap, n_out);
    k_counts_compact<<<grid_for(n, 256, 148 * 8), 256, 0, st>>>(sp, counts, n, pairs, cap, n_out);
    return cudaGetLastError();
}

cudaError_t launch_counts_scatter_add(const SparseView &sp, uint32_t *counts, uint64_t n_counts,
                                      const unsigned long long *pairs, uint64_t n_pairs, cudaStream_t st)
{
    if (!n_pairs) return cudaSuccess;
    k_counts_scatter_add<<<grid_for(n_pairs, 256, 148 * 8), 256, 0, st>>>(sp, counts, n_counts, pairs, n_pairs);
    return cudaGetLastError();
}

cudaError_t launch_counts_absorb(const SparseView &sp, uint32_t *counts, uint64_t n_counts,
                                 const unsigned long long *rows, uint32_t n_rows, uint32_t cap, uint32_t skip,
                                 int sm_count, cudaStream_t st)
{
    if (!n_rows || !cap) return cudaSuccess;
    k_counts_absorb<<<(uint32_t)sm_count * 8u, 256, 0, st>>>(sp, counts, n_counts, rows, n_rows, cap, skip);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// Multi-GPU mixture: union of the ranks' bottom-s lists, its s smallest, and S10 -- on the device,
// so that the exchange needs no host round trip between the collectives and the reduction.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_mixture_gather(const unsigned long long *rows, uint32_t n_rows, uint32_t s_cap,
                                                        uint64_t *work, uint32_t work_cap, SparseState *st)
{
    // row r = [length | s_cap hashes]; the value 2^64-1 is a legal hash but also the sort's padding:
    // it is set aside here (st->mix_has_max = seen) and appended again after the unique pass
    const size_t stride = (size_t)s_cap + 1;
    for (uint32_t x = blockIdx.x * blockDim.x + threadIdx.x; x < work_cap; x += gridDim.x * blockDim.x) {
        uint64_t v = kEmptyKey;
        if (x < n_rows * s_cap) {
            const uint32_t r = x / s_cap, i = x % s_cap;
            const unsigned long long len64 = rows[r * stride];
            if (len64 == kMixUnsettled) { if (i == 0) atomicExch(&st->mix_unsettled, 1u); }   // that rank's selection fell through
            const uint32_t len = len64 == kMixUnsettled ? 0u : (uint32_t)min((unsigned long long)s_cap, len64);
            if (i < len) {
                v = rows[r * stride + 1 + i];
                if (v == kEmptyKey) atomicExch(&st->mix_has_max, 1u);
            }
        }
        work[x] = v;
    }
}

__global__ void k_mixture_finish(const uint64_t *sorted, const uint32_t *n_unique, uint32_t s, const uint32_t *seg_s,
                                 uint32_t n_seg, int use64, uint64_t *out, SparseState *st)
{
    uint32_t n = min(*n_unique, s);
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) out[i] = sorted[i];
    __syncthreads();
    if (threadIdx.x == 0) {
        if (st->mix_has_max && n < s) out[n++] = kEmptyKey;
        st->n_mix = n;
        for (uint32_t j = 0; j < n_seg && j < 8u; j++) {
            // S10: (uint64) (2^W * |M| / max(M)) in double, M = the seg_s[j] smallest
            const uint32_t m = min(n, seg_s[j]);
            unsigned long long v = 0;
            if (m) {
                const double est = ldexp(1.0, use64 ? 64 : 32) * (double)m / (double)out[m - 1];
                v = est < 18446744073709551615.0 ? (unsigned long long)est : ~0ull;
            }
            st->set_size[j] = v;
        }
    }
}

// the device-side selection's own verdict (the host applies the same test to the state it gets back)
__global__ void __launch_bounds__(256) k_mix_record(const MixView v, uint32_t s, uint32_t sel_pad, const uint64_t *cand,
                                                    unsigned long long *record, int force_unsettled)
{
    const MixState *st = v.st;
    const bool ok = !force_unsettled && !st->overflow && !st->sel_too_many && st->n_out <= sel_pad &&
                    (st->n_unique >= s || st->tau == ~0ull);
    uint32_t n = min(st->n_unique, s);
    for (uint32_t i = threadIdx.x; i < s; i += blockDim.x) record[1 + i] = (ok && i < n) ? cand[i] : 0ull;
    __syncthreads();
    if (threadIdx.x == 0) {
        if (ok && st->has_max && n < s) record[1 + n++] = kEmptyKey;   // hash == 2^64-1 present
        record[0] = ok ? (unsigned long long)n : kMixUnsettled;
    }
}

cudaError_t launch_mix_record(const MixView &v, uint32_t s, uint32_t sel_pad, const uint64_t *cand, unsigned long long *record,
                              int force_unsettled, cudaStream_t st)
{
    k_mix_record<<<1, 256, 0, st>>>(v, s, sel_pad, cand, record, force_unsettled);
    return cudaGetLastError();
}

cudaError_t launch_mixture_merge(const unsigned long long *rows, uint32_t n_rows, uint32_t s_cap, uint32_t s,
                                 const uint32_t *seg_s, uint32_t n_seg, bool use64, uint64_t *work, uint32_t work_cap,
                                 uint64_t *scratch, uint64_t *out, SparseState *st, cudaStream_t stm)
{
    if ((uint64_t)n_rows * s_cap > work_cap) return cudaErrorInvalidValue;
    static_assert(offsetof(SparseState, mix_unsettled) == offsetof(SparseState, mix_has_max) + 4, "cleared together");
    cudaError_t e = cudaMemsetAsync(&st->mix_has_max, 0, 2 * sizeof(uint32_t), stm);
    if (e != cudaSuccess) return e;
    k_mixture_gather<<<grid_for(work_cap, 256, 148 * 4), 256, 0, stm>>>(rows, n_rows, s_cap, work, work_cap, st);
    if ((e = launch_sort_unique(work, work_cap, scratch, &st->n_mix, stm)) != cudaSuccess) return e;
    k_mixture_finish<<<1, 256, 0, stm>>>(work, &st->n_mix, s, seg_s, n_seg, use64 ? 1 : 0, out, st);
    return cudaGetLastError();
}

}  // namespace hs
