// abi.cu -- the C ABI of libhymet_screen.so (include/hymet_screen.h): handle
// lifetimes, HBM layout, stream orchestration.  All arithmetic of the hot path runs
// in the kernels of screen_kernels.cu; the only host arithmetic here is control
// logic (thresholds, S10's one-line set-size formula, merging <= G*s mixture hashes).
// There is deliberately no CPU implementation of any kernel in this library.
#include <cuda_runtime.h>
#include <math.h>
#include <stddef.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <ctype.h>
#include <fcntl.h>
#include <sched.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/hymet_screen.h"
#include "fasta_pack.h"
#include "kmer_core.cuh"
#include "lca_kernels.h"
#include "msh_capnp.h"
#include "screen_kernels.h"

#define HS_API extern "C" __attribute__((visibility("default")))

using namespace hs;

namespace {

thread_local std::string g_err;
// hs_init() binds the CALLING THREAD: one thread per GPU can each build its own db (HYMET_SCREEN_GPUS)
thread_local int g_device = -1;
thread_local int g_sm = 0;
bool g_debug_timing = false;

int fail(int code, const std::string &msg)
{
    g_err = msg;
    return code;
}
#define CU(x)                                                                                         \
    do {                                                                                              \
        cudaError_t e_ = (x);                                                                         \
        if (e_ != cudaSuccess) return fail(HS_ECUDA, std::string(#x) + ": " + cudaGetErrorString(e_)); \
    } while (0)
// Entry points without a handle run on the device of the latest hs_init(); handles remember the
// device they were created on (one process may drive several GPUs, one db + screen per GPU).
#define NEED_DEVICE()                                                                                      \
    do {                                                                                                   \
        if (g_device < 0) return fail(HS_ENODEV, "hs_init() has not bound an sm_100 device (no CPU fallback)"); \
        CU(cudaSetDevice(g_device));                                                                       \
    } while (0)
#define ON_DEVICE(dev) CU(cudaSetDevice(dev))

// device allocations of a build step: freed on every return path unless released to their owner
struct DevBufs {
    std::vector<void *> p;
    template <class T> cudaError_t alloc(T **out, size_t bytes)
    {
        void *q = nullptr;
        cudaError_t e = cudaMalloc(&q, bytes ? bytes : 1);
        if (e == cudaSuccess) { p.push_back(q); *out = (T *)q; }
        return e;
    }
    ~DevBufs() { for (void *q : p) cudaFree(q); }
};

double now_s()
{
    return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

uint64_t tiles_for(uint64_t n_bases) { return ((n_bases + 31) / 32 + kTileWords - 1) / kTileWords; }

// ---- device arena for query chunks ------------------------------------------
struct Arena {
    struct Slab { char *p; size_t cap, used; };
    std::vector<Slab> slabs;
    size_t slab_bytes = (size_t)256 << 20;
    size_t total = 0, cur = 0;
    cudaError_t alloc(size_t n, void **out)
    {
        n = (n + 255) & ~(size_t)255;
        while (cur < slabs.size() && slabs[cur].used + n > slabs[cur].cap) cur++;
        if (cur == slabs.size()) {
            Slab s{nullptr, std::max(n, slab_bytes), 0};
            cudaError_t e = cudaMalloc((void **)&s.p, s.cap);
            if (e != cudaSuccess) return e;
            slabs.push_back(s);
            total += s.cap;
        }
        *out = slabs[cur].p + slabs[cur].used;
        slabs[cur].used += n;
        return cudaSuccess;
    }
    void reset()
    {   // slabs stay allocated: a steady-state screen never calls cudaMalloc/cudaFree
        for (auto &s : slabs) s.used = 0;
        cur = 0;
    }
    void release()
    {
        for (auto &s : slabs) cudaFree(s.p);
        slabs.clear();
        total = 0; cur = 0;
    }
};

struct Chunk {
    const uint64_t *d_seq;
    const uint32_t *d_inv;
    uint64_t n_bases;                                // exact, or an upper bound when n_dev is set
    const unsigned long long *n_dev = nullptr;       // device-parsed chunk: true length lives in HBM
};

// ---- device-side FASTA ingest: raw text slots + scan scratch ------------------------
struct Ingest {
    static constexpr int kSlots = 4;
    struct Slot { uint8_t *raw = nullptr, *codes = nullptr; size_t cap = 0; cudaEvent_t done = nullptr, copied = nullptr; };
    Slot slots[kSlots];
    int next = 0;
    FaScratch sc{};
    size_t tile_cap = 0;
    std::vector<unsigned long long *> counter_blocks;   // per-chunk position counters (512 per block)
    size_t counters_used = 0;
    unsigned long long *d_totals = nullptr;             // [0] positions [1] bases [2] records
    bool ready = false;

    int ensure(size_t bytes, cudaStream_t st)
    {
        if (!ready) {
            CU(cudaMalloc((void **)&d_totals, 4 * sizeof(unsigned long long)));
            // on the stream that will accumulate into it: the legacy default stream is not ordered
            // against a non-blocking stream
            CU(cudaMemsetAsync(d_totals, 0, 4 * sizeof(unsigned long long), st));
            for (auto &sl : slots) {
                CU(cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming | cudaEventBlockingSync));
                CU(cudaEventCreateWithFlags(&sl.copied, cudaEventDisableTiming));
            }
            ready = true;
        }
        const size_t tiles = (bytes + kFaTileBytes - 1) / kFaTileBytes + 1;
        if (tiles > tile_cap) {
            cudaDeviceSynchronize();
            cudaFree(sc.tile_event); cudaFree(sc.tile_carry); cudaFree(sc.tile_event_b); cudaFree(sc.tile_carry_b);
            cudaFree(sc.tile_count); cudaFree(sc.tile_offset); cudaFree(sc.masks); cudaFree(sc.emit);
            tile_cap = tiles + tiles / 4;
            CU(cudaMalloc((void **)&sc.masks, tile_cap * 256 * sizeof(uint4)));
            CU(cudaMalloc((void **)&sc.emit, tile_cap * 256 * sizeof(uint2)));
            CU(cudaMalloc((void **)&sc.tile_event, tile_cap * 4));
            CU(cudaMalloc((void **)&sc.tile_carry, tile_cap * 4));
            CU(cudaMalloc((void **)&sc.tile_event_b, tile_cap * 4));
            CU(cudaMalloc((void **)&sc.tile_carry_b, tile_cap * 4));
            CU(cudaMalloc((void **)&sc.tile_count, tile_cap * 4));
            CU(cudaMalloc((void **)&sc.tile_offset, tile_cap * 8));
        }
        sc.totals = d_totals;
        return HS_OK;
    }
    int slot_for(size_t bytes, Slot **out)
    {
        Slot &sl = slots[next];
        next = (next + 1) % kSlots;
        CU(cudaEventSynchronize(sl.done));  // throttle: at most kSlots chunks of raw text in flight
        if (sl.cap < bytes) {
            cudaFree(sl.raw); cudaFree(sl.codes);
            sl.cap = bytes + bytes / 8 + 64;
            CU(cudaMalloc((void **)&sl.raw, sl.cap));
            CU(cudaMalloc((void **)&sl.codes, sl.cap));
        }
        *out = &sl;
        return HS_OK;
    }
    int counter(unsigned long long **out)
    {
        if (counters_used == counter_blocks.size() * 512) {
            unsigned long long *b = nullptr;
            CU(cudaMalloc((void **)&b, 512 * sizeof(unsigned long long)));
            counter_blocks.push_back(b);
        }
        *out = counter_blocks[counters_used / 512] + counters_used % 512;
        counters_used++;
        return HS_OK;
    }
    void release()
    {
        for (auto &sl : slots) {
            cudaFree(sl.raw); cudaFree(sl.codes);
            if (sl.done) cudaEventDestroy(sl.done);
            if (sl.copied) cudaEventDestroy(sl.copied);
        }
        cudaFree(sc.tile_event); cudaFree(sc.tile_carry); cudaFree(sc.tile_event_b); cudaFree(sc.tile_carry_b);
        cudaFree(sc.tile_count); cudaFree(sc.tile_offset); cudaFree(sc.masks); cudaFree(sc.emit); cudaFree(d_totals);
        for (auto *b : counter_blocks) cudaFree(b);
    }
};

// ---- mixture bottom-s engine (K3 control logic) --------------------------------
// The threshold tau and the live set are DEVICE state (MixState): streaming launches and
// their maintenance kernels are enqueued back to back, the host looks at the state only
// at flush.  Exactness: a value is dropped only when >= s smaller distinct values stay.
struct MixEngine {
    uint32_t s = 0, cap = 0, cand_cap = 0;
    bool use64 = true;     // 32-bit hashes (k <= 16) live in [0, 2^32): caps and tau start there
    uint64_t *d_set[2] = {nullptr, nullptr};
    MixState *d_state = nullptr;
    MixState *h_state = nullptr;  // pinned mirror, valid after sync_state()
    uint64_t *d_cand = nullptr, *d_scratch = nullptr;
    uint32_t *d_hist = nullptr;   // device-side selection: 2048 bins
    uint32_t sel_pad = 0;         // its sort capacity (power of two >= s + slack, <= cand_cap)
    bool fast_select = true;
    uint64_t *h_cand = nullptr;   // pinned: the settled mixture travels with the state, one sync for both
    bool auto_tau = true;  // first pass: cap tau per launch so expected offers stay <= cap/8
    uint32_t passes = 1;

    int init(uint32_t s_, bool use64_ = true)
    {
        s = s_ ? s_ : 1;
        use64 = use64_;
        cap = 1u << 20;
        while ((uint64_t)cap < 64ull * s) cap <<= 1;
        cand_cap = 8192;
        while (cand_cap < 4 * s) cand_cap <<= 1;
        for (int i = 0; i < 2; i++) CU(cudaMalloc((void **)&d_set[i], (size_t)cap * 8));
        CU(cudaMalloc((void **)&d_state, sizeof(MixState)));
        CU(cudaHostAlloc((void **)&h_state, sizeof(MixState), cudaHostAllocDefault));
        CU(cudaMalloc((void **)&d_cand, (size_t)cand_cap * 8));
        CU(cudaMalloc((void **)&d_scratch, (size_t)cand_cap * 8));
        CU(cudaMalloc((void **)&d_hist, (2 * 2048 + 8) * sizeof(uint32_t)));   // bin counts | bin starts | last bin
        sel_pad = 2048;
        while (sel_pad < s + 1024) sel_pad <<= 1;
        if (sel_pad > cand_cap) sel_pad = cand_cap;
        if (const char *e = getenv("HYMET_SCREEN_FAST_SELECT")) fast_select = atoi(e) != 0;
        CU(cudaHostAlloc((void **)&h_cand, (size_t)s * 8, cudaHostAllocDefault));
        return HS_OK;
    }
    void destroy()
    {
        for (int i = 0; i < 2; i++) cudaFree(d_set[i]);
        cudaFree(d_state); cudaFree(d_cand); cudaFree(d_scratch); cudaFree(d_hist);
        if (h_state) cudaFreeHost(h_state);
        if (h_cand) cudaFreeHost(h_cand);
    }
    uint32_t *field(size_t off) const { return reinterpret_cast<uint32_t *>(reinterpret_cast<char *>(d_state) + off); }
    int reset(cudaStream_t st, uint64_t new_tau = ~0ull, bool automatic = true)
    {
        CU(cudaMemsetAsync(d_set[0], 0xFF, (size_t)cap * 8, st));
        CU(launch_mix_state_init(d_state, new_tau, st));
        auto_tau = automatic;  // a re-offer pass runs at exactly the tau the finaliser chose
        return HS_OK;
    }
    // cap for a launch over n positions: expected offers <= capacity/8
    uint64_t launch_cap(uint64_t n) const
    {
        const uint64_t budget = cap / 8, space = use64 ? ~0ull : 0xFFFFFFFFull;
        if (!auto_tau || n <= budget) return ~0ull;
        const uint64_t c = (uint64_t)((unsigned __int128)space * budget / n);
        return c < 256 ? 256 : c;
    }
    MixView view(uint64_t tau_cap) const
    {
        MixView v;
        v.sets[0] = d_set[0]; v.sets[1] = d_set[1];
        v.mask = cap - 1; v.limit = cap / 2; v.tau_cap = tau_cap; v.st = d_state;
        return v;
    }
    int sync_state(cudaStream_t st)
    {
        CU(cudaMemcpyAsync(h_state, d_state, sizeof(MixState), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        return HS_OK;
    }
};

}  // namespace

// =============================================================================
// handles
// =============================================================================
struct hs_msh { MshData d; };

struct hs_db {
    int device = 0, sm = 0;
    uint32_t k = 0, s = 0, seed = 42;
    bool use64 = true;
    uint64_t n_refs = 0, n_entries = 0, n_distinct = 0, max_key = 0, dense_max = 0;
    std::vector<std::string> names, comments;
    std::vector<uint64_t> lengths, offsets;
    uint64_t *d_buckets = nullptr;           // n_buckets x 128 bytes: keys | canonical entry ids | overflow flag
    uint32_t n_buckets = 0, special = kNoEntry;
    uint32_t *d_canon = nullptr;             // per stored hash: canonical entry id of its key (reference -> hashes, dense path)
    uint32_t *d_next = nullptr;              // per stored hash: next entry holding the same key (hash -> references, sparse path)
    uint64_t *d_offsets = nullptr, *d_lengths = nullptr, *d_seg_begin = nullptr;
    uint32_t *d_seg_s = nullptr;
    uint64_t device_bytes = 0;
    double t_parse = 0, t_build = 0;
    uint32_t *d_bloom = nullptr;
    uint32_t bloom_mask = 0;
    uint64_t bloom_keys = 0;                 // keys above dense_max (what the Bloom filter holds)
    // Several .msh files screened in one pass (run_hymet_cami.sh:85-97 streams the query three times):
    // references [seg_begin[j], seg_begin[j+1]) came from file j, whose sketch size was seg_s[j].
    std::vector<uint64_t> seg_begin;
    std::vector<uint32_t> seg_s;
    TableView view() const { return TableView{d_buckets, n_buckets, max_key, special, d_bloom, bloom_mask, d_bloom ? dense_max : max_key}; }
};

// pinned ring the file readers pread() into: two slots per reader thread
struct FileRing {
    char *base = nullptr;
    size_t slot_cap = 0;
    std::vector<cudaEvent_t> free_ev;   // recorded on the copy stream once a slot's text is in HBM
    void release()
    {
        if (base) cudaFreeHost(base);
        base = nullptr; slot_cap = 0;
        for (auto e : free_ev) cudaEventDestroy(e);
        free_ev.clear();
    }
};

struct Staging {
    uint64_t *seq = nullptr;
    uint32_t *inv = nullptr;
    uint64_t cap_words = 0;
    cudaEvent_t free_ev = nullptr;
};

struct hs_screen {
    hs_db *db = nullptr;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaStream_t copy_stream = nullptr;      // H2D of query chunks overlaps the kernels of earlier chunks
    std::vector<cudaEvent_t> copy_evs;
    size_t copy_ev_used = 0;
    Ingest ingest;
    int ingest_mode = 2;   // 0 = host packer only, 1 = device parser only, 2 = both compete for chunks (pinned text)
    uint64_t text_chunk = (uint64_t)256 << 20;   // gzip / stdin input: bytes inflated per hand-over to the packers
    FileRing ring;
    // plain FASTA files: nominal bytes per reader block and reader threads.  Pinning the ring costs
    // ~0.5 ms per MB once per handle (measured), which a one-shot `mash screen` pays in full: the
    // defaults keep it at 96 MB (1 GB file: ~50 ms + 40 ms); a long-lived handle is better off with
    // 8 readers x 16 MB (28 ms per GB, bench.py's e2e_file)
    uint64_t file_block = (uint64_t)8 << 20;
    int file_readers = 4;
    int file_mode = -1;   // plain FASTA files: 0 pread ring + device parser, 1 mmap + host packers, -1 by host capability
    std::mutex ingest_mu;                       // one thread at a time hands a span to the device parser
    std::mutex giant_mu;                        // records larger than a ring slot take the host path, one at a time
    uint32_t *d_counts = nullptr;
    unsigned long long *d_stats = nullptr;
    // O(present hashes) bookkeeping (SparseState): ids of the non-zero counts, references with hits,
    // their depth segments.  touched_valid: the list covers every non-zero count as far as the HOST
    // knows (a dense all-reduce into counts[] invalidates it; the device flags overflow and wraps).
    SparseState *d_sparse = nullptr, *h_sparse = nullptr;
    uint32_t *d_touched = nullptr, *d_hit = nullptr, *d_seg_start = nullptr, *d_seg_fill = nullptr, *d_plain = nullptr;
    uint32_t *d_depths = nullptr;
    uint32_t touched_cap = 0, pair_cap = 0;
    bool touched_valid = true, sparse_enabled = true;
    uint32_t last_reduce_dense = 0;
    // multi-GPU: mixture merged on the device (hs_screen_mixture_merge_device)
    uint64_t *d_mixture = nullptr, *d_merge_work = nullptr, *d_merge_scratch = nullptr, *h_mixture = nullptr;
    uint32_t merge_cap = 0;
    bool mixture_on_device = false;
    cudaEvent_t rst0 = nullptr, rst1 = nullptr;
    bool rst_pending = false;
    // result rows of the references with hits (hs_screen_finish_hits): pinned, host-mapped, written by the GPU
    char *h_rows = nullptr;
    HitRows rows_host{}, rows_dev{};
    std::vector<uint32_t> hit_order;   // indices into the rows, ascending by reference, shared > 0 only
    MixEngine mix;
    std::vector<uint64_t> mixture;  // settled s smallest distinct hashes, ascending
    bool flushed = false;
    bool flush_pending = false;   // hs_screen_flush_async: selection enqueued, verdict read after the next synchronisation
    bool flush_parsed = false;    // ... and it fetched the device parser's totals
    int force_unsettled = 0;      // tests: the next mixture record says "not settled" (HYMET_SCREEN_FORCE_UNSETTLED)
    uint32_t *d_shared = nullptr, *d_median = nullptr;
    double *d_identity = nullptr, *d_pvalue = nullptr;
    unsigned long long *d_best_score = nullptr, *d_best_len = nullptr;
    uint32_t *d_winner = nullptr;
    Arena arena;
    std::vector<Chunk> chunks;
    std::vector<Staging> staging;
    std::mutex mu;  // serialises arena + launches when packer threads feed concurrently
    bool filter = true;
    uint64_t chunk_text = (uint64_t)16 << 20;
    hs_stats_t st;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev_pool;
    size_t ev_used = 0;
    cudaEvent_t red0 = nullptr, red1 = nullptr, red2 = nullptr, red3 = nullptr;
    unsigned long long *h_stats = nullptr;   // pinned: [0, ST_COUNT) kernel counters, then 4 device-parser totals
    char *h_result = nullptr;   // pinned landing zone for the four result columns (24 B per sketch):
                                // a D2H copy into the caller's pageable arrays costs ~0.3 ms at N = 50 000
};

namespace {

// Two-tier pre-filter: where does the dense range end?  Sketches of ordinary genomes keep hashes
// below ~2^64 * s / genome k-mers; sketches of genomes with fewer than ~s k-mers (viruses, plasmids)
// reach up to 2^64.  Probing directly costs a DRAM line per k-mer <= T, the Bloom tier an L2 word per
// k-mer in (T, max_key] plus a probe per false positive.  T runs over the references' largest hashes;
// keys above T are estimated per reference as size * (1 - T / max) (uniform below its own max).
struct FilterPlan { uint64_t dense_max; uint64_t words; double keys_above; bool bloom; };

FilterPlan plan_filter(const hs_db *db, const uint64_t *hashes)
{
    FilterPlan best{db->max_key, 0, 0.0, false};
    const double kSpace = 18446744073709551616.0, kProbeCost = 8.0, kBloomCost = 1.0, kMaxBits = 32.0 * 8 * 1048576;   // <= 32 MB: it has to stay in L2 next to the streaming query (64 MB: 16 % of its reads went to DRAM, ncu r02)
    struct R { double mx, size; };
    std::vector<R> r;
    for (uint64_t i = 0; i < db->n_refs; i++)
        if (db->offsets[i + 1] > db->offsets[i])
            r.push_back({(double)hashes[db->offsets[i + 1] - 1], (double)(db->offsets[i + 1] - db->offsets[i])});
    if (r.empty()) return best;
    std::sort(r.begin(), r.end(), [](const R &a, const R &b) { return a.mx < b.mx; });
    double suf_size = 0, suf_ratio = 0;   // over references whose max lies above the candidate
    double best_cost = (double)db->max_key / kSpace * kProbeCost;   // no Bloom tier: probe everything in range
    std::vector<double> ss(r.size() + 1, 0.0), sr(r.size() + 1, 0.0);
    for (size_t i = r.size(); i-- > 0;) {
        suf_size += r[i].size; suf_ratio += r[i].size / std::max(r[i].mx, 1.0);
        ss[i] = suf_size; sr[i] = suf_ratio;
    }
    const size_t step = std::max<size_t>(1, r.size() / 4096);
    for (size_t i = 0; i + 1 < r.size(); i += step) {
        const double T = r[i].mx;
        const double above = std::max(0.0, ss[i + 1] - T * sr[i + 1]);
        double bits = 4096.0 * 32;
        while (bits < above * 16.0 && bits < kMaxBits) bits *= 2;
        const double fp = pow(1.0 - exp(-3.0 * above / bits), 3.0) * 1.5;   // blocked filter: somewhat worse than the textbook rate
        const double p_direct = T / kSpace, p_bloom = ((double)db->max_key - T) / kSpace;
        const double cost = p_direct * kProbeCost + p_bloom * (kBloomCost + fp * kProbeCost);
        if (cost < best_cost) { best_cost = cost; best = FilterPlan{(uint64_t)T, (uint64_t)(bits / 32), above, true}; }
    }
    return best;
}

int db_build(hs_db *db, const uint64_t *hashes)
{
    const double t0 = now_s();
    const uint64_t E = db->n_entries, N = db->n_refs;
    db->device = g_device; db->sm = g_sm;
    if (E > 0xFFFFFFF0ull) return fail(HS_EUNSUPPORTED, "more than 2^32 stored hashes");
    if (N > 0xFFFFFFF0ull) return fail(HS_EUNSUPPORTED, "more than 2^32 references");
    if (db->k == 0 || db->k > 32) return fail(HS_EUNSUPPORTED, "k-mer size must be 1..32");
    uint64_t nb = (E + 4) / 5 + 1;  // 10 slots per bucket -> load factor <= 0.5: 1.4 % of the buckets overflow (0.6: 4.3 %)
    if (nb < 16) nb = 16;
    if (nb > 0xFFFFFFF0ull) return fail(HS_EUNSUPPORTED, "hash table too large");
    db->n_buckets = (uint32_t)nb;
    db->max_key = 0;
    for (uint64_t i = 0; i < N; i++)
        if (db->offsets[i + 1] > db->offsets[i]) db->max_key = std::max(db->max_key, hashes[db->offsets[i + 1] - 1]);
    for (uint64_t i = 0; i < N; i++)  // ascending order is part of the format; verify instead of trusting
        for (uint64_t e = db->offsets[i] + 1; e < db->offsets[i + 1]; e++)
            if (hashes[e] <= hashes[e - 1]) return fail(HS_EFORMAT, "sketch hashes are not strictly ascending");
    if (db->seg_begin.empty()) { db->seg_begin = {0, N}; db->seg_s = {db->s}; }
    if (db->seg_s.size() > 8) return fail(HS_EUNSUPPORTED, "more than 8 sketch files in one table");

    DevBufs tmp;   // build scratch: released on every path out of here
    uint64_t *d_hashes = nullptr;
    uint32_t *d_flags = nullptr;
    unsigned long long *d_nd = nullptr;
    // the handle owns what it was given so far: hs_db_free() releases it if a later step fails
    CU(cudaMalloc((void **)&db->d_buckets, nb * kBucketWords * 8));
    CU(cudaMalloc((void **)&db->d_canon, std::max<uint64_t>(E, 1) * 4));
    CU(cudaMalloc((void **)&db->d_next, std::max<uint64_t>(E, 1) * 4));
    CU(cudaMalloc((void **)&db->d_offsets, (N + 1) * 8));
    CU(cudaMalloc((void **)&db->d_lengths, std::max<uint64_t>(N, 1) * 8));
    CU(cudaMalloc((void **)&db->d_seg_begin, db->seg_begin.size() * 8));
    CU(cudaMalloc((void **)&db->d_seg_s, db->seg_s.size() * 4));
    CU(tmp.alloc(&d_hashes, E * 8));
    CU(tmp.alloc(&d_flags, 2 * sizeof(uint32_t)));
    CU(tmp.alloc(&d_nd, sizeof(unsigned long long)));
    db->device_bytes = nb * kBucketWords * 8 + E * 8 + (N + 1) * 8 + N * 8;
    CU(cudaMemset(db->d_next, 0xFF, std::max<uint64_t>(E, 1) * 4));   // kNoEntry = end of chain
    CU(cudaMemset(d_flags, 0xFF, sizeof(uint32_t)));      // [0] special = kNoEntry
    CU(cudaMemset(d_flags + 1, 0, sizeof(uint32_t)));     // [1] fail
    CU(cudaMemset(d_nd, 0, sizeof(unsigned long long)));
    if (E) CU(cudaMemcpy(d_hashes, hashes, E * 8, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(db->d_offsets, db->offsets.data(), (N + 1) * 8, cudaMemcpyHostToDevice));
    if (N) CU(cudaMemcpy(db->d_lengths, db->lengths.data(), N * 8, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(db->d_seg_begin, db->seg_begin.data(), db->seg_begin.size() * 8, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(db->d_seg_s, db->seg_s.data(), db->seg_s.size() * 4, cudaMemcpyHostToDevice));
    CU(launch_table_insert(db->d_buckets, db->n_buckets, d_hashes, E, d_flags, d_flags + 1, 0));
    uint32_t flags[2];
    CU(cudaMemcpy(flags, d_flags, sizeof flags, cudaMemcpyDeviceToHost));
    if (flags[1]) return fail(HS_ECUDA, "hash table build failed (table full)");
    db->special = flags[0];
    if (db->special != kNoEntry) db->max_key = ~0ull;
    db->dense_max = db->max_key;
    {
        // Second tier: worth it when the range test lets more than ~1 % of uniformly distributed query
        // hashes through.
        const double pass = (double)db->max_key / 18446744073709551615.0;
        const FilterPlan plan = plan_filter(db, hashes);
        if (pass > 0.01 && plan.bloom && E) {
            uint64_t words = 4096;
            while (words < plan.words) words <<= 1;
            CU(cudaMalloc((void **)&db->d_bloom, words * 4));
            CU(cudaMemset(db->d_bloom, 0, words * 4));
            db->bloom_mask = (uint32_t)(words - 1);
            db->dense_max = plan.dense_max;
            db->bloom_keys = (uint64_t)plan.keys_above;
            CU(launch_bloom_build(db->d_bloom, db->bloom_mask, db->dense_max, db->use64, d_hashes, E, 0));
            db->device_bytes += words * 4;
        }
    }
    CU(launch_table_canon(db->view(), d_hashes, E, db->d_canon, db->d_next, d_nd, 0));
    unsigned long long nd = 0;
    CU(cudaMemcpy(&nd, d_nd, sizeof nd, cudaMemcpyDeviceToHost));
    db->n_distinct = nd;
    db->t_build = now_s() - t0;
    return HS_OK;
}

void fill_info(const hs_db *db, hs_db_info_t *o)
{
    memset(o, 0, sizeof *o);
    o->k = db->k; o->s = db->s; o->seed = db->seed; o->use64 = db->use64;
    o->n_refs = db->n_refs; o->n_entries = db->n_entries; o->n_distinct = db->n_distinct;
    o->n_buckets = db->n_buckets; o->max_key = db->max_key; o->device_bytes = db->device_bytes;
    o->bloom_bytes = db->d_bloom ? ((uint64_t)db->bloom_mask + 1) * 4 : 0;
    o->dense_max = db->d_bloom ? db->dense_max : db->max_key;
    o->bloom_keys = db->bloom_keys;
    o->t_parse_s = db->t_parse; o->t_build_s = db->t_build;
}

StreamArgs base_args(const Chunk &c, uint32_t k, uint32_t seed, bool use64)
{
    StreamArgs a;
    memset(&a, 0, sizeof a);
    a.seq = c.d_seq; a.inv = c.d_inv; a.n_bases = c.n_bases;
    a.n_tiles = (uint32_t)tiles_for(c.n_bases);
    a.k = (int)k; a.seed = seed; a.use64 = use64;
    return a;
}

// launch the streaming kernel for tiles [tile_begin, tile_end) of one chunk (caller holds s->mu);
// tile_end == 0 means the whole chunk
int launch_chunk(hs_screen *s, const Chunk &c, bool count, bool mix, uint64_t tile_begin = 0, uint64_t tile_end = 0)
{
    if (!c.n_bases) return HS_OK;
    if (tiles_for(c.n_bases) > 0xFFFFFFFFull) return fail(HS_EINVAL, "chunk too large");
    if (!tile_end) tile_end = tiles_for(c.n_bases);
    StreamArgs a = base_args(c, s->db->k, s->db->seed, s->db->use64);
    a.n_bases_dev = c.n_dev;
    a.tile_begin = (uint32_t)tile_begin; a.n_tiles = (uint32_t)tile_end;
    a.do_count = count; a.do_filter = s->filter; a.do_mix = mix;
    a.tab = s->db->view(); a.counts = s->d_counts;
    // the range test removes probes only when the keys are confined to a sliver of the hash range; a db
    // whose keys cover a quarter of it or more and has no Bloom tier probes for most k-mers: that is
    // the warp-cooperative kernel's job, as is "filter" = 0
    a.probe_all = !s->filter || (!s->db->d_bloom && s->db->max_key >= ((uint64_t)1 << 62));
    if (count && s->sparse_enabled) a.sparse = SparseView{s->d_touched, s->touched_cap, s->d_sparse};
    const uint64_t launch_positions = (tile_end - tile_begin) * kTileWords * 32;
    a.mix = s->mix.view(mix ? s->mix.launch_cap(launch_positions) : ~0ull);
    a.stats = count ? s->d_stats : s->d_stats + ST_COUNT;  // re-offer passes must not double count
    if (s->ev_used == s->ev_pool.size()) {
        cudaEvent_t e0, e1;
        CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
        s->ev_pool.emplace_back(e0, e1);
    }
    auto &ev = s->ev_pool[s->ev_used++];
    CU(cudaEventRecord(ev.first, s->stream));
    CU(launch_stream(a, s->db->sm, s->stream));
    CU(cudaEventRecord(ev.second, s->stream));
    s->st.n_launches++;
    if (mix) {
        CU(launch_mix_maintain(a.mix, s->stream));
        s->st.n_launches += 3;
    }
    if (!c.n_dev)  // device-parsed chunks are accounted from the parser's own totals at flush
        s->st.n_positions += std::min<uint64_t>(c.n_bases, tile_end * kTileWords * 32) - tile_begin * kTileWords * 32;
    return HS_OK;
}

SparseView sparse_view(const hs_screen *s) { return SparseView{s->sparse_enabled ? s->d_touched : nullptr, s->touched_cap, s->d_sparse}; }

int screen_zero(hs_screen *s)
{
    CU(cudaEventRecord(s->rst0, s->stream));
    if (s->sparse_enabled && s->touched_valid) {
        // counts[] back to zero in O(touched); if the list overflowed on the device, the conditional
        // dense clear does the work instead (both are enqueued, one of them returns at once)
        CU(launch_sparse_reset(sparse_view(s), s->d_counts, s->db->sm, s->stream));
        CU(launch_counts_clear_if_overflow(sparse_view(s), s->d_counts, s->db->n_entries, s->stream));
    } else {
        CU(cudaMemsetAsync(s->d_counts, 0, std::max<uint64_t>(s->db->n_entries, 1) * 4, s->stream));
    }
    CU(cudaMemsetAsync(s->d_sparse, 0, sizeof(SparseState), s->stream));
    s->touched_valid = true;
    s->mixture_on_device = false;
    CU(cudaMemsetAsync(s->d_stats, 0, 2 * ST_COUNT * sizeof(unsigned long long), s->stream));
    int rc = s->mix.reset(s->stream);
    if (rc) return rc;
    CU(cudaEventRecord(s->rst1, s->stream));
    s->rst_pending = true;
    s->mix.passes = 1;
    s->mixture.clear();
    s->flushed = false;
    s->flush_pending = false;
    s->chunks.clear();
    if (s->copy_stream) CU(cudaStreamSynchronize(s->copy_stream));
    s->arena.reset();
    s->ev_used = 0;
    s->copy_ev_used = 0;
    s->ingest.counters_used = 0;
    if (s->ingest.ready) CU(cudaMemsetAsync(s->ingest.d_totals, 0, 4 * sizeof(unsigned long long), s->stream));
    memset(&s->st, 0, sizeof s->st);
    return HS_OK;
}

// Settle the s smallest distinct hashes of everything streamed so far (K3).
// rehash(tau) re-offers every resident chunk to a fresh set when the set lost
// elements (overflow) or tau was lowered further than the data supports.
template <class Rehash>
int mix_finalize(MixEngine &m, cudaStream_t st, std::vector<uint64_t> &out, uint32_t &n_launches, Rehash &&rehash)
{
    if (m.fast_select) {
        // Common case in ONE synchronisation: the device picks the threshold (histogram of the live set),
        // collects, sorts and dedups; state and the s smallest come back together.  Anything unusual --
        // the set overflowed, fewer than s values below tau, a crowded histogram bin -- is left to the
        // iterative path below, which starts from the same device state.
        CU(launch_mix_select(m.view(~0ull), m.s, m.use64, m.d_hist, m.d_cand, m.sel_pad, m.d_scratch, st));
        n_launches += 4;
        CU(cudaMemcpyAsync(m.h_cand, m.d_cand, (size_t)m.s * 8, cudaMemcpyDeviceToHost, st));
        int rc = m.sync_state(st);
        if (rc) return rc;
        const MixState &hs_ = *m.h_state;
        if (!hs_.overflow && !hs_.sel_too_many && hs_.n_out <= m.sel_pad && (hs_.n_unique >= m.s || hs_.tau == ~0ull)) {
            const uint32_t nu = std::min(hs_.n_unique, m.s);
            out.assign(m.h_cand, m.h_cand + nu);
            if (hs_.has_max && out.size() < m.s) out.push_back(~0ull);  // hash == 2^64-1 present
            return HS_OK;
        }
    }
    for (int round = 0; round < 40; round++) {
        int rc = m.sync_state(st);
        if (rc) return rc;
        if (m.h_state->overflow) {  // too many distinct values below tau: lower it and re-offer
            const uint64_t nt = m.h_state->tau >> 4;
            rc = m.reset(st, nt ? nt : 1, false);
            if (rc) return rc;
            m.passes++;
            rc = rehash();
            if (rc) return rc;
            continue;
        }
        const uint64_t tau = m.h_state->tau;
        const uint64_t *live = m.d_set[m.h_state->cur & 1u];
        // distinct values <= tau (older, larger ones may linger from before tau dropped)
        uint64_t thr = tau;
        uint32_t M = 0;
        for (int iter = 0; iter < 64; iter++) {
            CU(cudaMemsetAsync(m.field(offsetof(MixState, n_out)), 0, sizeof(uint32_t), st));
            CU(launch_mix_collect(live, m.cap, thr, m.d_cand, m.cand_cap, m.field(offsetof(MixState, n_out)), st));
            n_launches++;
            rc = m.sync_state(st);
            if (rc) return rc;
            M = m.h_state->n_out;
            if (M <= m.cand_cap && (M >= m.s || thr == tau)) break;
            if (M > m.cand_cap) {
                // aim for ~1.5 s candidates assuming hashes are uniform below thr
                const long double f = ((long double)m.s * 1.5L + 64.0L) / (long double)M;
                thr = (uint64_t)((long double)thr * (f < 0.9L ? f : 0.9L));
            } else {
                thr = (thr > tau / 2) ? tau : thr * 2;
            }
        }
        if (M > m.cand_cap) return fail(HS_ECUDA, "mixture candidate selection did not converge");
        if (M < m.s && tau != ~0ull) {
            // complete below tau but fewer than s distinct values there (very repetitive
            // input): raise tau and re-offer everything
            const uint64_t nt = (tau > (~0ull >> 4)) ? ~0ull : (tau ? tau << 4 : 16);
            rc = m.reset(st, nt, false);
            if (rc) return rc;
            m.passes++;
            rc = rehash();
            if (rc) return rc;
            continue;
        }
        out.clear();
        if (M) {
            CU(launch_sort_unique(m.d_cand, M, m.d_scratch, m.field(offsetof(MixState, n_unique)), st));
            n_launches++;
            const uint32_t take = std::min(M, m.s);   // >= what is kept (n_unique <= M)
            CU(cudaMemcpyAsync(m.h_cand, m.d_cand, (size_t)take * 8, cudaMemcpyDeviceToHost, st));
            rc = m.sync_state(st);
            if (rc) return rc;
            const uint32_t nu = std::min(m.h_state->n_unique, take);
            out.assign(m.h_cand, m.h_cand + nu);
        }
        if (m.h_state->has_max && out.size() < m.s) out.push_back(~0ull);  // hash == 2^64-1 present
        return HS_OK;
    }
    return fail(HS_ECUDA, "mixture threshold search did not settle");
}

uint64_t set_size_of(const std::vector<uint64_t> &mix, bool use64, uint64_t s_limit = ~0ull)
{   // S10: (uint64) (2^W * |M| / max(M)), W = 64 or 32, in double; M = the s_limit smallest of mix
    const uint64_t n = std::min<uint64_t>(mix.size(), s_limit);
    if (!n) return 0;
    const double est = pow(2.0, use64 ? 64.0 : 32.0) * (double)n / (double)mix[n - 1];
    if (!(est < 18446744073709551615.0)) return ~0ull;
    return (uint64_t)est;
}

int collect_stream_ms(hs_screen *s)
{
    float total = 0;
    for (size_t i = 0; i < s->ev_used; i++) {
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, s->ev_pool[i].first, s->ev_pool[i].second));
        total += ms;
    }
    s->st.ms_stream = total;
    return HS_OK;
}

}  // namespace

// =============================================================================
// library
// =============================================================================
HS_API const char *hs_version(void) { return "hymet-screen-b200 0.1 (sm_100a)"; }
HS_API const char *hs_last_error(void) { return g_err.c_str(); }
HS_API int hs_sm_count(void) { return g_sm; }

namespace {
// Host side of the feed path: the packer/reader threads and the pinned buffers they fill should sit on
// the NUMA node the GPU hangs off -- on a two-socket 8-GPU box a rank whose pinned text lives on the
// other socket pulls it across the inter-socket link (round 1: 8 ranks together read host memory at
// 174 GB/s, a third of what eight PCIe 5 x16 links carry).  Threads inherit the caller's affinity
// and pinned pages are placed on first touch, so narrowing THIS thread's CPU set to the GPU's node
// (never widening it, never leaving it empty) is enough.  HYMET_SCREEN_NUMA=0 leaves it alone.
int g_numa_node = -1, g_numa_cpus = 0;
void bind_to_gpu_numa_node(int device)
{
    g_numa_node = -1; g_numa_cpus = 0;
    if (const char *e = getenv("HYMET_SCREEN_NUMA")) if (atoi(e) == 0) return;
    char bus[32] = {0};
    if (cudaDeviceGetPCIBusId(bus, sizeof bus, device) != cudaSuccess) { cudaGetLastError(); return; }
    for (char *c = bus; *c; c++) *c = (char)tolower(*c);
    char path[160];
    snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", bus);
    FILE *f = fopen(path, "r");
    if (!f) return;
    int node = -1;
    if (fscanf(f, "%d", &node) != 1) node = -1;
    fclose(f);
    if (node < 0) return;
    snprintf(path, sizeof path, "/sys/devices/system/node/node%d/cpulist", node);
    f = fopen(path, "r");
    if (!f) return;
    char list[4096] = {0};
    const bool ok = fgets(list, sizeof list, f) != nullptr;
    fclose(f);
    if (!ok) return;
    cpu_set_t cur, want;
    CPU_ZERO(&want);
    if (sched_getaffinity(0, sizeof cur, &cur) != 0) return;
    for (char *tok = strtok(list, ",\n"); tok; tok = strtok(nullptr, ",\n")) {
        int a = 0, b = 0;
        const int k = sscanf(tok, "%d-%d", &a, &b);
        if (k == 1) b = a;
        if (k < 1) continue;
        for (int c = a; c <= b && c < CPU_SETSIZE; c++)
            if (CPU_ISSET(c, &cur)) CPU_SET(c, &want);
    }
    const int n = CPU_COUNT(&want);
    if (n < 1 || n == CPU_COUNT(&cur)) { g_numa_node = node; g_numa_cpus = CPU_COUNT(&cur); return; }   // nothing to narrow
    if (sched_setaffinity(0, sizeof want, &want) == 0) { g_numa_node = node; g_numa_cpus = n; }
}
}  // namespace

HS_API int hs_host_placement(int *numa_node, int *cpus)
{
    if (numa_node) *numa_node = g_numa_node;
    if (cpus) *cpus = g_numa_cpus;
    return HS_OK;
}

HS_API int hs_init(int device)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(HS_ENODEV, std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "count is 0") +
                                   " (this library has no CPU fallback)");
    if (device < 0 || device >= n) return fail(HS_EINVAL, "device ordinal out of range");
    cudaDeviceProp p;
    CU(cudaGetDeviceProperties(&p, device));
    if (p.major != 10)
        return fail(HS_ENODEV, std::string("device ") + p.name + " is sm_" + std::to_string(p.major) + std::to_string(p.minor) +
                                   "; this build carries sm_100a code only");
    CU(cudaSetDevice(device));
    if (g_device != device) bind_to_gpu_numa_node(device);
    g_device = device;
    g_sm = p.multiProcessorCount;
    g_debug_timing = getenv("HYMET_SCREEN_DEBUG_TIMING") != nullptr;
    return HS_OK;
}

// =============================================================================
// .msh on the host
// =============================================================================
HS_API int hs_msh_open(const char *path, hs_msh **out)
{
    if (!path || !out) return fail(HS_EINVAL, "null argument");
    auto *m = new hs_msh();
    std::string err;
    int rc = msh_read(path, m->d, err);
    if (rc) { delete m; return fail(rc, err); }
    *out = m;
    return HS_OK;
}
HS_API int hs_msh_info(const hs_msh *m, hs_db_info_t *info)
{
    if (!m || !info) return fail(HS_EINVAL, "null argument");
    memset(info, 0, sizeof *info);
    info->k = m->d.k; info->s = m->d.s; info->seed = m->d.seed; info->use64 = m->d.use64;
    info->n_refs = m->d.offsets.size() - 1; info->n_entries = m->d.hashes.size();
    info->t_parse_s = m->d.t_parse_s;
    for (uint64_t h : m->d.hashes) info->max_key = std::max(info->max_key, h);
    return HS_OK;
}
HS_API int hs_msh_ref(const hs_msh *m, uint64_t i, const char **name, const char **comment, uint64_t *length,
                      uint64_t *n_hashes, const uint64_t **hashes)
{
    if (!m || i + 1 >= m->d.offsets.size()) return fail(HS_EINVAL, "reference index out of range");
    if (name) *name = m->d.names[i].c_str();
    if (comment) *comment = m->d.comments[i].c_str();
    if (length) *length = m->d.lengths[i];
    if (n_hashes) *n_hashes = m->d.offsets[i + 1] - m->d.offsets[i];
    if (hashes) *hashes = m->d.hashes.data() + m->d.offsets[i];
    return HS_OK;
}
HS_API void hs_msh_free(hs_msh *m) { delete m; }

// =============================================================================
// database on the GPU
// =============================================================================
HS_API int hs_db_from_msh(const hs_msh *m, hs_db **out)
{
    if (!m || !out) return fail(HS_EINVAL, "null argument");
    NEED_DEVICE();
    auto *db = new hs_db();
    db->k = m->d.k; db->s = m->d.s; db->seed = m->d.seed; db->use64 = m->d.use64;
    db->n_refs = m->d.offsets.size() - 1; db->n_entries = m->d.hashes.size();
    db->names = m->d.names; db->comments = m->d.comments; db->lengths = m->d.lengths; db->offsets = m->d.offsets;
    db->t_parse = m->d.t_parse_s;
    int rc = db_build(db, m->d.hashes.data());
    if (rc) { hs_db_free(db); return rc; }
    *out = db;
    return HS_OK;
}

HS_API int hs_db_from_msh_multi(const hs_msh *const *ms, uint32_t n, hs_db **out)
{
    if (!ms || !n || !out) return fail(HS_EINVAL, "null argument");
    NEED_DEVICE();
    for (uint32_t j = 0; j < n; j++) {
        if (!ms[j]) return fail(HS_EINVAL, "null sketch handle");
        if (ms[j]->d.k != ms[0]->d.k || ms[j]->d.seed != ms[0]->d.seed || ms[j]->d.use64 != ms[0]->d.use64)
            return fail(HS_EUNSUPPORTED, "sketch files differ in k-mer size, seed or hash width: screen them one at a time");
    }
    auto *db = new hs_db();
    db->k = ms[0]->d.k; db->seed = ms[0]->d.seed; db->use64 = ms[0]->d.use64;
    std::vector<uint64_t> hashes;
    db->offsets.push_back(0);
    db->seg_begin.push_back(0);
    for (uint32_t j = 0; j < n; j++) {
        const MshData &d = ms[j]->d;
        db->s = std::max(db->s, d.s);       // the mixture keeps max s; each file's set size uses its own prefix (S9, S10)
        db->t_parse += d.t_parse_s;
        const uint64_t base = hashes.size();
        hashes.insert(hashes.end(), d.hashes.begin(), d.hashes.end());
        for (size_t i = 1; i < d.offsets.size(); i++) db->offsets.push_back(base + d.offsets[i]);
        db->names.insert(db->names.end(), d.names.begin(), d.names.end());
        db->comments.insert(db->comments.end(), d.comments.begin(), d.comments.end());
        db->lengths.insert(db->lengths.end(), d.lengths.begin(), d.lengths.end());
        db->seg_begin.push_back(db->offsets.size() - 1);
        db->seg_s.push_back(d.s);
    }
    db->n_refs = db->offsets.size() - 1; db->n_entries = hashes.size();
    int rc = db_build(db, hashes.data());
    if (rc) { hs_db_free(db); return rc; }
    *out = db;
    return HS_OK;
}

HS_API int hs_db_segments(const hs_db *db, uint32_t *n_segments, uint64_t *ref_begin, uint32_t *seg_s)
{
    if (!db || !n_segments) return fail(HS_EINVAL, "null argument");
    *n_segments = (uint32_t)db->seg_s.size();
    if (ref_begin) memcpy(ref_begin, db->seg_begin.data(), db->seg_begin.size() * 8);
    if (seg_s) memcpy(seg_s, db->seg_s.data(), db->seg_s.size() * 4);
    return HS_OK;
}

HS_API int hs_db_load_msh(const char *path, hs_db **out)
{
    hs_msh *m = nullptr;
    int rc = hs_msh_open(path, &m);
    if (rc) return rc;
    rc = hs_db_from_msh(m, out);
    hs_msh_free(m);
    return rc;
}

HS_API int hs_db_from_arrays(uint32_t k, uint32_t s, uint32_t seed, uint64_t n_refs, const uint64_t *offsets,
                             const uint64_t *hashes, const uint64_t *lengths, hs_db **out)
{
    if (!offsets || !out || (!hashes && offsets[n_refs])) return fail(HS_EINVAL, "null argument");
    NEED_DEVICE();
    auto *db = new hs_db();
    db->k = k; db->s = s; db->seed = seed;
    db->use64 = pow(4.0, (double)k) > pow(2.0, 32.0);
    db->n_refs = n_refs; db->n_entries = offsets[n_refs];
    db->offsets.assign(offsets, offsets + n_refs + 1);
    if (lengths) db->lengths.assign(lengths, lengths + n_refs); else db->lengths.assign(n_refs, 0);
    db->names.assign(n_refs, std::string()); db->comments.assign(n_refs, std::string());
    int rc = db_build(db, hashes);
    if (rc) { hs_db_free(db); return rc; }
    *out = db;
    return HS_OK;
}

HS_API int hs_db_info(const hs_db *db, hs_db_info_t *info)
{
    if (!db || !info) return fail(HS_EINVAL, "null argument");
    fill_info(db, info);
    return HS_OK;
}
HS_API int hs_db_ref(const hs_db *db, uint64_t i, const char **name, const char **comment, uint64_t *length,
                     uint64_t *n_hashes)
{
    if (!db || i >= db->n_refs) return fail(HS_EINVAL, "reference index out of range");
    if (name) *name = db->names[i].c_str();
    if (comment) *comment = db->comments[i].c_str();
    if (length) *length = db->lengths[i];
    if (n_hashes) *n_hashes = db->offsets[i + 1] - db->offsets[i];
    return HS_OK;
}
HS_API void hs_db_free(hs_db *db)
{
    if (!db) return;
    cudaSetDevice(db->device);
    cudaFree(db->d_buckets); cudaFree(db->d_canon); cudaFree(db->d_next); cudaFree(db->d_offsets); cudaFree(db->d_lengths);
    cudaFree(db->d_seg_begin); cudaFree(db->d_seg_s); cudaFree(db->d_bloom);
    delete db;
}

// =============================================================================
// screen
// =============================================================================
HS_API int hs_screen_new(hs_db *db, hs_screen **out)
{
    if (!db || !out) return fail(HS_EINVAL, "null argument");
    ON_DEVICE(db->device);
    auto *s = new hs_screen();
    s->db = db;
    const uint64_t N = std::max<uint64_t>(db->n_refs, 1), E = std::max<uint64_t>(db->n_entries, 1);
    const uint64_t E4 = (E + 3) / 4 * 4;
    auto bail = [&](int rc) { hs_screen_free(s); return rc; };
#define CUB(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { fail(HS_ECUDA, std::string(#x) + ": " + cudaGetErrorString(e_)); return bail(HS_ECUDA); } } while (0)
    CUB(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
    s->own_stream = true;
    CUB(cudaStreamCreateWithFlags(&s->copy_stream, cudaStreamNonBlocking));
    CUB(cudaMalloc((void **)&s->d_counts, E4 * 4));
    CUB(cudaMemsetAsync(s->d_counts, 0, E4 * 4, s->stream));
    CUB(cudaMalloc((void **)&s->d_stats, 2 * ST_COUNT * sizeof(unsigned long long)));
    // the four result columns share one allocation (identity | p-value | shared | median) so that
    // they travel to the host in a single copy
    CUB(cudaMalloc((void **)&s->d_identity, N * 24));
    s->d_pvalue = s->d_identity + N;
    s->d_shared = reinterpret_cast<uint32_t *>(s->d_pvalue + N);
    s->d_median = s->d_shared + N;
    // sparse bookkeeping: room for one hash in eight to be present (a metagenome touches a small part
    // of a RefSeq-sized table); beyond that the dense kernels take over
    s->touched_cap = (uint32_t)std::min<uint64_t>(E, std::max<uint64_t>((uint64_t)1 << 22, E / 8));
    s->pair_cap = (uint32_t)std::min<uint64_t>(E, std::max<uint64_t>((uint64_t)1 << 23, E / 4));
    if (const char *e = getenv("HYMET_SCREEN_TOUCHED_CAP")) s->touched_cap = (uint32_t)std::max(1ll, atoll(e));   // tests: force the fallbacks
    if (const char *e = getenv("HYMET_SCREEN_PAIR_CAP")) s->pair_cap = (uint32_t)std::max(1ll, atoll(e));
    if (const char *e = getenv("HYMET_SCREEN_FORCE_UNSETTLED")) s->force_unsettled = atoi(e);
    CUB(cudaMalloc((void **)&s->d_sparse, sizeof(SparseState)));
    CUB(cudaMemsetAsync(s->d_sparse, 0, sizeof(SparseState), s->stream));
    CUB(cudaHostAlloc((void **)&s->h_sparse, sizeof(SparseState), cudaHostAllocDefault));
    CUB(cudaMalloc((void **)&s->d_touched, (size_t)s->touched_cap * 4));
    CUB(cudaMalloc((void **)&s->d_depths, (size_t)s->pair_cap * 4));
    CUB(cudaMalloc((void **)&s->d_hit, N * 16));   // hit | seg_start | seg_fill | plain
    s->d_seg_start = s->d_hit + N; s->d_seg_fill = s->d_seg_start + N; s->d_plain = s->d_seg_fill + N;
    CUB(cudaEventCreate(&s->red0));
    CUB(cudaEventCreate(&s->red1));
    CUB(cudaEventCreate(&s->red2));
    CUB(cudaEventCreate(&s->red3));
    CUB(cudaEventCreate(&s->rst0));
    CUB(cudaEventCreate(&s->rst1));
    CUB(cudaHostAlloc((void **)&s->h_result, N * 24, cudaHostAllocDefault));
    CUB(cudaHostAlloc((void **)&s->h_stats, (ST_COUNT + 4) * sizeof(unsigned long long), cudaHostAllocDefault));
    CUB(cudaHostAlloc((void **)&s->h_mixture, ((size_t)db->s + 1) * 8, cudaHostAllocDefault));
#undef CUB
    int rc = s->mix.init(db->s, db->use64);
    if (rc) return bail(rc);
    s->touched_valid = false;   // nothing recorded yet and counts[] was just cleared: screen_zero need not walk a list
    rc = screen_zero(s);
    if (rc) return bail(rc);
    *out = s;
    return HS_OK;
}

HS_API int hs_screen_set_stream(hs_screen *s, void *cuda_stream)
{
    if (!s) return fail(HS_EINVAL, "null handle");
    ON_DEVICE(s->db->device);
    CU(cudaStreamSynchronize(s->stream));
    if (s->own_stream) { cudaStreamDestroy(s->stream); s->own_stream = false; }
    if (cuda_stream) {
        s->stream = (cudaStream_t)cuda_stream;
    } else {
        CU(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
        s->own_stream = true;
    }
    return HS_OK;
}

HS_API int hs_screen_set_option(hs_screen *s, const char *key, int64_t value)
{
    if (!s || !key) return fail(HS_EINVAL, "null argument");
    if (!strcmp(key, "filter")) s->filter = value != 0;
    else if (!strcmp(key, "chunk_bases")) s->chunk_text = value > 4096 ? (uint64_t)value : 4096;
    else if (!strcmp(key, "ingest")) s->ingest_mode = (int)value;
    else if (!strcmp(key, "text_chunk_bytes")) s->text_chunk = value > 4096 ? (uint64_t)value : 4096;
    else if (!strcmp(key, "file_block_bytes")) s->file_block = value > 65536 ? (uint64_t)value : 65536;
    else if (!strcmp(key, "file_mode")) s->file_mode = value < 0 ? -1 : (value ? 1 : 0);
    else if (!strcmp(key, "file_readers")) s->file_readers = value < 1 ? 1 : (value > 16 ? 16 : (int)value);
    else if (!strcmp(key, "sparse")) { s->sparse_enabled = value != 0; s->touched_valid = false; }
    else return fail(HS_EINVAL, std::string("unknown option ") + key);
    return HS_OK;
}

HS_API uint64_t hs_packed_words(uint64_t n_bases) { return tiles_for(n_bases) * kTileWords; }

HS_API int hs_pack_text(const char *text, size_t n, uint64_t *seq2, uint32_t *inv, uint64_t cap_words,
                        uint64_t *n_bases, hs_stats_t *stats)
{
    if ((!text && n) || !seq2 || !inv || !n_bases) return fail(HS_EINVAL, "null argument");
    if (cap_words < pack_words_bound(n)) return fail(HS_EINVAL, "capacity below hs pack bound (n/32 + 4 words)");
    PackStats ps;
    pack_text_span(text, n, seq2, inv, &ps);
    *n_bases = ps.n_positions;
    if (stats) { memset(stats, 0, sizeof *stats); stats->n_bases = ps.n_seq_bases; stats->n_records = ps.n_records; stats->n_positions = ps.n_positions; }
    return HS_OK;
}

namespace {

constexpr uint64_t kPieceWords = ((uint64_t)32 << 20) / 32;   // 32 Mi positions per piece, a whole number of tiles
static_assert(kPieceWords % kTileWords == 0, "pieces must be whole tiles");

// copy a packed host chunk into the arena (padding flagged invalid) and launch it, in
// pieces: the copy of piece i+1 (copy stream) overlaps the kernel of piece i (compute stream)
int feed_host_chunk(hs_screen *s, const uint64_t *seq, const uint32_t *inv, uint64_t n_bases, cudaEvent_t done_ev)
{
    if (!n_bases) return HS_OK;
    const uint64_t words = (n_bases + 31) / 32, alloc = hs_packed_words(n_bases);
    void *dseq = nullptr, *dinv = nullptr;
    CU(s->arena.alloc(alloc * 8, &dseq));
    CU(s->arena.alloc(alloc * 4, &dinv));
    Chunk c{(const uint64_t *)dseq, (const uint32_t *)dinv, n_bases};
    s->chunks.push_back(c);
    s->st.h2d_bytes += words * 12;
    for (uint64_t w0 = 0; w0 < alloc; w0 += kPieceWords) {
        const uint64_t w1 = std::min(alloc, w0 + kPieceWords);      // tile aligned
        const uint64_t cw1 = std::min(words, w1);                   // words that exist in the host buffer
        if (cw1 > w0) {
            CU(cudaMemcpyAsync((char *)dseq + w0 * 8, seq + w0, (cw1 - w0) * 8, cudaMemcpyHostToDevice, s->copy_stream));
            CU(cudaMemcpyAsync((char *)dinv + w0 * 4, inv + w0, (cw1 - w0) * 4, cudaMemcpyHostToDevice, s->copy_stream));
        }
        if (w1 > cw1) {
            const uint64_t p0 = std::max(cw1, w0);
            CU(cudaMemsetAsync((char *)dseq + p0 * 8, 0, (w1 - p0) * 8, s->copy_stream));
            CU(cudaMemsetAsync((char *)dinv + p0 * 4, 0xFF, (w1 - p0) * 4, s->copy_stream));
        }
        if (s->copy_ev_used == s->copy_evs.size()) {
            cudaEvent_t e;
            CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            s->copy_evs.push_back(e);
        }
        cudaEvent_t ev = s->copy_evs[s->copy_ev_used++];
        CU(cudaEventRecord(ev, s->copy_stream));
        CU(cudaStreamWaitEvent(s->stream, ev, 0));
        int rc = launch_chunk(s, c, true, true, w0 / kTileWords, w1 / kTileWords);
        if (rc) return rc;
    }
    if (done_ev) CU(cudaEventRecord(done_ev, s->copy_stream));  // the host buffer may be reused
    return HS_OK;
}

// Row a6 on the GPU: upload one record-aligned span of raw FASTA text, parse + pack it on
// the device, stream it.  Everything is enqueued; the host only waits for a free slot.
int feed_span_device(hs_screen *s, const char *text, size_t len, cudaEvent_t host_free_ev = nullptr)
{
    if (!len) return HS_OK;
    if (len >= ((size_t)1 << 30)) return fail(HS_EINVAL, "text chunk too large for the device parser");
    Ingest &in = s->ingest;
    Ingest::Slot *sl = nullptr;
    {
        std::lock_guard<std::mutex> lk(s->mu);
        int rc = in.ensure(len, s->stream);
        if (rc) return rc;
    }
    int rc = in.slot_for(len, &sl);   // may wait for the GPU (outside the lock)
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(s->mu);
    unsigned long long *d_npos = nullptr;
    rc = in.counter(&d_npos);
    if (rc) return rc;
    const uint64_t alloc = hs_packed_words(len);      // positions <= bytes
    void *dseq = nullptr, *dinv = nullptr;
    CU(s->arena.alloc(alloc * 8, &dseq));
    CU(s->arena.alloc(alloc * 4, &dinv));
    CU(cudaMemcpyAsync(sl->raw, text, len, cudaMemcpyHostToDevice, s->copy_stream));
    CU(cudaEventRecord(sl->copied, s->copy_stream));
    if (host_free_ev) CU(cudaEventRecord(host_free_ev, s->copy_stream));
    CU(cudaStreamWaitEvent(s->stream, sl->copied, 0));
    FaScratch sc = in.sc;
    sc.chunk_positions = d_npos;
    CU(launch_fasta_to_codes(sl->raw, (uint32_t)len, sl->codes, sc, s->stream));
    CU(launch_pack_codes_dyn(sl->codes, d_npos, (uint64_t *)dseq, (uint32_t *)dinv, alloc, s->stream));
    CU(cudaEventRecord(sl->done, s->stream));
    s->st.n_launches += 7;
    s->st.h2d_bytes += len;
    Chunk c{(const uint64_t *)dseq, (const uint32_t *)dinv, (uint64_t)len, d_npos};
    s->chunks.push_back(c);
    return launch_chunk(s, c, true, true);
}

bool is_pinned_host(const void *p)
{
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost;
}

int feed_text_impl(hs_screen *s, const char *text, size_t n, int threads)
{
    if (s->flushed || s->flush_pending) return fail(HS_ESTATE, "screen already flushed; call hs_screen_reset first");
    if (threads < 0) threads = 0;
    if (threads > 64) threads = 64;
    const int parts = (int)std::min<uint64_t>(1u << 20, n / s->chunk_text + 1);
    auto spans = split_records(text, n, parts, 1 << 16);
    // the device parser handles FASTA ('>' records) whose text the DMA engine can read directly
    size_t first = 0;
    while (first < n && (text[first] == '\n' || text[first] == '\r')) first++;
    const bool fasta = first < n && text[first] != '@';
    // (a single record of a GiB or more cannot go through the device parser's 32-bit offsets: such a feed is
    // packed on the host as a whole)
    size_t longest = 0;
    for (const auto &sp : spans) longest = std::max(longest, sp.second - sp.first);
    const bool device_ok = fasta && s->ingest_mode != 0 && longest < ((size_t)1 << 28) && is_pinned_host(text) &&
                           is_pinned_host(text + n - 1);
    const bool use_device = device_ok;
    if (s->ingest_mode == 1 && device_ok) threads = 0;          // device parser only
    // a handful of packer threads next to the DMA engine only adds host-memory traffic (8 GPUs x 4
    // threads measured: 150 Gbp/s with them, 168 without; 4 x 8 threads: 112 with, 105 without)
    if (s->ingest_mode == 2 && device_ok && threads < 6) threads = 0;
    if (!use_device && threads < 1) threads = 1;
    if ((int)spans.size() < threads) threads = (int)spans.size();
    if (spans.empty()) return HS_OK;
    // two staging buffers per packer thread (pinned), reused through events
    const size_t need = (size_t)threads * 2;
    while (s->staging.size() < need) {
        Staging g;
        CU(cudaEventCreateWithFlags(&g.free_ev, cudaEventDisableTiming));
        s->staging.push_back(g);
    }
    std::atomic<size_t> next{0};
    std::atomic<int> rc_all{HS_OK};
    std::atomic<int> dev_us_per_span{350};  // measured pace of the device-ingest worker
    std::atomic<int> pack_us_per_span{(int)(s->chunk_text / 5000) + 1};   // pace of one packer thread (EMA; ~5 GB/s to start with)
    std::string err_all;
    std::mutex err_mu;
    // Each side may leave the rest of the spans to the other (below); `device_quit` and `packers_alive` make
    // sure the two never do so at the same time: whoever wants to stop announces it first and then looks at
    // the other's announcement (sequentially consistent atomics: at least one of them sees the other's).
    std::atomic<bool> device_quit{!use_device};
    std::atomic<int> packers_alive{threads};
    auto worker = [&](int t, bool may_yield) {
        cudaSetDevice(s->db->device);
        int flip = 0;
        double my_ms = 4.0;  // how long this thread needs to pack one span
        for (;;) {
            if (use_device && may_yield && !device_quit.load()) {
                // do not start a span the DMA + device parser would finish before we do: near the end
                // of the input a slow packer thread would otherwise be the tail of the whole feed
                const size_t nx = next.load();
                if (nx >= spans.size()) break;
                if ((double)(spans.size() - nx) * dev_us_per_span.load() * 1e-3 < my_ms) {
                    packers_alive.fetch_sub(1);
                    if (!device_quit.load()) return;     // the device worker is still there and will see one packer fewer
                    packers_alive.fetch_add(1);          // it has stopped taking spans: stay
                }
            }
            const size_t i = next.fetch_add(1);
            if (i >= spans.size() || rc_all.load() != HS_OK) break;
            Staging &g = s->staging[(size_t)t * 2 + (flip ^= 1)];
            const size_t len = spans[i].second - spans[i].first;
            const uint64_t bound = pack_words_bound(len);
            int rc = HS_OK;
            if (g.cap_words < bound) {
                if (g.seq) { cudaEventSynchronize(g.free_ev); cudaFreeHost(g.seq); cudaFreeHost(g.inv); g.seq = nullptr; g.inv = nullptr; }
                g.cap_words = bound + bound / 8;
                if (cudaHostAlloc((void **)&g.seq, g.cap_words * 8, cudaHostAllocDefault) != cudaSuccess ||
                    cudaHostAlloc((void **)&g.inv, g.cap_words * 4, cudaHostAllocDefault) != cudaSuccess) {
                    g.cap_words = 0;
                    rc = fail(HS_ENOMEM, "pinned staging allocation failed");
                }
            } else {
                cudaEventSynchronize(g.free_ev);  // previous H2D from this buffer has finished
            }
            PackStats ps;
            if (rc == HS_OK) {
                const double t0 = now_s();
                pack_text_span(text + spans[i].first, len, g.seq, g.inv, &ps);
                const double t1 = now_s();
                my_ms = 1e3 * (t1 - t0);
                pack_us_per_span.store((pack_us_per_span.load() * 3 + (int)(1e3 * my_ms)) / 4);
                std::lock_guard<std::mutex> lk(s->mu);
                const double t2 = now_s();
                s->st.n_bases += ps.n_seq_bases;
                s->st.n_records += ps.n_records;
                rc = feed_host_chunk(s, g.seq, g.inv, ps.n_positions, g.free_ev);
                if (g_debug_timing)
                    fprintf(stderr, "[hs] span %zu thr %d: %zu B pack %.2f ms (%.2f GB/s) lock-wait %.2f ms feed %.2f ms\n", i, t,
                            len, 1e3 * (t1 - t0), len / (t1 - t0) / 1e9, 1e3 * (t2 - t1), 1e3 * (now_s() - t2));
            }
            if (rc != HS_OK) {
                std::lock_guard<std::mutex> lk(err_mu);
                if (rc_all.load() == HS_OK) { rc_all = rc; err_all = g_err; }
                break;
            }
        }
        if (may_yield) packers_alive.fetch_sub(1);
    };
    // the device-ingest worker competes with the packer threads for spans: it costs no CPU
    // (one cudaMemcpyAsync + kernel launches per span) and is throttled by its raw-text slots
    auto device_worker = [&]() {
        cudaSetDevice(s->db->device);
        // consecutive spans are contiguous text: take a few at a time so that the parser and
        // stream kernels run on >= 48 MB launches (fewer, fuller waves; fewer host wake-ups)
        const size_t batch = threads > 0 ? 2 : 4;
        for (;;) {
            if (threads > 0) {
                // The mirror image of the packers' rule: a batch taken now completes after everything already
                // queued on this path (raw text moves at ~1 byte per base over PCIe).  If the packer threads
                // would be through with ALL that is left before then, taking it only lengthens the tail --
                // with the AVX-512 packer the feed used to return after 9 ms and the GPU worked off this
                // path's backlog for another 6.
                const size_t nx = next.load();
                if (nx >= spans.size()) break;
                int busy = 0;
                for (int q = 0; q < Ingest::kSlots; q++)
                    if (s->ingest.slots[q].done && cudaEventQuery(s->ingest.slots[q].done) == cudaErrorNotReady) busy++;
                cudaGetLastError();
                const int alive = packers_alive.load();
                const double rest_ms = (double)(spans.size() - nx) * pack_us_per_span.load() * 1e-3 / (alive > 0 ? alive : 1);
                const double mine_ms = (double)(busy + 1) * (double)batch * dev_us_per_span.load() * 1e-3 + 0.3;
                if (alive > 0 && rest_ms < mine_ms) {
                    device_quit.store(true);
                    if (packers_alive.load() > 0) break;   // somebody is left to take the rest
                    device_quit.store(false);              // the last packer has just left it to us
                }
            }
            const size_t i = next.fetch_add(batch);
            if (i >= spans.size() || rc_all.load() != HS_OK) break;
            const size_t last = std::min(spans.size(), i + batch) - 1;
            const size_t len = spans[last].second - spans[i].first;
            const double t0 = now_s();
            int rc = feed_span_device(s, text + spans[i].first, len);
            {   // pace = wall time per span including the wait for a free slot (EMA)
                // never faster than the PCIe link can move the raw text (~60 GB/s)
                const int floor_us = (int)(len / (last - i + 1) / 60000) + 1;
                const int us = (int)(1e6 * (now_s() - t0) / (double)(last - i + 1));
                dev_us_per_span.store((dev_us_per_span.load() * 3 + std::max(us, floor_us)) / 4);
            }
            if (g_debug_timing)
                fprintf(stderr, "[hs] spans %zu-%zu device-ingest: %zu B enqueue+wait %.2f ms\n", i, last, len,
                        1e3 * (now_s() - t0));
            if (rc != HS_OK) {
                std::lock_guard<std::mutex> lk(err_mu);
                if (rc_all.load() == HS_OK) { rc_all = rc; err_all = g_err; }
                break;
            }
        }
    };
    if (threads == 1 && !use_device) {
        worker(0, false);
    } else {
        std::vector<std::thread> pool;
        if (use_device) pool.emplace_back(device_worker);
        for (int t = 0; t < threads; t++) pool.emplace_back(worker, t, true);
        for (auto &th : pool) th.join();
    }
    // belt and braces: every span is fed exactly once whatever the two sides decided
    if (rc_all == HS_OK && next.load() < spans.size()) {
        while (s->staging.size() < 2) {
            Staging g;
            CU(cudaEventCreateWithFlags(&g.free_ev, cudaEventDisableTiming));
            s->staging.push_back(g);
        }
        worker(0, false);
    }
    if (rc_all != HS_OK) return fail(rc_all, err_all);
    return HS_OK;
}

size_t pread_full(int fd, char *dst, size_t n, uint64_t off)
{
    size_t got = 0;
    while (got < n) {
        const ssize_t r = pread(fd, dst + got, n - got, (off_t)(off + got));
        if (r <= 0) break;
        got += (size_t)r;
    }
    return got;
}

// index of the first record start ('>' right after a newline) in buf[from, n), or n
size_t find_record_start(const char *buf, size_t from, size_t n)
{
    if (from < 1) from = 1;
    while (from < n) {
        const char *p = (const char *)memchr(buf + from, '>', n - from);
        if (!p) return n;
        const size_t i = (size_t)(p - buf);
        if (buf[i - 1] == '\n') return i;
        from = i + 1;
    }
    return n;
}

// Row a6 for a plain FASTA file: reader threads pread() disjoint blocks of the file into a
// pinned ring; each block is trimmed to whole records (it starts at the first record start at or
// after its nominal begin and runs to the first record start at or after its nominal end, so
// blocks are independent of each other) and handed to the device parser.  File -> page-cache
// copy -> DMA -> parse/pack/hash on the GPU; no host-side parsing at all.
// [range_begin, range_end) restricts the call to the records that START in that byte range (a record that
// starts before range_end is read to its end, the one straddling range_begin belongs to whoever owns the
// bytes before it), so N callers with adjacent ranges cover the file exactly once.
int feed_file_stream(hs_screen *s, int fd, uint64_t size, int threads, uint64_t range_begin = 0, uint64_t range_end = ~0ull)
{
    if (s->flushed || s->flush_pending) return fail(HS_ESTATE, "screen already flushed; call hs_screen_reset first");
    range_end = std::min(range_end, size);
    if (range_begin >= range_end) return HS_OK;
    const uint64_t B = s->file_block;
    const uint64_t n_blocks = (range_end - range_begin + B - 1) / B;
    int T = std::max(1, std::min(threads, s->file_readers));
    if ((uint64_t)T > n_blocks) T = (int)n_blocks;
    const size_t cap = (size_t)(B + B / 2 + 4096);
    if (s->ring.slot_cap < cap || s->ring.free_ev.size() < (size_t)2 * T) {
        CU(cudaStreamSynchronize(s->copy_stream));
        s->ring.release();
        CU(cudaHostAlloc((void **)&s->ring.base, cap * 2 * T, cudaHostAllocDefault));
        s->ring.slot_cap = cap;
        for (int i = 0; i < 2 * T; i++) {
            cudaEvent_t e;
            CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            s->ring.free_ev.push_back(e);
        }
    }
    std::atomic<uint64_t> next{0};
    std::atomic<int> rc_all{HS_OK};
    std::string err_all;
    std::mutex err_mu;
    auto reader = [&](int t) {
        cudaSetDevice(s->db->device);
        int flip = 0;
        auto bail = [&](int rc) {
            std::lock_guard<std::mutex> lk(err_mu);
            if (rc_all.load() == HS_OK) { rc_all = rc; err_all = g_err; }
        };
        for (;;) {
            const uint64_t j = next.fetch_add(1);
            if (j >= n_blocks || rc_all.load() != HS_OK) break;
            const size_t slot = (size_t)t * 2 + (size_t)(flip ^= 1);
            char *buf = s->ring.base + slot * s->ring.slot_cap;
            if (cudaEventSynchronize(s->ring.free_ev[slot]) != cudaSuccess) { bail(fail(HS_ECUDA, "ring event")); break; }
            const double t0 = now_s();
            const uint64_t nominal_begin = range_begin + j * B;
            const uint64_t off0 = nominal_begin ? nominal_begin - 1 : 0;   // one byte early: is there a newline before the block?
            const uint64_t nominal_end = std::min(range_end, nominal_begin + B);
            size_t got = pread_full(fd, buf, (size_t)std::min<uint64_t>(size - off0, nominal_end - off0 + std::min<uint64_t>(65536, B / 4)), off0);
            if (off0 + got < nominal_end) { bail(fail(HS_EIO, "short read")); break; }
            // first record that starts inside this block (block 0 starts at the top of the file)
            size_t b = 0;
            if (nominal_begin) {
                b = find_record_start(buf, 1, (size_t)(nominal_end - off0));
                if (b >= nominal_end - off0) continue;        // no record starts here: an earlier block owns these bytes
            }
            // first record start at or after the nominal end: read on until it shows up
            size_t e = got, from = (size_t)(nominal_end - off0);
            bool giant = false;
            for (;;) {
                e = find_record_start(buf, from, got);
                if (e < got || off0 + got >= size) break;
                if (got >= cap) { giant = true; break; }
                from = got;
                const size_t more = (size_t)std::min<uint64_t>(std::min<uint64_t>(cap - got, size - off0 - got), (uint64_t)4 << 20);
                const size_t r = pread_full(fd, buf + got, more, off0 + got);
                if (!r) { bail(fail(HS_EIO, "short read")); break; }
                got += r;
            }
            if (rc_all.load() != HS_OK) break;
            const double t1 = now_s();
            int rc = HS_OK;
            if (giant) {
                // a record longer than a ring slot: find its end, read it into ordinary memory and let
                // the host packer take it (rare: chromosome-sized contigs)
                std::vector<char> tmp((size_t)1 << 20);
                uint64_t pos = off0 + got, end = size;
                char prev = buf[got - 1];
                while (pos < size) {
                    const size_t r = pread_full(fd, tmp.data(), tmp.size(), pos);
                    if (!r) break;
                    size_t hit = r;
                    if (tmp[0] == '>' && prev == '\n') hit = 0; else hit = find_record_start(tmp.data(), 1, r);
                    if (hit < r) { end = pos + hit; break; }
                    prev = tmp[r - 1];
                    pos += r;
                }
                std::vector<char> rec((size_t)(end - (off0 + b)));
                if (pread_full(fd, rec.data(), rec.size(), off0 + b) != rec.size()) { bail(fail(HS_EIO, "short read")); break; }
                std::lock_guard<std::mutex> lk(s->giant_mu);
                rc = feed_text_impl(s, rec.data(), rec.size(), 1);
            } else {
                std::lock_guard<std::mutex> lk(s->ingest_mu);
                rc = feed_span_device(s, buf + b, e - b, s->ring.free_ev[slot]);
            }
            if (g_debug_timing)
                fprintf(stderr, "[hs] block %llu reader %d: %zu B read %.2f ms (%.2f GB/s) submit %.2f ms%s\n", (unsigned long long)j,
                        t, got, 1e3 * (t1 - t0), got / (t1 - t0) / 1e9, 1e3 * (now_s() - t1), giant ? " [giant record: host path]" : "");
            if (rc != HS_OK) { bail(rc); break; }
        }
    };
    if (T == 1) {
        reader(0);
    } else {
        std::vector<std::thread> pool;
        for (int t = 0; t < T; t++) pool.emplace_back(reader, t);
        for (auto &th : pool) th.join();
    }
    if (rc_all != HS_OK) return fail(rc_all, err_all);
    return HS_OK;
}

// Row a6 for a plain FASTA file, second form: map the file and let the host packer threads read the page
// cache where it lies -- no copy into a pinned ring, and 3/8 of a byte per base over PCIe instead of a
// whole one.  Worth it when the packers are fast (AVX-512 hosts: pack_level() == 2); the pread ring feeds
// the device parser otherwise.  Same range rule as feed_file_stream.
bool file_wants_mmap(const hs_screen *s, int threads) { return s->file_mode == 1 || (s->file_mode < 0 && pack_level() >= 2 && threads >= 4); }

int feed_file_mmap(hs_screen *s, int fd, uint64_t size, int threads, uint64_t range_begin = 0, uint64_t range_end = ~0ull)
{
    if (s->flushed || s->flush_pending) return fail(HS_ESTATE, "screen already flushed; call hs_screen_reset first");
    range_end = std::min(range_end, size);
    if (range_begin >= range_end) return HS_OK;
    void *m = mmap(nullptr, (size_t)size, PROT_READ, MAP_PRIVATE, fd, 0);
    if (m == MAP_FAILED) return fail(HS_EIO, "mmap failed");
    madvise(m, (size_t)size, MADV_SEQUENTIAL);
    const char *t = (const char *)m;
    // a record belongs to the range in which its first byte falls
    auto cut = [&](uint64_t pos) -> uint64_t { return pos == 0 ? 0 : (pos >= size ? size : find_record_start(t, (size_t)pos, (size_t)size)); };
    const uint64_t b = cut(range_begin), e = cut(range_end);
    int rc = HS_OK;
    if (e > b) rc = feed_text_impl(s, t + b, (size_t)(e - b), threads);
    // the packers have read everything (their H2D copies come from pinned staging, not from the mapping)
    munmap(m, (size_t)size);
    return rc;
}

}  // namespace

HS_API int hs_screen_feed_text(hs_screen *s, const char *text, size_t n, int host_threads)
{
    if (!s || (!text && n)) return fail(HS_EINVAL, "null argument");
    ON_DEVICE(s->db->device);
    return feed_text_impl(s, text, n, host_threads);
}

HS_API int hs_screen_feed_fasta(hs_screen *s, const char *path, int host_threads)
{
    if (!s || !path) return fail(HS_EINVAL, "null argument");
    ON_DEVICE(s->db->device);
    // plain FASTA in a regular file: stream it through the pinned ring to the device parser
    if (strcmp(path, "-") != 0) {
        const int fd = open(path, O_RDONLY);
        struct stat sb;
        if (fd >= 0 && fstat(fd, &sb) == 0 && S_ISREG(sb.st_mode) && sb.st_size > 0) {
            char head[256];
            const size_t hn = pread_full(fd, head, sizeof head, 0);
            size_t first = 0;
            while (first < hn && (head[first] == '\n' || head[first] == '\r')) first++;
            if (first < hn && head[first] == '>') {   // not gzip (1f 8b), not FASTQ
                // ("ingest" 0 = host packer only: the mapped form IS the host path, minus a copy)
                const int rc = (s->ingest_mode == 0 || file_wants_mmap(s, host_threads))
                                   ? feed_file_mmap(s, fd, (uint64_t)sb.st_size, host_threads)
                                   : feed_file_stream(s, fd, (uint64_t)sb.st_size, host_threads);
                close(fd);
                return rc;
            }
        }
        if (fd >= 0) close(fd);
    }
    // gzip / stdin / FASTQ: decompress on this thread in chunks of whole FASTA records and hand every
    // chunk to the host packer threads, so memory stays bounded and the GPU works on chunk i while
    // chunk i+1 is being inflated.  FASTQ is cut where the packer's own walk sees a header (record_starts:
    // '@' also starts quality lines), so read sets stay bounded in memory and use every packer thread too.
    gzFile f = strcmp(path, "-") == 0 ? gzdopen(0, "rb") : gzopen(path, "rb");
    if (!f) return fail(HS_EIO, std::string("could not open ") + path);
    gzbuffer(f, 1 << 20);
    const size_t chunk = (size_t)s->text_chunk;
    std::vector<char> buf;
    size_t len = 0, target = chunk;
    bool fastq = false, first = true, eof = false;
    int rc = HS_OK;
    while (!eof && rc == HS_OK) {
        while (len < target) {   // fill up to one chunk
            if (buf.size() - len < ((size_t)1 << 22)) buf.resize(std::max(buf.size() * 2, len + ((size_t)1 << 23)));
            const int r = gzread(f, buf.data() + len, 1u << 22);
            if (r < 0) { gzclose(f); return fail(HS_EIO, std::string("read error on ") + path); }
            if (r == 0) { eof = true; break; }
            len += (size_t)r;
            if (first) {
                size_t q = 0;
                while (q < len && (buf[q] == '\n' || buf[q] == '\r')) q++;
                if (q < len) { fastq = buf[q] == '@'; first = false; }
            }
        }
        size_t cut = len;
        if (!eof) {   // last record start in the buffer: everything before it is whole records
            cut = 0;
            if (fastq) {   // '@' also starts quality lines: only the packer's own walk knows a header from one
                const std::vector<size_t> starts = record_starts(buf.data(), len, 1);
                if (starts.size() > 1) cut = starts.back();
            } else {
                for (size_t i = len - 1; i > 0; i--)
                    if (buf[i] == '>' && buf[i - 1] == '\n') { cut = i; break; }
            }
            if (!cut) { target = len + chunk; continue; }   // one record larger than the chunk: keep reading
        }
        rc = feed_text_impl(s, buf.data(), cut, host_threads);
        memmove(buf.data(), buf.data() + cut, len - cut);
        len -= cut;
        target = chunk;
    }
    gzclose(f);
    return rc;
}

HS_API int hs_screen_feed_fasta_range(hs_screen *s, const char *path, uint64_t begin, uint64_t end, int host_threads)
{
    if (!s || !path) return fail(HS_EINVAL, "null argument");
    ON_DEVICE(s->db->device);
    const int fd = open(path, O_RDONLY);
    if (fd < 0) return fail(HS_EIO, std::string("could not open ") + path);
    struct stat sb;
    char head[256];
    size_t hn = 0, first = 0;
    const bool regular = fstat(fd, &sb) == 0 && S_ISREG(sb.st_mode) && sb.st_size > 0;
    if (regular) {
        hn = pread_full(fd, head, sizeof head, 0);
        while (first < hn && (head[first] == '\n' || head[first] == '\r')) first++;
    }
    if (!regular || first >= hn || head[first] != '>') {
        close(fd);
        return fail(HS_EUNSUPPORTED, "byte ranges need a plain FASTA file (gzip, FASTQ and pipes cannot be cut): feed it whole");
    }
    const int rc = file_wants_mmap(s, host_threads) ? feed_file_mmap(s, fd, (uint64_t)sb.st_size, host_threads, begin, end)
                                                    : feed_file_stream(s, fd, (uint64_t)sb.st_size, host_threads, begin, end);
    close(fd);
    return rc;
}

HS_API int hs_screen_feed_packed(hs_screen *s, const uint64_t *seq2, const uint32_t *inv, uint64_t n_bases)
{
    if (!s || ((!seq2 || !inv) && n_bases)) return fail(HS_EINVAL, "null argument");
    ON_DEVICE(s->db->device);
    if (s->flushed || s->flush_pending) return fail(HS_ESTATE, "screen already flushed; call hs_screen_reset first");
    std::lock_guard<std::mutex> lk(s->mu);
    s->st.n_bases += n_bases;
    return feed_host_chunk(s, seq2, inv, n_bases, nullptr);
}

HS_API int hs_screen_feed_packed_device(hs_screen *s, const void *d_seq2, const void *d_inv, uint64_t n_bases)
{
    if (!s || ((!d_seq2 || !d_inv) && n_bases)) return fail(HS_EINVAL, "null argument");
    ON_DEVICE(s->db->device);
    if (s->flushed || s->flush_pending) return fail(HS_ESTATE, "screen already flushed; call hs_screen_reset first");
    if (((uintptr_t)d_seq2 & 15) || ((uintptr_t)d_inv & 15)) return fail(HS_EINVAL, "packed device buffers must be 16-byte aligned");
    std::lock_guard<std::mutex> lk(s->mu);
    s->st.n_bases += n_bases;
    Chunk c{(const uint64_t *)d_seq2, (const uint32_t *)d_inv, n_bases};
    s->chunks.push_back(c);
    return launch_chunk(s, c, true, true);
}

namespace {

// what hs_screen_flush does once the stream has been synchronised: counters, timings, state
int flush_epilogue(hs_screen *s, bool parsed)
{
    unsigned long long *h = s->h_stats, *t = s->h_stats + ST_COUNT;
    if (parsed) { s->st.n_positions += t[0]; s->st.n_bases += t[1]; s->st.n_records += t[2]; }
    s->st.n_valid_kmers = h[ST_VALID]; s->st.n_probes = h[ST_PROBES]; s->st.n_bucket_reads = h[ST_BUCKETS];
    s->st.n_hits = h[ST_HITS]; s->st.n_mix_inserts = h[ST_MIXINS];
    s->st.n_mix_passes = s->mix.passes;
    s->st.n_mixture = s->mixture.size();
    s->st.set_size = set_size_of(s->mixture, s->db->use64, s->db->seg_s[0]);
    int rc = collect_stream_ms(s);
    if (rc) return rc;
    if (s->rst_pending) {
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, s->rst0, s->rst1));
        s->st.ms_reset = ms;
        s->rst_pending = false;
    }
    return HS_OK;
}

}  // namespace

// Rows a8-a10 without waiting: the device-side selection of the local bottom-s is ENQUEUED, its result and
// the counters travel to pinned memory behind it, and nothing is looked at until the caller's next
// synchronisation (hs_screen_finish*), which then completes the flush.  In between the caller may
// enqueue the whole multi-GPU exchange -- hs_screen_mixture_record reads the selection where it lies on
// the device -- so that one screen is ONE host synchronisation and the host runs ahead of the GPU from
// the first feed to the result.  If the selection does not hold (set overflowed, fewer than s values
// below tau, a crowded bin) the record says so, every rank sees it after the all-gather
// (hs_stats_t.mix_unsettled), and the caller falls back to hs_screen_flush + the synchronous exchange.
HS_API int hs_screen_flush_async(hs_screen *s)
{
    if (!s) return fail(HS_EINVAL, "null handle");
    ON_DEVICE(s->db->device);
    if (s->flushed || s->flush_pending) return HS_OK;
    if (!s->mix.fast_select) return hs_screen_flush(s);
    std::lock_guard<std::mutex> lk(s->mu);
    CU(cudaEventRecord(s->red0, s->stream));
    const bool parsed = s->ingest.ready && s->ingest.counters_used;
    CU(cudaMemcpyAsync(s->h_stats, s->d_stats, ST_COUNT * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s->stream));
    if (parsed) {
        CU(cudaMemcpyAsync(s->h_stats + ST_COUNT, s->ingest.d_totals, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s->stream));
        CU(cudaMemsetAsync(s->ingest.d_totals, 0, 4 * sizeof(unsigned long long), s->stream));
    }
    MixEngine &m = s->mix;
    CU(launch_mix_select(m.view(~0ull), m.s, m.use64, m.d_hist, m.d_cand, m.sel_pad, m.d_scratch, s->stream));
    s->st.n_launches += 4;
    CU(cudaMemcpyAsync(m.h_cand, m.d_cand, (size_t)m.s * 8, cudaMemcpyDeviceToHost, s->stream));
    CU(cudaMemcpyAsync(m.h_state, m.d_state, sizeof(MixState), cudaMemcpyDeviceToHost, s->stream));
    s->flush_pending = true;
    s->flush_parsed = parsed;
    return HS_OK;
}

HS_API int hs_screen_flush(hs_screen *s)
{
    if (!s) return fail(HS_EINVAL, "null handle");
    ON_DEVICE(s->db->device);
    if (s->flushed) return HS_OK;
    std::lock_guard<std::mutex> lk(s->mu);
    if (s->flush_pending) {
        // an enqueued selection is abandoned (its verdict was "not settled", or the caller changed its mind):
        // the iterative finaliser below starts from the same device state
        CU(cudaStreamSynchronize(s->stream));
        if (s->flush_parsed) {   // the parser totals were folded into h_stats and cleared on the device: keep them
            unsigned long long *t = s->h_stats + ST_COUNT;
            s->st.n_positions += t[0]; s->st.n_bases += t[1]; s->st.n_records += t[2];
        }
        s->flush_pending = false;
    }
    CU(cudaEventRecord(s->red0, s->stream));
    // the counters are final once the streaming launches are (re-offer passes count elsewhere): fetch
    // them with the first synchronisation of the mixture finaliser instead of one of their own
    unsigned long long *h = s->h_stats, *t = s->h_stats + ST_COUNT;
    const bool parsed = s->ingest.ready && s->ingest.counters_used;
    CU(cudaMemcpyAsync(h, s->d_stats, ST_COUNT * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s->stream));
    if (parsed) {
        CU(cudaMemcpyAsync(t, s->ingest.d_totals, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s->stream));
        CU(cudaMemsetAsync(s->ingest.d_totals, 0, 4 * sizeof(unsigned long long), s->stream));  // folded: do not fold twice
    }
    int rc = mix_finalize(s->mix, s->stream, s->mixture, s->st.n_launches, [&]() -> int {
        for (const Chunk &c : s->chunks) {
            int r = launch_chunk(s, c, false, true);
            if (r) return r;
            if (!c.n_dev) s->st.n_positions -= c.n_bases;  // a mixture-only second pass is not new input
        }
        return HS_OK;
    });
    if (rc) return rc;
    CU(cudaEventRecord(s->red1, s->stream));
    CU(cudaEventSynchronize(s->red1));   // mix_finalize ended on a synchronisation: nothing is left to wait for
    rc = flush_epilogue(s, parsed);
    if (rc) return rc;
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, s->red0, s->red1));
    s->st.ms_reduce = ms;
    s->flushed = true;
    return HS_OK;
}

HS_API int hs_screen_counts_devptr(hs_screen *s, void **d_counts, uint64_t *n)
{
    if (!s || !d_counts || !n) return fail(HS_EINVAL, "null argument");
    *d_counts = s->d_counts;
    *n = s->db->n_entries;
    // whoever asks for the raw vector may add to it (the dense all-reduce): the record of which
    // counts are non-zero no longer covers it, so reduction and reset take their dense forms
    s->touched_valid = false;
    return HS_OK;
}

HS_API int hs_screen_counts_compact_async(hs_screen *s, void *d_pairs, uint32_t cap, void *d_n_out)
{
    if (!s || !d_pairs || !d_n_out) return fail(HS_EINVAL, "null argument");
    ON_DEVICE(s->db->device);
    // no flush needed: counts[] is final, in stream order, as soon as the last feed has been enqueued
    // (the mixture finaliser never touches it), so the exchange can start underneath hs_screen_flush
    CU(cudaMemsetAsync(d_n_out, 0, sizeof(uint32_t), s->stream));
    SparseView sp = sparse_view(s);
    if (!s->touched_valid) sp.touched = nullptr;
    CU(launch_counts_compact(sp, s->d_counts, s->db->n_entries, (unsigned long long *)d_pairs, cap, (uint32_t *)d_n_out, s->stream));
    s->st.n_launches += sp.touched ? 2 : 1;
    return HS_OK;
}

HS_API int hs_screen_counts_absorb(hs_screen *s, const void *d_rows, uint32_t n_rows, uint32_t cap, uint32_t skip_row)
{
    if (!s || (!d_rows && n_rows)) return fail(HS_EINVAL, "null argument");
    ON_DEVICE(s->db->device);
    SparseView sp = sparse_view(s);
    if (!s->touched_valid) sp.touched = nullptr;
    CU(launch_counts_absorb(sp, s->d_counts, s->db->n_entries, (const unsigned long long *)d_rows, n_rows, cap, skip_row,
                            s->db->sm, s->stream));
    s->st.n_launches++;
    return HS_OK;
}

namespace {

// [length | s hashes, zero padded]: a settled mixture (<= s values) as one row of the mixture merge
void mixture_row(const hs_screen *s, uint64_t *row)
{
    const size_t n = s->mixture.size();
    memset(row, 0, ((size_t)s->db->s + 1) * 8);
    row[0] = n;
    if (n) memcpy(row + 1, s->mixture.data(), n * 8);
}

// what hs_screen_mixture_merge_device left in h_sparse / h_mixture becomes the screen's mixture
void adopt_merged_mixture(hs_screen *s)
{
    const uint32_t nm = std::min<uint32_t>(s->h_sparse->n_mix, s->db->s);
    s->mixture.assign(s->h_mixture, s->h_mixture + nm);
    s->st.n_mixture = nm;
    s->st.set_size = s->h_sparse->set_size[0];
}

}  // namespace

HS_API int hs_screen_absorb_screens(hs_screen *dst, hs_screen *const *src, uint32_t n_src)
{
    // every check before any device work: a refused call leaves every handle as it was
    if (!dst || !src || !n_src) return fail(HS_EINVAL, "a screen and at least one source are needed");
    for (uint32_t i = 0; i < n_src; i++) {
        if (!src[i] || src[i] == dst) return fail(HS_EINVAL, "every source must be a screen other than dst");
        for (uint32_t j = 0; j < i; j++)
            if (src[j] == src[i]) return fail(HS_EINVAL, "a source is listed twice: it would be counted twice");
    }
    if (dst->mixture_on_device) return fail(HS_ESTATE, "this screen has already absorbed others; call hs_screen_reset first");
    if (!dst->flushed) return fail(HS_ESTATE, "flush every screen first");
    const hs_db *db = dst->db;
    for (uint32_t i = 0; i < n_src; i++) {
        const hs_screen *s = src[i];
        if (!s->flushed) return fail(HS_ESTATE, "flush every screen first");
        if (s->mixture_on_device) return fail(HS_ESTATE, "a source has merged mixtures on the device: its own is stale");
        if (s->db->n_entries != db->n_entries || s->db->k != db->k || s->db->s != db->s || s->db->seg_s.size() != db->seg_s.size())
            return fail(HS_EINVAL, "the screens are not over the same sketch database");
    }
    // The distributed exchange with peer copies instead of the all-gather: each source's pair record
    // [n | (entry id << 32 | count) ...] is built on its own device, copied into row 1 + i of a buffer on
    // dst's device (row 0, dst's own, is empty and skipped), and hs_screen_counts_absorb and
    // hs_screen_mixture_merge_device take it from there.
    std::vector<unsigned long long *> rec(n_src, nullptr);
    unsigned long long *rows = nullptr;
    const int rc = [&]() -> int {
        std::vector<uint32_t> n(n_src);
        uint32_t cap = 1;
        for (uint32_t i = 0; i < n_src; i++) {
            hs_screen *s = src[i];
            ON_DEVICE(s->db->device);
            CU(cudaMemcpyAsync(s->h_sparse, s->d_sparse, sizeof(SparseState), cudaMemcpyDeviceToHost, s->stream));
            CU(cudaStreamSynchronize(s->stream));
            const bool listed = s->sparse_enabled && s->touched_valid && s->h_sparse->n_touched <= s->touched_cap;
            const uint64_t rcap = listed ? s->h_sparse->n_touched : db->n_entries;
            CU(cudaMalloc((void **)&rec[i], (rcap + 1) * 8));
            CU(cudaMemsetAsync(rec[i], 0, 8, s->stream));
            int r = hs_screen_counts_compact_async(s, rec[i] + 1, (uint32_t)rcap, rec[i]);
            if (r) return r;
            CU(cudaMemcpyAsync(&n[i], rec[i], sizeof(uint32_t), cudaMemcpyDeviceToHost, s->stream));
            CU(cudaStreamSynchronize(s->stream));
            cap = std::max(cap, n[i]);
        }
        ON_DEVICE(db->device);
        const size_t R = (size_t)n_src + 1, stride = (size_t)cap + 1, mstride = (size_t)db->s + 1;
        CU(cudaMalloc((void **)&rows, R * (stride + mstride) * 8));
        unsigned long long *mix = rows + R * stride;
        CU(cudaMemsetAsync(rows, 0, 8, dst->stream));
        for (uint32_t i = 0; i < n_src; i++)
            CU(cudaMemcpyPeerAsync(rows + (i + 1) * stride, db->device, rec[i], src[i]->db->device, ((size_t)n[i] + 1) * 8,
                                   dst->stream));
        std::vector<uint64_t> h_mix(R * mstride);
        mixture_row(dst, h_mix.data());
        for (uint32_t i = 0; i < n_src; i++) mixture_row(src[i], h_mix.data() + (i + 1) * mstride);
        CU(cudaMemcpyAsync(mix, h_mix.data(), h_mix.size() * 8, cudaMemcpyHostToDevice, dst->stream));
        int r = hs_screen_counts_absorb(dst, rows, (uint32_t)R, cap, 0);
        if (!r) r = hs_screen_mixture_merge_device(dst, mix, (uint32_t)R);
        if (r) return r;
        // the merged mixture and its set size now, as for a single screen after flush (stats read before finish)
        CU(cudaMemcpyAsync(dst->h_sparse, dst->d_sparse, sizeof(SparseState), cudaMemcpyDeviceToHost, dst->stream));
        if (db->s) CU(cudaMemcpyAsync(dst->h_mixture, dst->d_mixture, (size_t)db->s * 8, cudaMemcpyDeviceToHost, dst->stream));
        CU(cudaStreamSynchronize(dst->stream));
        adopt_merged_mixture(dst);
        for (uint32_t i = 0; i < n_src; i++) {
            const hs_stats_t &t = src[i]->st;
            dst->st.n_bases += t.n_bases; dst->st.n_records += t.n_records; dst->st.n_positions += t.n_positions;
            dst->st.n_valid_kmers += t.n_valid_kmers; dst->st.n_probes += t.n_probes;
            dst->st.n_bucket_reads += t.n_bucket_reads; dst->st.n_hits += t.n_hits;
            dst->st.n_mix_inserts += t.n_mix_inserts; dst->st.h2d_bytes += t.h2d_bytes;
            dst->st.n_launches += t.n_launches;
            dst->st.ms_stream = std::max(dst->st.ms_stream, t.ms_stream);
        }
        return HS_OK;
    }();
    if (rows && cudaSetDevice(db->device) == cudaSuccess) cudaFree(rows);
    for (uint32_t i = 0; i < n_src; i++)
        if (rec[i] && cudaSetDevice(src[i]->db->device) == cudaSuccess) cudaFree(rec[i]);
    return rc;
}

HS_API int hs_screen_mixture_get(hs_screen *s, uint64_t *hashes, uint32_t *n)
{
    if (!s || !n) return fail(HS_EINVAL, "null argument");
    if (!s->flushed) return fail(HS_ESTATE, "call hs_screen_flush first");
    *n = (uint32_t)s->mixture.size();
    if (hashes) memcpy(hashes, s->mixture.data(), s->mixture.size() * 8);
    return HS_OK;
}

HS_API int hs_screen_mixture_record(hs_screen *s, void *d_record)
{
    if (!s || !d_record) return fail(HS_EINVAL, "null argument");
    ON_DEVICE(s->db->device);
    if (s->flush_pending) {
        // the selection is still on its way: the record is cut out of it on the device, verdict included
        CU(launch_mix_record(s->mix.view(~0ull), s->db->s, s->mix.sel_pad, s->mix.d_cand, (unsigned long long *)d_record,
                             s->force_unsettled, s->stream));
        s->force_unsettled = 0;
        s->st.n_launches++;
        return HS_OK;
    }
    if (!s->flushed) return fail(HS_ESTATE, "call hs_screen_flush first");
    // what every rank contributes to the mixture all-gather: it goes up from pinned memory on the
    // screen's stream and the record stays on the device for the collective
    mixture_row(s, s->h_mixture);
    CU(cudaMemcpyAsync(d_record, s->h_mixture, ((size_t)s->db->s + 1) * 8, cudaMemcpyHostToDevice, s->stream));
    return HS_OK;
}

HS_API int hs_screen_mixture_merge_device(hs_screen *s, const void *d_rows, uint32_t n_rows)
{
    if (!s || !d_rows || !n_rows) return fail(HS_EINVAL, "null argument");
    ON_DEVICE(s->db->device);
    if (!s->flushed && !s->flush_pending) return fail(HS_ESTATE, "call hs_screen_flush first");
    const uint32_t sc = s->db->s;
    uint32_t need = 2;
    while (need < (uint64_t)n_rows * sc) need <<= 1;
    if (s->merge_cap < need) {
        cudaFree(s->d_merge_work); cudaFree(s->d_merge_scratch); cudaFree(s->d_mixture);
        s->d_merge_work = s->d_merge_scratch = s->d_mixture = nullptr;
        CU(cudaMalloc((void **)&s->d_merge_work, (size_t)need * 8));
        CU(cudaMalloc((void **)&s->d_merge_scratch, (size_t)need * 8));
        CU(cudaMalloc((void **)&s->d_mixture, (size_t)std::max<uint32_t>(sc, 1) * 8));
        s->merge_cap = need;
    }
    CU(launch_mixture_merge((const unsigned long long *)d_rows, n_rows, sc, sc, s->db->d_seg_s, (uint32_t)s->db->seg_s.size(),
                            s->db->use64, s->d_merge_work, need, s->d_merge_scratch, s->d_mixture, s->d_sparse, s->stream));
    s->st.n_launches += 3;
    s->mixture_on_device = true;   // finish reads the set sizes from the device and brings the mixture back with the results
    return HS_OK;
}

HS_API int hs_screen_segment_set_size(hs_screen *s, uint32_t segment, uint64_t *set_size)
{
    if (!s || !set_size) return fail(HS_EINVAL, "null argument");
    if (!s->flushed) return fail(HS_ESTATE, "call hs_screen_flush first");
    if (segment >= s->db->seg_s.size()) return fail(HS_EINVAL, "segment index out of range");
    *set_size = set_size_of(s->mixture, s->db->use64, s->db->seg_s[segment]);
    return HS_OK;
}

namespace {

// rows a11-a13 enqueued on the screen's stream: the O(present) kernels, or the dense ones
int enqueue_reduce(hs_screen *s, bool wta, bool dense)
{
    hs_db *db = s->db;
    const uint64_t N = db->n_refs, E = db->n_entries;
    const size_t n_seg = db->seg_s.size();
    if (!N) return HS_OK;
    if (!dense) {
        CU(cudaMemsetAsync(s->d_shared, 0, N * 8, s->stream));   // shared | median are adjacent
        static_assert(offsetof(SparseState, overflow) == offsetof(SparseState, n_hit) + 8, "n_hit, n_pairs, overflow are cleared together");
        CU(cudaMemsetAsync(&s->d_sparse->n_hit, 0, 3 * sizeof(uint32_t), s->stream));
        SparseReduceArgs a;
        memset(&a, 0, sizeof a);
        a.sp = sparse_view(s);
        a.counts = s->d_counts; a.next = db->d_next; a.offsets = db->d_offsets; a.n_refs = (uint32_t)N;
        a.lengths = db->d_lengths; a.seg_begin = db->d_seg_begin; a.n_seg = (uint32_t)n_seg;
        a.shared = s->d_shared; a.median = s->d_median; a.plain = s->d_plain; a.hit = s->d_hit;
        a.seg_start = s->d_seg_start; a.seg_fill = s->d_seg_fill; a.depths = s->d_depths; a.pair_cap = s->pair_cap;
        a.ref_scale = (E && N <= E) ? (uint64_t)((((unsigned __int128)N) << 64) / ((unsigned __int128)E + 1)) : 0;
        CU(launch_sparse_reduce(a, wta, db->sm, s->stream));
        s->st.n_launches += wta ? 7 : 4;
        return HS_OK;
    }
    CU(launch_sketch_reduce(db->d_offsets, N, db->d_canon, s->d_counts, nullptr, s->d_shared, s->d_median, db->sm, s->stream));
    s->st.n_launches++;
    if (wta && E) {
        if (!s->d_winner) {
            CU(cudaMalloc((void **)&s->d_best_score, E * 8));
            CU(cudaMalloc((void **)&s->d_best_len, E * 8));
            CU(cudaMalloc((void **)&s->d_winner, E * 4));
        }
        for (size_t j = 0; j < n_seg; j++) {   // -w is a competition among the references of one .msh (S12)
            const uint64_t b = db->seg_begin[j], n = db->seg_begin[j + 1] - b;
            if (!n) continue;
            CU(launch_winner(db->d_offsets + b, n, db->d_canon, s->d_counts, s->d_shared + b, db->d_lengths + b,
                             s->d_best_score, s->d_best_len, s->d_winner, E, db->sm, s->stream));
            CU(launch_sketch_reduce(db->d_offsets + b, n, db->d_canon, s->d_counts, s->d_winner, s->d_shared + b,
                                    s->d_median + b, db->sm, s->stream));
            s->st.n_launches += 5;   // k_winner x4 (clear, score, length, index) + the reduction
        }
    }
    return HS_OK;
}

// rows a14/a15 + the trip home: statistics per source file, the result columns, the sparse state
int enqueue_stats_and_copy(hs_screen *s)
{
    hs_db *db = s->db;
    const uint64_t N = db->n_refs;
    for (size_t j = 0; j < db->seg_s.size(); j++) {
        const uint64_t b = db->seg_begin[j], n = db->seg_begin[j + 1] - b;
        if (!n) continue;
        CU(launch_stats(db->k, set_size_of(s->mixture, db->use64, db->seg_s[j]),
                        s->mixture_on_device ? &s->d_sparse->set_size[j] : nullptr, n, s->d_shared + b, nullptr,
                        db->d_offsets + b, nullptr, s->d_identity + b, s->d_pvalue + b, s->stream));
        s->st.n_launches++;
    }
    const uint64_t NA = std::max<uint64_t>(N, 1);   // layout of the allocation (hs_screen_new)
    if (N) CU(cudaMemcpyAsync(s->h_result, s->d_identity, NA * 24, cudaMemcpyDeviceToHost, s->stream));
    CU(cudaMemcpyAsync(s->h_sparse, s->d_sparse, sizeof(SparseState), cudaMemcpyDeviceToHost, s->stream));
    if (s->mixture_on_device && db->s)
        CU(cudaMemcpyAsync(s->h_mixture, s->d_mixture, (size_t)db->s * 8, cudaMemcpyDeviceToHost, s->stream));
    return HS_OK;
}

}  // namespace

namespace {

// rows a14-a16 for the references with hits only, written by the GPU into host-mapped rows
int enqueue_hits(hs_screen *s, bool dense)
{
    hs_db *db = s->db;
    const uint64_t N = db->n_refs;
    if (N && !s->h_rows) {
        const size_t n3 = (N * 12 + 7) & ~(size_t)7;
        CU(cudaHostAlloc((void **)&s->h_rows, n3 + N * 16, cudaHostAllocMapped));
        char *d = nullptr;
        CU(cudaHostGetDevicePointer((void **)&d, s->h_rows, 0));
        auto lay = [&](char *base) {
            HitRows r;
            r.ref = reinterpret_cast<uint32_t *>(base); r.shared = r.ref + N; r.median = r.shared + N;
            r.identity = reinterpret_cast<double *>(base + n3); r.pvalue = r.identity + N;
            r.cap = (uint32_t)N;
            return r;
        };
        s->rows_host = lay(s->h_rows);
        s->rows_dev = lay(d);
    }
    if (N) {
        StatsHitArgs a;
        memset(&a, 0, sizeof a);
        a.k = db->k; a.n_seg = (uint32_t)db->seg_s.size();
        for (size_t j = 0; j < db->seg_s.size(); j++) a.set_size[j] = set_size_of(s->mixture, db->use64, db->seg_s[j]);
        a.set_size_dev = s->mixture_on_device ? s->d_sparse->set_size : nullptr;
        a.seg_begin = db->d_seg_begin; a.hit = s->d_hit; a.n_hit = &s->d_sparse->n_hit;
        a.shared = s->d_shared; a.median = s->d_median; a.offsets = db->d_offsets; a.rows = s->rows_dev;
        CU(launch_stats_hits(a, dense, (uint32_t)N, s->d_hit, &s->d_sparse->n_hit, db->sm, s->stream));
        s->st.n_launches += dense ? 2 : 1;
    }
    CU(cudaMemcpyAsync(s->h_sparse, s->d_sparse, sizeof(SparseState), cudaMemcpyDeviceToHost, s->stream));
    if (s->mixture_on_device && db->s)
        CU(cudaMemcpyAsync(s->h_mixture, s->d_mixture, (size_t)db->s * 8, cudaMemcpyDeviceToHost, s->stream));
    return HS_OK;
}

// the common part of hs_screen_finish / hs_screen_finish_hits: settle the mixture, reduce, statistics,
// results on the host (all N references as columns, or only the references with hits as rows)
int finish_core(hs_screen *s, bool wta, bool hits)
{
    // Single-GPU order: the per-sketch reduction needs only counts[], so it is enqueued BEFORE the
    // mixture is settled and runs underneath the host round trips of that (flush); a caller that
    // flushed first (multi-GPU: flush -> exchange -> finish) gets it here, after the exchange.
    const bool pending = s->flush_pending;
    const bool early = !s->flushed && !pending;
    bool dense = !(s->sparse_enabled && s->touched_valid);
    int rc;
    if (early) {
        CU(cudaEventRecord(s->red2, s->stream));
        if ((rc = enqueue_reduce(s, wta, dense)) != HS_OK) return rc;
        CU(cudaEventRecord(s->red3, s->stream));
    }
    if (!pending) {
        rc = hs_screen_flush(s);
        if (rc) return rc;
        CU(cudaEventRecord(s->red0, s->stream));
    }   // (pending: red0 was recorded by hs_screen_flush_async -- the exchange in between is part of the figure)
    if (early) {
        float ems = 0;
        CU(cudaEventElapsedTime(&ems, s->red2, s->red3));   // flush synchronised the stream
        s->st.ms_reduce += ems;
    }
    if (!early && (rc = enqueue_reduce(s, wta, dense)) != HS_OK) return rc;
    if ((rc = hits ? enqueue_hits(s, dense) : enqueue_stats_and_copy(s)) != HS_OK) return rc;
    CU(cudaEventRecord(s->red1, s->stream));
    CU(cudaStreamSynchronize(s->stream));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, s->red0, s->red1));
    s->st.ms_reduce = pending ? ms : s->st.ms_reduce + ms;
    s->st.mix_unsettled = 0;
    if (pending) {
        // the one synchronisation of this screen has happened: complete the flush from what came back with it
        const MixState &hs_ = *s->mix.h_state;
        const bool held = !s->force_unsettled && !hs_.overflow && !hs_.sel_too_many && hs_.n_out <= s->mix.sel_pad &&
                          (hs_.n_unique >= s->mix.s || hs_.tau == ~0ull);
        s->force_unsettled = 0;   // (tests; the multi-GPU path has already spent it in its mixture record)
        const bool all_held = s->mixture_on_device ? !s->h_sparse->mix_unsettled : held;
        if (!all_held) {
            if (s->mixture_on_device) {
                // some rank's selection fell through: every rank knows (the gathered records say so) and the
                // CALLER redoes flush + mixture exchange synchronously; the counts were absorbed and stay
                s->st.mix_unsettled = 1;
                s->st.exchange_overflow = s->h_sparse->xchg_overflow;
                s->st.exchange_max_pairs = s->h_sparse->xchg_max;
                return HS_OK;
            }
            rc = hs_screen_flush(s);              // single process: the iterative finaliser, then everything again
            if (rc) return rc;
            return finish_core(s, wta, hits);
        }
        s->mixture.assign(s->mix.h_cand, s->mix.h_cand + std::min(hs_.n_unique, s->mix.s));
        if (hs_.has_max && s->mixture.size() < s->mix.s) s->mixture.push_back(~0ull);
        s->flush_pending = false;
        rc = flush_epilogue(s, s->flush_parsed);
        if (rc) return rc;
        s->flushed = true;
    }
    if (s->mixture_on_device) adopt_merged_mixture(s);   // the merged mixture and its set size arrive with the results
    s->st.exchange_overflow = s->h_sparse->xchg_overflow;
    s->st.exchange_max_pairs = s->h_sparse->xchg_max;
    if (!dense && (s->h_sparse->n_touched > s->touched_cap || s->h_sparse->wrapped || s->h_sparse->overflow)) {
        // the O(present) bookkeeping did not hold this query (more present hashes than its buffers, or a
        // count that wrapped): the dense kernels give the answer, and the next reset clears every count
        dense = true;
        const uint32_t n_touched = s->h_sparse->n_touched;
        CU(cudaEventRecord(s->red0, s->stream));
        if ((rc = enqueue_reduce(s, wta, true)) != HS_OK) return rc;
        if ((rc = hits ? enqueue_hits(s, true) : enqueue_stats_and_copy(s)) != HS_OK) return rc;
        CU(cudaEventRecord(s->red1, s->stream));
        CU(cudaStreamSynchronize(s->stream));
        CU(cudaEventElapsedTime(&ms, s->red0, s->red1));
        s->st.ms_reduce += ms;
        s->h_sparse->n_touched = n_touched;
    }
    s->st.reduce_path = dense ? 1u : 0u;
    s->st.n_touched = s->h_sparse->n_touched;
    s->st.n_hit_refs = (dense && !hits) ? 0u : s->h_sparse->n_hit;
    s->st.n_pairs = dense ? 0u : s->h_sparse->n_pairs;
    return HS_OK;
}

}  // namespace

HS_API int hs_screen_finish(hs_screen *s, int wta, uint64_t *shared, uint32_t *median, double *identity,
                            double *pvalue, hs_stats_t *stats)
{
    if (!s) return fail(HS_EINVAL, "null handle");
    ON_DEVICE(s->db->device);
    int rc = finish_core(s, wta != 0, false);
    if (rc) return rc;
    const uint64_t N = s->db->n_refs, NA = std::max<uint64_t>(N, 1);   // layout of the allocation (hs_screen_new)
    double *h_id = reinterpret_cast<double *>(s->h_result), *h_pv = h_id + NA;
    uint32_t *h_sh = reinterpret_cast<uint32_t *>(h_pv + NA), *h_md = h_sh + NA;
    if (shared) for (uint64_t i = 0; i < N; i++) shared[i] = h_sh[i];
    if (median && N) memcpy(median, h_md, N * 4);
    if (identity && N) memcpy(identity, h_id, N * 8);
    if (pvalue && N) memcpy(pvalue, h_pv, N * 8);
    s->st.d2h_bytes += N * 24;
    if (stats) *stats = s->st;
    return HS_OK;
}

HS_API int hs_screen_finish_hits(hs_screen *s, int wta, uint32_t *n_hits, hs_stats_t *stats)
{
    if (!s || !n_hits) return fail(HS_EINVAL, "null argument");
    ON_DEVICE(s->db->device);
    int rc = finish_core(s, wta != 0, true);
    if (rc) return rc;
    const uint32_t n = (uint32_t)std::min<uint64_t>(s->h_sparse->n_hit, s->db->n_refs);
    s->hit_order.clear();
    for (uint32_t q = 0; q < n; q++)
        if (s->rows_host.shared[q]) s->hit_order.push_back(q);   // -w leaves references that lost every hash: not reported
    const uint32_t *ref = s->rows_host.ref;
    std::sort(s->hit_order.begin(), s->hit_order.end(), [ref](uint32_t a, uint32_t b) { return ref[a] < ref[b]; });
    *n_hits = (uint32_t)s->hit_order.size();
    s->st.d2h_bytes += (uint64_t)n * 28;
    if (stats) *stats = s->st;
    return HS_OK;
}

HS_API int hs_screen_hits_copy(hs_screen *s, uint32_t cap, uint32_t *ref, uint64_t *shared, uint32_t *median,
                               double *identity, double *pvalue)
{
    if (!s) return fail(HS_EINVAL, "null handle");
    const uint32_t n = (uint32_t)std::min<size_t>(cap, s->hit_order.size());
    for (uint32_t i = 0; i < n; i++) {
        const uint32_t q = s->hit_order[i];
        if (ref) ref[i] = s->rows_host.ref[q];
        if (shared) shared[i] = s->rows_host.shared[q];
        if (median) median[i] = s->rows_host.median[q];
        if (identity) identity[i] = s->rows_host.identity[q];
        if (pvalue) pvalue[i] = s->rows_host.pvalue[q];
    }
    return HS_OK;
}

HS_API int hs_screen_reset(hs_screen *s)
{
    if (!s) return fail(HS_EINVAL, "null handle");
    ON_DEVICE(s->db->device);
    CU(cudaStreamSynchronize(s->stream));
    return screen_zero(s);
}

HS_API int hs_screen_stats(hs_screen *s, hs_stats_t *stats)
{
    if (!s || !stats) return fail(HS_EINVAL, "null argument");
    *stats = s->st;
    return HS_OK;
}

HS_API void hs_screen_free(hs_screen *s)
{
    if (!s) return;
    if (s->db) cudaSetDevice(s->db->device);
    if (s->stream) cudaStreamSynchronize(s->stream);
    cudaFree(s->d_counts); cudaFree(s->d_stats);
    cudaFree(s->d_sparse); cudaFree(s->d_touched); cudaFree(s->d_depths); cudaFree(s->d_hit);
    cudaFree(s->d_mixture); cudaFree(s->d_merge_work); cudaFree(s->d_merge_scratch);
    if (s->h_sparse) cudaFreeHost(s->h_sparse);
    if (s->h_mixture) cudaFreeHost(s->h_mixture);
    if (s->h_rows) cudaFreeHost(s->h_rows);
    if (s->rst0) cudaEventDestroy(s->rst0);
    if (s->rst1) cudaEventDestroy(s->rst1);
    cudaFree(s->d_identity);   // one block: identity | p-value | shared | median
    cudaFree(s->d_best_score); cudaFree(s->d_best_len); cudaFree(s->d_winner);
    s->mix.destroy();
    s->arena.release();
    s->ingest.release();
    s->ring.release();
    for (auto &g : s->staging) {
        if (g.seq) cudaFreeHost(g.seq);
        if (g.inv) cudaFreeHost(g.inv);
        if (g.free_ev) cudaEventDestroy(g.free_ev);
    }
    for (auto &e : s->ev_pool) { cudaEventDestroy(e.first); cudaEventDestroy(e.second); }
    if (s->red0) cudaEventDestroy(s->red0);
    if (s->red1) cudaEventDestroy(s->red1);
    if (s->red2) cudaEventDestroy(s->red2);
    if (s->red3) cudaEventDestroy(s->red3);
    if (s->h_result) cudaFreeHost(s->h_result);
    if (s->h_stats) cudaFreeHost(s->h_stats);
    if (s->own_stream && s->stream) cudaStreamDestroy(s->stream);
    if (s->copy_stream) { cudaStreamSynchronize(s->copy_stream); cudaStreamDestroy(s->copy_stream); }
    for (auto &e : s->copy_evs) cudaEventDestroy(e);
    delete s;
}

// =============================================================================
// single stages
// =============================================================================
HS_API int hs_hash_packed(uint32_t k, uint32_t seed, const uint64_t *seq2, const uint32_t *inv, uint64_t n_bases,
                          uint64_t *out_hash, uint8_t *out_valid)
{
    if (!seq2 || !inv || !out_hash || !out_valid) return fail(HS_EINVAL, "null argument");
    if (k == 0 || k > 32) return fail(HS_EUNSUPPORTED, "k-mer size must be 1..32");
    NEED_DEVICE();
    if (!n_bases) return HS_OK;
    const uint64_t words = (n_bases + 31) / 32, alloc = hs_packed_words(n_bases);
    uint64_t *dseq = nullptr, *dh = nullptr;
    uint32_t *dinv = nullptr;
    uint8_t *dv = nullptr;
    unsigned long long *dst = nullptr;
    CU(cudaMalloc((void **)&dseq, alloc * 8));
    CU(cudaMalloc((void **)&dinv, alloc * 4));
    CU(cudaMalloc((void **)&dh, n_bases * 8));
    CU(cudaMalloc((void **)&dv, n_bases));
    CU(cudaMalloc((void **)&dst, ST_COUNT * sizeof(unsigned long long)));
    CU(cudaMemset(dseq, 0, alloc * 8));
    CU(cudaMemset(dinv, 0xFF, alloc * 4));
    CU(cudaMemset(dh, 0, n_bases * 8));
    CU(cudaMemset(dv, 0, n_bases));
    CU(cudaMemset(dst, 0, ST_COUNT * sizeof(unsigned long long)));
    CU(cudaMemcpy(dseq, seq2, words * 8, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dinv, inv, words * 4, cudaMemcpyHostToDevice));
    Chunk c{dseq, dinv, n_bases};
    StreamArgs a = base_args(c, k, seed, pow(4.0, (double)k) > pow(2.0, 32.0));
    a.emit_hash = dh; a.emit_valid = dv; a.stats = dst;
    CU(launch_stream(a, g_sm, 0));
    CU(cudaMemcpy(out_hash, dh, n_bases * 8, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(out_valid, dv, n_bases, cudaMemcpyDeviceToHost));
    cudaFree(dseq); cudaFree(dinv); cudaFree(dh); cudaFree(dv); cudaFree(dst);
    return HS_OK;
}

HS_API int hs_pack_text_device(const char *text, size_t n, uint64_t *seq2, uint32_t *inv, uint64_t cap_words,
                               uint64_t *n_bases, hs_stats_t *stats)
{
    if ((!text && n) || !seq2 || !inv || !n_bases) return fail(HS_EINVAL, "null argument");
    if (n >= ((size_t)1 << 30)) return fail(HS_EINVAL, "text too large for one device-parser chunk");
    NEED_DEVICE();
    *n_bases = 0;
    if (stats) memset(stats, 0, sizeof *stats);
    if (!n) return HS_OK;
    const uint64_t alloc = hs_packed_words(n);
    Ingest in;
    int rc = in.ensure(n, 0);
    if (rc) return rc;
    uint8_t *raw = nullptr, *codes = nullptr;
    uint64_t *dseq = nullptr;
    uint32_t *dinv = nullptr;
    unsigned long long *d_npos = nullptr, tot[4] = {0, 0, 0, 0};
    CU(cudaMalloc((void **)&raw, n + 64)); CU(cudaMalloc((void **)&codes, n + 64));
    CU(cudaMalloc((void **)&dseq, alloc * 8)); CU(cudaMalloc((void **)&dinv, alloc * 4));
    CU(cudaMalloc((void **)&d_npos, sizeof(unsigned long long)));
    CU(cudaMemcpy(raw, text, n, cudaMemcpyHostToDevice));
    FaScratch sc = in.sc;
    sc.chunk_positions = d_npos;
    CU(launch_fasta_to_codes(raw, (uint32_t)n, codes, sc, 0));
    CU(launch_pack_codes_dyn(codes, d_npos, dseq, dinv, alloc, 0));
    CU(cudaMemcpy(tot, in.d_totals, sizeof tot, cudaMemcpyDeviceToHost));
    const uint64_t words = (tot[0] + 31) / 32;
    if (words > cap_words) rc = fail(HS_EINVAL, "output capacity too small");
    if (rc == HS_OK && words) {
        CU(cudaMemcpy(seq2, dseq, words * 8, cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(inv, dinv, words * 4, cudaMemcpyDeviceToHost));
    }
    *n_bases = tot[0];
    if (stats) { stats->n_positions = tot[0]; stats->n_bases = tot[1]; stats->n_records = tot[2]; }
    cudaFree(raw); cudaFree(codes); cudaFree(dseq); cudaFree(dinv); cudaFree(d_npos);
    in.release();
    return rc;
}

HS_API int hs_db_probe(hs_db *db, const uint64_t *hashes, uint64_t n, uint32_t *out_entry)
{
    if (!db || (!hashes && n) || (!out_entry && n)) return fail(HS_EINVAL, "null argument");
    ON_DEVICE(db->device);
    if (!n) return HS_OK;
    uint64_t *dh = nullptr;
    uint32_t *de = nullptr;
    unsigned long long *dst = nullptr;
    CU(cudaMalloc((void **)&dh, n * 8));
    CU(cudaMalloc((void **)&de, n * 4));
    CU(cudaMalloc((void **)&dst, 2 * sizeof(unsigned long long)));
    CU(cudaMemset(dst, 0, 2 * sizeof(unsigned long long)));
    CU(cudaMemcpy(dh, hashes, n * 8, cudaMemcpyHostToDevice));
    CU(launch_probe(db->view(), dh, n, de, dst, db->sm, 0));
    CU(cudaMemcpy(out_entry, de, n * 4, cudaMemcpyDeviceToHost));
    cudaFree(dh); cudaFree(de); cudaFree(dst);
    return HS_OK;
}

HS_API int hs_db_probe_device(hs_db *db, const void *d_hashes, uint64_t n, uint64_t *n_hits, uint64_t *n_bucket_reads,
                              float *ms)
{
    if (!db || (!d_hashes && n)) return fail(HS_EINVAL, "null argument");
    ON_DEVICE(db->device);
    unsigned long long *dst = nullptr, h[2] = {0, 0};
    cudaEvent_t e0, e1;
    CU(cudaMalloc((void **)&dst, 2 * sizeof(unsigned long long)));
    CU(cudaMemset(dst, 0, 2 * sizeof(unsigned long long)));
    CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
    CU(cudaEventRecord(e0, 0));
    CU(launch_probe(db->view(), (const uint64_t *)d_hashes, n, nullptr, dst, db->sm, 0));
    CU(cudaEventRecord(e1, 0));
    CU(cudaEventSynchronize(e1));
    float t = 0;
    CU(cudaEventElapsedTime(&t, e0, e1));
    CU(cudaMemcpy(h, dst, sizeof h, cudaMemcpyDeviceToHost));
    if (n_hits) *n_hits = h[0];
    if (n_bucket_reads) *n_bucket_reads = h[1];
    if (ms) *ms = t;
    cudaFree(dst); cudaEventDestroy(e0); cudaEventDestroy(e1);
    return HS_OK;
}

HS_API int hs_gather_bench(const void *d_buf, uint64_t bytes, uint64_t n_reads, float *ms)
{
    if (!d_buf || bytes < 64 || !ms) return fail(HS_EINVAL, "bad argument");
    NEED_DEVICE();
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
    CU(launch_gather_bench(d_buf, bytes, n_reads, g_sm, 0));  // warm-up
    CU(cudaEventRecord(e0, 0));
    CU(launch_gather_bench(d_buf, bytes, n_reads, g_sm, 0));
    CU(cudaEventRecord(e1, 0));
    CU(cudaEventSynchronize(e1));
    CU(cudaEventElapsedTime(ms, e0, e1));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    return HS_OK;
}

HS_API int hs_db_entry_ids(hs_db *db, uint32_t *out)
{
    if (!db || !out) return fail(HS_EINVAL, "null argument");
    ON_DEVICE(db->device);
    if (db->n_entries) CU(cudaMemcpy(out, db->d_canon, db->n_entries * 4, cudaMemcpyDeviceToHost));
    return HS_OK;
}

HS_API int hs_stat_batch(uint32_t k, uint64_t set_size, uint64_t n, const uint64_t *shared, const uint64_t *size,
                         double *identity, double *pvalue)
{
    if ((!shared || !size || !identity || !pvalue) && n) return fail(HS_EINVAL, "null argument");
    NEED_DEVICE();
    if (!n) return HS_OK;
    uint64_t *dx = nullptr, *dn = nullptr;
    double *di = nullptr, *dp = nullptr;
    CU(cudaMalloc((void **)&dx, n * 8)); CU(cudaMalloc((void **)&dn, n * 8));
    CU(cudaMalloc((void **)&di, n * 8)); CU(cudaMalloc((void **)&dp, n * 8));
    CU(cudaMemcpy(dx, shared, n * 8, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dn, size, n * 8, cudaMemcpyHostToDevice));
    CU(launch_stats(k, set_size, nullptr, n, nullptr, dx, nullptr, dn, di, dp, 0));
    CU(cudaMemcpy(identity, di, n * 8, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(pvalue, dp, n * 8, cudaMemcpyDeviceToHost));
    cudaFree(dx); cudaFree(dn); cudaFree(di); cudaFree(dp);
    return HS_OK;
}

// =============================================================================
// `mash sketch` of a genome collection (SURVEY.md 8f rank 1)
// =============================================================================
// Host threads read, inflate and pack whole files; the calling thread lays the packed genomes out
// in batches -- every genome on a tile boundary, followed by at least one invalid position -- and
// hashes a batch with one k_stream launch (MODE 4), each genome into its own set of the distinct
// hashes <= its threshold tau.  One launch of k_sketch_select then sorts every set.
//
// Threshold.  With L = the genome's valid positions (>= its valid k-mers >= its distinct k-mers D),
// tau = lambda / L of the hash range makes the set expect D * lambda / L <= lambda values, lambda =
// s + 6 sqrt(s) + 8, and the set takes lambda + 6 sqrt(lambda) + 8 before it overflows (tau = the top
// of the range, and room for L values, when L is smaller than that).
// Exactness.  Without overflow the set holds every distinct hash <= tau, so its s smallest are the
// sketch when it holds >= s of them or when tau is the top of the range.  Otherwise the genome is
// streamed again with another tau: higher when it held too few (D << L: repeats), lower when it
// overflowed.  The number of distinct hashes <= tau, N(tau), is monotone in tau.  A genome keeps the
// largest tau known to give N < s (lo) and the smallest known to overflow (hi, N > limit > s); once
// both exist the next tau is their midpoint, which lies strictly between them (N(hi) - N(lo) >= 3,
// and distinct hashes are distinct integers), so the interval shrinks every pass.  Before that, tau
// only grows (at least x2, to the top at most) or only shrinks (/8, and N(0) <= 1 cannot overflow):
// the search ends, at the latest, after a few dozen passes.
namespace {

constexpr uint32_t kSketchBatchTiles = 4096;              // 32 M positions, 12 MB of packed words per batch
constexpr uint64_t kSketchSetWords = (uint64_t)8 << 20;   // 64 MB of sets per batch: L2 holds them while they fill
constexpr uint32_t kSketchMaxCap = 1u << 24;              // mixset_slot spreads a set over at most 2^24 slots
constexpr uint64_t kTilePositions = (uint64_t)kTileWords * kBasesPerWord;

// a buffer with a single owner that grows on demand (device memory, or pinned host memory)
template <class T, bool HOST>
struct Grow {
    T *p = nullptr;
    size_t cap = 0;
    cudaError_t need(size_t n)
    {
        if (n <= cap) return cudaSuccess;
        release();
        n = std::max<size_t>(n + n / 2, 64);
        const cudaError_t e = HOST ? cudaHostAlloc((void **)&p, n * sizeof(T), cudaHostAllocDefault)
                                   : cudaMalloc((void **)&p, n * sizeof(T));
        if (e == cudaSuccess) cap = n; else p = nullptr;
        return e;
    }
    void release()
    {
        if (p) { if (HOST) cudaFreeHost(p); else cudaFree(p); }
        p = nullptr; cap = 0;
    }
};

// every CUDA resource of a sketcher, released in one place
struct SketchDev {
    bool ready = false;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[4] = {};
    unsigned long long *stats = nullptr;
    Grow<uint64_t, false> seq, sets, out, out_off;
    Grow<uint32_t, false> inv, tile_genome, n_out;
    Grow<SketchSlot, false> slots;
    Grow<uint64_t, true> h_seq, h_out, h_out_off;
    Grow<uint32_t, true> h_inv, h_tile_genome, h_n_out;
    Grow<SketchSlot, true> h_slots;
    int init()
    {
        if (ready) return HS_OK;
        ready = true;   // from here on release() owns whatever was created
        CU(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        for (auto &e : ev) CU(cudaEventCreate(&e));
        CU(cudaMalloc((void **)&stats, ST_COUNT * sizeof(unsigned long long)));
        CU(cudaMemsetAsync(stats, 0, ST_COUNT * sizeof(unsigned long long), stream));
        return HS_OK;
    }
    void release()
    {
        if (stream) cudaStreamSynchronize(stream);
        seq.release(); sets.release(); out.release(); out_off.release(); inv.release(); tile_genome.release();
        n_out.release(); slots.release(); h_seq.release(); h_out.release(); h_out_off.release(); h_inv.release();
        h_tile_genome.release(); h_n_out.release(); h_slots.release();
        cudaFree(stats); stats = nullptr;
        for (auto &e : ev) { if (e) cudaEventDestroy(e); e = nullptr; }
        if (stream) cudaStreamDestroy(stream);
        stream = nullptr;
        ready = false;
    }
};

struct SkInput {
    std::string path;                    // a file ...
    const char *text = nullptr;          // ... or text in host memory (hs_sketch_text) ...
    size_t n = 0;
    bool packed = false;                 // ... or packed words already copied into the genome (hs_sketch_packed_device)
};

struct SkGenome {
    std::vector<uint64_t> seq;           // packed words, kept until the sketch is final (a re-stream needs them)
    std::vector<uint32_t> inv;
    uint64_t n_pos = 0, valid = 0, length = 0, n_records = 0;
    std::string header, err;
    std::vector<uint64_t> hashes;
    double t_read = 0, t_pack = 0;
    uint64_t tau = 0, lo = 0, hi = 0;    // threshold, and the bounds of its search (see above)
    bool has_lo = false, has_hi = false;
    uint32_t cap = 0;                    // set slots
    uint64_t tiles() const { return n_pos / kTilePositions + 1; }   // >= 1 invalid position at the end
};

}  // namespace

struct hs_sketcher {
    int device = 0;
    uint32_t k = 21, s = 1000, seed = 42;
    bool use64 = true;
    int threads = 1;
    bool ran = false;
    std::vector<SkInput> inputs;
    std::vector<SkGenome> gen;
    std::vector<uint32_t> retry;         // genomes whose pass did not settle their sketch
    hs_sketch_stats_t st{};
    SketchDev dev;
    uint64_t top() const { return use64 ? ~0ull : 0xFFFFFFFFull; }
    double lambda() const { return (double)s + 6.0 * sqrt((double)s) + 8.0; }
};

namespace {

// read + inflate + pack one input (host thread; no CUDA calls, no hs_last_error)
void sketch_ingest(SkGenome &g, const SkInput &in)
{
    if (in.packed) return;
    std::vector<char> buf;
    const char *t = in.text;
    size_t n = in.n;
    double t0 = now_s();
    if (!in.path.empty()) {
        std::string err;
        if (!slurp_file(in.path, buf, err)) { g.err = "could not open " + in.path + " for reading."; return; }
        t = buf.data(); n = buf.size();
        const double t1 = now_s();
        g.t_read = t1 - t0;
        t0 = t1;
    }
    // what the .msh comment is made of (cli.py): records = "\n>" count + a leading '>', first header line
    g.n_records = (n && t[0] == '>') ? 1 : 0;
    for (const char *p = t; n && (p = (const char *)memmem(p, (size_t)(t + n - p), "\n>", 2)); p += 2) g.n_records++;
    if (n && t[0] == '>') {
        const char *nl = (const char *)memchr(t, '\n', n);
        const size_t end = nl ? (size_t)(nl - t) : n - 1;   // Python's text[1:text.find(b"\n")]
        if (end > 1) g.header.assign(t + 1, end - 1);
    }
    g.seq.resize(pack_words_bound(n));
    g.inv.resize(pack_words_bound(n));
    PackStats ps;
    pack_text_span(t, n, g.seq.data(), g.inv.data(), &ps);
    const uint64_t words = (ps.n_positions + 31) / 32;
    g.seq.resize(words); g.inv.resize(words);
    g.n_pos = ps.n_positions;
    g.length = ps.n_seq_bases;
    for (uint32_t w : g.inv) g.valid += 32 - (uint64_t)__builtin_popcount(w);
    g.t_pack = now_s() - t0;
}

// first threshold and set size of a genome
int sketch_plan(hs_sketcher *sk, SkGenome &g)
{
    const double lam = sk->lambda(), room = lam + 6.0 * sqrt(lam) + 8.0;
    uint64_t need;
    if ((double)g.valid <= room) {
        g.tau = sk->top();
        need = g.valid;
    } else {
        const long double t = (long double)lam / (long double)g.valid * (sk->use64 ? 18446744073709551616.0L : 4294967296.0L);
        g.tau = t >= (long double)sk->top() ? sk->top() : (uint64_t)t;
        need = (uint64_t)ceil(room);
    }
    uint64_t cap = 64;
    while (cap < 2 * need + 2) cap <<= 1;
    if (cap > kSketchMaxCap) return fail(HS_EUNSUPPORTED, "sketch size too large for a genome of this size");
    g.cap = (uint32_t)cap;
    return HS_OK;
}

// the genome's words [w0, w1) into the staging at tile t0, padded with invalid positions to `tiles` tiles
uint32_t sketch_stage(SketchDev &d, const SkGenome &g, uint64_t w0, uint64_t w1, uint32_t tiles, uint32_t t0, uint32_t slot)
{
    uint64_t *sq = d.h_seq.p + (size_t)t0 * kTileWords;
    uint32_t *iv = d.h_inv.p + (size_t)t0 * kTileWords;
    memcpy(sq, g.seq.data() + w0, (w1 - w0) * 8);
    memcpy(iv, g.inv.data() + w0, (w1 - w0) * 4);
    const size_t pad = (size_t)tiles * kTileWords - (w1 - w0);
    memset(sq + (w1 - w0), 0, pad * 8);
    memset(iv + (w1 - w0), 0xFF, pad * 4);
    for (uint32_t t = 0; t < tiles; t++) d.h_tile_genome.p[t0 + t] = slot;
    return tiles;
}

// hash the staged tiles [0, tiles) into the batch's sets
int sketch_launch(hs_sketcher *sk, uint32_t tiles)
{
    SketchDev &d = sk->dev;
    const size_t words = (size_t)tiles * kTileWords;
    CU(d.seq.need(words)); CU(d.inv.need(words)); CU(d.tile_genome.need(tiles));
    CU(cudaMemcpyAsync(d.seq.p, d.h_seq.p, words * 8, cudaMemcpyHostToDevice, d.stream));
    CU(cudaMemcpyAsync(d.inv.p, d.h_inv.p, words * 4, cudaMemcpyHostToDevice, d.stream));
    CU(cudaMemcpyAsync(d.tile_genome.p, d.h_tile_genome.p, (size_t)tiles * 4, cudaMemcpyHostToDevice, d.stream));
    StreamArgs a;
    memset(&a, 0, sizeof a);
    a.seq = d.seq.p; a.inv = d.inv.p; a.n_bases = tiles * kTilePositions; a.n_tiles = tiles;
    a.k = (int)sk->k; a.seed = sk->seed; a.use64 = sk->use64; a.stats = d.stats;
    a.sk = SketchView{d.tile_genome.p, d.slots.p, d.sets.p};
    CU(cudaEventRecord(d.ev[0], d.stream));
    CU(launch_stream(a, g_sm, d.stream));
    CU(cudaEventRecord(d.ev[1], d.stream));
    // the staging is refilled next: wait for the copies (and take the kernel time with them)
    CU(cudaEventSynchronize(d.ev[1]));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, d.ev[0], d.ev[1]));
    sk->st.ms_stream += ms;
    sk->st.n_launches++;
    return HS_OK;
}

// one batch: genomes ids (all of them fit kSketchBatchTiles, or a single genome streamed piece by piece)
int sketch_batch(hs_sketcher *sk, const std::vector<uint32_t> &ids)
{
    SketchDev &d = sk->dev;
    const uint32_t n = (uint32_t)ids.size();
    CU(d.h_slots.need(n)); CU(d.slots.need(n)); CU(d.h_out_off.need(n)); CU(d.out_off.need(n));
    CU(d.h_n_out.need(n)); CU(d.n_out.need(n));
    uint64_t set_words = 0, out_words = 0, tiles = 0;
    uint32_t max_cap = 0;
    for (uint32_t j = 0; j < n; j++) {
        const SkGenome &g = sk->gen[ids[j]];
        SketchSlot &sl = d.h_slots.p[j];
        memset(&sl, 0, sizeof sl);
        sl.st.tau = g.tau;
        sl.set_off = set_words;
        sl.mask = g.cap - 1; sl.limit = g.cap / 2;
        d.h_out_off.p[j] = out_words;
        set_words += g.cap;
        out_words += std::min<uint64_t>(sk->s, g.cap);
        max_cap = std::max(max_cap, g.cap);
        tiles += g.tiles();
    }
    CU(d.sets.need(set_words)); CU(d.out.need(out_words)); CU(d.h_out.need(out_words));
    const uint64_t stage_tiles = std::min<uint64_t>(tiles, kSketchBatchTiles);
    CU(d.h_seq.need(stage_tiles * kTileWords)); CU(d.h_inv.need(stage_tiles * kTileWords)); CU(d.h_tile_genome.need(stage_tiles));
    CU(cudaMemcpyAsync(d.slots.p, d.h_slots.p, n * sizeof(SketchSlot), cudaMemcpyHostToDevice, d.stream));
    CU(cudaMemcpyAsync(d.out_off.p, d.h_out_off.p, n * 8, cudaMemcpyHostToDevice, d.stream));
    CU(cudaMemsetAsync(d.sets.p, 0xFF, set_words * 8, d.stream));
    sk->st.n_batches++;
    if (tiles <= kSketchBatchTiles) {
        uint32_t t = 0;
        for (uint32_t j = 0; j < n; j++) {
            const SkGenome &g = sk->gen[ids[j]];
            t += sketch_stage(d, g, 0, g.seq.size(), (uint32_t)g.tiles(), t, j);
        }
        int rc = sketch_launch(sk, t);
        if (rc) return rc;
    } else {
        // a genome larger than a batch: pieces of one launch each, into the same set.  Each piece after the
        // first starts one word early: k-mers that end in its second word read their first bases there
        // (k <= 32), and the k-mers that end in the repeated word were offered before (sets keep one copy).
        const SkGenome &g = sk->gen[ids[0]];
        const uint64_t nw = g.seq.size(), piece = (uint64_t)kSketchBatchTiles * kTileWords - 1;
        for (uint64_t w0 = 0;;) {
            const uint64_t w1 = std::min(nw, w0 + piece);
            int rc = sketch_launch(sk, sketch_stage(d, g, w0, w1, (uint32_t)((w1 - w0 + kTileWords - 1) / kTileWords), 0, 0));
            if (rc) return rc;
            if (w1 == nw) break;
            w0 = w1 - 1;
        }
    }
    CU(cudaEventRecord(d.ev[2], d.stream));
    CU(launch_sketch_select(d.slots.p, n, max_cap, d.sets.p, sk->s, d.out_off.p, d.out.p, d.n_out.p, d.stream));
    CU(cudaEventRecord(d.ev[3], d.stream));
    sk->st.n_launches++;
    CU(cudaMemcpyAsync(d.h_slots.p, d.slots.p, n * sizeof(SketchSlot), cudaMemcpyDeviceToHost, d.stream));
    CU(cudaMemcpyAsync(d.h_n_out.p, d.n_out.p, n * 4, cudaMemcpyDeviceToHost, d.stream));
    CU(cudaMemcpyAsync(d.h_out.p, d.out.p, out_words * 8, cudaMemcpyDeviceToHost, d.stream));
    CU(cudaStreamSynchronize(d.stream));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, d.ev[2], d.ev[3]));
    sk->st.ms_select += ms;
    // settle or re-stream each genome (see the argument at the top of this section)
    const uint64_t top = sk->top();
    for (uint32_t j = 0; j < n; j++) {
        SkGenome &g = sk->gen[ids[j]];
        const MixState &r = d.h_slots.p[j].st;
        const uint64_t have = (uint64_t)r.count + (r.has_max ? 1 : 0);
        if (!r.overflow && (have >= sk->s || g.tau == top)) {
            const uint64_t *h = d.h_out.p + d.h_out_off.p[j];
            g.hashes.assign(h, h + d.h_n_out.p[j]);
            if (r.has_max && g.hashes.size() < sk->s) g.hashes.push_back(~0ull);   // hash 2^64-1 (kEmptyKey) is never stored in a set
            std::vector<uint64_t>().swap(g.seq);
            std::vector<uint32_t>().swap(g.inv);
            continue;
        }
        if (r.overflow) { g.hi = g.tau; g.has_hi = true; }
        else { g.lo = g.tau; g.has_lo = true; }
        if (g.has_lo && g.has_hi) {
            g.tau = g.lo + (g.hi - g.lo) / 2;
        } else if (g.has_hi) {
            g.tau /= 8;
        } else {
            const long double f = std::max(2.0L, (long double)sk->lambda() / (long double)std::max<uint32_t>(r.count, 1));
            const long double t = (long double)g.tau * f + 1.0L;
            g.tau = t >= (long double)top ? top : (uint64_t)t;
        }
        sk->retry.push_back(ids[j]);
        sk->st.n_passes++;
    }
    return HS_OK;
}

// batch the genomes in `order` (in that order) and sketch them
template <class Next>
int sketch_genomes(hs_sketcher *sk, Next &&next)
{
    std::vector<uint32_t> cur;
    uint64_t cur_tiles = 0, cur_sets = 0;
    auto flush = [&]() -> int {
        if (cur.empty()) return HS_OK;
        int rc = sketch_batch(sk, cur);
        cur.clear(); cur_tiles = 0; cur_sets = 0;
        return rc;
    };
    for (;;) {
        int64_t i = -1;
        int rc = next(i);
        if (rc) return rc;
        if (i < 0) break;
        const SkGenome &g = sk->gen[(size_t)i];
        if (!g.n_pos) continue;   // empty: an empty sketch
        const uint64_t tg = g.tiles();
        if (tg > kSketchBatchTiles) {
            if ((rc = flush()) || (rc = sketch_batch(sk, {(uint32_t)i}))) return rc;
            continue;
        }
        if (cur_tiles + tg > kSketchBatchTiles || (!cur.empty() && cur_sets + g.cap > kSketchSetWords))
            if ((rc = flush())) return rc;
        cur.push_back((uint32_t)i);
        cur_tiles += tg; cur_sets += g.cap;
    }
    return flush();
}

int sketcher_run(hs_sketcher *sk)
{
    int rc = sk->dev.init();
    if (rc) return rc;
    const size_t n = sk->inputs.size();
    sk->gen.resize(n);
    // host threads take whole inputs in order and run at most ~two batches of positions ahead of the GPU
    const uint64_t ahead_max = 2ull * kSketchBatchTiles * kTilePositions;
    std::mutex mu;
    std::condition_variable cv;
    std::vector<char> ready(n, 0);
    size_t next_in = 0, consumed = 0;
    uint64_t ahead = 0;
    bool stop = false;
    auto worker = [&]() {
        for (;;) {
            size_t i;
            {
                std::unique_lock<std::mutex> lk(mu);
                cv.wait(lk, [&] { return stop || next_in >= n || next_in <= consumed || ahead < ahead_max; });
                if (stop || next_in >= n) return;
                i = next_in++;
            }
            sketch_ingest(sk->gen[i], sk->inputs[i]);
            {
                std::lock_guard<std::mutex> lk(mu);
                ready[i] = 1;
                ahead += sk->gen[i].n_pos;
            }
            cv.notify_all();
        }
    };
    std::vector<std::thread> pool;
    for (int t = 0; t < std::min<int>(sk->threads, (int)std::max<size_t>(n, 1)); t++) pool.emplace_back(worker);
    size_t at = 0;
    rc = sketch_genomes(sk, [&](int64_t &i) -> int {
        if (at == n) return HS_OK;
        const double t0 = now_s();
        {
            std::unique_lock<std::mutex> lk(mu);
            cv.wait(lk, [&] { return ready[at] != 0; });
            consumed = at + 1;
            ahead -= sk->gen[at].n_pos;
        }
        cv.notify_all();
        sk->st.t_wait_s += now_s() - t0;
        SkGenome &g = sk->gen[at];
        if (!g.err.empty()) return fail(HS_EIO, g.err);
        if (g.n_pos) {
            int r = sketch_plan(sk, g);
            if (r) return r;
        }
        i = (int64_t)at++;
        return HS_OK;
    });
    {
        std::lock_guard<std::mutex> lk(mu);
        stop = true;
    }
    cv.notify_all();
    for (auto &t : pool) t.join();
    // re-streams: genomes whose first pass did not settle, batched again with their new thresholds
    while (rc == HS_OK && !sk->retry.empty()) {
        std::vector<uint32_t> again;
        again.swap(sk->retry);
        size_t r = 0;
        rc = sketch_genomes(sk, [&](int64_t &i) -> int {
            i = r < again.size() ? (int64_t)again[r++] : -1;
            return HS_OK;
        });
    }
    for (const SkGenome &g : sk->gen) {
        sk->st.n_bases += g.length;
        sk->st.n_positions += g.n_pos;
        sk->st.t_read_s += g.t_read;
        sk->st.t_pack_s += g.t_pack;
    }
    sk->st.n_genomes = n;
    return rc;
}

int sketcher_new(uint32_t k, uint32_t s_, uint32_t seed, int threads, hs_sketcher **out)
{
    if (!out) return fail(HS_EINVAL, "null argument");
    if (k == 0 || k > 32) return fail(HS_EUNSUPPORTED, "k-mer size must be 1..32");
    if (s_ == 0) return fail(HS_EINVAL, "sketch size must be positive");
    NEED_DEVICE();
    auto *sk = new hs_sketcher();
    sk->device = g_device;
    sk->k = k; sk->s = s_; sk->seed = seed;
    sk->use64 = k > 16;   // 4^k > 2^32: 64-bit hashes (S1)
    sk->threads = threads < 1 ? 1 : threads;
    *out = sk;
    return HS_OK;
}

// a batch of one, for the single-genome entry points
int sketch_one(hs_sketcher *sk, uint64_t *out_hashes, uint32_t *n_out, uint64_t *length)
{
    sk->ran = true;
    int rc = sketcher_run(sk);
    if (rc) return rc;
    const SkGenome &g = sk->gen[0];
    *n_out = (uint32_t)g.hashes.size();
    memcpy(out_hashes, g.hashes.data(), g.hashes.size() * 8);
    if (length) *length = g.length;
    return HS_OK;
}

}  // namespace

HS_API int hs_sketcher_new(uint32_t k, uint32_t s_, uint32_t seed, int host_threads, hs_sketcher **out)
{
    return sketcher_new(k, s_, seed, host_threads, out);
}

HS_API int hs_sketcher_add_file(hs_sketcher *sk, const char *path)
{
    if (!sk || !path) return fail(HS_EINVAL, "null argument");
    if (sk->ran) return fail(HS_ESTATE, "the sketcher has already run");
    SkInput in;
    in.path = path;
    if (in.path.empty()) return fail(HS_EINVAL, "empty path");
    sk->inputs.push_back(in);
    return HS_OK;
}

HS_API int hs_sketcher_run(hs_sketcher *sk)
{
    if (!sk) return fail(HS_EINVAL, "null argument");
    if (sk->ran) return fail(HS_ESTATE, "the sketcher has already run");
    ON_DEVICE(sk->device);
    sk->ran = true;
    const double t0 = now_s();
    const int rc = sketcher_run(sk);
    sk->st.t_total_s = now_s() - t0;
    return rc;
}

HS_API int hs_sketcher_result(const hs_sketcher *sk, uint64_t i, const uint64_t **hashes, uint32_t *n, uint64_t *length,
                              uint64_t *n_records, const char **header, uint64_t *header_len)
{
    if (!sk) return fail(HS_EINVAL, "null argument");
    if (!sk->ran || sk->gen.size() != sk->inputs.size()) return fail(HS_ESTATE, "hs_sketcher_run has not completed");
    if (i >= sk->gen.size()) return fail(HS_EINVAL, "input index out of range");
    const SkGenome &g = sk->gen[i];
    if (hashes) *hashes = g.hashes.data();
    if (n) *n = (uint32_t)g.hashes.size();
    if (length) *length = g.length;
    if (n_records) *n_records = g.n_records;
    if (header) *header = g.header.data();
    if (header_len) *header_len = g.header.size();
    return HS_OK;
}

HS_API int hs_sketcher_stats(const hs_sketcher *sk, hs_sketch_stats_t *stats)
{
    if (!sk || !stats) return fail(HS_EINVAL, "null argument");
    *stats = sk->st;
    return HS_OK;
}

HS_API void hs_sketcher_free(hs_sketcher *sk)
{
    if (!sk) return;
    if (sk->dev.ready) {
        cudaSetDevice(sk->device);
        sk->dev.release();
    }
    delete sk;
}

HS_API int hs_sketch_packed_device(uint32_t k, uint32_t s_, uint32_t seed, const void *d_seq2, const void *d_inv,
                                   uint64_t n_bases, uint64_t *out_hashes, uint32_t *n_out)
{
    if (!out_hashes || !n_out || ((!d_seq2 || !d_inv) && n_bases)) return fail(HS_EINVAL, "null argument");
    hs_sketcher *sk = nullptr;
    int rc = sketcher_new(k, s_ ? s_ : 1, seed, 1, &sk);
    if (rc) return rc;
    *n_out = 0;
    SkInput in;
    in.packed = true;
    sk->inputs.push_back(in);
    sk->gen.resize(1);
    SkGenome &g = sk->gen[0];
    const uint64_t words = (n_bases + 31) / 32;
    g.seq.resize(words); g.inv.resize(words);
    cudaError_t e = cudaMemcpy(g.seq.data(), d_seq2, words * 8, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(g.inv.data(), d_inv, words * 4, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) rc = fail(HS_ECUDA, std::string("copying the packed genome: ") + cudaGetErrorString(e));
    if (rc == HS_OK) {
        if (n_bases % 32) g.inv[words - 1] |= (1u << (32 - n_bases % 32)) - 1u;   // positions >= n_bases are not the genome's
        g.n_pos = n_bases;
        for (uint32_t w : g.inv) g.valid += 32 - (uint64_t)__builtin_popcount(w);
        rc = sketch_one(sk, out_hashes, n_out, nullptr);
    }
    hs_sketcher_free(sk);
    return rc;
}

HS_API int hs_sketch_text(uint32_t k, uint32_t s_, uint32_t seed, const char *text, size_t n, uint64_t *out_hashes,
                          uint32_t *n_out, uint64_t *length)
{
    if ((!text && n) || !out_hashes || !n_out) return fail(HS_EINVAL, "null argument");
    hs_sketcher *sk = nullptr;
    int rc = sketcher_new(k, s_ ? s_ : 1, seed, 1, &sk);
    if (rc) return rc;
    *n_out = 0;
    SkInput in;
    in.text = text; in.n = n;
    sk->inputs.push_back(in);
    rc = sketch_one(sk, out_hashes, n_out, length);
    hs_sketcher_free(sk);
    return rc;
}

HS_API int hs_pack_codes_device(const void *d_codes, uint64_t n, void *d_seq2, void *d_inv, void *cuda_stream)
{
    if ((!d_codes && n) || !d_seq2 || !d_inv) return fail(HS_EINVAL, "null argument");
    NEED_DEVICE();
    CU(launch_pack_codes((const uint8_t *)d_codes, n, (uint64_t *)d_seq2, (uint32_t *)d_inv, hs_packed_words(n),
                         (cudaStream_t)cuda_stream));
    return HS_OK;
}

// =============================================================================
// SURVEY.md 8f rank 4: weighted-LCA vote (classification_cami.py:251-308)
// =============================================================================
HS_API int hs_lca_weighted(uint64_t n_q, const uint64_t *q_off, const int32_t *tax, const double *w, uint64_t n_tax,
                           const uint32_t *names, uint32_t *out_names, uint32_t *out_depth, double *out_conf, uint8_t *out_any)
{
    if (n_q && (!q_off || !out_names || !out_depth || !out_conf || !out_any)) return fail(HS_EINVAL, "null argument");
    NEED_DEVICE();
    if (!n_q) return HS_OK;
    const uint64_t n_a = q_off[n_q];
    if (n_a && (!tax || !w)) return fail(HS_EINVAL, "null argument");
    if (n_tax && !names) return fail(HS_EINVAL, "null argument");
    for (uint64_t j = 0; j < n_a; j++)
        if (tax[j] >= 0 && (uint64_t)tax[j] >= n_tax) return fail(HS_EINVAL, "taxid row out of range");
    DevBufs d;
    LcaArgs a;
    memset(&a, 0, sizeof a);
    uint64_t *d_off = nullptr;
    int32_t *d_tax = nullptr;
    double *d_w = nullptr;
    uint32_t *d_names = nullptr;
    CU(d.alloc(&d_off, (n_q + 1) * 8));
    CU(d.alloc(&d_tax, n_a * 4)); CU(d.alloc(&d_w, n_a * 8)); CU(d.alloc(&d_names, n_tax * kLcaRanks * 4));
    CU(d.alloc(&a.s_tax, n_a * 4)); CU(d.alloc(&a.s_w, n_a * 8)); CU(d.alloc(&a.s_name, n_a * 4)); CU(d.alloc(&a.s_nw, n_a * 8));
    CU(d.alloc(&a.out_names, n_q * kLcaRanks * 4)); CU(d.alloc(&a.out_depth, n_q * 4));
    CU(d.alloc(&a.out_conf, n_q * 8)); CU(d.alloc(&a.out_any, n_q));
    CU(cudaMemcpy(d_off, q_off, (n_q + 1) * 8, cudaMemcpyHostToDevice));
    if (n_a) { CU(cudaMemcpy(d_tax, tax, n_a * 4, cudaMemcpyHostToDevice)); CU(cudaMemcpy(d_w, w, n_a * 8, cudaMemcpyHostToDevice)); }
    if (n_tax) CU(cudaMemcpy(d_names, names, n_tax * kLcaRanks * 4, cudaMemcpyHostToDevice));
    CU(cudaMemset(a.out_names, 0, n_q * kLcaRanks * 4));
    a.n_q = n_q; a.q_off = d_off; a.tax = d_tax; a.w = d_w; a.names = d_names;
    CU(launch_weighted_lca(a, g_sm, 0));
    CU(cudaMemcpy(out_names, a.out_names, n_q * kLcaRanks * 4, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(out_depth, a.out_depth, n_q * 4, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(out_conf, a.out_conf, n_q * 8, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(out_any, a.out_any, n_q, cudaMemcpyDeviceToHost));
    return HS_OK;
}
