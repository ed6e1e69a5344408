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
#include <errno.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <type_traits>
#include <vector>

#include "../../include/hymet_screen.h"
#include "cuda_owned.h"
#include "distance_kernels.h"
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

double now_s()
{
    return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

uint64_t tiles_for(uint64_t n_bases) { return ((n_bases + 31) / 32 + kTileWords - 1) / kTileWords; }

// ---- device arena for query chunks ------------------------------------------
struct Arena {
    struct Slab { DevBuf<char> mem; size_t used = 0; };
    std::vector<Slab> slabs;
    size_t slab_bytes = (size_t)256 << 20;
    size_t cur = 0;
    cudaError_t alloc(size_t n, void **out)
    {
        n = (n + 255) & ~(size_t)255;
        while (cur < slabs.size() && slabs[cur].used + n > slabs[cur].mem.cap()) cur++;
        if (cur == slabs.size()) {
            Slab s;
            cudaError_t e = s.mem.grow(std::max(n, slab_bytes));
            if (e != cudaSuccess) return e;
            slabs.push_back(std::move(s));
        }
        *out = slabs[cur].mem.get() + slabs[cur].used;
        slabs[cur].used += n;
        return cudaSuccess;
    }
    void reset()
    {   // slabs stay allocated: a steady-state screen never calls cudaMalloc/cudaFree
        for (auto &s : slabs) s.used = 0;
        cur = 0;
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
    struct Slot { DevBuf<uint8_t> raw, codes; Event done, copied; };
    Slot slots[kSlots];
    int next = 0;
    DevBuf<char> scan;                                  // the eight FaScratch arrays (carve)
    FaScratch sc{};
    size_t tile_cap = 0;
    std::vector<DevBuf<unsigned long long>> counter_blocks;   // per-chunk position counters (512 per block)
    size_t counters_used = 0;
    DevBuf<unsigned long long> d_totals;                // [0] positions [1] bases [2] records
    bool ready = false;

    // points sc's arrays into base (tile capacity cap), each on a 256-byte boundary as if allocated
    // alone; returns the bytes they take
    size_t carve(char *base, size_t cap)
    {
        size_t off = 0;
        auto part = [&](auto *&p, size_t n) {
            p = reinterpret_cast<std::remove_reference_t<decltype(p)>>(reinterpret_cast<uintptr_t>(base) + off);
            off += (n * sizeof(*p) + 255) & ~(size_t)255;
        };
        part(sc.masks, cap * 256); part(sc.emit, cap * 256);
        part(sc.tile_event, cap); part(sc.tile_carry, cap); part(sc.tile_event_b, cap); part(sc.tile_carry_b, cap);
        part(sc.tile_count, cap); part(sc.tile_offset, cap);
        return off;
    }
    int ensure(size_t bytes, cudaStream_t st)
    {
        if (!ready) {
            CU(d_totals.grow(4));
            // on the stream that will accumulate into it: the legacy default stream is not ordered
            // against a non-blocking stream
            CU(cudaMemsetAsync(d_totals.get(), 0, 4 * sizeof(unsigned long long), st));
            for (auto &sl : slots) {
                CU(sl.done.create(cudaEventDisableTiming | cudaEventBlockingSync));
                CU(sl.copied.create(cudaEventDisableTiming));
            }
            ready = true;
        }
        const size_t tiles = (bytes + kFaTileBytes - 1) / kFaTileBytes + 1;
        if (tiles > tile_cap) {
            cudaDeviceSynchronize();
            tile_cap = 0;   // sc points nowhere until the new scratch is carved
            const size_t cap = tiles + tiles / 4;
            CU(scan.grow(carve(nullptr, cap)));
            carve(scan.get(), cap);
            tile_cap = cap;
        }
        sc.totals = d_totals.get();
        return HS_OK;
    }
    int slot_for(size_t bytes, Slot **out)
    {
        Slot &sl = slots[next];
        next = (next + 1) % kSlots;
        CU(cudaEventSynchronize(sl.done.get()));  // throttle: at most kSlots chunks of raw text in flight
        if (sl.raw.cap() < bytes || sl.codes.cap() < bytes) {
            const size_t cap = bytes + bytes / 8 + 64;
            sl.raw.reset(); sl.codes.reset();   // both go before either grows
            CU(sl.raw.grow(cap));
            CU(sl.codes.grow(cap));
        }
        *out = &sl;
        return HS_OK;
    }
    int counter(unsigned long long **out)
    {
        if (counters_used == counter_blocks.size() * 512) {
            DevBuf<unsigned long long> b;
            CU(b.grow(512));
            counter_blocks.push_back(std::move(b));
        }
        *out = counter_blocks[counters_used / 512].get() + counters_used % 512;
        counters_used++;
        return HS_OK;
    }
};

// ---- mixture bottom-s engine (K3 control logic) --------------------------------
// The threshold tau and the live set are DEVICE state (MixState): streaming launches and
// their maintenance kernels are enqueued back to back, the host looks at the state only
// at flush.  Exactness: a value is dropped only when >= s smaller distinct values stay.
struct MixEngine {
    uint32_t s = 0, cap = 0, cand_cap = 0;
    bool use64 = true;     // 32-bit hashes (k <= 16) live in [0, 2^32): caps and tau start there
    DevBuf<uint64_t> d_set[2];
    DevBuf<MixState> d_state;
    PinnedBuf<MixState> h_state;  // pinned mirror, valid after sync_state()
    DevBuf<uint64_t> d_cand, d_scratch;
    DevBuf<uint32_t> d_hist;      // device-side selection: 2048 bins
    uint32_t sel_pad = 0;         // its sort capacity (power of two >= s + slack, <= cand_cap)
    bool fast_select = true;
    PinnedBuf<uint64_t> h_cand;   // pinned: the settled mixture travels with the state, one sync for both
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
        for (int i = 0; i < 2; i++) CU(d_set[i].grow(cap));
        CU(d_state.grow(1));
        CU(h_state.grow(1));
        CU(d_cand.grow(cand_cap));
        CU(d_scratch.grow(cand_cap));
        CU(d_hist.grow(2 * 2048 + 8));   // bin counts | bin starts | last bin
        sel_pad = 2048;
        while (sel_pad < s + 1024) sel_pad <<= 1;
        if (sel_pad > cand_cap) sel_pad = cand_cap;
        if (const char *e = getenv("HYMET_SCREEN_FAST_SELECT")) fast_select = atoi(e) != 0;
        CU(h_cand.grow(s));
        return HS_OK;
    }
    uint32_t *field(size_t off) const { return reinterpret_cast<uint32_t *>(reinterpret_cast<char *>(d_state.get()) + off); }
    int reset(cudaStream_t st, uint64_t new_tau = ~0ull, bool automatic = true)
    {
        CU(cudaMemsetAsync(d_set[0].get(), 0xFF, (size_t)cap * 8, st));
        CU(launch_mix_state_init(d_state.get(), new_tau, st));
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
        v.sets[0] = d_set[0].get(); v.sets[1] = d_set[1].get();
        v.mask = cap - 1; v.limit = cap / 2; v.tau_cap = tau_cap; v.st = d_state.get();
        return v;
    }
    int sync_state(cudaStream_t st)
    {
        CU(cudaMemcpyAsync(h_state.get(), d_state.get(), sizeof(MixState), cudaMemcpyDeviceToHost, st));
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
    DevBuf<uint64_t> d_buckets;              // n_buckets x 128 bytes: keys | canonical entry ids | overflow flag
    uint32_t n_buckets = 0, special = kNoEntry;
    DevBuf<uint32_t> d_canon;                // per stored hash: canonical entry id of its key (reference -> hashes, dense path)
    DevBuf<uint32_t> d_next;                 // per stored hash: next entry holding the same key (hash -> references, sparse path)
    DevBuf<uint64_t> d_offsets, d_lengths, d_seg_begin;
    DevBuf<uint32_t> d_seg_s;
    uint64_t device_bytes = 0;
    double t_parse = 0, t_build = 0;
    DevBuf<uint32_t> d_bloom;
    uint32_t bloom_mask = 0;
    uint64_t bloom_keys = 0;                 // keys above dense_max (what the Bloom filter holds)
    // Several .msh files screened in one pass (run_hymet_cami.sh:85-97 streams the query three times):
    // references [seg_begin[j], seg_begin[j+1]) came from file j, whose sketch size was seg_s[j].
    std::vector<uint64_t> seg_begin;
    std::vector<uint32_t> seg_s;
    TableView view() const
    {
        return TableView{d_buckets.get(), n_buckets, max_key, special, d_bloom.get(), bloom_mask, d_bloom.get() ? dense_max : max_key};
    }
};

// pinned ring the file readers pread() into: two slots per reader thread
struct FileRing {
    PinnedBuf<char> base;
    size_t slot_cap = 0;
    std::vector<Event> free_ev;   // recorded on the copy stream once a slot's text is in HBM
};

struct Staging {
    PinnedBuf<uint64_t> seq;
    PinnedBuf<uint32_t> inv;
    uint64_t cap_words = 0;
    Event free_ev;
};

struct hs_screen {
    hs_db *db = nullptr;
    // declared first, so released last (members go in reverse order, after the destructor's wait)
    Stream stream;                           // the handle's own, or the caller's (hs_screen_set_stream)
    Stream copy_stream;                      // H2D of query chunks overlaps the kernels of earlier chunks
    std::vector<Event> copy_evs;
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
    DevBuf<uint32_t> d_counts;
    DevBuf<unsigned long long> d_stats;
    // O(present hashes) bookkeeping (SparseState): ids of the non-zero counts, references with hits,
    // their depth segments.  touched_valid: the list covers every non-zero count as far as the HOST
    // knows (a dense all-reduce into counts[] invalidates it; the device flags overflow and wraps).
    DevBuf<SparseState> d_sparse;
    PinnedBuf<SparseState> h_sparse;
    DevBuf<uint32_t> d_touched, d_depths;
    DevBuf<uint32_t> d_ref_rows;   // one block: hit | seg_start | seg_fill | plain
    uint32_t *d_hit = nullptr, *d_seg_start = nullptr, *d_seg_fill = nullptr, *d_plain = nullptr;
    uint32_t touched_cap = 0, pair_cap = 0;
    bool touched_valid = true, sparse_enabled = true;
    uint32_t last_reduce_dense = 0;
    // multi-GPU: mixture merged on the device (hs_screen_mixture_merge_device)
    DevBuf<uint64_t> d_mixture, d_merge_work, d_merge_scratch;
    PinnedBuf<uint64_t> h_mixture;
    bool mixture_on_device = false;
    Event rst0, rst1;
    bool rst_pending = false;
    // result rows of the references with hits (hs_screen_finish_hits): pinned, host-mapped, written by the GPU
    PinnedBuf<char> h_rows;
    HitRows rows_host{}, rows_dev{};
    std::vector<uint32_t> hit_order;   // indices into the rows, ascending by reference, shared > 0 only
    MixEngine mix;
    std::vector<uint64_t> mixture;  // settled s smallest distinct hashes, ascending
    bool flushed = false;
    bool flush_pending = false;   // hs_screen_flush_async: selection enqueued, verdict read after the next synchronisation
    bool flush_parsed = false;    // ... and it fetched the device parser's totals
    int force_unsettled = 0;      // tests: the next mixture record says "not settled" (HYMET_SCREEN_FORCE_UNSETTLED)
    DevBuf<double> d_result;   // one block: identity | p-value | shared | median
    uint32_t *d_shared = nullptr, *d_median = nullptr;
    double *d_identity = nullptr, *d_pvalue = nullptr;
    DevBuf<char> d_win;        // -w on the dense path: best score | best length | winner
    Arena arena;
    std::vector<Chunk> chunks;
    std::vector<Staging> staging;
    std::mutex mu;  // serialises arena + launches when packer threads feed concurrently
    bool filter = true;
    uint64_t chunk_text = (uint64_t)16 << 20;
    hs_stats_t st;
    std::vector<std::pair<Event, Event>> ev_pool;
    size_t ev_used = 0;
    Event red0, red1, red2, red3;
    PinnedBuf<unsigned long long> h_stats;   // pinned: [0, ST_COUNT) kernel counters, then 4 device-parser totals
    PinnedBuf<char> h_result;   // pinned landing zone for the four result columns (24 B per sketch):
                                // a D2H copy into the caller's pageable arrays costs ~0.3 ms at N = 50 000
    ~hs_screen()
    {   // the copy stream reads the staging and the ring; both streams write buffers released below
        if (stream.get()) cudaStreamSynchronize(stream.get());
        if (copy_stream.get()) cudaStreamSynchronize(copy_stream.get());
    }
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

    // build scratch; the handle's buffers are its own from here on (deleting it releases them)
    DevBuf<uint64_t> d_hashes;
    DevBuf<uint32_t> d_flags;
    DevBuf<unsigned long long> d_nd;
    CU(db->d_buckets.grow(nb * kBucketWords));
    CU(db->d_canon.grow(std::max<uint64_t>(E, 1)));
    CU(db->d_next.grow(std::max<uint64_t>(E, 1)));
    CU(db->d_offsets.grow(N + 1));
    CU(db->d_lengths.grow(std::max<uint64_t>(N, 1)));
    CU(db->d_seg_begin.grow(db->seg_begin.size()));
    CU(db->d_seg_s.grow(db->seg_s.size()));
    CU(d_hashes.grow(std::max<uint64_t>(E, 1)));
    CU(d_flags.grow(2));
    CU(d_nd.grow(1));
    db->device_bytes = nb * kBucketWords * 8 + E * 8 + (N + 1) * 8 + N * 8;
    CU(cudaMemset(db->d_next.get(), 0xFF, std::max<uint64_t>(E, 1) * 4));   // kNoEntry = end of chain
    CU(cudaMemset(d_flags.get(), 0xFF, sizeof(uint32_t)));      // [0] special = kNoEntry
    CU(cudaMemset(d_flags.get() + 1, 0, sizeof(uint32_t)));     // [1] fail
    CU(cudaMemset(d_nd.get(), 0, sizeof(unsigned long long)));
    if (E) CU(cudaMemcpy(d_hashes.get(), hashes, E * 8, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(db->d_offsets.get(), db->offsets.data(), (N + 1) * 8, cudaMemcpyHostToDevice));
    if (N) CU(cudaMemcpy(db->d_lengths.get(), db->lengths.data(), N * 8, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(db->d_seg_begin.get(), db->seg_begin.data(), db->seg_begin.size() * 8, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(db->d_seg_s.get(), db->seg_s.data(), db->seg_s.size() * 4, cudaMemcpyHostToDevice));
    CU(launch_table_insert(db->d_buckets.get(), db->n_buckets, d_hashes.get(), E, d_flags.get(), d_flags.get() + 1, 0));
    uint32_t flags[2];
    CU(cudaMemcpy(flags, d_flags.get(), sizeof flags, cudaMemcpyDeviceToHost));
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
            CU(db->d_bloom.grow(words));
            CU(cudaMemset(db->d_bloom.get(), 0, words * 4));
            db->bloom_mask = (uint32_t)(words - 1);
            db->dense_max = plan.dense_max;
            db->bloom_keys = (uint64_t)plan.keys_above;
            CU(launch_bloom_build(db->d_bloom.get(), db->bloom_mask, db->dense_max, db->use64, d_hashes.get(), E, 0));
            db->device_bytes += words * 4;
        }
    }
    CU(launch_table_canon(db->view(), d_hashes.get(), E, db->d_canon.get(), db->d_next.get(), d_nd.get(), 0));
    unsigned long long nd = 0;
    CU(cudaMemcpy(&nd, d_nd.get(), sizeof nd, cudaMemcpyDeviceToHost));
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
    o->bloom_bytes = db->d_bloom.get() ? ((uint64_t)db->bloom_mask + 1) * 4 : 0;
    o->dense_max = db->d_bloom.get() ? db->dense_max : db->max_key;
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
    a.tab = s->db->view(); a.counts = s->d_counts.get();
    // the range test removes probes only when the keys are confined to a sliver of the hash range; a db
    // whose keys cover a quarter of it or more and has no Bloom tier probes for most k-mers: that is
    // the warp-cooperative kernel's job, as is "filter" = 0
    a.probe_all = !s->filter || (!s->db->d_bloom.get() && s->db->max_key >= ((uint64_t)1 << 62));
    if (count && s->sparse_enabled) a.sparse = SparseView{s->d_touched.get(), s->touched_cap, s->d_sparse.get()};
    const uint64_t launch_positions = (tile_end - tile_begin) * kTileWords * 32;
    a.mix = s->mix.view(mix ? s->mix.launch_cap(launch_positions) : ~0ull);
    a.stats = count ? s->d_stats.get() : s->d_stats.get() + ST_COUNT;  // re-offer passes must not double count
    if (s->ev_used == s->ev_pool.size()) {
        Event e0, e1;
        CU(e0.create()); CU(e1.create());
        s->ev_pool.emplace_back(std::move(e0), std::move(e1));
    }
    auto &ev = s->ev_pool[s->ev_used++];
    CU(cudaEventRecord(ev.first.get(), s->stream.get()));
    CU(launch_stream(a, s->db->sm, s->stream.get()));
    CU(cudaEventRecord(ev.second.get(), s->stream.get()));
    s->st.n_launches++;
    if (mix) {
        CU(launch_mix_maintain(a.mix, s->stream.get()));
        s->st.n_launches += 3;
    }
    if (!c.n_dev)  // device-parsed chunks are accounted from the parser's own totals at flush
        s->st.n_positions += std::min<uint64_t>(c.n_bases, tile_end * kTileWords * 32) - tile_begin * kTileWords * 32;
    return HS_OK;
}

SparseView sparse_view(const hs_screen *s) { return SparseView{s->sparse_enabled ? s->d_touched.get() : nullptr, s->touched_cap, s->d_sparse.get()}; }

int screen_zero(hs_screen *s)
{
    CU(cudaEventRecord(s->rst0.get(), s->stream.get()));
    if (s->sparse_enabled && s->touched_valid) {
        // counts[] back to zero in O(touched); if the list overflowed on the device, the conditional
        // dense clear does the work instead (both are enqueued, one of them returns at once)
        CU(launch_sparse_reset(sparse_view(s), s->d_counts.get(), s->db->sm, s->stream.get()));
        CU(launch_counts_clear_if_overflow(sparse_view(s), s->d_counts.get(), s->db->n_entries, s->stream.get()));
    } else {
        CU(cudaMemsetAsync(s->d_counts.get(), 0, std::max<uint64_t>(s->db->n_entries, 1) * 4, s->stream.get()));
    }
    CU(cudaMemsetAsync(s->d_sparse.get(), 0, sizeof(SparseState), s->stream.get()));
    s->touched_valid = true;
    s->mixture_on_device = false;
    CU(cudaMemsetAsync(s->d_stats.get(), 0, 2 * ST_COUNT * sizeof(unsigned long long), s->stream.get()));
    int rc = s->mix.reset(s->stream.get());
    if (rc) return rc;
    CU(cudaEventRecord(s->rst1.get(), s->stream.get()));
    s->rst_pending = true;
    s->mix.passes = 1;
    s->mixture.clear();
    s->flushed = false;
    s->flush_pending = false;
    s->chunks.clear();
    if (s->copy_stream.get()) CU(cudaStreamSynchronize(s->copy_stream.get()));
    s->arena.reset();
    s->ev_used = 0;
    s->copy_ev_used = 0;
    s->ingest.counters_used = 0;
    if (s->ingest.ready) CU(cudaMemsetAsync(s->ingest.d_totals.get(), 0, 4 * sizeof(unsigned long long), s->stream.get()));
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
        CU(launch_mix_select(m.view(~0ull), m.s, m.use64, m.d_hist.get(), m.d_cand.get(), m.sel_pad, m.d_scratch.get(), st));
        n_launches += 4;
        CU(cudaMemcpyAsync(m.h_cand.get(), m.d_cand.get(), (size_t)m.s * 8, cudaMemcpyDeviceToHost, st));
        int rc = m.sync_state(st);
        if (rc) return rc;
        const MixState &hs_ = *m.h_state.get();
        if (!hs_.overflow && !hs_.sel_too_many && hs_.n_out <= m.sel_pad && (hs_.n_unique >= m.s || hs_.tau == ~0ull)) {
            const uint32_t nu = std::min(hs_.n_unique, m.s);
            out.assign(m.h_cand.get(), m.h_cand.get() + nu);
            if (hs_.has_max && out.size() < m.s) out.push_back(~0ull);  // hash == 2^64-1 present
            return HS_OK;
        }
    }
    for (int round = 0; round < 40; round++) {
        int rc = m.sync_state(st);
        if (rc) return rc;
        if (m.h_state.get()->overflow) {  // too many distinct values below tau: lower it and re-offer
            const uint64_t nt = m.h_state.get()->tau >> 4;
            rc = m.reset(st, nt ? nt : 1, false);
            if (rc) return rc;
            m.passes++;
            rc = rehash();
            if (rc) return rc;
            continue;
        }
        const uint64_t tau = m.h_state.get()->tau;
        const uint64_t *live = m.d_set[m.h_state.get()->cur & 1u].get();
        // distinct values <= tau (older, larger ones may linger from before tau dropped)
        uint64_t thr = tau;
        uint32_t M = 0;
        for (int iter = 0; iter < 64; iter++) {
            CU(cudaMemsetAsync(m.field(offsetof(MixState, n_out)), 0, sizeof(uint32_t), st));
            CU(launch_mix_collect(live, m.cap, thr, m.d_cand.get(), m.cand_cap, m.field(offsetof(MixState, n_out)), st));
            n_launches++;
            rc = m.sync_state(st);
            if (rc) return rc;
            M = m.h_state.get()->n_out;
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
            CU(launch_sort_unique(m.d_cand.get(), M, m.d_scratch.get(), m.field(offsetof(MixState, n_unique)), st));
            n_launches++;
            const uint32_t take = std::min(M, m.s);   // >= what is kept (n_unique <= M)
            CU(cudaMemcpyAsync(m.h_cand.get(), m.d_cand.get(), (size_t)take * 8, cudaMemcpyDeviceToHost, st));
            rc = m.sync_state(st);
            if (rc) return rc;
            const uint32_t nu = std::min(m.h_state.get()->n_unique, take);
            out.assign(m.h_cand.get(), m.h_cand.get() + nu);
        }
        if (m.h_state.get()->has_max && out.size() < m.s) out.push_back(~0ull);  // hash == 2^64-1 present
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
        CU(cudaEventElapsedTime(&ms, s->ev_pool[i].first.get(), s->ev_pool[i].second.get()));
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
HS_API void hs_db_free(hs_db *db) { if (db) delete db; }

// =============================================================================
// screen
// =============================================================================
HS_API int hs_screen_new(hs_db *db, hs_screen **out)
{
    if (!db || !out) return fail(HS_EINVAL, "null argument");
    ON_DEVICE(db->device);
    std::unique_ptr<hs_screen> s(new hs_screen());   // a failed step below deletes the half-built handle
    s->db = db;
    const uint64_t N = std::max<uint64_t>(db->n_refs, 1), E = std::max<uint64_t>(db->n_entries, 1);
    const uint64_t E4 = (E + 3) / 4 * 4;
    CU(s->stream.create());
    CU(s->copy_stream.create());
    CU(s->d_counts.grow(E4));
    CU(cudaMemsetAsync(s->d_counts.get(), 0, E4 * 4, s->stream.get()));
    CU(s->d_stats.grow(2 * ST_COUNT));
    // the four result columns share one allocation (identity | p-value | shared | median) so that
    // they travel to the host in a single copy
    CU(s->d_result.grow(N * 3));
    s->d_identity = s->d_result.get();
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
    CU(s->d_sparse.grow(1));
    CU(cudaMemsetAsync(s->d_sparse.get(), 0, sizeof(SparseState), s->stream.get()));
    CU(s->h_sparse.grow(1));
    CU(s->d_touched.grow(s->touched_cap));
    CU(s->d_depths.grow(s->pair_cap));
    CU(s->d_ref_rows.grow(N * 4));
    s->d_hit = s->d_ref_rows.get();
    s->d_seg_start = s->d_hit + N; s->d_seg_fill = s->d_seg_start + N; s->d_plain = s->d_seg_fill + N;
    for (Event *e : {&s->red0, &s->red1, &s->red2, &s->red3, &s->rst0, &s->rst1}) CU(e->create());
    CU(s->h_result.grow(N * 24));
    CU(s->h_stats.grow(ST_COUNT + 4));
    CU(s->h_mixture.grow((size_t)db->s + 1));
    int rc = s->mix.init(db->s, db->use64);
    if (rc) return rc;
    s->touched_valid = false;   // nothing recorded yet and counts[] was just cleared: screen_zero need not walk a list
    rc = screen_zero(s.get());
    if (rc) return rc;
    *out = s.release();
    return HS_OK;
}

HS_API int hs_screen_set_stream(hs_screen *s, void *cuda_stream)
{
    if (!s) return fail(HS_EINVAL, "null handle");
    ON_DEVICE(s->db->device);
    CU(cudaStreamSynchronize(s->stream.get()));
    if (cuda_stream) s->stream.borrow((cudaStream_t)cuda_stream);
    else CU(s->stream.create());
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
            CU(cudaMemcpyAsync((char *)dseq + w0 * 8, seq + w0, (cw1 - w0) * 8, cudaMemcpyHostToDevice, s->copy_stream.get()));
            CU(cudaMemcpyAsync((char *)dinv + w0 * 4, inv + w0, (cw1 - w0) * 4, cudaMemcpyHostToDevice, s->copy_stream.get()));
        }
        if (w1 > cw1) {
            const uint64_t p0 = std::max(cw1, w0);
            CU(cudaMemsetAsync((char *)dseq + p0 * 8, 0, (w1 - p0) * 8, s->copy_stream.get()));
            CU(cudaMemsetAsync((char *)dinv + p0 * 4, 0xFF, (w1 - p0) * 4, s->copy_stream.get()));
        }
        if (s->copy_ev_used == s->copy_evs.size()) {
            Event e;
            CU(e.create(cudaEventDisableTiming));
            s->copy_evs.push_back(std::move(e));
        }
        cudaEvent_t ev = s->copy_evs[s->copy_ev_used++].get();
        CU(cudaEventRecord(ev, s->copy_stream.get()));
        CU(cudaStreamWaitEvent(s->stream.get(), ev, 0));
        int rc = launch_chunk(s, c, true, true, w0 / kTileWords, w1 / kTileWords);
        if (rc) return rc;
    }
    if (done_ev) CU(cudaEventRecord(done_ev, s->copy_stream.get()));  // the host buffer may be reused
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
        int rc = in.ensure(len, s->stream.get());
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
    CU(cudaMemcpyAsync(sl->raw.get(), text, len, cudaMemcpyHostToDevice, s->copy_stream.get()));
    CU(cudaEventRecord(sl->copied.get(), s->copy_stream.get()));
    if (host_free_ev) CU(cudaEventRecord(host_free_ev, s->copy_stream.get()));
    CU(cudaStreamWaitEvent(s->stream.get(), sl->copied.get(), 0));
    FaScratch sc = in.sc;
    sc.chunk_positions = d_npos;
    CU(launch_fasta_to_codes(sl->raw.get(), (uint32_t)len, sl->codes.get(), sc, s->stream.get()));
    CU(launch_pack_codes_dyn(sl->codes.get(), d_npos, (uint64_t *)dseq, (uint32_t *)dinv, alloc, s->stream.get()));
    CU(cudaEventRecord(sl->done.get(), s->stream.get()));
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
        CU(g.free_ev.create(cudaEventDisableTiming));
        s->staging.push_back(std::move(g));
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
                if (g.seq.get()) cudaEventSynchronize(g.free_ev.get());
                g.seq.reset(); g.inv.reset();   // both go before either grows
                g.cap_words = 0;
                const uint64_t cap = bound + bound / 8;
                if (g.seq.grow(cap) != cudaSuccess || g.inv.grow(cap) != cudaSuccess)
                    rc = fail(HS_ENOMEM, "pinned staging allocation failed");
                else
                    g.cap_words = cap;
            } else {
                cudaEventSynchronize(g.free_ev.get());  // previous H2D from this buffer has finished
            }
            PackStats ps;
            if (rc == HS_OK) {
                const double t0 = now_s();
                pack_text_span(text + spans[i].first, len, g.seq.get(), g.inv.get(), &ps);
                const double t1 = now_s();
                my_ms = 1e3 * (t1 - t0);
                pack_us_per_span.store((pack_us_per_span.load() * 3 + (int)(1e3 * my_ms)) / 4);
                std::lock_guard<std::mutex> lk(s->mu);
                const double t2 = now_s();
                s->st.n_bases += ps.n_seq_bases;
                s->st.n_records += ps.n_records;
                rc = feed_host_chunk(s, g.seq.get(), g.inv.get(), ps.n_positions, g.free_ev.get());
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
                    if (s->ingest.slots[q].done.get() && cudaEventQuery(s->ingest.slots[q].done.get()) == cudaErrorNotReady) busy++;
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
            CU(g.free_ev.create(cudaEventDisableTiming));
            s->staging.push_back(std::move(g));
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
        CU(cudaStreamSynchronize(s->copy_stream.get()));
        s->ring = FileRing();
        CU(s->ring.base.grow(cap * 2 * T));
        s->ring.slot_cap = cap;
        for (int i = 0; i < 2 * T; i++) {
            Event e;
            CU(e.create(cudaEventDisableTiming));
            s->ring.free_ev.push_back(std::move(e));
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
            char *buf = s->ring.base.get() + slot * s->ring.slot_cap;
            if (cudaEventSynchronize(s->ring.free_ev[slot].get()) != cudaSuccess) { bail(fail(HS_ECUDA, "ring event")); break; }
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
                rc = feed_span_device(s, buf + b, e - b, s->ring.free_ev[slot].get());
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
    unsigned long long *h = s->h_stats.get(), *t = s->h_stats.get() + ST_COUNT;
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
        CU(cudaEventElapsedTime(&ms, s->rst0.get(), s->rst1.get()));
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
    CU(cudaEventRecord(s->red0.get(), s->stream.get()));
    const bool parsed = s->ingest.ready && s->ingest.counters_used;
    CU(cudaMemcpyAsync(s->h_stats.get(), s->d_stats.get(), ST_COUNT * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s->stream.get()));
    if (parsed) {
        CU(cudaMemcpyAsync(s->h_stats.get() + ST_COUNT, s->ingest.d_totals.get(), 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s->stream.get()));
        CU(cudaMemsetAsync(s->ingest.d_totals.get(), 0, 4 * sizeof(unsigned long long), s->stream.get()));
    }
    MixEngine &m = s->mix;
    CU(launch_mix_select(m.view(~0ull), m.s, m.use64, m.d_hist.get(), m.d_cand.get(), m.sel_pad, m.d_scratch.get(), s->stream.get()));
    s->st.n_launches += 4;
    CU(cudaMemcpyAsync(m.h_cand.get(), m.d_cand.get(), (size_t)m.s * 8, cudaMemcpyDeviceToHost, s->stream.get()));
    CU(cudaMemcpyAsync(m.h_state.get(), m.d_state.get(), sizeof(MixState), cudaMemcpyDeviceToHost, s->stream.get()));
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
        CU(cudaStreamSynchronize(s->stream.get()));
        if (s->flush_parsed) {   // the parser totals were folded into h_stats and cleared on the device: keep them
            unsigned long long *t = s->h_stats.get() + ST_COUNT;
            s->st.n_positions += t[0]; s->st.n_bases += t[1]; s->st.n_records += t[2];
        }
        s->flush_pending = false;
    }
    CU(cudaEventRecord(s->red0.get(), s->stream.get()));
    // the counters are final once the streaming launches are (re-offer passes count elsewhere): fetch
    // them with the first synchronisation of the mixture finaliser instead of one of their own
    unsigned long long *h = s->h_stats.get(), *t = s->h_stats.get() + ST_COUNT;
    const bool parsed = s->ingest.ready && s->ingest.counters_used;
    CU(cudaMemcpyAsync(h, s->d_stats.get(), ST_COUNT * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s->stream.get()));
    if (parsed) {
        CU(cudaMemcpyAsync(t, s->ingest.d_totals.get(), 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s->stream.get()));
        CU(cudaMemsetAsync(s->ingest.d_totals.get(), 0, 4 * sizeof(unsigned long long), s->stream.get()));  // folded: do not fold twice
    }
    int rc = mix_finalize(s->mix, s->stream.get(), s->mixture, s->st.n_launches, [&]() -> int {
        for (const Chunk &c : s->chunks) {
            int r = launch_chunk(s, c, false, true);
            if (r) return r;
            if (!c.n_dev) s->st.n_positions -= c.n_bases;  // a mixture-only second pass is not new input
        }
        return HS_OK;
    });
    if (rc) return rc;
    CU(cudaEventRecord(s->red1.get(), s->stream.get()));
    CU(cudaEventSynchronize(s->red1.get()));   // mix_finalize ended on a synchronisation: nothing is left to wait for
    rc = flush_epilogue(s, parsed);
    if (rc) return rc;
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, s->red0.get(), s->red1.get()));
    s->st.ms_reduce = ms;
    s->flushed = true;
    return HS_OK;
}

HS_API int hs_screen_counts_devptr(hs_screen *s, void **d_counts, uint64_t *n)
{
    if (!s || !d_counts || !n) return fail(HS_EINVAL, "null argument");
    *d_counts = s->d_counts.get();
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
    CU(cudaMemsetAsync(d_n_out, 0, sizeof(uint32_t), s->stream.get()));
    SparseView sp = sparse_view(s);
    if (!s->touched_valid) sp.touched = nullptr;
    CU(launch_counts_compact(sp, s->d_counts.get(), s->db->n_entries, (unsigned long long *)d_pairs, cap, (uint32_t *)d_n_out, s->stream.get()));
    s->st.n_launches += sp.touched ? 2 : 1;
    return HS_OK;
}

HS_API int hs_screen_counts_absorb(hs_screen *s, const void *d_rows, uint32_t n_rows, uint32_t cap, uint32_t skip_row)
{
    if (!s || (!d_rows && n_rows)) return fail(HS_EINVAL, "null argument");
    ON_DEVICE(s->db->device);
    SparseView sp = sparse_view(s);
    if (!s->touched_valid) sp.touched = nullptr;
    CU(launch_counts_absorb(sp, s->d_counts.get(), s->db->n_entries, (const unsigned long long *)d_rows, n_rows, cap, skip_row,
                            s->db->sm, s->stream.get()));
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
    const uint32_t nm = std::min<uint32_t>(s->h_sparse.get()->n_mix, s->db->s);
    s->mixture.assign(s->h_mixture.get(), s->h_mixture.get() + nm);
    s->st.n_mixture = nm;
    s->st.set_size = s->h_sparse.get()->set_size[0];
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
    // temporaries on several devices: each is released on its own when the call returns
    std::vector<DevBuf<unsigned long long>> rec(n_src);
    DevBuf<unsigned long long> rows_buf;
    std::vector<uint32_t> n(n_src);
    uint32_t cap = 1;
    for (uint32_t i = 0; i < n_src; i++) {
        hs_screen *s = src[i];
        ON_DEVICE(s->db->device);
        CU(cudaMemcpyAsync(s->h_sparse.get(), s->d_sparse.get(), sizeof(SparseState), cudaMemcpyDeviceToHost, s->stream.get()));
        CU(cudaStreamSynchronize(s->stream.get()));
        const bool listed = s->sparse_enabled && s->touched_valid && s->h_sparse.get()->n_touched <= s->touched_cap;
        const uint64_t rcap = listed ? s->h_sparse.get()->n_touched : db->n_entries;
        CU(rec[i].grow(rcap + 1));
        CU(cudaMemsetAsync(rec[i].get(), 0, 8, s->stream.get()));
        int r = hs_screen_counts_compact_async(s, rec[i].get() + 1, (uint32_t)rcap, rec[i].get());
        if (r) return r;
        CU(cudaMemcpyAsync(&n[i], rec[i].get(), sizeof(uint32_t), cudaMemcpyDeviceToHost, s->stream.get()));
        CU(cudaStreamSynchronize(s->stream.get()));
        cap = std::max(cap, n[i]);
    }
    ON_DEVICE(db->device);
    const size_t R = (size_t)n_src + 1, stride = (size_t)cap + 1, mstride = (size_t)db->s + 1;
    CU(rows_buf.grow(R * (stride + mstride)));
    unsigned long long *rows = rows_buf.get(), *mix = rows + R * stride;
    CU(cudaMemsetAsync(rows, 0, 8, dst->stream.get()));
    for (uint32_t i = 0; i < n_src; i++)
        CU(cudaMemcpyPeerAsync(rows + (i + 1) * stride, db->device, rec[i].get(), src[i]->db->device, ((size_t)n[i] + 1) * 8,
                               dst->stream.get()));
    std::vector<uint64_t> h_mix(R * mstride);
    mixture_row(dst, h_mix.data());
    for (uint32_t i = 0; i < n_src; i++) mixture_row(src[i], h_mix.data() + (i + 1) * mstride);
    CU(cudaMemcpyAsync(mix, h_mix.data(), h_mix.size() * 8, cudaMemcpyHostToDevice, dst->stream.get()));
    int r = hs_screen_counts_absorb(dst, rows, (uint32_t)R, cap, 0);
    if (!r) r = hs_screen_mixture_merge_device(dst, mix, (uint32_t)R);
    if (r) return r;
    // the merged mixture and its set size now, as for a single screen after flush (stats read before finish)
    CU(cudaMemcpyAsync(dst->h_sparse.get(), dst->d_sparse.get(), sizeof(SparseState), cudaMemcpyDeviceToHost, dst->stream.get()));
    if (db->s) CU(cudaMemcpyAsync(dst->h_mixture.get(), dst->d_mixture.get(), (size_t)db->s * 8, cudaMemcpyDeviceToHost, dst->stream.get()));
    CU(cudaStreamSynchronize(dst->stream.get()));
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
        CU(launch_mix_record(s->mix.view(~0ull), s->db->s, s->mix.sel_pad, s->mix.d_cand.get(), (unsigned long long *)d_record,
                             s->force_unsettled, s->stream.get()));
        s->force_unsettled = 0;
        s->st.n_launches++;
        return HS_OK;
    }
    if (!s->flushed) return fail(HS_ESTATE, "call hs_screen_flush first");
    // what every rank contributes to the mixture all-gather: it goes up from pinned memory on the
    // screen's stream and the record stays on the device for the collective
    mixture_row(s, s->h_mixture.get());
    CU(cudaMemcpyAsync(d_record, s->h_mixture.get(), ((size_t)s->db->s + 1) * 8, cudaMemcpyHostToDevice, s->stream.get()));
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
    if (s->d_merge_work.cap() < need || s->d_merge_scratch.cap() < need) {
        s->d_merge_work.reset(); s->d_merge_scratch.reset();   // both go before either grows
        CU(s->d_merge_work.grow(need));
        CU(s->d_merge_scratch.grow(need));
    }
    CU(s->d_mixture.grow(std::max<uint32_t>(sc, 1)));
    CU(launch_mixture_merge((const unsigned long long *)d_rows, n_rows, sc, sc, s->db->d_seg_s.get(), (uint32_t)s->db->seg_s.size(),
                            s->db->use64, s->d_merge_work.get(), need, s->d_merge_scratch.get(), s->d_mixture.get(),
                            s->d_sparse.get(), s->stream.get()));
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
        CU(cudaMemsetAsync(s->d_shared, 0, N * 8, s->stream.get()));   // shared | median are adjacent
        static_assert(offsetof(SparseState, overflow) == offsetof(SparseState, n_hit) + 8, "n_hit, n_pairs, overflow are cleared together");
        CU(cudaMemsetAsync(&s->d_sparse.get()->n_hit, 0, 3 * sizeof(uint32_t), s->stream.get()));
        SparseReduceArgs a;
        memset(&a, 0, sizeof a);
        a.sp = sparse_view(s);
        a.counts = s->d_counts.get(); a.next = db->d_next.get(); a.offsets = db->d_offsets.get(); a.n_refs = (uint32_t)N;
        a.lengths = db->d_lengths.get(); a.seg_begin = db->d_seg_begin.get(); a.n_seg = (uint32_t)n_seg;
        a.shared = s->d_shared; a.median = s->d_median; a.plain = s->d_plain; a.hit = s->d_hit;
        a.seg_start = s->d_seg_start; a.seg_fill = s->d_seg_fill; a.depths = s->d_depths.get(); a.pair_cap = s->pair_cap;
        a.ref_scale = (E && N <= E) ? (uint64_t)((((unsigned __int128)N) << 64) / ((unsigned __int128)E + 1)) : 0;
        CU(launch_sparse_reduce(a, wta, db->sm, s->stream.get()));
        s->st.n_launches += wta ? 7 : 4;
        return HS_OK;
    }
    CU(launch_sketch_reduce(db->d_offsets.get(), N, db->d_canon.get(), s->d_counts.get(), nullptr, s->d_shared, s->d_median, db->sm, s->stream.get()));
    s->st.n_launches++;
    if (wta && E) {
        CU(s->d_win.grow(E * 20));
        auto *best_score = reinterpret_cast<unsigned long long *>(s->d_win.get()), *best_len = best_score + E;
        auto *winner = reinterpret_cast<uint32_t *>(best_len + E);
        for (size_t j = 0; j < n_seg; j++) {   // -w is a competition among the references of one .msh (S12)
            const uint64_t b = db->seg_begin[j], n = db->seg_begin[j + 1] - b;
            if (!n) continue;
            CU(launch_winner(db->d_offsets.get() + b, n, db->d_canon.get(), s->d_counts.get(), s->d_shared + b, db->d_lengths.get() + b,
                             best_score, best_len, winner, E, db->sm, s->stream.get()));
            CU(launch_sketch_reduce(db->d_offsets.get() + b, n, db->d_canon.get(), s->d_counts.get(), winner, s->d_shared + b,
                                    s->d_median + b, db->sm, s->stream.get()));
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
                        s->mixture_on_device ? &s->d_sparse.get()->set_size[j] : nullptr, n, s->d_shared + b, nullptr,
                        db->d_offsets.get() + b, nullptr, s->d_identity + b, s->d_pvalue + b, s->stream.get()));
        s->st.n_launches++;
    }
    const uint64_t NA = std::max<uint64_t>(N, 1);   // layout of the allocation (hs_screen_new)
    if (N) CU(cudaMemcpyAsync(s->h_result.get(), s->d_identity, NA * 24, cudaMemcpyDeviceToHost, s->stream.get()));
    CU(cudaMemcpyAsync(s->h_sparse.get(), s->d_sparse.get(), sizeof(SparseState), cudaMemcpyDeviceToHost, s->stream.get()));
    if (s->mixture_on_device && db->s)
        CU(cudaMemcpyAsync(s->h_mixture.get(), s->d_mixture.get(), (size_t)db->s * 8, cudaMemcpyDeviceToHost, s->stream.get()));
    return HS_OK;
}

}  // namespace

namespace {

// rows a14-a16 for the references with hits only, written by the GPU into host-mapped rows
int enqueue_hits(hs_screen *s, bool dense)
{
    hs_db *db = s->db;
    const uint64_t N = db->n_refs;
    if (N && !s->rows_host.ref) {   // (laid out once the pinned rows and their device address both exist)
        const size_t n3 = (N * 12 + 7) & ~(size_t)7;
        CU(s->h_rows.grow(n3 + N * 16, cudaHostAllocMapped));
        char *d = nullptr;
        CU(cudaHostGetDevicePointer((void **)&d, s->h_rows.get(), 0));
        auto lay = [&](char *base) {
            HitRows r;
            r.ref = reinterpret_cast<uint32_t *>(base); r.shared = r.ref + N; r.median = r.shared + N;
            r.identity = reinterpret_cast<double *>(base + n3); r.pvalue = r.identity + N;
            r.cap = (uint32_t)N;
            return r;
        };
        s->rows_host = lay(s->h_rows.get());
        s->rows_dev = lay(d);
    }
    if (N) {
        StatsHitArgs a;
        memset(&a, 0, sizeof a);
        a.k = db->k; a.n_seg = (uint32_t)db->seg_s.size();
        for (size_t j = 0; j < db->seg_s.size(); j++) a.set_size[j] = set_size_of(s->mixture, db->use64, db->seg_s[j]);
        a.set_size_dev = s->mixture_on_device ? s->d_sparse.get()->set_size : nullptr;
        a.seg_begin = db->d_seg_begin.get(); a.hit = s->d_hit; a.n_hit = &s->d_sparse.get()->n_hit;
        a.shared = s->d_shared; a.median = s->d_median; a.offsets = db->d_offsets.get(); a.rows = s->rows_dev;
        CU(launch_stats_hits(a, dense, (uint32_t)N, s->d_hit, &s->d_sparse.get()->n_hit, db->sm, s->stream.get()));
        s->st.n_launches += dense ? 2 : 1;
    }
    CU(cudaMemcpyAsync(s->h_sparse.get(), s->d_sparse.get(), sizeof(SparseState), cudaMemcpyDeviceToHost, s->stream.get()));
    if (s->mixture_on_device && db->s)
        CU(cudaMemcpyAsync(s->h_mixture.get(), s->d_mixture.get(), (size_t)db->s * 8, cudaMemcpyDeviceToHost, s->stream.get()));
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
        CU(cudaEventRecord(s->red2.get(), s->stream.get()));
        if ((rc = enqueue_reduce(s, wta, dense)) != HS_OK) return rc;
        CU(cudaEventRecord(s->red3.get(), s->stream.get()));
    }
    if (!pending) {
        rc = hs_screen_flush(s);
        if (rc) return rc;
        CU(cudaEventRecord(s->red0.get(), s->stream.get()));
    }   // (pending: red0 was recorded by hs_screen_flush_async -- the exchange in between is part of the figure)
    if (early) {
        float ems = 0;
        CU(cudaEventElapsedTime(&ems, s->red2.get(), s->red3.get()));   // flush synchronised the stream
        s->st.ms_reduce += ems;
    }
    if (!early && (rc = enqueue_reduce(s, wta, dense)) != HS_OK) return rc;
    if ((rc = hits ? enqueue_hits(s, dense) : enqueue_stats_and_copy(s)) != HS_OK) return rc;
    CU(cudaEventRecord(s->red1.get(), s->stream.get()));
    CU(cudaStreamSynchronize(s->stream.get()));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, s->red0.get(), s->red1.get()));
    s->st.ms_reduce = pending ? ms : s->st.ms_reduce + ms;
    s->st.mix_unsettled = 0;
    if (pending) {
        // the one synchronisation of this screen has happened: complete the flush from what came back with it
        const MixState &hs_ = *s->mix.h_state.get();
        const bool held = !s->force_unsettled && !hs_.overflow && !hs_.sel_too_many && hs_.n_out <= s->mix.sel_pad &&
                          (hs_.n_unique >= s->mix.s || hs_.tau == ~0ull);
        s->force_unsettled = 0;   // (tests; the multi-GPU path has already spent it in its mixture record)
        const bool all_held = s->mixture_on_device ? !s->h_sparse.get()->mix_unsettled : held;
        if (!all_held) {
            if (s->mixture_on_device) {
                // some rank's selection fell through: every rank knows (the gathered records say so) and the
                // CALLER redoes flush + mixture exchange synchronously; the counts were absorbed and stay
                s->st.mix_unsettled = 1;
                s->st.exchange_overflow = s->h_sparse.get()->xchg_overflow;
                s->st.exchange_max_pairs = s->h_sparse.get()->xchg_max;
                return HS_OK;
            }
            rc = hs_screen_flush(s);              // single process: the iterative finaliser, then everything again
            if (rc) return rc;
            return finish_core(s, wta, hits);
        }
        s->mixture.assign(s->mix.h_cand.get(), s->mix.h_cand.get() + std::min(hs_.n_unique, s->mix.s));
        if (hs_.has_max && s->mixture.size() < s->mix.s) s->mixture.push_back(~0ull);
        s->flush_pending = false;
        rc = flush_epilogue(s, s->flush_parsed);
        if (rc) return rc;
        s->flushed = true;
    }
    if (s->mixture_on_device) adopt_merged_mixture(s);   // the merged mixture and its set size arrive with the results
    s->st.exchange_overflow = s->h_sparse.get()->xchg_overflow;
    s->st.exchange_max_pairs = s->h_sparse.get()->xchg_max;
    if (!dense && (s->h_sparse.get()->n_touched > s->touched_cap || s->h_sparse.get()->wrapped || s->h_sparse.get()->overflow)) {
        // the O(present) bookkeeping did not hold this query (more present hashes than its buffers, or a
        // count that wrapped): the dense kernels give the answer, and the next reset clears every count
        dense = true;
        const uint32_t n_touched = s->h_sparse.get()->n_touched;
        CU(cudaEventRecord(s->red0.get(), s->stream.get()));
        if ((rc = enqueue_reduce(s, wta, true)) != HS_OK) return rc;
        if ((rc = hits ? enqueue_hits(s, true) : enqueue_stats_and_copy(s)) != HS_OK) return rc;
        CU(cudaEventRecord(s->red1.get(), s->stream.get()));
        CU(cudaStreamSynchronize(s->stream.get()));
        CU(cudaEventElapsedTime(&ms, s->red0.get(), s->red1.get()));
        s->st.ms_reduce += ms;
        s->h_sparse.get()->n_touched = n_touched;
    }
    s->st.reduce_path = dense ? 1u : 0u;
    s->st.n_touched = s->h_sparse.get()->n_touched;
    s->st.n_hit_refs = (dense && !hits) ? 0u : s->h_sparse.get()->n_hit;
    s->st.n_pairs = dense ? 0u : s->h_sparse.get()->n_pairs;
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
    double *h_id = reinterpret_cast<double *>(s->h_result.get()), *h_pv = h_id + NA;
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
    const uint32_t n = (uint32_t)std::min<uint64_t>(s->h_sparse.get()->n_hit, s->db->n_refs);
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
    CU(cudaStreamSynchronize(s->stream.get()));
    return screen_zero(s);
}

HS_API int hs_screen_stats(hs_screen *s, hs_stats_t *stats)
{
    if (!s || !stats) return fail(HS_EINVAL, "null argument");
    *stats = s->st;
    return HS_OK;
}

HS_API void hs_screen_free(hs_screen *s) { if (s) delete s; }

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
    DevBuf<uint64_t> dseq, dh;
    DevBuf<uint32_t> dinv;
    DevBuf<uint8_t> dv;
    DevBuf<unsigned long long> dst;
    CU(dseq.grow(alloc));
    CU(dinv.grow(alloc));
    CU(dh.grow(n_bases));
    CU(dv.grow(n_bases));
    CU(dst.grow(ST_COUNT));
    CU(cudaMemset(dseq.get(), 0, alloc * 8));
    CU(cudaMemset(dinv.get(), 0xFF, alloc * 4));
    CU(cudaMemset(dh.get(), 0, n_bases * 8));
    CU(cudaMemset(dv.get(), 0, n_bases));
    CU(cudaMemset(dst.get(), 0, ST_COUNT * sizeof(unsigned long long)));
    CU(cudaMemcpy(dseq.get(), seq2, words * 8, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dinv.get(), inv, words * 4, cudaMemcpyHostToDevice));
    Chunk c{dseq.get(), dinv.get(), n_bases};
    StreamArgs a = base_args(c, k, seed, pow(4.0, (double)k) > pow(2.0, 32.0));
    a.emit_hash = dh.get(); a.emit_valid = dv.get(); a.stats = dst.get();
    CU(launch_stream(a, g_sm, 0));
    CU(cudaMemcpy(out_hash, dh.get(), n_bases * 8, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(out_valid, dv.get(), n_bases, cudaMemcpyDeviceToHost));
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
    DevBuf<uint8_t> raw, codes;
    DevBuf<uint64_t> dseq;
    DevBuf<uint32_t> dinv;
    DevBuf<unsigned long long> d_npos;
    unsigned long long tot[4] = {0, 0, 0, 0};
    CU(raw.grow(n + 64)); CU(codes.grow(n + 64));
    CU(dseq.grow(alloc)); CU(dinv.grow(alloc));
    CU(d_npos.grow(1));
    CU(cudaMemcpy(raw.get(), text, n, cudaMemcpyHostToDevice));
    FaScratch sc = in.sc;
    sc.chunk_positions = d_npos.get();
    CU(launch_fasta_to_codes(raw.get(), (uint32_t)n, codes.get(), sc, 0));
    CU(launch_pack_codes_dyn(codes.get(), d_npos.get(), dseq.get(), dinv.get(), alloc, 0));
    CU(cudaMemcpy(tot, in.d_totals.get(), sizeof tot, cudaMemcpyDeviceToHost));
    const uint64_t words = (tot[0] + 31) / 32;
    if (words > cap_words) rc = fail(HS_EINVAL, "output capacity too small");
    if (rc == HS_OK && words) {
        CU(cudaMemcpy(seq2, dseq.get(), words * 8, cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(inv, dinv.get(), words * 4, cudaMemcpyDeviceToHost));
    }
    *n_bases = tot[0];
    if (stats) { stats->n_positions = tot[0]; stats->n_bases = tot[1]; stats->n_records = tot[2]; }
    return rc;
}

HS_API int hs_db_probe(hs_db *db, const uint64_t *hashes, uint64_t n, uint32_t *out_entry)
{
    if (!db || (!hashes && n) || (!out_entry && n)) return fail(HS_EINVAL, "null argument");
    ON_DEVICE(db->device);
    if (!n) return HS_OK;
    DevBuf<uint64_t> dh;
    DevBuf<uint32_t> de;
    DevBuf<unsigned long long> dst;
    CU(dh.grow(n));
    CU(de.grow(n));
    CU(dst.grow(2));
    CU(cudaMemset(dst.get(), 0, 2 * sizeof(unsigned long long)));
    CU(cudaMemcpy(dh.get(), hashes, n * 8, cudaMemcpyHostToDevice));
    CU(launch_probe(db->view(), dh.get(), n, de.get(), dst.get(), db->sm, 0));
    CU(cudaMemcpy(out_entry, de.get(), n * 4, cudaMemcpyDeviceToHost));
    return HS_OK;
}

HS_API int hs_db_probe_device(hs_db *db, const void *d_hashes, uint64_t n, uint64_t *n_hits, uint64_t *n_bucket_reads,
                              float *ms)
{
    if (!db || (!d_hashes && n)) return fail(HS_EINVAL, "null argument");
    ON_DEVICE(db->device);
    unsigned long long h[2] = {0, 0};
    DevBuf<unsigned long long> dst;
    Event e0, e1;
    CU(dst.grow(2));
    CU(cudaMemset(dst.get(), 0, 2 * sizeof(unsigned long long)));
    CU(e0.create()); CU(e1.create());
    CU(cudaEventRecord(e0.get(), 0));
    CU(launch_probe(db->view(), (const uint64_t *)d_hashes, n, nullptr, dst.get(), db->sm, 0));
    CU(cudaEventRecord(e1.get(), 0));
    CU(cudaEventSynchronize(e1.get()));
    float t = 0;
    CU(cudaEventElapsedTime(&t, e0.get(), e1.get()));
    CU(cudaMemcpy(h, dst.get(), sizeof h, cudaMemcpyDeviceToHost));
    if (n_hits) *n_hits = h[0];
    if (n_bucket_reads) *n_bucket_reads = h[1];
    if (ms) *ms = t;
    return HS_OK;
}

HS_API int hs_gather_bench(const void *d_buf, uint64_t bytes, uint64_t n_reads, float *ms)
{
    if (!d_buf || bytes < 64 || !ms) return fail(HS_EINVAL, "bad argument");
    NEED_DEVICE();
    Event e0, e1;
    CU(e0.create()); CU(e1.create());
    CU(launch_gather_bench(d_buf, bytes, n_reads, g_sm, 0));  // warm-up
    CU(cudaEventRecord(e0.get(), 0));
    CU(launch_gather_bench(d_buf, bytes, n_reads, g_sm, 0));
    CU(cudaEventRecord(e1.get(), 0));
    CU(cudaEventSynchronize(e1.get()));
    CU(cudaEventElapsedTime(ms, e0.get(), e1.get()));
    return HS_OK;
}

HS_API int hs_db_entry_ids(hs_db *db, uint32_t *out)
{
    if (!db || !out) return fail(HS_EINVAL, "null argument");
    ON_DEVICE(db->device);
    if (db->n_entries) CU(cudaMemcpy(out, db->d_canon.get(), db->n_entries * 4, cudaMemcpyDeviceToHost));
    return HS_OK;
}

HS_API int hs_stat_batch(uint32_t k, uint64_t set_size, uint64_t n, const uint64_t *shared, const uint64_t *size,
                         double *identity, double *pvalue)
{
    if ((!shared || !size || !identity || !pvalue) && n) return fail(HS_EINVAL, "null argument");
    NEED_DEVICE();
    if (!n) return HS_OK;
    DevBuf<uint64_t> dx, dn;
    DevBuf<double> di, dp;
    CU(dx.grow(n)); CU(dn.grow(n));
    CU(di.grow(n)); CU(dp.grow(n));
    CU(cudaMemcpy(dx.get(), shared, n * 8, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dn.get(), size, n * 8, cudaMemcpyHostToDevice));
    CU(launch_stats(k, set_size, nullptr, n, nullptr, dx.get(), nullptr, dn.get(), di.get(), dp.get(), 0));
    CU(cudaMemcpy(identity, di.get(), n * 8, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(pvalue, dp.get(), n * 8, cudaMemcpyDeviceToHost));
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

// room for n elements in a buffer that grows on demand: half as much again when it has to (at least 64)
template <class B>
cudaError_t need(B &b, size_t n)
{
    return n <= b.cap() ? cudaSuccess : b.grow(std::max<size_t>(n + n / 2, 64));
}

// every CUDA resource of a sketcher; the stream (declared first) is released last
struct SketchDev {
    Stream stream;
    Event ev[4];
    DevBuf<unsigned long long> stats;
    DevBuf<uint64_t> seq, sets, out, out_off;
    DevBuf<uint32_t> inv, tile_genome, n_out;
    DevBuf<SketchSlot> slots;
    PinnedBuf<uint64_t> h_seq, h_out, h_out_off;
    PinnedBuf<uint32_t> h_inv, h_tile_genome, h_n_out;
    PinnedBuf<SketchSlot> h_slots;
    int init()
    {
        CU(stream.create());
        for (auto &e : ev) CU(e.create());
        CU(stats.grow(ST_COUNT));
        CU(cudaMemsetAsync(stats.get(), 0, ST_COUNT * sizeof(unsigned long long), stream.get()));
        return HS_OK;
    }
    ~SketchDev()
    {   // nothing is released while the stream may still use it
        if (stream.get()) cudaStreamSynchronize(stream.get());
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
    uint64_t *sq = d.h_seq.get() + (size_t)t0 * kTileWords;
    uint32_t *iv = d.h_inv.get() + (size_t)t0 * kTileWords;
    memcpy(sq, g.seq.data() + w0, (w1 - w0) * 8);
    memcpy(iv, g.inv.data() + w0, (w1 - w0) * 4);
    const size_t pad = (size_t)tiles * kTileWords - (w1 - w0);
    memset(sq + (w1 - w0), 0, pad * 8);
    memset(iv + (w1 - w0), 0xFF, pad * 4);
    for (uint32_t t = 0; t < tiles; t++) d.h_tile_genome.get()[t0 + t] = slot;
    return tiles;
}

// hash the staged tiles [0, tiles) into the batch's sets
int sketch_launch(hs_sketcher *sk, uint32_t tiles)
{
    SketchDev &d = sk->dev;
    const size_t words = (size_t)tiles * kTileWords;
    CU(need(d.seq, words)); CU(need(d.inv, words)); CU(need(d.tile_genome, tiles));
    CU(cudaMemcpyAsync(d.seq.get(), d.h_seq.get(), words * 8, cudaMemcpyHostToDevice, d.stream.get()));
    CU(cudaMemcpyAsync(d.inv.get(), d.h_inv.get(), words * 4, cudaMemcpyHostToDevice, d.stream.get()));
    CU(cudaMemcpyAsync(d.tile_genome.get(), d.h_tile_genome.get(), (size_t)tiles * 4, cudaMemcpyHostToDevice, d.stream.get()));
    StreamArgs a;
    memset(&a, 0, sizeof a);
    a.seq = d.seq.get(); a.inv = d.inv.get(); a.n_bases = tiles * kTilePositions; a.n_tiles = tiles;
    a.k = (int)sk->k; a.seed = sk->seed; a.use64 = sk->use64; a.stats = d.stats.get();
    a.sk = SketchView{d.tile_genome.get(), d.slots.get(), d.sets.get()};
    CU(cudaEventRecord(d.ev[0].get(), d.stream.get()));
    CU(launch_stream(a, g_sm, d.stream.get()));
    CU(cudaEventRecord(d.ev[1].get(), d.stream.get()));
    // the staging is refilled next: wait for the copies (and take the kernel time with them)
    CU(cudaEventSynchronize(d.ev[1].get()));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, d.ev[0].get(), d.ev[1].get()));
    sk->st.ms_stream += ms;
    sk->st.n_launches++;
    return HS_OK;
}

// one batch: genomes ids (all of them fit kSketchBatchTiles, or a single genome streamed piece by piece)
int sketch_batch(hs_sketcher *sk, const std::vector<uint32_t> &ids)
{
    SketchDev &d = sk->dev;
    const uint32_t n = (uint32_t)ids.size();
    CU(need(d.h_slots, n)); CU(need(d.slots, n)); CU(need(d.h_out_off, n)); CU(need(d.out_off, n));
    CU(need(d.h_n_out, n)); CU(need(d.n_out, n));
    uint64_t set_words = 0, out_words = 0, tiles = 0;
    uint32_t max_cap = 0;
    for (uint32_t j = 0; j < n; j++) {
        const SkGenome &g = sk->gen[ids[j]];
        SketchSlot &sl = d.h_slots.get()[j];
        memset(&sl, 0, sizeof sl);
        sl.st.tau = g.tau;
        sl.set_off = set_words;
        sl.mask = g.cap - 1; sl.limit = g.cap / 2;
        d.h_out_off.get()[j] = out_words;
        set_words += g.cap;
        out_words += std::min<uint64_t>(sk->s, g.cap);
        max_cap = std::max(max_cap, g.cap);
        tiles += g.tiles();
    }
    CU(need(d.sets, set_words)); CU(need(d.out, out_words)); CU(need(d.h_out, out_words));
    const uint64_t stage_tiles = std::min<uint64_t>(tiles, kSketchBatchTiles);
    CU(need(d.h_seq, stage_tiles * kTileWords)); CU(need(d.h_inv, stage_tiles * kTileWords)); CU(need(d.h_tile_genome, stage_tiles));
    CU(cudaMemcpyAsync(d.slots.get(), d.h_slots.get(), n * sizeof(SketchSlot), cudaMemcpyHostToDevice, d.stream.get()));
    CU(cudaMemcpyAsync(d.out_off.get(), d.h_out_off.get(), n * 8, cudaMemcpyHostToDevice, d.stream.get()));
    CU(cudaMemsetAsync(d.sets.get(), 0xFF, set_words * 8, d.stream.get()));
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
    CU(cudaEventRecord(d.ev[2].get(), d.stream.get()));
    CU(launch_sketch_select(d.slots.get(), n, max_cap, d.sets.get(), sk->s, d.out_off.get(), d.out.get(), d.n_out.get(), d.stream.get()));
    CU(cudaEventRecord(d.ev[3].get(), d.stream.get()));
    sk->st.n_launches++;
    CU(cudaMemcpyAsync(d.h_slots.get(), d.slots.get(), n * sizeof(SketchSlot), cudaMemcpyDeviceToHost, d.stream.get()));
    CU(cudaMemcpyAsync(d.h_n_out.get(), d.n_out.get(), n * 4, cudaMemcpyDeviceToHost, d.stream.get()));
    CU(cudaMemcpyAsync(d.h_out.get(), d.out.get(), out_words * 8, cudaMemcpyDeviceToHost, d.stream.get()));
    CU(cudaStreamSynchronize(d.stream.get()));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, d.ev[2].get(), d.ev[3].get()));
    sk->st.ms_select += ms;
    // settle or re-stream each genome (see the argument at the top of this section)
    const uint64_t top = sk->top();
    for (uint32_t j = 0; j < n; j++) {
        SkGenome &g = sk->gen[ids[j]];
        const MixState &r = d.h_slots.get()[j].st;
        const uint64_t have = (uint64_t)r.count + (r.has_max ? 1 : 0);
        if (!r.overflow && (have >= sk->s || g.tau == top)) {
            const uint64_t *h = d.h_out.get() + d.h_out_off.get()[j];
            g.hashes.assign(h, h + d.h_n_out.get()[j]);
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

HS_API void hs_sketcher_free(hs_sketcher *sk) { if (sk) delete sk; }

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
    // every array has at least one element: no kernel argument is a null pointer
    const uint64_t na1 = std::max<uint64_t>(n_a, 1), nt1 = std::max<uint64_t>(n_tax, 1);
    DevBuf<uint64_t> d_off;
    DevBuf<int32_t> d_tax, s_tax;
    DevBuf<double> d_w, s_w, s_nw, o_conf;
    DevBuf<uint32_t> d_names, s_name, o_names, o_depth;
    DevBuf<uint8_t> o_any;
    CU(d_off.grow(n_q + 1));
    CU(d_tax.grow(na1)); CU(d_w.grow(na1)); CU(d_names.grow(nt1 * kLcaRanks));
    CU(s_tax.grow(na1)); CU(s_w.grow(na1)); CU(s_name.grow(na1)); CU(s_nw.grow(na1));
    CU(o_names.grow(n_q * kLcaRanks)); CU(o_depth.grow(n_q)); CU(o_conf.grow(n_q)); CU(o_any.grow(n_q));
    LcaArgs a;
    memset(&a, 0, sizeof a);
    a.s_tax = s_tax.get(); a.s_w = s_w.get(); a.s_name = s_name.get(); a.s_nw = s_nw.get();
    a.out_names = o_names.get(); a.out_depth = o_depth.get(); a.out_conf = o_conf.get(); a.out_any = o_any.get();
    CU(cudaMemcpy(d_off.get(), q_off, (n_q + 1) * 8, cudaMemcpyHostToDevice));
    if (n_a) { CU(cudaMemcpy(d_tax.get(), tax, n_a * 4, cudaMemcpyHostToDevice)); CU(cudaMemcpy(d_w.get(), w, n_a * 8, cudaMemcpyHostToDevice)); }
    if (n_tax) CU(cudaMemcpy(d_names.get(), names, n_tax * kLcaRanks * 4, cudaMemcpyHostToDevice));
    CU(cudaMemset(a.out_names, 0, n_q * kLcaRanks * 4));
    a.n_q = n_q; a.q_off = d_off.get(); a.tax = d_tax.get(); a.w = d_w.get(); a.names = d_names.get();
    CU(launch_weighted_lca(a, g_sm, 0));
    CU(cudaMemcpy(out_names, a.out_names, n_q * kLcaRanks * 4, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(out_depth, a.out_depth, n_q * 4, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(out_conf, a.out_conf, n_q * 8, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(out_any, a.out_any, n_q, cudaMemcpyDeviceToHost));
    return HS_OK;
}

// =============================================================================
// `mash dist` (DESIGN.md §5 "mash dist"): one reference .msh against query sketches, exactly
// =============================================================================
namespace {

constexpr uint64_t kDistBlockBytes = 48ull << 20;   // bitmap rows + query hashes of one block: stays in L2 (126 MB)
constexpr uint32_t kDistMaxBlock = 1u << 16;        // queries per block at most
constexpr uint32_t kDistResultRows = 1u << 19;      // candidate rows one block holds (at least one query's worth)

struct DistQuery {
    std::string name, comment;
    uint64_t length = 0;
    uint32_t sp = 0;        // min(reference file's s, this query file's s)
};

struct DistSlot {
    DevBuf<DistRow> d_rows;
    PinnedBuf<DistRow> h_rows;
    PinnedBuf<unsigned long long> h_total;
    Event ev_t0, ev_t1, ev_t2, ev_done, ev_copied;   // t0 mark t1 count + scan + compact t2 merge done
    uint32_t q0 = 0, n_q = 0;
};

}  // namespace

struct hs_distance {
    int device = 0, sm = 0;
    std::unique_ptr<hs_db, void (*)(hs_db *)> db{nullptr, hs_db_free};
    DevBuf<uint64_t> d_ref_hashes;           // the references' sorted hashes, flat (hs_db keeps only its table)
    std::vector<uint64_t> ref_sizes;
    uint64_t ref_scale = 0;
    std::vector<DistQuery> q;
    std::vector<uint64_t> q_off{0}, q_hashes;
    bool uploaded = false;
    DevBuf<uint64_t> d_q_off, d_q_hashes, d_q_len;
    DevBuf<uint32_t> d_q_sp, d_bitmap;
    DevBuf<unsigned long long> d_row_start;
    DistSlot slot[2];
    Stream st, st_copy;
    std::vector<DistRow> rows;               // hs_distance_run_rows
    hs_distance_stats_t stats{};
};

namespace {

int dist_add(hs_distance *d, const char *name, const char *comment, uint64_t length, uint32_t s_q, const uint64_t *h, uint64_t n)
{
    for (uint64_t i = 1; i < n; i++)
        if (h[i] <= h[i - 1]) return fail(HS_EFORMAT, "sketch hashes are not strictly ascending");
    if (d->q.size() >= 0xFFFFFFF0ull) return fail(HS_EUNSUPPORTED, "more than 2^32 query sketches");
    DistQuery x;
    x.name = name ? name : "";
    x.comment = comment ? comment : "";
    x.length = length;
    x.sp = std::min(d->db->s, s_q);
    d->q.push_back(std::move(x));
    d->q_hashes.insert(d->q_hashes.end(), h, h + n);
    d->q_off.push_back(d->q_hashes.size());
    d->uploaded = false;
    return HS_OK;
}

int dist_upload(hs_distance *d)
{
    if (d->uploaded) return HS_OK;
    const uint64_t nq = d->q.size();
    std::vector<uint64_t> len(std::max<uint64_t>(nq, 1), 0);
    std::vector<uint32_t> sp(std::max<uint64_t>(nq, 1), 0);
    for (uint64_t i = 0; i < nq; i++) { len[i] = d->q[i].length; sp[i] = d->q[i].sp; }
    d->d_q_off.reset(); d->d_q_hashes.reset(); d->d_q_len.reset(); d->d_q_sp.reset();
    CU(d->d_q_off.grow(nq + 1));
    CU(d->d_q_hashes.grow(std::max<uint64_t>(d->q_hashes.size(), 1)));
    CU(d->d_q_len.grow(len.size()));
    CU(d->d_q_sp.grow(sp.size()));
    CU(cudaMemcpy(d->d_q_off.get(), d->q_off.data(), (nq + 1) * 8, cudaMemcpyHostToDevice));
    if (!d->q_hashes.empty())
        CU(cudaMemcpy(d->d_q_hashes.get(), d->q_hashes.data(), d->q_hashes.size() * 8, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d->d_q_len.get(), len.data(), len.size() * 8, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d->d_q_sp.get(), sp.data(), sp.size() * 4, cudaMemcpyHostToDevice));
    d->uploaded = true;
    return HS_OK;
}

// D2 from the exact integers, with the double expression of Mash's CommandDistance
double dist_value(uint64_t common, uint64_t denom, uint32_t k)
{
    if (common == denom) return 0.0;
    if (common == 0) return 1.0;
    const double jaccard = double(common) / denom;
    const double distance = -log(2 * jaccard / (1. + jaccard)) / k;
    return distance > 1 ? 1 : distance;
}

// The block pipeline.  Blocks of queries go through the kernels on `st`; while the device computes
// block b + 1, the candidate rows of block b are copied (on `st_copy`) into that slot's pinned buffer
// and handed to `sink` on the calling thread, in query order.  A block whose candidates overflow the
// result buffer is redone as blocks half its size, and so are the blocks after it (the one already in
// flight is dropped).
template <class Sink>
int dist_pipeline(hs_distance *d, double max_d, Sink &&sink)
{
    ON_DEVICE(d->device);
    int rc = dist_upload(d);
    if (rc) return rc;
    const hs_db *db = d->db.get();
    const uint64_t nq = d->q.size(), nr = db->n_refs;
    const uint32_t words = (uint32_t)((nr + 31) / 32);
    const double avg_q = nq ? (double)d->q_hashes.size() / (double)nq : 0.0;
    const double per_q = (double)words * 4 + avg_q * 8 + 8;
    uint64_t block = (uint64_t)((double)kDistBlockBytes / per_q);
    block = std::max<uint64_t>(1, std::min<uint64_t>({block, (uint64_t)kDistMaxBlock, std::max<uint64_t>(nq, 1)}));
    const uint32_t cap = (uint32_t)std::max<uint64_t>(kDistResultRows, nr);
    d->stats.block_queries = (uint32_t)block;
    d->stats.result_cap = cap;
    if (!nq) return HS_OK;

    if (!d->st.get()) { CU(d->st.create()); CU(d->st_copy.create()); }
    if (d->d_bitmap.cap() < block * words) {
        CU(d->d_bitmap.grow(std::max<uint64_t>(block * words, 1)));
        CU(cudaMemset(d->d_bitmap.get(), 0, d->d_bitmap.cap() * 4));   // k_dist_compact leaves it zero again
    }
    CU(d->d_row_start.grow(block + 1));
    for (DistSlot &s : d->slot) {
        CU(s.d_rows.grow(cap));
        CU(s.h_total.grow(1));
        if (!s.ev_done.get()) {
            CU(s.ev_t0.create()); CU(s.ev_t1.create()); CU(s.ev_t2.create()); CU(s.ev_done.create());
            CU(s.ev_copied.create(cudaEventDisableTiming));
            CU(cudaEventRecord(s.ev_copied.get(), d->st_copy.get()));
        }
    }
    const cudaStream_t st = d->st.get(), stc = d->st_copy.get();
    DistArgs a;
    memset(&a, 0, sizeof a);
    a.tab = db->view(); a.next = db->d_next.get();
    a.ref_off = db->d_offsets.get(); a.ref_hashes = d->d_ref_hashes.get(); a.ref_len = db->d_lengths.get();
    a.n_refs = (uint32_t)nr; a.ref_scale = d->ref_scale;
    a.q_off = d->d_q_off.get(); a.q_hashes = d->d_q_hashes.get(); a.q_len = d->d_q_len.get(); a.q_sp = d->d_q_sp.get();
    a.bitmap = d->d_bitmap.get(); a.words = words; a.row_start = d->d_row_start.get();
    a.cap = cap; a.k = db->k; a.max_d = max_d;

    uint64_t q_next = 0, blk = block;   // next block: [q_next, q_next + blk)
    int prev = -1, next_slot = 0;
    while (q_next < nq || prev >= 0) {
        int cur = -1;
        if (q_next < nq) {
            DistSlot &s = d->slot[next_slot];
            s.q0 = (uint32_t)q_next; s.n_q = (uint32_t)std::min<uint64_t>(blk, nq - q_next);
            q_next += s.n_q;
            a.q0 = s.q0; a.n_q = s.n_q; a.rows = s.d_rows.get();
            CU(cudaStreamWaitEvent(st, s.ev_copied.get(), 0));   // this slot's previous rows are home
            CU(cudaEventRecord(s.ev_t0.get(), st));
            CU(launch_dist_candidates(a, d->sm, s.ev_t1.get(), st));
            CU(cudaEventRecord(s.ev_t2.get(), st));
            CU(launch_dist_merge(a, d->sm, st));
            CU(cudaMemcpyAsync(s.h_total.get(), d->d_row_start.get() + s.n_q, sizeof(unsigned long long),
                               cudaMemcpyDeviceToHost, st));
            CU(cudaEventRecord(s.ev_done.get(), st));
            d->stats.n_blocks++;
            cur = next_slot;
            next_slot ^= 1;
        }
        if (prev >= 0) {
            DistSlot &s = d->slot[prev];
            CU(cudaEventSynchronize(s.ev_done.get()));
            float ms[3] = {0, 0, 0};
            CU(cudaEventElapsedTime(ms, s.ev_t0.get(), s.ev_t1.get()));
            CU(cudaEventElapsedTime(ms + 1, s.ev_t1.get(), s.ev_t2.get()));
            CU(cudaEventElapsedTime(ms + 2, s.ev_t2.get(), s.ev_done.get()));
            d->stats.ms_mark += ms[0]; d->stats.ms_compact += ms[1]; d->stats.ms_merge += ms[2];
            const unsigned long long n = *s.h_total.get();
            if (n > cap) {
                // redo from this block on (the one in flight behind it is dropped) with blocks half its size;
                // a block of one query always fits (cap >= references)
                CU(cudaStreamSynchronize(st));
                q_next = s.q0;
                blk = std::max<uint64_t>(1, s.n_q / 2);
                d->stats.n_splits++;
                prev = -1;
                next_slot = 0;
                continue;
            }
            uint64_t want = 1;
            while (want < n) want <<= 1;
            CU(s.h_rows.grow(want));
            CU(cudaStreamWaitEvent(stc, s.ev_done.get(), 0));
            if (n) CU(cudaMemcpyAsync(s.h_rows.get(), s.d_rows.get(), n * sizeof(DistRow), cudaMemcpyDeviceToHost, stc));
            CU(cudaEventRecord(s.ev_copied.get(), stc));
            CU(cudaEventSynchronize(s.ev_copied.get()));
            d->stats.n_candidates += n;
            if ((rc = sink(s.q0, s.n_q, s.h_rows.get(), (uint64_t)n))) return rc;
        }
        prev = cur;
    }
    return HS_OK;
}

void put_g(std::string &o, double x)
{
    char b[32];
    o.append(b, (size_t)snprintf(b, sizeof b, "%g", x));
}
void put_u(std::string &o, uint64_t x)
{
    char b[24];
    o.append(b, (size_t)snprintf(b, sizeof b, "%llu", (unsigned long long)x));
}

int write_all(int fd, const std::string &s)
{
    size_t off = 0;
    while (off < s.size()) {
        const ssize_t w = ::write(fd, s.data() + off, s.size() - off);
        if (w < 0) {
            if (errno == EINTR) continue;
            return fail(HS_EIO, std::string("writing the output: ") + strerror(errno));
        }
        off += (size_t)w;
    }
    return HS_OK;
}

struct DistFormat {
    const hs_distance *d;
    double max_d, max_p;
    bool table, comments;
    std::vector<std::string> ref_names;      // name or name:comment
    bool implicit_all;                        // non-candidate pairs pass D4 (-d >= 1 and -v >= 1)

    std::string qname(uint64_t q) const
    {
        const DistQuery &x = d->q[q];
        return comments ? x.name + ":" + x.comment : x.name;
    }
    // the lines of query q; its candidate rows are [r0, r1) in reference order.  Returns lines written.
    uint64_t query(uint64_t q, const DistRow *r0, const DistRow *r1, std::string &o) const
    {
        const hs_db *db = d->db.get();
        const uint32_t k = db->k;
        const uint64_t nr = db->n_refs, qsize = d->q_off[q + 1] - d->q_off[q];
        const uint32_t sp = d->q[q].sp;
        const std::string qn = qname(q);
        const bool empties = qsize == 0 && max_p >= 1;   // pairs of two empty sketches: distance 0, p-value 1
        auto line = [&](uint64_t r, uint64_t common, uint64_t denom, double dist, double p) {
            o += ref_names[r]; o += '\t'; o += qn; o += '\t';
            put_g(o, dist); o += '\t'; put_g(o, p); o += '\t';
            put_u(o, common); o += '/'; put_u(o, denom); o += '\n';
        };
        if (table) {
            o += qn;
            const DistRow *c = r0;
            for (uint64_t r = 0; r < nr; r++) {
                o += '\t';
                uint64_t common = 0, denom;
                double p = 1.0;
                if (c < r1 && c->r == r) { common = c->common; denom = c->denom; p = c->p; c++; }
                else denom = std::min<uint64_t>(sp, d->ref_sizes[r] + qsize);
                const double dist = dist_value(common, denom, k);
                if (dist > max_d || p > max_p) continue;
                put_g(o, dist);
            }
            o += '\n';
            return 1;
        }
        uint64_t n = 0;
        if (implicit_all || empties) {
            const DistRow *c = r0;
            for (uint64_t r = 0; r < nr; r++) {
                if (c < r1 && c->r == r) {
                    const double dist = dist_value(c->common, c->denom, k);
                    if (!(dist > max_d) && !(c->p > max_p)) { line(r, c->common, c->denom, dist, c->p); n++; }
                    c++;
                    continue;
                }
                const uint64_t denom = std::min<uint64_t>(sp, d->ref_sizes[r] + qsize);
                if (denom == 0 ? max_p >= 1 : implicit_all) { line(r, 0, denom, denom == 0 ? 0.0 : 1.0, 1.0); n++; }
            }
            return n;
        }
        for (const DistRow *c = r0; c < r1; c++) {
            const double dist = dist_value(c->common, c->denom, k);
            if (dist > max_d || c->p > max_p) continue;
            line(c->r, c->common, c->denom, dist, c->p);
            n++;
        }
        return n;
    }
};

}  // namespace

HS_API int hs_distance_new(const hs_msh *ref, hs_distance **out)
{
    if (!ref || !out) return fail(HS_EINVAL, "null argument");
    NEED_DEVICE();
    std::unique_ptr<hs_distance> d(new hs_distance());
    d->device = g_device; d->sm = g_sm;
    hs_db *db = nullptr;
    int rc = hs_db_from_msh(ref, &db);
    if (rc) return rc;
    d->db.reset(db);
    const uint64_t N = db->n_refs, E = db->n_entries;
    d->ref_sizes.resize(N);
    for (uint64_t i = 0; i < N; i++) d->ref_sizes[i] = db->offsets[i + 1] - db->offsets[i];
    d->ref_scale = (E && N <= E) ? (uint64_t)((((unsigned __int128)N) << 64) / ((unsigned __int128)E + 1)) : 0;
    CU(d->d_ref_hashes.grow(std::max<uint64_t>(E, 1)));
    if (E) CU(cudaMemcpy(d->d_ref_hashes.get(), ref->d.hashes.data(), E * 8, cudaMemcpyHostToDevice));
    d->stats.n_refs = N;
    *out = d.release();
    return HS_OK;
}

HS_API int hs_distance_add_msh(hs_distance *d, const hs_msh *m)
{
    if (!d || !m) return fail(HS_EINVAL, "null argument");
    const hs_db *db = d->db.get();
    if (m->d.k != db->k || m->d.seed != db->seed || m->d.use64 != db->use64)
        return fail(HS_EUNSUPPORTED, "query sketch file differs from the reference in k-mer size (" + std::to_string(m->d.k) +
                                         " vs " + std::to_string(db->k) + "), seed (" + std::to_string(m->d.seed) + " vs " +
                                         std::to_string(db->seed) + ") or hash width");
    const uint64_t n = m->d.offsets.size() - 1;
    for (uint64_t i = 0; i < n; i++) {
        const uint64_t b = m->d.offsets[i], e = m->d.offsets[i + 1];
        const int rc = dist_add(d, m->d.names[i].c_str(), m->d.comments[i].c_str(), m->d.lengths[i], m->d.s,
                                m->d.hashes.data() + b, e - b);
        if (rc) return rc;
    }
    return HS_OK;
}

HS_API int hs_distance_add_sketch(hs_distance *d, const char *name, const char *comment, uint64_t length, uint32_t s,
                                  const uint64_t *hashes, uint64_t n)
{
    if (!d || (!hashes && n)) return fail(HS_EINVAL, "null argument");
    if (s == 0) return fail(HS_EINVAL, "sketch size must be positive");
    return dist_add(d, name, comment, length, s, hashes, n);
}

HS_API int hs_distance_run(hs_distance *d, int fd, double max_distance, double max_pvalue, int table, int comments,
                           int host_threads)
{
    if (!d) return fail(HS_EINVAL, "null handle");
    if (!(max_distance >= 0 && max_distance <= 1) || !(max_pvalue >= 0 && max_pvalue <= 1))
        return fail(HS_EINVAL, "maximum distance and p-value must be in [0, 1]");
    const double t0 = now_s();
    const hs_db *db = d->db.get();
    DistFormat f;
    f.d = d; f.max_d = max_distance; f.max_p = max_pvalue; f.table = table != 0; f.comments = comments != 0;
    f.implicit_all = max_distance >= 1 && max_pvalue >= 1;
    f.ref_names.resize(db->n_refs);
    for (uint64_t r = 0; r < db->n_refs; r++)
        f.ref_names[r] = f.comments ? db->names[r] + ":" + db->comments[r] : db->names[r];
    const int threads = std::max(1, host_threads);
    double t_write = 0;
    int rc = HS_OK;
    if (table) {
        std::string h = "#query";
        for (const std::string &n : f.ref_names) { h += '\t'; h += n; }
        h += '\n';
        if ((rc = write_all(fd, h))) return rc;
    }
    std::vector<std::string> out(threads);
    std::vector<uint64_t> lines(threads);
    rc = dist_pipeline(d, max_distance, [&](uint32_t q0, uint32_t n_q, const DistRow *rows, uint64_t n) -> int {
        const double tw = now_s();
        // query q's rows start at the first row whose q is >= q
        auto first_of = [&](uint64_t q) { return std::lower_bound(rows, rows + n, q, [](const DistRow &x, uint64_t v) { return x.q < v; }); };
        const uint32_t nt = (uint32_t)std::min<uint64_t>((uint64_t)threads, n_q);
        auto part = [&](uint32_t t) {
            const uint64_t qa = q0 + (uint64_t)n_q * t / nt, qb = q0 + (uint64_t)n_q * (t + 1) / nt;
            std::string &o = out[t];
            o.clear();
            lines[t] = 0;
            const DistRow *c = first_of(qa);
            for (uint64_t q = qa; q < qb; q++) {
                const DistRow *e = first_of(q + 1);
                lines[t] += f.query(q, c, e, o);
                c = e;
            }
        };
        if (nt <= 1) part(0);
        else {
            std::vector<std::thread> th;
            for (uint32_t t = 1; t < nt; t++) th.emplace_back(part, t);
            part(0);
            for (auto &x : th) x.join();
        }
        for (uint32_t t = 0; t < nt; t++) {
            const int r = write_all(fd, out[t]);
            if (r) return r;
            d->stats.n_lines += lines[t];
        }
        t_write += now_s() - tw;
        return HS_OK;
    });
    d->stats.t_write_s += t_write;
    d->stats.t_total_s += now_s() - t0;
    return rc;
}

HS_API int hs_distance_run_rows(hs_distance *d, double max_distance, uint64_t *n_rows)
{
    if (!d || !n_rows) return fail(HS_EINVAL, "null argument");
    if (!(max_distance >= 0 && max_distance <= 1)) return fail(HS_EINVAL, "maximum distance must be in [0, 1]");
    const double t0 = now_s();
    d->rows.clear();
    const int rc = dist_pipeline(d, max_distance, [&](uint32_t, uint32_t, const DistRow *rows, uint64_t n) -> int {
        d->rows.insert(d->rows.end(), rows, rows + n);
        return HS_OK;
    });
    d->stats.t_total_s += now_s() - t0;
    *n_rows = d->rows.size();
    return rc;
}

HS_API int hs_distance_rows_copy(const hs_distance *d, uint64_t cap, uint32_t *q, uint32_t *r, uint32_t *common,
                                 uint32_t *denom, double *pvalue)
{
    if (!d) return fail(HS_EINVAL, "null handle");
    const uint64_t n = std::min<uint64_t>(cap, d->rows.size());
    for (uint64_t i = 0; i < n; i++) {
        const DistRow &x = d->rows[i];
        if (q) q[i] = x.q;
        if (r) r[i] = x.r;
        if (common) common[i] = x.common;
        if (denom) denom[i] = x.denom;
        if (pvalue) pvalue[i] = x.p;
    }
    return HS_OK;
}

HS_API int hs_distance_stats(const hs_distance *d, hs_distance_stats_t *stats)
{
    if (!d || !stats) return fail(HS_EINVAL, "null argument");
    *stats = d->stats;
    stats->n_queries = d->q.size();
    return HS_OK;
}

HS_API void hs_distance_free(hs_distance *d)
{
    if (!d) return;
    int cur = -1;
    const bool other = cudaGetDevice(&cur) == cudaSuccess && cur != d->device;
    if (other) cudaSetDevice(d->device);
    if (d->st.get()) cudaStreamSynchronize(d->st.get());
    if (d->st_copy.get()) cudaStreamSynchronize(d->st_copy.get());
    if (other) cudaSetDevice(cur);
    delete d;
}
