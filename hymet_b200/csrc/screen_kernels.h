// screen_kernels.h -- launch interface of the hand-written sm_100a kernels.
// Internal to libhymet_screen.so (the public surface is include/hymet_screen.h).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "kmer_core.cuh"

namespace hs {

constexpr int kTileWords = 256;    // 256 words = 8192 bases; the stream kernel's CTAs take 1 or 2 tiles per pass
constexpr uint32_t kNoEntry = 0xFFFFFFFFu;

// counters accumulated by the streaming kernel (device, 64-bit each)
enum StatSlot { ST_VALID = 0, ST_PROBES, ST_BUCKETS, ST_HITS, ST_MIXINS, ST_COUNT };

struct TableView {
    const uint64_t *buckets; // n_buckets * kBucketWords: keys | canonical entry ids | overflow flag (kmer_core.cuh)
    uint32_t n_buckets;
    uint64_t max_key;       // largest stored key (exact range pre-filter)
    uint32_t special;       // canonical entry id of key == kEmptyKey, or kNoEntry
    // Two-tier pre-filter for databases whose keys are spread over the whole hash range (sketches
    // of viral/plasmid-sized genomes keep ALL their k-mer hashes, so max_key ~ 2^64 and the range
    // test alone stops helping).  Keys <= dense_max -- where the sketches of ordinary genomes
    // live, a sliver of the hash range -- are probed directly; the keys above it are few and go
    // through a blocked Bloom filter (32-bit blocks, 3 bits per key, L2 resident) first.  No false
    // negatives => results unchanged.  bloom == NULL: every hash <= max_key is probed.
    const uint32_t *bloom;
    uint32_t bloom_mask;    // words - 1 (power of two)
    uint64_t dense_max;
};

// Per-screen record of WHICH counts are non-zero, so that everything after the streaming pass
// (count exchange, "Summing shared", -w, medians, reset) is O(present hashes), as it is in mash
// itself (SURVEY.md 8a row a11), not O(stored hashes).
struct SparseState {
    uint32_t n_touched;     // entry ids appended to touched[] (> cap: the list is incomplete)
    uint32_t wrapped;       // a count passed 2^32 (S8 wraps): a zero may be a present key
    uint32_t n_hit;         // references with shared > 0
    uint32_t n_pairs;       // depth slots handed out
    uint32_t overflow;      // a sparse buffer was too small -> the caller reruns the dense reduction
    uint32_t xchg_overflow; // multi-GPU: some rank's record held more pairs than its capacity
    uint32_t xchg_max;      // multi-GPU: the largest pair count among the ranks' records
    uint32_t n_mix;         // merged mixture length (device-side merge)
    uint32_t mix_has_max;   // the value 2^64-1 is in the merged mixture (it doubles as the sort padding)
    uint32_t mix_unsettled; // some rank's mixture record said "not settled" (device-side selection fell through)
    unsigned long long set_size[8];   // S10 per source file, when the mixture was merged on the device
};
struct SparseView {
    uint32_t *touched;      // canonical entry ids whose count left zero, in arrival order
    uint32_t cap;
    SparseState *st;
};

// Mixture bottom-s state lives on the device so that streaming never waits for the host:
// the threshold is lowered by a maintenance kernel after each chunk, not by a host check.
struct MixState {
    unsigned long long tau;  // accept h <= tau (min over launches of their caps, /4 per shrink)
    uint32_t count;          // distinct values in sets[cur]
    uint32_t new_count;      // scratch while rebuilding into sets[cur ^ 1]
    uint32_t overflow;       // an insert was dropped: the set is incomplete below tau
    uint32_t has_max;        // hash == kEmptyKey seen (only possible while tau == 2^64-1)
    uint32_t cur;            // live set
    uint32_t n_out, n_unique;  // finalisation scratch
    uint32_t rebuilds;
    uint32_t sel_too_many;   // device-side selection: more candidates than the sort holds (host falls back)
    unsigned long long sel_thr;  // device-side selection: values <= sel_thr were collected
};
struct MixView {
    uint64_t *sets[2];      // open addressing, capacity mask+1, kEmptyKey = free
    uint32_t mask;
    uint32_t limit;         // max distinct before `overflow` is raised
    uint64_t tau_cap;       // this launch's cap: expected offers stay <= capacity/8
    MixState *st;
};

// `mash sketch` of many genomes in one launch (k_stream MODE 4).  Every genome starts on a tile
// boundary of the batch and ends with at least one invalid position, so no k-mer spans two genomes,
// and tile_genome[] names each tile's genome.  A genome's set holds the distinct hashes <= its own
// threshold st.tau; mix_insert sees st (count, overflow, has_max) as it sees the mixture's.
struct SketchSlot {
    MixState st;
    uint64_t set_off;       // its set: SketchView::sets + set_off, mask + 1 slots (a power of two)
    uint32_t mask, limit;   // limit: distinct values before `overflow` is raised
};
struct SketchView {
    const uint32_t *tile_genome;   // slot index of every tile of the launch
    SketchSlot *slots;             // NULL: not a sketch launch
    uint64_t *sets;
};

struct StreamArgs {
    const uint64_t *seq;    // packed words (16-byte aligned), n_tiles * kTileWords allocated
    const uint32_t *inv;
    uint64_t n_bases;       // positions >= n_bases are invalid whatever inv says
    const unsigned long long *n_bases_dev;  // if set, the length is read from HBM (device-parsed chunks)
    uint32_t n_tiles;       // END tile (exclusive) of this launch
    uint32_t tile_begin;    // first tile of this launch (> 0: a later piece of the same chunk, halo is real data)
    int k;
    uint32_t seed;
    int use64;
    int do_count;           // probe + count
    int do_filter;          // skip probes for h > max_key
    int do_mix;             // offer hashes <= tau to the mixture set
    TableView tab;
    uint32_t *counts;       // per canonical entry id
    SparseView sparse;      // touched == NULL: do not record
    MixView mix;
    unsigned long long *stats;  // ST_COUNT slots
    uint64_t *emit_hash;    // optional: per position hash (K1 parity), n_bases entries
    uint8_t *emit_valid;
    int probe_all;          // (nearly) every k-mer probes: use the warp-cooperative instantiation
    SketchView sk;          // sk.slots set: per-genome bottom-s sets, nothing else (do_count = do_mix = 0)
};

// ---- streaming (K1+K2+K3 insert) -------------------------------------------
cudaError_t launch_stream(const StreamArgs &a, int sm_count, cudaStream_t st);

// ---- database build (row a5) -------------------------------------------------
cudaError_t launch_table_insert(uint64_t *buckets, uint32_t n_buckets, const uint64_t *hashes,
                                uint64_t n_entries, uint32_t *special, uint32_t *fail, cudaStream_t st);
// canon[e] = canonical id of entry e's key; next[] links the entries that hold the same key into a
// chain that starts at the canonical one (next[] must be filled with kNoEntry beforehand)
cudaError_t launch_table_canon(const TableView &t, const uint64_t *hashes, uint64_t n_entries, uint32_t *canon,
                               uint32_t *next, unsigned long long *n_distinct, cudaStream_t st);
cudaError_t launch_bloom_build(uint32_t *bloom, uint32_t bloom_mask, uint64_t dense_max, bool use64,
                               const uint64_t *hashes, uint64_t n, cudaStream_t st);
// standalone probe (K2), warp-cooperative: eight lanes read one 128-byte bucket.  out_entry may be
// NULL; stats[0]=hits, stats[1]=bucket reads
cudaError_t launch_probe(const TableView &t, const uint64_t *hashes, uint64_t n, uint32_t *out_entry,
                         unsigned long long *stats, int sm_count, cudaStream_t st);

// random 32-byte sector reads over `bytes` of device memory (measurement reference for K2)
cudaError_t launch_gather_bench(const void *buf, uint64_t bytes, uint64_t total_reads, int sm_count, cudaStream_t st);

// ---- mixture bottom-s (K3) ---------------------------------------------------
// MixState := {tau, everything else 0} without a host buffer (no synchronisation to reuse one)
cudaError_t launch_mix_state_init(MixState *st, uint64_t tau, cudaStream_t stm);
// copy keys <= thr from the set into out (append with atomic cursor); counts all <= thr
cudaError_t launch_mix_collect(const uint64_t *set, uint32_t cap, uint64_t thr, uint64_t *out, uint32_t out_cap,
                               uint32_t *n_out, cudaStream_t st);
// after a streaming launch: fold its cap into tau and, if the live set is more than a
// quarter full, rebuild it at tau/4 into the other buffer (exact: >= s smaller values stay)
cudaError_t launch_mix_maintain(const MixView &v, cudaStream_t st);
// The whole selection on the device, no host decision in between: histogram of the live set below
// tau (2048 bins) -> smallest threshold with >= s values under it -> collect -> sort + unique.
// out[] (capacity n_pad, a power of two >= s + slack) ends up ascending and distinct, st->n_unique
// long; st->sel_too_many is raised when more than n_pad values lay under the threshold.
cudaError_t launch_mix_select(const MixView &v, uint32_t s, bool use64, uint32_t *hist /*2 * 2048 + 8*/, uint64_t *out,
                              uint32_t n_pad, uint64_t *scratch, cudaStream_t st);
// sort ascending + unique in place (n <= cap_pow2 handled by padding); *n_unique out
cudaError_t launch_sort_unique(uint64_t *data, uint32_t n, uint64_t *scratch, uint32_t *n_unique, cudaStream_t st);
// one CTA per genome of a sketch batch: sort its set and write its min(s, count) smallest values to
// out + out_off[g], the number to n_out[g].  Sets larger than the shared-memory sort are sorted in place.
cudaError_t launch_sketch_select(const SketchSlot *slots, uint32_t n_slots, uint32_t max_cap, uint64_t *sets, uint32_t s,
                                 const uint64_t *out_off, uint64_t *out, uint32_t *n_out, cudaStream_t st);

// ---- per-sketch reduction (K4), winner-take-all (K5), statistics (K6) ---------
// DENSE forms (O(stored hashes)): the fallback when the touched list overflowed or counts wrapped
cudaError_t launch_sketch_reduce(const uint64_t *offsets, uint64_t n_refs, const uint32_t *canon,
                                 const uint32_t *counts, const uint32_t *winner /*nullable*/, uint32_t *shared,
                                 uint32_t *median, int sm_count, cudaStream_t st);
cudaError_t launch_winner(const uint64_t *offsets, uint64_t n_refs, const uint32_t *canon, const uint32_t *counts,
                          const uint32_t *shared, const uint64_t *lengths, unsigned long long *best_score,
                          unsigned long long *best_len, uint32_t *winner, uint64_t n_entries, int sm_count,
                          cudaStream_t st);
// set_size_dev != NULL: read S10's set size from device memory instead of the argument
cudaError_t launch_stats(uint32_t k, uint64_t set_size, const unsigned long long *set_size_dev, uint64_t n,
                         const uint32_t *shared32, const uint64_t *shared64, const uint64_t *offsets,
                         const uint64_t *sizes, double *identity, double *pvalue, cudaStream_t st);

// rows a14-a16 for the references with hits only; the rows live in host-mapped pinned memory
struct HitRows { uint32_t *ref, *shared, *median; double *identity, *pvalue; uint32_t cap; };
struct StatsHitArgs {
    uint32_t k, n_seg;
    unsigned long long set_size[8];           // S10 per source file (host value) ...
    const unsigned long long *set_size_dev;   // ... or, when not NULL, read from device memory
    const uint64_t *seg_begin;                // n_seg + 1 (device)
    const uint32_t *hit, *n_hit;              // references with hits, how many (device)
    const uint32_t *shared, *median;          // per reference
    const uint64_t *offsets;
    HitRows rows;
};
// from_dense: build hit[] / n_hit from shared[] first (the dense reduction leaves no hit list)
cudaError_t launch_stats_hits(const StatsHitArgs &a, bool from_dense, uint32_t n_refs, uint32_t *hit, uint32_t *n_hit,
                              int sm_count, cudaStream_t st);

// SPARSE forms (O(present hashes)), rows a11-a13: walk the touched list and, per present key, the
// chain of references that hold it.
struct SparseReduceArgs {
    SparseView sp;
    const uint32_t *counts, *next;
    const uint64_t *offsets;       // n_refs + 1
    uint32_t n_refs;
    const uint64_t *lengths;       // S18, for -w ties
    const uint64_t *seg_begin;     // n_seg + 1 reference indices: -w competes inside one source file
    uint32_t n_seg;
    uint32_t *shared, *median;     // n_refs each, zeroed by the caller
    uint32_t *plain;               // n_refs: shared counts before -w (its scores)
    uint32_t *hit;                 // n_refs: references with hits, arrival order
    uint32_t *seg_start, *seg_fill;// n_refs each
    uint32_t *depths;              // pair_cap
    uint32_t pair_cap;
    uint64_t ref_scale;            // floor(2^64 * n_refs / stored hashes): first guess of an entry's reference (0: none)
};
cudaError_t launch_sparse_reduce(const SparseReduceArgs &a, bool wta, int sm_count, cudaStream_t st);
// counts[touched[i]] = 0 for the recorded ids; the second launch clears every count instead when the
// list is incomplete (decided on the device: one of the two returns at once).  counts[] must be
// allocated in multiples of four entries.
cudaError_t launch_sparse_reset(const SparseView &sp, uint32_t *counts, int sm_count, cudaStream_t st);
cudaError_t launch_counts_clear_if_overflow(const SparseView &sp, uint32_t *counts, uint64_t n, cudaStream_t st);

// ---- count exchange (multi-GPU) -----------------------------------------------------
// (entry id << 32 | count) pairs of the touched ids; *n_out = how many there are (may exceed cap:
// then the pairs are incomplete).  Falls back, on the device, to scanning all counts when the
// touched list itself overflowed.
cudaError_t launch_counts_compact(const SparseView &sp, const uint32_t *counts, uint64_t n, unsigned long long *pairs,
                                  uint32_t cap, uint32_t *n_out, cudaStream_t st);
// All ranks' records at once: rows of (1 + cap) words, word 0 = pair count; row `skip` is this
// rank's own.  Nothing is added (and xchg_overflow is raised) if any row holds more than cap pairs.
cudaError_t launch_counts_absorb(const SparseView &sp, uint32_t *counts, uint64_t n_counts,
                                 const unsigned long long *rows, uint32_t n_rows, uint32_t cap, uint32_t skip,
                                 int sm_count, cudaStream_t st);
// Union of n_rows ascending hash lists (row = [length | s_cap hashes]) -> out[<= s] ascending distinct,
// length in st->n_mix, and S10's set size for each of n_seg sketch sizes in st->set_size[]
cudaError_t launch_mixture_merge(const unsigned long long *rows, uint32_t n_rows, uint32_t s_cap, uint32_t s,
                                 const uint32_t *seg_s, uint32_t n_seg, bool use64, uint64_t *work, uint32_t work_cap,
                                 uint64_t *scratch, uint64_t *out, SparseState *st, cudaStream_t stm);
// this rank's record for the mixture all-gather, written on the device from the device-side selection:
// [length | s hashes, zero padded], or length = kMixUnsettled when the selection did not hold
constexpr unsigned long long kMixUnsettled = ~0ull;
cudaError_t launch_mix_record(const MixView &v, uint32_t s, uint32_t sel_pad, const uint64_t *cand, unsigned long long *record,
                              int force_unsettled, cudaStream_t st);

// ---- device-side packer (codes -> 2-bit words + invalid mask) -------------------
cudaError_t launch_pack_codes(const uint8_t *codes, uint64_t n, uint64_t *seq, uint32_t *inv, uint64_t n_words_alloc,
                              cudaStream_t st);

}  // namespace hs

// ---- device-side FASTA ingest (row a6 on the GPU) --------------------------------
// Raw FASTA bytes in HBM -> base codes (0..3, 4 = invalid / record separator), compacted:
// headers and line ends removed, one separator per record, exactly like fasta_pack.cpp.
namespace hs {
constexpr int kFaTileBytes = 8192;   // 256 threads x 32 bytes
struct FaScratch {
    uint32_t *tile_event;   // per tile: its last newline/header-start event code (0 = none)
    uint32_t *tile_carry;   // exclusive prefix max of tile_event
    uint32_t *tile_event_b; // per tile: its last header-start/'+'-line event code
    uint32_t *tile_carry_b; // exclusive prefix max of tile_event_b, seeded "skipping"
    uint4 *masks;           // per 32 input bytes: newline / header-start / '+'-start / dropped-CR masks
    uint2 *emit;            // per 32 input bytes: emitted-byte mask, separator mask
    uint32_t *tile_count;   // per tile: positions emitted
    uint64_t *tile_offset;  // exclusive prefix sum of tile_count
    unsigned long long *totals;  // [0] positions, [1] sequence bases, [2] records  (accumulated)
    unsigned long long *chunk_positions;  // positions of THIS chunk (read by the pack/stream launches)
};
// text: n bytes (n < 2^30) starting at a record header; codes: capacity >= n
cudaError_t launch_fasta_to_codes(const uint8_t *text, uint32_t n, uint8_t *codes, const FaScratch &sc, cudaStream_t st);
// k_pack_codes / k_stream variants whose length comes from device memory (no host sync)
cudaError_t launch_pack_codes_dyn(const uint8_t *codes, const unsigned long long *n_dev, uint64_t *seq, uint32_t *inv,
                                  uint64_t n_words_alloc, cudaStream_t st);
}  // namespace hs
