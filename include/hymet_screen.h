/*
 * hymet_screen.h -- C ABI of libhymet_screen.so: the B200-native `mash screen`.
 *
 * What it replaces.  HYMET's candidate selection calls an external process,
 *     mash screen -p 8 -v 0.9 "$MASH_SCREEN" "$INPUT_DIR"/ *.fna > "$SCREEN_TAB"
 * (/root/reference/scripts/mash.sh:14; three times per run from
 * /root/reference/run_hymet_cami.sh:85-96 and main.pl:94-104).  The reference
 * has no FFI for this path -- the process boundary is the interface -- so the
 * drop-in has two layers:
 *   1. bin/mash (Python) keeps the CLI and the TSV byte-for-byte, and
 *   2. this header is what that shim binds with ctypes.  Each entry point is
 *      annotated with the step of `mash screen` it stands for (SURVEY.md 8a
 *      rows a4..a16; Mash's own source is third-party and not under
 *      /root/reference, so rows cite the survey's restated rules S1..S22).
 *
 * Conventions: plain C, no C++/torch types; every function returns HS_OK (0) or
 * a negative HS_E* code and leaves a message for hs_last_error() (thread local).
 * The caller allocates every output array.  There is no CPU fallback: without an
 * sm_100 device hs_init() fails and every device entry point returns HS_ENODEV.
 * One hs_screen is one query stream; handles are not re-entrant.
 */
#ifndef HYMET_SCREEN_H
#define HYMET_SCREEN_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HS_OK 0
#define HS_EINVAL (-1)       /* bad argument */
#define HS_ENODEV (-2)       /* no sm_100 (B200) device / hs_init not called */
#define HS_ECUDA (-3)        /* CUDA runtime error (message has the detail) */
#define HS_EIO (-4)          /* could not open / read an input */
#define HS_EFORMAT (-5)      /* malformed .msh */
#define HS_ENOMEM (-6)
#define HS_EUNSUPPORTED (-7) /* S22: protein / noncanonical / preserveCase sketches, k > 32 */
#define HS_ENOSEQ (-8)       /* S6: "Did not find sequence records in inputs" */
#define HS_ESTATE (-9)       /* call order violated */

typedef struct hs_msh hs_msh;       /* a parsed .msh on the host */
typedef struct hs_db hs_db;         /* a sketch database resident on one GPU */
typedef struct hs_screen hs_screen; /* one screen (query stream) against a db */

typedef struct {
    uint32_t k, s, seed, use64;   /* from the sketch file, never from the CLI (Appendix A) */
    uint64_t n_refs, n_entries;   /* N sketches, E stored hashes */
    uint64_t n_distinct;          /* D distinct hashes (device dbs only, else 0) */
    uint64_t n_buckets;           /* hash-table buckets: 128-byte lines of 10 keys + their ids (device dbs only) */
    uint64_t max_key;             /* largest stored hash: exact range pre-filter */
    uint64_t device_bytes;        /* HBM held by the db */
    uint64_t bloom_bytes;         /* size of the L2-resident Bloom second-tier filter (0 = not built) */
    double t_parse_s, t_build_s;  /* .msh parse / GPU table build, seconds */
    uint64_t dense_max;           /* hashes <= dense_max are probed directly, (dense_max, max_key] go through the
                                     Bloom tier first (== max_key when that tier was not built) */
    uint64_t bloom_keys;          /* estimate of the stored hashes above dense_max */
} hs_db_info_t;

typedef struct {
    uint64_t n_bases;        /* characters inside sequence records ("query bases", the Mbp of Mbp/s) */
    uint64_t n_records;
    uint64_t n_positions;    /* packed positions streamed (bases + record separators + padding) */
    uint64_t n_valid_kmers;  /* K: k-mers hashed (S4) */
    uint64_t n_probes;       /* P: table probes issued (<= K when the range pre-filter is on) */
    uint64_t n_bucket_reads; /* 128-byte bucket lines read by those probes */
    uint64_t n_hits;         /* H: probes that found a key (count updates) */
    uint64_t n_mix_inserts;  /* hashes offered to the mixture bottom-s set */
    uint64_t set_size;       /* S10, printed by mash as "Estimated distinct k-mers in mixture" */
    uint64_t n_mixture;      /* |M| <= s (S9) */
    uint64_t h2d_bytes, d2h_bytes;
    uint32_t n_launches;     /* kernels launched for this screen so far */
    uint32_t n_mix_passes;   /* hashing passes needed for the mixture set (1 unless re-thresholded) */
    float ms_stream;         /* device time of the k-mer/probe kernels (CUDA events) */
    float ms_reduce;         /* device time of mixture finalise + per-sketch reduction */
    float ms_reset;          /* device time of the reset that preceded this screen (counts, mixture set) */
    uint32_t reduce_path;    /* 0 = O(present hashes) kernels, 1 = dense O(stored hashes) kernels */
    uint32_t n_touched;      /* distinct stored hashes present in the query (non-zero counts) */
    uint32_t n_hit_refs;     /* references with shared > 0 (sparse path) */
    uint32_t n_pairs;        /* (present hash, reference holding it) pairs walked (sparse path) */
    uint32_t exchange_overflow; /* multi-GPU: a rank's pair record was too small, nothing was added
                                   (hs_screen_counts_absorb): redo the exchange densely */
    uint32_t exchange_max_pairs; /* multi-GPU: largest pair count among the ranks' records (sizes the next one) */
    uint32_t mix_unsettled;      /* multi-GPU after hs_screen_flush_async: some rank's bottom-s selection did not hold; the
                                    counts are merged, the mixture is not: hs_screen_flush, exchange the mixture again, finish again */
} hs_stats_t;

/* ---- library ------------------------------------------------------------ */
const char *hs_version(void);
const char *hs_last_error(void);
/* Select CUDA device `device` (ordinal) for the handles THIS THREAD creates from now on and for the
 * handle-less entry points it calls.  Fails with HS_ENODEV unless the device is compute capability 10.x.
 * A db and its screens stay on the device they were created on, so one process can drive
 * several GPUs: hs_init(0), build db 0, hs_init(1), build db 1, ... */
int hs_init(int device);
/* Where hs_init placed the calling thread: it narrows the thread's CPU affinity to the NUMA node the GPU
 * hangs off (packer/reader threads inherit it, pinned buffers are first-touched there), unless
 * HYMET_SCREEN_NUMA=0.  numa_node = -1: unknown or left alone; cpus = CPUs the thread may run on. */
int hs_host_placement(int *numa_node, int *cpus);
/* Number of SMs of the bound device (148 on B200); 0 before hs_init. */
int hs_sm_count(void);

/* ---- .msh on the host (row a4: Sketch::initFromFiles) --------------------- */
int hs_msh_open(const char *path, hs_msh **out);
int hs_msh_info(const hs_msh *m, hs_db_info_t *info);
/* name/comment stay owned by the hs_msh; hashes -> pointer to n_hashes ascending
 * 64-bit values (32-bit sketches are widened). length = S18. */
int hs_msh_ref(const hs_msh *m, uint64_t i, const char **name, const char **comment, uint64_t *length,
               uint64_t *n_hashes, const uint64_t **hashes);
void hs_msh_free(hs_msh *m);

/* ---- database on the GPU (row a5: the "Loading..." hash-table build) ------- */
int hs_db_from_msh(const hs_msh *m, hs_db **out);
int hs_db_load_msh(const char *path, hs_db **out); /* open + from_msh */
/* Row a3 (run_hymet_cami.sh:85-97 screens the same contigs against data/sketch1-3.msh, one mash
 * process each): ONE table over the references of n sketch files, in file order, so that a single
 * pass over the query serves all of them.  Reference indices of file j are
 * [ref_begin[j], ref_begin[j+1]) (hs_db_segments).  Counts and the mixture do not depend on the
 * file; winner-take-all and the set size (hence p-values) are evaluated per file, with that
 * file's sketch size.  The files must agree in k, seed and hash width (HS_EUNSUPPORTED if not). */
int hs_db_from_msh_multi(const hs_msh *const *ms, uint32_t n, hs_db **out);
/* n_segments = number of files the db was built from (1 for the other constructors);
 * ref_begin[n_segments+1], seg_s[n_segments] may be NULL. */
int hs_db_segments(const hs_db *db, uint32_t *n_segments, uint64_t *ref_begin, uint32_t *seg_s);
/* Build from flat host arrays: offsets[n_refs+1], hashes[offsets[n_refs]] ascending per
 * reference, lengths[n_refs] (may be NULL -> 0).  Names are empty. */
int hs_db_from_arrays(uint32_t k, uint32_t s, uint32_t seed, uint64_t n_refs, const uint64_t *offsets,
                      const uint64_t *hashes, const uint64_t *lengths, hs_db **out);
int hs_db_info(const hs_db *db, hs_db_info_t *info);
int hs_db_ref(const hs_db *db, uint64_t i, const char **name, const char **comment, uint64_t *length,
              uint64_t *n_hashes);
void hs_db_free(hs_db *db);

/* ---- one screen ---------------------------------------------------------- */
int hs_screen_new(hs_db *db, hs_screen **out);
/* Run on a caller-owned CUDA stream (cudaStream_t as void*; NULL = library's own). */
int hs_screen_set_stream(hs_screen *s, void *cuda_stream);
/* Options: "filter" 1/0 = skip probes for hashes above the db's largest key (exact;
 * default 1); "sparse" 1/0 = O(present hashes) reduction and reset (default 1; 0 = always the dense kernels);
 * "chunk_bases" = host packer chunk size;
 * "ingest" 0/1/2 = host packer only / device parser only / both compete (default; packer
 * threads join when at least six were asked for); "file_readers", "file_block_bytes" = reader
 * threads and nominal block size of the pinned ring that streams plain FASTA files (defaults
 * 4 x 8 MiB: sized for a one-shot process, pinning costs ~0.5 ms per MB); "file_mode" 0/1/-1 = plain
 * FASTA files go through that ring to the device parser / are mapped and packed by the host threads
 * where the page cache holds them / chosen by host capability (default: mapped when the packer has
 * its AVX-512 path and at least four threads); "text_chunk_bytes" =
 * bytes of gzip / stdin FASTA inflated per hand-over to the packer threads (default 256 MiB;
 * cut at record starts -- FASTQ too, where the packer's own walk tells a header from a quality line that starts with '@').
 * Any other key is refused with HS_EINVAL.  Packed query chunks stay in HBM until reset (the mixture
 * threshold may have to be revisited): one screen holds 3/8 byte per query base, i.e. ~480 Gbp fit a
 * 180 GB B200 -- split larger read sets across screens and GPUs. */
int hs_screen_set_option(hs_screen *s, const char *key, int64_t value);

/* rows a6/a7: stream FASTA/FASTQ (plain or gzip; "-" = stdin).  A plain FASTA file is read by
 * up to `host_threads` reader threads (pread of record-aligned blocks into a pinned ring) and
 * parsed, packed and hashed on the GPU; gzip, FASTQ and stdin are packed on the host into
 * pinned 2-bit buffers with `host_threads` threads while the GPU consumes. */
int hs_screen_feed_fasta(hs_screen *s, const char *path, int host_threads);
/* The records of a plain FASTA file that START in the byte range [begin, end): N callers with adjacent
 * ranges (N GPUs in one process, or N ranks) cover the file exactly once and no k-mer spans two of them.
 * HS_EUNSUPPORTED for gzip / FASTQ / pipes, which cannot be cut: feed those whole to one screen. */
int hs_screen_feed_fasta_range(hs_screen *s, const char *path, uint64_t begin, uint64_t end, int host_threads);
/* Same, text already in host memory. */
int hs_screen_feed_text(hs_screen *s, const char *text, size_t n, int host_threads);
/* Pre-packed HOST buffers (layout: hs_packed_words()).  n_bases positions. */
int hs_screen_feed_packed(hs_screen *s, const uint64_t *seq2, const uint32_t *inv, uint64_t n_bases);
/* Pre-packed DEVICE buffers, used in place (must stay alive until finish; allocation
 * must hold hs_packed_words(n_bases) words of each array). */
int hs_screen_feed_packed_device(hs_screen *s, const void *d_seq2, const void *d_inv, uint64_t n_bases);
/* Words each packed array must hold for n_bases positions (tile padding included). */
uint64_t hs_packed_words(uint64_t n_bases);
/* Host packer alone (no GPU): text -> seq2/inv with capacity cap_words each; returns
 * positions in *n_bases.  stats may be NULL. */
int hs_pack_text(const char *text, size_t n, uint64_t *seq2, uint32_t *inv, uint64_t cap_words,
                 uint64_t *n_bases, hs_stats_t *stats);

/* Device parser alone (row a6 on the GPU): same contract and same output as hs_pack_text,
 * computed by the FASTA-ingest kernels ('>' records only; FASTQ goes through the host
 * packer).  Used by the parity tests; the streaming path calls the same kernels when
 * hs_screen_feed_text is given pinned host memory (option "ingest": 0 host packer,
 * 1 device parser, 2 both compete for chunks -- default). */
int hs_pack_text_device(const char *text, size_t n, uint64_t *seq2, uint32_t *inv, uint64_t cap_words,
                        uint64_t *n_bases, hs_stats_t *stats);

/* rows a8-a10 complete: wait for the stream, settle the local mixture bottom-s. */
int hs_screen_flush(hs_screen *s);
/* The same without waiting: the device-side selection of the bottom-s is enqueued, and the next
 * hs_screen_finish / _finish_hits completes the flush with its own (single) synchronisation.  In between,
 * hs_screen_mixture_record, hs_screen_mixture_merge_device, hs_screen_counts_compact_async and
 * hs_screen_counts_absorb may be enqueued: a whole multi-GPU screen then synchronises with the host
 * once.  See hs_stats_t.mix_unsettled for the (rare) fallback. */
int hs_screen_flush_async(hs_screen *s);

/* Multi-GPU seam (SURVEY.md 8e): after flush, counts[] (uint32, one per stored hash
 * entry id; device pointer) may be summed across ranks in place, and every rank's local
 * mixture hashes merged into every other rank, before finish. */
int hs_screen_counts_devptr(hs_screen *s, void **d_counts, uint64_t *n);
/* Sparse form of the same exchange, for when few hashes were hit: compact the non-zero counts into
 * (entry id << 32 | count) pairs in a DEVICE buffer of `cap` pairs.  The pairs come from the screen's
 * record of which counts left zero -- O(present hashes) -- or, when that record overflowed, from a
 * scan of all counts.  Enqueued on the screen's stream without waiting: the pair count goes to the
 * uint32 at d_n_out (device memory; it may exceed cap: then the pairs are incomplete), so a whole
 * exchange needs a single host synchronisation.  May be called before hs_screen_flush (after the last
 * feed): counts[] no longer changes, and the collective that carries the pairs can then run
 * underneath the flush. */
int hs_screen_counts_compact_async(hs_screen *s, void *d_pairs, uint32_t cap, void *d_n_out);
/* The whole exchange in one launch: d_rows = what an all-gather of every rank's record leaves in
 * DEVICE memory, n_rows records of (1 + cap) 64-bit words each, word 0 = that rank's pair count, then
 * its pairs; row `skip_row` (this rank's own) is not added.  If any record holds more than cap pairs
 * nothing is added and hs_stats_t.exchange_overflow is set by the next hs_screen_finish -- every rank
 * sees the same records, so every rank takes the same decision.  No host synchronisation. */
int hs_screen_counts_absorb(hs_screen *s, const void *d_rows, uint32_t n_rows, uint32_t cap, uint32_t skip_row);
/* Several GPUs in ONE process (HYMET_SCREEN_GPUS): add the counts and mixtures of n_src flushed screens
 * into dst (flushed too; all over copies of the same sketch database, one per GPU).  The in-process form
 * of the distributed exchange: each source's pair record is built on its own device and peer-copied
 * (over NVLink when the GPUs are peers) to dst's, then hs_screen_counts_absorb and
 * hs_screen_mixture_merge_device do the rest.  dst then finishes for everybody.  Refused, with every
 * handle left as it was: dst among the sources, a source listed twice, an unflushed screen, or a dst
 * that has already absorbed since its last reset (HS_EINVAL / HS_ESTATE). */
int hs_screen_absorb_screens(hs_screen *dst, hs_screen *const *src, uint32_t n_src);
int hs_screen_mixture_get(hs_screen *s, uint64_t *hashes /*[s]*/, uint32_t *n);
/* Mixture exchange without the host: write this rank's record [length | s hashes, zero padded]
 * ((s + 1) 64-bit words, DEVICE memory) after flush; after the all-gather, merge n_rows such records
 * on the device (sort + unique, keep the s smallest, S10's set size per source file).  hs_screen_finish
 * then takes the set size from device memory and returns the merged mixture with the results. */
int hs_screen_mixture_record(hs_screen *s, void *d_record);
int hs_screen_mixture_merge_device(hs_screen *s, const void *d_rows, uint32_t n_rows);
/* Set size (S10) used for the p-values of one file of a multi-file db (after flush). */
int hs_screen_segment_set_size(hs_screen *s, uint32_t segment, uint64_t *set_size);

/* rows a11-a15: shared, median multiplicity, identity, p-value for every sketch, in
 * sketch order.  winner_take_all = mash's -w (S17).  Arrays have n_refs elements.
 * The work is O(hashes present in the query) -- the streaming kernel records which counts left
 * zero, and every stored hash is chained to the references that hold it -- with the dense
 * O(stored hashes) kernels as the fallback when that record overflows (hs_stats_t.reduce_path). */
int hs_screen_finish(hs_screen *s, int winner_take_all, uint64_t *shared, uint32_t *median,
                     double *identity, double *pvalue, hs_stats_t *stats);
/* The same reduction, but only the references mash would print (shared > 0; S15) come back: rows a14-a16
 * are computed for those alone and the GPU writes them into pinned host rows, so the trip home is
 * O(references with hits) instead of 24 bytes for each of N.  *n_hits = how many there are;
 * hs_screen_hits_copy then fills the caller's arrays (`cap` elements each, NULL to skip a column) in
 * ascending reference order -- the line order of the TSV. */
int hs_screen_finish_hits(hs_screen *s, int winner_take_all, uint32_t *n_hits, hs_stats_t *stats);
int hs_screen_hits_copy(hs_screen *s, uint32_t cap, uint32_t *ref, uint64_t *shared, uint32_t *median,
                        double *identity, double *pvalue);
/* Forget the query (counts, mixture, stats) so the handle can screen another one. */
int hs_screen_reset(hs_screen *s);
int hs_screen_stats(hs_screen *s, hs_stats_t *stats);
void hs_screen_free(hs_screen *s);

/* ---- single stages, for parity tests and per-kernel measurement ------------ */
/* K1 alone (row a7/a8): hash every k-mer of a packed host buffer.  out_hash/out_valid
 * have n_bases elements, indexed by the position of the k-mer's LAST base. */
int hs_hash_packed(uint32_t k, uint32_t seed, const uint64_t *seq2, const uint32_t *inv, uint64_t n_bases,
                   uint64_t *out_hash, uint8_t *out_valid);
/* K2 alone (row a10): probe n host hashes; out_entry[i] = canonical entry id of the
 * key (index into the db's flat hash array of its first occurrence) or 0xFFFFFFFF. */
int hs_db_probe(hs_db *db, const uint64_t *hashes, uint64_t n, uint32_t *out_entry);
/* K2 alone on DEVICE hashes, timed: increments nothing, returns hits and device ms. */
int hs_db_probe_device(hs_db *db, const void *d_hashes, uint64_t n, uint64_t *n_hits,
                       uint64_t *n_bucket_reads, float *ms);
/* Measurement reference for K2: time n_reads independent random 32-byte sector reads over a
 * device buffer of `bytes` (make it much larger than L2). */
int hs_gather_bench(const void *d_buf, uint64_t bytes, uint64_t n_reads, float *ms);
/* canonical entry id of every stored entry (n_entries values). */
int hs_db_entry_ids(hs_db *db, uint32_t *out);
/* K6 alone (rows a14/a15). */
int hs_stat_batch(uint32_t k, uint64_t set_size, uint64_t n, const uint64_t *shared, const uint64_t *size,
                  double *identity, double *pvalue);
/* ---- `mash sketch` of a genome collection (SURVEY.md 8f rank 1) ------------------------------------
 * One sketch per input file: the s smallest distinct canonical k-mer hashes of all its records.
 * host_threads threads each take whole files (plain or gzip FASTA/FASTQ), inflate and pack them while
 * the GPU hashes the previous batch; a batch holds many genomes and one kernel pass gives each its own
 * bottom-s set.  Results come back in the order the files were added. */
typedef struct hs_sketcher hs_sketcher;
typedef struct {
    uint64_t n_genomes;      /* inputs sketched */
    uint64_t n_bases;        /* sequence bases of all inputs */
    uint64_t n_positions;    /* packed positions hashed by first passes (bases + record separators) */
    uint32_t n_batches;      /* batches sent to the GPU, re-stream batches included */
    uint32_t n_launches;     /* kernels launched */
    uint32_t n_passes;       /* genome re-streams the exactness check asked for (threshold raised or lowered) */
    float ms_stream;         /* device time of the hashing launches (CUDA events) */
    float ms_select;         /* device time of the per-genome selections */
    double t_read_s;         /* host thread-seconds reading and inflating files */
    double t_pack_s;         /* host thread-seconds packing text */
    double t_wait_s;         /* time the GPU-feeding thread waited for packed genomes */
    double t_total_s;        /* wall clock of hs_sketcher_run */
} hs_sketch_stats_t;

/* k 1..32, s >= 1; host_threads < 1 means 1. */
int hs_sketcher_new(uint32_t k, uint32_t s, uint32_t seed, int host_threads, hs_sketcher **out);
/* Queue one file; it is read by hs_sketcher_run (HS_EIO there if it cannot be read). */
int hs_sketcher_add_file(hs_sketcher *sk, const char *path);
/* Sketch everything queued.  Once per handle. */
int hs_sketcher_run(hs_sketcher *sk);
/* Input i after run: n ascending hashes (owned by the handle), total sequence length, record count
 * (occurrences of "\n>" plus one if the text starts with '>') and the bytes of the first header line
 * after its '>' (empty unless the text starts with '>'; not NUL-terminated: header_len bytes). */
int hs_sketcher_result(const hs_sketcher *sk, uint64_t i, const uint64_t **hashes, uint32_t *n, uint64_t *length,
                       uint64_t *n_records, const char **header, uint64_t *header_len);
int hs_sketcher_stats(const hs_sketcher *sk, hs_sketch_stats_t *stats);
void hs_sketcher_free(hs_sketcher *sk);

/* `mash sketch` of one genome held as FASTA text: s smallest distinct hashes (a sketcher batch of one). */
int hs_sketch_text(uint32_t k, uint32_t s, uint32_t seed, const char *text, size_t n, uint64_t *out_hashes,
                   uint32_t *n_out, uint64_t *length);

/* Same, for a genome already packed in DEVICE memory (hs_packed_words() layout). */
int hs_sketch_packed_device(uint32_t k, uint32_t s, uint32_t seed, const void *d_seq2, const void *d_inv,
                            uint64_t n_bases, uint64_t *out_hashes, uint32_t *n_out);
/* Device-side packer: n base codes (uint8: 0..3 = A,C,G,T, anything else = invalid position)
 * in DEVICE memory -> packed DEVICE arrays of hs_packed_words(n) words (padding flagged
 * invalid).  Runs on `cuda_stream` (NULL = default stream) and returns without syncing. */
int hs_pack_codes_device(const void *d_codes, uint64_t n, void *d_seq2, void *d_inv, void *cuda_stream);

/* ---- `mash dist`: one reference sketch file against query sketches (DESIGN.md §5 "mash dist") ------------------
 * Every (query, reference) pair gets Mash 2.3's exact (common, denom) -- its merge of the two sorted
 * sketches truncated at s_p, the smaller of the two files' sketch sizes -- its distance and its p-value.
 * On the device: the pairs that share a hash (found through the reference key table, one query block at
 * a time), the merge and the p-value.  On the host: the distance and both filters, from the exact
 * integers with libm, and the TSV.  Pairs that share no hash are written without device work. */
typedef struct hs_distance hs_distance;
typedef struct {
    uint64_t n_queries, n_refs;
    uint64_t n_candidates;   /* pairs that share a hash (computed blocks, redone ones excluded) */
    uint64_t n_lines;        /* lines written (-t: query rows) */
    uint32_t n_blocks;       /* query blocks sent to the device, redone ones included */
    uint32_t n_splits;       /* blocks whose candidates overflowed the result buffer: redone at half the size */
    uint32_t block_queries;  /* queries per block (chosen so that the block's bitmap and sketches stay in L2) */
    uint32_t result_cap;     /* candidate pairs one block's result buffer holds */
    float ms_mark;           /* device time: probes + chain walks marking candidate pairs (CUDA events) */
    float ms_compact;        /* device time: popcount, scan, compaction into (q, r) rows */
    float ms_merge;          /* device time: truncated merges + p-values */
    double t_write_s;        /* host seconds formatting and writing lines */
    double t_total_s;        /* wall clock of the runs */
} hs_distance_stats_t;

/* The reference side: a key table over the sketches of `ref` on the bound device. */
int hs_distance_new(const hs_msh *ref, hs_distance **out);
/* Queue every sketch of one query file, in file order.  HS_EUNSUPPORTED if its k-mer size, seed or hash
 * width differs from the reference's.  Its sketch size sets s_p for its pairs. */
int hs_distance_add_msh(hs_distance *d, const hs_msh *m);
/* Queue one sketch (a sketcher result): n ascending hashes, sketch size s of the file it stands for. */
int hs_distance_add_sketch(hs_distance *d, const char *name, const char *comment, uint64_t length, uint32_t s,
                           const uint64_t *hashes, uint64_t n);
/* Write `mash dist` output for every queued query (queries outer, references inner) to fd.  Pairs with
 * distance > max_distance or p-value > max_pvalue (both in [0, 1]) are left out; table = -t (one row
 * per query, distances only), comments = -C (name:comment); host_threads format disjoint query ranges. */
int hs_distance_run(hs_distance *d, int fd, double max_distance, double max_pvalue, int table, int comments,
                    int host_threads);
/* The same pipeline without output: keeps the candidate pairs (those that share a hash) in (query,
 * reference) order; *n_rows = how many.  p-value < 0: not computed, the pair is farther than max_distance.
 * hs_distance_rows_copy fills the caller's arrays (cap elements each, NULL to skip a column). */
int hs_distance_run_rows(hs_distance *d, double max_distance, uint64_t *n_rows);
int hs_distance_rows_copy(const hs_distance *d, uint64_t cap, uint32_t *q, uint32_t *r, uint32_t *common,
                          uint32_t *denom, double *pvalue);
/* Counters accumulated over the handle's runs. */
int hs_distance_stats(const hs_distance *d, hs_distance_stats_t *stats);
void hs_distance_free(hs_distance *d);

/* ---- SURVEY.md 8f rank 4: the classifier's weighted-LCA vote ----------------------------------------
 * /root/reference/scripts/classification_cami.py:251-308 (_weighted_lca, _process_one) for n_q queries
 * at once, one GPU thread per query, bit-exact with the reference's double arithmetic (sums in dict
 * insertion order, first maximum wins).  Alignments of query q are [q_off[q], q_off[q+1]); tax[j] = row of
 * `names` for the target's taxid or -1, w[j] = coverage x reference abundance; names[n_tax][8] = name id
 * per rank (superkingdom..strain), 0 = none.  out_names[q][0..out_depth[q]) = chosen names, out_depth = 0
 * means "Unknown"; out_any[q] = some alignment had a taxid. */
int hs_lca_weighted(uint64_t n_q, const uint64_t *q_off, const int32_t *tax, const double *w, uint64_t n_tax,
                    const uint32_t *names, uint32_t *out_names, uint32_t *out_depth, double *out_conf, uint8_t *out_any);

#ifdef __cplusplus
}
#endif
#endif /* HYMET_SCREEN_H */
