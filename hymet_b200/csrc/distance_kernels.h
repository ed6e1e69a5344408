// distance_kernels.h -- launch interface of the `mash dist` kernels (distance_kernels.cu).
// Internal to libhymet_screen.so (the public surface is include/hymet_screen.h).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "screen_kernels.h"

namespace hs {

// One candidate pair of a query block: k_dist_compact writes (q, r), k_dist_merge the rest.
// p < 0: not computed, because the pair is certainly farther than -d (the host drops it).
struct DistRow {
    uint32_t q, r;          // query (global index), reference
    uint32_t common, denom; // Mash's truncated merge (DESIGN.md §5 "mash dist", D1)
    double p;               // D3
};
static_assert(sizeof(DistRow) == 24, "DistRow is copied to the host as is");

struct DistArgs {
    TableView tab;               // the reference sketches' key table (hs_db)
    const uint32_t *next;        // hash -> references chains of that table
    const uint64_t *ref_off;     // n_refs + 1
    const uint64_t *ref_hashes;  // ascending per reference
    const uint64_t *ref_len;     // sequence lengths (S18)
    uint32_t n_refs;
    uint64_t ref_scale;          // first guess of an entry's reference (ref_of_entry)
    const uint64_t *q_off;       // all queries: n_queries + 1
    const uint64_t *q_hashes;
    const uint64_t *q_len;
    const uint32_t *q_sp;        // per query: the smaller of its file's and the reference file's sketch size
    uint32_t q0, n_q;            // this block: queries [q0, q0 + n_q)
    uint32_t *bitmap;            // n_q rows of `words` words; all zero on entry, left all zero by k_dist_compact
    uint32_t words;              // (n_refs + 31) / 32
    unsigned long long *row_start;  // n_q + 1: exclusive scan of the rows' popcounts, [n_q] = candidates
    DistRow *rows;               // cap rows, in (q, r) order
    uint32_t cap;
    uint32_t k;
    double max_d;                // -d: p-values are skipped for pairs certainly farther than this
};

// mark + count + scan + compact: the block's candidate pairs (the pairs that share a hash) in rows[],
// their number in row_start[n_q] (it may exceed cap: then rows[] holds the first cap of them).
// ev_mid, when not NULL, is recorded after the marking kernel.
cudaError_t launch_dist_candidates(const DistArgs &a, int sm_count, cudaEvent_t ev_mid, cudaStream_t st);
// k_dist_merge: (common, denom, p) of rows [0, min(row_start[n_q], cap)).
cudaError_t launch_dist_merge(const DistArgs &a, int sm_count, cudaStream_t st);

}  // namespace hs
