// Append stage: merge of a finalized index A with the index B of one more batch into a compact index C.  Internal
// interface (api.cu <-> append.cu).
//
// Every protein of B has an id above every protein of A, so for an equal hash A's groups and postings come before B's and
// no two postings are ever compared: C is A with B's rows inserted at known points.  Per B key j the locate kernel finds
// the insertion key in A (lower bound through A's directory), whether the hash is already there, the insertion group and
// the insertion posting; a scan of the matched flags gives M, the shared keys (U_C = U_A + U_B - M, G_C = G_A + G_B,
// n_C = n_A + n_B).  Between two insertion points A's elements move as one run with a constant shift, so every output
// element of C finds its source with a binary search over the insertion points of its tile (a few entries, L1-resident).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "index_build.cuh"

namespace ks {

// One input of the merge in the compact layout: keys[U], key_grp[U + 1], grp_start[G + 1], loc[n].
struct MergeSide {
    const uint64_t* keys = nullptr;
    const uint32_t* key_grp = nullptr;
    const uint32_t* grp_start = nullptr;
    const uint64_t* loc = nullptr;
    uint64_t U = 0, G = 0, n = 0;
};

// Segmented layout -> compact (keys[U], key_grp[U + 1], grp_start[G + 1]; counts[0] = U, counts[1] = G): one CTA per sort
// bucket after a scan of the buckets' key and group counts.  `pre` holds 2 * seg_nb words.
cudaError_t launch_compact_segmented(const CsrView& v, uint64_t U, uint64_t G, uint32_t* pre, uint64_t* keys,
                                     uint32_t* key_grp, uint32_t* grp_start, uint64_t* counts, cudaStream_t stream,
                                     uint64_t* n_launches);

struct AppendArgs {
    MergeSide a, b;
    const uint32_t* dir_a = nullptr;  // A's compact directory (dir_bits_a / dir_shift_a)
    int dir_bits_a = 0, dir_shift_a = 0;
    uint32_t p_a = 0;                  // proteins of A: added to B's protein ids
    // out (device, preallocated): keys[U_A + U_B], key_grp[U_A + U_B + 1], grp_start[G_A + G_B + 1], loc[n_A + n_B];
    // d_counts[0] = U_C, [1] = G_C, [2] = M
    uint64_t* keys = nullptr;
    uint32_t *key_grp = nullptr, *grp_start = nullptr;
    uint64_t* loc = nullptr;
    uint64_t* d_counts = nullptr;
    void* work = nullptr;  // append_work_bytes(b.U)
    size_t work_bytes = 0;
};
size_t append_work_bytes(uint64_t u_b);

// locate + scan + the three copy kernels (keys with key_grp, grp_start, loc).  No synchronisation.
cudaError_t launch_append_merge(const AppendArgs& m, cudaStream_t stream, uint64_t* n_launches);

}  // namespace ks
