// Fused sketch stage: internal interface between the C ABI (api.cu) and the kernels (sketch.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "dense_scatter.cuh"

namespace ks {

constexpr int SK_THREADS = 256;
constexpr int SK_ROWS = 8;                         // windows per thread
constexpr int SK_TILE = SK_THREADS * SK_ROWS;      // window start positions per CTA
constexpr int SK_MAX_TEMPLATE_K = 32;              // k above this takes the generic (byte-loop) kernel
constexpr int SK_MAX_K = 256;                      // bound of the generic kernel's halo

struct Lut256 { uint8_t b[256]; };

struct SketchArgs {
    const uint8_t* residues;   // device, 16 B aligned.  packed == 0: n_res bytes + >= 64 readable pad bytes;
                               // packed == 1: 5-bit codes, 8 residues per 5 bytes (pack_residues), + >= 72 pad bytes
    int packed = 0;
    const uint64_t* offsets;   // device, n_prot + 1
    uint64_t n_res;
    uint64_t n_prot;
    uint32_t k;
    int moltype;               // 0 protein (identity), 1 dayhoff, 2 hp
    uint64_t max_hash;
    uint32_t pid_base;         // added to the local protein index in the emitted tuples
    uint64_t* out_hash;        // device, capacity entries (already offset to the append position)
    uint64_t* out_loc;         // (pid << 32) | pos
    uint64_t capacity;
    uint64_t* d_count;         // device u64[2]: [0] tuples kept by this launch (may exceed capacity: nothing is written
                               // past it); [1] high word != 0: a zero hash was met on the exact path
    PairScatter scatter{};     // scatter.out_key != nullptr: the tuples leave the kernel partitioned by the top bits of the
                               // hash (first level of an unstable partition, dense_scatter.cuh) instead of in (protein,
                               // pos) order; out_hash / out_loc / capacity are not used, d_count[0] still gets the total
    uint32_t* t_abund = nullptr;  // scatter mode with scaled > 1: kept windows per protein are counted here (device, n_prot,
                                  // zeroed by the caller): there is no (protein, pos)-ordered tuple array to count them from
    int force_general;         // 1: take the look-back path even when scaled == 1
    uint32_t tile_begin = 0, tile_end = 0;  // exact path: launch_sketch_tiles covers [tile_begin, tile_end); 0,0 = all
    int unordered = 0;         // the output does not need the tiles' exact bases (scatter modes set it: the tiles add their
                               // totals to d_count[0] instead, and launch_sketch_prepare skips the count + scan launches)
    int count_zeroed = 0;      // the caller has zeroed d_count[0..1] on the stream already
    void* workspace;           // sketch_workspace_bytes(n_res)
};

// Dense k-mer space path (hp, DENSE_MIN_K <= k <= DENSE_MAX_K, scaled == 1): see sketch_dense_kernel.
constexpr int DENSE_MIN_K = 8;
constexpr int DENSE_MAX_K = 24;
constexpr int DENSE_PREFIX_BITS = 16;  // a pattern's code starts with the top 16 bits of its hash
// Order-preserving code of a pattern (per-handle table, dense.cu): with p = the top DENSE_PREFIX_BITS bits of the pattern's
// hash and l = the pattern's rank among the patterns that share p,
//     code = p << rb | (2 l + 1)
// Codes sort like the hashes, and a code's top bits ARE its hash's top bits, so a bucket of the key sort is a hash-prefix
// range (the directory the search uses is over hash prefixes).  A window with a residue of neither class has no pattern:
// it is hashed from its bytes and gets the EVEN code p << rb | 2 x (patterns of its prefix group below its hash), which
// sorts it between the right two patterns (or onto a pattern with the very same hash: then the odd code).
// When code | protein | position would not fit 64 bits with the parity bit but does without it (parity == 0), codes are
// p << rb | l and a window without a pattern makes the batch take the general path (handle_exceptions must be 0).
struct DenseSketchArgs {
    const uint32_t* code_of_pattern;  // device, 2^k entries
    const uint64_t* sorted_hash;      // device, 2^k entries: the patterns' hashes in increasing order
    const uint32_t* group_base;       // device, 2^16 + 1 entries: first entry of sorted_hash of every prefix group
    int rb;                           // bits of a code below the prefix (the parity bit included)
    int parity;                       // 1: the lowest code bit tells patterns (1) from exception keys (0)
    uint64_t* out_keys;               // device, capacity entries: code << (pid_bits + pos_bits) | protein << pos_bits | position
    int pid_bits, pos_bits;
    int handle_exceptions;         // 0: such a window only raises exception_flag[0] (the caller takes the general path)
    uint32_t* exception_flag;      // device u32[2]: [0] unhandled exception / zero hash, [1] exception keys were emitted
    DenseScatter scatter;          // scatter.out != nullptr: the keys leave the kernel partitioned by their top bits
                                   // (first level of the key sort, dense_scatter.cuh) instead of in tile order
};
// launch_sketch_prepare first (exact path: scaled == 1); then this instead of launch_sketch_tiles.
cudaError_t launch_sketch_dense(const SketchArgs& a, const DenseSketchArgs& d, cudaStream_t stream, uint64_t* n_launches);

size_t sketch_workspace_bytes(uint64_t n_res);
// Enqueues memset + tile->protein map + the fused kernel on `stream`; adds the number of kernels launched.
cudaError_t launch_sketch(const SketchArgs& a, cudaStream_t stream, uint64_t* n_launches);
// The same in three steps, so that the host can stream the residues in while earlier tiles are hashed:
// prepare needs only the offsets; tiles [tile_begin, tile_end) need the residues up to tile_end * SK_TILE + k.
cudaError_t launch_sketch_prepare(const SketchArgs& a, cudaStream_t stream, uint64_t* n_launches);
cudaError_t launch_sketch_tiles(const SketchArgs& a, cudaStream_t stream, uint64_t* n_launches);
cudaError_t launch_sketch_finish(const SketchArgs& a, cudaStream_t stream);
void fill_lut(int moltype, Lut256* lut);
// 5-bit residue codes for the packed upload format: 'A'..'Z' -> 1..26, '*' -> 27, 0 = padding.  Returns false (and
// leaves `out` unspecified) when a byte has no code.  out must hold packed_bytes(n) bytes.
bool pack_residues(const uint8_t* res, uint64_t n, uint8_t* out);
inline uint64_t packed_bytes(uint64_t n) { return (n + 7) / 8 * 5 + 72; }

}  // namespace ks
