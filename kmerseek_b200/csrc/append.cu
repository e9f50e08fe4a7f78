// Append stage (append.cuh): A (finalized index) + B (index of one batch, protein ids above A's) -> compact C.
#include <cub/cub.cuh>

#include "append.cuh"

namespace ks {

namespace {

constexpr int MT = 256;                    // threads of a merge CTA
constexpr int MI = 8;                      // outputs per thread and tile
constexpr uint64_t TILE = (uint64_t)MT * MI;
constexpr unsigned MAX_GRID = 148 * 16;

inline size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }
inline unsigned grid_for(uint64_t n, uint64_t per) {
    const uint64_t g = (n + per - 1) / per;
    return (unsigned)std::max<uint64_t>(1, std::min<uint64_t>(g, MAX_GRID));
}

// ---- segmented -> compact ---------------------------------------------------------------------------------------------
// One CTA: exclusive scans of the keys and groups per sort bucket.  seg_counts[b] = keys | groups << 32, and both totals
// are below 2^31, so the packed words add up without a carry between the halves.
__global__ void __launch_bounds__(1024) seg_prefix_kernel(const uint64_t* __restrict__ seg_counts, uint32_t nb,
                                                          uint32_t* __restrict__ kpre, uint32_t* __restrict__ gpre) {
    __shared__ uint64_t s_w[32];
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t per = (nb + blockDim.x - 1) / blockDim.x;
    const uint32_t b0 = min(tid * per, nb), b1 = min(b0 + per, nb);
    uint64_t sum = 0;
    for (uint32_t b = b0; b < b1; b++) sum += seg_counts[b];
    uint64_t v = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint64_t t = __shfl_up_sync(0xffffffffu, v, o);
        if ((int)lane >= o) v += t;
    }
    if (lane == 31) s_w[warp] = v;
    __syncthreads();
    if (warp == 0) {
        uint64_t w = lane < (blockDim.x >> 5) ? s_w[lane] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint64_t t = __shfl_up_sync(0xffffffffu, w, o);
            if ((int)lane >= o) w += t;
        }
        s_w[lane] = w;
    }
    __syncthreads();
    uint64_t excl = v - sum + (warp ? s_w[warp - 1] : 0);
    for (uint32_t b = b0; b < b1; b++) {
        kpre[b] = (uint32_t)excl;
        gpre[b] = (uint32_t)(excl >> 32);
        excl += seg_counts[b];
    }
}

// One CTA per sort bucket: its keys at seg_start[b] + b + i go to kpre[b] + i, its groups (same base) to gpre[b] + i.
__global__ void __launch_bounds__(256) seg_compact_kernel(CsrView v, const uint32_t* __restrict__ kpre,
                                                          const uint32_t* __restrict__ gpre, uint64_t U, uint64_t G,
                                                          uint64_t* __restrict__ keys, uint32_t* __restrict__ key_grp,
                                                          uint32_t* __restrict__ grp_start, uint64_t* __restrict__ counts) {
    const uint32_t b = blockIdx.x;
    const uint32_t kb = v.seg_start[b] + b;
    const uint64_t c = v.seg_counts[b];
    const uint32_t tk = (uint32_t)c, tg = (uint32_t)(c >> 32), ko = kpre[b], go = gpre[b];
    for (uint32_t i = threadIdx.x; i < tk; i += blockDim.x) {
        keys[ko + i] = v.keys[kb + i];
        key_grp[ko + i] = v.key_grp[kb + i] - kb + go;
    }
    for (uint32_t i = threadIdx.x; i < tg; i += blockDim.x) grp_start[go + i] = v.grp_start[kb + i];
    if (b == 0 && threadIdx.x == 0) {
        key_grp[U] = (uint32_t)G;
        grp_start[G] = (uint32_t)v.n;
        counts[0] = U;
        counts[1] = G;
    }
}

// ---- merge --------------------------------------------------------------------------------------------------------------
// Per B key j (and j = U_B, the end): the insertion key `ins` in A, the matched flag, the first group and posting of the
// key's block in C (gstart / tstart) and B's own first group and posting (bg / bt).
struct Work {
    uint32_t *ins, *matched, *mx, *gstart, *tstart, *bg, *bt;
    void* scan_temp;
    size_t scan_bytes;
};

Work carve(void* p, uint64_t u_b, size_t scan_bytes) {
    char* w = (char*)p;
    const size_t arr = align256((u_b + 1) * 4);
    Work k;
    uint32_t** a[7] = {&k.ins, &k.matched, &k.mx, &k.gstart, &k.tstart, &k.bg, &k.bt};
    for (int i = 0; i < 7; i++) *a[i] = (uint32_t*)(w + i * arr);
    k.scan_temp = w + 7 * arr;
    k.scan_bytes = scan_bytes;
    return k;
}

size_t scan_temp_bytes(uint64_t u_b) {
    size_t bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, bytes, (const uint32_t*)nullptr, (uint32_t*)nullptr, (int64_t)(u_b + 1));
    return align256(bytes);
}

__global__ void __launch_bounds__(256) locate_kernel(MergeSide A, MergeSide B, const uint32_t* __restrict__ dir,
                                                     int dir_bits, int dir_shift, Work w) {
    const uint64_t j = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (j > B.U) return;
    uint32_t ins = (uint32_t)A.U, m = 0, ins_g = (uint32_t)A.G, ins_p = (uint32_t)A.n, bg = (uint32_t)B.G, bt = (uint32_t)B.n;
    if (j < B.U) {
        const uint64_t h = B.keys[j];
        uint32_t lo = 0, hi = (uint32_t)A.U;
        if (A.U) {
            const uint64_t x = h >> dir_shift;
            if (x < (1ull << dir_bits)) { lo = dir[x]; hi = dir[x + 1]; } else lo = hi;
        }
        while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if (A.keys[mid] < h) lo = mid + 1; else hi = mid;
        }
        ins = lo;
        m = (lo < A.U && A.keys[lo] == h) ? 1u : 0u;
        // matched: behind A's groups of the key; else in front of the next key's
        ins_g = lo + m < A.U ? A.key_grp[lo + m] : (uint32_t)A.G;
        ins_p = ins_g < A.G ? A.grp_start[ins_g] : (uint32_t)A.n;
        bg = B.key_grp[j];
        bt = B.grp_start[bg];
    }
    w.ins[j] = ins;
    w.matched[j] = m;
    w.gstart[j] = ins_g + bg;
    w.tstart[j] = ins_p + bt;
    w.bg[j] = bg;
    w.bt[j] = bt;
}

// Number of j in [0, U_B] whose block starts at or before output o, known to lie in [lo, hi].
template <class S>
__device__ __forceinline__ uint32_t count_le(const S& s, uint64_t o, uint32_t lo, uint32_t hi) {
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (s(mid) <= o) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// Tiles of TILE consecutive outputs [0, total): two threads bound the tile's insertion points with a search over all of
// them, then every output searches that range only and calls f(o, c), c = number of B blocks starting at or before o.
template <class S, class F>
__device__ __forceinline__ void merge_tiles(const S& s, uint32_t n_blocks, uint64_t total, const F& f) {
    __shared__ uint32_t s_rng[2];
    for (uint64_t o0 = blockIdx.x * TILE; o0 < total; o0 += (uint64_t)gridDim.x * TILE) {
        const uint64_t o_last = min(o0 + TILE, total) - 1;
        if (threadIdx.x < 2) s_rng[threadIdx.x] = count_le(s, threadIdx.x ? o_last : o0, 0u, n_blocks);
        __syncthreads();
        const uint32_t lo = s_rng[0], hi = s_rng[1];
        __syncthreads();
#pragma unroll
        for (int r = 0; r < MI; r++) {
            const uint64_t o = o0 + (uint64_t)r * MT + threadIdx.x;
            if (o <= o_last) f(o, count_le(s, o, lo, hi));
        }
    }
}

// keys and key_grp.  B key j starts at ins + j - mx[j] (unmatched keys before it); a matched key inserts nothing.
__global__ void __launch_bounds__(MT) merge_keys_kernel(MergeSide A, MergeSide B, Work w, uint64_t* __restrict__ keys,
                                                        uint32_t* __restrict__ key_grp, uint64_t* __restrict__ d_counts) {
    const uint32_t nb = (uint32_t)B.U + 1;
    const uint64_t M = w.mx[B.U];
    const uint64_t U = A.U + B.U - M, G = A.G + B.G;
    if (blockIdx.x == 0 && threadIdx.x == 0) { d_counts[0] = U; d_counts[1] = G; d_counts[2] = M; }
    auto s = [&](uint32_t j) -> uint64_t { return (uint64_t)w.ins[j] + j - w.mx[j]; };
    merge_tiles(s, nb, U + 1, [&](uint64_t o, uint32_t c) {
        if (o == U) { key_grp[o] = (uint32_t)G; return; }
        const bool at = c && o == s(c - 1);                  // B's key c - 1 starts here
        const bool mt = c && w.mx[c] != w.mx[c - 1];         // ... and it is a matched key (it inserts no key)
        if (at && !mt) {                                     // B's key c - 1
            keys[o] = B.keys[c - 1];
            key_grp[o] = w.gstart[c - 1];
        } else {  // A's key a: B's unmatched keys before it moved it up; a matched B key at a puts its groups behind a's
            const uint64_t a = o - (c - w.mx[c]);
            keys[o] = A.keys[a];
            key_grp[o] = A.key_grp[a] + w.bg[c - (at ? 1 : 0)];
        }
    });
}

// grp_start: B's groups of key j start at gstart[j]; A's groups move up by B's groups before them, their postings by
// B's postings before them.
__global__ void __launch_bounds__(MT) merge_groups_kernel(MergeSide A, MergeSide B, Work w, uint32_t* __restrict__ grp_start) {
    const uint64_t G = A.G + B.G;
    auto s = [&](uint32_t j) -> uint64_t { return w.gstart[j]; };
    merge_tiles(s, (uint32_t)B.U + 1, G + 1, [&](uint64_t o, uint32_t c) {
        if (o == G) { grp_start[o] = (uint32_t)(A.n + B.n); return; }
        if (c && o - w.gstart[c - 1] < w.bg[c] - w.bg[c - 1]) {
            const uint64_t gb = w.bg[c - 1] + (o - w.gstart[c - 1]);
            grp_start[o] = (w.tstart[c - 1] - w.bt[c - 1]) + B.grp_start[gb];
        } else {
            grp_start[o] = A.grp_start[o - w.bg[c]] + w.bt[c];
        }
    });
}

// loc: the bulk of the bytes.  B's postings get A's protein count added to their protein ids.
__global__ void __launch_bounds__(MT) merge_loc_kernel(MergeSide A, MergeSide B, Work w, uint32_t p_a, uint64_t* __restrict__ loc) {
    auto s = [&](uint32_t j) -> uint64_t { return w.tstart[j]; };
    const uint64_t pid_add = (uint64_t)p_a << 32;
    merge_tiles(s, (uint32_t)B.U + 1, A.n + B.n, [&](uint64_t o, uint32_t c) {
        if (c && o - w.tstart[c - 1] < w.bt[c] - w.bt[c - 1]) loc[o] = B.loc[w.bt[c - 1] + (o - w.tstart[c - 1])] + pid_add;
        else loc[o] = A.loc[o - w.bt[c]];
    });
}

}  // namespace

cudaError_t launch_compact_segmented(const CsrView& v, uint64_t U, uint64_t G, uint32_t* pre, uint64_t* keys,
                                     uint32_t* key_grp, uint32_t* grp_start, uint64_t* counts, cudaStream_t stream,
                                     uint64_t* n_launches) {
    if (v.seg_nb == 0) return cudaErrorInvalidValue;
    seg_prefix_kernel<<<1, 1024, 0, stream>>>(v.seg_counts, v.seg_nb, pre, pre + v.seg_nb);
    seg_compact_kernel<<<v.seg_nb, 256, 0, stream>>>(v, pre, pre + v.seg_nb, U, G, keys, key_grp, grp_start, counts);
    if (n_launches) *n_launches += 2;
    return cudaGetLastError();
}

size_t append_work_bytes(uint64_t u_b) { return 7 * align256((u_b + 1) * 4) + scan_temp_bytes(u_b); }

cudaError_t launch_append_merge(const AppendArgs& m, cudaStream_t stream, uint64_t* n_launches) {
    const uint64_t nb = m.b.U + 1;
    const size_t scan_bytes = scan_temp_bytes(m.b.U);
    if (m.work_bytes < append_work_bytes(m.b.U)) return cudaErrorInvalidValue;
    const Work w = carve(m.work, m.b.U, scan_bytes);
    locate_kernel<<<(unsigned)((nb + 255) / 256), 256, 0, stream>>>(m.a, m.b, m.dir_a, m.dir_bits_a, m.dir_shift_a, w);
    size_t tb = scan_bytes;
    cudaError_t e = cub::DeviceScan::ExclusiveSum(w.scan_temp, tb, w.matched, w.mx, (int64_t)nb, stream);
    if (e != cudaSuccess) return e;
    merge_keys_kernel<<<grid_for(m.a.U + m.b.U + 1, TILE), MT, 0, stream>>>(m.a, m.b, w, m.keys, m.key_grp, m.d_counts);
    merge_groups_kernel<<<grid_for(m.a.G + m.b.G + 1, TILE), MT, 0, stream>>>(m.a, m.b, w, m.grp_start);
    merge_loc_kernel<<<grid_for(m.a.n + m.b.n, TILE), MT, 0, stream>>>(m.a, m.b, w, m.p_a, m.loc);
    if (n_launches) *n_launches += 5;
    return cudaGetLastError();
}

}  // namespace ks
