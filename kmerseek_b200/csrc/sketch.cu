// Sketch stage for sm_100a.
//
// For every k-mer window of every protein of the resident batch:
//   reduced-alphabet translation (256-entry LUT in shared memory)        -- src/rust/encoding.rs:43-53
//   MurmurHash3_x64_128(translated k-mer, seed 42), low word            -- sourmash::_hash_murmur, src/rust/index.rs:766
//   FracMinHash filter  h != 0 && h <= max_hash                          -- KmerMinHash::add_protein, src/rust/signature.rs:273-274
//   output of the surviving (hash, protein, pos) tuples                  -- process_kmers, src/rust/index.rs:749-786
// (paths relative to the reference repository).  Data layout and roofline: DESIGN.md section 3.
//
// Three kernels: sketch_quad_kernel (k <= 32: every lane hashes 4 consecutive windows), sketch_dense_kernel (hp,
// 8 <= k <= 24: a window's hash is a table entry and its tuple one 64-bit key) and sketch_kernel (k > 32: a byte loop per
// window).  All three cut the residue stream into tiles of SK_TILE window starts, one tile per CTA, and are built from
// the same parts: the tile's residues staged once, translated, in shared memory (stage_residues); the offsets of the
// proteins that intersect the tile (cache_offsets) and every lane's forward walk over them (first_protein,
// seek_protein); and the ordered output (warp_prefix, exact_base / lookback_base, write_warp).
//
// Ordered output is in (protein, pos) order, independent of scheduling, so the later stable sort by hash is
// deterministic: each row of windows is ranked with ballots into a per-warp staging area in shared memory, and every
// warp streams its staged entries to their final position with coalesced stores.  The tile's base is known up front on
// the exact path (scaled == 1: tile_count_kernel + scan, no cross-CTA dependency); otherwise CTAs take tiles by ticket
// (a tile's predecessors have always started) and chain the tile totals with a single-pass decoupled look-back.
// Unordered output (the quad kernel's SCATTER, the dense kernel's scatter) keeps the keys in registers and hands them
// straight to the first level of the partition (dense_scatter.cuh): no ranking and no staging in window order.
#include <cub/device/device_scan.cuh>

#include <cstring>
#include <type_traits>

#include "common.cuh"
#include "sketch.cuh"

namespace ks {

namespace {

constexpr int OFFS_CACHE = 256;  // offsets of the proteins that intersect a tile, cached in smem when they fit

struct Workspace {
    uint32_t* ticket;      // [0] tile ticket, [1] zero-hash flag (exact path)
    uint64_t* status;      // look-back words, one per tile
    uint32_t* tile_pid;    // [nt + 1]
    uint64_t* tile_cnt;    // [nt + 1] valid windows per tile (exact path)
    uint64_t* tile_base;   // [nt + 1] exclusive scan of tile_cnt
    void* scan_temp;
    size_t scan_temp_bytes;
};

__host__ __device__ inline uint64_t n_tiles_of(uint64_t n_res) { return (n_res + SK_TILE - 1) / SK_TILE; }

inline size_t scan_temp_bytes_for(uint64_t n) {
    size_t bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, bytes, (const uint64_t*)nullptr, (uint64_t*)nullptr, (int64_t)n);
    return (bytes + 255) & ~(size_t)255;
}

__host__ inline Workspace carve(void* ws, uint64_t n_res) {
    uint64_t nt = n_tiles_of(n_res);
    char* p = (char*)ws;
    Workspace w;
    w.ticket = (uint32_t*)p;
    w.status = (uint64_t*)(p + 16);
    w.tile_pid = (uint32_t*)(p + 16 + nt * 8);
    size_t off = (16 + nt * 8 + (nt + 1) * 4 + 15) & ~(size_t)15;
    w.tile_cnt = (uint64_t*)(p + off);
    w.tile_base = w.tile_cnt + nt + 1;
    off += 2 * (nt + 1) * 8;
    w.scan_temp = p + off;
    w.scan_temp_bytes = scan_temp_bytes_for(nt + 1);
    return w;
}

// tile_pid[t] = index of the protein that contains residue t*SK_TILE (last p with offsets[p] <= that
// position, clipped to n_prot-1); one entry past the last tile bounds the last tile's protein range.
// One thread per protein: a non-empty protein [a, b) owns the tile starts inside it (most own none or one), so the map
// costs two coalesced reads per protein instead of a 20-step binary search per tile (9 us on a 12 M-residue shard).
__global__ void tile_pid_kernel(const uint64_t* __restrict__ offsets, uint64_t n_prot, uint64_t n_tiles,
                                uint32_t* __restrict__ tile_pid) {
    const uint64_t p = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (p >= n_prot) return;
    const uint64_t a = offsets[p], b = offsets[p + 1];
    for (uint64_t t = (a + SK_TILE - 1) / SK_TILE; t <= n_tiles && t * SK_TILE < b; t++) tile_pid[t] = (uint32_t)p;
    if (p == n_prot - 1)  // tile starts at or past the last residue (the bounding entry; n_tiles * SK_TILE >= n_res)
        for (uint64_t t = (b + SK_TILE - 1) / SK_TILE; t <= n_tiles; t++) tile_pid[t] = (uint32_t)p;
}

// Exact path (scaled == 1): the number of tuples a tile emits is its number of valid windows, known from the
// offsets alone (a hash of exactly 0 is the one exception, flagged by the kernel and redone on the general path).
__global__ void tile_count_kernel(const uint64_t* __restrict__ offsets, uint64_t n_res, uint32_t k, uint64_t n_tiles,
                                  const uint32_t* __restrict__ tile_pid, uint64_t* __restrict__ tile_cnt) {
    uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (t > n_tiles) return;
    if (t == n_tiles) { tile_cnt[t] = 0; return; }
    const uint64_t g0 = t * SK_TILE, g1 = g0 + SK_TILE;
    uint64_t c = 0;
    for (uint32_t p = tile_pid[t]; p <= tile_pid[t + 1]; p++) {
        const uint64_t a = offsets[p], b = offsets[p + 1];
        if (b - a < k) continue;
        const uint64_t lo = a > g0 ? a : g0;              // window starts of p inside the tile: [lo, hi)
        const uint64_t last = b - k + 1;                  // one past the last window start of p
        const uint64_t hi = last < g1 ? last : g1;
        if (hi > lo) c += hi - lo;
    }
    tile_cnt[t] = c;
}

// ---------------------------------------------------------------------------------------------
// Parts shared by the kernels
// ---------------------------------------------------------------------------------------------
constexpr int WARP_SLOTS = SK_TILE / (SK_THREADS / 32);  // staging slots per warp (256): one per window of the warp

// Entry c of the code table of the packed residue format (pack_residues: 'A'..'Z' -> 1..26, '*' -> 27), translated.
__device__ __forceinline__ uint8_t lut32_entry(const uint8_t* lut, uint32_t c) {
    return c == 0 ? 0 : c <= 26 ? lut['A' + c - 1] : c == 27 ? lut['*'] : 0;
}

// Residues [g0, g0 + n) of the batch into s_res as translated bytes (n + 15 bytes of room).  Packed residues: thread t
// unpacks the 5-bit groups t, t + SK_THREADS, ... (8 residues = 5 bytes) through s_lut32, which the caller has filled.
// Plain residues: coalesced 16-byte loads, translated through s_lut when TRANSLATE, 16-byte shared stores (n <= 16 *
// SK_THREADS).  Groups and chunks that start past the batch are not backed by memory and stage zeros.  The caller puts a
// barrier between this and the first read of s_res.
template <bool TRANSLATE>
__device__ __forceinline__ void stage_residues(uint32_t tid, uint32_t* s_res, const SketchArgs& a, bool packed, uint64_t g0,
                                               uint32_t n, const uint8_t* s_lut, const uint8_t* s_lut32) {
    if (packed) {
        const uint32_t n_groups = (n + 7) / 8;
        for (uint32_t grp = tid; grp < n_groups; grp += SK_THREADS) {
            const uint64_t group = g0 / 8 + grp;
            const uint64_t byte = group * 5;
            uint32_t w0 = 0, w1 = 0;
            if (group * 8 < a.n_res) {
                const uint32_t* w = reinterpret_cast<const uint32_t*>(a.residues + (byte & ~3ull));
                w0 = __ldg(w);
                w1 = __ldg(w + 1);
            }
            const uint32_t sh8 = (uint32_t)(byte & 3) * 8;
            const uint32_t lo = __funnelshift_r(w0, w1, sh8), hi = (w1 >> sh8) & 0xffu;  // 40 bits: lo | hi << 32
            uint32_t o0 = 0, o1 = 0;
#pragma unroll
            for (int i = 0; i < 4; i++) o0 |= (uint32_t)s_lut32[(lo >> (5 * i)) & 31u] << (8 * i);
            o1 |= (uint32_t)s_lut32[(lo >> 20) & 31u];
            o1 |= (uint32_t)s_lut32[(lo >> 25) & 31u] << 8;
            o1 |= (uint32_t)s_lut32[((lo >> 30) | (hi << 2)) & 31u] << 16;
            o1 |= (uint32_t)s_lut32[(hi >> 3) & 31u] << 24;
            s_res[2 * grp] = o0;
            s_res[2 * grp + 1] = o1;
        }
    } else {
        const uint32_t n_chunks = (n + 15) / 16;
        if (tid < n_chunks) {
            const uint64_t g = g0 + 16ull * tid;
            uint4 v = make_uint4(0, 0, 0, 0);
            if (g < a.n_res) v = __ldg(reinterpret_cast<const uint4*>(a.residues + g));
            if (TRANSLATE) {
                uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    const uint32_t x = w[i];
                    w[i] = (uint32_t)s_lut[x & 0xff] | ((uint32_t)s_lut[(x >> 8) & 0xff] << 8) |
                           ((uint32_t)s_lut[(x >> 16) & 0xff] << 16) | ((uint32_t)s_lut[x >> 24] << 24);
                }
                v = make_uint4(w[0], w[1], w[2], w[3]);
            }
            reinterpret_cast<uint4*>(s_res)[tid] = v;
        }
    }
}

// The proteins that intersect a tile are [p_lo, p_hi] = tile_pid[tile], tile_pid[tile + 1].  Caches their offsets,
// offsets[p_lo .. p_hi + 1], in s_offs when they fit; returns whether they do.  A barrier must follow before the first
// lookup.
__device__ __forceinline__ bool cache_offsets(uint32_t tid, const SketchArgs& a, uint64_t* s_offs, uint32_t p_lo, uint32_t p_hi) {
    const uint32_t n_off = p_hi - p_lo + 2;
    const bool cached = n_off <= OFFS_CACHE;
    if (cached)
        for (uint32_t i = tid; i < n_off; i += SK_THREADS) s_offs[i] = a.offsets[p_lo + i];
    return cached;
}

// Residues from the tile start g0 on, clamped (window w of the tile exists iff w < the result).
__device__ __forceinline__ uint32_t tile_residues(const SketchArgs& a, uint64_t g0) {
    const uint64_t left = a.n_res - g0;
    return left > 0x40000000ull ? 0x40000000u : (uint32_t)left;
}

// A lane's walk over the proteins of its tile.  Windows are named by their start w relative to the tile start g0, and
// a lane's windows only move forward.  The state is the lane's protein p, its start as the low 32 bits of the absolute
// position (positions within a protein fit 32 bits) and its end relative to the tile start, clamped so that 32-bit
// compares suffice (end_rel).  offs: offsets[], from the shared-memory cache when the tile's slice is there.
__device__ __forceinline__ uint32_t end_rel(uint64_t o, uint64_t g0) {
    const uint64_t d = o - g0;
    return d > 0x7fffffffull ? 0x7fffffffu : (uint32_t)d;
}
// the protein of window w (which exists): binary search over the tile's proteins [p_lo, p_hi]
__device__ __forceinline__ void first_protein(const uint64_t* offs, uint64_t g0, uint32_t p_lo, uint32_t p_hi, uint32_t w,
                                              uint32_t& p, uint32_t& pstart_lo, uint32_t& pend_rel) {
    const uint64_t g = g0 + w;
    uint32_t lo = p_lo, hi = p_hi;
    while (lo < hi) {
        const uint32_t mid = (lo + hi + 1) >> 1;
        if (offs[mid] <= g) lo = mid; else hi = mid - 1;
    }
    p = lo;
    pstart_lo = (uint32_t)offs[p];
    pend_rel = end_rel(offs[p + 1], g0);
}
// forward to the protein of window w (which exists and is not before the lane's current window)
__device__ __forceinline__ void seek_protein(const uint64_t* offs, uint64_t g0, uint32_t w, uint32_t& p, uint32_t& pstart_lo,
                                             uint32_t& pend_rel) {
    while (w >= pend_rel) { p++; pstart_lo = (uint32_t)offs[p]; pend_rel = end_rel(offs[p + 1], g0); }
}

// Ordered output, after every warp has staged its wcount entries: the warps' prefix over the staged counts (contains a
// barrier).  wprefix = entries of the warps before this one, btotal = entries of the tile.
struct WarpPrefix { uint32_t wprefix, btotal; };
__device__ __forceinline__ WarpPrefix warp_prefix(uint32_t tid, uint32_t* s_wtot, uint32_t wcount) {
    const uint32_t lane = tid & 31, warp = tid >> 5;
    if (lane == 0) s_wtot[warp] = wcount;
    __syncthreads();
    WarpPrefix r{0, 0};
#pragma unroll
    for (int i = 0; i < SK_THREADS / 32; i++) {
        const uint32_t t = s_wtot[i];
        if (i < (int)warp) r.wprefix += t;
        r.btotal += t;
    }
    return r;
}

// Output position of the tile's first entry, exact path: the tile's base from tile_count_kernel + scan.  The last tile
// sets d_count[0].
__device__ __forceinline__ uint64_t exact_base(uint32_t tid, const SketchArgs& a, uint32_t tile, const uint64_t* tile_base,
                                               uint32_t btotal) {
    const uint64_t base = tile_base[tile];
    if (tid == 0 && tile == n_tiles_of(a.n_res) - 1) *a.d_count = base + btotal;
    return base;
}

// The same on the look-back path: warp 0 chains the tile's total behind its predecessors' (contains a barrier).
__device__ __forceinline__ uint64_t lookback_base(uint32_t lane, uint32_t warp, const SketchArgs& a, uint32_t tile,
                                                  uint64_t* status, uint32_t btotal, uint64_t& s_base) {
    if (warp == 0) {
        const uint64_t excl = scan_lookback(status, tile, btotal);
        if (lane == 0) {
            s_base = excl;
            if (tile == n_tiles_of(a.n_res) - 1) *a.d_count = excl + btotal;
        }
    }
    __syncthreads();
    return s_base;
}

// A warp's share of the ordered output: its staged entries 0 .. wcount - 1 go to output positions base + i.  Positions
// at or past a.capacity are not written (the caller sees the full count in d_count and retries with room).  put(i)
// writes entry i.
template <class Put>
__device__ __forceinline__ void write_warp(uint32_t lane, const SketchArgs& a, uint64_t base, uint32_t wcount, Put put) {
    if (base + wcount <= a.capacity) {  // the usual case: the warp's 256 slots, 8 per lane, no per-element bound check
#pragma unroll
        for (uint32_t i0 = 0; i0 < WARP_SLOTS; i0 += 32) {
            const uint32_t i = i0 + lane;
            if (i0 >= wcount) break;  // uniform
            if (i < wcount) put(i);
        }
    } else {
        for (uint32_t i = lane; i < wcount; i += 32)
            if (base + i < a.capacity) put(i);
    }
}

// ---------------------------------------------------------------------------------------------
// Byte-loop kernel (k > 32): lane l of row r owns window (warp * SK_ROWS + r) * 32 + l and hashes its k bytes straight
// from shared memory; a row is compacted with one ballot (lanes write consecutive slots).  Ordered output on the
// look-back path only (exact_path and the scatter route take k <= 32).
// ---------------------------------------------------------------------------------------------
template <bool TRANSLATE>
__global__ void __launch_bounds__(SK_THREADS)
sketch_kernel(SketchArgs a, Lut256 lut, uint32_t* __restrict__ ticket, uint64_t* __restrict__ status,
              const uint32_t* __restrict__ tile_pid) {
    constexpr int RES_WORDS = (SK_TILE + SK_MAX_K + 16 + 3) / 4;
    __shared__ __align__(16) uint32_t s_res[RES_WORDS];
    __shared__ __align__(16) uint64_t s_hash[SK_TILE];
    __shared__ __align__(16) uint64_t s_loc[SK_TILE];
    __shared__ uint64_t s_offs[OFFS_CACHE];
    __shared__ uint8_t s_lut[256];
    __shared__ uint32_t s_wtot[SK_THREADS / 32];
    __shared__ uint32_t s_tile;
    __shared__ uint64_t s_base;

    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t k = a.k;

    if (tid == 0) s_tile = atomicAdd(ticket, 1u);
    if (TRANSLATE) s_lut[tid] = lut.b[tid];
    __syncthreads();
    const uint32_t tile = s_tile;
    const uint64_t g0 = (uint64_t)tile * SK_TILE;
    const uint32_t p_lo = tile_pid[tile], p_hi = tile_pid[tile + 1];
    const bool cached = cache_offsets(tid, a, s_offs, p_lo, p_hi);
    stage_residues<TRANSLATE>(tid, s_res, a, false, g0, SK_TILE + k - 1, s_lut, nullptr);  // (k > 32 is never uploaded packed)
    __syncthreads();

    const uint64_t* offs = cached ? (const uint64_t*)s_offs - p_lo : a.offsets;
    const uint32_t nres_rel = tile_residues(a, g0), g0_lo = (uint32_t)g0;
    const uint32_t w0 = warp * WARP_SLOTS + lane;  // the lane's window in row 0
    uint32_t p = p_lo, pstart_lo = 0, pend_rel = 0;
    if (w0 < nres_rel) first_protein(offs, g0, p_lo, p_hi, w0, p, pstart_lo, pend_rel);

    uint32_t wcount = 0;  // tuples staged by this warp so far (uniform across the warp)
#pragma unroll
    for (int r = 0; r < SK_ROWS; r++) {
        const uint32_t w = w0 + r * 32;
        bool valid = false;
        if (w < nres_rel) {
            seek_protein(offs, g0, w, p, pstart_lo, pend_rel);
            valid = w + k <= pend_rel;
        }
        const uint64_t h = valid ? murmur_bytes(reinterpret_cast<const uint8_t*>(s_res) + w, k) : 0;
        const bool keep = valid && h != 0 && h <= a.max_hash;
        const uint32_t bal = __ballot_sync(0xffffffffu, keep);
        if (keep) {
            const uint32_t slot = warp * WARP_SLOTS + wcount + __popc(bal & ((1u << lane) - 1u));
            s_hash[slot] = h;
            s_loc[slot] = ((uint64_t)(a.pid_base + p) << 32) | (uint64_t)(g0_lo + w - pstart_lo);
        }
        wcount += __popc(bal);
    }

    const WarpPrefix wp = warp_prefix(tid, s_wtot, wcount);
    const uint64_t base = lookback_base(lane, warp, a, tile, status, wp.btotal, s_base) + wp.wprefix;
    const uint32_t sbase = warp * WARP_SLOTS;
    write_warp(lane, a, base, wcount, [&](uint32_t i) {
        a.out_hash[base + i] = s_hash[sbase + i];
        a.out_loc[base + i] = s_loc[sbase + i];
    });
}

// ---------------------------------------------------------------------------------------------
// Fast path (k <= 32): every lane owns 4 consecutive windows ("a quad").
//
// The 4 + k - 1 bytes of a quad are 4-byte aligned in shared memory, so they are fetched once as whole words
// and each window is cut out with constant funnel shifts.  MurmurHash3 runs on explicit 32-bit limbs so that a
// 64-bit multiply by a constant is three IMADs and a 64-bit rotate two SHFs (left to the compiler, the same
// arithmetic took about twice the instructions, and the kernel is issue-bound before it is HBM-bound).
// Positions are tile-relative 32-bit values.  Ordered output stages kept tuples in shared memory at their ordered
// slot; the slot -> address map interleaves the four windows of a quad over four segments so that both the quad
// writes and the linear read-out are bank-conflict free.
// ---------------------------------------------------------------------------------------------
struct L64 { uint32_t lo, hi; };

__device__ __forceinline__ L64 mul_c(L64 a, uint64_t c) {
    const uint32_t clo = (uint32_t)c, chi = (uint32_t)(c >> 32);
    uint32_t t = a.lo * chi;
    t = a.hi * clo + t;
    const uint64_t p = (uint64_t)a.lo * clo + ((uint64_t)t << 32);
    return {(uint32_t)p, (uint32_t)(p >> 32)};
}
__device__ __forceinline__ L64 rotl_c(L64 a, int r) {  // 0 < r < 64, r != 32
    if (r < 32) return {__funnelshift_l(a.hi, a.lo, r), __funnelshift_l(a.lo, a.hi, r)};
    return {__funnelshift_l(a.lo, a.hi, r - 32), __funnelshift_l(a.hi, a.lo, r - 32)};
}
__device__ __forceinline__ L64 xor_(L64 a, L64 b) { return {a.lo ^ b.lo, a.hi ^ b.hi}; }
__device__ __forceinline__ L64 add_(L64 a, L64 b) {
    const uint64_t s = (((uint64_t)a.hi << 32) | a.lo) + (((uint64_t)b.hi << 32) | b.lo);
    return {(uint32_t)s, (uint32_t)(s >> 32)};
}
__device__ __forceinline__ L64 mul5_add(L64 a, uint32_t c) {  // a * 5 + c
    const uint64_t p = (uint64_t)a.lo * 5u + c;
    return {(uint32_t)p, (uint32_t)(p >> 32) + a.hi * 5u};
}
__device__ __forceinline__ L64 fmix_l(L64 k) {
    k.lo ^= k.hi >> 1;  // k ^= k >> 33
    k = mul_c(k, 0xff51afd7ed558ccdULL);
    k.lo ^= k.hi >> 1;
    k = mul_c(k, 0xc4ceb9fe1a85ec53ULL);
    k.lo ^= k.hi >> 1;
    return k;
}
__device__ __forceinline__ L64 mix1(L64 k) { return mul_c(rotl_c(mul_c(k, C1), 31), C2); }
__device__ __forceinline__ L64 mix2(L64 k) { return mul_c(rotl_c(mul_c(k, C2), 33), C1); }

template <int K>
__device__ __forceinline__ uint64_t murmur_limbs(const uint32_t* a) {
    // a[] = the K translated bytes, little-endian packed, bytes past K zeroed.
    constexpr int NB = K / 16, REM = K % 16, NWORDS = (K + 3) / 4;
    L64 h1 = {(uint32_t)SEED, 0}, h2 = {(uint32_t)SEED, 0};
#pragma unroll
    for (int b = 0; b < NB; b++) {
        h1 = xor_(h1, mix1({a[4 * b], a[4 * b + 1]}));
        h1 = add_(rotl_c(h1, 27), h2);
        h1 = mul5_add(h1, 0x52dce729u);
        h2 = xor_(h2, mix2({a[4 * b + 2], a[4 * b + 3]}));
        h2 = add_(rotl_c(h2, 31), h1);
        h2 = mul5_add(h2, 0x38495ab5u);
    }
    auto word = [&](int i) -> uint32_t { return i < NWORDS ? a[i] : 0u; };
    if (REM > 8) h2 = xor_(h2, mix2({word(4 * NB + 2), word(4 * NB + 3)}));
    if (REM > 0) h1 = xor_(h1, mix1({word(4 * NB), word(4 * NB + 1)}));
    h1.lo ^= (uint32_t)K;
    h2.lo ^= (uint32_t)K;
    h1 = add_(h1, h2);
    h2 = add_(h2, h1);
    h1 = fmix_l(h1);
    h2 = fmix_l(h2);
    h1 = add_(h1, h2);
    return ((uint64_t)h1.hi << 32) | h1.lo;
}

constexpr int SQ_ROWS = SK_TILE / (SK_THREADS * 4);   // quad rows per warp (2)
constexpr int SQ_SEG = SK_TILE / 4 + 4;                // staging segment stride in slots: = 4 (mod 16)
__device__ __forceinline__ uint32_t stage_addr(uint32_t slot) { return (slot & 3u) * SQ_SEG + (slot >> 2); }
static_assert(DS_ITEMS == SQ_ROWS * 4, "a thread's windows are its scatter items");
static_assert(DS_THREADS == SK_THREADS && DS_TILE == SK_TILE, "one scatter tile per sketch tile");

// The bytes of quad q (windows 4q .. 4q + 3 of the tile): the aligned words of s_res that cover them.
template <int K>
struct Quad {
    static constexpr int NW = (K + 3 + 3) / 4;  // words that cover the 4 + K - 1 bytes of a quad
    static constexpr int KW = (K + 3) / 4;      // words of one window
    uint32_t x[NW + 1];
    __device__ __forceinline__ Quad(const uint32_t* s_res, uint32_t q) {
#pragma unroll
        for (int i = 0; i < NW; i++) x[i] = s_res[q + i];
        x[NW] = 0;
    }
    // MurmurHash3 of window j of the quad: its K bytes cut out with a funnel shift, bytes past K zeroed
    __device__ __forceinline__ uint64_t hash(int j) const {
        uint32_t b[KW];
#pragma unroll
        for (int i = 0; i < KW; i++) b[i] = j == 0 ? x[i] : __funnelshift_r(x[i], x[i + 1], 8 * j);
        if (K % 4) b[KW - 1] &= (1u << (8 * (K % 4))) - 1u;
        return murmur_limbs<K>(b);
    }
};

// Ordered staging of one quad row: the kept windows of the warp's 32 quads are ranked in window order (lane, then j) with
// four ballots, and put(j, addr) stores this lane's window j at its staging address.  wcount: entries the warp has
// staged so far (uniform across the warp).
template <class Put>
__device__ __forceinline__ void stage_row(uint32_t lane, uint32_t warp, const bool (&keep)[4], uint32_t& wcount, Put put) {
    const uint32_t lt = (1u << lane) - 1u;
    uint32_t below = 0, total = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const uint32_t bal = __ballot_sync(0xffffffffu, keep[j]);
        below += __popc(bal & lt);
        total += __popc(bal);
    }
    uint32_t slot = warp * WARP_SLOTS + wcount + below;
#pragma unroll
    for (int j = 0; j < 4; j++) {
        if (keep[j]) {
            put(j, stage_addr(slot));
            slot++;
        }
    }
    wcount += total;
}

#ifndef KS_SK_CTAS
#define KS_SK_CTAS 5
#endif
#ifndef KS_SK_CTAS_LB
#define KS_SK_CTAS_LB 6
#endif
// FULL (max_hash = 2^64 - 1, i.e. scaled == 1): tile bases come from tile_count_kernel + scan, so there is no ticket, no
// look-back chain and no cross-CTA dependency at all.  SCATTER: unordered output, the first level of the partition
// follows in this kernel; hashes stay in registers and a window's loc waits in its own staging slot.
// CTAs per SM the register allocation aims at (FULL: exact path / look-back path).  Measured (round 2, C4 slice, the
// look-back path): 4 / 5 / 6 CTAs 9.26 / 7.75 / 6.77 ms (left to the compiler the non-scatter instantiations took 62-64
// registers = 4 CTAs); the exact path is best at 5 (100 M-residue target run 0.90 ms against 0.97 ms at 6).
template <int K, bool TRANSLATE, bool FULL, bool SCATTER>
__global__ void __launch_bounds__(SK_THREADS, FULL ? KS_SK_CTAS : KS_SK_CTAS_LB)
sketch_quad_kernel(SketchArgs a, Lut256 lut, uint32_t* __restrict__ ticket, uint64_t* __restrict__ status,
                   const uint32_t* __restrict__ tile_pid, const uint64_t* __restrict__ tile_base) {
    constexpr int RES_WORDS = (SK_TILE + K + 16 + 3) / 4;
    __shared__ __align__(16) uint32_t s_res[RES_WORDS];
    __shared__ __align__(16) uint64_t s_hash[4 * SQ_SEG];
    __shared__ __align__(16) uint64_t s_loc[4 * SQ_SEG];
    __shared__ uint64_t s_offs[OFFS_CACHE];
    __shared__ uint8_t s_lut[256];
    __shared__ uint8_t s_lut32[32];
    __shared__ uint32_t s_wtot[SK_THREADS / 32];
    __shared__ uint32_t s_tile;
    __shared__ uint64_t s_base;
    constexpr bool COUNT_ABUND = SCATTER && !FULL;  // kept windows per protein, counted per tile in shared memory
    __shared__ uint32_t s_pcnt[COUNT_ABUND ? OFFS_CACHE : 1];

    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (COUNT_ABUND) s_pcnt[tid] = 0;  // OFFS_CACHE == SK_THREADS; ordered before the first count by the barriers below
    if (!FULL && tid == 0) s_tile = atomicAdd(ticket, 1u);
    if (TRANSLATE) s_lut[tid] = lut.b[tid];
    if (!FULL || TRANSLATE) __syncthreads();
    const uint32_t tile = FULL ? blockIdx.x + a.tile_begin : s_tile;
    const uint64_t g0 = (uint64_t)tile * SK_TILE;
    const uint32_t p_lo = tile_pid[tile], p_hi = tile_pid[tile + 1];
    const bool cached = cache_offsets(tid, a, s_offs, p_lo, p_hi);
    if (a.packed) {  // (the code table is filled here, behind its own barrier, only when it is used)
        if (tid < 32) s_lut32[tid] = lut32_entry(lut.b, tid);
        __syncthreads();
        stage_residues<TRANSLATE>(tid, s_res, a, true, g0, SK_TILE + K - 1, s_lut, s_lut32);
    } else {
        stage_residues<TRANSLATE>(tid, s_res, a, false, g0, SK_TILE + K - 1, s_lut, s_lut32);
    }
    __syncthreads();

    const uint64_t* offs = cached ? (const uint64_t*)s_offs - p_lo : a.offsets;
    const uint32_t nres_rel = tile_residues(a, g0), g0_lo = (uint32_t)g0;
    const uint32_t w_first = (warp * SQ_ROWS * 32 + lane) * 4;
    uint32_t p = p_lo, pstart_lo = 0, pend_rel = 0;
    if (w_first < nres_rel) first_protein(offs, g0, p_lo, p_hi, w_first, p, pstart_lo, pend_rel);

    bool zero_seen = false;
    uint32_t wcount = 0;  // tuples staged by this warp so far (uniform across the warp)
    uint64_t dkey[SCATTER ? DS_ITEMS : 1];
    uint32_t dvalid = 0;
#pragma unroll
    for (int rr = 0; rr < SQ_ROWS; rr++) {
        const uint32_t q = (warp * SQ_ROWS + rr) * 32 + lane;
        const Quad<K> quad(s_res, q);
        uint64_t h[4], loc[4];
        bool keep[4];
        // a quad that lies inside one protein with all four windows complete (9 in 10) skips the per-window walk
        const bool inside = q * 4 + 3 + K <= pend_rel;  // the lane's protein state only moves forward: q * 4 is in p
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const uint32_t w = q * 4 + j;
            bool valid = inside;
            if (!inside && w < nres_rel) {
                seek_protein(offs, g0, w, p, pstart_lo, pend_rel);
                valid = w + K <= pend_rel;
            }
            h[j] = quad.hash(j);
            if (FULL) {
                keep[j] = valid;  // the count was fixed in advance; a zero hash (1 in 2^64) sends the batch to the general path
                zero_seen |= valid && h[j] == 0;
            } else {
                keep[j] = valid && h[j] != 0 && h[j] <= a.max_hash;
                if (COUNT_ABUND && keep[j]) {
                    if (cached) atomicAdd(&s_pcnt[p - p_lo], 1u);
                    else atomicAdd(&a.t_abund[p], 1u);  // a tile of more than 254 tiny proteins
                }
            }
            loc[j] = ((uint64_t)(a.pid_base + p) << 32) | (uint64_t)(g0_lo + w - pstart_lo);
        }
        if (SCATTER) {
#pragma unroll
            for (int j = 0; j < 4; j++) {
                dkey[SCATTER ? rr * 4 + j : 0] = h[j];
                dvalid |= (keep[j] ? 1u : 0u) << (rr * 4 + j);
                s_loc[(rr * 4 + j) * SK_THREADS + tid] = loc[j];
            }
        } else {
            stage_row(lane, warp, keep, wcount, [&](int j, uint32_t ad) {
                s_hash[ad] = h[j];
                s_loc[ad] = loc[j];
            });
        }
    }

    if (FULL && zero_seen) atomicOr(reinterpret_cast<uint32_t*>(a.d_count + 1) + 1, 1u);
    if (SCATTER) {
        static_assert(OFFS_CACHE == SK_THREADS, "one protein counter per thread");
        __shared__ DenseScatterSmem s_sc;
        const uint32_t total = scatter_pairs(reinterpret_cast<const uint64_t (&)[DS_ITEMS]>(dkey), dvalid,
                                             [&](int it) { return s_loc[it * SK_THREADS + tid]; }, a.scatter, 0, s_sc, s_hash, s_loc);
        if (COUNT_ABUND && cached && tid < p_hi - p_lo + 1) {  // (the scatter's barriers ordered the counts before this read)
            const uint32_t c = s_pcnt[tid];
            if (c) atomicAdd(&a.t_abund[p_lo + tid], c);
        }
        if (tid == 0 && total) atomicAdd(reinterpret_cast<unsigned long long*>(a.d_count), (unsigned long long)total);
        return;
    }
    const WarpPrefix wp = warp_prefix(tid, s_wtot, wcount);
    const uint64_t base = wp.wprefix + (FULL ? exact_base(tid, a, tile, tile_base, wp.btotal)
                                             : lookback_base(lane, warp, a, tile, status, wp.btotal, s_base));
    const uint32_t sbase = warp * WARP_SLOTS;
    uint64_t* oh = a.out_hash + base;
    uint64_t* ol = a.out_loc + base;
    write_warp(lane, a, base, wcount, [&](uint32_t i) {
        const uint32_t ad = stage_addr(sbase + i);
        oh[i] = s_hash[ad];
        ol[i] = s_loc[ad];
    });
}

// ---------------------------------------------------------------------------------------------
// Dense k-mer space (two-letter hp alphabet, K <= 24, scaled == 1; DESIGN.md 3.3): a window is a K-bit pattern, its hash
// a function of the pattern, and its tuple ONE 64-bit key  code | protein | position.  `code_of_pattern` (a per-handle
// table, dense.cu) gives every pattern an order-preserving code: the top DENSE_PREFIX_BITS bits of its hash, then its rank
// among the patterns of that hash prefix (sketch.cuh), so keys sort like (hash, protein, position) tuples.  This is the
// exact-path sketch kernel with the hash replaced by a table read: residues are staged and translated once per tile,
// turned into two bit streams (hydrophobic / neither class), and a window's pattern is one funnel shift.  A complete
// window that holds a residue of neither class (X, U, O, *) has no pattern: with handle_exceptions it is hashed from its
// bytes and placed among the patterns' hashes (an even code); without, the kernel flags it and the host builds the batch
// on the general path.  The keys leave either through the first level of the key sort (d.scatter.out != nullptr) or in
// tile order at the tiles' exact bases (d.out_keys, sorted by the library afterwards).
// ---------------------------------------------------------------------------------------------
// 5 CTAs per SM: measured 2.41 ms (4), 1.78 ms (5), 1.89 ms (6, 40 registers) on C2
#ifndef KS_DK_CTAS
#define KS_DK_CTAS 5
#endif

template <int K>
__global__ void __launch_bounds__(SK_THREADS, KS_DK_CTAS)
sketch_dense_kernel(SketchArgs a, Lut256 lut, const uint32_t* __restrict__ tile_pid, const uint64_t* __restrict__ tile_base,
                    DenseSketchArgs d) {
    constexpr int RES_WORDS = (SK_TILE + K + 16 + 3) / 4;
    constexpr int N_BITW = (SK_TILE + K - 2) / 32 + 2;  // words of the bit streams a tile's windows reach
    __shared__ __align__(16) uint32_t s_res[RES_WORDS];
    __shared__ __align__(16) uint64_t s_key[4 * SQ_SEG];
    __shared__ uint32_t s_hb[N_BITW], s_eb[N_BITW];
    __shared__ uint64_t s_offs[OFFS_CACHE];
    __shared__ uint8_t s_lut[256];
    __shared__ uint8_t s_lut32[32];
    __shared__ uint32_t s_wtot[SK_THREADS / 32];

    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    s_lut[tid] = lut.b[tid];
    if (tid < 32) s_lut32[tid] = lut32_entry(lut.b, tid);
    __syncthreads();
    const uint32_t tile = blockIdx.x + a.tile_begin;
    const uint64_t g0 = (uint64_t)tile * SK_TILE;
    const uint32_t p_lo = tile_pid[tile], p_hi = tile_pid[tile + 1];
    const bool cached = cache_offsets(tid, a, s_offs, p_lo, p_hi);
    stage_residues<true>(tid, s_res, a, a.packed, g0, SK_TILE + K - 1, s_lut, s_lut32);
    __syncthreads();
    // bit streams over the staged residues: bit i of word w = residue 32 w + i is hydrophobic / of neither class
    for (uint32_t wd = tid; wd < (uint32_t)N_BITW; wd += SK_THREADS) {
        uint32_t hb = 0, eb = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const uint32_t wi = wd * 8 + i;
            const uint32_t x = wi < (uint32_t)RES_WORDS ? s_res[wi] : 0u;
#pragma unroll
            for (int c = 0; c < 4; c++) {
                const uint32_t ch = (x >> (8 * c)) & 0xffu;
                hb |= (ch == 'h' ? 1u : 0u) << (4 * i + c);
                eb |= ((ch != 'h' && ch != 'p') ? 1u : 0u) << (4 * i + c);
            }
        }
        s_hb[wd] = hb;
        s_eb[wd] = eb;
    }
    __syncthreads();

    const uint64_t* offs = cached ? (const uint64_t*)s_offs - p_lo : a.offsets;
    const uint32_t nres_rel = tile_residues(a, g0), g0_lo = (uint32_t)g0;
    const uint32_t w_first = (warp * SQ_ROWS * 32 + lane) * 4;
    uint32_t p = p_lo, pstart_lo = 0, pend_rel = 0;
    if (w_first < nres_rel) first_protein(offs, g0, p_lo, p_hi, w_first, p, pstart_lo, pend_rel);

    constexpr uint32_t KMASK = K >= 32 ? 0xffffffffu : ((1u << (K & 31)) - 1u);
    const int loc_bits = d.pid_bits + d.pos_bits;
    bool exc_seen = false, exc_emitted = false;
    uint32_t wcount = 0;  // keys staged by this warp so far (uniform across the warp)
    const bool scatter = d.scatter.out != nullptr;
    uint64_t dkey[DS_ITEMS];
    uint32_t dvalid = 0;
#pragma unroll
    for (int rr = 0; rr < SQ_ROWS; rr++) {
        const uint32_t q = (warp * SQ_ROWS + rr) * 32 + lane;
        const uint32_t hlo = s_hb[q >> 3], hhi = s_hb[(q >> 3) + 1];
        const uint32_t elo = s_eb[q >> 3], ehi = s_eb[(q >> 3) + 1];
        const bool inside = q * 4 + 3 + K <= pend_rel;  // the lane's protein state only moves forward: q * 4 is in p
        uint32_t code[4], rank[4];
        uint64_t locp[4];
        bool keep[4], is_exc[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const uint32_t w = q * 4 + j;
            bool valid = inside;
            if (!inside && w < nres_rel) {
                seek_protein(offs, g0, w, p, pstart_lo, pend_rel);
                valid = w + K <= pend_rel;
            }
            const uint32_t bsh = ((q & 7u) << 2) + j;  // bit offset of window w in its stream word: (4q + j) mod 32
            code[j] = __funnelshift_r(hlo, hhi, bsh) & KMASK;
            is_exc[j] = valid && (__funnelshift_r(elo, ehi, bsh) & KMASK) != 0;
            keep[j] = valid;
            locp[j] = ((uint64_t)p << d.pos_bits) | (uint64_t)(g0_lo + w - pstart_lo);
        }
#pragma unroll
        for (int j = 0; j < 4; j++) rank[j] = __ldg(d.code_of_pattern + code[j]);
#pragma unroll
        for (int j = 0; j < 4; j++) {
            if (is_exc[j]) {  // rare: hash the translated bytes, place the hash among the patterns' hashes
                if (!d.handle_exceptions) { exc_seen = true; continue; }
                const uint64_t h = Quad<K>(s_res, q).hash(j);
                const uint32_t pfx = (uint32_t)(h >> (64 - DENSE_PREFIX_BITS));
                const uint32_t gb0 = __ldg(d.group_base + pfx), gb1 = __ldg(d.group_base + pfx + 1);
                uint32_t lo = gb0, hi = gb1;  // first pattern hash >= h inside the prefix group
                while (lo < hi) {
                    const uint32_t mid = (lo + hi) >> 1;
                    if (__ldg(d.sorted_hash + mid) < h) lo = mid + 1; else hi = mid;
                }
                const bool same = lo < gb1 && __ldg(d.sorted_hash + lo) == h;  // a pattern with this very hash
                rank[j] = (pfx << d.rb) | (2u * (lo - gb0) + (same ? 1u : 0u));
                if (h == 0) exc_seen = true;  // would have to be dropped: general path
                exc_emitted = true;
            }
        }
        if (scatter) {
#pragma unroll
            for (int j = 0; j < 4; j++) {
                dkey[rr * 4 + j] = ((uint64_t)rank[j] << loc_bits) | locp[j];
                dvalid |= (keep[j] ? 1u : 0u) << (rr * 4 + j);
            }
        } else {
            stage_row(lane, warp, keep, wcount, [&](int j, uint32_t ad) { s_key[ad] = ((uint64_t)rank[j] << loc_bits) | locp[j]; });
        }
    }
    if (exc_seen) atomicOr(d.exception_flag, 1u);
    if (exc_emitted) atomicOr(d.exception_flag + 1, 1u);
    if (scatter) {
        __shared__ DenseScatterSmem s_sc;
        const uint32_t total = scatter_keys(dkey, dvalid, d.scatter, 0, s_sc, s_key);
        if (tid == 0 && total) atomicAdd(reinterpret_cast<unsigned long long*>(a.d_count), (unsigned long long)total);
        return;
    }
    const WarpPrefix wp = warp_prefix(tid, s_wtot, wcount);
    const uint64_t base = exact_base(tid, a, tile, tile_base, wp.btotal) + wp.wprefix;
    const uint32_t sbase = warp * WARP_SLOTS;
    uint64_t* ok = d.out_keys + base;
#pragma unroll
    for (uint32_t i0 = 0; i0 < WARP_SLOTS; i0 += 32) {  // (one checked pass: write_warp's unrolled copy costs C2's scatter path 3 %)
        const uint32_t i = i0 + lane;
        if (i0 >= wcount) break;  // uniform
        if (i < wcount && base + i < a.capacity) ok[i] = s_key[stage_addr(sbase + i)];
    }
}

// Calls f(std::integral_constant<int, V>()) for the run-time value v = V in [LO, HI]; cudaErrorInvalidValue outside.
template <int LO, int HI, class F>
cudaError_t dispatch(int v, F&& f) {
    if constexpr (LO > HI) return cudaErrorInvalidValue;
    else return v == HI ? f(std::integral_constant<int, HI>()) : dispatch<LO, HI - 1>(v, f);
}

// Tiles [a.tile_begin, a.tile_end) of the batch, or all tiles when the range is empty (the look-back path takes tiles by
// ticket: its ranges must be launched in order, each exactly once).
unsigned grid_of(const SketchArgs& a, uint64_t n_tiles) {
    return a.tile_end > a.tile_begin ? (unsigned)(a.tile_end - a.tile_begin) : (unsigned)n_tiles;
}

}  // namespace

bool pack_residues(const uint8_t* res, uint64_t n, uint8_t* out) {
    const uint64_t groups = (n + 7) / 8;
    for (uint64_t g = 0; g < groups; g++) {
        uint64_t v = 0;
        for (int i = 0; i < 8; i++) {
            const uint64_t idx = g * 8 + i;
            if (idx >= n) break;
            const uint8_t c = res[idx];
            uint32_t code;
            if (c >= 'A' && c <= 'Z') code = c - 'A' + 1;
            else if (c == '*') code = 27;
            else return false;
            v |= (uint64_t)code << (5 * i);
        }
        for (int b = 0; b < 5; b++) out[g * 5 + b] = (uint8_t)(v >> (8 * b));
    }
    memset(out + groups * 5, 0, 72);
    return true;
}

void fill_lut(int moltype, Lut256* lut) {
    for (int i = 0; i < 256; i++) {
        uint8_t c = (uint8_t)i, o = c;
        if (moltype == 1) {
            switch (c) {
                case '*': o = '*'; break;
                case 'C': o = 'a'; break;
                case 'A': case 'G': case 'P': case 'S': case 'T': o = 'b'; break;
                case 'D': case 'E': case 'N': case 'Q': o = 'c'; break;
                case 'H': case 'K': case 'R': o = 'd'; break;
                case 'I': case 'L': case 'M': case 'V': o = 'e'; break;
                case 'F': case 'W': case 'Y': o = 'f'; break;
                default: o = 'X';
            }
        } else if (moltype == 2) {
            switch (c) {
                case '*': o = '*'; break;
                case 'A': case 'F': case 'G': case 'I': case 'L': case 'M': case 'P': case 'V': case 'W': case 'Y':
                    o = 'h'; break;
                case 'C': case 'D': case 'E': case 'H': case 'K': case 'N': case 'Q': case 'R': case 'S': case 'T':
                    o = 'p'; break;
                default: o = 'X';
            }
        }
        lut->b[i] = o;
    }
}

size_t sketch_workspace_bytes(uint64_t n_res) {
    const uint64_t nt = n_tiles_of(n_res);
    return ((16 + nt * 8 + (nt + 1) * 4 + 15) & ~(size_t)15) + 2 * (nt + 1) * 8 + scan_temp_bytes_for(nt + 1) + 64;
}

static bool exact_path(const SketchArgs& a) {
    return a.max_hash == ~0ull && !a.force_general && a.k <= (uint32_t)SK_MAX_TEMPLATE_K;
}

cudaError_t launch_sketch_prepare(const SketchArgs& a, cudaStream_t stream, uint64_t* n_launches) {
    if (a.n_res == 0 || a.n_prot == 0) return a.count_zeroed ? cudaSuccess : cudaMemsetAsync(a.d_count, 0, 16, stream);
    const uint64_t nt = n_tiles_of(a.n_res);
    Workspace w = carve(a.workspace, a.n_res);
    const bool exact = exact_path(a);
    const bool unordered = a.unordered || a.scatter.out_key != nullptr;
    cudaError_t e = cudaSuccess;
    if (!exact) e = cudaMemsetAsync(a.workspace, 0, 16 + nt * 8, stream);  // ticket + look-back status
    if (e != cudaSuccess) return e;
    // exact path: [1] collects the zero-hash flag; unordered output: the tiles add their totals up in [0]
    if ((exact || unordered) && !a.count_zeroed) {
        e = cudaMemsetAsync(a.d_count, 0, 16, stream);
        if (e != cudaSuccess) return e;
    }
    tile_pid_kernel<<<(unsigned)((a.n_prot + 255) / 256), 256, 0, stream>>>(a.offsets, a.n_prot, nt, w.tile_pid);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    if (n_launches) *n_launches += 1;
    if (exact && !unordered) {  // ordered output: the exact number of windows per tile, scanned
        tile_count_kernel<<<(unsigned)((nt + 1 + 255) / 256), 256, 0, stream>>>(a.offsets, a.n_res, a.k, nt, w.tile_pid, w.tile_cnt);
        size_t tb = w.scan_temp_bytes;
        e = cub::DeviceScan::ExclusiveSum(w.scan_temp, tb, w.tile_cnt, w.tile_base, (int64_t)(nt + 1), stream);
        if (e != cudaSuccess) return e;
        if (n_launches) *n_launches += 3;
    }
    return cudaSuccess;
}

// The sketch kernel over tiles [a.tile_begin, a.tile_end) (0, 0 = all tiles).
cudaError_t launch_sketch_tiles(const SketchArgs& a, cudaStream_t stream, uint64_t* n_launches) {
    if (a.n_res == 0 || a.n_prot == 0) return cudaSuccess;
    const Workspace w = carve(a.workspace, a.n_res);
    const unsigned grid = grid_of(a, n_tiles_of(a.n_res));
    Lut256 lut;
    fill_lut(a.moltype, &lut);
    if (n_launches) *n_launches += 1;
    if (a.k > (uint32_t)SK_MAX_TEMPLATE_K) {
        if (a.moltype == 0) sketch_kernel<false><<<grid, SK_THREADS, 0, stream>>>(a, lut, w.ticket, w.status, w.tile_pid);
        else sketch_kernel<true><<<grid, SK_THREADS, 0, stream>>>(a, lut, w.ticket, w.status, w.tile_pid);
        return cudaGetLastError();
    }
    const bool translate = a.moltype != 0, full = exact_path(a), scatter = a.scatter.out_key != nullptr;
    return dispatch<1, SK_MAX_TEMPLATE_K>((int)a.k, [&](auto K) {
        return dispatch<0, 1>(translate, [&](auto T) {
            return dispatch<0, 1>(full, [&](auto F) {
                return dispatch<0, 1>(scatter, [&](auto S) {
                    sketch_quad_kernel<K, T != 0, F != 0, S != 0>
                        <<<grid, SK_THREADS, 0, stream>>>(a, lut, w.ticket, w.status, w.tile_pid, w.tile_base);
                    return cudaGetLastError();
                });
            });
        });
    });
}

// Look-back path: d_count[1] <- 0 (no zero-hash flag there: such a hash fails h != 0 and is dropped in the kernel).  The
// exact path sets the flag in d_count[1] itself.
cudaError_t launch_sketch_finish(const SketchArgs& a, cudaStream_t stream) {
    if (a.n_res == 0 || a.n_prot == 0 || exact_path(a)) return cudaSuccess;
    return cudaMemsetAsync(a.d_count + 1, 0, 8, stream);
}

cudaError_t launch_sketch(const SketchArgs& a, cudaStream_t stream, uint64_t* n_launches) {
    cudaError_t e = launch_sketch_prepare(a, stream, n_launches);
    if (e != cudaSuccess) return e;
    e = launch_sketch_tiles(a, stream, n_launches);
    if (e != cudaSuccess) return e;
    return launch_sketch_finish(a, stream);
}

// Dense path: tile -> protein map, exact tile bases (launch_sketch_prepare), then the rank kernel over all tiles (or
// [tile_begin, tile_end) when a.tile_end > a.tile_begin).  a.out_hash / a.out_loc are not used.
cudaError_t launch_sketch_dense(const SketchArgs& a, const DenseSketchArgs& d, cudaStream_t stream, uint64_t* n_launches) {
    if (a.n_res == 0 || a.n_prot == 0) return cudaSuccess;
    if (a.moltype != 2 || a.k < (uint32_t)DENSE_MIN_K || a.k > (uint32_t)DENSE_MAX_K || a.max_hash != ~0ull) return cudaErrorInvalidValue;
    const Workspace w = carve(a.workspace, a.n_res);
    const unsigned grid = grid_of(a, n_tiles_of(a.n_res));
    Lut256 lut;
    fill_lut(a.moltype, &lut);
    if (n_launches) *n_launches += 1;
    return dispatch<DENSE_MIN_K, DENSE_MAX_K>((int)a.k, [&](auto K) {
        sketch_dense_kernel<K><<<grid, SK_THREADS, 0, stream>>>(a, lut, w.tile_pid, w.tile_base, d);
        return cudaGetLastError();
    });
}

}  // namespace ks
