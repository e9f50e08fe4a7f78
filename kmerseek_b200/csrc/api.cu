// C ABI of the kmerseek B200 sketch-and-search path (include/kmerseek_b200.h).
// Host orchestration only: pinned packing, H2D streaming, stage launches, result hand-back.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <new>
#include <time.h>

#include <nccl.h>  // types and prototypes only: the library is bound with dlopen (NcclApi), never linked

#include "append.cuh"
#include "dense.cuh"
#include "host_util.hpp"
#include "ingest.hpp"
#include "index_build.cuh"
#include "search.cuh"
#include "sketch.cuh"
#include "util.cuh"

using namespace ks;

// ------------------------------------------------------------------------------------------------
// error slot
// ------------------------------------------------------------------------------------------------
namespace {
thread_local std::string g_err;
thread_local uint32_t g_err_ch = 0;
thread_local uint64_t g_err_pos = 0, g_err_protein = 0;

ks_status set_error(ks_status s, const std::string& m) { g_err = m; return s; }

template <class F>
ks_status guarded(F&& f) {
    try {
        f();
        return KS_OK;
    } catch (const KsError& e) {
        return set_error(e.status, e.message);
    } catch (const std::bad_alloc&) {
        return set_error(KS_ERR_OUT_OF_MEMORY, "out of host memory");
    } catch (const std::exception& e) {
        return set_error(KS_ERR_VALIDATION, e.what());
    }
}

[[noreturn]] void fail_residue(const InvalidResidue& b) {
    g_err_ch = b.ch; g_err_pos = b.pos; g_err_protein = b.protein;
    char msg[128];
    // src/rust/errors.rs:14-15
    snprintf(msg, sizeof msg, "Invalid amino acid '%c' found at position %llu", (char)b.ch, (unsigned long long)b.pos);
    fail(KS_ERR_INVALID_AMINO_ACID, msg);
}

int clz64(uint64_t x) { return x ? __builtin_clzll(x) : 64; }
}  // namespace

// ------------------------------------------------------------------------------------------------
// proteome (host buffers: the upload formats pinned, from a pool that outlives the objects)
// ------------------------------------------------------------------------------------------------
namespace {

// Pinned blocks are recycled (proteomes, search results): cudaHostAlloc of a few hundred MB costs more than filling them.
std::mutex g_pin_mu;
std::vector<std::pair<void*, size_t>> g_pin_free;
size_t g_pin_pooled = 0;

void* pinned_try_get(size_t bytes, size_t* got) {  // nullptr when there is no device to pin for
    {
        std::lock_guard<std::mutex> lk(g_pin_mu);
        int best = -1;
        for (size_t i = 0; i < g_pin_free.size(); i++)
            if (g_pin_free[i].second >= bytes && (best < 0 || g_pin_free[i].second < g_pin_free[best].second)) best = (int)i;
        if (best >= 0 && g_pin_free[best].second <= 2 * bytes + (1u << 20)) {
            auto b = g_pin_free[best];
            g_pin_free.erase(g_pin_free.begin() + best);
            g_pin_pooled -= b.second;
            *got = b.second;
            return b.first;
        }
    }
    const size_t want = bytes + bytes / 8 + (1u << 16);
    void* p = nullptr;
    if (cudaHostAlloc(&p, want, cudaHostAllocDefault) != cudaSuccess) { (void)cudaGetLastError(); return nullptr; }
    *got = want;
    return p;
}

void* pinned_get(size_t bytes, size_t* got) {
    void* p = pinned_try_get(bytes, got);
    if (!p) fail(KS_ERR_OUT_OF_MEMORY, "cudaHostAlloc failed");
    return p;
}

void pinned_put(void* p, size_t bytes) {
    if (!p) return;
    std::lock_guard<std::mutex> lk(g_pin_mu);
    if (g_pin_pooled + bytes > (8ull << 30)) { cudaFreeHost(p); return; }
    g_pin_free.emplace_back(p, bytes);
    g_pin_pooled += bytes;
}

struct HostBuf {
    void* p = nullptr;
    size_t bytes = 0;  // of the block (pinned: as the pool knows it)
    bool pinned = false;
    // pinned (pooled) when a device is there and `want_pinned`; pageable otherwise (CPU-only host tests, or buffers that are
    // not an upload format)
    void alloc(size_t n, bool want_pinned) {
        release();
        if (want_pinned) {
            p = pinned_try_get(n, &bytes);
            pinned = p != nullptr;
        }
        if (!p) {
            p = malloc(n ? n : 1);
            if (!p) throw std::bad_alloc();
            bytes = n;
            pinned = false;
        }
    }
    void release() {
        if (!p) return;
        if (pinned) pinned_put(p, bytes); else free(p);
        p = nullptr; bytes = 0; pinned = false;
    }
};

}  // namespace

struct ks_proteome {
    uint8_t* residues = nullptr;  // normalised residues (+ 64 zero bytes); pageable when the packed copy is the upload format
    uint64_t* offsets = nullptr;  // pinned
    uint64_t n_prot = 0, n_res = 0;
    // upload format: 5-bit codes, 8 residues per 5 bytes, pinned (null when a byte outside A-Z and '*' is present: the
    // residues themselves are then pinned and uploaded)
    uint8_t* packed = nullptr;
    HostBuf b_res, b_offs, b_packed;
    std::string name_blob;  // NUL-terminated names back to back; empty when no names were given
    std::vector<uint64_t> name_off;
    // shape of the batch, computed once per k-mer size (one pass over the offsets; every add of the proteome needs it)
    std::mutex shape_mu;
    bool shape_valid = false;
    uint32_t shape_k = 0;
    uint64_t shape_windows = 0, shape_max_len = 0;
    ~ks_proteome() { b_res.release(); b_offs.release(); b_packed.release(); }
};

namespace {

// residues are in p->residues (pageable): build the packed upload copy, or pin the residues when they cannot be packed.
// `prepacked`: the caller has packed into p->packed already (the FASTA parser does it while it fills the residues);
// 1 = every byte had a code, 0 = some byte had none.
void finish_proteome(ks_proteome* p, int prepacked = -1) {
    memset(p->residues + p->n_res, 0, 64);
    if (prepacked < 0) {
        p->b_packed.alloc(packed_bytes(p->n_res), true);
        p->packed = (uint8_t*)p->b_packed.p;
    }
    if (prepacked < 0 ? !pack_residues_parallel(p->residues, p->n_res, p->packed) : prepacked == 0) {
        p->b_packed.release();
        p->packed = nullptr;
        HostBuf pin;
        pin.alloc(p->n_res + 64, true);
        memcpy(pin.p, p->residues, p->n_res + 64);
        p->b_res.release();
        p->b_res = pin;
        p->residues = (uint8_t*)pin.p;
    }
}

ks_proteome* new_proteome(uint64_t n_res, uint64_t n_prot) {
    ks_proteome* p = new ks_proteome();
    try {
        p->b_res.alloc(n_res + 64, false);
        p->b_offs.alloc((n_prot + 1) * 8, true);
    } catch (...) {
        delete p;
        throw;
    }
    p->residues = (uint8_t*)p->b_res.p;
    p->offsets = (uint64_t*)p->b_offs.p;
    p->n_prot = n_prot;
    p->n_res = n_res;
    return p;
}

ks_proteome* make_proteome(const uint8_t* res, uint64_t n_res, const uint64_t* offs, uint64_t n_prot) {
    ks_proteome* p = new_proteome(n_res, n_prot);
    try {
        if (n_res) {  // first touch of a fresh buffer: all host threads copy (and fault the pages in) at once
            const int t = ingest_threads((size_t)n_res);
            parallel_chunks(t, [&](int i) {
                const uint64_t a = n_res * (uint64_t)i / t, b = n_res * (uint64_t)(i + 1) / t;
                memcpy(p->residues + a, res + a, b - a);
            });
        }
        memcpy(p->offsets, offs, (n_prot + 1) * 8);
        finish_proteome(p);
    } catch (...) {
        delete p;
        throw;
    }
    return p;
}

void set_names(ks_proteome* p, const std::vector<std::string>& names) {
    p->name_off.resize(names.size());
    size_t total = 0;
    for (auto& n : names) total += n.size() + 1;
    p->name_blob.resize(total);
    size_t at = 0;
    for (size_t i = 0; i < names.size(); i++) {
        p->name_off[i] = at;
        memcpy(&p->name_blob[at], names[i].c_str(), names[i].size() + 1);
        at += names[i].size() + 1;
    }
}

double wall_ms() {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6;
}

ks_proteome* proteome_from_fasta(const char* path, uint64_t ambig_seed, NormalizeMode mode) {
    static const bool timing = getenv("KS_TIMING") != nullptr;  // read once
    const double t0 = timing ? wall_ms() : 0;
    FastaBytes fb;
    load_fasta_bytes(path, &fb);
    const double t1 = timing ? wall_ms() : 0;
    FastaParser parser(fb.data, fb.size, mode, ambig_seed);
    const ParsedFasta t = parser.count();
    const double t2 = timing ? wall_ms() : 0;
    ks_proteome* p = new_proteome(t.n_res, t.n_rec);
    try {
        p->name_blob.resize(t.name_bytes);
        p->name_off.resize(t.n_rec);
        p->b_packed.alloc(packed_bytes(t.n_res), true);  // the upload copy is packed in the same pass as the residues
        p->packed = (uint8_t*)p->b_packed.p;
        const double t3 = timing ? wall_ms() : 0;
        InvalidResidue bad;
        bool packed_ok = true;
        if (!parser.fill(p->residues, p->offsets, t.name_bytes ? &p->name_blob[0] : nullptr, p->name_off.data(), &bad, p->packed,
                         &packed_ok))
            fail_residue(bad);
        for (uint64_t i = 0; i < t.n_rec; i++)
            if (p->offsets[i + 1] - p->offsets[i] > 0xffffffffull) fail(KS_ERR_CAPACITY, "protein longer than 2^32-1 residues");
        const double t4 = timing ? wall_ms() : 0;
        finish_proteome(p, packed_ok ? 1 : 0);
        if (timing) fprintf(stderr, "[ks] from_fasta: map %.1f ms, count %.1f, alloc %.1f, fill + pack %.1f, finish %.1f ms\n", t1 - t0, t2 - t1,
                            t3 - t2, t4 - t3, wall_ms() - t4);
    } catch (...) {
        delete p;
        throw;
    }
    return p;
}
}  // namespace

extern "C" {

const char* ks_last_error_message(void) { return g_err.c_str(); }
void ks_last_error_detail(uint32_t* ch, uint64_t* pos, uint64_t* protein_index) {
    if (ch) *ch = g_err_ch;
    if (pos) *pos = g_err_pos;
    if (protein_index) *protein_index = g_err_protein;
}
int ks_abi_version(void) { return KS_ABI_VERSION; }
int ks_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { (void)cudaGetLastError(); return 0; }
    return n;
}

ks_status ks_moltype_from_str(const char* m, ks_moltype* out) {
    std::string s = m ? m : "";
    if (s == "protein" || s == "raw") { *out = KS_PROTEIN; return KS_OK; }
    if (s == "hp") { *out = KS_HP; return KS_OK; }
    if (s == "dayhoff") { *out = KS_DAYHOFF; return KS_OK; }
    // src/rust/encoding.rs:22-25
    return set_error(KS_ERR_INVALID_MOLTYPE, "Invalid moltype: " + s + ", only 'protein', 'hp', or 'dayhoff' are supported");
}
const char* ks_moltype_name(ks_moltype m) { return m == KS_DAYHOFF ? "dayhoff" : m == KS_HP ? "hp" : "protein"; }

uint64_t ks_max_hash(uint32_t scaled) {
    if (scaled == 0) return 0;
    if (scaled == 1) return UINT64_MAX;
    return (uint64_t)(18446744073709551616.0 / (double)scaled);
}
uint8_t ks_translate_residue(uint8_t aa, ks_moltype m) {
    Lut256 lut;
    fill_lut((int)m, &lut);
    return lut.b[aa];
}
void ks_md5_of_mins(const uint64_t* mins, uint64_t n, uint32_t ksize, char out[33]) {
    Md5 md;
    char buf[32];
    int l = snprintf(buf, sizeof buf, "%u", ksize * KS_PROTEIN_TO_MINHASH_RATIO);
    md.update(buf, l);
    for (uint64_t i = 0; i < n; i++) {
        l = snprintf(buf, sizeof buf, "%llu", (unsigned long long)mins[i]);
        md.update(buf, l);
    }
    md.hex(out);
}
void ks_id_of_mins(const uint64_t* mins, uint64_t n, char out[17]) {
    uint64_t s = 0;
    for (uint64_t i = 0; i < n; i++) s += mins[i];
    snprintf(out, 17, "%llx", (unsigned long long)s);
}

// ---- ingest -------------------------------------------------------------------------------------
ks_status ks_proteome_from_sequences_mode(const char* const* seqs, const uint64_t* lens, const char* const* names, uint64_t n,
                                          uint64_t ambig_seed, int mode, ks_proteome** out) {
    return guarded([&] {
        if (!out || (n && (!seqs || !lens))) fail(KS_ERR_VALIDATION, "Validation error: null argument");
        if (mode != KS_NORMALIZE_KMERSEEK && mode != KS_NORMALIZE_SOURMASH) fail(KS_ERR_VALIDATION, "Validation error: unknown normalisation mode");
        std::vector<uint8_t> res;
        std::vector<uint64_t> offs(n + 1, 0);
        uint64_t total = 0;
        for (uint64_t i = 0; i < n; i++) total += lens[i];
        res.reserve(total);
        for (uint64_t i = 0; i < n; i++) {
            InvalidResidue bad;
            if (!normalize_into(seqs[i], lens[i], i, ambig_seed, mode == KS_NORMALIZE_SOURMASH, res, &bad)) fail_residue(bad);
            if (res.size() - offs[i] > 0xffffffffull) fail(KS_ERR_CAPACITY, "protein longer than 2^32-1 residues");
            offs[i + 1] = res.size();
        }
        ks_proteome* p = make_proteome(res.data(), res.size(), offs.data(), n);
        if (names) {
            std::vector<std::string> nm;
            nm.reserve(n);
            for (uint64_t i = 0; i < n; i++) nm.emplace_back(names[i] ? names[i] : "");
            set_names(p, nm);
        }
        *out = p;
    });
}
ks_status ks_proteome_from_sequences(const char* const* seqs, const uint64_t* lens, const char* const* names, uint64_t n,
                                     uint64_t ambig_seed, ks_proteome** out) {
    return ks_proteome_from_sequences_mode(seqs, lens, names, n, ambig_seed, KS_NORMALIZE_KMERSEEK, out);
}

ks_status ks_proteome_from_fasta_mode(const char* path, uint64_t ambig_seed, int mode, ks_proteome** out) {
    return guarded([&] {
        if (!out || !path) fail(KS_ERR_VALIDATION, "Validation error: null argument");
        if (mode != KS_NORMALIZE_KMERSEEK && mode != KS_NORMALIZE_SOURMASH) fail(KS_ERR_VALIDATION, "Validation error: unknown normalisation mode");
        *out = proteome_from_fasta(path, ambig_seed, (NormalizeMode)mode);
    });
}
ks_status ks_proteome_from_fasta(const char* path, uint64_t ambig_seed, ks_proteome** out) {
    return ks_proteome_from_fasta_mode(path, ambig_seed, KS_NORMALIZE_KMERSEEK, out);
}

ks_status ks_proteome_from_packed(const uint8_t* residues, const uint64_t* offsets, uint64_t n_proteins, ks_proteome** out) {
    return guarded([&] {
        if (!out || !offsets || (offsets[n_proteins] && !residues)) fail(KS_ERR_VALIDATION, "Validation error: null argument");
        if (offsets[0] != 0) fail(KS_ERR_VALIDATION, "Validation error: offsets[0] must be 0");
        for (uint64_t i = 0; i < n_proteins; i++) {
            if (offsets[i + 1] < offsets[i]) fail(KS_ERR_VALIDATION, "Validation error: offsets must be non-decreasing");
            if (offsets[i + 1] - offsets[i] > 0xffffffffull) fail(KS_ERR_CAPACITY, "protein longer than 2^32-1 residues");
        }
        *out = make_proteome(residues, offsets[n_proteins], offsets, n_proteins);
    });
}

uint64_t ks_proteome_n_proteins(const ks_proteome* p) { return p ? p->n_prot : 0; }
uint64_t ks_proteome_n_residues(const ks_proteome* p) { return p ? p->n_res : 0; }
const uint8_t* ks_proteome_residues(const ks_proteome* p) { return p ? p->residues : nullptr; }
const uint64_t* ks_proteome_offsets(const ks_proteome* p) { return p ? p->offsets : nullptr; }
const uint8_t* ks_proteome_packed(const ks_proteome* p, uint64_t* n_bytes) {
    if (n_bytes) *n_bytes = (p && p->packed) ? packed_bytes(p->n_res) : 0;
    return p ? p->packed : nullptr;
}
const char* ks_proteome_name(const ks_proteome* p, uint64_t i) {
    return (p && i < p->name_off.size()) ? p->name_blob.data() + p->name_off[i] : "";
}
void ks_proteome_free(ks_proteome* p) { delete p; }

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// index handle
// ------------------------------------------------------------------------------------------------
namespace {

// Grow-only device buffer: steady-state steps (clear + build again) never go back to the allocator.
struct Buf {
    void* p = nullptr;
    size_t bytes = 0;
    template <class T>
    T* ensure(Arena* ar, size_t n) {
        const size_t need = (n ? n : 1) * sizeof(T);
        if (need > bytes) {
            if (p) ar->release(p);
            p = ar->alloc<char>(need);
            bytes = need;
        }
        return (T*)p;
    }
};

struct DeviceBatch {  // residues + offsets resident in HBM
    uint8_t* res = nullptr;
    uint64_t* offs = nullptr;
    Buf b_res, b_offs;  // (a batch of the handle)
    uint64_t n_prot = 0, n_res = 0, n_windows = 0;
    uint64_t max_len = 0;  // longest protein of the batch
    bool valid = false;
    bool packed = false;  // res holds 5-bit codes
    uint64_t res_bytes() const { return packed ? packed_bytes(n_res) : n_res + 64; }
};

// k-mer windows and longest protein of a proteome for k-mer size k (cached on the proteome: one pass per k)
void proteome_shape(const ks_proteome* cp, uint32_t k, uint64_t* n_windows, uint64_t* max_len) {
    ks_proteome* p = const_cast<ks_proteome*>(cp);
    std::lock_guard<std::mutex> g(p->shape_mu);
    if (!p->shape_valid || p->shape_k != k) {
        uint64_t w = 0, m = 0;
        const uint64_t* offs = p->offsets;
        for (uint64_t i = 0; i < p->n_prot; i++) {
            const uint64_t len = offs[i + 1] - offs[i];
            m = std::max(m, len);
            if (len >= k) w += len - k + 1;
        }
        p->shape_windows = w; p->shape_max_len = m; p->shape_k = k; p->shape_valid = true;
    }
    *n_windows = p->shape_windows;
    *max_len = p->shape_max_len;
}

// What a handle holds.  The four values between Tuples and Finalized are a pending batch: the resident batch, added as the
// handle's only content by a route that finalize completes.  n_tuples / n_prot / n_res / n_windows count it already.
enum class Build {
    Tuples,              // (protein, pos)-ordered tuples in d_hash / d_loc [0, n_tuples), possibly none: finalize sorts them
    DenseDeferred,       // the batch is counted, not sketched: finalize runs the dense path's rank kernel over it, then
                         // builds from the keys
    DenseRanked,         // the pipelined add has run the rank kernel: the keys are in the dense work buffer (in d_hash when
                         // the library sorts them), the kernel's flags in d_status; finalize builds from them
    Scattered,           // the tuples are in the first-level regions of the unstable partition (b_pair_work, pair_plan) and
                         // the kernel's count has been checked; scaled > 1: t_abund holds the kept windows per protein.
                         // finalize runs the second level and the bin kernel, the postings go to d_loc
    ScatteredUnchecked,  // as Scattered, at scaled == 1: the kernel's count and zero-hash flag (d_count) are read back with
                         // finalize's results
    Finalized,           // csr is the index; adds fail until ks_index_clear
};

// The finalized index: views into the handle's grow-only buffers and, for the segmented layout, into the build's scratch
// (which stays with the handle until the next build).  Meaningful in state Finalized only.
struct Csr {
    uint64_t* keys = nullptr;
    uint32_t *key_grp = nullptr, *grp_start = nullptr, *t_size = nullptr, *t_abund = nullptr, *dir = nullptr;
    uint64_t* d_counts = nullptr;
    int dir_bits = 0, dir_shift = 0;
    int dir_sub = DIR_SUB_COMPACT;  // layout of keys / key_grp / grp_start (index_build.cuh): compact, or segmented
    uint32_t seg_nb = 0;
    const uint32_t* seg_start = nullptr;
    const uint64_t* seg_counts = nullptr;
    uint64_t* hash = nullptr;  // sorted tuples: the hash column (see hash_col_valid) and the postings
    uint64_t* loc = nullptr;
    uint64_t U = 0, G = 0, n_ids = 0;
    bool hash_col_valid = true;  // false: the sorted hash column is rebuilt on demand (ks_index_export)
};

// Buffers of a finalized index of its own: where an index extended by ks_index_append_* lives (two sets, ping-pong: the
// next append merges from one into the other, and a build never touches either).
struct CsrSet {
    Buf keys, key_grp, grp_start, t_size, t_abund, dir, hash, loc, seg_start, seg_counts;
};

// The device words a build reports through (ks_index::d_status), one block so that they are zeroed and read back together.
struct StatusBlock {
    uint64_t U, G;         // CSR totals (d_counts)
    uint64_t produced;     // tuples of the sketch kernel (d_count[0])
    uint64_t zero_flag;    // high word != 0: a zero hash on the exact path (d_count[1])
    uint64_t dense_flags;  // dense path, u32 pair: unhandled exception | exception keys emitted
    uint64_t overflow;     // u32: a sort bucket of the dense path overflowed (the unstable partition's own flag is read here)
};

}  // namespace

// Test / experiment hooks, read from the environment ONCE when the handle is created (never on the hot path).
struct Hooks {
    bool sketch_general = false;  // KS_SKETCH_GENERAL: take the look-back sketch path at scaled == 1
    int dense = -1;               // KS_DENSE: 0 switches the dense k-mer space path off, 1 drops its coverage condition
    bool scatter_off = false;     // KS_SCATTER=0: no unstable partition on the general path
    bool no_pipeline = false;     // KS_NO_PIPELINE: one copy + one launch instead of the chunked upload
    bool dense_sort_library = false;  // KS_DENSE_SORT=library: the dense path's keys sorted by the library
    bool timing = false;          // KS_TIMING: host-side stage timings on stderr
    bool search_legacy = false;   // KS_SEARCH_LEGACY: the library-sorted query path for every batch
    int ls_variant = 0;           // KS_LS_VARIANT = rep | bn | bs: bucket-sort variant of the stable path (1 / 2 / 3)
    int append_fail = 0;          // KS_APPEND_FAIL = build | merge: an append fails as an allocation would, after the
                                  // batch's build (1) or after the merge kernels (2), to test that the index is restored
    void read() {
        sketch_general = getenv("KS_SKETCH_GENERAL") != nullptr;
        const char* d = getenv("KS_DENSE");
        dense = d ? (d[0] == '0' ? 0 : d[0] == '1' ? 1 : -1) : -1;
        const char* sc = getenv("KS_SCATTER");
        scatter_off = sc && sc[0] == '0';
        no_pipeline = getenv("KS_NO_PIPELINE") != nullptr;
        const char* ds = getenv("KS_DENSE_SORT");
        dense_sort_library = ds && ds[0] == 'l';
        timing = getenv("KS_TIMING") != nullptr;
        search_legacy = getenv("KS_SEARCH_LEGACY") != nullptr;
        const char* lv = getenv("KS_LS_VARIANT");
        ls_variant = !lv ? 0 : lv[0] == 'r' ? 1 : (lv[0] == 'b' && lv[1] == 's') ? 3 : lv[0] == 'b' ? 2 : 0;
        const char* af = getenv("KS_APPEND_FAIL");
        append_fail = !af ? 0 : af[0] == 'b' ? 1 : af[0] == 'm' ? 2 : 0;
    }
};

struct ks_index {
    ks_params params{};
    Hooks hooks;
    uint64_t max_hash = 0;
    int lz = 0;  // known-zero leading bits of every kept hash
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;  // H2D of residue chunks while earlier tiles are being hashed
    cudaEvent_t ev_chunk[17] = {};
    cudaEvent_t ev[13] = {};
    uint64_t live_bytes = 0;
    Arena* arena = nullptr;

    DeviceBatch batch, qbatch;
    Build state = Build::Tuples;
    // tuples
    uint64_t *d_hash = nullptr, *d_loc = nullptr;
    uint64_t cap = 0, n_tuples = 0;
    uint64_t n_prot = 0, n_res = 0, n_windows = 0;
    uint64_t* d_status = nullptr;  // StatusBlock
    uint64_t* d_count = nullptr;   // d_status + 2
    void* ws = nullptr;
    size_t ws_bytes = 0;
    // dense k-mer space path (hp, 8 <= k <= 24, scaled == 1): per-handle rank tables; a batch that qualifies is not
    // sketched when it is added but built as a whole by finalize (Build::DenseDeferred)
    int dense_state = 0;  // 0: tables not built, 1: ready, -1: unusable for this k (two patterns share a hash)
    uint32_t* dense_code = nullptr;   // pattern -> order-preserving code (DenseSketchArgs, sketch.cuh)
    uint64_t* dense_hash = nullptr;   // the patterns' hashes in increasing order
    uint32_t* dense_group = nullptr;  // first entry of every 16-bit hash-prefix group
    int dense_rb_full = 0;            // bits of a code below the hash prefix, parity bit included
    int dense_rb = 0, dense_parity = 1;   // layout of this build: rb = dense_rb_full - (1 - parity)
    int dense_table_parity = -1;      // layout the code table currently holds
    uint32_t* dense_por = nullptr;    // pattern of every rank (to rebuild the code table in the other layout)
    uint32_t* dense_flags = nullptr;  // device u32[4], table build: [0] table check, [3] largest rank of a pattern inside
                                      // its prefix group
    Buf b_dense_code, b_dense_hash, b_dense_group, b_dense_por, b_dense_flags, b_dense_work;
    PairSortPlan pair_plan;  // of a scattered batch
    Buf b_pair_work;
    uint32_t build_path = 0;  // ks_stats.build_path of the last finalize (ks_index_clear keeps it)
    DenseSortPlan dense_plan;
    int dense_pid_bits = 0, dense_pos_bits = 0;
    Csr csr;
    Buf b_keys, b_key_grp, b_grp_start, b_t_size, b_t_abund, b_dir, b_alt_hash, b_alt_loc, b_temp;
    // append: the index lives in the build's buffers (home -1) or in app[home]; scratch of the merge (compact copies of
    // segmented inputs, the per-key insertion points)
    CsrSet app[2];
    int home = -1;
    bool appended = false;  // the index holds batches merged by ks_index_append_* (no sharded search)
    Buf b_ca_keys, b_ca_kg, b_ca_gs, b_ca_dir, b_cb_keys, b_cb_kg, b_cb_gs, b_m_pre, b_m_counts, b_m_work;
    // query path: per-handle scratch (grow-only) and a pinned word block for the counts the host reads back
    Buf b_q_ecount, b_q_pcount, b_q_hcount, b_q_sig, b_q_poff, b_q_hoff, b_q_ent_hash, b_q_ent_abund, b_q_win_key,
        b_q_win_hoff, b_q_stage, b_q_totals;
    uint64_t* h_words = nullptr;  // pinned u64[H_WORDS]
    // bookkeeping
    uint64_t l_sketch = 0, l_sort = 0, l_csr = 0, l_search = 0;
    bool t_upload = false, t_sketch = false, t_sort = false, t_csr = false;
    float ms_search = 0;

    void use() { KS_CUDA(cudaSetDevice(params.device)); }
    int end_bit() const { return 64 - lz; }
    bool finalized() const { return state == Build::Finalized; }
};

namespace {

enum { EV_UP0, EV_UP1, EV_SK0, EV_SK1, EV_SO0, EV_SO1, EV_CS0, EV_CS1, EV_Q0, EV_Q1, EV_PART, EV_M0, EV_M1 };
// pinned words of a handle: [0, QT_WORDS) totals of the query kernels; then this rank's header of a sharded search;
// then every rank's header
enum { HW_TOTALS = 0, HW_HDR = QT_WORDS, HW_ALL = QT_WORDS + 8, H_WORDS = QT_WORDS + 8 + 4 * MAX_SHARDS };
static_assert(sizeof(StatusBlock) == 48 && sizeof(StatusBlock) <= QT_WORDS * 8, "the status block is read into the totals words");

void ensure_ws(ks_index* x, size_t bytes) {
    if (bytes <= x->ws_bytes) return;
    if (x->ws) x->arena->release(x->ws);
    x->ws = x->arena->alloc<char>(bytes);
    x->ws_bytes = bytes;
}

// Buffers and shape of batch b for proteome p, its residues as 5-bit codes when `packed`; the caller copies the data in.
void reserve_batch(ks_index* x, DeviceBatch& b, const ks_proteome* p, bool packed) {
    if (p->n_prot >= 0xffffffffull) fail(KS_ERR_CAPACITY, "more than 2^32-2 proteins in one batch");
    b.packed = packed;
    b.n_prot = p->n_prot;
    b.n_res = p->n_res;
    b.res = b.b_res.ensure<uint8_t>(x->arena, b.res_bytes());
    b.offs = b.b_offs.ensure<uint64_t>(x->arena, p->n_prot + 1);
    proteome_shape(p, x->params.ksize, &b.n_windows, &b.max_len);
    b.valid = true;
}

void upload_batch(ks_index* x, DeviceBatch& b, const ks_proteome* p, bool allow_packed = false) {
    reserve_batch(x, b, p, allow_packed && p->packed && x->params.ksize <= (uint32_t)SK_MAX_TEMPLATE_K);
    KS_CUDA(cudaMemcpyAsync(b.res, b.packed ? p->packed : p->residues, b.res_bytes(), cudaMemcpyHostToDevice, x->stream));
    KS_CUDA(cudaMemcpyAsync(b.offs, p->offsets, (p->n_prot + 1) * 8, cudaMemcpyHostToDevice, x->stream));
}

// The handle holds nothing afterwards (ks_index_clear, and a pending batch about to be sketched again).  The buffers stay
// with the handle (grow-only), and so does build_path.
void drop_content(ks_index* x) {
    x->state = Build::Tuples;
    x->csr = Csr();
    x->home = -1;
    x->appended = false;
    x->n_tuples = x->n_prot = x->n_res = x->n_windows = 0;
}

// The resident batch has been added with n tuples and the handle now holds `state`: the one place a batch is counted.
void commit_batch(ks_index* x, uint64_t n, Build state) {
    const DeviceBatch& b = x->batch;
    x->state = state;
    x->n_tuples += n;
    x->n_prot += b.n_prot;
    x->n_res += b.n_res;
    x->n_windows += b.n_windows;
}

// Room for `need` tuples.  keep = false: the tuples held are dropped (the buffers may be replaced without a copy).
void grow_tuples(ks_index* x, uint64_t need, bool keep = true) {
    if (need <= x->cap) return;
    const uint64_t held = keep ? x->n_tuples : 0;
    uint64_t ncap = std::max<uint64_t>(need, held ? x->cap + x->cap / 2 : need);
    uint64_t* nh = x->arena->alloc<uint64_t>(ncap);
    uint64_t* nl = x->arena->alloc<uint64_t>(ncap);
    if (held) {
        KS_CUDA(cudaMemcpyAsync(nh, x->d_hash, held * 8, cudaMemcpyDeviceToDevice, x->stream));
        KS_CUDA(cudaMemcpyAsync(nl, x->d_loc, held * 8, cudaMemcpyDeviceToDevice, x->stream));
    }
    if (x->d_hash) x->arena->release(x->d_hash);
    if (x->d_loc) x->arena->release(x->d_loc);
    x->d_hash = nh; x->d_loc = nl; x->cap = ncap;
}

uint64_t expected_kept(const ks_index* x, uint64_t windows) {
    if (x->params.scaled <= 1) return windows;
    double e = (double)windows / (double)x->params.scaled;
    uint64_t est = (uint64_t)(e * 1.05 + 8.0 * std::sqrt(e + 1.0)) + 1024;
    return std::min(windows, est);
}

// One status block read-back: its first `bytes` (the other words keep the values of `st`), and the unstable partition's
// overflow flag into st.overflow when `part_overflow` is given.
StatusBlock read_status(ks_index* x, const StatusBlock& st, size_t bytes, const uint32_t* part_overflow = nullptr) {
    StatusBlock* h = (StatusBlock*)(x->h_words + HW_TOTALS);
    *h = st;
    KS_CUDA(cudaMemcpyAsync(h, x->d_status, bytes, cudaMemcpyDeviceToHost, x->stream));
    if (part_overflow) KS_CUDA(cudaMemcpyAsync(&h->overflow, part_overflow, 4, cudaMemcpyDeviceToHost, x->stream));
    KS_CUDA(cudaStreamSynchronize(x->stream));
    return *h;
}

// A sketch launch over batch b: everything but the output (out_hash / out_loc / capacity, or the scatter), the tile range
// and force_general, which callers set.  d_count / ws: the counter pair and workspace of the launch, the handle's own by
// default.
SketchArgs sketch_args(const ks_index* x, const DeviceBatch& b, uint32_t pid_base, uint64_t* d_count = nullptr, void* ws = nullptr) {
    SketchArgs a;
    a.residues = b.res; a.packed = b.packed ? 1 : 0; a.offsets = b.offs; a.n_res = b.n_res; a.n_prot = b.n_prot;
    a.k = x->params.ksize; a.moltype = x->params.moltype; a.max_hash = x->max_hash; a.pid_base = pid_base;
    a.out_hash = nullptr; a.out_loc = nullptr; a.capacity = 0;
    a.d_count = d_count ? d_count : x->d_count; a.workspace = d_count ? ws : x->ws;
    a.force_general = 0;
    return a;
}

// Sketch batch `b` into (out_hash, out_loc) of `capacity`; returns the number of tuples the batch produces
// (which may exceed capacity, in which case nothing past capacity was written).  d_count / ws: the counter pair and
// workspace of the launch -- the handle's own for its batches, private ones for ks_sketch_batch and the query sketch (a
// pipelined dense batch that is still pending keeps its counts in the handle's).
uint64_t run_sketch(ks_index* x, const DeviceBatch& b, uint32_t pid_base, uint64_t* out_hash, uint64_t* out_loc,
                    uint64_t capacity, uint64_t* d_count = nullptr, void* ws = nullptr) {
    if (!d_count) ensure_ws(x, sketch_workspace_bytes(b.n_res));
    SketchArgs a = sketch_args(x, b, pid_base, d_count, ws);
    a.out_hash = out_hash; a.out_loc = out_loc; a.capacity = capacity;
    a.force_general = x->hooks.sketch_general ? 1 : 0;  // test hook: exercise the look-back path at scaled == 1
    uint64_t r[2] = {0, 0};
    for (int attempt = 0; attempt < 2; attempt++) {
        KS_CUDA(launch_sketch(a, x->stream, &x->l_sketch));
        KS_CUDA(cudaMemcpyAsync(r, a.d_count, 16, cudaMemcpyDeviceToHost, x->stream));
        KS_CUDA(cudaStreamSynchronize(x->stream));
        if ((r[1] >> 32) == 0) break;  // no zero hash on the exact path
        a.force_general = 1;           // a hash of exactly 0 must be dropped: redo on the look-back path
    }
    return r[0];
}

int bits_for_value(uint64_t v) {  // bits needed to hold values 0 .. v
    int b = 1;
    while (b < 64 && (v >> b)) b++;
    return b;
}

// Dense k-mer space path (sketch_dense_kernel): the batch must be the index's only content, its k-mer space small and
// well covered (otherwise the tables cost more than they save), and rank | protein | position must fit 64 bits.
// KS_DENSE=0 switches the path off, KS_DENSE=1 drops the coverage condition (test hooks).
bool dense_eligible(const ks_index* x, const DeviceBatch& b) {
    if (x->hooks.dense == 0) return false;
    const uint32_t k = x->params.ksize;
    if (x->params.moltype != KS_HP || k < (uint32_t)DENSE_MIN_K || k > (uint32_t)DENSE_MAX_K || x->max_hash != ~0ull) return false;
    if (x->dense_state < 0 || x->n_prot || x->n_tuples || b.n_prot == 0 || b.n_res >= (1ull << 32)) return false;
    if (x->hooks.dense != 1 && b.n_windows < (1ull << k) / 4) return false;
    // a key is code | protein | position; the code takes DENSE_PREFIX_BITS + rb bits (rb is known once the tables exist:
    // at most k + 1 when every pattern shared one hash prefix)
    // (without the parity bit -- then a window without a pattern sends the batch to the general path -- one bit less)
    int rb_full = x->dense_rb_full;
    if (x->dense_state != 1) {  // tables not built yet: the largest prefix group is about lambda + 6 sqrt(lambda) patterns
        const double lambda = k > (uint32_t)DENSE_PREFIX_BITS ? std::ldexp(1.0, (int)k - DENSE_PREFIX_BITS) : 1.0;
        rb_full = bits_for_value((uint64_t)(2.0 * (lambda + 6.0 * std::sqrt(lambda) + 4.0) + 2.0));
    }
    const int code_bits = DENSE_PREFIX_BITS + rb_full - 1;
    return code_bits + bits_for_value(b.n_prot - 1) + bits_for_value(b.max_len) <= 64;
}

// tuples per possible hash: distinct k-mers under this alphabet (hp k=24 has 2^24 of them for ~2*10^8 tuples on C2)
double avg_postings(const ks_index* x, uint64_t n) {
    const double alphabet = x->params.moltype == KS_HP ? 2.0 : x->params.moltype == KS_DAYHOFF ? 6.0 : 20.0;
    const double space = std::pow(alphabet, (double)x->params.ksize) / (double)x->params.scaled;
    return (double)n / space;
}
bool repeat_heavy(const ks_index* x, uint64_t n) { return avg_postings(x, n) > 0.25; }

// Unstable partition of the general path (dense_scatter.cuh, PairSortPlan): the batch is the index's only content, hashes
// rarely repeat (the bucket sort orders equal hashes by loc, pair by pair) and the tuple count fits two scatter levels.  KS_SCATTER=0 switches it off (test hook).
bool scatter_eligible(const ks_index* x, const DeviceBatch& b, PairSortPlan* plan) {
    if (x->hooks.scatter_off) return false;
    if (x->params.ksize > (uint32_t)SK_MAX_TEMPLATE_K || x->hooks.sketch_general) return false;
    if (x->n_prot || x->n_tuples || b.n_prot == 0 || b.n_windows > MAX_TUPLES) return false;
    const uint64_t n_est = expected_kept(x, b.n_windows);  // exact for scaled == 1
    // measured: with hashes that repeat the stable path wins -- the C4 slice (protein k7 scaled 10, every hash twice on
    // average) takes 4.5 ms in the bin kernel with loc tie-breaks against 2.8 ms in the two-pass stable bucket sort
    if (repeat_heavy(x, n_est)) return false;
    *plan = pair_sort_plan(n_est, x->end_bit(), x->max_hash);
    return plan->custom != 0;
}

// How a batch of this shape is added to the handle, by the resident and the pipelined add alike: the dense k-mer space
// path, the unstable partition of the general path (*plan), or the ordered sketch.
enum class Route { Dense, Scatter, Ordered };
Route choose_route(const ks_index* x, const DeviceBatch& b, PairSortPlan* plan) {
    const bool dense = dense_eligible(x, b);
    if (x->hooks.timing) fprintf(stderr, "[ks] dense eligible: %d (state %d, prot before %llu, tuples before %llu, windows %llu)\n", (int)dense,
                                 x->dense_state, (unsigned long long)x->n_prot, (unsigned long long)x->n_tuples,
                                 (unsigned long long)b.n_windows);
    if (dense) return Route::Dense;
    return scatter_eligible(x, b, plan) ? Route::Scatter : Route::Ordered;
}

void scatter_args(ks_index* x, SketchArgs* a) {
    const PairSortPlan& pl = x->pair_plan;
    char* w = (char*)x->b_pair_work.p;
    a->scatter.out_key = (uint64_t*)(w + pl.off_r1_hash);
    a->scatter.out_val = (uint64_t*)(w + pl.off_r1_loc);
    a->scatter.cursor = (uint32_t*)(w + pl.off_cursor1);
    a->scatter.cap = pl.cap1;
    a->scatter.shift = 64 - pl.l1;
    a->scatter.bits = pl.l1;
    a->scatter.lz = x->lz;
    a->scatter.overflow = (uint32_t*)(w + pl.off_overflow);
    a->t_abund = x->max_hash != ~0ull ? (uint32_t*)x->b_t_abund.p : nullptr;
}

void scatter_begin(ks_index* x, const PairSortPlan& plan, uint64_t n_prot) {
    x->pair_plan = plan;
    char* w = x->b_pair_work.ensure<char>(x->arena, plan.bytes);
    KS_CUDA(cudaMemsetAsync(w + plan.off_small, 0, plan.small_bytes, x->stream));
    if (x->max_hash != ~0ull) {  // scaled > 1: the sketch kernel counts the kept windows per protein (finalize's t_abund)
        uint32_t* t_abund = x->b_t_abund.ensure<uint32_t>(x->arena, n_prot);
        KS_CUDA(cudaMemsetAsync(t_abund, 0, n_prot * 4, x->stream));
    }
}

bool dense_begin(ks_index* x);
void dense_rank_tiles(ks_index* x, uint32_t t0, uint32_t t1);

// Ordered route: the resident batch (valid, the handle not finalized) sketched in (protein, pos) order behind the
// tuples the handle holds.
void sketch_ordered(ks_index* x) {
    DeviceBatch& b = x->batch;
    if (x->n_prot + b.n_prot >= 0xffffffffull) fail(KS_ERR_CAPACITY, "more than 2^32-2 proteins on one shard");
    grow_tuples(x, x->n_tuples + expected_kept(x, b.n_windows));
    KS_CUDA(cudaEventRecord(x->ev[EV_SK0], x->stream));
    uint64_t n = run_sketch(x, b, (uint32_t)x->n_prot, x->d_hash + x->n_tuples, x->d_loc + x->n_tuples, x->cap - x->n_tuples);
    if (n > x->cap - x->n_tuples) {  // estimate for scaled > 1 was short: grow to the exact size and redo
        grow_tuples(x, x->n_tuples + n);
        KS_CUDA(cudaEventRecord(x->ev[EV_SK0], x->stream));
        n = run_sketch(x, b, (uint32_t)x->n_prot, x->d_hash + x->n_tuples, x->d_loc + x->n_tuples, x->cap - x->n_tuples);
    }
    KS_CUDA(cudaEventRecord(x->ev[EV_SK1], x->stream));
    x->t_sketch = true;
    commit_batch(x, n, Build::Tuples);
}

// A pending batch is sketched again, in order: something else is about to touch the tuples or the resident batch, or
// finalize found that its route does not apply after all.
void materialize_pending(ks_index* x) {
    if (x->state == Build::Tuples || x->finalized()) return;
    drop_content(x);
    sketch_ordered(x);
}

// Scatter route, after the sketch kernel: r = its count and zero-hash flag, or nullptr when they are read by finalize
// (scaled == 1).  A zero hash on the exact path (it must be dropped), or more tuples than the partition takes, sends the
// batch to the ordered route.
void scatter_done(ks_index* x, const uint64_t* r) {
    const DeviceBatch& b = x->batch;
    if (!r) return commit_batch(x, b.n_windows, Build::ScatteredUnchecked);
    const bool exact = x->max_hash == ~0ull;
    if (exact ? ((r[1] >> 32) != 0 || r[0] != b.n_windows) : r[0] > MAX_TUPLES) return sketch_ordered(x);
    commit_batch(x, r[0], Build::Scattered);
}

void sketch_resident(ks_index* x) {
    DeviceBatch& b = x->batch;
    if (!b.valid) fail(KS_ERR_VALIDATION, "Validation error: no batch is resident (call ks_index_upload first)");
    if (x->finalized()) fail(KS_ERR_VALIDATION, "Validation error: index is finalized; ks_index_clear before adding more");
    materialize_pending(x);  // the resident batch was already added once and is being added again
    PairSortPlan plan;
    const Route route = choose_route(x, b, &plan);
    if (route == Route::Dense) return commit_batch(x, b.n_windows, Build::DenseDeferred);  // finalize builds it in one go
    if (route == Route::Ordered) return sketch_ordered(x);
    scatter_begin(x, plan, b.n_prot);
    ensure_ws(x, sketch_workspace_bytes(b.n_res));
    SketchArgs a = sketch_args(x, b, 0);
    scatter_args(x, &a);
    KS_CUDA(cudaEventRecord(x->ev[EV_SK0], x->stream));
    KS_CUDA(launch_sketch(a, x->stream, &x->l_sketch));
    KS_CUDA(cudaEventRecord(x->ev[EV_SK1], x->stream));
    x->t_sketch = true;
    // scaled == 1: the tuple count is known from the offsets; the kernel's own count and its zero-hash flag are read
    // together with the build's results at the end of finalize (no host round trip here)
    if (x->max_hash == ~0ull) return scatter_done(x, nullptr);
    uint64_t r[2] = {0, 0};
    KS_CUDA(cudaMemcpyAsync(r, x->d_count, 16, cudaMemcpyDeviceToHost, x->stream));
    KS_CUDA(cudaStreamSynchronize(x->stream));
    scatter_done(x, r);
}

// upload + sketch with the residues streamed in: the offsets go first (everything the tile -> protein map and
// the exact tile bases need), then the residues in chunks on the copy stream; the fused kernel runs over the
// tile range of a chunk as soon as that chunk has landed.  On the exact path (scaled == 1) tile bases are known
// before any hash; on the look-back path (scaled > 1) tiles are taken by ticket, which simply continues across the
// chunk launches.  Returns false when the batch does not qualify (caller takes upload + sketch_resident).
bool add_proteome_pipelined(ks_index* x, const ks_proteome* p) {
    constexpr int CHUNKS = 16;  // (the last chunk's kernel is all that is not hidden behind the copy)
    if (x->params.ksize > (uint32_t)SK_MAX_TEMPLATE_K || x->hooks.no_pipeline)  // (test hook)
        return false;
    if (p->n_res < (64u << 20) || p->n_prot == 0) return false;  // small batches: one copy, one launch
    if (x->finalized()) fail(KS_ERR_VALIDATION, "Validation error: index is finalized; ks_index_clear before adding more");
    materialize_pending(x);
    if (x->n_prot + p->n_prot >= 0xffffffffull) fail(KS_ERR_CAPACITY, "more than 2^32-2 proteins on one shard");
    DeviceBatch& b = x->batch;
    reserve_batch(x, b, p, p->packed != nullptr);  // 5 bits per residue over PCIe instead of 8
    PairSortPlan plan;
    Route route = choose_route(x, b, &plan);  // dense: the rank kernel follows the chunks instead of the sketch kernel
    const uint8_t* host_res = b.packed ? p->packed : p->residues;
    const uint64_t res_bytes = b.res_bytes();
    const uint64_t tile_bytes = b.packed ? SK_TILE / 8 * 5 : SK_TILE;
    if (route == Route::Ordered) grow_tuples(x, x->n_tuples + expected_kept(x, b.n_windows));
    if (route == Route::Scatter) scatter_begin(x, plan, p->n_prot);
    ensure_ws(x, sketch_workspace_bytes(b.n_res));
    KS_CUDA(cudaEventRecord(x->ev[EV_UP0], x->stream));
    KS_CUDA(cudaEventRecord(x->ev[EV_SK0], x->stream));
    KS_CUDA(cudaMemcpyAsync(b.offs, p->offsets, (p->n_prot + 1) * 8, cudaMemcpyHostToDevice, x->stream));
    if (route == Route::Dense && !dense_begin(x)) {  // the tables turned out unusable for this k: the ordered route after all
        route = Route::Ordered;
        grow_tuples(x, x->n_tuples + expected_kept(x, b.n_windows));
    }
    // buffers were (re)allocated in compute-stream order: the copy stream must not run ahead of that
    KS_CUDA(cudaEventRecord(x->ev_chunk[CHUNKS], x->stream));
    KS_CUDA(cudaStreamWaitEvent(x->copy_stream, x->ev_chunk[CHUNKS], 0));
    SketchArgs a = sketch_args(x, b, (uint32_t)x->n_prot);
    a.force_general = x->hooks.sketch_general ? 1 : 0;  // test hook: the look-back path at scaled == 1
    if (route == Route::Scatter) {
        scatter_args(x, &a);
    } else {
        a.out_hash = x->d_hash + x->n_tuples; a.out_loc = x->d_loc + x->n_tuples; a.capacity = x->cap - x->n_tuples;
    }
    if (route != Route::Dense) KS_CUDA(launch_sketch_prepare(a, x->stream, &x->l_sketch));  // (dense_begin has done it)
    const uint64_t nt = (b.n_res + SK_TILE - 1) / SK_TILE;
    const uint64_t per = (nt + CHUNKS - 1) / CHUNKS;
    for (int c = 0; c < CHUNKS; c++) {
        const uint64_t t0 = (uint64_t)c * per, t1 = std::min<uint64_t>(nt, t0 + per);
        if (t0 >= t1) break;
        const uint64_t byte0 = t0 * tile_bytes;
        const uint64_t byte1 = std::min<uint64_t>(res_bytes, t1 * tile_bytes + 64);  // halo of the last tile included
        KS_CUDA(cudaMemcpyAsync(b.res + byte0, host_res + byte0, byte1 - byte0, cudaMemcpyHostToDevice, x->copy_stream));
        KS_CUDA(cudaEventRecord(x->ev_chunk[c], x->copy_stream));
        KS_CUDA(cudaStreamWaitEvent(x->stream, x->ev_chunk[c], 0));
        a.tile_begin = (uint32_t)t0; a.tile_end = (uint32_t)t1;
        if (route == Route::Dense) dense_rank_tiles(x, (uint32_t)t0, (uint32_t)t1);
        else KS_CUDA(launch_sketch_tiles(a, x->stream, &x->l_sketch));
    }
    uint64_t r[2] = {0, 0};
    if (route != Route::Dense) {
        KS_CUDA(launch_sketch_finish(a, x->stream));
        KS_CUDA(cudaMemcpyAsync(r, x->d_count, 16, cudaMemcpyDeviceToHost, x->stream));
    }
    KS_CUDA(cudaEventRecord(x->ev[EV_UP1], x->stream));
    KS_CUDA(cudaEventRecord(x->ev[EV_SK1], x->stream));
    KS_CUDA(cudaStreamSynchronize(x->stream));
    x->t_upload = x->t_sketch = true;
    if (route == Route::Dense) commit_batch(x, b.n_windows, Build::DenseRanked);  // finalize takes it from here
    else if (route == Route::Scatter) scatter_done(x, r);
    // a zero hash on the exact path, or more tuples than the estimate for scaled > 1 allowed for: redo the batch (now
    // resident) on the ordered route, which takes the look-back kernel / grows the buffer as needed
    else if ((r[1] >> 32) != 0 || r[0] > x->cap - x->n_tuples) sketch_ordered(x);
    else commit_batch(x, r[0], Build::Tuples);
    return true;
}

// ---- dense path (sketch_dense_kernel, dense.cu) -------------------------------------------------------------------
void dense_kernel_args(ks_index* x, SketchArgs* a, DenseSketchArgs* d) {
    const DenseSortPlan& plan = x->dense_plan;
    *a = sketch_args(x, x->batch, 0);
    a->capacity = x->cap;
    d->code_of_pattern = x->dense_code; d->out_keys = x->d_hash; d->pid_bits = x->dense_pid_bits; d->pos_bits = x->dense_pos_bits;
    d->sorted_hash = x->dense_hash; d->group_base = x->dense_group; d->rb = x->dense_rb; d->parity = x->dense_parity;
    d->exception_flag = (uint32_t*)(x->d_status + 4);
    // the library-sorted variant and the layout without the parity bit have no exception handling: general path then
    d->handle_exceptions = plan.custom && x->dense_parity ? 1 : 0;
    d->scatter = DenseScatter{nullptr, nullptr, 0, 0, 0, nullptr};
    if (plan.custom) {
        char* work = (char*)x->b_dense_work.p;
        d->scatter.out = (uint64_t*)(work + plan.off_region1);
        d->scatter.cursor = (uint32_t*)(work + plan.off_cursor1);
        d->scatter.cap = plan.cap1;
        d->scatter.shift = DENSE_PREFIX_BITS + x->dense_rb + x->dense_pid_bits + x->dense_pos_bits - plan.l1;
        d->scatter.bits = plan.l1;
        d->scatter.overflow = (uint32_t*)(x->d_status + 5);
        a->unordered = 1;
    }
    a->count_zeroed = 1;  // (dense_begin zeroes the status block)
}

// Tables (first use of the handle), sort plan, buffers, tile -> protein map and exact tile bases.  The offsets of the
// batch must be on their way to the device on x->stream.  Returns false when the tables are unusable for this k.
bool dense_begin(ks_index* x) {
    DeviceBatch& b = x->batch;
    const uint32_t k = x->params.ksize;
    Arena* ar = x->arena;
    x->dense_flags = x->b_dense_flags.ensure<uint32_t>(ar, 4);
    if (x->dense_state == 0) {  // first use of the handle: the tables (two steps, one host read in between)
        x->dense_code = x->b_dense_code.ensure<uint32_t>(ar, (size_t)1 << k);
        x->dense_hash = x->b_dense_hash.ensure<uint64_t>(ar, (size_t)1 << k);
        x->dense_group = x->b_dense_group.ensure<uint32_t>(ar, ((size_t)1 << DENSE_PREFIX_BITS) + 1);
        x->dense_por = x->b_dense_por.ensure<uint32_t>(ar, (size_t)1 << k);
        const size_t tb = dense_table_temp_bytes(k);
        void* tmp = x->b_temp.ensure<char>(ar, tb);
        KS_CUDA(dense_build_tables(k, x->dense_hash, x->dense_group, x->dense_por, tmp, tb, x->dense_flags, x->stream, &x->l_sketch));
        uint32_t fl[4] = {0, 0, 0, 0};
        KS_CUDA(cudaMemcpyAsync(fl, x->dense_flags, 16, cudaMemcpyDeviceToHost, x->stream));
        KS_CUDA(cudaStreamSynchronize(x->stream));
        x->dense_state = fl[0] ? -1 : 1;
        x->dense_rb_full = bits_for_value(2ull * fl[3] + 2);  // even codes go up to 2 x (group size), odd ones to 2 x rank + 1
        if (DENSE_PREFIX_BITS + x->dense_rb_full > 32) x->dense_state = -1;  // (codes are 32-bit table entries)
        x->dense_table_parity = -1;
    }
    if (x->hooks.timing) fprintf(stderr, "[ks] dense begin: state %d rb %d\n", x->dense_state, x->dense_rb_full);
    if (x->dense_state < 0) return false;
    const uint64_t n = b.n_windows;
    if (n > MAX_TUPLES) fail(KS_ERR_CAPACITY, "more than 2^31-1 tuples on one shard: shard the proteome over more GPUs");
    x->dense_pid_bits = bits_for_value(b.n_prot - 1);
    x->dense_pos_bits = bits_for_value(b.max_len);
    grow_tuples(x, n, false);  // d_hash: the keys when the library sorts them; d_loc: the postings
    // the key sort: hand-written (two scatter levels + a shared-memory sort per bucket) when the input fits its scheme,
    // the library's otherwise (KS_DENSE_SORT=library is a test hook)
    // layout of the keys: with the parity bit (exception windows handled) when code | protein | position fits 64 bits
    const int loc_bits = x->dense_pid_bits + x->dense_pos_bits;
    if (DENSE_PREFIX_BITS + x->dense_rb_full + loc_bits <= 64) x->dense_parity = 1;
    else if (DENSE_PREFIX_BITS + x->dense_rb_full - 1 + loc_bits <= 64) x->dense_parity = 0;
    else return false;  // (the estimate of dense_eligible was short)
    x->dense_rb = x->dense_rb_full - (1 - x->dense_parity);
    if (x->dense_table_parity != x->dense_parity) {
        KS_CUDA(dense_build_codes(k, x->dense_hash, x->dense_group, x->dense_por, x->dense_rb, x->dense_parity, x->dense_code, x->stream,
                                  &x->l_sketch));
        x->dense_table_parity = x->dense_parity;
    }
    const int code_bits = DENSE_PREFIX_BITS + x->dense_rb;
    x->dense_plan = x->hooks.dense_sort_library ? DenseSortPlan()
                                                : dense_sort_plan(n, code_bits, code_bits + x->dense_pid_bits + x->dense_pos_bits, (int)k);
    if (x->dense_plan.custom) {
        char* work = x->b_dense_work.ensure<char>(ar, x->dense_plan.bytes);
        KS_CUDA(cudaMemsetAsync(work + x->dense_plan.off_small, 0, x->dense_plan.small_bytes, x->stream));
    }
    ensure_ws(x, sketch_workspace_bytes(b.n_res));
    SketchArgs a;
    DenseSketchArgs d;
    dense_kernel_args(x, &a, &d);
    KS_CUDA(cudaMemsetAsync(x->d_status, 0, 64, x->stream));  // totals, count, flags, overflow: one memset, one read at the end
    KS_CUDA(launch_sketch_prepare(a, x->stream, &x->l_sketch));
    return true;
}

// The rank kernel over tiles [t0, t1) of the resident batch (0, 0 = all).
void dense_rank_tiles(ks_index* x, uint32_t t0, uint32_t t1) {
    SketchArgs a;
    DenseSketchArgs d;
    dense_kernel_args(x, &a, &d);
    a.tile_begin = t0; a.tile_end = t1;
    KS_CUDA(launch_sketch_dense(a, d, x->stream, &x->l_sketch));
}

// The CSR's buffers for n tuples of P proteins.  The directory has about 4 tuples (<= 4 keys) per bucket, so that it stays
// small next to the keys, and at least the 2^top_bits buckets of the key sort (a directory bucket must not span two of
// them); the key, group and directory arrays get `slack` more slots.
int dir_bits_for(uint64_t n) {
    int bits = 8;
    while (bits < 24 && (4ull << bits) < n) bits++;
    return bits;
}

Csr reserve_csr(ks_index* x, uint64_t n, uint32_t P, int top_bits, uint64_t slack) {
    Arena* ar = x->arena;
    Csr c;
    c.dir_bits = std::max(dir_bits_for(n), top_bits);
    c.dir_shift = 64 - x->lz - c.dir_bits;
    c.t_abund = x->b_t_abund.ensure<uint32_t>(ar, P);
    c.t_size = x->b_t_size.ensure<uint32_t>(ar, P);
    c.keys = x->b_keys.ensure<uint64_t>(ar, n + slack);
    c.key_grp = x->b_key_grp.ensure<uint32_t>(ar, n + slack);
    c.grp_start = x->b_grp_start.ensure<uint32_t>(ar, n + slack);
    c.dir = x->b_dir.ensure<uint32_t>(ar, (1ull << c.dir_bits) + slack);
    c.d_counts = x->d_status;
    return c;
}

// Build the index of the pending batch on the dense path.  Returns false (nothing changed that matters) when the path
// turns out not to apply: the tables are unusable for this k, a window holds a residue of neither hp class, or heavy
// repeats of one k-mer overflowed a sort bucket.
bool dense_finalize(ks_index* x) {
    DeviceBatch& b = x->batch;
    const uint32_t k = x->params.ksize;
    Arena* ar = x->arena;
    if (x->state == Build::DenseDeferred) {
        KS_CUDA(cudaEventRecord(x->ev[EV_SK0], x->stream));
        if (!dense_begin(x)) return false;
        dense_rank_tiles(x, 0, 0);
        KS_CUDA(cudaEventRecord(x->ev[EV_SK1], x->stream));
    }
    const uint64_t n = b.n_windows;
    const uint32_t P = (uint32_t)b.n_prot;
    const DenseSortPlan plan = x->dense_plan;
    char* work = (char*)x->b_dense_work.p;
    // No host round trip between the rank kernel and the CSR: the kernels read the rank kernel's flags on the device, and
    // everything the host has to know (flags, counts, overflow) comes back in ONE read at the end.
    const uint64_t slack = (plan.custom ? (1ull << plan.total) : 0) + 2;  // segmented layout: a sentinel slot per bucket
    Csr cs = reserve_csr(x, n, P, plan.custom ? plan.total : 0, slack);
    DenseCsrArgs c;
    c.dir = cs.dir; c.dir_bits = cs.dir_bits;
    c.out_dir_sub = &cs.dir_sub; c.out_seg_nb = &cs.seg_nb; c.out_seg_start = &cs.seg_start; c.out_seg_counts = &cs.seg_counts;
    c.plan = plan; c.work = work;
    c.keys_a = x->d_hash; c.keys_b = plan.custom ? nullptr : x->b_alt_hash.ensure<uint64_t>(ar, n);
    c.n = n; c.n_prot = P; c.k = k;
    c.rank_bits = DENSE_PREFIX_BITS + x->dense_rb; c.rb = x->dense_rb; c.parity = x->dense_parity;
    c.pid_bits = x->dense_pid_bits; c.pos_bits = x->dense_pos_bits;
    c.offsets = b.offs; c.sorted_hash = x->dense_hash; c.group_base = x->dense_group;
    c.residues = b.res; c.packed = b.packed ? 1 : 0;
    c.skip_flag = (uint32_t*)(x->d_status + 4); c.exc_flag = c.skip_flag + 1; c.overflow = (uint32_t*)(x->d_status + 5);
    c.counts_zeroed = 1;
    c.loc = x->d_loc; c.keys = cs.keys; c.key_grp = cs.key_grp; c.grp_start = cs.grp_start;
    c.t_size = cs.t_size; c.t_abund = cs.t_abund; c.d_counts = cs.d_counts;
    c.temp_bytes = dense_csr_temp_bytes(n);
    c.temp = x->b_temp.ensure<char>(ar, c.temp_bytes);
    c.ev_sorted = x->ev[EV_PART];
    KS_CUDA(cudaEventRecord(x->ev[EV_SO0], x->stream));
    KS_CUDA(dense_build_csr(c, x->stream, &x->l_sort, &x->l_csr));
    KS_CUDA(cudaEventRecord(x->ev[EV_SO1], x->stream));
    if (cs.dir_sub == DIR_SUB_COMPACT) {  // library-sorted keys: compact layout, the directory in its own pass
        KS_CUDA(launch_directory(cs.keys, cs.d_counts, cs.dir, cs.dir_bits, cs.dir_shift, x->stream));
        x->l_csr += 1;
    }
    KS_CUDA(cudaEventRecord(x->ev[EV_CS1], x->stream));
    x->t_sketch = x->t_sort = x->t_csr = true;
    const StatusBlock st = read_status(x, StatusBlock{}, sizeof(StatusBlock));
    const uint32_t unhandled = (uint32_t)st.dense_flags;  // an exception the path does not handle, or a zero hash
    if (x->hooks.timing)
        fprintf(stderr, "[ks] dense finalize: n %llu produced %llu unhandled %u exc %u overflow %u U %llu G %llu plan l1 %d l2 %d rb %d\n",
                (unsigned long long)n, (unsigned long long)st.produced, unhandled, (uint32_t)(st.dense_flags >> 32),
                (uint32_t)st.overflow, (unsigned long long)st.U, (unsigned long long)st.G, plan.l1, plan.l2, x->dense_rb);
    if (unhandled) return false;
    if (st.produced != n) fail(KS_ERR_CUDA, "internal error: dense path produced an unexpected number of tuples");
    if ((uint32_t)st.overflow) return false;  // heavy repeats of one k-mer overflowed a sort bucket: the general path handles those
    cs.U = st.U; cs.G = st.G;
    cs.hash_col_valid = false;  // d_hash holds code keys: the sorted hash column is rebuilt from the CSR on demand
    cs.hash = x->d_hash; cs.loc = x->d_loc;
    x->csr = cs;
    x->build_path = plan.custom ? 1u : 2u;
    x->state = Build::Finalized;
    return true;
}

void finalize(ks_index* x) {
    if (x->finalized()) return;
    if (x->state == Build::DenseDeferred || x->state == Build::DenseRanked) {
        if (dense_finalize(x)) return;
        materialize_pending(x);  // not applicable after all: the general path from here on
    }
    const bool dbg = x->hooks.timing;
    double t0 = dbg ? wall_ms() : 0;
    const uint64_t n = x->n_tuples;
    if (n > MAX_TUPLES) fail(KS_ERR_CAPACITY, "more than 2^31-1 tuples on one shard: shard the proteome over more GPUs");
    const uint32_t P = (uint32_t)x->n_prot;
    const bool scattered = x->state == Build::Scattered || x->state == Build::ScatteredUnchecked;
    // the bucket sort writes the CSR in the segmented layout: a directory bucket must not span two sort buckets, and the
    // key / group arrays carry one sentinel slot per sort bucket
    const int top_bits = scattered ? x->pair_plan.total : build_top_bits(n, x->end_bit(), x->max_hash, avg_postings(x, n));
    const uint64_t slack = std::max<uint64_t>(build_slack(n), top_bits > 0 ? (1ull << top_bits) + 2 : 2);
    Csr cs = reserve_csr(x, n, P, top_bits, slack);
    Arena* ar = x->arena;
    // the second tuple pair is the sort's ping-pong partner; a scattered batch has its regions instead
    uint64_t* hb = scattered ? nullptr : x->b_alt_hash.ensure<uint64_t>(ar, n);
    uint64_t* lb = scattered ? nullptr : x->b_alt_loc.ensure<uint64_t>(ar, n);
    if (scattered) grow_tuples(x, n, false);  // the tuples sit in the regions of the unstable partition; the postings go to d_loc
    BuildArgs a;
    a.hash_a = x->d_hash; a.loc_a = x->d_loc; a.hash_b = hb; a.loc_b = lb;
    a.n = n; a.n_prot = P; a.end_bit = x->end_bit(); a.max_hash = x->max_hash;
    a.repeat_heavy = repeat_heavy(x, n) ? 1 : 0;  // measured: the bin kernel only wins when repeats are rare
    a.ls_variant = x->hooks.ls_variant;
    a.avg_postings = avg_postings(x, n);
    a.out_dir_sub = &cs.dir_sub; a.out_seg_nb = &cs.seg_nb; a.out_seg_start = &cs.seg_start; a.out_seg_counts = &cs.seg_counts;
    const uint32_t* d_overflow = nullptr;  // device flag of the unstable partition (a region overflowed)
    if (scattered) {
        a.plan = x->pair_plan; a.work = x->b_pair_work.p; a.offsets = x->batch.offs; a.k = x->params.ksize;
        a.overflow_dev = &d_overflow;
        a.abund_ready = x->max_hash != ~0ull ? 1 : 0;
    }
    a.keys = cs.keys; a.key_grp = cs.key_grp; a.grp_start = cs.grp_start; a.t_size = cs.t_size; a.t_abund = cs.t_abund;
    a.d_counts = cs.d_counts; a.dir = cs.dir; a.dir_bits = cs.dir_bits; a.dir_shift = cs.dir_shift;
    a.temp_bytes = build_temp_bytes(n, x->end_bit());
    a.temp = x->b_temp.ensure<char>(ar, a.temp_bytes);
    a.ev_sorted = x->ev[EV_SO1];
    a.ev_partitioned = x->ev[EV_PART];
    int in_a = 1, hash_written = 1;
    a.hash_written = &hash_written;
    double t1 = dbg ? wall_ms() : 0;
    KS_CUDA(cudaEventRecord(x->ev[EV_SO0], x->stream));
    KS_CUDA(build_index(a, x->stream, &in_a, &x->l_sort, &x->l_csr));
    KS_CUDA(cudaEventRecord(x->ev[EV_CS1], x->stream));
    double t2 = dbg ? wall_ms() : 0;
    x->t_sort = x->t_csr = true;
    // everything the host has to know comes back in ONE read: the CSR totals, and for a scattered batch the partition's
    // overflow flag and (when the sketch was not checked yet) the sketch kernel's count and zero-hash flag
    StatusBlock st{};
    st.produced = n;
    st = read_status(x, st, x->state == Build::ScatteredUnchecked ? 32 : 16, d_overflow);
    if (scattered && ((uint32_t)st.overflow != 0 || st.produced != n || (st.zero_flag >> 32) != 0)) {
        // a k-mer repeated thousands of times filled a region, or a window hashed to exactly 0 (it must be dropped):
        // sketch again in order, stable partition
        materialize_pending(x);
        finalize(x);
        return;
    }
    if (!in_a) {  // the sorted tuples sit in the alternate pair: swap roles, nothing is freed
        std::swap(x->d_hash, hb); std::swap(x->d_loc, lb);
        const size_t cap_bytes = x->cap * 8;
        x->cap = x->b_alt_hash.bytes / 8;
        x->b_alt_hash.p = hb; x->b_alt_hash.bytes = cap_bytes;
        x->b_alt_loc.p = lb; x->b_alt_loc.bytes = cap_bytes;
    }
    cs.U = st.U; cs.G = st.G;
    cs.hash_col_valid = hash_written != 0;
    cs.hash = x->d_hash; cs.loc = x->d_loc;
    x->csr = cs;
    x->build_path = scattered ? 3u : 0u;
    x->state = Build::Finalized;
    if (dbg) fprintf(stderr, "[ks] finalize: alloc %.3f ms, build_index (host) %.3f ms, tail %.3f ms\n", t1 - t0, t2 - t1, wall_ms() - t2);
}

CsrView view_of(const ks_index* x) {
    const Csr& c = x->csr;
    CsrView v;
    v.hash = c.hash; v.loc = c.loc; v.keys = c.keys; v.key_grp = c.key_grp; v.grp_start = c.grp_start;
    v.t_size = c.t_size; v.t_abund = c.t_abund; v.dir = c.dir; v.d_counts = c.d_counts; v.n = x->n_tuples;
    v.n_prot = (uint32_t)x->n_prot; v.dir_bits = c.dir_bits; v.dir_shift = c.dir_shift;
    v.dir_sub = c.dir_sub; v.seg_nb = c.seg_nb; v.seg_start = c.seg_start; v.seg_counts = c.seg_counts;
    return v;
}

// The resident batch replaced by p (ks_index_upload).
void upload_resident(ks_index* x, const ks_proteome* p) {
    materialize_pending(x);  // the resident batch is about to be replaced
    KS_CUDA(cudaEventRecord(x->ev[EV_UP0], x->stream));
    upload_batch(x, x->batch, p, true);
    KS_CUDA(cudaEventRecord(x->ev[EV_UP1], x->stream));
    x->t_upload = true;
}

// ks_index_add_proteome: the pipelined add, or upload + sketch of the resident batch.
void add_proteome(ks_index* x, const ks_proteome* p) {
    if (add_proteome_pipelined(x, p)) return;
    upload_resident(x, p);
    sketch_resident(x);
}

// The postings of host tuples with protein ids local to their batch (+ pid_base); checks range and (protein, pos) order.
std::vector<uint64_t> tuple_locs(const uint32_t* pid, const uint32_t* pos, uint64_t n, uint64_t n_proteins, uint32_t pid_base) {
    std::vector<uint64_t> loc(n);
    for (uint64_t i = 0; i < n; i++) {
        if (pid[i] >= n_proteins) fail(KS_ERR_VALIDATION, "Validation error: tuple protein index out of range");
        loc[i] = ((uint64_t)(pid[i] + pid_base) << 32) | pos[i];
        if (i && loc[i] <= loc[i - 1]) fail(KS_ERR_VALIDATION, "Validation error: tuples must be ordered by (protein, pos)");
    }
    return loc;
}

// Tuples behind the ones the (not finalized) handle holds, n_proteins more proteins.
void push_tuples(ks_index* x, const uint64_t* hash, const std::vector<uint64_t>& loc, uint64_t n_proteins) {
    const uint64_t n = loc.size();
    grow_tuples(x, x->n_tuples + n);
    if (n) {
        KS_CUDA(cudaMemcpyAsync(x->d_hash + x->n_tuples, hash, n * 8, cudaMemcpyHostToDevice, x->stream));
        KS_CUDA(cudaMemcpyAsync(x->d_loc + x->n_tuples, loc.data(), n * 8, cudaMemcpyHostToDevice, x->stream));
        KS_CUDA(cudaStreamSynchronize(x->stream));
    }
    x->n_tuples += n;
    x->n_prot += n_proteins;
}

// ---- append (ks_index_append_*) -----------------------------------------------------------------------------------------
// The finalized index A is parked, the batch is built as the handle's only content by the usual routes (B), and the two
// are merged into a compact index C in the append set A does not occupy.  A failure anywhere puts A back as it was.
struct Parked {
    Csr csr;
    uint64_t n_tuples = 0, n_prot = 0, n_res = 0, n_windows = 0;
    uint32_t build_path = 0;
    int home = -1;
    bool appended = false;
};

// An index in the build's buffers moves to app[0]: its buffers are swapped with the set's (no copy), the tuple pair too;
// the segmented layout's bucket tables live in the build's scratch and are copied.  An index in an append set stays.
// Everything that can fail (the tables' allocations and copies) comes first: the swaps that follow cannot, so the index
// is either where it was or wholly in app[0] with home = 0.
void park_index(ks_index* x) {
    if (x->home >= 0) return;
    CsrSet& s = x->app[0];
    Csr& c = x->csr;
    const uint32_t* seg_start = c.seg_start;
    const uint64_t* seg_counts = c.seg_counts;
    if (c.dir_sub != DIR_SUB_COMPACT) {
        uint32_t* st = s.seg_start.ensure<uint32_t>(x->arena, (uint64_t)c.seg_nb + 1);
        uint64_t* sc = s.seg_counts.ensure<uint64_t>(x->arena, c.seg_nb);
        KS_CUDA(cudaMemcpyAsync(st, c.seg_start, ((uint64_t)c.seg_nb + 1) * 4, cudaMemcpyDeviceToDevice, x->stream));
        KS_CUDA(cudaMemcpyAsync(sc, c.seg_counts, (uint64_t)c.seg_nb * 8, cudaMemcpyDeviceToDevice, x->stream));
        seg_start = st; seg_counts = sc;
    }
    std::swap(x->b_keys, s.keys); std::swap(x->b_key_grp, s.key_grp); std::swap(x->b_grp_start, s.grp_start);
    std::swap(x->b_t_size, s.t_size); std::swap(x->b_t_abund, s.t_abund); std::swap(x->b_dir, s.dir);
    Buf h{x->d_hash, x->cap * 8}, l{x->d_loc, x->cap * 8};
    std::swap(h, s.hash); std::swap(l, s.loc);
    if (h.p && l.p) {  // the set's former pair becomes the build's tuple pair
        x->d_hash = (uint64_t*)h.p; x->d_loc = (uint64_t*)l.p; x->cap = std::min(h.bytes, l.bytes) / 8;
    } else {
        if (h.p) x->arena->release(h.p);
        if (l.p) x->arena->release(l.p);
        x->d_hash = x->d_loc = nullptr; x->cap = 0;
    }
    c.seg_start = seg_start; c.seg_counts = seg_counts;
    x->home = 0;
}

void restore_index(ks_index* x, const Parked& a) {
    x->csr = a.csr;
    x->n_tuples = a.n_tuples; x->n_prot = a.n_prot; x->n_res = a.n_res; x->n_windows = a.n_windows;
    x->build_path = a.build_path; x->home = a.home; x->appended = a.appended;
    x->state = Build::Finalized;
    try {  // the batch's build has overwritten the totals the device reads (d_counts)
        const uint64_t ug[2] = {a.csr.U, a.csr.G};
        KS_CUDA(cudaMemcpyAsync(x->d_status, ug, 16, cudaMemcpyHostToDevice, x->stream));
        KS_CUDA(cudaStreamSynchronize(x->stream));
    } catch (...) {
    }
}

// One input of the merge in the compact layout: a segmented index is compacted into scratch (keys, key_grp, grp_start).
MergeSide merge_side(ks_index* x, const Csr& c, uint64_t n, Buf& bk, Buf& bkg, Buf& bgs, uint64_t* counts) {
    MergeSide m;
    m.U = c.U; m.G = c.G; m.n = n; m.loc = c.loc;
    if (c.dir_sub == DIR_SUB_COMPACT) {
        m.keys = c.keys; m.key_grp = c.key_grp; m.grp_start = c.grp_start;
        return m;
    }
    Arena* ar = x->arena;
    uint64_t* keys = bk.ensure<uint64_t>(ar, c.U);
    uint32_t* kg = bkg.ensure<uint32_t>(ar, c.U + 1);
    uint32_t* gs = bgs.ensure<uint32_t>(ar, c.G + 1);
    uint32_t* pre = x->b_m_pre.ensure<uint32_t>(ar, 2ull * c.seg_nb);
    CsrView v;
    v.keys = c.keys; v.key_grp = c.key_grp; v.grp_start = c.grp_start; v.n = n;
    v.seg_nb = c.seg_nb; v.seg_start = c.seg_start; v.seg_counts = c.seg_counts;
    KS_CUDA(launch_compact_segmented(v, c.U, c.G, pre, keys, kg, gs, counts, x->stream, &x->l_csr));
    m.keys = keys; m.key_grp = kg; m.grp_start = gs;
    return m;
}

// A (parked) + B (the handle's finalized batch) -> C in the other append set.
void merge_appended(ks_index* x, const Parked& A, double batch_ms) {
    Arena* ar = x->arena;
    const Csr B = x->csr;
    const uint64_t n_b = x->n_tuples, p_b = x->n_prot;
    const uint64_t n = A.n_tuples + n_b, P = A.n_prot + p_b, G = A.csr.G + B.G, U_max = A.csr.U + B.U;
    if (n > MAX_TUPLES) fail(KS_ERR_CAPACITY, "more than 2^31-1 tuples on one shard: shard the proteome over more GPUs");
    const int dst = 1 - A.home;
    CsrSet& out = x->app[dst];
    uint64_t* counts = x->b_m_counts.ensure<uint64_t>(ar, 4);
    KS_CUDA(cudaEventRecord(x->ev[EV_M0], x->stream));
    const MergeSide a = merge_side(x, A.csr, A.n_tuples, x->b_ca_keys, x->b_ca_kg, x->b_ca_gs, counts);
    const MergeSide b = merge_side(x, B, n_b, x->b_cb_keys, x->b_cb_kg, x->b_cb_gs, counts + 2);
    const uint32_t* dir_a = A.csr.dir;
    if (A.csr.dir_sub != DIR_SUB_COMPACT) {  // a directory over the compacted keys (same bits)
        uint32_t* d = x->b_ca_dir.ensure<uint32_t>(ar, (1ull << A.csr.dir_bits) + 1);
        KS_CUDA(launch_directory(a.keys, counts, d, A.csr.dir_bits, A.csr.dir_shift, x->stream));
        x->l_csr += 1;
        dir_a = d;
    }
    Csr c;
    c.dir_bits = dir_bits_for(n);
    c.dir_shift = 64 - x->lz - c.dir_bits;
    c.keys = out.keys.ensure<uint64_t>(ar, U_max);
    c.key_grp = out.key_grp.ensure<uint32_t>(ar, U_max + 1);
    c.grp_start = out.grp_start.ensure<uint32_t>(ar, G + 1);
    c.t_size = out.t_size.ensure<uint32_t>(ar, P);
    c.t_abund = out.t_abund.ensure<uint32_t>(ar, P);
    c.dir = out.dir.ensure<uint32_t>(ar, (1ull << c.dir_bits) + 2);
    c.hash = out.hash.ensure<uint64_t>(ar, n);
    c.loc = out.loc.ensure<uint64_t>(ar, n);
    c.d_counts = x->d_status;
    AppendArgs m;
    m.a = a; m.b = b; m.dir_a = dir_a; m.dir_bits_a = A.csr.dir_bits; m.dir_shift_a = A.csr.dir_shift; m.p_a = (uint32_t)A.n_prot;
    m.keys = c.keys; m.key_grp = c.key_grp; m.grp_start = c.grp_start; m.loc = c.loc; m.d_counts = x->d_status;
    m.work_bytes = append_work_bytes(B.U);
    m.work = x->b_m_work.ensure<char>(ar, m.work_bytes);
    KS_CUDA(launch_append_merge(m, x->stream, &x->l_csr));
    KS_CUDA(launch_directory(c.keys, x->d_status, c.dir, c.dir_bits, c.dir_shift, x->stream));
    x->l_csr += 1;
    if (A.n_prot) {
        KS_CUDA(cudaMemcpyAsync(c.t_size, A.csr.t_size, A.n_prot * 4, cudaMemcpyDeviceToDevice, x->stream));
        KS_CUDA(cudaMemcpyAsync(c.t_abund, A.csr.t_abund, A.n_prot * 4, cudaMemcpyDeviceToDevice, x->stream));
    }
    if (p_b) {
        KS_CUDA(cudaMemcpyAsync(c.t_size + A.n_prot, B.t_size, p_b * 4, cudaMemcpyDeviceToDevice, x->stream));
        KS_CUDA(cudaMemcpyAsync(c.t_abund + A.n_prot, B.t_abund, p_b * 4, cudaMemcpyDeviceToDevice, x->stream));
    }
    KS_CUDA(cudaEventRecord(x->ev[EV_M1], x->stream));
    const StatusBlock st = read_status(x, StatusBlock{}, 24);  // U_C, G_C, M: the one host read of the merge
    if (st.G != G || st.U + st.produced != U_max) fail(KS_ERR_CUDA, "internal error: the merged index does not add up");
    if (x->hooks.append_fail == 2) fail(KS_ERR_OUT_OF_MEMORY, "KS_APPEND_FAIL: append failed after the merge (test hook)");
    c.U = st.U; c.G = st.G;
    c.hash_col_valid = false;  // rebuilt from the CSR on demand (ks_index_export)
    if (x->hooks.timing) {
        float ms = 0;
        KS_CUDA(cudaEventElapsedTime(&ms, x->ev[EV_M0], x->ev[EV_M1]));
        fprintf(stderr, "[ks] append: batch_path %u A_layout %s B_layout %s U_A %llu U_B %llu matched %llu n_C %llu batch_ms %.3f merge_ms %.3f\n",
                x->build_path, A.csr.dir_sub == DIR_SUB_COMPACT ? "compact" : "seg", B.dir_sub == DIR_SUB_COMPACT ? "compact" : "seg",
                (unsigned long long)A.csr.U, (unsigned long long)B.U, (unsigned long long)st.produced, (unsigned long long)n,
                batch_ms, ms);
    }
    x->csr = c;
    x->n_tuples = n; x->n_prot = P; x->n_res += A.n_res; x->n_windows += A.n_windows;
    x->build_path = 4;
    x->home = dst;
    x->appended = true;
}

// Extend the finalized index by the batch add_batch() adds.
template <class F>
void append_batch(ks_index* x, F&& add_batch) {
    const double t0 = wall_ms();
    park_index(x);
    Parked A;
    A.csr = x->csr; A.n_tuples = x->n_tuples; A.n_prot = x->n_prot; A.n_res = x->n_res; A.n_windows = x->n_windows;
    A.build_path = x->build_path; A.home = x->home; A.appended = x->appended;
    try {
        drop_content(x);
        add_batch();
        finalize(x);
        if (x->hooks.append_fail == 1) fail(KS_ERR_OUT_OF_MEMORY, "KS_APPEND_FAIL: append failed after the batch's build (test hook)");
        if (x->hooks.timing) KS_CUDA(cudaStreamSynchronize(x->stream));
        merge_appended(x, A, wall_ms() - t0);
    } catch (...) {
        restore_index(x, A);
        throw;
    }
}

template <class T>
T* to_host(const T* d, uint64_t n, cudaStream_t st) {
    T* h = (T*)malloc((n ? n : 1) * sizeof(T));
    if (!h) throw std::bad_alloc();
    if (n) KS_CUDA(cudaMemcpyAsync(h, d, n * sizeof(T), cudaMemcpyDeviceToHost, st));
    return h;
}

// Fill a ks_sketch from grouped tuples.  tuple_hash/tuple_loc: the tuple list to export alongside.
ks_sketch* sketch_to_host(const Grouped& g, const uint64_t* tuple_hash, const uint64_t* tuple_loc, uint64_t n,
                          uint64_t n_prot, cudaStream_t st) {
    ks_sketch* s = (ks_sketch*)calloc(1, sizeof(ks_sketch));
    if (!s) throw std::bad_alloc();
    s->n_proteins = n_prot;
    s->n_tuples = n;
    s->hash = to_host(tuple_hash, n, st);
    uint64_t* loc = to_host(tuple_loc, n, st);
    s->sig_ptr = to_host(g.sig_ptr, n_prot + 1, st);
    s->mins = to_host(g.ent_hash, g.n_entries, st);
    uint32_t* first = to_host(g.ent_first, g.n_entries + 1, st);
    KS_CUDA(cudaStreamSynchronize(st));
    s->pid = (uint32_t*)malloc((n ? n : 1) * 4);
    s->pos = (uint32_t*)malloc((n ? n : 1) * 4);
    s->abunds = (uint64_t*)malloc((g.n_entries ? g.n_entries : 1) * 8);
    if (!s->pid || !s->pos || !s->abunds) throw std::bad_alloc();
    for (uint64_t i = 0; i < n; i++) { s->pid[i] = (uint32_t)(loc[i] >> 32); s->pos[i] = (uint32_t)loc[i]; }
    for (uint64_t e = 0; e < g.n_entries; e++) s->abunds[e] = first[e + 1] - first[e];
    free(loc);
    free(first);
    return s;
}

// What a ks_search_result owns besides its struct: the device block (until it has been copied out, or for as long as the
// result lives with KS_SEARCH_DEVICE_ONLY) and the pinned host copy; both have layout L (search.cuh).
struct ResultDevice {
    Arena* arena = nullptr;  // owns `block`
    void* block = nullptr;
    ResultLayout L;
    void* pinned = nullptr;
    size_t pinned_bytes = 0;
};

}  // namespace

extern "C" {

ks_status ks_index_create(const ks_params* params, ks_index** out) {
    return guarded([&] {
        if (!params || !out) fail(KS_ERR_VALIDATION, "Validation error: null argument");
        if (params->moltype < 0 || params->moltype > 2)
            fail(KS_ERR_INVALID_MOLTYPE, "Invalid moltype: " + std::to_string(params->moltype) +
                                             ", only 'protein', 'hp', or 'dayhoff' are supported");
        if (params->ksize == 0 || params->ksize > (uint32_t)SK_MAX_K)
            fail(KS_ERR_INVALID_KSIZE, "Invalid k-mer size: " + std::to_string(params->ksize));  // errors.rs:20-21
        if (params->scaled == 0) fail(KS_ERR_VALIDATION, "Validation error: scaled must be >= 1");
        int n = ks_device_count();
        if (n == 0) fail(KS_ERR_NO_DEVICE, "no CUDA device: kmerseek_b200 has no CPU fallback");
        if (params->device < 0 || params->device >= n) fail(KS_ERR_NO_DEVICE, "CUDA device ordinal out of range");
        ks_index* x = new ks_index();
        x->params = *params;
        x->hooks.read();
        x->max_hash = ks_max_hash(params->scaled);
        x->lz = clz64(x->max_hash);
        try {
            x->use();
            KS_CUDA(cudaStreamCreateWithFlags(&x->stream, cudaStreamNonBlocking));
            KS_CUDA(cudaStreamCreateWithFlags(&x->copy_stream, cudaStreamNonBlocking));
            for (auto& e : x->ev_chunk) KS_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            for (auto& e : x->ev) KS_CUDA(cudaEventCreate(&e));
            cudaMemPool_t pool;
            KS_CUDA(cudaDeviceGetDefaultMemPool(&pool, params->device));
            uint64_t thr = UINT64_MAX;  // keep freed blocks in the pool: steady-state steps never reach the driver
            KS_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr));
            x->arena = new Arena(x->stream, &x->live_bytes);
            x->d_status = x->arena->alloc<uint64_t>(8);
            x->d_count = x->d_status + 2;
            KS_CUDA(cudaHostAlloc((void**)&x->h_words, H_WORDS * 8, cudaHostAllocDefault));
        } catch (...) {
            ks_index_destroy(x);
            throw;
        }
        *out = x;
    });
}

void ks_index_destroy(ks_index* x) {
    if (!x) return;
    cudaSetDevice(x->params.device);
    if (x->stream) cudaStreamSynchronize(x->stream);
    delete x->arena;
    if (x->stream) cudaStreamSynchronize(x->stream);
    for (auto& e : x->ev) if (e) cudaEventDestroy(e);
    for (auto& e : x->ev_chunk) if (e) cudaEventDestroy(e);
    if (x->h_words) cudaFreeHost(x->h_words);
    if (x->copy_stream) { cudaStreamSynchronize(x->copy_stream); cudaStreamDestroy(x->copy_stream); }
    if (x->stream) cudaStreamDestroy(x->stream);
    delete x;
}

ks_status ks_index_params(const ks_index* x, ks_params* out) {
    if (!x || !out) return set_error(KS_ERR_VALIDATION, "Validation error: null argument");
    *out = x->params;
    return KS_OK;
}
void* ks_index_stream(const ks_index* x) { return x ? (void*)x->stream : nullptr; }
ks_status ks_index_sync(ks_index* x) {
    return guarded([&] { x->use(); KS_CUDA(cudaStreamSynchronize(x->stream)); });
}

ks_status ks_index_upload(ks_index* x, const ks_proteome* p) {
    return guarded([&] {
        if (!x || !p) fail(KS_ERR_VALIDATION, "Validation error: null argument");
        x->use();
        upload_resident(x, p);
    });
}
ks_status ks_index_sketch_resident(ks_index* x) {
    return guarded([&] { x->use(); sketch_resident(x); });
}
ks_status ks_index_add_proteome(ks_index* x, const ks_proteome* p) {
    return guarded([&] {
        if (!x || !p) fail(KS_ERR_VALIDATION, "Validation error: null argument");
        x->use();
        add_proteome(x, p);
    });
}
ks_status ks_index_finalize(ks_index* x) {
    return guarded([&] { x->use(); finalize(x); });
}
ks_status ks_index_clear(ks_index* x) {
    return guarded([&] {
        x->use();
        drop_content(x);
    });
}
ks_status ks_index_process_fasta(ks_index* x, const char* path, uint64_t ambig_seed) {
    ks_proteome* p = nullptr;
    ks_status s = ks_proteome_from_fasta(path, ambig_seed, &p);
    if (s != KS_OK) return s;
    s = ks_index_add_proteome(x, p);
    ks_proteome_free(p);
    return s != KS_OK ? s : ks_index_finalize(x);
}

ks_status ks_index_add_tuples(ks_index* x, const uint64_t* hash, const uint32_t* pid, const uint32_t* pos, uint64_t n,
                              uint64_t n_proteins) {
    return guarded([&] {
        if (!x || (n && (!hash || !pid || !pos))) fail(KS_ERR_VALIDATION, "Validation error: null argument");
        x->use();
        materialize_pending(x);
        if (x->n_prot + n_proteins >= 0xffffffffull) fail(KS_ERR_CAPACITY, "more than 2^32-2 proteins on one shard");
        const std::vector<uint64_t> loc = tuple_locs(pid, pos, n, n_proteins, (uint32_t)x->n_prot);
        if (x->finalized()) fail(KS_ERR_VALIDATION, "Validation error: index is finalized; ks_index_clear before adding more");
        push_tuples(x, hash, loc, n_proteins);
    });
}

ks_status ks_index_append_proteome(ks_index* x, const ks_proteome* p) {
    return guarded([&] {
        if (!x || !p) fail(KS_ERR_VALIDATION, "Validation error: null argument");
        if (!x->finalized()) fail(KS_ERR_NOT_FINALIZED, "index is not finalized: ks_index_finalize before appending");
        x->use();
        if (x->n_prot + p->n_prot >= 0xffffffffull) fail(KS_ERR_CAPACITY, "more than 2^32-2 proteins on one shard");
        uint64_t windows = 0, max_len = 0;
        proteome_shape(p, x->params.ksize, &windows, &max_len);
        if (x->max_hash == ~0ull && x->n_tuples + windows > MAX_TUPLES)  // scaled 1: every window is a tuple
            fail(KS_ERR_CAPACITY, "more than 2^31-1 tuples on one shard: shard the proteome over more GPUs");
        append_batch(x, [&] { add_proteome(x, p); });
    });
}

ks_status ks_index_append_tuples(ks_index* x, const uint64_t* hash, const uint32_t* pid, const uint32_t* pos, uint64_t n,
                                 uint64_t n_proteins) {
    return guarded([&] {
        if (!x || (n && (!hash || !pid || !pos))) fail(KS_ERR_VALIDATION, "Validation error: null argument");
        if (!x->finalized()) fail(KS_ERR_NOT_FINALIZED, "index is not finalized: ks_index_finalize before appending");
        x->use();
        if (x->n_prot + n_proteins >= 0xffffffffull) fail(KS_ERR_CAPACITY, "more than 2^32-2 proteins on one shard");
        if (x->n_tuples + n > MAX_TUPLES) fail(KS_ERR_CAPACITY, "more than 2^31-1 tuples on one shard: shard the proteome over more GPUs");
        const std::vector<uint64_t> loc = tuple_locs(pid, pos, n, n_proteins, 0);  // the batch's own ids: it is built alone
        append_batch(x, [&] { push_tuples(x, hash, loc, n_proteins); });
    });
}

ks_status ks_index_stats(ks_index* x, ks_stats* out) {
    return guarded([&] {
        if (!x || !out) fail(KS_ERR_VALIDATION, "Validation error: null argument");
        x->use();
        KS_CUDA(cudaStreamSynchronize(x->stream));
        ks_stats s{};
        s.n_proteins = x->n_prot; s.n_residues = x->n_res; s.n_windows = x->n_windows; s.n_tuples = x->n_tuples;
        s.n_unique_hashes = x->csr.U; s.n_groups = x->csr.G; s.n_distinct_ids = x->csr.n_ids; s.device_bytes = x->live_bytes;
        s.sketch_launches = x->l_sketch; s.sort_launches = x->l_sort; s.csr_launches = x->l_csr; s.search_launches = x->l_search;
        if (x->t_upload) KS_CUDA(cudaEventElapsedTime(&s.ms_upload, x->ev[EV_UP0], x->ev[EV_UP1]));
        if (x->t_sketch) KS_CUDA(cudaEventElapsedTime(&s.ms_sketch, x->ev[EV_SK0], x->ev[EV_SK1]));
        if (x->t_sort) {
            KS_CUDA(cudaEventElapsedTime(&s.ms_sort, x->ev[EV_SO0], x->ev[EV_SO1]));
            KS_CUDA(cudaEventElapsedTime(&s.ms_sort_partition, x->ev[EV_SO0], x->ev[EV_PART]));
            KS_CUDA(cudaEventElapsedTime(&s.ms_sort_bucket, x->ev[EV_PART], x->ev[EV_SO1]));
        }
        if (x->t_csr) KS_CUDA(cudaEventElapsedTime(&s.ms_csr, x->ev[EV_SO1], x->ev[EV_CS1]));
        s.ms_search = x->ms_search;
        s.finalized = x->finalized() ? 1 : 0;
        s.build_path = x->build_path;
        *out = s;
    });
}

// signature_count() (src/rust/index.rs:514-516): signatures are keyed by their id string -- the hex of the wrapping sum of
// the sketch's mins (signature.rs:277-279) -- and equal ids overwrite (DashMap insert, index.rs:817-820), so the count is
// the number of distinct sums over the proteins.  Sums on the device from the CSR, distinct count on the host.
ks_status ks_index_signature_count(ks_index* x, uint64_t* out) {
    return guarded([&] {
        if (!x || !out) fail(KS_ERR_VALIDATION, "Validation error: null argument");
        if (!x->finalized()) fail(KS_ERR_NOT_FINALIZED, "index is not finalized");
        x->use();
        const uint64_t P = x->n_prot;
        std::vector<uint64_t> sums(P ? P : 1, 0);
        if (P) {
            Arena tmp(x->stream, &x->live_bytes);
            unsigned long long* d = (unsigned long long*)tmp.alloc<uint64_t>(P);
            KS_CUDA(cudaMemsetAsync(d, 0, P * 8, x->stream));
            KS_CUDA(launch_id_sums(view_of(x), x->csr.U, d, x->stream));
            KS_CUDA(cudaMemcpyAsync(sums.data(), d, P * 8, cudaMemcpyDeviceToHost, x->stream));
            KS_CUDA(cudaStreamSynchronize(x->stream));
        }
        std::sort(sums.begin(), sums.begin() + P);
        x->csr.n_ids = (uint64_t)(std::unique(sums.begin(), sums.begin() + P) - sums.begin());
        *out = x->csr.n_ids;
    });
}

// ---- sketch export ------------------------------------------------------------------------------
ks_status ks_sketch_batch(ks_index* x, const ks_proteome* p, ks_sketch** out) {
    return guarded([&] {
        if (!x || !p || !out) fail(KS_ERR_VALIDATION, "Validation error: null argument");
        x->use();
        DeviceBatch b;
        Arena keep(x->stream, &x->live_bytes), tmp(x->stream, &x->live_bytes);
        // a private batch: the index's resident batch and tuples are left alone
        b.res = keep.alloc<uint8_t>(p->n_res + 64);
        b.offs = keep.alloc<uint64_t>(p->n_prot + 1);
        KS_CUDA(cudaMemcpyAsync(b.res, p->residues, p->n_res + 64, cudaMemcpyHostToDevice, x->stream));
        KS_CUDA(cudaMemcpyAsync(b.offs, p->offsets, (p->n_prot + 1) * 8, cudaMemcpyHostToDevice, x->stream));
        b.n_prot = p->n_prot; b.n_res = p->n_res;
        proteome_shape(p, x->params.ksize, &b.n_windows, &b.max_len);
        b.valid = true;
        const uint64_t cap = b.n_windows;
        uint64_t* h = keep.alloc<uint64_t>(cap);
        uint64_t* l = keep.alloc<uint64_t>(cap);
        uint64_t* cnt = tmp.alloc<uint64_t>(2);  // private: a pending pipelined batch keeps its counts in the handle's
        void* ws = tmp.alloc<char>(sketch_workspace_bytes(b.n_res));
        uint64_t n = run_sketch(x, b, 0, h, l, cap, cnt, ws);
        Grouped g;
        group_by_owner(keep, tmp, h, l, n, (uint32_t)p->n_prot, x->end_bit(), &g, &x->l_sketch);
        *out = sketch_to_host(g, h, l, n, p->n_prot, x->stream);
    });
}

ks_status ks_index_export(ks_index* x, ks_sketch** out) {
    return guarded([&] {
        if (!x || !out) fail(KS_ERR_VALIDATION, "Validation error: null argument");
        if (!x->finalized()) fail(KS_ERR_NOT_FINALIZED, "index is not finalized");
        x->use();
        Arena keep(x->stream, &x->live_bytes), tmp(x->stream, &x->live_bytes);
        Grouped g;
        if (!x->csr.hash_col_valid) {
            KS_CUDA(expand_sorted_hash(view_of(x), x->csr.hash, x->stream));
            x->csr.hash_col_valid = true;
        }
        group_by_owner(keep, tmp, x->csr.hash, x->csr.loc, x->n_tuples, (uint32_t)x->n_prot, x->end_bit(), &g, &x->l_csr);
        *out = sketch_to_host(g, x->csr.hash, x->csr.loc, x->n_tuples, x->n_prot, x->stream);
    });
}

void ks_sketch_free(ks_sketch* s) {
    if (!s) return;
    free(s->hash); free(s->pid); free(s->pos); free(s->sig_ptr); free(s->mins); free(s->abunds);
    free(s);
}

ks_status ks_index_csr(ks_index* x, ks_csr** out) {
    return guarded([&] {
        if (!x || !out) fail(KS_ERR_VALIDATION, "Validation error: null argument");
        if (!x->finalized()) fail(KS_ERR_NOT_FINALIZED, "index is not finalized");
        x->use();
        ks_csr* c = (ks_csr*)calloc(1, sizeof(ks_csr));
        if (!c) throw std::bad_alloc();
        c->n_keys = x->csr.U; c->n_postings = x->n_tuples;
        const bool seg = x->csr.dir_sub != DIR_SUB_COMPACT;
        const uint64_t span = seg ? x->n_tuples + x->csr.seg_nb + 1 : x->csr.U + 1;  // key / group positions in use
        uint64_t* keys = to_host(x->csr.keys, seg ? span : x->csr.U, x->stream);
        uint32_t* kg = to_host(x->csr.key_grp, span, x->stream);
        uint32_t* gs = to_host(x->csr.grp_start, seg ? span : x->csr.G + 1, x->stream);
        uint64_t* loc = to_host(x->csr.loc, x->n_tuples, x->stream);
        uint32_t* st = seg ? to_host(x->csr.seg_start, (uint64_t)x->csr.seg_nb + 1, x->stream) : nullptr;
        uint64_t* sc = seg ? to_host(x->csr.seg_counts, x->csr.seg_nb, x->stream) : nullptr;
        KS_CUDA(cudaStreamSynchronize(x->stream));
        c->row_ptr = (uint64_t*)malloc((x->csr.U + 1) * 8);
        c->pid = (uint32_t*)malloc((x->n_tuples ? x->n_tuples : 1) * 4);
        c->pos = (uint32_t*)malloc((x->n_tuples ? x->n_tuples : 1) * 4);
        if (!c->row_ptr || !c->pid || !c->pos) throw std::bad_alloc();
        if (!seg) {
            c->keys = keys;
            for (uint64_t u = 0; u <= x->csr.U; u++) c->row_ptr[u] = gs[kg[u]];
        } else {  // segmented layout -> the compact table: bucket by bucket, keys at seg_start[b] + b + i
            c->keys = (uint64_t*)malloc((x->csr.U ? x->csr.U : 1) * 8);
            if (!c->keys) throw std::bad_alloc();
            uint64_t u = 0;
            for (uint32_t b = 0; b < x->csr.seg_nb; b++) {
                const uint64_t kb = (uint64_t)st[b] + b, tk = (uint32_t)sc[b];
                for (uint64_t i = 0; i < tk && u < x->csr.U; i++, u++) { c->keys[u] = keys[kb + i]; c->row_ptr[u] = gs[kg[kb + i]]; }
            }
            if (u != x->csr.U) fail(KS_ERR_CUDA, "internal error: segmented CSR does not add up");
            c->row_ptr[x->csr.U] = x->n_tuples;
            free(keys);
        }
        for (uint64_t i = 0; i < x->n_tuples; i++) { c->pid[i] = (uint32_t)(loc[i] >> 32); c->pos[i] = (uint32_t)loc[i]; }
        free(kg); free(gs); free(loc); free(st); free(sc);
        *out = c;
    });
}
void ks_csr_free(ks_csr* c) {
    if (!c) return;
    free(c->keys); free(c->row_ptr); free(c->pid); free(c->pos);
    free(c);
}

// ---- search --------------------------------------------------------------------------------------
}  // extern "C"

namespace {

QueryScratch ensure_query_scratch(ks_index* x, uint64_t nq, uint64_t n_res, bool hits) {
    Arena* ar = x->arena;
    QueryScratch s;
    s.e_count = x->b_q_ecount.ensure<uint32_t>(ar, nq);
    s.p_count = x->b_q_pcount.ensure<uint32_t>(ar, nq);
    s.h_count = x->b_q_hcount.ensure<uint64_t>(ar, nq);
    s.sig_ptr = x->b_q_sig.ensure<uint64_t>(ar, nq + 1);
    s.pair_off = x->b_q_poff.ensure<uint64_t>(ar, nq + 1);
    s.hit_off = x->b_q_hoff.ensure<uint64_t>(ar, nq + 1);
    s.ent_hash = x->b_q_ent_hash.ensure<uint64_t>(ar, n_res);
    s.ent_abund = x->b_q_ent_abund.ensure<uint32_t>(ar, n_res);
    if (hits) {
        s.win_key = x->b_q_win_key.ensure<uint32_t>(ar, n_res);
        s.win_hoff = x->b_q_win_hoff.ensure<uint32_t>(ar, n_res);
    }
    const uint64_t want = std::max<uint64_t>(1u << 16, n_res / 2);  // first guess; grows to what a batch needed
    if (x->b_q_stage.bytes < want * sizeof(StagedPair)) x->b_q_stage.ensure<StagedPair>(ar, want);
    s.stage = (StagedPair*)x->b_q_stage.p;
    s.stage_cap = x->b_q_stage.bytes / sizeof(StagedPair);
    s.totals = x->b_q_totals.ensure<uint64_t>(ar, QT_WORDS);
    return s;
}

struct SearchOut {
    void* block = nullptr;
    ResultLayout L;
};

// Device side of one search of the resident query batch; the result block is allocated from `keep`.  Synchronises the
// stream once on the hand-written path (the totals that size the block).
SearchOut search_resident_device(ks_index* x, Arena& keep, bool hits, bool sketches, bool wire, uint32_t pid_base) {
    cudaStream_t st = x->stream;
    const DeviceBatch& qb = x->qbatch;
    const uint32_t k = x->params.ksize;
    const uint64_t maxw = qb.max_len >= k ? qb.max_len - k + 1 : 0;
    SearchOut o;
    KS_CUDA(cudaEventRecord(x->ev[EV_Q0], st));
    if (maxw > QK_MAX_WINDOWS || x->hooks.search_legacy) {
        if (wire) fail(KS_ERR_CAPACITY, "sharded search: queries of more than 4096 k-mer windows are not supported");
        Arena tmp(st, &x->live_bytes);
        uint64_t* qh = tmp.alloc<uint64_t>(qb.n_windows);
        uint64_t* ql = tmp.alloc<uint64_t>(qb.n_windows);
        uint64_t* cnt = tmp.alloc<uint64_t>(2);
        void* ws = tmp.alloc<char>(sketch_workspace_bytes(qb.n_res));
        const uint64_t nqt = run_sketch(x, qb, 0, qh, ql, qb.n_windows, cnt, ws);
        search_device_legacy(tmp, view_of(x), qh, ql, nqt, (uint32_t)qb.n_prot, k, x->end_bit(), hits, sketches, pid_base, keep,
                             &o.block, &o.L, &x->l_search);
    } else {
        QueryScratch s = ensure_query_scratch(x, qb.n_prot, qb.n_res, hits);
        QueryBatchView qv{qb.res, qb.offs, (uint32_t)qb.n_prot, qb.n_res, (uint32_t)maxw};
        uint64_t* t = x->h_words + HW_TOTALS;
        for (int attempt = 0;; attempt++) {
            KS_CUDA(launch_query_phase1(qv, view_of(x), k, x->params.moltype, x->max_hash, hits, s, st, &x->l_search));
            KS_CUDA(cudaMemcpyAsync(t, s.totals, QT_WORDS * 8, cudaMemcpyDeviceToHost, st));
            KS_CUDA(cudaStreamSynchronize(st));
            if (t[QT_FLAGS] & QF_HITS_OVERFLOW) fail(KS_ERR_CAPACITY, "one query has 2^32 or more hits");
            if (t[QT_PAIRS] <= s.stage_cap) break;
            if (attempt) fail(KS_ERR_CUDA, "internal error: the pair staging buffer overflowed twice");
            x->b_q_stage.ensure<StagedPair>(x->arena, t[QT_PAIRS] + t[QT_PAIRS] / 4);  // counted in full: now it fits
            s.stage = (StagedPair*)x->b_q_stage.p;
            s.stage_cap = x->b_q_stage.bytes / sizeof(StagedPair);
        }
        o.L = result_layout(qb.n_prot, t[QT_PAIRS], t[QT_HITS], t[QT_ENTRIES], hits, sketches, wire, qb.n_res);
        o.block = keep.alloc<char>(o.L.bytes);
        KS_CUDA(launch_query_phase2(qv, view_of(x), k, pid_base, s, o.L, o.block, st, &x->l_search));
    }
    KS_CUDA(cudaEventRecord(x->ev[EV_Q1], st));
    return o;
}

void set_host_columns(ks_search_result* r, const ResultLayout& L, char* base) {
    r->q_sig_ptr = (uint64_t*)(base + L.off_sig_ptr);
    uint32_t** u32[N_PAIR_U32] = {&r->pair_qid, &r->pair_pid, &r->intersect_hashes, &r->q_size, &r->t_size};
    for (int i = 0; i < N_PAIR_U32; i++) *u32[i] = (uint32_t*)(base + L.off_u32[i]);
    r->n_weighted_found = (uint64_t*)(base + L.off_u64[0]);
    r->total_weighted_hashes = (uint64_t*)(base + L.off_u64[1]);
    double** sc[N_SCORE_COLS] = {&r->containment, &r->containment_target_in_query, &r->max_containment, &r->jaccard,
                                 &r->query_containment_ani, &r->match_containment_ani, &r->average_containment_ani,
                                 &r->max_containment_ani, &r->average_abund, &r->median_abund, &r->std_abund,
                                 &r->f_weighted_target_in_query};
    for (int i = 0; i < N_SCORE_COLS; i++) *sc[i] = (double*)(base + L.off_score[i]);
    if (L.hits) {
        uint32_t** h32[N_HIT_U32] = {&r->hit_qid, &r->hit_pid, &r->hit_qpos, &r->hit_tpos};
        for (int i = 0; i < N_HIT_U32; i++) *h32[i] = (uint32_t*)(base + L.off_hit32[i]);
        r->hit_hash = (uint64_t*)(base + L.off_hit_hash);
    }
    if (L.sketches) {
        r->q_mins = (uint64_t*)(base + L.off_q_mins);
        r->q_abunds = (uint64_t*)(base + L.off_q_abunds);
    }
}

// One D2H copy of the whole block into a pooled pinned block; the device block is given back.
void result_to_host(ks_index* x, ks_search_result* r, ResultDevice* rd) {
    rd->pinned = pinned_get(rd->L.bytes, &rd->pinned_bytes);
    KS_CUDA(cudaMemcpyAsync(rd->pinned, rd->block, rd->L.bytes, cudaMemcpyDeviceToHost, x->stream));
    KS_CUDA(cudaStreamSynchronize(x->stream));
    set_host_columns(r, rd->L, (char*)rd->pinned);
    // the host copy is complete: give the device block back now, so that the result no longer depends on the index
    // (and its stream) staying alive
    delete rd->arena;
    rd->arena = nullptr;
    rd->block = nullptr;
}

ks_search_result* new_result(ks_index* x, ResultDevice** rd_out) {
    ks_search_result* r = (ks_search_result*)calloc(1, sizeof(ks_search_result));
    if (!r) throw std::bad_alloc();
    ResultDevice* rd = new ResultDevice();
    rd->arena = new Arena(x->stream, &x->live_bytes);
    r->device_block = rd;
    *rd_out = rd;
    return r;
}

// ---- NCCL, bound at run time (the library loads without it; multi-GPU calls then return KS_ERR_NCCL) ------------------
struct NcclApi {
    DlLib lib;
    decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
    decltype(&ncclCommInitRank) CommInitRank = nullptr;
    decltype(&ncclCommDestroy) CommDestroy = nullptr;
    decltype(&ncclAllGather) AllGather = nullptr;
    decltype(&ncclSend) Send = nullptr;
    decltype(&ncclRecv) Recv = nullptr;
    decltype(&ncclGroupStart) GroupStart = nullptr;
    decltype(&ncclGroupEnd) GroupEnd = nullptr;
    decltype(&ncclGetErrorString) GetErrorString = nullptr;
    bool ok = false;
    static const char* const* names() {
        static const char* const n[] = {"libnccl.so.2", "libnccl.so", nullptr};
        return n;
    }
    NcclApi() : lib(names()) {
        GetUniqueId = lib.sym<decltype(GetUniqueId)>("ncclGetUniqueId");
        CommInitRank = lib.sym<decltype(CommInitRank)>("ncclCommInitRank");
        CommDestroy = lib.sym<decltype(CommDestroy)>("ncclCommDestroy");
        AllGather = lib.sym<decltype(AllGather)>("ncclAllGather");
        Send = lib.sym<decltype(Send)>("ncclSend");
        Recv = lib.sym<decltype(Recv)>("ncclRecv");
        GroupStart = lib.sym<decltype(GroupStart)>("ncclGroupStart");
        GroupEnd = lib.sym<decltype(GroupEnd)>("ncclGroupEnd");
        GetErrorString = lib.sym<decltype(GetErrorString)>("ncclGetErrorString");
        ok = GetUniqueId && CommInitRank && CommDestroy && AllGather && Send && Recv && GroupStart && GroupEnd && GetErrorString;
    }
};

NcclApi& nccl() {
    static NcclApi api;  // process-wide; under torch this resolves to the libnccl.so.2 torch has already loaded
    if (!api.ok) fail(KS_ERR_NCCL, "NCCL error: libnccl.so.2 could not be loaded");
    return api;
}

void nccl_check(ncclResult_t r, const char* what) {
    if (r == ncclSuccess) return;
    fail(KS_ERR_NCCL, std::string("NCCL error: ") + nccl().GetErrorString(r) + " (" + what + ")");
}
#define KS_NCCL(x) nccl_check((x), #x)

}  // namespace

struct ks_comm {
    ncclComm_t comm = nullptr;
    int rank = 0, world = 1, device = 0;
};

extern "C" {

ks_status ks_query_upload(ks_index* x, const ks_proteome* q) {
    return guarded([&] {
        if (!x || !q) fail(KS_ERR_VALIDATION, "Validation error: null argument");
        x->use();
        upload_batch(x, x->qbatch, q);
    });
}

ks_status ks_search_resident(ks_index* x, uint32_t flags, ks_search_result** out) {
    return guarded([&] {
        if (!x || !out) fail(KS_ERR_VALIDATION, "Validation error: null argument");
        if (!x->finalized()) fail(KS_ERR_NOT_FINALIZED, "index is not finalized");
        if (!x->qbatch.valid) fail(KS_ERR_VALIDATION, "Validation error: no query batch is resident");
        x->use();
        ResultDevice* rd = nullptr;
        ks_search_result* r = new_result(x, &rd);
        const bool dbg = x->hooks.timing;
        const double t0 = dbg ? wall_ms() : 0;
        try {
            const SearchOut o = search_resident_device(x, *rd->arena, (flags & KS_SEARCH_HITS) != 0,
                                                       (flags & KS_SEARCH_QUERY_SKETCHES) != 0, false, 0);
            const double t1 = dbg ? wall_ms() : 0;
            rd->block = o.block;
            rd->L = o.L;
            r->n_queries = o.L.nq;
            r->n_pairs = o.L.n_pairs;
            r->n_hits = o.L.n_hits;
            if (flags & KS_SEARCH_DEVICE_ONLY) KS_CUDA(cudaStreamSynchronize(x->stream));
            else result_to_host(x, r, rd);
            KS_CUDA(cudaEventElapsedTime(&r->ms_device, x->ev[EV_Q0], x->ev[EV_Q1]));
            x->ms_search = r->ms_device;
            if (dbg) fprintf(stderr, "[ks] search: device %.3f ms; host: kernels + count read-back %.3f ms, block read-back %.3f ms\n",
                             r->ms_device, t1 - t0, wall_ms() - t1);
        } catch (...) {
            ks_search_result_free(r);
            throw;
        }
        *out = r;
    });
}

ks_status ks_search_batch(ks_index* x, const ks_proteome* queries, uint32_t flags, ks_search_result** out) {
    ks_status s = ks_query_upload(x, queries);
    return s != KS_OK ? s : ks_search_resident(x, flags, out);
}

void* ks_search_result_device_column(const ks_search_result* r, const char* name) {
    if (!r || !r->device_block || !name) return nullptr;
    const ResultDevice* rd = (const ResultDevice*)r->device_block;
    if (!rd->block) return nullptr;
    char* b = (char*)rd->block;
    const ResultLayout& L = rd->L;
    static const char* u32n[N_PAIR_U32] = {"pair_qid", "pair_pid", "intersect_hashes", "q_size", "t_size"};
    static const char* u64n[N_PAIR_U64] = {"n_weighted_found", "total_weighted_hashes"};
    static const char* scn[N_SCORE_COLS] = {
        "containment", "containment_target_in_query", "max_containment", "jaccard", "query_containment_ani",
        "match_containment_ani", "average_containment_ani", "max_containment_ani", "average_abund", "median_abund",
        "std_abund", "f_weighted_target_in_query"};
    static const char* h32n[N_HIT_U32] = {"hit_qid", "hit_pid", "hit_qpos", "hit_tpos"};
    for (int i = 0; i < N_PAIR_U32; i++) if (!strcmp(name, u32n[i])) return b + L.off_u32[i];
    for (int i = 0; i < N_PAIR_U64; i++) if (!strcmp(name, u64n[i])) return b + L.off_u64[i];
    for (int i = 0; i < N_SCORE_COLS; i++) if (!strcmp(name, scn[i])) return b + L.off_score[i];
    if (L.hits) {
        for (int i = 0; i < N_HIT_U32; i++) if (!strcmp(name, h32n[i])) return b + L.off_hit32[i];
        if (!strcmp(name, "hit_hash")) return b + L.off_hit_hash;
    }
    if (!strcmp(name, "q_sig_ptr")) return b + L.off_sig_ptr;
    if (L.sketches && !strcmp(name, "q_mins")) return b + L.off_q_mins;
    if (L.sketches && !strcmp(name, "q_abunds")) return b + L.off_q_abunds;
    return nullptr;
}

void ks_search_result_free(ks_search_result* r) {
    if (!r) return;
    if (r->device_block) {  // every column lives in the pinned block (or on the device only)
        ResultDevice* rd = (ResultDevice*)r->device_block;
        pinned_put(rd->pinned, rd->pinned_bytes);
        delete rd->arena;
        delete rd;
    }
    free(r);
}

// ---- multi-GPU: one process per GPU, the proteome sharded by protein ------------------------------------------------
ks_status ks_comm_unique_id(uint8_t id[KS_COMM_ID_BYTES]) {
    return guarded([&] {
        if (!id) fail(KS_ERR_VALIDATION, "Validation error: null argument");
        static_assert(sizeof(ncclUniqueId) == KS_COMM_ID_BYTES, "ncclUniqueId is 128 bytes");
        ncclUniqueId u;
        KS_NCCL(nccl().GetUniqueId(&u));
        memcpy(id, &u, sizeof u);
    });
}

ks_status ks_comm_create(const uint8_t id[KS_COMM_ID_BYTES], int rank, int world, int device, ks_comm** out) {
    return guarded([&] {
        if (!id || !out) fail(KS_ERR_VALIDATION, "Validation error: null argument");
        if (world < 1 || world > MAX_SHARDS || rank < 0 || rank >= world)
            fail(KS_ERR_VALIDATION, "Validation error: rank / world out of range (at most 16 shards)");
        const int n = ks_device_count();
        if (n == 0) fail(KS_ERR_NO_DEVICE, "no CUDA device: kmerseek_b200 has no CPU fallback");
        if (device < 0 || device >= n) fail(KS_ERR_NO_DEVICE, "CUDA device ordinal out of range");
        KS_CUDA(cudaSetDevice(device));
        ncclUniqueId u;
        memcpy(&u, id, sizeof u);
        ks_comm* c = new ks_comm();
        c->rank = rank; c->world = world; c->device = device;
        try {
            KS_NCCL(nccl().CommInitRank(&c->comm, world, u, rank));
        } catch (...) {
            delete c;
            throw;
        }
        *out = c;
    });
}

void ks_comm_destroy(ks_comm* c) {
    if (!c) return;
    if (c->comm) {
        cudaSetDevice(c->device);
        try { nccl().CommDestroy(c->comm); } catch (...) {}
    }
    delete c;
}
int ks_comm_rank(const ks_comm* c) { return c ? c->rank : 0; }
int ks_comm_world(const ks_comm* c) { return c ? c->world : 1; }

ks_status ks_shard_search_batch(ks_index* x, ks_comm* c, const ks_proteome* queries, uint32_t flags, uint64_t pid_base,
                                ks_search_result** out) {
    ks_status up = ks_query_upload(x, queries);
    if (up != KS_OK) return up;
    return guarded([&] {
        if (!c || !out) fail(KS_ERR_VALIDATION, "Validation error: null argument");
        if (!x->finalized()) fail(KS_ERR_NOT_FINALIZED, "index is not finalized");
        if (x->appended)
            fail(KS_ERR_VALIDATION, "Validation error: a sharded search needs an index built by adds and one finalize; this one was "
                                    "extended by ks_index_append_* (rebuild it: ks_index_clear, add every batch, finalize)");
        if (c->device != x->params.device) fail(KS_ERR_VALIDATION, "Validation error: communicator and index are on different devices");
        if (pid_base + x->n_prot > 0xffffffffull) fail(KS_ERR_CAPACITY, "more than 2^32-1 proteins over all shards");
        x->use();
        cudaStream_t st = x->stream;
        NcclApi& N = nccl();
        const bool hits = (flags & KS_SEARCH_HITS) != 0;
        const bool root = c->rank == 0;
        const bool sketches = root && (flags & KS_SEARCH_QUERY_SKETCHES) != 0;  // replicated queries: rank 0's copy is the result's
        ResultDevice* rd = nullptr;
        ks_search_result* r = new_result(x, &rd);
        try {
            Arena tmp(st, &x->live_bytes);
            // 1. this shard, in wire layout (the merge offsets travel with the block); protein ids already index-wide
            const SearchOut mine = search_resident_device(x, tmp, hits, sketches, true, (uint32_t)pid_base);
            // 2. every rank's counts: one all-gather of four words
            uint64_t* hdr = x->h_words + HW_HDR;
            hdr[0] = mine.L.n_pairs; hdr[1] = mine.L.n_hits; hdr[2] = mine.L.n_entries; hdr[3] = mine.L.bytes;
            uint64_t* d_hdr = tmp.alloc<uint64_t>(4);
            uint64_t* d_all = tmp.alloc<uint64_t>(4 * (size_t)c->world);
            KS_CUDA(cudaMemcpyAsync(d_hdr, hdr, 32, cudaMemcpyHostToDevice, st));
            KS_NCCL(N.AllGather(d_hdr, d_all, 4, ncclUint64, c->comm, st));
            uint64_t* all = x->h_words + HW_ALL;
            KS_CUDA(cudaMemcpyAsync(all, d_all, 32 * (size_t)c->world, cudaMemcpyDeviceToHost, st));
            KS_CUDA(cudaStreamSynchronize(st));
            r->n_queries = mine.L.nq;
            if (!root) {
                // 3. ship the block to rank 0: one send
                KS_NCCL(N.GroupStart());
                KS_NCCL(N.Send(mine.block, mine.L.bytes, ncclUint8, 0, c->comm, st));
                KS_NCCL(N.GroupEnd());
                KS_CUDA(cudaStreamSynchronize(st));
                r->n_pairs = mine.L.n_pairs;  // this shard's counts; the columns are on rank 0
                r->n_hits = mine.L.n_hits;
            } else {
                MergeArgs m;
                m.n_shards = c->world; m.nq = (uint32_t)mine.L.nq; m.q_offs = x->qbatch.offs; m.k = x->params.ksize;
                m.shard[0].block = mine.block; m.shard[0].layout = mine.L;
                uint64_t np = mine.L.n_pairs, nh = mine.L.n_hits;
                KS_NCCL(N.GroupStart());
                for (int s = 1; s < c->world; s++) {
                    const uint64_t* h = all + 4 * s;
                    const ResultLayout Ls = result_layout(mine.L.nq, h[0], h[1], 0, hits, false, true, x->qbatch.n_res);
                    if (Ls.bytes != h[3]) fail(KS_ERR_NCCL, "NCCL error: shard result layout mismatch between ranks");
                    void* blk = tmp.alloc<char>(Ls.bytes);
                    KS_NCCL(N.Recv(blk, Ls.bytes, ncclUint8, s, c->comm, st));
                    m.shard[s].block = blk; m.shard[s].layout = Ls;
                    np += h[0]; nh += h[1];
                }
                KS_NCCL(N.GroupEnd());
                // 4. merge by counting (launch_merge): (query, target) order over ascending shards
                rd->L = result_layout(mine.L.nq, np, nh, mine.L.n_entries, hits, sketches);
                rd->block = rd->arena->alloc<char>(rd->L.bytes);
                m.out_block = rd->block; m.out_layout = rd->L;
                KS_CUDA(launch_merge(m, st, &x->l_search));
                r->n_pairs = np;
                r->n_hits = nh;
                if (flags & KS_SEARCH_DEVICE_ONLY) KS_CUDA(cudaStreamSynchronize(st));
                else result_to_host(x, r, rd);
            }
            KS_CUDA(cudaEventElapsedTime(&r->ms_device, x->ev[EV_Q0], x->ev[EV_Q1]));
            x->ms_search = r->ms_device;
        } catch (...) {
            ks_search_result_free(r);
            throw;
        }
        *out = r;
    });
}

}  // extern "C"
