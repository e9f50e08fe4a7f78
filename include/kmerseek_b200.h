/*
 * kmerseek_b200.h -- C ABI of the B200-native sketch-and-search path of kmerseek.
 *
 * The reference (seanome/kmerseek) exposes no FFI seam on this path: callers use the Rust type
 * `kmerseek::index::ProteomeIndex` directly (src/rust/lib.rs:25) and search lives in Python on top
 * of sourmash_plugin_branchwater (src/python/kmerseek/search.py:125-141).  This header is the seam a
 * maintainer would bind instead (Rust `extern "C"` block / bindgen: see INTEGRATION.md and
 * rust/kmerseek-b200-sys).  Every entry point names the reference item it replaces; paths are
 * relative to the reference repository.
 *
 * Conventions
 *   - plain C types only; opaque handles; no exceptions cross the boundary, nothing aborts.
 *   - every call returns ks_status; on error ks_last_error_message() (thread-local, valid until the
 *     next call on this thread) holds the reference's own error text where one exists.
 *   - inputs are borrowed for the duration of the call; every library-allocated result is released
 *     by the matching *_free.
 *   - a handle owns one device, two CUDA streams and its device buffers.  It is thread-compatible,
 *     not re-entrant: concurrent calls on different handles are safe, on the same handle are not.
 *     (The reference's `&self` methods are called from rayon workers, src/rust/index.rs:993-1005;
 *     callers of this ABI batch instead of calling per protein.)
 *   - there is no CPU fallback: without a CUDA device every compute entry point returns
 *     KS_ERR_NO_DEVICE.
 */
#ifndef KMERSEEK_B200_H
#define KMERSEEK_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KS_ABI_VERSION 1

/* Status codes.  1..19 mirror IndexError (src/rust/errors.rs:4-55); >=100 are device-side. */
typedef enum ks_status {
    KS_OK = 0,
    KS_ERR_INVALID_MOLTYPE = 1,    /* errors.rs:8-9; text from src/rust/encoding.rs:22-25 */
    KS_ERR_INVALID_AMINO_ACID = 2, /* errors.rs:14-15 "Invalid amino acid '{0}' found at position {1}" */
    KS_ERR_INVALID_KSIZE = 3,      /* errors.rs:20-21 */
    KS_ERR_NO_SAVED_STATE = 4,     /* errors.rs:23-24 */
    KS_ERR_IO = 5,                 /* errors.rs:26-27 */
    KS_ERR_UTF8 = 6,               /* errors.rs:29-30 */
    KS_ERR_PARSE = 7,              /* errors.rs:41-42 (needletail errors, src/rust/index.rs:920-928) */
    KS_ERR_BUILDER = 8,            /* errors.rs:35-36 (src/rust/index.rs:3021-3036) */
    KS_ERR_VALIDATION = 9,         /* errors.rs:47-48: a bad argument to this ABI */
    KS_ERR_NOT_FINALIZED = 10,     /* search / export before ks_index_finalize */
    KS_ERR_CUDA = 100,
    KS_ERR_NCCL = 101,
    KS_ERR_OUT_OF_MEMORY = 102,
    KS_ERR_NO_DEVICE = 103,
    KS_ERR_CAPACITY = 104          /* more than 2^32-1 tuples, proteins or residues-per-protein on one shard */
} ks_status;

/* Moltypes: src/rust/encoding.rs:17-27.  "raw" is an alias of protein. */
typedef enum ks_moltype { KS_PROTEIN = 0, KS_DAYHOFF = 1, KS_HP = 2 } ks_moltype;

#define KS_SEED 42u                   /* src/rust/signature.rs:12 */
#define KS_PROTEIN_TO_MINHASH_RATIO 3 /* src/rust/signature.rs:13 */

const char *ks_last_error_message(void);
/* Detail of the last KS_ERR_INVALID_AMINO_ACID: the (upper-cased) character, its 1-based position
 * in the processed sequence (src/rust/aminoacid.rs:85-87) and the 0-based protein index. */
void ks_last_error_detail(uint32_t *ch, uint64_t *pos, uint64_t *protein_index);
int ks_abi_version(void);
/* Number of visible CUDA devices (0 when there is no driver/device). */
int ks_device_count(void);

/* encoding.rs:17-27: "protein"|"raw"|"hp"|"dayhoff"; otherwise KS_ERR_INVALID_MOLTYPE with the
 * reference's message "Invalid moltype: {}, only 'protein', 'hp', or 'dayhoff' are supported". */
ks_status ks_moltype_from_str(const char *moltype, ks_moltype *out);
const char *ks_moltype_name(ks_moltype m);
/* sourmash max_hash_for_scaled, reached via KmerMinHash::new (src/rust/signature.rs:124-131). */
uint64_t ks_max_hash(uint32_t scaled);
/* One residue through aa_to_dayhoff / aa_to_hp / identity (src/rust/encoding.rs:43-53). */
uint8_t ks_translate_residue(uint8_t aa, ks_moltype m);
/* sourmash md5sum of a sketch: MD5(ascii(3*ksize) || ascii(min_0) || ...) -> 32 hex chars + NUL. */
void ks_md5_of_mins(const uint64_t *mins, uint64_t n, uint32_t ksize, char out[33]);
/* kmerseek's id string: lowercase hex of the wrapping sum of mins (src/rust/signature.rs:277-279). */
void ks_id_of_mins(const uint64_t *mins, uint64_t n, char out[17]);

/* ---------------------------------------------------------------------------------------------
 * Ingest: FASTA / sequences -> packed residues + offsets in pinned host memory.
 * Replaces needletail::parse_fastx_file + the per-record Vec copies (src/rust/index.rs:920-935),
 * `to_uppercase` (:1000) and AminoAcidAmbiguity::validate_and_resolve (src/rust/aminoacid.rs:74-105).
 * Normalisation (KS_NORMALIZE_KMERSEEK, the index path of the Rust crate): upper-case; keep and stop at the first '*';
 * reject anything outside the 20 standard letters + X U O * + B Z J.  B/Z/J are resolved to D|N, E|Q, I|L -- at random in
 * the reference (rand::rng(), aminoacid.rs:45-54); here reproducibly:
 *     choice = splitmix64(ambig_seed ^ position_in_output) & 1          (0 -> D/E/I, 1 -> N/Q/L)
 * which is one of the outcomes the reference can produce, and depends on the residue's position in its own sequence only
 * (the same sequence resolves the same way wherever it stands, so a query that copies a target matches it fully).
 * KS_NORMALIZE_SOURMASH is what `kmerseek search` does to both of its inputs (src/python/kmerseek/sketch.py:28-40 ->
 * branchwater manysketch -> sourmash add_protein): upper-case only -- no validation, no '*' truncation, no resolution
 * (B/Z/J and anything else unknown translate to 'X' under dayhoff / hp and are hashed as they are under protein).
 * FASTA files are parsed by all host threads at once (KS_INGEST_THREADS overrides the count), straight into the
 * pinned upload buffers.
 * ------------------------------------------------------------------------------------------- */
#define KS_NORMALIZE_KMERSEEK 0
#define KS_NORMALIZE_SOURMASH 1
typedef struct ks_proteome ks_proteome;

/* plain, gzip, zstd, bzip2 or xz FASTA; names are the full header line without '>' (needletail id()). */
ks_status ks_proteome_from_fasta(const char *path, uint64_t ambig_seed, ks_proteome **out);
ks_status ks_proteome_from_fasta_mode(const char *path, uint64_t ambig_seed, int mode, ks_proteome **out);
/* n sequences (not NUL-terminated; lens in bytes); names may be NULL. */
ks_status ks_proteome_from_sequences(const char *const *seqs, const uint64_t *lens, const char *const *names,
                                     uint64_t n, uint64_t ambig_seed, ks_proteome **out);
ks_status ks_proteome_from_sequences_mode(const char *const *seqs, const uint64_t *lens, const char *const *names,
                                          uint64_t n, uint64_t ambig_seed, int mode, ks_proteome **out);
/* already-normalised residues: copied as is (no validation); offsets has n_proteins+1 entries. */
ks_status ks_proteome_from_packed(const uint8_t *residues, const uint64_t *offsets, uint64_t n_proteins,
                                  ks_proteome **out);
uint64_t ks_proteome_n_proteins(const ks_proteome *p);
uint64_t ks_proteome_n_residues(const ks_proteome *p);
const uint8_t *ks_proteome_residues(const ks_proteome *p); /* n_residues bytes (+64 zero pad) */
const uint64_t *ks_proteome_offsets(const ks_proteome *p); /* pinned, n_proteins+1 */
/* The upload copy: 5-bit codes (A-Z = 1..26, '*' = 27), 8 residues per 5 bytes little-endian, + 72 zero bytes; NULL
 * (*n_bytes = 0) when a byte outside A-Z and '*' is present -- the residues themselves are uploaded then. */
const uint8_t *ks_proteome_packed(const ks_proteome *p, uint64_t *n_bytes);
const char *ks_proteome_name(const ks_proteome *p, uint64_t i); /* "" when no names were given */
void ks_proteome_free(ks_proteome *p);

/* ---------------------------------------------------------------------------------------------
 * Index handle.  Replaces ProteomeIndex::new (src/rust/index.rs:130-225) minus RocksDB.
 * ------------------------------------------------------------------------------------------- */
typedef struct ks_index ks_index;

typedef struct ks_params {
    uint32_t ksize;              /* residues per k-mer (sourmash ksize is 3x this) */
    uint32_t scaled;             /* FracMinHash scaled; max_hash = ks_max_hash(scaled) */
    int32_t moltype;             /* ks_moltype */
    int32_t store_raw_sequences; /* recorded only (ks_index_params hands it back): the raw sequences of index.rs:737-743
                                    are strings of the host mirror; the device keeps no residues beyond the resident batch */
    int32_t device;              /* CUDA device ordinal */
    uint32_t reserved;
} ks_params;

ks_status ks_index_create(const ks_params *params, ks_index **out);
void ks_index_destroy(ks_index *idx);
ks_status ks_index_params(const ks_index *idx, ks_params *out);
/* The handle's compute stream as a cudaStream_t (for event timing by the caller). */
void *ks_index_stream(const ks_index *idx);
ks_status ks_index_sync(ks_index *idx);

/* Staged build (each stage is asynchronous on the handle's stream unless stated):
 *   upload   : pinned host residues/offsets -> HBM (cudaMemcpyAsync), replacing the resident batch
 *   sketch   : fused translate/window/MurmurHash3/filter/compaction kernel over the resident batch;
 *              appends (hash, protein, pos) tuples; protein ids continue from the proteins already added.
 *              = create_protein_signature's add_protein + process_kmers for the whole batch
 *              (src/rust/index.rs:719-786) followed by store_signatures (:800-830).
 *   finalize : radix sort by hash + CSR build (unique hashes, postings, per-protein sketch sizes).
 *              = the end state of combined_minhash / signatures after process_fasta (:907-961).
 * ks_index_add_proteome = upload + sketch (residues streamed in chunks, hashed as they land).  ks_index_clear drops
 * tuples and the CSR and keeps the resident batch: clear + ks_index_sketch_resident + ks_index_finalize builds it again
 * (the benchmark loop).  A build costs ONE host read-back (counts and flags, at the end of finalize).
 * A finalized index takes no more adds; ks_index_append_* extends it instead: the batch is built on its own by the same
 * stages and merged into the index on the device (one pass over the old postings, no rebuild, the old residues are not
 * needed), and the index is finalized again on return.  */
ks_status ks_index_upload(ks_index *idx, const ks_proteome *p);
ks_status ks_index_sketch_resident(ks_index *idx);
ks_status ks_index_add_proteome(ks_index *idx, const ks_proteome *p);
ks_status ks_index_finalize(ks_index *idx);
ks_status ks_index_clear(ks_index *idx);
/* process_fasta (src/rust/index.rs:907-961) minus save_state: read, add, finalize. */
ks_status ks_index_process_fasta(ks_index *idx, const char *path, uint64_t ambig_seed);
/* store_signatures (src/rust/index.rs:800-830) for sketches that were produced by ks_sketch_batch:
 * tuples with protein ids local to the batch (0..n_proteins-1). */
ks_status ks_index_add_tuples(ks_index *idx, const uint64_t *hash, const uint32_t *pid, const uint32_t *pos,
                              uint64_t n, uint64_t n_proteins);
/* Extend a FINALIZED index by one batch; the index is finalized again on return.  The batch's proteins get the ids
 * n_proteins .. n_proteins + batch - 1.  The result is the index that add(old batches) + add(batch) + finalize gives
 * (CSR, export, combined sketch, signature_count, search); stats count the merged totals and build_path is 4.
 * = a repeated process_fasta (src/rust/index.rs:907-961) on the same index.  Not finalized: KS_ERR_NOT_FINALIZED;
 * more than 2^31-1 tuples or 2^32-2 proteins in the merged index: KS_ERR_CAPACITY.  A failed append leaves the index as
 * it was.  The appended batch becomes the resident batch.  Device memory while appending: about twice the index.
 * An appended index cannot take part in ks_shard_search_batch (KS_ERR_VALIDATION). */
ks_status ks_index_append_proteome(ks_index *idx, const ks_proteome *p);
/* store_signatures (src/rust/index.rs:800-830) on a finalized index: arguments as ks_index_add_tuples. */
ks_status ks_index_append_tuples(ks_index *idx, const uint64_t *hash, const uint32_t *pid, const uint32_t *pos,
                                 uint64_t n, uint64_t n_proteins);

typedef struct ks_stats {
    uint64_t n_proteins;      /* proteins added (signatures incl. ones whose id collides) */
    uint64_t n_residues;
    uint64_t n_windows;       /* k-mer windows examined */
    uint64_t n_tuples;        /* kept (hash, protein, pos) occurrences */
    uint64_t n_unique_hashes; /* combined_minhash_size(), src/rust/index.rs:519-521 (after finalize) */
    uint64_t n_groups;        /* distinct (hash, protein) pairs = sum of per-protein sketch sizes */
    uint64_t n_distinct_ids;  /* signature_count(): what the last ks_index_signature_count() returned (0 before) */
    uint64_t device_bytes;    /* bytes currently allocated on the device by this handle */
    uint64_t sketch_launches, sort_launches, csr_launches, search_launches; /* kernels launched so far */
    float ms_upload, ms_sketch, ms_sort, ms_csr; /* device time of the last run of each stage (CUDA events) */
    float ms_search;
    float ms_sort_partition; /* part of ms_sort: partition by the top hash bits (library onesweep passes); dense path: the
                                second scatter level (or the library's key sort) */
    float ms_sort_bucket;    /* part of ms_sort: the bucket sort kernel (+ bucket table kernels); dense path: dense_bucket_kernel
                                (or the two streaming CSR passes) */
    uint32_t finalized;
    uint32_t build_path;     /* how the last finalize built the index: 0 general (hash tuples, partition + bucket sort),
                                1 dense k-mer space (hp, 8 <= k <= 24, scaled 1: rank keys), 2 the same with the keys
                                sorted by the library, 3 general with the unstable two-level partition (one batch of
                                hashes that rarely repeat), 4 a finalized index extended by ks_index_append_*, compact
                                layout */
} ks_stats;
/* Synchronises the handle's stream. */
ks_status ks_index_stats(ks_index *idx, ks_stats *out);
/* signature_count() (src/rust/index.rs:514-516): the signatures map is keyed by the id string (hex of the wrapping sum of
 * the sketch's mins, src/rust/signature.rs:277-279) and equal ids overwrite (:817-820), so this is the number of DISTINCT
 * ids over the proteins added.  Computed on demand from the finalized index (per-protein sums on the device). */
ks_status ks_index_signature_count(ks_index *idx, uint64_t *out);

/* ---------------------------------------------------------------------------------------------
 * Sketch export.  Replaces the accessors of ProteinSignature (src/rust/signature.rs:305-317):
 * signature().get_minhash().mins()/abunds(), kmer_infos(), and ProteinSignatureData
 * (signature.rs:322-335).  One batch call instead of one call per protein.
 * ------------------------------------------------------------------------------------------- */
typedef struct ks_sketch {
    uint64_t n_proteins;
    uint64_t n_tuples;   /* every kept window occurrence, in (protein, pos) order */
    uint64_t *hash;      /* [n_tuples] */
    uint32_t *pid;       /* [n_tuples] protein index within the batch */
    uint32_t *pos;       /* [n_tuples] 0-based window start in the processed sequence (index.rs:758-780) */
    uint64_t *sig_ptr;   /* [n_proteins+1] CSR into mins/abunds */
    uint64_t *mins;      /* per protein: sorted distinct hashes  (KmerMinHash.mins) */
    uint64_t *abunds;    /* per protein: occurrences of each min (KmerMinHash.abunds) */
} ks_sketch;
/* create_protein_signature (src/rust/index.rs:719-747) for a batch; does not modify the index's tuples. */
ks_status ks_sketch_batch(ks_index *idx, const ks_proteome *p, ks_sketch **out);
void ks_sketch_free(ks_sketch *s);
/* Per-protein sketches of everything in a finalized index (same layout; hash/pid/pos are the
 * postings in (hash, protein, pos) order). */
ks_status ks_index_export(ks_index *idx, ks_sketch **out);

/* The CSR table of a finalized index (host copies; free with ks_csr_free):
 * keys[U] sorted unique hashes = combined_minhash mins; row_ptr[U+1] into pid/pos; abundance of key u
 * in the combined sketch = row_ptr[u+1]-row_ptr[u] (src/rust/index.rs:802-827). */
typedef struct ks_csr {
    uint64_t n_keys, n_postings;
    uint64_t *keys;
    uint64_t *row_ptr;
    uint32_t *pid;
    uint32_t *pos;
} ks_csr;
ks_status ks_index_csr(ks_index *idx, ks_csr **out);
void ks_csr_free(ks_csr *c);

/* ---------------------------------------------------------------------------------------------
 * Search.  Replaces sourmash_plugin_branchwater.do_manysearch as called at
 * src/python/kmerseek/search.py:125-141 (threshold 0, abundance on, only pairs with overlap) and the
 * k-mer join of search.py:204-213 / sig2kmer.py:113-155 (hit positions).
 * Scores follow SURVEY.md Appendix A.6; float columns are fp64.
 * ------------------------------------------------------------------------------------------- */
#define KS_SEARCH_HITS 1u           /* also produce the hit list */
#define KS_SEARCH_DEVICE_ONLY 2u    /* leave results on the device; host arrays are NULL, counts are set */
#define KS_SEARCH_QUERY_SKETCHES 4u /* also return the queries' sketches (q_mins / q_abunds; needed for query_md5) */

typedef struct ks_search_result {
    uint64_t n_queries;
    /* per query: sketch (sorted distinct mins + abundances), CSR by query.  q_sig_ptr always comes back (|Q| of query q
     * = q_sig_ptr[q+1] - q_sig_ptr[q]); q_mins / q_abunds only with KS_SEARCH_QUERY_SKETCHES, else NULL. */
    uint64_t *q_sig_ptr; /* [n_queries+1] */
    uint64_t *q_mins;
    uint64_t *q_abunds;
    /* scored pairs, ordered by (query, target) */
    uint64_t n_pairs;
    uint32_t *pair_qid, *pair_pid;   /* pid is the index-wide protein id */
    uint32_t *intersect_hashes;      /* |Q n T| */
    uint32_t *q_size, *t_size;       /* |Q|, |T| (distinct hashes) */
    uint64_t *n_weighted_found;      /* sum of target abundances over the intersection */
    uint64_t *total_weighted_hashes; /* sum of all target abundances */
    double *containment, *containment_target_in_query, *max_containment, *jaccard;
    double *query_containment_ani, *match_containment_ani, *average_containment_ani, *max_containment_ani;
    double *average_abund, *median_abund, *std_abund, *f_weighted_target_in_query;
    /* hit list (KS_SEARCH_HITS), ordered by (query, qpos, target, tpos) */
    uint64_t n_hits;
    uint32_t *hit_qid, *hit_pid, *hit_qpos, *hit_tpos;
    uint64_t *hit_hash;
    /* Owner of the result's memory.  A result is ONE contiguous block -- every column above points into a single pinned
     * host block that one cudaMemcpyAsync filled -- and, with KS_SEARCH_DEVICE_ONLY, one device block that stays valid until
     * ks_search_result_free (which must then precede ks_index_destroy); see ks_search_result_device_column(). */
    void *device_block;
    float ms_device; /* device time of the search (query sketch + lookup + aggregation + scores [+ hits]) */
} ks_search_result;

ks_status ks_search_batch(ks_index *idx, const ks_proteome *queries, uint32_t flags, ks_search_result **out);
void ks_search_result_free(ks_search_result *r);
/* Device pointer of a named pair/hit column of a result ("pair_qid", "containment", "hit_tpos", ...),
 * or NULL.  Element counts are n_pairs / n_hits. */
void *ks_search_result_device_column(const ks_search_result *r, const char *name);
/* Split search for benchmarking with the query batch already resident in HBM. */
ks_status ks_query_upload(ks_index *idx, const ks_proteome *queries);
ks_status ks_search_resident(ks_index *idx, uint32_t flags, ks_search_result **out);

/* ---------------------------------------------------------------------------------------------
 * Multi-GPU (SURVEY.md section 8e; the reference is single-process, src/rust/index.rs:993-1005 is its only parallel
 * region).  One process per GPU; the proteome is sharded by protein in contiguous ranges (rank r owns index-wide protein
 * ids [pid_base_r, pid_base_r + n_proteins_r), ascending with the rank); every rank builds its own index with the calls
 * above -- the build has no collective.  Queries are replicated.  A target lives on exactly one shard, so each (query,
 * target) pair is scored completely by its owner and the merge on rank 0 is a concatenation in (query, target) order.
 * NCCL is bound at run time (dlopen of libnccl.so.2): without it these calls return KS_ERR_NCCL.
 * ------------------------------------------------------------------------------------------- */
typedef struct ks_comm ks_comm;
#define KS_COMM_ID_BYTES 128
/* ncclGetUniqueId: call on one rank, hand the bytes to every rank (any side channel), then ks_comm_create everywhere. */
ks_status ks_comm_unique_id(uint8_t id[KS_COMM_ID_BYTES]);
/* ncclCommInitRank on `device`; collective over all `world` ranks (at most 16). */
ks_status ks_comm_create(const uint8_t id[KS_COMM_ID_BYTES], int rank, int world, int device, ks_comm **out);
void ks_comm_destroy(ks_comm *c);
int ks_comm_rank(const ks_comm *c);
int ks_comm_world(const ks_comm *c);
/* ks_search_batch over all shards; collective.  Every rank passes the same query batch and its shard's pid_base.  Per
 * batch: one ncclAllGather (four counts per rank), one grouped ncclSend/ncclRecv of each shard's result block (exact
 * sizes) to rank 0 over NVLink, and a counting merge kernel there (no sort).  On rank 0 *out is the merged result
 * (protein ids index-wide, pairs ordered by (query, target), hits by (query, qpos, target, tpos)); on the other ranks
 * *out carries only this shard's n_pairs / n_hits.  Queries of more than 4096 windows: KS_ERR_CAPACITY. */
ks_status ks_shard_search_batch(ks_index *idx, ks_comm *comm, const ks_proteome *queries, uint32_t flags, uint64_t pid_base,
                                ks_search_result **out);

#ifdef __cplusplus
}
#endif
#endif /* KMERSEEK_B200_H */
