//! NOT COMPILED IN THIS REPOSITORY'S BUILD ENVIRONMENT (no cargo/rustc in the image).
//! Hand-written mirror of include/kmerseek_b200.h (what bindgen would emit), plus the thin safe wrapper that
//! keeps kmerseek's `ProteomeIndex` surface (src/rust/index.rs:104-1017) on top of it.
#![allow(non_camel_case_types)]
use libc::{c_char, c_int, c_void};

#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct ks_params {
    pub ksize: u32,
    pub scaled: u32,
    pub moltype: i32, // 0 protein | 1 dayhoff | 2 hp  (src/rust/encoding.rs:17-27)
    pub store_raw_sequences: i32,
    pub device: i32,
    pub reserved: u32,
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct ks_stats {
    pub n_proteins: u64,
    pub n_residues: u64,
    pub n_windows: u64,
    pub n_tuples: u64,
    pub n_unique_hashes: u64, // combined_minhash_size(), src/rust/index.rs:519-521
    pub n_groups: u64,
    pub n_distinct_ids: u64,
    pub device_bytes: u64,
    pub sketch_launches: u64,
    pub sort_launches: u64,
    pub csr_launches: u64,
    pub search_launches: u64,
    pub ms_upload: f32,
    pub ms_sketch: f32,
    pub ms_sort: f32,
    pub ms_csr: f32,
    pub ms_search: f32,
    pub ms_sort_partition: f32,
    pub ms_sort_bucket: f32,
    pub finalized: u32,
    pub build_path: u32, // 0 general, 1 dense k-mer space, 2 dense with the library's key sort, 3 general / unstable partition
}

#[repr(C)]
pub struct ks_sketch {
    pub n_proteins: u64,
    pub n_tuples: u64,
    pub hash: *mut u64,
    pub pid: *mut u32,
    pub pos: *mut u32,
    pub sig_ptr: *mut u64,
    pub mins: *mut u64,
    pub abunds: *mut u64,
}

pub enum ks_index {}
pub enum ks_proteome {}
pub enum ks_search_result {} // field layout: see the header; read through accessors in the safe wrapper
pub enum ks_comm {}

pub const KS_SEARCH_HITS: u32 = 1;
pub const KS_SEARCH_DEVICE_ONLY: u32 = 2;
pub const KS_SEARCH_QUERY_SKETCHES: u32 = 4;
pub const KS_NORMALIZE_KMERSEEK: c_int = 0; // index path: validate_and_resolve (src/rust/aminoacid.rs:74-105)
pub const KS_NORMALIZE_SOURMASH: c_int = 1; // search path: upper-case only (sourmash add_protein)
pub const KS_COMM_ID_BYTES: usize = 128;

extern "C" {
    pub fn ks_last_error_message() -> *const c_char;
    pub fn ks_last_error_detail(ch: *mut u32, pos: *mut u64, protein_index: *mut u64);
    pub fn ks_moltype_from_str(moltype: *const c_char, out: *mut c_int) -> c_int;
    pub fn ks_max_hash(scaled: u32) -> u64;
    pub fn ks_proteome_from_fasta(path: *const c_char, ambig_seed: u64, out: *mut *mut ks_proteome) -> c_int;
    pub fn ks_proteome_from_sequences(seqs: *const *const c_char, lens: *const u64, names: *const *const c_char,
                                      n: u64, ambig_seed: u64, out: *mut *mut ks_proteome) -> c_int;
    pub fn ks_proteome_from_fasta_mode(path: *const c_char, ambig_seed: u64, mode: c_int, out: *mut *mut ks_proteome) -> c_int;
    pub fn ks_proteome_from_sequences_mode(seqs: *const *const c_char, lens: *const u64, names: *const *const c_char,
                                           n: u64, ambig_seed: u64, mode: c_int, out: *mut *mut ks_proteome) -> c_int;
    pub fn ks_proteome_packed(p: *const ks_proteome, n_bytes: *mut u64) -> *const u8;
    pub fn ks_proteome_free(p: *mut ks_proteome);
    pub fn ks_index_create(params: *const ks_params, out: *mut *mut ks_index) -> c_int;
    pub fn ks_index_destroy(idx: *mut ks_index);
    pub fn ks_index_add_proteome(idx: *mut ks_index, p: *const ks_proteome) -> c_int;
    pub fn ks_index_finalize(idx: *mut ks_index) -> c_int;
    pub fn ks_index_process_fasta(idx: *mut ks_index, path: *const c_char, ambig_seed: u64) -> c_int;
    // a repeated process_fasta / store_signatures (src/rust/index.rs:800-830, 907-961) on a finalized index
    pub fn ks_index_append_proteome(idx: *mut ks_index, p: *const ks_proteome) -> c_int;
    pub fn ks_index_append_tuples(idx: *mut ks_index, hash: *const u64, pid: *const u32, pos: *const u32, n: u64,
                                  n_proteins: u64) -> c_int;
    pub fn ks_index_stats(idx: *mut ks_index, out: *mut ks_stats) -> c_int;
    pub fn ks_index_signature_count(idx: *mut ks_index, out: *mut u64) -> c_int; // src/rust/index.rs:514-516
    pub fn ks_sketch_batch(idx: *mut ks_index, p: *const ks_proteome, out: *mut *mut ks_sketch) -> c_int;
    pub fn ks_sketch_free(s: *mut ks_sketch);
    pub fn ks_search_batch(idx: *mut ks_index, queries: *const ks_proteome, flags: u32,
                           out: *mut *mut ks_search_result) -> c_int;
    pub fn ks_search_result_free(r: *mut ks_search_result);
    pub fn ks_search_result_device_column(r: *const ks_search_result, name: *const c_char) -> *mut c_void;
    // multi-GPU: one process per GPU, proteome sharded by protein (no precedent in the reference, which is single-process)
    pub fn ks_comm_unique_id(id: *mut u8) -> c_int;
    pub fn ks_comm_create(id: *const u8, rank: c_int, world: c_int, device: c_int, out: *mut *mut ks_comm) -> c_int;
    pub fn ks_comm_destroy(c: *mut ks_comm);
    pub fn ks_shard_search_batch(idx: *mut ks_index, comm: *mut ks_comm, queries: *const ks_proteome, flags: u32,
                                 pid_base: u64, out: *mut *mut ks_search_result) -> c_int;
}

/// How `IndexError` (src/rust/errors.rs:4-55) is rebuilt from a status code.
pub fn status_to_index_error(status: c_int) -> String {
    let msg = unsafe { std::ffi::CStr::from_ptr(ks_last_error_message()) }.to_string_lossy().into_owned();
    match status {
        1 => format!("InvalidMoltype: {msg}"),
        2 => msg, // already "Invalid amino acid '{c}' found at position {p}" (errors.rs:14-15)
        7 => format!("ParseError: {msg}"),
        8 => format!("BuilderError: {msg}"),
        _ => msg,
    }
}
