// kmerseek_b200.hpp -- header-only C++ facade over the C ABI (kmerseek_b200.h) with the names of the
// reference's Rust API: kmerseek::ProteomeIndex / ProteomeIndexBuilder (src/rust/index.rs:104-1017,
// 2975-3061), ProteinSignature accessors (src/rust/signature.rs:305-317), IndexError (src/rust/errors.rs).
// This is the host layer a compiled caller links against; it adds no compute of its own.
#pragma once
#include <cstdint>
#include <map>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "kmerseek_b200.h"

namespace kmerseek {

// IndexError (src/rust/errors.rs:4-55): one exception type carrying the status code and the message.
class IndexError : public std::runtime_error {
  public:
    IndexError(ks_status s, const std::string& m) : std::runtime_error(m), status(s) {}
    ks_status status;
};

inline void check(ks_status s) {
    if (s != KS_OK) throw IndexError(s, ks_last_error_message());
}

struct KmerInfo {  // src/rust/kmer.rs:7-12
    size_t ksize = 0;
    uint64_t hashval = 0;
    std::string encoded_kmer;
    std::map<std::string, std::vector<size_t>> original_kmer_to_position;
};

class ProteinSignature {  // src/rust/signature.rs:100-317
  public:
    std::string name;
    std::string md5sum;  // kmerseek id: hex of the wrapping sum of mins (signature.rs:277-279)
    std::vector<uint64_t> mins, abunds;
    std::vector<uint64_t> hashes;   // every kept window, position order
    std::vector<uint32_t> positions;
    std::string sequence;           // processed sequence (kept for kmer_infos / raw sequence storage)
    uint32_t protein_ksize = 0;
    std::string moltype;
    uint32_t minhash_ksize() const { return protein_ksize * KS_PROTEIN_TO_MINHASH_RATIO; }
    std::string sourmash_md5() const {
        char out[33];
        ks_md5_of_mins(mins.data(), mins.size(), protein_ksize, out);
        return out;
    }
    // hashval -> KmerInfo (src/rust/index.rs:770-780)
    std::map<uint64_t, KmerInfo> kmer_infos() const {
        std::map<uint64_t, KmerInfo> out;
        ks_moltype m;
        check(ks_moltype_from_str(moltype.c_str(), &m));
        for (size_t i = 0; i < hashes.size(); i++) {
            const std::string orig = sequence.substr(positions[i], protein_ksize);
            KmerInfo& ki = out[hashes[i]];
            if (ki.encoded_kmer.empty()) {
                ki.ksize = protein_ksize;
                ki.hashval = hashes[i];
                for (char c : orig) ki.encoded_kmer.push_back((char)ks_translate_residue((uint8_t)c, m));
            }
            ki.original_kmer_to_position[orig].push_back(positions[i]);
        }
        return out;
    }
};

class ProteomeIndexBuilder;

class ProteomeIndex {
  public:
    // ProteomeIndex::new (src/rust/index.rs:130-136); `path` names the index (persistence is out of scope)
    ProteomeIndex(const std::string& path, uint32_t ksize, uint32_t scaled, const std::string& moltype,
                  bool store_raw_sequences, int device = 0)
        : path_(path), moltype_(moltype) {
        ks_moltype m;
        check(ks_moltype_from_str(moltype.c_str(), &m));
        ks_params p{ksize, scaled, (int32_t)m, store_raw_sequences ? 1 : 0, device, 0};
        params_ = p;
        check(ks_index_create(&p, &h_));
    }
    ProteomeIndex(const ProteomeIndex&) = delete;
    ProteomeIndex& operator=(const ProteomeIndex&) = delete;
    ProteomeIndex(ProteomeIndex&& o) noexcept : h_(o.h_), params_(o.params_), path_(std::move(o.path_)), moltype_(std::move(o.moltype_)) { o.h_ = nullptr; }
    ~ProteomeIndex() { ks_index_destroy(h_); }

    static ProteomeIndexBuilder builder();
    // src/rust/index.rs:655-673
    static ProteomeIndex new_with_auto_filename(const std::string& base_path, uint32_t ksize, uint32_t scaled,
                                                const std::string& moltype, bool store_raw_sequences, int device = 0) {
        const size_t slash = base_path.find_last_of('/');
        const std::string dir = slash == std::string::npos ? "" : base_path.substr(0, slash + 1);
        const std::string file = slash == std::string::npos ? base_path : base_path.substr(slash + 1);
        return ProteomeIndex(dir + file + "." + moltype + ".k" + std::to_string(ksize) + ".scaled" +
                                 std::to_string(scaled) + ".kmerseek.rocksdb",
                             ksize, scaled, moltype, store_raw_sequences, device);
    }
    std::string generate_filename(const std::string& base) const {  // src/rust/index.rs:647-652
        return base + "." + moltype_ + ".k" + std::to_string(params_.ksize) + ".scaled" + std::to_string(params_.scaled) +
               ".kmerseek.rocksdb";
    }

    // create_protein_signature (src/rust/index.rs:719-747)
    ProteinSignature create_protein_signature(const std::string& sequence, const std::string& name) {
        const char* seqs[1] = {sequence.data()};
        const uint64_t lens[1] = {sequence.size()};
        const char* names[1] = {name.c_str()};
        ks_proteome* p = nullptr;
        check(ks_proteome_from_sequences(seqs, lens, names, 1, 0, &p));
        ks_sketch* s = nullptr;
        ks_status st = ks_sketch_batch(h_, p, &s);
        ProteinSignature sig;
        if (st == KS_OK) {
            sig.name = name;
            sig.protein_ksize = params_.ksize;
            sig.moltype = moltype_;
            sig.mins.assign(s->mins, s->mins + s->sig_ptr[1]);
            sig.abunds.assign(s->abunds, s->abunds + s->sig_ptr[1]);
            sig.hashes.assign(s->hash, s->hash + s->n_tuples);
            sig.positions.assign(s->pos, s->pos + s->n_tuples);
            sig.sequence.assign((const char*)ks_proteome_residues(p), ks_proteome_n_residues(p));
            char id[17];
            ks_id_of_mins(sig.mins.data(), sig.mins.size(), id);
            sig.md5sum = id;
            ks_sketch_free(s);
        }
        ks_proteome_free(p);
        check(st);
        return sig;
    }
    // store_signatures (src/rust/index.rs:800-830)
    void store_signatures(const std::vector<ProteinSignature>& sigs) {
        std::vector<uint64_t> h;
        std::vector<uint32_t> pid, pos;
        for (size_t i = 0; i < sigs.size(); i++) {
            h.insert(h.end(), sigs[i].hashes.begin(), sigs[i].hashes.end());
            pos.insert(pos.end(), sigs[i].positions.begin(), sigs[i].positions.end());
            pid.insert(pid.end(), sigs[i].hashes.size(), (uint32_t)i);
        }
        check(ks_index_add_tuples(h_, h.data(), pid.data(), pos.data(), h.size(), sigs.size()));
    }
    // store_signatures on a finalized index: the signatures are merged into it (ks_index_append_tuples)
    void append_signatures(const std::vector<ProteinSignature>& sigs) {
        std::vector<uint64_t> h;
        std::vector<uint32_t> pid, pos;
        for (size_t i = 0; i < sigs.size(); i++) {
            h.insert(h.end(), sigs[i].hashes.begin(), sigs[i].hashes.end());
            pos.insert(pos.end(), sigs[i].positions.begin(), sigs[i].positions.end());
            pid.insert(pid.end(), sigs[i].hashes.size(), (uint32_t)i);
        }
        check(ks_index_append_tuples(h_, h.data(), pid.data(), pos.data(), h.size(), sigs.size()));
    }
    // a repeated process_fasta on a finalized index: read, then merge the batch in (ks_index_append_proteome)
    void append_fasta(const std::string& fasta_path) {
        ks_proteome* p = nullptr;
        check(ks_proteome_from_fasta(fasta_path.c_str(), 0, &p));
        const ks_status st = ks_index_append_proteome(h_, p);
        ks_proteome_free(p);
        check(st);
    }
    // process_fasta (src/rust/index.rs:907-961); progress_interval / batch_size kept for signature parity
    void process_fasta(const std::string& fasta_path, uint32_t /*progress_interval*/ = 0, size_t /*batch_size*/ = 1000) {
        check(ks_index_process_fasta(h_, fasta_path.c_str(), 0));
    }
    size_t combined_minhash_size() {  // src/rust/index.rs:519-521
        check(ks_index_finalize(h_));
        ks_stats s;
        check(ks_index_stats(h_, &s));
        return s.n_unique_hashes;
    }
    size_t signature_count() {  // src/rust/index.rs:514-516: distinct ids (equal ids overwrite, :817-820)
        check(ks_index_finalize(h_));
        uint64_t n = 0;
        check(ks_index_signature_count(h_, &n));
        return (size_t)n;
    }
    ks_stats stats() {
        ks_stats s;
        check(ks_index_stats(h_, &s));
        return s;
    }
    bool store_raw_sequences() const { return params_.store_raw_sequences != 0; }
    ks_index* handle() { return h_; }

  private:
    ks_index* h_ = nullptr;
    ks_params params_{};
    std::string path_, moltype_;
};

// ProteomeIndexBuilder (src/rust/index.rs:2975-3061): same setters, same "... is required" messages
class ProteomeIndexBuilder {
  public:
    ProteomeIndexBuilder& path(const std::string& p) { path_ = p; has_path_ = true; return *this; }
    ProteomeIndexBuilder& ksize(uint32_t k) { ksize_ = k; has_k_ = true; return *this; }
    ProteomeIndexBuilder& scaled(uint32_t s) { scaled_ = s; has_s_ = true; return *this; }
    ProteomeIndexBuilder& moltype(const std::string& m) { moltype_ = m; has_m_ = true; return *this; }
    ProteomeIndexBuilder& store_raw_sequences(bool b) { raw_ = b; return *this; }
    ProteomeIndexBuilder& device(int d) { device_ = d; return *this; }
    ProteomeIndex build() {
        require("Database path is required");
        return ProteomeIndex(path_, ksize_, scaled_, moltype_, raw_, device_);
    }
    ProteomeIndex build_with_auto_filename() {
        require("Base path is required");
        return ProteomeIndex::new_with_auto_filename(path_, ksize_, scaled_, moltype_, raw_, device_);
    }

  private:
    void require(const char* path_msg) const {
        if (!has_path_) throw IndexError(KS_ERR_BUILDER, std::string("Builder error: ") + path_msg);
        if (!has_k_) throw IndexError(KS_ERR_BUILDER, "Builder error: K-mer size is required");
        if (!has_s_) throw IndexError(KS_ERR_BUILDER, "Builder error: Scaled value is required");
        if (!has_m_) throw IndexError(KS_ERR_BUILDER, "Builder error: Molecular type is required");
    }
    std::string path_, moltype_;
    uint32_t ksize_ = 0, scaled_ = 0;
    bool has_path_ = false, has_k_ = false, has_s_ = false, has_m_ = false, raw_ = false;
    int device_ = 0;
};

inline ProteomeIndexBuilder ProteomeIndex::builder() { return ProteomeIndexBuilder(); }

}  // namespace kmerseek
