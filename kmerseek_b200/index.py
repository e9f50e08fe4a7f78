"""Host-side mirror of the reference's index API over the C ABI.

Same names, argument meaning and error behaviour as `kmerseek::index::ProteomeIndex`,
`ProteomeIndexBuilder` (src/rust/index.rs:104-1017, 2975-3061), `ProteinSignature`
(src/rust/signature.rs:100-317) and `KmerInfo` (src/rust/kmer.rs:7-12), so that parity tests read like
the reference's own.  All compute goes through libkmerseek_b200.so (CUDA, sm_100a); nothing here hashes.
"""
import ctypes as C
import os

import numpy as np

from . import _ffi
from .errors import BuilderError, ValidationError, check

SEED = 42  # src/rust/signature.rs:12
PROTEIN_TO_MINHASH_RATIO = 3  # src/rust/signature.rs:13
MOLTYPE_IDS = {"protein": 0, "dayhoff": 1, "hp": 2}


def _moltype_id(moltype: str) -> int:
    out = C.c_int(0)
    check(_ffi.lib().ks_moltype_from_str(moltype.encode(), C.byref(out)))
    return out.value


def _np(ptr, n, dtype):
    if n == 0:
        return np.zeros(0, dtype=dtype)
    return np.ctypeslib.as_array(ptr, shape=(n,)).astype(dtype, copy=True)


def translate(seq: str, moltype: str) -> str:
    """encode_kmer (src/rust/encoding.rs:68-81) through the library's table."""
    m = _moltype_id(moltype)
    L = _ffi.lib()
    return "".join(chr(L.ks_translate_residue(ord(c), m)) for c in seq)


def max_hash(scaled: int) -> int:
    return _ffi.lib().ks_max_hash(scaled)


def md5_of_mins(mins, ksize: int) -> str:
    mins = np.ascontiguousarray(mins, dtype=np.uint64)
    buf = C.create_string_buffer(33)
    _ffi.lib().ks_md5_of_mins(mins.ctypes.data_as(_ffi.u64p), len(mins), ksize, buf)
    return buf.value.decode()


def id_of_mins(mins) -> str:
    mins = np.ascontiguousarray(mins, dtype=np.uint64)
    buf = C.create_string_buffer(17)
    _ffi.lib().ks_id_of_mins(mins.ctypes.data_as(_ffi.u64p), len(mins), buf)
    return buf.value.decode()


class Proteome:
    """Packed, normalised sequences in pinned host memory (ks_proteome)."""

    def __init__(self, handle):
        self._h = handle

    MODES = {"kmerseek": _ffi.KS_NORMALIZE_KMERSEEK, "sourmash": _ffi.KS_NORMALIZE_SOURMASH}

    @classmethod
    def from_fasta(cls, path, ambig_seed=0, mode="kmerseek"):
        """mode "kmerseek": the Rust crate's index path (upper-case, '*' truncation, B/Z/J resolved, validation);
        "sourmash": what `kmerseek search` does to both inputs (upper-case only)."""
        h = C.c_void_p()
        check(_ffi.lib().ks_proteome_from_fasta_mode(os.fspath(path).encode(), ambig_seed, cls.MODES[mode], C.byref(h)))
        return cls(h)

    @classmethod
    def from_sequences(cls, seqs, names=None, ambig_seed=0, mode="kmerseek"):
        n = len(seqs)
        raw = [s.encode() if isinstance(s, str) else bytes(s) for s in seqs]
        arr = (C.c_char_p * max(n, 1))(*raw)
        lens = (C.c_uint64 * max(n, 1))(*[len(r) for r in raw])
        nm = None
        if names is not None:
            nm = (C.c_char_p * max(n, 1))(*[x.encode() for x in names])
        h = C.c_void_p()
        check(_ffi.lib().ks_proteome_from_sequences_mode(arr, lens, nm, n, ambig_seed, cls.MODES[mode], C.byref(h)))
        return cls(h)

    @classmethod
    def from_packed(cls, residues, offsets):
        residues = np.ascontiguousarray(residues, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        h = C.c_void_p()
        rp = residues.ctypes.data_as(_ffi.u8p) if len(residues) else None
        check(_ffi.lib().ks_proteome_from_packed(rp, offsets.ctypes.data_as(_ffi.u64p), len(offsets) - 1, C.byref(h)))
        return cls(h)

    @property
    def n_proteins(self):
        return _ffi.lib().ks_proteome_n_proteins(self._h)

    @property
    def n_residues(self):
        return _ffi.lib().ks_proteome_n_residues(self._h)

    def _view(self, ptr, n, dtype):
        """Read-only numpy view of one of the proteome's pinned buffers (no copy; valid until close())."""
        if n == 0:
            return np.zeros(0, dtype=dtype)
        a = np.ctypeslib.as_array(ptr, shape=(n,))
        a.flags.writeable = False
        return a

    @property
    def residues(self):
        """The normalised residues: a read-only view of the pinned buffer (copy it to keep it past close())."""
        return self._view(_ffi.lib().ks_proteome_residues(self._h), self.n_residues, np.uint8)

    @property
    def offsets(self):
        return self._view(_ffi.lib().ks_proteome_offsets(self._h), self.n_proteins + 1, np.uint64)

    def name(self, i):
        return _ffi.lib().ks_proteome_name(self._h, i).decode("utf-8", "replace")

    @property
    def names(self):
        return [self.name(i) for i in range(self.n_proteins)]

    def sequence(self, i):
        o = self.offsets  # views: a call costs the protein's own bytes, not the proteome's
        return self.residues[int(o[i]):int(o[i + 1])].tobytes().decode()

    def close(self):
        if self._h:
            _ffi.lib().ks_proteome_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class KmerInfo:
    """src/rust/kmer.rs:7-12"""

    def __init__(self, ksize, hashval, encoded_kmer):
        self.ksize, self.hashval, self.encoded_kmer = ksize, hashval, encoded_kmer
        self.original_kmer_to_position = {}

    def unique_kmer_count(self):
        return len(self.original_kmer_to_position)

    def total_occurrences(self):
        return sum(len(v) for v in self.original_kmer_to_position.values())

    def has_position(self, position):
        return any(position in v for v in self.original_kmer_to_position.values())


class ProteinSignature:
    """One protein's sketch + k-mer positions (src/rust/signature.rs:100-317).

    `md5sum` is kmerseek's id string (hex of the wrapping sum of mins, signature.rs:277-279);
    `sourmash_md5()` is the real sourmash md5sum used in .sig files and manysearch rows."""

    def __init__(self, name, moltype, protein_ksize, scaled, mins, abunds, hashes, positions, sequence, store_raw):
        self.name = name
        self._moltype, self._ksize, self._scaled = moltype, protein_ksize, scaled
        self._mins, self._abunds = mins, abunds
        self._hashes, self._positions = hashes, positions  # every kept window, in position order
        self._sequence = sequence
        self._store_raw = store_raw
        self.md5sum = id_of_mins(mins)
        self._infos = None

    def protein_ksize(self):
        return self._ksize

    def minhash_ksize(self):
        return self._ksize * PROTEIN_TO_MINHASH_RATIO

    def moltype(self):
        return self._moltype

    def scaled(self):
        return self._scaled

    def mins(self):
        return self._mins

    def abunds(self):
        return self._abunds

    def size(self):
        return len(self._mins)

    def sourmash_md5(self):
        return md5_of_mins(self._mins, self._ksize)

    def get_raw_sequence(self):
        return self._sequence if self._store_raw else None

    def has_efficient_data(self):
        """src/rust/signature.rs: the raw sequence is there (store_raw_sequences)."""
        return self._store_raw

    def kmer_infos(self):
        """hashval -> KmerInfo (src/rust/index.rs:770-780)."""
        if self._infos is None:
            infos = {}
            for h, p in zip(self._hashes.tolist(), self._positions.tolist()):
                orig = self._sequence[p:p + self._ksize]
                ki = infos.get(h)
                if ki is None:
                    ki = infos[h] = KmerInfo(self._ksize, h, translate(orig, self._moltype))
                ki.original_kmer_to_position.setdefault(orig, []).append(p)
            self._infos = infos
        return self._infos


class StoredSignature(tuple):
    """A signature as the index holds it (the value type of get_signatures()): unpacks as (name, mins, abunds) and
    carries the raw sequence when the index was created with store_raw_sequences (src/rust/index.rs:737-743,
    signature.rs:305-317)."""

    def __new__(cls, name, mins, abunds, raw_sequence=None):
        self = super().__new__(cls, (name, mins, abunds))
        self.name, self.raw_sequence = name, raw_sequence
        return self

    def mins(self):
        return self[1]

    def abunds(self):
        return self[2]

    def get_raw_sequence(self):
        return self.raw_sequence

    def has_efficient_data(self):
        return self.raw_sequence is not None


class ProteomeIndexBuilder:
    """src/rust/index.rs:2975-3061"""

    def __init__(self):
        self._path = self._ksize = self._scaled = self._moltype = None
        self._store_raw = False
        self._device = 0

    def path(self, path):
        self._path = path
        return self

    def ksize(self, ksize):
        self._ksize = ksize
        return self

    def scaled(self, scaled):
        self._scaled = scaled
        return self

    def moltype(self, moltype):
        self._moltype = moltype
        return self

    def store_raw_sequences(self, flag):
        self._store_raw = bool(flag)
        return self

    def device(self, device):
        self._device = device
        return self

    def _required(self, path_msg):
        if self._path is None:
            raise BuilderError(path_msg)
        if self._ksize is None:
            raise BuilderError("K-mer size is required")
        if self._scaled is None:
            raise BuilderError("Scaled value is required")
        if self._moltype is None:
            raise BuilderError("Molecular type is required")

    def build(self):
        self._required("Database path is required")
        return ProteomeIndex(self._path, self._ksize, self._scaled, self._moltype, self._store_raw, device=self._device)

    def build_with_auto_filename(self):
        self._required("Base path is required")
        return ProteomeIndex.new_with_auto_filename(self._path, self._ksize, self._scaled, self._moltype,
                                                    self._store_raw, device=self._device)


class ProteomeIndex:
    """GPU-resident proteome index (ks_index).  Mirrors src/rust/index.rs:104-1017 without RocksDB:
    `path` is kept as the index's name only (persistence is SURVEY section 8f row N2)."""

    def __init__(self, path, ksize, scaled, moltype, store_raw_sequences=False, device=0, ambig_seed=0):
        self.path = os.fspath(path)
        self.ksize, self.scaled, self.moltype = int(ksize), int(scaled), moltype
        self._store_raw = bool(store_raw_sequences)
        self.ambig_seed = ambig_seed
        self._names = []
        self._raw = []  # raw sequences, protein order (only with store_raw_sequences)
        self._h = None
        p = _ffi.ks_params(self.ksize, self.scaled, _moltype_id(moltype), int(self._store_raw), device, 0)
        h = C.c_void_p()
        check(_ffi.lib().ks_index_create(C.byref(p), C.byref(h)))
        self._h = h

    # -- constructors ---------------------------------------------------------------------------
    @classmethod
    def new(cls, path, ksize, scaled, moltype, store_raw_sequences=False, **kw):
        return cls(path, ksize, scaled, moltype, store_raw_sequences, **kw)

    @staticmethod
    def builder():
        return ProteomeIndexBuilder()

    @classmethod
    def new_with_auto_filename(cls, base_path, ksize, scaled, moltype, store_raw_sequences=False, **kw):
        base_path = os.fspath(base_path)
        name = f"{os.path.basename(base_path)}.{moltype}.k{ksize}.scaled{scaled}.kmerseek.rocksdb"
        return cls(os.path.join(os.path.dirname(base_path), name), ksize, scaled, moltype, store_raw_sequences, **kw)

    def generate_filename(self, base_name):
        return f"{base_name}.{self.moltype}.k{self.ksize}.scaled{self.scaled}.kmerseek.rocksdb"

    def store_raw_sequences(self):
        return self._store_raw

    # -- sketching --------------------------------------------------------------------------------
    def create_protein_signatures(self, sequences, names):
        """Batch form of create_protein_signature: one kernel launch for all sequences."""
        prot = Proteome.from_sequences(sequences, names, self.ambig_seed)
        out = C.POINTER(_ffi.ks_sketch)()
        check(_ffi.lib().ks_sketch_batch(self._h, prot._h, C.byref(out)))
        try:
            s = out.contents
            n, P = s.n_tuples, s.n_proteins
            hashes, pid, pos = _np(s.hash, n, np.uint64), _np(s.pid, n, np.uint32), _np(s.pos, n, np.uint32)
            sig_ptr = _np(s.sig_ptr, P + 1, np.uint64)
            E = int(sig_ptr[-1]) if P else 0
            mins, abunds = _np(s.mins, E, np.uint64), _np(s.abunds, E, np.uint64)
        finally:
            _ffi.lib().ks_sketch_free(out)
        bounds = np.searchsorted(pid, np.arange(P + 1))
        sigs = []
        for i in range(P):
            a, b = int(sig_ptr[i]), int(sig_ptr[i + 1])
            t0, t1 = int(bounds[i]), int(bounds[i + 1])
            sigs.append(ProteinSignature(names[i], self.moltype, self.ksize, self.scaled, mins[a:b], abunds[a:b],
                                         hashes[t0:t1], pos[t0:t1], prot.sequence(i), self._store_raw))
        prot.close()
        return sigs

    def sketch_proteome(self, proteome: "Proteome"):
        """[(mins, abunds)] for every protein of a packed proteome (ks_sketch_batch); the index is left untouched."""
        out = C.POINTER(_ffi.ks_sketch)()
        check(_ffi.lib().ks_sketch_batch(self._h, proteome._h, C.byref(out)))
        try:
            s = out.contents
            P = s.n_proteins
            sig_ptr = _np(s.sig_ptr, P + 1, np.uint64)
            E = int(sig_ptr[-1]) if P else 0
            mins, abunds = _np(s.mins, E, np.uint64), _np(s.abunds, E, np.uint64)
        finally:
            _ffi.lib().ks_sketch_free(out)
        return [(mins[int(sig_ptr[i]):int(sig_ptr[i + 1])], abunds[int(sig_ptr[i]):int(sig_ptr[i + 1])]) for i in range(P)]

    def create_protein_signature(self, sequence, name):
        """src/rust/index.rs:719-747"""
        return self.create_protein_signatures([sequence], [name])[0]

    def store_signatures(self, protein_signatures):
        """src/rust/index.rs:800-830: add already-made signatures to the index."""
        if not protein_signatures:
            return
        h, pid, pos = self._signature_tuples(protein_signatures)
        check(_ffi.lib().ks_index_add_tuples(self._h, h.ctypes.data_as(_ffi.u64p), pid.ctypes.data_as(_ffi.u32p),
                                             pos.ctypes.data_as(_ffi.u32p), len(h), len(protein_signatures)))
        self._names.extend(s.name for s in protein_signatures)
        if self._store_raw:
            self._raw.extend(s._sequence for s in protein_signatures)

    @staticmethod
    def _signature_tuples(protein_signatures):
        """(hash, protein, pos) of every kept window, protein ids local to the list."""
        if not protein_signatures:
            return np.zeros(0, np.uint64), np.zeros(0, np.uint32), np.zeros(0, np.uint32)
        h = np.concatenate([s._hashes for s in protein_signatures]).astype(np.uint64)
        pos = np.concatenate([s._positions for s in protein_signatures]).astype(np.uint32)
        pid = np.concatenate([np.full(len(s._hashes), i, dtype=np.uint32) for i, s in enumerate(protein_signatures)])
        return h, pid, pos

    def store_signatures_batch(self, protein_signatures):
        self.store_signatures(list(protein_signatures))

    def add_proteome(self, proteome: Proteome):
        check(_ffi.lib().ks_index_add_proteome(self._h, proteome._h))
        self._names.extend(proteome.names)
        if self._store_raw:
            self._raw.extend(proteome.sequence(i) for i in range(proteome.n_proteins))

    def process_fasta(self, fasta_path, progress_interval=0, batch_size=1000):
        """src/rust/index.rs:907-961.  `batch_size` is accepted for signature parity; the whole file is one
        device batch (the reference batches only to bound rayon's working set)."""
        if progress_interval:
            print("Reading FASTA file with automatic compression detection and parallel processing...")
        prot = Proteome.from_fasta(fasta_path, self.ambig_seed)
        self.add_proteome(prot)
        n = prot.n_proteins
        prot.close()
        self.finalize()
        if progress_interval:
            print(f"Successfully processed and stored {n} sequences.")

    def append_proteome(self, proteome: Proteome):
        """Extend the finalized index by one batch (ks_index_append_proteome): the batch is built on the device and merged
        into the index, which stays finalized; its proteins take the ids after the ones already there."""
        check(_ffi.lib().ks_index_append_proteome(self._h, proteome._h))
        self._names.extend(proteome.names)
        if self._store_raw:
            self._raw.extend(proteome.sequence(i) for i in range(proteome.n_proteins))

    def append_fasta(self, fasta_path):
        """A repeated process_fasta (src/rust/index.rs:907-961) on a finalized index: read, then append_proteome."""
        prot = Proteome.from_fasta(fasta_path, self.ambig_seed)
        try:
            self.append_proteome(prot)
        finally:
            prot.close()

    def append_signatures(self, protein_signatures):
        """store_signatures (src/rust/index.rs:800-830) on a finalized index (ks_index_append_tuples)."""
        h, pid, pos = self._signature_tuples(protein_signatures)
        check(_ffi.lib().ks_index_append_tuples(self._h, h.ctypes.data_as(_ffi.u64p), pid.ctypes.data_as(_ffi.u32p),
                                                pos.ctypes.data_as(_ffi.u32p), len(h), len(protein_signatures)))
        self._names.extend(s.name for s in protein_signatures)
        if self._store_raw:
            self._raw.extend(s._sequence for s in protein_signatures)

    def finalize(self):
        check(_ffi.lib().ks_index_finalize(self._h))

    def clear(self):
        check(_ffi.lib().ks_index_clear(self._h))
        self._names = []
        self._raw = []

    # -- accessors ----------------------------------------------------------------------------------
    def stats(self):
        s = _ffi.ks_stats()
        check(_ffi.lib().ks_index_stats(self._h, C.byref(s)))
        return {n: getattr(s, n) for n, _ in _ffi.ks_stats._fields_}

    def names(self):
        return list(self._names)

    def combined_minhash_size(self):
        """src/rust/index.rs:519-521"""
        self.finalize()
        return self.stats()["n_unique_hashes"]

    def get_combined_minhash(self):
        """(mins, abunds) of combined_minhash (src/rust/index.rs:802-827)."""
        keys, row_ptr, _, _ = self.csr()
        return keys, np.diff(row_ptr)

    def csr(self):
        self.finalize()
        out = C.POINTER(_ffi.ks_csr)()
        check(_ffi.lib().ks_index_csr(self._h, C.byref(out)))
        try:
            c = out.contents
            return (_np(c.keys, c.n_keys, np.uint64), _np(c.row_ptr, c.n_keys + 1, np.uint64),
                    _np(c.pid, c.n_postings, np.uint32), _np(c.pos, c.n_postings, np.uint32))
        finally:
            _ffi.lib().ks_csr_free(out)

    def export_sketches(self):
        """Per-protein (mins, abunds) for everything in the index, in protein order."""
        self.finalize()
        out = C.POINTER(_ffi.ks_sketch)()
        check(_ffi.lib().ks_index_export(self._h, C.byref(out)))
        try:
            s = out.contents
            P = s.n_proteins
            sig_ptr = _np(s.sig_ptr, P + 1, np.uint64)
            E = int(sig_ptr[-1]) if P else 0
            mins, abunds = _np(s.mins, E, np.uint64), _np(s.abunds, E, np.uint64)
        finally:
            _ffi.lib().ks_sketch_free(out)
        return [(mins[int(sig_ptr[i]):int(sig_ptr[i + 1])], abunds[int(sig_ptr[i]):int(sig_ptr[i + 1])]) for i in range(P)]

    def get_signatures(self):
        """id string -> StoredSignature (name, mins, abunds, raw sequence when the index stores them); equal ids overwrite,
        last in input order wins (DashMap insert at src/rust/index.rs:817-820)."""
        out = {}
        for i, (m, a) in enumerate(self.export_sketches()):
            raw = self._raw[i] if (self._store_raw and i < len(self._raw)) else None
            out[id_of_mins(m)] = StoredSignature(self._names[i] if i < len(self._names) else str(i), m, a, raw)
        return out

    def signature_count(self):
        """src/rust/index.rs:514-516: distinct ids (equal ids overwrite), counted by the library from the device index."""
        self.finalize()
        out = C.c_uint64(0)
        check(_ffi.lib().ks_index_signature_count(self._h, C.byref(out)))
        return out.value

    def print_stats(self):
        """src/rust/index.rs:628-639"""
        print("ProteomeIndex Statistics:")
        print(f"  K-mer size: {self.ksize}")
        print(f"  Scaled: {self.scaled}")
        print(f"  Molecular type: {self.moltype}")
        print(f"  Combined minhash size: {self.combined_minhash_size()}")
        print(f"  Raw sequence storage: {'enabled' if self._store_raw else 'disabled'}")

    def is_equivalent_to(self, other):
        """src/rust/index.rs:523-626: same parameters, same signatures, same combined mins."""
        if (self.ksize, self.scaled, self.moltype) != (other.ksize, other.scaled, other.moltype):
            return False
        a, b = self.get_signatures(), other.get_signatures()
        if set(a) != set(b):
            return False
        for k in a:
            if not (np.array_equal(a[k][1], b[k][1]) and np.array_equal(a[k][2], b[k][2])):
                return False
        return np.array_equal(self.get_combined_minhash()[0], other.get_combined_minhash()[0])

    # -- lifecycle ----------------------------------------------------------------------------------
    def close(self):
        if self._h:
            _ffi.lib().ks_index_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()
