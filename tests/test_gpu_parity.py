"""Parity of the CUDA path (through the C ABI) against the oracle and the reference's golden vectors.
Bit-exact for hashes, retained k-mers, positions, postings and hit lists; scores within 1e-6 relative
(the tolerance BASELINE.json's north_star states).  Needs a GPU: run with -m gpu."""
import csv
import io
import os

import numpy as np
import pytest

from conftest import fasta_path

pytestmark = pytest.mark.gpu

SCORE_RTOL = 1e-6  # north_star: "floating-point scores within 1e-6 relative"


@pytest.fixture(scope="module")
def K():
    import kmerseek_b200
    return kmerseek_b200


@pytest.fixture(scope="module")
def O():
    from oracle import oracle
    return oracle


def _oracle_tuples(O, prot, k, moltype, scaled):
    return O.sketch_tuples(prot.residues, prot.offsets, k, moltype, scaled)


def _gpu_tuples(K, prot, k, moltype, scaled):
    """(hash, pid, pos) in (pid, pos) order + per-protein sketches, via ks_sketch_batch."""
    import ctypes as C
    from kmerseek_b200 import _ffi
    from kmerseek_b200.errors import check
    from kmerseek_b200.index import _np
    with K.ProteomeIndex("t", k, scaled, moltype) as idx:
        out = C.POINTER(_ffi.ks_sketch)()
        check(_ffi.lib().ks_sketch_batch(idx._h, prot._h, C.byref(out)))
        s = out.contents
        n, P = s.n_tuples, s.n_proteins
        h, pid, pos = _np(s.hash, n, np.uint64), _np(s.pid, n, np.uint32), _np(s.pos, n, np.uint32)
        sp = _np(s.sig_ptr, P + 1, np.uint64)
        E = int(sp[-1]) if P else 0
        mins, ab = _np(s.mins, E, np.uint64), _np(s.abunds, E, np.uint64)
        _ffi.lib().ks_sketch_free(out)
    return h, pid, pos, [(mins[int(sp[i]):int(sp[i + 1])], ab[int(sp[i]):int(sp[i + 1])]) for i in range(P)]


# ---- golden vectors of the reference -------------------------------------------------------------
@pytest.mark.parametrize("moltype", ["protein", "dayhoff", "hp"])
def test_golden_kmer_infos(K, golden_rust, moltype):
    g = golden_rust["kmer_tables"][moltype]  # src/rust/index.rs:1084-1103,1187-1205,1309-1326
    with K.ProteomeIndex("t", g["ksize"], g["scaled"], moltype) as idx:
        sig = idx.create_protein_signature(g["sequence"], "test_protein")
        infos = sig.kmer_infos()
        assert len(infos) == len(g["rows"])
        for row in g["rows"]:
            ki = infos[int(row["hash"])]
            if row["encoded"] is not None:
                assert ki.encoded_kmer == row["encoded"]
            assert set(ki.original_kmer_to_position) == set(row["originals"])
            assert sorted(p for v in ki.original_kmer_to_position.values() for p in v) == sorted(row["positions"])
        idx.store_signatures([sig])  # src/rust/index.rs:1414-1441
        assert idx.signature_count() == 1
        assert idx.combined_minhash_size() == len(g["rows"])


@pytest.mark.parametrize("moltype", ["protein", "dayhoff", "hp"])
def test_golden_two_record_fasta(K, golden_rust, moltype, tmp_path):
    g = golden_rust["index_tests"][f"test_process_fasta_moltype_{moltype}"]
    f = tmp_path / "test.fasta"
    f.write_text(golden_rust["fixtures"]["TEST_FASTA_CONTENT"])
    with K.ProteomeIndex(tmp_path / "db", g["ksize"], g["scaled"], moltype) as idx:
        idx.process_fasta(f, 0, 1000)
        sigs = idx.get_signatures()
        assert len(sigs) == g["n_signatures"]
        for i, n in g["ids"].items():
            assert len(sigs[i][1]) == n
        assert idx.combined_minhash_size() == g["combined_size"]


@pytest.mark.parametrize("test", ["test_process_fasta_gz_moltype_protein", "test_process_fasta_gz_moltype_dayhoff",
                                  "test_process_fasta_gz_moltype_hp", "test_manual_vs_auto_index_equivalence"])
def test_golden_bcl2_first25(K, golden_rust, test):
    g = golden_rust["index_tests"][test]  # src/rust/index.rs:1812-1843,1871-1902,1937-1968,2403-2418
    with K.ProteomeIndex("db", g["ksize"], g["scaled"], g["moltype"]) as idx:
        idx.process_fasta(fasta_path("bcl2_first25.fasta.gz"), 0, 1000)
        sigs = idx.get_signatures()
        assert len(sigs) == 25 and idx.signature_count() == 25
        for i, n in g["ids"].items():
            assert len(sigs[i][1]) == n
        assert idx.combined_minhash_size() == g["combined_size"]
        st = idx.stats()
        assert st["n_proteins"] == 25 and st["n_residues"] == 9288


@pytest.mark.parametrize("key,k", [("hp.k16.scaled5", 16), ("hp.k15.scaled5", 15), ("hp.k24.scaled5", 24)])
def test_golden_sig_zip_and_kmers(K, golden_sigs, golden_kmers, key, k):
    prot = K.Proteome.from_fasta(fasta_path("bcl2_first25.fasta.gz"))
    names = prot.names
    h, pid, pos, sk = _gpu_tuples(K, prot, k, "hp", 5)
    by_name = dict(zip(names, sk))
    for g in golden_sigs[key]["signatures"]:
        mins, ab = by_name[g["name"]]
        assert [int(x) for x in g["mins"]] == mins.tolist()
        assert g["abundances"] == ab.tolist()
        assert g["md5sum"] == K.md5_of_mins(mins, k)
        assert int(g["max_hash"]) == K.max_hash(5)
    seqs = [prot.sequence(i) for i in range(prot.n_proteins)]
    mine = set()
    for hv, p, s in zip(h.tolist(), pid.tolist(), pos.tolist()):
        km = seqs[p][s:s + k]
        mine.add((names[p], s, hv if hv < 2**63 else hv - 2**64, km, K.translate(km, "hp")))
    gold = {(r["name"], r["start"], int(r["hashval"]), r["kmer"], r["encoded"]) for r in golden_kmers[key]}
    assert gold == mine


def _ced9_vs_bcl2(K):
    q = K.Proteome.from_fasta(fasta_path("ced9.fasta"))
    t = K.Proteome.from_fasta(fasta_path("bcl2_first25.fasta.gz"))
    idx = K.ProteomeIndex("db", 16, 5, "hp")
    idx.add_proteome(t)
    res = K.search(idx, q, hits=True)
    return idx, q, t, res


def test_golden_manysearch(K, golden_search):
    idx, q, t, res = _ced9_vs_bcl2(K)
    rows = K.manysearch_rows(res, idx, q.names)
    gold = list(csv.DictReader(io.StringIO(golden_search["manysearch_csv"])))  # tests/test_search.py:33-39
    assert len(rows) == len(gold) == 5
    by = {r["match_name"]: r for r in rows}
    for g in gold:
        r = by[g["match_name"]]
        for col, v in r.items():
            if isinstance(v, float):
                assert v == pytest.approx(float(g[col]), rel=SCORE_RTOL, abs=0), col
            else:
                assert str(v) == g[col], col
    idx.close()


def test_golden_stitched(K, golden_search):
    idx, q, t, res = _ced9_vs_bcl2(K)
    qs = [q.sequence(i) for i in range(q.n_proteins)]
    ts = [t.sequence(i) for i in range(t.n_proteins)]
    rows = K.stitch_hits(res, idx, qs, ts, q.names, t.names)
    gold = list(csv.DictReader(io.StringIO(golden_search["stitched_csv"])))  # tests/test_search.py:88-94
    assert len(rows) == len(gold) == 5
    by = {r["match_name"]: r for r in rows}
    for g in gold:
        for col, v in by[g["match_name"]].items():
            assert str(v) == g[col], col
    idx.close()


def test_ambiguous_residues_self_match_and_sourmash_mode(K, O):
    """A query that is a copy of a target record must match it fully, B/Z/J included: the resolution depends on the seed
    and the position in the sequence, not on the record's index.  In "sourmash" mode (what `kmerseek search` does to both
    inputs) nothing is resolved, truncated or rejected: B/Z/J translate to X under dayhoff / hp, an inner '*' stays."""
    rng = np.random.default_rng(21)
    letters = list("ACDEFGHIKLMNPQRSTVWY")
    seqs = []
    for i in range(40):
        s = rng.choice(letters, size=int(rng.integers(60, 200)))
        s[rng.integers(0, len(s), size=6)] = rng.choice(list("BZJ"), size=6)
        seqs.append("".join(s))
    seqs[7] = seqs[7][:50] + "*" + seqs[7][50:]
    seqs[9] = seqs[9].lower()
    names = [f"p{i}" for i in range(len(seqs))]
    for mode in ("kmerseek", "sourmash"):
        for k, moltype in ((7, "protein"), (10, "dayhoff"), (14, "hp")):
            t = K.Proteome.from_sequences(seqs, names, mode=mode)
            q = K.Proteome.from_sequences([seqs[33], seqs[7], seqs[9]], ["a", "b", "c"], mode=mode)  # other record indices
            with K.ProteomeIndex("db", k, 1, moltype) as idx:
                idx.add_proteome(t)
                r = K.search(idx, q, hits=False)
                p = r.pairs
                for qi, ti in ((0, 33), (1, 7), (2, 9)):
                    j = [x for x in range(r.n_pairs) if p["pair_qid"][x] == qi and p["pair_pid"][x] == ti]
                    assert len(j) == 1 and p["containment"][j[0]] == 1.0 and p["jaccard"][j[0]] == 1.0, (mode, moltype, qi)
                # against the oracle on the oracle's own normalisation
                norm = [O.normalize(s, i, 0, mode) for i, s in enumerate(seqs)]
                assert [t.sequence(i) for i in range(len(seqs))] == norm
                res, offs = O.pack(norm)
                qres, qoffs = O.pack([O.normalize(s, 0, 0, mode) for s in (seqs[33], seqs[7], seqs[9])])
                _search_equals_oracle(K, O, idx, res, offs, qres, qoffs, k, moltype, 1)
    assert "*" in K.Proteome.from_sequences(seqs, names, mode="sourmash").sequence(7)[:-1]
    assert K.Proteome.from_sequences(seqs, names).sequence(7).endswith("*") and len(K.Proteome.from_sequences(seqs, names).sequence(7)) == 51
    K.Proteome.from_sequences(["AC1-DE"], ["x"], mode="sourmash")  # nothing is rejected on this path
    with pytest.raises(K.InvalidAminoAcid):
        K.Proteome.from_sequences(["AC1-DE"], ["x"])


def test_stitch_groups_by_match_name_like_the_reference(K, O):
    """stitch_kmers_per_gene groups by match_name only (src/python/kmerseek/search.py:222-240): two queries that hit one
    match end in ONE stitched row, labelled with the query of the smallest query start."""
    rng = np.random.default_rng(3)
    letters = list("ACDEFGHIKLMNPQRSTVWY")
    tseqs = ["".join(rng.choice(letters, size=150)) for _ in range(5)]
    # (the two queries share their offset into t2: with unrelated offsets the reference's own length assertion fails,
    # search.py:87-88, and so does stitch_hits)
    qseqs = [tseqs[2][20:60], tseqs[2][20:75], tseqs[4][10:70]]
    k = 9
    t = K.Proteome.from_sequences(tseqs, [f"t{i}" for i in range(5)])
    q = K.Proteome.from_sequences(qseqs, ["qa", "qb", "qc"])
    with K.ProteomeIndex("db", k, 1, "dayhoff") as idx:
        idx.add_proteome(t)
        res = K.search(idx, q, hits=True)
        rows = K.stitch_hits(res, idx, qseqs, tseqs, q.names, t.names)
    assert sorted(r["match_name"] for r in rows) == ["t2", "t4"]
    h = res.hits
    merged = {}
    for i in range(res.n_hits):
        qi, ti, a, b = int(h["hit_qid"][i]), int(h["hit_pid"][i]), int(h["hit_qpos"][i]), int(h["hit_tpos"][i])
        qk = qseqs[qi][a:a + k]
        merged.setdefault(ti, []).append((a, b, qk, tseqs[ti][b:b + k], O.translate(qk, "dayhoff"), qi))
    for r in rows:
        ti = int(r["match_name"][1:])
        o = O.stitch_pair([x[:5] for x in merged[ti]])
        for col, v in o.items():
            assert r[col] == v, col
        first = sorted(merged[ti], key=lambda x: x[0])[0]
        assert r["query_name"] == q.names[first[5]]
    t2 = [r for r in rows if r["match_name"] == "t2"][0]
    assert t2["query_name"] == "qa" and t2["length"] > 75 - 20  # both queries' k-mers in one row (duplicates concatenated)


def test_raw_sequence_storage_and_signature_count(K):
    """src/rust/index.rs:2713-2844 (raw-sequence storage) and :514-516 / :817-820 (signature_count: the signatures map is
    keyed by the id, equal sketches overwrite)."""
    seq = "ACDEFGHIKLMNPQRSTVWY"
    for store in (True, False):
        with K.ProteomeIndex("db", 5, 1, "protein", store_raw_sequences=store) as idx:
            sig = idx.create_protein_signature(seq, "test_protein")
            assert sig.has_efficient_data() == store
            assert sig.get_raw_sequence() == (seq if store else None)
            idx.store_signatures([sig])
            assert idx.store_raw_sequences() == store and idx.signature_count() == 1
            stored = next(iter(idx.get_signatures().values()))
            assert stored.has_efficient_data() == store and stored.get_raw_sequence() == (seq if store else None)
            assert stored.name == "test_protein" and np.array_equal(stored.mins(), sig.mins())
    # duplicates overwrite: 5 records, two of them copies, one too short to have a sketch ("0" is an id too)
    seqs = [seq, "PLANTANDANIMALGENQMES", seq, "LIVINGALIVEANDWELL", "ACD", "PLANTANDANIMALGENQMES", "AC"]
    with K.ProteomeIndex("db", 5, 1, "protein", store_raw_sequences=True) as idx:
        idx.add_proteome(K.Proteome.from_sequences(seqs, [f"p{i}" for i in range(len(seqs))]))
        idx.finalize()
        assert idx.signature_count() == 4 == len(idx.get_signatures())
        assert idx.stats()["n_distinct_ids"] == 4 and idx.stats()["n_proteins"] == 7
        sigs = idx.get_signatures()
        assert sorted(s.name for s in sigs.values()) == ["p2", "p3", "p5", "p6"]  # the last of equal ids wins
        assert all(s.get_raw_sequence() == seqs[int(s.name[1:])] for s in sigs.values())


def test_invalid_residue_and_moltype_errors(K, golden_rust):
    with K.ProteomeIndex("db", 5, 1, "protein") as idx:
        for e in golden_rust["errors"]:  # src/rust/index.rs:2031-2046
            with pytest.raises(K.InvalidAminoAcid) as ei:
                idx.create_protein_signature(e["sequence"], "test_protein")
            assert e["message"] in str(ei.value)
        for seq in ["PLANTANDANIMALGENBMES", "PLANTANDANIMALGENZMES", "PLANTANDANIMALGENJMES"]:
            assert idx.create_protein_signature(seq, "p").size() == 17  # resolved, not rejected (index.rs:2052-2075)
    with pytest.raises(K.InvalidMoltype):
        K.ProteomeIndex("db", 5, 1, "dna")


# ---- against the oracle on seeded synthetic inputs -----------------------------------------------------
def _edge_proteome(K, seed, n_res=300_000):
    """Synthetic proteome with the awkward cases mixed in: empty and shorter-than-k proteins, a protein much
    longer than a tile, runs of tiny proteins (more boundaries than the kernel's offsets cache), X/U/O/*,
    lower case, low-complexity repeats (duplicate hashes)."""
    from kmerseek_b200 import synth
    rng = np.random.default_rng(seed)
    res, offs = synth.proteome(n_res, seed)
    seqs = [res[int(offs[i]):int(offs[i + 1])].tobytes().decode() for i in range(len(offs) - 1)]
    seqs[3] = ""
    seqs[4] = "AC"
    seqs[5] = seqs[5].lower()
    seqs[6] = seqs[6][:40] + "XUO" + seqs[6][40:80] + "*" + seqs[6][80:]
    seqs[7] = "A" * 700 + "ACDEFGHIKL" * 50
    seqs[8] = "".join(rng.choice(list("ACDEFGHIKLMNPQRSTVWY"), size=9000))
    tiny = ["".join(rng.choice(list("ACDEFGHIKLMNPQRSTVWY"), size=int(n))) for n in rng.integers(0, 6, size=900)]
    seqs = seqs[:20] + tiny + seqs[20:] + ["", "M", ""]
    return K.Proteome.from_sequences(seqs, [f"p{i}" for i in range(len(seqs))]), seqs


SWEEP = [(k, m, 1) for k in (1, 2, 5, 7, 8, 9, 12, 15, 16, 17, 21, 24, 25, 31, 32, 33, 40) for m in ("protein", "dayhoff", "hp")]
SWEEP += [(7, "protein", 10), (16, "dayhoff", 5), (24, "hp", 100), (10, "hp", 2), (5, "protein", 1000)]


@pytest.mark.parametrize("k,moltype,scaled", SWEEP)
def test_sketch_tuples_bit_exact(K, O, k, moltype, scaled):
    prot, _ = _edge_proteome(K, 1234, 120_000)
    h, pid, pos, sk = _gpu_tuples(K, prot, k, moltype, scaled)
    oh, opid, opos = _oracle_tuples(O, prot, k, moltype, scaled)
    assert len(h) == len(oh)
    assert np.array_equal(h, oh) and np.array_equal(pid, opid) and np.array_equal(pos, opos)
    osk = O.protein_sketches(oh, opid, prot.n_proteins)
    assert len(sk) == len(osk)
    for (m, a), (om, oa) in zip(sk, osk):
        assert np.array_equal(m, om) and np.array_equal(a, oa)


@pytest.mark.parametrize("k,moltype,scaled", [(5, "protein", 1), (16, "dayhoff", 1), (24, "hp", 1), (7, "protein", 10),
                                              (12, "hp", 5)])
def test_index_csr_and_search_bit_exact(K, O, k, moltype, scaled):
    from kmerseek_b200 import synth
    prot, seqs = _edge_proteome(K, 99, 400_000)
    res, offs = prot.residues, prot.offsets
    qres, qoffs, _ = synth.queries(res, offs, 64, 7, min_len=max(30, k + 3), max_len=200)
    queries = K.Proteome.from_packed(qres, qoffs)
    with K.ProteomeIndex("db", k, scaled, moltype) as idx:
        idx.add_proteome(prot)
        idx.finalize()
        keys, row_ptr, pid, pos = idx.csr()
        oh, opid, opos = _oracle_tuples(O, prot, k, moltype, scaled)
        okeys, orow, ops, oqs = O.build_index(oh, opid, opos)
        assert np.array_equal(keys, okeys) and np.array_equal(row_ptr, orow)
        assert np.array_equal(pid, ops) and np.array_equal(pos, oqs)
        st = idx.stats()
        assert st["n_tuples"] == len(oh) and st["n_unique_hashes"] == len(okeys)
        osk = O.protein_sketches(oh, opid, prot.n_proteins)
        assert st["n_groups"] == sum(len(m) for m, _ in osk)
        sk = idx.export_sketches()
        for (m, a), (om, oa) in zip(sk, osk):
            assert np.array_equal(m, om) and np.array_equal(a, oa)
        cm, ca = idx.get_combined_minhash()
        ocm, oca = O.combined_sketch(osk)
        assert np.array_equal(cm, ocm) and np.array_equal(ca, oca)

        r = K.search(idx, queries, hits=True)
        qh, qid, qpos = O.sketch_tuples(qres, qoffs, k, moltype, scaled)
        ohits = O.hits(qh, qid, qpos, oh, opid, opos)
        hh = r.hits
        mine = list(zip(hh["hit_qid"].tolist(), hh["hit_pid"].tolist(), hh["hit_hash"].tolist(),
                        hh["hit_qpos"].tolist(), hh["hit_tpos"].tolist()))
        assert mine == ohits  # same rows, same (query, qpos, target, tpos) order
        assert len(mine) > 0

        qsk = O.protein_sketches(qh, qid, queries.n_proteins)
        for (m, a), (om, oa) in zip(r.query_sketches, qsk):
            assert np.array_equal(m, om) and np.array_equal(a, oa)
        orows = O.manysearch(qsk, osk, k, scaled, moltype)
        p = r.pairs
        assert r.n_pairs == len(orows)
        for j, o in enumerate(orows):
            assert (int(p["pair_qid"][j]), int(p["pair_pid"][j])) == (o["qid"], o["pid"])
            assert int(p["intersect_hashes"][j]) == o["intersect_hashes"]
            assert int(p["n_weighted_found"][j]) == o["n_weighted_found"]
            assert int(p["total_weighted_hashes"][j]) == o["total_weighted_hashes"]
            for c in ("containment", "containment_target_in_query", "max_containment", "jaccard",
                      "query_containment_ani", "match_containment_ani", "average_containment_ani",
                      "max_containment_ani", "average_abund", "median_abund", "std_abund",
                      "f_weighted_target_in_query"):
                assert float(p[c][j]) == pytest.approx(o[c], rel=SCORE_RTOL, abs=1e-12), (c, j)


SCORE_NAMES = ("containment", "containment_target_in_query", "max_containment", "jaccard", "query_containment_ani",
               "match_containment_ani", "average_containment_ani", "max_containment_ani", "average_abund", "median_abund",
               "std_abund", "f_weighted_target_in_query")


def _search_equals_oracle(K, O, idx, res, offs, qres, qoffs, k, moltype, scaled, hits=True):
    """Pairs (bit-exact integers, scores within SCORE_RTOL), hit list and query sketches of one search vs the oracle."""
    queries = K.Proteome.from_packed(qres, qoffs)
    r = K.search(idx, queries, hits=hits)
    oh, opid, opos = O.sketch_tuples(res, offs, k, moltype, scaled)
    qh, qid, qpos = O.sketch_tuples(qres, qoffs, k, moltype, scaled)
    osk = O.protein_sketches(oh, opid, len(offs) - 1)
    qsk = O.protein_sketches(qh, qid, len(qoffs) - 1)
    for (m, a), (om, oa) in zip(r.query_sketches, qsk):
        assert np.array_equal(m, om) and np.array_equal(a, oa)
    assert np.array_equal(r.q_sizes, [len(m) for m, _ in qsk])
    orows = O.manysearch(qsk, osk, k, scaled, moltype)
    p = r.pairs
    assert r.n_pairs == len(orows)
    assert np.array_equal(p["pair_qid"], [o["qid"] for o in orows]) and np.array_equal(p["pair_pid"], [o["pid"] for o in orows])
    for c in ("intersect_hashes", "n_weighted_found", "total_weighted_hashes"):
        assert np.array_equal(p[c], [o[c] for o in orows]), c
    for c in SCORE_NAMES:
        np.testing.assert_allclose(p[c], [o[c] for o in orows], rtol=SCORE_RTOL, atol=1e-12, err_msg=c)
    if hits:
        ohits = O.hits(qh, qid, qpos, oh, opid, opos)
        hh = r.hits
        mine = list(zip(hh["hit_qid"].tolist(), hh["hit_pid"].tolist(), hh["hit_hash"].tolist(), hh["hit_qpos"].tolist(),
                        hh["hit_tpos"].tolist()))
        assert mine == ohits
    return r


def test_search_query_size_classes_and_library_path(K, O, monkeypatch):
    """The hand-written query kernel has two instantiations (queries of up to 512 and up to 4096 windows); longer queries
    and KS_SEARCH_LEGACY take the library-sorted path.  All must give the oracle's rows, a batch that mixes the classes
    included, with empty / shorter-than-k queries in between."""
    from kmerseek_b200 import synth
    res, offs = synth.proteome(600_000, 2718)
    rng = np.random.default_rng(5)
    k, moltype = 12, "dayhoff"

    def slices(lengths):
        parts, lens = [], []
        for n in lengths:
            a = int(rng.integers(0, len(res) - n - 1)) if n else 0
            piece = res[a:a + n].copy()
            if n > 20:
                piece[rng.integers(0, n, size=n // 12)] = ord("A")  # substitutions: hits are partial
            parts.append(piece)
            lens.append(n)
        return np.concatenate(parts), np.cumsum([0] + lens).astype(np.uint64)

    with K.ProteomeIndex("db", k, 1, moltype) as idx:
        idx.add_proteome(K.Proteome.from_packed(res, offs))
        idx.finalize()
        for lengths in ([60, 0, 5, 523, 300, 11, 12], [3000, 100, 0, 4107, 700], [200, 9000, 50]):
            qres, qoffs = slices(lengths)
            _search_equals_oracle(K, O, idx, res, offs, qres, qoffs, k, moltype, 1)
    monkeypatch.setenv("KS_SEARCH_LEGACY", "1")
    with K.ProteomeIndex("db", k, 1, moltype) as idx:
        idx.add_proteome(K.Proteome.from_packed(res, offs))
        idx.finalize()
        qres, qoffs = slices([60, 0, 523, 300])
        _search_equals_oracle(K, O, idx, res, offs, qres, qoffs, k, moltype, 1)


def test_search_many_targets_per_query(K, O):
    """A tiny k-mer space (hp k = 8): every query hash has thousands of postings, a query meets every target and its
    (target, abundance) records overflow the shared-memory window many times over (the protein-id windows of the query
    kernel), abundances vary (median / deviation over more than ones), and the batch's pairs overflow the first staging
    buffer (65 536 pairs) so that the retry path runs."""
    from kmerseek_b200 import synth
    res, offs = synth.proteome(300_000, 99)
    qres, qoffs, _ = synth.queries(res, offs, 96, 13, min_len=60, max_len=400)
    with K.ProteomeIndex("db", 8, 1, "hp") as idx:
        idx.add_proteome(K.Proteome.from_packed(res, offs))
        idx.finalize()
        r = _search_equals_oracle(K, O, idx, res, offs, qres, qoffs, 8, "hp", 1, hits=False)
        assert r.n_pairs > 65_536 and float(np.max(r.pairs["std_abund"])) > 0
        r2 = K.search(idx, K.Proteome.from_packed(qres, qoffs), hits=False, query_sketches=False)  # buffers now sized
        assert r2.query_sketches is None and r2.n_pairs == r.n_pairs
        assert np.array_equal(r2.pairs["pair_pid"], r.pairs["pair_pid"]) and np.array_equal(r2.pairs["jaccard"], r.pairs["jaccard"])
    # scaled > 1 and a handful of queries, with hits
    qres, qoffs, _ = synth.queries(res, offs, 6, 14, min_len=60, max_len=200)
    with K.ProteomeIndex("db", 9, 3, "hp") as idx:
        idx.add_proteome(K.Proteome.from_packed(res, offs))
        idx.finalize()
        _search_equals_oracle(K, O, idx, res, offs, qres, qoffs, 9, "hp", 3, hits=True)


def test_empty_and_degenerate_inputs(K, O):
    with K.ProteomeIndex("db", 7, 1, "dayhoff") as idx:
        idx.add_proteome(K.Proteome.from_sequences([], []))
        idx.finalize()
        assert idx.stats()["n_tuples"] == 0 and idx.combined_minhash_size() == 0
    with K.ProteomeIndex("db", 7, 1, "dayhoff") as idx:
        prot = K.Proteome.from_sequences(["", "ACD", "ACDEFG"], ["a", "b", "c"])
        idx.add_proteome(prot)
        idx.finalize()
        assert idx.stats()["n_tuples"] == 0
        r = K.search(idx, K.Proteome.from_sequences(["ACDEFGHIKLMN"], ["q"]))
        assert r.n_pairs == 0 and r.n_hits == 0
    with K.ProteomeIndex("db", 7, 1, "dayhoff") as idx:
        prot = K.Proteome.from_sequences(["ACDEFGHIKLMNPQRSTVWY" * 3], ["a"])
        idx.add_proteome(prot)
        r = K.search(idx, K.Proteome.from_sequences(["", "AC", "WWWWWWWWWWWW"], ["q0", "q1", "q2"]))
        assert r.n_pairs == 0


def test_tile_boundary_sizes(K, O):
    # residue counts exactly at, one below and one above the kernel tile (2048 window starts)
    rng = np.random.default_rng(3)
    for n in (2047, 2048, 2049, 4096, 4096 + 23):
        seq = "".join(rng.choice(list("ACDEFGHIKLMNPQRSTVWY"), size=n))
        prot = K.Proteome.from_sequences([seq[:1000], seq[1000:]], ["a", "b"])
        h, pid, pos, _ = _gpu_tuples(K, prot, 24, "hp", 1)
        oh, opid, opos = _oracle_tuples(O, prot, 24, "hp", 1)
        assert np.array_equal(h, oh) and np.array_equal(pid, opid) and np.array_equal(pos, opos)


def test_batches_append_and_store_signatures(K, O):
    prot, seqs = _edge_proteome(K, 5, 60_000)
    half = len(seqs) // 2
    a = K.Proteome.from_sequences(seqs[:half], [f"p{i}" for i in range(half)])
    b = K.Proteome.from_sequences(seqs[half:], [f"p{i}" for i in range(half, len(seqs))])
    with K.ProteomeIndex("one", 9, 1, "dayhoff") as one, K.ProteomeIndex("two", 9, 1, "dayhoff") as two, \
            K.ProteomeIndex("three", 9, 1, "dayhoff") as three:
        one.add_proteome(prot)
        two.add_proteome(a)
        two.add_proteome(b)
        sigs = three.create_protein_signatures(seqs[:50], [f"p{i}" for i in range(50)])
        three.store_signatures(sigs)
        three.store_signatures(three.create_protein_signatures(seqs[50:], [f"p{i}" for i in range(50, len(seqs))]))
        c1, c2, c3 = one.csr(), two.csr(), three.csr()
        for x, y, z in zip(c1, c2, c3):
            assert np.array_equal(x, y) and np.array_equal(x, z)
        assert one.is_equivalent_to(two) and one.is_equivalent_to(three)


def test_medium_scale_against_oracle(K, O):
    """20 M residues, the C2 alphabet/k: tuples are compared through order-sensitive checksums, the CSR fully."""
    from kmerseek_b200 import synth
    res, offs = synth.proteome(20_000_000, 20260102)
    prot = K.Proteome.from_packed(res, offs)
    with K.ProteomeIndex("db", 24, 1, "hp") as idx:
        idx.add_proteome(prot)
        idx.finalize()
        keys, row_ptr, pid, pos = idx.csr()
        oh, opid, opos = O.sketch_tuples(res, offs, 24, "hp", 1)
        okeys, orow, ops, oqs = O.build_index(oh, opid, opos)
        assert np.array_equal(keys, okeys) and np.array_equal(row_ptr, orow)
        assert np.array_equal(pid, ops) and np.array_equal(pos, oqs)
        assert idx.stats()["build_path"] == 1  # the dense k-mer space path took it (the C2 configuration's path)


def test_bucket_sort_path_with_oversize_buckets(K, O):
    """Enough tuples for the hand-written bucket sort (needs >= 2^12 buckets) plus low-complexity proteins whose
    repeated hashes overflow a shared-memory bucket (library-sort fallback for those ranges)."""
    from kmerseek_b200 import synth
    res, offs = synth.proteome(14_000_000, 4242)
    seqs_extra = ["A" * 30000, "AG" * 9000, "ACDEFGHIKL" * 2500, "M" + "L" * 7000]
    extra = np.frombuffer("".join(seqs_extra).encode(), dtype=np.uint8)
    eoffs = np.cumsum([0] + [len(s) for s in seqs_extra]).astype(np.uint64)
    res2 = np.concatenate([res[: int(offs[1000])], extra, res[int(offs[1000]):]])
    offs2 = np.concatenate([offs[:1001], offs[1000] + eoffs[1:], offs[1001:] + eoffs[-1]])
    prot = K.Proteome.from_packed(res2, offs2)
    for k, moltype, scaled in ((16, "dayhoff", 1), (24, "hp", 1)):
        with K.ProteomeIndex("db", k, scaled, moltype) as idx:
            idx.add_proteome(prot)
            idx.finalize()
            keys, row_ptr, pid, pos = idx.csr()
            oh, opid, opos = O.sketch_tuples(res2, offs2, k, moltype, scaled)
            okeys, orow, ops, oqs = O.build_index(oh, opid, opos)
            assert np.array_equal(keys, okeys) and np.array_equal(row_ptr, orow)
            assert np.array_equal(pid, ops) and np.array_equal(pos, oqs)
            assert int(np.diff(orow).max()) > 4096  # a hash that alone overflows a bucket


def test_bucket_sort_path_scaled(K, O):
    from kmerseek_b200 import synth
    res, offs = synth.proteome(30_000_000, 777)
    prot = K.Proteome.from_packed(res, offs)
    with K.ProteomeIndex("db", 7, 10, "protein") as idx:  # the C4 alphabet / k / scaled
        idx.add_proteome(prot)
        idx.finalize()
        keys, row_ptr, pid, pos = idx.csr()
        oh, opid, opos = O.sketch_tuples(res, offs, 7, "protein", 10)
        okeys, orow, ops, oqs = O.build_index(oh, opid, opos)
        assert np.array_equal(keys, okeys) and np.array_equal(row_ptr, orow)
        assert np.array_equal(pid, ops) and np.array_equal(pos, oqs)


def _csr_equals_oracle(K, O, res, offs, k, moltype, scaled=1, path=None, idx=None):
    """idx: a handle that (res, offs) has been added to; a new one takes them otherwise."""
    if idx is None:
        prot = K.Proteome.from_packed(res, offs)
        with K.ProteomeIndex("db", k, scaled, moltype) as idx:
            idx.add_proteome(prot)
            return _csr_equals_oracle(K, O, res, offs, k, moltype, scaled, path, idx)
    idx.finalize()
    keys, row_ptr, pid, pos = idx.csr()
    oh, opid, opos = O.sketch_tuples(res, offs, k, moltype, scaled)
    okeys, orow, ops, oqs = O.build_index(oh, opid, opos)
    assert np.array_equal(keys, okeys) and np.array_equal(row_ptr, orow), (k, moltype)
    assert np.array_equal(pid, ops) and np.array_equal(pos, oqs), (k, moltype)
    st = idx.stats()
    assert st["n_tuples"] == len(oh) and st["n_unique_hashes"] == len(okeys)
    assert path is None or st["build_path"] == path, (st["build_path"], path)
    sk = idx.export_sketches()
    osk = O.protein_sketches(oh, opid, len(offs) - 1)
    assert len(sk) == len(osk)
    for (m, a), (om, oa) in zip(sk, osk):
        assert np.array_equal(m, om) and np.array_equal(a, oa)
    return st


def test_dense_kmer_space_path(K, O, monkeypatch):
    """hp, 8 <= k <= 24, scaled == 1: the index is built from the ranks of the k-bit patterns (per-handle table, 8-byte
    keys, library sort on the rank bits, no bucket sort).  Forced on for small inputs here; must equal the oracle for
    every k, with proteins shorter than k, and fall back to the general path -- same result -- when a window holds a
    residue of neither class (X, U, O, *) or when a second batch is added."""
    from kmerseek_b200 import synth
    monkeypatch.setenv("KS_DENSE", "1")
    res, offs = synth.proteome(400_000, 606)
    # a few degenerate proteins: empty, shorter than k, exactly k
    extra = [b"", b"ACDEF", b"ACDEFGHIKLMNPQRSTVWYACDE", b"LLLLLLLLLLLLLLLLLLLLLLLLLLLLLLLLLLLLLLLL"]
    eres = np.frombuffer(b"".join(extra), dtype=np.uint8)
    eoffs = np.cumsum([0] + [len(e) for e in extra]).astype(np.uint64)
    res2 = np.concatenate([res, eres])
    offs2 = np.concatenate([offs, offs[-1] + eoffs[1:]])
    for k in (8, 9, 15, 16, 17, 21, 24):
        # (with 2^8 or 2^9 patterns a sort bucket is a single, unevenly frequent pattern: it may overflow and send the
        # batch to the general path, which is what the overflow flag is for)
        _csr_equals_oracle(K, O, res2, offs2, k, "hp", path=1 if k >= 15 else None)
    monkeypatch.setenv("KS_DENSE_SORT", "library")  # the keys sorted by the library instead of the two scatter levels
    for k in (8, 16, 24):
        _csr_equals_oracle(K, O, res2, offs2, k, "hp", path=2)
    monkeypatch.delenv("KS_DENSE_SORT")
    # exceptions: windows with X / * / U / O have no pattern; they are hashed from their bytes and ranked between the
    # patterns.  A few of them, then thousands (with k = 15 / 16 many different exception hashes fall between the same
    # two patterns and share a rank', the case the bucket kernel re-orders by recomputed hash)
    res3 = res2.copy()
    res3[[1000, 5000, 123456]] = [ord("X"), ord("*"), ord("U")]
    _csr_equals_oracle(K, O, res3, offs2, 24, "hp", path=1)
    rng = np.random.default_rng(11)
    res4 = res2.copy()
    res4[rng.integers(0, len(res4), size=3000)] = rng.choice(np.frombuffer(b"XUO*", dtype=np.uint8), size=3000)
    res4[200_000:200_060] = ord("X")  # a run of X: the same exception k-mer many times
    for k in (15, 16, 24):
        _csr_equals_oracle(K, O, res4, offs2, k, "hp", path=1)
    monkeypatch.setenv("KS_DENSE_SORT", "library")  # no exception handling with the library's key sort: general path
    _csr_equals_oracle(K, O, res4, offs2, 16, "hp", path=0)
    monkeypatch.delenv("KS_DENSE_SORT")
    # two batches: the first is deferred, the second forces it through the general sketch
    half = len(offs) // 2
    a = K.Proteome.from_packed(res[: int(offs[half])], offs[: half + 1])
    b = K.Proteome.from_packed(res[int(offs[half]):], offs[half:] - offs[half])
    with K.ProteomeIndex("db", 16, 1, "hp") as idx:
        idx.add_proteome(a)
        idx.add_proteome(b)
        idx.finalize()
        keys, row_ptr, pid, pos = idx.csr()
        oh, opid, opos = O.sketch_tuples(res, offs, 16, "hp", 1)
        okeys, orow, ops, oqs = O.build_index(oh, opid, opos)
        assert np.array_equal(keys, okeys) and np.array_equal(row_ptr, orow)
        assert np.array_equal(pid, ops) and np.array_equal(pos, oqs)
    # search on a densely built index
    qres, qoffs, _ = synth.queries(res, offs, 64, 5)
    prot, queries = K.Proteome.from_packed(res, offs), K.Proteome.from_packed(qres, qoffs)
    with K.ProteomeIndex("db", 16, 1, "hp") as idx:
        idx.add_proteome(prot)
        r = K.search(idx, queries, hits=True)
        qh, qid, qpos = O.sketch_tuples(qres, qoffs, 16, "hp", 1)
        oh, opid, opos = O.sketch_tuples(res, offs, 16, "hp", 1)
        ohits = O.hits(qh, qid, qpos, oh, opid, opos)
        h = r.hits
        mine = list(zip(h["hit_qid"].tolist(), h["hit_pid"].tolist(), h["hit_hash"].tolist(), h["hit_qpos"].tolist(),
                        h["hit_tpos"].tolist()))
        assert mine == ohits and len(mine) > 0
        rows = O.manysearch(O.protein_sketches(qh, qid, len(qoffs) - 1), O.protein_sketches(oh, opid, len(offs) - 1), 16, 1, "hp")
        assert len(rows) == r.n_pairs
        for j, row in enumerate(rows):
            assert (int(r.pairs["pair_qid"][j]), int(r.pairs["pair_pid"][j])) == (row["qid"], row["pid"])
            assert int(r.pairs["intersect_hashes"][j]) == row["intersect_hashes"]
            assert float(r.pairs["containment"][j]) == pytest.approx(row["containment"], rel=SCORE_RTOL)
            assert float(r.pairs["median_abund"][j]) == pytest.approx(row["median_abund"], rel=SCORE_RTOL)


def test_dense_path_two_scatter_levels(K, O):
    """14 M residues of hp k=24 / k=16 take the dense path on their own (the k-mer space is covered) with both scatter
    levels of the key sort (more than 2^8 x 3072 keys); a proteome with a heavily repeated k-mer overflows a sort bucket
    and must come out of the general path with the same index."""
    from kmerseek_b200 import synth
    res, offs = synth.proteome(14_000_000, 515)
    for k in (24, 16):
        _csr_equals_oracle(K, O, res, offs, k, "hp", path=1)
    rep = np.frombuffer(("AL" * 40_000).encode(), dtype=np.uint8)  # two patterns, ~40 000 windows each
    res2 = np.concatenate([res, rep])
    offs2 = np.concatenate([offs, [offs[-1] + len(rep)]]).astype(np.uint64)
    _csr_equals_oracle(K, O, res2, offs2, 24, "hp", path=0)


def test_unstable_partition_of_the_general_path(K, O, monkeypatch):
    """Hashes that rarely repeat, scaled == 1, one batch: the sketch kernel scatters the tuples straight into the
    first-level regions of an unstable partition, a second level follows, and the bin kernel orders equal hashes by
    their loc (build_path 3).  Checked on a proteome with thousands of duplicated proteins (equal hashes at different
    positions, arriving in arbitrary order) at a size that needs both scatter levels, against the stable path and the
    oracle; a k-mer repeated tens of thousands of times overflows a region and must come out of the stable path."""
    from kmerseek_b200 import synth
    res, offs = synth.proteome(14_000_000, 808)
    # duplicate 3 000 proteins twice each (paralogs): every k-mer of theirs occurs three times
    lens = np.diff(offs.astype(np.int64))
    pick = np.arange(1000, 4000)
    dup = np.concatenate([res[int(offs[p]):int(offs[p + 1])] for p in pick])
    res2 = np.concatenate([res, dup, dup])
    offs2 = np.concatenate([offs, offs[-1] + np.cumsum(np.tile(lens[pick], 2)).astype(np.uint64)])
    for k, moltype in ((16, "dayhoff"), (7, "protein")):
        st = _csr_equals_oracle(K, O, res2, offs2, k, moltype, path=3)
        assert st["n_unique_hashes"] < st["n_tuples"]
    # scaled > 1: the look-back sketch path scatters too (kept windows per protein counted by the sketch kernel)
    for k, moltype, scaled in ((7, "protein", 10), (16, "dayhoff", 5)):
        _csr_equals_oracle(K, O, res2, offs2, k, moltype, scaled=scaled, path=3)
    rep = np.frombuffer(("ACDEFGHIKLMNPQRSTVWY" * 3000).encode(), dtype=np.uint8)  # 20 k-mers, 3 000 times each
    res3 = np.concatenate([res, rep])
    offs3 = np.concatenate([offs, [offs[-1] + len(rep)]]).astype(np.uint64)
    _csr_equals_oracle(K, O, res3, offs3, 16, "dayhoff", path=0)
    monkeypatch.setenv("KS_SCATTER", "0")
    _csr_equals_oracle(K, O, res2, offs2, 16, "dayhoff", path=0)


def test_general_sketch_path_at_scaled_1(K, O, monkeypatch):
    """scaled == 1 normally takes the chain-free exact path; the look-back path must give the same tuples
    (it is what a batch is redone on if a hash of exactly 0 ever shows up)."""
    monkeypatch.setenv("KS_SKETCH_GENERAL", "1")
    prot, _ = _edge_proteome(K, 1234, 120_000)
    for k, moltype in ((24, "hp"), (16, "dayhoff"), (5, "protein")):
        h, pid, pos, _ = _gpu_tuples(K, prot, k, moltype, 1)
        oh, opid, opos = _oracle_tuples(O, prot, k, moltype, 1)
        assert np.array_equal(h, oh) and np.array_equal(pid, opid) and np.array_equal(pos, opos)


@pytest.mark.parametrize("variant", ["rep", "bs", "bn"])
def test_bucket_sort_both_variants(K, O, monkeypatch, variant):
    """The bucket sort picks the bin kernel (hashes rarely repeat) or the two-pass stable kernel (small k-mer space,
    repeat-heavy); every variant must give the same index on both kinds of data."""
    from kmerseek_b200 import synth
    monkeypatch.setenv("KS_LS_VARIANT", variant)
    monkeypatch.setenv("KS_DENSE", "0")    # the stable partition + bucket sort of the general path is what is under test
    monkeypatch.setenv("KS_SCATTER", "0")
    res, offs = synth.proteome(14_000_000, 2024)
    prot = K.Proteome.from_packed(res, offs)
    for k, moltype in ((24, "hp"), (16, "dayhoff")):
        with K.ProteomeIndex("db", k, 1, moltype) as idx:
            idx.add_proteome(prot)
            idx.finalize()
            keys, row_ptr, pid, pos = idx.csr()
            oh, opid, opos = O.sketch_tuples(res, offs, k, moltype, 1)
            okeys, orow, ops, oqs = O.build_index(oh, opid, opos)
            assert np.array_equal(keys, okeys) and np.array_equal(row_ptr, orow)
            assert np.array_equal(pid, ops) and np.array_equal(pos, oqs)


def test_cli_search_and_index_against_goldens(K, golden_search, golden_sigs, tmp_path):
    """`python -m kmerseek_b200 search|index` end to end (tests/test_search.py:9-60,63-139, src/rust/tests/test_cli.rs)."""
    import json
    import subprocess
    import sys
    import zipfile
    import gzip
    from conftest import ROOT
    env = dict(os.environ, PYTHONPATH=ROOT)
    base = [sys.executable, "-m", "kmerseek_b200"]
    r = subprocess.run(base + ["search", "--ksize", "16", fasta_path("ced9.fasta"), fasta_path("bcl2_first25.fasta.gz")],
                       capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr
    got = {x["match_name"]: x for x in csv.DictReader(io.StringIO(r.stdout))}
    gold = list(csv.DictReader(io.StringIO(golden_search["manysearch_csv"])))
    assert len(got) == len(gold) == 5
    for g in gold:
        for c, v in g.items():
            try:
                assert float(got[g["match_name"]][c]) == pytest.approx(float(v), rel=SCORE_RTOL), c
            except ValueError:
                assert got[g["match_name"]][c] == v, c
    r = subprocess.run(base + ["search", "--extract-kmers", "--ksize", "16", fasta_path("ced9.fasta"),
                               fasta_path("bcl2_first25.fasta.gz")], capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr
    key = lambda x: x["match_name"]
    assert sorted(csv.DictReader(io.StringIO(r.stdout)), key=key) == \
        sorted(csv.DictReader(io.StringIO(golden_search["stitched_csv"])), key=key)
    assert "query: MSIGESIDGKINDWEEPGIVGVVVCGRMMFSLK (59-92)" in r.stderr  # tests/test_search.py:112-117
    out = tmp_path / "db"
    r = subprocess.run(base + ["index", "--input", fasta_path("bcl2_first25.fasta.gz"), "--output", str(out), "--ksize", "16",
                               "--scaled", "5", "--encoding", "hp"], capture_output=True, text=True, env=env)
    assert r.returncode == 0 and "Indexing completed successfully!" in r.stdout and out.exists()  # test_cli.rs:46
    z = zipfile.ZipFile(out / "bcl2_first25.fasta.gz.hp.k16.scaled5.sig.zip")
    for s in golden_sigs["hp.k16.scaled5"]["signatures"]:
        sk = json.loads(gzip.decompress(z.read(f"signatures/{s['md5sum']}.sig.gz")))[0]["signatures"][0]
        assert [str(x) for x in sk["mins"]] == s["mins"] and sk["abundances"] == s["abundances"]
    r = subprocess.run(base + ["index", "--input", str(tmp_path / "nope.fasta")], capture_output=True, text=True, env=env)
    assert r.returncode != 0 and "No such file or directory" in r.stderr  # test_cli.rs:125
    r = subprocess.run(base + ["index"], capture_output=True, text=True, env=env)
    assert r.returncode != 0 and "required" in r.stderr  # test_cli.rs:135


@pytest.mark.parametrize("k,moltype,scaled", [(16, "dayhoff", 1), (7, "protein", 10)])
def test_pipelined_upload_matches_single_copy(K, monkeypatch, k, moltype, scaled):
    """Batches above 64 MB stream the residues in chunks while earlier tiles are hashed (ks_index_add_proteome), on
    the exact path (scaled == 1) and on the look-back path (scaled > 1, tiles taken by ticket across the chunk
    launches); the index must be identical to the one built from a single copy + single launch."""
    from kmerseek_b200 import synth
    res, offs = synth.proteome(80_000_000, 31337)
    prot = K.Proteome.from_packed(res, offs)
    lens = np.diff(offs.astype(np.int64))
    out = []
    for no_pipe in (False, True):
        if no_pipe:
            monkeypatch.setenv("KS_NO_PIPELINE", "1")
        with K.ProteomeIndex("db", k, scaled, moltype) as idx:
            idx.add_proteome(prot)
            idx.finalize()
            st = idx.stats()
            if scaled == 1:
                assert st["n_tuples"] == int(np.maximum(lens - (k - 1), 0).sum())
            else:
                assert 0.09 < st["n_tuples"] / float(np.maximum(lens - (k - 1), 0).sum()) < 0.11
            out.append(idx.csr())
    for a, b in zip(*out):
        assert np.array_equal(a, b)


def test_unpackable_residues_take_the_byte_path(K, O, monkeypatch):
    """Index builds upload 5-bit packed residues; a proteome handed over with bytes outside A-Z and '*'
    (ks_proteome_from_packed does not validate) cannot be packed and must go through the plain byte path, on every
    route of the sketch kernels: the ordered sketch, the dense path with its own key sort (every hp window of these bytes
    has a residue of neither class: exception keys) and with the library's (no exception handling: general path), and,
    on a batch large enough for the unstable partition, the sketch kernel's scatter at scaled 1 and at scaled > 1.  The
    large batch has a run of 1 000 proteins of 0-3 residues, more than the sketch kernel's offsets cache holds for one
    tile, so that kept windows are counted per protein both in shared memory and in global memory."""
    rng = np.random.default_rng(8)
    alphabet = np.frombuffer(b"ACDEFGHIKLMNPQRSTVWYacdxyz@#1", dtype=np.uint8)
    res = rng.choice(alphabet, size=50_000)
    offs = np.array([0, 10_000, 10_000, 35_000, 50_000], dtype=np.uint64)
    lens = np.concatenate([np.full(100, 3000), rng.integers(0, 4, size=1000), np.full(166, 3000)])
    big_offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    big_res = rng.choice(alphabet, size=int(big_offs[-1]))
    # (residues, offsets, k, moltype, scaled, KS_DENSE_SORT, build_path): 0 general (ordered sketch), 1 dense with the
    # hand-written key sort, 3 general with the unstable partition
    cases = [(res, offs, 7, "protein", 1, None, 0), (res, offs, 12, "hp", 1, None, 1), (res, offs, 12, "hp", 1, "library", 0),
             (big_res, big_offs, 7, "protein", 1, None, 3), (big_res, big_offs, 7, "protein", 10, None, 3)]
    for r, o, k, moltype, scaled, dense_sort, path in cases:
        if dense_sort:
            monkeypatch.setenv("KS_DENSE_SORT", dense_sort)
        else:
            monkeypatch.delenv("KS_DENSE_SORT", raising=False)
        _csr_equals_oracle(K, O, r, o, k, moltype, scaled=scaled, path=path)


def test_golden_zstd_fasta(K, golden_rust):
    g = golden_rust["index_tests"]["test_process_fasta_zstd_moltype_protein"]  # src/rust/index.rs:1734-1789
    with K.ProteomeIndex("db", g["ksize"], g["scaled"], g["moltype"]) as idx:
        idx.process_fasta(fasta_path("test_compression.fasta.zst"), 0, 1000)
        sigs = idx.get_signatures()
        assert len(sigs) == g["n_signatures"] == 2
        for i, n in g["ids"].items():
            assert len(sigs[i][1]) == n
        assert idx.combined_minhash_size() == g["combined_size"] == 24
