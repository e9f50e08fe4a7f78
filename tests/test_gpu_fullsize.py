"""BASELINE.json's full-size configurations on one B200, checked through size-independent properties (the oracle
takes minutes at these sizes): the sort is a permutation of the sketch output, rows are ordered, counts add up, and
planted queries find the protein they were cut from.  C2: 570 k proteins / 200 M residues, hp k=24 scaled=1 (index
build); C3 on one GPU: 10 000 planted domains against the same proteome, dayhoff k=16.
And against the oracle itself on the subsamples BASELINE.md section 4 names: C2 on a 10 M-residue prefix, C3 with 1 000
queries against a 10 M-residue prefix (hit lists bit-exact, scores within 1e-6), C4 on a 50 M-residue prefix."""
import re

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def K():
    import kmerseek_b200
    return kmerseek_b200


@pytest.fixture(scope="module")
def proteome():
    from kmerseek_b200 import synth
    return synth.proteome(200_000_000, 20260102)


def _check_index(K, res, offs, k, moltype, expect_max_unique=None):
    prot = K.Proteome.from_packed(res, offs)
    lens = np.diff(offs.astype(np.int64))
    windows = np.maximum(lens - (k - 1), 0)
    with K.ProteomeIndex("full", k, 1, moltype) as idx:
        idx.add_proteome(prot)
        idx.finalize()
        st = idx.stats()
        n = int(windows.sum())
        assert st["n_tuples"] == n  # scaled == 1: every complete window is kept
        keys, row_ptr, pid, pos = idx.csr()
        U = len(keys)
        assert U == st["n_unique_hashes"] and (expect_max_unique is None or U <= expect_max_unique)
        assert np.all(keys[1:] > keys[:-1])                      # combined sketch: strictly increasing
        assert row_ptr[0] == 0 and row_ptr[-1] == n and np.all(row_ptr[1:] > row_ptr[:-1])  # no empty row
        # the postings are a permutation of all windows: every (protein, position) exactly once ...
        g = offs[:-1].astype(np.int64)[pid] + pos.astype(np.int64)   # global residue index of the window start
        assert np.all(pos.astype(np.int64) < windows[pid])
        seen = np.zeros(len(res), dtype=np.uint8)
        seen[g] = 1
        assert int(seen.sum()) == n
        # ... and inside a row they are ordered by (protein, position)
        loc = (pid.astype(np.uint64) << np.uint64(32)) | pos.astype(np.uint64)
        inner = np.ones(n, dtype=bool)
        inner[row_ptr[:-1].astype(np.int64)] = False               # first posting of every row
        assert np.all(loc[1:][inner[1:]] > loc[:-1][inner[1:]])
        # per-protein sketch sizes: distinct hashes per protein add up to the (hash, protein) groups
        grp_head = ~inner
        grp_head[1:] |= pid[1:] != pid[:-1]
        assert int(grp_head.sum()) == st["n_groups"]
        return st, (keys, row_ptr, pid, pos)


def test_c2_index_build_properties(K, proteome, monkeypatch, capfd):
    """... and the keys against the oracle on a seeded sample of postings: C2's dense keys need 16 + 10 + 20 + 19 = 65 bits
    with the parity bit, so they are built without it (code = prefix << 9 | rank in the prefix group, all 64 bits)."""
    from oracle import oracle as O
    res, offs = proteome
    k = 24
    assert (len(offs) - 2).bit_length() == 20 and int(np.diff(offs.astype(np.int64)).max()).bit_length() == 19
    monkeypatch.setenv("KS_TIMING", "1")  # (read when the handle is created)
    capfd.readouterr()
    st, (keys, row_ptr, pid, pos) = _check_index(K, res, offs, k, "hp", expect_max_unique=1 << 24)
    err = capfd.readouterr().err
    begin = re.search(r"^\[ks\] dense begin: state 1 rb (\d+)$", err, re.M)
    fin = re.search(r"^\[ks\] dense finalize: .* unhandled 0 .* rb (\d+)$", err, re.M)
    assert begin and fin and (int(begin.group(1)), int(fin.group(1))) == (10, 9), err  # no parity bit
    assert st["build_path"] == 1
    # the key of a posting's row is the hash of the posting's window: the sampled windows, one per protein, to the oracle
    j = np.random.default_rng(20260109).integers(0, len(pid), size=4096)
    row = np.searchsorted(row_ptr, j, "right") - 1
    start = offs[:-1].astype(np.int64)[pid[j]] + pos[j].astype(np.int64)
    wres = res[start[:, None] + np.arange(k)].ravel()
    woffs = np.arange(0, k * len(j) + 1, k, dtype=np.uint64)
    oh, opid, opos = O.sketch_tuples(wres, woffs, k, "hp", 1)
    assert np.array_equal(opid, np.arange(len(j))) and not opos.any()
    assert np.array_equal(keys[row], oh)


def test_c3_planted_queries_find_their_source(K, proteome):
    from kmerseek_b200 import synth
    res, offs = proteome
    k, moltype = 16, "dayhoff"
    prot = K.Proteome.from_packed(res, offs)
    qres, qoffs, src = synth.queries(res, offs, 10_000, 79)
    queries = K.Proteome.from_packed(qres, qoffs)
    with K.ProteomeIndex("full", k, 1, moltype) as idx:
        idx.add_proteome(prot)
        idx.finalize()
        r = K.search(idx, queries, hits=True)
        p, h = r.pairs, r.hits
        # ordered by (query, target); every pair has a positive overlap that fits both sketches
        key = (p["pair_qid"].astype(np.uint64) << np.uint64(32)) | p["pair_pid"].astype(np.uint64)
        assert np.all(key[1:] > key[:-1])
        assert np.all(p["intersect_hashes"] > 0)
        assert np.all(p["intersect_hashes"] <= p["q_size"]) and np.all(p["intersect_hashes"] <= p["t_size"])
        np.testing.assert_allclose(p["containment"], p["intersect_hashes"] / p["q_size"], rtol=1e-12)
        np.testing.assert_allclose(p["jaccard"], p["intersect_hashes"] /
                                   (p["q_size"].astype(np.float64) + p["t_size"] - p["intersect_hashes"]), rtol=1e-12)
        # a query with an unmutated 16-mer must hit the protein it was cut from; with 10 % substitutions and
        # 50-300 residues nearly all have one (the few that do not may legitimately have no pair)
        found = set(zip(p["pair_qid"].tolist(), p["pair_pid"].tolist()))
        n_found = sum((q, int(s)) in found for q, s in enumerate(src))
        assert n_found >= 0.9 * len(src)
        # hit list: ordered by (query, qpos, target, tpos); every hit belongs to a scored pair; hits per pair >= overlap
        hk1 = (h["hit_qid"].astype(np.uint64) << np.uint64(32)) | h["hit_qpos"].astype(np.uint64)
        hk2 = (h["hit_pid"].astype(np.uint64) << np.uint64(32)) | h["hit_tpos"].astype(np.uint64)
        assert np.all((hk1[1:] > hk1[:-1]) | ((hk1[1:] == hk1[:-1]) & (hk2[1:] > hk2[:-1])))
        hp = np.unique((h["hit_qid"].astype(np.uint64) << np.uint64(32)) | h["hit_pid"].astype(np.uint64))
        assert np.array_equal(hp, key)
        assert len(h["hit_qid"]) >= int(p["intersect_hashes"].sum())
        # a hit is a real shared window: same translated 16-mer in query and target
        from kmerseek_b200.index import translate
        rng = np.random.default_rng(5)
        for i in rng.integers(0, len(h["hit_qid"]), size=200):
            q, t = int(h["hit_qid"][i]), int(h["hit_pid"][i])
            a, b = int(qoffs[q]) + int(h["hit_qpos"][i]), int(offs[t]) + int(h["hit_tpos"][i])
            qs, ts = qres[a:a + k].tobytes().decode(), res[b:b + k].tobytes().decode()
            assert translate(qs, moltype) == translate(ts, moltype)


SCORES = ("containment", "containment_target_in_query", "max_containment", "jaccard", "query_containment_ani",
          "match_containment_ani", "average_containment_ani", "max_containment_ani", "average_abund", "median_abund",
          "std_abund", "f_weighted_target_in_query")


def _index_equals_oracle(K, res, offs, k, moltype, scaled, path=None):
    from oracle import oracle as O
    with K.ProteomeIndex("prefix", k, scaled, moltype) as idx:
        idx.add_proteome(K.Proteome.from_packed(res, offs))
        idx.finalize()
        keys, row_ptr, pid, pos = idx.csr()
        st = idx.stats()
    oh, opid, opos = O.sketch_tuples(res, offs, k, moltype, scaled)
    okeys, orow, ops, oqs = O.build_index(oh, opid, opos)
    assert np.array_equal(keys, okeys) and np.array_equal(row_ptr, orow)
    assert np.array_equal(pid, ops) and np.array_equal(pos, oqs)
    assert path is None or st["build_path"] in path, st["build_path"]
    return oh, opid, opos


def _prefix(res, offs, n_res):
    p = int(np.searchsorted(offs, n_res))
    return res[:int(offs[p])], offs[:p + 1]


def test_c2_prefix_equals_oracle(K, proteome):
    """BASELINE.md section 4, C2: equality vs the CPU oracle on a 10 M-residue prefix (dense k-mer space path)."""
    res, offs = _prefix(*proteome, 10_000_000)
    _index_equals_oracle(K, res, offs, 24, "hp", 1, path=(1,))


def test_c3_subsample_equals_oracle(K, proteome):
    """BASELINE.md section 4, C3: 1 000 planted queries against a 10 M-residue prefix, dayhoff k=16 -- pairs and hit lists
    bit-exact, scores within 1e-6 relative, against the oracle (indexed restatement of manysearch)."""
    from kmerseek_b200 import synth
    from oracle import oracle as O
    res, offs = _prefix(*proteome, 10_000_000)
    k, moltype = 16, "dayhoff"
    qres, qoffs, _ = synth.queries(res, offs, 1000, 79)
    with K.ProteomeIndex("c3", k, 1, moltype) as idx:
        idx.add_proteome(K.Proteome.from_packed(res, offs))
        idx.finalize()
        r = K.search(idx, K.Proteome.from_packed(qres, qoffs), hits=True)
        p, h = r.pairs, r.hits
        oh, opid, opos = O.sketch_tuples(res, offs, k, moltype, 1)
        qh, qid, qpos = O.sketch_tuples(qres, qoffs, k, moltype, 1)
        qsk = O.protein_sketches(qh, qid, len(qoffs) - 1)
        for (m, a), (om, oa) in zip(r.query_sketches, qsk):
            assert np.array_equal(m, om) and np.array_equal(a, oa)
        rows = O.manysearch_indexed(qsk, oh, opid, k, 1, moltype)
        assert r.n_pairs == len(rows) > 900
        assert np.array_equal(p["pair_qid"], [x["qid"] for x in rows]) and np.array_equal(p["pair_pid"], [x["pid"] for x in rows])
        for c in ("intersect_hashes", "n_weighted_found", "total_weighted_hashes"):
            assert np.array_equal(p[c], [x[c] for x in rows]), c
        for c in SCORES:
            np.testing.assert_allclose(p[c], [x[c] for x in rows], rtol=1e-6, atol=0, err_msg=c)
        ohits = O.hits(qh, qid, qpos, oh, opid, opos)
        mine = list(zip(h["hit_qid"].tolist(), h["hit_pid"].tolist(), h["hit_hash"].tolist(), h["hit_qpos"].tolist(),
                        h["hit_tpos"].tolist()))
        assert mine == ohits and len(mine) > 10_000


def test_c4_prefix_equals_oracle(K):
    """BASELINE.md section 4, C4 (protein k=7 scaled=10): equality vs the oracle on a 50 M-residue prefix."""
    from kmerseek_b200 import synth
    res, offs = synth.proteome(50_000_000, 20260104)
    _index_equals_oracle(K, res, offs, 7, "protein", 10)
