"""ks_index_append_proteome / ks_index_append_tuples: a finalized index extended by a batch must equal the oracle's index
of the concatenation, and a second handle's add(A) + add(B) + finalize byte for byte, on every build route of the old
index and of the batch, in both layouts of the old index.  Each case reads the handle's KS_TIMING lines to check the route
and layout it targets.  Needs a GPU: run with -m gpu."""
import ctypes as C
import re

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

KS_ERR_VALIDATION, KS_ERR_NOT_FINALIZED, KS_ERR_CAPACITY = 9, 10, 104
SCORE_RTOL = 1e-6
SCORE_NAMES = ("containment", "containment_target_in_query", "max_containment", "jaccard", "query_containment_ani",
               "match_containment_ani", "average_containment_ani", "max_containment_ani", "average_abund", "median_abund",
               "std_abund", "f_weighted_target_in_query")

# route -> (k, moltype, scaled, environment, build_path of one add) as in test_gpu_handle_state, plus the dense route with
# the library's key sort, whose index has the compact layout
ROUTES = {
    "dense": (16, "hp", 1, {"KS_DENSE": "1"}, 1),
    "scatter": (16, "dayhoff", 1, {}, 3),
    "ordered": (16, "dayhoff", 1, {"KS_SCATTER": "0"}, 0),
    "scatter_scaled": (7, "protein", 10, {}, 3),
    "ordered_repeats": (24, "hp", 1, {"KS_DENSE": "0"}, 0),
    "dense_library": (16, "hp", 1, {"KS_DENSE": "1", "KS_DENSE_SORT": "library"}, 2),
}
APPEND = re.compile(r"\[ks\] append: batch_path (\d+) A_layout (\w+) B_layout (\w+) U_A (\d+) U_B (\d+) matched (\d+) "
                    r"n_C (\d+)")


@pytest.fixture(scope="module")
def K():
    import kmerseek_b200
    return kmerseek_b200


@pytest.fixture(scope="module")
def O():
    from oracle import oracle
    return oracle


def _short_proteins(n, k, seed):
    """n proteins, each shorter than k: no window, no key."""
    rng = np.random.default_rng(seed)
    lens = rng.integers(1, k, size=n)
    offs = np.zeros(n + 1, np.uint64)
    np.cumsum(lens, out=offs[1:])
    from kmerseek_b200 import synth
    return synth.residues_iid(int(offs[-1]), rng), offs


class Data:
    """Proteomes as (residues, offsets) and handles; the oracle's tuples and indexes of concatenations per configuration."""

    def __init__(self, K, O):
        self.K, self.O = K, O
        self.raw, self.prot, self.cache, self.cfg = {}, {}, {}, None

    def put(self, name, res, offs):
        self.raw[name] = (res, offs)
        self.prot[name] = self.K.Proteome.from_packed(res, offs)

    def add(self, name, n_residues, seed):
        from kmerseek_b200 import synth
        self.put(name, *synth.proteome(n_residues, seed))

    def concat(self, names):
        res = np.concatenate([self.raw[n][0] for n in names]) if names else np.zeros(0, np.uint8)
        offs, base = [np.zeros(1, np.uint64)], 0
        for n in names:
            offs.append(self.raw[n][1][1:] + np.uint64(base))
            base += len(self.raw[n][0])
        return res, np.concatenate(offs)

    def n_proteins(self, names):
        return sum(len(self.raw[n][1]) - 1 for n in names)

    def _key(self, cfg):
        if tuple(cfg[:3]) != self.cfg:
            self.cache, self.cfg = {}, tuple(cfg[:3])

    def tuples(self, names, cfg):
        self._key(cfg)
        if ("t", names) not in self.cache:
            k, moltype, scaled = cfg[:3]
            self.cache[("t", names)] = self.O.sketch_tuples(*self.concat(names), k, moltype, scaled)
        return self.cache[("t", names)]

    def index(self, names, cfg):
        t = self.tuples(names, cfg)
        if ("i", names) not in self.cache:
            self.cache[("i", names)] = self.O.build_index(*t)
        return self.cache[("i", names)]


@pytest.fixture(scope="module")
def small(K, O):
    d = Data(K, O)
    d.add("A", 2_000_000, 4101)
    d.add("A14", 14_000_000, 4104)  # the repeat-heavy route's old index
    d.add("B", 300_000, 4102)
    d.add("C", 2_000_000, 4103)
    d.put("short", *_short_proteins(64, 16, 4105))
    d.put("one", *_one_protein(4106))
    d.put("empty", np.zeros(0, np.uint8), np.zeros(1, np.uint64))
    return d


def _one_protein(seed):
    from kmerseek_b200 import synth
    res, _ = synth.proteome(2_000, seed)
    return res[:700].copy(), np.array([0, 700], np.uint64)


def _handle(K, monkeypatch, cfg):
    k, moltype, scaled, env, _ = cfg
    for name in ("KS_DENSE", "KS_SCATTER", "KS_NO_PIPELINE", "KS_SKETCH_GENERAL", "KS_DENSE_SORT", "KS_APPEND_FAIL"):
        monkeypatch.delenv(name, raising=False)
    monkeypatch.setenv("KS_TIMING", "1")
    for name, value in env.items():
        monkeypatch.setenv(name, value)  # read once, when the handle is created
    return K.ProteomeIndex("db", k, scaled, moltype)


def _lib():
    from kmerseek_b200 import _ffi
    return _ffi.lib()


def _ok(status):
    from kmerseek_b200.errors import check
    check(status)


def _append_line(capfd):
    lines = APPEND.findall(capfd.readouterr().err)
    assert len(lines) == 1, lines
    p, a, b, ua, ub, m, n = lines[0]
    return {"batch_path": int(p), "A_layout": a, "B_layout": b, "U_A": int(ua), "U_B": int(ub), "matched": int(m),
            "n_C": int(n)}


def _equals_oracle(d, idx, names, cfg, path=4):
    """CSR, per-protein sketches, signature_count and stats against the oracle of the concatenation of `names`."""
    O = d.O
    keys, row_ptr, pid, pos = idx.csr()
    okeys, orow, opid, opos = d.index(names, cfg)
    assert np.array_equal(keys, okeys) and np.array_equal(row_ptr, orow), names
    assert np.array_equal(pid, opid) and np.array_equal(pos, opos), names
    P = d.n_proteins(names)
    oh, otp, _ = d.tuples(names, cfg)
    osk = O.protein_sketches(oh, otp, P)
    sk = idx.export_sketches()
    assert len(sk) == len(osk) == P
    for (m, a), (om, oa) in zip(sk, osk):
        assert np.array_equal(m, om) and np.array_equal(a, oa)
    assert idx.signature_count() == len({O.signature_id(m) for m, _ in osk})
    st = idx.stats()
    assert st["finalized"] == 1 and st["n_proteins"] == P and st["n_tuples"] == len(opid)
    assert st["n_unique_hashes"] == len(okeys) and st["n_groups"] == sum(len(m) for m, _ in osk)
    assert path is None or st["build_path"] == path, (st["build_path"], path)
    return st


def _two_add_equal(K, monkeypatch, cfg, idx, prots):
    """The appended index against a second handle's add(...) + finalize: CSR and export byte for byte."""
    with _handle(K, monkeypatch, cfg) as ref:
        for p in prots:
            ref.add_proteome(p)
        ref.finalize()
        for x, y in zip(idx.csr(), ref.csr()):
            assert np.array_equal(x, y)
        a, b = idx.export_sketches(), ref.export_sketches()
        assert len(a) == len(b)
        for (m, ab), (rm, rab) in zip(a, b):
            assert np.array_equal(m, rm) and np.array_equal(ab, rab)


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


# ---- 1 + 2: routes x layouts, and the same as the multi-add build -----------------------------------------------------
@pytest.mark.parametrize("route", list(ROUTES))
def test_append_equals_oracle_and_two_adds(K, small, monkeypatch, capfd, route):
    cfg = ROUTES[route]
    first = "A14" if route == "ordered_repeats" else "A"
    with _handle(K, monkeypatch, cfg) as idx:
        idx.add_proteome(small.prot[first])
        idx.finalize()
        assert idx.stats()["build_path"] == cfg[4]
        assert idx.signature_count() > 0 and idx.stats()["n_distinct_ids"] > 0
        capfd.readouterr()
        idx.append_proteome(small.prot["B"])
        line = _append_line(capfd)
        assert idx.stats()["n_distinct_ids"] == 0  # (until signature_count runs on the merged index)
        assert line["A_layout"] == ("compact" if cfg[4] == 2 else "seg"), line
        # the batch takes the route of the old index, except where its size rules that out: at scaled 10 its 30 k tuples
        # are too few for the unstable partition, and 300 k residues are not repeat-heavy at hp k24
        if route != "ordered_repeats":
            assert line["batch_path"] == (0 if route == "scatter_scaled" else cfg[4]), line
        if route == "scatter_scaled":  # scaled 10: few of the batch's hashes are in the old index
            assert 0 < line["matched"] < line["U_B"] // 10, line
        st = _equals_oracle(small, idx, (first, "B"), cfg)
        assert st["n_residues"] == len(small.raw[first][0]) + len(small.raw["B"][0])
        assert st["n_distinct_ids"] > 0  # (signature_count has run)
        assert line["n_C"] == st["n_tuples"] and line["U_A"] + line["U_B"] - line["matched"] == st["n_unique_hashes"]
        _two_add_equal(K, monkeypatch, cfg, idx, [small.prot[first], small.prot["B"]])


# ---- 3: chains and edge batches ---------------------------------------------------------------------------------------
def test_append_chain_and_edge_batches(K, small, monkeypatch, capfd):
    cfg = ROUTES["scatter"]
    with _handle(K, monkeypatch, cfg) as idx:
        idx.add_proteome(small.prot["A"])
        idx.finalize()
        names = ("A",)
        for step, name in enumerate(("B", "C", "short", "one", "empty")):
            capfd.readouterr()
            idx.append_proteome(small.prot[name])
            line = _append_line(capfd)
            assert line["A_layout"] == ("seg" if step == 0 else "compact"), line
            names = names + (name,)
            _equals_oracle(small, idx, names, cfg)
            if name == "short":
                assert line["U_B"] == 0
        assert idx.names() == sum((small.prot[n].names for n in names), [])
    with _handle(K, monkeypatch, cfg) as idx:  # onto a finalized empty index
        idx.finalize()
        idx.append_proteome(small.prot["B"])
        _equals_oracle(small, idx, ("B",), cfg)


# ---- 4: key overlap extremes ------------------------------------------------------------------------------------------
def test_append_a_copy_matches_every_key(K, small, monkeypatch, capfd):
    cfg = ROUTES["dense"]
    with _handle(K, monkeypatch, cfg) as idx:
        idx.add_proteome(small.prot["A"])
        idx.finalize()
        capfd.readouterr()
        idx.append_proteome(small.prot["A"])
        line = _append_line(capfd)
        assert line["matched"] == line["U_B"] == line["U_A"], line
        keys, row_ptr, _, _ = idx.csr()
        ok, orow, _, _ = small.index(("A",), cfg)
        assert np.array_equal(keys, ok) and np.array_equal(np.diff(row_ptr), 2 * np.diff(orow))
        _equals_oracle(small, idx, ("A", "A"), cfg)


# ---- 5: search after append -------------------------------------------------------------------------------------------
def test_search_after_append(K, O, small, monkeypatch):
    from kmerseek_b200 import synth
    cfg = ROUTES["dense"]
    k, moltype, scaled = cfg[:3]
    P_A = small.n_proteins(("A",))
    with _handle(K, monkeypatch, cfg) as idx:
        idx.add_proteome(small.prot["A"])
        idx.finalize()
        res, offs = small.raw["A"]
        qres, qoffs, _ = synth.queries(res, offs, 64, 11, min_len=k + 14, max_len=200)
        _search_equals_oracle(K, O, idx, res, offs, qres, qoffs, k, moltype, scaled)  # search -> append -> search
        idx.append_proteome(small.prot["B"])
        res, offs = small.concat(("A", "B"))
        qres, qoffs, src = synth.queries(res, offs, 256, 12, min_len=k + 14, max_len=200)
        assert (src >= P_A).any() and (src < P_A).any()
        r = _search_equals_oracle(K, O, idx, res, offs, qres, qoffs, k, moltype, scaled)
        assert (r.pairs["pair_pid"] >= P_A).any() and (r.hits["hit_pid"] >= P_A).any()


# ---- 6: tuples ----------------------------------------------------------------------------------------------------------
def test_append_tuples_and_signatures(K, small, monkeypatch):
    from kmerseek_b200 import _ffi
    from kmerseek_b200.index import _np
    cfg = ROUTES["scatter"]
    L = _lib()
    with _handle(K, monkeypatch, cfg) as idx:
        idx.add_proteome(small.prot["A"])
        idx.finalize()
        out = C.POINTER(_ffi.ks_sketch)()
        _ok(L.ks_sketch_batch(idx._h, small.prot["B"]._h, C.byref(out)))
        try:
            s = out.contents
            n, P = s.n_tuples, s.n_proteins
            h, pid, pos = _np(s.hash, n, np.uint64), _np(s.pid, n, np.uint32), _np(s.pos, n, np.uint32)
        finally:
            L.ks_sketch_free(out)
        _ok(L.ks_index_append_tuples(idx._h, h.ctypes.data_as(_ffi.u64p), pid.ctypes.data_as(_ffi.u32p),
                                     pos.ctypes.data_as(_ffi.u32p), n, P))
        _equals_oracle(small, idx, ("A", "B"), cfg)
    with _handle(K, monkeypatch, cfg) as idx:  # the Python mirror: store_signatures on a finalized index
        idx.add_proteome(small.prot["A"])
        idx.finalize()
        prot = small.prot["B"]
        sigs = idx.create_protein_signatures([prot.sequence(i) for i in range(prot.n_proteins)], prot.names)
        idx.append_signatures(sigs)
        _equals_oracle(small, idx, ("A", "B"), cfg)
        assert idx.names()[small.n_proteins(("A",)):] == prot.names


# ---- 7: errors leave the index intact -----------------------------------------------------------------------------------
def _snapshot(K, idx, queries):
    r = K.search(idx, queries, hits=True)
    return idx.csr(), idx.export_sketches(), r.pairs, r.hits, idx.stats()


@pytest.mark.parametrize("when", ["build", "merge"])
@pytest.mark.parametrize("route", ["scatter", "dense_library"])
def test_failed_append_restores_the_index(K, O, small, monkeypatch, route, when):
    """An append that fails after the old index was parked -- after the batch's build, or after the merge kernels have
    overwritten the device totals -- puts the old index back: the same CSR, export, search results and stats, and the
    oracle's index.  Old index in the segmented layout (scatter) and the compact one (dense_library, whose export reads
    the totals on the device).  KS_APPEND_FAIL makes the append fail as an allocation would."""
    from kmerseek_b200 import _ffi, synth
    cfg = ROUTES[route]
    k, moltype, scaled = cfg[:3]
    cfg_fail = cfg[:3] + ({**cfg[3], "KS_APPEND_FAIL": when}, cfg[4])
    L = _lib()
    with _handle(K, monkeypatch, cfg_fail) as idx:
        idx.add_proteome(small.prot["A"])
        idx.finalize()
        idx.signature_count()
        res, offs = small.raw["A"]
        qres, qoffs, _ = synth.queries(res, offs, 32, 14, min_len=k + 14, max_len=200)
        queries = K.Proteome.from_packed(qres, qoffs)
        before = _snapshot(K, idx, queries)
        assert L.ks_index_append_proteome(idx._h, small.prot["B"]._h) == 102  # KS_ERR_OUT_OF_MEMORY
        after = _snapshot(K, idx, queries)
        for x, y in zip(before[0], after[0]):
            assert np.array_equal(x, y)
        assert len(before[1]) == len(after[1])
        for (m, a), (rm, ra) in zip(before[1], after[1]):
            assert np.array_equal(m, rm) and np.array_equal(a, ra)
        for c in ("pair_qid", "pair_pid", "intersect_hashes", "n_weighted_found", "total_weighted_hashes", "containment"):
            assert np.array_equal(before[2][c], after[2][c]), c
        for c in ("hit_qid", "hit_pid", "hit_qpos", "hit_tpos", "hit_hash"):
            assert np.array_equal(before[3][c], after[3][c]), c
        for f in ("n_proteins", "n_residues", "n_windows", "n_tuples", "n_unique_hashes", "n_groups", "n_distinct_ids",
                  "finalized", "build_path"):
            assert before[4][f] == after[4][f], f
        _equals_oracle(small, idx, ("A",), cfg, path=cfg[4])
        _search_equals_oracle(K, O, idx, res, offs, qres, qoffs, k, moltype, scaled)


def test_append_errors_leave_the_index(K, O, small, monkeypatch):
    from kmerseek_b200 import _ffi, synth
    cfg = ROUTES["scatter"]
    k, moltype, scaled = cfg[:3]
    L = _lib()
    with _handle(K, monkeypatch, cfg) as idx:
        _ok(L.ks_index_add_proteome(idx._h, small.prot["A"]._h))  # pending, not finalized
        assert L.ks_index_append_proteome(idx._h, small.prot["B"]._h) == KS_ERR_NOT_FINALIZED
        assert L.ks_index_append_tuples(idx._h, None, None, None, 0, 1) == KS_ERR_NOT_FINALIZED
        _equals_oracle(small, idx, ("A",), cfg, path=cfg[4])  # (finalizes what was added)
        before = idx.csr()
        res, offs = small.raw["A"]
        qres, qoffs, _ = synth.queries(res, offs, 32, 13, min_len=k + 14, max_len=200)
        r0 = _search_equals_oracle(K, O, idx, res, offs, qres, qoffs, k, moltype, scaled)
        P_A = small.n_proteins(("A",))
        assert L.ks_index_append_tuples(idx._h, None, None, None, 0, (1 << 32) - 1 - P_A) == KS_ERR_CAPACITY
        assert L.ks_index_append_proteome(None, small.prot["B"]._h) == KS_ERR_VALIDATION
        assert L.ks_index_append_proteome(idx._h, None) == KS_ERR_VALIDATION
        assert L.ks_index_append_tuples(idx._h, None, None, None, 5, 1) == KS_ERR_VALIDATION
        h = np.array([5, 3], np.uint64)
        bad_pid, pos = np.array([0, 2], np.uint32), np.array([0, 1], np.uint32)  # protein index out of range
        assert L.ks_index_append_tuples(idx._h, h.ctypes.data_as(_ffi.u64p), bad_pid.ctypes.data_as(_ffi.u32p),
                                        pos.ctypes.data_as(_ffi.u32p), 2, 1) == KS_ERR_VALIDATION
        for x, y in zip(before, idx.csr()):
            assert np.array_equal(x, y)
        r1 = _search_equals_oracle(K, O, idx, res, offs, qres, qoffs, k, moltype, scaled)
        assert r0.n_pairs == r1.n_pairs and r0.n_hits == r1.n_hits
        assert idx.stats()["build_path"] == cfg[4]
        # an append, then clear + add C + finalize: the ping-pong buffers carry nothing over
        idx.append_proteome(small.prot["B"])
        idx.clear()
        idx.add_proteome(small.prot["C"])
        _equals_oracle(small, idx, ("C",), cfg, path=cfg[4])


# ---- 8: a pipelined (streamed dense) batch ------------------------------------------------------------------------------
def test_append_pipelined_batch(K, monkeypatch, capfd):
    from kmerseek_b200 import synth
    cfg = (24, "hp", 1, {}, 1)
    a = K.Proteome.from_packed(*synth.proteome(2_000_000, 4301))
    b = K.Proteome.from_packed(*synth.proteome(68_000_000, 4302))
    with _handle(K, monkeypatch, cfg) as idx:
        idx.add_proteome(a)
        idx.finalize()
        capfd.readouterr()
        idx.append_proteome(b)
        line = _append_line(capfd)
        assert line["batch_path"] == 1, line
        assert idx.stats()["build_path"] == 4
        _two_add_equal(K, monkeypatch, cfg, idx, [a, b])


# ---- 9: full size -------------------------------------------------------------------------------------------------------
def test_append_to_c2(K, O, monkeypatch, capfd):
    """C2 (200 M residues, hp k24: the no-parity dense layout) + a 2 M-residue append, against the two-add build, and a
    seeded sample of 4 096 postings against the oracle's hash of each posting's window."""
    from kmerseek_b200 import synth
    cfg = (24, "hp", 1, {}, 1)
    k = cfg[0]
    ra, oa = synth.proteome(200_000_000, 2024)
    rb, ob = synth.proteome(2_000_000, 4401)
    a, b = K.Proteome.from_packed(ra, oa), K.Proteome.from_packed(rb, ob)
    with _handle(K, monkeypatch, cfg) as idx:
        idx.add_proteome(a)
        idx.finalize()
        assert idx.stats()["build_path"] == 1
        capfd.readouterr()
        idx.append_proteome(b)
        line = _append_line(capfd)
        assert line["A_layout"] == "seg", line
        keys, row_ptr, pid, pos = idx.csr()
        _two_add_equal(K, monkeypatch, cfg, idx, [a, b])
    res = np.concatenate([ra, rb])
    offs = np.concatenate([oa, ob[1:] + np.uint64(len(ra))])
    j = np.random.default_rng(20261021).integers(0, len(pid), size=4096)
    row = np.searchsorted(row_ptr, j, "right") - 1
    start = offs[:-1].astype(np.int64)[pid[j]] + pos[j].astype(np.int64)
    wres = res[start[:, None] + np.arange(k)].ravel()
    woffs = np.arange(0, k * len(j) + 1, k, dtype=np.uint64)
    oh, opid, opos = O.sketch_tuples(wres, woffs, k, "hp", 1)
    assert np.array_equal(opid, np.arange(len(j))) and not opos.any()
    assert np.array_equal(keys[row], oh)
    assert (pid[j] >= len(oa) - 1).any()  # the sample holds postings of the appended proteins
