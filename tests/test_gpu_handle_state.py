"""Index handle state: sequences of adds, clears, uploads, tuple adds and finalizes through the C ABI and the Python
wrapper, on every build route, must give the oracle's index and the route's build_path.  The routes are forced with
the handle's environment switches on small proteomes; the pipelined add (batches above 64 M residues) runs on one
proteome of 68 M residues.  Needs a GPU: run with -m gpu."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

KS_ERR_VALIDATION, KS_ERR_NOT_FINALIZED = 9, 10

# route -> (k, moltype, scaled, environment, build_path of one add); routes of one configuration next to each other, so
# that the oracle's results are computed once for them
ROUTES = {
    "dense": (16, "hp", 1, {"KS_DENSE": "1"}, 1),
    "scatter": (16, "dayhoff", 1, {}, 3),
    "ordered": (16, "dayhoff", 1, {"KS_SCATTER": "0"}, 0),
    "scatter_scaled": (7, "protein", 10, {}, 3),
    # ~0.8 tuples per possible hash at 14 M residues: the partition turns it down on its own
    "ordered_repeats": (24, "hp", 1, {"KS_DENSE": "0"}, 0),
}
# the pipelined add; its dense route takes the C2 configuration (hp k24), with which no sort bucket of the dense path
# overflows at this size
PIPELINED = {
    "dense": (24, "hp", 1, {}, 1),
    "scatter": (16, "dayhoff", 1, {}, 3),
    "ordered": (16, "dayhoff", 1, {"KS_SCATTER": "0"}, 0),
    "scatter_scaled": (7, "protein", 10, {}, 3),
}
BIG_RESIDUES = 68_000_000  # above the 64 M residues (2^26) from which ks_index_add_proteome streams the upload


@pytest.fixture(scope="module")
def K():
    import kmerseek_b200
    return kmerseek_b200


@pytest.fixture(scope="module")
def O():
    from oracle import oracle
    return oracle


class Data:
    """Proteomes as (residues, offsets) and as handles, and the oracle's indexes of them and of their concatenations
    (kept for one configuration at a time)."""

    def __init__(self, K, O):
        self.K, self.O = K, O
        self.raw, self.prot, self.cache, self.cfg = {}, {}, {}, None

    def add(self, name, n_residues, seed):
        from kmerseek_b200 import synth
        self.raw[name] = synth.proteome(n_residues, seed)
        self.prot[name] = self.K.Proteome.from_packed(*self.raw[name])

    def n_proteins(self, names):
        return sum(len(self.raw[n][1]) - 1 for n in names)

    def tuples(self, names, cfg):
        k, moltype, scaled = cfg[:3]
        if (k, moltype, scaled) != self.cfg:
            self.cache, self.cfg = {}, (k, moltype, scaled)
        if ("t", names) not in self.cache:
            res = np.concatenate([self.raw[n][0] for n in names])
            offs, base = [np.zeros(1, np.uint64)], 0
            for n in names:
                offs.append(self.raw[n][1][1:] + np.uint64(base))
                base += len(self.raw[n][0])
            self.cache[("t", names)] = self.O.sketch_tuples(res, np.concatenate(offs), k, moltype, scaled)
        return self.cache[("t", names)]

    def index(self, names, cfg):
        self.tuples(names, cfg)
        if ("i", names) not in self.cache:
            self.cache[("i", names)] = self.O.build_index(*self.cache.pop(("t", names)))
        return self.cache[("i", names)]


@pytest.fixture(scope="module")
def small(K, O):
    d = Data(K, O)
    d.add("A", 2_000_000, 4101)
    d.add("A14", 14_000_000, 4104)  # the repeat-heavy route's first batch
    d.add("B", 300_000, 4102)  # a second batch
    d.add("C", 2_000_000, 4103)  # different content for a rebuild
    return d


def _handle(K, monkeypatch, cfg):
    k, moltype, scaled, env, _ = cfg
    for name in ("KS_DENSE", "KS_SCATTER", "KS_NO_PIPELINE", "KS_SKETCH_GENERAL", "KS_DENSE_SORT"):
        monkeypatch.delenv(name, raising=False)
    for name, value in env.items():
        monkeypatch.setenv(name, value)  # read once, when the handle is created
    return K.ProteomeIndex("db", k, scaled, moltype)


def _lib():
    from kmerseek_b200 import _ffi
    return _ffi.lib()


def _ok(status):
    from kmerseek_b200.errors import check
    check(status)


def _csr_equals(d, idx, names, cfg, path):
    keys, row_ptr, pid, pos = idx.csr()  # (finalizes)
    okeys, orow, opid, opos = d.index(names, cfg)
    assert np.array_equal(keys, okeys) and np.array_equal(row_ptr, orow), names
    assert np.array_equal(pid, opid) and np.array_equal(pos, opos), names
    st = idx.stats()
    assert st["finalized"] == 1 and st["n_proteins"] == d.n_proteins(names)
    assert st["n_tuples"] == len(opid) and st["n_unique_hashes"] == len(okeys)
    assert path is None or st["build_path"] == path, (st["build_path"], path)
    return keys, row_ptr, pid, pos


# ---- the sequences: `first` is the name of the first batch, B the second -----------------------------------------------
def seq_rebuild_from_the_resident_batch(d, idx, first, cfg):
    """add -> finalize, then clear -> ks_index_sketch_resident -> finalize twice (the benchmark's loop): the same index
    and build_path every time."""
    idx.add_proteome(d.prot[first])
    ref = _csr_equals(d, idx, (first,), cfg, cfg[4])
    for _ in range(2):
        _ok(_lib().ks_index_clear(idx._h))
        assert idx.stats()["build_path"] == cfg[4]  # the last finalize's, until the next one
        _ok(_lib().ks_index_sketch_resident(idx._h))
        for x, y in zip(ref, _csr_equals(d, idx, (first,), cfg, cfg[4])):
            assert np.array_equal(x, y)


def seq_clear_drops_a_pending_batch(d, idx, first, cfg):
    """add -> clear -> add -> finalize: the first add, still pending, is gone."""
    idx.add_proteome(d.prot[first])
    idx.clear()
    st = idx.stats()
    assert st["n_tuples"] == 0 and st["n_proteins"] == 0 and st["finalized"] == 0
    idx.add_proteome(d.prot[first])
    _csr_equals(d, idx, (first,), cfg, cfg[4])


def seq_second_add(d, idx, first, cfg):
    """add -> add a second batch -> finalize: the pending first batch is sketched in order, then the second."""
    idx.add_proteome(d.prot[first])
    idx.add_proteome(d.prot["B"])
    _csr_equals(d, idx, (first, "B"), cfg, 0)


def seq_upload_another(d, idx, first, cfg):
    """add -> ks_index_upload of another proteome -> ks_index_sketch_resident -> finalize: replacing the resident batch
    keeps the pending one."""
    idx.add_proteome(d.prot[first])
    _ok(_lib().ks_index_upload(idx._h, d.prot["B"]._h))
    _ok(_lib().ks_index_sketch_resident(idx._h))
    _csr_equals(d, idx, (first, "B"), cfg, 0)


def seq_add_tuples(d, idx, first, cfg):
    """add -> ks_sketch_batch of another proteome (private counters: a pending batch keeps the handle's) ->
    ks_index_add_tuples of its tuples -> finalize."""
    from kmerseek_b200 import _ffi
    from kmerseek_b200.index import _np
    idx.add_proteome(d.prot[first])
    out = C.POINTER(_ffi.ks_sketch)()
    _ok(_lib().ks_sketch_batch(idx._h, d.prot["B"]._h, C.byref(out)))
    try:
        s = out.contents
        n, P = s.n_tuples, s.n_proteins
        h, pid, pos = _np(s.hash, n, np.uint64).copy(), _np(s.pid, n, np.uint32).copy(), _np(s.pos, n, np.uint32).copy()
    finally:
        _lib().ks_sketch_free(out)
    _ok(_lib().ks_index_add_tuples(idx._h, h.ctypes.data_as(_ffi.u64p), pid.ctypes.data_as(_ffi.u32p),
                                   pos.ctypes.data_as(_ffi.u32p), n, P))
    _csr_equals(d, idx, (first, "B"), cfg, 0)


SEQUENCES = [seq_rebuild_from_the_resident_batch, seq_clear_drops_a_pending_batch, seq_second_add, seq_upload_another,
             seq_add_tuples]


@pytest.mark.parametrize("seq", SEQUENCES, ids=[s.__name__[4:] for s in SEQUENCES])
@pytest.mark.parametrize("route", list(ROUTES))
def test_sequence(K, small, monkeypatch, route, seq):
    cfg = ROUTES[route]
    with _handle(K, monkeypatch, cfg) as idx:
        seq(small, idx, "A14" if route == "ordered_repeats" else "A", cfg)


@pytest.fixture(scope="module")
def big(K, O):
    d = Data(K, O)
    d.add("A", BIG_RESIDUES, 4201)
    d.add("B", 300_000, 4102)
    return d


@pytest.mark.parametrize("route", list(PIPELINED))
def test_pipelined_sequences(K, big, monkeypatch, route):
    """Every sequence above with a first batch that takes the pipelined add (the dense route then leaves the rank kernel
    run, the scatter routes a checked count).  One test per route: the oracle's indexes are kept for one configuration."""
    cfg = PIPELINED[route]
    for seq in SEQUENCES:
        with _handle(K, monkeypatch, cfg) as idx:
            seq(big, idx, "A", cfg)


def _search_equals(d, idx, name, cfg, seed):
    from kmerseek_b200 import synth
    k, moltype, scaled = cfg[:3]
    O = d.O
    res, offs = d.raw[name]
    qres, qoffs, _ = synth.queries(res, offs, 32, seed, min_len=max(30, k + 3), max_len=200)
    r = d.K.search(idx, d.K.Proteome.from_packed(qres, qoffs), hits=True)
    oh, opid, opos = O.sketch_tuples(res, offs, k, moltype, scaled)
    qh, qid, qpos = O.sketch_tuples(qres, qoffs, k, moltype, scaled)
    hh = r.hits
    mine = list(zip(hh["hit_qid"].tolist(), hh["hit_pid"].tolist(), hh["hit_hash"].tolist(), hh["hit_qpos"].tolist(),
                    hh["hit_tpos"].tolist()))
    assert mine == O.hits(qh, qid, qpos, oh, opid, opos) and len(mine) > 0
    orows = O.manysearch(O.protein_sketches(qh, qid, len(qoffs) - 1), O.protein_sketches(oh, opid, len(offs) - 1), k,
                         scaled, moltype)
    p = r.pairs
    assert r.n_pairs == len(orows)
    assert np.array_equal(p["pair_qid"], [o["qid"] for o in orows]) and np.array_equal(p["pair_pid"], [o["pid"] for o in orows])
    for c in ("intersect_hashes", "n_weighted_found", "total_weighted_hashes"):
        assert np.array_equal(p[c], [o[c] for o in orows]), c
    np.testing.assert_allclose(p["containment"], [o["containment"] for o in orows], rtol=1e-6, atol=1e-12)
    return oh, opid


@pytest.mark.parametrize("route", list(ROUTES))
def test_search_rebuild_search(K, small, monkeypatch, route):
    """finalize -> search -> clear -> add different content -> finalize -> search: the second search answers for the new
    content, and export works twice in a row (after a dense build the sorted hash column is rebuilt on the first)."""
    cfg = ROUTES[route]
    first = "A14" if route == "ordered_repeats" else "A"
    with _handle(K, monkeypatch, cfg) as idx:
        idx.add_proteome(small.prot[first])
        _csr_equals(small, idx, (first,), cfg, cfg[4])
        _search_equals(small, idx, first, cfg, 7)
        idx.clear()
        idx.add_proteome(small.prot["C"])
        _csr_equals(small, idx, ("C",), cfg, None if route == "ordered_repeats" else cfg[4])
        oh, opid = _search_equals(small, idx, "C", cfg, 8)
        osk = small.O.protein_sketches(oh, opid, small.n_proteins(("C",)))
        for _ in range(2):
            sk = idx.export_sketches()
            assert len(sk) == len(osk)
            for (m, a), (om, oa) in zip(sk, osk):
                assert np.array_equal(m, om) and np.array_equal(a, oa)


@pytest.mark.parametrize("route", list(ROUTES))
def test_add_after_finalize_and_search_before(K, small, monkeypatch, route):
    """An add to a finalized index fails with KS_ERR_VALIDATION and leaves the index as it was; a search of an index
    that is not finalized fails with KS_ERR_NOT_FINALIZED.  Through the C ABI: the Python wrapper finalizes on its own."""
    from kmerseek_b200 import _ffi
    cfg = ROUTES[route]
    first = "A14" if route == "ordered_repeats" else "A"
    L = _lib()
    with _handle(K, monkeypatch, cfg) as idx:
        _ok(L.ks_index_add_proteome(idx._h, small.prot[first]._h))
        out = C.POINTER(_ffi.ks_search_result)()
        assert L.ks_search_batch(idx._h, small.prot["B"]._h, _ffi.KS_SEARCH_HITS, C.byref(out)) == KS_ERR_NOT_FINALIZED
        _ok(L.ks_index_finalize(idx._h))
        assert L.ks_index_add_proteome(idx._h, small.prot["B"]._h) == KS_ERR_VALIDATION
        assert L.ks_index_add_tuples(idx._h, None, None, None, 0, 0) == KS_ERR_VALIDATION
        _csr_equals(small, idx, (first,), cfg, cfg[4])
