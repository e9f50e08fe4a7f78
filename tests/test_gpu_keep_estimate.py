"""Batches at scaled > 1 that keep more tuples than the host estimates (expected_kept, csrc/api.cu), on every build route,
against the oracle.  The host cannot know how many windows the FracMinHash filter keeps, so the ordered route's tuple
buffer and the unstable partition's plan are sized from an estimate; a batch that keeps more takes code of its own: the
sketch kernels' bounded write past capacity, the grow-and-redo of sketch_ordered (with held tuples too), the redo of a
pipelined add, a region or bucket overflow that sends a scattered batch back to the ordered route in finalize, and the
sketch kernel's per-protein counts when the partition holds more tuples than planned but does not overflow.

The inputs raise the keep rate with proteins of exactly k residues, each a window the oracle keeps (drawn with
replacement from a synthetic proteome's kept windows): every such protein is one kept tuple, and the hashes stay spread,
so nothing overflows unless the count does.  Low-complexity runs (one kept hash thousands of times) are the other kind.
Every case asserts its build_path, the oracle's CSR, per-protein sketches and stats, that the sketch was redone (more
sketch launches than a control build of the synthetic part alone, on the same route), and where marked a search against
the oracle.  Needs a GPU: run with -m gpu."""
import math

import numpy as np
import pytest

from test_gpu_append import _append_line, _handle, _two_add_equal
from test_gpu_parity import SCORE_NAMES, SCORE_RTOL, _csr_equals_oracle

pytestmark = pytest.mark.gpu

PIPELINE_MIN_RESIDUES = 64 << 20  # add_proteome_pipelined streams batches of at least this many residues


@pytest.fixture(scope="module")
def K():
    import kmerseek_b200
    return kmerseek_b200


@pytest.fixture(scope="module")
def O():
    from oracle import oracle
    return oracle


def expected_kept(windows, scaled):
    """csrc/api.cu expected_kept: the tuples the host plans for."""
    if scaled <= 1:
        return windows
    e = windows / scaled
    return min(windows, int(e * 1.05 + 8.0 * math.sqrt(e + 1.0)) + 1024)


def _windows(offs, k):
    return int(np.maximum(np.diff(offs.astype(np.int64)) - (k - 1), 0).sum())


def _cat(parts):
    res = np.concatenate([r for r, _ in parts])
    offs, base = [np.zeros(1, np.uint64)], 0
    for r, o in parts:
        offs.append(o[1:] + np.uint64(base))
        base += len(r)
    return res, np.concatenate(offs)


def _run(letter, n):
    return np.frombuffer((letter * n).encode(), np.uint8).copy(), np.array([0, n], np.uint64)


def _n_groups(h, pid):
    """(hash, protein) groups: the sum of the per-protein sketch sizes."""
    if len(h) == 0:
        return 0
    o = np.lexsort((pid, h))
    hs, ps = h[o], pid[o]
    return int(1 + np.count_nonzero((hs[1:] != hs[:-1]) | (ps[1:] != ps[:-1])))


class Inputs:
    """Seeded synthetic proteomes and one-window proteins, built once per module."""

    def __init__(self, O):
        self.O = O
        self.cache = {}

    def _get(self, key, make):
        if key not in self.cache:
            self.cache[key] = make()
        return self.cache[key]

    def synth(self, n_residues, seed):
        from kmerseek_b200 import synth
        return self._get(("synth", n_residues, seed), lambda: synth.proteome(n_residues, seed))

    def kept(self, k, moltype, scaled, n, seed):
        """n proteins of exactly k residues, each a window the oracle keeps, drawn with replacement from the kept windows
        of a 4 M-residue synthetic proteome."""
        def make():
            res, offs = self.synth(4_000_000, 7001)
            _, pid, pos = self._get(("pool", k, moltype, scaled),
                                    lambda: self.O.sketch_tuples(res, offs, k, moltype, scaled))
            pick = np.random.default_rng(seed).integers(0, len(pid), size=n)
            start = offs[:-1].astype(np.int64)[pid[pick]] + pos[pick].astype(np.int64)
            return res[start[:, None] + np.arange(k)].ravel(), np.arange(0, k * n + 1, k, dtype=np.uint64)
        return self._get(("kept", k, moltype, scaled, n, seed), make)


@pytest.fixture(scope="module")
def data(O):
    return Inputs(O)


def _ratio(O, res, offs, k, moltype, scaled):
    """Oracle tuples of the batch and its kept count over the host's estimate."""
    t = O.sketch_tuples(res, offs, k, moltype, scaled)
    return t, len(t[0]) / expected_kept(_windows(offs, k), scaled)


def _control(K, monkeypatch, cfg, parts):
    """sketch_launches and build_path of a fresh handle that adds each of `parts` and finalizes."""
    with _handle(K, monkeypatch, cfg) as idx:
        for res, offs in parts:
            idx.add_proteome(K.Proteome.from_packed(res, offs))
        idx.finalize()
        st = idx.stats()
    return st["sketch_launches"], st["build_path"]


def _report(name, path, launches, control, ratio):
    print(f"[keep] {name}: build_path {path} sketch_launches {launches} (control {control}) kept/estimate {ratio:.2f}")


def _search_equals_indexed_oracle(K, O, idx, tuples, n_prot, qres, qoffs, k, moltype, scaled):
    """test_gpu_parity._search_equals_oracle with the target's oracle tuples given and the pairs from
    oracle.manysearch_indexed: the same rows as manysearch (test_oracle_golden checks it), without an all-pairs scan over
    hundreds of thousands of one-window targets.  Query sketches, every pair column (integers bit-exact, the 12 scores
    within SCORE_RTOL) and the hit list."""
    oh, opid, opos = tuples
    r = K.search(idx, K.Proteome.from_packed(qres, qoffs), hits=True)
    qh, qid, qpos = O.sketch_tuples(qres, qoffs, k, moltype, scaled)
    qsk = O.protein_sketches(qh, qid, len(qoffs) - 1)
    for (m, a), (om, oa) in zip(r.query_sketches, qsk):
        assert np.array_equal(m, om) and np.array_equal(a, oa)
    assert np.array_equal(r.q_sizes, [len(m) for m, _ in qsk])
    assert int(opid.max()) < n_prot
    orows = O.manysearch_indexed(qsk, oh, opid, k, scaled, moltype)
    p = r.pairs
    assert r.n_pairs == len(orows) > 0
    assert np.array_equal(p["pair_qid"], [o["qid"] for o in orows]) and np.array_equal(p["pair_pid"], [o["pid"] for o in orows])
    for c in ("intersect_hashes", "n_weighted_found", "total_weighted_hashes"):
        assert np.array_equal(p[c], [o[c] for o in orows]), c
    for c in SCORE_NAMES:
        np.testing.assert_allclose(p[c], [o[c] for o in orows], rtol=SCORE_RTOL, atol=1e-12, err_msg=c)
    ohits = O.hits(qh, qid, qpos, oh, opid, opos)
    hh = r.hits
    mine = list(zip(hh["hit_qid"].tolist(), hh["hit_pid"].tolist(), hh["hit_hash"].tolist(), hh["hit_qpos"].tolist(),
                    hh["hit_tpos"].tolist()))
    assert mine == ohits
    return r


def _queries(syn, kept, k, letter, seed, n_synth=24):
    """Planted queries over the synthetic part, four of twelve concatenated kept windows each, and a run of k + 2 residues
    of `letter` (three windows: against a 20 k-residue run of the same letter that is 60 k hits already)."""
    from kmerseek_b200 import synth
    parts = [synth.queries(*syn, n_synth, seed, min_len=k + 30, max_len=240)[:2]]
    kres, koffs = kept
    rng = np.random.default_rng(seed)
    for _ in range(4):
        j = rng.integers(0, len(koffs) - 1, size=12)
        q = kres[(j[:, None] * k + np.arange(k)).ravel()]
        parts.append((q, np.array([0, len(q)], np.uint64)))
    parts.append(_run(letter, k + 2))
    return _cat(parts)


# ---- one batch, one add: the ordered route (A, A', E), the scatter route with an overflow (B, D) and without (C) ---------
# name -> (k, moltype, scaled, environment, build_path, control's build_path), the synthetic part (residues, seed), the
# one-window proteins (count, seed), a low-complexity run (letter, length), the keep rate over the estimate the case is
# built for, whether the sketch is redone, and whether the index is searched
ONE_BATCH = {
    # the ordered route: sketch_ordered's first launch writes up to the estimate, grows the buffer and runs again
    "A": ((7, "protein", 10, {"KS_SCATTER": "0"}, 0), 0, (2_000_000, 4101), (300_000, 7101), None, 2.0, True, True),
    # the same in the hp alphabet: at k12 s5 every batch is repeat-heavy and takes the ordered route on its own
    "A_hp": ((12, "hp", 5, {}, 0), 0, (2_000_000, 4101), (400_000, 7102), None, 1.5, True, False),
    # the scatter route: the plan has 2^9 final buckets (msd_top_bits raises tb to 12 - lz = 9 at scaled 10), about 4 900
    # tuples each against LS_CAP = 4 096: they overflow, finalize sketches the batch again in order (which also runs short)
    "B": ((7, "protein", 10, {}, 0), 3, (2_000_000, 4101), (1_800_000, 7103), None, 4.5, True, True),
    # the scatter route with 8 % more tuples than planned and no overflow (tb 9, about 2 250 per final bucket): no redo,
    # and t_abund / t_size come from the sketch kernel's per-protein counts
    "C": ((7, "protein", 10, {}, 3), 3, (8_000_000, 808), (134_000, 7104), None, 1.05, False, True),
    # C's input and 30 000 L: one kept hash overflows its bucket, the ordered redo takes the stable path, whose oversize
    # bucket takes the library sort
    "D": ((7, "protein", 10, {}, 0), 3, (8_000_000, 808), (134_000, 7104), ("L", 30_000), 1.05, True, False),
    # k > 32: the byte-loop kernel (look-back path only) writes up to the estimate, then the redo
    "E": ((40, "protein", 10, {}, 0), 0, (2_000_000, 4101), (60_000, 7105), ("A", 20_000), 1.25, True, True),
}


@pytest.mark.parametrize("case", list(ONE_BATCH))
def test_one_batch_beyond_the_estimate(K, O, data, monkeypatch, case):
    cfg, control_path, (n_syn, syn_seed), (n_kept, kept_seed), run, min_ratio, redo, search = ONE_BATCH[case]
    k, moltype, scaled, _, path = cfg
    syn = data.synth(n_syn, syn_seed)
    kept = data.kept(k, moltype, scaled, n_kept, kept_seed)
    res, offs = _cat([syn, kept] + ([_run(*run)] if run else []))
    tuples, ratio = _ratio(O, res, offs, k, moltype, scaled)
    assert ratio > min_ratio, ratio  # the input still runs short of the estimate by the factor the case is built for
    if run:  # every window of the run is the same kept hash
        _, counts = np.unique(tuples[0], return_counts=True)
        assert counts.max() >= run[1] - k + 1
    with _handle(K, monkeypatch, cfg) as idx:
        idx.add_proteome(K.Proteome.from_packed(res, offs))
        idx.finalize()
        st = idx.stats()  # (before any export or search)
        launches = st["sketch_launches"]
        _csr_equals_oracle(K, O, res, offs, k, moltype, scaled, path=path, idx=idx)
        assert st["n_groups"] == _n_groups(tuples[0], tuples[1])
        if search:
            qres, qoffs = _queries(syn, kept, k, run[0] if run else "L", 300 + k)
            r = _search_equals_indexed_oracle(K, O, idx, tuples, len(offs) - 1, qres, qoffs, k, moltype, scaled)
            assert r.n_hits < 200_000
            if case == "E":  # a batch with a query of more than 4 096 windows: the library-sorted query path
                long_q = syn[0][1000:7000].copy()
                qres2, qoffs2 = _cat([(long_q, np.array([0, len(long_q)], np.uint64)), (qres, qoffs)])
                assert len(long_q) - k + 1 > 4096
                _search_equals_indexed_oracle(K, O, idx, tuples, len(offs) - 1, qres2, qoffs2, k, moltype, scaled)
    control, cpath = _control(K, monkeypatch, cfg, [syn])
    _report(case, st["build_path"], launches, control, ratio)
    assert cpath == control_path
    assert launches > control if redo else launches == control, (launches, control)


# ---- F: a second add behind held tuples -----------------------------------------------------------------------------------
def test_second_add_beyond_the_estimate_keeps_the_held_tuples(K, O, data, monkeypatch):
    """add(300 k) then add(A's input): the second add takes the ordered route behind the first batch's tuples; growing the
    buffer for the redo must copy them."""
    cfg = (7, "protein", 10, {}, 0)
    k, moltype, scaled = cfg[:3]
    first = data.synth(300_000, 4102)
    syn = data.synth(2_000_000, 4101)
    second = _cat([syn, data.kept(k, moltype, scaled, 300_000, 7101)])
    _, ratio = _ratio(O, *second, k, moltype, scaled)
    assert ratio > 2.0, ratio
    res, offs = _cat([first, second])
    with _handle(K, monkeypatch, cfg) as idx:
        idx.add_proteome(K.Proteome.from_packed(*first))
        idx.add_proteome(K.Proteome.from_packed(*second))
        idx.finalize()
        st = idx.stats()
        launches = st["sketch_launches"]
        _csr_equals_oracle(K, O, res, offs, k, moltype, scaled, path=0, idx=idx)
        assert st["n_groups"] == _n_groups(*O.sketch_tuples(res, offs, k, moltype, scaled)[:2])
    control, cpath = _control(K, monkeypatch, cfg, [first, syn])
    _report("F", st["build_path"], launches, control, ratio)
    assert cpath == 0 and launches > control, (launches, control)


# ---- G: an append whose batch overflows the partition ---------------------------------------------------------------------
def test_append_of_a_batch_beyond_the_estimate(K, O, data, monkeypatch, capfd):
    """A finalized 2 M-residue index (unstable partition, path 3), then B's batch appended: the batch is built alone while
    the old index is parked, overflows its buckets and is redone in order (batch_path 0).  Must equal the oracle's index
    of the concatenation and a second handle's add + add + finalize."""
    cfg = (7, "protein", 10, {}, 3)
    k, moltype, scaled = cfg[:3]
    old = data.synth(2_000_000, 4201)
    syn = data.synth(2_000_000, 4101)
    kept = data.kept(k, moltype, scaled, 1_800_000, 7103)
    batch = _cat([syn, kept])
    _, ratio = _ratio(O, *batch, k, moltype, scaled)
    assert ratio > 4.5, ratio
    res, offs = _cat([old, batch])
    tuples = O.sketch_tuples(res, offs, k, moltype, scaled)
    prots = [K.Proteome.from_packed(*old), K.Proteome.from_packed(*batch)]
    with _handle(K, monkeypatch, cfg) as idx:
        idx.add_proteome(prots[0])
        idx.finalize()
        assert idx.stats()["build_path"] == 3
        capfd.readouterr()
        idx.append_proteome(prots[1])
        line = _append_line(capfd)
        st = idx.stats()
        launches = st["sketch_launches"]
        assert line["batch_path"] == 0, line
        _csr_equals_oracle(K, O, res, offs, k, moltype, scaled, path=4, idx=idx)
        assert st["n_groups"] == _n_groups(tuples[0], tuples[1])
        _two_add_equal(K, monkeypatch, cfg, idx, prots)
        qres, qoffs = _queries(_cat([old, syn]), kept, k, "L", 317)
        _search_equals_indexed_oracle(K, O, idx, tuples, len(offs) - 1, qres, qoffs, k, moltype, scaled)
    with _handle(K, monkeypatch, cfg) as idx:  # control: the same append of the synthetic part alone
        idx.add_proteome(prots[0])
        idx.finalize()
        capfd.readouterr()
        idx.append_proteome(K.Proteome.from_packed(*syn))
        control_line = _append_line(capfd)
        control = idx.stats()["sketch_launches"]
    _report("G", line["batch_path"], launches, control, ratio)
    assert control_line["batch_path"] == 3, control_line
    assert launches > control, (launches, control)


# ---- H: pipelined adds (batches of at least 64 Mi residues) ----------------------------------------------------------------
@pytest.fixture(scope="module")
def big(O, data):
    """A 68 M-residue batch: 20 M synthetic residues and 48 M residues of one-window 7-mers (6.9 M proteins), with its
    oracle tuples; and a synthetic proteome of the same size, the controls' batch."""
    k, moltype, scaled = 7, "protein", 10
    syn = data.synth(20_000_000, 9001)
    res, offs = _cat([syn, data.kept(k, moltype, scaled, 48_000_000 // k, 7106)])
    assert len(res) >= PIPELINE_MIN_RESIDUES
    tuples, ratio = _ratio(O, res, offs, k, moltype, scaled)
    return res, offs, tuples, ratio, data.synth(len(res), 9002)


def _csr_equals_tuples(O, idx, tuples, st):
    """CSR and stats against oracle.build_index of the given tuples (no per-protein sketch lists: millions of proteins)."""
    keys, row_ptr, pid, pos = idx.csr()
    okeys, orow, opid, opos = O.build_index(*tuples)
    assert np.array_equal(keys, okeys) and np.array_equal(row_ptr, orow)
    assert np.array_equal(pid, opid) and np.array_equal(pos, opos)
    assert st["n_tuples"] == len(tuples[0]) and st["n_unique_hashes"] == len(okeys)
    assert st["n_groups"] == _n_groups(tuples[0], tuples[1])


def test_pipelined_scatter_batch_beyond_the_estimate(K, O, big, monkeypatch):
    """One pipelined add on the scatter route: the first-level regions (planned for 2.8 M tuples) overflow, finalize redoes
    the batch in order."""
    cfg = (7, "protein", 10, {}, 0)
    res, offs, tuples, ratio, control_batch = big
    assert ratio > 3.0, ratio
    with _handle(K, monkeypatch, cfg) as idx:
        idx.add_proteome(K.Proteome.from_packed(res, offs))
        idx.finalize()
        st = idx.stats()
        launches = st["sketch_launches"]
        assert st["build_path"] == 0
        _csr_equals_tuples(O, idx, tuples, st)
    control, cpath = _control(K, monkeypatch, cfg, [control_batch])
    _report("H1", st["build_path"], launches, control, ratio)
    assert cpath == 3 and launches > control, (launches, control)


def test_pipelined_ordered_batch_beyond_the_estimate(K, O, data, big, monkeypatch):
    """add(300 k), then the 68 M-residue batch: a pipelined add on the ordered route behind held tuples, whose chunked
    launches run past their capacity; the batch is sketched again through sketch_ordered."""
    cfg = (7, "protein", 10, {}, 0)
    k, moltype, scaled = cfg[:3]
    res, offs, (h, pid, pos), ratio, control_batch = big
    first = data.synth(300_000, 4102)
    h0, pid0, pos0 = O.sketch_tuples(*first, k, moltype, scaled)
    p0 = len(first[1]) - 1
    tuples = (np.concatenate([h0, h]), np.concatenate([pid0, pid + np.uint32(p0)]), np.concatenate([pos0, pos]))
    with _handle(K, monkeypatch, cfg) as idx:
        idx.add_proteome(K.Proteome.from_packed(*first))
        idx.add_proteome(K.Proteome.from_packed(res, offs))
        idx.finalize()
        st = idx.stats()
        launches = st["sketch_launches"]
        assert st["build_path"] == 0 and st["n_proteins"] == p0 + len(offs) - 1
        _csr_equals_tuples(O, idx, tuples, st)
    control, cpath = _control(K, monkeypatch, cfg, [first, control_batch])
    _report("H2", st["build_path"], launches, control, ratio)
    assert cpath == 0 and launches > control, (launches, control)
