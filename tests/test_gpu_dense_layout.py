"""The dense k-mer space path (hp, 8 <= k <= 24, scaled 1) with keys that fill all 64 bits.

A key of the dense path is code | protein | position.  dense_begin (api.cu) lays it out WITH the parity bit -- the code's
lowest bit tells pattern windows (odd) from windows with an X / U / O / * (even, hashed from their bytes) -- when
16 + rb_full + pid_bits + pos_bits <= 64, and WITHOUT it (rb = rb_full - 1, a window without a pattern sends the batch to
the general path) when only that fits.  C2 (570 k proteins, 200 M residues, hp k=24) needs 65 bits with the parity bit and
runs the second layout.  Every proteome here is sized so that its keys are exactly 64 bits wide: short proteins, then one
long protein LAST, so that the largest protein id and the largest positions are in the same keys.  Each build proves from
the handle's KS_TIMING lines the layout, the bucket bits of the key sort and the build path it targets, and must equal the
oracle's index.  Needs a GPU: run with -m gpu."""
import re

import numpy as np
import pytest

from test_gpu_parity import _csr_equals_oracle, _search_equals_oracle

pytestmark = pytest.mark.gpu

# rb_full = bits_for_value(2 x largest 16-bit hash-prefix group + 2): 320 patterns at k=24, 180 at k=23
RB_FULL = {24: 10, 23: 9}

# name: k, short proteins, their length range, long protein, parity layout, bucket bits of the key sort, build_path
CASES = {
    # 16 + 10 + 16 + 22 = 64 bits; ~9.2 M windows: 12 bucket bits, 52 key bits below them (the bucket kernel's limit)
    "k24_parity": (24, 65_535, (90, 110), 2**22 - 1, 1, 12, 1),
    # 16 + 9 + 17 + 22 = 64 bits
    "k24_no_parity": (24, 65_536, (90, 110), 2**22 - 1, 0, 12, 1),
    # ~5.3 M windows: 11 bucket bits would leave 53 key bits below them, more than the bucket kernel keeps beside a
    # key's slot: the library sorts the keys
    "k24_parity_library": (24, 65_535, (36, 44), 2**22 - 1, 1, None, 2),
    # 16 + 9 + 16 + 23 = 64 bits; 13 bucket bits put the parity bit among the 13 bin bits of the bucket kernel (squeeze)
    "k23_parity_squeeze": (23, 65_535, (90, 110), 2**23 - 1, 1, 13, 1),
    # 16 + 8 + 17 + 23 = 64 bits
    "k23_no_parity": (23, 65_536, (90, 110), 2**23 - 1, 0, 13, 1),
}
SEEDS = {name: 7100 + i for i, name in enumerate(CASES)}

ELIGIBLE = re.compile(r"^\[ks\] dense eligible: (\d) ", re.M)
BEGIN = re.compile(r"^\[ks\] dense begin: state (-?\d+) rb (\d+)$", re.M)
FINALIZE = re.compile(r"^\[ks\] dense finalize: n (\d+) produced \d+ unhandled (\d+) exc (\d+) overflow (\d+) U \d+ G \d+ "
                      r"plan l1 (\d+) l2 (\d+) rb (\d+)$", re.M)


@pytest.fixture(scope="module")
def K():
    import kmerseek_b200
    return kmerseek_b200


@pytest.fixture(scope="module")
def O():
    from oracle import oracle
    return oracle


class _Kept:
    """The oracle, with its results kept per argument arrays: a proteome is checked against it more than once."""

    def __init__(self, O):
        self._O, self._kept = O, {}

    def __getattr__(self, name):
        return getattr(self._O, name)

    def _once(self, name, *args):
        key = (name,) + tuple(id(a) if isinstance(a, np.ndarray) else a for a in args)
        if key not in self._kept:  # (the arguments are kept too: their ids stay theirs)
            self._kept[key] = (args, getattr(self._O, name)(*args))
        return self._kept[key][1]

    def sketch_tuples(self, *args):
        return self._once("sketch_tuples", *args)

    def build_index(self, *args):
        return self._once("build_index", *args)

    def protein_sketches(self, *args):
        return self._once("protein_sketches", *args)


def _proteome(n_short, short_len, long_len, seed):
    """n_short proteins of short_len[0] .. short_len[1] residues, then one of long_len; i.i.d. residues."""
    from kmerseek_b200 import synth
    rng = np.random.Generator(np.random.PCG64(seed))
    lens = np.append(rng.integers(short_len[0], short_len[1] + 1, size=n_short), long_len)
    offs = np.zeros(len(lens) + 1, dtype=np.uint64)
    np.cumsum(lens, out=offs[1:])
    return synth.residues_iid(int(offs[-1]), rng), offs


@pytest.fixture(scope="module")
def data():
    made = {}

    def get(name):
        if name not in made:
            made[name] = _proteome(*CASES[name][1:4], SEEDS[name])
        return made[name]
    return get


def _bits_for_value(v):  # api.cu: bits that hold the values 0 .. v
    return max(1, int(v).bit_length())


def _widths(offs):
    """(pid_bits, pos_bits) of a batch, as dense_begin derives them."""
    return _bits_for_value(len(offs) - 2), _bits_for_value(int(np.diff(offs.astype(np.int64)).max()))


def _windows(offs, k):
    return int(np.maximum(np.diff(offs.astype(np.int64)) - (k - 1), 0).sum())


def _env(monkeypatch, **values):
    for name in ("KS_DENSE", "KS_DENSE_SORT", "KS_SCATTER", "KS_NO_PIPELINE", "KS_SKETCH_GENERAL"):
        monkeypatch.delenv(name, raising=False)
    monkeypatch.setenv("KS_TIMING", "1")  # read when a handle is created
    for name, value in values.items():
        monkeypatch.setenv(name, value)


def _layout(err):
    """What the KS_TIMING lines of one add + finalize say: whether the dense path took the batch and, when it did, the
    layout of its keys (parity = the code width of the build is rb_full), the bucket bits of the key sort (0: the
    library sorts the keys) and the rank kernel's flags."""
    el = ELIGIBLE.findall(err)
    assert len(el) == 1, err
    if el[0] == "0":
        assert not BEGIN.search(err) and not FINALIZE.search(err), err
        return {"eligible": 0}
    b, f = BEGIN.findall(err), FINALIZE.findall(err)
    assert len(b) == 1 and len(f) == 1, err
    state, rb_full = map(int, b[0])
    n, unhandled, exc, overflow, l1, l2, rb = map(int, f[0])
    assert rb in (rb_full, rb_full - 1), err
    return {"eligible": 1, "state": state, "rb_full": rb_full, "parity": int(rb == rb_full), "total": l1 + l2, "n": n,
            "unhandled": unhandled, "exc": exc, "overflow": overflow}


def _check(K, O, capfd, res, offs, k, path, expect, idx=None):
    """One build (a new handle, or `idx` that the batch has been added to) against the oracle, and its layout."""
    st = _csr_equals_oracle(K, O, res, offs, k, "hp", path=path, idx=idx)
    lay = _layout(capfd.readouterr().err)
    assert {name: lay.get(name) for name in expect} == expect, lay
    return st, lay


def _full_width(offs, k, parity):
    pid_bits, pos_bits = _widths(offs)
    return 16 + RB_FULL[k] - (1 - parity) + pid_bits + pos_bits


@pytest.mark.parametrize("case", list(CASES))
def test_full_width_keys_equal_oracle(K, O, data, monkeypatch, capfd, case):
    k, _, _, long_len, parity, total, path = CASES[case]
    res, offs = data(case)
    assert _widths(offs) == (16 + (1 - parity), _bits_for_value(long_len))
    assert _full_width(offs, k, parity) == 64 and (parity or _full_width(offs, k, 1) == 65)
    O = _Kept(O)
    _env(monkeypatch)
    capfd.readouterr()
    n = _windows(offs, k)
    expect = {"eligible": 1, "state": 1, "rb_full": RB_FULL[k], "parity": parity, "unhandled": 0, "exc": 0, "overflow": 0,
              "n": n, "total": total if path == 1 else 0}
    _check(K, O, capfd, res, offs, k, path, expect)
    if path == 2:  # no hook: the slot guard of dense_sort_plan turned the hand-written sort down
        need = 0
        while (n >> need) > 3072:
            need += 1
        assert 64 - need == 53, need
        return
    # the same keys sorted by the library (KS_DENSE_SORT=library, k=24 only: the sort's key width, not the squeeze, is
    # what this varies)
    if k == 24:
        _env(monkeypatch, KS_DENSE_SORT="library")
        _check(K, O, capfd, res, offs, k, 2, dict(expect, total=0))


@pytest.mark.parametrize("k", [24, 23])
def test_one_bit_too_many_is_not_dense(K, O, monkeypatch, capfd, k):
    """65 bits even without the parity bit: dense_eligible turns the batch down (its estimate of rb_full, the tables are
    not built yet), and with more than 0.25 tuples per possible hash it takes the ordered route."""
    res, offs = _proteome(65_536, (90, 110), 2**(47 - k) - 1, 7200 + k)
    assert _widths(offs) == (17, 47 - k) and _full_width(offs, k, 0) == 65
    _env(monkeypatch)
    capfd.readouterr()
    _check(K, O, capfd, res, offs, k, 0, {"eligible": 0})


@pytest.mark.parametrize("case", ["k24_parity", "k23_parity_squeeze", "k24_no_parity", "k23_no_parity"])
def test_exception_windows_at_full_width(K, O, data, monkeypatch, capfd, case):
    """X / U / O / * in short proteins and in the long one past position 2^(pos_bits - 1), plus a run of X: with the
    parity bit the exception keys are built on the dense path (their hash recomputed from offsets[pid] + pos of
    full-width fields in the bucket kernel); without it the batch goes to the general path."""
    k, _, _, _, parity, total, _ = CASES[case]
    res, offs = data(case)
    assert _full_width(offs, k, parity) == 64
    res = res.copy()
    rng = np.random.default_rng(SEEDS[case])
    long0, long_len = int(offs[-2]), int(offs[-1] - offs[-2])
    half = 1 << (_widths(offs)[1] - 1)
    at = np.concatenate([rng.integers(0, long0, size=2000), long0 + rng.integers(half, long_len, size=2000)])
    res[at] = rng.choice(np.frombuffer(b"XUO*", dtype=np.uint8), size=len(at))
    run = long0 + long_len - 5000
    res[run:run + 60] = ord("X")  # one exception k-mer many times
    _env(monkeypatch)
    capfd.readouterr()
    if parity:
        _check(K, O, capfd, res, offs, k, 1, {"parity": 1, "total": total, "unhandled": 0, "exc": 1, "overflow": 0})
    else:
        _check(K, O, capfd, res, offs, k, 0, {"parity": 0, "total": total, "unhandled": 1})


def test_one_handle_across_layouts(K, O, data, monkeypatch, capfd):
    """parity -> clear -> no parity -> clear -> parity on ONE handle: the pattern -> code table is rebuilt at each switch
    (dense_table_parity), and a search of the index without the parity bit answers like the oracle."""
    from kmerseek_b200 import synth
    O = _Kept(O)
    _env(monkeypatch)
    capfd.readouterr()
    with K.ProteomeIndex("db", 24, 1, "hp") as idx:
        for case in ("k24_parity", "k24_no_parity", "k24_parity"):
            parity = CASES[case][4]
            res, offs = data(case)
            assert _full_width(offs, 24, parity) == 64
            prot = K.Proteome.from_packed(res, offs)
            idx.add_proteome(prot)
            _check(K, O, capfd, res, offs, 24, 1, {"eligible": 1, "state": 1, "parity": parity, "total": 12, "unhandled": 0},
                   idx=idx)
            if not parity:
                # planted queries, and one cut from the long protein past position 2^21 (the top bit of the position field)
                qres, qoffs, _ = synth.queries(res, offs, 6, 31, min_len=40, max_len=200)
                a = int(offs[-2]) + 3_000_000
                qres = np.concatenate([qres, res[a:a + 150]])
                qoffs = np.append(qoffs, qoffs[-1] + np.uint64(150))
                r = _search_equals_oracle(K, O, idx, res, offs, qres, qoffs, 24, "hp", 1, hits=True)
                h = r.hits
                assert np.any((h["hit_pid"] == len(offs) - 2) & (h["hit_tpos"] >= 1 << 21))
            idx.clear()
            prot.close()


def test_c2_layout_on_the_pipelined_add(K, O, monkeypatch, capfd):
    """C2's key layout (18 protein bits + 21 position bits: no parity bit) on a batch of more than 2^26 residues, which
    ks_index_add_proteome streams in while the rank kernel runs over the chunks that have landed (Build::DenseRanked)."""
    from kmerseek_b200 import synth
    res, offs = synth.proteome(65_500_000, 20260107)
    long = synth.residues_iid(2**21 - 1, np.random.Generator(np.random.PCG64(20260108)))
    res = np.concatenate([res, long])
    offs = np.append(offs, offs[-1] + np.uint64(len(long)))
    assert len(res) >= 1 << 26
    assert _widths(offs) == (18, 21) and _full_width(offs, 24, 0) == 64  # (the generator may lengthen its last protein)
    _env(monkeypatch)
    capfd.readouterr()
    prot = K.Proteome.from_packed(res, offs)
    with K.ProteomeIndex("db", 24, 1, "hp") as idx:
        idx.add_proteome(prot)
        added = capfd.readouterr().err
        assert BEGIN.search(added) and not FINALIZE.search(added), added  # the rank kernel ran during the add
        st = _csr_equals_oracle(K, O, res, offs, 24, "hp", path=1, idx=idx)
        lay = _layout(added + capfd.readouterr().err)
    assert lay == {"eligible": 1, "state": 1, "rb_full": 10, "parity": 0, "total": 15, "n": st["n_tuples"], "unhandled": 0,
                   "exc": 0, "overflow": 0}, lay
    prot.close()
