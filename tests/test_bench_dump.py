"""bench.py --dump-outputs on the host: how one result table becomes float64 arrays (CPU only)."""
import hashlib

import numpy as np

import bench


def test_small_table_is_dumped_whole_and_exact():
    keys = np.array([0, 1, 2**53 + 1, 2**64 - 1], dtype=np.uint64)
    pid = np.array([7, 0, 3, 2**32 - 1], dtype=np.uint32)
    score = np.array([0.1, 1.0, 1e-300, 0.3333333333333333])
    out = bench.dump_columns("t_", {"hash": keys, "pid": pid, "score": score})
    assert sorted(out) == ["t_hash_hi", "t_hash_lo", "t_hash_sha256", "t_pid", "t_pid_sha256", "t_score"]
    assert all(a.dtype == np.float64 for a in out.values())
    back = (out["t_hash_hi"].astype(np.uint64) << np.uint64(32)) | out["t_hash_lo"].astype(np.uint64)
    assert np.array_equal(back, keys)  # a float64 alone would round 2^53 + 1 and 2^64 - 1
    assert np.array_equal(out["t_pid"], pid) and np.array_equal(out["t_score"], score)
    words = np.frombuffer(hashlib.sha256(pid.tobytes()).digest(), dtype="<u4")
    assert np.array_equal(out["t_pid_sha256"], words)


def test_large_table_is_sampled_by_the_same_seeded_rows():
    n = bench.DUMP_ROWS * 5 + 3
    rng = np.random.default_rng(1)
    pid = rng.integers(0, 2**32, size=n, dtype=np.uint64).astype(np.uint32)
    pos = np.arange(n, dtype=np.uint32)
    a = bench.dump_columns("p_", {"pid": pid, "pos": pos})
    b = bench.dump_columns("p_", {"pid": pid.copy(), "pos": pos.copy()})
    assert all(np.array_equal(a[k], b[k]) for k in a)  # same input, same files
    assert len(a["p_pos"]) == len(a["p_pid"]) == bench.DUMP_ROWS
    rows = a["p_pos"].astype(np.int64)  # pos is the row number: the sample is sorted and has no repeats
    assert np.all(rows[1:] > rows[:-1]) and rows[-1] < n
    assert np.array_equal(a["p_pid"], pid[rows])  # every column keeps the same rows
    changed = pid.copy()
    changed[np.setdiff1d(np.arange(n), rows)[0]] ^= 1  # a row outside the sample
    c = bench.dump_columns("p_", {"pid": changed, "pos": pos})
    assert np.array_equal(c["p_pid"], a["p_pid"]) and not np.array_equal(c["p_pid_sha256"], a["p_pid_sha256"])


def test_largest_dump_stays_under_64_mb(tmp_path):
    """Two indexes, a pair table and a hit table, each longer than the sample, written as bench.py writes them."""
    from kmerseek_b200.search import HIT_COLUMNS, PAIR_INT_COLUMNS
    from kmerseek_b200._ffi import SCORE_COLUMNS
    n = bench.DUMP_ROWS + 1

    class Index:
        def csr(self):
            return (np.arange(n, dtype=np.uint64), np.arange(n + 1, dtype=np.uint64), np.zeros(2 * n, np.uint32),
                    np.ones(2 * n, np.uint32))

    pairs = {c: np.zeros(n, dtype=t) for c, t in PAIR_INT_COLUMNS.items()}
    pairs.update({c: np.zeros(n) for c in SCORE_COLUMNS})
    hits = {c: np.zeros(n, dtype=t) for c, t in HIT_COLUMNS.items()}
    dump = {**bench.dump_index("index_", Index()), **bench.dump_columns("search_", pairs),
            **bench.dump_columns("search_", hits), **bench.dump_index("target_index_", Index())}
    bench.write_dump(str(tmp_path / "out"), dump)
    files = list((tmp_path / "out").iterdir())
    assert len(files) == len(dump) and all(f.suffix == ".npy" for f in files)
    assert all(np.load(f).dtype == np.float64 for f in files)
    assert sum(f.stat().st_size for f in files) <= 64 << 20
