"""bench.py --dump-outputs: the sample of the timed path's rows and the per-piece fingerprints, checked on made-up rows. CPU only."""
import numpy as np

import bench
from modkit_b200 import ROW_DTYPE


def made_up_rows(n, start, seed):
    rng = np.random.default_rng(seed)
    r = np.zeros(n, dtype=ROW_DTYPE)
    r["pos"] = start + np.sort(rng.choice(50_000_000, n, replace=False))
    r["code"] = rng.choice([ord("h"), ord("m"), 0x80000000 | 76792], n)
    r["strand"] = rng.choice([ord("+"), ord("-")], n)
    r["primary_base"] = rng.integers(0, 4, n)
    for f in bench.ROW_FIELDS[4:]:
        r[f] = rng.integers(0, 60, n)
    return r


def test_dump_is_seeded_exact_and_bounded():
    pieces = [(0, 0, 50_000_000), (1, 0, 100_000), (1, 200_000_000, 250_000_000)]
    rows = [made_up_rows(3000, 0, 1), made_up_rows(0, 0, 2), made_up_rows(5000, 200_000_000, 3)]
    a = bench.output_arrays(pieces, rows, 1000, 7)
    b = bench.output_arrays(pieces, [r.copy() for r in rows], 1000, 7)
    assert sorted(a) == sorted(b) and all(np.array_equal(a[k], b[k]) for k in a)
    assert all(v.dtype == np.float64 for v in a.values())
    # the sample: rows of the concatenated output, in order, every field exact (positions beyond float32's integers)
    flat = np.concatenate(rows)
    idx = a["rows_index"].astype(np.int64)
    assert len(idx) == 1000 and (np.diff(idx) > 0).all() and idx[-1] >= 3000
    for f in bench.ROW_FIELDS:
        assert np.array_equal(a["rows_" + f], flat[f][idx].astype(np.float64)), f
    assert np.array_equal(a["rows_contig"], np.where(idx < 3000, 0, 1))
    assert a["pieces"].tolist() == [list(p) for p in pieces] and a["piece_rows"].tolist() == [3000, 0, 5000]
    # a change to one count of one row outside the sample shows in that piece's checksum only
    k = next(i for i in range(5000) if 3000 + i not in set(idx.tolist()))
    rows[2]["n_nocall"][k] += 1
    c = bench.output_arrays(pieces, rows, 1000, 7)
    assert c["piece_crc32"][2] != a["piece_crc32"][2] and c["piece_crc32"][0] == a["piece_crc32"][0]
    assert all(np.array_equal(c[k], a[k]) for k in a if k.startswith("rows_"))
    # fewer rows than the sample size: all of them
    d = bench.output_arrays(pieces[:1], rows[:1], 10_000, 7)
    assert d["rows_index"].tolist() == list(range(3000))


def test_dump_stays_within_64_mb():
    n = bench.DUMP_ROWS + 12345
    rows = [made_up_rows(n // 2, 0, 4), made_up_rows(n - n // 2, 60_000_000, 5)]
    a = bench.output_arrays([(0, 0, 60_000_000), (0, 60_000_000, 120_000_000)], rows, bench.DUMP_ROWS, 1)
    assert len(a["rows_index"]) == bench.DUMP_ROWS
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
