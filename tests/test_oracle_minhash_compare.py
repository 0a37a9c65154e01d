"""The numpy reference of the all-pairs sketch comparison (sketch_reference.minhash_compare) against brute force over Python sets:
shared = |A ∩ B| and shared_bottom = |S_s(A ∪ B) ∩ A ∩ B|, S_s = the s smallest values, rows read up to min(length, s)."""
import numpy as np
import pytest

import sketch_reference as ref

ALL = (1 << 64) - 1


def brute(rows_a, rows_b, s):
    shared = np.zeros((len(rows_a), len(rows_b)), dtype=np.uint32)
    bottom = np.zeros_like(shared)
    for i, x in enumerate(rows_a):
        for j, y in enumerate(rows_b):
            x, y = set(x), set(y)
            shared[i, j] = len(x & y)
            smallest = set(sorted(x | y)[:s])
            bottom[i, j] = len(smallest & x & y)
    return shared, bottom


def pack(rows, s, extra_len=0):
    a = np.full((len(rows), s), ALL, dtype=np.uint64)
    n = np.zeros(len(rows), dtype=np.uint32)
    for i, r in enumerate(rows):
        r = sorted(r)[:s]
        a[i, : len(r)] = np.array(r, dtype=np.uint64)
        n[i] = len(r) + (extra_len if len(r) == s else 0)
    return a, n


@pytest.mark.parametrize("s", [1, 2, 5, 17, 64])
def test_oracle_compare_matches_python_sets(s):
    rng = np.random.default_rng(s)
    universe = [int(v) for v in rng.integers(0, 2**64, size=3 * s + 5, dtype=np.uint64)] + [0, ALL]
    universe = sorted(set(universe))
    full = universe[:s]
    rows = [
        [],                                   # empty
        full,                                 # s values
        full,                                 # identical
        universe[s: 2 * s],                   # disjoint from `full`
        full[: max(1, s // 2)],               # nested
        sorted(set(universe[-s:]) | {ALL}),   # ~0 as a real last value
    ]
    for _ in range(12):
        m = int(rng.integers(0, s + 1))
        rows.append(sorted(int(v) for v in rng.choice(np.array(universe, dtype=np.uint64), size=m, replace=False)))
    rows_s = [sorted(r)[:s] for r in rows]
    a, a_n = pack(rows, s)
    b, b_n = pack(rows[::-1], s, extra_len=3)  # a length above s is read as s
    got = ref.minhash_compare(a, a_n, b, b_n, s)
    want = brute(rows_s, rows_s[::-1], s)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    # A against itself: symmetric, the diagonal is every row's length
    sh, bt = ref.minhash_compare(a, a_n, a, a_n, s)
    assert np.array_equal(sh, sh.T) and np.array_equal(bt, bt.T)
    assert np.array_equal(np.diag(sh), [len(r) for r in rows_s]) and np.array_equal(np.diag(bt), np.diag(sh))
