"""The chunk-delta oracle (oracle/chunk_delta.py) against a brute-force restatement with Python sets and lists.

The GPU tests check the engine's statuses, counts and index rows against this oracle, so the oracle itself is pinned
here on the CPU: duplicates, empty inputs, rows that share their 64-bit prefix (the K3 key) and rows at the ends of
the order (prefixes 00.. and ff..).
"""
import numpy as np
import pytest

from oracle import chunk_delta as cd


def _brute_classify(digests, index_rows):
    idx = {bytes(r) for r in index_rows}
    seen, out = set(), []
    for d in digests:
        b = bytes(d)
        if b in idx:
            out.append(0)
        elif b in seen:
            out.append(2)
        else:
            out.append(1)
            seen.add(b)
    return np.array(out, dtype=np.uint8)


def _brute_union(a, b):
    rows = sorted({bytes(r) for r in a} | {bytes(r) for r in b})
    return np.frombuffer(b"".join(rows), dtype=np.uint8).reshape(-1, 32)


def _digests(rng, n, pool=None, prefix_share=0, edges=False):
    """n digests; drawn with repetition from `pool` distinct ones if given; `prefix_share` of the distinct digests get
    one common 64-bit prefix; `edges` puts some at prefix 00.. and ff.."""
    k = pool or n
    base = rng.integers(0, 256, (max(k, 1), 32), dtype=np.uint8)
    if prefix_share:
        base[:prefix_share, :8] = base[0, :8]
    if edges and k >= 4:
        base[0, :8] = 0
        base[1, :] = 0
        base[2, :8] = 0xFF
        base[3, :] = 0xFF
    if pool:
        return base[rng.integers(0, k, n)] if n else base[:0]
    return base[:n]


def _sorted_unique(rows):
    return _brute_union(rows, rows[:0])


CASES = [
    dict(n=0, pool=None, ix=0),
    dict(n=1, pool=None, ix=0),
    dict(n=300, pool=None, ix=0),
    dict(n=500, pool=40, ix=0),                          # duplicates only
    dict(n=500, pool=40, ix=20),                          # index drawn from the same pool
    dict(n=800, pool=200, ix=100, prefix_share=60),       # 60 digests with one 64-bit prefix
    dict(n=800, pool=200, ix=100, edges=True),            # 00.. and ff.. prefixes
    dict(n=0, pool=None, ix=50),                          # empty session, non-empty index
    dict(n=1000, pool=1000, ix=300, prefix_share=300, edges=True),
]


@pytest.mark.parametrize("case", range(len(CASES)))
def test_classify_matches_brute_force(case):
    c = CASES[case]
    rng = np.random.default_rng(100 + case)
    dig = _digests(rng, c["n"], c["pool"], c.get("prefix_share", 0), c.get("edges", False))
    # index: some of the session's digests plus unrelated rows (with the same prefix games)
    own = dig[rng.permutation(len(dig))[: c["ix"] // 2]] if len(dig) else dig[:0]
    other = _digests(rng, c["ix"] - len(own), None, c.get("prefix_share", 0) // 2, c.get("edges", False))
    index_rows = _sorted_unique(np.concatenate([own, other]))
    got = cd.classify(dig, index_rows)
    want = _brute_classify(dig, index_rows)
    np.testing.assert_array_equal(got, want)
    # invariants of the delta result
    n_unique = len({bytes(d) for d in dig})
    known_unique = len({bytes(d) for d in dig} & {bytes(r) for r in index_rows})
    assert (got == cd.NEW).sum() == n_unique - known_unique
    assert (got == cd.KNOWN).sum() + (got == cd.NEW).sum() + (got == cd.REPEAT).sum() == len(dig)
    lens = rng.integers(1, 100000, len(dig)).astype(np.uint64)
    cnt = cd.counts(got, lens)
    assert cnt["known_bytes"] + cnt["new_bytes"] + cnt["repeat_bytes"] == int(lens.sum())
    assert cnt["new_chunks"] == n_unique - known_unique


@pytest.mark.parametrize("case", range(len(CASES)))
def test_union_matches_brute_force(case):
    c = CASES[case]
    rng = np.random.default_rng(200 + case)
    a = _sorted_unique(_digests(rng, c["n"], c["pool"], c.get("prefix_share", 0), c.get("edges", False)))
    b = _digests(rng, c["ix"], None, c.get("prefix_share", 0), c.get("edges", False))
    if len(a):
        b = np.concatenate([b, a[: len(a) // 3]])           # overlap
    b = _sorted_unique(b)
    got = cd.union(a, b)
    np.testing.assert_array_equal(got, _brute_union(a, b))
    np.testing.assert_array_equal(cd.union(b, a), got)
    np.testing.assert_array_equal(cd.union(got, got), got)
    assert cd.union(a[:0], a[:0]).shape == (0, 32)


def test_contains_and_chunk_lens():
    rng = np.random.default_rng(7)
    rows = _sorted_unique(_digests(rng, 100, edges=True))
    probe = np.concatenate([rows[::3], _digests(rng, 20)])
    want = np.array([bytes(p) in {bytes(r) for r in rows} for p in probe])
    np.testing.assert_array_equal(cd.contains(rows, probe), want)
    assert cd.contains(rows[:0], probe).sum() == 0
    # files at 0 (1000 B, chunks end 400, 1000), 1024 (0 B), 1024 (600 B, one chunk), 2048 (5000 B, ends 4048, 7048)
    ends = np.array([400, 1000, 1624, 6048, 7048], dtype=np.uint64)
    np.testing.assert_array_equal(cd.chunk_lens(ends, [0, 1024, 1024, 2048], [1000, 0, 600, 5000]),
                                  [400, 600, 600, 4000, 1000])
