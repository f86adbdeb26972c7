"""The grouped-session reference (tests/chunk_groups_ref.py) against a literal restatement of its definition: the
sequential per-layer flow "for g in 0..G-1: classify the chunks of group g against the index, then add group g's table
to the index", written with oracle/chunk_delta.py's classify and union.  The GPU tests check the engine's grouped
statuses, counts and group tables against this reference."""
import numpy as np
import pytest

from oracle import chunk_delta as cd
from tests import chunk_groups_ref as gr


def _sequential(digests, groups, index_rows, n_groups):
    """Statuses and per-group tables of the sequential flow; the index the flow ends with."""
    d = np.ascontiguousarray(digests, dtype=np.uint8).reshape(-1, 32)
    g = np.asarray(groups)
    status = np.zeros(len(d), dtype=np.uint8)
    ix = np.ascontiguousarray(index_rows, dtype=np.uint8).reshape(-1, 32)
    tables = []
    for k in range(n_groups):
        sel = np.flatnonzero(g == k)
        status[sel] = cd.classify(d[sel], ix)
        table = cd.union(d[sel][:0], d[sel])
        tables.append(table)
        ix = cd.union(ix, table)
    return status, tables, ix


def _digests(rng, n, pool):
    base = rng.integers(0, 256, (max(pool, 1), 32), dtype=np.uint8)
    base[: pool // 4, :8] = base[0, :8]                   # a quarter of the pool shares one 64-bit prefix
    return base[rng.integers(0, pool, n)] if n else base[:0]


def _index(rng, dig, n_own, n_other):
    own = dig[rng.permutation(len(dig))[:n_own]] if len(dig) else dig[:0]
    other = rng.integers(0, 256, (n_other, 32), dtype=np.uint8)
    return cd.union(own, other)


def _check(dig, groups, index_rows, n_groups):
    want_status, want_tables, _ = _sequential(dig, groups, index_rows, n_groups)
    got = gr.classify_groups(dig, groups, index_rows)
    np.testing.assert_array_equal(got, want_status)
    tables = gr.group_tables(dig, groups, n_groups)
    assert len(tables) == n_groups
    for t, w in zip(tables, want_tables):
        np.testing.assert_array_equal(t, w)
    return got


@pytest.mark.parametrize("seed,n,pool,G,ix_own,ix_other", [
    (1, 600, 150, 5, 20, 30),
    (2, 2000, 300, 17, 0, 0),
    (3, 2000, 2000, 3, 100, 100),                         # almost no repeats
    (4, 1500, 40, 9, 5, 10),                              # heavy repeats across groups
    (5, 0, 10, 4, 0, 10),                                 # no chunks at all
])
def test_random_groups(seed, n, pool, G, ix_own, ix_other):
    rng = np.random.default_rng(seed)
    dig = _digests(rng, n, pool)
    groups = rng.integers(0, G, n)
    _check(dig, groups, _index(rng, dig, ix_own, ix_other), G)


def test_digest_first_seen_in_a_later_group():
    rng = np.random.default_rng(11)
    a, b, c = rng.integers(0, 256, (3, 32), dtype=np.uint8)
    # positions:      0  1  2  3  4  5   groups: 2 1 2 0 1 0
    dig = np.stack([a, b, a, c, a, b])
    groups = np.array([2, 1, 2, 0, 1, 0])
    got = _check(dig, groups, np.zeros((0, 32), np.uint8), 3)
    # c: NEW in group 0.  b: NEW at 5 (group 0), KNOWN at 1 (group 1 > 0).  a: NEW at 4 (group 1, its lowest group),
    # KNOWN at 0 and 2 (group 2)
    np.testing.assert_array_equal(got, [cd.KNOWN, cd.KNOWN, cd.KNOWN, cd.NEW, cd.NEW, cd.NEW])
    # the same digest twice in its lowest group: the lower position is NEW
    got = _check(np.stack([a, a, a]), np.array([1, 0, 0]), np.zeros((0, 32), np.uint8), 2)
    np.testing.assert_array_equal(got, [cd.KNOWN, cd.NEW, cd.REPEAT])


def test_empty_groups():
    rng = np.random.default_rng(12)
    dig = _digests(rng, 400, 100)
    groups = rng.choice([1, 4, 6], 400)                   # groups 0, 2, 3, 5, 7 hold nothing
    _check(dig, groups, _index(rng, dig, 10, 10), 8)
    tables = gr.group_tables(dig, groups, 8)
    assert [len(tables[k]) for k in (0, 2, 3, 5, 7)] == [0] * 5


def test_one_group_is_the_plain_delta():
    rng = np.random.default_rng(13)
    dig = _digests(rng, 900, 200)
    ix = _index(rng, dig, 30, 30)
    got = _check(dig, np.zeros(900, dtype=np.int64), ix, 1)
    np.testing.assert_array_equal(got, cd.classify(dig, ix))
    np.testing.assert_array_equal(gr.group_tables(dig, np.zeros(900), 1)[0], cd.union(dig[:0], dig))


def test_every_chunk_in_one_group_of_many():
    rng = np.random.default_rng(14)
    dig = _digests(rng, 700, 150)
    ix = _index(rng, dig, 25, 25)
    got = _check(dig, np.full(700, 3), ix, 6)
    np.testing.assert_array_equal(got, cd.classify(dig, ix))


def test_counts_sum_to_the_batch():
    rng = np.random.default_rng(15)
    dig = _digests(rng, 1200, 250)
    groups = rng.integers(0, 7, 1200)
    st = gr.classify_groups(dig, groups, np.zeros((0, 32), np.uint8))
    lens = rng.integers(1, 1 << 17, 1200).astype(np.uint64)
    tot = cd.counts(st, lens)
    per = [cd.counts(st[groups == k], lens[groups == k]) for k in range(7)]
    for key in tot:
        assert sum(p[key] for p in per) == tot[key]
    # NEW over all groups = distinct digests of the batch (each is new exactly once, in its lowest group)
    assert tot["new_chunks"] == len({bytes(r) for r in dig})
