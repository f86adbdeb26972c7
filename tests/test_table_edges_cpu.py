"""The plain references of tests/table_ref.py, the prefix-twin fixture, and oracle/chunk_delta.py on rows that share long
prefixes.  ref_table / ref_merkle are pinned here against oracle/mkoracle.c at every Merkle level boundary up to three
levels, so the GPU tests of tests/test_gpu_table_edges.py can use either."""
import hashlib

import numpy as np
import pytest

from oracle import chunk_delta as cd
from tests.table_ref import NEAR_TWIN_BYTES, TWINS_PATH, msg, near_twins, ref_merkle, ref_table, rows, twins


def _twin_digests():
    return [d for kind in ("pairs", "triples") for g in twins(kind) for _, d in g]


def test_fixture_groups_share_32_bits_and_differ_after_them():
    import json
    with open(TWINS_PATH) as f:
        fx = json.load(f)
    assert len(fx["tag"].encode("ascii")) == 24 and fx["bound"] == 1 << 24
    assert len(fx["pairs"]) >= 8500 and len(fx["triples"]) >= 30
    seen = set()
    for kind, size in (("pairs", 2), ("triples", 3)):
        for g in fx[kind]:
            assert len(g) >= size and len(set(g)) == len(g)
            assert all(0 <= c < fx["bound"] for c in g)
            assert seen.isdisjoint(g)
            seen.update(g)
            ds = [hashlib.sha256(fx["tag"].encode("ascii") + c.to_bytes(8, "little")).digest() for c in g]
            assert len(msg(g[0])) == 32 and hashlib.sha256(msg(g[0])).digest() == ds[0]
            assert len({d[:4] for d in ds}) == 1, g
            assert len(set(ds)) == len(ds), g
    # twins() returns each group in ascending digest order
    for g in twins("triples"):
        assert [d for _, d in g] == sorted(d for _, d in g)


@pytest.mark.parametrize("u", [0, 1, 2, 255, 256, 257, 511, 512, 513, 65535, 65536, 65537])
def test_ref_table_and_merkle_against_the_c_oracle(oracle_lib, u):
    rng = np.random.default_rng(u)
    uniq = rng.integers(0, 256, (u, 32), dtype=np.uint8)
    dup = uniq[rng.integers(0, max(u, 1), u // 3)] if u else uniq
    digests = np.concatenate([uniq, dup])[rng.permutation(u + len(dup))]
    tab = ref_table(digests)
    assert len(tab) == u
    c_tab = oracle_lib.sort_unique(digests)
    assert c_tab.tobytes() == b"".join(tab)
    assert ref_merkle(tab) == oracle_lib.merkle_root(c_tab)
    if u == 0:
        assert ref_merkle(tab) == hashlib.sha256(b"").digest()
    if u == 1:
        assert ref_merkle(tab) == hashlib.sha256(tab[0]).digest()


def test_ref_table_and_merkle_on_twin_sets(oracle_lib):
    d = _twin_digests()
    rng = np.random.default_rng(11)
    for n in (2, 3, 257, 5000, len(d)):
        part = [d[i] for i in rng.permutation(len(d))[:n]]
        rep = part + part[: n // 2]                                  # duplicates of some of them
        tab = ref_table(rep)
        assert len(tab) == n
        c_tab = oracle_lib.sort_unique(rows(rep))
        assert c_tab.tobytes() == b"".join(tab)
        assert ref_merkle(tab) == oracle_lib.merkle_root(c_tab)
    pre = [r[:4] for r in ref_table(d)]
    assert sum(a == b for a, b in zip(pre, pre[1:])) >= 8500        # ties on the 32-bit key, adjacent in the table


def _classify_by_sets(chunks, index):
    ix, seen, out = set(index), set(), []
    for c in chunks:
        out.append(cd.KNOWN if c in ix else (cd.REPEAT if c in seen else cd.NEW))
        seen.add(c)
    return np.array(out, dtype=np.uint8)


@pytest.mark.parametrize("n_pairs", [3, 2000])
def test_chunk_delta_oracle_on_near_twin_rows(n_pairs):
    groups = twins("pairs")[:n_pairs] + twins("triples")[:2]
    table = ref_table([d for g in groups for _, d in g])
    nt = near_twins(table)
    assert len(nt) > 15 * len(table)
    t0 = table[0]
    for j in NEAR_TWIN_BYTES:                                       # both neighbours of t0 at each position
        both = {bytes(t0[:j]) + bytes([(t0[j] + d) & 0xFF]) + t0[j + 1:] for d in (1, 255)}
        assert both <= set(nt) and t0 not in set(nt)
    rng = np.random.default_rng(n_pairs)
    chunks = [table[i] for i in rng.integers(0, len(table), 3 * len(table))] + [nt[0]]
    subset = table[::3]
    for index in (nt, ref_table(nt + subset), ref_table(nt + table), []):
        got_u = cd.union(rows(index) if index else np.zeros((0, 32), np.uint8), rows(table))
        assert got_u.tobytes() == b"".join(ref_table(index + table))
        got_c = cd.contains(rows(index) if index else np.zeros((0, 32), np.uint8), rows(chunks))
        in_index = set(index)
        assert got_c.tolist() == [c in in_index for c in chunks]
        st = cd.classify(rows(chunks), rows(index) if index else np.zeros((0, 32), np.uint8))
        np.testing.assert_array_equal(st, _classify_by_sets(chunks, index))
        c = cd.counts(st, [32] * len(chunks))
        assert c["known_chunks"] + c["new_chunks"] + c["repeat_chunks"] == len(chunks)
        assert c["new_chunks"] == len(set(chunks) - set(index))
    assert not cd.classify(rows(table), rows(nt)).__eq__(cd.KNOWN).any()
    assert cd.classify(rows([nt[0]]), rows(nt)).tolist() == [cd.KNOWN]
