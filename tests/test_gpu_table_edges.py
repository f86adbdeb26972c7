"""-m gpu: the table stages on digests that share long prefixes, and the Merkle root at its level boundaries.

Random content almost never gives two digests that share the 32-bit key the sort orders on, nor index rows that agree
with a chunk's digest in all but a few bytes.  Here every chunk is a 32-byte message of the prefix-twin fixture (a file
shorter than the minimum chunk size is one chunk, digest = SHA-256 of the file), so K3 meets ties of every run length
it treats differently, the index meets rows that differ from a chunk only in one byte of any word, and fixed-size
chunks (min = normal = max = 64) pin the table size to the Merkle level boundaries.  Every session checks the chunk
digests against hashlib in chunk order, and the table and root against tests/table_ref.py."""
import hashlib

import numpy as np
import pytest

from oracle import chunk_delta as cd
from tests.table_ref import msg, near_twins, ref_merkle, ref_table, rows, twins

pytestmark = pytest.mark.gpu

E_INVAL = -1
FIX_SHORT, FIX_LONG_CAP = 64, 8192   # the tie fix-up's run-length split and long-run list size (mksnap_kernels.cuh)
FIXED64 = (64, 64, 64, 16, 12)


@pytest.fixture(scope="module")
def eng():
    from makisu_b200.abi import Engine
    e = Engine(device=0, device_arena_bytes=16 << 20, max_extents=1 << 20)
    yield e
    e.close()


def _extents(offs, lens):
    from makisu_b200.abi import Extent, MKSNAP_X_CDC
    n = len(offs)
    arr = (Extent * n)()
    a = np.frombuffer(arr, dtype=np.uint64).reshape(n, 4)
    a[:, 0] = offs
    a[:, 1] = lens
    a[:, 2] = 0
    a[:, 3] = MKSNAP_X_CDC            # flags (low half), reserved = 0
    return arr


def _check(e, res, want_digests, want_ends):
    """chunk digests and ends in chunk order, n_unique, table and root"""
    assert res.n_chunks == len(want_digests)
    ends, dig = e.get_chunks(res.n_chunks)
    assert dig.tobytes() == b"".join(want_digests)
    np.testing.assert_array_equal(ends, np.asarray(want_ends, dtype=np.uint64))
    tab = ref_table(want_digests)
    assert res.n_unique == len(tab)
    assert e.get_table(res.n_unique).tobytes() == b"".join(tab)
    assert bytes(res.root) == ref_merkle(tab)
    return tab


def _twin_session(e, counters, submits=1):
    """One session whose chunks are msg(c) for c in `counters`, in that order; the arena holds each message once and the
    extents repeat it.  The extents are split evenly over `submits` submits of the same arena."""
    uniq = sorted(set(counters))
    at = {c: 32 * i for i, c in enumerate(uniq)}
    arena = np.frombuffer(b"".join(msg(c) for c in uniq), dtype=np.uint8)
    offs = np.array([at[c] for c in counters], dtype=np.uint64)
    e.begin()
    e.device_upload(0, 0, arena)
    bounds = np.linspace(0, len(offs), submits + 1).astype(int)
    ends = []
    for k, (a, b) in enumerate(zip(bounds[:-1], bounds[1:])):
        e.device_submit(0, arena.size, _extents(offs[a:b], np.full(b - a, 32, np.uint64)))
        ends.append(offs[a:b] + 32 + k * arena.size)      # ends count in the concatenation of the submitted arenas
    res = e.finish()
    dig = {c: hashlib.sha256(msg(c)).digest() for c in uniq}
    tab = _check(e, res, [dig[c] for c in counters], np.concatenate(ends))
    return res, tab, dig


def _runs_of(tab):
    """lengths of the runs of equal 32-bit key in a sorted table"""
    k = np.frombuffer(b"".join(t[:4] for t in tab), dtype=">u4")
    starts = np.flatnonzero(np.r_[True, k[1:] != k[:-1]])
    return np.diff(np.r_[starts, len(k)])


PAIR_COUNTS = [(1, 1), (62, 1), (1, 62), (1, 63), (33, 32), (64, 1)]           # runs of 2, 63, 63, 64, 65, 65 rows
TRIPLE_COUNTS = [(1, 1, 1), (61, 1, 1), (1, 62, 1), (1, 1, 63), (22, 21, 22)]  # runs of 3, 63, 64, 65, 65 rows


def _short_run_counters():
    """pairs and triples, each member repeated so that the group's run has 2, 3, 63, 64 or 65 rows; even groups emit
    their members in ascending digest order, odd groups in descending order, every fifth group interleaved"""
    rng = np.random.default_rng(1)
    out = []
    groups = [(g, PAIR_COUNTS[i % len(PAIR_COUNTS)]) for i, g in enumerate(twins("pairs")[:1500])]
    groups += [(g, TRIPLE_COUNTS[i % len(TRIPLE_COUNTS)]) for i, g in enumerate(twins("triples"))]
    for i, (g, mult) in enumerate(groups):
        seq = [c for (c, _), m in zip(g, mult) for _ in range(m)]
        if i % 2:
            seq = seq[::-1]
        if i % 5 == 4:
            seq = [seq[j] for j in rng.permutation(len(seq))]
        out += seq
    return out


@pytest.mark.parametrize("submits", [1, 2])
def test_short_runs_of_tied_digests(eng, submits):
    res, tab, _ = _twin_session(eng, _short_run_counters(), submits)
    runs = _runs_of(tab)
    assert (runs == 2).sum() >= 1500 and (runs == 3).sum() >= 30      # every group is a run of its distinct members
    assert res.n_chunks - res.n_unique > 50_000


def test_long_runs_of_distinct_digests(eng):
    """runs longer than FIX_SHORT that hold distinct digests: the long-run kernel must sort them (inversions <= 1e5)"""
    p, t = twins("pairs")[2000:2010], twins("triples")
    lo, hi = (lambda g: g[0][0]), (lambda g: g[-1][0])
    counters = ([hi(p[0])] * 1000 + [lo(p[0])]                     # smaller digest last
                + [hi(p[1])] + [lo(p[1])] * 1000                   # larger digest first
                + [lo(p[2])] * 2500 + [hi(p[2])] + [lo(p[2])] * 2500
                + [hi(p[3])] * 200 + [lo(p[3])] * 200              # 40 000 inversions
                + [t[0][2][0]] * 300 + [t[0][0][0]] * 2 + [t[0][1][0]]
                + [t[1][1][0]] * 100 + [t[1][2][0]] * 3 + [t[1][0][0]] * 100
                + [lo(p[4])] * (FIX_SHORT + 1) + [hi(p[4])])       # already in order
    res, tab, _ = _twin_session(eng, counters)
    assert res.n_unique == 5 * 2 + 2 * 3
    _twin_session(eng, counters, submits=2)


def test_more_long_runs_than_the_list_holds(eng):
    """8 400 runs of A x 65 + B x 1, every one out of order: the runs beyond FIX_LONG_CAP are sorted by their own thread"""
    n_runs = 8400
    assert n_runs > FIX_LONG_CAP
    counters = []
    for i, g in enumerate(twins("pairs")[:n_runs]):
        rep, single = (g[0], g[1]) if i % 2 else (g[1], g[0])
        a = [rep[0]] * (FIX_SHORT + 1)
        counters += a + [single[0]] if single[1] < rep[1] else [single[0]] + a   # B after A's if smaller, else before
    res, tab, _ = _twin_session(eng, counters)
    assert res.n_chunks == n_runs * (FIX_SHORT + 2) and res.n_unique == 2 * n_runs
    assert (_runs_of(tab) == 2).sum() == n_runs


def _check_delta(e, ix, res, counters):
    d = e.delta(ix)
    _, dig = e.get_chunks(res.n_chunks)
    st = e.chunk_status(res.n_chunks)
    want = cd.classify(dig, ix.get(e))
    np.testing.assert_array_equal(st, want)
    c = cd.counts(want, np.full(len(counters), 32))
    assert (d.known_chunks, d.new_chunks, d.repeat_chunks) == (c["known_chunks"], c["new_chunks"], c["repeat_chunks"])
    assert (d.known_bytes, d.new_bytes, d.repeat_bytes) == (c["known_bytes"], c["new_bytes"], c["repeat_bytes"])
    assert d.index_rows == ix.rows()
    return st


def test_delta_on_twins(eng):
    """an index of one member of each twin group: the other member is NEW at its first chunk, REPEAT after"""
    from makisu_b200.abi import ChunkIndex
    groups = twins("pairs")[3000:6000] + twins("triples")
    counters, known = [], set()
    for i, g in enumerate(groups):
        a, b = g[i % len(g)][0], g[(i + 1) % len(g)][0]
        known.add(a)
        counters += [b, a, b, a] if i % 2 else [a, b, b]
    res, tab, dig = _twin_session(eng, counters)
    with ChunkIndex(eng, 10_000) as ix:
        ix.add_rows(eng, rows(ref_table([dig[c] for c in known])))
        st = _check_delta(eng, ix, res, counters)
        seen = set()
        for c, s in zip(counters, st):
            assert s == (cd.KNOWN if c in known else cd.REPEAT if c in seen else cd.NEW)
            seen.add(c)


@pytest.mark.parametrize("n_pairs", [4, 6000])
def test_near_twin_index_rows(eng, n_pairs):
    """index rows equal to a chunk's digest except one byte: never a hit; the merge orders them by their tail words;
    strict ascent is checked on all 32 bytes"""
    from makisu_b200.abi import ChunkIndex, MksnapError
    groups = twins("pairs")[:n_pairs]
    counters = [c for g in groups for c, _ in g] + [g[0][0] for g in groups[::2]]
    res, tab, _ = _twin_session(eng, counters)
    nt = near_twins(tab)
    assert len(nt) >= 8 and (n_pairs < 100 or len(nt) >= 100_000)
    subset = tab[::3]
    with ChunkIndex(eng, len(nt) + len(tab) + 64) as ix:
        ix.add_rows(eng, rows(nt))
        assert ix.get(eng).tobytes() == b"".join(nt)
        st = _check_delta(eng, ix, res, counters)
        assert (st != cd.KNOWN).all()
        ix.add_rows(eng, rows(subset))
        assert ix.get(eng).tobytes() == b"".join(ref_table(nt + subset))
        st = _check_delta(eng, ix, res, counters)
        s = set(subset)
        _, dig = eng.get_chunks(res.n_chunks)
        np.testing.assert_array_equal(st == cd.KNOWN, [r.tobytes() in s for r in dig])
        ix.add_table(eng)                                           # merge path: the session table into near twins
        before = ix.get(eng)
        np.testing.assert_array_equal(before, cd.union(rows(nt + subset), rows(tab)))
        assert before.tobytes() == b"".join(ref_table(nt + tab))
        assert (_check_delta(eng, ix, res, counters) == cd.KNOWN).all()
        # a run ascending only in its last byte, and the same run made invalid
        run = [tab[-1][:31] + bytes([k]) for k in range(0, 256, 5)]
        for bad in (run[:10] + [run[11], run[10]] + run[12:], run[:20] + [run[19]] + run[20:],
                    [nt[0], nt[2], nt[1]] + nt[3:40], nt[:30] + [nt[29]] + nt[30:60]):
            with pytest.raises(MksnapError) as ei:
                ix.add_rows(eng, rows(bad))
            assert ei.value.code == E_INVAL
            np.testing.assert_array_equal(ix.get(eng), before)
        ix.add_rows(eng, rows(run))
        np.testing.assert_array_equal(ix.get(eng), rows(ref_table(nt + tab + run)))
    with ChunkIndex(eng, len(run)) as fresh:
        fresh.add_rows(eng, rows(run))
        assert fresh.get(eng).tobytes() == b"".join(run)


MERKLE_U = [1, 2, 255, 256, 257, 511, 512, 513, 65535, 65536, 65537]


@pytest.fixture(scope="module")
def eng64():
    from makisu_b200.abi import CdcParams, Engine
    e = Engine(device=0, device_arena_bytes=16 << 20, max_extents=1 << 12, cdc=CdcParams(*FIXED64))
    yield e
    e.close()


@pytest.mark.parametrize("u", MERKLE_U)
def test_merkle_level_boundaries(eng64, oracle_lib, u):
    """fixed 64-byte chunks of synth_fill content (one seed per file): exactly u distinct chunks, plus a second extent
    over the first file"""
    rng = np.random.default_rng(u)
    sizes = []
    while sum(sizes) < u:
        sizes.append(min(int(rng.integers(1, 700)), u - sum(sizes)))
    offs, pos = [], 0
    for i, k in enumerate(sizes):
        offs.append(pos)
        eng64.synth_fill(0, pos, 64 * k, 0x7000 + i)
        pos += (64 * k + 511) // 512 * 512
    offs.append(offs[0])
    sizes.append(sizes[0])
    eng64.begin()
    eng64.device_submit(0, pos, _extents(offs, [64 * k for k in sizes]))
    res = eng64.finish()
    digests, ends = [], []
    for i, (o, k) in enumerate(zip(offs, sizes)):
        data = oracle_lib.synth_fill(o, 64 * k, 0x7000 + (i if i < len(sizes) - 1 else 0)).tobytes()
        digests += [hashlib.sha256(data[64 * j:64 * j + 64]).digest() for j in range(k)]
        ends += [o + 64 * (j + 1) for j in range(k)]
    tab = _check(eng64, res, digests, ends)
    assert len(tab) == u


def test_merkle_levels_around_2_24(oracle_lib):
    """4096 files of 256 KiB in a 1 GiB arena, 64-byte chunks: 2^24 - 1, 2^24 and 2^24 + 1 distinct chunks (the last
    file shortened or lengthened by one chunk)"""
    from makisu_b200.abi import CdcParams, Engine
    fb, nf = 256 << 10, 4096
    offs = [i * fb for i in range(nf)]
    prm = CdcParams(*FIXED64)
    arena = np.empty((nf - 1) * fb, dtype=np.uint8)
    for i, o in enumerate(offs[:-1]):
        arena[o:o + fb] = oracle_lib.synth_fill(o, fb, i)
    common = oracle_lib.chunk_table(arena, offs[:-1], [fb] * (nf - 1), oracle_lib.CdcParams(*FIXED64))
    del arena
    last_data = oracle_lib.synth_fill(offs[-1], fb + 64, nf - 1).tobytes()
    last_dig = np.frombuffer(b"".join(hashlib.sha256(last_data[j:j + 64]).digest() for j in range(0, fb + 64, 64)),
                             dtype=np.uint8).reshape(-1, 32)
    tv = np.ascontiguousarray(common["table"]).view("V32").ravel()
    with Engine(device=0, device_arena_bytes=nf * fb + 512, max_extents=nf + 16, cdc=prm) as e:
        for i, o in enumerate(offs[:-1]):
            e.synth_fill(0, o, fb, i)
        e.synth_fill(0, offs[-1], fb + 64, nf - 1)
        for last in (fb - 64, fb, fb + 64):
            e.begin()
            e.device_submit(0, nf * fb + 64, _extents(offs, [fb] * (nf - 1) + [last]))
            res = e.finish()
            k = last // 64
            assert res.n_chunks == (1 << 24) + k - fb // 64
            ends, dig = e.get_chunks(res.n_chunks)
            n0 = common["n_chunks"]
            np.testing.assert_array_equal(dig[:n0], common["digests"])
            np.testing.assert_array_equal(dig[n0:], last_dig[:k])
            np.testing.assert_array_equal(ends[:n0], common["ends"])
            np.testing.assert_array_equal(ends[n0:], offs[-1] + 64 * np.arange(1, k + 1, dtype=np.uint64))
            lv = np.sort(np.ascontiguousarray(last_dig[:k]).view("V32").ravel())
            table = np.insert(tv, np.searchsorted(tv, lv), lv).view(np.uint8).reshape(-1, 32)
            assert res.n_unique == len(table) == res.n_chunks
            np.testing.assert_array_equal(e.get_table(res.n_unique), table)
            assert bytes(res.root) == oracle_lib.merkle_root(table)


def test_world_of_one_allgather_on_twins():
    from makisu_b200.abi import Engine
    with Engine(device=0, device_arena_bytes=16 << 20, max_extents=1 << 16) as e:
        e.comm_init(Engine.comm_unique_id(), 1, 0)
        counters = _short_run_counters()[:20_000]
        res, tab, _ = _twin_session(e, counters)
        g = e.allgather_tables()
        assert (g.n_chunks, g.n_unique, bytes(g.root)) == (res.n_chunks, len(tab), ref_merkle(tab))
        assert e.get_table(g.n_unique).tobytes() == b"".join(tab)
