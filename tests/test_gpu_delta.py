"""-m gpu: the chunk index and the chunk delta (mksnap_index_* / mksnap_delta) against oracle/chunk_delta.py.

Every status vector, count and index row set is compared bit-exact with the oracle, which consumes the engine's own
get_chunks digests (pinned to oracle/mkoracle.c by test_gpu_parity.py; at small sizes they are re-checked here).
"""
import io
import os
import tarfile

import numpy as np
import pytest

from oracle import chunk_delta as cd
from tests.util import pack, cdc_extents

pytestmark = pytest.mark.gpu

E_INVAL, E_CAPACITY, E_STATE = -1, -4, -5


@pytest.fixture(scope="module")
def eng():
    from makisu_b200.abi import Engine
    e = Engine(device=0, device_arena_bytes=64 << 20, n_host_arenas=2, host_arena_bytes=16 << 20, max_extents=1 << 14)
    yield e
    e.close()


def _rand(rng, n):
    return rng.integers(0, 256, n, dtype=np.uint8)


def _session(e, segs):
    arena, offs = pack(segs)
    lens = [len(s) for s in segs]
    e.begin()
    e.device_upload(0, 0, arena)
    e.device_submit(0, arena.size, cdc_extents(offs, lens))
    res = e.finish()
    return res, arena, offs, lens


def _sorted_rows(rng, n, top=None):
    r = _rand(rng, n * 32).reshape(n, 32)
    if top is not None:
        r[:, :3] = top
    return cd.union(r[:0], r)


def _check_delta(e, ix, res, lens_of_chunks=None):
    """delta against the oracle; returns (delta result, statuses, digests)"""
    index_rows = ix.get(e)
    d = e.delta(ix)
    ends, dig = e.get_chunks(res.n_chunks)
    st = e.chunk_status(res.n_chunks)
    want = cd.classify(dig, index_rows)
    np.testing.assert_array_equal(st, want)
    assert d.index_rows == len(index_rows)
    assert d.known_chunks + d.new_chunks + d.repeat_chunks == res.n_chunks
    assert d.known_bytes + d.new_bytes + d.repeat_bytes == res.cdc_bytes
    n_known_unique = int(cd.contains(index_rows, e.get_table(res.n_unique)).sum())
    assert d.new_chunks == res.n_unique - n_known_unique
    assert (d.known_chunks, d.new_chunks, d.repeat_chunks) == tuple(int((want == k).sum()) for k in (0, 1, 2))
    if lens_of_chunks is not None:
        c = cd.counts(want, lens_of_chunks)
        assert (d.known_bytes, d.new_bytes, d.repeat_bytes) == (c["known_bytes"], c["new_bytes"], c["repeat_bytes"])
    return d, st, dig


def _mixed(rng):
    blob = _rand(rng, 400_000)
    return [_rand(rng, 300_000), blob, np.zeros(700_000, dtype=np.uint8), _rand(rng, 5), blob.copy(),
            np.tile(_rand(rng, 37), 20000), np.zeros(300_000, dtype=np.uint8), _rand(rng, 131_072 * 2), b"", blob[:200_000]]


def test_delta_against_empty_index(eng, oracle_lib):
    from makisu_b200.abi import ChunkIndex
    rng = np.random.default_rng(1)
    segs = _mixed(rng)
    res, arena, offs, lens = _session(eng, segs)
    want = oracle_lib.chunk_table(arena, offs, lens)
    with ChunkIndex(eng, 1000) as ix:
        d, st, dig = _check_delta(eng, ix, res)
        ends, _ = eng.get_chunks(res.n_chunks)
        np.testing.assert_array_equal(dig, want["digests"])
        np.testing.assert_array_equal(ends, want["ends"])
        lens_c = cd.chunk_lens(ends, offs, lens)
        _check_delta(eng, ix, res, lens_c)
        assert d.known_chunks == 0 and d.new_chunks == res.n_unique
        assert d.repeat_chunks == res.n_chunks - res.n_unique > 0
        assert d.new_bytes + d.repeat_bytes == res.cdc_bytes == sum(lens)


def _edit(rng, segs):
    """B from A: edited bytes, an insertion, deleted files, duplicated files, new files"""
    b = [s.copy() if isinstance(s, np.ndarray) else np.frombuffer(bytes(s), dtype=np.uint8).copy() for s in segs]
    b[0][150_000] ^= 0xFF
    b[1] = np.concatenate([b[1][:100_000], _rand(rng, 777), b[1][100_000:]])
    del b[3]
    b.append(b[2].copy())
    b.append(_rand(rng, 250_000))
    b.insert(1, b[5].copy())
    return b


def test_delta_after_edits_and_against_itself(eng, oracle_lib):
    from makisu_b200.abi import ChunkIndex
    rng = np.random.default_rng(2)
    a_segs = [_rand(rng, int(n)) for n in rng.integers(1000, 600_000, 24)] + _mixed(rng)
    res_a, *_ = _session(eng, a_segs)
    with ChunkIndex(eng, 100_000) as ix:
        ix.add_table(eng)
        np.testing.assert_array_equal(ix.get(eng), eng.get_table(res_a.n_unique))
        b_segs = _edit(rng, a_segs)
        res_b, arena, offs, lens = _session(eng, b_segs)
        want = oracle_lib.chunk_table(arena, offs, lens)
        d, st, dig = _check_delta(eng, ix, res_b)
        np.testing.assert_array_equal(dig, want["digests"])
        assert d.known_chunks > 0 and d.new_chunks > 0
        ends, _ = eng.get_chunks(res_b.n_chunks)
        _check_delta(eng, ix, res_b, cd.chunk_lens(ends, offs, lens))
    with ChunkIndex(eng, 100_000) as ix2:          # B against its own table: everything is known
        ix2.add_table(eng)
        d2, st2, _ = _check_delta(eng, ix2, res_b)
        assert d2.known_chunks == res_b.n_chunks and d2.known_bytes == res_b.cdc_bytes and not st2.any()


@pytest.mark.parametrize("n", [0, 1, 255, 256, 257, 1 << 20])
def test_union_sizes_overlap_and_round_trip(eng, n):
    from makisu_b200.abi import ChunkIndex
    rng = np.random.default_rng(n + 3)
    a = _sorted_rows(rng, n)
    b = cd.union(_sorted_rows(rng, n // 2 + 1), a[::2])          # overlaps a
    with ChunkIndex(eng, 2 * n + 8) as ix:
        ix.add_rows(eng, a)
        assert ix.rows() == len(a)
        np.testing.assert_array_equal(ix.get(eng), a)
        ix.add_rows(eng, b)
        want = cd.union(a, b)
        got = ix.get(eng)
        np.testing.assert_array_equal(got, want)
        ix.add_rows(eng, a)                                     # nothing novel
        np.testing.assert_array_equal(ix.get(eng), want)
        with ChunkIndex(eng, len(got)) as fresh:                # persisted form: get -> add_rows
            fresh.add_rows(eng, got)
            np.testing.assert_array_equal(fresh.get(eng), got)


def test_union_and_lookup_of_a_skewed_table(eng, oracle_lib):
    """every row shares its top 24 bits: one directory bucket holds the whole table"""
    from makisu_b200.abi import ChunkIndex
    rng = np.random.default_rng(4)
    skew = _sorted_rows(rng, 5000, top=[0x12, 0x34, 0x56])
    res, *_ = _session(eng, [_rand(rng, 200_000), _rand(rng, 90_000)])
    _, dig = eng.get_chunks(res.n_chunks)
    mixed = cd.union(skew, dig[::2])
    with ChunkIndex(eng, 20_000) as ix:
        ix.add_rows(eng, skew[::2])
        ix.add_rows(eng, mixed)
        np.testing.assert_array_equal(ix.get(eng), cd.union(skew[::2], mixed))
        _check_delta(eng, ix, res)


def test_rejections_leave_the_index_unchanged(eng):
    from makisu_b200.abi import ChunkIndex, MksnapError
    rng = np.random.default_rng(5)
    a = _sorted_rows(rng, 600)
    with ChunkIndex(eng, 1000) as ix:
        ix.add_rows(eng, a)
        before = ix.get(eng)
        bad = [a[::-1][:10], np.concatenate([a[:5], a[4:6]]), np.concatenate([a[100:110], a[50:60]])]
        fresh = _sorted_rows(rng, 50)
        bad.append(cd.union(fresh, fresh)[np.r_[0:20, 20, 20, 21:50]])   # one duplicate row
        for rows in bad:
            with pytest.raises(MksnapError) as ei:
                ix.add_rows(eng, rows)
            assert ei.value.code == E_INVAL
            np.testing.assert_array_equal(ix.get(eng), before)
        over = _sorted_rows(rng, 401)                               # 600 + 401 > 1000
        with pytest.raises(MksnapError) as ei:
            ix.add_rows(eng, over)
        assert ei.value.code == E_CAPACITY
        np.testing.assert_array_equal(ix.get(eng), before)
        with pytest.raises(MksnapError) as ei:
            ix.add_rows(eng, _sorted_rows(rng, 1001))
        assert ei.value.code == E_CAPACITY
        fits = cd.union(a[:450], _sorted_rows(rng, 400))            # 600 + 850 > 1000, but the union is 1000
        ix.add_rows(eng, fits)
        assert ix.rows() == 1000
        np.testing.assert_array_equal(ix.get(eng), cd.union(a, fits))
        # a session table whose union would not fit
        res, *_ = _session(eng, [_rand(rng, 2_000_000)])
        full = ix.get(eng)
        with pytest.raises(MksnapError) as ei:
            ix.add_table(eng)
        assert ei.value.code == E_CAPACITY
        np.testing.assert_array_equal(ix.get(eng), full)
    with ChunkIndex(eng, 10) as small:                              # the session table alone exceeds the capacity
        small.add_rows(eng, a[:3])
        with pytest.raises(MksnapError) as ei:
            small.add_table(eng)
        assert ei.value.code == E_CAPACITY
        np.testing.assert_array_equal(small.get(eng), a[:3])


def test_state_rules(eng):
    from makisu_b200.abi import ChunkIndex, Engine, MksnapError
    rng = np.random.default_rng(6)
    segs = [_rand(rng, 500_000), _rand(rng, 300_000)]
    with ChunkIndex(eng, 10_000) as ix:
        eng.begin()
        with pytest.raises(MksnapError) as ei:
            eng.delta(ix)
        assert ei.value.code == E_STATE
        with pytest.raises(MksnapError) as ei:
            ix.add_table(eng)
        assert ei.value.code == E_STATE
        eng.finish()
        res, *_ = _session(eng, segs)
        with pytest.raises(MksnapError) as ei:                      # no delta in this session yet
            eng.chunk_status(res.n_chunks)
        assert ei.value.code == E_STATE
        eng.delta(ix)
        eng.chunk_status(res.n_chunks)
        eng.begin()
        with pytest.raises(MksnapError) as ei:
            eng.chunk_status(res.n_chunks)
        assert ei.value.code == E_STATE
        eng.finish()
        # an index created on one handle works with another handle on the same device
        with Engine(device=0, device_arena_bytes=16 << 20, max_extents=256) as e2:
            res2, *_ = _session(e2, segs)
            ix.add_table(e2)
            np.testing.assert_array_equal(ix.get(eng), e2.get_table(res2.n_unique))
            d, st, _ = _check_delta(e2, ix, res2)
            assert d.known_chunks == res2.n_chunks
        # after a local exchange the handles' tables are shards: E_STATE
        with Engine(device=0, device_arena_bytes=16 << 20, max_extents=256) as x0, \
                Engine(device=0, device_arena_bytes=16 << 20, max_extents=256) as x1:
            _session(x0, segs[:1])
            _session(x1, segs[1:])
            Engine.exchange_tables_local([x0, x1])
            for x in (x0, x1):
                for call in (lambda: x.delta(ix), lambda: ix.add_table(x), lambda: x.chunk_status(0)):
                    with pytest.raises(MksnapError) as ei:
                        call()
                    assert ei.value.code == E_STATE


def test_files_larger_than_an_arena(oracle_lib):
    """files split over submits (MKSNAP_X_MORE / MKSNAP_X_CONT) give the statuses of the undivided files"""
    from makisu_b200.abi import ChunkIndex, Engine
    from tests.test_gpu_parity import _split_submit
    rng = np.random.default_rng(7)
    big = _rand(rng, 9_000_000)
    zr = _rand(rng, 1_500_000)
    zr[200_000:900_000] = 0
    files = [_rand(rng, 70_000), big, zr, big.copy(), _rand(rng, 300_000)]
    pieces = [[70_000], [3_145_728, 3_145_728, 9_000_000 - 2 * 3_145_728], [524_288 - 512, 512 * 3, 1_500_000 - 524_288 - 1024],
              [4_000_000, 5_000_000], [300_000]]
    arena, offs = pack(files)
    want = oracle_lib.chunk_table(arena, offs, [len(f) for f in files])
    with Engine(device=0, device_arena_bytes=8 << 20, max_extents=256) as e:
        with ChunkIndex(e, 10_000) as ix:
            ix.add_rows(e, cd.union(want["digests"][:0], want["digests"][::3]))
            carry = e.limits().carry_bytes
            res = _split_submit(e, files, pieces, carry, False)
            d, st, dig = _check_delta(e, ix, res)
            np.testing.assert_array_equal(dig, want["digests"])
            np.testing.assert_array_equal(st, cd.classify(want["digests"], ix.get(e)))
            assert d.known_bytes + d.new_bytes + d.repeat_bytes == res.cdc_bytes == sum(len(f) for f in files)
            # the same bytes of every class as the undivided files (chunk lengths from the oracle's ends)
            c = cd.counts(st, cd.chunk_lens(want["ends"], offs, [len(f) for f in files]))
            assert (d.known_bytes, d.new_bytes, d.repeat_bytes) == (c["known_bytes"], c["new_bytes"], c["repeat_bytes"])


def test_delta_and_union_leave_the_session_untouched(eng):
    from makisu_b200.abi import ChunkIndex
    rng = np.random.default_rng(8)
    res, *_ = _session(eng, _mixed(rng))
    ends0, dig0 = eng.get_chunks(res.n_chunks)
    tab0 = eng.get_table(res.n_unique)
    with ChunkIndex(eng, 200_000) as ix:
        ix.add_rows(eng, _sorted_rows(rng, 100_000))
        eng.delta(ix)
        ix.add_table(eng)
        eng.delta(ix)
        ends1, dig1 = eng.get_chunks(res.n_chunks)
        np.testing.assert_array_equal(ends1, ends0)
        np.testing.assert_array_equal(dig1, dig0)
        np.testing.assert_array_equal(eng.get_table(res.n_unique), tab0)
        assert eng.table_rows() == res.n_unique
    from oracle import lib as olib
    assert olib.merkle_root(tab0) == bytes(res.root)


def _tar(files):
    buf = io.BytesIO()
    with tarfile.open(fileobj=buf, mode="w", format=tarfile.PAX_FORMAT) as tf:
        for name, data in files:
            ti = tarfile.TarInfo(name)
            ti.mode, ti.mtime, ti.uid, ti.gid, ti.size = 0o644, 1_500_000_000, 7, 8, len(data)
            tf.addfile(ti, io.BytesIO(data))
    return buf.getvalue()


def test_end_to_end_through_the_host_library(tmp_path, oracle_lib):
    """base layer -> MemFS.update_from_tar -> add_table; a COPY layer holding byte-identical copies of half the base
    files plus new files -> commit_copy_ops -> delta: every chunk of a copied file is known"""
    from makisu_b200 import host
    from makisu_b200.abi import ChunkIndex, Engine
    rng = np.random.default_rng(9)
    base = [(f"usr/lib/f{i:02d}.bin", _rand(rng, int(rng.integers(1, 900_000))).tobytes()) for i in range(12)]
    tar_path = tmp_path / "base.tar"
    tar_path.write_bytes(_tar(base))
    ctx = tmp_path / "ctx"
    ctx.mkdir()
    copied = base[::2]
    for name, data in copied:
        (ctx / os.path.basename(name)).write_bytes(data)
    for i in range(4):
        (ctx / f"new{i}.bin").write_bytes(_rand(rng, int(rng.integers(1000, 700_000))).tobytes())
    root = tmp_path / "root"
    root.mkdir()
    os.chmod(root, 0o755)
    with Engine(device=0, device_arena_bytes=8 << 20, n_host_arenas=2, host_arena_bytes=8 << 20, max_extents=1 << 12) as e:
        with ChunkIndex(e, 100_000) as ix:
            h = host.MemFS(str(root))
            with open(tar_path, "rb") as f:
                got = h.update_from_tar(e, 1_600_000_000, f.fileno())
            ix.add_table(e)
            assert ix.rows() == got["n_unique"]
            base_digests = set()
            for _, data in base:
                a = np.frombuffer(data, dtype=np.uint8)
                base_digests |= {bytes(r) for r in oracle_lib.chunk_table(a, [0], [a.size])["digests"]}
            assert {bytes(r) for r in ix.get(e)} == base_digests
            layer = h.commit_copy_ops(e, 1_600_000_000, [host.CopyOperation(["/"], str(ctx), "/", "/app/", 3, 4)])
            n = layer["n_chunks"]
            d = e.delta(ix)
            ends, dig = e.get_chunks(n)
            st = e.chunk_status(n)
            np.testing.assert_array_equal(st, cd.classify(dig, ix.get(e)))
            copied_digests = set()
            for _, data in copied:
                a = np.frombuffer(data, dtype=np.uint8)
                copied_digests |= {bytes(r) for r in oracle_lib.chunk_table(a, [0], [a.size])["digests"]}
            in_copied = np.array([bytes(r) in copied_digests for r in dig])
            assert in_copied.sum() >= len(copied) and (st[in_copied] == 0).all()
            assert d.known_chunks + d.new_chunks + d.repeat_chunks == n
            assert d.known_bytes >= sum(len(x) for _, x in copied)
            assert d.new_chunks > 0
            h.close()


def test_scale_device_resident_session(oracle_lib):
    """a multi-GiB device-resident session against its own table plus 10 M random rows, 10 % of files re-seeded"""
    from makisu_b200.abi import ChunkIndex, Engine
    n_files, fb = 8192, 512 << 10
    size = n_files * fb                                                   # 4 GiB
    offs = [i * fb for i in range(n_files)]
    ext = cdc_extents(offs, [fb] * n_files)
    rng = np.random.default_rng(10)
    with Engine(device=0, device_arena_bytes=size, max_extents=n_files + 16) as e:
        e.synth_fill(0, 0, size, 0xA1)
        e.begin()
        e.device_submit(0, size, ext)
        res_a = e.finish()
        extra = _sorted_rows(rng, 10_000_000)
        with ChunkIndex(e, res_a.n_unique + len(extra)) as ix:
            ix.add_table(e)
            ix.add_rows(e, extra)
            want_rows = cd.union(e.get_table(res_a.n_unique), extra)
            assert ix.rows() == len(want_rows)
            np.testing.assert_array_equal(ix.get(e), want_rows)
            for k in rng.choice(n_files, n_files // 10, replace=False):
                e.synth_fill(0, int(k) * fb, fb, 0xB000 + int(k))
            e.begin()
            e.device_submit(0, size, ext)
            res_b = e.finish()
            d, st, dig = _check_delta(e, ix, res_b)
            assert 0.8 < d.known_chunks / res_b.n_chunks < 0.95
            assert d.new_chunks > 0
            ends, _ = e.get_chunks(res_b.n_chunks)
            c = cd.counts(st, cd.chunk_lens(ends, offs, [fb] * n_files))
            assert (d.known_bytes, d.new_bytes, d.repeat_bytes) == (c["known_bytes"], c["new_bytes"], c["repeat_bytes"])
