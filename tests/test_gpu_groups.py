"""-m gpu: grouped sessions (mksnap_begin_groups ... mksnap_delta_groups, DESIGN.md section 3c).

Every group table, root, status and count is compared bit for bit with (a) one ungrouped session per group, built from
the same files on the same engine, and (b) tests/chunk_groups_ref.py on the engine's downloaded digests; every batch
output of a grouped session is compared with an ungrouped session of the same submits.
"""
import ctypes
import os

import numpy as np
import pytest

from oracle import chunk_delta as cd
from tests import chunk_groups_ref as ref
from tests.table_ref import msg, ref_merkle, twins

pytestmark = pytest.mark.gpu

E_INVAL, E_STATE = -1, -5
FIXED64 = (64, 64, 64, 16, 12)


# ---- plans: a session as data, replayed grouped, ungrouped, or restricted to one group -----------------------------
def _sub(arena, ext, grp, pinned=False):
    """one submit: the arena bytes, extents (off, len, flags[, reserved]) and one group per extent"""
    return dict(arena=np.ascontiguousarray(arena, dtype=np.uint8), ext=[tuple(x) for x in ext], grp=list(grp), pinned=pinned)


def _extents(items):
    from makisu_b200.abi import Extent
    if not items:
        return []
    arr = (Extent * len(items))()
    for k, x in enumerate(items):
        arr[k].arena_off, arr[k].len, arr[k].crc_suffix, arr[k].flags = x[0], x[1], 0, x[2]
        arr[k].reserved = x[3] if len(x) > 3 else 0
    return arr


def _run(e, plan, G=None, only=None):
    """G: a grouped session; only: an ungrouped session of group `only`'s CDC extents (same submits, same order)"""
    if G is not None:
        e.begin_groups(G)
    else:
        e.begin()
    for sub in plan:
        items = [(x, g) for x, g in zip(sub["ext"], sub["grp"]) if only is None or g == only]
        ext = _extents([x for x, _ in items])
        grp = [g for _, g in items] if G is not None else None
        a = sub["arena"]
        if sub["pinned"]:
            ptr, cap, aid = e.arena_acquire()
            ctypes.memmove(ptr, a.ctypes.data, a.size)
            e.arena_submit(aid, a.size, ext, groups=grp)
        else:
            e.device_upload(0, 0, a)
            e.device_submit(0, a.size, ext, groups=grp)
    return e.finish()


def _res(r):
    return (r.crc_pure, r.crc_bytes, r.cdc_bytes, r.n_files, r.n_chunks, r.n_unique, bytes(r.root), r.n_streams)


def _outputs(e, r):
    ends, dig = e.get_chunks(r.n_chunks)
    return dict(res=_res(r), ends=ends.copy(), dig=dig.copy(), tab=e.get_table(r.n_unique).copy())


def _same(a, b):
    assert a["res"] == b["res"]
    for k in ("ends", "dig", "tab"):
        np.testing.assert_array_equal(a[k], b[k])


def _check_grouped(e, plan, G):
    """grouped == ungrouped for the batch; every group == its own ungrouped session == the reference"""
    plain = _outputs(e, _run(e, plan))
    grouped = _outputs(e, _run(e, plan, G=G))
    _same(grouped, plain)
    n = grouped["res"][4]
    gres = e.group_results(G)
    tabs = [e.group_table(g, gres[g].n_unique).copy() for g in range(G)]
    cg = e.chunk_groups(n).copy()
    ref_tabs = ref.group_tables(grouped["dig"], cg, G)
    row = 0
    for g in range(G):
        np.testing.assert_array_equal(tabs[g], ref_tabs[g])
        assert bytes(gres[g].root) == ref_merkle(tabs[g]), g
        assert gres[g].first_row == row
        row += gres[g].n_unique
    assert sum(r.n_files for r in gres) == grouped["res"][3]
    assert sum(r.cdc_bytes for r in gres) == grouped["res"][2]
    assert sum(r.n_chunks for r in gres) == n
    for g in range(G):
        alone = _outputs(e, _run(e, plan, only=g))
        r = gres[g]
        assert (r.n_files, r.cdc_bytes, r.n_chunks, r.n_unique, bytes(r.root)) == \
            (alone["res"][3], alone["res"][2], alone["res"][4], alone["res"][5], alone["res"][6]), g
        np.testing.assert_array_equal(tabs[g], alone["tab"])
        np.testing.assert_array_equal(grouped["dig"][cg == g], alone["dig"])   # group order = the standalone order
    return grouped, gres, tabs, cg


def _check_delta_groups(e, plan, G, index_rows):
    """delta_groups == the sequential flow (per-group session -> delta -> add_table) and the reference; ix unchanged;
    add_table after the grouped batch and add_group for g = 0..G-1 end where the sequential flow ends"""
    from makisu_b200.abi import ChunkIndex
    index_rows = np.ascontiguousarray(index_rows, dtype=np.uint8).reshape(-1, 32)
    cap = len(index_rows) + 4 * sum(sum(1 for x in s["ext"]) for s in plan) + 200_000
    with ChunkIndex(e, cap) as ix:
        if len(index_rows):
            ix.add_rows(e, index_rows)
        r = _run(e, plan, G=G)
        n = r.n_chunks
        _, dig = e.get_chunks(n)
        cg = e.chunk_groups(n).copy()
        before = ix.get(e).copy()
        out = e.delta_groups(ix, G)
        st = e.chunk_status(n).copy()
        np.testing.assert_array_equal(ix.get(e), before)          # the call does not change the index
        np.testing.assert_array_equal(st, ref.classify_groups(dig, cg, before))
        ix.add_table(e)
        after_table = ix.get(e).copy()
    with ChunkIndex(e, cap) as ix:
        if len(index_rows):
            ix.add_rows(e, index_rows)
        _run(e, plan, G=G)
        for g in range(G):
            ix.add_group(e, g)
        after_groups = ix.get(e).copy()
    with ChunkIndex(e, cap) as seq:
        if len(index_rows):
            seq.add_rows(e, index_rows)
        for g in range(G):
            rg = _run(e, plan, only=g)
            d = e.delta(seq)
            np.testing.assert_array_equal(e.chunk_status(rg.n_chunks), st[cg == g])
            o = out[g]
            assert (o.known_chunks, o.new_chunks, o.repeat_chunks, o.known_bytes, o.new_bytes, o.repeat_bytes) == \
                (d.known_chunks, d.new_chunks, d.repeat_chunks, d.known_bytes, d.new_bytes, d.repeat_bytes), g
            assert o.index_rows == len(before)
            seq.add_table(e)
        final = seq.get(e).copy()
    np.testing.assert_array_equal(after_table, final)
    np.testing.assert_array_equal(after_groups, final)
    return out, st, cg


# ---- content -----------------------------------------------------------------------------------------------------
def _rand(rng, n):
    return rng.integers(0, 256, n, dtype=np.uint8)


def _pack(files, base=0, align=512):
    offs, pos = [], base
    for f in files:
        pos = (pos + align - 1) // align * align
        offs.append(pos)
        pos += len(f)
    arena = np.zeros((pos + 511) // 512 * 512 or 512, dtype=np.uint8)
    for f, o in zip(files, offs):
        arena[o:o + len(f)] = f
    return arena, offs


def _mixed_plan(rng, G, n_submits=3, pinned=()):
    """files of every kind, groups interleaved within and across submits, the same content in several groups"""
    shared = _rand(rng, 350_000)
    plan = []
    for s in range(n_submits):
        files, grp = [], []
        for k in range(12):
            kind = int(rng.integers(0, 5))
            f = [_rand(rng, int(rng.integers(1, 400_000))), shared, np.zeros(int(rng.integers(1, 300_000)), np.uint8),
                 np.tile(_rand(rng, 41), 3000), _rand(rng, int(rng.integers(1, 3000)))][kind]
            files.append(f)
            grp.append(int(rng.integers(0, G)))
        arena, offs = _pack(files)
        plan.append(_sub(arena, [(o, len(f), 2) for o, f in zip(offs, files)], grp, pinned=s in pinned))
    return plan


@pytest.fixture(scope="module")
def eng():
    from makisu_b200.abi import Engine
    e = Engine(device=0, device_arena_bytes=32 << 20, n_host_arenas=2, host_arena_bytes=16 << 20, max_extents=1 << 14)
    yield e
    e.close()


# ---- tests -------------------------------------------------------------------------------------------------------
def test_grouped_session_equals_one_session_per_group(eng):
    rng = np.random.default_rng(1)
    plan = _mixed_plan(rng, 5)
    _check_grouped(eng, plan, 5)


def test_one_group_is_the_ungrouped_session(eng):
    from makisu_b200.abi import ChunkIndex
    rng = np.random.default_rng(2)
    plan = _mixed_plan(rng, 1)
    grouped, gres, tabs, cg = _check_grouped(eng, plan, 1)
    np.testing.assert_array_equal(tabs[0], grouped["tab"])
    assert bytes(gres[0].root) == grouped["res"][6]
    assert not cg.any()
    extra = cd.union(grouped["tab"][:0], _rand(rng, 32 * 5000).reshape(-1, 32))
    index_rows = cd.union(extra, grouped["tab"][::4])
    with ChunkIndex(eng, 100_000) as ix:
        ix.add_rows(eng, index_rows)
        r = _run(eng, plan)
        d = eng.delta(ix)
        st = eng.chunk_status(r.n_chunks).copy()
        _run(eng, plan, G=1)
        (g,) = eng.delta_groups(ix)
        np.testing.assert_array_equal(eng.chunk_status(r.n_chunks), st)
        assert (g.known_chunks, g.new_chunks, g.repeat_chunks, g.known_bytes, g.new_bytes, g.repeat_bytes, g.index_rows) == \
            (d.known_chunks, d.new_chunks, d.repeat_chunks, d.known_bytes, d.new_bytes, d.repeat_bytes, d.index_rows)
    _check_delta_groups(eng, plan, 1, index_rows)


def test_pinned_and_device_submits_split_file_empty_and_one_row_groups(eng):
    """groups interleaved over pinned arenas and device slots; a 9 MB file of group 2 split over two arenas
    (MKSNAP_X_MORE / MKSNAP_X_CONT); group 4 empty; groups 5 and 6 one small file each (one row)"""
    rng = np.random.default_rng(3)
    carry = eng.limits().carry_bytes
    big = _rand(rng, 9_000_000)
    head, tail = big[:5_000_000], big[5_000_000:]
    small = [_rand(rng, int(rng.integers(1000, 300_000))) for _ in range(10)]
    a0, o0 = _pack(small[:4] + [head])
    s0 = _sub(a0, [(o, len(f), 2) for o, f in zip(o0[:4], small[:4])] + [(o0[4], len(head), 2 | 4, len(tail))],
              [0, 1, 3, 0, 2], pinned=True)
    files1 = [tail] + small[4:7] + [_rand(rng, 100)]
    a1, o1 = _pack(files1, base=carry)
    s1 = _sub(a1, [(o1[0], len(tail), 2 | 8)] + [(o, len(f), 2) for o, f in zip(o1[1:], files1[1:])],
              [2, 1, 0, 3, 5], pinned=False)
    files2 = small[7:] + [small[0], _rand(rng, 3000)]
    a2, o2 = _pack(files2)
    s2 = _sub(a2, [(o, len(f), 2) for o, f in zip(o2, files2)], [3, 0, 1, 2, 6], pinned=True)
    plan = [s0, s1, s2]
    _, gres, tabs, _ = _check_grouped(eng, plan, 7)
    assert gres[4].n_unique == 0 and bytes(gres[4].root) == ref_merkle([])
    assert gres[5].n_unique == 1 and gres[6].n_unique == 1
    ix_rows = cd.union(tabs[0][:0], np.concatenate([tabs[1][::2], tabs[2][:3], _rand(rng, 32 * 1000).reshape(-1, 32)]))
    _check_delta_groups(eng, plan, 7, ix_rows)


def test_prefix_twins_in_the_same_and_in_different_groups(eng):
    """32-byte files whose digests share their 32-bit sort key: pairs inside one group, pairs split over two groups,
    triples over three, every member repeated"""
    rng = np.random.default_rng(4)
    pairs, triples = twins("pairs")[:300], twins("triples")[:100]
    items = []
    for i, p in enumerate(pairs):
        for k, (c, _) in enumerate(p):
            g = 0 if i % 2 == 0 else 1 + k                          # even pairs in group 0, odd pairs over groups 1 and 2
            items += [(c, g)] * int(rng.integers(1, 4))
    for t in triples:
        items += [(c, 3 + k) for k, (c, _) in enumerate(t)] * 2
    order = rng.permutation(len(items))
    items = [items[i] for i in order]
    uniq = sorted({c for c, _ in items})
    at = {c: 32 * i for i, c in enumerate(uniq)}
    arena = np.frombuffer(b"".join(msg(c) for c in uniq), dtype=np.uint8)
    half = len(items) // 2
    plan = [_sub(arena, [(at[c], 32, 2) for c, _ in part], [g for _, g in part]) for part in (items[:half], items[half:])]
    _, _, tabs, _ = _check_grouped(eng, plan, 6)
    _check_delta_groups(eng, plan, 6, cd.union(tabs[1][:0], np.concatenate([tabs[1][::3], tabs[4][::2]])))


@pytest.fixture(scope="module")
def eng64():
    from makisu_b200.abi import CdcParams, Engine
    e = Engine(device=0, device_arena_bytes=16 << 20, max_extents=1 << 12, cdc=CdcParams(*FIXED64))
    yield e
    e.close()


def test_merkle_level_boundaries_per_group(eng64):
    """fixed 64-byte chunks of synth_fill content: groups of 255, 256, 257, 65 537, 1 and 0 distinct rows, their
    files interleaved, and a repeat of group 0's first file in group 1"""
    sizes = {0: 255, 1: 256, 2: 257, 3: 65_537, 4: 1, 5: 0}
    rng = np.random.default_rng(5)
    files = []
    for g, u in sizes.items():
        left = u
        while left:
            k = min(int(rng.integers(1, 3000)), left)
            files.append((g, k))
            left -= k
    files = [files[i] for i in rng.permutation(len(files))]
    ext, grp, pos = [], [], 0
    for i, (g, k) in enumerate(files):
        eng64.synth_fill(0, pos, 64 * k, 0x5100 + i)
        ext.append((pos, 64 * k, 2))
        grp.append(g)
        pos += (64 * k + 511) // 512 * 512
    first0 = next(x for x, g in zip(ext, grp) if g == 0)
    ext.append(first0)
    grp.append(1)
    arena = eng64.device_download(0, 0, pos)
    plan = [_sub(arena, ext, grp)]
    _, gres, _, _ = _check_grouped(eng64, plan, 6)
    first_len = first0[1] // 64
    assert [r.n_unique for r in gres] == [255, 256 + first_len, 257, 65_537, 1, 0]


def test_rejections_leave_the_session_unchanged(eng):
    from makisu_b200.abi import ChunkIndex, MksnapError
    rng = np.random.default_rng(6)
    plan = _mixed_plan(rng, 3, n_submits=2)
    want = _outputs(eng, _run(eng, plan))
    # grouped getters on an ungrouped (finished) session
    with ChunkIndex(eng, 1000) as ix:
        for call in (lambda: eng.group_results(3), lambda: eng.group_table(0, 10), lambda: eng.chunk_groups(10),
                     lambda: eng.delta_groups(ix, 3), lambda: ix.add_group(eng, 0)):
            with pytest.raises(MksnapError) as ei:
                call()
            assert ei.value.code == E_STATE
    for bad in (0, 65_537):
        with pytest.raises(MksnapError) as ei:
            eng.begin_groups(bad)
        assert ei.value.code == E_INVAL
    # a grouped submit in an ungrouped session
    eng.begin()
    sub = plan[0]
    eng.device_upload(0, 0, sub["arena"])
    with pytest.raises(MksnapError) as ei:
        eng.device_submit(0, sub["arena"].size, _extents(sub["ext"]), groups=sub["grp"])
    assert ei.value.code == E_STATE
    # inside a grouped session: a plain submit, a group out of range, getters before finish, then the real submits
    eng.begin_groups(3)
    with pytest.raises(MksnapError) as ei:
        eng.device_submit(0, sub["arena"].size, _extents(sub["ext"]))
    assert ei.value.code == E_STATE
    bad = list(sub["grp"])
    bad[1] = 3
    with pytest.raises(MksnapError) as ei:
        eng.device_submit(0, sub["arena"].size, _extents(sub["ext"]), groups=bad)
    assert ei.value.code == E_INVAL
    with pytest.raises(MksnapError) as ei:
        eng.group_results(3)
    assert ei.value.code == E_STATE
    for s in plan:
        eng.device_upload(0, 0, s["arena"])
        eng.device_submit(0, s["arena"].size, _extents(s["ext"]), groups=s["grp"])
    _same(_outputs(eng, eng.finish()), want)
    gres = eng.group_results(3)
    with pytest.raises(MksnapError) as ei:
        eng.group_results(2)
    assert ei.value.code == E_INVAL
    with pytest.raises(MksnapError) as ei:
        eng.group_table(3, 10)
    assert ei.value.code == E_INVAL
    # the groups match a clean grouped run of the same plan
    clean = _run(eng, plan, G=3)
    assert [bytes(r.root) for r in eng.group_results(3)] == [bytes(r.root) for r in gres]
    assert _res(clean) == want["res"]


def test_continuation_must_keep_its_group(eng):
    from makisu_b200.abi import MksnapError
    rng = np.random.default_rng(7)
    carry = eng.limits().carry_bytes
    big = _rand(rng, 3_000_000)
    a0, o0 = _pack([big[:1_000_000]])
    a1, o1 = _pack([big[1_000_000:]], base=carry)
    eng.begin_groups(2)
    eng.device_upload(0, 0, a0)
    eng.device_submit(0, a0.size, _extents([(o0[0], 1_000_000, 2 | 4, 2_000_000)]), groups=[1])
    eng.device_upload(0, 0, a1)
    with pytest.raises(MksnapError) as ei:
        eng.device_submit(0, a1.size, _extents([(o1[0], 2_000_000, 2 | 8)]), groups=[0])
    assert ei.value.code == E_INVAL
    eng.device_submit(0, a1.size, _extents([(o1[0], 2_000_000, 2 | 8)]), groups=[1])
    r = eng.finish()
    gres = eng.group_results(2)
    assert (gres[0].n_chunks, gres[1].n_chunks, gres[1].n_files, gres[1].cdc_bytes) == (0, r.n_chunks, 1, 3_000_000)
    assert bytes(gres[1].root) == bytes(r.root)


NOW = 1_600_000_000


def _mk(root, rel, data=b"", mode=0o644, mtime=1_500_000_000):
    p = os.path.join(root, rel)
    os.makedirs(os.path.dirname(p), exist_ok=True)
    with open(p, "wb") as f:
        f.write(data)
    os.chmod(p, mode)
    os.utime(p, (mtime, mtime))


def test_commit_layers_with_layer_tables_end_to_end(tmp_path):
    """mkhost_memfs_commit_layers(MKHOST_LAYER_TABLES) on the 6-layer spec of test_gpu_host's batch test: every layer's
    root / n_chunks / n_unique, chunk digests, delta statuses and counts equal six sequential commit_copy_ops + delta +
    add_table, and the TarDigests equal the ungrouped batch's"""
    from makisu_b200 import host
    from makisu_b200.abi import ChunkIndex, Engine
    c = str(tmp_path / "ctx")
    rng = np.random.default_rng(42)
    _mk(c, "Dockerfile", b"FROM scratch\nCOPY . /app/\n")
    for d in range(4):
        for i in range(12):
            _mk(c, f"d{d}/f{i:03d}.bin", rng.integers(0, 256, int(rng.integers(0, 600_000)), dtype=np.uint8).tobytes())
    _mk(c, "d3/dup.bin", open(os.path.join(c, "d0/f000.bin"), "rb").read())
    _mk(c, "big.bin", rng.integers(0, 256, 11_000_000, dtype=np.uint8).tobytes())
    _mk(c, "empty", b"")
    _mk(c, "zeros", bytes(300_000))
    os.symlink("big.bin", os.path.join(c, "link"))
    specs = [(["/d0"], "/app/d0/"), (["/d1", "/d2"], "/app/"), (["/zeros", "/empty"], "/app/"), (["/d3"], "/srv/"),
             (["/d0"], "/app/d0/"), (["/link"], "/app/")]
    ops = [[host.CopyOperation(s, c, "/", d)] for s, d in specs]
    L = len(specs)
    for arena in (16 << 20, 64 << 20):
        roots = []
        for k in range(2):
            r = tmp_path / ("root%d_%d" % (k, arena))
            r.mkdir()
            os.chmod(r, 0o755)
            roots.append(str(r))
        with Engine(device=0, device_arena_bytes=arena, n_host_arenas=2, host_arena_bytes=arena, max_extents=1 << 12) as eng:
            with ChunkIndex(eng, 1 << 20) as ix:
                ix.add_rows(eng, cd.union(np.zeros((0, 32), np.uint8), rng.integers(0, 256, (5000, 32), dtype=np.uint8)))
                start_rows = ix.get(eng).copy()
                # sequential: one commit per layer, delta, add_table
                h = host.MemFS(roots[0])
                seq = []
                for layer in ops:
                    got = h.commit_copy_ops(eng, NOW, layer)
                    d = eng.delta(ix)
                    _, dig = eng.get_chunks(got["n_chunks"])
                    seq.append((got, d, eng.chunk_status(got["n_chunks"]).copy(), dig.copy()))
                    ix.add_table(eng)
                seq_rows = ix.get(eng).copy()
                h.close()
            with ChunkIndex(eng, 1 << 20) as ix:
                ix.add_rows(eng, start_rows)
                h = host.MemFS(roots[1])
                got = h.commit_layers(eng, NOW, ops, layer_tables=True)
                h.close()
                n = sum(g["n_chunks"] for g in got)
                _, dig = eng.get_chunks(n)
                cg = eng.chunk_groups(n)
                out = eng.delta_groups(ix, L)
                st = eng.chunk_status(n)
                for i, (g1, d1, st1, dig1) in enumerate(seq):
                    for k in ("tar_digest", "root", "n_chunks", "n_unique"):
                        assert got[i][k] == g1[k], (i, k, arena)
                    np.testing.assert_array_equal(dig[cg == i], dig1)
                    np.testing.assert_array_equal(st[cg == i], st1)
                    o = out[i]
                    assert (o.known_chunks, o.new_chunks, o.repeat_chunks, o.known_bytes, o.new_bytes, o.repeat_bytes) == \
                        (d1.known_chunks, d1.new_chunks, d1.repeat_chunks, d1.known_bytes, d1.new_bytes, d1.repeat_bytes)
                for i in range(L):
                    ix.add_group(eng, i)
                np.testing.assert_array_equal(ix.get(eng), seq_rows)
    assert len({g["root"] for g in got}) >= L - 1                  # the layers have their own content addresses


def test_four_gib_session_with_256_groups_against_a_large_index():
    """4 GiB device resident, 256 groups of 64 files of 256 KiB, every group repeating four files of other groups,
    against a 3 M-row index holding every fifth row of the batch: grouped delta, group tables and roots against the
    reference on the downloaded digests"""
    from makisu_b200.abi import ChunkIndex, Engine
    G, per, fb = 256, 64, 256 << 10
    total = G * per * fb
    rng = np.random.default_rng(9)
    with Engine(device=0, device_arena_bytes=total, max_extents=1 << 15) as e:
        e.synth_fill(0, 0, total, 0xC0FFEE)
        ext, grp = [], []
        for f in range(G * per):
            ext.append((f * fb, fb, 2))
            grp.append(f % G)                                       # groups interleaved file by file
        for g in range(G):
            for f in rng.integers(0, G * per, 4):
                ext.append((int(f) * fb, fb, 2))
                grp.append(g)
        e.begin_groups(G)
        e.device_submit(0, total, _extents(ext), groups=grp)
        r = e.finish()
        n = r.n_chunks
        ends, dig = e.get_chunks(n)
        cg = e.chunk_groups(n).copy()
        tab = e.get_table(r.n_unique)
        gres = e.group_results(G)
        ref_tabs = ref.group_tables(dig, cg, G)
        for g in range(G):
            t = e.group_table(g, gres[g].n_unique)
            np.testing.assert_array_equal(t, ref_tabs[g])
            assert bytes(gres[g].root) == ref_merkle(t)
        with ChunkIndex(e, 4_000_000) as ix:
            ix.add_rows(e, cd.union(tab[::5], rng.integers(0, 256, (3_000_000, 32), dtype=np.uint8)))
            before = ix.get(e)
            out = e.delta_groups(ix, G)
            st = e.chunk_status(n)
            want = ref.classify_groups(dig, cg, before)
            np.testing.assert_array_equal(st, want)
            np.testing.assert_array_equal(ix.get(e), before)
        # per-group counts: chunks from the statuses, bytes from the chunk lengths
        lens = np.empty(n, dtype=np.uint64)
        k, prev = 0, None
        for i in range(n):
            off, ln, _ = ext[k]
            start = off if prev is None else prev
            lens[i] = int(ends[i]) - start
            if int(ends[i]) == off + ln:
                k, prev = k + 1, None
            else:
                prev = int(ends[i])
        for g in range(G):
            c = cd.counts(want[cg == g], lens[cg == g])
            o = out[g]
            assert (o.known_chunks, o.new_chunks, o.repeat_chunks, o.known_bytes, o.new_bytes, o.repeat_bytes) == \
                (c["known_chunks"], c["new_chunks"], c["repeat_chunks"], c["known_bytes"], c["new_bytes"], c["repeat_bytes"])
        assert sum(o.new_chunks for o in out) == r.n_unique - int(cd.contains(before, tab).sum())
