"""-m gpu (one device): the range-partitioned exchange (mksnap_exchange_tables) run between R engines of one process
through the local transport -- the same phase code NCCL drives, so every R and every awkward distribution (empty
ranks, ranks with fewer than 256 rows, a Merkle group straddling several ranks) is covered on a single GPU.
Expected values: the oracle's Merkle root over the union, and makisu_b200.shard.exchange_tables_model."""
import ctypes
import hashlib

import numpy as np
import pytest

from tests.util import pack, cdc_extents, crc_extents

pytestmark = pytest.mark.gpu


def _random_segs(per_rank_lens, seed, dup_from_rank0=0):
    """Random files of the given lengths per rank; with dup_from_rank0, every non-empty rank's first file is one shared
    file of that length"""
    rng = np.random.default_rng(seed)
    shared = rng.integers(0, 256, dup_from_rank0, dtype=np.uint8) if dup_from_rank0 else None
    out = []
    for lens in per_rank_lens:
        segs = [rng.integers(0, 256, n, dtype=np.uint8) for n in lens]
        if shared is not None and lens:
            segs[0] = shared.copy()   # the same file on every rank
        out.append(segs)
    return out


def _run(oracle_lib, per_rank_segs, **engine_kw):
    """One local exchange of R engines, engine r holding per_rank_segs[r] (files, each one CRC + CDC extent)"""
    from makisu_b200 import shard
    from makisu_b200.abi import Engine, MKSNAP_X_CDC
    from tests.table_ref import ref_merkle
    kw = {**dict(device=0, device_arena_bytes=24 << 20, max_extents=1 << 10, max_chunks=1 << 14), **engine_kw}
    engines, tables, sums = [], [], dict(n_chunks=0, n_files=0, cdc_bytes=0, crc=0, crc_bytes=0)
    try:
        for r, segs in enumerate(per_rank_segs):
            e = Engine(**kw)
            engines.append(e)
            lens = [len(s) for s in segs]
            e.begin()
            if lens:
                arena, offs = pack(segs)
                ext, _ = crc_extents(offs, lens, list(range(len(lens))), flags_extra=[MKSNAP_X_CDC] * len(lens))
                e.device_upload(0, 0, arena)
                e.device_submit(0, arena.size, ext)
            res = e.finish()
            tables.append(e.get_table(res.n_unique).copy())
            sums["n_chunks"] += res.n_chunks
            sums["n_files"] += res.n_files
            sums["cdc_bytes"] += res.cdc_bytes
            sums["crc_bytes"] += res.crc_bytes
            sums["crc"] ^= res.crc_pure
        outs = Engine.exchange_tables_local(engines)
        union = sorted({bytes(row) for t in tables for row in t})
        cat = np.frombuffer(b"".join(union), dtype=np.uint8).reshape(-1, 32) if union else np.zeros((0, 32), np.uint8)
        want_root = (ctypes.c_uint8 * 32)()
        oracle_lib.L().mko_merkle_root(np.ascontiguousarray(cat).ctypes.data if union else None, len(union), want_root)
        model_root, model_ranges = shard.exchange_tables_model(tables, lambda b: hashlib.sha256(b).digest())
        assert model_root == bytes(want_root) == ref_merkle(union)
        got_ranges = []
        for r, (e, o) in enumerate(zip(engines, outs)):
            assert bytes(o.root) == bytes(want_root), (r, [len(t) for t in tables])
            assert o.n_unique == len(union) and o.n_chunks == sums["n_chunks"] and o.n_files == sums["n_files"]
            assert o.cdc_bytes == sums["cdc_bytes"] and o.crc_bytes == sums["crc_bytes"] and o.crc_pure == sums["crc"]
            rows = e.get_table(e.table_rows())
            np.testing.assert_array_equal(rows, model_ranges[r])
            got_ranges.append(rows.tobytes())
        assert b"".join(got_ranges) == b"".join(union)
        return len(union), [len(t) for t in tables]
    finally:
        for e in engines:
            e.close()


@pytest.mark.parametrize("per_rank", [
    [[3_000_000]],                                                   # R=1: the exchange degenerates to finish()
    [[2_000_000, 500_000], [1_500_000]],                             # R=2
    [[], [70_000], [4_000_000], []],                                 # empty ranks, a rank with a handful of rows
    [[100], [], [5], [9_000_000], [4096 * 3], [1], [], [200_000]],   # R=8, most ranks below one Merkle group
    [[], [], []],                                                    # nothing anywhere: root = SHA-256("")
    [[5], [], [], [], []],                                           # one row in total
    [[6_000_000], [6_000_000], [6_000_000]],                         # several groups per rank, straddling boundaries
])
def test_local_exchange_equals_single_table(oracle_lib, per_rank):
    _run(oracle_lib, _random_segs(per_rank, seed=len(per_rank) * 7 + sum(map(len, per_rank))))


def test_local_exchange_dedups_across_ranks(oracle_lib):
    n, sizes = _run(oracle_lib, _random_segs([[900_000, 300_000], [900_000], [900_000, 10], [900_000]], seed=5,
                                         dup_from_rank0=900_000))
    assert n < sum(sizes)          # the shared 900 kB region is counted once globally


@pytest.mark.parametrize("n_ranks", [2, 3, 8])
def test_local_exchange_of_prefix_twins(oracle_lib, n_ranks):
    """digests sharing their 32-bit sort key, the members of each group on different ranks, and duplicates of some on
    every rank: every receiving rank sorts ties of its slices"""
    from tests.table_ref import msg, twins
    segs = [[] for _ in range(n_ranks)]
    pairs, triples = twins("pairs")[:600], twins("triples")[:12]
    for i, g in enumerate(pairs + triples):
        for k, (c, _) in enumerate(g):
            segs[(i + k) % n_ranks].append(msg(c))
    for g in pairs[:40] + triples[:4]:
        for r in range(n_ranks):
            segs[r].append(msg(g[r % len(g)][0]))
    n, sizes = _run(oracle_lib, segs, max_extents=1 << 12)
    assert n == 2 * len(pairs) + sum(len(g) for g in triples)


@pytest.mark.parametrize("n_ranks", [3, 8])
@pytest.mark.parametrize("u", [256, 257, 65536, 65537])
def test_local_exchange_of_fixed_size_chunks(oracle_lib, n_ranks, u):
    """min = normal = max = 64: exactly `u` distinct chunks in the union, at the Merkle level boundaries; ranks hold
    uneven shares (one holds none of its own) and a copy of rank 0's first file"""
    from makisu_b200.abi import CdcParams
    rng = np.random.default_rng(u * 10 + n_ranks)
    share = rng.dirichlet(np.ones(n_ranks)) * u
    share[1] = 0
    counts = np.floor(share).astype(int)
    counts[0] += u - counts.sum()
    segs = []
    for r, k in enumerate(counts):
        cuts = np.sort(rng.integers(0, k + 1, 2)) if k else np.zeros(2, int)
        segs.append([rng.integers(0, 256, 64 * int(n), dtype=np.uint8) for n in np.diff(np.r_[0, cuts, k]) if n])
    first = segs[0][0]
    for r in range(1, n_ranks):
        segs[r].append(first.copy())
    n, sizes = _run(oracle_lib, segs, cdc=CdcParams(64, 64, 64, 16, 12), max_chunks=1 << 17)
    assert n == u
