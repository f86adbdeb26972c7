#!/usr/bin/env python
"""bench_groups.py -- cost of per-layer chunk tables (grouped sessions) on the flagship context.

  python bench_groups.py --reps 20 --warmup 3          (C3: 100k files x 512 KiB, device resident, 256 groups)

Workload (BASELINE configs[2], the layout of bench.py's context_layout): session A fills a chunk index with A's table
plus 3x as many random rows (the 4x index of bench_delta.py); session B is A with 10 % of the files re-seeded on the
device.  B is submitted with one group per directory (256 groups, as if its 256 directories were 256 layers committed
together).  Measured: the host clock around mksnap_finish for the same submits grouped and ungrouped, alternating,
after a device synchronize that ends the submit (so only finish is timed); and mksnap_delta_groups against the 4x index
(ms_device = CUDA events around its kernels, and a host clock around the call).

Before anything is timed ("gate"): the grouped batch outputs equal the ungrouped ones, every group table equals the
sorted-unique digests of its chunks and every group root the fan-out-256 Merkle root of its table (on B's downloaded
digests), and the grouped statuses and per-group counts equal tests/chunk_groups_ref.py.  Median, min and max over
--reps after --warmup.  Prints one JSON line; writes nothing in the tree.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from bench import context_layout, ext_ptr  # noqa: E402
from bench_delta import card, stats  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--files", type=int, default=100_000)
    ap.add_argument("--file-kib", type=int, default=512)
    ap.add_argument("--dirs", type=int, default=256)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reseed", type=float, default=0.10)
    ap.add_argument("--step-ms", type=float, default=73.0, help="the C3 step time the shares are quoted against")
    args = ap.parse_args()
    real_stdout = os.dup(1)
    os.dup2(2, 1)  # library chatter goes to stderr; the JSON line alone to stdout

    from makisu_b200.abi import ChunkIndex, Engine
    from oracle import chunk_delta as cd
    from tests import chunk_groups_ref as ref
    from tests.table_ref import ref_merkle

    fb = args.file_kib << 10
    lay = context_layout(args.files, fb, args.dirs, 0)
    ext, used = lay["ext"], lay["used"]
    n_ext = len(ext)
    per_dir = (args.files + args.dirs - 1) // args.dirs
    groups = np.zeros(n_ext, dtype=np.uint32)
    is_file = (ext["flags"] & 2) != 0
    groups[is_file] = np.arange(args.files, dtype=np.uint32) // per_dir   # files come in file order
    G = int(groups.max()) + 1
    arena_bytes = (used + (1 << 20)) // 512 * 512
    out = {"metric": "chunk_groups", "card": card(),
           "workload": f"{args.files} files x {args.file_kib} KiB device resident (BASELINE configs[2]), {G} groups "
                       f"(one per directory); B = A with {args.reseed:.0%} of the files re-seeded"}
    eng = Engine(device=0, device_arena_bytes=arena_bytes, n_host_arenas=0, max_extents=n_ext + 16,
                 max_chunks=max(arena_bytes, lay["data_bytes"]) // 4096 + n_ext + 1024)

    def session(grouped):
        """-> (result, host ms of finish alone)"""
        if grouped:
            eng.begin_groups(G)
            rc = eng.lib.mksnap_device_submit_groups(eng.h, 0, used, ext_ptr(ext), n_ext, groups.ctypes.data, None, 0)
        else:
            eng.begin()
            rc = eng.lib.mksnap_device_submit(eng.h, 0, used, ext_ptr(ext), n_ext, None, 0)
        eng._ck(rc, "submit")
        eng.sync()
        t = time.perf_counter()
        res = eng.finish()
        return res, (time.perf_counter() - t) * 1e3

    eng.synth_fill(0, 0, (lay["data_bytes"] + 15) // 16 * 16, 0xC3)
    eng.device_upload(0, lay["meta_base"], np.frombuffer(lay["blob"], dtype=np.uint8))
    eng.sync()
    res_a, _ = session(False)
    table_a = eng.get_table(res_a.n_unique)
    rng = np.random.default_rng(0xDE17A)
    for k in rng.choice(args.files, int(args.files * args.reseed), replace=False):
        eng.synth_fill(0, int(lay["file_off"][k]), fb, 0xB000 + int(k))
    eng.sync()

    # ---- gate ----
    res_p, _ = session(False)
    ends_p, dig_p = eng.get_chunks(res_p.n_chunks)
    tab_p = eng.get_table(res_p.n_unique)
    res_g, _ = session(True)
    ends_g, dig_g = eng.get_chunks(res_g.n_chunks)
    tab_g = eng.get_table(res_g.n_unique)
    fields = ("crc_pure", "crc_bytes", "cdc_bytes", "n_files", "n_chunks", "n_unique")
    batch_ok = all(getattr(res_p, f) == getattr(res_g, f) for f in fields) and bytes(res_p.root) == bytes(res_g.root) and \
        np.array_equal(ends_p, ends_g) and np.array_equal(dig_p, dig_g) and np.array_equal(tab_p, tab_g)
    n = int(res_g.n_chunks)
    cg = eng.chunk_groups(n)
    gres = eng.group_results(G)
    want_tabs = ref.group_tables(dig_g, cg, G)
    tables_ok = True
    for g in range(G):
        t = eng.group_table(g, gres[g].n_unique)
        tables_ok &= bool(np.array_equal(t, want_tabs[g])) and bytes(gres[g].root) == ref_merkle(t) and \
            gres[g].n_chunks == int((cg == g).sum())
    tables_ok &= sum(r.n_files for r in gres) == res_g.n_files and sum(r.cdc_bytes for r in gres) == res_g.cdc_bytes
    extra = np.random.default_rng(0x4A).integers(0, 256, (3 * len(table_a), 32), dtype=np.uint8)
    rows_4x = cd.union(table_a, extra)
    # chunk lengths: files are back to back and every chunk ends inside its file
    e64 = ends_g.astype(np.int64)
    file_start = (e64 - 1) // fb * fb
    same_file = np.r_[False, file_start[1:] == file_start[:-1]]
    lens = np.where(same_file, e64 - np.r_[0, e64[:-1]], e64 - file_start).astype(np.uint64)
    with ChunkIndex(eng, len(rows_4x)) as ix:
        ix.add_rows(eng, rows_4x)
        dg = eng.delta_groups(ix, G)
        st = eng.chunk_status(n)
        want = ref.classify_groups(dig_g, cg, rows_4x)
        delta_ok = bool(np.array_equal(st, want)) and bool(np.array_equal(ix.get(eng), rows_4x))
        for g in range(G):
            c = cd.counts(want[cg == g], lens[cg == g])
            o = dg[g]
            delta_ok &= (o.known_chunks, o.new_chunks, o.repeat_chunks, o.known_bytes, o.new_bytes, o.repeat_bytes) == \
                (c["known_chunks"], c["new_chunks"], c["repeat_chunks"], c["known_bytes"], c["new_bytes"], c["repeat_bytes"])
        delta_ok &= sum(o.known_bytes + o.new_bytes + o.repeat_bytes for o in dg) == res_g.cdc_bytes
        gate = bool(batch_ok and tables_ok and delta_ok)
        out["gate_detail"] = {"batch": bool(batch_ok), "group_tables_and_roots": bool(tables_ok), "delta_groups": bool(delta_ok)}
        out["session"] = {"n_chunks": n, "n_unique": int(res_g.n_unique), "cdc_bytes": int(res_g.cdc_bytes), "groups": G,
                          "group_unique_rows_total": int(sum(r.n_unique for r in gres))}

        # ---- delta_groups timing (B is the finished grouped session) ----
        for _ in range(args.warmup):
            eng.delta_groups(ix, G)
        dev, host = [], []
        for _ in range(args.reps):
            t = time.perf_counter()
            r = eng.delta_groups(ix, G)
            host.append((time.perf_counter() - t) * 1e3)
            dev.append(r[0].ms_device)
        known = sum(o.known_chunks for o in dg) / n
        out["delta_groups"] = {"index_rows": len(rows_4x), "ms_device": stats(dev), "ms_host": stats(host),
                               "share_of_step_device": float(np.median(dev)) / args.step_ms, "target_ms_device": 0.5,
                               "known_frac": known}

    # ---- finish: grouped vs ungrouped, alternating ----
    fin = {False: [], True: []}
    for i in range(args.warmup + args.reps):
        for grouped in (False, True):
            _, ms = session(grouped)
            if i >= args.warmup:
                fin[grouped].append(ms)
    extra_ms = float(np.median(fin[True]) - np.median(fin[False]))
    out["finish"] = {"ungrouped_ms_host": stats(fin[False]), "grouped_ms_host": stats(fin[True]),
                     "grouped_minus_ungrouped_ms": extra_ms, "target_extra_ms": 1.5,
                     "extra_share_of_step": extra_ms / args.step_ms}
    out["gate"] = gate
    eng.close()
    os.dup2(real_stdout, 1)
    print(json.dumps(out), flush=True)
    return 0 if gate else 1


if __name__ == "__main__":
    sys.exit(main())
