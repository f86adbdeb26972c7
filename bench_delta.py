#!/usr/bin/env python
"""bench_delta.py -- cost of the chunk delta and the chunk-index union on the flagship context.

  python bench_delta.py --reps 20 --warmup 3          (C3: 100k files x 512 KiB, device resident)

Workload (BASELINE configs[2], the layout of bench.py's context_layout): session A fills the index; session B is A with
10 % of the files re-seeded on the device (synth_fill), i.e. a layer whose content mostly exists already.  B is
classified against three indexes: empty, A's table (1x), and A's table plus 3x as many random rows (4x).  The union
adds B's table to the 4x index.  configs[4] (dup, 80 % repeated files) against an empty index must give
new_chunks / n_chunks = its dedup ratio (0.2000).

Before anything is timed every status vector and count is checked against oracle/chunk_delta.py on B's downloaded
digests ("gate").  Delta: ms_device (CUDA events around the delta's kernels) and a host clock around the call (which
ends in a device synchronize).  Union: host clock around mksnap_index_add_table on a fresh copy of the 4x index each
repetition.  Median, min and max over --reps after --warmup.  Prints one JSON line; writes nothing in the tree.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time
from types import SimpleNamespace

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from bench import context_layout, ext_ptr, special_layout  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, pl = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": pl}
    except Exception as ex:  # noqa: BLE001
        return {"name": None, "power_limit": None, "error": str(ex)}


def stats(xs):
    a = np.asarray(xs, dtype=np.float64)
    return {"median": float(np.median(a)), "min": float(a.min()), "max": float(a.max()), "n": int(a.size)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--files", type=int, default=100_000)
    ap.add_argument("--file-kib", type=int, default=512)
    ap.add_argument("--dirs", type=int, default=256)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--union-reps", type=int, default=7)
    ap.add_argument("--reseed", type=float, default=0.10)
    ap.add_argument("--step-ms", type=float, default=73.0, help="the C3 step time the shares are quoted against")
    args = ap.parse_args()
    real_stdout = os.dup(1)
    os.dup2(2, 1)  # library chatter goes to stderr; the JSON line alone to stdout

    from makisu_b200.abi import ChunkIndex, Engine
    from oracle import chunk_delta as cd

    fb = args.file_kib << 10
    lay = context_layout(args.files, fb, args.dirs, 0)
    ext, used = lay["ext"], lay["used"]
    n_ext = len(ext)
    arena_bytes = (used + (1 << 20)) // 512 * 512
    out = {"metric": "chunk_delta", "card": card(),
           "workload": f"{args.files} files x {args.file_kib} KiB device resident (BASELINE configs[2]); "
                       f"B = A with {args.reseed:.0%} of the files re-seeded"}
    eng = Engine(device=0, device_arena_bytes=arena_bytes, n_host_arenas=0, max_extents=n_ext + 16,
                 max_chunks=max(arena_bytes, lay["data_bytes"]) // 4096 + n_ext + 1024)

    def session():
        t = time.perf_counter()
        eng.begin()
        eng.lib.mksnap_device_submit(eng.h, 0, used, ext_ptr(ext), n_ext, None, 0)
        res = eng.finish()
        return res, (time.perf_counter() - t) * 1e3

    eng.synth_fill(0, 0, (lay["data_bytes"] + 15) // 16 * 16, 0xC3)
    eng.device_upload(0, lay["meta_base"], np.frombuffer(lay["blob"], dtype=np.uint8))
    eng.sync()
    res_a, _ = session()
    table_a = eng.get_table(res_a.n_unique)
    rng = np.random.default_rng(0xDE17A)
    for k in rng.choice(args.files, int(args.files * args.reseed), replace=False):
        eng.synth_fill(0, int(lay["file_off"][k]), fb, 0xB000 + int(k))
    eng.sync()
    steps = [session()[1] for _ in range(3)]
    res_b, _ = session()
    _, dig_b = eng.get_chunks(res_b.n_chunks)
    table_b = eng.get_table(res_b.n_unique)
    out["session"] = {"n_chunks_a": int(res_a.n_chunks), "n_unique_a": int(res_a.n_unique),
                      "n_chunks_b": int(res_b.n_chunks), "n_unique_b": int(res_b.n_unique),
                      "cdc_bytes_b": int(res_b.cdc_bytes), "step_ms_host": stats(steps)}

    extra = np.random.default_rng(0x4A).integers(0, 256, (3 * len(table_a), 32), dtype=np.uint8)
    rows_4x = cd.union(table_a, extra)
    indexes = {"0": table_a[:0], "1x": table_a, "4x": rows_4x}
    delta_out, gate = {}, True
    for name, rows in indexes.items():
        with ChunkIndex(eng, max(1, len(rows))) as ix:
            ix.add_rows(eng, rows)
            d = eng.delta(ix)
            st = eng.chunk_status(res_b.n_chunks)
            want = cd.classify(dig_b, rows)
            ok = bool(np.array_equal(st, want)) and (d.known_chunks, d.new_chunks, d.repeat_chunks) == tuple(
                int((want == k).sum()) for k in (0, 1, 2)) and \
                d.known_bytes + d.new_bytes + d.repeat_bytes == res_b.cdc_bytes and \
                d.new_chunks == res_b.n_unique - int(cd.contains(rows, table_b).sum())
            gate &= ok
            for _ in range(args.warmup):
                eng.delta(ix)
            dev, host = [], []
            for _ in range(args.reps):
                t = time.perf_counter()
                r = eng.delta(ix)
                host.append((time.perf_counter() - t) * 1e3)
                dev.append(r.ms_device)
            n = res_b.n_chunks
            delta_out[name] = {"index_rows": int(d.index_rows), "gate": ok, "ms_device": stats(dev), "ms_host": stats(host),
                               "share_of_step_device": float(np.median(dev)) / args.step_ms,
                               "known_frac": d.known_chunks / n, "new_frac": d.new_chunks / n, "repeat_frac": d.repeat_chunks / n,
                               "new_bytes": int(d.new_bytes)}
    out["delta"] = delta_out

    # union: B's table into a fresh copy of the 4x index per repetition
    want_union = cd.union(rows_4x, table_b)
    union_ms, union_ok = [], True
    for i in range(args.warmup + args.union_reps):
        with ChunkIndex(eng, len(rows_4x) + len(table_b)) as ix:
            ix.add_rows(eng, rows_4x)
            eng.sync()
            t = time.perf_counter()
            ix.add_table(eng)
            ms = (time.perf_counter() - t) * 1e3
            if i == 0:
                union_ok = bool(np.array_equal(ix.get(eng), want_union))
            if i >= args.warmup:
                union_ms.append(ms)
    gate &= union_ok
    out["union"] = {"index_rows": len(rows_4x), "added_rows": int(res_b.n_unique), "result_rows": len(want_union),
                    "gate": union_ok, "ms_host": stats(union_ms),
                    "share_of_step": float(np.median(union_ms)) / args.step_ms}

    # dup (configs[4]) against an empty index: new / chunks = the dedup ratio
    dargs = SimpleNamespace(files=args.files, file_kib=args.file_kib, dirs=args.dirs, workload="dup")
    dl, _ = special_layout(dargs, 0, 1)
    eng.synth_fill(0, 0, (dl["fill_bytes"] + 15) // 16 * 16, 0x5C0)
    eng.device_upload(0, dl["meta_base"], np.frombuffer(dl["blob"], dtype=np.uint8))
    eng.sync()
    eng.begin()
    eng.lib.mksnap_device_submit(eng.h, 0, dl["used"], ext_ptr(dl["ext"]), len(dl["ext"]), None, 0)
    rd = eng.finish()
    with ChunkIndex(eng, 1) as ix0:
        dd = eng.delta(ix0)
    dup_ok = dd.new_chunks == rd.n_unique and dd.known_chunks == 0
    gate &= dup_ok
    out["dup_empty_index"] = {"n_chunks": int(rd.n_chunks), "new_chunks": int(dd.new_chunks),
                              "new_over_chunks": dd.new_chunks / rd.n_chunks, "gate": dup_ok}
    out["gate"] = bool(gate)
    eng.close()
    os.dup2(real_stdout, 1)
    print(json.dumps(out), flush=True)
    return 0 if gate else 1


if __name__ == "__main__":
    sys.exit(main())
