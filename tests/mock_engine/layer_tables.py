"""Entry point of a FRESH process (tests/test_host_layer_tables_cpu.py spawns it), like run.py: load the CPU mock of
the engine with the grouped-session calls (mock_mksnap_groups.cpp) with RTLD_GLOBAL first, so that libmkhost's
mksnap_* references bind to it, then commit a batch of layers with per-layer chunk tables.
    python -m tests.mock_engine.layer_tables <mock.so> <tmpdir>"""
import ctypes as C
import io
import os
import sys
import tarfile

import numpy as np


def batch_of_layers_with_layer_tables(make_engine, tmp):
    """mkhost_memfs_commit_layers(..., MKHOST_LAYER_TABLES): one grouped engine session (layer i = group i), and every
    layer's root / n_chunks / n_unique equal those of a separate commit_copy_ops of that layer (and the oracle's chunk
    table of its files); TarDigests and tar bytes stay what the ungrouped batch gives.  No chown: owners stay 0."""
    from makisu_b200 import host
    from oracle import layer_tar as lt
    from oracle import lib as olib
    from tests.mock_engine.scenarios import NOW, _ctx, _layer_expectations
    ctx = _ctx(tmp)
    root = os.path.join(tmp, "root")
    os.mkdir(root)
    os.chmod(root, 0o755)
    specs = [(["/d0"], "/app/d0/"), (["/d1", "/d2"], "/app/"), (["/big.bin"], "/data/big.bin"), (["/empty", "/zeros"], "/app/"),
             (["/d0"], "/app/d0/"),                                # identical to layer 0: only re-added ancestors remain
             (["/link"], "/app/")]
    o = lt.MemFS(lambda: NOW, root)
    want = []
    for srcs, dst in specs:
        entries = o.add_layer_by_copy_ops([lt.CopyOperation.new(srcs, ctx, "/", dst)])
        blob, table = _layer_expectations(entries)
        want.append((lt.tar_digest(entries), blob, table))
    ops = [[host.CopyOperation(s, ctx, "/", d)] for s, d in specs]
    # the separate commits: one session per layer, each diffed against the tree its predecessors left
    eng = make_engine(8 << 20)
    seq = host.MemFS(root)
    separate = [seq.commit_copy_ops(eng, NOW, layer) for layer in ops]
    seq.close()
    for arena_bytes in (2 << 20, 8 << 20):
        eng = make_engine(arena_bytes, n_host_arenas=2)
        h = host.MemFS(root)
        got = h.commit_layers(eng, NOW, ops, layer_tables=True)
        assert eng.n_groups == len(specs)
        for i, (dig, blob, table) in enumerate(want):
            assert got[i]["tar_digest"] == dig == separate[i]["tar_digest"], (i, arena_bytes)
            assert got[i]["tar_bytes"] == len(blob)
            for k in ("root", "n_chunks", "n_unique"):
                assert got[i][k] == separate[i][k], (i, k, arena_bytes)
            assert (got[i]["root"], got[i]["n_chunks"], got[i]["n_unique"]) == (table["root"], table["n_chunks"], table["n_unique"])
        h.close()
    assert len({g["root"] for g in got}) > 2                       # the layers really differ
    # without the flag: the batch's table under every layer, as before
    eng = make_engine(8 << 20)
    plain = host.MemFS(root).commit_layers(eng, NOW, ops)
    batch = olib.chunk_table(np.frombuffer(b"".join(w[1] for w in want), dtype=np.uint8), *_batch_files(want))
    assert all((p["root"], p["n_chunks"]) == (batch["root"], batch["n_chunks"]) for p in plain)
    assert [p["tar_digest"] for p in plain] == [g["tar_digest"] for g in got]


def _batch_files(want):
    """File offsets and lengths of the layer blobs laid end to end (for the batch's chunk table)."""
    offs, lens, base = [], [], 0
    for _, blob, _ in want:
        with tarfile.open(fileobj=io.BytesIO(blob)) as tf:
            for m in tf.getmembers():
                if m.isreg() and m.size:
                    offs.append(base + m.offset_data)
                    lens.append(m.size)
        base += len(blob)
    return offs, lens


def main():
    mock_path, tmp = sys.argv[1:3]
    mock = C.CDLL(mock_path, mode=C.RTLD_GLOBAL)          # BEFORE anything loads libmksnap / libmkhost
    from makisu_b200 import host
    from tests.mock_engine.scenarios import MockEngineFactory
    host.load()
    for name in ("mksnap_begin", "mksnap_begin_groups", "mksnap_arena_submit_groups", "mksnap_get_group_results"):
        ours = C.cast(getattr(mock, name), C.c_void_p).value
        seen = C.cast(getattr(C.CDLL(None), name), C.c_void_p).value
        assert ours == seen, "libmkhost is not bound to the mock engine (%s)" % name
    batch_of_layers_with_layer_tables(MockEngineFactory(mock), tmp)
    print("SCENARIO-OK batch_of_layers_with_layer_tables")


if __name__ == "__main__":
    main()
