"""CPU restatement of grouped sessions (DESIGN.md section 3c), test infrastructure only, in numpy on top of
oracle/chunk_delta.py.  Like that oracle it consumes chunk digests the engine returned (mksnap_get_chunks) together
with the group of every chunk (mksnap_get_chunk_groups), so GPU-scale grouped sessions can be checked without hashing
on the CPU.

  - group g's table is the bytewise-sorted unique digests of the chunks tagged g;
  - the grouped delta equals "for g in 0..G-1: classify(chunks of g, index) -> index = union(index, table of g)":
    a chunk of group g is KNOWN if its digest is in the index or occurs in a group < g, NEW at the lowest position of
    group g carrying the digest, REPEAT otherwise.
"""
from __future__ import annotations

import numpy as np

from oracle.chunk_delta import KNOWN, NEW, REPEAT, contains  # noqa: F401  (re-exported for the tests)


def _v(rows) -> np.ndarray:
    return np.ascontiguousarray(rows, dtype=np.uint8).reshape(-1, 32).view("V32").ravel()


def _groups(groups, n) -> np.ndarray:
    g = np.asarray(groups, dtype=np.int64).ravel()
    assert g.size == n, "one group per chunk"
    return g


def group_tables(digests, groups, n_groups: int | None = None) -> list:
    """One (n_g, 32) uint8 array per group: the sorted-unique digests of its chunks."""
    d = _v(digests)
    g = _groups(groups, d.size)
    G = int(n_groups if n_groups is not None else (g.max() + 1 if g.size else 0))
    out = []
    for k in range(G):
        u = np.unique(d[g == k])
        out.append(np.ascontiguousarray(u).view(np.uint8).reshape(-1, 32))
    return out


def classify_groups(digests, groups, index_rows) -> np.ndarray:
    """uint8 status per chunk, in chunk order (the order of mksnap_get_chunks)."""
    d = _v(digests)
    g = _groups(groups, d.size)
    status = np.full(d.size, REPEAT, dtype=np.uint8)
    if d.size == 0:
        return status
    pos = np.arange(d.size)
    # the first chunk of every digest in (group, position) order: its group is the lowest carrying the digest
    order = np.lexsort((pos, g, d))
    ds = d[order]
    head = np.ones(d.size, dtype=bool)
    head[1:] = ds[1:] != ds[:-1]
    run = np.cumsum(head) - 1                    # digest run of each sorted chunk
    first = order[head][run]                     # per sorted chunk: the first chunk of its digest
    first_of = np.empty(d.size, dtype=np.int64)
    first_of[order] = first
    status[pos == first_of] = NEW
    status[g > g[first_of]] = KNOWN
    status[contains(index_rows, digests)] = KNOWN
    return status
