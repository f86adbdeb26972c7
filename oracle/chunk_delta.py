"""CPU restatement of the chunk delta and the chunk-index union (test infrastructure only).

It consumes chunk digests the engine returned through mksnap_get_chunks (which the parity tests pin bit-exact to
oracle/mkoracle.c), so GPU-scale sessions can be checked without hashing on the CPU.  Frozen semantics (DESIGN.md
section 3b):
  - rows are ordered bytewise over all 32 bytes;
  - a chunk is KNOWN (0) if its digest is in the index, else NEW (1) at the lowest chunk position carrying the
    digest in the session, else REPEAT (2);
  - a union is the sorted set of index rows and incoming rows.
Digests are compared as numpy 32-byte void scalars, whose order is bytewise.
"""
from __future__ import annotations

import numpy as np

KNOWN, NEW, REPEAT = 0, 1, 2


def _v(rows) -> np.ndarray:
    a = np.ascontiguousarray(rows, dtype=np.uint8).reshape(-1, 32)
    return a.view("V32").ravel()


def _rows(v: np.ndarray) -> np.ndarray:
    return np.ascontiguousarray(v).view(np.uint8).reshape(-1, 32)


def contains(index_rows, digests) -> np.ndarray:
    """bool per digest: is it a row of the sorted-unique table `index_rows`?"""
    ix, d = _v(index_rows), _v(digests)
    if ix.size == 0 or d.size == 0:
        return np.zeros(d.size, dtype=bool)
    at = np.searchsorted(ix, d)
    hit = at < ix.size
    hit[hit] = ix[at[hit]] == d[hit]
    return hit


def classify(chunk_digests, index_rows) -> np.ndarray:
    """uint8 status per chunk, in chunk order."""
    d = _v(chunk_digests)
    status = np.full(d.size, REPEAT, dtype=np.uint8)
    if d.size == 0:
        return status
    _, first, inv = np.unique(d, return_index=True, return_inverse=True)
    status[np.arange(d.size) == first[inv.ravel()]] = NEW
    status[contains(index_rows, chunk_digests)] = KNOWN
    return status


def counts(status, chunk_lens) -> dict:
    """Per-class chunk and byte counts, named like mksnap_delta_result."""
    st = np.asarray(status)
    ln = np.asarray(chunk_lens, dtype=np.uint64)
    out = {}
    for name, k in (("known", KNOWN), ("new", NEW), ("repeat", REPEAT)):
        m = st == k
        out[name + "_chunks"] = int(m.sum())
        out[name + "_bytes"] = int(ln[m].sum())
    return out


def chunk_lens(ends, offs, lens) -> np.ndarray:
    """Chunk lengths from mksnap_get_chunks end offsets of one arena whose files start at `offs` and are `lens` long
    (files in ascending offset order): a chunk starts where the previous chunk of its file ended, or at its file."""
    e = np.asarray(ends, dtype=np.int64)
    o = np.asarray(offs, dtype=np.int64)
    fe = o + np.asarray(lens, dtype=np.int64)
    f = np.searchsorted(fe, e, side="left")          # file whose end is the first at or after the chunk end
    start = o[f].copy()
    same = np.zeros(e.size, dtype=bool)
    same[1:] = f[1:] == f[:-1]
    start[same] = e[:-1][same[1:]]
    return (e - start).astype(np.uint64)


def union(index_rows, rows) -> np.ndarray:
    """Sorted-unique rows of both inputs, as an (n, 32) uint8 array."""
    v = np.concatenate([_v(index_rows), _v(rows)])
    return _rows(np.unique(v))
