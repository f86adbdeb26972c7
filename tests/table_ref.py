"""Plain references for the table stages, written straight from DESIGN.md section 3 with hashlib and Python sets, and
the prefix-twin fixture (tests/golden/sha256_prefix32_twins.json, written by tests/golden/make_prefix_twins.py)."""
from __future__ import annotations

import functools
import hashlib
import json
import os
import struct

import numpy as np

TWINS_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sha256_prefix32_twins.json")


def _as_bytes(rows):
    if isinstance(rows, np.ndarray):
        return [r.tobytes() for r in np.ascontiguousarray(rows, dtype=np.uint8).reshape(-1, 32)]
    return [bytes(r) for r in rows]


def ref_table(digests) -> list:
    """Table = bytewise-sorted unique digests, as a list of 32-byte strings."""
    return sorted(set(_as_bytes(digests)))


def ref_merkle(table) -> bytes:
    """Root = fan-out-256 Merkle: level_{k+1}[j] = SHA256(level_k[256j : 256j+256]), hashed at least once and until
    one digest remains; SHA256("") for an empty table."""
    level = _as_bytes(table)
    if not level:
        return hashlib.sha256(b"").digest()
    while True:
        level = [hashlib.sha256(b"".join(level[j:j + 256])).digest() for j in range(0, len(level), 256)]
        if len(level) == 1:
            return level[0]


def rows(table) -> np.ndarray:
    """A list of 32-byte strings as an (n, 32) uint8 array."""
    return np.frombuffer(b"".join(table), dtype=np.uint8).reshape(-1, 32).copy()


NEAR_TWIN_BYTES = (31, 30, 24, 16, 15, 8, 7, 4, 3, 0)   # last and first byte of each 64-bit word, and a few inside


def near_twins(table, positions=NEAR_TWIN_BYTES) -> list:
    """Rows equal to a row of `table` except one byte at `positions`, changed by +1 and by -1 (mod 256), that are not
    rows of `table` themselves: sorted and unique."""
    tab = set(_as_bytes(table))
    out = set()
    for r in tab:
        for j in positions:
            for d in (1, 255):
                b = bytearray(r)
                b[j] = (b[j] + d) & 0xFF
                out.add(bytes(b))
    return sorted(out - tab)


@functools.lru_cache(maxsize=None)
def _fixture():
    with open(TWINS_PATH) as f:
        return json.load(f)


def msg(c: int) -> bytes:
    """The 32-byte message of counter c: the fixture's tag, then c as a u64 little-endian."""
    return _fixture()["tag"].encode("ascii") + struct.pack("<Q", c)


def twins(kind: str = "pairs") -> list:
    """Groups of counters ("pairs" or "triples") whose messages' SHA-256 digests share their first 4 bytes, each
    group in ascending order of its digests: [[(counter, digest), ...], ...]."""
    out = []
    for g in _fixture()[kind]:
        out.append(sorted(((c, hashlib.sha256(msg(c)).digest()) for c in g), key=lambda t: t[1]))
    return out
