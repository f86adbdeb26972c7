"""Writes tests/golden/sha256_prefix32_twins.json: counters c whose 32-byte messages msg(c) = TAG + c (u64 little-endian)
have SHA-256 digests sharing their first 4 bytes (the 32-bit sort key of the table stages) with another counter's.

  python tests/golden/make_prefix_twins.py [output path]

SHA-256 of every msg(c), c in [0, BOUND), is hashed once and grouped by its first 4 bytes. Every group of three or
more is kept, and the first N_PAIRS groups of two in ascending order of their smaller counter. A file shorter than
the minimum chunk size is one chunk whose digest is the SHA-256 of its bytes, so each group gives the table stages
digests that tie on the sort key and differ after it. The output depends only on TAG, BOUND and N_PAIRS: running
this again reproduces the committed file byte for byte.
"""
import hashlib
import json
import os
import struct
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
TAG = b"makisu-b200 prefix twin "   # 24 bytes; msg(c) is 32 bytes
BOUND = 1 << 24
N_PAIRS = 9000


def msg(c: int) -> bytes:
    return TAG + struct.pack("<Q", c)


def main(path):
    assert len(TAG) == 24
    key = np.empty(BOUND, dtype=np.uint32)
    h, pack = hashlib.sha256, struct.Struct("<Q").pack
    for c in range(BOUND):
        key[c] = int.from_bytes(h(TAG + pack(c)).digest()[:4], "big")
    order = np.argsort(key, kind="stable")          # equal keys keep ascending counters
    k = key[order]
    starts = np.flatnonzero(np.r_[True, k[1:] != k[:-1]])
    lens = np.diff(np.r_[starts, BOUND])
    groups = [order[s:s + n].tolist() for s, n in zip(starts, lens) if n >= 2]
    groups.sort(key=lambda g: g[0])
    pairs = [g for g in groups if len(g) == 2]
    triples = [g for g in groups if len(g) >= 3]
    out = {
        "tag": TAG.decode("ascii"),
        "bound": BOUND,
        "message": "tag bytes followed by the counter as u64 little-endian",
        "pairs_found": len(pairs),
        "pairs": pairs[:N_PAIRS],
        "triples": triples,
    }
    with open(path, "w") as f:
        json.dump(out, f, separators=(",", ":"))
        f.write("\n")
    print(f"{path}: {min(len(pairs), N_PAIRS)} of {len(pairs)} pairs, {len(triples)} groups of 3 or more")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "sha256_prefix32_twins.json"))
