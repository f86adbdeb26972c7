"""Generates the files under tests/golden/ from the fixtures of a makisu checkout (uber/makisu @5fdc8f4).  The tests
read only what this writes, so they run without that checkout.

  python tests/golden/make_golden.py <path of the makisu checkout>

- reference_fixtures.json: SHA-256 / CRC values the reference's tests pin (SURVEY.md section 8c) plus, for the
  Go-written USTAR fixture testdata/files/busybox/393c.../layer.tar, a per-header digest list so the header
  re-encoding test has something to chew on without the 1.3 MB tarball.
- alpine_test_image_config: testdata/files/alpine/test_image_config, byte for byte.
- alpine_test_layer_zeroed.tar.gz: the Go-written tar inside testdata/files/alpine/test_layer.tar with the bodies of
  its two large files (alpine_test_layer_zeroed_members) zero-filled: every header, hard link and small body as in
  the original, 6 KB instead of 660 KB.
- reference_build_contexts.json: the files of every testdata/build-context/* directory (relative path -> text).
- build_context_cacheids.json: cacheIDs of every testdata/build-context/* directory under `COPY . /app/`,
  computed with Python's zlib.crc32 (independent of oracle/mkoracle.c) in the reference byte order.
- cdc_vectors.json: Roll-32 multiplier / cut points / table roots of seeded inputs (our frozen spec).
"""
import base64
import gzip
import hashlib
import io
import json
import os
import sys
import tarfile
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import ctx_crc, lib as olib  # noqa: E402

ZEROED_ABOVE = 4096  # regular files of the alpine layer larger than this are zero-filled in the stored copy


def zeroed_layer(tar: bytes):
    """(the tar with the bodies of its regular files above ZEROED_ABOVE bytes zero-filled, their names)"""
    out, names = bytearray(tar), []
    for m in tarfile.open(fileobj=io.BytesIO(tar)).getmembers():
        if m.isreg() and m.size > ZEROED_ABOVE:
            out[m.offset_data:m.offset_data + m.size] = bytes(m.size)
            names.append(m.name)
    return bytes(out), names


def main(ref):
    out = {}
    p = f"{ref}/testdata/files/alpine/test_layer.tar"
    gz = open(p, "rb").read()
    out["alpine_test_layer_gzip_sha256"] = hashlib.sha256(gz).hexdigest()
    tar = gzip.decompress(gz)
    out["alpine_test_layer_tar_sha256"] = hashlib.sha256(tar).hexdigest()
    out["alpine_test_layer_tar_len"] = len(tar)
    busy = open(f"{ref}/testdata/files/busybox/393ccd5c4dd90344c9d725125e13f636ce0087c62f5ca89050faaacbb9e3ed5b/layer.tar", "rb").read()
    assert busy == tar
    cfg = open(f"{ref}/testdata/files/alpine/test_image_config", "rb").read()
    out["alpine_test_image_config_sha256"] = hashlib.sha256(cfg).hexdigest()
    open(f"{HERE}/alpine_test_image_config", "wb").write(cfg)
    zeroed, names = zeroed_layer(tar)
    out["alpine_test_layer_zeroed_members"] = names
    out["alpine_test_layer_zeroed_tar_sha256"] = hashlib.sha256(zeroed).hexdigest()
    open(f"{HERE}/alpine_test_layer_zeroed.tar.gz", "wb").write(gzip.compress(zeroed, 9, mtime=0))
    out["empty_tar_go_sha256"] = hashlib.sha256(b"\0" * 1024).hexdigest()
    out["empty_tar_gnu_sha256"] = hashlib.sha256(b"\0" * 10240).hexdigest()
    out["crc32_check_123456789"] = "%08x" % zlib.crc32(b"123456789")
    # header blocks of the Go-written fixture, base64 (390 x 512 B = 200 KB -> keep raw, gz+b64 ~ 12 KB)
    hdrs, pos = [], 0
    while pos + 512 <= len(tar):
        blk = tar[pos:pos + 512]
        if blk == b"\0" * 512:
            break
        size = int(blk[124:135].rstrip(b"\0 ") or b"0", 8)
        hdrs.append(blk)
        pos += 512 + (size + 511) // 512 * 512
    out["busybox_n_headers"] = len(hdrs)
    out["busybox_trailer_len"] = len(tar) - pos
    out["busybox_headers_gz_b64"] = base64.b64encode(gzip.compress(b"".join(hdrs), 9, mtime=0)).decode()
    json.dump(out, open(f"{HERE}/reference_fixtures.json", "w"), indent=1, sort_keys=True)

    ids, files = {}, {}
    base = f"{ref}/testdata/build-context"
    seed0 = ctx_crc.plan_seed(True, False)
    seed1 = ctx_crc.from_step_cache_id(seed0, "scratch")
    for d in sorted(os.listdir(base)):
        ctx = os.path.join(base, d)
        n_files = sum(len(f) for _, _, f in os.walk(ctx))
        ids[d] = {"copy_dot_app": ctx_crc.copy_step_cache_id(seed1, "COPY", ". /app/", ctx, ["."]), "n_files": n_files}
        files[d] = {os.path.relpath(os.path.join(p, f), ctx): open(os.path.join(p, f), "rb").read().decode()
                    for p, _, fs in os.walk(ctx) for f in fs}
    json.dump({"plan_seed": seed0, "from_scratch": seed1, "contexts": ids},
              open(f"{HERE}/build_context_cacheids.json", "w"), indent=1, sort_keys=True)
    json.dump(files, open(f"{HERE}/reference_build_contexts.json", "w"), indent=1, sort_keys=True)

    probe = olib.synth_fill(0, 4096, 99)
    vec = {"roll_multiplier": olib.roll_multiplier(),
           "roll_probe_seed99": [olib.roll_at(probe, i) for i in (0, 1, 2, 3, 30, 31, 32, 1000, 4095)], "cases": []}
    for seed, n in [(1, 0), (2, 100), (3, 4096), (4, 4097), (5, 100000), (6, 1 << 20), (7, 3000001)]:
        d = olib.synth_fill(0, (n + 7) // 8 * 8, seed)[:n]
        t = olib.chunk_table(d, [0], [n])
        vec["cases"].append({"seed": seed, "len": n, "ends": [int(x) for x in t["ends"]],
                             "n_unique": t["n_unique"], "root": t["root"].hex(),
                             "first_digest": t["digests"][0].tobytes().hex() if t["n_chunks"] else ""})
    z = np.zeros(300000, dtype=np.uint8)
    t = olib.chunk_table(z, [0], [z.size])
    vec["zeros_300000"] = {"ends": [int(x) for x in t["ends"]], "n_unique": t["n_unique"], "root": t["root"].hex()}
    json.dump(vec, open(f"{HERE}/cdc_vectors.json", "w"), indent=1, sort_keys=True)

    # BASELINE configs[1] exactly (1k files x 1 MiB, device generator seed 0xC2): what the GPU test diffs against
    n, fb = 1000, 1 << 20
    arena = olib.synth_fill(0, n * fb, 0xC2)
    t = olib.chunk_table(arena, [i * fb for i in range(n)], [fb] * n)
    c1 = {"files": n, "file_bytes": fb, "seed": 0xC2, "n_chunks": t["n_chunks"], "n_unique": t["n_unique"], "root": t["root"].hex(),
          "crc32_of_content": zlib.crc32(arena.tobytes()),
          "sha256_of_chunk_ends_u64le": hashlib.sha256(np.asarray(t["ends"], dtype=np.uint64).tobytes()).hexdigest(),
          "sha256_of_chunk_digests": hashlib.sha256(np.ascontiguousarray(t["digests"]).tobytes()).hexdigest(),
          "first_ends": [int(x) for x in t["ends"][:4]]}
    json.dump(c1, open(f"{HERE}/config1_1k_x_1MiB.json", "w"), indent=1, sort_keys=True)
    print("wrote", os.listdir(HERE))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
