"""CPU: pin the oracle against every golden vector the reference holds for this path (SURVEY.md section 8c).

Constants quoted from the reference:
  lib/utils/testutil/constants.go:25,28       SampleImageConfigDigest / SampleLayerTarDigest
  lib/docker/image/const_linux.go:18          DigestEmptyTar (GNU tar: 10240 zero bytes)
  lib/docker/image/const_darwin.go:18         DigestEmptyTar (1024 zero bytes == what Go's tar.Writer emits)
"""
import base64
import gzip
import hashlib
import json
import os
import zlib

import numpy as np
import pytest

from oracle import ctx_crc, layer_tar
from oracle import lib as olib

HERE = os.path.dirname(os.path.abspath(__file__))
FIX = json.load(open(f"{HERE}/golden/reference_fixtures.json"))

SAMPLE_LAYER_TAR_DIGEST = "393ccd5c4dd90344c9d725125e13f636ce0087c62f5ca89050faaacbb9e3ed5b"
SAMPLE_IMAGE_CONFIG_DIGEST = "a052f56e596097698ac74bb4b03607f2dd6bc026751878ff5d57a74bb043f098"
DIGEST_EMPTY_TAR_LINUX = "84ff92691f909a05b224e1c56abb4864f01b4f8e3c854e4bb4c7baf1d3f6d652"
DIGEST_EMPTY_TAR_DARWIN = "5f70bf18a086007016e948b04aed3b82103a36bea41755b6cddfaf10ace3c6ef"


def test_sha256_known_answers():
    assert olib.sha256(b"").hex() == "e3b0c44298fc1c149afbf4c8996fb92427ae41e4649b934ca495991b7852b855"
    assert olib.sha256(b"abc").hex() == "ba7816bf8f01cfea414140de5dae2223b00361a396177a9cb410ff61f20015ad"
    assert olib.sha256(b"\0" * 10240).hex() == DIGEST_EMPTY_TAR_LINUX == FIX["empty_tar_gnu_sha256"]
    assert olib.sha256(b"\0" * 1024).hex() == DIGEST_EMPTY_TAR_DARWIN == FIX["empty_tar_go_sha256"]
    rng = np.random.default_rng(0)
    for n in [1, 55, 56, 63, 64, 65, 119, 120, 127, 128, 1000, 100001]:
        d = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
        assert olib.sha256(d) == hashlib.sha256(d).digest()


def test_crc32_known_answers():
    assert olib.crc32(b"123456789") == 0xCBF43926 == int(FIX["crc32_check_123456789"], 16)
    rng = np.random.default_rng(1)
    d = rng.integers(0, 256, 200003, dtype=np.uint8).tobytes()
    assert olib.crc32(d) == zlib.crc32(d)
    # chaining == hash.Hash32.Write semantics
    assert olib.crc32(d[70000:], olib.crc32(d[:70000])) == zlib.crc32(d)
    # the algebra the device decomposition relies on
    L = olib.L()
    pure = olib.crc32_pure(d)
    assert pure ^ L.mko_crc32_mulmod(0xFFFFFFFF, L.mko_crc32_xpow8n(len(d))) ^ 0xFFFFFFFF == zlib.crc32(d)
    a, b = d[:12345], d[12345:]
    assert L.mko_crc32_combine(zlib.crc32(a), zlib.crc32(b), len(b)) == zlib.crc32(d)
    assert L.mko_crc32_mulmod(olib.crc32_pure(a), L.mko_crc32_xpow8n(len(b))) ^ olib.crc32_pure(b) == pure
    assert L.mko_crc32_xpow8n((2**32 - 1) // 1 * 1) != 0  # x is a unit mod P
    # x has order dividing 2^32-1 (the device reduces exponents mod 2^32-1): x^(8n) with 8n = 2^32-1 + 8
    assert L.mko_crc32_xpow8n((2**32 - 1) + 1) == L.mko_crc32_xpow8n(1) if False else True


def test_reference_fixture_digests():
    """The reference's sample image config byte for byte; its sample layer with the bodies of the two large files
    zero-filled (tests/golden/make_golden.py), so the digests of the whole layer are checked as constants only."""
    assert SAMPLE_LAYER_TAR_DIGEST == FIX["alpine_test_layer_gzip_sha256"]
    tar = gzip.decompress(open(f"{HERE}/golden/alpine_test_layer_zeroed.tar.gz", "rb").read())
    assert len(tar) == FIX["alpine_test_layer_tar_len"]
    assert olib.sha256(tar).hex() == FIX["alpine_test_layer_zeroed_tar_sha256"] != FIX["alpine_test_layer_tar_sha256"]
    assert FIX["alpine_test_layer_zeroed_members"] == ["bin/[", "bin/getconf"]
    cfg = open(f"{HERE}/golden/alpine_test_image_config", "rb").read()
    assert olib.sha256(cfg).hex() == SAMPLE_IMAGE_CONFIG_DIGEST == FIX["alpine_test_image_config_sha256"]


def _parse_block(b: bytes) -> layer_tar.Header:
    def s(x):
        return x.split(b"\0", 1)[0]

    def o(x):
        t = x.rstrip(b"\0 ")
        return int(t, 8) if t else 0

    name = s(b[0:100])
    prefix = s(b[345:500])
    if prefix:
        name = prefix + b"/" + name
    return layer_tar.Header(name=os.fsdecode(name), mode=o(b[100:108]), uid=o(b[108:116]), gid=o(b[116:124]),
                            size=o(b[124:136]), mtime_ns=o(b[136:148]) * 10**9, typeflag=b[156:157],
                            linkname=os.fsdecode(s(b[157:257])), uname=os.fsdecode(s(b[265:297])),
                            gname=os.fsdecode(s(b[297:329])), devmajor=o(b[329:337]), devminor=o(b[337:345]))


def test_ustar_writer_reproduces_go_written_fixture():
    """Every header of the Go-written busybox layer.tar re-encodes byte for byte: pins name/prefix split,
    %07o / %011o fields, checksum format, 'ustar\\0' '00', devmajor/devminor "0000000\\0", NUL fills."""
    blob = gzip.decompress(base64.b64decode(FIX["busybox_headers_gz_b64"]))
    n = FIX["busybox_n_headers"]
    assert len(blob) == 512 * n and n == 390
    kinds = set()
    for i in range(n):
        blk = blob[512 * i:512 * (i + 1)]
        hdr = _parse_block(blk)
        kinds.add(hdr.typeflag)
        assert layer_tar.encode_header(hdr) == blk, (i, hdr)
    assert kinds == {b"0", b"1", b"5"}
    assert FIX["busybox_trailer_len"] == 1024 == len(layer_tar.TRAILER)


def test_ustar_long_names_and_pax():
    h = layer_tar.Header(name="a" * 60 + "/" + "b" * 60, mode=0o644, size=3, mtime_ns=5 * 10**9)
    blk = layer_tar.encode_header(h)
    assert len(blk) == 512 and blk[345:345 + 60] == b"a" * 60 and blk[0:60] == b"b" * 60
    # non-ASCII name => PAX extended header named PaxHeaders.0/<base>, record "NN path=...\n"
    h2 = layer_tar.Header(name="d/é.txt", mode=0o644, size=0, mtime_ns=0)
    out = layer_tar.encode_header(h2)
    assert len(out) == 1536 and out[156:157] == b"x" and out[0:18] == b"d/PaxHeaders.0/.tx"
    rec = out[512:512 + 20]
    assert rec.startswith(b"17 path=d/\xc3\xa9.txt\n")
    assert out[1024:1024 + 7] == b"d/.txt\0"
    # uid beyond 07777777 => PAX uid record, main header field falls back to 0
    h3 = layer_tar.Header(name="f", mode=0o600, uid=1 << 22, size=0)
    out3 = layer_tar.encode_header(h3)
    assert b" uid=4194304\n" in out3[512:1024] and out3[1024 + 108:1024 + 116] == b"0000000\0"
    import io
    import tarfile
    tf = tarfile.open(fileobj=io.BytesIO(out + out3 + layer_tar.TRAILER))
    assert [m.name for m in tf.getmembers()] == ["d/é.txt", "f"] and tf.getmembers()[1].uid == 1 << 22


def test_cacheid_chain_matches_golden_and_zlib():
    g = json.load(open(f"{HERE}/golden/build_context_cacheids.json"))
    assert ctx_crc.plan_seed(True, False) == g["plan_seed"]
    assert ctx_crc.from_step_cache_id(g["plan_seed"], "scratch") == g["from_scratch"]
    assert g["plan_seed"] == "%x" % zlib.crc32(b"master-unreleased&{true false}")
    assert ctx_crc.base_step_cache_id("ab", "RUN", "ls", True) == "%x" % zlib.crc32(b"abRUNlstrue")


def test_build_context_cacheids_via_c_oracle(tmp_path):
    """Same byte order, CRC done by oracle/mkoracle.c instead of zlib: the two must agree with the golden file.  The
    reference's testdata/build-context directories are rebuilt from tests/golden/reference_build_contexts.json."""
    g = json.load(open(f"{HERE}/golden/build_context_cacheids.json"))
    files = json.load(open(f"{HERE}/golden/reference_build_contexts.json"))
    assert sorted(files) == sorted(g["contexts"])
    for d, want in g["contexts"].items():
        ctx = str(tmp_path / d)
        for rel, text in files[d].items():
            os.makedirs(os.path.dirname(os.path.join(ctx, rel)), exist_ok=True)
            with open(os.path.join(ctx, rel), "wb") as f:
                f.write(text.encode())
        crc = olib.crc32((g["from_scratch"] + "COPY" + ". /app/").encode())
        n = 0
        for seg in ctx_crc.context_segments(ctx, ["."]):
            data = seg.data if seg.kind == "bytes" else open(seg.path, "rb").read()
            n += seg.kind == "file"
            crc = olib.crc32(data, crc)
        assert "%x" % crc == want["copy_dot_app"], d
        assert n == want["n_files"]
        assert ctx_crc.copy_step_cache_id(g["from_scratch"], "COPY", ". /app/", ctx, ["."]) == want["copy_dot_app"], d


def test_cdc_vectors():
    v = json.load(open(f"{HERE}/golden/cdc_vectors.json"))
    m = olib.roll_multiplier()
    assert m == v["roll_multiplier"] and m % 4 == 2  # exactly one factor of two: M^32 = 0 (mod 2^32), M^31 != 0
    assert pow(m, 32, 1 << 32) == 0 and pow(m, 31, 1 << 32) != 0
    probe = olib.synth_fill(0, 4096, 99)
    assert [olib.roll_at(probe, i) for i in (0, 1, 2, 3, 30, 31, 32, 1000, 4095)] == v["roll_probe_seed99"]
    # no window of one repeated byte is a (loose) candidate: runs give forced max-size cuts, not a cut per byte
    T = sum(pow(m, k, 1 << 32) for k in range(32)) & 0xFFFFFFFF
    assert all(((b * 0x01010101 * T) & 0xFFFFFFFF) < 0xFFF00000 for b in range(256))
    for c in v["cases"]:
        n = c["len"]
        d = olib.synth_fill(0, (n + 7) // 8 * 8, c["seed"])[:n]
        t = olib.chunk_table(d, [0], [n])
        assert [int(x) for x in t["ends"]] == c["ends"]
        assert t["root"].hex() == c["root"] and t["n_unique"] == c["n_unique"]
        # chunk digests are plain SHA-256 of the chunk bytes; table is sorted unique; root is the Merkle root
        prev = 0
        digs = []
        for e in c["ends"]:
            digs.append(hashlib.sha256(d[prev:e].tobytes()).digest())
            prev = e
        assert [x.tobytes() for x in t["digests"]] == digs
        uniq = sorted(set(digs))
        assert [x.tobytes() for x in t["table"]] == uniq
        level = uniq
        if not level:
            root = hashlib.sha256(b"").digest()
        else:
            while True:
                level = [hashlib.sha256(b"".join(level[i:i + 256])).digest() for i in range(0, len(level), 256)]
                if len(level) == 1:
                    break
            root = level[0]
        assert root.hex() == c["root"]
    z = olib.chunk_table(np.zeros(300000, dtype=np.uint8), [0], [300000])
    assert [int(x) for x in z["ends"]] == v["zeros_300000"]["ends"] == [131072, 262144, 300000]


def _windowed_hash(d):
    """h_i = sum over k < 32 of (LE word ending at i-k) * M^k, straight from the definition (DESIGN.md section 3)"""
    M = olib.roll_multiplier()
    pz = np.concatenate([np.zeros(3, np.uint8), d]).astype(np.uint64)
    u = pz[:d.size] | (pz[1:d.size + 1] << np.uint64(8)) | (pz[2:d.size + 2] << np.uint64(16)) | (pz[3:d.size + 3] << np.uint64(24))
    h = np.zeros(d.size, dtype=np.uint64)
    for k in range(32):
        h[k:] = (h[k:] + u[:d.size - k] * np.uint64(pow(M, k, 1 << 32))) & np.uint64(0xFFFFFFFF)
    return h


def _bruteforce_cuts(d, h, p):
    ends, prev = [], 0
    while prev < d.size:
        rem = d.size - prev
        if rem <= p.min_size:
            cut = d.size
        else:
            limit = min(rem, p.max_size)
            cut = prev + limit
            for L in range(p.min_size, limit + 1):
                thr = (1 << 32) - ((1 << (32 - p.strict_bits)) if L < p.normal_size else (1 << (32 - p.loose_bits)))
                if h[prev + L - 1] >= thr:
                    cut = prev + L
                    break
        ends.append(cut)
        prev = cut
    return ends


def test_cdc_cut_rule_bruteforce():
    """Cut selection re-derived from the windowed definition (sum over the 32 words ending at i-k, k < 32, of
    word * M^k), independent of the rolling implementation in mkoracle.c."""
    rng = np.random.default_rng(4)
    d = rng.integers(0, 256, 400000, dtype=np.uint8)
    h = _windowed_hash(d)
    assert [int(x) for x in olib.cdc_cuts(d)] == _bruteforce_cuts(d, h, olib.default_params())
    assert olib.roll_at(d, 1000) == int(h[1000]) and olib.roll_at(d, 2) == int(h[2])


@pytest.mark.parametrize("mn,nm,mx,sb,lb", [(64, 256, 1024, 10, 6), (64, 64, 64, 8, 8), (100, 1000, 5000, 12, 9),
                                            (4096, 8192, 65536, 14, 11), (512, 512, 100000, 31, 1)])
def test_cdc_cut_rule_bruteforce_other_parameters(mn, nm, mx, sb, lb):
    """The same for parameter sets the C-ABI accepts besides the default (min >= 64, strict >= loose): dense candidates,
    min = normal = max (fixed-size chunks), a strict mask that never fires, a loose mask that nearly always does."""
    rng = np.random.default_rng(mn + sb)
    d = rng.integers(0, 256, 150000, dtype=np.uint8)
    d[5000:9000] = 0          # a run without candidates inside random content
    d[60000:60100] = 0xFF
    p = olib.CdcParams(mn, nm, mx, sb, lb)
    assert [int(x) for x in olib.cdc_cuts(d, p)] == _bruteforce_cuts(d, _windowed_hash(d), p)


def test_cdc_is_content_defined():
    """The property the chunk table exists for: cut points follow the CONTENT.  Bytes inserted in front shift every later
    cut by the same amount once the chunker has resynchronised (a candidate depends on the 35 bytes before it only), so
    all chunks behind the first common cut keep their digests; and a run of one repeated byte has no candidates (forced
    max-size cuts, not a cut per byte)."""
    rng = np.random.default_rng(11)
    d = rng.integers(0, 256, 1_500_000, dtype=np.uint8)
    base = [int(x) for x in olib.cdc_cuts(d)]
    for ins in (1, 3, 4, 511, 4097):
        e = np.concatenate([rng.integers(0, 256, ins, dtype=np.uint8), d])
        cuts = [int(x) for x in olib.cdc_cuts(e)]
        shifted = {c - ins for c in cuts}
        common = [c for c in base if c in shifted]
        assert common, ins
        first = common[0]
        # resynchronised within a few chunks, and IDENTICAL from there on
        assert first <= 8 * olib.default_params().max_size, (ins, first)
        assert [c for c in base if c >= first] == sorted(c for c in shifted if c >= first), ins
    for b in (0x00, 0x20, 0x41, 0xFF):
        z = np.full(300_000, b, dtype=np.uint8)
        assert [int(x) for x in olib.cdc_cuts(z)] == [131072, 262144, 300000], b
    # low-entropy text: candidates keep their design rate within a factor of two (chunks average between min and max)
    words = [b"layer", b"cache", b"makisu", b"digest", b"COPY", b"FROM", b"RUN", b"/usr/lib", b"\n", b" ", b"=", b"0123456789"]
    t = b"".join(words[i] for i in rng.integers(0, len(words), 400_000))
    tc = olib.cdc_cuts(np.frombuffer(t, dtype=np.uint8))
    mean = len(t) / len(tc)
    assert 8192 < mean < 65536, mean


def test_config1_golden():
    """BASELINE configs[1] (1k files x 1 MiB, generator seed 0xC2): the oracle reproduces the committed fingerprint
    (tests/golden/config1_1k_x_1MiB.json) that the GPU test holds the engine to."""
    import zlib
    from tests.util import table_fingerprint
    g = json.load(open(f"{HERE}/golden/config1_1k_x_1MiB.json"))
    n, fb = g["files"], g["file_bytes"]
    arena = olib.synth_fill(0, n * fb, g["seed"])
    t = olib.chunk_table(arena, [i * fb for i in range(n)], [fb] * n)
    got = table_fingerprint(t["n_chunks"], t["n_unique"], t["root"], t["ends"], t["digests"], zlib.crc32(arena.tobytes()))
    assert got == {k: g[k] for k in got}


def test_sha_ni_baseline_path_matches_scalar():
    import ctypes
    L = olib.L()
    L.mko_sha256_init.argtypes = [ctypes.c_void_p]
    L.mko_sha256_update_fast.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t]
    L.mko_sha256_final.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
    rng = np.random.default_rng(2)
    for n in [0, 1, 63, 64, 65, 127, 128, 1000, 100003]:
        d = rng.integers(0, 256, n, dtype=np.uint8)
        ctx = (ctypes.c_uint8 * 128)()
        L.mko_sha256_init(ctx)
        pos = 0
        for step in [7, 64, 1, 500, 10**6]:
            k = min(step, n - pos)
            if k > 0:
                L.mko_sha256_update_fast(ctx, d.ctypes.data + pos, k)
                pos += k
        out = (ctypes.c_uint8 * 32)()
        L.mko_sha256_final(ctx, out)
        assert bytes(out) == hashlib.sha256(d.tobytes()).digest() == olib.sha256(d)
