"""Scenarios run against the CPU mock engine (see run.py).  They drive the real libmkhost packers -- layer commit over
several arenas, tar ingest, per-file digests, untar / materialise from the arena, content-aware scan -- and check the
results against the oracle, exactly like the -m gpu host tests do on a B200."""
import ctypes as C
import hashlib
import io
import os
import stat
import tarfile

import numpy as np

from makisu_b200 import abi, host
from oracle import copier as oc
from oracle import ctx_crc
from oracle import layer_tar as lt
from oracle import lib as olib

NOW = 1_600_000_000
T = 1_500_000_000


class MockEngine:
    def __init__(self, mock, host_arena_bytes, n_host_arenas=2, max_extents=1 << 12):
        self.mock = mock
        cfg = abi.Config()
        cfg.device, cfg.n_host_arenas, cfg.host_arena_bytes = 0, n_host_arenas, host_arena_bytes
        cfg.device_arena_bytes, cfg.max_extents = host_arena_bytes, max_extents
        self.h = C.c_void_p()
        mock.mksnap_create.argtypes = [C.POINTER(abi.Config), C.POINTER(C.c_void_p)]
        assert mock.mksnap_create(C.byref(cfg), C.byref(self.h)) == 0
        mock.mock_submits.restype = C.c_uint64
        mock.mock_submits.argtypes = [C.c_void_p]

    def submits(self):
        return int(self.mock.mock_submits(self.h))


class MockEngineFactory:
    def __init__(self, mock):
        self.mock = mock

    def __call__(self, host_arena_bytes, **kw):
        return MockEngine(self.mock, host_arena_bytes, **kw)


def _mk(root, rel, data=b"", mode=0o644, mtime=T):
    p = os.path.join(root, rel)
    os.makedirs(os.path.dirname(p), exist_ok=True)
    with open(p, "wb") as f:
        f.write(data)
    os.chmod(p, mode)
    os.utime(p, (mtime, mtime))
    return p


def _ctx(tmp, seed=42):
    c = os.path.join(tmp, "ctx")
    rng = np.random.default_rng(seed)
    _mk(c, "Dockerfile", b"FROM scratch\nCOPY . /app/\n")
    for d in range(3):
        for i in range(6):
            _mk(c, f"d{d}/f{i:03d}.bin", rng.integers(0, 256, int(rng.integers(0, 300_000)), dtype=np.uint8).tobytes())
    _mk(c, "big.bin", rng.integers(0, 256, 1_500_000, dtype=np.uint8).tobytes())
    _mk(c, "empty", b"")
    _mk(c, "zeros", bytes(200_000))
    os.symlink("big.bin", os.path.join(c, "link"))
    for d, _, _ in os.walk(c):
        os.utime(d, (T, T))
    return c


def _tree(root, mtimes=False):
    out = {}
    for d, dirs, files in os.walk(root):
        for n in sorted(dirs + files):
            p = os.path.join(d, n)
            st = os.lstat(p)
            rel = os.path.relpath(p, root)
            if stat.S_ISLNK(st.st_mode):
                out[rel] = ("l", os.readlink(p), st.st_uid, st.st_gid)
            elif stat.S_ISDIR(st.st_mode):
                out[rel] = ("d", stat.S_IMODE(st.st_mode), st.st_uid, st.st_gid) + ((st.st_mtime_ns,) if mtimes else ())
            else:
                out[rel] = ("f", stat.S_IMODE(st.st_mode), st.st_uid, st.st_gid) + ((st.st_mtime_ns, st.st_nlink) if mtimes else ()) \
                    + (open(p, "rb").read(),)
    return out


def _layer_expectations(entries):
    blob = b"".join(lt.layer_tar_chunks(entries))
    arena = np.frombuffer(blob, dtype=np.uint8)
    offs, lens, pos = [], [], 0
    for e in entries:
        pos += len(lt.entry_header_bytes(e))
        if not e.whiteout and e.hdr.typeflag == lt.TYPE_REG and e.hdr.size:
            offs.append(pos)
            lens.append(e.hdr.size)
            pos += (e.hdr.size + 511) // 512 * 512
    return blob, olib.chunk_table(arena, offs, lens)


def cache_id_and_commit(make_engine, tmp):
    """cacheID through the packer (several arenas, files split across them) and a layer commit whose tar stream spans
    many arenas (stream continuation), with tar emission -- against the oracle."""
    ctx = _ctx(tmp)
    seed = ctx_crc.from_step_cache_id(ctx_crc.plan_seed(True, False), "scratch")
    eng = make_engine(1 << 20)                                    # 1 MiB arenas: big.bin alone needs two
    for args, paths in [(". /app/", ["."]), ("d1 d2 big.bin /x/", ["d1", "d2", "big.bin"]), ("d*/f00?.bin /y/", ["d*/f00?.bin"])]:
        assert host.copy_step_cache_id(eng, seed, "COPY", args, ctx, paths) == ctx_crc.copy_step_cache_id(seed, "COPY", args, ctx, paths)
    assert eng.submits() > 6
    root = os.path.join(tmp, "root")
    os.mkdir(root)
    os.chmod(root, 0o755)
    fs = lt.MemFS(lambda: NOW, root)
    entries = fs.add_layer_by_copy_ops([lt.CopyOperation.new(["/"], ctx, "/", "/app/", uid=3, gid=4)])
    blob, want = _layer_expectations(entries)
    for arena_bytes in (8 << 20, 2 << 20):                        # one arena / many arenas (big.bin = 1.5 MB fits 2 MiB)
        eng = make_engine(arena_bytes)
        tar_path = os.path.join(tmp, "layer%d.tar" % arena_bytes)
        with open(tar_path, "wb") as f:
            got = host.commit_copy_ops(eng, root, NOW, [host.CopyOperation(["/"], ctx, "/", "/app/", 3, 4)], tar_fd=f.fileno())
        assert open(tar_path, "rb").read() == blob
        assert got["tar_digest"] == "sha256:" + hashlib.sha256(blob).hexdigest() == lt.tar_digest(entries)
        assert (got["n_entries"], got["tar_bytes"]) == (len(entries), len(blob))
        assert (got["n_chunks"], got["n_unique"], got["root"]) == (want["n_chunks"], want["n_unique"], want["root"])
    assert eng.submits() >= 3
    # big.bin (1.5 MB) is larger than a 1 MiB arena: it travels in pieces (MKSNAP_X_MORE / MKSNAP_X_CONT, per-file
    # stream continued) and everything equals the single-arena result -- tario.WriteEntry copies any size (write.go:45)
    eng = make_engine(1 << 20)
    tar_path = os.path.join(tmp, "layer_split.tar")
    with open(tar_path, "wb") as f:
        got = host.commit_copy_ops(eng, root, NOW, [host.CopyOperation(["/"], ctx, "/", "/app/", 3, 4)], tar_fd=f.fileno())
    assert open(tar_path, "rb").read() == blob
    assert got["tar_digest"] == lt.tar_digest(entries) and (got["n_entries"], got["tar_bytes"]) == (len(entries), len(blob))
    assert (got["n_chunks"], got["n_unique"], got["root"]) == (want["n_chunks"], want["n_unique"], want["root"])
    h = host.MemFS(root)
    got = h.commit_copy_ops(make_engine(1 << 20), NOW, [host.CopyOperation(["/"], ctx, "/", "/app/", 3, 4)], flags=host.MKHOST_FILE_DIGESTS)
    assert got["root"] == want["root"] and h.file_digest("/app/big.bin") == hashlib.sha256(open(os.path.join(ctx, "big.bin"), "rb").read()).digest()
    try:                                                          # too small to carry a file across submits: refused loudly
        host.commit_copy_ops(make_engine(128 << 10), root, NOW, [host.CopyOperation(["/"], ctx, "/", "/app/", 3, 4)])
        raise AssertionError("expected a capacity error")
    except host.HostError as e:
        assert "exceeds the arena" in str(e)


def _base_tar(rng):
    buf = io.BytesIO()
    with tarfile.open(fileobj=buf, mode="w", format=tarfile.PAX_FORMAT) as tf:
        def add(name, type_=tarfile.REGTYPE, data=b"", link="", mode=0o644):
            ti = tarfile.TarInfo(name)
            ti.type, ti.mode, ti.mtime, ti.linkname, ti.uid, ti.gid = type_, mode, T, link, 7, 8
            ti.size = len(data) if type_ == tarfile.REGTYPE else 0
            tf.addfile(ti, io.BytesIO(data) if ti.size else None)
        add("usr/", tarfile.DIRTYPE, mode=0o755)
        add("usr/lib/", tarfile.DIRTYPE, mode=0o2755)
        shared = rng.integers(0, 256, 300_000, dtype=np.uint8).tobytes()
        for i in range(8):
            add(f"usr/lib/lib{i}.so", data=rng.integers(0, 256, int(rng.integers(1, 400_000)), dtype=np.uint8).tobytes(), mode=0o755)
        add("usr/lib/copy_a.bin", data=shared)
        add("usr/lib/" + "d" * 150 + "/", tarfile.DIRTYPE, mode=0o755)
        add("usr/lib/" + "d" * 150 + "/copy_b.bin", data=shared)
        add("usr/lib/alias.so", tarfile.LNKTYPE, link="usr/lib/lib0.so", mode=0o755)
        add("lib", tarfile.SYMTYPE, link="usr/lib", mode=0o777)
        add("etc/", tarfile.DIRTYPE, mode=0o755)
        add("etc/empty", data=b"")
        add("etc/.wh.stale", data=b"")
        add("dev/null", tarfile.CHRTYPE)
    return buf.getvalue()


def ingest_untar_and_file_digests(make_engine, tmp):
    """mkhost_memfs_update_from_tar: DiffID + chunk table over 1 MiB arenas, record padding after the end marker,
    a pipe as the source, per-file digests, and MKHOST_UNTAR writing the members from the arena."""
    rng = np.random.default_rng(5)
    data = _base_tar(rng)
    assert len(data) % 10240 == 0
    tar_path = os.path.join(tmp, "base.tar")
    open(tar_path, "wb").write(data)
    members = [m for m in lt.read_tar(data) if m.hdr.typeflag == lt.TYPE_REG and m.data_len]
    want = olib.chunk_table(np.frombuffer(data, dtype=np.uint8), [m.data_off for m in members], [m.data_len for m in members])
    # 1. untar=false, FILE_DIGESTS
    root = os.path.join(tmp, "r1")
    os.mkdir(root)
    o = lt.MemFS(lambda: NOW, root)
    want_layer = o.update_from_tar(data, remember=True)
    eng = make_engine(1 << 20)
    h = host.MemFS(root)
    with open(tar_path, "rb") as f:
        got = h.update_from_tar(eng, NOW, f.fileno(), flags=host.MKHOST_FILE_DIGESTS)
    assert eng.submits() >= 3
    assert got["tar_digest"] == "sha256:" + hashlib.sha256(data).hexdigest() and got["tar_bytes"] == len(data)
    assert got["n_entries"] == len(want_layer)
    assert (got["n_chunks"], got["n_unique"], got["root"]) == (want["n_chunks"], want["n_unique"], want["root"])
    assert got["n_unique"] < got["n_chunks"]
    for m in members:
        dst = lt.abs_path(m.hdr.name)
        assert h.file_digest(dst) == hashlib.sha256(data[m.data_off:m.data_off + m.data_len]).digest(), dst
    assert h.file_digest("/etc/empty") is None and h.file_digest("/usr") is None
    # 2. through a pipe, digest left to the caller
    r, w = os.pipe()
    import threading
    t = threading.Thread(target=lambda: (os.write(w, data), os.close(w)))
    t.start()
    piped = host.MemFS(root).update_from_tar(make_engine(1 << 20), NOW, r, flags=host.MKHOST_NO_TAR_DIGEST)
    t.join()
    os.close(r)
    assert piped["root"] == got["root"] and piped["tar_digest"] == "sha256:" + "00" * 32
    # 3. untar=true from the arena == the oracle's untar
    disks, counts = [], []
    for impl in ("oracle", "engine"):
        rr = os.path.join(tmp, "untar_" + impl)
        os.makedirs(os.path.join(rr, "etc"))
        open(os.path.join(rr, "etc", "stale"), "wb").write(b"to be whited out")
        os.chmod(os.path.join(rr, "etc"), 0o700)
        for d in (os.path.join(rr, "etc"), rr):
            os.utime(d, (1_400_000_000, 1_400_000_000))
        if impl == "oracle":
            counts.append(len(lt.MemFS(lambda: NOW, rr).update_from_tar(data, untar=True)))
        else:
            with open(tar_path, "rb") as f:
                g = host.MemFS(rr).update_from_tar(make_engine(1 << 20), NOW, f.fileno(), flags=host.MKHOST_UNTAR)
            assert g["tar_digest"] == got["tar_digest"] and g["root"] == got["root"]
            counts.append(g["n_entries"])
        disks.append(_tree(rr, mtimes=True))
    assert counts[0] == counts[1] and disks[0] == disks[1]
    assert "etc/stale" not in disks[1] and disks[1]["usr/lib/alias.so"][5] == 2
    # 4. a truncated blob is refused
    open(tar_path, "wb").write(data[:5000])
    try:
        with open(tar_path, "rb") as f:
            host.MemFS(root).update_from_tar(make_engine(1 << 20), NOW, f.fileno())
        raise AssertionError("expected unexpected EOF")
    except host.HostError as e:
        assert "unexpected EOF" in str(e)


def content_aware_scan(make_engine, tmp):
    """MKHOST_FILE_DIGESTS at commit, then MKHOST_SCAN_CONTENT: same-second same-size edits are caught; the digest pass
    streams a file larger than an arena across submits."""
    rng = np.random.default_rng(11)
    root = os.path.join(tmp, "root")
    _mk(root, "d/a.txt", b"A" * 5000)
    _mk(root, "d/b.bin", rng.integers(0, 256, 300_000, dtype=np.uint8).tobytes())
    _mk(root, "d/big.bin", rng.integers(0, 256, 2_500_000, dtype=np.uint8).tobytes())
    _mk(root, "e/c.txt", b"c")
    _mk(root, "e/empty", b"")
    for d, _, _ in os.walk(root):
        os.utime(d, (T, T))
    o = lt.MemFS(lambda: NOW, root)
    h = host.MemFS(root)
    eng = make_engine(4 << 20)
    l1 = o.add_layer_by_scan()
    o.remember_content(l1)
    g1 = h.commit_scan(eng, NOW, flags=host.MKHOST_FILE_DIGESTS)
    assert g1["tar_digest"] == lt.tar_digest(l1) and g1["n_entries"] == len(l1) == 7

    def edit(rel, off):
        p = os.path.join(root, rel)
        st = os.lstat(p)
        with open(p, "r+b") as f:
            f.seek(off)
            b = f.read(1)
            f.seek(off)
            f.write(bytes([b[0] ^ 0x5A]))
        os.utime(p, ns=(st.st_atime_ns, st.st_mtime_ns))
    edit("d/b.bin", 123_456)
    edit("d/big.bin", 2_499_999)
    assert o.add_layer_by_scan() == [] and h.commit_scan(eng, NOW)["n_entries"] == 0       # the reference misses it
    l3 = o.add_layer_by_scan(content_aware=True)
    o.remember_content(l3)
    assert [e.dst for e in l3] == ["/d", "/d/b.bin", "/d/big.bin"]
    g3 = h.commit_scan(eng, NOW, flags=host.MKHOST_SCAN_CONTENT)
    assert g3["n_entries"] == 3 and g3["tar_digest"] == lt.tar_digest(l3)
    small = make_engine(1 << 20)                                  # big.bin (2.5 MB) streams through 1 MiB arenas
    assert o.add_layer_by_scan(content_aware=True) == []
    assert h.commit_scan(small, NOW, flags=host.MKHOST_SCAN_CONTENT)["n_entries"] == 0
    assert small.submits() >= 4
    edit("d/big.bin", 0)
    l4 = o.add_layer_by_scan(content_aware=True)
    assert [e.dst for e in l4] == ["/d", "/d/big.bin"]
    g4 = h.commit_scan(small, NOW, flags=host.MKHOST_SCAN_CONTENT)   # the 2.5 MB entry is committed in pieces (1 MiB arenas)
    assert g4["n_entries"] == 2 and g4["tar_digest"] == lt.tar_digest(l4)
    assert h.file_digest("/d/big.bin") == hashlib.sha256(open(os.path.join(root, "d/big.bin"), "rb").read()).digest()


def materialize_from_the_arena(make_engine, tmp):
    """MKHOST_MATERIALIZE: the COPY step's file copy fed from the arena of the layer commit == CopyOperation.Execute by
    the oracle's Copier; the layer itself is unchanged."""
    rng = np.random.default_rng(3)
    ctx = os.path.join(tmp, "ctx")
    os.makedirs(os.path.join(ctx, "app", "sub"))
    for rel, n, mode in [("app/a.bin", 700_000, 0o644), ("app/sub/b.bin", 1_200_000, 0o755), ("app/empty", 0, 0o600), ("conf.txt", 900, 0o640)]:
        p = os.path.join(ctx, rel)
        open(p, "wb").write(rng.integers(0, 256, n, dtype=np.uint8).tobytes())
        os.chmod(p, mode)
        os.utime(p, (T, T))
    os.symlink("a.bin", os.path.join(ctx, "app", "link"))
    for d, _, _ in os.walk(ctx):
        os.utime(d, (T, T))
    roots = {k: os.path.join(tmp, k) for k in ("fused", "plain", "oracle")}
    for r in roots.values():
        os.mkdir(r)
        os.chmod(r, 0o755)
    ops = [host.CopyOperation(["/app"], ctx, "/", "/srv/app/", 5, 6), host.CopyOperation(["/conf.txt"], ctx, "/", "/etc/conf.txt", 7, 8)]
    eng = make_engine(2 << 20)                                    # the layer spans two arenas
    fused = host.MemFS(roots["fused"]).commit_copy_ops(eng, NOW, ops, flags=host.MKHOST_MATERIALIZE | host.MKHOST_MATERIALIZE_CHOWN)
    plain = host.MemFS(roots["plain"]).commit_copy_ops(make_engine(2 << 20), NOW, ops)
    assert fused == plain and _tree(roots["plain"]) == {}
    oc.execute_copy_op(ctx, ["/app"], roots["oracle"] + "/srv/app/", 5, 6, True, False, False, [])
    oc.execute_copy_op(ctx, ["/conf.txt"], roots["oracle"] + "/etc/conf.txt", 7, 8, True, False, False, [])
    got, want = _tree(roots["fused"]), _tree(roots["oracle"])
    assert got == want
    assert got["srv/app/sub/b.bin"][1:4] == (0o755, 5, 6) and got["etc/conf.txt"][1:4] == (0o640, 7, 8)
    assert got["srv/app/link"][:2] == ("l", "a.bin") and got["srv/app"] == ("d", 0o755, 5, 6)
    fs = lt.MemFS(lambda: NOW, roots["oracle"])
    entries = fs.add_layer_by_copy_ops([lt.CopyOperation.new(["/app"], ctx, "/", "/srv/app/", uid=5, gid=6),
                                        lt.CopyOperation.new(["/conf.txt"], ctx, "/", "/etc/conf.txt", uid=7, gid=8)])
    assert fused["tar_digest"] == lt.tar_digest(entries)
    # a second commit of the same ops: nothing new for the layer except re-added ancestors, files copied from disk
    again = host.MemFS(roots["fused"]).commit_copy_ops(make_engine(2 << 20), NOW, ops, flags=host.MKHOST_MATERIALIZE | host.MKHOST_MATERIALIZE_CHOWN)
    assert again["n_entries"] == fused["n_entries"] and _tree(roots["fused"]) == want


def random_trees_small_arenas(make_engine, tmp):
    """Arena-boundary arithmetic: random build contexts committed and fingerprinted through arenas of 8 KiB .. 1 MiB
    (every flush condition is hit: entry does not fit the remainder, trailer does not fit, file split across arenas for
    the CRC stream at 16-byte granularity) -- tar bytes, TarDigest, chunk table root and cacheID against the oracle."""
    from tests.test_host_fuzz_cpu import _random_tree
    seedid = ctx_crc.from_step_cache_id(ctx_crc.plan_seed(True, False), "scratch")
    for seed in range(10):
        rng = np.random.default_rng(77 + seed)
        ctx = os.path.join(tmp, "ctx%d" % seed)
        os.mkdir(ctx)
        _random_tree(ctx, rng)
        with open(os.path.join(ctx, "blob"), "wb") as f:          # one file that spans several small arenas in the CRC stream
            f.write(bytes(rng.integers(0, 256, 40_000 + seed, dtype=np.uint8)))
        for d, dirs, files in os.walk(ctx):
            for n in dirs + files:
                os.utime(os.path.join(d, n), (T, T), follow_symlinks=False)
        os.utime(ctx, (T, T))
        root = os.path.join(tmp, "root%d" % seed)
        os.mkdir(root)
        os.chmod(root, 0o755)
        try:
            entries = lt.MemFS(lambda: NOW, root).add_layer_by_copy_ops([lt.CopyOperation.new(["/"], ctx, "/", "/app/", uid=1, gid=2)])
            want_id = ctx_crc.copy_step_cache_id(seedid, "COPY", ". /app/", ctx, ["."])
        except (OSError, ValueError):
            continue                                              # e.g. an absolute symlink out of the tree: both sides refuse (test_host_fuzz_cpu)
        blob, want = _layer_expectations(entries)
        for arena in (8 << 10, 12 << 10, 64 << 10, 1 << 20):
            assert host.copy_step_cache_id(make_engine(arena), seedid, "COPY", ". /app/", ctx, ["."]) == want_id, (seed, arena)
            if arena < 48 << 10:
                continue                                          # the 40 kB blob must fit one arena for the layer
            tar_path = os.path.join(tmp, "t%d_%d.tar" % (seed, arena))
            with open(tar_path, "wb") as f:
                got = host.commit_copy_ops(make_engine(arena), root, NOW, [host.CopyOperation(["/"], ctx, "/", "/app/", 1, 2)],
                                           tar_fd=f.fileno())
            assert open(tar_path, "rb").read() == blob, (seed, arena)
            assert got["tar_digest"] == lt.tar_digest(entries) and got["root"] == want["root"] and got["n_chunks"] == want["n_chunks"]


def table_limits_and_arena_leases(make_engine, tmp):
    """ADVICE round 1: (a) a context of many tiny files fills max_extents long before it fills an arena -- the packers
    flush early instead of failing with E_CAPACITY (the reference handles any file count, add_copy_step.go:153-169);
    (b) a packer that throws between acquire and submit gives its arena back (ArenaLease): the handle survives more
    failures than it has arenas."""
    ctx = os.path.join(tmp, "tiny")
    rng = np.random.default_rng(11)
    for i in range(300):
        _mk(ctx, "d%02d/f%04d" % (i % 7, i), rng.integers(0, 256, int(rng.integers(0, 40)), dtype=np.uint8).tobytes())
    for d, _, _ in os.walk(ctx):
        os.utime(d, (T, T))
    seed = ctx_crc.from_step_cache_id(ctx_crc.plan_seed(True, False), "scratch")
    eng = make_engine(1 << 20, max_extents=16)                      # 300 files x 2 extents each >> 16
    assert host.copy_step_cache_id(eng, seed, "COPY", ". /app/", ctx, ["."]) == ctx_crc.copy_step_cache_id(seed, "COPY", ". /app/", ctx, ["."])
    assert eng.submits() >= 300 * 2 // 16
    root = os.path.join(tmp, "root")
    os.mkdir(root)
    entries = lt.MemFS(lambda: NOW, root).add_layer_by_copy_ops([lt.CopyOperation.new(["/"], ctx, "/", "/app/")])
    blob, want = _layer_expectations(entries)
    eng = make_engine(1 << 20, max_extents=16)
    got = host.commit_copy_ops(eng, root, NOW, [host.CopyOperation(["/"], ctx, "/", "/app/")])
    assert got["tar_digest"] == lt.tar_digest(entries) and got["root"] == want["root"] and got["n_chunks"] == want["n_chunks"]
    # per-file digests: one stream slot per file is a session-wide need, refused with a clear message when too small
    h = host.MemFS(root)
    try:
        h.commit_copy_ops(make_engine(1 << 20, max_extents=16), NOW, [host.CopyOperation(["/"], ctx, "/", "/app/")],
                          flags=host.MKHOST_FILE_DIGESTS)
        raise AssertionError("expected a capacity error")
    except host.HostError as e:
        assert "stream slot per regular file" in str(e)
    h2 = host.MemFS(root)
    got2 = h2.commit_copy_ops(make_engine(1 << 20, max_extents=512), NOW, [host.CopyOperation(["/"], ctx, "/", "/app/")],
                              flags=host.MKHOST_FILE_DIGESTS)
    assert got2["tar_digest"] == got["tar_digest"]
    # (b) failures between acquire and submit: a damaged archive, n_host_arenas + 2 times on ONE handle, then a good one
    rng = np.random.default_rng(5)
    data = _base_tar(rng)
    bad = bytearray(data)
    victim = [m for m in lt.read_tar(data) if m.hdr.typeflag == lt.TYPE_REG and m.data_len][3]
    bad[victim.data_off - 512 + 150] ^= 0x55                        # break a header checksum a few members in
    eng = make_engine(1 << 20, n_host_arenas=2)
    for _ in range(4):
        r, w = os.pipe()
        import threading
        t = threading.Thread(target=lambda: (os.write(w, bytes(bad)), os.close(w)))
        t.start()
        try:
            host.MemFS(root).update_from_tar(eng, NOW, r)
            raise AssertionError("expected a damaged-archive error")
        except host.HostError:
            pass
        finally:
            os.close(r)
            t.join()
    good = os.path.join(tmp, "good.tar")
    open(good, "wb").write(data)
    with open(good, "rb") as f:
        ok = host.MemFS(root).update_from_tar(eng, NOW, f.fileno())
    assert ok["tar_digest"] == "sha256:" + hashlib.sha256(data).hexdigest()


def batch_of_layers_in_one_session(make_engine, tmp):
    """mkhost_memfs_commit_layers: N consecutive COPY layers packed together (every arena carries a piece of every open
    layer, one SHA-256 stream per layer continued across submits) == N sequential commits: per-layer TarDigest and tar
    bytes equal the oracle's, later layers are diffed against the tree the earlier ones left."""
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
        entries = o.add_layer_by_copy_ops([lt.CopyOperation.new(srcs, ctx, "/", dst, uid=5, gid=6)])
        want.append((lt.tar_digest(entries), b"".join(lt.layer_tar_chunks(entries)), len(entries)))
    for arena_bytes in (2 << 20, 8 << 20):                         # shares of 341 KiB / 1.3 MiB per layer
        eng = make_engine(arena_bytes, n_host_arenas=2)
        h = host.MemFS(root)
        paths = [os.path.join(tmp, "l%d_%d.tar" % (i, arena_bytes)) for i in range(len(specs))]
        files = [open(p, "wb") for p in paths]
        got = h.commit_layers(eng, NOW, [[host.CopyOperation(s, ctx, "/", d, 5, 6)] for s, d in specs],
                              tar_fds=[f.fileno() for f in files])
        for f in files:
            f.close()
        for i, (dig, blob, n) in enumerate(want):
            assert got[i]["tar_digest"] == dig, (i, arena_bytes)
            assert open(paths[i], "rb").read() == blob, (i, arena_bytes)
            assert (got[i]["n_entries"], got[i]["tar_bytes"]) == (n, len(blob))
        assert eng.submits() >= 2
        h.close()
    # the union chunk table equals the one over the concatenation of the layers' files
    # without digests
    eng = make_engine(8 << 20)
    got = host.MemFS(root).commit_layers(eng, NOW, [[host.CopyOperation(s, ctx, "/", d, 5, 6)] for s, d in specs],
                                        flags=host.MKHOST_NO_TAR_DIGEST)
    assert all(g["tar_digest"] == "sha256:" + "00" * 32 for g in got)
    try:
        host.MemFS(root).commit_layers(make_engine(1 << 20), NOW, [[host.CopyOperation(["/big.bin"], ctx, "/", "/x")]])
        raise AssertionError("expected a capacity error")
    except host.HostError as e:
        assert "exceeds the arena" in str(e)


def ingest_member_larger_than_the_arena(make_engine, tmp):
    """mkhost_memfs_update_from_tar with members of 3.2 MB and 1.1 MB through 1 MiB arenas: the bodies travel in pieces
    (MKSNAP_X_MORE / MKSNAP_X_CONT), DiffID, chunk table and per-file digests equal those of the undivided archive;
    MKHOST_UNTAR, which needs a contiguous body, refuses loudly."""
    rng = np.random.default_rng(12)
    bodies = {"big/one.bin": rng.integers(0, 256, 3_200_001, dtype=np.uint8).tobytes(),
              "big/two.bin": bytes(700_000) + rng.integers(0, 256, 400_123, dtype=np.uint8).tobytes(),
              "small.txt": b"hello"}
    buf = io.BytesIO()
    with tarfile.open(fileobj=buf, mode="w", format=tarfile.PAX_FORMAT) as tf:
        # members owned by the caller: the untar below must reach the capacity check, not fail on chown
        d = tarfile.TarInfo("big/")
        d.type, d.mode, d.mtime, d.uid, d.gid = tarfile.DIRTYPE, 0o755, T, os.getuid(), os.getgid()
        tf.addfile(d)
        for name, data in bodies.items():
            ti = tarfile.TarInfo(name)
            ti.size, ti.mode, ti.mtime, ti.uid, ti.gid = len(data), 0o644, T, os.getuid(), os.getgid()
            tf.addfile(ti, io.BytesIO(data))
    data = buf.getvalue()
    path = os.path.join(tmp, "big.tar")
    open(path, "wb").write(data)
    members = [m for m in lt.read_tar(data) if m.hdr.typeflag == lt.TYPE_REG and m.data_len]
    want = olib.chunk_table(np.frombuffer(data, dtype=np.uint8), [m.data_off for m in members], [m.data_len for m in members])
    root = os.path.join(tmp, "r")
    os.mkdir(root)
    for arena in (1 << 20, 8 << 20):
        eng = make_engine(arena)
        h = host.MemFS(root)
        with open(path, "rb") as f:
            got = h.update_from_tar(eng, NOW, f.fileno(), flags=host.MKHOST_FILE_DIGESTS)
        assert got["tar_digest"] == "sha256:" + hashlib.sha256(data).hexdigest() and got["tar_bytes"] == len(data), arena
        assert (got["n_chunks"], got["n_unique"], got["root"]) == (want["n_chunks"], want["n_unique"], want["root"]), arena
        for name, body in bodies.items():
            assert h.file_digest("/" + name) == hashlib.sha256(body).digest(), (arena, name)
        h.close()
    assert make_engine(1 << 20).submits() == 0
    try:
        with open(path, "rb") as f:
            host.MemFS(root).update_from_tar(make_engine(1 << 20), NOW, f.fileno(), flags=host.MKHOST_UNTAR)
        raise AssertionError("expected a capacity error")
    except host.HostError as e:
        assert "exceeds the arena" in str(e)


def incremental_cache_id(make_engine, tmp):
    """mkhost_context_crc32_cached: the first build fills the cache (every file travels), the second build of the
    unchanged context sends NO file bytes and returns the identical cacheID, an edit re-sends exactly the edited file;
    the value always equals the oracle's full computation (zlib over the reference's byte order), also through small
    arenas that split files into several extents and through a saved + reloaded cache."""
    ctx = _ctx(tmp)
    seed = ctx_crc.from_step_cache_id(ctx_crc.plan_seed(True, False), "scratch")
    prefix = (seed + "COPY" + ". /app/").encode()

    def want():
        return int(ctx_crc.copy_step_cache_id(seed, "COPY", ". /app/", ctx, ["."]), 16)
    regular = [os.path.join(d, f) for d, _, fs in os.walk(ctx) for f in fs if not os.path.islink(os.path.join(d, f))]
    n_files, total = len(regular), sum(os.path.getsize(p) for p in regular)
    eng = make_engine(1 << 20)                                    # big.bin (1.5 MB) is split over two arenas
    cache = host.CrcCache()
    crc, slen, st = cache.context_crc32(eng, prefix, ctx, ["."])
    assert crc == want() and st == {"files_total": n_files, "files_reused": 0, "bytes_total": total, "bytes_sent": total}
    assert len(cache) == n_files
    before = eng.submits()
    crc2, slen2, st2 = cache.context_crc32(eng, prefix, ctx, ["."])
    assert (crc2, slen2) == (crc, slen) and st2["files_reused"] == n_files and st2["bytes_sent"] == 0
    assert eng.submits() - before == 1                            # one arena of path strings, no file bytes
    assert host.context_crc32(eng, prefix, ctx, ["."])[0] == crc  # the uncached entry point agrees
    # a different prefix (seed / directive / args) reuses the same per-file values: they are position independent
    crc3, _, st3 = cache.context_crc32(eng, b"other" + prefix, ctx, ["."])
    assert st3["bytes_sent"] == 0 and "%x" % crc3 == ctx_crc.copy_step_cache_id("other" + seed, "COPY", ". /app/", ctx, ["."])
    # edit one file (same size): exactly that file travels again
    p = os.path.join(ctx, "d1", "f003.bin")
    size = os.path.getsize(p)
    with open(p, "r+b") as f:
        f.write(b"EDIT")
    crc4, _, st4 = cache.context_crc32(eng, prefix, ctx, ["."])
    assert crc4 == want() != crc and st4["files_reused"] == n_files - 1 and st4["bytes_sent"] == size
    # grow big.bin (split across arenas): its pieces are joined into one remembered value
    with open(os.path.join(ctx, "big.bin"), "ab") as f:
        f.write(b"tail" * 1000)
    crc5, _, st5 = cache.context_crc32(eng, prefix, ctx, ["."])
    assert crc5 == want() and st5["files_reused"] == n_files - 1
    crc6, _, st6 = cache.context_crc32(eng, prefix, ctx, ["."])
    assert crc6 == crc5 and st6["bytes_sent"] == 0
    # save / load: a later process starts warm; a stale entry (file replaced: new inode) is not trusted
    path = os.path.join(tmp, "crc.cache")
    cache.save(path)
    warm = host.CrcCache(path)
    assert len(warm) == len(cache)
    q = os.path.join(ctx, "d0", "f001.bin")
    data = open(q, "rb").read()
    stq = os.stat(q)
    os.rename(q, q + ".old")
    with open(q, "wb") as f:
        f.write(data[::-1])
    os.utime(q, ns=(stq.st_atime_ns, stq.st_mtime_ns))
    os.remove(q + ".old")
    crc7, _, st7 = warm.context_crc32(make_engine(8 << 20), prefix, ctx, ["."])
    assert crc7 == want() and st7["files_reused"] == n_files - 1 and st7["bytes_sent"] == len(data)
