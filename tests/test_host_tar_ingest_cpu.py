"""CPU: UpdateFromTarReader(untar=false) -- the go1.14 archive/tar Reader restatement and the MemFS merge, C++ host
side (libmkhost) against the oracle, and the oracle's reader against Python's independent `tarfile`.

Reference: lib/snapshot/mem_fs.go:165-255 (UpdateFromTarReader), mem_fs_test.go:31-117 (TestUntarFromPath: the
layer counts 7 and 2 are the reference's own assertions)."""
import base64
import gzip
import io
import json
import os
import tarfile

import pytest

from makisu_b200 import host
from oracle import layer_tar as lt
from tests.test_host_cpu import _desc_from_oracle, _mk

HERE = os.path.dirname(os.path.abspath(__file__))
NOW = 1_600_000_000


def _go_fixture_stream() -> bytes:
    """The 390 Go-written USTAR headers of the reference's busybox layer (tests/golden), each followed by a zero body
    of its padded size, plus the two-block end marker: same member layout as the original archive."""
    fix = json.load(open(f"{HERE}/golden/reference_fixtures.json"))
    blob = gzip.decompress(base64.b64decode(fix["busybox_headers_gz_b64"]))
    out = bytearray()
    for i in range(fix["busybox_n_headers"]):
        blk = blob[512 * i:512 * (i + 1)]
        out += blk
        if blk[156:157] in (b"0", b"\0"):
            size = int(blk[124:135], 8)
            out += b"\0" * ((size + 511) // 512 * 512)
    return bytes(out) + b"\0" * 1024


def _check_against_tarfile(data: bytes):
    ms = lt.read_tar(data)
    infos = tarfile.open(fileobj=io.BytesIO(data)).getmembers()
    assert len(ms) == len(infos)
    for m, i in zip(ms, infos):
        assert m.hdr.name.rstrip("/") == i.name.rstrip("/")
        assert m.hdr.typeflag == i.type
        assert m.hdr.mode == i.mode and m.hdr.uid == i.uid and m.hdr.gid == i.gid
        assert m.hdr.mtime_ns // 10**9 == int(i.mtime // 1)
        assert m.hdr.linkname == i.linkname
        if i.isreg():
            assert m.hdr.size == i.size and m.data_len == i.size and m.data_off == i.offset_data
    return ms


def _pipe_fd(data: bytes):
    """A real fd carrying the stream (the C entry points take an fd: file or pipe)."""
    import tempfile
    f = tempfile.TemporaryFile()
    f.write(data)
    f.seek(0)
    return f


def _both(root, blacklist, streams, now=NOW):
    """Run the same sequence of tar streams through the oracle MemFS and the C++ MemFS; return the last layers."""
    o = lt.MemFS(lambda: now, str(root), blacklist=list(blacklist))
    h = host.MemFS(str(root), list(blacklist))
    got = want = None
    for data in streams:
        want = _desc_from_oracle(o.update_from_tar(data))
        with _pipe_fd(data) as f:
            got = h.describe_update_from_tar(now, f.fileno())
        assert got == want
    return o, h, got


def test_reader_and_merge_on_go_written_headers(tmp_path):
    data = _go_fixture_stream()
    ms = _check_against_tarfile(data)
    assert len(ms) == 390 and sum(m.hdr.typeflag == b"1" for m in ms) == 372
    root = tmp_path / "root"
    root.mkdir()
    _, h, got = _both(root, [], [data])
    assert len(got) == 390
    # hard links carry an absolute Linkname in the tree (mem_fs.go:221-223), regular entries keep theirs
    links = [l for l in got if l.startswith("1 ")]
    assert len(links) == 372
    # the same layer again: every header is "similar" to what the tree holds => empty layer
    _, _, again = _both(root, [], [data, data])
    assert again == []
    h.close()


def _add(tf, name, type_=tarfile.REGTYPE, data=b"", mode=0o644, link="", uid=0, gid=0, mtime=1_500_000_000):
    ti = tarfile.TarInfo(name)
    ti.type, ti.mode, ti.uid, ti.gid, ti.mtime, ti.linkname = type_, mode, uid, gid, mtime, link
    ti.size = len(data) if type_ == tarfile.REGTYPE else 0
    tf.addfile(ti, io.BytesIO(data) if ti.size else None)


def _sample_tar(fmt) -> bytes:
    buf = io.BytesIO()
    with tarfile.open(fileobj=buf, mode="w", format=fmt) as tf:
        _add(tf, "usr/", tarfile.DIRTYPE, mode=0o755)
        _add(tf, "usr/bin/", tarfile.DIRTYPE, mode=0o755)
        _add(tf, "bin", tarfile.SYMTYPE, link="usr/bin", mode=0o777)
        _add(tf, "usr/bin/tool", data=b"#!/bin/sh\n" * 700, mode=0o4755, uid=3, gid=4)
        _add(tf, "usr/bin/alias", tarfile.LNKTYPE, link="usr/bin/tool", mode=0o4755, uid=3, gid=4)
        _add(tf, "./etc/passwd", data=b"root:x:0:0\n", mode=0o100644)          # foreign writer: type bits in Mode
        _add(tf, "etc/" + "n" * 120 + "/" + "f" * 90 + ".conf", data=b"x" * 513)   # needs prefix split / long-name record
        _add(tf, "etc/" + "p" * 200 + "/" + "q" * 150, data=b"")                  # too long for USTAR
        _add(tf, "srv/déjà.txt", data=b"accent")                        # non-ASCII
        _add(tf, "big/uid", data=b"1", uid=3_000_000, gid=5_000_000)              # > 7 octal digits
        _add(tf, "lnk/" + "l" * 130, tarfile.SYMTYPE, link="t" * 140)             # long link target
        _add(tf, "dev/null", tarfile.CHRTYPE, mode=0o666)                         # special: skipped
        _add(tf, "run/fifo", tarfile.FIFOTYPE)                                    # special: skipped
        _add(tf, ".wh..wh.plnk/", tarfile.DIRTYPE)                                # AUFS metadata: skipped
        _add(tf, "proc/", tarfile.DIRTYPE)                                        # blacklisted
        _add(tf, "proc/cpuinfo", data=b"no")                                      # blacklisted
        _add(tf, "opt/deep/er/file", data=b"ancestors are synthesized")           # parents missing from the archive
        _add(tf, "frac", data=b"", mtime=1_500_000_000.75)
    return buf.getvalue()


@pytest.mark.parametrize("fmt", [tarfile.USTAR_FORMAT, tarfile.PAX_FORMAT, tarfile.GNU_FORMAT])
def test_formats_against_tarfile_and_cpp_against_oracle(tmp_path, fmt):
    if fmt == tarfile.USTAR_FORMAT:
        buf = io.BytesIO()
        with tarfile.open(fileobj=buf, mode="w", format=fmt) as tf:  # only what plain USTAR can express
            _add(tf, "usr/", tarfile.DIRTYPE, mode=0o755)
            _add(tf, "usr/" + "n" * 120 + "/" + "f" * 90, data=b"x" * 1000)
            _add(tf, "usr/h", tarfile.LNKTYPE, link="usr/" + "n" * 90)
            _add(tf, "usr/s", tarfile.SYMTYPE, link="../x")
        data = buf.getvalue()
    else:
        data = _sample_tar(fmt)
    _check_against_tarfile(data)
    root = tmp_path / "root"
    root.mkdir()
    bl = [str(root / "proc")]
    o, h, got = _both(root, bl, [data])
    dsts = [l.split(" ")[6] for l in got]
    assert dsts == sorted(dsts, key=os.fsencode)
    if fmt != tarfile.USTAR_FORMAT:
        assert "/dev/null" not in dsts and "/run/fifo" not in dsts and "/proc/cpuinfo" not in dsts
        assert not any(".wh..wh." in d for d in dsts)
        assert {"/opt", "/opt/deep", "/opt/deep/er", "/opt/deep/er/file", "/etc/passwd", "/usr/bin/alias"} <= set(dsts)
        # a COPY on top of the ingested tree: /bin is a symlink to usr/bin in the base layer, so the ancestors of the
        # destination resolve through it (mem_fs.go:509-569)
        ctx = tmp_path / "ctx"
        _mk(ctx, "n/new.txt", b"new")
        for d, _, _ in os.walk(ctx):
            os.utime(d, (1_500_000_000, 1_500_000_000))
        want = _desc_from_oracle(o.add_layer_by_copy_ops([lt.CopyOperation.new(["/n"], str(ctx), "/", "/bin/sub/", uid=1, gid=2)]))
        got2 = h.describe_copy_ops(NOW, [host.CopyOperation(["/n"], str(ctx), "/", "/bin/sub/", 1, 2)])
        assert got2 == want
        assert "/usr/bin/sub/new.txt" in [l.split(" ")[6] for l in got2]
    h.close()


def test_untar_from_path_layer_counts(tmp_path):
    """mem_fs_test.go:31-117 with untar=false: 7 headers from the first archive, 2 whiteouts from the second."""
    root = tmp_path / "root"
    _mk(root, "test1/test1.txt", b"TEST1")
    (root / "mydir").mkdir()
    b1 = io.BytesIO()
    with tarfile.open(fileobj=b1, mode="w", format=tarfile.USTAR_FORMAT) as tf:  # filepath.Walk order of `src`
        _add(tf, "mydir", tarfile.SYMTYPE, link="/target.txt", mode=0o777)
        _add(tf, "target.txt", data=b"TARGET", mode=0o677)
        _add(tf, "test.txt", data=b"TEST", mode=0o677)
        _add(tf, "test1/", tarfile.DIRTYPE, mode=0o755)
        _add(tf, "test1/test1.txt", data=b"TEST1", mode=0o677)
        _add(tf, "test2/", tarfile.DIRTYPE, mode=0o755)
        _add(tf, "test2.txt", data=b"TEST1", mode=0o677)
    b2 = io.BytesIO()
    with tarfile.open(fileobj=b2, mode="w", format=tarfile.USTAR_FORMAT) as tf:
        _add(tf, ".wh.test.txt/", tarfile.DIRTYPE, mode=0o755)
        _add(tf, ".wh.test1/", tarfile.DIRTYPE, mode=0o755)
    o = lt.MemFS(lambda: NOW, str(root))
    h = host.MemFS(str(root))
    l1 = o.update_from_tar(b1.getvalue())
    with _pipe_fd(b1.getvalue()) as f:
        g1 = h.describe_update_from_tar(NOW, f.fileno())
    assert len(l1) == 7 and g1 == _desc_from_oracle(l1)
    l2 = o.update_from_tar(b2.getvalue())
    with _pipe_fd(b2.getvalue()) as f:
        g2 = h.describe_update_from_tar(NOW, f.fileno())
    assert len(l2) == 2 and g2 == _desc_from_oracle(l2)
    assert [e.whiteout for e in l2] == [True, True]
    assert sorted(e.deleted for e in l2) == ["/test.txt", "/test1"]
    assert "test1" not in o.tree.children and "test.txt" not in o.tree.children
    h.close()


@pytest.mark.parametrize("damage", ["checksum", "truncated_header", "truncated_body", "garbage_after_zero_block", "global_pax"])
def test_malformed_streams_are_rejected_by_both(tmp_path, damage):
    root = tmp_path / "root"
    root.mkdir()
    buf = io.BytesIO()
    with tarfile.open(fileobj=buf, mode="w", format=tarfile.USTAR_FORMAT) as tf:
        _add(tf, "a.txt", data=b"a" * 700)
        _add(tf, "b.txt", data=b"b")
    data = bytearray(buf.getvalue())
    if damage == "checksum":
        data[3] ^= 1
    elif damage == "truncated_header":
        data = data[:1536 + 100]
    elif damage == "truncated_body":
        data = data[:512 + 600]
    elif damage == "garbage_after_zero_block":
        end = 512 + 1024 + 512 + 512
        data = data[:end] + b"\0" * 512 + b"x" * 512
    elif damage == "global_pax":
        g = io.BytesIO()
        with tarfile.open(fileobj=g, mode="w", format=tarfile.PAX_FORMAT, pax_headers={"comment": "hello"}) as tf:
            _add(tf, "a.txt", data=b"a")
        data = bytearray(g.getvalue())
    data = bytes(data)
    with pytest.raises(ValueError):
        lt.MemFS(lambda: NOW, str(root)).update_from_tar(data)
    h = host.MemFS(str(root))
    with _pipe_fd(data) as f, pytest.raises(host.HostError) as ei:
        h.describe_update_from_tar(NOW, f.fileno())
    assert "update memfs from tar" in str(ei.value)
    h.close()


def test_base256_numeric_fields_and_old_v7(tmp_path):
    """GNU base-256 size/uid fields and a V7 header without magic (strconv.go parseNumeric, format.go getFormat)."""
    def block(name, size_field, uid_field, typeflag=b"0", magic=b"ustar\x0000"):
        b = bytearray(512)
        b[0:len(name)] = name
        b[100:108] = b"0000644\0"
        b[108:116] = uid_field
        b[116:124] = b"0000000\0"
        b[124:136] = size_field
        b[136:148] = b"13142405000\0"
        b[148:156] = b" " * 8
        b[156:157] = typeflag
        b[257:265] = magic
        b[148:156] = b"%06o\0 " % sum(b)
        return bytes(b)
    big_uid = bytes([0x80]) + (3_000_000).to_bytes(7, "big")
    size600 = bytes([0x80]) + (600).to_bytes(11, "big")
    data = (block(b"bin256", size600, big_uid, magic=b"ustar  \0") + b"z" * 600 + b"\0" * 424 +
            block(b"oldv7/", b"00000000000\0", b"0000001\0", typeflag=b"\0", magic=b"\0" * 8) +
            block(b"oldreg", b"00000000003\0", b"0000001\0", typeflag=b"\0", magic=b"\0" * 8) + b"abc" + b"\0" * 509 +
            b"\0" * 1024)
    ms = lt.read_tar(data)
    assert [(m.hdr.name, m.hdr.typeflag, m.hdr.size, m.hdr.uid) for m in ms] == \
        [("bin256", b"0", 600, 3_000_000), ("oldv7/", b"5", 0, 1), ("oldreg", b"0", 3, 1)]
    root = tmp_path / "root"
    root.mkdir()
    _both(root, [], [data])[1].close()


# ---- untar=true (mem_fs.go:574-716, lib/tario/apply.go) ----------------------------------------------------------
import stat as _stat

needs_root = pytest.mark.skipif(os.geteuid() != 0, reason="chown needs root")


def _disk(root):
    out = {}
    for d, dirs, files in os.walk(root):
        for n in sorted(dirs + files):
            p = os.path.join(d, n)
            st = os.lstat(p)
            rel = os.path.relpath(p, root)
            if _stat.S_ISLNK(st.st_mode):
                out[rel] = ("l", os.readlink(p).replace(str(root), "$ROOT"), st.st_uid, st.st_gid)
            elif _stat.S_ISDIR(st.st_mode):
                out[rel] = ("d", _stat.S_IMODE(st.st_mode), st.st_uid, st.st_gid, st.st_mtime_ns)
            else:
                out[rel] = ("f", _stat.S_IMODE(st.st_mode), st.st_uid, st.st_gid, st.st_mtime_ns, st.st_nlink, open(p, "rb").read())
    return out


@needs_root
def test_untar_from_path_like_the_reference(tmp_path):
    """mem_fs_test.go:31-117 (TestUntarFromPath), assertions copied: contents of test.txt and test1/test1.txt, mydir
    replaced by the symlink (reads TARGET through it), 7 headers; then the whiteout archive removes test.txt, 2 headers."""
    b1 = io.BytesIO()
    with tarfile.open(fileobj=b1, mode="w", format=tarfile.USTAR_FORMAT) as tf:
        _add(tf, "mydir", tarfile.SYMTYPE, link="/target.txt", mode=0o777)
        _add(tf, "target.txt", data=b"TARGET", mode=0o677)
        _add(tf, "test.txt", data=b"TEST", mode=0o677)
        _add(tf, "test1/", tarfile.DIRTYPE, mode=0o755)
        _add(tf, "test1/test1.txt", data=b"TEST1", mode=0o677)
        _add(tf, "test2/", tarfile.DIRTYPE, mode=0o755)
        _add(tf, "test2.txt", tarfile.LNKTYPE, link="test1/test1.txt", mode=0o677)
    b2 = io.BytesIO()
    with tarfile.open(fileobj=b2, mode="w", format=tarfile.USTAR_FORMAT) as tf:
        _add(tf, ".wh.test.txt/", tarfile.DIRTYPE, mode=0o755)
        _add(tf, ".wh.test1/", tarfile.DIRTYPE, mode=0o755)
    disks = []
    for impl in ("oracle", "cpp"):
        root = tmp_path / impl
        _mk(root, "test1/test1.txt", b"TEST1", mode=0o677)
        (root / "mydir").mkdir()
        if impl == "oracle":
            fs = lt.MemFS(lambda: NOW, str(root))
            n1 = len(fs.update_from_tar(b1.getvalue(), untar=True))
        else:
            fs = host.MemFS(str(root))
            with _pipe_fd(b1.getvalue()) as f:
                n1 = len(fs.describe_update_from_tar(NOW, f.fileno(), host.MKHOST_UNTAR))
        assert n1 == 7
        assert (root / "test.txt").read_bytes() == b"TEST" and (root / "test1" / "test1.txt").read_bytes() == b"TEST1"
        assert os.path.islink(root / "mydir") and (root / "mydir").read_bytes() == b"TARGET"
        assert os.stat(root / "test2.txt").st_nlink == 2
        if impl == "oracle":
            n2 = len(fs.update_from_tar(b2.getvalue(), untar=True))
        else:
            with _pipe_fd(b2.getvalue()) as f:
                n2 = len(fs.describe_update_from_tar(NOW, f.fileno(), host.MKHOST_UNTAR))
            fs.close()
        assert n2 == 2 and not (root / "test.txt").exists() and not (root / "test1").exists()
        disks.append(_disk(root))
    assert disks[0] == disks[1]


@needs_root
@pytest.mark.parametrize("seed", range(18))
def test_untar_random_archives_cpp_equals_oracle(tmp_path, seed):
    """Two random archives untarred one after the other onto a pre-populated root: the second one meets what the first
    left (similar entries skipped, directories updated in place, files replaced, whiteouts).  Disk state (type, mode,
    owner, mtime, link count, content), merged layers and failures must be the same for both implementations."""
    import numpy as np
    from tests.test_host_fuzz_cpu import _random_tar
    results = []
    for impl in ("oracle", "cpp"):
        rng = np.random.default_rng(4000 + seed)
        fmt = [tarfile.USTAR_FORMAT, tarfile.PAX_FORMAT, tarfile.GNU_FORMAT][seed % 3]
        root = tmp_path / impl
        _mk(root, "a/keep.txt", b"k")
        _mk(root, "b", b"file where an archive may want a directory")
        for d in (root / "a", root):
            os.utime(d, (1_400_000_000, 1_400_000_000))
        fs = lt.MemFS(lambda: NOW, str(root)) if impl == "oracle" else host.MemFS(str(root))
        log = []
        for _ in range(2):
            data = _random_tar(rng, fmt)
            try:
                if impl == "oracle":
                    layer = _desc_from_oracle(fs.update_from_tar(data, untar=True))
                else:
                    with _pipe_fd(data) as f:
                        layer = fs.describe_update_from_tar(NOW, f.fileno(), host.MKHOST_UNTAR)
                log.append(("ok", [l.split(" ")[6] for l in layer]))
            except (OSError, ValueError, host.HostError):
                log.append(("err",))
                break
        if impl == "cpp":
            fs.close()
        results.append((log, _disk(root)))
    assert results[0][0] == results[1][0]
    a, b = results[0][1], results[1][1]
    if ("err",) in results[0][0]:
        # an aborted ingest (e.g. a hard link whose target is a directory) never reaches the step that restores the
        # parent directories' mtimes: those carry the wall clock of each run
        drop = lambda t: {k: (v[:4] if v[0] == "d" else v) for k, v in t.items()}  # noqa: E731
        a, b = drop(a), drop(b)
    assert a == b


REF_LAYER = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "alpine_test_layer_zeroed.tar.gz")


def test_reference_layer_archive_end_to_end(tmp_path):
    """The reference's own layer (testutil.SampleLayerTarDigest, lib/utils/testutil/constants.go:28): the Go-written tar
    inside it (SHA-256 4ac76077...caba, SURVEY section 8c), stored with the bodies of bin/[ and bin/getconf zero-filled
    (tests/golden/make_golden.py).  Reader == tarfile, C++ merge == oracle merge, and an untar by both leaves identical
    trees whose hard links share inodes (372 of the 390 members are hard links)."""
    import hashlib
    data = gzip.decompress(open(REF_LAYER, "rb").read())
    assert hashlib.sha256(data).hexdigest() == "0785eb88355b58156ea158d14d9bc66b62871f95c3da416b455c8ee1145fcf1b"
    assert len(data) == 1_308_672
    ms = _check_against_tarfile(data)
    assert len(ms) == 390
    root = tmp_path / "merge"
    root.mkdir()
    _both(root, [], [data])[1].close()
    if os.geteuid() != 0:
        return
    disks = []
    for impl in ("oracle", "cpp"):
        r = tmp_path / impl
        r.mkdir()
        os.utime(r, (1_400_000_000, 1_400_000_000))
        if impl == "oracle":
            n = len(lt.MemFS(lambda: NOW, str(r)).update_from_tar(data, untar=True))
        else:
            fs = host.MemFS(str(r))
            with _pipe_fd(data) as f:
                n = len(fs.describe_update_from_tar(NOW, f.fileno(), host.MKHOST_UNTAR))
            fs.close()
        assert n == 390
        disks.append(_disk(r))
    assert disks[0] == disks[1]
    busybox = [v for k, v in disks[0].items() if k == "bin/busybox" or k.endswith("/busybox")]
    assert busybox and busybox[0][5] > 300                          # st_nlink: the applets are hard links to it
