"""CPU: symlink handling on the layer path, replayed from the reference's own tests.

  * TestEvalSymlink (lib/snapshot/utils_test.go:86-147) -- the three scenarios with the values the reference asserts,
    on the oracle (oracle/copier.py) and on the C++ host side (mkhost_eval_symlinks).
  * MemFS.addToLayer resolves every SOURCE through evalSymlinks before walking it (lib/snapshot/mem_fs.go:380-384):
    `COPY linkdir /dst` copies the link target's contents, `COPY link.txt /dst/` lands under the TARGET's base name,
    a symlinked intermediate component is followed.  Expected entries are written out by hand from the reference code,
    so a checker that shares the product's omission cannot hide it (round-1 VERDICT, "What's weak" #1).
  * TestGetAncestors (lib/snapshot/mem_fs_test.go:340-570): FollowSymlinkFullResolve, FollowSymlinkPartialResolve,
    DetectSymlinkInfiniteLoop and FillNonexistent rebuilt through the public surface: the tree state comes from a scan
    of a directory holding the same directories and links, the addAncestors call is the one a COPY onto that
    destination makes (mem_fs.go:369), and the layer must hold exactly the entries the reference's test counts.
"""
import os

import numpy as np

import pytest

from makisu_b200 import host
from oracle import copier as oc, layer_tar as lt
from tests.test_host_cpu import _desc_from_oracle, _mk

NOW = 1_600_000_000
T0 = 1_500_000_000


def _both_eval(path, root):
    a = oc.eval_symlinks(path, root)
    b = host.eval_symlinks(path, root)
    assert a == b, (path, a, b)
    return a


def test_eval_symlink_no_symlinks(tmp_path):  # utils_test.go:87-103
    root = str(tmp_path)
    _mk(root, "dir1/tmp1")
    assert _both_eval(os.path.join("dir1", "tmp1"), root) == "/dir1/tmp1"


def test_eval_symlink_simple_case(tmp_path):  # utils_test.go:105-125
    root = str(tmp_path)
    _mk(root, "test1")
    os.symlink("test1", os.path.join(root, "link2"))
    os.symlink(os.path.join(root, "link2"), os.path.join(root, "link3"))  # absolute target inside the root
    assert _both_eval("link2", root) == "/test1"
    assert _both_eval("link3", root) == "/test1"


def test_eval_symlink_layered(tmp_path):  # utils_test.go:127-146
    root = str(tmp_path)
    _mk(root, "dir1/tmp1")
    os.mkdir(os.path.join(root, "dir2"))
    os.symlink(os.path.join(root, "dir1"), os.path.join(root, "dir2", "dir3"))
    assert _both_eval(os.path.join("dir2", "dir3", "tmp1"), root) == "/dir1/tmp1"


def test_eval_symlink_forms_and_errors(tmp_path):
    root = str(tmp_path)
    _mk(root, "real/sub/f.txt", b"x")
    os.symlink("real", os.path.join(root, "alias"))
    os.symlink("../real/sub", os.path.join(root, "real", "up"))       # relative, with ..
    os.symlink("/etc", os.path.join(root, "escape"))
    os.symlink("loop_b", os.path.join(root, "loop_a"))
    os.symlink("loop_a", os.path.join(root, "loop_b"))
    assert _both_eval("", root) == ""                                   # utils.go:250-252
    assert _both_eval("/", root) == "/"
    assert _both_eval("/alias/sub/f.txt", root) == "/real/sub/f.txt"    # TrimRoot leaves a leading slash
    assert _both_eval("alias/up/f.txt", root) == "/real/sub/f.txt"
    assert _both_eval("real/sub/", root) == "/real/sub"
    for bad, msg in [("escape", "link points outside of root"), ("loop_a", "too many links"), ("nothing", "lstat")]:
        with pytest.raises(OSError) as eo:
            oc.eval_symlinks(bad, root)
        with pytest.raises(host.HostError) as eh:
            host.eval_symlinks(bad, root)
        assert msg in str(eh.value) and (msg in str(eo.value) or msg == "lstat")


@pytest.fixture
def linked_ctx(tmp_path):
    c = str(tmp_path / "ctx")
    _mk(c, "real/a.txt", b"A" * 10)
    _mk(c, "real/sub/b.txt", b"B" * 20)
    _mk(c, "file.txt", b"F" * 30)
    os.symlink("real", os.path.join(c, "linkdir"))             # link to a directory
    os.symlink("file.txt", os.path.join(c, "link.txt"))        # link to a file
    os.symlink("real/sub", os.path.join(c, "deep"))            # link used as an intermediate component
    os.symlink("a.txt", os.path.join(c, "real", "inner"))      # a link INSIDE the walked tree stays a link
    for d, _, _ in os.walk(c):
        os.utime(d, (T0, T0))
    return c


def _layer_both(tmp_path, ctx, srcs, dst, uid=7, gid=8):
    root = tmp_path / "root"
    root.mkdir(exist_ok=True)
    fs = lt.MemFS(lambda: NOW, str(root))
    want = _desc_from_oracle(fs.add_layer_by_copy_ops([lt.CopyOperation.new(srcs, ctx, "/", dst, uid=uid, gid=gid)]))
    got = host.describe_layer(str(root), NOW, [host.CopyOperation(srcs, ctx, "/", dst, uid, gid)])
    assert got == want
    return [(l.split(" ")[0], l.split(" ")[6], l.split(" ")[8] if len(l.split(" ")) > 8 else "") for l in got]


def test_copy_symlinked_source_dir_copies_the_target(tmp_path, linked_ctx):
    """COPY linkdir /dst : evalSymlinks("linkdir") = "/real", so the walk root is real/ (a directory: its CONTENTS go
    under /dst, mem_fs.go:389-394) -- not one symlink header, which is what an unresolved Lstat walk would emit."""
    ents = _layer_both(tmp_path, linked_ctx, ["/linkdir"], "/dst")
    assert ents == [
        ("5", "/dst", "/"),                                                     # addAncestors(inclusive): no source
        ("0", "/dst/a.txt", linked_ctx + "/real/a.txt"),
        ("2", "/dst/inner", linked_ctx + "/real/inner"),                        # links inside the tree are kept
        ("5", "/dst/sub", linked_ctx + "/real/sub"),
        ("0", "/dst/sub/b.txt", linked_ctx + "/real/sub/b.txt"),
    ]


def test_copy_symlinked_source_file_uses_the_target_name(tmp_path, linked_ctx):
    """COPY link.txt /dst/ : os.Stat follows the link => not a dir => createDst=false (mem_fs.go:357-365);
    evalSymlinks gives "/file.txt", so currDst = /dst/ + Base(src) = /dst/file.txt, a REGULAR file of 30 bytes."""
    ents = _layer_both(tmp_path, linked_ctx, ["/link.txt"], "/dst/")
    assert ents == [("5", "/dst", "/"), ("0", "/dst/file.txt", linked_ctx + "/file.txt")]
    # file -> file form keeps the destination name
    ents = _layer_both(tmp_path, linked_ctx, ["/link.txt"], "/dst/renamed")
    assert ents == [("5", "/dst", "/"), ("0", "/dst/renamed", linked_ctx + "/file.txt")]


def test_copy_through_symlinked_intermediate_component(tmp_path, linked_ctx):
    ents = _layer_both(tmp_path, linked_ctx, ["/deep/b.txt", "/linkdir/sub"], "/out/")
    assert ents == [("5", "/out", "/"), ("0", "/out/b.txt", linked_ctx + "/real/sub/b.txt")]  # second src: same b.txt


def test_copy_source_link_leaving_the_context_is_an_error(tmp_path, linked_ctx):
    os.symlink("/etc/hostname", os.path.join(linked_ctx, "escape"))
    root = tmp_path / "root"
    root.mkdir()
    with pytest.raises(host.HostError) as eh:
        host.describe_layer(str(root), NOW, [host.CopyOperation(["/escape"], linked_ctx, "/", "/dst/")])
    assert "eval symlinks for" in str(eh.value) and "link points outside of root" in str(eh.value)
    with pytest.raises(OSError):
        lt.MemFS(lambda: NOW, str(root)).add_layer_by_copy_ops([lt.CopyOperation.new(["/escape"], linked_ctx, "/", "/dst/")])


def test_layer_and_on_disk_copy_agree_on_symlinked_sources(tmp_path, linked_ctx):
    """The layer (addToLayer) and the on-disk copy (CopyOperation.Execute) of the same operation describe the same
    files -- they disagreed while only Execute resolved its sources."""
    dst_root = tmp_path / "fsroot"
    dst_root.mkdir()
    # --chown to the caller (without it the copy is owned by 0:0), so the copy needs no privilege
    host.copy_op_execute(host.CopyOperation(["/linkdir"], linked_ctx, "/", str(dst_root / "dst"), os.getuid(), os.getgid()),
                         host.MKHOST_COPY_CHOWN)
    on_disk = sorted(os.path.relpath(os.path.join(d, f), dst_root) for d, ds, fs in os.walk(dst_root) for f in fs + ds)
    ents = _layer_both(tmp_path, linked_ctx, ["/linkdir"], "/dst")
    assert on_disk == sorted(e[1].lstrip("/") for e in ents)


# ---- TestGetAncestors (mem_fs_test.go:340-570) through scan + copy -----------------------------------------------
def _scan_both(root):
    for d, _, _ in os.walk(root):
        os.utime(d, (T0, T0))
    o = lt.MemFS(lambda: NOW, str(root))
    h = host.MemFS(str(root))
    assert h.describe_scan(NOW) == _desc_from_oracle(o.add_layer_by_scan())
    return o, h


def _copy_both(o, h, ctx, dst):
    got = h.describe_copy_ops(NOW, [host.CopyOperation(["/payload"], ctx, "/", dst)])
    want = _desc_from_oracle(o.add_layer_by_copy_ops([lt.CopyOperation.new(["/payload"], ctx, "/", dst)]))
    assert got == want
    return [(l.split(" ")[0], l.split(" ")[6]) for l in got]


@pytest.fixture
def payload_ctx(tmp_path):
    c = str(tmp_path / "ctx")
    _mk(c, "payload/p.txt", b"p")
    for d, _, _ in os.walk(c):
        os.utime(d, (T0, T0))
    return c


def test_get_ancestors_follow_symlink_full_resolve(tmp_path, payload_ctx):  # mem_fs_test.go:437-482
    root = tmp_path / "r"
    for d in ["test11/test12/ignore1", "test21/test22/ignore2"]:
        os.makedirs(root / d)
    os.symlink(str(root) + "/test11", root / "test21" / "test22" / "link")  # createHeader trims the root: Linkname "/test11"
    o, h = _scan_both(root)
    # addAncestors(l, "/test21/test22/link/test12", inclusive) resolves to /test11/test12 and re-adds the four
    # ancestors the reference's test requires (n21, n22, n23 = the link, n11) plus test12 itself (inclusive)
    ents = _copy_both(o, h, payload_ctx, "/test21/test22/link/test12/")
    assert ents == [("5", "/test11"), ("5", "/test11/test12"), ("0", "/test11/test12/p.txt"), ("5", "/test21"),
                    ("5", "/test21/test22"), ("2", "/test21/test22/link")]
    h.close()


def test_get_ancestors_follow_symlink_partial_resolve(tmp_path, payload_ctx):  # mem_fs_test.go:484-536
    root = tmp_path / "r"
    os.makedirs(root / "test11" / "test12")
    os.chmod(root / "test11" / "test12", 0o777)
    os.makedirs(root / "test21" / "test22")
    os.symlink(str(root) + "/test11", root / "test21" / "test22" / "link")  # createHeader trims the root: Linkname "/test11"
    o, h = _scan_both(root)
    got = h.describe_copy_ops(NOW + 9, [host.CopyOperation(["/payload"], payload_ctx, "/", "/test21/test22/link/test12/test13/nonexistent/")])
    dsts = [(l.split(" ")[0], l.split(" ")[6]) for l in got]
    assert dsts == [("5", "/test11"), ("5", "/test11/test12"), ("5", "/test11/test12/test13"),
                    ("5", "/test11/test12/test13/nonexistent"), ("0", "/test11/test12/test13/nonexistent/p.txt"),
                    ("5", "/test21"), ("5", "/test21/test22"), ("2", "/test21/test22/link")]
    # hdr13 = createHeader(root, "", "/test11/test12/test13", n12.hdr.FileInfo()); ModTime = clk.Now()  (:522-524):
    # the synthesized directories take test12's mode (0777) and the injected clock
    syn = {l.split(" ")[6]: l.split(" ") for l in got}
    for p in ("/test11/test12/test13", "/test11/test12/test13/nonexistent"):
        assert syn[p][1] == "777" and syn[p][5] == str(NOW + 9) and syn[p][8:] == ["/"]
    o.now = lambda: NOW + 9
    want = _desc_from_oracle(o.add_layer_by_copy_ops(
        [lt.CopyOperation.new(["/payload"], payload_ctx, "/", "/test21/test22/link/test12/test13/nonexistent/")]))
    assert got == want
    h.close()


def test_get_ancestors_detect_symlink_infinite_loop(tmp_path, payload_ctx):  # mem_fs_test.go:538-569
    root = tmp_path / "r"
    os.makedirs(root / "test11")
    os.makedirs(root / "test21")
    os.symlink(str(root) + "/test21/link", root / "test11" / "link")
    os.symlink(str(root) + "/test11/link", root / "test21" / "link")
    o, h = _scan_both(root)
    with pytest.raises(host.HostError) as eh:
        h.describe_copy_ops(NOW, [host.CopyOperation(["/payload"], payload_ctx, "/", "/test21/link/nonexistent/")])
    assert "symlink loop" in str(eh.value)
    with pytest.raises(Exception) as eo:
        o.add_layer_by_copy_ops([lt.CopyOperation.new(["/payload"], payload_ctx, "/", "/test21/link/nonexistent/")])
    assert "symlink loop" in str(eo.value)
    h.close()


def test_get_ancestors_fill_nonexistent_and_inclusive(tmp_path, payload_ctx):  # mem_fs_test.go:341-435
    root = tmp_path / "r"
    os.makedirs(root / "test1" / "test2")
    os.chmod(root / "test1", 0o766)
    os.chmod(root / "test1" / "test2", 0o777)
    o, h = _scan_both(root)
    ents = _copy_both(o, h, payload_ctx, "/test1/test2/")          # Inclusive: both existing ancestors re-added
    assert ents == [("5", "/test1"), ("5", "/test1/test2"), ("0", "/test1/test2/p.txt")]
    ents = _copy_both(o, h, payload_ctx, "/nonexistent1/nonexistent2/")
    assert ents == [("5", "/nonexistent1"), ("5", "/nonexistent1/nonexistent2"), ("0", "/nonexistent1/nonexistent2/p.txt")]
    h.close()


# ---- random contexts full of symlinks: the C++ layer builder against the oracle ------------------------------------
def _random_linked_tree(root, rng):
    """files, directories and symlinks (relative, absolute-inside-the-root, chains, dangling, escaping) under root;
    returns every path (relative, with a leading slash) that exists as a name -- usable as a COPY source."""
    names, dirs = [], [""]
    for i in range(int(rng.integers(6, 14))):
        parent = dirs[int(rng.integers(0, len(dirs)))]
        nm = parent + "/" + "".join(rng.choice(list("abXY01_"), size=int(rng.integers(1, 5)))) + str(i)
        kind = rng.random()
        p = root + nm
        if os.path.lexists(p):
            continue
        if kind < 0.3:
            os.mkdir(p)
            dirs.append(nm)
        elif kind < 0.6 or len(names) < 2:
            with open(p, "wb") as f:
                f.write(bytes(rng.integers(0, 256, int(rng.integers(0, 300)), dtype=np.uint8)))
        else:
            target = names[int(rng.integers(0, len(names)))]
            form = rng.random()
            if form < 0.45:
                os.symlink(os.path.relpath(root + target, os.path.dirname(p)), p)      # relative
            elif form < 0.8:
                os.symlink(root + target, p)                                           # absolute, inside the root
            elif form < 0.9:
                os.symlink("nowhere/at/all", p)                                        # dangling
            else:
                os.symlink("/etc/hostname", p)                                         # escapes the root
        names.append(nm)
    for d, _, _ in os.walk(root):
        os.utime(d, (T0, T0))
    return names


@pytest.mark.parametrize("seed", range(24))
def test_random_symlinked_sources_layer_matches_oracle(tmp_path, seed):
    """COPY <any name of a random symlink-ridden context> <dst>: the layer the C++ side builds (entries, header fields,
    source paths, or the error) equals the oracle's -- both now resolve sources like mem_fs.go:380 does."""
    rng = np.random.default_rng(1000 + seed)
    ctx = str(tmp_path / "ctx")
    os.mkdir(ctx)
    names = _random_linked_tree(ctx, rng)
    root = tmp_path / "root"
    root.mkdir()
    for k in range(6):
        src = names[int(rng.integers(0, len(names)))]
        dst = ["/out%d/" % k, "/out%d/sub/" % k, "/file%d" % k][int(rng.integers(0, 3))]
        try:
            want = _desc_from_oracle(lt.MemFS(lambda: NOW, str(root)).add_layer_by_copy_ops(
                [lt.CopyOperation.new([src], ctx, "/", dst, uid=1, gid=2)]))
            werr = None
        except (OSError, ValueError) as e:
            want, werr = None, e
        try:
            got = host.describe_layer(str(root), NOW, [host.CopyOperation([src], ctx, "/", dst, 1, 2)])
            gerr = None
        except host.HostError as e:
            got, gerr = None, e
        assert (werr is None) == (gerr is None), (src, dst, werr, gerr)
        assert got == want, (src, dst)
