"""ctypes binding of libmkhost.so (include/mkhost.h): the C++ host side above the mksnap C-ABI.

Mirrors the reference names: context_crc32 ~ addCopyStep.SetCacheID, commit_copy_ops ~ commitLayer over
MemFS.AddLayerByCopyOps, encode_tar_header ~ tario.WriteHeader.  No hashing happens here or in libmkhost.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from pathlib import Path
from typing import List, Optional, Sequence

from . import abi

LIB_PATH = Path(__file__).resolve().parent / "lib" / "libmkhost.so"


class TarHeader(C.Structure):
    _fields_ = [("name", C.c_char_p), ("linkname", C.c_char_p), ("mode", C.c_int64), ("uid", C.c_int64),
                ("gid", C.c_int64), ("size", C.c_int64), ("mtime_ns", C.c_int64), ("typeflag", C.c_char)]


class CopyOp(C.Structure):
    _fields_ = [("src_root", C.c_char_p), ("srcs", C.POINTER(C.c_char_p)), ("n_srcs", C.c_size_t),
                ("work_dir", C.c_char_p), ("dst", C.c_char_p), ("uid", C.c_int32), ("gid", C.c_int32)]


class CrcCacheStats(C.Structure):
    _fields_ = [("files_total", C.c_uint64), ("files_reused", C.c_uint64), ("bytes_total", C.c_uint64), ("bytes_sent", C.c_uint64)]


class LayerSpec(C.Structure):
    _fields_ = [("ops", C.POINTER(CopyOp)), ("n_ops", C.c_size_t), ("tar_fd", C.c_int)]


class LayerResult(C.Structure):
    _fields_ = [("tar_digest", C.c_uint8 * 32), ("root", C.c_uint8 * 32), ("n_entries", C.c_uint64),
                ("tar_bytes", C.c_uint64), ("n_chunks", C.c_uint64), ("n_unique", C.c_uint64)]


_P = C.c_void_p
SYMBOLS = [
    ("mkhost_encode_tar_header", C.c_size_t, [C.POINTER(TarHeader), _P, C.c_size_t]),
    ("mkhost_context_crc32", C.c_int, [_P, _P, C.c_size_t, C.c_char_p, C.POINTER(C.c_char_p), C.c_size_t, C.c_int,
                                       C.POINTER(C.c_uint32), C.POINTER(C.c_uint64), C.c_char_p, C.c_size_t]),
    ("mkhost_crc_cache_new", _P, []),
    ("mkhost_crc_cache_free", None, [_P]),
    ("mkhost_crc_cache_size", C.c_uint64, [_P]),
    ("mkhost_crc_cache_save", C.c_int, [_P, C.c_char_p, C.c_char_p, C.c_size_t]),
    ("mkhost_crc_cache_load", C.c_int, [_P, C.c_char_p, C.c_char_p, C.c_size_t]),
    ("mkhost_context_crc32_cached", C.c_int, [_P, _P, _P, C.c_size_t, C.c_char_p, C.POINTER(C.c_char_p), C.c_size_t, C.c_int,
                                              C.POINTER(C.c_uint32), C.POINTER(C.c_uint64), C.POINTER(CrcCacheStats), C.c_char_p,
                                              C.c_size_t]),
    ("mkhost_commit_copy_ops", C.c_int, [_P, C.c_char_p, C.c_int64, C.POINTER(CopyOp), C.c_size_t, C.c_int,
                                         C.POINTER(LayerResult), C.c_char_p, C.c_size_t]),
    ("mkhost_commit_copy_ops_to_fd", C.c_int, [_P, C.c_char_p, C.c_int64, C.POINTER(CopyOp), C.c_size_t, C.c_int, C.c_int,
                                               C.POINTER(LayerResult), C.c_char_p, C.c_size_t]),
    ("mkhost_commit_copy_ops_ex", C.c_int, [_P, C.c_char_p, C.c_int64, C.POINTER(CopyOp), C.c_size_t, C.c_int, C.c_int,
                                            C.c_uint32, C.POINTER(LayerResult), C.c_char_p, C.c_size_t]),
    ("mkhost_memfs_new", _P, [C.c_char_p, C.POINTER(C.c_char_p), C.c_size_t, C.c_char_p, C.c_size_t]),
    ("mkhost_memfs_free", None, [_P]),
    ("mkhost_memfs_file_digest", C.c_int, [_P, C.c_char_p, C.POINTER(C.c_uint8)]),
    ("mkhost_memfs_commit_copy_ops", C.c_int, [_P, _P, C.c_int64, C.POINTER(CopyOp), C.c_size_t, C.c_int, C.c_int, C.c_uint32,
                                               C.POINTER(LayerResult), C.c_char_p, C.c_size_t]),
    ("mkhost_memfs_commit_layers", C.c_int, [_P, _P, C.c_int64, C.POINTER(LayerSpec), C.c_size_t, C.c_int, C.c_uint32,
                                             C.POINTER(LayerResult), C.c_char_p, C.c_size_t]),
    ("mkhost_memfs_commit_scan", C.c_int, [_P, _P, C.c_int64, C.c_int, C.c_int, C.c_uint32, C.POINTER(LayerResult),
                                           C.c_char_p, C.c_size_t]),
    ("mkhost_memfs_describe_copy_ops", C.c_size_t, [_P, C.c_int64, C.POINTER(CopyOp), C.c_size_t, C.c_char_p, C.c_size_t,
                                                    C.c_char_p, C.c_size_t]),
    ("mkhost_memfs_describe_scan", C.c_size_t, [_P, C.c_int64, C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t]),
    ("mkhost_memfs_update_from_tar", C.c_int, [_P, _P, C.c_int64, C.c_int, C.c_uint32, C.POINTER(LayerResult), C.c_char_p,
                                               C.c_size_t]),
    ("mkhost_memfs_describe_update_from_tar_ex", C.c_size_t, [_P, C.c_int64, C.c_int, C.c_uint32, C.c_char_p, C.c_size_t,
                                                              C.c_char_p, C.c_size_t]),
    ("mkhost_memfs_describe_update_from_tar", C.c_size_t, [_P, C.c_int64, C.c_int, C.c_char_p, C.c_size_t, C.c_char_p,
                                                           C.c_size_t]),
    ("mkhost_copy_op_execute", C.c_int, [C.POINTER(CopyOp), C.c_uint32, C.POINTER(C.c_char_p), C.c_size_t, C.c_char_p, C.c_size_t]),
    ("mkhost_eval_symlinks", C.c_size_t, [C.c_char_p, C.c_char_p, C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t]),
    ("mkhost_cache_key", C.c_size_t, [C.c_char_p, C.c_int, C.c_char_p, C.c_size_t]),
    ("mkhost_cache_entry_create", C.c_size_t, [C.c_char_p, C.c_char_p, C.c_char_p, C.c_size_t]),
    ("mkhost_cache_entry_parse", C.c_int, [C.c_char_p, C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t]),
    ("mkhost_cache_chunk_entry_create", C.c_size_t, [C.POINTER(C.c_uint8), C.c_uint64, C.c_char_p, C.c_size_t]),
    ("mkhost_cache_chunk_entry_parse", C.c_int, [C.c_char_p, C.POINTER(C.c_uint8), C.POINTER(C.c_uint64), C.c_char_p,
                                                 C.c_size_t]),
    ("mkhost_describe_context_stream", C.c_size_t, [C.c_char_p, C.POINTER(C.c_char_p), C.c_size_t, C.c_char_p,
                                                    C.c_size_t, C.c_char_p, C.c_size_t]),
    ("mkhost_describe_layer", C.c_size_t, [C.c_char_p, C.c_int64, C.POINTER(CopyOp), C.c_size_t, C.c_char_p,
                                           C.c_size_t, C.c_char_p, C.c_size_t]),
]

_lib = None


def load() -> C.CDLL:
    global _lib
    if _lib is None:
        abi.load()  # libmksnap first (libmkhost links against it)
        if not LIB_PATH.exists():
            raise FileNotFoundError(f"{LIB_PATH} not found: run __graft_entry__.build()")
        lib = C.CDLL(str(LIB_PATH))
        for name, res, args in SYMBOLS:
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


class HostError(RuntimeError):
    pass


def _strs(items: Sequence[str]):
    arr = (C.c_char_p * max(1, len(items)))(*[os.fsencode(s) for s in items])
    return arr


@dataclass
class CopyOperation:
    """snapshot.NewCopyOperation(srcs, srcRoot, workDir, dst, chown...) (lib/snapshot/copy_op.go:45)."""
    srcs: List[str]
    src_root: str
    work_dir: str
    dst: str
    uid: int = 0
    gid: int = 0


def _ops(ops: Sequence[CopyOperation]):
    keep = []
    arr = (CopyOp * max(1, len(ops)))()
    for i, o in enumerate(ops):
        s = _strs(o.srcs)
        keep.append(s)
        arr[i].src_root = os.fsencode(o.src_root)
        arr[i].srcs = s
        arr[i].n_srcs = len(o.srcs)
        arr[i].work_dir = os.fsencode(o.work_dir)
        arr[i].dst = os.fsencode(o.dst)
        arr[i].uid, arr[i].gid = o.uid, o.gid
    return arr, keep


def encode_tar_header(name: str, mode: int, uid: int, gid: int, size: int, mtime_ns: int, typeflag: bytes,
                      linkname: str = "") -> bytes:
    h = TarHeader(os.fsencode(name), os.fsencode(linkname), mode, uid, gid, size, mtime_ns, typeflag)
    buf = C.create_string_buffer(8192)
    n = load().mkhost_encode_tar_header(C.byref(h), buf, len(buf))
    if n == 0:
        raise HostError("header not encodable")
    return buf.raw[:n]


def describe_context_stream(context_dir: str, from_paths: Sequence[str]) -> List[str]:
    err = C.create_string_buffer(1024)
    p = _strs(from_paths)
    n = load().mkhost_describe_context_stream(os.fsencode(context_dir), p, len(from_paths), None, 0, err, len(err))
    if n == 0:
        raise HostError(err.value.decode())
    buf = C.create_string_buffer(n)
    load().mkhost_describe_context_stream(os.fsencode(context_dir), p, len(from_paths), buf, n, err, len(err))
    return [l for l in os.fsdecode(buf.value).split("\n") if l]


def describe_layer(root_dir: str, now_unix: int, ops: Sequence[CopyOperation]) -> List[str]:
    err = C.create_string_buffer(1024)
    arr, keep = _ops(ops)
    n = load().mkhost_describe_layer(os.fsencode(root_dir), now_unix, arr, len(ops), None, 0, err, len(err))
    if n == 0:
        raise HostError(err.value.decode())
    buf = C.create_string_buffer(n)
    arr, keep = _ops(ops)
    load().mkhost_describe_layer(os.fsencode(root_dir), now_unix, arr, len(ops), buf, n, err, len(err))
    return [l for l in os.fsdecode(buf.value).split("\n") if l]


def context_crc32(eng: abi.Engine, prefix: bytes, context_dir: str, from_paths: Sequence[str], n_threads: int = 0):
    """-> (crc32 value as checksum.Sum32() would return it, stream length)."""
    err = C.create_string_buffer(1024)
    crc, slen = C.c_uint32(), C.c_uint64()
    rc = load().mkhost_context_crc32(eng.h, prefix, len(prefix), os.fsencode(context_dir), _strs(from_paths),
                                     len(from_paths), n_threads, C.byref(crc), C.byref(slen), err, len(err))
    if rc:
        raise HostError(err.value.decode())
    return crc.value, slen.value


def copy_step_cache_id(eng: abi.Engine, seed: str, directive: str, args: str, context_dir: str,
                       from_paths: Sequence[str]) -> str:
    crc, _ = context_crc32(eng, (seed + directive + args).encode(), context_dir, from_paths)
    return "%x" % crc  # add_copy_step.go:119


MKHOST_NO_TAR_DIGEST = 1
MKHOST_FILE_DIGESTS = 2   # remember per-file SHA-256 in the MemFS tree
MKHOST_SCAN_CONTENT = 4   # content-aware AddLayerByScan (implies FILE_DIGESTS)
MKHOST_MATERIALIZE = 8    # commit_copy_ops also performs the copy onto the file system, from the arena
MKHOST_MATERIALIZE_CHOWN = 16
MKHOST_UNTAR = 32         # UpdateFromTarReader(untar=true): also write the members under the root
MKHOST_LAYER_TABLES = 64  # commit_layers: per-layer chunk tables (a grouped engine session, layer i = group i)
MKHOST_COPY_CHOWN, MKHOST_COPY_INTERNAL, MKHOST_COPY_PRESERVE_OWNER, MKHOST_COPY_DEFERRED = 1, 2, 4, 8


def commit_copy_ops(eng: abi.Engine, root_dir: str, now_unix: int, ops: Sequence[CopyOperation], n_threads: int = 0,
                    tar_fd: int = -1, flags: int = 0):
    """commitLayer over AddLayerByCopyOps; tar_fd >= 0 also receives the uncompressed layer tar."""
    err = C.create_string_buffer(1024)
    arr, keep = _ops(ops)
    out = LayerResult()
    rc = load().mkhost_commit_copy_ops_ex(eng.h, os.fsencode(root_dir), now_unix, arr, len(ops), n_threads, tar_fd, flags,
                                          C.byref(out), err, len(err))
    if rc:
        raise HostError(err.value.decode())
    return {"tar_digest": "sha256:" + bytes(out.tar_digest).hex(), "root": bytes(out.root), "n_entries": out.n_entries,
            "tar_bytes": out.tar_bytes, "n_chunks": out.n_chunks, "n_unique": out.n_unique}


def _layer_dict(out: LayerResult):
    return {"tar_digest": "sha256:" + bytes(out.tar_digest).hex(), "root": bytes(out.root), "n_entries": out.n_entries,
            "tar_bytes": out.tar_bytes, "n_chunks": out.n_chunks, "n_unique": out.n_unique}


class MemFS:
    """snapshot.NewMemFS(clk, root, blacklist): layers accumulate; AddLayerByCopyOps / AddLayerByScan either
    described as text (no GPU) or committed through an Engine."""
    _BUF = 16 << 20

    def __init__(self, root: str, blacklist: Sequence[str] = ()):
        err = C.create_string_buffer(1024)
        self._bl = _strs(list(blacklist))
        self.h = load().mkhost_memfs_new(os.fsencode(root), self._bl, len(blacklist), err, len(err))
        if not self.h:
            raise HostError(err.value.decode())

    def close(self):
        if getattr(self, "h", None):
            load().mkhost_memfs_free(self.h)
            self.h = None

    __del__ = close

    def describe_copy_ops(self, now_unix: int, ops: Sequence[CopyOperation]) -> List[str]:
        err, buf = C.create_string_buffer(1024), C.create_string_buffer(self._BUF)
        arr, keep = _ops(ops)
        n = load().mkhost_memfs_describe_copy_ops(self.h, now_unix, arr, len(ops), buf, len(buf), err, len(err))
        if n == 0 or n > len(buf):
            raise HostError(err.value.decode() or "describe buffer too small")
        return [l for l in os.fsdecode(buf.value).split("\n") if l]

    def describe_scan(self, now_unix: int) -> List[str]:
        err, buf = C.create_string_buffer(1024), C.create_string_buffer(self._BUF)
        n = load().mkhost_memfs_describe_scan(self.h, now_unix, buf, len(buf), err, len(err))
        if n == 0 or n > len(buf):
            raise HostError(err.value.decode() or "describe buffer too small")
        return [l for l in os.fsdecode(buf.value).split("\n") if l]

    def commit_copy_ops(self, eng: abi.Engine, now_unix: int, ops: Sequence[CopyOperation], n_threads: int = 0,
                        tar_fd: int = -1, flags: int = 0):
        err, out = C.create_string_buffer(1024), LayerResult()
        arr, keep = _ops(ops)
        if load().mkhost_memfs_commit_copy_ops(self.h, eng.h, now_unix, arr, len(ops), n_threads, tar_fd, flags,
                                               C.byref(out), err, len(err)):
            raise HostError(err.value.decode())
        return _layer_dict(out)

    def commit_layers(self, eng: abi.Engine, now_unix: int, layers: Sequence[Sequence[CopyOperation]], n_threads: int = 0,
                      tar_fds: Optional[Sequence[int]] = None, flags: int = 0, layer_tables: bool = False):
        """Consecutive layers of one build in ONE engine session (all TarDigest chains advance together).  root /
        n_chunks / n_unique describe the whole batch, or with layer_tables=True each layer's own chunk table; the
        grouped session then stays open on eng for delta_groups / group_table / ChunkIndex.add_group."""
        err = C.create_string_buffer(1024)
        n = len(layers)
        if layer_tables:
            flags |= MKHOST_LAYER_TABLES
        specs, keep, outs = (LayerSpec * max(1, n))(), [], (LayerResult * max(1, n))()
        for i, ops in enumerate(layers):
            arr, k = _ops(ops)
            keep.append((arr, k))
            specs[i].ops, specs[i].n_ops = arr, len(ops)
            specs[i].tar_fd = tar_fds[i] if tar_fds is not None else -1
        if load().mkhost_memfs_commit_layers(self.h, eng.h, now_unix, specs, n, n_threads, flags, outs, err, len(err)):
            raise HostError(err.value.decode())
        eng.n_groups = n if flags & MKHOST_LAYER_TABLES else 0
        return [_layer_dict(outs[i]) for i in range(n)]

    def file_digest(self, dst: str) -> Optional[bytes]:
        """SHA-256 the tree remembers for the regular file at dst, or None."""
        out = (C.c_uint8 * 32)()
        return bytes(out) if load().mkhost_memfs_file_digest(self.h, os.fsencode(dst), out) == 0 else None

    def describe_update_from_tar(self, now_unix: int, tar_fd: int, flags: int = 0) -> List[str]:
        """UpdateFromTarReader without a GPU: the merged layer as text (flags: MKHOST_UNTAR writes the members)."""
        err, buf = C.create_string_buffer(1024), C.create_string_buffer(self._BUF)
        n = load().mkhost_memfs_describe_update_from_tar_ex(self.h, now_unix, tar_fd, flags, buf, len(buf), err, len(err))
        if n == 0 or n > len(buf):
            raise HostError(err.value.decode() or "describe buffer too small")
        return [l for l in os.fsdecode(buf.value).split("\n") if l]

    def update_from_tar(self, eng: abi.Engine, now_unix: int, tar_fd: int, flags: int = 0):
        """UpdateFromTarReader(untar=false) through the GPU: DiffID of the blob + chunk table of its files."""
        err, out = C.create_string_buffer(1024), LayerResult()
        if load().mkhost_memfs_update_from_tar(self.h, eng.h, now_unix, tar_fd, flags, C.byref(out), err, len(err)):
            raise HostError(err.value.decode())
        return _layer_dict(out)

    def commit_scan(self, eng: abi.Engine, now_unix: int, n_threads: int = 0, tar_fd: int = -1, flags: int = 0):
        err, out = C.create_string_buffer(1024), LayerResult()
        if load().mkhost_memfs_commit_scan(self.h, eng.h, now_unix, n_threads, tar_fd, flags, C.byref(out), err, len(err)):
            raise HostError(err.value.decode())
        return _layer_dict(out)


# ---- cache.Manager wire format (lib/cache/cache_manager.go:34-35,239-252) --------------------------
def cache_key(cache_id: str, chunk_table: bool = False) -> str:
    buf = C.create_string_buffer(len(cache_id) + 64)
    load().mkhost_cache_key(cache_id.encode(), int(chunk_table), buf, len(buf))
    return buf.value.decode()


def cache_entry_create(tar_hex: Optional[str], gzip_hex: str = "") -> str:
    buf = C.create_string_buffer(len(tar_hex or "") + len(gzip_hex) + 32)
    load().mkhost_cache_entry_create(None if tar_hex is None else tar_hex.encode(), gzip_hex.encode(), buf, len(buf))
    return buf.value.decode()


def cache_entry_parse(entry: str):
    t, g, err = C.create_string_buffer(len(entry) + 16), C.create_string_buffer(len(entry) + 16), C.create_string_buffer(512)
    if load().mkhost_cache_entry_parse(entry.encode(), t, len(t), g, len(g), err, len(err)):
        raise HostError(err.value.decode())
    return t.value.decode(), g.value.decode()


def cache_chunk_entry_create(root: bytes, n_unique: int) -> str:
    buf = C.create_string_buffer(128)
    load().mkhost_cache_chunk_entry_create((C.c_uint8 * 32).from_buffer_copy(root), n_unique, buf, len(buf))
    return buf.value.decode()


def cache_chunk_entry_parse(entry: str):
    root, n, err = (C.c_uint8 * 32)(), C.c_uint64(), C.create_string_buffer(512)
    if load().mkhost_cache_chunk_entry_parse(entry.encode(), root, C.byref(n), err, len(err)):
        raise HostError(err.value.decode())
    return bytes(root), n.value


def copy_op_execute(op: "CopyOperation", mode: int = 0, blacklist: Sequence[str] = ()) -> None:
    """CopyOperation.Execute (lib/snapshot/copy_op.go:82-147) through fileio.Copier's rules."""
    err = C.create_string_buffer(1024)
    arr, keep = _ops([op])
    bl = _strs(list(blacklist))
    if load().mkhost_copy_op_execute(arr, mode, bl, len(blacklist), err, len(err)):
        raise HostError(err.value.decode())


def eval_symlinks(path: str, src_root: str) -> str:
    """evalSymlinks(p, srcRoot) (lib/snapshot/utils.go:249-324)."""
    err, buf = C.create_string_buffer(1024), C.create_string_buffer(8192)
    n = load().mkhost_eval_symlinks(os.fsencode(path), os.fsencode(src_root), buf, len(buf), err, len(err))
    if n == 0 or n > len(buf):
        raise HostError(err.value.decode() or "path too long")
    return os.fsdecode(buf.value)


class CrcCache:
    """pure(file content) per context file, remembered between builds: unchanged files are folded into the cacheID on
    the host, only changed files travel to the device (include/mkhost.h, "Incremental cacheID")."""

    def __init__(self, path: Optional[str] = None):
        self.h = load().mkhost_crc_cache_new()
        if path is not None and os.path.exists(path):
            err = C.create_string_buffer(512)
            if load().mkhost_crc_cache_load(self.h, os.fsencode(path), err, len(err)):
                raise HostError(err.value.decode())

    def __len__(self):
        return int(load().mkhost_crc_cache_size(self.h))

    def save(self, path: str):
        err = C.create_string_buffer(512)
        if load().mkhost_crc_cache_save(self.h, os.fsencode(path), err, len(err)):
            raise HostError(err.value.decode())

    def close(self):
        if getattr(self, "h", None):
            load().mkhost_crc_cache_free(self.h)
            self.h = None

    __del__ = close

    def context_crc32(self, eng: abi.Engine, prefix: bytes, context_dir: str, from_paths: Sequence[str], n_threads: int = 0):
        """-> (crc32 as checksum.Sum32() returns it, stream length, stats dict)."""
        err = C.create_string_buffer(1024)
        crc, slen, st = C.c_uint32(), C.c_uint64(), CrcCacheStats()
        rc = load().mkhost_context_crc32_cached(eng.h, self.h, prefix, len(prefix), os.fsencode(context_dir), _strs(from_paths),
                                                len(from_paths), n_threads, C.byref(crc), C.byref(slen), C.byref(st), err, len(err))
        if rc:
            raise HostError(err.value.decode())
        return crc.value, slen.value, {k: getattr(st, k) for k, _ in CrcCacheStats._fields_}
