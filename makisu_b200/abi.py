"""ctypes binding of libmksnap.so (include/mksnap.h).

This is the Python face of the C-ABI that a cgo shim would bind (INTEGRATION.md).
It is a thin 1:1 wrapper: every method is one C call.  There is no CPU
fallback: importing works anywhere (so the symbol table can be checked on a
CPU-only box), but creating an engine without a usable B200 raises.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "lib" / "libmksnap.so"

MKSNAP_X_CRC = 1
MKSNAP_X_CDC = 2
MKSNAP_X_MORE = 4   # CDC extent whose file continues in the next submit (reserved = bytes that follow)
MKSNAP_X_CONT = 8   # CDC extent that continues the MORE extent of the previous submit

ERRORS = {0: "OK", -1: "E_INVAL", -2: "E_CUDA", -3: "E_NOMEM", -4: "E_CAPACITY", -5: "E_STATE", -6: "E_NCCL"}


class MksnapError(RuntimeError):
    def __init__(self, code: int, where: str, msg: str):
        super().__init__(f"{where}: {ERRORS.get(code, code)}: {msg}")
        self.code = code


class CdcParams(C.Structure):
    _fields_ = [("min_size", C.c_uint32), ("normal_size", C.c_uint32), ("max_size", C.c_uint32),
                ("strict_bits", C.c_uint32), ("loose_bits", C.c_uint32)]


class Config(C.Structure):
    _fields_ = [("device", C.c_int32), ("n_host_arenas", C.c_uint32), ("host_arena_bytes", C.c_uint64),
                ("device_arena_bytes", C.c_uint64), ("n_device_slots", C.c_uint32), ("reserved0", C.c_uint32),
                ("max_extents", C.c_uint64), ("max_chunks", C.c_uint64), ("cdc", CdcParams)]


class Extent(C.Structure):
    _fields_ = [("arena_off", C.c_uint64), ("len", C.c_uint64), ("crc_suffix", C.c_uint64),
                ("flags", C.c_uint32), ("reserved", C.c_uint32)]


class Range(C.Structure):
    _fields_ = [("arena_off", C.c_uint64), ("len", C.c_uint64), ("stream", C.c_uint32), ("flags", C.c_uint32)]


MKSNAP_R_MORE = 1


class Result(C.Structure):
    _fields_ = [("crc_pure", C.c_uint32), ("reserved", C.c_uint32), ("crc_bytes", C.c_uint64),
                ("cdc_bytes", C.c_uint64), ("n_files", C.c_uint64), ("n_chunks", C.c_uint64),
                ("n_unique", C.c_uint64), ("root", C.c_uint8 * 32), ("n_streams", C.c_uint64)]


class Stats(C.Structure):
    _fields_ = [("ms_total", C.c_float), ("ms_crc", C.c_float), ("ms_scan", C.c_float), ("ms_select", C.c_float),
                ("ms_sha", C.c_float), ("ms_stream", C.c_float), ("ms_h2d", C.c_float), ("ms_sort", C.c_float),
                ("ms_root", C.c_float), ("ms_gather", C.c_float), ("kernel_launches", C.c_uint64),
                ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64)]


class Limits(C.Structure):
    _fields_ = [("max_extents", C.c_uint64), ("max_streams", C.c_uint64), ("max_chunks", C.c_uint64),
                ("host_arena_bytes", C.c_uint64), ("device_arena_bytes", C.c_uint64), ("n_host_arenas", C.c_uint32),
                ("n_device_slots", C.c_uint32), ("carry_bytes", C.c_uint64)]


MKSNAP_CHUNK_KNOWN = 0   # digest is in the index
MKSNAP_CHUNK_NEW = 1     # not in the index; lowest chunk position carrying this digest in the session
MKSNAP_CHUNK_REPEAT = 2  # not in the index; an earlier chunk of the session has the same digest


class DeltaResult(C.Structure):
    _fields_ = [("index_rows", C.c_uint64), ("known_chunks", C.c_uint64), ("new_chunks", C.c_uint64),
                ("repeat_chunks", C.c_uint64), ("known_bytes", C.c_uint64), ("new_bytes", C.c_uint64),
                ("repeat_bytes", C.c_uint64), ("ms_device", C.c_float), ("reserved", C.c_uint32)]


# every symbol include/mksnap.h declares: (name, restype, argtypes)
_P = C.c_void_p
SYMBOLS = [
    ("mksnap_abi_version", C.c_int, []),
    ("mksnap_create", C.c_int, [C.POINTER(Config), C.POINTER(_P)]),
    ("mksnap_destroy", None, [_P]),
    ("mksnap_last_error", C.c_char_p, [_P]),
    ("mksnap_begin", C.c_int, [_P]),
    ("mksnap_arena_acquire", C.c_int, [_P, C.POINTER(_P), C.POINTER(C.c_uint64), C.POINTER(C.c_int32)]),
    ("mksnap_arena_release", C.c_int, [_P, C.c_int32]),
    ("mksnap_get_limits", C.c_int, [_P, C.POINTER(Limits)]),
    ("mksnap_arena_submit", C.c_int, [_P, C.c_int32, C.c_uint64, C.POINTER(Extent), C.c_uint64, C.POINTER(Range), C.c_uint64]),
    ("mksnap_device_arena", C.c_int, [_P, C.c_uint32, C.POINTER(_P), C.POINTER(C.c_uint64)]),
    ("mksnap_device_upload", C.c_int, [_P, C.c_uint32, C.c_uint64, _P, C.c_uint64]),
    ("mksnap_device_submit", C.c_int, [_P, C.c_uint32, C.c_uint64, C.POINTER(Extent), C.c_uint64, C.POINTER(Range), C.c_uint64]),
    ("mksnap_finish", C.c_int, [_P, C.POINTER(Result)]),
    ("mksnap_ctx_crc32", C.c_uint32, [C.POINTER(Result)]),
    ("mksnap_crc_add", C.c_int, [_P, C.c_uint32, C.c_uint64, C.c_uint64]),
    ("mksnap_crc_concat", C.c_uint32, [C.c_uint32, C.c_uint32, C.c_uint64]),
    ("mksnap_get_extent_crcs", C.c_int, [_P, _P, C.c_uint64, C.POINTER(C.c_uint64)]),
    ("mksnap_get_chunks", C.c_int, [_P, _P, _P, C.c_uint64]),
    ("mksnap_get_table", C.c_int, [_P, _P, C.c_uint64]),
    ("mksnap_get_stream_digests", C.c_int, [_P, _P, C.c_uint64]),
    ("mksnap_index_create", C.c_int, [_P, C.c_uint64, C.POINTER(_P)]),
    ("mksnap_index_destroy", None, [_P]),
    ("mksnap_index_rows", C.c_uint64, [_P]),
    ("mksnap_index_add_rows", C.c_int, [_P, _P, _P, C.c_uint64]),
    ("mksnap_index_add_table", C.c_int, [_P, _P]),
    ("mksnap_index_get", C.c_int, [_P, _P, _P, C.c_uint64]),
    ("mksnap_delta", C.c_int, [_P, _P, C.POINTER(DeltaResult)]),
    ("mksnap_get_chunk_status", C.c_int, [_P, _P, C.c_uint64]),
    ("mksnap_comm_unique_id", C.c_int, [_P]),
    ("mksnap_comm_init", C.c_int, [_P, _P, C.c_int32, C.c_int32]),
    ("mksnap_table_rows", C.c_uint64, [_P]),
    ("mksnap_allgather_tables", C.c_int, [_P, C.POINTER(Result)]),
    ("mksnap_exchange_tables", C.c_int, [_P, C.POINTER(Result)]),
    ("mksnap_exchange_tables_local", C.c_int, [C.POINTER(_P), C.c_int32, C.POINTER(Result)]),
    ("mksnap_exchange_plan", C.c_int, [C.POINTER(C.c_uint64), C.c_int32, C.c_int32, C.POINTER(C.c_uint64)]),
    ("mksnap_synth_fill", C.c_int, [_P, C.c_uint32, C.c_uint64, C.c_uint64, C.c_uint64]),
    ("mksnap_memset", C.c_int, [_P, C.c_uint32, C.c_uint64, C.c_uint64, C.c_int]),
    ("mksnap_device_download", C.c_int, [_P, C.c_uint32, C.c_uint64, _P, C.c_uint64]),
    ("mksnap_sync", C.c_int, [_P]),
    ("mksnap_stats", C.c_int, [_P, C.POINTER(Stats)]),
    ("mksnap_default_cdc", None, [C.POINTER(CdcParams)]),
    ("mksnap_roll_multiplier", C.c_uint32, []),
]

_lib = None


def load() -> C.CDLL:
    """Load libmksnap.so and bind every declared symbol.  Raises if the library
    is missing: the product has no other code path."""
    global _lib
    if _lib is not None:
        return _lib
    path = str(LIB_PATH)  # the in-tree build only: no environment override, nothing else may stand in for the engine
    if not os.path.exists(path):
        raise FileNotFoundError(
            f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  makisu_b200 has no CPU fallback.")
    lib = C.CDLL(path, mode=C.RTLD_GLOBAL)  # libmkhost resolves mksnap_* against it
    for name, res, args in SYMBOLS:
        fn = getattr(lib, name)  # AttributeError here = ABI drift
        fn.restype = res
        fn.argtypes = args
    if lib.mksnap_abi_version() != 1:
        raise RuntimeError("libmksnap ABI version mismatch")
    _lib = lib
    return lib


def default_cdc() -> CdcParams:
    p = CdcParams()
    load().mksnap_default_cdc(C.byref(p))
    return p


class Engine:
    """One mksnap handle (one GPU)."""

    def __init__(self, device: int = 0, device_arena_bytes: int = 1 << 30, n_host_arenas: int = 0,
                 host_arena_bytes: int = 0, max_extents: int = 1 << 20, max_chunks: int = 0,
                 n_device_slots: int = 0, cdc: CdcParams | None = None):
        self.lib = load()
        cfg = Config()
        cfg.device = device
        cfg.n_host_arenas = n_host_arenas
        cfg.host_arena_bytes = host_arena_bytes
        cfg.device_arena_bytes = device_arena_bytes
        cfg.n_device_slots = n_device_slots
        cfg.max_extents = max_extents
        cfg.max_chunks = max_chunks
        if cdc is not None:
            cfg.cdc = cdc
        self.cfg = cfg
        self.h = _P()
        rc = self.lib.mksnap_create(C.byref(cfg), C.byref(self.h))
        if rc:
            raise MksnapError(rc, "mksnap_create", (self.lib.mksnap_last_error(None) or b"").decode())

    # -- helpers -------------------------------------------------------
    def _ck(self, rc: int, where: str):
        if rc:
            raise MksnapError(rc, where, (self.lib.mksnap_last_error(self.h) or b"").decode())

    def close(self):
        if getattr(self, "h", None):
            self.lib.mksnap_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- session -------------------------------------------------------
    def begin(self):
        self._ck(self.lib.mksnap_begin(self.h), "mksnap_begin")

    def arena_acquire(self):
        ptr, cap, aid = _P(), C.c_uint64(), C.c_int32()
        self._ck(self.lib.mksnap_arena_acquire(self.h, C.byref(ptr), C.byref(cap), C.byref(aid)), "mksnap_arena_acquire")
        return ptr.value, cap.value, aid.value

    def crc_add(self, pure: int, length: int, crc_suffix: int):
        self._ck(self.lib.mksnap_crc_add(self.h, pure, length, crc_suffix), "mksnap_crc_add")

    def get_extent_crcs(self):
        import numpy as np
        n = C.c_uint64()
        self.lib.mksnap_get_extent_crcs(self.h, None, 0, C.byref(n))
        out = np.empty(max(1, n.value), dtype=np.uint32)
        self._ck(self.lib.mksnap_get_extent_crcs(self.h, out.ctypes.data, out.size, C.byref(n)), "mksnap_get_extent_crcs")
        return out[:n.value]

    def arena_release(self, arena_id: int):
        self._ck(self.lib.mksnap_arena_release(self.h, arena_id), "mksnap_arena_release")

    def limits(self) -> Limits:
        out = Limits()
        self._ck(self.lib.mksnap_get_limits(self.h, C.byref(out)), "mksnap_get_limits")
        return out

    @staticmethod
    def _tables(extents, ranges):
        ne = len(extents) if extents is not None else 0
        nr = len(ranges) if ranges is not None else 0
        ea = extents if isinstance(extents, C.Array) else (Extent * max(ne, 1))(*(extents or []))
        ra = ranges if isinstance(ranges, C.Array) else (Range * max(nr, 1))(*(ranges or []))
        return ea, ne, ra, nr

    def arena_submit(self, arena_id: int, used: int, extents, ranges=None):
        ea, ne, ra, nr = self._tables(extents, ranges)
        self._ck(self.lib.mksnap_arena_submit(self.h, arena_id, used, ea, ne, ra, nr), "mksnap_arena_submit")

    def device_submit(self, slot: int, used: int, extents, ranges=None):
        ea, ne, ra, nr = self._tables(extents, ranges)
        self._ck(self.lib.mksnap_device_submit(self.h, slot, used, ea, ne, ra, nr), "mksnap_device_submit")

    def device_upload(self, slot: int, dst_off: int, data):
        import numpy as np
        a = np.ascontiguousarray(np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else data)
        self._ck(self.lib.mksnap_device_upload(self.h, slot, dst_off, a.ctypes.data, a.nbytes), "mksnap_device_upload")

    def device_download(self, slot: int, src_off: int, n: int):
        import numpy as np
        out = np.empty(n, dtype=np.uint8)
        self._ck(self.lib.mksnap_device_download(self.h, slot, src_off, out.ctypes.data, n), "mksnap_device_download")
        return out

    def synth_fill(self, slot: int, byte_off: int, n: int, seed: int):
        self._ck(self.lib.mksnap_synth_fill(self.h, slot, byte_off, n, seed), "mksnap_synth_fill")

    def memset(self, slot: int, byte_off: int, n: int, value: int):
        self._ck(self.lib.mksnap_memset(self.h, slot, byte_off, n, value), "mksnap_memset")

    def finish(self) -> Result:
        r = Result()
        self._ck(self.lib.mksnap_finish(self.h, C.byref(r)), "mksnap_finish")
        return r

    def ctx_crc32(self, res: Result) -> int:
        return int(self.lib.mksnap_ctx_crc32(C.byref(res)))

    def get_chunks(self, n: int):
        import numpy as np
        ends = np.empty(max(n, 1), dtype=np.uint64)
        dig = np.empty((max(n, 1), 32), dtype=np.uint8)
        self._ck(self.lib.mksnap_get_chunks(self.h, ends.ctypes.data, dig.ctypes.data, n), "mksnap_get_chunks")
        return ends[:n], dig[:n]

    def get_table(self, n: int):
        import numpy as np
        t = np.empty((max(n, 1), 32), dtype=np.uint8)
        self._ck(self.lib.mksnap_get_table(self.h, t.ctypes.data, n), "mksnap_get_table")
        return t[:n]

    def table_rows(self) -> int:
        return int(self.lib.mksnap_table_rows(self.h))

    def get_stream_digests(self, n: int):
        import numpy as np
        t = np.empty((max(n, 1), 32), dtype=np.uint8)
        self._ck(self.lib.mksnap_get_stream_digests(self.h, t.ctypes.data, n), "mksnap_get_stream_digests")
        return t[:n]

    def sync(self):
        self._ck(self.lib.mksnap_sync(self.h), "mksnap_sync")

    def stats(self) -> Stats:
        s = Stats()
        self._ck(self.lib.mksnap_stats(self.h, C.byref(s)), "mksnap_stats")
        return s

    # -- chunk delta ---------------------------------------------------
    def delta(self, ix: "ChunkIndex") -> DeltaResult:
        """Classify every chunk of the finished session against `ix` (MKSNAP_CHUNK_KNOWN / NEW / REPEAT)."""
        r = DeltaResult()
        self._ck(self.lib.mksnap_delta(self.h, ix.ix, C.byref(r)), "mksnap_delta")
        return r

    def chunk_status(self, n: int):
        """The statuses of the last delta, one uint8 per chunk in get_chunks order."""
        import numpy as np
        out = np.empty(max(n, 1), dtype=np.uint8)
        self._ck(self.lib.mksnap_get_chunk_status(self.h, out.ctypes.data, n), "mksnap_get_chunk_status")
        return out[:n]

    # -- multi GPU -----------------------------------------------------
    @staticmethod
    def comm_unique_id() -> bytes:
        buf = (C.c_uint8 * 128)()
        rc = load().mksnap_comm_unique_id(buf)
        if rc:
            raise MksnapError(rc, "mksnap_comm_unique_id", (load().mksnap_last_error(None) or b"").decode())
        return bytes(buf)

    def comm_init(self, uid: bytes, n_ranks: int, rank: int):
        buf = (C.c_uint8 * 128).from_buffer_copy(uid)
        self._ck(self.lib.mksnap_comm_init(self.h, buf, n_ranks, rank), "mksnap_comm_init")

    def allgather_tables(self) -> Result:
        r = Result()
        self._ck(self.lib.mksnap_allgather_tables(self.h, C.byref(r)), "mksnap_allgather_tables")
        return r

    def exchange_tables(self) -> Result:
        """Range-partitioned form of the exchange step (NCCL all-to-all); get_table then returns this rank's range."""
        r = Result()
        self._ck(self.lib.mksnap_exchange_tables(self.h, C.byref(r)), "mksnap_exchange_tables")
        return r

    @staticmethod
    def exchange_tables_local(engines) -> list:
        """The same exchange between engines of this process on one device (engine i = rank i)."""
        n = len(engines)
        hs = (_P * n)(*[e.h for e in engines])
        outs = (Result * n)()
        rc = engines[0].lib.mksnap_exchange_tables_local(hs, n, outs)
        if rc:
            msgs = [(e.lib.mksnap_last_error(e.h) or b"").decode() for e in engines]
            raise MksnapError(rc, "mksnap_exchange_tables_local", "; ".join(m for m in msgs if m))
        return [outs[i] for i in range(n)]


class ChunkIndex:
    """A device-resident sorted-unique set of chunk digests (mksnap_index_*), created on `eng`'s device.  Every call
    takes an engine on that device; close() before the engine it was created on is closed."""

    def __init__(self, eng: Engine, capacity_rows: int):
        self.lib = eng.lib
        self.capacity = capacity_rows
        self.ix = _P()
        eng._ck(self.lib.mksnap_index_create(eng.h, capacity_rows, C.byref(self.ix)), "mksnap_index_create")

    def rows(self) -> int:
        return int(self.lib.mksnap_index_rows(self.ix))

    def add_rows(self, eng: Engine, rows):
        """Union with host rows: an (n, 32) uint8 array, strictly ascending bytewise."""
        import numpy as np
        a = np.ascontiguousarray(rows, dtype=np.uint8).reshape(-1, 32)
        eng._ck(self.lib.mksnap_index_add_rows(eng.h, self.ix, a.ctypes.data if a.size else None, a.shape[0]),
                "mksnap_index_add_rows")

    def add_table(self, eng: Engine):
        """Union with eng's finished session table."""
        eng._ck(self.lib.mksnap_index_add_table(eng.h, self.ix), "mksnap_index_add_table")

    def get(self, eng: Engine):
        import numpy as np
        n = self.rows()
        out = np.empty((max(n, 1), 32), dtype=np.uint8)
        eng._ck(self.lib.mksnap_index_get(eng.h, self.ix, out.ctypes.data, n), "mksnap_index_get")
        return out[:n]

    def close(self):
        if getattr(self, "ix", None):
            self.lib.mksnap_index_destroy(self.ix)
            self.ix = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


def exchange_plan(rows_per_rank, rank: int) -> dict:
    """mksnap_exchange_plan: the device code's own statement of shard.level0_plan (host arithmetic only)."""
    n = len(rows_per_rank)
    arr = (C.c_uint64 * n)(*[int(x) for x in rows_per_rank])
    out = (C.c_uint64 * 7)()
    rc = load().mksnap_exchange_plan(arr, n, rank, out)
    if rc:
        raise MksnapError(rc, "mksnap_exchange_plan", "")
    return dict(zip(["U", "g0", "lead", "full", "tail_own", "borrowed", "groups"], [int(v) for v in out]))


def roll_multiplier() -> int:
    return int(load().mksnap_roll_multiplier())
