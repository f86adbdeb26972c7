#!/usr/bin/env python
"""bench.py -- snapshot+hash throughput of the B200 path, next to the reference-equivalent CPU path.

  python bench.py --gpus 1 --steps 5 --warmup 3                 (own arm, default)
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
         --master-port P bench.py --gpus N --steps K --warmup W   (N > 1, one rank per GPU)
  python bench.py --impl reference --gpus 1 --steps 3 --warmup 1  (reference arm: oracle port on host cores)
  python bench.py --gpus 1 --steps 5 --warmup 3 --dump-outputs DIR  (also writes the last step's outputs as .npy)

A "step" = one pass of the hot path over one build context per GPU:
  CRC-32 context fingerprint (cacheID, bit-exact reference arithmetic) + Roll-32 CDC + per-chunk SHA-256
  + sort/unique + Merkle root [+ the NCCL table exchange when N > 1: range-partitioned all-to-all by default
  (checked untimed against the all-gather merge first, fallback to it on disagreement), --merge allgather for the other].
Workload = BASELINE.json configs[2]: 100k files x 512 KiB (48.83 GiB) synthetic, per GPU (weak scaling:
the file list shards by rank, every rank owns a full-size shard).  Inputs are 48.8 GiB >> 126 MB L2, so no
L2 flush is needed between timed iterations.

value  : device-resident arena (bytes already in HBM), wall time around K steps with a barrier + device
         synchronize on both sides, max over ranks.
e2e    : same work through mksnap_arena_acquire/submit with PINNED HOST arenas: every step copies the whole
         context host->device in batches (overlapped with compute) and reads the result struct back.
TarDigest (serial SHA-256 per layer stream) is reported separately in "tar_digest" (DESIGN.md section 5).
cpu_baseline    : the reference-equivalent CPU path (single thread like the reference's goroutines) on a bounded sample.
cpu_best_effort : all host threads doing the SAME work as the GPU step (CRC-32 + Roll-32 CDC + SHA-NI chunk SHA-256).
"""
from __future__ import annotations

import argparse
import ctypes
import hashlib
import json
import os
import subprocess
import sys
import threading
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GiB = float(1 << 30)
EXT_DT = np.dtype([("arena_off", "<u8"), ("len", "<u8"), ("crc_suffix", "<u8"), ("flags", "<u4"), ("reserved", "<u4")])


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--files", type=int, default=100_000)
    ap.add_argument("--file-kib", type=int, default=512)
    ap.add_argument("--dirs", type=int, default=256)
    ap.add_argument("--batch-mib", type=int, default=1024, help="pinned host arena size for the e2e path")
    ap.add_argument("--host-pool", type=int, default=8, help="distinct pinned arenas cycled by the e2e path")
    ap.add_argument("--cpu-sample-mib", type=int, default=1536)
    ap.add_argument("--merge", default="exchange", choices=["exchange", "allgather"],
                    help="N>1: range-partitioned all-to-all exchange (default) or all-gather of whole tables")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--workload", default="uniform", choices=["uniform", "dup", "zipf"],
                    help="uniform = BASELINE configs[2] (the bench line); dup = configs[4] (80 %% repeated content); "
                         "zipf = configs[3] (Zipf-sized files 10 B..1 GiB, LPT-sharded by rank)")
    ap.add_argument("--tar-files", type=int, default=256, help="files in the TarDigest side measurement")
    ap.add_argument("--fs-files", type=int, default=16384, help="files of the e2e_fs leg (real files on tmpfs); 0 = skip")
    ap.add_argument("--fs-dir", default="/dev/shm")
    ap.add_argument("--fs-threads", type=int, default=16, help="reader threads of the e2e_fs leg (16 measured best on the 2-socket box: profiles/r2b_fs_threads.txt)")
    ap.add_argument("--fs-arena-mib", type=int, default=1024)
    ap.add_argument("--fs-only", action="store_true", help="run only the e2e_fs leg and print its object (tuning aid, not the bench line)")
    ap.add_argument("--strong", action="store_true", help="run the strong-scaling legs at N=1 too (always run at N>1)")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--no-deliverables", action="store_true", help="skip the {cacheID, TarDigest} same-deliverables leg")
    ap.add_argument("--deliv-one-layer-mib", type=int, default=256, help="sample size of the ONE-layer TarDigest run")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last device-resident step computed to DIR/<name>.npy "
                         "(single-process runs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_ROWS = 65536  # chunk-table rows kept by --dump-outputs: a seeded sample when the table is longer (about 18 MB in all)


def dump_outputs(eng, res, out_dir: str):
    """What a caller of the device-resident path receives from one step, as float64 / float32 arrays (every value is
    exact in them): the result struct, the context CRC-32 (cacheID), and the same seeded sample of rows of the chunk
    list (end offset + SHA-256) and of the sorted unique-digest table."""
    os.makedirs(out_dir, exist_ok=True)
    n_chunks, n_unique = int(res.n_chunks), int(res.n_unique)
    ends, digs = eng.get_chunks(n_chunks)
    table = eng.get_table(n_unique)

    def rows(n):
        if n <= DUMP_ROWS:
            return np.arange(n)
        return np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))
    ci, ti = rows(n_chunks), rows(n_unique)
    arrays = {
        "result_counts": np.array([res.crc_bytes, res.cdc_bytes, res.n_files, n_chunks, n_unique], dtype=np.float64),
        "cache_id_crc32": np.array([eng.ctx_crc32(res)], dtype=np.float64),
        "merkle_root": np.frombuffer(bytes(res.root), dtype=np.uint8).astype(np.float32),
        "chunk_rows": ci.astype(np.float64),
        "chunk_ends": ends[ci].astype(np.float64),
        "chunk_sha256": digs[ci].astype(np.float32),
        "table_rows": ti.astype(np.float64),
        "table_sha256": table[ti].astype(np.float32),
    }
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ----------------------------------------------------------------------------------------------------
# workload description (pure host arithmetic, vectorised)
# ----------------------------------------------------------------------------------------------------
def context_layout(n_files: int, file_bytes: int, n_dirs: int, rank: int):
    """Files d%03d/f%06d.bin in filepath.Walk order.  Returns (file offsets, meta blob, meta offsets, extents)
    where the CRC stream is: ".", then per dir its relpath, then per file relpath + content
    (reference add_copy_step.go:194-238)."""
    per_dir = (n_files + n_dirs - 1) // n_dirs
    names, kinds, fidx = [b"."], [0], [-1]
    k = 0
    for d in range(n_dirs):
        if k >= n_files:
            break
        dn = b"d%03d" % d
        names.append(dn); kinds.append(0); fidx.append(-1)
        for _ in range(min(per_dir, n_files - k)):
            names.append(dn + b"/f%06d_r%d.bin" % (k, rank)); kinds.append(1); fidx.append(k)
            k += 1
    stride = file_bytes  # multiple of 512: files are packed back to back, tar-block aligned
    file_off = np.arange(n_files, dtype=np.uint64) * np.uint64(stride)
    data_end = int(n_files) * stride
    # meta region: path strings, each 16-byte aligned
    lens = np.array([len(n) for n in names], dtype=np.uint64)
    moff = np.zeros(len(names), dtype=np.uint64)
    pos = 0
    blob = bytearray()
    for i, n in enumerate(names):
        moff[i] = pos
        blob += n + b"\0" * (-len(n) % 16)
        pos += (len(n) + 15) // 16 * 16
    blob += b"\0" * (-len(blob) % 512)
    meta_base = (data_end + 511) // 512 * 512
    # stream segments in order: name_i [, content_i]
    kinds_a = np.array(kinds)
    fidx_a = np.array(fidx)
    nseg = len(names) + int((kinds_a == 1).sum())
    ext = np.zeros(nseg, dtype=EXT_DT)
    is_file = kinds_a == 1
    pos_name = np.arange(len(names)) + np.concatenate([[0], np.cumsum(is_file)[:-1]])
    ext["arena_off"][pos_name] = moff + np.uint64(meta_base)
    ext["len"][pos_name] = lens
    ext["flags"][pos_name] = 1
    pos_file = pos_name[is_file] + 1
    ext["arena_off"][pos_file] = file_off[fidx_a[is_file]]
    ext["len"][pos_file] = file_bytes
    ext["flags"][pos_file] = 1 | 2
    total = int(ext["len"].sum())
    ext["crc_suffix"] = np.uint64(total) - np.cumsum(ext["len"]).astype(np.uint64)
    used = meta_base + len(blob)
    return dict(file_off=file_off, blob=bytes(blob), meta_base=meta_base, ext=ext, used=used, stream_len=total,
                data_bytes=data_end)


def layout_from_files(names, file_off, file_len, data_end):
    """CRC stream = name_i || content_i in list order; every file is also a CDC extent.  Paths go to a meta
    region after the data.  file_off may repeat (dup workload: several files share one pool region)."""
    n = len(names)
    lens = np.array([len(x) for x in names], dtype=np.uint64)
    moff = np.concatenate([[0], np.cumsum((lens + 15) // 16 * 16)[:-1]]).astype(np.uint64)
    blob = bytearray(int(((lens + 15) // 16 * 16).sum()))
    for i, x in enumerate(names):
        blob[int(moff[i]):int(moff[i]) + len(x)] = x
    blob += b"\0" * (-len(blob) % 512)
    meta_base = (int(data_end) + 511) // 512 * 512
    ext = np.zeros(2 * n, dtype=EXT_DT)
    ext["arena_off"][0::2] = moff + np.uint64(meta_base)
    ext["len"][0::2] = lens
    ext["flags"][0::2] = 1
    ext["arena_off"][1::2] = file_off
    ext["len"][1::2] = file_len
    ext["flags"][1::2] = 3
    total = int(ext["len"].sum())
    ext["crc_suffix"] = np.uint64(total) - np.cumsum(ext["len"]).astype(np.uint64)
    return dict(blob=bytes(blob), meta_base=meta_base, ext=ext, used=meta_base + len(blob), stream_len=total,
                data_bytes=int(np.asarray(file_len, dtype=np.uint64).sum()), fill_bytes=int(data_end))


def special_layout(args, rank, world):
    """dup: n files of file_kib drawn (with repetition) from a pool holding 20 % as many distinct regions.
    zipf: sizes ~ Zipf(1.1)*10 B clipped to [10 B, 1 GiB] until ~files*file_kib bytes in total, whole list LPT-sharded."""
    from makisu_b200 import shard
    fb = args.file_kib << 10
    rng = np.random.default_rng(0xC5 if args.workload == "dup" else 0xC4)
    if args.workload == "dup":
        pool = max(1, args.files // 5)
        pick = rng.integers(0, pool, args.files)
        pick[:pool] = np.arange(pool)  # every pool region appears at least once
        names = [b"d%03d/f%06d_r%d.bin" % (i % args.dirs, i, rank) for i in range(args.files)]
        return layout_from_files(names, pick.astype(np.uint64) * np.uint64(fb), np.full(args.files, fb, dtype=np.uint64), pool * fb), None
    target = args.files * fb
    sizes = []
    tot = 0
    while tot < target:
        z = np.clip(rng.zipf(1.1, 4096).astype(np.float64) * 10, 10, 1 << 30).astype(np.int64)
        for v in z:
            if tot >= target:
                break
            sizes.append(int(v))
            tot += int(v)
    sizes = np.array(sizes, dtype=np.int64)
    shards = shard.lpt_shard(sizes, world)
    mine = shards[rank]
    ml = sizes[mine]
    off = np.concatenate([[0], np.cumsum((ml + 511) // 512 * 512)[:-1]]).astype(np.uint64)
    data_end = int(off[-1] + (ml[-1] + 511) // 512 * 512) if len(ml) else 0
    names = [b"z/f%07d.bin" % i for i in mine]
    info = {"n_files_total": int(len(sizes)), "imbalance": shard.imbalance(sizes, shards), "largest_file": int(sizes.max())}
    return layout_from_files(names, off, ml.astype(np.uint64), data_end), info


def global_sharded_layout(names, sizes, rank, world, region_of=None, region_bytes=0, n_regions=0):
    """ONE global context (stream = name_i || content_i, i ascending) whose files are LPT-sharded over `world` ranks:
    the strong-scaling form of the path (SURVEY section 8e).  A rank packs its own files (512-aligned, or -- dup --
    the shared pool regions they point at) and their names; crc_suffix is GLOBAL, so the XOR of the rank partials is
    the cacheID of the whole context and the exchanged table is the table of the whole context at every N."""
    from makisu_b200 import shard
    sizes = np.asarray(sizes, dtype=np.uint64)
    n = len(names)
    nlen = np.array([len(x) for x in names], dtype=np.uint64)
    seg = np.empty(2 * n, dtype=np.uint64)
    seg[0::2], seg[1::2] = nlen, sizes
    total = int(seg.sum())
    suffix = (np.uint64(total) - np.cumsum(seg)).astype(np.uint64)
    shards = shard.lpt_shard(sizes.tolist(), world) if world > 1 else [list(range(n))]
    mine = np.array(shards[rank], dtype=np.int64)
    ml = sizes[mine]
    if region_of is None:
        pad = (ml + np.uint64(511)) // np.uint64(512) * np.uint64(512)
        off = (np.cumsum(pad) - pad).astype(np.uint64)
        data_end = int(pad.sum())
        fill = data_end
    else:
        off = (np.asarray(region_of)[mine].astype(np.uint64) * np.uint64(region_bytes))
        data_end = fill = n_regions * region_bytes
    mlen = nlen[mine]
    mpad = (mlen + np.uint64(15)) // np.uint64(16) * np.uint64(16)
    moff = (np.cumsum(mpad) - mpad).astype(np.uint64)
    blob = bytearray(int(mpad.sum()))
    for j, i in enumerate(mine):
        x = names[i]
        blob[int(moff[j]):int(moff[j]) + len(x)] = x
    blob += b"\0" * (-len(blob) % 512)
    meta_base = (data_end + 511) // 512 * 512
    ext = np.zeros(2 * len(mine), dtype=EXT_DT)
    ext["arena_off"][0::2] = moff + np.uint64(meta_base)
    ext["len"][0::2] = mlen
    ext["flags"][0::2] = 1
    ext["crc_suffix"][0::2] = suffix[2 * mine]
    ext["arena_off"][1::2] = off
    ext["len"][1::2] = ml
    ext["flags"][1::2] = 3
    ext["crc_suffix"][1::2] = suffix[2 * mine + 1]
    loads = [int(sizes[np.array(s_, dtype=np.int64)].sum()) if len(s_) else 0 for s_ in shards]
    info = {"n_files_total": n, "bytes_total": int(sizes.sum()), "files_this_rank": int(len(mine)),
            "imbalance_max_over_mean": max(loads) / (sum(loads) / len(loads)) if sum(loads) else 1.0,
            "largest_file": int(sizes.max()) if n else 0}
    return dict(blob=bytes(blob), meta_base=meta_base, ext=ext, used=meta_base + len(blob), stream_len=total,
                data_bytes=int(ml.sum()), fill_bytes=int(fill)), info


def strong_contexts(args):
    """The fixed-size contexts of BASELINE configs[2..4], as (names, sizes, region_of, n_regions) generators."""
    fb = args.file_kib << 10

    def uniform():
        names = [b"d%03d/f%06d.bin" % (i * args.dirs // args.files, i) for i in range(args.files)]
        return names, np.full(args.files, fb, dtype=np.uint64), None, 0

    def dup():
        rng = np.random.default_rng(0xC5)
        pool = max(1, args.files // 5)
        pick = rng.integers(0, pool, args.files)
        pick[:pool] = np.arange(pool)
        names = [b"d%03d/f%06d.bin" % (i % args.dirs, i) for i in range(args.files)]
        return names, np.full(args.files, fb, dtype=np.uint64), pick, pool

    def zipf():
        rng = np.random.default_rng(0xC4)
        target = args.files * fb
        sizes, tot = [], 0
        while tot < target:
            z = np.clip(rng.zipf(1.1, 4096).astype(np.float64) * 10, 10, 1 << 30).astype(np.int64)
            for v in z:
                if tot >= target:
                    break
                sizes.append(int(v))
                tot += int(v)
        names = [b"z/f%07d.bin" % i for i in range(len(sizes))]
        return names, np.array(sizes, dtype=np.uint64), None, 0
    return {"uniform": uniform, "dup": dup, "zipf": zipf}


def ext_ptr(a: np.ndarray):
    from makisu_b200.abi import Extent
    return ctypes.cast(a.ctypes.data, ctypes.POINTER(Extent))


# ----------------------------------------------------------------------------------------------------
def clocks_sampler(dev_index: int, stop: threading.Event, out: list):
    """SM clock + throttle reasons of this rank's GPU DURING the timed region.  NVML polled every 20 ms (a timed region
    is only a few hundred ms; spawning nvidia-smi can take longer than that on an 8-GPU box); nvidia-smi -lms as the
    fallback when NVML cannot be used.  Rows: [sm_mhz, sm_max_mhz, hw_slowdown, hw_thermal, sw_thermal, sw_power_cap]."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(dev_index)
        mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
        bits = [0x8, 0x40, 0x20, 0x4]  # HwSlowdown, HwThermalSlowdown, SwThermalSlowdown, SwPowerCap
        pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
        pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
    except Exception:
        h = None
    if h is not None:
        while not stop.is_set():
            try:
                sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                r = int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                out.append([str(sm), str(mx)] + [("Active" if r & b else "Not Active") for b in bits])
            except Exception:
                break
            stop.wait(0.02)
        return
    q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    try:
        p = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(dev_index),
                              "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    except Exception:
        return
    try:
        while not stop.is_set():
            line = p.stdout.readline()
            if not line:
                break
            out.append([x.strip() for x in line.split(",")])
    finally:
        p.terminate()


def summarize_clocks(rows):
    if not rows:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
    sm = sorted(int(r[0]) for r in rows if r[0].isdigit())
    mx = max(int(r[1]) for r in rows if r[1].isdigit())
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].startswith("Active") for r in rows)]
    return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": reasons, "samples": len(rows)}


def bind_to_gpu_numa_node(dev: int) -> str:
    """Pin this process to the CPUs next to its GPU before any pinned arena is allocated, so the e2e path's
    host buffers sit on the GPU's socket (first touch) and H2D does not cross the inter-socket link."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(dev)
        n = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, n)
        cpus = [64 * i + b for i, w in enumerate(mask) for b in range(64) if (w >> b) & 1]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return f"cpus {cpus[0]}-{cpus[-1]} ({len(cpus)})"
    except Exception as e:  # affinity is an optimisation, never a requirement
        return f"unbound ({type(e).__name__})"
    return "unbound"


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------------------------
# CPU side: the oracle port of the reference path, timed on a bounded sample
# ----------------------------------------------------------------------------------------------------
def cpu_reference_pass(sample_mib: int, file_bytes: int):
    """One pass of the reference-equivalent CPU path over `sample_mib` of the same workload, single thread
    like the reference (one goroutine for the CRC walk, add_copy_step.go:153-169; one for tar -> SHA-256,
    common.go:53-58; gzip excluded, which favours the reference):
      pass 1  crc32 over relpath + content of every file   (cacheID)
      pass 3  SHA-256 over header + padded content          (TarDigest)"""
    import oracle.lib as o
    L = o.L()
    n_files = max(1, (sample_mib << 20) // file_bytes)
    buf = o.synth_fill(0, n_files * file_bytes, 0xC3)
    t0 = time.perf_counter()
    crc = 0
    for i in range(n_files):
        name = b"d%03d/f%06d.bin" % (i % 256, i)
        crc = zlib.crc32(name, crc)
        crc = L.mko_crc32_update(crc, buf.ctypes.data + i * file_bytes, file_bytes)
    t1 = time.perf_counter()
    hdr = np.zeros(512, dtype=np.uint8)
    ctx = (ctypes.c_uint8 * 128)()
    L.mko_sha256_init.argtypes = [ctypes.c_void_p]
    L.mko_sha256_update_fast.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t]
    L.mko_sha256_final.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
    L.mko_sha256_init(ctx)
    for i in range(n_files):  # SHA-NI when the host has it: at least as fast as Go 1.14's AVX2 assembly
        L.mko_sha256_update_fast(ctx, hdr.ctypes.data, 512)
        L.mko_sha256_update_fast(ctx, buf.ctypes.data + i * file_bytes, file_bytes)
    out = (ctypes.c_uint8 * 32)()
    L.mko_sha256_final(ctx, out)
    t2 = time.perf_counter()
    nbytes = n_files * file_bytes
    return dict(bytes=nbytes, s_crc=t1 - t0, s_sha=t2 - t1, s_total=t2 - t0, crc="%x" % crc, n_files=n_files,
                sha_impl="SHA-NI" if L.mko_have_sha_ni() else "scalar")


def cpu_reference_extras(file_bytes: int, threads: int):
    """Two informational figures SURVEY section 8d asks for next to the CPU baseline (they do NOT enter cpu_baseline.value, which
    stays the most favourable reading of the reference): SHA-256 without the x86 SHA extensions (Go 1.14's crypto/sha256
    had none), and a deflate level-6 sink on `threads` threads over 1 MiB blocks standing in for pgzip (the reference
    joins tar->sha256 and tar->pgzip per 32 KiB write, so its layer pass runs at the slower of the two)."""
    import oracle.lib as o
    L = o.L()
    n = 64 << 20
    buf = o.synth_fill(0, n, 0xC3)
    out = (ctypes.c_uint8 * 32)()
    t0 = time.perf_counter()
    L.mko_sha256(buf.ctypes.data, n, out)                       # the scalar FIPS 180-4 restatement
    sha_scalar = n / GiB / (time.perf_counter() - t0)
    blocks = [bytes(buf[i:i + (1 << 20)]) for i in range(0, n, 1 << 20)] * max(1, threads // 8)
    idx = iter(range(len(blocks)))
    lock = threading.Lock()

    def work():
        while True:
            with lock:
                i = next(idx, None)
            if i is None:
                return
            zlib.compress(blocks[i], 6)                          # releases the GIL
    ths = [threading.Thread(target=work) for _ in range(threads)]
    t0 = time.perf_counter()
    for th in ths:
        th.start()
    for th in ths:
        th.join()
    gz = len(blocks) * (1 << 20) / GiB / (time.perf_counter() - t0)
    return {"sha256_scalar_GiBps": sha_scalar, "deflate6_GiBps": gz, "deflate_threads": threads,
            "note": "synthetic content is incompressible: deflate runs at its slowest here"}


def cpu_same_work_pass(file_bytes: int, threads: int, files_per_thread: int = 192):
    """Best-effort CPU figure (SURVEY section 8d): the SAME work as one GPU step -- CRC-32 of every file, Roll-32 CDC, SHA-256
    of every chunk (SHA-NI when present) -- on `threads` host threads over disjoint slices of files
    (oracle/mkoracle.c mko_step_same_work; ctypes releases the GIL).  Sort/unique/root are left out (tiny)."""
    import oracle.lib as o
    L = o.L()
    n_files = threads * files_per_thread
    buf = o.synth_fill(0, n_files * file_bytes, 0xC3)
    offs = np.arange(n_files, dtype=np.uint64) * np.uint64(file_bytes)
    lens = np.full(n_files, file_bytes, dtype=np.uint64)
    prm = o.default_params()
    sinks = (ctypes.c_uint32 * threads)()
    counts = [0] * threads

    def work(t):
        lo = t * files_per_thread
        counts[t] = L.mko_step_same_work(buf.ctypes.data, offs[lo:].ctypes.data, lens[lo:].ctypes.data, files_per_thread,
                                         ctypes.byref(prm), None, None, 0, ctypes.byref(sinks, 4 * t))
    ths = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
    t0 = time.perf_counter()
    for th in ths:
        th.start()
    for th in ths:
        th.join()
    dt = time.perf_counter() - t0
    return dict(bytes=n_files * file_bytes, s=dt, n_files=n_files, chunks=sum(counts),
                sha_impl="SHA-NI" if L.mko_have_sha_ni() else "scalar")


def fs_leg(args, local, rank):
    """e2e_fs: the same path from REAL FILES on tmpfs through the C++ host side (libmkhost: filepath.Walk-ordered
    walker, parallel pread into the pinned arenas, tar headers) -- what a `makisu build` would actually drive:
      cacheID          mkhost_context_crc32                      (add_copy_step.go:102-122)
      commit           mkhost_memfs_commit_copy_ops, 1 layer     (common.go:67-111; chunk table, TarDigest left to the caller)
      commit_layers    mkhost_memfs_commit_layers, one layer per directory WITH TarDigest (the reference's deliverables)
    Gate: cacheID and TarDigest of a sub-context against the oracle's file-based restatement (zlib / hashlib)."""
    import shutil
    from concurrent.futures import ThreadPoolExecutor
    from makisu_b200 import host
    from makisu_b200.abi import Engine
    from oracle import ctx_crc, layer_tar as lt
    fb = args.file_kib << 10
    n_files, n_dirs = args.fs_files, min(args.dirs, max(1, args.fs_files // 8))
    base = os.path.join(args.fs_dir, "mkbench_r%d" % rank)
    shutil.rmtree(base, ignore_errors=True)
    ctx, root = os.path.join(base, "ctx"), os.path.join(base, "root")
    os.makedirs(root)
    for d in range(n_dirs):
        os.makedirs(os.path.join(ctx, "d%03d" % d))
    total = n_files * fb
    threads = max(1, min(len(os.sched_getaffinity(0)), args.fs_threads))
    arena = args.fs_arena_mib << 20
    t_create = time.perf_counter()
    with Engine(device=local, device_arena_bytes=arena, n_host_arenas=max(4, (4 << 30) // arena), host_arena_bytes=arena, n_device_slots=2,
                max_extents=1 << 16, max_chunks=total // 4096 + n_files + (1 << 16)) as eng:
        # content: device generator -> host -> files (written by a few threads; tmpfs)
        per = max(1, arena // fb)
        def write_one(args_):
            path, buf = args_
            with open(path, "wb") as f:
                f.write(buf)
        with ThreadPoolExecutor(max_workers=min(16, threads)) as ex:
            for b0 in range(0, n_files, per):
                nb = min(per, n_files - b0)
                eng.synth_fill(0, 0, nb * fb, 0xF5 + 1000 * rank + b0)
                blob = eng.device_download(0, 0, nb * fb)
                list(ex.map(write_one, [(os.path.join(ctx, "d%03d" % ((b0 + i) * n_dirs // n_files), "f%06d.bin" % (b0 + i)),
                                         blob[i * fb:(i + 1) * fb]) for i in range(nb)]))
        for d, _, _ in os.walk(ctx):
            os.utime(d, (1_500_000_000, 1_500_000_000))
        t_create = time.perf_counter() - t_create
        seed = ctx_crc.from_step_cache_id(ctx_crc.plan_seed(True, False), "scratch")
        prefix = (seed + "COPY" + ". /app/").encode()
        # gate on a sub-context (2 directories): GPU vs the oracle's zlib / hashlib restatement
        sub = ["d000", "d001"] if n_dirs > 1 else ["d000"]
        want_id = ctx_crc.copy_step_cache_id(seed, "COPY", " ".join(sub) + " /app/", ctx, sub)
        got_id = host.copy_step_cache_id(eng, seed, "COPY", " ".join(sub) + " /app/", ctx, sub)
        assert got_id == want_id, ("e2e_fs cacheID gate", got_id, want_id)
        o = lt.MemFS(lambda: 1_600_000_000, root)
        want_td = [lt.tar_digest(o.add_layer_by_copy_ops([lt.CopyOperation.new(["/" + d], ctx, "/", "/app/%s/" % d)])) for d in sub]
        got_l = host.MemFS(root).commit_layers(eng, 1_600_000_000, [[host.CopyOperation(["/" + d], ctx, "/", "/app/%s/" % d)] for d in sub],
                                               n_threads=threads)
        assert [g["tar_digest"] for g in got_l] == want_td, "e2e_fs TarDigest gate"
        out = {"files": n_files, "file_kib": args.file_kib, "dirs": n_dirs, "GiB": total / GiB, "tmpfs": args.fs_dir,
               "host_threads": threads, "create_s": t_create, "arena_MiB": arena >> 20,
               "gate": "cacheID and per-layer TarDigest of %d directories equal the oracle's file-based restatement" % len(sub)}
        host.context_crc32(eng, prefix, ctx, ["."], threads)  # warm: page cache, reader pool
        best = {}
        for rep in range(2):
            t0 = time.perf_counter()
            crc, slen = host.context_crc32(eng, prefix, ctx, ["."], threads)
            t1 = time.perf_counter()
            lay1 = host.MemFS(root).commit_copy_ops(eng, 1_600_000_000, [host.CopyOperation(["/"], ctx, "/", "/app/")], threads,
                                                    flags=host.MKHOST_NO_TAR_DIGEST)
            t2 = time.perf_counter()
            layn = host.MemFS(root).commit_layers(eng, 1_600_000_000,
                                                  [[host.CopyOperation(["/d%03d" % d], ctx, "/", "/app/d%03d/" % d)] for d in range(n_dirs)],
                                                  n_threads=threads)
            t3 = time.perf_counter()
            for k, v in (("cacheid_s", t1 - t0), ("commit_1layer_no_tardigest_s", t2 - t1), ("commit_layers_with_tardigest_s", t3 - t2)):
                best[k] = min(best.get(k, 1e30), v)
        out.update(best)
        out.update(cache_id="%x" % crc, n_layers=n_dirs, n_chunks=int(lay1["n_chunks"]),
                   cacheid_GiBps=total / GiB / best["cacheid_s"],
                   commit_1layer_no_tardigest_GiBps=total / GiB / best["commit_1layer_no_tardigest_s"],
                   commit_layers_with_tardigest_GiBps=total / GiB / best["commit_layers_with_tardigest_s"],
                   deliverables_GiBps=total / GiB / (best["cacheid_s"] + best["commit_layers_with_tardigest_s"]),
                   deliverables_note="cacheID pass + commit of %d layers with TarDigest, back to back (the reference reads the context "
                                     "once for each, add_copy_step.go:153 and common.go:69)" % n_dirs)
    shutil.rmtree(base, ignore_errors=True)
    return out


def run_reference_arm(args, emit):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    file_bytes = args.file_kib << 10
    sample_mib = min(args.cpu_sample_mib, 512)
    for _ in range(args.warmup):
        cpu_reference_pass(min(sample_mib, 64), file_bytes)
    tot, dt = 0, 0.0
    last = None
    for _ in range(args.steps):
        last = cpu_reference_pass(sample_mib, file_bytes)  # synthetic content is generated outside the timed part
        tot += last["bytes"]
        dt += last["s_total"]
    v = tot / GiB / dt
    try:  # the same passes with scalar SHA-256 (Go 1.14 had no SHA-extension path): lower bracket of the reference
        sc = cpu_reference_extras(file_bytes, 1)["sha256_scalar_GiBps"]
        v_scalar = last["bytes"] / GiB / (last["s_crc"] + last["bytes"] / GiB / sc)
    except Exception:  # noqa: BLE001
        sc, v_scalar = None, None
    line = {
        "impl": "reference", "metric": "snapshot_hash_throughput", "value": v, "unit": "GiB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": f"{args.files} files x {args.file_kib} KiB per GPU (BASELINE configs[2]); each step = "
                               f"{sample_mib} MiB bounded sample of it", "path": "crc32 context pass + tar SHA-256 pass"},
        "cpu_baseline": {"value": v, "unit": "GiB/s", "cores": 1, "kind": "port",
                         "sample": f"{sample_mib} MiB/step, oracle/mkoracle.c (slicing-8 CRC-32, {last['sha_impl']} SHA-256), single "
                                   f"thread like the reference's goroutine; crc {last['s_crc']:.2f}s sha {last['s_sha']:.2f}s",
                         "value_without_sha_extensions": v_scalar, "sha256_scalar_GiBps": sc,
                         "note": "value uses SHA-NI (generous to the reference: Go 1.14 has no SHA-extension path); "
                                 "value_without_sha_extensions is the lower bracket"},
        "e2e": {"value": v, "unit": "GiB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ----------------------------------------------------------------------------------------------------
def main():
    args = parse()
    if os.environ.get("MKSNAP_BENCH_WATCHDOG"):  # debugging aid: dump every thread's Python stack if the run is still alive after N s
        import faulthandler
        faulthandler.dump_traceback_later(int(os.environ["MKSNAP_BENCH_WATCHDOG"]), repeat=True, file=sys.stderr)
    # stdout carries exactly ONE JSON line: libraries (NCCL prints its version there) get stderr until the end
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(obj), flush=True)
        os.dup2(2, 1)

    if args.impl == "reference":
        run_reference_arm(args, emit)
        return
    if args.fs_only:
        import torch
        torch.cuda.set_device(0)
        bind_to_gpu_numa_node(0)
        emit(fs_leg(args, 0, 0))
        return

    import torch
    import torch.distributed as dist
    from makisu_b200.abi import Engine, Range

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and world > 1:
        raise SystemExit("bench.py: --dump-outputs is for single-process runs (the chunk list of a rank is not the exchanged table's)")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 path has no CPU fallback")
    torch.cuda.set_device(local)
    affinity_note = bind_to_gpu_numa_node(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    file_bytes = args.file_kib << 10
    wl_info = None
    if args.workload == "uniform":
        lay = context_layout(args.files, file_bytes, args.dirs, rank)
        lay["fill_bytes"] = lay["data_bytes"]
    else:
        lay, wl_info = special_layout(args, rank, world)
        args.no_e2e = True  # the e2e leg is defined on the uniform workload
    used = lay["used"]
    arena_bytes = (used + (1 << 20)) // 512 * 512
    n_ext = len(lay["ext"])

    cdc = None
    if os.environ.get("MKSNAP_BENCH_CDC"):  # experiment knob: "min,normal,max,strict_bits,loose_bits" (not the bench line)
        from makisu_b200.abi import CdcParams
        cdc = CdcParams(*[int(v) for v in os.environ["MKSNAP_BENCH_CDC"].split(",")])
    eng = Engine(device=local, device_arena_bytes=arena_bytes, n_host_arenas=0, max_extents=n_ext + 16,
                 max_chunks=max(arena_bytes, lay["data_bytes"]) // 4096 + n_ext + 1024, cdc=cdc)
    if world > 1:
        uid = [Engine.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        eng.comm_init(uid[0], world, rank)

    # ---- synthetic context, generated on the device (seed differs per rank: shards are distinct) ----
    eng.synth_fill(0, 0, (lay["fill_bytes"] + 15) // 16 * 16, 0xC3 + 1000 * rank)
    eng.device_upload(0, lay["meta_base"], np.frombuffer(lay["blob"], dtype=np.uint8))
    eng.sync()
    ext = lay["ext"]

    merge = {"mode": args.merge}

    def one_step():
        eng.begin()
        eng.lib.mksnap_device_submit(eng.h, 0, used, ext_ptr(ext), n_ext, None, 0)
        res = eng.finish()
        if world > 1:
            res = eng.exchange_tables() if merge["mode"] == "exchange" else eng.allgather_tables()
        return res

    if world > 1 and merge["mode"] == "exchange":
        # self-check before anything is timed: the range-partitioned exchange must give the root, CRC and counters of the
        # all-gather merge on this very workload; if any rank disagrees every rank falls back to the all-gather.
        merge["mode"] = "allgather"
        ra = one_step()
        merge["mode"] = "exchange"
        try:
            rx = one_step()
            ok = (bytes(rx.root) == bytes(ra.root) and rx.n_unique == ra.n_unique and rx.crc_pure == ra.crc_pure
                  and rx.n_chunks == ra.n_chunks)
        except Exception as ex:  # noqa: BLE001
            print("exchange failed:", ex, file=sys.stderr)
            ok = False
        flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 0:
            merge["mode"] = "allgather"
            merge["note"] = "exchange self-check failed, fell back to all-gather"

    # ---- correctness gate on a sample (stdlib zlib / hashlib, not the oracle) ----
    gate_files = min(args.files, 8)
    sample = eng.device_download(0, 0, gate_files * file_bytes)
    res0 = one_step()
    res1 = one_step()
    assert bytes(res0.root) == bytes(res1.root) and res0.crc_pure == res1.crc_pure, "non-deterministic digests"
    if world == 1 and args.workload == "uniform":
        eng.begin()
        sub = context_layout(gate_files, file_bytes, 1, rank)
        # same bytes, sub-context of the first files: needs its own meta strings
        eng.device_upload(0, lay["meta_base"], np.frombuffer(sub["blob"], dtype=np.uint8))
        e2 = sub["ext"].copy()
        e2["arena_off"][e2["flags"] == 1] += np.uint64(lay["meta_base"] - sub["meta_base"])
        eng.lib.mksnap_device_submit(eng.h, 0, used, ext_ptr(e2), len(e2), None, 0)
        rs = eng.finish()
        crc = 0
        for i in range(len(e2)):
            if e2["flags"][i] == 1:
                o = int(e2["arena_off"][i]) - lay["meta_base"]
                crc = zlib.crc32(sub["blob"][o:o + int(e2["len"][i])], crc)
            else:
                o = int(e2["arena_off"][i])
                crc = zlib.crc32(sample[o:o + file_bytes].tobytes(), crc)
        assert eng.ctx_crc32(rs) == crc, "CRC-32 gate failed: %x != %x" % (eng.ctx_crc32(rs), crc)
        ends, digs = eng.get_chunks(rs.n_chunks)
        prev = 0
        for e_, d_ in zip(ends[:64], digs[:64]):
            e_ = int(e_)
            if e_ <= prev or e_ > sample.size:
                prev = e_
                continue
            assert hashlib.sha256(sample[prev:e_].tobytes()).digest() == d_.tobytes(), "chunk SHA-256 gate failed"
            prev = e_
        eng.device_upload(0, lay["meta_base"], np.frombuffer(lay["blob"], dtype=np.uint8))
        # same gate at the far end of the arena (offsets ~48.8 GiB): the last file alone
        last_off = (args.files - 1) * file_bytes
        tail = eng.device_download(0, last_off, file_bytes)
        one = np.zeros(1, dtype=EXT_DT)
        one["arena_off"], one["len"], one["crc_suffix"], one["flags"] = last_off, file_bytes, 0, 3
        eng.begin()
        eng.lib.mksnap_device_submit(eng.h, 0, used, ext_ptr(one), 1, None, 0)
        rt = eng.finish()
        assert eng.ctx_crc32(rt) == zlib.crc32(tail.tobytes()), "CRC-32 gate failed at high offset"
        ends, digs = eng.get_chunks(rt.n_chunks)
        prev = last_off
        for e_, d_ in zip(ends, digs):
            e_ = int(e_)
            assert hashlib.sha256(tail[prev - last_off:e_ - last_off].tobytes()).digest() == d_.tobytes(), \
                "chunk SHA-256 gate failed at high offset"
            prev = e_
        assert prev == last_off + file_bytes

    # ---- device-resident timing ----
    for _ in range(args.warmup):
        one_step()
    st0 = eng.stats()
    stop, rows = threading.Event(), []
    th = threading.Thread(target=clocks_sampler, args=(local, stop, rows), daemon=True)
    if rank == 0:
        th.start()
    kern = {k: 0.0 for k in ["ms_crc", "ms_scan", "ms_select", "ms_sha", "ms_sort", "ms_root", "ms_gather"]}
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = one_step()
        s = eng.stats()
        for k in kern:
            kern[k] += getattr(s, k)
    barrier()
    dt = time.perf_counter() - t0
    stop.set()
    st1 = eng.stats()
    dt = max_over_ranks(dt)
    launches = int(st1.kernel_launches - st0.kernel_launches)
    if args.dump_outputs:
        dump_outputs(eng, res, args.dump_outputs)
    ms_step = dt / args.steps * 1e3
    ctx_bytes = lay["data_bytes"]
    value = world * ctx_bytes / GiB / (dt / args.steps)
    for k in kern:
        kern[k] /= args.steps
    peak, peak_src = measured_peak()
    gbs = lambda ms: (ctx_bytes / 1e9) / (ms / 1e3) if ms > 0 else None  # noqa: E731
    kernels = [
        {"name": "K1 k_roll_scan", "bound": "hbm", "ms": kern["ms_scan"], "algorithmic_GBps": gbs(kern["ms_scan"])},
        {"name": "K0 k_crc32_extents", "bound": "hbm", "ms": kern["ms_crc"], "algorithmic_GBps": gbs(kern["ms_crc"])},
        {"name": "K2 k_sha256_ranges(chunks)", "bound": "int-alu", "ms": kern["ms_sha"], "algorithmic_GBps": gbs(kern["ms_sha"])},
        {"name": "K1b k_select_cuts+scan", "bound": "latency", "ms": kern["ms_select"]},
        {"name": "K3 radix sort+unique", "bound": "hbm(small)", "ms": kern["ms_sort"]},
        {"name": "merkle root", "bound": "latency", "ms": kern["ms_root"]},
        {"name": "nccl table exchange (" + merge["mode"] + ")", "bound": "nvlink(small)", "ms": kern["ms_gather"]},
    ]
    for k in kernels:
        if k.get("algorithmic_GBps"):
            k["frac_of_hbm_peak"] = k["algorithmic_GBps"] / peak
        k["share_of_step"] = k["ms"] / ms_step if ms_step else None
    traffic, traffic_src = None, None
    try:  # DRAM bytes of the launch from the committed ncu capture of the FULL-SIZE launch (scaled only when --files differs)
        tj = json.load(open(os.path.join(ROOT, "profiles", "r2b_traffic.json")))["k_roll_scan"]
        if ctx_bytes == tj["algorithmic_bytes"]:
            traffic, traffic_src = tj["dram_bytes_read"] + tj["dram_bytes_write"], tj["source"]
        else:
            traffic, traffic_src = tj["ratio"] * ctx_bytes, tj["source"] + " [scaled by algorithmic bytes]"
    except Exception:
        pass
    roofline = {"kernel": "k_roll_scan (north_star's rolling-hash kernel)", "bound": "hbm",
                "achieved": gbs(kern["ms_scan"]), "peak": peak, "unit": "GB/s",
                "frac": (gbs(kern["ms_scan"]) or 0) / peak, "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": peak_src,
                "algorithmic_bytes_per_launch": ctx_bytes,
                "note": "dominant kernel BY TIME is K2 (SHA-256, integer-ALU bound, not HBM): see kernels[]"}

    # ---- end-to-end: pinned host arenas, H2D inside the timed region ----
    e2e = None
    if not args.no_e2e:
        batch = args.batch_mib << 20
        files_per_batch = max(1, (batch - (1 << 20)) // file_bytes)
        n_batches = (args.files + files_per_batch - 1) // files_per_batch
        pool = min(args.host_pool, n_batches)
        blay = context_layout(files_per_batch, file_bytes, 1, rank)
        # suffixes are per session: recompute per batch below (cheap, vectorised)
        eng2 = Engine(device=local, device_arena_bytes=batch, n_host_arenas=pool, host_arena_bytes=batch,
                      n_device_slots=2, max_extents=len(blay["ext"]) + 16,
                      max_chunks=ctx_bytes // 4096 + args.files + 1024)
        if world > 1:
            uid = [Engine.comm_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(uid, src=0)
            eng2.comm_init(uid[0], world, rank)
        # fill the pool: device generator -> D2H straight into the C-owned pinned arenas
        ids = []
        eng2.begin()
        for b in range(pool):
            ptr, cap, aid = eng2.arena_acquire()
            eng2.synth_fill(0, 0, blay["data_bytes"], 0xE2E + 1000 * rank + b)
            eng2._ck(eng2.lib.mksnap_device_download(eng2.h, 0, 0, ptr, blay["data_bytes"]), "download")
            ctypes.memmove(ptr + blay["meta_base"], blay["blob"], len(blay["blob"]))
            ids.append((ptr, aid))
            eng2.arena_submit(aid, blay["used"], [])  # hand it back (no work)
        eng2.finish()
        stream_total = blay["stream_len"] * n_batches
        per_batch_ext = []
        for b in range(n_batches):
            e = blay["ext"].copy()
            e["crc_suffix"] += np.uint64(blay["stream_len"] * (n_batches - 1 - b))
            per_batch_ext.append(e)

        def e2e_step():
            eng2.begin()
            for b in range(n_batches):
                ptr, cap, aid = eng2.arena_acquire()
                e = per_batch_ext[b]
                eng2._ck(eng2.lib.mksnap_arena_submit(eng2.h, aid, blay["used"], ext_ptr(e), len(e), None, 0), "submit")
            r = eng2.finish()
            if world > 1:
                r = eng2.exchange_tables() if merge["mode"] == "exchange" else eng2.allgather_tables()
            return r

        e2e_step()
        s0 = eng2.stats()
        barrier()
        t0 = time.perf_counter()
        n_e2e = args.steps
        for _ in range(n_e2e):
            r = e2e_step()
        barrier()
        dte = max_over_ranks(time.perf_counter() - t0)
        s1 = eng2.stats()
        e2e_bytes = n_batches * blay["data_bytes"]
        e2e = {"value": world * e2e_bytes / GiB / (dte / n_e2e), "unit": "GiB/s",
               "h2d_bytes_per_step": int((s1.h2d_bytes - s0.h2d_bytes) // n_e2e),
               "d2h_bytes_per_step": int((s1.d2h_bytes - s0.d2h_bytes) // n_e2e),
               "ms_per_step": dte / n_e2e * 1e3, "steps": n_e2e,
               "note": f"{n_batches} batches x {args.batch_mib} MiB pinned arenas/step, pool of {pool} distinct arenas cycled; "
                       f"2 device slots, H2D overlapped with kernels; api = mksnap_arena_acquire/submit/finish"}
        launches_e2e = int(s1.kernel_launches - s0.kernel_launches) // n_e2e
        e2e["gpu_launches_per_step"] = launches_e2e

        # ---- same deliverables as the reference: {cacheID, TarDigest per layer}, host buffers, H2D in the timed region ----
        # The reference commits one layer per step (common.go:67-111); TarDigest is one serial SHA-256 chain per layer.
        # Every pinned arena is split into L equal regions = the pieces of L layer streams (MKSNAP_R_MORE until the last
        # batch), next to the CRC extents of the cacheID: what mkhost_memfs_commit_layers submits for L layers.
        def stream_ranges(L, b, nb, span):
            reg = span // L // 64 * 64
            r = (Range * L)()
            for i in range(L):
                r[i].arena_off = i * reg
                r[i].len = reg if i < L - 1 else span - reg * (L - 1)
                r[i].stream, r[i].flags = i, (1 if b < nb - 1 else 0)
            return r

        def deliv_step(L, nb, with_table, span, check=None):
            eng2.begin()
            seen = []
            for b in range(nb):
                ptr, cap, aid = eng2.arena_acquire()
                seen.append(ptr)
                e = per_batch_ext[b] if with_table else per_batch_crc[b]
                eng2._ck(eng2.lib.mksnap_arena_submit(eng2.h, aid, blay["used"], ext_ptr(e), len(e), stream_ranges(L, b, nb, span), L),
                         "submit")
            r = eng2.finish()
            d = eng2.get_stream_digests(L)
            if check is not None:  # untimed: stdlib SHA-256 over the same pinned bytes
                reg = span // L // 64 * 64
                for i in check:
                    hh = hashlib.sha256()
                    ln = reg if i < L - 1 else span - reg * (L - 1)
                    for ptr in seen:
                        hh.update(ctypes.string_at(ptr + i * reg, ln))
                    assert hh.digest() == d[i].tobytes(), "TarDigest stream %d of %d mismatch" % (i, L)
            return r

        per_batch_crc = []
        for e in per_batch_ext:
            c = e.copy()
            c["flags"] = 1
            per_batch_crc.append(c)
        deliv = {"unit": "GiB/s", "what": "cacheID (CRC-32 of the context stream) + one TarDigest (serial SHA-256) per layer, "
                 "pinned host arenas -> H2D -> kernels -> digests read back; layers = equal slices of the context "
                 "(C3 has 256 directories: 256 = one COPY per directory)", "runs": []}
        if not args.no_deliverables:
            span = blay["data_bytes"]
            for L, with_table in ((256, False), (256, True), (1024, False)):
                if L + 16 > len(blay["ext"]):
                    continue
                deliv_step(L, min(2, n_batches), with_table, span, check=[0, L - 1])
                barrier()
                t0 = time.perf_counter()
                deliv_step(L, n_batches, with_table, span)
                barrier()
                dtd = max_over_ranks(time.perf_counter() - t0)
                deliv["runs"].append({"layers": L, "chunk_table_too": with_table, "bytes_per_gpu": e2e_bytes, "s": dtd,
                                      "value": world * e2e_bytes / GiB / dtd, "sample": "full context"})
            # ONE layer: one chain for the whole context is latency-bound (~0.09 GB/s): bounded sample, extrapolated
            one_span = min(span, args.deliv_one_layer_mib << 20) // 64 * 64
            deliv_step(1, 1, False, one_span, check=[0])
            barrier()
            t0 = time.perf_counter()
            deliv_step(1, 1, False, one_span)
            barrier()
            dt1 = max_over_ranks(time.perf_counter() - t0)
            deliv["runs"].append({"layers": 1, "chunk_table_too": False, "bytes_per_gpu": one_span, "s": dt1,
                                  "value": world * one_span / GiB / dt1,
                                  "sample": f"first {one_span >> 20} MiB of one batch: a single SHA-256 chain cannot be split; "
                                            f"the whole context as ONE layer would take ~{e2e_bytes / one_span * dt1:.0f} s"})
        # ---- strong scaling end to end: the SAME fixed context (args.files files in total) split over the N ranks ----
        if (world > 1 or args.strong) and not args.no_strong:
            counts = [args.files // world + (1 if r_ < args.files % world else 0) for r_ in range(world)]

            def rank_plan(r_):
                nbf_, k_ = divmod(counts[r_], files_per_batch)
                slp = context_layout(k_, file_bytes, 1, r_)["stream_len"] if k_ else 0
                return nbf_, k_, nbf_ * blay["stream_len"] + slp
            plans = [rank_plan(r_) for r_ in range(world)]
            total_stream = sum(p_[2] for p_ in plans)
            after = total_stream - sum(p_[2] for p_ in plans[:rank])
            nbf, k_last, _ = plans[rank]
            sexts = []
            for _ in range(nbf):
                after -= blay["stream_len"]
                e = blay["ext"].copy()
                e["crc_suffix"] += np.uint64(after)
                sexts.append((e, blay["used"], None))
            if k_last:
                lp = context_layout(k_last, file_bytes, 1, rank)
                after -= lp["stream_len"]
                e = lp["ext"].copy()
                e["crc_suffix"] += np.uint64(after)
                sexts.append((e, lp["used"], lp))

            def strong_e2e_step():
                eng2.begin()
                for e, used_b, lp in sexts:
                    ptr, cap, aid = eng2.arena_acquire()
                    if lp is not None:  # the names of a partial batch are packed behind its last file
                        ctypes.memmove(ptr + lp["meta_base"], lp["blob"], len(lp["blob"]))
                    eng2._ck(eng2.lib.mksnap_arena_submit(eng2.h, aid, used_b, ext_ptr(e), len(e), None, 0), "submit")
                r_ = eng2.finish()
                if world > 1:
                    r_ = eng2.exchange_tables() if merge["mode"] == "exchange" else eng2.allgather_tables()
                return r_
            strong_e2e_step()
            barrier()
            t0 = time.perf_counter()
            for _ in range(n_e2e):
                strong_e2e_step()
            barrier()
            dse = max_over_ranks(time.perf_counter() - t0) / n_e2e
            e2e["strong"] = {"value": args.files * file_bytes / GiB / dse, "unit": "GiB/s", "ms_per_step": dse * 1e3,
                             "context_GiB": args.files * file_bytes / GiB, "files_per_rank": counts[rank],
                             "note": "the ONE 100k-file context of BASELINE configs[2] split over the N ranks, pinned host arenas, "
                                     "H2D inside the timed region, table exchange included"}
        eng2.close()

    # ---- strong scaling: ONE fixed-size context sharded over the N ranks (BASELINE configs[2],[3],[4]) ----
    strong = None
    if (world > 1 or args.strong) and args.workload == "uniform" and not args.no_strong:
        strong = {"what": "one GLOBAL context LPT-sharded by file over the N ranks (whole files; global crc_suffix); a step = "
                          "every rank digests its shard + the table exchange; value = bytes of the WHOLE context / max-over-ranks time",
                  "runs": {}}
        fb = file_bytes
        for kind, gen in strong_contexts(args).items():
            names, sizes, region_of, n_regions = gen()
            slay, sinfo = global_sharded_layout(names, sizes, rank, world, region_of, fb, n_regions)
            sa = (slay["used"] + (1 << 20)) // 512 * 512
            ne = len(slay["ext"])
            se = Engine(device=local, device_arena_bytes=sa, n_host_arenas=0, max_extents=ne + 16,
                        max_chunks=max(sa, slay["data_bytes"]) // 4096 + ne + 1024)
            if world > 1:
                uid = [Engine.comm_unique_id() if rank == 0 else None]
                dist.broadcast_object_list(uid, src=0)
                se.comm_init(uid[0], world, rank)
            # dup: the pool (same bytes on every rank: seed and offsets are global); else the rank's own files
            se.synth_fill(0, 0, (slay["fill_bytes"] + 15) // 16 * 16, 0x5C0 + (0 if kind == "dup" else 1000 * rank))
            se.device_upload(0, slay["meta_base"], np.frombuffer(slay["blob"], dtype=np.uint8))
            se.sync()

            def sstep():
                se.begin()
                se.lib.mksnap_device_submit(se.h, 0, slay["used"], ext_ptr(slay["ext"]), ne, None, 0)
                r_ = se.finish()
                if world > 1:
                    r_ = se.exchange_tables() if merge["mode"] == "exchange" else se.allgather_tables()
                return r_
            for _ in range(max(1, args.warmup)):
                sstep()
            barrier()
            t0 = time.perf_counter()
            n_s = args.steps
            for _ in range(n_s):
                sr = sstep()
            barrier()
            dts = max_over_ranks(time.perf_counter() - t0) / n_s
            sst = se.stats()
            run = {"value": sinfo["bytes_total"] / GiB / dts, "unit": "GiB/s", "ms_per_step": dts * 1e3, "steps": n_s,
                   "context_GiB": sinfo["bytes_total"] / GiB, "n_files": sinfo["n_files_total"],
                   "imbalance_max_over_mean": sinfo["imbalance_max_over_mean"], "largest_file": sinfo["largest_file"],
                   "n_chunks": int(sr.n_chunks), "n_unique": int(sr.n_unique),
                   "dedup_ratio_unique_over_total": int(sr.n_unique) / int(sr.n_chunks) if sr.n_chunks else None,
                   "cache_id": "%x" % se.ctx_crc32(sr), "root": bytes(sr.root).hex(),
                   "rank0_ms": {"crc": sst.ms_crc, "scan": sst.ms_scan, "select": sst.ms_select, "sha": sst.ms_sha,
                                "sort": sst.ms_sort, "root": sst.ms_root, "exchange": sst.ms_gather}}
            strong["runs"][kind] = run
            se.close()
    # ---- TarDigest side measurement: serial SHA-256 streams (one per layer) ----
    tar = None
    if rank == 0 and args.tar_files > 0:
        nf = min(args.tar_files, args.files)
        for streams in (1, 64, 256):
            per = nf // streams
            rng_ = (Range * streams)()
            for s_ in range(streams):
                rng_[s_].arena_off = s_ * per * file_bytes
                rng_[s_].len = per * file_bytes
                rng_[s_].stream, rng_[s_].flags = s_, 0
            eng.begin()
            eng.lib.mksnap_device_submit(eng.h, 0, used, None, 0, rng_, streams)
            eng.finish()
            ms = eng.stats().ms_stream
            tar = (tar or []) + [{"streams": streams, "bytes_per_stream": per * file_bytes, "ms": ms,
                                  "GBps": streams * per * file_bytes / 1e9 / (ms / 1e3) if ms else None}]

    # ---- CPU baseline on this box's host cores (rank 0, N == 1 only) ----
    cpu = None
    cpu_best = None
    if rank == 0 and world == 1 and not args.no_cpu:
        c = cpu_reference_pass(args.cpu_sample_mib, file_bytes)
        cpu = {"value": c["bytes"] / GiB / c["s_total"], "unit": "GiB/s", "cores": 1, "kind": "port",
               "sample": f"{c['n_files']} files x {args.file_kib} KiB ({c['bytes'] / GiB:.2f} GiB) of the same workload; "
                         f"crc32 pass {c['s_crc']:.2f}s (slicing-8) + tar SHA-256 pass {c['s_sha']:.2f}s ({c['sha_impl']}), single thread (the reference "
                         f"path is single-goroutine); gzip and the >=1 s sync() floor excluded",
               "host_cpus": os.cpu_count()}
        try:
            cpu["extras"] = cpu_reference_extras(file_bytes, max(1, min(len(os.sched_getaffinity(0)), 64)))
            # Go 1.14's crypto/sha256 has no SHA-extension path (AVX2 assembly, ~0.4-0.5 GB/s): the same two passes with
            # the scalar SHA-256 figure bracket the reference from below, `value` (SHA-NI) from above
            sc = cpu["extras"]["sha256_scalar_GiBps"]
            cpu["value_without_sha_extensions"] = c["bytes"] / GiB / (c["s_crc"] + c["bytes"] / GiB / sc)
            cpu["note"] = "value uses the x86 SHA extensions (generous to the reference); value_without_sha_extensions = same CRC pass + " \
                          "scalar SHA-256 (%.3f GiB/s): Go 1.14's AVX2 assembly sits between the two" % sc
        except Exception as ex:  # noqa: BLE001
            cpu["extras"] = {"unavailable": repr(ex)}
        try:  # honesty figure: all host threads doing what the GPU step does (not the reference's algorithm)
            nt = max(1, min(len(os.sched_getaffinity(0)), 64))
            b = cpu_same_work_pass(file_bytes, nt)
            cpu_best = {"value": b["bytes"] / GiB / b["s"], "unit": "GiB/s", "cores": nt, "kind": "port",
                        "sample": f"{b['n_files']} files x {args.file_kib} KiB ({b['bytes'] / GiB:.2f} GiB): crc32 (slicing-8) + roll32 CDC + "
                                  f"chunk SHA-256 ({b['sha_impl']}) per file on {nt} threads, {b['chunks']} chunks; sort/unique/root excluded"}
        except Exception as ex:  # noqa: BLE001
            cpu_best = {"unavailable": repr(ex)}

    e2e_fs = None
    if rank == 0 and world == 1 and args.fs_files > 0 and args.workload == "uniform" and not args.no_e2e:
        try:
            e2e_fs = fs_leg(args, local, rank)
            if cpu is not None:
                e2e_fs["speedup_vs_cpu_reference_deliverables"] = e2e_fs["deliverables_GiBps"] / cpu["value"]
        except AssertionError:
            raise
        except Exception as ex:  # noqa: BLE001  (tmpfs too small, ...): reported, not fatal for the contract line
            e2e_fs = {"unavailable": repr(ex)}
    deliverables = None
    if e2e is not None:
        deliverables = deliv
        if cpu is not None:  # the reference path's time does not depend on the layer count: one goroutine, layer after layer
            deliverables["cpu_reference_GiBps"] = cpu["value"]
            deliverables["cpu_reference_s_for_context"] = ctx_bytes / GiB / cpu["value"]
            deliverables["cpu_note"] = "oracle port, 1 thread, CRC pass + tar SHA-256 pass (cpu_baseline), extrapolated from its sample"
            for r_ in deliverables["runs"]:
                r_["speedup_vs_cpu_reference"] = r_["value"] / cpu["value"]
    if rank == 0:
        line = {
            "metric": "snapshot_hash_throughput", "value": value, "unit": "GiB/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": f"{args.files} files x {args.file_kib} KiB ({ctx_bytes / GiB:.2f} GiB) per GPU, "
                                   f"{args.dirs} dirs, BASELINE configs[2]",
                       "per_step": "crc32 cacheID + roll32 CDC + chunk SHA-256 + sort/unique + merkle root"
                                   + ((" + nccl " + merge["mode"] + " of the tables" + (" [" + merge["note"] + "]" if "note" in merge else ""))
                                      if world > 1 else ""),
                       "l2": "inputs (48.8 GiB) >> L2 (126 MB): no flush needed", "sharding": f"files by rank, dp{world}",
                       "host_affinity": affinity_note,
                       "n_chunks": int(res.n_chunks), "n_unique": int(res.n_unique), "cache_id": "%x" % eng.ctx_crc32(res),
                       "dedup_ratio_unique_over_total": (int(res.n_unique) / int(res.n_chunks)) if res.n_chunks else None,
                       "workload_kind": args.workload, "workload_info": wl_info,
                       "root": bytes(res.root).hex()},
            "roofline": roofline, "kernels": kernels, "cpu_baseline": cpu, "cpu_best_effort": cpu_best, "e2e": e2e,
            "deliverables": deliverables, "e2e_fs": e2e_fs, "strong": strong,
            "gpu_launches": launches,
            "gpu_launches_per_step": launches // max(1, args.steps), "tar_digest": tar,
            "clocks": summarize_clocks(rows),
        }
        emit(line)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
