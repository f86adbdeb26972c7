/*
 * mksnap.h — C-ABI of libmksnap.so: the B200-native snapshot+hash engine that
 * replaces the CPU arithmetic on makisu's build-context fingerprint and layer
 * digest path.  Plain C, plain pointers and sizes; no torch / C++ types.
 *
 * The reference (uber/makisu @5fdc8f4) has NO FFI on this path: it is direct Go
 * calls inside a CGO_ENABLED=0 binary (reference Makefile:46-49).  The entry
 * points below are what a cgo shim would bind at the three seams SURVEY.md
 * section 8(b) identifies; each one cites the reference code it replaces.  The Go-side
 * stubs are shown in INTEGRATION.md.
 *
 * Model: a handle owns one CUDA device, its streams, a ring of pinned host
 * arenas and device arena slots.  A *session* (begin ... finish) digests one
 * build context / layer: the host packs file bytes into an arena in layer-tar
 * order (512-byte aligned, zero padded -- i.e. the arena *is* the tar stream),
 * describes what to hash with extent / range tables, and submits.  All
 * arithmetic runs on the device; there is no CPU fallback: every call fails
 * with MKSNAP_E_CUDA if no device is usable.
 *
 * Threading: one session per handle at a time, calls on a handle must be
 * serialised by the caller (the reference calls these seams from one goroutine
 * per build: lib/builder/build_plan.go:174, lib/stream/multi_writer.go:60);
 * different handles may be used concurrently.  Every entry point does its own
 * cudaSetDevice, so a goroutine may migrate between OS threads.
 *
 * Errors: 0 = ok, negative = MKSNAP_E_*; text via mksnap_last_error().  A Go
 * wrapper maps them to fmt.Errorf("...: %s", err) like lib/builder/step/common.go:59.
 */
#ifndef MKSNAP_H
#define MKSNAP_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MKSNAP_ABI_VERSION 1

enum {
    MKSNAP_OK = 0,
    MKSNAP_E_INVAL = -1,    /* bad argument / misuse */
    MKSNAP_E_CUDA = -2,     /* CUDA runtime / driver failure, or no device */
    MKSNAP_E_NOMEM = -3,    /* allocation failed */
    MKSNAP_E_CAPACITY = -4, /* batch / table exceeds a configured capacity */
    MKSNAP_E_STATE = -5,    /* call out of sequence */
    MKSNAP_E_NCCL = -6      /* NCCL unavailable or failed */
};

typedef struct mksnap mksnap_t;

/* Content-defined chunking parameters (DESIGN.md section 3; no reference counterpart). */
typedef struct {
    uint32_t min_size;    /* default 4096   (must be >= 64)                     */
    uint32_t normal_size; /* default 16384  (strict mask below, loose at/after) */
    uint32_t max_size;    /* default 131072                                     */
    uint32_t strict_bits; /* default 16: candidate iff the top bits of roll32 are all ones */
    uint32_t loose_bits;  /* default 12                                         */
} mksnap_cdc_params;

typedef struct {
    int32_t device;              /* CUDA ordinal                                      */
    uint32_t n_host_arenas;      /* pinned staging arenas; 0 = device-resident use    */
    uint64_t host_arena_bytes;   /* capacity of each pinned arena                     */
    uint64_t device_arena_bytes; /* capacity of each device arena slot                */
    uint32_t n_device_slots;     /* 0 = auto (2 if host arenas are used, else 1)      */
    uint32_t reserved0;
    uint64_t max_extents;        /* per submit                                        */
    uint64_t max_chunks;         /* per session; 0 = device_arena_bytes/min_size + 3*max_extents + 64 */
    mksnap_cdc_params cdc;       /* all-zero = defaults                               */
} mksnap_config;

/* One contiguous piece of an arena.  Offsets are relative to the arena that is
 * being submitted and must be multiples of 16. */
#define MKSNAP_X_CRC 1u /* part of the CRC-32 context stream */
#define MKSNAP_X_CDC 2u /* chunk + digest this extent as one file */
/* A file larger than one arena (tario.WriteEntry copies any size, lib/tario/write.go:45): its pieces travel in
 * consecutive submits.  Every piece but the last carries MKSNAP_X_MORE, must be the LAST CDC extent of its submit and
 * states in `reserved` how many bytes of the file follow in later submits (saturate at 0xFFFFFFFF); every piece but
 * the first carries MKSNAP_X_CONT, must be the FIRST CDC extent of the next submit and start at arena offset >=
 * mksnap_limits.carry_bytes (the engine copies the chunk left open at the end of the previous piece in front of it).
 * Chunks and digests are exactly those of the undivided file.  CRC extents need none of this: they split anywhere. */
#define MKSNAP_X_MORE 4u
#define MKSNAP_X_CONT 8u
typedef struct {
    uint64_t arena_off;
    uint64_t len;
    /* MKSNAP_X_CRC: number of context-stream bytes that FOLLOW this extent's last
     * byte (over the whole session, across submits).  The stream is the byte
     * sequence the reference feeds to crc32 in lib/builder/step/add_copy_step.go:104-119,
     * 194-238: seed+directive+args, then relpath / link target / file content
     * per walked path, no separators. */
    uint64_t crc_suffix;
    uint32_t flags;
    uint32_t reserved; /* MKSNAP_X_MORE: bytes of this file in later submits (saturated); otherwise 0 */
} mksnap_extent;

/* A piece of a serial SHA-256 stream (replaces the tarDigester sha256.New() sink of
 * lib/builder/step/common.go:44-55: every tar.Writer write lands in one stream).  arena_off multiple of 16.
 * `stream` is a caller-chosen slot in [0, max_extents): the digest of the stream lands in row `stream` of the
 * stream-digest table.  A stream may span several submits (a layer tar larger than one arena): every piece but
 * the last carries MKSNAP_R_MORE and a length that is a multiple of 64; the device keeps the SHA-256 midstate
 * between submits.  At most one piece per stream per submit. */
#define MKSNAP_R_MORE 1u
typedef struct {
    uint64_t arena_off;
    uint64_t len;
    uint32_t stream;
    uint32_t flags;
} mksnap_range;

typedef struct {
    uint32_t crc_pure;      /* GF(2)-linear accumulator; use mksnap_ctx_crc32() */
    uint32_t reserved;
    uint64_t crc_bytes;     /* context-stream bytes seen */
    uint64_t cdc_bytes;     /* bytes chunked             */
    uint64_t n_files;       /* MKSNAP_X_CDC extents      */
    uint64_t n_chunks;
    uint64_t n_unique;      /* rows of the sorted-unique table */
    uint8_t root[32];       /* fan-out-256 Merkle root of the table = layer content address */
    uint64_t n_streams;     /* rows of the stream-digest table (highest finished stream slot + 1) */
} mksnap_result;

typedef struct {
    /* device time of the most recent submit, CUDA events on the compute stream */
    float ms_total;
    float ms_crc;     /* K0  crc32 extents          */
    float ms_scan;    /* K1  rolling-hash candidate scan */
    float ms_select;  /* K1b cut selection          */
    float ms_sha;     /* K2  per-chunk SHA-256      */
    float ms_stream;  /* K4  serial-stream SHA-256  */
    float ms_h2d;     /* host->device copy (copy stream) */
    /* device time of the most recent finish */
    float ms_sort;    /* K3  radix sort + unique    */
    float ms_root;    /* Merkle root                */
    float ms_gather;  /* NCCL all-gather + merge    */
    uint64_t kernel_launches; /* kernels launched by this handle since create */
    uint64_t h2d_bytes;       /* since create */
    uint64_t d2h_bytes;       /* since create */
} mksnap_stats_t;

/* ---- lifetime --------------------------------------------------------- */
int mksnap_abi_version(void);
int mksnap_create(const mksnap_config *cfg, mksnap_t **out);
void mksnap_destroy(mksnap_t *h);
const char *mksnap_last_error(const mksnap_t *h); /* h may be NULL: create() errors */

/* ---- session ---------------------------------------------------------- */
/* Start digesting a new context/layer: clears the CRC accumulator and the
 * chunk table.  Replaces crc32.NewIEEE() (add_copy_step.go:104) +
 * sha256.New() (common.go:44-45). */
int mksnap_begin(mksnap_t *h);

/* Borrow a C-owned pinned host arena (cudaHostAlloc).  Blocks until one is
 * free.  The caller writes file bytes into it (the Go side through
 * unsafe.Slice; no Go-heap pointer crosses the boundary) and hands it back
 * with mksnap_arena_submit. */
int mksnap_arena_acquire(mksnap_t *h, void **host_ptr, uint64_t *capacity, int32_t *arena_id);

/* Give an acquired arena back without submitting it (error unwinding in a packer: a file vanished, a damaged
 * archive).  mksnap_begin() also reclaims every arena that was acquired and never submitted. */
int mksnap_arena_release(mksnap_t *h, int32_t arena_id);

/* Capacities of this handle, so that a packer can flush an arena BEFORE a table limit is hit (a context of 500k tiny
 * files fills max_extents long before it fills a 1 GiB arena; the reference handles any file count,
 * add_copy_step.go:153-169). */
typedef struct {
    uint64_t max_extents;        /* extents, and ranges, per submit */
    uint64_t max_streams;        /* serial-stream slots per session */
    uint64_t max_chunks;         /* chunk-table rows per session */
    uint64_t host_arena_bytes;
    uint64_t device_arena_bytes;
    uint32_t n_host_arenas;
    uint32_t n_device_slots;
    uint64_t carry_bytes;        /* earliest arena offset of a MKSNAP_X_CONT extent (max chunk size, 512-aligned) */
} mksnap_limits;
int mksnap_get_limits(const mksnap_t *h, mksnap_limits *out);

/* Async: copy arena[0,used) host->device, then run CRC over MKSNAP_X_CRC
 * extents, CDC + per-chunk SHA-256 over MKSNAP_X_CDC extents and one serial
 * SHA-256 per range.  Returns once everything is enqueued; the arena becomes
 * acquirable again when its copy has completed.  Replaces the io.Copy(checksum, fh)
 * loop of add_copy_step.go:230-237 and the tario.WriteEntry -> ConcurrentMultiWriter
 * fan-out of lib/tario/write.go:28-52 / lib/stream/multi_writer.go:35-66. */
int mksnap_arena_submit(mksnap_t *h, int32_t arena_id, uint64_t used,
                        const mksnap_extent *extents, uint64_t n_extents,
                        const mksnap_range *ranges, uint64_t n_ranges);

/* Device-resident variant: the bytes are already in device slot `slot`
 * (written by mksnap_synth_fill, a previous upload, or a GPUDirect producer). */
int mksnap_device_arena(mksnap_t *h, uint32_t slot, void **device_ptr, uint64_t *capacity);
int mksnap_device_upload(mksnap_t *h, uint32_t slot, uint64_t dst_off, const void *src, uint64_t n);
int mksnap_device_submit(mksnap_t *h, uint32_t slot, uint64_t used,
                         const mksnap_extent *extents, uint64_t n_extents,
                         const mksnap_range *ranges, uint64_t n_ranges);

/* Finish the session: sort + unique the chunk digests, Merkle root, wait for
 * the device, fill *out.  On a handle that is one rank of SEVERAL (mksnap_comm_init with n_ranks > 1) out->root is
 * left zeroed: the content address is the root of the global table, which mksnap_exchange_tables /
 * mksnap_allgather_tables return. */
int mksnap_finish(mksnap_t *h, mksnap_result *out);

/* cacheID arithmetic: the value checksum.Sum32() returns at
 * add_copy_step.go:119 for a context stream of stream_len bytes whose pure
 * accumulator is res->crc_pure. */
uint32_t mksnap_ctx_crc32(const mksnap_result *res);

/* ---- incremental cacheID: CRC-32 is linear, so a file's contribution can be reused without its bytes ----
 * With pure(M) = M(x) * x^32 mod P (what the engine accumulates), the context stream's value is the XOR over its
 * segments of pure(segment) * x^(8 * bytes after the segment).  mksnap_get_extent_crcs returns pure(extent) for every
 * MKSNAP_X_CRC extent of the finished session, in submission order; a caller that remembers pure(file content) per
 * file (keyed like MemFS keys a file: size + mtime, lib/tario/compare.go:104-120) folds an UNCHANGED file into a later
 * session with mksnap_crc_add -- no read, no H2D copy, no kernel -- and only changed files travel.  The cacheID is
 * bit-identical to the full computation (add_copy_step.go:102-122) as long as the remembered values are current.
 * mksnap_crc_concat joins the values of two adjacent pieces: pure(A||B) from pure(A), pure(B), len(B). */
int mksnap_crc_add(mksnap_t *h, uint32_t pure, uint64_t len, uint64_t crc_suffix); /* between begin and finish */
uint32_t mksnap_crc_concat(uint32_t pure_a, uint32_t pure_b, uint64_t len_b);
int mksnap_get_extent_crcs(mksnap_t *h, uint32_t *pure, uint64_t capacity, uint64_t *n_out);

/* ---- result tables (valid after mksnap_finish, until the next begin) ---- */
/* chunk END offsets (exclusive; position in the concatenation of all submitted
 * arenas) and digests, in (submit, extent, position) order. */
int mksnap_get_chunks(mksnap_t *h, uint64_t *ends, uint8_t *digests, uint64_t capacity);
/* sorted-unique 32-byte digest table */
int mksnap_get_table(mksnap_t *h, uint8_t *table, uint64_t capacity_rows);
/* rows the handle's table currently holds: result.n_unique after finish / allgather, this rank's range after exchange */
uint64_t mksnap_table_rows(mksnap_t *h);
/* stream digests, row = stream slot: the TarDigest bytes of
 * lib/builder/step/common.go:86 (hex-encode and prefix "sha256:" on the host). */
int mksnap_get_stream_digests(mksnap_t *h, uint8_t *digests, uint64_t capacity);

/* ---- chunk index and chunk delta (DESIGN.md section 3b) ----
 * A chunk index is a sorted-unique set of 32-byte chunk digests that lives in HBM and outlives sessions (the layers a
 * registry or cache already holds).  Rows are ordered bytewise over all 32 bytes -- the order of mksnap_get_table --
 * and mksnap_index_get returns that order, so an index persists as get -> store anywhere -> add_rows.
 * An index works with any handle on the device it was created on (another device: MKSNAP_E_INVAL).  add_rows and
 * add_table return MKSNAP_E_CAPACITY only when the UNION would exceed capacity_rows; on any error the index is
 * unchanged.  add_rows checks strict ascent on the device (violation: MKSNAP_E_INVAL).
 * mksnap_delta, add_table and get_chunk_status need a finished session whose table is still its own: before finish,
 * after the next begin, on one rank of several, or after an exchange / all-gather they return MKSNAP_E_STATE.
 * Per layer: finish -> delta(ix) -> add_table(ix).  The delta classifies against the index as it is at call time;
 * statuses stay valid until the next begin. */
typedef struct mksnap_index mksnap_index_t;
int mksnap_index_create(mksnap_t *h, uint64_t capacity_rows, mksnap_index_t **out); /* on h's device; capacity < 2^32 */
void mksnap_index_destroy(mksnap_index_t *ix);                                        /* before the handle it was created on */
uint64_t mksnap_index_rows(const mksnap_index_t *ix);
int mksnap_index_add_rows(mksnap_t *h, mksnap_index_t *ix, const uint8_t *rows, uint64_t n); /* host rows, strictly ascending */
int mksnap_index_add_table(mksnap_t *h, mksnap_index_t *ix);      /* union with h's finished session table */
int mksnap_index_get(mksnap_t *h, mksnap_index_t *ix, uint8_t *rows, uint64_t capacity_rows);

#define MKSNAP_CHUNK_KNOWN 0u  /* digest is in the index */
#define MKSNAP_CHUNK_NEW 1u    /* not in the index; lowest chunk position carrying this digest in the session */
#define MKSNAP_CHUNK_REPEAT 2u /* not in the index; an earlier chunk of the session has the same digest */
typedef struct {
    uint64_t index_rows;
    uint64_t known_chunks, new_chunks, repeat_chunks;
    uint64_t known_bytes, new_bytes, repeat_bytes; /* sum to mksnap_result.cdc_bytes */
    float ms_device;                               /* CUDA events around the delta's kernels */
    uint32_t reserved;
} mksnap_delta_result;
int mksnap_delta(mksnap_t *h, const mksnap_index_t *ix, mksnap_delta_result *out); /* after mksnap_finish */
int mksnap_get_chunk_status(mksnap_t *h, uint8_t *status, uint64_t capacity);      /* one byte per chunk, mksnap_get_chunks order */

/* ---- multi-GPU: one process per GPU, files sharded, one exchange step ---- */
/* NCCL is dlopen()ed (libnccl.so.2); rank 0 creates the id, the host side
 * distributes it (any out-of-band channel), every rank calls comm_init. */
int mksnap_comm_unique_id(uint8_t id[128]);
int mksnap_comm_init(mksnap_t *h, const uint8_t id[128], int32_t n_ranks, int32_t rank);
/* After mksnap_finish on every rank: all-gather the per-rank sorted-unique
 * tables (ncclAllGather of counts, then of padded rows), merge + unique on the
 * device, XOR-combine the CRC partials.  *out is identical on every rank and
 * equal to what a single GPU would produce for the whole context. */
int mksnap_allgather_tables(mksnap_t *h, mksnap_result *out);
/* The scalable form of the same step: the global table stays RANGE-PARTITIONED.  Rank r ends up owning the digests
 * whose big-endian 64-bit prefix p has floor(p * n_ranks / 2^64) == r: slices of the per-rank tables travel once
 * (ncclSend/ncclRecv all-to-all over NVLink), every rank sorts only its range, Merkle level 0 is computed where the
 * rows are (a group of 256 consecutive global rows by the rank owning its first row, the missing rows of a group
 * that straddles a range end come from an all-gather of every rank's first 255 rows), level-1 digests are
 * all-gathered and the upper levels run everywhere.  *out (root, CRC, counters, n_unique = GLOBAL unique rows) is
 * identical on every rank and equal to the single-GPU result; afterwards mksnap_get_table returns THIS rank's range
 * (ascending; the ranges of ranks 0..n-1 concatenated are the global table).  Work per rank stays ~constant as
 * n_ranks grows, where mksnap_allgather_tables sorts n_ranks times more rows on every rank. */
int mksnap_exchange_tables(mksnap_t *h, mksnap_result *out);
/* The same exchange between n handles of ONE process on ONE device (device copies instead of NCCL; no comm_init):
 * handle i plays rank i, outs[i] receives its result.  Used to run the exchange logic for any n on a single GPU. */
int mksnap_exchange_tables_local(mksnap_t **handles, int32_t n, mksnap_result *outs);
/* Host arithmetic of the exchange, no device needed: given the rows every rank holds after the all-to-all, which
 * groups of 256 global rows does `rank` hash?  out = {U total rows, g0 first global row of the rank, lead rows that
 * belong to a predecessor's group, full groups, own rows in the tail group, rows borrowed from successors, groups}. */
int mksnap_exchange_plan(const uint64_t *rows_per_rank, int32_t n_ranks, int32_t rank, uint64_t out[7]);

/* ---- utilities --------------------------------------------------------- */
/* Deterministic synthetic content, generated on the device into slot bytes
 * [byte_off, byte_off+n) (multiples of 16): little-endian u64 word i (absolute
 * word index in the slot) = mix64(seed + (i+1)*0x9E3779B97F4A7C15). */
int mksnap_synth_fill(mksnap_t *h, uint32_t slot, uint64_t byte_off, uint64_t n, uint64_t seed);
int mksnap_memset(mksnap_t *h, uint32_t slot, uint64_t byte_off, uint64_t n, int value);
int mksnap_device_download(mksnap_t *h, uint32_t slot, uint64_t src_off, void *dst, uint64_t n);
int mksnap_sync(mksnap_t *h);
int mksnap_stats(mksnap_t *h, mksnap_stats_t *out);
void mksnap_default_cdc(mksnap_cdc_params *p);
/* the multiplier M of the frozen rolling hash h_i = h_{i-1}*M + (LE word ending at byte i) (for cross-checking against
 * the oracle) */
uint32_t mksnap_roll_multiplier(void);

#ifdef __cplusplus
}
#endif
#endif
