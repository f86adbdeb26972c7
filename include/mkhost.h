/*
 * mkhost.h — host side ABOVE the mksnap C-ABI, in C++ (libmkhost.so), C interface.
 *
 * The reference's host code on this path is Go; no Go toolchain exists in the build image, so the
 * packer / walker / tar-header logic a cgo build would keep in Go is implemented here in C++ with the
 * reference's names, argument meaning and error behaviour, and is what the tests drive.  It contains NO
 * hashing: every digest comes from libmksnap (the GPU); without a device these calls fail.
 *
 *   mkhost_context_crc32      = addCopyStep.SetCacheID + calculateContextChecksum + checksumPathContents
 *                               reference lib/builder/step/add_copy_step.go:102-122,153-184,194-238
 *   mkhost_commit_copy_ops    = MemFS.AddLayerByCopyOps + commitLayer + tario.WriteEntry, digested on the GPU
 *                               reference lib/snapshot/mem_fs.go:276-289,353-433,509-569, mem_layer.go:152-244,
 *                               lib/tario/write.go:28-68, lib/builder/step/common.go:35-111
 *   mkhost_memfs_update_from_tar = MemFS.UpdateFromTarReader (untar=false) + go1.14 archive/tar Reader, with blob
 *                               verification (DiffID) and the chunk table on the GPU
 *                               reference lib/snapshot/mem_fs.go:165-255
 *   mkhost_encode_tar_header  = tario.WriteHeader + go1.14 archive/tar Writer.WriteHeader (USTAR / PAX)
 *   mkhost_describe_*         = the same host logic without a GPU (entry order / stream order as text), so the
 *                               CPU test-suite can diff it against the oracle.
 */
#ifndef MKHOST_H
#define MKHOST_H

#include <stddef.h>
#include <stdint.h>

#include "mksnap.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct {
    const char *name;     /* as stored in tar.Header.Name (WriteHeader strips leading '/') */
    const char *linkname;
    int64_t mode;         /* perm | 04000 | 02000 | 01000, no type bits (FileInfoHeader) */
    int64_t uid, gid;
    int64_t size;
    int64_t mtime_ns;     /* truncated to the second by tario.WriteHeader (write.go:61) */
    char typeflag;        /* '0' reg, '1' link, '2' symlink, '5' dir, ... */
} mkhost_tar_header;

/* Returns the number of bytes written (512 for USTAR, 1536+ for PAX), 0 on error (cap too small /
 * field not encodable). */
size_t mkhost_encode_tar_header(const mkhost_tar_header *h, uint8_t *out, size_t cap);

/* snapshot.CopyOperation (lib/snapshot/copy_op.go:29-80).  srcs are relative to src_root (leading '/'
 * allowed, as TrimRoot produces them); dst is absolute or relative to work_dir. */
typedef struct {
    const char *src_root;
    const char *const *srcs;
    size_t n_srcs;
    const char *work_dir;
    const char *dst;
    int32_t uid, gid;
} mkhost_copy_op;

typedef struct {
    uint8_t tar_digest[32]; /* DigestPair.TarDigest bytes */
    uint8_t root[32];       /* chunk-table content address */
    uint64_t n_entries;     /* tar entries */
    uint64_t tar_bytes;     /* length of the uncompressed tar stream */
    uint64_t n_chunks, n_unique;
} mkhost_layer_result;

/* cacheID arithmetic of a COPY/ADD step from the build context.  prefix = seed+directive+args.
 * from_paths are the directive's sources (globbed and joined like resolveFromPaths).  *crc_out is what
 * checksum.Sum32() returns; format it with "%x" for the cacheID.  n_threads: file readers (0 = default). */
int mkhost_context_crc32(mksnap_t *eng, const void *prefix, size_t prefix_len, const char *context_dir,
                         const char *const *from_paths, size_t n_paths, int n_threads, uint32_t *crc_out,
                         uint64_t *stream_len_out, char *err, size_t errlen);

/* Incremental cacheID.  CRC-32 is linear: the context value is the XOR over its segments of pure(segment) shifted to
 * the segment's place, so pure(file content) -- 32 bits -- remembered from an earlier build lets an UNCHANGED file be
 * folded in on the host (mksnap_crc_add): no read, no copy to the device, no kernel.  "Unchanged" = same device, inode,
 * size, mtime and ctime (nanoseconds) as when the value was remembered -- stricter than the reference's own notion of an
 * unchanged file (tario.IsSimilarHeader: mtime to the second + size, lib/tario/compare.go:104-120).  Path strings,
 * link targets and the prefix are always streamed (tiny).  The result is bit-identical to mkhost_context_crc32 /
 * addCopyStep.SetCacheID whenever the remembered values are current; a cold cache degrades to the full computation and
 * fills itself.  The cache object belongs to the caller (one per build context); save/load keep it between processes. */
typedef struct mkhost_crc_cache mkhost_crc_cache;
typedef struct {
    uint64_t files_total, files_reused; /* regular files in the stream / folded from the cache */
    uint64_t bytes_total, bytes_sent;   /* file bytes in the stream / file bytes that travelled to the device */
} mkhost_crc_cache_stats;
mkhost_crc_cache *mkhost_crc_cache_new(void);
void mkhost_crc_cache_free(mkhost_crc_cache *c);
uint64_t mkhost_crc_cache_size(const mkhost_crc_cache *c);
int mkhost_crc_cache_save(const mkhost_crc_cache *c, const char *path, char *err, size_t errlen);
int mkhost_crc_cache_load(mkhost_crc_cache *c, const char *path, char *err, size_t errlen);
int mkhost_context_crc32_cached(mksnap_t *eng, mkhost_crc_cache *cache, const void *prefix, size_t prefix_len,
                                const char *context_dir, const char *const *from_paths, size_t n_paths, int n_threads,
                                uint32_t *crc_out, uint64_t *stream_len_out, mkhost_crc_cache_stats *stats, char *err,
                                size_t errlen);

/* Commit one layer from copy operations against an EMPTY MemFS rooted at root_dir (FROM scratch): packs
 * the sorted entries as a tar stream into one arena, digests it (TarDigest) and chunks every regular
 * file (chunk table).  now_unix = clk.Now() for synthesized ancestors (mem_fs.go:562). */
int mkhost_commit_copy_ops(mksnap_t *eng, const char *root_dir, int64_t now_unix, const mkhost_copy_op *ops,
                           size_t n_ops, int n_threads, mkhost_layer_result *out, char *err, size_t errlen);
/* Same, and additionally writes the uncompressed layer tar (the packed arenas, byte for byte what
 * tar.Writer would have produced) to tar_fd -- the stream the Go side feeds to pgzip (common.go:47-55,
 * SURVEY section 8f-1).  SHA-256 of those bytes == out->tar_digest. */
int mkhost_commit_copy_ops_to_fd(mksnap_t *eng, const char *root_dir, int64_t now_unix, const mkhost_copy_op *ops,
                                 size_t n_ops, int n_threads, int tar_fd, mkhost_layer_result *out, char *err,
                                 size_t errlen);
/* flags for mkhost_commit_copy_ops_ex */
#define MKHOST_NO_TAR_DIGEST 1u /* leave TarDigest to the caller (Go's sha256.New() fed from the same bytes, see
                                   INTEGRATION.md section 3): out->tar_digest is zeroed, no serial stream is submitted */
/* MemFS entry points only (they need a tree to remember into):
 * MKHOST_FILE_DIGESTS  also hash every regular file of the layer (one serial SHA-256 stream per file, stream slots
 *                      1..n; the engine needs max_extents > n) and remember the digest in the tree.
 * MKHOST_SCAN_CONTENT  mkhost_memfs_commit_scan: content-aware change detection (SURVEY section 8f-3).  Files the
 *                      reference's IsSimilarHeader calls unchanged (same mtime second, size, mode, owner) are
 *                      re-hashed on the GPU and compared with the remembered digest; a difference puts the file into
 *                      the layer.  Removes the need for the sync() + 1 s sleep of mem_fs.go:291-311.  Implies
 *                      MKHOST_FILE_DIGESTS.  No reference counterpart: with the flag clear the scan is the reference's. */
#define MKHOST_FILE_DIGESTS 2u
#define MKHOST_SCAN_CONTENT 4u
int mkhost_commit_copy_ops_ex(mksnap_t *eng, const char *root_dir, int64_t now_unix, const mkhost_copy_op *ops,
                              size_t n_ops, int n_threads, int tar_fd, uint32_t flags, mkhost_layer_result *out,
                              char *err, size_t errlen);

/* Persistent mirror of snapshot.MemFS (lib/snapshot/mem_fs.go:60-83): layers accumulate in the merged tree, later
 * layers contain only entries whose header is not "similar" (lib/tario/compare.go) to what the tree holds, scans
 * emit whiteouts for children that vanished (mem_fs.go:459-480), `blacklist` as in NewMemFS(clk, root, blacklist). */
typedef struct mkhost_memfs mkhost_memfs;
mkhost_memfs *mkhost_memfs_new(const char *root_dir, const char *const *blacklist, size_t n_blacklist, char *err,
                               size_t errlen);
void mkhost_memfs_free(mkhost_memfs *m);
/* SHA-256 of the content the tree remembers for the regular file at dst (MKHOST_FILE_DIGESTS / MKHOST_SCAN_CONTENT
 * commits and ingests); returns 0 and fills out, or 1 when nothing is remembered for that path. */
int mkhost_memfs_file_digest(mkhost_memfs *m, const char *dst, uint8_t out[32]);
/* AddLayerByCopyOps / AddLayerByScan followed by commitLayer on the GPU (flags: MKHOST_NO_TAR_DIGEST). */
int mkhost_memfs_commit_copy_ops(mkhost_memfs *m, mksnap_t *eng, int64_t now_unix, const mkhost_copy_op *ops, size_t n_ops,
                                 int n_threads, int tar_fd, uint32_t flags, mkhost_layer_result *out, char *err,
                                 size_t errlen);
int mkhost_memfs_commit_scan(mkhost_memfs *m, mksnap_t *eng, int64_t now_unix, int n_threads, int tar_fd, uint32_t flags,
                             mkhost_layer_result *out, char *err, size_t errlen);
/* Several consecutive layers of ONE build committed in one engine session.  Equivalent to calling
 * mkhost_memfs_commit_copy_ops once per layer, in order (same entries, same tar bytes to each layer's tar_fd, same
 * TarDigest per layer) -- but every pinned arena carries a piece of EVERY unfinished layer, so the serial SHA-256
 * chains (one per layer, lib/builder/step/common.go:44-55) advance together on the device instead of one after the
 * other.  This is what makes TarDigest on the GPU worthwhile: one chain runs at ~0.09 GB/s, 256 chains at ~23 GB/s.
 * The reference commits layer by layer (build_node.go:102-107); COPY/ADD steps that do not modify the file system
 * (no RUN in between) can be deferred and committed together, which is what a cgo caller would do (INTEGRATION.md).
 * outs[i].tar_digest / tar_bytes / n_entries are per layer; root / n_chunks / n_unique describe the chunk table of the
 * whole batch (one session) -- unless MKHOST_LAYER_TABLES is set: then the session is grouped (layer i = group i,
 * mksnap_begin_groups) and they are layer i's own, equal to what a separate mkhost_memfs_commit_copy_ops of that layer
 * returns; the engine's session stays open for mksnap_delta_groups / mksnap_get_group_table / mksnap_index_add_group.
 * flags: MKHOST_NO_TAR_DIGEST, MKHOST_LAYER_TABLES.  tar_fd < 0: that layer's tar is not emitted. */
#define MKHOST_LAYER_TABLES 64u
typedef struct {
    const mkhost_copy_op *ops;
    size_t n_ops;
    int tar_fd;
} mkhost_layer_spec;
int mkhost_memfs_commit_layers(mkhost_memfs *m, mksnap_t *eng, int64_t now_unix, const mkhost_layer_spec *layers,
                               size_t n_layers, int n_threads, uint32_t flags, mkhost_layer_result *outs, char *err,
                               size_t errlen);
/* the same two without a GPU: entry list as text (format below); they DO merge the layer into the tree */
size_t mkhost_memfs_describe_copy_ops(mkhost_memfs *m, int64_t now_unix, const mkhost_copy_op *ops, size_t n_ops, char *out,
                                      size_t cap, char *err, size_t errlen);
size_t mkhost_memfs_describe_scan(mkhost_memfs *m, int64_t now_unix, char *out, size_t cap, char *err, size_t errlen);

/* UpdateFromTarReader(r, untar=false) (lib/snapshot/mem_fs.go:165-255; FROM / cache-hit path, from_step.go:118-134):
 * merge an UNCOMPRESSED layer tar read from tar_fd (file or pipe; gunzip stays in Go, lib/tario/gzip.go) into the tree,
 * hard links in a second pass, nothing written to disk.  The stream goes through the pinned arenas once:
 * out->tar_digest = SHA-256 of every byte read up to EOF (the layer's DiffID: compare with the image config to
 * verify the pulled blob, lib/docker/image/digest.go:42-50), out->root / n_chunks / n_unique = chunk table of the
 * regular-file members (so base layers join the chunk-granular dedup), out->n_entries = headers merged (the
 * count the reference logs).  flags: MKHOST_NO_TAR_DIGEST, MKHOST_FILE_DIGESTS, MKHOST_UNTAR.  A regular-file member
 * larger than one arena travels in pieces (MKSNAP_X_MORE / MKSNAP_X_CONT); only MKHOST_UNTAR, which writes a member
 * from one contiguous body, still needs every member to fit an arena. */
int mkhost_memfs_update_from_tar(mkhost_memfs *m, mksnap_t *eng, int64_t now_unix, int tar_fd, uint32_t flags,
                                 mkhost_layer_result *out, char *err, size_t errlen);
/* the same merge without a GPU: merged layer as text (format below) */
size_t mkhost_memfs_describe_update_from_tar(mkhost_memfs *m, int64_t now_unix, int tar_fd, char *out, size_t cap,
                                             char *err, size_t errlen);
/* MKHOST_UNTAR (flag of mkhost_memfs_update_from_tar and of the _ex describe): UpdateFromTarReader(r, untar=true) --
 * every member is also written under the root (untarOneItem, lib/snapshot/mem_fs.go:574-716: whiteouts delete,
 * existing directories are updated in place, similar entries are left alone, anything else is replaced; hard links
 * last; tario.ApplyHeader sets owner, mode and mtime; parent directory mtimes are restored).  On the GPU path the file
 * bodies are written straight from the arena that is being digested. */
#define MKHOST_UNTAR 32u
size_t mkhost_memfs_describe_update_from_tar_ex(mkhost_memfs *m, int64_t now_unix, int tar_fd, uint32_t flags, char *out,
                                                size_t cap, char *err, size_t errlen);

/* CopyOperation.Execute (lib/snapshot/copy_op.go:82-147) with fileio.Copier (lib/fileio/copy.go): what a COPY/ADD step
 * does to the file system when it runs with --modifyfs.  op->dst is used as the on-disk destination exactly like the
 * reference does (resolved against op->work_dir when relative).  mode selects the Copier of copy_op.go:98-124:
 * MKHOST_COPY_CHOWN (--chown: op->uid/gid), MKHOST_COPY_INTERNAL (--from=<stage>: no blacklist, owners preserved),
 * MKHOST_COPY_PRESERVE_OWNER (--from --archive).  mode 0 = copy from the build context (owner root).
 * MKHOST_COPY_DEFERRED runs the traversal (directories, symlinks, chmod of existing targets) first and writes the
 * regular files afterwards from buffers read once -- the path mkhost_memfs_commit_copy_ops(…, MKHOST_MATERIALIZE)
 * takes with its arena; here the buffers are plain reads, so the deferred machinery can be exercised without a GPU. */
#define MKHOST_COPY_CHOWN 1u
#define MKHOST_COPY_INTERNAL 2u
#define MKHOST_COPY_PRESERVE_OWNER 4u
#define MKHOST_COPY_DEFERRED 8u
int mkhost_copy_op_execute(const mkhost_copy_op *op, uint32_t mode, const char *const *blacklist, size_t n_blacklist,
                           char *err, size_t errlen);
/* evalSymlinks(p, srcRoot) (lib/snapshot/utils.go:249-324): the root-relative path after following every symlink on
 * it, links confined to src_root (absolute targets must carry the root prefix, which is trimmed), at most 255 links.
 * Both CopyOperation.Execute (copy_op.go:86) and MemFS.addToLayer (mem_fs.go:380) resolve each source through it.
 * Returns the number of bytes needed including NUL (nothing written if > cap), 0 on error. */
size_t mkhost_eval_symlinks(const char *path, const char *src_root, char *out, size_t cap, char *err, size_t errlen);
/* flag for mkhost_memfs_commit_copy_ops: also perform the copy (as mkhost_copy_op_execute with `copy_mode` 0 / CHOWN
 * decided by MKHOST_MATERIALIZE_CHOWN), writing regular files from the arena the layer is packed in: the context is
 * read once for the copy, the layer, its digest and its chunk table (SURVEY section 8f-4). */
#define MKHOST_MATERIALIZE 8u
#define MKHOST_MATERIALIZE_CHOWN 16u

/* cache.Manager wire format (lib/cache/cache_manager.go:34-35,239-252).  key = "makisu_builder_cache_" + cacheID;
 * entry = "<tarHex>,<gzipHex>" (createEntry), or "MAKISU_CACHE_EMPTY" for a nil pair (tar_hex == NULL).
 * parse = parseEntry: error when there is no ',', otherwise SplitN(entry, ",", 2) -- no hex validation, like
 * the reference.  Because old readers keep everything after the first ',' as the gzip digest, the chunk-table
 * root cannot ride in the same value: it is stored under its own key "<key>_chunks" = "<rootHex>,<n_unique>",
 * which readers that do not know it never fetch (SURVEY section 8f-1: "old readers must still parse").
 * All return the number of bytes needed including NUL (nothing written if > cap), 0 on error. */
size_t mkhost_cache_key(const char *cache_id, int chunk_table, char *out, size_t cap);
size_t mkhost_cache_entry_create(const char *tar_hex, const char *gzip_hex, char *out, size_t cap);
int mkhost_cache_entry_parse(const char *entry, char *tar_digest, size_t tar_cap, char *gzip_digest, size_t gzip_cap,
                             char *err, size_t errlen);
size_t mkhost_cache_chunk_entry_create(const uint8_t root[32], uint64_t n_unique, char *out, size_t cap);
int mkhost_cache_chunk_entry_parse(const char *entry, uint8_t root[32], uint64_t *n_unique, char *err, size_t errlen);

/* No-GPU introspection for the CPU tests: one line per item, '\n' separated, NUL terminated.
 *   stream : "P <relpath>" | "L <target>" | "F <size> <abs path>"   in CRC stream order
 *   layer  : "<typeflag> <mode octal> <uid> <gid> <size> <mtime> <dst> <hdr.Name> <src>"  in tar order
 * Return the number of bytes needed (including NUL); if > cap nothing is written. */
size_t mkhost_describe_context_stream(const char *context_dir, const char *const *from_paths, size_t n_paths,
                                      char *out, size_t cap, char *err, size_t errlen);
size_t mkhost_describe_layer(const char *root_dir, int64_t now_unix, const mkhost_copy_op *ops, size_t n_ops,
                             char *out, size_t cap, char *err, size_t errlen);

#ifdef __cplusplus
}
#endif
#endif
