// +build mksnap

// Package mksnap binds libmksnap.so (include/mksnap.h: the B200 snapshot+hash engine) and libmkhost.so
// (include/mkhost.h: walker, tar headers and arena packers above it) into makisu.
//
// Drop this directory into the reference tree as lib/mksnap, apply integration/patches/*.patch and build with
//   CGO_ENABLED=1 go build -tags mksnap ./bin/makisu
// Without the tag the stock pure-Go files are compiled unchanged.  The engine has no CPU fallback: New fails when no
// sm_100 device is usable, and so does the build that asked for it.
//
// NOTE: the image this repository is built in has no Go toolchain, so these files have been reviewed against
// include/*.h but never compiled; the same C entry points are exercised from Python (makisu_b200/abi.py, host.py).
package mksnap

/*
#cgo LDFLAGS: -lmkhost -lmksnap
#include <stdlib.h>
#include "mksnap.h"
#include "mkhost.h"
*/
import "C"

import (
	"encoding/hex"
	"fmt"
	"os"
	"runtime"
	"unsafe"
)

// Engine owns one GPU: streams, pinned host arenas, device slots.  One session at a time; the reference drives the
// seams from the plan goroutine (lib/builder/build_plan.go:174), which is what the C side expects.
type Engine struct{ h *C.mksnap_t }

// New creates an engine on `device` with nArenas pinned host arenas of arenaBytes each (1 GiB and 3 are good
// defaults: one being filled, one in flight, one on the device).
func New(device int, arenaBytes uint64, nArenas int) (*Engine, error) {
	cfg := C.mksnap_config{
		device:             C.int32_t(device),
		n_host_arenas:      C.uint32_t(nArenas),
		host_arena_bytes:   C.uint64_t(arenaBytes),
		device_arena_bytes: C.uint64_t(arenaBytes),
		max_extents:        1 << 20,
	}
	e := &Engine{}
	if rc := C.mksnap_create(&cfg, &e.h); rc != 0 {
		return nil, fmt.Errorf("mksnap create: %s", C.GoString(C.mksnap_last_error(nil)))
	}
	runtime.SetFinalizer(e, func(e *Engine) { e.Close() })
	return e, nil
}

// Close releases the device.
func (e *Engine) Close() {
	if e.h != nil {
		C.mksnap_destroy(e.h)
		e.h = nil
	}
}

const errLen = 1024

func cStrings(ss []string) (**C.char, func()) {
	arr := C.malloc(C.size_t(len(ss)+1) * C.size_t(unsafe.Sizeof(uintptr(0))))
	view := (*[1 << 28]*C.char)(arr)[: len(ss)+1 : len(ss)+1]
	for i, s := range ss {
		view[i] = C.CString(s)
	}
	view[len(ss)] = nil
	return (**C.char)(arr), func() {
		for i := range ss {
			C.free(unsafe.Pointer(view[i]))
		}
		C.free(arr)
	}
}

// ContextCRC32 replaces the crc32.NewIEEE() / filepath.Walk / io.Copy chain of
// addCopyStep.SetCacheID (lib/builder/step/add_copy_step.go:102-122,153-238): prefix is seed+directive+args,
// fromPaths are the directive's sources exactly as resolveFromPaths receives them.  The result is what
// checksum.Sum32() returns; format it with "%x".
func (e *Engine) ContextCRC32(prefix []byte, contextDir string, fromPaths []string, threads int) (uint32, error) {
	var crc C.uint32_t
	var n C.uint64_t
	errBuf := (*C.char)(C.malloc(errLen))
	defer C.free(unsafe.Pointer(errBuf))
	cdir := C.CString(contextDir)
	defer C.free(unsafe.Pointer(cdir))
	paths, free := cStrings(fromPaths)
	defer free()
	var p unsafe.Pointer
	if len(prefix) > 0 {
		p = C.CBytes(prefix)
		defer C.free(p)
	}
	if rc := C.mkhost_context_crc32(e.h, p, C.size_t(len(prefix)), cdir, paths, C.size_t(len(fromPaths)),
		C.int(threads), &crc, &n, errBuf, errLen); rc != 0 {
		return 0, fmt.Errorf("%s", C.GoString(errBuf)) // already "hash context sources: ..." like add_copy_step.go:116
	}
	return uint32(crc), nil
}

// CopyOp mirrors snapshot.CopyOperation (lib/snapshot/copy_op.go:29-80).
type CopyOp struct {
	SrcRoot, WorkDir, Dst string
	Srcs                  []string
	UID, GID              int
}

// LayerResult carries what commitLayer needs (lib/builder/step/common.go:86-110) plus the chunk-table address.
type LayerResult struct {
	TarDigest        string // "sha256:<hex>" == image.DigestPair.TarDigest
	ChunkRoot        [32]byte
	Entries, TarSize uint64
	Chunks, Unique   uint64
}

func toResult(r *C.mkhost_layer_result) LayerResult {
	out := LayerResult{Entries: uint64(r.n_entries), TarSize: uint64(r.tar_bytes), Chunks: uint64(r.n_chunks), Unique: uint64(r.n_unique)}
	out.TarDigest = "sha256:" + hex.EncodeToString(C.GoBytes(unsafe.Pointer(&r.tar_digest[0]), 32))
	copy(out.ChunkRoot[:], C.GoBytes(unsafe.Pointer(&r.root[0]), 32))
	return out
}

// MemFS is the C++ mirror of snapshot.MemFS (lib/snapshot/mem_fs.go:60-83): the merged tree lives on the C side, so
// the entry order, the headers and the tar bytes are produced next to the arenas they are packed into.
type MemFS struct{ m *C.mkhost_memfs }

// NewMemFS = snapshot.NewMemFS(clk, root, blacklist); the clock is passed per call (now) instead.
func NewMemFS(root string, blacklist []string) (*MemFS, error) {
	errBuf := (*C.char)(C.malloc(errLen))
	defer C.free(unsafe.Pointer(errBuf))
	croot := C.CString(root)
	defer C.free(unsafe.Pointer(croot))
	bl, free := cStrings(blacklist)
	defer free()
	m := C.mkhost_memfs_new(croot, bl, C.size_t(len(blacklist)), errBuf, errLen)
	if m == nil {
		return nil, fmt.Errorf("new memfs: %s", C.GoString(errBuf))
	}
	fs := &MemFS{m: m}
	runtime.SetFinalizer(fs, func(fs *MemFS) { C.mkhost_memfs_free(fs.m) })
	return fs, nil
}

type cOps struct {
	arr   *C.mkhost_copy_op
	n     int
	frees []func()
}

func newCOps(ops []CopyOp) *cOps {
	c := &cOps{n: len(ops)}
	c.arr = (*C.mkhost_copy_op)(C.calloc(C.size_t(len(ops)+1), C.size_t(unsafe.Sizeof(C.mkhost_copy_op{}))))
	view := (*[1 << 20]C.mkhost_copy_op)(unsafe.Pointer(c.arr))[:len(ops):len(ops)]
	for i, o := range ops {
		srcs, free := cStrings(o.Srcs)
		c.frees = append(c.frees, free)
		view[i].src_root, view[i].work_dir, view[i].dst = C.CString(o.SrcRoot), C.CString(o.WorkDir), C.CString(o.Dst)
		view[i].srcs, view[i].n_srcs = srcs, C.size_t(len(o.Srcs))
		view[i].uid, view[i].gid = C.int32_t(o.UID), C.int32_t(o.GID)
	}
	return c
}

func (c *cOps) free() {
	view := (*[1 << 20]C.mkhost_copy_op)(unsafe.Pointer(c.arr))[:c.n:c.n]
	for i := range view {
		C.free(unsafe.Pointer(view[i].src_root))
		C.free(unsafe.Pointer(view[i].work_dir))
		C.free(unsafe.Pointer(view[i].dst))
	}
	for _, f := range c.frees {
		f()
	}
	C.free(unsafe.Pointer(c.arr))
}

// Flags of the commit calls (include/mkhost.h).
const (
	NoTarDigest uint32 = 1 // leave TarDigest to the caller (keep sha256.New() on the host for a single huge layer)
	FileDigests uint32 = 2
	ScanContent uint32 = 4
	Materialize uint32 = 8
)

// CommitCopyOps = MemFS.AddLayerByCopyOps + commitLayer's tar/SHA-256 half (mem_fs.go:276-289, common.go:35-63).
// The uncompressed layer tar is written to tarOut (feed it to pgzip); TarDigest comes back from the GPU.
func (fs *MemFS) CommitCopyOps(e *Engine, now int64, ops []CopyOp, tarOut *os.File, threads int, flags uint32) (LayerResult, error) {
	c := newCOps(ops)
	defer c.free()
	errBuf := (*C.char)(C.malloc(errLen))
	defer C.free(unsafe.Pointer(errBuf))
	fd := C.int(-1)
	if tarOut != nil {
		fd = C.int(tarOut.Fd())
	}
	var r C.mkhost_layer_result
	if rc := C.mkhost_memfs_commit_copy_ops(fs.m, e.h, C.int64_t(now), c.arr, C.size_t(c.n), C.int(threads), fd,
		C.uint32_t(flags), &r, errBuf, errLen); rc != 0 {
		return LayerResult{}, fmt.Errorf("%s", C.GoString(errBuf)) // "failed to generate diff layer: ..." (common.go:82)
	}
	return toResult(&r), nil
}

// CommitScan = MemFS.AddLayerByScan + the same digest half (mem_fs.go:260-270).
func (fs *MemFS) CommitScan(e *Engine, now int64, tarOut *os.File, threads int, flags uint32) (LayerResult, error) {
	errBuf := (*C.char)(C.malloc(errLen))
	defer C.free(unsafe.Pointer(errBuf))
	fd := C.int(-1)
	if tarOut != nil {
		fd = C.int(tarOut.Fd())
	}
	var r C.mkhost_layer_result
	if rc := C.mkhost_memfs_commit_scan(fs.m, e.h, C.int64_t(now), C.int(threads), fd, C.uint32_t(flags), &r, errBuf, errLen); rc != 0 {
		return LayerResult{}, fmt.Errorf("%s", C.GoString(errBuf))
	}
	return toResult(&r), nil
}

// LayerTables (flag of CommitLayers, MKHOST_LAYER_TABLES): give every layer of the batch its own chunk table -- ChunkRoot,
// Chunks and Unique of result i are what CommitCopyOps of layer i alone returns -- and leave the grouped session open
// for Engine.DeltaGroups / GroupTable / Index.AddGroup (layer i = group i).
const LayerTables = 64

// CommitLayers commits consecutive COPY/ADD layers of one build in ONE engine session: every TarDigest chain
// advances together on the device (one chain runs at ~0.09 GB/s, 256 chains at ~23 GB/s).  tarOuts[i] may be nil.
// Without LayerTables in flags, ChunkRoot / Chunks / Unique of every result describe the batch as a whole.
func (fs *MemFS) CommitLayers(e *Engine, now int64, layers [][]CopyOp, tarOuts []*os.File, threads int, flags uint32) ([]LayerResult, error) {
	n := len(layers)
	specs := (*C.mkhost_layer_spec)(C.calloc(C.size_t(n+1), C.size_t(unsafe.Sizeof(C.mkhost_layer_spec{}))))
	defer C.free(unsafe.Pointer(specs))
	sview := (*[1 << 20]C.mkhost_layer_spec)(unsafe.Pointer(specs))[:n:n]
	for i, ops := range layers {
		c := newCOps(ops)
		defer c.free()
		sview[i].ops, sview[i].n_ops, sview[i].tar_fd = c.arr, C.size_t(c.n), -1
		if tarOuts != nil && tarOuts[i] != nil {
			sview[i].tar_fd = C.int(tarOuts[i].Fd())
		}
	}
	outs := (*C.mkhost_layer_result)(C.calloc(C.size_t(n+1), C.size_t(unsafe.Sizeof(C.mkhost_layer_result{}))))
	defer C.free(unsafe.Pointer(outs))
	errBuf := (*C.char)(C.malloc(errLen))
	defer C.free(unsafe.Pointer(errBuf))
	if rc := C.mkhost_memfs_commit_layers(fs.m, e.h, C.int64_t(now), specs, C.size_t(n), C.int(threads), C.uint32_t(flags),
		outs, errBuf, errLen); rc != 0 {
		return nil, fmt.Errorf("%s", C.GoString(errBuf))
	}
	oview := (*[1 << 20]C.mkhost_layer_result)(unsafe.Pointer(outs))[:n:n]
	res := make([]LayerResult, n)
	for i := range res {
		res[i] = toResult(&oview[i])
	}
	return res, nil
}

// UpdateFromTar = MemFS.UpdateFromTarReader (mem_fs.go:165-255) on an UNCOMPRESSED tar stream (gunzip stays Go):
// the blob's DiffID and the chunk table come back; untar also writes the members under the root from the arena.
func (fs *MemFS) UpdateFromTar(e *Engine, now int64, tarIn *os.File, untar bool, flags uint32) (LayerResult, error) {
	if untar {
		flags |= 32 // MKHOST_UNTAR
	}
	errBuf := (*C.char)(C.malloc(errLen))
	defer C.free(unsafe.Pointer(errBuf))
	var r C.mkhost_layer_result
	if rc := C.mkhost_memfs_update_from_tar(fs.m, e.h, C.int64_t(now), C.int(tarIn.Fd()), C.uint32_t(flags), &r, errBuf, errLen); rc != 0 {
		return LayerResult{}, fmt.Errorf("%s", C.GoString(errBuf))
	}
	return toResult(&r), nil
}

// CrcCache remembers pure(file content) per context file between builds (include/mkhost.h, "Incremental cacheID"):
// unchanged files (same device, inode, size, mtime, ctime) are folded into the cacheID on the host, only changed files
// travel to the device.  One cache per build context; Save/Load keep it between makisu invocations.
type CrcCache struct{ c *C.mkhost_crc_cache }

// NewCrcCache loads `path` when it exists ("" = start cold).
func NewCrcCache(path string) (*CrcCache, error) {
	cc := &CrcCache{c: C.mkhost_crc_cache_new()}
	runtime.SetFinalizer(cc, func(cc *CrcCache) { C.mkhost_crc_cache_free(cc.c) })
	if path == "" {
		return cc, nil
	}
	if _, err := os.Stat(path); err != nil {
		return cc, nil
	}
	errBuf := (*C.char)(C.malloc(errLen))
	defer C.free(unsafe.Pointer(errBuf))
	cpath := C.CString(path)
	defer C.free(unsafe.Pointer(cpath))
	if C.mkhost_crc_cache_load(cc.c, cpath, errBuf, errLen) != 0 {
		return nil, fmt.Errorf("%s", C.GoString(errBuf))
	}
	return cc, nil
}

// Save writes the cache next to the build context (or into makisu's storage dir).
func (cc *CrcCache) Save(path string) error {
	errBuf := (*C.char)(C.malloc(errLen))
	defer C.free(unsafe.Pointer(errBuf))
	cpath := C.CString(path)
	defer C.free(unsafe.Pointer(cpath))
	if C.mkhost_crc_cache_save(cc.c, cpath, errBuf, errLen) != 0 {
		return fmt.Errorf("%s", C.GoString(errBuf))
	}
	return nil
}

// ContextCRC32Cached is ContextCRC32 with the cache in the loop; sent = file bytes that travelled to the device.
func (e *Engine) ContextCRC32Cached(cc *CrcCache, prefix []byte, contextDir string, fromPaths []string, threads int) (crc uint32, sent uint64, err error) {
	var c C.uint32_t
	var n C.uint64_t
	var st C.mkhost_crc_cache_stats
	errBuf := (*C.char)(C.malloc(errLen))
	defer C.free(unsafe.Pointer(errBuf))
	cdir := C.CString(contextDir)
	defer C.free(unsafe.Pointer(cdir))
	paths, free := cStrings(fromPaths)
	defer free()
	var p unsafe.Pointer
	if len(prefix) > 0 {
		p = C.CBytes(prefix)
		defer C.free(p)
	}
	if rc := C.mkhost_context_crc32_cached(e.h, cc.c, p, C.size_t(len(prefix)), cdir, paths, C.size_t(len(fromPaths)),
		C.int(threads), &c, &n, &st, errBuf, errLen); rc != 0 {
		return 0, 0, fmt.Errorf("%s", C.GoString(errBuf))
	}
	return uint32(c), uint64(st.bytes_sent), nil
}

// Index is a device-resident sorted-unique set of chunk digests (mksnap_index_*): the chunks of the base image and of
// the layers already pushed or cached.  It lives on the engine's device and outlives sessions; Close it before the
// engine it was created on.
type Index struct {
	ix *C.mksnap_index_t
	e  *Engine
}

// NewIndex creates an empty index of capacityRows rows (< 2^32) on e's device.
func (e *Engine) NewIndex(capacityRows uint64) (*Index, error) {
	x := &Index{e: e}
	if rc := C.mksnap_index_create(e.h, C.uint64_t(capacityRows), &x.ix); rc != 0 {
		return nil, fmt.Errorf("mksnap index create: %s", C.GoString(C.mksnap_last_error(e.h)))
	}
	return x, nil
}

// Close releases the index's device memory.
func (x *Index) Close() {
	if x.ix != nil {
		C.mksnap_index_destroy(x.ix)
		x.ix = nil
	}
}

// Rows is the number of digests the index holds.
func (x *Index) Rows() uint64 { return uint64(C.mksnap_index_rows(x.ix)) }

// AddTable adds the chunk table of e's finished session (base-layer ingest or a committed layer).
func (x *Index) AddTable(e *Engine) error {
	if rc := C.mksnap_index_add_table(e.h, x.ix); rc != 0 {
		return fmt.Errorf("mksnap index add table: %s", C.GoString(C.mksnap_last_error(e.h)))
	}
	return nil
}

// AddRows adds persisted rows: n*32 bytes, strictly ascending (what Rows returned, stored anywhere).
func (x *Index) AddRows(rows []byte) error {
	if len(rows)%32 != 0 {
		return fmt.Errorf("mksnap index add rows: %d bytes is not a multiple of 32", len(rows))
	}
	if len(rows) == 0 {
		return nil
	}
	p := C.CBytes(rows)
	defer C.free(p)
	if rc := C.mksnap_index_add_rows(x.e.h, x.ix, (*C.uint8_t)(p), C.uint64_t(len(rows)/32)); rc != 0 {
		return fmt.Errorf("mksnap index add rows: %s", C.GoString(C.mksnap_last_error(x.e.h)))
	}
	return nil
}

// Get returns the index rows in bytewise order, 32 bytes each: the persisted form of the index.
func (x *Index) Get() ([]byte, error) {
	n := x.Rows()
	if n == 0 {
		return nil, nil
	}
	buf := C.malloc(C.size_t(n * 32))
	defer C.free(buf)
	if rc := C.mksnap_index_get(x.e.h, x.ix, (*C.uint8_t)(buf), C.uint64_t(n)); rc != 0 {
		return nil, fmt.Errorf("mksnap index get: %s", C.GoString(C.mksnap_last_error(x.e.h)))
	}
	return C.GoBytes(buf, C.int(n*32)), nil
}

// Chunk statuses of Delta / ChunkStatus.
const (
	ChunkKnown  = 0 // the digest is in the index
	ChunkNew    = 1 // not in the index; the first chunk of the layer carrying it
	ChunkRepeat = 2 // not in the index; an earlier chunk of the layer has the same digest
)

// DeltaResult counts the chunks and bytes of each status.  NewBytes is what a chunk-granular push would send.
type DeltaResult struct {
	IndexRows                            uint64
	KnownChunks, NewChunks, RepeatChunks uint64
	KnownBytes, NewBytes, RepeatBytes    uint64
	DeviceMs                             float32
}

// Delta classifies every chunk of e's finished session against x.  Call it before x.AddTable(e) for the same layer.
func (e *Engine) Delta(x *Index) (DeltaResult, error) {
	var r C.mksnap_delta_result
	if rc := C.mksnap_delta(e.h, x.ix, &r); rc != 0 {
		return DeltaResult{}, fmt.Errorf("mksnap delta: %s", C.GoString(C.mksnap_last_error(e.h)))
	}
	return DeltaResult{IndexRows: uint64(r.index_rows), KnownChunks: uint64(r.known_chunks), NewChunks: uint64(r.new_chunks),
		RepeatChunks: uint64(r.repeat_chunks), KnownBytes: uint64(r.known_bytes), NewBytes: uint64(r.new_bytes),
		RepeatBytes: uint64(r.repeat_bytes), DeviceMs: float32(r.ms_device)}, nil
}

// ChunkStatus returns one status byte per chunk of the last Delta, in chunk order (valid until the next session).
func (e *Engine) ChunkStatus(nChunks uint64) ([]byte, error) {
	if nChunks == 0 {
		return nil, nil
	}
	buf := C.malloc(C.size_t(nChunks))
	defer C.free(buf)
	if rc := C.mksnap_get_chunk_status(e.h, (*C.uint8_t)(buf), C.uint64_t(nChunks)); rc != 0 {
		return nil, fmt.Errorf("mksnap chunk status: %s", C.GoString(C.mksnap_last_error(e.h)))
	}
	return C.GoBytes(buf, C.int(nChunks)), nil
}

// GroupResult is one group (layer) of a grouped session: its own chunk table, as if it had been committed alone.
type GroupResult struct {
	Files, CdcBytes, Chunks, Unique, FirstRow uint64
	Root                                      [32]byte
}

// GroupResults returns the per-group results of e's finished grouped session (CommitLayers with LayerTables).
func (e *Engine) GroupResults(nGroups int) ([]GroupResult, error) {
	if nGroups <= 0 {
		return nil, fmt.Errorf("mksnap group results: %d groups", nGroups)
	}
	buf := (*C.mksnap_group_result)(C.calloc(C.size_t(nGroups), C.size_t(unsafe.Sizeof(C.mksnap_group_result{}))))
	defer C.free(unsafe.Pointer(buf))
	if rc := C.mksnap_get_group_results(e.h, buf, C.uint32_t(nGroups)); rc != 0 {
		return nil, fmt.Errorf("mksnap group results: %s", C.GoString(C.mksnap_last_error(e.h)))
	}
	view := (*[1 << 20]C.mksnap_group_result)(unsafe.Pointer(buf))[:nGroups:nGroups]
	out := make([]GroupResult, nGroups)
	for i := range out {
		r := &view[i]
		out[i] = GroupResult{Files: uint64(r.n_files), CdcBytes: uint64(r.cdc_bytes), Chunks: uint64(r.n_chunks),
			Unique: uint64(r.n_unique), FirstRow: uint64(r.first_row)}
		copy(out[i].Root[:], C.GoBytes(unsafe.Pointer(&r.root[0]), 32))
	}
	return out, nil
}

// GroupTable returns group g's sorted-unique chunk table (rows = its GroupResult.Unique), 32 bytes per row: the rows
// to persist next to that layer's <key>_chunks entry.
func (e *Engine) GroupTable(g int, rows uint64) ([]byte, error) {
	if rows == 0 {
		return nil, nil
	}
	buf := C.malloc(C.size_t(rows * 32))
	defer C.free(buf)
	if rc := C.mksnap_get_group_table(e.h, C.uint32_t(g), (*C.uint8_t)(buf), C.uint64_t(rows)); rc != 0 {
		return nil, fmt.Errorf("mksnap group table: %s", C.GoString(C.mksnap_last_error(e.h)))
	}
	return C.GoBytes(buf, C.int(rows*32)), nil
}

// DeltaGroups is "for every layer g in order: Delta(x), then x.AddTable" over a grouped session in one call, without
// changing x: a chunk of layer g is known if x holds it or an earlier layer of the batch has it.  ChunkStatus then
// returns these statuses.
func (e *Engine) DeltaGroups(x *Index, nGroups int) ([]DeltaResult, error) {
	if nGroups <= 0 {
		return nil, fmt.Errorf("mksnap delta groups: %d groups", nGroups)
	}
	buf := (*C.mksnap_delta_result)(C.calloc(C.size_t(nGroups), C.size_t(unsafe.Sizeof(C.mksnap_delta_result{}))))
	defer C.free(unsafe.Pointer(buf))
	if rc := C.mksnap_delta_groups(e.h, x.ix, buf, C.uint32_t(nGroups)); rc != 0 {
		return nil, fmt.Errorf("mksnap delta groups: %s", C.GoString(C.mksnap_last_error(e.h)))
	}
	view := (*[1 << 20]C.mksnap_delta_result)(unsafe.Pointer(buf))[:nGroups:nGroups]
	out := make([]DeltaResult, nGroups)
	for i := range out {
		r := &view[i]
		out[i] = DeltaResult{IndexRows: uint64(r.index_rows), KnownChunks: uint64(r.known_chunks), NewChunks: uint64(r.new_chunks),
			RepeatChunks: uint64(r.repeat_chunks), KnownBytes: uint64(r.known_bytes), NewBytes: uint64(r.new_bytes),
			RepeatBytes: uint64(r.repeat_bytes), DeviceMs: float32(r.ms_device)}
	}
	return out, nil
}

// AddGroup adds the chunk table of group g of e's finished grouped session.
func (x *Index) AddGroup(e *Engine, g int) error {
	if rc := C.mksnap_index_add_group(e.h, x.ix, C.uint32_t(g)); rc != 0 {
		return fmt.Errorf("mksnap index add group: %s", C.GoString(C.mksnap_last_error(e.h)))
	}
	return nil
}
