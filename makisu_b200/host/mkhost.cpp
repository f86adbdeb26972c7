// mkhost.cpp — host side above the mksnap C-ABI (see include/mkhost.h).
//
// C++ stand-in for the Go code a cgo build of makisu would keep on this path: the filepath.Walk-ordered
// context stream (cacheID), the MemFS copy-op layer (entry order + tar headers) and the arena packer.
// It does no hashing; digests come from libmksnap (GPU).  Reference line numbers are cited per function.
//
// One translation unit: the *.inc files in this directory are fragments of the anonymous namespace below, included in
// dependency order (Go path helpers, Walk/Glob, context stream, file reader pool, tar writer, tar reader, Copier,
// MemFS, arena packers); this file holds the C entry points.
#include "../../include/mkhost.h"

#include <dirent.h>
#include <errno.h>
#include <fcntl.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <array>
#include <atomic>
#include <condition_variable>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <chrono>
#include <string>
#include <thread>
#include <vector>

namespace {

struct HostError : std::runtime_error {
    using std::runtime_error::runtime_error;
};

std::string errno_str(const std::string &what, const std::string &path)
{
    return what + " " + path + ": " + strerror(errno);
}

#include "gopath.inc"
#include "gowalk.inc"
#include "context_stream.inc"
#include "reads.inc"
#include "tar_writer.inc"
#include "tar_reader.inc"
#include "copier.inc"
#include "memfs.inc"
#include "packer.inc"

} // namespace

// pure(file content) per context file, remembered between builds (incremental cacheID, include/mkhost.h)
struct mkhost_crc_cache {
    struct Entry {
        uint64_t dev, ino, size;
        int64_t mtime_ns, ctime_ns;
        uint32_t pure;
    };
    std::map<std::string, Entry> files; // key: absolute path
};

// persistent snapshot.MemFS mirror (layers accumulate in the merged tree, like context.BuildContext.MemFS)
struct mkhost_memfs {
    MemFS fs;
    mkhost_memfs(const std::string &root, std::vector<std::string> bl) : fs(root, 0, std::move(bl)) {}
};

// =====================================================================================================
extern "C" {

size_t mkhost_encode_tar_header(const mkhost_tar_header *h, uint8_t *out, size_t cap)
{
    try {
        Hdr x;
        x.name = h->name ? h->name : "";
        while (!x.name.empty() && x.name[0] == '/') // write.go:57 strings.TrimLeft(h.Name, "/")
            x.name.erase(0, 1);
        x.linkname = h->linkname ? h->linkname : "";
        x.mode = h->mode; x.uid = h->uid; x.gid = h->gid; x.size = h->size; x.mtime_ns = h->mtime_ns;
        x.typeflag = h->typeflag;
        std::string b = encode_header(x);
        if (b.size() > cap)
            return 0;
        memcpy(out, b.data(), b.size());
        return b.size();
    } catch (const std::exception &) {
        return 0;
    }
}

size_t mkhost_describe_context_stream(const char *context_dir, const char *const *from_paths, size_t n_paths, char *out,
                                      size_t cap, char *err, size_t errlen)
{
    try {
        std::string s;
        for (const auto &g : context_segments(go_clean(context_dir), from_paths, n_paths, 4)) { // 4: the parallel walk is what the parity tests see
            if (g.kind == 'F')
                s += "F " + std::to_string(g.size) + " " + g.path + "\n";
            else
                s += std::string(1, g.kind) + " " + g.bytes + "\n";
        }
        if (s.size() + 1 <= cap)
            memcpy(out, s.c_str(), s.size() + 1);
        return s.size() + 1;
    } catch (const std::exception &e) {
        set_err(err, errlen, std::string("hash context sources: ") + e.what());
        return 0;
    }
}

size_t mkhost_describe_layer(const char *root_dir, int64_t now_unix, const mkhost_copy_op *ops, size_t n_ops, char *out,
                             size_t cap, char *err, size_t errlen)
{
    try {
        MemFS fs(root_dir, now_unix);
        return emit_text(describe_layer_text(fs.add_layer_by_copy_ops(ops, n_ops)), out, cap);
    } catch (const std::exception &e) {
        set_err(err, errlen, std::string("create layer by copy ops: ") + e.what());
        return 0;
    }
}

mkhost_memfs *mkhost_memfs_new(const char *root_dir, const char *const *blacklist, size_t n_blacklist, char *err,
                               size_t errlen)
{
    try {
        std::vector<std::string> bl;
        for (size_t i = 0; i < n_blacklist; ++i)
            bl.emplace_back(blacklist[i]);
        return new mkhost_memfs(root_dir, std::move(bl));
    } catch (const std::exception &e) {
        set_err(err, errlen, e.what());
        return nullptr;
    }
}

void mkhost_memfs_free(mkhost_memfs *m) { delete m; }

int mkhost_memfs_file_digest(mkhost_memfs *m, const char *dst, uint8_t out[32])
{
    return m && dst && m->fs.get_digest(abs_path(dst), out) ? 0 : 1;
}

size_t mkhost_memfs_describe_copy_ops(mkhost_memfs *m, int64_t now_unix, const mkhost_copy_op *ops, size_t n_ops, char *out,
                                      size_t cap, char *err, size_t errlen)
{
    try {
        m->fs.set_now(now_unix);
        return emit_text(describe_layer_text(m->fs.add_layer_by_copy_ops(ops, n_ops)), out, cap);
    } catch (const std::exception &e) {
        set_err(err, errlen, std::string("create layer by copy ops: ") + e.what());
        return 0;
    }
}

size_t mkhost_memfs_describe_scan(mkhost_memfs *m, int64_t now_unix, char *out, size_t cap, char *err, size_t errlen)
{
    try {
        m->fs.set_now(now_unix);
        return emit_text(describe_layer_text(m->fs.add_layer_by_scan()), out, cap);
    } catch (const std::exception &e) {
        set_err(err, errlen, std::string("create layer by scan: ") + e.what());
        return 0;
    }
}

size_t mkhost_eval_symlinks(const char *path, const char *src_root, char *out, size_t cap, char *err, size_t errlen)
{
    try {
        return emit_text(eval_symlinks(path ? path : "", src_root ? src_root : ""), out, cap);
    } catch (const std::exception &e) {
        set_err(err, errlen, std::string("eval symlinks for ") + (path ? path : "") + ": " + e.what());
        return 0;
    }
}

int mkhost_copy_op_execute(const mkhost_copy_op *op, uint32_t mode, const char *const *blacklist, size_t n_blacklist,
                           char *err, size_t errlen)
{
    try {
        if (!op || op->n_srcs == 0)
            throw HostError("check copy param: srcs cannot be empty");
        std::vector<std::string> bl;
        for (size_t i = 0; i < n_blacklist; ++i)
            bl.emplace_back(blacklist[i]);
        std::multimap<std::string, DeferredFile> deferred;
        std::vector<Copier> copiers;
        execute_copy_op(*op, mode, bl, (mode & MKHOST_COPY_DEFERRED) ? &deferred : nullptr, &copiers);
        for (const auto &kv : deferred) { // stand-in for the arena: one read of each source, written from memory
            std::vector<uint8_t> buf((size_t)kv.second.st.st_size);
            std::vector<ReadJob> job{ReadJob{kv.first, 0, (uint64_t)buf.size(), buf.data()}};
            run_reads(job, 1);
            copiers[kv.second.copier].finish_regular(kv.second.st, kv.first, kv.second.dst, buf.data(), buf.size());
        }
        return 0;
    } catch (const std::exception &e) {
        set_err(err, errlen, e.what());
        return -1;
    }
}

int mkhost_memfs_commit_copy_ops(mkhost_memfs *m, mksnap_t *eng, int64_t now_unix, const mkhost_copy_op *ops, size_t n_ops,
                                 int n_threads, int tar_fd, uint32_t flags, mkhost_layer_result *out, char *err,
                                 size_t errlen)
{
    try {
        m->fs.set_now(now_unix);
        if (!(flags & MKHOST_MATERIALIZE)) {
            commit_layer(eng, m->fs.add_layer_by_copy_ops(ops, n_ops), n_threads, tar_fd, flags, out, &m->fs);
            return 0;
        }
        // SURVEY section 8f-4: the copy onto the file system (CopyOperation.Execute) and the layer share one read of the
        // context.  Directories, symlinks and chmods first; regular files are written from the arena as it fills;
        // what the layer did not need to read (entries the tree already holds) is copied from disk at the end.
        std::multimap<std::string, DeferredFile> deferred;
        std::vector<Copier> copiers;
        const uint32_t mode = (flags & MKHOST_MATERIALIZE_CHOWN) ? MKHOST_COPY_CHOWN : 0u;
        for (size_t i = 0; i < n_ops; ++i) {
            mkhost_copy_op on_disk = ops[i];
            std::string dst = ops[i].dst ? ops[i].dst : "";
            const bool dir_fmt = (!dst.empty() && dst.back() == '/') || dst == "." || dst == "..";
            if (dst.empty() || dst[0] != '/') {
                if (!ops[i].work_dir || ops[i].work_dir[0] != '/')
                    throw HostError("check copy param: dst is not absolute path, must specify absolute working directory");
                dst = go_join(ops[i].work_dir, dst);
            }
            dst = go_join(m->fs.root(), dst) + (dir_fmt ? "/" : ""); // image path -> path under the MemFS root ("/" in a real build)
            on_disk.dst = dst.c_str();
            execute_copy_op(on_disk, mode, m->fs.blacklist(), &deferred, &copiers);
        }
        auto write_from_arena = [&](const std::vector<ReadJob> &jobs) {
            for (const auto &j : jobs) {
                if (j.file_off != 0)
                    continue;
                auto range = deferred.equal_range(j.path);
                if (range.first == range.second || (uint64_t)range.first->second.st.st_size != j.len)
                    continue; // a piece of a file larger than the arena: that file is copied from disk at the end
                for (auto it = range.first; it != range.second; ++it)
                    copiers[it->second.copier].finish_regular(it->second.st, j.path, it->second.dst, j.dst, j.len);
                deferred.erase(range.first, range.second);
            }
        };
        commit_layer(eng, m->fs.add_layer_by_copy_ops(ops, n_ops), n_threads, tar_fd, flags, out, &m->fs, write_from_arena);
        for (const auto &kv : deferred)
            copiers[kv.second.copier].finish_regular(kv.second.st, kv.first, kv.second.dst, nullptr, 0);
        return 0;
    } catch (const std::exception &e) {
        set_err(err, errlen, std::string("failed to generate diff layer: ") + e.what());
        return -1;
    }
}

int mkhost_memfs_commit_layers(mkhost_memfs *m, mksnap_t *eng, int64_t now_unix, const mkhost_layer_spec *specs, size_t n_layers,
                               int n_threads, uint32_t flags, mkhost_layer_result *outs, char *err, size_t errlen)
{
    try {
        if (!m || !eng || (!specs && n_layers) || (!outs && n_layers))
            throw HostError("null argument");
        if (flags & ~(uint32_t)(MKHOST_NO_TAR_DIGEST | MKHOST_LAYER_TABLES))
            throw HostError("commit layers: only MKHOST_NO_TAR_DIGEST and MKHOST_LAYER_TABLES are supported for a batch");
        m->fs.set_now(now_unix);
        // the layer maps are built in order -- each AddLayerByCopyOps sees the tree its predecessors left
        // (mem_fs.go:276-289) -- and only then packed together
        std::vector<std::map<std::string, MemFile>> maps;
        maps.reserve(n_layers);
        for (size_t i = 0; i < n_layers; ++i)
            maps.push_back(m->fs.add_layer_by_copy_ops(specs[i].ops, specs[i].n_ops));
        std::vector<BatchLayer> bl;
        for (size_t i = 0; i < n_layers; ++i)
            bl.push_back(BatchLayer{&maps[i], specs[i].tar_fd});
        commit_layers_batch(eng, bl, n_threads, flags, outs);
        return 0;
    } catch (const std::exception &e) {
        set_err(err, errlen, std::string("failed to generate diff layers: ") + e.what());
        return -1;
    }
}

int mkhost_memfs_commit_scan(mkhost_memfs *m, mksnap_t *eng, int64_t now_unix, int n_threads, int tar_fd, uint32_t flags,
                             mkhost_layer_result *out, char *err, size_t errlen)
{
    try {
        m->fs.set_now(now_unix);
        if (!(flags & MKHOST_SCAN_CONTENT)) {
            commit_layer(eng, m->fs.add_layer_by_scan(), n_threads, tar_fd, flags, out, &m->fs);
            return 0;
        }
        // content-aware scan (SURVEY section 8f-3): the reference trusts mtime+size and therefore sync()s and sleeps
        // a second before every scan (mem_fs.go:291-311); here files the metadata calls unchanged are re-hashed on
        // the GPU and compared with the digest remembered when they were committed.
        std::vector<Suspect> suspects;
        std::map<std::string, MemFile> layer = m->fs.add_layer_by_scan(&suspects);
        const std::vector<std::array<uint8_t, 32>> now = digest_files(eng, suspects, n_threads);
        for (size_t k = 0; k < suspects.size(); ++k)
            if (now[k] != suspects[k].known)
                m->fs.add_changed(layer, suspects[k]);
        commit_layer(eng, layer, n_threads, tar_fd, flags, out, &m->fs);
        return 0;
    } catch (const std::exception &e) {
        set_err(err, errlen, std::string("failed to generate diff layer: ") + e.what());
        return -1;
    }
}

size_t mkhost_memfs_describe_update_from_tar_ex(mkhost_memfs *m, int64_t now_unix, int tar_fd, uint32_t flags, char *out,
                                                size_t cap, char *err, size_t errlen)
{
    try {
        m->fs.set_now(now_unix);
        std::vector<uint8_t> buf;
        uint8_t tmp[65536];
        for (;;) {
            ssize_t r = read(tar_fd, tmp, sizeof tmp);
            if (r < 0) {
                if (errno == EINTR)
                    continue;
                throw HostError(std::string("read header: ") + strerror(errno));
            }
            if (r == 0)
                break;
            buf.insert(buf.end(), tmp, tmp + r);
        }
        MemTarSource src(buf.data(), buf.size());
        if (flags & MKHOST_UNTAR) {
            MemFS::Untar u;
            read_tar(src, [&](const TarMember &mem, const uint8_t *body) { m->fs.untar_member(u, mem, body); });
            return emit_text(describe_layer_text(m->fs.untar_finish(u)), out, cap);
        }
        return emit_text(describe_layer_text(m->fs.update_from_tar(read_tar(src))), out, cap);
    } catch (const std::exception &e) {
        set_err(err, errlen, std::string("update memfs from tar: ") + e.what());
        return 0;
    }
}

size_t mkhost_memfs_describe_update_from_tar(mkhost_memfs *m, int64_t now_unix, int tar_fd, char *out, size_t cap, char *err,
                                             size_t errlen)
{
    return mkhost_memfs_describe_update_from_tar_ex(m, now_unix, tar_fd, 0, out, cap, err, errlen);
}

int mkhost_memfs_update_from_tar(mkhost_memfs *m, mksnap_t *eng, int64_t now_unix, int tar_fd, uint32_t flags,
                                 mkhost_layer_result *out, char *err, size_t errlen)
{
    try {
        m->fs.set_now(now_unix);
        const bool want_digest = !(flags & MKHOST_NO_TAR_DIGEST);
        ck(eng, mksnap_begin(eng), "begin");
        const bool file_digests = (flags & MKHOST_FILE_DIGESTS) != 0;
        ArenaTarSource src(eng, tar_fd, want_digest, file_digests);
        const bool untar = (flags & MKHOST_UNTAR) != 0;
        src.allow_split = !untar; // untarOneItem writes a member from one contiguous body
        MemFS::Untar u;
        const std::vector<TarMember> members =
            untar ? read_tar(src, [&](const TarMember &mem, const uint8_t *body) { m->fs.untar_member(u, mem, body); }) // files written from the arena
                  : read_tar(src);
        src.flush(true);
        mksnap_result res;
        ck(eng, mksnap_finish(eng, &res), "finish");
        memset(out->tar_digest, 0, 32);
        std::vector<uint8_t> d((size_t)(src.n_file_streams + 1) * 32);
        if (want_digest || src.n_file_streams)
            ck(eng, mksnap_get_stream_digests(eng, d.data(), src.n_file_streams + 1), "stream digests");
        if (want_digest)
            memcpy(out->tar_digest, d.data(), 32);
        memcpy(out->root, res.root, 32);
        const std::map<std::string, MemFile> layer = untar ? m->fs.untar_finish(u) : m->fs.update_from_tar(members);
        out->n_entries = layer.size();
        if (file_digests) { // remember the content digest of every regular member that made it into the tree
            uint32_t k = 0;
            for (const auto &mem : members) {
                if (mem.hdr.typeflag != '0' || mem.data_len == 0)
                    continue;
                ++k;
                const std::string dst = abs_path(mem.hdr.name);
                auto it = layer.find(dst);
                if (it != layer.end() && !it->second.whiteout && it->second.hdr.typeflag == '0')
                    m->fs.set_digest(dst, d.data() + 32 * k);
            }
        }
        out->tar_bytes = src.tar_bytes;
        out->n_chunks = res.n_chunks;
        out->n_unique = res.n_unique;
        return 0;
    } catch (const std::exception &e) {
        set_err(err, errlen, std::string("update memfs from tar: ") + e.what());
        return -1;
    }
}

// ---- cache.Manager wire format (lib/cache/cache_manager.go:34-35,239-252) ----
size_t mkhost_cache_key(const char *cache_id, int chunk_table, char *out, size_t cap)
{
    return emit_text(std::string("makisu_builder_cache_") + (cache_id ? cache_id : "") + (chunk_table ? "_chunks" : ""), out, cap);
}

size_t mkhost_cache_entry_create(const char *tar_hex, const char *gzip_hex, char *out, size_t cap)
{
    if (!tar_hex) // createEntry(nil)
        return emit_text("MAKISU_CACHE_EMPTY", out, cap);
    return emit_text(std::string(tar_hex) + "," + (gzip_hex ? gzip_hex : ""), out, cap);
}

int mkhost_cache_entry_parse(const char *entry, char *tar_digest, size_t tar_cap, char *gzip_digest, size_t gzip_cap,
                             char *err, size_t errlen)
{
    const std::string e = entry ? entry : "";
    const size_t c = e.find(',');
    if (c == std::string::npos) {
        set_err(err, errlen, "parse redis entry: " + e);
        return -1;
    }
    const std::string t = "sha256:" + e.substr(0, c), g = "sha256:" + e.substr(c + 1); // SplitN(entry, ",", 2)
    if (t.size() + 1 > tar_cap || g.size() + 1 > gzip_cap) {
        set_err(err, errlen, "parse redis entry: output buffer too small");
        return -1;
    }
    memcpy(tar_digest, t.c_str(), t.size() + 1);
    memcpy(gzip_digest, g.c_str(), g.size() + 1);
    return 0;
}

size_t mkhost_cache_chunk_entry_create(const uint8_t root[32], uint64_t n_unique, char *out, size_t cap)
{
    static const char *hx = "0123456789abcdef";
    std::string s;
    for (int i = 0; i < 32; ++i) {
        s += hx[root[i] >> 4];
        s += hx[root[i] & 15];
    }
    return emit_text(s + "," + std::to_string(n_unique), out, cap);
}

int mkhost_cache_chunk_entry_parse(const char *entry, uint8_t root[32], uint64_t *n_unique, char *err, size_t errlen)
{
    const std::string e = entry ? entry : "";
    auto nib = [](char c) { return c >= '0' && c <= '9' ? c - '0' : (c >= 'a' && c <= 'f' ? c - 'a' + 10 : -1); };
    bool ok = e.size() > 65 && e[64] == ',';
    for (int i = 0; ok && i < 64; ++i)
        ok = nib(e[i]) >= 0;
    uint64_t n = 0;
    for (size_t i = 65; ok && i < e.size(); ++i) {
        ok = e[i] >= '0' && e[i] <= '9' && n <= (UINT64_MAX - 9) / 10;
        n = n * 10 + (uint64_t)(e[i] - '0');
    }
    if (!ok) {
        set_err(err, errlen, "parse chunk table entry: " + e);
        return -1;
    }
    for (int i = 0; i < 32; ++i)
        root[i] = (uint8_t)(nib(e[2 * i]) * 16 + nib(e[2 * i + 1]));
    *n_unique = n;
    return 0;
}

static int context_crc32_impl(mksnap_t *eng, mkhost_crc_cache *cache, mkhost_crc_cache_stats *stats, const void *prefix,
                              size_t prefix_len, const char *context_dir, const char *const *from_paths, size_t n_paths,
                              int n_threads, uint32_t *crc_out, uint64_t *stream_len_out, char *err, size_t errlen)
{
    try {
        const bool trace = getenv("MKHOST_TRACE") != nullptr; // phase times on stderr
        const auto t_start = std::chrono::steady_clock::now();
        auto ms_since = [&](std::chrono::steady_clock::time_point t) {
            return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t).count();
        };
        double ms_reads = 0, ms_submit = 0, ms_acquire = 0;
        std::vector<Seg> segs = context_segments(go_clean(context_dir), from_paths, n_paths, n_threads);
        const double ms_walk = ms_since(t_start);
        uint64_t total = prefix_len;
        for (const auto &g : segs)
            total += g.kind == 'F' ? g.size : g.bytes.size();
        ck(eng, mksnap_begin(eng), "begin");

        const mksnap_limits lim = engine_limits(eng);
        void *hp = nullptr;
        uint64_t cap = 0;
        ArenaLease lease(eng);
        int32_t &aid = lease.id;
        uint64_t pos = 0;
        std::vector<mksnap_extent> ext;
        std::vector<ReadJob> jobs;
        auto acquire = [&]() {
            const auto t = std::chrono::steady_clock::now();
            ck(eng, mksnap_arena_acquire(eng, &hp, &cap, &aid), "arena acquire");
            ms_acquire += ms_since(t);
            pos = 0;
            ext.clear();
            jobs.clear();
        };
        auto flush = [&]() {
            auto t = std::chrono::steady_clock::now();
            run_reads(jobs, n_threads);
            ms_reads += ms_since(t);
            t = std::chrono::steady_clock::now();
            ck(eng, mksnap_arena_submit(eng, aid, pos, ext.data(), ext.size(), nullptr, 0), "arena submit");
            ms_submit += ms_since(t);
            aid = -1;
        };
        acquire();
        uint64_t after = total; // stream bytes not yet placed
        uint64_t n_crc_ext = 0; // CRC extents submitted so far in this session (index into mksnap_get_extent_crcs)
        struct Sent {           // a file that travelled: its extents [first, first + pieces) and their lengths
            const Seg *seg;
            uint64_t first;
            std::vector<uint64_t> piece_len;
        };
        std::vector<Sent> sent;
        mkhost_crc_cache_stats st{};
        auto put_bytes = [&](const void *p, size_t n) {
            if (n == 0)
                return;
            uint64_t o = align_up(pos, 16);
            if (o + n > cap || ext.size() >= lim.max_extents) { // the extent table fills before the arena on tiny files

                flush();
                acquire();
                o = 0;
            }
            if (n > cap)
                throw HostError("path string larger than the arena");
            memcpy((uint8_t *)hp + o, p, n);
            after -= n;
            ext.push_back(mksnap_extent{o, n, after, MKSNAP_X_CRC, 0});
            ++n_crc_ext;
            pos = o + n;
        };
        put_bytes(prefix, prefix_len);
        for (const auto &g : segs) {
            if (g.kind != 'F') {
                put_bytes(g.bytes.data(), g.bytes.size());
                continue;
            }
            ++st.files_total;
            st.bytes_total += g.size;
            if (cache) { // unchanged since a build that remembered it: fold pure(content) in, send nothing
                auto it = cache->files.find(g.path);
                if (it != cache->files.end() && it->second.dev == g.dev && it->second.ino == g.ino && it->second.size == g.size &&
                    it->second.mtime_ns == g.mtime_ns && it->second.ctime_ns == g.ctime_ns) {
                    after -= g.size;
                    ck(eng, mksnap_crc_add(eng, it->second.pure, g.size, after), "crc add");
                    ++st.files_reused;
                    continue;
                }
            }
            st.bytes_sent += g.size;
            if (cache)
                sent.push_back(Sent{&g, n_crc_ext, {}});
            uint64_t done = 0; // CRC is linear: a file may be split across arenas at any 16-byte boundary
            while (done < g.size) {
                uint64_t o = align_up(pos, 512);
                if (o + 4096 > cap || ext.size() >= lim.max_extents) {
                    flush();
                    acquire();
                    o = 0;
                }
                uint64_t n = std::min<uint64_t>(g.size - done, (cap - o) / 16 * 16);
                jobs.push_back(ReadJob{g.path, done, n, (uint8_t *)hp + o});
                after -= n;
                ext.push_back(mksnap_extent{o, n, after, MKSNAP_X_CRC, 0});
                ++n_crc_ext;
                if (cache)
                    sent.back().piece_len.push_back(n);
                pos = o + n;
                done += n;
            }
        }
        flush();
        mksnap_result res;
        const auto t_fin = std::chrono::steady_clock::now();
        ck(eng, mksnap_finish(eng, &res), "finish");
        if (trace)
            fprintf(stderr, "[mkhost] context crc32: %zu segments, %.1f MiB; walk %.2f ms, reads %.2f, acquire waits %.2f, submit %.2f, "
                            "finish %.2f, total %.2f ms\n",
                    segs.size(), (double)total / 1048576.0, ms_walk, ms_reads, ms_acquire, ms_submit, ms_since(t_fin), ms_since(t_start));
        if (res.crc_bytes != total)
            throw HostError("internal: stream length mismatch");
        *crc_out = mksnap_ctx_crc32(&res);
        if (stream_len_out)
            *stream_len_out = total;
        if (cache) { // remember pure(content) of every file that travelled (pieces joined: pure(A||B) = pure(A) x^(8|B|) ^ pure(B))
            std::vector<uint32_t> pure(std::max<uint64_t>(1, n_crc_ext));
            uint64_t n_got = 0;
            ck(eng, mksnap_get_extent_crcs(eng, pure.data(), pure.size(), &n_got), "extent crcs");
            if (n_got != n_crc_ext)
                throw HostError("internal: extent count mismatch");
            for (const Sent &f : sent) {
                uint32_t v = 0; // pure of the empty string
                for (size_t k = 0; k < f.piece_len.size(); ++k)
                    v = mksnap_crc_concat(v, pure[f.first + k], f.piece_len[k]);
                cache->files[f.seg->path] =
                    mkhost_crc_cache::Entry{f.seg->dev, f.seg->ino, f.seg->size, f.seg->mtime_ns, f.seg->ctime_ns, v};
            }
        }
        if (stats)
            *stats = st;
        return 0;
    } catch (const std::exception &e) {
        set_err(err, errlen, std::string("hash context sources: ") + e.what());
        return -1;
    }
}

int mkhost_context_crc32(mksnap_t *eng, const void *prefix, size_t prefix_len, const char *context_dir,
                         const char *const *from_paths, size_t n_paths, int n_threads, uint32_t *crc_out,
                         uint64_t *stream_len_out, char *err, size_t errlen)
{
    return context_crc32_impl(eng, nullptr, nullptr, prefix, prefix_len, context_dir, from_paths, n_paths, n_threads, crc_out,
                              stream_len_out, err, errlen);
}

mkhost_crc_cache *mkhost_crc_cache_new(void) { return new mkhost_crc_cache; }
void mkhost_crc_cache_free(mkhost_crc_cache *c) { delete c; }
uint64_t mkhost_crc_cache_size(const mkhost_crc_cache *c) { return c ? c->files.size() : 0; }

int mkhost_crc_cache_save(const mkhost_crc_cache *c, const char *path, char *err, size_t errlen)
{
    FILE *f = c && path ? fopen(path, "w") : nullptr;
    if (!f) {
        set_err(err, errlen, std::string("save crc cache: ") + strerror(errno));
        return -1;
    }
    fprintf(f, "mkhost-crc-cache 1\n");
    for (const auto &kv : c->files) // path last: it may hold spaces (newlines in file names are not cached)
        if (kv.first.find('\n') == std::string::npos)
            fprintf(f, "%llu %llu %llu %lld %lld %08x %s\n", (unsigned long long)kv.second.dev, (unsigned long long)kv.second.ino,
                    (unsigned long long)kv.second.size, (long long)kv.second.mtime_ns, (long long)kv.second.ctime_ns, kv.second.pure,
                    kv.first.c_str());
    const bool ok = fclose(f) == 0;
    if (!ok)
        set_err(err, errlen, std::string("save crc cache: ") + strerror(errno));
    return ok ? 0 : -1;
}

int mkhost_crc_cache_load(mkhost_crc_cache *c, const char *path, char *err, size_t errlen)
{
    FILE *f = c && path ? fopen(path, "r") : nullptr;
    if (!f) {
        set_err(err, errlen, std::string("load crc cache: ") + strerror(errno));
        return -1;
    }
    char *line = nullptr;
    size_t cap = 0;
    ssize_t n = getline(&line, &cap, f);
    bool ok = n > 0 && strncmp(line, "mkhost-crc-cache 1", 18) == 0;
    while (ok && (n = getline(&line, &cap, f)) > 0) {
        if (line[n - 1] == '\n')
            line[--n] = 0;
        unsigned long long dev, ino, size;
        long long mt, ct;
        unsigned pure;
        int used = 0;
        if (sscanf(line, "%llu %llu %llu %lld %lld %x %n", &dev, &ino, &size, &mt, &ct, &pure, &used) != 6 || used <= 0 || used >= n) {
            ok = false;
            break;
        }
        c->files[line + used] = mkhost_crc_cache::Entry{dev, ino, size, mt, ct, (uint32_t)pure};
    }
    free(line);
    fclose(f);
    if (!ok)
        set_err(err, errlen, "load crc cache: not a mkhost-crc-cache file");
    return ok ? 0 : -1;
}

int mkhost_context_crc32_cached(mksnap_t *eng, mkhost_crc_cache *cache, const void *prefix, size_t prefix_len,
                                const char *context_dir, const char *const *from_paths, size_t n_paths, int n_threads,
                                uint32_t *crc_out, uint64_t *stream_len_out, mkhost_crc_cache_stats *stats, char *err, size_t errlen)
{
    if (!cache) {
        set_err(err, errlen, "hash context sources: no cache object");
        return -1;
    }
    return context_crc32_impl(eng, cache, stats, prefix, prefix_len, context_dir, from_paths, n_paths, n_threads, crc_out,
                              stream_len_out, err, errlen);
}

int mkhost_commit_copy_ops(mksnap_t *eng, const char *root_dir, int64_t now_unix, const mkhost_copy_op *ops, size_t n_ops,
                           int n_threads, mkhost_layer_result *out, char *err, size_t errlen)
{
    return mkhost_commit_copy_ops_to_fd(eng, root_dir, now_unix, ops, n_ops, n_threads, -1, out, err, errlen);
}

int mkhost_commit_copy_ops_to_fd(mksnap_t *eng, const char *root_dir, int64_t now_unix, const mkhost_copy_op *ops,
                                 size_t n_ops, int n_threads, int tar_fd, mkhost_layer_result *out, char *err,
                                 size_t errlen)
{
    return mkhost_commit_copy_ops_ex(eng, root_dir, now_unix, ops, n_ops, n_threads, tar_fd, 0, out, err, errlen);
}

int mkhost_commit_copy_ops_ex(mksnap_t *eng, const char *root_dir, int64_t now_unix, const mkhost_copy_op *ops,
                              size_t n_ops, int n_threads, int tar_fd, uint32_t flags, mkhost_layer_result *out,
                              char *err, size_t errlen)
{
    try {
        MemFS fs(root_dir, now_unix);
        commit_layer(eng, fs.add_layer_by_copy_ops(ops, n_ops), n_threads, tar_fd, flags, out);
        return 0;
    } catch (const std::exception &e) {
        set_err(err, errlen, std::string("failed to generate diff layer: ") + e.what());
        return -1;
    }
}

} // extern "C"
