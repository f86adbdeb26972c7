// mksnap.cu — C-ABI implementation of include/mksnap.h (libmksnap.so).
//
// Host-side orchestration only: arena ring, extent tables, stream/event
// plumbing, result tables.  All arithmetic happens in the kernels of
// mksnap_kernels.cuh; there is deliberately no CPU fallback.
#include "../../include/mksnap.h"
#include "mksnap_kernels.cuh"
#include "mksnap_index.cuh"

#include <dlfcn.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include <algorithm>
#include <string>
#include <vector>

using namespace mk;

struct Id128 {
    char b[128];
};

namespace {

thread_local std::string g_create_error;

constexpr uint64_t SLOT_SLACK = 8192;
constexpr int N_EV = 8; // timing marks per submit
constexpr uint32_t MAX_SLOTS = 4;
constexpr int GH_WORDS = 8; // u64 words per rank in the all-gather header

struct MetaSet {
    // pinned host staging
    CrcExtent *h_crc = nullptr;
    uint32_t *h_piece_base = nullptr;
    CdcFile *h_files = nullptr;
    uint64_t *h_rstart = nullptr, *h_rlen = nullptr;
    uint32_t *h_rstream = nullptr, *h_rflags = nullptr;
    // device mirrors
    CrcExtent *d_crc = nullptr;
    uint32_t *d_piece_base = nullptr;
    uint32_t *d_ext_pure = nullptr; // pure(extent) of this submit's CRC extents
    CdcFile *d_files = nullptr;
    uint64_t *d_rstart = nullptr, *d_rlen = nullptr;
    uint32_t *d_rstream = nullptr, *d_rflags = nullptr;
    cudaEvent_t ev_done = nullptr; // kernels that read this set have finished
    bool in_flight = false;
};

struct HostArena {
    uint8_t *ptr = nullptr;
    cudaEvent_t ev_h2d = nullptr;
    bool in_flight = false;
    bool acquired = false;
};

// NCCL via dlopen: only the handful of entry points we need
struct NcclApi {
    void *lib = nullptr;
    int (*GetUniqueId)(void *) = nullptr;
    int (*CommInitRank)(void **, int, /* ncclUniqueId by value */ Id128, int) = nullptr;
    int (*AllGather)(const void *, void *, size_t, int, void *, cudaStream_t) = nullptr;
    int (*Send)(const void *, size_t, int, int, void *, cudaStream_t) = nullptr;
    int (*Recv)(void *, size_t, int, int, void *, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    int (*CommDestroy)(void *) = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
};

} // namespace

struct mksnap {
    mksnap_config cfg;
    CdcParamsDev prm;
    std::string err;
    int sm_count = 148;
    cudaStream_t s_comp = nullptr, s_copy = nullptr;

    uint32_t n_slots = 0;
    uint8_t *d_slot[MAX_SLOTS] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t ev_slot_free[MAX_SLOTS] = {nullptr, nullptr, nullptr, nullptr};
    bool slot_used[MAX_SLOTS] = {false, false, false, false};

    std::vector<HostArena> arenas;
    uint32_t next_arena = 0;

    std::vector<MetaSet> meta;
    uint64_t submit_idx = 0;

    CrcConsts *d_consts = nullptr;
    SessionCounters *d_sc = nullptr;
    SessionCounters *h_sc = nullptr; // pinned

    TileRec *d_tiles = nullptr;
    CUtensorMap tm_main[MAX_SLOTS]; // per slot: arena viewed as [rows][128 B]
    int scan_cfg = 0; // index into SCAN_SHAPES
    bool sha_fma = true; // chunk SHA-256: additions on the FMA pipe
    uint32_t *d_pool = nullptr;
    uint32_t pool_cap = 0;
    uint32_t *d_pool_count = nullptr;
    uint32_t *d_counts = nullptr, *d_bases = nullptr;
    uint32_t *d_scan_tmp = nullptr; // block sums for the generic scan (several levels)
    uint64_t scan_tmp_words = 0;

    // session tables
    uint64_t max_chunks = 0;
    uint64_t *d_chunk_start = nullptr, *d_chunk_len = nullptr, *d_chunk_end = nullptr;
    uint32_t *d_order = nullptr; // K2 work order of the current batch (batch-relative chunk indices)
    bool sha_order = true;
    uint8_t *d_digests = nullptr;
    uint64_t max_streams = 0;
    uint8_t *d_stream_digests = nullptr;
    StreamState *d_stream_state = nullptr;
    std::vector<uint32_t> stream_stamp; // submit epoch that last used the stream slot (one piece per stream per submit)
    uint32_t stamp_epoch = 0;
    uint64_t n_streams = 0;
    uint64_t stream_base = 0; // bytes of arenas submitted before the current one
    uint64_t crc_bytes = 0;
    uint32_t *d_crc_session = nullptr; // pure(extent) of every CRC extent of the session, submission order
    uint64_t crc_session_cap = 0, crc_session_n = 0;
    uint32_t crc_host_acc = 0;         // contributions folded on the host (mksnap_crc_add)
    uint64_t crc_host_bytes = 0;
    bool open_file = false;      // the last submit ended with a MKSNAP_X_MORE extent: the next must start with its continuation
    uint8_t *d_carry = nullptr;  // open chunk of that file (k_carry_out -> k_carry_in)
    uint64_t carry_cap = 0;

    // sort / table
    uint64_t *d_keys[2] = {nullptr, nullptr};
    uint32_t *d_idx[2] = {nullptr, nullptr};
    uint8_t *d_sorted = nullptr, *d_table = nullptr;
    uint32_t *d_flags = nullptr, *d_pos = nullptr, *d_hist = nullptr;
    uint8_t *d_merkle[2] = {nullptr, nullptr};
    uint64_t table_cap = 0; // rows the sort buffers can hold
    uint64_t n_unique = 0;
    uint8_t root[32];
    bool finished = false;
    bool in_session = false;
    bool table_own = false; // d_table is the finished session's own table (set by finish; cleared by begin, exchange, all-gather)
    mksnap_result last_result;

    // chunk delta: allocated by the first mksnap_delta, sized for max_chunks
    uint32_t *d_dfirst = nullptr; // per session-table row: lowest non-known chunk carrying it
    uint32_t *d_duidx = nullptr;  // per chunk: its session-table row (IDX_NONE = known)
    uint32_t *d_ddir = nullptr;   // prefix directory of d_table
    uint8_t *d_dstatus = nullptr; // per chunk: MKSNAP_CHUNK_*
    unsigned long long *d_dcnt = nullptr;
    cudaEvent_t ev_delta[2] = {nullptr, nullptr};
    bool delta_done = false; // d_dstatus holds this session's statuses

    // multi-GPU
    NcclApi nccl;
    void *comm = nullptr;
    int n_ranks = 1, rank = 0;
    uint8_t *d_gather = nullptr; // n_ranks * pad_rows * 32
    uint64_t gather_rows = 0;
    unsigned long long *d_gcount = nullptr; // n_ranks * GH_WORDS header words
    uint8_t *d_concat = nullptr;            // dense concatenation of all ranks' tables
    uint64_t concat_rows = 0;
    // range-partitioned exchange (mksnap_exchange_tables): small fixed-size scratch
    unsigned long long *d_xbounds = nullptr; // R+1 slice boundaries of my table
    unsigned long long *d_xhdr = nullptr;    // R * (GH_WORDS + R) header words
    uint8_t *d_xrec = nullptr;               // R records of XREC_BYTES: u64 rows-in-range, then the first 255 rows
    uint8_t *d_xtail = nullptr;              // 256 rows: the Merkle group that straddles the end of my range
    int x_ranks = 0;

    // timing
    cudaEvent_t ev[N_EV];
    cudaEvent_t ev_copy0 = nullptr, ev_copy1 = nullptr, ev_copy_done = nullptr;
    cudaEvent_t ev_fin[4];
    bool have_submit_times = false, have_h2d_time = false, have_fin_times = false, have_gather_time = false;
    mksnap_stats_t stats;
};

namespace {

int fail(mksnap *h, int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (h)
        h->err = buf;
    else
        g_create_error = buf;
    return code;
}

#define CK(h, call)                                                                                   \
    do {                                                                                              \
        cudaError_t e__ = (call);                                                                     \
        if (e__ != cudaSuccess)                                                                       \
            return fail((h), e__ == cudaErrorMemoryAllocation ? MKSNAP_E_NOMEM : MKSNAP_E_CUDA,       \
                        "%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__));          \
    } while (0)

#define LAUNCH_OK(h)                                                                                  \
    do {                                                                                              \
        cudaError_t e__ = cudaGetLastError();                                                         \
        if (e__ != cudaSuccess)                                                                       \
            return fail((h), MKSNAP_E_CUDA, "%s:%d kernel launch: %s", __FILE__, __LINE__,            \
                        cudaGetErrorString(e__));                                                     \
        (h)->stats.kernel_launches++;                                                                 \
    } while (0)

uint32_t xpow_bits(uint64_t bits) // x^bits mod P, reflected
{
    uint32_t result = 0x80000000u, sq = 0x40000000u; // x^0, x^1
    while (bits) {
        if (bits & 1)
            result = crc_mulmod(result, sq);
        sq = crc_mulmod(sq, sq);
        bits >>= 1;
    }
    return result;
}

void build_crc_consts(CrcConsts *c)
{
    const uint32_t x4096 = xpow_bits(4096);
    for (int t = 0; t < 4; t++)
        for (uint32_t v = 0; v < 256; v++)
            c->mulk[t][v] = crc_mulmod(v << (8 * t), x4096);
    for (int l = 0; l < 32; l++)
        for (int k = 0; k < 4; k++)
            c->lane_c[l * 4 + k] = xpow_bits(32 + 8 * (508 - 16 * l - 4 * k));
    uint32_t sq = 0x40000000u;
    for (int i = 0; i < 32; i++) {
        c->xp[i] = sq;
        sq = crc_mulmod(sq, sq);
    }
}

// generic device exclusive scan (u32), in -> out (may alias), n elements; block sums go to h->d_scan_tmp unless the
// caller brings its own temporary
int scan_u32(mksnap *h, const uint32_t *in, uint32_t *out, uint64_t n, cudaStream_t s, uint32_t *tmp = nullptr,
             uint64_t tmp_words = 0)
{
    if (!tmp) {
        tmp = h->d_scan_tmp;
        tmp_words = h->scan_tmp_words;
    }
    if (n == 0)
        return 0;
    // level sizes
    std::vector<uint64_t> sizes;
    sizes.push_back(n);
    while (sizes.back() > SCAN_ITEMS)
        sizes.push_back((sizes.back() + SCAN_ITEMS - 1) / SCAN_ITEMS);
    // temp layout: level l (l>=1) sums at offset
    std::vector<uint64_t> off(sizes.size(), 0);
    uint64_t total = 0;
    for (size_t l = 1; l < sizes.size(); l++) {
        off[l] = total;
        total += sizes[l];
    }
    if (total > tmp_words)
        return fail(h, MKSNAP_E_CAPACITY, "scan temp too small (%llu > %llu)", (unsigned long long)total,
                    (unsigned long long)tmp_words);
    // up-sweep: reduce each level into the next
    for (size_t l = 0; l + 1 < sizes.size(); l++) {
        const uint32_t *src = l == 0 ? in : tmp + off[l];
        uint32_t nb = (uint32_t)sizes[l + 1];
        k_scan_reduce<<<nb, 256, 0, s>>>(src, sizes[l], tmp + off[l + 1]);
        LAUNCH_OK(h);
    }
    // top level fits one block: scan in place
    for (size_t l = sizes.size(); l-- > 0;) {
        const uint32_t *src = l == 0 ? in : tmp + off[l];
        uint32_t *dst = l == 0 ? out : tmp + off[l];
        const uint32_t *boff = (l + 1 < sizes.size()) ? tmp + off[l + 1] : nullptr;
        uint32_t nb = (uint32_t)((sizes[l] + SCAN_ITEMS - 1) / SCAN_ITEMS);
        k_scan_apply<<<nb, 256, 0, s>>>(src, sizes[l], boff, dst);
        LAUNCH_OK(h);
    }
    return 0;
}

int sha_grid(const mksnap *h) { return h->sm_count * 8; }

// sort n digests at `src` -> sorted unique table at h->d_table; sets h->n_unique, root
int sort_unique_root(mksnap *h, const uint8_t *src, uint64_t n, cudaStream_t s)
{
    if (n > h->table_cap)
        return fail(h, MKSNAP_E_CAPACITY, "table of %llu rows exceeds capacity %llu", (unsigned long long)n,
                    (unsigned long long)h->table_cap);
    h->n_unique = 0;
    if (n) {
        const uint32_t tb = 256;
        k_make_keys<<<(uint32_t)((n + tb - 1) / tb), tb, 0, s>>>(src, n, h->d_keys[0], h->d_idx[0]);
        LAUNCH_OK(h);
        const uint32_t nblocks = (uint32_t)((n + SORT_TILE - 1) / SORT_TILE);
        int cur = 0;
        for (int pass = 0; pass < SORT_KEY_BITS / 8; pass++) {
            const int shift = 64 - SORT_KEY_BITS + pass * 8;
            k_radix_hist<<<nblocks, SORT_THREADS, 0, s>>>(h->d_keys[cur], n, shift, h->d_hist, nblocks);
            LAUNCH_OK(h);
            int rc = scan_u32(h, h->d_hist, h->d_hist, (uint64_t)256 * nblocks, s);
            if (rc)
                return rc;
            k_radix_scatter<<<nblocks, SORT_THREADS, 0, s>>>(h->d_keys[cur], h->d_idx[cur], n, shift, h->d_hist,
                                                             nblocks, h->d_keys[cur ^ 1], h->d_idx[cur ^ 1]);
            LAUNCH_OK(h);
            cur ^= 1;
        }
        k_gather_digests<<<(uint32_t)((2 * n + tb - 1) / tb), tb, 0, s>>>(src, h->d_idx[cur], n, h->d_sorted);
        LAUNCH_OK(h);
        // long runs (duplicates) are listed in the idle flag buffer and handled by whole CTAs
        uint2 *long_runs = reinterpret_cast<uint2 *>(h->d_hist); // sized for FIX_LONG_CAP entries in alloc_table_buffers
        uint32_t *n_long = h->d_pos;
        CK(h, cudaMemsetAsync(n_long, 0, 4, s));
        k_fix_ties<<<(uint32_t)((n + tb - 1) / tb), tb, 0, s>>>(h->d_keys[cur], n, h->d_sorted, 64 - SORT_KEY_BITS, long_runs, n_long);
        LAUNCH_OK(h);
        k_fix_long_runs<<<h->sm_count, 256, 0, s>>>(h->d_sorted, long_runs, n_long);
        LAUNCH_OK(h);
        k_unique_flags<<<(uint32_t)((n + tb - 1) / tb), tb, 0, s>>>(h->d_sorted, n, h->d_flags);
        LAUNCH_OK(h);
        int rc = scan_u32(h, h->d_flags, h->d_pos, n, s);
        if (rc)
            return rc;
        k_compact_digests<<<(uint32_t)((2 * n + tb - 1) / tb), tb, 0, s>>>(h->d_sorted, h->d_flags, h->d_pos, n,
                                                                            h->d_table);
        LAUNCH_OK(h);
        uint32_t last_pos = 0, last_flag = 0;
        CK(h, cudaMemcpyAsync(&last_pos, h->d_pos + (n - 1), 4, cudaMemcpyDeviceToHost, s));
        CK(h, cudaMemcpyAsync(&last_flag, h->d_flags + (n - 1), 4, cudaMemcpyDeviceToHost, s));
        CK(h, cudaStreamSynchronize(s));
        h->n_unique = (uint64_t)last_pos + last_flag;
    }
    return 0;
}

// hash level after level (groups of 256 digests = 8 KiB) starting from `cur_n` digests at `cur`; always at least once
int merkle_from(mksnap *h, const uint8_t *cur, uint64_t cur_n, cudaStream_t s)
{
    int which = 0;
    for (;;) {
        const uint64_t next_n = cur_n == 0 ? 1 : (cur_n + 255) / 256;
        // a Merkle group is one 8 KiB serial SHA-256: the warp-pair stream kernel (next block prefetched, rounds and
        // schedule on separate warps) does a level in ~0.14 ms where one lane per group of the chunk kernel, waiting
        // for its un-prefetched loads with a handful of warps per SM, took ~0.8 ms
        CK(h, cudaMemsetAsync(&h->d_sc->work, 0, 4, s));
        k_sha256_streams<<<(uint32_t)std::min<uint64_t>((next_n + 31) / 32, (uint64_t)h->sm_count * 4), SS_THREADS, 0, s>>>(
            cur, nullptr, nullptr, (uint32_t)next_n, nullptr, nullptr, nullptr, h->d_merkle[which], &h->d_sc->work, 32u, 1u, 8192,
            cur_n * 32);
        LAUNCH_OK(h);
        cur = h->d_merkle[which];
        cur_n = next_n;
        which ^= 1;
        if (cur_n == 1)
            break;
    }
    CK(h, cudaMemcpyAsync(h->root, cur, 32, cudaMemcpyDeviceToHost, s));
    h->stats.d2h_bytes += 32;
    return 0;
}
int merkle_root(mksnap *h, cudaStream_t s) { return merkle_from(h, h->d_table, h->n_unique, s); } // level 0 = table

} // namespace

// ---------------------------------------------------------------------------
extern "C" {

int mksnap_abi_version(void) { return MKSNAP_ABI_VERSION; }

void mksnap_default_cdc(mksnap_cdc_params *p)
{
    p->min_size = 4096;
    p->normal_size = 16384;
    p->max_size = 131072;
    p->strict_bits = 16;
    p->loose_bits = 12;
}

uint32_t mksnap_roll_multiplier(void) { return ROLL_MULT; }

const char *mksnap_last_error(const mksnap_t *h) { return h ? h->err.c_str() : g_create_error.c_str(); }

} // extern "C" (helpers below are C++)

// cuTensorMapEncodeTiled through the runtime's driver entry point (no -lcuda link dependency)
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int make_row_map(mksnap *h, EncodeTiledFn enc, CUtensorMap *out, void *base, uint64_t n_rows, uint32_t box_rows)
{
    const cuuint64_t dims[2] = {128, n_rows};
    const cuuint64_t strides[1] = {128};
    const cuuint32_t box[2] = {128, box_rows};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
        return fail(h, MKSNAP_E_CUDA, "cuTensorMapEncodeTiled failed (%d) rows=%llu box=%u", (int)r,
                    (unsigned long long)n_rows, box_rows);
    return 0;
}

// (re)allocate everything whose size follows the number of table rows: radix keys/payload, sorted and unique
// tables, flags/positions, histograms, Merkle levels, scan temporaries.  Called at create (rows = max_chunks)
// and again by mksnap_comm_init (rows = max_chunks x ranks: every rank merges the union of all tables).
static int alloc_table_buffers(mksnap *h, uint64_t rows)
{
    for (int k = 0; k < 2; k++) {
        cudaFree(h->d_keys[k]); cudaFree(h->d_idx[k]); cudaFree(h->d_merkle[k]);
        h->d_keys[k] = nullptr; h->d_idx[k] = nullptr; h->d_merkle[k] = nullptr;
    }
    cudaFree(h->d_sorted); cudaFree(h->d_table); cudaFree(h->d_flags); cudaFree(h->d_pos); cudaFree(h->d_hist);
    cudaFree(h->d_scan_tmp);
    h->d_sorted = h->d_table = nullptr;
    h->d_flags = h->d_pos = h->d_hist = h->d_scan_tmp = nullptr;
    h->table_cap = 0;
    for (int k = 0; k < 2; k++) {
        CK(h, cudaMalloc(&h->d_keys[k], rows * 8));
        CK(h, cudaMalloc(&h->d_idx[k], rows * 4));
    }
    CK(h, cudaMalloc(&h->d_sorted, rows * 32));
    CK(h, cudaMalloc(&h->d_table, rows * 32));
    CK(h, cudaMalloc(&h->d_flags, rows * 4));
    CK(h, cudaMalloc(&h->d_pos, rows * 4));
    const uint64_t hist_words = std::max<uint64_t>(256ull * ((rows + SORT_TILE - 1) / SORT_TILE + 1), 2ull * FIX_LONG_CAP + 64); // also holds k_fix_ties' long-run list
    CK(h, cudaMalloc(&h->d_hist, hist_words * 4));
    const uint64_t merkle_rows = rows / 256 + 2;
    CK(h, cudaMalloc(&h->d_merkle[0], merkle_rows * 32));
    CK(h, cudaMalloc(&h->d_merkle[1], (merkle_rows / 256 + 2) * 32));
    h->scan_tmp_words = std::max(rows, std::max<uint64_t>(hist_words, h->cfg.max_extents)) / SCAN_ITEMS * 2 + 4096;
    CK(h, cudaMalloc(&h->d_scan_tmp, h->scan_tmp_words * 4));
    h->table_cap = rows;
    return 0;
}

template <int GROUPS, int TW, int ST> static int launch_scan(mksnap *h, uint32_t slot, uint32_t n_regions, cudaStream_t sk)
{
    using Cfg = ScanCfg<GROUPS, TW, ST>;
    const uint32_t n_tiles = (n_regions + Cfg::TILE_WARPS - 1) / Cfg::TILE_WARPS;
    const uint32_t grid = std::min<uint32_t>(n_tiles, (uint32_t)h->sm_count);
    k_roll_scan<GROUPS, TW, ST><<<grid, Cfg::THREADS, Cfg::SMEM, sk>>>(h->tm_main[slot], n_tiles, h->prm.strict_lim, h->prm.loose_lim,
                                                                     h->d_tiles, h->d_pool, h->pool_cap, h->d_pool_count, &h->d_sc->err);
    LAUNCH_OK(h);
    return 0;
}

// the k_roll_scan shapes that are compiled in: {groups, warps per tile, stages}; MKSNAP_SCAN_CFG picks one (0 = default)
struct ScanShape {
    int groups, tile_warps, stages;
};
#define MK_SCAN_SHAPES(X) X(0, 4, 6, 8) X(1, 3, 6, 8) X(2, 2, 6, 8) X(3, 4, 4, 12) X(4, 3, 4, 12) X(5, 2, 4, 12) X(6, 3, 7, 7) X(7, 2, 7, 7) \
    X(8, 4, 3, 16) X(9, 6, 4, 12) X(10, 4, 7, 7) X(11, 5, 5, 9)
#define MK_SHAPE_ROW(I, G, T, S) {G, T, S},
static const ScanShape SCAN_SHAPES[] = {MK_SCAN_SHAPES(MK_SHAPE_ROW)};
#undef MK_SHAPE_ROW
constexpr int N_SCAN_SHAPES = (int)(sizeof(SCAN_SHAPES) / sizeof(SCAN_SHAPES[0]));

static int launch_scan_cfg(mksnap *h, uint32_t slot, uint32_t n_regions, cudaStream_t sk)
{
    switch (h->scan_cfg) {
#define MK_SHAPE_CASE(I, G, T, S) \
    case I: return launch_scan<G, T, S>(h, slot, n_regions, sk);
        MK_SCAN_SHAPES(MK_SHAPE_CASE)
#undef MK_SHAPE_CASE
    default: return launch_scan<4, 6, 8>(h, slot, n_regions, sk);
    }
}

extern "C" {

static int create_impl(mksnap *h)
{
    const mksnap_config &c = h->cfg;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(h, MKSNAP_E_CUDA, "no CUDA device usable (%s); libmksnap has no CPU fallback",
                    e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    if (c.device < 0 || c.device >= ndev)
        return fail(h, MKSNAP_E_INVAL, "device %d out of range [0,%d)", c.device, ndev);
    CK(h, cudaSetDevice(c.device));
    cudaDeviceProp prop;
    CK(h, cudaGetDeviceProperties(&prop, c.device));
    if (prop.major != 10)
        return fail(h, MKSNAP_E_CUDA, "device %d is sm_%d%d; libmksnap is built for sm_100a only", c.device,
                    prop.major, prop.minor);
    h->sm_count = prop.multiProcessorCount;
    CK(h, cudaStreamCreateWithFlags(&h->s_comp, cudaStreamNonBlocking));
    CK(h, cudaStreamCreateWithFlags(&h->s_copy, cudaStreamNonBlocking));

    h->n_slots = c.n_device_slots ? c.n_device_slots : (c.n_host_arenas ? 2u : 1u);
    if (h->n_slots > MAX_SLOTS)
        return fail(h, MKSNAP_E_INVAL, "n_device_slots > %u", MAX_SLOTS);
    for (uint32_t s = 0; s < h->n_slots; s++) {
        CK(h, cudaMalloc(&h->d_slot[s], c.device_arena_bytes + SLOT_SLACK));
        CK(h, cudaMemsetAsync(h->d_slot[s] + c.device_arena_bytes, 0, SLOT_SLACK, h->s_comp));
        CK(h, cudaEventCreateWithFlags(&h->ev_slot_free[s], cudaEventDisableTiming));
    }
    h->arenas.resize(c.n_host_arenas);
    for (auto &a : h->arenas) {
        CK(h, cudaHostAlloc(&a.ptr, c.host_arena_bytes, cudaHostAllocDefault));
        CK(h, cudaEventCreateWithFlags(&a.ev_h2d, cudaEventDisableTiming));
    }
    const uint64_t mx = c.max_extents;
    h->meta.resize(std::max<uint32_t>(2, h->n_slots));
    for (auto &m : h->meta) {
        CK(h, cudaHostAlloc(&m.h_crc, mx * sizeof(CrcExtent), cudaHostAllocDefault));
        CK(h, cudaHostAlloc(&m.h_piece_base, (mx + 1) * 4, cudaHostAllocDefault));
        CK(h, cudaHostAlloc(&m.h_files, mx * sizeof(CdcFile), cudaHostAllocDefault));
        CK(h, cudaHostAlloc(&m.h_rstart, mx * 8, cudaHostAllocDefault));
        CK(h, cudaHostAlloc(&m.h_rlen, mx * 8, cudaHostAllocDefault));
        CK(h, cudaHostAlloc(&m.h_rstream, mx * 4, cudaHostAllocDefault));
        CK(h, cudaHostAlloc(&m.h_rflags, mx * 4, cudaHostAllocDefault));
        CK(h, cudaMalloc(&m.d_crc, mx * sizeof(CrcExtent)));
        CK(h, cudaMalloc(&m.d_piece_base, (mx + 1) * 4));
        CK(h, cudaMalloc(&m.d_ext_pure, mx * 4));
        CK(h, cudaMalloc(&m.d_files, mx * sizeof(CdcFile)));
        CK(h, cudaMalloc(&m.d_rstart, mx * 8));
        CK(h, cudaMalloc(&m.d_rlen, mx * 8));
        CK(h, cudaMalloc(&m.d_rstream, mx * 4));
        CK(h, cudaMalloc(&m.d_rflags, mx * 4));
        CK(h, cudaEventCreateWithFlags(&m.ev_done, cudaEventDisableTiming));
    }

    CrcConsts *hc = new CrcConsts;
    build_crc_consts(hc);
    CK(h, cudaMalloc(&h->d_consts, sizeof(CrcConsts)));
    CK(h, cudaMemcpy(h->d_consts, hc, sizeof(CrcConsts), cudaMemcpyHostToDevice));
    delete hc;
    CK(h, cudaMalloc(&h->d_sc, sizeof(SessionCounters)));
    CK(h, cudaMemset(h->d_sc, 0, sizeof(SessionCounters)));
    CK(h, cudaHostAlloc(&h->h_sc, sizeof(SessionCounters), cudaHostAllocDefault));

    const uint64_t n_tiles = c.device_arena_bytes / SCAN_TILE + 128; // one TileRec per 4 KiB region (+ tile round-up)
    CK(h, cudaMalloc(&h->d_tiles, n_tiles * sizeof(TileRec)));
    {
        EncodeTiledFn enc = nullptr;
        cudaDriverEntryPointQueryResult qres;
        CK(h, cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", (void **)&enc, cudaEnableDefault, &qres));
        if (!enc || qres != cudaDriverEntryPointSuccess)
            return fail(h, MKSNAP_E_CUDA, "cuTensorMapEncodeTiled entry point unavailable");
        const char *e = getenv("MKSNAP_SCAN_CFG"); // tuning knob: index into SCAN_SHAPES (0 = default)
        if (e && e[0] >= '0' && e[0] <= '9' && atoi(e) < N_SCAN_SHAPES)
            h->scan_cfg = atoi(e);
        const uint64_t n_rows = (c.device_arena_bytes + SLOT_SLACK) / 128;
        const uint32_t box_rows = (uint32_t)SCAN_SHAPES[h->scan_cfg].tile_warps * 32u + 1u; // the row above the tile travels with it
        for (uint32_t s = 0; s < h->n_slots; s++) {
            int rc;
            if ((rc = make_row_map(h, enc, &h->tm_main[s], h->d_slot[s], n_rows, box_rows)))
                return rc;
        }
#define MK_SET_SMEM(I, G, T, S) \
    CK(h, cudaFuncSetAttribute(k_roll_scan<G, T, S>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ScanCfg<G, T, S>::SMEM));
        MK_SCAN_SHAPES(MK_SET_SMEM)
#undef MK_SET_SMEM
        const char *e2 = getenv("MKSNAP_SHA_FMA"); // tuning knob: 0 = plain adds in the chunk SHA-256 kernel
        if (e2 && e2[0] == '0')
            h->sha_fma = false;
        const char *e3 = getenv("MKSNAP_SHA_ORDER"); // tuning knob: 0 = hash chunks in file order instead of longest first
        if (e3 && e3[0] == '0')
            h->sha_order = false;
    }
    // expected candidates = bytes >> loose_bits; 8x headroom (32x at the default 12 bits would be wasteful for
    // dense parameter sets), plus one private block per resident scan warp (x2)
    uint64_t pc = std::max<uint64_t>(1u << 20, (c.device_arena_bytes >> h->cfg.cdc.loose_bits) * 8) +
                  2ull * h->sm_count * 32 * SCAN_POOL_BLOCK;
    if (pc > 0xFFFFFFF0ull)
        pc = 0xFFFFFFF0ull;
    h->pool_cap = (uint32_t)pc;
    CK(h, cudaMalloc(&h->d_pool, (uint64_t)h->pool_cap * 4));
    CK(h, cudaMalloc(&h->d_pool_count, 4));
    h->crc_session_cap = std::max<uint64_t>(4 * mx, 1ull << 20);
    CK(h, cudaMalloc(&h->d_crc_session, h->crc_session_cap * 4));
    h->carry_cap = ((uint64_t)h->prm.max_size + 511) / 512 * 512;
    CK(h, cudaMalloc(&h->d_carry, h->carry_cap));
    CK(h, cudaMalloc(&h->d_counts, mx * 4));
    CK(h, cudaMalloc(&h->d_bases, mx * 4));

    // default: every byte in min-size chunks, plus per file the end-of-file chunk and the two spare cut-list slots of the big-file path
    h->max_chunks = c.max_chunks ? c.max_chunks : c.device_arena_bytes / h->prm.min_size + 3 * mx + 64;
    const uint64_t mc = h->max_chunks;
    CK(h, cudaMalloc(&h->d_chunk_start, mc * 8));
    CK(h, cudaMalloc(&h->d_chunk_len, mc * 8));
    CK(h, cudaMalloc(&h->d_order, mc * 4));
    CK(h, cudaMalloc(&h->d_chunk_end, mc * 8));
    CK(h, cudaMalloc(&h->d_digests, mc * 32));
    h->max_streams = mx;
    CK(h, cudaMalloc(&h->d_stream_digests, h->max_streams * 32));
    CK(h, cudaMalloc(&h->d_stream_state, h->max_streams * sizeof(StreamState)));
    CK(h, cudaMemset(h->d_stream_state, 0, h->max_streams * sizeof(StreamState)));
    h->stream_stamp.assign(h->max_streams, 0);

    {
        int rc = alloc_table_buffers(h, mc);
        if (rc)
            return rc;
    }

    for (int i = 0; i < N_EV; i++)
        CK(h, cudaEventCreate(&h->ev[i]));
    for (int i = 0; i < 4; i++)
        CK(h, cudaEventCreate(&h->ev_fin[i]));
    CK(h, cudaEventCreate(&h->ev_copy0));
    CK(h, cudaEventCreate(&h->ev_copy1));
    CK(h, cudaEventCreateWithFlags(&h->ev_copy_done, cudaEventDisableTiming));
    CK(h, cudaFuncSetAttribute(k_crc32_extents, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CRC_SMEM));
    CK(h, cudaFuncSetAttribute(k_select_cuts_big, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SELB_SMEM));
    CK(h, cudaStreamSynchronize(h->s_comp));
    memset(&h->stats, 0, sizeof h->stats);
    return 0;
}

int mksnap_create(const mksnap_config *cfg, mksnap_t **out)
{
    if (!cfg || !out)
        return fail(nullptr, MKSNAP_E_INVAL, "null argument");
    *out = nullptr;
    mksnap *h = new mksnap;
    h->cfg = *cfg;
    mksnap_cdc_params p = cfg->cdc;
    if (p.min_size == 0 && p.max_size == 0)
        mksnap_default_cdc(&p);
    h->cfg.cdc = p;
    if (p.min_size < 64 || p.normal_size < p.min_size || p.max_size < p.normal_size || p.strict_bits < p.loose_bits ||
        p.strict_bits > 31 || p.loose_bits < 1) {
        g_create_error = "invalid cdc parameters";
        delete h;
        return MKSNAP_E_INVAL;
    }
    h->prm.min_size = p.min_size;
    h->prm.normal_size = p.normal_size;
    h->prm.max_size = p.max_size;
    h->prm.strict_lim = 1u << (32 - p.strict_bits);
    h->prm.loose_lim = 1u << (32 - p.loose_bits);
    if (cfg->device_arena_bytes == 0 || cfg->device_arena_bytes % 512 || cfg->max_extents == 0 ||
        (cfg->n_host_arenas && (cfg->host_arena_bytes == 0 || cfg->host_arena_bytes > cfg->device_arena_bytes))) {
        g_create_error = "invalid arena configuration (sizes must be non-zero, device arena multiple of 512, host arena <= device arena)";
        delete h;
        return MKSNAP_E_INVAL;
    }
    int rc = create_impl(h);
    if (rc) {
        g_create_error = h->err;
        mksnap_destroy(h);
        return rc;
    }
    *out = h;
    return 0;
}

void mksnap_destroy(mksnap_t *h)
{
    if (!h)
        return;
    cudaSetDevice(h->cfg.device);
    cudaDeviceSynchronize();
    if (h->comm && h->nccl.CommDestroy)
        h->nccl.CommDestroy(h->comm);
    for (uint32_t s = 0; s < MAX_SLOTS; s++) {
        cudaFree(h->d_slot[s]);
        if (h->ev_slot_free[s])
            cudaEventDestroy(h->ev_slot_free[s]);
    }
    for (auto &a : h->arenas) {
        cudaFreeHost(a.ptr);
        if (a.ev_h2d)
            cudaEventDestroy(a.ev_h2d);
    }
    for (auto &m : h->meta) {
        cudaFreeHost(m.h_crc); cudaFreeHost(m.h_piece_base); cudaFreeHost(m.h_files);
        cudaFreeHost(m.h_rstart); cudaFreeHost(m.h_rlen); cudaFreeHost(m.h_rstream); cudaFreeHost(m.h_rflags);
        cudaFree(m.d_rstream); cudaFree(m.d_rflags);
        cudaFree(m.d_ext_pure);
        cudaFree(m.d_crc); cudaFree(m.d_piece_base); cudaFree(m.d_files); cudaFree(m.d_rstart); cudaFree(m.d_rlen);
        if (m.ev_done)
            cudaEventDestroy(m.ev_done);
    }
    cudaFree(h->d_consts); cudaFree(h->d_sc); cudaFreeHost(h->h_sc);
    cudaFree(h->d_carry);
    cudaFree(h->d_crc_session);
    cudaFree(h->d_tiles); cudaFree(h->d_pool); cudaFree(h->d_pool_count); cudaFree(h->d_counts); cudaFree(h->d_bases);
    cudaFree(h->d_scan_tmp);
    cudaFree(h->d_order); cudaFree(h->d_chunk_start); cudaFree(h->d_chunk_len); cudaFree(h->d_chunk_end); cudaFree(h->d_digests);
    cudaFree(h->d_stream_digests); cudaFree(h->d_stream_state);
    for (int k = 0; k < 2; k++) {
        cudaFree(h->d_keys[k]); cudaFree(h->d_idx[k]); cudaFree(h->d_merkle[k]);
    }
    cudaFree(h->d_sorted); cudaFree(h->d_table); cudaFree(h->d_flags); cudaFree(h->d_pos); cudaFree(h->d_hist);
    cudaFree(h->d_gather); cudaFree(h->d_gcount); cudaFree(h->d_concat);
    cudaFree(h->d_xbounds); cudaFree(h->d_xhdr); cudaFree(h->d_xrec); cudaFree(h->d_xtail);
    cudaFree(h->d_dfirst); cudaFree(h->d_duidx); cudaFree(h->d_ddir); cudaFree(h->d_dstatus); cudaFree(h->d_dcnt);
    for (int i = 0; i < 2; i++)
        if (h->ev_delta[i])
            cudaEventDestroy(h->ev_delta[i]);
    if (h->s_comp) cudaStreamDestroy(h->s_comp);
    if (h->s_copy) cudaStreamDestroy(h->s_copy);
    delete h;
}

int mksnap_begin(mksnap_t *h)
{
    if (!h)
        return MKSNAP_E_INVAL;
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaStreamSynchronize(h->s_comp));
    CK(h, cudaMemsetAsync(h->d_sc, 0, sizeof(SessionCounters), h->s_comp));
    CK(h, cudaMemsetAsync(h->d_stream_state, 0, h->max_streams * sizeof(StreamState), h->s_comp));
    for (auto &a : h->arenas) // an arena acquired but never submitted (a packer that failed half way) is reclaimed here
        a.acquired = false;
    h->n_streams = 0;
    h->stream_base = 0;
    h->crc_bytes = 0;
    h->crc_session_n = 0;
    h->crc_host_acc = 0;
    h->crc_host_bytes = 0;
    h->open_file = false;
    h->n_unique = 0;
    h->finished = false;
    h->table_own = false;
    h->delta_done = false;
    h->in_session = true;
    return 0;
}

int mksnap_arena_acquire(mksnap_t *h, void **host_ptr, uint64_t *capacity, int32_t *arena_id)
{
    if (!h || !host_ptr || !capacity || !arena_id)
        return MKSNAP_E_INVAL;
    if (h->arenas.empty())
        return fail(h, MKSNAP_E_STATE, "handle was created with n_host_arenas = 0");
    CK(h, cudaSetDevice(h->cfg.device));
    const uint32_t n = (uint32_t)h->arenas.size();
    for (uint32_t k = 0; k < n; k++) {
        uint32_t i = (h->next_arena + k) % n;
        HostArena &a = h->arenas[i];
        if (a.acquired)
            continue;
        if (a.in_flight) {
            CK(h, cudaEventSynchronize(a.ev_h2d));
            a.in_flight = false;
        }
        a.acquired = true;
        h->next_arena = (i + 1) % n;
        *host_ptr = a.ptr;
        *capacity = h->cfg.host_arena_bytes;
        *arena_id = (int32_t)i;
        return 0;
    }
    return fail(h, MKSNAP_E_STATE, "all %u host arenas are acquired and not yet submitted", n);
}

int mksnap_arena_release(mksnap_t *h, int32_t arena_id)
{
    if (!h)
        return MKSNAP_E_INVAL;
    if (arena_id < 0 || (size_t)arena_id >= h->arenas.size() || !h->arenas[arena_id].acquired)
        return fail(h, MKSNAP_E_STATE, "arena %d was not acquired", arena_id);
    h->arenas[arena_id].acquired = false;
    return 0;
}

int mksnap_get_limits(const mksnap_t *h, mksnap_limits *out)
{
    if (!h || !out)
        return MKSNAP_E_INVAL;
    out->max_extents = h->cfg.max_extents;
    out->max_streams = h->max_streams;
    out->max_chunks = h->max_chunks;
    out->host_arena_bytes = h->cfg.host_arena_bytes;
    out->device_arena_bytes = h->cfg.device_arena_bytes;
    out->n_host_arenas = (uint32_t)h->arenas.size();
    out->n_device_slots = h->n_slots;
    out->carry_bytes = h->carry_cap;
    return 0;
}

static int submit_common(mksnap *h, uint32_t slot, uint64_t used, const mksnap_extent *ext, uint64_t n_ext,
                         const mksnap_range *rng, uint64_t n_rng, HostArena *src)
{
    if (!h->in_session || h->finished)
        return fail(h, MKSNAP_E_STATE, "submit outside begin/finish");
    if (used > h->cfg.device_arena_bytes)
        return fail(h, MKSNAP_E_CAPACITY, "used %llu > device arena %llu", (unsigned long long)used,
                    (unsigned long long)h->cfg.device_arena_bytes);
    if (n_ext > h->cfg.max_extents || n_rng > h->cfg.max_extents)
        return fail(h, MKSNAP_E_CAPACITY, "too many extents/ranges (%llu/%llu > %llu)", (unsigned long long)n_ext,
                    (unsigned long long)n_rng, (unsigned long long)h->cfg.max_extents);

    MetaSet &m = h->meta[h->submit_idx % h->meta.size()];
    if (m.in_flight) {
        CK(h, cudaEventSynchronize(m.ev_done));
        m.in_flight = false;
    }
    uint64_t n_crc = 0, n_files = 0, pieces = 0, cdc_bytes = 0, crc_bytes = 0, big_slots = 0, cont_off = 0;
    bool have_cont = false, have_more = false;
    for (uint64_t i = 0; i < n_ext; i++) {
        const mksnap_extent &x = ext[i];
        if ((x.arena_off & 15) || x.arena_off > used || x.len > used - x.arena_off)
            return fail(h, MKSNAP_E_INVAL, "extent %llu out of bounds or not 16-byte aligned", (unsigned long long)i);
        if (x.flags & MKSNAP_X_CRC) {
            m.h_crc[n_crc].off = x.arena_off;
            m.h_crc[n_crc].len = x.len;
            m.h_crc[n_crc].suffix = x.crc_suffix;
            m.h_piece_base[n_crc] = (uint32_t)pieces;
            pieces += (x.len + CRC_PIECE - 1) / CRC_PIECE;
            if (pieces > 0xFFFFFFF0ull)
                return fail(h, MKSNAP_E_CAPACITY, "too many CRC pieces");
            crc_bytes += x.len;
            n_crc++;
        }
        if (x.flags & MKSNAP_X_CDC) {
            const bool cont = (x.flags & MKSNAP_X_CONT) != 0, more = (x.flags & MKSNAP_X_MORE) != 0;
            if (cont) {
                if (n_files != 0 || !h->open_file)
                    return fail(h, MKSNAP_E_STATE, "extent %llu: MKSNAP_X_CONT must be the first CDC extent of the submit that follows a MKSNAP_X_MORE extent",
                                (unsigned long long)i);
                if (x.arena_off < h->carry_cap)
                    return fail(h, MKSNAP_E_INVAL, "extent %llu: a continuation starts at arena offset >= %llu (room for the open chunk)",
                                (unsigned long long)i, (unsigned long long)h->carry_cap);
                have_cont = true;
                cont_off = x.arena_off;
            }
            if (have_more)
                return fail(h, MKSNAP_E_INVAL, "extent %llu: a MKSNAP_X_MORE extent must be the last CDC extent of its submit", (unsigned long long)i);
            if (more) {
                if (x.len == 0 || x.reserved == 0)
                    return fail(h, MKSNAP_E_INVAL, "extent %llu: MKSNAP_X_MORE needs a non-empty piece and the bytes that follow in `reserved`",
                                (unsigned long long)i);
                have_more = true;
            }
            m.h_files[n_files].off = x.arena_off;
            m.h_files[n_files].len = x.len;
            m.h_files[n_files].scratch = big_slots;
            m.h_files[n_files].more_after = more ? x.reserved : 0u;
            m.h_files[n_files].cont = cont ? 1u : 0u;
            if (x.len + (cont ? h->carry_cap : 0) >= SELECT_BIG_FILE) // a continuation is widened by its open chunk on the device
                big_slots += (x.len + (cont ? h->carry_cap : 0)) / h->prm.min_size + 2;
            cdc_bytes += x.len;
            n_files++;
        } else if (x.flags & (MKSNAP_X_MORE | MKSNAP_X_CONT)) {
            return fail(h, MKSNAP_E_INVAL, "extent %llu: MKSNAP_X_MORE / MKSNAP_X_CONT apply to MKSNAP_X_CDC extents", (unsigned long long)i);
        }
    }
    m.h_piece_base[n_crc] = (uint32_t)pieces;
    if (h->open_file && !have_cont)
        return fail(h, MKSNAP_E_STATE, "the previous submit left a file open (MKSNAP_X_MORE): this one must start with its MKSNAP_X_CONT extent");
    if (big_slots > h->table_cap) // the cut lists of the big files live in the (idle) radix key buffer
        return fail(h, MKSNAP_E_CAPACITY, "big-file cut lists need %llu slots, max_chunks allows %llu",
                    (unsigned long long)big_slots, (unsigned long long)h->table_cap);
    if (++h->stamp_epoch == 0) { // epoch wrapped: forget every stamp
        std::fill(h->stream_stamp.begin(), h->stream_stamp.end(), 0);
        h->stamp_epoch = 1;
    }
    for (uint64_t i = 0; i < n_rng; i++) {
        if ((rng[i].arena_off & 15) || rng[i].arena_off > used || rng[i].len > used - rng[i].arena_off)
            return fail(h, MKSNAP_E_INVAL, "range %llu out of bounds or not 16-byte aligned", (unsigned long long)i);
        if (rng[i].stream >= h->max_streams)
            return fail(h, MKSNAP_E_CAPACITY, "range %llu: stream slot %u >= %llu", (unsigned long long)i, rng[i].stream,
                        (unsigned long long)h->max_streams);
        if ((rng[i].flags & MKSNAP_R_MORE) && (rng[i].len == 0 || rng[i].len % 64))
            return fail(h, MKSNAP_E_INVAL, "range %llu: a piece with MKSNAP_R_MORE must be a non-empty multiple of 64 bytes",
                        (unsigned long long)i);
        if (h->stream_stamp[rng[i].stream] == h->stamp_epoch)
            return fail(h, MKSNAP_E_INVAL, "range %llu: stream slot %u already has a piece in this submit (one piece per stream per submit)",
                        (unsigned long long)i, rng[i].stream);
        h->stream_stamp[rng[i].stream] = h->stamp_epoch;
        m.h_rstart[i] = rng[i].arena_off;
        m.h_rlen[i] = rng[i].len;
        m.h_rstream[i] = rng[i].stream;
        m.h_rflags[i] = rng[i].flags;
    }

    uint8_t *d_arena = h->d_slot[slot];
    // ---- copy stream: arena + tables ----
    cudaStream_t sc = h->s_copy, sk = h->s_comp;
    if (h->slot_used[slot])
        CK(h, cudaStreamWaitEvent(sc, h->ev_slot_free[slot], 0));
    if (src) {
        CK(h, cudaEventRecord(h->ev_copy0, sc));
        CK(h, cudaMemcpyAsync(d_arena, src->ptr, used, cudaMemcpyHostToDevice, sc));
        // zero the tail up to the next 512 so row-granular readers see zeros
        const uint64_t padded = std::min<uint64_t>((used + 511) & ~511ull, h->cfg.device_arena_bytes);
        if (padded > used)
            CK(h, cudaMemsetAsync(d_arena + used, 0, padded - used, sc));
        CK(h, cudaEventRecord(h->ev_copy1, sc));
        CK(h, cudaEventRecord(src->ev_h2d, sc));
        src->in_flight = true;
        src->acquired = false;
        h->stats.h2d_bytes += used;
        h->have_h2d_time = true;
    }
    if (n_crc) {
        CK(h, cudaMemcpyAsync(m.d_crc, m.h_crc, n_crc * sizeof(CrcExtent), cudaMemcpyHostToDevice, sc));
        CK(h, cudaMemcpyAsync(m.d_piece_base, m.h_piece_base, (n_crc + 1) * 4, cudaMemcpyHostToDevice, sc));
    }
    if (n_files)
        CK(h, cudaMemcpyAsync(m.d_files, m.h_files, n_files * sizeof(CdcFile), cudaMemcpyHostToDevice, sc));
    if (n_rng) {
        CK(h, cudaMemcpyAsync(m.d_rstart, m.h_rstart, n_rng * 8, cudaMemcpyHostToDevice, sc));
        CK(h, cudaMemcpyAsync(m.d_rlen, m.h_rlen, n_rng * 8, cudaMemcpyHostToDevice, sc));
        CK(h, cudaMemcpyAsync(m.d_rstream, m.h_rstream, n_rng * 4, cudaMemcpyHostToDevice, sc));
        CK(h, cudaMemcpyAsync(m.d_rflags, m.h_rflags, n_rng * 4, cudaMemcpyHostToDevice, sc));
    }
    h->stats.h2d_bytes += n_crc * sizeof(CrcExtent) + (n_crc ? (n_crc + 1) * 4 : 0) + n_files * sizeof(CdcFile) + n_rng * 16;
    CK(h, cudaEventRecord(h->ev_copy_done, sc));

    // ---- compute stream ----
    CK(h, cudaStreamWaitEvent(sk, h->ev_copy_done, 0));
    if (have_cont) { // prepend the open chunk of the file that continues here (before anything scans the arena)
        k_carry_in<<<1, 256, 0, sk>>>(h->d_carry, d_arena, cont_off, m.d_files, 0u, h->d_sc);
        LAUNCH_OK(h);
    }
    CK(h, cudaEventRecord(h->ev[0], sk));
    if (n_crc && pieces) {
        const uint32_t grid = (uint32_t)std::min<uint64_t>(h->sm_count, (pieces + 31) / 32);
        CK(h, cudaMemsetAsync(m.d_ext_pure, 0, n_crc * 4, sk));
        k_crc32_extents<<<grid, CRC_THREADS, CRC_SMEM, sk>>>(d_arena, m.d_crc, m.d_piece_base, (uint32_t)n_crc,
                                                            (uint32_t)pieces, h->d_consts, m.d_ext_pure, &h->d_sc->crc_acc);
        LAUNCH_OK(h);
    }
    if (n_crc) { // pure(extent) of this submit's extents joins the session table (zero-length extents keep their slot)
        if (!pieces)
            CK(h, cudaMemsetAsync(m.d_ext_pure, 0, n_crc * 4, sk));
        if (h->crc_session_n < h->crc_session_cap)
            CK(h, cudaMemcpyAsync(h->d_crc_session + h->crc_session_n, m.d_ext_pure,
                                  std::min<uint64_t>(n_crc, h->crc_session_cap - h->crc_session_n) * 4, cudaMemcpyDeviceToDevice, sk));
        h->crc_session_n += n_crc;
    }
    CK(h, cudaEventRecord(h->ev[1], sk));
    if (n_files) {
        const uint32_t n_regions = (uint32_t)((used + SCAN_TILE - 1) / SCAN_TILE);
        CK(h, cudaMemsetAsync(h->d_pool_count, 0, 4, sk));
        int rc = launch_scan_cfg(h, slot, n_regions, sk);
        if (rc)
            return rc;
    }
    CK(h, cudaEventRecord(h->ev[2], sk));
    if (n_files) {
        const uint32_t nb = (uint32_t)((n_files + 127) / 128);
        k_select_cuts<0><<<nb, 128, 0, sk>>>(m.d_files, (uint32_t)n_files, h->prm, h->d_tiles, h->d_pool, h->d_counts,
                                             nullptr, h->d_sc, h->max_chunks, 0, nullptr, nullptr, nullptr);
        LAUNCH_OK(h);
        const bool big_files = big_slots != 0;
        if (big_files) {
            k_select_cuts_big<<<(uint32_t)n_files, SELB_THREADS, SELB_SMEM, sk>>>(m.d_files, (uint32_t)n_files, h->prm, h->d_tiles,
                                                                       h->d_pool, h->d_counts, h->d_keys[0], h->d_sc);
            LAUNCH_OK(h);
        }
        int rc = scan_u32(h, h->d_counts, h->d_bases, n_files, sk);
        if (rc)
            return rc;
        k_batch_begin<<<1, 64, 0, sk>>>(h->d_sc, h->d_counts, h->d_bases, (uint32_t)n_files, h->max_chunks, cdc_bytes, have_cont ? 1u : 0u);
        LAUNCH_OK(h);
        k_select_cuts<1><<<nb, 128, 0, sk>>>(m.d_files, (uint32_t)n_files, h->prm, h->d_tiles, h->d_pool, h->d_counts,
                                             h->d_bases, h->d_sc, h->max_chunks, h->stream_base, h->d_chunk_start,
                                             h->d_chunk_len, h->d_chunk_end);
        LAUNCH_OK(h);
        if (big_files) {
            k_expand_big_cuts<<<(uint32_t)n_files, 256, 0, sk>>>(m.d_files, (uint32_t)n_files, h->d_counts, h->d_bases,
                                                              h->d_keys[0], h->d_sc, h->max_chunks, h->stream_base,
                                                              h->d_chunk_start, h->d_chunk_len, h->d_chunk_end);
            LAUNCH_OK(h);
        }
    }
    CK(h, cudaEventRecord(h->ev[3], sk));
    if (n_files) {
        const uint32_t *order = nullptr;
        if (h->sha_order) { // longest chunks first (see k_len_order)
            k_len_hist<<<h->sm_count * 2, LEN_THREADS, 0, sk>>>(h->d_chunk_len, h->d_sc);
            LAUNCH_OK(h);
            k_len_order<<<h->sm_count * 2, LEN_THREADS, 0, sk>>>(h->d_chunk_len, h->d_sc, h->d_order);
            LAUNCH_OK(h);
            order = h->d_order;
        }
        if (h->sha_fma)
            k_sha256_ranges<true><<<sha_grid(h), SHA_THREADS, 0, sk>>>(d_arena, h->d_chunk_start, h->d_chunk_len,
                                                                      &h->d_sc->batch_chunks, 0, &h->d_sc->n_chunks, 0, 0,
                                                                      0, h->d_digests, &h->d_sc->work, &h->d_sc->err, 1u, nullptr, nullptr,
                                                                      nullptr, order);
        else
            k_sha256_ranges<false><<<sha_grid(h), SHA_THREADS, 0, sk>>>(d_arena, h->d_chunk_start, h->d_chunk_len,
                                                                       &h->d_sc->batch_chunks, 0, &h->d_sc->n_chunks, 0,
                                                                       0, 0, h->d_digests, &h->d_sc->work, &h->d_sc->err, 1u, nullptr, nullptr,
                                                                      nullptr, order);
        LAUNCH_OK(h);
        k_batch_end<<<1, 32, 0, sk>>>(h->d_sc);
        LAUNCH_OK(h);
        if (have_more) { // park the open chunk before this slot is recycled
            k_carry_out<<<1, 256, 0, sk>>>(d_arena, h->d_carry, h->carry_cap, h->d_sc);
            LAUNCH_OK(h);
        }
    }
    CK(h, cudaEventRecord(h->ev[4], sk));
    if (n_rng) {
        // K4: warp pairs, 32 streams each, spread one pair per SM first (a pair then owns its two sub-partitions)
        CK(h, cudaMemsetAsync(&h->d_sc->work, 0, 4, sk));
        const uint32_t pairs = (uint32_t)((n_rng + 31) / 32);
        k_sha256_streams<<<std::min<uint32_t>(pairs, (uint32_t)h->sm_count * 4), SS_THREADS, 0, sk>>>(
            d_arena, m.d_rstart, m.d_rlen, (uint32_t)n_rng, m.d_rstream, m.d_rflags, h->d_stream_state, h->d_stream_digests,
            &h->d_sc->work, 32u, 1u);
        LAUNCH_OK(h);
        CK(h, cudaMemsetAsync(&h->d_sc->work, 0, 4, sk));
    }
    CK(h, cudaEventRecord(h->ev[5], sk));
    CK(h, cudaEventRecord(h->ev_slot_free[slot], sk));
    CK(h, cudaEventRecord(m.ev_done, sk));
    m.in_flight = true;
    h->slot_used[slot] = true;
    h->have_submit_times = true;
    for (uint64_t i = 0; i < n_rng; i++)
        if (!(rng[i].flags & MKSNAP_R_MORE))
            h->n_streams = std::max<uint64_t>(h->n_streams, (uint64_t)rng[i].stream + 1);
    h->open_file = have_more;
    h->stream_base += used;
    h->crc_bytes += crc_bytes;
    h->submit_idx++;
    return 0;
}

int mksnap_arena_submit(mksnap_t *h, int32_t arena_id, uint64_t used, const mksnap_extent *extents,
                        uint64_t n_extents, const mksnap_range *ranges, uint64_t n_ranges)
{
    if (!h)
        return MKSNAP_E_INVAL;
    CK(h, cudaSetDevice(h->cfg.device));
    if (arena_id < 0 || (size_t)arena_id >= h->arenas.size() || !h->arenas[arena_id].acquired)
        return fail(h, MKSNAP_E_STATE, "arena %d was not acquired", arena_id);
    if (used > h->cfg.host_arena_bytes)
        return fail(h, MKSNAP_E_CAPACITY, "used %llu > host arena %llu", (unsigned long long)used,
                    (unsigned long long)h->cfg.host_arena_bytes);
    const uint32_t slot = (uint32_t)(h->submit_idx % h->n_slots);
    return submit_common(h, slot, used, extents, n_extents, ranges, n_ranges, &h->arenas[arena_id]);
}

int mksnap_device_arena(mksnap_t *h, uint32_t slot, void **device_ptr, uint64_t *capacity)
{
    if (!h || slot >= h->n_slots || !device_ptr || !capacity)
        return MKSNAP_E_INVAL;
    *device_ptr = h->d_slot[slot];
    *capacity = h->cfg.device_arena_bytes;
    return 0;
}

int mksnap_device_upload(mksnap_t *h, uint32_t slot, uint64_t dst_off, const void *src, uint64_t n)
{
    if (!h || slot >= h->n_slots || dst_off > h->cfg.device_arena_bytes || n > h->cfg.device_arena_bytes - dst_off)
        return MKSNAP_E_INVAL;
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaStreamSynchronize(h->s_comp));
    CK(h, cudaMemcpy(h->d_slot[slot] + dst_off, src, n, cudaMemcpyHostToDevice));
    h->stats.h2d_bytes += n;
    return 0;
}

int mksnap_device_download(mksnap_t *h, uint32_t slot, uint64_t src_off, void *dst, uint64_t n)
{
    if (!h || slot >= h->n_slots || src_off > h->cfg.device_arena_bytes || n > h->cfg.device_arena_bytes - src_off)
        return MKSNAP_E_INVAL;
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaStreamSynchronize(h->s_comp));
    CK(h, cudaMemcpy(dst, h->d_slot[slot] + src_off, n, cudaMemcpyDeviceToHost));
    h->stats.d2h_bytes += n;
    return 0;
}

int mksnap_device_submit(mksnap_t *h, uint32_t slot, uint64_t used, const mksnap_extent *extents, uint64_t n_extents,
                         const mksnap_range *ranges, uint64_t n_ranges)
{
    if (!h || slot >= h->n_slots)
        return MKSNAP_E_INVAL;
    CK(h, cudaSetDevice(h->cfg.device));
    return submit_common(h, slot, used, extents, n_extents, ranges, n_ranges, nullptr);
}

int mksnap_synth_fill(mksnap_t *h, uint32_t slot, uint64_t byte_off, uint64_t n, uint64_t seed)
{
    if (!h || slot >= h->n_slots || (byte_off & 15) || (n & 15) || byte_off > h->cfg.device_arena_bytes ||
        n > h->cfg.device_arena_bytes - byte_off)
        return MKSNAP_E_INVAL;
    CK(h, cudaSetDevice(h->cfg.device));
    if (n == 0)
        return 0;
    k_synth_fill<<<h->sm_count * 8, 256, 0, h->s_comp>>>(reinterpret_cast<uint64_t *>(h->d_slot[slot] + byte_off),
                                                         byte_off / 8, n / 8, seed);
    LAUNCH_OK(h);
    return 0;
}

int mksnap_memset(mksnap_t *h, uint32_t slot, uint64_t byte_off, uint64_t n, int value)
{
    if (!h || slot >= h->n_slots || byte_off > h->cfg.device_arena_bytes || n > h->cfg.device_arena_bytes - byte_off)
        return MKSNAP_E_INVAL;
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaMemsetAsync(h->d_slot[slot] + byte_off, value, n, h->s_comp));
    return 0;
}

int mksnap_sync(mksnap_t *h)
{
    if (!h)
        return MKSNAP_E_INVAL;
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaStreamSynchronize(h->s_copy));
    CK(h, cudaStreamSynchronize(h->s_comp));
    return 0;
}

int mksnap_finish(mksnap_t *h, mksnap_result *out)
{
    if (!h || !out)
        return MKSNAP_E_INVAL;
    if (!h->in_session)
        return fail(h, MKSNAP_E_STATE, "finish without begin");
    CK(h, cudaSetDevice(h->cfg.device));
    cudaStream_t s = h->s_comp;
    CK(h, cudaMemcpyAsync(h->h_sc, h->d_sc, sizeof(SessionCounters), cudaMemcpyDeviceToHost, s));
    CK(h, cudaStreamSynchronize(s));
    h->stats.d2h_bytes += sizeof(SessionCounters);
    if (h->h_sc->err & 1u)
        return fail(h, MKSNAP_E_CAPACITY, "candidate pool overflow (capacity %u entries): pathologically dense candidates", h->pool_cap);
    if (h->h_sc->err & 4u)
        return fail(h, MKSNAP_E_CUDA, "k_gear_scan: dynamic shared memory does not start where the layout plan assumes");
    if (h->h_sc->err & 8u)
        return fail(h, MKSNAP_E_STATE, "internal: open chunk of a continued file exceeds the carry buffer");
    if (h->open_file)
        return fail(h, MKSNAP_E_STATE, "finish: the last submit left a file open (MKSNAP_X_MORE without its continuation)");
    if (h->h_sc->err & 2u)
        return fail(h, MKSNAP_E_CAPACITY, "chunk table overflow (max_chunks = %llu)", (unsigned long long)h->max_chunks);
    const uint64_t n = h->h_sc->n_chunks;
    CK(h, cudaEventRecord(h->ev_fin[0], s));
    int rc = sort_unique_root(h, h->d_digests, n, s);
    if (rc)
        return rc;
    CK(h, cudaEventRecord(h->ev_fin[1], s));
    if (h->n_ranks > 1) {
        // one rank of several: the content address is the root of the GLOBAL table, computed by the exchange step;
        // a root over this rank's shard would be ~1 ms of Merkle levels nobody reads
        memset(h->root, 0, 32);
    } else {
        rc = merkle_root(h, s);
        if (rc)
            return rc;
    }
    CK(h, cudaEventRecord(h->ev_fin[2], s));
    CK(h, cudaStreamSynchronize(s));
    h->have_fin_times = true;
    memset(out, 0, sizeof *out);
    out->crc_pure = h->h_sc->crc_acc ^ h->crc_host_acc;
    out->crc_bytes = h->crc_bytes + h->crc_host_bytes;
    out->cdc_bytes = h->h_sc->cdc_bytes;
    out->n_files = h->h_sc->n_files;
    out->n_chunks = n;
    out->n_unique = h->n_unique;
    memcpy(out->root, h->root, 32);
    out->n_streams = h->n_streams;
    h->last_result = *out;
    h->finished = true;
    h->table_own = h->n_ranks == 1;
    return 0;
}

uint32_t mksnap_ctx_crc32(const mksnap_result *res)
{
    // standard CRC = pure ^ (0xFFFFFFFF * x^(8L)) ^ 0xFFFFFFFF
    const uint64_t M = 0xFFFFFFFFull;
    const uint64_t bits = ((res->crc_bytes % M) * 8ull) % M;
    return res->crc_pure ^ crc_mulmod(0xFFFFFFFFu, xpow_bits(bits)) ^ 0xFFFFFFFFu;
}

int mksnap_crc_add(mksnap_t *h, uint32_t pure, uint64_t len, uint64_t crc_suffix)
{
    if (!h)
        return MKSNAP_E_INVAL;
    if (!h->in_session || h->finished)
        return fail(h, MKSNAP_E_STATE, "crc_add outside begin/finish");
    const uint64_t M = 0xFFFFFFFFull;
    h->crc_host_acc ^= crc_mulmod(pure, xpow_bits(((crc_suffix % M) * 8ull) % M));
    h->crc_host_bytes += len;
    return 0;
}

uint32_t mksnap_crc_concat(uint32_t pure_a, uint32_t pure_b, uint64_t len_b)
{
    const uint64_t M = 0xFFFFFFFFull;
    return crc_mulmod(pure_a, xpow_bits(((len_b % M) * 8ull) % M)) ^ pure_b;
}

int mksnap_get_extent_crcs(mksnap_t *h, uint32_t *pure, uint64_t capacity, uint64_t *n_out)
{
    if (!h || !h->finished || !n_out)
        return h ? fail(h, MKSNAP_E_STATE, "get_extent_crcs before finish") : MKSNAP_E_INVAL;
    CK(h, cudaSetDevice(h->cfg.device));
    *n_out = h->crc_session_n;
    if (h->crc_session_n > h->crc_session_cap)
        return fail(h, MKSNAP_E_CAPACITY, "the session submitted %llu CRC extents, the per-extent table keeps %llu",
                    (unsigned long long)h->crc_session_n, (unsigned long long)h->crc_session_cap);
    if (!pure || h->crc_session_n > capacity)
        return fail(h, MKSNAP_E_CAPACITY, "need %llu entries", (unsigned long long)h->crc_session_n);
    if (h->crc_session_n)
        CK(h, cudaMemcpy(pure, h->d_crc_session, h->crc_session_n * 4, cudaMemcpyDeviceToHost));
    h->stats.d2h_bytes += h->crc_session_n * 4;
    return 0;
}

int mksnap_get_chunks(mksnap_t *h, uint64_t *ends, uint8_t *digests, uint64_t capacity)
{
    if (!h || !h->finished)
        return h ? fail(h, MKSNAP_E_STATE, "get_chunks before finish") : MKSNAP_E_INVAL;
    CK(h, cudaSetDevice(h->cfg.device));
    const uint64_t n = h->last_result.n_chunks;
    if (n > capacity)
        return fail(h, MKSNAP_E_CAPACITY, "need %llu rows", (unsigned long long)n);
    if (ends && n)
        CK(h, cudaMemcpy(ends, h->d_chunk_end, n * 8, cudaMemcpyDeviceToHost));
    if (digests && n)
        CK(h, cudaMemcpy(digests, h->d_digests, n * 32, cudaMemcpyDeviceToHost));
    h->stats.d2h_bytes += (ends ? n * 8 : 0) + (digests ? n * 32 : 0);
    return 0;
}

uint64_t mksnap_table_rows(mksnap_t *h) { return h && h->finished ? h->n_unique : 0; }

int mksnap_get_table(mksnap_t *h, uint8_t *table, uint64_t capacity_rows)
{
    if (!h || !h->finished || !table)
        return h ? fail(h, MKSNAP_E_STATE, "get_table before finish") : MKSNAP_E_INVAL;
    CK(h, cudaSetDevice(h->cfg.device));
    if (h->n_unique > capacity_rows)
        return fail(h, MKSNAP_E_CAPACITY, "need %llu rows", (unsigned long long)h->n_unique);
    if (h->n_unique)
        CK(h, cudaMemcpy(table, h->d_table, h->n_unique * 32, cudaMemcpyDeviceToHost));
    h->stats.d2h_bytes += h->n_unique * 32;
    return 0;
}

int mksnap_get_stream_digests(mksnap_t *h, uint8_t *digests, uint64_t capacity)
{
    if (!h || !digests)
        return MKSNAP_E_INVAL;
    CK(h, cudaSetDevice(h->cfg.device));
    if (h->n_streams > capacity)
        return fail(h, MKSNAP_E_CAPACITY, "need %llu rows", (unsigned long long)h->n_streams);
    CK(h, cudaStreamSynchronize(h->s_comp));
    if (h->n_streams)
        CK(h, cudaMemcpy(digests, h->d_stream_digests, h->n_streams * 32, cudaMemcpyDeviceToHost));
    h->stats.d2h_bytes += h->n_streams * 32;
    return 0;
}

int mksnap_stats(mksnap_t *h, mksnap_stats_t *out)
{
    if (!h || !out)
        return MKSNAP_E_INVAL;
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaStreamSynchronize(h->s_copy));
    CK(h, cudaStreamSynchronize(h->s_comp));
    if (h->have_submit_times) {
        float t[5];
        for (int i = 0; i < 5; i++)
            CK(h, cudaEventElapsedTime(&t[i], h->ev[i], h->ev[i + 1]));
        h->stats.ms_crc = t[0];
        h->stats.ms_scan = t[1];
        h->stats.ms_select = t[2];
        h->stats.ms_sha = t[3];
        h->stats.ms_stream = t[4];
        CK(h, cudaEventElapsedTime(&h->stats.ms_total, h->ev[0], h->ev[5]));
    }
    if (h->have_h2d_time)
        CK(h, cudaEventElapsedTime(&h->stats.ms_h2d, h->ev_copy0, h->ev_copy1));
    if (h->have_fin_times) {
        CK(h, cudaEventElapsedTime(&h->stats.ms_sort, h->ev_fin[0], h->ev_fin[1]));
        CK(h, cudaEventElapsedTime(&h->stats.ms_root, h->ev_fin[1], h->ev_fin[2]));
    }
    *out = h->stats;
    return 0;
}
// ---- chunk index and chunk delta (DESIGN.md section 3b) ---------------------------------------------------------
struct mksnap_index {
    int device = 0;
    uint64_t cap = 0, n = 0;
    uint32_t bits = 0;                 // directory bits of the current table
    int cur = 0;                       // rows[cur] / dir[cur] hold the index; the other pair is the spare a union builds
    uint8_t *rows[2] = {nullptr, nullptr};
    uint32_t *dir[2] = {nullptr, nullptr};
    uint8_t *novel = nullptr;          // compacted rows a union adds
    uint8_t *stage = nullptr;          // uploaded rows of add_rows (allocated by the first add_rows)
    uint32_t *flags = nullptr, *pos = nullptr, *scan_tmp = nullptr;
    uint64_t scan_words = 0;
    uint32_t *d_bad = nullptr;
};

static mk::RowSet index_view(const mksnap_index *ix)
{
    return mk::RowSet{ix->rows[ix->cur], ix->dir[ix->cur], (uint32_t)ix->n, ix->bits};
}

static uint32_t grid_for(uint64_t n, uint32_t tb) { return (uint32_t)std::max<uint64_t>(1, (n + tb - 1) / tb); }

// delta / add_table / get_chunk_status need the finished session's own table on a single-rank handle
static int own_table_check(mksnap *h, const mksnap_index *ix, const char *what)
{
    if (ix && ix->device != h->cfg.device)
        return fail(h, MKSNAP_E_INVAL, "%s: index lives on device %d, handle on device %d", what, ix->device, h->cfg.device);
    if (!h->finished)
        return fail(h, MKSNAP_E_STATE, "%s needs a finished session", what);
    if (h->n_ranks > 1)
        return fail(h, MKSNAP_E_STATE, "%s: the handle is one rank of %d (its table is a shard)", what, h->n_ranks);
    if (!h->table_own)
        return fail(h, MKSNAP_E_STATE, "%s: an exchange or all-gather replaced the session's table", what);
    return 0;
}

static void index_free(mksnap_index *ix)
{
    for (int k = 0; k < 2; k++) {
        cudaFree(ix->rows[k]);
        cudaFree(ix->dir[k]);
    }
    cudaFree(ix->novel); cudaFree(ix->stage); cudaFree(ix->flags); cudaFree(ix->pos); cudaFree(ix->scan_tmp); cudaFree(ix->d_bad);
    delete ix;
}

int mksnap_index_create(mksnap_t *h, uint64_t capacity_rows, mksnap_index_t **out)
{
    if (!h || !out)
        return MKSNAP_E_INVAL;
    *out = nullptr;
    if (capacity_rows >= (1ull << 32))
        return fail(h, MKSNAP_E_INVAL, "index capacity %llu rows: must be below 2^32", (unsigned long long)capacity_rows);
    CK(h, cudaSetDevice(h->cfg.device));
    mksnap_index *ix = new mksnap_index;
    ix->device = h->cfg.device;
    ix->cap = capacity_rows;
    const uint64_t rows = std::max<uint64_t>(1, capacity_rows);
    const uint64_t dir_words = (1ull << mk::dir_bits(capacity_rows)) + 1;
    ix->scan_words = rows / SCAN_ITEMS * 2 + 4096;
    cudaError_t e = cudaSuccess;
    for (int k = 0; k < 2 && e == cudaSuccess; k++) {
        e = cudaMalloc(&ix->rows[k], rows * 32);
        if (e == cudaSuccess)
            e = cudaMalloc(&ix->dir[k], dir_words * 4);
    }
    if (e == cudaSuccess) e = cudaMalloc(&ix->novel, rows * 32);
    if (e == cudaSuccess) e = cudaMalloc(&ix->flags, rows * 4);
    if (e == cudaSuccess) e = cudaMalloc(&ix->pos, rows * 4);
    if (e == cudaSuccess) e = cudaMalloc(&ix->scan_tmp, ix->scan_words * 4);
    if (e == cudaSuccess) e = cudaMalloc(&ix->d_bad, 4);
    if (e == cudaSuccess) {
        k_dir_build<<<1, 256, 0, h->s_comp>>>(ix->rows[0], 0, 0, ix->dir[0]); // the empty index: dir = {0, 0}
        e = cudaGetLastError();
        if (e == cudaSuccess)
            e = cudaStreamSynchronize(h->s_comp);
    }
    if (e != cudaSuccess) {
        index_free(ix);
        return fail(h, e == cudaErrorMemoryAllocation ? MKSNAP_E_NOMEM : MKSNAP_E_CUDA, "mksnap_index_create: %s",
                    cudaGetErrorString(e));
    }
    h->stats.kernel_launches++;
    *out = ix;
    return 0;
}

void mksnap_index_destroy(mksnap_index_t *ix)
{
    if (!ix)
        return;
    cudaSetDevice(ix->device);
    index_free(ix);
}

uint64_t mksnap_index_rows(const mksnap_index_t *ix) { return ix ? ix->n : 0; }

// index := index U src[0, m) (src sorted-unique, on the device).  Novel rows = rows the index lookup misses, compacted
// with scan_u32; the merge writes into the spare buffer and the pair is swapped only when everything succeeded.
static int index_union(mksnap *h, mksnap_index *ix, const uint8_t *src, uint64_t m, bool check_ascent)
{
    if (m > ix->cap) // m distinct rows: the union holds at least m
        return fail(h, MKSNAP_E_CAPACITY, "%llu incoming rows exceed the index capacity %llu", (unsigned long long)m,
                    (unsigned long long)ix->cap);
    cudaStream_t s = h->s_comp;
    if (check_ascent) {
        CK(h, cudaMemsetAsync(ix->d_bad, 0, 4, s));
        if (m > 1) {
            k_check_ascent<<<grid_for(m - 1, 256), 256, 0, s>>>(src, (uint32_t)m, ix->d_bad);
            LAUNCH_OK(h);
        }
    }
    k_novel_flags<<<grid_for(m, 256), 256, 0, s>>>(src, (uint32_t)m, index_view(ix), ix->flags);
    LAUNCH_OK(h);
    int rc = scan_u32(h, ix->flags, ix->pos, m, s, ix->scan_tmp, ix->scan_words);
    if (rc)
        return rc;
    uint32_t tail[3] = {0, 0, 0}; // last pos, last flag, ascent violated
    CK(h, cudaMemcpyAsync(&tail[0], ix->pos + (m - 1), 4, cudaMemcpyDeviceToHost, s));
    CK(h, cudaMemcpyAsync(&tail[1], ix->flags + (m - 1), 4, cudaMemcpyDeviceToHost, s));
    if (check_ascent)
        CK(h, cudaMemcpyAsync(&tail[2], ix->d_bad, 4, cudaMemcpyDeviceToHost, s));
    CK(h, cudaStreamSynchronize(s));
    h->stats.d2h_bytes += check_ascent ? 12 : 8;
    if (tail[2])
        return fail(h, MKSNAP_E_INVAL, "index_add_rows: rows are not strictly ascending");
    const uint64_t novel = (uint64_t)tail[0] + tail[1];
    if (ix->n + novel > ix->cap)
        return fail(h, MKSNAP_E_CAPACITY, "union of %llu index rows and %llu new rows exceeds capacity %llu",
                    (unsigned long long)ix->n, (unsigned long long)novel, (unsigned long long)ix->cap);
    if (novel == 0)
        return 0;
    k_compact_digests<<<grid_for(2 * m, 256), 256, 0, s>>>(src, ix->flags, ix->pos, m, ix->novel);
    LAUNCH_OK(h);
    const int nxt = ix->cur ^ 1;
    const uint64_t total = ix->n + novel;
    k_merge_rows<<<grid_for(total, MERGE_TILE), MERGE_THREADS, 0, s>>>(ix->rows[ix->cur], (uint32_t)ix->n, ix->novel,
                                                                      (uint32_t)novel, ix->rows[nxt]);
    LAUNCH_OK(h);
    const uint32_t bits = mk::dir_bits(total);
    k_dir_build<<<grid_for(total + 1, 256), 256, 0, s>>>(ix->rows[nxt], (uint32_t)total, bits, ix->dir[nxt]);
    LAUNCH_OK(h);
    CK(h, cudaStreamSynchronize(s));
    ix->cur = nxt;
    ix->n = total;
    ix->bits = bits;
    return 0;
}

int mksnap_index_add_rows(mksnap_t *h, mksnap_index_t *ix, const uint8_t *rows, uint64_t n)
{
    if (!h || !ix || (n && !rows))
        return MKSNAP_E_INVAL;
    if (ix->device != h->cfg.device)
        return fail(h, MKSNAP_E_INVAL, "index_add_rows: index lives on device %d, handle on device %d", ix->device, h->cfg.device);
    if (n == 0)
        return 0;
    if (n > ix->cap) // before the upload: the staging buffer holds capacity rows
        return fail(h, MKSNAP_E_CAPACITY, "index_add_rows: %llu rows exceed capacity %llu", (unsigned long long)n,
                    (unsigned long long)ix->cap);
    CK(h, cudaSetDevice(h->cfg.device));
    if (!ix->stage)
        CK(h, cudaMalloc(&ix->stage, std::max<uint64_t>(1, ix->cap) * 32));
    // on the compute stream: a pageable cudaMemcpy may return before its DMA lands, and nothing would order the
    // kernels that read the rows after it
    CK(h, cudaMemcpyAsync(ix->stage, rows, n * 32, cudaMemcpyHostToDevice, h->s_comp));
    h->stats.h2d_bytes += n * 32;
    return index_union(h, ix, ix->stage, n, true);
}

int mksnap_index_add_table(mksnap_t *h, mksnap_index_t *ix)
{
    if (!h || !ix)
        return MKSNAP_E_INVAL;
    int rc = own_table_check(h, ix, "index_add_table");
    if (rc)
        return rc;
    CK(h, cudaSetDevice(h->cfg.device));
    return h->n_unique ? index_union(h, ix, h->d_table, h->n_unique, false) : 0;
}

int mksnap_index_get(mksnap_t *h, mksnap_index_t *ix, uint8_t *rows, uint64_t capacity_rows)
{
    if (!h || !ix || (ix->n && !rows))
        return MKSNAP_E_INVAL;
    if (ix->device != h->cfg.device)
        return fail(h, MKSNAP_E_INVAL, "index_get: index lives on device %d, handle on device %d", ix->device, h->cfg.device);
    if (ix->n > capacity_rows)
        return fail(h, MKSNAP_E_CAPACITY, "index_get: need %llu rows", (unsigned long long)ix->n);
    CK(h, cudaSetDevice(h->cfg.device));
    if (ix->n) {
        CK(h, cudaStreamSynchronize(h->s_comp));
        CK(h, cudaMemcpy(rows, ix->rows[ix->cur], ix->n * 32, cudaMemcpyDeviceToHost));
    }
    h->stats.d2h_bytes += ix->n * 32;
    return 0;
}

int mksnap_delta(mksnap_t *h, const mksnap_index_t *ix, mksnap_delta_result *out)
{
    if (!h || !ix || !out)
        return MKSNAP_E_INVAL;
    int rc = own_table_check(h, ix, "delta");
    if (rc)
        return rc;
    CK(h, cudaSetDevice(h->cfg.device));
    if (!h->d_dstatus) { // first use: the delta's buffers, sized for the session
        const uint64_t mc = std::max<uint64_t>(1, h->max_chunks);
        CK(h, cudaMalloc(&h->d_dfirst, mc * 4));
        CK(h, cudaMalloc(&h->d_duidx, mc * 4));
        CK(h, cudaMalloc(&h->d_ddir, ((1ull << mk::dir_bits(mc)) + 1) * 4));
        CK(h, cudaMalloc(&h->d_dcnt, 6 * sizeof(unsigned long long)));
        CK(h, cudaMalloc(&h->d_dstatus, mc));
        for (int i = 0; i < 2; i++)
            CK(h, cudaEventCreate(&h->ev_delta[i]));
    }
    cudaStream_t s = h->s_comp;
    const uint64_t n = h->last_result.n_chunks, u = h->n_unique;
    CK(h, cudaEventRecord(h->ev_delta[0], s));
    CK(h, cudaMemsetAsync(h->d_dcnt, 0, 6 * sizeof(unsigned long long), s));
    if (n) {
        CK(h, cudaMemsetAsync(h->d_dfirst, 0xFF, u * 4, s));
        const uint32_t tbits = mk::dir_bits(u);
        k_dir_build<<<grid_for(u + 1, 256), 256, 0, s>>>(h->d_table, (uint32_t)u, tbits, h->d_ddir);
        LAUNCH_OK(h);
        k_delta_lookup<<<grid_for(n, 256), 256, 0, s>>>(h->d_digests, (uint32_t)n, index_view(ix),
                                                        mk::RowSet{h->d_table, h->d_ddir, (uint32_t)u, tbits}, h->d_dstatus,
                                                        h->d_duidx, h->d_dfirst);
        LAUNCH_OK(h);
        const uint32_t grid = (uint32_t)std::min<uint64_t>(grid_for(n, DELTA_THREADS), (uint64_t)h->sm_count * 8);
        k_delta_classify<<<grid, DELTA_THREADS, 0, s>>>((uint32_t)n, h->d_duidx, h->d_dfirst, h->d_chunk_len, h->d_dstatus,
                                                        h->d_dcnt);
        LAUNCH_OK(h);
    }
    CK(h, cudaEventRecord(h->ev_delta[1], s));
    unsigned long long c[6];
    CK(h, cudaMemcpyAsync(c, h->d_dcnt, sizeof c, cudaMemcpyDeviceToHost, s));
    CK(h, cudaStreamSynchronize(s));
    h->stats.d2h_bytes += sizeof c;
    memset(out, 0, sizeof *out);
    out->index_rows = ix->n;
    out->known_chunks = c[0];
    out->new_chunks = c[1];
    out->repeat_chunks = c[2];
    out->known_bytes = c[3];
    out->new_bytes = c[4];
    out->repeat_bytes = c[5];
    CK(h, cudaEventElapsedTime(&out->ms_device, h->ev_delta[0], h->ev_delta[1]));
    h->delta_done = true;
    return 0;
}

int mksnap_get_chunk_status(mksnap_t *h, uint8_t *status, uint64_t capacity)
{
    if (!h)
        return MKSNAP_E_INVAL;
    int rc = own_table_check(h, nullptr, "get_chunk_status");
    if (rc)
        return rc;
    if (!h->delta_done)
        return fail(h, MKSNAP_E_STATE, "get_chunk_status before mksnap_delta in this session");
    const uint64_t n = h->last_result.n_chunks;
    if (n > capacity || (n && !status))
        return fail(h, MKSNAP_E_CAPACITY, "need %llu bytes", (unsigned long long)n);
    CK(h, cudaSetDevice(h->cfg.device));
    if (n)
        CK(h, cudaMemcpy(status, h->d_dstatus, n, cudaMemcpyDeviceToHost));
    h->stats.d2h_bytes += n;
    return 0;
}

#include "mksnap_comm.inc"

} // extern "C"
