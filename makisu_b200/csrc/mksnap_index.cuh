// mksnap_index.cuh — kernels of the chunk index and the chunk delta (DESIGN.md section 3b).
//
// A table here is a sorted-unique array of 32-byte digests in bytewise order (the order of mksnap_get_table).  Lookups
// go through a prefix directory: with B directory bits, dir[b] is the first row whose top-B prefix (of the big-endian
// 64-bit key, the K3 key) is >= b, and dir[2^B] = rows.  A lookup reads its bucket's bounds and binary-searches inside
// the bucket, comparing the 64-bit key first and the remaining 192 bits only on key equality.  Digests are uniform, so
// B = log2(rows) - 2 leaves a handful of rows per bucket; a skewed table (every row in one bucket) is still correct,
// the search just covers more rows.
#pragma once

#include "mksnap_kernels.cuh"

namespace mk {

constexpr uint32_t DIR_MAX_BITS = 24;
constexpr uint32_t IDX_NONE = 0xFFFFFFFFu;

// directory bits for a table of n rows: about four rows per bucket, at most 2^24 buckets
__host__ __device__ inline uint32_t dir_bits(uint64_t n)
{
    uint32_t l = 0;
    while (l < 63 && (2ull << l) <= n)
        ++l; // l = floor(log2(n)) for n >= 1
    return n < 8 ? 0u : (l - 2 < DIR_MAX_BITS ? l - 2 : DIR_MAX_BITS);
}

struct RowSet {
    const uint8_t *rows;
    const uint32_t *dir;
    uint32_t n;
    uint32_t bits;
};

struct Row {
    uint64_t w[4]; // big-endian words: w[0] is the K3 key
};

__device__ __forceinline__ uint64_t be64(uint32_t lo_word, uint32_t hi_word)
{
    return ((uint64_t)__byte_perm(lo_word, 0, 0x0123) << 32) | __byte_perm(hi_word, 0, 0x0123);
}

__device__ __forceinline__ uint64_t row_key(const uint8_t *p)
{
    const uint2 v = *reinterpret_cast<const uint2 *>(p);
    return be64(v.x, v.y);
}

__device__ __forceinline__ Row load_row(const uint8_t *p)
{
    const uint4 a = reinterpret_cast<const uint4 *>(p)[0], b = reinterpret_cast<const uint4 *>(p)[1];
    Row r;
    r.w[0] = be64(a.x, a.y);
    r.w[1] = be64(a.z, a.w);
    r.w[2] = be64(b.x, b.y);
    r.w[3] = be64(b.z, b.w);
    return r;
}

// the last three words of row p compared with q's: -1, 0, 1
__device__ __forceinline__ int tail_cmp(const uint8_t *p, const Row &q)
{
    const uint2 a = reinterpret_cast<const uint2 *>(p)[1];
    const uint4 b = reinterpret_cast<const uint4 *>(p)[1];
    const uint64_t w1 = be64(a.x, a.y), w2 = be64(b.x, b.y), w3 = be64(b.z, b.w);
    if (w1 != q.w[1])
        return w1 < q.w[1] ? -1 : 1;
    if (w2 != q.w[2])
        return w2 < q.w[2] ? -1 : 1;
    if (w3 != q.w[3])
        return w3 < q.w[3] ? -1 : 1;
    return 0;
}

__device__ __forceinline__ bool row_less(const Row &a, const Row &b)
{
    if (a.w[0] != b.w[0])
        return a.w[0] < b.w[0];
    if (a.w[1] != b.w[1])
        return a.w[1] < b.w[1];
    if (a.w[2] != b.w[2])
        return a.w[2] < b.w[2];
    return a.w[3] < b.w[3];
}

__device__ __forceinline__ uint32_t key_prefix(uint64_t key, uint32_t bits) { return bits ? (uint32_t)(key >> (64 - bits)) : 0u; }

// row index of q in t, or IDX_NONE
__device__ __forceinline__ uint32_t rowset_find(const RowSet &t, const Row &q)
{
    const uint32_t b = key_prefix(q.w[0], t.bits);
    uint32_t lo = t.dir[b], hi = t.dir[b + 1];
    while (lo < hi) { // lower bound of q in [lo, hi)
        const uint32_t mid = lo + (hi - lo) / 2;
        const uint8_t *p = t.rows + (uint64_t)mid * 32;
        const uint64_t k = row_key(p);
        const bool less = k != q.w[0] ? k < q.w[0] : tail_cmp(p, q) < 0;
        if (less)
            lo = mid + 1;
        else
            hi = mid;
    }
    if (lo < t.dir[b + 1]) {
        const uint8_t *p = t.rows + (uint64_t)lo * 32;
        if (row_key(p) == q.w[0] && tail_cmp(p, q) == 0)
            return lo;
    }
    return IDX_NONE;
}

// one thread per row i in [0, n]: dir[b] = i for every bucket b in (prefix(i-1), prefix(i)]; thread n closes the
// directory up to the sentinel dir[2^bits] = n.  An empty table gets dir = {0, 0, ...}.
__global__ void __launch_bounds__(256) k_dir_build(const uint8_t *__restrict__ rows, uint32_t n, uint32_t bits,
                                                   uint32_t *__restrict__ dir)
{
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n)
        return;
    const uint64_t lo = i == 0 ? 0 : (uint64_t)key_prefix(row_key(rows + (i - 1) * 32), bits) + 1;
    const uint64_t hi = i == n ? (1ull << bits) : key_prefix(row_key(rows + i * 32), bits);
    for (uint64_t b = lo; b <= hi; ++b)
        dir[b] = (uint32_t)i;
}

// status[i] = KNOWN if chunk i's digest is in the index; otherwise uidx[i] = its row in the session table and
// first[row] = the lowest such chunk (atomicMin)
__global__ void __launch_bounds__(256) k_delta_lookup(const uint8_t *__restrict__ digests, uint32_t n, RowSet ix, RowSet tab,
                                                      uint8_t *__restrict__ status, uint32_t *__restrict__ uidx,
                                                      uint32_t *__restrict__ first)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n)
        return;
    const Row q = load_row(digests + (uint64_t)i * 32);
    if (rowset_find(ix, q) != IDX_NONE) {
        status[i] = 0; // MKSNAP_CHUNK_KNOWN
        uidx[i] = IDX_NONE;
        return;
    }
    const uint32_t u = rowset_find(tab, q); // always found: the session table holds every chunk digest of the session
    uidx[i] = u;
    if (u != IDX_NONE)
        atomicMin(first + u, i);
}

constexpr int DELTA_THREADS = 256;

// status = NEW for the first chunk of each non-known digest, REPEAT for the rest; per-class chunk and byte counts
// (cnt[0..2] chunks, cnt[3..5] bytes: known, new, repeat), reduced per warp, then per CTA, then one 64-bit atomic
__global__ void __launch_bounds__(DELTA_THREADS) k_delta_classify(uint32_t n, const uint32_t *__restrict__ uidx,
                                                                  const uint32_t *__restrict__ first,
                                                                  const uint64_t *__restrict__ len, uint8_t *__restrict__ status,
                                                                  unsigned long long *__restrict__ cnt)
{
    __shared__ unsigned long long s_acc[DELTA_THREADS / 32][6];
    uint32_t c[3] = {0, 0, 0};
    uint64_t by[3] = {0, 0, 0};
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint32_t u = uidx[i];
        const uint32_t cls = u == IDX_NONE ? 0u : (first[u] == i ? 1u : 2u);
        if (cls)
            status[i] = (uint8_t)cls;
        const uint64_t l = len[i];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            c[k] += cls == (uint32_t)k;
            by[k] += cls == (uint32_t)k ? l : 0;
        }
    }
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        c[k] = __reduce_add_sync(0xFFFFFFFFu, c[k]);
#pragma unroll
        for (int s = 16; s > 0; s >>= 1)
            by[k] += __shfl_xor_sync(0xFFFFFFFFu, by[k], s);
    }
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            s_acc[warp][k] = c[k];
            s_acc[warp][3 + k] = by[k];
        }
    }
    __syncthreads();
    if (threadIdx.x < 6) {
        unsigned long long t = 0;
#pragma unroll
        for (int w = 0; w < DELTA_THREADS / 32; ++w)
            t += s_acc[w][threadIdx.x];
        if (t)
            atomicAdd(cnt + threadIdx.x, t);
    }
}

// flags[j] = 1 if row j of src is not in the index (the rows a union adds)
__global__ void __launch_bounds__(256) k_novel_flags(const uint8_t *__restrict__ src, uint32_t m, RowSet ix,
                                                     uint32_t *__restrict__ flags)
{
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m)
        return;
    flags[j] = rowset_find(ix, load_row(src + (uint64_t)j * 32)) == IDX_NONE ? 1u : 0u;
}

// *bad = 1 unless rows are strictly ascending
__global__ void __launch_bounds__(256) k_check_ascent(const uint8_t *__restrict__ rows, uint32_t m, uint32_t *__restrict__ bad)
{
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x + 1;
    if (j >= m)
        return;
    if (!row_less(load_row(rows + (uint64_t)(j - 1) * 32), load_row(rows + (uint64_t)j * 32)))
        *bad = 1u;
}

// ---- merge path of two disjoint sorted tables A (na rows) and B (nb rows) into C ----
constexpr uint32_t MERGE_THREADS = 128;
constexpr uint32_t MERGE_ITEMS = 8;
constexpr uint32_t MERGE_TILE = MERGE_THREADS * MERGE_ITEMS;

// rows of A among the first d rows of the merge, searched in A[a_lo, a_hi) against B[b_lo, b_hi) (a 256-bit binary
// search along the cross diagonal; A and B share no row, so there are no ties)
__device__ __forceinline__ uint64_t merge_path(const uint8_t *A, const uint8_t *B, uint64_t d, uint64_t a_lo, uint64_t a_hi,
                                               uint64_t b_lo, uint64_t b_hi)
{
    uint64_t lo = d > b_hi ? (d - b_hi > a_lo ? d - b_hi : a_lo) : a_lo;
    uint64_t hi = d - b_lo < a_hi ? d - b_lo : a_hi;
    while (lo < hi) {
        const uint64_t mid = lo + (hi - lo) / 2;
        if (row_less(load_row(A + mid * 32), load_row(B + (d - 1 - mid) * 32)))
            lo = mid + 1;
        else
            hi = mid;
    }
    return lo;
}

__device__ __forceinline__ void copy_row(uint8_t *dst, const uint8_t *src)
{
    reinterpret_cast<uint4 *>(dst)[0] = reinterpret_cast<const uint4 *>(src)[0];
    reinterpret_cast<uint4 *>(dst)[1] = reinterpret_cast<const uint4 *>(src)[1];
}

// each CTA finds where its tile of MERGE_TILE output rows starts and ends on A, then each thread finds its own
// MERGE_ITEMS-row diagonal inside the tile and merges sequentially
__global__ void __launch_bounds__(MERGE_THREADS) k_merge_rows(const uint8_t *__restrict__ A, uint32_t na, const uint8_t *__restrict__ B,
                                                             uint32_t nb, uint8_t *__restrict__ C)
{
    __shared__ uint64_t s_a[2];
    const uint64_t total = (uint64_t)na + nb;
    const uint64_t d0 = (uint64_t)blockIdx.x * MERGE_TILE, d1 = d0 + MERGE_TILE < total ? d0 + MERGE_TILE : total;
    if (threadIdx.x < 2)
        s_a[threadIdx.x] = merge_path(A, B, threadIdx.x ? d1 : d0, 0, na, 0, nb);
    __syncthreads();
    const uint64_t a0 = s_a[0], a1 = s_a[1], b0 = d0 - a0, b1 = d1 - a1;
    const uint64_t t0 = d0 + (uint64_t)threadIdx.x * MERGE_ITEMS;
    if (t0 >= d1)
        return;
    const uint64_t t1 = t0 + MERGE_ITEMS < d1 ? t0 + MERGE_ITEMS : d1;
    uint64_t i = merge_path(A, B, t0, a0, a1, b0, b1), j = t0 - i;
    for (uint64_t o = t0; o < t1; ++o) {
        const bool take_a = i < na && (j >= nb || row_less(load_row(A + i * 32), load_row(B + j * 32)));
        if (take_a) {
            copy_row(C + o * 32, A + i * 32);
            ++i;
        } else {
            copy_row(C + o * 32, B + j * 32);
            ++j;
        }
    }
}

} // namespace mk
