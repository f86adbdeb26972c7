// mksnap_groups.cuh — kernels of grouped sessions (DESIGN.md section 3c): per-group chunk tables, roots and deltas.
//
// A grouped session tags every CDC file with a group (a layer).  Finish then builds, next to the batch table, one
// sorted-unique table per group: each chunk is mapped to its batch-table row by lookup (the K3 payload is not usable,
// k_fix_ties reorders digests without it), the exact integer keys (group << rbits) | row are radix-sorted on only the
// bits they use, and unique keys are compacted.  The batch table is sorted, so rows inside a group come out in
// bytewise digest order.  Per-group Merkle levels run through the K4 stream kernel with explicit range lists.  None of
// these kernels runs in an ungrouped session.
#pragma once

#include "mksnap_index.cuh"

namespace mk {

constexpr uint32_t GROUPS_MAX = 65536;
constexpr uint32_t GD_SMEM_GROUPS = 512;                 // the grouped delta reduces in shared memory up to this many groups
constexpr unsigned long long GD_KNOWN = ~1ull;           // first64[row]: the row is in the index
constexpr unsigned long long GD_NONE = ~0ull;

// chunk -> group, one warp per file of the submit (run after the cut selection, before k_batch_end)
__global__ void __launch_bounds__(256) k_group_tag(uint32_t n_files, const uint32_t *__restrict__ file_group,
                                                   const uint32_t *__restrict__ counts, const uint32_t *__restrict__ bases,
                                                   const SessionCounters *__restrict__ sc, uint64_t max_chunks,
                                                   uint32_t *__restrict__ chunk_group)
{
    const uint32_t f = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (f >= n_files || sc->err)
        return;
    const uint64_t out = sc->n_chunks + bases[f];
    const uint32_t c = counts[f], g = file_group[f];
    for (uint32_t j = lane; j < c; j += 32)
        if (out + j < max_chunks)
            chunk_group[out + j] = g;
}

// chunk -> batch-table row (lookup in the finished table), and its sort key (group << rbits) | row
__global__ void __launch_bounds__(256) k_group_keys(const uint8_t *__restrict__ digests, uint32_t n, RowSet tab,
                                                    const uint32_t *__restrict__ chunk_group, uint32_t rbits,
                                                    uint32_t *__restrict__ row_of, uint64_t *__restrict__ keys)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n)
        return;
    const uint32_t r = rowset_find(tab, load_row(digests + (uint64_t)i * 32)); // always found: the table holds every digest
    row_of[i] = r;
    keys[i] = ((uint64_t)chunk_group[i] << rbits) | r;
}

__global__ void __launch_bounds__(256) k_group_flags(const uint64_t *__restrict__ keys, uint32_t n, uint32_t *__restrict__ flags)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n)
        flags[i] = (i == 0 || keys[i] != keys[i - 1]) ? 1u : 0u;
}

// gtable[pos[i]] = table[row of key i] for the first key of every run (two threads per 32-byte row)
__global__ void __launch_bounds__(256) k_group_compact(const uint64_t *__restrict__ keys, const uint32_t *__restrict__ flags,
                                                       const uint32_t *__restrict__ pos, uint32_t n, uint32_t rbits,
                                                       const uint8_t *__restrict__ table, uint8_t *__restrict__ gtable)
{
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t i = t >> 1;
    if (i >= n || !flags[i])
        return;
    const uint64_t r = keys[i] & ((1ull << rbits) - 1);
    reinterpret_cast<uint4 *>(gtable + (uint64_t)pos[i] * 32)[t & 1] = reinterpret_cast<const uint4 *>(table + r * 32)[t & 1];
}

// group offsets over the sorted keys, one thread per position i in [0, n]: every group g in (group(i-1), group(i)]
// starts at chunk i and at unique row pos[i]; thread n closes the lists at n_groups (cstart/ustart hold n_groups + 1)
__global__ void __launch_bounds__(256) k_group_bounds(const uint64_t *__restrict__ keys, const uint32_t *__restrict__ flags,
                                                      const uint32_t *__restrict__ pos, uint32_t n, uint32_t rbits,
                                                      uint32_t n_groups, uint32_t *__restrict__ cstart, uint32_t *__restrict__ ustart)
{
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n)
        return;
    const int64_t lo = i == 0 ? 0 : (int64_t)(keys[i - 1] >> rbits) + 1;
    const int64_t hi = i == n ? (int64_t)n_groups : (int64_t)(keys[i] >> rbits);
    const uint32_t u = i == n ? (n ? pos[n - 1] + flags[n - 1] : 0u) : pos[i];
    for (int64_t g = lo; g <= hi; ++g) {
        cstart[g] = (uint32_t)i;
        ustart[g] = u;
    }
}

// ---- grouped delta ----
// per batch-table row: in the index (GD_KNOWN) or not yet claimed (GD_NONE)
__global__ void __launch_bounds__(256) k_gdelta_rows(const uint8_t *__restrict__ table, uint32_t u, RowSet ix,
                                                     unsigned long long *__restrict__ first)
{
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < u)
        first[r] = rowset_find(ix, load_row(table + (uint64_t)r * 32)) != IDX_NONE ? GD_KNOWN : GD_NONE;
}

// first[row] = min over the row's chunks of (group << 32) | chunk: the lowest group carrying the digest, and in it the
// lowest chunk position
__global__ void __launch_bounds__(256) k_gdelta_first(const uint32_t *__restrict__ row_of, const uint32_t *__restrict__ chunk_group,
                                                      uint32_t n, unsigned long long *__restrict__ first)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n)
        return;
    const uint32_t r = row_of[i];
    if (first[r] != GD_KNOWN)
        atomicMin(first + r, ((unsigned long long)chunk_group[i] << 32) | i);
}

// status per chunk (KNOWN: in the index or first seen in an earlier group; NEW: the lowest position of its group
// carrying the digest; REPEAT otherwise) and per-group counts cnt[g * 6 + {known, new, repeat} chunks, then bytes].
// A warp whose 32 chunks share one group (the common case: chunks come file by file) reduces by shuffles and adds
// once; otherwise each lane adds its own chunk.  SMEM: the counters of every group live in shared memory per CTA.
template <bool SMEM>
__global__ void __launch_bounds__(DELTA_THREADS) k_gdelta_classify(uint32_t n, const uint32_t *__restrict__ row_of,
                                                                   const uint32_t *__restrict__ chunk_group,
                                                                   const unsigned long long *__restrict__ first,
                                                                   const uint64_t *__restrict__ len, uint32_t n_groups,
                                                                   uint8_t *__restrict__ status,
                                                                   unsigned long long *__restrict__ cnt)
{
    __shared__ unsigned long long s_cnt[SMEM ? GD_SMEM_GROUPS * 6 : 1];
    unsigned long long *acc = SMEM ? s_cnt : cnt;
    if (SMEM) {
        for (uint32_t j = threadIdx.x; j < n_groups * 6; j += blockDim.x)
            s_cnt[j] = 0;
        __syncthreads();
    }
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t stride = gridDim.x * blockDim.x;
    const uint32_t n_round = (n + 31) / 32 * 32; // whole warps stay in the loop together for the shuffles
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_round; i += stride) {
        const bool ok = i < n;
        uint32_t g = 0, cls = 3;
        uint64_t l = 0;
        if (ok) {
            g = chunk_group[i];
            const unsigned long long f = first[row_of[i]];
            cls = (f == GD_KNOWN || (uint32_t)(f >> 32) < g) ? 0u : ((uint32_t)f == i ? 1u : 2u);
            status[i] = (uint8_t)cls;
            l = len[i];
        }
        const uint32_t g0 = __shfl_sync(0xFFFFFFFFu, g, 0);
        const bool ok0 = __shfl_sync(0xFFFFFFFFu, ok ? 1u : 0u, 0) != 0;
        if (__all_sync(0xFFFFFFFFu, !ok || g == g0) && ok0) {
            uint32_t c[3];
            uint64_t by[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                c[k] = __reduce_add_sync(0xFFFFFFFFu, cls == (uint32_t)k ? 1u : 0u);
                by[k] = cls == (uint32_t)k ? l : 0;
#pragma unroll
                for (int s = 16; s > 0; s >>= 1)
                    by[k] += __shfl_xor_sync(0xFFFFFFFFu, by[k], s);
            }
            if (lane < 6) {
                const uint64_t v = lane == 0 ? c[0] : lane == 1 ? c[1] : lane == 2 ? c[2] : lane == 3 ? by[0] : lane == 4 ? by[1] : by[2];
                if (v)
                    atomicAdd(acc + (uint64_t)g0 * 6 + lane, (unsigned long long)v);
            }
        } else if (ok) {
            atomicAdd(acc + (uint64_t)g * 6 + cls, 1ull);
            if (l)
                atomicAdd(acc + (uint64_t)g * 6 + 3 + cls, (unsigned long long)l);
        }
    }
    if (SMEM) {
        __syncthreads();
        for (uint32_t j = threadIdx.x; j < n_groups * 6; j += blockDim.x)
            if (s_cnt[j])
                atomicAdd(cnt + j, s_cnt[j]);
    }
}

} // namespace mk
