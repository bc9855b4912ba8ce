// The overlap graph R from the resident alignments: the prune between PairwiseAlignment and TransitiveReduction
// (src/main.cpp:300-313), restated in tests/tr_inputs.py::overlap_graph.
//
// Over the alignments of all ranks: C = { row(p) : passed(p) and containedQ(p) } U { col(p) : passed(p) and containedT(p) };
// p stays in R iff passed(p) and neither of its reads is in C.  An entry of R carries its row, its column and the four
// fields TransitiveReduction reads (direction, directionT, suffix, suffixT).  R keeps the order of the alignments.
//
//   k_og_contained   one thread per alignment: stores 1 into the contained flag (one byte per read of the whole job) of the
//                    row or column read it finds contained.  Racing stores write the same value.
//   k_og_count       |C|: the set flags, summed per warp, one atomic per warp
//   k_og_keep        one thread per alignment: 1 if it stays in R (and a 0 past the end, for the exclusive scan)
//   k_og_compact     the kept alignments at their scanned positions: job-relative row / column, 4 fields, source index
//   k_og_ids         job-relative ids back to global ones for the copy to the host
//
// Read ids inside are relative to the first read of rank 0, so that the flags and the transitive-reduction kernels index
// [0, reads of the job).  Everything is a few bytes per alignment and launch-bound.
#pragma once
#include "common.cuh"

namespace elba {

static constexpr int OG_FIELDS = 13, OG_PASSED = 6, OG_CONT_Q = 7, OG_CONT_T = 8, OG_DIR = 9;     // Overlap's fields as k_xdrop writes them

// row_base / col_base: job-relative id of the block's first row / column read (pair ids are local to the block of B)
__global__ void k_og_contained(const u32 *__restrict__ prow, const u32 *__restrict__ pcol, const int32_t *__restrict__ fields, u64 np,
                               u32 row_base, u32 col_base, uint8_t *__restrict__ contained)
{
    const u64 p = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= np) return;
    const int32_t *f = fields + (u64)OG_FIELDS * p;
    if (f[OG_PASSED] == 0) return;
    if (f[OG_CONT_Q] != 0) contained[row_base + prow[p]] = 1;
    if (f[OG_CONT_T] != 0) contained[col_base + pcol[p]] = 1;
}

__global__ void k_og_count(const uint8_t *__restrict__ flag, u64 n, u64 *__restrict__ total)
{
    u32 c = 0;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) c += flag[i];
    c = __reduce_add_sync(0xFFFFFFFFu, c);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(total, (u64)c);
}

__global__ void k_og_keep(const u32 *__restrict__ prow, const u32 *__restrict__ pcol, const int32_t *__restrict__ fields, u64 np,
                          u32 row_base, u32 col_base, const uint8_t *__restrict__ contained, u64 *__restrict__ keep)
{
    const u64 p = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (p > np) return;
    u64 k = 0;
    if (p < np && fields[(u64)OG_FIELDS * p + OG_PASSED] != 0)
        k = (!contained[row_base + prow[p]] && !contained[col_base + pcol[p]]) ? 1ull : 0ull;
    keep[p] = k;
}

// rank = exclusive scan of k_og_keep's flags: alignment p is kept iff rank[p + 1] != rank[p]
__global__ void k_og_compact(const u32 *__restrict__ prow, const u32 *__restrict__ pcol, const int32_t *__restrict__ fields, u64 np,
                             u32 row_base, u32 col_base, const u64 *__restrict__ rank,
                             int64_t *__restrict__ row, int64_t *__restrict__ col, int32_t *__restrict__ of, u64 *__restrict__ src)
{
    const u64 p = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= np) return;
    const u64 o = rank[p];
    if (rank[p + 1] == o) return;
    const int32_t *f = fields + (u64)OG_FIELDS * p;
    row[o] = (int64_t)(row_base + prow[p]); col[o] = (int64_t)(col_base + pcol[p]);
    of[4 * o] = f[OG_DIR]; of[4 * o + 1] = f[OG_DIR + 1]; of[4 * o + 2] = f[OG_DIR + 2]; of[4 * o + 3] = f[OG_DIR + 3];
    src[o] = p;
}

__global__ void k_og_ids(const int64_t *__restrict__ rrow, const int64_t *__restrict__ rcol, u64 n, int64_t base,
                         int64_t *__restrict__ row, int64_t *__restrict__ col)
{
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { row[i] = rrow[i] + base; col[i] = rcol[i] + base; }
}

} // namespace elba
