// Contigs from the string graph S (the stage GenerateContigs(S, mydna, dfd) runs in the reference, src/main.cpp:320).  The
// reference's ContigGeneration.cpp is not pinned; the rule is written down in DESIGN.md §3d and restated in
// tests/contig_inputs.py.  In short: a read is a branch if it has more than two entries in S, or two that leave from the same
// end; the chain graph G keeps the entries of S between two reads that are not branches (and whose mirror is in S); every
// component of G with two or more reads is a path or a cycle and becomes one contig.
//
// Input: S row-major (rows ascending, columns ascending within a row) with global ids, base = global id of read 0 of the
// job; per read its length and its place in a DnaBuffer arena.
//
//   k_ct_rowptr    ptr[v] = first entry of row v, one binary search per read
//   k_ct_branch    degree and branch flag, one thread per read
//   k_ct_slots     two slots per read, indexed by t = (dir >> 1) & 1: the entry of G that leaves the read through its 3' end
//                  (slot 0) or its 5' end (slot 1).  A slot also says which way a walk through the read is heading.
//   k_ct_init      list ranking over 2 n states (v, d) = "at v, leaving through slot d": the successor is (w, the other slot of
//                  w), dist 1; a state whose slot is empty is terminal (its own successor, dist 0)
//   k_ct_jump      one round of Wyllie's pointer jumping (successor, distance and minimum read id doubled), double-buffered
//   k_ct_cut       after a first ranking (minimum id): the smallest read s of a cycle drops the edge to the larger of its two
//                  neighbours, so every component is a path.  A second ranking then gives every state its terminal and distance.
//   k_ct_place     per read: its start (the smaller of its two terminals), its position from the start, which slot leads on
//   k_ct_clen      reads per contig, at the contig id the scan of the start flags gives (contigs in start-id order)
//   k_ct_layout    every read at contig offset + position: (global id, reversed, beg, end) and its segment length
//   k_ct_block     bases and bytes of the contigs of this rank's block
//   k_ct_pack      the sequences, output-driven: one thread per output byte finds its contig and segment by binary search, so
//                  segments that share a byte never race
#pragma once
#include "common.cuh"

namespace elba {

static constexpr u32 CT_NONE = 0xFFFFFFFFu;

__device__ __forceinline__ int ct_t(const int32_t *f, u64 e) { return (__ldg(f + 4 * e) >> 1) & 1; }

__global__ void k_ct_rowptr(const int64_t *__restrict__ row, u64 m, u32 n, int64_t base, u64 *__restrict__ ptr)
{
    const u64 v = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (v > n) return;
    const int64_t want = base + (int64_t)v;
    u64 lo = 0, hi = m;
    while (lo < hi) { const u64 mid = (lo + hi) >> 1; if (__ldg(row + mid) < want) lo = mid + 1; else hi = mid; }
    ptr[v] = lo;
}

__global__ void k_ct_branch(const u64 *__restrict__ ptr, const int32_t *__restrict__ f, u32 n, uint8_t *__restrict__ branch)
{
    const u32 v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n) return;
    const u64 b = ptr[v], deg = ptr[v + 1] - b;
    branch[v] = (deg > 2 || (deg == 2 && ct_t(f, b) == ct_t(f, b + 1))) ? 1 : 0;
}

__global__ void k_ct_slots(const u64 *__restrict__ ptr, const int64_t *__restrict__ col, const int32_t *__restrict__ f, u32 n, int64_t base,
                           const uint8_t *__restrict__ branch, u32 *__restrict__ slot)
{
    const u32 v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n) return;
    u32 s[2] = {CT_NONE, CT_NONE};
    if (!branch[v])
        for (u64 e = ptr[v]; e < ptr[v + 1]; ++e)
        {
            const u32 c = (u32)(__ldg(col + e) - base);
            if (branch[c]) continue;
            bool mirror = false;                                       // c is not a branch: at most two entries to look at
            for (u64 q = ptr[c]; q < ptr[c + 1]; ++q) mirror |= __ldg(col + q) == base + (int64_t)v;
            if (mirror) s[ct_t(f, e)] = (u32)e;
        }
    slot[2 * v] = s[0]; slot[2 * v + 1] = s[1];
}

// the slot of w whose entry leads to v (w is a neighbour of v in G, and G is symmetric)
__device__ __forceinline__ u32 ct_back(const u32 *slot, const int64_t *col, int64_t base, u32 w, u32 v)
{
    const u32 e = slot[2 * w];
    return (e != CT_NONE && __ldg(col + e) == base + (int64_t)v) ? 0u : 1u;
}

// mn may be NULL (second ranking), dist may be NULL (first ranking)
__global__ void k_ct_init(const u32 *__restrict__ slot, const int64_t *__restrict__ col, u32 n, int64_t base,
                          u32 *__restrict__ succ, u32 *__restrict__ dist, u32 *__restrict__ mn)
{
    const u64 x = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= 2ull * n) return;
    const u32 v = (u32)(x >> 1), e = slot[x];
    if (e == CT_NONE) { succ[x] = (u32)x; if (dist) dist[x] = 0; }
    else
    {
        const u32 w = (u32)(__ldg(col + e) - base);
        succ[x] = 2 * w + (1 - ct_back(slot, col, base, w, v)); if (dist) dist[x] = 1;
    }
    if (mn) mn[x] = v;
}

__global__ void k_ct_jump(u64 ns, const u32 *__restrict__ succ, const u32 *__restrict__ dist, const u32 *__restrict__ mn,
                          u32 *__restrict__ succ2, u32 *__restrict__ dist2, u32 *__restrict__ mn2)
{
    const u64 x = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= ns) return;
    const u32 s = succ[x];
    succ2[x] = succ[s];
    if (dist) dist2[x] = dist[x] + dist[s];
    if (mn) mn2[x] = min(mn[x], mn[s]);
}

// after the first ranking: a state whose successor still has a slot is on a cycle (a path's states reach their terminal
// within 2^rounds >= n hops).  Only the cycle's smallest read writes, and only slots of its own cycle.
__global__ void k_ct_cut(u32 *__restrict__ slot, const int64_t *__restrict__ col, int64_t base, const u32 *__restrict__ succ,
                         const u32 *__restrict__ mn, u32 n, uint8_t *__restrict__ cycle_start)
{
    const u32 v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n) return;
    uint8_t start = 0;
    if (slot[2 * v] != CT_NONE && slot[2 * v + 1] != CT_NONE && slot[succ[2 * v]] != CT_NONE && mn[2 * v] == v)
    {
        const u32 a = (u32)(__ldg(col + slot[2 * v]) - base), b = (u32)(__ldg(col + slot[2 * v + 1]) - base);
        const u32 u = a < b ? b : a;
        slot[2 * u + ct_back(slot, col, base, u, v)] = CT_NONE;
        slot[2 * v + (a < b ? 1 : 0)] = CT_NONE;
        start = 1;
    }
    cycle_start[v] = start;
}

// after the second ranking.  next = the slot that leads away from the start (2: the read is in no contig); flag = 1 for a
// start read (an exclusive scan of the flags numbers the contigs in start-id order); L = reads of the read's contig.
__global__ void k_ct_place(const u32 *__restrict__ succ, const u32 *__restrict__ dist, u32 n, u64 *__restrict__ flag,
                           u32 *__restrict__ start, u32 *__restrict__ pos, uint8_t *__restrict__ next, u32 *__restrict__ L)
{
    const u32 v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v > n) return;
    if (v == n) { flag[n] = 0; return; }
    const u32 e0 = succ[2 * v] >> 1, e1 = succ[2 * v + 1] >> 1, d0 = dist[2 * v], d1 = dist[2 * v + 1];
    const u32 len = d0 + d1 + 1;
    if (len < 2) { next[v] = 2; flag[v] = 0; return; }
    const bool from0 = e0 < e1;                   // the start lies behind slot 0: the walk leaves v through slot 1
    start[v] = from0 ? e0 : e1; pos[v] = from0 ? d0 : d1; next[v] = from0 ? 1 : 0; L[v] = len;
    flag[v] = (from0 ? d0 : d1) == 0 ? 1ull : 0ull;
}

// cid = exclusive scan of the start flags; clen[c] = reads of contig c (zeroed beforehand, n + 1 entries for the scan)
__global__ void k_ct_clen(const u64 *__restrict__ cid, const u32 *__restrict__ L, u32 n, u64 *__restrict__ clen)
{
    const u32 v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n || cid[v + 1] == cid[v]) return;
    clen[cid[v]] = L[v];
}

struct CtReads { const uint8_t *buf; const u64 *off; const u32 *len; };

// every read of a contig at cptr[contig] + pos: its segment (rule 6 of DESIGN.md §3d)
__global__ void k_ct_layout(const u32 *__restrict__ slot, const int64_t *__restrict__ col, const int32_t *__restrict__ f, int64_t base, u32 n,
                            const u64 *__restrict__ cid, const u64 *__restrict__ cptr, const u32 *__restrict__ start, const u32 *__restrict__ pos,
                            const uint8_t *__restrict__ next, CtReads rd, int64_t *__restrict__ oread, uint8_t *__restrict__ orev,
                            u32 *__restrict__ obeg, u32 *__restrict__ oend, u64 *__restrict__ seglen)
{
    const u32 v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n || next[v] == 2) return;
    const u32 nx = next[v], len = __ldg(rd.len + v);
    const u64 o = cptr[cid[start[v]]] + pos[v];
    u32 b = 0, e = len;
    if (pos[v] != 0)
    {
        const u32 p = (u32)(__ldg(col + slot[2 * v + (1 - nx)]) - base);      // the read before v; its next slot leads to v
        const int32_t suf = __ldg(f + 4 * (u64)slot[2 * p + next[p]] + 2);
        const u32 s = suf < 0 ? 0u : min((u32)suf, len);
        if (nx == 0) b = len - s; else e = s;
    }
    oread[o] = base + (int64_t)v; orev[o] = nx; obeg[o] = b; oend[o] = e; seglen[o] = e - b;
}

// contig first + i of this rank's block: bases and bytes (count + 1 entries of bytes for the scan)
__global__ void k_ct_block(const u64 *__restrict__ cptr, const u64 *__restrict__ boff, u64 first, u64 count, u64 *__restrict__ blen, u64 *__restrict__ bbytes)
{
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > count) return;
    if (i == count) { bbytes[i] = 0; return; }
    const u64 l = boff[cptr[first + i + 1]] - boff[cptr[first + i]];
    blen[i] = l; bbytes[i] = (l + 3) / 4;
}

__device__ __forceinline__ u32 ct_base(const CtReads &rd, u32 v, u32 i)
{
    return (__ldg(rd.buf + __ldg(rd.off + v) + (i >> 2)) >> (6 - 2 * (i & 3))) & 3u;
}

// bbyte = exclusive scan of the block's bytes per contig (count + 1 entries); boff = exclusive scan of the segment lengths
__global__ void k_ct_pack(const u64 *__restrict__ bbyte, u64 count, u64 first, const u64 *__restrict__ cptr, const u64 *__restrict__ boff,
                          const int64_t *__restrict__ oread, const uint8_t *__restrict__ orev, const u32 *__restrict__ obeg, const u32 *__restrict__ oend,
                          int64_t base, CtReads rd, uint8_t *__restrict__ out)
{
    const u64 total = bbyte[count];
    const u64 B = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (B >= total) return;
    u64 lo = 0, hi = count;                                        // last contig with bbyte <= B (empty contigs come before it)
    while (hi - lo > 1) { const u64 mid = (lo + hi) >> 1; if (bbyte[mid] <= B) lo = mid; else hi = mid; }
    const u64 c = first + lo, s0 = cptr[c], s1 = cptr[c + 1];
    const u64 g0 = boff[s0] + 4 * (B - bbyte[lo]), gend = boff[s1];
    u64 a = s0, z = s1;                                            // last segment with boff <= g0 (empty segments come before it)
    while (z - a > 1) { const u64 mid = (a + z) >> 1; if (boff[mid] <= g0) a = mid; else z = mid; }
    u32 byte = 0;
    for (u32 j = 0; j < 4; ++j)
    {
        const u64 g = g0 + j;
        if (g >= gend) break;
        while (boff[a + 1] <= g) ++a;
        const u32 o = (u32)(g - boff[a]), v = (u32)(oread[a] - base);
        const u32 x = orev[a] ? 3u - ct_base(rd, v, oend[a] - 1 - o) : ct_base(rd, v, obeg[a] + o);
        byte |= x << (6 - 2 * j);
    }
    out[B] = (uint8_t)byte;
}

} // namespace elba
