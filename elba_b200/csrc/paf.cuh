// PAF text of the overlap graph and of the string graph, formatted on the device (the reference writes <prefix>.overlap.paf
// and <prefix>.string.paf, src/main.cpp:303,317).  The format is defined in DESIGN.md §3d and include/elba_fe.h and restated
// in tests/paf_inputs.py.  One line per alignment, 13 tab-separated columns:
//
//   qname qlen begQ endQ strand tname tlen begT endT score max(endQ - begQ, endT - begT) 255 dr:i:<direction>\n
//
// q = the alignment's row read, t = its column read, strand '-' iff rc; integers in plain decimal.
//
//   k_paf_len          one thread per line: the byte length of the line from the digit counts of its nine integers, the two
//                      name lengths and the 22 constant bytes (12 tabs, strand, "255", "dr:i:", "\n")
//   (CUB scan)         line offsets = exclusive scan of the lengths
//   k_paf_write        a CTA takes PAF_THREADS consecutive lines, whose bytes are one contiguous range of the output: every
//                      thread formats its line into shared memory, staged at the same offset mod 16 as in the output, then
//                      the CTA stores the range with coalesced 16-byte stores (byte stores for the partial chunks at its two
//                      ends).  A run longer than the staging buffer (very long names) is written directly by each thread.
//   k_paf_flags        string graph: 1 for the entries of S with transposed == 0 (the lines), for the scan
//   k_paf_string_lines string graph: line i's reads, direction and, where this rank owns the source alignment, its six
//                      printed fields (zeros otherwise; several GPUs sum the ranks' arrays)
#pragma once
#include "common.cuh"

namespace elba {

static constexpr int PAF_THREADS = 256, PAF_STAGE = 32768, PAF_CONST_BYTES = 22, PAF_XD_FIELDS = 13;

// where the fields of line i come from
struct PafSrc
{
    const u32 *q, *t;                  // row / column read of line i, relative to qbase / tbase (then job-relative)
    u32 qbase, tbase;
    const int32_t *v; u32 vstride;     // begQ endQ begT endT score rc of line i at v[vstride * i + 0..5]
    const int32_t *dir; u32 dstride;   // direction of line i at dir[dstride * i]
    const u32 *len;                    // read lengths, job-relative ids
    const char *names; const u64 *name_off;   // name of read r = names[name_off[r], name_off[r + 1]); names == NULL: id_base + r
    int64_t id_base;
};

__device__ __forceinline__ int paf_digits(u64 v)
{
    int d = 1;
    while (d < 20 && v >= 10ull) { v /= 10ull; ++d; }
    return d;
}
__device__ __forceinline__ int paf_digits_i(int64_t v) { return v < 0 ? 1 + paf_digits(0ull - (u64)v) : paf_digits((u64)v); }

__device__ __forceinline__ char *paf_put(char *p, int64_t v)
{
    u64 u = (u64)v;
    if (v < 0) { *p++ = '-'; u = 0ull - (u64)v; }
    const int n = paf_digits(u);
    for (int k = n - 1; k >= 0; --k) { p[k] = (char)('0' + (int)(u % 10ull)); u /= 10ull; }
    return p + n;
}

__device__ __forceinline__ int paf_name_len(const PafSrc &s, u32 r)
{
    return s.names ? (int)(s.name_off[r + 1] - s.name_off[r]) : paf_digits_i(s.id_base + (int64_t)r);
}

__device__ __forceinline__ char *paf_put_name(const PafSrc &s, u32 r, char *p)
{
    if (!s.names) return paf_put(p, s.id_base + (int64_t)r);
    for (u64 b = s.name_off[r], e = s.name_off[r + 1]; b < e; ++b) *p++ = s.names[b];
    return p;
}

struct PafLine { u32 q, t; int32_t f[6], dir; };

__device__ __forceinline__ PafLine paf_line(const PafSrc &s, u64 i)
{
    PafLine L;
    L.q = s.qbase + s.q[i]; L.t = s.tbase + s.t[i];
    const int32_t *v = s.v + (u64)s.vstride * i;
#pragma unroll
    for (int j = 0; j < 6; ++j) L.f[j] = v[j];
    L.dir = s.dir[(u64)s.dstride * i];
    return L;
}

__device__ __forceinline__ int64_t paf_block(const PafLine &L)
{
    const int64_t a = (int64_t)L.f[1] - L.f[0], b = (int64_t)L.f[3] - L.f[2];
    return a > b ? a : b;
}

// len[i] = bytes of line i for i < n, len[n] = 0 (the exclusive scan then ends with the total)
__global__ void k_paf_len(PafSrc s, u64 n, u64 *__restrict__ len)
{
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n) return;
    if (i == n) { len[n] = 0; return; }
    const PafLine L = paf_line(s, i);
    int b = PAF_CONST_BYTES + paf_name_len(s, L.q) + paf_name_len(s, L.t);
    b += paf_digits(s.len[L.q]) + paf_digits(s.len[L.t]);
#pragma unroll
    for (int j = 0; j < 5; ++j) b += paf_digits_i(L.f[j]);
    b += paf_digits_i(paf_block(L)) + paf_digits_i(L.dir);
    len[i] = (u64)b;
}

__device__ __forceinline__ void paf_format(const PafSrc &s, u64 i, char *p)
{
    const PafLine L = paf_line(s, i);
    p = paf_put_name(s, L.q, p); *p++ = '\t';
    p = paf_put(p, s.len[L.q]); *p++ = '\t';
    p = paf_put(p, L.f[0]); *p++ = '\t';
    p = paf_put(p, L.f[1]); *p++ = '\t';
    *p++ = L.f[5] ? '-' : '+'; *p++ = '\t';
    p = paf_put_name(s, L.t, p); *p++ = '\t';
    p = paf_put(p, s.len[L.t]); *p++ = '\t';
    p = paf_put(p, L.f[2]); *p++ = '\t';
    p = paf_put(p, L.f[3]); *p++ = '\t';
    p = paf_put(p, L.f[4]); *p++ = '\t';
    p = paf_put(p, paf_block(L)); *p++ = '\t';
    *p++ = '2'; *p++ = '5'; *p++ = '5'; *p++ = '\t';
    *p++ = 'd'; *p++ = 'r'; *p++ = ':'; *p++ = 'i'; *p++ = ':';
    p = paf_put(p, L.dir); *p = '\n';
}

// lines [first, first + count) of the source; off = the exclusive scan of k_paf_len (absolute), out = the text of these lines
// (16-byte aligned), line first at out[0]
__global__ void __launch_bounds__(PAF_THREADS) k_paf_write(PafSrc s, const u64 *__restrict__ off, u64 first, u64 count, char *__restrict__ out)
{
    __shared__ uint4 stage4[PAF_STAGE / 16 + 1];
    char *stage = reinterpret_cast<char*>(stage4);
    const u64 l0 = first + (u64)blockIdx.x * PAF_THREADS, end = first + count;
    const u64 l1 = l0 + PAF_THREADS < end ? l0 + PAF_THREADS : end;
    const u64 obase = off[first], b0 = off[l0] - obase, b1 = off[l1] - obase;
    const u64 a0 = b0 & ~15ull;                 // the 16-byte chunk the run starts in
    const u64 i = l0 + threadIdx.x;
    if (b1 - a0 > (u64)PAF_STAGE)
    {
        if (i < l1) paf_format(s, i, out + (off[i] - obase));
        return;
    }
    if (i < l1) paf_format(s, i, stage + (off[i] - obase - a0));
    __syncthreads();
    for (u64 c = a0 + 16ull * threadIdx.x; c < b1; c += 16ull * PAF_THREADS)
    {
        if (c >= b0 && c + 16 <= b1) *reinterpret_cast<uint4*>(out + c) = stage4[(c - a0) >> 4];
        else
        {
            const u64 lo = c > b0 ? c : b0, hi = c + 16 < b1 ? c + 16 : b1;
            for (u64 b = lo; b < hi; ++b) out[b] = stage[b - a0];
        }
    }
}

__global__ void k_paf_flags(const uint8_t *__restrict__ transposed, u64 m, u64 *__restrict__ flag)
{
    const u64 e = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (e <= m) flag[e] = (e < m && transposed[e] == 0) ? 1ull : 0ull;
}

// S entry e with transposed == 0 is line line_of[e].  R entries [r_lo, r_hi) are this rank's alignments, og_src[r] the index
// of entry r's alignment among them; base = global id of read 0 of the job
__global__ void k_paf_string_lines(const uint8_t *__restrict__ transposed, const u64 *__restrict__ line_of, u64 m,
                                   const int64_t *__restrict__ srow, const int64_t *__restrict__ scol, const int32_t *__restrict__ sf,
                                   const u64 *__restrict__ ssrc, int64_t base, const u64 *__restrict__ og_src, u64 r_lo, u64 r_hi,
                                   const int32_t *__restrict__ afields, u32 *__restrict__ q, u32 *__restrict__ t,
                                   int32_t *__restrict__ dir, int32_t *__restrict__ v)
{
    const u64 e = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= m || transposed[e]) return;
    const u64 i = line_of[e], r = ssrc[e];
    q[i] = (u32)(srow[e] - base); t[i] = (u32)(scol[e] - base); dir[i] = sf[4 * e];
    if (r >= r_lo && r < r_hi)
    {
        const int32_t *a = afields + (u64)PAF_XD_FIELDS * og_src[r];
#pragma unroll
        for (int j = 0; j < 6; ++j) v[6 * i + j] = a[j];
    }
    else
    {
#pragma unroll
        for (int j = 0; j < 6; ++j) v[6 * i + j] = 0;
    }
}

} // namespace elba
