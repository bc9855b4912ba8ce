// C ABI of the B200-native ELBA front end (include/elba_fe.h): context, HBM buffers, phase orchestration.
// Host code is C++; CUDA is reached only from here.  sm_100a only, no CPU fallback.
#include "../../include/elba_fe.h"
#include "common.cuh"
#include "kmer_count.cuh"
#include "sketch.cuh"
#include "matrix_build.cuh"
#include "spgemm.cuh"
#include "spgemm2.cuh"
#include "superkmer.cuh"
#include "skm_count.cuh"
#include "xdrop.cuh"
#include "digest.cuh"
#include "fasta_ingest.cuh"
#include "dcsc.cuh"
#include "transitive.cuh"
#include "overlap_graph.cuh"
#include "contigs.cuh"
#include "paf.cuh"
#include "comm.cuh"
#include <cub/cub.cuh>
#include <string>
#include <vector>
#include <cstring>
#include <cstdlib>
#include <cstdio>
#include <cmath>
#include <algorithm>

using namespace elba;

namespace {

thread_local std::string g_create_error;

struct DevBuf
{
    void *p = nullptr; size_t cap = 0;
    template <class T> T *as() const { return reinterpret_cast<T*>(p); }
    cudaError_t ensure(size_t bytes)
    {
        if (bytes <= cap) return cudaSuccess;
        // a buffer that has to grow grows with headroom: sizes that wobble from pass to pass (chunked lists) must not
        // cost a cudaFree + cudaMalloc (a device-wide synchronisation) per pass
        size_t want = (bytes + 255) & ~size_t(255);
        if (p) { cudaFree(p); p = nullptr; cap = 0; want = (want + want / 8 + 255) & ~size_t(255); }
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want; else p = nullptr;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

struct EventPair { cudaEvent_t a = nullptr, b = nullptr; };

// A device buffer other GPUs of the job write into: peer[r] is rank r's buffer mapped into this process (CUDA IPC),
// peer[me] the local one.  With one rank it is a plain buffer.
struct Window { DevBuf buf; void *peer[elba::SK_MAXW] = {}; bool mapped = false; };

// geometry of the bucket count kernel (skm_count.cuh): 4 CTAs x 256 threads per SM, 2048-slot tables, 960-record staging buffers
constexpr int SK4_THREADS = 256, SK4_SLOTS = 2048, SK4_RMAX = 736, SK4_POOL = 1536, SK4_RETRY = 64, SK4_MINB = 4;

} // namespace

struct elba_fe_ctx
{
    elba_fe_config cfg;
    cudaStream_t stream = nullptr; bool own_stream = false;
    int sm_count = 148;
    std::string err;
    int phase = 0;                      // 0 none, 1 reads, 2 counted, 3 A built, 4 B built
    // reads
    DevBuf packed, off, len64, len32, chunk_start, kmer_start, nks_start;
    u32 n = 0; u64 packed_bytes = 0, nchunks = 0, M = 0, Ms = 0; int64_t read_id_offset = 0;
    // an upload from host memory arrives in slices on a second stream; the scatter of slice s starts when slice s + 1 is there
    static constexpr int UP_SLICES = 8;
    int up_n = 0; u64 up_chunk_end[UP_SLICES] = {}; cudaEvent_t up_ev[UP_SLICES] = {}; cudaEvent_t up_t0 = nullptr;
    // counting
    DevBuf table, cand, ctr, partbuf, phist, pcursor, rel_key, rel_cnt, rel_key_s, rel_cnt_s, lut, filter;
    DevBuf plan, bfill, ovf, scratch[2];
    u64 ovf_cap = 0;
    DevBuf skm_slab, skm_fill, skm_ovf;      // super-k-mer path: record slabs, per-bucket fill, overflow records
    u64 skm_ovf_cap = 0;
    bool seeds_fused = false; u64 nseeds_fused = 0;      // counting already wrote the seed list (ctx->seeds) of this pass
    DevBuf seeds, perm, rel_idx, rel_idx_s;              // super-k-mer path: {list index, pos, read} seeds; list index -> column id; sort payload
    u64 seed_cap = 0, seed_id_base = 0; double hist_dm = 0.0;              // seed-list capacity; distinct / instances of the last pass (sizes the buckets)
    u64 skm_reliable = 0;                                // super-k-mer path: reliable k-mers among the (holey) list entries handed out
    // several GPUs, super-k-mer path: every GPU parses its own reads and writes the records into the owners' slabs (peer memory)
    Window w_slab, w_ovf, w_octr, w_rkey, w_rpos, w_rcnt;     // record slabs, overflow list + its counters, routed seed triples + their counts
    DevBuf agpad, skm_fillin, skm_plan, skm_stage, skm_foff, skm_inoff, d_roff, route_cur, rel_gid, glob_key, glob_cnt, glob_gid, glob_cnt_in;
    std::vector<u64> roff;                                   // [W + 1] first global read id of every rank's block
    int64_t read_base0 = 0;                                  // global id of the first read of rank 0
    bool p2p = false, kmers_distributed = false; u64 R_local = 0; std::vector<u64> rel_counts;
    u64 Ms_total = 0, Ms_max = 0, route_cap = 0; u64 setup_sig[3] = {0, 0, 0}; bool setup_valid = false;
    cudaStream_t aux = nullptr; cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_x0 = nullptr, ev_x1 = nullptr;
    u64 exchange_bytes = 0, panel_bytes = 0;
    u64 scratch_mb = 64;
    u32 lut_slots = 0; u64 rel_cap = 0; u32 filter_words = 0; u64 cand_cap = 0;
    // A
    DevBuf seed_key, seed_pos, seed_key2, seed_pos2, idx, a_key, a_rowptr, a_col, a_pos, at_key, at_key2, at_pos2, at_colptr, at_row, at_pos, prod;
    int col_bits = 1, read_bits = 1; bool at_built = false;
    // B
    DevBuf sp_ptr, sp_ent;               // the right operand by column as the SpGEMM reads it: 32-bit column pointers, {row, pos} entries
    DevBuf at_ptr32, at_ent, lp_ptr, lp_ent, sp_col, sp_col2, sp_val, sp_val2, tup_cnt, tup_cur, tuples;      // left operand by column (several GPUs); sort scratch; tuple regions
    const u32 *op_l_cptr = nullptr; const uint2 *op_l_cent = nullptr; u32 op_r_rows = 0;
    DevBuf xd_flag, xd_rowof, xd_prow, xd_pcol, xd_sq, xd_st, xd_nz, xd_out, xd_scratch, xd_max;      // elba_fe_align
    u64 xd_pairs = 0; bool xd_done = false; cudaEvent_t xd_e0 = nullptr, xd_e1 = nullptr;
    DevBuf t_col, t_num, t_seeds, row_off, row_nnz, bins, small_rows, mid_rows, big_rows, ovf_rows, gscratch, b_rowptr, b_col, b_num, b_seeds;
    u64 b_cap_hint = 0;
    DevBuf cubtmp, hll_regs, bloom;
    DevBuf tr_in_row, tr_in_col, tr_in_f, tr_key, tr_key2, tr_val, tr_val2, tr_head, tr_okey, tr_row, tr_col, tr_dir, tr_dirT, tr_suf, tr_sufT, tr_src, tr_tr,
           tr_rowptr, tr_I, tr_T, tr_keep, tr_orow, tr_ocol, tr_of, tr_osrc, tr_otr;      // elba_fe_transitive_reduction
    u64 tr_out = 0; bool tr_done = false;
    bool tr_resident = false;                               // the tr_* output is the reduction of the current resident R (not of a host R)
    // elba_fe_overlap_graph: contained flags, keep scan, this rank's kept alignments (several GPUs), the whole R (job-relative ids)
    DevBuf og_cont, og_keep, og_lrow, og_lcol, og_lf, og_lsrc, og_row, og_col, og_f, og_src;
    // og_aligned: the resident alignments are those of the current B (count, build_A and spgemm clear it, align sets it)
    u64 og_nnz = 0, og_nreads = 0; int64_t og_base = 0; std::vector<u64> og_counts; bool og_aligned = false, og_done = false; cudaEvent_t og_e0 = nullptr, og_e1 = nullptr;
    DevBuf xa_buf, xa_off, xa_len;                          // elba_fe_align on several GPUs: arena and read tables of all ranks
    u64 read_gen = 0, xd_read_gen = 0;                      // bumped by every upload / set / ingest of reads; its value at elba_fe_align
    // elba_fe_contigs: S uploaded by contigs_from_graph, per-read scratch, the layout, this rank's sequences
    DevBuf ct_in_row, ct_in_col, ct_in_f, ct_ptr, ct_branch, ct_slot, ct_succ[2], ct_dist[2], ct_mn[2], ct_cyc, ct_flag, ct_start, ct_pos, ct_next, ct_L,
           ct_cptr, ct_read, ct_rev, ct_beg, ct_end, ct_boff, ct_blen, ct_bbyte, ct_packed;
    elba_fe_contig_info_t ct_info; bool ct_done = false; cudaEvent_t ct_e0 = nullptr, ct_e1 = nullptr;
    // elba_fe_paf: read names of the job (char arena + offsets), line lengths / offsets, string-graph lines, the text of this rank
    DevBuf pf_names, pf_noff, pf_len, pf_flag, pf_q, pf_t, pf_dir, pf_v, pf_text;
    u64 pf_nnames = 0; bool pf_has_names = false;
    elba_fe_paf_info_t pf_info; bool pf_done = false; cudaEvent_t pf_e0 = nullptr, pf_e1 = nullptr;
    DevBuf fa_raw, fa_rec, fa_items;                       // elba_fe_ingest_fasta: the raw FASTA chunk, its .fai records, first work item of every read
    DevBuf dc_key, dc_key2, dc_val, dc_val2, dc_head, dc_jc, dc_cp, dc_ir, dc_num, dc_seeds; u64 dc_nzc = 0; bool dc_built = false;      // B by column (DCSC)
    // multi-GPU
    Comm comm;
    u64 N_total = 0;
    DevBuf recvbuf, recvcnt, tmp64, rel_all_key, rel_all_cnt, g_key, g_pos, pack_key, l_rowptr, l_col, r_key, r_key2, r_pos, r_colptr, r_row, r_ptr;
    // SpGEMM operands: left rows (CSR) x right rows by column (CSC); one GPU: A and its transpose
    struct { const int64_t *l_rowptr; const u32 *l_col, *l_pos; u32 l_rows; u64 l_nnz; const int64_t *r_colptr; const u32 *r_row, *r_pos; u64 r_nnz; int64_t row0, col0; } op;
    u32 b_rows = 0;
    elba_fe_sizes_t sz;
    elba_fe_timings_t tm;
    cudaEvent_t ev[8];
    bool trace = false; std::vector<std::pair<const char*, cudaEvent_t>> marks; size_t marks_used = 0;      // ELBA_FE_TRACE=1: sub-phase device times on stderr
    std::vector<EventPair> kev; size_t kev_used = 0;      // per-kernel event pairs (count kernels)
    std::vector<EventPair> sev; size_t sev_used = 0;      // spgemm numeric kernels
    std::vector<EventPair> pev; size_t pev_used = 0;      // partition kernels
    std::vector<EventPair> lev; size_t lev_used = 0;      // lookup kernel
};

extern "C" { static void window_release(elba_fe_ctx *ctx, Window &w); }

namespace {

int fail(elba_fe_ctx *c, int code, const std::string &msg) { if (c) c->err = msg; else g_create_error = msg; return code; }

#define CK(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) { \
    return fail(ctx, e__ == cudaErrorMemoryAllocation ? ELBA_FE_ERR_OOM : ELBA_FE_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__)); } } while (0)
#define CKL() CK(cudaGetLastError())
#define LAUNCHED(ctx) ((ctx)->tm.kernel_launches++)

inline u32 nblk(u64 n, u32 b) { return (u32)((n + b - 1) / b); }
inline u64 next_pow2(u64 v) { u64 p = 1; while (p < v) p <<= 1; return p; }
inline int bits_for(u64 v) { int b = 1; while ((1ull << b) < v) ++b; return b; }   // bits to hold values < v

EventPair &next_pair(std::vector<EventPair> &v, size_t &used)
{
    if (used == v.size()) { EventPair p; cudaEventCreate(&p.a); cudaEventCreate(&p.b); v.push_back(p); }
    return v[used++];
}
float sum_pairs(std::vector<EventPair> &v, size_t used)
{
    float tot = 0; for (size_t i = 0; i < used; ++i) { float ms = 0; if (cudaEventElapsedTime(&ms, v[i].a, v[i].b) == cudaSuccess) tot += ms; } return tot;
}

ReadsView view(elba_fe_ctx *c)
{
    ReadsView rv; rv.buf = c->packed.as<uint8_t>(); rv.off = c->off.as<u64>(); rv.len = c->len32.as<u32>();
    rv.chunk_start = c->chunk_start.as<u64>(); rv.kmer_start = c->kmer_start.as<u64>(); rv.n = c->n; rv.nchunks = c->nchunks;
    return rv;
}

template <class T> int exclusive_scan_inplace(elba_fe_ctx *ctx, T *d, u64 n)
{
    size_t need = 0;
    CK(cub::DeviceScan::ExclusiveSum(nullptr, need, d, d, (int64_t)n, ctx->stream));
    CK(ctx->cubtmp.ensure(need));
    CK(cub::DeviceScan::ExclusiveSum(ctx->cubtmp.p, need, d, d, (int64_t)n, ctx->stream));
    ctx->tm.kernel_launches += 2;
    return 0;
}

int sort_pairs(elba_fe_ctx *ctx, const u64 *kin, u64 *kout, const u32 *vin, u32 *vout, u64 n, int begin_bit, int end_bit)
{
    if (n == 0) return 0;
    size_t need = 0;
    CK(cub::DeviceRadixSort::SortPairs(nullptr, need, kin, kout, vin, vout, (int64_t)n, begin_bit, end_bit, ctx->stream));
    CK(ctx->cubtmp.ensure(need));
    CK(cub::DeviceRadixSort::SortPairs(ctx->cubtmp.p, need, kin, kout, vin, vout, (int64_t)n, begin_bit, end_bit, ctx->stream));
    ctx->tm.kernel_launches += (u32)((end_bit - begin_bit + 7) / 8 + 1);
    return 0;
}

int sort_pairs_u32_u64(elba_fe_ctx *ctx, const u32 *kin, u32 *kout, const u64 *vin, u64 *vout, u64 n, int begin_bit, int end_bit)
{
    if (n == 0) return 0;
    size_t need = 0;
    CK(cub::DeviceRadixSort::SortPairs(nullptr, need, kin, kout, vin, vout, (int64_t)n, begin_bit, end_bit, ctx->stream));
    CK(ctx->cubtmp.ensure(need));
    CK(cub::DeviceRadixSort::SortPairs(ctx->cubtmp.p, need, kin, kout, vin, vout, (int64_t)n, begin_bit, end_bit, ctx->stream));
    ctx->tm.kernel_launches += (u32)((end_bit - begin_bit + 7) / 8 + 1);
    return 0;
}

int grid_for(elba_fe_ctx *c, int per_sm) { return c->sm_count * per_sm; }

// ELBA_FE_TRACE=1: record a named point of the stream; trace_flush prints the device time between consecutive points
void mark(elba_fe_ctx *c, const char *name)
{
    if (!c->trace) return;
    if (c->marks_used == c->marks.size()) { cudaEvent_t e; cudaEventCreate(&e); c->marks.push_back({name, e}); }
    c->marks[c->marks_used].first = name;
    cudaEventRecord(c->marks[c->marks_used++].second, c->stream);
}
void trace_flush(elba_fe_ctx *c, const char *phase)
{
    if (!c->trace || c->marks_used < 2) { c->marks_used = 0; return; }
    cudaStreamSynchronize(c->stream);
    std::string line = std::string("[elba_fe trace] rank ") + std::to_string(c->comm.rank) + " " + phase + ":";
    for (size_t i = 1; i < c->marks_used; ++i)
    {
        float ms = 0; cudaEventElapsedTime(&ms, c->marks[i - 1].second, c->marks[i].second);
        char b[96]; snprintf(b, sizeof b, " %s %.3f", c->marks[i].first, ms); line += b;
    }
    fprintf(stderr, "%s\n", line.c_str());
    c->marks_used = 0;
}

// after the reads are resident: per-read tables and totals
int prepare_reads(elba_fe_ctx *ctx)
{
    u32 n = ctx->n;
    CK(ctx->len32.ensure(sizeof(u32) * (size_t)(n + 1)));
    CK(ctx->chunk_start.ensure(sizeof(u64) * (size_t)(n + 1)));
    CK(ctx->kmer_start.ensure(sizeof(u64) * (size_t)(n + 1)));
    CK(ctx->nks_start.ensure(sizeof(u64) * (size_t)(n + 1)));
    k_prep_reads<<<nblk((u64)n + 1, 256), 256, 0, ctx->stream>>>(ctx->len64.as<u64>(), n, ctx->cfg.k, ctx->cfg.stride,
        ctx->len32.as<u32>(), ctx->chunk_start.as<u64>(), ctx->kmer_start.as<u64>(), ctx->nks_start.as<u64>());
    CKL(); LAUNCHED(ctx);
    int rc;
    if ((rc = exclusive_scan_inplace(ctx, ctx->chunk_start.as<u64>(), (u64)n + 1))) return rc;
    if ((rc = exclusive_scan_inplace(ctx, ctx->kmer_start.as<u64>(), (u64)n + 1))) return rc;
    if ((rc = exclusive_scan_inplace(ctx, ctx->nks_start.as<u64>(), (u64)n + 1))) return rc;
    u64 tot[3];
    CK(cudaMemcpyAsync(&tot[0], ctx->chunk_start.as<u64>() + n, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&tot[1], ctx->kmer_start.as<u64>() + n, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&tot[2], ctx->nks_start.as<u64>() + n, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->nchunks = tot[0]; ctx->M = tot[1]; ctx->Ms = tot[2];
    std::memset(&ctx->sz, 0, sizeof ctx->sz);
    ctx->sz.nreads = n; ctx->sz.num_kmers = ctx->Ms;
    ctx->phase = 1;
    return 0;
}

} // namespace

extern "C" {

int elba_fe_version(void) { return ELBA_FE_VERSION; }

int elba_fe_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

void elba_fe_default_config(elba_fe_config *cfg)
{
    std::memset(cfg, 0, sizeof *cfg);
    cfg->k = 31; cfg->lower = 15; cfg->upper = 35;     /* reference Makefile:1-3 */
    cfg->stride = 1; cfg->seed_count = 2; cfg->device = 0; cfg->num_partitions = 0; cfg->flags = 0;
}

const char *elba_fe_last_error(const elba_fe_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int elba_fe_create(const elba_fe_config *cfg, elba_fe_ctx **out)
{
    elba_fe_ctx *ctx = nullptr;
    if (!cfg || !out) return fail(nullptr, ELBA_FE_ERR_INVALID, "null argument");
    *out = nullptr;
    if (cfg->k < 3 || cfg->k > ELBA_FE_MAX_KMER_SIZE) return fail(nullptr, ELBA_FE_ERR_INVALID, "k must be in 3..32 (one 64-bit word, include/Kmer.hpp:95-97)");
    if (cfg->stride < 1) return fail(nullptr, ELBA_FE_ERR_INVALID, "stride must be >= 1");
    if (cfg->seed_count < 1 || cfg->seed_count > 2) return fail(nullptr, ELBA_FE_ERR_INVALID, "seed_count must be 1 or 2 (SharedSeeds::seeds[2], include/SharedSeeds.hpp:94)");
    if (cfg->lower < 2) return fail(nullptr, ELBA_FE_ERR_INVALID, "lower must be >= 2: with LOWER_KMER_FREQ=1 the reference's result depends on Bloom false positives");
    if (cfg->upper < cfg->lower || cfg->upper > 65535) return fail(nullptr, ELBA_FE_ERR_INVALID, "need lower <= upper <= 65535 (include/compiletime.h:21)");
    if (cfg->num_partitions < 0 || cfg->num_partitions > 4096) return fail(nullptr, ELBA_FE_ERR_INVALID, "num_partitions must be in 0..4096");
    if (cfg->flags != 0) return fail(nullptr, ELBA_FE_ERR_INVALID, "unsupported flags");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, ELBA_FE_ERR_NO_DEVICE, std::string("no CUDA device (there is no CPU fallback): ") + cudaGetErrorString(e));
    if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, ELBA_FE_ERR_INVALID, "device ordinal out of range");
    e = cudaSetDevice(cfg->device);
    if (e != cudaSuccess) return fail(nullptr, ELBA_FE_ERR_CUDA, cudaGetErrorString(e));
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, cfg->device);
    if (e != cudaSuccess) return fail(nullptr, ELBA_FE_ERR_CUDA, cudaGetErrorString(e));
    if (prop.major != 10 || prop.minor != 0) return fail(nullptr, ELBA_FE_ERR_NO_DEVICE, "device is not sm_100 (this library carries sm_100a code only)");
    ctx = new elba_fe_ctx;
    ctx->cfg = *cfg;
    ctx->sm_count = prop.multiProcessorCount;
    std::memset(&ctx->sz, 0, sizeof ctx->sz); std::memset(&ctx->tm, 0, sizeof ctx->tm);
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return fail(nullptr, ELBA_FE_ERR_CUDA, "cudaStreamCreate failed"); }
    ctx->own_stream = true;
    for (auto &ev : ctx->ev) cudaEventCreate(&ev);
    // random 16-byte table probes: do not let L2 pull whole 128-byte lines from HBM for them (profiles/r1_count_v0.md)
    cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, 32);
    cudaStreamCreateWithFlags(&ctx->aux, cudaStreamNonBlocking);
    for (auto &e : ctx->up_ev) cudaEventCreate(&e);
    cudaEventCreate(&ctx->up_t0);
    cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming); cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming);
    cudaEventCreate(&ctx->ev_x0); cudaEventCreate(&ctx->ev_x1); cudaEventCreate(&ctx->xd_e0); cudaEventCreate(&ctx->xd_e1);
    cudaEventCreate(&ctx->og_e0); cudaEventCreate(&ctx->og_e1); cudaEventCreate(&ctx->ct_e0); cudaEventCreate(&ctx->ct_e1);
    cudaEventCreate(&ctx->pf_e0); cudaEventCreate(&ctx->pf_e1);
    if (ctx->tmp64.ensure(8192) != cudaSuccess || ctx->ctr.ensure(128) != cudaSuccess) { elba_fe_destroy(ctx); return fail(nullptr, ELBA_FE_ERR_OOM, "cudaMalloc failed"); }
    if (const char *e = getenv("ELBA_FE_TRACE")) ctx->trace = atoi(e) != 0;
    if (const char *e = getenv("ELBA_FE_SCRATCH_MB")) { long v = atol(e); if (v >= 8 && v <= 65536) ctx->scratch_mb = (u64)v; }
    // opt in to large dynamic shared memory
    cudaFuncSetAttribute(k_scatter1<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(u64) * S1_TILE + 2 * sizeof(u32) * MAX_P1));
    cudaFuncSetAttribute(k_scatter1<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(u64) * S1_TILE + 2 * sizeof(u32) * MAX_P1));
    cudaFuncSetAttribute(k_scatter2<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(u64) * S2_TILE + 2 * sizeof(u32) * MAX_P2));
    cudaFuncSetAttribute(k_scatter2<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(u64) * S2_TILE + 2 * sizeof(u32) * MAX_P2));
    cudaFuncSetAttribute(k_count_buckets, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)((sizeof(u64) + sizeof(u32)) * BUCKET_SLOTS));
    if (cudaFuncSetAttribute(k_skm_count4<SK4_THREADS, SK4_SLOTS, SK4_RMAX, SK4_POOL, SK4_RETRY, SK4_MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sk4_smem(SK4_SLOTS, SK4_RMAX, SK4_POOL, SK4_RETRY, SK4_THREADS)) != cudaSuccess)
    { elba_fe_destroy(ctx); return fail(nullptr, ELBA_FE_ERR_CUDA, "cudaFuncSetAttribute(k_skm_count4) failed"); }
    *out = ctx;
    return 0;
}

int elba_fe_destroy(elba_fe_ctx *ctx)
{
    if (!ctx) return 0;
    cudaSetDevice(ctx->cfg.device);
    cudaStreamSynchronize(ctx->stream);
    DevBuf *all[] = { &ctx->packed, &ctx->off, &ctx->len64, &ctx->len32, &ctx->chunk_start, &ctx->kmer_start, &ctx->nks_start,
        &ctx->table, &ctx->cand, &ctx->ctr, &ctx->partbuf, &ctx->phist, &ctx->pcursor, &ctx->rel_key, &ctx->rel_cnt, &ctx->rel_key_s, &ctx->rel_cnt_s, &ctx->lut, &ctx->filter,
        &ctx->seed_key, &ctx->seed_pos, &ctx->seed_key2, &ctx->seed_pos2, &ctx->idx, &ctx->a_key, &ctx->a_rowptr, &ctx->a_col, &ctx->a_pos,
        &ctx->at_key, &ctx->at_key2, &ctx->at_pos2, &ctx->at_colptr, &ctx->at_row, &ctx->at_pos, &ctx->prod,
        &ctx->t_col, &ctx->t_num, &ctx->t_seeds, &ctx->row_off, &ctx->row_nnz, &ctx->sp_ptr, &ctx->sp_ent, &ctx->at_ptr32, &ctx->at_ent, &ctx->lp_ptr, &ctx->lp_ent, &ctx->sp_col, &ctx->sp_col2, &ctx->sp_val, &ctx->sp_val2, &ctx->tup_cnt, &ctx->tup_cur, &ctx->tuples, &ctx->xd_flag, &ctx->xd_rowof, &ctx->xd_prow, &ctx->xd_pcol, &ctx->xd_sq, &ctx->xd_st, &ctx->xd_nz, &ctx->xd_out, &ctx->xd_scratch, &ctx->xd_max, &ctx->agpad, &ctx->skm_fillin, &ctx->skm_plan, &ctx->skm_stage, &ctx->skm_foff, &ctx->skm_inoff, &ctx->d_roff, &ctx->route_cur, &ctx->rel_gid, &ctx->glob_key, &ctx->glob_cnt, &ctx->glob_gid, &ctx->glob_cnt_in, &ctx->bins, &ctx->small_rows, &ctx->mid_rows, &ctx->big_rows, &ctx->ovf_rows, &ctx->gscratch,
        &ctx->b_rowptr, &ctx->b_col, &ctx->b_num, &ctx->b_seeds, &ctx->cubtmp, &ctx->hll_regs, &ctx->bloom,
        &ctx->tr_in_row, &ctx->tr_in_col, &ctx->tr_in_f, &ctx->tr_key, &ctx->tr_key2, &ctx->tr_val, &ctx->tr_val2, &ctx->tr_head, &ctx->tr_okey, &ctx->tr_row, &ctx->tr_col,
        &ctx->tr_dir, &ctx->tr_dirT, &ctx->tr_suf, &ctx->tr_sufT, &ctx->tr_src, &ctx->tr_tr, &ctx->tr_rowptr, &ctx->tr_I, &ctx->tr_T, &ctx->tr_keep, &ctx->tr_orow, &ctx->tr_ocol,
        &ctx->tr_of, &ctx->tr_osrc, &ctx->tr_otr,
        &ctx->og_cont, &ctx->og_keep, &ctx->og_lrow, &ctx->og_lcol, &ctx->og_lf, &ctx->og_lsrc, &ctx->og_row, &ctx->og_col, &ctx->og_f, &ctx->og_src,
        &ctx->xa_buf, &ctx->xa_off, &ctx->xa_len,
        &ctx->ct_in_row, &ctx->ct_in_col, &ctx->ct_in_f, &ctx->ct_ptr, &ctx->ct_branch, &ctx->ct_slot, &ctx->ct_succ[0], &ctx->ct_succ[1], &ctx->ct_dist[0], &ctx->ct_dist[1],
        &ctx->ct_mn[0], &ctx->ct_mn[1], &ctx->ct_cyc, &ctx->ct_flag, &ctx->ct_start, &ctx->ct_pos, &ctx->ct_next, &ctx->ct_L, &ctx->ct_cptr, &ctx->ct_read, &ctx->ct_rev,
        &ctx->ct_beg, &ctx->ct_end, &ctx->ct_boff, &ctx->ct_blen, &ctx->ct_bbyte, &ctx->ct_packed,
        &ctx->pf_names, &ctx->pf_noff, &ctx->pf_len, &ctx->pf_flag, &ctx->pf_q, &ctx->pf_t, &ctx->pf_dir, &ctx->pf_v, &ctx->pf_text, &ctx->fa_raw, &ctx->fa_rec, &ctx->fa_items, &ctx->dc_key, &ctx->dc_key2, &ctx->dc_val, &ctx->dc_val2, &ctx->dc_head, &ctx->dc_jc, &ctx->dc_cp, &ctx->dc_ir, &ctx->dc_num, &ctx->dc_seeds,
        &ctx->plan, &ctx->bfill, &ctx->ovf, &ctx->scratch[0], &ctx->scratch[1], &ctx->skm_slab, &ctx->skm_fill, &ctx->skm_ovf, &ctx->seeds, &ctx->perm, &ctx->rel_idx, &ctx->rel_idx_s,
        &ctx->recvbuf, &ctx->recvcnt, &ctx->tmp64, &ctx->rel_all_key, &ctx->rel_all_cnt, &ctx->g_key, &ctx->g_pos, &ctx->pack_key, &ctx->l_rowptr, &ctx->l_col,
        &ctx->r_key, &ctx->r_key2, &ctx->r_pos, &ctx->r_colptr, &ctx->r_row, &ctx->r_ptr };
    for (Window *w : { &ctx->w_slab, &ctx->w_ovf, &ctx->w_octr, &ctx->w_rkey, &ctx->w_rpos, &ctx->w_rcnt }) window_release(ctx, *w);
    for (DevBuf *b : all) b->release();
    for (auto &ev : ctx->ev) cudaEventDestroy(ev);
    for (auto *v : { &ctx->kev, &ctx->sev, &ctx->pev, &ctx->lev }) for (auto &p : *v) { cudaEventDestroy(p.a); cudaEventDestroy(p.b); }
    if (ctx->comm.comm) ctx->comm.api->CommDestroy(ctx->comm.comm);
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    if (ctx->aux) cudaStreamDestroy(ctx->aux);
    for (auto &e : ctx->up_ev) if (e) cudaEventDestroy(e);
    if (ctx->up_t0) cudaEventDestroy(ctx->up_t0);
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
    if (ctx->ev_x0) cudaEventDestroy(ctx->ev_x0);
    if (ctx->ev_x1) cudaEventDestroy(ctx->ev_x1);
    if (ctx->xd_e0) cudaEventDestroy(ctx->xd_e0);
    if (ctx->xd_e1) cudaEventDestroy(ctx->xd_e1);
    if (ctx->og_e0) cudaEventDestroy(ctx->og_e0);
    if (ctx->og_e1) cudaEventDestroy(ctx->og_e1);
    if (ctx->ct_e0) cudaEventDestroy(ctx->ct_e0);
    if (ctx->ct_e1) cudaEventDestroy(ctx->ct_e1);
    if (ctx->pf_e0) cudaEventDestroy(ctx->pf_e0);
    if (ctx->pf_e1) cudaEventDestroy(ctx->pf_e1);
    delete ctx;
    return 0;
}

int elba_fe_set_stream(elba_fe_ctx *ctx, void *cuda_stream)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->own_stream) { cudaStreamDestroy(ctx->stream); ctx->own_stream = false; }
    ctx->stream = (cudaStream_t)cuda_stream;
    return 0;
}

int elba_fe_synchronize(elba_fe_ctx *ctx) { if (!ctx) return ELBA_FE_ERR_INVALID; CK(cudaStreamSynchronize(ctx->stream)); return 0; }

// every consumer of the arena other than the sliced scatter: the whole upload must have arrived
static int wait_reads(elba_fe_ctx *ctx)
{
    if (ctx->up_n > 0) CK(cudaStreamWaitEvent(ctx->stream, ctx->up_ev[ctx->up_n - 1], 0));
    return 0;
}

static int stage_reads(elba_fe_ctx *ctx, const uint8_t *packed, uint64_t packed_bytes, const uint64_t *byte_off, const uint64_t *len,
                       uint64_t nreads, int64_t read_id_offset, cudaMemcpyKind kind)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (nreads >= 0xFFFFFFF0ull) return fail(ctx, ELBA_FE_ERR_INVALID, "too many reads for one context (local read ids are 32-bit)");
    if (nreads && (!byte_off || !len)) return fail(ctx, ELBA_FE_ERR_INVALID, "null read tables");
    if (packed_bytes && !packed) return fail(ctx, ELBA_FE_ERR_INVALID, "null arena");
    CK(cudaSetDevice(ctx->cfg.device));
    ctx->phase = 0; ++ctx->read_gen; ctx->ct_done = ctx->pf_done = false;
    ctx->n = (u32)nreads; ctx->packed_bytes = packed_bytes; ctx->read_id_offset = read_id_offset;
    cudaStream_t st = ctx->stream;
    CK(cudaEventRecord(ctx->ev[0], st));
    CK(ctx->packed.ensure(packed_bytes + 64));
    CK(ctx->off.ensure(sizeof(u64) * (size_t)(nreads + 1)));
    CK(ctx->len64.ensure(sizeof(u64) * (size_t)(nreads + 1)));
    // A large arena coming from the host travels in slices on the second stream while the read tables are prepared and the
    // first slices are already parsed (count_superkmers).  The caller's buffer must stay valid until the next call that
    // synchronises (elba_fe_count / elba_fe_run do).
    const bool sliced = kind == cudaMemcpyHostToDevice && packed_bytes >= (64ull << 20) && nreads >= 4096;
    ctx->up_n = 0;
    // the read tables first: a copy engine serves its copies in issue order, and the table preparation must not queue behind the arena
    if (nreads)
    {
        CK(cudaMemcpyAsync(ctx->off.p, byte_off, sizeof(u64) * nreads, kind, st));
        CK(cudaMemcpyAsync(ctx->len64.p, len, sizeof(u64) * nreads, kind, st));
    }
    std::vector<u64> slice_read;                         // first read of every slice (host side: byte_off is a host array here)
    if (sliced)
    {
        const int S = elba_fe_ctx::UP_SLICES;
        CK(cudaEventRecord(ctx->ev_fork, st));           // the previous pass has finished with the old arena before it is overwritten
        CK(cudaStreamWaitEvent(ctx->aux, ctx->ev_fork, 0));
        CK(cudaEventRecord(ctx->up_t0, ctx->aux));
        slice_read.assign(S + 1, nreads);
        slice_read[0] = 0;
        for (int i = 1; i < S; ++i) slice_read[i] = (u64)(std::lower_bound(byte_off, byte_off + nreads, packed_bytes / S * (u64)i) - byte_off);
        for (int i = 0; i < S; ++i)
        {
            const u64 b0 = slice_read[i] < nreads ? byte_off[slice_read[i]] : packed_bytes, b1 = slice_read[i + 1] < nreads ? byte_off[slice_read[i + 1]] : packed_bytes;
            if (b1 > b0) CK(cudaMemcpyAsync(ctx->packed.as<uint8_t>() + b0, packed + b0, b1 - b0, kind, ctx->aux));
            if (i == S - 1) CK(cudaMemsetAsync(ctx->packed.as<uint8_t>() + packed_bytes, 0, 64, ctx->aux));
            CK(cudaEventRecord(ctx->up_ev[i], ctx->aux));
        }
        ctx->up_n = S;
    }
    else
    {
        CK(cudaMemsetAsync(ctx->packed.as<uint8_t>() + packed_bytes, 0, 64, st));
        if (packed_bytes) CK(cudaMemcpyAsync(ctx->packed.p, packed, packed_bytes, kind, st));
    }
    CK(cudaEventRecord(ctx->ev[1], st));
    int rc = prepare_reads(ctx);
    if (rc) return rc;
    if (sliced)
    {
        // chunk index where every slice ends (the scatter is launched per slice)
        const int S = elba_fe_ctx::UP_SLICES;
        u64 ends[elba_fe_ctx::UP_SLICES];
        for (int i = 0; i < S; ++i) CK(cudaMemcpyAsync(&ends[i], ctx->chunk_start.as<u64>() + slice_read[i + 1], 8, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        for (int i = 0; i < S; ++i) ctx->up_chunk_end[i] = ends[i];
    }
    float ms = 0; cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]); ctx->tm.upload_ms = ms;
    return 0;
}

int elba_fe_upload_reads(elba_fe_ctx *ctx, const uint8_t *packed, uint64_t packed_bytes, const uint64_t *byte_off, const uint64_t *len,
                         uint64_t nreads, int64_t read_id_offset)
{
    return stage_reads(ctx, packed, packed_bytes, byte_off, len, nreads, read_id_offset, cudaMemcpyHostToDevice);
}

int elba_fe_set_reads_device(elba_fe_ctx *ctx, const uint8_t *d_packed, uint64_t packed_bytes, const uint64_t *d_byte_off, const uint64_t *d_len,
                             uint64_t nreads, int64_t read_id_offset)
{
    // device-to-device into the context's padded, aligned arena (the parse kernels read whole 32-bit words past a read's last byte)
    return stage_reads(ctx, d_packed, packed_bytes, d_byte_off, d_len, nreads, read_id_offset, cudaMemcpyDeviceToDevice);
}

// ---- the step before the path: FASTA ingest (fasta_ingest.cuh) ---------------------------------------------------
// FastaIndex::getmydna (src/FastaIndex.cpp:191-290): the rank's chunk of the file + the .fai records of its reads -> DnaBuffer.
// The raw chunk crosses PCIe in slices on the second stream; the pack kernel of a slice starts when the slice is there.
int elba_fe_ingest_fasta(elba_fe_ctx *ctx, const char *chunk, uint64_t chunk_bytes, uint64_t chunk_pos, const uint64_t *records,
                         uint64_t nreads, int64_t read_id_offset)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (nreads >= 0xFFFFFFF0ull) return fail(ctx, ELBA_FE_ERR_INVALID, "too many reads for one context (local read ids are 32-bit)");
    if (nreads && !records) return fail(ctx, ELBA_FE_ERR_INVALID, "null FASTA index records");
    if (chunk_bytes && !chunk) return fail(ctx, ELBA_FE_ERR_INVALID, "null FASTA chunk");
    CK(cudaSetDevice(ctx->cfg.device));
    // layout of the arena (DnaBuffer::computebufsize, src/DnaBuffer.cpp:16-20) and of the work items; every record must lie in the chunk
    std::vector<u64> off(nreads + 1), items(nreads + 1), len(nreads ? nreads : 1);
    u64 head = 0, nitems = 0; bool ordered = true; u64 prev_end = chunk_pos;
    for (u64 r = 0; r < nreads; ++r)
    {
        const u64 l = records[3 * r], pos = records[3 * r + 1], bases = records[3 * r + 2];
        off[r] = head; items[r] = nitems; len[r] = l;
        if (pos < prev_end || pos - chunk_pos > chunk_bytes) ordered = false;      // (an empty read's position is never dereferenced)
        if (l)
        {
            if (bases == 0) return fail(ctx, ELBA_FE_ERR_INVALID, "FASTA index record with zero bases per line");
            if (pos < chunk_pos) return fail(ctx, ELBA_FE_ERR_INVALID, "FASTA index record starts before the chunk");
            const u64 last = pos + (l - 1) + (l - 1) / bases;          // file offset of the read's last base
            if (last < pos || last - chunk_pos >= chunk_bytes) return fail(ctx, ELBA_FE_ERR_INVALID, "FASTA index record ends behind the chunk");
            prev_end = last + 1;
        }
        const u64 nb = (l + 3) / 4;
        head += nb; nitems += (nb + FI_ITEM_BYTES - 1) / FI_ITEM_BYTES;
    }
    off[nreads] = head; items[nreads] = nitems;
    ctx->phase = 0; ++ctx->read_gen; ctx->ct_done = ctx->pf_done = false;
    ctx->n = (u32)nreads; ctx->packed_bytes = head; ctx->read_id_offset = read_id_offset; ctx->up_n = 0;
    cudaStream_t st = ctx->stream;
    CK(cudaEventRecord(ctx->ev[0], st));
    CK(ctx->packed.ensure(head + 64));
    CK(ctx->off.ensure(sizeof(u64) * (size_t)(nreads + 1)));
    CK(ctx->len64.ensure(sizeof(u64) * (size_t)(nreads + 1)));
    CK(ctx->fa_raw.ensure(chunk_bytes + 64));
    CK(ctx->fa_rec.ensure(24 * (size_t)std::max<u64>(nreads, 1)));
    CK(ctx->fa_items.ensure(sizeof(u64) * (size_t)(nreads + 1)));
    CK(cudaMemcpyAsync(ctx->off.p, off.data(), sizeof(u64) * (nreads + 1), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(ctx->fa_items.p, items.data(), sizeof(u64) * (nreads + 1), cudaMemcpyHostToDevice, st));
    if (nreads)
    {
        CK(cudaMemcpyAsync(ctx->len64.p, len.data(), sizeof(u64) * nreads, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(ctx->fa_rec.p, records, 24 * nreads, cudaMemcpyHostToDevice, st));
    }
    CK(cudaMemsetAsync(ctx->packed.as<uint8_t>() + head, 0, 64, st));
    FastaView fv; fv.raw = ctx->fa_raw.as<uint8_t>(); fv.rec = ctx->fa_rec.as<u64>(); fv.off = ctx->off.as<u64>(); fv.item_start = ctx->fa_items.as<u64>();
    fv.chunk_pos = chunk_pos; fv.n = (u32)nreads;
    // slices end where a read begins (records in file order, the .fai's own order; otherwise one slice)
    const int S = (ordered && chunk_bytes >= (64ull << 20) && nreads >= 4096) ? elba_fe_ctx::UP_SLICES : 1;
    std::vector<u64> slice_read(S + 1, nreads);
    slice_read[0] = 0;
    for (int i = 1; i < S; ++i)
    {
        const u64 want = chunk_pos + chunk_bytes / S * (u64)i;          // the first read that starts at or behind this file offset
        u64 lo = slice_read[i - 1], hi = nreads;
        while (lo < hi) { const u64 mid = (lo + hi) / 2; if (records[3 * mid + 1] < want) lo = mid + 1; else hi = mid; }
        slice_read[i] = lo;
    }
    CK(cudaEventRecord(ctx->ev_fork, st));                   // the previous pass has finished with the old chunk before it is overwritten
    CK(cudaStreamWaitEvent(ctx->aux, ctx->ev_fork, 0));
    for (int i = 0; i < S; ++i)
    {
        const u64 r0 = slice_read[i], r1 = slice_read[i + 1];
        const u64 p0 = (i == 0 || r0 >= nreads) ? (i == 0 ? 0 : chunk_bytes) : records[3 * r0 + 1] - chunk_pos;
        const u64 p1 = (i == S - 1 || r1 >= nreads) ? chunk_bytes : records[3 * r1 + 1] - chunk_pos;
        if (p1 > p0) CK(cudaMemcpyAsync(ctx->fa_raw.as<uint8_t>() + p0, chunk + p0, p1 - p0, cudaMemcpyHostToDevice, ctx->aux));
        CK(cudaEventRecord(ctx->up_ev[i], ctx->aux));
        CK(cudaStreamWaitEvent(st, ctx->up_ev[i], 0));
        const u64 i0 = items[r0], i1 = items[r1];
        if (i1 > i0)
        {
            const u32 g = (u32)std::min<u64>((i1 - i0 + 7) / 8, (u64)grid_for(ctx, 8));
            k_fasta_pack<<<g, 256, 0, st>>>(fv, i0, i1, ctx->packed.as<uint8_t>()); CKL(); LAUNCHED(ctx);
        }
    }
    CK(cudaEventRecord(ctx->ev[1], st));
    int rc = prepare_reads(ctx);                              // synchronises: the caller's chunk and records are free again
    if (rc) return rc;
    float ms = 0; cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]); ctx->tm.upload_ms = ms;
    return 0;
}

int elba_fe_reads_size(elba_fe_ctx *ctx, uint64_t *nreads, uint64_t *packed_bytes)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (ctx->phase < 1) return fail(ctx, ELBA_FE_ERR_STATE, "no reads resident");
    if (nreads) *nreads = ctx->n; if (packed_bytes) *packed_bytes = ctx->packed_bytes;
    return 0;
}

// the resident DnaBuffer back to the host (the stages behind the path still read it there: src/main.cpp:150,289)
int elba_fe_get_reads(elba_fe_ctx *ctx, uint8_t *packed, uint64_t *byte_off, uint64_t *len)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (ctx->phase < 1) return fail(ctx, ELBA_FE_ERR_STATE, "no reads resident");
    CK(cudaSetDevice(ctx->cfg.device));
    { int rcw = wait_reads(ctx); if (rcw) return rcw; }
    cudaEvent_t a = ctx->ev[0], b = ctx->ev[1];
    CK(cudaEventRecord(a, ctx->stream));
    if (packed && ctx->packed_bytes) CK(cudaMemcpyAsync(packed, ctx->packed.p, ctx->packed_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    if (byte_off && ctx->n) CK(cudaMemcpyAsync(byte_off, ctx->off.p, 8 * (size_t)ctx->n, cudaMemcpyDeviceToHost, ctx->stream));
    if (len && ctx->n) CK(cudaMemcpyAsync(len, ctx->len64.p, 8 * (size_t)ctx->n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaEventRecord(b, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    float ms = 0; cudaEventElapsedTime(&ms, a, b); ctx->tm.download_ms = ms;
    return 0;
}

// -------------------------------------------------------------------------------------------------
#define NC(call) do { ncclResult_t r__ = (call); if (r__ != ncclSuccess) \
    return fail(ctx, ELBA_FE_ERR_COMM, std::string(#call) + ": " + ctx->comm.api->GetErrorString(r__)); } while (0)

static int allreduce_u64(elba_fe_ctx *ctx, u64 *vals, int n, ncclRedOp_t op)
{
    if (ctx->comm.nranks == 1) return 0;
    CK(ctx->tmp64.ensure(8 * (size_t)std::max(n, 64)));
    CK(cudaMemcpyAsync(ctx->tmp64.p, vals, 8 * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    NC(ctx->comm.api->AllReduce(ctx->tmp64.p, ctx->tmp64.p, (size_t)n, ncclUint64, op, ctx->comm.comm, ctx->stream));
    CK(cudaMemcpyAsync(vals, ctx->tmp64.p, 8 * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

static int allgather_u64(elba_fe_ctx *ctx, u64 mine, std::vector<u64> &all)
{
    const int W = ctx->comm.nranks;
    all.assign(W, mine);
    if (W == 1) return 0;
    CK(ctx->tmp64.ensure(8 * (size_t)std::max(W + 1, 64)));
    CK(cudaMemcpyAsync(ctx->tmp64.as<u64>() + W, &mine, 8, cudaMemcpyHostToDevice, ctx->stream));
    NC(ctx->comm.api->AllGather(ctx->tmp64.as<u64>() + W, ctx->tmp64.p, 1, ncclUint64, ctx->comm.comm, ctx->stream));
    CK(cudaMemcpyAsync(all.data(), ctx->tmp64.p, 8 * (size_t)W, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

// every rank contributes count[r] elements of `esize` bytes; recv holds them in rank order
static int allgatherv(elba_fe_ctx *ctx, const void *send, void *recv, const std::vector<u64> &count, size_t esize)
{
    const int W = ctx->comm.nranks, me = ctx->comm.rank;
    u64 mx = 0, tot = 0;
    for (int r = 0; r < W; ++r) { mx = std::max(mx, count[r]); tot += count[r]; }
    if (tot == 0) return 0;
    if (mx * (u64)W <= tot + tot / 4 + 4096 && ctx->comm.api->AllGather)
    {
        // balanced blocks (the usual case): one ncclAllGather of blocks padded to the largest (NVSwitch: every GPU receives from all
        // others at once), then the blocks are closed up by device-to-device copies
        const size_t blk = (size_t)mx * esize;
        CK(ctx->agpad.ensure(blk * (size_t)(W + 1)));
        char *pad = ctx->agpad.as<char>();
        if (count[me]) CK(cudaMemcpyAsync(pad + blk * (size_t)W, send, count[me] * esize, cudaMemcpyDeviceToDevice, ctx->stream));
        NC(ctx->comm.api->AllGather(pad + blk * (size_t)W, pad, blk, ncclUint8, ctx->comm.comm, ctx->stream));
        u64 off = 0;
        for (int r = 0; r < W; ++r)
        {
            if (count[r]) CK(cudaMemcpyAsync((char*)recv + off * esize, pad + blk * (size_t)r, count[r] * esize, cudaMemcpyDeviceToDevice, ctx->stream));
            off += count[r];
        }
        return 0;
    }
    // uneven blocks: every rank sends its block to every other rank and receives theirs, W - 1 point-to-point transfers in each
    // direction in one group; the own block is a local copy
    u64 off = 0, myoff = 0;
    for (int r = 0; r < me; ++r) myoff += count[r];
    if (count[me]) CK(cudaMemcpyAsync((char*)recv + myoff * esize, send, count[me] * esize, cudaMemcpyDeviceToDevice, ctx->stream));
    NC(ctx->comm.api->GroupStart());
    for (int r = 0; r < W; ++r)
    {
        if (r != me)
        {
            if (count[me]) NC(ctx->comm.api->Send(send, count[me] * esize, ncclUint8, r, ctx->comm.comm, ctx->stream));
            if (count[r]) NC(ctx->comm.api->Recv((char*)recv + off * esize, count[r] * esize, ncclUint8, r, ctx->comm.comm, ctx->stream));
        }
        off += count[r];
    }
    NC(ctx->comm.api->GroupEnd());
    return 0;
}

// Slow, always-correct counting of one set of h slabs with a global table (heavy-hitter partitions, direct mode).
static int count_with_global_table(elba_fe_ctx *ctx, const std::vector<std::pair<const u64*, u64>> &slabs, u64 total, u64 rel_cap)
{
    cudaStream_t st = ctx->stream;
    u64 *d_ctr = ctx->ctr.as<u64>(); u32 *d_err = reinterpret_cast<u32*>(d_ctr + 3);
    u64 slots = std::max<u64>(2 * total + 64, 1024);
    if (slots >= (1ull << 32)) return fail(ctx, ELBA_FE_ERR_INVALID, "a k-mer partition needs a count table of more than 2^32 slots");
    CK(ctx->table.ensure(sizeof(Slot) * slots));
    k_table_clear<<<grid_for(ctx, 8), 256, 0, st>>>(ctx->table.as<Slot>(), slots, EMPTY_H); CKL(); LAUNCHED(ctx);
    TableRef T{ctx->table.as<Slot>(), (u32)slots};
    for (auto &sl : slabs)
        if (sl.second) { k_count_array<<<grid_for(ctx, 4), 256, 0, st>>>(sl.first, sl.second, T, d_err, d_ctr + 2); CKL(); LAUNCHED(ctx); }
    k_table_collect<<<grid_for(ctx, 8), 256, 0, st>>>(T.tab, T.slots, (u32)ctx->cfg.lower, (u32)ctx->cfg.upper, ctx->rel_key.as<u64>(), ctx->rel_cnt.as<u32>(), d_ctr, rel_cap);
    CKL(); LAUNCHED(ctx);
    return 0;
}

// Counting through super-k-mers (superkmer.cuh), one GPU: reads -> 16-byte records in minimizer buckets -> one CTA per
// bucket counts in shared memory.  Appends the reliable {h, count} to rel_key / rel_cnt exactly as the hash path does,
// and (fused pass 2) every instance of a reliable k-mer to the seed list ctx->cand, so build_A has no second sweep.
// retry: the overflow list or the seed list was too small (their exact sizes are known now).
// What the super-k-mer path counts: one GPU: its own reads, all buckets.  Several GPUs: ALL reads, the buckets of this rank.
struct SkmPlan { ReadsView rv; u64 Ms; u32 read_base; int nranks, rank; };

// ---- peer-memory windows -----------------------------------------------------------------------------------
static void window_unmap(elba_fe_ctx *ctx, Window &w)
{
    if (!w.mapped) return;
    for (int r = 0; r < ctx->comm.nranks && r < SK_MAXW; ++r) if (r != ctx->comm.rank && w.peer[r]) cudaIpcCloseMemHandle(w.peer[r]);
    for (auto &p : w.peer) p = nullptr;
    w.mapped = false;
}
static void window_release(elba_fe_ctx *ctx, Window &w) { window_unmap(ctx, w); w.buf.release(); }

// COLLECTIVE over the ranks when there are several (every rank calls it with the same `bytes`): (re)allocates the buffer if
// it is too small and maps every rank's buffer into every process.  The handles travel over NCCL.
static int window_ensure(elba_fe_ctx *ctx, Window &w, size_t bytes)
{
    const int W = ctx->comm.nranks, me = ctx->comm.rank;
    bytes = std::max<size_t>(bytes, 256);
    if (W == 1) { CK(w.buf.ensure(bytes)); w.peer[0] = w.buf.p; return 0; }
    if (w.mapped && bytes <= w.buf.cap) return 0;
    // nobody may still be writing into (or have mapped) the old buffer: two barriers around the unmap
    u64 one = 1; int rc;
    CK(cudaStreamSynchronize(ctx->stream));
    if ((rc = allreduce_u64(ctx, &one, 1, ncclSum))) return rc;
    window_unmap(ctx, w);
    one = 1; if ((rc = allreduce_u64(ctx, &one, 1, ncclSum))) return rc;
    CK(w.buf.ensure(bytes));
    cudaIpcMemHandle_t mine;
    CK(cudaIpcGetMemHandle(&mine, w.buf.p));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    CK(ctx->tmp64.ensure(64 * (size_t)(W + 1) + 512));
    char *d = ctx->tmp64.as<char>() + 512;                      // [0, 512) is the scratch of the scalar collectives
    CK(cudaMemcpyAsync(d + 64 * (size_t)W, &mine, 64, cudaMemcpyHostToDevice, ctx->stream));
    NC(ctx->comm.api->AllGather(d + 64 * (size_t)W, d, 64, ncclUint8, ctx->comm.comm, ctx->stream));
    std::vector<cudaIpcMemHandle_t> all(W);
    CK(cudaMemcpyAsync(all.data(), d, 64 * (size_t)W, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (int r = 0; r < W; ++r)
    {
        if (r == me) { w.peer[r] = w.buf.p; continue; }
        cudaError_t e = cudaIpcOpenMemHandle(&w.peer[r], all[r], cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) { w.peer[r] = nullptr; w.mapped = true; window_unmap(ctx, w); return fail(ctx, ELBA_FE_ERR_COMM, std::string("cudaIpcOpenMemHandle: ") + cudaGetErrorString(e)); }
    }
    w.mapped = true;
    return 0;
}

// all ranks reach this point of their streams before any of them goes on (device-side: no host synchronisation)
static int stream_barrier(elba_fe_ctx *ctx)
{
    if (ctx->comm.nranks == 1) return 0;
    CK(ctx->tmp64.ensure(1024));
    NC(ctx->comm.api->AllReduce(ctx->tmp64.as<u64>() + 48, ctx->tmp64.as<u64>() + 48, 1, ncclUint64, ncclSum, ctx->comm.comm, ctx->stream));
    return 0;
}

// Several GPUs: what every rank must know before the super-k-mer path can run across them: the blocks of reads are
// consecutive in rank order (global read ids travel as 32 bits in the records), the total number of instances (bucket
// geometry) and that every GPU can address every other one.  ok = false: use the hash path with its NCCL all-to-all.
static int multi_setup(elba_fe_ctx *ctx, bool &ok)
{
    const int W = ctx->comm.nranks;
    int rc;
    // the layout of the reads over the ranks rarely changes between passes: one scalar collective says whether anybody's did
    const u64 sig[3] = { (u64)ctx->n, (u64)ctx->read_id_offset, ctx->Ms };
    u64 changed = !ctx->setup_valid || sig[0] != ctx->setup_sig[0] || sig[1] != ctx->setup_sig[1] || sig[2] != ctx->setup_sig[2];
    if ((rc = allreduce_u64(ctx, &changed, 1, ncclMax))) return rc;
    if (!changed) { ok = ctx->p2p; return 0; }
    ctx->setup_valid = false;
    std::vector<u64> nr, ro, ms;
    if ((rc = allgather_u64(ctx, ctx->n, nr))) return rc;
    if ((rc = allgather_u64(ctx, (u64)ctx->read_id_offset, ro))) return rc;
    if ((rc = allgather_u64(ctx, ctx->Ms, ms))) return rc;
    u64 Nt = 0, Mt = 0, Mx = 0; ok = W <= SK_MAXW;
    for (int r = 0; r < W; ++r) { if (ro[r] != ro[0] + Nt) ok = false; Nt += nr[r]; Mt += ms[r]; Mx = std::max(Mx, ms[r]); }
    if (ro[0] + Nt >= 0xFFFFFFF0ull) ok = false;
    ctx->N_total = Nt; ctx->Ms_total = Mt; ctx->Ms_max = Mx; ctx->read_base0 = (int64_t)ro[0];
    ctx->roff.assign(W + 1, ro[0] + Nt);
    for (int r = 0; r < W; ++r) ctx->roff[r] = ro[r];
    if (ok)
    {
        CK(ctx->d_roff.ensure(8 * (size_t)(W + 1)));
        CK(cudaMemcpyAsync(ctx->d_roff.p, ctx->roff.data(), 8 * (size_t)(W + 1), cudaMemcpyHostToDevice, ctx->stream));
        // peer access from this GPU to every other GPU of the job
        std::vector<u64> dev;
        if ((rc = allgather_u64(ctx, (u64)ctx->cfg.device, dev))) return rc;
        u64 can = 1;
        for (int r = 0; r < W; ++r)
            if (r != ctx->comm.rank)
            {
                int a = 0;
                if ((int)dev[r] == ctx->cfg.device || cudaDeviceCanAccessPeer(&a, ctx->cfg.device, (int)dev[r]) != cudaSuccess || !a) can = 0;
            }
        if (const char *e = getenv("ELBA_FE_P2P")) { if (atoi(e) == 0) can = 0; }
        if ((rc = allreduce_u64(ctx, &can, 1, ncclMin))) return rc;
        if (!can) ok = false;
    }
    ctx->p2p = ok;
    ctx->setup_sig[0] = sig[0]; ctx->setup_sig[1] = sig[1]; ctx->setup_sig[2] = sig[2]; ctx->setup_valid = true;
    return 0;
}

static __global__ void k_add_u64(u64 *__restrict__ v, u64 n, u64 add)
{
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) v[i] += add;
}

static __global__ void k_remote_records(const u64 *__restrict__ fill, u64 nbg, u32 nb_own, u32 me, u64 *__restrict__ out)
{
    u64 acc = 0;
    for (u64 b = (u64)blockIdx.x * blockDim.x + threadIdx.x; b < nbg; b += (u64)gridDim.x * blockDim.x)
        if (b / nb_own != me) acc += (u32)fill[b];
    for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0 && acc) atomicAdd(out, acc);
}

static int count_superkmers(elba_fe_ctx *ctx, const SkmPlan &plan, int m, int Wm, u64 rel_cap, bool &retry)
{
    cudaStream_t st = ctx->stream;
    const ReadsView rv = plan.rv;
    const int k = ctx->cfg.k; const u32 lower = ctx->cfg.lower, upper = ctx->cfg.upper;
    const u64 Ms = plan.Ms;                                 // instances of the reads of ALL GPUs: decides the bucket geometry
    const u64 Ms_own = Ms / (u64)plan.nranks + 1;           // what this GPU expects to count: decides the list capacities
    const int W = plan.nranks, me = plan.rank;
    u64 *d_ctr = ctx->ctr.as<u64>(); u32 *d_err = reinterpret_cast<u32*>(d_ctr + 3);
    int rc;
    retry = false;
    const u32 slots = SK4_SLOTS, bcap = sk4_cap(SK4_THREADS);
    const double avg_run = 32.0 / (64.0 / (double)(Wm + 1) + 1.0);    // a chunk of 32 window starts holds 32 * 2 / (W + 1) minimizer runs plus the one its start cuts
    // mean bucket: a third of the table in DISTINCT k-mers (distinct / instances of the last pass, else a guess), records well inside the staging
    // buffer, instances within 2 / 5 of the capacity (a bucket is a handful of genomic super-k-mers times the coverage: CV ~ 0.4)
    const double dm = ctx->hist_dm > 0.0 ? std::min(1.0, std::max(0.05, ctx->hist_dm)) : 0.3;
    u64 mean_inst = (u64)std::min({ (double)bcap * 0.4, 0.36 * (double)slots / dm, (double)SK4_RMAX / 2.7 * avg_run });      // measured: profiles/r2_v11_tune_bucket_mean.log
    mean_inst = std::max<u64>(mean_inst, 64);
    if (const char *e = getenv("ELBA_FE_SKM_MEAN")) { long v = atol(e); if (v >= 64 && v <= (long)bcap) mean_inst = (u64)v; }
    u64 NBg = std::max<u64>(1, (Ms + mean_inst - 1) / mean_inst);
    if (ctx->cfg.num_partitions > 1) NBg = std::max<u64>(NBg, (u64)ctx->cfg.num_partitions);
    const u64 NB = (NBg + plan.nranks - 1) / plan.nranks;   // buckets of this GPU: [rank * NB, (rank + 1) * NB) of NBg
    NBg = NB * (u64)plan.nranks;
    if (NBg >= (1ull << 31)) return fail(ctx, ELBA_FE_ERR_INVALID, "too many minimizer buckets for one context");
    // records per (bucket, source GPU): the bucket sizes vary by ~40 % whatever the number of sources, the share of one
    // source adds its own (Poisson-like) spread
    double slack = 2.5;
    if (const char *e = getenv("ELBA_FE_SKM_SLACK")) { double v = atof(e); if (v >= 1.0 && v <= 16.0) slack = v; }
    const double mean_rec = (double)Ms / (double)NBg / avg_run / (double)W;
    u64 rcap = (u64)(mean_rec * slack + (W > 1 ? 4.0 * std::sqrt(1.5 * mean_rec) : 0.0)) + (W > 1 ? 16 : 32);
    rcap = std::min<u64>(rcap, SK4_RMAX);
    ctx->sz.partitions = NBg; ctx->sz.table_slots = slots;
    // every rank computes the same capacities from the same global numbers: the windows are (re)allocated collectively
    const u64 ovf_cap = std::max<u64>(ctx->skm_ovf_cap, std::max<u64>(Ms_own / 64, 1u << 16));
    if ((rc = window_ensure(ctx, ctx->w_slab, sizeof(SkmRec) * NB * (u64)W * rcap))) return rc;
    if ((rc = window_ensure(ctx, ctx->w_ovf, sizeof(SkmRec) * ovf_cap))) return rc;
    if ((rc = window_ensure(ctx, ctx->w_octr, 64))) return rc;
    CK(ctx->skm_fill.ensure(sizeof(u64) * NBg));
    if (W > 1) { CK(ctx->skm_fillin.ensure(sizeof(u64) * NBg)); CK(ctx->skm_plan.ensure(sizeof(u64) * NB)); CK(ctx->skm_stage.ensure(sizeof(SkmRec) * NBg * rcap)); }
    ctx->skm_ovf_cap = ovf_cap;
    u64 *d_octr = ctx->w_octr.buf.as<u64>();                              // [0] records, [1] instances in my overflow list
    // seed list: {list index, pos, read} of every instance of a reliable k-mer; the size of the last pass, else a guess
    const u64 gc_max = (u64)grid_for(ctx, SK4_MINB);                  // CTAs of the count kernel: each may leave one chunk partly used
    u64 seed_guess = Ms_own / 16 + (1u << 20) + gc_max * SK4_CHUNK;
    if (const char *e = getenv("ELBA_FE_SEED_CAP")) { long long v = atoll(e); if (v >= 1) seed_guess = (u64)v; }      // tests: force the resize
    const u64 seed_cap = std::max<u64>(ctx->seed_cap, seed_guess);
    CK(ctx->seeds.ensure(sizeof(Seed) * seed_cap));
    ctx->seed_cap = seed_cap;
    if (rel_cap >= 0xFFFFFFF0ull) return fail(ctx, ELBA_FE_ERR_INVALID, "more than 2^32 entries in the reliable list of one context");
    SeedSink2 seeds; seeds.out = ctx->seeds.as<Seed>(); seeds.cursor = d_ctr + 7; seeds.cap = seed_cap;
    CK(cudaMemsetAsync(ctx->skm_fill.p, 0, sizeof(u64) * NBg, st));
    CK(cudaMemsetAsync(d_octr, 0, 64, st));
    // several GPUs: nobody writes into a slab (or bumps an overflow counter) that its owner still reads from the previous pass
    if ((rc = stream_barrier(ctx))) return rc;
    RecSink sink; std::memset(&sink, 0, sizeof sink);
    for (int r = 0; r < W; ++r) { sink.ovf[r] = (SkmRec*)ctx->w_ovf.peer[r]; sink.ovf_ctr[r] = (u64*)ctx->w_octr.peer[r]; }
    sink.slab = ctx->w_slab.buf.as<SkmRec>(); sink.stage = ctx->skm_stage.as<SkmRec>();
    sink.fill = ctx->skm_fill.as<u64>(); sink.rcap = (u32)rcap; sink.nb_own = (u32)NB; sink.nsrc = (u32)W; sink.me = (u32)me;
    sink.read_base = plan.read_base; sink.ovf_cap = ovf_cap;
    const u32 nmax = skm_nmax(k);
    mark(ctx, "setup");
    EventPair &pp = next_pair(ctx->pev, ctx->pev_used);
    CK(cudaEventRecord(pp.a, st));
    if (rv.nchunks)
    {
        int contig = 1, nr = SK_NR;
        if (const char *e = getenv("ELBA_FE_SKM_ORDER")) contig = std::strcmp(e, "strided") != 0;
        if (const char *e = getenv("ELBA_FE_SKM_NR")) nr = atoi(e);
        // one launch over all chunks, or one per slice of an upload that is still arriving (slice s needs slice s + 1: a chunk's
        // 64-base window may reach into the next read)
        const int nlaunch = ctx->up_n > 0 ? ctx->up_n : 1;
        u64 gb = 0;
        for (int sl = 0; sl < nlaunch; ++sl)
        {
            const u64 ge = ctx->up_n > 0 ? ctx->up_chunk_end[sl] : rv.nchunks;
            if (ctx->up_n > 0) CK(cudaStreamWaitEvent(st, ctx->up_ev[std::min(sl + 1, ctx->up_n - 1)], 0));
            const u64 nch = ge - gb;
            if (nch == 0) continue;
            const u32 g1 = (u32)std::min<u64>((nch + SK_THREADS - 1) / SK_THREADS, (u64)grid_for(ctx, 4));
            const u64 it1 = (nch + (u64)g1 * SK_THREADS - 1) / ((u64)g1 * SK_THREADS);
            switch (Wm)
            {
                case 8:  k_skm_scatter<8, SK_NR><<<g1, SK_THREADS, 0, st>>>(rv, k, m, nmax, sink, it1, contig, gb, ge); break;
                case 12: k_skm_scatter<12, SK_NR><<<g1, SK_THREADS, 0, st>>>(rv, k, m, nmax, sink, it1, contig, gb, ge); break;
                case 16: if (nr == 1) k_skm_scatter<16, 1><<<g1, SK_THREADS, 0, st>>>(rv, k, m, nmax, sink, it1, contig, gb, ge);
                         else k_skm_scatter<16, SK_NR><<<g1, SK_THREADS, 0, st>>>(rv, k, m, nmax, sink, it1, contig, gb, ge);
                         break;
                case 17: k_skm_scatter<17, SK_NR><<<g1, SK_THREADS, 0, st>>>(rv, k, m, nmax, sink, it1, contig, gb, ge); break;
                default: return fail(ctx, ELBA_FE_ERR_INVALID, "no super-k-mer kernel for this minimizer window");
            }
            CKL(); LAUNCHED(ctx);
            gb = ge;
        }
    }
    CK(cudaEventRecord(pp.b, st));
    mark(ctx, "scatter");
    RecSlabs in; in.slab = ctx->w_slab.buf.as<SkmRec>(); in.fill = ctx->skm_fill.as<u64>(); in.plan = in.fill; in.off = nullptr; in.rcap = (u32)rcap; in.nsrc = (u32)W; in.nb = (u32)NB; in.me = (u32)me;
    if (W > 1)
    {
        // the staged records of the other GPUs' buckets go into their owners' slabs through peer memory, packed: where a bucket
        // starts inside the region = the exclusive scan of the record counts (the owner redoes that scan from the fill words)
        CK(ctx->skm_foff.ensure(8 * (NBg + 1))); CK(ctx->skm_inoff.ensure(8 * (NBg + 1)));
        k_skm_forward_counts<<<nblk(NBg + 1, 256), 256, 0, st>>>(ctx->skm_fill.as<u64>(), NBg, (u32)rcap, ctx->skm_foff.as<u64>()); CKL(); LAUNCHED(ctx);
        if ((rc = exclusive_scan_inplace(ctx, ctx->skm_foff.as<u64>(), NBg + 1))) return rc;
        RecForward fw; std::memset(&fw, 0, sizeof fw);
        for (int r = 0; r < W; ++r) fw.slab[r] = (SkmRec*)ctx->w_slab.peer[r];
        fw.stage = ctx->skm_stage.as<SkmRec>(); fw.fill = ctx->skm_fill.as<u64>(); fw.off = ctx->skm_foff.as<u64>(); fw.rcap = (u32)rcap; fw.nb_own = (u32)NB; fw.nsrc = (u32)W; fw.me = (u32)me;
        CK(cudaEventRecord(ctx->ev_x0, st));                 // exchange_ms = the push through peer memory + the fill words
        k_skm_forward<<<grid_for(ctx, 8), 256, 0, st>>>(fw); CKL(); LAUNCHED(ctx);
        mark(ctx, "forward");
        // the reservation words follow the records: rank d gets, from every source, the fill words of its own buckets.  Stream
        // order makes this exchange the barrier behind the peer-memory stores of the scatter.
        NC(ctx->comm.api->GroupStart());
        for (int r = 0; r < W; ++r)
        {
            NC(ctx->comm.api->Send(ctx->skm_fill.as<u64>() + NB * (u64)r, NB, ncclUint64, r, ctx->comm.comm, st));
            NC(ctx->comm.api->Recv(ctx->skm_fillin.as<u64>() + NB * (u64)r, NB, ncclUint64, r, ctx->comm.comm, st));
        }
        NC(ctx->comm.api->GroupEnd());
        CK(cudaEventRecord(ctx->ev_x1, st));
        k_skm_plan<<<nblk(NB, 256), 256, 0, st>>>(ctx->skm_fillin.as<u64>(), (u32)NB, (u32)W, (u32)rcap, ctx->skm_plan.as<u64>()); CKL(); LAUNCHED(ctx);
        k_skm_forward_counts<<<nblk(NBg + 1, 256), 256, 0, st>>>(ctx->skm_fillin.as<u64>(), NBg, (u32)rcap, ctx->skm_inoff.as<u64>()); CKL(); LAUNCHED(ctx);
        if ((rc = exclusive_scan_inplace(ctx, ctx->skm_inoff.as<u64>(), NBg + 1))) return rc;
        in.off = ctx->skm_inoff.as<u64>();
        k_remote_records<<<grid_for(ctx, 2), 256, 0, st>>>(ctx->skm_fill.as<u64>(), NBg, (u32)NB, (u32)me, d_ctr + 9); CKL(); LAUNCHED(ctx);
        in.fill = ctx->skm_fillin.as<u64>(); in.plan = ctx->skm_plan.as<u64>();
        mark(ctx, "fill_exchange");
    }
    RecOverflow ovf; ovf.list = ctx->w_ovf.buf.as<SkmRec>(); ovf.cursor = d_octr; ovf.inst = d_octr + 1; ovf.cap = ovf_cap;
    EventPair &ep = next_pair(ctx->kev, ctx->kev_used);
    CK(cudaEventRecord(ep.a, st));
    {
        const u32 gc = (u32)std::min<u64>(NB, gc_max);
        k_skm_count4<SK4_THREADS, SK4_SLOTS, SK4_RMAX, SK4_POOL, SK4_RETRY, SK4_MINB><<<gc, SK4_THREADS, sk4_smem(SK4_SLOTS, SK4_RMAX, SK4_POOL, SK4_RETRY, SK4_THREADS), st>>>(in, (u32)NB, k, ovf, lower, upper,
            ctx->rel_key.as<u64>(), ctx->rel_cnt.as<u32>(), d_ctr, rel_cap, seeds);
    }
    CKL(); LAUNCHED(ctx);
    CK(cudaEventRecord(ep.b, st));
    mark(ctx, "count_kernel");
    u64 o[2] = {0, 0};
    CK(cudaMemcpyAsync(o, d_octr, 16, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    const u64 novf = o[0], ninst = o[1];
    {
        // an overflow list that was too small anywhere: every rank redoes the pass with the largest need (the windows are collective)
        u64 need = novf > ovf_cap ? novf + (novf >> 3) : 0;
        if (W > 1 && (rc = allreduce_u64(ctx, &need, 1, ncclMax))) return rc;
        if (need) { ctx->skm_ovf_cap = std::max(ctx->skm_ovf_cap, need); retry = true; return 0; }
    }
    ctx->sz.slow_partitions = 0; ctx->sz.overflow_instances = ninst;
    if (novf)
    {
        // buckets that overflowed their record capacity, 6144 instances or 3/4 of the table: exact count in one global table
        const u64 gslots = std::max<u64>(2 * ninst + 64, 1024);
        if (gslots >= (1ull << 32)) return fail(ctx, ELBA_FE_ERR_INVALID, "the overflow of the minimizer buckets needs a count table of more than 2^32 slots");
        CK(ctx->table.ensure(sizeof(Slot) * gslots));
        k_table_clear<<<grid_for(ctx, 8), 256, 0, st>>>(ctx->table.as<Slot>(), gslots, EMPTY_KEY); CKL(); LAUNCHED(ctx);
        TableRef T{ctx->table.as<Slot>(), (u32)gslots};
        k_skm4_count_global<<<grid_for(ctx, 4), 256, 0, st>>>(ctx->w_ovf.buf.as<SkmRec>(), d_octr, ovf_cap, k, T, d_err, d_ctr + 2); CKL(); LAUNCHED(ctx);
        k_skm4_collect_global<<<grid_for(ctx, 8), 256, 0, st>>>(T.tab, T.slots, lower, upper, ctx->rel_key.as<u64>(), ctx->rel_cnt.as<u32>(), d_ctr, rel_cap); CKL(); LAUNCHED(ctx);
        k_skm4_emit_global<<<grid_for(ctx, 4), 256, 0, st>>>(ctx->w_ovf.buf.as<SkmRec>(), d_octr, ovf_cap, k, T, lower, upper, seeds); CKL(); LAUNCHED(ctx);
    }
    mark(ctx, "fallback");
    ctx->seeds_fused = false;
    {
        // [0] list entries handed out (chunks with holes + what the fallback appended), [1] sum of reliable counts, [2] distinct,
        // [7] seed entries handed out, [8] reliable k-mers
        u64 h[10];
        CK(cudaMemcpyAsync(h, d_ctr, sizeof h, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        ctx->skm_reliable = h[8];
        ctx->exchange_bytes = 32 * h[9];                      // records this GPU wrote into other GPUs' slabs
        {
            u64 again = h[7] > seed_cap;
            if (again) ctx->seed_cap = h[7] + (h[7] >> 4) + 1024;
            if (W > 1 && (rc = allreduce_u64(ctx, &again, 1, ncclMax))) return rc;
            if (again) { retry = true; return 0; }
        }
        if (h[0] <= rel_cap && h[7] < h[1])
        {
            char b[160]; snprintf(b, sizeof b, "fused seed emission handed out %llu entries, the counts promise %llu", (unsigned long long)h[7], (unsigned long long)h[1]);
            return fail(ctx, ELBA_FE_ERR_CUDA, b);
        }
        ctx->seeds_fused = true; ctx->nseeds_fused = h[7];
        if (Ms) ctx->hist_dm = (double)h[2] / (double)Ms_own;
    }
    return 0;
}

int elba_fe_count(elba_fe_ctx *ctx)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (ctx->phase < 1) return fail(ctx, ELBA_FE_ERR_STATE, "elba_fe_count: no reads uploaded");
    ctx->og_aligned = ctx->og_done = ctx->ct_done = ctx->pf_done = false;
    CK(cudaSetDevice(ctx->cfg.device));
    const int k = ctx->cfg.k, stride = ctx->cfg.stride; const u32 lower = ctx->cfg.lower, upper = ctx->cfg.upper;
    cudaStream_t st = ctx->stream;
    ReadsView rv = view(ctx);
    CK(cudaEventRecord(ctx->ev[2], st));
    ctx->seeds_fused = false;
    mark(ctx, "begin");

    // counters: [0] R cursor, [1] sum of reliable counts, [2] distinct, [3] (u32) table-overflow flag, [4] (u32) level-1 overflow flag
    CK(ctx->ctr.ensure(128));
    u64 *d_ctr = ctx->ctr.as<u64>();
    u32 *d_err = reinterpret_cast<u32*>(d_ctr + 3);
    u32 *d_flag1 = reinterpret_cast<u32*>(d_ctr + 4);

    const u64 Ms = ctx->Ms;
    const int W = ctx->comm.nranks, me = ctx->comm.rank;
    // instances over all GPUs decide the partitioning; the largest local share decides the slab capacity
    u64 Ms_total = Ms, Ms_max = Ms;
    bool p2p_ok = false;
    ctx->p2p = W > 1 ? ctx->p2p : false;
    if (W > 1)
    {
        int rc0 = multi_setup(ctx, p2p_ok);          // collective: read layout over the ranks, totals, peer access
        if (rc0) return rc0;
        Ms_total = ctx->Ms_total; Ms_max = ctx->Ms_max;
    }
    else ctx->N_total = ctx->n;
    // balanced digits: P1 ~ P2 ~ sqrt(#sub-buckets); both scatters then write runs of similar length
    u64 PART_TARGET = std::max<u64>(1u << 16, (u64)std::sqrt((double)Ms_total * (double)BUCKET_CAP / 1.4));
    if (const char *e = getenv("ELBA_FE_PART_TARGET")) { long long v = atoll(e); if (v >= 4096) PART_TARGET = (u64)v; }
    u32 P1 = (u32)ctx->cfg.num_partitions;
    const bool direct = W == 1 && ((P1 == 1) || (P1 == 0 && Ms <= 65536));
    if (P1 == 0) P1 = (u32)std::min<u64>(MAX_P1, std::max<u64>(1, (Ms_total + PART_TARGET - 1) / PART_TARGET));
    if (direct) P1 = 1;
    // k >= 20, one GPU, every window start: super-k-mers in minimizer buckets (superkmer.cuh); else the two-level hash partition
    int skm_m = 0, skm_W = 0;
    // (several GPUs: every GPU parses all reads and counts the buckets it owns, no record crosses NVLink)
    bool use_skm = !direct && stride == 1 && skm_geometry(k, skm_m, skm_W);
    if (const char *e = getenv("ELBA_FE_COUNT_PATH")) { if (!std::strcmp(e, "hash")) use_skm = false; }
    SkmPlan plan; plan.rv = rv; plan.Ms = Ms; plan.read_base = 0; plan.nranks = 1; plan.rank = 0;
    ctx->kmers_distributed = false;
    if (W == 1) ctx->read_base0 = ctx->read_id_offset;
    else
    {
        // every GPU parses ITS OWN reads; the records go into the owners' slabs through peer memory (superkmer.cuh)
        if (use_skm && !p2p_ok) use_skm = false;                         // read blocks not consecutive over the ranks / no peer access: hash path
        if (use_skm) { plan.Ms = ctx->Ms_total; plan.read_base = (u32)ctx->read_id_offset; plan.nranks = W; plan.rank = me; }
    }
    if (!use_skm) { int rcw = wait_reads(ctx); if (rcw) return rcw; }                 // only the super-k-mer scatter follows an upload slice by slice
    if (W > 1) { P1 = (P1 + W - 1) / W * W; if (P1 > MAX_P1) P1 = MAX_P1 / W * W; }      // every rank owns P1 / W partitions
    const u32 Pown = P1 / (u32)W;
    ctx->sz.partitions = P1;

    u64 rel_cap = Ms_max / lower + 1;
    if (rel_cap * 12 > (1ull << 30)) rel_cap = std::max<u64>(ctx->rel_cap, std::max<u64>(Ms_max / 8, (1ull << 30) / 12));
    if (use_skm) rel_cap += (u64)grid_for(ctx, SK4_MINB) * SK4_CHUNK;           // the bucket kernel hands the list out in chunks
    u64 R = 0, sumcnt = 0, D = 0;
    for (int attempt = 0; attempt < 4; ++attempt)
    {
        CK(ctx->rel_key.ensure(sizeof(u64) * rel_cap)); CK(ctx->rel_cnt.ensure(sizeof(u32) * rel_cap));
        ctx->rel_cap = rel_cap;
        CK(cudaMemsetAsync(ctx->ctr.p, 0, 128, st));
        ctx->kev_used = 0; ctx->pev_used = 0;
        if (direct)
        {
            u64 slots = std::max<u64>(2 * Ms + 64, 1024);
            if (slots >= (1ull << 32)) return fail(ctx, ELBA_FE_ERR_INVALID, "single-partition mode needs < 2^31 k-mer instances; use num_partitions = 0");
            CK(ctx->table.ensure(sizeof(Slot) * slots));
            ctx->sz.table_slots = slots;
            k_table_clear<<<grid_for(ctx, 8), 256, 0, st>>>(ctx->table.as<Slot>(), slots, EMPTY_H); CKL(); LAUNCHED(ctx);
            TableRef T{ctx->table.as<Slot>(), (u32)slots};
            EventPair &ep = next_pair(ctx->kev, ctx->kev_used);
            CK(cudaEventRecord(ep.a, st));
            if (ctx->nchunks) { k_count_direct<<<grid_for(ctx, 8), 256, 0, st>>>(rv, k, stride, T, d_err, d_ctr + 2); CKL(); LAUNCHED(ctx); }
            CK(cudaEventRecord(ep.b, st));
            k_table_collect<<<grid_for(ctx, 8), 256, 0, st>>>(T.tab, T.slots, lower, upper, ctx->rel_key.as<u64>(), ctx->rel_cnt.as<u32>(), d_ctr, rel_cap);
            CKL(); LAUNCHED(ctx);
        }
        else if (use_skm)
        {
            bool again = false;
            int rc0 = count_superkmers(ctx, plan, skm_m, skm_W, rel_cap, again);
            if (rc0) return rc0;
            if (again)
            {
                if (attempt == 3) return fail(ctx, ELBA_FE_ERR_CUDA, "overflow list resize did not converge");
                continue;
            }
        }
        else
        {
            ctx->sz.table_slots = BUCKET_SLOTS;
            // ---- level 1: optimistic uniform regions; exact regions from a histogram if one overflows
            const u64 mean = (Ms_max + P1 - 1) / P1;
            u64 cap1 = (u64)((double)mean * 1.03) + 4096; cap1 = (cap1 + 15) & ~15ull;
            if (cap1 >= (1ull << 32)) return fail(ctx, ELBA_FE_ERR_INVALID, "level-1 partition exceeds 2^32 instances");
            std::vector<u64> start(P1 + 1);
            for (u32 p = 0; p <= P1; ++p) start[p] = (u64)p * cap1;
            std::vector<u32> cnt(P1, 0);
            CK(ctx->phist.ensure(sizeof(u64) * (P1 + 1))); CK(ctx->pcursor.ensure(sizeof(u32) * (P1 + 1)));
            const size_t smem1 = sizeof(u64) * S1_TILE + 2 * sizeof(u32) * P1;
            EventPair &pp = next_pair(ctx->pev, ctx->pev_used);
            CK(cudaEventRecord(pp.a, st));
            bool uniform = true;
            for (int lay = 0; lay < 2; ++lay)
            {
                CK(ctx->partbuf.ensure(sizeof(u64) * std::max<u64>(start[P1], 1)));
                CK(cudaMemcpyAsync(ctx->phist.p, start.data(), sizeof(u64) * (P1 + 1), cudaMemcpyHostToDevice, st));
                CK(cudaMemsetAsync(ctx->pcursor.p, 0, sizeof(u32) * (P1 + 1), st));
                CK(cudaMemsetAsync(d_flag1, 0, 4, st));
                if (uniform) k_scatter1<true><<<grid_for(ctx, 2), S1_THREADS, smem1, st>>>(rv, k, stride, P1, (u32)cap1, ctx->phist.as<u64>(), ctx->pcursor.as<u32>(), ctx->partbuf.as<u64>(), d_flag1);
                else         k_scatter1<false><<<grid_for(ctx, 2), S1_THREADS, smem1, st>>>(rv, k, stride, P1, 0u, ctx->phist.as<u64>(), ctx->pcursor.as<u32>(), ctx->partbuf.as<u64>(), d_flag1);
                CKL(); LAUNCHED(ctx);
                u32 flag = 0;
                CK(cudaMemcpyAsync(cnt.data(), ctx->pcursor.p, sizeof(u32) * P1, cudaMemcpyDeviceToHost, st));
                CK(cudaMemcpyAsync(&flag, d_flag1, 4, cudaMemcpyDeviceToHost, st));
                CK(cudaStreamSynchronize(st));
                u64 anyflag = flag;
                if (W > 1) { int rc0 = allreduce_u64(ctx, &anyflag, 1, ncclMax); if (rc0) return rc0; }
                if (!anyflag) break;
                if (lay == 1) return fail(ctx, ELBA_FE_ERR_CUDA, "level-1 scatter overflowed an exact layout");
                // skewed partition sizes (heavy hitters): exact histogram, exact regions
                CK(ctx->lut.ensure(sizeof(u64) * (P1 + 1)));
                CK(cudaMemsetAsync(ctx->lut.p, 0, sizeof(u64) * (P1 + 1), st));
                k_hist1<<<grid_for(ctx, 4), 256, sizeof(u32) * P1, st>>>(rv, k, stride, P1, ctx->lut.as<u64>()); CKL(); LAUNCHED(ctx);
                std::vector<u64> hist(P1);
                CK(cudaMemcpyAsync(hist.data(), ctx->lut.p, sizeof(u64) * P1, cudaMemcpyDeviceToHost, st));
                CK(cudaStreamSynchronize(st));
                u64 hmax = 0;
                for (u32 p = 0; p < P1; ++p) hmax = std::max(hmax, hist[p]);
                if (W > 1)
                {
                    // slabs must have one shape on every rank: uniform regions of the largest partition anywhere
                    int rc0 = allreduce_u64(ctx, &hmax, 1, ncclMax); if (rc0) return rc0;
                    cap1 = (hmax + 15) & ~15ull;
                    if (cap1 >= (1ull << 32)) return fail(ctx, ELBA_FE_ERR_INVALID, "level-1 partition exceeds 2^32 instances");
                    for (u32 p = 0; p <= P1; ++p) start[p] = (u64)p * cap1;
                }
                else
                {
                    if (hmax >= (1ull << 32)) return fail(ctx, ELBA_FE_ERR_INVALID, "level-1 partition exceeds 2^32 instances");
                    for (u32 p = 0; p < P1; ++p) start[p + 1] = start[p] + ((hist[p] + 15) & ~15ull);
                    uniform = false;
                }
            }
            CK(cudaEventRecord(pp.b, st));

            // ---- several GPUs: partition p belongs to rank p / Pown; one personalised all-to-all of the slabs
            //      (the reference's Alltoallv of 8-byte k-mers, src/KmerOps.cpp:151) and of their fill counts
            const u64 *lvl2_in = ctx->partbuf.as<u64>();
            u64 slab_stride = 0;
            std::vector<u32> cnt_all;                   // [W][Pown] fills of my partitions in every rank's slab
            if (W > 1)
            {
                const u64 slab = (u64)Pown * cap1;
                CK(ctx->recvbuf.ensure(sizeof(u64) * slab * W)); CK(ctx->recvcnt.ensure(sizeof(u32) * (size_t)P1));
                CK(cudaEventRecord(ctx->ev_x0, st));
                NC(ctx->comm.api->GroupStart());
                for (int r = 0; r < W; ++r)
                {
                    NC(ctx->comm.api->Send(ctx->partbuf.as<u64>() + slab * r, slab, ncclUint64, r, ctx->comm.comm, st));
                    NC(ctx->comm.api->Recv(ctx->recvbuf.as<u64>() + slab * r, slab, ncclUint64, r, ctx->comm.comm, st));
                    NC(ctx->comm.api->Send(ctx->pcursor.as<u32>() + (size_t)Pown * r, Pown, ncclUint32, r, ctx->comm.comm, st));
                    NC(ctx->comm.api->Recv(ctx->recvcnt.as<u32>() + (size_t)Pown * r, Pown, ncclUint32, r, ctx->comm.comm, st));
                }
                NC(ctx->comm.api->GroupEnd());
                CK(cudaEventRecord(ctx->ev_x1, st));
                cnt_all.resize(P1);
                CK(cudaMemcpyAsync(cnt_all.data(), ctx->recvcnt.p, sizeof(u32) * (size_t)P1, cudaMemcpyDeviceToHost, st));
                CK(cudaStreamSynchronize(st));
                lvl2_in = ctx->recvbuf.as<u64>(); slab_stride = slab;
                ctx->exchange_bytes = sizeof(u64) * slab * (W - 1);
            }
            else cnt_all = cnt;

            // ---- plan of level 2 over MY partitions (all of them on one GPU)
            std::vector<u32> plan(4 * (size_t)Pown + 2, 0);
            u32 *pn = plan.data(), *pp2 = pn + Pown, *ptile = pp2 + Pown, *pbucket = ptile + Pown + 1;
            std::vector<u32> slow;
            std::vector<u64> ntot(Pown, 0);
            for (u32 p = 0; p < Pown; ++p)
            {
                u64 n = 0;
                for (int j = 0; j < W; ++j) n += cnt_all[(size_t)j * Pown + p];
                ntot[p] = n;
                if (n >= (1ull << 32)) return fail(ctx, ELBA_FE_ERR_INVALID, "level-1 partition exceeds 2^32 instances");
                // mean fill = BUCKET_CAP / 1.4: with repeats the bucket sizes are compound-Poisson (sigma ~ sqrt(mean * copy number))
                u64 p2 = n ? std::max<u64>(1, (n * 7 / 5 + BUCKET_CAP - 1) / BUCKET_CAP) : 0;
                if (p2 > MAX_P2) { slow.push_back(p); n = 0; p2 = 0; }
                pn[p] = (u32)n; pp2[p] = (u32)p2;
                ptile[p + 1] = ptile[p] + (u32)((n + S2_TILE - 1) / S2_TILE);
                pbucket[p + 1] = pbucket[p] + (u32)p2;
            }
            const u32 nbuckets = pbucket[Pown];
            CK(ctx->plan.ensure(sizeof(u32) * plan.size()));
            CK(cudaMemcpyAsync(ctx->plan.p, plan.data(), sizeof(u32) * plan.size(), cudaMemcpyHostToDevice, st));
            CK(ctx->bfill.ensure(sizeof(u32) * ((size_t)nbuckets + 1)));
            u64 ovf_cap = std::max<u64>(ctx->ovf_cap, std::max<u64>(Ms_max / 16, 1u << 20));
            CK(ctx->ovf.ensure(sizeof(u64) * ovf_cap)); ctx->ovf_cap = ovf_cap;
            Overflow ovf{ctx->ovf.as<u64>(), d_ctr + 5, ovf_cap};
            CK(cudaMemsetAsync(ctx->bfill.p, 0, sizeof(u32) * ((size_t)nbuckets + 1), st));
            PartPlan pl; pl.n = ctx->plan.as<u32>(); pl.p2 = pl.n + Pown; pl.tile_start = pl.p2 + Pown; pl.bucket_start = pl.tile_start + Pown + 1;
            // my partitions start at region me * Pown of every slab; on one GPU that is region 0 of the only slab
            PartInput pi; pi.in = lvl2_in; pi.W = (u32)W; pi.slab_stride = slab_stride; pi.part_start = ctx->phist.as<u64>(); pi.P = Pown;
            pi.cnt = W > 1 ? ctx->recvcnt.as<u32>() : ctx->pcursor.as<u32>();

            // ---- groups of partitions whose sub-buckets fit one scratch buffer; two buffers, two streams
            const u64 group_buckets = std::max<u64>(MAX_P2, (ctx->scratch_mb << 20) / (sizeof(u64) * BUCKET_CAP));
            for (int b = 0; b < 2; ++b) CK(ctx->scratch[b].ensure(sizeof(u64) * BUCKET_CAP * std::min<u64>(group_buckets, std::max<u32>(nbuckets, 1))));
            const size_t smemc = (sizeof(u64) + sizeof(u32)) * BUCKET_SLOTS;
            EventPair &ep = next_pair(ctx->kev, ctx->kev_used);
            CK(cudaEventRecord(ep.a, st));
            CK(cudaEventRecord(ctx->ev_fork, st));
            CK(cudaStreamWaitEvent(ctx->aux, ctx->ev_fork, 0));
            int which = 0; bool used_aux = false;
            for (u32 g0 = 0; g0 < Pown;)
            {
                u32 g1 = g0 + 1;
                while (g1 < Pown && (u64)(pbucket[g1 + 1] - pbucket[g0]) <= group_buckets) ++g1;
                const u32 nt = ptile[g1] - ptile[g0], nb = pbucket[g1] - pbucket[g0];
                u32 p2max = 1; for (u32 p = g0; p < g1; ++p) p2max = std::max(p2max, pp2[p]);
                if (nt)
                {
                    cudaStream_t s2 = which ? ctx->aux : st; used_aux |= which != 0;
                    const size_t smem2 = sizeof(u64) * S2_TILE + 2 * sizeof(u32) * p2max;
                    if (W == 1) k_scatter2<true><<<std::min<u32>(nt, grid_for(ctx, 5)), S2_THREADS, smem2, s2>>>(pi, pl, P1, g0, g1, p2max, ctx->scratch[which].as<u64>(), ctx->bfill.as<u32>(), ovf);
                    else        k_scatter2<false><<<std::min<u32>(nt, grid_for(ctx, 5)), S2_THREADS, smem2, s2>>>(pi, pl, P1, g0, g1, p2max, ctx->scratch[which].as<u64>(), ctx->bfill.as<u32>(), ovf);
                    CKL(); LAUNCHED(ctx);
                    k_count_buckets<<<std::min<u32>(nb, grid_for(ctx, 2)), CB_THREADS, smemc, s2>>>(pl, g0, g1, ctx->scratch[which].as<u64>(), ctx->bfill.as<u32>(), ovf,
                        lower, upper, ctx->rel_key.as<u64>(), ctx->rel_cnt.as<u32>(), d_ctr, rel_cap);
                    CKL(); LAUNCHED(ctx);
                    which ^= 1;
                }
                g0 = g1;
            }
            if (used_aux) { CK(cudaEventRecord(ctx->ev_join, ctx->aux)); CK(cudaStreamWaitEvent(st, ctx->ev_join, 0)); }
            CK(cudaEventRecord(ep.b, st));

            // ---- what the fast path gave up on: instances of overflowing sub-buckets (repeat-rich / heavy hitters) and
            //      partitions too large for MAX_P2 sub-buckets -> exact global-table count
            u64 novf = 0;
            CK(cudaMemcpyAsync(&novf, d_ctr + 5, 8, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            u64 retry = novf > ovf_cap;
            if (retry) ctx->ovf_cap = novf + (novf >> 3);      // the list length does not depend on scheduling: exact next time
            if (W > 1) { int rc0 = allreduce_u64(ctx, &retry, 1, ncclMax); if (rc0) return rc0; }      // collective: everybody redoes the exchange
            if (retry)
            {
                if (attempt == 3) return fail(ctx, ELBA_FE_ERR_CUDA, "overflow list resize did not converge");
                continue;
            }
            ctx->sz.slow_partitions = slow.size(); ctx->sz.overflow_instances = novf;
            if (novf)
            {
                std::vector<std::pair<const u64*, u64>> slabs{{ctx->ovf.as<u64>(), novf}};
                int rc = count_with_global_table(ctx, slabs, novf, rel_cap);
                if (rc) return rc;
            }
            for (u32 p : slow)
            {
                std::vector<std::pair<const u64*, u64>> slabs;
                for (int j = 0; j < W; ++j)
                    slabs.push_back({lvl2_in + (u64)j * slab_stride + (W > 1 ? (u64)p * cap1 : start[p]), (u64)cnt_all[(size_t)j * Pown + p]});
                int rc = count_with_global_table(ctx, slabs, ntot[p], rel_cap);
                if (rc) return rc;
            }
        }
        u64 h[4];
        CK(cudaMemcpyAsync(h, d_ctr, sizeof h, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        R = h[0]; sumcnt = h[1]; D = h[2];
        if ((u32)h[3] != 0) return fail(ctx, ELBA_FE_ERR_CUDA, "count table overflow");
        u64 retry = R > rel_cap;
        if (W > 1) { int rc0 = allreduce_u64(ctx, &retry, 1, ncclMax); if (rc0) return rc0; }
        if (!retry) break;
        if (attempt == 3) return fail(ctx, ELBA_FE_ERR_CUDA, "reliable list overflow after resize");
        rel_cap = std::max(rel_cap, R);       // exact; redo the count
    }
    ctx->sz.distinct = D; ctx->sz.nnzA_pre = sumcnt;
    // super-k-mer path: the list has holes (h = EMPTY_H -> k-mer = all ones, sorted behind every k-mer); R_list entries, R k-mers
    u64 R_list = R;
    if (use_skm) R = ctx->skm_reliable;

    u64 *rk = ctx->rel_key.as<u64>(); u32 *rc_ = ctx->rel_cnt.as<u32>();
    if (W > 1 && ctx->seeds_fused)
    {
        // ---- several GPUs, super-k-mer path: NOTHING is replicated.  Every GPU sorts the reliable k-mers it owns; the sorted
        // runs are all-gathered (8 B per k-mer) and the column id of a k-mer = its rank in the own run + the number of smaller
        // k-mers in every other run (binary searches, k_rank_global).  (reference: the Allreduce / Exscan of src/KmerOps.cpp:371-374)
        const u64 Rl = ctx->skm_reliable;
        if (R_list >= 0xFFFFFFF0ull) return fail(ctx, ELBA_FE_ERR_INVALID, "more than 2^32 entries in the reliable list of one context");
        CK(ctx->rel_key_s.ensure(8 * std::max<u64>(R_list, 1))); CK(ctx->rel_cnt_s.ensure(4 * std::max<u64>(R_list, 1)));
        CK(ctx->rel_idx.ensure(4 * std::max<u64>(R_list, 1))); CK(ctx->rel_idx_s.ensure(4 * std::max<u64>(R_list, 1))); CK(ctx->perm.ensure(4 * std::max<u64>(R_list, 1)));
        CK(ctx->rel_gid.ensure(4 * std::max<u64>(Rl, 1)));
        if (R_list) { k_iota_u32<<<nblk(R_list, 256), 256, 0, st>>>(ctx->rel_idx.as<u32>(), R_list); CKL(); LAUNCHED(ctx); }
        int rc1 = sort_pairs(ctx, rk, ctx->rel_key_s.as<u64>(), ctx->rel_idx.as<u32>(), ctx->rel_idx_s.as<u32>(), R_list, 64 - 2 * k, 64);
        if (rc1) return rc1;
        mark(ctx, "sort_own_kmers");
        if ((rc1 = allgather_u64(ctx, Rl, ctx->rel_counts))) return rc1;
        u64 Rt = 0; for (u64 v : ctx->rel_counts) Rt += v;
        if (Rt >= 0xFFFFFFFFull) return fail(ctx, ELBA_FE_ERR_INVALID, "more than 2^32 reliable k-mers");
        CK(ctx->rel_all_key.ensure(8 * std::max<u64>(Rt, 1)));
        if ((rc1 = allgatherv(ctx, ctx->rel_key_s.p, ctx->rel_all_key.p, ctx->rel_counts, 8))) return rc1;
        mark(ctx, "allgather_runs");
        RankRuns runs; std::memset(&runs, 0, sizeof runs);
        { u64 o = 0; for (int r = 0; r < W; ++r) { runs.off[r] = o; runs.n[r] = ctx->rel_counts[r]; o += ctx->rel_counts[r]; } }
        runs.nruns = (u32)W; runs.me = (u32)me;
        if (Rl) { k_rank_global<<<nblk(Rl, RG_KEYS), 256, 0, st>>>(ctx->rel_key_s.as<u64>(), ctx->rel_idx_s.as<u32>(), rc_, Rl, ctx->rel_all_key.as<u64>(), runs,
                      ctx->perm.as<u32>(), ctx->rel_cnt_s.as<u32>(), ctx->rel_gid.as<u32>()); CKL(); LAUNCHED(ctx); }
        ctx->R_local = Rl; ctx->kmers_distributed = true; ctx->seed_id_base = 0;
        ctx->sz.reliable = Rt;
        CK(cudaEventRecord(ctx->ev[3], st));
        mark(ctx, "rank_global"); trace_flush(ctx, "count");
        ctx->phase = 2;
        return 0;
    }
    // ---- several GPUs, hash path: every rank needs the whole reliable list (column ids are ranks among ALL reliable k-mers)
    if (W > 1)
    {
        std::vector<u64> Rr;
        int rc0 = allgather_u64(ctx, R_list, Rr); if (rc0) return rc0;
        if ((rc0 = allreduce_u64(ctx, &R, 1, ncclSum))) return rc0;       // k-mers (the lists may hold holes)
        u64 Rt = 0; for (u64 v : Rr) Rt += v;
        CK(ctx->rel_all_key.ensure(sizeof(u64) * std::max<u64>(Rt, 1))); CK(ctx->rel_all_cnt.ensure(sizeof(u32) * std::max<u64>(Rt, 1)));
        if ((rc0 = allgatherv(ctx, ctx->rel_key.p, ctx->rel_all_key.p, Rr, sizeof(u64)))) return rc0;
        if ((rc0 = allgatherv(ctx, ctx->rel_cnt.p, ctx->rel_all_cnt.p, Rr, sizeof(u32)))) return rc0;
        rk = ctx->rel_all_key.as<u64>(); rc_ = ctx->rel_all_cnt.as<u32>(); R_list = Rt;
    }
    ctx->seed_id_base = 0;
    if (R >= 0xFFFFFFFFull) return fail(ctx, ELBA_FE_ERR_INVALID, "more than 2^32 reliable k-mers on one context");
    ctx->sz.reliable = R;

    CK(ctx->rel_key_s.ensure(sizeof(u64) * std::max<u64>(R_list, 1))); CK(ctx->rel_cnt_s.ensure(sizeof(u32) * std::max<u64>(R_list, 1)));
    int rc;
    if (ctx->seeds_fused)
    {
        // super-k-mer path: the list holds the k-mers themselves (holes = all ones, sorted behind every k-mer) and the seeds name
        // their k-mer by its list index: column id = rank by value = where the sort puts the entry; perm[list index] = column id.
        // No k-mer -> column hash table is built (round 1: 34 M random CAS into an 826 MB table per pass).
        if (R_list >= 0xFFFFFFF0ull) return fail(ctx, ELBA_FE_ERR_INVALID, "more than 2^32 entries in the reliable lists");
        CK(ctx->rel_idx.ensure(4 * std::max<u64>(R_list, 1))); CK(ctx->rel_idx_s.ensure(4 * std::max<u64>(R_list, 1))); CK(ctx->perm.ensure(4 * std::max<u64>(R_list, 1)));
        if (R_list) { k_iota_u32<<<nblk(R_list, 256), 256, 0, st>>>(ctx->rel_idx.as<u32>(), R_list); CKL(); LAUNCHED(ctx); }
        rc = sort_pairs(ctx, rk, ctx->rel_key_s.as<u64>(), ctx->rel_idx.as<u32>(), ctx->rel_idx_s.as<u32>(), R_list, 64 - 2 * k, 64);
        if (rc) return rc;
        if (R) { k_rank_finish<<<nblk(R, 256), 256, 0, st>>>(ctx->rel_idx_s.as<u32>(), rc_, R, ctx->perm.as<u32>(), ctx->rel_cnt_s.as<u32>()); CKL(); LAUNCHED(ctx); }
    }
    else
    {
    // the lists hold h = mix64(k-mer): back to k-mers, then column ids = rank by k-mer value: sort (key, count) by key
    if (R_list) { k_unmix<<<nblk(R_list, 256), 256, 0, st>>>(rk, R_list); CKL(); LAUNCHED(ctx); }
    rc = sort_pairs(ctx, rk, ctx->rel_key_s.as<u64>(), rc_, ctx->rel_cnt_s.as<u32>(), R_list, 64 - 2 * k, 64);    // the first R of R_list are k-mers
    if (rc) return rc;
    // k-mer -> column id table in HBM, fronted by a blocked Bloom filter sized to stay L2-resident
    u64 lslots = std::max<u64>(R + R / 2 + 64, 1024);
    if (lslots >= (1ull << 32)) return fail(ctx, ELBA_FE_ERR_INVALID, "too many reliable k-mers for the column table");
    CK(ctx->lut.ensure(sizeof(Slot) * lslots));
    ctx->lut_slots = (u32)lslots;
    const u64 bits_per_key = (R * 2 <= (32ull << 20)) ? 16 : (R * 3 / 2 <= (64ull << 20)) ? 12 : 8;
    u64 fwords = std::max<u64>((R * bits_per_key + 63) / 64, 1024);
    CK(ctx->filter.ensure(8 * fwords));
    ctx->filter_words = (u32)fwords;
    CK(cudaMemsetAsync(ctx->filter.p, 0, 8 * fwords, st));
    k_table_clear<<<grid_for(ctx, 4), 256, 0, st>>>(ctx->lut.as<Slot>(), lslots, EMPTY_KEY); CKL(); LAUNCHED(ctx);
    if (R) { k_lookup_build<<<nblk(R, 256), 256, 0, st>>>(ctx->rel_key_s.as<u64>(), ctx->rel_cnt_s.as<u32>(), (u32)R, ctx->lut.as<Slot>(), ctx->lut_slots,
                                                       ctx->filter.as<u64>(), ctx->filter_words); CKL(); LAUNCHED(ctx); }
    }
    CK(cudaEventRecord(ctx->ev[3], st));
    mark(ctx, "column_ids"); trace_flush(ctx, "count");
    ctx->phase = 2;
    return 0;
}

// Several GPUs: block (i, j) of B = A[R_i, :] (x) A[C_j, :]^T on rank i * pc + j, inner (k-mer) dimension unsplit, so every
// nonzero is folded on exactly one GPU in the canonical order and no partial results are merged across GPUs (the
// reference's Sparse SUMMA, src/SharedSeeds.cpp:7, broadcasts panels stage by stage and merges).  Every rank built the
// rows of A of its own reads; one all-gather of those row blocks gives each GPU all of A (read-major, already sorted,
// since the ranks hold consecutive read ranges), from which it slices R_i as the left CSR and re-sorts C_j as the
// right CSC.
static int operands_from_gathered(elba_fe_ctx *ctx, u64 tot);

static int gather_operands(elba_fe_ctx *ctx)
{
    cudaStream_t st = ctx->stream;
    const u64 nnzA = ctx->sz.nnzA; const u32 N = ctx->n;
    std::vector<u64> nz;
    int rc = allgather_u64(ctx, nnzA, nz); if (rc) return rc;
    u64 tot = 0; for (u64 v : nz) tot += v;
    CK(ctx->pack_key.ensure(8 * std::max<u64>(nnzA, 1)));
    CK(ctx->g_key.ensure(8 * std::max<u64>(tot, 1))); CK(ctx->g_pos.ensure(4 * std::max<u64>(tot, 1)));
    if (N) { k_pack_rows<<<nblk((u64)N * 32, 256), 256, 0, st>>>(ctx->a_rowptr.as<int64_t>(), ctx->a_col.as<u32>(), N, (u64)ctx->read_id_offset, ctx->pack_key.as<u64>()); CKL(); LAUNCHED(ctx); }
    if ((rc = allgatherv(ctx, ctx->pack_key.p, ctx->g_key.p, nz, 8))) return rc;
    if ((rc = allgatherv(ctx, ctx->a_pos.p, ctx->g_pos.p, nz, 4))) return rc;
    ctx->panel_bytes += 12 * (tot - nnzA);
    mark(ctx, "allgather_A");
    return operands_from_gathered(ctx, tot);
}

// g_key (global read << 32 | column, ascending) / g_pos hold ALL of A (tot entries): slice R_i as the left CSR, re-sort C_j as the right CSC
static int operands_from_gathered(elba_fe_ctx *ctx, u64 tot)
{
    cudaStream_t st = ctx->stream;
    const int me = ctx->comm.rank, pr = ctx->comm.grid_rows, pc = ctx->comm.grid_cols;
    const u64 R = ctx->sz.reliable;
    int rc;
    const int bi = me / pc, bj = me % pc;
    int64_t row0, nr, col0, ncb;
    block_extent((int64_t)ctx->N_total, pr, bi, row0, nr);
    block_extent((int64_t)ctx->N_total, pc, bj, col0, ncb);
    row0 += ctx->read_base0; col0 += ctx->read_base0;                    // the gathered keys carry GLOBAL read ids, which start at rank 0's offset
    // left: rows R_i are one contiguous slice
    CK(ctx->l_rowptr.ensure(8 * ((size_t)nr + 2))); CK(ctx->r_ptr.ensure(8 * ((size_t)ncb + 2)));
    k_read_ptr<<<nblk((u64)nr + 1, 256), 256, 0, st>>>(ctx->g_key.as<u64>(), tot, (u64)row0, (u64)nr, ctx->l_rowptr.as<int64_t>()); CKL(); LAUNCHED(ctx);
    k_read_ptr<<<nblk((u64)ncb + 1, 256), 256, 0, st>>>(ctx->g_key.as<u64>(), tot, (u64)col0, (u64)ncb, ctx->r_ptr.as<int64_t>()); CKL(); LAUNCHED(ctx);
    int64_t lb = 0, le = 0, rb = 0, re = 0;
    CK(cudaMemcpyAsync(&lb, ctx->l_rowptr.as<int64_t>(), 8, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&le, ctx->l_rowptr.as<int64_t>() + nr, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&rb, ctx->r_ptr.as<int64_t>(), 8, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&re, ctx->r_ptr.as<int64_t>() + ncb, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    const u64 ln = (u64)(le - lb), rn = (u64)(re - rb);
    CK(ctx->l_col.ensure(4 * std::max<u64>(ln, 1)));
    k_sub_base<<<nblk((u64)nr + 1, 256), 256, 0, st>>>(ctx->l_rowptr.as<int64_t>(), (u64)nr, lb); CKL(); LAUNCHED(ctx);
    if (ln) { k_slice_left<<<nblk(ln, 256), 256, 0, st>>>(ctx->g_key.as<u64>(), (u64)lb, ln, ctx->l_col.as<u32>()); CKL(); LAUNCHED(ctx); }
    // both operands by column for the expand step (spgemm2.cuh): the slices are sorted by read, a STABLE sort by the column id
    // alone (4 radix passes instead of 6) leaves the reads ascending inside every column
    const int cb = bits_for(std::max<u64>(R, 2));
    if (ln >= (1ull << 32) || rn >= (1ull << 32)) return fail(ctx, ELBA_FE_ERR_INVALID, "an SpGEMM operand of one GPU exceeds 2^32 entries");
    const u64 mx = std::max<u64>(std::max(ln, rn), 1);
    CK(ctx->sp_col.ensure(4 * mx)); CK(ctx->sp_col2.ensure(4 * mx)); CK(ctx->sp_val.ensure(8 * mx)); CK(ctx->sp_val2.ensure(8 * mx));
    CK(ctx->lp_ptr.ensure(4 * (R + 2))); CK(ctx->lp_ent.ensure(8 * std::max<u64>(ln, 1)));
    CK(ctx->sp_ptr.ensure(4 * (R + 2))); CK(ctx->sp_ent.ensure(8 * std::max<u64>(rn, 1)));
    for (int side = 0; side < 2; ++side)
    {
        const u64 b0 = side ? (u64)rb : (u64)lb, n = side ? rn : ln, r0 = side ? (u64)col0 : (u64)row0;
        u32 *cptr = side ? ctx->sp_ptr.as<u32>() : ctx->lp_ptr.as<u32>(); uint2 *ent = side ? ctx->sp_ent.as<uint2>() : ctx->lp_ent.as<uint2>();
        if (n) { k_sp2_slice<<<nblk(n, 256), 256, 0, st>>>(ctx->g_key.as<u64>(), ctx->g_pos.as<u32>(), b0, n, r0, ctx->sp_col.as<u32>(), ctx->sp_val.as<u64>()); CKL(); LAUNCHED(ctx); }
        if ((rc = sort_pairs_u32_u64(ctx, ctx->sp_col.as<u32>(), ctx->sp_col2.as<u32>(), ctx->sp_val.as<u64>(), ctx->sp_val2.as<u64>(), n, 0, cb))) return rc;
        k_sp2_colptr<<<nblk(n + 1, 256), 256, 0, st>>>(ctx->sp_col2.as<u32>(), n, R, cptr); CKL(); LAUNCHED(ctx);
        if (n) { k_sp2_unpack_val<<<nblk(n, 256), 256, 0, st>>>(ctx->sp_val2.as<u64>(), n, ent); CKL(); LAUNCHED(ctx); }
    }
    ctx->op.l_rowptr = ctx->l_rowptr.as<int64_t>(); ctx->op.l_col = ctx->l_col.as<u32>(); ctx->op.l_pos = ctx->g_pos.as<u32>() + lb; ctx->op.l_rows = (u32)nr; ctx->op.l_nnz = ln;
    ctx->op.r_colptr = nullptr; ctx->op.r_row = nullptr; ctx->op.r_pos = nullptr; ctx->op.r_nnz = rn;
    ctx->op.row0 = row0; ctx->op.col0 = col0; ctx->op_r_rows = (u32)ncb;
    ctx->op_l_cptr = ctx->lp_ptr.as<u32>(); ctx->op_l_cent = ctx->lp_ent.as<uint2>();
    return 0;
}

// A^T of the rows of this GPU (src/main.cpp:272-273) in the form the SpGEMM reads: 32-bit column pointers, {row, pos} entries.
// A is sorted by (read, column): a STABLE sort by the column id alone (4 radix passes of a 32-bit key instead of 6 of a 64-bit
// one) leaves the reads ascending inside every column; the column pointers come from the boundaries of the sorted ids.
static int build_local_transpose(elba_fe_ctx *ctx, u32 *cptr, uint2 *ent)
{
    cudaStream_t st = ctx->stream;
    const u64 nnzA = ctx->sz.nnzA, R = ctx->sz.reliable;
    const int cb = ctx->col_bits;
    int rc;
    const u64 na = std::max<u64>(nnzA, 1);
    CK(ctx->sp_col.ensure(4 * na)); CK(ctx->sp_col2.ensure(4 * na)); CK(ctx->sp_val.ensure(8 * na)); CK(ctx->sp_val2.ensure(8 * na));
    if (nnzA) { k_csr_to_colsort<<<nblk(nnzA, 256), 256, 0, st>>>(ctx->a_key.as<u64>(), ctx->a_pos.as<u32>(), nnzA, cb, ctx->sp_col.as<u32>(), ctx->sp_val.as<u64>()); CKL(); LAUNCHED(ctx); }
    if ((rc = sort_pairs_u32_u64(ctx, ctx->sp_col.as<u32>(), ctx->sp_col2.as<u32>(), ctx->sp_val.as<u64>(), ctx->sp_val2.as<u64>(), nnzA, 0, cb))) return rc;
    k_sp2_colptr<<<nblk(nnzA + 1, 256), 256, 0, st>>>(ctx->sp_col2.as<u32>(), nnzA, R, cptr); CKL(); LAUNCHED(ctx);
    if (nnzA) { k_sp2_unpack_val<<<nblk(nnzA, 256), 256, 0, st>>>(ctx->sp_val2.as<u64>(), nnzA, ent); CKL(); LAUNCHED(ctx); }
    return 0;
}

// -------------------------------------------------------------------------------------------------
int elba_fe_build_A(elba_fe_ctx *ctx)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (ctx->phase < 2) return fail(ctx, ELBA_FE_ERR_STATE, "elba_fe_build_A: call elba_fe_count first");
    ctx->og_aligned = ctx->og_done = ctx->ct_done = ctx->pf_done = false;
    CK(cudaSetDevice(ctx->cfg.device));
    cudaStream_t st = ctx->stream;
    ReadsView rv = view(ctx);
    const u64 R = ctx->sz.reliable; u64 npre = ctx->sz.nnzA_pre; const u32 N = ctx->n;
    const int W = ctx->comm.nranks;
    CK(cudaEventRecord(ctx->ev[4], st));
    mark(ctx, "begin");
    ctx->lev_used = 0; ctx->panel_bytes = 0;
    { int rcw = wait_reads(ctx); if (rcw) return rcw; }
    const int cb = bits_for(std::max<u64>(R, 2)), rb = bits_for(std::max<u64>(N, 2));
    ctx->col_bits = cb; ctx->read_bits = rb;
    u64 *d_ctr = ctx->ctr.as<u64>();
    CK(cudaMemsetAsync(d_ctr, 0, 64, st));
    // one GPU: counting already told how many instances belong to reliable k-mers.  Several GPUs: that number is
    // known per OWNER, not per reader, so the triple buffers are sized by what arrives.
    u64 cap = std::max<u64>(npre, 1);
    const bool fused = ctx->seeds_fused;
    const bool routed = fused && W > 1;                    // several GPUs, super-k-mer path: the k-mer owners send the triples to the read owners
    u64 nsort = 0;                                         // entries handed to the (read, column) sort
    bool holes = false;                                    // ... some of which are holes of the chunked seed list (sorted behind the triples)
    if (fused && !routed) cap = std::max<u64>(ctx->nseeds_fused, 1);
    if ((W == 1 || fused) && !routed) { CK(ctx->seed_key.ensure(8 * cap)); CK(ctx->seed_pos.ensure(4 * cap)); }
    // sweep 2: every instance of a reliable k-mer -> (read, column, pos)
    u64 emitted = 0;
    {
        EventPair &lp = next_pair(ctx->lev, ctx->lev_used);
        CK(cudaEventRecord(lp.a, st));
        if (routed)
        {
            // The seeds lie with the OWNERS of the k-mers; the rows of A belong to the owners of the reads.  Every GPU turns its
            // seeds into (global read, column, pos) and stores each straight into the read owner's receive window through peer
            // memory (region [source][route_cap] of that window; the slot comes from a local cursor per destination): the
            // reference's second exchange (src/KmerOps.cpp:274) without packing, 12 B per instance of a reliable k-mer.
            const u64 ncand = ctx->nseeds_fused;
            ctx->sz.candidates = ncand;
            u64 most = ncand; int rc0;
            if ((rc0 = allreduce_u64(ctx, &most, 1, ncclMax))) return rc0;
            const u64 rcap_t = std::max<u64>(ctx->route_cap, most / (u64)W + most / (u64)(2 * W) + (1u << 16));      // same on every rank
            ctx->route_cap = rcap_t;
            if ((rc0 = window_ensure(ctx, ctx->w_rkey, 8 * rcap_t * (u64)W))) return rc0;
            if ((rc0 = window_ensure(ctx, ctx->w_rpos, 4 * rcap_t * (u64)W))) return rc0;
            if ((rc0 = window_ensure(ctx, ctx->w_rcnt, 8 * (size_t)SK_MAXW))) return rc0;
            CK(ctx->route_cur.ensure(8 * (size_t)SK_MAXW));
            CK(cudaMemsetAsync(ctx->route_cur.p, 0, 8 * (size_t)SK_MAXW, st));
            if ((rc0 = stream_barrier(ctx))) return rc0;          // the windows of the previous pass have been read
            RouteSink rs; std::memset(&rs, 0, sizeof rs);
            for (int r = 0; r < W; ++r) { rs.key[r] = (u64*)ctx->w_rkey.peer[r]; rs.pos[r] = (u32*)ctx->w_rpos.peer[r]; rs.cnt[r] = (u64*)ctx->w_rcnt.peer[r]; rs.first[r] = ctx->roff[r]; }
            rs.first[W] = ctx->roff[W]; rs.nranks = (u32)W; rs.me = (u32)ctx->comm.rank; rs.cap = rcap_t; rs.cursor = ctx->route_cur.as<u64>();
            if (ncand) { k_seed_route<<<grid_for(ctx, 4), 256, 0, st>>>(ctx->seeds.as<Seed>(), ncand, ctx->perm.as<u32>(), rs); CKL(); LAUNCHED(ctx); }
            k_route_publish<<<1, 32, 0, st>>>(rs); CKL(); LAUNCHED(ctx);
            if ((rc0 = stream_barrier(ctx))) return rc0;          // every source has stored its triples and its counts
            u64 got[SK_MAXW];
            CK(cudaMemcpyAsync(got, ctx->w_rcnt.buf.p, 8 * (size_t)W, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            u64 tot = 0, over = 0;
            for (int r = 0; r < W; ++r) { if (got[r] > rcap_t) over = std::max(over, got[r]); tot += std::min(got[r], rcap_t); }
            if ((rc0 = allreduce_u64(ctx, &over, 1, ncclMax))) return rc0;
            if (over) { ctx->route_cap = over + over / 8; return fail(ctx, ELBA_FE_ERR_CUDA, "seed routing window too small (the reads are very unevenly distributed over the GPUs): call elba_fe_build_A again"); }
            const u64 t1 = std::max<u64>(tot, 1);
            CK(ctx->seed_key.ensure(8 * t1)); CK(ctx->seed_pos.ensure(4 * t1));
            u64 o = 0;
            for (int r = 0; r < W; ++r)
            {
                if (got[r]) { k_route_unpack<<<nblk(got[r], 256), 256, 0, st>>>(ctx->w_rkey.buf.as<u64>() + rcap_t * (u64)r, ctx->w_rpos.buf.as<u32>() + rcap_t * (u64)r, got[r],
                                  (u64)ctx->read_id_offset, cb, ctx->seed_key.as<u64>() + o, ctx->seed_pos.as<u32>() + o); CKL(); LAUNCHED(ctx); }
                o += got[r];
            }
            ctx->panel_bytes = 12 * (tot - got[ctx->comm.rank]);
            CK(cudaMemsetAsync(d_ctr, 0, 8, st));
            emitted = tot; nsort = tot;
        }
        else if (fused)
        {
            // counting already listed every instance of a reliable k-mer as {list index, pos, read} (skm_count.cuh): the column id
            // is perm[list index]; holes keep a key that sorts behind every entry
            const u64 ncand = ctx->nseeds_fused;
            ctx->sz.candidates = ncand;
            nsort = ncand; holes = true;
            const u64 hole_key = 1ull << (cb + rb);
            if (ncand) { k_seed_keys<<<grid_for(ctx, 8), 256, 0, st>>>(ctx->seeds.as<Seed>(), ncand, ctx->perm.as<u32>(), 0u, cb, hole_key,
                             ctx->seed_key.as<u64>(), ctx->seed_pos.as<u32>(), d_ctr); CKL(); LAUNCHED(ctx); }
        }
        else if (ctx->nchunks && R)
        {
            // candidates = true instances + filter false positives (a few % of all instances); exact size after one try
            const u64 chunk_slack = (u64)grid_for(ctx, 2) * (PF_THREADS / 32) * PF_CHUNK;     // every warp may leave one chunk partly used
            u64 ccap = std::max<u64>(ctx->cand_cap, npre + std::max<u64>(ctx->Ms / 32, 1u << 16) + chunk_slack);
            for (int attempt = 0; attempt < 3; ++attempt)
            {
                CK(ctx->cand.ensure(sizeof(Candidate) * ccap));
                ctx->cand_cap = ccap;
                CK(cudaMemsetAsync(d_ctr, 0, 64, st));
                k_probe_filter<<<grid_for(ctx, 2), PF_THREADS, 0, st>>>(rv, ctx->cfg.k, ctx->cfg.stride, ctx->filter.as<u64>(), ctx->filter_words,
                    ctx->cand.as<Candidate>(), d_ctr + 1, ccap);
                CKL(); LAUNCHED(ctx);
                u64 ncand = 0;
                CK(cudaMemcpyAsync(&ncand, d_ctr + 1, 8, cudaMemcpyDeviceToHost, st));
                CK(cudaStreamSynchronize(st));
                ctx->sz.candidates = ncand;
                if (ncand > ccap) { if (attempt == 2) return fail(ctx, ELBA_FE_ERR_CUDA, "candidate list overflow after resize"); ccap = ncand + ncand / 8 + chunk_slack; continue; }
                if (W > 1) { cap = std::max<u64>(ncand, 1); CK(ctx->seed_key.ensure(8 * cap)); CK(ctx->seed_pos.ensure(4 * cap)); }
                if (ncand) { k_resolve<<<grid_for(ctx, 8), 256, 0, st>>>(ctx->cand.as<Candidate>(), ncand, ctx->lut.as<Slot>(), ctx->lut_slots,
                                 ctx->seed_key.as<u64>(), ctx->seed_pos.as<u32>(), d_ctr, cap, cb); CKL(); LAUNCHED(ctx); }
                break;
            }
        }
        CK(cudaEventRecord(lp.b, st));
        if (!routed)
        {
            CK(cudaMemcpyAsync(&emitted, d_ctr, 8, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
        }
    }
    {
        // every instance of a reliable k-mer must have been found again: emitted == what counting promised (summed over the GPUs)
        u64 chk[2] = {emitted, npre};
        if (W > 1) { int rc0 = allreduce_u64(ctx, chk, 2, ncclSum); if (rc0) return rc0; }
        if (chk[0] != chk[1]) { char b[160]; snprintf(b, sizeof b, "seed emission produced %llu triples, counting promised %llu", (unsigned long long)chk[0], (unsigned long long)chk[1]); return fail(ctx, ELBA_FE_ERR_CUDA, b); }
        npre = emitted;
        if (!fused) nsort = npre;
        const u64 ns1 = std::max<u64>(nsort, 1);
        CK(ctx->seed_key.ensure(8 * ns1)); CK(ctx->seed_pos.ensure(4 * ns1));
        CK(ctx->seed_key2.ensure(8 * ns1)); CK(ctx->seed_pos2.ensure(4 * ns1));
    }

    mark(ctx, "seeds_to_triples");
    int rc;
    u64 nnzA = 0;
    // sort by (read, column); merge duplicates keeping the largest position
    if ((rc = sort_pairs(ctx, ctx->seed_key.as<u64>(), ctx->seed_key2.as<u64>(), ctx->seed_pos.as<u32>(), ctx->seed_pos2.as<u32>(), nsort, 0, cb + rb + (holes ? 1 : 0)))) return rc;      // the first npre are triples, holes behind
    CK(ctx->idx.ensure(8 * (npre + 1)));
    k_mark_run_ends<<<nblk(npre + 1, 256), 256, 0, st>>>(ctx->seed_key2.as<u64>(), npre, ctx->idx.as<u64>()); CKL(); LAUNCHED(ctx);
    if ((rc = exclusive_scan_inplace(ctx, ctx->idx.as<u64>(), npre + 1))) return rc;
    CK(cudaMemcpyAsync(&nnzA, ctx->idx.as<u64>() + npre, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    ctx->sz.nnzA = nnzA;
    const u64 na = std::max<u64>(nnzA, 1);
    CK(ctx->a_key.ensure(8 * na)); CK(ctx->a_pos.ensure(4 * na)); CK(ctx->a_col.ensure(4 * na)); CK(ctx->a_rowptr.ensure(8 * ((size_t)N + 2)));
    if (npre) { k_dedupe_write<<<nblk(npre, 256), 256, 0, st>>>(ctx->seed_key2.as<u64>(), ctx->seed_pos2.as<u32>(), ctx->idx.as<u64>(), npre, ctx->a_key.as<u64>(), ctx->a_pos.as<u32>()); CKL(); LAUNCHED(ctx); }
    k_segment_ptr<<<nblk((u64)N + 1, 256), 256, 0, st>>>(ctx->a_key.as<u64>(), nnzA, N, cb, ctx->a_rowptr.as<int64_t>()); CKL(); LAUNCHED(ctx);
    if (nnzA) { k_split_swap<<<nblk(nnzA, 256), 256, 0, st>>>(ctx->a_key.as<u64>(), nnzA, cb, rb, ctx->a_col.as<u32>(), nullptr); CKL(); LAUNCHED(ctx); }
    mark(ctx, "sort_dedupe_csr");
    // transpose: the same entries by column.  One GPU: it is both operands of the expand step.  Several GPUs: the operands are
    // built from the gathered rows (gather_operands); the transpose of the own rows is only made when somebody asks for it (elba_fe_get_AT)
    ctx->at_built = false;
    ctx->op.l_rowptr = ctx->a_rowptr.as<int64_t>(); ctx->op.l_col = ctx->a_col.as<u32>(); ctx->op.l_pos = ctx->a_pos.as<u32>(); ctx->op.l_rows = N; ctx->op.l_nnz = nnzA;
    ctx->op.r_colptr = nullptr; ctx->op.r_row = nullptr; ctx->op.r_pos = nullptr; ctx->op.r_nnz = nnzA;
    ctx->op.row0 = ctx->op.col0 = ctx->read_id_offset;
    if (W == 1)
    {
        if (nnzA >= (1ull << 32)) return fail(ctx, ELBA_FE_ERR_INVALID, "the SpGEMM operand of one GPU exceeds 2^32 entries");
        CK(ctx->sp_ptr.ensure(4 * (R + 2))); CK(ctx->sp_ent.ensure(8 * na));
        if ((rc = build_local_transpose(ctx, ctx->sp_ptr.as<u32>(), ctx->sp_ent.as<uint2>()))) return rc;
        ctx->op_l_cptr = ctx->sp_ptr.as<u32>(); ctx->op_l_cent = ctx->sp_ent.as<uint2>(); ctx->op_r_rows = N;
    }
    mark(ctx, "csc");
    if (W > 1) { rc = gather_operands(ctx); if (rc) return rc; mark(ctx, "gather_operands"); }
    // products per row, F
    CK(ctx->prod.ensure(8 * ((size_t)ctx->op.l_rows + 1)));
    CK(cudaMemsetAsync(d_ctr, 0, 64, st));
    if (ctx->op.l_rows) { k_row_products32<<<nblk((u64)ctx->op.l_rows * 32, 256), 256, 0, st>>>(ctx->op.l_rowptr, ctx->op.l_col, ctx->sp_ptr.as<u32>(), ctx->op.l_rows, ctx->prod.as<u64>(), d_ctr); CKL(); LAUNCHED(ctx); }
    u64 F = 0;
    CK(cudaMemcpyAsync(&F, d_ctr, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaEventRecord(ctx->ev[5], st));
    CK(cudaStreamSynchronize(st));
    ctx->sz.products = F;
    mark(ctx, "spgemm_operand+row_products"); trace_flush(ctx, "build_A");
    ctx->phase = 3;
    return 0;
}

// rows with more distinct columns than the shared-memory table holds: global-memory tables (the rows are in ctx->ovf_rows)
static int spgemm_overflow_rows(elba_fe_ctx *ctx, const Sp2Args &A, u64 novf, u64 maxprod)
{
    cudaStream_t st = ctx->stream;
    u64 TS = next_pow2(2 * std::min<u64>(maxprod, (u64)ctx->op_r_rows) + 2);
    if (TS < 2 * SPG_BLOCK_TS) TS = 2 * SPG_BLOCK_TS;
    const u32 grid = (u32)std::min<u64>(novf, 64);
    CK(ctx->gscratch.ensure(sizeof(u32) * 5 * TS * grid));
    k_sp2_global<<<grid, SPG_BLOCK_THREADS, 0, st>>>(A, ctx->ovf_rows.as<u32>(), (u32)novf, ctx->gscratch.as<u32>(), (u32)TS); CKL(); LAUNCHED(ctx);
    return 0;
}

// -------------------------------------------------------------------------------------------------
int elba_fe_spgemm(elba_fe_ctx *ctx)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (ctx->phase < 3) return fail(ctx, ELBA_FE_ERR_STATE, "elba_fe_spgemm: call elba_fe_build_A first");
    ctx->og_aligned = ctx->og_done = ctx->ct_done = ctx->pf_done = false;
    CK(cudaSetDevice(ctx->cfg.device));
    cudaStream_t st = ctx->stream;
    const u32 N = ctx->op.l_rows; const u64 nnzA = ctx->op.l_nnz;       // rows of this GPU's block of B
    const u64 R = ctx->sz.reliable, F = ctx->sz.products;
    ctx->b_rows = N;
    CK(cudaEventRecord(ctx->ev[6], st));
    mark(ctx, "begin");
    ctx->sev_used = 0;
    CK(ctx->row_off.ensure(8 * ((size_t)N + 1))); CK(ctx->row_nnz.ensure(4 * ((size_t)N + 1)));
    CK(ctx->small_rows.ensure(4 * ((size_t)N + 1))); CK(ctx->mid_rows.ensure(4 * ((size_t)N + 1))); CK(ctx->big_rows.ensure(4 * ((size_t)N + 1))); CK(ctx->ovf_rows.ensure(4 * ((size_t)N + 1)));
    CK(ctx->bins.ensure(64)); CK(ctx->b_rowptr.ensure(8 * ((size_t)N + 2)));
    CK(ctx->tup_cnt.ensure(8 * ((size_t)N + 2))); CK(ctx->tup_cur.ensure(4 * ((size_t)N + 1)));
    // the tuple regions: row i gets exactly its products (minus the pairs of a read with itself, diagonal blocks only)
    k_sp2_tuple_counts<<<nblk((u64)N + 1, 256), 256, 0, st>>>(ctx->prod.as<u64>(), ctx->op.l_rowptr, N, ctx->op.row0, ctx->op.col0, ctx->op_r_rows, ctx->tup_cnt.as<u64>()); CKL(); LAUNCHED(ctx);
    int rc = exclusive_scan_inplace(ctx, ctx->tup_cnt.as<u64>(), (u64)N + 1);
    if (rc) return rc;
    // rounds: the tuples of all rows at once if they fit the budget (16 B each), else consecutive row ranges
    u64 budget = 48ull << 30;
    if (const char *e = getenv("ELBA_FE_TUPLE_MB")) { long long v = atoll(e); if (v >= 1) budget = (u64)v << 20; }
    std::vector<u32> cut{0, N};
    u64 tup_cap = std::max<u64>(F, 1);
    if (F * sizeof(Sp2Tuple) > budget && N > 1)
    {
        std::vector<u64> off((size_t)N + 1);
        CK(cudaMemcpyAsync(off.data(), ctx->tup_cnt.p, 8 * ((size_t)N + 1), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        cut.assign(1, 0); tup_cap = 1;
        const u64 per = budget / sizeof(Sp2Tuple);
        u32 r = 0;
        while (r < N)
        {
            u32 e = r + 1;                                              // at least one row per round, whatever its size
            while (e < N && off[e + 1] - off[r] <= per) ++e;
            tup_cap = std::max(tup_cap, off[e] - off[r]);
            cut.push_back(e); r = e;
        }
    }
    CK(ctx->tuples.ensure(sizeof(Sp2Tuple) * tup_cap));
    u64 cap = std::max<u64>(ctx->b_cap_hint, std::max<u64>(nnzA + N, 1024));
    u64 *d_ctr = ctx->ctr.as<u64>();
    u64 h[4] = {0, 0, 0, 0};
    for (int attempt = 0; attempt < 2; ++attempt)
    {
        CK(ctx->t_col.ensure(4 * cap)); CK(ctx->t_num.ensure(4 * cap)); CK(ctx->t_seeds.ensure(16 * cap));
        CK(cudaMemsetAsync(d_ctr, 0, 64, st)); CK(cudaMemsetAsync(ctx->bins.p, 0, 64, st));
        u32 *d_bins = ctx->bins.as<u32>(); u64 *d_maxprod = reinterpret_cast<u64*>(d_bins + 4);
        Sp2Operands op; op.l_cptr = ctx->op_l_cptr; op.l_cent = ctx->op_l_cent; op.r_cptr = ctx->sp_ptr.as<u32>(); op.r_cent = ctx->sp_ent.as<uint2>();
        op.ncol = R; op.row0 = ctx->op.row0; op.col0 = ctx->op.col0; op.l_rows = N; op.r_rows = ctx->op_r_rows;
        Sp2Args A;
        A.a_rowptr = ctx->op.l_rowptr; A.a_col = ctx->op.l_col; A.a_pos = ctx->op.l_pos;
        A.tup_off = ctx->tup_cnt.as<u64>(); A.tuples = ctx->tuples.as<Sp2Tuple>(); A.ra = 0; A.rb = N;
        A.row0 = ctx->op.row0; A.col0 = ctx->op.col0; A.r_rows = ctx->op_r_rows;
        A.nrows = N; A.seed_count = ctx->cfg.seed_count;
        A.t_col = ctx->t_col.as<u32>(); A.t_num = ctx->t_num.as<int32_t>(); A.t_seeds = ctx->t_seeds.as<u32>(); A.cap = cap;
        A.counters = d_ctr; A.row_off = ctx->row_off.as<u64>(); A.row_nnz = ctx->row_nnz.as<u32>();
        if (N)
        {
            // rows by their product count: a warp per light row (256-slot table), a CTA per heavy row (2048 slots), global tables beyond
            k_spgemm_bin<<<nblk(N, 256), 256, 0, st>>>(ctx->prod.as<u64>(), N, ctx->small_rows.as<u32>(), ctx->mid_rows.as<u32>(), ctx->big_rows.as<u32>(), d_bins, A.row_off, A.row_nnz, d_maxprod, 0u, SP2_WARP_MAXPROD);
            CKL(); LAUNCHED(ctx);
            EventPair &sp = next_pair(ctx->sev, ctx->sev_used);
            CK(cudaEventRecord(sp.a, st));
            for (size_t rd = 0; rd + 1 < cut.size(); ++rd)
            {
                A.ra = cut[rd]; A.rb = cut[rd + 1];
                CK(cudaMemsetAsync(ctx->tup_cur.p, 0, 4 * ((size_t)N + 1), st));
                if (R) { k_sp2_expand<<<grid_for(ctx, 8), 256, 0, st>>>(op, A.tup_off, ctx->tup_cur.as<u32>(), A.ra, A.rb, ctx->tuples.as<Sp2Tuple>()); CKL(); LAUNCHED(ctx); }
                if (cut.size() == 2) mark(ctx, "expand");
                k_sp2_warp<<<grid_for(ctx, 8), 32 * SP2_WARPS, 0, st>>>(A, ctx->small_rows.as<u32>(), d_bins, ctx->big_rows.as<u32>(), d_bins + 1); CKL(); LAUNCHED(ctx);
                if (cut.size() == 2) mark(ctx, "rows_warp");
                k_sp2_block<<<grid_for(ctx, 4), SPG_BLOCK_THREADS, 0, st>>>(A, ctx->big_rows.as<u32>(), d_bins + 1, ctx->ovf_rows.as<u32>()); CKL(); LAUNCHED(ctx);
                if (cut.size() == 2) mark(ctx, "rows_cta");
                if (cut.size() > 2)
                {
                    // several rounds: the rows of this round that overflowed the shared-memory table, before their tuples are overwritten
                    u64 hc[3];
                    CK(cudaMemcpyAsync(hc, d_ctr, sizeof hc, cudaMemcpyDeviceToHost, st));
                    u64 hbm[3];
                    CK(cudaMemcpyAsync(hbm, ctx->bins.p, sizeof hbm, cudaMemcpyDeviceToHost, st));
                    CK(cudaStreamSynchronize(st));
                    if (hc[2])
                    {
                        int rc2 = spgemm_overflow_rows(ctx, A, hc[2], hbm[2]); if (rc2) return rc2;
                        CK(cudaMemsetAsync(d_ctr + 2, 0, 8, st));
                    }
                }
            }
            CK(cudaEventRecord(sp.b, st));
        }
        u64 hb[6];
        CK(cudaMemcpyAsync(h, d_ctr, sizeof h, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(hb, ctx->bins.p, sizeof hb, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (h[2] && cut.size() == 2)
        {
            EventPair &sp = next_pair(ctx->sev, ctx->sev_used);
            CK(cudaEventRecord(sp.a, st));
            A.ra = 0; A.rb = N;
            int rc2 = spgemm_overflow_rows(ctx, A, h[2], hb[2]); if (rc2) return rc2;
            CK(cudaEventRecord(sp.b, st));
            CK(cudaMemcpyAsync(h, d_ctr, sizeof h, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
        }
        if (h[0] <= cap) break;
        if (attempt == 1) return fail(ctx, ELBA_FE_ERR_CUDA, "B storage overflow after resize");
        cap = h[0];
    }
    ctx->b_cap_hint = cap;
    const u64 nnzB = h[0];
    ctx->sz.nnzB = nnzB; ctx->sz.nnzB_pre = h[1];
    // CSR order
    CK(ctx->b_col.ensure(4 * std::max<u64>(nnzB, 1))); CK(ctx->b_num.ensure(4 * std::max<u64>(nnzB, 1))); CK(ctx->b_seeds.ensure(16 * std::max<u64>(nnzB, 1)));
    k_u32_to_u64<<<nblk((u64)N + 1, 256), 256, 0, st>>>(ctx->row_nnz.as<u32>(), N, reinterpret_cast<u64*>(ctx->b_rowptr.p)); CKL(); LAUNCHED(ctx);
    rc = exclusive_scan_inplace(ctx, reinterpret_cast<u64*>(ctx->b_rowptr.p), (u64)N + 1);
    if (rc) return rc;
    if (N)
    {
        k_gather_B<<<nblk((u64)N * 32, 256), 256, 0, st>>>(ctx->row_off.as<u64>(), ctx->row_nnz.as<u32>(), ctx->b_rowptr.as<int64_t>(), N,
            ctx->t_col.as<u32>(), ctx->t_num.as<int32_t>(), ctx->t_seeds.as<u32>(), ctx->b_col.as<u32>(), ctx->b_num.as<int32_t>(), ctx->b_seeds.as<u32>());
        CKL(); LAUNCHED(ctx);
    }
    CK(cudaEventRecord(ctx->ev[7], st));
    mark(ctx, "spgemm"); trace_flush(ctx, "spgemm");
    ctx->phase = 4; ctx->dc_built = false;
    return 0;
}

int elba_fe_run(elba_fe_ctx *ctx)
{
    int rc;
    if ((rc = elba_fe_count(ctx))) return rc;
    if ((rc = elba_fe_build_A(ctx))) return rc;
    if ((rc = elba_fe_spgemm(ctx))) return rc;
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int elba_fe_sizes(elba_fe_ctx *ctx, elba_fe_sizes_t *out)
{
    if (!ctx || !out) return ELBA_FE_ERR_INVALID;
    CK(cudaStreamSynchronize(ctx->stream));
    *out = ctx->sz;
    return 0;
}

int elba_fe_timings(elba_fe_ctx *ctx, elba_fe_timings_t *out)
{
    if (!ctx || !out) return ELBA_FE_ERR_INVALID;
    CK(cudaStreamSynchronize(ctx->stream));
    float ms;
    if (ctx->up_n > 0 && cudaEventElapsedTime(&ms, ctx->up_t0, ctx->up_ev[ctx->up_n - 1]) == cudaSuccess) ctx->tm.upload_ms = ms;      // the sliced H2D copy on the second stream
    if (ctx->phase >= 2 && cudaEventElapsedTime(&ms, ctx->ev[2], ctx->ev[3]) == cudaSuccess) ctx->tm.count_ms = ms;
    if (ctx->phase >= 3 && cudaEventElapsedTime(&ms, ctx->ev[4], ctx->ev[5]) == cudaSuccess) ctx->tm.build_ms = ms;
    if (ctx->phase >= 4 && cudaEventElapsedTime(&ms, ctx->ev[6], ctx->ev[7]) == cudaSuccess) ctx->tm.spgemm_ms = ms;
    if (ctx->phase >= 2) { ctx->tm.count_kernel_ms = sum_pairs(ctx->kev, ctx->kev_used); ctx->tm.partition_ms = sum_pairs(ctx->pev, ctx->pev_used); }
    if (ctx->phase >= 3) ctx->tm.lookup_ms = sum_pairs(ctx->lev, ctx->lev_used);
    if (ctx->phase >= 2 && ctx->comm.nranks > 1 && cudaEventElapsedTime(&ms, ctx->ev_x0, ctx->ev_x1) == cudaSuccess) ctx->tm.exchange_ms = ms;
    ctx->tm.exchange_mbytes = (float)((double)ctx->exchange_bytes / 1e6); ctx->tm.panel_mbytes = (float)((double)ctx->panel_bytes / 1e6);
    if (ctx->phase >= 4) ctx->tm.spgemm_kernel_ms = sum_pairs(ctx->sev, ctx->sev_used);
    *out = ctx->tm;
    return 0;
}

int elba_fe_reset_timings(elba_fe_ctx *ctx) { if (!ctx) return ELBA_FE_ERR_INVALID; std::memset(&ctx->tm, 0, sizeof ctx->tm); return 0; }


// ---- multi-GPU ------------------------------------------------------------------------------------------
int elba_fe_comm_get_id(elba_fe_comm_id *id)
{
    elba_fe_ctx *ctx = nullptr;
    if (!id) return fail(nullptr, ELBA_FE_ERR_INVALID, "null argument");
    static_assert(sizeof(elba_fe_comm_id) >= sizeof(ncclUniqueId), "elba_fe_comm_id must hold an ncclUniqueId");
    std::string err;
    NcclApi *api = nccl_api(err);
    if (!api) return fail(nullptr, ELBA_FE_ERR_COMM, err);
    ncclUniqueId nid;
    ncclResult_t r = api->GetUniqueId(&nid);
    if (r != ncclSuccess) return fail(nullptr, ELBA_FE_ERR_COMM, std::string("ncclGetUniqueId: ") + api->GetErrorString(r));
    std::memset(id, 0, sizeof *id);
    std::memcpy(id, &nid, sizeof nid);
    (void)ctx;
    return 0;
}

int elba_fe_comm_init(elba_fe_ctx *ctx, const elba_fe_comm_id *id, int rank, int nranks)
{
    if (!ctx || !id) return ELBA_FE_ERR_INVALID;
    if (nranks < 1 || rank < 0 || rank >= nranks) return fail(ctx, ELBA_FE_ERR_INVALID, "bad rank / nranks");
    if (nranks > 64) return fail(ctx, ELBA_FE_ERR_INVALID, "at most 64 ranks");
    if (ctx->comm.comm) return fail(ctx, ELBA_FE_ERR_STATE, "communicator already initialised");
    CK(cudaSetDevice(ctx->cfg.device));
    ctx->comm.rank = rank; ctx->comm.nranks = nranks;
    default_grid(nranks, ctx->comm.grid_rows, ctx->comm.grid_cols);
    if (nranks == 1) return 0;
    std::string err;
    ctx->comm.api = nccl_api(err);
    if (!ctx->comm.api) return fail(ctx, ELBA_FE_ERR_COMM, err);
    ncclUniqueId nid;
    std::memcpy(&nid, id, sizeof nid);
    NC(ctx->comm.api->CommInitRank(&ctx->comm.comm, nranks, nid, rank));
    return 0;
}

int elba_fe_comm_set_grid(elba_fe_ctx *ctx, int grid_rows, int grid_cols)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (grid_rows < 1 || grid_cols < 1 || grid_rows * grid_cols != ctx->comm.nranks) return fail(ctx, ELBA_FE_ERR_INVALID, "grid_rows * grid_cols must equal the number of ranks");
    ctx->comm.grid_rows = grid_rows; ctx->comm.grid_cols = grid_cols;
    return 0;
}

int elba_fe_comm_info(elba_fe_ctx *ctx, int *rank, int *nranks, int *grid_rows, int *grid_cols, int64_t *row0, int64_t *nrows, int64_t *col0, int64_t *ncols)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (rank) *rank = ctx->comm.rank; if (nranks) *nranks = ctx->comm.nranks;
    if (grid_rows) *grid_rows = ctx->comm.grid_rows; if (grid_cols) *grid_cols = ctx->comm.grid_cols;
    int64_t o, l;
    const int64_t Nt = ctx->comm.nranks > 1 ? (int64_t)ctx->N_total : (int64_t)ctx->n;
    if (ctx->comm.nranks > 1) { block_extent(Nt, ctx->comm.grid_rows, ctx->comm.rank / ctx->comm.grid_cols, o, l); o += ctx->read_base0; } else { o = ctx->read_id_offset; l = ctx->n; }
    if (row0) *row0 = o; if (nrows) *nrows = l;
    if (ctx->comm.nranks > 1) { block_extent(Nt, ctx->comm.grid_cols, ctx->comm.rank % ctx->comm.grid_cols, o, l); o += ctx->read_base0; } else { o = ctx->read_id_offset; l = ctx->n; }
    if (col0) *col0 = o; if (ncols) *ncols = l;
    return 0;
}

void elba_fe_block_extent(int64_t n, int parts, int idx, int64_t *offset, int64_t *length)
{
    int64_t o = 0, l = 0;
    if (parts > 0 && idx >= 0 && idx < parts) block_extent(n, parts, idx, o, l);
    if (offset) *offset = o; if (length) *length = l;
}

int elba_fe_sizes_global(elba_fe_ctx *ctx, elba_fe_sizes_t *out)
{
    if (!ctx || !out) return ELBA_FE_ERR_INVALID;
    CK(cudaStreamSynchronize(ctx->stream));
    *out = ctx->sz;
    if (ctx->comm.nranks == 1) return 0;
    // sums over the GPUs; reliable / partitions / table_slots are global already
    u64 v[10] = { ctx->sz.nreads, ctx->sz.num_kmers, ctx->sz.distinct, ctx->sz.nnzA_pre, ctx->sz.nnzA, ctx->sz.products, ctx->sz.nnzB_pre, ctx->sz.nnzB,
                  ctx->sz.candidates, ctx->sz.overflow_instances };
    int rc = allreduce_u64(ctx, v, 10, ncclSum);
    if (rc) return rc;
    out->nreads = v[0]; out->num_kmers = v[1]; out->distinct = v[2]; out->nnzA_pre = v[3]; out->nnzA = v[4]; out->products = v[5];
    out->nnzB_pre = v[6]; out->nnzB = v[7]; out->candidates = v[8]; out->overflow_instances = v[9];
    return 0;
}

// ---- result digests (digest.cuh): global values, identical for any number of GPUs -------------------------------
int elba_fe_digests(elba_fe_ctx *ctx, uint64_t out[4])
{
    if (!ctx || !out) return ELBA_FE_ERR_INVALID;
    if (ctx->phase < 2) return fail(ctx, ELBA_FE_ERR_STATE, "elba_fe_digests: call elba_fe_count first");
    CK(cudaSetDevice(ctx->cfg.device));
    cudaStream_t st = ctx->stream;
    CK(ctx->tmp64.ensure(8 * 64));
    u64 *d = ctx->tmp64.as<u64>() + 8;              // [8..11]: the four sums ([0..7] is the scratch of allreduce_u64)
    CK(cudaMemsetAsync(d, 0, 32, st));
    const u64 R = ctx->sz.reliable;
    // the reliable list: every GPU's own share (super-k-mer path on several GPUs), else replicated: one rank contributes it
    if (ctx->kmers_distributed) { if (ctx->R_local) { k_digest_kmers<<<grid_for(ctx, 4), 256, 0, st>>>(ctx->rel_key_s.as<u64>(), ctx->rel_cnt_s.as<u32>(), ctx->R_local, d); CKL(); LAUNCHED(ctx); } }
    else if (R && ctx->comm.rank == 0) { k_digest_kmers<<<grid_for(ctx, 4), 256, 0, st>>>(ctx->rel_key_s.as<u64>(), ctx->rel_cnt_s.as<u32>(), R, d); CKL(); LAUNCHED(ctx); }
    if (ctx->phase >= 3 && ctx->n) { k_digest_A<<<grid_for(ctx, 4), 256, 0, st>>>(ctx->a_rowptr.as<int64_t>(), ctx->a_col.as<u32>(), ctx->a_pos.as<u32>(), ctx->n, (u64)ctx->read_id_offset, d + 1); CKL(); LAUNCHED(ctx); }
    if (ctx->phase >= 4 && ctx->b_rows) { k_digest_B<<<grid_for(ctx, 4), 256, 0, st>>>(ctx->b_rowptr.as<int64_t>(), ctx->b_col.as<u32>(), ctx->b_num.as<int32_t>(), ctx->b_seeds.as<u32>(), ctx->b_rows,
                                                (u64)ctx->op.row0, (u64)ctx->op.col0, d + 2, d + 3); CKL(); LAUNCHED(ctx); }
    u64 h[4];
    CK(cudaMemcpyAsync(h, d, 32, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    int rc = allreduce_u64(ctx, h, 4, ncclSum);
    if (rc) return rc;
    for (int i = 0; i < 4; ++i) out[i] = h[i];
    return 0;
}

// ---- results ---------------------------------------------------------------------------------------
#define D2H(dst, src, bytes) do { if ((bytes) && (dst)) CK(cudaMemcpyAsync((dst), (src), (bytes), cudaMemcpyDeviceToHost, ctx->stream)); } while (0)

int elba_fe_get_kmers(elba_fe_ctx *ctx, uint64_t *kmer, uint32_t *count)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (ctx->phase < 2) return fail(ctx, ELBA_FE_ERR_STATE, "no counts yet");
    u64 R = ctx->sz.reliable;
    if (ctx->kmers_distributed)
    {
        // several GPUs, super-k-mer path: every GPU holds the k-mers it owns (sorted) with their global column ids; the whole
        // list is assembled on request (COLLECTIVE): all-gather of the counts and ids, then every entry goes to its rank
        const int W = ctx->comm.nranks; cudaStream_t st = ctx->stream; int rc;
        CK(ctx->glob_key.ensure(8 * std::max<u64>(R, 1))); CK(ctx->glob_cnt.ensure(4 * std::max<u64>(R, 1)));
        CK(ctx->glob_gid.ensure(4 * std::max<u64>(R, 1))); CK(ctx->glob_cnt_in.ensure(4 * std::max<u64>(R, 1)));
        if ((rc = allgatherv(ctx, ctx->rel_gid.p, ctx->glob_gid.p, ctx->rel_counts, 4))) return rc;
        if ((rc = allgatherv(ctx, ctx->rel_cnt_s.p, ctx->glob_cnt_in.p, ctx->rel_counts, 4))) return rc;
        (void)W;
        if (R) { k_place_by_id<<<nblk(R, 256), 256, 0, st>>>(ctx->rel_all_key.as<u64>(), ctx->glob_cnt_in.as<u32>(), ctx->glob_gid.as<u32>(), R, ctx->glob_key.as<u64>(), ctx->glob_cnt.as<u32>()); CKL(); LAUNCHED(ctx); }
        D2H(kmer, ctx->glob_key.p, 8 * R); D2H(count, ctx->glob_cnt.p, 4 * R);
        CK(cudaStreamSynchronize(st));
        return 0;
    }
    D2H(kmer, ctx->rel_key_s.p, 8 * R); D2H(count, ctx->rel_cnt_s.p, 4 * R);
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int elba_fe_get_A(elba_fe_ctx *ctx, int64_t *rowptr, uint32_t *col, uint32_t *pos)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (ctx->phase < 3) return fail(ctx, ELBA_FE_ERR_STATE, "A not built");
    D2H(rowptr, ctx->a_rowptr.p, 8 * ((size_t)ctx->n + 1)); D2H(col, ctx->a_col.p, 4 * ctx->sz.nnzA); D2H(pos, ctx->a_pos.p, 4 * ctx->sz.nnzA);
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int elba_fe_get_AT(elba_fe_ctx *ctx, int64_t *colptr, uint32_t *row, uint32_t *pos)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (ctx->phase < 3) return fail(ctx, ELBA_FE_ERR_STATE, "A not built");
    if (!ctx->at_built)
    {
        // the API's form of the transpose (64-bit column pointers, rows and positions apart), made on request
        const u64 R = ctx->sz.reliable, na = std::max<u64>(ctx->sz.nnzA, 1);
        CK(ctx->at_colptr.ensure(8 * (R + 2))); CK(ctx->at_row.ensure(4 * na)); CK(ctx->at_pos.ensure(4 * na));
        const u32 *cptr = ctx->sp_ptr.as<u32>(); const uint2 *ent = ctx->sp_ent.as<uint2>();
        if (ctx->comm.nranks > 1)
        {
            // several GPUs: sp_ptr / sp_ent hold the gathered right operand; transpose the own rows into the left-operand scratch
            CK(ctx->at_ptr32.ensure(4 * (R + 2))); CK(ctx->at_ent.ensure(8 * na));
            int rc = build_local_transpose(ctx, ctx->at_ptr32.as<u32>(), ctx->at_ent.as<uint2>()); if (rc) return rc;
            cptr = ctx->at_ptr32.as<u32>(); ent = ctx->at_ent.as<uint2>();
        }
        k_transpose_api<<<nblk(std::max<u64>(R + 1, ctx->sz.nnzA), 256), 256, 0, ctx->stream>>>(cptr, ent, R, ctx->sz.nnzA, ctx->at_colptr.as<int64_t>(), ctx->at_row.as<u32>(), ctx->at_pos.as<u32>());
        CKL(); LAUNCHED(ctx);
        ctx->at_built = true;
    }
    D2H(colptr, ctx->at_colptr.p, 8 * (ctx->sz.reliable + 1)); D2H(row, ctx->at_row.p, 4 * ctx->sz.nnzA); D2H(pos, ctx->at_pos.p, 4 * ctx->sz.nnzA);
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int elba_fe_get_B(elba_fe_ctx *ctx, int64_t *rowptr, uint32_t *col, int32_t *numshared, uint32_t *seeds)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (ctx->phase < 4) return fail(ctx, ELBA_FE_ERR_STATE, "B not built");
    cudaEvent_t a = ctx->ev[0], b = ctx->ev[1];
    CK(cudaEventRecord(a, ctx->stream));
    D2H(rowptr, ctx->b_rowptr.p, 8 * ((size_t)ctx->b_rows + 1)); D2H(col, ctx->b_col.p, 4 * ctx->sz.nnzB);
    D2H(numshared, ctx->b_num.p, 4 * ctx->sz.nnzB); D2H(seeds, ctx->b_seeds.p, 16 * ctx->sz.nnzB);
    CK(cudaEventRecord(b, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    float ms = 0; cudaEventElapsedTime(&ms, a, b); ctx->tm.download_ms = ms;
    return 0;
}

int elba_fe_get_B_triples(elba_fe_ctx *ctx, int64_t *row, int64_t *col, int32_t *numshared, uint32_t *seeds)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (ctx->phase < 4) return fail(ctx, ELBA_FE_ERR_STATE, "B not built");
    u64 nnz = ctx->sz.nnzB; u32 N = ctx->b_rows;
    std::vector<int64_t> rp((size_t)N + 1); std::vector<u32> c32(nnz);
    int rc = elba_fe_get_B(ctx, rp.data(), c32.data(), numshared, seeds);
    if (rc) return rc;
    // global ids: this GPU's block starts at (row0, col0); on one GPU both are the caller's read offset
    for (u32 r = 0; r < N; ++r) for (int64_t p = rp[r]; p < rp[r + 1]; ++p) { if (row) row[p] = (int64_t)r + ctx->op.row0; if (col) col[p] = (int64_t)c32[p] + ctx->op.col0; }
    return 0;
}

int elba_fe_device_B(elba_fe_ctx *ctx, const int64_t **rowptr, const uint32_t **col, const int32_t **numshared, const uint32_t **seeds)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (ctx->phase < 4) return fail(ctx, ELBA_FE_ERR_STATE, "B not built");
    if (rowptr) *rowptr = ctx->b_rowptr.as<int64_t>(); if (col) *col = ctx->b_col.as<u32>();
    if (numshared) *numshared = ctx->b_num.as<int32_t>(); if (seeds) *seeds = ctx->b_seeds.as<u32>();
    return 0;
}

int elba_fe_device_A(elba_fe_ctx *ctx, const int64_t **rowptr, const uint32_t **col, const uint32_t **pos)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (ctx->phase < 3) return fail(ctx, ELBA_FE_ERR_STATE, "A not built");
    if (rowptr) *rowptr = ctx->a_rowptr.as<int64_t>(); if (col) *col = ctx->a_col.as<u32>(); if (pos) *pos = ctx->a_pos.as<u32>();
    return 0;
}

// ---- B by column, doubly compressed (dcsc.cuh): the layout the reference's consumer walks (src/PairwiseAlignment.cpp:16-56) ----
int elba_fe_B_dcsc(elba_fe_ctx *ctx, uint64_t *nzc)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (ctx->phase < 4) return fail(ctx, ELBA_FE_ERR_STATE, "B not built");
    CK(cudaSetDevice(ctx->cfg.device));
    cudaStream_t st = ctx->stream;
    const u64 nnz = ctx->sz.nnzB; const u32 N = ctx->b_rows;
    if (nnz >= 0xFFFFFFF0ull) return fail(ctx, ELBA_FE_ERR_INVALID, "B block with more than 2^32 nonzeros");
    if (!ctx->dc_built)
    {
        int rc;
        CK(ctx->dc_key.ensure(4 * (nnz + 1))); CK(ctx->dc_key2.ensure(4 * (nnz + 1))); CK(ctx->dc_val.ensure(8 * (nnz + 1))); CK(ctx->dc_val2.ensure(8 * (nnz + 1)));
        CK(ctx->dc_head.ensure(8 * (nnz + 1)));
        CK(ctx->dc_ir.ensure(8 * (nnz + 1))); CK(ctx->dc_num.ensure(4 * (nnz + 1))); CK(ctx->dc_seeds.ensure(16 * (nnz + 1)));
        CK(ctx->dc_jc.ensure(8 * (nnz + 1))); CK(ctx->dc_cp.ensure(8 * (nnz + 2)));
        u64 h_nzc = 0;
        if (nnz)
        {
            // the widest column id of the block decides the sorted bits
            int64_t ncols = (int64_t)N;
            if (ctx->comm.nranks > 1) { int64_t o, l; elba_fe_block_extent((int64_t)ctx->N_total, ctx->comm.grid_cols, ctx->comm.rank % ctx->comm.grid_cols, &o, &l); ncols = l; }
            k_dcsc_keys<<<nblk(nnz, 256), 256, 0, st>>>(ctx->b_rowptr.as<int64_t>(), ctx->b_col.as<u32>(), N, nnz, ctx->dc_key.as<u32>(), ctx->dc_val.as<u64>()); CKL(); LAUNCHED(ctx);
            if ((rc = sort_pairs_u32_u64(ctx, ctx->dc_key.as<u32>(), ctx->dc_key2.as<u32>(), ctx->dc_val.as<u64>(), ctx->dc_val2.as<u64>(), nnz, 0, bits_for((u64)std::max<int64_t>(ncols, 2))))) return rc;
            k_dcsc_heads<<<nblk(nnz + 1, 256), 256, 0, st>>>(ctx->dc_key2.as<u32>(), nnz, ctx->dc_head.as<u64>()); CKL(); LAUNCHED(ctx);
            if ((rc = exclusive_scan_inplace(ctx, ctx->dc_head.as<u64>(), nnz + 1))) return rc;
            k_dcsc_write<<<nblk(nnz + 1, 256), 256, 0, st>>>(ctx->dc_key2.as<u32>(), ctx->dc_val2.as<u64>(), ctx->dc_head.as<u64>(), nnz, ctx->b_num.as<int32_t>(),
                ctx->b_seeds.as<uint4>(), ctx->dc_jc.as<int64_t>(), ctx->dc_cp.as<int64_t>(), ctx->dc_ir.as<int64_t>(), ctx->dc_num.as<int32_t>(), ctx->dc_seeds.as<uint4>()); CKL(); LAUNCHED(ctx);
            CK(cudaMemcpyAsync(&h_nzc, ctx->dc_head.as<u64>() + nnz, 8, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
        }
        else CK(cudaMemsetAsync(ctx->dc_cp.p, 0, 8, st));
        ctx->dc_nzc = h_nzc; ctx->dc_built = true;
    }
    if (nzc) *nzc = ctx->dc_nzc;
    return 0;
}

int elba_fe_get_B_dcsc(elba_fe_ctx *ctx, int64_t *jc, int64_t *cp, int64_t *ir, int32_t *numshared, uint32_t *seeds)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    int rc = elba_fe_B_dcsc(ctx, nullptr);
    if (rc) return rc;
    cudaEvent_t a = ctx->ev[0], b = ctx->ev[1];
    CK(cudaEventRecord(a, ctx->stream));
    D2H(jc, ctx->dc_jc.p, 8 * ctx->dc_nzc); D2H(cp, ctx->dc_cp.p, 8 * (ctx->dc_nzc + 1)); D2H(ir, ctx->dc_ir.p, 8 * ctx->sz.nnzB);
    D2H(numshared, ctx->dc_num.p, 4 * ctx->sz.nnzB); D2H(seeds, ctx->dc_seeds.p, 16 * ctx->sz.nnzB);
    CK(cudaEventRecord(b, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    float ms = 0; cudaEventElapsedTime(&ms, a, b); ctx->tm.download_ms = ms;
    return 0;
}

int elba_fe_device_B_dcsc(elba_fe_ctx *ctx, const int64_t **jc, const int64_t **cp, const int64_t **ir, const int32_t **numshared, const uint32_t **seeds)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    int rc = elba_fe_B_dcsc(ctx, nullptr);
    if (rc) return rc;
    if (jc) *jc = ctx->dc_jc.as<int64_t>(); if (cp) *cp = ctx->dc_cp.as<int64_t>(); if (ir) *ir = ctx->dc_ir.as<int64_t>();
    if (numshared) *numshared = ctx->dc_num.as<int32_t>(); if (seeds) *seeds = ctx->dc_seeds.as<u32>();
    return 0;
}

// ---- the consumer of B: X-drop alignment of its nonzeros (xdrop.cuh) ----------------------------------------
int elba_fe_align(elba_fe_ctx *ctx, int mat, int mis, int gap, int dropoff, uint64_t *npairs)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (ctx->phase < 4) return fail(ctx, ELBA_FE_ERR_STATE, "elba_fe_align: call elba_fe_spgemm first");
    if (mat <= 0 || mis > 0 || gap >= 0 || dropoff < 0) return fail(ctx, ELBA_FE_ERR_INVALID, "elba_fe_align: need mat > 0, mis <= 0, gap < 0, dropoff >= 0");
    ctx->og_aligned = ctx->og_done = ctx->ct_done = ctx->pf_done = false;
    CK(cudaSetDevice(ctx->cfg.device));
    cudaStream_t st = ctx->stream;
    const u64 nnz = ctx->sz.nnzB; const u32 N = ctx->b_rows;
    ctx->xd_done = false;
    { int rcw = wait_reads(ctx); if (rcw) return rcw; }
    CK(cudaEventRecord(ctx->xd_e0, st));
    CK(ctx->xd_flag.ensure(8 * (nnz + 2))); CK(ctx->xd_rowof.ensure(4 * (nnz + 1))); CK(ctx->xd_max.ensure(64));
    int rc;
    // the reads the pairs of this block name: one GPU: its own.  Several GPUs: block (i, j) needs the reads of R_i and C_j, which
    // other ranks hold (the reference exchanges them in DistributedFastaData, src/DistributedFastaData.cpp:98-232): the arenas
    // and read tables of all ranks are all-gathered over NVLink (0.25 B per base) and indexed by global read id.
    const int W = ctx->comm.nranks;
    const uint8_t *x_buf = ctx->packed.as<uint8_t>(); const u64 *x_off = ctx->off.as<u64>(); const u32 *x_len = ctx->len32.as<u32>();
    u64 x_n = ctx->n; u32 row_base = 0, col_base = 0;
    if (W > 1)
    {
        std::vector<u64> nb, nr, ro;
        if ((rc = allgather_u64(ctx, ctx->packed_bytes, nb))) return rc;
        if ((rc = allgather_u64(ctx, (u64)ctx->n, nr))) return rc;
        if ((rc = allgather_u64(ctx, (u64)ctx->read_id_offset, ro))) return rc;
        u64 Nt = 0, Bt = 0;
        for (int r = 0; r < W; ++r)
        {
            if (ro[r] != ro[0] + Nt) return fail(ctx, ELBA_FE_ERR_INVALID, "elba_fe_align: the ranks must hold consecutive blocks of reads in rank order");
            Nt += nr[r]; Bt += nb[r];
        }
        if (Nt >= 0xFFFFFFF0ull) return fail(ctx, ELBA_FE_ERR_INVALID, "elba_fe_align: too many reads");
        CK(ctx->xa_buf.ensure(Bt + 64)); CK(ctx->xa_off.ensure(8 * (Nt + 1))); CK(ctx->xa_len.ensure(4 * (Nt + 1)));
        if ((rc = allgatherv(ctx, ctx->packed.p, ctx->xa_buf.p, nb, 1))) return rc;
        if ((rc = allgatherv(ctx, ctx->off.p, ctx->xa_off.p, nr, 8))) return rc;
        if ((rc = allgatherv(ctx, ctx->len32.p, ctx->xa_len.p, nr, 4))) return rc;
        CK(cudaMemsetAsync(ctx->xa_buf.as<uint8_t>() + Bt, 0, 64, st));
        u64 r0 = 0, b0 = 0;
        for (int r = 0; r < W; ++r)
        {
            // rank r's offsets count from its own arena: move them behind the arenas of the ranks before it
            if (nr[r] && b0) { k_add_u64<<<nblk(nr[r], 256), 256, 0, st>>>(ctx->xa_off.as<u64>() + r0, nr[r], b0); CKL(); LAUNCHED(ctx); }
            r0 += nr[r]; b0 += nb[r];
        }
        x_buf = ctx->xa_buf.as<uint8_t>(); x_off = ctx->xa_off.as<u64>(); x_len = ctx->xa_len.as<u32>(); x_n = Nt;
        row_base = (u32)((u64)ctx->op.row0 - ro[0]); col_base = (u32)((u64)ctx->op.col0 - ro[0]);
        ctx->panel_bytes += Bt + 12 * Nt - ctx->packed_bytes - 12 * (u64)ctx->n;
    }
    const int global_rule = ctx->comm.grid_rows != ctx->comm.grid_cols;
    k_xdrop_select<<<nblk(nnz + 1, 256), 256, 0, st>>>(ctx->b_rowptr.as<int64_t>(), ctx->b_col.as<u32>(), N, nnz, ctx->op.row0, ctx->op.col0,
        global_rule, ctx->xd_flag.as<u64>(), ctx->xd_rowof.as<u32>());
    CKL(); LAUNCHED(ctx);
    rc = exclusive_scan_inplace(ctx, ctx->xd_flag.as<u64>(), nnz + 1);
    if (rc) return rc;
    CK(cudaMemsetAsync(ctx->xd_max.p, 0, 64, st));
    if (x_n) { k_max_u32<<<grid_for(ctx, 2), 256, 0, st>>>(x_len, x_n, ctx->xd_max.as<u32>()); CKL(); LAUNCHED(ctx); }
    u64 np = 0; u32 maxlen = 0;
    CK(cudaMemcpyAsync(&np, ctx->xd_flag.as<u64>() + nnz, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&maxlen, ctx->xd_max.p, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    const u64 n1 = std::max<u64>(np, 1);
    CK(ctx->xd_prow.ensure(4 * n1)); CK(ctx->xd_pcol.ensure(4 * n1)); CK(ctx->xd_sq.ensure(4 * n1)); CK(ctx->xd_st.ensure(4 * n1)); CK(ctx->xd_nz.ensure(8 * n1));
    CK(ctx->xd_out.ensure(4 * XD_FIELDS * n1));
    if (nnz) { k_xdrop_pairs<<<nblk(nnz, 256), 256, 0, st>>>(ctx->xd_flag.as<u64>(), ctx->xd_rowof.as<u32>(), ctx->b_col.as<u32>(), ctx->b_seeds.as<u32>(), nnz,
                   ctx->xd_prow.as<u32>(), ctx->xd_pcol.as<u32>(), ctx->xd_sq.as<u32>(), ctx->xd_st.as<u32>(), ctx->xd_nz.as<u64>()); CKL(); LAUNCHED(ctx); }
    if (np)
    {
        const u32 warps_per_cta = 4;
        const u32 grid = (u32)std::min<u64>((np + warps_per_cta - 1) / warps_per_cta, (u64)grid_for(ctx, 8));
        XdropArgs A;
        A.buf = x_buf; A.off = x_off; A.len = x_len; A.row_base = row_base; A.col_base = col_base;
        A.k = ctx->cfg.k; A.mat = mat; A.mis = mis; A.gap = gap; A.drop = dropoff;
        A.prow = ctx->xd_prow.as<u32>(); A.pcol = ctx->xd_pcol.as<u32>(); A.sq = ctx->xd_sq.as<u32>(); A.st = ctx->xd_st.as<u32>(); A.npairs = np;
        A.stride = (u64)maxlen + 4;
        CK(ctx->xd_scratch.ensure(sizeof(int) * 3 * A.stride * (u64)grid * warps_per_cta));
        A.scratch = ctx->xd_scratch.as<int>(); A.out = ctx->xd_out.as<int32_t>();
        k_xdrop<<<grid, 32 * warps_per_cta, 0, st>>>(A); CKL(); LAUNCHED(ctx);
    }
    CK(cudaEventRecord(ctx->xd_e1, st));
    CK(cudaStreamSynchronize(st));
    float ms = 0; if (cudaEventElapsedTime(&ms, ctx->xd_e0, ctx->xd_e1) == cudaSuccess) ctx->tm.align_ms = ms;
    ctx->xd_pairs = np; ctx->xd_done = true; ctx->og_aligned = true; ctx->xd_read_gen = ctx->read_gen;
    if (npairs) *npairs = np;
    return 0;
}

static __global__ void k_xdrop_ids(const u32 *__restrict__ prow, const u32 *__restrict__ pcol, u64 n, int64_t row0, int64_t col0, int64_t *__restrict__ row, int64_t *__restrict__ col)
{
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { row[i] = row0 + prow[i]; col[i] = col0 + pcol[i]; }
}

int elba_fe_get_alignments(elba_fe_ctx *ctx, int64_t *row, int64_t *col, int32_t *fields)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (!ctx->xd_done || ctx->phase < 4) return fail(ctx, ELBA_FE_ERR_STATE, "elba_fe_get_alignments: call elba_fe_align first");
    const u64 np = ctx->xd_pairs;
    if (!np) return 0;
    DevBuf tmp;
    CK(tmp.ensure(16 * np));
    k_xdrop_ids<<<nblk(np, 256), 256, 0, ctx->stream>>>(ctx->xd_prow.as<u32>(), ctx->xd_pcol.as<u32>(), np, ctx->op.row0, ctx->op.col0, tmp.as<int64_t>(), tmp.as<int64_t>() + np);
    LAUNCHED(ctx);
    D2H(row, tmp.p, 8 * np); D2H(col, tmp.as<int64_t>() + np, 8 * np); D2H(fields, ctx->xd_out.p, 4 * (size_t)XD_FIELDS * np);
    CK(cudaStreamSynchronize(ctx->stream));
    tmp.release();
    return 0;
}

// ---- transitive reduction of the overlap graph (transitive.cuh): TransitiveReduction(R), src/TransitiveReduction.cpp:3-92 ----
// The kernel chain on nnz device-resident triples with read ids in [0, n); id_base is added to the string graph's rows and
// columns.  The caller has recorded ev[0] on the stream; this ends with ev[1], a stream synchronise and tr_done set.
static int tr_reduce_device(elba_fe_ctx *ctx, const int64_t *row, const int64_t *col, const int32_t *fields, u64 nnz, u32 n, int32_t fuzz,
                            int64_t id_base, uint64_t *nnz_out)
{
    cudaStream_t st = ctx->stream;
    const u64 m2 = 2 * nnz;
    int rc;
    u64 M = 0;
    if (nnz)
    {
        CK(ctx->tr_key.ensure(8 * m2)); CK(ctx->tr_key2.ensure(8 * m2)); CK(ctx->tr_val.ensure(4 * m2)); CK(ctx->tr_val2.ensure(4 * m2)); CK(ctx->tr_head.ensure(8 * (m2 + 1)));
        k_tr_items<<<nblk(nnz, 256), 256, 0, st>>>(row, col, nnz, ctx->tr_key.as<u64>(), ctx->tr_val.as<u32>()); CKL(); LAUNCHED(ctx);
        if ((rc = sort_pairs(ctx, ctx->tr_key.as<u64>(), ctx->tr_key2.as<u64>(), ctx->tr_val.as<u32>(), ctx->tr_val2.as<u32>(), m2, 0, 32 + bits_for(std::max<u64>(n, 2))))) return rc;
        k_tr_heads<<<nblk(m2 + 1, 256), 256, 0, st>>>(ctx->tr_key2.as<u64>(), m2, ctx->tr_head.as<u64>()); CKL(); LAUNCHED(ctx);
        if ((rc = exclusive_scan_inplace(ctx, ctx->tr_head.as<u64>(), m2 + 1))) return rc;
        CK(cudaMemcpyAsync(&M, ctx->tr_head.as<u64>() + m2, 8, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    }
    if (M)
    {
        CK(ctx->tr_okey.ensure(8 * M)); CK(ctx->tr_row.ensure(4 * M)); CK(ctx->tr_col.ensure(4 * M)); CK(ctx->tr_dir.ensure(4 * M)); CK(ctx->tr_dirT.ensure(4 * M));
        CK(ctx->tr_suf.ensure(4 * M)); CK(ctx->tr_sufT.ensure(4 * M)); CK(ctx->tr_src.ensure(4 * M)); CK(ctx->tr_tr.ensure(M)); CK(ctx->tr_rowptr.ensure(8 * ((u64)n + 2)));
        CK(ctx->tr_I.ensure(M)); CK(ctx->tr_T.ensure(M)); CK(ctx->tr_keep.ensure(8 * (M + 1)));
        k_tr_entries<<<nblk(m2, 256), 256, 0, st>>>(ctx->tr_key2.as<u64>(), ctx->tr_val2.as<u32>(), ctx->tr_head.as<u64>(), m2, nnz, fields,
            ctx->tr_okey.as<u64>(), ctx->tr_row.as<u32>(), ctx->tr_col.as<u32>(), ctx->tr_dir.as<int32_t>(), ctx->tr_dirT.as<int32_t>(), ctx->tr_suf.as<int32_t>(), ctx->tr_sufT.as<int32_t>(),
            ctx->tr_src.as<u32>(), ctx->tr_tr.as<uint8_t>()); CKL(); LAUNCHED(ctx);
        k_segment_ptr<<<nblk((u64)n + 1, 256), 256, 0, st>>>(ctx->tr_okey.as<u64>(), M, n, 32, ctx->tr_rowptr.as<int64_t>()); CKL(); LAUNCHED(ctx);
        TrGraph g; g.rowptr = ctx->tr_rowptr.as<int64_t>(); g.row = ctx->tr_row.as<u32>(); g.col = ctx->tr_col.as<u32>(); g.dir = ctx->tr_dir.as<int32_t>(); g.dirT = ctx->tr_dirT.as<int32_t>();
        g.suf = ctx->tr_suf.as<int32_t>(); g.sufT = ctx->tr_sufT.as<int32_t>(); g.m = M; g.n = n;
        CK(cudaMemsetAsync(ctx->tr_T.p, 0, M, st));
        k_tr_mark<<<nblk(M, 128), 128, 0, st>>>(g, fuzz, ctx->tr_I.as<uint8_t>()); CKL(); LAUNCHED(ctx);
        k_tr_symmetric<<<nblk(M, 256), 256, 0, st>>>(g, ctx->tr_I.as<uint8_t>(), ctx->tr_T.as<uint8_t>()); CKL(); LAUNCHED(ctx);
        k_tr_keep<<<nblk(M + 1, 256), 256, 0, st>>>(g, ctx->tr_T.as<uint8_t>(), ctx->tr_keep.as<u64>()); CKL(); LAUNCHED(ctx);
        if ((rc = exclusive_scan_inplace(ctx, ctx->tr_keep.as<u64>(), M + 1))) return rc;
        u64 S = 0;
        CK(cudaMemcpyAsync(&S, ctx->tr_keep.as<u64>() + M, 8, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        const u64 S1 = std::max<u64>(S, 1);
        CK(ctx->tr_orow.ensure(8 * S1)); CK(ctx->tr_ocol.ensure(8 * S1)); CK(ctx->tr_of.ensure(16 * S1)); CK(ctx->tr_osrc.ensure(8 * S1)); CK(ctx->tr_otr.ensure(S1));
        k_tr_output<<<nblk(M, 256), 256, 0, st>>>(g, ctx->tr_T.as<uint8_t>(), ctx->tr_keep.as<u64>(), ctx->tr_src.as<u32>(), ctx->tr_tr.as<uint8_t>(),
            ctx->tr_orow.as<int64_t>(), ctx->tr_ocol.as<int64_t>(), ctx->tr_of.as<int32_t>(), ctx->tr_osrc.as<u64>(), ctx->tr_otr.as<uint8_t>()); CKL(); LAUNCHED(ctx);
        if (id_base && S)
        {
            k_add_u64<<<nblk(S, 256), 256, 0, st>>>(ctx->tr_orow.as<u64>(), S, (u64)id_base); CKL(); LAUNCHED(ctx);
            k_add_u64<<<nblk(S, 256), 256, 0, st>>>(ctx->tr_ocol.as<u64>(), S, (u64)id_base); CKL(); LAUNCHED(ctx);
        }
        ctx->tr_out = S;
    }
    CK(cudaEventRecord(ctx->ev[1], st));
    CK(cudaStreamSynchronize(st));
    float ms = 0; if (cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]) == cudaSuccess) ctx->tm.transitive_ms = ms;
    ctx->tr_done = true;
    if (nnz_out) *nnz_out = ctx->tr_out;
    return 0;
}

int elba_fe_transitive_reduction(elba_fe_ctx *ctx, const int64_t *row, const int64_t *col, const int32_t *fields, uint64_t nnz, int64_t nreads,
                                 int32_t fuzz, uint64_t *nnz_out)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (nreads < 0 || nreads >= 0xFFFFFFF0ll) return fail(ctx, ELBA_FE_ERR_INVALID, "elba_fe_transitive_reduction: bad number of reads");
    if (nnz >= (1ull << 31)) return fail(ctx, ELBA_FE_ERR_INVALID, "elba_fe_transitive_reduction: more than 2^31 overlaps");
    if (nnz && (!row || !col || !fields)) return fail(ctx, ELBA_FE_ERR_INVALID, "elba_fe_transitive_reduction: null triples");
    for (u64 e = 0; e < nnz; ++e)
    {
        if (row[e] < 0 || row[e] >= nreads || col[e] < 0 || col[e] >= nreads) return fail(ctx, ELBA_FE_ERR_INVALID, "elba_fe_transitive_reduction: read id out of range");
        if (fields[4 * e] < -1 || fields[4 * e] > 3 || fields[4 * e + 1] < -1 || fields[4 * e + 1] > 3)
            return fail(ctx, ELBA_FE_ERR_INVALID, "elba_fe_transitive_reduction: direction outside -1..3 (include/Overlap.hpp:36-44)");
    }
    CK(cudaSetDevice(ctx->cfg.device));
    cudaStream_t st = ctx->stream;
    ctx->tr_done = ctx->tr_resident = ctx->ct_done = ctx->pf_done = false; ctx->tr_out = 0;
    CK(cudaEventRecord(ctx->ev[0], st));
    if (nnz)
    {
        CK(ctx->tr_in_row.ensure(8 * nnz)); CK(ctx->tr_in_col.ensure(8 * nnz)); CK(ctx->tr_in_f.ensure(16 * nnz));
        CK(cudaMemcpyAsync(ctx->tr_in_row.p, row, 8 * nnz, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(ctx->tr_in_col.p, col, 8 * nnz, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(ctx->tr_in_f.p, fields, 16 * nnz, cudaMemcpyHostToDevice, st));
    }
    return tr_reduce_device(ctx, ctx->tr_in_row.as<int64_t>(), ctx->tr_in_col.as<int64_t>(), ctx->tr_in_f.as<int32_t>(), nnz, (u32)nreads, fuzz, 0, nnz_out);
}

// ---- the overlap graph R from the resident alignments (overlap_graph.cuh): the prunes of src/main.cpp:300-313 ------------
int elba_fe_overlap_graph(elba_fe_ctx *ctx, uint64_t *nnz, uint64_t *ncontained)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (!ctx->og_aligned || !ctx->xd_done || ctx->phase < 4) return fail(ctx, ELBA_FE_ERR_STATE, "elba_fe_overlap_graph: call elba_fe_align first");
    CK(cudaSetDevice(ctx->cfg.device));
    cudaStream_t st = ctx->stream;
    ctx->og_done = ctx->tr_resident = ctx->ct_done = ctx->pf_done = false;
    const int W = ctx->comm.nranks;
    const u64 np = ctx->xd_pairs, Nt = W > 1 ? ctx->N_total : (u64)ctx->n;
    // job-relative id of this block's first row / column read (one GPU: 0)
    const u32 row_base = (u32)(ctx->op.row0 - ctx->read_base0), col_base = (u32)(ctx->op.col0 - ctx->read_base0);
    const u32 *prow = ctx->xd_prow.as<u32>(), *pcol = ctx->xd_pcol.as<u32>(); const int32_t *fields = ctx->xd_out.as<int32_t>();
    int rc;
    CK(cudaEventRecord(ctx->og_e0, st));
    // C over the alignments of every rank: local flags, then one max-all-reduce of the bytes
    CK(ctx->og_cont.ensure(std::max<u64>(Nt, 1))); CK(ctx->og_keep.ensure(8 * (np + 2)));      // np + 1 keep flags, |C| behind them
    if (Nt) CK(cudaMemsetAsync(ctx->og_cont.p, 0, Nt, st));
    if (np) { k_og_contained<<<nblk(np, 256), 256, 0, st>>>(prow, pcol, fields, np, row_base, col_base, ctx->og_cont.as<uint8_t>()); CKL(); LAUNCHED(ctx); }
    if (W > 1 && Nt) NC(ctx->comm.api->AllReduce(ctx->og_cont.p, ctx->og_cont.p, (size_t)Nt, ncclUint8, ncclMax, ctx->comm.comm, st));
    u64 *d_ncont = ctx->og_keep.as<u64>() + np + 1;
    CK(cudaMemsetAsync(d_ncont, 0, 8, st));
    if (Nt) { k_og_count<<<(u32)std::min<u64>(nblk(Nt, 256), (u64)grid_for(ctx, 4)), 256, 0, st>>>(ctx->og_cont.as<uint8_t>(), Nt, d_ncont); CKL(); LAUNCHED(ctx); }
    // keep flags -> positions -> this rank's part of R
    k_og_keep<<<nblk(np + 1, 256), 256, 0, st>>>(prow, pcol, fields, np, row_base, col_base, ctx->og_cont.as<uint8_t>(), ctx->og_keep.as<u64>()); CKL(); LAUNCHED(ctx);
    if ((rc = exclusive_scan_inplace(ctx, ctx->og_keep.as<u64>(), np + 1))) return rc;
    u64 h[2] = {0, 0};
    CK(cudaMemcpyAsync(&h[0], ctx->og_keep.as<u64>() + np, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&h[1], d_ncont, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    const u64 kept = h[0];
    DevBuf *dst[4] = { &ctx->og_row, &ctx->og_col, &ctx->og_f, &ctx->og_src };
    if (W > 1) { dst[0] = &ctx->og_lrow; dst[1] = &ctx->og_lcol; dst[2] = &ctx->og_lf; dst[3] = &ctx->og_lsrc; }
    const u64 k1 = std::max<u64>(kept, 1);
    CK(dst[0]->ensure(8 * k1)); CK(dst[1]->ensure(8 * k1)); CK(dst[2]->ensure(16 * k1)); CK(dst[3]->ensure(8 * k1));
    if (kept)
    {
        k_og_compact<<<nblk(np, 256), 256, 0, st>>>(prow, pcol, fields, np, row_base, col_base, ctx->og_keep.as<u64>(),
            dst[0]->as<int64_t>(), dst[1]->as<int64_t>(), dst[2]->as<int32_t>(), dst[3]->as<u64>()); CKL(); LAUNCHED(ctx);
    }
    // several GPUs: every rank gets the whole R, the ranks' parts in rank order
    u64 total = kept;
    if ((rc = allgather_u64(ctx, kept, ctx->og_counts))) return rc;
    if (W > 1)
    {
        total = 0; for (u64 c : ctx->og_counts) total += c;
        const u64 t1 = std::max<u64>(total, 1);
        CK(ctx->og_row.ensure(8 * t1)); CK(ctx->og_col.ensure(8 * t1)); CK(ctx->og_f.ensure(16 * t1)); CK(ctx->og_src.ensure(8 * t1));
        if ((rc = allgatherv(ctx, ctx->og_lrow.p, ctx->og_row.p, ctx->og_counts, 8))) return rc;
        if ((rc = allgatherv(ctx, ctx->og_lcol.p, ctx->og_col.p, ctx->og_counts, 8))) return rc;
        if ((rc = allgatherv(ctx, ctx->og_lf.p, ctx->og_f.p, ctx->og_counts, 16))) return rc;
        if ((rc = allgatherv(ctx, ctx->og_lsrc.p, ctx->og_src.p, ctx->og_counts, 8))) return rc;
    }
    CK(cudaEventRecord(ctx->og_e1, st));
    CK(cudaStreamSynchronize(st));
    float ms = 0; if (cudaEventElapsedTime(&ms, ctx->og_e0, ctx->og_e1) == cudaSuccess) ctx->tm.overlap_ms = ms;
    ctx->og_nnz = total; ctx->og_nreads = Nt; ctx->og_base = ctx->read_base0; ctx->og_done = true;
    if (nnz) *nnz = total;
    if (ncontained) *ncontained = h[1];
    return 0;
}

int elba_fe_get_overlap_graph(elba_fe_ctx *ctx, int64_t *row, int64_t *col, int32_t *fields, int32_t *src_rank, uint64_t *src_pair)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (!ctx->og_done) return fail(ctx, ELBA_FE_ERR_STATE, "elba_fe_get_overlap_graph: call elba_fe_overlap_graph first");
    CK(cudaSetDevice(ctx->cfg.device));
    const u64 m = ctx->og_nnz;
    if (!m) return 0;
    DevBuf tmp;
    if (row || col)
    {
        CK(tmp.ensure(16 * m));
        k_og_ids<<<nblk(m, 256), 256, 0, ctx->stream>>>(ctx->og_row.as<int64_t>(), ctx->og_col.as<int64_t>(), m, ctx->og_base, tmp.as<int64_t>(), tmp.as<int64_t>() + m);
        LAUNCHED(ctx);
    }
    D2H(row, tmp.p, 8 * m); D2H(col, tmp.as<int64_t>() + m, 8 * m); D2H(fields, ctx->og_f.p, 16 * m); D2H(src_pair, ctx->og_src.p, 8 * m);
    if (src_rank)
    {
        u64 o = 0;
        for (size_t r = 0; r < ctx->og_counts.size(); ++r) for (u64 i = 0; i < ctx->og_counts[r]; ++i) src_rank[o++] = (int32_t)r;
    }
    CK(cudaStreamSynchronize(ctx->stream));
    tmp.release();
    return 0;
}

int elba_fe_reduce_overlap_graph(elba_fe_ctx *ctx, int32_t fuzz, uint64_t *nnz_out)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (!ctx->og_done) return fail(ctx, ELBA_FE_ERR_STATE, "elba_fe_reduce_overlap_graph: call elba_fe_overlap_graph first");
    const u64 nnz = ctx->og_nnz, Nt = ctx->og_nreads;
    if (Nt >= 0xFFFFFFF0ull) return fail(ctx, ELBA_FE_ERR_INVALID, "elba_fe_reduce_overlap_graph: too many reads");
    if (nnz >= (1ull << 31)) return fail(ctx, ELBA_FE_ERR_INVALID, "elba_fe_reduce_overlap_graph: more than 2^31 overlaps");
    CK(cudaSetDevice(ctx->cfg.device));
    ctx->tr_done = ctx->ct_done = ctx->pf_done = false; ctx->tr_out = 0;
    CK(cudaEventRecord(ctx->ev[0], ctx->stream));
    const int rc = tr_reduce_device(ctx, ctx->og_row.as<int64_t>(), ctx->og_col.as<int64_t>(), ctx->og_f.as<int32_t>(), nnz, (u32)Nt, fuzz, ctx->og_base, nnz_out);
    if (rc == 0) ctx->tr_resident = true;
    return rc;
}

int elba_fe_get_string_graph(elba_fe_ctx *ctx, int64_t *row, int64_t *col, int32_t *fields, uint64_t *src, uint8_t *transposed)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (!ctx->tr_done) return fail(ctx, ELBA_FE_ERR_STATE, "elba_fe_get_string_graph: call elba_fe_transitive_reduction first");
    const u64 S = ctx->tr_out;
    D2H(row, ctx->tr_orow.p, 8 * S); D2H(col, ctx->tr_ocol.p, 8 * S); D2H(fields, ctx->tr_of.p, 16 * S); D2H(src, ctx->tr_osrc.p, 8 * S); D2H(transposed, ctx->tr_otr.p, S);
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

// ---- contigs from the string graph (contigs.cuh): the stage GenerateContigs runs in the reference (src/main.cpp:320) ------
// S: m entries row-major with global ids, base = global id of read 0 of the job, n reads in rd (job-relative ids).  Builds the
// whole layout on every rank (no collective) and the sequences of the contigs [block of rank / nranks].
static int contigs_device(elba_fe_ctx *ctx, const int64_t *row, const int64_t *col, const int32_t *f, u64 m, u32 n, int64_t base,
                          CtReads rd, int rank, int nranks, elba_fe_contig_info_t *info)
{
    cudaStream_t st = ctx->stream;
    int rc;
    const u64 n1 = (u64)n + 1, ns = 2ull * n;
    CK(cudaEventRecord(ctx->ct_e0, st));
    CK(ctx->ct_ptr.ensure(8 * n1)); CK(ctx->ct_branch.ensure(n1)); CK(ctx->ct_slot.ensure(4 * (ns + 2))); CK(ctx->ct_cyc.ensure(n1));
    for (int i = 0; i < 2; ++i) { CK(ctx->ct_succ[i].ensure(4 * (ns + 2))); CK(ctx->ct_dist[i].ensure(4 * (ns + 2))); CK(ctx->ct_mn[i].ensure(4 * (ns + 2))); }
    CK(ctx->ct_flag.ensure(8 * n1)); CK(ctx->ct_start.ensure(4 * n1)); CK(ctx->ct_pos.ensure(4 * n1)); CK(ctx->ct_next.ensure(n1)); CK(ctx->ct_L.ensure(4 * n1));
    CK(ctx->ct_cptr.ensure(8 * n1)); CK(ctx->ct_read.ensure(8 * n1)); CK(ctx->ct_rev.ensure(n1)); CK(ctx->ct_beg.ensure(4 * n1)); CK(ctx->ct_end.ensure(4 * n1));
    CK(ctx->ct_boff.ensure(8 * n1)); CK(ctx->tmp64.ensure(64));
    u64 *d_cnt = ctx->tmp64.as<u64>();                    // [0] branches, [1] cycles
    CK(cudaMemsetAsync(d_cnt, 0, 16, st));
    CK(cudaMemsetAsync(ctx->ct_cptr.p, 0, 8 * n1, st)); CK(cudaMemsetAsync(ctx->ct_boff.p, 0, 8 * n1, st));
    if (n)
    {
        const u32 gn = nblk(n, 256), gs = nblk(ns, 256);
        u32 *slot = ctx->ct_slot.as<u32>();
        k_ct_rowptr<<<nblk(n1, 256), 256, 0, st>>>(row, m, n, base, ctx->ct_ptr.as<u64>()); CKL(); LAUNCHED(ctx);
        k_ct_branch<<<gn, 256, 0, st>>>(ctx->ct_ptr.as<u64>(), f, n, ctx->ct_branch.as<uint8_t>()); CKL(); LAUNCHED(ctx);
        k_ct_slots<<<gn, 256, 0, st>>>(ctx->ct_ptr.as<u64>(), col, f, n, base, ctx->ct_branch.as<uint8_t>(), slot); CKL(); LAUNCHED(ctx);
        // list ranking: rounds doubles the hops every state has looked ahead; 2^rounds >= n covers the longest chain
        const int rounds = bits_for(std::max<u64>(n, 2));
        int cur = 0;
        k_ct_init<<<gs, 256, 0, st>>>(slot, col, n, base, ctx->ct_succ[0].as<u32>(), nullptr, ctx->ct_mn[0].as<u32>()); CKL(); LAUNCHED(ctx);
        for (int r = 0; r < rounds; ++r, cur ^= 1)
        {
            k_ct_jump<<<gs, 256, 0, st>>>(ns, ctx->ct_succ[cur].as<u32>(), nullptr, ctx->ct_mn[cur].as<u32>(), ctx->ct_succ[cur ^ 1].as<u32>(), nullptr, ctx->ct_mn[cur ^ 1].as<u32>());
            CKL(); LAUNCHED(ctx);
        }
        k_ct_cut<<<gn, 256, 0, st>>>(slot, col, base, ctx->ct_succ[cur].as<u32>(), ctx->ct_mn[cur].as<u32>(), n, ctx->ct_cyc.as<uint8_t>()); CKL(); LAUNCHED(ctx);
        cur = 0;
        k_ct_init<<<gs, 256, 0, st>>>(slot, col, n, base, ctx->ct_succ[0].as<u32>(), ctx->ct_dist[0].as<u32>(), nullptr); CKL(); LAUNCHED(ctx);
        for (int r = 0; r < rounds; ++r, cur ^= 1)
        {
            k_ct_jump<<<gs, 256, 0, st>>>(ns, ctx->ct_succ[cur].as<u32>(), ctx->ct_dist[cur].as<u32>(), nullptr, ctx->ct_succ[cur ^ 1].as<u32>(), ctx->ct_dist[cur ^ 1].as<u32>(), nullptr);
            CKL(); LAUNCHED(ctx);
        }
        k_ct_place<<<nblk(n1, 256), 256, 0, st>>>(ctx->ct_succ[cur].as<u32>(), ctx->ct_dist[cur].as<u32>(), n, ctx->ct_flag.as<u64>(), ctx->ct_start.as<u32>(),
            ctx->ct_pos.as<u32>(), ctx->ct_next.as<uint8_t>(), ctx->ct_L.as<u32>()); CKL(); LAUNCHED(ctx);
        if ((rc = exclusive_scan_inplace(ctx, ctx->ct_flag.as<u64>(), n1))) return rc;
        k_ct_clen<<<gn, 256, 0, st>>>(ctx->ct_flag.as<u64>(), ctx->ct_L.as<u32>(), n, ctx->ct_cptr.as<u64>()); CKL(); LAUNCHED(ctx);
        if ((rc = exclusive_scan_inplace(ctx, ctx->ct_cptr.as<u64>(), n1))) return rc;
        k_ct_layout<<<gn, 256, 0, st>>>(slot, col, f, base, n, ctx->ct_flag.as<u64>(), ctx->ct_cptr.as<u64>(), ctx->ct_start.as<u32>(), ctx->ct_pos.as<u32>(),
            ctx->ct_next.as<uint8_t>(), rd, ctx->ct_read.as<int64_t>(), ctx->ct_rev.as<uint8_t>(), ctx->ct_beg.as<u32>(), ctx->ct_end.as<u32>(), ctx->ct_boff.as<u64>());
        CKL(); LAUNCHED(ctx);
        if ((rc = exclusive_scan_inplace(ctx, ctx->ct_boff.as<u64>(), n1))) return rc;
        const u32 gc = (u32)std::min<u64>(gn, (u64)grid_for(ctx, 4));
        k_og_count<<<gc, 256, 0, st>>>(ctx->ct_branch.as<uint8_t>(), n, d_cnt); CKL(); LAUNCHED(ctx);
        k_og_count<<<gc, 256, 0, st>>>(ctx->ct_cyc.as<uint8_t>(), n, d_cnt + 1); CKL(); LAUNCHED(ctx);
    }
    // totals: contigs, reads in contigs, bases (the scans end at n: entries past the last contig / read are zero)
    u64 h[5] = {0, 0, 0, 0, 0};
    if (n) CK(cudaMemcpyAsync(&h[0], ctx->ct_flag.as<u64>() + n, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&h[1], ctx->ct_cptr.as<u64>() + n, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&h[2], ctx->ct_boff.as<u64>() + n, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&h[3], d_cnt, 16, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    elba_fe_contig_info_t I; std::memset(&I, 0, sizeof I);
    I.ncontigs = h[0]; I.contig_reads = h[1]; I.bases = h[2]; I.branches = h[3]; I.cycles = h[4];
    int64_t first = 0, count = 0;
    elba_fe_block_extent((int64_t)I.ncontigs, nranks, rank, &first, &count);
    I.first = (u64)first; I.count = (u64)count;
    // this rank's block: bases and bytes per contig, byte offsets, then the packed sequences
    const u64 c1 = I.count + 1;
    CK(ctx->ct_blen.ensure(8 * c1)); CK(ctx->ct_bbyte.ensure(8 * c1));
    k_ct_block<<<nblk(c1, 256), 256, 0, st>>>(ctx->ct_cptr.as<u64>(), ctx->ct_boff.as<u64>(), I.first, I.count, ctx->ct_blen.as<u64>(), ctx->ct_bbyte.as<u64>()); CKL(); LAUNCHED(ctx);
    if ((rc = exclusive_scan_inplace(ctx, ctx->ct_bbyte.as<u64>(), c1))) return rc;
    u64 b[3] = {0, 0, 0};
    CK(cudaMemcpyAsync(&b[0], ctx->ct_bbyte.as<u64>() + I.count, 8, cudaMemcpyDeviceToHost, st));
    u64 cp[2] = {0, 0};
    CK(cudaMemcpyAsync(&cp[0], ctx->ct_cptr.as<u64>() + I.first, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&cp[1], ctx->ct_cptr.as<u64>() + I.first + I.count, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    CK(cudaMemcpyAsync(&b[1], ctx->ct_boff.as<u64>() + cp[0], 8, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&b[2], ctx->ct_boff.as<u64>() + cp[1], 8, cudaMemcpyDeviceToHost, st));
    CK(ctx->ct_packed.ensure(b[0] + 64));
    if (b[0])
    {
        k_ct_pack<<<nblk(b[0], 256), 256, 0, st>>>(ctx->ct_bbyte.as<u64>(), I.count, I.first, ctx->ct_cptr.as<u64>(), ctx->ct_boff.as<u64>(), ctx->ct_read.as<int64_t>(),
            ctx->ct_rev.as<uint8_t>(), ctx->ct_beg.as<u32>(), ctx->ct_end.as<u32>(), base, rd, ctx->ct_packed.as<uint8_t>()); CKL(); LAUNCHED(ctx);
    }
    CK(cudaEventRecord(ctx->ct_e1, st));
    CK(cudaStreamSynchronize(st));
    I.my_bytes = b[0]; I.my_bases = b[2] - b[1];
    float ms = 0; if (cudaEventElapsedTime(&ms, ctx->ct_e0, ctx->ct_e1) == cudaSuccess) I.ms = ms;
    ctx->ct_info = I; ctx->ct_done = true;
    if (info) *info = I;
    return 0;
}

int elba_fe_contigs(elba_fe_ctx *ctx, elba_fe_contig_info_t *info)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (!ctx->og_done || !ctx->tr_done || !ctx->tr_resident)
        return fail(ctx, ELBA_FE_ERR_STATE, "elba_fe_contigs: needs the string graph of elba_fe_reduce_overlap_graph of the current overlap graph");
    if (ctx->read_gen != ctx->xd_read_gen || ctx->phase < 4) return fail(ctx, ELBA_FE_ERR_STATE, "elba_fe_contigs: the reads changed after elba_fe_align");
    const u64 Nt = ctx->og_nreads, m = ctx->tr_out;
    if (Nt >= 0xFFFFFFF0ull || m >= 0xFFFFFFF0ull) return fail(ctx, ELBA_FE_ERR_INVALID, "elba_fe_contigs: too many reads or string-graph entries");
    CK(cudaSetDevice(ctx->cfg.device));
    ctx->ct_done = false;
    { int rcw = wait_reads(ctx); if (rcw) return rcw; }
    CtReads rd;
    if (ctx->comm.nranks > 1) { rd.buf = ctx->xa_buf.as<uint8_t>(); rd.off = ctx->xa_off.as<u64>(); rd.len = ctx->xa_len.as<u32>(); }
    else { rd.buf = ctx->packed.as<uint8_t>(); rd.off = ctx->off.as<u64>(); rd.len = ctx->len32.as<u32>(); }
    return contigs_device(ctx, ctx->tr_orow.as<int64_t>(), ctx->tr_ocol.as<int64_t>(), ctx->tr_of.as<int32_t>(), m, (u32)Nt, ctx->og_base, rd,
                          ctx->comm.rank, std::max(ctx->comm.nranks, 1), info);
}

int elba_fe_contigs_from_graph(elba_fe_ctx *ctx, const int64_t *row, const int64_t *col, const int32_t *fields, uint64_t nnz, elba_fe_contig_info_t *info)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (ctx->phase < 1) return fail(ctx, ELBA_FE_ERR_STATE, "elba_fe_contigs_from_graph: no reads resident");
    if (nnz >= 0xFFFFFFF0ull) return fail(ctx, ELBA_FE_ERR_INVALID, "elba_fe_contigs_from_graph: too many entries");
    if (nnz && (!row || !col || !fields)) return fail(ctx, ELBA_FE_ERR_INVALID, "elba_fe_contigs_from_graph: null triples");
    const int64_t base = ctx->read_id_offset, n = (int64_t)ctx->n;
    // validate, and sort row-major: key = local row << 32 | local column
    std::vector<std::pair<u64, u64>> key(nnz);
    for (u64 e = 0; e < nnz; ++e)
    {
        if (row[e] < base || row[e] >= base + n || col[e] < base || col[e] >= base + n)
            return fail(ctx, ELBA_FE_ERR_INVALID, "elba_fe_contigs_from_graph: read id outside this context's reads");
        if (row[e] == col[e]) return fail(ctx, ELBA_FE_ERR_INVALID, "elba_fe_contigs_from_graph: diagonal entry");
        if (fields[4 * e] < 0 || fields[4 * e] > 3) return fail(ctx, ELBA_FE_ERR_INVALID, "elba_fe_contigs_from_graph: direction outside 0..3");
        key[e] = { ((u64)(row[e] - base) << 32) | (u64)(col[e] - base), e };
    }
    std::sort(key.begin(), key.end());
    for (u64 e = 0; e < nnz; ++e)
    {
        if (e && key[e].first == key[e - 1].first) return fail(ctx, ELBA_FE_ERR_INVALID, "elba_fe_contigs_from_graph: repeated coordinate");
        const u64 mirror = (key[e].first << 32) | (key[e].first >> 32);
        if (!std::binary_search(key.begin(), key.end(), std::make_pair(mirror, (u64)0), [](const std::pair<u64, u64> &a, const std::pair<u64, u64> &b) { return a.first < b.first; }))
            return fail(ctx, ELBA_FE_ERR_INVALID, "elba_fe_contigs_from_graph: not symmetric");
    }
    std::vector<int64_t> r(nnz), c(nnz); std::vector<int32_t> f(4 * nnz);
    for (u64 e = 0; e < nnz; ++e)
    {
        const u64 s = key[e].second;
        r[e] = row[s]; c[e] = col[s]; for (int j = 0; j < 4; ++j) f[4 * e + j] = fields[4 * s + j];
    }
    CK(cudaSetDevice(ctx->cfg.device));
    ctx->ct_done = false;
    { int rcw = wait_reads(ctx); if (rcw) return rcw; }
    cudaStream_t st = ctx->stream;
    CK(ctx->ct_in_row.ensure(8 * nnz + 8)); CK(ctx->ct_in_col.ensure(8 * nnz + 8)); CK(ctx->ct_in_f.ensure(16 * nnz + 16));
    if (nnz)
    {
        CK(cudaMemcpyAsync(ctx->ct_in_row.p, r.data(), 8 * nnz, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(ctx->ct_in_col.p, c.data(), 8 * nnz, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(ctx->ct_in_f.p, f.data(), 16 * nnz, cudaMemcpyHostToDevice, st));
    }
    CtReads rd; rd.buf = ctx->packed.as<uint8_t>(); rd.off = ctx->off.as<u64>(); rd.len = ctx->len32.as<u32>();
    return contigs_device(ctx, ctx->ct_in_row.as<int64_t>(), ctx->ct_in_col.as<int64_t>(), ctx->ct_in_f.as<int32_t>(), nnz, ctx->n, base, rd, 0, 1, info);
}

int elba_fe_get_contig_layout(elba_fe_ctx *ctx, uint64_t *ptr, int64_t *read, uint8_t *reverse, uint32_t *beg, uint32_t *end)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (!ctx->ct_done) return fail(ctx, ELBA_FE_ERR_STATE, "elba_fe_get_contig_layout: call elba_fe_contigs first");
    CK(cudaSetDevice(ctx->cfg.device));
    const u64 C = ctx->ct_info.ncontigs, R = ctx->ct_info.contig_reads;
    if (ptr && C) D2H(ptr, ctx->ct_cptr.p, 8 * (C + 1));
    if (ptr && !C) ptr[0] = 0;
    D2H(read, ctx->ct_read.p, 8 * R); D2H(reverse, ctx->ct_rev.p, R); D2H(beg, ctx->ct_beg.p, 4 * R); D2H(end, ctx->ct_end.p, 4 * R);
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int elba_fe_get_contigs(elba_fe_ctx *ctx, uint8_t *packed, uint64_t *byte_off, uint64_t *len)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (!ctx->ct_done) return fail(ctx, ELBA_FE_ERR_STATE, "elba_fe_get_contigs: call elba_fe_contigs first");
    CK(cudaSetDevice(ctx->cfg.device));
    const u64 K = ctx->ct_info.count;
    D2H(packed, ctx->ct_packed.p, ctx->ct_info.my_bytes); D2H(byte_off, ctx->ct_bbyte.p, 8 * K); D2H(len, ctx->ct_blen.p, 8 * K);
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int elba_fe_device_contigs(elba_fe_ctx *ctx, const uint8_t **packed, const uint64_t **byte_off, const uint64_t **len)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (!ctx->ct_done) return fail(ctx, ELBA_FE_ERR_STATE, "elba_fe_device_contigs: call elba_fe_contigs first");
    if (packed) *packed = ctx->ct_packed.as<uint8_t>();
    if (byte_off) *byte_off = ctx->ct_bbyte.as<uint64_t>();
    if (len) *len = ctx->ct_blen.as<uint64_t>();
    return 0;
}

// ---- PAF text of the overlap graph and of the string graph (paf.cuh): the files src/main.cpp:303,317 write -----------------
int elba_fe_set_read_names(elba_fe_ctx *ctx, const char *names, const uint64_t *name_off, uint64_t nreads)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (nreads && (!names || !name_off)) return fail(ctx, ELBA_FE_ERR_INVALID, "elba_fe_set_read_names: null names");
    if (nreads >= 0xFFFFFFF0ull) return fail(ctx, ELBA_FE_ERR_INVALID, "elba_fe_set_read_names: too many reads");
    for (u64 r = 0; r < nreads; ++r)
        if (name_off[r + 1] <= name_off[r]) return fail(ctx, ELBA_FE_ERR_INVALID, "elba_fe_set_read_names: empty name (offsets must increase)");
    const u64 b0 = nreads ? name_off[0] : 0, nb = nreads ? name_off[nreads] - b0 : 0;
    for (u64 b = 0; b < nb; ++b)
        if ((unsigned char)names[b0 + b] <= 0x20) return fail(ctx, ELBA_FE_ERR_INVALID, "elba_fe_set_read_names: a name holds a byte <= 0x20 (blank or control)");
    CK(cudaSetDevice(ctx->cfg.device));
    ctx->pf_done = ctx->pf_has_names = false; ctx->pf_nnames = 0;
    if (!nreads) return 0;
    std::vector<u64> off(nreads + 1);
    for (u64 r = 0; r <= nreads; ++r) off[r] = name_off[r] - b0;
    CK(ctx->pf_names.ensure(nb + 16)); CK(ctx->pf_noff.ensure(8 * (nreads + 1)));
    CK(cudaMemcpyAsync(ctx->pf_names.p, names + b0, nb, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->pf_noff.p, off.data(), 8 * (nreads + 1), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->pf_has_names = true; ctx->pf_nnames = nreads;
    return 0;
}

// the n lines of s: lengths and offsets, then the text of lines [first, first + count) into pf_text.
// h = {offset of line first, bytes of lines [first, first + count), bytes of all n lines}
static int paf_text(elba_fe_ctx *ctx, const PafSrc &s, u64 n, u64 first, u64 count, u64 h[3])
{
    cudaStream_t st = ctx->stream;
    int rc;
    CK(ctx->pf_len.ensure(8 * (n + 1)));
    u64 *off = ctx->pf_len.as<u64>();
    k_paf_len<<<nblk(n + 1, 256), 256, 0, st>>>(s, n, off); CKL(); LAUNCHED(ctx);
    if ((rc = exclusive_scan_inplace(ctx, off, n + 1))) return rc;
    u64 b[3] = {0, 0, 0};
    CK(cudaMemcpyAsync(&b[0], off + first, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&b[1], off + first + count, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&b[2], off + n, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    h[0] = b[0]; h[1] = b[1] - b[0]; h[2] = b[2];
    CK(ctx->pf_text.ensure(h[1] + 16));
    if (count) { k_paf_write<<<nblk(count, PAF_THREADS), PAF_THREADS, 0, st>>>(s, off, first, count, ctx->pf_text.as<char>()); CKL(); LAUNCHED(ctx); }
    return 0;
}

int elba_fe_paf(elba_fe_ctx *ctx, int which, elba_fe_paf_info_t *info)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (which != ELBA_FE_PAF_OVERLAP && which != ELBA_FE_PAF_STRING) return fail(ctx, ELBA_FE_ERR_INVALID, "elba_fe_paf: which must be ELBA_FE_PAF_OVERLAP or ELBA_FE_PAF_STRING");
    if (!ctx->og_aligned || !ctx->xd_done || ctx->phase < 4) return fail(ctx, ELBA_FE_ERR_STATE, "elba_fe_paf: call elba_fe_align first");
    if (which == ELBA_FE_PAF_STRING)
    {
        if (!ctx->og_done || !ctx->tr_done || !ctx->tr_resident)
            return fail(ctx, ELBA_FE_ERR_STATE, "elba_fe_paf: needs the string graph of elba_fe_reduce_overlap_graph of the current overlap graph");
        if (ctx->read_gen != ctx->xd_read_gen) return fail(ctx, ELBA_FE_ERR_STATE, "elba_fe_paf: the reads changed after elba_fe_align");
    }
    const int W = std::max(ctx->comm.nranks, 1), me = ctx->comm.rank;
    const u64 Nt = W > 1 ? ctx->N_total : (u64)ctx->n;
    if (ctx->pf_has_names && ctx->pf_nnames != Nt) return fail(ctx, ELBA_FE_ERR_STATE, "elba_fe_paf: the read names are not those of the job's reads (count differs)");
    CK(cudaSetDevice(ctx->cfg.device));
    ctx->pf_done = false;
    { int rcw = wait_reads(ctx); if (rcw) return rcw; }
    cudaStream_t st = ctx->stream;
    int rc;
    CK(cudaEventRecord(ctx->pf_e0, st));
    PafSrc s;
    s.len = W > 1 ? ctx->xa_len.as<u32>() : ctx->len32.as<u32>();
    s.names = ctx->pf_has_names ? ctx->pf_names.as<char>() : nullptr; s.name_off = ctx->pf_noff.as<u64>(); s.id_base = ctx->read_base0;
    elba_fe_paf_info_t I; std::memset(&I, 0, sizeof I);
    u64 h[3];
    if (which == ELBA_FE_PAF_OVERLAP)
    {
        // this rank's alignments, in the order of elba_fe_get_alignments; the ranks' parts follow in rank order
        const u64 np = ctx->xd_pairs;
        s.q = ctx->xd_prow.as<u32>(); s.t = ctx->xd_pcol.as<u32>();
        s.qbase = (u32)(ctx->op.row0 - ctx->read_base0); s.tbase = (u32)(ctx->op.col0 - ctx->read_base0);
        s.v = ctx->xd_out.as<int32_t>(); s.vstride = PAF_XD_FIELDS; s.dir = ctx->xd_out.as<int32_t>() + OG_DIR; s.dstride = PAF_XD_FIELDS;
        if ((rc = paf_text(ctx, s, np, 0, np, h))) return rc;
        I.lines = np; I.bytes = h[1];
        std::vector<u64> bytes, lines;
        if ((rc = allgather_u64(ctx, I.bytes, bytes))) return rc;
        if ((rc = allgather_u64(ctx, I.lines, lines))) return rc;
        for (int r = 0; r < W; ++r)
        {
            if (r < me) I.offset += bytes[r];
            I.total_bytes += bytes[r]; I.total_lines += lines[r];
        }
    }
    else
    {
        // lines = the entries of S with transposed == 0, in S's order; the printed fields come from the source alignment, which
        // one rank holds: every rank fills those of its own, the others are zero, and one sum all-reduce completes them
        const u64 m = ctx->tr_out;
        CK(ctx->pf_flag.ensure(8 * (m + 1)));
        k_paf_flags<<<nblk(m + 1, 256), 256, 0, st>>>(ctx->tr_otr.as<uint8_t>(), m, ctx->pf_flag.as<u64>()); CKL(); LAUNCHED(ctx);
        if ((rc = exclusive_scan_inplace(ctx, ctx->pf_flag.as<u64>(), m + 1))) return rc;
        u64 L = 0;
        CK(cudaMemcpyAsync(&L, ctx->pf_flag.as<u64>() + m, 8, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        const u64 L1 = std::max<u64>(L, 1);
        CK(ctx->pf_q.ensure(4 * L1)); CK(ctx->pf_t.ensure(4 * L1)); CK(ctx->pf_dir.ensure(4 * L1)); CK(ctx->pf_v.ensure(24 * L1));
        u64 r_lo = 0;
        for (int r = 0; r < me; ++r) r_lo += ctx->og_counts[r];
        const u64 r_hi = r_lo + ctx->og_counts[me];
        if (m)
        {
            k_paf_string_lines<<<nblk(m, 256), 256, 0, st>>>(ctx->tr_otr.as<uint8_t>(), ctx->pf_flag.as<u64>(), m, ctx->tr_orow.as<int64_t>(), ctx->tr_ocol.as<int64_t>(),
                ctx->tr_of.as<int32_t>(), ctx->tr_osrc.as<u64>(), ctx->og_base, ctx->og_src.as<u64>(), r_lo, r_hi, ctx->xd_out.as<int32_t>(),
                ctx->pf_q.as<u32>(), ctx->pf_t.as<u32>(), ctx->pf_dir.as<int32_t>(), ctx->pf_v.as<int32_t>()); CKL(); LAUNCHED(ctx);
        }
        if (W > 1 && L) NC(ctx->comm.api->AllReduce(ctx->pf_v.p, ctx->pf_v.p, (size_t)(6 * L), ncclInt32, ncclSum, ctx->comm.comm, st));
        s.q = ctx->pf_q.as<u32>(); s.t = ctx->pf_t.as<u32>(); s.qbase = s.tbase = 0;
        s.v = ctx->pf_v.as<int32_t>(); s.vstride = 6; s.dir = ctx->pf_dir.as<int32_t>(); s.dstride = 1;
        int64_t first = 0, count = 0;
        elba_fe_block_extent((int64_t)L, W, me, &first, &count);
        if ((rc = paf_text(ctx, s, L, (u64)first, (u64)count, h))) return rc;
        I.lines = (u64)count; I.bytes = h[1]; I.offset = h[0]; I.total_lines = L; I.total_bytes = h[2];
    }
    CK(cudaEventRecord(ctx->pf_e1, st));
    CK(cudaStreamSynchronize(st));
    float ms = 0; if (cudaEventElapsedTime(&ms, ctx->pf_e0, ctx->pf_e1) == cudaSuccess) I.ms = ms;
    ctx->pf_info = I; ctx->pf_done = true;
    if (info) *info = I;
    return 0;
}

int elba_fe_get_paf(elba_fe_ctx *ctx, char *text)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (!ctx->pf_done) return fail(ctx, ELBA_FE_ERR_STATE, "elba_fe_get_paf: call elba_fe_paf first");
    CK(cudaSetDevice(ctx->cfg.device));
    D2H(text, ctx->pf_text.p, ctx->pf_info.bytes);
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int elba_fe_device_paf(elba_fe_ctx *ctx, const char **text)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (!ctx->pf_done) return fail(ctx, ELBA_FE_ERR_STATE, "elba_fe_device_paf: call elba_fe_paf first");
    if (text) *text = ctx->pf_text.as<char>();
    return 0;
}

// ---- sketches ---------------------------------------------------------------------------------------
int elba_fe_hll(elba_fe_ctx *ctx, uint8_t *registers, double *estimate)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (ctx->phase < 1) return fail(ctx, ELBA_FE_ERR_STATE, "no reads uploaded");
    CK(cudaSetDevice(ctx->cfg.device));
    { int rcw = wait_reads(ctx); if (rcw) return rcw; }
    CK(ctx->hll_regs.ensure(4 * ELBA_FE_HLL_REGISTERS));
    CK(cudaMemsetAsync(ctx->hll_regs.p, 0, 4 * ELBA_FE_HLL_REGISTERS, ctx->stream));
    if (ctx->nchunks) { k_hll<<<grid_for(ctx, 4), 256, 0, ctx->stream>>>(view(ctx), ctx->cfg.k, ctx->cfg.stride, ctx->hll_regs.as<u32>()); CKL(); LAUNCHED(ctx); }
    std::vector<u32> regs(ELBA_FE_HLL_REGISTERS);
    CK(cudaMemcpyAsync(regs.data(), ctx->hll_regs.p, 4 * ELBA_FE_HLL_REGISTERS, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    // estimate(): src/HyperLogLog.cpp:52-76, same double arithmetic in the same order
    const double size = 4096.0;
    const double alpha_mm = (0.7213 / (1.0 + (1.079 / size))) * size * size;
    double sum = 0.0; uint32_t zeros = 0;
    for (int i = 0; i < ELBA_FE_HLL_REGISTERS; ++i) { sum += 1.0 / (double)(1 << regs[i]); zeros += (regs[i] == 0); if (registers) registers[i] = (uint8_t)regs[i]; }
    double est = alpha_mm / sum;
    if (est <= 2.5 * size && zeros) est = size * std::log(size / zeros);
    if (estimate) *estimate = est;
    return 0;
}

int elba_fe_bloom(elba_fe_ctx *ctx, int64_t entries, double error, int64_t *bits_out, int32_t *hashes_out, int64_t *bytes_out, uint8_t *bf)
{
    if (!ctx) return ELBA_FE_ERR_INVALID;
    if (entries < 1 || !(error > 0 && error < 1)) return fail(ctx, ELBA_FE_ERR_INVALID, "Bloom needs entries >= 1 and 0 < error < 1 (src/Bloom.cpp:8)");
    // sizing: src/Bloom.cpp:10-22
    double bpe = -(std::log(error) / 0.480453013918201);
    int64_t bits = (int64_t)((double)entries * bpe);
    int64_t bytes = (bits / 8) + !!(bits % 8);
    int hashes = (int)std::ceil(0.693147180559945 * bpe);
    if (bits_out) *bits_out = bits; if (hashes_out) *hashes_out = hashes; if (bytes_out) *bytes_out = bytes;
    if (!bf) return 0;
    if (ctx->phase < 1) return fail(ctx, ELBA_FE_ERR_STATE, "no reads uploaded");
    if (bits < 1) return fail(ctx, ELBA_FE_ERR_INVALID, "Bloom filter has no bits");
    CK(cudaSetDevice(ctx->cfg.device));
    size_t words = (size_t)(bytes + 3) / 4;
    { int rcw = wait_reads(ctx); if (rcw) return rcw; }
    CK(ctx->bloom.ensure(4 * words));
    CK(cudaMemsetAsync(ctx->bloom.p, 0, 4 * words, ctx->stream));
    if (ctx->nchunks) { k_bloom_add<<<grid_for(ctx, 4), 256, 0, ctx->stream>>>(view(ctx), ctx->cfg.k, ctx->cfg.stride, ctx->bloom.as<u32>(), (u64)bits, hashes); CKL(); LAUNCHED(ctx); }
    CK(cudaMemcpyAsync(bf, ctx->bloom.p, (size_t)bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int elba_fe_get_kmer_stream(elba_fe_ctx *ctx, uint64_t *out)
{
    if (!ctx || !out) return ELBA_FE_ERR_INVALID;
    if (ctx->phase < 1) return fail(ctx, ELBA_FE_ERR_STATE, "no reads uploaded");
    CK(cudaSetDevice(ctx->cfg.device));
    DevBuf tmp;
    { int rcw = wait_reads(ctx); if (rcw) return rcw; }
    CK(tmp.ensure(8 * std::max<u64>(ctx->M, 1)));
    if (ctx->nchunks) { k_kmer_stream<<<grid_for(ctx, 8), 256, 0, ctx->stream>>>(view(ctx), ctx->cfg.k, tmp.as<u64>()); LAUNCHED(ctx); }
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, tmp.p, 8 * ctx->M, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    tmp.release();
    if (e != cudaSuccess) return fail(ctx, ELBA_FE_ERR_CUDA, cudaGetErrorString(e));
    return 0;
}

} // extern "C"
