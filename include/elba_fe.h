/*
 * elba_fe.h — C ABI of the B200-native ELBA overlap-detection front end.
 *
 * Drop-in boundary for ONE path of PASSIONLab/ELBA (reference commit 4b75895a):
 *
 *     get_kmer_count_map_keys  ->  get_kmer_count_map_values  ->  create_kmer_matrix
 *       ->  Transpose  ->  create_seed_matrix          (reference src/main.cpp:191-282)
 *
 * The reference has no FFI layer; its interface for this path is five C++ free
 * functions (include/KmerOps.hpp:24-31, include/SharedSeeds.hpp:98-99).  The
 * C++ shim elba_b200/host/elba_fe_shim.cpp keeps those five signatures and implements
 * them on top of the symbols below, so src/main.cpp compiles unchanged (see
 * INTEGRATION.md).  Everything here is plain C: pointers and sizes, no C++/torch
 * types.  Every function returns 0 on success or a negative elba_fe_status;
 * elba_fe_last_error() gives the message.  There is NO CPU fallback: without a
 * CUDA device (sm_100a) elba_fe_create fails with ELBA_FE_ERR_NO_DEVICE.
 *
 * Results are bit-exact against the reference on the same inputs and
 * parameters for everything the reference's own code defines (k-mer stream,
 * reliable k-mer set and counts, A after max-position dedupe, pattern of B,
 * shared-seed counts, prune); which two seed pairs a nonzero retains is decided
 * inside CombBLAS in the reference (unpinned external dependency) and follows
 * the documented canonical rule here (DESIGN.md §"Seed rule").
 *
 * Threading: a context is not thread-safe; all work is enqueued on the
 * context's stream.  Multi-GPU: one context per GPU/process; see
 * elba_fe_comm_* (the calls are collective across the participating contexts).
 */
#ifndef ELBA_FE_H
#define ELBA_FE_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ELBA_FE_VERSION 1
#define ELBA_FE_MAX_KMER_SIZE 32      /* README.md:55-57 MAX_KMER_SIZE; one 64-bit word, Kmer<1> (include/Kmer.hpp:95-97) */
#define ELBA_FE_HLL_REGISTERS 4096    /* HyperLogLog(bits=12), include/HyperLogLog.hpp:17 */

typedef enum {
    ELBA_FE_OK = 0,
    ELBA_FE_ERR_INVALID = -1,      /* bad argument / parameter out of contract */
    ELBA_FE_ERR_NO_DEVICE = -2,    /* no usable CUDA device: there is no CPU fallback */
    ELBA_FE_ERR_CUDA = -3,         /* a CUDA call failed */
    ELBA_FE_ERR_OOM = -4,          /* device allocation failed */
    ELBA_FE_ERR_STATE = -5,        /* call sequence violated (e.g. spgemm before build_A) */
    ELBA_FE_ERR_COMM = -6          /* NCCL / multi-GPU failure */
} elba_fe_status;

/*
 * Run-time parameters.  In the reference k / LOWER / UPPER are compile-time
 * macros (Makefile:1-6, include/compiletime.h:7-22), stride is hard-wired to 1
 * (include/KmerOps.hpp:106-136) and the seed count to 2 (include/SharedSeeds.hpp:94).
 */
typedef struct {
    int32_t k;              /* KMER_SIZE, 3..32; parity pinned for odd k <= 31 */
    int32_t stride;         /* visit window starts p with p % stride == 0; reference == 1 */
    int32_t seed_count;     /* seed pairs kept per read pair, 1..2; reference == 2 */
    int32_t lower;          /* LOWER_KMER_FREQ, >= 2 (with 1 the reference depends on Bloom false positives) */
    int32_t upper;          /* UPPER_KMER_FREQ, lower..65535 (include/compiletime.h:21) */
    int32_t device;         /* CUDA device ordinal */
    int32_t num_partitions; /* level-1 k-mer partitions: 0 = choose (~1 M instances each); 1 = direct (one global table, no partition pass); 2..4096 */
    int32_t flags;          /* ELBA_FE_FLAG_* */
} elba_fe_config;

#define ELBA_FE_FLAG_UPPER_TRIANGLE 1   /* keep only B(i,j), i <= j ... reserved, not implemented: rejected */

typedef struct elba_fe_ctx elba_fe_ctx;

/* ---- lifetime ------------------------------------------------------------------ */
void        elba_fe_default_config(elba_fe_config *cfg);     /* k=31 L=15 U=35 (Makefile:1-3), stride 1, seeds 2 */
/* create: needs a compute-capability 10.0 device (the library carries sm_100a code only).  Side effect on the process:
 * cudaLimitMaxL2FetchGranularity is set to 32 bytes for the device (sector-random table probes and 32-byte records). */
int         elba_fe_create(const elba_fe_config *cfg, elba_fe_ctx **out);
int         elba_fe_destroy(elba_fe_ctx *ctx);
const char *elba_fe_last_error(const elba_fe_ctx *ctx);      /* ctx may be NULL: error of the last failed create */
int         elba_fe_version(void);
int         elba_fe_device_count(void);                      /* usable (sm_100) CUDA devices this process sees; 0 if none */
/* Use an existing cudaStream_t (e.g. torch's current stream) instead of the context's own. */
int         elba_fe_set_stream(elba_fe_ctx *ctx, void *cuda_stream);

/* ---- input: the reference's DnaBuffer (include/DnaBuffer.hpp, src/DnaBuffer.cpp:5-29) ---------
 * packed:   the arena, 4 bases/byte, base i of a read at bits 6-2*(i%4) of its byte i/4,
 *           A=0 C=1 G=2 T=3 (N was already folded to A by DnaSeq::compress, src/DnaSeq.cpp:7-29)
 * byte_off: offset of read i's first byte in the arena (DnaBuffer::getbufoffset(i) - getbufoffset(0))
 * len:      bases in read i (DnaSeq::size())
 * read_id_offset: global id of local read 0 (the MPI_Exscan of src/KmerOps.cpp:215-216)
 * upload_reads copies from host memory (pinned or pageable): the read tables on the context's stream, a large arena in
 * slices on a second stream so that parsing starts while it arrives (the caller's buffers must stay valid until the
 * next call that synchronises: elba_fe_count / elba_fe_run do).
 * set_reads_device takes pointers already resident in HBM and COPIES them device-to-device into the context's own padded,
 * 4-byte-aligned arena (the parse kernels read whole 32-bit words past a read's last byte); the caller's buffers are
 * free again when the call returns.
 */
int elba_fe_upload_reads(elba_fe_ctx *ctx, const uint8_t *packed, uint64_t packed_bytes,
                         const uint64_t *byte_off, const uint64_t *len, uint64_t nreads, int64_t read_id_offset);
int elba_fe_set_reads_device(elba_fe_ctx *ctx, const uint8_t *d_packed, uint64_t packed_bytes,
                             const uint64_t *d_byte_off, const uint64_t *d_len, uint64_t nreads, int64_t read_id_offset);

/* ---- the step before the path: FASTA ingest on the device (SURVEY.md 8f-2) ------------------------------------
 * Replaces FastaIndex::getmydna (src/FastaIndex.cpp:191-290: one core per rank copies every record line by line and
 * packs it with DnaSeq::compress, src/DnaSeq.cpp:7-29).  chunk = the bytes [chunk_pos, chunk_pos + chunk_bytes) of the
 * FASTA file in host memory (what MPI_File_read_at_all delivers, :236); records = the rank's .fai records exactly as
 * FastaIndex::getmyrecords() holds them (include/FastaIndex.hpp:10: nreads x {size_t len, pos, bases}; base i of a read
 * is the byte at pos + i + i / bases).  The arena it leaves resident is byte-for-byte the reference's DnaBuffer
 * (code table include/DnaSeq.hpp:136-154; N/n -> A; lower case accepted); afterwards the context is in the same state
 * as after elba_fe_upload_reads.  A record that leaves the chunk is ELBA_FE_ERR_INVALID (the reference reads past it). */
int elba_fe_ingest_fasta(elba_fe_ctx *ctx, const char *chunk, uint64_t chunk_bytes, uint64_t chunk_pos,
                         const uint64_t *records /* nreads x 3 */, uint64_t nreads, int64_t read_id_offset);
/* the resident DnaBuffer: its sizes, then arena + tables to the host for the stages that still read it there
 * (DnaBuffer(bufsize, numreads, buf, readlens), src/DnaBuffer.cpp:5-14); any pointer may be NULL */
int elba_fe_reads_size(elba_fe_ctx *ctx, uint64_t *nreads, uint64_t *packed_bytes);
int elba_fe_get_reads(elba_fe_ctx *ctx, uint8_t *packed, uint64_t *byte_off /*nreads*/, uint64_t *len /*nreads*/);

/* ---- the path ------------------------------------------------------------------------------- */
/* get_kmer_count_map_keys + get_kmer_count_map_values (src/KmerOps.cpp:18-350):
 * reliable k-mers {x : lower <= count(x) <= upper}, exact instance counts, column id = rank of x. */
int elba_fe_count(elba_fe_ctx *ctx);
/* create_kmer_matrix + Transpose (src/KmerOps.cpp:361-401, src/main.cpp:272-273):
 * A (reads x reliable k-mers, value = position, duplicates keep the largest position) in device CSR and CSC. */
int elba_fe_build_A(elba_fe_ctx *ctx);
/* create_seed_matrix (src/SharedSeeds.cpp:4-10): B = A (x) A^T under SharedSeeds::Semiring, pruned numshared <= 1. */
int elba_fe_spgemm(elba_fe_ctx *ctx);
/* all three, then a stream synchronize */
int elba_fe_run(elba_fe_ctx *ctx);
int elba_fe_synchronize(elba_fe_ctx *ctx);

/* ---- several GPUs: one context per GPU / process --------------------------------------------------------
 * Replaces the MPI collectives of the path (SURVEY.md §2.2) with NCCL over NVLink: the personalised all-to-all of
 * k-mers (src/KmerOps.cpp:151; the second exchange :274 is not needed), the k-mer id Allreduce/Exscan (:371-374) and
 * the operand broadcasts of the Sparse SUMMA (src/SharedSeeds.cpp:7).  Call order on every rank:
 *   create -> comm_init -> [comm_set_grid] -> upload_reads(own contiguous block of reads, read_id_offset = its first
 *   global id; ranks hold consecutive ranges in rank order) -> count -> build_A -> spgemm   (all collective).
 * After count every rank holds the WHOLE reliable k-mer list (get_kmers); A / A^T are the rows of the rank's own
 * reads (global column ids); B is block (i, j) of the pr x pc grid, rank = i * pc + j, block extents as CombBLAS
 * distributes them (n / parts, remainder to the last; src/DistributedFastaData.cpp:21-29).  Results do not depend
 * on the number of GPUs.  NCCL (libnccl.so.2) is loaded at comm_init with more than one rank, never before. */
typedef struct { char internal[128]; } elba_fe_comm_id;
int  elba_fe_comm_get_id(elba_fe_comm_id *id);                  /* on one rank; ship the bytes to the others (MPI_Bcast, a file, torch.distributed) */
int  elba_fe_comm_init(elba_fe_ctx *ctx, const elba_fe_comm_id *id, int rank, int nranks);
int  elba_fe_comm_set_grid(elba_fe_ctx *ctx, int grid_rows, int grid_cols);   /* default: 1x1, 1x2, 2x2, 2x4, ... (rows <= cols, most square) */
/* this rank's place: grid, and the extent of its block of B (rows [row0, row0+nrows), columns [col0, col0+ncols)) */
int  elba_fe_comm_info(elba_fe_ctx *ctx, int *rank, int *nranks, int *grid_rows, int *grid_cols, int64_t *row0, int64_t *nrows, int64_t *col0, int64_t *ncols);
void elba_fe_block_extent(int64_t n, int parts, int idx, int64_t *offset, int64_t *length);

/* ---- sizes (valid after the phase that produces them; synchronizes the stream) ----------------------- */
typedef struct {
    uint64_t nreads;        /* N (local) */
    uint64_t num_kmers;     /* M: k-mer instances visited */
    uint64_t distinct;      /* D: distinct canonical k-mers */
    uint64_t reliable;      /* R */
    uint64_t nnzA_pre;      /* instances of reliable k-mers (triples before dedupe) */
    uint64_t nnzA;          /* after (read,column) dedupe */
    uint64_t products;      /* F = sum over columns of count^2 (semiring multiplies) */
    uint64_t nnzB_pre;      /* nonzeros of A*A^T before Prune */
    uint64_t nnzB;          /* after Prune(numshared <= 1) */
    uint64_t partitions;    /* k-mer partitions actually used */
    uint64_t table_slots;   /* slots of one count table */
    uint64_t slow_partitions; /* partitions too large for the sub-bucket fan-out, counted whole with the global-table kernel */
    uint64_t candidates;    /* sweep-2 candidate slots (filter hits: true instances + false positives, + chunk padding) */
    uint64_t overflow_instances; /* instances of overflowing sub-buckets (heavy hitters / repeats), counted with the global-table kernel */
    uint64_t reserved[2];
} elba_fe_sizes_t;
int elba_fe_sizes(elba_fe_ctx *ctx, elba_fe_sizes_t *out);
/* the same summed over the GPUs (collective); equals elba_fe_sizes on one GPU */
int elba_fe_sizes_global(elba_fe_ctx *ctx, elba_fe_sizes_t *out);

/* ---- result digests: what a run produced, without moving it to the host -------------------------------------------
 * Order-independent 64-bit multiset hashes (sum mod 2^64 of one mix per entry, GLOBAL ids; elba_b200/csrc/digest.cuh,
 * restated in numpy in tests/common.py): out[0] reliable k-mers + counts (the KmerCountMap of src/KmerOps.cpp:18-350),
 * out[1] A = (read, column id, position) (src/KmerOps.cpp:361-401), out[2] B = (row, column, numshared) after Prune
 * (src/SharedSeeds.cpp:4-10), out[3] B's retained seed positions (include/SharedSeeds.hpp:94-95).  Entries of phases
 * not run yet are 0.  Collective over the GPUs: every rank gets the whole-job values, which do not depend on the
 * number of GPUs or on the grid. */
int elba_fe_digests(elba_fe_ctx *ctx, uint64_t out[4]);

/* ---- results to host (caller allocates from elba_fe_sizes) ------------------------------------------- */
/* reliable k-mers ascending by 64-bit value (== column id order) and their counts */
int elba_fe_get_kmers(elba_fe_ctx *ctx, uint64_t *kmer /*R*/, uint32_t *count /*R*/);
/* A in CSR: rowptr[N+1], col[nnzA] ascending within a row, pos[nnzA] */
int elba_fe_get_A(elba_fe_ctx *ctx, int64_t *rowptr, uint32_t *col, uint32_t *pos);
/* A^T (= A in CSC): colptr[R+1], row[nnzA] (local read ids ascending within a column), pos[nnzA] */
int elba_fe_get_AT(elba_fe_ctx *ctx, int64_t *colptr, uint32_t *row, uint32_t *pos);
/* B in CSR (several GPUs: this rank's block, nrows of elba_fe_comm_info, local row / column ids): rowptr[N+1], col[nnzB] ascending, numshared[nnzB], seeds[nnzB*4] = {s0.q, s0.t, s1.q, s1.t}
 * (SharedSeeds::seeds[2] + numshared, include/SharedSeeds.hpp:94-95; q = position in the row read, t = in the column read) */
int elba_fe_get_B(elba_fe_ctx *ctx, int64_t *rowptr, uint32_t *col, int32_t *numshared, uint32_t *seeds);
/* the same as (row, col, ...) triples with GLOBAL ids, the layout the SpParMat triple constructor takes */
int elba_fe_get_B_triples(elba_fe_ctx *ctx, int64_t *row, int64_t *col, int32_t *numshared, uint32_t *seeds);

/* device pointers of the same arrays (zero-copy hand-off to a device consumer); any may be NULL */
int elba_fe_device_B(elba_fe_ctx *ctx, const int64_t **rowptr, const uint32_t **col, const int32_t **numshared, const uint32_t **seeds);
int elba_fe_device_A(elba_fe_ctx *ctx, const int64_t **rowptr, const uint32_t **col, const uint32_t **pos);

/* B column-major and doubly compressed (SURVEY.md 8f-3): the arrays of CombBLAS' Dcsc<int64_t, SharedSeeds> exactly as the
 * consumer walks them (src/PairwiseAlignment.cpp:16-56: nzc, cp[nzc+1], jc[nzc], ir[nnz], numx[nnz]; row ids ascending
 * within a column; LOCAL row / column indices of this rank's block), made on the device: a host that builds
 * SpDCCols(nrow, ncol, Dcsc*) copies them in as they are, no tuple sort.  elba_fe_B_dcsc builds (once per B) and
 * returns the number of nonempty columns; get_ copies to caller-allocated arrays, device_ hands out the pointers. */
int elba_fe_B_dcsc(elba_fe_ctx *ctx, uint64_t *nzc);
int elba_fe_get_B_dcsc(elba_fe_ctx *ctx, int64_t *jc, int64_t *cp, int64_t *ir, int32_t *numshared, uint32_t *seeds);
int elba_fe_device_B_dcsc(elba_fe_ctx *ctx, const int64_t **jc, const int64_t **cp, const int64_t **ir, const int32_t **numshared, const uint32_t **seeds);

/* ---- the consumer of B (next row of the hot path; first version of the kernel) --------------------------------------- */
/* X-drop seed-and-extend of B's nonzeros: PairwiseAlignment (src/PairwiseAlignment.cpp:5-106) keeps the strict upper
 * triangle of the local block (:52) and runs Overlap(len, seeds[0]).extend_overlap on each (:90-91; src/Overlap.cpp:20-73;
 * xdrop_aligner + classify_alignment, src/XDropAligner.cpp:7-282).  mat / mis / gap / dropoff: src/main.cpp:53-56
 * (1, -1, -1, 15).  *npairs = number of aligned pairs of THIS rank.
 * Several GPUs: COLLECTIVE (every rank calls it): rank (i, j) aligns the nonzeros of its block of B; the reads of the other
 * ranks it needs are all-gathered over NVLink inside the call (the reference: DistributedFastaData, src/DistributedFastaData.cpp:
 * 98-232).  Pairs are selected by the reference's block-local rule (:52) on a square grid and by the global upper triangle
 * (row < column) on the others, where the block-local rule would lose pairs: every unordered pair exactly once either way. */
#define ELBA_FE_ALIGN_FIELDS 13   /* begQ endQ begT endT score rc passed containedQ containedT direction directionT suffix suffixT */
int elba_fe_align(elba_fe_ctx *ctx, int mat, int mis, int gap, int dropoff, uint64_t *npairs);
/* the aligned pairs in B's row-major order: global row / column read ids and ELBA_FE_ALIGN_FIELDS ints each = the fields of
 * the reference's Overlap (include/Overlap.hpp:25-31) that extend_overlap sets */
int elba_fe_get_alignments(elba_fe_ctx *ctx, int64_t *row, int64_t *col, int32_t *fields);

/* ---- behind the consumer: transitive reduction of the overlap graph (SURVEY.md 8f-4; first version, one GPU) ----------
 * TransitiveReduction(R) (src/TransitiveReduction.cpp:3-92; functors include/TransitiveReduction.hpp:19-110).  R comes as nnz
 * triples with distinct coordinates (the matrix src/PairwiseAlignment.cpp:97-103 builds, after the prunes of
 * src/main.cpp:305-311): global read ids in [0, nreads) and four ints per entry = Overlap's direction, directionT, suffix,
 * suffixT (include/Overlap.hpp:27-29), the only fields the algorithm reads.  fuzz = FUZZ (include/TransitiveReduction.hpp:15:
 * 1000).  The string graph S (symmetric: every surviving overlap in both orientations) stays on the device;
 * get_string_graph returns it row-major: coordinates, the four fields as they stand at that coordinate, src = index of the
 * input triple the entry came from and transposed = 1 where it is that triple's mirror image (the host applies
 * Overlap::Transpose, include/Overlap.hpp:46-74, to the rest of the payload).  The matrix is small: every rank may run it
 * on the whole R (replicas only, no collective). */
int elba_fe_transitive_reduction(elba_fe_ctx *ctx, const int64_t *row, const int64_t *col, const int32_t *fields /* nnz x 4 */, uint64_t nnz,
                                 int64_t nreads, int32_t fuzz, uint64_t *nnz_out);
int elba_fe_get_string_graph(elba_fe_ctx *ctx, int64_t *row, int64_t *col, int32_t *fields /* nnz_out x 4 */, uint64_t *src, uint8_t *transposed);

/* ---- from the alignments to the string graph without leaving the device ---------------------------------------------
 * The prunes between PairwiseAlignment and TransitiveReduction (src/main.cpp:300-313) on the alignments elba_fe_align left
 * resident, restated in tests/tr_inputs.py::overlap_graph: over the alignments of ALL ranks, C = the rows of the passed
 * alignments with containedQ and the columns of those with containedT; an alignment stays in the overlap graph R iff it
 * passed and neither of its reads is in C.  An entry of R is (global row, global column, direction, directionT, suffix,
 * suffixT); R is the ranks' kept alignments concatenated in rank order, each rank's in the order of elba_fe_get_alignments.
 * overlap_graph: after elba_fe_align; COLLECTIVE on several GPUs (one all-reduce of one byte per read, then all-gathers):
 * every rank ends up holding the whole R.  *nnz = entries of R, *ncontained = reads in C.  Only scalars reach the host.
 * get_overlap_graph: R to the host; any pointer may be NULL; src_rank / src_pair = which rank's alignment the entry is
 * (the index into that rank's elba_fe_get_alignments order).
 * reduce_overlap_graph: TransitiveReduction of the resident R, the kernels and semantics of elba_fe_transitive_reduction with
 * nreads = the reads of the whole job; no collective (every rank reduces its replica).  The result is read with
 * elba_fe_get_string_graph, where src indexes R.  More than 2^31 entries in R is ELBA_FE_ERR_INVALID.
 * elba_fe_count, elba_fe_build_A, elba_fe_spgemm and elba_fe_align discard R: the calls after them are ELBA_FE_ERR_STATE
 * until the next elba_fe_overlap_graph. */
int elba_fe_overlap_graph(elba_fe_ctx *ctx, uint64_t *nnz, uint64_t *ncontained);
int elba_fe_get_overlap_graph(elba_fe_ctx *ctx, int64_t *row, int64_t *col, int32_t *fields /* nnz x 4 */,
                              int32_t *src_rank, uint64_t *src_pair);
int elba_fe_reduce_overlap_graph(elba_fe_ctx *ctx, int32_t fuzz, uint64_t *nnz_out);

/* ---- contigs from the string graph (the stage GenerateContigs runs in the reference, src/main.cpp:320) -------------------
 * The rule (DESIGN.md §3d; restated in tests/contig_inputs.py; parity with the reference's own contig output is UNPINNED):
 * entry e = (i, j) of S has t(e) = (dir >> 1) & 1, the end of read i it leaves from (0 = 3' end, 1 = 5' start), and suffix =
 * the bases j adds beyond i.  A read is a branch if its row of S has more than two entries, or two with the same t.  The
 * chain graph G = the entries of S between two reads that are not branches (and whose mirror is in S); every component of G
 * with two or more reads is a path or a cycle and gives one contig.  A path starts at the smaller of its two end reads; a cycle
 * at its smallest read s, first towards the smaller of s's two neighbours (the edge to the other one is cut; counted in
 * cycles).  On the walk v0 .. vm, v_k (k < m) is forward iff t(v_k -> v_k+1) == 0 and vm iff t(vm -> vm-1) == 1; v0 adds
 * [0, len), v_k (k >= 1) with s = clamp(suffix(v_k-1 -> v_k), 0, len) adds [len - s, len) forward or [0, s) reverse-complemented.
 * Contigs are numbered in ascending order of their start read's global id, whatever the number of GPUs.
 * contigs: from the S that elba_fe_reduce_overlap_graph left on the device for the current R, and the reads elba_fe_align saw
 *   (ELBA_FE_ERR_STATE otherwise: a host-route elba_fe_transitive_reduction, reads replaced after align).  No collective:
 *   every rank builds the whole layout and the sequences of its block of contigs, elba_fe_block_extent(ncontigs, nranks, rank).
 * contigs_from_graph: S from the host in the layout of elba_fe_get_string_graph over this context's own reads (global ids in
 *   [read_id_offset, read_id_offset + nreads)); checked on the host: ids, dir in 0..3, no diagonal, distinct coordinates,
 *   symmetric coordinates (ELBA_FE_ERR_INVALID otherwise).  No collective; builds every contig.
 * get_contig_layout: the whole job: ptr[ncontigs + 1] into the contig_reads arrays read (global id), reverse (1 = reverse
 *   complemented), beg / end (the segment [beg, end) of the read, before reverse complementing); any pointer may be NULL.
 * get_contigs / device_contigs: this rank's block as a DnaBuffer: 2-bit packed, every contig byte-aligned at byte_off[count],
 *   len[count] bases (u64 both: the device arrays can go straight into elba_fe_set_reads_device of another context).
 * Calls that discard R or replace S or the reads discard the contigs: the getters are ELBA_FE_ERR_STATE until the next call. */
typedef struct {
    uint64_t ncontigs, contig_reads, bases;    /* whole job */
    uint64_t branches, cycles;
    uint64_t first, count, my_bases, my_bytes; /* this rank's block of contigs */
    float ms; float reserved;                  /* device time of the call */
} elba_fe_contig_info_t;
int elba_fe_contigs(elba_fe_ctx *ctx, elba_fe_contig_info_t *info);
int elba_fe_contigs_from_graph(elba_fe_ctx *ctx, const int64_t *row, const int64_t *col, const int32_t *fields /* nnz x 4 */, uint64_t nnz,
                               elba_fe_contig_info_t *info);
int elba_fe_get_contig_layout(elba_fe_ctx *ctx, uint64_t *ptr /* ncontigs + 1 */, int64_t *read, uint8_t *reverse, uint32_t *beg, uint32_t *end);
int elba_fe_get_contigs(elba_fe_ctx *ctx, uint8_t *packed, uint64_t *byte_off, uint64_t *len);
int elba_fe_device_contigs(elba_fe_ctx *ctx, const uint8_t **packed, const uint64_t **byte_off, const uint64_t **len);

/* ---- PAF text of the overlap graph and of the string graph (the reference's <prefix>.overlap.paf / .string.paf,
 * src/main.cpp:303,317), formatted on the device.  The format (DESIGN.md §3d; restated in tests/paf_inputs.py; parity with the
 * reference's own writer is UNPINNED): one line per alignment, 13 tab-separated columns, ending in '\n':
 *     qname qlen begQ endQ strand tname tlen begT endT score max(endQ - begQ, endT - begT) 255 dr:i:<direction>
 * q = the alignment's row read, t = its column read, strand '-' iff rc, the fields those of ELBA_FE_ALIGN_FIELDS (begT / endT
 * are forward-strand coordinates of t); integers in plain decimal (int32 fields may be negative).  A read's name is the one
 * elba_fe_set_read_names gave, else its global id in decimal.
 * set_read_names: the names of the whole job's reads, job-relative: read r (global id = first id of rank 0 + r) is
 *   names[name_off[r], name_off[r + 1]).  Checked on the host: every name non-empty, no byte <= 0x20 (ELBA_FE_ERR_INVALID).
 *   The names stay until replaced; nreads == 0 clears them.  A count other than the job's reads makes elba_fe_paf
 *   ELBA_FE_ERR_STATE.
 * paf(ELBA_FE_PAF_OVERLAP): one line per alignment elba_fe_align made, passed or not (R before the prunes), in the order of
 *   elba_fe_get_alignments; on several GPUs the ranks' parts follow in rank order (COLLECTIVE: one all-gather of the byte counts
 *   gives offset and the totals; every rank formats its own alignments).  After elba_fe_align, else ELBA_FE_ERR_STATE.
 * paf(ELBA_FE_PAF_STRING): one line per entry of the resident S with transposed == 0, in S's row-major order (each surviving
 *   overlap once, in the orientation the aligner produced), printed from the entry's source alignment.  Needs the S that
 *   elba_fe_reduce_overlap_graph left for the current R and the reads elba_fe_align saw (ELBA_FE_ERR_STATE otherwise).  Several
 *   GPUs: COLLECTIVE (one sum all-reduce of 6 int32 per line); every rank formats the lines elba_fe_block_extent(lines, nranks,
 *   rank).  The bytes of the whole file do not depend on the number of GPUs or the grid.
 * info: this rank's part (lines, bytes, its byte offset in the whole file) and the whole file's totals; the rank parts laid
 *   end to end at their offsets are the file.  get_paf copies this rank's part (info.bytes) to the host, device_paf hands out
 *   the device pointer.  The text is that of the last elba_fe_paf; calls that discard the alignments, R or S, replace the reads
 *   or set the names discard it (the getters are ELBA_FE_ERR_STATE until the next elba_fe_paf). */
#define ELBA_FE_PAF_OVERLAP 0
#define ELBA_FE_PAF_STRING  1
typedef struct {
    uint64_t lines, bytes;              /* this rank's part */
    uint64_t offset;                    /* byte offset of this rank's part in the whole file */
    uint64_t total_lines, total_bytes;  /* whole job */
    float ms; float reserved;           /* device time of the call */
} elba_fe_paf_info_t;
int elba_fe_set_read_names(elba_fe_ctx *ctx, const char *names, const uint64_t *name_off /* nreads + 1 */, uint64_t nreads);
int elba_fe_paf(elba_fe_ctx *ctx, int which, elba_fe_paf_info_t *info);
int elba_fe_get_paf(elba_fe_ctx *ctx, char *text /* info.bytes */);
int elba_fe_device_paf(elba_fe_ctx *ctx, const char **text);

/* ---- the reference's sizing sketches, bit-exact (not needed for the result when lower >= 2) ----------- */
/* HyperLogLog over the canonical k-mers of the uploaded reads exactly as KmerEstimateHandler drives it
 * (include/KmerOps.hpp:58-69, src/HyperLogLog.cpp:40-76): registers[4096] and estimate(). */
int elba_fe_hll(elba_fe_ctx *ctx, uint8_t *registers /*4096 or NULL*/, double *estimate);
/* Bloom sized as Bloom(entries, error) (src/Bloom.cpp:6-27) with every canonical k-mer of the uploaded reads
 * added (src/Bloom.cpp:44-73).  bits/hashes/bytes are outputs; bf (bytes long) may be NULL to size only. */
int elba_fe_bloom(elba_fe_ctx *ctx, int64_t entries, double error, int64_t *bits, int32_t *hashes, int64_t *bytes, uint8_t *bf);
/* the canonical k-mer stream itself (ForeachKmer, include/KmerOps.hpp:106-136): out[M], read order then position order */
int elba_fe_get_kmer_stream(elba_fe_ctx *ctx, uint64_t *out /*M*/);

/* ---- measurement ---------------------------------------------------------------------------------------- */
typedef struct {
    float upload_ms;        /* H2D of the reads (upload_reads) */
    float count_ms;         /* elba_fe_count, device time */
    float build_ms;         /* elba_fe_build_A */
    float spgemm_ms;        /* elba_fe_spgemm */
    float download_ms;      /* last get_* */
    float count_kernel_ms;  /* the dominant counting kernel(s) only (sum over partitions) */
    float spgemm_kernel_ms; /* the numeric SpGEMM kernel(s) only */
    uint32_t kernel_launches; /* kernels of this library launched since create/reset */
    float partition_ms;     /* histogram + scatter kernels */
    float lookup_ms;        /* second sweep (seed emission) kernel */
    float exchange_ms;      /* several GPUs: the k-mer exchange: super-k-mer records pushed into the owners' slabs through peer memory + the
                               fill words (k >= 20), or the all-to-all of the level-1 partitions (k < 20) */
    float exchange_mbytes;  /* MB this rank sent in it */
    float panel_mbytes;     /* MB this rank received as routed seed triples and in the all-gather of A's row blocks */
    float align_ms;         /* elba_fe_align: pair selection + the X-drop kernel */
    float transitive_ms;    /* elba_fe_transitive_reduction, elba_fe_reduce_overlap_graph */
    float overlap_ms;       /* elba_fe_overlap_graph (several GPUs: with its all-reduce and all-gathers) */
} elba_fe_timings_t;
int elba_fe_timings(elba_fe_ctx *ctx, elba_fe_timings_t *out);
int elba_fe_reset_timings(elba_fe_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif /* ELBA_FE_H */
