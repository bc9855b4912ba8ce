"""Host-side mirror of the reference's interface for the overlap-detection front end.

The reference exposes this path as five C++ free functions
(`include/KmerOps.hpp:24-31`, `include/SharedSeeds.hpp:98-99`) sequenced by
`src/main.cpp:191-282`.  This module keeps their names and argument meaning on
top of the C ABI (`include/elba_fe.h`, built into ``elba_b200/lib/libelba_fe.so``):

    kmermap = get_kmer_count_map_keys(myreads, params)      # pass 1
    get_kmer_count_map_values(myreads, kmermap)             # pass 2 (counts + filter)
    A  = create_kmer_matrix(myreads, kmermap)               # reads x reliable k-mers
    AT = A.transpose()                                      # main.cpp:272-273
    B  = create_seed_matrix(A, AT)                          # SharedSeeds SpGEMM + Prune

All compute happens in the CUDA library.  There is no CPU fallback: importing this
module works anywhere, but creating a context without the library or without a B200
raises ``FrontEndError``.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

from .dnabuffer import DnaBuffer

_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "libelba_fe.so")


class FrontEndError(RuntimeError):
    pass


class _Config(C.Structure):
    _fields_ = [("k", C.c_int32), ("stride", C.c_int32), ("seed_count", C.c_int32), ("lower", C.c_int32),
                ("upper", C.c_int32), ("device", C.c_int32), ("num_partitions", C.c_int32), ("flags", C.c_int32)]


class Sizes(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("nreads", "num_kmers", "distinct", "reliable", "nnzA_pre", "nnzA", "products",
                                          "nnzB_pre", "nnzB", "partitions", "table_slots", "slow_partitions", "candidates", "overflow_instances")] + [("reserved", C.c_uint64 * 2)]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_ if n != "reserved"}


class Timings(C.Structure):
    _fields_ = [("upload_ms", C.c_float), ("count_ms", C.c_float), ("build_ms", C.c_float), ("spgemm_ms", C.c_float),
                ("download_ms", C.c_float), ("count_kernel_ms", C.c_float), ("spgemm_kernel_ms", C.c_float),
                ("kernel_launches", C.c_uint32), ("partition_ms", C.c_float), ("lookup_ms", C.c_float), ("exchange_ms", C.c_float),
                ("exchange_mbytes", C.c_float), ("panel_mbytes", C.c_float), ("align_ms", C.c_float), ("transitive_ms", C.c_float), ("overlap_ms", C.c_float)]

    def as_dict(self):
        return {n: (int(getattr(self, n)) if n == "kernel_launches" else float(getattr(self, n))) for n, _ in self._fields_}


class ContigInfo(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("ncontigs", "contig_reads", "bases", "branches", "cycles", "first", "count", "my_bases", "my_bytes")] + \
               [("ms", C.c_float), ("reserved", C.c_float)]

    def as_dict(self):
        return {n: (float(getattr(self, n)) if n == "ms" else int(getattr(self, n))) for n, _ in self._fields_ if n != "reserved"}


@dataclass
class Contigs:
    """What elba_fe_contigs leaves: the whole job's layout (contig c = entries ptr[c] .. ptr[c + 1] of read, reverse, beg, end) and
    this rank's block of contigs [info["first"], + info["count"]) as packed sequences."""
    info: dict
    ptr: np.ndarray
    read: np.ndarray
    reverse: np.ndarray
    beg: np.ndarray
    end: np.ndarray
    seqs: DnaBuffer


def write_contigs_fa(path: str, seqs: DnaBuffer, first: int = 0, mode: str = "w"):
    """Write contigs as FASTA (`.contigs.fa`): one record `>contig_<id>` per contig, the sequence on one line; ids count from
    `first` (a rank's block appends with mode "a" and its own first id)."""
    with open(path, mode) as fa:
        for i in range(seqs.size()):
            fa.write(f">contig_{first + i}\n{seqs.read_ascii(i)}\n")


def write_at(path: str, data: bytes, offset: int, total: int, dist=None):
    """One file written by every rank at once: rank 0 creates it and sets its size to `total` bytes, then (after a barrier) every
    rank writes its `data` at `offset` with os.pwrite; returns when every rank's part is in.  `dist`: an initialised
    torch.distributed, or None for one process."""
    rank = dist.get_rank() if dist is not None else 0
    if rank == 0:
        fd = os.open(path, os.O_WRONLY | os.O_CREAT | os.O_TRUNC, 0o644)
        os.ftruncate(fd, total)
        os.close(fd)
    if dist is not None:
        dist.barrier()
    fd = os.open(path, os.O_WRONLY)
    try:
        view, pos = memoryview(data), 0
        while pos < len(view):
            pos += os.pwrite(fd, view[pos:], offset + pos)
    finally:
        os.close(fd)
    if dist is not None:
        dist.barrier()


def write_contigs_fa_parallel(path: str, seqs: DnaBuffer, first: int = 0, dist=None):
    """The `.contigs.fa` of write_contigs_fa(path, all contigs) written by every rank at once: each rank's block of contigs
    (ids from `first`) goes to its byte offset, found by all-gathering the ranks' byte counts over `dist` (torch.distributed)."""
    data = "".join(f">contig_{first + i}\n{seqs.read_ascii(i)}\n" for i in range(seqs.size())).encode()
    sizes = [len(data)]
    if dist is not None:
        sizes = [None] * dist.get_world_size()
        dist.all_gather_object(sizes, len(data))
    rank = dist.get_rank() if dist is not None else 0
    write_at(path, data, sum(sizes[:rank]), sum(sizes), dist)


PAF_OVERLAP, PAF_STRING = 0, 1


class PafInfo(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("lines", "bytes", "offset", "total_lines", "total_bytes")] + [("ms", C.c_float), ("reserved", C.c_float)]

    def as_dict(self):
        return {n: (float(getattr(self, n)) if n == "ms" else int(getattr(self, n))) for n, _ in self._fields_ if n != "reserved"}


def check_read_names(names):
    """The names as bytes, checked as elba_fe_set_read_names checks them: every name non-empty, no byte <= 0x20 (PAF columns are
    tab-separated and a FASTA name ends at the first blank).  Raises ValueError."""
    out = []
    for i, n in enumerate(names):
        b = n.encode() if isinstance(n, str) else bytes(n)
        if not b:
            raise ValueError(f"read name {i} is empty")
        if min(b) <= 0x20:
            raise ValueError(f"read name {i} ({b[:40]!r}) holds a blank or control byte")
        out.append(b)
    return out


def write_paf(path: str, ctx: "Context", which: int, dist=None) -> dict:
    """`<prefix>.overlap.paf` (which = PAF_OVERLAP) or `.string.paf` (PAF_STRING) formatted on the device (Context.paf) and
    written by every rank at its offset into one file; collective on several GPUs.  Returns the info dict."""
    text, info = ctx.paf(which)
    write_at(path, text, info["offset"], info["total_bytes"], dist)
    return info


# every symbol include/elba_fe.h declares (tests check the library exports all of them)
ABI_SYMBOLS = (
    "elba_fe_default_config", "elba_fe_create", "elba_fe_destroy", "elba_fe_last_error", "elba_fe_version", "elba_fe_set_stream",
    "elba_fe_upload_reads", "elba_fe_set_reads_device", "elba_fe_count", "elba_fe_build_A", "elba_fe_spgemm", "elba_fe_run",
    "elba_fe_synchronize", "elba_fe_sizes", "elba_fe_get_kmers", "elba_fe_get_A", "elba_fe_get_AT", "elba_fe_get_B",
    "elba_fe_get_B_triples", "elba_fe_device_B", "elba_fe_device_A", "elba_fe_hll", "elba_fe_bloom", "elba_fe_get_kmer_stream",
    "elba_fe_timings", "elba_fe_reset_timings", "elba_fe_align", "elba_fe_get_alignments",
    "elba_fe_comm_get_id", "elba_fe_comm_init", "elba_fe_comm_set_grid", "elba_fe_comm_info", "elba_fe_block_extent", "elba_fe_sizes_global",
    "elba_fe_digests", "elba_fe_device_count",
    "elba_fe_transitive_reduction", "elba_fe_get_string_graph",
    "elba_fe_overlap_graph", "elba_fe_get_overlap_graph", "elba_fe_reduce_overlap_graph",
    "elba_fe_ingest_fasta", "elba_fe_reads_size", "elba_fe_get_reads", "elba_fe_B_dcsc", "elba_fe_get_B_dcsc", "elba_fe_device_B_dcsc",
    "elba_fe_contigs", "elba_fe_contigs_from_graph", "elba_fe_get_contig_layout", "elba_fe_get_contigs", "elba_fe_device_contigs",
    "elba_fe_set_read_names", "elba_fe_paf", "elba_fe_get_paf", "elba_fe_device_paf",
)

_lib = None


def load_library():
    """dlopen the C-ABI library.  Raises FrontEndError (never falls back) if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            raise FrontEndError(f"{_LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                                "(nvcc, sm_100a). There is no CPU fallback.")
        L = C.CDLL(_LIB_PATH)
        L.elba_fe_last_error.restype = C.c_char_p
        L.elba_fe_last_error.argtypes = [C.c_void_p]
        for name in ABI_SYMBOLS:
            getattr(L, name)
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


@dataclass
class Params:
    """Run-time equivalents of the reference's compile-time macros (Makefile:1-6)."""
    k: int = 31
    lower: int = 15
    upper: int = 35
    stride: int = 1
    seed_count: int = 2
    device: int = 0
    num_partitions: int = 0


class Context:
    """One elba_fe_ctx: owns every device buffer of the path for one set of reads."""

    def __init__(self, params: Params):
        self.L = load_library()
        self.params = params
        cfg = _Config(params.k, params.stride, params.seed_count, params.lower, params.upper, params.device, params.num_partitions, 0)
        h = C.c_void_p()
        rc = self.L.elba_fe_create(C.byref(cfg), C.byref(h))
        if rc != 0:
            raise FrontEndError(f"elba_fe_create failed ({rc}): {self.L.elba_fe_last_error(None).decode()}")
        self.h = h
        self.nreads = 0

    def _ck(self, rc):
        if rc != 0:
            raise FrontEndError(f"elba_fe error {rc}: {self.L.elba_fe_last_error(self.h).decode()}")

    def close(self):
        if getattr(self, "h", None):
            self.L.elba_fe_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- input ----------------------------------------------------------------
    def upload(self, dna: DnaBuffer, read_id_offset: int = 0):
        self.nreads = dna.size()
        self._keep = dna
        self._ck(self.L.elba_fe_upload_reads(self.h, _p(dna.buf), C.c_uint64(dna.buf.shape[0]), _p(dna.offsets), _p(dna.lengths),
                                             C.c_uint64(dna.size()), C.c_int64(read_id_offset)))

    def upload_raw(self, buf_ptr: int, nbytes: int, off_ptr: int, len_ptr: int, nreads: int, read_id_offset: int = 0):
        """Host pointers (e.g. pinned torch tensors)."""
        self.nreads = nreads
        self._ck(self.L.elba_fe_upload_reads(self.h, C.c_void_p(buf_ptr), C.c_uint64(nbytes), C.c_void_p(off_ptr), C.c_void_p(len_ptr),
                                             C.c_uint64(nreads), C.c_int64(read_id_offset)))

    def set_reads_device(self, buf_ptr: int, nbytes: int, off_ptr: int, len_ptr: int, nreads: int, read_id_offset: int = 0):
        """Device pointers (reads already resident in HBM)."""
        self.nreads = nreads
        self._ck(self.L.elba_fe_set_reads_device(self.h, C.c_void_p(buf_ptr), C.c_uint64(nbytes), C.c_void_p(off_ptr), C.c_void_p(len_ptr),
                                                 C.c_uint64(nreads), C.c_int64(read_id_offset)))

    def ingest_fasta(self, chunk, chunk_pos: int, records: np.ndarray, read_id_offset: int = 0):
        """FastaIndex::getmydna on the device (src/FastaIndex.cpp:191-290): `chunk` = the bytes [chunk_pos, chunk_pos + len(chunk))
        of the FASTA file (bytes / uint8 array), `records` = (nreads, 3) uint64 .fai records (len, pos, bases)."""
        rec = np.ascontiguousarray(records, dtype=np.uint64).reshape(-1, 3)
        raw = np.frombuffer(chunk, dtype=np.uint8) if isinstance(chunk, (bytes, bytearray, memoryview)) else np.ascontiguousarray(chunk, dtype=np.uint8)
        self.nreads = len(rec)
        self._ck(self.L.elba_fe_ingest_fasta(self.h, _p(raw) if raw.size else None, C.c_uint64(raw.size), C.c_uint64(chunk_pos),
                                             _p(rec) if len(rec) else None, C.c_uint64(len(rec)), C.c_int64(read_id_offset)))

    def reads(self) -> DnaBuffer:
        """The resident DnaBuffer back on the host (arena, offsets, lengths)."""
        n, nb = C.c_uint64(), C.c_uint64()
        self._ck(self.L.elba_fe_reads_size(self.h, C.byref(n), C.byref(nb)))
        buf, off, lens = np.zeros(nb.value, np.uint8), np.zeros(n.value, np.uint64), np.zeros(n.value, np.uint64)
        self._ck(self.L.elba_fe_get_reads(self.h, _p(buf), _p(off), _p(lens)))
        return DnaBuffer(buf, off.astype(np.uint64), lens.astype(np.uint64))

    def set_stream(self, cuda_stream: int):
        self._ck(self.L.elba_fe_set_stream(self.h, C.c_void_p(cuda_stream)))

    # -- phases ----------------------------------------------------------------
    def count(self):
        self._ck(self.L.elba_fe_count(self.h))

    def build_A(self):
        self._ck(self.L.elba_fe_build_A(self.h))

    def spgemm(self):
        self._ck(self.L.elba_fe_spgemm(self.h))

    def run(self):
        self._ck(self.L.elba_fe_run(self.h))

    def synchronize(self):
        self._ck(self.L.elba_fe_synchronize(self.h))

    def sizes(self) -> dict:
        s = Sizes()
        self._ck(self.L.elba_fe_sizes(self.h, C.byref(s)))
        return s.as_dict()

    def sizes_global(self) -> dict:
        s = Sizes()
        self._ck(self.L.elba_fe_sizes_global(self.h, C.byref(s)))
        return s.as_dict()

    def digests(self) -> dict:
        """Whole-job multiset hashes of the results (elba_fe_digests; collective on several GPUs): hex strings."""
        d = (C.c_uint64 * 4)()
        self._ck(self.L.elba_fe_digests(self.h, d))
        return {n: f"{int(d[i]):016x}" for i, n in enumerate(("kmers", "A", "B", "seeds"))}

    # -- several GPUs (one Context per process / GPU) ---------------------------------------------
    @staticmethod
    def comm_get_id() -> bytes:
        L = load_library()
        buf = C.create_string_buffer(128)
        rc = L.elba_fe_comm_get_id(buf)
        if rc != 0:
            raise FrontEndError(f"elba_fe_comm_get_id failed ({rc}): {L.elba_fe_last_error(None).decode()}")
        return buf.raw

    def comm_init(self, comm_id: bytes, rank: int, nranks: int, grid=None):
        buf = C.create_string_buffer(bytes(comm_id), 128)
        self._ck(self.L.elba_fe_comm_init(self.h, buf, C.c_int(rank), C.c_int(nranks)))
        if grid is not None:
            self._ck(self.L.elba_fe_comm_set_grid(self.h, C.c_int(grid[0]), C.c_int(grid[1])))

    def comm_info(self) -> dict:
        i = [C.c_int() for _ in range(4)]
        e = [C.c_int64() for _ in range(4)]
        self._ck(self.L.elba_fe_comm_info(self.h, *[C.byref(x) for x in i], *[C.byref(x) for x in e]))
        return dict(rank=i[0].value, nranks=i[1].value, grid_rows=i[2].value, grid_cols=i[3].value,
                    row0=e[0].value, nrows=e[1].value, col0=e[2].value, ncols=e[3].value)

    def timings(self) -> dict:
        t = Timings()
        self._ck(self.L.elba_fe_timings(self.h, C.byref(t)))
        return t.as_dict()

    def reset_timings(self):
        self._ck(self.L.elba_fe_reset_timings(self.h))

    # -- results -----------------------------------------------------------------
    def kmers(self):
        R = self.sizes()["reliable"]
        k, c = np.zeros(R, np.uint64), np.zeros(R, np.uint32)
        self._ck(self.L.elba_fe_get_kmers(self.h, _p(k), _p(c)))
        return k, c

    def A(self):
        s = self.sizes()
        rp, col, pos = np.zeros(s["nreads"] + 1, np.int64), np.zeros(s["nnzA"], np.uint32), np.zeros(s["nnzA"], np.uint32)
        self._ck(self.L.elba_fe_get_A(self.h, _p(rp), _p(col), _p(pos)))
        return rp, col, pos

    def AT(self):
        s = self.sizes()
        cp, row, pos = np.zeros(s["reliable"] + 1, np.int64), np.zeros(s["nnzA"], np.uint32), np.zeros(s["nnzA"], np.uint32)
        self._ck(self.L.elba_fe_get_AT(self.h, _p(cp), _p(row), _p(pos)))
        return cp, row, pos

    def B(self):
        s = self.sizes()
        rp, col = np.zeros(self.comm_info()["nrows"] + 1, np.int64), np.zeros(s["nnzB"], np.uint32)
        num, seeds = np.zeros(s["nnzB"], np.int32), np.zeros((s["nnzB"], 4), np.uint32)
        self._ck(self.L.elba_fe_get_B(self.h, _p(rp), _p(col), _p(num), _p(seeds)))
        return rp, col, num, seeds

    def B_dcsc(self):
        """B column-major and doubly compressed, CombBLAS' Dcsc arrays (src/PairwiseAlignment.cpp:16-56): (jc, cp, ir, numshared, seeds),
        local indices of this rank's block, rows ascending within a column."""
        nzc = C.c_uint64()
        self._ck(self.L.elba_fe_B_dcsc(self.h, C.byref(nzc)))
        nnz = self.sizes()["nnzB"]
        jc, cp, ir = np.zeros(nzc.value, np.int64), np.zeros(nzc.value + 1, np.int64), np.zeros(nnz, np.int64)
        num, seeds = np.zeros(nnz, np.int32), np.zeros((nnz, 4), np.uint32)
        self._ck(self.L.elba_fe_get_B_dcsc(self.h, _p(jc), _p(cp), _p(ir), _p(num), _p(seeds)))
        return jc, cp, ir, num, seeds

    def B_triples(self):
        s = self.sizes()
        row, col = np.zeros(s["nnzB"], np.int64), np.zeros(s["nnzB"], np.int64)
        num, seeds = np.zeros(s["nnzB"], np.int32), np.zeros((s["nnzB"], 4), np.uint32)
        self._ck(self.L.elba_fe_get_B_triples(self.h, _p(row), _p(col), _p(num), _p(seeds)))
        return row, col, num, seeds

    ALIGN_FIELDS = ("begQ", "endQ", "begT", "endT", "score", "rc", "passed", "containedQ", "containedT", "direction", "directionT", "suffix", "suffixT")

    def align(self, mat: int = 1, mis: int = -1, gap: int = -1, dropoff: int = 15, fetch: bool = True):
        """X-drop seed-and-extend of B's nonzeros (PairwiseAlignment, src/PairwiseAlignment.cpp:5-106; defaults src/main.cpp:53-56):
        (rows, cols, fields[npairs, 13]) with global read ids, pairs in B's row-major order.  fetch=False leaves the alignments
        on the device and returns only their number."""
        n = C.c_uint64()
        self._ck(self.L.elba_fe_align(self.h, C.c_int(mat), C.c_int(mis), C.c_int(gap), C.c_int(dropoff), C.byref(n)))
        if not fetch:
            return int(n.value)
        rows, cols = np.zeros(n.value, np.int64), np.zeros(n.value, np.int64)
        out = np.zeros((n.value, len(self.ALIGN_FIELDS)), np.int32)
        self._ck(self.L.elba_fe_get_alignments(self.h, _p(rows), _p(cols), _p(out)))
        return rows, cols, out

    TR_FIELDS = ("direction", "directionT", "suffix", "suffixT")

    def transitive_reduction(self, nreads: int, rows, cols, fields, fuzz: int = 1000):
        """TransitiveReduction(R) (src/TransitiveReduction.cpp:3-92) on the device.  R = triples (row, col, fields[nnz, 4] =
        direction, directionT, suffix, suffixT).  Returns the string graph S row-major: (rows, cols, fields[nnzS, 4], src, transposed)."""
        rows, cols = np.ascontiguousarray(rows, np.int64), np.ascontiguousarray(cols, np.int64)
        fields = np.ascontiguousarray(fields, np.int32).reshape(-1, 4)
        n = C.c_uint64()
        self._ck(self.L.elba_fe_transitive_reduction(self.h, _p(rows) if len(rows) else None, _p(cols) if len(rows) else None, _p(fields) if len(rows) else None,
                                                     C.c_uint64(len(rows)), C.c_int64(nreads), C.c_int32(fuzz), C.byref(n)))
        m = n.value
        orow, ocol, of = np.zeros(m, np.int64), np.zeros(m, np.int64), np.zeros((m, 4), np.int32)
        osrc, otr = np.zeros(m, np.uint64), np.zeros(m, np.uint8)
        self._ck(self.L.elba_fe_get_string_graph(self.h, _p(orow), _p(ocol), _p(of), _p(osrc), _p(otr)))
        return orow, ocol, of, osrc, otr

    def overlap_graph(self):
        """The overlap graph R from the resident alignments (the prunes of src/main.cpp:300-313, elba_fe_overlap_graph; collective
        on several GPUs, where every rank gets the whole R): (rows, cols, fields[nnz, 4] = direction, directionT, suffix, suffixT,
        src_rank, src_pair, ncontained) with global read ids; src_rank / src_pair name the alignment of `align()` on that rank."""
        n, nc = C.c_uint64(), C.c_uint64()
        self._ck(self.L.elba_fe_overlap_graph(self.h, C.byref(n), C.byref(nc)))
        m = n.value
        rows, cols, f = np.zeros(m, np.int64), np.zeros(m, np.int64), np.zeros((m, 4), np.int32)
        src_rank, src_pair = np.zeros(m, np.int32), np.zeros(m, np.uint64)
        self._ck(self.L.elba_fe_get_overlap_graph(self.h, _p(rows), _p(cols), _p(f), _p(src_rank), _p(src_pair)))
        return rows, cols, f, src_rank, src_pair, int(nc.value)

    def string_graph(self, fuzz: int = 1000):
        """TransitiveReduction of the resident R (elba_fe_reduce_overlap_graph; call overlap_graph first): the same
        (rows, cols, fields[nnzS, 4], src, transposed) as transitive_reduction, src indexing R."""
        n = C.c_uint64()
        self._ck(self.L.elba_fe_reduce_overlap_graph(self.h, C.c_int32(fuzz), C.byref(n)))
        m = n.value
        orow, ocol, of = np.zeros(m, np.int64), np.zeros(m, np.int64), np.zeros((m, 4), np.int32)
        osrc, otr = np.zeros(m, np.uint64), np.zeros(m, np.uint8)
        self._ck(self.L.elba_fe_get_string_graph(self.h, _p(orow), _p(ocol), _p(of), _p(osrc), _p(otr)))
        return orow, ocol, of, osrc, otr

    def _contigs_result(self, info: ContigInfo) -> Contigs:
        d = info.as_dict()
        nc, nr, k = d["ncontigs"], d["contig_reads"], d["count"]
        ptr, read, rev = np.zeros(nc + 1, np.uint64), np.zeros(nr, np.int64), np.zeros(nr, np.uint8)
        beg, end = np.zeros(nr, np.uint32), np.zeros(nr, np.uint32)
        self._ck(self.L.elba_fe_get_contig_layout(self.h, _p(ptr), _p(read), _p(rev), _p(beg), _p(end)))
        packed, off, lens = np.zeros(d["my_bytes"], np.uint8), np.zeros(k, np.uint64), np.zeros(k, np.uint64)
        self._ck(self.L.elba_fe_get_contigs(self.h, _p(packed), _p(off), _p(lens)))
        return Contigs(d, ptr, read, rev, beg, end, DnaBuffer(packed, off, lens))

    def contigs(self) -> Contigs:
        """Contigs from the string graph string_graph() left on the device (elba_fe_contigs; the rule is in include/elba_fe.h):
        the whole job's layout and this rank's block of sequences."""
        info = ContigInfo()
        self._ck(self.L.elba_fe_contigs(self.h, C.byref(info)))
        return self._contigs_result(info)

    def contigs_from_graph(self, rows, cols, fields) -> Contigs:
        """The same from a string graph given on the host (elba_fe_contigs_from_graph) over this context's own reads:
        (rows, cols, fields[nnz, 4] = direction, directionT, suffix, suffixT) with global read ids."""
        rows, cols = np.ascontiguousarray(rows, np.int64), np.ascontiguousarray(cols, np.int64)
        fields = np.ascontiguousarray(fields, np.int32).reshape(-1, 4)
        info = ContigInfo()
        self._ck(self.L.elba_fe_contigs_from_graph(self.h, _p(rows) if len(rows) else None, _p(cols) if len(rows) else None,
                                                   _p(fields) if len(rows) else None, C.c_uint64(len(rows)), C.byref(info)))
        return self._contigs_result(info)

    def set_read_names(self, names):
        """The names of the whole job's reads for the PAF text (elba_fe_set_read_names): names[r] is read r of the job (global id =
        first id of rank 0 + r); str or bytes, checked by check_read_names.  An empty list clears them."""
        b = check_read_names(names)
        off = np.zeros(len(b) + 1, np.uint64)
        off[1:] = np.cumsum([len(x) for x in b], dtype=np.uint64)
        arena = np.frombuffer(b"".join(b), np.uint8) if b else np.zeros(0, np.uint8)
        self._ck(self.L.elba_fe_set_read_names(self.h, _p(arena) if len(b) else None, _p(off) if len(b) else None, C.c_uint64(len(b))))

    def paf(self, which: int = PAF_OVERLAP):
        """PAF text formatted on the device (elba_fe_paf; the format is in include/elba_fe.h): (this rank's part as bytes, info
        dict with lines, bytes, offset, total_lines, total_bytes, ms).  Collective on several GPUs."""
        info = PafInfo()
        self._ck(self.L.elba_fe_paf(self.h, C.c_int(which), C.byref(info)))
        text = np.empty(max(info.bytes, 1), np.uint8)
        self._ck(self.L.elba_fe_get_paf(self.h, _p(text)))
        return text[:info.bytes].tobytes(), info.as_dict()

    def hll(self):
        regs, est = np.zeros(4096, np.uint8), C.c_double()
        self._ck(self.L.elba_fe_hll(self.h, _p(regs), C.byref(est)))
        return float(est.value), regs

    def bloom(self, entries: int, error: float = 0.05, fetch: bool = True):
        bits, hashes, nbytes = C.c_int64(), C.c_int32(), C.c_int64()
        self._ck(self.L.elba_fe_bloom(self.h, C.c_int64(entries), C.c_double(error), C.byref(bits), C.byref(hashes), C.byref(nbytes), None))
        bf = None
        if fetch:
            bf = np.zeros(nbytes.value, np.uint8)
            self._ck(self.L.elba_fe_bloom(self.h, C.c_int64(entries), C.c_double(error), C.byref(bits), C.byref(hashes), C.byref(nbytes), _p(bf)))
        return int(bits.value), int(hashes.value), bf

    def kmer_stream(self):
        M = self._keep.num_kmers(self.params.k) if getattr(self, "_keep", None) is not None else self.sizes()["num_kmers"]
        out = np.zeros(M, np.uint64)
        self._ck(self.L.elba_fe_get_kmer_stream(self.h, _p(out)))
        return out


# ---------------------------------------------------------------------------------------------------------
# The reference's five functions (same names, same order of use as src/main.cpp:191-282)
# ---------------------------------------------------------------------------------------------------------
class KmerCountMap:
    """Stands for `std::unique_ptr<KmerCountMap>` (include/KmerOps.hpp:20-22); the table itself lives in HBM."""

    def __init__(self, ctx: Context):
        self.ctx = ctx
        self.filled = False

    def size(self) -> int:
        return self.ctx.sizes()["reliable"]

    def items(self):
        """(k-mer value, count) of every reliable k-mer, ascending by value == column id order."""
        return self.ctx.kmers()


class KmerMatrix:
    """`CT<PosInRead>::PSpParMat` A (reads x reliable k-mers) or its transpose; device-resident CSR/CSC."""

    def __init__(self, ctx: Context, transposed: bool = False):
        self.ctx, self.transposed = ctx, transposed

    def getnrow(self):
        s = self.ctx.sizes()
        return s["reliable"] if self.transposed else s["nreads"]

    def getncol(self):
        s = self.ctx.sizes()
        return s["nreads"] if self.transposed else s["reliable"]

    def getnnz(self):
        return self.ctx.sizes()["nnzA"]

    def transpose(self) -> "KmerMatrix":
        """`AT = *A; AT->Transpose()` (src/main.cpp:272-273): the CSC view built together with A."""
        return KmerMatrix(self.ctx, not self.transposed)

    def csr(self):
        return self.ctx.AT() if self.transposed else self.ctx.A()


class SeedMatrix:
    """`CT<SharedSeeds>::PSpParMat` B: reads x reads, values (seeds[2], numshared) (include/SharedSeeds.hpp:94-95)."""

    def __init__(self, ctx: Context):
        self.ctx = ctx

    def getnnz(self):
        return self.ctx.sizes()["nnzB"]

    def csr(self):
        return self.ctx.B()

    def triples(self):
        return self.ctx.B_triples()


def get_kmer_count_map_keys(myreads: DnaBuffer, params: Params, read_id_offset: int = 0) -> KmerCountMap:
    """Pass 1 (src/KmerOps.cpp:18-204): uploads the reads.  On the GPU the keys and the values are produced by
    one exact counting pass, which runs in get_kmer_count_map_values; this call only stages the input."""
    ctx = Context(params)
    ctx.upload(myreads, read_id_offset)
    return KmerCountMap(ctx)


def get_kmer_count_map_values(myreads: DnaBuffer, kmermap: KmerCountMap) -> None:
    """Pass 2 (src/KmerOps.cpp:206-350): counts, UPPER/LOWER filter -> the reliable k-mer table."""
    kmermap.ctx.count()
    kmermap.filled = True


def create_kmer_matrix(myreads: DnaBuffer, kmermap: KmerCountMap) -> KmerMatrix:
    """src/KmerOps.cpp:361-401."""
    if not kmermap.filled:
        raise FrontEndError("create_kmer_matrix: call get_kmer_count_map_values first")
    kmermap.ctx.build_A()
    return KmerMatrix(kmermap.ctx)


def create_seed_matrix(A: KmerMatrix, AT: KmerMatrix) -> SeedMatrix:
    """src/SharedSeeds.cpp:4-10."""
    if A.ctx is not AT.ctx or A.transposed or not AT.transposed:
        raise FrontEndError("create_seed_matrix(A, AT): AT must be A.transpose()")
    A.ctx.spgemm()
    return SeedMatrix(A.ctx)


def overlap_front_end(myreads: DnaBuffer, params: Params, read_id_offset: int = 0):
    """The whole path as main.cpp sequences it; returns (kmermap, A, B)."""
    kmermap = get_kmer_count_map_keys(myreads, params, read_id_offset)
    get_kmer_count_map_values(myreads, kmermap)
    A = create_kmer_matrix(myreads, kmermap)
    AT = A.transpose()
    B = create_seed_matrix(A, AT)
    return kmermap, A, B
