"""From the resident alignments to the string graph on the device: elba_fe_overlap_graph (the prunes between PairwiseAlignment
and TransitiveReduction, src/main.cpp:300-313, as tests/tr_inputs.py::overlap_graph restates them), elba_fe_get_overlap_graph
and elba_fe_reduce_overlap_graph.  R must be exactly the prune of what align() returns, S exactly what the host route
(get_alignments, prune on the CPU, elba_fe_transitive_reduction) gives, and on the stored fixtures the committed digests."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from common import digest
import tr_inputs

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLD = os.path.join(HERE, "golden", "golden_tr.json")
PASSED, CONT_Q, CONT_T = 6, 7, 8
TR_COLS = [9, 10, 11, 12]       # direction, directionT, suffix, suffixT


def prune(rows, cols, fields):
    """The rule of tr_inputs.overlap_graph on alignments (rows, cols, fields[npairs, 13]): (indices of the kept alignments, C)."""
    passed = fields[:, PASSED] != 0
    C = set(rows[passed & (fields[:, CONT_Q] != 0)].tolist()) | set(cols[passed & (fields[:, CONT_T] != 0)].tolist())
    Ca = np.fromiter(C, np.int64, len(C))
    keep = passed & ~np.isin(rows, Ca) & ~np.isin(cols, Ca)
    return np.nonzero(keep)[0], C


def _ctx(k, lo, up):
    from elba_b200 import frontend
    return frontend.Context(frontend.Params(k=k, lower=lo, upper=up, device=0))


def _same(got, want, what):
    for a, b, name in zip(got, want, ("row", "col", "fields", "src", "transposed")):
        assert np.array_equal(a, b), (what, name, len(a), len(b))


def _check_against_host_route(ctx, nreads, base, scoring, what):
    """align -> overlap_graph -> string_graph against the prune of align()'s output and the host transitive reduction."""
    ar, ac, af = ctx.align(*scoring)
    rows, cols, f, src_rank, src_pair, ncont = ctx.overlap_graph()
    idx, C = prune(ar, ac, af)
    assert np.array_equal(rows, ar[idx]) and np.array_equal(cols, ac[idx]), what
    assert np.array_equal(f, af[idx][:, TR_COLS]), what
    assert np.array_equal(src_pair, idx) and (src_rank == 0).all(), what
    assert ncont == len(C), (what, ncont, len(C))
    S = ctx.string_graph()
    _same(S, ctx.transitive_reduction(base + nreads, ar[idx], ac[idx], af[idx][:, TR_COLS]), what)
    return len(ar), int((af[:, PASSED] != 0).sum()), len(C), len(idx), len(S[0])


def test_golden_chain_one_gpu(fixtures):
    from oracle import oracle as O
    g = json.load(open(GOLD))
    for key, want in g.items():
        dna = fixtures(want["fixture"])
        ctx = _ctx(want["k"], want["lower"], want["upper"])
        ctx.upload(dna)
        ctx.run()
        ctx.align(1, -1, -1, 15)
        rows, cols, f, src_rank, src_pair, ncont = ctx.overlap_graph()
        n, er, ec, ef = tr_inputs.overlap_graph(dna, want["k"], want["lower"], want["upper"])
        assert np.array_equal(rows, er) and np.array_equal(cols, ec) and np.array_equal(f, ef), key
        assert len(rows) == want["nnzR"] and digest(rows, cols, f) == want["input_digest"], key
        r, c, of, src, tr = S = ctx.string_graph()
        assert len(r) == want["nnzS"] and digest(r, c, of) == want["digest"], key
        _same(S, ctx.transitive_reduction(n, rows, cols, f), key)
        _same(S, O.transitive_reduction(n, rows, cols, f), key)
        tm = ctx.timings()
        assert tm["overlap_ms"] > 0 and tm["transitive_ms"] > 0
        ctx.close()


@pytest.mark.parametrize("kind,k,lo,up,scoring,base", [
    ("clr", 17, 2, 8, (2, -3, -2, 25), 0),
    ("clr", 17, 2, 8, (1, -1, -1, 15), 1000),          # most pairs fail; every passed pair touches a contained read
    ("clr_large", 17, 2, 8, (2, -3, -2, 25), 123456),
    ("hifi", 31, 2, 4, (1, -1, -1, 15), 1000),
    ("hifi", 31, 2, 4, (1, -2, -1, 7), 0),
])
def test_synthetic_reads_vs_host_route(kind, k, lo, up, scoring, base):
    from elba_b200.synth import make_dnabuffer
    if kind == "clr_large":
        dna = make_dnabuffer(genome_len=120_000, n_reads=300, mean_len=8000, sd_len=1000, err=0.12, seed=3)
    else:
        dna = make_dnabuffer(genome_len=60_000, n_reads=160, mean_len=6000, sd_len=857, err=0.12 if kind == "clr" else 0.01, seed=11)
    ctx = _ctx(k, lo, up)
    ctx.upload(dna, base)
    ctx.run()
    pairs, passed, ncont, kept, nS = _check_against_host_route(ctx, dna.size(), base, scoring, (kind, scoring, base))
    assert pairs > 300 and ncont > 0
    if kind == "clr":
        assert passed < pairs, "CLR-like reads: some alignments fail"
    if kind == "clr" and scoring == (1, -1, -1, 15):
        assert passed > 0 and kept == 0
    else:
        assert 0 < kept < passed and nS > 0
    ctx.close()


def test_edges():
    """No alignments at all; every alignment failing (dovetails shorter than 500 bases); every pair touching a contained read
    (identical copies: all but the last copy are contained).  Each gives an empty R and an empty S, no error."""
    from elba_b200.dnabuffer import DnaBuffer
    rng = np.random.default_rng(4)
    g = "".join("ACGT"[c] for c in rng.integers(0, 4, 5000))
    cases = (("no alignments", DnaBuffer.from_strings(["ACGTACGTACGTACGTACGTAAA", "TTTTGGGGCCCCAAAATTTTGGGC"]), 0, 0),
             ("all fail", DnaBuffer.from_strings([g[200 * i: 200 * i + 400] for i in range(10)]), 9, 0),
             ("all contained", DnaBuffer.from_strings([g[0:2000]] * 4), 6, 3))
    for what, dna, npairs, ncontained in cases:
        for base in (0, 50):
            ctx = _ctx(17, 2, 8)
            ctx.upload(dna, base)
            ctx.run()
            ar, ac, af = ctx.align(1, -1, -1, 15)
            assert len(ar) == npairs, what
            rows, cols, f, src_rank, src_pair, ncont = ctx.overlap_graph()
            assert len(rows) == 0 and f.shape == (0, 4) and ncont == ncontained, what
            r, c, of, src, tr = ctx.string_graph()
            assert len(r) == 0 and of.shape == (0, 4), what
            ctx.close()


def test_call_order_errors():
    from elba_b200 import frontend
    from elba_b200.synth import make_dnabuffer
    import ctypes as C
    dna = make_dnabuffer(genome_len=60_000, n_reads=160, mean_len=6000, sd_len=857, err=0.01, seed=11)
    ctx = _ctx(31, 2, 4)
    L, h = ctx.L, ctx.h

    def get_R():
        return L.elba_fe_get_overlap_graph(h, None, None, None, None, None)

    def reduce_R():
        return L.elba_fe_reduce_overlap_graph(h, C.c_int32(1000), None)
    for call in (ctx.overlap_graph, ctx.string_graph):
        with pytest.raises(frontend.FrontEndError):
            call()                                    # no reads
    assert get_R() == -5 and reduce_R() == -5
    ctx.upload(dna, 7)
    ctx.run()
    with pytest.raises(frontend.FrontEndError):
        ctx.overlap_graph()                           # B, but no alignments
    ctx.align()
    assert get_R() == -5 and reduce_R() == -5        # alignments, but no R
    with pytest.raises(frontend.FrontEndError):
        ctx.string_graph()
    R = ctx.overlap_graph()
    assert len(R[0]) > 0 and get_R() == 0
    S = ctx.string_graph()
    # each of count, build_A, spgemm and align discards R; the first three also the alignments (they belong to the old B)
    redo = {"run": (), "count": ("build_A", "spgemm"), "build_A": ("spgemm",), "spgemm": (), "align": None}
    for step, rest in redo.items():
        ctx.overlap_graph()
        getattr(ctx, step)()
        assert get_R() == -5 and reduce_R() == -5, step
        with pytest.raises(frontend.FrontEndError):
            ctx.string_graph()
        if rest is not None:
            with pytest.raises(frontend.FrontEndError):
                ctx.overlap_graph()
            for s in rest:
                getattr(ctx, s)()
            ctx.align()
    R2 = ctx.overlap_graph()
    for a, b in zip(R, R2):
        assert np.array_equal(a, b)
    _same(ctx.string_graph(), S, "after a second run")
    ctx.close()


def test_host_reduction_interleaved():
    """The host entry point and the resident route share the string-graph buffers: each call's results are its own, and the
    host call leaves the resident R alone."""
    from oracle import oracle as O
    from elba_b200.synth import make_dnabuffer
    dna = make_dnabuffer(genome_len=60_000, n_reads=160, mean_len=6000, sd_len=857, err=0.01, seed=11)
    ctx = _ctx(31, 2, 4)
    ctx.upload(dna, 300)
    ctx.run()
    ar, ac, af = ctx.align()
    R = ctx.overlap_graph()
    S = ctx.string_graph()
    rng = np.random.default_rng(5)
    n = 40
    rows, cols, f = tr_inputs.random_graph(rng, n, density=0.4)
    want = O.transitive_reduction(n, rows, cols, f)
    _same(ctx.transitive_reduction(n, rows, cols, f), want, "host after resident")
    _same(ctx.string_graph(), S, "resident after host")
    _same(ctx.transitive_reduction(n, rows, cols, f), want, "host again")
    got = ctx.L.elba_fe_get_overlap_graph(ctx.h, None, None, None, None, None)
    assert got == 0
    idx, _ = prune(ar, ac, af)
    _same(ctx.string_graph(), ctx.transitive_reduction(300 + dna.size(), ar[idx], ac[idx], af[idx][:, TR_COLS]), "resident vs host")
    assert np.array_equal(R[0], ar[idx])
    ctx.close()


# ---- several GPUs ----------------------------------------------------------------------------------------------------
def _ngpus():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


def _launch(world, args, port):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(HERE, "multi_gpu_string_graph_worker.py")] + [str(a) for a in args]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0 and "MULTI-GPU STRING GRAPH OK" in p.stdout, p.stdout[-3000:] + p.stderr[-3000:]


@pytest.mark.parametrize("world,grid", [(2, "-"), (2, "2x1"), (4, "2x2")])
@pytest.mark.parametrize("base", [0, 77])
def test_multi_gpu_string_graph(world, grid, base):
    """R is identical on every rank, equals the prune over all ranks' alignments in rank order and (as a set of unordered pairs)
    the one-GPU R; S equals the oracle's transitive reduction of that R."""
    if _ngpus() < world:
        pytest.skip(f"needs {world} GPUs")
    port = 29741 + 10 * world + (0 if grid == "-" else 1) + (2 if base else 0)
    _launch(world, ["reads_fa", 17, 2, 8, grid, base], port)
