"""Contigs on the device (elba_fe_contigs, elba_fe_contigs_from_graph) against the rule of tests/contig_inputs.py: the layout and
the sequences must be exactly the rule's, on the resident string graph of real and synthetic read sets, on random bidirected
graphs given from the host, and on error-free reads where every contig is an exact substring of the genome."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import contig_inputs as CI

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def _ctx(k, lo, up):
    from elba_b200 import frontend
    return frontend.Context(frontend.Params(k=k, lower=lo, upper=up, device=0))


def check(got, rows, cols, fields, dna, base, what):
    """got (frontend.Contigs) == the rule on S over dna (ids from base): layout, totals, sequences of the block."""
    contigs, branches, cycles = CI.rule(rows, cols, fields, dna.lengths, base)
    for a, b, name in zip((got.ptr, got.read, got.reverse, got.beg, got.end), CI.layout(contigs), ("ptr", "read", "reverse", "beg", "end")):
        assert np.array_equal(a, b), (what, name, len(a), len(b))
    seqs = CI.sequences(contigs, dna, base)
    i = got.info
    assert (i["ncontigs"], i["contig_reads"], i["bases"], i["branches"], i["cycles"]) == \
        (len(contigs), int(got.ptr[-1]), sum(len(s) for s in seqs), branches, cycles), (what, i)
    first, count = i["first"], i["count"]
    assert got.seqs.size() == count and i["my_bases"] == sum(len(s) for s in seqs[first:first + count]), (what, i)
    assert i["my_bytes"] == sum((len(s) + 3) // 4 for s in seqs[first:first + count]), (what, i)
    for c in range(count):
        assert np.array_equal(got.seqs.read_codes(c), seqs[first + c]), (what, "sequence", first + c)
    return contigs


def _resident(ctx, dna, base, scoring):
    ctx.upload(dna, base)
    ctx.run()
    ctx.align(*scoring)
    ctx.overlap_graph()
    S = ctx.string_graph()
    return S, ctx.contigs()


@pytest.mark.parametrize("kind,k,lo,up,scoring,base", [
    ("reads_fa", 17, 2, 8, (1, -1, -1, 15), 0),
    ("reads_fa", 17, 2, 8, (1, -1, -1, 15), 4321),
    ("clr", 17, 2, 8, (2, -3, -2, 25), 77),
    ("hifi", 31, 2, 4, (1, -1, -1, 15), 1000),
])
def test_resident_vs_rule(kind, k, lo, up, scoring, base, fixtures):
    from elba_b200.synth import make_dnabuffer
    if kind == "reads_fa":
        dna = fixtures("reads_fa")
    else:
        dna = make_dnabuffer(genome_len=60_000, n_reads=160, mean_len=6000, sd_len=857, err=0.12 if kind == "clr" else 0.01, seed=11)
    ctx = _ctx(k, lo, up)
    (rows, cols, f, _, _), got = _resident(ctx, dna, base, scoring)
    contigs = check(got, rows, cols, f, dna, base, (kind, base))
    if kind == "hifi":
        assert len(contigs) > 0
    assert got.info["ms"] > 0
    # the same S given from the host (shuffled: the call sorts it) gives the same contigs
    p = np.random.default_rng(1).permutation(len(rows))
    check(ctx.contigs_from_graph(rows[p], cols[p], f[p]), rows, cols, f, dna, base, (kind, base, "from_graph"))
    ctx.close()


@pytest.mark.parametrize("circular", [False, True])
def test_error_free_genome_substrings(circular):
    dna, g = CI.error_free_reads(2, circular=circular)
    ctx = _ctx(31, 2, 100)
    (rows, cols, f, _, _), got = _resident(ctx, dna, 500, (1, -1, -1, 15))
    check(got, rows, cols, f, dna, 500, circular)
    assert got.info["ncontigs"] == 1 and got.info["cycles"] == (1 if circular else 0)
    s = got.seqs.read_codes(0)
    assert len(s) > 0.95 * len(g) and CI.is_substring(s, g, circular)
    ctx.close()


def _random_graph(rng, n):
    """A symmetric bidirected graph on n reads: a few random paths and cycles (long chains) plus random extra edges (branches);
    mirror entry = the two bits of direction swapped, suffix <-> suffixT."""
    perm = rng.permutation(n)
    pairs, i = set(), 0
    while i < n - 1:
        L = int(rng.integers(2, max(3, n // 3)))
        chain = perm[i:i + L].tolist()
        pairs |= {(min(a, b), max(a, b)) for a, b in zip(chain, chain[1:])}
        if len(chain) > 2 and rng.random() < 0.4:
            pairs.add((min(chain[0], chain[-1]), max(chain[0], chain[-1])))
        i += L
    for _ in range(int(rng.integers(0, n // 4 + 1))):
        a, b = rng.integers(0, n, 2).tolist()
        if a != b:
            pairs.add((min(a, b), max(a, b)))
    rows, cols, f = [], [], []
    for a, b in sorted(pairs):
        d = int(rng.integers(0, 4)); dT = ((d & 1) << 1) | (d >> 1)
        s, sT = rng.integers(-20, 120, 2).tolist()
        rows += [a, b]; cols += [b, a]; f += [[d, dT, s, sT], [dT, d, sT, s]]
    return np.array(rows, np.int64), np.array(cols, np.int64), np.array(f, np.int32).reshape(-1, 4)


def test_random_graphs_from_graph():
    from elba_b200.dnabuffer import DnaBuffer
    rng = np.random.default_rng(7)
    ctx = _ctx(17, 2, 8)
    cycles = branches = 0
    for it in range(200):
        n = int(rng.integers(1, 60))
        lens = rng.integers(0, 100, n)
        dna = DnaBuffer.from_codes(rng.integers(0, 4, int(lens.sum())).astype(np.uint8), lens)
        base = int(rng.choice([0, 1000, 123456789]))
        ctx.upload(dna, base)
        rows, cols, f = _random_graph(rng, n)
        got = ctx.contigs_from_graph(rows + base, cols + base, f)
        check(got, rows + base, cols + base, f, dna, base, it)
        cycles += got.info["cycles"]; branches += got.info["branches"]
    assert cycles > 0 and branches > 0
    ctx.close()


def test_state_errors():
    from elba_b200 import frontend
    from elba_b200.synth import make_dnabuffer
    dna = make_dnabuffer(genome_len=60_000, n_reads=160, mean_len=6000, sd_len=857, err=0.01, seed=11)
    ctx = _ctx(31, 2, 4)
    L, h = ctx.L, ctx.h

    def getters():
        return (L.elba_fe_get_contig_layout(h, None, None, None, None, None), L.elba_fe_get_contigs(h, None, None, None),
                L.elba_fe_device_contigs(h, None, None, None))
    assert getters() == (-5, -5, -5)
    with pytest.raises(frontend.FrontEndError):
        ctx.contigs()                                  # nothing resident
    S, first = _resident(ctx, dna, 9, (1, -1, -1, 15))
    assert getters() == (0, 0, 0)
    # a host-route reduction overwrites S: no contigs from it, and the old ones are gone
    ctx.transitive_reduction(9 + dna.size(), S[0], S[1], S[2])
    assert getters() == (-5, -5, -5)
    with pytest.raises(frontend.FrontEndError):
        ctx.contigs()
    ctx.string_graph()
    again = ctx.contigs()
    assert np.array_equal(again.read, first.read) and np.array_equal(again.seqs.buf, first.seqs.buf)
    # a new R discards S's contigs
    ctx.overlap_graph()
    assert getters() == (-5, -5, -5)
    with pytest.raises(frontend.FrontEndError):
        ctx.contigs()
    ctx.string_graph()
    ctx.contigs()
    # reads uploaded again after align: the arena is not the one S was built from
    ctx.upload(dna, 9)
    assert getters() == (-5, -5, -5)
    with pytest.raises(frontend.FrontEndError):
        ctx.contigs()
    # host S: validation
    r, c, f = np.array([9, 10], np.int64), np.array([10, 9], np.int64), np.array([[1, 2, 5, 5], [2, 1, 5, 5]], np.int32)
    ctx.contigs_from_graph(r, c, f)
    for bad in ((r[:1], c[:1], f[:1]),                                    # not symmetric
                (np.array([9]), np.array([9]), f[:1]),                    # diagonal
                (r - 1, c - 1, f),                                        # id below read_id_offset
                (r + dna.size(), c + dna.size(), f),                      # id past the reads
                (r, c, np.array([[4, 2, 5, 5], [2, 1, 5, 5]], np.int32)),    # direction 4
                (np.concatenate([r, r]), np.concatenate([c, c]), np.concatenate([f, f]))):   # repeated coordinates
        with pytest.raises(frontend.FrontEndError):
            ctx.contigs_from_graph(*bad)
    ctx.close()


def test_device_handoff():
    """The contigs' device arrays go straight into set_reads_device of a second context and read back equal."""
    from elba_b200.synth import make_dnabuffer
    dna = make_dnabuffer(genome_len=60_000, n_reads=160, mean_len=6000, sd_len=857, err=0.01, seed=11)
    ctx = _ctx(31, 2, 4)
    _, got = _resident(ctx, dna, 0, (1, -1, -1, 15))
    assert got.seqs.size() > 0
    p, o, l = C.c_void_p(), C.c_void_p(), C.c_void_p()
    ctx._ck(ctx.L.elba_fe_device_contigs(ctx.h, C.byref(p), C.byref(o), C.byref(l)))
    ctx2 = _ctx(31, 2, 4)
    ctx2.set_reads_device(p.value, got.info["my_bytes"], o.value, l.value, got.info["count"], 0)
    back = ctx2.reads()
    assert np.array_equal(back.lengths, got.seqs.lengths) and np.array_equal(back.offsets, got.seqs.offsets)
    assert np.array_equal(back.buf, got.seqs.buf)
    ctx2.close()
    ctx.close()


# ---- several GPUs ----------------------------------------------------------------------------------------------------
def _ngpus():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.parametrize("world,grid", [(2, "-"), (2, "2x1"), (4, "2x2")])
@pytest.mark.parametrize("base", [0, 77])
def test_multi_gpu_contigs(world, grid, base):
    """Every rank holds the same layout, equal to the rule on its S; the ranks' sequences in rank order are the rule's."""
    if _ngpus() < world:
        pytest.skip(f"needs {world} GPUs")
    port = 29841 + 10 * world + (0 if grid == "-" else 1) + (2 if base else 0)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(HERE, "multi_gpu_contigs_worker.py"), "reads_fa", "17", "2", "8", grid, str(base)]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0 and "MULTI-GPU CONTIGS OK" in p.stdout, p.stdout[-3000:] + p.stderr[-3000:]
