"""The contig rule of tests/contig_inputs.py on hand-built string graphs, and on the error-free oracle chain (reads -> overlap
graph -> transitive reduction -> contigs), where every contig must be an exact substring of the genome.  CPU only: these pin
the rule the device is checked against in test_gpu_contigs.py."""
import numpy as np
import pytest

import contig_inputs as CI
import tr_inputs
from elba_b200.dnabuffer import DnaBuffer


def swap(d):
    return ((d & 1) << 1) | (d >> 1)


def sym(edges):
    """edges (i, j, direction of (i, j), suffix of (i, j), suffix of (j, i)) -> S with both orientations, row-major."""
    ent = []
    for i, j, d, s, sT in edges:
        ent.append((i, j, [d, swap(d), s, sT]))
        ent.append((j, i, [swap(d), d, sT, s]))
    ent.sort(key=lambda x: (x[0], x[1]))
    return (np.array([e[0] for e in ent], np.int64), np.array([e[1] for e in ent], np.int64),
            np.array([e[2] for e in ent], np.int32).reshape(-1, 4))


def rc(x):
    return (3 - x[::-1]).astype(np.uint8)


G = np.random.default_rng(0).integers(0, 4, 30).astype(np.uint8)
PIECES = ((0, 12), (8, 20), (15, 30))          # consecutive overlaps of 4 and 5 bases: suffixes 8 and 10


def test_forward_path():
    dna = DnaBuffer.from_codes(np.concatenate([G[a:b] for a, b in PIECES]), [b - a for a, b in PIECES])
    rows, cols, f = sym([(0, 1, 1, 8, 4), (1, 2, 1, 10, 5)])         # leave i's 3' end, enter j's 5' start
    contigs, branches, cycles = CI.rule(rows, cols, f, dna.lengths)
    assert contigs == [[(0, False, 0, 12), (1, False, 4, 12), (2, False, 5, 15)]] and branches == 0 and cycles == 0
    assert np.array_equal(CI.sequences(contigs, dna)[0], G)


def test_reversed_path():
    """Every read stored reverse-complemented: the overlaps leave through the 5' starts, every read is reversed, the contig is G."""
    dna = DnaBuffer.from_codes(np.concatenate([rc(G[a:b]) for a, b in PIECES]), [b - a for a, b in PIECES])
    rows, cols, f = sym([(0, 1, 2, 8, 4), (1, 2, 2, 10, 5)])
    contigs, _, _ = CI.rule(rows, cols, f, dna.lengths)
    assert contigs == [[(0, True, 0, 12), (1, True, 0, 8), (2, True, 0, 10)]]
    assert np.array_equal(CI.sequences(contigs, dna)[0], G)


def test_nonzero_base():
    dna = DnaBuffer.from_codes(np.concatenate([G[a:b] for a, b in PIECES]), [b - a for a, b in PIECES])
    rows, cols, f = sym([(0, 1, 1, 8, 4), (1, 2, 1, 10, 5)])
    contigs, _, _ = CI.rule(rows + 500, cols + 500, f, dna.lengths, base=500)
    assert [x[0] for x in contigs[0]] == [500, 501, 502]
    assert np.array_equal(CI.sequences(contigs, dna, base=500)[0], G)


def test_degree3_branch_splits_a_path():
    lens = np.full(6, 100, np.uint64)
    rows, cols, f = sym([(0, 1, 1, 10, 10), (1, 2, 1, 10, 10), (2, 3, 1, 10, 10), (3, 4, 1, 10, 10), (2, 5, 1, 20, 20)])
    contigs, branches, cycles = CI.rule(rows, cols, f, lens)
    assert [[x[0] for x in c] for c in contigs] == [[0, 1], [3, 4]]        # read 5 alone: its only neighbour is a branch
    assert branches == 1 and cycles == 0


def test_same_end_branch():
    """Read 2 has two entries, both leaving from its 3' end: no walk passes through it."""
    lens = np.full(5, 100, np.uint64)
    rows, cols, f = sym([(0, 1, 1, 10, 10), (2, 1, 0, 10, 10), (2, 3, 1, 10, 10), (3, 4, 1, 10, 10)])
    contigs, branches, _ = CI.rule(rows, cols, f, lens)
    assert [[x[0] for x in c] for c in contigs] == [[0, 1], [3, 4]] and branches == 1
    assert contigs[0] == [(0, False, 0, 100), (1, False, 90, 100)]      # 0's 3' end overlaps 1's 5' start: both forward


def test_cycle():
    """Four reads around a circular genome of 40 bases, ids 0, 3, 1, 2 in genome order: the walk starts at 0 and goes first to
    the smaller of its neighbours 3 and 2, i.e. against the genome; the edge 0 - 3 is cut."""
    g = np.random.default_rng(1).integers(0, 4, 40).astype(np.uint8)
    gg = np.concatenate([g, g])
    order = [0, 3, 1, 2]
    reads = {rid: gg[10 * k: 10 * k + 15] for k, rid in enumerate(order)}
    dna = DnaBuffer.from_codes(np.concatenate([reads[i] for i in range(4)]), [15] * 4)
    rows, cols, f = sym([(order[k], order[(k + 1) % 4], 1, 10, 10) for k in range(4)])
    contigs, branches, cycles = CI.rule(rows, cols, f, dna.lengths)
    assert [x[0] for x in contigs[0]] == [0, 2, 1, 3] and all(x[1] for x in contigs[0]) and cycles == 1 and branches == 0
    s = CI.sequences(contigs, dna)[0]
    assert len(s) == 45 and CI.is_substring(s, g, circular=True)


def test_suffix_clamped():
    lens = np.array([12, 12, 12], np.uint64)
    rows, cols, f = sym([(0, 1, 1, -5, 3), (1, 2, 1, 100, 3)])
    contigs, _, _ = CI.rule(rows, cols, f, lens)
    assert contigs == [[(0, False, 0, 12), (1, False, 12, 12), (2, False, 0, 12)]]


def test_empty_graph():
    z = np.zeros(0, np.int64)
    assert CI.rule(z, z, np.zeros((0, 4), np.int32), np.zeros(3, np.uint64)) == ([], 0, 0)
    ptr, read, rev, beg, end = CI.layout([])
    assert list(ptr) == [0] and len(read) == 0


@pytest.mark.parametrize("circular", [False, True])
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_error_free_oracle_chain(seed, circular):
    """Error-free reads through the CPU oracle (overlap graph, transitive reduction) and the rule: one contig, an exact substring
    of the genome (linear) or of g + g + g (circular, a cut cycle)."""
    from oracle import oracle as O
    dna, g = CI.error_free_reads(seed, circular=circular)
    n, r, c, f = tr_inputs.overlap_graph(dna, 31, 2, 100)
    S = O.transitive_reduction(n, r, c, f)
    contigs, branches, cycles = CI.rule(S[0], S[1], S[2], dna.lengths)
    seqs = CI.sequences(contigs, dna)
    assert len(contigs) == 1 and cycles == (1 if circular else 0) and branches == 0
    assert len(seqs[0]) > 0.95 * len(g) and CI.is_substring(seqs[0], g, circular)


def test_write_contigs_fa(tmp_path):
    from elba_b200.frontend import write_contigs_fa
    seqs = DnaBuffer.from_strings(["ACGTTGCA", "", "GGGAC"])
    p = tmp_path / "x.contigs.fa"
    write_contigs_fa(str(p), seqs, first=5)
    assert p.read_text() == ">contig_5\nACGTTGCA\n>contig_6\n\n>contig_7\nGGGAC\n"
