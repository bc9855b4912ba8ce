"""The PAF format (tests/paf_inputs.py, the restatement of elba_fe_paf) on hand-built alignments, the choice of string-graph
lines, read-name validation and the command line of the driver; none of it needs a GPU."""
import os
import subprocess
import sys

import numpy as np
import pytest

import paf_inputs as PI

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _aln(*rows):
    """13-field alignments from (begQ, endQ, begT, endT, score, rc, direction)."""
    f = np.zeros((len(rows), 13), np.int32)
    for i, (bq, eq, bt, et, sc, rc, d) in enumerate(rows):
        f[i, [0, 1, 2, 3, 4, 5, 9]] = (bq, eq, bt, et, sc, rc, d)
        f[i, 6] = d != -1
    return f


def test_lines_by_hand():
    lens = np.array([5000, 4200, 3100], np.uint32)
    f = _aln((10, 4000, 0, 3990, 3900, 0, 1), (0, 1500, 2000, 3600, -7, 1, -1))
    got = PI.lines(np.array([100, 101]), np.array([101, 102]), f, lens, base=100)
    assert got == [b"100\t5000\t10\t4000\t+\t101\t4200\t0\t3990\t3900\t3990\t255\tdr:i:1\n",
                   b"101\t4200\t0\t1500\t-\t102\t3100\t2000\t3600\t-7\t1600\t255\tdr:i:-1\n"]
    named = PI.lines(np.array([100, 101]), np.array([101, 102]), f, lens, base=100, names=["a", b"read/2", "c_3"])
    assert named[0].startswith(b"a\t5000\t") and b"\tread/2\t4200\t" in named[0]
    assert named[1].startswith(b"read/2\t4200\t") and b"\tc_3\t3100\t" in named[1]


def test_block_length_takes_the_longer_side():
    lens = np.array([9000, 9000], np.uint32)
    a = PI.lines([0], [1], _aln((100, 200, 0, 900, 5, 0, 2)), lens)[0].split(b"\t")
    b = PI.lines([0], [1], _aln((0, 800, 100, 200, 5, 0, 2)), lens)[0].split(b"\t")
    assert a[10] == b"900" and b[10] == b"800"


def test_paf_columns_parse():
    """12 mandatory PAF columns with integers where PAF has them, the 13th a SAM-style tag; one line per alignment."""
    rng = np.random.default_rng(3)
    n, N = 200, 50
    lens = rng.integers(1, 20000, N).astype(np.uint32)
    rows, cols = rng.integers(7, 7 + N, n), rng.integers(7, 7 + N, n)
    f = np.zeros((n, 13), np.int32)
    f[:, :6] = np.stack([rng.integers(-5, 9000, n), rng.integers(-5, 9000, n), rng.integers(-5, 9000, n), rng.integers(-5, 9000, n),
                         rng.integers(-2**31, 2**31 - 1, n), rng.integers(0, 2, n)], 1)
    f[:, 9] = rng.integers(-1, 4, n)
    t = PI.text(rows, cols, f, lens, base=7)
    assert t.endswith(b"\n") and t.count(b"\n") == n
    for line, r, c, a in zip(t.decode().splitlines(), rows, cols, f):
        x = line.split("\t")
        assert len(x) == 13
        assert (x[0], x[5]) == (str(r), str(c)) and x[4] in "+-" and (x[4] == "-") == bool(a[5])
        assert [int(x[i]) for i in (1, 2, 3, 6, 7, 8, 9, 10, 11)] == \
            [lens[r - 7], a[0], a[1], lens[c - 7], a[2], a[3], a[4], max(int(a[1]) - int(a[0]), int(a[3]) - int(a[2])), 255]
        assert x[12] == f"dr:i:{a[9]}"


def test_string_lines_follow_src():
    # S: 5 entries, two of them mirrors; R: 3 entries from two ranks
    transposed = np.array([0, 1, 0, 1, 0], np.uint8)
    src = np.array([2, 2, 0, 1, 1], np.uint64)
    src_rank, src_pair = np.array([0, 1, 1], np.int32), np.array([4, 0, 3], np.uint64)
    assert PI.string_lines(transposed, src, src_rank, src_pair) == [(1, 3), (0, 4), (1, 0)]
    # and the text is printed from those alignments
    al = {0: (np.arange(5) + 10, np.arange(5) + 20, _aln(*[(i, i + 1, i, i + 2, i, 0, 1) for i in range(5)])),
          1: (np.arange(4) + 30, np.arange(4) + 40, _aln(*[(i, i + 3, i, i + 1, i, 1, 2) for i in range(4)]))}
    S = (None, None, None, src, transposed)
    R = (None, None, None, src_rank, src_pair)
    lens = np.full(60, 1000, np.uint32)
    got = PI.string_text(S, R, al, lens)
    assert got.splitlines()[0].split(b"\t")[:2] == [b"33", b"1000"] and got.splitlines()[1].startswith(b"14\t")
    assert PI.string_text((None, None, None, src[:0], transposed[:0]), R, al, lens) == b""


def test_read_names_checked():
    from elba_b200 import frontend
    assert frontend.check_read_names(["a", b"r/1", "x" * 2000]) == [b"a", b"r/1", b"x" * 2000]
    for bad in (["a", ""], ["a b"], ["a\tb"], ["x\n"], [b"\x01"], ["\x7f ok"]):
        with pytest.raises(ValueError):
            frontend.check_read_names(bad)


def test_assemble_help():
    p = subprocess.run([sys.executable, "-m", "elba_b200.assemble", "--help"], capture_output=True, text=True, cwd=ROOT, timeout=300)
    assert p.returncode == 0 and "--prefix" in p.stdout and "--xdrop" in p.stdout


def test_assemble_without_device(tmp_path):
    import torch
    from elba_b200 import frontend
    from elba_b200.assemble import assemble
    from elba_b200.fasta import write_fasta
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    fa = str(tmp_path / "r.fa")
    write_fasta(fa, ["ACGT" * 50, "TTGCA" * 40], names=["r1", "r2"])
    with pytest.raises(frontend.FrontEndError) as e:
        assemble(fa, str(tmp_path / "out"), frontend.Params(k=17, lower=2, upper=8))
    assert "no CUDA device" in str(e.value) or "-2" in str(e.value)
    assert not os.path.exists(str(tmp_path / "out.overlap.paf"))
