"""The PAF format of elba_fe_paf (DESIGN.md §3d, include/elba_fe.h) restated in Python: the text the device must write, byte
for byte.  One line per alignment, 13 tab-separated columns:

    qname qlen begQ endQ strand tname tlen begT endT score max(endQ - begQ, endT - begT) 255 dr:i:<direction>

q = the alignment's row read, t = its column read, strand '-' iff rc; a read's name is names[id - base], or its global id in
decimal without names."""
import numpy as np

BEG_Q, END_Q, BEG_T, END_T, SCORE, RC, DIR = 0, 1, 2, 3, 4, 5, 9


def _name(r, names, base):
    if names is None:
        return str(r).encode()
    n = names[r - base]
    return n.encode() if isinstance(n, str) else bytes(n)


def lines(rows, cols, fields, lens, base=0, names=None):
    """The PAF lines (bytes, '\\n' included) of alignments (global row / column ids, fields[n, 13] as elba_fe_get_alignments
    returns them); lens[r - base] = bases of read r; names[r - base] = its name, or None for decimal ids."""
    out = []
    f = np.asarray(fields).reshape(-1, 13).tolist()
    for q, t, a in zip(np.asarray(rows).tolist(), np.asarray(cols).tolist(), f):
        block = max(a[END_Q] - a[BEG_Q], a[END_T] - a[BEG_T])
        cols_ = [_name(q, names, base), b"%d" % int(lens[q - base]), b"%d" % a[BEG_Q], b"%d" % a[END_Q], b"-" if a[RC] else b"+",
                 _name(t, names, base), b"%d" % int(lens[t - base]), b"%d" % a[BEG_T], b"%d" % a[END_T], b"%d" % a[SCORE],
                 b"%d" % block, b"255", b"dr:i:%d" % a[DIR]]
        out.append(b"\t".join(cols_) + b"\n")
    return out


def text(rows, cols, fields, lens, base=0, names=None) -> bytes:
    return b"".join(lines(rows, cols, fields, lens, base, names))


def string_lines(transposed, src, src_rank, src_pair):
    """The lines of string.paf as (rank, alignment index on that rank): the entries of S with transposed == 0 in S's order,
    each followed through src into R (src_rank / src_pair of elba_fe_get_overlap_graph)."""
    out = []
    for tr, s in zip(np.asarray(transposed).tolist(), np.asarray(src).tolist()):
        if tr == 0:
            out.append((int(src_rank[s]), int(src_pair[s])))
    return out


def string_text(S, R, alignments, lens, base=0, names=None) -> bytes:
    """string.paf from S = (rows, cols, fields, src, transposed), R = (rows, cols, fields, src_rank, src_pair, ...) and
    alignments[rank] = (rows, cols, fields[n, 13]) of every rank."""
    pick = string_lines(S[4], S[3], R[3], R[4])
    rows = np.array([alignments[r][0][p] for r, p in pick], np.int64)
    cols = np.array([alignments[r][1][p] for r, p in pick], np.int64)
    f = np.array([alignments[r][2][p] for r, p in pick], np.int32).reshape(-1, 13)
    return text(rows, cols, f, lens, base, names)
