"""The contig rule (DESIGN.md §3d, include/elba_fe.h: elba_fe_contigs) restated in Python, and error-free read sets whose contigs
must be exact substrings of the genome they were drawn from.

Entry e = (i, j) of the string graph S: t(e) = (direction >> 1) & 1 is the end of read i the overlap leaves from (0 = 3' end,
1 = 5' start), suffix(e) the bases j adds beyond i."""
import numpy as np

from elba_b200.dnabuffer import DnaBuffer


def _t(f):
    return (f[0] >> 1) & 1


def rule(rows, cols, fields, lens, base=0):
    """S (global ids, any order) and the read lengths (indexed by id - base) -> (contigs, branches, cycles); a contig is a list of
    (global read id, reversed, beg, end) in walk order, contigs in ascending order of their start read."""
    adj = {}
    for r, c, f in zip(np.asarray(rows).tolist(), np.asarray(cols).tolist(), np.asarray(fields).reshape(-1, 4).tolist()):
        adj.setdefault(r, []).append((c, f))
    # 1-2: branches
    branch = {v for v, es in adj.items() if len(es) > 2 or (len(es) == 2 and _t(es[0][1]) == _t(es[1][1]))}
    # 3: the chain graph G, as two slots per read indexed by t; an entry counts only if its mirror is in S
    slot, ent = {}, {}
    for v, es in adj.items():
        if v in branch:
            continue
        for c, f in es:
            if c in branch or not any(cc == v for cc, _ in adj.get(c, ())):
                continue
            slot.setdefault(v, [None, None])[_t(f)] = c
            ent[(v, c)] = f

    def nbrs(v):
        return [c for c in slot.get(v, (None, None)) if c is not None]
    seen, walks, cycles = set(), [], 0
    for v in sorted(slot):
        if v in seen:
            continue
        comp, stack = [], [v]
        seen.add(v)
        while stack:
            u = stack.pop()
            comp.append(u)
            for w in nbrs(u):
                if w not in seen:
                    seen.add(w)
                    stack.append(w)
        if len(comp) < 2:
            continue
        ends = [u for u in comp if len(nbrs(u)) < 2]
        # 4: where the walk starts
        if ends:
            s = min(ends)
            walk, prev, cur = [s], None, s
            while True:
                nxt = [w for w in nbrs(cur) if w != prev]
                if not nxt:
                    break
                prev, cur = cur, nxt[0]
                walk.append(cur)
        else:
            cycles += 1
            s = min(comp)
            walk, prev, cur = [s], s, min(nbrs(s))
            while cur != s:
                walk.append(cur)
                nxt = [w for w in nbrs(cur) if w != prev][0]
                prev, cur = cur, nxt
        walks.append(walk)
    walks.sort(key=lambda w: w[0])                     # 7
    contigs = []
    for walk in walks:
        m = len(walk) - 1
        out = []
        for k, v in enumerate(walk):
            n = int(lens[v - base])
            fwd = _t(ent[(v, walk[k + 1])]) == 0 if k < m else _t(ent[(v, walk[k - 1])]) == 1      # 5
            b, e = 0, n
            if k:                                                                                   # 6
                s = min(max(ent[(walk[k - 1], v)][2], 0), n)
                b, e = (n - s, n) if fwd else (0, s)
            out.append((v, not fwd, b, e))
        contigs.append(out)
    return contigs, len(branch), cycles


def layout(contigs):
    """The arrays of elba_fe_get_contig_layout: ptr, read, reverse, beg, end."""
    ptr = np.zeros(len(contigs) + 1, np.uint64)
    ptr[1:] = np.cumsum([len(c) for c in contigs]) if contigs else []
    flat = [x for c in contigs for x in c]
    return (ptr, np.array([x[0] for x in flat], np.int64), np.array([x[1] for x in flat], np.uint8),
            np.array([x[2] for x in flat], np.uint32), np.array([x[3] for x in flat], np.uint32))


def sequences(contigs, dna: DnaBuffer, base=0):
    """2-bit codes of every contig: the segments concatenated, a reversed one reverse-complemented (3 - c, in reverse order)."""
    out = []
    for c in contigs:
        parts = []
        for v, rev, b, e in c:
            x = dna.read_codes(v - base)[b:e]
            parts.append((3 - x[::-1]) if rev else x)
        out.append(np.concatenate(parts).astype(np.uint8) if parts else np.zeros(0, np.uint8))
    return out


def error_free_reads(seed, genome_len=60_000, n_reads=200, lo=3000, hi=6000, circular=False):
    """Reads of random length in [lo, hi] from a random genome g on random strands, without errors; circular: drawn from g + g
    (they may wrap around).  -> (DnaBuffer, g as codes)."""
    rng = np.random.default_rng(seed)
    g = rng.integers(0, 4, genome_len).astype(np.uint8)
    src = np.concatenate([g, g]) if circular else g
    reads = []
    for _ in range(n_reads):
        n = int(rng.integers(lo, hi + 1))
        p = int(rng.integers(0, genome_len if circular else genome_len - n + 1))
        x = src[p:p + n]
        reads.append(3 - x[::-1] if rng.integers(0, 2) else x)
    lens = np.array([len(r) for r in reads], np.int64)
    return DnaBuffer.from_codes(np.concatenate(reads), lens), g


def is_substring(codes, g, circular=False):
    """codes (or its reverse complement) occurs in g (circular: in g + g + g)."""
    hay = (np.concatenate([g, g, g]) if circular else g).tobytes()
    return codes.tobytes() in hay or (3 - codes[::-1]).astype(np.uint8).tobytes() in hay
