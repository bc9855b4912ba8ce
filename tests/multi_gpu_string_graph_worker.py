"""One rank of the multi-GPU string-graph check (launched by torchrun from test_gpu_string_graph.py, or by hand):
every rank runs the front end and the X-drop alignment on its block of reads, builds the overlap graph R on the device
(collective) and reduces it to the string graph S.  Every rank checks its own R and S."""
import hashlib
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from elba_b200 import frontend, distributed as D  # noqa: E402
from elba_b200.dnabuffer import DnaBuffer  # noqa: E402
from test_gpu_string_graph import TR_COLS, prune  # noqa: E402
import tr_inputs  # noqa: E402


def main():
    fixture, k, lo, up = sys.argv[1], int(sys.argv[2]), int(sys.argv[3]), int(sys.argv[4])
    grid = tuple(int(x) for x in sys.argv[5].split("x")) if len(sys.argv) > 5 and sys.argv[5] != "-" else None
    base = int(sys.argv[6]) if len(sys.argv) > 6 else 0      # global id of the first read of rank 0
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dna = DnaBuffer.load(os.path.join(ROOT, "tests", "golden", fixture + ".npz"))
    mine, first = D.local_reads(dna, rank, world)
    ctx = frontend.Context(frontend.Params(k=k, lower=lo, upper=up, device=local))
    D.bootstrap_comm(ctx, dist, device=torch.device("cuda", local), grid=grid)
    ctx.upload(mine, first + base)
    ctx.run()
    aligned = ctx.align(1, -1, -1, 15)
    rows, cols, f, src_rank, src_pair, ncont = ctx.overlap_graph()
    S = ctx.string_graph()
    h = hashlib.sha256()
    for a in (rows, cols, f, src_rank, src_pair):
        h.update(np.ascontiguousarray(a).tobytes())
    mine_out = dict(aligned=aligned, digest=h.hexdigest())
    everyone = [None] * world
    dist.all_gather_object(everyone, mine_out)
    ok = True
    try:
        assert len({e["digest"] for e in everyone}) == 1, "R differs between the ranks"
        # R = the prune over all ranks' alignments, concatenated in rank order
        ar = np.concatenate([e["aligned"][0] for e in everyone]); ac = np.concatenate([e["aligned"][1] for e in everyone])
        af = np.concatenate([e["aligned"][2] for e in everyone])
        ranks = np.concatenate([np.full(len(e["aligned"][0]), r, np.int32) for r, e in enumerate(everyone)])
        local_idx = np.concatenate([np.arange(len(e["aligned"][0]), dtype=np.uint64) for e in everyone])
        idx, C = prune(ar, ac, af)
        assert np.array_equal(rows, ar[idx]) and np.array_equal(cols, ac[idx]) and np.array_equal(f, af[idx][:, TR_COLS]), "R vs the prune"
        assert np.array_equal(src_rank, ranks[idx]) and np.array_equal(src_pair, local_idx[idx]), "source of R's entries"
        assert ncont == len(C), (ncont, len(C))
        # the same unordered pairs as the one-GPU R (square grids may orient a pair the other way)
        n, er, ec, ef = tr_inputs.overlap_graph(dna, k, lo, up)
        got = sorted((min(int(r), int(c)), max(int(r), int(c))) for r, c in zip(rows - base, cols - base))
        want = sorted((int(r), int(c)) for r, c in zip(er, ec))
        assert got == want, ("pairs of R vs one GPU", len(got), len(want))
        if grid is not None and grid[0] != grid[1]:
            assert (rows < cols).all()
        # S = the oracle's transitive reduction of this R
        from oracle import oracle as O
        wantS = O.transitive_reduction(base + dna.size(), rows, cols, f)
        for a, b, name in zip(S, wantS, ("row", "col", "fields", "src", "transposed")):
            assert np.array_equal(a, b), ("S", name, len(a), len(b))
        assert len(rows) > 0 and len(S[0]) > 0
        print(f"rank {rank}: R={len(rows)} C={ncont} S={len(S[0])} overlap_ms={ctx.timings()['overlap_ms']:.3f}", flush=True)
    except AssertionError as e:
        import traceback
        traceback.print_exc()
        print(f"rank {rank}: MULTI-GPU STRING GRAPH FAILED", e, flush=True)
        ok = False
    flags = [None] * world
    dist.all_gather_object(flags, ok)
    if rank == 0 and all(flags):
        print(f"MULTI-GPU STRING GRAPH OK world={world} grid={sys.argv[5] if len(sys.argv) > 5 else '-'} base={base} N={dna.size()}", flush=True)
    ctx.close()
    dist.destroy_process_group()
    sys.exit(0 if all(flags) else 1)


if __name__ == "__main__":
    main()
