"""One rank of the multi-GPU contig check (launched by torchrun from test_gpu_contigs.py, or by hand): every rank runs the
chain to the string graph S on its block of reads, then elba_fe_contigs (no collective).  Checks: the same layout on every
rank, equal to the rule of tests/contig_inputs.py on the rank's S; the ranks' sequences, concatenated in rank order, are the
rule's."""
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
import contig_inputs as CI  # noqa: E402


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
    ctx.align(1, -1, -1, 15)
    ctx.overlap_graph()
    rows, cols, f, _, _ = ctx.string_graph()
    got = ctx.contigs()
    h = hashlib.sha256()
    for a in (got.ptr, got.read, got.reverse, got.beg, got.end):
        h.update(np.ascontiguousarray(a).tobytes())
    mine_out = dict(digest=h.hexdigest(), first=got.info["first"], seqs=[got.seqs.read_codes(i) for i in range(got.seqs.size())])
    everyone = [None] * world
    dist.all_gather_object(everyone, mine_out)
    ok = True
    try:
        assert len({e["digest"] for e in everyone}) == 1, "the layout differs between the ranks"
        contigs, branches, cycles = CI.rule(rows, cols, f, dna.lengths, base)
        for a, b, name in zip((got.ptr, got.read, got.reverse, got.beg, got.end), CI.layout(contigs), ("ptr", "read", "reverse", "beg", "end")):
            assert np.array_equal(a, b), ("layout vs the rule", name)
        assert (got.info["branches"], got.info["cycles"]) == (branches, cycles)
        want = CI.sequences(contigs, dna, base)
        seqs = [s for e in everyone for s in e["seqs"]]
        assert [e["first"] for e in everyone] == sorted(e["first"] for e in everyone)
        assert len(seqs) == len(want) and all(np.array_equal(a, b) for a, b in zip(seqs, want)), "sequences vs the rule"
        print(f"rank {rank}: S={len(rows)} contigs={len(contigs)} mine={got.info['count']} bases={got.info['bases']} "
              f"ms={got.info['ms']:.3f}", flush=True)
    except AssertionError as e:
        import traceback
        traceback.print_exc()
        print(f"rank {rank}: MULTI-GPU CONTIGS FAILED", e, flush=True)
        ok = False
    flags = [None] * world
    dist.all_gather_object(flags, ok)
    if rank == 0 and all(flags):
        print(f"MULTI-GPU CONTIGS OK world={world} grid={sys.argv[5] if len(sys.argv) > 5 else '-'} base={base} N={dna.size()}", flush=True)
    ctx.close()
    dist.destroy_process_group()
    sys.exit(0 if all(flags) else 1)


if __name__ == "__main__":
    main()
