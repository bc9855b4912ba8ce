"""One rank of the multi-GPU PAF check (launched by torchrun from test_gpu_paf.py, or by hand):

    torchrun --nproc-per-node=N tests/multi_gpu_paf_worker.py <grid RxC or -> <first read id> <output directory>

Step by step on every rank's block of reads (first id nonzero), and then through the driver on a FASTA file: overlap.paf,
string.paf and contigs.fa written by all ranks at their offsets.  Rank 0 then runs the same on one GPU and checks: string.paf
and contigs.fa byte-identical, overlap.paf the same lines (their order follows the grid)."""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from elba_b200 import frontend, distributed as D  # noqa: E402
from elba_b200.assemble import assemble  # noqa: E402
from elba_b200.fasta import write_fasta  # noqa: E402
from elba_b200.synth import make_dnabuffer  # noqa: E402


def chain(ctx, dna, base, names, prefix, d):
    """align -> overlap.paf -> R -> S -> string.paf -> contigs.fa, every file written at the ranks' offsets."""
    ctx.upload(dna, base)
    ctx.set_read_names(names)
    ctx.run()
    ctx.align(fetch=False)
    frontend.write_paf(prefix + ".overlap.paf", ctx, frontend.PAF_OVERLAP, d)
    ctx.overlap_graph()
    ctx.string_graph()
    frontend.write_paf(prefix + ".string.paf", ctx, frontend.PAF_STRING, d)
    cg = ctx.contigs()
    frontend.write_contigs_fa_parallel(prefix + ".contigs.fa", cg.seqs, cg.info["first"], d)


def same(a, b, sort_lines=False):
    x, y = open(a, "rb").read(), open(b, "rb").read()
    if sort_lines:
        x, y = sorted(x.splitlines(True)), sorted(y.splitlines(True))
    return x == y and len(x) > 0


def main():
    grid = tuple(int(x) for x in sys.argv[1].split("x")) if sys.argv[1] != "-" else None
    base, out = int(sys.argv[2]), sys.argv[3]
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dna = make_dnabuffer(genome_len=60_000, n_reads=160, mean_len=6000, sd_len=857, err=0.01, seed=11)
    names = [f"m54/{i}/ccs" for i in range(dna.size())]
    params = frontend.Params(k=31, lower=2, upper=4, device=local)
    fa = os.path.join(out, "reads.fa")
    if rank == 0:
        write_fasta(fa, [dna.read_ascii(i) for i in range(dna.size())], names=names)
    mine, first = D.local_reads(dna, rank, world)
    ctx = frontend.Context(params)
    D.bootstrap_comm(ctx, dist, device=torch.device("cuda", local), grid=grid)
    chain(ctx, mine, first + base, names, os.path.join(out, "multi"), dist)
    ctx.close()
    assemble(fa, os.path.join(out, "drv_multi"), params, dist=dist, grid=grid)
    ok = True
    if rank == 0:
        one = frontend.Context(params)
        chain(one, dna, base, names, os.path.join(out, "single"), None)
        one.close()
        assemble(fa, os.path.join(out, "drv_single"), params)
        for a, b in (("multi", "single"), ("drv_multi", "drv_single")):
            pa, pb = os.path.join(out, a), os.path.join(out, b)
            checks = dict(string=same(pa + ".string.paf", pb + ".string.paf"), contigs=same(pa + ".contigs.fa", pb + ".contigs.fa"),
                          overlap=same(pa + ".overlap.paf", pb + ".overlap.paf", sort_lines=True))
            print(f"{a} vs {b}: {checks}; overlap.paf {os.path.getsize(pa + '.overlap.paf')} B, string.paf "
                  f"{os.path.getsize(pa + '.string.paf')} B, contigs.fa {os.path.getsize(pa + '.contigs.fa')} B", flush=True)
            ok = ok and all(checks.values())
    flags = [None] * world
    dist.all_gather_object(flags, ok)
    if rank == 0 and all(flags):
        print(f"MULTI-GPU PAF OK world={world} grid={sys.argv[1]} base={base} N={dna.size()}", flush=True)
    dist.destroy_process_group()
    sys.exit(0 if all(flags) else 1)


if __name__ == "__main__":
    main()
