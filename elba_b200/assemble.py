"""From a FASTA file to ELBA's three outputs, `<prefix>.overlap.paf`, `<prefix>.string.paf` and `<prefix>.contigs.fa`
(src/main.cpp:303,317,332-345), on one GPU or on several (one process per GPU under torchrun):

    python -m elba_b200.assemble reads.fa -k 31 -l 15 -u 35 -o prefix [--xdrop 15 --mat 1 --mis -1 --gap -1 --fuzz 1000]
    torchrun --nproc-per-node=4 -m elba_b200.assemble reads.fa -k 31 -l 15 -u 35 -o prefix [--grid 2x2]

The FASTA needs its .fai next to it (samtools faidx).  Every stage runs on the device: FASTA ingest, counting, A and B, X-drop
alignment, the prunes to the overlap graph R, transitive reduction to the string graph S, contigs and the PAF text.  What
reaches the host is the text of the files, which every rank writes at its own offset of one shared file.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

from . import frontend
from .fasta import FastaIndex


def assemble(fasta: str, prefix: str, params: frontend.Params, scoring=(1, -1, -1, 15), fuzz: int = 1000, dist=None, grid=None) -> dict:
    """Run the whole chain on `fasta` and write the three files; collective over `dist` (an initialised torch.distributed with
    one process per GPU; params.device = this process' GPU) when given.  scoring = (mat, mis, gap, xdrop).  Returns the
    sizes and the device time of every stage (this rank's)."""
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist is not None else (0, 1)
    ctx = frontend.Context(params)
    try:
        if dist is not None:
            import torch
            from .distributed import bootstrap_comm
            bootstrap_comm(ctx, dist, device=torch.device("cuda", params.device), grid=grid)
        fi = FastaIndex(fasta, rank, world)
        fi.getmydna(ctx, fetch=False)
        ctx.set_read_names(fi.rootnames)
        ctx.run()
        npairs = ctx.align(*scoring, fetch=False)
        ov = frontend.write_paf(prefix + ".overlap.paf", ctx, frontend.PAF_OVERLAP, dist)
        R = ctx.overlap_graph()
        S = ctx.string_graph(fuzz)
        sg = frontend.write_paf(prefix + ".string.paf", ctx, frontend.PAF_STRING, dist)
        cg = ctx.contigs()
        frontend.write_contigs_fa_parallel(prefix + ".contigs.fa", cg.seqs, cg.info["first"], dist)
        tm = ctx.timings()
        return dict(reads=fi.gettotrecords(), pairs=npairs, R=len(R[0]), contained=R[5], S=len(S[0]), contigs=cg.info["ncontigs"],
                    contig_bases=cg.info["bases"], overlap_paf_lines=ov["total_lines"], overlap_paf_bytes=ov["total_bytes"],
                    string_paf_lines=sg["total_lines"], string_paf_bytes=sg["total_bytes"],
                    ms=dict(ingest=tm["upload_ms"], count=tm["count_ms"], build_A=tm["build_ms"], spgemm=tm["spgemm_ms"],
                            align=tm["align_ms"], overlap_paf=ov["ms"], overlap_graph=tm["overlap_ms"], string_graph=tm["transitive_ms"],
                            string_paf=sg["ms"], contigs=cg.info["ms"]))
    finally:
        ctx.close()


def main(argv=None):
    ap = argparse.ArgumentParser(prog="python -m elba_b200.assemble", description=__doc__.split("\n\n")[0])
    ap.add_argument("fasta", help="reads; the .fai index must sit next to it")
    ap.add_argument("-k", type=int, default=31, help="k-mer length (default 31)")
    ap.add_argument("-l", "--lower", type=int, default=15, help="lowest count of a reliable k-mer (default 15)")
    ap.add_argument("-u", "--upper", type=int, default=35, help="highest count of a reliable k-mer (default 35)")
    ap.add_argument("-o", "--prefix", required=True, help="output prefix: <prefix>.overlap.paf, .string.paf, .contigs.fa")
    ap.add_argument("--xdrop", type=int, default=15, help="X-drop cut-off (default 15)")
    ap.add_argument("--mat", type=int, default=1, help="match score (default 1)")
    ap.add_argument("--mis", type=int, default=-1, help="mismatch score (default -1)")
    ap.add_argument("--gap", type=int, default=-1, help="gap score (default -1)")
    ap.add_argument("--fuzz", type=int, default=1000, help="transitive-reduction fuzz (default 1000)")
    ap.add_argument("--grid", default=None, help="process grid RxC on several GPUs (default: the most square)")
    a = ap.parse_args(argv)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    dist, device = None, 0
    if world > 1:
        import torch
        import torch.distributed as dist
        device = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(device)
        dist.init_process_group("nccl", device_id=torch.device("cuda", device))
    grid = tuple(int(x) for x in a.grid.split("x")) if a.grid else None
    params = frontend.Params(k=a.k, lower=a.lower, upper=a.upper, device=device)
    try:
        out = assemble(a.fasta, a.prefix, params, (a.mat, a.mis, a.gap, a.xdrop), a.fuzz, dist=dist, grid=grid)
        if dist is None or dist.get_rank() == 0:
            print(json.dumps(out), flush=True)
    finally:
        if dist is not None:
            dist.destroy_process_group()


if __name__ == "__main__":
    sys.exit(main())
