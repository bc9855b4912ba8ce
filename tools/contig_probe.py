"""From the resident string graph S to contigs: the device route against the host route, on the same S and reads.

    python tools/contig_probe.py [--genome 8000000] [--reads 80000] [--mean 4000] [--upper 40] [--reps 5]

One synthetic HiFi-like read set (elba_b200.synth, generated on the GPU; the defaults of tools/string_graph_probe.py) goes
through elba_fe_run, elba_fe_align, elba_fe_overlap_graph and elba_fe_reduce_overlap_graph once.  Then each route runs --reps
times (host clock; every call ends in a stream synchronise):
  resident: elba_fe_contigs (layout and sequences on the device; only scalars cross PCIe)
  host:     S and the whole read arena to the host (elba_fe_get_string_graph, elba_fe_get_reads), then the rule of
            tests/contig_inputs.py in Python
The device contigs are fetched outside the timed region; layout and sequences of both routes must be identical.  Prints the
card's name and power limit with the numbers."""
import argparse
import ctypes as C
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from elba_b200 import frontend, synth  # noqa: E402
import contig_inputs as CI  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return q.stdout.strip()
    except Exception as e:      # nvidia-smi missing: the name at least
        return f"{torch.cuda.get_device_name()} (nvidia-smi: {e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--genome", type=int, default=8_000_000)
    ap.add_argument("--reads", type=int, default=80_000)
    ap.add_argument("--mean", type=int, default=4000)
    ap.add_argument("--sd", type=int, default=500)
    ap.add_argument("--err", type=float, default=0.01)
    ap.add_argument("--k", type=int, default=31)
    ap.add_argument("--lower", type=int, default=2)
    ap.add_argument("--upper", type=int, default=40)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("contig_probe: no CUDA device (the measurement needs a B200)")
    print(f"[probe] card: {card()}", flush=True)
    t0 = time.perf_counter()
    buf, off, lens = synth.make_reads(a.genome, a.reads, a.mean, a.sd, a.err, 313, device="cuda")
    torch.cuda.synchronize()
    ctx = frontend.Context(frontend.Params(k=a.k, lower=a.lower, upper=a.upper))
    ctx.set_reads_device(buf.data_ptr(), buf.numel(), off.data_ptr(), lens.data_ptr(), lens.numel(), 0)
    ctx.run()
    npairs, nR, nC, nS = C.c_uint64(), C.c_uint64(), C.c_uint64(), C.c_uint64()
    ctx._ck(ctx.L.elba_fe_align(ctx.h, 1, -1, -1, 15, C.byref(npairs)))
    ctx._ck(ctx.L.elba_fe_overlap_graph(ctx.h, C.byref(nR), C.byref(nC)))
    ctx._ck(ctx.L.elba_fe_reduce_overlap_graph(ctx.h, C.c_int32(1000), C.byref(nS)))
    t1 = time.perf_counter()
    print(f"[probe] {a.reads} reads of mean {a.mean} (genome {a.genome}, err {a.err}), k={a.k} L={a.lower} U={a.upper}: aligned pairs={npairs.value} "
          f"R={nR.value} S={nS.value}; generate + run + align + string graph {t1 - t0:.1f} s", flush=True)
    m = nS.value
    info = frontend.ContigInfo()

    def resident():
        ctx._ck(ctx.L.elba_fe_contigs(ctx.h, C.byref(info)))

    def host():
        S = (np.zeros(m, np.int64), np.zeros(m, np.int64), np.zeros((m, 4), np.int32))
        ctx._ck(ctx.L.elba_fe_get_string_graph(ctx.h, *[frontend._p(x) for x in S], None, None))
        dna = ctx.reads()
        contigs, branches, cycles = CI.rule(*S, dna.lengths)
        return contigs, CI.sequences(contigs, dna), branches, cycles

    times = {"resident": [], "host": []}
    dev = []
    for rep in range(a.reps + 1):                      # rep 0 warms both routes up and is not counted
        torch.cuda.synchronize()
        ts = time.perf_counter(); resident(); te = time.perf_counter()
        got = ctx._contigs_result(info)
        hs = time.perf_counter(); contigs, seqs, branches, cycles = host(); he = time.perf_counter()
        same = all(np.array_equal(x, y) for x, y in zip((got.ptr, got.read, got.reverse, got.beg, got.end), CI.layout(contigs)))
        same = same and (got.info["branches"], got.info["cycles"]) == (branches, cycles) and got.seqs.size() == len(seqs)
        same = same and all(np.array_equal(got.seqs.read_codes(i), s) for i, s in enumerate(seqs))
        if not same:
            raise SystemExit(f"contig_probe: the routes disagree (contigs {got.info['ncontigs']} vs {len(contigs)})")
        if rep:
            times["resident"].append(1e3 * (te - ts)); times["host"].append(1e3 * (he - hs)); dev.append(got.info["ms"])
        lens_ = np.array([len(s) for s in seqs])
        print(f"[probe] rep {rep}{' (warm-up)' if not rep else ''}: resident {1e3 * (te - ts):.2f} ms (device {got.info['ms']:.3f}), host {1e3 * (he - hs):.0f} ms; "
              f"contigs={got.info['ncontigs']} reads in contigs={got.info['contig_reads']} bases={got.info['bases']} branches={branches} cycles={cycles} "
              f"longest={lens_.max() if len(lens_) else 0} mean={lens_.mean() if len(lens_) else 0:.0f}; layout and sequences identical", flush=True)
    med = {k: float(np.median(v)) for k, v in times.items()}
    print(f"[probe] median of {a.reps}: resident {med['resident']:.2f} ms (device {np.median(dev):.3f} ms), host {med['host']:.0f} ms, "
          f"host / resident = {med['host'] / med['resident']:.0f}x; S={m} contigs={info.ncontigs}; card: {card()}", flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
