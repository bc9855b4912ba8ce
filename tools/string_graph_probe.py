"""From resident alignments to the string graph S: the device route against the host route, on the same alignments.

    python tools/string_graph_probe.py [--genome 8000000] [--reads 80000] [--mean 4000] [--upper 40] [--reps 5]

One synthetic HiFi-like read set (elba_b200.synth, generated on the GPU) goes through elba_fe_run and elba_fe_align once.
Then, from the same resident alignments, each route runs --reps times (host clock; every call ends in a stream synchronise):
  resident: elba_fe_overlap_graph + elba_fe_reduce_overlap_graph (only scalars cross PCIe)
  host:     elba_fe_get_alignments (13 fields per pair to the host) + the prune in numpy + elba_fe_transitive_reduction
            (host validation, R back to the device)
Both leave S on the device; it is fetched outside the timed region and the two must be identical.  Prints the card's
name and power limit with the numbers."""
import argparse
import ctypes as C
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
from elba_b200 import frontend, synth  # noqa: E402

PASSED, CONT_Q, CONT_T = 6, 7, 8


def host_prune(rows, cols, fields):
    passed = fields[:, PASSED] != 0
    C_ = np.union1d(rows[passed & (fields[:, CONT_Q] != 0)], cols[passed & (fields[:, CONT_T] != 0)])
    keep = passed & ~np.isin(rows, C_) & ~np.isin(cols, C_)
    return rows[keep], cols[keep], np.ascontiguousarray(fields[keep][:, 9:13]), len(C_)


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
        raise SystemExit("string_graph_probe: no CUDA device (the measurement needs a B200)")
    print(f"[probe] card: {card()}", flush=True)
    t0 = time.perf_counter()
    buf, off, lens = synth.make_reads(a.genome, a.reads, a.mean, a.sd, a.err, 313, device="cuda")
    torch.cuda.synchronize()
    ctx = frontend.Context(frontend.Params(k=a.k, lower=a.lower, upper=a.upper))
    ctx.set_reads_device(buf.data_ptr(), buf.numel(), off.data_ptr(), lens.data_ptr(), lens.numel(), 0)
    ctx.run()
    t1 = time.perf_counter()
    npairs = C.c_uint64()
    ctx._ck(ctx.L.elba_fe_align(ctx.h, 1, -1, -1, 15, C.byref(npairs)))
    t2 = time.perf_counter()
    P = npairs.value
    print(f"[probe] {a.reads} reads of mean {a.mean} (genome {a.genome}, err {a.err}), k={a.k} L={a.lower} U={a.upper}: nnzB={ctx.sizes()['nnzB']} "
          f"aligned pairs={P}; generate + run {t1 - t0:.1f} s, align {t2 - t1:.1f} s", flush=True)

    rows, cols = np.zeros(P, np.int64), np.zeros(P, np.int64)
    fields = np.zeros((P, 13), np.int32)
    nR, nC, nS = C.c_uint64(), C.c_uint64(), C.c_uint64()

    def resident():
        ctx._ck(ctx.L.elba_fe_overlap_graph(ctx.h, C.byref(nR), C.byref(nC)))
        ctx._ck(ctx.L.elba_fe_reduce_overlap_graph(ctx.h, C.c_int32(1000), C.byref(nS)))

    def host():
        ctx._ck(ctx.L.elba_fe_get_alignments(ctx.h, frontend._p(rows), frontend._p(cols), frontend._p(fields)))
        r, c, f, nc = host_prune(rows, cols, fields)
        ctx._ck(ctx.L.elba_fe_transitive_reduction(ctx.h, frontend._p(r) if len(r) else None, frontend._p(c) if len(r) else None,
                                                   frontend._p(f) if len(r) else None, C.c_uint64(len(r)), C.c_int64(a.reads), C.c_int32(1000), C.byref(nS)))
        return len(r), nc

    def fetch_S():
        m = nS.value
        out = (np.zeros(m, np.int64), np.zeros(m, np.int64), np.zeros((m, 4), np.int32), np.zeros(m, np.uint64), np.zeros(m, np.uint8))
        ctx._ck(ctx.L.elba_fe_get_string_graph(ctx.h, *[frontend._p(x) for x in out]))
        return out

    times = {"resident": [], "host": []}
    dev = {"overlap_ms": [], "transitive_ms": []}
    for rep in range(a.reps + 1):                      # rep 0 warms both routes up and is not counted
        torch.cuda.synchronize()
        ts = time.perf_counter(); resident(); te = time.perf_counter()
        tm = ctx.timings()
        S_res = fetch_S()
        nR_res, nC_res = nR.value, nC.value
        torch.cuda.synchronize()
        hs = time.perf_counter(); nR_host, nC_host = host(); he = time.perf_counter()
        S_host = fetch_S()
        same = nR_res == nR_host and nC_res == nC_host and all(np.array_equal(x, y) for x, y in zip(S_res, S_host))
        if not same:
            raise SystemExit(f"string_graph_probe: the routes disagree (R {nR_res} vs {nR_host}, C {nC_res} vs {nC_host}, S {len(S_res[0])} vs {len(S_host[0])})")
        if rep:
            times["resident"].append(1e3 * (te - ts)); times["host"].append(1e3 * (he - hs))
            dev["overlap_ms"].append(tm["overlap_ms"]); dev["transitive_ms"].append(tm["transitive_ms"])
        print(f"[probe] rep {rep}{' (warm-up)' if not rep else ''}: resident {1e3 * (te - ts):.2f} ms (device: overlap {tm['overlap_ms']:.2f} + "
              f"reduction {tm['transitive_ms']:.2f}), host {1e3 * (he - hs):.2f} ms; R={nR_res} contained={nC_res} S={len(S_res[0])}; S identical", flush=True)
    med = {k: float(np.median(v)) for k, v in times.items()}
    print(f"[probe] median of {a.reps}: resident {med['resident']:.2f} ms (device overlap {np.median(dev['overlap_ms']):.2f} + reduction "
          f"{np.median(dev['transitive_ms']):.2f}), host {med['host']:.2f} ms, host / resident = {med['host'] / med['resident']:.1f}x; "
          f"pairs={P} R={nR.value} S={nS.value}; card: {card()}", flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
