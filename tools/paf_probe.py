"""PAF text on the device against the host route, on the same resident alignments and string graph.

    python tools/paf_probe.py [--genome 8000000] [--reads 80000] [--mean 4000] [--upper 40] [--reps 5] [--host-reps 1]

The HiFi-like read set of tools/string_graph_probe.py (elba_b200.synth, generated on the GPU) goes through elba_fe_run,
elba_fe_align, elba_fe_overlap_graph and elba_fe_reduce_overlap_graph once.  Then, --reps times each (rep 0 warms up):
  device:  elba_fe_paf for overlap.paf and for string.paf (its device time, info.ms), then elba_fe_get_paf (the text to a host
           buffer; host clock)
  host:    elba_fe_get_alignments (13 fields per pair to the host) + the formatter of tests/paf_inputs.py (Python), for
           overlap.paf only (--host-reps times)
The two routes' bytes must be identical.  Prints the card's name and power limit with the numbers."""
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
import paf_inputs as PI  # noqa: E402


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
    ap.add_argument("--host-reps", type=int, default=1)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("paf_probe: no CUDA device (the measurement needs a B200)")
    print(f"[probe] card: {card()}", flush=True)
    t0 = time.perf_counter()
    buf, off, lens = synth.make_reads(a.genome, a.reads, a.mean, a.sd, a.err, 313, device="cuda")
    torch.cuda.synchronize()
    hlens = lens.cpu().numpy().astype(np.uint64)
    ctx = frontend.Context(frontend.Params(k=a.k, lower=a.lower, upper=a.upper))
    ctx.set_reads_device(buf.data_ptr(), buf.numel(), off.data_ptr(), lens.data_ptr(), lens.numel(), 0)
    ctx.run()
    P = ctx.align(fetch=False)
    ctx.overlap_graph()
    ctx.string_graph()
    t1 = time.perf_counter()
    print(f"[probe] {a.reads} reads of mean {a.mean} (genome {a.genome}, err {a.err}), k={a.k} L={a.lower} U={a.upper}: aligned pairs={P}; "
          f"generate .. string graph {t1 - t0:.1f} s", flush=True)

    dev = {}
    for which, name in ((frontend.PAF_OVERLAP, "overlap"), (frontend.PAF_STRING, "string")):
        ms, copy, text = [], [], None
        for rep in range(a.reps + 1):
            info = frontend.PafInfo()
            ctx._ck(ctx.L.elba_fe_paf(ctx.h, C.c_int(which), C.byref(info)))
            host = np.empty(max(info.bytes, 1), np.uint8)
            ts = time.perf_counter()
            ctx._ck(ctx.L.elba_fe_get_paf(ctx.h, frontend._p(host)))
            te = time.perf_counter()
            if rep:
                ms.append(info.ms); copy.append(1e3 * (te - ts))
            text = host[:info.bytes].tobytes()
        m, c = float(np.median(ms)), float(np.median(copy))
        dev[name] = text
        print(f"[probe] {name}.paf: {info.lines} lines, {info.bytes} bytes ({info.bytes / max(info.lines, 1):.1f} B/line); elba_fe_paf device "
              f"median {m:.3f} ms (min {min(ms):.3f}, max {max(ms):.3f}) = {info.bytes / m / 1e6:.1f} GB/s of text; get_paf to pageable host "
              f"memory median {c:.2f} ms = {info.bytes / c / 1e6:.1f} GB/s", flush=True)

    rows, cols = np.zeros(P, np.int64), np.zeros(P, np.int64)
    fields = np.zeros((P, 13), np.int32)
    host_ms = []
    for rep in range(a.host_reps):
        ts = time.perf_counter()
        ctx._ck(ctx.L.elba_fe_get_alignments(ctx.h, frontend._p(rows), frontend._p(cols), frontend._p(fields)))
        tg = time.perf_counter()
        text = PI.text(rows, cols, fields, hlens, 0, None)
        te = time.perf_counter()
        host_ms.append((1e3 * (tg - ts), 1e3 * (te - tg)))
        same = text == dev["overlap"]
        print(f"[probe] host route rep {rep}: get_alignments {host_ms[-1][0]:.1f} ms + Python formatter {host_ms[-1][1]:.0f} ms; "
              f"{len(text)} bytes; identical to the device text: {same}", flush=True)
        if not same:
            raise SystemExit("paf_probe: the routes disagree")
    print(f"[probe] card: {card()}", flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
