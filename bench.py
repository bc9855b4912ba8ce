#!/usr/bin/env python
"""Benchmark of the ELBA overlap-detection front end (k-mer count -> A -> A*A^T SpGEMM) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic reads:
  value  reads/s with the packed reads already resident in HBM when the timed region starts
  e2e    reads/s through the C ABI with HOST (pinned) buffers: H2D of the reads and D2H of B inside the timed region
One JSON line on stdout (rank 0).  See DESIGN.md "Measurement" for the roofline accounting.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# stdout carries ONE JSON line: whatever NCCL logs (its version banner under NCCL_DEBUG=VERSION, for one) goes to stderr
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

import numpy as np  # noqa: E402
import torch  # noqa: E402

# BASELINE.json configs: 2 = example_medium (fixture), 3 = E. coli 30X CLR, 4 = C. elegans 40X HiFi, 5 = human 10X CLR
WORKLOADS = {
    "example_medium_k17": dict(fixture="example_medium", k=17, lower=2, upper=8, desc="BASELINE configs[1]: example_medium/reads.fa k=17 L=2 U=8"),
    "ecoli30x_clr": dict(shape="ecoli30x_clr", desc="BASELINE configs[2]: synthetic E. coli 30X CLR, 16,890 reads, k=17 U=8"),
    "celegans40x_hifi": dict(shape="celegans40x_hifi", desc="BASELINE configs[3]: synthetic C. elegans 40X HiFi shape, 275,699 reads, k=31 U=4"),
    "human10x_clr": dict(shape="human10x_clr", desc="BASELINE configs[4]: synthetic human 10X CLR shape, 4,421,593 reads, k=17 U=4"),
}
DEFAULT_WORKLOAD = "celegans40x_hifi"     # the config BASELINE.json quotes at 1/2/4/8 GPUs; fits one B200
METRIC = "reads/s through k-mer count + A*A^T SpGEMM"


def ncu_traffic(workload: str):
    """DRAM bytes per launch of the counting chain's kernels from the committed `ncu --set full` capture of this workload
    (profiles/traffic.json, written by tools/ncu_traffic.py from dram__bytes_read.sum + dram__bytes_write.sum); None if absent."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)
        return t.get(workload)
    except Exception:
        return None


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region."""

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index), "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [int(r[0]) for r in self.rows if r and r[0].isdigit()]
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": int(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


def load_workload(name: str, rank: int, world: int, device, scale: float = 1.0):
    """Returns (buf uint8, off int64, lens int64) torch tensors on `device` for THIS rank's contiguous block of reads
    plus (k, lower, upper, total_reads, read_id_offset)."""
    from elba_b200.dnabuffer import DnaBuffer
    from elba_b200 import synth
    w = WORKLOADS[name]
    if "fixture" in w:
        dna = DnaBuffer.load(os.path.join(ROOT, "tests", "golden", w["fixture"] + ".npz"))
        k, lo, up = w["k"], w["lower"], w["upper"]
        total = dna.size()
        r0, r1 = total * rank // world, total * (rank + 1) // world
        d = dna.slice(r0, r1)
        return (torch.from_numpy(d.buf).to(device), torch.from_numpy(d.offsets.astype(np.int64)).to(device),
                torch.from_numpy(d.lengths.astype(np.int64)).to(device), k, lo, up, total, r0)
    s = synth.SHAPES[w["shape"]]
    genome, reads = int(s["genome"] * scale), int(s["reads"] * scale)
    r0, r1 = reads * rank // world, reads * (rank + 1) // world
    buf, off, lens = synth.make_reads_block(genome, reads, s["mean"], s["sd"], s["err"], 313, device, r0, r1)
    return buf, off, lens, s["k"], s["lower"], s["upper"], reads, r0


def check_digests(workload: str, scale: float, input_digest: str, digests: dict, digests_e2e: dict) -> str:
    """The timed result against tests/golden/bench_digests.json (pinned by tests/test_gpu_fullscale.py: the CPU oracle where it
    can run the workload, N = 1 == N = 8 everywhere).  A mismatch makes the number invalid: say so loudly."""
    if digests != digests_e2e:
        print("bench.py: INVALID RUN: the resident and the end-to-end passes disagree: " + json.dumps([digests, digests_e2e]), file=sys.stderr, flush=True)
        return "MISMATCH between the resident and the end-to-end pass"
    try:
        with open(os.path.join(ROOT, "tests", "golden", "bench_digests.json")) as f:
            gold = json.load(f).get(f"{workload}@{scale:g}")
    except Exception:
        gold = None
    if not gold:
        return "no golden for this workload/scale"
    if gold.get("input_digest") != input_digest:
        print(f"bench.py: INVALID RUN: input digest {input_digest} != golden {gold.get('input_digest')}", file=sys.stderr, flush=True)
        return "MISMATCH: the generated input differs from the golden input"
    if {a: gold.get(a) for a in digests} != digests:
        print("bench.py: INVALID RUN: result digests differ from tests/golden/bench_digests.json: " + json.dumps(digests), file=sys.stderr, flush=True)
        return "MISMATCH: results differ from the golden digests"
    return "match (" + gold.get("pinned_by", "golden") + ")"


# share of a synthetic workload the CPU arms run (the reference's own code needs minutes per 10^9 k-mer instances):
# config 3 in full (the same reads the GPU arm times), config 4 at 10 %, config 5 at 0.4 %
CPU_SAMPLE = {"ecoli30x_clr": 1.0, "celegans40x_hifi": 0.10, "human10x_clr": 0.004}


def cpu_reference_sample(name: str, frac: float | None = None):
    """The input of the CPU leg: (DnaBuffer, k, lower, upper, description, same_as_gpu_arm).  frac = 1: the very reads the GPU
    arm times (same generator, same seeds); frac < 1: the same shape (coverage, read length, error rate) over a genome and a
    read count both scaled by frac.  Generated on the GPU when there is one (seconds instead of minutes)."""
    from elba_b200.dnabuffer import DnaBuffer
    from elba_b200 import synth
    w = WORKLOADS[name]
    if "fixture" in w:
        dna = DnaBuffer.load(os.path.join(ROOT, "tests", "golden", w["fixture"] + ".npz"))
        return dna, w["k"], w["lower"], w["upper"], f"all {dna.size()} reads of {w['fixture']}", True
    s = synth.SHAPES[w["shape"]]
    if frac is None:
        # the sample that takes a 16-thread host 10-20 s per pass; fewer host threads get a proportionally smaller one,
        # so that W + K passes of the reference arm still end within a few minutes
        frac = CPU_SAMPLE.get(w["shape"], 0.05)
        if frac < 1.0:
            frac = max(frac * min(1.0, square_ranks()[0] / 16.0), 0.01)
    genome, reads = max(int(s["genome"] * frac), 100_000), max(int(s["reads"] * frac), 64)
    dev = torch.device("cuda", 0) if torch.cuda.is_available() else torch.device("cpu")
    buf, off, lens = synth.make_reads_block(genome, reads, s["mean"], s["sd"], s["err"], 313, dev, 0, reads)
    dna = synth.to_dnabuffer(buf, off, lens)
    del buf, off, lens
    if frac >= 1.0:
        desc = f"all {reads} reads of the workload (the same reads the GPU arm times)"
    else:
        desc = f"{reads} reads over a {genome} bp genome: the {w['shape']} shape (same coverage, read length, error rate) scaled by {frac:.4g}"
    return dna, s["k"], s["lower"], s["upper"], desc, frac >= 1.0 and dev.type == "cuda"


def run_cpu_reference(dna, k, lo, up, ranks: int):
    """One pass of the reference's own CPU implementation (oracle/_ref when built for this (k,L,U), else the oracle port)."""
    from oracle import oracle as O
    t = time.perf_counter()
    if O.ref_available(k, lo, up):
        r = O.ref_run(dna, k, lo, up, nranks=ranks, fetch=False)
        kind, cores, secs = "reference", ranks, r.secs
    else:
        r = O.run(dna, k, lo, up, threads=ranks)
        kind, cores, secs = "port", 1, r.secs
    dt = time.perf_counter() - t
    return dna.size() / dt, kind, cores, {a: float(b) for a, b in secs.items()}


DUMP_SAMPLE = 1 << 18       # entries kept of each large output: at most 2^18 x (3 + 3 + 7) float64 values, 27 MB in all
DUMP_SIZES = ("nreads", "num_kmers", "distinct", "reliable", "nnzA_pre", "nnzA", "products", "nnzB_pre", "nnzB")


def _sample(n: int, m: int) -> np.ndarray:
    """Sorted indices of a fixed, seeded sample of m out of n entries (all of them when n <= m)."""
    if n <= m:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, m, replace=False))


def dump_outputs(ctx, out_dir: str, sizes: dict, rank: int, world: int, r0: int):
    """Write what the last resident step (the timed value) returned to its caller as float64 .npy files under out_dir,
    so that two builds can be compared output for output.  Called on every rank: on several GPUs ctx.kmers() is
    collective (the super-k-mer path all-gathers the list from its owners).  The files:
      sizes.npy   the whole-job sizes of DUMP_SIZES
      kmers.npy   [value >> 32, value & 0xffffffff, count] of the reliable k-mers (float64 is exact below 2^53 only)
      A.npy       [read, k-mer column, position] of A's entries
      B.npy       [row read, column read, numshared, s0.q, s0.t, s1.q, s1.t] of B's entries
    Global read ids; A and B row-major, k-mers ascending.  Large outputs are sampled by _sample, the same entry indices
    for the same sizes.  On several GPUs every rank writes its own block of A and B (file names end in .rank<r>), and
    each rank keeps a 1/world share of the sample."""
    os.makedirs(out_dir, exist_ok=True)
    m = DUMP_SAMPLE // world
    tag = "" if world == 1 else f".rank{rank}"

    def save(name, cols):
        np.save(os.path.join(out_dir, name + ".npy"), np.stack([np.asarray(c, np.float64) for c in cols], axis=1))

    kmers, counts = ctx.kmers()             # the whole list on every rank
    if rank == 0:
        np.save(os.path.join(out_dir, "sizes.npy"), np.array([sizes[a] for a in DUMP_SIZES], np.float64))
        i = _sample(len(kmers), m)
        save("kmers", (kmers[i] >> np.uint64(32), kmers[i] & np.uint64(0xFFFFFFFF), counts[i]))
    rp, col, pos = ctx.A()                  # the rows of this rank's reads, global column ids
    i = _sample(len(col), m)
    save("A" + tag, (np.searchsorted(rp, i, side="right") - 1 + r0, col[i], pos[i]))
    rp, col, num, seeds = ctx.B()           # this rank's block of B, local row / column ids
    info = ctx.comm_info()
    i = _sample(len(col), m)
    save("B" + tag, (np.searchsorted(rp, i, side="right") - 1 + info["row0"], col[i].astype(np.int64) + info["col0"], num[i], *seeds[i].T))


def square_ranks():
    cores = os.cpu_count() or 1
    q = int(np.floor(np.sqrt(min(cores, 64))))
    return max(1, q * q), cores


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--partitions", type=int, default=0)
    ap.add_argument("--scale", type=float, default=1.0, help="shrink a synthetic workload (debug only; the JSON says so)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed resident steps, write a sample of what the last one computed as .npy files")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    w = WORKLOADS[args.workload]

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        dna, k, lo, up, sample, same = cpu_reference_sample(args.workload)
        ranks, cores = square_ranks()
        times = []
        for i in range(args.warmup + args.steps):
            rps, kind, used, secs = run_cpu_reference(dna, k, lo, up, ranks)
            if i >= args.warmup:
                times.append(dna.size() / rps)
        ms = 1000.0 * float(np.mean(times)) if times else float("nan")
        val = dna.size() / (ms / 1000.0)
        line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "reads/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
                "config": {"workload": args.workload, "desc": w["desc"], "k": k, "lower": lo, "upper": up},
                "same_input_as_gpu_arm": same,
                "cpu_baseline": {"value": val, "unit": "reads/s", "cores": used, "kind": kind, "host_cores": cores,
                                 "sample": sample + "; reference KmerOps.cpp/SharedSeeds.cpp compiled unmodified, MPI ranks emulated as threads, CombBLAS restated (oracle/stubs)",
                                 "stage_secs": secs},
                "e2e": {"value": val, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        print(json.dumps(line), flush=True)
        return

    # ------------------------------------------------------------------ our arm (B200)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from elba_b200 import frontend

    buf, off, lens, k, lo, up, total_reads, r0 = load_workload(args.workload, rank, world, dev, args.scale)
    nreads = lens.numel()
    M = int((lens - k + 1).clamp(min=0).sum().item())
    # what is being timed: a digest of the input that does not depend on how the reads are split over the GPUs
    from elba_b200 import synth as _synth
    nbytes_all = torch.tensor([buf.numel() if r == rank else 0 for r in range(world)], device=dev, dtype=torch.int64)
    if world > 1:
        dist.all_reduce(nbytes_all)
    din = _synth.input_digest_parts(buf, lens, int(nbytes_all[:rank].sum().item()), r0)
    din_t = torch.tensor([x - (1 << 64) if x >= (1 << 63) else x for x in din], device=dev, dtype=torch.int64)
    if world > 1:
        dist.all_reduce(din_t)            # int64 sums wrap mod 2^64
    input_digest = "".join(f"{int(x) & 0xFFFFFFFFFFFFFFFF:016x}" for x in din_t.tolist())
    # host (pinned) copies for the end-to-end leg
    hbuf, hoff, hlen = (t.cpu().pin_memory() for t in (buf, off, lens))
    torch.cuda.synchronize()

    ctx = frontend.Context(frontend.Params(k=k, lower=lo, upper=up, device=local, num_partitions=args.partitions))
    # run the library on torch's current stream so that torch CUDA events bracket its kernels
    ctx.set_stream(torch.cuda.current_stream().cuda_stream)
    if world > 1:
        from elba_b200 import distributed as D
        D.bootstrap_comm(ctx, dist, device=dev)      # the library's own NCCL communicator (k-mer all-to-all, panel all-gather)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def step_resident():
        ctx.set_reads_device(buf.data_ptr(), buf.numel(), off.data_ptr(), lens.data_ptr(), nreads, r0)
        ctx.run()

    out_host = {}

    def step_e2e():
        ctx.upload_raw(hbuf.data_ptr(), hbuf.numel(), hoff.data_ptr(), hlen.data_ptr(), nreads, r0)
        ctx.run()
        s = ctx.sizes()
        n = s["nnzB"]
        if out_host.get("cap", -1) < n:
            out_host["rp"] = torch.empty(ctx.comm_info()["nrows"] + 1, dtype=torch.int64).pin_memory()
            out_host["col"] = torch.empty(max(n, 1), dtype=torch.int32).pin_memory()
            out_host["num"] = torch.empty(max(n, 1), dtype=torch.int32).pin_memory()
            out_host["seeds"] = torch.empty(max(n, 1) * 4, dtype=torch.int32).pin_memory()
            out_host["cap"] = n
        import ctypes as C
        ctx._ck(ctx.L.elba_fe_get_B(ctx.h, C.c_void_p(out_host["rp"].data_ptr()), C.c_void_p(out_host["col"].data_ptr()),
                                    C.c_void_p(out_host["num"].data_ptr()), C.c_void_p(out_host["seeds"].data_ptr())))
        return s

    def timed(fn, steps, warmup):
        import gc
        for _ in range(warmup):
            fn()
        gc.collect()
        gc.disable()            # a generation-2 collection of the interpreter on one rank stalls every rank at the next collective
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ctx.reset_timings()
        acc = {}
        e0.record()
        for _ in range(steps):
            fn()
            for a, b in ctx.timings().items():
                acc[a] = acc.get(a, 0.0) + b
        e1.record()
        barrier()
        gc.enable()
        ms = torch.tensor([e0.elapsed_time(e1) / steps], device=dev, dtype=torch.float64)   # device time, CUDA events on the launching stream
        if dist is not None:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), {a: b / steps for a, b in acc.items()}

    # one sampler for the job (rank 0's GPU): eight nvidia-smi loops on one box were seen to stall kernel launches for tens of ms
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ms_res, tm = timed(step_resident, args.steps, args.warmup)
    clocks = sampler.stop() if sampler else None
    sizes_local = ctx.sizes()
    sizes = ctx.sizes_global()              # whole-job totals (collective)
    digests = ctx.digests()                 # whole-job result digests of the last timed pass (collective)
    if args.dump_outputs:
        dump_outputs(ctx, args.dump_outputs, sizes, rank, world, r0)
    ms_e2e, tm_e2e = timed(step_e2e, args.steps, 1)
    sizes_e2e = ctx.sizes()
    digests_e2e = ctx.digests()
    info = ctx.comm_info()

    # per-phase device times: the slowest rank
    keys = sorted(a for a in tm if a.endswith("_ms"))
    tvec = torch.tensor([tm[a] for a in keys], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(tvec, op=dist.ReduceOp.MAX)
    tm.update({a: float(v) for a, v in zip(keys, tvec.tolist())})
    io = torch.tensor([hbuf.numel() + 16 * nreads, 8 * (info["nrows"] + 1) + 24 * sizes_e2e["nnzB"]], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(io)
    tot_reads, tot_M, tot_nnzA, tot_F, tot_nnzB_pre, tot_nnzB, tot_R = [float(sizes[a]) for a in ("nreads", "num_kmers", "nnzA", "products", "nnzB_pre", "nnzB", "reliable")]
    M = int(tot_M)

    if rank == 0:
        peak, peak_src = measured_peaks()
        # counting = everything the reference does in get_kmer_count_map_keys/values: our count phase + the seed-emission sweep
        t_count = (tm["count_ms"] + tm["lookup_ms"]) / 1000.0
        bytes_count = 28.5 * M / world              # SURVEY.md §8(d): 8 + 20 + 2*0.25 bytes per k-mer instance; per GPU
        ach = bytes_count / t_count / 1e9 if t_count > 0 else 0.0
        t_sp = tm["spgemm_kernel_ms"] / 1000.0
        bytes_sp = 8.0 * sizes_local["products"] + 8.0 * sizes_local["nnzA"] + 28.0 * sizes_local["nnzB_pre"]      # rank 0's block
        ach_sp = bytes_sp / t_sp / 1e9 if t_sp > 0 else 0.0
        Mg = max(M / world, 1)
        skm = sizes["table_slots"] == 2048 and k >= 20       # the super-k-mer path ran (superkmer.cuh, skm_count.cuh)
        names = (("k_skm_scatter", "k_skm_count4", "k_seed_keys") if skm else ("k_scatter1", "k_scatter2+k_count_buckets", "k_probe_filter+k_resolve"))
        chain = (("k_skm_scatter (own reads) -> k_skm_forward (records into the owners' slabs through peer memory) -> " if world > 1 else "k_skm_scatter -> ") +
                 "k_skm_count4 (bulk-copied slabs, pass 2 fused: reliable list + seed list) -> radix sort of the reliable k-mers, k_rank_finish" +
                 (" / k_rank_global" if world > 1 else "") + " -> k_seed_keys" if skm else
                 "k_scatter1 -> k_scatter2 -> k_count_buckets -> k_unmix, radix sort, k_lookup_build -> k_probe_filter -> k_resolve")
        kt = {names[0]: tm["partition_ms"], names[1]: tm["count_kernel_ms"], names[2]: tm["lookup_ms"]}
        if world > 1:
            kt["k_skm_forward + fill words" if skm else "all-to-all"] = tm.get("exchange_ms", 0.0)
        kt["rest (column ids: sort + rank, fallback for spilled buckets, host)"] = max(0.0, 1000.0 * t_count - sum(kt.values()))
        traffic = ncu_traffic(args.workload) if world == 1 and args.scale == 1.0 else None
        roofline = {"bound": "hbm", "kernel": "counting chain per GPU = everything the reference does in get_kmer_count_map_keys/values: " + chain,
                    "dominant_kernel": max(kt, key=kt.get), "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "traffic": (traffic or {}).get("chain_dram_bytes"), "traffic_source": (traffic or {}).get("source"), "traffic_per_kernel": (traffic or {}).get("kernels"),
                    "peak_source": peak_src, "algorithmic_bytes": bytes_count, "algorithmic_bytes_per_instance": 28.5, "seconds": t_count,
                    "kernels_ms": {a: round(b, 4) for a, b in kt.items()},
                    "kernels_share_of_step": {a: round(b / ms_res, 4) for a, b in kt.items()},
                    "kernels_ps_per_instance": {a: 1e9 * b / Mg for a, b in kt.items()},
                    "budget_ps_per_instance_at_50pct": 1e12 * 28.5 / (0.5 * peak * 1e9)}
        line = {
            "metric": METRIC, "value": tot_reads / (ms_res / 1000.0), "unit": "reads/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_res, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64", "data": "synthetic" if "shape" in w else "reference fixture",
            "config": {"workload": args.workload, "desc": w["desc"] + (f" (scaled x{args.scale})" if args.scale != 1.0 else ""), "k": k, "lower": lo, "upper": up,
                       "reads": int(tot_reads), "kmer_instances": int(tot_M), "reliable_kmers": int(tot_R), "nnzA": int(tot_nnzA), "products": int(tot_F),
                       "nnzB": int(tot_nnzB), "partitions": sizes["partitions"], "grid": f"{info['grid_rows']}x{info['grid_cols']}", "l2_policy": "inputs larger than L2 / every step rewrites count tables and partition buffers",
                       "timing": "CUDA events on the launching stream around K steps, max over ranks; per-phase numbers from the library's own CUDA events on the same stream"},
            "input_digest": input_digest, "digests": digests, "digest_check": check_digests(args.workload, args.scale, input_digest, digests, digests_e2e),
            "phases_ms": {a: round(b, 4) for a, b in tm.items() if a.endswith("_ms")},
            "roofline": roofline,
            "roofline_spgemm": {"bound": "hbm", "kernel": "k_sp2_expand + k_sp2_warp + k_sp2_block (rank 0's block of B)", "achieved": ach_sp, "peak": peak, "unit": "GB/s", "frac": ach_sp / peak,
                                "algorithmic_bytes": bytes_sp, "algorithmic_bytes_formula": "8 F + 8 nnzA + 28 nnzB_pre (SURVEY.md 8d)", "seconds": t_sp,
                                "traffic": ((traffic or {}).get("spgemm_dram_bytes"))},
            "roofline_build_A": {"bound": "hbm", "kernel": "seed keys, radix sorts by (read, column) and (column, read), dedupe, CSR + CSC (rank 0)",
                                 "achieved": 40.0 * sizes_local["nnzA"] / (tm["build_ms"] / 1e3) / 1e9 if tm["build_ms"] > 0 else 0.0, "peak": peak, "unit": "GB/s",
                                 "frac": (40.0 * sizes_local["nnzA"] / (tm["build_ms"] / 1e3) / 1e9 / peak) if tm["build_ms"] > 0 else 0.0,
                                 "algorithmic_bytes": 40.0 * sizes_local["nnzA"], "algorithmic_bytes_formula": "40 B per nnzA (SURVEY.md 8d)", "seconds": tm["build_ms"] / 1e3},
            "e2e": {"value": tot_reads / (ms_e2e / 1000.0), "unit": "reads/s", "h2d_bytes_per_step": int(io[0].item()),
                    "d2h_bytes_per_step": int(io[1].item()), "ms_per_step": ms_e2e},
            "gpu_launches": int(tm["kernel_launches"]), "clocks": clocks,
        }
        if world > 1:
            # NVLink side of the roofline (SURVEY §8d): what this rank received in the counting exchange over its device time
            try:
                xb, xs = float(tm.get("exchange_mbytes", 0.0)) * 1e6, float(tm.get("exchange_ms", 0.0)) / 1e3
                line["roofline_nvlink"] = {"bound": "nvlink", "exchange": ("super-k-mer records pushed into the owners' slabs through peer memory (k_skm_forward) + fill words" if skm else "all-to-all of the level-1 k-mer partitions"),
                                           "bytes_per_gpu": xb, "seconds": xs, "achieved": (xb / xs / 1e9) if xs > 0 else 0.0, "peak": 770.0, "unit": "GB/s",
                                           "frac": (xb / xs / 1e9 / 770.0) if xs > 0 else 0.0, "peak_source": "measured peer copy, 770 GB/s per direction per GPU (B200_PROFILING.md; nominal 900)",
                                           "panel_bytes_per_gpu": float(tm.get("panel_mbytes", 0.0)) * 1e6}
            except Exception as ex:          # never lose the bench line over a reporting extra
                line["roofline_nvlink"] = {"error": str(ex)}
        if world == 1 and not args.no_cpu_baseline:
            ranks, cores = square_ranks()
            dna, ck, cl, cu, sample, same = cpu_reference_sample(args.workload)
            rps, kind, used, secs = run_cpu_reference(dna, ck, cl, cu, ranks)
            line["cpu_baseline"] = {"value": rps, "unit": "reads/s", "cores": used, "kind": kind, "host_cores": cores, "same_input_as_gpu_arm": same,
                                    "sample": sample + "; reference KmerOps.cpp/SharedSeeds.cpp compiled unmodified, MPI ranks emulated as threads, CombBLAS restated (oracle/stubs)",
                                    "stage_secs": secs}
            if "shape" in w and not same:
                # the rate at a quarter of the sample: how flat the CPU rate is in the input size (hash maps leave the caches)
                dna2, _, _, _, sample2, _ = cpu_reference_sample(args.workload, max(CPU_SAMPLE.get(w["shape"], 0.05) * min(1.0, ranks / 16.0), 0.01) / 4)
                rps2, _, _, _ = run_cpu_reference(dna2, ck, cl, cu, ranks)
                line["cpu_baseline"]["rate_by_sample"] = [{"sample": sample2, "reads_per_s": rps2}, {"sample": sample, "reads_per_s": rps}]
        print(json.dumps(line), flush=True)
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
