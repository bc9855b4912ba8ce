"""PAF text on the device (elba_fe_paf) against the format of tests/paf_inputs.py, byte for byte: overlap.paf from the resident
alignments and string.paf from the resident string graph, with and without read names, on the reads fixture, the CLR- and
HiFi-like synthetic sets and a set large enough for thousands of CTAs of the write kernel; the empty cases, the state rules, the
device pointer, and the driver (python -m elba_b200.assemble) from a FASTA file to its three files."""
import os
import subprocess
import sys

import numpy as np
import pytest

import paf_inputs as PI

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
HIFI = dict(genome_len=60_000, n_reads=160, mean_len=6000, sd_len=857, err=0.01, seed=11)


def _ctx(k, lo, up):
    from elba_b200 import frontend
    return frontend.Context(frontend.Params(k=k, lower=lo, upper=up, device=0))


def _names(n, kind, seed=0):
    if kind is None:
        return None
    rng = np.random.default_rng(seed)
    if kind == "short":
        return ["ACGTacgt!~"[i % 10] for i in range(n)]
    if kind == "long":
        return [f"read{i}_" + "x" * int(rng.integers(1900, 2100)) for i in range(n)]
    return [f"m54{i % 7}/{i}/ccs_{int(rng.integers(0, 10**6))}" for i in range(n)]


def run_and_check(ctx, dna, base, scoring, names, what):
    """Upload, align, both PAF files; each must equal the formatter.  Returns (overlap info, string info, alignments)."""
    from elba_b200 import frontend
    ctx.upload(dna, base)
    ctx.set_read_names(names if names is not None else [])      # names stay until replaced: clear those of an earlier run
    ctx.run()
    al = ctx.align(*scoring)
    text, info = ctx.paf(frontend.PAF_OVERLAP)
    want = PI.text(*al, dna.lengths, base, names)
    assert text == want, (what, "overlap", len(text), len(want))
    assert (info["lines"], info["total_lines"], info["bytes"], info["total_bytes"], info["offset"]) == \
        (len(al[0]), len(al[0]), len(want), len(want), 0), (what, info)
    R = ctx.overlap_graph()
    S = ctx.string_graph()
    stext, sinfo = ctx.paf(frontend.PAF_STRING)
    swant = PI.string_text(S, R, {0: al}, dna.lengths, base, names)
    assert stext == swant, (what, "string", len(stext), len(swant))
    assert sinfo["lines"] == sinfo["total_lines"] == int((S[4] == 0).sum()) and sinfo["total_bytes"] == len(swant), (what, sinfo)
    return info, sinfo, al


@pytest.mark.parametrize("names", [None, "given"])
@pytest.mark.parametrize("kind,k,lo,up,scoring,base", [
    ("reads_fa", 17, 2, 8, (1, -1, -1, 15), 0),
    ("reads_fa", 17, 2, 8, (1, -1, -1, 15), 4321),
    ("clr", 17, 2, 8, (2, -3, -2, 25), 77),
    ("hifi", 31, 2, 4, (1, -1, -1, 15), 1000),
])
def test_paf_vs_format(kind, k, lo, up, scoring, base, names, fixtures):
    from elba_b200.synth import make_dnabuffer
    dna = fixtures("reads_fa") if kind == "reads_fa" else make_dnabuffer(**dict(HIFI, err=0.12 if kind == "clr" else 0.01))
    ctx = _ctx(k, lo, up)
    info, sinfo, al = run_and_check(ctx, dna, base, scoring, _names(dna.size(), names), (kind, base, names))
    assert len(al[0]) > 0 and sinfo["lines"] > 0 and info["ms"] > 0
    ctx.close()


@pytest.mark.parametrize("names", ["short", "long"])
def test_name_lengths(names):
    """1-byte names (a run of lines fits the staging buffer) and ~2,000-byte names (no run fits: every thread writes its own line
    directly)."""
    from elba_b200.synth import make_dnabuffer
    dna = make_dnabuffer(**HIFI)
    ctx = _ctx(31, 2, 4)
    info, sinfo, _ = run_and_check(ctx, dna, 5, (1, -1, -1, 15), _names(dna.size(), names), names)
    if names == "long":
        assert info["bytes"] / max(info["lines"], 1) > 4000 and info["lines"] > 256
    ctx.close()


def test_large_set():
    """HiFi-like, 40x: 8,000 reads of 4 kb on an 800 kb genome; hundreds of thousands of lines, thousands of CTAs."""
    import torch
    from elba_b200 import synth
    buf, off, lens = synth.make_reads(800_000, 8000, 4000, 500, 0.01, 313, device="cuda")
    dna = synth.to_dnabuffer(buf.cpu(), off.cpu(), lens.cpu())
    torch.cuda.synchronize()
    ctx = _ctx(31, 2, 40)
    names = _names(dna.size(), "given", 5)
    info, sinfo, al = run_and_check(ctx, dna, 12345, (1, -1, -1, 15), names, "large")
    assert info["lines"] > 1000 * 256, info
    print(f"large: {info['lines']} lines {info['bytes']} bytes {info['ms']:.3f} ms; string {sinfo['lines']} lines {sinfo['ms']:.3f} ms")
    ctx.close()


def _random_reads(rng, n, length):
    return ["".join("ACGT"[c] for c in rng.integers(0, 4, length)) for _ in range(n)]


def test_empty_cases():
    from elba_b200 import frontend
    from elba_b200.dnabuffer import DnaBuffer
    rng = np.random.default_rng(2)
    ctx = _ctx(31, 2, 8)
    # no alignments: reads without a shared k-mer
    info, sinfo, al = run_and_check(ctx, DnaBuffer.from_strings(_random_reads(rng, 4, 3000)), 3, (1, -1, -1, 15), None, "none")
    assert len(al[0]) == 0 and info["total_bytes"] == 0 and sinfo["total_lines"] == 0 and sinfo["total_bytes"] == 0
    # every alignment failing: a 300-base repeat inside reads whose flanks differ (too short an overlap for its overhangs)
    seqs = []
    for _ in range(3):
        r = _random_reads(rng, 1, 300)[0]
        x, w = _random_reads(rng, 2, 1000)
        y, z = _random_reads(rng, 2, 500)
        seqs += [x + r + y, z + r + w]
    info, sinfo, al = run_and_check(ctx, DnaBuffer.from_strings(seqs), 0, (1, -1, -1, 15), ["r%d" % i for i in range(len(seqs))], "failing")
    assert len(al[0]) >= 3 and not al[2][:, 6].any() and info["total_bytes"] > 0
    assert sinfo["total_lines"] == 0 and sinfo["total_bytes"] == 0
    # every alignment passing but contained (identical reads): R and S are empty
    s = _random_reads(rng, 2, 2000)
    info, sinfo, al = run_and_check(ctx, DnaBuffer.from_strings([s[0], s[0], s[1], s[1]]), 9, (1, -1, -1, 15), None, "contained")
    assert len(al[0]) == 2 and al[2][:, 6].all() and sinfo["total_bytes"] == 0
    assert ctx.paf(frontend.PAF_STRING)[0] == b""
    ctx.close()


def test_state_errors():
    from elba_b200 import frontend
    from elba_b200.synth import make_dnabuffer
    dna = make_dnabuffer(**HIFI)
    ctx = _ctx(31, 2, 4)
    L, h = ctx.L, ctx.h
    OV, ST = frontend.PAF_OVERLAP, frontend.PAF_STRING

    def getters():
        import ctypes as C
        p = C.c_void_p()
        return L.elba_fe_get_paf(h, None), L.elba_fe_device_paf(h, C.byref(p))

    def refused(which, code=-5):
        with pytest.raises(frontend.FrontEndError) as e:
            ctx.paf(which)
        assert f"error {code}" in str(e.value), str(e.value)
    assert getters() == (-5, -5)
    refused(OV)
    ctx.upload(dna, 9)
    ctx.run()
    refused(OV); refused(ST)                                # before align
    refused(7, -1)                                          # neither file
    ctx.align()
    ctx.paf(OV)
    assert getters() == (0, 0)
    refused(ST)                                             # before string_graph
    ctx.overlap_graph()
    assert getters() == (-5, -5)                            # a new R discards the text
    refused(ST)
    S = ctx.string_graph()
    ctx.paf(ST)
    assert getters() == (0, 0)
    ctx.transitive_reduction(9 + dna.size(), S[0], S[1], S[2])
    assert getters() == (-5, -5)
    refused(ST)                                             # S of the host route
    ctx.paf(OV)
    ctx.string_graph()
    ctx.paf(ST)
    # names: wrong count, bad names, names replaced
    ctx.set_read_names(["n%d" % i for i in range(dna.size() - 1)])
    assert getters() == (-5, -5)
    refused(OV); refused(ST)
    with pytest.raises(ValueError):
        ctx.set_read_names(["a b"] * dna.size())
    import ctypes as C
    bad = np.frombuffer(b"ab c", np.uint8)
    off = np.array([0, 2, 4], np.uint64)
    assert L.elba_fe_set_read_names(h, frontend._p(bad), frontend._p(off), C.c_uint64(2)) == -1          # blank inside a name
    off = np.array([0, 2, 2], np.uint64)
    assert L.elba_fe_set_read_names(h, frontend._p(bad), frontend._p(off), C.c_uint64(2)) == -1          # empty name
    ctx.set_read_names([])
    ctx.paf(ST)
    # reads replaced after align
    ctx.upload(dna, 9)
    assert getters() == (-5, -5)
    refused(OV); refused(ST)
    ctx.run()
    refused(OV)                                             # a new B: its alignments are not there yet
    ctx.close()


def test_device_paf_equals_get_paf():
    import ctypes as C
    import torch
    from elba_b200 import frontend
    from elba_b200.synth import make_dnabuffer
    dna = make_dnabuffer(**HIFI)
    ctx = _ctx(31, 2, 4)
    run_and_check(ctx, dna, 0, (1, -1, -1, 15), None, "device")
    for which in (frontend.PAF_OVERLAP, frontend.PAF_STRING):
        text, info = ctx.paf(which)
        p = C.c_void_p()
        ctx._ck(ctx.L.elba_fe_device_paf(ctx.h, C.byref(p)))

        class Dev:
            __cuda_array_interface__ = {"shape": (info["bytes"],), "typestr": "|u1", "data": (p.value, False), "version": 3}
        dev = torch.as_tensor(Dev(), device="cuda").cpu().numpy().tobytes()
        assert len(text) > 0 and dev == text
    ctx.close()


def test_driver(tmp_path):
    """python -m elba_b200.assemble on a FASTA with named records: the three files equal the step-by-step route."""
    from elba_b200 import frontend
    from elba_b200.assemble import assemble
    from elba_b200.fasta import write_fasta
    from elba_b200.synth import make_dnabuffer
    dna = make_dnabuffer(**HIFI)
    names = _names(dna.size(), "given", 9)
    fa = str(tmp_path / "reads.fa")
    write_fasta(fa, [dna.read_ascii(i) for i in range(dna.size())], width=60, names=names)
    prefix = str(tmp_path / "out")
    params = frontend.Params(k=31, lower=2, upper=4, device=0)
    out = assemble(fa, prefix, params)
    # the same through the command line
    p = subprocess.run([sys.executable, "-m", "elba_b200.assemble", fa, "-k", "31", "-l", "2", "-u", "4", "-o", prefix + "_cli"],
                       capture_output=True, text=True, cwd=os.path.dirname(HERE), timeout=900)
    assert p.returncode == 0, p.stderr[-3000:]
    # step by step
    ctx = frontend.Context(params)
    ctx.upload(dna, 0)
    ctx.set_read_names(names)
    ctx.run()
    al = ctx.align()
    R = ctx.overlap_graph()
    S = ctx.string_graph()
    cg = ctx.contigs()
    frontend.write_contigs_fa(str(tmp_path / "want.contigs.fa"), cg.seqs, cg.info["first"])
    ctx.close()
    read = lambda f: open(f, "rb").read()  # noqa: E731
    for pre in (prefix, prefix + "_cli"):
        assert read(pre + ".overlap.paf") == PI.text(*al, dna.lengths, 0, names)
        assert read(pre + ".string.paf") == PI.string_text(S, R, {0: al}, dna.lengths, 0, names)
        assert read(pre + ".contigs.fa") == read(str(tmp_path / "want.contigs.fa"))
    assert out["contigs"] == cg.info["ncontigs"] > 0 and out["pairs"] == len(al[0]) and out["S"] == len(S[0])
    assert out["overlap_paf_bytes"] == os.path.getsize(prefix + ".overlap.paf")


# ---- several GPUs ----------------------------------------------------------------------------------------------------
def _ngpus():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.parametrize("world,grid", [(2, "-"), (2, "2x1"), (4, "2x2")])
def test_multi_gpu_paf(world, grid, tmp_path):
    """string.paf and contigs.fa byte-identical to one GPU, overlap.paf the same lines; step by step with a nonzero first id,
    and through the driver."""
    if _ngpus() < world:
        pytest.skip(f"needs {world} GPUs")
    port = 29941 + 10 * world + (0 if grid == "-" else 1)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(HERE, "multi_gpu_paf_worker.py"), grid, "321", str(tmp_path)]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=1500)
    assert p.returncode == 0 and "MULTI-GPU PAF OK" in p.stdout, p.stdout[-3000:] + p.stderr[-3000:]
