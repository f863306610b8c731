"""The drop-in executables (vcfx_b200/bin/VCFX_*) against the reference tools (tests/reference_runs.py: the reference
build where there is one, else recorded outputs): same argv, same stdin/file, stdout and exit code must be identical."""
import gzip
import os
import subprocess
from pathlib import Path

import pytest

import reference_runs
import vcfgen
from vcfx_b200 import synth

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
BIN = ROOT / "vcfx_b200" / "bin"


def run(exe, args, stdin=None, env=None):
    e = dict(os.environ)
    if env:
        e.update(env)
    r = subprocess.run([str(exe), *args], input=stdin if stdin is not None else b"", capture_output=True, timeout=120, env=e)
    return r.returncode, r.stdout, r.stderr


def both(tool, args, stdin=None, env=None):
    mine = BIN / f"VCFX_{tool}"
    assert mine.exists(), f"{mine} not built (python -c 'import __graft_entry__ as g; g.build()')"
    a = run(mine, args, stdin, env)
    b = reference_runs.run(tool, args, stdin)
    assert a[0] == b[0], (tool, args, a[0], b[0], a[2][-300:], b[2][-300:])
    assert a[1] == b[1], (tool, args, a[1][:300], repr(b[1])[:300])
    return a, b


@pytest.fixture(scope="module")
def files(tmp_path_factory):
    """Few files on purpose: every invocation is a fresh process with its own CUDA context, and the
    per-record behaviour is already covered through the C ABI in test_gpu_parity.py."""
    d = tmp_path_factory.mktemp("vcf")
    out = {}
    out["c3"] = d / "c3.vcf"; out["c3"].write_bytes(synth.make_vcf(3, 600, 300, seed=4))
    spec = {"late": dict(header="late"), "crlf": dict(crlf=True), "nonl": dict(final_newline=False)}
    for i, (k, kw) in enumerate(spec.items()):
        p = d / f"{k}.vcf"
        p.write_bytes(vcfgen.make_vcf(500 + i, n_lines=150, n_samples=3 + 4 * i, **kw))
        out[k] = p
    return out


SMALL_CHUNK = {"VCFX_CHUNK_BYTES": str(48 << 10)}


@pytest.mark.parametrize("tool", ["allele_freq_calc", "hwe_tester", "missing_detector"])
def test_file_and_stdin(files, tool):
    extra = ["-t", "1"] if tool == "missing_detector" else []
    stdin_args = ["-q"] if tool != "hwe_tester" else []
    for name, p in files.items():
        both(tool, ["-q", *extra, "-i", str(p)])
        both(tool, stdin_args, stdin=p.read_bytes())
    # several newline-aligned chunks through the three-slot pipeline, partial last lines carried over
    both(tool, ["-q", *extra, "-i", str(files["c3"])], env=SMALL_CHUNK)
    both(tool, stdin_args, stdin=files["nonl"].read_bytes(), env={"VCFX_CHUNK_BYTES": "4096"})


def test_variant_counter(files):
    for name, p in files.items():
        a, b = both("variant_counter", [str(p)])
        assert sorted(a[2].splitlines()) == sorted(b[2].splitlines())
        a, b = both("variant_counter", ["--strict", str(p)])
        assert a[2] == b[2]
        a, b = both("variant_counter", [], stdin=p.read_bytes())
        assert a[2] == b[2]
    p = files["late"]
    both("variant_counter", ["--strict"], stdin=p.read_bytes())
    both("variant_counter", [], stdin=gzip.compress(p.read_bytes()))
    both("variant_counter", [str(files["c3"])], env=SMALL_CHUNK)
    both("variant_counter", [str(p)], env={"VCFX_CHUNK_BYTES": "4096"})


def test_nonref_filter(files, tmp_path):
    """VCFX_nonref_filter (SURVEY §8 f2): file (-i and positional), "-" and stdin, several chunks, the quirks fixture."""
    import golden_util
    q = tmp_path / "q.vcf"; q.write_bytes(golden_util.load()["nr_quirks"][0])
    homref = tmp_path / "h.vcf"
    rows = [b"21\t%d\t.\tA\tG\t.\tPASS\t.\tGT\t" % (i + 1) + b"\t".join([b"0|0"] * 299 + [b"0|1" if i % 3 == 0 else b"0|0"]) for i in range(400)]
    homref.write_bytes(b"##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + b"\t".join(b"S%d" % i for i in range(300)) + b"\n" + b"\n".join(rows) + b"\n")
    for p in (files["late"], files["crlf"], q, homref):          # (every invocation is a process with its own CUDA context)
        both("nonref_filter", ["-i", str(p)])
        both("nonref_filter", [], stdin=p.read_bytes())
    both("nonref_filter", [str(q)])
    both("nonref_filter", ["-"], stdin=q.read_bytes())
    both("nonref_filter", ["-i", str(homref)], env=SMALL_CHUNK)
    both("nonref_filter", [], stdin=files["nonl"].read_bytes(), env={"VCFX_CHUNK_BYTES": "4096"})
    both("nonref_filter", ["-i", str(files["c3"])], env=SMALL_CHUNK)


def test_phase_checker(files, tmp_path):
    """VCFX_phase_checker (SURVEY §8 f2): stdout and the messages on stderr, file (-i and positional) and stdin ("-": the
    reference shows its help text when started without arguments before anything can be read from the pipe), -q,
    several chunks (messages stay in line order; file mode's FORMAT cache spans the chunk borders)."""
    import golden_util
    q = tmp_path / "q.vcf"; q.write_bytes(golden_util.load()["pc_quirks"][0])
    fc = tmp_path / "fc.vcf"; fc.write_bytes(golden_util.load()["pc_format_cache"][0])
    phased = tmp_path / "p.vcf"
    rows = [b"21\t%d\t.\tA\tG\t.\tPASS\t.\tGT\t" % (i + 1) + b"\t".join([b"0|1"] * 299 + [b"0/1" if i % 3 == 0 else b"1|0"]) for i in range(400)]
    phased.write_bytes(b"##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + b"\t".join(b"S%d" % i for i in range(300)) + b"\n" + b"\n".join(rows) + b"\n")
    for p in (files["crlf"], q, fc, phased):
        a, b = both("phase_checker", ["-i", str(p)])
        assert a[2] == b[2]
        a, b = both("phase_checker", ["-"], stdin=p.read_bytes())
        assert a[2] == b[2]
    a, b = both("phase_checker", [str(q)])
    assert a[2] == b[2]
    a, b = both("phase_checker", ["-q", "-i", str(q)])
    assert a[2] == b[2] == b""
    a, b = both("phase_checker", ["--quiet"], stdin=q.read_bytes())
    assert a[2] == b[2] == b""
    for f, env in ((phased, SMALL_CHUNK), (fc, {"VCFX_CHUNK_BYTES": "128"}), (files["c3"], SMALL_CHUNK)):
        a, b = both("phase_checker", ["-i", str(f)], env=env)
        assert a[2] == b[2]
    a, b = both("phase_checker", ["-"], stdin=files["nonl"].read_bytes(), env={"VCFX_CHUNK_BYTES": "4096"})
    assert a[2] == b[2]


def test_dosage_calculator(files, tmp_path):
    """VCFX_dosage_calculator (SURVEY §8 f2): stdout, stderr and exit code, file and stdin, -q (which the stdin path ignores),
    several chunks, the quirks fixture, a data line in front of the header (nothing on stdout, exit code 1 in file mode)."""
    import golden_util
    q = tmp_path / "q.vcf"; q.write_bytes(golden_util.load()["ds_quirks"][0])
    nohdr = tmp_path / "n.vcf"; nohdr.write_bytes(b"##f\n1\t1\t.\tA\tG\t.\t.\t.\tGT\t0/1\n#CHROM\tP\tI\tR\tA\tQ\tF\tI\tFORMAT\tS1\n")
    for p, arg_sets in ((files["crlf"], ([],)), (q, ([], ["-q"])), (nohdr, ([],))):
        for args in arg_sets:
            a, b = both("dosage_calculator", [*args, "-i", str(p)])
            assert a[2] == b[2]
            a, b = both("dosage_calculator", args, stdin=p.read_bytes())
            assert a[2] == b[2]
    a, b = both("dosage_calculator", [str(q)])
    assert a[2] == b[2]
    both("dosage_calculator", ["-q", "-i", str(files["c3"])], env=SMALL_CHUNK)
    both("dosage_calculator", ["-q"], stdin=files["c3"].read_bytes(), env=SMALL_CHUNK)
    both("dosage_calculator", ["-q"], stdin=files["nonl"].read_bytes(), env={"VCFX_CHUNK_BYTES": "4096"})


def test_genotype_query(files, tmp_path):
    """VCFX_genotype_query (SURVEY §8 f2): stdout and stderr, file and stdin, flexible and strict, several chunks (stdin mode's
    '#' lines wait for a data line across chunk borders), the run that ends at a data line in front of the header."""
    import golden_util
    q = tmp_path / "q.vcf"; q.write_bytes(golden_util.load()["gq_quirks"][0])
    tails = tmp_path / "t.vcf"
    body = synth.make_vcf(3, 300, 60, seed=31)
    tails.write_bytes(body + b"#t1\n\n#t2\n" + b"#pad\n" * 2000)                      # '#' lines behind the last data line, several chunks of them
    nohdr = tmp_path / "n.vcf"; nohdr.write_bytes(b"##f\n#x\n1\t1\t.\tA\tG\t.\t.\t.\tGT\t0/1\n" + body)
    for p, arg_sets in ((files["crlf"], (["-g", "0/1"],)), (q, (["-g", "0/1"], ["-g", "1|1", "--strict"])), (tails, (["-g", "1|1", "--strict"],)), (nohdr, (["-g", "0/1"],))):
        for args in arg_sets:          # (every invocation is a process with its own CUDA context: about a second each)
            a, b = both("genotype_query", [*args, "-i", str(p)])
            assert a[2] == b[2]
            a, b = both("genotype_query", args, stdin=p.read_bytes())
            assert a[2] == b[2]
    a, b = both("genotype_query", ["-g", "0/1", "-q", str(q)])
    assert a[2] == b[2] == b""
    a, b = both("genotype_query", ["--genotype-query", "1/0", "--quiet"], stdin=q.read_bytes())
    assert a[2] == b[2] == b""
    for f, env in ((tails, {"VCFX_CHUNK_BYTES": "4096"}), (files["c3"], SMALL_CHUNK), (q, {"VCFX_CHUNK_BYTES": "256"})):
        a, b = both("genotype_query", ["-g", "0/1", "-i", str(f)], env=env)
        assert a[2] == b[2]
        a, b = both("genotype_query", ["-g", "0/1"], stdin=f.read_bytes(), env=env)
        assert a[2] == b[2]
    a, b = both("genotype_query", ["-g", "2/2", "-i", str(files["c3"])], env=SMALL_CHUNK)     # nothing matches: the header alone
    assert a[2] == b[2]


def test_inbreeding_calculator(files, tmp_path):
    """VCFX_inbreeding_calculator (SURVEY §8 f3): file (-i and positional) and stdin, every option, several chunks (the
    per-sample sums are carried from chunk to chunk in file order), the quirks fixture, the fixed messages."""
    import golden_util
    q = tmp_path / "q.vcf"; q.write_bytes(golden_util.load()["ib_quirks"][0])
    wide = tmp_path / "w.vcf"; wide.write_bytes(synth.make_vcf(3, 1500, 300, seed=21))
    for p in (files["crlf"], q, wide):
        a, b = both("inbreeding_calculator", ["-q", "-i", str(p)])
        assert a[2] == b[2]
        a, b = both("inbreeding_calculator", ["-q"], stdin=p.read_bytes())
        assert a[2] == b[2]
    a, b = both("inbreeding_calculator", [str(q)])
    assert a[2] == b[2]                                  # "Processing <file> (<n> bytes)..."
    for args in (["--freq-mode", "global"], ["--skip-boundary"], ["--skip-boundary", "--count-boundary-as-used"], ["--freq-mode", "bogus"]):
        a, b = both("inbreeding_calculator", ["-q", *args, "-i", str(q)])
        assert a[2] == b[2]
    both("inbreeding_calculator", ["-q", "--skip-boundary", "--count-boundary-as-used"], stdin=wide.read_bytes(), env=SMALL_CHUNK)
    both("inbreeding_calculator", ["-q", "--freq-mode", "global"], stdin=wide.read_bytes(), env=SMALL_CHUNK)
    both("inbreeding_calculator", ["-q", "-i", str(wide)], env=SMALL_CHUNK)
    both("inbreeding_calculator", ["-q", "-i", str(files["c3"])], env={"VCFX_CHUNK_BYTES": str(wide.stat().st_size // 3)})
    both("inbreeding_calculator", ["-q"], stdin=files["nonl"].read_bytes(), env={"VCFX_CHUNK_BYTES": "4096"})
    multi = tmp_path / "m.vcf"                           # every site multi-allelic: "No biallelic variants found."
    multi.write_bytes(b"##f\n#CHROM\tP\tI\tR\tA\tQ\tF\tI\tFORMAT\tA\tB\n1\t1\t.\tA\tG,T\t.\t.\t.\tGT\t0/1\t1/1\n")
    a, b = both("inbreeding_calculator", [], stdin=multi.read_bytes())
    assert a[2] == b[2]
    hdr_only = tmp_path / "h.vcf"; hdr_only.write_bytes(b"##f\n#CHROM\tP\tI\tR\tA\tQ\tF\tI\tFORMAT\tA\tB\n")
    for p in (hdr_only,):
        a, b = both("inbreeding_calculator", ["-q", "-i", str(p)])
        assert a[2] == b[2]
        a, b = both("inbreeding_calculator", ["-q"], stdin=p.read_bytes())
        assert a[2] == b[2]
    nohdr = tmp_path / "n.vcf"; nohdr.write_bytes(b"##f\n1\t1\t.\tA\tG\t.\t.\t.\tGT\t0/1\t1/1\n")
    a, b = both("inbreeding_calculator", ["-q", "-i", str(nohdr)])
    assert a[2] == b[2]
    a, b = both("inbreeding_calculator", ["-q"], stdin=nohdr.read_bytes())
    assert a[2] == b[2]


def test_indexer(files, tmp_path):
    """VCFX_indexer (SURVEY §8 f4): file argument and stdin, several chunks (offsets stay absolute), the quirks fixture."""
    import golden_util
    q = tmp_path / "q.vcf"; q.write_bytes(golden_util.load()["ix_quirks"][0])
    for p in (files["late"], files["crlf"], q):
        a, b = both("indexer", [str(p)])
        assert a[2] == b[2]
        a, b = both("indexer", [], stdin=p.read_bytes())
        assert a[2] == b[2]
    both("indexer", [str(files["c3"])], env=SMALL_CHUNK)
    both("indexer", [], stdin=files["c3"].read_bytes(), env=SMALL_CHUNK)
    both("indexer", [], stdin=files["nonl"].read_bytes(), env={"VCFX_CHUNK_BYTES": "4096"})


@pytest.mark.parametrize("tool", ["allele_freq_calc", "hwe_tester", "missing_detector", "variant_counter", "allele_counter", "nonref_filter", "indexer", "phase_checker", "inbreeding_calculator", "genotype_query", "dosage_calculator"])
def test_flags(tool, files):
    for args in (["--help"], ["-v"]):
        both(tool, args)
    if tool == "genotype_query":
        a, b = both(tool, ["-g", "0/1", "-i", "/nonexistent/file.vcf"]); assert a[2] == b[2]
        a, b = both(tool, ["-g", "0/1"], stdin=b""); assert a[2] == b[2]
        return
    a, b = both(tool, ["/nonexistent/file.vcf"] if tool == "variant_counter" else (["-i", "/nonexistent/file.vcf"] if tool in ("nonref_filter", "phase_checker", "dosage_calculator") else ["/nonexistent/file.vcf"] if tool == "indexer" else ["-q", "-i", "/nonexistent/file.vcf"]))
    assert a[2] == b[2]
    # empty stdin: per-tool behaviour (help+rc1 / header only / nothing / Total 0); phase_checker without arguments prints its
    # help text unless stdin is readable at that very moment (a race with the parent closing the pipe): give it an argument
    both(tool, ["-q"] if tool == "phase_checker" else [], stdin=b"")


def test_allele_counter(tmp_path):
    a = tmp_path / "a.vcf"; a.write_bytes(vcfgen.make_vcf(901, n_lines=120, n_samples=6, domain="ac"))
    b = tmp_path / "b.vcf"; b.write_bytes(synth.make_vcf(3, 300, 40, seed=8))
    c = tmp_path / "c.vcf"; c.write_bytes(vcfgen.make_vcf(902, n_lines=40, n_samples=3, domain="ac", header="double", final_newline=False))
    for p in (a, b, c):
        both("allele_counter", ["-q", "-i", str(p)])
        both("allele_counter", ["-q", str(p)])
        both("allele_counter", ["-q"], stdin=p.read_bytes())
        both("allele_counter", ["-q", "-a", "-i", str(p)])
        both("allele_counter", ["-q", "-b", "-i", str(p)])
        both("allele_counter", ["-q", "-l", "2", "-i", str(p)])
    both("allele_counter", ["-q", "-s", "S1 S0", "-i", str(a)])
    both("allele_counter", ["-q", "-s", "S1 S0"], stdin=a.read_bytes())
    both("allele_counter", ["-q", "-s", "S1 nope", "-i", str(a)])
    both("allele_counter", ["-q", "-a", "-s", "S2 S0", "-i", str(a)])
    both("allele_counter", ["-q", "-i", str(b)], env={"VCFX_CHUNK_BYTES": str(16 << 10)})
    # -z: the gzip container may differ, the payload may not
    mine = run(BIN / "VCFX_allele_counter", ["-q", "-z", "-i", str(a)])
    ref = reference_runs.run("allele_counter", ["-q", "-z", "-i", str(a)])          # (its stdout: the payload of the reference's stream)
    assert mine[0] == ref[0] == 0 and gzip.decompress(mine[1]) == ref[1]
    # header-less inputs
    both("allele_counter", ["-q"], stdin=b"##only\n")
    both("allele_counter", ["-q"], stdin=b"1\t1\t.\tA\tG\t.\t.\t.\tGT\t0/1\n")


def test_large_file_parallel_io(tmp_path):
    """Files past the 8 MiB mark take the multi-threaded pread / pwrite paths of the host reader:
    output to a regular file must be byte-identical to the reference's, with one and with eight I/O
    threads (VCFX_IO_THREADS), and identical to the pipe path."""
    src = tmp_path / "big.vcf"
    src.write_bytes(synth.make_vcf(3, 9000, 600, seed=21))          # ~ 22 MB, dots on most lines
    assert src.stat().st_size > (20 << 20)

    def to_file(exe, args, out, env=None):
        e = dict(os.environ); e.update(env or {})
        with open(out, "wb") as f:
            r = subprocess.run([str(exe), *args], stdout=f, stderr=subprocess.PIPE, timeout=300, env=e)
        return r.returncode

    for tool, args in (("missing_detector", ["-q", "-t", "1", "-i", str(src)]), ("allele_freq_calc", ["-q", "-i", str(src)])):
        rc, want, _ = reference_runs.run(tool, args)
        assert rc == 0
        for threads in ("1", "8"):
            out = tmp_path / f"{tool}.{threads}"
            assert to_file(BIN / f"VCFX_{tool}", args, out, {"VCFX_IO_THREADS": threads}) == 0
            assert out.read_bytes() == want, (tool, threads)
        rc, piped, _ = run(BIN / f"VCFX_{tool}", args)
        assert rc == 0 and piped == want


def test_multi_gpu_same_bytes(tmp_path):
    """VCFX_CUDA_DEVICES: one context per GPU in one process, chunks dealt round-robin, text drained in submission order
    (the reference's own decomposition, allele_counter.cpp:870-947: newline-aligned ranges, results written in order).
    The bytes must be those of the one-GPU run and of the reference tool, for all five tools."""
    import ctypes
    n = ctypes.c_int(0)
    lib = ctypes.CDLL(str(ROOT / "vcfx_b200" / "libvcfx_cuda.so"))
    lib.vcfx_cuda_device_count(ctypes.byref(n))
    if n.value < 2:
        pytest.skip("needs at least two GPUs")
    src = tmp_path / "m.vcf"
    src.write_bytes(synth.make_vcf(3, 3000, 300, seed=33))           # ~3.6 MB: dozens of 128 KiB chunks over the GPUs
    late = tmp_path / "late.vcf"
    late.write_bytes(vcfgen.make_vcf(77, n_lines=3000, n_samples=6, header="late"))
    env_multi = {"VCFX_CUDA_DEVICES": "all", "VCFX_CHUNK_BYTES": str(128 << 10)}
    env_one = {"VCFX_CHUNK_BYTES": str(128 << 10)}
    cases = [("allele_freq_calc", ["-q", "-i"]), ("hwe_tester", ["-q", "-i"]), ("missing_detector", ["-q", "-t", "1", "-i"]),
             ("variant_counter", []), ("allele_counter", ["-q", "-i"]), ("allele_counter", ["-q", "-a", "-i"]), ("nonref_filter", ["-i"]), ("indexer", []), ("phase_checker", ["-i"]),
             ("genotype_query", ["-g", "0/1", "-i"]), ("dosage_calculator", ["-q", "-i"]), ("inbreeding_calculator", ["-q", "-i"])]
    for f in (src, late):
        for tool, args in cases:
            one = run(BIN / f"VCFX_{tool}", [*args, str(f)], env=env_one)
            many = run(BIN / f"VCFX_{tool}", [*args, str(f)], env=env_multi)
            assert one[0] == many[0] and one[1] == many[1], (tool, f.name)
            both(tool, [*args, str(f)], env=env_multi)
    both("variant_counter", ["--strict", str(late)], env=env_multi)
