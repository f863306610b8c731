"""VCFX_plink_bed (vcfx_b200/bin): PLINK 1 .bed / .bim / .fam from a VCF.  The tool has no reference counterpart, so its
files are checked against what the published format says they hold, built from the oracle's dosage text: the .bed is
decoded here (magic bytes, variant-major, two bits a sample with the low bits first) and compared call for call, and
its bytes with the numpy packing of test_gpu_dosage_bed.py; the .bim against the first five columns of the oracle's
rows; the .fam against the "#CHROM" line.  test_emu_plink_cli.py runs the same tests with the executable linked against
the warp emulator, with one and with three devices."""
import os
import subprocess
from pathlib import Path

import numpy as np
import pytest

import golden_util
import test_gpu_dosage_bed as DB
import test_gpu_dosage_matrix as D
import vcfgen
from vcfx_b200 import synth

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
BIN = ROOT / "vcfx_b200" / "bin"
FILE = 0
MAGIC = b"\x6c\x1b\x01"
SHORT_WARNING = b"Warning: Skipping VCF line with fewer than 10 fields.\n"


def run(args, stdin=None, env=None, cwd=None):
    exe = BIN / "VCFX_plink_bed"
    assert exe.exists(), f"{exe} not built (python -c 'import __graft_entry__ as g; g.build()')"
    e = dict(os.environ)
    if env:
        e.update(env)
    r = subprocess.run([str(exe), *args], input=stdin if stdin is not None else b"", capture_output=True, timeout=300, env=e, cwd=cwd)
    return r.returncode, r.stdout, r.stderr


def decode_bed(raw, n_samples):
    """A variant-major PLINK 1 .bed as an int matrix: A1 (ALT) allele counts, -1 missing."""
    assert raw[:3] == MAGIC, raw[:3]
    B = (n_samples + 3) // 4
    body = np.frombuffer(raw, dtype=np.uint8, offset=3)
    assert len(body) % B == 0 if B else len(body) == 0
    rows = len(body) // B if B else 0
    bits = np.stack([(body >> (2 * k)) & 3 for k in range(4)], axis=-1).reshape(rows, 4 * B)[:, :n_samples]
    return np.select([bits == 0, bits == 2, bits == 3], [2, 1, 0], default=-1)


def expected(O, data):
    """(.bed bytes, .bim bytes, .fam bytes, the calls) the tool should write for `data` (file-mode rules)."""
    from vcfx_b200 import api
    names = api._ds_prescan(data, FILE)[2]
    W = len(names)
    codes, fields = DB.oracle_codes(O, data, FILE, W)
    bed = MAGIC + DB.pack(codes, W).tobytes()
    bim = b"".join(b"\t".join((f[0], f[2], b"0", f[1], f[4], f[3])) + b"\n" for f in fields)
    fam = b"".join(b"%s\t%s\t0\t0\t0\t-9\n" % (n, n) for n in names)
    return bed, bim, fam, np.where(codes < 0, -1, codes)


def read3(prefix):
    return tuple(Path(f"{prefix}{e}").read_bytes() for e in (".bed", ".bim", ".fam"))


def leftovers(d, stem):
    return sorted(p.name for p in Path(d).iterdir() if p.name.startswith(stem + "."))


@pytest.fixture(scope="module")
def files(tmp_path_factory):
    d = tmp_path_factory.mktemp("plink")
    out = {}
    corpora = {
        "c3": synth.make_vcf(3, 600, 301, seed=4),
        "late": vcfgen.make_vcf(500, n_lines=150, n_samples=3, header="late"),
        "crlf": vcfgen.make_vcf(501, n_lines=150, n_samples=7, crlf=True),
        "nonl": vcfgen.make_vcf(502, n_lines=150, n_samples=11, final_newline=False),
        "lattice": D.ds_lattice_input(129),
        "literal": DB.literal_input(True),
        "ragged": D.ragged_input(),
        "quirks": golden_util.load()["ds_quirks"][0],
    }
    for k, data in corpora.items():
        p = d / f"{k}.vcf"
        p.write_bytes(data)
        out[k] = p
    return out


def check_run(O, data, prefix, args, stdin=None, env=None):
    rc, so, se = run(["--out", str(prefix), *args], stdin, env)
    assert rc == 0 and so == b"", (args, rc, se[-300:])
    bed, bim, fam = read3(prefix)
    want_bed, want_bim, want_fam, calls = expected(O, data)
    assert bed == want_bed, (args, len(bed), len(want_bed))
    assert bim == want_bim and fam == want_fam, args
    got = decode_bed(bed, fam.count(b"\n"))
    assert np.array_equal(got, calls), args
    assert leftovers(prefix.parent, prefix.name) == [prefix.name + e for e in (".bed", ".bim", ".fam")]
    return se


def test_file_positional_and_stdin(oracle, files, tmp_path):
    """Each corpus through -i FILE, a positional FILE and stdin, at the default chunk size and at small chunks: the same
    three files, equal to the format's reading of the oracle's rows."""
    for name, p in files.items():
        data = p.read_bytes()
        o = oracle.dosage(data, FILE)
        if o.first_bad_line:
            continue
        small = {"VCFX_CHUNK_BYTES": str(D.small_chunk(data))}
        for k, (args, stdin, env) in enumerate(((["-q", "-i", str(p)], None, None), (["-q", str(p)], None, small),
                                                (["-q"], data, None), (["-q"], data, small))):
            check_run(oracle, data, tmp_path / f"{name}{k}", args, stdin, env)


def test_warnings_and_quiet(oracle, files, tmp_path):
    """A line with fewer than ten fields: one warning each, none with -q; rows wider than the "#CHROM" line: one warning
    with their count, with or without -q."""
    data = files["literal"].read_bytes()
    se = check_run(oracle, data, tmp_path / "w", ["-i", str(files["literal"])])
    assert se.count(SHORT_WARNING) == oracle.dosage(data, FILE).warnings == 1
    assert b"Warning: 1 variant line(s) have more sample columns" in se
    se = check_run(oracle, data, tmp_path / "q", ["-q"], stdin=data)
    assert SHORT_WARNING not in se and b"Warning: 1 variant line(s)" in se
    ragged = files["ragged"].read_bytes()
    se = check_run(oracle, ragged, tmp_path / "r", [str(files["ragged"])])
    assert se == b"Warning: 1 variant line(s) have more sample columns than the #CHROM line names; the extra columns were dropped.\n"
    se = check_run(oracle, files["c3"].read_bytes(), tmp_path / "c", [str(files["c3"])])
    assert se == b""


def test_header_only(oracle, tmp_path):
    """A "#CHROM" line and no data: a 3-byte .bed, an empty .bim and a full .fam."""
    data = b"##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\ts1\ts2\ts3\n"
    check_run(oracle, data, tmp_path / "h", [], stdin=data)
    assert read3(tmp_path / "h") == (MAGIC, b"", b"s1\ts1\t0\t0\t0\t-9\ns2\ts2\t0\t0\t0\t-9\ns3\ts3\t0\t0\t0\t-9\n")


def test_errors_leave_no_files(files, tmp_path):
    """Each failure exits 1 with a message and leaves no PREFIX.* file behind."""
    hdr = b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tA\tB\n"
    line = b"1\t100\trs1\tA\tG\t.\tPASS\t.\tGT\t0/1\t1/1\n"
    bad_input = tmp_path / "early.vcf"
    bad_input.write_bytes(line + hdr + line)
    cases = [
        (["--out", "{p}", "-i", str(bad_input)], None, None, b"Error: VCF header (#CHROM) not found before variant records.\n"),
        (["--out", "{p}"], line + hdr + line, None, b"Error: VCF header (#CHROM) not found before variant records.\n"),
        (["--out", "{p}"], b"##fileformat=VCFv4.2\n", None, b"Error: no #CHROM header line in the input.\n"),
        (["--out", "{p}"], b"", None, b"Error: no #CHROM header line in the input.\n"),
        (["-i", str(files["c3"])], None, None, b"Error: --out PREFIX is required.\n"),
        (["--out", "{p}", "-i", str(tmp_path / "missing.vcf")], None, None, b"Error: cannot open file"),
        (["--out", str(tmp_path / "no_such_dir" / "x")], hdr + line, None, b"Error: cannot create"),
        (["--out", "{p}"], hdr.replace(b"\tB\n", b"\tB C\n") + line, None, b"contains a blank"),
        (["--out", "{p}"], hdr.replace(b"\tA\t", b"\t\t") + line, None, b"is empty or contains a blank"),
        (["--out", "{p}"], hdr + line * 50 + b"1\t2\t" + b"x" * 9000 + b"\n", {"VCFX_CHUNK_BYTES": "4096"}, b"Error: "),
    ]
    for k, (args, stdin, env, msg) in enumerate(cases):
        prefix = tmp_path / f"err{k}"
        rc, so, se = run([a.replace("{p}", str(prefix)) for a in args], stdin, env)
        assert rc == 1 and so == b"" and msg in se, (k, rc, se)
        assert leftovers(tmp_path, f"err{k}") == [], (k, leftovers(tmp_path, f"err{k}"))
    assert not (tmp_path / "no_such_dir").exists()


def test_help():
    rc, so, se = run(["--help"])
    assert rc == 0 and b"no counterpart" in so and b"any non-REF allele" in so


def test_multi_gpu_same_bytes(oracle, files, tmp_path):
    """VCFX_CUDA_DEVICES=all: chunks dealt round-robin over the GPUs, the same three files as one GPU."""
    data = files["c3"].read_bytes()
    env = {"VCFX_CHUNK_BYTES": str(64 << 10)}
    check_run(oracle, data, tmp_path / "one", ["-q", str(files["c3"])], env={**env, "VCFX_CUDA_DEVICES": "0"})
    check_run(oracle, data, tmp_path / "all", ["-q", str(files["c3"])], env={**env, "VCFX_CUDA_DEVICES": "all"})
    assert read3(tmp_path / "one") == read3(tmp_path / "all")
