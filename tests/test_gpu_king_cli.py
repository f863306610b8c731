"""VCFX_king (vcfx_b200/bin): PREFIX.kin0 from a VCF.  The tool has no reference counterpart: its bytes are checked against
text built here from numpy counts of the oracle's dosage rows (test_gpu_king.py's planes and products), printed as the
tool documents it (tab-separated, pairs i < j with i outer, KINSHIP with %.6g or NA).  test_emu_king_cli.py runs the same
tests with the executable linked against the warp emulator, with one and with three devices."""
import os
import subprocess
from pathlib import Path

import numpy as np
import pytest

import test_gpu_dosage_bed as DB
import test_gpu_dosage_matrix as D
import test_gpu_king as K
import vcfgen
from vcfx_b200 import synth

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
BIN = ROOT / "vcfx_b200" / "bin"
FILE = 0
SHORT_WARNING = b"Warning: Skipping VCF line with fewer than 10 fields.\n"
HEADER = b"#ID1\tID2\tNSNP\tHETHET\tIBS0\tHET1\tHET2\tKINSHIP\n"


def run(args, stdin=None, env=None):
    exe = BIN / "VCFX_king"
    assert exe.exists(), f"{exe} not built (python -c 'import __graft_entry__ as g; g.build()')"
    e = dict(os.environ)
    if env:
        e.update(env)
    r = subprocess.run([str(exe), *args], input=stdin if stdin is not None else b"", capture_output=True, timeout=300, env=e)
    return r.returncode, r.stdout, r.stderr


def expected(O, data, min_kinship=None):
    from vcfx_b200 import api
    names = api._ds_prescan(data, FILE)[2]
    W = len(names)
    v = K.bed_codes(DB.oracle_codes(O, data, FILE, W)[0])
    cc, hh, ab, hc = K.expected_counts(v) if W else [np.zeros((0, 0), dtype=np.int64)] * 4
    kin = K.expected_kinship(cc, hh, ab, hc)
    out = [HEADER]
    for i in range(W):
        for j in range(i + 1, W):
            k = kin[i, j]
            if min_kinship is not None and not (k >= min_kinship):
                continue
            out.append(b"%s\t%s\t%d\t%d\t%d\t%d\t%d\t%s\n" % (names[i], names[j], cc[i, j], hh[i, j], ab[i, j] + ab[j, i], hc[i, j], hc[j, i],
                                                            b"NA" if np.isnan(k) else b"%.6g" % k))
    return b"".join(out)


def leftovers(d, stem):
    return sorted(p.name for p in Path(d).iterdir() if p.name.startswith(stem + "."))


@pytest.fixture(scope="module")
def files(tmp_path_factory):
    d = tmp_path_factory.mktemp("king")
    corpora = {
        "c3": synth.make_vcf(3, 600, 301, seed=4),
        "late": vcfgen.make_vcf(500, n_lines=150, n_samples=3, header="late"),
        "crlf": vcfgen.make_vcf(501, n_lines=150, n_samples=7, crlf=True),
        "nonl": vcfgen.make_vcf(502, n_lines=150, n_samples=11, final_newline=False),
        "lattice": D.ds_lattice_input(129),
        "literal": DB.literal_input(True),
        "ragged": D.ragged_input(),
    }
    out = {}
    for k, data in corpora.items():
        p = d / f"{k}.vcf"
        p.write_bytes(data)
        out[k] = p
    return out


def check_run(O, data, prefix, args, stdin=None, env=None, min_kinship=None):
    rc, so, se = run(["--out", str(prefix), *args], stdin, env)
    assert rc == 0 and so == b"", (args, rc, se[-300:])
    got = Path(f"{prefix}.kin0").read_bytes()
    want = expected(O, data, min_kinship)
    assert got == want, (args, len(got), len(want), got[:300], want[:300])
    assert leftovers(prefix.parent, prefix.name) == [prefix.name + ".kin0"]
    return se


def test_file_positional_and_stdin(oracle, files, tmp_path):
    """Each corpus through -i FILE, a positional FILE and stdin, at the default chunk size and at small chunks."""
    for name, p in files.items():
        data = p.read_bytes()
        if oracle.dosage(data, FILE).first_bad_line:
            continue
        small = {"VCFX_CHUNK_BYTES": str(D.small_chunk(data))}
        for k, (args, stdin, env) in enumerate(((["-q", "-i", str(p)], None, None), (["-q", str(p)], None, small),
                                                (["-q"], data, None), (["-q"], data, small))):
            check_run(oracle, data, tmp_path / f"{name}{k}", args, stdin, env)


def test_min_kinship(oracle, files, tmp_path):
    """--min-kinship X keeps the pairs with kinship >= X and drops NA pairs; a value strtod does not consume is an error."""
    data = files["c3"].read_bytes()
    kin = np.array([float(l.split(b"\t")[7]) for l in expected(oracle, data).split(b"\n")[1:-1] if not l.endswith(b"NA")])
    cut = float(np.quantile(kin, 0.9))
    for k, x in enumerate((str(cut), repr(float(kin.max())), "-1", "1e9")):
        check_run(oracle, data, tmp_path / f"m{k}", ["-q", "--min-kinship", x, str(files["c3"])], min_kinship=float(x))
    hdr = b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tA\tB\tC\n"            # B is never het: NA with everyone
    nas = hdr + b"".join(b"1\t%d\t.\tA\tG\t.\t.\t.\tGT\t%s\t0/0\t%s\n" % (i, [b"0/1", b"1/1"][i % 2], [b"0/1", b"0/0", b"1/1"][i % 3])
                         for i in range(1, 40))
    check_run(oracle, nas, tmp_path / "na", ["-q", "-m", "-100"], stdin=nas, min_kinship=-100.0)
    assert Path(f"{tmp_path / 'na'}.kin0").read_bytes().count(b"\n") == 2
    for k, bad in enumerate(("", "0.1x", "abc", "0.1 ")):
        rc, so, se = run(["--out", str(tmp_path / f"bad{k}"), "--min-kinship", bad, str(files["c3"])])
        assert rc == 1 and b"Error: invalid --min-kinship value" in se, (bad, se)
        assert leftovers(tmp_path, f"bad{k}") == []


def test_warnings_and_quiet(oracle, files, tmp_path):
    """A line with fewer than ten fields: one warning each, none with -q; rows wider than the "#CHROM" line: one warning."""
    data = files["literal"].read_bytes()
    se = check_run(oracle, data, tmp_path / "w", ["-i", str(files["literal"])])
    assert se.count(SHORT_WARNING) == oracle.dosage(data, FILE).warnings == 1
    assert b"Warning: 1 variant line(s) have more sample columns" in se
    se = check_run(oracle, data, tmp_path / "q", ["-q"], stdin=data)
    assert SHORT_WARNING not in se and b"Warning: 1 variant line(s)" in se
    se = check_run(oracle, files["c3"].read_bytes(), tmp_path / "c", [str(files["c3"])])
    assert se == b""


def test_header_only_and_no_samples(oracle, tmp_path):
    """No data lines: every pair with NSNP 0 and NA; no samples: the header line alone."""
    data = b"##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\ts1\ts2\ts3\n"
    check_run(oracle, data, tmp_path / "h", [], stdin=data)
    assert Path(f"{tmp_path / 'h'}.kin0").read_bytes() == HEADER + b"s1\ts2\t0\t0\t0\t0\t0\tNA\ns1\ts3\t0\t0\t0\t0\t0\tNA\ns2\ts3\t0\t0\t0\t0\t0\tNA\n"
    data = b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\n1\t1\t.\tA\tG\t.\t.\t.\tGT\n"
    check_run(oracle, data, tmp_path / "n", [], stdin=data)
    assert Path(f"{tmp_path / 'n'}.kin0").read_bytes() == HEADER


def test_errors_leave_no_files(files, tmp_path):
    """Each failure exits 1 with a message and leaves no PREFIX.kin0 behind."""
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
        (["--out", "{p}"], hdr.replace(b"\tB\n", b"\tB C\n") + line, None, b"contains a blank; .kin0 is whitespace-delimited"),
        (["--out", "{p}"], hdr.replace(b"\tA\t", b"\t\t") + line, None, b"is empty or contains a blank"),
        (["--out", "{p}"], hdr + line * 50 + b"1\t2\t" + b"x" * 9000 + b"\n", {"VCFX_CHUNK_BYTES": "4096"}, b"Error: "),
        (["--out", "{p}", "--min-kinship", "0.2.5", str(files["c3"])], None, None, b"Error: invalid --min-kinship value '0.2.5'\n"),
    ]
    for k, (args, stdin, env, msg) in enumerate(cases):
        prefix = tmp_path / f"err{k}"
        rc, so, se = run([a.replace("{p}", str(prefix)) for a in args], stdin, env)
        assert rc == 1 and so == b"" and msg in se, (k, rc, se)
        assert leftovers(tmp_path, f"err{k}") == [], (k, leftovers(tmp_path, f"err{k}"))
    assert not (tmp_path / "no_such_dir").exists()


def test_help():
    rc, so, se = run(["--help"])
    assert rc == 0 and b"no counterpart" in so and b"--min-kinship" in so


def test_multi_gpu_same_bytes(oracle, files, tmp_path):
    """VCFX_CUDA_DEVICES=all: the scan's chunks dealt round-robin over the GPUs, the same .kin0 as one GPU."""
    data = files["c3"].read_bytes()
    env = {"VCFX_CHUNK_BYTES": str(64 << 10)}
    check_run(oracle, data, tmp_path / "one", ["-q", str(files["c3"])], env={**env, "VCFX_CUDA_DEVICES": "0"})
    check_run(oracle, data, tmp_path / "all", ["-q", str(files["c3"])], env={**env, "VCFX_CUDA_DEVICES": "all"})
    assert Path(f"{tmp_path / 'one'}.kin0").read_bytes() == Path(f"{tmp_path / 'all'}.kin0").read_bytes()
