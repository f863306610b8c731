"""Paths of the executables that never reach the GPU — help, version, unopenable input, bad options —
against the reference tools (tests/reference_runs.py: the reference build where there is one, else recorded
outputs): same stdout, stderr and exit code.  (Everything that parses data is in tests/test_gpu_cli.py.)"""
import subprocess
from pathlib import Path

import pytest

import reference_runs

ROOT = Path(__file__).resolve().parent.parent
BIN = ROOT / "vcfx_b200" / "bin"
TOOLS = ["allele_freq_calc", "hwe_tester", "missing_detector", "variant_counter", "allele_counter", "nonref_filter", "indexer", "phase_checker", "inbreeding_calculator", "genotype_query", "dosage_calculator"]


def run(exe, args):
    r = subprocess.run([str(exe), *args], input=b"", capture_output=True, timeout=60)
    # getopt prefixes its own messages with argv[0]: compare them without the directory
    err = r.stderr.replace(str(exe).encode(), exe.name.encode())
    return r.returncode, r.stdout, err


@pytest.fixture(scope="module", autouse=True)
def built():
    from vcfx_b200 import build
    build.build_cuda(); build.build_tools()


@pytest.mark.parametrize("tool", TOOLS)
@pytest.mark.parametrize("args", [["--help"], ["-h"], ["--version"], ["-v"], ["-i", "/nonexistent/x.vcf"], ["/nonexistent/x.vcf"],
                                  ["--no-such-option"], ["-q", "-i", "/nonexistent/x.vcf"], ["--help", "--version"], ["-g", "0/1", "-i", "/nonexistent/x.vcf"]])
def test_same_as_reference_without_a_device(tool, args):
    mine = run(BIN / f"VCFX_{tool}", args)
    ref = reference_runs.run(tool, args)
    assert mine == ref, (tool, args, mine, ref)


def test_genotype_query_without_a_query_prints_its_usage_line():
    for args in ([], ["-q"], ["-i", "/nonexistent/x.vcf"], ["-g", ""]):
        mine = run(BIN / "VCFX_genotype_query", args)
        ref = reference_runs.run("genotype_query", args)
        assert mine == ref, (args, mine, ref)
