"""The oracle (CPU restatement, oracle/vcfx_oracle.c) against the committed outputs of the reference
tools (tests/golden/reference_outputs.json), and on seeded inputs against tests/reference_runs.py: the reference
build where there is one, else outputs recorded from the drop-in tools (see there).  This is what pins the oracle;
the GPU parity tests then compare the CUDA path with the oracle."""
import os
import tempfile

import pytest

import golden_util
import reference_runs
import vcfgen
from vcfx_b200 import synth

GOLD = golden_util.load()


def check_case(O, data, exp, name):
    for mode_name, mode in (("file", O.FILE), ("stdin", O.STDIN)):
        for tool, fn in (("allele_freq_calc", O.allele_freq), ("hwe_tester", O.hwe), ("missing_detector", O.missing)):
            key = f"{tool}.{mode_name}"
            if key in exp:
                r = fn(data, mode)
                assert (r.rc, r.out) == exp[key][:2], (name, key)
        key = f"indexer.{mode_name}"
        if key in exp:
            r = O.indexer(data, mode)
            assert (r.rc, r.out, r.warnings) == tuple(exp[key][:3]), (name, key)
        key = f"nonref_filter.{mode_name}"
        if key in exp:
            r = O.nonref_filter(data, mode)
            assert (r.rc, r.out, r.warnings) == tuple(exp[key][:3]), (name, key)
        key = f"phase_checker.{mode_name}"
        if key in exp:
            r = O.phase_checker(data, mode)
            assert (r.rc, r.out, O.phase_checker_stderr(data, mode)) == tuple(exp[key][:3]), (name, key)
        for strict in (0, 1):
            key = f"variant_counter.{mode_name}.strict{strict}"
            r = O.variant_count(data, mode, bool(strict))
            assert (r.rc, r.out) == exp[key][:2], (name, key)
            if not strict:
                assert r.warnings == exp[key][2], (name, key)
    for key, mode in (("file", O.FILE), ("stdin", O.STDIN)):
        k = f"dosage_calculator.{key}"
        if k in exp:
            r = O.dosage(data, mode)
            assert (r.rc, r.out, O.DS_ERROR if r.first_bad_line else O.DS_WARNING * r.warnings) == tuple(exp[k][:3]), (name, k)
    for key, mode, q, strict in (("file.het", O.FILE, "0/1", False), ("stdin.het", O.STDIN, "1/0", False),
                                 ("file.strict", O.FILE, "0|1", True), ("stdin.strict", O.STDIN, "1/1", True)):
        k = f"genotype_query.{key}"
        if k in exp:
            r, err = O.genotype_query(data, q, mode, strict)
            assert (r.rc, r.out, err) == tuple(exp[k][:3]), (name, k)
    for key, mode, flags in (("file", O.FILE, 0), ("stdin", O.STDIN, 0), ("file.global", O.FILE, O.IB_GLOBAL),
                             ("file.skipcount", O.FILE, O.IB_SKIP_BOUNDARY | O.IB_COUNT_BOUNDARY), ("stdin.skip", O.STDIN, O.IB_SKIP_BOUNDARY)):
        k = f"inbreeding_calculator.{key}"
        if k in exp:
            r = O.inbreeding(data, mode, flags | O.IB_QUIET)
            assert (r.rc, r.out, O.IB_MESSAGES[r.warnings]) == tuple(exp[k][:3]), (name, k)
    for key, (path, fmt, limit) in {"mt": (O.AC_MT_TEXT, O.AC_TEXT, 0), "stream": (O.AC_STREAM, O.AC_TEXT, 0),
                                    "agg": (O.AC_UNIFIED, O.AC_AGGREGATE, 0), "bin": (O.AC_UNIFIED, O.AC_BINARY, 0),
                                    "limit2": (O.AC_UNIFIED, O.AC_TEXT, 2)}.items():
        k = f"allele_counter.{key}"
        if k in exp:
            r = O.allele_counter(data, path, fmt, limit)
            assert (r.rc, r.out) == exp[k][:2], (name, k)


@pytest.mark.parametrize("name", sorted(GOLD))
def test_oracle_matches_reference_outputs(oracle, name):
    data, exp = GOLD[name]
    check_case(oracle, data, exp, name)


def test_golden_covers_the_modes_that_differ():
    """The fixtures hold the two facts the reference's own tests never pin (SURVEY.md finding 1):
    FILE and STDIN mode print different text for an AF tie and for HWE p-values."""
    _, exp = GOLD["af_tie"]
    assert b"0.0313" in exp["allele_freq_calc.file"][1] and b"0.0312" in exp["allele_freq_calc.stdin"][1]
    differ = sum(GOLD[n][1]["hwe_tester.file"][1] != GOLD[n][1]["hwe_tester.stdin"][1] for n in GOLD)
    assert differ >= 3


@pytest.mark.parametrize("seed", range(25))
def test_oracle_matches_reference_binaries_fuzz(oracle, seed):
    """Seeded inputs against the reference tools (tests/reference_runs.py)."""
    O = oracle
    hdr = ["normal", "normal", "late", "none", "double"][seed % 5]
    data = vcfgen.make_vcf(9000 + seed, n_lines=30, n_samples=1 + seed % 7, crlf=(seed % 7 == 3), final_newline=(seed % 5 != 2), header=hdr)
    with tempfile.NamedTemporaryFile(suffix=".vcf") as f:
        f.write(data); f.flush()
        for tool, fn in (("allele_freq_calc", O.allele_freq), ("hwe_tester", O.hwe), ("missing_detector", O.missing)):
            extra = ["-t", "1"] if tool == "missing_detector" else []
            rc, out, _ = reference_runs.run(tool, ["-q", *extra, "-i", f.name]); r = fn(data, O.FILE)
            assert (r.rc, r.out) == (rc, out), (tool, "file")
            rc, out, _ = reference_runs.run(tool, ["-q"] if tool != "hwe_tester" else [], stdin=data); r = fn(data, O.STDIN)
            assert (r.rc, r.out) == (rc, out), (tool, "stdin")
        rc, out, err = reference_runs.run("indexer", [f.name]); r = O.indexer(data, O.FILE)
        assert (r.rc, r.out, r.warnings) == (rc, out, err.count(b"no #CHROM")), "indexer file"
        rc, out, err = reference_runs.run("indexer", [], stdin=data); r = O.indexer(data, O.STDIN)
        assert (r.rc, r.out, r.warnings) == (rc, out, err.count(b"no #CHROM")), "indexer stdin"
        rc, out, err = reference_runs.run("nonref_filter", ["-i", f.name]); r = O.nonref_filter(data, O.FILE)
        assert (r.rc, r.out, r.warnings) == (rc, out, err.count(b"Warning")), "nonref_filter file"
        rc, out, err = reference_runs.run("nonref_filter", [], stdin=data); r = O.nonref_filter(data, O.STDIN)
        assert (r.rc, r.out, r.warnings) == (rc, out, err.count(b"Warning")), "nonref_filter stdin"
        rc, out, err = reference_runs.run("phase_checker", ["-i", f.name]); r = O.phase_checker(data, O.FILE)
        assert (r.rc, r.out, O.phase_checker_stderr(data, O.FILE)) == (rc, out, err), "phase_checker file"
        rc, out, err = reference_runs.run("phase_checker", ["-"], stdin=data); r = O.phase_checker(data, O.STDIN)
        assert (r.rc, r.out, O.phase_checker_stderr(data, O.STDIN)) == (rc, out, err), "phase_checker stdin"
        rc, out, err = reference_runs.run("phase_checker", ["-q"], stdin=data)
        assert (rc, out, err) == (r.rc, r.out, b""), "phase_checker -q"
        rc, out, err = reference_runs.run("dosage_calculator", ["-i", f.name]); r = O.dosage(data, O.FILE)
        assert (r.rc, r.out, O.DS_ERROR if r.first_bad_line else O.DS_WARNING * r.warnings) == (rc, out, err), "dosage_calculator file"
        rc, out, err = reference_runs.run("dosage_calculator", ["-q"], stdin=data); r = O.dosage(data, O.STDIN)
        assert (r.rc, r.out, O.DS_ERROR if r.first_bad_line else O.DS_WARNING * r.warnings) == (rc, out, err), "dosage_calculator stdin"
        for q, strict in (("0/1", False), ("1|1", True), ("2/0", False)):
            a = ["-g", q] + (["--strict"] if strict else [])
            rc, out, err = reference_runs.run("genotype_query", [*a, "-i", f.name]); r, e = O.genotype_query(data, q, O.FILE, strict)
            assert (r.rc, r.out, e) == (rc, out, err), ("genotype_query file", a)
            rc, out, err = reference_runs.run("genotype_query", a, stdin=data); r, e = O.genotype_query(data, q, O.STDIN, strict)
            assert (r.rc, r.out, e) == (rc, out, err), ("genotype_query stdin", a)
        for flags, args in ((0, []), (O.IB_GLOBAL, ["--freq-mode", "global"]), (O.IB_SKIP_BOUNDARY, ["--skip-boundary"]),
                            (O.IB_SKIP_BOUNDARY | O.IB_COUNT_BOUNDARY, ["--skip-boundary", "--count-boundary-as-used"])):
            rc, out, err = reference_runs.run("inbreeding_calculator", ["-q", *args, "-i", f.name]); r = O.inbreeding(data, O.FILE, flags | O.IB_QUIET)
            assert (r.rc, r.out, O.IB_MESSAGES[r.warnings]) == (rc, out, err), ("inbreeding_calculator file", args)
            rc, out, err = reference_runs.run("inbreeding_calculator", ["-q", *args], stdin=data); r = O.inbreeding(data, O.STDIN, flags | O.IB_QUIET)
            assert (r.rc, r.out, O.IB_MESSAGES[r.warnings]) == (rc, out, err), ("inbreeding_calculator stdin", args)
        for strict in (False, True):
            a = ["--strict"] if strict else []
            rc, out, err = reference_runs.run("variant_counter", [*a, f.name]); r = O.variant_count(data, O.FILE, strict)
            assert (r.rc, r.out) == (rc, out)
            if strict and rc:
                assert b"line %d " % r.first_bad_line in err
        data = vcfgen.make_vcf(9100 + seed, n_lines=30, n_samples=1 + seed % 7, domain="ac", final_newline=(seed % 5 != 2), header=hdr)
        f.seek(0); f.truncate(); f.write(data); f.flush()
        rc, out, _ = reference_runs.run("allele_counter", ["-q", "-i", f.name]); r = O.allele_counter(data, O.AC_MT_TEXT)
        assert (r.rc, r.out) == (rc, out)
        rc, out, _ = reference_runs.run("allele_counter", ["-q"], stdin=data); r = O.allele_counter(data, O.AC_STREAM)
        assert (r.rc, r.out) == (rc, out)
        rc, out, _ = reference_runs.run("allele_counter", ["-q", "-a", "-i", f.name]); r = O.allele_counter(data, O.AC_UNIFIED, O.AC_AGGREGATE)
        assert (r.rc, r.out) == (rc, out)


def test_oracle_matches_reference_binaries_shapes(oracle):
    O = oracle
    for shape, V, S in ((1, 400, 100), (2, 60, 2504), (3, 60, 2504), (4, 150, 33)):
        data = synth.make_vcf(shape, V, S, seed=shape)
        with tempfile.NamedTemporaryFile(suffix=".vcf") as f:
            f.write(data); f.flush()
            for tool, fn in (("allele_freq_calc", O.allele_freq), ("hwe_tester", O.hwe), ("missing_detector", O.missing)):
                extra = ["-t", "1"] if tool == "missing_detector" else []
                rc, out, _ = reference_runs.run(tool, ["-q", *extra, "-i", f.name])
                assert (fn(data, O.FILE).out) == out, (shape, tool)
            rc, out, _ = reference_runs.run("variant_counter", [f.name])
            assert O.variant_count(data).out == out
            rc, out, _ = reference_runs.run("nonref_filter", ["-i", f.name])
            assert O.nonref_filter(data, O.FILE).out == out, (shape, "nonref_filter")
            rc, out, err = reference_runs.run("inbreeding_calculator", ["-q", "-i", f.name])
            assert O.inbreeding(data, O.FILE, O.IB_QUIET).out == out, (shape, "inbreeding_calculator")
            rc, out, err = reference_runs.run("phase_checker", ["-i", f.name])
            assert (O.phase_checker(data, O.FILE).out, O.phase_checker_stderr(data, O.FILE)) == (out, err), (shape, "phase_checker")


def test_hwe_numbers_and_formatters(oracle):
    """Non-trivial p-values (the reference's tests only pin 1.000000) and both formatters."""
    O = oracle
    assert O.fmt("af_file", 1 / 32) == b"0.0313" and O.fmt("af_stdin", 1 / 32) == b"0.0312"
    p = O.hwe_pvalue(50, 20, 30)
    assert 0 < p < 1e-6
    assert O.fmt("p_file", 0.1234567) == b"0.123456" and O.fmt("p_stdin", 0.1234567) == b"0.123457"
    assert O.hwe_pvalue(0, 0, 0) == 1.0 and O.hwe_pvalue(10, 0, 0) == 1.0
