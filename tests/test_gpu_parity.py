"""Parity of the CUDA path (through the C ABI) with the oracle, byte for byte.

Every case runs the same bytes through libvcfx_cuda (streaming entry points, host buffers)
and through the CPU restatement in oracle/, in both input modes of the reference.
"""
import pytest

import vcfgen
from vcfx_b200 import synth

pytestmark = pytest.mark.gpu

MODES = [0, 1]


def _cmp(name, got, exp):
    if got != exp:
        i = next((k for k in range(min(len(got), len(exp))) if got[k] != exp[k]), min(len(got), len(exp)))
        raise AssertionError(f"{name}: first difference at byte {i} (len {len(got)} vs {len(exp)}):\n"
                             f"  got {got[max(0, i - 60): i + 60]!r}\n  exp {exp[max(0, i - 60): i + 60]!r}")


def run_all(api, O, data, tag, chunk_bytes=0, tile_bytes=0, tools=("af", "hwe", "vc", "md", "nr", "ix", "pc", "ib", "gq", "ds")):
    kw = dict(chunk_bytes=chunk_bytes, tile_bytes=tile_bytes)
    for mode in MODES:
        if "af" in tools:
            r = api.allele_freq_calc(data, mode, **kw); o = O.allele_freq(data, mode)
            _cmp(f"{tag} af mode{mode}", r.out, o.out)
            assert r.rc == o.rc
            if o.rc == 0:
                assert r.totals.rows == o.rows
                assert r.totals.pre_header + (r.totals.short_lines if mode == 1 else 0) == o.warnings
        if "hwe" in tools:
            r = api.hwe_tester(data, mode, **kw); o = O.hwe(data, mode)
            _cmp(f"{tag} hwe mode{mode}", r.out, o.out)
        if "md" in tools and not (mode == 0 and max((len(l) for l in data.split(b"\n")), default=0) > 60000):
            # (FILE mode of the reference overflows its 64 KB line buffer on longer lines: no oracle there)
            r = api.missing_detector(data, mode, **kw); o = O.missing(data, mode)
            _cmp(f"{tag} md mode{mode}", r.out, o.out)
            assert r.totals.flagged == o.flagged or (mode == 0 and r.totals.dots_terminated == 0)
        if "ix" in tools:
            r = api.indexer(data, mode, **kw); o = O.indexer(data, mode)
            _cmp(f"{tag} ix mode{mode}", r.out, o.out)
            assert (r.totals.rows, r.totals.pre_header) == (o.rows, o.warnings)
        if "nr" in tools:
            r = api.nonref_filter(data, mode, **kw); o = O.nonref_filter(data, mode)
            _cmp(f"{tag} nr mode{mode}", r.out, o.out)
            assert (r.totals.rows, r.totals.pre_header) == (o.rows, o.warnings)
        if "pc" in tools:
            r = api.phase_checker(data, mode, **kw); o = O.phase_checker(data, mode)
            _cmp(f"{tag} pc mode{mode}", r.out, o.out)
            _cmp(f"{tag} pc mode{mode} stderr", r.err, O.phase_checker_stderr(data, mode))
            assert (r.totals.rows, r.totals.pre_header, r.totals.flagged) == (o.rows, o.warnings, o.flagged + o.warnings)
        if "ds" in tools:
            r = api.dosage_calculator(data, mode, **kw); o = O.dosage(data, mode)
            _cmp(f"{tag} ds mode{mode}", r.out, o.out)
            assert (r.rc, r.err) == (o.rc, O.DS_ERROR if o.first_bad_line else O.DS_WARNING * o.warnings)
        if "gq" in tools:
            for q, strict in ((("0/1", False), ("1|1", True)) if mode == 0 else (("1/1", False), ("0|1", True))):
                r = api.genotype_query(data, q, mode, strict, **kw); o, e = O.genotype_query(data, q, mode, strict)
                _cmp(f"{tag} gq {q} strict{strict} mode{mode}", r.out, o.out)
                _cmp(f"{tag} gq {q} strict{strict} mode{mode} stderr", r.err, e)
        if "ib" in tools:
            for fl in ((0, 6) if mode == 0 else (0, 1)):
                r = api.inbreeding_calculator(data, mode, bool(fl & 1), bool(fl & 2), bool(fl & 4), quiet=False, **kw); o = O.inbreeding(data, mode, fl)
                _cmp(f"{tag} ib mode{mode} flags{fl}", r.out, o.out)
                assert r.err == O.IB_MESSAGES[o.warnings]
                if o.warnings in (0, 3):
                    assert r.totals.rows == o.rows
        if "vc" in tools:
            for strict in (False, True):
                r = api.variant_counter(data, mode, strict, **kw); o = O.variant_count(data, mode, strict)
                _cmp(f"{tag} vc mode{mode} strict{strict}", r.out, o.out)
                assert r.rc == o.rc
                if strict and o.rc:
                    assert r.totals.first_short_line == o.first_bad_line
                if not strict:
                    assert r.totals.short_lines == o.warnings
                    assert len(r.totals.short_line_numbers) == o.warnings


# the inputs below are shared with test_gpu_resident.py, which runs them through the device-resident entry point
SHAPES = [(1, 2000, 100), (2, 200, 2504), (3, 200, 2504), (4, 40, 2504), (2, 3000, 7), (3, 3000, 33), (4, 500, 21), (1, 1, 1), (2, 50, 0)]


def shape_input(shape, V, S):
    return synth.make_vcf(shape, V, S, seed=100 + shape)


def adversarial_input(seed):
    """vcfgen: both header kinds and the broken ones, CRLF, no final newline."""
    hdr = ["normal", "normal", "late", "none", "double"][seed % 5]
    return vcfgen.make_vcf(seed, n_lines=60, n_samples=1 + seed % 9, crlf=(seed % 7 == 3),
                           final_newline=(seed % 4 != 1), header=hdr)


DEGENERATE = (b"", b"\n", b"\n\n\n", b"#only header\n", b"#CHROM\tPOS\n", b"1\t2\t3", b"\t\t\t\t\t\t\t\tGT\n",
              b"#CHROM\n\t\t\t\t\t\t\t\tGT", b"#CHROM\n1\t1\t.\tA\tG\t.\t.\t.\tGT\t0/1\r\n",
              b"#CHROM\n1\t1\t.\tA\tG\t.\t.\t.\tGT\t\n", b"#CHROM\n1\t1\t.\tA\tG\t.\t.\t.\tGT\t0/1\t")

SWEEP_S = list(range(1, 34, 2)) + list(range(100, 134, 3)) + [119, 120, 121, 127, 128, 129, 255, 256, 257, 383, 511, 640]


def sweep_input(shape, S):
    return synth.make_vcf(shape, 150 if S < 300 else 40, S, seed=1000 * shape + S)


@pytest.mark.parametrize("shape,V,S", SHAPES)
def test_synthetic_shapes(cuda_api, oracle, shape, V, S):
    data = shape_input(shape, V, S)
    run_all(cuda_api, oracle, data, f"shape{shape} {V}x{S}")


@pytest.mark.parametrize("seed", range(40))
def test_adversarial(cuda_api, oracle, seed):
    data = adversarial_input(seed)
    run_all(cuda_api, oracle, data, f"fuzz{seed}")


@pytest.mark.parametrize("tile", [512, 1024, 4096])
def test_small_tiles_many_boundaries(cuda_api, oracle, tile):
    """Tiny tiles put tile boundaries everywhere: inside headers, samples, at '\\n', at CRLF."""
    for seed in range(6):
        data = vcfgen.make_vcf(1000 + seed, n_lines=80, n_samples=3 + 5 * seed, crlf=(seed == 2),
                               final_newline=(seed != 3))
        run_all(cuda_api, oracle, data, f"tile{tile} fuzz{seed}", tile_bytes=tile)
    data = synth.make_vcf(3, 300, 300, seed=5)
    run_all(cuda_api, oracle, data, f"tile{tile} shape3", tile_bytes=tile)


def test_multi_chunk_stream(cuda_api, oracle):
    """Several newline-aligned chunks through the 3-slot pipeline, order preserved."""
    data = synth.make_vcf(3, 4000, 200, seed=9)
    run_all(cuda_api, oracle, data, "chunks", chunk_bytes=256 << 10)
    data = vcfgen.make_vcf(77, n_lines=3000, n_samples=6, header="late")
    run_all(cuda_api, oracle, data, "chunks-fuzz", chunk_bytes=64 << 10)


def test_empty_and_degenerate(cuda_api, oracle):
    for data in DEGENERATE:
        run_all(cuda_api, oracle, data, repr(data[:20]))


def test_missing_detector_cases(cuda_api, oracle):
    H = b"##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tS1\tS2\n"
    L = lambda info, s1, s2: b"1\t100\t.\tA\tG\t.\tPASS\t" + info + b"\tGT:DP\t" + s1 + b"\t" + s2
    cases = [
        H + L(b"DP=25", b"0/1:3", b"./.:0") + b"\n",
        H + L(b"DP=25;", b"0/1:3", b".") + b"\n",
        H + L(b".", b".|.", b"0/0") + b"\n" + L(b"", b"0/.", b"1/1") + b"\n",
        H + L(b"AF=0.5", b"0/1:0.5", b"1/1:.") + b"\n",                # dots outside the first piece only
        H + L(b"DP=1", b"0/1", b"0/.") ,                                  # unterminated + flagged, only dot (pre-scan quirk)
        H + L(b"DP=1", b"./.", b"0/0") + b"\n" + L(b"DP=2", b"0/1", b"0/.") ,   # ... with another dotted line before it
        H + L(b"DP=1", b"0/1", b"0/0") + b"\r\n" + L(b"DP=2", b"0.", b"./1") + b"\r\n",
        H + L(b"DP=1", b"0.5", b"1.5") + b"\n" + L(b"DP=1", b"0/1:.", b".:1") + b"\n",
        H + b"1\t100\t.\tA\tG\t.\tPASS\tDP=3\tGT\n" + b"1\t100\t.\tA\tG\t.\tPASS\tDP=3\tGT\t\n" + b"\n#x\t.\n",
        H + L(b"DP=1", b"0/1", b"0/1").replace(b"0/1\t0/1", b"0/1\t\t.\t") + b"\n",
    ]
    for i, data in enumerate(cases):
        run_all(cuda_api, oracle, data, f"mdcase{i}", tools=("md",))
        run_all(cuda_api, oracle, data, f"mdcase{i}-tile512", tile_bytes=512, tools=("md",))


def _ac_all(api, O, data, tag, **kw):
    cases = [(O.AC_MT_TEXT, O.AC_TEXT, 0, None), (O.AC_STREAM, O.AC_TEXT, 0, None), (O.AC_UNIFIED, O.AC_AGGREGATE, 0, None),
             (O.AC_UNIFIED, O.AC_BINARY, 0, None), (O.AC_UNIFIED, O.AC_TEXT, 2, None),
             (O.AC_MT_TEXT, O.AC_TEXT, 0, "S1 S0"), (O.AC_STREAM, O.AC_TEXT, 0, "S1 S0"), (O.AC_UNIFIED, O.AC_AGGREGATE, 0, "S2 S0 S1"),
             (O.AC_MT_TEXT, O.AC_TEXT, 0, "S0 nope")]
    for path, fmt, limit, samples in cases:
        o = O.allele_counter(data, path, fmt, limit, samples)
        r = api.allele_counter(data, path, fmt, limit, samples, **kw)
        assert r.rc == o.rc, (tag, path, fmt, limit, samples, r.rc, o.rc)
        _cmp(f"{tag} ac path{path} fmt{fmt} l{limit} s{samples}", r.out, o.out)


@pytest.mark.parametrize("seed", range(16))
def test_allele_counter_adversarial(cuda_api, oracle, seed):
    hdr = ["normal", "normal", "late", "none", "double"][seed % 5]
    data = vcfgen.make_vcf(2000 + seed, n_lines=50, n_samples=1 + seed % 8, domain="ac", final_newline=(seed % 4 != 1), header=hdr)
    _ac_all(cuda_api, oracle, data, f"acfuzz{seed}")
    if seed % 4 == 0:
        _ac_all(cuda_api, oracle, data, f"acfuzz{seed}-tile512", tile_bytes=512)


@pytest.mark.parametrize("shape,V,S", [(1, 300, 100), (2, 60, 2504), (3, 60, 2504), (4, 100, 33), (3, 500, 9)])
def test_allele_counter_shapes(cuda_api, oracle, shape, V, S):
    data = synth.make_vcf(shape, V, S, seed=300 + shape)
    for path, fmt in ((oracle.AC_MT_TEXT, oracle.AC_TEXT), (oracle.AC_UNIFIED, oracle.AC_AGGREGATE), (oracle.AC_UNIFIED, oracle.AC_BINARY)):
        o = oracle.allele_counter(data, path, fmt)
        r = cuda_api.allele_counter(data, path, fmt)
        assert r.rc == o.rc
        _cmp(f"ac shape{shape} path{path} fmt{fmt}", r.out, o.out)
    # several chunks; the first one overflows the default output slot and is re-run with exact sizes
    r = cuda_api.allele_counter(data, oracle.AC_MT_TEXT, chunk_bytes=256 << 10)
    _cmp(f"ac shape{shape} chunks", r.out, oracle.allele_counter(data).out)


def test_gpu_matches_reference_golden(cuda_api):
    """The CUDA path against the committed outputs of the reference tools themselves."""
    import golden_util
    api = cuda_api
    for name, (data, exp) in sorted(golden_util.load().items()):
        for mode_name, mode in (("file", 0), ("stdin", 1)):
            for tool, fn in (("allele_freq_calc", api.allele_freq_calc), ("hwe_tester", api.hwe_tester), ("missing_detector", api.missing_detector)):
                key = f"{tool}.{mode_name}"
                if key in exp:
                    r = fn(data, mode)
                    assert r.rc == exp[key][0], (name, key)
                    if r.rc == 0:
                        _cmp(f"golden {name} {key}", r.out, exp[key][1])
            key = f"indexer.{mode_name}"
            if key in exp:
                r = api.indexer(data, mode)
                assert (r.rc, r.totals.pre_header) == (exp[key][0], exp[key][2]), (name, key)
                _cmp(f"golden {name} {key}", r.out, exp[key][1])
            key = f"nonref_filter.{mode_name}"
            if key in exp:
                r = api.nonref_filter(data, mode)
                assert (r.rc, r.totals.pre_header) == (exp[key][0], exp[key][2]), (name, key)
                _cmp(f"golden {name} {key}", r.out, exp[key][1])
            for strict in (0, 1):
                key = f"variant_counter.{mode_name}.strict{strict}"
                r = api.variant_counter(data, mode, bool(strict))
                assert (r.rc, r.out) == exp[key][:2], (name, key)
        for key, (path, fmt, limit) in {"mt": (0, 0, 0), "stream": (1, 0, 0), "agg": (2, 1, 0), "bin": (2, 2, 0), "limit2": (2, 0, 2)}.items():
            k = f"allele_counter.{key}"
            if k in exp:
                r = api.allele_counter(data, path, fmt, limit)
                assert r.rc == exp[k][0], (name, k)
                _cmp(f"golden {name} {k}", r.out, exp[k][1])


def test_shared_upload_feeds_two_tools(cuda_api, oracle):
    """vcfx_cuda_submit_shared: variant_counter runs on the bytes allele_freq_calc uploaded."""
    import ctypes as C
    api = cuda_api
    data = synth.make_vcf(3, 3000, 120, seed=13)
    chunk = 256 << 10
    af = api.Context(api.OP_ALLELE_FREQ, api.FILE, chunk_bytes=chunk, n_slots=3)
    vc = api.Context(api.OP_VARIANT_COUNT, api.FILE, chunk_bytes=chunk, n_slots=3)
    keep = C.create_string_buffer(data, len(data))
    base = C.addressof(keep)
    valid_abs = api.find_chrom_header(data)
    out_af, rows_vc = [], 0

    def drain():
        nonlocal rows_vc
        o, st, _ = vc.next_output(); rows_vc += st.rows
        o, st, _ = af.next_output(); out_af.append(o)

    n = len(data)
    for s, e in api.chunk_bounds(data, chunk):
        vf = min(max(valid_abs - s, 0), e - s)
        while not af.submit_host(base + s, e - s, valid_from=vf, is_final=(e == n)):
            drain()
        assert vc.submit_shared(af, is_final=(e == n))
    while af.in_flight():
        drain()
    af.close(); vc.close()
    assert api.AF_HEADER + b"".join(out_af) == oracle.allele_freq(data, 0).out
    assert rows_vc == oracle.variant_count(data, 0).rows


def test_line_lengths_sweep(cuda_api, oracle):
    """Lines of every length class against the 512-byte windows: a line inside one window, ending in
    the first bytes of the next one, phase shifts (haploid / missing calls) right before a window or
    line end — the places where the lattice tiers hand over to the exact path."""
    for shape in (1, 2, 3):
        for S in SWEEP_S:
            data = sweep_input(shape, S)
            run_all(cuda_api, oracle, data, f"sweep shape{shape} S{S}", tools=("af", "hwe"))
    data = synth.make_vcf(3, 3000, 120, seed=13)
    run_all(cuda_api, oracle, data, "sweep regression S120", chunk_bytes=256 << 10)


def _mutate_genotypes(data, seed, per_line, forms, crlf_every=0):
    """Replace `per_line` random sample fields of every data line with one of `forms`."""
    import random
    rng = random.Random(seed)
    out = []
    for k, line in enumerate(data.split(b"\n")):
        if line and not line.startswith(b"#"):
            f = line.split(b"\t")
            if len(f) > 9:
                for _ in range(per_line):
                    f[rng.randrange(9, len(f))] = rng.choice(forms)
                line = b"\t".join(f)
                if crlf_every and k % crlf_every == 0:
                    line += b"\r"
        out.append(line)
    return b"\n".join(out)


def test_tier1_rounds_long_lines_and_sparse_exceptions(cuda_api, oracle):
    """The steady tier-1 rounds: lines long enough to hit the periodic flush of the packed sums
    (64 iterations of 2 KiB), and otherwise regular lines with a few genotypes that are not
    `a<sep>b` — each one stops the rounds, goes through the exact path and the rounds resume."""
    for shape in (1, 2):                                   # unphased / phased GT-only
        data = synth.make_vcf(shape, 6, 40000, seed=77 + shape)
        run_all(cuda_api, oracle, data, f"long lines shape{shape}", tools=("af", "hwe"))
    forms = [b".", b"./.", b".|.", b"0", b"1", b"2|1", b"0/1", b"1|0", b"10|1", b"0|1:5", b"", b"./1", b"0|.", b"1/1/1"]
    base = synth.make_vcf(2, 120, 2504, seed=5)
    for per_line, seed in ((1, 1), (3, 2), (12, 3)):
        data = _mutate_genotypes(base, seed, per_line, forms, crlf_every=7 if seed == 2 else 0)
        run_all(cuda_api, oracle, data, f"sparse exceptions x{per_line}", tools=("af", "hwe", "md", "vc"))
        run_all(cuda_api, oracle, data, f"sparse exceptions x{per_line} small tiles", tile_bytes=4096, tools=("af", "hwe"))


def test_multikey_format_exceptions(cuda_api, oracle):
    """Lines whose FORMAT has several keys (GT:AD:DP:GQ:PL) run through the skip-ahead loop: a lane decides the one
    sample that starts in it from four bytes.  Everything else — haploid and missing calls, multi-digit alleles, a
    leading blank, empty columns, samples short enough for two to start in one lane, CRLF — must leave the loop
    and come out of the exact path unchanged."""
    forms = [b".", b"./.:.:.:.:.", b"0:1,2:3", b"10/1:5,5:10:50:0,1,2", b"0/10:5,5:10:50:0,1,2", b"0/1", b"1|1:9", b" 0/1:3",
             b"", b"0/1/1:2,2:4:9:1,2,3", b".|.:1", b"1", b"0|2:3,4:7:20:9,8,7", b"./1:2", b"0/.:2", b"00/1:3", b"0/1:", b"1/1\r"]
    base = synth.make_vcf(4, 60, 2504, seed=21)
    for per_line, seed in ((1, 1), (6, 2), (60, 3)):
        data = _mutate_genotypes(base, seed, per_line, forms, crlf_every=5 if seed == 2 else 0)
        run_all(cuda_api, oracle, data, f"multikey exceptions x{per_line}", tools=("af", "hwe", "vc"))
        run_all(cuda_api, oracle, data, f"multikey exceptions x{per_line} small tiles", tile_bytes=8192, tools=("af", "hwe"))
    # GT first with other keys behind it, every sample one of the short forms: two or more sample starts per lane
    short = synth.make_vcf(4, 30, 300, seed=22)
    data = _mutate_genotypes(short, 4, 250, [b".", b"0/1", b"1", b"./.", b"0|0:1"])
    run_all(cuda_api, oracle, data, "multikey short samples", tools=("af", "hwe"))


def test_digit_path_exceptions(cuda_api, oracle):
    """GT-only lines off the lattice run through the digit path (every byte classified, digits counted); a token of
    more than one character, a ':' piece, a high byte, CRLF in stdin mode make it decline and the exact path takes the
    line: multi-digit alleles, junk bytes, pieces, empty tokens — at every distance from the window borders."""
    forms = [b".", b"./.", b".|.", b"0", b"1", b"0/1", b"1|0", b"./1", b"0|.", b"", b"2|1", b"9/0"]
    odd_forms = [b"10|1", b"0|1:5", b"1/1/1", b"0x/1", b"1.", b".1", b"0/:/1", b":", b"/", b"||", b"1\xc3\xa9", b"01/0", b" 0/1", b"0/1 "]
    base = synth.make_vcf(3, 80, 2504, seed=31)
    for per_line, seed in ((0, 1), (2, 2), (30, 3)):
        data = _mutate_genotypes(base, seed, 40, forms, crlf_every=6 if seed == 2 else 0)
        if per_line:
            data = _mutate_genotypes(data, seed + 10, per_line, odd_forms)
        run_all(cuda_api, oracle, data, f"digit path x{per_line}", tools=("af", "hwe", "md", "vc"))
        run_all(cuda_api, oracle, data, f"digit path x{per_line} small tiles", tile_bytes=4096, tools=("af",))
        for path, fmt in ((oracle.AC_UNIFIED, oracle.AC_AGGREGATE),):
            if per_line == 0:                      # (allele_counter's reference loops forever on bytes outside [0-9./|:]: no oracle there)
                o = oracle.allele_counter(data, path, fmt)
                r = cuda_api.allele_counter(data, path, fmt)
                _cmp(f"digit path ac -a x{per_line}", r.out, o.out)
    # one odd genotype at every offset of a 2 KiB stretch: each position relative to the 512-byte windows and the lanes
    line_hdr = b"##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + b"\t".join(b"S%d" % i for i in range(700)) + b"\n"
    body = []
    for k in range(700):
        gts = [b"0|1", b"1/1", b".", b"0", b"./."] * 140
        gts[k] = [b"10|1", b"0|1:5", b"1.", b"11"][k % 4]
        body.append(b"1\t%d\t.\tA\tG\t.\tPASS\t.\tGT\t" % (k + 1) + b"\t".join(gts))
    data = line_hdr + b"\n".join(body) + b"\n"
    run_all(cuda_api, oracle, data, "digit path, one odd genotype at every offset", tools=("af",))


def test_indexer_cases(cuda_api, oracle):
    """VCFX_indexer: CHROM / POS as the two modes read them, and byte offsets that must be absolute — across tiles, across
    the chunks of the streaming path, and beyond 4 GiB (a chunk submitted with a large file_offset)."""
    import golden_util
    data, _ = golden_util.load()["ix_quirks"]
    for kw in ({}, {"tile_bytes": 512}, {"chunk_bytes": 4096}):
        run_all(cuda_api, oracle, data, f"ix quirks {kw}", tools=("ix",), **kw)
    data = synth.make_vcf(2, 3000, 40, seed=77)
    run_all(cuda_api, oracle, data, "ix chunks", chunk_bytes=64 << 10, tools=("ix",))
    # one chunk far into a large file: the offsets are the chunk's plus 5 GiB
    api = cuda_api
    body = data[api.find_chrom_header(data):]
    base = 5 << 30
    ctx = api.Context(api.OP_INDEX, api.FILE, chunk_bytes=1 << 20)
    buf, cap = ctx.acquire()
    import ctypes as C
    C.memmove(buf, body, len(body))
    ctx.submit(len(body), valid_from=0, is_final=True, file_offset=base)
    out, st, _ = ctx.next_output()
    ctx.close()
    exp = oracle.indexer(data, 0).out.split(b"\n")[1:-1]
    got = out.split(b"\n")[:-1]
    shift = base - api.find_chrom_header(data)
    assert len(got) == len(exp) == 3000
    for g, e in zip(got, exp):
        c1, p1, o1 = g.split(b"\t"); c2, p2, o2 = e.split(b"\t")
        assert (c1, p1) == (c2, p2) and int(o1) == int(o2) + shift


def test_nonref_filter_cases(cuda_api, oracle):
    """VCFX_nonref_filter: the two meanings of "definitely hom-ref" (file mode: three bytes must be 0/0 or 0|0; stdin mode: nothing
    but 0 / |), empty columns, GT not the first key, a final tab, CRLF, lines in front of the header, all-hom-ref lines of every
    length against the 512-byte windows."""
    import golden_util
    data, _ = golden_util.load()["nr_quirks"]
    for kw in ({}, {"tile_bytes": 512}, {"chunk_bytes": 4096}):
        run_all(cuda_api, oracle, data, f"nr quirks {kw}", tools=("nr",), **kw)
    hdr = b"##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t"
    # GT not the first key: a column that is just "0|0" has no GT piece at all — not hom-ref, the line stays (found by fuzzing)
    data = hdr + b"S1\tS2\n" + b"".join(b"1\t%d\t.\tT\tG\t.\tq10\tDP=3;\t%s\t%s\t%s\n" % (k + 1, f, a, b2) for k, (f, a, b2) in enumerate(
        [(b"DP:GQ:GT", b"0|0", b"0/1:35:0/0"), (b"DP:GQ:GT", b"3:35:0/0", b"0/0"), (b"DP:GT", b"0/0", b"0|0"), (b"DP:GT", b"1:0/0", b"2:0|0"),
         (b"GT:DP", b"0|0", b"0/0:3"), (b"DP:GT", b"0/0:0/0", b"0|0:0|0")]))
    for kw in ({}, {"tile_bytes": 512}):
        run_all(cuda_api, oracle, data, f"nr GT not first {kw}", tools=("nr", "pc", "gq", "ds"), **kw)
    for S in (1, 2, 100, 126, 127, 128, 129, 255, 256, 257, 700):
        names = b"\t".join(b"S%d" % i for i in range(S))
        lines = []
        for k in range(60):
            gts = [b"0|0" if (i + k) % 3 else b"0/0" for i in range(S)]
            if k % 4 == 1:
                gts[(k * 37) % S] = [b"0|1", b".", b"0", b"./.", b"0/0/0", b"000", b"1"][k % 7]
            lines.append(b"1\t%d\t.\tA\tG\t.\tPASS\t.\tGT\t" % (k + 1) + b"\t".join(gts))
        data = hdr + names + b"\n" + b"\n".join(lines) + (b"\n" if S % 2 else b"")
        run_all(cuda_api, oracle, data, f"nr S{S}", tools=("nr",))
        run_all(cuda_api, oracle, data, f"nr S{S} tile512", tile_bytes=512, tools=("nr",))


def test_phase_checker_cases(cuda_api, oracle):
    """VCFX_phase_checker: what "fully phased" means, empty columns, GT not the first key / no GT key, short lines, CRLF, lines in
    front of the header, file mode's FORMAT cache that starts as ("", GT first); every dropped line with the message the tool
    prints for it; all-phased lines of every length against the 512-byte windows; -q prints nothing."""
    import golden_util
    for name in ("pc_quirks", "pc_format_cache", "nr_quirks"):
        data, _ = golden_util.load()[name]
        for kw in ({}, {"tile_bytes": 512}, {"chunk_bytes": 4096}):
            run_all(cuda_api, oracle, data, f"{name} {kw}", tools=("pc",), **kw)
    # the FORMAT cache across chunk borders: no non-empty FORMAT for the first chunks
    hdr = b"##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t"
    lines = [b"1\t%d\t.\tA\tG\t.\tPASS\t.\t\t%s\t1|0" % (k + 1, [b"0|1", b"0/1", b"1|1:7"][k % 3]) for k in range(200)]
    lines += [b"1\t900\t.\tA\tG\t.\tPASS\t.\tGT\t0|1\t1|0"] + lines[:50]
    data = hdr + b"S1\tS2\n" + b"\n".join(lines) + b"\n"
    for kw in ({}, {"chunk_bytes": 1024}, {"tile_bytes": 512}):
        run_all(cuda_api, oracle, data, f"pc format cache {kw}", tools=("pc",), **kw)
    assert cuda_api.phase_checker(data, 0, quiet=True).err == b""
    for S in (1, 2, 100, 126, 127, 128, 129, 255, 256, 257, 700):
        names = b"\t".join(b"S%d" % i for i in range(S))
        lines = []
        for k in range(60):
            gts = [b"0|1" if (i + k) % 3 else b"1|0" for i in range(S)]
            if k % 4 == 1:
                gts[(k * 37) % S] = [b"0/1", b".", b"0", b".|.", b"0|1|1", b"0|.", b"10|11"][k % 7]
            lines.append(b"%d\t%d\t.\tA\tG\t.\tPASS\t.\tGT\t" % (k % 22 + 1, k + 1) + b"\t".join(gts))
        data = hdr + names + b"\n" + b"\n".join(lines) + (b"\n" if S % 2 else b"")
        run_all(cuda_api, oracle, data, f"pc S{S}", tools=("pc",))
        run_all(cuda_api, oracle, data, f"pc S{S} tile512", tile_bytes=512, tools=("pc",))


def pc_dropped_lines_input():
    """(input, lines phase_checker drops): 2^20 + 5000 short lines, more than the first event list holds."""
    hdr = b"##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tA\n"
    n = (1 << 20) + 5000
    return hdr + b"1\t2\n" * n + b"1\t7\t.\tA\tG\t.\t.\t.\tGT\t0|1\n", n


def test_phase_checker_more_dropped_lines_than_the_event_list(cuda_api, oracle):
    """Every dropped line is reported; the list starts with room for 2^20 of them and the chunk is run again with a longer
    one when that is not enough."""
    data, n = pc_dropped_lines_input()
    r = cuda_api.phase_checker(data, 0)
    o = oracle.phase_checker(data, 0)
    assert r.out == o.out and r.totals.flagged == n
    assert r.err == b"Warning: Invalid VCF line with fewer than 10 columns; skipping line.\n" * n


def test_dosage_calculator_cases(cuda_api, oracle):
    """VCFX_dosage_calculator: the quirks fixture; lines on the four-byte lattice of every length and phase with samples that
    leave it; several chunks and tiny tiles; the run that ends at a data line in front of the header."""
    import golden_util
    data, _ = golden_util.load()["ds_quirks"]
    for kw in ({}, {"tile_bytes": 512}, {"chunk_bytes": 4096}):
        run_all(cuda_api, oracle, data, f"ds quirks {kw}", tools=("ds",), **kw)
    hdr = b"##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t"
    for S in (1, 2, 100, 126, 127, 128, 129, 255, 256, 257, 700):
        lines = []
        for k in range(48):
            gts = [[b"0|1", b"1|1", b"0/0", b"2|0", b"./."][(i * 7 + k) % 5] for i in range(S)]
            if k % 4 == 1:
                gts[(k * 37) % S] = [b"0", b".", b"0/1/1", b"0|1:3", b"10|1", b"", b" 0|1"][k % 7]
            lines.append(b"%d\t%d\t%s\tA\tG\t.\tPASS\t.\tGT\t" % (k % 22 + 1, 10 ** (k % 7), b"r" * (k % 5)) + b"\t".join(gts))
        data = hdr + b"\t".join(b"S%d" % i for i in range(S)) + b"\n" + b"\n".join(lines) + (b"\n" if S % 2 else b"")
        run_all(cuda_api, oracle, data, f"ds S{S}", tools=("ds",))
        run_all(cuda_api, oracle, data, f"ds S{S} tile512", tile_bytes=512, tools=("ds",))
    for data in (b"##f\n1\t1\t.\tA\tG\t.\t.\t.\tGT\t0/1\n" + hdr + b"S1\n", hdr + b"S1\n", b"", b"\n", b"##f\n"):
        run_all(cuda_api, oracle, data, "ds stream edges", tools=("ds",))


def test_genotype_query_cases(cuda_api, oracle):
    """VCFX_genotype_query: flexible and strict queries (also ones the reference's parser gives up on half way), the quirks
    fixture, lines on the four-byte lattice of every length where only the LAST sample — or none — has the genotype."""
    import golden_util
    data, _ = golden_util.load()["gq_quirks"]
    for kw in ({}, {"tile_bytes": 512}, {"chunk_bytes": 4096}):
        for mode in MODES:
            for q, strict in (("0/1", False), ("1/0", False), ("0|1", True), ("1/1", False), ("0/x", False), ("x/0", False), ("./.", True), ("./.", False),
                              ("10/1", False), ("0/01", False), ("0", True), ("1/0:4", True), ("0/1\r", True)):
                r = cuda_api.genotype_query(data, q, mode, strict, **kw); o, e = oracle.genotype_query(data, q, mode, strict)
                _cmp(f"gq quirks {kw} mode{mode} {q!r} strict{strict}", r.out, o.out)
                _cmp(f"gq quirks {kw} mode{mode} {q!r} strict{strict} stderr", r.err, e)
    hdr = b"##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t"
    for S in (1, 2, 100, 127, 128, 129, 256, 257, 700):
        lines = []
        for k in range(40):
            gts = [b"0|0" if (i + k) % 3 else b"0/0" for i in range(S)]
            if k % 3 == 1:
                gts[-1] = [b"0|1", b"1/0", b"1|1", b"0/1:5", b"01/0"][k % 5]
            if k % 7 == 3:
                gts[(k * 11) % S] = b"1|0"
            lines.append(b"%d\t%d\t%s\tA\tG\t.\tPASS\t.\tGT\t" % (k % 22 + 1, 10 ** (k % 6), b"r" * (k % 4)) + b"\t".join(gts))
        data = hdr + b"\t".join(b"S%d" % i for i in range(S)) + b"\n" + b"\n".join(lines) + (b"\n" if S % 2 else b"")
        run_all(cuda_api, oracle, data, f"gq S{S}", tools=("gq",))
        run_all(cuda_api, oracle, data, f"gq S{S} tile512", tile_bytes=512, tools=("gq",))
    # the run ends at a data line in front of the header; '#' lines behind the last data line (stdin mode drops them)
    for data in (b"##f\n1\t1\t.\tA\tG\t.\t.\t.\tGT\t0/1\n" + hdr + b"S1\n1\t1\t.\tA\tG\t.\t.\t.\tGT\t0/1\n",
                 hdr + b"S1\n1\t1\t.\tA\tG\t.\t.\t.\tGT\t0/1\n#a\n\n#b\n", hdr + b"S1\n#only\n", b"##f\n#x\n", b"", b"\n\n"):
        run_all(cuda_api, oracle, data, "gq stream edges", tools=("gq",))


def test_inbreeding_calculator_cases(cuda_api, oracle):
    """VCFX_inbreeding_calculator: what a genotype code is, lines with fewer columns than samples (the file mode takes the code
    of the last line that had the column), multi-allelic / empty ALT, two "#CHROM" lines, every option; sums that need the
    sites in file order (thousands of sites, hundreds of samples, several chunks and tiny tiles); two streams through one
    context one after the other."""
    import golden_util
    data, _ = golden_util.load()["ib_quirks"]
    for kw in ({}, {"tile_bytes": 512}, {"chunk_bytes": 4096}):
        for mode in MODES:
            for fl in range(8):
                r = cuda_api.inbreeding_calculator(data, mode, bool(fl & 1), bool(fl & 2), bool(fl & 4), quiet=False, **kw)
                o = oracle.inbreeding(data, mode, fl)
                _cmp(f"ib quirks {kw} mode{mode} flags{fl}", r.out, o.out)
                assert r.err == oracle.IB_MESSAGES[o.warnings]
    for shape, V, S in ((2, 3000, 300), (3, 2000, 257), (4, 300, 64), (2, 40, 2504)):
        data = synth.make_vcf(shape, V, S, seed=40 + shape)
        run_all(cuda_api, oracle, data, f"ib shape{shape}", tools=("ib",))
        run_all(cuda_api, oracle, data, f"ib shape{shape} chunks", chunk_bytes=1 << 20 if S > 1000 else 64 << 10, tools=("ib",))
    run_all(cuda_api, oracle, synth.make_vcf(3, 400, 100, seed=77), "ib tile512", tile_bytes=512, tools=("ib",))
    # lines on the four-byte lattice (d|d + tab) of every length and phase against the 512-byte windows, a sample that leaves
    # the lattice here and there (the rest of such a line goes tab by tab), three-byte samples that are not genotypes
    hdr9 = b"##f\n#CHROM\tP\tI\tR\tA\tQ\tF\tI\tFORMAT\t"
    for S in (100, 126, 127, 128, 129, 255, 256, 257, 700):
        lines = []
        for k in range(48):
            gts = [[b"0|1", b"1|1", b"0/0", b"1|0"][(i * 7 + k) % 4] for i in range(S)]
            if k % 4 == 1:
                gts[(k * 37) % S] = [b"0", b".", b"./.", b"0|1:3", b"10|1", b"2|1", b" 0|1"][k % 7]
            lines.append(b"%d\t%d\t%s\tA\tG\t.\tPASS\t.\tGT\t" % (k % 22 + 1, 10 ** (k % 7), b"r" * (k % 5)) + b"\t".join(gts))
        data = hdr9 + b"\t".join(b"S%d" % i for i in range(S)) + b"\n" + b"\n".join(lines) + (b"\n" if S % 2 else b"")
        run_all(cuda_api, oracle, data, f"ib lattice S{S}", tools=("ib",))
        run_all(cuda_api, oracle, data, f"ib lattice S{S} tile512", tile_bytes=512, tools=("ib",))
    # thousands of samples in the header, two columns on most lines: more rows x samples than the panels were sized for — the
    # chunk is run again with larger ones, and the chunks behind it (already launched) wait their turn and are run again too
    data = ib_few_columns_input()
    for kw in ({"chunk_bytes": 16 << 10}, {}):
        run_all(cuda_api, oracle, data, f"ib few columns {kw}", tools=("ib",), **kw)
    # a context is good for one stream after the other: the sums start again behind a final chunk
    a = synth.make_vcf(3, 200, 20, seed=5); b = synth.make_vcf(2, 150, 20, seed=6)
    names = [b"S%d" % i for i in range(20)]

    def body(d):
        return d[cuda_api._ib_header(d, 0)[1]:]
    ctx = cuda_api.Context(cuda_api.OP_INBREEDING, cuda_api.FILE, chunk_bytes=1 << 20, sel_cols=list(range(20)), sel_names=names)
    for d in (a, b, a):
        outs, _ = cuda_api.stream_bytes(ctx, body(d), 16 << 10)
        exp = oracle.inbreeding(d, 0, 0).out
        got = cuda_api.IB_HEADER + b"".join(outs)
        # (the names of the synthetic header are not S0..S19: compare the numbers)
        assert [l.split(b"\t")[1] for l in got.splitlines()[1:]] == [l.split(b"\t")[1] for l in exp.splitlines()[1:]]
    ctx.close()


def ib_few_columns_input():
    S = 4000
    hdr = b"##f\n#CHROM\tP\tI\tR\tA\tQ\tF\tI\tFORMAT\t" + b"\t".join(b"N%d" % i for i in range(S)) + b"\n"
    g = [b"0/1", b"1/1", b"0/0", b"0|1", b"./."]
    lines = [b"1\t%d\t.\tA\tG\t.\t.\t.\tGT\t%s\t%s" % (k + 1, g[k % 5], g[(k * 3 + 1) % 5]) for k in range(2500)]
    lines[7] += b"\t" + b"\t".join(g[(j * 7) % 5] for j in range(S - 2))
    return hdr + b"\n".join(lines) + b"\n"


def two_digit_counts_input():
    hdr = b"##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tA\tB\tC\n"
    deca = b"/".join([b"0"] * 10)
    wrap = b"|".join([b"1"] * 130)
    body = b"".join(b"1\t%d\trs%d\tA\tG\t.\tPASS\t.\tGT\t0|1\t%s\t1/1\n" % (100 + i, i, deca if i % 7 == 3 else (wrap if i % 11 == 5 else b"0/0"))
                    for i in range(60))
    return hdr + body


def test_allele_counter_two_digit_counts(cuda_api, oracle):
    """allele_counter TEXT rows are sized without looking at the genotypes (one digit per count); a
    sample with ten or more alleles of a kind, or 128+ (int8 wrap to a negative number), breaks that
    guess: the write pass notices and the chunk is run again with exact sizes."""
    data = two_digit_counts_input()
    for kw in ({}, {"chunk_bytes": 4096}, {"tile_bytes": 512}):
        o = oracle.allele_counter(data)
        r = cuda_api.allele_counter(data, **kw)
        assert r.rc == o.rc
        _cmp(f"ac two-digit counts {kw}", r.out, o.out)
    # and the plain case right after it through a fresh context
    data2 = synth.make_vcf(2, 40, 64, seed=9)
    _cmp("ac after exact", cuda_api.allele_counter(data2).out, oracle.allele_counter(data2).out)


def more_rows_input():
    """130,000 lines of 36 bytes: more rows than the default record capacity of a 4 MiB chunk."""
    hdr = b"##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tA\tB\n"
    gts = [b"0|1", b"1|1", b"0|0", b"./.", b"1|0"]
    body = b"".join(b"1\t%d\t.\tA\tG\t.\t.\t.\tGT\t%s\t%s\n" % (i + 1, gts[i % 5], gts[(i * 7 + 3) % 5]) for i in range(130000))
    return hdr + body


def test_more_rows_than_the_default_record_capacity(cuda_api, oracle):
    """Row records are sized for one row per 256 input bytes (+64 Ki); a chunk of very short lines has
    more: the launch reports it and is repeated with the exact count (block-wise slot reservation
    included), through the streaming path and through several chunks."""
    data = more_rows_input()
    chunk = 4 << 20                                       # the slot's capacity is sized from the chunk size
    assert len(data) <= chunk and chunk // 256 + 65536 < 130000
    run_all(cuda_api, oracle, data, "many short lines, one 4 MiB chunk", chunk_bytes=chunk, tools=("af", "hwe", "md", "vc"))
    run_all(cuda_api, oracle, data, "many short lines, 1 MiB chunks", chunk_bytes=1 << 20, tools=("af", "md"))
