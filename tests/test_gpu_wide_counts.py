"""Exact per-variant counts on lines of 30,000 to 1,000,000 samples.

Past about 5,000 diploid samples allele_freq_calc's four-digit text stands for several alt counts, so a kernel that
drops or double-counts a sample can print the oracle's bytes.  Here the expected counts do not come from the oracle:
a numpy generator draws a genotype table (variants x samples), writes it out as VCF text and sums every token's
contribution, read once from the oracle on a one-sample line.  The AF rows are pinned to rounding edges of their mode's
formatter and the HWE cohorts are chosen where every one-sample move changes the p-value text, so the text is lossless
for the mistakes that matter; the test asserts that before any device run.

The lines are written four ways: on the lattice with one separator (tier 1, whose periodic flush folds the packed
16-bit sums every 32,768 samples), on the lattice with both separators (general kernel and exact path), GT-only with
tokens off the lattice (digit path) and as GT:AD:DP:GQ:PL (skip-ahead loop).  The ID column is 0 to 3 bytes long so
that the sample region shifts against the 512-byte windows, and the non-reference alleles sit where the kernel
changes state: around every flush point, in the first and last window of the line and at window borders.

Every case runs through the streaming path (default chunks and chunks of one to three lines), 512-byte tiles, and the
device-resident entry point with and without a line hint (without it the tiles are far smaller than the lines, and on
the 4 MB lines most tiles hold no line start).  test_emu_wide_counts.py runs the same checks at a few widths under the
warp emulator.
"""
import ctypes as C
import math
from dataclasses import dataclass
from functools import lru_cache

import numpy as np
import pytest

import test_gpu_parity as G
import test_gpu_resident as R

pytestmark = pytest.mark.gpu

FLUSH = 32768                  # 4-byte samples per flush of tier 1's packed sums: ITMAX = 64 iterations of 2 KiB
NEAR = (-128, -32, -31, -1, 1, 31, 32, 128)
WIDTHS = sorted({k * FLUSH + d for k in (1, 2, 3) for d in NEAR} | {100_000, 250_000, 1_000_000})
DECIDER_WIDTHS = (FLUSH + 1, 2 * FLUSH - 1, 3 * FLUSH + 32, 100_000, 250_000, 1_000_000)
AC_WIDTHS = (FLUSH - 31, 2 * FLUSH + 1, 3 * FLUSH - 128, 100_000, 250_000, 1_000_000)
IB_WIDTHS = (FLUSH + 128, 2 * FLUSH - 32, 100_000, 250_000)
MODES = (0, 1)

# ----------------------------------------------------------------------------- tokens
TOKENS = (b"0|0", b"0|1", b"1|0", b"1|1", b"0/0", b"0/1", b"1/0", b"1/1", b".", b"./.", b"0", b"1", b"2|1", b"10|1", b"0|1:5")
TI = {t: i for i, t in enumerate(TOKENS)}
LAT = np.array([[[TI[b"%d%s%d" % (a, s, b)] for b in (0, 1)] for a in (0, 1)] for s in (b"|", b"/")])   # [sep, a, b]
MK_FORMAT, MK_SUFFIX = b"GT:AD:DP:GQ:PL", b":3,4:7:50:0,10,100"
# tokens off the lattice each encoding mixes in, and how often
ODD = {"tier1": ((), 0.0), "mixed": ((b"10|1", b"0|1:5"), 2e-4), "digits": ((b".", b"./.", b"0", b"1", b"2|1"), 0.08),
       "multikey": ((b"./.", b"."), 0.01)}
ENCODINGS = tuple(ODD)
GQ_QUERY = {0: "0/1", 1: "1/1"}                       # (non-strict, as test_gpu_resident.GQ_QUERIES)
H1 = b"##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tS0\n"


def one_sample_line(tok, fmt=b"GT"):
    return b"1\t100\trs1\tA\tG\t.\tPASS\t.\t%s\t%s\n" % (fmt, tok + (MK_SUFFIX if fmt == MK_FORMAT else b""))


@dataclass
class Tokens:
    """What one token adds, read from the oracle: AF alt / total, HWE class (= inbreeding code: the two parse a sample
    alike), allele_counter ref / alt, dosage code per FORMAT (-1 "NA"), and per mode whether a one-sample line with it is
    kept by nonref_filter / phase_checker / genotype_query and rewritten by missing_detector."""
    af_alt: np.ndarray
    af_tot: np.ndarray
    hwe: np.ndarray
    ac_ref: np.ndarray
    ac_alt: np.ndarray
    ds: dict
    keep: dict                                          # (tool, mode) -> bool array


@lru_cache(maxsize=None)
def _tokens(O):
    l = O.lib()
    n = len(TOKENS)
    af_alt, af_tot, ac_ref, ac_alt, hwe = (np.zeros(n, np.int64) for _ in range(5))
    for i, t in enumerate(TOKENS):
        a, b = C.c_int(0), C.c_int(0)
        g = t.split(b":")[0]                            # both tools count the GT piece (GT is the first key here)
        l.oracle_af_counts(g, len(g), C.byref(a), C.byref(b))
        af_alt[i], af_tot[i] = a.value, b.value
        l.oracle_ac_counts(g, len(g), C.byref(a), C.byref(b))
        ac_ref[i], ac_alt[i] = a.value, b.value
        hwe[i] = l.oracle_hwe_class(t, len(t))
    ds = {}
    for fmt in (b"GT", MK_FORMAT):
        codes = []
        for t in TOKENS:
            row = O.dosage(H1 + one_sample_line(t, fmt), 0).out.split(b"\n")[1]
            v = row.rsplit(b"\t", 1)[1]
            codes.append(-1 if v == b"NA" else int(v))
        ds[fmt] = np.array(codes, np.int64)
    keep = {}
    for mode in MODES:
        k = {"nr": [], "pc": [], "gq": [], "md": []}
        for t in TOKENS:
            L = one_sample_line(t)
            k["nr"].append(O.nonref_filter(H1 + L, mode).out.endswith(L))
            k["pc"].append(O.phase_checker(H1 + L, mode).out.endswith(L))
            k["gq"].append(O.genotype_query(H1 + L, GQ_QUERY[mode], mode)[0].out.endswith(L))
            k["md"].append(O.missing(H1 + L, mode).out != H1 + L)
        for tool, v in k.items():
            keep[tool, mode] = np.array(v)
    return Tokens(af_alt, af_tot, hwe, ac_ref, ac_alt, ds, keep)


def serialise(ids, texts):
    """b"\\t".join(texts[i] for i in ids), vectorised."""
    lens = np.array([len(t) + 1 for t in texts], np.int64)
    blob = np.frombuffer(b"".join(t + b"\t" for t in texts), np.uint8)
    offs = np.cumsum(lens) - lens
    L = lens[ids]
    ends = np.cumsum(L)
    idx = np.repeat(offs[ids] - (ends - L), L) + np.arange(int(ends[-1]))
    return blob[idx[:-1]].tobytes()


@lru_cache(maxsize=8)
def header(W):
    return (b"##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t"
            + b"\t".join(b"S%d" % i for i in range(W)) + b"\n")


def hot_mask(W):
    """Samples where the kernel changes state: the first and last 160 (a 512-byte window, plus the header's share of
    the first one), ~1,200 around every flush point, and the two on each side of every 128-sample window border."""
    i = np.arange(W)
    m = (i < 160) | (i >= W - 160) | np.isin(i % 128, (0, 1, 126, 127))
    for c in range(FLUSH, W, FLUSH):
        m |= (i >= c - 512) & (i < c + 672)
    return m


# ----------------------------------------------------------------------------- rows whose text is lossless
def af_text(O, mode, alt, tot):
    return O.fmt("af_file" if mode == 0 else "af_stdin", alt / tot if tot > 0 else 0.0)


def p_text(O, mode, hr, het, ha):
    return O.fmt("p_file" if mode == 0 else "p_stdin", O.hwe_pvalue(hr, het, ha))


def pin_alt(O, mode, tot, start, edge):
    """The first alt count from `start` on that sits on a rounding edge of the mode's AF text: at a lower edge alt - 1
    and alt / (tot + 2) print differently, at an upper edge alt + 1 and alt / (tot - 2) do.  The search only goes up:
    the row reaches the count by adding alt alleles, never by taking them away."""
    a = start
    while True:
        s = af_text(O, mode, a, tot)
        if edge == "lo" and af_text(O, mode, a - 1, tot) != s and af_text(O, mode, a, tot + 2) != s:
            return a
        if edge == "hi" and af_text(O, mode, a + 1, tot) != s and af_text(O, mode, a, tot - 2) != s:
            return a
        a += 1


def assert_af_lossless(O, mode, alt, tot, edge, tag):
    s = af_text(O, mode, alt, tot)
    if edge == "lo":
        assert af_text(O, mode, alt - 1, tot) != s, (tag, "alt - 1 prints the same", alt, tot)
        assert af_text(O, mode, alt, tot + 2) != s, (tag, "one more hom-ref sample prints the same", alt, tot)
    else:
        assert af_text(O, mode, alt + 1, tot) != s, (tag, "alt + 1 prints the same", alt, tot)
        assert af_text(O, mode, alt, tot - 2) != s, (tag, "one hom-ref sample less prints the same", alt, tot)


def assert_hwe_sensitive(O, mode, c, tag):
    """Every move of one sample from one class to another, and one sample more or less in any class, changes the text."""
    s = p_text(O, mode, *c)
    for i in range(3):
        for d in (-1, 1):
            m = list(c); m[i] += d
            assert p_text(O, mode, *m) != s, (tag, "one sample more / less", c, m)
        for j in range(3):
            if i != j:
                m = list(c); m[i] -= 1; m[j] += 1
                assert p_text(O, mode, *m) != s, (tag, "one sample moved", c, m)


@dataclass
class Row:
    enc: str
    ids: np.ndarray            # token per sample
    text: bytes                # the line, without '\n'
    edge: str = ""


def _row_text(k, id_len, fmt, samples):
    return b"%d\t%d\t%s\tA\tG\t.\tPASS\t.\t%s\t" % (k % 22 + 1, 1000 + k, b"rs7"[:id_len], fmt) + samples


def draw_row(O, tab, mode, enc, W, edge, rng, k):
    """One line of W samples in encoding `enc`, its AF count pinned to `edge` of the mode's formatter and its HWE cohort
    at a moderate chi-square (2 to 6, either sign of the deviation)."""
    hot = hot_mask(W)
    q = rng.uniform(0.6, 0.85)
    F = rng.choice((-1.0, 1.0)) * math.sqrt(rng.uniform(2.0, 6.0) / W)
    het = int(round(2 * q * (1 - q) * (1 - F) * W))
    ha = int(round((q * q + F * q * (1 - q)) * W))
    cls = np.repeat(np.array([0, 1, 2]), [W - het - ha, het, ha])
    rng.shuffle(cls)
    # the non-reference alleles where the kernel changes state
    h0, c1 = np.flatnonzero(hot & (cls == 0)), np.flatnonzero(~hot & (cls != 0))
    m = min(len(h0), len(c1))
    cls[h0[:m]], cls[c1[:m]] = cls[c1[:m]], 0
    cls[0] = cls[-1] = 2
    a = (cls == 2) | ((cls == 1) & (rng.random(W) < 0.5))
    b = (cls == 2) | ((cls == 1) & ~a)
    sep = rng.integers(0, 2, W) if enc == "mixed" else np.full(W, k % 2)
    pool, rate = ODD[enc]
    odd = np.zeros(W, bool)
    odd_ids = np.zeros(W, np.int64)
    if pool:
        odd = rng.random(W) < rate
        odd[[0, -1]] = False
        if enc == "mixed":                                   # every line leaves the lattice at least twice
            odd[rng.integers(1, W - 1, 2)] = True
        odd_ids[odd] = rng.choice([TI[t] for t in pool], int(odd.sum()))

    def ids():
        return np.where(odd, odd_ids, LAT[sep, a.astype(int), b.astype(int)])
    x = ids()
    alt, tot = int(tab.af_alt[x].sum()), int(tab.af_tot[x].sum())
    want = pin_alt(O, mode, tot, alt, edge)
    # reach it by turning first alleles of lattice samples away from the hot spots 0 -> 1 (each adds one alt allele)
    free = ~hot & ~odd
    free[[0, -1]] = False
    cand = np.flatnonzero(free & ~a)
    assert want - alt <= len(cand), (enc, W, want, alt)
    a[rng.choice(cand, want - alt, replace=False)] = True
    x = ids()
    assert int(tab.af_alt[x].sum()) == want and int(tab.af_tot[x].sum()) == tot
    fmt = MK_FORMAT if enc == "multikey" else b"GT"
    texts = [t + MK_SUFFIX for t in TOKENS] if enc == "multikey" else list(TOKENS)
    return Row(enc, x, _row_text(k, (k + W) % 4, fmt, serialise(x, texts)), edge)


@dataclass
class Wide:
    W: int
    mode: int                  # the mode whose formatters the rows are pinned for
    rows: list
    data: bytes


def encodings_for(W):
    return ENCODINGS if W <= 250_000 else ("tier1", "digits")


@lru_cache(maxsize=2)
def wide_input(O, W, mode, encodings=None):
    """Per encoding a row at a lower and at an upper edge (the 22-byte multi-key samples: one, alternating with W)."""
    tab = _tokens(O)
    rng = np.random.default_rng(W * 2 + mode)
    rows = []
    for enc in encodings or encodings_for(W):
        edges = ("lo", "hi") if enc != "multikey" else (("lo", "hi")[(W + mode) % 2],)
        for edge in edges:
            rows.append(draw_row(O, tab, mode, enc, W, edge, rng, len(rows)))
    return Wide(W, mode, rows, header(W) + b"".join(r.text + b"\n" for r in rows))


def counts(tab, row):
    cls = tab.hwe[row.ids]
    return (int(tab.af_alt[row.ids].sum()), int(tab.af_tot[row.ids].sum()),
            (int((cls == 0).sum()), int((cls == 1).sum()), int((cls == 2).sum())))


def self_check(O, wide):
    """The generator still gives lossless rows: fails before any device run when it drifts."""
    tab = _tokens(O)
    for k, row in enumerate(wide.rows):
        alt, tot, c = counts(tab, row)
        tag = f"W{wide.W} mode{wide.mode} row{k} {row.enc}"
        assert_af_lossless(O, wide.mode, alt, tot, row.edge, tag)
        assert_hwe_sensitive(O, wide.mode, c, tag)


def expected_af_hwe(O, api, wide):
    """allele_freq_calc's and hwe_tester's stdout from the numpy counts."""
    tab = _tokens(O)
    af, hwe = [api.AF_HEADER], [api.HWE_HEADER]
    for row in wide.rows:
        alt, tot, c = counts(tab, row)
        lead = b"\t".join(row.text.split(b"\t", 5)[:5]) + b"\t"
        af.append(lead + af_text(O, wide.mode, alt, tot) + b"\n")
        hwe.append(lead + p_text(O, wide.mode, *c) + b"\n")
    return b"".join(af), b"".join(hwe)


# ----------------------------------------------------------------------------- geometries
def longest_line(data):
    return max(len(l) for l in data.split(b"\n")) + 1


def stream_kw(data):
    """Default chunks, chunks of one to three lines, 512-byte tiles."""
    return ({}, {"chunk_bytes": 2 * longest_line(data) + 64}, {"tile_bytes": 512})


def resident_geoms(data):
    """(tile_bytes, line hint): default tiles without a hint (much smaller than the lines) and with one, 512-byte tiles."""
    return ((0, None), (0, longest_line(data)), (512, None))


def run_resident_jobs(api, O, mem, data, mode, ops, tag):
    """Each job of test_gpu_resident.jobs through vcfx_cuda_run_device at every resident geometry: compared with the
    oracle, or with the streaming path where the tool has host rules or the oracle has no answer."""
    ran = []
    for job in R.jobs(api, O, data, mode, ops):
        want = job.expect() if job.expect else None
        stream = R.streamed(api, job, R.chunk_info(api, job.op, mode, job.data)) if want is None else None
        for tile, hint in resident_geoms(data):
            got = R.run_resident(mem, api, job.op, mode, job.data, tile_bytes=tile, line_hint=hint, ctx_kw=job.ctx_kw)
            R.check(api, job, f"{tag} tile{tile} hint{hint}", got, stream, want)
        ran.append(job.name)
    return ran


# ----------------------------------------------------------------------------- 1. AF and HWE
def check_af_hwe(api, O, mem, W, encodings=None):
    for mode in MODES:
        wide = wide_input(O, W, mode, encodings)
        self_check(O, wide)
        data = wide.data
        exp_af, exp_hwe = expected_af_hwe(O, api, wide)
        o_af, o_hwe = O.allele_freq(data, mode), O.hwe(data, mode)
        G._cmp(f"W{W} mode{mode} oracle af vs numpy", o_af.out, exp_af)
        G._cmp(f"W{W} mode{mode} oracle hwe vs numpy", o_hwe.out, exp_hwe)
        for kw in stream_kw(data):
            r = api.allele_freq_calc(data, mode, **kw)
            G._cmp(f"W{W} af mode{mode} {kw}", r.out, exp_af)
            assert r.totals.rows == len(wide.rows)
            G._cmp(f"W{W} hwe mode{mode} {kw}", api.hwe_tester(data, mode, **kw).out, exp_hwe)
        assert run_resident_jobs(api, O, mem, data, mode, ("af", "hwe"), f"W{W}") == ["af", "hwe"]


@pytest.fixture
def mem():
    return R.TorchMem()


@pytest.mark.parametrize("W", WIDTHS)
def test_af_hwe_counts_at_width(cuda_api, oracle, mem, W):
    check_af_hwe(cuda_api, oracle, mem, W)


# ----------------------------------------------------------------------------- 2. allele_counter, dosage, inbreeding
def ac_selection(W):
    """Column 0, the last column and (where the line has them) columns above 65,535, in mixed order."""
    cols = [W - 1, 0, W // 2] + ([65_536, W - 2] if W > 65_537 else [])
    return cols, " ".join(f"S{c}" for c in cols)


def check_allele_counter(api, O, mem, W):
    tab = _tokens(O)
    wide = wide_input(O, W, 0)
    data = wide.data
    lead = [b"\t".join(r.text.split(b"\t", 5)[:5]) + b"\t" for r in wide.rows]
    # -a: per line the sums over every sample, as integers
    exp = api.AC_AGG_HEADER + b"".join(l + b"%d\t%d\t%d\n" % (tab.ac_ref[r.ids].sum(), tab.ac_alt[r.ids].sum(), W)
                                         for l, r in zip(lead, wide.rows))
    G._cmp(f"W{W} ac -a oracle vs numpy", O.allele_counter(data, O.AC_UNIFIED, O.AC_AGGREGATE).out, exp)
    for kw in stream_kw(data):
        r = api.allele_counter(data, api.AC_UNIFIED, api.AC_AGGREGATE, **kw)
        got = [tuple(map(int, l.split(b"\t")[5:])) for l in r.out.splitlines()[1:]]
        assert got == [(int(tab.ac_ref[x.ids].sum()), int(tab.ac_alt[x.ids].sum()), W) for x in wide.rows], (W, kw)
        G._cmp(f"W{W} ac -a {kw}", r.out, exp)
    # TEXT (both paths) and -b with a selection
    cols, sel = ac_selection(W)
    for path in (api.AC_MT_TEXT, api.AC_STREAM):
        # the stream path walks the columns forward only: a selected column left of the one it stands on reads that one
        at = np.maximum.accumulate(cols) if path == api.AC_STREAM else cols
        exp = api.AC_TEXT_HEADER + b"".join(l + b"S%d\t%d\t%d\n" % (c, tab.ac_ref[r.ids[x]], tab.ac_alt[r.ids[x]])
                                              for l, r in zip(lead, wide.rows) for c, x in zip(cols, at))
        G._cmp(f"W{W} ac path{path} oracle vs numpy", O.allele_counter(data, path, O.AC_TEXT, 0, sel).out, exp)
        for kw in stream_kw(data):
            G._cmp(f"W{W} ac path{path} {sel} {kw}", api.allele_counter(data, path, api.AC_TEXT, 0, sel, **kw).out, exp)
    o = O.allele_counter(data, O.AC_UNIFIED, O.AC_BINARY, 0, sel)
    assert o.rc == 0
    for kw in stream_kw(data):
        G._cmp(f"W{W} ac -b {sel} {kw}", api.allele_counter(data, api.AC_UNIFIED, api.AC_BINARY, 0, sel, **kw).out, o.out)
    assert run_resident_jobs(api, O, mem, data, 0, ("ac path2",), f"W{W}") == ["ac path2 fmt1", "ac path2 fmt2"]


@pytest.mark.parametrize("W", AC_WIDTHS)
def test_allele_counter_at_width(cuda_api, oracle, mem, W):
    check_allele_counter(cuda_api, oracle, mem, W)


def check_dosage(api, O, mem, W):
    tab = _tokens(O)
    for mode in MODES:
        wide = wide_input(O, W, mode)
        data = wide.data
        codes = np.stack([tab.ds[MK_FORMAT if r.enc == "multikey" else b"GT"][r.ids] for r in wide.rows])
        lead = [b"\t".join(r.text.split(b"\t", 5)[:5]) + b"\t" for r in wide.rows]
        txt = [b"NA", b"0", b"1", b"2"]
        exp = api.DS_HEADER + b"".join(l + b",".join(txt[c + 1] for c in row) + b"\n" for l, row in zip(lead, codes.tolist()))
        G._cmp(f"W{W} ds mode{mode} oracle vs numpy", O.dosage(data, mode).out, exp)
        for kw in stream_kw(data):
            G._cmp(f"W{W} ds mode{mode} {kw}", api.dosage_calculator(data, mode, **kw).out, exp)
            m = api.dosage_matrix(data, mode, **kw)
            assert m.codes.shape == (len(wide.rows), W) and np.array_equal(m.codes.numpy(), codes), (W, mode, kw)
        assert run_resident_jobs(api, O, mem, data, mode, ("ds",), f"W{W}") == ["ds"]
        if isinstance(mem, R.TorchMem):
            d_in = mem.input(data, api.DEVICE_PAD).t
            for hint in (0, longest_line(data)):
                m = api.dosage_matrix_device(d_in, len(data), mode, line_hint=hint)
                assert np.array_equal(m.codes.cpu().numpy(), codes), (W, mode, hint)


@pytest.mark.parametrize("W", AC_WIDTHS)
def test_dosage_at_width(cuda_api, oracle, mem, W):
    check_dosage(cuda_api, oracle, mem, W)


def ib_expected(O, api, W, code_rows):
    """The tool's text from numpy: per site, in file order, each sample's expected heterozygosity from the allele
    frequency of the other samples, summed in float64; F = 1 - het / sum, printed by the oracle's formatter."""
    s = np.zeros(W); het = np.zeros(W); used = np.zeros(W, np.int64)
    for code in code_rows:
        good = code >= 0
        n_good, alt_sum = int(good.sum()), int(code[good].sum())
        freq = (alt_sum - code[good]) / (2.0 * (n_good - 1))
        s[good] += 2.0 * freq * (1.0 - freq)
        het[good] += code[good] == 1
        used[good] += 1
    out = [api.IB_HEADER]
    for i in range(W):
        v = b"NA" if used[i] == 0 else (b"1.000000" if s[i] <= 0.0 else O.fmt("p_file", 1.0 - het[i] / s[i]))
        out.append(b"S%d\t%s\n" % (i, v))
    return b"".join(out)


def check_inbreeding(api, O, mem, W):
    tab = _tokens(O)
    for mode in MODES:
        wide = wide_input(O, W, mode)
        data = wide.data
        exp = ib_expected(O, api, W, [tab.hwe[r.ids] for r in wide.rows])
        G._cmp(f"W{W} ib mode{mode} oracle vs numpy", O.inbreeding(data, mode, 0).out, exp)
        for kw in stream_kw(data):
            G._cmp(f"W{W} ib mode{mode} {kw}", api.inbreeding_calculator(data, mode, **kw).out, exp)
        assert run_resident_jobs(api, O, mem, data, mode, ("ib",), f"W{W}")


@pytest.mark.parametrize("W", IB_WIDTHS)
def test_inbreeding_at_width(cuda_api, oracle, mem, W):
    check_inbreeding(cuda_api, oracle, mem, W)


# ----------------------------------------------------------------------------- 3. one deciding sample per line
DECIDERS = (b"1|1", b"0/0", b"0|1", b"./.")     # against a background of 0|0: each changes the verdict of some tools


def decider_positions(W):
    p = {0, 3, 4, 127, 128, 249_999, W - 1}
    for c in list(range(FLUSH, W, FLUSH))[:3] + [(W - 1) // FLUSH * FLUSH]:
        p |= {c - 1, c, c + 1}
    return sorted(x for x in p if 0 <= x < W)


@lru_cache(maxsize=2)
def decider_input(W):
    rows = []
    bg = TI[b"0|0"]
    for k, p in enumerate(decider_positions(W) + [None]):
        ids = np.full(W, bg, np.int64)
        if p is not None:
            ids[p] = TI[DECIDERS[k % len(DECIDERS)]]
        rows.append(Row("decider", ids, _row_text(k, k % 4, b"GT", serialise(ids, TOKENS))))
    return rows, header(W) + b"".join(r.text + b"\n" for r in rows)


def check_deciders(api, O, mem, W):
    tab = _tokens(O)
    rows, data = decider_input(W)
    hdr = header(W)
    for mode in MODES:
        keep = {t: [bool(tab.keep[t, mode][r.ids].any()) if t != "pc" else bool(tab.keep[t, mode][r.ids].all()) for r in rows]
                for t in ("nr", "pc", "gq", "md")}
        assert all(any(v) and not all(v) for v in keep.values()), keep     # every tool keeps some lines and drops others
        exp = {t: hdr + b"".join(r.text + b"\n" for r, k in zip(rows, keep[t]) if k) for t in ("nr", "pc", "gq")}
        G._cmp(f"W{W} nr mode{mode} oracle vs numpy", O.nonref_filter(data, mode).out, exp["nr"])
        G._cmp(f"W{W} pc mode{mode} oracle vs numpy", O.phase_checker(data, mode).out, exp["pc"])
        G._cmp(f"W{W} gq mode{mode} oracle vs numpy", O.genotype_query(data, GQ_QUERY[mode], mode)[0].out, exp["gq"])
        md = O.missing(data, mode).out if mode == 1 else None      # (file mode: no oracle on lines past 60,000 bytes)
        if md is not None:
            changed = [a != b for a, b in zip(md.split(b"\n")[2:], data.split(b"\n")[2:])]
            assert changed[:len(rows)] == keep["md"], (W, "md")
        for kw in stream_kw(data):
            G._cmp(f"W{W} nr mode{mode} {kw}", api.nonref_filter(data, mode, **kw).out, exp["nr"])
            G._cmp(f"W{W} pc mode{mode} {kw}", api.phase_checker(data, mode, quiet=True, **kw).out, exp["pc"])
            G._cmp(f"W{W} gq mode{mode} {kw}", api.genotype_query(data, GQ_QUERY[mode], mode, quiet=True, **kw).out, exp["gq"])
            r = api.missing_detector(data, mode, **kw)
            assert r.totals.flagged == sum(keep["md"]), (W, mode, kw)
            if md is not None:
                G._cmp(f"W{W} md mode{mode} {kw}", r.out, md)
        run_resident_jobs(api, O, mem, data, mode, ("md", "nr", "pc", "gq 0/1 strict0", "gq 1/1 strict0"), f"W{W} deciders")


@pytest.mark.parametrize("W", DECIDER_WIDTHS)
def test_deciding_sample_at_width(cuda_api, oracle, mem, W):
    check_deciders(cuda_api, oracle, mem, W)
