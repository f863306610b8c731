"""dosage_calculator's matrix mode (VCFX_OP_DOSAGE + VCFX_F_DS_MATRIX): the genotypes as an int8 variants x samples
matrix with 16 bytes of metadata per row, through the streaming path (api.dosage_matrix), the device-resident entry point
(vcfx_cuda_run_device) and the torch wrapper (api.dosage_matrix_device).

A matrix row is exactly the row dosage_calculator prints, in binary.  The central check rebuilds the tool's stdout from
the matrix and the input bytes (render) and compares it byte for byte with the oracle and with the text path; the
literal-codes case writes its expected matrix out instead.  test_emu_dosage_matrix.py runs the same tests under the warp
emulator, except the launch past 4 GiB and the device half of the torch wrapper test.
"""
import ctypes as C
import functools
import time

import pytest

import golden_util
import test_gpu_parity as G
import test_gpu_resident as R
from vcfx_b200 import synth

pytestmark = pytest.mark.gpu

MODES = (0, 1)
TILES = (0, 512, 4096)
E_OUTPUT_TOO_BIG = -7


@pytest.fixture
def mem():
    return R.TorchMem()


@pytest.fixture
def resident(mem):
    return functools.partial(R.run_resident, mem)


# ----------------------------------------------------------------------------- helpers
TXT = {0: b"0", 1: b"1", 2: b"2", -1: b"NA"}


def render(data, m):
    """dosage_calculator's stdout without its header row, rebuilt from the matrix: the line's bytes up to its fifth tab,
    then "NA" for a line without a GT key, else the n_cols codes as 0 / 1 / 2 / NA joined by ','."""
    out = []
    codes = m.codes.tolist()
    for i, (off, n, nogt) in enumerate(zip(m.line_offset.tolist(), m.n_cols.tolist(), m.no_gt.tolist())):
        p = off
        for _ in range(5):
            p = data.index(b"\t", p) + 1
        assert n <= len(codes[i]), "render needs every column: a width of at least the widest line"
        out.append(bytes(data[off:p]) + (b"NA" if nogt else b",".join(TXT[c] for c in codes[i][:n])) + b"\n")
    return b"".join(out)


def widest(data):
    """Sample columns of the widest line (a width that keeps every column)."""
    return max(0, max((l.count(b"\t") for l in data.split(b"\n")), default=0) - 8)


def small_chunk(data):
    """4096-byte chunks, or more when a line does not fit one."""
    longest = max((len(l) + 1 for l in data.split(b"\n")), default=1)
    return max(4096, (2 * longest + 4095) & ~4095)


def out_cap_for(data, W):
    return (data.count(b"\n") + 1) * (16 + W) + 16


def check_shape(api, m, W, tag):
    """What every matrix satisfies: -2 past a line's columns, -1 in the columns of a line without a GT key, codes in
    {-1, 0, 1, 2} elsewhere, flagged = rows with more columns than W."""
    import torch
    rows = m.line_offset.numel()
    assert m.codes.shape == (rows, W) and m.codes.dtype == torch.int8, (tag, m.codes.shape)
    assert m.n_cols.numel() == rows and m.no_gt.numel() == rows and m.totals.rows == rows, tag
    s = torch.arange(W, device=m.codes.device)[None, :]
    past = s >= m.n_cols.to(torch.int64)[:, None]
    assert bool((m.codes[past] == -2).all()), tag
    inside = ~past
    assert bool((m.codes[inside & m.no_gt[:, None]] == -1).all()), tag
    c = m.codes[inside]
    assert bool(((c >= -1) & (c <= 2)).all()), tag
    assert m.totals.flagged == int((m.n_cols > W).sum()), (tag, m.totals.flagged)
    assert m.totals.bytes_out == rows * (16 + W), tag


def check_text(api, O, data, mode, m, tag):
    """The matrix against dosage_calculator's text: the oracle and the library's text path, with the same counters."""
    text = api.dosage_calculator(data, mode)
    o = O.dosage(data, mode)
    if mode == api.FILE and not data:
        assert m.totals.rows == 0 and text.out == o.out == b"", tag
        return
    got = api.DS_HEADER + render(data, m)
    G._cmp(f"{tag} matrix vs oracle", got, o.out)
    G._cmp(f"{tag} matrix vs text path", got, text.out)
    for f in ("rows", "data_lines", "short_lines"):
        assert getattr(m.totals, f) == getattr(text.totals, f), (tag, f)
    assert m.err == text.err, tag


def same(a, b, tag):
    """Two matrices (on any devices) are equal tensor for tensor."""
    import torch
    for f in ("codes", "line_offset", "n_cols", "no_gt"):
        x, y = getattr(a, f).cpu(), getattr(b, f).cpu()
        assert x.dtype == y.dtype and x.shape == y.shape and torch.equal(x, y), (tag, f, x.shape, y.shape)
    assert a.samples == b.samples, tag


def from_resident(api, got, W, samples=()):
    """A DosageMatrix from one resident result (raw bytes, stats, events)."""
    import numpy as np
    import torch
    raw, st, _ = got
    assert st.bytes_out == st.rows * (16 + W) and len(raw) == st.bytes_out
    meta, codes = api._ds_split(raw, W)
    tot = api.Totals()
    tot.add(st, 0, [])
    return api.DosageMatrix(list(samples), torch.from_numpy(np.array(codes)), torch.from_numpy(meta["line_offset"].astype(np.int64)),
                            torch.from_numpy(meta["n_cols"].astype(np.int32)), torch.from_numpy((meta["flags"] & 1).astype(bool)),
                            tot, api.DS_WARNING * tot.short_lines)


def matrix_kw(api, W):
    return dict(flags=api.F_DS_MATRIX, width=W)


def run_corpus(api, O, resident, data, tag, tiles=TILES):
    """Both modes: the streaming path at the default chunk size and at small chunks, the resident path at each tile size;
    all equal, and equal to the tool's text."""
    for mode in MODES:
        o = O.dosage(data, mode)
        if o.first_bad_line:                      # a data line in front of "#CHROM": the tool stops with its error
            with pytest.raises(api.VcfxCudaError, match=r"VCF header \(#CHROM\) not found"):
                api.dosage_matrix(data, mode)
            continue
        W = widest(data)
        m = api.dosage_matrix(data, mode, width=W)
        t = f"{tag} mode{mode} W{W}"
        check_shape(api, m, W, t)
        check_text(api, O, data, mode, m, t)
        ms = api.dosage_matrix(data, mode, width=W, chunk_bytes=small_chunk(data))
        same(ms, m, f"{t} small chunks")
        assert (ms.totals.rows, ms.totals.data_lines, ms.totals.short_lines, ms.totals.flagged) == \
               (m.totals.rows, m.totals.data_lines, m.totals.short_lines, m.totals.flagged), t
        if mode == api.FILE and not data:
            continue
        for tile in tiles:
            got = resident(api, api.OP_DOSAGE, mode, data, tile_bytes=tile, out_cap=out_cap_for(data, W), ctx_kw=matrix_kw(api, W))
            r = from_resident(api, got, W, m.samples)
            same(r, m, f"{t} resident tile{tile}")
            for f in ("rows", "data_lines", "short_lines", "flagged", "bytes_out"):
                assert getattr(got[1], f) == getattr(m.totals, f), (t, tile, f)


# ----------------------------------------------------------------------------- 1. the corpora
SWEEP = R.SWEEP
DS_S = (1, 2, 100, 126, 127, 128, 129, 255, 256, 257, 700)


def ds_lattice_input(S):
    """test_dosage_calculator_cases' input: lines on the four-byte lattice with samples that leave it."""
    hdr = b"##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t"
    lines = []
    for k in range(48):
        gts = [[b"0|1", b"1|1", b"0/0", b"2|0", b"./."][(i * 7 + k) % 5] for i in range(S)]
        if k % 4 == 1:
            gts[(k * 37) % S] = [b"0", b".", b"0/1/1", b"0|1:3", b"10|1", b"", b" 0|1"][k % 7]
        lines.append(b"%d\t%d\t%s\tA\tG\t.\tPASS\t.\tGT\t" % (k % 22 + 1, 10 ** (k % 7), b"r" * (k % 5)) + b"\t".join(gts))
    return hdr + b"\t".join(b"S%d" % i for i in range(S)) + b"\n" + b"\n".join(lines) + (b"\n" if S % 2 else b"")


@pytest.mark.parametrize("shape,V,S", G.SHAPES)
def test_matrix_synthetic_shapes(cuda_api, oracle, resident, shape, V, S):
    run_corpus(cuda_api, oracle, resident, G.shape_input(shape, V, S), f"shape{shape} {V}x{S}")


@pytest.mark.parametrize("seed", range(40))
def test_matrix_adversarial(cuda_api, oracle, resident, seed):
    run_corpus(cuda_api, oracle, resident, G.adversarial_input(seed), f"fuzz{seed}")


def test_matrix_empty_and_degenerate(cuda_api, oracle, resident):
    for data in G.DEGENERATE:
        run_corpus(cuda_api, oracle, resident, data, repr(data[:20]))


def test_matrix_ds_quirks_fixture(cuda_api, oracle, resident):
    data, _ = golden_util.load()["ds_quirks"]
    run_corpus(cuda_api, oracle, resident, data, "ds_quirks")


@pytest.mark.parametrize("S", DS_S)
def test_matrix_dosage_lattice_sweep(cuda_api, oracle, resident, S):
    run_corpus(cuda_api, oracle, resident, ds_lattice_input(S), f"ds S{S}")


@pytest.mark.parametrize("shape,S", SWEEP)
def test_matrix_line_lengths_sweep(cuda_api, oracle, resident, shape, S):
    run_corpus(cuda_api, oracle, resident, G.sweep_input(shape, S), f"sweep shape{shape} S{S}")


# ----------------------------------------------------------------------------- 2. literal codes
LITERAL_LINES = (
    b"1\t100\trs1\tA\tG\t.\tPASS\t.\tGT\t0/0\t0|1\t1/1\t2|0\t./.\t.\t0\t0/1/1\t1/0:3\t\t1|1",
    b"1\t200\trs2\tA\tC\t.\tPASS\t.\tGT\t1|1\t0/1\t",                   # a trailing tab: no third column
    b"1\t300\trs3\tA\tT\t.\tPASS\t.\tDP\t5\t7\t9",                      # no GT key
    b"1\t400\trs4\tG\tA\t.\tPASS\t.\tDP:GT\t3:0/1\t4:1|1",
    b"1\t500\trs5\tG\tA\t.\tPASS",                                     # fewer than ten columns: no row, one warning
)
X = -2
LITERAL_WANT = [                                   # (n_cols, no_gt, the 11 codes) per row, '\n' line ends, either mode
    (11, False, [0, 1, 2, 1, -1, -1, -1, -1, 1, -1, 2]),
    (2, False, [2, 1, X, X, X, X, X, X, X, X, X]),
    (3, True, [-1, -1, -1, X, X, X, X, X, X, X, X]),
    (2, False, [1, 2, X, X, X, X, X, X, X, X, X]),
]
LITERAL_WANT_CRLF_STDIN = [                        # stdin mode keeps the '\r': it spoils the last column, or is one
    (11, False, [0, 1, 2, 1, -1, -1, -1, -1, 1, -1, -1]),
    (3, False, [2, 1, -1, X, X, X, X, X, X, X, X]),
    (3, True, [-1, -1, -1, X, X, X, X, X, X, X, X]),
    (2, False, [1, -1, X, X, X, X, X, X, X, X, X]),
]


def literal_input(crlf):
    eol = b"\r\n" if crlf else b"\n"
    hdr = b"##fileformat=VCFv4.2" + eol + b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + b"\t".join(b"ABCDEFGHIJK"[i:i + 1] for i in range(11)) + eol
    return hdr + b"".join(l + eol for l in LITERAL_LINES)


def test_matrix_literal_codes(cuda_api, oracle, resident):
    import torch
    api = cuda_api
    for crlf in (False, True):
        data = literal_input(crlf)
        for mode in MODES:
            want = LITERAL_WANT_CRLF_STDIN if (crlf and mode == api.STDIN) else LITERAL_WANT
            starts = [data.index(l) for l in LITERAL_LINES[:4]]
            tag = f"literal crlf{int(crlf)} mode{mode}"
            m = api.dosage_matrix(data, mode)
            assert m.samples == [bytes([c]) for c in b"ABCDEFGHIJK"], (tag, m.samples)
            got = from_resident(api, resident(api, api.OP_DOSAGE, mode, data, out_cap=out_cap_for(data, 11), ctx_kw=matrix_kw(api, 11)), 11, m.samples)
            for mm in (m, got):
                assert mm.codes.tolist() == [c for _, _, c in want], (tag, mm.codes.tolist())
                assert mm.n_cols.tolist() == [n for n, _, _ in want], (tag, mm.n_cols.tolist())
                assert mm.no_gt.tolist() == [g for _, g, _ in want], tag
                assert mm.line_offset.tolist() == starts, tag
                assert (mm.totals.rows, mm.totals.short_lines, mm.totals.flagged) == (4, 1, 0), tag
                assert mm.err == api.DS_WARNING, tag
            assert m.codes.dtype == torch.int8 and m.line_offset.dtype == torch.int64 and m.n_cols.dtype == torch.int32
            check_text(api, oracle, data, mode, m, tag)


# ----------------------------------------------------------------------------- 3. width
def ragged_input():
    """40 samples in the header; lines of 40 columns, a line of 20 and a line of 50."""
    data = synth.make_vcf(2, 60, 40, seed=77)
    lines = data.split(b"\n")
    first = next(i for i, l in enumerate(lines) if l and not l.startswith(b"#"))
    f = lines[first + 3].split(b"\t")
    lines[first + 3] = b"\t".join(f[:9 + 20])
    f = lines[first + 7].split(b"\t")
    lines[first + 7] = b"\t".join(f + [b"1|0"] * 10)
    return b"\n".join(lines)


def test_matrix_width(cuda_api, oracle, resident):
    """W from the header, and width 0, 1 and header + 5: a shorter line has a -2 tail, a longer one is cut at W with its
    true n_cols and is counted in flagged."""
    import torch
    api = cuda_api
    data = ragged_input()
    for mode in MODES:
        full = api.dosage_matrix(data, mode, width=50)
        check_text(api, oracle, data, mode, full, f"ragged mode{mode}")
        n = full.n_cols.tolist()
        assert n.count(20) == 1 and n.count(50) == 1 and all(c in (20, 40, 50) for c in n)
        d = api.dosage_matrix(data, mode)
        assert len(d.samples) == 40 and d.codes.shape[1] == 40
        for W in (None, 0, 1, 45):
            tag = f"ragged mode{mode} width{W}"
            m = api.dosage_matrix(data, mode, width=W)
            w = 40 if W is None else W
            check_shape(api, m, w, tag)
            assert torch.equal(m.codes, full.codes[:, :w]), tag
            assert torch.equal(m.n_cols, full.n_cols) and torch.equal(m.line_offset, full.line_offset), tag
            assert m.totals.flagged == sum(c > w for c in n), tag
            r = from_resident(api, resident(api, api.OP_DOSAGE, mode, data, out_cap=out_cap_for(data, w), ctx_kw=matrix_kw(api, w)), w, m.samples)
            same(r, m, tag + " resident")
            assert r.totals.flagged == m.totals.flagged, tag


# ----------------------------------------------------------------------------- 4. re-runs and capacity
def test_matrix_more_rows_than_records(cuda_api, oracle, resident):
    """More rows than the default record capacity: vcfx_cuda_sync runs the launch again; a second launch on the grown
    context is right too."""
    api = cuda_api
    data = G.more_rows_input()
    assert len(data) // 256 + 65536 < data.count(b"\n") - 2
    for mode in MODES:
        m = api.dosage_matrix(data, mode, width=2)
        check_text(api, oracle, data, mode, m, f"more rows mode{mode}")
        ctx = api.Context(api.OP_DOSAGE, mode, **matrix_kw(api, 2))
        try:
            for k in range(2):
                got = resident(api, api.OP_DOSAGE, mode, data, ctx=ctx, out_cap=out_cap_for(data, 2))
                same(from_resident(api, got, 2, m.samples), m, f"more rows mode{mode} launch{k}")
        finally:
            ctx.close()


def test_matrix_stream_slot_grows(cuda_api, oracle):
    """A streaming output slot far too small for a chunk's matrix is grown and the chunk run again."""
    api = cuda_api
    data = G.shape_input(2, 200, 2504)
    for mode in MODES:
        want = api.dosage_matrix(data, mode)
        assert want.totals.bytes_out > 100 * 4096
        m = api.dosage_matrix(data, mode, out_bytes=4096)
        same(m, want, f"tiny slot mode{mode}")
        assert (m.totals.rows, m.totals.bytes_out) == (want.totals.rows, want.totals.bytes_out)


def test_matrix_run_device_output_too_big(cuda_api, oracle, mem):
    """run_device into too small an output: VCFX_E_OUTPUT_TOO_BIG with stats.rows filled; a second run sized from them
    is right.  An output that is not 16-byte aligned is refused."""
    api = cuda_api
    data = G.shape_input(3, 200, 2504)
    W = 2504
    for mode in MODES:
        want = api.dosage_matrix(data, mode)
        ctx = api.Context(api.OP_DOSAGE, mode, **matrix_kw(api, W))
        try:
            d_in = mem.input(data, api.DEVICE_PAD)
            small = mem.output(100 * (16 + W))
            ctx.run_device(d_in.addr, len(data), small.addr, small.cap)
            st = api.ChunkStats()
            assert ctx._l.vcfx_cuda_sync(ctx._h, C.byref(st)) == E_OUTPUT_TOO_BIG
            assert st.rows == want.totals.rows > 100 and st.bytes_out == st.rows * (16 + W)
            out = mem.output(int(st.bytes_out))
            ctx.run_device(d_in.addr, len(data), out.addr, int(st.bytes_out))
            st2 = ctx.sync()
            same(from_resident(api, (out.read(0, int(st2.bytes_out)), st2, []), W, want.samples), want, f"sized from stats mode{mode}")
            with pytest.raises(api.VcfxCudaError) as e:
                ctx.run_device(d_in.addr, len(data), out.addr + 8, int(st.bytes_out) - 8)
            assert e.value.code == -1
        finally:
            ctx.close()


# ----------------------------------------------------------------------------- 5. reuse, queued launches, a shared upload
def test_matrix_context_reuse_and_queued_launches(cuda_api, oracle, resident, mem):
    """One context for a large, a small and the large input again; N launches queued before one sync give one launch's
    result."""
    api = cuda_api
    large = synth.make_vcf(3, 3000, 120, seed=13)
    small = synth.make_vcf(2, 30, 120, seed=14)
    W = 120
    for mode in MODES:
        ref = {id(d): api.dosage_matrix(d, mode) for d in (large, small)}
        ctx = api.Context(api.OP_DOSAGE, mode, **matrix_kw(api, W))
        try:
            for k, d in enumerate((large, small, large)):
                got = resident(api, api.OP_DOSAGE, mode, d, ctx=ctx, out_cap=out_cap_for(d, W))
                same(from_resident(api, got, W, ref[id(d)].samples), ref[id(d)], f"reuse mode{mode} step{k}")
            d_in = mem.input(large, api.DEVICE_PAD)
            out = mem.output(out_cap_for(large, W))
            for _ in range(4):
                ctx.run_device(d_in.addr, len(large), out.addr, out.cap)
            st = ctx.sync()
            same(from_resident(api, (out.read(0, int(st.bytes_out)), st, []), W, ref[id(large)].samples), ref[id(large)], f"queued mode{mode}")
        finally:
            ctx.close()


def test_matrix_shared_upload_next_to_text(cuda_api, oracle):
    """A matrix context fed by submit_shared from a text dosage context's upload: both give what they give alone."""
    api = cuda_api
    data = synth.make_vcf(3, 1500, 64, seed=31)
    chunk = 32 << 10
    for mode in MODES:
        text_ctx = api.Context(api.OP_DOSAGE, mode, chunk_bytes=chunk)
        mat_ctx = api.Context(api.OP_DOSAGE, mode, chunk_bytes=chunk, **matrix_kw(api, 64))
        texts, metas, codes = [], [], []
        try:
            pieces = list(api.chunk_bounds(data, chunk))
            assert len(pieces) > 4
            for s, e in pieces:
                buf, cap = text_ctx.acquire()
                C.memmove(buf, data[s:e], e - s)
                text_ctx.submit(e - s, is_final=(e == len(data)), file_offset=s)
                assert mat_ctx.submit_shared(text_ctx, is_final=(e == len(data)), file_offset=s)
                texts.append(text_ctx.next_output()[0])
                mm, cc = api._ds_split(mat_ctx.next_output()[0], 64)
                metas.append(mm); codes.append(cc)
        finally:
            text_ctx.close(); mat_ctx.close()
        import numpy as np
        G._cmp(f"shared upload text mode{mode}", api.DS_HEADER + b"".join(texts), api.dosage_calculator(data, mode).out)
        want = api.dosage_matrix(data, mode)
        meta = np.concatenate(metas)
        assert np.array_equal(np.concatenate(codes), want.codes.numpy()), mode
        assert meta["line_offset"].tolist() == want.line_offset.tolist() and meta["n_cols"].tolist() == want.n_cols.tolist(), mode


# ----------------------------------------------------------------------------- 6. codes past 2^32 bytes in one launch
def test_matrix_codes_past_4_gib(cuda_api):
    """70,000 sample names, about 70,000 one-sample lines: a few MB of input, ~4.9 GB of codes in one launch.  Column 0
    holds the expected codes, every other column is -2, and the rows around byte 2^32 are right (checked on the device)."""
    import torch
    api = cuda_api
    t0 = time.perf_counter()
    S, V = 70000, 70000
    gts, want = (b"0/0", b"0|1", b"1/1", b"./."), (0, 1, 2, -1)
    hdr = b"##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + b"\t".join(b"S%d" % i for i in range(S)) + b"\n"
    lines = [b"1\t%d\t.\tA\tG\t.\t.\t.\tGT\t%s\n" % (i + 1, gts[i % 4]) for i in range(V)]
    data = hdr + b"".join(lines)
    assert V * S > 1 << 32
    need = V * (16 + S) + len(data) * 4 + (2 << 30)
    free, total = torch.cuda.mem_get_info()
    if free < need:
        pytest.skip(f"needs {need / 1e9:.1f} GB of free device memory, {free / 1e9:.1f} GB are free")
    dev = torch.device("cuda", 0)
    d_in = torch.empty(len(data) + api.DEVICE_PAD, dtype=torch.uint8, device=dev)
    d_in[:len(data)].copy_(torch.frombuffer(bytearray(data), dtype=torch.uint8))
    m = api.dosage_matrix_device(d_in, len(data))
    assert len(m.samples) == S and m.codes.shape == (V, S) and m.totals.rows == V
    expect0 = torch.tensor(want, dtype=torch.int8, device=dev).repeat(V // 4 + 1)[:V]
    assert torch.equal(m.codes[:, 0], expect0)
    for r0 in range(0, V, 8192):
        assert bool((m.codes[r0:r0 + 8192, 1:] == -2).all()), r0
    starts = [len(hdr)]
    for l in lines[:-1]:
        starts.append(starts[-1] + len(l))
    assert m.line_offset.cpu().tolist() == starts and bool((m.n_cols == 1).all()) and not bool(m.no_gt.any())
    r = (1 << 32) // S
    for i in range(r - 2, r + 3):                      # rows that straddle byte 2^32 of the codes
        row = m.codes[i].cpu().tolist()
        assert row == [want[i % 4]] + [-2] * (S - 1), i
    print(f"\ncodes past 2^32: {V} x {S} = {V * S / 1e9:.2f} GB in one launch, {m.totals.kernel_ms:.1f} ms of kernels, "
          f"whole test {time.perf_counter() - t0:.1f} s")


# ----------------------------------------------------------------------------- 7. the torch wrappers
def test_matrix_torch_wrapper_host(cuda_api, resident):
    """dosage_matrix hands back CPU tensors of the documented types, the header's sample names, and what one resident
    launch over the same bytes gives, on a C2-shaped input."""
    import torch
    api = cuda_api
    data = synth.make_vcf(2, 300, 2504, seed=2)
    m = api.dosage_matrix(data)
    names = api._ds_prescan(data, api.FILE)[2]
    assert m.samples == names and len(names) == 2504
    for f, dt in (("codes", torch.int8), ("line_offset", torch.int64), ("n_cols", torch.int32), ("no_gt", torch.bool)):
        t = getattr(m, f)
        assert t.device.type == "cpu" and t.dtype == dt, f
    assert m.codes.shape == (300, 2504) and m.totals.rows == 300
    got = resident(api, api.OP_DOSAGE, api.FILE, data, out_cap=out_cap_for(data, 2504), ctx_kw=matrix_kw(api, 2504))
    same(from_resident(api, got, 2504, names), m, "host wrapper vs resident")


def test_matrix_torch_wrapper_device(cuda_api):
    """dosage_matrix_device on a 50,000-variant C2-shaped input equals dosage_matrix on the same bytes; its output feeds
    a torch op on the current stream without an explicit synchronize."""
    import torch
    api = cuda_api
    data = synth.make_vcf(2, 50000, 2504, seed=2)
    host = api.dosage_matrix(data)
    assert host.codes.shape == (50000, 2504)
    dev = torch.device("cuda", 0)
    d_in = torch.empty(len(data) + api.DEVICE_PAD, dtype=torch.uint8, device=dev)
    side = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(side):
        d_in[:len(data)].copy_(torch.frombuffer(bytearray(data), dtype=torch.uint8).to(dev, non_blocking=True))
        m = api.dosage_matrix_device(d_in, len(data))
        alt = m.codes.clamp(min=0).sum(dim=1, dtype=torch.int64)      # queued on `side` behind the library's kernels
        alt_host = alt.cpu()
    same(m, host, "device wrapper vs streaming")
    assert torch.equal(alt_host, host.codes.clamp(min=0).sum(dim=1, dtype=torch.int64))
    assert m.codes.device == dev and m.codes.untyped_storage().data_ptr() == m.line_offset.untyped_storage().data_ptr()
    assert (m.totals.rows, m.totals.short_lines, m.err) == (host.totals.rows, host.totals.short_lines, host.err)
