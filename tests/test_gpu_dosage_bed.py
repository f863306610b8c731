"""dosage_calculator's .bed mode (VCFX_OP_DOSAGE + VCFX_F_DS_BED): the genotypes as PLINK 1 .bed rows, two bits a call,
with the matrix mode's 16 bytes of metadata per row, through the streaming path (api.dosage_bed), the device-resident
entry point (vcfx_cuda_run_device) and the torch wrapper (api.dosage_bed_device).

The expected rows do not come from the library: they are packed in numpy from the oracle's dosage text (each row cut
after its fifth tab, "NA" / 0 / 1 / 2 per column, missing past the row's columns).  As a second check they equal the int8
matrix of the same input, packed.  The literal case writes its bytes out.  test_emu_dosage_bed.py runs the same tests
under the warp emulator, except the launch past 4 GiB and the device half of the torch wrapper test.
"""
import ctypes as C
import functools
import time

import numpy as np
import pytest

import golden_util
import test_gpu_dosage_matrix as D
import test_gpu_parity as G
import test_gpu_resident as R
from vcfx_b200 import synth

pytestmark = pytest.mark.gpu

MODES = (0, 1)
TILES = (0, 512, 4096)
E_INVALID, E_OUTPUT_TOO_BIG = -1, -7


@pytest.fixture
def mem():
    return R.TorchMem()


@pytest.fixture
def resident(mem):
    return functools.partial(R.run_resident, mem)


# ----------------------------------------------------------------------------- helpers
def row_bytes(W):
    return (W + 3) // 4


def pack(codes, W):
    """PLINK 1 .bed rows of an int matrix of dosage codes (2 / 1 / 0, -1 "NA", -2 no such column), W columns: 2 -> 00,
    1 -> 10, 0 -> 11, anything else -> 01; sample s at bits 2 (s & 3) of byte s >> 2, padding 00."""
    codes = np.asarray(codes, dtype=np.int64)
    assert codes.ndim == 2 and codes.shape[1] == W
    v = np.ones(codes.shape, dtype=np.uint8)
    v[codes == 2] = 0
    v[codes == 1] = 2
    v[codes == 0] = 3
    B = row_bytes(W)
    full = np.zeros((codes.shape[0], 4 * B), dtype=np.uint8)
    full[:, :W] = v
    q = full.reshape(codes.shape[0], B, 4)
    return (q[:, :, 0] | (q[:, :, 1] << 2) | (q[:, :, 2] << 4) | (q[:, :, 3] << 6)).astype(np.uint8)


def oracle_codes(O, data, mode, W):
    """The oracle's dosage rows as an int matrix of W columns (-1 "NA", -2 past the row's columns), and the rows' first five
    fields (CHROM, POS, ID, REF, ALT).  An empty dosage field is a row of no columns."""
    text = O.dosage(data, mode).out
    rows = text.split(b"\n")[1:-1] if text else []
    codes = np.full((len(rows), W), -2, dtype=np.int64)
    fields = []
    for i, r in enumerate(rows):
        f = r.split(b"\t", 5)
        fields.append(f[:5])
        vals = [-1 if t == b"NA" else int(t) for t in f[5].split(b",")][:W] if f[5] else []      # (no column at all)
        assert all(v in (-1, 0, 1, 2) for v in vals), r
        codes[i, :len(vals)] = vals
    return codes, fields


def expected_bed(O, data, mode, W):
    return pack(oracle_codes(O, data, mode, W)[0], W)


def out_cap_for(data, W):
    return (data.count(b"\n") + 1) * (16 + row_bytes(W)) + 16


def bed_kw(api, W):
    return dict(flags=api.F_DS_BED, width=W)


def from_resident(api, got, W, samples=()):
    """A DosageBed from one resident result (raw bytes, stats, events)."""
    import torch
    raw, st, _ = got
    assert st.bytes_out == st.rows * (16 + row_bytes(W)) and len(raw) == st.bytes_out
    meta, packed = api._ds_split(raw, W, api.F_DS_BED)
    tot = api.Totals()
    tot.add(st, 0, [])
    return api.DosageBed(list(samples), W, torch.from_numpy(np.array(packed)), *api._ds_meta_host(meta), tot, api.DS_WARNING * tot.short_lines)


def same(a, b, tag):
    """Two DosageBed results (on any devices) are equal tensor for tensor."""
    import torch
    for f in ("packed", "line_offset", "n_cols", "no_gt"):
        x, y = getattr(a, f).cpu(), getattr(b, f).cpu()
        assert x.dtype == y.dtype and x.shape == y.shape and torch.equal(x, y), (tag, f, x.shape, y.shape)
    assert a.samples == b.samples and a.width == b.width, tag


def check_bed(api, O, data, mode, b, W, tag):
    """b against the numpy rows from the oracle's text, and against the int8 matrix of the same input: packed bytes, the
    metadata and the counters."""
    import torch
    rows = b.line_offset.numel()
    assert b.packed.dtype == torch.uint8 and b.packed.shape == (rows, row_bytes(W)) and b.width == W, (tag, b.packed.shape)
    want = expected_bed(O, data, mode, W)
    assert np.array_equal(b.packed.cpu().numpy(), want), (tag, "vs oracle")
    m = api.dosage_matrix(data, mode, width=W)
    assert np.array_equal(pack(m.codes.numpy(), W), want), (tag, "packed matrix vs oracle")
    for f in ("line_offset", "n_cols", "no_gt"):
        assert torch.equal(getattr(b, f).cpu(), getattr(m, f)), (tag, f)
    for f in ("rows", "data_lines", "short_lines", "flagged"):
        assert getattr(b.totals, f) == getattr(m.totals, f), (tag, f)
    assert b.totals.bytes_out == rows * (16 + row_bytes(W)) and b.err == m.err and b.samples == m.samples, tag


def run_corpus(api, O, resident, data, tag, widths=None, tiles=TILES):
    """Both modes and each width (default: the widest line's): the streaming path at the default chunk size and at small
    chunks, the resident path at each tile size; all equal, and equal to the oracle's rows packed."""
    for mode in MODES:
        if O.dosage(data, mode).first_bad_line:       # a data line in front of "#CHROM": the tool stops with its error
            with pytest.raises(api.VcfxCudaError, match=r"VCF header \(#CHROM\) not found"):
                api.dosage_bed(data, mode)
            continue
        for W in widths or (D.widest(data),):
            t = f"{tag} mode{mode} W{W}"
            b = api.dosage_bed(data, mode, width=W)
            check_bed(api, O, data, mode, b, W, t)
            bs = api.dosage_bed(data, mode, width=W, chunk_bytes=D.small_chunk(data))
            same(bs, b, f"{t} small chunks")
            assert (bs.totals.rows, bs.totals.short_lines, bs.totals.flagged) == (b.totals.rows, b.totals.short_lines, b.totals.flagged), t
            if mode == api.FILE and not data:
                continue
            for tile in tiles:
                got = resident(api, api.OP_DOSAGE, mode, data, tile_bytes=tile, out_cap=out_cap_for(data, W), ctx_kw=bed_kw(api, W))
                same(from_resident(api, got, W, b.samples), b, f"{t} resident tile{tile}")
                for f in ("rows", "data_lines", "short_lines", "flagged", "bytes_out"):
                    assert getattr(got[1], f) == getattr(b.totals, f), (t, tile, f)


# ----------------------------------------------------------------------------- 1. the corpora
@pytest.mark.parametrize("shape,V,S", G.SHAPES)
def test_bed_synthetic_shapes(cuda_api, oracle, resident, shape, V, S):
    run_corpus(cuda_api, oracle, resident, G.shape_input(shape, V, S), f"shape{shape} {V}x{S}")


@pytest.mark.parametrize("seed", range(40))
def test_bed_adversarial(cuda_api, oracle, resident, seed):
    run_corpus(cuda_api, oracle, resident, G.adversarial_input(seed), f"fuzz{seed}")


def test_bed_empty_and_degenerate(cuda_api, oracle, resident):
    for data in G.DEGENERATE:
        run_corpus(cuda_api, oracle, resident, data, repr(data[:20]))


def test_bed_ds_quirks_fixture(cuda_api, oracle, resident):
    data, _ = golden_util.load()["ds_quirks"]
    run_corpus(cuda_api, oracle, resident, data, "ds_quirks")


def odd_row_width(S):
    """A width >= S whose rows take an odd number of bytes (and end in padding): 16 rows in a row then start at every
    offset modulo 16."""
    B = row_bytes(S)
    return 4 * (B if B % 2 else B + 1) - 1


@pytest.mark.parametrize("S", D.DS_S)
def test_bed_dosage_lattice_sweep(cuda_api, oracle, resident, S):
    data = D.ds_lattice_input(S)
    W = odd_row_width(S)
    rows = 48
    assert {(16 * rows + i * row_bytes(W)) % 16 for i in range(rows)} == set(range(16))
    run_corpus(cuda_api, oracle, resident, data, f"ds S{S}", widths=(S, W))


@pytest.mark.parametrize("shape,S", R.SWEEP)
def test_bed_line_lengths_sweep(cuda_api, oracle, resident, shape, S):
    run_corpus(cuda_api, oracle, resident, G.sweep_input(shape, S), f"sweep shape{shape} S{S}")


# ----------------------------------------------------------------------------- 2. literal bytes
LITERAL_HEADER = b"##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tA\tB\tC\tD\tE\n"
LITERAL_LINES = (
    b"1\t100\trs1\tA\tG\t.\tPASS\t.\tGT\t0/0\t0|1\t1/1\t./.\t1",               # 0 1 2 NA NA (haploid: NA)
    b"1\t200\trs2\tA\tC,T\t.\tPASS\t.\tGT:DP\t10|1:3\t2/0:4\t0/2\t1|2\t0|0",   # 2 1 1 2 0 (every allele > 0 counts)
    b"1\t300\trs3\tA\tT\t.\tPASS\t.\tDP\t5\t7\t9\t1\t2",                      # no GT key: all missing
    b"1\t400\trs4\tG\tA\t.\tPASS\t.\tGT\t1|1\t0/1",                           # ragged: 2 1, then no column
    b"1\t500\trs5\tG\tA\t.\tPASS",                                           # fewer than ten columns: no row, one warning
    b"2\t600\trs6\tC\tG\t.\tPASS\t.\tGT\t0|0\t1|0\t0/0\t1/1\t0/1\t1/1",        # six columns: 0 1 0 2 1 | 2
    b"2\t700\trs7\tC\tG\t.\tPASS\t.\tGT\t0\t.\t0|1\t1/1/1\t1",                # NA NA 1 NA NA
)
# the .bed rows at widths 1 .. 5: 2 -> 00, 1 -> 10, 0 -> 11, missing -> 01, padding 00; low bits first
LITERAL_BED = {
    1: [b"\x03", b"\x00", b"\x01", b"\x00", b"\x03", b"\x01"],
    2: [b"\x0b", b"\x08", b"\x05", b"\x08", b"\x0b", b"\x05"],
    3: [b"\x0b", b"\x28", b"\x15", b"\x18", b"\x3b", b"\x25"],
    4: [b"\x4b", b"\x28", b"\x55", b"\x58", b"\x3b", b"\x65"],
    5: [b"\x4b\x01", b"\x28\x03", b"\x55\x01", b"\x58\x01", b"\x3b\x02", b"\x65\x01"],
}
LITERAL_N_COLS = [5, 5, 5, 2, 6, 5]


def literal_input(crlf):
    data = LITERAL_HEADER + b"".join(l + b"\n" for l in LITERAL_LINES)
    return data.replace(b"\n", b"\r\n") if crlf else data


def test_bed_literal_bytes(cuda_api, oracle, resident):
    api = cuda_api
    for crlf in (False, True):
        data = literal_input(crlf)
        starts = [data.index(l) for i, l in enumerate(LITERAL_LINES) if i != 4]
        for mode in MODES:
            for W, want in LITERAL_BED.items():
                tag = f"literal crlf{int(crlf)} mode{mode} W{W}"
                b = api.dosage_bed(data, mode, width=W)
                r = from_resident(api, resident(api, api.OP_DOSAGE, mode, data, out_cap=out_cap_for(data, W), ctx_kw=bed_kw(api, W)), W, b.samples)
                same(r, b, tag)
                check_bed(api, oracle, data, mode, b, W, tag)
                assert b.samples == [bytes([c]) for c in b"ABCDE"], tag
                assert b.line_offset.tolist() == starts and b.n_cols.tolist() == LITERAL_N_COLS, tag
                assert b.no_gt.tolist() == [False, False, True, False, False, False], tag
                assert (b.totals.rows, b.totals.short_lines, b.totals.flagged) == (6, 1, sum(n > W for n in LITERAL_N_COLS)), tag
                assert b.err == api.DS_WARNING, tag
                if crlf and mode == api.STDIN:                 # stdin mode keeps the '\r': it spoils each line's last column
                    continue
                assert [bytes(row) for row in b.packed.numpy()] == want, (tag, b.packed.tolist())
            b = api.dosage_bed(data, mode)
            assert b.width == 5 and b.packed.shape == (6, 2), (crlf, mode)


# ----------------------------------------------------------------------------- 3. widths and flags
def test_bed_width(cuda_api, oracle, resident):
    """W from the header, 0 (rows of metadata only), 1, the header's and header + 5 on ragged lines."""
    import torch
    api = cuda_api
    data = D.ragged_input()
    for mode in MODES:
        full = api.dosage_matrix(data, mode, width=50)
        for W in (None, 0, 1, 40, 45):
            tag = f"ragged mode{mode} width{W}"
            b = api.dosage_bed(data, mode, width=W)
            w = 40 if W is None else W
            check_bed(api, oracle, data, mode, b, w, tag)
            assert np.array_equal(b.packed.numpy(), pack(full.codes[:, :w].numpy(), w)), tag
            assert torch.equal(b.n_cols, full.n_cols), tag
            r = from_resident(api, resident(api, api.OP_DOSAGE, mode, data, out_cap=out_cap_for(data, w), ctx_kw=bed_kw(api, w)), w, b.samples)
            same(r, b, tag + " resident")
            if w == 0:
                assert b.totals.bytes_out == 16 * b.totals.rows and r.packed.shape == (b.totals.rows, 0), tag


def test_bed_and_matrix_flags_together_are_invalid(cuda_api):
    api = cuda_api
    for mode in MODES:
        with pytest.raises(api.VcfxCudaError) as e:
            api.Context(api.OP_DOSAGE, mode, flags=api.F_DS_MATRIX | api.F_DS_BED, width=8)
        assert e.value.code == E_INVALID


# ----------------------------------------------------------------------------- 4. re-runs and capacity
def test_bed_more_rows_than_records(cuda_api, oracle, resident):
    """More rows than the default record capacity: vcfx_cuda_sync runs the launch again; a second launch on the grown
    context is right too."""
    api = cuda_api
    data = G.more_rows_input()
    assert len(data) // 256 + 65536 < data.count(b"\n") - 2
    for mode in MODES:
        b = api.dosage_bed(data, mode, width=2)
        check_bed(api, oracle, data, mode, b, 2, f"more rows mode{mode}")
        ctx = api.Context(api.OP_DOSAGE, mode, **bed_kw(api, 2))
        try:
            for k in range(2):
                got = resident(api, api.OP_DOSAGE, mode, data, ctx=ctx, out_cap=out_cap_for(data, 2))
                same(from_resident(api, got, 2, b.samples), b, f"more rows mode{mode} launch{k}")
        finally:
            ctx.close()


def test_bed_stream_slot_grows(cuda_api, oracle):
    """A streaming output slot far too small for a chunk's rows is grown and the chunk run again."""
    api = cuda_api
    data = G.shape_input(2, 200, 2504)
    for mode in MODES:
        want = api.dosage_bed(data, mode)
        assert want.totals.bytes_out > 25 * 4096
        b = api.dosage_bed(data, mode, out_bytes=4096)
        same(b, want, f"tiny slot mode{mode}")
        assert (b.totals.rows, b.totals.bytes_out) == (want.totals.rows, want.totals.bytes_out)


def test_bed_run_device_output_too_big(cuda_api, oracle, mem):
    """run_device into an output one byte short: VCFX_E_OUTPUT_TOO_BIG with stats.rows filled; a second run sized from
    them is right.  An output that is not 16-byte aligned is refused."""
    api = cuda_api
    data = G.shape_input(3, 200, 2504)
    W = 2504
    for mode in MODES:
        want = api.dosage_bed(data, mode)
        need = want.totals.rows * (16 + row_bytes(W))
        ctx = api.Context(api.OP_DOSAGE, mode, **bed_kw(api, W))
        try:
            d_in = mem.input(data, api.DEVICE_PAD)
            small = mem.output(need - 1)
            ctx.run_device(d_in.addr, len(data), small.addr, need - 1)
            st = api.ChunkStats()
            assert ctx._l.vcfx_cuda_sync(ctx._h, C.byref(st)) == E_OUTPUT_TOO_BIG
            assert st.rows == want.totals.rows and st.bytes_out == need
            out = mem.output(int(st.bytes_out))
            ctx.run_device(d_in.addr, len(data), out.addr, int(st.bytes_out))
            st2 = ctx.sync()
            same(from_resident(api, (out.read(0, int(st2.bytes_out)), st2, []), W, want.samples), want, f"sized from stats mode{mode}")
            with pytest.raises(api.VcfxCudaError) as e:
                ctx.run_device(d_in.addr, len(data), out.addr + 8, int(st.bytes_out) - 8)
            assert e.value.code == E_INVALID
        finally:
            ctx.close()


# ----------------------------------------------------------------------------- 5. reuse, queued launches, a shared upload
def test_bed_context_reuse_and_queued_launches(cuda_api, oracle, resident, mem):
    """One context for a large, a small and the large input again; N launches queued before one sync give one launch's
    result."""
    api = cuda_api
    large = synth.make_vcf(3, 3000, 121, seed=13)
    small = synth.make_vcf(2, 30, 121, seed=14)
    W = 121
    for mode in MODES:
        ref = {id(d): api.dosage_bed(d, mode) for d in (large, small)}
        ctx = api.Context(api.OP_DOSAGE, mode, **bed_kw(api, W))
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


def test_bed_shared_upload_next_to_text(cuda_api, oracle):
    """A .bed context fed by submit_shared from a text dosage context's upload: both give what they give alone."""
    api = cuda_api
    data = synth.make_vcf(3, 1500, 66, seed=31)
    chunk = 32 << 10
    for mode in MODES:
        text_ctx = api.Context(api.OP_DOSAGE, mode, chunk_bytes=chunk)
        bed_ctx = api.Context(api.OP_DOSAGE, mode, chunk_bytes=chunk, **bed_kw(api, 66))
        texts, metas, packed = [], [], []
        try:
            pieces = list(api.chunk_bounds(data, chunk))
            assert len(pieces) > 4
            for s, e in pieces:
                buf, cap = text_ctx.acquire()
                C.memmove(buf, data[s:e], e - s)
                text_ctx.submit(e - s, is_final=(e == len(data)), file_offset=s)
                assert bed_ctx.submit_shared(text_ctx, is_final=(e == len(data)), file_offset=s)
                texts.append(text_ctx.next_output()[0])
                mm, pp = api._ds_split(bed_ctx.next_output()[0], 66, api.F_DS_BED)
                metas.append(mm); packed.append(pp)
        finally:
            text_ctx.close(); bed_ctx.close()
        G._cmp(f"shared upload text mode{mode}", api.DS_HEADER + b"".join(texts), api.dosage_calculator(data, mode).out)
        want = api.dosage_bed(data, mode)
        meta = np.concatenate(metas)
        assert np.array_equal(np.concatenate(packed), want.packed.numpy()), mode
        assert meta["line_offset"].tolist() == want.line_offset.tolist() and meta["n_cols"].tolist() == want.n_cols.tolist(), mode


# ----------------------------------------------------------------------------- 6. rows past 2^32 bytes in one launch
def test_bed_rows_past_4_gib(cuda_api):
    """140,000 sample names, 125,000 one-sample lines: about 5 MB of input, 4.4 GB of packed rows (35,000 bytes each) in
    one launch.  Sample 0 holds the expected call, every other sample is missing (0x55 bytes), and the rows around byte
    2^32 are right (checked on the device)."""
    import torch
    api = cuda_api
    t0 = time.perf_counter()
    S, V = 140000, 125000
    B = row_bytes(S)
    gts, want = (b"0/0", b"0|1", b"1/1", b"./."), (3, 2, 0, 1)
    hdr = b"##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + b"\t".join(b"S%d" % i for i in range(S)) + b"\n"
    lines = [b"1\t%d\t.\tA\tG\t.\t.\t.\tGT\t%s\n" % (i + 1, gts[i % 4]) for i in range(V)]
    data = hdr + b"".join(lines)
    assert V * B > 1 << 32 and S % 4 == 0
    need = V * (16 + B) + len(data) * 4 + (2 << 30)
    free, total = torch.cuda.mem_get_info()
    if free < need:
        pytest.skip(f"needs {need / 1e9:.1f} GB of free device memory, {free / 1e9:.1f} GB are free")
    dev = torch.device("cuda", 0)
    d_in = torch.empty(len(data) + api.DEVICE_PAD, dtype=torch.uint8, device=dev)
    d_in[:len(data)].copy_(torch.frombuffer(bytearray(data), dtype=torch.uint8))
    b = api.dosage_bed_device(d_in, len(data))
    assert len(b.samples) == S and b.packed.shape == (V, B) and b.totals.rows == V
    expect0 = (torch.tensor(want, dtype=torch.uint8, device=dev) | 0x54).repeat(V // 4 + 1)[:V]
    assert torch.equal(b.packed[:, 0], expect0)
    for r0 in range(0, V, 8192):
        assert bool((b.packed[r0:r0 + 8192, 1:] == 0x55).all()), r0
    starts = [len(hdr)]
    for l in lines[:-1]:
        starts.append(starts[-1] + len(l))
    assert b.line_offset.cpu().tolist() == starts and bool((b.n_cols == 1).all()) and not bool(b.no_gt.any())
    r = (1 << 32) // B
    for i in range(r - 2, r + 3):                      # rows that straddle byte 2^32 of the packed part
        row = b.packed[i]
        assert int(row[0]) == want[i % 4] | 0x54 and bool((row[1:] == 0x55).all()), i
    print(f"\nrows past 2^32: {V} x {B} = {V * B / 1e9:.2f} GB in one launch, {b.totals.kernel_ms:.1f} ms of kernels, "
          f"whole test {time.perf_counter() - t0:.1f} s")


# ----------------------------------------------------------------------------- 7. the torch wrappers
def test_bed_torch_wrapper_host(cuda_api, resident):
    """dosage_bed hands back CPU tensors of the documented types, the header's sample names, and what one resident
    launch over the same bytes gives, on a C2-shaped input."""
    import torch
    api = cuda_api
    data = synth.make_vcf(2, 300, 2504, seed=2)
    b = api.dosage_bed(data)
    names = api._ds_prescan(data, api.FILE)[2]
    assert b.samples == names and b.width == len(names) == 2504
    for f, dt in (("packed", torch.uint8), ("line_offset", torch.int64), ("n_cols", torch.int32), ("no_gt", torch.bool)):
        t = getattr(b, f)
        assert t.device.type == "cpu" and t.dtype == dt, f
    assert b.packed.shape == (300, 626) and b.totals.rows == 300
    got = resident(api, api.OP_DOSAGE, api.FILE, data, out_cap=out_cap_for(data, 2504), ctx_kw=bed_kw(api, 2504))
    same(from_resident(api, got, 2504, names), b, "host wrapper vs resident")


def test_bed_torch_wrapper_device(cuda_api):
    """dosage_bed_device on a 50,000-variant C2-shaped input equals dosage_bed on the same bytes; its output feeds a torch
    op on the current stream without an explicit synchronize."""
    import torch
    api = cuda_api
    data = synth.make_vcf(2, 50000, 2504, seed=2)
    host = api.dosage_bed(data)
    assert host.packed.shape == (50000, 626)
    dev = torch.device("cuda", 0)
    d_in = torch.empty(len(data) + api.DEVICE_PAD, dtype=torch.uint8, device=dev)
    side = torch.cuda.Stream(device=dev)

    def hom_a2(p):                                     # calls 11 per row: the samples with dosage 0
        p = p.to(torch.int32)
        return sum(((p >> (2 * k)) & 3 == 3).sum(dim=1) for k in range(4))

    with torch.cuda.stream(side):
        d_in[:len(data)].copy_(torch.frombuffer(bytearray(data), dtype=torch.uint8).to(dev, non_blocking=True))
        b = api.dosage_bed_device(d_in, len(data))
        n = hom_a2(b.packed)                           # queued on `side` behind the library's kernels
        n_host = n.cpu()
    same(b, host, "device wrapper vs streaming")
    assert torch.equal(n_host, hom_a2(host.packed))
    assert b.packed.device == dev and b.packed.dtype == torch.uint8
    assert b.packed.untyped_storage().data_ptr() == b.line_offset.untyped_storage().data_ptr()
    assert (b.totals.rows, b.totals.short_lines, b.err) == (host.totals.rows, host.totals.short_lines, host.err)
