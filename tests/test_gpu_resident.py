"""The device-resident entry point (vcfx_cuda_run_device + vcfx_cuda_sync) — the path bench.py times — for every op in
both input modes, compared two ways:

(a) with the streaming entry points on the same bytes (stream_bytes, one chunk covering the whole input): the text, the
    counters of the stats and the event list must be identical; neither side has host logic the other lacks;
(b) with the oracle, the tool's header row put in front of the resident text, for the ops whose host side is only that
    header row (allele_freq_calc, hwe_tester, missing_detector, nonref_filter, indexer, phase_checker, variant_counter,
    allele_counter, inbreeding_calculator).

genotype_query and dosage_calculator keep host rules in vcfx_b200/api.py — the run ends at a data line in front of the
"#CHROM" line, and genotype_query's stdin mode holds '#' lines back until a data line follows — so they are compared
with (a) only, and only on inputs those rules leave as they are.

Device buffers follow the ABI: the input 16-byte aligned and readable for nbytes + DEVICE_PAD bytes.  On the GPU they
are torch tensors; test_emu_resident.py runs the same tests under the warp emulator, where device memory is host
memory, with aligned ctypes buffers (the `mem` fixture chooses).
"""
import ctypes as C
import functools
import time
from dataclasses import dataclass, field

import pytest

import golden_util
import test_gpu_parity as G
import vcfgen
from vcfx_b200 import synth

pytestmark = pytest.mark.gpu

MODES = (0, 1)
TILES = (0, 512, 4096)


# ----------------------------------------------------------------------------- device memory
class _TorchBuf:
    def __init__(self, t):
        self.t, self.addr, self.cap = t, t.data_ptr(), t.numel()

    def read(self, off, n):
        return self.t[off:off + n].cpu().numpy().tobytes() if n else b""


class TorchMem:
    """Device buffers on cuda:0."""

    def __init__(self):
        import torch
        self.torch = torch
        self.dev = torch.device("cuda", 0)
        self.sm_count = torch.cuda.get_device_properties(0).multi_processor_count

    def input(self, data, pad):
        t = self.torch.empty(len(data) + pad, dtype=self.torch.uint8, device=self.dev)
        if data:
            t[:len(data)].copy_(self.torch.frombuffer(bytearray(data), dtype=self.torch.uint8))
        self.torch.cuda.synchronize()            # the library launches on its own non-blocking stream
        assert t.data_ptr() % 16 == 0
        return _TorchBuf(t)

    def output(self, cap):
        return _TorchBuf(self.torch.empty(max(cap, 1), dtype=self.torch.uint8, device=self.dev))

    def stream(self):
        s = self.torch.cuda.Stream(device=self.dev)
        return s, s.cuda_stream


class _HostBuf:
    def __init__(self, n):
        self.keep = C.create_string_buffer(n + 16)
        self.addr = (C.addressof(self.keep) + 15) & ~15
        self.cap = n

    def read(self, off, n):
        return C.string_at(self.addr + off, n) if n else b""


class HostMem:
    """The warp emulator's device memory is host memory: 16-byte aligned ctypes buffers."""
    sm_count = 2                                  # what the emulator reports (VCFX_EMU_SMS)

    def input(self, data, pad):
        b = _HostBuf(len(data) + pad)
        C.memmove(b.addr, data, len(data))
        return b

    def output(self, cap):
        return _HostBuf(max(cap, 1))

    def stream(self):
        s = C.c_int(0)                            # the emulator runs everything in order and never looks at the handle
        return s, C.addressof(s)


@pytest.fixture
def mem():
    return TorchMem()


# ----------------------------------------------------------------------------- one resident run
def chunk_info(api, op, mode, data):
    """What the streaming wrappers in api.py pass for a whole input, computed by the same helpers."""
    if op in (api.OP_ALLELE_FREQ, api.OP_NONREF_FILTER, api.OP_PHASE_CHECK):
        vf = api.find_chrom_header(data)
        fc = api.first_format_line(data, vf) if (op == api.OP_PHASE_CHECK and mode == api.FILE) else 0
        return dict(valid_from=vf, format_cache_from=fc)
    if op == api.OP_MISSING_DETECT:
        return dict(valid_from=api.first_data_offset(data))
    if op == api.OP_INDEX:
        return dict(valid_from=api._index_header(data, mode)[0])
    return {}


def short_lines(ctx, st):
    n = int(st.n_events)
    if not n:
        return []
    arr = (C.c_uint64 * n)()
    got = C.c_size_t()
    ctx._check(ctx._l.vcfx_cuda_short_lines(ctx._h, arr, n, C.byref(got)))
    return list(arr[:got.value])


def default_out_cap(op, flags, n, n_sel=0):
    text_rows = op == 4 and not (flags & 3)                 # allele_counter TEXT: a row per sample
    return (12 if text_rows else 2) * n + 64 * n_sel + (1 << 20)


def run_resident(mem, api, op, mode, data, *, tile_bytes=0, line_hint=None, out_cap=None, info=None, ctx_kw=None, ctx=None):
    """(text, stats, events) of one vcfx_cuda_run_device over `data` + vcfx_cuda_sync, on `ctx` or a fresh context."""
    ctx_kw = ctx_kw or {}
    own = ctx is None
    if own:
        ctx = api.Context(op, mode, tile_bytes=tile_bytes, **ctx_kw)
    try:
        if line_hint is not None:
            ctx.set_line_hint(line_hint)
        d_in = mem.input(data, api.DEVICE_PAD)
        d_out = mem.output(out_cap or default_out_cap(op, ctx_kw.get("flags", 0), len(data), len(ctx_kw.get("sel_names") or ())))
        ctx.run_device(d_in.addr, len(data), d_out.addr, d_out.cap, **(chunk_info(api, op, mode, data) if info is None else info))
        st = ctx.sync()
        return d_out.read(0, int(st.bytes_out)), st, short_lines(ctx, st)
    finally:
        if own:
            ctx.close()


@pytest.fixture
def resident(mem):
    """resident(api, op, mode, data, *, tile_bytes=0, line_hint=None, out_cap=None, info=None, ctx_kw=None, ctx=None)."""
    return functools.partial(run_resident, mem)


# ----------------------------------------------------------------------------- what each tool hands the library
@dataclass
class Job:
    name: str
    op: int
    mode: int
    data: bytes                      # the bytes the library gets
    ctx_kw: dict = field(default_factory=dict)
    head: bytes = b""                # the header row the tool prints in front of the library's text
    expect: object = None            # () -> the oracle's stdout, or None: compared with the streaming path only
    src: bytes = b""                 # the whole input (missing_detector's last-line rule looks at it)


def _library_request(api, target, call):
    """Run the wrapper `call` with api.<target> replaced by a recorder: ((args, kwargs) it was handed, or None when the
    wrapper answered without the library; the wrapper's result)."""
    seen = []
    real = getattr(api, target)

    def record(*a, **kw):
        seen.append((a, kw))
        return (b"", api.Totals()) if target == "_run" else ([], api.Totals())
    setattr(api, target, record)
    try:
        r = call()
    finally:
        setattr(api, target, real)
    return (seen[0] if seen else None), r


GQ_QUERIES = {0: (("0/1", False), ("1|1", True)), 1: (("1/1", False), ("0|1", True))}
IB_FLAGS = {0: (0, 6), 1: (0, 1)}


def jobs(api, O, data, mode, ops=None):
    """Every op (allele_counter as TEXT, -a and -b in file mode, the stream path in stdin mode) on `data` in `mode`."""
    J = []

    def wanted(name):
        return ops is None or any(name.startswith(o) for o in ops)

    def add(name, op, **kw):
        if wanted(name):
            J.append(Job(name, op, mode, kw.pop("d", data), src=data, **kw))
    add("af", api.OP_ALLELE_FREQ, head=api.AF_HEADER,
        expect=None if (mode == api.STDIN and not data) else (lambda: O.allele_freq(data, mode).out))
    add("hwe", api.OP_HWE, head=api.HWE_HEADER, expect=None if (mode == api.FILE and not data) else (lambda: O.hwe(data, mode).out))
    long_lines = max((len(l) for l in data.split(b"\n")), default=0) > 60000
    # (the reference's file mode overflows its 64 KB line buffer on longer lines: no oracle there)
    add("md", api.OP_MISSING_DETECT, expect=None if (mode == api.FILE and long_lines) else (lambda: O.missing(data, mode).out))
    add("nr", api.OP_NONREF_FILTER, expect=lambda: O.nonref_filter(data, mode).out)
    add("ix", api.OP_INDEX, head=api.INDEX_HEADER if api._index_header(data, mode)[0] < len(data) else b"",
        expect=lambda: O.indexer(data, mode).out)
    add("pc", api.OP_PHASE_CHECK, expect=lambda: O.phase_checker(data, mode).out)
    add("vc", api.OP_VARIANT_COUNT, expect=lambda: O.variant_count(data, mode).out)
    names, start = api._ib_header(data, mode)
    if names and not (mode == api.FILE and not data):
        for fl in IB_FLAGS[mode]:
            add(f"ib flags{fl}", api.OP_INBREEDING, d=data[start:], head=api.IB_HEADER, expect=lambda fl=fl: O.inbreeding(data, mode, fl).out,
                ctx_kw=dict(flags=fl, sel_cols=list(range(len(names))), sel_names=names))
    for q, strict in GQ_QUERIES[mode]:
        if not wanted(f"gq {q} strict{int(strict)}"):
            continue
        req, _ = _library_request(api, "stream_bytes", lambda: api.genotype_query(data, q, mode, strict))
        if req is not None and req[0][1] == data:          # the host rules leave the input as it is
            add(f"gq {q} strict{int(strict)}", api.OP_GENOTYPE_QUERY, ctx_kw=dict(query=q.encode(), flags=api.F_GQ_STRICT if strict else 0))
    req, _ = _library_request(api, "_run", lambda: api.dosage_calculator(data, mode)) if wanted("ds") else (None, None)
    if req is not None:
        add("ds", api.OP_DOSAGE)
    for path, fmt in (((api.AC_MT_TEXT, api.AC_TEXT), (api.AC_UNIFIED, api.AC_AGGREGATE), (api.AC_UNIFIED, api.AC_BINARY))
                      if mode == api.FILE else ((api.AC_STREAM, api.AC_TEXT),)):
        name = f"ac path{path} fmt{fmt}"
        if not wanted(name):
            continue
        req, r = _library_request(api, "_run", lambda: api.allele_counter(data, path, fmt))
        if req is not None:
            (_, _, ac_mode, _), kw = req
            assert ac_mode == mode
            J.append(Job(name, api.OP_ALLELE_COUNT, mode, data, {k: kw[k] for k in ("flags", "sel_cols", "sel_names")}, r.out,
                         lambda path=path, fmt=fmt: _ac_oracle(O, data, path, fmt), data))
    return J


def _ac_oracle(O, data, path, fmt):
    o = O.allele_counter(data, path, fmt)
    assert o.rc == 0
    return o.out


# ----------------------------------------------------------------------------- the two comparisons
STAT_FIELDS = ("bytes_out", "lines", "data_lines", "rows", "flagged", "pre_header", "short_lines", "first_short_line",
               "dots_terminated", "last_unterminated_flagged")


def streamed(api, job, info):
    """(text, Totals, raw events) of the streaming path over job.data as one chunk."""
    n = len(job.data)
    chunk = max(n, 1 << 16)
    events = []
    ctx = api.Context(job.op, job.mode, chunk_bytes=chunk, **job.ctx_kw)
    try:
        if n:
            outs, tot = api.stream_bytes(ctx, job.data, chunk, info.get("valid_from", 0), lambda s, ev: events.extend(ev),
                                         info.get("format_cache_from", 0))
            return b"".join(outs), tot, events
        ctx.acquire()                              # (stream_bytes submits nothing for no bytes; a final chunk of none still reports)
        ctx.submit(0, **info)
        out, st, ev = ctx.next_output()
        tot = api.Totals()
        tot.add(st, 0, [])
        return out, tot, ev
    finally:
        ctx.close()


def tool_stdout(api, job, text, st):
    """What the tool prints for the library's result."""
    if job.op == api.OP_VARIANT_COUNT:
        return b"Total Variants: %d\n" % st.rows
    if job.op == api.OP_MISSING_DETECT and job.mode == api.FILE and st.last_unterminated_flagged and st.dots_terminated == 0:
        # the reference's pre-scan ignores an unterminated last line (api.missing_detector)
        return text[:len(text) - st.last_unterminated_flagged] + job.src[job.src.rfind(b"\n") + 1:]
    return job.head + text


def check(api, job, tag, got, stream=None, want=None):
    """Compare one resident result (text, stats, events) with the streaming result (a) and the oracle's stdout (b)."""
    text, st, events = got
    tag = f"{tag} {job.name} mode{job.mode}"
    assert len(events) == st.n_events, (tag, len(events), st.n_events)
    if stream is not None:
        s_text, s_tot, s_events = stream
        G._cmp(f"{tag} resident vs streaming", text, s_text)
        for f in STAT_FIELDS:
            assert getattr(st, f) == getattr(s_tot, f), (tag, f, getattr(st, f), getattr(s_tot, f))
        assert events == s_events, (tag, "events", events[:8], s_events[:8])
    if want is not None:
        G._cmp(f"{tag} resident vs oracle", tool_stdout(api, job, text, st), want)


def run_jobs(resident, api, O, data, tag, tiles=TILES, modes=MODES, ops=None):
    for mode in modes:
        for job in jobs(api, O, data, mode, ops):
            info = chunk_info(api, job.op, mode, job.data)
            stream = streamed(api, job, info)
            want = job.expect() if job.expect else None
            for tile in tiles:
                got = resident(api, job.op, mode, job.data, tile_bytes=tile, ctx_kw=job.ctx_kw)
                check(api, job, f"{tag} tile{tile}", got, stream, want)


# ----------------------------------------------------------------------------- 1. every op on the parity corpora
SWEEP = [(shape, S) for shape in (1, 2, 3) for S in G.SWEEP_S if 119 <= S <= 130 or S in (255, 256, 257, 511)]
QUIRKS = sorted(k for k in golden_util.load() if k.endswith("_quirks"))


@pytest.mark.parametrize("shape,V,S", G.SHAPES)
def test_resident_synthetic_shapes(cuda_api, oracle, resident, shape, V, S):
    run_jobs(resident, cuda_api, oracle, G.shape_input(shape, V, S), f"shape{shape} {V}x{S}")


@pytest.mark.parametrize("seed", range(40))
def test_resident_adversarial(cuda_api, oracle, resident, seed):
    run_jobs(resident, cuda_api, oracle, G.adversarial_input(seed), f"fuzz{seed}")


def test_resident_empty_and_degenerate(cuda_api, oracle, resident):
    for data in G.DEGENERATE:
        run_jobs(resident, cuda_api, oracle, data, repr(data[:20]))


@pytest.mark.parametrize("name", QUIRKS)
def test_resident_quirks_fixtures(cuda_api, oracle, resident, name):
    data, _ = golden_util.load()[name]
    run_jobs(resident, cuda_api, oracle, data, name)


@pytest.mark.parametrize("shape,S", SWEEP)
def test_resident_line_lengths_sweep(cuda_api, oracle, resident, shape, S):
    run_jobs(resident, cuda_api, oracle, G.sweep_input(shape, S), f"sweep shape{shape} S{S}")


# ----------------------------------------------------------------------------- 2. line hints change no result
WARPS_PER_CTA = 8                                  # vcfx_kernels.cuh
MIN_TILE, MAX_TILE = 32 << 10, 256 << 10


def tile_for(nbytes, warps, line_hint=0):
    """vcfx_api.cu tile_for, restated: about four tiles per resident warp within [32 KiB, 256 KiB]; a line hint asks for at
    least eight lines per tile while every resident warp still gets two tiles."""
    t = nbytes // (warps * 4 + 1)
    t = min(MAX_TILE, max(MIN_TILE, (t + 511) & ~511))
    if line_hint:
        want = min((line_hint * 8 + 511) & ~511, 8 << 20)
        room = (nbytes // (warps * 2 + 1)) & ~511
        t = max(t, min(want, room))
    return t


def blocks_per_sm(mem, op):
    """The library's CTAs per SM: the occupancy query capped at the kernels' __launch_bounds__ minimum (five for
    variant_counter, four for the others), which sm_100a reaches; the warp emulator reports one."""
    return 1 if isinstance(mem, HostMem) else (5 if op == 0 else 4)


def test_resident_line_hints_change_no_result(cuda_api, oracle, resident, mem):
    """vcfx_cuda_set_line_hint picks larger tiles for long lines and "changes no result" (vcfx_cuda.h): no hint, the right
    one, 1 byte and 6 MiB give the same text, stats and events, on an input large enough for them to give different tiles."""
    api, O = cuda_api, oracle
    warps = mem.sm_count * blocks_per_sm(mem, 1) * WARPS_PER_CTA
    S = 1250                                         # 5 KB lines: eight of them fill a tile between the two bounds below
    V = int(1.45 * MIN_TILE * (2 * warps + 1)) // (4 * S + 40)
    data = synth.make_vcf(3, V, S, seed=61)
    fd = api.first_data_offset(data)
    line = data.index(b"\n", fd) + 1 - fd
    hints = (None, line, 1, 6 << 20)
    for op in (0, 1):
        w = mem.sm_count * blocks_per_sm(mem, op) * WARPS_PER_CTA
        none, right, one, huge = (tile_for(len(data), w, h or 0) for h in hints)
        assert one == none and huge != none, (op, none, right, huge)
        if op:
            assert none < right < huge, (none, right, huge)
    # (allele_counter's TEXT rows would be ten times the input here: its -a / -b forms stand for it)
    ops = ("af", "hwe", "md", "nr", "ix", "pc", "vc", "ib", "gq", "ds", "ac path2")
    for mode in MODES:
        for job in jobs(api, O, data, mode, ops):
            base = resident(api, job.op, mode, job.data, ctx_kw=job.ctx_kw)
            check(api, job, "hints none", base, streamed(api, job, chunk_info(api, job.op, mode, job.data)) if job.expect is None else None,
                  job.expect() if job.expect else None)
            for h in hints[1:]:
                got = resident(api, job.op, mode, job.data, ctx_kw=job.ctx_kw, line_hint=h)
                check(api, job, f"hint {h}", got, (base[0], base[1], base[2]))


# ----------------------------------------------------------------------------- 3. vcfx_cuda_sync runs a launch again
def launch_twice(resident, api, O, data, tag, ops, modes=MODES):
    """Each job on one context, twice: the first launch outgrows what the context was sized for and is run again inside
    vcfx_cuda_sync; the second finds the grown buffers.  Both equal the oracle."""
    ran = set()
    for mode in modes:
        for job in jobs(api, O, data, mode, ops):
            want = job.expect()
            ctx = api.Context(job.op, mode, **job.ctx_kw)
            try:
                for k in range(2):
                    got = resident(api, job.op, mode, job.data, ctx=ctx, ctx_kw=job.ctx_kw)
                    check(api, job, f"{tag} launch{k}", got, None, want)
            finally:
                ctx.close()
            ran.add(job.name.split()[0] if not job.name.startswith("ac") else job.name)
    return ran


def test_resident_rerun_more_rows_than_records(cuda_api, oracle, resident):
    data = G.more_rows_input()
    rows = data.count(b"\n") - 2
    assert len(data) // 256 + 65536 < rows           # default_rec_cap (vcfx_api.cu): too few records for the first launch
    ran = launch_twice(resident, cuda_api, oracle, data, "more rows", ("af", "hwe", "md", "ix", "ac path2 fmt1"))
    assert ran == {"af", "hwe", "md", "ix", "ac path2 fmt1"}


def test_resident_rerun_allele_counter_row_sizes(cuda_api, oracle, resident):
    """allele_counter TEXT rows are sized for one-digit counts; two-digit and wrapped counts make the launch run again."""
    ran = launch_twice(resident, cuda_api, oracle, G.two_digit_counts_input(), "two-digit counts", ("ac path0",), modes=(0,))
    assert ran == {"ac path0 fmt0"}


def test_resident_rerun_inbreeding_panels(cuda_api, oracle, resident):
    """4,000 samples, two columns on most lines: more rows x samples than the panels were sized for."""
    launch_twice(resident, cuda_api, oracle, G.ib_few_columns_input(), "ib few columns", ("ib",))


def test_resident_phase_checker_event_list_grows(cuda_api, oracle, resident):
    data, n = G.pc_dropped_lines_input()
    launch_twice(resident, cuda_api, oracle, data, "pc 2^20+ dropped", ("pc",), modes=(0,))
    text, st, events = resident(cuda_api, cuda_api.OP_PHASE_CHECK, 0, data)
    assert st.flagged == n and len(events) == n and all(e & 3 == cuda_api.PC_SHORT for e in events)


# ----------------------------------------------------------------------------- 4. one context, large / small / large
def test_resident_context_reuse_across_sizes(cuda_api, oracle, resident):
    """Tile arrays, records and tile_resume sized for a large launch are reused by a small one and the large one again:
    nothing stale may leak from one launch into the next."""
    api, O = cuda_api, oracle
    large = synth.make_vcf(3, 3000, 120, seed=13)
    small = synth.make_vcf(2, 30, 120, seed=14)
    assert api._ib_header(large, 0)[0] == api._ib_header(small, 0)[0]
    for mode in MODES:
        jl = {j.name: j for j in jobs(api, O, large, mode)}
        js = {j.name: j for j in jobs(api, O, small, mode)}
        assert jl.keys() == js.keys()
        for name, job in jl.items():
            assert js[name].ctx_kw == job.ctx_kw
            ref = {}
            for j in (job, js[name]):
                ref[id(j)] = (streamed(api, j, chunk_info(api, j.op, mode, j.data)), j.expect() if j.expect else None)
            ctx = api.Context(job.op, mode, **job.ctx_kw)
            try:
                for k, j in enumerate((job, js[name], job)):
                    check(api, j, f"reuse step{k}", resident(api, j.op, mode, j.data, ctx=ctx, ctx_kw=j.ctx_kw), *ref[id(j)])
            finally:
                ctx.close()


# ----------------------------------------------------------------------------- 5. queued launches, as bench.py times them
def test_resident_queued_launches(cuda_api, oracle, resident, mem):
    """N run_device calls queued before one sync give one launch's text and stats; allele_freq_calc and variant_counter on
    two contexts that share one stream, queued step after step, as bench.py's headline loop runs them."""
    api, O = cuda_api, oracle
    data = synth.make_vcf(3, 2000, 64, seed=21)
    N = 4
    for mode in MODES:
        for job in jobs(api, O, data, mode):
            one = resident(api, job.op, mode, job.data, ctx_kw=job.ctx_kw)
            ctx = api.Context(job.op, mode, **job.ctx_kw)
            try:
                d_in = mem.input(job.data, api.DEVICE_PAD)
                d_out = mem.output(default_out_cap(job.op, job.ctx_kw.get("flags", 0), len(job.data), len(job.ctx_kw.get("sel_names") or ())))
                for _ in range(N):
                    ctx.run_device(d_in.addr, len(job.data), d_out.addr, d_out.cap, **chunk_info(api, job.op, mode, job.data))
                st = ctx.sync()
                check(api, job, f"queued x{N}", (d_out.read(0, int(st.bytes_out)), st, short_lines(ctx, st)), (one[0], one[1], one[2]))
            finally:
                ctx.close()
    data = vcfgen.make_vcf(5, n_lines=3000, n_samples=6, header="late")      # short lines and data in front of the header
    keep, stream = mem.stream()
    d_in = mem.input(data, api.DEVICE_PAD)
    d_out = mem.output(4 << 20)
    af = api.Context(api.OP_ALLELE_FREQ, api.FILE, stream=stream)
    vc = api.Context(api.OP_VARIANT_COUNT, api.FILE, stream=stream)
    try:
        vf = api.find_chrom_header(data)
        for _ in range(N):
            af.run_device(d_in.addr, len(data), d_out.addr, d_out.cap, valid_from=vf)
            vc.run_device(d_in.addr, len(data), 0, 0)
        st_af, st_vc = af.sync(), vc.sync()
        ev_vc = short_lines(vc, st_vc)
        G._cmp("shared stream af", api.AF_HEADER + d_out.read(0, int(st_af.bytes_out)), O.allele_freq(data, 0).out)
        o = O.variant_count(data, 0)
        assert (st_vc.rows, st_vc.short_lines, len(ev_vc)) == (o.rows, o.warnings, o.warnings)
        assert st_vc.short_lines > 0 and st_af.pre_header > 0
        _, tot, ev = streamed(api, Job("vc", api.OP_VARIANT_COUNT, 0, data), {})
        assert ev_vc == ev and st_vc.first_short_line == tot.first_short_line
    finally:
        af.close(); vc.close()
    del keep


# ----------------------------------------------------------------------------- 6. inbreeding_calculator across resident calls
def test_resident_inbreeding_across_calls(cuda_api, oracle, resident, mem):
    """The per-sample sums live in the context from call to call: newline-aligned pieces with is_final=0 on all but the
    last give the one-shot result; a second stream through the same context starts again."""
    api, O = cuda_api, oracle
    first = synth.make_vcf(3, 2000, 40, seed=5)
    second = synth.make_vcf(2, 1500, 40, seed=6)
    for mode in MODES:
        names, _ = api._ib_header(first, mode)
        assert names == api._ib_header(second, mode)[0]
        for fl in IB_FLAGS[mode]:
            kw = dict(flags=fl, sel_cols=list(range(len(names))), sel_names=names)
            ctx = api.Context(api.OP_INBREEDING, mode, **kw)
            try:
                for data in (first, second, first):
                    body = data[api._ib_header(data, mode)[1]:]
                    one = resident(api, api.OP_INBREEDING, mode, body, ctx_kw=kw)
                    want = O.inbreeding(data, mode, fl).out
                    G._cmp(f"ib one shot mode{mode} flags{fl}", api.IB_HEADER + one[0], want)
                    pieces = list(api.chunk_bounds(body, 16 << 10))
                    assert len(pieces) > 3
                    d_out = mem.output(1 << 20)
                    rows = 0
                    for s, e in pieces:
                        d_in = mem.input(body[s:e], api.DEVICE_PAD)
                        ctx.run_device(d_in.addr, e - s, d_out.addr, d_out.cap, is_final=(e == len(body)), file_offset=s)
                        st = ctx.sync()
                        rows += st.rows
                    G._cmp(f"ib pieces mode{mode} flags{fl}", api.IB_HEADER + d_out.read(0, int(st.bytes_out)), want)
                    assert rows == one[1].rows
            finally:
                ctx.close()


# ----------------------------------------------------------------------------- 7. one launch past 4 GiB
BIG_BYTES = 9 << 29                                   # 4.5 GiB
BIG_HEADER = (b"##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t"
              + b"\t".join(b"S%d" % i for i in range(100)) + b"\n")


def big_piece():
    """100 data lines, self-contained (starts at a line start, ends with '\\n', needs nothing from the lines in front):
    a short line (variant_counter's numbers and events, phase_checker drops it), a line with missing calls
    (missing_detector rewrites it, phase_checker drops it), an all-hom-ref line (nonref_filter and genotype_query drop
    it) and an unphased one (phase_checker drops it).  The first line has a FORMAT column, so phase_checker's FORMAT
    cache is the same in every copy; every copy has a dotted line, so missing_detector's pre-scan finds one in the piece
    as in the whole file."""
    gts = [b"0|1", b"1|0", b"1|1", b"0|0"]
    lines = []
    for k in range(100):
        g = [gts[(i * 3 + k) % 4] for i in range(100)]
        g[k % 100] = b"0|1"
        if k == 30:
            lines.append(b"2\t%d\tshort\n" % (k + 1))
            continue
        if k == 50:
            g[7] = b"./."; g[60] = b"0|."
        if k == 70:
            g = [b"0|0"] * 100
        if k == 90:
            g[11] = b"0/1"
        lines.append(b"1\t%d\trs%d\tA\tG\t50\tPASS\tDP=%d\tGT\t" % (1000 + k, k, k) + b"\t".join(g) + b"\n")
    return b"".join(lines)


def test_resident_one_launch_past_4_gib(cuda_api, oracle, mem):
    """One launch over ~4.6 GB (header + k copies of big_piece): output offsets of the copy ops, indexer's file offsets,
    variant_counter's line numbers and every op's row count pass 2^32.  The expected text follows from the oracle on the
    header plus one piece; the device output is compared copy by copy on the device, and a copy that differs is copied
    back and shown."""
    import torch
    api, O = cuda_api, oracle
    t_all = time.perf_counter()
    H, P = BIG_HEADER, big_piece()
    k = (BIG_BYTES - len(H)) // len(P) + 1
    n = len(H) + k * len(P)
    one = H + P
    # expected: header part + k x piece part, for the ops whose text has no absolute numbers
    fixed = {}
    for name, fn, head in (("af", lambda d: O.allele_freq(d, 0).out, api.AF_HEADER), ("hwe", lambda d: O.hwe(d, 0).out, api.HWE_HEADER),
                           ("md", lambda d: O.missing(d, 0).out, b""), ("nr", lambda d: O.nonref_filter(d, 0).out, b""),
                           ("pc", lambda d: O.phase_checker(d, 0).out, b""), ("gq 0/1 strict0", lambda d: O.genotype_query(d, "0/1", 0, False)[0].out, b""),
                           ("ds", lambda d: O.dosage(d, 0).out, api.DS_HEADER), ("ac path2 fmt1", lambda d: O.allele_counter(d, O.AC_UNIFIED, O.AC_AGGREGATE).out, api.AC_AGG_HEADER)):
        a, b = fn(H), fn(one)
        assert a.startswith(head) and b.startswith(a), name
        fixed[name] = (a[len(head):], b[len(a):])
    for name in ("md", "nr", "pc", "gq 0/1 strict0"):
        x, y = fixed[name]
        assert len(x) + k * len(y) > (1 << 32) + (64 << 20), (name, len(x) + k * len(y))     # output offsets past 2^32
    ix_one = O.indexer(one, 0).out.split(b"\n")[1:-1]
    vc_job = jobs(api, O, one, 0, ("vc",))[0]
    _, vc_tot, vc_ev = streamed(api, vc_job, {})
    assert vc_tot.short_lines == 1 and vc_ev == [H.count(b"\n") + 31]
    out_cap = max(len(x) + k * len(y) for x, y in fixed.values()) + (1 << 20)
    free, total = torch.cuda.mem_get_info()
    need = (n + api.DEVICE_PAD) + out_cap + n + (2 << 30)     # input, output, dosage_calculator's code per input byte, work
    if free < need:
        pytest.skip(f"needs {need / 1e9:.1f} GB of free device memory, {free / 1e9:.1f} GB of {total / 1e9:.1f} GB are free")
    dev = torch.device("cuda", 0)
    d_in = torch.empty(n + api.DEVICE_PAD, dtype=torch.uint8, device=dev)
    d_in[:len(H)].copy_(torch.frombuffer(bytearray(H), dtype=torch.uint8))
    d_in[len(H):n].view(k, len(P)).copy_(torch.frombuffer(bytearray(P), dtype=torch.uint8).to(dev).expand(k, len(P)))
    d_out = torch.empty(out_cap, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    times = {}

    def launch(job):
        t0 = time.perf_counter()
        ctx = api.Context(job.op, api.FILE, **job.ctx_kw)
        try:
            ctx.run_device(d_in.data_ptr(), n, d_out.data_ptr(), out_cap, **chunk_info(api, job.op, api.FILE, one))
            st = ctx.sync()
            ev = short_lines(ctx, st)
        finally:
            ctx.close()
        times[job.name] = time.perf_counter() - t0
        return st, ev

    def compare_copies(tag, off, y):
        yd = torch.frombuffer(bytearray(y), dtype=torch.uint8).to(dev)
        per = max(1, (256 << 20) // len(y))
        for j in range(0, k, per):
            m = min(per, k - j)
            blk = d_out[off + j * len(y): off + (j + m) * len(y)].view(m, len(y))
            bad = (blk != yd).any(dim=1)
            if bool(bad.any()):
                c = j + int(bad.nonzero()[0])
                G._cmp(f"{tag}: copy {c} of {k} (output offset {off + c * len(y)})", blk[c - j].cpu().numpy().tobytes(), y)

    all_jobs = {j.name: j for j in jobs(api, O, one, 0)}
    for name, (x, y) in fixed.items():
        st, _ = launch(all_jobs[name])
        assert st.bytes_out == len(x) + k * len(y), (name, st.bytes_out, len(x) + k * len(y))
        G._cmp(f">4 GiB {name} header part", d_out[:len(x)].cpu().numpy().tobytes(), x)
        compare_copies(f">4 GiB {name}", len(x), y)
    # indexer: the file offsets of copy c are those of the first copy plus c x len(piece)
    st, _ = launch(all_jobs["ix"])
    rows = [(l.rsplit(b"\t", 1)[0] + b"\t", int(l.rsplit(b"\t", 1)[1])) for l in ix_one]
    assert st.rows == k * len(rows)
    pos, per = 0, 4096
    for c0 in range(0, k, per):
        exp = b"".join(pre + b"%d\n" % (off + c * len(P)) for c in range(c0, min(k, c0 + per)) for pre, off in rows)
        G._cmp(f">4 GiB ix copies {c0}..", d_out[pos:pos + len(exp)].cpu().numpy().tobytes(), exp)
        pos += len(exp)
    assert pos == st.bytes_out and rows[-1][1] + (k - 1) * len(P) > 1 << 32
    # variant_counter: k x the rows, short-line numbers shifted by the lines of a piece
    st, ev = launch(all_jobs["vc"])
    o = O.variant_count(one, 0)
    lines_p = P.count(b"\n")
    assert (st.rows, st.short_lines, st.first_short_line) == (k * o.rows, k, vc_ev[0])
    assert ev == [vc_ev[0] + c * lines_p for c in range(k)]
    print(f"\n>4 GiB launch: {n} bytes ({k} copies of a {len(P)}-byte piece); seconds per op (launch + sync): "
          + ", ".join(f"{a} {b:.2f}" for a, b in times.items()) + f"; whole test {time.perf_counter() - t_all:.1f} s")
