"""ctypes mirror of ``include/vcfx_cuda.h`` plus the host-side logic the five tools share.

This is the Python twin of the C++ host code in ``vcfx_b200/tools``: header pre-parse,
newline-aligned chunking, the fixed header rows, and totals — everything per-record happens
in ``libvcfx_cuda.so`` on the GPU.  There is no CPU fallback: if the library is missing, or
no CUDA device is usable, the calls raise :class:`VcfxCudaError`.

Function names follow the reference tools (``allele_freq_calc``, ``hwe_tester``,
``missing_detector``, ``variant_counter``, ``allele_counter``) and take the same two input
modes the reference has: ``FILE`` (``tool -i file``, mmap semantics) and ``STDIN``.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from pathlib import Path

from . import build as _build

OP_VARIANT_COUNT, OP_ALLELE_FREQ, OP_HWE, OP_MISSING_DETECT, OP_ALLELE_COUNT, OP_NONREF_FILTER, OP_INDEX, OP_PHASE_CHECK, OP_INBREEDING, OP_GENOTYPE_QUERY, OP_DOSAGE = range(11)
FILE, STDIN = 0, 1
F_AC_AGGREGATE, F_AC_BINARY, F_AC_FORWARD = 1, 2, 4
DEVICE_PAD = 8192

E_BUSY, E_EMPTY = -5, -6

AF_HEADER = b"CHROM\tPOS\tID\tREF\tALT\tAllele_Frequency\n"      # allele_freq_calc.cpp:353
HWE_HEADER = b"CHROM\tPOS\tID\tREF\tALT\tHWE_pvalue\n"            # hwe_tester.cpp:463
AC_TEXT_HEADER = b"CHROM\tPOS\tID\tREF\tALT\tSample\tRef_Count\tAlt_Count\n"            # allele_counter.cpp:908
AC_AGG_HEADER = b"CHROM\tPOS\tID\tREF\tALT\tTotal_Ref\tTotal_Alt\tSample_Count\n"        # :1359


class VcfxCudaError(RuntimeError):
    def __init__(self, code: int, what: str):
        super().__init__(f"libvcfx_cuda: {what} (code {code})")
        self.code = code


class Cfg(C.Structure):
    _fields_ = [("device", C.c_int32), ("op", C.c_int32), ("mode", C.c_int32), ("flags", C.c_uint32),
                ("chunk_bytes", C.c_size_t), ("out_bytes", C.c_size_t), ("n_slots", C.c_int32),
                ("tile_bytes", C.c_int32), ("stream", C.c_void_p),
                ("n_sel", C.c_uint32), ("sel_col", C.POINTER(C.c_uint32)), ("sel_names", C.c_char_p),
                ("sel_name_off", C.POINTER(C.c_uint32))]


class ChunkInfo(C.Structure):
    _fields_ = [("data_valid_from", C.c_uint64), ("is_final", C.c_int32), ("reserved", C.c_int32), ("file_offset", C.c_uint64),
                ("format_cache_from", C.c_uint64)]


class ChunkStats(C.Structure):
    _fields_ = [("bytes_in", C.c_uint64), ("bytes_out", C.c_uint64), ("lines", C.c_uint64),
                ("data_lines", C.c_uint64), ("rows", C.c_uint64), ("flagged", C.c_uint64),
                ("pre_header", C.c_uint64), ("short_lines", C.c_uint64), ("first_short_line", C.c_uint64),
                ("n_events", C.c_uint64), ("dots_terminated", C.c_uint64),
                ("last_unterminated_flagged", C.c_uint64), ("kernel_ms", C.c_float), ("reserved", C.c_float)]


EXPORTS = ["vcfx_cuda_abi_version", "vcfx_cuda_device_count", "vcfx_cuda_strerror", "vcfx_cuda_last_error",
           "vcfx_cuda_create", "vcfx_cuda_destroy", "vcfx_cuda_acquire_input", "vcfx_cuda_submit",
           "vcfx_cuda_submit_host", "vcfx_cuda_submit_shared", "vcfx_cuda_set_line_hint", "vcfx_cuda_next_output", "vcfx_cuda_in_flight", "vcfx_cuda_short_lines",
           "vcfx_cuda_run_device", "vcfx_cuda_sync", "vcfx_cuda_hwe_pvalues",
           "vcfx_cuda_king_create", "vcfx_cuda_king_destroy", "vcfx_cuda_king_add", "vcfx_cuda_king_counts", "vcfx_cuda_king_slab_rows"]

_lib = None


def lib_path() -> Path:
    import os
    alt = os.environ.get("VCFX_CUDA_LIB")          # an alternative build of the same library (kernel experiments)
    return Path(alt) if alt else _build.CUDA_LIB


def load():
    """Load libvcfx_cuda.so (building it is the job of __graft_entry__.build / build.build_cuda)."""
    global _lib
    if _lib is None:
        p = lib_path()
        if not p.exists():
            raise VcfxCudaError(-2, f"{p} is not built; run `python -c 'import __graft_entry__ as g; g.build()'`"
                                    " — there is no CPU fallback")
        l = C.CDLL(str(p))
        l.vcfx_cuda_strerror.restype = C.c_char_p
        l.vcfx_cuda_last_error.restype = C.c_char_p
        l.vcfx_cuda_last_error.argtypes = [C.c_void_p]
        l.vcfx_cuda_create.argtypes = [C.POINTER(Cfg), C.POINTER(C.c_void_p)]
        l.vcfx_cuda_destroy.argtypes = [C.c_void_p]
        l.vcfx_cuda_acquire_input.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]
        l.vcfx_cuda_submit.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(ChunkInfo)]
        l.vcfx_cuda_submit_host.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(ChunkInfo)]
        l.vcfx_cuda_submit_shared.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(ChunkInfo)]
        l.vcfx_cuda_set_line_hint.argtypes = [C.c_void_p, C.c_size_t]
        l.vcfx_cuda_next_output.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.POINTER(ChunkStats)]
        l.vcfx_cuda_in_flight.argtypes = [C.c_void_p]
        l.vcfx_cuda_short_lines.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.c_size_t, C.POINTER(C.c_size_t)]
        l.vcfx_cuda_run_device.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(ChunkInfo), C.c_void_p, C.c_size_t]
        l.vcfx_cuda_sync.argtypes = [C.c_void_p, C.POINTER(ChunkStats)]
        l.vcfx_cuda_hwe_pvalues.argtypes = [C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]
        l.vcfx_cuda_king_create.argtypes = [C.c_int, C.c_uint32, C.c_void_p, C.POINTER(C.c_void_p)]
        l.vcfx_cuda_king_destroy.argtypes = [C.c_void_p]
        l.vcfx_cuda_king_add.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int]
        l.vcfx_cuda_king_counts.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_uint64)]
        l.vcfx_cuda_king_slab_rows.argtypes = [C.c_void_p]
        l.vcfx_cuda_king_slab_rows.restype = C.c_uint64
        _lib = l
    return _lib


def hwe_pvalues(counts, device: int = 0):
    """hwe_tester's p-value computed on the device for an int32 array [n, 3] of (homRef, het, homAlt)."""
    import numpy as np
    c = np.ascontiguousarray(counts, dtype=np.int32).reshape(-1, 3)
    out = np.empty(len(c), dtype=np.float64)
    rc = load().vcfx_cuda_hwe_pvalues(device, c.ctypes.data, len(c), out.ctypes.data)
    if rc != 0:
        raise VcfxCudaError(rc, load().vcfx_cuda_strerror(rc).decode())
    return out


def device_count() -> int:
    n = C.c_int(0)
    load().vcfx_cuda_device_count(C.byref(n))
    return n.value


@dataclass
class Totals:
    bytes_in: int = 0
    bytes_out: int = 0
    lines: int = 0
    data_lines: int = 0
    rows: int = 0
    flagged: int = 0
    pre_header: int = 0
    short_lines: int = 0
    first_short_line: int = 0          # 1-based, over the whole input
    short_line_numbers: list = field(default_factory=list)
    dots_terminated: int = 0
    last_unterminated_flagged: int = 0
    kernel_ms: float = 0.0
    chunks: int = 0

    def add(self, s: ChunkStats, line_base: int, events):
        self.bytes_in += s.bytes_in; self.bytes_out += s.bytes_out
        self.data_lines += s.data_lines; self.rows += s.rows; self.flagged += s.flagged
        self.pre_header += s.pre_header; self.short_lines += s.short_lines
        if s.first_short_line and not self.first_short_line:
            self.first_short_line = line_base + s.first_short_line
        self.short_line_numbers += [line_base + e for e in events]
        self.lines += s.lines
        self.dots_terminated += s.dots_terminated
        self.last_unterminated_flagged = s.last_unterminated_flagged
        self.kernel_ms += s.kernel_ms; self.chunks += 1


class Context:
    """One GPU context (``vcfx_ctx``)."""

    def __init__(self, op: int, mode: int = FILE, device: int = 0, flags: int = 0, chunk_bytes: int = 0,
                 out_bytes: int = 0, n_slots: int = 0, tile_bytes: int = 0, stream: int | None = None,
                 sel_cols=None, sel_names=None, query: bytes | None = None, width: int | None = None):
        self._l = load()
        self._h = C.c_void_p()
        cfg = Cfg(device=device, op=op, mode=mode, flags=flags, chunk_bytes=chunk_bytes, out_bytes=out_bytes,
                  n_slots=n_slots, tile_bytes=tile_bytes, stream=stream)
        self._keep = []
        if sel_cols is not None:
            n = len(sel_cols)
            cols = (C.c_uint32 * max(n, 1))(*sel_cols)
            blob = b"".join(nm + b"\t" for nm in sel_names)
            offs = [0]
            for nm in sel_names:
                offs.append(offs[-1] + len(nm) + 1)
            off_arr = (C.c_uint32 * (n + 1))(*offs)
            cfg.n_sel = n; cfg.sel_col = cols; cfg.sel_names = blob; cfg.sel_name_off = off_arr
            self._keep = [cols, blob, off_arr]
        if query is not None:                      # genotype_query: the -g argument travels in sel_names, its length in n_sel
            cfg.n_sel = len(query); cfg.sel_names = query
            self._keep = [query]
        if width is not None:                      # dosage_calculator matrix mode: W, the sample columns of the matrix
            cfg.n_sel = int(width)
        self._check(self._l.vcfx_cuda_create(C.byref(cfg), C.byref(self._h)))
        self.op, self.mode = op, mode

    def _check(self, rc: int):
        if rc != 0:
            msg = self._l.vcfx_cuda_strerror(rc).decode()
            if self._h:
                extra = self._l.vcfx_cuda_last_error(self._h).decode()
                if extra:
                    msg += ": " + extra
            raise VcfxCudaError(rc, msg)

    def close(self):
        if self._h:
            self._l.vcfx_cuda_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- streaming path ------------------------------------------------------------------
    def acquire(self):
        buf = C.c_void_p(); cap = C.c_size_t()
        rc = self._l.vcfx_cuda_acquire_input(self._h, C.byref(buf), C.byref(cap))
        if rc == E_BUSY:
            return None, 0
        self._check(rc)
        return buf.value, cap.value

    def submit(self, nbytes: int, valid_from: int = 0, is_final: bool = True, file_offset: int = 0, format_cache_from: int = 0):
        info = ChunkInfo(valid_from, int(is_final), 0, file_offset, format_cache_from)
        self._check(self._l.vcfx_cuda_submit(self._h, nbytes, C.byref(info)))

    def submit_host(self, host_ptr: int, nbytes: int, valid_from: int = 0, is_final: bool = True, file_offset: int = 0, format_cache_from: int = 0) -> bool:
        """Submit a chunk straight from caller memory; False when every slot is in flight."""
        info = ChunkInfo(valid_from, int(is_final), 0, file_offset, format_cache_from)
        rc = self._l.vcfx_cuda_submit_host(self._h, host_ptr, nbytes, C.byref(info))
        if rc == E_BUSY:
            return False
        self._check(rc)
        return True

    def submit_shared(self, primary: "Context", valid_from: int = 0, is_final: bool = True, file_offset: int = 0, format_cache_from: int = 0) -> bool:
        """Run this context's op on the chunk last submitted to ``primary`` (no second upload)."""
        info = ChunkInfo(valid_from, int(is_final), 0, file_offset, format_cache_from)
        rc = self._l.vcfx_cuda_submit_shared(self._h, primary._h, C.byref(info))
        if rc == E_BUSY:
            return False
        self._check(rc)
        return True

    def set_line_hint(self, line_bytes: int) -> None:
        """Typical bytes per data line, for run_device callers (the host never sees their bytes)."""
        self._check(self._l.vcfx_cuda_set_line_hint(self._h, int(line_bytes)))

    def in_flight(self) -> int:
        return self._l.vcfx_cuda_in_flight(self._h)

    def next_output(self):
        text = C.c_void_p(); n = C.c_size_t(); st = ChunkStats()
        self._check(self._l.vcfx_cuda_next_output(self._h, C.byref(text), C.byref(n), C.byref(st)))
        out = C.string_at(text.value, n.value) if n.value else b""
        events = []
        if st.n_events:
            cap = int(st.n_events)
            arr = (C.c_uint64 * cap)(); got = C.c_size_t()
            self._check(self._l.vcfx_cuda_short_lines(self._h, arr, cap, C.byref(got)))
            events = list(arr[: got.value])
        return out, st, events

    def next_output_raw(self):
        """Like next_output, without copying the text out of the library's pinned buffer: (address, length, stats).
        The buffer is valid until the next call on this context."""
        text = C.c_void_p(); n = C.c_size_t(); st = ChunkStats()
        self._check(self._l.vcfx_cuda_next_output(self._h, C.byref(text), C.byref(n), C.byref(st)))
        return text.value, n.value, st

    # -- device-resident path ------------------------------------------------------------
    def run_device(self, d_in: int, nbytes: int, d_out: int, out_cap: int, valid_from: int = 0, is_final: bool = True, file_offset: int = 0, format_cache_from: int = 0):
        info = ChunkInfo(valid_from, int(is_final), 0, file_offset, format_cache_from)
        self._check(self._l.vcfx_cuda_run_device(self._h, d_in, nbytes, C.byref(info), d_out, out_cap))

    def sync(self) -> ChunkStats:
        st = ChunkStats()
        self._check(self._l.vcfx_cuda_sync(self._h, C.byref(st)))
        return st


# ----------------------------------------------------------------------------- host logic
def find_chrom_header(data) -> int:
    """Offset of the first line that starts with ``#CHROM`` (len(data) if none): data lines
    before it are skipped by allele_freq_calc (allele_freq_calc.cpp:372-386, 492-502)."""
    if bytes(data[:6]) == b"#CHROM":
        return 0
    i = data.find(b"\n#CHROM")
    return len(data) if i < 0 else i + 1


def chunk_bounds(data, chunk_bytes: int):
    """Newline-aligned [start, end) pieces of at most chunk_bytes (the last may be unterminated)."""
    n = len(data)
    pos = 0
    while pos < n:
        end = min(n, pos + chunk_bytes)
        if end < n:
            cut = data.rfind(b"\n", pos, end)
            if cut < 0:
                raise VcfxCudaError(-1, f"a line longer than chunk_bytes={chunk_bytes} starts at byte {pos}")
            end = cut + 1
        yield pos, end
        pos = end


def stream_bytes(ctx: Context, data, chunk_bytes: int, valid_abs: int = 0, on_events=None, fmt0_abs: int = 0):
    """Push ``data`` through ctx's streaming pipeline; returns (list of output pieces, Totals).  ``on_events(chunk_start,
    events)`` is called per drained chunk, in order, with its raw event list (phase_checker) instead of adding the
    events to the totals as line numbers."""
    tot = Totals()
    outs = []
    line_base = 0
    starts = []

    def drain():
        nonlocal line_base
        out, st, ev = ctx.next_output()
        outs.append(out)
        start = starts.pop(0)
        if on_events is not None:
            if ev:
                on_events(start, ev)
            ev = []
        tot.add(st, line_base, ev)
        line_base += st.lines

    mv = memoryview(data)
    n = len(data)
    for s, e in chunk_bounds(data, chunk_bytes):
        buf, cap = ctx.acquire()
        while buf is None:
            drain()
            buf, cap = ctx.acquire()
        assert e - s <= cap
        C.memmove(buf, (C.c_char * (e - s)).from_buffer_copy(mv[s:e]), e - s)
        vf = min(max(valid_abs - s, 0), e - s)
        ctx.submit(e - s, valid_from=vf, is_final=(e == n), file_offset=s, format_cache_from=min(max(fmt0_abs - s, 0), e - s))
        starts.append(s)
        # line numbers: chunks are drained in order, so the base is exact when drained
    while ctx.in_flight():
        drain()
    return outs, tot


_ctx_cache: dict = {}


def _cached_context(op, mode, device, flags, chunk_bytes, **kw):
    """Contexts are reusable once drained; creating one costs pinned and device allocations, so the
    helpers below keep a few around (allele_counter contexts carry a selection and are not cached)."""
    if "sel_cols" in kw and op != OP_INBREEDING:
        return Context(op, mode, device=device, flags=flags, chunk_bytes=chunk_bytes, **kw), False
    key = (op, mode, device, flags, chunk_bytes, tuple(sorted((k, tuple(v) if isinstance(v, list) else v) for k, v in kw.items())))
    ctx = _ctx_cache.get(key)
    if ctx is None:
        if len(_ctx_cache) >= 24:
            _ctx_cache.pop(next(iter(_ctx_cache))).close()
        ctx = _ctx_cache[key] = Context(op, mode, device=device, flags=flags, chunk_bytes=chunk_bytes, **kw)
    return ctx, True


def close_cached_contexts():
    while _ctx_cache:
        _ctx_cache.popitem()[1].close()


import atexit  # noqa: E402
atexit.register(close_cached_contexts)


def _stream(op: int, data, mode: int, chunk_bytes: int, flags: int = 0, device: int = 0, valid_abs: int = 0, fmt0_abs: int = 0,
            on_events=None, final_if_empty: bool = False, **kw):
    """One stream of ``data`` through a context of ``op`` from _cached_context: (list of output pieces, Totals), as
    stream_bytes.  The chunk size defaults to the input rounded up to 1 MiB, at most 64 MiB (pinned allocations are not
    free).  On any exception the context leaves the cache and is closed: chunks of the failed stream may still be in
    flight in it, and the next stream would drain them.  ``final_if_empty``: no bytes are still submitted, as one final
    chunk (inbreeding_calculator reports with its final chunk)."""
    chunk_bytes = chunk_bytes or min(64 << 20, max(1 << 20, (len(data) + (1 << 20) - 1) & ~((1 << 20) - 1)))
    ctx, cached = _cached_context(op, mode, device, flags, chunk_bytes, **kw)
    try:
        if len(data) == 0 and final_if_empty:
            ctx.acquire()
            ctx.submit(0, is_final=True)
            out, st, _ = ctx.next_output()
            tot = Totals(); tot.add(st, 0, [])
            outs = [out]
        else:
            outs, tot = stream_bytes(ctx, data, chunk_bytes, valid_abs, on_events, fmt0_abs)
    except Exception:
        if cached:
            _ctx_cache.pop(next(k for k, v in _ctx_cache.items() if v is ctx), None)
        ctx.close()
        raise
    if not cached:
        ctx.close()
    return outs, tot


def _run(op: int, data: bytes, mode: int, chunk_bytes: int, **kw):
    valid_abs = find_chrom_header(data) if op in (OP_ALLELE_FREQ, OP_NONREF_FILTER, OP_PHASE_CHECK) else 0
    fmt0_abs = first_format_line(data, valid_abs) if (op == OP_PHASE_CHECK and mode == FILE) else 0
    outs, tot = _stream(op, data, mode, chunk_bytes, valid_abs=valid_abs, fmt0_abs=fmt0_abs, **kw)
    return b"".join(outs), tot


@dataclass
class ToolResult:
    out: bytes
    rc: int
    totals: Totals
    err: bytes = b""            # what the tool prints on stderr (phase_checker)


def allele_freq_calc(data: bytes, mode: int = FILE, chunk_bytes: int = 0, **kw) -> ToolResult:
    if mode == STDIN and len(data) == 0:          # allele_freq_calc.cpp:638-641 prints help, rc 1
        return ToolResult(b"", 1, Totals())
    body, tot = _run(OP_ALLELE_FREQ, data, mode, chunk_bytes, **kw)
    return ToolResult(AF_HEADER + body, 0, tot)


def hwe_tester(data: bytes, mode: int = FILE, chunk_bytes: int = 0, **kw) -> ToolResult:
    if mode == FILE and len(data) == 0:           # hwe_tester.cpp:456 no header for an empty file
        return ToolResult(b"", 0, Totals())
    body, tot = _run(OP_HWE, data, mode, chunk_bytes, **kw)
    return ToolResult(HWE_HEADER + body, 0, tot)


def first_data_offset(data) -> int:
    """Offset of the first line that does not start with '#': the end of the leading header block
    (missing_detector.cpp:378-383 starts its pre-scan there)."""
    pos = 0
    n = len(data)
    while pos < n and data[pos:pos + 1] == b"#":
        nl = data.find(b"\n", pos)
        if nl < 0:
            return n
        pos = nl + 1
    return pos


def first_format_line(data, start: int = 0) -> int:
    """Offset of the first data line at or behind ``start`` that has eight tabs and a non-empty FORMAT column behind them
    (len(data) when there is none): VCFX_phase_checker's file mode treats an empty FORMAT column as "GT first" for the
    lines in front of it (its FORMAT cache starts as ("", 0), VCFX_phase_checker.cpp:486-488, :313-316)."""
    pos, n = start, len(data)
    while pos < n:
        nl = data.find(b"\n", pos)
        le = n if nl < 0 else nl
        line = bytes(data[pos:le])
        if line.endswith(b"\r"):
            line = line[:-1]
        if line and not line.startswith(b"#"):
            f = line.split(b"\t", 9)
            if len(f) >= 9 and f[8] != b"":
                return pos
        pos = le + 1
    return n


def missing_detector(data: bytes, mode: int = FILE, chunk_bytes: int = 0, **kw) -> ToolResult:
    outs, tot = _stream(OP_MISSING_DETECT, data, mode, chunk_bytes, valid_abs=first_data_offset(data), **kw)
    if mode == FILE and tot.last_unterminated_flagged and tot.dots_terminated == 0:
        # The reference's pre-scan ignores an unterminated last line (missing_detector.cpp:354): when
        # no other line has a '.' in its sample columns it copies the file verbatim, so that last
        # line stays as it was.
        body = b"".join(outs)
        cut = len(body) - tot.last_unterminated_flagged
        last = data[data.rfind(b"\n") + 1:]
        return ToolResult(body[:cut] + last, 0, tot)
    return ToolResult(b"".join(outs), 0, tot)


INDEX_HEADER = b"CHROM\tPOS\tFILE_OFFSET\n"                     # VCFX_indexer.cpp:283 / :364


def _index_header(data: bytes, mode: int):
    """(offset of the first line VCFX_indexer takes for the "#CHROM" line or len(data), whether a data line came before
    any '#' line).  File mode: blanks / tabs, then "#CHROM" (VCFX_indexer.cpp:108-122); stdin mode: white space, then a
    first field that is exactly "#CHROM" with a second field behind it (:349-356)."""
    pos, n, saw_hash, warned = 0, len(data), False, False
    ws = b" \t" if mode == FILE else b" \t\n\v\f\r"
    while pos < n:
        nl = data.find(b"\n", pos)
        le = n if nl < 0 else nl
        line = data[pos:le]
        if line.endswith(b"\r"):
            line = line[:-1]
        if line:
            t = line.lstrip(ws)
            if t.startswith(b"#"):
                saw_hash = True
                if (mode == FILE and len(line) >= 6 and t.startswith(b"#CHROM")) or (mode == STDIN and t.startswith(b"#CHROM\t")):
                    return pos, warned
            elif not saw_hash:
                warned = True
        pos = le + 1
    return n, warned


def indexer(data: bytes, mode: int = FILE, chunk_bytes: int = 0, **kw) -> ToolResult:
    """VCFX_indexer: CHROM, POS and byte offset of every data line behind the "#CHROM" line.  totals.pre_header = 1 when
    the tool prints "Error: no #CHROM header found before variant lines."."""
    hdr_off, warned = _index_header(data, mode)
    outs, tot = _stream(OP_INDEX, data, mode, chunk_bytes, valid_abs=hdr_off, **kw)
    tot.pre_header = int(warned)
    return ToolResult((INDEX_HEADER if hdr_off < len(data) else b"") + b"".join(outs), 0, tot)


def nonref_filter(data: bytes, mode: int = FILE, chunk_bytes: int = 0, **kw) -> ToolResult:
    """VCFX_nonref_filter: data lines behind the "#CHROM" line whose samples are all homozygous reference are dropped,
    every other line is written as its content + '\\n' (VCFX_nonref_filter.cpp:458-548 file mode, :553-631 stdin mode).
    totals.pre_header = data lines in front of the header (each prints a warning), totals.flagged = lines dropped."""
    body, tot = _run(OP_NONREF_FILTER, data, mode, chunk_bytes, **kw)
    return ToolResult(body, 0, tot)


F_IB_GLOBAL, F_IB_SKIP_BOUNDARY, F_IB_COUNT_BOUNDARY = 1, 2, 4
IB_HEADER = b"Sample\tInbreedingCoefficient\n"                    # VCFX_inbreeding_calculator.cpp:639
IB_MESSAGES = {0: b"", 1: b"Error: Empty file.\n", 2: b"Error: No #CHROM line or no samples found.\n", 3: b"No biallelic variants found.\n",
               4: b"Error: No #CHROM line found.\n", 5: b"Error: No sample columns found.\n"}


def _ib_header(data: bytes, mode: int):
    """(sample names or None when no "#CHROM" line was found, offset the data lines start at).  File mode: the leading block
    of '#' and empty lines; EVERY line in it that starts with "#CHROM" adds its columns 10.. (VCFX_inbreeding_calculator.cpp
    :474-513).  Stdin mode: the first '#' line that contains "#CHROM" anywhere; lines in front of it do not count (:689-706)."""
    names, found, pos, n = [], False, 0, len(data)
    while pos < n:
        nl = data.find(b"\n", pos)
        le = n if nl < 0 else nl
        line = data[pos:le]
        if line.endswith(b"\r"):
            line = line[:-1]
        nxt = le + 1
        if mode == FILE:
            if line:
                if not line.startswith(b"#"):
                    return (names if found else None), pos
                if line.startswith(b"#CHROM"):
                    found = True
                    f = line.split(b"\t")
                    if f and f[-1] == b"":                 # nothing is read behind a final tab
                        f = f[:-1]
                    names += f[9:]
        elif line.startswith(b"#") and b"#CHROM" in line:
            return line.split(b"\t")[9:], nxt
        pos = nxt
    return (names if found else None), n


def inbreeding_calculator(data: bytes, mode: int = FILE, freq_global: bool = False, skip_boundary: bool = False,
                          count_boundary: bool = False, quiet: bool = True, chunk_bytes: int = 0, **kw) -> ToolResult:
    """VCFX_inbreeding_calculator: per-sample F = 1 - observed / expected heterozygotes over the biallelic sites, the
    expectation summed in file order (calculateInbreedingMmap :456-668, calculateInbreedingStdin :670-826).  The scan leaves
    a genotype code per sample column, a second pass walks the sites in order with one thread per sample; the state lives
    in the context from chunk to chunk and the text arrives with the final chunk.  ``err`` = what goes to stderr,
    totals.rows = sites used."""
    if mode == FILE and len(data) == 0:
        return ToolResult(IB_HEADER, 0, Totals(), IB_MESSAGES[1])
    names, start = _ib_header(data, mode)
    if mode == FILE and not names:
        return ToolResult(IB_HEADER, 0, Totals(), IB_MESSAGES[2])
    if mode == STDIN and names is None:
        return ToolResult(IB_HEADER, 0, Totals(), IB_MESSAGES[4])
    if mode == STDIN and not names:
        return ToolResult(IB_HEADER, 0, Totals(), IB_MESSAGES[5])
    flags = (F_IB_GLOBAL if freq_global else 0) | (F_IB_SKIP_BOUNDARY if skip_boundary else 0) | (F_IB_COUNT_BOUNDARY if count_boundary else 0)
    # (a context is good for one stream after the other: the per-sample state starts again behind a final chunk; with no
    # data line at all, a final chunk of nothing still reports)
    outs, tot = _stream(OP_INBREEDING, data[start:], mode, chunk_bytes, flags=flags, final_if_empty=True,
                        sel_cols=list(range(len(names))), sel_names=names, **kw)
    err = IB_MESSAGES[3] if (tot.rows == 0 and not quiet) else b""
    return ToolResult(IB_HEADER + b"".join(outs), 0, tot, err)


DS_HEADER = b"CHROM\tPOS\tID\tREF\tALT\tDosages\n"           # VCFX_dosage_calculator.cpp:414
DS_WARNING = b"Warning: Skipping VCF line with fewer than 10 fields.\n"
DS_ERROR = b"Error: VCF header (#CHROM) not found before variant records.\n"


def _ds_prescan(data, mode: int):
    """dosage_calculator's host rule, applied to the lines up to the first data line: (offset of the first data line or
    len(data), whether a "#CHROM" line came before it, the sample names of the first "#CHROM" line — its columns from index
    9, a '\\r' in front of the '\\n' and an empty column behind a final tab left out)."""
    pos, n, found, names = 0, len(data), False, []
    while pos < n:                                       # up to the first data line
        nl = data.find(b"\n", pos)
        le = n if nl < 0 else nl
        line = data[pos:le]
        if mode == FILE and line.endswith(b"\r"):
            line = line[:-1]
        if line:
            if not line.startswith(b"#"):
                return pos, found, names
            if line.startswith(b"#CHROM") and not found:
                found = True
                f = bytes(line[:-1] if (mode != FILE and line.endswith(b"\r")) else line).split(b"\t")[9:]
                names = f[:-1] if f and f[-1] == b"" else f
        pos = le + 1
    return n, found, names


def dosage_calculator(data: bytes, mode: int = FILE, quiet: bool = False, chunk_bytes: int = 0, **kw) -> ToolResult:
    """VCFX_dosage_calculator: per data line "CHROM..ALT \\t d,d,NA,.." (processFileMmap :375-591, calculateDosage :209-366).
    A data line in front of the "#CHROM" line ends the run with nothing on stdout (exit code 1 in file mode); an empty FILE
    gives nothing at all; stdin mode prints its warnings even with -q."""
    if mode == FILE and len(data) == 0:
        return ToolResult(b"", 0, Totals())
    first_data, found, _ = _ds_prescan(data, mode)
    if first_data < len(data) and not found:
        return ToolResult(b"", 1 if mode == FILE else 0, Totals(), DS_ERROR)
    body, tot = _run(OP_DOSAGE, data, mode, chunk_bytes, **kw)
    warn = b"" if (quiet and mode == FILE) else DS_WARNING * tot.short_lines
    return ToolResult(DS_HEADER + body, 0, tot, warn)


F_DS_MATRIX, F_DS_BED = 1, 2
DS_ROW_BYTES = 16                                      # vcfx_ds_row: uint64 line_offset, uint32 n_cols, uint32 flags
BED_MAGIC = b"\x6c\x1b\x01"                            # PLINK 1 .bed: the two magic bytes, then 01 = variant-major


@dataclass
class DosageMatrix:
    """dosage_calculator's rows as numbers: row i is the row the tool prints for the line at byte line_offset[i].
    codes[i, s] = 0 / 1 / 2 the dosage, -1 "NA" (every column of a line without a GT key too), -2 the line has no column s;
    columns beyond the width are dropped (n_cols keeps the true count, totals.flagged counts such rows)."""
    samples: list                  # the "#CHROM" line's columns from index 9
    codes: object                  # int8 [rows, W]
    line_offset: object            # int64 [rows]
    n_cols: object                 # int32 [rows]
    no_gt: object                  # bool [rows]: the line has no GT key (the tool prints "NA" alone)
    totals: Totals
    err: bytes = b""               # the warnings the tool prints on stderr


@dataclass
class DosageBed:
    """The same rows as PLINK 1 .bed rows (variant-major, A1 = ALT, A2 = REF): packed[i] holds the calls of row i, sample s
    at bits 2 (s & 3) of byte s >> 2 — 00 dosage 2 (on a multi-allelic line: two non-REF alleles), 10 dosage 1, 11
    dosage 0, 01 missing ("NA", no GT key, or no column s), 00 padding from the width on.  BED_MAGIC followed by the rows
    of packed is a .bed file."""
    samples: list                  # the "#CHROM" line's columns from index 9
    width: int                     # W: samples per row
    packed: object                 # uint8 [rows, ceil(W / 4)]
    line_offset: object            # int64 [rows]
    n_cols: object                 # int32 [rows]
    no_gt: object                  # bool [rows]
    totals: Totals
    err: bytes = b""


def _ds_matrix_prescan(data, mode: int):
    """(sample names) after dosage_calculator's host rule: a data line in front of the "#CHROM" line ends the tool's run."""
    first_data, found, names = _ds_prescan(data, mode)
    if first_data < len(data) and not found:
        raise VcfxCudaError(-1, DS_ERROR.decode().rstrip("\n"))
    return names


def _ds_row_bytes(flags: int, width: int) -> int:
    """Bytes of a row behind its metadata: W int8 codes, or ceil(W / 4) packed .bed bytes."""
    return (width + 3) // 4 if flags & F_DS_BED else width


def _ds_split(piece: bytes, width: int, flags: int = F_DS_MATRIX):
    """(metadata, codes or packed bytes) numpy views of one chunk's matrix or .bed output."""
    import numpy as np
    nb = _ds_row_bytes(flags, width)
    rows = len(piece) // (DS_ROW_BYTES + nb)
    meta = np.frombuffer(piece, dtype=np.dtype([("line_offset", "<u8"), ("n_cols", "<u4"), ("flags", "<u4")]), count=rows)
    body = np.frombuffer(piece, dtype=np.uint8 if flags & F_DS_BED else np.int8, count=rows * nb, offset=DS_ROW_BYTES * rows)
    return meta, body.reshape(rows, nb)


def _ds_host(data, mode: int, width, chunk_bytes: int, flags: int, kw):
    """One stream of host bytes in the matrix or .bed layout: (names, W, metadata, rows of codes or packed bytes, Totals)."""
    import numpy as np
    names = [] if (mode == FILE and len(data) == 0) else _ds_matrix_prescan(data, mode)
    W = len(names) if width is None else int(width)
    metas, bodies, tot = [], [], Totals()
    if len(data):
        outs, tot = _stream(OP_DOSAGE, data, mode, chunk_bytes, flags=flags, width=W, **kw)
        for piece in outs:
            m, b = _ds_split(piece, W, flags)
            metas.append(m); bodies.append(b)
    empty = _ds_split(b"", W, flags)
    meta = np.concatenate(metas) if metas else empty[0]
    body = np.ascontiguousarray(np.concatenate(bodies)) if bodies else empty[1].copy()
    return names, W, meta, body, tot


def _ds_meta_host(meta):
    """line_offset, n_cols, no_gt as CPU tensors."""
    import numpy as np
    import torch
    return (torch.from_numpy(meta["line_offset"].astype(np.int64)), torch.from_numpy(meta["n_cols"].astype(np.int32)),
            torch.from_numpy((meta["flags"] & 1).astype(bool)))


def dosage_matrix(data: bytes, mode: int = FILE, width: int | None = None, chunk_bytes: int = 0, **kw) -> DosageMatrix:
    """dosage_calculator's genotypes as an int8 variants x samples matrix (CPU tensors), through the streaming path.  The
    width defaults to the number of samples of the "#CHROM" line.  Raises VcfxCudaError with the tool's error text when a
    data line comes before the "#CHROM" line."""
    import torch
    names, W, meta, code, tot = _ds_host(data, mode, width, chunk_bytes, F_DS_MATRIX, kw)
    return DosageMatrix(names, torch.from_numpy(code), *_ds_meta_host(meta), tot, DS_WARNING * tot.short_lines)


def dosage_bed(data: bytes, mode: int = FILE, width: int | None = None, chunk_bytes: int = 0, **kw) -> DosageBed:
    """dosage_calculator's genotypes as PLINK 1 .bed rows (CPU tensors), through the streaming path; otherwise as
    dosage_matrix.  BED_MAGIC + packed.numpy().tobytes() is the .bed file of the rows."""
    import torch
    names, W, meta, packed, tot = _ds_host(data, mode, width, chunk_bytes, F_DS_BED, kw)
    return DosageBed(names, W, torch.from_numpy(packed), *_ds_meta_host(meta), tot, DS_WARNING * tot.short_lines)


def _ds_device_head(d_in, nbytes: int, mode: int):
    """The sample names, read back from the leading lines of a device input only: the bytes up to the first data line."""
    k = min(nbytes, 1 << 16)
    while True:
        head = d_in[:k].cpu().numpy().tobytes()
        cut = k if k == nbytes else head.rfind(b"\n") + 1         # complete lines only, unless that is the whole input
        first_data, _, _ = _ds_prescan(head[:cut], mode)
        if first_data < cut or k == nbytes:
            return _ds_matrix_prescan(head[:cut], mode)
        k = min(nbytes, 4 * k)


def _ds_device(d_in, nbytes: int, mode: int, width, line_hint: int, flags: int):
    """One resident launch in the matrix or .bed layout on torch's current stream: (names, W, metadata views, rows of codes
    or packed bytes as a uint8 view, Totals), the views into one output tensor."""
    import torch
    if d_in.dtype != torch.uint8 or not d_in.is_cuda or d_in.numel() < nbytes + DEVICE_PAD or d_in.data_ptr() % 16:
        raise VcfxCudaError(-1, "d_in must be a 16-byte aligned uint8 CUDA tensor of at least nbytes + DEVICE_PAD bytes")
    names = [] if (mode == FILE and nbytes == 0) else _ds_device_head(d_in, nbytes, mode)
    W = len(names) if width is None else int(width)
    nb = _ds_row_bytes(flags, W)
    lines = 1
    for s in range(0, nbytes, 1 << 28):                     # (bounded temporaries for inputs of several GB)
        lines += int((d_in[s:min(nbytes, s + (1 << 28))] == 10).sum())
    out = torch.empty(max(lines * (DS_ROW_BYTES + nb), DS_ROW_BYTES), dtype=torch.uint8, device=d_in.device)
    stream = torch.cuda.current_stream(d_in.device)
    tot = Totals()
    rows = 0
    if nbytes:
        with Context(OP_DOSAGE, mode, device=d_in.device.index or 0, flags=flags, width=W, stream=stream.cuda_stream) as ctx:
            if line_hint:
                ctx.set_line_hint(line_hint)
            ctx.run_device(d_in.data_ptr(), nbytes, out.data_ptr(), out.numel())
            st = ctx.sync()
        tot.add(st, 0, [])
        rows = int(st.rows)
    meta = out[:DS_ROW_BYTES * rows].view(rows, DS_ROW_BYTES)
    body = out[DS_ROW_BYTES * rows:DS_ROW_BYTES * rows + rows * nb].view(rows, nb)
    return names, W, (meta.view(torch.int64)[:, 0], meta.view(torch.int32)[:, 2], meta[:, 12].view(torch.bool)), body, tot


def dosage_matrix_device(d_in, nbytes: int, mode: int = FILE, width: int | None = None, line_hint: int = 0) -> DosageMatrix:
    """dosage_matrix for an input already on the device: d_in is a uint8 CUDA tensor of at least nbytes + DEVICE_PAD bytes
    (16-byte aligned).  Only the leading '#' block comes back to the host.  The output is sized from a newline count on
    the device (rows <= lines) and the library runs on torch.cuda.current_stream(), so torch work behind it is ordered
    after it; codes, line_offset, n_cols and no_gt are views into one output tensor on the same device."""
    import torch
    names, W, meta, body, tot = _ds_device(d_in, nbytes, mode, width, line_hint, F_DS_MATRIX)
    return DosageMatrix(names, body.view(torch.int8), *meta, tot, DS_WARNING * tot.short_lines)


def dosage_bed_device(d_in, nbytes: int, mode: int = FILE, width: int | None = None, line_hint: int = 0) -> DosageBed:
    """dosage_bed for an input already on the device, as dosage_matrix_device: packed, line_offset, n_cols and no_gt are
    views into one output tensor on the same device, written on torch.cuda.current_stream()."""
    names, W, meta, body, tot = _ds_device(d_in, nbytes, mode, width, line_hint, F_DS_BED)
    return DosageBed(names, W, body, *meta, tot, DS_WARNING * tot.short_lines)


@dataclass
class KingCounts:
    """KING-robust relatedness counts over every ordered pair of samples (include/vcfx_cuda.h, "pairwise relatedness"):
    cc[i, j] both called, hh[i, j] both het, ab[i, j] i hom A2 (REF/REF) and j hom A1, hc[i, j] i het and j called.
    int64 tensors [n, n] (CUDA tensors unless counts(device=False) asked for CPU ones)."""
    cc: object
    hh: object
    ab: object
    hc: object
    rows: int                      # rows added
    samples: list | None = None    # the "#CHROM" line's sample names (king() only)

    @property
    def nsnp(self):
        return self.cc

    @property
    def hethet(self):
        return self.hh

    @property
    def ibs0(self):
        return self.ab + self.ab.T

    @property
    def het1(self):
        return self.hc

    @property
    def het2(self):
        return self.hc.T

    def kinship(self):
        """KING's between-family robust kinship, float64 [n, n]:
        0.5 - (HET1 + HET2 - 2 HETHET + 4 IBS0) / (4.0 * min(HET1, HET2)), NaN where min(HET1, HET2) = 0."""
        import torch
        het1, het2 = self.het1, self.het2
        num = (het1 + het2 - 2 * self.hh + 4 * self.ibs0).double()
        den = torch.minimum(het1, het2)
        k = 0.5 - num / (4.0 * den.double())
        return torch.where(den == 0, torch.full_like(k, float("nan")), k)


class King:
    """Accumulator of KING counts (``vcfx_king``) on one GPU.  add() takes PLINK 1 .bed rows — a DosageBed, or a uint8
    tensor [rows, ceil(n_samples / 4)] on the CPU or on this device — and counts() returns a KingCounts.  The library
    runs on `stream` (a cudaStream_t handle, 0 = the default stream; None = torch's current stream of the device).
    Device rows given to add() and the tensor counts() writes are ordered after the work queued on torch's current stream
    at the call, and device rows stay allocated until the library's stream has read them, whichever stream that is."""

    def __init__(self, n_samples: int, device: int = 0, stream: int | None = None):
        self._l = load()
        self._h = C.c_void_p()
        self.n_samples, self.device = int(n_samples), int(device)
        if self.n_samples <= 0:
            raise ValueError("King needs at least one sample")
        if self.n_samples > 0xFFFFFFFF:
            raise ValueError(f"{self.n_samples} samples do not fit the library's uint32 n_samples")
        if stream is None:
            import torch
            stream = torch.cuda.current_stream(self.device).cuda_stream
        self._stream = int(stream or 0)
        rc = self._l.vcfx_cuda_king_create(self.device, self.n_samples, stream or None, C.byref(self._h))
        if rc != 0:
            raise VcfxCudaError(rc, self._l.vcfx_cuda_strerror(rc).decode())
        self.row_bytes = (self.n_samples + 3) // 4
        self.slab_rows = int(self._l.vcfx_cuda_king_slab_rows(self._h))

    def close(self):
        if self._h:
            self._l.vcfx_cuda_king_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        self.close()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _add(self, ptr: int, n_rows: int, on_device: bool):
        rc = self._l.vcfx_cuda_king_add(self._h, ptr, n_rows, int(on_device))
        if rc != 0:
            raise VcfxCudaError(rc, self._l.vcfx_cuda_strerror(rc).decode())

    def _after_current_stream(self, *used):
        """The library's stream waits for the work queued so far on torch's current stream (which writes the tensors the
        library is about to touch), and the caching allocator reuses none of `used` before the library's stream has
        read it.  Nothing to do when the library runs on the current stream."""
        import torch
        cur = torch.cuda.current_stream(self.device)
        if cur.cuda_stream == self._stream:
            return
        mine = torch.cuda.ExternalStream(self._stream, device=self.device) if self._stream else torch.cuda.default_stream(self.device)
        mine.wait_stream(cur)
        for t in used:
            t.record_stream(mine)

    def add(self, x) -> None:
        import numpy as np
        import torch
        if isinstance(x, DosageBed):
            if x.width != self.n_samples:
                raise ValueError(f"the rows are {x.width} samples wide, the accumulator has {self.n_samples}")
            x = x.packed
        if isinstance(x, np.ndarray):
            x = torch.from_numpy(x)
        if x.dtype != torch.uint8 or x.dim() != 2 or x.shape[1] != self.row_bytes:
            raise ValueError(f"want uint8 rows [n, {self.row_bytes}] for {self.n_samples} samples, got {x.dtype} {tuple(x.shape)}")
        if x.is_cuda and x.device.index != self.device:
            raise ValueError(f"the rows are on cuda:{x.device.index}, the accumulator on cuda:{self.device}")
        x = x.contiguous()
        if x.is_cuda:
            self._after_current_stream(x)
        self._add(x.data_ptr(), x.shape[0], x.is_cuda)

    def counts(self, device: bool = True) -> KingCounts:
        """Waits for the rows added so far and returns their counts (int64 tensors on this device, or on the CPU)."""
        import torch
        n = self.n_samples
        rows = C.c_uint64(0)
        if device:
            out = torch.empty((4, n, n), dtype=torch.int32, device=f"cuda:{self.device}")
            self._after_current_stream()                # (out is not recorded: the call returns once its stream wrote it)
            rc = self._l.vcfx_cuda_king_counts(self._h, out.data_ptr(), 1, C.byref(rows))
            big = out.to(torch.int64) & 0xFFFFFFFF
        else:
            import numpy as np
            out = np.empty((4, n, n), dtype=np.uint32)
            rc = self._l.vcfx_cuda_king_counts(self._h, out.ctypes.data, 0, C.byref(rows))
            big = torch.from_numpy(out.astype(np.int64))
        if rc != 0:
            raise VcfxCudaError(rc, self._l.vcfx_cuda_strerror(rc).decode())
        return KingCounts(big[0], big[1], big[2], big[3], int(rows.value))


def king(data: bytes, mode: int = FILE, width: int | None = None, chunk_bytes: int = 0, **kw) -> KingCounts:
    """KING counts of a VCF's genotypes: dosage_bed's rows (the streaming path, same rules and errors) into one King on
    device 0.  Raises ValueError when there are no samples."""
    bed = dosage_bed(data, mode, width, chunk_bytes, **kw)
    with King(bed.width) as k:
        k.add(bed)
        r = k.counts()
    r.samples = bed.samples
    return r


F_GQ_STRICT = 1


def genotype_query(data: bytes, query: str, mode: int = FILE, strict: bool = False, quiet: bool = False, chunk_bytes: int = 0, **kw) -> ToolResult:
    """VCFX_genotype_query -g query [--strict]: '#' lines pass, empty lines vanish, a data line passes when one of its
    samples has the queried genotype (VCFX_genotype_query.cpp:433-517 file mode, :527-614 stdin mode).  What depends on
    the lines before or behind is settled here: the run ends at a data line that comes before the "#CHROM" line (file
    mode has written the '#' lines in front of it by then, stdin mode nothing), and stdin mode holds '#' lines back until
    the next data line, so those behind the last data line never appear.  ``err`` = the text on stderr without -q."""
    q = query.encode()
    assert q, "the tool prints its usage line for an empty query"
    n, pos, found, first_data, last_data_end = len(data), 0, False, None, 0
    while pos < n:
        nl = data.find(b"\n", pos)
        le = n if nl < 0 else nl
        if le > pos:
            if data[pos:pos + 1] == b"#":
                if first_data is None and data[pos:pos + 6] == b"#CHROM":
                    found = True
            else:
                if first_data is None:
                    first_data = pos
                    if not found:
                        break
                last_data_end = min(le + 1, n)
        pos = le + 1
    msgs = []
    if first_data is not None and not found:
        body = data[:first_data] if mode == FILE else b""
        msgs.append(b"Error: No #CHROM header found before data lines.\n")
    elif first_data is None:
        body = data if mode == FILE else b""
        if mode == STDIN and not found:
            msgs.append(b"Error: No #CHROM line found in VCF.\n")
    else:
        body = data if mode == FILE else data[:last_data_end]
    warn = []

    def on_events(start, events):
        for ev in events:
            off = start + (ev >> 2)
            nl = body.find(b"\n", off)
            line = bytes(body[off:len(body) if nl < 0 else nl])
            warn.append(b"Warning: skipping line with <9 fields" + (b"" if mode == FILE else b": " + line) + b"\n")

    tot = Totals(); out = b""
    if body:
        outs, tot = _stream(OP_GENOTYPE_QUERY, body, mode, chunk_bytes, flags=F_GQ_STRICT if strict else 0, on_events=on_events,
                            query=q, **kw)
        out = b"".join(outs)
    return ToolResult(out, 0, tot, b"" if quiet else b"".join(warn + msgs))


PC_UNPHASED, PC_PRE_HEADER, PC_SHORT, PC_NO_GT = range(4)      # why VCFX_OP_PHASE_CHECK dropped a line (event & 3)


def phase_checker(data: bytes, mode: int = FILE, quiet: bool = False, chunk_bytes: int = 0, **kw) -> ToolResult:
    """VCFX_phase_checker: '#' lines and empty lines pass, a data line passes when it lies behind the "#CHROM" line, has
    ten columns and a GT key and every sample is fully phased (VCFX_phase_checker.cpp:470-558 file mode, :563-650 stdin
    mode).  The device reports every dropped line (offset, reason); ``err`` is the text the tool prints for them on
    stderr without -q.  totals.flagged = lines dropped."""
    msgs = []

    def on_events(start, events):
        for ev in events:
            off, why = start + (ev >> 2), ev & 3
            if why == PC_PRE_HEADER:
                msgs.append(b"Warning: Data line encountered before #CHROM header; skipping line.\n")
            elif why == PC_SHORT:
                msgs.append(b"Warning: Invalid VCF line with fewer than 10 columns; skipping line.\n")
            elif why == PC_NO_GT:
                msgs.append(b"Warning: GT field not found; skipping line.\n")
            else:
                nl = data.find(b"\n", off)
                line = bytes(data[off:len(data) if nl < 0 else nl])
                if mode == FILE and line.endswith(b"\r"):
                    line = line[:-1]
                f = line.split(b"\t", 2)
                if len(f) == 3:
                    msgs.append(b"Unphased genotype found at CHROM=" + f[0] + b", POS=" + f[1] + b"; line skipped.\n")

    body, tot = _run(OP_PHASE_CHECK, data, mode, chunk_bytes, on_events=None if quiet else on_events, **kw)
    return ToolResult(body, 0, tot, b"".join(msgs))


def variant_counter(data: bytes, mode: int = FILE, strict: bool = False, chunk_bytes: int = 0, **kw) -> ToolResult:
    _, tot = _run(OP_VARIANT_COUNT, data, mode, chunk_bytes, **kw)
    if strict and tot.short_lines:                # variant_counter.cpp:373-377, 175-177
        return ToolResult(b"", 1, tot)
    return ToolResult(b"Total Variants: %d\n" % tot.rows, 0, tot)


# ----------------------------------------------------------------------------- allele_counter
AC_MT_TEXT, AC_STREAM, AC_UNIFIED = 0, 1, 2          # code paths of the reference (allele_counter.cpp:1522-1533)
AC_TEXT, AC_AGGREGATE, AC_BINARY = 0, 1, 2


def _ac_header_names(data: bytes):
    """Sample names of the leading '#' block (fields 10.. of every "#CHROM" line, accumulated) and
    the offset of the first non-'#' line (allele_counter.cpp:806-829, 1285-1307)."""
    names, pos, n = [], 0, len(data)
    while pos < n and data[pos:pos + 1] == b"#":
        nl = data.find(b"\n", pos)
        end = n if nl < 0 else nl
        line = data[pos:end]
        if line.startswith(b"#CHROM"):
            f = line.split(b"\t")
            if len(f) > 9:
                cols = f[9:]
                if cols and cols[-1] == b"":      # nothing is pushed for an empty tail after a final tab
                    cols = cols[:-1]
                names += cols
        pos = n if nl < 0 else nl + 1
    return names, pos


def _ac_parse_samples(arg: str | None):
    """The -s argument: split on ' ', drop empties, trim (allele_counter.cpp:355-373)."""
    if not arg:
        return []
    out = []
    for tok in arg.encode().split(b" "):
        if tok:
            t = tok.strip(b" \t\n\r")
            out.append(t if t else tok)
    return out


def allele_counter(data: bytes, path: int = AC_MT_TEXT, fmt: int = AC_TEXT, limit: int = 0,
                   samples: str | None = None, chunk_bytes: int = 0, **kw) -> ToolResult:
    """Host side of VCFX_allele_counter (header parse, sample selection, fixed header rows); the
    per-line work (processChunk / countAllelesStream / countAllelesUnified) runs in libvcfx_cuda."""
    req = _ac_parse_samples(samples)
    if path != AC_STREAM:
        if len(data) == 0:
            return ToolResult(b"", 1, Totals())                       # "Error: Empty file"
        names, data_pos = _ac_header_names(data)
        if not names:
            return ToolResult(b"", 1, Totals())                       # "Error: No samples found in VCF"
        if path == AC_MT_TEXT and data_pos >= len(data):
            return ToolResult(b"", 1, Totals())                       # "Error: No data lines found"
    else:
        # the stream path meets lines one by one: every "#CHROM" line APPENDS its names and then appends
        # a full selection over all names so far (allele_counter.cpp:1139-1178); blank lines are skipped;
        # a data line before any "#CHROM" line is an error with nothing written; no header at all ends
        # with the header row and rc 1
        names, cols, pos, n, saw_chrom = [], [], 0, len(data), False
        while pos < n and data[pos:pos + 1] in (b"#", b"\n"):
            nl = data.find(b"\n", pos)
            line = data[pos:(n if nl < 0 else nl)]
            if line.startswith(b"#CHROM"):
                saw_chrom = True
                f = line.split(b"\t")
                add = f[9:] if len(f) > 9 else []
                if add and add[-1] == b"":
                    add = add[:-1]
                names += add
                if req:
                    last = {nm: i for i, nm in enumerate(names)}
                    if any(r not in last for r in req):
                        return ToolResult(b"", 1, Totals())
                    cols += [last[r] for r in req]
                else:
                    cols += list(range(len(names)))
            pos = n if nl < 0 else nl + 1
        if not saw_chrom:
            has_data = any(l and not l.startswith(b"#") for l in data[pos:].split(b"\n"))
            return ToolResult(b"" if has_data else AC_TEXT_HEADER, 1, Totals())
    if path != AC_STREAM:
        if req:
            last = {nm: i for i, nm in enumerate(names)}                  # duplicates: the last column wins (:845-847)
            if any(r not in last for r in req):
                return ToolResult(b"", 1, Totals())                       # "Error: Sample 'x' not found"
            cols = [last[r] for r in req]
        else:
            cols = list(range(len(names)))
        if path == AC_UNIFIED and limit > 0 and len(cols) > limit:
            cols = cols[:limit]
    if not cols:
        # a "#CHROM" line without sample columns: nothing can be selected, every data line yields no row
        return ToolResult(AC_TEXT_HEADER, 0, Totals())
    sel_names = [names[c] for c in cols]
    flags = 0
    if path == AC_STREAM or (path == AC_UNIFIED and fmt == AC_TEXT):
        flags = F_AC_FORWARD
    elif path == AC_UNIFIED and fmt == AC_AGGREGATE:
        flags = F_AC_AGGREGATE
    elif path == AC_UNIFIED and fmt == AC_BINARY:
        flags = F_AC_BINARY
    body, tot = _run(OP_ALLELE_COUNT, data, FILE if path != AC_STREAM else STDIN, chunk_bytes, flags=flags,
                     sel_cols=cols, sel_names=sel_names, **kw)
    if flags == F_AC_AGGREGATE:
        head = AC_AGG_HEADER
    elif flags == F_AC_BINARY:
        import struct
        head = b"VCAC" + struct.pack("<IIQ", 1, len(cols), 0)        # BinaryHeader, packed (:326-333)
    else:
        head = AC_TEXT_HEADER
    return ToolResult(head + body, 0, tot)
