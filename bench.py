#!/usr/bin/env python
"""bench.py — throughput of the VCFX hot path on B200 (BASELINE.json metric).

Headline (the contractual JSON line): one "step" = the job of BASELINE config 2, VCFX_allele_freq_calc +
VCFX_variant_counter over one synthetic 1000G-chr21-shape VCF (427,409 variants x 2,504 samples, phased
GT-only, ~4.3 GB) — each tool makes its own full pass, exactly like the two reference processes.

  value     input GB/s of that job with the file already resident in HBM (kernel-only)
  e2e       the same job through the C ABI from HOST memory (vcfx_cuda_submit_host / next_output): every
            step re-uploads the file in pinned 64 MiB chunks and reads the text back; beside it the bare
            pinned host->device copy rate of this box at the same rank count (`h2d_ceiling`)
  roofline  the allele_freq_calc kernels of that job against the measured HBM peak
  parity    byte comparison of what the timed kernels wrote: the full-size resident output against the CPU
            restatement (oracle/, all host cores) and its first rows against the unmodified reference tool
  configs   the other tools and BASELINE shapes, one entry each: kernel time, fraction of the HBM peak,
            end to end from host memory, parity against the reference tool on a prefix sample
  cli       wall clock of the drop-in executables on the 4.3 GB file (page cache), reference tools beside them
  --impl reference : the unmodified reference tools (oracle/_ref/VCFX_*, built by oracle/Makefile from the
            reference sources) on this box's host cores, each step on a bounded sample of the same workload
  --dump-outputs DIR : what the timed job computed in its last step, as DIR/<name>.npy (float32 / float64)

N > 1 (torchrun, one rank per GPU): every rank owns its own newline-aligned shard of the same synthetic
stream (weak scaling, no data-path collective); the scalar totals cross ranks in one tiny NCCL all-reduce
per step.  Each rank binds itself to the cores of its GPU's NUMA node before it allocates pinned memory.
"""
from __future__ import annotations

import argparse
import concurrent.futures as cf
import hashlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

C2_VARIANTS = 427_409
SAMPLES = 2_504
CHUNK = 64 << 20
CPU_SAMPLE_VARIANTS = 60_000          # ~0.6 GB: ~3-4 s of allele_freq_calc on one core
C4_VARIANTS = 60_000                  # BASELINE config 4 names 1 M variants (~66 GB); scaled to ~4 GB, V stated


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ----------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons through NVML while the timed region runs."""

    def __init__(self, indices):
        """indices: physical GPU indices to watch (rank 0 watches every GPU of the job: one NVML poller
        per node instead of one per rank, so the polling itself does not perturb the launches)."""
        super().__init__(daemon=True)
        self.indices = list(indices)
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.hs = [pynvml.nvmlDeviceGetHandleByIndex(i) for i in self.indices]
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.hs[0], pynvml.NVML_CLOCK_SM) if self.hs else None
            self.ok = bool(self.hs)
        except Exception as e:  # pragma: no cover
            log(f"[bench] NVML unavailable: {e}")

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._halt.is_set():
            for h in self.hs:
                try:
                    self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                    try:
                        r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                    except Exception:
                        r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    for bit, name in names.items():
                        if r & bit:
                            self.reasons.add(name)
                except Exception:
                    pass
            time.sleep(0.003)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None,
                "sm_mhz_min": min(self.samples) if self.samples else None, "gpus_watched": len(getattr(self, "hs", [])),
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ----------------------------------------------------------------------------------------
def physical_gpu_index(local_rank: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


def bind_to_gpu_numa_node(local_rank: int):
    """Run this rank on the cores next to its GPU, BEFORE pinned memory is allocated: Linux places pages
    on the node of the thread that first touches them, and cudaMallocHost touches them here.  Returns what
    was done (for the JSON line)."""
    info = {"bound": False}
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(physical_gpu_index(local_rank))
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:           # NVML prints an 8-digit domain, sysfs a 4-digit one
            bus = bus[4:]
        base = Path("/sys/bus/pci/devices") / bus
        node = int((base / "numa_node").read_text().strip())
        cpus = (base / "local_cpulist").read_text().strip()
        info.update({"pci": bus, "numa_node": node, "local_cpulist": cpus})
        ids = set()
        for part in cpus.split(","):
            if "-" in part:
                a, b = part.split("-"); ids.update(range(int(a), int(b) + 1))
            elif part:
                ids.add(int(part))
        allowed = os.sched_getaffinity(0)
        ids &= allowed
        if ids and ids != allowed:
            os.sched_setaffinity(0, ids)
            info["bound"] = True
        info["cpus_used"] = len(os.sched_getaffinity(0))
    except Exception as e:
        info["error"] = str(e)[:120]
    return info


def sha256_file(path) -> str:
    h = hashlib.sha256()
    with open(path, "rb") as f:
        while True:
            b = f.read(1 << 24)
            if not b:
                break
            h.update(b)
    return h.hexdigest()


def shm_dir() -> str:
    return "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()


def ref_tool(name: str):
    p = ROOT / "oracle" / "_ref" / f"VCFX_{name}"
    return p if p.exists() else None


def run_to_file(cmd, out_path, stdin_path=None, timeout=900):
    """Wall clock of one process with stdout into a file (the reference's benchmark method:
    benchmarks/scripts/run_comprehensive_benchmark.sh:122-146, with the output kept for the comparison)."""
    t0 = time.perf_counter()
    with open(out_path, "wb") as fo:
        fi = open(stdin_path, "rb") if stdin_path else None
        try:
            r = subprocess.run([str(c) for c in cmd], stdout=fo, stderr=subprocess.DEVNULL, stdin=fi, timeout=timeout)
        finally:
            if fi:
                fi.close()
    return time.perf_counter() - t0, r.returncode


# ----------------------------------------------------------------------------------------
def cpu_reference_run(sample_variants: int, steps: int, warmup: int, keep_outputs: dict | None = None):
    """Time the reference's own CPU tools (allele_freq_calc -q -i + variant_counter, the headline job) on a
    bounded sample of the workload (rank 0 only); with keep_outputs the stdout of the last run is hashed."""
    from vcfx_b200 import synth
    af, vc = ref_tool("allele_freq_calc"), ref_tool("variant_counter")
    if not (af and vc):
        return None
    data = synth.make_vcf(2, sample_variants, SAMPLES, seed=2)
    fd, path = tempfile.mkstemp(suffix=".vcf", dir=shm_dir())
    out_af, out_vc = path + ".af", path + ".vc"
    times = []
    try:
        with os.fdopen(fd, "wb") as f:
            f.write(data)
        with open(path, "rb") as f:        # warm the page cache
            while f.read(1 << 24):
                pass
        for i in range(warmup + steps):
            t_af, rc1 = run_to_file([af, "-q", "-i", path], out_af)
            t_vc, rc2 = run_to_file([vc, path], out_vc)
            if rc1 or rc2:
                return None
            if i >= warmup:
                times.append(t_af + t_vc)
        if keep_outputs is not None:
            keep_outputs["allele_freq_calc"] = open(out_af, "rb").read()
            keep_outputs["variant_counter"] = open(out_vc, "rb").read()
            keep_outputs["input"] = data
    finally:
        for p in (path, out_af, out_vc):
            if os.path.exists(p):
                os.unlink(p)
    nbytes = len(data)
    return {"bytes": nbytes, "variants": sample_variants, "times": times,
            "gbps": nbytes / (sum(times) / len(times)) / 1e9}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    warm = max(0, min(args.warmup, 1))        # one warm-up run is enough for a process that streams a cached file
    r = cpu_reference_run(CPU_SAMPLE_VARIANTS, args.steps, warm)
    if r is None:
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/VCFX_* not built (make -C oracle ref REFERENCE=<VCFX source tree>)"}))
        return 0
    ms = 1e3 * sum(r["times"]) / len(r["times"])
    sample = (f"{r['variants']} variants x {SAMPLES} samples ({r['bytes'] / 1e9:.2f} GB): a prefix of the C2 stream, file in page cache; "
              f"allele_freq_calc -q -i + variant_counter are single-threaded (1 of {os.cpu_count()} cores busy)")
    cfg = workload_config()
    cfg["reference_sample"] = sample
    cfg["reference_warmup_runs"] = warm
    line = {
        "impl": "reference", "metric": "vcf_input_GB_per_s", "value": r["gbps"], "unit": "GB/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": warm, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": cfg,
        "genotypes_per_s": r["variants"] * SAMPLES / (ms / 1e3),
        "cpu_baseline": {"value": r["gbps"], "unit": "GB/s", "cores": 1, "kind": "reference", "sample": sample},
        "e2e": {"value": r["gbps"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


DUMP_SAMPLE_ROWS = 4096


def dump_outputs(np, out_dir: Path, suffix: str, af_text: bytes, af_rows: int, vc_rows: int):
    """What one step of the timed job hands its caller, as float arrays (DIR/<name><suffix>.npy), so that two builds
    can be compared output for output: POS and allele frequency of every allele_freq_calc row, the text of a fixed,
    seeded sample of its rows as byte values, and the row counts of both tools."""
    rows = af_text.splitlines(keepends=True)
    assert len(rows) == af_rows, (len(rows), af_rows)
    cols = [r.split(b"\t") for r in rows]
    pick = np.sort(np.random.default_rng(0).choice(len(rows), min(DUMP_SAMPLE_ROWS, len(rows)), replace=False))
    arrays = {
        "allele_freq_calc_pos": np.array([float(c[1]) for c in cols], dtype=np.float64),
        "allele_freq_calc_af": np.array([float(c[-1]) for c in cols], dtype=np.float64),
        "allele_freq_calc_text_sample": np.frombuffer(b"".join(rows[i] for i in pick), dtype=np.uint8).astype(np.float32),
        "row_counts": np.array([af_rows, vc_rows], dtype=np.float64),
    }
    out_dir.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(out_dir / f"{name}{suffix}.npy", a)
    log(f"[bench] wrote {', '.join(f'{n}{suffix}.npy' for n in arrays)} to {out_dir} ({sum(a.nbytes for a in arrays.values()) / 1e6:.1f} MB)")


def workload_config():
    return {"workload": "C2: VCFX_allele_freq_calc + VCFX_variant_counter (FILE semantics) on a synthetic "
                        "1000G chr21-shape VCF, 427409 variants x 2504 samples, phased GT-only, ~4.3 GB per GPU",
            "variants_per_gpu": C2_VARIANTS, "samples": SAMPLES, "chunk_bytes": CHUNK,
            "l2": "inputs (4.3 GB) are larger than L2 (126 MB); no explicit flush",
            "sharding": "one newline-aligned shard of the stream per GPU; the scalar totals of the timed jobs are merged by one NCCL all-reduce inside the timed region"}


# ----------------------------------------------------------------------------------------
class Shard:
    """A synthetic stream generated straight into pinned host memory and copied to the device."""

    def __init__(self, torch, np, synth, api, dev, shape, first, count, with_header, threads):
        t0 = time.perf_counter()
        self.shape, self.V = shape, count
        self.hdr = synth.header(shape, SAMPLES, shape) if with_header else b""
        cap = len(self.hdr) + synth.line_bound(shape, SAMPLES) * count
        self.host = torch.empty(cap, dtype=torch.uint8, pin_memory=True)
        self.hnp = self.host.numpy()
        self.hnp[: len(self.hdr)] = np.frombuffer(self.hdr, dtype=np.uint8)
        nbody = synth.lines_into(self.hnp[len(self.hdr):], shape, SAMPLES, first, count, seed=shape, threads=threads)
        self.nbytes = len(self.hdr) + nbody
        self.line_len = int(np.argmax(self.hnp[len(self.hdr):len(self.hdr) + (4 << 20)] == 10)) + 1
        self.d_in = torch.empty(self.nbytes + api.DEVICE_PAD, dtype=torch.uint8, device=dev)
        self.d_in[:self.nbytes].copy_(self.host[:self.nbytes], non_blocking=False)
        torch.cuda.synchronize()
        self.bounds = []
        pos = 0
        while pos < self.nbytes:
            end = min(self.nbytes, pos + CHUNK)
            if end < self.nbytes:
                end = pos + int(np.flatnonzero(self.hnp[pos:end] == 10)[-1]) + 1
            self.bounds.append((pos, end)); pos = end
        self.gen_s = time.perf_counter() - t0

    def prefix_bytes(self, np, n_variants: int) -> bytes:
        """The header and the first n_variants lines."""
        body = self.hnp[len(self.hdr):self.nbytes]
        # the k-th newline of the body
        step = 64 << 20
        seen = 0; pos = 0
        while pos < len(body):
            nl = np.flatnonzero(body[pos:pos + step] == 10)
            if seen + len(nl) >= n_variants:
                end = pos + int(nl[n_variants - seen - 1]) + 1
                return self.hdr + body[:end].tobytes()
            seen += len(nl); pos += step
        return self.hdr + body.tobytes()


def oracle_parallel(O, fn_name, shard, np, pieces=48, **kw):
    """The CPU restatement (oracle/, the checker) over a whole shard: newline-aligned pieces, every piece with
    the header in front, one thread per piece (ctypes releases the GIL); returns sha256 and length of the
    concatenated data rows."""
    fn = getattr(O, fn_name)
    body0 = len(shard.hdr)
    n = shard.nbytes
    cuts = [body0]
    for i in range(1, pieces):
        target = body0 + (n - body0) * i // pieces
        nl = np.flatnonzero(shard.hnp[target:min(n, target + (1 << 20))] == 10)
        cuts.append(target + int(nl[0]) + 1 if len(nl) else n)
    cuts.append(n)
    cuts = sorted(set(cuts))

    def one(i):
        data = shard.hdr + shard.hnp[cuts[i]:cuts[i + 1]].tobytes()
        r = fn(data, 0, **kw) if fn_name != "allele_counter" else fn(data, **kw)
        out = r.out
        return out[out.index(b"\n") + 1:] if out else out            # drop the fixed header row of the piece

    h = hashlib.sha256(); total = 0
    with cf.ThreadPoolExecutor(max_workers=min(pieces, os.cpu_count() or 8)) as ex:
        for out in ex.map(one, range(len(cuts) - 1)):
            h.update(out); total += len(out)
    return h.hexdigest(), total


def measure_h2d_ceiling(torch, shard, dev, dist, world, seconds=1.0):
    """Bare pinned host->device copies of the shard's own 64 MiB chunks on three streams (what the streaming
    path does, without any kernel), all ranks at once: the ceiling of `e2e` on this box."""
    K = 6                                          # copies in flight (the streaming path keeps three slots per context busy)
    streams = [torch.cuda.Stream(device=dev) for _ in range(K)]
    bufs = [torch.empty(CHUNK, dtype=torch.uint8, device=dev) for _ in range(K)]

    def one_pass():
        for i, (s, e) in enumerate(shard.bounds):
            with torch.cuda.stream(streams[i % K]):
                bufs[i % K][: e - s].copy_(shard.host[s:e], non_blocking=True)
    one_pass(); torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter(); n = 0
    while True:
        one_pass(); n += 1
        torch.cuda.synchronize()
        if time.perf_counter() - t0 > seconds:
            break
    dt = time.perf_counter() - t0
    t = torch.tensor([dt / n], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return world * shard.nbytes / float(t.item()) / 1e9


def measure_bidir_ceiling(torch, shard, dev, seconds=1.0):
    """The same bare host->device copies with an equally large device->host copy under way for every chunk (pinned
    buffers, streams of their own): what the link gives the INPUT while an output as large as the input goes back —
    the ceiling of `e2e` for missing_detector / nonref_filter / phase_checker / genotype_query style tools."""
    K = 3
    up = [torch.cuda.Stream(device=dev) for _ in range(K)]
    down = [torch.cuda.Stream(device=dev) for _ in range(K)]
    bufs = [torch.empty(CHUNK, dtype=torch.uint8, device=dev) for _ in range(K)]
    back_d = [torch.empty(CHUNK, dtype=torch.uint8, device=dev) for _ in range(K)]
    back_h = [torch.empty(CHUNK, dtype=torch.uint8, pin_memory=True) for _ in range(K)]

    def one_pass():
        for i, (s, e) in enumerate(shard.bounds):
            with torch.cuda.stream(up[i % K]):
                bufs[i % K][: e - s].copy_(shard.host[s:e], non_blocking=True)
            with torch.cuda.stream(down[i % K]):
                back_h[i % K][: e - s].copy_(back_d[i % K][: e - s], non_blocking=True)
    one_pass(); torch.cuda.synchronize()
    t0 = time.perf_counter(); n = 0
    while True:
        one_pass(); n += 1
        torch.cuda.synchronize()
        if time.perf_counter() - t0 > seconds:
            break
    return shard.nbytes / ((time.perf_counter() - t0) / n) / 1e9


# ----------------------------------------------------------------------------------------
def e2e_stream(api, ctx, shard, valid_abs, steps):
    """One tool through the streaming C ABI from the shard's pinned host memory: H2D, kernels and D2H per chunk."""
    base_ptr = shard.host.data_ptr()

    def step():
        rows = nout = 0
        for (s, e) in shard.bounds:
            vf = min(max(valid_abs - s, 0), e - s)
            while not ctx.submit_host(base_ptr + s, e - s, valid_from=vf, is_final=(e == shard.nbytes), file_offset=s):
                _, n, st = ctx.next_output_raw(); rows += st.rows; nout += n      # the text is in the library's pinned buffer: on the host
        while ctx.in_flight():
            _, n, st = ctx.next_output_raw(); rows += st.rows; nout += n
        return rows, nout
    step()
    t0 = time.perf_counter()
    for _ in range(steps):
        rows, nout = step()
    dt = (time.perf_counter() - t0) / steps
    return {"value": shard.nbytes / dt / 1e9, "unit": "GB/s", "ms_per_step": dt * 1e3, "steps": steps,
            "h2d_bytes_per_step": shard.nbytes, "d2h_bytes_per_step": int(nout)}, rows


def config_entries(torch, np, api, synth, O, dev, peak, threads, only=None):
    """The other tools and shapes (N = 1): kernel time resident in HBM, fraction of the HBM peak on algorithmic
    bytes (input + stdout, each once), end to end from host memory, parity against the reference tool."""
    names = [b"HG%05d" % (96 + i) for i in range(SAMPLES)]
    sel = dict(sel_cols=list(range(SAMPLES)), sel_names=names)
    plans = [
        ("C2", 2, C2_VARIANTS, [("hwe_tester", api.OP_HWE, 0, {}, 20000), ("nonref_filter", api.OP_NONREF_FILTER, 0, {}, 20000),
                                ("indexer", api.OP_INDEX, 0, {}, 60000), ("phase_checker", api.OP_PHASE_CHECK, 0, {}, 20000),
                                ("inbreeding_calculator", api.OP_INBREEDING, 0, sel, 20000),
                                ("genotype_query -g 1/1", api.OP_GENOTYPE_QUERY, 0, dict(query=b"1/1"), 20000),
                                ("dosage_calculator", api.OP_DOSAGE, 0, {}, 20000)]),
        ("C3", 3, C2_VARIANTS, [("missing_detector", api.OP_MISSING_DETECT, 0, {}, 20000),
                                ("allele_counter", api.OP_ALLELE_COUNT, 0, sel, 4000),
                                ("allele_counter -a", api.OP_ALLELE_COUNT, api.F_AC_AGGREGATE, sel, 400),
                                ("allele_freq_calc", api.OP_ALLELE_FREQ, 0, {}, 20000),
                                ("inbreeding_calculator", api.OP_INBREEDING, 0, sel, 20000)]),
        ("C4", 4, C4_VARIANTS, [("hwe_tester", api.OP_HWE, 0, {}, 3000),
                                ("allele_freq_calc", api.OP_ALLELE_FREQ, 0, {}, 3000)]),
    ]
    entries = []
    for cname, shape, V, tools in plans:
        if only and cname not in only:
            continue
        sh = Shard(torch, np, synth, api, dev, shape, 0, V, True, threads)
        bidir = measure_bidir_ceiling(torch, sh, dev)
        log(f"[bench] {cname}: {sh.nbytes / 1e9:.2f} GB, {V} variants generated in {sh.gen_s:.1f}s; input rate with an equal output going back: {bidir:.1f} GB/s")
        for tname, op, flags, kw, ref_variants in tools:
            out_cap = 64 << 20
            if op in (api.OP_MISSING_DETECT, api.OP_NONREF_FILTER, api.OP_PHASE_CHECK, api.OP_GENOTYPE_QUERY, api.OP_DOSAGE):
                out_cap = sh.nbytes + sh.nbytes // 50 + (1 << 20)
            if op == api.OP_ALLELE_COUNT and flags == 0:
                out_cap = int(sh.nbytes * 9.5) + (1 << 20)
            d_out = torch.empty(out_cap, dtype=torch.uint8, device=dev)
            ctx = api.Context(op, api.FILE, flags=flags, **kw)
            ctx.set_line_hint(sh.line_len)
            vf = api.find_chrom_header(sh.hdr) if op in (api.OP_ALLELE_FREQ, api.OP_NONREF_FILTER, api.OP_INDEX, api.OP_PHASE_CHECK) else (api.first_data_offset(sh.hdr) if op == api.OP_MISSING_DETECT else 0)
            fc = api.first_format_line(sh.prefix_bytes(np, 4), vf) if op == api.OP_PHASE_CHECK else 0     # (every line of these shapes has a FORMAT)
            ms = []
            for i in range(5):
                ctx.run_device(sh.d_in.data_ptr(), sh.nbytes, d_out.data_ptr(), out_cap, valid_from=vf, format_cache_from=fc)
                st = ctx.sync()
                if i >= 2:
                    ms.append(st.kernel_ms)
            k = statistics.median(ms)
            alg = sh.nbytes + int(st.bytes_out)
            ent = {"config": cname, "tool": tname, "variants": V, "samples": SAMPLES, "input_bytes": sh.nbytes, "output_bytes": int(st.bytes_out),
                   "kernel_ms": k, "algorithmic_bytes": alg, "achieved_GBps": alg / k / 1e6, "frac": alg / k / 1e6 / peak,
                   "input_GBps": sh.nbytes / k / 1e6, "genotypes_per_s": V * SAMPLES / (k / 1e3), "rows": int(st.rows)}
            ctx.close()
            # full-size byte parity of the resident output against the CPU restatement (small outputs only)
            if tname in ("hwe_tester", "allele_freq_calc", "allele_counter -a", "dosage_calculator"):
                got = hashlib.sha256(d_out[:int(st.bytes_out)].cpu().numpy().tobytes()).hexdigest()
                if tname == "allele_counter -a":
                    exp, n_exp = oracle_parallel(O, "allele_counter", sh, np, path=O.AC_UNIFIED, fmt=O.AC_AGGREGATE)
                else:
                    exp, n_exp = oracle_parallel(O, {"hwe_tester": "hwe", "allele_freq_calc": "allele_freq", "dosage_calculator": "dosage"}[tname], sh, np)
                ent["parity_full"] = {"against": "oracle port, all host cores, the whole input", "bytes": int(st.bytes_out),
                                      "equal": got == exp and n_exp == int(st.bytes_out), "sha256": got}
            if tname == "inbreeding_calculator":
                # the sums depend on the order of the sites: the restatement walks the whole input on one core
                got_b = d_out[:int(st.bytes_out)].cpu().numpy().tobytes()
                t0 = time.perf_counter()
                exp_b = O.inbreeding(sh.hnp[:sh.nbytes].tobytes(), 0, O.IB_QUIET).out[len(api.IB_HEADER):]
                ent["parity_full"] = {"against": "oracle port, one core, the whole input in file order", "bytes": len(got_b), "equal": got_b == exp_b,
                                      "sha256": hashlib.sha256(got_b).hexdigest(), "oracle_seconds": time.perf_counter() - t0}
            del d_out
            torch.cuda.empty_cache()
            # end to end from pinned host memory
            if op == api.OP_ALLELE_COUNT and flags == 0:
                sctx = api.Context(op, api.FILE, flags=flags, chunk_bytes=16 << 20, n_slots=3, **kw)
                e2e_chunk = 16 << 20
            else:
                sctx = api.Context(op, api.FILE, flags=flags, chunk_bytes=CHUNK, n_slots=3, **kw)
                e2e_chunk = CHUNK
            if e2e_chunk != CHUNK:                                   # re-cut the shard for the smaller slots
                keep = sh.bounds
                sh.bounds = []
                pos = 0
                while pos < sh.nbytes:
                    end = min(sh.nbytes, pos + e2e_chunk)
                    if end < sh.nbytes:
                        end = pos + int(np.flatnonzero(sh.hnp[pos:end] == 10)[-1]) + 1
                    sh.bounds.append((pos, end)); pos = end
            ent["e2e"], rows = e2e_stream(api, sctx, sh, vf, 2)
            ent["e2e"]["chunk_bytes"] = e2e_chunk
            if sh.nbytes // 2 <= ent["e2e"]["d2h_bytes_per_step"] <= 2 * sh.nbytes:      # an output about as large as the input: both directions of the link are busy
                ent["e2e"]["bidir_ceiling_GBps"] = bidir
                ent["e2e"]["frac_of_bidir_ceiling"] = ent["e2e"]["value"] / bidir
            elif ent["e2e"]["d2h_bytes_per_step"] > 2 * sh.nbytes:                        # the text going back is the bound: its own rate
                ent["e2e"]["d2h_GBps"] = ent["e2e"]["d2h_bytes_per_step"] / (ent["e2e"]["ms_per_step"] * 1e6)
            if e2e_chunk != CHUNK:
                sh.bounds = keep
            sctx.close()
            # parity against the unmodified reference tool on a prefix of the same stream
            ent["parity"] = parity_vs_reference(api, O, np, sh, tname, ref_variants)
            entries.append(ent)
            log(f"[bench] {cname} {tname}: {k:.3f} ms, {100 * ent['frac']:.1f}% of HBM peak, e2e {ent['e2e']['value']:.1f} GB/s, parity {ent['parity'].get('equal')}")
        del sh
        torch.cuda.empty_cache()
    return entries


def parity_vs_reference(api, O, np, shard, tname, n_variants):
    """GPU tool output (through the C ABI, FILE semantics) against the stdout of the unmodified reference tool
    on the first n_variants lines of the shard."""
    tool = {"hwe_tester": "hwe_tester", "allele_freq_calc": "allele_freq_calc", "missing_detector": "missing_detector",
            "allele_counter": "allele_counter", "allele_counter -a": "allele_counter", "variant_counter": "variant_counter", "nonref_filter": "nonref_filter", "indexer": "indexer", "phase_checker": "phase_checker", "inbreeding_calculator": "inbreeding_calculator", "genotype_query -g 1/1": "genotype_query", "dosage_calculator": "dosage_calculator"}[tname]
    exe = ref_tool(tool)
    data = shard.prefix_bytes(np, n_variants)
    if tname == "hwe_tester":
        got = api.hwe_tester(data, api.FILE).out; args = ["-q", "-i"]
    elif tname == "allele_freq_calc":
        got = api.allele_freq_calc(data, api.FILE).out; args = ["-q", "-i"]
    elif tname == "missing_detector":
        got = api.missing_detector(data, api.FILE).out; args = ["-q", "-t", "1", "-i"]   # default threads abort on dotted files >= 10 MB (SURVEY finding 2)
    elif tname == "nonref_filter":
        got = api.nonref_filter(data, api.FILE).out; args = ["-i"]
    elif tname == "indexer":
        got = api.indexer(data, api.FILE).out; args = []
    elif tname == "phase_checker":
        got = api.phase_checker(data, api.FILE, quiet=True).out; args = ["-q", "-i"]
    elif tname == "inbreeding_calculator":
        got = api.inbreeding_calculator(data, api.FILE).out; args = ["-q", "-i"]
    elif tname == "genotype_query -g 1/1":
        got = api.genotype_query(data, "1/1", api.FILE, quiet=True).out; args = ["-q", "-g", "1/1", "-i"]
    elif tname == "dosage_calculator":
        got = api.dosage_calculator(data, api.FILE, quiet=True).out; args = ["-q", "-i"]
    elif tname == "allele_counter":
        got = api.allele_counter(data, api.AC_MT_TEXT, api.AC_TEXT).out; args = ["-q", "-i"]
    elif tname == "allele_counter -a":
        got = api.allele_counter(data, api.AC_UNIFIED, api.AC_AGGREGATE).out; args = ["-q", "-a", "-i"]
    else:
        got = api.variant_counter(data, api.FILE).out; args = []
    res = {"tool": tname, "variants": n_variants, "input_bytes": len(data), "bytes": len(got), "sha256": hashlib.sha256(got).hexdigest()}
    if exe is None:
        # no reference binary on this box: the CPU restatement (pinned to the reference by tests/) stands in
        fn = {"hwe_tester": lambda: O.hwe(data, 0), "allele_freq_calc": lambda: O.allele_freq(data, 0), "missing_detector": lambda: O.missing(data, 0),
              "nonref_filter": lambda: O.nonref_filter(data, 0), "indexer": lambda: O.indexer(data, 0), "phase_checker": lambda: O.phase_checker(data, 0), "inbreeding_calculator": lambda: O.inbreeding(data, 0, O.IB_QUIET), "genotype_query -g 1/1": lambda: O.genotype_query(data, "1/1", 0)[0], "dosage_calculator": lambda: O.dosage(data, 0), "allele_counter": lambda: O.allele_counter(data), "allele_counter -a": lambda: O.allele_counter(data, O.AC_UNIFIED, O.AC_AGGREGATE),
              "variant_counter": lambda: O.variant_count(data, 0)}[tname]
        exp = fn().out
        res.update({"against": "oracle port (reference binary not built on this box)", "equal": exp == got})
        return res
    fd, path = tempfile.mkstemp(suffix=".vcf", dir=shm_dir())
    outp = path + ".out"
    try:
        with os.fdopen(fd, "wb") as f:
            f.write(data)
        secs, rc = run_to_file([exe, *args, path], outp)
        exp_sha = sha256_file(outp)
        res.update({"against": f"oracle/_ref/VCFX_{tool} {' '.join(args)} (unmodified reference tool)", "reference_seconds": secs, "reference_rc": rc,
                    "reference_GBps": len(data) / secs / 1e9, "equal": rc == 0 and exp_sha == res["sha256"] and os.path.getsize(outp) == len(got)})
    finally:
        for p in (path, outp):
            if os.path.exists(p):
                os.unlink(p)
    return res


def cli_leg(np, shard):
    """The drop-in boundary itself: wall clock of the executables on the full file (page cache), the reference's own
    method (benchmarks/scripts/run_comprehensive_benchmark.sh:122-146), with the reference tools on the same file."""
    bin_dir = ROOT / "vcfx_b200" / "bin"
    if not (bin_dir / "VCFX_allele_freq_calc").exists():
        return {"unavailable": "vcfx_b200/bin not built"}
    path = os.path.join(shm_dir(), f"vcfx_bench_{os.getpid()}.vcf")
    res = {"file_bytes": shard.nbytes, "where": shm_dir()}
    try:
        with open(path, "wb") as f:
            step = 256 << 20
            for pos in range(0, shard.nbytes, step):
                f.write(shard.hnp[pos:min(shard.nbytes, pos + step)].tobytes())
        outs = {}
        for tool, args in (("allele_freq_calc", ["-q", "-i", path]), ("variant_counter", [path])):
            best = None
            for rep in range(2):
                secs, rc = run_to_file([bin_dir / f"VCFX_{tool}", *args], path + f".{tool}.gpu")
                best = secs if best is None else min(best, secs)
            outs[tool] = {"gpu_seconds": best, "gpu_rc": rc, "gpu_GBps": shard.nbytes / best / 1e9, "sha256": sha256_file(path + f".{tool}.gpu")}
            exe = ref_tool(tool)
            if exe:
                secs, rc = run_to_file([exe, *args], path + f".{tool}.ref", timeout=600)
                outs[tool].update({"reference_seconds": secs, "reference_rc": rc, "reference_GBps": shard.nbytes / secs / 1e9,
                                   "equal": sha256_file(path + f".{tool}.ref") == outs[tool]["sha256"], "ratio": secs / best})
        res["tools"] = outs
        g = sum(v["gpu_seconds"] for v in outs.values())
        res["job_gpu_seconds"] = g
        res["job_GBps"] = shard.nbytes / g / 1e9
        if all("reference_seconds" in v for v in outs.values()):
            r = sum(v["reference_seconds"] for v in outs.values())
            res["job_reference_seconds"] = r
            res["job_ratio"] = r / g
        res["note"] = "one process per tool, CUDA context creation included; best of 2 runs for the GPU tools, one run for the reference"
    except Exception as e:
        res["error"] = str(e)[:200]
    finally:
        for suffix in ("", ".allele_freq_calc.gpu", ".variant_counter.gpu", ".allele_freq_calc.ref", ".variant_counter.ref"):
            if os.path.exists(path + suffix):
                os.unlink(path + suffix)
    return res


def hwe_pvalue_report(api, O, np):
    sys.path.insert(0, str(ROOT / "tests"))
    from hwe_triples import triples
    c = triples()
    dev = api.hwe_pvalues(c)
    ref = O.hwe_pvalues(c)
    nz = ref != 0
    rel = np.abs(dev[nz] - ref[nz]) / np.abs(ref[nz])
    fd, sd = O.p_text_diffs(dev, ref)
    return {"triples": int(len(c)), "max_relative_difference": float(rel.max()), "values_not_bit_identical": int((dev != ref).sum()),
            "file_mode_texts_that_differ": int(fd), "stdin_mode_texts_that_differ": int(sd), "tolerance": 1e-12,
            "within_tolerance": bool(rel.max() <= 1e-12 and np.array_equal(dev == 0, ref == 0)),
            "note": "device exp() vs glibc exp(); every other operation is bit-identical by construction"}


# ----------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10,
                    help="timed steps of the headline (resident) and e2e legs; the per-kernel medians and the configs entries use fixed counts")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="vcfx_b200", choices=["vcfx_b200", "reference"])
    ap.add_argument("--variants", type=int, default=C2_VARIANTS, help="variants per GPU (default: full C2)")
    ap.add_argument("--tile", type=int, default=0, help="tile_bytes for the resident path (0 = library default)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-tool / per-shape entries (N = 1 only)")
    ap.add_argument("--no-cli", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--configs", default="", help="comma-separated subset of C2,C3,C4 for the configs array")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed job computed in its last step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 0)

    if args.impl == "reference":
        return run_reference_arm(args)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    affinity = bind_to_gpu_numa_node(local_rank)      # before torch creates threads or pins memory

    import numpy as np
    import torch
    import torch.distributed as dist

    from vcfx_b200 import api, synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libvcfx_cuda has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    V = args.variants
    warmup = max(args.warmup, 3)
    threads = min(max(1, len(os.sched_getaffinity(0)) // (1 if affinity.get("bound") else max(world, 1))), 48)

    # ---- this rank's shard of the stream, generated straight into pinned host memory
    sh = Shard(torch, np, synth, api, dev, 2, rank * V, V, rank == 0, threads)
    nbytes = sh.nbytes
    log(f"[bench r{rank}] generated {nbytes / 1e9:.3f} GB ({V} variants) in {sh.gen_s:.1f}s; affinity {affinity}")
    d_in = sh.d_in
    out_cap = 64 << 20
    d_out = torch.empty(out_cap, dtype=torch.uint8, device=dev)
    # a real (non-default) stream: the library launches on it and torch's events time it
    tstream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    assert stream != 0

    ctx_af = api.Context(api.OP_ALLELE_FREQ, api.FILE, device=local_rank, stream=stream, chunk_bytes=CHUNK, tile_bytes=args.tile)
    ctx_vc = api.Context(api.OP_VARIANT_COUNT, api.FILE, device=local_rank, stream=stream, chunk_bytes=CHUNK, tile_bytes=args.tile)
    valid_from = 0 if rank else api.find_chrom_header(sh.hdr)
    totals = torch.zeros(2, dtype=torch.int64, device=dev)

    def step_resident():
        ctx_af.run_device(d_in.data_ptr(), nbytes, d_out.data_ptr(), out_cap, valid_from=valid_from)
        ctx_vc.run_device(d_in.data_ptr(), nbytes, 0, 0)

    def reduce_totals(n_jobs: int):
        """The path's only exchange: the scalar totals of the jobs just run, merged with ONE all-reduce
        (a [jobs x 2] int64 tensor) inside the timed region: the shards never talk to each other while they
        are being parsed, so no rank waits for another one between two jobs."""
        if world > 1:
            dist.all_reduce(totals.repeat(max(n_jobs, 1), 1))

    # ---- correctness gate (size-independent properties at full size)
    step_resident()
    torch.cuda.synchronize()
    st_af, st_vc = ctx_af.sync(), ctx_vc.sync()
    assert st_af.rows == V and st_vc.rows == V, (st_af.rows, st_vc.rows, V)
    out_bytes_af = int(st_af.bytes_out)
    head = bytes(d_out[:64].cpu().numpy())
    assert head.startswith(b"21\t"), head
    totals[0] = st_af.rows; totals[1] = st_vc.rows

    for _ in range(warmup):
        step_resident()
    reduce_totals(warmup)
    torch.cuda.synchronize()
    # NVML is set up BEFORE the barrier: done after it, the few milliseconds it takes on rank 0 made rank 0
    # enter the timed region late and every other rank wait for it at the closing all-reduce
    sampler = ClockSampler([physical_gpu_index(r) for r in range(world)] if rank == 0 else [])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.start()
    e0.record()
    t_host0 = time.perf_counter()
    for _ in range(args.steps):
        step_resident()
    reduce_totals(args.steps)
    e1.record()
    host_ms_per_step = (time.perf_counter() - t_host0) * 1e3 / args.steps      # enqueue time only (no sync yet)
    torch.cuda.synchronize()
    clocks = sampler.stop()
    ms_total = e0.elapsed_time(e1)
    st_af, st_vc = ctx_af.sync(), ctx_vc.sync()
    if args.dump_outputs:
        dump_outputs(np, Path(args.dump_outputs), "" if world == 1 else f".rank{rank}",
                     d_out[:int(st_af.bytes_out)].cpu().numpy().tobytes(), int(st_af.rows), int(st_vc.rows))
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    per_rank_ms = [ms_total / args.steps]
    if world > 1:                      # every rank's own time, for the record (value uses the slowest)
        g = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
        dist.all_gather(g, torch.tensor([ms_total / args.steps], dtype=torch.float64, device=dev))
        per_rank_ms = [round(float(x.item()), 4) for x in g]
    log(f"[bench r{rank}] timed region: {ms_total / args.steps:.3f} ms/step on the device, {host_ms_per_step:.3f} ms/step of host enqueue")
    value = world * nbytes / (ms_step / 1e3) / 1e9

    # per-kernel durations (CUDA events around each tool's kernels on the launch stream)
    af_ms, vc_ms = [], []
    for _ in range(5):
        ctx_af.run_device(d_in.data_ptr(), nbytes, d_out.data_ptr(), out_cap, valid_from=valid_from)
        af_ms.append(ctx_af.sync().kernel_ms)
        ctx_vc.run_device(d_in.data_ptr(), nbytes, 0, 0)
        vc_ms.append(ctx_vc.sync().kernel_ms)
    af_k, vc_k = statistics.median(af_ms), statistics.median(vc_ms)
    log(f"[bench r{rank}] kernels alone: allele_freq_calc {af_k:.3f} ms, variant_counter {vc_k:.3f} ms")

    # ---- parity of the timed job: what the full-size resident launch wrote, byte for byte
    parity = None
    ref_outputs = {}
    cpu_run = None
    if rank == 0 and world == 1 and not args.no_parity:
        from oracle import oracle as O
        ctx_af.run_device(d_in.data_ptr(), nbytes, d_out.data_ptr(), out_cap, valid_from=valid_from)
        st_af = ctx_af.sync()
        gpu_out = d_out[:int(st_af.bytes_out)].cpu().numpy().tobytes()
        t0 = time.perf_counter()
        exp_sha, exp_n = oracle_parallel(O, "allele_freq", sh, np)
        parity = {"allele_freq_calc_full": {"against": "oracle port (oracle/vcfx_oracle.c) over the whole 4.3 GB input, all host cores",
                                            "bytes": len(gpu_out), "sha256": hashlib.sha256(gpu_out).hexdigest(),
                                            "equal": hashlib.sha256(gpu_out).hexdigest() == exp_sha and exp_n == len(gpu_out),
                                            "oracle_seconds": time.perf_counter() - t0},
                  "variant_counter_full": {"against": "line count of the generator", "rows": int(st_vc.rows), "equal": int(st_vc.rows) == V}}
        if not args.no_cpu_baseline and V >= CPU_SAMPLE_VARIANTS:
            cpu_run = cpu_reference_run(CPU_SAMPLE_VARIANTS, 2, 1, keep_outputs=ref_outputs)
            if cpu_run and "allele_freq_calc" in ref_outputs:
                ref_af = ref_outputs["allele_freq_calc"]
                body = ref_af[len(api.AF_HEADER):]
                parity["allele_freq_calc_vs_reference_tool"] = {
                    "against": f"oracle/_ref/VCFX_allele_freq_calc -q -i on the first {CPU_SAMPLE_VARIANTS} variants (unmodified reference tool)",
                    "bytes": len(body), "equal": ref_af.startswith(api.AF_HEADER) and gpu_out[:len(body)] == body,
                    "what": "the first rows of the FULL-SIZE resident output against the reference tool's stdout"}
                parity["variant_counter_vs_reference_tool"] = {
                    "against": "oracle/_ref/VCFX_variant_counter on the same prefix", "equal": ref_outputs["variant_counter"] == b"Total Variants: %d\n" % CPU_SAMPLE_VARIANTS}
        parity["hwe_pvalue"] = hwe_pvalue_report(api, O, np)
        parity["all_equal"] = all(v.get("equal", True) for v in parity.values() if isinstance(v, dict)) and parity["hwe_pvalue"]["within_tolerance"]
        log(f"[bench] parity: {json.dumps({k: (v.get('equal', v.get('within_tolerance')) if isinstance(v, dict) else v) for k, v in parity.items()})}")

    # ---- e2e: host buffers through the streaming C ABI, H2D + D2H inside the timed region
    e2e = None
    h2d_ceiling = None
    if not args.no_e2e:
        ctx_af_s = api.Context(api.OP_ALLELE_FREQ, api.FILE, device=local_rank, chunk_bytes=CHUNK, n_slots=3)
        ctx_vc_s = api.Context(api.OP_VARIANT_COUNT, api.FILE, device=local_rank, chunk_bytes=CHUNK, n_slots=3)
        bounds = sh.bounds
        base_ptr = sh.host.data_ptr()

        def step_e2e():
            """The job through the C ABI from host memory: every chunk is uploaded ONCE
            (vcfx_cuda_submit_host on the allele_freq_calc context) and variant_counter runs on the same
            device bytes (vcfx_cuda_submit_shared); both texts come back to the host."""
            rows_af = rows_vc = nout = 0

            def drain_pair():
                nonlocal rows_af, rows_vc, nout
                out, st, _ = ctx_vc_s.next_output(); rows_vc += st.rows; nout += len(out)
                out, st, _ = ctx_af_s.next_output(); rows_af += st.rows; nout += len(out)

            for (s, e) in bounds:
                vf = min(max(valid_from - s, 0), e - s)
                while not ctx_af_s.submit_host(base_ptr + s, e - s, valid_from=vf, is_final=(e == nbytes)):
                    drain_pair()
                ok = ctx_vc_s.submit_shared(ctx_af_s, is_final=(e == nbytes))
                assert ok
            while ctx_af_s.in_flight():
                drain_pair()
            assert rows_af == V and rows_vc == V, (rows_af, rows_vc)
            if world > 1:
                dist.all_reduce(totals)
            return nout

        for _ in range(2):
            d2h = step_e2e()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e2e_steps = args.steps
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            d2h = step_e2e()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        t = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item()) / e2e_steps
        ctx_af_s.close(); ctx_vc_s.close()
        h2d_ceiling = measure_h2d_ceiling(torch, sh, dev, dist, world)
        e2e = {"value": world * nbytes / e2e_s / 1e9, "unit": "GB/s", "ms_per_step": e2e_s * 1e3, "steps": e2e_steps,
               "h2d_bytes_per_step": nbytes, "d2h_bytes_per_step": int(d2h),
               "h2d_ceiling_GBps": h2d_ceiling, "frac_of_h2d_ceiling": (world * nbytes / e2e_s / 1e9) / h2d_ceiling if h2d_ceiling else None,
               "note": "pinned host memory -> 64 MiB chunks, 3 slots in flight; each chunk is uploaded once and feeds both tools (vcfx_cuda_submit_host + vcfx_cuda_submit_shared); "
                       "h2d_ceiling = the same chunks copied host->device with no kernel, all ranks at once"}

    # ---- roofline of the dominant kernel
    peaks_path = ROOT / "MEASURED_PEAKS.json"
    if peaks_path.exists():
        peak = float(json.loads(peaks_path.read_text())["hbm_gbs"]); peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)"
    else:
        peak = 6650.0; peak_src = "B200_PROFILING.md fallback (of fallback)"
    alg_bytes = nbytes + out_bytes_af
    achieved = alg_bytes / (af_k / 1e3) / 1e9
    # DRAM traffic of the dominant kernel from the committed ncu --set full capture of this workload
    traffic = None
    for prof in (ROOT / "profiles" / "r2_ncu_full_c2.json", ROOT / "profiles" / "r1_ncu_full_c2.json"):
        if prof.exists() and V == C2_VARIANTS:
            try:
                ks = [k for k in json.loads(prof.read_text()) if "vcfx_scan_kernel<1>" in k["Kernel Name"] or "(int)1" in k["Kernel Name"]]
                k = ks[0]

                def gb(v):
                    num, unit = v.split()[:2]
                    return float(num) * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}[unit]
                traffic = gb(k["dram__bytes_read.sum"]) + gb(k["dram__bytes_write.sum"])
                break
            except Exception:
                traffic = None
    roofline = {"bound": "hbm", "kernel": "vcfx_scan_kernel<OP_AF> (+ tile_scan + format_rows: the tool's kernels)", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "algorithmic_bytes_per_launch": alg_bytes,
                "kernel_ms": af_k, "peak_source": peak_src,
                "other_kernels": {"vcfx_scan_kernel<OP_VC>+resolve_events": {"kernel_ms": vc_k,
                                  "achieved": nbytes / (vc_k / 1e3) / 1e9, "frac": nbytes / (vc_k / 1e3) / 1e9 / peak}}}

    ctx_af.close(); ctx_vc.close()
    configs = None
    cli = None
    if rank == 0 and world == 1:
        from oracle import oracle as O
        if not args.no_cli and V == C2_VARIANTS:
            cli = cli_leg(np, sh)
            log(f"[bench] cli: {json.dumps(cli)[:400]}")
        del d_in, d_out
        sh_hdr = sh.hdr
        del sh
        torch.cuda.empty_cache()
        if not args.no_configs:
            only = set(args.configs.split(",")) if args.configs else None
            configs = config_entries(torch, np, api, synth, O, dev, peak, threads, only)

    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline and world == 1:      # reported at N=1 only
            r = cpu_run or cpu_reference_run(CPU_SAMPLE_VARIANTS, 2, 1)
            if not r:
                log("[bench] reference tools not built (oracle/_ref/VCFX_*, make -C oracle ref REFERENCE=<VCFX source tree>): "
                    "no cpu_baseline, and the parity entries compare with the oracle instead")
            if r:
                cpu = {"value": r["gbps"], "unit": "GB/s", "cores": 1, "kind": "reference",
                       "sample": f"{r['variants']} variants x {SAMPLES} samples ({r['bytes'] / 1e9:.2f} GB) of the C2 stream, "
                                 f"allele_freq_calc -q -i + variant_counter, best-effort warm cache, {os.cpu_count()} host cores present"}
        line = {
            "metric": "vcf_input_GB_per_s", "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps,
            "warmup": warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": workload_config(),
            "genotypes_per_s": world * V * SAMPLES / (ms_step / 1e3),
            "variants_per_s": world * V / (ms_step / 1e3),
            "bytes_per_gpu": nbytes,
            "e2e": e2e, "gpu_launches": 5 * args.steps, "per_rank_ms_per_step": per_rank_ms, "clocks": clocks,
            "roofline": roofline, "cpu_baseline": cpu, "parity": parity, "configs": configs, "cli": cli,
            "affinity": affinity,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
