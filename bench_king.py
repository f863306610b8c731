"""KING relatedness on the tensor cores: king_planes_kernel and king_mma_kernel timed on one slab of .bed rows, next to
torch._int_mm on the same planes, with the counts checked exactly against float64 torch.matmul.

    python bench_king.py [--reps R] [--warmup W]

Two shapes: C2 (2,504 samples x 427,409 variants from synth, as bench.py's C2) and a compute-heavy one (10,000 samples x
100,000 variants).  The .bed rows are built on the device by dosage_bed_device.  One slab (the rows one planes buffer
holds, vcfx_cuda_king_slab_rows) is added R times after W warm-up adds; CUDA events around each add give the slab time
(device copy of the rows + planes + MMA), and torch.profiler in a separate pass gives each kernel's device time by name.
Medians.  Algorithmic int8 ops per slab: 2 K (2 S (S + 1) / 2 + 2 S^2) for K rows and S samples (HH and CC are symmetric,
AB and HC are not).  The share of peak is over the data sheet's dense INT8 rate, 4,500 TOPS for one B200 (it prints 72
POPS for eight GPUs with sparsity).  The card's name and power limit are read in the same run.  Prints one JSON line and
writes nothing in the tree.
"""
from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

PEAK_INT8_TOPS = 4500.0
SHAPES = {"C2": (2504, 427409), "heavy": (10000, 100000)}


def gpu_facts():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    name, power = [x.strip() for x in r.stdout.strip().split(",")] if r.returncode == 0 else ("unknown", "unknown")
    return name, power


def planes_of(packed, n):
    """int8 planes A, H, B, C [n, rows] of .bed rows [rows, ceil(n / 4)], unpacked by torch."""
    import torch
    shifts = torch.arange(0, 8, 2, device=packed.device, dtype=torch.uint8)
    x = ((packed[:, :, None] >> shifts) & 3).reshape(packed.shape[0], -1)[:, :n].T.contiguous()
    return [(x == 3).to(torch.int8), (x == 2).to(torch.int8), (x == 0).to(torch.int8), (x != 1).to(torch.int8)]


def run_shape(tag, S, V, reps, warmup):
    import torch
    from vcfx_b200 import api, synth
    data = synth.make_vcf(2, V, S, seed=7)
    d_in = torch.zeros(len(data) + api.DEVICE_PAD, dtype=torch.uint8, device="cuda")
    d_in[:len(data)] = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    del data
    bed = api.dosage_bed_device(d_in, len(d_in) - api.DEVICE_PAD)
    del d_in
    assert bed.width == S and bed.packed.shape[0] == V, (bed.width, bed.packed.shape)
    k = api.King(S)
    K = min(k.slab_rows, V)
    slab = bed.packed[:K].contiguous()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    times = []
    for i in range(warmup + reps):
        ev[0].record()
        k.add(slab)                                  # exactly one slab: one planes and one MMA launch
        ev[1].record()
        torch.cuda.synchronize()
        if i >= warmup:
            times.append(ev[0].elapsed_time(ev[1]))
    c = k.counts()
    assert c.rows == (warmup + reps) * K
    # the counts of one slab, exactly, against float64 products of the planes
    A, H, B, Cc = planes_of(slab, S)
    reps_total = warmup + reps
    for name, got, (p, q) in zip(("CC", "HH", "AB", "HC"), (c.cc, c.hh, c.ab, c.hc), ((Cc, Cc), (H, H), (A, B), (H, Cc))):
        want = (p.double() @ q.double().T).round().to(torch.int64) * reps_total
        assert torch.equal(got, want), f"{tag}: {name} differs from float64 torch.matmul"
    del c
    # per-kernel device times in a separate, profiled pass
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            k.add(slab)
        torch.cuda.synchronize()
    kern = {"king_planes_kernel": [], "king_mma_kernel": []}
    for e in prof.events():
        for name in kern:
            if name in e.name and e.device_type.name == "CUDA":
                kern[name].append(e.time_range.elapsed_us() / 1e3)
    k.close()
    # torch._int_mm on the same planes: the four full S x S products
    Bt = {id(q): q.T.contiguous() for q in (Cc, H, B)}
    def int_mm_only():
        return [torch._int_mm(p, Bt[id(q)]) for p, q in ((Cc, Cc), (H, H), (A, B), (H, Cc))]
    mm_times = []
    for i in range(warmup + reps):
        ev[0].record()
        out = int_mm_only()
        ev[1].record()
        torch.cuda.synchronize()
        if i >= warmup:
            mm_times.append(ev[0].elapsed_time(ev[1]))
    for name, got, (p, q) in zip(("CC", "HH", "AB", "HC"), out, ((Cc, Cc), (H, H), (A, B), (H, Cc))):
        assert torch.equal(got.to(torch.int64), (p.double() @ q.double().T).round().to(torch.int64)), f"{tag}: _int_mm {name}"
    del out, Bt
    ops = 2.0 * K * (2 * S * (S + 1) / 2 + 2 * S * S)
    med = {n: statistics.median(v) if v else None for n, v in kern.items()}
    t_slab, t_mm = statistics.median(times), statistics.median(mm_times)
    t_mma = med["king_mma_kernel"]
    bytes_planes = 4 * K * S + K * ((S + 3) // 4)
    res = {
        "shape": tag, "samples": S, "variants": V, "slab_rows": K,
        "int8_ops_per_slab": ops,
        "slab_ms": round(t_slab, 4),
        "planes_kernel_ms": round(med["king_planes_kernel"], 4) if med["king_planes_kernel"] else None,
        "mma_kernel_ms": round(t_mma, 4) if t_mma else None,
        "mma_tops": round(ops / (t_mma * 1e-3) / 1e12, 1) if t_mma else None,
        "mma_share_of_int8_peak": round(ops / (t_mma * 1e-3) / 1e12 / PEAK_INT8_TOPS, 4) if t_mma else None,
        "slab_tops": round(ops / (t_slab * 1e-3) / 1e12, 1),
        "int_mm_ms": round(t_mm, 4),
        "int_mm_tops": round(ops / (t_mm * 1e-3) / 1e12, 1),
        "planes_bytes_written_read": bytes_planes,
        "bound": "compute (int8 tensor-core ops; the planes pass is memory-bound)",
        "counts_exact": True,
    }
    del A, H, B, Cc, slab, bed
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--shapes", default="C2,heavy")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_king.py needs a CUDA device: there is no CPU path")
    name, power = gpu_facts()
    out = {"metric": "king_counts", "gpu": name, "power_limit": power, "peak_int8_tops_datasheet": PEAK_INT8_TOPS,
           "shapes": [run_shape(t, *SHAPES[t], a.reps, a.warmup) for t in a.shapes.split(",")]}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
