#!/usr/bin/env python
"""bench_ops.py — kernel-only throughput of every op on the BASELINE shapes (1 GPU, data resident
in HBM).  Complements bench.py (which reports the contractual C2 line): one JSON line per
(config, tool) with the event-timed kernel time, algorithmic bytes (input + output) per second and
the fraction of the measured HBM peak.

  C2  427,409 x 2,504 phased GT                      allele_freq_calc, variant_counter, hwe_tester
  C3  C2 shape + 5 % missing / unphased / haploid    missing_detector, allele_counter (TEXT, -a), allele_freq_calc
  C2, C3 also: dosage_calculator as text, as its int8 matrix (dosage_matrix, VCFX_F_DS_MATRIX, width = S) and as
              PLINK 1 .bed rows (dosage_bed, VCFX_F_DS_BED, width = S)
  C4  GT:AD:DP:GQ:PL multi-allelic (scaled to ~4 GB) hwe_tester, allele_freq_calc
"""
from __future__ import annotations

import argparse
import json
import statistics
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the full variant counts")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--configs", default="C2,C3,C4")
    ap.add_argument("--tools", default="", help="comma-separated substrings: only tools whose name contains one of them")
    ap.add_argument("--warm", type=int, default=2, help="untimed runs per tool (0 under ncu: one launch per kernel)")
    args = ap.parse_args()

    import numpy as np
    import torch
    from vcfx_b200 import api, synth

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    peak = 6545.3
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        peak = float(json.loads(p.read_text())["hbm_gbs"])
    S = 2504
    plans = {
        "C2": (2, int(427409 * args.scale), [("allele_freq_calc", api.OP_ALLELE_FREQ, 0), ("variant_counter", api.OP_VARIANT_COUNT, 0),
                                             ("hwe_tester", api.OP_HWE, 0), ("nonref_filter", api.OP_NONREF_FILTER, 0), ("phase_checker", api.OP_PHASE_CHECK, 0),
                                             ("indexer", api.OP_INDEX, 0), ("inbreeding_calculator", api.OP_INBREEDING, 0), ("genotype_query", api.OP_GENOTYPE_QUERY, 0), ("dosage_calculator", api.OP_DOSAGE, 0),
                                             ("dosage_matrix", api.OP_DOSAGE, api.F_DS_MATRIX), ("dosage_bed", api.OP_DOSAGE, api.F_DS_BED)]),
        "C3": (3, int(427409 * args.scale), [("missing_detector", api.OP_MISSING_DETECT, 0), ("allele_counter -a", api.OP_ALLELE_COUNT, api.F_AC_AGGREGATE),
                                             ("allele_counter", api.OP_ALLELE_COUNT, 0), ("allele_freq_calc", api.OP_ALLELE_FREQ, 0),
                                             ("inbreeding_calculator", api.OP_INBREEDING, 0), ("dosage_calculator", api.OP_DOSAGE, 0),
                                             ("dosage_matrix", api.OP_DOSAGE, api.F_DS_MATRIX), ("dosage_bed", api.OP_DOSAGE, api.F_DS_BED)]),
        "C4": (4, int(60000 * args.scale), [("hwe_tester", api.OP_HWE, 0), ("allele_freq_calc", api.OP_ALLELE_FREQ, 0)]),
    }
    for cname in args.configs.split(","):
        shape, V, tools = plans[cname]
        hdr = synth.header(shape, S, shape)
        cap = len(hdr) + synth.line_bound(shape, S) * V
        host = torch.empty(cap, dtype=torch.uint8, pin_memory=True)
        hnp = host.numpy()
        hnp[: len(hdr)] = np.frombuffer(hdr, dtype=np.uint8)
        t0 = time.perf_counter()
        nbytes = len(hdr) + synth.lines_into(hnp[len(hdr):], shape, S, 0, V, seed=shape)
        first_nl = int(np.argmax(hnp[len(hdr):len(hdr) + (4 << 20)] == 10))
        line_len = first_nl + 1                       # what a streaming caller's library measures by itself
        d_in = torch.empty(nbytes + api.DEVICE_PAD, dtype=torch.uint8, device=dev)
        d_in[:nbytes].copy_(host[:nbytes]); torch.cuda.synchronize()
        print(f"[{cname}] {nbytes / 1e9:.2f} GB, {V} variants, generated in {time.perf_counter() - t0:.1f}s", file=sys.stderr, flush=True)
        del host
        names = [b"HG%05d" % (96 + i) for i in range(S)]
        for tname, op, flags in tools:
            if args.tools and not any(t == tname for t in args.tools.split(",")):
                continue
            out_cap = 64 << 20
            if op in (api.OP_MISSING_DETECT, api.OP_NONREF_FILTER, api.OP_PHASE_CHECK, api.OP_GENOTYPE_QUERY, api.OP_DOSAGE):
                out_cap = nbytes + nbytes // 50 + (1 << 20)
            if op == api.OP_ALLELE_COUNT and flags == 0:
                out_cap = int(nbytes * 9.5) + (1 << 20)
            if op == api.OP_DOSAGE and flags == api.F_DS_MATRIX:
                out_cap = (V + hdr.count(b"\n") + 1) * (16 + S)          # rows <= lines, 16 + W bytes a row
            if op == api.OP_DOSAGE and flags == api.F_DS_BED:
                out_cap = (V + hdr.count(b"\n") + 1) * (16 + (S + 3) // 4)
            d_out = torch.empty(out_cap, dtype=torch.uint8, device=dev)
            kw = dict(sel_cols=list(range(S)), sel_names=names) if op in (api.OP_ALLELE_COUNT, api.OP_INBREEDING) else (dict(query=b"1/1") if op == api.OP_GENOTYPE_QUERY
                                                                                                                   else dict(width=S) if (op == api.OP_DOSAGE and flags) else {})
            ctx = api.Context(op, api.FILE, flags=flags, **kw)
            ctx.set_line_hint(line_len)
            vf = api.find_chrom_header(hdr) if op in (api.OP_ALLELE_FREQ, api.OP_NONREF_FILTER, api.OP_PHASE_CHECK, api.OP_INDEX) else (api.first_data_offset(hdr) if op == api.OP_MISSING_DETECT else 0)
            ms = []
            st = None
            for i in range(args.reps + args.warm):
                ctx.run_device(d_in.data_ptr(), nbytes, d_out.data_ptr(), out_cap, valid_from=vf)
                st = ctx.sync()
                if i >= args.warm:
                    ms.append(st.kernel_ms)
            k = statistics.median(ms)
            alg = nbytes + int(st.bytes_out)
            line = {"config": cname, "tool": tname, "variants": V, "samples": S, "input_GB": nbytes / 1e9, "output_GB": st.bytes_out / 1e9,
                    "kernel_ms": k, "input_GB_per_s": nbytes / k / 1e6, "algorithmic_GB_per_s": alg / k / 1e6,
                    "frac_of_measured_hbm_peak": alg / k / 1e6 / peak, "genotypes_per_s": V * S / (k / 1e3),
                    "rows": int(st.rows), "flagged": int(st.flagged), "data_lines": int(st.data_lines)}
            print(json.dumps(line), flush=True)
            ctx.close()
            del d_out
            torch.cuda.empty_cache()
        del d_in
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
