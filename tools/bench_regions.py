#!/usr/bin/env python
"""Many small regions with paired reads: three ways to the same [H_g, T_g] template matrices of a batch of C1-shaped regions
(default 1 000 regions x 1 000 reads x 8 haplotypes, L = 150, Lh = 300, band 8; reads paired into two-read templates, a seeded 5 %
singletons; production mode: per-region flank states, naive shortcut, device k-mer mapper):

  a  one phmm_populate_templates call per region (what a caller does without a many-regions call)
  b  one phmm_populate_regions call (per-read values), the template sums in numpy on the host
  c  one phmm_populate_regions_ex call with the templates (sums fused into the epilogue kernel)

(a) and (c) must be bit-identical, and so must (b). Timing: host clock around the synchronous calls, after a warm-up, in windows of
at least --window-s seconds, the three ways alternating window by window, --windows windows each; the spread over the windows is
reported. Writes bench_regions.json to --out and prints it as one line. There is no CPU fallback: without a GPU it stops at the
first device call."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def make_workload(n_regions, n_reads, n_haps, seed=2026):
    from octopus_b200 import synth
    from octopus_b200.batch import concat_blocks, concat_templates
    rng = np.random.default_rng(seed)
    c = synth.CONFIGS["C1"]
    hap_blocks, read_blocks, toffs, flanks = [], [], [], []
    for _ in range(n_regions):
        h = synth.make_haplotypes(rng, n_haps, c["hap_len"])
        r = synth.make_reads(rng, h, n_reads, c["read_lens"], c["band"], c["quals"])
        sizes = []
        while sum(sizes) < n_reads:
            sizes.append(1 if (rng.random() < 0.05 or sum(sizes) == n_reads - 1) else 2)
        hap_blocks.append(h); read_blocks.append(r)
        toffs.append(np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64))
        flanks.append((int(rng.integers(20, 61)), int(rng.integers(20, 61))))
    haps, reads, hf, rf = concat_blocks(hap_blocks, read_blocks)
    toff, tf = concat_templates(toffs)
    return dict(hap_blocks=hap_blocks, read_blocks=read_blocks, toffs=toffs, flanks=flanks, haps=haps, reads=reads, hf=hf, rf=rf,
                toff=toff, tf=tf, band=c["band"])


def sum_templates_host(flat, hf, rf, toff, tf):
    """(b)'s host step: per-read [H_g, R_g] matrices back to back -> the regions' [H_g, T_g] template matrices back to back. Each sum
    runs in read order from the first read (np.add.reduceat over at most two reads per template: (0.0 + x) + y == x + y)."""
    out = np.empty(int((np.diff(hf).astype(np.int64) * np.diff(tf)).sum()))
    o_in = o_out = 0
    for g in range(len(hf) - 1):
        H, R, T = int(hf[g + 1] - hf[g]), int(rf[g + 1] - rf[g]), int(tf[g + 1] - tf[g])
        m = flat[o_in:o_in + H * R].reshape(H, R)
        starts = toff[tf[g]:tf[g + 1]] - rf[g]
        out[o_out:o_out + H * T] = np.add.reduceat(m, starts, axis=1).reshape(-1)
        o_in += H * R; o_out += H * T
    return out


def gpu_identity():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return {"gpu": name, "nvidia_smi": q}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--regions", type=int, default=1000)
    ap.add_argument("--reads", type=int, default=1000)
    ap.add_argument("--haps", type=int, default=8)
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--window-s", type=float, default=1.0)
    ap.add_argument("--tiny", action="store_true", help="8 regions x 40 reads: a rehearsal of the whole script")
    ap.add_argument("--out", required=True, help="directory for bench_regions.json (created if missing)")
    a = ap.parse_args()
    if a.tiny:
        a.regions, a.reads = 8, 40
    t0 = time.perf_counter()
    w = make_workload(a.regions, a.reads, a.haps)
    setup_s = time.perf_counter() - t0
    from octopus_b200 import HaplotypeLikelihoodModel, PairHMMEngine, PhmmError
    try:
        eng = PairHMMEngine(0)
    except PhmmError as e:
        sys.exit("bench_regions: no usable GPU (%s); there is no CPU fallback" % e)
    cfg = HaplotypeLikelihoodModel.Config(max_indel_error=w["band"])          # production defaults: shortcut on, device mapper on
    haps, reads = w["haps"].pin(), w["reads"].pin()
    hf, rf, toff, tf, flanks = w["hf"], w["rf"], w["toff"], w["tf"], w["flanks"]

    def run_a():
        parts, cells = [], 0
        for h, r, to, fl in zip(w["hap_blocks"], w["read_blocks"], w["toffs"], flanks):
            parts.append(eng.populate_templates(cfg, h, r, to, flank_state=fl).reshape(-1))
            cells += eng.last_dp_cells()
        return np.concatenate(parts), cells, 0.0

    def run_b():
        flat, _ = eng.populate_regions(cfg, haps, reads, hf, rf, flank_states=flanks)
        cells = eng.last_dp_cells()
        t = time.perf_counter()
        out = sum_templates_host(flat, hf, rf, toff, tf)
        return out, cells, time.perf_counter() - t

    def run_c():
        flat, _ = eng.populate_regions(cfg, haps, reads, hf, rf, flank_states=flanks, templates=(toff, tf))
        return flat, eng.last_dp_cells(), 0.0

    ways = {"a_per_region_templates": run_a, "b_regions_plus_host_sums": run_b, "c_regions_templates": run_c}
    results = {}
    for k, f in ways.items():                  # warm-up of every shape, and the answers
        f()
        results[k] = f()[0]
    same_ac = results["a_per_region_templates"].tobytes() == results["c_regions_templates"].tobytes()
    same_bc = results["b_regions_plus_host_sums"].tobytes() == results["c_regions_templates"].tobytes()
    assert same_ac, "(a) and (c) differ"
    windows = {k: [] for k in ways}
    for _ in range(a.windows):
        for k, f in ways.items():
            n, host_only, cells = 0, 0.0, 0
            t = time.perf_counter()
            while True:
                _, cells, h = f()
                n += 1; host_only += h
                el = time.perf_counter() - t
                if el >= a.window_s:
                    break
            windows[k].append({"ms_per_batch": 1e3 * el / n, "engine_ms_per_batch": 1e3 * (el - host_only) / n, "batches": n, "cells": cells})
    summary = {}
    for k, ws in windows.items():
        ms = np.array([x["ms_per_batch"] for x in ws]); ems = np.array([x["engine_ms_per_batch"] for x in ws])
        cells = ws[-1]["cells"]
        summary[k] = {"ms_per_batch_median": float(np.median(ms)), "ms_per_batch_min": float(ms.min()), "ms_per_batch_max": float(ms.max()),
                      "engine_ms_per_batch_median": float(np.median(ems)), "dp_cells": int(cells),
                      "gcups_median": cells / (np.median(ms) / 1e3) / 1e9, "windows": ws}
    b, c, aa = summary["b_regions_plus_host_sums"], summary["c_regions_templates"], summary["a_per_region_templates"]
    rec = {"what": "bench_regions", "regions": a.regions, "reads_per_region": a.reads, "haps_per_region": a.haps, "read_len": 150,
           "hap_len": 300, "band": w["band"], "templates": int(len(toff) - 1), "mode": "flank state + naive shortcut + device mapper",
           "window_s": a.window_s, "setup_s": setup_s, "a_equals_c_bitwise": same_ac, "b_equals_c_bitwise": same_bc,
           "c_engine_over_b_engine": c["engine_ms_per_batch_median"] / b["engine_ms_per_batch_median"],
           "a_over_c": aa["ms_per_batch_median"] / c["ms_per_batch_median"], "results": summary}
    rec.update(gpu_identity())
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "bench_regions.json"), "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({k: v for k, v in rec.items() if k != "results"} | {k: {m: v[m] for m in v if m != "windows"} for k, v in summary.items()}))


if __name__ == "__main__":
    main()
