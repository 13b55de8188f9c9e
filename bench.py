#!/usr/bin/env python
"""bench.py — pair-HMM GCUPS of the B200 engine on BASELINE.json's (reads x haplotypes) workload.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config C3] [--reads R] [--haps H]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

A step = one pass of the hot path (HaplotypeLikelihoodArray::populate semantics, one mapping position per pair, naive
shortcut disabled so that CPU and GPU do identical DP work) over one synthetic batch. Metric: banded DP cell-updates/s,
cells per alignment = 2*(L+band)*band (simd_pair_hmm.hpp:271). Prints ONE JSON line on rank 0.

  value  device-resident inputs → device-resident double matrix (+ gather to rank 0 when N > 1), max over ranks
  e2e    the same call through the C ABI with pinned HOST buffers: H2D of the batch and D2H of the matrix inside the timed region
  roofline / cpu_baseline / clocks: see DESIGN.md "Measurement"
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C3", help="BASELINE config name (octopus_b200.synth.CONFIGS)")
    ap.add_argument("--reads", type=int, default=None, help="override reads per GPU (debug)")
    ap.add_argument("--haps", type=int, default=None)
    ap.add_argument("--cpu-sample-reads", type=int, default=None, help="reads in the CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    # non-headline modes (diagnostics; the headline is the default: one position per pair, DP for every pair, no flank state)
    ap.add_argument("--flank", default=None, help="LHS,RHS flank sizes: exercises the traceback + flank-discount path")
    ap.add_argument("--shortcut", action="store_true", help="enable the reference's naive shortcut (reference behaviour)")
    ap.add_argument("--map", action="store_true", help="candidate positions from the device k-mer mapper (reference behaviour)")
    ap.add_argument("--band", type=int, default=None, help="override the config's band (wide-band diagnostics)")
    ap.add_argument("--hap-len", type=int, default=None, help="override the haplotype length")
    ap.add_argument("--read-lens", default=None, help="override the read lengths, comma separated")
    ap.add_argument("--int-scores", action="store_true", help="HaplotypeLikelihoodModel::Config::use_int_scores (reference: int32 lanes)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: every rank owns a batch of the config's shape; strong: the config's reads are split over the ranks (SURVEY.md §8e, C3) "
                         "and the [H, R] matrix is re-assembled on rank 0")
    ap.add_argument("--regions", type=int, default=None, help="regions per rank and step (C5: 1k regions over 8 GPUs = 125 per rank); each its own reads and haplotypes")
    ap.add_argument("--batch-regions", type=int, default=None,
                    help="regions per CALL: the rank's regions go to the GPU in one phmm_populate_regions call (Octopus's real call shape: many small "
                         "active regions) instead of one phmm_populate call per region")
    ap.add_argument("--reserve-sms", type=int, default=0,
                    help="SMs kept free of persistent DP blocks for a collective that runs beside the next call (phmm_reserve_sms)")
    ap.add_argument("--unordered-penalties", action="store_true",
                    help="draw gap_extend without the cap at gap_open (only the PacBio / custom error models produce such arrays); the DP kernels detect it and run their general (6 ALU-op) deletion update")
    ap.add_argument("--gather", choices=["peer", "nccl"], default="peer",
                    help="several ranks: how the values reach rank 0 — peer (each rank's epilogue stores into rank 0's HBM through a CUDA IPC mapping) or nccl (gather collective)")
    ap.add_argument("--error-model", default=None, help="haplotype penalty arrays from the reference's error models (reset()), e.g. PCR-free.HiSeq-2500, instead of i.i.d. draws")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write the ln-likelihood matrices of the last timed step (rank 0's) to DIR/<name>.npy, "
                         "float64; above %d MB in all, a seeded sample of each matrix's columns (indices in <name>_columns.npy)" % (DUMP_BYTES // 10**6))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_BYTES = 64_000_000


def dump_outputs(dirname, outputs):
    """outputs: [(name, [H, R] float64 tensor)]. Every matrix whole, or, when they would take more than DUMP_BYTES together, the
    same seeded sample of columns (reads) of each in every run with the same arguments, so that two builds compare value for value."""
    import torch
    os.makedirs(dirname, exist_ok=True)
    budget = (DUMP_BYTES - (1 << 20)) // len(outputs)                 # 1 MB for the .npy headers
    sample = sum(t.numel() for _, t in outputs) * 8 > DUMP_BYTES - (1 << 20)
    for name, t in outputs:
        H, R = t.shape
        if sample:
            k = max(1, min(R, budget // (8 * (H + 1))))
            cols = np.sort(np.random.default_rng(0).choice(R, k, replace=False))
            np.save(os.path.join(dirname, name + "_columns.npy"), cols.astype(np.float64))
            t = t[:, torch.as_tensor(cols, device=t.device)]
        np.save(os.path.join(dirname, name + ".npy"), t.cpu().numpy().astype(np.float64, copy=False))


METRIC = "pair-HMM GCUPS (DP cell-updates/s)"


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def issue_roofline(kernel_gcups, reads, band, clocks, alu_ops):
    """The binding roofline of the packed DP (DESIGN.md section 4): `alu_ops` half-rate ALU-pipe instructions per cell pair (5 when
    gap_open >= gap_extend everywhere — the OGE deletion update — else 6) at 64 thread-instructions/clk/SM; beside it the issue
    bound of the steady-state loop (9.6 warp instructions per cell pair, SASS). Both in the reference's cell count 2(L+B)B per
    alignment (the column sweep itself touches 2LB cells)."""
    lens = np.diff(np.asarray(reads.off))
    mean_ratio = float(((lens + band) / lens).mean())
    mhz = (clocks or {}).get("sm_mhz") or 1965.0
    peak = 148 * mhz * 1e6 * (64.0 * 2.0 / alu_ops) * mean_ratio / 1e9
    issue_peak = 148 * mhz * 1e6 * (4 * 64.0 / 9.6) * mean_ratio / 1e9
    return {"bound": "alu-pipe (DPX packed-16)", "achieved": kernel_gcups, "peak": peak, "unit": "GCUPS", "frac": kernel_gcups / peak,
            "alu_instr_per_cell_pair": alu_ops, "alu_thread_instr_per_clk_per_sm": 64, "sm_mhz": mhz,
            "issue_peak": issue_peak, "issue_frac": kernel_gcups / issue_peak, "warp_instr_per_cell_pair": 9.6}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def host_threads():
    """Host threads the CPU arm may use: the cgroup CPU quota when there is one (a 128-thread box may grant a pod only a
    few CPUs' worth of time), else the online CPU count."""
    n = os.cpu_count() or 1
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(round(int(quota) / int(period)))))
    except Exception:
        pass
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    return n


def calibrated_sample(haps, reads, band, threads, target_s):
    """Number of reads whose (reads x all haplotypes) CPU pass takes about target_s seconds (measured on a small probe)."""
    probe = min(reads.n, max(64, 16 * threads))
    cpu_reference_run(haps, reads, band, probe, threads)
    g, dt, _, _, _ = cpu_reference_run(haps, reads, band, probe, threads)
    per_read = max(dt / probe, 1e-7)
    return int(max(probe, min(reads.n, target_s / per_read)))


def reference_batch_dict(haps, reads):
    return dict(read_bases=reads.bases, read_quals=reads.quals, read_off=reads.off, hap_seq=haps.seq,
                hap_mask_fwd=haps.snv_mask_fwd, hap_prior_fwd=haps.snv_prior_fwd, hap_mask_rev=haps.snv_mask_rev,
                hap_prior_rev=haps.snv_prior_rev, hap_gap_open=haps.gap_open, hap_gap_extend=haps.gap_extend, hap_off=haps.off)


def cpu_reference_run(haps, reads, band, n_sample_reads, threads, isa=None, want_scores=False):
    """Time the reference's own SIMD kernel (oracle/_ref; the build its -march=native would select = what BASELINE names) — or,
    where that build is absent, the C port — on the first n_sample_reads reads x all haplotypes, one mapping position per pair.
    Returns (gcups, seconds, kind, isa_name, cells[, integer scores [n, H] or None])."""
    from oracle.oracle import COracle, RefKernel, available_ref_isas
    n = min(n_sample_reads, reads.n)
    H = haps.n
    lens = np.diff(reads.off[:n + 1])
    cells = int((2 * (lens + band) * band).sum()) * H
    isas = available_ref_isas()
    if isas:
        isa = isa or isas[0]   # the widest build this host runs == what the reference's -march=native build would select
        k = RefKernel(isa)
        batch = reference_batch_dict(haps, reads)
        ridx = np.repeat(np.arange(n, dtype=np.int32), H)
        hidx = np.tile(np.arange(H, dtype=np.int32), n)
        woff = np.repeat((reads.begin[:n] - band).astype(np.int32), H)
        rev = np.repeat(reads.reverse[:n].astype(bool), H)
        parts = []
        for strand in (False, True):
            sel = rev == strand
            if sel.any():
                parts.append((strand, sel, np.ascontiguousarray(ridx[sel]), np.ascontiguousarray(hidx[sel]), np.ascontiguousarray(woff[sel])))
        scores = np.empty(n * H, dtype=np.int32) if want_scores else None
        t0 = time.perf_counter()
        for strand, sel, a, b, c in parts:
            out = k.align_batch(band, batch, a, b, c, nuc_prior=2, nthreads=threads, strand_rev=strand)
            if want_scores:
                scores[sel] = out
        dt = time.perf_counter() - t0
        res = (cells / dt / 1e9, dt, "reference", "%s<%d,short> (%s build)" % (k.name(band), band, isa), cells)
        return res + (scores.reshape(n, H),) if want_scores else res
    from octopus_b200.batch import ReadBlock
    a = int(reads.off[n])
    sub = ReadBlock(reads.off[:n + 1], reads.bases[:a], reads.quals[:a], reads.mapq[:n], reads.reverse[:n], reads.begin[:n])
    o = COracle()
    t0 = time.perf_counter()
    o.populate(band, haps, sub, dp_only=True)
    dt = time.perf_counter() - t0
    res = (cells / dt / 1e9, dt, "port", "scalar C restatement", cells)
    return res + (None,) if want_scores else res


def sample_reads(reads, n):
    from octopus_b200.batch import ReadBlock
    n = min(n, reads.n)
    a = int(reads.off[n])
    return ReadBlock(reads.off[:n + 1], reads.bases[:a], reads.quals[:a], reads.mapq[:n], reads.reverse[:n], reads.begin[:n])


def parity_gate(eng, haps, reads, band, flank_state, shortcut, mapit, int_scores, ref_scores, n_ref):
    """BASELINE.md §3 "parity gate before any timing counts", inside the timed run's process. Headline mode: the reference SIMD
    kernel's INTEGER scores of the cpu_baseline sample (already computed) against the GPU's, recovered exactly from a second call on
    the same reads with mapping-quality mixing off (ln-likelihood = -ln10/10 * integer). Other modes: the GPU's ln-likelihoods of a
    small sample against the oracle's populate in the same mode (1e-4 relative, integers exact)."""
    from octopus_b200 import HaplotypeLikelihoodModel
    c = 0.230258509299404568401799145468436420760110148862877297603
    if ref_scores is not None and flank_state is None and not shortcut and not mapit:
        sub = sample_reads(reads, n_ref)
        cfg = HaplotypeLikelihoodModel.Config(max_indel_error=band, disable_naive_shortcut=True, map_positions=False, use_mapping_quality=False,
                                              use_int_scores=int_scores)
        lnl = eng.populate(cfg, haps, sub)                       # [H, n]
        got = np.rint(-lnl / c).astype(np.int64)
        exact = np.abs(-c * got - lnl) <= 1e-9 * np.maximum(1.0, np.abs(lnl))
        mism = int((got != ref_scores.T.astype(np.int64)).sum() + (~exact).sum())
        return {"pairs": int(got.size), "mismatches": mism, "against": "reference SIMD kernel, integer scores of the cpu_baseline sample"}
    from oracle.oracle import COracle
    sub = sample_reads(reads, 48)
    hs = haps
    if haps.n > 64:                                              # keep the scalar oracle's share of the run small
        from octopus_b200.batch import HaplotypeBlock
        e = int(haps.off[64])
        hs = HaplotypeBlock(haps.off[:65], haps.seq[:e], haps.snv_mask_fwd[:e], haps.snv_prior_fwd[:e], haps.snv_mask_rev[:e],
                            haps.snv_prior_rev[:e], haps.gap_open[:e], haps.gap_extend[:e], haps.begin[:64])
    cfg = HaplotypeLikelihoodModel.Config(max_indel_error=band, disable_naive_shortcut=not shortcut, map_positions=mapit, use_int_scores=int_scores)
    got, st = eng.populate(cfg, hs, sub, flank_state=flank_state, want_status=True)
    rc, want, wst = COracle().populate(band, hs, sub, None, flank_state, dp_only=not shortcut, map_positions=mapit)
    ok = wst == 0
    rel = np.abs(got[ok] - want[ok]) / np.maximum(np.abs(want[ok]), 1e-300)
    return {"pairs": int(ok.sum()), "mismatches": int((rel > 1e-4).sum() + (st[~ok] != wst[~ok]).sum()),
            "against": "oracle populate in the same mode (C restatement pinned to the compiled reference), 1e-4 relative"}


def measured_traffic(config, R, H, band, mode_key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed ncu --set full captures
    (profiles/traffic.json, written by tools/ncu_traffic.py from the .ncu-rep files); None when this workload was never captured."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)
        return t.get("%s:%d:%d:%d:%s" % (config, R, H, band, mode_key))
    except Exception:
        return None


def workload_name(config, R, lens, H, hap_len, band):
    return ("%s per GPU: %d reads (L=%s) x %d haplotypes (%d bp), band=%d, one mapping position per pair, "
            "naive shortcut disabled (every pair runs the DP), mapq mixing on, double [H][R] out" % (config, R, lens, H, hap_len, band))


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from octopus_b200 import synth
    cfg = synth.CONFIGS[args.config]
    threads = host_threads()
    # a bounded sample of the workload per step: sized so that the whole --steps/--warmup run takes about a minute
    haps, reads, band = synth.make_batch(args.config, n_reads=min(cfg["n_reads"], 200_000), n_haps=args.haps, ordered_penalties=not args.unordered_penalties)
    n_sample = args.cpu_sample_reads or calibrated_sample(haps, reads, band, threads, 60.0 / max(1, args.steps + args.warmup))
    for _ in range(max(1, args.warmup)):
        cpu_reference_run(haps, reads, band, n_sample, threads)
    t_total, cells_total, info = 0.0, 0, None
    for _ in range(args.steps):
        g, dt, kind, name, cells = cpu_reference_run(haps, reads, band, n_sample, threads)
        t_total += dt; cells_total += cells; info = (kind, name)
    value = cells_total / t_total / 1e9
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "GCUPS", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int16", "data": "synthetic",
            # the same workload as the GPU arm (same generator, shapes, band and mode); each step times a bounded sample of it
            "config": {"workload": workload_name(args.config, args.reads or cfg["n_reads"], "/".join(map(str, cfg["read_lens"])), haps.n, cfg["hap_len"], band),
                       "sample_reads_per_step": n_sample,
                       "mode": {"flank_state": None, "naive_shortcut": False, "kmer_mapper": False}},
            "cpu_baseline": {"value": value, "unit": "GCUPS", "cores": threads, "kind": info[0], "sample": "%d reads x %d haplotypes per step; %s" % (n_sample, haps.n, info[1])},
            "e2e": {"value": value, "unit": "GCUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
        return
    import torch
    import torch.distributed as dist
    from octopus_b200 import ErrorModel, HaplotypeLikelihoodModel, PairHMMEngine, shard, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    cfg = synth.CONFIGS[args.config]
    read_lens = tuple(int(x) for x in args.read_lens.split(",")) if args.read_lens else None
    strong = args.scaling == "strong" and world > 1
    n_regions = args.batch_regions or (args.regions if args.regions else (125 if args.config == "C5" else 1))

    def make_region(seed):
        h, r, b = synth.make_batch(args.config, n_reads=args.reads, n_haps=args.haps, seed=seed, band=args.band, hap_len=args.hap_len, read_lens=read_lens,
                                   ordered_penalties=not args.unordered_penalties)
        if args.error_model:       # penalty arrays as the reference's error models assign them (tandem-repeat structured), not i.i.d.
            h = ErrorModel(args.error_model).reset_block(h.off, h.seq, h.begin)
        return h, r, b

    # weak scaling: every rank owns its own batch(es) of the named shape (its own regions' reads and haplotypes);
    # strong scaling: ONE batch of the named shape, its reads split contiguously over the ranks, haplotypes replicated
    if strong:
        haps, all_reads, band = make_region(cfg["seed"])
        reads, (lo, hi) = shard.shard_reads(all_reads, world, rank)
        regions = [(haps, reads)]
        R_total = all_reads.n
        cells_rank_total = synth.total_cells(haps, all_reads, band)          # the whole job's cells (all ranks together)
    else:
        regions = []
        for g in range(n_regions):
            h, r, band = make_region(cfg["seed"] + 1000 * rank + 7919 * g)
            regions.append((h, r))
        haps, reads = regions[0]
        cells_rank_total = sum(synth.total_cells(h, r, band) for h, r in regions) * world
    H, R = haps.n, reads.n
    model_cfg = HaplotypeLikelihoodModel.Config(max_indel_error=band, disable_naive_shortcut=not args.shortcut, map_positions=args.map,
                                                use_int_scores=args.int_scores)
    flank_state = tuple(int(x) for x in args.flank.split(",")) if args.flank else None
    eng = PairHMMEngine(local)
    reserve = args.reserve_sms
    eng.reserve_sms(reserve)
    d_regions = [(h.to_device(dev), r.to_device(dev)) for h, r in regions]
    # Several ranks: the values have to end up on rank 0.
    #   --gather peer (default): rank 0 owns a ring of result slots mapped into every rank (CUDA IPC); each rank's epilogue kernel
    #     stores its slab — its columns of the [H, R_total] matrix (strong) or its [H, R] matrix of the per-rank stack (weak) —
    #     straight into rank 0's HBM over NVLink; one barrier per step tells rank 0 the step has landed (octopus_b200/peer.py).
    #   --gather nccl: a ring of local output buffers and an NCCL gather per step, asynchronous on torch's stream; before a buffer is
    #     re-used the engine waits (on the device) for the event recorded after its gather.
    n_buf = 3 if world > 1 else 1
    peer_ring = None
    max_region_bytes = max(h.n * r.n for h, r in regions) * 8
    gather_note = None
    if world > 1 and args.gather == "peer":
        from octopus_b200.peer import PeerRing
        slot_bytes = H * R_total * 8 if strong else world * max_region_bytes
        try:
            peer_ring = PeerRing(slot_bytes, local, rank, world, n_buf=n_buf)
            ok = 1
        except (RuntimeError, MemoryError) as exc:       # no peer access between these GPUs / IPC refused in this container
            peer_ring, ok, gather_note = None, 0, str(exc)
        flag = torch.tensor([ok], dtype=torch.int32, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)      # all ranks take the same path
        if int(flag.item()) == 0:
            if peer_ring is not None:
                peer_ring.close()
                peer_ring = None
            gather_note = "peer mapping unavailable on some rank (%s): NCCL gather instead" % (gather_note or "another rank")
            sys.stderr.write(gather_note + "\n")
    gather_buffers = [dict() for _ in range(n_buf)]
    d_out = [torch.empty((H, R), dtype=torch.float64, device=dev) for _ in range(n_buf)] if peer_ring is None else None
    gather_done = [None] * n_buf
    recv = None
    if world > 1 and rank == 0 and not strong and peer_ring is None:
        recv = [[torch.empty_like(d_out[0]) for _ in range(world)] for _ in range(n_buf)]
    state = {"k": 0, "gather_ms": [], "launches": 0, "keep": None}

    def keep(out, reused=False):
        """--dump-outputs: hold what the last timed step returned. A buffer that a later region of the step writes again is
        copied first, and the engine's stream waits for the copy."""
        if state["keep"] is None:
            return
        if reused:
            out = out.clone()
            ev = torch.cuda.Event()
            ev.record()
            eng.wait_event(ev)
        state["keep"].append(out)

    def one_region(dh, dr):
        k = state["k"]
        b = k % n_buf
        state["k"] += 1
        if peer_ring is not None:
            peer_ring.wait_slot(eng, k)
            if strong:
                lo, _ = shard.split_range(R_total, world, rank)
                out = peer_ring.window(k, lo * 8, dh.n, dr.n, ld=R_total)
            else:
                out = peer_ring.window(k, rank * max_region_bytes, dh.n, dr.n)
            eng.populate(model_cfg, dh, dr, flank_state=flank_state, out=out)
            keep(out, reused=len(d_regions) > 1)
            dp = eng.last_dp_kernel_ms()
            state["launches"] += eng.launch_count()
            g0 = torch.cuda.Event(enable_timing=True)
            g0.record()
            g1 = peer_ring.publish(k)
            state["gather_ms"].append((g0, g1))        # here: the barrier alone (the stores are part of the populate call)
            return dp
        if gather_done[b] is not None:
            eng.wait_event(gather_done[b])
        out = d_out[b] if (dh.n, dr.n) == (H, R) else None
        out = eng.populate(model_cfg, dh, dr, flank_state=flank_state, out=out)
        keep(out, reused=len(d_regions) > 1)
        dp = eng.last_dp_kernel_ms()
        state["launches"] += eng.launch_count()
        if world > 1:
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            if strong:
                shard.gather_likelihoods(out, R_total, world, rank, buffers=gather_buffers[b])   # the [H, R_total] matrix re-assembled on rank 0
            else:
                shard.gather_slabs(out, world, rank, recv=recv[b] if recv else None)   # per-rank matrices straight into rank 0's slabs
            g1.record()
            gather_done[b] = g1
            state["gather_ms"].append((g0, g1))
        return dp

    batched = None
    if args.batch_regions:
        from octopus_b200.batch import concat_blocks
        bh, br, hf, rf = concat_blocks([h for h, r in regions], [r for h, r in regions])
        batched = (bh.to_device(dev), br.to_device(dev), hf, rf, bh, br)
        flat_out = torch.empty(int(sum(h.n * r.n for h, r in regions)), dtype=torch.float64, device=dev)

    def step():
        if batched is not None:
            _, off = eng.populate_regions(model_cfg, batched[0], batched[1], batched[2], batched[3],
                                          flank_states=[flank_state] * len(regions) if flank_state else None, out=flat_out)
            state["launches"] += eng.launch_count()
            for m in PairHMMEngine.split_regions(flat_out, off, batched[2], batched[3]):
                keep(m)
            return eng.last_dp_kernel_ms()
        return sum(one_region(dh, dr) for dh, dr in d_regions)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(local)
    sync_all()
    state["gather_ms"] = []
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dp_ms = []
    state["launches"] = 0
    sync_all()
    ev0.record()
    for i in range(args.steps):
        if args.dump_outputs and rank == 0 and i == args.steps - 1:
            state["keep"] = []
        dp_ms.append(step())
    ev1.record()
    launches = state["launches"]
    sync_all()
    ms = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    total_ms = float(ms.item())
    gather_ms = float(np.mean([a.elapsed_time(b) for a, b in state["gather_ms"]])) if state["gather_ms"] else 0.0
    clocks = sampler.stop() if rank == 0 else None
    kept, state["keep"] = state["keep"], None
    if kept:
        dump_outputs(args.dump_outputs, [("likelihoods" if len(kept) == 1 else "likelihoods_region%04d" % g, t) for g, t in enumerate(kept)])

    # Did every rank's values land on rank 0? Each rank recomputes its last region locally; rank 0 compares an order-independent bit
    # digest (int64 sum of the float64 bit patterns) of every rank's window of the last slot with that rank's own digest.
    gather_check = None
    if peer_ring is not None:
        k_last = state["k"] - 1
        dh, dr = d_regions[-1]
        mine = eng.populate(model_cfg, dh, dr, flank_state=flank_state)
        dig = torch.stack([mine.view(torch.int64).sum(), torch.tensor(dh.n, device=dev), torch.tensor(dr.n, device=dev)]).to(torch.int64)
        digs = [torch.zeros_like(dig) for _ in range(world)] if rank == 0 else None
        dist.gather(dig, digs, dst=0)
        if rank == 0:
            torch.cuda.synchronize()
            bad = 0
            for k in range(world):
                want, rows, cols = (int(x) for x in digs[k].tolist())
                if strong:
                    lo, hi = shard.split_range(R_total, world, k)
                    win = peer_ring.owner_slot(k_last, (H, R_total))[:, lo:hi].contiguous()
                else:
                    win = peer_ring.owner_slot(k_last, (rows, cols), byte_offset=k * max_region_bytes)
                bad += int(tuple(win.shape) != (rows, cols) or int(win.view(torch.int64).sum().item()) != want)
            gather_check = {"ranks_checked": world, "ranks_mismatched": bad,
                            "what": "bit digest of every rank's window of rank 0's last result slot vs the rank's own recomputation"}
        sync_all()

    # e2e: the same call through the C ABI with pinned HOST buffers: H2D of the batch and D2H of the matrix inside the timed region
    # (and, with several ranks, the gather of the host matrices' device copies is replaced by each rank's own D2H: the per-rank
    # results land in host memory of the rank that computed them)
    p_regions = [(h.pin(), r.pin()) for h, r in regions]
    p_out_t = torch.empty((H, R), dtype=torch.float64).pin_memory()
    p_out = p_out_t.numpy()

    p_batched = (batched[4].pin(), batched[5].pin()) if batched is not None else None
    p_flat = torch.empty(int(sum(h.n * r.n for h, r in regions)), dtype=torch.float64).pin_memory().numpy() if batched is not None else None

    def e2e_step():
        if batched is not None:
            eng.populate_regions(model_cfg, p_batched[0], p_batched[1], batched[2], batched[3],
                                 flank_states=[flank_state] * len(regions) if flank_state else None, out=p_flat)
            return
        for ph, pr in p_regions:
            eng.populate(model_cfg, ph, pr, flank_state=flank_state, out=p_out if (ph.n, pr.n) == (H, R) else None)

    for _ in range(2):
        e2e_step()
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        e2e_step()
    e1.record()
    sync_all()
    ems = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ems, op=dist.ReduceOp.MAX)
    e2e_ms = float(ems.item())
    h2d = sum(sum(int(a.nbytes) for a in h.arrays().values()) + sum(int(a.nbytes) for a in r.arrays().values()) for h, r in regions)
    d2h = sum(h.n * r.n * 8 for h, r in regions)

    if rank == 0:
        value = cells_rank_total * args.steps / (total_ms / 1e3) / 1e9
        e2e = cells_rank_total * args.steps / (e2e_ms / 1e3) / 1e9
        kernel_ms = float(np.mean(dp_ms))                      # DP kernel time per step on this rank (all its regions)
        cells_rank = sum(synth.total_cells(h, r, band) for h, r in regions)
        # algorithmic HBM bytes of the dominant DP kernel per step, SURVEY.md §8(d): 4 B per pair (integer score out) + the read row
        # half-words (2 B per read base, read once per read pair) + both strand column tables (16 B per haplotype base)
        alg_bytes = sum(4 * h.n * r.n + 2 * int(r.off[-1]) + 16 * int(h.off[-1]) for h, r in regions)
        peak, peak_src = peaks()
        achieved = alg_bytes / (kernel_ms / 1e3) / 1e9
        mode_key = "flank" if flank_state else ("ref" if (args.shortcut or args.map) else "dp")
        traffic = measured_traffic(args.config, R, H, band, mode_key)
        role_warps = band in (32, 64) and H >= 17 and not os.environ.get("PHMM_NO_ROLE_WARPS")     # the engine's own rule (populate_impl)
        flank_fb = band <= 16 and not args.int_scores and not os.environ.get("PHMM_NO_FLANK_FB")          # the engine's own rule (populate_impl)
        kernel_name = ("k_flank_fwd<%d> + k_flank_bwd<%d> (+ score-only and labelled flank kernels of the tile)" % (band, band)) if flank_state and flank_fb else \
                      ("k_populate_flank_acc<%d> (+ score-only and crossing-cell flank kernels of the tile)" % band) if flank_state and band <= 32 else \
                      ("k_populate_wide (32-bit lanes, band %d)" % band) if args.int_scores else \
                      ("k_populate_roles<%d> (one warp per 32 diagonals)" % band) if role_warps else "k_populate_fast<%d>" % band
        how = "none: one rank" if world == 1 else ("peer stores: every rank's epilogue kernel writes into rank 0's HBM through a CUDA IPC mapping, one barrier per step"
                                                   if peer_ring is not None else "NCCL gather per step, overlapped with the next step's compute")
        line = {
            "metric": METRIC, "value": value, "unit": "GCUPS", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": "int32" if args.int_scores else "int16", "data": "synthetic",
            "config": {"workload": workload_name(args.config, R, (args.read_lens or "/".join(map(str, cfg["read_lens"]))).replace(",", "/"), H, args.hap_len or cfg["hap_len"], band),
                       "regions_per_rank_and_step": len(regions), "regions_per_call": len(regions) if args.batch_regions else 1,
                       "alignments_per_step": haps.n * R_total if strong else sum(h.n * r.n for h, r in regions) * world,
                       "cells_per_step": cells_rank_total,
                       "l2": "inputs+outputs (%.0f MB) larger than the 126 MB L2" % ((h2d + d2h + 4 * H * R) / 1e6),
                       "parallelism": ("one batch, reads split over %d rank(s), [H, R_total] matrix assembled on rank 0 (%s)" % (world, how)) if strong else
                                      ("every rank its own region(s), haplotypes per region, the per-rank matrices collected on rank 0 (%d rank(s), %s)" % (world, how)),
                       "gather": (None if world == 1 else ("peer" if peer_ring is not None else "nccl")), "gather_note": gather_note,
                       "reserved_sms": reserve,
                       "penalties": args.error_model or ("i.i.d. draws from the error-model tables' value range" +
                                                         (", gap_extend unconstrained (general deletion update)" if args.unordered_penalties else
                                                          ", gap_extend capped at gap_open as in every short-read error model")),
                       "mode": {"flank_state": flank_state, "naive_shortcut": bool(args.shortcut), "kmer_mapper": bool(args.map), "use_int_scores": bool(args.int_scores)}},
            "e2e": {"value": e2e, "unit": "GCUPS", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / args.steps},
            "gpu_launches": launches,
            "clocks": clocks,
            "gather_ms_per_region": gather_ms,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "peak_source": peak_src, "kernel": kernel_name, "kernel_ms": kernel_ms,
                         "algorithmic_bytes_per_launch": alg_bytes,
                         "note": "the path is integer-issue bound, not HBM bound (SURVEY.md F3); see DESIGN.md for the issue-rate roofline",
                         "kernel_gcups": cells_rank / (kernel_ms / 1e3) / 1e9},
            # The binding roofline (DESIGN.md §4): the packed cell costs 5 (6 for unordered penalties) ALU-pipe instructions per 2 cells
            # and the ALU pipe issues 64 thread-instructions/clk/SM (profiles/r01_ubench_int.txt).
            "issue_roofline": issue_roofline(cells_rank / (kernel_ms / 1e3) / 1e9, reads, band, clocks,
                                             5 if all(bool((np.asarray(h.gap_open) >= np.asarray(h.gap_extend)).all()) for h, _ in regions) else 6),
        }
        ref_scores, n_ref = None, 0
        if not args.no_cpu_baseline:
            threads = host_threads()
            n_sample = args.cpu_sample_reads or calibrated_sample(haps, reads, band, threads, 12.0)
            g, dt, kind, name, _, ref_scores = cpu_reference_run(haps, reads, band, n_sample, threads, want_scores=True)
            n_ref = n_sample
            line["cpu_baseline"] = {"value": g, "unit": "GCUPS", "cores": threads, "kind": kind,
                                    "sample": "first %d reads x %d haplotypes of the same batch, %.1f s; %s" % (n_sample, H, dt, name)}
            # BASELINE.md §3: one thread, and the AVX2-forced build next to what -march=native selects (they differ for band 32 on AVX-512 hosts)
            from oracle.oracle import available_ref_isas
            variants = {}
            n1 = max(64, n_sample // (4 * max(1, threads)))
            variants["1_thread"] = {"value": cpu_reference_run(haps, reads, band, n1, 1)[0], "sample_reads": n1}
            for isa in available_ref_isas():
                v = cpu_reference_run(haps, reads, band, max(64, n_sample // 4), threads, isa=isa)
                variants["%s_build_all_threads" % isa] = {"value": v[0], "kernel": v[3]}
            line["cpu_baseline"]["variants"] = variants
        if gather_check is not None:
            line["gather_check"] = gather_check
            if gather_check["ranks_mismatched"]:
                sys.stderr.write("GATHER CHECK FAILED: %r\n" % (gather_check,))
        line["parity"] = parity_gate(eng, haps, reads, band, flank_state, args.shortcut, args.map, args.int_scores, ref_scores, n_ref)
        print(json.dumps(line))
        if line["parity"]["mismatches"]:
            sys.stderr.write("PARITY GATE FAILED: %r\n" % (line["parity"],))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
