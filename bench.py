#!/usr/bin/env python
"""bench.py -- POA windows/sec of the B200-native engine (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torchrun, one rank per GPU)
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   (+ the last timed step's results, see dump_outputs)
    python bench.py --impl reference --gpus N --steps K --warmup W

Headline workload (config.workload): BASELINE.json configs[1] -- "single B200: 10k windows, 500 bp x 32 reads,
15% ONT error, banded width 256" -- synthetic windows (racon_gpu_b200/windows.py, SURVEY.md 8d), per GPU (weak
scaling).  One step = one pass of the hot path over the whole batch of windows.

  value      windows/s, whole job, inputs ALREADY RESIDENT IN HBM: K back-to-back launches of the POA
             kernel timed with CUDA events on the launching stream, max over ranks.
  e2e        the same metric through the public host API (api.Polisher.polish == racon's GPU window
             scheduler) with HOST buffers: pinned staging + H2D + kernel + D2H + coverage trim every
             step (+ the NCCL gather of the consensus to rank 0 when N > 1, overlapped with the next step).
  roofline   the DP-fill kernel against the measured HBM peak: algorithmic bytes = DP cells
             x 2 B x 2 (one write + one read), SURVEY.md 8(d) / BASELINE.md 4.
  cpu_baseline  the reference's own CPU path (oracle/_ref: racon::Window + spoa AVX2) timed on this
             box's host cores over a bounded sample of the same windows (rank 0, N=1).
  extra      (N=1 only, outside the headline timing) the overlap aligner (SURVEY 8f-4) on real overlaps, and
             the same measurements for BASELINE configs[2]
             (A_full: full band, the bit-exact mode) and configs[4]'s shape (B_banded: 1024 bp x 64 reads, 12 %,
             band 256, max_sequence_size 1279), and the headline workload with the MSA output switched on.

`--impl reference` times that CPU path as the job itself (all usable host threads, bounded sample per step).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

M, X, G = 3, -5, -4
WORKLOADS = {
    # name: (windows per GPU, backbone length, reads per window, error rate, banded, max_sequence_size, BASELINE.json configs[i])
    "A_banded": (10000, 500, 32, 0.15, True, 1023, 1),   # headline
    "A_full": (10000, 500, 32, 0.15, False, 1023, 2),
    "B_banded": (4096, 1024, 64, 0.12, True, 1279, 4),   # long-window stress shape
    "C_small": (100, 500, 8, 0.05, False, 1023, 0),
    # BASELINE configs[3] per GPU: 1M windows over 8 GPUs, cudapoa-batches=8 -> 125k windows and 8 batch processors per GPU
    "A_banded_1M": (125000, 500, 32, 0.15, True, 1023, 3),
}


def usable_cores():
    """Host cores this process can actually run on: scheduler affinity AND the cgroup CPU quota (a 1-GPU lease of
    a 128-thread host is a cgroup slice; os.cpu_count() reports the whole host)."""
    aff = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    try:  # cgroup v2
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            quota = float(q) / float(p)
    except (OSError, ValueError):
        try:  # cgroup v1
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / p
        except (OSError, ValueError):
            pass
    eff = aff if quota is None else max(1, min(aff, int(quota + 0.5)))
    return eff, {"os_cpu_count": os.cpu_count(), "sched_affinity": aff, "cgroup_quota": quota}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index: int):
        self.index, self.rows, self.proc, self.thr = index, [], None, None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            return
        self.thr = threading.Thread(target=self._read, daemon=True)
        self.thr.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.thr.join(timeout=2)
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower() == "active"})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def measured_hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def recorded_traffic(workload: str, nwin: int):
    """DRAM bytes per launch of `nwin` windows, scaled from the committed `ncu --set full` capture of this workload
    (profiles/traffic.json).  A constant from a profile, not a per-run measurement: see traffic_source."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(path):
        rec = json.load(open(path))
        if workload in rec and isinstance(rec[workload], dict):
            r = rec[workload]
            return float(r["dram_bytes_per_launch"]) * nwin / float(r["windows_per_launch"]), r.get("source")
    return None, None


def cpu_reference_rate(batch, L, seconds_target, threads, core_info):
    """Times the reference's CPU path on a bounded sample; returns the cpu_baseline dict."""
    from oracle_lib import Oracle, Ref
    ref = Ref()
    est = 40.0 * threads * (500.0 / L) ** 2  # windows/s guess (SURVEY.md 6: ~50 windows/s/thread on config A)
    n = int(max(threads * 2, min(batch.n_windows, seconds_target * est)))
    sample = batch.slice(0, n)
    t0 = time.perf_counter()
    if ref.available:
        ref.polish(sample, M, X, G, tgs=True, trim=True, threads=threads, window_length=L)
        kind = "reference"
    else:  # the restatement, when oracle/_ref did not travel
        from racon_gpu_b200 import api
        Oracle().polish(sample, api.processing_order(sample), M, X, G, tgs=True, trim=True, threads=threads)
        kind = "port"
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": "windows/s", "cores": threads, "kind": kind, "host": core_info,
            "sample": f"first {n} windows of the workload, {dt:.1f} s, racon::Window::generate_consensus + spoa "
                      f"(kNW {M}/{X}/{G}, unbanded), one engine per thread, {threads} threads = usable cores"}


def algorithmic_bytes_per_window(batch, banded, sample=48):
    """SURVEY.md 8(d): sum over reads of rows x cols DP cells (rows from the oracle's trace) x 2 B x 2."""
    from oracle_lib import Oracle
    from racon_gpu_b200 import api
    sub = batch.slice(0, min(sample, batch.n_windows))
    _, _, _, st = Oracle().polish(sub, api.processing_order(sub), M, X, G, tgs=False, trim=False,
                                  threads=min(16, usable_cores()[0]), want_stats=True)
    cells = st[:, 4].mean() if banded else st[:, 2].mean()
    return float(cells) * 4.0, float(cells)


def workload_label(name, nwin):
    _, L, D, err, banded, max_seq, cfg = WORKLOADS[name]
    return (f"{name}: {nwin} windows per GPU, {L} bp x {D} reads, {err:.0%} error, "
            f"{'static band 256' if banded else 'full band'}, m{M}/x{X}/g{G}, max_sequence_size {max_seq} "
            f"(BASELINE.json configs[{cfg}]{' shape' if name == 'B_banded' else ''})")


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path as the job itself."""
    if rank != 0:
        return
    from racon_gpu_b200.windows import synth_windows
    nwin, L, D, err, banded, _, _ = WORKLOADS[args.workload]
    threads, core_info = usable_cores()
    per_step = int(max(threads * 2, min(nwin, 6.0 * 40.0 * threads * (500.0 / L) ** 2)))  # ~6 s of CPU work per step
    batch = synth_windows(per_step, L, D, err, seed=args.seed)
    from oracle_lib import Oracle, Ref
    ref = Ref()

    def step():
        if ref.available:
            ref.polish(batch, M, X, G, tgs=True, trim=True, threads=threads, window_length=L)
        else:
            from racon_gpu_b200 import api
            Oracle().polish(batch, api.processing_order(batch), M, X, G, tgs=True, trim=True, threads=threads)
    for _ in range(min(args.warmup, 1)):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    value = per_step * args.steps / dt
    print(json.dumps({
        "impl": "reference", "metric": "POA windows/sec", "value": value, "unit": "windows/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": min(args.warmup, 1), "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int16", "data": "synthetic",
        "config": {"workload": f"{args.workload}: {L} bp x {D} reads, {err:.0%} error, m{M}/x{X}/g{G}; CPU path is unbanded "
                               f"(spoa has no band); bounded sample of {per_step} windows per step"},
        "cpu_baseline": {"value": value, "unit": "windows/s", "cores": threads, "host": core_info,
                         "kind": "reference" if ref.available else "port",
                         "sample": f"{per_step} windows per step x {args.steps} steps, {threads} threads = usable cores"},
        "e2e": {"value": value, "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def measure(name, args, rank, world, local_rank, device, steps, warmup, nwin=None, sample_clocks=True, keep_outputs=False):
    """Kernel-only and end-to-end legs of one workload on this rank.  Returns a dict of per-rank raw numbers (and, with
    keep_outputs, what each leg's last timed step returned)."""
    import torch
    import torch.distributed as dist
    from racon_gpu_b200 import api
    from racon_gpu_b200.shard import ConsensusGather
    from racon_gpu_b200.windows import synth_windows

    nwin0, L, D, err, banded, max_seq, _ = WORKLOADS[name]
    nwin = nwin or nwin0
    if nwin * (D + 1) * L > (1 << 30):  # the 1M-window configuration: more pinned staging than the 3 GiB default
        os.environ.setdefault("B200POA_MAX_STAGING_MB", str(int(nwin * (D + 1) * L * 4.5) >> 20))
    batch = synth_windows(nwin, L, D, err, seed=args.seed + 1000003 * rank)  # each rank its own windows

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    free_b, _ = torch.cuda.mem_get_info()
    mem = int(min(0.6 * free_b, 64 << 30))

    # ---------------- value: kernel with inputs resident in HBM -------------------------------------
    stream = torch.cuda.Stream(device=device)
    pb = api.PoaBatch(device=local_rank, stream=stream.cuda_stream, max_gpu_mem=mem, banded=banded,
                      gap=G, mismatch=X, match=M, max_sequence_size=max_seq)
    n_added, _ = pb.add_windows(batch)
    if n_added != nwin:
        raise SystemExit(f"bench.py: batch accepted {n_added}/{nwin} windows; raise the memory budget")
    pb.upload()
    info = pb.info()
    sampler = ClockSampler(local_rank)
    if sample_clocks:
        sampler.start()  # started before the warm-up: nvidia-smi needs ~1 s to deliver its first sample
    with torch.cuda.stream(stream):
        for _ in range(warmup):
            pb.launch()
        barrier()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        t0 = time.perf_counter()
        for a, b in ev:
            a.record(stream)
            pb.launch()
            b.record(stream)
        barrier()
        wall = time.perf_counter() - t0
        clocks = sampler.stop() if sample_clocks else None
    dev_ms = float(sum(a.elapsed_time(b) for a, b in ev))
    pb.download()
    cons_k, cov_k, status_k = pb.get_consensus()
    n_fail = int((status_k != 0).sum())
    pb.close()

    # ---------------- e2e: host buffers through the public API -------------------------------------
    pol = api.Polisher(devices=[local_rank], batches_per_device=args.batches, mem_per_batch=mem // args.batches,
                       banded=banded, match=M, mismatch=X, gap=G, max_sequence_size=max_seq)
    chunk = max(256, int(-(-nwin // (args.batches * args.rounds))))  # windows per launch of a batch processor
    stride = 2 * max_seq + 2
    bufs = [None, None]  # double-buffered outputs: step k's gather overlaps step k+1's polish
    gather = ConsensusGather(device, nwin) if world > 1 else None
    # the windows as racon's Polisher::initialize would leave them for the GPU path: a columnar arena in pinned host
    # memory (b200poa_arena_*; built once, outside the timed region, like window construction upstream of the hot path)
    arena = api.WindowArena.from_batch(batch)
    for k in range(warmup):
        out_t = pol.polish_arena(arena, tgs=True, trim=True, max_windows_per_round=chunk, stride=stride, out=bufs[k % 2])
        bufs[k % 2] = (out_t[0], out_t[1], out_t[2].astype(np.uint8), out_t[3])
        if gather:
            gather.start(out_t[0], out_t[1])
            gather.wait()
    barrier()
    t0 = time.perf_counter()
    e2e_launches = 0
    for k in range(steps):
        cons, clen, polished, status = pol.polish_arena(arena, tgs=True, trim=True, max_windows_per_round=chunk,
                                                        stride=stride, out=bufs[k % 2])
        e2e_launches += pol.last["kernel_launches"]
        if gather:
            gather.wait()           # the previous step's consensus is on rank 0 (pinned host memory) ...
            gather.start(cons, clen)  # ... this step's travels while the next one is computed
    if gather:
        gather.wait()
    barrier()
    e2e_s = time.perf_counter() - t0
    h2d, d2h = pol.last["h2d_bytes"], pol.last["d2h_bytes"]
    n_unpolished = int((~polished).sum())
    pol.close()
    arena.close()
    out = {"batch": batch, "nwin": nwin, "L": L, "banded": banded, "info": info, "dev_ms": dev_ms, "e2e_s": e2e_s,
           "wall": wall, "failures": n_fail + n_unpolished, "h2d": h2d, "d2h": d2h, "clocks": clocks,
           "launches": steps + warmup + e2e_launches, "timed_launches": steps + e2e_launches}
    if keep_outputs:
        out["outputs"] = {"kernel": (cons_k, cov_k, status_k), "e2e": (cons, clen, polished, status)}
    return out


DUMP_BYTES = 63_000_000  # data of all --dump-outputs files; the .npy headers stay within 64 MB with it


def dump_outputs(out_dir, outputs):
    """--dump-outputs: the results of the last timed step as float32 .npy files.  Kernel leg (the headline `value`):
    what PoaBatch.get_consensus returns -- untrimmed consensus, its per-base coverage, status per window.  e2e leg: what
    Polisher.polish_arena returns -- trimmed consensus, polished flag, status per window.  Consensus and coverage are
    concatenated over windows, with the lengths beside them.  When the worst case of all windows (every consensus as
    long as the output stride) would exceed DUMP_BYTES, a fixed seeded sample of windows is written (window_index)."""
    cons_k, cov_k, status_k = outputs["kernel"]
    cons_e, clen_e, polished_e, status_e = outputs["e2e"]
    nwin, stride = len(cons_k), cons_e.shape[1]
    per_window = 4 * (3 * stride + 6)
    idx = np.arange(nwin)
    if nwin * per_window > DUMP_BYTES:
        idx = np.sort(np.random.default_rng(0).choice(nwin, DUMP_BYTES // per_window, replace=False))
    arrays = {
        "window_index": idx,
        "consensus": np.frombuffer(b"".join(cons_k[i] for i in idx), dtype=np.uint8),
        "consensus_length": np.asarray([len(cons_k[i]) for i in idx]),
        "coverage": np.concatenate([cov_k[i] for i in idx]),
        "status": status_k[idx],
        "e2e_consensus": np.concatenate([cons_e[i, :clen_e[i]] for i in idx]),
        "e2e_consensus_length": clen_e[idx],
        "e2e_polished": polished_e[idx],
        "e2e_status": status_e[idx],
    }
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float32))


def measure_msa(args, local_rank, device, steps=3, warmup=3):
    """extra: the headline workload with OutputType::msa added to the output mask (Batch::get_msa): kernel rate with the
    inputs resident, and the bytes / time of the compact MSA download."""
    import torch
    from racon_gpu_b200 import api
    from racon_gpu_b200.windows import synth_windows
    nwin, L, D, err, banded, max_seq, _ = WORKLOADS["A_banded"]
    batch = synth_windows(nwin, L, D, err, seed=args.seed)
    free_b, _ = torch.cuda.mem_get_info()
    stream = torch.cuda.Stream(device=device)
    pb = api.PoaBatch(device=local_rank, stream=stream.cuda_stream, max_gpu_mem=int(min(0.6 * free_b, 64 << 30)),
                      banded=banded, gap=G, mismatch=X, match=M, max_sequence_size=max_seq,
                      output_mask=api.OUTPUT_CONSENSUS | api.OUTPUT_MSA)
    n_added, _ = pb.add_windows(batch)
    pb.upload()
    with torch.cuda.stream(stream):
        for _ in range(warmup):
            pb.launch()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(steps):
            pb.launch()
        b.record(stream)
        torch.cuda.synchronize()
    ms = a.elapsed_time(b) / steps
    pb.download()
    t0 = time.perf_counter()
    msa, status = pb.get_msa()
    dt = time.perf_counter() - t0
    ok = [m for m in msa if m is not None]
    msa_bytes = sum(len(m) * len(m[0]) for m in ok)
    pb.close()
    return {"workload": workload_label("A_banded", n_added) + " + OutputType::msa", "steps": steps, "warmup": warmup,
            "value": n_added / (ms / 1e3), "unit": "windows/s", "ms_per_step": ms, "windows": n_added,
            "failed_windows": int((status != 0).sum()), "msa_bytes_per_window": msa_bytes / max(len(ok), 1),
            "msa_d2h_and_unpack_s": dt,
            "note": "kernel with consensus + MSA, inputs resident; the MSA download moves exactly the bytes produced"}


def measure_aligner(args, local_rank, rep=32, steps=3, warmup=2, cpu_seconds=6.0):
    """extra: the overlap alignment step before the POA path (SURVEY 8f-4, CUDABatchAligner; include/b200aln.h) on REAL
    overlaps -- the 181 read-to-contig overlaps of the reference's lambda-phage test data (tests/golden/lambda_overlaps.npz,
    1.4-11 kb, cut like src/overlap.cpp:186-199), replicated `rep` times.  e2e = host buffers in, CIGAR bytes out through
    the C ABI (staging, H2D, all launches, D2H); kernel = distance-matrix cells computed / device time of the launches."""
    from concurrent.futures import ThreadPoolExecutor
    from common import overlap_fixture
    from racon_gpu_b200.aligner import AlignerPool, CUDABatchAligner, pack_pairs, pinned
    fx = overlap_fixture()
    pairs = [(f["q"], f["t"]) for f in fx] * rep
    q, qo, t, to = pack_pairs(pairs)
    matrix = float(sum(len(x) * len(y) for x, y in pairs))
    # kernel leg: one batch, device time of its launches (CUDA events inside the library)
    al = CUDABatchAligner(device_id=local_rank, max_gpu_memory=32 << 30)
    recs = []
    for it in range(warmup + steps):
        first, rec, eds = 0, {"kernel_ms": 0.0, "cells": 0, "h2d": 0, "d2h": 0, "launches": 0, "team_launches": 0, "batches": 0}, []
        while first < len(pairs):
            first += al.add_overlaps(q, qo, t, to, first)
            al.align_all()
            text, off, ln, ed = al.cigars()
            info = al.info()
            al.reset()
            eds.append(ed)
            for k, kk in (("kernel_ms", "kernel_ms"), ("cells", "cells"), ("h2d", "h2d_bytes"), ("d2h", "d2h_bytes"),
                          ("launches", "kernel_launches"), ("team_launches", "team_launches")):
                rec[k] += info[kk]
            rec["batches"] += 1
            rec["slots"], rec["levels"] = info["n_slots"], info["levels"]
        if it == 0 and [int(x) for x in np.concatenate(eds)[:len(fx)]] != [f["score"] for f in fx]:
            raise RuntimeError("aligner: edit distances differ from the committed edlib results")
        if it >= warmup:
            recs.append(rec)
    al.close()
    # e2e leg: the pool (three batches on the device, a host thread each, like racon --cudaaligner-batches 3): host buffers in,
    # CIGAR bytes out, staging / H2D / D2H of one batch under the other's kernels
    pool = AlignerPool(devices=(local_rank,), batches_per_device=3, max_gpu_memory_per_batch=20 << 30)
    walls = []
    with pinned(q, t):  # the caller's segment buffers are page-locked once (like the POA arena at finalize); every step
        for it in range(warmup + steps):  # uploads from them, runs all launches and brings the CIGAR bytes back
            t0 = time.perf_counter()
            ed, buf, off, ln, pinfo = pool.align(q, qo, t, to)
            dt = time.perf_counter() - t0
            if it == 0 and [int(x) for x in ed[:len(fx)]] != [f["score"] for f in fx]:
                raise RuntimeError("aligner pool: edit distances differ from the committed edlib results")
            if it >= warmup:
                walls.append(dt)
    pool.close()
    for r in recs:
        r["wall_s"] = sum(walls) / len(walls)
    wall = sum(r["wall_s"] for r in recs) / len(recs)
    kms = sum(r["kernel_ms"] for r in recs) / len(recs)
    r0 = recs[0]
    sm_mhz = 1965.0
    peak = 148 * 4 * sm_mhz * 1e6 / (2.0 * 24.0) * 2048.0  # see DESIGN.md section 11: ALU pipe, 24 instructions a step
    out = {"workload": f"real lambda-phage overlaps x{rep}: {len(pairs)} pairs, {int(qo[-1] + to[-1])} bases, "
                       f"{matrix:.3g} matrix cells, unit-cost NW with path (edlib's alignment, bit-exact)",
           "steps": steps, "warmup": warmup, "unit": "overlaps/s",
           "e2e": len(pairs) / wall, "value": len(pairs) / (kms / 1e3), "ms_per_step": kms, "e2e_ms_per_step": wall * 1e3,
           "matrix_gcups_e2e": matrix / wall / 1e9, "h2d_bytes_per_step": r0["h2d"], "d2h_bytes_per_step": r0["d2h"],
           "gpu_launches_per_step": r0["launches"], "team_launches_per_step": r0["team_launches"], "levels": r0["levels"],
           "resident_warps": r0["slots"], "batches_per_step": r0["batches"],
           "e2e_api": "b200aln_aligner_align: 3 batches on the device, one host thread each (racon --cudaaligner-batches 3), "
                      "segments in page-locked host buffers, uploaded without a staging copy",
           "roofline": {"bound": "alu", "achieved": r0["cells"] / (kms / 1e3) / 1e9, "peak": peak / 1e9, "unit": "Gcell/s",
                        "frac": r0["cells"] / (kms / 1e3) / peak, "traffic": None,
                        "kernel": "aln_split_kernel / aln_split_team_kernel / aln_leaf_kernel (all launches of a step)",
                        "cells_computed_per_step": r0["cells"],
                        "peak_source": "148 SMs x 4 schedulers x 1965 MHz / (24 ALU-pipe instructions x 2 cycles) per "
                                       "32-lane x 64-row step (SASS count, DESIGN.md section 11)"}}
    try:  # CPU side: the unmodified edlib as racon calls it (oracle/_ref), bounded sample, usable cores
        from oracle_lib import Ref, ref_align
        r = Ref()
        if r.available and not args.no_cpu_baseline:
            threads, core_info = usable_cores()
            t0, done = time.perf_counter(), 0
            with ThreadPoolExecutor(threads) as ex:
                while time.perf_counter() - t0 < cpu_seconds:
                    list(ex.map(lambda p: ref_align(r, p[0], p[1])[1], pairs[:len(fx)]))
                    done += len(fx)
            dt = time.perf_counter() - t0
            out["cpu_baseline"] = {"value": done / dt, "unit": "overlaps/s", "cores": threads, "kind": "reference",
                                   "sample": f"{done} alignments ({done // len(fx)} passes over the 181 overlaps), {dt:.1f} s, "
                                             f"edlibAlign(NW, path) + edlibAlignmentToCigar as src/overlap.cpp:205-224"}
    except Exception as e:  # the product's numbers do not depend on the checker
        out["cpu_baseline"] = {"unavailable": str(e)}
    try:  # long reads (what current ONT / HiFi overlaps look like): 40 kb pairs at 10 % edits, seeded
        from common import random_pairs
        base = random_pairs(4242, [(40000, 0.10)] * 24)
        lp = base * 20
        q2, qo2, t2, to2 = pack_pairs(lp)
        pool = AlignerPool(devices=(local_rank,), batches_per_device=3, max_gpu_memory_per_batch=20 << 30)
        walls = []
        with pinned(q2, t2):
            for it in range(2 + steps):  # the first rounds also teach every batch its band guess (verified on the device)
                t0 = time.perf_counter()
                ed2, buf2, off2, ln2, pinfo2 = pool.align(q2, qo2, t2, to2)
                if it >= 2:
                    walls.append(time.perf_counter() - t0)
        pool.close()
        lr = {"workload": f"synthetic long reads: {len(lp)} pairs of 40 kb, 10 % edits ({len(base)} distinct, seeded), "
                          f"{float(sum(len(a) * len(b) for a, b in lp)):.3g} matrix cells",
              "e2e": len(lp) / (sum(walls) / len(walls)), "unit": "overlaps/s", "e2e_ms_per_step": 1e3 * sum(walls) / len(walls),
              "cells_computed_per_step": pinfo2["cells"], "gpu_launches_per_step": pinfo2["kernel_launches"]}
        from oracle_lib import Ref, ref_align
        r = Ref()
        if r.available and not args.no_cpu_baseline:
            threads, core_info = usable_cores()
            ref_scores = [ref_align(r, a, b)[1] for a, b in base[:4]]
            if [int(x) for x in ed2[:4]] != ref_scores:
                raise RuntimeError("aligner (long reads): edit distances differ from edlib's")
            t0, done = time.perf_counter(), 0
            with ThreadPoolExecutor(threads) as ex:
                while time.perf_counter() - t0 < cpu_seconds / 2:
                    list(ex.map(lambda p: ref_align(r, p[0], p[1])[1], base * 4))
                    done += 4 * len(base)
            dt = time.perf_counter() - t0
            lr["cpu_baseline"] = {"value": done / dt, "unit": "overlaps/s", "cores": threads, "kind": "reference",
                                  "sample": f"{done} alignments of the same pairs, {dt:.1f} s, edlib as above"}
        out["long_reads"] = lr
    except Exception as e:
        out["long_reads"] = {"error": f"{type(e).__name__}: {e}"}
    return out


def roofline_block(name, m, steps):
    bytes_per_window, cells = algorithmic_bytes_per_window(m["batch"], m["banded"])
    peak, peak_src = measured_hbm_peak()
    launch_s = (m["dev_ms"] / 1e3) / steps
    achieved = bytes_per_window * m["nwin"] / launch_s / 1e9
    traffic, tsrc = recorded_traffic(name, m["nwin"])
    return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": traffic, "traffic_source": tsrc or "none (no ncu --set full capture committed for this workload)",
            "kernel": "poa_window_kernel", "algorithmic_bytes_per_window": bytes_per_window,
            "dp_cells_per_window": cells, "launch_ms": launch_s * 1e3, "peak_source": peak_src}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="A_banded", choices=sorted(WORKLOADS))
    ap.add_argument("--windows", type=int, default=0, help="override windows per GPU")
    ap.add_argument("--seed", type=int, default=12345)
    ap.add_argument("--batches", type=int, default=2, help="batch processors per GPU for the e2e leg (racon -c)")
    ap.add_argument("--rounds", type=float, default=1.0, help="e2e leg: launches per batch processor per step (chunk = windows / (batches x rounds))")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the A_full / B_banded block (N=1 only anyway)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (rank 0's windows) as DIR/<name>.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 0)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device visible (the engine has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    warmup = max(args.warmup, 3)

    m = measure(args.workload, args, rank, world, local_rank, device, args.steps, warmup, nwin=args.windows or None,
                keep_outputs=bool(args.dump_outputs) and rank == 0)

    # ---------------- reduce over ranks ---------------------------------------------------------------
    dev_ms, e2e_s, wall, failures = m["dev_ms"], m["e2e_s"], m["wall"], m["failures"]
    t = torch.tensor([dev_ms, e2e_s, wall, float(failures)], dtype=torch.float64, device=device)
    if world > 1:
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone()
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        dev_ms, e2e_s, wall = float(tmax[0]), float(tmax[1]), float(tmax[2])
        failures = int(tsum[3])
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    if args.dump_outputs:
        dump_outputs(args.dump_outputs, m.pop("outputs"))
    nwin, info = m["nwin"], m["info"]
    total_windows = nwin * world
    m["dev_ms"] = dev_ms
    result = {
        "metric": "POA windows/sec", "value": total_windows * args.steps / (dev_ms / 1e3), "unit": "windows/s",
        "n_gpus": world, "steps": args.steps, "warmup": warmup, "ms_per_step": dev_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int16", "data": "synthetic",
        "config": {"workload": workload_label(args.workload, nwin), "windows_per_gpu": nwin,
                   "l2": f"inputs larger than L2: {info['n_slots']} resident window workspaces x "
                         f"{info['slot_bytes'] / 1048576:.1f} MB are rewritten every step",
                   "resident_warps": info["n_slots"], "blocks_per_sm": info["blocks_per_sm"],
                   "e2e_batches_per_gpu": args.batches, "failed_windows": failures},
        "e2e": {"value": total_windows * args.steps / e2e_s, "unit": "windows/s", "h2d_bytes_per_step": m["h2d"],
                "d2h_bytes_per_step": m["d2h"],
                "api": "api.Polisher.polish_arena (b200poa_polisher_polish_arena): windows in a pinned columnar arena (host buffers), per batch: tables + H2D straight from the arena + kernel + D2H + trim"
                       + (" + NCCL gather of the compact consensus to rank 0, overlapped with the next step" if world > 1 else "")},
        "gpu_launches": m["timed_launches"],
        "clocks": m["clocks"],
        "roofline": roofline_block(args.workload, m, args.steps),
        "wall_s_timed_region": wall,
    }
    if world == 1 and not args.no_cpu_baseline:
        threads, core_info = usable_cores()
        result["cpu_baseline"] = cpu_reference_rate(m["batch"], m["L"], 12.0, threads, core_info)
    if world == 1 and not args.no_extra and args.workload == "A_banded" and not args.windows:
        extra = {}
        for name in ("A_full", "B_banded"):
            x = measure(name, args, rank, world, local_rank, device, 3, 3, sample_clocks=False)
            extra[name] = {
                "workload": workload_label(name, x["nwin"]), "steps": 3, "warmup": 3,
                "value": x["nwin"] * 3 / (x["dev_ms"] / 1e3), "e2e": x["nwin"] * 3 / x["e2e_s"], "unit": "windows/s",
                "ms_per_step": x["dev_ms"] / 3, "failed_windows": x["failures"],
                "h2d_bytes_per_step": x["h2d"], "d2h_bytes_per_step": x["d2h"],
                "resident_warps": x["info"]["n_slots"], "roofline": roofline_block(name, x, 3)}
        extra["A_banded_msa"] = measure_msa(args, local_rank, device)
        try:  # a separate step of the pipeline (SURVEY 8f-4): its block must never cost the headline line
            extra["overlap_aligner"] = measure_aligner(args, local_rank)
        except Exception as e:
            extra["overlap_aligner"] = {"error": f"{type(e).__name__}: {e}"}
        result["extra"] = extra
    print(json.dumps(result))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
