#!/usr/bin/env python
"""bench.py -- NanoRepeat's repeat-size estimation hot path (rounds 1-3) on a B200.

Headline workload: BASELINE.json's config 2 (the configuration the metric is quoted on): the HTT amplicon, 5 000 synthetic
ONT reads, quantified as the two BED rows of example_data/HTT_repeat_region.bed (CAG and CCG) -> 10 000 (read, region)
units per pass, each aligned against its round-2 template and its round-3 ladder (31+ rungs).  A STEP is `--passes`
(default 20) passes over that batch, so that 20 steps keep the GPU busy for about a second.

  value     GCUPS = algorithmic DP cells (full rectangles |core| x |template|, SURVEY.md 8d) per second, inputs resident
            in HBM, CUDA-event time of the kernel launches, summed over the K steps, max over ranks.
  e2e       the same metric through the public operator API (nanorepeat_b200.estimate_regions on RepeatRegion / Read
            objects): host strings in, Read.round{1,2,3}_repeat_size out; packing, H2D, kernels, D2H, selection inside.
  roofline  DPX / integer-pipe bound of the dominant kernel: executed cells / CUDA-event time of its launches against
            SMs x sm_max_mhz x 64 DPX lanes/clk/SM x 2 cells per lane-instr / 7 DPX instr per cell pair (u16x2 kernels),
            x 1 / 6 for the 32-bit kernels.  `useful` = the same with padding rows removed.
  configs   the other four configs of BASELINE.json (1, 3 slice, 4, 5 sample), each with device time, per-kernel
            rooflines, e2e and a random sample of reads checked against the CPU oracle.
  strong    ONE workload (the config-5 sample) split over the ranks by sharding.estimate_regions_sharded (LPT by
            predicted cells, host gather inside the timed region): strong scaling next to the weak-scaling `value`.
  cpu_baseline / --impl reference   the CPU oracle port (oracle/nr_oracle.c: scalar full-rectangle DP, pthreads) on the
            host cores, on a bounded sample of the headline workload.  The reference's own engine (pyminimap2, a banded
            seed-chain-extend aligner) is not installable here; a banded SIMD aligner would be much faster than this port.

N > 1 (torchrun): every rank runs its own config-2 batch (seed + 1000 * rank) -- weak scaling, no data-path collective;
NCCL carries the barrier and the max-over-ranks of the times only.
"""
import argparse
import gc
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "GCUPS"
UNIT = "GCUPS (1e9 DP cells/s, full rectangles)"          # the same string in both arms
DPX_LANES_PER_CLK_PER_SM = 64       # measured: tools/microbench/pipe_rates.cu -> profiles/r01_pipe_rates.jsonl
DPX_INSTR_PER_CELL = 6              # 32-bit word: 2 (five-way max + floor for H) + 4 (E1, E2, F1, F2 updates)
DPX_INSTR_PER_CELL_PAIR = 7         # u16x2 words (two cells per instruction): 3 for H (no .RELU on unsigned halves) + 4
HEADLINE = "config 2: HTT CAG/CCG amplicon, 5k ONT reads, two BED rows, rounds 1-3"
DUMP_MAX_BYTES = 64_000_000         # --dump-outputs in all, headers included; above it a seeded sample of reads is written
NPY_HEADER_BYTES = 128              # header of a 1-D .npy file (format 1.0)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback"


def load_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed ncu capture of
    this command (profiles/r02_traffic.json, written by tools/ncu_traffic.py on the GPU box); None if absent."""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f)
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu_index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
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
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            c = [x.strip() for x in ln.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2]))
            except ValueError:
                continue
            for n, v in zip(names, c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        busy = [s for s in sm if s > 0.5 * max(sm)]
        return {"sm_mhz": statistics.median(busy), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm)}


def clock_snapshot(gpu_index):
    """One reading of the SM clock and the throttle reasons (outside any timed section)."""
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={ClockSampler.Q}", "--format=csv,noheader,nounits", "-i", str(gpu_index)],
                             capture_output=True, text=True, timeout=10).stdout.strip().split(",")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        return {"sm_mhz": float(out[1]), "sm_max_mhz": float(out[2]),
                "reasons": [n for n, v in zip(names, out[5:9]) if v.strip().lower().startswith("active")]}
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        return None


def headline_config(args):
    """`config` of the JSON line: the same dictionary in both arms (the driver compares them)."""
    return {"workload": HEADLINE, "reads": args.reads, "regions": 2, "seed": args.seed, "passes_per_step": args.passes,
            "l2": "not flushed" if args.no_flush else "flushed between timed steps (256 MB fill)"}


def region_cells(reg, T, kmin, kmax, ok):
    from nanorepeat_b200 import synth
    nl, nr_, m = len(reg.left_anchor_seq), len(reg.right_anchor_seq), len(reg.repeat_unit_seq)
    c2 = c3 = 0
    for i, core in enumerate(reg.core_seqs):
        c2 += len(core) * (nl + m * T)
        if ok[i]:
            c3 += synth.algorithmic_cells(nl, nr_, m, len(core), T, int(kmin[i]), int(kmax[i]))[1]
    return c2, c3


def oracle_pass(regs, threads):
    """Rounds 1-3 of `regs` on the CPU oracle -> (algorithmic cells, per-region results)."""
    from oracle import selection
    cells, out = 0, []
    for reg in regs:
        res = selection.estimate_region(reg.left_anchor_seq, reg.right_anchor_seq, reg.repeat_unit_seq, reg.core_seqs,
                                        reg.dist_between_anchors, n_threads=threads)
        ok = [r is not None for r in res["r2"]]
        c2, c3 = region_cells(reg, res["T"], [k if k is not None else 0 for k in res["kmin"]],
                              [k if k is not None else -1 for k in res["kmax"]], ok)
        cells += c2 + c3
        out.append(res)
    return cells, out


def run_reference_arm(args, rank):
    """The reference's CPU path for this metric: the oracle port on all host cores (pyminimap2 is not installable here).
    Each step is a bounded sample of the headline workload."""
    if rank != 0:
        return
    from nanorepeat_b200 import synth
    from oracle import nr_oracle
    nr_oracle.build()
    threads = nr_oracle.max_threads()
    n_sample = args.cpu_sample_reads
    regs = synth.config2(seed=args.seed, n_reads=n_sample)
    warm = min(args.warmup, 8)          # a CPU pass over the sample takes seconds: the driver's W is honoured up to 8
    for _ in range(warm):
        oracle_pass(regs, threads)
    t0 = time.perf_counter()
    cells = 0
    for _ in range(args.steps):
        cells += oracle_pass(regs, threads)[0]
    dt = time.perf_counter() - t0
    gcups = cells / dt / 1e9
    units = 2 * n_sample * args.steps
    sample = (f"{n_sample} of the workload's {args.reads} reads (same seed), both regions, rounds 1-3, full rectangles, "
              f"{threads} pthreads, one pass per step")
    line = {
        "impl": "reference", "metric": METRIC, "value": gcups, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": warm, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "reads_per_s": units / dt, "config": headline_config(args),
        "cpu_baseline": {"value": gcups, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": gcups, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "the reference's engine (pyminimap2 >= 2.30, a banded seed-chain-extend aligner) is absent and not "
                "installable offline; this arm times the CPU oracle port of the exact DP (oracle/nr_oracle.c, scalar, "
                "~0.25 GCUPS per thread)",
    }
    print(json.dumps(line), flush=True)


class Workload:
    """One synthetic workload on this rank's GPU: resident batches for the device-timed leg, the operator API for e2e."""

    def __init__(self, name, regs, data_type="ont", fast_mode=False):
        import nanorepeat_b200 as nrb
        from nanorepeat_b200 import engine
        from nanorepeat_b200.estimation import ladder_bounds_array
        self.name, self.regs, self.data_type, self.fast_mode = name, regs, data_type, fast_mode
        self.nrb, self.engine = nrb, engine
        self.sc = engine.get_preset(data_type)
        self.units = sum(len(r.core_seqs) for r in regs)
        # one pass through the public API: warm-up, and the round-2 sizes the resident round-3 batch is built from
        self.rrs = self.e2e_pass(self.fresh())
        self.T, self.kmin, self.kmax, self.valid = [], [], [], []
        cells2 = cells3 = 0
        for reg, rr in zip(regs, self.rrs):
            m = len(reg.repeat_unit_seq)
            r1max = max(float(d) / m for d in reg.dist_between_anchors)
            T = int(r1max * 1.5) + 1
            if T < r1max + 10:
                T = int(r1max + 10)
            r2 = [rr.read_dict[n].round2_repeat_size for n in reg.read_names]
            ok = np.array([v is not None for v in r2], bool)
            lo = np.zeros(len(r2), np.int32); hi = np.full(len(r2), -1, np.int32)
            if ok.any():
                lo[ok], hi[ok] = ladder_bounds_array(np.array([v for v in r2 if v is not None]), fast_mode)
            self.T.append(T); self.kmin.append(lo); self.kmax.append(hi); self.valid.append(ok)
            c2, c3 = region_cells(reg, T, lo, hi, ok)
            cells2 += c2; cells3 += c3
        self.cells = cells2 + cells3
        # resident batches: round 2 over all regions, round 3 over the reads round 2 left in HBM (the production flow)
        self.b2 = engine.Batch.begin(self.sc, "round2_flags")
        for reg, T in zip(regs, self.T):
            self.b2.add_round2(reg.left_anchor_seq, reg.repeat_unit_seq, T, reg.core_seqs)
        self.b2.commit()
        self.b3 = engine.Batch.begin_round3_from(self.b2)
        for i, (reg, lo, hi) in enumerate(zip(regs, self.kmin, self.kmax)):
            self.b3.add_round3_reuse(i, reg.right_anchor_seq, lo, hi)
        self.b3.commit()
        self.stats = [self.b2.stats(), self.b3.stats()]
        assert sum(s["algorithmic_cells"] for s in self.stats) == self.cells, (self.name, self.stats, self.cells)
        self.executed = sum(s["executed_cells"] for s in self.stats)
        self.h2d = sum(s["h2d_bytes"] for s in self.stats)
        self.d2h = sum(s["d2h_bytes"] for s in self.stats)

    def fresh(self):
        return [self.nrb.RepeatRegion.from_synth(reg) for reg in self.regs]

    def e2e_pass(self, rrs):
        self.nrb.estimate_regions(rrs, self.data_type, self.fast_mode)
        return rrs

    def resident_pass(self, stream):
        self.b2.run(stream)
        self.b3.run(stream)

    def close(self):
        self.b3.close(); self.b2.close()

    def check_against_oracle(self, n_sample, seed, threads, max_cells=4e10):
        """A random sample of reads per region against the CPU oracle's rounds 1-3 (r1, r2, r3 bit for bit), bounded
        by `max_cells` of oracle work (the longest reads of configs 4 and 5 are 10^10 cells each)."""
        from oracle import selection
        rng = np.random.default_rng(seed)
        checked = cells = 0
        order = rng.permutation(len(self.regs))
        for gi in order:
            reg, rr = self.regs[gi], self.rrs[gi]
            idx = rng.choice(len(reg.read_names), min(n_sample, len(reg.read_names)), replace=False)
            cost = sum(len(reg.core_seqs[i]) for i in idx) * 31.0 * (len(reg.left_anchor_seq) + len(reg.right_anchor_seq) +
                                                                     max(reg.dist_between_anchors))
            if cells and cells + cost > max_cells:
                continue
            cells += cost
            exp = selection.estimate_region(reg.left_anchor_seq, reg.right_anchor_seq, reg.repeat_unit_seq,
                                            [reg.core_seqs[i] for i in idx], [reg.dist_between_anchors[i] for i in idx],
                                            fast_mode=self.fast_mode, n_threads=threads, max_dist=max(reg.dist_between_anchors))
            for j, i in enumerate(idx):
                rd = rr.read_dict[reg.read_names[i]]
                g3, e3 = rd.round3_repeat_size, exp["r3"][j]
                assert rd.round1_repeat_size == exp["r1"][j] and rd.round2_repeat_size == exp["r2"][j] and \
                    (None if g3 is None else float(g3)) == (None if e3 is None else float(e3)), \
                    f"{self.name}: read {reg.read_names[i]} differs from the oracle: {rd.round2_repeat_size} {g3} vs {exp['r2'][j]} {e3}"
                checked += 1
        return checked


def dump_outputs(out_dir, arrays):
    """arrays: name -> one value per read, all of the same length -> out_dir/<name>.npy as float64, and the reads'
    positions in read_index.npy.  Above DUMP_MAX_BYTES in all, every file holds the same seeded sample of the reads."""
    os.makedirs(out_dir, exist_ok=True)
    n = len(next(iter(arrays.values())))
    n_files = len(arrays) + 1
    keep = (DUMP_MAX_BYTES - NPY_HEADER_BYTES * n_files) // (8 * n_files)
    idx = np.arange(n) if n <= keep else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    np.save(os.path.join(out_dir, "read_index.npy"), idx.astype(np.float64))
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64)
        assert len(a) == n, (name, len(a), n)
        np.save(os.path.join(out_dir, name + ".npy"), a[idx])


def sizes_or_nan(rrs, attr):
    return [np.nan if v is None else float(v) for rr in rrs for v in (getattr(rd, attr) for rd in rr.read_dict.values())]


def kernel_table(linfo, kern_ms, launches, peak16, peak32):
    """Per-kernel rooflines from nr_batch_launch_info: executed cells per launch / mean CUDA-event time per launch."""
    names = [("pair_round2_kernel (round 2, u16x2 pairs + 32-bit entries beside them)", 0, "paired"),
             ("exact_kernel (round 2, 32-bit, separate launch)", 0, "rest"),
             ("pair_ladder_kernel (round 3, u16x2 pairs + 32-bit entries beside them)", 1, "paired"),
             ("ladder_kernel (round 3, 32-bit flag words, separate launch)", 1, "rest")]
    out = {}
    for name, b, kind in names:
        ms = kern_ms[b][kind + "_ms"]
        if ms <= 0:
            continue
        li = linfo[b]
        if kind == "paired":       # the fused launch runs the batch's 32-bit entries too: both classes against their peaks
            ideal = li["paired_cells"] / peak16 + li["rest_cells"] / peak32
            useful = li["paired_useful_cells"] / peak16 + li["rest_useful_cells"] / peak32
            cells = li["paired_cells"] + li["rest_cells"]
        else:
            ideal = li["rest_cells"] / peak32
            useful = li["rest_useful_cells"] / peak32
            cells = li["rest_cells"]
        per = ms / launches * 1e-3
        out[name] = {"ms_per_launch": ms / launches, "executed_cells_per_launch": cells,
                     "achieved": cells / per / 1e9, "frac": ideal / 1e9 / per, "frac_useful": useful / 1e9 / per,
                     "u16x2_share_of_cells": li["paired_cells"] / cells if kind == "paired" and cells else 0.0}
    return out


def time_resident(wl, torch, stream, flush, steps, passes, engine):
    """K steps of `passes` passes each; CUDA events around every step on the launching stream; L2 flushed between steps
    (inside a step consecutive passes stream 10^5 different reads, far more state than L2 re-use could help)."""
    kern_ms = [dict(paired_ms=0.0, rest_ms=0.0, redo_ms=0.0) for _ in range(2)]
    dev_ms = []
    engine.set_timing(True)
    for _ in range(steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _p in range(passes):
            wl.resident_pass(stream.cuda_stream)
            for acc, b in zip(kern_ms, (wl.b2, wl.b3)):      # (waits for this pass: the per-launch events are per batch)
                li = b.launch_info()
                for key in acc:
                    acc[key] += li[key]
        e1.record(stream)
        e1.synchronize()
        dev_ms.append(e0.elapsed_time(e1))
    engine.set_timing(False)
    return dev_ms, kern_ms


def time_resident_async(wl, torch, stream, flush, steps, passes):
    """The same without per-kernel events: passes queued back to back (no host wait inside a step)."""
    dev_ms = []
    for _ in range(steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _p in range(passes):
            wl.resident_pass(stream.cuda_stream)
        e1.record(stream)
        e1.synchronize()
        dev_ms.append(e0.elapsed_time(e1))
    return dev_ms


def time_e2e(wl, torch, passes_total):
    """Public operator API, fresh RepeatRegion / Read objects per pass (built outside the timed sections).  Two untimed
    passes first: the resident batches built after the workload's first call hold the buffers that call had cached, so
    the next call allocates device and pinned memory anew (hundreds of milliseconds once, nothing to do with a pass)."""
    warm = 2
    total = 0.0
    wl.e2e_pass_ms = []
    gc.collect()
    gc.freeze()              # this process holds five workloads' worth of objects: keep the collector from walking them
    try:                     # inside the timed calls (its cost there would be an artefact of the bench); GC stays enabled
        for i in range(warm + passes_total):
            rrs = wl.fresh()
            t0 = time.perf_counter()
            wl.e2e_pass(rrs)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if i < warm:     # same flow as the timed passes: with three calls in flight the library may need a third set of
                continue     # buffers that an earlier, differently interleaved pass never asked for (a one-off 100 ms)
            total += dt
            wl.e2e_pass_ms.append(round(dt * 1e3, 3))
            wl.last_rrs = rrs
    finally:
        gc.unfreeze()
    return total


def time_c_abi(wl, torch, passes_total):
    """The same work through the C ABI's one call: lists of host strings in, numpy arrays out, no Read objects."""
    lefts = [r.left_anchor_seq for r in wl.regs]
    rights = [r.right_anchor_seq for r in wl.regs]
    motifs = [r.repeat_unit_seq for r in wl.regs]
    cores = [list(r.core_seqs) for r in wl.regs]
    dists = np.array([d for r in wl.regs for d in r.dist_between_anchors], dtype=np.int32)
    wl.engine.estimate_regions(wl.sc, wl.fast_mode, lefts, rights, motifs, cores, dists)
    t0 = time.perf_counter()
    for _ in range(passes_total):
        wl.engine.estimate_regions(wl.sc, wl.fast_mode, lefts, rights, motifs, cores, dists)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / passes_total * 1e3


def measure_config(name, regs, torch, stream, flush, engine, peak16, peak32, steps, passes, e2e_passes, threads, check):
    t0 = time.perf_counter()
    wl = Workload(name, regs)
    for _ in range(3):
        wl.resident_pass(stream.cuda_stream)
    torch.cuda.synchronize()
    dev_ms, kern_ms = time_resident(wl, torch, stream, flush, steps, passes, engine)
    linfo = [wl.b2.launch_info(), wl.b3.launch_info()]
    e2e_s = time_e2e(wl, torch, e2e_passes)
    c_abi_ms = time_c_abi(wl, torch, e2e_passes)
    n_pass = steps * passes
    dev_s = sum(dev_ms) * 1e-3
    res = {
        "reads": wl.units, "regions": len(regs), "core_len_median": float(np.median([len(c) for r in regs for c in r.core_seqs])),
        "core_len_max": int(max(len(c) for r in regs for c in r.core_seqs)),
        "cells_per_pass": wl.cells, "executed_cells_per_pass": wl.executed,
        "value": wl.cells * n_pass / dev_s / 1e9, "unit": UNIT, "reads_per_s": wl.units * n_pass / dev_s,
        "ms_per_pass": dev_s / n_pass * 1e3, "executed_gcups": wl.executed * n_pass / dev_s / 1e9,
        "e2e": {"value": wl.cells * e2e_passes / e2e_s / 1e9, "unit": UNIT, "reads_per_s": wl.units * e2e_passes / e2e_s,
                "ms_per_pass": e2e_s / e2e_passes * 1e3, "passes_ms": wl.e2e_pass_ms, "c_abi_ms_per_pass": c_abi_ms,
                "h2d_bytes_per_pass": wl.h2d, "d2h_bytes_per_pass": wl.d2h},
        "kernels": kernel_table(linfo, kern_ms, n_pass, peak16, peak32),
        "redo_reads_per_pass": linfo[1]["n_redo"], "unscored_reads": sum(s["n_skipped"] for s in wl.stats),
    }
    if check:
        res["oracle_checked_reads"] = wl.check_against_oracle(check, 7, threads)
    res["setup_s"] = time.perf_counter() - t0
    wl.close()
    return res


def measure_joint(torch, engine, peak32, threads, n_reads=1000, n_check=48):
    """Config 2 read as what BASELINE.json literally names -- HTT CAG/CCG JOINT quantification: nanoRepeat-joint's grid
    rounds 2 and 3 (nanoRepeat_joint.py:234-273) for one locus through nr_joint_grid: one backward sweep per (read, strand)
    and one forward sweep per k1 with a junction per k2 (nr_window_ladder.cuh); `cells` counts every grid point's full
    rectangle (the algorithmic work the reference does), the window score comes out of the DP.  A sample of grid points
    is checked against the CPU oracle."""
    from nanorepeat_b200 import joint, synth
    from oracle import nr_oracle
    loc = synth.joint_locus(seed=7, n_reads=n_reads)
    args = (loc["reads"], loc["left"], loc["mid"], loc["right"], "CAG", "CCG", loc["range1"], loc["range2"], 200, 50)
    counted = {"points": 0, "cells": 0}

    def counting_grid(sc, left, mid, right, m1, m2, reads, pr, p1, p2):
        counted["points"] += len(pr)
        lens = np.array([len(r) for r in reads], dtype=np.int64)
        tlen = len(left) + len(mid) + len(right) + len(m1) * np.asarray(p1, dtype=np.int64) + len(m2) * np.asarray(p2, dtype=np.int64)
        counted["cells"] += int((2 * lens[np.asarray(pr, dtype=np.int64)] * tlen).sum())
        counted["last"] = (pr, p1, p2)
        rec, strand = engine.joint_grid(sc, left, mid, right, m1, m2, reads, pr, p1, p2)
        counted["rec"], counted["strand"] = rec, strand
        return rec, strand

    joint.quantify_two_repeats(*args)                       # warm-up
    counted.update(points=0, cells=0)
    t0 = time.perf_counter()
    res = joint.quantify_two_repeats(*args, align=counting_grid)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    # parity spot check on the last round's grid points
    pr, p1, p2 = counted["last"]
    rng = np.random.default_rng(3)
    for i in rng.choice(len(pr), min(n_check, len(pr)), replace=False):
        r, k1, k2 = int(pr[i]), int(p1[i]), int(p2[i])
        tpl = loc["left"] + "CAG" * k1 + loc["mid"] + "CCG" * k2 + loc["right"]
        a, b = max(len(loc["left"]) - 10, 0), min(len(loc["left"]) + 3 * k1 + len(loc["mid"]) + 3 * k2 + 10, len(tpl))
        f = nr_oracle.align_window(loc["reads"][r], tpl, a, b, reverse=False)
        v = nr_oracle.align_window(loc["reads"][r], tpl, a, b, reverse=True)
        exp = v if v > f else f
        got = (int(counted["rec"]["score"][i]), int(counted["rec"]["window_score"][i]))
        assert got == exp, f"joint grid point {i}: {got} vs oracle {exp}"
    good = sum(abs(float(a) - t[0]) <= 1 and abs(float(b) - t[1]) <= 1
               for a, b, t in zip(res["size1"], res["size2"], loc["truth"]) if a is not None)
    return {"workload": f"HTT-like locus, {n_reads} raw amplicon reads (either strand), grid rounds 2 and 3 of nanoRepeat-joint",
            "reads": n_reads, "grid_points": int(counted["points"]), "cells": int(counted["cells"]), "s": dt, "reads_per_s": n_reads / dt,
            "value": counted["cells"] / dt / 1e9, "unit": UNIT, "algorithmic_gcups_over_32bit_peak": counted["cells"] / dt / 1e9 / peak32,
            "oracle_checked_points": min(n_check, len(pr)), "reads_within_1_unit_of_both_simulated_counts": good,
            "path": "joint.quantify_two_repeats -> nr_joint_grid (host strings in, sizes out; both strands of every grid point; "
                    "time includes template building, packing, both launches and the selection)"}


def measure_phasing(torch, engine, n_loci=2000, reads_per_locus=30, n_cpu=6):
    """Step 4 for a config-3 slice: 1-D allele phasing of n_loci regions x reads_per_locus round-3 sizes in one
    nr_phase_1d call (trim, 100x bootstrap, auto-GMM with 10 starts per fit, labels), beside the reference's recipe --
    scikit-learn's GaussianMixture driven the way split_alleles.auto_GMM_1d drives it -- on n_cpu of the loci, one thread
    (the reference pins MKL / OMP to one thread, split_alleles.py:30-32)."""
    import math
    import warnings
    from oracle import gmm as ogmm
    rng = np.random.default_rng(11)
    loci, truth = [], []
    for g in range(n_loci):
        het = rng.random() < 0.6
        a = int(rng.integers(5, 120))
        b = a + int(rng.integers(6, 60)) if het else a
        ks = np.where(rng.random(reads_per_locus) < 0.5, a, b)
        loci.append(list(np.round(ks + rng.normal(0, 0.01 * (10 + ks)), 2)))
        truth.append(2 if het else 1)
    params = engine.GmmParams(error_rate=0.07, max_mutual_overlap=0.15, max_components=22, seed=5)
    engine.phase_1d(params, loci[:64])                                              # warm-up
    t0 = time.perf_counter()
    fits = engine.phase_1d(params, loci)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    agree = int(sum(f["n"] == t for f, t in zip(fits, truth)))
    # config 2's shape: two regions of 5 000 reads (500 000 bootstrapped samples each: a cluster of thread blocks per fit)
    big = [list(np.round(np.where(rng.random(5000) < 0.5, a, b) + rng.normal(0, 0.4, 5000), 2)) for a, b in ((17, 55), (7, 10))]
    engine.phase_1d(params, big)
    t0 = time.perf_counter()
    big_fits = engine.phase_1d(params, big)
    torch.cuda.synchronize()
    big_dt = time.perf_counter() - t0
    # the reference recipe on a few loci
    from sklearn.mixture import GaussianMixture
    z = ogmm.std_isf(0.15)
    t0 = time.perf_counter()
    same = 0
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for g in range(n_cpu):
            xs = np.array(loci[g])
            lo, hi = ogmm.outlier_cutoffs(xs)
            kept = xs[(xs >= lo) & (xs <= hi)]
            sim = np.tile(kept, 100)
            sim = (sim + rng.normal(0, 1, len(sim)) * 0.07 * (10 + sim)).reshape(-1, 1)
            best = 22
            for n in range(2, 23):
                gm = GaussianMixture(n_components=n, covariance_type="diag", n_init=10).fit(sim)
                sd = np.maximum(1.0, np.sqrt(gm.covariances_[:, 0]))
                m = gm.means_[:, 0]
                if any(max(m[i] - z * sd[i], m[j] - z * sd[j]) - min(m[i] + z * sd[i], m[j] + z * sd[j]) <= 0
                       for i in range(n) for j in range(i + 1, n)):
                    best = n - 1
                    break
            GaussianMixture(n_components=best, covariance_type="diag", n_init=10).fit(sim)
            same += int(best == fits[g]["n"])
    cpu_dt = time.perf_counter() - t0
    return {"workload": f"{n_loci} loci x {reads_per_locus} round-3 sizes (60 % heterozygous), error_rate 0.07, overlap 0.15, up to 22 components",
            "s": dt, "loci_per_s": n_loci / dt, "samples_fitted": n_loci * reads_per_locus * 100,
            "loci_with_the_simulated_number_of_alleles": agree,
            "config2_shape": {"regions": 2, "reads_per_region": 5000, "s": big_dt, "alleles": [int(f["n"]) for f in big_fits],
                              "means": [[round(float(m), 2) for m in f["means"]] for f in big_fits]},
            "path": "engine.phase_1d -> nr_phase_1d (host sizes in, mixtures + labels out)",
            "cpu_reference_recipe": {"loci": n_cpu, "s": cpu_dt, "loci_per_s": n_cpu / cpu_dt, "threads": 1,
                                     "same_number_of_alleles": same,
                                     "what": "scikit-learn GaussianMixture(n, 'diag', n_init=10) for n = 2.. until overlap + refit, as split_alleles.auto_GMM_1d"}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of `value` (each --passes passes over the batch); the end-to-end and C-ABI legs time "
                         "as many passes, the per-kernel event leg a quarter as many steps (at least one)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--reads", type=int, default=5000, help="reads in the headline batch (config 2: 5000)")
    ap.add_argument("--passes", type=int, default=20, help="passes over the batch per step")
    ap.add_argument("--seed", type=int, default=2)
    ap.add_argument("--cpu-sample-reads", type=int, default=400)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the other four configs and the strong-scaling leg")
    ap.add_argument("--no-flush", action="store_true", help="no L2 flush between steps (for ncu traffic captures)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the headline batch's results of the last timed step (and of the last e2e pass) as "
                         "DIR/<name>.npy, one float64 value per read, so that two builds can be compared (rank 0)")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the GPU arm's results; --impl reference has none")
        run_reference_arm(args, rank)
        return

    args.warmup = max(args.warmup, 3)
    import torch
    import torch.distributed as dist
    from nanorepeat_b200 import engine, sharding, synth
    import nanorepeat_b200 as nrb

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    engine.init(local_rank)
    info = engine.device_info()
    peaks, peak_src = load_peaks()
    sm_max = float(peaks.get("sm_max_mhz", 1965.0))
    peak32 = info["sm_count"] * sm_max * 1e6 * DPX_LANES_PER_CLK_PER_SM / DPX_INSTR_PER_CELL / 1e9
    peak16 = info["sm_count"] * sm_max * 1e6 * DPX_LANES_PER_CLK_PER_SM * 2 / DPX_INSTR_PER_CELL_PAIR / 1e9
    stream = torch.cuda.Stream()
    flush = torch.empty((1 if args.no_flush else 256) * 1024 * 1024, dtype=torch.uint8, device="cuda")     # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- headline: config 2, every rank its own batch (weak scaling) ----
    wl = Workload(HEADLINE, synth.config2(seed=args.seed + 1000 * rank, n_reads=args.reads))
    K, P = args.steps, args.passes
    for _ in range(args.warmup * min(P, 4)):
        wl.resident_pass(stream.cuda_stream)
    torch.cuda.synchronize()
    launches_pass = sum(b.stats()["kernel_launches"] for b in (wl.b2, wl.b3))
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    wall0 = time.perf_counter()
    dev_ms = time_resident_async(wl, torch, stream, flush, K, P)                 # the number `value` is made of
    barrier()
    wall = time.perf_counter() - wall0
    if args.dump_outputs:
        r2_score, r2_tend, r2_starts = wl.b2.fetch_round2()
        r3_sum_k, r3_n_k, r3_top = wl.b3.fetch_round3()
    ev_ms, kern_ms = time_resident(wl, torch, stream, flush, max(1, K // 4), P, engine)      # per-kernel event times
    linfo = [wl.b2.launch_info(), wl.b3.launch_info()]
    n_ev = max(1, K // 4) * P
    # the 100 ms clock poll covers the device-timed region above and stops here: every NVML query stalls the CUDA calls
    # of this process for a while, which a host-timed 6 ms pass feels (measured: +0.8 ms per pass under the poll); the e2e
    # passes get one clock reading before and one after instead
    clocks = sampler.stop()
    clocks["e2e_before"] = clock_snapshot(local_rank)
    # e2e through the operator API
    e2e_passes = K
    for _ in range(2):
        wl.e2e_pass(wl.fresh())
    barrier()
    e2e_s = time_e2e(wl, torch, e2e_passes)
    c_abi_ms = time_c_abi(wl, torch, e2e_passes)
    barrier()
    clocks["e2e_after"] = clock_snapshot(local_rank)
    total_ms = float(sum(dev_ms))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {
            "round2_score": r2_score, "round2_tend": r2_tend, "round2_starts_by_left": r2_starts,
            "round3_sum_k": r3_sum_k, "round3_n_k": r3_n_k, "round3_top_score": r3_top,
            **{f"e2e_{a}": sizes_or_nan(wl.last_rrs, a) for a in ("round1_repeat_size", "round2_repeat_size", "round3_repeat_size")}})

    # resumed round 3 (from round 2's kept state) == a fresh round-3 batch (full forward sweeps): checked on every run
    s3 = wl.b3.fetch_round3()
    with engine.Batch.begin(wl.sc, "round3") as fresh3:
        for reg, lo, hi, ok in zip(wl.regs, wl.kmin, wl.kmax, wl.valid):
            idx = np.flatnonzero(ok)
            fresh3.add_round3(reg.left_anchor_seq, reg.right_anchor_seq, reg.repeat_unit_seq,
                              [reg.core_seqs[i] for i in idx], lo[idx], hi[idx])
        s3_fresh = fresh3.commit().run().fetch_round3()
    vmask = np.concatenate(wl.valid)
    assert all(np.array_equal(x[vmask], y) for x, y in zip(s3, s3_fresh)), "resumed and fresh round-3 results differ"

    # ---- strong scaling: ONE workload (config-5 sample, same seed on every rank) split by estimate_regions_sharded ----
    strong = None
    if not args.no_configs:          # (at every N: this is the leg whose time must fall with N)
        sregs = synth.config5(seed=5, n_reads=10000)
        def sharded_pass():
            rrs = [nrb.RepeatRegion.from_synth(r) for r in sregs]
            gc.collect()
            barrier()
            t0 = time.perf_counter()
            sharding.estimate_regions_sharded(rrs, "ont", False, rank=rank, world_size=world, gather=world > 1)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            return dt, rrs
        sharded_pass()
        times = []
        for _ in range(3):
            dt, srrs = sharded_pass()
            times.append(dt)
        t = torch.tensor(times, dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        best = float(t.min())
        n_r3 = sum(rd.round3_repeat_size is not None for rr in srrs for rd in rr.read_dict.values())
        strong = {"workload": "config 5 sample: 200 regions x 50 reads (1 % of 1M), k log-uniform 1..2000, ont / clr profiles, same seed on every rank",
                  "reads": sum(len(r.core_seqs) for r in sregs), "reads_with_round3_on_every_rank": n_r3,
                  "s_per_pass": best, "reads_per_s": sum(len(r.core_seqs) for r in sregs) / best,
                  "path": "sharding.estimate_regions_sharded: region pieces dealt by LPT on predicted cells, rounds 1-3 on each rank's GPU, "
                          "host gather of (r1, r2, r3) per read inside the timed region; max over ranks, best of 3 passes",
                  "note": "strong-scaling efficiency at N GPUs = s_per_pass(N=1) / (N * s_per_pass(N))"}

    if world > 1:
        t = torch.tensor([total_ms, e2e_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, e2e_s = float(t[0]), float(t[1])
        c = torch.tensor([wl.cells, wl.executed, wl.units], dtype=torch.float64, device="cuda")
        dist.all_reduce(c, op=dist.ReduceOp.SUM)
        cells_all, executed_all, units_all = (float(x) for x in c)
    else:
        cells_all, executed_all, units_all = wl.cells, wl.executed, wl.units

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    n_pass = K * P
    value = cells_all * n_pass / (total_ms * 1e-3) / 1e9
    kernels = kernel_table(linfo, kern_ms, n_ev, peak16, peak32)
    # the dominant kernel; when another launch is within 5 % of it, the one further below its roofline is reported
    # (config 2's two kernels take 1.22 and 1.23 ms: which is "longest" would flip from run to run)
    longest = max(v["ms_per_launch"] for v in kernels.values())
    dom_name = min((k for k in kernels if kernels[k]["ms_per_launch"] >= 0.95 * longest), key=lambda k: kernels[k]["frac"])
    dom = kernels[dom_name]
    step_ms = total_ms / K
    ideal_ms_pass = sum((li["paired_cells"] / peak16 + li["rest_cells"] / peak32) / 1e9 * 1e3 for li in linfo)
    useful_ms_pass = sum((li["paired_useful_cells"] / peak16 + li["rest_useful_cells"] / peak32) / 1e9 * 1e3 for li in linfo)
    traffic = load_traffic()
    if traffic and "per_kernel" in traffic:
        hit = [v for k, v in traffic["per_kernel"].items() if k in dom_name]
        traffic = dict(traffic, **hit[0]) if hit else None
    from oracle import nr_oracle
    nr_oracle.build()
    threads = nr_oracle.max_threads()
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": args.warmup,
        "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u16x2 (2*score + mark + 64 per half, two reads per word); s32 (score*65536 - span) for reads > 384 bases",
        "data": "synthetic", "reads_per_s": units_all * n_pass / (total_ms * 1e-3),
        "executed_gcups": executed_all * n_pass / (total_ms * 1e-3) / 1e9,
        "config": headline_config(args),
        "workload_size": {"units_per_pass_per_gpu": wl.units, "cells_per_pass_per_gpu": wl.cells},
        "e2e": {"value": cells_all * e2e_passes / e2e_s / 1e9, "unit": UNIT,
                "h2d_bytes_per_step": wl.h2d * P, "d2h_bytes_per_step": wl.d2h * P,
                "h2d_bytes_per_pass": wl.h2d, "d2h_bytes_per_pass": wl.d2h,
                "reads_per_s": units_all * e2e_passes / e2e_s, "ms_per_pass": e2e_s / e2e_passes * 1e3,
                "device_ms_per_pass": total_ms / n_pass, "passes_timed": e2e_passes, "passes_ms": wl.e2e_pass_ms,
                "c_abi_ms_per_pass": c_abi_ms,
                "c_abi_path": "engine.estimate_regions: lists of host strings in, numpy arrays out (the same nr_estimate_regions "
                              "call without the per-Read attribute traffic of the operator API)",
                "path": "nanorepeat_b200.estimate_regions on RepeatRegion / Read objects (host strings in, "
                        "Read.round{1,2,3}_repeat_size out) -> nr_estimate_regions (one C-ABI call, rounds 1-3)"},
        "gpu_launches": int(launches_pass * n_pass * world),
        "clocks": clocks,
        "roofline": {"bound": "dpx", "kernel": dom_name, "achieved": dom["achieved"],
                     "peak": dom["executed_cells_per_launch"] / 1e9 / (dom["frac"] * dom["ms_per_launch"] * 1e-3) if dom["frac"] else peak16,
                     "unit": "GCUPS", "frac": dom["frac"], "frac_useful": dom["frac_useful"], "ms_per_launch": dom["ms_per_launch"],
                     "traffic": traffic["bytes_per_launch"] if traffic else None,
                     "traffic_source": traffic["source"] if traffic else None,
                     "algorithmic_bytes_per_launch": wl.stats[1]["h2d_bytes"] + wl.stats[1]["d2h_bytes"],
                     "kernels": kernels,
                     "step": {"frac": ideal_ms_pass * P / step_ms, "frac_useful": useful_ms_pass * P / step_ms, "ms": step_ms,
                              "dpx_ideal_ms": ideal_ms_pass * P,
                              "def": "sum over kernels of executed (useful: unpadded) cells / that kernel class's DPX peak, "
                                     "over the step's device time"},
                     "peak_def": f"{info['sm_count']} SMs x {sm_max:.0f} MHz ({peak_src}) x {DPX_LANES_PER_CLK_PER_SM} DPX lanes/clk/SM "
                                 f"(measured) x 2 cells per lane-instr / {DPX_INSTR_PER_CELL_PAIR} DPX instr per cell pair = "
                                 f"{peak16:.0f} GCUPS (u16x2 kernels); x 1 / {DPX_INSTR_PER_CELL} = {peak32:.0f} GCUPS (32-bit kernels); "
                                 "a fused launch is held to the mix of both",
                     "executed_cells_per_pass": wl.executed, "algorithmic_cells_per_pass": wl.cells,
                     "useful_cell_fraction": (sum(li["paired_useful_cells"] + li["rest_useful_cells"] for li in linfo) /
                                              max(1, sum(li["paired_cells"] + li["rest_cells"] for li in linfo))),
                     "hbm_gbs_algorithmic": (wl.h2d + wl.d2h) / (total_ms / n_pass * 1e-3) / 1e9,
                     "hbm_peak_gbs": peaks.get("hbm_gbs")},
        "wall_s_timed_region": wall,
    }
    if strong:
        line["strong"] = strong
    if not args.no_configs and world == 1:
        cfgs = {}
        plan = [("config 1: 15 STR regions x 30 ont_q20 reads", lambda: synth.config1(seed=1), 5, 20, 10, 30),
                ("config 3 (slice): 2000 of 100k loci x 30 HiFi reads, 2-6 bp motifs", lambda: synth.config3(seed=3, n_loci=2000), 4, 2, 6, 2),
                ("config 4: C9orf72 ~1000 x GGGGCC and FMR1 ~500 x CGG, 200 R9 reads per locus", lambda: synth.config4(seed=4, reads_per_locus=200), 4, 2, 5, 3),
                ("config 5 (1 % sample): 200 regions x 50 reads, k log-uniform 1..2000, ont / clr", lambda: synth.config5(seed=5, n_reads=10000), 3, 1, 4, 2)]
        for name, make, steps, passes, e2e_passes_c, check in plan:
            cfgs[name] = measure_config(name, make(), torch, stream, flush, engine, peak16, peak32, steps, passes,
                                        e2e_passes_c, threads, check)
        line["configs"] = cfgs
    if not args.no_configs and world == 1:
        line["joint"] = measure_joint(torch, engine, peak32, threads)
        line["phasing"] = measure_phasing(torch, engine)
    if not args.no_cpu_baseline:
        sample = synth.config2(seed=args.seed, n_reads=args.cpu_sample_reads)
        t0 = time.perf_counter()
        c, _ = oracle_pass(sample, threads)
        dt = time.perf_counter() - t0
        line["cpu_baseline"] = {"value": c / dt / 1e9, "unit": UNIT, "cores": threads, "kind": "port",
                                "sample": f"{args.cpu_sample_reads} of the workload's {args.reads} reads x 2 regions, rounds 1-3, {dt:.1f} s; "
                                          "scalar full-rectangle DP (oracle/nr_oracle.c), not the reference's banded aligner",
                                "executed_cell_ratio_note": "the GPU executes ~22x fewer cells than it is credited with (shared ladder "
                                                            "prefixes / suffixes): executed_gcups / cpu value is the like-for-like rate ratio"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
