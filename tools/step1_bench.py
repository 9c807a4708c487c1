#!/usr/bin/env python
"""Step 1 (anchor finding, core positions) on the GPU: the per-region path (one nr_score_tasks call of four exact
32-bit alignments per read for every region, the rules in Python -- the package's path before nr_anchor_regions) against
the batched call (nr_anchor_regions: both anchors per read strand on u16x2 words, one launch; start recovery, a second).

Shapes: config 1 (15 regions x 30 reads), a 2 000-locus x 30-read catalog slice (50 simulated loci, each taken 40 times:
same cells, 240 MB of reads, more than L2), config 2's shape (2 amplicon regions x 5 000 reads).  Per shape: end-to-end
wall time of both paths (mean of --reps calls after a warm-up), kernel time of the batched call per kernel from a
torch.profiler run of its own, GCUPS of algorithmic cells (2 (|left| + |right|) |read| per read), the anchor kernel's
share of the u16x2 DPX peak (DESIGN.md section 7: 148 SMs x SM clock x 64 lanes x 2 cells / 7 DPX) and the second
launch's share of the device time.  Both paths must accept the same reads at the same positions.
Writes one JSON document (--out) with the card name, power limit and SM clock read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)


from nanorepeat_b200 import engine, synth  # noqa: E402
from nanorepeat_b200.anchoring import rev_comp  # noqa: E402


def per_region(sc, left, right, seqs):
    """The per-region path: -> {read index: (strand, dist, core_start, core_end)} of the accepted reads."""
    if not seqs:
        return {}
    q, t = [], []
    for s in seqs:
        r = rev_comp(s)
        q += [left, left, right, right]
        t += [s, r, s, r]
    recs = engine.score_tasks(q, t, sc)
    out = {}
    for i, s in enumerate(seqs):
        best = []
        for a in range(2):
            hits = [(int(recs[4 * i + 2 * a + d]["score"]), "+-"[d], int(recs[4 * i + 2 * a + d]["tstart"]), int(recs[4 * i + 2 * a + d]["tend"]))
                    for d in range(2) if recs[4 * i + 2 * a + d]["score"] >= max(1, sc.min_dp_score)]
            hits.sort(key=lambda h: h[0], reverse=True)
            best.append(hits[0] if len(hits) == 1 or (len(hits) == 2 and hits[0][0] > 1.5 * hits[1][0]) else None)
        if best[0] is None or best[1] is None:
            continue
        dist = best[1][2] - best[0][3] if best[0][1] == best[1][1] else 0
        if dist > -10:
            out[i] = (best[0][1], dist, max(best[0][3] - 100, 0), min(best[1][2] + 100, len(s)))
    return out


def shapes():
    loci = []
    for g in range(50):
        reg, _n, seqs, _t = synth.region_reads(seed=300 + g, n_reads=30, motif=("CAG", "GGGGCC", "AT", "TTTCA")[g % 4], alleles=(15, 45))
        loci.append((reg.left_anchor_seq, reg.right_anchor_seq, seqs, reg.repeat_unit_seq))
    amp = []
    for g, motif in enumerate(("CAG", "CCG")):
        reg, _n, seqs, _t = synth.region_reads(seed=400 + g, n_reads=5000, motif=motif, alleles=(20, 40), outer=150)
        amp.append((reg.left_anchor_seq, reg.right_anchor_seq, seqs, reg.repeat_unit_seq))
    return {"config1_15x30": loci[:15], "catalog_2000x30": [loci[g % 50] for g in range(2000)], "config2_2x5000": amp}


def kernel_ms(fn):
    """device time per kernel name of one call, from torch.profiler (CUDA activities)"""
    import torch
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.events():
        if ev.device_type.name == "CUDA" and "kernel" in ev.name.lower():
            key = "anchor_pair_kernel" if "anchor_pair_kernel" in ev.name else ("exact_kernel" if "exact_kernel" in ev.name else ev.name[:60])
            out[key] = out.get(key, 0.0) + ev.device_time / 1e3
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_step1_bench.json"))
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()[0].split(", ")
    sm_mhz = float(q[2].split()[0])
    engine.init(0)
    import torch
    torch.cuda.init()
    sc = engine.get_preset("ont")
    n_sm = engine.device_info()["sm_count"]
    peak16 = n_sm * sm_mhz * 1e6 * 64 * 2 / 7 / 1e9
    doc = {"gpu": q[0], "power_limit": q[1], "sm_clock_max_mhz": sm_mhz, "sm_clock_now": q[3], "u16x2_peak_gcups": peak16, "shapes": {}}
    for name, regs in shapes().items():
        lefts, rights, reads = [r[0] for r in regs], [r[1] for r in regs], [r[2] for r in regs]
        batched = lambda: engine.anchor_regions(sc, lefts, rights, reads)      # noqa: E731
        res, stats = batched()
        # same accepted reads, strands, distances and cores as the per-region path
        i = 0
        for (l, r, seqs, _m) in regs[:200]:
            want = per_region(sc, l, r, seqs)
            got = {j: (chr(res[i + j]["strand"]), int(res[i + j]["dist_between_anchors"]), int(res[i + j]["core_start"]),
                       int(res[i + j]["core_end"])) for j in range(len(seqs)) if res[i + j]["accepted"]}
            assert got == want, (name, i)
            i += len(seqs)
        t = []
        for _ in range(args.reps):
            t0 = time.perf_counter(); batched(); t.append(time.perf_counter() - t0)
        e2e_new = sum(t) / len(t)
        per_region(sc, *regs[0][:3])
        t0 = time.perf_counter()
        for l, r, seqs, _m in regs:
            per_region(sc, l, r, seqs)
        e2e_old = time.perf_counter() - t0
        k_new = kernel_ms(batched)
        k_old = kernel_ms(lambda: [engine.score_tasks([x for _s in seqs for x in (l, l, r, r)],
                                                      [x for s in seqs for x in (s, rev_comp(s), s, rev_comp(s))], sc) for l, r, seqs, _m in regs])
        cells = stats["algorithmic_cells"]
        dev_new = sum(k_new.values())
        dev_old = sum(k_old.values())
        pair_ms = k_new.get("anchor_pair_kernel", 0.0)
        # cells the anchor kernel executes: both halves of 32 R S rows per read strand (nr_anchor.cu, pair_shape)
        rows = lambda n: (lambda S: S * 32 * next(h for h in (4, 6, 8, 12, 16) if h * 32 * S >= n))(max(1, -(-n // 512)))  # noqa: E731
        pair_cells = sum(2 * 2 * rows(max(len(l), len(r))) * len(s) for l, r, seqs, _m in regs for s in seqs)
        doc["shapes"][name] = {
            "regions": len(regs), "reads": sum(map(len, reads)), "algorithmic_cells": cells, "stats": stats,
            "per_region": {"e2e_ms": e2e_old * 1e3, "device_ms": dev_old, "kernels_ms": k_old, "gcups_e2e": cells / e2e_old / 1e9,
                           "gcups_device": cells / dev_old / 1e6 if dev_old else None},
            "batched": {"e2e_ms": e2e_new * 1e3, "device_ms": dev_new, "kernels_ms": k_new, "gcups_e2e": cells / e2e_new / 1e9,
                        "gcups_device": cells / dev_new / 1e6 if dev_new else None,
                        "anchor_kernel_frac_u16x2_peak": pair_cells / (pair_ms * 1e-3) / 1e9 / peak16 if pair_ms else None,
                        "second_launch_share": (dev_new - pair_ms) / dev_new if dev_new else None},
            "speedup_e2e": e2e_old / e2e_new, "speedup_device": dev_old / dev_new if dev_new else None}
        print(name, json.dumps(doc["shapes"][name]["batched"]), "per-region e2e %.1f ms" % (e2e_old * 1e3), flush=True)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(doc, f, indent=1)


if __name__ == "__main__":
    main()
