#!/usr/bin/env python
"""Fingerprints of the library's launch plans (tests/test_gpu_plan_identity.py).

A committed batch's plan decides which reads share a warp, the stripe heights of the long reads, the entry order of
the 32-bit launch and the layout of the uploaded blob.  `nr_batch_stats` and `nr_batch_launch_info` of a committed
batch summarise it: cells and useful cells of both launches, the pair count, the entry count (`n_rest`) and the bytes
of every blob section (`h2d_bytes`).  Any change to what gets paired, to a stripe height or to an entry moves at least
one of them.  The cases cover both rounds on every kind and ladder mode, round 3 resumed from round 2, the long pairs
of both rounds, the commit-time knobs NR_ROUND2_EXIT, NR_NO_LONG_PAIRS and NR_COOP_ROWS, a region whose anchor holds
an N, and a task batch.  Batches are committed only, never run.

Stripe heights depend on the device's SM count, which the fixture records.

Usage (on a GPU): python tests/golden/make_golden_plan.py   -> tests/golden/plan_fingerprints.json
"""
import functools
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from nanorepeat_b200 import engine, synth                     # noqa: E402
from nanorepeat_b200.estimation import ladder_bounds_array    # noqa: E402

OUT = os.path.join(HERE, "plan_fingerprints.json")
LAUNCH_FIELDS = ("paired_cells", "rest_cells", "paired_useful_cells", "rest_useful_cells", "planned_paired_cells",
                 "planned_paired_useful_cells", "n_pairs", "n_rest")


@functools.lru_cache(maxsize=None)
def dataset(name):
    """-> list of (left, right, motif, T, cores, kmin, kmax) per region; bounds from the round-1 sizes."""
    if name == "cfg1":
        regs = synth.config1(seed=11, n_regions=6, reads_per_region=20)
        # a region whose left anchor holds an N: not scored in either round, its reads count as skipped
        bad = synth.make_region(np.random.default_rng(12), "cfg1_n", "AAAG", [12, 20], 10, "ont_q20")
        bad.left_anchor_seq = bad.left_anchor_seq[:500] + "N" + bad.left_anchor_seq[501:]
        regs.insert(3, bad)
    elif name == "cfg2":
        regs = synth.config2(seed=12, n_reads=300)
    elif name == "cfg4":
        regs = synth.config4(seed=14, reads_per_locus=16)
    elif name == "cfg5":
        # a config-5 sample: short and medium regions, and one of 2 000 six-base units (reads up to 12.6 kb)
        regs = synth.config5(seed=15, n_reads=400, reads_per_region=10, k_max=400)
        rng = np.random.default_rng(16)
        regs.append(synth.make_region(rng, "cfg5_long", "ACGGTC", [2000, 1600], 9, "clr"))
        regs.append(synth.make_region(rng, "cfg5_mid", "TTAGG", [700, 650], 7, "ont"))
    else:
        raise KeyError(name)
    out = []
    for reg in regs:
        m = len(reg.repeat_unit_seq)
        r1 = np.array(reg.dist_between_anchors, dtype=np.float64) / m
        r1max = float(r1.max())
        T = int(r1max * 1.5) + 1
        if T < r1max + 10:
            T = int(r1max + 10)
        kmin, kmax = ladder_bounds_array(np.maximum(r1, 0.0), False)
        out.append((reg.left_anchor_seq, reg.right_anchor_seq, reg.repeat_unit_seq, T, list(reg.core_seqs), kmin, kmax))
    return out


class knobs:
    """Environment knobs read at commit time, and the process-wide ladder mode."""

    def __init__(self, env=None, mode=3):
        self.env, self.mode = dict(env or {}), mode

    def __enter__(self):
        self.old = {k: os.environ.get(k) for k in self.env}
        os.environ.update(self.env)
        engine.set_ladder_mode(self.mode)

    def __exit__(self, *exc):
        for k, v in self.old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
        engine.set_ladder_mode(3)


def fingerprint(b):
    li = b.launch_info()
    return {"stats": b.stats(), "launch": {k: int(li[k]) for k in LAUNCH_FIELDS}}


def round2(data, kind, env=None):
    sc = engine.get_preset("ont")
    with knobs(env):
        with engine.Batch.begin(sc, kind) as b:
            for left, _right, motif, T, cores, _lo, _hi in data:
                b.add_round2(left, motif, T, cores)
            return [fingerprint(b.commit())]


def round3(data, mode, env=None):
    sc = engine.get_preset("ont")
    with knobs(env, mode):
        with engine.Batch.begin(sc, "round3") as b:
            for left, right, motif, _T, cores, lo, hi in data:
                b.add_round3(left, right, motif, cores, lo, hi)
            return [fingerprint(b.commit())]


def resumed(data, mode, env=None):
    """Round 2 on flag words, then round 3 over its reads (nr_batch_begin_round3_from / nr_batch_add_round3_reuse)."""
    sc = engine.get_preset("ont")
    with knobs(env, mode):
        with engine.Batch.begin(sc, "round2_flags") as b2:
            for left, _right, motif, T, cores, _lo, _hi in data:
                b2.add_round2(left, motif, T, cores)
            b2.commit()
            with engine.Batch.begin_round3_from(b2) as b3:
                for i, (_left, right, _motif, _T, _cores, lo, hi) in enumerate(data):
                    b3.add_round3_reuse(i, right, lo, hi)
                return [fingerprint(b2), fingerprint(b3.commit())]


def tasks():
    """What Step 1's second launch makes: anchors against read windows and whole reads, some of them with an N."""
    sc = engine.get_preset("ont")
    qs, ts = [], []
    for left, right, _motif, _T, cores, _lo, _hi in dataset("cfg1") + dataset("cfg5")[-2:]:
        for i, core in enumerate(cores[:4]):
            qs.append(left if i % 2 == 0 else right)
            ts.append(core if i != 3 else core[:40] + "N" + core[41:])
    qs.append(dataset("cfg5")[-2][4][0])                # a long query: cut into stripes
    ts.append(dataset("cfg5")[-2][0] + dataset("cfg5")[-2][4][0])
    with knobs():
        with engine.Batch.tasks(sc, qs, ts) as b:
            return [fingerprint(b)]


def cases():
    """name -> function that returns the fingerprints of the case's committed batches."""
    out = {}
    for ds in ("cfg1", "cfg2", "cfg4", "cfg5"):
        d = functools.partial(dataset, ds)
        out[f"{ds}-round2"] = lambda d=d: round2(d(), "round2")
        out[f"{ds}-round2_flags"] = lambda d=d: round2(d(), "round2_flags")
        out[f"{ds}-round2_flags-exit0"] = lambda d=d: round2(d(), "round2_flags", {"NR_ROUND2_EXIT": "0"})
        for mode in range(4):
            out[f"{ds}-round3-mode{mode}"] = lambda d=d, mode=mode: round3(d(), mode)
        for mode in (1, 2, 3):
            out[f"{ds}-resumed-mode{mode}"] = lambda d=d, mode=mode: resumed(d(), mode)
        out[f"{ds}-resumed-exit0"] = lambda d=d: resumed(d(), 3, {"NR_ROUND2_EXIT": "0"})
    for ds in ("cfg4", "cfg5"):
        d = functools.partial(dataset, ds)
        for tag, env in (("no_long_pairs", {"NR_NO_LONG_PAIRS": "1"}), ("coop_rows4", {"NR_COOP_ROWS": "4"}),
                         ("coop_rows12", {"NR_COOP_ROWS": "12"})):
            out[f"{ds}-resumed-{tag}"] = lambda d=d, env=env: resumed(d(), 3, env)
            out[f"{ds}-round3-mode3-{tag}"] = lambda d=d, env=env: round3(d(), 3, env)
            out[f"{ds}-round3-mode2-{tag}"] = lambda d=d, env=env: round3(d(), 2, env)
    out["tasks"] = tasks
    return out


def main():
    engine.lib()
    engine.init(0)
    fixture = {"sm_count": engine.device_info()["sm_count"], "cases": {k: f() for k, f in cases().items()}}
    with open(OUT, "w") as f:
        json.dump(fixture, f, indent=1, sort_keys=True)
        f.write("\n")
    print(f"{len(fixture['cases'])} cases -> {OUT}")


if __name__ == "__main__":
    main()
