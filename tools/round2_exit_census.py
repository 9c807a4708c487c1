"""CPU census of round 2's dominance exit (DESIGN.md section 4.9): the share of round-2 DP cells that need not be
swept because every column right of some cut is dominated by the column one period earlier.

Full DP per read (tools/round2_exit_census.c, compiled into a temporary directory), the bench's T rule, checks every
P = lcm(16, |motif|) columns from the column the library starts checking at (|left| + read length + OFFSET, the
host's rule in nr_api.cu).  Prints the skippable fraction per region and per config.

    python tools/round2_exit_census.py [--configs 2,3,5] [--offset -192] [--loci 300] [--reads5 2000]
"""
import argparse
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from nanorepeat_b200 import synth  # noqa: E402


def bench_T(reg):
    m = len(reg.repeat_unit_seq)
    r1max = max(float(d) / m for d in reg.dist_between_anchors)
    T = int(r1max * 1.5) + 1
    return int(r1max + 10) if T < r1max + 10 else T


def regions(cfg, loci, reads5):
    if cfg == 2:
        return synth.config2(seed=2)
    if cfg == 3:
        return synth.config3(seed=3, n_loci=loci)
    if cfg == 5:
        return synth.config5(seed=5, n_reads=reads5)
    raise ValueError(cfg)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="2,3,5")
    ap.add_argument("--offset", type=int, default=-192, help="first checked column = |left| + read length + offset")
    ap.add_argument("--loci", type=int, default=300, help="config 3: loci in the slice")
    ap.add_argument("--reads5", type=int, default=2000, help="config 5: reads in the slice")
    ap.add_argument("--per-region", action="store_true")
    a = ap.parse_args()
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "census")
        subprocess.check_call(["cc", "-O2", "-o", exe, os.path.join(ROOT, "tools", "round2_exit_census.c")])
        for cfg in (int(c) for c in a.configs.split(",")):
            regs = [r for r in regions(cfg, a.loci, a.reads5) if r.left_anchor_seq and r.core_seqs]
            lines = []
            for reg in regs:
                lines.append(f"R {reg.left_anchor_seq} {reg.repeat_unit_seq} {bench_T(reg)} {len(reg.core_seqs)} {a.offset}")
                lines.extend(reg.core_seqs)
            out = subprocess.run([exe], input="\n".join(lines) + "\n", capture_output=True, text=True, check=True).stdout
            tot = skip = 0
            for reg, line in zip(regs, out.splitlines()):
                f = line.split()
                cells, skipped, n = int(f[1]), int(f[3]), int(f[7])
                tot += cells; skip += skipped
                if a.per_region or len(regs) <= 4:
                    print(f"config {cfg} {reg.name}: |L|={len(reg.left_anchor_seq)} m={len(reg.repeat_unit_seq)} "
                          f"T={bench_T(reg)} reads={n}: round-2 cells {cells:.3e}, skippable {100.0 * skipped / cells:.1f} %, "
                          f"mean exit column |L| + {int(f[5]) / n:.0f}")
            print(f"config {cfg} total: round-2 cells {tot:.4e}, skippable {100.0 * skip / max(tot, 1):.1f} % "
                  f"(checks every lcm(16, m) columns from |L| + read length {a.offset:+d})", flush=True)


if __name__ == "__main__":
    main()
