#!/usr/bin/env python
"""Steps 1-4 from raw reads on one GPU (pipeline.quantify_regions) and sharded over ranks (sharding.quantify_regions_sharded,
one process per rank under torch.distributed.run, started here on a free port) for two shapes of tools/step1_bench.py:
the 2 000-locus x 30-read catalog slice and config 2's shape (2 amplicon regions x 5 000 reads).

Per run: the wall time of every pass (fresh RepeatRegion objects each pass, built outside the timed region; a barrier
before each pass; a pass's time is the slowest rank's), and per rank its wall time in Step 1 (cut, deal, anchors,
cores), the T exchange, rounds 1-3, the gather (exchange, rebuilding every region, cutting every core) and the phasing,
with its Step-1 cells and predicted round-1-3 cells (the balance).  The one-GPU run reports Step 1 (the anchor call),
rounds 1-3 and the phasing the same way.  Every sharded run compares all its regions -- every Read attribute with its
type, the cores, buffer_len, the alleles -- with the one-GPU run and the script exits 1 when one differs.  Ranks go to
GPU local_rank mod the visible count: with fewer GPUs than ranks (--ranks) they share, and the JSON says so.
Writes one JSON document (--out) with the card name, power limit and SM clock read in the same run."""
import argparse
import json
import os
import pickle
import signal
import socket
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

SHAPES = ("catalog_2000x30", "config2_2x5000")


def _value(v):
    if hasattr(v, "__slots__"):
        return type(v), [(k, type(getattr(v, k)), getattr(v, k)) for k in v.__slots__]
    if hasattr(v, "__dict__"):
        return type(v), [(k, type(x), x) for k, x in sorted(vars(v).items())]
    return type(v), v


def _state(rr):
    """Everything quantify_regions leaves on a region, with the type of every value."""
    alleles = getattr(rr, "allele_list", None)
    return (sorted(vars(rr)), [(n, [(k, _value(v)) for k, v in sorted(vars(rd).items())]) for n, rd in rr.read_dict.items()],
            list(rr.read_core_seq_dict.items()), getattr(rr, "buffer_len", None),
            [_value(a) for a in alleles] if alleles else alleles, getattr(rr, "num_removed_reads", None))


def _timed(fn, stats, key):
    def run(*a, **kw):
        t0 = time.perf_counter()
        out = fn(*a, **kw)
        stats[key] = stats.get(key, 0.0) + time.perf_counter() - t0
        return out
    return run


def worker(args):
    import torch
    import torch.distributed as dist
    import nanorepeat_b200 as nrb
    from nanorepeat_b200 import anchoring, engine, phasing, pipeline, sharding
    from step1_bench import shapes
    world, rank, local = int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0))
    if world > 1:
        dist.init_process_group("gloo")
    device = local % torch.cuda.device_count()
    engine.init(device)
    data = shapes()
    out = {}
    for shape in SHAPES:
        regs = data[shape]
        reads = [([f"read{i}" for i in range(len(seqs))], seqs) for _l, _r, seqs, _m in regs]
        walls, stats = [], []
        for p in range(args.warmup + args.reps):
            regions = []
            for left, right, _seqs, motif in regs:
                rr = nrb.RepeatRegion()
                rr.left_anchor_seq, rr.right_anchor_seq, rr.repeat_unit_seq = left, right, motif
                regions.append(rr)
            st = {}
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            if world == 1:
                pipeline.quantify_regions(regions, reads, phase=True,
                                          anchor_fn=_timed(anchoring.find_anchor_locations_in_regions, st, "step1_anchor_s"),
                                          estimate_fn=_timed(nrb.estimate_regions, st, "rounds_s"),
                                          phase_fn=_timed(phasing.phase_regions_1d, st, "phase_s"))
            else:
                sharding.quantify_regions_sharded(regions, reads, phase=True, stats=st)
            wall = time.perf_counter() - t0
            if p >= args.warmup:
                walls.append(wall)
                stats.append(st)
        states = [_state(rr) for rr in regions]
        base = os.path.join(args.tmp, shape + ".baseline.pkl")
        equal = None
        if world == 1:
            with open(base, "wb") as f:
                pickle.dump(states, f, protocol=pickle.HIGHEST_PROTOCOL)
        else:
            with open(base, "rb") as f:
                equal = pickle.load(f) == states
        mine = dict(rank=rank, device=device, wall_s=walls, equal=equal,
                    phases_s={k: [s[k] for s in stats] for k in stats[0] if k.endswith("_s")},
                    loads={k: stats[0][k] for k in stats[0] if not k.endswith("_s")})
        ranks = [mine]
        if world > 1:
            ranks = [None] * world
            dist.all_gather_object(ranks, mine)
        out[shape] = dict(regions=len(regs), reads=sum(len(s) for _l, _r, s, _m in regs),
                          accepted_reads=sum(len(rr.read_dict) for rr in regions),
                          pass_ms=[1e3 * max(r["wall_s"][i] for r in ranks) for i in range(args.reps)],
                          equal_to_one_gpu=all(r["equal"] for r in ranks) if world > 1 else None, ranks=ranks)
        if rank == 0:
            print(f"world {world} {shape}: pass ms {[round(x, 1) for x in out[shape]['pass_ms']]} "
                  f"equal {out[shape]['equal_to_one_gpu']}", flush=True)
    if rank == 0:
        with open(os.path.join(args.tmp, f"world{world}.json"), "w") as f:
            json.dump(dict(world=world, gpus_visible=torch.cuda.device_count(), shapes=out), f)
    if world > 1:
        dist.destroy_process_group()


def _run(cmd, timeout):
    """Run cmd in its own process group; on a timeout the whole group (torchrun and every rank) is killed."""
    proc = subprocess.Popen(cmd, cwd=ROOT, start_new_session=True)
    try:
        rc = proc.wait(timeout=timeout)
    except subprocess.TimeoutExpired:
        os.killpg(proc.pid, signal.SIGKILL)
        proc.wait()
        raise
    if rc != 0:
        raise SystemExit(f"{cmd[:6]} ... exited {rc}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--ranks", type=int, nargs="*", help="world sizes (default: 2, 4, 8 up to the visible GPU count)")
    ap.add_argument("--timeout", type=int, default=1500, help="seconds per run")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_pipeline_sharded_bench.json"))
    ap.add_argument("--worker", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--tmp", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.worker:
        return worker(args)

    def smi():
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, check=True).stdout.strip().splitlines()
    cards = smi()
    n_gpu = len(cards)
    worlds = args.ranks if args.ranks else [w for w in (2, 4, 8) if w <= n_gpu]
    with tempfile.TemporaryDirectory(prefix="pipeline_sharded_bench_") as tmp:
        common = [os.path.abspath(__file__), "--worker", "--tmp", tmp, "--reps", str(args.reps), "--warmup", str(args.warmup)]
        _run([sys.executable] + common, args.timeout)
        for w in worlds:
            s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
            _run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(w), "--master-addr",
                  "127.0.0.1", "--master-port", str(port)] + common, args.timeout)
        runs = {}
        for w in [1] + worlds:
            with open(os.path.join(tmp, f"world{w}.json")) as f:
                runs[w] = json.load(f)
    first = cards[0].split(", ")
    doc = dict(gpu=first[0], gpus_visible=n_gpu, power_limit=first[1], sm_clock_max=first[2],
               sm_clock_at_start=[c.split(", ")[3] for c in cards], sm_clock_at_end=[c.split(", ")[3] for c in smi()],
               host_cpus=os.cpu_count(), reps=args.reps, warmup=args.warmup,
               runs={str(w): dict(r, ranks_per_gpu=max(1, -(-w // n_gpu))) for w, r in runs.items()})
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(doc, f, indent=1)
    bad = [(w, s) for w in worlds for s, v in runs[w]["shapes"].items() if not v["equal_to_one_gpu"]]
    if bad:
        raise SystemExit(f"sharded runs differ from the one-GPU run: {bad}")
    print("all sharded runs equal the one-GPU run;", args.out)


if __name__ == "__main__":
    main()
