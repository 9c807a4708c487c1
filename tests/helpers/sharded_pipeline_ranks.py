"""Run under torchrun by tests/test_gpu_multi_pipeline.py: Steps 1-4 of one raw-read workload split over the ranks by
sharding.quantify_regions_sharded (each rank its own GPU); rank 0 compares every region with one
pipeline.quantify_regions(phase=True) call on its GPU and prints a JSON verdict.  --one-gpu puts every rank on GPU 0
(a functional check on a box with one GPU)."""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

import numpy as np                                   # noqa: E402
import torch.distributed as dist                     # noqa: E402
import nanorepeat_b200 as nrb                        # noqa: E402
from nanorepeat_b200 import engine, sharding, synth  # noqa: E402
from helpers.pipeline_state import region_state, first_difference  # noqa: E402

MAX_READS = 2048


def workload():
    """config-1-like regions; a config-2-sized region cut into three pieces, with reads Step 1 leaves unscored (one
    holding N, one over 65 471 bases, an empty one) in different pieces; a region with a repeated read name; a region
    whose left anchor holds an N."""
    rng = np.random.default_rng(17)
    regions, reads = [], []

    def add(reg, names, seqs, left=None):
        rr = nrb.RepeatRegion()
        rr.left_anchor_seq, rr.right_anchor_seq, rr.repeat_unit_seq = left or reg.left_anchor_seq, reg.right_anchor_seq, reg.repeat_unit_seq
        regions.append(rr); reads.append((list(names), list(seqs)))

    for g, motif in enumerate(("CAG", "GGGGCC", "AT", "TTTCA", "CAG", "CCG")):
        add(*synth.region_reads(seed=60 + g, n_reads=30, motif=motif, alleles=(12 + g, 40 + 2 * g))[:3])
    reg, names, seqs, _t = synth.region_reads(seed=70, n_reads=5000, motif="CAG", alleles=(20, 40), outer=150)
    names, seqs = list(names), list(seqs)
    seqs[100] = seqs[100][:300] + "N" + seqs[100][301:]
    seqs[2100] = synth.random_seq(rng, 70000)
    seqs[4500] = ""
    add(reg, names, seqs)
    reg, names, seqs, _t = synth.region_reads(seed=71, n_reads=40, motif="CAG", alleles=(15, 33))
    names = list(names)
    names[7], names[20] = names[3], names[11]
    add(reg, names, seqs)
    reg, names, seqs, _t = synth.region_reads(seed=72, n_reads=25, motif="CAG", alleles=(18, 30))
    add(reg, names, seqs, left=reg.left_anchor_seq[:400] + "N" + reg.left_anchor_seq[401:])
    return regions, reads


def main():
    rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    dist.init_process_group("gloo")                  # the only collectives are host-side exchanges
    device = 0 if "--one-gpu" in sys.argv else local
    engine.init(device)
    assert engine.device_info()["device"] == device
    regions, reads = workload()
    mine = sharding.quantify_regions_sharded(regions, reads, phase=True, max_reads_per_piece=MAX_READS)
    got = [region_state(rr) for rr in regions]
    all_mine = [None] * dist.get_world_size()
    dist.all_gather_object(all_mine, mine)
    states = [None] * dist.get_world_size()
    dist.all_gather_object(states, got)
    if rank == 0:
        whole, whole_reads = workload()
        nrb.quantify_regions(whole, whole_reads, phase=True)
        want = [region_state(rr) for rr in whole]
        spans = sharding.cut_pieces(whole_reads, MAX_READS)
        big = [s for s in spans if s[0] == 6]
        print(json.dumps({
            "equal": all(s == want for s in states),
            "difference": next((d for d in (first_difference(s, want) for s in states) if d), None),
            "pieces_per_rank": [len(m) for m in all_mine],
            "disjoint": sorted(i for m in all_mine for i in m) == list(range(len(spans))),
            "big_region_pieces": len(big), "repeated_name_region_pieces": sum(s[0] == 7 for s in spans),
            "unscored_pieces": sorted({next(k for k, (_r, a, b) in enumerate(big) if a <= i < b) for i in (100, 2100, 4500)}),
            "accepted_reads": sum(len(rr.read_dict) for rr in whole),
            "phased_regions": sum(rr.allele_list is not None for rr in whole),
            "anchor_n_region_reads": len(whole[8].read_dict)}))
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
