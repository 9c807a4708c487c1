"""Steps 1-4 sharded (sharding.quantify_regions_sharded / anchor_regions_sharded) on CPU: gloo ranks in spawned
processes, with the three library-backed steps replaced by stand-ins -- Step 1 built on oracle/anchoring.records and
filled through the helper the library path uses, rounds 1-3 on oracle/selection, and a phasing that answers with the
region id it was given -- so that cutting, dealing, the T exchange, the gather and the phasing blocks are checked
against one single-process pipeline.quantify_regions call without a GPU."""
import os
import socket
import sys

import numpy as np
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import ROOT
from helpers.pipeline_state import region_state

PHASE_CALLS = []          # region ids each phase stand-in call was given, in this process


def _oracle_anchor(data_type, regions, region_reads):
    """Same contract as anchoring.find_anchor_locations_in_regions, the alignments by the oracle."""
    from nanorepeat_b200 import anchoring
    from oracle import anchoring as oanchor
    for rr, reads in zip(regions, region_reads):
        names, seqs = anchoring._reads_of(rr, reads)
        acc = [(n, o) for n, o in zip(names, oanchor.records(rr.left_anchor_seq, rr.right_anchor_seq, seqs)) if o["accepted"]]
        col = {f: [] for f in anchoring.STEP1_FIELDS}
        for _n, o in acc:
            for f in ("read_len", "dist_between_anchors", "core_start", "core_end", "mid_start", "mid_end", "left_buffer",
                      "right_buffer"):
                col[f].append(o[f])
            for f in ("strand", "left_strand", "right_strand"):
                col[f].append(ord(o[f]))
            for side in ("left", "right"):
                for f, v in zip(("score", "tstart", "tend"), o[side]):
                    col[side + f].append(v)
        anchoring.add_accepted_reads(rr, [n for n, _o in acc], col, range(len(acc)))


def _oracle_estimate(regions, data_type=None, fast_mode=False):
    """Same contract as nanorepeat_b200.estimate_regions (round1_max_dist honoured), computed by the oracle."""
    from oracle import selection
    for rr in regions:
        names = [n for n in rr.read_dict if n in rr.read_core_seq_dict]
        if not names:
            continue
        m = len(rr.repeat_unit_seq)
        dists = [rr.read_dict[n].dist_between_anchors for n in names]
        res = selection.estimate_region(rr.left_anchor_seq, rr.right_anchor_seq, rr.repeat_unit_seq,
                                        [rr.read_core_seq_dict[n] for n in names], dists, fast_mode=fast_mode,
                                        n_threads=2, max_dist=getattr(rr, "round1_max_dist", None))
        for i, n in enumerate(names):
            rd = rr.read_dict[n]
            rd.round1_repeat_size = float(dists[i]) / m
            rd.round2_repeat_size = res["r2"][i]
            rd.round3_repeat_size = res["r3"][i]


def _phase_by_id(sizes, ploidy=2, error_rate=0.07, max_mutual_overlap=0.15, max_num_components=-1,
                 remove_noisy_reads=False, seed=0, region_id_base=0):
    """phasing.phase_regions_1d's shape; the answer names the region id and the sizes it was given."""
    ids = list(range(region_id_base, region_id_base + len(sizes)))
    PHASE_CALLS.append(ids)
    return [None if len(d) < 2 else ([("region", g, seed), sorted((k, float(v)) for k, v in d.items())], g % 3)
            for g, d in zip(ids, sizes)]


def _workload():
    """(regions, reads): synth.region_reads regions (200-base anchors, so that the oracle is quick), plus a region with
    no accepted read, one with no reads, one with a repeated read name and one whose longest dist is in its last read."""
    import nanorepeat_b200 as nrb
    from nanorepeat_b200 import synth

    def region(reg):
        rr = nrb.RepeatRegion()
        rr.left_anchor_seq, rr.right_anchor_seq, rr.repeat_unit_seq = reg.left_anchor_seq, reg.right_anchor_seq, reg.repeat_unit_seq
        return rr

    kw = dict(flank=200, outer=300)
    regions, reads = [], []
    for seed, motif, alleles, n in ((31, "CAG", (12, 30), 23), (32, "GGGGCC", (5, 14), 17), (33, "AT", (20,), 9)):
        reg, names, seqs, _t = synth.region_reads(seed=seed, n_reads=n, motif=motif, alleles=alleles, **kw)
        regions.append(region(reg)); reads.append((names, seqs))
    rng = np.random.default_rng(7)
    reg, _n, _s, _t = synth.region_reads(seed=36, n_reads=1, **kw)
    regions.append(region(reg)); reads.append(([f"junk{i}" for i in range(6)], [synth.random_seq(rng, 800) for _ in range(6)]))
    regions.append(region(reg)); reads.append(([], []))
    reg, names, seqs, _t = synth.region_reads(seed=34, n_reads=12, motif="CAG", alleles=(10, 25), **kw)
    names = list(names)
    names[5], names[9] = names[2], names[0]
    regions.append(region(reg)); reads.append((names, seqs))
    # the right anchor starts with 30 of the reads' 40 repeat units, so a core holds more units than its dist says and
    # round 2 sees the template's length: T must come from the region's longest dist, in the region's last read
    reg, names, seqs, _t = synth.region_reads(seed=35, n_reads=13, motif="CAG", alleles=(40,), **kw)
    _reg, names2, seqs2, _t = synth.region_reads(seed=35, n_reads=1, motif="CAG", alleles=(80,), **kw)
    rr = region(reg)
    rr.right_anchor_seq = "CAG" * 30 + reg.right_anchor_seq[:110]
    regions.append(rr); reads.append((names + ["long0"], seqs + seqs2))
    return regions, reads


def _single(max_reads=None, sharded=False):
    from nanorepeat_b200 import pipeline, sharding
    regions, reads = _workload()
    kw = dict(phase=True, anchor_fn=_oracle_anchor, estimate_fn=_oracle_estimate, phase_fn=_phase_by_id)
    if sharded:
        mine = sharding.quantify_regions_sharded(regions, reads, max_reads_per_piece=max_reads, **kw)
    else:
        mine = None
        pipeline.quantify_regions(regions, reads, **kw)
    return [region_state(rr) for rr in regions], mine


def _worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from nanorepeat_b200 import sharding
    out = {}
    for max_reads in (4, 7):
        regions, reads = _workload()
        PHASE_CALLS.clear()
        mine = sharding.quantify_regions_sharded(regions, reads, phase=True, max_reads_per_piece=max_reads,
                                                 anchor_fn=_oracle_anchor, estimate_fn=_oracle_estimate,
                                                 phase_fn=_phase_by_id)
        out[max_reads] = (mine, [region_state(rr) for rr in regions], list(PHASE_CALLS))
    regions, reads = _workload()
    mine = sharding.anchor_regions_sharded(regions, reads, max_reads_per_piece=4, gather=False, anchor_fn=_oracle_anchor)
    out["local"] = (mine, [(list(rr.read_dict), dict(rr.read_core_seq_dict)) for rr in regions])
    q.put((rank, out))
    dist.barrier()
    dist.destroy_process_group()


def _run(world):
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = [q.get(timeout=600) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    return [out for _r, out in sorted(got, key=lambda x: x[0])]


def _check_world(world, oracle):
    from nanorepeat_b200 import sharding
    expect, _ = _single()
    assert sum(len(e["reads"]) for e in expect) > 40
    r3_types = [dict(a)["round3_repeat_size"][0] for e in expect for _n, a in e["reads"]]
    assert r3_types.count(np.float64) > 10 and r3_types.count(float) + r3_types.count(type(None)) > 0
    dists = {n: dict(a)["dist_between_anchors"][1] for n, a in expect[6]["reads"]}
    assert "long0" in dists and dists["long0"] > max(d for n, d in dists.items() if n != "long0")   # in the last piece
    assert expect[3]["reads"] == [] and expect[4]["reads"] == [] and expect[3]["alleles"] is None
    outs = _run(world)
    regions, reads = _workload()
    for max_reads in (4, 7):
        spans = sharding.cut_pieces(reads, max_reads)
        mines = [out[max_reads][0] for out in outs]
        assert all(mines) and sorted(i for m in mines for i in m) == list(range(len(spans)))     # disjoint, all, none empty
        for out in outs:
            assert out[max_reads][1] == expect                       # every rank ends with the single-process result
        ids = [i for out in outs for call in out[max_reads][2] for i in call]
        assert ids == list(range(len(regions)))                      # contiguous blocks, in rank order
        assert all(call == list(range(call[0], call[0] + len(call))) for out in outs for call in out[max_reads][2])
    # gather=False: a rank holds its own pieces' reads; together the ranks hold Step 1's whole answer
    spans = sharding.cut_pieces(reads, 4)
    for r, (e, rr_reads) in enumerate(zip(expect, reads)):
        held = [out["local"][1][r] for out in outs]
        assert sorted(n for keys, _c in held for n in keys) == sorted(n for n, _a in e["reads"])
        for out, (keys, cores) in zip(outs, held):
            own = {n for i in out["local"][0] if spans[i][0] == r for n in rr_reads[0][spans[i][1]:spans[i][2]]}
            assert set(keys) <= own and cores == {n: c for n, c in e["cores"] if n in keys}


def test_two_ranks_equal_single_process(oracle):
    _check_world(2, oracle)


def test_three_ranks_equal_single_process(oracle):
    _check_world(3, oracle)


def test_one_rank_without_process_group_is_quantify_regions(oracle):
    from nanorepeat_b200 import sharding
    expect, _ = _single()
    got, mine = _single(max_reads=4, sharded=True)
    assert got == expect
    _regions, reads = _workload()
    assert mine == list(range(len(sharding.cut_pieces(reads, 4))))


def test_pieces_and_dealing_are_deterministic():
    from nanorepeat_b200 import sharding
    regions, reads = _workload()
    spans = sharding.cut_pieces(reads, 4)
    assert spans == sharding.cut_pieces(reads, 4)
    assert [s for s in spans if s[0] == 0] == [(0, 0, 4), (0, 4, 8), (0, 8, 12), (0, 12, 16), (0, 16, 20), (0, 20, 23)]
    assert [s for s in spans if s[0] == 4] == []                     # no reads, no piece
    assert [s for s in spans if s[0] == 5] == [(5, 0, 12)]           # a repeated name: one piece, more than 4 reads
    costs = [2 * (len(regions[r].left_anchor_seq) + len(regions[r].right_anchor_seq)) * sum(map(len, reads[r][1][s:e]))
             for r, s, e in spans]
    for world in (2, 3):
        assert sharding.partition(costs, world) == sharding.partition(costs, world)
    assert spans[-1] == (6, 12, 14) and sharding.cut_pieces(reads, 7)[-1] == (6, 7, 14)
    assert sharding._phase_blocks([3, 3, 3, 3], 2) == [(0, 2), (2, 4)]
    assert sharding._phase_blocks([0, 0], 3) == [(0, 1), (1, 1), (1, 2)]
    assert sharding._phase_blocks([5, 0, 1, 1, 1, 1, 1], 2) == [(0, 1), (1, 7)]
