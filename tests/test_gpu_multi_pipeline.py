"""Steps 1-4 sharded on real GPUs (sharding.quantify_regions_sharded): one rank equals pipeline.quantify_regions; the
phasing of a region list equals the same list phased in two calls with the right region_id_base (the premise of the
sharded Step 4); two ranks on two GPUs under torchrun equal one quantify_regions call (needs two visible GPUs; with one
the test says so)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers.pipeline_state import first_difference, region_state, value

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _regions():
    import nanorepeat_b200 as nrb
    from nanorepeat_b200 import synth
    regions, reads = [], []
    for g, (motif, n) in enumerate((("CAG", 40), ("GGGGCC", 25), ("AT", 1), ("CAG", 0), ("TTTCA", 30), ("CAG", 300))):
        reg, names, seqs, _t = synth.region_reads(seed=80 + g, n_reads=max(n, 1), motif=motif, alleles=(14 + g, 35 + g))
        rr = nrb.RepeatRegion()
        rr.left_anchor_seq, rr.right_anchor_seq, rr.repeat_unit_seq = reg.left_anchor_seq, reg.right_anchor_seq, motif
        regions.append(rr); reads.append((names[:n], seqs[:n]))
    return regions, reads


def test_one_rank_equals_quantify_regions(engine):
    import nanorepeat_b200 as nrb
    from nanorepeat_b200 import sharding
    want, reads = _regions()
    nrb.quantify_regions(want, reads, phase=True)
    got, reads2 = _regions()
    mine = sharding.quantify_regions_sharded(got, reads2, phase=True, max_reads_per_piece=64, world_size=1)
    a, b = [region_state(rr) for rr in got], [region_state(rr) for rr in want]
    assert a == b, first_difference(a, b)
    assert mine == list(range(len(sharding.cut_pieces(reads, 64))))
    assert sum(len(rr.read_dict) for rr in want) > 250 and sum(rr.allele_list is not None for rr in want) >= 3


def test_phasing_in_blocks_equals_one_call(engine):
    from nanorepeat_b200 import phasing
    rng = np.random.default_rng(5)
    sizes = []
    for g in range(9):
        n = (1, 40, 7, 60, 0, 25, 33, 2, 50)[g]
        a, b = 10 + 3 * g, 30 + 5 * g
        sizes.append({f"r{i}": float(rng.normal(a if i % 2 else b, 0.6)) for i in range(n)})
    params = engine.GmmParams(error_rate=0.07, max_mutual_overlap=0.15, max_components=22, seed=3)
    lists = [list(d.values()) for d in sizes]
    whole = engine.phase_1d(params, lists)
    whole_alleles = phasing.phase_regions_1d(sizes, 2, 0.07, 0.15, -1, True, 3)
    for cut in (1, 4, 8):
        parts = engine.phase_1d(params, lists[:cut]) + engine.phase_1d(params, lists[cut:], region_id_base=cut)
        for x, y in zip(whole, parts):
            assert x["n"] == y["n"]
            for k in ("weights", "means", "variances", "label", "proba"):
                assert np.array_equal(x[k], y[k]), (cut, k)
        alleles = (phasing.phase_regions_1d(sizes[:cut], 2, 0.07, 0.15, -1, True, 3) +
                   phasing.phase_regions_1d(sizes[cut:], 2, 0.07, 0.15, -1, True, 3, region_id_base=cut))
        assert [None if r is None else ([value(a) for a in r[0]], r[1]) for r in alleles] == \
               [None if r is None else ([value(a) for a in r[0]], r[1]) for r in whole_alleles]
    assert sum(x["n"] >= 2 for x in whole) >= 5


def test_two_ranks_on_two_gpus_equal_quantify_regions():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs (the multi-rank logic is covered on CPU by tests/test_sharding_pipeline.py)")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29619",
                          os.path.join(ROOT, "tests", "helpers", "sharded_pipeline_ranks.py")],
                         capture_output=True, text=True, timeout=1200)
    assert out.returncode == 0, out.stderr[-3000:]
    res = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
    assert res["equal"], res
    assert res["disjoint"] and min(res["pieces_per_rank"]) >= 1, res
    assert res["big_region_pieces"] == 3 and res["repeated_name_region_pieces"] == 1 and res["unscored_pieces"] == [0, 1, 2], res
    assert res["accepted_reads"] > 4000 and res["phased_regions"] >= 6, res
