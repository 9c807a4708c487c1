"""Step 1 for many regions in one call (nr_anchor_regions: anchor pairs on u16x2 words + start recovery) against
(a) the CPU restatement oracle/anchoring.step1 and (b) the per-region rules of the previous Python layer, restated here
over engine.score_tasks (four exact alignments per read, one library call per region)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

COMP = str.maketrans("ACGTacgtNn", "TGCAtgcaNn")


def rc(s):
    return s.translate(COMP)[::-1]


def per_region_rules(engine, left, right, names, seqs):
    """The per-region path as it was: score_tasks over (anchor, strand) and the reference's rules in Python."""
    sc = engine.get_preset("ont")
    q, t = [], []
    for s in seqs:
        q += [left, left, right, right]
        t += [s, rc(s), s, rc(s)]
    recs = engine.score_tasks(q, t, sc) if q else []
    out = {}
    for r, (name, seq) in enumerate(zip(names, seqs)):
        best = []
        for a in range(2):
            hits = []
            for sd, strand in enumerate("+-"):
                rec = recs[4 * r + 2 * a + sd]
                if rec["score"] > 0 and rec["score"] >= sc.min_dp_score:
                    hits.append((int(rec["score"]), strand, int(rec["tstart"]), int(rec["tend"])))
            hits.sort(key=lambda h: h[0], reverse=True)
            ok = len(hits) == 1 or (len(hits) == 2 and hits[0][3] - hits[0][2] >= 10 and hits[0][0] > 1.5 * hits[1][0])
            best.append(hits[0] if ok else None)
        if best[0] is None or best[1] is None:
            continue
        (ls, lst, lqs, lqe), (rs, rst, rqs, rqe) = best
        dist = rqs - lqe if lst == rst else 0
        if not dist > -10:
            continue
        cs, ce = max(lqe - 100, 0), min(rqs + 100, len(seq))
        oriented = rc(seq) if lst == "-" else seq
        out[name] = dict(strand=lst, dist=dist, core_start=cs, core_end=ce, mid_start=lqe, mid_end=rqs, left_buffer=lqe - cs,
                         right_buffer=ce - rqs, core=oriented[cs:ce], left=(lst, ls, lqs, lqe), right=(rst, rs, rqs, rqe))
    return out


def build_cases():
    from nanorepeat_b200 import synth
    rng = np.random.default_rng(41)
    regions = []            # (left, right, names, seqs)
    for seed, motif, alleles, n in ((6, "CAG", (17, 55), 33), (7, "GGGGCC", (8, 60), 20), (8, "AT", (12,), 1), (9, "CAG", (20,), 0),
                                    (10, "TTTCA", (9, 30), 25)):
        reg, names, seqs, _truth = synth.region_reads(seed=seed, n_reads=max(n, 1), motif=motif, alleles=alleles)
        regions.append((reg.left_anchor_seq, reg.right_anchor_seq, names[:n], seqs[:n]))
    # anchors of 1000 and 600, and of at most one stripe (512 and 300); an anchor holding N
    for seed, cut_l, cut_r, n_in_anchor in ((12, 1000, 600, False), (13, 512, 300, False), (14, 1000, 1000, True)):
        reg, names, seqs, _truth = synth.region_reads(seed=seed, n_reads=18, motif="CAG", alleles=(15, 40))
        left, right = reg.left_anchor_seq[-cut_l:], reg.right_anchor_seq[:cut_r]
        if n_in_anchor:
            left = left[:400] + "N" + left[401:]
        regions.append((left, right, names, seqs))
    # edge reads in one region: shorter than an anchor, holding N, over the template limit, empty, anchors on different
    # strands (dist 0), the anchor twice (equal scores on both strands), lower case
    reg, names, seqs, _truth = synth.region_reads(seed=15, n_reads=6, motif="CAG", alleles=(20,))
    L, R = reg.left_anchor_seq, reg.right_anchor_seq
    mid = "CAG" * 20
    extra = {"short": L[200:700], "has_n": seqs[0][:500] + "N" + seqs[0][501:], "huge": synth.random_seq(rng, 70000),
             "empty": "", "strands": L + mid + rc(R), "both_strands": L + mid + R + synth.random_seq(rng, 50) + rc(L),
             "lower": seqs[1].lower(), "just_anchors": L + R, "overlap": L + R[5:]}
    regions.append((L, R, names + list(extra), seqs + list(extra.values())))
    return regions


def test_anchor_regions_equal_both_references(engine, oracle):
    from nanorepeat_b200 import anchoring, RepeatRegion
    from oracle import anchoring as oanchor
    regions = build_cases()
    rrs = []
    for left, right, _names, _seqs in regions:
        rr = RepeatRegion()
        rr.left_anchor_seq, rr.right_anchor_seq = left, right
        rrs.append(rr)
    anchoring.find_anchor_locations_in_regions("ont", rrs, [(names, seqs) for _l, _r, names, seqs in regions])
    n_accepted = 0
    for rr, (left, right, names, seqs) in zip(rrs, regions):
        anchoring.make_core_seq_fastq(rr, reads=(names, seqs), write_files=False)
        want = per_region_rules(engine, left, right, names, seqs)
        # the oracle scores every read; the library leaves reads with N and reads over the template limit unscored
        keep = [i for i, n in enumerate(names) if n not in ("has_n", "huge")]
        ora = oanchor.step1(left, right, [names[i] for i in keep], [seqs[i].upper() for i in keep], n_threads=oracle.max_threads())
        assert set(rr.read_dict) == set(want), set(rr.read_dict) ^ set(want)
        assert set(want) == set(ora), set(want) ^ set(ora)
        for name, w in want.items():
            rd = rr.read_dict[name]
            got = dict(strand=rd.strand, dist=rd.dist_between_anchors, core_start=rd.core_seq_start_pos, core_end=rd.core_seq_end_pos,
                       mid_start=rd.mid_seq_start_pos, mid_end=rd.mid_seq_end_pos, left_buffer=rd.left_buffer_len,
                       right_buffer=rd.right_buffer_len, core=rr.read_core_seq_dict[name],
                       left=(rd.left_anchor_paf.strand, rd.left_anchor_paf.align_score, rd.left_anchor_paf.qstart, rd.left_anchor_paf.qend),
                       right=(rd.right_anchor_paf.strand, rd.right_anchor_paf.align_score, rd.right_anchor_paf.qstart,
                              rd.right_anchor_paf.qend))
            assert got == w, (name, got, w)
            if name in ora:
                o = ora[name]
                assert (o["strand"], o["dist"], o["core_start"], o["core_end"], o["mid_start"], o["mid_end"], o["left_buffer"],
                        o["right_buffer"]) == tuple(w[k] for k in ("strand", "dist", "core_start", "core_end", "mid_start", "mid_end",
                                                                   "left_buffer", "right_buffer")), name
            assert rd.full_read_len == len(seqs[names.index(name)])
            n_accepted += 1
    assert n_accepted > 100
    last = rrs[-1].read_dict
    assert "strands" in last and last["strands"].dist_between_anchors == 0
    assert not ({"has_n", "huge", "empty", "short"} & set(last))


def test_anchor_regions_two_launches_for_many_regions(engine):
    from nanorepeat_b200 import synth
    sc = engine.get_preset("ont")
    lefts, rights, reads = [], [], []
    for g in range(200):
        reg, _names, seqs, _truth = synth.region_reads(seed=100 + g, n_reads=3, motif="CAG", alleles=(12, 30))
        lefts.append(reg.left_anchor_seq); rights.append(reg.right_anchor_seq); reads.append(seqs)
    res, stats = engine.anchor_regions(sc, lefts, rights, reads)
    assert stats["kernel_launches"] <= 2
    assert stats["algorithmic_cells"] == sum(2 * (len(l) + len(r)) * len(s) for l, r, ss in zip(lefts, rights, reads) for s in ss)
    assert int(res["accepted"].sum()) > 300


def test_quantify_regions_equals_per_region_chain(engine):
    import nanorepeat_b200 as nrb
    from nanorepeat_b200 import anchoring, synth
    batch, single, region_reads = [], [], []
    for seed, motif in ((21, "CAG"), (22, "GGGGCC"), (23, "AT"), (24, "CAG")):
        reg, names, seqs, _truth = synth.region_reads(seed=seed, n_reads=20, motif=motif, alleles=(14, 33))
        for lst in (batch, single):
            rr = nrb.RepeatRegion()
            rr.left_anchor_seq, rr.right_anchor_seq, rr.repeat_unit_seq = reg.left_anchor_seq, reg.right_anchor_seq, motif
            lst.append(rr)
        region_reads.append((names, seqs))
    nrb.quantify_regions(batch, region_reads)
    for rr, reads in zip(single, region_reads):
        anchoring.find_anchor_locations_in_reads("ont", rr, 1, reads=reads)
        anchoring.make_core_seq_fastq(rr, reads=reads, write_files=False)
        nrb.round1_and_round2_estimation("ont", rr, 1)
        nrb.round3_estimation("ont", False, rr, 1)
    for a, b in zip(batch, single):
        assert list(a.read_dict) == list(b.read_dict)
        for name in a.read_dict:
            x, y = a.read_dict[name], b.read_dict[name]
            assert (x.round1_repeat_size, x.round2_repeat_size) == (y.round1_repeat_size, y.round2_repeat_size), name
            assert (x.round3_repeat_size is None) == (y.round3_repeat_size is None), name
            assert x.round3_repeat_size is None or float(x.round3_repeat_size) == float(y.round3_repeat_size), name
