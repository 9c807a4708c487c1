"""CPU restatement of Step 1 (anchor finding + core extraction) for the tests (TEST INFRASTRUCTURE ONLY).

Follows reference src/NanoRepeat/nanoRepeat_bam.py:165-234 (acceptance rules, distances, core positions) and :308-316
(slicing) with the alignment engine replaced by oracle/nr_oracle (PARITY UNPINNED for the engine: minimap2's seeding,
secondary-hit and mapq heuristics are not modelled; the candidate hits of an anchor are its best exact alignment on each
strand at or above minimap2's -s).  Written independently of nanorepeat_b200/anchoring.py: plain tuples, no shared code.
"""
from . import nr_oracle

COMP = {"A": "T", "C": "G", "G": "C", "T": "A", "a": "t", "c": "g", "g": "c", "t": "a", "N": "N", "n": "n"}


def revcomp(s):
    return "".join(COMP[c] for c in reversed(s))


def records(left_anchor, right_anchor, seqs, min_dp_score=80, n_threads=1):
    """-> per read, what nr_anchor_read_t holds: dict(accepted, left_good, right_good, strand, left_strand, right_strand,
    read_len, dist_between_anchors, core_start, core_end, mid_start, mid_end, left_buffer, right_buffer, left, right).

    left / right: the anchor's best hit as (score, qstart, qend), (0, -1, 0) without a hit, qstart -1 unless the anchor is
    good; strands are '+', '-' or '' (no hit; strand: '' unless accepted); dist_between_anchors is set when both anchors
    are good, the core and middle fields when the read is accepted (else 0).  Also `cands`: the four raw alignments of
    the read as ((left '+', left '-'), (right '+', right '-')), each (score, tstart, tend)."""
    q, t = [], []
    for s in seqs:
        r = revcomp(s)
        q += [left_anchor, left_anchor, right_anchor, right_anchor]
        t += [s, r, s, r]
    recs = nr_oracle.align_batch(q, t, n_threads=n_threads)

    def good(hits):                                           # :165-179
        if not hits:
            return False
        if len(hits) == 1:
            return True
        if hits[0][3] - hits[0][2] < 10:
            return False
        return hits[0][0] > 1.5 * hits[1][0]

    out = []
    for i, seq in enumerate(seqs):
        o = dict(accepted=0, left_good=0, right_good=0, strand="", left_strand="", right_strand="", read_len=len(seq),
                 dist_between_anchors=0, core_start=0, core_end=0, mid_start=0, mid_end=0, left_buffer=0, right_buffer=0,
                 left=(0, -1, 0), right=(0, -1, 0))
        o["cands"] = tuple(tuple(tuple(int(x) for x in recs[4 * i + 2 * a + s]) for s in range(2)) for a in range(2))
        best = []
        for a, side in enumerate(("left", "right")):
            hits = []
            for s, strand in enumerate("+-"):
                score, ts, te = o["cands"][a][s]
                if score > 0 and score >= min_dp_score:
                    hits.append((score, strand, ts, te))
            hits.sort(key=lambda h: -h[0])                    # stable: '+' first on a tie
            ok = good(hits)
            o[side + "_good"] = int(ok)
            if hits:
                score, strand, ts, te = hits[0]
                o[side] = (score, ts if ok else -1, te)
                o[side + "_strand"] = strand
            best.append(hits[0] if ok else None)
        out.append(o)
        if best[0] is None or best[1] is None:
            continue
        (_ls, lstrand, _lqs, lqe), (_rs, rstrand, rqs, _rqe) = best
        dist = rqs - lqe if lstrand == rstrand else 0         # :204-207
        o["dist_between_anchors"] = dist
        if not dist > -10:                                    # :209-211
            continue
        core_start, core_end = max(lqe - 100, 0), min(rqs + 100, len(seq))       # :221-234
        o.update(accepted=1, strand=lstrand, core_start=core_start, core_end=core_end, mid_start=lqe, mid_end=rqs,
                 left_buffer=lqe - core_start, right_buffer=core_end - rqs)
    return out


def step1(left_anchor, right_anchor, names, seqs, min_dp_score=80, n_threads=1):
    """-> {name: dict(strand, dist, core_start, core_end, mid_start, mid_end, left_buffer, right_buffer, core, mid)} for
    the reads the reference's rules accept (the accepted reads of records())."""
    out = {}
    for name, seq, o in zip(names, seqs, records(left_anchor, right_anchor, seqs, min_dp_score, n_threads)):
        if not o["accepted"]:
            continue
        oriented = revcomp(seq) if o["strand"] == "-" else seq
        out[name] = dict(strand=o["strand"], dist=o["dist_between_anchors"], core_start=o["core_start"], core_end=o["core_end"],
                         mid_start=o["mid_start"], mid_end=o["mid_end"], left_buffer=o["left_buffer"],
                         right_buffer=o["right_buffer"], core=oriented[o["core_start"]:o["core_end"]],
                         mid=oriented[o["mid_start"]:o["mid_end"]])
    return out
