"""CPU companion of tests/test_gpu_joint_edges.py: each boundary that file names really occurs in its inputs
(tests/helpers/joint_edges.py).  The oracle's traceback gives the optimal path's CIGAR; walked from tstart it shows where
every gap sits and, through oracle/joint.window_stats (the reference's window re-scoring), whether it was charged."""
import re

from helpers import joint_edges as je
from oracle import joint


def _gaps(cigar, tstart):
    """-> (insertions [(template position, length)], deletions [(first template position, length)])"""
    ins, dels, p = [], [], tstart
    for n, op in re.findall(r"(\d+)([=XID])", cigar):
        n = int(n)
        if op == "I":
            ins.append((p, n))
        elif op == "D":
            dels.append((p, n))
        if op != "I":
            p += n
    return ins, dels


def _aln(oracle, read, tpl, a, b):
    score, pay, ts, te, cigar = oracle.align_window(read, tpl, a, b, want_cigar=True)
    assert joint.window_stats(cigar, ts, te, a, b)["score"] == pay
    ins, dels = _gaps(cigar, ts)
    return score, pay, ins, dels


def _by_tag(cases, tag):
    (c,) = [c for c in cases if c["tag"] == tag]
    return c


def test_window_edge_cases_hit_their_boundaries(oracle):
    cases = je.window_cases()
    # insertions at a and b - 1 are not charged, at a + 1 and b - 2 they are (a < p < b - 1)
    for p, charged in ((je.A, False), (je.A + 1, True), (je.B - 2, True), (je.B - 1, False)):
        c = _by_tag(cases, f"ins 3 at {p}")
        _, pay, ins, dels = _aln(oracle, c["read"], c["tpl"], je.A, je.B)
        assert ins == [(p, 3)] and not dels, (p, ins, dels)
        assert (pay == 2 * (je.B - je.A) - 4 - 2 * 2) == charged and (pay == 2 * (je.B - je.A)) == (not charged), (p, pay)
    # the optimal path enters the window by a deletion at a - 1: its first in-window base is charged -4
    c = _by_tag(cases, "del from a-1")
    _, pay, ins, dels = _aln(oracle, c["read"], c["tpl"], je.A, je.B)
    assert dels == [(je.A - 1, 3)] and not ins
    assert pay == 2 * (je.B - je.A - 2) - 4 - 2
    for tag, at in (("del from a", je.A), ("del to b-1", je.B - 3), ("del over window", je.A - 2), ("del 19", je.A + 30),
                    ("del 21", je.A + 30), ("del 21 from a-1", je.A - 1)):
        c = _by_tag(cases, tag)
        assert [d[0] for d in _aln(oracle, c["read"], c["tpl"], je.A, je.B)[3]] == [at], tag
    # b = a + 3 is the first window with a charged insertion position (a + 1)
    c = _by_tag(cases, "window [200, 203)")
    assert _aln(oracle, c["read"], c["tpl"], 200, 203)[2] == [(201, 3)]
    assert oracle.align_window(c["read"], c["tpl"], 200, 203)[1] == 2 * 3 - 4 - 2 * 2
    assert oracle.align_window(c["read"], c["tpl"], 200, 202)[1] == 2 * 2
    # N sits at the stated rows of the oriented read
    for row in (255, 256, 257):
        assert _by_tag(cases, f"N at row {row}")["read"][row] == "N"
    # the shapes: every stripe height against every ramp width
    assert {(len(c["read"]), len(c["tpl"])) for c in cases if c["tag"].startswith("shape")} == \
        {(q, t) for q in je.READ_LENS for t in je.TPL_LENS}


def test_grid_junction_reads_hit_the_junction(oracle):
    """On the loci with long anchors: insertions at J + 8 (charged) and J + 9 (not), a deletion that spans J by each affine
    piece, deletions from R[9] (charged) and R[10] (outside the window)."""
    seen = 0
    for locus in je.geometry_loci():
        if len(locus["left"]) != 42 or len(locus["right"]) < 41:
            continue
        seen += 1
        T = je.template(locus, je.K1T, je.K2T)
        J = je.junction(locus, je.K1T, je.K2T)
        a, b = je.window_of(locus, je.K1T, je.K2T)
        assert b == J + 10
        rd = dict(zip(locus["tags"], locus["reads"]))
        fwd = {t: (je.revcomp(r) if i % 2 else r) for i, (t, r) in enumerate(rd.items())}
        full = 2 * (b - a)
        _, pay, ins, dels = _aln(oracle, fwd["ins at J+8"], T, a, b)
        assert ins == [(J + 8, 2)] and pay == full - 6
        _, pay, ins, dels = _aln(oracle, fwd["ins at J+9"], T, a, b)
        assert ins == [(J + 9, 2)] and pay == full
        for tag, n in (("del over J (E1)", 6), ("del over J (E2)", 25)):
            _, pay, ins, dels = _aln(oracle, fwd[tag], T, a, b)
            assert len(dels) == 1 and dels[0][0] < J < dels[0][0] + dels[0][1] and dels[0][1] == n, (tag, dels)
            m = min(dels[0][0] + n, b) - dels[0][0]                                   # its bases inside the window
            assert pay == full - 2 * m - 4 - 2 * (m - 1)
        _, pay, ins, dels = _aln(oracle, fwd["del from R[9]"], T, a, b)
        assert dels == [(J + 9, 1)] and pay == full - 2 - 4
        _, pay, ins, dels = _aln(oracle, fwd["del from R[10]"], T, a, b)
        assert dels == [(J + 10, 1)] and pay == full
        pal = rd["palindrome"]
        assert pal == je.revcomp(pal)
    assert seen == 3


def test_grid_shapes_reach_the_limits():
    loc = je.shape_locus()
    pr, p1, p2 = loc["points"]
    k = {r: (sorted({p1[i] for i in range(len(pr)) if pr[i] == r}), sorted({p2[i] for i in range(len(pr)) if pr[i] == r}))
         for r in set(pr)}
    assert [len(k[r][1]) for r in (0, 1)] == [64, 65] and [len(k[r][0]) for r in (2, 3)] == [64, 65]
    assert 8 not in k and loc["reads"][9] == "" and len(pr) > len(set(zip(pr, p1, p2)))
    lim = je.window_limit_locus()
    widths = sorted(je.window_of(lim, k1, k2)[1] - je.window_of(lim, k1, k2)[0] for k1, k2 in zip(*lim["points"][1:]))
    assert widths[-2:] == [8000, 8002]
    long_reads = je.long_read_locus()["reads"]
    assert 6 * 40000 * 9100 > 2 ** 31 and all(len(r) == 40000 for r in long_reads)
    # |K1| = 2: 12 state words per read base; the 2^29-word budget lasts 1 118 of 1 200 reads
    assert (2 ** 29 - 1) // (12 * 40000) == 1118


def test_window_limit_records(oracle):
    """The +16 000 payload ceiling of an 8 000-base window and the payload floor at the score limit: 60 from the
    16-bit decode limit."""
    lim = {c["tag"]: c for c, _ in je.limit_cases()}
    c = lim["window 8000"]
    assert oracle.align_window(c["read"], c["tpl"], c["a"], c["b"]) == (16000, 16000)
    for g, rec in je.PAYLOAD_FLOOR.items():
        c = je.payload_floor_case(g)
        assert 2 * min(len(c["read"]), len(c["tpl"])) == 32766
        assert oracle.align_window(c["read"], c["tpl"], c["a"], c["b"]) == rec
    assert -32768 + 60 == je.PAYLOAD_FLOOR[16356][1]
