"""Step 1 (nr_anchor_regions) read by read against the exact DP: every field of nr_anchor_read_t -- each anchor's best hit
(score, qstart, qend), its strand, left_good / right_good, acceptance, distance, core and middle -- of every read, accepted
or rejected, equals oracle/anchoring.records bit for bit.

The regions cover what the anchor kernel (nr_launch_anchor.cu) and its host side (nr_anchor.cu) do differently by shape:
every stripe height R and stripe counts S = 1..32 of pair_shape, a half that is mostly padding, an empty anchor, the
16-bit score and column limits, the whole-strand 32-bit fallback for long anchors and its own score limit, N at stripe
edges, and the reference's rules at their boundaries.  Each boundary case asserts, on the oracle's records, that the
boundary really occurs in its inputs (test_boundary_cases_occur runs without a GPU)."""
import numpy as np
import pytest

from oracle import anchoring as oanchor

COMP = str.maketrans("ACGTacgtNn", "TGCAtgcaNn")
MAX_TLEN = 65535 - 64               # nr_limits' template limit
MAX_SCORE = 32767                   # nr_limits' score limit (match * min(|anchor|, |read|))
MATCH = 2                           # map-ont
MIN_DP_SCORE = 80
MAX_PAIR_ANCHOR = (65535 - 65) // 4   # longest anchor of a 16-bit half: an exact hit fills it to 2 * 32 734 + 65
# the stripe shapes to cover: every R of pair_shape (4, 6, 8, 12, 16) and S = 1 .. 32
SHAPE_PAIRS = ((1537, 40), (41, 128), (127, 192), (129, 256), (193, 257), (384, 41), (385, 511), (513, 512), (768, 127),
               (769, 1000), (1024, 1025), (40, 1536), (4097, 384))
FIELDS = ("accepted", "left_good", "right_good", "strand", "left_strand", "right_strand", "read_len", "dist_between_anchors",
          "core_start", "core_end", "mid_start", "mid_end", "left_buffer", "right_buffer", "left", "right")


def rc(s):
    return s.translate(COMP)[::-1]


def pair_shape(rows):
    """nr_anchor.cu's pair_shape: -> (R, S)."""
    S = max(1, -(-rows // 512))
    need = -(-rows // (32 * S))
    return next(h for h in (4, 6, 8, 12, 16) if h >= need), S


def stripes(left, right):
    """stripes of a region's anchor pairs (0: both anchors are over 16 367 bases or empty)"""
    rows = max(n if n <= MAX_PAIR_ANCHOR else 0 for n in (len(left), len(right)))
    return pair_shape(rows)[1] if rows else 0


def rand(rng, n):
    return "".join("ACGT"[i] for i in rng.integers(0, 4, size=n))


def mutate(rng, s, rate=0.03):
    """deletions, substitutions and insertions, each at rate / 3; other characters than ACGTacgt become bases"""
    out = []
    for c in s:
        u = rng.random()
        if u < rate / 3:
            continue
        if u < 2 * rate / 3:
            out.append("ACGT"[("ACGT".index(c.upper()) + int(rng.integers(1, 4))) % 4] if c.upper() in "ACGT" else "A")
            continue
        out.append(c if c in "ACGTacgt" else "ACGT"[int(rng.integers(0, 4))])
        if u < rate:
            out.append("ACGT"[int(rng.integers(0, 4))])
    return "".join(out)


def acgt(s):
    """a read the library scores: its N / lower case become bases"""
    return "".join(c if c in "ACGTacgt" else "A" for c in s)


def shape_reads(rng, left, right):
    """mutated copies of both anchors on both strands at random offsets, an exact copy, the anchors on different strands,
    a read shorter than the anchors and an unrelated read"""
    L, R = acgt(left), acgt(right)
    mid = rand(rng, int(rng.integers(20, 200)))
    reads = [rand(rng, int(rng.integers(0, 300))) + mutate(rng, L) + mid + mutate(rng, R) + rand(rng, int(rng.integers(0, 300))),
             rc(rand(rng, int(rng.integers(0, 300))) + mutate(rng, L) + mid + mutate(rng, R) + rand(rng, 50)),
             rand(rng, int(rng.integers(1, 100))) + L + mid + R + rand(rng, int(rng.integers(1, 100))),
             rand(rng, 30) + mutate(rng, L) + mid + rc(mutate(rng, R)),
             (L + mid + R)[len(L) // 3: len(L) // 3 + max(len(L), len(R)) // 2 + 1],
             rand(rng, len(L) + len(R) + 40)]
    return reads


def unscored(read_len):
    return dict(accepted=0, left_good=0, right_good=0, strand="", left_strand="", right_strand="", read_len=read_len,
                dist_between_anchors=0, core_start=0, core_end=0, mid_start=0, mid_end=0, left_buffer=0, right_buffer=0,
                left=(0, -1, 0), right=(0, -1, 0))


def scored_read(s):
    return 0 < len(s) <= MAX_TLEN and not set(s) - set("ACGTacgt")


def anchor_scored(anchor, read):
    """an anchor's score fits a DP word on this read (else the library leaves it without a hit and counts it)"""
    return MATCH * min(len(anchor), len(read)) <= MAX_SCORE


def expected(left, right, reads, n_threads):
    """-> (records per read, n_skipped, algorithmic cells) of one region as the library defines them"""
    out = [None] * len(reads)
    groups = {}
    skipped = cells = 0
    for i, s in enumerate(reads):
        if not scored_read(s):
            out[i] = unscored(len(s))
            skipped += len(s) > 0
            continue
        cells += 2 * (len(left) + len(right)) * len(s)
        lq = left if anchor_scored(left, s) else ""
        rq = right if anchor_scored(right, s) else ""
        skipped += (lq != left) + (rq != right)
        groups.setdefault((lq, rq), []).append(i)
    for (lq, rq), idx in groups.items():
        for i, o in zip(idx, oanchor.records(lq, rq, [reads[i] for i in idx], MIN_DP_SCORE, n_threads)):
            out[i] = o
    return out, skipped, cells


def got_records(res):
    """ANCHOR_READ_DTYPE rows -> the records' dicts"""
    out = []
    for r in res:
        d = {k: int(r[k]) for k in FIELDS if k not in ("left", "right")}
        for k in ("strand", "left_strand", "right_strand"):
            d[k] = chr(d[k]) if d[k] else ""
        for k in ("left", "right"):
            d[k] = (int(r[k]["score"]), int(r[k]["tstart"]), int(r[k]["tend"]))
        out.append(d)
    return out


def assert_same(name, got, want):
    assert len(got) == len(want), name
    for i, (g, w) in enumerate(zip(got, want)):
        bad = {k: (g[k], w[k]) for k in FIELDS if g[k] != w[k]}
        assert not bad, (name, i, bad)


# ---------------------------------------------------------------- regions

def ambiguous(rng, n, R_S):
    """an anchor of n bases with N at row 0, at 32R - 1 and 32R of every stripe edge and at the last row"""
    R, S = R_S
    rows = {0, n - 1}
    for s in range(1, S):
        rows |= {s * 32 * R - 1, s * 32 * R}
    a = list(rand(rng, n))
    for r in rows:
        if r < n:
            a[r] = "N"
    return "".join(a), sorted(r for r in rows if r < n)


def shape_regions(rng):
    regs = {}
    for nl, nr in SHAPE_PAIRS:
        left, right = rand(rng, nl), rand(rng, nr)
        regs[f"shape_{nl}_{nr}"] = (left, right, shape_reads(rng, left, right))
    for nl, nr in ((0, 500), (500, 0)):
        left, right = rand(rng, nl), rand(rng, nr)
        regs[f"empty_{nl}_{nr}"] = (left, right, shape_reads(rng, left, right))
    # N at the stripe edges, in the left half (the longer anchor) and in the right half
    for nl, nr in ((1537, 1000), (700, 1025)):
        shape = pair_shape(max(nl, nr))
        left, _ = ambiguous(rng, nl, shape)
        right, _ = ambiguous(rng, nr, shape)
        regs[f"ambiguous_{nl}_{nr}"] = (left, right, shape_reads(rng, left, right))
    left, right = rand(rng, 800).lower(), rand(rng, 150) + rand(rng, 150).lower()
    regs["lower_case"] = (left, right, shape_reads(rng, left, right))
    # low complexity anchors and reads: ties of score and end everywhere
    left, right = "CAG" * 40, "AT" * 45 + "T" * 30
    reads = ["CAG" * 90 + "AT" * 80 + "T" * 40, "CAGCAGCAACAG" * 25 + "AT" * 100, rc("CAG" * 60 + rand(rng, 30) + "AT" * 60),
             "A" * 500, "AT" * 300, "CAG" * 20 + "CTG" * 40 + "TA" * 70 + "T" * 50, mutate(rng, "CAG" * 120 + "AT" * 90 + "T" * 60)]
    regs["low_complexity"] = (left, right, reads)
    return regs


def limit_regions(rng):
    regs = {}
    # an exact 16 367-base hit fills its half to 2 * 32 734 + 65 = 65 533; the other half holds a 600-base anchor's hit
    L, R = rand(rng, 16367), rand(rng, 600)
    regs["score_limit"] = (L, R, [rand(rng, 40) + L + rand(rng, 80) + mutate(rng, R), rc(L + rand(rng, 60) + R),
                                  rand(rng, 100) + R + rand(rng, 50)])
    # whole-strand fallback (anchors over 16 367 bases), scored; the first read holds the anchor on both strands
    L, R = rand(rng, 16368), rand(rng, 200)
    regs["whole_strand_16368"] = (L, R, [L + rc(L), rand(rng, 50) + L + rand(rng, 70) + R, rc(mutate(rng, L) + rand(rng, 20) + R)])
    L, R = rand(rng, 300), rand(rng, 16383)
    regs["whole_strand_16383"] = (L, R, [rand(rng, 10) + L + rand(rng, 90) + R, rc(L + rand(rng, 30) + R)])
    # a 16 384-base anchor does not fit a 32-bit task on reads over 16 383 bases: no hit, counted; on a shorter read it is scored
    L, R = rand(rng, 16384), rand(rng, 300)
    regs["unscored_16384"] = (L, R, [L + rand(rng, 60) + R, rc(rand(rng, 5) + L + rand(rng, 60) + R),
                                     L[-15000:] + rand(rng, 60) + R, L[:16383]])
    # the template limit: hits ending at the last column of 65 471-base reads; a read of 65 472 bases is not scored
    L, R = rand(rng, 500), rand(rng, 300)
    body = L + rand(rng, 45) + R
    regs["column_limit"] = (L, R, [rand(rng, MAX_TLEN - len(body)) + body, rc(rand(rng, MAX_TLEN - len(body)) + body),
                                   rand(rng, MAX_TLEN + 1 - len(body)) + body, rand(rng, MAX_TLEN)])
    # tiny reads (1 - 33 bases) and reads shorter than the anchor
    L, R = rand(rng, 100), rand(rng, 64)
    regs["tiny_reads"] = (L, R, [L[:k] for k in range(1, 34)] + [L[10:90], R[:50], rc(L[:70]), ""])
    return regs


def score_of(anchor, read):
    from oracle import nr_oracle
    return nr_oracle.align(anchor, read)[0]


def ratio_read(rng, A, tail, delta):
    """a read holding A[:j] on '+' and A[:k] on '-' with 2 * AS0 - 3 * AS1 == delta (found on the oracle's scores)"""
    f1, f2, g1, g2 = (rand(rng, 40) for _ in range(4))
    plus = {j: score_of(A, f1 + acgt(A[:j]) + f2) for j in range(60, len(A) + 1)}
    minus = {k: score_of(A, g1 + acgt(A[:k]) + g2) for k in range(40, len(A) + 1)}
    for j, s0 in plus.items():
        for k, s1 in minus.items():
            if s1 >= MIN_DP_SCORE and 2 * s0 - 3 * s1 == delta:
                read = f1 + acgt(A[:j]) + f2 + rc(g1 + acgt(A[:k]) + g2) + tail
                o = oanchor.records(A, "", [read])[0]
                (p, _, _), (m, _, _) = o["cands"][0]
                if p > m and 2 * p - 3 * m == delta:
                    return read
    raise AssertionError(f"no read with 2 * AS0 - 3 * AS1 == {delta}")


def rule_regions(rng):
    regs = {}
    # 2 * AS0 == 3 * AS1 (not good) and one point above it (good); the N makes odd scores possible
    A = rand(rng, 150) + "N" + rand(rng, 149)
    B = rand(rng, 400)
    tail = rand(rng, 30) + B
    regs["ratio"] = (A, B, [ratio_read(rng, A, tail, 0), ratio_read(rng, A, tail, 1)])
    # a 40-base exact hit scores min_dp_score; one mismatch drops it below; a 41-base anchor with an N scores one below
    L, R = rand(rng, 40), rand(rng, 20) + "N" + rand(rng, 20)
    Lm = L[:20] + "ACGT"[("ACGT".index(L[20]) + 1) % 4] + L[21:]
    regs["min_score"] = (L, R, [rand(rng, 30) + L + rand(rng, 50) + acgt(R) + rand(rng, 9),
                                rand(rng, 30) + Lm + rand(rng, 50) + R.replace("N", "C")])
    # dist = -10 (rejected) and -9 (accepted): the right anchor begins with the left anchor's last j bases
    L = rand(rng, 300)
    rest = rand(rng, 290)
    for j in (10, 9):
        R = L[-j:] + rest
        regs[f"dist_{j}"] = (L, R, [rand(rng, 70) + L + R[j:] + rand(rng, 40), rc(L + R[j:] + rand(rng, 15))])
    # equal scores on both strands; tandem copies (smallest tend, then largest tstart); hits at the first and last column
    L, R = rand(rng, 250), rand(rng, 260)
    mid = rand(rng, 90)
    regs["ties"] = (L, R, [rand(rng, 20) + L + mid + R + rand(rng, 33) + rc(L),
                           rand(rng, 20) + L + mid + R + rand(rng, 33) + rc(R),
                           rand(rng, 20) + L + L + mid + R + R + rand(rng, 12),
                           rc(L + L + mid + R + rand(rng, 5)),
                           L + mid + R, rc(L + mid + R)])
    # core clamped at 0 and at read_len (anchors under 100 bases), and not clamped
    L, R = rand(rng, 60), rand(rng, 70)
    mid = rand(rng, 40)
    regs["clamps"] = (L, R, [L + mid + R, rc(rand(rng, 3) + L + mid + R), rand(rng, 100) + L + mid + R + rand(rng, 100)])
    return regs


def check_rule_cases(regs, exp):
    """each boundary occurs in its inputs, on the oracle's records"""
    r0, r1 = exp["ratio"]
    for o, delta, good in ((r0, 0, 0), (r1, 1, 1)):
        (p, _, _), (m, _, _) = o["cands"][0]
        assert 2 * max(p, m) - 3 * min(p, m) == delta and min(p, m) >= MIN_DP_SCORE and o["left_good"] == good, (delta, o)
    a, b = exp["min_score"]
    assert a["left"][0] == MIN_DP_SCORE and a["left_good"] and a["cands"][1][0][0] == MIN_DP_SCORE - 1 and not a["right_strand"]
    assert max(c[0] for c in b["cands"][0]) < MIN_DP_SCORE and not b["left_strand"]
    for j, acc in ((10, 0), (9, 1)):
        for o in exp[f"dist_{j}"]:
            assert o["left_good"] and o["right_good"] and o["dist_between_anchors"] == -j and o["accepted"] == acc, (j, o)
    t = exp["ties"]
    L, R = regs["ties"][0], regs["ties"][1]
    assert t[0]["cands"][0][0][0] == t[0]["cands"][0][1][0] == 2 * len(L) and t[0]["left_strand"] == "+" and not t[0]["left_good"]
    assert t[1]["cands"][1][0][0] == t[1]["cands"][1][1][0] == 2 * len(R) and t[1]["right_strand"] == "+" and not t[1]["right_good"]
    assert t[2]["left"] == (2 * len(L), 20, 20 + len(L)) and t[2]["accepted"]                  # the first of two copies
    assert t[2]["right"][0] == 2 * len(R) and t[2]["right"][2] == t[2]["right"][1] + len(R)
    assert t[3]["left"] == (2 * len(L), 0, len(L)) and t[3]["strand"] == "-"          # on the strand of the hit
    for o in t[4:]:
        assert o["accepted"] and o["left"][1] == 0 and o["right"][2] == o["read_len"], o
    c = exp["clamps"]
    for o in c[:2]:
        assert o["accepted"] and o["core_start"] == 0 and o["left"][2] < 100 and o["core_end"] == o["read_len"] and \
            o["right"][1] + 100 > o["read_len"], o
    assert c[2]["accepted"] and c[2]["core_start"] > 0 and c[2]["core_end"] < c[2]["read_len"]


def check_limit_cases(regs, exp):
    o = exp["score_limit"][0]
    assert o["left"][0] == 2 * 16367 and o["right"][0] > 0 and o["accepted"]
    assert exp["score_limit"][1]["left"][0] == 2 * 16367 and exp["score_limit"][1]["strand"] == "-"
    o = exp["whole_strand_16368"][0]
    assert o["cands"][0][0][0] == o["cands"][0][1][0] == 2 * 16368 and not o["left_good"] and o["left"][1] == -1
    assert exp["whole_strand_16368"][1]["accepted"] and exp["whole_strand_16383"][0]["right"][0] == 2 * 16383
    u = exp["unscored_16384"]
    assert u[0]["left"] == u[1]["left"] == (0, -1, 0) and u[0]["right_good"] and u[2]["left_good"] and u[2]["accepted"]
    c = exp["column_limit"]
    assert len(regs["column_limit"][2][0]) == MAX_TLEN and c[0]["right"][2] == MAX_TLEN and c[0]["accepted"]
    assert c[1]["right"][2] == MAX_TLEN and c[1]["strand"] == "-" and c[2] == unscored(MAX_TLEN + 1)
    reads = regs["tiny_reads"][2]
    assert {len(s) for s in reads[:33]} == set(range(1, 34))
    assert exp["tiny_reads"][33]["left_good"] and len(reads[33]) < len(regs["tiny_reads"][0])


def all_regions():
    rng = np.random.default_rng(2024)
    regs = {}
    regs.update(shape_regions(rng))
    regs.update(limit_regions(rng))
    regs.update(rule_regions(rng))
    return regs


@pytest.fixture(scope="module")
def cases(oracle):
    regs = all_regions()
    exp, skipped, cells = {}, {}, {}
    for name, (left, right, reads) in regs.items():
        exp[name], skipped[name], cells[name] = expected(left, right, reads, oracle.max_threads())
    return regs, exp, skipped, cells


def test_boundary_cases_occur(oracle):
    """the rules' boundaries, without a GPU: each case is built from the inputs and happens on the oracle's records"""
    rng = np.random.default_rng(7)
    regs = rule_regions(rng)
    exp = {name: expected(l, r, reads, oracle.max_threads())[0] for name, (l, r, reads) in regs.items()}
    check_rule_cases(regs, exp)


def test_shapes_cover_every_stripe_height():
    shapes = {pair_shape(max(nl, nr)) for nl, nr in SHAPE_PAIRS} | {pair_shape(16367)}
    assert {R for R, _S in shapes} == {4, 6, 8, 12, 16}
    assert {1, 2, 3, 4, 9, 32} <= {S for _R, S in shapes}


@pytest.mark.gpu
def test_every_field_of_every_read_in_one_call(engine, cases):
    regs, exp, skipped, cells = cases
    check_rule_cases(regs, {k: exp[k] for k in regs if k in ("ratio", "min_score", "dist_10", "dist_9", "ties", "clamps")})
    check_limit_cases(regs, exp)
    sc = engine.get_preset("ont")
    names = list(regs)
    res, stats = engine.anchor_regions(sc, [regs[n][0] for n in names], [regs[n][1] for n in names], [regs[n][2] for n in names])
    assert stats["kernel_launches"] <= 2
    assert stats["algorithmic_cells"] == sum(cells.values())
    assert stats["n_skipped"] == sum(skipped.values())
    got = got_records(res)
    n_accepted = n_rejected = pos = 0
    for n in names:
        k = len(regs[n][2])
        assert_same(n, got[pos:pos + k], exp[n])
        n_accepted += sum(o["accepted"] for o in exp[n])
        n_rejected += sum(not o["accepted"] for o in exp[n])
        # the same region called alone
        alone, st = engine.anchor_regions(sc, [regs[n][0]], [regs[n][1]], [regs[n][2]])
        assert np.array_equal(alone, res[pos:pos + k]), n
        assert st["n_skipped"] == skipped[n] and st["algorithmic_cells"] == cells[n], (n, st)
        pos += k
    assert n_accepted > 50 and n_rejected > 50


@pytest.mark.gpu
def test_long_anchor_qstart_only_for_good_anchors(engine, cases):
    regs, exp, _skipped, _cells = cases
    left, right, reads = regs["whole_strand_16368"]
    res, _st = engine.anchor_regions(engine.get_preset("ont"), [left], [right], [reads])
    got = got_records(res)
    assert got[0]["left"] == (2 * 16368, -1, 16368) and not got[0]["left_good"]      # a hit on both strands: not good
    assert_same("whole_strand_16368", got, exp["whole_strand_16368"])


@pytest.mark.gpu
def test_unscored_long_anchor_is_counted(engine, cases):
    regs, exp, skipped, _cells = cases
    left, right, reads = regs["unscored_16384"]
    res, st = engine.anchor_regions(engine.get_preset("ont"), [left], [right], [reads])
    assert skipped["unscored_16384"] == 2 and st["n_skipped"] == 2
    assert_same("unscored_16384", got_records(res), exp["unscored_16384"])


@pytest.mark.gpu
def test_calls_back_to_back_reuse_the_scratch(engine, cases, oracle):
    """after the call above, a call with shorter multi-stripe reads, then one with longer ones: the per-warp scratch rows
    come back from the caching allocator holding entries of the earlier calls under the same tag"""
    regs, exp, _skipped, _cells = cases
    sc = engine.get_preset("ont")
    names = list(regs)
    engine.anchor_regions(sc, [regs[n][0] for n in names], [regs[n][1] for n in names], [regs[n][2] for n in names])
    longest = max(len(s) for n in names for s in regs[n][2] if scored_read(s) and stripes(regs[n][0], regs[n][1]) > 1)
    rng = np.random.default_rng(99)
    for nl, nr, read_len in ((1025, 769, 2500), (1537, 513, longest + 7000)):
        left, right = rand(rng, nl), rand(rng, nr)
        reads = [rand(rng, 30) + mutate(rng, left) + rand(rng, 50) + mutate(rng, right),
                 rc(left + rand(rng, 20) + right),
                 rand(rng, read_len - nl - nr - 60) + left + rand(rng, 60) + right,
                 rc(rand(rng, read_len - nl - nr - 61) + mutate(rng, left) + rand(rng, 61) + right)]
        assert stripes(left, right) > 1 and (max(map(len, reads)) < longest if read_len < longest else min(map(len, reads[2:])) > longest)
        res, st = engine.anchor_regions(sc, [left], [right], [reads])
        want, _sk, cells = expected(left, right, reads, oracle.max_threads())
        assert st["kernel_launches"] <= 2 and st["algorithmic_cells"] == cells
        assert_same(f"reuse_{read_len}", got_records(res), want)
        assert sum(o["accepted"] for o in want) >= 3
