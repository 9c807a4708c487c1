"""Inputs of the joint path's edge tests: tests/test_gpu_joint_edges.py holds nr_window_tasks and nr_joint_grid to the
CPU oracle on them, tests/test_oracle_joint_edges.py checks on the CPU that each named boundary really occurs in them.

Every read is built in template orientation by applying edits at stated template positions (`edit`); the GPU tests feed
it as given and as its reverse complement with reverse = 1, so both strands align the same oriented read.  Template
positions follow the window rule of tk.py:435-500 as the kernels restate it: an insertion placed before template base p
sits at position p and is charged when a < p < b - 1; a deletion's bases are charged where they lie in [a, b)."""
import os
import random
from concurrent.futures import ThreadPoolExecutor

COMP = {"A": "T", "C": "G", "G": "C", "T": "A", "N": "N"}
BASES = "ACGT"


def rs(rng, n):
    return "".join(rng.choice(BASES) for _ in range(n))


def revcomp(s):
    return "".join(COMP[c] for c in reversed(s))


def other(c, *avoid):
    """The first base that is neither c nor any of avoid."""
    return next(x for x in BASES if x != c and x not in avoid)


def edit(tpl, lo, hi, subs=(), dels=(), ins=None):
    """tpl[lo:hi] with mismatches at the positions in subs, deletions (start, length) and insertions {p: bases} placed
    before template base p (p == hi: after the last base)."""
    ins = ins or {}
    gone = {p for s, n in dels for p in range(s, s + n)}
    out = []
    for p in range(lo, hi):
        out.append(ins.get(p, ""))
        if p in gone:
            continue
        out.append(other(tpl[p]) if p in subs else tpl[p])
    out.append(ins.get(hi, ""))
    return "".join(out)


def pin_del(t, s, n):
    """Make a deletion of t[s:s+n] the only placement of its score (no shift left or right): t is a list, changed in place."""
    if s >= 1 and t[s - 1] == t[s + n - 1]:
        t[s - 1] = other(t[s + n - 1], t[s - 2] if s >= 2 else "")
    if s + n < len(t) and t[s] == t[s + n]:
        t[s + n] = other(t[s], t[s + n + 1] if s + n + 1 < len(t) else "")


def ins_bases(t, p, n):
    """n inserted bases that cannot slide off position p: none equals t[p - 1] or t[p]."""
    avoid = {t[p - 1] if p >= 1 else "", t[p] if p < len(t) else ""}
    pool = [c for c in BASES if c not in avoid]
    return "".join(pool[i % len(pool)] for i in range(n))


def clamp(a, b, t_len):
    """The window nr_window_tasks scores: [max(a, 0), min(b, |t|))."""
    return max(a, 0), min(b, t_len)


def oracle_map(oracle, jobs):
    """oracle.align_window over (query, target, a, b, reverse) jobs on a thread pool (ctypes releases the GIL)."""
    with ThreadPoolExecutor(max_workers=max(1, min(32, os.cpu_count() or 1))) as ex:
        return list(ex.map(lambda j: oracle.align_window(*j), jobs))


# ---- nr_window_tasks ---------------------------------------------------------------------------------------------------
READ_LENS = [1, 255, 256, 257, 511, 512, 513, 2049]
TPL_LENS = [1, 30, 31, 32, 33, 63, 64]
A, B = 150, 250                               # the window of the edge family, on a 400-base template; reads span [20, 380)


def window_cases():
    """Small nr_window_tasks cases: dicts (read, tpl, a, b, tag); `read` is the oriented read, a / b as passed."""
    rng = random.Random(2101)
    out = []
    # the 256-row stripes against the guarded ramps (31 steps) and the unrolled loop's odd / even trip count
    for q_len in READ_LENS:
        for t_len in TPL_LENS:
            tpl = rs(rng, t_len)
            if q_len <= t_len:
                s = (t_len - q_len) // 2
                read = edit(tpl, s, s + q_len, subs={s + q_len // 2} if q_len >= 3 else ())
            else:
                ins = {t_len // 2: ins_bases(tpl, t_len // 2, 2)} if t_len >= 30 else {}
                core = edit(tpl, 0, t_len, ins=ins)
                flank = max(0, min(256 - t_len // 2, q_len - len(core)))      # the alignment crosses row 256
                read = rs(rng, flank) + core
                read = (read + rs(rng, q_len))[:q_len]
            for a, b in ((t_len // 4, t_len - t_len // 4), (0, t_len)):
                out.append(dict(read=read, tpl=tpl, a=a, b=b, tag=f"shape q{q_len} t{t_len}"))
    # N in the read at rows 255, 256, 257 (stripe edge), inside the window and outside it
    tpl = rs(rng, 700)
    base = edit(tpl, 50, 650)
    for row in (255, 256, 257, 300, 100):
        out.append(dict(read=base[:row] + "N" + base[row + 1:], tpl=tpl, a=280, b=420, tag=f"N at row {row}"))
    # windows at and beyond the template's ends, empty, one to three bases (the insertion range a < p < b - 1 opens at
    # b = a + 3), reversed, and the whole template; the read has an insertion at 201, a deletion at 150, a mismatch at 260
    t = list(rs(rng, 400))
    pin_del(t, 150, 4)
    tpl = "".join(t)
    read = edit(tpl, 20, 380, subs={260}, dels=[(150, 4)], ins={201: ins_bases(tpl, 201, 3)})
    for a, b in ((-5, 100), (0, 120), (200, 200), (200, 201), (200, 202), (200, 203), (300, 400), (300, 450), (400, 500),
                 (450, 460), (250, 200), (0, 400), (-20, 999)):
        out.append(dict(read=read, tpl=tpl, a=a, b=b, tag=f"window [{a}, {b})"))
    # edits at the window's edges
    for p in (A - 1, A, B - 1, B):
        tpl = rs(rng, 400)
        out.append(dict(read=edit(tpl, 20, 380, subs={p}), tpl=tpl, a=A, b=B, tag=f"mismatch at {p}"))
    for s, n, tag in ((A - 1, 3, "del from a-1"), (A, 3, "del from a"), (B - 3, 3, "del to b-1"), (A - 2, B - A + 4, "del over window"),
                      (A + 30, 19, "del 19"), (A + 30, 20, "del 20"), (A + 30, 21, "del 21"), (A + 30, 35, "del 35"),
                      (A - 1, 19, "del 19 from a-1"), (A - 1, 21, "del 21 from a-1"), (B - 21, 21, "del 21 to b-1")):
        t = list(rs(rng, 400))
        pin_del(t, s, n)
        tpl = "".join(t)
        lo, hi = (0, 400) if n > 100 else (20, 380)
        out.append(dict(read=edit(tpl, lo, hi, dels=[(s, n)]), tpl=tpl, a=A, b=B, tag=tag))
    for p, n in ((A, 3), (A + 1, 3), (B - 2, 3), (B - 1, 3), (A + 1, 25), (B - 2, 1), (B - 1, 1)):
        tpl = rs(rng, 400)
        out.append(dict(read=edit(tpl, 20, 380, ins={p: ins_bases(tpl, p, n)}), tpl=tpl, a=A, b=B, tag=f"ins {n} at {p}"))
    return out


def n_template_case():
    rng = random.Random(2102)
    tpl = rs(rng, 100)
    return dict(read=tpl, tpl=tpl[:50] + "N" + tpl[51:], a=0, b=100, tag="template with N")


def limit_cases():
    """(case, skipped): the score, window and payload limits of nr_window_tasks, and reads as long as the joint CLI feeds."""
    rng = random.Random(2103)
    out = []
    t = rs(rng, 16384)
    out.append((dict(read=t[:16383], tpl=t[:16383], a=8000, b=8100, tag="score limit"), False))
    out.append((dict(read=t, tpl=t, a=8000, b=8100, tag="score limit + 1"), True))
    t = rs(rng, 8001)
    out.append((dict(read=t[:8000], tpl=t[:8000], a=0, b=8000, tag="window 8000"), False))
    out.append((dict(read=t, tpl=t, a=0, b=8001, tag="window 8001"), True))
    for g in (16355, 16356):
        c = payload_floor_case(g)
        out.append((c, False))
    for q_len, t_len in ((20000, 2000), (40000, 3000)):
        tpl = rs(rng, t_len)
        mid = edit(tpl, 0, t_len, subs=set(range(7, t_len, 97)), dels=[(t_len // 3, 5)], ins={2 * t_len // 3: "ACG"})
        read = rs(rng, (q_len - len(mid)) // 2) + mid
        read += rs(rng, q_len - len(read))
        out.append((dict(read=read, tpl=tpl, a=t_len // 4, b=3 * t_len // 4, tag=f"raw read {q_len}"), False))
    return out


PAYLOAD_FLOOR = {16355: (16387, -32706), 16356: (16386, -32708)}


def payload_floor_case(g):
    """Two 8 190-base flanks around a 3-base window [8190, 8193) (|t| = 16 383, 2 min(q, t) = 32 766: scored) and a read
    with g random bases inserted after the window's first base: the insertion is charged in full, -4 - 2 (g - 1)."""
    rng = random.Random(7)
    tpl = rs(rng, 8190 + 3 + 8190)
    read = tpl[:8191] + rs(rng, g) + tpl[8191:]
    return dict(read=read, tpl=tpl, a=8190, b=8193, tag=f"payload floor g={g}")


def template_limit_cases():
    """A 2^20-base template is scored, 2^20 + 1 bases are skipped (a call of its own: the scratch row is per template)."""
    rng = random.Random(2104)
    t = rs(rng, (1 << 20) + 1)
    read = t[500000:500200]
    return [(dict(read=read, tpl=t[:1 << 20], a=499990, b=500210, tag="template 2^20"), False),
            (dict(read=read, tpl=t, a=499990, b=500210, tag="template 2^20 + 1"), True)]


# ---- nr_joint_grid -----------------------------------------------------------------------------------------------------
MOTIF_PAIRS = [(1, 2), (2, 3), (3, 1), (4, 6), (5, 1), (6, 4)]


def template(locus, k1, k2):
    return locus["left"] + locus["m1"] * k1 + locus["mid"] + locus["m2"] * k2 + locus["right"]


def window_of(locus, k1, k2):
    """The window nanoRepeat-joint re-scores for grid point (k1, k2): [|L| - 10, J + 10) clamped to the template."""
    L, J = len(locus["left"]), junction(locus, k1, k2)
    return max(L - 10, 0), min(J + 10, len(template(locus, k1, k2)))


def junction(locus, k1, k2):
    return len(locus["left"]) + len(locus["m1"]) * k1 + len(locus["mid"]) + len(locus["m2"]) * k2


def _grid(reads, grids):
    pr, p1, p2 = [], [], []
    for r, (K1, K2) in enumerate(grids):
        for k1 in K1:
            for k2 in K2:
                pr.append(r); p1.append(k1); p2.append(k2)
    return pr, p1, p2


K1T, K2T = 3, 2                               # the true repeat counts of the geometry loci's reads


def junction_reads(locus, rng):
    """Reads of (K1T, K2T) with edits at the junction J and at the right anchor's window edge; dict tag -> read (template
    orientation)."""
    T = template(locus, K1T, K2T)
    J, nR = junction(locus, K1T, K2T), len(locus["right"])
    rd = {"whole": edit(T, 0, len(T), subs={J // 2})}
    for d in (0, 8, 9):
        rd[f"ins at J+{d}"] = edit(T, 0, len(T), ins={J + d: ins_bases(T, J + d, 2)})
    if J >= 3:
        rd["del over J (E1)"] = edit(T, 0, len(T), dels=[(J - 3, 6)])
    if J >= 12 and nR >= 13:
        rd["del over J (E2)"] = edit(T, 0, len(T), dels=[(J - 12, 25)])
    rd["del from R[9]"] = edit(T, 0, len(T), dels=[(J + 9, 1)])
    if nR >= 11:
        rd["del from R[10]"] = edit(T, 0, len(T), dels=[(J + 10, 1)])
    rd["ends at J"] = T[:J]
    rd["R only"] = locus["right"]
    rd["L only"] = locus["left"]
    x = T[max(0, J - 20):J]
    rd["palindrome"] = x + revcomp(x)
    return rd


def geometry_loci():
    """|R| in {10, 11, 41, 42, 43} x |L| in {1, 9, 10, 11, 12, 42}; mid '', one base or 12 bases; motifs of 1-6 bases with
    m1 != m2.  Grids: K1 and K2 from 0 (arithmetic), a single k1, steps above 1."""
    rng = random.Random(2201)
    loci = []
    for i, (nR, nL) in enumerate((r, l) for r in (10, 11, 41, 42, 43) for l in (1, 9, 10, 11, 12, 42)):
        m1n, m2n = MOTIF_PAIRS[i % len(MOTIF_PAIRS)]
        locus = dict(left=rs(rng, nL), mid=rs(rng, (0, 1, 12)[i % 3]), right=rs(rng, nR), m1=rs(rng, m1n), m2=rs(rng, m2n))
        while locus["m2"] == locus["m1"][:m2n]:
            locus["m2"] = rs(rng, m2n)
        rd = junction_reads(locus, rng)
        tags, reads, grids = [], [], []
        for j, (tag, read) in enumerate(rd.items()):
            tags.append(tag)
            reads.append(revcomp(read) if j % 2 else read)
            g = j % 4
            grids.append(([0, 1, 2, 3, 4, 5], [0, 1, 2, 3]) if g == 0 else ([K1T], [0, 1, 2, 3, 4]) if g == 1 else
                         ([1, 3, 5], [0, 2, 4]) if g == 2 else ([2, 3, 4], [1, 2, 3]))
        locus.update(reads=reads, tags=tags, points=_grid(reads, grids))
        loci.append(locus)
    return loci


def shape_locus():
    """|K2| = 64 (shared sweeps) and 65 (rectangles); |K1| = 64 (2-D sharing) and 65 (one sweep per k1); duplicated
    points, a grid that is not full, a read with no points and an empty read."""
    rng = random.Random(2202)
    locus = dict(left=rs(rng, 60), mid=rs(rng, 5), right=rs(rng, 60), m1="C", m2="AG")
    reads = []
    for k1, k2 in ((30, 20), (30, 20), (40, 10), (40, 10), (5, 5), (5, 5), (5, 5), (7, 3)):
        T = template(locus, k1, k2)
        reads.append(edit(T, 20, len(T) - 20, subs={len(T) // 2}, ins={len(T) // 3: "TT"}))
    reads[1], reads[3], reads[5] = revcomp(reads[1]), revcomp(reads[3]), revcomp(reads[5])
    reads += [reads[0][:50], ""]
    grids = [(range(0, 3), range(0, 64)), (range(0, 3), range(0, 65)), (range(0, 64), range(8, 11)), (range(0, 65), range(8, 11)),
             ([5], [2, 5, 8]), ([2, 5, 8], [5]), ([4, 5], [5, 6]), ([7], [3])]
    pr, p1, p2 = _grid(reads, grids + [([], []), ([1], [1])])
    pr += [4, 4, 7, 7, 7]; p1 += [5, 5, 7, 9, 9]; p2 += [5, 2, 3, 3, 4]           # duplicates; read 7's grid not full
    locus.update(reads=reads, tags=[f"shape read {r}" for r in range(len(reads))], points=(pr, p1, p2))
    return locus


def window_limit_locus():
    """One read whose largest template's window is 8 002 bases: its points of exactly 8 000 and less are scored, that one
    is skipped."""
    rng = random.Random(2203)
    locus = dict(left=rs(rng, 20), mid=rs(rng, 12), right=rs(rng, 30), m1="ACGA", m2="TC")
    read = locus["left"] + locus["m1"] * 100
    locus.update(reads=[read], tags=["window limit"], points=_grid([read], [([1989, 1990, 1991, 1992], [0, 1])]))
    return locus


def long_read_locus(n_distinct=4, q_len=40000):
    """A small locus and n_distinct reads of q_len bases holding its amplicon (k1, k2) = (2, 1) among random bases."""
    rng = random.Random(2204)
    locus = dict(left=rs(rng, 11), mid="", right=rs(rng, 10), m1="A", m2="C")
    reads = []
    for i in range(n_distinct):
        amp = edit(template(locus, 2, 1), 0, 24, subs={5 + i})
        s = rng.randint(0, q_len - len(amp))
        reads.append(rs(rng, s) + amp + rs(rng, q_len - s - len(amp)))
    locus["reads"] = reads
    return locus
