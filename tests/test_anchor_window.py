"""The start-recovery lemma of nr_anchor_regions (nr_anchor.cu), on the CPU oracle: for an anchor's best hit (S, tend) on
a read, the exact record of the anchor against read[a, tend), a = max(0, tend - W),
W = n + max(0, (match * n - S - min(q, q2)) // min(e, e2)), is (S, tstart - a, tend - a) -- the full read's record."""
import numpy as np

from nanorepeat_b200.synth import mutate, random_seq

MATCH, Q1, Q2, E1, E2 = 2, 4, 24, 2, 1          # map-ont


def window_of(n, score, tend):
    w = n + max(0, (MATCH * n - score - min(Q1, Q2)) // min(E1, E2))
    return max(0, tend - w)


def check(oracle, anchor, reads):
    full = oracle.align_batch([anchor] * len(reads), reads)
    cases = [(r, int(f["score"]), int(f["tstart"]), int(f["tend"])) for r, f in zip(reads, full) if f["score"] > 0]
    wins = [window_of(len(anchor), s, te) for _r, s, _ts, te in cases]
    got = oracle.align_batch([anchor] * len(cases), [r[a:te] for (r, _s, _ts, te), a in zip(cases, wins)])
    for (r, s, ts, te), a, g in zip(cases, wins, got):
        assert (int(g["score"]), a + int(g["tstart"]), a + int(g["tend"])) == (s, ts, te), (len(anchor), len(r), s, ts, te, a)
    return len(cases)


def test_window_record_equals_full_read_record_random(oracle):
    rng = np.random.default_rng(11)
    for n in (1000, 600, 97, 12):
        anchor = random_seq(rng, n)
        reads = []
        for _ in range(12):
            hit = mutate(rng, anchor, 0.05, 0.03, 0.03)
            reads.append(random_seq(rng, int(rng.integers(0, 900))) + hit + random_seq(rng, int(rng.integers(0, 900))))
        reads += [random_seq(rng, int(rng.integers(1, 3000))) for _ in range(4)]            # unrelated reads
        assert check(oracle, anchor, reads) >= 12


def test_window_record_equals_full_read_record_adversarial(oracle):
    rng = np.random.default_rng(12)
    anchor = random_seq(rng, 300)
    reads = []
    # long deletions inside the alignment, up to the bound: the read holds the anchor with l extra bases in its middle
    for l in (1, 50, 250, 500, 560, 590, 595, 700):
        reads.append(random_seq(rng, 40) + anchor[:150] + random_seq(rng, l) + anchor[150:] + random_seq(rng, 40))
        reads.append(anchor[:150] + "A" * l + anchor[150:])
        reads.append(anchor[:20] + random_seq(rng, l) + anchor[20:])
    # the anchor twice on one strand with equal scores: the smallest tend wins
    reads.append(random_seq(rng, 30) + anchor + random_seq(rng, 77) + anchor + random_seq(rng, 12))
    reads.append(anchor + anchor)
    # hits at the read's start and end, and reads shorter than the anchor
    reads += [anchor + random_seq(rng, 100), random_seq(rng, 100) + anchor, anchor, anchor[40:260], anchor[:100], anchor[-90:]]
    reads.append(mutate(rng, anchor, 0.1, 0.1, 0.1))
    assert check(oracle, anchor, reads) == len(reads)
    short = random_seq(rng, 45)                                                               # short anchors
    assert check(oracle, short, [short, "GG" + short + "TT", short[:30] + random_seq(rng, 60) + short[30:], short + short]) == 4
