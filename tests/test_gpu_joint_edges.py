"""The joint path at its edges (SURVEY.md 8a row a7): nr_window_tasks (nr_window_kernel.cuh) and nr_joint_grid (the
shared sweeps of nr_window_ladder.cuh and their fall-backs) against the CPU oracle on EVERY task and grid point, with
edits placed on the window's edges, the junction J = |L| + m1 k1 + |mid| + m2 k2, the right anchor's window edge, the
256-row stripes, the 31-step ramps, and at the score, window, template, K2 / K1, 2-D state and offset limits.  The
inputs live in tests/helpers/joint_edges.py; tests/test_oracle_joint_edges.py checks on the CPU that each named
boundary really occurs in them."""
import numpy as np
import pytest

from helpers import joint_edges as je

pytestmark = pytest.mark.gpu


def _window_run(engine, oracle, cases, skipped=None):
    """Both strands of every case through one nr_window_tasks call; -> (got records, expected, stats).  The oracle is not
    run on the cases marked skipped (their expected record is None)."""
    sc = engine.get_preset("ont")
    qs, ts, aa, bb, rv, jobs = [], [], [], [], [], []
    for c in cases:
        a, b = je.clamp(c["a"], c["b"], len(c["tpl"]))
        for rev in (0, 1):
            q = je.revcomp(c["read"]) if rev else c["read"]
            qs.append(q); ts.append(c["tpl"]); aa.append(c["a"]); bb.append(c["b"]); rv.append(rev)
            jobs.append((q, c["tpl"], a, b, bool(rev)))
    got = engine.window_tasks(qs, ts, aa, bb, sc, reverse=rv)
    st = engine.last_stats()
    run = [i for i in range(len(jobs)) if not (skipped and skipped[i // 2])]
    exp = [None] * len(jobs)
    for i, e in zip(run, je.oracle_map(oracle, [jobs[i] for i in run])):
        exp[i] = e
    return [(int(g["score"]), int(g["window_score"])) for g in got], exp, st


def _assert_same(cases, got, exp, per=2):
    bad = [(i, cases[i // per]["tag"], got[i], exp[i]) for i in range(len(got)) if got[i] != exp[i]]
    assert not bad, (len(bad), len(got), bad[:10])


def test_window_tasks_edges_equal_oracle(engine, oracle):
    """Stripe heights x ramp widths, N at the stripe edge and in the window, every window shape, edits at a - 1, a, b - 1,
    b, deletions on both sides of the 20-base affine crossover, insertions at a, a + 1, b - 2, b - 1; a template holding
    N is (0, 0) and counted."""
    cases = je.window_cases()
    got, exp, st = _window_run(engine, oracle, cases + [je.n_template_case()])
    assert got[-2:] == [(0, 0), (0, 0)]
    _assert_same(cases, got[:-2], exp[:-2])
    assert st["n_tasks"] == 2 * len(cases) + 2 and st["n_skipped"] == 2 and st["kernel_launches"] == 1, st
    # both strands align the same oriented read
    assert got[0:-2:2] == got[1:-2:2]


def test_window_tasks_limits(engine, oracle):
    """Score limit 16 383 x 16 383 scored, one more base skipped; an 8 000-base window gives +16 000, 8 001 skipped; the
    payload floor (60 from the 16-bit decode limit); 20 kb and 40 kb raw reads against short templates."""
    lim = je.limit_cases()
    cases = [c for c, _ in lim]
    got, exp, st = _window_run(engine, oracle, cases, [s for _, s in lim])
    for i, (c, skipped) in enumerate(lim):
        for s in (0, 1):
            want = (0, 0) if skipped else exp[2 * i + s]
            assert got[2 * i + s] == want, (c["tag"], s, got[2 * i + s], exp[2 * i + s])
    by_tag = {c["tag"]: got[2 * i] for i, c in enumerate(cases)}
    assert by_tag["window 8000"] == (16000, 16000)
    assert by_tag["score limit"][0] == 2 * 16383
    for g, rec in je.PAYLOAD_FLOOR.items():
        assert by_tag[f"payload floor g={g}"] == rec
    assert st["n_skipped"] == 2 * sum(s for _, s in lim) and st["n_tasks"] == 2 * len(lim), st


def test_window_tasks_template_limit(engine, oracle):
    """A 2^20-base template with a 200-base read is scored; 2^20 + 1 bases are skipped and counted."""
    lim = je.template_limit_cases()
    cases = [c for c, _ in lim]
    got, exp, st = _window_run(engine, oracle, cases, [s for _, s in lim])
    assert got[:2] == exp[:2] == [(400, 400), (400, 400)]
    assert got[2:] == [(0, 0), (0, 0)]
    assert st["n_skipped"] == 2, st


def _grid_expected(oracle, locus, reads=None):
    """Per point max(align_window(read, tpl, a, b, 0), align_window(..., 1)), strand '+' on a full tie."""
    reads = locus["reads"] if reads is None else reads
    pr, p1, p2 = locus["points"]
    jobs = []
    for r, k1, k2 in zip(pr, p1, p2):
        tpl = je.template(locus, k1, k2)
        a, b = je.window_of(locus, k1, k2)
        jobs += [(reads[r], tpl, a, b, False), (reads[r], tpl, a, b, True)]
    res = je.oracle_map(oracle, jobs)
    exp = []
    for i in range(len(pr)):
        f, v = res[2 * i], res[2 * i + 1]
        exp.append((v, 1) if v > f else (f, 0))
    return exp


def _grid(engine, locus, reads=None, points=None):
    sc = engine.get_preset("ont")
    reads = locus["reads"] if reads is None else reads
    pr, p1, p2 = locus["points"] if points is None else points
    got, strand = engine.joint_grid(sc, locus["left"], locus["mid"], locus["right"], locus["m1"], locus["m2"], reads, pr, p1, p2)
    return [((int(g["score"]), int(g["window_score"])), int(s)) for g, s in zip(got, strand)], engine.last_stats()


def _check_locus(engine, oracle, locus, monkeypatch):
    got, st = _grid(engine, locus)
    exp = _grid_expected(oracle, locus)
    pr = locus["points"][0]
    bad = [(i, locus["tags"][pr[i]], got[i], exp[i]) for i in range(len(pr)) if got[i] != exp[i]]
    assert not bad, (len(locus["left"]), len(locus["mid"]), len(locus["right"]), locus["m1"], locus["m2"], len(bad), len(pr), bad[:8])
    assert st["n_tasks"] == len(pr) and st["n_skipped"] == 0, st
    # the same records on every path: one sweep per k1, and rectangles only
    for var in ("NR_JOINT_NO_2D", "NR_JOINT_RECTANGLES"):
        monkeypatch.setenv(var, "1")
        assert _grid(engine, locus)[0] == got, var
        monkeypatch.delenv(var)
    # each read alone equals its result inside the call
    for r in range(len(locus["reads"])):
        idx = [i for i in range(len(pr)) if pr[i] == r]
        if idx:
            pts = ([0] * len(idx), [locus["points"][1][i] for i in idx], [locus["points"][2][i] for i in idx])
            assert _grid(engine, locus, reads=[locus["reads"][r]], points=pts)[0] == [got[i] for i in idx], (locus["tags"][r])


def test_joint_grid_geometry_and_junction_edits_equal_oracle(engine, oracle, monkeypatch):
    """|R| in {10, 11, 41, 42, 43} x |L| in {1, 9, 10, 11, 12, 42}, mid of 0 / 1 / 12 bases, motifs of 1-6 bases; reads
    with insertions at J, J + 8, J + 9, junction-spanning deletions, deletions from R[9] and R[10], reads that end at J,
    lie in R or L only, and a palindrome."""
    for locus in je.geometry_loci():
        _check_locus(engine, oracle, locus, monkeypatch)


def test_joint_grid_shapes_equal_oracle(engine, oracle, monkeypatch):
    """|K2| = 64 / 65, |K1| = 64 / 65, duplicates, a grid that is not full, a read without points, an empty read."""
    _check_locus(engine, oracle, je.shape_locus(), monkeypatch)


def test_joint_grid_window_limit(engine, oracle):
    """The read's largest template has an 8 002-base window: that point is (0, 0) and counted once (not per strand); its
    8 000-base and smaller ones are scored."""
    locus = je.window_limit_locus()
    got, st = _grid(engine, locus)
    exp = _grid_expected(oracle, locus)
    pr, p1, p2 = locus["points"]
    for i in range(len(pr)):
        a, b = je.window_of(locus, p1[i], p2[i])
        if b - a > 8000:
            assert got[i] == ((0, 0), 0), (p1[i], p2[i])
        else:
            assert got[i] == exp[i] and exp[i][0][0] > 0, (p1[i], p2[i], got[i], exp[i])
    assert sum(je.window_of(locus, k1, k2)[1] - je.window_of(locus, k1, k2)[0] == 8000 for k1, k2 in zip(p1, p2)) == 1
    assert st["n_skipped"] == 1 and st["n_tasks"] == len(pr), st


def _copies(locus, n_reads, k1s, k2s):
    """n_reads copies of the locus's distinct reads, each with the grid k1s x k2s."""
    d = locus["reads"]
    reads = [d[r % len(d)] for r in range(n_reads)]
    pr, p1, p2 = [], [], []
    for r in range(n_reads):
        for k1 in k1s:
            for k2 in k2s:
                pr.append(r); p1.append(k1); p2.append(k2)
    return reads, (pr, p1, p2)


def _check_copies(engine, oracle, locus, reads, points, got):
    """Every copy equals its distinct read's result in a call of its own, and that equals the oracle."""
    d = locus["reads"]
    pr, p1, p2 = points
    n_per = len(pr) // len(reads)
    rows = np.array([[g[0][0], g[0][1], g[1]] for g in got]).reshape(len(reads), n_per, 3)
    for j in range(len(d)):
        idx = list(range(j * n_per, (j + 1) * n_per))
        pts = ([0] * n_per, [p1[i] for i in idx], [p2[i] for i in idx])
        alone, _ = _grid(engine, locus, reads=[d[j]], points=pts)
        exp = _grid_expected(oracle, dict(locus, points=pts), reads=[d[j]])
        assert alone == exp, (j, alone, exp)
        want = np.array([[g[0][0], g[0][1], g[1]] for g in alone])
        same = (rows[j::len(d)] == want[None]).all(axis=(1, 2))
        assert same.all(), (j, int((~same).sum()), np.nonzero(~same)[0][:5])


def test_joint_grid_2d_budget_runs_out_part_way(engine, oracle):
    """|K1| = 2 on 1 200 reads of 40 kb: the 2-D state budget (2^29 words, 12 per read base here) lasts for 1 118 reads,
    the rest take one sweep per k1; every read equals its result alone."""
    locus = je.long_read_locus()
    reads, points = _copies(locus, 1200, [1, 2], [1])
    got, st = _grid(engine, locus, reads=reads, points=points)
    assert st["n_skipped"] == 0 and st["n_tasks"] == len(points[0]), st
    _check_copies(engine, oracle, locus, reads, points, got)


def test_joint_grid_junction_vectors_past_2_31_words(engine, oracle):
    """9 100 reads of 40 kb with one point each: 6 junction-vector words per read base, 2.18 G words in all, so the reads
    after the first ~8 948 sit past 2^31 words (64-bit offsets)."""
    locus = je.long_read_locus()
    reads, points = _copies(locus, 9100, [2], [1])
    assert 6 * sum(len(r) for r in reads) > 2 ** 31
    got, st = _grid(engine, locus, reads=reads, points=points)
    assert st["n_skipped"] == 0, st
    _check_copies(engine, oracle, locus, reads, points, got)
