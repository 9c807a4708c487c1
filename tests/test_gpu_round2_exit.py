"""Round 2's dominance exit (nr_pair_kernels.cuh, Sweep::run; DESIGN.md section 4.9): a pair's sweep ends once the DP
cut is dominated by the cut one period earlier.  Records must be bit for bit those of the full sweep and of the oracle,
with the exit on and off (NR_ROUND2_EXIT=0, read when a batch is committed)."""
import os
import random

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _rand_seq(rng, n):
    return "".join(rng.choice("ACGT") for _ in range(n))


def _mutate(rng, s, rate):
    out = []
    for c in s:
        u = rng.random()
        if u < rate / 3:
            continue                                   # deletion
        if u < 2 * rate / 3:
            out.append(rng.choice("ACGT"))             # substitution
        elif u < rate:
            out.append(c + rng.choice("ACGT"))         # insertion
        else:
            out.append(c)
    return "".join(out)


def _run(engine, sc, left, motif, T, cores, exit_on):
    old = os.environ.get("NR_ROUND2_EXIT")
    os.environ["NR_ROUND2_EXIT"] = "1" if exit_on else "0"
    try:
        with engine.Batch.begin(sc, "round2_flags") as b:
            b.add_round2(left, motif, T, cores)
            res = b.commit().run().fetch_round2()
            return res, b.launch_info()
    finally:
        if old is None:
            del os.environ["NR_ROUND2_EXIT"]
        else:
            os.environ["NR_ROUND2_EXIT"] = old


def _check(engine, oracle, left, motif, T, cores, what):
    sc = engine.get_preset("ont")
    ref = oracle.align_batch(cores, [left + motif * T] * len(cores), n_threads=oracle.max_threads())
    (on, li_on), (off, li_off) = _run(engine, sc, left, motif, T, cores, True), _run(engine, sc, left, motif, T, cores, False)
    for a, b in zip(on, off):
        assert np.array_equal(a, b), what
    score, tend, inside = on
    assert np.array_equal(score, ref["score"]), what
    spans = ref["tend"] >= len(left)
    assert np.array_equal(tend[spans], ref["tend"][spans]), what
    live = (ref["score"] > 0) & spans
    assert np.array_equal(inside[live], (ref["tstart"] <= len(left))[live]), what
    assert li_off["paired_cells"] == li_off["planned_paired_cells"], what
    assert li_on["planned_paired_cells"] == li_off["planned_paired_cells"], what
    assert li_on["paired_cells"] <= li_on["planned_paired_cells"], what
    return li_on


def _flanked(rng, left, motif, k, rate, right_len=100):
    return _mutate(rng, left[-100:] + motif * k + _rand_seq(rng, right_len), rate)


@pytest.mark.parametrize("m", [1, 2, 3, 4, 5, 6])
def test_long_template_short_repeats(engine, oracle, m):
    """T far beyond the reads' repeats: the exit fires (fewer cells than planned) and every record stays exact;
    motif lengths 1-6, including lengths that do not divide 16."""
    rng = random.Random(100 + m)
    left = _rand_seq(rng, 400)
    motif = _rand_seq(rng, m) if m > 1 else "A"
    while m > 1 and len(set(motif)) == 1:
        motif = _rand_seq(rng, m)
    T = 600 // m
    cores = [_flanked(rng, left, motif, rng.randint(3, 60 // m + 5), rng.choice([0.0, 0.05, 0.1])) for _ in range(40)]
    li = _check(engine, oracle, left, motif, T, cores, f"m={m}")
    assert li["paired_cells"] < li["planned_paired_cells"], m
    assert li["paired_useful_cells"] < li["planned_paired_useful_cells"], m


def test_short_template_does_not_fire(engine, oracle):
    rng = random.Random(7)
    left, motif = _rand_seq(rng, 200), "CAG"
    cores = [_flanked(rng, left, motif, rng.randint(5, 20), 0.05) for _ in range(20)]
    li = _check(engine, oracle, left, motif, 22, cores, "T = 22")
    assert li["paired_cells"] == li["planned_paired_cells"]


def test_ties_marks_halves_and_ambiguous_bases(engine, oracle):
    """Equal scores later in the template (smallest tend must survive), best alignments that start inside the left
    anchor and after it, pairs whose halves are dominated at very different columns, reads with N."""
    rng = random.Random(11)
    left, motif = _rand_seq(rng, 300), "CAG"
    T = 250
    cores = []
    for i in range(96):
        kind = i % 6
        k = rng.randint(2, 40)
        if kind == 0:
            cores.append(motif * k)                                        # starts past |left|; ties along the repeat
        elif kind == 1:
            cores.append(left[-1:] + motif * k)                            # one flank base: ties on tstart
        elif kind == 2:
            cores.append(_flanked(rng, left, motif, k, 0.05))
        elif kind == 3:
            cores.append(_flanked(rng, left, motif, rng.randint(150, 200), 0.03, 20))   # dominated much later
        elif kind == 4:
            s = list(_flanked(rng, left, motif, k, 0.02))
            for _ in range(rng.randint(1, 8)):
                s[rng.randrange(len(s))] = "N"
            cores.append("".join(s))
        else:
            cores.append(_rand_seq(rng, rng.randint(20, 120)))             # unrelated
    li = _check(engine, oracle, left, motif, T, cores, "mixed")
    assert li["paired_cells"] < li["planned_paired_cells"]


def test_round3_resumed_from_exited_round2(engine, oracle):
    """Round 3 resumes from the state round 2 keeps at column |left| - 2, before any exit: the same selections as a
    fresh round 3 over the same reads, with the exit on and off."""
    rng = random.Random(23)
    left, right, motif = _rand_seq(rng, 300), _rand_seq(rng, 200), "CAG"
    ks = [rng.choice([17, 55]) for _ in range(60)]
    cores = [_mutate(rng, left[-100:] + motif * k + right[:100], 0.04) for k in ks]
    kmin = np.array([max(0, k - 3) for k in ks], np.int32)
    kmax = np.array([k + 3 for k in ks], np.int32)
    sc = engine.get_preset("ont")
    with engine.Batch.round3(sc, left, right, motif, cores, kmin, kmax) as b:
        fresh = b.run().fetch_round3()
    for exit_on in (True, False):
        os.environ["NR_ROUND2_EXIT"] = "1" if exit_on else "0"
        try:
            with engine.Batch.begin(sc, "round2_flags") as b2:
                b2.add_round2(left, motif, 120, cores).commit().run()
                with engine.Batch.begin_round3_from(b2) as b3:
                    got = b3.add_round3_reuse(0, right, kmin, kmax).commit().run().fetch_round3()
                if exit_on:
                    li = b2.launch_info()
                    assert li["paired_cells"] < li["planned_paired_cells"]
        finally:
            del os.environ["NR_ROUND2_EXIT"]
        for a, b in zip(got, fresh):
            assert np.array_equal(a, b), exit_on
