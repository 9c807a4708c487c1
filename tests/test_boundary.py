"""The drop-in boundary as the reference would use it (SURVEY.md section 8b): install() on a module of the reference's
shape, the reference's own Read / RepeatRegion classes, pickling through the result queue, fork-after-load with several
workers, and the pymm2.main-shaped shim."""
import inspect
import json
import os
import pickle
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# the original NanoRepeat's src/ directory; it is not part of this repository: given, the boundary shape stored under
# tests/golden is re-checked against it and the shim runs under the reference's own round functions
REF_SRC = os.environ.get("NANOREPEAT_REFERENCE_SRC", "")
NO_REF = "needs the original NanoRepeat sources: set NANOREPEAT_REFERENCE_SRC to its src/ directory"


def _import_reference_module():
    """NanoRepeat.nanoRepeat_bam from REF_SRC with its absent third-party imports stubbed."""
    sys.path.insert(0, REF_SRC)
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import make_golden
    return make_golden.import_reference()


def test_install_matches_the_reference_module_shape():
    """install() patches exactly the names quantify1repeat_from_bam calls, with the reference's parameter lists; the
    package's Read / RepeatRegion carry every attribute the operators read or write, with the reference's defaults
    (tests/golden/boundary_shape.json).  With the reference sources given, the stored shape is re-derived from them and
    install() is run on the reference's own module as well."""
    import types
    import nanorepeat_b200 as nrb
    from conftest import load_golden
    want = load_golden("boundary_shape")
    del want["source"]
    assert set(want["quantify1repeat_from_bam_calls"]) == set(want["signatures"])       # looked up in module globals
    modules = [types.ModuleType("nanoRepeat_bam")]
    if os.path.isdir(REF_SRC):
        ref_bam, ref_rr = _import_reference_module()
        import make_golden_boundary
        assert make_golden_boundary.shape(ref_bam, ref_rr) == want
        pickle.dumps(ref_rr.RepeatRegion())
        modules.append(ref_bam)
    for mod in modules:
        before = dict(vars(mod))
        try:
            nrb.install(mod)
            changed = {n for n, v in vars(mod).items() if before.get(n, None) is not v}
            assert changed == set(want["signatures"]), changed
            for name, params in want["signatures"].items():
                assert getattr(mod, name) is getattr(nrb, name)
                assert list(inspect.signature(getattr(nrb, name)).parameters) == params, name
        finally:
            for name in want["signatures"]:
                if name in before:
                    setattr(mod, name, before[name])
    rd, rr = nrb.Read(), nrb.RepeatRegion()
    for attr in want["read_defaults_none"]:
        assert hasattr(rd, attr) and getattr(rd, attr) is None, attr
    for attr in want["repeat_region_attributes"]:
        assert hasattr(rr, attr), attr
    pickle.dumps(rr)


@pytest.mark.skipif(not os.path.isdir(REF_SRC), reason=NO_REF)
def test_shim_feeds_the_unmodified_reference_functions(monkeypatch, tmp_path):
    """The reference's UNMODIFIED round1_and_round2_estimation / round3_estimation on top of pymm2_shim.main, with the
    engine call inside the shim answered by the oracle (no GPU here): the shim's file handling, command recognition and
    PAF text must give the reference's functions what the golden fixtures say."""
    from conftest import load_golden
    from nanorepeat_b200 import pymm2_shim, engine
    from oracle import nr_oracle
    ref_bam, ref_rr = _import_reference_module()
    monkeypatch.setattr(engine, "get_preset", lambda dt: nr_oracle.scoring())
    monkeypatch.setattr(engine, "score_tasks", lambda q, t, sc: nr_oracle.align_batch(q, t, sc, n_threads=nr_oracle.max_threads()))
    monkeypatch.setattr(ref_bam, "pymm2", pymm2_shim)
    doc = load_golden("cfg1_small")
    reg = doc["regions"][0]
    R = ref_rr.RepeatRegion()
    R.left_anchor_seq, R.right_anchor_seq, R.repeat_unit_seq = reg["left"], reg["right"], reg["motif"]
    R.left_anchor_len, R.right_anchor_len = len(reg["left"]), len(reg["right"])
    R.temp_out_dir = str(tmp_path)
    R.core_seq_fq_file = str(tmp_path / "core_sequences.fastq")
    with open(R.core_seq_fq_file, "w") as f:
        for name, core, dist in zip(reg["read_names"], reg["cores"], reg["dists"]):
            rd = ref_rr.Read()
            rd.read_name, rd.dist_between_anchors = name, dist
            R.read_dict[name] = rd
            R.read_core_seq_dict[name] = core
            f.write(f"@{name}\n{core}\n+\n{'0' * len(core)}\n")
    ref_bam.round1_and_round2_estimation(reg["data_type"], R, 1)
    ref_bam.round3_estimation(reg["data_type"], doc["fast_mode"], R, 1)
    for name, exp in zip(reg["read_names"], reg["expected"]):
        rd = R.read_dict[name]
        assert (rd.round1_repeat_size, rd.round2_repeat_size) == (exp["r1"], exp["r2"])
        assert (None if rd.round3_repeat_size is None else float(rd.round3_repeat_size)) == exp["r3"]


def test_shim_prints_the_paf_the_golden_fixtures_were_made_from(monkeypatch, tmp_path):
    """The part of the test above that needs no reference sources: on the reference's round-2 command and, for every
    read round 2 placed, its round-3 command over the ladder the reference builds (oracle/selection.ladder_bounds,
    nanoRepeat_bam.py:463-472), pymm2_shim.main (engine call answered by the oracle) prints, line for line, the columns
    the reference reads (query, target, target length, target start / end, AS) as the stand-in aligner whose PAF the
    reference's functions turned into tests/golden/cfg1_small.json (tests/golden/make_golden.py).  Any other command
    (Step 1's anchor search) is refused."""
    from conftest import load_golden
    from nanorepeat_b200 import pymm2_shim, engine
    from oracle import nr_oracle, selection
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import make_golden
    monkeypatch.setattr(engine, "get_preset", lambda dt: nr_oracle.scoring())
    monkeypatch.setattr(engine, "score_tasks", lambda q, t, sc: nr_oracle.align_batch(q, t, sc, n_threads=nr_oracle.max_threads()))
    doc = load_golden("cfg1_small")
    reg = doc["regions"][0]
    left, right, motif = reg["left"], reg["right"], reg["motif"]
    r1_max = max(reg["dists"]) / len(motif)                                   # round-2 template, :339-355
    T = int(r1_max * 1.5) + 1
    if T < r1_max + 10:
        T = int(r1_max + 10)
    (tmp_path / "round1_ref.fasta").write_text(f">{T}\n{left}{motif * T}\n")
    with open(tmp_path / "core_sequences.fastq", "w") as f:
        for name, core in zip(reg["read_names"], reg["cores"]):
            f.write(f"@{name}\n{core}\n+\n{'0' * len(core)}\n")
    cmds = [f"-c -t 1 -x map-ont -f 0.0 {tmp_path}/round1_ref.fasta {tmp_path}/core_sequences.fastq"]
    for i, (name, core, exp) in enumerate(zip(reg["read_names"], reg["cores"], reg["expected"])):
        if exp["r2"] is None:
            continue
        kmin, kmax = selection.ladder_bounds(exp["r2"], doc["fast_mode"])
        ladder = tmp_path / f"round3_reference.{kmin}-{kmax}.fasta"
        ladder.write_text("".join(f">{k}\n{left}{motif * k}{right}\n" for k in range(kmin, kmax + 1)))
        (tmp_path / f"round3_input.read{i}.fasta").write_text(f">{name}\n{core}\n")
        cmds.append(f"-x map-ont -f 0.0 -N 100 -c --eqx -t 1 {ladder} {tmp_path}/round3_input.read{i}.fasta")
    assert len(cmds) >= 4

    def columns(paf):
        return [[r[i] for i in (0, 5, 6, 7, 8, 12)] for r in (ln.split("\t") for ln in paf.splitlines())]
    for cmd in cmds:
        got, want = pymm2_shim.main(cmd)[0], make_golden.fake_pymm2_main(cmd)[0]
        assert len(columns(got)) >= 2 and columns(got) == columns(want), cmd
    with pytest.raises(NotImplementedError):
        pymm2_shim.main("-c -t 4 -x map-ont anchors.fasta region.fastq")       # Step 1's command is not this library's


@pytest.mark.gpu
def test_installed_operators_on_reference_shaped_objects_pickle(engine):
    """install() on a module of the reference's shape; its driver calls the two names through the module globals on
    objects with the reference's attribute set; the region then pickles (it crosses a multiprocessing queue in the
    reference, nanoRepeat_bam.py:610) after EACH operator, and the results equal the direct calls."""
    import nanorepeat_b200 as nrb
    from nanorepeat_b200 import synth
    from helpers import refshape
    own = (refshape.round1_and_round2_estimation, refshape.round3_estimation)
    nrb.install(refshape)
    try:
        regs = synth.config1(seed=5, n_regions=3, reads_per_region=10)
        for mode in (3, 0):                        # the production ladder and the independent-rectangle checking mode
            engine.set_ladder_mode(mode)
            for reg in regs:
                rr = refshape.region_from_synth(reg)
                refshape.round1_and_round2_estimation("ont", rr, 4)
                mid = pickle.loads(pickle.dumps(rr))                 # between the two operators
                assert [rd.round2_repeat_size for rd in mid.read_dict.values()] == [rd.round2_repeat_size for rd in rr.read_dict.values()]
                refshape.round3_estimation("ont", False, rr, 4)
                back = pickle.loads(pickle.dumps(rr))
                direct = nrb.RepeatRegion.from_synth(reg)
                nrb.estimate_regions([direct], "ont", False)
                for name, rd in direct.read_dict.items():
                    o = back.read_dict[name]
                    assert (rd.round1_repeat_size, rd.round2_repeat_size, rd.round3_repeat_size) == \
                           (o.round1_repeat_size, o.round2_repeat_size, o.round3_repeat_size), (mode, name)
                assert not [k for k in vars(rr) if k.startswith("_nr")]      # nothing of ours is left on the object
                assert sum(rd.round3_repeat_size is not None for rd in rr.read_dict.values()) >= 8
    finally:
        engine.set_ladder_mode(3)
        refshape.round1_and_round2_estimation, refshape.round3_estimation = own


@pytest.mark.gpu
def test_fork_after_load_four_workers():
    """The reference forks up to 16 workers after importing everything (nanoRepeat_bam.py:719-724): the library is loaded
    before the fork, every worker initialises CUDA on its own, results come back pickled and equal the parent's."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "helpers", "fork_workers.py"), "4"],
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    res = json.loads(out.stdout.strip().splitlines()[-1])
    assert res["exitcodes"] == [0, 0, 0, 0] and res["regions_back"] == 12 and res["equal"], res
    assert res["reads_with_round3"] > 80


@pytest.mark.gpu
def test_pymm2_shim_on_the_gpu(engine, oracle, tmp_path):
    """The two hot-path command shapes through pymm2_shim.main on the CUDA engine: PAF text whose AS / tstart / tend are
    the oracle's, one line per template at or above minimap2's -s, best first."""
    from nanorepeat_b200 import pymm2_shim, synth
    reg = synth.config1(seed=9, n_regions=1, reads_per_region=7)[0]
    m = len(reg.repeat_unit_seq)
    tpl = reg.left_anchor_seq + reg.repeat_unit_seq * 70
    (tmp_path / "round1_ref.fasta").write_text(f">70\n{tpl}\n")
    with open(tmp_path / "core_sequences.fastq", "w") as f:
        for n, c in zip(reg.read_names, reg.core_seqs):
            f.write(f"@{n}\n{c}\n+\n{'0' * len(c)}\n")
    out, err = pymm2_shim.main(f"-c -t 4  -x map-ont  -f 0.0 {tmp_path}/round1_ref.fasta {tmp_path}/core_sequences.fastq")
    ref = oracle.align_batch(reg.core_seqs, [tpl] * len(reg.core_seqs))
    rows = [ln.split("\t") for ln in out.strip().split("\n")]
    assert [r[0] for r in rows] == reg.read_names
    for r, a in zip(rows, ref):
        assert (int(r[7]), int(r[8]), r[12]) == (int(a["tstart"]), int(a["tend"]), f"AS:i:{int(a['score'])}") and r[5] == "70"
    # round 3: one read against a ladder file
    ks = list(range(3, 12))
    with open(tmp_path / "round3_reference.3-11.fasta", "w") as f:
        for k in ks:
            f.write(f">{k}\n{reg.left_anchor_seq}{reg.repeat_unit_seq * k}{reg.right_anchor_seq}\n")
    (tmp_path / "round3_input.read0.fasta").write_text(f">{reg.read_names[0]}\n{reg.core_seqs[0]}\n")
    out, err = pymm2_shim.main(f" -x map-ont  -f 0.0 -N 100 -c --eqx -t 4 {tmp_path}/round3_reference.3-11.fasta {tmp_path}/round3_input.read0.fasta")
    ref, _off = oracle.align_ladders([reg.core_seqs[0]], reg.left_anchor_seq, reg.right_anchor_seq, reg.repeat_unit_seq, [3], [11])
    rows = {int(r[5]): r for r in (ln.split("\t") for ln in out.strip().split("\n"))}
    for k, a in zip(ks, ref):
        if a["score"] >= 80:
            assert (int(rows[k][7]), int(rows[k][8]), rows[k][12]) == (int(a["tstart"]), int(a["tend"]), f"AS:i:{int(a['score'])}")
            assert int(rows[k][6]) == len(reg.left_anchor_seq) + m * k + len(reg.right_anchor_seq)
        else:
            assert k not in rows
    scores = [int(ln.split("\t")[12][5:]) for ln in out.strip().split("\n")]
    assert scores == sorted(scores, reverse=True)
