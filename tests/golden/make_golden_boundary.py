#!/usr/bin/env python
"""Generate tests/golden/boundary_shape.json: the slice of the reference's NanoRepeat.nanoRepeat_bam that install()
depends on, read from the reference's own, unmodified sources (NANOREPEAT_REFERENCE_SRC = its src/ directory).

  signatures                       parameter lists of the two functions install() replaces (nanoRepeat_bam.py:334, :446)
  quantify1repeat_from_bam_calls   which of them quantify1repeat_from_bam calls by name, i.e. through the module's
                                   globals, so that patching the module takes effect (:675-679)
  read_defaults_none               the Read attributes the operators read or write that a fresh Read holds as None
  repeat_region_attributes         the RepeatRegion attributes the operators read (repeat_region.py:32-55, :116-151)

tests/test_boundary.py asserts install() and the package's own Read / RepeatRegion against this file, and re-derives
it with shape() when the reference sources are given.

Usage: NANOREPEAT_REFERENCE_SRC=<NanoRepeat>/src python tests/golden/make_golden_boundary.py
"""
import inspect
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))

PATCHED = ("round1_and_round2_estimation", "round3_estimation")
READ_ATTRS = ("dist_between_anchors", "round1_repeat_size", "round2_repeat_size", "round3_repeat_size")
REGION_ATTRS = ("left_anchor_seq", "right_anchor_seq", "repeat_unit_seq", "read_dict", "read_core_seq_dict")


def shape(ref_bam, ref_rr):
    """The dictionary stored in boundary_shape.json, from the reference's nanoRepeat_bam and repeat_region modules."""
    src = inspect.getsource(ref_bam.quantify1repeat_from_bam)
    rd, rr = ref_rr.Read(), ref_rr.RepeatRegion()
    return dict(signatures={n: list(inspect.signature(getattr(ref_bam, n)).parameters) for n in PATCHED},
                quantify1repeat_from_bam_calls=[n for n in PATCHED if n + "(" in src],
                read_defaults_none=[a for a in READ_ATTRS if hasattr(rd, a) and getattr(rd, a) is None],
                repeat_region_attributes=[a for a in REGION_ATTRS if hasattr(rr, a)])


def main():
    sys.path.insert(0, os.environ["NANOREPEAT_REFERENCE_SRC"])
    sys.path.insert(0, HERE)
    import make_golden
    doc = dict(source="NanoRepeat.nanoRepeat_bam / repeat_region (reference, unmodified), tests/golden/make_golden_boundary.py",
               **shape(*make_golden.import_reference()))
    path = os.path.join(HERE, "boundary_shape.json")
    with open(path, "w") as f:
        json.dump(doc, f, indent=1)
        f.write("\n")
    print("wrote", path)


if __name__ == "__main__":
    main()
