"""Step 1 of the reference's per-region pipeline on the GPU: locate the two anchors in every read and cut the core.

    find_anchor_locations_in_regions <- reference src/NanoRepeat/nanoRepeat_bam.py:260-286 (+ :165-258), many regions
    find_anchor_locations_in_reads   <- the same for one region
    make_core_seq_fastq              <- reference src/NanoRepeat/nanoRepeat_bam.py:288-331

The reference aligns every read of the region to `left_anchor` / `right_anchor` (<= 1000 bp each) with
`minimap2 -c -x map-ont` and keeps a read when both anchors are found unambiguously on one strand (:165-219); the core
handed to rounds 1-3 is read[left.qend - 100 : right.qstart + 100] in the read's orientation (:221-234, :308-316).
Here the four alignments per read (two anchors x two strands) are exact local alignments on the CUDA engine with the
ANCHOR as the DP's query and the READ as its target, so the record's (tstart, tend) are the read coordinates the rules
need (paf.qstart / paf.qend in the read's orientation, paf.py:70-74).

What is the reference's and what is not.  The acceptance rules -- one hit: good; several: best AS > 1.5 x second AS;
both anchors good and on one strand; dist = right.qstart - left.qend > -10; the core / mid slicing with its 100-base
buffers and clamps -- are the reference's, line for line.  What minimap2 decides heuristically is replaced by a stated
rule: the candidate hits of an anchor are its best exact alignment on each strand that reaches minimap2's -s (80), so
"second AS" is the other strand's; `mapq > 30` is taken as true whenever the 1.5 x rule holds (mapq is a function of
exactly that score ratio and chain properties this engine does not have); `align_len < 10` cannot occur above -s.
A read longer than the engine's template limit (65 471 bases) is left out, as a read minimap2 printed nothing for.
The rules run inside the library (nr_anchor_regions, include/nanorepeat_b200.h), one call for any number of regions.
"""
import os

import numpy as np

from . import engine
from .presets import get_preset_for_minimap2

_COMP = str.maketrans("ACGTacgtNn", "TGCAtgcaNn")
BUFFER_LEN = 100                       # nanoRepeat_bam.py:221


def rev_comp(seq):
    """tk.rev_comp (tk.py:346-355) -- which raises on anything but ACGT; here N stays N."""
    return seq.translate(_COMP)[::-1]


def read_fastq(path):
    """-> ([name, ...], [sequence, ...]) exactly as make_core_seq_fastq walks the file (:298-309)."""
    names, seqs = [], []
    with open(path) as f:
        while True:
            l1, l2, l3, l4 = f.readline(), f.readline(), f.readline(), f.readline()
            if not l1 or not l2 or not l3 or not l4:
                break
            names.append(l1.strip()[1:])
            seqs.append(l2.strip())
    return names, seqs


class AnchorHit:
    """The slice of a PAF record Step 1 reads (paf.py:39-74), coordinates in the read's orientation."""
    __slots__ = ("strand", "align_score", "qstart", "qend", "align_len", "mapq")

    def __init__(self, strand, align_score, qstart, qend):
        self.strand, self.align_score, self.qstart, self.qend = strand, align_score, qstart, qend
        self.align_len = qend - qstart
        self.mapq = 60


def _reads_of(repeat_region, reads):
    """(names, sequences) of a region's reads: given as such, as {name: sequence}, or (None) from its region FASTQ."""
    if reads is None:
        return read_fastq(repeat_region.region_fq_file)
    if isinstance(reads, dict):
        return list(reads), list(reads.values())
    return reads


def find_anchor_locations_in_regions(data_type, repeat_regions, region_reads, read_class=None):
    """Reference nanoRepeat_bam.py:260-286 + :181-234 for many regions in ONE library call (nr_anchor_regions: two
    kernel launches however many regions): fills every region's read_dict with a Read per accepted read
    (dist_between_anchors, strand, core / mid positions, buffer lengths, left_anchor_paf / right_anchor_paf).
    region_reads: per region (names, sequences), {name: sequence} or None (the region's region_fq_file, which is what the
    reference hands minimap2, :279).  read_class: the Read class to instantiate (default: this package's)."""
    if len(repeat_regions) != len(region_reads):
        raise ValueError("one read set per region")
    get_preset_for_minimap2(data_type)
    sc = engine.get_preset(data_type)
    if read_class is None:
        from .repeat_region import Read as read_class
    named = [_reads_of(rr, reads) for rr, reads in zip(repeat_regions, region_reads)]
    res, _stats = engine.anchor_regions(sc, [rr.left_anchor_seq for rr in repeat_regions],
                                        [rr.right_anchor_seq for rr in repeat_regions], [list(seqs) for _names, seqs in named])
    col = {k: res[k].tolist() for k in ("read_len", "dist_between_anchors", "core_start", "core_end", "mid_start", "mid_end",
                                        "left_buffer", "right_buffer", "strand", "left_strand", "right_strand")}
    for side in ("left", "right"):
        for f in ("score", "tstart", "tend"):
            col[side + f] = res[side][f].tolist()
    accepted = np.flatnonzero(res["accepted"]).tolist()
    first = 0
    a = 0
    for rr, (names, _seqs) in zip(repeat_regions, named):
        end = first + len(names)
        rows = []
        while a < len(accepted) and accepted[a] < end:
            rows.append(accepted[a])
            a += 1
        add_accepted_reads(rr, [names[i - first] for i in rows], col, rows, read_class)
        first = end
    return


# The per-read Step-1 columns add_accepted_reads reads (strands as character codes), in the order
# sharding.anchor_regions_sharded sends them between ranks.
STEP1_FIELDS = ("read_len", "dist_between_anchors", "core_start", "core_end", "mid_start", "mid_end", "left_buffer",
                "right_buffer", "strand", "left_strand", "right_strand", "leftscore", "lefttstart", "lefttend",
                "rightscore", "righttstart", "righttend")


def add_accepted_reads(repeat_region, names, col, rows, read_class=None):
    """A Read per accepted read into repeat_region.read_dict, in the order given (:181-234): names[j] is the read whose
    Step-1 fields are row rows[j] of the columns `col` ({STEP1_FIELDS name: sequence}).  A name given twice keeps its
    first position in read_dict and the later read's fields, as the reference's dictionary does."""
    if read_class is None:
        from .repeat_region import Read as read_class
    for name, i in zip(names, rows):
        read = read_class()
        read.read_name = name
        read.full_read_len = col["read_len"][i]
        read.left_anchor_is_good = read.right_anchor_is_good = read.both_anchors_are_good = True
        read.left_anchor_paf = AnchorHit(chr(col["left_strand"][i]), col["leftscore"][i], col["lefttstart"][i], col["lefttend"][i])
        read.right_anchor_paf = AnchorHit(chr(col["right_strand"][i]), col["rightscore"][i], col["righttstart"][i],
                                          col["righttend"][i])
        read.dist_between_anchors = col["dist_between_anchors"][i]
        repeat_region.read_dict[name] = read
        repeat_region.buffer_len = BUFFER_LEN
        read.core_seq_start_pos, read.core_seq_end_pos = col["core_start"][i], col["core_end"][i]
        read.mid_seq_start_pos, read.mid_seq_end_pos = col["mid_start"][i], col["mid_end"][i]
        read.left_buffer_len, read.right_buffer_len = col["left_buffer"][i], col["right_buffer"][i]
        read.strand = chr(col["strand"][i])


def find_anchor_locations_in_reads(data_type, repeat_region, num_cpu=1, reads=None, read_class=None):
    """Reference nanoRepeat_bam.py:260-286 + :181-234 for one region (find_anchor_locations_in_regions).
    reads: (names, sequences) or {name: sequence}; default: repeat_region.region_fq_file."""
    find_anchor_locations_in_regions(data_type, [repeat_region], [reads], read_class)


def make_core_seq_fastq(repeat_region, reads=None, write_files=None):
    """Reference nanoRepeat_bam.py:288-331: the core (and middle) sequence of every accepted read, in the read's
    orientation, into repeat_region.read_core_seq_dict.  The two FASTQ files the reference also writes (the unmodified
    round1_and_round2_estimation reads core_sequences.fastq) are written when the region has a temp_out_dir, or on
    request; this package's own operators read the dictionary."""
    names, seqs = _reads_of(repeat_region, reads)
    if write_files is None:
        write_files = bool(getattr(repeat_region, "temp_out_dir", None))
    core_f = mid_f = None
    if write_files:
        repeat_region.core_seq_fq_file = os.path.join(repeat_region.temp_out_dir, "core_sequences.fastq")
        repeat_region.mid_seq_fq_file = os.path.join(repeat_region.temp_out_dir, "middle_sequences.fastq")
        repeat_region.temp_file_list += [repeat_region.core_seq_fq_file, repeat_region.mid_seq_fq_file]
        core_f, mid_f = open(repeat_region.core_seq_fq_file, "w"), open(repeat_region.mid_seq_fq_file, "w")
    for name, seq in zip(names, seqs):
        read = repeat_region.read_dict.get(name)
        if read is None:
            continue
        if read.strand == "-":
            seq = rev_comp(seq)                                             # :311-312
        core = seq[read.core_seq_start_pos:read.core_seq_end_pos]
        mid = seq[read.mid_seq_start_pos:read.mid_seq_end_pos]
        repeat_region.read_core_seq_dict[name] = core
        if core_f:
            core_f.write(f"@{name}\n{core}\n+\n{'0' * len(core)}\n")
            mid_f.write(f"@{name}\n{mid}\n+\n{'0' * len(mid)}\n")
    if core_f:
        core_f.close(); mid_f.close()
    return
