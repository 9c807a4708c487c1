"""Steps 1-4 of the reference's per-region pipeline for MANY regions, in memory.

The reference runs quantify1repeat_from_bam (nanoRepeat_bam.py:614-686) once per region inside forked workers, and
between its steps everything travels through files: the region's reads as FASTQ (:577-600), anchors.fasta and PAF text
(:260-286), core_sequences.fastq / middle_sequences.fastq (:288-331), round1_ref.fasta, one ladder FASTA and one read
FASTA per read (:349-355, :474-493), and the finished RepeatRegion objects -- with every read's round3_paf_text -- are
pickled through a multiprocessing queue (:602-612).  quantify_regions() does the same steps for a list of regions with the
reads handed over in memory: Step 1 (anchors, cores) and rounds 1-3 each as a few batched launches over ALL regions,
no temp files, no PAF text, nothing to pickle; with phase=True also Step 4 (:684, split_allele_using_gmm_1d), the
mixture fits of all regions in one call.  BAM / reference-FASTA IO, the motif check (:139-154) and the output files stay
with the caller, as in the reference.
"""
from . import anchoring, phasing
from .estimation import estimate_regions


def quantify_regions(repeat_regions, region_reads, data_type="ont", fast_mode=False, phase=False, ploidy=2,
                     max_mutual_overlap=0.15, max_num_components=-1, remove_noisy_reads=False, seed=0,
                     anchor_fn=None, estimate_fn=None, phase_fn=None):
    """repeat_regions: RepeatRegion-like objects with left_anchor_seq / right_anchor_seq / repeat_unit_seq set (what
    extract_ref_sequence leaves, :76-136); region_reads: per region (names, sequences) or {name: sequence} -- the reads
    extract_fastq_from_bam would have written for it (:577-600).
    Fills read_dict (accepted reads with dist_between_anchors, strand, core positions, round{1,2,3}_repeat_size) and
    read_core_seq_dict of every region, like Steps 1-3 of quantify1repeat_from_bam (:669-679).  Returns the regions.
    phase=True: also Step 4; every region gets `allele_list` (Allele objects sorted by gmm_mean1, or None when the
    reference would not phase it) and `num_removed_reads`.
    anchor_fn / estimate_fn / phase_fn stand in for anchoring.find_anchor_locations_in_regions, estimate_regions and
    phasing.phase_regions_1d (same arguments; default: those)."""
    if len(repeat_regions) != len(region_reads):
        raise ValueError("one read set per region")
    anchor_fn = anchor_fn or anchoring.find_anchor_locations_in_regions
    estimate_fn = estimate_fn or estimate_regions
    phase_fn = phase_fn or phasing.phase_regions_1d
    anchor_fn(data_type, repeat_regions, region_reads)                                  # Step 1 (:669-672), one call
    for rr, reads in zip(repeat_regions, region_reads):
        anchoring.make_core_seq_fastq(rr, reads=reads, write_files=False)
    estimate_fn(repeat_regions, data_type, fast_mode)                                   # Steps 2 and 3 (:675-679), batched
    if phase:                                                                          # Step 4 (:684), batched
        sizes = [{name: read.round3_repeat_size for name, read in rr.read_dict.items() if read.round3_repeat_size is not None}
                 for rr in repeat_regions]
        res = phase_fn(sizes, ploidy, phasing.error_rate_of(data_type), max_mutual_overlap, max_num_components,
                       remove_noisy_reads, seed)
        for rr, r in zip(repeat_regions, res):
            rr.allele_list, rr.num_removed_reads = (None, 0) if r is None else r
    return repeat_regions
