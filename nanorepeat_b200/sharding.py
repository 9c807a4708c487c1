"""Sharding the hot path across the GPUs of one box (one process per GPU, torch.distributed for the plumbing).

The path is embarrassingly parallel (SURVEY.md section 8e): every (read, rung) task is independent and the only
dependencies are host-side scalars (round 2 -> ladder bounds per read, T per region).  So regions are dealt to ranks
by predicted DP cells -- the reference stripes regions over worker processes the same way, region i -> worker
i mod P (nanoRepeat_bam.py:604) -- each rank runs rounds 1-3 on its own GPU with no data-path collective, and the
per-read results (three numbers per read) are gathered on the host.  A region with very many reads (config 2: 5 000
reads in 2 regions) is first cut into contiguous read batches; T is a region-wide scalar, so it is computed before the
cut and pinned on every piece.

quantify_regions_sharded does the same for Steps 1-4 from raw reads (DESIGN.md section 5): pieces of raw reads dealt by
Step-1 cost, Step 1 and rounds 1-3 of a piece on one rank, T settled by one host exchange, the phasing in contiguous
blocks of regions; every rank ends with what one pipeline.quantify_regions call leaves.
"""
import copy
import time

import numpy as np

from . import anchoring


def predicted_cells(rr):
    """Executed-cell estimate for one region from what Step 1 hands over (no alignment needed):
    sum over reads of |core| * (round-2 template + backward |R| + forward |L| + m * k)."""
    m = max(1, len(rr.repeat_unit_seq))
    n_left, n_right = len(rr.left_anchor_seq), len(rr.right_anchor_seq)
    dists = [max(0, rd.dist_between_anchors) for rd in rr.read_dict.values()]
    if not dists:
        return 0
    r1max = max(dists) / m
    T = max(int(r1max * 1.5) + 1, int(r1max + 10))
    total = 0
    for name, rd in rr.read_dict.items():
        q = len(rr.read_core_seq_dict.get(name, ""))
        k = max(0, rd.dist_between_anchors) / m
        total += q * (n_left + m * T + n_right + n_left + int(m * (k + max(15, 0.05 * k))))
    return int(total)


def partition(costs, world_size):
    """Longest-processing-time greedy: item indices per rank, deterministic (ties by index), each rank's list
    in increasing index order."""
    order = sorted(range(len(costs)), key=lambda i: (-costs[i], i))
    load = [0] * world_size
    parts = [[] for _ in range(world_size)]
    for i in order:
        r = min(range(world_size), key=lambda w: (load[w], w))
        parts[r].append(i)
        load[r] += costs[i]
    return [sorted(p) for p in parts]


def split_region(rr, max_reads):
    """Cut one region into pieces of at most max_reads reads (contiguous in read_dict order).  Round 1's T depends
    on the region's maximum r1 (nanoRepeat_bam.py:344-347), so every piece carries the whole region's longest
    dist_between_anchors as `round1_max_dist` for the operator layer to honour."""
    names = list(rr.read_dict)
    if len(names) <= max_reads:
        return [rr]
    max_dist = max(rr.read_dict[n].dist_between_anchors for n in names)
    pieces = []
    for s in range(0, len(names), max_reads):
        p = copy.copy(rr)
        p.read_dict = {n: rr.read_dict[n] for n in names[s:s + max_reads]}
        p.read_core_seq_dict = {n: rr.read_core_seq_dict[n] for n in p.read_dict if n in rr.read_core_seq_dict}
        p.round1_max_dist = max_dist
        pieces.append(p)
    return pieces


def _world(rank, world_size):
    """(rank, world size) of the default process group where not given; (0, 1) without one."""
    import torch.distributed as dist
    up = dist.is_available() and dist.is_initialized()
    if world_size is None:
        world_size = dist.get_world_size() if up else 1
    if rank is None:
        rank = dist.get_rank() if up else 0
    return rank, world_size


def estimate_regions_sharded(regions, data_type=None, fast_mode=False, max_reads_per_piece=2048, estimate_fn=None,
                             rank=None, world_size=None, gather=True):
    """Rounds 1-3 over `regions` with the work split across the ranks of the default process group.

    Every rank passes the same `regions` list (same order).  Rank r computes the pieces dealt to it on its own GPU
    (estimate_fn defaults to nanorepeat_b200.estimate_regions), then -- gather=True -- the per-read results are
    exchanged on the host (all_gather_object of three float arrays per rank, no NCCL data path) and written into every rank's
    Read objects.  Returns the list of piece indices this rank computed."""
    import torch.distributed as dist
    if estimate_fn is None:
        from .estimation import estimate_regions as estimate_fn
    rank, world_size = _world(rank, world_size)
    pieces = []
    for rr in regions:
        for p in split_region(rr, max_reads_per_piece):
            if data_type is None and not hasattr(p, "data_type"):
                p.data_type = "ont"
            pieces.append(p)
    costs = [predicted_cells(p) for p in pieces]
    parts = partition(costs, world_size)
    mine = parts[rank]
    estimate_fn([pieces[i] for i in mine], data_type, fast_mode)
    if gather and world_size > 1:
        # host-side gather: every rank holds the same pieces in the same order, so three float arrays (NaN = None) and a
        # flag array per rank say everything -- no names, no per-read Python objects on the wire
        reads = [rd for i in mine for rd in pieces[i].read_dict.values()]
        nan = float("nan")
        r1 = np.fromiter((nan if r.round1_repeat_size is None else r.round1_repeat_size for r in reads), np.float64, len(reads))
        r2 = np.fromiter((nan if r.round2_repeat_size is None else r.round2_repeat_size for r in reads), np.float64, len(reads))
        r3 = np.fromiter((nan if r.round3_repeat_size is None else r.round3_repeat_size for r in reads), np.float64, len(reads))
        is_np = np.fromiter((isinstance(r.round3_repeat_size, np.floating) for r in reads), np.bool_, len(reads))
        gathered = [None] * world_size
        dist.all_gather_object(gathered, (mine, r1, r2, r3, is_np))
        for src, (theirs, g1, g2, g3, gnp) in enumerate(gathered):
            if src == rank:
                continue
            v1, v2, v3, fl = g1.tolist(), g2.tolist(), g3.tolist(), gnp.tolist()
            pos = 0
            for i in theirs:
                for read in pieces[i].read_dict.values():
                    a, b, c = v1[pos], v2[pos], v3[pos]
                    read.round1_repeat_size = None if a != a else a
                    read.round2_repeat_size = None if b != b else b
                    read.round3_repeat_size = None if c != c else (np.float64(c) if fl[pos] else c)
                    pos += 1
    return mine


# ---- Steps 1-4 sharded: Step 1 and rounds 1-3 of a piece on the rank that holds its reads ----

def cut_pieces(named, max_reads):
    """Step 1's pieces: every region's raw reads cut into contiguous ranges of at most max_reads reads, in input order,
    as (region index, start, end).  Step 1 has no region-wide value, so any cut is exact -- except in a region whose
    read names repeat: there the later read of a name wins at the first one's place in read_dict and the cores are cut
    with it (make_core_seq_fastq), which only the whole region reproduces, so such a region is one piece.
    named: per region (names, sequences)."""
    out = []
    for r, (names, _seqs) in enumerate(named):
        n = len(names)
        step = n if len(set(names)) < n else max_reads
        out.extend((r, s, min(s + step, n)) for s in range(0, n, step))
    return out


def _step1_sharded(repeat_regions, region_reads, data_type, max_reads, rank, world, anchor_fn, stats):
    """Cut, deal by Step-1 cells (2 (|left| + |right|) |read|, nr_stats_t.algorithmic_cells), and run Step 1 and the
    core cut of this rank's pieces: one anchor_fn call over all of them.  -> (named, spans, mine, pieces), pieces[j]
    being a copy of piece mine[j]'s region that holds only that piece's reads."""
    if len(repeat_regions) != len(region_reads):
        raise ValueError("one read set per region")
    t0 = time.perf_counter()
    named = [anchoring._reads_of(rr, reads) for rr, reads in zip(repeat_regions, region_reads)]
    spans = cut_pieces(named, max_reads)
    costs = [2 * (len(repeat_regions[r].left_anchor_seq) + len(repeat_regions[r].right_anchor_seq)) *
             sum(map(len, named[r][1][s:e])) for r, s, e in spans]
    mine = partition(costs, world)[rank]
    pieces, reads = [], []
    for i in mine:
        r, s, e = spans[i]
        p = copy.copy(repeat_regions[r])
        p.read_dict, p.read_core_seq_dict = {}, {}
        pieces.append(p)
        reads.append((named[r][0][s:e], named[r][1][s:e]))
    if pieces:
        anchor_fn(data_type, pieces, reads)
    for p, rd in zip(pieces, reads):
        anchoring.make_core_seq_fastq(p, reads=rd, write_files=False)
    if stats is not None:
        stats.update(step1_s=time.perf_counter() - t0, pieces=len(mine), step1_cells=sum(costs[i] for i in mine))
    return named, spans, mine, pieces


def _pin_region_max_dist(spans, mine, pieces, world):
    """Round 1's T is region-wide (nanoRepeat_bam.py:344-347): every piece of a region that was cut gets the whole
    region's longest dist_between_anchors as `round1_max_dist` (one all_gather_object of each piece's longest, None
    for a piece without an accepted read).  A region in one piece gets nothing: its call is the single-GPU call."""
    import torch.distributed as dist
    local = [max((rd.dist_between_anchors for rd in p.read_dict.values()), default=None) for p in pieces]
    gathered = [None] * world
    dist.all_gather_object(gathered, (mine, local))
    n_pieces, longest = {}, {}
    for r, _s, _e in spans:
        n_pieces[r] = n_pieces.get(r, 0) + 1
    for theirs, dists in gathered:
        for i, d in zip(theirs, dists):
            r = spans[i][0]
            if d is not None and (r not in longest or d > longest[r]):
                longest[r] = d
    for i, p in zip(mine, pieces):
        r = spans[i][0]
        if n_pieces[r] > 1 and r in longest:
            p.round1_max_dist = longest[r]


def _pack(spans, mine, pieces, named, with_rounds):
    """This rank's results as numpy arrays: per accepted read (in read_dict order, piece by piece) its index in the
    region's read list and its Step-1 fields (anchoring.STEP1_FIELDS, int64), with_rounds also round{1,2,3}_repeat_size
    (float64, NaN = None) and whether round 3 is an np.float64.  No sequence, no name, no per-read object."""
    idx, ints, counts = [], [], []
    for i, p in zip(mine, pieces):
        r, s, e = spans[i]
        first = {}
        for j, name in enumerate(named[r][0][s:e], s):
            first.setdefault(name, j)
        counts.append(len(p.read_dict))
        for name, rd in p.read_dict.items():
            la, ra = rd.left_anchor_paf, rd.right_anchor_paf
            idx.append(first[name])
            ints.append((rd.full_read_len, rd.dist_between_anchors, rd.core_seq_start_pos, rd.core_seq_end_pos,
                         rd.mid_seq_start_pos, rd.mid_seq_end_pos, rd.left_buffer_len, rd.right_buffer_len, ord(rd.strand),
                         ord(la.strand), ord(ra.strand), la.align_score, la.qstart, la.qend, ra.align_score, ra.qstart, ra.qend))
    out = dict(mine=list(mine), counts=np.array(counts, np.int64), idx=np.array(idx, np.int64),
               fields=np.array(ints, np.int64).reshape(len(ints), len(anchoring.STEP1_FIELDS)))
    if with_rounds:
        reads = [rd for p in pieces for rd in p.read_dict.values()]
        nan = float("nan")
        out["rounds"] = np.array([[nan if v is None else v for v in (rd.round1_repeat_size, rd.round2_repeat_size,
                                                                     rd.round3_repeat_size)] for rd in reads],
                                 np.float64).reshape(len(reads), 3)
        out["r3_is_np"] = np.array([isinstance(rd.round3_repeat_size, np.floating) for rd in reads], np.bool_)
    return out


def _unpack(repeat_regions, named, spans, gathered, with_rounds):
    """Every gathered read into its region's read_dict, regions and pieces in input order, through the helper Step 1
    itself uses (anchoring.add_accepted_reads); then every region's cores are cut from this rank's own reads as the
    single-GPU path cuts them (make_core_seq_fastq)."""
    where, parts = {}, []                     # piece -> (part, first row, rows)
    for k, g in enumerate(gathered):
        row = 0
        for i, c in zip(g["mine"], g["counts"].tolist()):
            where[i] = (k, row, c)
            row += c
    cols = [{f: g["fields"][:, j].tolist() for j, f in enumerate(anchoring.STEP1_FIELDS)} for g in gathered]
    idx = [g["idx"].tolist() for g in gathered]
    rounds = [(g["rounds"].tolist(), g["r3_is_np"].tolist()) for g in gathered] if with_rounds else None
    for i, (r, _s, _e) in enumerate(spans):
        if i not in where:
            continue
        k, row, c = where[i]
        rr, names = repeat_regions[r], named[r][0]
        rows = range(row, row + c)
        piece_names = [names[idx[k][j]] for j in rows]
        anchoring.add_accepted_reads(rr, piece_names, cols[k], rows)
        if with_rounds:
            vals, is_np = rounds[k]
            for name, j in zip(piece_names, rows):
                rd = rr.read_dict[name]
                a, b, c3 = vals[j]
                rd.round1_repeat_size = None if a != a else a
                rd.round2_repeat_size = None if b != b else b
                rd.round3_repeat_size = None if c3 != c3 else (np.float64(c3) if is_np[j] else c3)
    for rr, reads in zip(repeat_regions, named):
        anchoring.make_core_seq_fastq(rr, reads=reads, write_files=False)


def _gather_into(repeat_regions, named, spans, mine, pieces, world, gather, with_rounds, stats):
    import torch.distributed as dist
    t0 = time.perf_counter()
    local = _pack(spans, mine, pieces, named, with_rounds)
    gathered = [local]
    if gather and world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, local)
    _unpack(repeat_regions, named, spans, gathered, with_rounds)
    if stats is not None:
        stats["gather_s"] = time.perf_counter() - t0


def anchor_regions_sharded(repeat_regions, region_reads, data_type="ont", max_reads_per_piece=2048, rank=None,
                           world_size=None, gather=True, anchor_fn=None, stats=None):
    """Step 1 (anchors, cores) of many regions with the work split across the ranks of the default process group: what
    anchoring.find_anchor_locations_in_regions + make_core_seq_fastq leave, for the same regions and reads.

    Every rank passes the same regions (empty read_dict) and reads (the forms find_anchor_locations_in_regions takes),
    in the same order.  The regions' reads are cut into pieces (cut_pieces), dealt by LPT on Step-1 cells, and each
    rank runs Step 1 on its pieces in one anchor_fn call (default: find_anchor_locations_in_regions).  gather=True: the
    Step-1 fields of every accepted read are exchanged (all_gather_object of integer arrays) and every rank fills every
    region's read_dict in input order and cuts read_core_seq_dict from its own reads; gather=False: only this rank's
    pieces' reads.  stats: a dict to receive this rank's wall times and Step-1 cells.  Returns this rank's piece
    indices (into cut_pieces)."""
    anchor_fn = anchor_fn or anchoring.find_anchor_locations_in_regions
    rank, world = _world(rank, world_size)
    named, spans, mine, pieces = _step1_sharded(repeat_regions, region_reads, data_type, max_reads_per_piece, rank, world,
                                                anchor_fn, stats)
    _gather_into(repeat_regions, named, spans, mine, pieces, world, gather, False, stats)
    return mine


def _phase_blocks(counts, world):
    """[start, end) of world contiguous blocks of regions, balanced by the number of sizes to phase."""
    total, acc, bounds = sum(counts), 0, [0]
    for j, c in enumerate(counts):
        acc += c
        while len(bounds) < world and acc * world >= total * len(bounds):
            bounds.append(j + 1)
    bounds += [len(counts)] * (world + 1 - len(bounds))
    return list(zip(bounds[:-1], bounds[1:]))


def quantify_regions_sharded(repeat_regions, region_reads, data_type="ont", fast_mode=False, phase=False, ploidy=2,
                             max_mutual_overlap=0.15, max_num_components=-1, remove_noisy_reads=False, seed=0,
                             max_reads_per_piece=2048, rank=None, world_size=None, gather=True, anchor_fn=None,
                             estimate_fn=None, phase_fn=None, stats=None):
    """pipeline.quantify_regions (Steps 1-4 in memory) with the work split across the ranks of the default process
    group; the regions end as one quantify_regions call would leave them.

    Every rank passes the same regions and reads in the same order.  Step 1 as anchor_regions_sharded; then round 1's
    region-wide T is settled by one exchange of each piece's longest dist_between_anchors (pinned on the pieces of a
    region that was cut as `round1_max_dist`), and rounds 1-3 of a piece run on the rank that ran its Step 1, in one
    estimate_fn call: no core travels.  gather=True: the Step-1 fields and round{1,2,3}_repeat_size of every read
    are exchanged and every region is filled on every rank; gather=False: only this rank's pieces' reads.
    phase=True (needs gather=True): Step 4 on contiguous blocks of regions, one per rank, balanced by the number of sizes;
    a block is phased with region_id_base = its first region's index, so every region draws what the single call gives
    it (nr_phase_1d keys its generator by (seed, region id)); the results are exchanged and set on every region.
    anchor_fn / estimate_fn / phase_fn stand in for the three library-backed steps (as in pipeline.quantify_regions);
    stats: a dict to receive this rank's wall time per phase and its Step-1 and predicted round-1-3 cells.
    With one rank this is pipeline.quantify_regions.  Returns this rank's piece indices (into cut_pieces)."""
    from . import phasing, pipeline
    if phase and not gather:
        raise ValueError("phase=True needs gather=True")
    rank, world = _world(rank, world_size)
    if world == 1:
        if len(repeat_regions) != len(region_reads):
            raise ValueError("one read set per region")
        named = [anchoring._reads_of(rr, reads) for rr, reads in zip(repeat_regions, region_reads)]
        pipeline.quantify_regions(repeat_regions, named, data_type, fast_mode, phase, ploidy, max_mutual_overlap,
                                  max_num_components, remove_noisy_reads, seed, anchor_fn, estimate_fn, phase_fn)
        return list(range(len(cut_pieces(named, max_reads_per_piece))))
    import torch.distributed as dist
    anchor_fn = anchor_fn or anchoring.find_anchor_locations_in_regions
    if estimate_fn is None:
        from .estimation import estimate_regions as estimate_fn
    phase_fn = phase_fn or phasing.phase_regions_1d
    named, spans, mine, pieces = _step1_sharded(repeat_regions, region_reads, data_type, max_reads_per_piece, rank, world,
                                                anchor_fn, stats)
    t0 = time.perf_counter()
    _pin_region_max_dist(spans, mine, pieces, world)
    t1 = time.perf_counter()
    if pieces:
        estimate_fn(pieces, data_type, fast_mode)
    t2 = time.perf_counter()
    if stats is not None:
        stats.update(t_exchange_s=t1 - t0, rounds_s=t2 - t1, round_cells=sum(predicted_cells(p) for p in pieces))
    _gather_into(repeat_regions, named, spans, mine, pieces, world, gather, True, stats)
    if phase:
        t0 = time.perf_counter()
        sizes = [{name: read.round3_repeat_size for name, read in rr.read_dict.items() if read.round3_repeat_size is not None}
                 for rr in repeat_regions]
        a, b = _phase_blocks([len(s) for s in sizes], world)[rank]
        res = phase_fn(sizes[a:b], ploidy, phasing.error_rate_of(data_type), max_mutual_overlap, max_num_components,
                       remove_noisy_reads, seed, region_id_base=a) if b > a else []
        gathered = [None] * world
        dist.all_gather_object(gathered, res)
        for rr, r in zip(repeat_regions, (r for part in gathered for r in part)):
            rr.allele_list, rr.num_removed_reads = (None, 0) if r is None else r
        if stats is not None:
            stats["phase_s"] = time.perf_counter() - t0
    return mine
