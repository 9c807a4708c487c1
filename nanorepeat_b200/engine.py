"""ctypes binding of libnanorepeat_b200.so (C ABI in include/nanorepeat_b200.h).

The library is built in-tree by __graft_entry__.build() / `make -C nanorepeat_b200/csrc`.  A missing library or
a missing GPU is an error -- there is no fallback path.
"""
import ctypes
import itertools
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libnanorepeat_b200.so")

NR_OK = 0
ERROR_NAMES = {-1: "NR_ERR_CUDA", -2: "NR_ERR_ARG", -3: "NR_ERR_BAD_BASE", -4: "NR_ERR_TOO_LARGE",
               -5: "NR_ERR_NOMEM", -6: "NR_ERR_UNKNOWN_TYPE"}


class Scoring(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in
                ("match", "mismatch", "gap_open1", "gap_ext1", "gap_open2", "gap_ext2", "ambiguous", "min_dp_score")]


class Stats(ctypes.Structure):
    _fields_ = [("algorithmic_cells", ctypes.c_int64), ("executed_cells", ctypes.c_int64),
                ("n_tasks", ctypes.c_int64), ("kernel_launches", ctypes.c_int32), ("n_skipped", ctypes.c_int32),
                ("h2d_bytes", ctypes.c_int64), ("d2h_bytes", ctypes.c_int64)]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_ if n != "reserved"}


class LaunchInfo(ctypes.Structure):
    _fields_ = [("paired_cells", ctypes.c_int64), ("rest_cells", ctypes.c_int64), ("n_pairs", ctypes.c_int32),
                ("n_rest", ctypes.c_int32), ("n_redo", ctypes.c_int32), ("reserved", ctypes.c_int32),
                ("paired_ms", ctypes.c_float), ("rest_ms", ctypes.c_float), ("redo_ms", ctypes.c_float),
                ("reserved2", ctypes.c_float), ("paired_useful_cells", ctypes.c_int64), ("rest_useful_cells", ctypes.c_int64),
                ("planned_paired_cells", ctypes.c_int64), ("planned_paired_useful_cells", ctypes.c_int64)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_ if not n.startswith("reserved")}


class RegionIn(ctypes.Structure):
    """nr_region_t: one region of nr_estimate_regions."""
    _fields_ = [("left", ctypes.c_char_p), ("n_left", ctypes.c_int32), ("right", ctypes.c_char_p), ("n_right", ctypes.c_int32),
                ("motif", ctypes.c_char_p), ("motif_len", ctypes.c_int32), ("n_reads", ctypes.c_int32),
                ("reads", ctypes.c_void_p), ("reads_len", ctypes.c_int64),
                ("dist_between_anchors", ctypes.POINTER(ctypes.c_int32)),
                ("has_round1_max_dist", ctypes.c_int32), ("round1_max_dist", ctypes.c_int64)]


ALN_DTYPE = np.dtype([("score", "<i4"), ("tstart", "<i4"), ("tend", "<i4")])
RUNG_DTYPE = np.dtype([("score", "<i4"), ("starts_in_left", "u1"), ("ends_in_right", "u1"), ("pad", "u1", (2,))])


class GmmParams(ctypes.Structure):
    """nr_gmm_params_t (include/nanorepeat_b200.h); defaults = the reference's (split_alleles.py:174, nanoRepeat.py:123,
    :159-160 with ploidy 2) and scikit-learn's."""
    _fields_ = [("max_components", ctypes.c_int32), ("n_init", ctypes.c_int32), ("max_iter", ctypes.c_int32),
                ("reserved", ctypes.c_int32), ("error_rate", ctypes.c_double), ("max_mutual_overlap", ctypes.c_double),
                ("tol", ctypes.c_double), ("reg_covar", ctypes.c_double), ("seed", ctypes.c_uint64)]

    def __init__(self, error_rate=0.03, max_mutual_overlap=0.15, max_components=22, seed=0, n_init=10, max_iter=100, tol=1e-3,
                 reg_covar=1e-6):
        super().__init__(max_components, n_init, max_iter, 0, error_rate, max_mutual_overlap, tol, reg_covar, seed)


GMM_MAX_COMPONENTS = 32


class NanoRepeatB200Error(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"{ERROR_NAMES.get(code, code)}: {message}")
        self.code = code


_lib = None

_cpp = ctypes.POINTER(ctypes.c_char_p)
_i32p = ctypes.POINTER(ctypes.c_int32)
_i64p = ctypes.POINTER(ctypes.c_int64)
_scp = ctypes.POINTER(Scoring)
_f64p = ctypes.POINTER(ctypes.c_double)
_gmp = ctypes.POINTER(GmmParams)

# name -> (restype, argtypes): every symbol include/nanorepeat_b200.h declares
SYMBOLS = {
    "nr_get_preset": (ctypes.c_int, [ctypes.c_char_p, _scp]),
    "nr_init": (ctypes.c_int, [ctypes.c_int]),
    "nr_shutdown": (ctypes.c_int, []),
    "nr_last_error": (ctypes.c_char_p, []),
    "nr_device_info": (ctypes.c_int, [_i32p, _i32p, _i32p]),
    "nr_limits": (ctypes.c_int, [_i32p, _i32p]),
    "nr_set_ladder_mode": (ctypes.c_int, [ctypes.c_int]),
    "nr_score_tasks": (ctypes.c_int, [_scp, ctypes.c_int32, _cpp, _i32p, _cpp, _i32p, ctypes.c_void_p]),
    "nr_round2_region": (ctypes.c_int, [_scp, ctypes.c_char_p, ctypes.c_int32, ctypes.c_char_p, ctypes.c_int32,
                                        ctypes.c_int32, ctypes.c_int32, _cpp, _i32p, ctypes.c_void_p]),
    "nr_round3_region": (ctypes.c_int, [_scp, ctypes.c_char_p, ctypes.c_int32, ctypes.c_char_p, ctypes.c_int32,
                                        ctypes.c_char_p, ctypes.c_int32, ctypes.c_int32, _cpp, _i32p, _i32p, _i32p,
                                        _i64p, ctypes.c_void_p, _i64p, _i32p, _i32p]),
    "nr_batch_create_tasks": (ctypes.c_void_p, [_scp, ctypes.c_int32, _cpp, _i32p, _cpp, _i32p]),
    "nr_batch_create_round2": (ctypes.c_void_p, [_scp, ctypes.c_char_p, ctypes.c_int32, ctypes.c_char_p,
                                                 ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, _cpp, _i32p]),
    "nr_batch_create_round3": (ctypes.c_void_p, [_scp, ctypes.c_char_p, ctypes.c_int32, ctypes.c_char_p,
                                                 ctypes.c_int32, ctypes.c_char_p, ctypes.c_int32, ctypes.c_int32,
                                                 _cpp, _i32p, _i32p, _i32p]),
    "nr_batch_begin": (ctypes.c_void_p, [_scp, ctypes.c_int32]),
    "nr_batch_add_round2": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_int32, ctypes.c_char_p,
                                           ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_char_p, _i64p]),
    "nr_batch_add_round2_lines": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_int32, ctypes.c_char_p,
                                                 ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p,
                                                 ctypes.c_int64]),
    "nr_batch_add_round3": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_int32, ctypes.c_char_p,
                                           ctypes.c_int32, ctypes.c_char_p, ctypes.c_int32, ctypes.c_int32,
                                           ctypes.c_char_p, _i64p, _i32p, _i32p]),
    "nr_batch_begin_round3_from": (ctypes.c_void_p, [ctypes.c_void_p]),
    "nr_batch_add_round3_reuse": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_char_p, ctypes.c_int32,
                                                 _i32p, _i32p]),
    "nr_batch_commit": (ctypes.c_int, [ctypes.c_void_p]),
    "nr_batch_run": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p]),
    "nr_batch_fetch_alns": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p]),
    "nr_batch_fetch_round2": (ctypes.c_int, [ctypes.c_void_p, _i32p, _i32p, ctypes.c_void_p]),
    "nr_batch_fetch_round3": (ctypes.c_int, [ctypes.c_void_p, _i64p, ctypes.c_void_p, _i64p, _i32p, _i32p]),
    "nr_batch_stats": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(Stats)]),
    "nr_set_timing": (ctypes.c_int, [ctypes.c_int]),
    "nr_batch_launch_info": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(LaunchInfo)]),
    "nr_batch_destroy": (None, [ctypes.c_void_p]),
    "nr_last_stats": (ctypes.c_int, [ctypes.POINTER(Stats)]),
    "nr_anchor_regions": (ctypes.c_int, [_scp, ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p, ctypes.POINTER(Stats)]),
    "nr_window_tasks": (ctypes.c_int, [_scp, ctypes.c_int32, _cpp, _i32p, _cpp, _i32p, _i32p, _i32p, ctypes.c_void_p, ctypes.c_void_p]),
    "nr_joint_grid": (ctypes.c_int, [_scp, ctypes.c_char_p, ctypes.c_int32, ctypes.c_char_p, ctypes.c_int32, ctypes.c_char_p,
                                     ctypes.c_int32, ctypes.c_char_p, ctypes.c_int32, ctypes.c_char_p, ctypes.c_int32,
                                     ctypes.c_int32, _cpp, _i32p, ctypes.c_int32, _i32p, _i32p, _i32p, ctypes.c_void_p,
                                     ctypes.c_void_p]),
    "nr_phase_1d": (ctypes.c_int, [_gmp, ctypes.c_int32, _i64p, _f64p, ctypes.c_int64, _i32p, _f64p, _f64p, _f64p, _i32p, _f64p]),
    "nr_gmm_bootstrap": (ctypes.c_int, [_gmp, ctypes.c_int32, _i64p, _f64p, ctypes.c_int64, _f64p]),
    "nr_gmm1d_fit": (ctypes.c_int, [_gmp, ctypes.c_int32, _i64p, _f64p, _i32p, _i64p, _f64p, _i32p, _f64p, _f64p, _f64p]),
    "nr_estimate_regions": (ctypes.c_int, [_scp, ctypes.c_int32, ctypes.c_int32, ctypes.POINTER(RegionIn),
                                           ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double), ctypes.c_void_p,
                                           ctypes.POINTER(ctypes.c_double), ctypes.c_void_p, _i32p, ctypes.POINTER(Stats)]),
}


def lib():
    """Load the shared library (no CUDA call happens at load time)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(nanorepeat_b200 has no CPU fallback)")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def _check(rc):
    if rc != NR_OK:
        raise NanoRepeatB200Error(rc, lib().nr_last_error().decode(errors="replace"))


def get_preset(data_type):
    sc = Scoring()
    rc = lib().nr_get_preset(data_type.encode(), ctypes.byref(sc))
    if rc != NR_OK:
        raise ValueError(lib().nr_last_error().decode())
    return sc


def init(device=-1):
    _check(lib().nr_init(int(device)))


def device_info():
    d, s, c = ctypes.c_int32(), ctypes.c_int32(), ctypes.c_int32()
    _check(lib().nr_device_info(ctypes.byref(d), ctypes.byref(s), ctypes.byref(c)))
    return dict(device=d.value, sm_count=s.value, clock_khz=c.value)


_ladder_mode = 3


def set_ladder_mode(mode):
    """3 (default): paired flag ladder (two reads per warp on u16x2 words); 2: flag ladder (score + span predicates per
    rung); 1: shared sweeps with exact (tstart, tend) per rung; 0: every rung is its own full rectangle.  Same scores,
    predicates and selection either way."""
    global _ladder_mode
    _check(lib().nr_set_ladder_mode(int(mode)))
    _ladder_mode = int(mode)


def ladder_mode():
    return _ladder_mode


def set_timing(on):
    """Bracket every kernel of Batch.run() with CUDA events (read back through Batch.launch_info())."""
    _check(lib().nr_set_timing(int(bool(on))))


def last_stats():
    st = Stats()
    _check(lib().nr_last_stats(ctypes.byref(st)))
    return st.as_dict()


def _cstrs(seqs):
    bs = [s.encode() if isinstance(s, str) else s for s in seqs]
    arr = (ctypes.c_char_p * len(bs))(*bs)
    lens = np.fromiter((len(b) for b in bs), dtype=np.int32, count=len(bs))
    return bs, arr, lens


def _concat(seqs):
    """list of str / bytes -> (one bytes buffer, int64 offsets[n + 1]): how reads cross the C ABI in bulk."""
    n = len(seqs)
    off = np.zeros(n + 1, dtype=np.int64)
    if n == 0:
        return b"", off
    if isinstance(seqs[0], str):
        buf = "".join(seqs).encode("ascii", "replace")     # a non-ASCII character becomes '?': an ambiguous base
    else:
        buf = b"".join(seqs)
    np.cumsum(np.fromiter(map(len, seqs), dtype=np.int64, count=n), out=off[1:])
    if off[-1] != len(buf):
        raise ValueError("mixed str / bytes reads")
    return buf, off


def _b(s):
    return s.encode() if isinstance(s, str) else s


# const char* PyUnicode_AsUTF8AndSize(PyObject*, Py_ssize_t*): for an ASCII str this is its own buffer, valid while
# the str is alive
_utf8 = ctypes.pythonapi.PyUnicode_AsUTF8AndSize
_utf8.restype = ctypes.c_void_p
_utf8.argtypes = [ctypes.py_object, ctypes.POINTER(ctypes.c_ssize_t)]


def score_tasks(queries, targets, sc):
    """Generic engine: (score, tstart, tend) for every (query, target) pair."""
    n = len(queries)
    if n != len(targets):
        raise ValueError("queries and targets differ in length")
    out = np.zeros(n, dtype=ALN_DTYPE)
    _qb, qa, ql = _cstrs(queries)
    _tb, ta, tl = _cstrs(targets)
    _check(lib().nr_score_tasks(ctypes.byref(sc), n, qa, ql.ctypes.data_as(_i32p), ta, tl.ctypes.data_as(_i32p),
                                out.ctypes.data))
    return out


def rung_offsets(kmin, kmax):
    n_rungs = np.maximum(kmax.astype(np.int64) - kmin.astype(np.int64) + 1, 0)
    off = np.zeros(len(kmin) + 1, dtype=np.int64)
    np.cumsum(n_rungs, out=off[1:])
    return off


NR_KIND_ROUND2, NR_KIND_ROUND3, NR_KIND_ROUND2_FLAGS = 1, 2, 3
_KINDS = {"round2": NR_KIND_ROUND2, "round3": NR_KIND_ROUND3, "round2_flags": NR_KIND_ROUND2_FLAGS}


class Batch:
    """Device-resident batch over one or more regions: reads are packed and uploaded by commit(), run() launches
    kernels only (asynchronously), fetch_*() synchronises and copies the records back."""

    def __init__(self, handle, kind):
        if not handle:
            raise NanoRepeatB200Error(-2, lib().nr_last_error().decode(errors="replace"))
        self._h = ctypes.c_void_p(handle)
        self.kind = kind
        self.n_items = 0          # reads (round 2 / 3) or tasks
        self._kmin, self._kmax = [], []
        self._region_reads = []   # round 2: reads per region, in add order

    # ---- construction -------------------------------------------------------------------------------------
    @classmethod
    def begin(cls, sc, kind):
        """kind: "round2" (exact (score, tstart, tend) records), "round2_flags" (score, tend and the span predicate
        tstart <= |left|: what nanoRepeat_bam.py:364-384 reads; paired u16x2 kernel) or "round3"."""
        return cls(lib().nr_batch_begin(ctypes.byref(sc), _KINDS[kind]), kind)

    @classmethod
    def begin_round3_from(cls, round2_batch):
        """Round-3 batch over the reads of a committed round-2 batch (they stay packed on the device)."""
        b = cls(lib().nr_batch_begin_round3_from(round2_batch._h), "round3")
        b._region_reads = list(round2_batch._region_reads)
        return b

    def add_round3_reuse(self, region_index, right, kmin, kmax):
        """kmin / kmax over ALL reads of that round-2 region, kmax < kmin skips a read."""
        kmin = np.ascontiguousarray(kmin, dtype=np.int32)
        kmax = np.ascontiguousarray(kmax, dtype=np.int32)
        n = self._region_reads[region_index]
        if len(kmin) != n or len(kmax) != n:
            raise ValueError("kmin / kmax must cover every read of the round-2 region")
        rb = _b(right)
        _check(lib().nr_batch_add_round3_reuse(self._h, int(region_index), rb, len(rb), kmin.ctypes.data_as(_i32p),
                                               kmax.ctypes.data_as(_i32p)))
        self.n_items += n
        self._kmin.append(kmin)
        self._kmax.append(kmax)
        return self

    def add_round2(self, left, motif, T, cores, lines=True):
        lb, mb = _b(left), _b(motif)
        if lines and cores and isinstance(cores[0], str):
            # one join, no per-read lengths, no encode: the joined str's own (ASCII == UTF-8) buffer crosses the ABI
            joined = "\n".join(cores)
            size = ctypes.c_ssize_t()
            ptr = _utf8(joined, ctypes.byref(size))
            if not ptr:
                raise ValueError("reads are not valid text")
            _check(lib().nr_batch_add_round2_lines(self._h, lb, len(lb), mb, len(mb), int(T), len(cores), ptr, size.value))
        else:
            buf, off = _concat(cores)
            _check(lib().nr_batch_add_round2(self._h, lb, len(lb), mb, len(mb), int(T), len(cores), buf,
                                             off.ctypes.data_as(_i64p)))
        self._region_reads.append(len(cores))
        self.n_items += len(cores)
        return self

    def add_round3(self, left, right, motif, cores, kmin, kmax):
        kmin = np.ascontiguousarray(kmin, dtype=np.int32)
        kmax = np.ascontiguousarray(kmax, dtype=np.int32)
        if len(kmin) != len(cores) or len(kmax) != len(cores):
            raise ValueError("kmin / kmax / cores differ in length")
        buf, off = _concat(cores)
        lb, rb, mb = _b(left), _b(right), _b(motif)
        _check(lib().nr_batch_add_round3(self._h, lb, len(lb), rb, len(rb), mb, len(mb), len(cores), buf,
                                         off.ctypes.data_as(_i64p), kmin.ctypes.data_as(_i32p),
                                         kmax.ctypes.data_as(_i32p)))
        self.n_items += len(cores)
        self._kmin.append(kmin)
        self._kmax.append(kmax)
        return self

    def commit(self):
        _check(lib().nr_batch_commit(self._h))
        return self

    @classmethod
    def tasks(cls, sc, queries, targets):
        _qb, qa, ql = _cstrs(queries)
        _tb, ta, tl = _cstrs(targets)
        b = cls(lib().nr_batch_create_tasks(ctypes.byref(sc), len(queries), qa, ql.ctypes.data_as(_i32p), ta,
                                            tl.ctypes.data_as(_i32p)), "tasks")
        b.n_items = len(queries)
        return b

    @classmethod
    def round2(cls, sc, left, motif, T, cores):
        return cls.begin(sc, "round2").add_round2(left, motif, T, cores).commit()

    @classmethod
    def round3(cls, sc, left, right, motif, cores, kmin, kmax):
        return cls.begin(sc, "round3").add_round3(left, right, motif, cores, kmin, kmax).commit()

    # ---- execution ----------------------------------------------------------------------------------------
    def run(self, stream=None):
        _check(lib().nr_batch_run(self._h, ctypes.c_void_p(stream) if stream else None))
        return self

    def fetch_alns(self):
        st = self.stats()
        out = np.zeros(st["n_tasks"], dtype=ALN_DTYPE)
        _check(lib().nr_batch_fetch_alns(self._h, out.ctypes.data))
        return out

    def fetch_round2(self):
        """-> (score, tend, starts_by_left) per read; starts_by_left = tstart <= |left| (nanoRepeat_bam.py:373)."""
        n = self.n_items
        score = np.zeros(n, dtype=np.int32)
        tend = np.zeros(n, dtype=np.int32)
        inside = np.zeros(n, dtype=np.uint8)
        _check(lib().nr_batch_fetch_round2(self._h, score.ctypes.data_as(_i32p), tend.ctypes.data_as(_i32p),
                                           inside.ctypes.data))
        return score, tend, inside.astype(bool)

    def fetch_round3(self, want_rungs=False):
        n = self.n_items
        kmin = np.concatenate(self._kmin) if self._kmin else np.zeros(0, np.int32)
        kmax = np.concatenate(self._kmax) if self._kmax else np.zeros(0, np.int32)
        sum_k = np.zeros(n, dtype=np.int64)
        n_k = np.zeros(n, dtype=np.int32)
        top = np.zeros(n, dtype=np.int32)
        off = rung_offsets(kmin, kmax) if want_rungs else None
        rungs = np.zeros(int(off[-1]), dtype=RUNG_DTYPE) if want_rungs else None
        _check(lib().nr_batch_fetch_round3(self._h, off.ctypes.data_as(_i64p) if want_rungs else None,
                                           rungs.ctypes.data if want_rungs else None,
                                           sum_k.ctypes.data_as(_i64p), n_k.ctypes.data_as(_i32p),
                                           top.ctypes.data_as(_i32p)))
        if want_rungs:
            return sum_k, n_k, top, rungs, off
        return sum_k, n_k, top

    def stats(self):
        st = Stats()
        _check(lib().nr_batch_stats(self._h, ctypes.byref(st)))
        return st.as_dict()

    def launch_info(self):
        """How the last run() split its work between the paired and the 32-bit kernels (+ event times, set_timing)."""
        li = LaunchInfo()
        _check(lib().nr_batch_launch_info(self._h, ctypes.byref(li)))
        return li.as_dict()

    def close(self):
        if self._h:
            lib().nr_batch_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def round2_regions(sc, regions):
    """regions: iterable of (left, motif, T, cores) -> one ALN_DTYPE array over all reads, in order."""
    with Batch.begin(sc, "round2") as b:
        for left, motif, T, cores in regions:
            b.add_round2(left, motif, T, cores)
        return b.commit().run().fetch_alns()


def round3_regions(sc, regions, want_rungs=False):
    """regions: iterable of (left, right, motif, cores, kmin, kmax) -> (sum_k, n_k, top_score[, rungs, rung_offset])
    over all reads, in order."""
    with Batch.begin(sc, "round3") as b:
        for left, right, motif, cores, kmin, kmax in regions:
            b.add_round3(left, right, motif, cores, kmin, kmax)
        return b.commit().run().fetch_round3(want_rungs)


def round2_region(sc, left, motif, T, cores):
    return round2_regions(sc, [(left, motif, T, cores)])


def round3_region(sc, left, right, motif, cores, kmin, kmax, want_rungs=False):
    """-> (sum_k, n_k, top_score[, rungs, rung_offset])."""
    return round3_regions(sc, [(left, right, motif, cores, kmin, kmax)], want_rungs)


# nr_region_t as a numpy record (same layout: natural alignment), so that a table of regions is filled column by column
REGION_DTYPE = np.dtype([("left", "<u8"), ("n_left", "<i4"), ("right", "<u8"), ("n_right", "<i4"), ("motif", "<u8"),
                         ("motif_len", "<i4"), ("n_reads", "<i4"), ("reads", "<u8"), ("reads_len", "<i8"),
                         ("dist_between_anchors", "<u8"), ("has_round1_max_dist", "<i4"), ("round1_max_dist", "<i8")],
                        align=True)
assert REGION_DTYPE.itemsize == ctypes.sizeof(RegionIn)


def _joined(strings):
    """list of str -> (one str, its buffer address, int64 start offsets[n + 1]); the str must outlive the pointer."""
    big = "".join(strings)
    size = ctypes.c_ssize_t()
    ptr = _utf8(big, ctypes.byref(size))
    off = np.zeros(len(strings) + 1, np.int64)
    np.cumsum(np.fromiter(map(len, strings), np.int64, len(strings)), out=off[1:])
    if not ptr or size.value != off[-1]:
        raise ValueError("sequences must be ASCII text")
    return big, ptr, off


def estimate_regions(sc, fast_mode, lefts, rights, motifs, cores, dists, max_dists=None, on_ready=None, n_reads=None):
    """nr_estimate_regions: rounds 1-3 of many regions in one call into the library.
    lefts / rights / motifs: one str per region; cores: one list of str per region (at least one read each) -- or, with
    n_reads given (reads per region), ONE flat list of all regions' reads in order; dists: all reads'
    dist_between_anchors, flat, in the same order; max_dists: per region None or the whole region's longest distance when
    the region is a piece of a split one.
    on_ready: called once the arguments are built, right before the library is entered (where ctypes drops the GIL) -- a
    caller that runs this on a worker thread uses it to know when its own Python work can go on without competing.
    -> dict of arrays over all reads in order: r1, r2, r2_valid, r3, r3_state (0 None / 1 mean of rungs / 2 = r2), plus T
    per region and the summed stats.  The table of regions is built column by column (no per-region ctypes work) and the
    reads travel as ONE buffer of lines (a single join)."""
    n = len(lefts)
    dists = np.ascontiguousarray(dists, dtype=np.int32)
    if n_reads is None:
        n_reads = np.fromiter(map(len, cores), np.int64, n)
        cores = list(itertools.chain.from_iterable(cores))
    else:
        n_reads = np.ascontiguousarray(n_reads, dtype=np.int64)
    total = int(n_reads.sum())
    if total != len(dists) or total != len(cores) or len(n_reads) != n:
        raise ValueError("cores and dist_between_anchors differ in length")
    if n and int(n_reads.min()) < 1:
        raise ValueError("every region needs at least one read")
    tab = np.zeros(max(n, 1), REGION_DTYPE)
    keep = []
    for name, seqs in (("left", lefts), ("right", rights), ("motif", motifs)):
        big, ptr, off = _joined(seqs)
        keep.append(big)
        tab[name][:n] = ptr + off[:-1]
        tab["n_" + name if name != "motif" else "motif_len"][:n] = off[1:] - off[:-1]
    big = "\n".join(cores)                               # every read a line; a region = n_reads consecutive lines
    size = ctypes.c_ssize_t()
    ptr = _utf8(big, ctypes.byref(size))
    keep.append(big)
    first = np.zeros(n + 1, np.int64)
    np.cumsum(n_reads, out=first[1:])
    if n == 1:
        llen = np.array([len(big)], np.int64)                                 # one region: all the lines are its lines
    else:
        clen = np.fromiter(map(len, cores), np.int64, total)
        csum = np.zeros(total + 1, np.int64)
        np.cumsum(clen, out=csum[1:])
        llen = csum[first[1:]] - csum[first[:-1]] + (n_reads - 1)             # a region's lines with the breaks between them
    start = np.zeros(n + 1, np.int64)
    np.cumsum(llen + 1, out=start[1:])
    if not ptr or (n and size.value != start[-1] - 1):
        raise ValueError("reads must be ASCII text")
    tab["reads"][:n] = ptr + start[:-1]
    tab["reads_len"][:n] = llen
    tab["n_reads"][:n] = n_reads
    tab["dist_between_anchors"][:n] = dists.ctypes.data + 4 * first[:-1]
    if max_dists is not None:
        has = np.fromiter((d is not None for d in max_dists), np.bool_, n)
        tab["has_round1_max_dist"][:n] = has
        tab["round1_max_dist"][:n] = np.fromiter((0 if d is None else d for d in max_dists), np.int64, n)
    r1 = np.zeros(total, np.float64); r2 = np.zeros(total, np.float64); r3 = np.zeros(total, np.float64)
    r2_valid = np.zeros(total, np.uint8); r3_state = np.zeros(total, np.uint8)
    T = np.zeros(max(n, 1), np.int32)
    st = Stats()
    dp = ctypes.POINTER(ctypes.c_double)
    if on_ready is not None:
        on_ready()
    _check(lib().nr_estimate_regions(ctypes.byref(sc), int(bool(fast_mode)), n, ctypes.cast(tab.ctypes.data, ctypes.POINTER(RegionIn)),
                                     r1.ctypes.data_as(dp), r2.ctypes.data_as(dp), r2_valid.ctypes.data, r3.ctypes.data_as(dp),
                                     r3_state.ctypes.data, T.ctypes.data_as(_i32p), ctypes.byref(st)))
    del keep
    return dict(r1=r1, r2=r2, r2_valid=r2_valid.astype(bool), r3=r3, r3_state=r3_state, T=T[:n], stats=st.as_dict())


# nr_anchor_region_t / nr_anchor_read_t as numpy records (same layout)
ANCHOR_REGION_DTYPE = np.dtype([("left", "<u8"), ("n_left", "<i4"), ("right", "<u8"), ("n_right", "<i4"), ("n_reads", "<i4"),
                                ("reads", "<u8"), ("reads_len", "<i8")], align=True)
ANCHOR_READ_DTYPE = np.dtype([("accepted", "u1"), ("left_good", "u1"), ("right_good", "u1"), ("strand", "u1"),
                              ("left_strand", "u1"), ("right_strand", "u1"), ("pad", "u1", (2,)), ("read_len", "<i4"),
                              ("dist_between_anchors", "<i4"), ("core_start", "<i4"), ("core_end", "<i4"), ("mid_start", "<i4"),
                              ("mid_end", "<i4"), ("left_buffer", "<i4"), ("right_buffer", "<i4"), ("left", ALN_DTYPE),
                              ("right", ALN_DTYPE)], align=True)
assert ANCHOR_REGION_DTYPE.itemsize == 48 and ANCHOR_READ_DTYPE.itemsize == 64


def anchor_regions(sc, lefts, rights, reads):
    """nr_anchor_regions: Step 1 (anchors, acceptance, core positions) of many regions in one call into the library.
    lefts / rights: one str per region; reads: per region a list of str (raw reads, any strand).
    -> (ANCHOR_READ_DTYPE array over all reads in region order, stats dict)."""
    n = len(lefts)
    if len(rights) != n or len(reads) != n:
        raise ValueError("one left anchor, right anchor and read list per region")
    n_reads = np.fromiter(map(len, reads), np.int64, n)
    flat = list(itertools.chain.from_iterable(reads))
    # a read that holds a newline (or any other character than ACGT) is not scored: it travels as one of N, never as
    # two lines
    flat = [r.replace("\n", "N") if "\n" in r else r for r in flat]
    tab = np.zeros(max(n, 1), ANCHOR_REGION_DTYPE)
    keep = []
    for name, seqs in (("left", lefts), ("right", rights)):
        big, ptr, off = _joined([s.encode("ascii", "replace").decode() for s in seqs])
        keep.append(big)
        tab[name][:n] = ptr + off[:-1]
        tab["n_" + name][:n] = off[1:] - off[:-1]
    big = "\n".join(flat).encode("ascii", "replace")          # a non-ASCII character becomes '?': the read is not scored
    keep.append(big)
    base = ctypes.cast(ctypes.c_char_p(big), ctypes.c_void_p).value or 0
    clen = np.fromiter(map(len, flat), np.int64, len(flat))
    csum = np.zeros(len(flat) + 1, np.int64)
    np.cumsum(clen + 1, out=csum[1:])                          # start of every line
    first = np.zeros(n + 1, np.int64)
    np.cumsum(n_reads, out=first[1:])
    tab["reads"][:n] = base + csum[first[:-1]]
    tab["reads_len"][:n] = np.maximum(csum[first[1:]] - csum[first[:-1]] - 1, 0)
    tab["n_reads"][:n] = n_reads
    out = np.zeros(max(len(flat), 1), ANCHOR_READ_DTYPE)
    st = Stats()
    _check(lib().nr_anchor_regions(ctypes.byref(sc), n, tab.ctypes.data, out.ctypes.data, ctypes.byref(st)))
    del keep
    return out[:len(flat)], st.as_dict()


WINDOW_DTYPE = np.dtype([("score", "<i4"), ("window_score", "<i4")])


def window_tasks(queries, targets, win_a, win_b, sc, reverse=None):
    """nr_window_tasks: (alignment score, window score of the optimal alignment inside [win_a, win_b)) per task."""
    n = len(queries)
    out = np.zeros(n, dtype=WINDOW_DTYPE)
    _qb, qa, ql = _cstrs(queries)
    _tb, ta, tl = _cstrs(targets)
    a = np.ascontiguousarray(win_a, dtype=np.int32)
    b = np.ascontiguousarray(win_b, dtype=np.int32)
    rv = None if reverse is None else np.ascontiguousarray(reverse, dtype=np.uint8)
    if len(targets) != n or len(a) != n or len(b) != n or (rv is not None and len(rv) != n):
        raise ValueError("task arrays differ in length")
    _check(lib().nr_window_tasks(ctypes.byref(sc), n, qa, ql.ctypes.data_as(_i32p), ta, tl.ctypes.data_as(_i32p),
                                 a.ctypes.data_as(_i32p), b.ctypes.data_as(_i32p), rv.ctypes.data if rv is not None else None,
                                 out.ctypes.data))
    return out


def joint_grid(sc, left, mid, right, motif1, motif2, reads, point_read, point_k1, point_k2):
    """nr_joint_grid: read point_read[i] against left + motif1*k1 + mid + motif2*k2 + right for (k1, k2) = point i.
    -> (records (score, window_score), strand (0 '+', 1 '-')), the better strand of every point."""
    _rb, ra, rl = _cstrs(reads)
    pr = np.ascontiguousarray(point_read, dtype=np.int32)
    k1 = np.ascontiguousarray(point_k1, dtype=np.int32)
    k2 = np.ascontiguousarray(point_k2, dtype=np.int32)
    n = len(pr)
    if len(k1) != n or len(k2) != n:
        raise ValueError("grid point arrays differ in length")
    out = np.zeros(n, dtype=WINDOW_DTYPE)
    strand = np.zeros(n, dtype=np.uint8)
    lb, mb, rb, m1b, m2b = _b(left), _b(mid), _b(right), _b(motif1), _b(motif2)
    _check(lib().nr_joint_grid(ctypes.byref(sc), lb, len(lb), mb, len(mb), rb, len(rb), m1b, len(m1b), m2b, len(m2b), len(reads), ra,
                               rl.ctypes.data_as(_i32p), n, pr.ctypes.data_as(_i32p), k1.ctypes.data_as(_i32p),
                               k2.ctypes.data_as(_i32p), out.ctypes.data, strand.ctypes.data))
    return out, strand


def _ragged(lists):
    """list of float sequences -> (offsets int64 [n + 1], values float64)"""
    off = np.zeros(len(lists) + 1, dtype=np.int64)
    if lists:
        np.cumsum([len(v) for v in lists], out=off[1:])
    flat = np.ascontiguousarray(np.concatenate([np.asarray(v, dtype=np.float64) for v in lists]) if off[-1] else np.zeros(0))
    return off, flat


def gmm_bootstrap(params, size_lists, region_id_base=0):
    """nr_gmm_bootstrap -> list of arrays (100 x len(sizes) samples per region)"""
    off, flat = _ragged(size_lists)
    out = np.zeros(100 * int(off[-1]), dtype=np.float64)
    _check(lib().nr_gmm_bootstrap(ctypes.byref(params), len(size_lists), off.ctypes.data_as(_i64p), flat.ctypes.data_as(_f64p),
                                  region_id_base, out.ctypes.data_as(_f64p)))
    return [out[100 * off[g]:100 * off[g + 1]] for g in range(len(size_lists))]


def gmm1d_fit(params, data_lists, n_components, region_ids=None):
    """nr_gmm1d_fit: best of params.n_init starts per problem -> dict(lower, iters, weights, means, variances), the last
    three as lists of arrays of n_components[i] entries."""
    off, flat = _ragged(data_lists)
    n = len(data_lists)
    nc = np.ascontiguousarray(n_components, dtype=np.int32)
    rid = None if region_ids is None else np.ascontiguousarray(region_ids, dtype=np.int64)
    C = params.max_components
    lower, iters = np.zeros(n), np.zeros(n, dtype=np.int32)
    w, m, v = np.zeros((n, C)), np.zeros((n, C)), np.zeros((n, C))
    _check(lib().nr_gmm1d_fit(ctypes.byref(params), n, off.ctypes.data_as(_i64p), flat.ctypes.data_as(_f64p), nc.ctypes.data_as(_i32p),
                              None if rid is None else rid.ctypes.data_as(_i64p), lower.ctypes.data_as(_f64p),
                              iters.ctypes.data_as(_i32p), w.ctypes.data_as(_f64p), m.ctypes.data_as(_f64p), v.ctypes.data_as(_f64p)))
    return dict(lower=lower, iters=iters, weights=[w[i, :nc[i]] for i in range(n)], means=[m[i, :nc[i]] for i in range(n)],
                variances=[v[i, :nc[i]] for i in range(n)])


def phase_1d(params, size_lists, region_id_base=0):
    """nr_phase_1d: every region's round-3 sizes -> per region dict(n, weights, means, variances, label, proba); label -1
    marks a size trimmed as an outlier (or a region with fewer than two sizes)."""
    off, flat = _ragged(size_lists)
    n = len(size_lists)
    C = params.max_components
    ncomp = np.zeros(n, dtype=np.int32)
    w, m, v = np.zeros((n, C)), np.zeros((n, C)), np.zeros((n, C))
    label = np.full(int(off[-1]), -1, dtype=np.int32)
    proba = np.zeros(int(off[-1]))
    _check(lib().nr_phase_1d(ctypes.byref(params), n, off.ctypes.data_as(_i64p), flat.ctypes.data_as(_f64p), region_id_base,
                             ncomp.ctypes.data_as(_i32p), w.ctypes.data_as(_f64p), m.ctypes.data_as(_f64p), v.ctypes.data_as(_f64p),
                             label.ctypes.data_as(_i32p), proba.ctypes.data_as(_f64p)))
    return [dict(n=int(ncomp[g]), weights=w[g, :ncomp[g]], means=m[g, :ncomp[g]], variances=v[g, :ncomp[g]],
                 label=label[off[g]:off[g + 1]], proba=proba[off[g]:off[g + 1]]) for g in range(n)]
