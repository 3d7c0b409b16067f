"""Deferred read validation (rcp_set_deferred_validation(1)), the mode bench.py measures in.

A deferred load returns before its map kernel is checked; the first call that uses the handle reads
the status words (reads_resolve, or the split path's own plan fetch, which also takes the give_up()
branch when the reads turn out too wide for the packed word).  Every load entry point is loaded
deferred and handed to every kind of first consumer; the result must equal the oracle
(oracle/recoup_oracle.py) bit for bit and what the same call gives after an eager load.

A deferred load of invalid reads succeeds; its first consumer raises the data error the eager load
raises, and so does every later consumer of the same handle (the handle never learnt its widths or
class counts, so anything else would be a wrong coverage returned as RCP_OK).  Under RCP_PATH_INDEX
the load is never deferred and raises itself.  Run the GPU tests with `-m gpu` on a B200."""
import contextlib
import ctypes as C
import os

import numpy as np
import pytest

from oracle import import_oracle as IO
from oracle import recoup_oracle as O
from tests.helpers import assert_coverage_equal, assert_matrix_close, synth_reads

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN_BAM = os.path.join(HERE, "golden", "WT_H4K20me1_5kr.bam")
CLEN = [60000, 25000, 8000]
SEED = 42
KINDS = ["dense", "device", "rle", "width", "width_runs", "select", "decoded", "decoded_select"]
CONSUMERS = ["cov_any", "cov_stranded", "cov_plus", "cov_minus_stranded", "list", "profile_fused",
             "profile_base", "profile_short"]


def _lib():
    from recoup_b200 import _lib as L
    return L


def vp(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def i64p(a):
    return a.ctypes.data_as(C.POINTER(C.c_int64))


def set_deferred(on):
    L = _lib()
    L.check(L.lib.rcp_set_deferred_validation(int(on)))


@pytest.fixture
def deferred(gpu):
    """gpu (every coverage path) with deferred validation on; always restored to off."""
    set_deferred(1)
    try:
        yield gpu
    finally:
        set_deferred(0)


@contextlib.contextmanager
def eager():
    set_deferred(0)
    try:
        yield
    finally:
        set_deferred(1)


def pool_used():
    """cudaMemPoolAttrUsedMemCurrent of device 0's default pool (driver API)."""
    cu = C.CDLL("libcuda.so.1")
    dev, pool, val = C.c_int(0), C.c_void_p(0), C.c_uint64(0)
    assert cu.cuDeviceGet(C.byref(dev), 0) == 0
    assert cu.cuDeviceGetDefaultMemPool(C.byref(pool), dev) == 0
    assert cu.cuMemPoolGetAttribute(pool, 7, C.byref(val)) == 0      # CU_MEMPOOL_ATTR_USED_MEM_CURRENT
    return val.value


# ---- one sample's reads, as every load entry point takes them ----------------------------------
class Sample:
    """Host arrays (kept alive until the handle is freed: a deferred load reads them late), the
    oracle's reads, and how to load them."""

    def __init__(self, kind, chrom, start, end, strand, clen, frag_len=0, width=None, select=None,
                 bam=None):
        self.kind = kind
        self.chrom = np.ascontiguousarray(chrom, dtype=np.int32)
        self.start = np.ascontiguousarray(start, dtype=np.int32)
        self.end = np.ascontiguousarray(end, dtype=np.int32)
        self.strand = None if strand is None else np.ascontiguousarray(strand, dtype=np.int8)
        self.clen = np.ascontiguousarray(clen, dtype=np.int64)
        self.frag_len = int(frag_len)
        self.width = width
        self.select = select            # (max_width, 1-based idx) for the select entry points
        self.bam = bam                  # bytes of a BAM file for the decoded entry points
        self._keep = []

    def oracle(self):
        c, s, e = self.chrom, self.start.astype(np.int64), self.end.astype(np.int64)
        st = np.zeros(c.shape[0], np.int64) if self.strand is None else self.strand.astype(np.int64)
        if self.select is not None:
            max_width, idx = self.select
            keep = np.flatnonzero(~((e - s + 1) > max_width))
            pick = keep[idx - 1]
            c, s, e, st = c[pick], s[pick], e[pick], st[pick]
        if self.frag_len:
            s, e = O.extend_fragments(s, e, st, self.frag_len, c, self.clen)
        return O.Reads(c, s, e, st, self.clen)

    def load(self):
        """The handle, or raises RecoupError."""
        L = _lib()
        lib = L.lib
        h = C.c_int(0)
        n, nc, cl = self.chrom.shape[0], self.clen.shape[0], i64p(self.clen)
        k = self.kind
        if k in ("dense", "device"):
            arrs = [self.chrom, self.start, self.end, self.strand]
            mem = L.MEM_HOST
            if k == "device":           # torch tensors, as bench.py passes them
                import torch
                dev = torch.device("cuda", 0)
                t = [None if a is None else torch.from_numpy(a).to(dev) for a in arrs]
                torch.cuda.synchronize()
                self._keep.append(t)
                p = [None if x is None else C.c_void_p(x.data_ptr()) for x in t]
                mem = L.MEM_DEVICE
            else:
                p = [vp(a) for a in arrs]
            rc = lib.rcp_reads_load(n, p[0], p[1], p[2], p[3], nc, cl, self.frag_len, mem, C.byref(h))
        elif k in ("rle", "width_runs"):
            from recoup_b200 import Rle
            r = Rle.encode(self.chrom)
            rv = np.ascontiguousarray(r.values, dtype=np.int32)
            rl = np.ascontiguousarray(r.lengths, dtype=np.int32)
            if getattr(self, "runs", None) is not None:      # explicit (possibly invalid) runs
                rv, rl = self.runs
            self._keep.append((rv, rl))
            if k == "rle":
                rc = lib.rcp_reads_load_rle(n, rv.shape[0], vp(rv), vp(rl), vp(self.start), vp(self.end),
                                            vp(self.strand), nc, cl, self.frag_len, L.MEM_HOST, C.byref(h))
            else:
                rc = lib.rcp_reads_load_width(n, None, rv.shape[0], vp(rv), vp(rl), vp(self.start),
                                              int(self.width), vp(self.strand), nc, cl, self.frag_len,
                                              L.MEM_HOST, C.byref(h))
        elif k == "width":
            rc = lib.rcp_reads_load_width(n, vp(self.chrom), 0, None, None, vp(self.start), int(self.width),
                                          vp(self.strand), nc, cl, self.frag_len, L.MEM_HOST, C.byref(h))
        elif k == "select":
            max_width, idx = self.select
            idx = np.ascontiguousarray(idx, dtype=np.int32)
            self._keep.append(idx)
            kept = C.c_int64(0)
            rc = lib.rcp_reads_load_select(n, vp(self.chrom), vp(self.start), vp(self.end), vp(self.strand),
                                           float(max_width), idx.shape[0], vp(idx), nc, cl, self.frag_len,
                                           L.MEM_HOST, C.byref(kept), C.byref(h))
        elif k in ("decoded", "decoded_select"):
            import recoup_b200 as rb
            gr = rb.readBam(self.bam)
            self._keep.append(gr)
            if k == "decoded":
                rc = lib.rcp_reads_load_decoded(gr.decoded_handle, nc, cl, self.frag_len, C.byref(h))
            else:
                max_width, idx = self.select
                idx = np.ascontiguousarray(idx, dtype=np.int32)
                self._keep.append(idx)
                kept = C.c_int64(0)
                rc = lib.rcp_reads_load_decoded_select(gr.decoded_handle, float(max_width), idx.shape[0], vp(idx),
                                                       nc, cl, self.frag_len, C.byref(kept), C.byref(h))
        else:
            raise ValueError(k)
        L.check(rc)
        return h.value


def _bam():
    data = open(GOLDEN_BAM, "rb").read()
    raw = IO.bgzf_inflate(data)
    _, lens, first = IO.bam_header(raw)
    c, s, e, st = IO.bam_decode(raw[first:], lens)
    return data, np.asarray(lens, np.int64), c, s, e, st


def make_sample(kind, seed=1):
    rng = np.random.default_rng(seed)
    if kind.startswith("decoded"):
        data, lens, c, s, e, st = _bam()
        sel = None
        if kind == "decoded_select":
            w = e.astype(np.int64) - s + 1
            max_width = float(np.quantile(w, 0.75))
            n_kept = int((~(w > max_width)).sum())
            sel = (max_width, np.sort(rng.choice(n_kept, size=n_kept * 2 // 3, replace=False) + 1))
        return Sample(kind, c, s, e, st, lens, select=sel, bam=data)
    if kind.startswith("width"):
        w = 50
        chrom, s, _, st = synth_reads(rng, 12000, CLEN, width=(w, w), sort=kind == "width_runs")
        return Sample(kind, chrom, s, s + w - 1, st, CLEN, width=w)
    chrom, s, e, st = synth_reads(rng, 15000, CLEN, width=(15, 400), sort=kind == "rle")
    sel = None
    if kind == "select":
        n_kept = int((~((e - s + 1) > 300)).sum())
        sel = (300.0, rng.integers(1, n_kept + 1, size=9000))        # with repeats, unsorted
    return Sample(kind, chrom, s, e, st, CLEN, select=sel)


# ---- masks -------------------------------------------------------------------------------------
def windows(rng, o_reads, n, lengths):
    """Windows around reads (and a few anywhere, some starting before position 1)."""
    nr = len(o_reads)
    clen = o_reads.chrom_len
    i = rng.integers(0, nr, size=n)
    chrom = o_reads.chrom[i].astype(np.int64)
    L = np.asarray(lengths, np.int64)[rng.integers(0, len(lengths), size=n)]
    start = o_reads.start[i] - rng.integers(0, L + 1)
    far = rng.random(n) < 0.15
    known = np.where(clen[chrom] > 0, clen[chrom], o_reads.end.max())
    start = np.where(far, (rng.random(n) * (known + 200)).astype(np.int64) - 100, start)
    strand = rng.choice(np.array([1, -1, 0]), size=n)
    return dict(chrom=chrom, start=start, end=start + L - 1, strand=strand)


def list_mask(rng, o_reads, n_el):
    """Exon-like elements: 1..5 ascending ranges on one chromosome, the first range's strand."""
    ptr, xc, xs, xe, xst = [0], [], [], [], []
    for _ in range(n_el):
        j = int(rng.integers(0, len(o_reads)))
        c, pos = int(o_reads.chrom[j]), int(o_reads.start[j]) - int(rng.integers(0, 800))
        gst = int(rng.choice([1, -1, 0]))
        for _ in range(int(rng.integers(1, 6))):
            w = int(rng.integers(10, 600))
            xc.append(c); xs.append(pos); xe.append(pos + w - 1); xst.append(gst)
            pos += w + int(rng.integers(0, 900))
        ptr.append(len(xs))
    if n_el > 3:
        ptr.insert(2, ptr[1])            # an empty element
    return dict(ptr=np.asarray(ptr, np.int64), chrom=np.asarray(xc, np.int64), start=np.asarray(xs, np.int64),
                end=np.asarray(xe, np.int64), strand=np.asarray(xst, np.int64))


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


# ---- consumers: the raw C calls, and the oracle's answer ----------------------------------------
CONSUMER_ARGS = {                   # ignore_strand, strand filter (None: any)
    "cov_any": (1, None), "cov_stranded": (0, None), "cov_plus": (1, 1), "cov_minus_stranded": (0, -1),
    "list": (0, None), "profile_fused": (1, None), "profile_base": (0, None), "profile_short": (1, -1),
}
PROFILE_SHAPE = {"profile_fused": (2000, 40), "profile_base": (300, 0), "profile_short": (40, 64)}


def make_mask(consumer, o_reads, seed=7):
    rng = np.random.default_rng(seed)
    if consumer == "list":
        return list_mask(rng, o_reads, 120)
    if consumer in PROFILE_SHAPE:
        return windows(rng, o_reads, 150, [PROFILE_SHAPE[consumer][0]])
    return windows(rng, o_reads, 250, [1, 37, 1024, 1025, 3000, 9000])


def consume(h, consumer, mask):
    """('cov', list of arrays / None) or ('mat', matrix, null flags); raises RecoupError."""
    from recoup_b200.coverage import CoverageList
    L = _lib()
    lib = L.lib
    ignore, filt = CONSUMER_ARGS[consumer]
    filt = L.STRAND_ANY if filt is None else filt
    c, s, e = _i32(mask["chrom"]), _i32(mask["start"]), _i32(mask["end"])
    st = np.ascontiguousarray(mask["strand"], dtype=np.int8)
    out = C.c_int(0)
    if consumer == "list":
        ptr = np.ascontiguousarray(mask["ptr"], dtype=np.int64)
        L.check(lib.rcp_coverage_list(h, ptr.shape[0] - 1, i64p(ptr), vp(c), vp(s), vp(e), vp(st), ignore, filt,
                                      L.MEM_HOST, C.byref(out)))
    elif consumer in PROFILE_SHAPE:
        Lw, n_bins = PROFILE_SHAPE[consumer]
        R = c.shape[0]
        ncols = n_bins if n_bins else Lw
        m = np.full((ncols, R), -7.0)            # column-major R x ncols, ld = R
        nul = np.full(R, 9, dtype=np.uint8)
        L.check(lib.rcp_coverage_profile(h, R, vp(c), vp(s), vp(e), vp(st), ignore, filt, n_bins, SEED, 0, 1.0,
                                         vp(m), R, vp(nul), L.MEM_HOST))
        return ("mat", m.T.copy(), nul.astype(bool))
    else:
        L.check(lib.rcp_coverage(h, c.shape[0], vp(c), vp(s), vp(e), vp(st), ignore, filt, L.MEM_HOST,
                                 C.byref(out)))
    cov = CoverageList(out.value)
    got = cov.to_list()
    cov.free()
    return ("cov", got)


def oracle_result(consumer, o_reads, mask):
    ignore, filt = CONSUMER_ARGS[consumer]
    want = O.calc_coverage(o_reads, mask, filt, bool(ignore))
    if consumer not in PROFILE_SHAPE:
        return ("cov", want)
    n_bins = PROFILE_SHAPE[consumer][1]
    bp = dict(flankBinSize=0, regionBinSize=n_bins, sumStat="mean", interpolation="auto")
    return ("mat", O.profile_matrix(want, (0, 0), bp, seed=SEED), np.asarray([w is None for w in want]))


def assert_same_result(got, want, exact):
    assert got[0] == want[0]
    if got[0] == "cov":
        assert_coverage_equal(got[1], want[1])
        return
    assert np.array_equal(got[2], want[2])
    if exact:
        assert np.array_equal(got[1], want[1])
    else:
        assert_matrix_close(got[1], want[1])


def check_against_oracle(got, want, consumer):
    # integer coverage and per-base rows are exact; bin means within the documented 1e-6
    assert_same_result(got, want, exact=consumer == "profile_base")


_ORACLE = {}


def _cached(kind, consumer):
    key = (kind, consumer)
    if key not in _ORACLE:
        smp = make_sample(kind)
        o_reads = smp.oracle()
        mask = make_mask(consumer, o_reads)
        follow = make_mask("cov_any", o_reads, seed=8)
        _ORACLE[key] = (mask, oracle_result(consumer, o_reads, mask), follow,
                        oracle_result("cov_any", o_reads, follow))
    return _ORACLE[key]


# ---- every load entry point x every kind of first consumer ------------------------------------
@pytest.mark.parametrize("consumer", CONSUMERS)
@pytest.mark.parametrize("kind", KINDS)
def test_deferred_load_then_first_consumer(deferred, kind, consumer):
    L = _lib()
    mask, want, follow, want_follow = _cached(kind, consumer)
    smp = make_sample(kind)
    h = smp.load()
    try:
        got = consume(h, consumer, mask)
        check_against_oracle(got, want, consumer)
        # the handle is usable afterwards: a GRanges call of another kind on it
        assert_same_result(consume(h, "cov_any", follow), want_follow, exact=True)
    finally:
        L.lib.rcp_reads_free(h)
    with eager():
        e_smp = make_sample(kind)
        he = e_smp.load()
        try:
            assert_same_result(consume(he, consumer, mask), got, exact=True)
        finally:
            L.lib.rcp_reads_free(he)


# ---- inputs that take the other branches of the load -------------------------------------------
def _run_both_modes(smp_fn, consumers, seed=3):
    """Deferred load -> each consumer in turn on ONE handle, against the oracle and against the
    same calls on an eager load."""
    L = _lib()
    smp = smp_fn()
    o_reads = smp.oracle()
    masks = [make_mask(c, o_reads, seed=seed + i) for i, c in enumerate(consumers)]
    h = smp.load()
    got = []
    try:
        for c, m in zip(consumers, masks):
            got.append(consume(h, c, m))
            check_against_oracle(got[-1], oracle_result(c, o_reads, m), c)
    finally:
        L.lib.rcp_reads_free(h)
    with eager():
        he = smp_fn().load()
        try:
            for c, m, g in zip(consumers, masks, got):
                assert_same_result(consume(he, c, m), g, exact=True)
        finally:
            L.lib.rcp_reads_free(he)


@pytest.mark.parametrize("kind", ["dense", "width", "width_runs"])
@pytest.mark.parametrize("first", ["cov_stranded", "list", "profile_fused"])
def test_fragment_extension_trimmed_at_chromosome_ends(deferred, kind, first):
    """frag_len > 0: one common width except the reads trim() shortens at either chromosome end
    (the uniform-width exception list)."""
    def smp_fn():
        rng = np.random.default_rng(5)
        w = 36
        chrom, s, _, st = synth_reads(rng, 8000, CLEN, width=(w, w), sort=kind == "width_runs")
        clen = np.asarray(CLEN)
        for j in range(0, 400, 2):               # '+' reads near the end, '-' reads near the start
            s[j] = clen[chrom[j]] - w + 1 - (j % 140)
            st[j] = 1 if j % 4 else 0
            s[j + 1] = 1 + (j % 150)
            st[j + 1] = -1
        return Sample(kind, chrom, s, s + w - 1, st, CLEN, frag_len=150, width=w)
    _run_both_modes(smp_fn, [first, "cov_any", "cov_plus"])


@pytest.mark.parametrize("kind", ["dense", "rle", "width"])
def test_unknown_seqlengths(deferred, kind):
    def smp_fn():
        smp = make_sample(kind, seed=9)
        smp.clen = np.asarray([-1, 25000, -1], dtype=np.int64)
        return smp
    _run_both_modes(smp_fn, ["cov_stranded", "list", "profile_base", "profile_fused"])


@pytest.mark.parametrize("first", ["cov_any", "cov_stranded", "list", "profile_fused"])
def test_strandless_reads(deferred, first):
    def smp_fn():
        smp = make_sample("dense", seed=4)
        smp.strand = None
        return smp
    _run_both_modes(smp_fn, [first, "cov_minus_stranded", "profile_short"])


def test_several_handles_pending_consumed_out_of_order(deferred):
    L = _lib()
    kinds = ["dense", "rle", "width", "select", "device"]
    smps = [make_sample(k, seed=20 + i) for i, k in enumerate(kinds)]
    hs = [s.load() for s in smps]                 # every map kernel queued, none checked yet
    order = [3, 0, 4, 2, 1]
    consumers = ["list", "cov_stranded", "profile_fused", "cov_any", "cov_plus"]
    try:
        for j, c in zip(order, consumers):
            o_reads = smps[j].oracle()
            m = make_mask(c, o_reads, seed=30 + j)
            check_against_oracle(consume(hs[j], c, m), oracle_result(c, o_reads, m), c)
    finally:
        for h in hs:
            L.lib.rcp_reads_free(h)


# ---- data errors of the reads ------------------------------------------------------------------
ERRORS = {                          # every one is RCP_ERR_DATA; the message index.cu gives
    "chrom_out_of_range": "a read has a chromosome id outside [0, n_chrom)",
    "start_below_1": "a read violates 1 <= start <= end",
    "start_after_end": "a read violates 1 <= start <= end",
    "start_past_chrom_end": "a read starts beyond the end of its chromosome",
    "negative_run": "a seqnames run has a negative length",
    "runs_short_of_n": "the seqnames run lengths sum to 1999, not to the 2000 reads",
}


def bad_sample(error):
    """The reads of `error` (None: the same reads, all valid)."""
    rng = np.random.default_rng(13)
    chrom, s, e, st = synth_reads(rng, 2000, CLEN, width=(20, 200), sort=True)
    kind = "rle" if error in ("negative_run", "runs_short_of_n", None) else "dense"
    smp = Sample(kind, chrom, s, e, st, CLEN)
    j = 777
    if error == "chrom_out_of_range":
        smp.chrom[j] = len(CLEN)
    elif error == "start_below_1":
        smp.start[j] = 0
    elif error == "start_after_end":
        smp.start[j] = smp.end[j] + 1
    elif error == "start_past_chrom_end":
        smp.start[j] = CLEN[smp.chrom[j]] + 3
        smp.end[j] = smp.start[j] + 10
    elif error is not None:
        from recoup_b200 import Rle
        r = Rle.encode(smp.chrom)
        rv = np.ascontiguousarray(r.values, dtype=np.int32)
        rl = np.ascontiguousarray(r.lengths, dtype=np.int32)
        if error == "negative_run":
            rl = np.concatenate([rl, [-1]]).astype(np.int32)
            rv = np.concatenate([rv, [0]]).astype(np.int32)
            rl[0] += 1
        else:
            rl[-1] -= 1
        smp.runs = (rv, rl)
    return smp


def _raises(fn):
    from recoup_b200 import RecoupError
    with pytest.raises(RecoupError) as ei:
        fn()
    return ei.value.code, str(ei.value)


ERROR_CONSUMERS = ["cov_stranded", "list", "profile_fused"]


@pytest.mark.parametrize("first", ERROR_CONSUMERS)
@pytest.mark.parametrize("error", sorted(ERRORS))
def test_a_failed_deferred_load_keeps_failing(deferred, request, error, first):
    L = _lib()
    lib = L.lib
    code, msg = L.RCP_ERR_DATA, ERRORS[error]
    # eager: the load raises
    with eager():
        got = _raises(bad_sample(error).load)
    assert got[0] == code and got[1].endswith(msg), got
    path = request.node.callspec.params["gpu"]
    if path == "index":
        # RCP_PATH_INDEX builds the sorted index inside the load: never deferred, the load raises
        assert _raises(bad_sample(error).load) == got
        return
    good = make_sample("dense", seed=17)
    o_good = good.oracle()
    masks = {c: make_mask(c, o_good, seed=40 + i) for i, c in enumerate(ERROR_CONSUMERS)}
    want_good = {c: oracle_result(c, o_good, m) for c, m in masks.items()}
    # warm-up on reads of the same shapes: blocks of 16 MiB and more return to the library's cache
    # (exact sizes), so the measured calls must meet the sizes the warm-up left there
    clean = bad_sample(None)
    warm = [clean, Sample("dense", clean.chrom, clean.start, clean.end, clean.strand, CLEN),
            make_sample("dense", seed=17)]
    for w in warm:
        hw = w.load()
        for c in ERROR_CONSUMERS:
            consume(hw, c, masks[c])
        lib.rcp_reads_free(hw)
    L.check(lib.rcp_sync())
    before = pool_used()
    bad = bad_sample(error)
    hb = bad.load()                                   # deferred: the load itself succeeds
    hg = good.load()                                  # a clean handle loaded in between
    order = [first] + [c for c in ERROR_CONSUMERS if c != first] + [first]
    for c in order:
        assert _raises(lambda: consume(hb, c, masks[c])) == got, c
    n, nchr = C.c_int64(0), C.c_int(0)
    L.check(lib.rcp_reads_info(hb, C.byref(n), C.byref(nchr), None))
    assert n.value == 2000 and nchr.value == len(CLEN)
    for c in ERROR_CONSUMERS:
        check_against_oracle(consume(hg, c, masks[c]), want_good[c], c)
    assert _raises(lambda: consume(hb, "cov_any", masks["cov_stranded"])) == got
    L.check(lib.rcp_reads_free(hb))
    L.check(lib.rcp_reads_free(hg))
    assert lib.rcp_reads_free(hb) == L.RCP_ERR_HANDLE
    L.check(lib.rcp_sync())
    assert pool_used() == before


def test_python_mirror_raises_on_every_call(deferred):
    """calcCoverage caches the device reads on the GRanges: a retry reuses the failed handle."""
    rb = deferred
    bad = rb.GRanges(np.zeros(3, np.int32), [5, 0, 40], [30, 9, 90], strand=np.array([1, -1, 0], np.int8),
                     seqlevels=["c0"], seqlengths=[100])
    mask = rb.GRanges(np.zeros(2, np.int32), [1, 20], [10, 60], seqlevels=["c0"])
    first = _raises(lambda: rb.calcCoverage(bad, mask))
    assert first[0] == _lib().RCP_ERR_DATA and "1 <= start <= end" in first[1]
    assert _raises(lambda: rb.calcCoverage(bad, mask)) == first
    assert _raises(lambda: rb.calcCoverage(bad, mask, ignore_strand=False)) == first
