"""Per-site modification frequency (``call_freq``) with the aggregation on the GPU.

Mirrors ``deepsignal_plant/call_mods_freq.py`` of the reference:

* ``calculate_mods_frequency(mods_files, prob_cf, contig_name=None)`` (``:29-74``)
* ``write_sitekey2stats(sitekey2stats, result_file, is_sort, is_bed, is_gzip)`` (``:77-122``)
* ``call_mods_frequency_to_file(args)`` (``:218-296``), including the ``--contigs`` per-contig mode
  (``:154-215,262-295``; same rows and order, one GPU pass instead of temp files + ``--nproc`` workers)

and ``utils/txt_formater.py`` (``ModRecord`` parsing rules, ``SiteStats`` attributes,
``split_key``).  The text is parsed into columns on the host, the segmented reduction --
callable filter, grouping by (chrom, pos), ordered float64 replay, integer counts, output
ordering -- runs in ``dsp_freq_aggregate`` (csrc/freq.cu), and the bytes written are
identical to the reference's.  Under ``torchrun`` (one process per GPU) ``call_mods_frequency_to_file`` hands
over to ``freq_dist.call_freq_distributed``: ranks parse contiguous byte shards, records are routed by site key
over NVLink peer memory (csrc/comm.cu) with no partial-sum merging, because float64 addition is order
sensitive, and every rank writes its own slice of the table.
"""
from __future__ import annotations

import ctypes as C
import gzip
import io
import os
import time

import numpy as np

from . import _native

key_sep = "||"
POS_BITS = 40


def split_key(key):
    """``utils/txt_formater.py:29-31``."""
    words = key.split(key_sep)
    return words[0], int(words[1])


class SiteStats:
    """``utils/txt_formater.py:34-46`` (attribute names kept)."""
    __slots__ = ("_strand", "_pos_in_strand", "_kmer", "_prob_0", "_prob_1", "_met", "_unmet", "_coverage")

    def __init__(self, strand, pos_in_strand, kmer):
        self._strand = strand
        self._pos_in_strand = pos_in_strand
        self._kmer = kmer
        self._prob_0 = 0.0
        self._prob_1 = 0.0
        self._met = 0
        self._unmet = 0
        self._coverage = 0


class Records:
    """Column form of call_mods lines (``utils/txt_formater.py:8-21``), file order.

    ``chrom`` / ``strand`` / ``kmer`` read as object arrays of ``str`` like the reference's fields.  Records
    that come from the native parser keep them compact instead -- chromosome codes + a name table, fixed-width
    byte cells -- and only turn the rows somebody asks for into Python strings (``meta_at``)."""
    FIELDS = ("chrom", "pos", "strand", "pos_in_strand", "p0", "p1", "label", "kmer")

    def __init__(self, chrom, pos, strand, pos_in_strand, p0, p1, label, kmer, chrom_codes=None):
        self._chrom = None if chrom is None else np.asarray(chrom, dtype=object)
        self._codes = chrom_codes                       # (int32 codes, list of names) or None
        self.pos = np.asarray(pos, dtype=np.int64)
        self._strand = strand if _is_cells(strand) else np.asarray(strand, dtype=object)
        self.pos_in_strand = np.asarray(pos_in_strand, dtype=np.int64)
        self.p0 = np.asarray(p0, dtype=np.float64)
        self.p1 = np.asarray(p1, dtype=np.float64)
        self.label = np.asarray(label, dtype=np.int32)
        self._kmer = kmer if _is_cells(kmer) else np.asarray(kmer, dtype=object)

    def __len__(self):
        return int(self.pos.shape[0])

    @property
    def chrom(self):
        if self._chrom is None:
            codes, names = self._codes
            self._chrom = np.asarray(names, dtype=object)[codes] if len(names) else np.empty(0, object)
        return self._chrom

    @property
    def strand(self):
        return _cells_to_str(self._strand)

    @property
    def kmer(self):
        return _cells_to_str(self._kmer)

    def meta_at(self, idx):
        """(strand, pos_in_strand, kmer) of the given records only, strings as object arrays."""
        return _cells_to_str(self._strand[idx]), self.pos_in_strand[idx], _cells_to_str(self._kmer[idx])

    def chrom_codes(self):
        """(int32 codes, list of names): the chromosome column as codes into a name table (any order)."""
        if self._codes is not None:
            return self._codes
        names, index = [], {}
        codes = np.fromiter((index.setdefault(c, len(index)) for c in self.chrom.tolist()), dtype=np.int32, count=len(self))
        return codes, list(index)

    def meta_cells(self, idx):
        """(strand, pos_in_strand, kmer) of the given records as fixed-width byte cells (S8 / int64 / S24) -- the form
        in which site rows carry their text columns between ranks."""
        def cells(a, width):
            a = a[idx]
            if _is_cells(a):
                return a.astype("S%d" % width)
            b = np.asarray([x.encode() for x in a.tolist()], dtype=object)
            if len(b) and max(len(x) for x in b) > width:
                raise ValueError("a strand / k-mer column wider than %d bytes cannot travel between ranks; "
                                 "run call_freq in one process for this input" % width)
            return b.astype("S%d" % width) if len(b) else np.empty(0, "S%d" % width)
        return cells(self._strand, 8), self.pos_in_strand[idx], cells(self._kmer, 24)

    def chrom_ranks(self):
        """(ids, names): chromosome ids by rank in Python string order, so that integer key order equals the
        reference's ``(chrom, pos)`` tuple order (``call_mods_freq.py:88``)."""
        if self._codes is None:
            return _chrom_ids(self.chrom)
        codes, names = self._codes
        order = sorted(range(len(names)), key=lambda i: names[i])
        rank = np.empty(len(names), np.int64)
        rank[order] = np.arange(len(names))
        return rank[codes], [names[i] for i in order]

    def chrom_in(self, wanted):
        """Boolean mask of the records whose chromosome is in the set ``wanted``."""
        if self._codes is None:
            return np.fromiter((c in wanted for c in self.chrom.tolist()), dtype=bool, count=len(self))
        codes, names = self._codes
        return np.array([nm in wanted for nm in names], bool)[codes] if len(names) else np.zeros(0, bool)

    def select(self, keep):
        codes = None if self._codes is None else (self._codes[0][keep], self._codes[1])
        return Records(None if codes is not None else self.chrom[keep], self.pos[keep], self._strand[keep],
                       self.pos_in_strand[keep], self.p0[keep], self.p1[keep], self.label[keep], self._kmer[keep], codes)

    @staticmethod
    def concat(parts):
        parts = [p for p in parts if len(p)]
        if not parts:
            return Records([], [], [], [], [], [], [], [])
        if len(parts) == 1:
            return parts[0]
        cat = lambda f: np.concatenate([getattr(p, f) for p in parts])
        compact = all(p._codes is not None and _is_cells(p._strand) and _is_cells(p._kmer) for p in parts)
        if not compact:
            return Records(cat("chrom"), cat("pos"), cat("strand"), cat("pos_in_strand"), cat("p0"), cat("p1"), cat("label"),
                           cat("kmer"))
        names, index, codes = [], {}, []
        for p in parts:                                  # one name table for all parts
            remap = np.array([index.setdefault(nm, len(index)) for nm in p._codes[1]], np.int32)
            names = list(index)
            codes.append(remap[p._codes[0]])
        return Records(None, cat("pos"), cat("_strand"), cat("pos_in_strand"), cat("p0"), cat("p1"), cat("label"), cat("_kmer"),
                       (np.concatenate(codes), names))


def _is_cells(a):
    return isinstance(a, np.ndarray) and a.dtype.kind == "S"


def _cells_to_str(a):
    return a.astype(str).astype(object) if _is_cells(a) else a


def parse_lines(lines):
    """Parse call_mods text lines (an iterable of str) into ``Records``.  Field rules of
    ``ModRecord.__init__``: ``line.strip().split('\\t')``; pos / pos_in_strand / label via
    ``int``; probabilities via ``float`` (correctly rounded decimal -> float64)."""
    chrom, pos, strand, pis, p0, p1, label, kmer = [], [], [], [], [], [], [], []
    for line in lines:
        w = line.strip().split("\t")
        chrom.append(w[0]); pos.append(int(w[1])); strand.append(w[2]); pis.append(int(w[3]))
        p0.append(float(w[6])); p1.append(float(w[7])); label.append(int(w[8])); kmer.append(w[9])
    return Records(chrom, pos, strand, pis, p0, p1, label, kmer)


def _shard_view(buf, byte_range):
    """The lines of ``buf`` whose first byte lies in [lo, hi): a line belongs to the shard it starts in."""
    lo, hi = byte_range
    n = buf.size

    def line_start_at_or_after(p):
        if p <= 0:
            return 0
        if p >= n:
            return n
        if buf[p - 1] == 10:
            return p
        blk = 1 << 16
        q = p
        while q < n:
            hit = np.flatnonzero(buf[q:q + blk] == 10)
            if hit.size:
                return q + int(hit[0]) + 1
            q += blk
        return n
    return buf[line_start_at_or_after(lo):line_start_at_or_after(hi)]


def _read_mods_file_native(path, nthreads=None, byte_range=None):
    """``dsp_parse_calls`` over the whole file (mapped in place, or decompressed) or over the lines that start inside
    ``byte_range``: compact ``Records``, or None when a strand / k-mer column is wider than the parser's fixed cells."""
    import mmap
    L = _native.lib()
    nthreads = int(nthreads or min(32, os.cpu_count() or 1))
    if path.endswith(".gz"):
        if byte_range is not None:
            raise ValueError("byte_range needs an uncompressed call_mods file")
        with gzip.open(path, "rb") as f:
            buf = np.frombuffer(f.read(), np.uint8)
        mm = None
    else:
        with open(path, "rb") as f:
            mm = mmap.mmap(f.fileno(), 0, access=mmap.ACCESS_READ)
        buf = np.frombuffer(mm, np.uint8)
    whole = buf
    if byte_range is not None:
        buf = _shard_view(buf, byte_range)
    try:
        return parse_calls_buffer(buf, nthreads, what=path)
    finally:
        del buf, whole
        if mm is not None:
            try:
                mm.close()
            except BufferError:
                pass


def parse_calls_buffer(buf, nthreads=None, what="<memory>"):
    """``dsp_parse_calls`` over call_mods lines held in memory (a uint8 array or bytes): compact ``Records``, or None
    when a strand / k-mer column is wider than the parser's fixed cells."""
    L = _native.lib()
    nthreads = int(nthreads or min(32, os.cpu_count() or 1))
    if not isinstance(buf, np.ndarray):
        buf = np.frombuffer(buf, np.uint8)
    if buf.size == 0:
        return Records([], [], [], [], [], [], [], [])
    n = C.c_int64(0)
    nb, nn = C.c_int64(0), C.c_int32(0)
    # first a counting pass (max_records = 0: newline scan only), then exactly sized columns: no oversized buffers, no copies
    _native.check(L.dsp_parse_calls(buf.ctypes.data, buf.size, 0, None, None, None, None, None, None, None, None, None, 0,
                                    C.byref(nb), C.byref(nn), C.byref(n), nthreads), "dsp_parse_calls(%s)" % what)
    cap = max(int(n.value), 1)
    code, pos, pis = np.empty(cap, np.int32), np.empty(cap, np.int64), np.empty(cap, np.int64)
    p0, p1, label = np.empty(cap, np.float64), np.empty(cap, np.float64), np.empty(cap, np.int32)
    strand, kmer = np.empty(cap, "S4"), np.empty(cap, "S24")
    names = np.empty(1 << 16, np.uint8)
    p = lambda a: a.ctypes.data
    while True:
        rc = L.dsp_parse_calls(buf.ctypes.data, buf.size, cap, p(code), p(pos), p(strand), p(pis), p(p0), p(p1), p(label),
                               p(kmer), p(names), names.size, C.byref(nb), C.byref(nn), C.byref(n), nthreads)
        if rc == 5:                                  # DSP_ERR_UNSUPPORTED: unusually wide strand / k-mer column
            return None
        if rc == 4 and nb.value > names.size:        # DSP_ERR_NOMEM: many long chromosome names
            names = np.empty(int(nb.value), np.uint8)
            continue
        _native.check(rc, "dsp_parse_calls(%s)" % what)
        break
    m = int(n.value)
    if m == 0:
        return Records([], [], [], [], [], [], [], [])
    table = names[:int(nb.value)].tobytes().decode().split("\n")[:int(nn.value)]
    return Records(None, pos[:m], strand[:m], pis[:m], p0[:m], p1[:m], label[:m], kmer[:m], (code[:m], table))


def read_mods_file(path, byte_range=None):
    """One call_mods file (plain or .gz, ``call_mods_freq.py:45-48``) -> ``Records``; ``byte_range=(lo, hi)`` keeps
    only the lines that start inside it (one rank's shard of an uncompressed file)."""
    if os.path.getsize(path) == 0:
        return Records([], [], [], [], [], [], [], [])
    rec = _read_mods_file_native(path, byte_range=byte_range)
    if rec is not None:
        return rec
    if byte_range is not None:
        with open(path, "rb") as f:
            data = np.frombuffer(f.read(), np.uint8)
        return parse_lines(_shard_view(data, byte_range).tobytes().decode().splitlines())
    import pandas as pd
    try:
        df = pd.read_csv(path, sep="\t", header=None, usecols=[0, 1, 2, 3, 6, 7, 8, 9],
                         names=list(range(10)), dtype={0: str, 2: str, 9: str, 1: np.int64, 3: np.int64,
                                                       6: np.float64, 7: np.float64, 8: np.int64},
                         float_precision="round_trip", na_filter=False, quoting=3,
                         compression="gzip" if path.endswith(".gz") else None, engine="c")
        return Records(df[0].str.strip().to_numpy(object), df[1].to_numpy(), df[2].to_numpy(object), df[3].to_numpy(),
                       df[6].to_numpy(), df[7].to_numpy(), df[8].to_numpy().astype(np.int32),
                       df[9].str.strip().to_numpy(object))
    except Exception:
        opener = gzip.open if path.endswith(".gz") else open
        with opener(path, "rt") as f:
            return parse_lines(f)


class FreqTable:
    """Result of the aggregation in column form, one row per site, in output order.
    Behaves like the reference's ``sitekey2stats`` dict (``"chrom||pos" -> SiteStats``) for
    callers that index it, without materialising one Python object per site."""

    def __init__(self, chrom, pos, strand, pos_in_strand, kmer, prob_0, prob_1, met, unmet, coverage,
                 first_index, n_records=0, n_used=0):
        self.chrom, self.pos, self.strand, self.pos_in_strand, self.kmer = chrom, pos, strand, pos_in_strand, kmer
        self.prob_0, self.prob_1, self.met, self.unmet, self.coverage = prob_0, prob_1, met, unmet, coverage
        self.first_index = first_index
        self.n_records, self.n_used = n_records, n_used
        self._index = None

    def __len__(self):
        return int(self.pos.shape[0])

    def keys(self):
        return [key_sep.join([c, str(p)]) for c, p in zip(self.chrom.tolist(), self.pos.tolist())]

    def __iter__(self):
        return iter(self.keys())

    def _row(self, i):
        s = SiteStats(self.strand[i], int(self.pos_in_strand[i]), self.kmer[i])
        s._prob_0, s._prob_1 = float(self.prob_0[i]), float(self.prob_1[i])
        s._met, s._unmet, s._coverage = int(self.met[i]), int(self.unmet[i]), int(self.coverage[i])
        return s

    def __getitem__(self, key):
        if self._index is None:
            self._index = {k: i for i, k in enumerate(self.keys())}
        return self._row(self._index[key])

    def items(self):
        return ((k, self._row(i)) for i, k in enumerate(self.keys()))

    def reorder(self, order):
        f = lambda a: a[order]
        return FreqTable(f(self.chrom), f(self.pos), f(self.strand), f(self.pos_in_strand), f(self.kmer),
                         f(self.prob_0), f(self.prob_1), f(self.met), f(self.unmet), f(self.coverage),
                         f(self.first_index), self.n_records, self.n_used)

    @staticmethod
    def concat(tables):
        tables = [t for t in tables if len(t)]
        if not tables:
            e = np.empty(0)
            return FreqTable(np.empty(0, object), e.astype(np.int64), np.empty(0, object), e.astype(np.int64), np.empty(0, object),
                             e, e, e.astype(np.int32), e.astype(np.int32), e.astype(np.int32), e.astype(np.int64))
        cat = lambda f: np.concatenate([getattr(t, f) for t in tables])
        return FreqTable(cat("chrom"), cat("pos"), cat("strand"), cat("pos_in_strand"), cat("kmer"), cat("prob_0"), cat("prob_1"),
                         cat("met"), cat("unmet"), cat("coverage"), cat("first_index"),
                         sum(t.n_records for t in tables), sum(t.n_used for t in tables))

    def sorted(self):
        """``sorted(keys, key=split_key)`` (``call_mods_freq.py:88``): (chrom str, pos int)."""
        uniq, inv = np.unique(self.chrom.astype(str), return_inverse=True)   # code-point order, like Python str
        return self.reorder(np.lexsort((self.pos, inv)))


def _chrom_ids(chrom):
    """Chromosome ids by rank in Python string order, so that integer key order equals the
    reference's ``(chrom, pos)`` tuple order."""
    names = sorted(set(chrom.tolist()))
    rank = {c: i for i, c in enumerate(names)}
    ids = np.fromiter((rank[c] for c in chrom.tolist()), dtype=np.int64, count=len(chrom))
    return ids, names


def make_keys(chrom_ids, pos):
    if len(pos) and (pos.min() < 0 or pos.max() >= (1 << POS_BITS)):
        raise ValueError("positions must be in [0, 2^%d)" % POS_BITS)
    return (chrom_ids.astype(np.uint64) << np.uint64(POS_BITS)) | pos.astype(np.uint64)


MAX_RECORDS_PER_PASS = 1 << 30       # dsp_freq_aggregate takes < 2^31 records; its scratch is ~100 B per record


def _aggregate_device(keys, p0, p1, label, prob_cf, sort_by_key, device, max_records=None):
    """numpy columns -> (key, first, s0, s1, met, unmet, cov) numpy arrays via the GPU.  More than ``max_records``
    records are aggregated in several passes over key-hash shards: a site's records never span two shards and keep
    their order inside one, so every sum is the same as in one pass; the rows are then put back in the one-pass
    order (a genome-scale run of > 2^31 calls, which the reference streams through a dict)."""
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("call_freq aggregation needs a CUDA device; there is no CPU path")
    n = int(keys.shape[0])
    limit = int(max_records or MAX_RECORDS_PER_PASS)
    dev = torch.device("cuda", device)

    def one_pass(k, a, b, lab, by_key):
        with torch.cuda.device(dev):
            t_key = torch.from_numpy(np.ascontiguousarray(k).view(np.int64)).to(dev)
            t_p0 = torch.from_numpy(np.ascontiguousarray(a)).to(dev)
            t_p1 = torch.from_numpy(np.ascontiguousarray(b)).to(dev)
            t_lab = torch.from_numpy(np.ascontiguousarray(lab, dtype=np.int32)).to(dev)
            out = _aggregate_tensors(t_key, t_p0, t_p1, t_lab, prob_cf, by_key, dev)
            return tuple(t.cpu().numpy() for t in out)
    if n <= limit:
        return one_pass(keys, p0, p1, label, sort_by_key)
    shards = -(-n // limit) * 2                        # hashing balances sites, not records: leave room
    owner = owner_of_key(keys, shards)
    parts = []
    for s in range(shards):
        idx = np.flatnonzero(owner == s)
        if idx.size == 0:
            continue
        if idx.size > limit:
            raise RuntimeError("one key-hash shard holds %d records (> %d): a single site dominates the input" % (idx.size, limit))
        k, first, s0, s1, met, unmet, cov = one_pass(keys[idx], p0[idx], p1[idx], label[idx], True)
        parts.append((k, idx[first], s0, s1, met, unmet, cov))
    if not parts:
        return one_pass(keys[:0], p0[:0], p1[:0], label[:0], sort_by_key)
    cols = [np.concatenate([p[i] for p in parts]) for i in range(7)]
    order = np.argsort(cols[0].view(np.uint64), kind="stable") if sort_by_key else np.argsort(cols[1], kind="stable")
    return tuple(c[order] for c in cols)


def _aggregate_compact(rec, prob_cf, sort_by_key, device):
    """``Records`` with chromosome codes -> (key, first, s0, s1, met, unmet, cov, names in rank order) through
    ``dsp_freq_aggregate_host``: host columns in, host rows out, site keys built on the device from the 4-byte codes and
    the positions.  No torch in this path: the ``call_freq`` command line does not pay its import."""
    codes, table = rec._codes
    order = sorted(range(len(table)), key=lambda i: table[i])           # Python string order = the reference's sort order
    rank = np.empty(max(len(table), 1), np.int64)
    rank[order] = np.arange(len(table))
    n = len(rec)
    L = _native.lib()
    c = lambda a, dt: np.ascontiguousarray(a, dtype=dt)
    code, pos, p0, p1, lab = c(codes, np.int32), c(rec.pos, np.int64), c(rec.p0, np.float64), c(rec.p1, np.float64), c(rec.label, np.int32)
    prof = os.environ.get("DSP_B200_PROFILE")
    t0 = time.perf_counter()
    cap = min(n, 1 << 22)
    while True:
        o_key, o_first = np.empty(cap, np.uint64), np.empty(cap, np.int64)
        o_p0, o_p1 = np.empty(cap, np.float64), np.empty(cap, np.float64)
        o_met, o_unmet, o_cov = np.empty(cap, np.int32), np.empty(cap, np.int32), np.empty(cap, np.int32)
        ns = C.c_int64(0)
        p = lambda a: a.ctypes.data
        rc = L.dsp_freq_aggregate_host(int(device), p(code), p(rank), len(rank), p(pos), p(p0), p(p1), p(lab), n, float(prob_cf),
                                       int(bool(sort_by_key)), p(o_key), p(o_first), p(o_p0), p(o_p1), p(o_met), p(o_unmet), p(o_cov),
                                       cap, C.byref(ns))
        if rc == 4 and ns.value > cap:               # more sites than the first guess: size the rows exactly and repeat
            cap = int(ns.value)
            continue
        if rc == 1 and b"positions must be" in (L.dsp_last_error() or b""):
            raise ValueError("positions must be in [0, 2^%d)" % POS_BITS)
        _native.check(rc, "dsp_freq_aggregate_host")
        break
    if prof:
        print("call_freq host seconds: upload + keys + aggregate + download %.3f (incl. CUDA context creation)" % (time.perf_counter() - t0))
    m = int(ns.value)
    return (o_key[:m].view(np.int64), o_first[:m], o_p0[:m], o_p1[:m], o_met[:m], o_unmet[:m], o_cov[:m], [table[i] for i in order])


def _aggregate_tensors(t_key, t_p0, t_p1, t_lab, prob_cf, sort_by_key, dev):
    """Device tensors in, device tensors out (rows = sites)."""
    import torch
    L = _native.lib()
    n = int(t_key.shape[0])
    o_key = torch.empty(n, dtype=torch.int64, device=dev)
    o_first = torch.empty(n, dtype=torch.int64, device=dev)
    o_p0 = torch.empty(n, dtype=torch.float64, device=dev)
    o_p1 = torch.empty(n, dtype=torch.float64, device=dev)
    o_met = torch.empty(n, dtype=torch.int32, device=dev)
    o_unmet = torch.empty(n, dtype=torch.int32, device=dev)
    o_cov = torch.empty(n, dtype=torch.int32, device=dev)
    nsites = C.c_int64(0)
    stream = torch.cuda.current_stream(dev).cuda_stream
    _native.check(L.dsp_freq_aggregate(dev.index, t_key.data_ptr(), t_p0.data_ptr(), t_p1.data_ptr(), t_lab.data_ptr(),
                                       n, float(prob_cf), int(bool(sort_by_key)),
                                       o_key.data_ptr(), o_first.data_ptr(), o_p0.data_ptr(), o_p1.data_ptr(),
                                       o_met.data_ptr(), o_unmet.data_ptr(), o_cov.data_ptr(),
                                       C.byref(nsites), stream), "dsp_freq_aggregate")
    m = int(nsites.value)
    return tuple(t[:m] for t in (o_key, o_first, o_p0, o_p1, o_met, o_unmet, o_cov))


def aggregate_records(rec, prob_cf, contig_name=None, sort_by_key=False, device=0):
    """``calculate_mods_frequency`` on parsed records -> ``FreqTable`` (rows ordered by first
    callable appearance, or by (chrom, pos) when ``sort_by_key``)."""
    n_total = len(rec)
    if contig_name is not None:                       # call_mods_freq.py:52
        rec = rec.select(rec.chrom_in({contig_name}))
    if len(rec) == 0:
        e = np.empty(0)
        return FreqTable(np.empty(0, object), e.astype(np.int64), np.empty(0, object), e.astype(np.int64), np.empty(0, object),
                         e, e, e.astype(np.int32), e.astype(np.int32), e.astype(np.int32), e.astype(np.int64), n_total, 0)
    if rec._codes is not None and len(rec) <= MAX_RECORDS_PER_PASS:
        # compact records (native parser): the site keys are built on the device from the 4-byte chromosome codes and
        # the positions -- no 8-byte id / key columns, no extra passes over the records on the host
        k, first, s0, s1, met, unmet, cov, names = _aggregate_compact(rec, prob_cf, sort_by_key, device)
    else:
        ids, names = rec.chrom_ranks()
        keys = make_keys(ids, rec.pos)
        k, first, s0, s1, met, unmet, cov = _aggregate_device(keys, rec.p0, rec.p1, rec.label, prob_cf, sort_by_key, device)
    k = k.view(np.uint64)
    names = np.asarray(names, dtype=object)
    chrom = names[(k >> np.uint64(POS_BITS)).astype(np.int64)]
    pos = (k & np.uint64((1 << POS_BITS) - 1)).astype(np.int64)
    strand, pis, kmer = rec.meta_at(first)
    return FreqTable(chrom, pos, strand, pis, kmer, s0, s1, met, unmet, cov, first, n_total, int(cov.sum()))


def _warm_device_in_background(device):
    import threading
    L = _native.lib()
    threading.Thread(target=lambda: L.dsp_device_warmup(int(device)), daemon=True).start()


# ---- bounded host memory: key-hash shards, the files re-read once per shard ---------------------------------------
# The reference streams its input line by line through a dict (``call_mods_freq.py:45-66``); what it keeps is one
# SiteStats per site.  Here the parsed columns of every record of a pass sit in host memory (HOST_RECORD_BYTES each)
# until the GPU has them, so an input that does not fit is aggregated shard by shard: shard s of S holds the records
# whose site key hashes to s.  A site's records never span two shards and keep their file order inside one, so every
# float64 sum is the one-pass sum; rows carry the global index of their first callable record, which restores the
# dict's insertion order at the end.  The price is parsing: the files are read S times (128 M records/s on 16 threads).

HOST_RECORD_BYTES = 80
STREAM_CHUNK_BYTES = 1 << 30


def default_host_record_budget():
    """Records whose parsed columns fit in half of the host memory that is available now (at most one aggregation pass)."""
    avail = None
    try:                                               # MemAvailable counts the page cache the kernel can drop (the input
        with open("/proc/meminfo") as f:               # files that were just read sit there); free pages alone do not
            for line in f:
                if line.startswith("MemAvailable:"):
                    avail = int(line.split()[1]) * 1024
                    break
    except (OSError, ValueError, IndexError):
        pass
    if avail is None:
        try:
            avail = os.sysconf("SC_AVPHYS_PAGES") * os.sysconf("SC_PAGE_SIZE")
        except (ValueError, OSError, AttributeError):
            avail = 16 << 30
    return int(min(MAX_RECORDS_PER_PASS, max(1 << 20, avail // 2 // HOST_RECORD_BYTES)))


def estimate_records(mods_files):
    """Upper-ish estimate of the number of call_mods lines without reading the files: bytes / (mean line length of the
    first plain file's first MB); a .gz file counts 5 x its size."""
    total, line = 0, None
    for f in mods_files:
        size = os.path.getsize(f)
        if f.endswith(".gz"):
            size *= 5
        elif line is None and size:
            with open(f, "rb") as fh:
                head = fh.read(1 << 20)
            if head.count(b"\n"):
                line = len(head) / head.count(b"\n")
        total += size
    return int(total / max(line or 50.0, 20.0) * 1.05) + 1


def _file_chunks(mods_files, chunk_bytes):
    """(path, byte_range) pieces in file order; a line belongs to the piece its first byte lies in; .gz files go whole."""
    for f in mods_files:
        size = os.path.getsize(f)
        if size == 0:
            continue
        if f.endswith(".gz") or size <= chunk_bytes:
            yield f, None
        else:
            for lo in range(0, size, chunk_bytes):
                yield f, (lo, min(lo + chunk_bytes, size))


def calculate_mods_frequency_streaming(mods_files, prob_cf, contigs=None, device=0, max_host_records=None, shards=None,
                                       chunk_bytes=None):
    """``calculate_mods_frequency`` with host memory bounded by ``max_host_records`` records (+ one chunk of the input):
    -> ``FreqTable`` with the same rows, order and bits as the one-pass result.  ``contigs``: None or the set of
    chromosome names to keep (``call_mods_freq.py:52``).  ``shards`` overrides the shard count derived from the
    estimated input size."""
    if type(mods_files) is str:
        mods_files = [mods_files, ]
    budget = int(max_host_records or default_host_record_budget())
    if shards is None:
        shards = max(1, -(-int(estimate_records(mods_files) * 1.25) // budget))       # hashing balances sites, not records
    shards = int(shards)
    chunk_bytes = int(chunk_bytes or STREAM_CHUNK_BYTES)
    wanted = None if contigs is None else set(contigs)
    gid = {}                                           # chromosome name -> id, first-seen order: the same in every pass
    tables, n_total = [], 0
    for s in range(shards):
        parts, gidx, base = [], [], 0
        for path, rng in _file_chunks(mods_files, chunk_bytes):
            rec = read_mods_file(path, byte_range=rng)
            n = len(rec)
            if n == 0:
                continue
            codes, table = rec.chrom_codes()
            ids = np.array([gid.setdefault(nm, len(gid)) for nm in table], np.int64)[codes]
            keep = owner_of_key(make_keys(ids, rec.pos), shards) == s if shards > 1 else np.ones(n, bool)
            if wanted is not None:
                keep &= rec.chrom_in(wanted)
            idx = np.flatnonzero(keep)
            if idx.size:
                parts.append(rec.select(idx))
                gidx.append(idx + base)
            base += n
            del rec, codes, ids, keep
        n_total = base
        if not parts:
            continue
        sub = Records.concat(parts)
        g = np.concatenate(gidx)
        del parts, gidx
        t = aggregate_records(sub, prob_cf, None, False, device)
        t.first_index = g[t.first_index]               # global record index of the site's first callable record
        tables.append(t)
        del sub, g
    table = FreqTable.concat(tables)
    table = table.reorder(np.argsort(table.first_index, kind="stable"))
    table.n_records = n_total
    return table


def calculate_mods_frequency(mods_files, prob_cf, contig_name=None, device=0, max_host_records=None):
    """call mod_freq from call_mods files (``call_mods_freq.py:29-74``).  Files are read in
    argument order; returns a ``FreqTable`` (dict-like ``sitekey2stats``).  An input whose parsed records would not
    fit in ``max_host_records`` (default: half of the available host memory) goes through
    ``calculate_mods_frequency_streaming``."""
    if type(mods_files) is str:
        mods_files = [mods_files, ]
    budget = int(max_host_records or default_host_record_budget())
    if estimate_records(mods_files) > budget:
        _warm_device_in_background(device)
        table = calculate_mods_frequency_streaming(mods_files, prob_cf, None if contig_name is None else {contig_name}, device, budget)
        count, used = table.n_records, table.n_used
        if count > 0:
            if contig_name is None:
                print("{:.2f}% ({} of {}) calls used..".format(used / float(count) * 100, used, count))
            else:
                print("{:.2f}% ({} of {}) calls used for {}..".format(used / float(count) * 100, used, count, contig_name))
        return table
    t0 = time.perf_counter()
    _warm_device_in_background(device)               # the CUDA context comes up while the files are parsed
    rec = Records.concat([read_mods_file(f) for f in mods_files])
    t1 = time.perf_counter()
    count = len(rec)
    table = aggregate_records(rec, prob_cf, contig_name, False, device)
    if os.environ.get("DSP_B200_PROFILE"):
        print("call_freq host seconds: parse %.3f, keys + upload + aggregate + rows %.3f" % (t1 - t0, time.perf_counter() - t1))
    used = table.n_used
    if count > 0:
        if contig_name is None:
            print("{:.2f}% ({} of {}) calls used..".format(used / float(count) * 100, used, count))
        else:
            print("{:.2f}% ({} of {}) calls used for {}..".format(used / float(count) * 100, used, count, contig_name))
    return table


def render_table(table, is_sort=False, is_bed=False):
    """Text of ``write_sitekey2stats`` (``call_mods_freq.py:87-120``) for a ``FreqTable``."""
    if not isinstance(table, FreqTable):
        table = _table_from_mapping(table)
    if is_sort:
        table = table.sorted()
    text = _render_native(table, is_bed)
    if text is not None:
        return text
    out = io.StringIO()
    chrom, pos, strand = table.chrom.tolist(), table.pos.tolist(), table.strand.tolist()
    cov, met, unmet = table.coverage.tolist(), table.met.tolist(), table.unmet.tolist()
    if is_bed:
        for c, p, s, cv, mt in zip(chrom, pos, strand, cov, met):
            if cv > 0:
                rmet = float(mt) / cv
                out.write("\t".join([c, str(p), str(p + 1), ".", str(cv), s, str(p), str(p + 1), "0,0,0", str(cv),
                                     str(int(round(rmet * 100 + 0.001, 0)))]) + "\n")
    else:
        pis, kmer = table.pos_in_strand.tolist(), table.kmer.tolist()
        s0, s1 = table.prob_0.tolist(), table.prob_1.tolist()
        for c, p, s, q, a, b, mt, um, cv, k in zip(chrom, pos, strand, pis, s0, s1, met, unmet, cov, kmer):
            if cv > 0:
                out.write("%s\t%d\t%s\t%d\t%.3f\t%.3f\t%d\t%d\t%d\t%.4f\t%s\n" % (c, p, s, q, a, b, mt, um, cv,
                                                                                 float(mt) / cv, k))
    return out.getvalue()


def _render_native(table, is_bed):
    """``dsp_format_freq`` (host threads); None when a text column holds a newline or NUL (the Python loop below
    prints anything)."""
    n = len(table)
    if n == 0:
        return ""
    cols = []
    for a in (table.chrom, table.strand, table.kmer):
        t = "\n".join(a.tolist())
        if t.count("\n") != n - 1 or "\0" in t:
            return None
        cols.append(t.encode())
    L = _native.lib()
    c = lambda a, dt: np.ascontiguousarray(a, dtype=dt)
    pos, pis = c(table.pos, np.int64), c(table.pos_in_strand, np.int64)
    s0, s1 = c(table.prob_0, np.float64), c(table.prob_1, np.float64)
    met, unmet, cov = c(table.met, np.int32), c(table.unmet, np.int32), c(table.coverage, np.int32)
    cap = sum(len(x) for x in cols) + n * 160
    p = lambda a: a.ctypes.data
    used = C.c_int64(0)
    while True:
        out = np.empty(cap, np.uint8)
        rc = L.dsp_format_freq(cols[0], cols[1], cols[2], p(pos), p(pis), p(s0), p(s1), p(met), p(unmet), p(cov), n,
                               int(bool(is_bed)), p(out), cap, C.byref(used), min(16, os.cpu_count() or 1))
        if rc == 4 and used.value > cap:
            cap = int(used.value)
            continue
        _native.check(rc, "dsp_format_freq")
        return out[:used.value].tobytes().decode()


def _table_from_mapping(d):
    keys = list(d.keys())
    rows = [d[k] for k in keys]
    cp = [split_key(k) for k in keys]
    obj = lambda xs: np.asarray(xs, dtype=object)
    return FreqTable(obj([c for c, _ in cp]), np.asarray([p for _, p in cp], np.int64), obj([r._strand for r in rows]),
                     np.asarray([r._pos_in_strand for r in rows], np.int64), obj([r._kmer for r in rows]),
                     np.asarray([r._prob_0 for r in rows], np.float64), np.asarray([r._prob_1 for r in rows], np.float64),
                     np.asarray([r._met for r in rows], np.int32), np.asarray([r._unmet for r in rows], np.int32),
                     np.asarray([r._coverage for r in rows], np.int32), np.arange(len(rows), dtype=np.int64))


def write_sitekey2stats(sitekey2stats, result_file, is_sort, is_bed, is_gzip):
    """write methylfreq of sites into files (``call_mods_freq.py:77-122``)."""
    t0 = time.perf_counter()
    text = render_table(sitekey2stats, is_sort, is_bed)
    if os.environ.get("DSP_B200_PROFILE"):
        print("call_freq host seconds: sort + render %.3f (%d bytes)" % (time.perf_counter() - t0, len(text)))
    if is_gzip:
        if not result_file.endswith(".gz"):
            result_file += ".gz"
        wf = gzip.open(result_file, "wt")
    else:
        wf = open(result_file, "w")
    wf.write(text)
    wf.flush()
    wf.close()


# ---- key-hash shards (multi-pass on one GPU here; the multi-GPU exchange lives in freq_dist.py / csrc/comm.cu) ----

def owner_of_key(keys, world):
    """Shard that owns a site key: multiplicative hash of the 64-bit key, its top 31 bits mapped onto [0, world) by
    multiply-shift (``route::owner_of_key`` in csrc/route.cuh is the same function on the device)."""
    h = (keys.astype(np.uint64) * np.uint64(0x9E3779B97F4A7C15)) >> np.uint64(33)
    return ((h * np.uint64(world)) >> np.uint64(31)).astype(np.int64)


def parse_contigs_arg(contigs):
    """``--contigs`` (``call_mods_freq.py:243-254``): a genome FASTA -> record names in file order
    (first word after ``>``); any other file -> its lines, de-duplicated and sorted; otherwise a
    comma-separated string, de-duplicated and sorted.  A file counts as FASTA by extension
    (.fa/.fasta/.fna) or when any of its lines starts with ``>`` (``:140-147``)."""
    if contigs is None:
        return None
    if not os.path.isfile(contigs):
        return sorted(set(contigs.strip().split(",")))
    with open(contigs, "r") as rf:
        lines = rf.read().splitlines()
    is_fasta = contigs.endswith((".fa", ".fasta", ".fna"))
    if not is_fasta:
        is_fasta = any(l.startswith(">") for l in lines)
    if is_fasta:
        return [l.strip()[1:].split(" ")[0] for l in lines if l.startswith(">")]
    return sorted(set(lines))


def order_by_contig(table, contigs, is_sort):
    """Row order of the reference's per-contig mode (``call_mods_freq.py:175-215``): every contig is
    aggregated and written on its own -- rows in first-appearance order, or by position with
    ``--sort`` -- and the per-contig files are concatenated in sorted FILE-NAME order, i.e. by
    ``contig + "."`` (the name is followed by ``.<uuid>`` in ``_call_and_write_modsfreq_process``)."""
    rank = {c: i for i, c in enumerate(sorted(set(contigs), key=lambda c: c + "."))}
    r = np.fromiter((rank[c] for c in table.chrom.tolist()), dtype=np.int64, count=len(table))
    if is_sort:
        order = np.lexsort((table.pos, r))
    else:
        order = np.argsort(r, kind="stable")          # insertion order inside a contig
    return table.reorder(order)


def call_mods_frequency_to_file(args):
    """``call_mods_freq.py:218-296``: collect files, aggregate, write.  With ``--contigs`` only the
    listed contigs are used and the rows come out contig by contig like the reference's per-contig
    mode (its temp files and ``--nproc`` worker processes are replaced by GPU passes, one contig at a time so
    that memory stays bounded by the largest contig).  Under ``torchrun`` (WORLD_SIZE > 1) the work is spread
    over the ranks' GPUs (``freq_dist.py``)."""
    print("[main]call_freq starts..")
    start = time.time()
    mods_files = []
    for ipath in args.input_path:
        input_path = os.path.abspath(ipath)
        if os.path.isdir(input_path):
            for ifile in os.listdir(input_path):
                if args.file_uid is None or ifile.find(args.file_uid) != -1:
                    mods_files.append("/".join([input_path, ifile]))
        elif os.path.isfile(input_path):
            mods_files.append(input_path)
        else:
            raise ValueError("--input_path is not a file or a directory!")
    print("get {} input file(s)..".format(len(mods_files)))
    contigs = parse_contigs_arg(getattr(args, "contigs", None))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        import torch.distributed as dist
        from . import freq_dist
        device = freq_dist.join_torchrun("call_freq aggregation")
        print("read the input files..")
        table, considered, path = freq_dist.call_freq_distributed(sorted(mods_files) if getattr(args, "sort_files", False) else mods_files,
                                                                  args.prob_cf, args.result_file, args.sort, args.bed, args.gzip,
                                                                  contigs=contigs, device=device)
        if dist.get_rank() == 0 and table.n_records > 0:
            print("{:.2f}% ({} of {}) calls used..".format(table.n_used / float(table.n_records) * 100, table.n_used, table.n_records))
            print("[main]call_freq costs %.1f seconds.." % (time.time() - start))
        return
    if contigs is None:
        print("read the input files..")
        sites_stats = calculate_mods_frequency(mods_files, args.prob_cf, max_host_records=int(getattr(args, "max_host_records", 0) or 0) or None)
        print("write the result..")
        write_sitekey2stats(sites_stats, args.result_file, args.sort, args.bed, args.gzip)
    else:
        # The reference splits the input by contig into temp files and aggregates one contig per worker
        # (call_mods_freq.py:154-200), so its memory is bounded by the largest contig.  Same bound here: the
        # records are parsed once file by file, kept only for the listed contigs, and aggregated one contig per
        # GPU pass in the reference's concatenation order.
        print("start processing {} contigs..".format(len(contigs)))
        wanted = set(contigs)
        budget = int(getattr(args, "max_host_records", 0) or 0) or default_host_record_budget()
        if estimate_records(mods_files) > budget:
            # too large to hold even once: the listed contigs in key-hash shards, rows put in the per-contig order afterwards
            table = calculate_mods_frequency_streaming(mods_files, args.prob_cf, wanted, 0, budget)
            print("{} of {} calls used for {} contigs..".format(table.n_used, table.n_records, len(contigs)))
            write_sitekey2stats(order_by_contig(table, contigs, args.sort), args.result_file, False, args.bed, args.gzip)
            print("[main]call_freq costs %.1f seconds.." % (time.time() - start))
            return
        parts, n_all = [], 0
        for f in mods_files:
            r = read_mods_file(f)
            n_all += len(r)
            parts.append(r.select(r.chrom_in(wanted)))
        rec = Records.concat(parts)
        del parts
        codes, names = rec.chrom_codes()
        tables, used = [], 0
        for contig in sorted(set(contigs), key=lambda c: c + "."):
            if contig not in names:
                continue
            sub = rec.select(codes == names.index(contig))
            t = aggregate_records(sub, args.prob_cf)
            used += t.n_used
            tables.append(t.sorted() if args.sort else t)
        print("{} of {} calls used for {} contigs..".format(used, len(rec), len(contigs)))
        table = FreqTable.concat(tables)
        write_sitekey2stats(table, args.result_file, False, args.bed, args.gzip)
    print("[main]call_freq costs %.1f seconds.." % (time.time() - start))
