"""Multi-GPU ``call_freq``: one process per GPU, records exchanged over NVLink peer memory.

The reference's parallel form of ``call_mods_frequency_to_file`` is per-contig worker processes over
temp files (``call_mods_freq.py:154-215,262-295``).  Here (``torchrun``, RANK/WORLD_SIZE set):

1. the input files are cut into contiguous byte shards in file order, one per rank; every rank parses its own
   shard with ``dsp_parse_calls`` (a line belongs to the shard its first byte lies in);
2. record counts and chromosome-name tables are all-gathered (small Python objects): global record index of a
   rank's first record, one name -> id table for everybody;
3. ``dsp_freq_aggregate_distributed`` (csrc/comm.cu): callable records go to rank ``hash(key) % world`` through
   a fused partition + all-to-all that stores straight into the owners' HBM over NVLink, are aggregated there
   by the single-GPU sort + ordered float64 replay (bit-identical sums, no partial-sum merging), and the
   finished site rows travel to the rank that parsed their first callable record -- the one that holds
   strand / pos_in_strand / k-mer (``call_mods_freq.py:55-59``);
4. rows never funnel through one rank: in the default order (dict insertion = first callable appearance) the table
   is cut into ``world`` ranges of the first-record index holding about equal numbers of rows (splitters from an
   all-gathered sample; with reads in random order almost every site is FIRST seen in rank 0's shard, so "home"
   placement would put the whole table on rank 0); a rank's rows, sorted by first record, ARE its slice.  The text
   columns of a site are then fetched from the rank that parsed that record (two small ``dsp_comm_route_rows``
   exchanges).  For ``--sort`` / ``--contigs`` the rows make one more hop to key-range owners and are sorted there;
5. every rank renders its slice (``dsp_format_freq``) and writes it at its byte offset of the result file.

The device steps sit behind a small backend interface so that the host logic above (sharding, tables, order,
writer) can be exercised by world-size-2 ``gloo`` tests on a CPU box with a stand-in that lives in ``tests/``;
the package itself has no CPU path: ``DeviceBackend`` raises without CUDA.
"""
from __future__ import annotations

import ctypes as C
import gzip
import os

import numpy as np

from . import _native
from . import call_mods_freq as cf

SITE_ROW = np.dtype([("key", "<u8"), ("first", "<u8"), ("s0", "<f8"), ("s1", "<f8"),
                     ("met", "<i4"), ("unmet", "<i4"), ("cov", "<i4"), ("pad", "<i4")])
FAT_ROW = np.dtype(SITE_ROW.descr + [("pis", "<i8"), ("strand", "S8"), ("kmer", "S24"), ("order", "<u8")])
# the text columns of a site live with the rank that parsed its first callable record: request / reply rows
META_REQ = np.dtype([("first", "<u8"), ("rank", "<u8"), ("idx", "<u8"), ("pad", "V24")])
META_REPLY = np.dtype([("rank", "<u8"), ("idx", "<u8"), ("pis", "<i8"), ("strand", "S8"), ("kmer", "S24"), ("pad", "V40")])
assert SITE_ROW.itemsize == 48 and FAT_ROW.itemsize == 96 and META_REQ.itemsize == 48 and META_REPLY.itemsize == 96
U64_MAX = np.uint64(0xFFFFFFFFFFFFFFFF)


# ---- input sharding ---------------------------------------------------------------------------------
def plan_units(mods_files, world):
    """Cut the concatenation of ``mods_files`` (argument order = record order, ``call_mods_freq.py:45-48``) into
    ``world`` contiguous shards of about equal bytes.  Returns per rank a list of ``(path, start, end)``; plain
    files are cut anywhere (the reader snaps to line starts), ``.gz`` files only as a whole."""
    sizes = [os.path.getsize(f) for f in mods_files]
    total = sum(sizes)
    shards = [[] for _ in range(world)]
    if total == 0:
        return shards
    pos = 0
    for f, sz in zip(mods_files, sizes):
        if sz == 0:
            continue
        if f.endswith(".gz"):
            r = min(world - 1, (pos + sz // 2) * world // total)
            shards[r].append((f, 0, sz))
        else:
            for r in range(world):
                lo, hi = max(pos, total * r // world), min(pos + sz, total * (r + 1) // world)
                if hi > lo:
                    shards[r].append((f, lo - pos, hi - pos))
        pos += sz
    # .gz files were placed by their midpoint: keep every rank's list in file order, and ranks monotone
    return shards


def read_units(units):
    """Parse a rank's units -> ``cf.Records`` in file order."""
    parts = []
    for path, lo, hi in units:
        whole = lo == 0 and hi >= os.path.getsize(path)
        parts.append(cf.read_mods_file(path) if whole else cf.read_mods_file(path, byte_range=(lo, hi)))
    return cf.Records.concat(parts)


# ---- device backend ----------------------------------------------------------------------------------
def open_comm(rank, world, device, window_bytes, all_gather_object):
    """A connected ``dsp_comm`` handle on ``device`` with two windows of ``window_bytes``: create, export, gather the
    blobs of all ranks through ``all_gather_object`` (collective), connect."""
    import torch
    L = _native.lib()
    h = C.c_void_p()
    with torch.cuda.device(torch.device("cuda", device)):
        _native.check(L.dsp_comm_create(C.byref(h), device, rank, world, int(window_bytes)), "dsp_comm_create")
        try:
            blob = np.zeros(512, np.uint8)
            nb = C.c_int64(0)
            _native.check(L.dsp_comm_export(h, blob.ctypes.data, blob.size, C.byref(nb)), "dsp_comm_export")
            blobs = all_gather_object(blob[:nb.value].tobytes())
            if world > 1:
                joined = np.frombuffer(b"".join(blobs), np.uint8).copy()
                _native.check(L.dsp_comm_connect(h, joined.ctypes.data, nb.value), "dsp_comm_connect")
        except BaseException:
            L.dsp_comm_destroy(h)
            raise
    return h


class DeviceBackend:
    """``dsp_comm_*`` / ``dsp_freq_aggregate_distributed`` behind the two calls the driver needs."""

    def __init__(self, rank, world, device, window_bytes, all_gather_object):
        import torch
        if not torch.cuda.is_available():
            raise RuntimeError("call_freq aggregation needs a CUDA device; there is no CPU path")
        self.torch = torch
        self.rank, self.world = rank, world
        self.dev = torch.device("cuda", device)
        self.L = _native.lib()
        self.h = C.c_void_p()
        self.window_bytes = int(window_bytes)
        self.h = open_comm(rank, world, device, self.window_bytes, all_gather_object)

    def close(self):
        if self.h:
            self.L.dsp_comm_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def aggregate_tensors(self, t_key, t_p0, t_p1, t_lab, gidx_base, bounds, prob_cf, balanced=True, rows_cap=None):
        """Device tensors in (this rank's records, file order) -> (rows tensor (m, 48) uint8 on the device: this rank's
        slice of the table, ordered by first callable record; callable records received; the world + 1 ``first``
        ranges of the slices).  ``balanced``: slices of about equal row count (sampled splitters); else rank r gets
        the rows whose first callable record lies in its own shard."""
        torch = self.torch
        n = int(t_key.shape[0])
        cap = int(rows_cap if rows_cap is not None else self.window_bytes // SITE_ROW.itemsize)
        out = torch.empty((max(cap, 1), SITE_ROW.itemsize), dtype=torch.uint8, device=self.dev)
        b = np.ascontiguousarray(bounds, dtype=np.uint64)
        assert b.shape[0] == self.world + 1
        used = np.zeros(self.world + 1, np.uint64)
        n_rows, n_call = C.c_int64(0), C.c_int64(0)
        with torch.cuda.device(self.dev):
            stream = torch.cuda.current_stream(self.dev).cuda_stream
            _native.check(self.L.dsp_freq_aggregate_distributed(
                self.h, t_key.data_ptr() if n else None, t_p0.data_ptr() if n else None, t_p1.data_ptr() if n else None,
                t_lab.data_ptr() if n else None, n, int(gidx_base), float(prob_cf), b.ctypes.data, 0 if balanced else 1,
                out.data_ptr(), cap, C.byref(n_rows), C.byref(n_call), used.ctypes.data, stream), "dsp_freq_aggregate_distributed")
        self.last_row_bounds = used
        return out[:n_rows.value], int(n_call.value)

    def aggregate(self, keys, p0, p1, label, gidx_base, bounds, prob_cf, balanced=True):
        """numpy columns in -> ``SITE_ROW`` array: this rank's slice of the table, ordered by first callable record."""
        torch = self.torch
        up = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a).astype(dt, copy=False)).to(self.dev)
        rows, _ = self.aggregate_tensors(up(keys.view(np.int64), np.int64), up(p0, np.float64), up(p1, np.float64),
                                         up(label, np.int32), gidx_base, bounds, prob_cf, balanced)
        return rows.cpu().numpy().reshape(-1).view(SITE_ROW)

    def route_rows(self, rows, field, bounds):
        """``FAT_ROW`` / ``SITE_ROW`` array -> the rows whose ``field`` falls in this rank's range, source-rank order."""
        torch = self.torch
        dt = rows.dtype
        off = dt.fields[field][1]
        t = torch.from_numpy(np.ascontiguousarray(rows).view(np.uint8).reshape(-1, dt.itemsize)).to(self.dev)
        cap = self.window_bytes // dt.itemsize
        out = torch.empty((max(cap, 1), dt.itemsize), dtype=torch.uint8, device=self.dev)
        b = np.ascontiguousarray(bounds, dtype=np.uint64)
        n_out = C.c_int64(0)
        with torch.cuda.device(self.dev):
            stream = torch.cuda.current_stream(self.dev).cuda_stream
            _native.check(self.L.dsp_comm_route_rows(self.h, t.data_ptr() if len(rows) else None, len(rows), dt.itemsize, off,
                                                     b.ctypes.data, out.data_ptr(), cap, C.byref(n_out), stream),
                          "dsp_comm_route_rows")
        return out[:n_out.value].cpu().numpy().reshape(-1).view(dt)

    def timing(self):
        ms = (C.c_float * 12)()
        _native.check(self.L.dsp_comm_last_timing(self.h, ms), "dsp_comm_last_timing")
        names = ("route_records_ms", "sort_replay_ms", "route_rows_ms", "order_ms",
                 "records_count_ms", "records_wait_counts_ms", "records_scatter_ms", "records_wait_stores_ms",
                 "rows_count_ms", "rows_wait_counts_ms", "rows_scatter_ms", "rows_wait_stores_ms")
        return dict(zip(names, [float(x) for x in ms]))


# ---- control plane ------------------------------------------------------------------------------------
def join_torchrun(what):
    """Under torchrun: join the default process group (if not yet joined), make this rank's GPU (LOCAL_RANK modulo the
    device count) current and return its index.  One GPU per rank: NCCL carries the (tiny) control plane; ranks sharing a
    GPU fall back to gloo for it -- the bulk data travels through CUDA IPC windows either way."""
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    ndev = torch.cuda.device_count()
    if ndev == 0:
        raise RuntimeError("%s needs a CUDA device; there is no CPU path" % what)
    if not dist.is_initialized():
        if ndev >= world:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        else:
            dist.init_process_group("gloo")
    device = local % ndev
    torch.cuda.set_device(device)
    return device


class TorchGroup:
    """The few small collectives of the control plane, on ``torch.distributed`` (any backend)."""

    def __init__(self, group=None):
        import torch.distributed as dist
        self.dist, self.group = dist, group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)

    def all_gather_object(self, obj):
        out = [None] * self.world
        self.dist.all_gather_object(out, obj, group=self.group)
        return out

    def barrier(self):
        self.dist.barrier(group=self.group)


class SoloGroup:
    rank, world = 0, 1

    def all_gather_object(self, obj):
        return [obj]

    def barrier(self):
        pass


def global_chrom_ids(rec, grp, contigs=None):
    """One chromosome-id table for all ranks.  ids follow Python string order of the names (so integer key order is
    the reference's ``(chrom, pos)`` sort order, ``call_mods_freq.py:88``) or, in ``--contigs`` mode, the order in which
    the reference concatenates its per-contig results: sorted by ``contig + "."`` (``:203-215``)."""
    codes, names = rec.chrom_codes()
    every = grp.all_gather_object(list(names))
    union = set()
    for t in every:
        union.update(t)
    ordered = sorted(union, key=(lambda c: c + ".") if contigs is not None else None)
    rank_of = {nm: i for i, nm in enumerate(ordered)}
    lut = np.array([rank_of[nm] for nm in names], np.int64) if len(names) else np.zeros(0, np.int64)
    return (lut[codes] if len(codes) else np.zeros(0, np.int64)), ordered


def _splitters_by_key(rows, grp, samples=512):
    """world + 1 ascending key bounds that cut the union of the ranks' rows into about equal parts."""
    k = np.sort(rows["key"])
    pick = k[np.linspace(0, len(k) - 1, min(samples, len(k))).astype(np.int64)] if len(k) else k
    allk = np.sort(np.concatenate([np.asarray(x, np.uint64) for x in grp.all_gather_object(pick)]))
    b = np.zeros(grp.world + 1, np.uint64)
    b[-1] = U64_MAX
    for w in range(1, grp.world):
        b[w] = allk[len(allk) * w // grp.world] if len(allk) else U64_MAX
    return np.maximum.accumulate(b)


def _splitters_by_chrom(rows, n_chrom, grp):
    """Key bounds at chromosome boundaries (a contig's rows stay on one rank), balanced by row count."""
    ids = (rows["key"] >> np.uint64(cf.POS_BITS)).astype(np.int64)
    cnt = np.sum(grp.all_gather_object(np.bincount(ids, minlength=n_chrom)), axis=0)
    cum = np.concatenate([[0], np.cumsum(cnt)])
    b = np.zeros(grp.world + 1, np.uint64)
    b[-1] = U64_MAX
    for w in range(1, grp.world):
        c = int(np.searchsorted(cum, cum[-1] * w / grp.world, side="left"))
        b[w] = np.uint64(min(c, n_chrom)) << np.uint64(cf.POS_BITS)
    return np.maximum.accumulate(b)


def distributed_table(rec, prob_cf, grp, backend, is_sort=False, contigs=None):
    """This rank's slice of the frequency table as a ``cf.FreqTable`` (rows in final output order; the slices of
    ranks 0..world-1 concatenate to the reference's table) and (records seen, records used) summed over ranks."""
    n_seen = len(rec)
    if contigs is not None:                                   # call_mods_freq.py:52 / :262-295
        rec = rec.select(rec.chrom_in(set(contigs)))
    counts = grp.all_gather_object((len(rec), n_seen))
    bounds = np.concatenate([[0], np.cumsum([c[0] for c in counts])]).astype(np.uint64)
    base = int(bounds[grp.rank])
    ids, names = global_chrom_ids(rec, grp, contigs)
    keys = cf.make_keys(ids, rec.pos) if len(rec) else np.zeros(0, np.uint64)
    rows = backend.aggregate(keys, rec.p0, rec.p1, rec.label, base, bounds, prob_cf)
    used = int(np.sum(grp.all_gather_object(int(rows["cov"].sum()))))
    # Text columns (strand, pos_in_strand, k-mer) of a site come from its first callable record (call_mods_freq.py:55-59),
    # which lives with the rank that parsed it: ask that rank (one exchange of 48-byte requests routed by `first` over
    # the ranks' record shards, one of 96-byte replies routed back by requesting rank).
    fat = np.zeros(len(rows), FAT_ROW)
    for f in SITE_ROW.names:
        fat[f] = rows[f]
    if grp.world > 1:
        req = np.zeros(len(rows), META_REQ)
        req["first"], req["rank"], req["idx"] = rows["first"], grp.rank, np.arange(len(rows), dtype=np.uint64)
        asked = backend.route_rows(req, "first", bounds)
        local = (asked["first"] - np.uint64(base)).astype(np.int64)
        assert len(local) == 0 or (local.min() >= 0 and local.max() < len(rec))
        strand, pis, kmer = rec.meta_cells(local)
        reply = np.zeros(len(asked), META_REPLY)
        reply["rank"], reply["idx"], reply["pis"], reply["strand"], reply["kmer"] = asked["rank"], asked["idx"], pis, strand, kmer
        back = backend.route_rows(reply, "rank", np.arange(grp.world + 1, dtype=np.uint64))
        assert len(back) == len(rows) and (back["rank"] == grp.rank).all()
        at = back["idx"].astype(np.int64)
        fat["pis"][at], fat["strand"][at], fat["kmer"][at] = back["pis"], back["strand"], back["kmer"]
    else:
        local = (rows["first"] - np.uint64(base)).astype(np.int64)
        strand, pis, kmer = rec.meta_cells(local)
        fat["pis"], fat["strand"], fat["kmer"] = pis, strand, kmer
    if is_sort or contigs is not None:
        if is_sort:
            b = _splitters_by_key(fat, grp)
        else:
            b = _splitters_by_chrom(fat, len(names), grp)
        fat = backend.route_rows(fat, "key", b) if grp.world > 1 else fat
        if is_sort:
            fat = fat[np.argsort(fat["key"], kind="stable")]
        else:                                                 # contig by contig, insertion order inside a contig
            fat = fat[np.lexsort((fat["first"], fat["key"] >> np.uint64(cf.POS_BITS)))]
    names_a = np.asarray(names, dtype=object)
    chrom = names_a[(fat["key"] >> np.uint64(cf.POS_BITS)).astype(np.int64)] if len(fat) else np.empty(0, object)
    pos = (fat["key"] & np.uint64((1 << cf.POS_BITS) - 1)).astype(np.int64)
    table = cf.FreqTable(chrom, pos, cf._cells_to_str(fat["strand"]), fat["pis"].astype(np.int64), cf._cells_to_str(fat["kmer"]),
                         fat["s0"].copy(), fat["s1"].copy(), fat["met"].copy(), fat["unmet"].copy(), fat["cov"].copy(),
                         fat["first"].astype(np.int64), sum(c[1] for c in counts), used)
    return table, sum(c[0] for c in counts)


def write_slices(text, result_file, is_gzip, grp):
    """Every rank writes its slice at its byte offset of ONE result file (``call_mods_freq.py:91-101`` names it).
    gzip: each slice is its own member; concatenated members are one valid gzip stream."""
    if is_gzip and not result_file.endswith(".gz"):
        result_file += ".gz"
    data = text.encode() if isinstance(text, str) else text
    if is_gzip:
        data = gzip.compress(data) if len(data) else b""
    sizes = grp.all_gather_object(len(data))
    off = int(sum(sizes[:grp.rank]))
    if grp.rank == 0:
        with open(result_file, "wb") as f:
            f.truncate(int(sum(sizes)))
    grp.barrier()
    if len(data):
        with open(result_file, "r+b") as f:
            f.seek(off)
            f.write(data)
    grp.barrier()
    return result_file


def default_window_bytes(n_local, grp):
    """Receive-window size: 1.3 x the per-rank share of all records (the key hash balances sites, not records)
    plus slack, in 32-byte records."""
    total = int(sum(grp.all_gather_object(int(n_local))))
    per = total // max(grp.world, 1)
    return max(int(per * 1.3) + (1 << 16), 1 << 16) * 32


def call_freq_distributed(mods_files, prob_cf, result_file, is_sort, is_bed, is_gzip, contigs=None, grp=None,
                          backend=None, device=0, records=None):
    """``call_mods_frequency_to_file`` across the ranks of ``grp`` (default: the initialised process group).
    ``records``: this rank's calls as ``cf.Records`` already in memory (contiguous shards in rank order, e.g. what
    ``call_mods --freq_out`` has just produced) instead of files to parse."""
    import time
    grp = grp or TorchGroup()
    t0 = time.perf_counter()
    rec = records if records is not None else read_units(plan_units(mods_files, grp.world)[grp.rank])
    t1 = time.perf_counter()
    own_backend = backend is None
    if own_backend:
        backend = DeviceBackend(grp.rank, grp.world, device, default_window_bytes(len(rec), grp), grp.all_gather_object)
    try:
        table, n_considered = distributed_table(rec, prob_cf, grp, backend, is_sort, contigs)
    finally:
        if own_backend:
            backend.close()
    t2 = time.perf_counter()
    text = cf.render_table(table, False, is_bed)
    t3 = time.perf_counter()
    path = write_slices(text, result_file, is_gzip, grp)
    if os.environ.get("DSP_B200_PROFILE"):
        print("call_freq rank %d host seconds: parse %.3f, exchange + aggregate + meta + order %.3f, render %.3f, write %.3f"
              % (grp.rank, t1 - t0, t2 - t1, t3 - t2, time.perf_counter() - t3))
    return table, n_considered, path


# ---- synthetic workload + measurement (BASELINE.json configs[4]; bench.py `freq` object, tools/bench_freq_dist.py) ----
def _synth_hash(lo, hi, dev, seed=1):
    """Two wrapping-int64 hashes of the global record indices [lo, hi): (site hash, probability hash)."""
    import torch

    def lsr(x, s):
        return (x >> s) & ((1 << (64 - s)) - 1)

    def mix(x):                                                  # splitmix64 finaliser on wrapping int64
        x = (x ^ lsr(x, 30)) * (-4658895280553007687)            # 0xBF58476D1CE4E5B9
        x = (x ^ lsr(x, 27)) * (-7723592293110705685)            # 0x94D049BB133111EB
        return x ^ lsr(x, 31)
    g = torch.arange(lo, hi, device=dev, dtype=torch.int64)
    h = mix(g * (-7046029254386353131) + seed)                   # 0x9E3779B97F4A7C15
    return h, mix(h)


def synth_keys(lo, hi, n_sites, dev, seed=1):
    """Site keys ((chrom << 40) | pos, int64) of the records [lo, hi) of the synthetic stream: 5 chromosomes,
    ``n_sites`` positions in all, uniformly hit."""
    h, _ = _synth_hash(lo, hi, dev, seed)
    site = (h & 0x7FFFFFFFFFFFFFFF) % n_sites
    return ((site % 5) << cf.POS_BITS) | (site // 5)


def synth_records(lo, hi, n_sites, dev, seed=1):
    """Records [lo, hi) of the synthetic call_mods stream of BASELINE.json configs[4] as device tensors: a pure
    function of the global record index (so any rank can produce any range and rank 0 can rebuild the whole stream
    for the bit-exactness check): keys from ``synth_keys``; prob_1 = m / 1e6 with m uniform in [0, 1e6],
    prob_0 = (1e6 - m) / 1e6 -- the 6-decimal values call_mods prints -- label = prob_1 > prob_0."""
    import torch
    h, h2 = _synth_hash(lo, hi, dev, seed)
    site = (h & 0x7FFFFFFFFFFFFFFF) % n_sites
    key = ((site % 5) << cf.POS_BITS) | (site // 5)
    m = (h2 & 0x7FFFFFFFFFFFFFFF) % 1000001
    p1 = m.to(torch.float64) / 1e6
    p0 = (1000000 - m).to(torch.float64) / 1e6
    return key, p0, p1, (p1 > p0).to(torch.int32)


def rows_checksum(rows):
    """Order-independent 64-bit checksum of a ``SITE_ROW`` array (sum of per-row hashes, wrapping) + row count."""
    if len(rows) == 0:
        return 0, 0
    w = np.ascontiguousarray(rows).view(np.uint64).reshape(len(rows), -1)[:, :5].copy()     # key, first, s0, s1, met|unmet
    w = np.concatenate([w, rows["cov"].astype(np.uint64)[:, None]], axis=1)
    h = np.zeros(len(rows), np.uint64)
    with np.errstate(over="ignore"):
        for j in range(w.shape[1]):
            h = (h ^ w[:, j]) * np.uint64(0x9E3779B97F4A7C15)
            h ^= h >> np.uint64(29)
        return int(h.sum(dtype=np.uint64)), len(rows)


def measure(grp, device, records_per_rank, coverage=20, prob_cf=0.5, iters=5, check=True, window_factor=1.3):
    """Time ``dsp_freq_aggregate_distributed`` on the synthetic stream with the records resident in HBM: every rank
    holds ``records_per_rank`` consecutive records; returns (on every rank) a dict with whole-job records/s from the
    slowest rank's wall clock around the synchronising call, the stage times, and -- ``check`` -- whether the
    table equals the single-GPU ``dsp_freq_aggregate`` of the whole stream on rank 0, row for row, bit for bit."""
    import time
    import torch
    dev = torch.device("cuda", device)
    world, rank = grp.world, grp.rank
    total = records_per_rank * world
    n_sites = max(total // coverage, 1)
    lo, hi = rank * records_per_rank, (rank + 1) * records_per_rank
    bounds = np.array([records_per_rank * r for r in range(world + 1)], np.uint64)
    key, p0, p1, lab = synth_records(lo, hi, n_sites, dev)
    win = (int(records_per_rank * window_factor) + (1 << 16)) * 32
    be = DeviceBackend(rank, world, device, win, grp.all_gather_object)
    try:
        times, stages = [], None
        rows = None
        for it in range(iters + 2):
            grp.barrier()
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            rows, n_call = be.aggregate_tensors(key, p0, p1, lab, lo, bounds, prob_cf)
            dt = time.perf_counter() - t0
            if it >= 2:
                times.append(max(grp.all_gather_object(dt)))
                stages = be.timing()
        mine = rows.cpu().numpy().reshape(-1).view(SITE_ROW)
        sums = grp.all_gather_object((rows_checksum(mine), int(mine["cov"].sum()), n_call,
                                      bool(len(mine) == 0 or (np.diff(mine["first"].astype(np.int64)) > 0).all()), len(mine)))
        every = grp.all_gather_object(stages)
        stage_max = {k: max(d[k] for d in every) for k in stages}
        stage_min = {k: min(d[k] for d in every) for k in stages}
    finally:
        be.close()
    del key, p0, p1, lab
    t = min(times)
    out = {"records": total, "world": world, "seconds": t, "seconds_mean": sum(times) / len(times), "iterations": len(times),
           "records_per_s": total / t, "sites": sum(s[0][1] for s in sums),
           "callable": sum(s[2] for s in sums), "coverage_sum_equals_callable": sum(s[1] for s in sums) == sum(s[2] for s in sums),
           "slices_ordered": all(s[3] for s in sums), "rows_per_rank": [s[4] for s in sums], "stage_ms_max_over_ranks": stage_max, "stage_ms_min_over_ranks": stage_min,
           "prob_cf": prob_cf,
           "bit_exact": None}
    if check:
        ok = None
        if rank == 0:
            torch.cuda.empty_cache()
            k, a, b, l = synth_records(0, total, n_sites, dev)
            one = cf._aggregate_tensors(k, a, b, l, prob_cf, True, dev)
            del k, a, b, l
            ref = np.zeros(int(one[0].shape[0]), SITE_ROW)
            for name, t_ in zip(("key", "first", "s0", "s1", "met", "unmet", "cov"), one):
                ref[name] = t_.cpu().numpy().view(ref.dtype[name]) if name in ("key", "first") else t_.cpu().numpy()
            want = rows_checksum(ref)
            got = (sum(s[0][0] for s in sums) & 0xFFFFFFFFFFFFFFFF, sum(s[0][1] for s in sums))
            ok = bool(want == got)
        out["bit_exact"] = grp.all_gather_object(ok)[0]
    return out
