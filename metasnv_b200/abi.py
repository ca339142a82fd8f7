"""ctypes binding of include/msnv.h (libmsnv_gpu.so). Thin: argument marshalling only.

Raises MsnvError when the library is missing or a call fails -- there is no Python or CPU
fallback behind these functions.
"""
import ctypes as C
import os

import numpy as np

from .paths import lib_path

TILE = 1024         # replaced by the library's own value on load()


class MsnvError(RuntimeError):
    pass


SAMPLE_ARRAYS = ("pos", "seg_off", "q4_off", "mate", "seg_pos", "seg_len", "seq2", "qual")   # order of msnv_sample_reads


class SampleReads(C.Structure):
    _fields_ = [("n_reads", C.c_uint32), ("max_span", C.c_uint32), ("reserved0", C.c_uint32), ("reserved1", C.c_uint32),
                ("pos", C.c_void_p), ("seg_off", C.c_void_p), ("q4_off", C.c_void_p), ("mate", C.c_void_p),
                ("seg_pos", C.c_void_p), ("seg_len", C.c_void_p), ("seq2", C.c_void_p), ("qual", C.c_void_p)]


class RawReads(C.Structure):
    _fields_ = [("n_reads", C.c_uint32), ("max_span", C.c_uint32), ("reserved0", C.c_uint32), ("reserved1", C.c_uint32),
                ("pos", C.c_void_p), ("mate", C.c_void_p), ("seg_off", C.c_void_p), ("q4_off", C.c_void_p), ("raw_off", C.c_void_p),
                ("n_cigar", C.c_void_p), ("l_seq", C.c_void_p), ("raw", C.c_void_p)]


RAW_ARRAYS = ("pos", "mate", "seg_off", "q4_off", "raw_off", "n_cigar", "l_seq", "raw")


class CallParams(C.Structure):
    _fields_ = [("min_coverage", C.c_int32), ("calling_threshold", C.c_int32), ("min_fraction", C.c_double)]


class Hits(C.Structure):
    _fields_ = [("n_hits", C.c_uint32), ("n_samples", C.c_uint32), ("pos", C.POINTER(C.c_uint32)),
                ("pop_mask", C.POINTER(C.c_uint8)), ("ind_mask", C.POINTER(C.c_uint8)), ("cov", C.POINTER(C.c_uint16)),
                ("allele", C.POINTER(C.c_uint16)), ("total", C.POINTER(C.c_uint32))]


class Timings(C.Structure):
    _fields_ = [("ms_index", C.c_float), ("ms_d2h", C.c_float), ("ms_pileup", C.c_float), ("ms_call", C.c_float),
                ("ms_compact", C.c_float), ("ms_gather", C.c_float), ("ms_total", C.c_float),
                ("n_items", C.c_uint64), ("n_reads", C.c_uint64), ("n_bases", C.c_uint64),
                ("n_tiles", C.c_uint32), ("kernel_launches", C.c_uint32), ("n_ranges", C.c_uint32), ("ms_mate", C.c_float),
                ("ms_cov_scatter", C.c_float), ("ms_cov_scan", C.c_float), ("reserved", C.c_uint32),
                ("cov_positions", C.c_uint64), ("cov_blocks", C.c_uint64)]


class CovBlocks(C.Structure):
    _fields_ = [("n_contigs", C.c_uint32), ("contig_len", C.c_void_p), ("blk_off", C.c_void_p), ("beg", C.c_void_p), ("end", C.c_void_p)]


class SynthDesc(C.Structure):
    _fields_ = [("seed", C.c_uint64)] + [(k, C.c_uint32) for k in (
        "n_samples", "read_len", "depth_x100", "presence_ppm", "paired_pct", "site_ppm", "err_ppm", "nbase_ppm", "refn_ppm",
        "indel_pct_x10", "clip_pct_x10", "mapq0_pct_x10", "n_contigs")] + [
        ("contig_len", C.c_void_p), ("contig_genome", C.c_void_p), ("n_genomes", C.c_uint32), ("genome_n_sub", C.c_void_p)]


class SampleSizes(C.Structure):
    _fields_ = [("n_reads", C.c_uint32), ("n_mated", C.c_uint32), ("max_span", C.c_uint32), ("reserved", C.c_uint32),
                ("n_segs", C.c_uint64), ("n_q4", C.c_uint64), ("n_aligned", C.c_uint64)]


class BgzfMember(C.Structure):
    _fields_ = [("coff", C.c_uint64), ("clen", C.c_uint32), ("isize", C.c_uint32), ("crc", C.c_uint32), ("reserved", C.c_uint32),
                ("ooff", C.c_uint64)]


# msnv_inflate_status
INFLATE_OK, INFLATE_TRUNCATED, INFLATE_BAD_CODE, INFLATE_BAD_DISTANCE, INFLATE_TOO_LONG, INFLATE_TOO_SHORT, INFLATE_BAD_CRC = range(7)

_lib = None


def load():
    """Load libmsnv_gpu.so (built in-tree by __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    p = lib_path()
    if not os.path.exists(p):
        raise MsnvError("%s is missing: run `python __graft_entry__.py` (build) first" % p)
    lib = C.CDLL(p)
    lib.msnv_abi_version.restype = C.c_int
    lib.msnv_tile.restype = C.c_int
    global TILE
    TILE = lib.msnv_tile()
    lib.msnv_device_count.restype = C.c_int
    lib.msnv_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    lib.msnv_destroy.argtypes = [C.c_void_p]
    lib.msnv_destroy.restype = None
    lib.msnv_last_error.argtypes = [C.c_void_p]
    lib.msnv_last_error.restype = C.c_char_p
    lib.msnv_shard_begin.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]
    lib.msnv_shard_add_sample.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(SampleReads)]
    lib.msnv_shard_mask_position.argtypes = [C.c_void_p, C.c_uint32]
    lib.msnv_shard_sync.argtypes = [C.c_void_p]
    lib.msnv_shard_run.argtypes = [C.c_void_p, C.POINTER(CallParams), C.POINTER(Hits)]
    lib.msnv_window_begin.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32]
    lib.msnv_window_add_sample.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(SampleReads)]
    lib.msnv_window_run.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(CallParams), C.POINTER(Hits)]
    lib.msnv_window_add_sample_raw.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(RawReads)]
    lib.msnv_expand_stats.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
    lib.msnv_shard_counts.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]
    lib.msnv_get_timings.argtypes = [C.c_void_p, C.POINTER(Timings)]
    lib.msnv_call_counts.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.POINTER(CallParams), C.POINTER(Hits)]
    lib.msnv_cov_run.argtypes = [C.c_void_p, C.POINTER(CovBlocks), C.c_uint32, C.c_void_p, C.c_void_p]
    lib.msnv_pinned_alloc.argtypes = [C.c_size_t]
    lib.msnv_pinned_alloc.restype = C.c_void_p
    lib.msnv_pinned_free.argtypes = [C.c_void_p]
    lib.msnv_pinned_free.restype = None
    lib.msnv_shard_synth.argtypes = [C.c_void_p, C.POINTER(SynthDesc), C.POINTER(C.c_int64)]
    lib.msnv_shard_sample_sizes.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(SampleSizes)]
    lib.msnv_window_sample_sizes.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(SampleSizes)]
    lib.msnv_shard_synth_ref.argtypes = [C.c_void_p, C.POINTER(SynthDesc), C.POINTER(C.c_int64)]
    lib.msnv_window_synth.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(SynthDesc), C.c_uint32, C.c_uint32]
    lib.msnv_shard_export_sample.argtypes = [C.c_void_p, C.c_uint32] + [C.c_void_p] * 8
    lib.msnv_shard_export_ref.argtypes = [C.c_void_p, C.c_void_p]
    lib.msnv_inflater_create.argtypes = [C.c_int, C.c_size_t, C.POINTER(C.c_void_p)]
    lib.msnv_inflate.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]
    lib.msnv_inflater_destroy.argtypes = [C.c_void_p]
    lib.msnv_inflater_destroy.restype = None
    lib.msnv_inflater_last_error.argtypes = [C.c_void_p]
    lib.msnv_inflater_last_error.restype = C.c_char_p
    lib.msnv_inflater_kernel_ms.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
    lib.msnv_inflater_max_members.argtypes = [C.c_size_t]
    lib.msnv_inflater_max_members.restype = C.c_uint32
    _lib = lib
    return lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


class PinnedArena:
    """Page-locked host memory from the library, carved out of 1 GiB slabs (cudaHostAlloc is slow per call).
    When the driver refuses to pin more, further slabs are ordinary (pageable) memory: copies from them are slower
    but still correct; `pageable_bytes` says how much that was."""
    SLAB = 1 << 30

    def __init__(self):
        self.lib = load()
        self.slabs = []          # (ptr, size)
        self.plain = []          # pageable slabs (numpy owns them)
        self.cur = None          # numpy view of the current slab
        self.off = 0
        self.bytes = 0
        self.pageable_bytes = 0

    def alloc(self, nbytes):
        n = (max(1, int(nbytes)) + 255) // 256 * 256
        if self.cur is None or self.off + n > self.cur.size:
            size = max(self.SLAB, n)
            p = None if self.plain else self.lib.msnv_pinned_alloc(size)      # once pinning failed, do not retry per slab
            if p:
                self.slabs.append((p, size))
                self.cur = np.ctypeslib.as_array((C.c_uint8 * size).from_address(p))
            else:
                try:
                    self.cur = np.empty(size, np.uint8)
                except MemoryError:
                    raise MsnvError("no host memory for another %d-byte staging slab" % size)
                self.plain.append(self.cur)
                self.pageable_bytes += size
            self.off = 0
        v = self.cur[self.off:self.off + n]
        self.off += n
        self.bytes += n
        return v

    def close(self):
        self.cur = None
        for p, _ in self.slabs:
            self.lib.msnv_pinned_free(p)
        self.slabs = []
        self.plain = []


class HitsView:
    """Numpy copies of a msnv_hits result."""

    def __init__(self, h):
        n, s = h.n_hits, h.n_samples
        self.n_hits, self.n_samples = n, s

        def arr(p, shape, dt):
            if n == 0:
                return np.zeros(shape, dt)
            return np.ctypeslib.as_array(p, shape=shape).astype(dt, copy=True)
        self.pos = arr(h.pos, (n,), np.uint32)
        self.pop_mask = arr(h.pop_mask, (n,), np.uint8)
        self.ind_mask = arr(h.ind_mask, (n,), np.uint8)
        self.cov = arr(h.cov, (n, s), np.uint16)
        self.allele = arr(h.allele, (n, 4, s), np.uint16)
        self.total = arr(h.total, (n, 5), np.uint32)


def device_count():
    """CUDA devices the library sees (0 without a GPU)."""
    return int(load().msnv_device_count())


class Context:
    def __init__(self, device=0):
        self.lib = load()
        self.h = C.c_void_p()
        rc = self.lib.msnv_create(device, C.byref(self.h))
        if rc != 0:
            msg = self.lib.msnv_last_error(self.h).decode()
            if self.h:
                self.lib.msnv_destroy(self.h)
            self.h = None
            raise MsnvError("msnv_create(%d) failed (%d): %s" % (device, rc, msg))
        self._keep = []

    def close(self):
        if self.h:
            self.lib.msnv_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc, what):
        if rc != 0:
            raise MsnvError("%s failed (%d): %s" % (what, rc, self.lib.msnv_last_error(self.h).decode()))

    def shard_begin(self, n_samples, ref):
        ref = np.ascontiguousarray(ref, dtype=np.uint8)
        self._keep = [ref]
        self._check(self.lib.msnv_shard_begin(self.h, n_samples, ref.size, _ptr(ref)), "msnv_shard_begin")

    def shard_add_sample(self, sample, arrays):
        """arrays: dict with pos, seg_off, q4_off, mate, seg_pos, seg_len, seq2, qual (numpy), max_span."""
        a = {k: np.ascontiguousarray(v) for k, v in arrays.items() if k != "max_span"}
        self._keep.append(a)
        r = SampleReads()
        r.n_reads = a["pos"].size
        r.max_span = int(arrays["max_span"])
        for k in SAMPLE_ARRAYS:
            setattr(r, k, _ptr(a[k]))
        self._check(self.lib.msnv_shard_add_sample(self.h, sample, C.byref(r)), "msnv_shard_add_sample")

    # ---- position windows (shards larger than device memory)
    def window_begin(self, slot, pos_lo, pos_hi):
        self._keep_win = getattr(self, "_keep_win", {})
        self._keep_win[slot] = []
        self._check(self.lib.msnv_window_begin(self.h, slot, pos_lo, pos_hi), "msnv_window_begin")

    def window_add_sample(self, slot, sample, arrays):
        a = {k: np.ascontiguousarray(v) for k, v in arrays.items() if k != "max_span"}
        self._keep_win[slot].append(a)
        r = SampleReads()
        r.n_reads = a["pos"].size
        r.max_span = int(arrays["max_span"])
        for k in SAMPLE_ARRAYS:
            setattr(r, k, _ptr(a[k]))
        self._check(self.lib.msnv_window_add_sample(self.h, slot, sample, C.byref(r)), "msnv_window_add_sample")

    def window_add_sample_raw(self, slot, sample, arrays):
        """arrays: pos, mate, seg_off, q4_off, raw_off, n_cigar, l_seq, raw (+ max_span): reads as BAM stores them; the device expands them."""
        a = {k: np.ascontiguousarray(arrays[k]) for k in RAW_ARRAYS}
        self._keep_win = getattr(self, "_keep_win", {})
        self._keep_win.setdefault(slot, []).append(a)
        r = RawReads()
        r.n_reads = a["pos"].size
        r.max_span = int(arrays["max_span"])
        for k in RAW_ARRAYS:
            setattr(r, k, _ptr(a[k]))
        self._check(self.lib.msnv_window_add_sample_raw(self.h, slot, sample, C.byref(r)), "msnv_window_add_sample_raw")

    def expand_stats(self):
        v = C.c_uint64(0)
        self._check(self.lib.msnv_expand_stats(self.h, C.byref(v)), "msnv_expand_stats")
        return int(v.value)

    def window_run(self, slot, min_coverage=4, calling_threshold=4, min_fraction=0.01, copy=True):
        p = CallParams(min_coverage, calling_threshold, min_fraction)
        h = Hits()
        self._check(self.lib.msnv_window_run(self.h, slot, C.byref(p), C.byref(h)), "msnv_window_run")
        return HitsView(h) if copy else h

    def shard_synth(self, desc, ref_only=False):
        """desc: the JSON dict printed by `msnv_synth --describe`. Returns (n_positions, first_column).
        ref_only: begin the shard and generate its reference; the reads come window by window (window_synth)."""
        cl = np.ascontiguousarray(desc["contig_len"], np.uint32)
        cg = np.ascontiguousarray(desc["contig_genome"], np.uint32)
        gs = np.ascontiguousarray(desc["genome_n_sub"], np.uint32)
        d = SynthDesc()
        d.seed = desc["seed"]
        for k in ("n_samples", "read_len", "depth_x100", "presence_ppm", "paired_pct", "site_ppm", "err_ppm", "nbase_ppm",
                  "refn_ppm", "indel_pct_x10", "clip_pct_x10", "mapq0_pct_x10"):
            setattr(d, k, int(desc[k]))
        d.n_contigs = cl.size
        d.contig_len, d.contig_genome, d.n_genomes, d.genome_n_sub = _ptr(cl), _ptr(cg), gs.size, _ptr(gs)
        first = C.c_int64(-1)
        self._synth = (d, cl, cg, gs)
        if ref_only:
            self._check(self.lib.msnv_shard_synth_ref(self.h, C.byref(d), C.byref(first)), "msnv_shard_synth_ref")
        else:
            self._check(self.lib.msnv_shard_synth(self.h, C.byref(d), C.byref(first)), "msnv_shard_synth")
        n_pos = int(sum((int(x) + TILE - 1) // TILE * TILE for x in cl))
        self.n_positions = n_pos
        return n_pos, first.value

    def window_synth(self, slot, ctg_lo, ctg_hi):
        """Reads of contigs [ctg_lo, ctg_hi) of the description given to shard_synth(ref_only=True) into a window slot."""
        self._check(self.lib.msnv_window_synth(self.h, slot, C.byref(self._synth[0]), ctg_lo, ctg_hi), "msnv_window_synth")

    def window_sample_sizes(self, slot, sample):
        z = SampleSizes()
        self._check(self.lib.msnv_window_sample_sizes(self.h, slot, sample, C.byref(z)), "msnv_window_sample_sizes")
        return z

    def sample_sizes(self, sample):
        z = SampleSizes()
        self._check(self.lib.msnv_shard_sample_sizes(self.h, sample, C.byref(z)), "msnv_shard_sample_sizes")
        return z

    def export_sample(self, sample, alloc=None):
        """Copy a sample of the open shard to host arrays. alloc(nbytes) -> writable uint8 numpy view (e.g. pinned)."""
        z = self.sample_sizes(sample)
        if alloc is None:
            def alloc(n):
                return np.empty(n, np.uint8)
        n, n1 = z.n_reads, z.n_reads + 1
        spec = [("pos", n, np.int32), ("seg_off", n1, np.uint32), ("q4_off", n1, np.uint32), ("mate", n, np.int32),
                ("seg_pos", z.n_segs, np.int32), ("seg_len", z.n_segs, np.uint16),
                ("seq2", z.n_q4, np.uint8), ("qual", z.n_q4 * 4, np.uint8)]
        out = {"max_span": z.max_span}
        for k, cnt, dt in spec:
            raw = alloc(max(1, int(cnt)) * np.dtype(dt).itemsize)
            out[k] = raw.view(dt)[:int(cnt)]
        if n:
            self._check(self.lib.msnv_shard_export_sample(self.h, sample, *[_ptr(out[k]) if out[k].size else None for k, _, _ in spec]),
                        "msnv_shard_export_sample")
        return out

    def export_ref(self, n_positions):
        ref = np.empty(n_positions, np.uint8)
        self._check(self.lib.msnv_shard_export_ref(self.h, _ptr(ref)), "msnv_shard_export_ref")
        return ref

    def shard_mask_position(self, pos):
        self._check(self.lib.msnv_shard_mask_position(self.h, pos), "msnv_shard_mask_position")

    def shard_sync(self):
        self._check(self.lib.msnv_shard_sync(self.h), "msnv_shard_sync")

    def shard_run(self, min_coverage=4, calling_threshold=4, min_fraction=0.01, copy=True):
        p = CallParams(min_coverage, calling_threshold, min_fraction)
        h = Hits()
        self._check(self.lib.msnv_shard_run(self.h, C.byref(p), C.byref(h)), "msnv_shard_run")
        return HitsView(h) if copy else h

    def shard_counts(self, sample, first, n):
        out = np.zeros((n, 5), np.uint16)
        self._check(self.lib.msnv_shard_counts(self.h, sample, first, n, _ptr(out)), "msnv_shard_counts")
        return out

    def timings(self):
        t = Timings()
        self._check(self.lib.msnv_get_timings(self.h, C.byref(t)), "msnv_get_timings")
        return {k: getattr(t, k) for k, _ in Timings._fields_}

    def call_counts(self, n_samples, ref, acgt, matches, min_coverage=4, calling_threshold=4, min_fraction=0.01):
        ref = np.ascontiguousarray(ref, np.uint8)
        acgt = np.ascontiguousarray(acgt, np.uint64)
        matches = np.ascontiguousarray(matches, np.uint16)
        p = CallParams(min_coverage, calling_threshold, min_fraction)
        h = Hits()
        self._check(self.lib.msnv_call_counts(self.h, n_samples, ref.size, _ptr(ref), _ptr(acgt), _ptr(matches), C.byref(p), C.byref(h)),
                    "msnv_call_counts")
        return HitsView(h)

    def cov_run(self, contig_len, blk_off, beg, end, max_cov):
        contig_len = np.ascontiguousarray(contig_len, np.uint32)
        blk_off = np.ascontiguousarray(blk_off, np.uint64)
        beg = np.ascontiguousarray(beg, np.uint32)
        end = np.ascontiguousarray(end, np.uint32)
        k = contig_len.size
        b = CovBlocks(k, _ptr(contig_len), _ptr(blk_off), _ptr(beg), _ptr(end))
        cov_sum = np.zeros(k, np.uint64)
        hist = np.zeros((k, max_cov + 1), np.uint64)
        self._check(self.lib.msnv_cov_run(self.h, C.byref(b), max_cov, _ptr(cov_sum), _ptr(hist)), "msnv_cov_run")
        return cov_sum, hist


def window_slice(arrays, pos_lo, pos_hi):
    """The reads of one sample (dict as returned by Context.export_sample) that a window [pos_lo, pos_hi) needs, as a
    new dict in the same layout: every read with pos < pos_hi that can reach pos_lo (pos + max_span > pos_lo), a
    contiguous run of the coordinate-sorted reads; offsets re-based to 0, mate links re-based to the run (links that
    leave it are dropped: such mates share no position inside the window)."""
    pos = arrays["pos"]
    span = int(arrays["max_span"])
    lo = int(np.searchsorted(pos, pos_lo - span + 1, side="left"))
    hi = int(np.searchsorted(pos, pos_hi, side="left"))
    if hi <= lo:
        return None
    s0, s1 = int(arrays["seg_off"][lo]), int(arrays["seg_off"][hi])
    q0, q1 = int(arrays["q4_off"][lo]), int(arrays["q4_off"][hi])
    mate = arrays["mate"][lo:hi].astype(np.int64) - lo
    mate[(mate < 0) | (mate >= hi - lo)] = -1
    return {"max_span": span, "pos": pos[lo:hi].copy(), "seg_off": (arrays["seg_off"][lo:hi + 1] - s0).astype(np.uint32),
            "q4_off": (arrays["q4_off"][lo:hi + 1] - q0).astype(np.uint32), "mate": mate.astype(np.int32),
            "seg_pos": arrays["seg_pos"][s0:s1].copy(), "seg_len": arrays["seg_len"][s0:s1].copy(),
            "seq2": arrays["seq2"][q0:q1].copy(), "qual": arrays["qual"][4 * q0:4 * q1].copy()}


class Inflater:
    """msnv_inflater: BGZF members inflated on the device. One thread at a time per inflater; several inflaters may run
    at once, next to a Context's calls."""

    def __init__(self, device=0, max_batch_bytes=8 << 20):
        self.lib = load()
        self.max_batch_bytes = max_batch_bytes
        h = C.c_void_p()
        rc = self.lib.msnv_inflater_create(device, max_batch_bytes, C.byref(h))
        if rc != 0:
            msg = self.lib.msnv_inflater_last_error(h).decode()
            self.lib.msnv_inflater_destroy(h)
            raise MsnvError("msnv_inflater_create failed (%d): %s" % (rc, msg))
        self.h = h

    def close(self):
        if self.h:
            self.lib.msnv_inflater_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def inflate(self, comp, members):
        """comp: uint8 array; members: numpy structured array with BgzfMember's fields (or a BgzfMember ctypes array).
        Returns (out uint8 array of max(ooff + isize) bytes, int32 status per member)."""
        import numpy as np
        comp = np.ascontiguousarray(comp, dtype=np.uint8)
        m = np.ascontiguousarray(members)
        n = len(m)
        out_bytes = int(max((int(x["ooff"]) + int(x["isize"]) for x in m), default=0))
        out = np.zeros(max(out_bytes, 1), np.uint8)
        status = np.full(max(n, 1), -1, np.int32)
        rc = self.lib.msnv_inflate(self.h, _ptr(comp), comp.size, m.ctypes.data_as(C.c_void_p), n, _ptr(out), _ptr(status))
        if rc != 0:
            raise MsnvError("msnv_inflate failed (%d): %s" % (rc, self.lib.msnv_inflater_last_error(self.h).decode()))
        return out[:out_bytes], status[:n]

    def kernel_ms(self):
        ms = C.c_float()
        self.lib.msnv_inflater_kernel_ms(self.h, C.byref(ms))
        return ms.value


MEMBER_DTYPE = [("coff", "<u8"), ("clen", "<u4"), ("isize", "<u4"), ("crc", "<u4"), ("reserved", "<u4"), ("ooff", "<u8")]


def bgzf_members(path_or_bytes):
    """The BGZF members of a file, as msnv_inflate takes them: (compressed bytes, structured array of members whose
    coff index the file and whose ooff lay the members out back to back). Parsed from the format (SAMv1 4.1)."""
    import numpy as np
    data = open(path_or_bytes, "rb").read() if isinstance(path_or_bytes, str) else bytes(path_or_bytes)
    rows, pos, ooff = [], 0, 0
    while pos < len(data):
        xlen = int.from_bytes(data[pos + 10:pos + 12], "little")
        bsize, off = None, 0
        while off + 4 <= xlen:
            x = pos + 12 + off
            slen = int.from_bytes(data[x + 2:x + 4], "little")
            if data[x:x + 2] == b"BC" and slen == 2:
                bsize = int.from_bytes(data[x + 4:x + 6], "little")
            off += 4 + slen
        if bsize is None:
            raise ValueError("BGZF member without BC subfield at %d" % pos)
        end = pos + bsize + 1
        crc = int.from_bytes(data[end - 8:end - 4], "little")
        isize = int.from_bytes(data[end - 4:end], "little")
        rows.append((pos + 12 + xlen, end - 8 - (pos + 12 + xlen), isize, crc, 0, ooff))
        ooff += isize
        pos = end
    return np.frombuffer(data, np.uint8), np.array(rows, dtype=MEMBER_DTYPE)


def bgzf_batches(comp, members, max_batch_bytes):
    """Cut a file's members (bgzf_members) into msnv_inflate batches of at most max_batch_bytes on either side: a list of
    (compressed bytes, members with coff and ooff relative to the batch)."""
    out, i, n = [], 0, len(members)
    while i < n:
        j, c0, o0 = i, int(members[i]["coff"]), int(members[i]["ooff"])
        while j < n and int(members[j]["ooff"]) + int(members[j]["isize"]) - o0 <= max_batch_bytes and \
                int(members[j]["coff"]) + int(members[j]["clen"]) - c0 <= max_batch_bytes:
            j += 1
        if j == i:
            raise ValueError("member %d does not fit a batch of %d bytes" % (i, max_batch_bytes))
        sub = members[i:j].copy()
        sub["coff"] -= c0
        sub["ooff"] -= o0
        out.append((comp[c0:int(sub[-1]["coff"]) + c0 + int(sub[-1]["clen"])], sub))
        i = j
    return out
