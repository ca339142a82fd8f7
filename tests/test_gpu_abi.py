"""The C ABI called directly (ctypes, numpy buffers) on the B200: msnv_call_counts against the snpCall oracle on
random count tiles, msnv_cov_run against a numpy difference-array restatement of qaCompute.cpp:142-165."""
import os
import subprocess

import numpy as np
import pytest

from metasnv_b200 import harness as H

pytestmark = pytest.mark.gpu


def _text_from_counts(cnt, match, ref):
    """cnt [L][S][4] letters, match [L][S] -> mpileup text (first line is a dummy the caller drops)."""
    L, S, _ = cnt.shape
    rows = ["x\t1\tA" + "\t1\t.\tI" * S]
    for i in range(L):
        cols = []
        for s in range(S):
            b = "." * int(match[i, s]) + "".join(ch * int(cnt[i, s, k]) for k, ch in enumerate("ACGT"))
            cols.append("%d\t%s\t%s" % (len(b), b if b else "*", "I" * len(b) if b else "*"))
        rows.append("ctg\t%d\t%s\t%s" % (i + 1, ref[i], "\t".join(cols)))
    return "\n".join(rows) + "\n"


def _expected_lines(h, ref, kind):
    out = []
    order = [0, 1, 3, 2]
    for i in range(h.n_hits):
        mask = int(h.pop_mask[i]) if kind == "pop" else int(h.ind_mask[i])
        if not mask:
            continue
        p = int(h.pos[i])
        ent = []
        for a in order:
            if mask >> a & 1:
                ent.append("%d|%s|.|%s" % (h.total[i, 1 + a], "ACGT"[a], "|".join(str(int(x)) for x in h.allele[i, a])))
        out.append("ctg\t-\t%d\t%s\t%s\t%s\n" % (p + 1, ref[p], "|".join(str(int(x)) for x in h.cov[i]), ",".join(ent)))
    return "".join(out)


# (c, t, p) with Poisson counts; (c, t, p, "placed"): every count is thr-1, thr or thr+1 (or small), so the integer test of
# the wide (text-mode) items decides on both sides of thresholds that take the HI_THR form of call_kernel (t > 128)
@pytest.mark.parametrize("S,L,seed,opts", [(3, 700, 1, (4, 4, 0.01)), (17, 1500, 2, (4, 4, 0.01)), (5, 512, 3, (10, 2, 0.3)), (1, 100, 4, (1, 1, 0.0))] +
                         [(4, 600, 10 + t, (4, t, p, "placed")) for t in (128, 129, 255, 256) for p in (0.01, 1.0)])
def test_call_counts_matches_snpcall_oracle(S, L, seed, opts, built, tmp_path):
    from metasnv_b200 import abi
    abi.load()
    TILE = abi.TILE
    rng = np.random.default_rng(seed)
    if len(opts) == 4:
        thr = opts[1]
        cnt = rng.choice(np.array([0, 0, 0, 1, 5, thr - 1, thr, thr + 1], np.uint64), (L, S, 4))
        match = rng.choice(np.array([0, 3, thr - 1, thr, thr + 1], np.uint16), (L, S))
    else:
        cnt = rng.poisson(0.6, (L, S, 4)).astype(np.uint64) * (rng.random((L, S, 4)) < 0.3)
        cnt[rng.random((L, S, 4)) < 0.01] = 40
        match = rng.poisson(6, (L, S)).astype(np.uint16)
    ref = "".join(rng.choice(list("ACGTacgtNnR"), L))
    P = (L + TILE - 1) // TILE * TILE
    nt = P // TILE
    acgt = np.zeros((nt, S, TILE), np.uint64)
    mt = np.zeros((nt, S, TILE), np.uint16)
    refb = np.zeros(P, np.uint8)
    refb[:L] = np.frombuffer(ref.encode(), np.uint8)
    for i in range(L):
        t, o = divmod(i, TILE)
        acgt[t, :, o] = cnt[i, :, 0] | (cnt[i, :, 1] << np.uint64(16)) | (cnt[i, :, 2] << np.uint64(32)) | (cnt[i, :, 3] << np.uint64(48))
        mt[t, :, o] = match[i]
    c, t_, p = opts[:3]
    with abi.Context(0) as ctx:
        h = ctx.call_counts(S, refb, acgt, mt, c, t_, p)
    assert np.all(np.diff(h.pos.astype(np.int64)) > 0)                    # ascending, no duplicates
    ind = str(tmp_path / "indiv")
    r = subprocess.run([H.oracle_bin("snpcall_oracle"), "-i", ind, "-c", str(c), "-t", str(t_), "-p", str(p)],
                       input=_text_from_counts(cnt, match, ref).encode(), capture_output=True)
    assert r.returncode == 0
    assert _expected_lines(h, ref, "pop") == r.stdout.decode()
    assert _expected_lines(h, ref, "ind") == open(ind).read()
    if len(opts) == 4:
        assert r.stdout if p < 1.0 else open(ind).read()          # p = 1.0: the individual test decides


@pytest.mark.parametrize("seed,max_cov", [(1, 10), (2, 30), (3, 1), (4, 1023), (5, 1024), (6, 5000)])
def test_cov_run_matches_numpy(seed, max_cov, built):
    """Random blocks, plus: one position under 10 000 blocks (coverage values above the 1024 bins held in shared memory),
    blocks that end exactly on a 4096-position chunk boundary, start on one, or cross several chunks, and contigs without
    blocks between contigs with blocks."""
    from metasnv_b200 import abi
    rng = np.random.default_rng(seed)
    lens = np.array([1, 5, 4095, 4096, 4097, 20000, 123457, 9000, 7, 50000], np.uint32)
    begs, ends, off = [], [], [0]
    for k, ln in enumerate(lens):
        n = int(rng.integers(0, 400)) if ln > 10 else 2
        if k in (7, 8):
            n = 0
        b = np.sort(rng.integers(0, max(1, ln - 1), n)).astype(np.uint32)
        e = np.minimum(b + rng.integers(1, 9000 if ln > 10000 else 150, n).astype(np.uint32), ln - 1).astype(np.uint32)
        if k == 5:                                    # 10 000 blocks over position 8192 (a chunk boundary), coverage ramps 0 -> 10 000
            b = np.concatenate([b, 8000 + np.arange(10000, dtype=np.uint32) % 193])
            e = np.concatenate([e, 8193 + np.arange(10000, dtype=np.uint32) % 211])
        if k == 9:                                    # ending on, starting on and crossing 4096-position chunks
            b = np.concatenate([b, np.array([100, 4096, 4095, 8191, 0, 12288, 5000, 40960 - 7], np.uint32)])
            e = np.concatenate([e, np.array([4096, 8192, 4097, 8192, 49999, 40960, 45000, 40960], np.uint32)])
        keep = e > b
        begs.append(b[keep]); ends.append(e[keep]); off.append(off[-1] + int(keep.sum()))
    beg = np.concatenate(begs) if off[-1] else np.zeros(0, np.uint32)
    end = np.concatenate(ends) if off[-1] else np.zeros(0, np.uint32)
    with abi.Context(0) as ctx:
        cov_sum, hist = ctx.cov_run(lens, np.array(off, np.uint64), beg, end, max_cov)
    top = 0
    for k, ln in enumerate(lens):
        d = np.zeros(int(ln) + 1, np.int64)
        np.add.at(d, begs[k], 1)
        np.add.at(d, ends[k], -1)
        cov = np.cumsum(d)[:ln]
        assert cov_sum[k] == cov.sum()
        want = np.bincount(np.minimum(cov, max_cov), minlength=max_cov + 1)
        assert np.array_equal(hist[k], want.astype(np.uint64)), k
        assert hist[k].sum() == ln
        top = max(top, int(cov.max()) if ln else 0)
    assert top >= 10000


def test_cov_run_refuses_histograms_above_the_limit(built):
    """max_cov = 0xFFFFFFFF (where max_cov + 1 wraps to 0 in 32 bits) and histograms beyond MSNV_COV_MAX_COUNTERS are refused
    with MSNV_E_LIMIT before anything is launched; the context stays usable."""
    import ctypes as C
    from metasnv_b200 import abi
    lens = np.array([5000, 7000], np.uint32)
    off = np.array([0, 1, 1], np.uint64)
    beg, end = np.array([10], np.uint32), np.array([20], np.uint32)
    b = abi.CovBlocks(2, abi._ptr(lens), abi._ptr(off), abi._ptr(beg), abi._ptr(end))
    cov_sum, hist = np.zeros(2, np.uint64), np.zeros(16, np.uint64)
    with abi.Context(0) as ctx:
        for max_cov in (0xFFFFFFFF, 1 << 27, (1 << 26)):
            assert ctx.lib.msnv_cov_run(ctx.h, C.byref(b), max_cov, abi._ptr(cov_sum), abi._ptr(hist)) == -4, max_cov     # MSNV_E_LIMIT
            assert "exceed the limit" in ctx.lib.msnv_last_error(ctx.h).decode()
        s, h = ctx.cov_run(lens, off, beg, end, 3)
    assert s.tolist() == [10, 0] and h[0].tolist() == [4990, 10, 0, 0] and h[1].tolist() == [7000, 0, 0, 0]


def test_cov_run_failed_allocation_leaves_the_context_usable(built):
    """A call whose difference array cannot be allocated (64 contigs of 2^32 - 1 positions: about 1.1 TiB) returns
    MSNV_E_CUDA. The buffer it could not grow is left empty and the runtime's error is cleared, so the next call on the
    same context allocates it again and gives the result it gave before."""
    import ctypes as C
    from metasnv_b200 import abi
    lens = np.array([5000, 7000], np.uint32)
    off = np.array([0, 1, 2], np.uint64)
    beg, end = np.array([10, 100], np.uint32), np.array([20, 4000], np.uint32)
    huge = np.full(64, 0xFFFFFFFF, np.uint32)
    huge_off = np.zeros(65, np.uint64)
    b = abi.CovBlocks(64, abi._ptr(huge), abi._ptr(huge_off), None, None)
    cov_sum, hist = np.zeros(64, np.uint64), np.zeros(64, np.uint64)
    with abi.Context(0) as ctx:
        s0, h0 = ctx.cov_run(lens, off, beg, end, 3)
        assert ctx.lib.msnv_cov_run(ctx.h, C.byref(b), 0, abi._ptr(cov_sum), abi._ptr(hist)) == -1     # MSNV_E_CUDA
        assert "out of memory" in ctx.lib.msnv_last_error(ctx.h).decode()
        s1, h1 = ctx.cov_run(lens, off, beg, end, 3)
    assert s0.tolist() == [10, 3900] and s1.tolist() == s0.tolist()
    assert np.array_equal(h1, h0)


def _called_positions(path, offsets):
    out = []
    for line in open(path):
        f = line.split("\t")
        out.append(offsets[f[0]] + int(f[2]) - 1)
    return np.array(out, np.int64)


@pytest.mark.parametrize("preset,scale,samples", [("c2", 0.003, 16), ("c1", 0.03, 10)])
def test_device_synth_equals_bam_pipeline(preset, scale, samples, built, tmp_path):
    """The device-side shard generator (used for the full-size benchmark shapes) and the BAM files written from the
    same model give identical per-sample counts and identical calls; exported host arrays re-uploaded through
    msnv_shard_add_sample() (the end-to-end path of bench.py) give the same hits again."""
    from metasnv_b200 import abi
    data = str(tmp_path / "data")
    H.synth(data, preset, scale, samples)
    dump = str(tmp_path / "counts.bin")
    rc, err = H.run_product_snpcall(data, str(tmp_path / "bam"), env=dict(os.environ, MSNV_DUMP_COUNTS=dump))
    assert rc == 0, err
    lay = [l.rstrip("\n").split("\t") for l in open(dump + ".layout")]
    S, P, first_bam = int(lay[0][0]), int(lay[0][1]), int(lay[0][2])
    offsets = {n: int(o) for n, o, _ in lay[1:]}
    want = np.fromfile(dump, np.uint16).reshape(S, P, 5)

    desc = H.describe(preset, scale, samples)
    with abi.Context(0) as ctx:
        n_pos, first = ctx.shard_synth(desc)
        assert (n_pos, first) == (P, first_bam)
        exported = [ctx.export_sample(s) for s in range(S)]
        ref = ctx.export_ref(P)
        ctx.shard_mask_position(first)
        h = ctx.shard_run()
        for s in range(S):
            got = ctx.shard_counts(s, 0, P)
            bad = np.argwhere(got != want[s])
            assert bad.size == 0, "sample %d first mismatch at %s: device-synth %s, BAM path %s" % (s, bad[0], got[tuple(bad[0])], want[s][tuple(bad[0])])
        pop = h.pos[h.pop_mask != 0].astype(np.int64)
        ind = h.pos[h.ind_mask != 0].astype(np.int64)
        assert np.array_equal(pop, _called_positions(str(tmp_path / "bam.called"), offsets))
        assert np.array_equal(ind, _called_positions(str(tmp_path / "bam.indiv"), offsets))
        t = ctx.timings()
        assert t["n_reads"] == sum(e["pos"].size for e in exported)
    with abi.Context(0) as ctx2:                       # host arrays -> add_sample: same result
        ctx2.shard_begin(S, ref)
        for s, e in enumerate(exported):
            if e["pos"].size:
                ctx2.shard_add_sample(s, e)
        ctx2.shard_mask_position(first)
        h2 = ctx2.shard_run()
        h3 = ctx2.shard_run()                          # repeated runs restore the qualities first
    for a in ("pos", "pop_mask", "ind_mask", "cov", "allele", "total"):
        assert np.array_equal(getattr(h, a), getattr(h2, a)), a
        assert np.array_equal(getattr(h, a), getattr(h3, a)), a


_FORM_KEYS = ("MSNV_PILEUP", "MSNV_MAX_READS", "MSNV_CHUNK_Q4", "MSNV_STAGES", "MSNV_CONSUMERS", "MSNV_PILEUP_CTAS")


@pytest.mark.parametrize("preset,scale,samples", [("c2", 0.003, 12), ("c4", 0.004, 4), ("c3", 0.0005, 12)])
def test_pileup_kernel_forms_agree(preset, scale, samples, built, monkeypatch):
    """The two forms of the pileup kernel (gather: counts in registers; scatter: shared-memory atomics) and their staging
    variants - items cut into several chunks, three stages, 256 consumers, deep items through the gather form's shared
    planes - give identical per-sample counts and identical hits on the same shard (ordinary depth with mate pairs, deep
    coverage with > 255 reads per tile, sparse multi-genome)."""
    from metasnv_b200 import abi
    desc = H.describe(preset, scale, samples)
    variants = [
        {},                                                                    # the library's own choice
        {"MSNV_PILEUP": "scatter"},
        {"MSNV_PILEUP": "gather"},
        {"MSNV_PILEUP": "gather", "MSNV_MAX_READS": "16", "MSNV_CHUNK_Q4": "1280"},          # narrow items in several chunks
        {"MSNV_PILEUP": "gather", "MSNV_STAGES": "3", "MSNV_PILEUP_CTAS": "2"},
        {"MSNV_PILEUP": "gather", "MSNV_CONSUMERS": "256"},
        {"MSNV_PILEUP": "scatter", "MSNV_MAX_READS": "16", "MSNV_CHUNK_Q4": "1280"},
    ]
    with abi.Context(0) as ctx:
        n_pos, first = ctx.shard_synth(desc)
        if first >= 0:
            ctx.shard_mask_position(first)
        S = desc["n_samples"]
        ref_hits = ref_counts = None
        for v in variants:
            for k in _FORM_KEYS:
                monkeypatch.delenv(k, raising=False)
            for k, val in v.items():
                monkeypatch.setenv(k, val)
            h = ctx.shard_run()
            hits = {a: np.array(getattr(h, a), copy=True) for a in ("pos", "pop_mask", "ind_mask", "cov", "allele", "total")}
            counts = [np.array(ctx.shard_counts(s, 0, n_pos), copy=True) for s in range(S)]
            if ref_hits is None:
                ref_hits, ref_counts = hits, counts
                assert sum(int(c.sum()) for c in counts) > 0
                continue
            for s, (a, b) in enumerate(zip(ref_counts, counts)):
                bad = np.argwhere(a != b)
                assert bad.size == 0, "%s: sample %d first mismatch at %s: %s against %s" % (v, s, bad[0], b[tuple(bad[0])], a[tuple(bad[0])])
            for a in ref_hits:
                assert np.array_equal(ref_hits[a], hits[a]), "%s: %s" % (v, a)


def test_full_size_shard_counts_recount_with_numpy(built):
    """BASELINE.json's headline shape at FULL size (5 Mb genome, 1000 samples at ~10x: 5e8 reads, 125 GB resident):
    the oracle cannot run at this size, so the device counts of whole samples are checked against the independent
    numpy recount of the same batches (tests/pileup_counts.py, itself pinned to the oracle on the CPU in
    tests/test_decode_cpu.py): one sample without overlapping mates, one with; plus size-independent properties:
    a second run is bit-identical, and every called position is covered where it says it is."""
    from metasnv_b200 import abi
    from pileup_counts import check_layout, numpy_counts
    desc = H.describe("c2", 1.0, 0)
    S = desc["n_samples"]
    assert S == 1000 and sum(desc["contig_len"]) == 5000000
    with abi.Context(0) as ctx:
        P, first = ctx.shard_synth(desc)
        ctx.shard_mask_position(first)
        h = ctx.shard_run()
        t = ctx.timings()
        assert t["n_reads"] >= 4.9e8 and t["n_items"] > 4.8e6
        picked = {}
        for s in range(S):
            z = ctx.sample_sizes(s)
            kind = "paired" if z.n_mated else "unpaired"
            if kind not in picked and z.n_reads:
                picked[kind] = s
            if len(picked) == 2:
                break
        assert set(picked) == {"paired", "unpaired"}
        for kind, s in picked.items():
            e = ctx.export_sample(s)
            assert (e["mate"] >= 0).any() == (kind == "paired")
            check_layout(e)
            want = numpy_counts(e, P)
            got = ctx.shard_counts(s, 0, P)
            bad = np.argwhere(got != want)
            assert bad.size == 0, "%s sample %d: first mismatch (pos, channel) %s: device %s, numpy %s" % (kind, s, bad[0], got[tuple(bad[0])], want[tuple(bad[0])])
            assert int(got.sum()) > 3e7
            # hits report this sample's coverage = counts of the four letters (+ N where the reference is N-like)
            cov = got[h.pos.astype(np.int64), :4].sum(axis=1)
            ref = ctx.export_ref(P)[h.pos.astype(np.int64)]
            acgt_ref = np.isin(ref, np.frombuffer(b"ACGTacgt", np.uint8))
            assert np.array_equal(h.cov[acgt_ref, s], cov[acgt_ref].astype(h.cov.dtype))
        h2 = ctx.shard_run()
        for a in ("pos", "pop_mask", "ind_mask", "cov", "allele", "total"):
            assert np.array_equal(getattr(h, a), getattr(h2, a)), a
        assert h.n_hits > 10000


def test_expand_kernel_builds_the_aligned_layout(built, tmp_path):
    """Reads handed over as BAM stores them (msnv_window_add_sample_raw): expand_kernel must build, byte for byte, the
    position-aligned arrays of msnv_decode_dump's host expansion (which tests/test_decode_cpu.py pins against the oracle):
    hand-written CIGAR cases and a synthetic set with indels, clips and N bases. Then the calls must be the same too."""
    import json
    from metasnv_b200 import abi
    from metasnv_b200.paths import bin_path
    from conftest import GOLDEN
    from pileup_counts import ARRAYS, RAW_ARRAYS
    tmp = str(tmp_path)
    bams = []
    for s in ("s1", "s2", "s4_ops", "s3_refskip", "s5_rules", "s6_leading_del"):
        out = os.path.join(tmp, s + ".bam")
        subprocess.run([bin_path("msnv_synth"), "--sam", os.path.join(GOLDEN, "hand", s + ".sam"), "--bam", out], check=True)
        bams.append(out)
    lst = os.path.join(tmp, "list")
    open(lst, "w").write("\n".join(bams) + "\n")
    data = os.path.join(tmp, "c1")
    H.synth(data, "c1", 0.05, 6)
    ctx = abi.Context(0)
    for i, (ref, l) in enumerate([(os.path.join(GOLDEN, "hand", "ref.fa"), lst), (os.path.join(data, "ref.fa"), os.path.join(data, "all_samples"))]):
        out = os.path.join(tmp, "dump%d" % i)
        os.makedirs(out)
        r = subprocess.run([bin_path("msnv_decode_dump"), ref, l, out], capture_output=True, text=True, env=dict(os.environ, MSNV_DUMP_RAW="1"))
        assert r.returncode == 0, r.stderr
        lay = json.load(open(os.path.join(out, "layout.json")))
        S, P = len(lay["samples"]), lay["n_positions"]
        refc = np.fromfile(os.path.join(out, "ref.bin"), np.uint8)
        host, raw = [], []
        for s, meta in enumerate(lay["samples"]):
            e = {k: np.fromfile(os.path.join(out, "s%d.%s.bin" % (s, k)), dt) for k, dt in ARRAYS}
            e["max_span"] = meta["max_span"]
            x = {k[4:] if k.startswith("raw_") and k != "raw_off" else k: np.fromfile(os.path.join(out, "s%d.%s.bin" % (s, k)), dt) for k, dt in RAW_ARRAYS}
            x["max_span"] = meta["max_span"]
            host.append(e); raw.append(x)
        # (a) device expansion == host layout
        ctx.shard_begin(S, refc)
        for s in range(S):
            if raw[s]["pos"].size:
                ctx.window_add_sample_raw(0, s, raw[s])
        n = 0
        for s in range(S):
            d = ctx.export_sample(s)
            for k, _ in ARRAYS:
                assert np.array_equal(d[k], host[s][k]), (i, s, k)
            n += d["pos"].size
        assert n > 20
        assert ctx.sample_sizes(0).n_aligned == int(host[0]["seg_len"].sum())
        h_raw = ctx.shard_run(min_coverage=2, calling_threshold=2)
        # (b) the same calls from either input form
        ctx.shard_begin(S, refc)
        for s in range(S):
            if host[s]["pos"].size:
                ctx.shard_add_sample(s, host[s])
        h_host = ctx.shard_run(min_coverage=2, calling_threshold=2)
        assert h_raw.n_hits == h_host.n_hits and h_raw.n_hits > 0
        for k in ("pos", "pop_mask", "ind_mask", "cov", "allele", "total"):
            assert np.array_equal(getattr(h_raw, k), getattr(h_host, k)), k
    assert ctx.expand_stats() == 0
    ctx.close()
