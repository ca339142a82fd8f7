"""Reads of long reference span on the GPU (B200 only: `pytest -m gpu`), on the span set of tests/golden/span_set.py: reads
of 4097..32768 positions (N and D) whose ends lie on, next to and just before tile boundaries, skips over whole tiles,
leading skips and deletions of 1..20 kb, items with more than 255 candidate reads of which a few touch the tile, mates
with gaps, the depth cap with long reads buffered, and the span limit (32768).
The index (both search paths), both pileup forms, the host- and device-built layouts, windows of one and three tiles and
ranges of tiles are compared with the oracle: per-sample per-position counts with the counts of its mpileup text, calls
byte for byte with `mpileup_oracle | snpCall`."""
import json
import os
import sys

import numpy as np
import pytest

from conftest import GOLDEN
from metasnv_b200 import abi
from metasnv_b200 import harness as H
from pileup_counts import decode_dump, first_difference, oracle_counts

sys.path.insert(0, GOLDEN)
import span_set as SP  # noqa: E402
from cases import file_digest  # noqa: E402

pytestmark = pytest.mark.gpu


class Span:
    def __init__(self, d):
        self.dir = d
        self.bed = os.path.join(d, "span.bed")
        self._want = None
        self.oracle = {}

    def want_counts(self, layout, P):
        """The oracle's [S][P][5] counts of the whole set (shard layout of the product)."""
        if self._want is None:
            self._want = oracle_counts(SP.oracle_pileup(self.dir), SP.N_SAMPLES, layout, P)
        return self._want

    def oracle_calls(self, opts):
        """Prefix of the oracle's .called / .indiv for one SPAN_CALLS entry, checked against the pinned digests
        (tests/golden/make_oracle_digests.py)."""
        key = SP.span_key(opts)
        if key not in self.oracle:
            prefix = os.path.join(self.dir, "oracle_%d" % len(self.oracle))
            rc, err = SP.run_oracle_calls(self.dir, opts, prefix)
            assert rc == 0, err
            want = json.load(open(os.path.join(GOLDEN, "oracle_digests.json")))
            for ext in (".called", ".indiv"):
                assert file_digest(prefix + ext) == want[key + ext], "oracle output %s%s differs from the pinned one" % (key, ext)
            self.oracle[key] = prefix
        return self.oracle[key]


@pytest.fixture(scope="module")
def span(built, tmp_path_factory):
    return Span(SP.write_span_set(str(tmp_path_factory.mktemp("span") / "set")))


def _same(a, b):
    d = H.first_diff(a, b)
    assert not d, "%s vs %s: %s" % (a, b, d)


# the library's choice; both pileup forms, also with the smallest stages (16 reads, one 4096-base read of quads); both
# search paths of the index; 256 consumer threads
COUNT_FORMS = [{}, {"MSNV_PILEUP": "scatter"}, {"MSNV_PILEUP": "gather"},
               {"MSNV_PILEUP": "scatter", "MSNV_MAX_READS": "16", "MSNV_CHUNK_Q4": "1280"},
               {"MSNV_PILEUP": "gather", "MSNV_MAX_READS": "16", "MSNV_CHUNK_Q4": "1280"},
               {"MSNV_INDEX_BITMAP": "0"}, {"MSNV_INDEX_BITMAP": "1"}, {"MSNV_CONSUMERS": "256"}]


@pytest.mark.parametrize("env", COUNT_FORMS, ids=lambda e: "-".join("%s=%s" % kv for kv in e.items()) or "library")
def test_span_counts_match_oracle_text(env, span, tmp_path):
    out = str(tmp_path / "gpu")
    dump = out + ".counts"
    rc, err = H.run_product_snpcall(span.dir, out, env=dict(os.environ, MSNV_DUMP_COUNTS=dump, **env))
    assert rc == 0, err
    lay = [l.rstrip("\n").split("\t") for l in open(dump + ".layout")]
    S, P = int(lay[0][0]), int(lay[0][1])
    layout = [(n, int(o), int(l)) for n, o, l in lay[1:]]
    got = np.fromfile(dump, np.uint16).reshape(S, P, 5)
    assert S == SP.N_SAMPLES and P == SP.N_TILES * abi.TILE
    want = span.want_counts(layout, P)
    d = first_difference(want, got, layout)
    assert not d, d


# (snpCall options, form): every SPAN_CALLS entry with the library's choice of pileup form and with both forced forms, in
# windows of one tile (a read of span 32768 crosses 33 of them) and of three tiles, and in ranges of tiles (a tile budget
# of 24 count-plane slots: a tile holds at most 11 items)
FORM_ENV = {"library": {}, "scatter": {"MSNV_PILEUP": "scatter"}, "gather": {"MSNV_PILEUP": "gather"},
            "windows1": {"MSNV_WINDOWS": str(SP.N_TILES)}, "windows3": {"MSNV_WINDOWS": str(SP.N_TILES // 3)},
            "ranges": {"MSNV_TILE_BUDGET_MB": "0.28125"}}
CALL_RUNS = [(o, f) for o in SP.SPAN_CALLS for f in FORM_ENV]


@pytest.mark.parametrize("opts,form", CALL_RUNS, ids=["%s-%s" % (SP.span_key(o)[5:], f) for o, f in CALL_RUNS])
def test_span_calls_match_oracle(opts, form, span, tmp_path):
    o = span.oracle_calls(opts)
    g = str(tmp_path / "gpu")
    kw = {k: v for k, v in opts.items() if k != "bed"}
    env = dict(os.environ, MSNV_PERF_JSON=g + ".perf", **FORM_ENV[form])
    rc, err = H.run_product_snpcall(span.dir, g, bed=span.bed if opts.get("bed") else None, env=env, **kw)
    assert rc == 0, err
    for ext in (".called", ".indiv"):
        _same(o + ext, g + ext)
    assert os.path.getsize(o + ".called") > 0
    perf = json.loads(open(g + ".perf").readline())
    n_windows = {"windows1": SP.N_TILES, "windows3": SP.N_TILES // 3}.get(form, 1)
    if opts.get("bed"):                                # (the shard holds the tiles of the BED's contigs only)
        assert (perf["windows"] > 1) == (n_windows > 1)
    else:
        assert perf["windows"] == n_windows
    if form == "ranges":
        assert perf["ranges"] > perf["windows"], "the tile budget should split the run into several ranges of tiles"
    else:
        assert perf["ranges"] == perf["windows"]


@pytest.fixture(scope="module")
def span_batches(span, tmp_path_factory):
    """The decoder's whole-shard batches of the span set and its shard reference."""
    d = str(tmp_path_factory.mktemp("span_dump"))
    lay, whole = decode_dump(os.path.join(span.dir, "ref.fa"), os.path.join(span.dir, "all_samples"), d)
    return lay, whole, np.fromfile(os.path.join(d, "ref.bin"), np.uint8)


@pytest.mark.parametrize("win_tiles", [1, 3])
def test_abi_windows_count_like_the_oracle(win_tiles, span, span_batches):
    """The C ABI's position windows: each window gets, per sample, the reads abi.window_slice cuts for it, uploaded into
    alternating slots one window ahead of the run; after each run, msnv_shard_counts over the window equals the oracle's
    counts there (snpCall's counts hook only sees one whole-shard window)."""
    lay, whole, ref = span_batches
    T, P = abi.TILE, lay["n_positions"]
    layout = [(c["name"], c["offset"], c["len"]) for c in lay["contigs"]]
    want = span.want_counts(layout, P)
    wins = [(lo, min(lo + win_tiles * T, P)) for lo in range(0, P, win_tiles * T)]
    with abi.Context(0) as ctx:
        ctx.shard_begin(SP.N_SAMPLES, ref)

        def upload(k):
            lo, hi = wins[k]
            ctx.window_begin(k & 1, lo, hi)
            for s, e in enumerate(whole):
                w = abi.window_slice(e, lo, hi) if e["pos"].size else None
                if w is not None:
                    ctx.window_add_sample(k & 1, s, w)
        upload(0)
        for k, (lo, hi) in enumerate(wins):
            if k + 1 < len(wins):
                upload(k + 1)
            ctx.window_run(k & 1)
            got = np.stack([ctx.shard_counts(s, lo, hi - lo) for s in range(SP.N_SAMPLES)])
            d = first_difference(want[:, lo:hi], got, [(n, o - lo, ln) for n, o, ln in layout if o < hi])
            assert not d, "window %d..%d: %s" % (lo, hi, d)


def test_snpcall_refuses_a_read_above_the_span_limit(span, tmp_path):
    """snpCall on a BAM holding a read of span 32769 stops with the decoder's message naming the BAM and the read."""
    over = os.path.join(span.dir, "over", "all_samples")
    rc, err = H.run_product_snpcall(span.dir, str(tmp_path / "gpu"), all_samples=over)
    assert rc != 0
    assert "over.bam: read too_long spans 32769 reference positions, more than the supported 32768" in err, err


def test_window_add_sample_span_limit(span, span_batches):
    """msnv_window_add_sample refuses a batch whose max_span is 32769 with MSNV_E_LIMIT; 32768 is accepted and the
    context stays usable: the run's counts equal the oracle's."""
    lay, whole, ref = span_batches
    P = lay["n_positions"]
    layout = [(c["name"], c["offset"], c["len"]) for c in lay["contigs"]]
    e = whole[0]
    assert e["max_span"] == SP.MAX_SPAN
    with abi.Context(0) as ctx:
        ctx.shard_begin(SP.N_SAMPLES, ref)
        with pytest.raises(abi.MsnvError, match=r"\(-4\).*reference span 32769 exceeds the limit of 32768"):
            ctx.shard_add_sample(0, dict(e, max_span=SP.MAX_SPAN + 1))
        for s, b in enumerate(whole):
            if b["pos"].size:
                ctx.shard_add_sample(s, b)
        ctx.shard_run()
        got = np.stack([ctx.shard_counts(s, 0, P) for s in range(SP.N_SAMPLES)])
    d = first_difference(span.want_counts(layout, P), got, layout)
    assert not d, d
