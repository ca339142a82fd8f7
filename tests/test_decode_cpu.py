"""CPU tests of the host BAM decoder (csrc/host/pileup_input.cc) and of the data layout of include/msnv.h:
`bin/msnv_decode_dump` writes the batches `snpCall` uploads, expanded on the host into the aligned layout; their structural
invariants are checked and a numpy recount of every sample (tests/pileup_counts.py) must equal the counts of the oracle's
mpileup text.
This covers, without a GPU, everything upstream of the kernels: mpileup's read filters, the depth cap, the overlap
pairing, the position-aligned segments with their zero padding, the reads carried from one position window to the
next, and the limits on read length and reference span."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import GOLDEN
from metasnv_b200 import abi
from metasnv_b200 import harness as H
from metasnv_b200.paths import bin_path
from pileup_counts import ARRAYS, check_layout, decode_dump, expand_raw, numpy_counts, oracle_counts

sys.path.insert(0, GOLDEN)
import edge_set  # noqa: E402
import span_set  # noqa: E402
from cases import oracle_mpileup  # noqa: E402
from edge_set import write_edge_set  # noqa: E402


def _compare(lay, samples, pile_path):
    P = lay["n_positions"]
    layout = [(c["name"], c["offset"], c["len"]) for c in lay["contigs"]]
    want = oracle_counts(pile_path, len(samples), layout, P)
    total = 0
    for s, e in enumerate(samples):
        if e["pos"].size:
            check_layout(e)
        got = numpy_counts(e, P)
        bad = np.argwhere(got != want[s])
        assert bad.size == 0, "sample %d first mismatch (pos, channel) %s: decoder+numpy %s, oracle %s" % (s, bad[0], got[tuple(bad[0])], want[s][tuple(bad[0])])
        total += int(got.sum())
    return total


def _touching(e, lo, hi):
    """Per read of batch e: does one of its segments cover a position of [lo, hi)?"""
    n = e["pos"].size
    if not n:
        return np.zeros(0, bool)
    sp, sl = e["seg_pos"].astype(np.int64), e["seg_len"].astype(np.int64)
    hit = (sp < hi) & (sp + sl > lo)
    return np.logical_or.reduceat(hit, e["seg_off"][:-1].astype(np.int64))


def _tiles_touched(e, tile):
    """{(tile, read)} of batch e: the read has a base in the tile."""
    sp, sl = e["seg_pos"].astype(np.int64), e["seg_len"].astype(np.int64)
    read = np.repeat(np.arange(e["pos"].size), np.diff(e["seg_off"].astype(np.int64)))
    return {(t, int(r)) for t_a, t_b, r in zip(sp // tile, (sp + sl - 1) // tile, read) for t in range(int(t_a), int(t_b) + 1)}


def _candidate_items(e, n_tiles, tile):
    """Per tile: (reads the index offers the tile - pos in [t0 - max_span + 1, t0 + TILE) - , reads that touch it)."""
    pos = e["pos"].astype(np.int64)
    t0 = np.arange(n_tiles, dtype=np.int64) * tile
    cand = np.searchsorted(pos, t0 + tile) - np.searchsorted(pos, t0 - int(e["max_span"]) + 1)
    touch = np.bincount([t for t, _ in _tiles_touched(e, tile)], minlength=n_tiles)
    return cand, touch


def _walk_skips(e, n_tiles, tile, back):
    """Tiles a read of batch e touches that the index's bitmap walk would skip with this `back`: mark_kernel sets a bit for
    the tile each read starts in, index_kernel searches a tile t only if a bit of [t - back, t] is set."""
    starts = np.zeros(n_tiles, bool)
    starts[e["pos"].astype(np.int64) // tile] = True
    return sorted({t for t, _ in _tiles_touched(e, tile) if not starts[max(t - back, 0):t + 1].any()})


def _at_k_lo(e, tile):
    """Tiles t touched by a read that starts exactly at t's k_lo = t * TILE - max_span + 1 (the first position the index's
    binary search takes)."""
    pos = e["pos"].astype(np.int64)
    return sorted({t for t, r in _tiles_touched(e, tile) if pos[r] == t * tile - int(e["max_span"]) + 1})


@pytest.mark.parametrize("preset,scale,samples", [("c1", 0.03, 8), ("c4", 0.002, 2), ("c5", 0.002, 4), ("c3", 0.0005, 6), ("edge", None, 310),
                                                  ("span", None, span_set.N_SAMPLES)])
def test_decoder_batches_recount_to_the_oracle_text(preset, scale, samples, datasets, tmp_path):
    """Synthetic sets, the edge set of tests/golden/edge_set.py (255 reads on one position in 270 samples, 250..260 reads
    on one tile, 1200x from one BAM, overlapping mates whose corrected qualities land on 12 and 13, reads of 4096 bases
    (one in 128 segments) at both ends of a contig whose length is not a multiple of 4), and the span set of
    tests/golden/span_set.py (reads of up to 32768 reference positions; there the BAM-shaped records are also expanded by the
Python restatement of expand_kernel)."""
    if preset == "edge":
        data = write_edge_set(str(tmp_path / "edge"))
    elif preset == "span":
        data = span_set.write_span_set(str(tmp_path / "span"))
    else:
        data = datasets(preset, scale, samples)
    lay, batches = decode_dump(os.path.join(data, "ref.fa"), os.path.join(data, "all_samples"), str(tmp_path / "dump"), raw=preset == "span")
    assert len(batches) == samples
    pile = oracle_mpileup(os.path.join(data, "ref.fa"), os.path.join(data, "all_samples"), str(tmp_path / "pile.txt"))
    assert _compare(lay, batches, pile) > 1000
    if preset == "span":
        # the BAM-shaped form, expanded as the device does, recounts to the same text
        assert _compare(lay, [dict(expand_raw(e), max_span=e["max_span"]) for e in batches], pile) > 1000
        # the set holds what it is meant to: spans up to the limit, items whose candidates mostly never touch their tile,
        # the depth cap with long reads buffered
        assert max(m["max_span"] for m in lay["samples"]) == span_set.MAX_SPAN
        cand, touch = _candidate_items(batches[1], lay["n_positions"] // lay["tile"], lay["tile"])
        assert ((cand > 255) & (touch * 10 <= cand)).any()
        assert lay["samples"][5]["dropped_by_cap"] > 0
        # ... and no column whose text snpCall would cut loses a base to the cut
        assert span_set.text_fits_snpcall(pile) == []
        assert lay["samples"][4]["pairs"] == 6
        # the index's reach is exact for every span of SPANS: its own sample (max_span == span) has a touched tile whose only
        # read starting in the bitmap walk's tiles [t - back, t] starts in t - back (so back - 1 would skip the tile and
        # lose its bases), and a touched tile whose read starts exactly at the tile's k_lo
        n_tiles, T = lay["n_positions"] // lay["tile"], lay["tile"]
        for s, e in enumerate(batches):
            back = (int(e["max_span"]) + T - 2) // T
            assert _walk_skips(e, n_tiles, T, back) == [], "sample %d: the walk must reach every touched tile" % s
        for span in span_set.SPANS:
            e = batches[span_set.ISOLATED + span_set.SPANS.index(span)]
            back = (span + T - 2) // T
            assert int(e["max_span"]) == span
            assert len(_walk_skips(e, n_tiles, T, back - 1)) >= 2, "span %d: back - 1 must skip a touched tile" % span
            assert len(_at_k_lo(e, T)) >= 2, "span %d: reads at k_lo" % span
    if preset == "c4":
        assert sum(m["dropped_by_cap"] for m in lay["samples"]) > 0, "the deep preset must exercise mpileup's depth cap"
    if preset == "c1":
        assert sum(m["pairs"] for m in lay["samples"]) > 0, "overlapping mates expected"
    if preset == "edge":
        assert max(m["max_span"] for m in lay["samples"]) == 4096 + 127 * 2, "the 128-segment read"
        assert lay["samples"][edge_set.MATES_SAMPLE]["pairs"] == 12


@pytest.mark.parametrize("sams,pile", [(("s1", "s2"), "expected.pileup"), (("s4_ops", "s1"), "expected_ops.pileup"),
                                       (("s3_refskip",), "expected_refskip.pileup"), (("s6_leading_del", "s1"), "expected_leading_del.pileup")])
def test_decoder_hand_written_cases(sams, pile, built, tmp_path):
    """The hand-written SAM files (indels, clips, =/X/P/N operations, overlapping mates with indels, filtered flags,
    orphans, N bases, CIGARs that open with a deletion) against the pinned pileup text."""
    tmp = str(tmp_path)
    bams = []
    for s in sams:
        out = os.path.join(tmp, s + ".bam")
        subprocess.run([bin_path("msnv_synth"), "--sam", os.path.join(GOLDEN, "hand", s + ".sam"), "--bam", out], check=True)
        bams.append(out)
    lst = os.path.join(tmp, "list")
    open(lst, "w").write("\n".join(bams) + "\n")
    lay, batches = decode_dump(os.path.join(GOLDEN, "hand", "ref.fa"), lst, os.path.join(tmp, "dump"))
    assert lay["tile"] == 1024 and lay["n_positions"] == 2048          # two 40-base contigs, one tile each
    assert _compare(lay, batches, os.path.join(GOLDEN, "hand", pile)) > 50


def test_bam_shaped_batches_expand_to_the_aligned_layout(built, tmp_path):
    """The decoder's batches - reads as BAM stores them, expanded on the device by expand_kernel - through two independent
    restatements of that expansion, msnv_decode_dump's host expansion and a plain-Python one, which must agree byte for
    byte: hand-written cases (indels, clips, =/X/P/N/H operations, N bases, one-base segments) and a small synthetic set."""
    tmp = str(tmp_path)
    bams = []
    for s in ("s1", "s2", "s4_ops", "s3_refskip", "s5_rules", "s6_leading_del"):
        out = os.path.join(tmp, s + ".bam")
        subprocess.run([bin_path("msnv_synth"), "--sam", os.path.join(GOLDEN, "hand", s + ".sam"), "--bam", out], check=True)
        bams.append(out)
    lst = os.path.join(tmp, "list")
    open(lst, "w").write("\n".join(bams) + "\n")
    sets = [(os.path.join(GOLDEN, "hand", "ref.fa"), lst)]
    data = os.path.join(tmp, "c1")
    H.synth(data, "c1", 0.004, 3)
    sets.append((os.path.join(data, "ref.fa"), os.path.join(data, "all_samples")))
    n_reads = 0
    for i, (ref, l) in enumerate(sets):
        lay, batches = decode_dump(ref, l, os.path.join(tmp, "dump%d" % i), raw=True)
        for e in batches:
            if not e["pos"].size:
                assert e["raw_pos"].size == 0
                continue
            x = expand_raw(e)
            for k, _ in ARRAYS:
                assert np.array_equal(x[k], e[k]), k
            n_reads += e["pos"].size
    assert n_reads > 1000


@pytest.mark.parametrize("what", ["bases", "segments"])
def test_decoder_refuses_reads_above_the_length_limits(what, built, tmp_path):
    """A read of 4097 bases, or of 129 aligned segments, is beyond MSNV_MAX_READ_BASES / MSNV_MAX_READ_SEGMENTS (the pileup
    kernel's smallest stage is sized for one read at these limits): the decoder stops with an error naming the read instead
    of handing it on. One read exactly at both limits (tests/golden/edge_set.py) decodes."""
    if what == "bases":
        cigar, n = "4097M", 4097
    else:
        cigar, n = "1M1D" * 128 + "1M", 129
    sam = str(tmp_path / "big.sam")
    open(sam, "w").write("@HD\tVN:1.6\tSO:coordinate\n@SQ\tSN:c\tLN:5000\n"
                         "ok\t0\tc\t1\t60\t10M\t*\t0\t0\t%s\t%s\n" % ("A" * 10, "I" * 10) +
                         "big\t0\tc\t5\t60\t%s\t*\t0\t0\t%s\t%s\n" % (cigar, "C" * n, "I" * n))
    bam = str(tmp_path / "big.bam")
    subprocess.run([bin_path("msnv_synth"), "--sam", sam, "--bam", bam], check=True)
    open(str(tmp_path / "list"), "w").write(bam + "\n")
    open(str(tmp_path / "ref.fa"), "w").write(">c\n" + "ACGT" * 1250 + "\n")
    os.makedirs(str(tmp_path / "dump"))
    r = subprocess.run([bin_path("msnv_decode_dump"), str(tmp_path / "ref.fa"), str(tmp_path / "list"), str(tmp_path / "dump")],
                       capture_output=True, text=True)
    assert r.returncode != 0
    assert "read big exceeds the supported length (4096 bases / 128 aligned segments)" in r.stderr, r.stderr


WINDOW_TILES = [1, 3, 7]


@pytest.fixture(scope="module")
def span_data(built, tmp_path_factory):
    """The span set, the decoder's whole-shard batches of it (expanded on the host) and the oracle's counts."""
    d = str(tmp_path_factory.mktemp("span"))
    data = span_set.write_span_set(os.path.join(d, "set"))
    lay, whole = decode_dump(os.path.join(data, "ref.fa"), os.path.join(data, "all_samples"), os.path.join(d, "dump"))
    layout = [(c["name"], c["offset"], c["len"]) for c in lay["contigs"]]
    want = oracle_counts(span_set.oracle_pileup(data), len(whole), layout, lay["n_positions"])
    return data, lay, whole, want


def _read_keys(e, idx):
    """Hashable contents of reads idx of batch e (position, segments, bases, qualities)."""
    so, qo = e["seg_off"].astype(np.int64), e["q4_off"].astype(np.int64)
    return [(int(e["pos"][i]), e["seg_pos"][so[i]:so[i + 1]].tobytes(), e["seg_len"][so[i]:so[i + 1]].tobytes(),
             e["seq2"][qo[i]:qo[i + 1]].tobytes(), e["qual"][4 * qo[i]:4 * qo[i + 1]].tobytes()) for i in idx]


@pytest.mark.parametrize("win_tiles", WINDOW_TILES)
def test_windowed_decoder_batches_recount_to_the_oracle(win_tiles, span_data, tmp_path):
    """snpCall decodes a shard window by window, and SampleDecoder::window carries the reads of the previous window that
    reach the next one. On the span set cut into windows of 1, 3 and 7 tiles (a read of span 32768 crosses up to 33 of
    them), each window's batch, expanded on the host and by the Python restatement, recounts to the oracle's counts over
    that window's positions, and holds every read that abi.window_slice offers the window and that touches it."""
    from collections import Counter
    data, lay0, whole, want = span_data
    T, P = lay0["tile"], lay0["n_positions"]
    assert P // T == span_set.N_TILES and span_set.N_TILES % win_tiles == 0
    lay, _, wins = decode_dump(os.path.join(data, "ref.fa"), os.path.join(data, "all_samples"), str(tmp_path / "dump"), raw=True,
                           windows=span_set.N_TILES // win_tiles)
    assert [(w["lo"], w["hi"]) for w in lay["windows"]] == [(lo, lo + win_tiles * T) for lo in range(0, P, win_tiles * T)]
    carried = 0
    for w, batches in zip(lay["windows"], wins):
        lo, hi = w["lo"], w["hi"]
        for s, e in enumerate(batches):
            if e["pos"].size:
                check_layout(e)
            got = numpy_counts(e, P)[lo:hi]
            bad = np.argwhere(got != want[s, lo:hi])
            assert bad.size == 0, "window %d..%d, sample %d, first mismatch (pos, channel) %s: decoder+numpy %s, oracle %s" % (
                lo, hi, s, bad[0] + [lo, 0], got[tuple(bad[0])], want[s, lo + bad[0][0], bad[0][1]])
            if e["raw_pos"].size:
                x = dict(expand_raw(e), max_span=e["raw_max_span"])
                got = numpy_counts(x, P)[lo:hi]
                bad = np.argwhere(got != want[s, lo:hi])
                assert bad.size == 0, "BAM-shaped form: window %d..%d, sample %d, first mismatch (pos, channel) %s" % (lo, hi, s, bad[0] + [lo, 0])
            sl = abi.window_slice(whole[s], lo, hi) if whole[s]["pos"].size else None
            if sl is None:
                continue
            need = Counter(_read_keys(sl, np.nonzero(_touching(sl, lo, hi))[0]))
            have = Counter(_read_keys(e, range(e["pos"].size)))
            assert not need - have, "window %d..%d, sample %d: %d reads reach the window but are not in its batch" % (lo, hi, s, sum((need - have).values()))
            carried += int((e["pos"] < lo).sum())
    assert carried > 100


def test_decoder_refuses_reads_above_the_span_limit(built, tmp_path):
    """A read of 32769 reference positions (50M 32669N 50M: 100 bases) is beyond MSNV_MAX_READ_SPAN: every item within the
    span is a candidate for the read, so the index and the pileup kernel bound it. The decoder stops with an error naming
    the BAM and the read instead of handing it on; reads of span 32768 (the span set) decode."""
    data = span_set.write_span_set(str(tmp_path / "span"))
    os.makedirs(str(tmp_path / "dump"))
    r = subprocess.run([bin_path("msnv_decode_dump"), os.path.join(data, "ref.fa"), os.path.join(data, "over", "all_samples"),
                        str(tmp_path / "dump")], capture_output=True, text=True)
    assert r.returncode != 0
    assert os.path.join(data, "over", "over.bam") + ": read too_long spans 32769 reference positions, more than the supported 32768" in r.stderr, r.stderr
