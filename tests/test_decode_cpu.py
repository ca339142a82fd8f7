"""CPU tests of the host BAM decoder (csrc/host/pileup_input.cc) and of the data layout of include/msnv.h:
`bin/msnv_decode_dump` writes the batches `snpCall` would upload; their structural invariants are checked and a
numpy recount of every sample (tests/pileup_counts.py) must equal the counts of the oracle's mpileup text.
This covers, without a GPU, everything upstream of the kernels: mpileup's read filters, the depth cap, the overlap
pairing, the position-aligned segments with their zero padding."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import GOLDEN
from metasnv_b200 import harness as H
from metasnv_b200.paths import bin_path
from pileup_counts import ARRAYS, RAW_ARRAYS, check_layout, expand_raw, numpy_counts, oracle_counts

sys.path.insert(0, GOLDEN)
import edge_set  # noqa: E402
from edge_set import write_edge_set  # noqa: E402


def _decode(ref, lst, out, raw=False):
    os.makedirs(out, exist_ok=True)
    env = dict(os.environ, MSNV_DUMP_RAW="1") if raw else None
    r = subprocess.run([bin_path("msnv_decode_dump"), ref, lst, out], capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr
    lay = json.load(open(os.path.join(out, "layout.json")))
    samples = []
    for s, meta in enumerate(lay["samples"]):
        e = {k: np.fromfile(os.path.join(out, "s%d.%s.bin" % (s, k)), dt) for k, dt in ARRAYS}
        e["max_span"] = meta["max_span"]
        if raw:
            for k, dt in RAW_ARRAYS:
                e[k] = np.fromfile(os.path.join(out, "s%d.%s.bin" % (s, k)), dt)
        assert e["pos"].size == meta["n_reads"] and e["seg_pos"].size == meta["n_segs"] and e["seq2"].size == meta["n_q4"]
        samples.append(e)
    return lay, samples


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


@pytest.mark.parametrize("preset,scale,samples", [("c1", 0.03, 8), ("c4", 0.002, 2), ("c5", 0.002, 4), ("c3", 0.0005, 6), ("edge", None, 310)])
def test_decoder_batches_recount_to_the_oracle_text(preset, scale, samples, datasets, tmp_path):
    """Synthetic sets, and the edge set of tests/golden/edge_set.py: 255 reads on one position in 270 samples, 250..260 reads
    on one tile, 1200x from one BAM, overlapping mates whose corrected qualities land on 12 and 13, reads of 4096 bases
    (one in 128 segments) at both ends of a contig whose length is not a multiple of 4."""
    if preset == "edge":
        data = write_edge_set(str(tmp_path / "edge"))
    else:
        data = datasets(preset, scale, samples)
    lay, batches = _decode(os.path.join(data, "ref.fa"), os.path.join(data, "all_samples"), str(tmp_path / "dump"))
    assert len(batches) == samples
    pile = str(tmp_path / "pile.txt")
    with open(pile, "wb") as f:
        subprocess.run([H.oracle_bin("mpileup_oracle"), "mpileup", "-f", os.path.join(data, "ref.fa"), "-B", "-b",
                        os.path.join(data, "all_samples")], stdout=f, check=True)
    assert _compare(lay, batches, pile) > 1000
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
    lay, batches = _decode(os.path.join(GOLDEN, "hand", "ref.fa"), lst, os.path.join(tmp, "dump"))
    assert lay["tile"] == 1024 and lay["n_positions"] == 2048          # two 40-base contigs, one tile each
    assert _compare(lay, batches, os.path.join(GOLDEN, "hand", pile)) > 50


def test_bam_shaped_batches_expand_to_the_aligned_layout(built, tmp_path):
    """The decoder's other output form - reads as BAM stores them, expanded on the device by expand_kernel - against the
    aligned layout the decoder builds itself, through a plain-Python restatement of the expansion: hand-written cases
    (indels, clips, =/X/P/N/H operations, N bases, one-base segments) and a small synthetic set."""
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
        lay, batches = _decode(ref, l, os.path.join(tmp, "dump%d" % i), raw=True)
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
