"""A small, deterministic data set of SAM-built BAMs aimed at the arithmetic boundaries of the pileup and call kernels
(byte-lane counters, the narrow/wide item switch, the 16-bit partial sums, the HI_THR threshold test, the fp64 fraction
test, the read-length limits) and at qaCompute's histogram above 1023. Needs neither pytest nor a GPU:

    from edge_set import write_edge_set
    write_edge_set(out_dir)          # ref.fa, sam/*.sam, bam/*.bam, all_samples, narrow_samples, stacks.bed

What each part pins (positions are 0-based contig coordinates; every contig starts on a tile, so a position's residue
mod 4 is its byte lane):
  deep, tile 0   samples 0..269 each hold exactly 255 reads over X1 (X1 % 4 == 0) with a non-reference G: the population
                 sum at X1 is 68 850 (> 65 535) and more than 256 narrow items of one tile carry 255 in one lane. Even
                 samples cover X1 alone (neighbour lanes empty), odd ones X1..X1+3 (255 T, 254 A + one base below Q13,
                 255 of the reference letter). Samples 270..309 add three reference bases each.
  deep, tile 1   samples 0..10 hold 250..260 reads at X2, all A: the narrow/wide switch on both sides.
  deep, tile 2   sample 20 (255 reads: narrow) and sample 21 (300 reads: wide) carry stacks of 127..300 bases of one
                 letter under an upper-case reference, N, R, Y, a lower-case base (its own allele and another) and the
                 expected letter itself; the rest of each read is a second non-reference letter.
  deep, tile 3   coverage / allele pairs on either side of an fp32-fp64 disagreement of cov*p, and overlapping mate
                 pairs whose corrected qualities land on 12 and 13.
  deep, tile 4   sample 0 reaches coverage 1200 (qaCompute -c above 1023).
  long           a 4096M read from position 1, a 4096M read ending on the last base of a contig of length 6143, a read of
                 4096 bases in 128 M segments (each starting at 3 mod 4, lengths 2 mod 4), short reads at both ends.
  bare           a contig without reads.
narrow_samples lists the samples without a wide item: as a shard of their own, its largest items hold exactly 255 reads.
"""
import os
import random
import subprocess

N_SAMPLES = 310
DEEP_LEN, LONG_LEN, BARE_LEN = 5120, 6143, 77
CONTIGS = [("deep", DEEP_LEN), ("long", LONG_LEN), ("bare", BARE_LEN)]

X1 = 64                                   # tile 0
BLOCK = range(0, 270)
X2 = 1024 + 128                           # tile 1
SWEEP = range(0, 11)
STACK_COUNTS_NARROW = [127, 128, 129, 200, 254, 255]
STACK_COUNTS_WIDE = [127, 128, 129, 200, 254, 255, 256, 257, 300]
NARROW_SAMPLE, NARROW_AT, NARROW_READS = 20, 2048 + 256, 255
WIDE_SAMPLE, WIDE_AT, WIDE_READS = 21, 2048 + 320, 300
# reference character, stacked letter, the letter of the other reads (None: keep the random reference base)
STACK_KINDS = [(None, None, None), ("N", "A", "C"), ("R", "A", "G"), ("Y", "C", "T"), ("c", "C", "A"), ("g", "T", "A"),
               ("T", "T", "A")]
# (sample, position, coverage, alleles, p): fp64 and fp32 cov*p fall on different sides of the allele count
FRACTION = [(30, 3072 + 16, 100, 7, 0.07), (31, 3072 + 20, 200, 14, 0.07), (32, 3072 + 24, 50, 15, 0.3)]
MATES_SAMPLE, MATES_AT = 33, 3072 + 100
DEEP_COV_SAMPLE, DEEP_COV_AT, DEEP_COV_READS = 0, 4096 + 300, 1200
SEGMENTS_AT = 999                         # 0-based, 3 mod 4

# snpCall options the edge set is called with (tests/test_gpu_kernel_edges.py, make_oracle_digests.py); "bed": restricted
# to stacks.bed
EDGE_CALLS = ([{}] + [dict(t=t, p=p) for t in (127, 128, 129, 200, 255, 256, 257, 300) for p in (0.01, 1.0)]
              + [dict(t=1, p=0.07), dict(t=1, p=0.3), dict(c=1, t=0, bed=True)])


# ... and the narrow_samples shard
NARROW_CALLS = [{}, dict(t=255, p=1.0), dict(t=128, p=1.0)]


def edge_key(opts, samples="all_samples"):
    """Name of one EDGE_CALLS / NARROW_CALLS entry in oracle_digests.json."""
    return ("edge/" if samples == "all_samples" else "edge-narrow/") + ("-".join("%s%s" % kv for kv in sorted(opts.items())) or "defaults")


def fraction_pairs_straddle():
    """Every FRACTION entry: the allele count passes `n >= cov*p` in exactly one of fp64 and fp32, and both directions occur."""
    import numpy as np
    sides = set()
    for _, _, cov, n, p in FRACTION:
        f64, f32 = n >= cov * p, n >= float(np.float32(cov) * np.float32(p))
        assert f64 != f32, (cov, n, p)
        sides.add(f64)
    assert sides == {True, False}
    return True


def _other(b, k=1):
    return "ACGT"[("ACGT".index(b.upper()) + k) % 4]


def _ref(rng):
    ref = {name: [rng.choice("ACGT") for _ in range(n)] for name, n in CONTIGS}
    d = ref["deep"]
    d[X1:X1 + 4] = list("ACGT")
    d[X2] = "C"
    for at, counts in ((NARROW_AT, STACK_COUNTS_NARROW), (WIDE_AT, STACK_COUNTS_WIDE)):
        for k, (rc, _, _) in enumerate(STACK_KINDS):
            if rc:
                for i in range(len(counts)):
                    d[at + k * len(counts) + i] = rc
    return ref


def _sam_line(name, flag, ctg, pos0, cigar, seq, qual, mate=None):
    rnext, pnext, tlen = ("=", mate[0] + 1, mate[1]) if mate else ("*", 0, 0)
    return "%s\t%d\t%s\t%d\t60\t%s\t%s\t%s\t%s\t%s\t%s\n" % (name, flag, ctg, pos0 + 1, cigar, rnext, pnext, tlen, seq, qual)


def _reads(ref, rng):
    """{sample: [(contig index, pos0, SAM line)]}"""
    out = {s: [] for s in range(N_SAMPLES)}
    ci = {name: k for k, (name, _) in enumerate(CONTIGS)}
    d = ref["deep"]

    def add(s, ctg, pos0, line):
        out[s].append((ci[ctg], pos0, line))

    # tile 0: 255 G at X1 in each of 270 samples
    for s in BLOCK:
        for j in range(255):
            if s % 2 == 0:
                add(s, "deep", X1, _sam_line("b%d" % j, 0, "deep", X1, "1M", "G", "I"))
            else:
                add(s, "deep", X1, _sam_line("b%d" % j, 0, "deep", X1, "4M", "GTA" + d[X1 + 3], "II" + ("#" if j == 7 else "I") + "I"))
    for s in range(BLOCK.stop, N_SAMPLES):
        for j in range(3):
            add(s, "deep", X1, _sam_line("e%d" % j, 0, "deep", X1, "1M", d[X1], "I"))
    # tile 1: 250..260 reads on one position
    for s in SWEEP:
        for j in range(250 + s):
            add(s, "deep", X2, _sam_line("w%d" % j, 0, "deep", X2, "1M", "A", "I"))
    for j in range(5):
        add(SWEEP.stop, "deep", X2, _sam_line("w%d" % j, 0, "deep", X2, "1M", d[X2], "I"))
    # tile 2: threshold stacks in a narrow and a wide item
    for s, at, n_reads, counts in ((NARROW_SAMPLE, NARROW_AT, NARROW_READS, STACK_COUNTS_NARROW),
                                   (WIDE_SAMPLE, WIDE_AT, WIDE_READS, STACK_COUNTS_WIDE)):
        cols = []
        for k, (rc, stack, filler) in enumerate(STACK_KINDS):
            for i, n in enumerate(counts):
                r = d[at + k * len(counts) + i]
                x, y = (stack, filler) if rc else (_other(r, 1 + i % 3), _other(r, 1 + (i + 1) % 3))
                cols.append((x, y, n))
        for j in range(n_reads):
            seq = "".join(x if j < n else y for x, y, n in cols)
            add(s, "deep", at, _sam_line("t%d" % j, 0, "deep", at, "%dM" % len(seq), seq, "I" * len(seq)))
    # tile 3: fraction boundaries
    for s, pos, cov, n, _ in FRACTION:
        for j in range(cov):
            add(s, "deep", pos, _sam_line("f%d" % j, 0, "deep", pos, "1M", _other(d[pos]) if j < n else d[pos], "I"))
    # tile 3: overlapping mates (10M + 10M, the later mate 4 bases further: 6 positions in both), overlap qualities
    # (earlier, later, same base): int(0.8*q) of the better read is 12 or 13, sums of equal bases are 12 or 13
    cases = [(6, 7, True), (6, 6, True), (16, 10, False), (17, 10, False), (10, 17, False), (10, 16, False), (16, 16, False),
             (17, 17, False), (13, 0, False), (12, 1, True), (40, 16, False), (17, 40, False)]
    for k, (qa, qb, same) in enumerate(cases):
        pa = MATES_AT + 12 * k
        pb = pa + 4
        sa = "".join(d[pa + i] for i in range(10))
        sb = "".join(d[pb + i] if (same or i >= 6) else _other(d[pb + i]) for i in range(10))
        qa_s = "".join(chr(33 + q) for q in [12, 13, 12, 13] + [qa] * 6)
        qb_s = "".join(chr(33 + q) for q in [qb] * 6 + [13, 12, 13, 12])
        add(MATES_SAMPLE, "deep", pa, _sam_line("m%d" % k, 99, "deep", pa, "10M", sa, qa_s, (pb, 14)))
        add(MATES_SAMPLE, "deep", pb, _sam_line("m%d" % k, 147, "deep", pb, "10M", sb, qb_s, (pa, -14)))
    # tile 4: coverage 1200 from one BAM
    for j in range(DEEP_COV_READS):
        pos = DEEP_COV_AT + j % 60
        seq = "".join(d[pos + i] if i != j % 53 else _other(d[pos + i]) for i in range(60))
        add(DEEP_COV_SAMPLE, "deep", pos, _sam_line("c%d" % j, 0, "deep", pos, "60M", seq, "I" * 60))
    # long contig: 4096-base reads, 128 segments, both contig ends
    g = ref["long"]

    def noisy(pos, n):
        return "".join(g[pos + i] if rng.random() > 0.05 else _other(g[pos + i], rng.randint(1, 3)) for i in range(n))

    def quals(n):
        return "".join(rng.choice("II-.") for _ in range(n))

    add(40, "long", 0, _sam_line("L0", 0, "long", 0, "4096M", noisy(0, 4096), quals(4096)))
    add(40, "long", LONG_LEN - 4, _sam_line("L1", 0, "long", LONG_LEN - 4, "4M", noisy(LONG_LEN - 4, 4), "IIII"))
    add(41, "long", LONG_LEN - 4096, _sam_line("L2", 0, "long", LONG_LEN - 4096, "4096M", noisy(LONG_LEN - 4096, 4096), quals(4096)))
    lens = [30 if k % 2 == 0 else 34 for k in range(128)]
    assert sum(lens) == 4096 and all(n % 4 == 2 for n in lens)
    cig, seq, pos = [], [], SEGMENTS_AT
    for k, n in enumerate(lens):
        assert pos % 4 == 3
        cig.append("%dM" % n)
        seq.append(noisy(pos, n))
        pos += n
        if k < 127:
            cig.append("2D")
            pos += 2
    assert pos <= LONG_LEN
    add(42, "long", SEGMENTS_AT, _sam_line("L3", 0, "long", SEGMENTS_AT, "".join(cig), "".join(seq), quals(4096)))
    for pos, n in ((0, 1), (0, 9), (LONG_LEN - 7, 7), (LONG_LEN - 3, 3), (LONG_LEN - 1, 1)):
        add(43, "long", pos, _sam_line("L%d_%d" % (pos, n), 0, "long", pos, "%dM" % n, noisy(pos, n), "I" * n))
    return out


def _reads_per_tile(reads, tile=1024):
    """{(contig index, tile): reads that touch it} of one sample's [(contig index, pos0, SAM line)]."""
    import re
    n = {}
    for c, pos, line in reads:
        span = sum(int(k) for k, op in re.findall(r"(\d+)([MDN=X])", line.split("\t")[5]))
        for t in range(pos // tile, (pos + span - 1) // tile + 1):
            n[(c, t)] = n.get((c, t), 0) + 1
    return n


def stack_intervals():
    """(contig, begin, end) of the stacked positions (0-based, half open)."""
    iv = [("deep", X1, X1 + 4), ("deep", X2, X2 + 1),
          ("deep", NARROW_AT, NARROW_AT + len(STACK_KINDS) * len(STACK_COUNTS_NARROW)),
          ("deep", WIDE_AT, WIDE_AT + len(STACK_KINDS) * len(STACK_COUNTS_WIDE))]
    return iv + [("deep", pos, pos + 1) for _, pos, _, _, _ in FRACTION]


def oracle_pileup(d, bed=False, samples="all_samples"):
    """The oracle's mpileup text of the set in d (or of its stacks.bed; samples: all_samples or narrow_samples), written
    once into d."""
    from cases import oracle_mpileup
    path = os.path.join(d, "pile_%s%s.txt" % (samples, "_bed" if bed else ""))
    if not os.path.exists(path):
        oracle_mpileup(os.path.join(d, "ref.fa"), os.path.join(d, samples), path, os.path.join(d, "stacks.bed") if bed else None)
    return path


def run_oracle_calls(d, opts, prefix, samples="all_samples"):
    """`mpileup_oracle | oracle snpCall` with one EDGE_CALLS entry -> prefix.called / prefix.indiv; returns (rc, stderr)."""
    from metasnv_b200 import harness as H
    kw = {k: v for k, v in opts.items() if k != "bed"}
    with open(oracle_pileup(d, opts.get("bed", False), samples), "rb") as fin, open(prefix + ".called", "wb") as fout:
        r = subprocess.run([H.oracle_snpcall()] + H.snpcall_args(os.path.join(d, "ref.fa"), prefix + ".indiv", **kw),
                           stdin=fin, stdout=fout, stderr=subprocess.PIPE)
    return r.returncode, r.stderr.decode(errors="replace")


def write_edge_set(out_dir, sam_to_bam=None):
    """Write the edge set into out_dir (created): ref.fa, sam/sNNN.sam, bam/sNNN.bam, all_samples, stacks.bed.
    sam_to_bam: the converter (default bin/msnv_synth of this tree)."""
    if sam_to_bam is None:
        from metasnv_b200.paths import bin_path
        sam_to_bam = bin_path("msnv_synth")
    fraction_pairs_straddle()
    rng = random.Random(20261020)
    ref = _ref(rng)
    reads = _reads(ref, rng)
    os.makedirs(os.path.join(out_dir, "sam"))
    os.makedirs(os.path.join(out_dir, "bam"))
    with open(os.path.join(out_dir, "ref.fa"), "w") as f:
        for name, _ in CONTIGS:
            s = "".join(ref[name])
            f.write(">%s\n" % name + "".join(s[i:i + 70] + "\n" for i in range(0, len(s), 70)))
    head = "@HD\tVN:1.6\tSO:coordinate\n" + "".join("@SQ\tSN:%s\tLN:%d\n" % c for c in CONTIGS)
    bams, narrow = [], []
    for s in range(N_SAMPLES):
        if max(_reads_per_tile(reads[s]).values(), default=0) <= 255:
            narrow.append(s)
        sam, bam = os.path.join(out_dir, "sam", "s%03d.sam" % s), os.path.join(out_dir, "bam", "s%03d.bam" % s)
        with open(sam, "w") as f:
            f.write(head + "".join(line for _, _, line in sorted(reads[s], key=lambda r: (r[0], r[1]))))
        subprocess.run([sam_to_bam, "--sam", sam, "--bam", bam], check=True)
        bams.append(bam)
    with open(os.path.join(out_dir, "all_samples"), "w") as f:
        f.write("\n".join(bams) + "\n")
    # the samples none of whose items is wide: a shard of them has items of exactly 255 reads and none above
    assert max(max(_reads_per_tile(reads[s]).values(), default=0) for s in narrow) == 255
    with open(os.path.join(out_dir, "narrow_samples"), "w") as f:
        f.write("\n".join(bams[s] for s in narrow) + "\n")
    with open(os.path.join(out_dir, "stacks.bed"), "w") as f:
        f.write("".join("%s\t%d\t%d\n" % iv for iv in stack_intervals()))
    return out_dir
