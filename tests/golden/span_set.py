"""A small, deterministic data set of SAM-built BAMs aimed at the reference span of reads (pos to the last covered
position, D and N included) rather than their base count: the index's reach (`max_span`, the bitmap walk's `back`),
items whose candidate reads mostly never touch their tile, the gather form's geometry for reads whose first segment lies
tiles behind their pos, the decoder's carry of reads from one window to the next, the depth cap with reads buffered
through a skip, and the span limit MSNV_MAX_READ_SPAN (32768). Needs neither pytest nor a GPU:

    from span_set import write_span_set
    write_span_set(out_dir)     # ref.fa, sam/*.sam, bam/*.bam, all_samples, span.bed, over/ (one read of span 32769)

Positions are 0-based contig coordinates; every contig starts on a tile (shard layout), so tile boundaries are multiples of
1024 in contig coordinates. Bases carry about 5 % noise, so low thresholds call most covered positions.
  sample 0  reach   for each span in SPANS and each of M..N..M / M..D..M: one read whose first base is on the last
                    position of a tile, one whose last base is the first position of a tile, one whose last base is the
                    position before a tile; every last aligned base is a non-reference base. The sample's max_span is
                    32768, so only its 32768 reads start at a tile's k_lo; the others are ordinary candidates.
  sample 1  reach   ~3x coverage of 100-base reads plus a few 32768-span reads: items with more than 255 candidate reads of
                    which a few touch the tile.
  sample 2  reach   only long reads of many operations (up to 32768 positions), one whose skip covers tiles 1..4 whole and
                    ends on a tile boundary; sparse, so the index's bitmap path is taken by default.
  sample 3  reach   the set's first read opens with an N (the first pileup line, which snpCall drops, has no base);
            lead    reads opening with 1..20 kb of N or D, each followed by reads starting inside the tile of its pos.
  sample 4  mates   overlapping proper pairs where one or both mates carry a 5..20 kb N or D; the overlap before the gap,
                    after it, and across a tile boundary; qualities around the 12 / 13 of the overlap rule.
  samples 6..10     one span of SPANS each (max_span is that span; its residues mod 1024 are 1, 0, 0, 1023, 0), reads
  reach, lead       of M..N..M and M..D..M, one per run of back + 1 tiles: a read whose first base is on the last position
                    of tile u ends in tile u + back, a read ending on the first position of tile m starts at k_lo of m
                    (in tile m - back), and no other read of the sample starts in between. The index's bitmap walk
                    (back = (max_span + TILE - 2) / TILE) and its binary search (k_lo = t0 - max_span + 1) find these
                    reads at exactly their reach.
  sample 5  lead    the depth cap: hundreds of long reads still buffered (covering the position through a skip) where
                    7900 reads start on ten positions.
snpCall reads a pileup column of at most 10000 characters and a deletion shows its deleted bases in the text, so the set
keeps every column whose text is longer than that free of bases behind the cut (text_fits_snpcall): the calls of the
oracle are then those of its counts.
span.bed holds an interval inside a read's N gap, one starting on a long read's last base, and a few ordinary ones.
"""
import os
import random
import subprocess

TILE = 1024
CONTIGS = [("reach", 110000), ("lead", 60000), ("mates", 44000)]        # 108 + 59 + 43 = 210 tiles
N_TILES = 210
N_SAMPLES = 11
SPANS = [4097, 8192, 16384, 32767, 32768]
MAX_SPAN = 32768                          # MSNV_MAX_READ_SPAN
ISOLATED = 6                              # samples 6..10: one span of SPANS each
CAP_AT, CAP_STARTS, CAP_READS, CAP_LONG = 30 * TILE + 500, 10, 790, 300     # reads start at CAP_AT .. CAP_AT + 9
GAP_READ = ("reach", 1000, [(24, "M"), (4 * TILE, "N"), (76, "M")])    # skip over tiles 1..4, ends on 5 * TILE
GAP_BED = ("reach", 2000, 2100)           # inside GAP_READ's skip (sample 2)

# snpCall options the span set is called with (tests/test_gpu_long_spans.py, make_oracle_digests.py); "bed": restricted to
# span.bed
SPAN_CALLS = [{}, dict(c=1, t=1), dict(c=1, t=0, bed=True)]


def span_key(opts):
    """Name of one SPAN_CALLS entry in oracle_digests.json."""
    return "span/" + ("-".join("%s%s" % kv for kv in sorted(opts.items())) or "defaults")


def _other(b, k=1):
    return "ACGT"[("ACGT".index(b.upper()) + k) % 4]


def span_of(ops):
    return sum(n for n, op in ops if op in "MDN=X")


def _sam_line(name, flag, ctg, pos0, ops, seq, qual, mate=None):
    rnext, pnext, tlen = ("=", mate[0] + 1, mate[1]) if mate else ("*", 0, 0)
    cigar = "".join("%d%s" % o for o in ops)
    return "%s\t%d\t%s\t%d\t60\t%s\t%s\t%d\t%d\t%s\t%s\n" % (name, flag, ctg, pos0 + 1, cigar, rnext, pnext, tlen, seq, qual)


class _Reads:
    def __init__(self, ref, rng):
        self.ref, self.rng = ref, rng
        self.out = {s: [] for s in range(N_SAMPLES)}
        self.ci = {name: k for k, (name, _) in enumerate(CONTIGS)}

    def seq(self, ctg, pos, ops, last_alt=True):
        """Bases of a read: the reference with ~5 % noise, inserted / clipped bases at random; the last aligned base is a
        non-reference base when last_alt."""
        g, rng = self.ref[ctg], self.rng
        out, x, last = [], pos, None
        for n, op in ops:
            if op == "M":
                out += [g[x + i] if rng.random() > 0.05 else _other(g[x + i], rng.randint(1, 3)) for i in range(n)]
                x += n
                last = (len(out) - 1, x - 1)           # (query index, reference position) of the last aligned base
            elif op in "DN":
                x += n
            elif op in "IS":
                out += [rng.choice("ACGT") for _ in range(n)]
        if last_alt:
            out[last[0]] = _other(g[last[1]])
        return "".join(out)

    def qual(self, n):
        """Mostly 40, some 12 and 13 (on both sides of mpileup's -Q 13); the last base 40."""
        q = [self.rng.choice("IIII-.5") for _ in range(n)]
        q[-1] = "I"
        return "".join(q)

    def add(self, s, name, ctg, pos, ops, flag=0, seq=None, qual=None, mate=None, last_alt=True):
        assert pos >= 0 and pos + span_of(ops) <= dict(CONTIGS)[ctg], (name, pos, ops)
        seq = seq if seq is not None else self.seq(ctg, pos, ops, last_alt)
        qual = qual if qual is not None else self.qual(len(seq))
        self.out[s].append((self.ci[ctg], pos, _sam_line(name, flag, ctg, pos, ops, seq, qual, mate)))


def _gap_ops(span, op, left=50, right=50):
    return [(left, "M"), (span - left - right, op), (right, "M")]


def _reads(ref, rng):
    """{sample: [(contig index, pos0, SAM line)]}"""
    R = _Reads(ref, rng)
    # sample 0: reach boundaries (ends on the last position of a tile, on the first, on the one before a tile)
    for i, (span, op) in enumerate((s, o) for s in SPANS for o in "ND"):
        k = 2 + 3 * i
        R.add(0, "a%d_%d%s" % (i, span, op), "reach", k * TILE + TILE - 1, _gap_ops(span, op))
        m = 40 + 3 * i
        R.add(0, "b%d_%d%s" % (i, span, op), "reach", m * TILE - span + 1, _gap_ops(span, op, 30 + i, 70 - i))
        m = 70 + 3 * i
        R.add(0, "c%d_%d%s" % (i, span, op), "reach", m * TILE - span, _gap_ops(span, op, 60, 40))
    # samples 6..10: one span each, so that the sample's max_span is that span, and reads isolated: one whose first base
    # is on the last position of tile u ends in tile u + back; one ending on the first position of tile m starts at that
    # tile's k_lo, in tile m - back; no other read of the sample starts in the tiles between (the bitmap walk's reach is
    # exact)
    for k, span in enumerate(SPANS):
        back = (span + TILE - 2) // TILE
        ctg, u = "reach", 1
        for name, op in (("a", "N"), ("b", "D"), ("a", "D"), ("b", "N")):
            if (u + back + 1) * TILE > dict(CONTIGS)[ctg]:
                ctg, u = "lead", 1
            if name == "a":
                pos, ops = u * TILE + TILE - 1, _gap_ops(span, op)
            else:
                pos, ops = (u + back) * TILE - span + 1, _gap_ops(span, op, 30, 70)
            assert pos // TILE == u and (pos + span - 1) // TILE == u + back
            R.add(ISOLATED + k, "%s_%d%s" % (name, span, op), ctg, pos, ops)
            u += back + 1
    # sample 1: ~3x coverage of 100-base reads plus four reads of span 32768
    for j in range(3300):
        R.add(1, "d%d" % j, "reach", rng.randint(10, 110000 - 100), [(100, "M")], last_alt=False)
    for j, pos in enumerate((5000, 30000, 50000, 70000)):
        R.add(1, "D%d" % j, "reach", pos, _gap_ops(MAX_SPAN, "N"))
    # sample 2: long reads of many operations only
    ctg, pos, ops = GAP_READ
    R.add(2, "gap", ctg, pos, ops)
    for j in range(14):
        span = rng.choice([5000, 9000, 15000, 24000, 32000, MAX_SPAN])
        parts, x = [(rng.randint(2, 5), "S")], 0
        while True:
            m, g = rng.randint(20, 60), rng.randint(200, 6000)
            if x + m + g + 40 > span:
                break
            parts += [(m, "M")] + ([(rng.randint(1, 3), "I")] if rng.random() < 0.3 else []) + [(g, rng.choice("ND"))]
            x += m + g
        rest = span - x
        parts += [(20, "M"), (rest - 60, rng.choice("ND")), (40, "M")] if rest > 100 else [(rest, "M")]
        assert span_of(parts) == span and len([p for p in parts if p[1] == "M"]) <= 128
        R.add(2, "x%d" % j, "reach", rng.randint(6000, 110000 - span), parts)
    # sample 3: the set's first read opens with an N; leading N / D of 1..20 kb on lead, each followed by reads that start
    # inside the tile of its pos
    R.add(3, "first", "reach", 0, [(3000, "N"), (60, "M")])
    for j in range(10):
        lead = [1000, 3000, 5000, 8000, 12000, 16000, 20000][j % 7] + rng.randint(0, 200)
        t = 1 + 4 * j
        pos = t * TILE + rng.randint(0, 600)
        R.add(3, "L%d" % j, "lead", pos, [(lead, "N" if j % 2 == 0 else "D"), (80, "M"), (500, "N"), (40, "M")])
        for k in range(3):
            R.add(3, "l%d_%d" % (j, k), "lead", rng.randint(pos + 1, (t + 1) * TILE - 1), [(100, "M")], last_alt=False)
    # sample 4: overlapping proper pairs with gaps
    qpool = [10, 12, 13, 16, 17, 40]

    def pair(name, pa, ops_a, pb, ops_b):
        ea, eb = pa + span_of(ops_a), pb + span_of(ops_b)
        tlen = max(ea, eb) - pa
        sa = R.seq("mates", pa, ops_a, last_alt=False)
        sb = list(R.seq("mates", pb, ops_b, last_alt=False))
        for i in range(len(sb)):
            if rng.random() < 0.3:
                sb[i] = _other(sb[i], rng.randint(1, 3))
        qa = "".join(chr(33 + rng.choice(qpool)) for _ in sa)
        qb = "".join(chr(33 + rng.choice(qpool)) for _ in sb)
        R.add(4, name, "mates", pa, ops_a, 99, sa, qa, (pb, tlen))
        R.add(4, name, "mates", pb, ops_b, 147, "".join(sb), qb, (pa, -tlen))

    a = 2 * TILE + 100
    pair("before", a, [(60, "M"), (8000, "N"), (40, "M")], a + 30, [(60, "M")])
    a = 3 * TILE + 300
    pair("after", a, [(40, "M"), (8000, "D"), (60, "M")], a + 8060, [(60, "M")])
    a = 12 * TILE + 700
    pair("both", a, [(50, "M"), (6000, "D"), (50, "M")], a + 20, [(30, "M"), (6000, "D"), (70, "M")])
    a = 22 * TILE - 40
    pair("cross", a, [(60, "M"), (10000, "N"), (40, "M")], a + 20, [(60, "M")])
    a = 4 * TILE + 500                        # the later mate overlaps the last 30 M of the earlier one on 20 * TILE - 10 ..
    pair("cross_after", a, [(40, "M"), (20 * TILE - 30 - 40 - a, "N"), (60, "M")], 20 * TILE - 10, [(30, "M"), (5000, "N"), (30, "M")])
    a = 14 * TILE + 10
    pair("both_n", a, [(45, "M"), (20000, "N"), (55, "M")], a + 5, [(40, "M"), (20000, "N"), (60, "M")])
    # sample 5: the depth cap with long reads still buffered, most of them covering CAP_AT.. through a skip; the reads
    # that fill the buffer start on ten positions, so that no pileup column is wider than the 10000 characters snpCall
    # reads (3 characters per starting read)
    starts = sorted(rng.randint(CAP_AT - 8000, CAP_AT - 1) for _ in range(CAP_LONG))
    for j, pos in enumerate(starts):
        R.add(5, "k%d" % j, "lead", pos, _gap_ops(rng.randint(10000, 20000), "N", 20, 20))
    for k in range(CAP_STARTS):
        for j in range(CAP_READS):
            R.add(5, "K%d_%d" % (k, j), "lead", CAP_AT + k, [(30, "M")], last_alt=False)
    return R.out


def bed_intervals(reads):
    """(contig, begin, end) of span.bed: inside GAP_READ's skip, one starting on the last base of sample 0's first read, and
    a few ordinary ones."""
    import re
    c, pos, line = reads[0][0]
    ops = re.findall(r"(\d+)([MIDNSHP=X])", line.split("\t")[5])
    last = pos + sum(int(n) for n, op in ops if op in "MDN=X") - 1
    return [GAP_BED, ("reach", last, last + 50), ("reach", 20000, 20400), ("lead", CAP_AT - 100, CAP_AT + 100),
            ("mates", 22 * TILE - 100, 22 * TILE + 100)]


def _bases(col):
    """Bases (not deleted-sequence letters, not start markers) in one mpileup column."""
    n = i = 0
    while i < len(col):
        ch = col[i]
        if ch == "^":
            i += 2
            continue
        if ch in "+-":
            j = i + 1
            while j < len(col) and col[j].isdigit():
                j += 1
            i = j + int(col[i + 1:j])
            continue
        n += ch in ".,ACGTNacgtn"
        i += 1
    return n


def text_fits_snpcall(pile_path, limit=10000):
    """[(contig, 1-based position, sample)] of the columns of mpileup text whose cut at `limit` characters (snpCall's
    toksplit) loses a base."""
    bad = []
    for line in open(pile_path):
        f = line.rstrip("\n").split("\t")
        for s in range((len(f) - 3) // 3):
            col = f[4 + 3 * s]
            if len(col) > limit and _bases(col) != _bases(col[:limit]):
                bad.append((f[0], int(f[1]), s))
    return bad


def oracle_pileup(d, bed=False, samples="all_samples"):
    """The oracle's mpileup text of the set in d (or of its span.bed), written once into d."""
    from cases import oracle_mpileup
    path = os.path.join(d, "pile_%s%s.txt" % (samples, "_bed" if bed else ""))
    if not os.path.exists(path):
        oracle_mpileup(os.path.join(d, "ref.fa"), os.path.join(d, samples), path, os.path.join(d, "span.bed") if bed else None)
    return path


def run_oracle_calls(d, opts, prefix):
    """`mpileup_oracle | oracle snpCall` with one SPAN_CALLS entry -> prefix.called / prefix.indiv; returns (rc, stderr)."""
    from metasnv_b200 import harness as H
    kw = {k: v for k, v in opts.items() if k != "bed"}
    with open(oracle_pileup(d, opts.get("bed", False)), "rb") as fin, open(prefix + ".called", "wb") as fout:
        r = subprocess.run([H.oracle_snpcall()] + H.snpcall_args(os.path.join(d, "ref.fa"), prefix + ".indiv", **kw),
                           stdin=fin, stdout=fout, stderr=subprocess.PIPE)
    return r.returncode, r.stderr.decode(errors="replace")


def write_span_set(out_dir, sam_to_bam=None):
    """Write the span set into out_dir (created): ref.fa, sam/sN.sam, bam/sN.bam, all_samples, span.bed, and over/: one
    read of span 32769 (over/all_samples; not part of the set's all_samples). sam_to_bam: the converter (default
    bin/msnv_synth of this tree)."""
    if sam_to_bam is None:
        from metasnv_b200.paths import bin_path
        sam_to_bam = bin_path("msnv_synth")
    rng = random.Random(20261021)
    ref = {name: [rng.choice("ACGT") for _ in range(n)] for name, n in CONTIGS}
    reads = _reads(ref, rng)
    for sub in ("sam", "bam", "over"):
        os.makedirs(os.path.join(out_dir, sub))
    with open(os.path.join(out_dir, "ref.fa"), "w") as f:
        for name, _ in CONTIGS:
            s = "".join(ref[name])
            f.write(">%s\n" % name + "".join(s[i:i + 70] + "\n" for i in range(0, len(s), 70)))
    head = "@HD\tVN:1.6\tSO:coordinate\n" + "".join("@SQ\tSN:%s\tLN:%d\n" % c for c in CONTIGS)

    def bam(sam_path, lines):
        with open(sam_path, "w") as f:
            f.write(head + "".join(line for _, _, line in sorted(lines, key=lambda r: (r[0], r[1]))))
        out = os.path.join(out_dir, "bam" if "over" not in sam_path else "over", os.path.basename(sam_path)[:-4] + ".bam")
        subprocess.run([sam_to_bam, "--sam", sam_path, "--bam", out], check=True)
        return out

    bams = [bam(os.path.join(out_dir, "sam", "s%d.sam" % s), reads[s]) for s in range(N_SAMPLES)]
    with open(os.path.join(out_dir, "all_samples"), "w") as f:
        f.write("\n".join(bams) + "\n")
    with open(os.path.join(out_dir, "span.bed"), "w") as f:
        f.write("".join("%s\t%d\t%d\n" % iv for iv in bed_intervals(reads)))
    # over the limit: one read of span MAX_SPAN + 1 behind an ordinary one
    R = _Reads(ref, rng)
    R.add(0, "ok", "reach", 10, [(100, "M")])
    R.add(0, "too_long", "reach", 100, _gap_ops(MAX_SPAN + 1, "N"))
    over = bam(os.path.join(out_dir, "over", "over.sam"), R.out[0])
    with open(os.path.join(out_dir, "over", "all_samples"), "w") as f:
        f.write(over + "\n")
    return out_dir
