#!/usr/bin/env python3
"""Regenerate tests/golden/oracle_digests.json: SHA-256 and line count of every oracle output that
tests/test_gpu_parity.py, tests/test_gpu_kernel_edges.py and tests/test_gpu_long_spans.py compare the product with, on the same seeded inputs. Needs no GPU:
    python tests/golden/make_oracle_digests.py
The oracle is `mpileup_oracle | snpCall`, with the upstream snpCall build when oracle/_ref has it and the
C restatement otherwise (the two agree on every vector of tests/golden/snpcall_vectors.json).
"""
import json
import os
import shutil
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import __graft_entry__  # noqa: E402
from metasnv_b200 import harness as H  # noqa: E402
from metasnv_b200.paths import bin_path  # noqa: E402
from cases import LIVE, WINDOWED, data_key, file_digest  # noqa: E402
import edge_set  # noqa: E402
import span_set  # noqa: E402

EMPTY_SAM = "@HD\tVN:1.6\tSO:coordinate\n@SQ\tSN:ctgA\tLN:40\n@SQ\tSN:ctgB\tLN:40\n"


def main():
    __graft_entry__.build()
    out = {}
    work = tempfile.mkdtemp(prefix="msnv_oracle_digests_")

    def oracle(key, data, **kw):
        prefix = os.path.join(work, "out")
        rc, err = H.run_oracle_snpcall(data, prefix, **kw)
        assert rc == 0, err
        for ext in (".called", ".indiv"):
            out[key + ext] = file_digest(prefix + ext)

    def synth(preset, scale, samples, **kw):
        d = os.path.join(work, data_key(preset, scale, samples, kw))
        if not os.path.isdir(d):
            H.synth(d, preset, scale, samples, **kw)
        return d

    def hand(name, sams):
        d = os.path.join(work, name)
        os.makedirs(d)
        bams = []
        for s in sams:
            b = os.path.join(d, s + ".bam")
            subprocess.run([bin_path("msnv_synth"), "--sam", os.path.join(HERE, "hand", s + ".sam"), "--bam", b], check=True)
            bams.append(b)
        open(os.path.join(d, "all_samples"), "w").write("\n".join(bams) + "\n")
        os.symlink(os.path.join(HERE, "hand", "ref.fa"), os.path.join(d, "ref.fa"))
        return d

    # test_live_parity and test_snpcall_in_windows_equals_oracle
    runs = [(p, s, n, kw, opts) for p, s, n, kw, opts in LIVE] + [(p, s, n, {}, {}) for p, s, n, _ in WINDOWED]
    for preset, scale, samples, kw, opts in runs:
        data = synth(preset, scale, samples, **kw)
        ann = os.path.join(data, "annotation.txt") if kw.get("annotation") else None
        bed = H.bed_header(data, os.path.join(data, "bed_header"))
        for mode, b in (("unsplit", None), ("split", bed)):
            oracle(data_key(preset, scale, samples, kw, opts) + "/" + mode, data, bed=b, ann=ann, **opts)

    # test_split_files_concatenate_to_whole: one genome per split
    data = synth("c1", 0.05, 12)
    for k, ln in enumerate(open(H.bed_header(data, os.path.join(data, "bed_header"))).read().splitlines()):
        sp = os.path.join(work, "best_split_%d" % k)
        open(sp, "w").write(ln + "\n")
        oracle(data_key("c1", 0.05, 12) + "/best_split_%d" % k, data, bed=sp)

    # test_two_splits_on_two_gpus: genomes dealt to two bins
    data = synth("c1", 0.1, 12)
    beds = []
    for k, line in enumerate(open(H.bed_header(data, os.path.join(data, "bed_header")))):
        p = os.path.join(work, "two_bins_%d" % (k % 2))
        open(p, "a").write(line)
        if p not in beds:
            beds.append(p)
    for k, bed in enumerate(beds):
        oracle(data_key("c1", 0.1, 12) + "/two_bins_%d" % k, data, bed=bed)

    # hand-written cases
    d = hand("rules", ["s5_rules", "s2"])
    oracle("hand/s5_rules+s2/whole", d, c=1, t=1)
    oracle("hand/s5_rules+s2/bed", d, bed=os.path.join(HERE, "hand", "rules.bed"), c=1, t=1)
    d = hand("leading_del", ["s6_leading_del", "s1"])
    oracle("hand/s6_leading_del+s1/whole", d, c=1, t=1)
    d = hand("empty", ["s1"])
    sam = os.path.join(d, "e.sam")
    open(sam, "w").write(EMPTY_SAM)
    e1, e2 = os.path.join(d, "e1.bam"), os.path.join(d, "e2.bam")
    for e in (e1, e2):
        subprocess.run([bin_path("msnv_synth"), "--sam", sam, "--bam", e], check=True)
    for name, bams in (("only_empty", [e1, e2]), ("mixed", [e1, os.path.join(d, "s1.bam"), e2])):
        lst = os.path.join(d, name + ".list")
        open(lst, "w").write("\n".join(bams) + "\n")
        oracle("hand/empty/" + name, d, all_samples=lst, c=1, t=1)

    # tests/test_gpu_kernel_edges.py: the edge set under every option set it is called with
    d = edge_set.write_edge_set(os.path.join(work, "edge"))
    for samples, calls in (("all_samples", edge_set.EDGE_CALLS), ("narrow_samples", edge_set.NARROW_CALLS)):
        for opts in calls:
            prefix = os.path.join(work, "out")
            rc, err = edge_set.run_oracle_calls(d, opts, prefix, samples)
            assert rc == 0, err
            for ext in (".called", ".indiv"):
                out[edge_set.edge_key(opts, samples) + ext] = file_digest(prefix + ext)

    # tests/test_gpu_long_spans.py: the span set under every option set it is called with
    d = span_set.write_span_set(os.path.join(work, "span"))
    for opts in span_set.SPAN_CALLS:
        prefix = os.path.join(work, "out")
        rc, err = span_set.run_oracle_calls(d, opts, prefix)
        assert rc == 0, err
        for ext in (".called", ".indiv"):
            out[span_set.span_key(opts) + ext] = file_digest(prefix + ext)

    with open(os.path.join(HERE, "oracle_digests.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    shutil.rmtree(work)
    print("oracle_digests.json: %d files (oracle snpCall: %s)" % (len(out), os.path.basename(H.oracle_snpcall())))


if __name__ == "__main__":
    main()
