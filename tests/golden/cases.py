"""Inputs and helpers shared by the tests and the scripts that regenerate the golden data under tests/golden/
(make_oracle_digests.py, make_filtering_golden.py). Needs neither pytest nor a GPU."""
import hashlib
import os

# test_gpu_parity.py::test_live_parity: preset, scale, samples, synth options, snpCall options
LIVE = [
    ("c1", 0.2, 40, {}, dict()),
    ("c1", 0.05, 12, {"seed": 7}, dict(c=10, t=2, p=0.2)),
    ("c1", 0.05, 12, {"seed": 8}, dict(c=1, t=1, p=0.0)),
    ("c3", 0.0005, 10, {}, dict()),
    ("c4", 0.005, 3, {}, dict()),
    ("c5", 0.004, 6, {"annotation": True}, dict()),
    ("c2", 0.004, 160, {}, dict()),
]

# test_gpu_parity.py::test_snpcall_in_windows_equals_oracle: preset, scale, samples, windows
WINDOWED = [("c1", 0.1, 12, 5), ("c4", 0.005, 3, 4), ("c3", 0.0005, 10, 7)]

# test_filtering_cpu.py::test_freq_files_identical_to_reference_script: metaSNV_Filtering options by name
FILTER_OPTS = {
    "defaults": [],
    "strict-positions": ["-c", "8", "-p", "0.9"],
    "few-samples-ind": ["-d", "10.2", "-b", "99.8", "-m", "1", "--ind"],
    "lenient-threads": ["-c", "1", "-p", "0.0", "--n_threads", "3"],
    "no-taxon": ["-m", "20"],
}


def oracle_mpileup(ref, samples, out, bed=None):
    """The oracle's mpileup text of the BAMs listed in `samples` (`mpileup_oracle mpileup -f ref [-l bed] -B -b samples`),
    written to out; returns out."""
    import subprocess
    from metasnv_b200 import harness as H
    with open(out, "wb") as f:
        subprocess.run([H.oracle_bin("mpileup_oracle"), "mpileup", "-f", ref] + (["-l", bed] if bed else []) + ["-B", "-b", samples],
                       stdout=f, check=True)
    return out


def file_digest(path):
    data = open(path, "rb").read()
    return {"sha256": hashlib.sha256(data).hexdigest(), "lines": data.count(b"\n")}


def tree_digests(root):
    """file_digest of every file under root, by path relative to it."""
    out = {}
    for d, _, fs in os.walk(root):
        for f in fs:
            p = os.path.join(d, f)
            out[os.path.relpath(p, root)] = file_digest(p)
    return out


def data_key(preset, scale, samples, kw=None, opts=None):
    """Name of a synthetic data set and its snpCall options in oracle_digests.json."""
    extra = sorted((kw or {}).items()) + sorted((opts or {}).items())
    return "-".join([preset, str(scale), str(samples)] + ["%s%s" % kv for kv in extra])


def write_cov_hand(d):
    """A project directory holding only qaCompute's files, made by hand: several contigs per taxon, a taxon that is not
    covered at all, lengths that make the weighted averages inexact in binary, sample names that sort differently as
    text and as numbers."""
    rows = [("101.pA.c1", 1000003, 12.34567, 900001, 800002), ("101.pA.c2", 7, 0.14286, 1, 0), ("101.pA.c3", 333331, 3.00001, 333331, 111110),
            ("202.pB.x", 4999999, 0.00000, 0, 0), ("303.c", 1234567, 107.10101, 1234567, 1234566), ("101.late", 11, 1.09091, 11, 1)]
    os.makedirs(os.path.join(d, "cov"))
    for s, scale in (("s2.bam", 1.0), ("s10.bam", 0.37), ("S1.bam", 2.5)):
        with open(os.path.join(d, "cov", s + ".cov"), "w") as f:
            f.write("Chromosome\tSeq_lem\tAvg_Cov\n")
            for n, L, avg, x1, x2 in rows:
                f.write("%s\t%d\t%3.5f\n" % (n, L, avg * scale))
            f.write("\n")
        with open(os.path.join(d, "cov", s + ".cov.detail"), "w") as f:
            for n, L, avg, x1, x2 in rows:
                f.write("%s\t%d\t%d\t%d\t0\t\n" % (n, L, int(x1 * min(1.0, scale)), int(x2 * min(1.0, scale))))
