"""metaSNV_coverage (B200 only: `pytest -m gpu`): a project's whole coverage pass in one process writes, for every BAM,
the same cov/<bam>.cov, .cov.detail and .cov.tidx as `qaCompute -c 10 -d -i` on that BAM alone (metaSNV.py:compute_opt),
and .cov / .cov.detail equal the committed golden files and qacompute_oracle."""
import filecmp
import json
import os
import random
import shutil
import subprocess
import sys

import pytest

from conftest import GOLDEN
from metasnv_b200 import harness as H
from metasnv_b200.paths import bin_path

pytestmark = pytest.mark.gpu

EXTS = (".cov", ".cov.detail", ".cov.tidx")


@pytest.fixture(scope="module")
def cov_built(built):
    if not os.path.exists(bin_path("metaSNV_coverage")):
        import __graft_entry__
        __graft_entry__.build()
    assert os.path.exists(bin_path("metaSNV_coverage"))
    return True


def _list(path, bams):
    with open(path, "w") as f:
        f.write("".join(b + "\n" for b in bams))
    return path


def run_coverage(project, all_samples, env=None):
    return subprocess.run([bin_path("metaSNV_coverage"), project, all_samples], capture_output=True, text=True,
                          env=dict(os.environ, **(env or {})))


def per_bam(project, bams):
    """What metaSNV.py:compute_opt leaves in <project>/cov: one qaCompute process per BAM."""
    os.makedirs(os.path.join(project, "cov"), exist_ok=True)
    for b in bams:
        r = H.run_qacompute(bin_path("qaCompute"), b, os.path.join(project, "cov", os.path.basename(b) + ".cov"))
        assert r.returncode == 0, r.stderr


def same_file(a, b):
    assert filecmp.cmp(a, b, shallow=False), "%s vs %s: %s" % (a, b, H.first_diff(a, b))


def same_tree(a, b, bams, exts=EXTS):
    assert sorted(os.listdir(os.path.join(a, "cov"))) == sorted(os.listdir(os.path.join(b, "cov")))
    for bam in bams:
        for e in exts:
            n = os.path.basename(bam) + e
            same_file(os.path.join(a, "cov", n), os.path.join(b, "cov", n))


def sam_to_bam(tmp, name, text):
    sam, bam = os.path.join(tmp, name + ".sam"), os.path.join(tmp, name + ".bam")
    with open(sam, "w") as f:
        f.write(text)
    subprocess.run([bin_path("msnv_synth"), "--sam", sam, "--bam", bam], check=True)
    os.remove(sam)
    return bam


def header(contigs):
    return "@HD\tVN:1.6\tSO:coordinate\n" + "".join("@SQ\tSN:%s\tLN:%d\n" % c for c in contigs)


# ---------------------------------------------------------------- committed golden files
@pytest.mark.parametrize("name", ["c1_tiny", "c4_tiny_deep", "c5_tiny_annotated"])
def test_golden_sets(name, cov_built, datasets, tmp_path):
    recipe = json.load(open(os.path.join(GOLDEN, name, "recipe.json")))
    data = datasets(recipe["preset"], recipe["scale"], recipe["samples"], **recipe["extra"])
    proj = str(tmp_path / "proj")
    r = run_coverage(proj, os.path.join(data, "all_samples"))
    assert r.returncode == 0, r.stderr
    bams = [l.strip() for l in open(os.path.join(data, "all_samples")) if l.strip()]
    for i, bam in enumerate(bams[:2]):
        for ext in ("", ".detail"):
            same_file(os.path.join(GOLDEN, name, "s%d.cov%s" % (i, ext)), os.path.join(proj, "cov", os.path.basename(bam) + ".cov" + ext))
    assert len(os.listdir(os.path.join(proj, "cov"))) == 3 * len(bams)


def test_hand_sams(cov_built, tmp_path):
    tmp = str(tmp_path)
    bams = []
    for s in ("s1", "s2"):
        out = os.path.join(tmp, s + ".bam")
        subprocess.run([bin_path("msnv_synth"), "--sam", os.path.join(GOLDEN, "hand", s + ".sam"), "--bam", out], check=True)
        bams.append(out)
    # surrounding white space and blank lines, as a hand-edited all_samples may have them
    lst = os.path.join(tmp, "all_samples")
    open(lst, "w").write("\n  %s\t\n\n%s" % (bams[0], bams[1]))
    proj = os.path.join(tmp, "proj")
    r = run_coverage(proj, lst)
    assert r.returncode == 0, r.stderr
    for s, bam in zip(("s1", "s2"), bams):
        for ext in ("", ".detail"):
            same_file(os.path.join(GOLDEN, "hand", "expected_%s.cov%s" % (s, ext)), os.path.join(proj, "cov", s + ".bam.cov" + ext))


# ---------------------------------------------------------------- seeded synthetic projects
SETS = [("c1", 0.2, 40, {}), ("c3", 0.0005, 10, {}), ("c4", 0.005, 3, {})]


@pytest.mark.parametrize("preset,scale,samples,kw", SETS, ids=["%s-%s-%d" % s[:3] for s in SETS])
def test_synthetic_project_equals_per_bam_runs(preset, scale, samples, kw, cov_built, datasets, tmp_path):
    data = datasets(preset, scale, samples, **kw)
    lst = os.path.join(data, "all_samples")
    bams = [l.strip() for l in open(lst) if l.strip()]
    one, per = str(tmp_path / "one"), str(tmp_path / "per")
    perf = str(tmp_path / "perf.jsonl")
    r = run_coverage(one, lst, env={"MSNV_PERF_JSON": perf})
    assert r.returncode == 0, r.stderr
    per_bam(per, bams)
    same_tree(one, per, bams)
    for bam in bams:
        o = str(tmp_path / "oracle.cov")
        assert H.run_qacompute(H.oracle_bin("qacompute_oracle"), bam, o).returncode == 0
        for ext in ("", ".detail"):
            same_file(o + ext, os.path.join(one, "cov", os.path.basename(bam) + ".cov" + ext))
    rec = json.loads(open(perf).read().splitlines()[-1])
    assert rec["tool"] == "metaSNV_coverage" and rec["bams"] == len(bams) and rec["bams_failed"] == 0
    assert rec["bam_bytes"] == sum(os.path.getsize(b) for b in bams)
    assert rec["peak_decoded_bams"] <= rec["decode_workers"] + 1
    assert rec["ms_cov_scatter"] > 0 and rec["ms_cov_scan"] > 0 and rec["cov_blocks"] > 0


def test_thread_counts_give_the_same_tree(cov_built, datasets, tmp_path):
    data = datasets("c1", 0.2, 40)
    lst = os.path.join(data, "all_samples")
    bams = [l.strip() for l in open(lst) if l.strip()]
    a, b = str(tmp_path / "a"), str(tmp_path / "b")
    perf = str(tmp_path / "perf.jsonl")
    assert run_coverage(a, lst, env={"MSNV_THREADS": "1", "MSNV_PERF_JSON": perf}).returncode == 0
    assert run_coverage(b, lst).returncode == 0
    same_tree(a, b, bams)
    rec = json.loads(open(perf).readline())
    assert rec["decode_workers"] == 1 and rec["inflate_threads"] == 1 and rec["peak_decoded_bams"] <= 2


# ---------------------------------------------------------------- awkward members of one project
@pytest.fixture(scope="module")
def awkward(cov_built, datasets, tmp_path_factory):
    """Tiny synthetic BAMs around four odd ones: only unmapped reads, header only, every read on one contig of 200, and
    one of more than 1.5e7 coverage blocks (reads of 2500 one-base M blocks, so that the file stays small)."""
    tmp = str(tmp_path_factory.mktemp("awkward"))
    data = datasets("c1", 0.02, 4)
    tiny = [l.strip() for l in open(os.path.join(data, "all_samples")) if l.strip()]
    ctgs = [("ctg%03d" % i, 5000 + 37 * i) for i in range(200)]
    unmapped = sam_to_bam(tmp, "unmapped", header(ctgs[:3]) + "".join(
        "u%d\t4\t*\t0\t0\t*\t*\t0\t0\tACGT\tIIII\n" % i for i in range(50)))
    header_only = sam_to_bam(tmp, "header_only", header(ctgs[:3]))
    rnd = random.Random(5)
    pos = sorted(rnd.randrange(1, 4900) for _ in range(300))
    one_contig = sam_to_bam(tmp, "one_contig", header(ctgs) + "".join(
        "r%d\t%d\tctg117\t%d\t%d\t50M\t*\t0\t0\t*\t*\n" % (i, rnd.choice((0, 16, 1024, 2)), p, rnd.choice((0, 5, 60)))
        for i, p in enumerate(pos)))
    big_ctgs = [("big%d" % i, 1000000) for i in range(3)]
    lines = []
    cig = "1M1D" * 2500
    for t, (n, ln) in enumerate(big_ctgs):
        for i, p in enumerate(sorted(rnd.randrange(1, ln - 6000) for _ in range(2100))):
            lines.append("b%d_%d\t0\t%s\t%d\t60\t%s\t*\t0\t0\t*\t*\n" % (t, i, n, p, cig))
    big = sam_to_bam(tmp, "big", header(big_ctgs) + "".join(lines))
    members = [tiny[0], unmapped, tiny[1], header_only, one_contig, tiny[2], big, tiny[3]]
    return tmp, members


def test_awkward_members(awkward, tmp_path):
    tmp, members = awkward
    lst = _list(str(tmp_path / "all_samples"), members)
    one, per = str(tmp_path / "one"), str(tmp_path / "per")
    perf = str(tmp_path / "perf.jsonl")
    r = run_coverage(one, lst, env={"MSNV_PERF_JSON": perf})
    assert r.returncode == 0, r.stderr
    per_bam(per, members)
    same_tree(one, per, members)
    rec = json.loads(open(perf).readline())
    assert rec["cov_blocks"] > 1.5e7
    # the three odd small ones: the header's contigs at zero, the read statistics as qaCompute counts them
    assert "Total number of reads: 50\n" in open(os.path.join(one, "cov", "unmapped.bam.cov")).read()
    assert open(os.path.join(one, "cov", "header_only.bam.cov")).read().count("\t0.00000\n") == 3
    det = open(os.path.join(one, "cov", "one_contig.bam.cov.detail")).read().splitlines()
    assert len(det) == 200 and sum(1 for l in det if l.split("\t")[2] != "0") == 1 and det[117].startswith("ctg117\t")


def test_failures_leave_the_other_bams_intact(cov_built, datasets, tmp_path):
    """An unreadable, an unsorted and a truncated BAM in the middle of the list: one message naming each, exit 1, and
    every other BAM's files identical to the clean run."""
    tmp = str(tmp_path)
    data = datasets("c1", 0.02, 4)
    good = [l.strip() for l in open(os.path.join(data, "all_samples")) if l.strip()]
    missing = os.path.join(tmp, "missing.bam")
    unsorted = sam_to_bam(tmp, "unsorted", header([("ctgA", 1000), ("ctgB", 1000)]) +
                          "r1\t0\tctgB\t10\t60\t20M\t*\t0\t0\t*\t*\nr2\t0\tctgA\t10\t60\t20M\t*\t0\t0\t*\t*\n")
    truncated = os.path.join(tmp, "truncated.bam")
    blob = open(good[0], "rb").read()
    open(truncated, "wb").write(blob[:len(blob) // 2])
    bad = [missing, unsorted, truncated]
    clean = str(tmp_path / "clean")
    assert run_coverage(clean, _list(os.path.join(tmp, "clean_list"), good)).returncode == 0
    proj = str(tmp_path / "proj")
    r = run_coverage(proj, _list(os.path.join(tmp, "list"), good[:2] + bad + good[2:]))
    assert r.returncode == 1
    msgs = [l for l in r.stderr.splitlines() if l.startswith("metaSNV_coverage:")]
    assert len(msgs) == 3, r.stderr
    for b in bad:
        assert sum(b in m for m in msgs) == 1, (b, r.stderr)
    assert "not coordinate sorted" in r.stderr
    same_tree(clean, proj, good)


# ---------------------------------------------------------------- the step behind: metaSNV_covSummary
def test_summaries_equal_those_of_the_per_bam_tree(cov_built, datasets, tmp_path):
    data = datasets("c1", 0.2, 40)
    lst = os.path.join(data, "all_samples")
    bams = [l.strip() for l in open(lst) if l.strip()]
    one, per = str(tmp_path / "a" / "proj"), str(tmp_path / "b" / "proj")
    os.makedirs(os.path.dirname(one))
    assert run_coverage(one, lst).returncode == 0
    per_bam(per, bams)
    for p in (one, per):
        r = subprocess.run([bin_path("metaSNV_covSummary"), p], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    same_tree(one, per, bams, exts=EXTS + (".cov.summary",))
    for f in ("proj.all_cov.tab", "proj.all_perc.tab"):
        same_file(os.path.join(one, f), os.path.join(per, f))
