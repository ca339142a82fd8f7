"""metaSNV_coverage's command line, checked without a GPU: argument count, an unreadable or empty all_samples, two BAMs
with the same basename (refused before anything is written), and no CUDA device."""
import os
import subprocess

import pytest

from metasnv_b200 import harness as H
from metasnv_b200.paths import bin_path


@pytest.fixture(scope="module")
def cov_bin(built):
    if not os.path.exists(bin_path("metaSNV_coverage")):
        import __graft_entry__
        __graft_entry__.build()
    assert os.path.exists(bin_path("metaSNV_coverage"))
    return bin_path("metaSNV_coverage")


def run(args, env=None):
    return subprocess.run([bin_path("metaSNV_coverage")] + args, capture_output=True, text=True, env=env)


def test_usage(cov_bin, tmp_path):
    for args in ([], [str(tmp_path / "p")], [str(tmp_path / "p"), "a", "b"]):
        r = run(args)
        assert r.returncode == 1 and "usage: metaSNV_coverage <project_dir> <all_samples>" in r.stderr
    assert not (tmp_path / "p").exists()


def test_missing_or_empty_all_samples(cov_bin, tmp_path):
    proj = str(tmp_path / "p")
    r = run([proj, str(tmp_path / "nonexistent")])
    assert r.returncode == 1 and "cannot read" in r.stderr
    empty = tmp_path / "empty"
    for text in ("", "\n \n\t\n"):
        empty.write_text(text)
        r = run([proj, str(empty)])
        assert r.returncode == 1 and "lists no BAM" in r.stderr
    assert not os.path.exists(proj)


def test_duplicate_basenames_are_refused(cov_bin, tmp_path):
    d = str(tmp_path / "d")
    H.synth(d, "c1", 0.02, 2)
    bams = [l.strip() for l in open(os.path.join(d, "all_samples"))]
    other = tmp_path / "other"
    other.mkdir()
    twin = str(other / os.path.basename(bams[0]))
    os.symlink(bams[0], twin)
    lst = tmp_path / "all_samples"
    lst.write_text("%s\n%s\n  %s\n" % (bams[0], bams[1], twin))
    proj = str(tmp_path / "p")
    r = run([proj, str(lst)])
    assert r.returncode == 1
    assert bams[0] in r.stderr and twin in r.stderr
    assert not os.path.exists(proj)


def test_fails_loudly_without_gpu(cov_bin, tmp_path):
    d = str(tmp_path / "d")
    H.synth(d, "c1", 0.02, 2)
    proj = str(tmp_path / "p")
    r = run([proj, os.path.join(d, "all_samples")], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 1 and "no usable CUDA device" in r.stderr
    assert not os.path.exists(proj)
