"""The pileup, call and coverage kernels at their arithmetic boundaries (B200 only: `pytest -m gpu`), on the edge set of
tests/golden/edge_set.py: byte-lane counters at 255 next to full and empty lanes, more than 256 narrow items of one tile
at 255 (the 16-bit partial sums of call_kernel, population sums above 65 535), 250..260 reads on one tile (the
narrow/wide item switch), stacks of 127..300 bases against thresholds on both sides of 128, 255 and 256 (the HI_THR
byte-lane test and the integer test of wide items) under every kind of reference character, cov*p next to an integer
(the fp64 fraction test), reads at the length limits, and coverage above 1023 (qaCompute -c).
Everything is compared with the oracle: per-sample per-position counts with the counts of its mpileup text, calls byte
for byte with `mpileup_oracle | snpCall`, coverage files byte for byte with qacompute_oracle."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import GOLDEN
from metasnv_b200 import harness as H
from metasnv_b200.paths import bin_path
from pileup_counts import first_difference, oracle_counts

sys.path.insert(0, GOLDEN)
import edge_set as E  # noqa: E402
from cases import file_digest  # noqa: E402

pytestmark = pytest.mark.gpu


class Edge:
    def __init__(self, d):
        self.dir = d
        self.bed = os.path.join(d, "stacks.bed")
        self.want_counts = None
        self.oracle = {}
        self.launches = {}

    def oracle_calls(self, opts, samples="all_samples"):
        """Prefix of the oracle's .called / .indiv for one EDGE_CALLS / NARROW_CALLS entry, checked against the pinned digests
        (tests/golden/make_oracle_digests.py): a change that moves the oracle and the product together fails here."""
        key = E.edge_key(opts, samples)
        if key not in self.oracle:
            prefix = os.path.join(self.dir, "oracle_%d" % len(self.oracle))
            rc, err = E.run_oracle_calls(self.dir, opts, prefix, samples)
            assert rc == 0, err
            want = json.load(open(os.path.join(GOLDEN, "oracle_digests.json")))
            for ext in (".called", ".indiv"):
                assert file_digest(prefix + ext) == want[key + ext], "oracle output %s%s differs from the pinned one" % (key, ext)
            self.oracle[key] = prefix
        return self.oracle[key]


@pytest.fixture(scope="module")
def edge(built, tmp_path_factory):
    return Edge(E.write_edge_set(str(tmp_path_factory.mktemp("edge") / "set")))


def _same(a, b):
    d = H.first_diff(a, b)
    assert not d, "%s vs %s: %s" % (a, b, d)


def _dump_counts(edge, out, env, samples="all_samples"):
    dump = out + ".counts"
    rc, err = H.run_product_snpcall(edge.dir, out, all_samples=os.path.join(edge.dir, samples),
                                    env=dict(os.environ, MSNV_DUMP_COUNTS=dump, MSNV_PERF_JSON=out + ".perf", **env))
    assert rc == 0, err
    lay = [l.rstrip("\n").split("\t") for l in open(dump + ".layout")]
    S, P = int(lay[0][0]), int(lay[0][1])
    layout = [(n, int(o), int(l)) for n, o, l in lay[1:]]
    return np.fromfile(dump, np.uint16).reshape(S, P, 5), layout, json.loads(open(out + ".perf").readline())


COUNT_FORMS = [{}, {"MSNV_PILEUP": "scatter"}, {"MSNV_PILEUP": "gather"},
               {"MSNV_PILEUP": "scatter", "MSNV_MAX_READS": "16", "MSNV_CHUNK_Q4": "1280"},     # smallest stage: one 4096-base read
               {"MSNV_PILEUP": "gather", "MSNV_MAX_READS": "16", "MSNV_CHUNK_Q4": "1280"},
               {"MSNV_CONSUMERS": "256"}, {"MSNV_STAGES": "3"}]


@pytest.mark.parametrize("env", COUNT_FORMS, ids=lambda e: "-".join("%s=%s" % kv for kv in e.items()) or "library")
def test_edge_counts_match_oracle_text(env, edge, tmp_path):
    got, layout, _ = _dump_counts(edge, str(tmp_path / "gpu"), env)
    S, P, _ = got.shape
    assert S == E.N_SAMPLES
    if edge.want_counts is None:
        want = oracle_counts(E.oracle_pileup(edge.dir), S, layout, P)
        deep = dict((n, o) for n, o, _ in layout)["deep"]
        # the set holds what it is meant to: 270 x 255 G at X1, 250..260 A at X2, 1200x from one BAM
        assert want[:, deep + E.X1, 2].sum() == 68850 and (want[:, deep + E.X1, 2] == 255).sum() == 270
        assert want[list(E.SWEEP), deep + E.X2, 0].tolist() == list(range(250, 261))
        assert want[E.DEEP_COV_SAMPLE, deep + E.DEEP_COV_AT:deep + E.DEEP_COV_AT + 200, :4].sum(axis=1).max() == 1200
        edge.want_counts = want
    d = first_difference(edge.want_counts, got, layout)
    assert not d, d


# (snpCall options, pileup form): every EDGE_CALLS entry with the library's choice; scatter and gather at the thresholds
# around the byte-lane forms; the count planes made and called in several ranges of tiles (a tile budget that holds the
# 310 items of the deepest tile but not the shard; the counts hook above only sees the last range), alone and in
# position windows
CALL_RUNS = ([(o, "library") for o in E.EDGE_CALLS] +
             [(o, f) for f in ("scatter", "gather") for o in E.EDGE_CALLS if o.get("t") in (128, 129, 256)] +
             [(o, f) for f in ("ranges", "windows") for o in E.EDGE_CALLS if o in ({}, dict(t=256, p=1.0), dict(t=129, p=1.0))])
FORM_ENV = {"library": {}, "scatter": {"MSNV_PILEUP": "scatter"}, "gather": {"MSNV_PILEUP": "gather"},
            "ranges": {"MSNV_TILE_BUDGET_MB": "3.75"}, "windows": {"MSNV_WINDOWS": "4", "MSNV_TILE_BUDGET_MB": "3.75"}}


@pytest.mark.parametrize("opts,form", CALL_RUNS, ids=["%s-%s" % (E.edge_key(o)[5:], f) for o, f in CALL_RUNS])
def test_edge_calls_match_oracle(opts, form, edge, tmp_path):
    o = edge.oracle_calls(opts)
    g = str(tmp_path / "gpu")
    kw = {k: v for k, v in opts.items() if k != "bed"}
    env = dict(os.environ, MSNV_PERF_JSON=g + ".perf", **FORM_ENV[form])
    rc, err = H.run_product_snpcall(edge.dir, g, bed=edge.bed if opts.get("bed") else None, env=env, **kw)
    assert rc == 0, err
    for ext in (".called", ".indiv"):
        _same(o + ext, g + ext)
    assert os.path.getsize(o + ".called") + os.path.getsize(o + ".indiv") > 0
    launches = json.loads(open(g + ".perf").readline())["launches"]
    if form == "library":
        edge.launches[E.edge_key(opts)] = launches
    elif form == "ranges" and E.edge_key(opts) in edge.launches:
        assert launches > edge.launches[E.edge_key(opts)], "the tile budget should split the shard into several ranges"


@pytest.mark.parametrize("opts", E.NARROW_CALLS, ids=[E.edge_key(o)[5:] for o in E.NARROW_CALLS])
def test_shard_whose_largest_items_hold_255_reads(opts, edge, tmp_path):
    """The samples without a wide item as a shard of their own: no item has more than 255 reads, many have exactly 255, so
    the pileup kernel is launched without its wide path and every item must be stored and read as narrow."""
    lst = os.path.join(edge.dir, "narrow_samples")
    if not opts:
        got, layout, _ = _dump_counts(edge, str(tmp_path / "counts"), {}, "narrow_samples")
        want = oracle_counts(E.oracle_pileup(edge.dir, samples="narrow_samples"), got.shape[0], layout, got.shape[1])
        assert (want.sum(axis=2) == 255).any() and not (want.sum(axis=2) > 255).any()
        d = first_difference(want, got, layout)
        assert not d, d
    o = edge.oracle_calls(opts, "narrow_samples")
    g = str(tmp_path / "gpu")
    rc, err = H.run_product_snpcall(edge.dir, g, all_samples=lst, **opts)
    assert rc == 0, err
    for ext in (".called", ".indiv"):
        _same(o + ext, g + ext)
    assert os.path.getsize(o + ".called") + os.path.getsize(o + ".indiv") > 0


@pytest.mark.parametrize("max_cov", [1, 1023, 1024, 5000])
def test_qacompute_above_1023_matches_oracle(max_cov, edge, tmp_path):
    """qaCompute -c on the BAM with 1200x: histogram bins above the 1024 held in shared memory."""
    bam = open(os.path.join(edge.dir, "all_samples")).readline().strip()
    outs = []
    for name, binary in (("oracle", H.oracle_bin("qacompute_oracle")), ("gpu", bin_path("qaCompute"))):
        out = str(tmp_path / (name + ".cov"))
        r = subprocess.run([binary, "-c", str(max_cov), "-d", "-i", bam, out], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        outs.append(out)
    for ext in ("", ".detail"):
        _same(outs[0] + ext, outs[1] + ext)
    if max_cov >= 1024:
        assert "\n1024\t" in open(outs[0]).read() and not open(outs[0]).read().split("\n1024\t")[1].startswith("0.00000\t0\n")
