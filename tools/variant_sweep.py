#!/usr/bin/env python3
"""Tuning aid: one device-generated shard, msnv_shard_run under several staging settings of the pileup kernel
(MSNV_PILEUP_CTAS : MSNV_CHUNK_Q4 : MSNV_MAX_READS : MSNV_CONSUMERS : MSNV_PILEUP : MSNV_STAGES, empty = the library's own choice)."""
import argparse, json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from metasnv_b200 import abi, harness as H

ap = argparse.ArgumentParser()
ap.add_argument("--preset", default="c2"); ap.add_argument("--scale", type=float, default=1.0)
ap.add_argument("--samples", type=int, default=0); ap.add_argument("--steps", type=int, default=3)
ap.add_argument("--no-hits", action="store_true", help="thresholds no position meets (no hits to gather and copy)")
ap.add_argument("--settings", default="::,2::,3::,4::,5::", help="comma list of <ctas per SM>:<chunk_q4>:<max_reads>, empty fields = default")
a = ap.parse_args()
desc = H.describe(a.preset, a.scale, a.samples)
ctx = abi.Context(0)
n_pos, first = ctx.shard_synth(desc)
if first >= 0:
    ctx.shard_mask_position(first)
ref_hits = None
for setting in a.settings.split(","):
    fields = (setting.split(":") + [""] * 6)[:6]
    for k, v in zip(("MSNV_PILEUP_CTAS", "MSNV_CHUNK_Q4", "MSNV_MAX_READS", "MSNV_CONSUMERS", "MSNV_PILEUP", "MSNV_STAGES"), fields):
        os.environ.pop(k, None)
        if v:
            os.environ[k] = v
    kw = dict(min_coverage=2000000000) if a.no_hits else {}
    ctx.shard_run(copy=False, **kw)
    ms = []
    for _ in range(a.steps):
        h = ctx.shard_run(copy=False, **kw)
        ms.append(ctx.timings()["ms_pileup"])
    if ref_hits is None:
        ref_hits = h.n_hits
    print(json.dumps({"setting": setting, "ms_pileup": sum(ms) / len(ms), "min": min(ms), "ms_mate": ctx.timings().get("ms_mate"), "hits_equal": h.n_hits == ref_hits}), flush=True)
