#!/usr/bin/env python3
"""BGZF inflate on the device (msnv_inflate) against the host's inflate, on one GPU, in one call:
  kernel     every member of the data set (bench.py's e2e BAM set by default) through msnv_inflate in batches of each
             --batch-mb size, warmed up first; the kernel's CUDA-event time (msnv_inflater_kernel_ms) summed over the
             batches -> inflated GB/s, and the call's wall time (staging copies and transfers included) alongside
             (members of all BAMs back to back, so that a batch may hold several files, as a member queue shared by
             the readers of one program would)
  bench      one plain `python bench.py` line, whose e2e pass inflates on the host
The arms alternate, --repeats times each. Writes one JSON line per measurement to --out, each with the card's name and
power limit read in the same call.

  python tools/inflate_compare.py --out profiles/r04_inflate_kernel.jsonl
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from metasnv_b200 import abi  # noqa: E402
from metasnv_b200 import harness as H  # noqa: E402
from metasnv_b200.paths import bin_path  # noqa: E402


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()
    name, power = [x.strip() for x in out[0].split(",")]
    return name, power


def bams_of(data):
    return [l.strip() for l in open(os.path.join(data, "all_samples")) if l.strip()]


def kernel_rate(data, batch_bytes=8 << 20):
    import numpy as np
    comps, ms, coff, ooff = [], [], 0, 0
    for b in bams_of(data):
        c, m = abi.bgzf_members(b)
        m["coff"] += coff
        m["ooff"] += ooff
        comps.append(c)
        ms.append(m)
        coff += c.size
        ooff += int(m["isize"].sum())
    batches = abi.bgzf_batches(np.concatenate(comps), np.concatenate(ms), batch_bytes)
    with abi.Inflater(0, batch_bytes) as inf:
        for c, m in batches[:8]:                        # warm-up
            inf.inflate(c, m)
        ms, wall, nbytes, members, bad = 0.0, 0.0, 0, 0, 0
        for c, m in batches:
            t0 = time.perf_counter()
            _, st = inf.inflate(c, m)
            wall += time.perf_counter() - t0
            ms += inf.kernel_ms()
            nbytes += int(m["isize"].sum())
            members += len(m)
            bad += int((st != 0).sum())
    return {"members": members, "batches": len(batches), "inflated_bytes": nbytes, "kernel_s": ms / 1e3, "call_wall_s": wall,
            "kernel_GBps": nbytes / (ms / 1e3) / 1e9, "call_GBps": nbytes / wall / 1e9, "members_refused": bad}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--set", default="c2:0.057:1000", help="preset:scale:samples (bench.py's e2e set)")
    ap.add_argument("--batch-mb", default="8,64,256", help="device batch sizes to time, MiB")
    a = ap.parse_args()
    name, power = gpu_info()
    work = tempfile.mkdtemp(prefix="msnv_inflate_cmp_")
    out = open(a.out, "a")

    def emit(rec):
        rec.update({"gpu": name, "power_limit": power, "host_cores": os.cpu_count()})
        out.write(json.dumps(rec) + "\n")
        out.flush()
        print(json.dumps(rec), flush=True)
    try:
        p, s, n = a.set.split(":")
        d = os.path.join(work, "set")
        H.synth(d, p, float(s), int(n))
        bam_bytes = sum(os.path.getsize(b) for b in bams_of(d))
        for rep in range(a.repeats):
            for mb in (int(x) for x in a.batch_mb.split(",")):
                emit(dict(kind="kernel", set=a.set, bam_bytes=bam_bytes, batch_mb=mb, rep=rep, **kernel_rate(d, mb << 20)))
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")], capture_output=True, text=True)
        line = [l for l in r.stdout.splitlines() if l.startswith("{")]
        emit(dict(kind="bench", rc=r.returncode, result=json.loads(line[-1]) if line else None, stderr=r.stderr[-1000:] if r.returncode else ""))
    finally:
        shutil.rmtree(work, ignore_errors=True)


if __name__ == "__main__":
    main()
