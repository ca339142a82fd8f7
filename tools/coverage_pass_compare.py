#!/usr/bin/env python3
"""The coverage pass of a metaSNV project two ways, on one GPU, alternating the arms:
  (a) per BAM, as metaSNV.py:compute_opt runs it: `qaCompute -c 10 -d -i <bam> <proj>/cov/<bam>.cov` for every BAM, in a
      pool of as many processes as the host has cores (every process creates its own CUDA context);
  (b) one `metaSNV_coverage <proj> <all_samples>` (one context).
Both arms run on device 0 (MSNV_DEVICE=0). Each run's cov/ tree is compared byte for byte with the first complete run of
arm (a) (every qaCompute exited 0). Writes one JSON line per run to --out: card name and power limit (read in the same
call), host cores, the data set, wall time, whether the tree is identical (null when no arm (a) run was complete), arm (b)'s
MSNV_PERF_JSON record, and the stderr of any process that failed.

  python tools/coverage_pass_compare.py --preset c1 --scale 0.5 --out profiles/r03_coverage_pass_c1.jsonl
  python tools/coverage_pass_compare.py --preset c2 --scale 0.057 --out profiles/r03_coverage_pass_c2.jsonl
"""
import argparse
import concurrent.futures
import filecmp
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from metasnv_b200 import harness as H  # noqa: E402
from metasnv_b200.paths import bin_path  # noqa: E402


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()
    name, power = [x.strip() for x in out[0].split(",")]
    return name, power


def arm_per_bam(proj, bams, cores, env):
    os.makedirs(os.path.join(proj, "cov"))

    def one(b):
        return subprocess.run([bin_path("qaCompute"), "-c", "10", "-d", "-i", b,
                               os.path.join(proj, "cov", os.path.basename(b) + ".cov")], capture_output=True, text=True, env=env)
    with concurrent.futures.ThreadPoolExecutor(max_workers=cores) as pool:
        runs = list(zip(bams, pool.map(one, bams)))
    failed = [{"bam": b, "rc": r.returncode, "stderr": r.stderr.strip()[-500:]} for b, r in runs if r.returncode != 0]
    return (1 if failed else 0), {"failed": failed}


def arm_one_process(proj, all_samples, env, perf):
    r = subprocess.run([bin_path("metaSNV_coverage"), proj, all_samples], capture_output=True, text=True,
                       env=dict(env, MSNV_PERF_JSON=perf))
    rec = json.loads(open(perf).read().splitlines()[-1]) if os.path.exists(perf) else {}
    if r.returncode != 0:
        rec["stderr"] = r.stderr.strip()[-2000:]
    return r.returncode, rec


def same_tree(a, b):
    fa, fb = sorted(os.listdir(a)), sorted(os.listdir(b))
    return fa == fb and all(filecmp.cmp(os.path.join(a, f), os.path.join(b, f), shallow=False) for f in fa)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--preset", required=True)
    ap.add_argument("--scale", type=float, required=True)
    ap.add_argument("--samples", type=int, default=0)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()

    gpu, power = gpu_info()
    cores = os.cpu_count()
    env = dict(os.environ, MSNV_DEVICE="0")
    work = tempfile.mkdtemp(prefix="covpass_")
    try:
        data = os.path.join(work, "data")
        t = time.time()
        st = H.synth(data, args.preset, args.scale, args.samples, threads=cores)
        synth_s = time.time() - t
        lst = os.path.join(data, "all_samples")
        bams = [l.strip() for l in open(lst) if l.strip()]
        bam_bytes = sum(os.path.getsize(b) for b in bams)
        base = {"gpu": gpu, "power_limit": power, "host_cores": cores, "preset": args.preset, "scale": args.scale,
                "bams": len(bams), "bam_bytes": bam_bytes, "reads": st["reads"], "synth_s": round(synth_s, 3)}
        print(json.dumps(base), flush=True)
        ref, pending = None, []          # runs not yet written: those before the first complete run of arm (a)
        with open(args.out, "a") as out:
            for rep in range(args.reps):
                for arm in (("a", "b") if rep % 2 == 0 else ("b", "a")):
                    proj = os.path.join(work, "proj_%s%d" % (arm, rep))
                    t = time.time()
                    if arm == "a":
                        rc, perf = arm_per_bam(proj, bams, cores, env)
                    else:
                        rc, perf = arm_one_process(proj, lst, env, os.path.join(work, "perf_%d.jsonl" % rep))
                    wall = time.time() - t
                    rec = dict(base, arm={"a": "qaCompute per BAM, %d processes at a time" % cores,
                                          "b": "one metaSNV_coverage"}[arm], rep=rep, rc=rc, wall_s=round(wall, 3), perf=perf)
                    print(json.dumps(rec), flush=True)
                    tree = os.path.join(proj, "cov")
                    if ref is None and arm == "a" and rc == 0:
                        ref = tree
                    pending.append((tree, rec))
                    if ref is None:
                        continue
                    for tr, rc_rec in pending:       # written as soon as they can be compared, so that a cut run keeps them
                        rc_rec["identical_to_first_complete_per_bam_tree"] = same_tree(ref, tr)
                        out.write(json.dumps(rc_rec) + "\n")
                        out.flush()
                        if tr != ref:
                            shutil.rmtree(os.path.dirname(tr))
                    pending = []
            for tr, rc_rec in pending:
                rc_rec["identical_to_first_complete_per_bam_tree"] = None
                out.write(json.dumps(rc_rec) + "\n")
            if ref is None:
                print("no run of arm (a) completed: nothing was compared", file=sys.stderr)
    finally:
        shutil.rmtree(work, ignore_errors=True)


if __name__ == "__main__":
    main()
