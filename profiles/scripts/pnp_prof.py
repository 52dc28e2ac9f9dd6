"""Batched P3P RANSAC (lorb_pnp_ransac_batched): time and throughput.

Two cases, 300 hypotheses each, 40 % mismatches, octave weights:
  reloc    30 problems x 300 correspondences: one relocalisation over 30 candidate keyframes
  offline  4096 problems x 1000 correspondences: offline re-tracking of many frames
Reported per case: ms per call (host clock around the whole call, which ends in a stream synchronise; it
includes the upload and download), problems/s and hypothesis x correspondence evaluations/s.  The roofline
line counts the fp64 operations of one evaluation from pnp_math.cuh::reproj2 and the inlier test and sets
them against lorb_microbench_fp64 (kind 0, scalar DFMA).  The CPU baseline is cv2.solvePnPRansac(SOLVEPNP_P3P,
300 iterations, reprojectionError sqrt(5.991)) over the box's host threads: different work (it refines the
best model and stops early once its confidence is reached), labelled as such.  The device results of the
reloc case are checked against the host restatement (tests/pnp_ref.py).

    python profiles/scripts/pnp_prof.py [--reps 5] [--out FILE]
"""
import argparse
import concurrent.futures as cf
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from lorb_slam_b200 import capi, synth  # noqa: E402

# one evaluation (pnp_math.cuh::reproj2 + the inlier test of pnp_score_kernel): R X + t is 9 mul + 9 add, then
# 1 division (1 / z), 2 x (2 mul + 2 add) for the two residuals, 2 mul + 1 add for |r|^2, 1 mul for w |r|^2
EVAL_ADD_MUL = 9 + 9 + 8 + 3 + 1
EVAL_DIV = 1


def gpu_state():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return dict(zip(q.split(","), (v.strip() for v in r.stdout.strip().split(",")))) if r.returncode == 0 else {}


def time_call(ctx, d, reps):
    run = lambda: ctx.pnp_ransac_batched(d["corr_off"], d["xw"], d["uv"], d["K"], info=d["info"])
    run()  # warm-up: scratch growth, module load
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        run()
        ts.append(1e3 * (time.perf_counter() - t0))
    return ts, run()


def cpu_baseline(d, n_problems):
    K = d["K"].astype(np.float64)
    Km = np.array([[K[0], 0, K[2]], [0, K[1], K[3]], [0, 0, 1]])
    off = d["corr_off"]

    def one(b):
        a, e = off[b], off[b + 1]
        return cv2.solvePnPRansac(d["xw"][a:e].astype(np.float64), d["uv"][a:e].astype(np.float64), Km, None,
                                  flags=cv2.SOLVEPNP_P3P, iterationsCount=300, reprojectionError=float(np.sqrt(5.991)))
    threads = os.cpu_count()
    t0 = time.perf_counter()
    with cf.ThreadPoolExecutor(threads) as ex:
        list(ex.map(one, range(n_problems)))
    dt = time.perf_counter() - t0
    return {"problems": n_problems, "threads": threads, "ms": 1e3 * dt, "problems_per_s": n_problems / dt,
            "note": "cv2.solvePnPRansac, SOLVEPNP_P3P, 300 iterations: refines and stops adaptively (different work)"}


def main():
    global cv2
    import cv2
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    out = {"gpu_before": gpu_state(), "hypotheses": 300, "outlier_fraction": 0.4,
           "fp64_ops_per_evaluation": {"add_mul": EVAL_ADD_MUL, "div": EVAL_DIV}}
    with capi.Context(0) as ctx:
        peak = ctx.microbench_fp64(0)
        out["fp64_dfma_flop_per_s"] = peak
        for name, B, n, cpu_n in (("reloc", 30, 300, 30), ("offline", 4096, 1000, 512)):
            d = synth.make_pnp_problems(1, n=n, n_problems=B, outlier_frac=0.4)
            ts, res = time_call(ctx, d, a.reps)
            ms = float(np.median(ts))
            evals = B * n * 300
            # the add/mul count over the DFMA instruction rate (peak flop / 2); the division costs more than one
            # instruction, so this bound is optimistic
            bound_s = evals * (EVAL_ADD_MUL + EVAL_DIV) / (peak / 2)
            row = {"problems": B, "correspondences": n, "ms_per_call": ms, "runs_ms": ts,
                   "problems_per_s": B / (ms * 1e-3), "evaluations_per_s": evals / (ms * 1e-3),
                   "fp64_bound_ms": 1e3 * bound_s, "share_of_fp64_bound": 1e3 * bound_s / ms,
                   "mean_inliers": float(np.mean(res[2]))}
            if name == "reloc":
                import pnp_ref as pr
                o = pr.ransac(d["corr_off"], d["xw"], d["uv"], d["K"], d["info"])
                row["parity_with_reference"] = bool(np.array_equal(res[1], o[1]) and np.array_equal(res[3], o[3])
                                                    and np.abs(res[0] - o[0]).max() <= 1e-12)
            row["cpu_baseline"] = cpu_baseline(d, cpu_n)
            if cpu_n < B:
                row["cpu_baseline"]["note"] += "; timed on the first %d problems" % cpu_n
            out[name] = row
            print(name, json.dumps({k: v for k, v in row.items() if k != "runs_ms"}), flush=True)
    out["gpu_after"] = gpu_state()
    js = json.dumps(out, indent=1)
    print(js)
    if a.out:
        with open(a.out, "w") as f:
            f.write(js + "\n")


if __name__ == "__main__":
    main()
