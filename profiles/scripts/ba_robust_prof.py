"""Cost of the robust losses in the BA solvers: trivial vs Huber vs Cauchy, ms per LM attempt and the
overhead over the trivial loss in %, on
    pose-only, n = 2000 (lorb_ba_pose_only, host buffers)
    BASELINE config 3 (10 keyframes, 5 000 points, resident problem, dense DMMA build)
    BASELINE config 4 (512 windows of config 3, one resident batch)
    BASELINE config 5 (200 keyframes, 200 000 points, 1.5 M observations, large path)
Every solve runs a fixed number of LM attempts (tolerances off), timed with CUDA events on the
library's stream as bench.py does; the three losses alternate inside each repetition and the median
of the repetitions is reported.  Inputs carry 10 % gross outliers (20-80 px), so the Huber and Cauchy
weights are not all 1.  Prints one JSON object; --out also writes it to a file.

    python profiles/scripts/ba_robust_prof.py [--reps 5] [--windows 512] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import robust_cases as rc  # noqa: E402
from lorb_slam_b200 import capi, synth  # noqa: E402

LOSSES = (("trivial", capi.LOSS_TRIVIAL), ("huber", capi.LOSS_HUBER), ("cauchy", capi.LOSS_CAUCHY))


def fixed_iters(n):
    # parameter_tolerance 0, not -1: the test is |step| <= tol (|x| + tol), which -1 turns true for |x| < 1
    return capi.ba_options(max_num_iterations=n, function_tolerance=-1.0, parameter_tolerance=0.0,
                           gradient_tolerance=-1.0, max_consecutive_invalid_steps=1 << 30)


def gpu_state():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks.mem"
    r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return dict(zip(q.split(","), (v.strip() for v in r.stdout.strip().split(",")))) if r.returncode == 0 else {}


def timed(ctx, run, iters, steps):
    """ms per LM attempt of `steps` calls of run() (each returns the summary or summaries)."""
    st = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", 0))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx.sync()
    e0.record(st)
    for _ in range(steps):
        s = run()
    e1.record(st)
    ctx.sync()
    s = s if isinstance(s, list) else [s]
    assert all(x["iterations"] == iters for x in s), s[0]
    return e0.elapsed_time(e1) / (steps * iters)


def measure(ctx, name, run, iters, steps, reps):
    ms = {k: [] for k, _ in LOSSES}
    for kind_name, kind in LOSSES:  # warm-up: module loads, cached buffers, every instantiation
        ctx.ba_set_loss(kind, rc.SCALE)
        run()
    for _ in range(reps):
        for kind_name, kind in LOSSES:
            ctx.ba_set_loss(kind, rc.SCALE)
            ms[kind_name].append(timed(ctx, run, iters, steps))
    ctx.ba_set_loss(capi.LOSS_TRIVIAL)
    med = {k: float(np.median(v)) for k, v in ms.items()}
    row = {"ms_per_lm_attempt": med, "runs_ms": ms,
           "overhead_pct": {k: 100.0 * (med[k] / med["trivial"] - 1.0) for k in med if k != "trivial"}}
    print(name, json.dumps(row["ms_per_lm_attempt"]), json.dumps(row["overhead_pct"]), flush=True)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--windows", type=int, default=512)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ba_robust_prof: needs a CUDA device")
    out = {"gpu_before": gpu_state(), "scale_px": rc.SCALE, "outlier_fraction": 0.1}
    ctx = capi.Context(0)

    po = rc.pose_only(0, 2000)
    opt = fixed_iters(10)
    out["pose_only_n2000"] = measure(
        ctx, "pose_only_n2000", lambda: ctx.ba_pose_only(po["xw"], po["uv"], po["K"], po["rt"], opt)[1], 10, 50, a.reps)

    pb = rc.local(0, C=10, P=5000)
    prob = ctx.ba_problem(pb)

    def cfg3():
        prob.reset()
        return prob.solve(opt)
    out["cfg3_10kf_5kpts"] = measure(ctx, "cfg3_10kf_5kpts", cfg3, 10, 10, a.reps)
    prob.close()

    bt = synth.batch_windows([rc.local(i, C=10, P=5000) for i in range(a.windows)])
    probb = ctx.ba_problem_batched(bt)
    opt4 = fixed_iters(4)

    def cfg4():
        probb.reset()
        return probb.solve(opt4)
    out["cfg4_%dwindows" % a.windows] = measure(ctx, "cfg4_%dwindows" % a.windows, cfg4, 4, 2, a.reps)
    probb.close()
    del bt

    pl = rc.local(0, C=200, P=200000, obs_per_point=(7, 8), traj_len=100.0)
    probl = ctx.ba_problem(pl)
    opt5 = fixed_iters(3)

    def cfg5():
        probl.reset()
        return probl.solve(opt5)
    out["cfg5_200kf_200kpts"] = measure(ctx, "cfg5_200kf_200kpts", cfg5, 3, 2, a.reps)
    probl.close()
    ctx.close()
    out["gpu_after"] = gpu_state()
    text = json.dumps(out, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
