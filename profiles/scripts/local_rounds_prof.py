"""Local BA with outlier rounds (lorb_ba_local_rounds_batched): time against the plain solves.

All runs: 2 rounds of 5 + 10 LM iterations (Huber sqrt(5.991) in round 0), octave weights, 10 % gross
outliers (robust_cases._move), every solve running its full budget (tolerances off).
    1. config-3 window (10 cameras, 5000 points): one rounds call against two lorb_ba_local calls with
       the same budgets (5 iterations under Huber, then 10 plain)
    2. 512 config-4 windows (10 cameras, 200 points each), batched: one rounds call against two
       lorb_ba_local_batched calls
    3. a config-5-sized window (200 cameras, 20000 points, work-list path): the same comparison
    4. the per-attempt cost of the weighted instantiation (config 3, one Huber round): the difference of
       a 15-iteration and a 0-iteration call over 15, against lorb_ba_local under the trivial and the
       Huber loss measured the same way
    5. the fixed cost of the 512-window batch: the rounds call and the two plain calls with 0-iteration
       budgets (staging, initial evaluations, weights and classification kernels, copies; no LM attempt)
    6. lorb_ba_local (10 iterations) of this build against an older build (--old-lib), the two
       alternating in one process, on the dense (config 3), privatised (14 cameras) and work-list
       (config-5-sized) paths
Times are CUDA events on the library's stream around the whole call (staging and copies included);
the median of --reps repetitions is reported.  Prints one JSON object; --out also writes it.

    python profiles/scripts/local_rounds_prof.py [--reps 7] [--old-lib PATH] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import local_rounds_cases as lc  # noqa: E402
import robust_cases as rc  # noqa: E402
from lorb_slam_b200 import capi, synth  # noqa: E402


def full_budget(n):
    return capi.ba_options(max_num_iterations=n, function_tolerance=-1.0, parameter_tolerance=0.0,
                           gradient_tolerance=-1.0, max_consecutive_invalid_steps=1 << 30)


def gpu_state():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return dict(zip(q.split(","), (v.strip() for v in r.stdout.strip().split(",")))) if r.returncode == 0 else {}


def timed(ctx, fn, reps):
    st = torch.cuda.ExternalStream(ctx._lib.lorb_ctx_stream(ctx._h), device=torch.device("cuda", 0))
    fn()  # warm-up: module load, cached problem buffers
    out = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(st)
        fn()
        e1.record(st)
        e1.synchronize()
        out.append(e0.elapsed_time(e1))
    return float(np.median(out))


def weights(n, seed):
    return lc.octave_weights(n, seed)


def compare(ctx, pb, batched, reps, iters=(5, 10)):
    """(rounds call ms, two plain calls ms) on one window or a batch."""
    O, F = len(pb["obs_cam"]), len(pb["fix_pt"]) if "fix_pt" in pb else 0
    w, fw = weights(O, 1), weights(F, 2)
    opts = [full_budget(iters[0]), full_budget(iters[1])]
    rounds = capi.local_rounds_options()
    ctx.ba_set_loss(*lc.HUBER)
    if batched:
        run_rounds = lambda: ctx.ba_local_rounds_batched(pb, w, fw, rounds, opts)  # noqa: E731
        plain = lambda o: ctx.ba_local_batched(pb, o)  # noqa: E731
    else:
        run_rounds = lambda: ctx.ba_local_rounds(pb, w, fw, rounds, opts)  # noqa: E731
        plain = lambda o: ctx.ba_local(pb, o)  # noqa: E731

    def two_plain():
        ctx.ba_set_loss(*lc.HUBER)
        plain(opts[0])
        ctx.ba_set_loss(capi.LOSS_TRIVIAL)
        plain(opts[1])
    t_rounds = timed(ctx, run_rounds, reps)
    t_plain = timed(ctx, two_plain, reps)
    ctx.ba_set_loss(capi.LOSS_TRIVIAL)
    return t_rounds, t_plain


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--old-lib")
    ap.add_argument("--out")
    a = ap.parse_args()
    ctx = capi.Context(0)
    res = {"gpu": gpu_state(), "rounds": "2 rounds x (5 + 10) LM iterations, Huber sqrt(5.991) in round 0",
           "outliers": 0.1, "reps": a.reps}
    cfg3 = rc.local(0, C=10, P=5000)
    cfg4 = synth.batch_windows([rc.local(1000 + i, C=10, P=200) for i in range(512)])
    cfg5 = rc.local(5, C=200, P=20000, obs_per_point=(6,), traj_len=40.0, fixed_frac=0.1)
    for key, pb, batched in (("config3_window", cfg3, False), ("config4_512_windows", cfg4, True),
                             ("config5_window", cfg5, False)):
        t_r, t_p = compare(ctx, pb, batched, a.reps)
        res[key] = {"rounds_call_ms": t_r, "two_plain_calls_ms": t_p, "ratio": t_r / t_p}
    t_r, t_p = compare(ctx, cfg4, True, a.reps, iters=(0, 0))
    res["config4_512_windows_no_iterations"] = {"rounds_call_ms": t_r, "two_plain_calls_ms": t_p}
    # per LM attempt: full budgets, so every call runs exactly its iterations
    per = {}
    for name, loss in (("plain", None), ("huber", lc.HUBER)):
        ctx.ba_set_loss(*(loss or (capi.LOSS_TRIVIAL,)))
        t15 = timed(ctx, lambda: ctx.ba_local(cfg3, full_budget(15)), a.reps)
        t0 = timed(ctx, lambda: ctx.ba_local(cfg3, full_budget(0)), a.reps)
        per[name] = (t15 - t0) / 15
    ctx.ba_set_loss(*lc.HUBER)
    O, F = len(cfg3["obs_cam"]), cfg3["F"]
    w, fw = weights(O, 1), weights(F, 2)
    r1 = capi.local_rounds_options(n_rounds=1, robust_rounds=1)
    t15 = timed(ctx, lambda: ctx.ba_local_rounds(cfg3, w, fw, r1, [full_budget(15)]), a.reps)
    t0 = timed(ctx, lambda: ctx.ba_local_rounds(cfg3, w, fw, r1, [full_budget(0)]), a.reps)
    per["weighted_huber"] = (t15 - t0) / 15
    ctx.ba_set_loss(capi.LOSS_TRIVIAL)
    res["config3_ms_per_lm_attempt"] = per
    if a.old_lib:
        lib_old = C.CDLL(os.path.abspath(a.old_lib))
        lib_old.lorb_last_error.restype = C.c_char_p
        lib_old.lorb_ctx_stream.restype = C.c_void_p
        lib_old.lorb_ctx_stream.argtypes = [C.c_void_p]
        saved = capi.load_library()
        priv = rc.local(12, C=14, P=5000, obs_per_point=(3, 4, 5), traj_len=5.0, fixed_frac=0.1)
        for key, pb in (("dense_config3", cfg3), ("privatised_14cams", priv), ("work_lists_config5", cfg5)):
            new_t, old_t = [], []
            try:
                for rep in range(a.reps):
                    for which, bucket in ((saved, new_t), (lib_old, old_t)):
                        capi._lib = which
                        c = capi.Context(0)
                        bucket.append(timed(c, lambda: c.ba_local(pb, full_budget(10)), 3))
                        c.close()
            finally:
                capi._lib = saved
            res["lorb_ba_local_10it_ms_" + key] = {"this_build": float(np.median(new_t)),
                                                   "older_build": float(np.median(old_t)),
                                                   "this_build_runs": new_t, "older_build_runs": old_t}
    ctx.close()
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
