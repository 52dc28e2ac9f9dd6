"""Pose-only BA with outlier rounds (lorb_ba_pose_rounds_batched): time and throughput.

    1. one frame, n = 300 / 1000 / 2000, 4 rounds x 10 LM iterations (Huber sqrt(5.991) in rounds
       0-2, octave weights, 20 % gross outliers): device-event time of one rounds call, against four
       sequential lorb_ba_pose_only calls of 10 iterations, and against the C++ reference rounds
       (tests/oracle_ext.py) on one host core
    2. batches of 1 / 64 / 512 / 2048 frames x 1000 observations: frames/s and observation-iterations/s
       (every LM pass visits all observations of its frame, flagged ones are skipped)
    3. lorb_ba_pose_only (n = 2000, 10 iterations) of this build against an older build of the library
       (--old-lib), the two alternating in one process
Every LM solve runs its full iteration budget (tolerances off).  Times are CUDA events on the library's
stream around the whole call (staging copies included); the median of --reps repetitions is reported.
Prints one JSON object; --out also writes it to a file.

    OMP_NUM_THREADS=1 python profiles/scripts/pose_rounds_prof.py [--reps 7] [--old-lib PATH] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

os.environ.setdefault("OMP_NUM_THREADS", "1")  # the reference on one host core
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import oracle_ext as rd  # noqa: E402
from lorb_slam_b200 import capi  # noqa: E402
from oracle import ref  # noqa: E402
from test_oracle_pose_rounds_cpu import planted  # noqa: E402

ITERS, ROUNDS, CHI2 = 10, 4, 5.991


def fixed_opts(mod):
    return mod.ba_options(max_num_iterations=ITERS, function_tolerance=-1.0, parameter_tolerance=0.0,
                          gradient_tolerance=-1.0, max_consecutive_invalid_steps=1 << 30)


def gpu_state():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks.mem"
    r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return dict(zip(q.split(","), (v.strip() for v in r.stdout.strip().split(",")))) if r.returncode == 0 else {}


def event_ms(stream_handle, run, sync, steps=1):
    st = torch.cuda.ExternalStream(stream_handle, device=torch.device("cuda", 0))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync()
    e0.record(st)
    for _ in range(steps):
        run()
    e1.record(st)
    sync()
    return e0.elapsed_time(e1) / steps


def frames(n, count):
    out = [planted(7000 + f, n, 0.2) for f in range(count)]
    return [(po, w) for po, w, _ in out]


def batch(fr, n_frames):
    pick = [fr[f % len(fr)] for f in range(n_frames)]
    off = np.arange(n_frames + 1, dtype=np.int32) * len(pick[0][0]["xw"])
    return (off, np.concatenate([p["xw"] for p, _ in pick]), np.concatenate([p["uv"] for p, _ in pick]),
            np.stack([p["rt"] for p, _ in pick]), np.concatenate([w for _, w in pick]))


def single_frame(ctx, reps):
    opt, rounds = fixed_opts(capi), capi.pose_rounds_options()
    rows = {}
    for n in (300, 1000, 2000):
        po, w = frames(n, 1)[0]
        ctx.ba_set_loss(capi.LOSS_HUBER, float(np.sqrt(CHI2)))
        g = ctx.ba_pose_rounds(po["xw"], po["uv"], po["K"], po["rt"], info=w, rounds=rounds, opt=opt)
        assert g[4] == ROUNDS and all(s["iterations"] == ITERS for s in g[5]), g[5]
        r_ms, p_ms, c_ms = [], [], []
        for _ in range(reps):
            ctx.ba_set_loss(capi.LOSS_HUBER, float(np.sqrt(CHI2)))
            r_ms.append(event_ms(ctx.stream, lambda: ctx.ba_pose_rounds(po["xw"], po["uv"], po["K"], po["rt"], info=w,
                                                                          rounds=rounds, opt=opt), ctx.sync))

            def four():  # the same work as four separate pose-only solves (no weights, no masks)
                for r in range(ROUNDS):
                    ctx.ba_set_loss(capi.LOSS_HUBER if r < 3 else capi.LOSS_TRIVIAL, float(np.sqrt(CHI2)))
                    ctx.ba_pose_only(po["xw"], po["uv"], po["K"], po["rt"], opt)
            p_ms.append(event_ms(ctx.stream, four, ctx.sync))
            t = time.perf_counter()
            o = rd.ba_pose_rounds(po["xw"], po["uv"], po["K"], po["rt"], w, opt=fixed_opts(ref),
                                  loss=(rd.LOSS_HUBER, float(np.sqrt(CHI2))))
            c_ms.append(1e3 * (time.perf_counter() - t))
        assert o[4] == ROUNDS
        med = lambda v: float(np.median(v))
        rows["n%d" % n] = {"rounds_call_ms": med(r_ms), "four_pose_only_calls_ms": med(p_ms),
                           "cpp_reference_one_core_ms": med(c_ms), "runs_rounds_ms": r_ms,
                           "runs_four_pose_only_ms": p_ms, "runs_cpp_ms": c_ms,
                           "speedup_vs_four_calls": med(p_ms) / med(r_ms), "speedup_vs_cpp": med(c_ms) / med(r_ms)}
        print("single n=%d" % n, json.dumps({k: v for k, v in rows["n%d" % n].items() if not k.startswith("runs")}),
              flush=True)
    ctx.ba_set_loss(capi.LOSS_TRIVIAL)
    return rows


def batched(ctx, reps):
    opt, rounds = fixed_opts(capi), capi.pose_rounds_options()
    fr = frames(1000, 64)
    rows = {}
    ctx.ba_set_loss(capi.LOSS_HUBER, float(np.sqrt(CHI2)))
    for nf in (1, 64, 512, 2048):
        off, xw, uv, rt, w = batch(fr, nf)
        B = ctx.ba_pose_rounds_batched(off, xw, uv, fr[0][0]["K"], rt, info=w, rounds=rounds, opt=opt)
        assert (B[4] == ROUNDS).all()
        obs_iters = sum(1000 * s["iterations"] for f in B[5] for s in f)
        ms = [event_ms(ctx.stream, lambda: ctx.ba_pose_rounds_batched(off, xw, uv, fr[0][0]["K"], rt, info=w,
                                                                       rounds=rounds, opt=opt), ctx.sync)
              for _ in range(reps)]
        m = float(np.median(ms))
        rows["frames%d" % nf] = {"call_ms": m, "frames_per_s": nf / (m * 1e-3),
                                 "obs_iterations_per_s": obs_iters / (m * 1e-3), "runs_ms": ms}
        print("batch %d" % nf, json.dumps({k: v for k, v in rows["frames%d" % nf].items() if k != "runs_ms"}),
              flush=True)
    ctx.ba_set_loss(capi.LOSS_TRIVIAL)
    return rows


class RawLib:
    """lorb_ctx_create / lorb_ba_pose_only of one build of the library, loaded on its own."""

    def __init__(self, path):
        self.lib = C.CDLL(path)
        self.lib.lorb_ctx_stream.restype = C.c_void_p
        self.lib.lorb_ctx_stream.argtypes = [C.c_void_p]
        self.h = C.c_void_p()
        assert self.lib.lorb_ctx_create(0, C.byref(self.h)) == 0
        self.stream = self.lib.lorb_ctx_stream(self.h)

    def pose_only(self, po, opt):
        rt, s = po["rt"].copy(), capi.BASummary()
        P = lambda a: a.ctypes.data_as(C.c_void_p)
        assert self.lib.lorb_ba_pose_only(self.h, len(po["xw"]), P(po["xw"]), P(po["uv"]), P(po["K"]), P(rt),
                                          C.byref(opt), C.byref(s)) == 0
        return rt, s

    def sync(self):
        self.lib.lorb_ctx_sync(self.h)


def old_vs_new(old_path, reps):
    po, _ = frames(2000, 1)[0]
    opt = fixed_opts(capi)
    libs = {"new": RawLib(capi.LIB_PATH), "old": RawLib(old_path)}
    out = {k: [] for k in libs}
    res = {k: lib.pose_only(po, opt) for k, lib in libs.items()}
    assert np.array_equal(res["new"][0], res["old"][0]), "old and new builds disagree"
    for _ in range(reps):
        for k, lib in libs.items():
            out[k].append(event_ms(lib.stream, lambda: lib.pose_only(po, opt), lib.sync, steps=50))
    med = {k: float(np.median(v)) for k, v in out.items()}
    row = {"pose_only_n2000_10iters_ms": med, "runs_ms": out, "change_pct": 100.0 * (med["new"] / med["old"] - 1.0),
           "spread_pct": {k: 100.0 * (max(v) - min(v)) / med[k] for k, v in out.items()}}
    print("old_vs_new", json.dumps({k: v for k, v in row.items() if k != "runs_ms"}), flush=True)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--old-lib", default=None, help="liblorb_cuda.so of the build to compare lorb_ba_pose_only with")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("pose_rounds_prof: needs a CUDA device")
    out = {"gpu_before": gpu_state(), "iterations_per_round": ITERS, "rounds": ROUNDS, "outlier_fraction": 0.2}
    ctx = capi.Context(0)
    out["single_frame"] = single_frame(ctx, a.reps)
    out["batched_1000obs"] = batched(ctx, a.reps)
    ctx.close()
    if a.old_lib:
        out["pose_only_old_vs_new"] = old_vs_new(a.old_lib, a.reps)
    out["gpu_after"] = gpu_state()
    text = json.dumps(out, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
