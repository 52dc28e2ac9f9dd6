#!/usr/bin/env python
"""bench.py — headline benchmark of the LORB-SLAM hot path on B200.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload NAME] [--dump-outputs DIR]

The default line carries all three BASELINE metrics: the keyframe-pair sweep is the top-level
record (descriptor-pairs/s); `ba_batched` (config 4: 512 windows split over the ranks) and
`ba_large` (config 5: 200 keyframes / 200k points / 1.5M observations, points sharded over the
ranks, NCCL all-reduce of the reduced camera system) are sub-objects with their own value, e2e,
roofline, cpu_baseline and an in-run parity check.  `--impl reference` prints the same structure
measured on the CPU path.

Headline workload (default, `sweep`): BASELINE.json config 5's keyframe-pair
matching sweep — a bank of 4096 keyframes x 2000 ORB descriptors (262 MB, larger
than the 126 MB L2) resident in HBM.  One step = every pair among one block of
128 consecutive keyframes (8128 keyframe pairs x 2000 x 2000 descriptor pairs),
a different block every step; rank r of N takes blocks r, r+N, ... (weak
scaling: per-GPU work fixed, no data-path collective).  metric =
descriptor-pairs/s (cross-checked Hamming match incl. the max(2*minDist,30)
filter), exact same result as the reference's BFMatcher path.

  value  whole-job pairs/s, bank and pair plan already in HBM, CUDA events on the
         library's stream, max over ranks.
  e2e    same step through the host-buffer C-ABI call (lorb_match_sweep): pinned
         host descriptors -> H2D -> kernels -> D2H of the per-pair results.

Other workloads (`--workload ba_batched | ba_large | ba_local | bf | proj`) put
another BASELINE config under the same contract; their short versions are also
reported in `extra` of the default line.

`--steps` sets the timed steps of the sweep and of both BA legs; the short `extra`
measurements keep their own fixed repetition counts.

`--dump-outputs DIR` writes, after the timed steps, what rank 0's last timed step of
every workload that ran handed back to its caller, as DIR/<name>.npy (integers as
float64): on several GPUs that is rank 0's block, window slice and point shard only.
An array above its share of 64 MB is cut to a fixed, seeded sample of its rows.  The inputs are seeded, so two builds run with the same arguments can be
compared output for output.  The sweep outputs are exact.  The BA outputs compare
to a tolerance: their partial sums are accumulated with atomics in no fixed order,
and the forced attempts past convergence accept or reject on that rounding noise,
so the trust-region radius and step counts of the BA summaries may differ.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_KF, N_DESC, BLOCK_KF = 4096, 2000, 128
PAIRS_PER_KF_PAIR = N_DESC * N_DESC


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def _tensor_peaks():
    """(bf16 dense TFLOP/s burst, sustained, source) from the driver-written MEASURED_PEAKS.json."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        if "bf16_tflops" in d:
            return (float(d["bf16_tflops"]), float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                    "measured (MEASURED_PEAKS.json: cuBLAS bf16 8192^3)")
    return 1640.0, 1390.0, "fallback (B200_PROFILING.md)"


def _rank_host_threads(world):
    """This rank's share of the host cores for the library's staging loops.  The oracle and the library
    share one OpenMP runtime, so every oracle leg that asks for all cores (rank 0's parity checks and CPU
    baselines) must be followed by this call again -- or rank 0 stages its e2e batches on every core of the
    box while the other ranks use their shares, and the max over the ranks is rank 0 fighting them."""
    from lorb_slam_b200 import capi
    capi.set_host_threads(int(os.environ.get("LORB_BENCH_HOST_THREADS", 0)) or
                          max(1, (os.cpu_count() or 1) // max(1, world)))


def _profile_traffic(key):
    """dram bytes per launch of a kernel from the committed ncu summary of this round, with its
    provenance; (None, None) when no capture has been committed for it."""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(p):
        d = json.load(open(p)).get(key)
        if d:
            return d.get("dram_bytes_per_launch"), d.get("source")
    return None, None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1]))
                smax = float(r[2])
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if r[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        # median of the upper half = clock under load (the sampler also sees idle edges)
        sm.sort()
        load = sm[len(sm) // 2:] if sm else []
        med = load[len(load) // 2] if load else None
        return {"sm_mhz": med, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


def _dist_setup(n_gpus):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, local


def _barrier(world):
    import torch
    import torch.distributed as dist
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def _max_over_ranks(x, world, local):
    import torch
    import torch.distributed as dist
    if world == 1:
        return x
    t = torch.tensor([x], dtype=torch.float64, device=torch.device("cuda", local))
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def _sum_over_ranks(x, world, local):
    import torch
    import torch.distributed as dist
    if world == 1:
        return x
    t = torch.tensor([x], dtype=torch.float64, device=torch.device("cuda", local))
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t.item())


def _events(ctx, local):
    import torch
    st = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", local))
    return st, torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


OUTPUTS = {}  # name -> what rank 0's last timed step returned (see --dump-outputs)
DUMP_BYTES = 64 * 10 ** 6
BA_SUMMARY_FIELDS = ("initial_cost", "final_cost", "final_radius", "final_gradient_max_norm", "iterations",
                     "num_successful_steps", "num_unsuccessful_steps", "termination")


def _ba_summary_rows(sums):
    return np.array([[s[k] for k in BA_SUMMARY_FIELDS] for s in sums], np.float64)


def write_outputs(out_dir):
    """OUTPUTS as out_dir/<name>.npy: float32 stays float32, everything else becomes float64.  Smallest
    first, every array gets an even share of what is left of DUMP_BYTES (what a small one does not use
    goes to the larger ones); an array above its share keeps a fixed, seeded sample of its rows (in row
    order)."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {name: np.ascontiguousarray(a, np.float32 if a.dtype == np.float32 else np.float64)
              for name, a in OUTPUTS.items()}
    left = DUMP_BYTES
    for k, name in enumerate(sorted(arrays, key=lambda n: arrays[n].nbytes)):
        a = arrays[name]
        share = left // (len(arrays) - k) - 1024  # room for the .npy header
        if a.nbytes > share:
            rows = np.random.default_rng(0).choice(len(a), share // (a.nbytes // len(a)), replace=False)
            a = a[np.sort(rows)]
        np.save(os.path.join(out_dir, name + ".npy"), a)
        left -= a.nbytes + 1024


# ----------------------------------------------------------------------- sweep
def _block_pairs():
    a, b = np.triu_indices(BLOCK_KF, k=1)
    return a.astype(np.int32), b.astype(np.int32)


def _make_bank(seed=0):
    rng = np.random.default_rng(seed)
    return rng.integers(0, 256, size=(N_KF, N_DESC, 32), dtype=np.uint8)


def _cpu_sweepers(bank_block):
    """-> [(kind, description, run(pa, pb), set_threads)], the reference's own compiled code first.

    "reference" = oracle/_ref: Matcher::SearchByProjection(curr, prev) of /root/reference's
    src/matcher.cpp compiled unmodified (descriptor gathering, minDist / max(2*minDist,30) filter)
    over the OpenCV stand-in's BFMatcher, OpenMP over keyframe pairs (the reference is
    single-threaded; OpenCV-C++ is not in the image).  "port" = oracle/match_ref.c."""
    from oracle import ref, reflib
    out = []
    if reflib.available():
        sw = reflib.Sweep(bank_block)
        out.append(("reference", "oracle/_ref (reference src/matcher.cpp compiled unmodified, -O2 -mpopcnt, "
                    "OpenCV stand-in BFMatcher), OpenMP over pairs", sw.run))
    out.append(("port", "oracle/match_ref.c -O2 -mpopcnt, OpenMP over pairs",
                lambda pa, pb: ref.sweep(bank_block, pa, pb)))
    return out


def cpu_baseline_sweep(bank, target_s=12.0):
    """The reference's CPU path on a bounded sample of the same workload, all host threads."""
    from oracle import ref
    cores = os.cpu_count() or 1
    cores = ref.set_num_threads(cores)  # one libgomp: also sets the team size of oracle/_ref
    pa, pb = _block_pairs()
    res = []
    for kind, desc, run in _cpu_sweepers(bank[:BLOCK_KF]):
        n0 = max(cores, 8)
        t0 = time.time()
        run(pa[:n0], pb[:n0])
        dt = time.time() - t0
        n = int(min(len(pa), max(n0, n0 * target_s / max(dt, 1e-3))))
        t0 = time.time()
        run(pa[:n], pb[:n])
        dt = time.time() - t0
        res.append({"value": n * PAIRS_PER_KF_PAIR / dt, "unit": "descriptor-pairs/s", "cores": cores,
                    "kind": kind,
                    "sample": "%d keyframe pairs (2000x2000 each) of the first block, %s" % (n, desc)})
    out = res[0]
    if len(res) > 1:
        out["port_value"] = res[1]["value"]
        out["port_sample"] = res[1]["sample"]
    try:  # the library routine the reference itself calls, for context
        import cv2
        cv2.setNumThreads(cores)
        m = cv2.BFMatcher(cv2.NORM_HAMMING, True)
        t0 = time.time()
        reps = 6
        for i in range(reps):
            m.match(bank[pa[i]], bank[pb[i]])
        out["cv2_bfmatcher_value"] = reps * PAIRS_PER_KF_PAIR / (time.time() - t0)
        out["cv2_threads"] = cores
    except Exception:
        pass
    return out



def run_sweep(args, rank, world, local):
    import torch
    from lorb_slam_b200 import capi
    ctx = capi.Context(local)
    ctx.sweep_set_impl(args.sweep_impl)
    tensor = args.sweep_impl == "tensor"
    bank = _make_bank(0)
    n_blocks = N_KF // BLOCK_KF
    pa, pb = _block_pairs()
    n_pairs = len(pa)
    ctx.bank_upload(bank)
    ctx.sweep_plan_upload(pa, pb)
    my_blocks = [(rank + i * world) % n_blocks for i in range(args.warmup + args.steps)]
    st, ev0, ev1 = _events(ctx, local)
    for i in range(args.warmup):
        ctx.sweep_plan_run(my_blocks[i] * BLOCK_KF)
    ctx.sync()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    _barrier(world)
    l0 = ctx.launch_count
    ev0.record(st)
    for i in range(args.steps):
        ctx.sweep_plan_run(my_blocks[args.warmup + i] * BLOCK_KF)
    ev1.record(st)
    ctx.sync()
    _barrier(world)
    launches = ctx.launch_count - l0
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if rank == 0 else None
    ms_max = _max_over_ranks(ms, world, local)
    step_ms = ms / args.steps
    kept_dev, matches_dev, min_dist_dev = ctx.sweep_plan_download()
    if rank == 0:
        OUTPUTS.update(sweep_kept=kept_dev, sweep_matches=matches_dev, sweep_min_dist=min_dist_dev)
    # the dominant kernel alone (the tensor form adds a small finalize kernel per step)
    kernel_ms = step_ms
    if tensor and rank == 0:
        ctx.profile(True)
        for i in range(min(3, args.steps)):
            ctx.sweep_plan_run(my_blocks[args.warmup + i] * BLOCK_KF)
        tot, cnt = ctx.profile_read(3)
        ctx.profile(False)
        if cnt:
            kernel_ms = tot / cnt

    # ---- e2e through the host-buffer entry point, pinned host inputs
    pinned = torch.empty((BLOCK_KF, N_DESC, 32), dtype=torch.uint8).pin_memory()
    host_blk = pinned.numpy()
    e2e_steps = args.steps
    for i in range(min(2, args.warmup)):
        host_blk[...] = bank[my_blocks[i] * BLOCK_KF:(my_blocks[i] + 1) * BLOCK_KF]
        ctx.match_sweep(host_blk, pa, pb)
    _barrier(world)
    t_e2e = 0.0
    kept_e2e = None
    for i in range(e2e_steps):
        b = my_blocks[args.warmup + i]
        host_blk[...] = bank[b * BLOCK_KF:(b + 1) * BLOCK_KF]  # staging of the step's input (untimed)
        t0 = time.perf_counter()
        kept_e2e, _, _ = ctx.match_sweep(host_blk, pa, pb)
        t_e2e += time.perf_counter() - t0
    assert np.array_equal(kept_e2e, kept_dev), "device-resident and host-buffer paths disagree"
    e2e_max = _max_over_ranks(t_e2e, world, local)
    total_pairs = float(world) * args.steps * n_pairs * PAIRS_PER_KF_PAIR
    value = total_pairs / (ms_max * 1e-3)
    e2e_value = total_pairs / e2e_max

    res = None
    if rank == 0:
        hbm_peak, peak_src = _peaks()
        pairs_per_launch = n_pairs * PAIRS_PER_KF_PAIR
        sm_max = (clocks or {}).get("sm_max_mhz") or 1965.0
        sm_count = torch.cuda.get_device_properties(local).multi_processor_count
        ctx.bank_upload(bank[:BLOCK_KF])  # small bank is enough for the micro-benchmarks
        if tensor:
            burst, sustained, tsrc = _tensor_peaks()
            mb = ctx.microbench_tensor_i8(4096)
            ops = pairs_per_launch * 512.0  # 256 multiply-adds per descriptor pair (the distance)
            traffic, traffic_src = _profile_traffic("tc_sweep_kernel")
            roof = {"bound": "tensor", "kernel": "tc_sweep_kernel (tcgen05.mma kind::i8, 128x256x32)",
                    "avg_launch_ms": kernel_ms,
                    "achieved": ops / (kernel_ms * 1e-3) / 1e12, "peak": mb / 1e12, "unit": "TOP/s (int8)",
                    "frac": ops / (kernel_ms * 1e-3) / mb,
                    "peak_source": "measured in this run: lorb_microbench_tensor_i8 = the kernel's own MMA stream "
                                   "(tcgen05.mma kind::i8 128x256x32) on zeroed operands, no TMA, no epilogue, whole GPU; "
                                   "MEASURED_PEAKS.json holds no int8 figure -- twice its bf16 numbers would be "
                                   "%.0f (sustained) / %.0f (burst), %s" % (2.0 * sustained, 2.0 * burst, tsrc),
                    "algorithmic_ops": "256 int8 multiply-adds (512 ops) per descriptor pair; executed: 288 per pair, "
                                       "the ninth k-step carries both tie-break index terms",
                    "frac_executed": ops * 288 / 256 / (kernel_ms * 1e-3) / mb,
                    "traffic": traffic, "traffic_source": traffic_src}
        else:
            alu_peak_pairs = 64.0 * sm_count * sm_max * 1e6 / 17.75
            peak_words = ctx.microbench_popc(1, 4096)
            traffic, traffic_src = _profile_traffic("sweep_kernel")
            roof = {"bound": "alu", "kernel": "sweep_kernel<4,true>", "avg_launch_ms": kernel_ms,
                    "achieved": pairs_per_launch * 8.0 / (kernel_ms * 1e-3) / 1e9, "peak": alu_peak_pairs * 8.0 / 1e9,
                    "unit": "G 32-bit words/s (1 descriptor pair = 8 words)",
                    "frac": pairs_per_launch / (kernel_ms * 1e-3) / alu_peak_pairs,
                    "peak_source": "hardware ALU issue ceiling: 64 lanes x %d SMs x %.0f MHz / 17.75 ALU "
                                   "thread-instructions per pair (SASS count, profiles/README.md)" % (sm_count, sm_max),
                    "loop_vs_register_body": pairs_per_launch * 8.0 / (kernel_ms * 1e-3) / peak_words,
                    "traffic": traffic, "traffic_source": traffic_src}
        popc_hw = 16.0 * sm_count * sm_max * 1e6  # SURVEY 8(d): 16 POPC / clk / SM
        alg_bytes = n_pairs * 2 * N_DESC * 32.0  # both descriptor blocks of every keyframe pair
        res = {
            "metric": "descriptor-pairs/s Hamming match", "value": value,
            "unit": "descriptor-pairs/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": "s8 (tcgen05.mma kind::i8 on +-32 expansions of the bit strings, s32 accumulate)" if tensor
                     else "u32 (xor/popc on 256-bit strings)",
            "data": "synthetic (uniform random 256-bit descriptors, seed 0)",
            "config": {"workload": "kf_pair_sweep: 4096 keyframes x 2000 descriptors resident "
                                   "(262 MB > 126 MB L2); step = all 8128 pairs of one 128-keyframe "
                                   "block, cross-check + max(2*minDist,30) filter",
                       "kernel": args.sweep_impl,
                       "keyframe_pairs_per_step_per_gpu": n_pairs,
                       "descriptor_pairs_per_step_per_gpu": n_pairs * PAIRS_PER_KF_PAIR,
                       "l2": "bank larger than L2; a different 8 MB block every step",
                       "sharding": "blocks round-robin over ranks, no collective"},
            "e2e": {"value": e2e_value, "unit": "descriptor-pairs/s",
                    "h2d_bytes_per_step": int(host_blk.nbytes + 2 * pa.nbytes),
                    "d2h_bytes_per_step": int(3 * 4 * n_pairs)},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roof,
            "roofline_popc_survey_8d": {
                "achieved": pairs_per_launch * 8.0 / (kernel_ms * 1e-3) / 1e9, "peak": popc_hw / 1e9,
                "unit": "G 32-bit words/s", "frac": pairs_per_launch * 8.0 / (kernel_ms * 1e-3) / popc_hw,
                "note": "SURVEY 8(d)'s definition (8 POPC per pair against 16 POPC/clk/SM at the max clock); "
                        "above 1 because neither kernel issues 8 POPC per pair (tensor: none; popc: 4, carry-save)"},
            "roofline_hbm": {"bound": "hbm", "achieved": alg_bytes / (kernel_ms * 1e-3) / 1e9,
                             "peak": hbm_peak, "unit": "GB/s",
                             "frac": alg_bytes / (kernel_ms * 1e-3) / 1e9 / hbm_peak,
                             "peak_source": peak_src,
                             "note": "algorithmic bytes = 2 x 64 KB descriptor blocks per keyframe "
                                     "pair; the kernel is not HBM-bound"},
        }
    ctx.close()
    return res, bank


def run_full_sweep(args, rank, world, local, bank):
    """BASELINE config 5's sweep in full, as SURVEY 8(e) row 1 specifies it: all 8 386 560 unordered
    keyframe pairs of the 4096-keyframe bank as an upper-triangular grid of 128 x 128-keyframe tiles
    dealt round-robin to the ranks (lorb_match_sweep_all), no collective during compute, then one
    gather (sum-reduce of the zero-initialised per-pair arrays, 33.5 MB) of the kept counts on rank 0;
    64 random off-diagonal keyframe pairs are checked against the oracle."""
    import torch
    import torch.distributed as dist
    from lorb_slam_b200 import capi
    ctx = capi.Context(local)
    ctx.sweep_set_impl(args.sweep_impl)
    ctx.bank_upload(bank)
    n_all = N_KF * (N_KF - 1) // 2
    pinned = torch.zeros(n_all, dtype=torch.int32).pin_memory()
    _barrier(world)
    l0 = ctx.launch_count
    t0 = time.perf_counter()
    kept, done = ctx.match_sweep_all(N_KF, BLOCK_KF, rank, world, out=pinned.numpy())
    ctx.sync()
    t_compute = _max_over_ranks(time.perf_counter() - t0, world, local)
    launches = ctx.launch_count - l0
    t1 = time.perf_counter()
    dev = pinned.cuda(non_blocking=True)
    if world > 1:
        dist.reduce(dev, 0, op=dist.ReduceOp.SUM)
    torch.cuda.synchronize()
    t_gather = _max_over_ranks(time.perf_counter() - t1, world, local)
    total_done = _sum_over_ranks(float(done), world, local)
    res = None
    if rank == 0:
        from oracle import ref
        allk = dev.cpu().numpy()
        OUTPUTS["full_sweep_kept"] = allk
        rng = np.random.default_rng(7)
        pa = rng.integers(0, N_KF, 64).astype(np.int32)
        pb = ((pa + rng.integers(BLOCK_KF, N_KF - BLOCK_KF, 64)) % N_KF).astype(np.int32)  # other blocks
        ref.set_num_threads(os.cpu_count() or 1)
        ok_kept = ref.sweep(bank, pa, pb)[0]
        got = np.array([allk[capi.sweep_pair_index(N_KF, int(a), int(b))] for a, b in zip(pa, pb)])
        wall = t_compute + t_gather
        res = {"metric": "descriptor-pairs/s Hamming match", "unit": "descriptor-pairs/s",
               "value": total_done * PAIRS_PER_KF_PAIR / wall, "n_gpus": world, "scaling": "strong",
               "keyframe_pairs": int(total_done), "descriptor_pairs": total_done * PAIRS_PER_KF_PAIR,
               "wall_s": wall, "compute_s": t_compute, "gather_s": t_gather,
               "gather_bytes": int(4 * n_all), "gpu_launches_rank0": int(launches),
               "config": {"workload": "whole keyframe-pair sweep: 4096 keyframes x 2000 descriptors, all %d unordered "
                                      "pairs = %d tiles of 128 x 128 keyframes, tile t on rank t %% %d, kept counts "
                                      "gathered on rank 0" % (n_all, N_KF // BLOCK_KF * (N_KF // BLOCK_KF + 1) // 2, world),
                          "kernel": args.sweep_impl},
               "kept_total": int(allk.sum(dtype=np.int64)),
               "parity": {"ok": bool(np.array_equal(got, ok_kept) and int(total_done) == n_all),
                          "checked": "64 random keyframe pairs from different blocks against the oracle "
                                     "(kept counts bit-exact); every pair processed exactly once: %s"
                                     % (int(total_done) == n_all)}}
    ctx.close()
    return res


# ------------------------------------------------------------------- BA extras
def _ba_opts_fixed_iters(mod, iters=10):
    """Exactly `iters` LM attempts: tolerances disabled (negative), as BASELINE's
    '10 LM iterations' asks."""
    return mod.ba_options(max_num_iterations=iters, function_tolerance=-1.0,
                          parameter_tolerance=-1.0, gradient_tolerance=-1.0,
                          max_consecutive_invalid_steps=1 << 30)


def extras(ctx, local):
    """Short versions of the other BASELINE configs (device-timed with CUDA
    events where a resident form exists, else wall clock through the C ABI)."""
    from lorb_slam_b200 import capi, synth
    out = {}
    rng = np.random.default_rng(0)
    # cfg 1: 1000 x 1000 brute force through the host-buffer call
    q, t = synth.descriptors_uniform(1000, rng), synth.descriptors_uniform(1000, rng)
    ctx.match_bf_crosscheck(q, t)
    t0 = time.perf_counter()
    reps = 200
    for _ in range(reps):
        ctx.match_bf_crosscheck(q, t)
    dt = (time.perf_counter() - t0) / reps
    out["bf_1000x1000_e2e"] = {"us_per_call": dt * 1e6, "descriptor_pairs_per_s": 1e6 / dt}
    # cfg 2: projection-guided search
    fr = synth.make_frame(2000, 0)
    pts = synth.make_proj_points(fr, 5000, 0)
    for th in (1.0, 15.0):
        r = ctx.search_proj_points(fr, pts, th)
        t0 = time.perf_counter()
        reps = 30
        for _ in range(reps):
            ctx.search_proj_points(fr, pts, th)
        dt = (time.perf_counter() - t0) / reps
        out["proj_5000pts_2000kp_th%g_e2e" % th] = {
            "us_per_call": dt * 1e6, "map_points_per_s": 5000 / dt,
            "candidate_pairs": r["n_candidates"], "candidate_pairs_per_s": r["n_candidates"] / dt}
    # next row: Frame::ComputeStereoMatches, 1000 features on a 640x480 stereo pair
    st = synth.make_stereo_pair(1000, 0)
    r = ctx.stereo_matches(st)
    t0 = time.perf_counter()
    reps = 30
    for _ in range(reps):
        ctx.stereo_matches(st)
    dt = (time.perf_counter() - t0) / reps
    out["stereo_matches_1000kp_640x480_e2e"] = {"us_per_call": dt * 1e6, "n_matched": r["n_matched"]}
    # cfg 0 / next row rank 5: ORBextractor::operator(), 1000 features on a 640x480 frame, then the
    # brute-force match of the frame pair (reference example/test.cpp)
    pat_path = os.path.join(ROOT, "tests", "golden", "orb_golden.npz")
    if os.path.exists(pat_path):
        pattern = np.load(pat_path)["orb/pattern"].astype(np.int32)
        img = synth.make_orb_image(0)
        img2 = synth.warp_orb_image(img)
        a = ctx.orb_extract(img, pattern)
        reps = 100
        t0 = time.perf_counter()
        for _ in range(reps):
            ctx.orb_extract(img, pattern)
        dt = (time.perf_counter() - t0) / reps
        b = ctx.orb_extract(img2, pattern)
        t0 = time.perf_counter()
        for _ in range(reps):
            m = ctx.match_bf_crosscheck(a["desc"], b["desc"])
        dtm = (time.perf_counter() - t0) / reps
        st0 = synth.make_stereo_pair(8, 0)
        sl, sr = st0["pyr_left"][0], st0["pyr_right"][0]
        sf = ctx.stereo_frame(sl, sr, pattern, float(st0["mbf"]), float(st0["mb"]))
        t0 = time.perf_counter()
        for _ in range(reps):
            ctx.stereo_frame(sl, sr, pattern, float(st0["mbf"]), float(st0["mb"]))
        dts = (time.perf_counter() - t0) / reps
        out["stereo_frame_2x640x480_e2e"] = {
            "us_per_frame_pair": dts * 1e6, "keypoints_left": int(sf[0]["n"]), "keypoints_right": int(sf[1]["n"]),
            "stereo_matches": int(sf[4])}
        out["orb_extract_1000f_640x480_e2e"] = {
            "us_per_frame": dt * 1e6, "frames_per_s": 1 / dt, "keypoints": int(a["n"]),
            "pair_match_us": dtm * 1e6, "pair_matches_kept": int(m["n_kept"])}
    # cfg 3: local BA, 10 LM iterations
    pb = synth.make_ba_problem(0, C=10, P=5000)
    opt = _ba_opts_fixed_iters(capi)
    prob = ctx.ba_problem(pb)
    prob.solve(opt)
    best = 1e9
    for _ in range(3):
        prob.reset()
        ctx.sync()
        t0 = time.perf_counter()
        s = prob.solve(opt)
        best = min(best, time.perf_counter() - t0)
    prob.close()
    ctx.ba_local(pb, opt)  # first call sizes the context's cached problem and staging
    e2e = 1e9
    for _ in range(3):
        t0 = time.perf_counter()
        ctx.ba_local(pb, opt)
        e2e = min(e2e, time.perf_counter() - t0)
    out["ba_local_10kf_5kpts_30kobs"] = {
        "ms_per_local_ba_resident": best * 1e3, "ms_per_local_ba_e2e": e2e * 1e3,
        "lm_iterations": s["iterations"],
        "obs_per_s_per_lm_iter": pb["O"] * s["iterations"] / best}
    return out



def _ba_rooflines(ctx, obs_per_launch, k_obs_per_point, n_reduced, prof, traffic_key):
    """roofline objects of one BA LM attempt from the library's own CUDA-event brackets
    (lorb_ctx_profile: slot 0 build pass, 1 back-substitution, 2 reduced-system solve).
    FLOP model of SURVEY 8(d): per observation 150 (linearise) + 216 (accumulate) + 216*k (Schur
    products, k observations per point) in the build pass, 60 in the back-substitution; the reduced
    solve is n^3/3 + 2 n^2.  Algorithmic bytes: 16 B per observation and pass (recompute-J design)."""
    hbm_peak, peak_src = _peaks()
    dfma = ctx.microbench_fp64(0, 4096)
    dmma = ctx.microbench_fp64(1, 4096)
    fp64_peak = max(dfma, dmma)
    build, backsub, solve = prof
    parts = {
        "build": (build, obs_per_launch * (150.0 + 216.0 + 216.0 * k_obs_per_point), obs_per_launch * 16.0),
        "backsub": (backsub, obs_per_launch * 60.0, obs_per_launch * 32.0),
        "reduced_solve": (solve, n_reduced ** 3 / 3.0 + 2.0 * n_reduced ** 2, n_reduced * n_reduced * 8.0),
    }
    name = max(parts, key=lambda k: parts[k][0][0])
    (ms_tot, n), flop, byt = parts[name]
    ms = ms_tot / max(1, n)
    shares = {k: v[0][0] for k, v in parts.items()}
    tot = sum(shares.values()) or 1.0
    traffic, traffic_src = _profile_traffic(traffic_key)
    roof = {"bound": "tensor", "bound_detail": "fp64: DMMA tensor-core contractions + DFMA Jacobians; latency-bound per ncu "
                                               "(profiles/README.md), HBM fraction below 1 %",
            "kernel": name, "avg_launch_ms": ms, "launches": int(n),
            "achieved": flop / (ms * 1e-3) / 1e12, "peak": fp64_peak / 1e12, "unit": "TFLOP/s",
            "frac": flop / (ms * 1e-3) / fp64_peak,
            "peak_source": "measured in this run: lorb_microbench_fp64 (DFMA %.1f, DMMA %.1f TFLOP/s), whole GPU"
                           % (dfma / 1e12, dmma / 1e12),
            "flop_model": "SURVEY 8(d): algorithmic flops of the kernel per launch",
            "share_of_attempt": {k: v / tot for k, v in shares.items()},
            "ms_per_attempt_by_part": {k: parts[k][0][0] / max(1, parts[k][0][1]) for k in parts},
            "traffic": traffic, "traffic_source": traffic_src}
    hbm = {"bound": "hbm", "kernel": name, "achieved": byt / (ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
           "frac": byt / (ms * 1e-3) / 1e9 / hbm_peak, "peak_source": peak_src,
           "note": "algorithmic bytes of the same kernel; BA on this design is not HBM-bound"}
    return roof, hbm


def _rel_err(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b) / (1e-8 + 1e-6 * np.abs(b)))) if a.size else 0.0


def cpu_baseline_ba_batched(pbs, iters=3):
    """The oracle port of BA::LocalPoseOptimization (oracle/ba_ref.cpp: Ceres' LM + DENSE_SCHUR restated,
    one thread per window as Ceres' num_threads=1) on a bounded sample: one window per host thread,
    `iters` LM iterations each, OpenMP over windows."""
    from lorb_slam_b200 import synth
    from oracle import ref
    cores = ref.set_num_threads(os.cpu_count() or 1)
    n = min(len(pbs), cores)
    bt = synth.batch_windows(pbs[:n])
    opt = _ba_opts_fixed_iters(ref, iters)
    t0 = time.perf_counter()
    _, _, sums = ref.ba_local_batched(bt["cam_off"], bt["cams"], bt["pt_off"], bt["pts"], bt["obs_off"],
                                      bt["obs_cam"], bt["obs_pt"], bt["obs_uv"], bt["K"], opt)
    dt = time.perf_counter() - t0
    it = sum(s["iterations"] for s in sums)
    return {"value": float(sum(p["O"] for p in pbs[:n])) * it / n / dt, "unit": "observations*iterations/s",
            "cores": cores, "kind": "port",
            "sample": "%d windows (10 keyframes / 5000 points / 30000 observations each), %d LM iterations each, "
                      "oracle/ba_ref.cpp -O2, OpenMP over windows (one thread per window)" % (n, iters)}


def cpu_baseline_ba_large(pb, iters=2):
    """The oracle port on the whole config-5 problem for `iters` LM iterations, one thread (Ceres'
    default num_threads=1; the reference sets no other)."""
    from oracle import ref
    opt = _ba_opts_fixed_iters(ref, iters)
    t0 = time.perf_counter()
    _, _, s = ref.ba_local(pb, opt)
    dt = time.perf_counter() - t0
    return {"value": pb["O"] * (s["iterations"] + 1) / dt, "unit": "observations*iterations/s", "cores": 1,
            "kind": "port",
            "sample": "%d LM iterations (+ the initial evaluation, counted as one) of the full problem "
                      "(%d keyframes / %d points / %d observations), oracle/ba_ref.cpp -O2, 1 thread"
                      % (s["iterations"], pb["C"], pb["P"], pb["O"])}


def run_ba_batched(args, rank, world, local, want_cpu=True):
    """BASELINE config 4: `--windows-total` (512) independent 10-keyframe windows split in contiguous
    slices over the ranks (strong scaling: the batch is fixed), every window its own LM loop."""
    import torch
    from lorb_slam_b200 import capi, sharding, synth
    _rank_host_threads(world)  # an earlier oracle leg may have taken every core for rank 0
    steps = args.steps
    warmup = max(3, min(args.warmup, 3))
    ctx = capi.Context(local)
    total = args.windows_total
    lo, hi = sharding.window_slice(rank, world, total)
    nw = hi - lo
    pbs = [synth.make_ba_problem(i, C=10, P=5000) for i in range(lo, hi)]
    bt = synth.batch_windows(pbs)
    opt = _ba_opts_fixed_iters(capi)
    obs = int(bt["obs_off"][-1])
    # ---- value: windows resident in HBM, only the solve is timed (reset + LM loop)
    prob = ctx.ba_problem_batched(bt)
    for _ in range(warmup):
        prob.reset()
        prob.solve(opt)
    st, ev0, ev1 = _events(ctx, local)
    _barrier(world)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = ctx.launch_count
    ctx.profile(True)
    ev0.record(st)
    for _ in range(steps):
        prob.reset()
        sums = prob.solve(opt)
    ev1.record(st)
    ctx.sync()
    dt = ev0.elapsed_time(ev1) * 1e-3
    launches = ctx.launch_count - l0
    prof = [ctx.profile_read(k) for k in range(3)]
    ctx.profile(False)
    clocks = sampler.stop() if rank == 0 else None
    dt_max = _max_over_ranks(dt, world, local)
    cams_res, pts_res = prob.download()
    if rank == 0:
        OUTPUTS.update(ba_batched_cams=cams_res, ba_batched_points=pts_res,
                       ba_batched_summaries=_ba_summary_rows(sums))
    # parity run: the same windows under Ceres' default tolerances (the timed runs force all 10
    # attempts, and attempts past convergence accept or reject on rounding noise, which makes their
    # end point a coin toss at the 1e-7 level -- not a fair thing to compare bit-for-tolerance)
    popt = capi.ba_options(max_num_iterations=10)
    prob.reset()
    psums = prob.solve(popt)
    pcams, ppts = prob.download()
    prob.close()
    iters = sum(s["iterations"] for s in sums) / len(sums)
    total_obs = _sum_over_ranks(float(obs), world, local)
    value = steps * total_obs * iters / dt_max
    # ---- e2e: the host-buffer call (upload of every window, solve, download) per step
    # (the call updates the caller's parameter arrays in place, as BA::LocalPoseOptimization's do;
    # restoring the initial values between steps is staging of the next step's input: untimed)
    io = dict(bt, cams=bt["cams"].copy(), pts=bt["pts"].copy())
    ctx.ba_local_batched(io, opt, inplace=True)
    _barrier(world)
    e2e_dt = 0.0
    for _ in range(steps):
        io["cams"][...] = bt["cams"]
        io["pts"][...] = bt["pts"]
        t0 = time.perf_counter()
        ctx.ba_local_batched(io, opt, inplace=True)
        e2e_dt += time.perf_counter() - t0
    e2e_dt = _max_over_ranks(e2e_dt, world, local)
    e2e_value = steps * total_obs * iters / e2e_dt
    # the host-buffer call against the resident solve, same default-tolerance options (the two sum their
    # partial results with atomics in no fixed order: compared by tolerance, not by bits)
    io["cams"][...] = bt["cams"]
    io["pts"][...] = bt["pts"]
    e_cams, e_pts, _ = ctx.ba_local_batched(io, popt, inplace=True)
    same = bool(max(_rel_err(e_cams, pcams), _rel_err(e_pts, ppts)) <= 1.0)
    res = None
    if rank == 0:
        from oracle import ref
        # parity inside the run: the first window of this rank against the oracle
        oc, op, so = ref.ba_local(pbs[0], ref.ba_options(max_num_iterations=10))
        pc, pp = pcams[:10], ppts[:pbs[0]["P"]]
        err = max(_rel_err(pc, oc), _rel_err(pp, op))
        sums = psums
        res = {"metric": "BA observations/s per LM iter", "value": value,
               "unit": "observations*iterations/s", "n_gpus": world, "steps": steps,
               "warmup": warmup, "ms_per_step": dt_max / steps * 1e3,
               "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
               "data": "synthetic (SURVEY 8(d) cfg 3 generator, window w = seed w)",
               "config": {"workload": "batched local BA (BASELINE config 4): %d independent windows split over "
                                      "%d rank(s) (%d on rank 0), each 10 keyframes / 5000 points / 30000 "
                                      "observations, 10 LM iterations (value: windows resident; e2e: "
                                      "lorb_ba_local_batched with host buffers)" % (total, world, nw),
                          "l2": "%.0f MB of observations and parameters on rank 0; parameters are "
                                "reset to the initial values before every step"
                                % ((bt["obs_uv"].nbytes + 2 * bt["obs_cam"].nbytes + bt["pts"].nbytes
                                    + bt["cams"].nbytes) / 1e6)},
               "e2e": {"value": e2e_value, "unit": "observations*iterations/s",
                       "h2d_bytes_per_step": int(bt["cams"].nbytes + bt["pts"].nbytes +
                                                 bt["obs_uv"].nbytes + 2 * bt["obs_cam"].nbytes),
                       "d2h_bytes_per_step": int(bt["cams"].nbytes + bt["pts"].nbytes)},
               "gpu_launches": int(launches), "clocks": clocks,
               "ms_per_local_ba": dt_max / steps / nw * 1e3, "lm_iterations": iters,
               "parity": {"ok": bool(err <= 1.0 and same), "max_err_over_tolerance": err,
                          "tolerance": "rtol 1e-6 + atol 1e-8 on final cameras and points",
                          "checked": "window %d (rank 0) against the oracle, Ceres' default tolerances, at most 10 "
                                     "LM iterations (the timed runs force all 10 attempts); host-buffer call == "
                                     "resident solve within the same tolerance: %s" % (lo, same),
                          "lm_iterations_ok_rejected_termination": {
                              "gpu": [sums[0]["iterations"], sums[0]["num_successful_steps"],
                                      sums[0]["num_unsuccessful_steps"], sums[0]["termination"]],
                              "oracle": [so["iterations"], so["num_successful_steps"],
                                         so["num_unsuccessful_steps"], so["termination"]]}}}
        res["roofline"], res["roofline_hbm"] = _ba_rooflines(ctx, obs, 6.0, 60, prof, "ba_build_dense_kernel")
        if world == 1 and want_cpu:
            res["cpu_baseline"] = cpu_baseline_ba_batched(pbs)
    ctx.close()
    return res


def run_ba_large(args, rank, world, local, want_cpu=True):
    """BASELINE config 5 BA: 200 keyframes / 200k points / 1.5M observations, points sharded over the
    ranks, reduced camera system all-reduced over NCCL every LM attempt.  Strong scaling."""
    import torch
    _rank_host_threads(world)  # an earlier oracle leg may have taken every core for rank 0
    import torch.distributed as dist
    from lorb_slam_b200 import capi, sharding, synth
    steps = args.steps
    warmup = max(3, min(args.warmup, 3))
    ctx = capi.Context(local)
    # the communicator exists at world 1 as well: the sharded code path (separate control kernel,
    # collectives) is then exercised and checked on a one-GPU box too
    uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
    if rank == 0:
        uid = torch.tensor(list(capi.Context.dist_unique_id()), dtype=torch.uint8, device="cuda")
    if world > 1:
        dist.broadcast(uid, 0)
    ctx.dist_init(bytes(uid.cpu().tolist()), rank, world)
    pb = synth.make_ba_problem(0, C=args.large_cams, P=args.large_points, obs_per_point=(7, 8),
                               traj_len=100.0 * args.large_cams / 200.0)
    sh = sharding.shard_ba_by_point(pb, rank, world)
    opt = _ba_opts_fixed_iters(capi)
    prob = ctx.ba_problem(sh)
    sharded = world > 1
    for _ in range(warmup):
        prob.reset()
        prob.solve(opt, sharded=sharded)
    st, ev0, ev1 = _events(ctx, local)
    _barrier(world)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = ctx.launch_count
    ctx.profile(True)
    ev0.record(st)
    for _ in range(steps):
        prob.reset()
        s = prob.solve(opt, sharded=sharded)
    ev1.record(st)
    ctx.sync()
    dt = ev0.elapsed_time(ev1) * 1e-3
    launches = ctx.launch_count - l0
    prof = [ctx.profile_read(k) for k in range(3)]
    coll_ms, coll_n = ctx.profile_read(4)  # the two all-reduces of every attempt, as seen by this rank
    ctx.profile(False)
    clocks = sampler.stop() if rank == 0 else None
    dt_max = _max_over_ranks(dt, world, local)
    cams_res, pts_res = prob.download()
    if rank == 0:
        OUTPUTS.update(ba_large_cams=cams_res, ba_large_points=pts_res, ba_large_summary=_ba_summary_rows([s]))
    # ---- parity inside the run: the un-sharded solve of the whole problem on rank 0 (at world 1: the
    # sharded code path over a one-rank communicator) must give the same cameras / points
    # Both sides run under Ceres' default tolerances (at most 10 iterations): the timed runs force all 10
    # attempts, and attempts past convergence accept or reject on rounding noise.
    popt = capi.ba_options(max_num_iterations=10)
    prob.reset()
    sp = prob.solve(popt, sharded=sharded)
    cams_res, pts_res = prob.download()
    parity = None
    if world == 1:
        prob.reset()
        s2 = prob.solve(popt, sharded=True)
        c2, p2 = prob.download()
        err = max(_rel_err(c2, cams_res), _rel_err(p2, pts_res))
        parity = {"ok": bool(err <= 1.0 and s2["iterations"] == sp["iterations"]), "max_err_over_tolerance": err,
                  "tolerance": "rtol 1e-6 + atol 1e-8 on final cameras and points",
                  "checked": "sharded code path (one-rank NCCL communicator) against the plain solve, default "
                             "tolerances, %d vs %d LM iterations, final cost %.9g vs %.9g"
                             % (s2["iterations"], sp["iterations"], s2["final_cost"], sp["final_cost"])}
    prob.close()
    if world > 1:
        camt = torch.from_numpy(cams_res).cuda()
        cam0 = camt.clone()
        dist.broadcast(cam0, 0)
        same_cams = torch.tensor([1.0 if torch.equal(camt, cam0) else 0.0], device="cuda")
        dist.all_reduce(same_cams, op=dist.ReduceOp.MIN)
        if rank == 0:
            full = ctx.ba_problem(pb)
            s1 = full.solve(popt)
            c1, p1 = full.download()
            full.close()
            err = max(_rel_err(cams_res, c1), _rel_err(pts_res, p1[sh["point_ids"]]))
            parity = {"ok": bool(err <= 1.0 and same_cams.item() == 1.0 and s1["iterations"] == sp["iterations"]),
                      "max_err_over_tolerance": err,
                      "tolerance": "rtol 1e-6 + atol 1e-8 on final cameras and rank 0's points",
                      "cameras_bit_identical_across_ranks": bool(same_cams.item() == 1.0),
                      "checked": "%d-rank sharded solve against the one-GPU solve of the whole problem on rank 0, "
                                 "default tolerances, %d vs %d LM iterations, final cost %.9g vs %.9g"
                                 % (world, sp["iterations"], s1["iterations"], sp["final_cost"], s1["final_cost"])}
    # ---- e2e: the host-buffer call every step (upload, device work lists, solve, download): lorb_ba_local
    # on one GPU, lorb_ba_local_shard (this rank's shard, collective) on several.
    _barrier(world)
    e2e_call = ctx.ba_local if world == 1 else ctx.ba_local_shard
    e2e_call(sh, opt)  # first call sizes the grow-only buffers of the ctx
    _barrier(world)
    t0 = time.perf_counter()
    for _ in range(steps):
        e2e_call(sh, opt)
    e2e = _max_over_ranks((time.perf_counter() - t0) / steps, world, local)
    O = pb["O"]
    value = steps * O * s["iterations"] / dt_max
    res = None
    if rank == 0:
        res = {"metric": "BA observations/s per LM iter", "value": value,
               "unit": "observations*iterations/s", "n_gpus": world, "steps": steps,
               "warmup": warmup, "ms_per_step": dt_max / steps * 1e3,
               "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
               "data": "synthetic (SURVEY 8(d) cfg 5 generator, seed 0)",
               "config": {"workload": "large BA (BASELINE config 5): %d keyframes / %d points / %d observations, 10 LM "
                                      "attempts, points sharded over %d rank(s) (by lowest observing camera, equal observation counts), NCCL all-reduce of the "
                                      "%dx%d reduced camera system per attempt"
                                      % (args.large_cams, args.large_points, O, world, 6 * args.large_cams,
                                         6 * args.large_cams),
                          "l2": "observations + points (%.0f MB) streamed per pass" % (O * 12 / 1e6)},
               "e2e": {"value": O * s["iterations"] / e2e, "unit": "observations*iterations/s",
                       "h2d_bytes_per_step": int(sh["obs_uv"].nbytes + 2 * sh["obs_cam"].nbytes +
                                                 sh["pts"].nbytes + sh["cams"].nbytes),
                       "d2h_bytes_per_step": int(sh["pts"].nbytes + sh["cams"].nbytes)},
               "gpu_launches": int(launches), "clocks": clocks,
               "ms_per_lm_iteration": dt_max / steps / s["iterations"] * 1e3,
               "lm_iterations": s["iterations"], "final_cost": s["final_cost"], "parity": parity}
        res["roofline"], res["roofline_hbm"] = _ba_rooflines(
            ctx, len(sh["obs_cam"]), 7.5, 6 * args.large_cams, prof, "ba_schur_pairs_kernel")
        attempts = max(1, prof[0][1])
        res["roofline"]["ms_per_attempt_by_part"]["collectives"] = coll_ms / attempts
        res["roofline"]["collectives_note"] = (
            "rank 0's CUDA-event brackets around the all-reduce of [packed S | H_cc | g_c | rhs | scalars | slots] "
            "(%.1f MB) after the build pass and of four scalars after the back-substitution, both per attempt; "
            "includes the wait for the slowest rank's build" % (6 * args.large_cams * (6 * args.large_cams + 7) * 4 / 1e6))
        if world == 1 and want_cpu:
            res["cpu_baseline"] = cpu_baseline_ba_large(pb)
    ctx.dist_finalize()
    ctx.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="lorb", choices=["lorb", "reference"])
    ap.add_argument("--workload", default="all", choices=["all", "sweep", "ba_batched", "ba_large"])
    ap.add_argument("--sweep-impl", default=os.environ.get("LORB_SWEEP_IMPL", "tensor"), choices=["tensor", "popc"])
    ap.add_argument("--windows-total", type=int, default=512)
    ap.add_argument("--large-cams", type=int, default=200)
    ap.add_argument("--large-points", type=int, default=200000)
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "lorb":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl lorb)")
    args.warmup = max(args.warmup, 3) if args.impl == "lorb" else args.warmup

    if args.impl == "reference":
        return reference_arm(args)

    rank, world, local = _dist_setup(args.gpus)
    want_cpu = not args.no_cpu_baseline
    # torchrun exports OMP_NUM_THREADS=1 to every rank: give each rank its share of the host cores
    # for the library's staging loops (the host-buffer calls of the e2e legs)
    _rank_host_threads(world)
    if args.workload == "ba_batched":
        res = run_ba_batched(args, rank, world, local, want_cpu=want_cpu)
    elif args.workload == "ba_large":
        res = run_ba_large(args, rank, world, local, want_cpu=want_cpu)
    else:
        res, bank = run_sweep(args, rank, world, local)
        if rank == 0:
            if not args.no_extras:
                from lorb_slam_b200 import capi
                ctx = capi.Context(local)
                try:
                    res["extra"] = extras(ctx, local)
                finally:
                    ctx.close()
            if world == 1 and want_cpu:
                res["cpu_baseline"] = cpu_baseline_sweep(bank)
        if args.workload == "all":
            f = run_full_sweep(args, rank, world, local, bank)
            if rank == 0:
                res["full_sweep"] = f
        del bank
        if args.workload == "all":
            # the other two BASELINE metrics, same contract
            b = run_ba_batched(args, rank, world, local, want_cpu=want_cpu)
            l = run_ba_large(args, rank, world, local, want_cpu=want_cpu)
            if rank == 0:
                res["ba_batched"] = b
                res["ba_large"] = l
    if rank == 0:
        if args.dump_outputs:
            write_outputs(args.dump_outputs)
        print(json.dumps(res), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


def _reference_sweep(args, cores):
    from oracle import ref
    bank = _make_bank(0)[:BLOCK_KF]
    pa, pb = _block_pairs()
    kind, desc, run = _cpu_sweepers(bank)[0]
    n = max(cores, 8) * (4 if kind == "reference" else 16)  # keyframe pairs per step (bounded sample)
    for _ in range(args.warmup):
        run(pa[:n], pb[:n])
    t0 = time.perf_counter()
    for s in range(args.steps):
        o = (s * n) % (len(pa) - n)
        run(pa[o:o + n], pb[o:o + n])
    dt = time.perf_counter() - t0
    value = args.steps * n * PAIRS_PER_KF_PAIR / dt
    sample = ("%d keyframe pairs (2000x2000 descriptors each) per step out of the 8128 of a block; %s"
              % (n, desc))
    return {"impl": "reference", "metric": "descriptor-pairs/s Hamming match", "value": value,
            "unit": "descriptor-pairs/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u64 popcnt", "data": "synthetic",
            "config": {"workload": "kf_pair_sweep (bounded sample): " + sample},
            "cpu_baseline": {"value": value, "unit": "descriptor-pairs/s", "cores": cores,
                             "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": "descriptor-pairs/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0}}


def _reference_ba(args, which):
    """CPU arm of a BA workload: the oracle port (oracle/_ref's Ceres stand-in is a dense
    normal-equations LM, 15 060 unknowns squared for one config-3 window: not runnable at these sizes)."""
    from lorb_slam_b200 import synth
    from oracle import ref
    cores = ref.set_num_threads(os.cpu_count() or 1)
    if which == "ba_batched":
        pbs = [synth.make_ba_problem(i, C=10, P=5000) for i in range(min(cores, args.windows_total))]
        t0 = time.perf_counter()
        cb = cpu_baseline_ba_batched(pbs, iters=3)
        metric_cfg = "batched local BA (bounded sample): " + cb["sample"]
    else:
        pb = synth.make_ba_problem(0, C=args.large_cams, P=args.large_points, obs_per_point=(7, 8),
                                   traj_len=100.0 * args.large_cams / 200.0)
        t0 = time.perf_counter()
        cb = cpu_baseline_ba_large(pb, iters=2)
        metric_cfg = "large BA (bounded sample): " + cb["sample"]
    dt = time.perf_counter() - t0
    return {"impl": "reference", "metric": "BA observations/s per LM iter", "value": cb["value"],
            "unit": "observations*iterations/s", "n_gpus": args.gpus, "steps": 1, "warmup": 0,
            "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": {"workload": metric_cfg}, "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": "observations*iterations/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0}}


def reference_arm(args):
    """The reference's own CPU path for the same metrics/configs, on the host cores of this box:
    the sweep through oracle/_ref (the reference's src/matcher.cpp compiled unmodified over the OpenCV
    stand-in; see oracle/ref_harness.cpp) when its library is present, else the oracle port; the two BA
    workloads through the oracle port -- the one other place bench.py may execute oracle/ -- each step
    a bounded sample of the workload.  Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import ref
    cores = os.cpu_count() or 1
    cores = ref.set_num_threads(cores)  # torchrun exports OMP_NUM_THREADS=1: use every host thread
    if args.workload in ("ba_batched", "ba_large"):
        out = _reference_ba(args, args.workload)
    else:
        out = _reference_sweep(args, cores)
        if args.workload == "all":
            out["ba_batched"] = _reference_ba(args, "ba_batched")
            out["ba_large"] = _reference_ba(args, "ba_large")
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
