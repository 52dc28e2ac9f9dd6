"""Launched by torchrun (one rank per GPU): the point-sharded large BA under the Huber loss against
the oracle.  Every rank sets the same loss on its ctx.  Prints SHARDED_BA_ROBUST_OK on rank 0."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import robust_cases as rc  # noqa: E402
import robust_ref as rr  # noqa: E402
from lorb_slam_b200 import capi  # noqa: E402


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = capi.Context(local)
    uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
    if rank == 0:
        uid = torch.tensor(list(capi.Context.dist_unique_id()), dtype=torch.uint8, device="cuda")
    dist.broadcast(uid, 0)
    ctx.dist_init(bytes(uid.cpu().tolist()), rank, world)
    ctx.ba_set_loss(capi.LOSS_HUBER, rc.SCALE)

    pb = rc.local(41, C=24, P=3000, obs_per_point=(5, 6, 7), traj_len=8.0, fixed_frac=0.05)
    opt = capi.ba_options(max_num_iterations=8)
    prob = ctx.ba_problem_sharded(pb, rank, world)
    s = prob.solve(opt, sharded=True)
    cams, pts = prob.download()
    ids = prob.point_ids
    prob.close()
    mx = len(pb["pts"])
    buf = torch.zeros((mx, 3), dtype=torch.float64, device="cuda")
    idx = torch.full((mx,), -1, dtype=torch.int64, device="cuda")
    buf[:len(pts)] = torch.from_numpy(pts).cuda()
    idx[:len(ids)] = torch.from_numpy(np.asarray(ids, np.int64)).cuda()
    allb = [torch.zeros_like(buf) for _ in range(world)]
    alli = [torch.zeros_like(idx) for _ in range(world)]
    dist.all_gather(allb, buf)
    dist.all_gather(alli, idx)
    camt = torch.from_numpy(cams).cuda()
    cam0 = camt.clone()
    dist.broadcast(cam0, 0)
    assert torch.equal(camt, cam0), "replicated cameras diverged between ranks"
    if rank == 0:
        full = np.full((mx, 3), np.nan)
        for b_, i_ in zip(allb, alli):
            i_ = i_.cpu().numpy()
            k = i_ >= 0
            full[i_[k]] = b_.cpu().numpy()[k]
        assert not np.isnan(full).any()
        from oracle import ref
        oc, op, so = rr.ba_local(pb, ref.ba_options(max_num_iterations=8), loss=(rr.LOSS_HUBER, rc.SCALE))
        np.testing.assert_allclose(cams, oc, rtol=1e-6, atol=1e-8)
        np.testing.assert_allclose(full, op, rtol=1e-6, atol=1e-8)
        assert s["iterations"] == so["iterations"] and s["termination"] == so["termination"], (s, so)
        np.testing.assert_allclose(s["final_cost"], so["final_cost"], rtol=1e-8)
        print("huber sharded ok", s)
    dist.barrier()
    ctx.dist_finalize()
    ctx.close()
    if rank == 0:
        print("SHARDED_BA_ROBUST_OK")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
