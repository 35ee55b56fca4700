"""Timing of sampled evaluation on row-sharded tables (not collected by pytest).  One process per GPU:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29651 \
        tests/sharded_eval_perf.py [--reps 3] [--out FILE]

cfg2 sizes: 200k recipes over the N ranks (recipe i on rank i % N), D = 128 fp32, and one shard of 1M test users per
GPU (N million users in all), 51 candidates each (the held-out item + 50 negatives, uniform over the catalog).
Reported by rank 0, in one JSON line:
  * ms per call of DistRunner.eval_sampled_topk (K = 10; CUDA events, one warm-up call; every rank evaluates its own
    1M users, so this is also ms per 1M test users per GPU);
  * at N = 1, Engine.eval_sampled_topk on the same tables in the same run (and a check that both rank identically);
  * bytes moved per test user: the distinct requested rows of other ranks (payload) and the fixed-capacity blocks the
    staged all-to-alls carry (requests + rows, own block excluded);
  * the card and its power limit, read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

U_LOCAL, I, D, STRIDE, K = 1_000_000, 200_000, 128, 51, 10


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def timed(fn, reps):
    fn()                                               # warm-up: module load, workspaces
    torch.cuda.synchronize(); dist.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = []
    for _ in range(reps):
        dist.barrier()
        a.record(); out = fn(); b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return ms, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from foodrec_b200 import Hyper, sharded
    from oracle import synth
    rank, W = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    dev = torch.device("cuda", torch.cuda.current_device())
    dist.init_process_group("nccl", device_id=dev)
    g = torch.Generator(device=dev); g.manual_seed(100 + rank)
    ipr = (I + W - 1) // W
    P = torch.randn((U_LOCAL, 5, D), generator=g, device=dev) * 0.1
    R = torch.randn((ipr, D), generator=g, device=dev) * 0.1
    g0 = torch.Generator(device=dev); g0.manual_seed(7)
    Cat = torch.randn((4, D), generator=g0, device=dev) * 0.1
    ic = synth.make_item_categories(I, seed=8)
    eng = sharded.ShardedEngine(Hyper(learner="sgd"), P, R, Cat, torch.zeros((9, 5, D), device=dev), rank, W, device=dev,
                                max_rows=256, item_cats_global=ic, adopt=True)
    del P, R
    run = sharded.DistRunner(eng)
    users = torch.arange(U_LOCAL, dtype=torch.int32, device=dev)
    cand = torch.randint(0, I, (U_LOCAL, STRIDE), generator=g, device=dev, dtype=torch.int32)
    nc = torch.full((U_LOCAL,), STRIDE, dtype=torch.int32, device=dev)
    ms, (ids, rk) = timed(lambda: run.eval_sampled_topk(users, cand, nc, K), args.reps)
    res = {"world": W, "users_per_gpu": U_LOCAL, "recipes": I, "D": D, "stride": STRIDE, "K": K,
           "round_users": sharded.EVAL_ROUND_USERS, "sharded_ms": ms, "sharded_ms_min": min(ms)}
    # bytes per test user: distinct rows of OTHER owners per round (payload) and the staged blocks (own block excluded)
    rn = min(sharded.EVAL_ROUND_USERS, U_LOCAL)
    cap = eng.eval_cap(rn, STRIDE)
    rounds = (U_LOCAL + rn - 1) // rn
    payload = 0
    for a in range(0, U_LOCAL, rn):
        u = torch.unique(cand[a:a + rn].reshape(-1))
        payload += int((u % W != rank).sum())
    row_bytes = D * 4
    res["payload_bytes_per_user"] = payload * (row_bytes + 4) / U_LOCAL
    res["staged_bytes_per_user"] = rounds * (W - 1) * cap * (row_bytes + 4) / U_LOCAL
    res["cap"] = cap
    if W == 1:                                         # the unsharded engine on the same tables, same run
        ms1, (ids1, rk1) = timed(lambda: eng.e.eval_sampled_topk(users, cand, nc, K), args.reps)
        res["engine_ms"] = ms1; res["engine_ms_min"] = min(ms1)
        res["identical_to_engine"] = bool(torch.equal(ids, ids1) and torch.equal(rk, rk1))
    res["gpu"] = gpu_info()
    if rank == 0:
        line = json.dumps(res)
        print(line, flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "a") as f:
                f.write(line + "\n")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
