"""Timing of full-ranking evaluation on row-sharded tables (not collected by pytest).  One process per GPU:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29667 \
        tests/full_ranking_sharded_perf.py [--reps 3] [--out FILE]

cfg2 sizes: 1M test users (every user of the table; user u on rank u % N), 200k recipes (recipe i on rank i % N),
D = 128 fp32, training histories of Zipf(1.05) recipes with geometric lengths of mean 20, one held-out recipe per user
(uniform over the catalog), K = 10 and 100.  Reported by rank 0, one JSON line per K:
  * ms per call of DistRunner.full_ranking with the default round size and with all users in one round (CUDA events
    on rank 0's stream after a barrier, one warm-up call first; the call reads each round's list size on the host, so
    the window holds that too).  All 1M test users are ranked per call: this is ms per 1M test users;
  * the exact-fallback rows (catalog_fallback_rows after the one-round call, summed over the ranks);
  * at N = 1: LocalRunner.full_ranking on the same engine and Engine.catalog_topk(users, K, exclude=...) on the same
    tables with the same lists, and whether all of them give the same positions;
  * the card, its power limit and max SM clock, read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

U, I, D = 1_000_000, 200_000, 128


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def timed(fn, reps):
    fn()                                               # warm-up: module load, workspaces, catalog index
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
    P = torch.randn((sharded.local_rows(U, W), 5, D), generator=g, device=dev) * 0.1
    R = torch.randn((sharded.local_rows(I, W), D), generator=g, device=dev) * 0.1
    g0 = torch.Generator(device=dev); g0.manual_seed(7)
    Cat = torch.randn((4, D), generator=g0, device=dev) * 0.1
    ic = synth.make_item_categories(I, seed=8)
    eng = sharded.ShardedEngine(Hyper(learner="sgd"), P, R, Cat, torch.zeros((9, 5, D), device=dev), rank, W, device=dev,
                                max_rows=256, item_cats_global=ic, adopt=True, num_users_global=U)
    del P, R
    rng = np.random.default_rng(5)                     # the same global draw on every rank
    lens = rng.geometric(1 / 20, U)
    off = np.zeros(U + 1, np.int64); off[1:] = np.cumsum(lens)
    ids = synth.zipf_items(rng, I, int(off[-1]))
    held = rng.integers(0, I, U)
    # resident device CSR of this rank's users: the timed window holds the evaluation, not the host -> device copy
    hist = tuple(torch.as_tensor(x).to(dev) for x in sharded.shard_label_csr(off, ids, rank, W, U))
    n = len(range(rank, U, W))
    users = torch.arange(n, dtype=torch.int32, device=dev)
    h = torch.as_tensor(held[rank::W]).to(dev)
    run = sharded.DistRunner(eng)
    for K in (10, 100):
        res = {"world": W, "test_users": U, "recipes": I, "D": D, "K": K, "history_entries": int(off[-1]),
               "round_users": sharded.FULL_RANKING_ROUND_USERS}
        ms, pos = timed(lambda: run.full_ranking(users, h, K, history=hist), args.reps)
        ms1, pos1 = timed(lambda: run.full_ranking(users, h, K, history=hist, round_users=n), args.reps)
        fb = torch.tensor([eng.e.catalog_fallback_rows()], dtype=torch.int64, device=dev)
        dist.all_reduce(fb)
        res.update(sharded_ms=ms, sharded_ms_min=min(ms), one_round_ms=ms1, one_round_ms_min=min(ms1),
                   fallback_rows=int(fb), hits=int((pos >= 0).sum()), rounds_identical=bool(torch.equal(pos, pos1)))
        if W == 1:                                     # LocalRunner and the unsharded entry on the same tables, same run
            lr = sharded.LocalRunner([eng])
            msl, posl = timed(lambda: lr.full_ranking([users], [h], K, history=[hist])[0], args.reps)
            _, excl = sharded._round_lists(users.long(), h, hist, 0, n, n)        # the same lists, built once
            mse, (eids, _) = timed(lambda: eng.e.catalog_topk(users=users, K=K, exclude=excl), args.reps)
            res.update(local_runner_ms=msl, local_runner_ms_min=min(msl), engine_ms=mse, engine_ms_min=min(mse),
                       engine_fallback_rows=eng.e.catalog_fallback_rows(),
                       identical_to_engine=bool(torch.equal(posl, pos) and torch.equal(sharded._positions(eids, h), pos)))
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
