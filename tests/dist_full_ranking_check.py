"""Multi-process check of full-ranking evaluation on row-sharded tables over NCCL: launched by
tests/test_gpu_full_ranking_sharded.py::test_nccl_full_ranking_equals_unsharded (needs >= 2 GPUs) or by hand:

  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
      --master-port 29665 tests/dist_full_ranking_check.py

Every rank trains its shard a few steps through DistRunner, then ranks its test users (rank 1 has few) through
DistRunner.full_ranking in several rounds, with the history set on the engine.  The tables are then gathered and every
rank compares its positions with an unsharded engine's catalog top-K over those tables (same exclusion lists);
evaluate_full_catalog_sharded must give evaluate_full_catalog's hits and NDCGs on every rank."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from foodrec_b200 import Hyper, Model, evaluate_full_catalog, evaluate_full_catalog_sharded, sharded   # noqa: E402
from oracle import synth                                                                               # noqa: E402
from tests.util import Problem, args_ns                                                                # noqa: E402


def main():
    rank, W = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    dev = torch.device("cuda", torch.cuda.current_device())
    dist.init_process_group("nccl", device_id=dev)
    p = Problem(1003, 2001, 9, 128, seed=73)
    p.item_cats[np.random.default_rng(1).choice(p.I, 30, replace=False)] = 0
    args = args_ns(p, learner="adam", lr=0.01)
    rows, cols = np.nonzero(p.user_labels)
    off = np.zeros(p.U + 1, np.int32); off[1:] = np.cumsum(np.bincount(rows, minlength=p.U))
    eng = sharded.ShardedEngine(Hyper.from_args(args), sharded.shard_rows(p.tb.P, rank, W), sharded.shard_rows(p.tb.R, rank, W),
                                p.tb.Cat, p.tb.G, rank, W, device=dev, max_rows=4096, adam_mode="lazy",
                                item_cats_global=p.item_cats, num_users_global=p.U,
                                user_label_csr_local=sharded.shard_label_csr(off, cols.astype(np.int32), rank, W, p.U),
                                max_label_entries=4096 * p.L)
    run = sharded.DistRunner(eng)
    live = p.item_cats.sum(1) > 0
    for s in range(3):
        f = p.bpr(1500, seed=95 + s)
        keep = live[f["item_input"]] & live[f["neg_item_input"]]      # a recipe without a category has no score
        u, it, neg = f["user_input"][keep], f["item_input"][keep], f["neg_item_input"][keep]
        ix = sharded.route_batch(u, W)[rank]
        eng.set_batch(u[ix] // W, it[ix], neg_items=neg[ix], global_batch=int(keep.sum()))
        assert run.step().cpu().numpy()[9] == 0
    rng = np.random.default_rng(5)                      # the same data on every rank
    train = {str(u): [int(x) for x in synth.zipf_items(rng, p.I, int(rng.geometric(1 / 20)))] for u in range(p.U) if u % 9}
    train["2"] = [int(x) for x in rng.permutation(p.I)[:1800]]          # every shard takes the exact fallback
    users = np.asarray([u for u in range(p.U) if u % W == 0 or u % 7 == 0], np.int64)
    held = rng.integers(0, p.I + 2, users.size)
    eng.e.flush()
    Ps = [torch.empty_like(eng.e.P) for _ in range(W)]; Rs = [torch.empty_like(eng.e.R) for _ in range(W)]
    dist.all_gather(Ps, eng.e.P.contiguous()); dist.all_gather(Rs, eng.e.R.contiguous())
    P = sharded.unshard_rows([x.cpu().numpy() for x in Ps], p.U)
    R = sharded.unshard_rows([x.cpu().numpy() for x in Rs], p.I)
    assert np.isfinite(P).all() and np.isfinite(R).all()
    m = Model(args, P, R, eng.e.Cat.cpu().numpy(), eng.e.G.cpu().numpy(), device=dev)
    m.engine.set_item_cats(p.item_cats)
    best, _ = m.engine.catalog_topk(users=users.astype(np.int32), K=30)
    pick = rng.random(users.size) < 0.6
    held[pick] = best.cpu().numpy()[pick, rng.integers(0, 30, int(pick.sum()))]
    test = {str(u): [int(h)] for u, h in zip(users, held)}
    d2c = {str(i): [[float(x)] for x in p.item_cats[i]] for i in range(p.I)}
    eng.set_user_history(train)
    for K in (10, 100):
        # positions of this rank's users through DistRunner.full_ranking, the history set on the engine
        mine = users % W == rank
        pos = run.full_ranking(torch.as_tensor(users[mine] // W, device=dev), held[mine], K, round_users=64)
        excl = [[i for i in train.get(str(u), []) if i != h] for u, h in zip(users[mine], held[mine])]
        ids, _ = m.engine.catalog_topk(users=users[mine].astype(np.int32), K=K, exclude=excl)
        hit = ids.cpu().numpy() == held[mine][:, None]
        want = np.where(hit.any(1), hit.argmax(1), -1)
        assert np.array_equal(pos.cpu().numpy(), want), K
        hits, ndcgs = evaluate_full_catalog_sharded(run, train, test, K, round_users=100)
        assert (hits, ndcgs) == evaluate_full_catalog(None, m, train, test, K, d2c), K
        assert 0 < sum(hits) < len(hits)
    sys.stdout.write(f"DIST_FULL_RANKING_CHECK_OK_{rank}\n"); sys.stdout.flush()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
