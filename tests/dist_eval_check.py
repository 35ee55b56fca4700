"""Multi-process check of sampled evaluation on row-sharded tables over NCCL: launched by
tests/test_gpu_sharded_eval.py::test_nccl_sharded_eval_equals_unsharded (needs >= 2 GPUs) or by hand:

  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
      --master-port 29643 tests/dist_eval_check.py

Every rank trains its shard a few steps through DistRunner, then evaluates its test users through
DistRunner.eval_sampled_topk (several rounds).  The tables are then gathered and every rank compares its ids, gt_rank
and scores, bit for bit, with an unsharded engine over those tables; evaluate_sharded must give evaluate_model's
hits and NDCGs on every rank."""
import math
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from foodrec_b200 import Engine, Hyper, evaluate_sharded, sharded    # noqa: E402
from foodrec_b200.evaluate import build_candidates                   # noqa: E402
from tests.util import Problem                                        # noqa: E402


def main():
    rank, W = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    dev = torch.device("cuda", torch.cuda.current_device())
    dist.init_process_group("nccl", device_id=dev)
    p = Problem(1003, 2001, 9, 128, seed=72)
    h = Hyper(learner="adam", lr=0.01)
    rows, cols = np.nonzero(p.user_labels)
    off = np.zeros(p.U + 1, np.int32); off[1:] = np.cumsum(np.bincount(rows, minlength=p.U))
    eng = sharded.ShardedEngine(h, sharded.shard_rows(p.tb.P, rank, W), sharded.shard_rows(p.tb.R, rank, W),
                                p.tb.Cat, p.tb.G, rank, W, device=dev, max_rows=4096, adam_mode="lazy",
                                item_cats_global=p.item_cats,
                                user_label_csr_local=sharded.shard_label_csr(off, cols.astype(np.int32), rank, W, p.U),
                                max_label_entries=4096 * p.L)
    run = sharded.DistRunner(eng)
    for s in range(3):
        f = p.bpr(1500, seed=95 + s)
        ix = sharded.route_batch(f["user_input"], W)[rank]
        eng.set_batch(f["user_input"][ix] // W, f["item_input"][ix], neg_items=f["neg_item_input"][ix], global_batch=1500)
        assert run.step().cpu().numpy()[9] == 0
    # this rank's test users (rank 1 has none: it only serves), 51 candidates with repeats and ids outside the catalog
    rng = np.random.default_rng(7)
    nl = len(range(rank, p.U, W))
    n = 700 if rank == 0 else 0
    u = rng.integers(0, nl, n).astype(np.int32)
    cand = rng.integers(0, p.I, (n, 51)).astype(np.int32)
    cand[:n // 20, 4] = p.I + 5
    cand[:n // 10, 9] = cand[:n // 10, 0]
    nc = np.full(n, 51, np.int32); nc[:n // 7] = rng.integers(0, 52, n // 7)
    dv = lambda x: torch.as_tensor(x, device=dev)
    ids, rk, sc = run.eval_sampled_topk(dv(u), dv(cand), nc, 10, return_scores=True, round_users=256)
    eng.e.flush()
    Ps = [torch.empty_like(eng.e.P) for _ in range(W)]; Rs = [torch.empty_like(eng.e.R) for _ in range(W)]
    dist.all_gather(Ps, eng.e.P.contiguous()); dist.all_gather(Rs, eng.e.R.contiguous())
    P = sharded.unshard_rows([x.cpu().numpy() for x in Ps], p.U)
    R = sharded.unshard_rows([x.cpu().numpy() for x in Rs], p.I)
    single = Engine(Hyper(learner="sgd"), P, R, eng.e.Cat.cpu().numpy(), eng.e.G.cpu().numpy(), device=dev, max_rows=256,
                    item_cats=p.item_cats)
    ids1, rk1, sc1 = single.eval_sampled_topk(dv(u.astype(np.int64) * W + rank).int(), dv(cand), nc, 10, return_scores=True)
    assert torch.equal(ids, ids1) and torch.equal(rk, rk1) and torch.equal(sc, sc1)
    # evaluate_sharded against evaluate_model's arithmetic on the same tables (the same test set on every rank)
    rng = np.random.default_rng(11)
    testR = {str(x): [int(rng.integers(0, p.I))] for x in range(0, p.U, 3)}
    testN = {k: [int(v) for v in rng.integers(0, p.I, 100)] for k in testR}
    d2c = {str(i): [[float(m)] for m in p.item_cats[i]] for i in range(p.I)}
    hits, ndcgs = evaluate_sharded(run, testR, testN, 10, d2c)
    users, c, ncs, cc = build_candidates(testR, testN, d2c)
    _, r1 = single.eval_sampled_topk(users, c, ncs, 10, cand_cats=cc)
    r1 = r1.cpu().numpy()
    assert hits == [1 if r >= 0 else 0 for r in r1]
    assert ndcgs == [math.log(2) / math.log(int(r) + 2) if r >= 0 else 0 for r in r1]
    sys.stdout.write(f"DIST_EVAL_CHECK_OK_{rank}\n"); sys.stdout.flush()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
