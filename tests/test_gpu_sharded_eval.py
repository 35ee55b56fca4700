"""Sampled evaluation (evaluate.py's protocol) on row-sharded tables, against the unsharded engine on the same global
tables.  The user owner ranks with the same kernel on the same fp32 values -- the recipe rows it received, addressed
by slot -- so ids, gt_rank and scores must be bit-identical, for every (user, candidate) case the kernel treats apart."""
import json
import os

import numpy as np
import pytest
import torch

from foodrec_b200 import sharded
from tests import sharded_eval_oracle as so
from tests.util import Problem, assert_close

pytestmark = pytest.mark.gpu

ALPHA = 0.35
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def dev32(x):
    return torch.as_tensor(np.ascontiguousarray(x, np.int32), device="cuda")


def label_csr(p):
    rows, cols = np.nonzero(p.user_labels)
    off = np.zeros(p.U + 1, np.int32); off[1:] = np.cumsum(np.bincount(rows, minlength=p.U))
    return off, cols.astype(np.int32)


def setup(p, W, learner="adagrad", bf16=False, health=False, G=None, **kw):
    from foodrec_b200 import Engine, Hyper
    h = Hyper(learner=learner, alpha=ALPHA, lr=0.01)
    G = p.tb.G if G is None else G
    td = "bf16" if bf16 else "float32"
    off, idx = label_csr(p)
    single = Engine(h, p.tb.P, p.tb.R, p.tb.Cat, G, max_rows=4096, item_cats=p.item_cats, user_label_csr=(off, idx),
                    max_label_entries=4096 * p.L, table_dtype=td, **kw)
    engs = [sharded.ShardedEngine(h, sharded.shard_rows(p.tb.P, r, W), sharded.shard_rows(p.tb.R, r, W), p.tb.Cat, G, r, W,
                                  max_rows=4096, item_cats_global=p.item_cats,
                                  user_label_csr_local=sharded.shard_label_csr(off, idx, r, W, p.U),
                                  max_label_entries=4096 * p.L, table_dtype=td, num_users_global=p.U, **kw)
            for r in range(W)]
    if health:
        single.set_health_blend(True)
        for g in engs:
            g.e.set_health_blend(True)
    return single, engs


def feed(rng, p, W, n_per_rank, stride, empty_rank=1):
    """Per rank: local users (a few outside Personal_Memory: the first row past the shard's users -- the padding row of
    the last user shard where there is one --, further past the shard's rows, or negative), candidates with
    ragged n_cand (0, 1 and the full stride among them), repeats within and across users, ids outside the catalog and
    in the padding of the last recipe shard.  ``empty_rank`` gets no test users."""
    I = p.I
    ipr = -(-I // W)
    pad = np.arange(I, W * ipr)
    out = []
    for r in range(W):
        n = 0 if r == empty_rank else n_per_rank
        nl = len(range(r, p.U, W))
        u = rng.integers(0, nl, n)
        bad = rng.random(n) < 0.03
        u[bad] = np.where(rng.random(int(bad.sum())) < 0.5, nl + rng.integers(0, 50, int(bad.sum())), -1)
        if n:
            u[4] = nl
        cand = rng.integers(0, I, (n, stride))
        m = rng.random((n, stride)) < 0.02
        cand[m] = np.where(rng.random(int(m.sum())) < 0.5, I + rng.integers(0, 1000, int(m.sum())), -1 - rng.integers(0, 9, int(m.sum())))
        if pad.size:
            m = rng.random((n, stride)) < 0.02
            cand[m] = rng.choice(pad, int(m.sum()))
        rep = rng.random(n) < 0.1
        cand[rep, 3] = cand[rep, 0]                                # the held-out item repeated
        cand[rep, stride - 1] = cand[rep, 5]
        cand[:n // 10, 7] = 13                                     # one recipe in many users' lists
        nc = np.full(n, stride, np.int32)
        if n:
            rag = rng.random(n) < 0.2
            nc[rag] = rng.integers(0, stride + 1, int(rag.sum()))
            nc[:3] = [0, 1, stride - 1]
        out.append((u.astype(np.int32), cand.astype(np.int32), nc))
    return out


def compare(single, engs, p, parts, K, cand_cats, round_users=None):
    W = len(engs)
    run = sharded.LocalRunner(engs)
    ccs = None
    if cand_cats:
        ccs = [p.item_cats[np.clip(c, 0, p.I - 1)].reshape(c.shape + (4,)) for _, c, _ in parts]
    kw = {} if round_users is None else {"round_users": round_users}
    outs = run.eval_sampled_topk([dev32(u) for u, _, _ in parts], [dev32(c) for _, c, _ in parts], [nc for _, _, nc in parts],
                                 K, cand_cats=ccs, return_scores=True, **kw)
    checked = 0
    for r, ((u, c, nc), (ids, rank, sc)) in enumerate(zip(parts, outs)):
        nl = len(range(r, p.U, W))
        gu = np.where((u >= 0) & (u < nl), u.astype(np.int64) * W + r, -1)
        ids1, rank1, sc1 = single.eval_sampled_topk(dev32(gu), dev32(c), nc, K, cand_cats=None if ccs is None else ccs[r],
                                                    return_scores=True)
        assert torch.equal(ids, ids1), f"rank {r}: ids"
        assert torch.equal(rank, rank1), f"rank {r}: gt_rank"
        assert torch.equal(sc.view(torch.int32), sc1.view(torch.int32)), f"rank {r}: scores"
        checked += len(u)
    assert checked > 0
    return outs


# D x stride x table format x health blend x K x W, with cand_cats given or taken from the global map
GRID = [
    (64, 51, False, False, 10, 2, True), (64, 100, True, True, 1, 3, False), (64, 51, True, False, 10, 8, False),
    (128, 51, False, True, 10, 3, False), (128, 100, False, False, 1, 8, True), (128, 51, True, True, 10, 2, True),
    (200, 51, False, False, 1, 8, False), (200, 100, True, False, 10, 2, False), (200, 51, False, True, 10, 3, True),
    (200, 100, False, True, 10, 8, False), (128, 100, True, False, 10, 3, True), (64, 100, False, True, 1, 2, False),
]


@pytest.mark.parametrize("D,stride,bf16,health,K,W,given", GRID)
def test_sharded_eval_equals_unsharded(D, stride, bf16, health, K, W, given):
    p = Problem(401, 1001, 7, D, seed=D + stride + W)          # 1001 recipes: padded last shard at W = 2, 3, 8
    G = (p.tb.G * 5).astype(np.float32)
    single, engs = setup(p, W, bf16=bf16, health=health, G=G)
    rng = np.random.default_rng(D * 7 + W)
    parts = feed(rng, p, W, 300, stride)
    compare(single, engs, p, parts, K, given)
    compare(single, engs, p, parts, K, given, round_users=64)       # several rounds, the empty rank in all of them


@pytest.mark.parametrize("W", [2, 3])
def test_device_plan_and_serve_equal_the_restatement(W):
    p = Problem(64, 1001, 5, 64, seed=9)
    _, engs = setup(p, W, bf16=True)
    rng = np.random.default_rng(W)
    u, cand, nc = feed(rng, p, W, 200, 51, empty_rank=-1)[0]
    g = engs[0]
    cap = g.eval_cap(200, 51)
    flag = torch.zeros(1, device="cuda")
    req = g.eval_plan(dev32(cand), nc, cap, flag=flag)
    ev = g._ev
    req0, slots0, ids0, over = so.eval_plan(cand, nc, W, p.I, cap)
    assert not over and float(flag) == 0
    np.testing.assert_array_equal(req.cpu().numpy(), req0)
    np.testing.assert_array_equal(ev["slots"].cpu().numpy(), slots0)
    np.testing.assert_array_equal(ev["slot_ids"].cpu().numpy(), ids0)
    valid = slots0 >= 0
    np.testing.assert_array_equal(ev["cats"].cpu().numpy()[valid], p.item_cats[cand[valid]])
    # serve: bf16 rows copied as stored (not widened), a zero row for an empty request
    rq = np.concatenate([req0[:cap], [-1, 0]])
    rows = g.eval_serve(dev32(rq))
    assert rows.dtype == torch.bfloat16
    want = g.e.R[torch.as_tensor(np.maximum(rq, 0), device="cuda").long()].clone()
    want[torch.as_tensor(rq < 0, device="cuda")] = 0
    assert torch.equal(rows.view(torch.int16), want.view(torch.int16))


@pytest.mark.parametrize("W", [2, 3])
def test_sharded_eval_after_training_serves_caught_up_rows(W):
    """Lazy Adam (fp32, single-pass step on): a few steps through the runner leave rows behind the step counter and
    Personal_Memory rows in the shadow.  The evaluation must see them caught up: equal, bit for bit, to an unsharded
    engine over the tables gathered afterwards -- and close to the unsharded engine trained on the same batches."""
    from foodrec_b200 import Engine, Hyper
    p = Problem(403, 1001, 9, 64, seed=61 + W)
    single, engs = setup(p, W, learner="adam", adam_mode="lazy")
    assert all(g.e.single_pass for g in engs)
    run = sharded.LocalRunner(engs)
    for s in range(4):
        f = p.bpr(300, seed=800 + s)
        single.train_step(f["user_input"], f["item_input"], categories=f["categories"], neg_items=f["neg_item_input"],
                          neg_categories=f["neg_categories"], user_one_hot_label=f["user_one_hot_label"])
        idx = sharded.route_batch(f["user_input"], W)
        for r, g in enumerate(engs):
            g.set_batch(f["user_input"][idx[r]] // W, f["item_input"][idx[r]], neg_items=f["neg_item_input"][idx[r]],
                        global_batch=300)
        assert run.step()[0].cpu().numpy()[9] == 0
    rng = np.random.default_rng(W)
    parts = feed(rng, p, W, 300, 51)
    outs = sharded.LocalRunner(engs).eval_sampled_topk([dev32(u) for u, _, _ in parts], [dev32(c) for _, c, _ in parts],
                                                       [nc for _, _, nc in parts], 10, return_scores=True)
    for g in engs:
        g.e.flush()
    P = sharded.unshard_rows([g.e.P.cpu().numpy() for g in engs], p.U)
    R = sharded.unshard_rows([g.e.R.cpu().numpy() for g in engs], p.I)
    off, idx = label_csr(p)
    fresh = Engine(Hyper(learner="sgd", alpha=ALPHA), P, R, engs[0].e.Cat.cpu().numpy(), engs[0].e.G.cpu().numpy(),
                   max_rows=256, item_cats=p.item_cats, user_label_csr=(off, idx))
    for r, ((u, c, nc), (ids, rank, sc)) in enumerate(zip(parts, outs)):
        nl = len(range(r, p.U, W))
        gu = dev32(np.where((u >= 0) & (u < nl), u.astype(np.int64) * W + r, -1))
        ids1, rank1, sc1 = fresh.eval_sampled_topk(gu, dev32(c), nc, 10, return_scores=True)
        assert torch.equal(ids, ids1) and torch.equal(rank, rank1) and torch.equal(sc, sc1), r
        if len(u):
            _, _, sc2 = single.eval_sampled_topk(gu, dev32(c), nc, 10, return_scores=True)
            assert_close(sc.cpu().numpy(), sc2.cpu().numpy(), rtol=1e-3, what=f"rank {r} vs unsharded training")


@pytest.mark.parametrize("W", [2, 3])
@pytest.mark.parametrize("K", [10, 3, 1])
def test_evaluate_sharded_reproduces_the_reference(W, K):
    """tests/test_reference_golden.py's fixture (a = 0, one-hot recipe rows, the score table in Personal_Memory slot 1:
    the logits ARE the table) through evaluate_sharded: the hits and NDCGs evaluate.py computed, in its order."""
    from foodrec_b200 import Hyper, evaluate_sharded
    load = lambda n: json.load(open(os.path.join(GOLD, n)))
    gd, ge = load("reference_dataset.json"), load("reference_evaluate.json")
    S = np.asarray(ge["S"], np.float32)
    U, I, D = S.shape[0], S.shape[1], 92
    P = np.zeros((U, 5, D), np.float32); P[:, 1, :I] = S
    R = np.zeros((I, D), np.float32); R[np.arange(I), np.arange(I)] = 1.0
    d2c = {str(i): [[1.0], [0.0], [0.0], [0.0]] for i in range(I)}
    ic = np.tile(np.array([1, 0, 0, 0], np.float32), (I, 1))
    h = Hyper(learner="sgd", high_level_score_coefficient=0.0)
    engs = [sharded.ShardedEngine(h, sharded.shard_rows(P, r, W), sharded.shard_rows(R, r, W), np.zeros((4, D), np.float32),
                                  np.zeros((5, 5, D), np.float32), r, W, max_rows=256, item_cats_global=ic, num_users_global=U)
            for r in range(W)]
    hits, ndcgs = evaluate_sharded(sharded.LocalRunner(engs), gd["testRatings"], gd["testNegatives"], K, d2c)
    assert [int(x) for x in hits] == ge[f"hits_K{K}"]
    assert [float(x) for x in ndcgs] == ge[f"ndcgs_K{K}"]
    hits2, _ = evaluate_sharded(sharded.LocalRunner(engs), gd["testRatings"], gd["testNegatives"], K, d2c, round_users=2)
    assert hits2 == hits
    # a test user past Personal_Memory raises, as in evaluate_model -- also one whose row would be a shard's padding
    tr, tn = dict(gd["testRatings"]), dict(gd["testNegatives"])
    tr[str(U)], tn[str(U)] = [0], tn[next(iter(tn))]
    with pytest.raises(IndexError):
        evaluate_sharded(sharded.LocalRunner(engs), tr, tn, K, d2c)


def test_small_capacity_raises():
    from foodrec_b200 import _lib as L
    W = 2
    p = Problem(101, 1001, 5, 64, seed=4)
    _, engs = setup(p, W)
    parts = feed(np.random.default_rng(0), p, W, 100, 51)
    run = sharded.LocalRunner(engs)
    args = ([dev32(u) for u, _, _ in parts], [dev32(c) for _, c, _ in parts], [nc for _, _, nc in parts], 10)
    with pytest.raises(L.FoodRecError, match="capacity"):
        run.eval_sampled_topk(*args, cap=16)
    run.eval_sampled_topk(*args)                    # the default capacity holds


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_nccl_sharded_eval_equals_unsharded():
    """DistRunner.eval_sampled_topk across real processes (torchrun x2, NCCL all-to-alls)."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29643",
                          os.path.join(root, "tests", "dist_eval_check.py")],
                         capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0 and out.stdout.count("DIST_EVAL_CHECK_OK_") == 2, out.stdout[-1500:] + out.stderr[-3000:]
