"""Full-ranking HR / NDCG on row-sharded tables (``LocalRunner.full_ranking``, ``evaluate_full_catalog_sharded``)
against one engine holding the same tables: every round is the item-sharded catalog top-K with the users' training
recipes excluded, whose merge is the unsharded engine's top-K, so positions, hits and NDCGs must be identical to
``evaluate_full_catalog`` through ``Model`` / ``Engine.catalog_topk``; a sample of users is checked against
tests/catalog_exclude_oracle.py on the same tables."""
import os

import numpy as np
import pytest
import torch

from foodrec_b200 import sharded
from oracle import synth
from oracle.recommender_oracle import Hyper as OHyper, OracleModel
from tests import catalog_exclude_oracle as xo
from tests.util import Problem, args_ns

pytestmark = pytest.mark.gpu

U, I = 403, 3001          # padding rows in the last user shard and the last recipe shard at W = 2, 3 and 8


def label_csr(p):
    rows, cols = np.nonzero(p.user_labels)
    off = np.zeros(p.U + 1, np.int32); off[1:] = np.cumsum(np.bincount(rows, minlength=p.U))
    return off, cols.astype(np.int32)


def trained(W, D, seed):
    """W engines over one Problem (some recipes without a category) after three BPR steps through the runner, and a
    Model over the tables gathered from them."""
    from foodrec_b200 import Hyper, Model
    p = Problem(U, I, 7, D, seed=seed)
    rng = np.random.default_rng(seed)
    p.item_cats[rng.choice(I, 40, replace=False)] = 0
    args = args_ns(p, learner="adam", lr=0.01)
    off, idx = label_csr(p)
    engs = [sharded.ShardedEngine(Hyper.from_args(args), sharded.shard_rows(p.tb.P, r, W), sharded.shard_rows(p.tb.R, r, W),
                                  p.tb.Cat, p.tb.G, r, W, max_rows=4096, item_cats_global=p.item_cats,
                                  user_label_csr_local=sharded.shard_label_csr(off, idx, r, W, U),
                                  max_label_entries=4096 * p.L, num_users_global=U)
            for r in range(W)]
    run = sharded.LocalRunner(engs)
    live = p.item_cats.sum(1) > 0
    for s in range(3):
        f = p.bpr(600, seed=300 + s)
        keep = live[f["item_input"]] & live[f["neg_item_input"]]      # a recipe without a category has no score
        u, it, neg = f["user_input"][keep], f["item_input"][keep], f["neg_item_input"][keep]
        ix = sharded.route_batch(u, W)
        for r, g in enumerate(engs):
            g.set_batch(u[ix[r]] // W, it[ix[r]], neg_items=neg[ix[r]], global_batch=int(keep.sum()))
        assert run.step()[0].cpu().numpy()[9] == 0
    for g in engs:
        g.e.flush()
    P = sharded.unshard_rows([g.e.P.cpu().numpy() for g in engs], U)
    R = sharded.unshard_rows([g.e.R.cpu().numpy() for g in engs], I)
    Cat, G = engs[0].e.Cat.cpu().numpy(), engs[0].e.G.cpu().numpy()
    assert all(np.isfinite(x).all() for x in (P, R, Cat, G))
    m = Model(args, P, R, Cat, G)
    m.engine.set_item_cats(p.item_cats)
    return p, run, m, OracleModel(P, R, Cat, G, OHyper(), dtype=np.float32)


def data(p, m, W, seed):
    """trainMatrix / testRatings: Zipf-ish histories (a few users without one, one empty, one of 2,600 recipes that
    takes the exact fallback on every shard), test users spread unevenly over the ranks, held-out recipes among the
    user's best (hits), at random, listed twice in the history, without a category, past the catalog and in the padding
    of the last recipe shard."""
    rng = np.random.default_rng(seed)
    train = {str(u): [int(x) for x in synth.zipf_items(rng, I, int(rng.geometric(1 / 20)))] for u in range(U) if u % 11}
    train["4"] = []
    heavy = 2 * W + 1                                   # owner rank 1
    train[str(heavy)] = [int(x) for x in rng.permutation(I)[:2600]]
    users = [u for u in range(U) if u % W != 1 or u % 5 == 0 or u == heavy]
    best, _ = m.engine.catalog_topk(users=np.asarray(users, np.int32), K=40)
    best = best.cpu().numpy()
    test = {}
    for j, u in enumerate(users):
        test[str(u)] = [int(best[j, rng.integers(0, 40)]) if rng.random() < 0.6 else int(rng.integers(0, I))]
    dead = np.nonzero(p.item_cats.sum(1) == 0)[0]
    a, b, c, dup = [u for u in users if u != heavy][:4]
    test[str(a)], test[str(b)], test[str(c)] = [int(dead[0])], [I + 3], [I]
    train[str(dup)] = [test[str(dup)][0]] * 2 + train.get(str(dup), [])
    return train, test


def positions(ids, held):
    hit = ids == held[:, None]
    return np.where(hit.any(1), hit.argmax(1), -1)


GRID = [(2, 1, 128), (2, 10, 64), (2, 100, 128), (3, 1, 64), (3, 10, 128), (3, 100, 64), (8, 1, 128), (8, 10, 64),
        (8, 100, 128)]


@pytest.mark.parametrize("W,K,D", GRID)
def test_full_ranking_equals_the_unsharded_engine(W, K, D):
    from foodrec_b200 import evaluate_full_catalog, evaluate_full_catalog_sharded
    p, run, m, om = trained(W, D, seed=W * 10 + K)
    train, test = data(p, m, W, seed=K + W)
    d2c = {str(i): [[float(x)] for x in p.item_cats[i]] for i in range(I)}
    want = evaluate_full_catalog(None, m, train, test, K, d2c)
    assert sum(want[0]) > 0 and sum(want[0]) < len(test)
    for ru in (None, 37):                                             # one round; several, the last one partial
        assert evaluate_full_catalog_sharded(run, train, test, K, round_users=ru) == want, ru
    # positions through full_ranking itself, with the histories set on the engines
    users = np.asarray([int(u) for u in test], np.int64)
    held = np.asarray([test[u][0] for u in test], np.int64)
    excl = [[i for i in train.get(str(u), []) if i != h] for u, h in zip(users, held)]
    ids, _ = m.engine.catalog_topk(users=users.astype(np.int32), K=K, exclude=excl)
    want_pos = positions(ids.cpu().numpy(), held)
    for g in run.engs:
        g.set_user_history(train)
    per = [np.nonzero(users % W == r)[0] for r in range(W)]
    assert len({len(ix) for ix in per}) > 1                           # uneven users per rank
    pos = run.full_ranking([torch.as_tensor(users[ix] // W, device="cuda") for ix in per], [held[ix] for ix in per], K,
                           round_users=16)
    for ix, ps in zip(per, pos):
        assert ps.is_cuda and ps.dtype == torch.int32
        np.testing.assert_array_equal(ps.cpu().numpy(), want_pos[ix])
    # the heavy history (2,600 of 3,001 recipes): K + its entries in every shard > 256, so every shard's exact fallback
    heavy = 2 * W + 1
    only = [np.asarray([heavy // W] if r == heavy % W else [], np.int64) for r in range(W)]
    hp = run.full_ranking(only, [np.asarray([test[str(heavy)][0]] if r == heavy % W else [], np.int64) for r in range(W)], K)
    assert all(g.e.catalog_fallback_rows() > 0 for g in run.engs)
    assert int(hp[heavy % W][0]) == int(want_pos[list(test).index(str(heavy))])
    # a sample of users against the oracle on the same tables (held-out ids inside the catalog: the oracle indexes them)
    rng = np.random.default_rng(K)
    keys = [k for k in test if test[k][0] < I]
    sample = [keys[i] for i in sorted(rng.choice(len(keys), 40, replace=False))]
    sub = {k: test[k] for k in sample}
    oh, on = xo.evaluate_full_catalog(om, train, sub, K, p.item_cats)
    assert oh == [want[0][list(test).index(k)] for k in sample]
    assert on == [want[1][list(test).index(k)] for k in sample]
    # a test user in the padding rows of the last user shard raises (W = 2, 3, 8: user 403's row is padding)
    with pytest.raises(IndexError):
        evaluate_full_catalog_sharded(run, train, dict(test, **{str(U): [0]}), K)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_nccl_full_ranking_equals_unsharded():
    """DistRunner.full_ranking / evaluate_full_catalog_sharded across real processes (torchrun x2, NCCL)."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29665",
                          os.path.join(root, "tests", "dist_full_ranking_check.py")],
                         capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0 and out.stdout.count("DIST_FULL_RANKING_CHECK_OK_") == 2, \
        out.stdout[-1500:] + out.stderr[-3000:]
