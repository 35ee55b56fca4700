"""``evaluate_model`` with the reference signature
(``/root/reference/Code/Recommender/evaluate.py:13``), batched on the GPU.

The reference runs one ``sess.run([model.logits])`` per test user (51 rows) and ranks
with ``heapq.nlargest`` over a dict in Python (``evaluate.py:35-66``).  Here every user's
candidate list -- ``[testRatings[u][0]] + testNegatives[u][50:100]`` (``:39-51``) -- goes
to the device in one padded [n_users, stride] array and ``fr_eval_sampled_topk`` does
scoring, dict-dedup and the stable top-K in one launch.  HR / NDCG use the same float64
``math.log`` expressions as ``getHitRatio`` / ``getNDCG`` (``:69-81``).

``evaluate_full_catalog`` is the full-ranking protocol (extension): the held-out item is ranked
against EVERY recipe the user did not train on, through the full-catalog top-K with the user's
training items excluded.

``evaluate_sharded`` is ``evaluate_model`` on row-sharded tables (``sharded.DistRunner`` / ``LocalRunner``).
"""
from __future__ import annotations

import math

import numpy as np


def build_candidates(testRatings, testNegatives, dish_to_category):
    users, cands = [], []
    for user in testRatings:                                   # :28
        if len(testRatings[str(user)]) == 0:                   # :37 (unreachable in the reference data)
            raise ValueError(f"user {user} has no test rating (evaluate.py:37 would return None and crash :29)")
        users.append(int(user))
        cands.append([int(testRatings[str(user)][0])] + [int(x) for x in testNegatives[str(user)][50:100]])
    n = len(users)
    stride = max((len(c) for c in cands), default=1)
    cand = np.zeros((n, stride), np.int32)
    ncand = np.zeros(n, np.int32)
    for r, c in enumerate(cands):
        cand[r, :len(c)] = c
        ncand[r] = len(c)
    # per-candidate category rows from the reference's json map (item -> [[m0],[m1],[m2],[m3]])
    uniq = np.unique(cand)
    lut = np.zeros((int(uniq.max()) + 1 if uniq.size else 1, 4), np.float32)
    for it in uniq:
        lut[it] = np.asarray(dish_to_category[str(int(it))], np.float32).reshape(4)
    return np.asarray(users, np.int32), cand, ncand, lut[cand]


def evaluate_model(sess, model, testRatings, testNegatives, K, dish_to_category):
    users, cand, ncand, ccats = build_candidates(testRatings, testNegatives, dish_to_category)
    if cand.shape[1] > 128:
        raise ValueError("at most 128 candidates per user are supported")
    _, rank = model.engine.eval_sampled_topk(users, cand, ncand, K, cand_cats=ccats)
    rank = rank.cpu().numpy()
    hits = [1 if r >= 0 else 0 for r in rank]                              # getHitRatio :69-73
    ndcgs = [math.log(2) / math.log(int(r) + 2) if r >= 0 else 0 for r in rank]   # getNDCG :76-81
    return hits, ndcgs


def evaluate_sharded(runner, testRatings, testNegatives, K, dish_to_category, round_users=None):
    """``evaluate_model`` on row-sharded tables: ``runner`` is a ``sharded.LocalRunner`` (all ranks in this process) or
    a ``sharded.DistRunner`` (this process is one rank; every rank passes the same ``testRatings`` / ``testNegatives``).
    Each test user is evaluated by its owner (user % W) through the runner's ``eval_sampled_topk``; the hits and NDCGs
    of every user come back in ``testRatings`` order, on every rank, equal to ``evaluate_model`` on the same tables."""
    import torch
    users, cand, ncand, ccats = build_candidates(testRatings, testNegatives, dish_to_category)
    if cand.shape[1] > 128:
        raise ValueError("at most 128 candidates per user are supported")
    kw = {} if round_users is None else {"round_users": int(round_users)}
    local = hasattr(runner, "engs")
    W = runner.W if local else runner.eng.world
    owner = users % W
    per = [np.nonzero(owner == r)[0] for r in range(W)]
    rank = np.empty(len(users), np.int64)
    if local:
        outs = runner.eval_sampled_topk([users[ix] // W for ix in per], [cand[ix] for ix in per], [ncand[ix] for ix in per],
                                        K, cand_cats=[ccats[ix] for ix in per], **kw)
        for ix, (_, rk) in zip(per, outs):
            rank[ix] = rk.cpu().numpy()
    else:
        g = runner.eng
        ix = per[g.rank]
        _, rk = runner.eval_sampled_topk(users[ix] // W, cand[ix], ncand[ix], K, cand_cats=ccats[ix], **kw)
        full = torch.zeros(len(users), dtype=torch.int32, device=rk.device)     # gt_rank + 1 at this rank's users
        full[torch.as_tensor(ix, dtype=torch.int64, device=rk.device)] = rk + 1
        runner.dist.all_reduce(full)
        rank[:] = full.cpu().numpy().astype(np.int64) - 1
    hits = [1 if r >= 0 else 0 for r in rank]                              # getHitRatio :69-73
    ndcgs = [math.log(2) / math.log(int(r) + 2) if r >= 0 else 0 for r in rank]   # getNDCG :76-81
    return hits, ndcgs


def evaluate_full_catalog(sess, model, trainMatrix, testRatings, K, dish_to_category):
    """Full-ranking HR / NDCG@K per test user, in ``testRatings`` order.  The held-out item is
    ``testRatings[u][0]`` (``evaluate.py:40``); the candidates are all recipes with a category except
    the user's training items (``trainMatrix.get(u, [])``, the held-out item itself kept)."""
    users, held, excl = [], [], {}
    for user in testRatings:
        if len(testRatings[str(user)]) == 0:
            raise ValueError(f"user {user} has no test rating (evaluate.py:37 would return None and crash :29)")
        h = int(testRatings[str(user)][0])
        users.append(int(user)); held.append(h)
        excl[str(int(user))] = [int(i) for i in trainMatrix.get(str(user), []) if int(i) != h]
    ids, _ = model.catalog_topk(users, K, dish_to_category, exclude=excl)
    hits, ndcgs = [], []
    for r, h in enumerate(held):
        pos = np.nonzero(ids[r] == h)[0]
        hits.append(1 if pos.size else 0)                                         # getHitRatio :69-73
        ndcgs.append(math.log(2) / math.log(int(pos[0]) + 2) if pos.size else 0)  # getNDCG :76-81
    return hits, ndcgs
