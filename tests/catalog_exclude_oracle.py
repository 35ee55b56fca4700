"""CPU definition of full-catalog top-K with per-user exclusion lists and of full-ranking evaluation -- TEST
INFRASTRUCTURE ONLY (not collected by pytest).

``catalog_topk_excluding`` is ``oracle/evaluate_oracle.catalog_topk`` (same GEMM-form scores, same (score desc, id asc)
order) with each row's listed recipes removed from the candidates before the sort; ids the table does not have are
ignored, and a row left with fewer than K candidates is padded with -1 / -inf.  ``evaluate_full_catalog`` restates the
full-ranking protocol: the held-out item ``testRatings[u][0]`` (``evaluate.py:40``) ranked against every recipe with a
category that is not among the user's training items, HR / NDCG as ``evaluate.py:69-81``."""
from __future__ import annotations

import math

import numpy as np


def catalog_scores(model, users, item_cats, dtype=np.float64):
    """[n, I] scores in the GEMM form of ``evaluate_oracle.catalog_topk`` (bit-identical to it)."""
    P = model.P.astype(dtype); R = model.R.astype(dtype); Cat = model.Cat.astype(dtype)
    cats = item_cats.astype(dtype)
    n = cats.sum(1, keepdims=True)
    w = cats / n
    a = dtype(model.a); b = dtype(model.one_minus_a)
    I, D = R.shape
    Q = np.empty((I, 5 * D), dtype)
    Q[:, :D] = a * (w @ Cat)
    for c in range(4):
        Q[:, (1 + c) * D:(2 + c) * D] = b * w[:, c:c + 1] * R
    users = np.asarray(users, np.int64)
    return P[users].reshape(len(users), 5 * D) @ Q.T


def catalog_topk_excluding(model, users, item_cats, K, exclude, dtype=np.float64):
    """Top-K by (score desc, id asc) per user row among the recipes not listed in ``exclude[row]``."""
    S = catalog_scores(model, users, item_cats, dtype)
    I = S.shape[1]
    ar = np.arange(I)
    ids = np.full((S.shape[0], K), -1, np.int64)
    sc = np.full((S.shape[0], K), -np.inf, dtype)
    for r in range(S.shape[0]):
        keep = np.ones(I, bool)
        ex = np.asarray(exclude[r], np.int64).reshape(-1)
        keep[ex[(ex >= 0) & (ex < I)]] = False
        cand = ar[keep]
        order = cand[np.lexsort((cand, -S[r, cand]))][:K]
        ids[r, :order.size], sc[r, :order.size] = order, S[r, order]
    return ids, sc


def evaluate_full_catalog(model, trainMatrix, testRatings, K, item_cats):
    """Full-ranking HR / NDCG@K per test user (``testRatings`` order); scores in float64, recipes without a category
    never ranked (the catalog path does not return them)."""
    P = model.P.astype(np.float64); R = model.R.astype(np.float64); Cat = model.Cat.astype(np.float64)
    cats = item_cats.astype(np.float64)
    n = cats.sum(1)
    live = n > 0
    w = np.where(live[:, None], cats / np.where(live, n, 1)[:, None], 0.0)
    a = np.float64(model.a); b = np.float64(model.one_minus_a)
    I = R.shape[0]
    hits, ndcgs = [], []
    for user in testRatings:
        u, h = int(user), int(testRatings[user][0])
        if not live[h]:
            hits.append(0); ndcgs.append(0)
            continue
        s = a * (w @ (Cat @ P[u, 0])) + b * ((R @ P[u, 1:].T) * w).sum(1)
        cand = live.copy()
        tr = np.asarray([int(i) for i in trainMatrix.get(user, []) if int(i) != h], np.int64)
        cand[tr[(tr >= 0) & (tr < I)]] = False
        cand[h] = True
        ids = np.nonzero(cand)[0]
        rank = int(((s[ids] > s[h]) | ((s[ids] == s[h]) & (ids < h))).sum())   # recipes ranked before h
        hits.append(1 if rank < K else 0)                                       # getHitRatio :69-73
        ndcgs.append(math.log(2) / math.log(rank + 2) if rank < K else 0)       # getNDCG :76-81
    return hits, ndcgs
