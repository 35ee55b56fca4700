"""Restatement of ``/root/reference/Code/Recommender/evaluate.py`` for the
oracle.  TEST INFRASTRUCTURE ONLY.

``evaluate_model`` (``evaluate.py:13-32``) loops every test user; per user
``eval_one_rating`` (``:35-66``) scores [held-out positive] + listed negatives
[50:100], collapses duplicate ids through a dict (later score wins, first
position kept, ``:60-61``), ranks with ``heapq.nlargest`` (stable: ties keep
insertion order, ``:63``) and reports HR (``:69-73``) and
NDCG = ln2/ln(rank+2) (``:76-81``).

Also the full-catalog top-K definition used by the catalog kernel (extension):
score every recipe with the same scorer, ties broken by ascending id.
"""
from __future__ import annotations

import heapq
import math

import numpy as np


def candidates_for(user, testRatings, testNegatives):
    pos = testRatings[str(user)][0]                        # :40
    return [pos] + list(testNegatives[str(user)][50:100])  # :46


def eval_one_rating(model, user, testRatings, testNegatives, K, item_cats):
    if str(user) not in testRatings or len(testRatings[str(user)]) == 0:   # :37
        return None
    cand = candidates_for(user, testRatings, testNegatives)
    u = np.full(len(cand), int(user), np.int64)
    it = np.asarray(cand, np.int64)
    pred = model.scores(u, it, item_cats[it])              # :55-59
    m = {}
    for i, c in enumerate(cand):                           # :60-61
        m[c] = pred[i]
    ranklist = heapq.nlargest(K, m, key=m.get)             # :63
    hr = 1 if cand[0] in ranklist else 0                   # :69-73
    ndcg = 0
    for i, item in enumerate(ranklist):                    # :76-81
        if item == cand[0]:
            ndcg = math.log(2) / math.log(i + 2)
            break
    return hr, ndcg, ranklist


def evaluate_model(model, testRatings, testNegatives, K, item_cats):
    hits, ndcgs, ranks = [], [], []
    for user in testRatings:                               # :28
        hr, ndcg, rl = eval_one_rating(model, user, testRatings, testNegatives, K, item_cats)
        hits.append(hr); ndcgs.append(ndcg); ranks.append(rl)
    return hits, ndcgs, ranks


def sampled_topk(scores, cand, n_cand, K, valid_user=None):
    """``eval_one_rating``'s ranking (dict of the candidates, later score wins,
    first position kept; ``heapq.nlargest``: score desc, ties in insertion
    order), vectorised over many users.  ``scores[r, j]`` is candidate j's score
    for row r.  Candidates past ``n_cand[r]`` and ids < 0 are not in the list.
    Returns top-K ids [n, K] padded with -1 and the rank of candidate 0's id in
    them (-1: not among them); rows with ``valid_user`` False get no list."""
    scores = np.asarray(scores, np.float64); cand = np.asarray(cand, np.int64)
    n, stride = cand.shape
    j = np.arange(stride)
    live = (j[None, :] < np.asarray(n_cand)[:, None]) & (cand >= 0)
    if valid_user is not None:
        live &= np.asarray(valid_user, bool)[:, None]
    r, p = np.nonzero(live)                      # row-major: positions ascending within a row
    c, s = cand[r, p], scores[r, p]
    # dict semantics: group equal (row, id); the first position survives with the last position's score
    o = np.lexsort((p, c, r))
    r, p, c, s = r[o], p[o], c[o], s[o]
    head = np.ones(len(r), bool); head[1:] = (r[1:] != r[:-1]) | (c[1:] != c[:-1])
    tail = np.ones(len(r), bool); tail[:-1] = head[1:]
    r, p, c, s = r[head], p[head], c[head], s[tail]
    # nlargest: score desc, then position asc
    o = np.lexsort((p, -s, r))
    r, c = r[o], c[o]
    start = np.searchsorted(r, np.arange(n))
    k = np.arange(len(r)) - start[r]
    ids = np.full((n, K), -1, np.int64)
    keep = k < K
    ids[r[keep], k[keep]] = c[keep]
    gt = np.where(live[:, 0], cand[:, 0], -1)
    hit = (ids == gt[:, None]) & (gt[:, None] >= 0)
    rank = np.where(hit.any(1), hit.argmax(1), -1)
    return ids, rank


def catalog_scores(model, users, item_cats, dtype=np.float64):
    """Score of every (user, recipe) pair, [len(users), I], by the GEMM form of
    ``inference`` (SURVEY App. A.1) in ``dtype``."""
    P = model.P.astype(dtype); R = model.R.astype(dtype); Cat = model.Cat.astype(dtype)
    cats = item_cats.astype(dtype)
    n = cats.sum(1, keepdims=True)
    w = cats / n
    a = dtype(model.a); b = dtype(model.one_minus_a)
    I, D = R.shape
    Q = np.empty((I, 5 * D), dtype)                       # GEMM form, SURVEY App. A.1
    Q[:, :D] = a * (w @ Cat)
    for c in range(4):
        Q[:, (1 + c) * D:(2 + c) * D] = b * w[:, c:c + 1] * R
    users = np.asarray(users, np.int64)
    return P[users].reshape(len(users), 5 * D) @ Q.T


def catalog_topk(model, users, item_cats, K, dtype=np.float64):
    """Full-catalog scoring (extension; definition = ``inference`` over every
    recipe).  Scores in ``dtype`` from the model's tables; top-K by
    (score desc, id asc)."""
    S = catalog_scores(model, users, item_cats, dtype)
    I = S.shape[1]
    ids = np.empty((len(users), K), np.int64)
    sc = np.empty((len(users), K), dtype)
    ar = np.arange(I)
    for r in range(len(users)):
        order = np.lexsort((ar, -S[r]))[:K]
        ids[r], sc[r] = order, S[r, order]
    return ids, sc
