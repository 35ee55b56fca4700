"""User histories for the tests of the history-aware negative sampler (CPU and GPU).  TEST INFRASTRUCTURE ONLY."""
from __future__ import annotations

import numpy as np

KINDS = ("empty", "short", "ninety", "all_but_one", "whole", "dups", "mixed")


def history_row(kind, I, rng):
    """One user's history (unsorted) of the given kind over a catalog of I recipes."""
    if kind == "empty":
        return np.zeros(0, np.int64)
    if kind == "short":
        return rng.choice(I, size=min(I, int(rng.integers(0, 6))), replace=False)
    if kind == "ninety":
        return rng.choice(I, size=int(0.9 * I), replace=False)
    if kind == "all_but_one":
        return rng.permutation(np.delete(np.arange(I), int(rng.integers(I))))
    if kind == "whole":
        return rng.permutation(I)
    if kind == "dups":
        r = rng.integers(0, I, int(rng.integers(0, 6)))
        return np.repeat(r, rng.integers(1, 4, r.size))
    raise ValueError(kind)


def make_history(kind, U, I, seed):
    """(off int32 [U+1], ids int32) with ascending rows; ``mixed`` cycles the other kinds over the users."""
    rng = np.random.default_rng(seed)
    rows = []
    for u in range(U):
        k = KINDS[u % (len(KINDS) - 1)] if kind == "mixed" else kind
        rows.append(np.sort(history_row(k, I, rng)))
    off = np.zeros(U + 1, np.int64)
    off[1:] = np.cumsum([r.size for r in rows])
    ids = np.concatenate(rows) if rows else np.zeros(0, np.int64)
    return off.astype(np.int32), ids.astype(np.int32)


def samples(U, I, n, seed, outside=True):
    """users [n] (a few outside [0, U) when ``outside``: they have no history) and anchors [n] in [0, I)."""
    rng = np.random.default_rng(seed)
    users = rng.integers(0, U, n)
    if outside and n >= 4:
        users[:2] = [U, -1]
    return users.astype(np.int32), rng.integers(0, I, n).astype(np.int32)


def check_rule(neg, users, pos, off, ids, I):
    """No draw is the anchor or in the user's history unless history and anchor cover the catalog (then (p+1) % I)."""
    rows = {}
    for s in range(neg.shape[0]):
        u, p = int(users[s]), int(pos[s])
        if u not in rows:
            rows[u] = set(ids[off[u]:off[u + 1]].tolist()) if 0 <= u < len(off) - 1 else set()
        seen = rows[u]
        full = len(seen) + (p not in seen) == I           # (histories hold ids in [0, I) only)
        for c in neg[s].tolist():
            assert 0 <= c < I
            if full:
                assert c == (p + 1) % I, (s, u, p, c)
            else:
                assert c != p and c not in seen, (s, u, p, c)
