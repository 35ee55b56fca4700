"""CPU restatement of the history-aware negative sampler (csrc/sampler.cu, fr_sample_batch).  TEST INFRASTRUCTURE ONLY.

Built on the pinned generator of ``oracle/sampler_oracle.py`` (Philox4x32-10, Random123 known-answer vectors), whose
``sample_negatives`` is the positive-only rule; with no history this module draws exactly that (the CPU tests check it,
including against ``tests/golden/negative_sampler.npz``).  The reference's negatives are listed items the user never
trained on (``Train_recommender.py:86-93``, ``evaluate.py:39-51``); the rule for sample index g, user u, anchor p,
negative j, catalog size I and history H(u):
  1. the first of 16 attempts cand = mulhi32(philox((g_lo, g_hi, j, a), seed).x0, I) with cand != p, cand not in H(u);
  2. else the first c of (p+1) % I, (p+2) % I, ... with c != p and c not in H(u);
  3. else (H(u) and p cover the catalog) (p + 1) % I."""
from __future__ import annotations

import numpy as np

from oracle.sampler_oracle import MASK, philox4x32_10


def _attempt(g, j, key, attempt, num_items):
    """cand = mulhi32(philox(ctr=(g_lo, g_hi, j, attempt), key).x0, I) for arrays g (uint64), j (uint32)."""
    ctr = np.stack([(g & MASK).astype(np.uint32), (g >> np.uint64(32)).astype(np.uint32), j,
                    np.full(g.shape, attempt, np.uint32)], -1)
    x0 = philox4x32_10(ctr, key)[..., 0].astype(np.uint64)
    return ((x0 * np.uint64(num_items)) >> np.uint64(32)).astype(np.int64)


def sample_negatives(pos_items, n_neg, num_items, seed, sample_offset=0, users=None, history=None):
    """int32 [n, n_neg]: negative j of sample s (index g = sample_offset + s, user u = users[s], anchor p = pos_items[s]
    in [0, I)) by the rule above.  ``history`` = (off, ids): H(u) = ids[off[u]:off[u+1]], every row ascending
    (duplicates allowed); a user outside [0, len(off) - 1) has an empty one, and so has every user without ``users`` /
    ``history``.  Step 1 is vectorised over the attempts; the rare step-2 draws take a loop."""
    pos = np.asarray(pos_items, np.int64).reshape(-1)
    n = pos.shape[0]
    g = (np.arange(n, dtype=np.uint64) + np.uint64(sample_offset))[:, None].repeat(n_neg, 1)
    j = np.arange(n_neg, dtype=np.uint32)[None, :].repeat(n, 0)
    key = np.empty((n, n_neg, 2), np.uint32)
    key[..., 0] = np.uint32(seed & 0xFFFFFFFF); key[..., 1] = np.uint32((seed >> 32) & 0xFFFFFFFF)
    p = pos[:, None].repeat(n_neg, 1)
    out = (p + 1) % num_items
    done = np.zeros((n, n_neg), bool)
    hist = history is not None and users is not None
    if hist:
        off, ids = (np.asarray(x, np.int64).reshape(-1) for x in history)
        rows = np.repeat(np.arange(off.shape[0] - 1, dtype=np.int64), np.diff(off))
        keys = rows * (1 << 32) + ids + (1 << 31)            # ascending: rows in order, each row ascending
        u = np.asarray(users, np.int64).reshape(-1)[:, None].repeat(n_neg, 1)
        has_row = (u >= 0) & (u < off.shape[0] - 1)
    for attempt in range(16):
        cand = _attempt(g, j, key, attempt, num_items)
        take = ~done & (cand != p)
        if hist and keys.size:
            q = u * (1 << 32) + cand + (1 << 31)
            k = np.minimum(np.searchsorted(keys, q), keys.size - 1)
            take &= ~(has_row & (keys[k] == q))
        out = np.where(take, cand, out)
        done |= take
        if done.all():
            break
    if hist:
        free = {}                                            # user -> sorted recipes of [0, I) outside the history
        for s, jj in zip(*np.nonzero(~done)):
            uu, pp = int(u[s, jj]), int(p[s, jj])
            if uu not in free:
                row = ids[off[uu]:off[uu + 1]] if has_row[s, jj] else ids[:0]
                free[uu] = np.setdiff1d(np.arange(num_items, dtype=np.int64), row)
            f = free[uu]
            if f.size == 0:
                continue                                     # step 3: (p + 1) % I is already in place
            k = int(np.searchsorted(f, (pp + 1) % num_items)) % f.size
            c = int(f[k])
            if c == pp:
                c = int(f[(k + 1) % f.size])
            if c != pp:
                out[s, jj] = c
    return out.astype(np.int32)


def sample_negatives_literal(pos_items, n_neg, num_items, seed, sample_offset=0, users=None, history=None):
    """The same rule as a literal loop over draws, attempts and the cyclic walk (the cross-check of the above)."""
    pos = [int(x) for x in np.asarray(pos_items).reshape(-1)]
    n = len(pos)
    g = (np.arange(n, dtype=np.uint64) + np.uint64(sample_offset))[:, None, None].repeat(n_neg, 1).repeat(16, 2)
    j = np.arange(n_neg, dtype=np.uint32)[None, :, None].repeat(n, 0).repeat(16, 2)
    key = np.empty((n, n_neg, 16, 2), np.uint32)
    key[..., 0] = np.uint32(seed & 0xFFFFFFFF); key[..., 1] = np.uint32((seed >> 32) & 0xFFFFFFFF)
    a = np.arange(16, dtype=np.uint32)[None, None, :].repeat(n, 0).repeat(n_neg, 1)
    ctr = np.stack([(g & MASK).astype(np.uint32), (g >> np.uint64(32)).astype(np.uint32), j, a], -1)
    x0 = philox4x32_10(ctr, key)[..., 0]
    out = np.empty((n, n_neg), np.int32)
    for s in range(n):
        seen = set()
        if history is not None and users is not None:
            off, ids = history
            u = int(np.asarray(users).reshape(-1)[s])
            if 0 <= u < len(off) - 1:
                seen = {int(x) for x in ids[int(off[u]):int(off[u + 1])]}
        p = pos[s]
        for jj in range(n_neg):
            item = None
            for att in range(16):
                cand = (int(x0[s, jj, att]) * num_items) >> 32
                if cand != p and cand not in seen:
                    item = cand
                    break
            if item is None:
                for k in range(1, num_items + 1):
                    c = (p + k) % num_items
                    if c != p and c not in seen:
                        item = c
                        break
            if item is None:
                item = (p + 1) % num_items
            out[s, jj] = item
    return out
