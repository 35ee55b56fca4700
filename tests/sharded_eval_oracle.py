"""numpy restatement of fr_shard_eval_plan (sampled evaluation on row-sharded tables; test-only helper).

A rank's candidates [n, stride] (GLOBAL recipe ids) become one request block per recipe owner o (the sorted unique
local rows id // W of the valid candidates with id % W == o, -1 padded to ``cap``) and a slot per candidate: owner o's
k-th requested row is slot o*cap + k of the received-row buffer.  A candidate is valid iff j < n_cand, 0 <= id and
id < n_items (the global catalog: ids in the padding of the last recipe shard are not valid)."""
from __future__ import annotations

import numpy as np


def eval_plan(cand, n_cand, world, n_items, cap):
    """-> (req [W*cap], slots [n, stride], slot_ids [W*cap], overflow).  An owner with more than ``cap`` distinct
    recipes keeps its ``cap`` smallest rows; the rest of its candidates get slot -1 and ``overflow`` is True."""
    cand = np.asarray(cand, np.int64)
    n, stride = cand.shape
    W = int(world)
    nc = np.clip(np.asarray(n_cand, np.int64).reshape(n), 0, stride)
    valid = (np.arange(stride)[None, :] < nc[:, None]) & (cand >= 0) & (cand < n_items)
    req = np.full(W * cap, -1, np.int64)
    slot_ids = np.full(W * cap, -1, np.int64)
    slots = np.full((n, stride), -1, np.int64)
    overflow = False
    for o in range(W):
        m = valid & (np.where(valid, cand, 0) % W == o)
        rows = np.unique(cand[m] // W)                       # sorted
        k = min(len(rows), cap)
        overflow |= len(rows) > cap
        req[o * cap:o * cap + k] = rows[:k]
        slot_ids[o * cap:o * cap + k] = rows[:k] * W + o
        pos = np.searchsorted(rows, cand[m] // W)
        slots[m] = np.where(pos < cap, o * cap + pos, -1)
    return req, slots, slot_ids, overflow


def serve(R_global, req_blocks, world):
    """What the owners send back: rbuf[o*cap + k] = R_global[req_o[k] * W + o] (a zero row for -1).  ``req_blocks``
    [W, cap] = the request block this rank sent to each owner."""
    W, cap = req_blocks.shape
    out = np.zeros((W * cap,) + R_global.shape[1:], R_global.dtype)
    for o in range(W):
        r = req_blocks[o]
        ok = r >= 0
        out[o * cap:(o + 1) * cap][ok] = R_global[r[ok] * W + o]
    return out
