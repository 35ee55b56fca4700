"""CPU tests of sampled evaluation on row-sharded tables: the numpy restatement of fr_shard_eval_plan (slot map and
request lists), the argument that ranking on slots equals ranking on global ids, and -- with a world_size-2 gloo
group -- which request and row blocks DistRunner.eval_sampled_topk sends where, round by round."""
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from oracle import evaluate_oracle
from tests import sharded_eval_oracle as so

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def check_plan(cand, n_cand, W, I, cap):
    req, slots, slot_ids, over = so.eval_plan(cand, n_cand, W, I, cap)
    assert not over
    cand = np.asarray(cand, np.int64)
    n, stride = cand.shape
    nc = np.clip(np.asarray(n_cand), 0, stride)
    valid = (np.arange(stride)[None] < nc[:, None]) & (cand >= 0) & (cand < I)
    assert ((slots >= 0) == valid).all()
    # every valid candidate maps back to its own global id, through its owner's block
    np.testing.assert_array_equal(slot_ids[slots[valid]], cand[valid])
    np.testing.assert_array_equal(slots[valid] // cap, cand[valid] % W)
    np.testing.assert_array_equal(req[slots[valid]], cand[valid] // W)
    # one slot per distinct id, shared by every repeat (within a user and across users)
    ids, first = np.unique(cand[valid], return_index=True)
    assert len(np.unique(slots[valid])) == len(ids)
    for o in range(W):
        blk = req[o * cap:(o + 1) * cap]
        used = blk[blk >= 0]
        assert (blk[len(used):] == -1).all()                     # front-packed
        assert (np.diff(used) > 0).all()                         # sorted, unique
        np.testing.assert_array_equal(used, np.unique(cand[valid & (np.where(valid, cand, 0) % W == o)] // W))
        assert (used * W + o < I).all()                          # padding rows of the last shard are never requested
    assert (slot_ids[req < 0] == -1).all()
    return req, slots, slot_ids


@pytest.mark.parametrize("W", [1, 2, 3, 8])
def test_plan_restatement_slot_map_and_requests(W):
    rng = np.random.default_rng(W)
    I = 101                                                       # 101 % W != 0 for W > 1: the last shard has padding
    ipr = -(-I // W)
    n, stride = 40, 51
    cand = rng.integers(0, I, (n, stride))
    cand[0, 1:10] = cand[0, 0]                                   # repeats of the held-out item within a user
    cand[1, 5] = cand[1, 20] = 7                                  # repeats within a user
    cand[2:6, 3] = 42                                             # repeats across users
    cand[6, :5] = [I, I + 3, -1, -7, 2**31 - 1]                   # outside the catalog
    pad = [i for i in range(I, W * ipr)]                          # the padding of the last recipe shard
    if pad:
        cand[7, :len(pad)] = pad
    n_cand = rng.integers(0, stride + 1, n)
    n_cand[:8] = stride
    n_cand[8], n_cand[9], n_cand[10] = 0, 1, -3                   # empty lists (a negative count is empty too)
    check_plan(cand, n_cand, W, I, cap=ipr)


def test_plan_restatement_edge_cases():
    # no users, every list empty, W = 1
    req, slots, _, over = so.eval_plan(np.zeros((0, 51), np.int64), np.zeros(0), 3, 100, 5)
    assert slots.shape == (0, 51) and (req == -1).all() and not over
    req, slots, _ = check_plan(np.arange(20).reshape(2, 10), [0, 0], 2, 20, 4)
    assert (slots == -1).all() and (req == -1).all()
    check_plan(np.arange(30).reshape(3, 10) % 13, [10, 4, 10], 1, 13, 13)
    # capacity: the owner keeps its cap smallest rows, the rest are dropped and reported
    req, slots, slot_ids, over = so.eval_plan(np.arange(0, 40, 2).reshape(1, 20), [20], 2, 40, 8)
    assert over and (slots[0, :8] == np.arange(8)).all() and (slots[0, 8:] == -1).all()
    assert (req[8:] == -1).all() and (slot_ids[:8] == np.arange(0, 16, 2)).all()


@pytest.mark.parametrize("W", [2, 3])
def test_ranking_on_slots_equals_ranking_on_global_ids(W):
    """evaluate.py's ranking (dict dedup, nlargest with ties by position) uses ids only for equality: ranking the
    slots and mapping the list back gives the ranking of the global ids.  Integer scores make ties common."""
    rng = np.random.default_rng(5 + W)
    I, n, stride, K = 60, 300, 51, 10
    cand = rng.integers(-2, I + 3, (n, stride))
    cand[::7, 1:4] = cand[::7, :1]
    n_cand = rng.integers(0, stride + 1, n)
    table = rng.integers(0, 6, (n, I + 3)).astype(np.float64)     # score of (user, id): the same for every repeat
    scores = table[np.arange(n)[:, None], np.clip(cand, 0, I + 2)]
    ids_ref, rank_ref = evaluate_oracle.sampled_topk(scores, np.where(cand < I, cand, -1), n_cand, K)
    req, slots, slot_ids = check_plan(cand, n_cand, W, I, cap=-(-I // W))
    ids_s, rank_s = evaluate_oracle.sampled_topk(scores, slots, n_cand, K)
    np.testing.assert_array_equal(np.where(ids_s >= 0, slot_ids[np.maximum(ids_s, 0)], -1), ids_ref)
    np.testing.assert_array_equal(rank_s, rank_ref)


def test_serve_restatement_places_rows_by_slot():
    W, I, D = 3, 50, 4
    R = np.arange(I * D, dtype=np.float32).reshape(I, D)
    cand = np.array([[5, 17, 5, 49, 3, 30]])
    req, slots, slot_ids, _ = so.eval_plan(cand, [6], W, I, 17)
    rbuf = so.serve(R, req.reshape(W, 17), W)
    np.testing.assert_array_equal(rbuf[slots[0]], R[cand[0]])


EVAL_WIRING = textwrap.dedent("""
    import os, sys, torch, torch.distributed as dist
    sys.path.insert(0, "__ROOT__")
    from foodrec_b200.sharded import DistRunner
    dist.init_process_group("gloo")
    r, W, cap, D, K, stride = dist.get_rank(), dist.get_world_size(), 3, 2, 4, 5
    n = 3 if r == 0 else 0                        # rank 1 has no test users: it still serves rank 0 in every round
    state = {"round": 0, "overflow": False}
    class Stub:                                   # the three phases on CPU tensors with recognisable payloads
        rank, world, device = r, W, "cpu"
        def eval_inputs(s, users, cand, n_cand, cc):
            return (torch.arange(n, dtype=torch.int32) * 10, torch.zeros((n, stride), dtype=torch.int32),
                    torch.full((n,), stride, dtype=torch.int32), None)
        def eval_cap(s, rn, st):
            assert (rn, st) == (2, stride), (rn, st)   # the round size and stride every rank agreed on
            return cap
        def eval_plan(s, cd, nc, cap_, cc, flag):  # request j to owner o carries 1000*round + 100*me + 10*o + j
            k = state["round"]
            assert cap_ == cap and cd.shape[0] == ([2, 1][k] if r == 0 else 0)
            if state["overflow"] and r == 1:
                flag.fill_(2.0)
            return torch.tensor([1000 * k + 100 * r + 10 * o + j for o in range(W) for j in range(cap)], dtype=torch.int32)
        def eval_serve(s, rreq):                  # I am the owner: block src = rank src's requests addressed to me
            k = state["round"]
            v = rreq.view(W, cap)
            for src in range(W):
                assert v[src].tolist() == [1000 * k + 100 * src + 10 * r + j for j in range(cap)], v
            return (rreq.float() + 0.5).unsqueeze(1).expand(-1, D).contiguous()
        def eval_rank(s, u, rbuf, K_, ids, rank, sc):   # rows come back in MY slot order o*cap + j
            k = state["round"]
            assert rbuf[:, 0].tolist() == [1000 * k + 100 * r + 10 * o + j + 0.5 for o in range(W) for j in range(cap)]
            ids.fill_(k); rank.copy_(u)
            state["round"] += 1
    run = DistRunner(Stub())
    ids, rank = run.eval_sampled_topk(None, None, None, K, round_users=2)
    assert state["round"] == 2                     # ceil(3 / 2) rounds on BOTH ranks
    if r == 0:
        assert ids.tolist() == [[0] * K, [0] * K, [1] * K] and rank.tolist() == [0, 10, 20]
    else:
        assert ids.shape == (0, K) and rank.shape == (0,)
    # an overflow on one rank is raised on every rank, after the last round
    state.update(round=0, overflow=True)
    try:
        run.eval_sampled_topk(None, None, None, K, round_users=2)
        raise SystemExit("no error")
    except Exception as ex:
        assert "capacity" in str(ex), ex
    assert state["round"] == 2
    sys.stdout.write("EVAL_WIRING_OK_%d\\n" % r); sys.stdout.flush()
""")


def test_dist_runner_eval_wiring_gloo_world2(tmp_path):
    """rounds agreed by all-reduce -> plan -> request blocks to the recipe owners -> serve -> rows back to the user
    owner, block o = owner o's rows -> rank; overflow flags all-reduced."""
    script = tmp_path / "eval_wiring.py"
    script.write_text(EVAL_WIRING.replace("__ROOT__", ROOT))
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29635", str(script)],
                         capture_output=True, text=True, timeout=300, env=env)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert out.stdout.count("EVAL_WIRING_OK_") == 2, out.stdout
