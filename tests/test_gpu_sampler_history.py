"""Negatives that skip each user's history (fr_set_user_history / fr_sample_batch) against the restatement in
tests/sampler_history_oracle.py: every layout and history shape bit for bit, the history-free path equal to the existing
entry points, the validation of the history, training and evaluation on the drawn batches, and row-sharded draws equal
to the single-GPU draws."""
import ctypes as C

import numpy as np
import pytest
import torch

from foodrec_b200 import Engine, Hyper, _lib as L, sharded
from oracle import evaluate_oracle, sampler_oracle as base, synth
from oracle.recommender_oracle import Hyper as OHyper, OracleModel
from tests import sampler_history_oracle as so
from tests.sampler_history_cases import KINDS, check_rule, make_history, samples
from tests.util import Problem, assert_close

pytestmark = pytest.mark.gpu


def dev32(x):
    return torch.as_tensor(np.ascontiguousarray(x, np.int32), device="cuda")


def sampler_engine(U, I):
    tb = synth.make_tables(U, min(I, 64), 3, 8, seed=1)
    return Engine(Hyper(learner="sgd"), tb.P, np.zeros((I, 8), np.float32), tb.Cat, tb.G, max_rows=128)


def layouts_equal_the_oracle(e, users, pos, n_neg, I, seed, offset, hist):
    """All four layouts of fr_sample_batch against the oracle's [n, n_neg] draws; returns them."""
    neg = so.sample_negatives(pos, n_neg, I, seed, offset, users=None if hist is None else users, history=hist)
    ex = hist is not None
    got = e.sample_negatives(pos, n_neg, seed, offset, exclude_seen=ex, users=users).cpu().numpy()
    assert np.array_equal(got, neg), "FR_SAMPLE_NEG"
    uu, it = e.sample_bpr_batch(users, pos, n_neg, seed, offset, exclude_seen=ex)
    it = it.cpu().numpy().reshape(-1, 2)
    assert np.array_equal(uu.cpu().numpy(), np.repeat(users, n_neg))
    assert np.array_equal(it[:, 0], np.repeat(pos, n_neg)) and np.array_equal(it[:, 1], neg.reshape(-1)), "FR_SAMPLE_BPR"
    pu, pi, pl = (x.cpu().numpy() for x in e.sample_pointwise_batch(users, pos, n_neg, seed, offset, exclude_seen=ex))
    assert np.array_equal(pu, np.repeat(users, 1 + n_neg))
    assert np.array_equal(pi, np.column_stack([pos, neg]).reshape(-1)), "FR_SAMPLE_POINTWISE"
    assert np.array_equal(pl, np.tile(np.r_[1.0, np.zeros(n_neg)], len(pos)).astype(np.float32))
    cand, nc = e.sample_eval_candidates(users, pos, n_neg, seed, offset, exclude_seen=ex)
    assert np.array_equal(cand.cpu().numpy(), np.column_stack([pos, neg])), "FR_SAMPLE_CAND"
    assert (nc.cpu().numpy() == 1 + n_neg).all()
    return neg


@pytest.mark.parametrize("I", [2, 5, 200_000, 1_000_003])
@pytest.mark.parametrize("kind", KINDS)
def test_every_layout_is_bit_exact(I, kind):
    U = 12 if I < 10_000 else 5
    off, ids = make_history(kind, U, I, seed=I % 997 + len(kind))
    users, pos = samples(U, I, 64, seed=I + 1)
    e = sampler_engine(U, I)
    e.set_user_history((off, ids))
    for n_neg, offset in ((1, 0), (8, 1 << 33), (50, 123_456_789)):
        neg = layouts_equal_the_oracle(e, users, pos, n_neg, I, 20260105 + n_neg, offset, (off, ids))
        check_rule(neg, users, pos, off, ids, I)
    e.close()


@pytest.mark.parametrize("I,n,n_neg,offset", [(200_000, 4096, 8, 0), (5, 3000, 8, 7), (2, 64, 4, 0),
                                              (200_000, 512, 8, 1 << 33), (1_000_003, 70_001, 1, 123456789)])
def test_without_history_equals_the_existing_entry_points(I, n, n_neg, offset):
    """use_history = 0 (with a history set or not) draws what fr_sample_negatives / fr_sample_bpr_batch draw."""
    e = sampler_engine(16, I)
    rng = np.random.default_rng(I + n)
    pos = dev32(rng.integers(0, I, n)); users = dev32(rng.integers(0, 16, n))
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    a = torch.empty((n, n_neg), dtype=torch.int32, device="cuda")
    L.check(e.handle, e.lib.fr_sample_negatives(e.handle, C.c_void_p(pos.data_ptr()), n, n_neg, 20260105, offset,
                                                C.c_void_p(a.data_ptr()), st))
    bu = torch.empty(n * n_neg, dtype=torch.int32, device="cuda"); bi = torch.empty(2 * n * n_neg, dtype=torch.int32, device="cuda")
    L.check(e.handle, e.lib.fr_sample_bpr_batch(e.handle, C.c_void_p(users.data_ptr()), C.c_void_p(pos.data_ptr()), n, n_neg,
                                                20260105, offset, 0, C.c_void_p(bu.data_ptr()), C.c_void_p(bi.data_ptr()), st))
    for with_history in (False, True):
        if with_history:
            e.set_user_history(make_history("whole", 16, I, seed=3) if I < 10 else make_history("short", 16, I, seed=3))
        assert torch.equal(e.sample_negatives(pos, n_neg, 20260105, offset), a)
        u2, i2 = e.sample_bpr_batch(users, pos, n_neg, 20260105, offset)
        assert torch.equal(u2, bu) and torch.equal(i2, bi)
    assert np.array_equal(a.cpu().numpy(), base.sample_negatives(pos.cpu().numpy(), n_neg, I, 20260105, offset))
    e.close()


def test_set_user_history_validates_and_clears():
    U, I = 6, 50
    e = sampler_engine(U, I)
    pos = np.arange(U, dtype=np.int32); users = np.arange(U, dtype=np.int32)
    with pytest.raises(L.FoodRecError, match="history"):
        e.sample_negatives(pos, 4, 1, exclude_seen=True, users=users)              # nothing set: FR_ERR_STATE
    good = make_history("short", U, I, seed=1)
    off, ids = dev32(good[0]), dev32(np.r_[good[1], 0])
    bad_rows = np.array([0, 2, 2, 4, 4, 4, 4], np.int32), np.array([5, 3, 1, 7], np.int32)
    bad_order = np.array([0, 2, 1, 4, 4, 4, 4], np.int32), np.array([3, 5, 1, 7], np.int32)
    bad_start = np.array([1, 2, 2, 4, 4, 4, 4], np.int32), np.array([3, 5, 1, 7], np.int32)
    for (o, i), msg in ((bad_rows, "ascending"), (bad_order, "non-decreasing"), (bad_start, r"off\[0\]")):
        e.set_user_history((off, ids))
        with pytest.raises(L.FoodRecError, match=msg):
            e.set_user_history((dev32(o), dev32(i)))                           # device tensors: the library checks
        with pytest.raises(L.FoodRecError, match="history"):
            e.sample_negatives(pos, 4, 1, exclude_seen=True, users=users)          # a rejected history is not kept
    e.set_user_history((off, ids))
    got = e.sample_negatives(pos, 4, 1, exclude_seen=True, users=users).cpu().numpy()
    assert np.array_equal(got, so.sample_negatives(pos, 4, I, 1, users=users, history=good))
    rc = e.lib.fr_sample_batch(e.handle, L.FR_SAMPLE_NEG, None, C.c_void_p(dev32(pos).data_ptr()), U, 4, 1, 0, 0, 1, None,
                               C.c_void_p(torch.empty(4 * U, dtype=torch.int32, device="cuda").data_ptr()), None, None)
    assert rc == L.FR_ERR_ARG                                                      # the history needs users
    e.set_user_history(None)
    rc = e.lib.fr_sample_batch(e.handle, L.FR_SAMPLE_NEG, C.c_void_p(dev32(users).data_ptr()), C.c_void_p(dev32(pos).data_ptr()),
                               U, 4, 1, 0, 0, 1, None, C.c_void_p(torch.empty(4 * U, dtype=torch.int32, device="cuda").data_ptr()),
                               None, None)
    assert rc == L.FR_ERR_STATE
    torch.cuda.synchronize()
    e.close()


# ---------------------------------------------------------------- training on the drawn batches
def label_csr(p):
    rows, cols = np.nonzero(p.user_labels)
    off = np.zeros(p.U + 1, np.int32); off[1:] = np.cumsum(np.bincount(rows, minlength=p.U))
    return off, cols.astype(np.int32)


def train_history(p, seed):
    """Training recipes per user: 30 to 200 of them (the whole range of the tiny catalog's re-draw rates)."""
    rng = np.random.default_rng(seed)
    return {str(u): rng.choice(p.I, int(rng.integers(30, 200)), replace=False).tolist() for u in range(p.U)}


@pytest.mark.parametrize("learner,mode", [("adagrad", "pointwise"), ("sgd", "pointwise"), ("adagrad", "bpr")])
def test_sampled_step_with_history_matches_oracle(learner, mode):
    from foodrec_b200 import history_csr
    p = Problem(300, 500, 9, 64, seed=5)
    e = Engine(Hyper(learner=learner, lr=0.05), p.tb.P, p.tb.R, p.tb.Cat, p.tb.G, max_rows=2 * 9 * 64,
               max_label_entries=2 * 9 * 64 * p.L, item_cats=p.item_cats, user_labels=p.user_labels)
    om = p.oracle(OHyper(learner=learner, lr=0.05))
    tm = train_history(p, 1)
    e.set_user_history(tm)
    hist = history_csr(tm, p.U)
    rng = np.random.default_rng(2)
    for s in range(2):
        users = rng.integers(0, p.U, 64).astype(np.int32); pos = rng.integers(0, p.I, 64).astype(np.int32)
        e.train_step_sampled(users, pos, 8, seed=99, sample_offset=64 * s, mode=mode, exclude_seen=True)
        e.read_scalars()
        neg = so.sample_negatives(pos, 8, p.I, seed=99, sample_offset=64 * s, users=users, history=hist)
        check_rule(neg, users, pos, *hist, p.I)
        if mode == "bpr":
            uu, pp, nn = np.repeat(users, 8), np.repeat(pos, 8), neg.reshape(-1)
            om.train_step_bpr(dict(user_input=uu, item_input=pp, neg_item_input=nn, categories=p.item_cats[pp],
                                   neg_categories=p.item_cats[nn], user_one_hot_label=p.user_labels[uu]))
        else:
            uu, it = np.repeat(users, 9), np.column_stack([pos, neg]).reshape(-1)
            y = np.tile(np.r_[1.0, np.zeros(8)], 64).astype(np.float32)
            om.train_step(dict(user_input=uu, item_input=it, labels=y, write_sign=np.where(y > 0.5, 1.0, -1.0).reshape(-1, 1),
                               categories=p.item_cats[it], user_one_hot_label=p.user_labels[uu]))
    t = e.tables()
    for k in ("P", "R", "Cat", "G"):
        assert_close(t[k], getattr(om, k), what=f"sampled {mode} {learner} {k}")
    e.close()


def bf16_ulps(x, ref):
    a = np.ascontiguousarray(x, np.float32).view(np.int32) >> 16
    b = np.ascontiguousarray(ref, np.float32).view(np.int32) >> 16
    return np.abs(a.astype(np.int64) - b.astype(np.int64))


def sharded_setup(p, W, bf16):
    h = Hyper(learner="adagrad", lr=0.05)
    td = "bf16" if bf16 else "float32"
    off, idx = label_csr(p)
    single = Engine(h, p.tb.P, p.tb.R, p.tb.Cat, p.tb.G, max_rows=4096, item_cats=p.item_cats, user_label_csr=(off, idx),
                    max_label_entries=4096 * p.L, table_dtype=td)
    engs = [sharded.ShardedEngine(h, sharded.shard_rows(p.tb.P, r, W), sharded.shard_rows(p.tb.R, r, W), p.tb.Cat, p.tb.G, r, W,
                                  max_rows=4096, item_cats_global=p.item_cats,
                                  user_label_csr_local=sharded.shard_label_csr(off, idx, r, W, p.U),
                                  max_label_entries=4096 * p.L, table_dtype=td, num_users_global=p.U)
            for r in range(W)]
    return single, engs


@pytest.mark.parametrize("W", [2, 3])
@pytest.mark.parametrize("bf16", [False, True])
@pytest.mark.parametrize("mode", ["pointwise", "bpr"])
def test_row_sharded_draws_and_step_equal_single_gpu(W, bf16, mode):
    p = Problem(403, 257, 9, 64, seed=61)
    single, engs = sharded_setup(p, W, bf16)
    tm = train_history(p, 4)
    single.set_user_history(tm)
    for g in engs:
        g.set_user_history(tm)
    rng = np.random.default_rng(9)
    n, n_neg = 120, 4
    users = rng.integers(0, p.U, n).astype(np.int32); pos = rng.integers(0, p.I, n).astype(np.int32)
    order = np.argsort(users % W, kind="stable")                  # pairs grouped by owner; sample index = position in this order
    users, pos = users[order], pos[order]
    group = 1 + n_neg if mode == "pointwise" else n_neg
    # the ranks' batches, together, are the single-GPU batch
    if mode == "pointwise":
        want = single.sample_pointwise_batch(users, pos, n_neg, 77, 5, exclude_seen=True)
    else:
        want = single.sample_bpr_batch(users, pos, n_neg, 77, 5, exclude_seen=True) + (None,)
    parts, start = [], 0
    for r, g in enumerate(engs):
        m = users % W == r
        if mode == "pointwise":
            got = g.e.sample_pointwise_batch(users[m] // W, pos[m], n_neg, 77, 5 + start, num_items=p.I, exclude_seen=True)
        else:
            got = g.e.sample_bpr_batch(users[m] // W, pos[m], n_neg, 77, 5 + start, num_items=p.I, exclude_seen=True) + (None,)
        parts.append([x if x is None else x.cpu().numpy() for x in got])
        parts[-1][0] = parts[-1][0] * W + r                       # local rows -> global users
        start += int(m.sum())
    for k in range(3):
        if want[k] is not None:
            assert np.array_equal(np.concatenate([q[k] for q in parts]), want[k].cpu().numpy()), (mode, k)
    # one step: the tables match the single engine's
    single.train_step_sampled(users, pos, n_neg, seed=77, sample_offset=5, mode=mode, exclude_seen=True)
    v1 = single.read_scalars().copy()
    start = 0
    for r, g in enumerate(engs):
        m = users % W == r
        g.set_batch_sampled(users[m] // W, pos[m], n_neg, seed=77, sample_offset=5 + start, global_batch=n * group, mode=mode,
                            exclude_seen=True)
        start += int(m.sum())
    v = sharded.LocalRunner(engs).step()[0].cpu().numpy()
    assert v[9] == 0 and v[0] == pytest.approx(v1[0], rel=1e-5)
    ts = {"P": sharded.unshard_rows([g.e.tables()["P"] for g in engs], p.U), "R": sharded.unshard_rows([g.e.tables()["R"] for g in engs], p.I)}
    tr = single.tables()
    for k in ("P", "R"):
        if bf16:
            d = bf16_ulps(ts[k], tr[k])
            assert (d <= 1).all() and (d == 0).mean() >= 0.999, (k, int((d > 1).sum()), float((d == 0).mean()))
        else:
            assert_close(ts[k], tr[k], what=f"W={W} {mode} {k}")
    single.close()


# ---------------------------------------------------------------- evaluation candidates
def test_eval_candidates_rank_like_the_reference_and_shard():
    """Candidates [held-out, 50 unseen negatives]: the kernel's HR / NDCG on them equal evaluate.py's (the oracle) on the
    same lists, and the row-sharded draws + sharded ranking equal the single engine's."""
    p = Problem(203, 700, 9, 64, seed=31)
    W = 3
    single, engs = sharded_setup(p, W, False)
    tm = train_history(p, 6)
    single.set_user_history(tm)
    for g in engs:
        g.set_user_history(tm)
    from foodrec_b200 import history_csr
    off, ids = history_csr(tm, p.U)
    users = np.argsort(np.arange(p.U) % W, kind="stable").astype(np.int32)     # test users grouped by owner
    held = np.array([tm[str(u)][0] for u in users], np.int32)                    # (a recipe the user has: the worst case)
    held[::3] = np.random.default_rng(1).integers(0, p.I, len(held[::3]))
    cand, nc = single.sample_eval_candidates(users, held, 50, seed=11)
    cand_h = cand.cpu().numpy()
    assert np.array_equal(cand_h[:, 0], held)
    for r, u in enumerate(users):
        seen = set(ids[off[u]:off[u + 1]].tolist())
        assert not (set(cand_h[r, 1:].tolist()) & (seen | {int(held[r])})), r
    want = so.sample_negatives(held, 50, p.I, 11, users=users, history=(off, ids))
    assert np.array_equal(cand_h[:, 1:], want)
    # HR / NDCG against evaluate.py on the same lists
    K = 10
    ids_k, rank = single.eval_sampled_topk(users, cand, nc, K)
    rank = rank.cpu().numpy()
    om = OracleModel(p.tb.P, p.tb.R, p.tb.Cat, p.tb.G, OHyper(), dtype=np.float64)
    tr = {str(int(u)): [int(h)] for u, h in zip(users, held)}
    tn = {str(int(u)): [0] * 50 + cand_h[r, 1:].tolist() for r, u in enumerate(users)}
    hits, ndcgs, _ = evaluate_oracle.evaluate_model(om, tr, tn, K, p.item_cats)
    for r, u in enumerate(users):
        s = om.scores(np.full(51, u), cand_h[r], p.item_cats[cand_h[r]])
        others = np.delete(s, np.nonzero(cand_h[r] == held[r])[0])
        if np.min(np.abs(others - s[0])) <= 1e-5 * np.abs(s).max():
            continue                                                              # a near tie with the held-out item
        assert hits[r] == int(rank[r] >= 0), r
        assert ndcgs[r] == pytest.approx(np.log(2) / np.log(rank[r] + 2) if rank[r] >= 0 else 0.0, rel=1e-12), r
    # row-sharded: each rank draws its users' lists with the global index of its first test user
    start, parts = 0, []
    for r, g in enumerate(engs):
        m = users % W == r
        c_r, n_r = g.sample_eval_candidates(users[m] // W, held[m], 50, seed=11, sample_offset=start)
        assert torch.equal(c_r, cand[start:start + int(m.sum())]), r
        parts.append((dev32(users[m] // W), c_r, n_r))
        start += int(m.sum())
    outs = sharded.LocalRunner(engs).eval_sampled_topk([u for u, _, _ in parts], [c for _, c, _ in parts],
                                                       [n for _, _, n in parts], K)
    start = 0
    for r, (ids_r, rank_r) in enumerate(outs):
        k = parts[r][0].numel()
        assert torch.equal(ids_r, ids_k[start:start + k]) and torch.equal(rank_r.cpu(), torch.as_tensor(rank[start:start + k])), r
        start += k
    single.close()


# ---------------------------------------------------------------- cfg5 shape
def test_cfg5_shape_is_bit_exact():
    """1M users, 200k recipes, Zipf(1.05) histories of mean length 20 (~20M ids), 32,768 positives x 8 negatives."""
    import synth_data
    U, I = 1_000_000, 200_000
    rng = np.random.default_rng(2026)
    lens = rng.geometric(1 / 20, U)
    off = np.zeros(U + 1, np.int64); off[1:] = np.cumsum(lens)
    ids = synth_data.zipf_items(rng, I, int(off[-1])).astype(np.int64)
    row = np.repeat(np.arange(U), lens)
    ids = ids[np.lexsort((ids, row))].astype(np.int32)
    off = off.astype(np.int32)
    assert 18e6 < ids.size < 22e6
    e = Engine(Hyper(learner="sgd"), np.zeros((U, 5, 4), np.float32), np.zeros((I, 4), np.float32), np.zeros((4, 4), np.float32),
               np.zeros((3, 5, 4), np.float32), max_rows=128)
    e.set_user_history((dev32(off), dev32(ids)))
    users = rng.integers(0, U, 32768).astype(np.int32)
    pos = synth_data.zipf_items(rng, I, 32768).astype(np.int32)
    for offset in (0, 1 << 33):
        _, items = e.sample_bpr_batch(users, pos, 8, 20260105, offset, exclude_seen=True)
        want = so.sample_negatives(pos, 8, I, 20260105, offset, users=users, history=(off, ids))
        assert np.array_equal(items.cpu().numpy().reshape(-1, 2)[:, 1], want.reshape(-1))
        plain = base.sample_negatives(pos, 8, I, 20260105, offset)
        assert (want != plain).any()                              # the history changed some draws ...
        for s in np.nonzero((want != plain).any(1))[0][:200]:     # ... each to one outside it
            assert not set(want[s].tolist()) & set(ids[off[users[s]]:off[users[s] + 1]].tolist())
    e.close()
