"""CPU tests of the oracle itself: the closed-form restatement against the literal
one-hot graph (torch autograd), against the committed golden vectors, and the TF-1.x
optimizer / clip semantics of SURVEY App. A.  (The reference ships no tests or golden
vectors of its own -- SURVEY 4 -- so parity is unpinned at the TF boundary.)"""
import importlib.util
import os

import numpy as np
import pytest

from oracle import evaluate_oracle, synth
from oracle.literal_graph import literal_step
from oracle.recommender_oracle import Hyper, OracleModel, sigmoid, sigmoid_ce
from tests.util import Problem, assert_close

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def load_make_golden():
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(GOLD, "make_golden.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


@pytest.mark.parametrize("dups", [False, True])
def test_closed_form_matches_literal_graph(dups):
    p = Problem(40, 30, 7, 8, seed=5)
    f = p.pointwise(24, seed=9)
    if dups:
        f = p.pointwise(24, seed=9, users=np.array([3] * 10 + [7] * 14))
    h = Hyper(learner="sgd", lr=0.05)
    lit = literal_step(p.tb.P, p.tb.R, p.tb.Cat, p.tb.G, f, h)
    om = p.oracle(h)
    s = om.scores(f["user_input"], f["item_input"], f["categories"])
    np.testing.assert_allclose(s, lit["scores"], atol=1e-15)
    P0 = om.P.copy()
    out = om.train_step(f, write_personal=True)
    assert abs(out["loss"] - lit["loss"]) < 1e-14
    assert abs(out["norm"] - lit["global_norm"]) < 1e-14
    dP = np.zeros_like(P0)
    np.add.at(dP, f["user_input"].astype(int), lit["dP_slices"])
    np.testing.assert_allclose(om.P, lit["P_after_write"] - h.lr * out["scale"] * dP, atol=1e-15)
    np.testing.assert_allclose(om.G, lit["G_after_write"], atol=1e-15)
    assert abs(out["general"] - lit["general"]) < 1e-15


def test_gemm_form_equals_inference():
    """App. A.1: s(u,i) = <P[u].reshape(5D), Q[i]> -- the catalog-scoring definition."""
    p = Problem(20, 50, 5, 12, seed=2)
    om = p.oracle(Hyper())
    users = np.arange(20)
    ids, sc = evaluate_oracle.catalog_topk(om, users, p.item_cats, K=50)
    for r in (0, 7, 19):
        ref = om.scores(np.full(50, r), np.arange(50), p.item_cats)
        np.testing.assert_allclose(sc[r], ref[ids[r]], atol=1e-14)
        assert (np.diff(sc[r]) <= 0).all()


def test_loss_and_sigmoid():
    s = np.array([-30.0, -1.5, 0.0, 2.0, 40.0])
    y = np.array([0.0, 1.0, 1.0, 0.0, 1.0])
    ref = np.logaddexp(0.0, s) - s * y          # -[y log sig(s) + (1-y) log(1-sig(s))]
    np.testing.assert_allclose(sigmoid_ce(s, y), ref, rtol=1e-12, atol=1e-16)
    np.testing.assert_allclose(sigmoid(s), 1 / (1 + np.exp(-s)), rtol=1e-12)


def test_clip_uses_undeduplicated_slices():
    """App. A.4: norm^2 = sum_b ||g_b||^2, not ||sum_b g_b||^2 -- differs with duplicates."""
    p = Problem(10, 10, 3, 8, seed=3, scale=30.0)   # large tables -> norm > 5 -> clip active
    f = p.pointwise(16, seed=1, users=np.zeros(16, np.int32))
    om = p.oracle(Hyper(learner="sgd"))
    out = om.train_step(f)
    assert out["norm"] > 5.0 and out["scale"] < 1.0
    np.testing.assert_allclose(out["scale"], 5.0 / out["norm"], rtol=1e-12)


def test_tf1_adam_moves_untouched_rows():
    """App. A.5: TF-1.x sparse Adam decays m,v and moves var for every row."""
    p = Problem(6, 6, 3, 4, seed=4)
    om = p.oracle(Hyper(learner="adam", lr=0.01))
    f1 = p.pointwise(4, seed=1, users=np.array([0, 0, 1, 1]))
    f2 = p.pointwise(4, seed=2, users=np.array([2, 2, 3, 3]))
    om.train_step(f1)
    P_after1 = om.P.copy()
    om.train_step(f2)
    assert np.abs(om.P[0] - P_after1[0]).max() > 0      # row 0 untouched in step 2, still moved
    assert np.abs(om.P[5] - p.tb.P[5]).max() == 0       # never touched, m == 0 -> frozen
    assert om.adam_lr_t(1) == pytest.approx(0.01 * np.sqrt(1 - 0.999) / (1 - 0.9), rel=1e-6)


def test_learner_fallback_is_sgd():
    p = Problem(6, 6, 3, 4)
    assert p.oracle(Hyper(learner="Adam")).learner == "adam"
    assert p.oracle(Hyper(learner="ftrl")).learner == "sgd"


@pytest.mark.parametrize("learner", ["sgd", "adagrad", "rmsprop", "adam"])
@pytest.mark.parametrize("mode", ["pointwise", "bpr"])
def test_oracle_reproduces_golden(learner, mode):
    mg = load_make_golden()
    g = np.load(os.path.join(GOLD, f"train_{learner}_{mode}.npz"))
    seed = int(g["seed"])
    tb, ic, ul = mg.problem(seed)
    om = OracleModel(tb.P, tb.R, tb.Cat, tb.G, Hyper(learner=learner, lr=0.01), dtype=np.float64)
    for s, f in enumerate(mg.feeds(ic, ul, seed, bpr=(mode == "bpr"))):
        o = om.train_step_bpr(f, write_personal=(s == 0)) if mode == "bpr" else om.train_step(f, write_personal=(s == 0))
        assert o["loss"] == pytest.approx(float(g[f"loss{s}"]), rel=1e-13)
        assert o["norm"] == pytest.approx(float(g[f"norm{s}"]), rel=1e-13)
    for k in ("P", "R", "Cat", "G"):
        np.testing.assert_allclose(getattr(om, k), g[k], rtol=1e-13, atol=1e-15)


@pytest.mark.parametrize("learner", ["sgd", "adagrad", "rmsprop", "adam"])
def test_fp32_oracle_within_tolerance_of_fp64(learner):
    p = Problem(200, 100, 9, 32, seed=11)
    h = Hyper(learner=learner, lr=0.01)
    o64, o32 = p.oracle(h, np.float64), p.oracle(h, np.float32)
    for s in range(3):
        f = p.contiguous(64, seed=20 + s, run=20) if s == 1 else p.pointwise(64, seed=20 + s)
        a, b = o64.train_step(f, write_personal=(s == 0)), o32.train_step(f, write_personal=(s == 0))
        assert b["loss"] == pytest.approx(a["loss"], rel=1e-5)
    for k in ("P", "R", "Cat", "G"):
        assert_close(getattr(o32, k), getattr(o64, k), what=k)


def test_bpr_equals_two_pointwise_rows_for_memory_write():
    """The BPR extension writes memory exactly as its two pointwise rows (+1 / -1)."""
    p = Problem(30, 20, 5, 8, seed=6)
    f = p.bpr(10, seed=3)
    h = Hyper(learner="sgd", lr=0.0)          # lr 0: only the memory write changes tables
    om = p.oracle(h); om.train_step_bpr(f, write_personal=True)
    users = np.repeat(f["user_input"], 2)
    items = np.stack([f["item_input"], f["neg_item_input"]], 1).reshape(-1)
    f2 = dict(user_input=users, item_input=items, labels=np.tile([1.0, 0.0], 10),
              write_sign=np.tile([1.0, -1.0], 10).reshape(-1, 1), categories=p.item_cats[items],
              user_one_hot_label=p.user_labels[users])
    o2 = p.oracle(h); o2.train_step(f2, write_personal=True)
    np.testing.assert_allclose(om.G, o2.G, atol=1e-15)
    np.testing.assert_allclose(om.P, o2.P, atol=1e-15)


def test_evaluate_restatement_semantics():
    """evaluate.py:60-63: dict collapse (first position, last score) + stable nlargest."""
    class Fake:
        def scores(self, u, it, cats):
            return np.array([{5: 1.0, 6: 2.0, 7: 2.0, 8: 0.5}[int(i)] for i in it])
    tr = {"0": [5]}
    tn = {"0": list(range(100, 150)) + [6, 7, 8, 5]}      # [50:100] = 6,7,8,5(dup of positive)
    hr, ndcg, rl = evaluate_oracle.eval_one_rating(Fake(), "0", tr, tn, 3, np.zeros((200, 4)))
    assert rl == [6, 7, 5] and hr == 1 and ndcg == pytest.approx(np.log(2) / np.log(4))


@pytest.mark.parametrize("K", [1, 3, 10, 60])
def test_vectorised_sampled_ranking_equals_eval_one_rating(K):
    """evaluate_oracle.sampled_topk (all users at once) against the per-user dict + heapq.nlargest of evaluate.py on
    lists drawn from 12 ids (repeats within a list, of the positive too) with integer scores per POSITION (exact ties,
    and a repeated id whose later occurrence carries a different score)."""
    rng = np.random.default_rng(K)
    n, stride = 400, 51
    cand = rng.integers(0, 12, (n, stride))
    n_cand = rng.integers(1, stride + 1, n)
    n_cand[:4] = [1, 2, 32, 33]
    scores = rng.integers(-3, 4, (n, stride)).astype(np.float64)

    class Fake:
        row = 0

        def scores(self, u, it, cats):
            return scores[self.row, :len(it)]
    fake = Fake()
    ids, rank = evaluate_oracle.sampled_topk(scores, cand, n_cand, K)
    for r in range(n):
        tr = {"0": [int(cand[r, 0])]}
        tn = {"0": [0] * 50 + cand[r, 1:n_cand[r]].tolist()}
        fake.row = r
        _, _, rl = evaluate_oracle.eval_one_rating(fake, "0", tr, tn, K, np.zeros((12, 4)))
        assert ids[r][ids[r] >= 0].tolist() == rl, r
        assert rank[r] == (rl.index(cand[r, 0]) if cand[r, 0] in rl else -1), r
    # ids < 0, positions past n_cand and rows of users outside the table are not ranked
    c2 = cand.copy(); c2[:, 0] = -1
    valid = np.arange(n) % 7 != 0
    ids2, rank2 = evaluate_oracle.sampled_topk(scores, c2, n_cand, K, valid_user=valid)
    assert (ids2[~valid] == -1).all() and (rank2 == -1).all()
    assert not np.isin(ids2[valid & (n_cand == 1)], np.arange(12)).any()


def test_get_train_instances_shape():
    p = Problem(12, 400, 5, 4, seed=8)
    train, tr, tn = synth.make_reference_dataset(12, 400, seed=1, pos_range=(3, 9))
    d2c, u2l = synth.reference_side_maps(p.item_cats, p.user_labels)
    u, i, y, c, ws, ul = synth.get_train_instances(train, tn, d2c, u2l, seed=3)
    assert len(u) == len(i) == len(y) == len(c) == len(ws) == len(ul)
    assert isinstance(u[0], str) and np.asarray(c).shape[1:] == (4, 1)
    first = [k for k in range(len(u)) if u[k] == "0"]
    assert first == list(range(len(first)))                # user-contiguous
    assert y[len(train["0"])] == 0 and ws[len(train["0"])] == [-1.0]


# ---------------------------------------------------------------- negative sampler
def test_philox_matches_random123_known_answers():
    """The sampler's generator is pinned to the PUBLISHED Philox4x32-10 known-answer vectors
    (Random123 v1.09 kat_vectors) -- the one part of this oracle with real golden vectors."""
    from oracle import sampler_oracle as so
    for ctr, key, want in so.KAT:
        got = so.philox4x32_10(np.array(ctr, np.uint32), np.array(key, np.uint32))
        assert got.tolist() == list(want)


def test_negative_sampler_properties_and_golden():
    from oracle import sampler_oracle as so
    rng = np.random.default_rng(1)
    pos = rng.integers(0, 50, 4000)
    neg = so.sample_negatives(pos, 8, 50, seed=20260105)
    assert neg.shape == (4000, 8) and neg.dtype == np.int32
    assert ((neg >= 0) & (neg < 50)).all() and (neg != pos[:, None]).all()          # never the positive
    cnt = np.bincount(neg.reshape(-1), minlength=50)
    assert cnt.min() > 0.7 * cnt.mean() and cnt.max() < 1.3 * cnt.mean()            # uniform over the catalog
    # a window of the stream equals the same rows of the whole stream (counter-based: no hidden state)
    np.testing.assert_array_equal(so.sample_negatives(pos[100:160], 8, 50, seed=20260105, sample_offset=100), neg[100:160])
    g = np.load(os.path.join(GOLD, "negative_sampler.npz"))
    np.testing.assert_array_equal(so.sample_negatives(g["pos"], int(g["n_neg"]), int(g["num_items"]), int(g["seed"]),
                                                      int(g["offset"])), g["neg"])
    # two recipes: every draw that hits the positive is re-drawn, the answer is forced
    two = so.sample_negatives(np.array([0, 1, 1, 0]), 4, 2, seed=3)
    np.testing.assert_array_equal(two, np.array([[1] * 4, [0] * 4, [0] * 4, [1] * 4], np.int32))
