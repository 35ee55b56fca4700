"""GPU parity tests: the CUDA path, called through the C ABI (ctypes), against the
CPU oracle on the same seeded inputs and against the committed golden vectors.

Tolerance (north_star): bit-exact for indices / top-K ids; 1e-5 relative for fp32
scores, losses and updated embeddings (tests/util.py:assert_close), judged against the
float64 oracle."""
import importlib.util
import os

import numpy as np
import pytest
import torch

from oracle import evaluate_oracle, synth
from oracle.recommender_oracle import Hyper as OHyper, OracleModel
from tests.util import Problem, args_ns, assert_close, assert_close_adam

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def make_engine(p, learner="adam", lr=0.01, adam_mode="lazy", max_rows=4096, resident=False, single_pass=None, **hk):
    from foodrec_b200 import Engine, Hyper
    h = Hyper(learner=learner, lr=lr, **hk)
    return Engine(h, p.tb.P, p.tb.R, p.tb.Cat, p.tb.G, max_rows=max_rows, adam_mode=adam_mode,
                  max_label_entries=max_rows * p.L, single_pass=single_pass,
                  item_cats=p.item_cats if resident else None,
                  user_labels=p.user_labels if resident else None)


def step_gpu(e, f, personal=False, bpr=False, compact=False):
    kw = {}
    if bpr:
        kw = dict(neg_items=f["neg_item_input"], neg_categories=None if compact else f["neg_categories"])
    e.train_step(f["user_input"], f["item_input"], labels=None if bpr else f["labels"],
                 categories=None if compact else f["categories"],
                 write_sign=None if (bpr or compact) else f["write_sign"],
                 user_one_hot_label=None if compact else f["user_one_hot_label"],
                 write_personal=personal, **kw)
    return e.read_scalars()


def compare_tables(e, om, what="", om32=None):
    """om32 (the float32 numpy oracle stepped on the same feeds) is given for Adam only:
    see tests/util.py:assert_close_adam."""
    t = e.tables()
    for k in ("P", "R", "Cat", "G"):
        if om32 is not None and k != "G":
            assert_close_adam(t[k], getattr(om, k), getattr(om32, k), what=f"{what}{k}")
        else:
            assert_close(t[k], getattr(om, k), what=f"{what}{k}")


# ---------------------------------------------------------------- sort
@pytest.mark.parametrize("n,nbits", [(1, 3), (31, 5), (2048, 8), (2049, 9), (5000, 20), (70000, 17), (100000, 1),
                                     (400000, 19)])     # > 128 tiles: separate scan path
def test_radix_sort_is_stable_and_exact(n, nbits):
    p = Problem(8, 8, 3, 8)
    e = make_engine(p, max_rows=max(n, 128))
    rng = np.random.default_rng(n)
    keys = rng.integers(0, 1 << nbits, n).astype(np.uint32)
    ok, oi = e.sort_pairs(keys, nbits)
    ref = np.argsort(keys, kind="stable")
    np.testing.assert_array_equal(oi, ref.astype(np.uint32))
    np.testing.assert_array_equal(ok, keys[ref])


# ---------------------------------------------------------------- forward
@pytest.mark.parametrize("D", [4, 16, 64, 128, 132, 200, 256])
def test_fwd_score_matches_oracle(D):
    p = Problem(300, 200, 7, D, seed=D)
    e = make_engine(p)
    f = p.pointwise(777, seed=1)
    got = e.score(f["user_input"], f["item_input"], f["categories"]).cpu().numpy()
    ref = p.oracle(OHyper()).scores(f["user_input"], f["item_input"], f["categories"])
    assert_close(got, ref, what="scores")


def test_fwd_score_general_float_category_weights():
    p = Problem(50, 40, 5, 32, seed=3)
    e = make_engine(p)
    f = p.pointwise(200, seed=2)
    cats = np.random.default_rng(0).random((200, 4, 1)).astype(np.float32) + 0.1
    got = e.score(f["user_input"], f["item_input"], cats).cpu().numpy()
    ref = p.oracle(OHyper()).scores(f["user_input"], f["item_input"], cats)
    assert_close(got, ref, what="scores")


# ---------------------------------------------------------------- train step
@pytest.mark.parametrize("learner,adam_mode", [("sgd", "dense"), ("adagrad", "dense"), ("rmsprop", "dense"),
                                               ("adam", "dense"), ("adam", "lazy_exact"), ("adam", "lazy")])
@pytest.mark.parametrize("D", [4, 64, 132, 200, 256])
def test_pointwise_steps_match_oracle(learner, adam_mode, D):
    p = Problem(500, 300, 9, D, seed=17)
    e = make_engine(p, learner=learner, adam_mode=adam_mode)
    om = p.oracle(OHyper(learner=learner, lr=0.01))
    om32 = p.oracle(OHyper(learner=learner, lr=0.01), dtype=np.float32) if learner == "adam" else None
    for s in range(5):
        if s == 1:
            f = p.contiguous(256, seed=40 + s, run=100)       # runs that cross 32-entry chunks
        elif s == 3:
            f = p.pointwise(200, seed=40 + s, users=np.full(200, 7))   # one user, one long run
        else:
            f = p.pointwise(300, seed=40 + s)
        o = om.train_step(f)
        if om32 is not None:
            om32.train_step(f)
        v = step_gpu(e, f)
        assert v[0] == pytest.approx(o["loss"], rel=1e-5), f"loss step {s}"
        assert v[1] == pytest.approx(o["norm"], rel=1e-5), f"norm step {s}"
        assert v[3] == pytest.approx(o["general"], rel=1e-5, abs=1e-5 * float(np.abs(om.G).mean())), f"general step {s}"
        assert int(v[6]) == len(np.unique(f["user_input"])) and int(v[7]) == len(np.unique(f["item_input"]))
    compare_tables(e, om, what=f"{learner}/{adam_mode}/D{D} ", om32=om32)


@pytest.mark.parametrize("learner", ["sgd", "adam"])
def test_bpr_steps_match_oracle(learner):
    p = Problem(400, 250, 9, 128, seed=23)
    e = make_engine(p, learner=learner)
    om = p.oracle(OHyper(learner=learner, lr=0.01))
    om32 = p.oracle(OHyper(learner=learner, lr=0.01), dtype=np.float32) if learner == "adam" else None
    for s in range(4):
        f = p.bpr(333, seed=70 + s, users=None if s != 2 else np.repeat(np.arange(9), 37))
        o = om.train_step_bpr(f, write_personal=(s == 0))
        if om32 is not None:
            om32.train_step_bpr(f, write_personal=(s == 0))
        v = step_gpu(e, f, personal=(s == 0), bpr=True)
        assert v[0] == pytest.approx(o["loss"], rel=1e-5)
        assert v[1] == pytest.approx(o["norm"], rel=1e-5)
        if s == 0:
            assert v[4] == pytest.approx(o["personal"], rel=1e-5, abs=1e-5 * float(np.abs(om.P).mean()))
    compare_tables(e, om, what=f"bpr/{learner} ", om32=om32)


@pytest.mark.parametrize("learner", ["sgd", "adagrad", "rmsprop", "adam"])
def test_personal_write_step_matches_oracle(learner):
    """Train_recommender.py:170-187: 16 mini-steps of 8 rows, each fetching model.personal."""
    p = Problem(60, 80, 9, 64, seed=29)
    e = make_engine(p, learner=learner)
    om = p.oracle(OHyper(learner=learner, lr=0.01))
    om32 = p.oracle(OHyper(learner=learner, lr=0.01), dtype=np.float32) if learner == "adam" else None
    f = p.contiguous(128, seed=5, run=40)
    for mini in range(16):
        sl = slice(mini * 8, mini * 8 + 8)
        fm = {k: v[sl] for k, v in f.items()}
        o = om.train_step(fm, write_personal=True)
        if om32 is not None:
            om32.train_step(fm, write_personal=True)
        v = step_gpu(e, fm, personal=True)
        assert v[0] == pytest.approx(o["loss"], rel=1e-5)
        assert v[4] == pytest.approx(o["personal"], rel=1e-5, abs=1e-5 * float(np.abs(om.P).mean()))
        assert v[3] == pytest.approx(o["general"], rel=1e-5, abs=1e-5 * float(np.abs(om.G).mean()))
    compare_tables(e, om, what=f"personal/{learner} ", om32=om32)


def test_clip_active_matches_oracle():
    p = Problem(50, 40, 5, 64, seed=31, scale=20.0)        # large tables -> global norm > 5
    e = make_engine(p, learner="sgd", lr=0.01)
    om = p.oracle(OHyper(learner="sgd", lr=0.01))
    f = p.pointwise(64, seed=3, users=np.zeros(64, np.int32))
    o = om.train_step(f)
    v = step_gpu(e, f)
    assert o["scale"] < 1.0
    assert v[2] == pytest.approx(o["scale"], rel=1e-5) and v[1] == pytest.approx(o["norm"], rel=1e-5)
    compare_tables(e, om, what="clip ")


def test_lazy_exact_adam_is_bit_identical_to_dense_sweep():
    """SURVEY hard part 1: lazy catch-up replays the skipped steps with identical
    arithmetic, so after a flush the tables equal the TF-1.x dense sweep bit for bit."""
    p = Problem(2000, 500, 9, 64, seed=37)
    ed = make_engine(p, adam_mode="dense")
    # (two-pass step on both sides: the single-pass kernel sums the dCat / loss partials in sorted-user order, which
    #  moves Category_Embedding in the last bits; its equality with the two-pass step is tests/test_gpu_single_pass.py)
    el = make_engine(p, adam_mode="lazy_exact", single_pass=False)
    for s in range(12):
        f = p.pointwise(256, seed=100 + s) if s % 3 else p.contiguous(256, seed=100 + s, run=64)
        step_gpu(ed, f); step_gpu(el, f)
    td, tl = ed.tables(), el.tables()
    for k in ("P", "R", "Cat", "G"):
        np.testing.assert_array_equal(td[k], tl[k], err_msg=k)
    for k in ("P", "R"):
        np.testing.assert_array_equal(ed.s1[k].cpu().numpy(), el.s1[k].cpu().numpy())
        np.testing.assert_array_equal(ed.s2[k].cpu().numpy(), el.s2[k].cpu().numpy())


def test_lazy_series_adam_equals_dense_sweep_to_rounding():
    """LAZY_SERIES (closed-form catch-up, O(1) per element) against the literal TF-1.x dense
    sweep over 80 steps with gaps from 1 to ~80 steps, plus a checkpoint round trip in the
    middle (fr_set_step rebuilds the coefficient table)."""
    p = Problem(4000, 600, 9, 64, seed=39)
    ed = make_engine(p, adam_mode="dense", lr=0.001)
    el = make_engine(p, adam_mode="lazy", lr=0.001)
    for s in range(80):
        f = p.pointwise(128, seed=300 + s)
        step_gpu(ed, f); step_gpu(el, f)
        if s == 40:
            sd = el.state_dict()
            el2 = make_engine(p, adam_mode="lazy", lr=0.001)
            el2.load_state_dict(sd)
            el = el2
    td, tl = ed.tables(), el.tables()
    for k in ("P", "R", "Cat", "G"):
        assert_close(tl[k], td[k], rtol=2e-6, what=f"series vs dense {k}")
    moved = np.abs(td["P"] - p.tb.P).max()
    assert moved > 1e-3          # the comparison is not vacuous: rows moved by many steps


def test_compact_feed_equals_dense_feed():
    """ids-only feed (resident dish_to_category / user-label tables) == reference dense feed."""
    p = Problem(300, 200, 9, 128, seed=41)
    ed, ec = make_engine(p), make_engine(p, resident=True)
    for s in range(3):
        f = p.pointwise(500, seed=7 + s)
        f["write_sign"] = np.where(f["labels"] > 0, 1.0, -1.0).astype(np.float32).reshape(-1, 1)
        a = step_gpu(ed, f).copy(); b = step_gpu(ec, f, compact=True).copy()
        np.testing.assert_array_equal(a[:6], b[:6])
    fb = p.bpr(400, seed=11)
    step_gpu(ed, fb, bpr=True); step_gpu(ec, fb, bpr=True, compact=True)
    td, tc = ed.tables(), ec.tables()
    for k in ("P", "R", "Cat", "G"):
        np.testing.assert_array_equal(td[k], tc[k], err_msg=k)


def test_host_buffer_entry_point_equals_device_entry_point():
    from foodrec_b200 import _lib as L
    p = Problem(300, 200, 9, 64, seed=43)
    e1, e2 = make_engine(p), make_engine(p)
    f = p.pointwise(256, seed=3)
    v1 = step_gpu(e1, f).copy()
    pin = lambda x, dt: torch.as_tensor(np.ascontiguousarray(x.astype(dt))).pin_memory()
    out = e2.train_step_host(L.FR_POINTWISE, 256, pin(f["user_input"], np.int32), pin(f["item_input"], np.int32),
                             pin(f["categories"].reshape(-1, 4), np.float32), pin(f["labels"], np.float32),
                             pin(f["write_sign"].reshape(-1), np.float32), pin(f["user_one_hot_label"], np.float32))
    torch.cuda.synchronize()
    np.testing.assert_array_equal(out.numpy()[:6], v1[:6])
    t1, t2 = e1.tables(), e2.tables()
    for k in ("P", "R", "Cat", "G"):
        np.testing.assert_array_equal(t1[k], t2[k], err_msg=k)


def test_label_overflow_is_reported():
    from foodrec_b200 import Engine, Hyper, _lib as L
    p = Problem(50, 40, 9, 16, seed=2)
    e = Engine(Hyper(), p.tb.P, p.tb.R, p.tb.Cat, p.tb.G, max_rows=256, max_label_entries=8)
    f = p.pointwise(64, seed=1)
    e.train_step(f["user_input"], f["item_input"], labels=f["labels"], categories=f["categories"],
                 write_sign=f["write_sign"], user_one_hot_label=f["user_one_hot_label"])
    with pytest.raises(L.FoodRecError, match="max_label_entries"):
        e.read_scalars()


def test_bad_batches_raise():
    from foodrec_b200 import _lib as L
    p = Problem(50, 40, 9, 16, seed=2)
    e = make_engine(p, max_rows=64)
    f = p.pointwise(100, seed=1)
    with pytest.raises(L.FoodRecError, match="max_rows"):
        step_gpu(e, f)
    f0 = {k: v[:0] for k, v in f.items()}
    with pytest.raises(L.FoodRecError, match="empty batch"):
        step_gpu(e, f0)


# ---------------------------------------------------------------- golden vectors
@pytest.mark.parametrize("learner", ["sgd", "adagrad", "rmsprop", "adam"])
@pytest.mark.parametrize("mode", ["pointwise", "bpr"])
def test_cuda_path_matches_golden(learner, mode):
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(GOLD, "make_golden.py"))
    mg = importlib.util.module_from_spec(spec); spec.loader.exec_module(mg)
    g = np.load(os.path.join(GOLD, f"train_{learner}_{mode}.npz"))
    seed = int(g["seed"])
    tb, ic, ul = mg.problem(seed)
    from foodrec_b200 import Engine, Hyper
    e = Engine(Hyper(learner=learner, lr=0.01), tb.P, tb.R, tb.Cat, tb.G, max_rows=512, max_label_entries=512 * mg.L)
    om32 = OracleModel(tb.P, tb.R, tb.Cat, tb.G, OHyper(learner=learner, lr=0.01), dtype=np.float32)
    for s, f in enumerate(mg.feeds(ic, ul, seed, bpr=(mode == "bpr"))):
        (om32.train_step_bpr if mode == "bpr" else om32.train_step)(f, write_personal=(s == 0))
        v = step_gpu(e, f, personal=(s == 0), bpr=(mode == "bpr"))
        assert v[0] == pytest.approx(float(g[f"loss{s}"]), rel=1e-5)
        assert v[1] == pytest.approx(float(g[f"norm{s}"]), rel=1e-5)
        # means of a table are sums that cancel: judged against the scale of the averaged terms
        assert v[3] == pytest.approx(float(g[f"general{s}"]), rel=1e-5, abs=1e-5 * float(np.abs(g["G"]).mean()))
        if s == 0:
            assert v[4] == pytest.approx(float(g["personal0"]), rel=1e-5, abs=1e-5 * float(np.abs(g["P"]).mean()))
    t = e.tables()
    for k in ("P", "R", "Cat", "G"):
        if learner == "adam" and k != "G":
            assert_close_adam(t[k], g[k], getattr(om32, k), what=f"golden {learner}/{mode} {k}")
        else:
            assert_close(t[k], g[k], what=f"golden {learner}/{mode} {k}")


# ---------------------------------------------------------------- evaluation
def test_sampled_eval_matches_evaluate_py_semantics():
    p = Problem(120, 400, 7, 64, seed=47)
    e = make_engine(p)
    train, tr, tn = synth.make_reference_dataset(120, 400, seed=5)
    tn["3"][60] = tr["3"][0]                # duplicate of the positive among the negatives
    tn["4"][70] = tn["4"][55]               # duplicate negative
    tn["5"] = tn["5"][:80]                  # ragged: only 30 eval negatives
    d2c, _ = synth.reference_side_maps(p.item_cats, p.user_labels)
    from foodrec_b200.evaluate import build_candidates
    users, cand, ncand, ccats = build_candidates(tr, tn, d2c)
    ids, rank, sc = e.eval_sampled_topk(users, cand, ncand, 10, cand_cats=ccats, return_scores=True)
    ids, rank, sc = ids.cpu().numpy(), rank.cpu().numpy(), sc.cpu().numpy()
    om = p.oracle(OHyper(), dtype=np.float64)
    hits, ndcgs, ranks = evaluate_oracle.evaluate_model(om, tr, tn, 10, p.item_cats)
    n_checked = 0
    for r, u in enumerate(tr):
        c = cand[r, :ncand[r]]
        ref = om.scores(np.full(len(c), int(u)), c, p.item_cats[c])
        assert_close(sc[r, :ncand[r]], ref, what=f"eval scores user {u}")
        # ids are bit-exact whenever the oracle's ranking is not decided by a sub-tolerance gap
        top = sorted(set(ref), reverse=True)[:11]
        if len(top) > 1 and np.min(-np.diff(top)) < 1e-6 * np.abs(ref).max():
            continue
        assert list(ids[r][ids[r] >= 0]) == ranks[r], f"user {u}"
        assert (rank[r] >= 0) == bool(hits[r])
        n_checked += 1
    assert n_checked > 100
    # dict semantics on exact ties / duplicates, independent of rounding:
    assert len(set(ids[3][ids[3] >= 0])) == len(ids[3][ids[3] >= 0])


def test_sampled_eval_tie_break_is_insertion_order():
    """All-equal scores (zero tables): nlargest keeps insertion order (evaluate.py:63)."""
    p = Problem(4, 100, 3, 16, seed=1)
    p.tb.P[:] = 0
    e = make_engine(p)
    cand = np.array([[9, 3, 7, 3, 1, 9, 2, 8, 6, 5, 4, 0]], np.int32)
    ids, rank = e.eval_sampled_topk(np.array([2]), cand, np.array([12]), 5, cand_cats=p.item_cats[cand])
    assert list(ids.cpu().numpy()[0]) == [9, 3, 7, 1, 2] and int(rank.cpu()[0]) == 0


@pytest.mark.parametrize("ncand", [51, 64, 100])
def test_sampled_eval_duplicates_across_slots(ncand):
    """Repeated ids anywhere in the candidate list -- inside the first 32 positions, beyond them, and straddling
    the two (the kernel detects them per 32-wide slot and across slots before it runs the dict fix-up) -- against
    evaluate.py's dict + nlargest, on integer-valued scores so that ties are exact (a = 0, one-hot recipe rows)."""
    rng = np.random.default_rng(ncand)
    U, I, D = 37, 120, 120
    p = Problem(U, I, 3, D, seed=3)
    p.tb.P[:] = 0; p.tb.P[:, 1, :I] = rng.integers(-3, 4, (U, I)).astype(np.float32)
    p.tb.R[:] = 0; p.tb.R[np.arange(I), np.arange(I)] = 1.0
    p.item_cats[:] = 0; p.item_cats[:, 0] = 1.0
    from foodrec_b200 import Engine, Hyper
    e = Engine(Hyper(learner="sgd", lr=0.01, high_level_score_coefficient=0.0), p.tb.P, p.tb.R, p.tb.Cat, p.tb.G,
               max_rows=256, max_label_entries=256 * p.L)
    cand = rng.integers(0, I, (U, ncand)).astype(np.int32)
    for u in range(U):            # plant repeats: within slot 0, within the upper slots, across them, of the positive
        k = u % 5
        if k == 0: cand[u, 20] = cand[u, 3]
        if k == 1: cand[u, ncand - 1] = cand[u, 33]
        if k == 2: cand[u, 40] = cand[u, 5]; cand[u, 45] = cand[u, 5]
        if k == 3: cand[u, ncand - 2] = cand[u, 0]
    nc = np.full(U, ncand, np.int32); nc[7] = 33; nc[8] = 32; nc[9] = 1
    ids, rank, sc = e.eval_sampled_topk(np.arange(U), cand, nc, 10, cand_cats=p.item_cats[cand], return_scores=True)
    ids, rank = ids.cpu().numpy(), rank.cpu().numpy()
    import heapq
    S = p.tb.P[:, 1, :I]
    for u in range(U):
        c = cand[u, :nc[u]].tolist()
        m = {}
        for it in c:
            m[it] = S[u, it]
        want = heapq.nlargest(10, m, key=m.get)
        got = [int(x) for x in ids[u] if x >= 0]
        assert got == want, (u, got, want)
        assert int(rank[u]) == (want.index(c[0]) if c[0] in want else -1)


# ---------------------------------------------------------------- reference driver protocol
def test_session_protocol_runs_the_reference_loop():
    """Train_recommender.py:156-205 + evaluate.py through the shim, with the reference's own
    feed types (python lists, str user ids, [4][1] category nesting)."""
    import foodrec_b200.tf_shim as tf
    from foodrec_b200 import Model, evaluate_model
    p = Problem(40, 300, 7, 32, seed=53)
    train, tr, tn = synth.make_reference_dataset(40, 300, seed=6, pos_range=(3, 12))
    d2c, u2l = synth.reference_side_maps(p.item_cats, p.user_labels)
    ui, ii, y, c, ws, ul = synth.get_train_instances(train, tn, d2c, u2l, seed=1)
    args = args_ns(p, learner="adam", lr=0.001, batch_size=128)
    om = p.oracle(OHyper(learner="adam", lr=0.001))
    om32 = p.oracle(OHyper(learner="adam", lr=0.001), dtype=np.float32)
    with tf.Session(config=tf.ConfigProto()) as sess:
        model = Model(args, p.tb.P, p.tb.R, p.tb.Cat, p.tb.G)
        sess.run(tf.global_variables_initializer())
        assert sess.run(model.epoch_step) == 0
        nb = len(ui) // 128
        for b in range(min(nb, 4)):
            start, end = b * 128, (b + 1) * 128
            if b == 0:                                    # :170-187
                for mini in range(16):
                    s0, s1 = start + mini * 8, start + (mini + 1) * 8
                    feed = {model.user_input: ui[s0:s1], model.item_input: ii[s0:s1], model.labels: y[s0:s1],
                            model.categories: c[s0:s1], model.user_one_hot_label: ul[s0:s1],
                            model.write_sign: ws[s0:s1], model.dropout_keep_prob: 0.8, model.is_training_flag: True}
                    loss, lr, personal, general, _ = sess.run(
                        [model.loss_value, model.learning_rate, model.personal, model.general, model.train_op], feed)
                    of = dict(user_input=np.asarray(ui[s0:s1]).astype(np.int32), item_input=ii[s0:s1],
                              labels=y[s0:s1], categories=c[s0:s1], write_sign=ws[s0:s1], user_one_hot_label=ul[s0:s1])
                    o = om.train_step(of, write_personal=True); om32.train_step(of, write_personal=True)
                    assert loss == pytest.approx(o["loss"], rel=1e-5) and personal == pytest.approx(o["personal"], rel=1e-5, abs=1e-5 * float(np.abs(om.P).mean()))
            else:                                         # :189-199
                feed = {model.user_input: ui[start:end], model.item_input: ii[start:end], model.labels: y[start:end],
                        model.categories: c[start:end], model.user_one_hot_label: ul[start:end],
                        model.write_sign: ws[start:end], model.dropout_keep_prob: 0.8, model.is_training_flag: True}
                loss, lr, general, _ = sess.run([model.loss_value, model.learning_rate, model.general, model.train_op], feed)
                of = dict(user_input=np.asarray(ui[start:end]).astype(np.int32), item_input=ii[start:end],
                          labels=y[start:end], categories=c[start:end], write_sign=ws[start:end],
                          user_one_hot_label=ul[start:end])
                o = om.train_step(of); om32.train_step(of)
                assert loss == pytest.approx(o["loss"], rel=1e-5) and general == pytest.approx(o["general"], rel=1e-5, abs=1e-5 * float(np.abs(om.G).mean()))
                assert lr == np.float32(0.001)
        sess.run(model.epoch_increment)
        assert sess.run(model.epoch_step) == 1
        # full-catalog top-K through the model object, fed with the reference's json map (extension)
        cid, csc = model.catalog_topk(["3", "17", "3"], 7, d2c)
        t = model.engine.tables()
        oc = OracleModel(t["P"], t["R"], t["Cat"], t["G"], OHyper(), dtype=np.float32)
        rid, rsc = evaluate_oracle.catalog_topk(oc, np.array([3, 17, 3]), p.item_cats, 7)
        assert np.array_equal(cid, rid) and np.abs(csc - rsc).max() <= 1e-12 * np.abs(rsc).max()
        hits, ndcgs = evaluate_model(sess, model, tr, tn, 10, d2c)
        oh, on, _ = evaluate_oracle.evaluate_model(om, tr, tn, 10, p.item_cats)
        assert len(hits) == len(tr) and abs(np.mean(hits) - np.mean(oh)) <= 2 / len(tr)
        assert abs(np.mean(ndcgs) - np.mean(on)) <= 2 / len(tr)
        compare_tables(model.engine, om, what="session ", om32=om32)
        # checkpoint round trip (Train_recommender.py:145-151,216-223)
        import tempfile
        d = tempfile.mkdtemp() + "/"
        saver = tf.train.Saver()
        saver.save(sess, d + "model.ckpt", global_step=0)
        assert os.path.exists(d + "checkpoint")
        before = model.engine.tables()
        model.engine.P.zero_()
        saver.restore(sess, tf.train.latest_checkpoint(d))
        np.testing.assert_array_equal(model.engine.tables()["P"], before["P"])
        assert sess.run(model.epoch_step) == 1 and model.engine.step == om.t


# ---------------------------------------------------------------- full-size properties (cfg2)
def test_cfg2_full_size_properties():
    """BASELINE cfg2 (1M users / 200k recipes / D=128) is too big for the numpy oracle;
    check size-independent properties instead: (1) lr=0 leaves P/R/Cat untouched while G
    moves by exactly the write; (2) a step followed by the same step with flipped labels and
    write signs restores G (linearity of Write_Memory); (3) only touched rows change;
    (4) the loss of an all-zero model is ln 2."""
    from foodrec_b200 import Engine, Hyper
    U, I, L, D, B = 1_000_000, 200_000, 95, 128, 65536
    g = torch.Generator(device="cuda"); g.manual_seed(1)
    P = torch.randn((U, 5, D), device="cuda", generator=g) * 0.1
    R = torch.randn((I, D), device="cuda", generator=g) * 0.1
    Cat = torch.randn((4, D), device="cuda", generator=g) * 0.1
    G = torch.randn((L, 5, D), device="cuda", generator=g) * 0.1
    ic = synth.make_item_categories(I); ul = synth.make_user_labels(U, L)
    e = Engine(Hyper(learner="sgd", lr=0.0), P, R, Cat, G, max_rows=2 * B, item_cats=ic, user_labels=ul)
    rng = np.random.default_rng(0)
    users = rng.integers(0, U, B).astype(np.int32); items = synth.zipf_items(rng, I, B)
    y = (rng.random(B) < 0.5).astype(np.float32)
    G0 = e.G.clone(); P0 = e.P.clone()
    e.train_step(users, items, labels=y); v = e.read_scalars()
    assert torch.equal(e.P, P0) and not torch.equal(e.G, G0)
    assert int(v[6]) == len(np.unique(users)) and int(v[7]) == len(np.unique(items))
    e.train_step(users, items, labels=1 - y); e.read_scalars()
    assert_close(e.G.cpu().numpy(), G0.cpu().numpy(), what="G after +/- write")
    del e, P0
    e = Engine(Hyper(learner="adam", lr=0.01), P, R, Cat, G, max_rows=2 * B, item_cats=ic, user_labels=ul)
    P0 = e.P.clone()
    e.train_step(users, items, labels=y); e.read_scalars(); e.flush()
    changed = (e.P != P0).reshape(U, -1).any(1).cpu().numpy()
    touched = np.zeros(U, bool); touched[users] = True
    assert (changed <= touched).all() and changed.sum() > 0.99 * touched.sum()
    del e, P0
    z = lambda t: torch.zeros_like(t)
    e = Engine(Hyper(learner="sgd", lr=0.1), z(P), z(R), z(Cat), z(G), max_rows=2 * B, item_cats=ic, user_labels=ul)
    e.train_step(users, items, labels=y)
    assert e.read_scalars()[0] == pytest.approx(np.log(2.0), rel=1e-6)


# ---------------------------------------------------------------- negative sampler (bit-exact)
def test_philox_kernel_matches_published_known_answers():
    from oracle import sampler_oracle as so
    p = Problem(8, 8, 3, 8)
    e = make_engine(p, max_rows=128)
    got = e.philox(np.array([list(c) + list(k) for c, k, _ in so.KAT], np.uint32))
    assert got.tolist() == [list(o) for _, _, o in so.KAT]
    e.close()


@pytest.mark.parametrize("I,n,n_neg,offset", [(200_000, 4096, 8, 0), (5, 3000, 8, 7), (2, 64, 4, 0),
                                              (200_000, 512, 8, 1 << 33), (1_000_003, 70_001, 1, 123456789)])
def test_negative_sampler_is_bit_exact(I, n, n_neg, offset):
    """Same (seed, sample index) -> same negatives on host and device, including re-draws when a draw
    hits the positive (tiny catalogs) and sample indices past 2^32."""
    from foodrec_b200 import Engine, Hyper
    from oracle import sampler_oracle as so
    tb = synth.make_tables(16, min(I, 64), 3, 8, seed=1)
    R = np.zeros((I, 8), np.float32)
    e = Engine(Hyper(learner="sgd"), tb.P, R, tb.Cat, tb.G, max_rows=128)
    pos = np.random.default_rng(I + n).integers(0, I, n).astype(np.int32)
    got = e.sample_negatives(pos, n_neg, seed=20260105, sample_offset=offset).cpu().numpy()
    want = so.sample_negatives(pos, n_neg, I, seed=20260105, sample_offset=offset)
    assert np.array_equal(got, want)
    assert (got != pos[:, None]).all()
    e.close()


def test_negative_sampler_golden_vectors():
    from foodrec_b200 import Engine, Hyper
    g = np.load(os.path.join(GOLD, "negative_sampler.npz"))
    tb = synth.make_tables(16, 64, 3, 8, seed=1)
    e = Engine(Hyper(learner="sgd"), tb.P, np.zeros((int(g["num_items"]), 8), np.float32), tb.Cat, tb.G, max_rows=128)
    got = e.sample_negatives(g["pos"], int(g["n_neg"]), int(g["seed"]), int(g["offset"])).cpu().numpy()
    assert np.array_equal(got, g["neg"])
    e.close()


def test_sampled_1_to_8_step_matches_oracle():
    """BASELINE configs[4] shape: 1:8 sampled negatives -> B*8 BPR triples; tables equal the oracle's on the
    triples the ORACLE sampler draws."""
    from oracle import sampler_oracle as so
    p = Problem(300, 500, 9, 64, seed=5)
    e = make_engine(p, learner="adagrad", lr=0.05, max_rows=2 * 8 * 64, resident=True)
    om = p.oracle(OHyper(learner="adagrad", lr=0.05))
    rng = np.random.default_rng(2)
    for s in range(2):
        users = rng.integers(0, p.U, 64).astype(np.int32); pos = rng.integers(0, p.I, 64).astype(np.int32)
        e.train_step_sampled(users, pos, 8, seed=99, sample_offset=64 * s)
        e.read_scalars()
        neg = so.sample_negatives(pos, 8, p.I, seed=99, sample_offset=64 * s)
        uu, pp, nn = np.repeat(users, 8), np.repeat(pos, 8), neg.reshape(-1)
        om.train_step_bpr(dict(user_input=uu, item_input=pp, neg_item_input=nn, categories=p.item_cats[pp],
                               neg_categories=p.item_cats[nn], user_one_hot_label=p.user_labels[uu]))
    compare_tables(e, om, "sampled 1:8 ")
    e.close()


def test_device_resident_instance_stream_equals_the_dense_feed_loop():
    """SURVEY 8f.1: instance arrays + side tables resident on the device, batches are device slices.  One epoch
    of Train_recommender.py:163-199 (first batch = 16 personal-memory steps of 8 rows) must leave exactly the
    tables the reference-format dense feed leaves."""
    from foodrec_b200 import Engine, Hyper
    from foodrec_b200.data import InstanceStream, build_instances, side_tables
    p = Problem(60, 400, 7, 32, seed=71)
    train, tr, tn = synth.make_reference_dataset(60, 400, seed=8, pos_range=(3, 12))
    d2c, u2l = synth.reference_side_maps(p.item_cats, p.user_labels)
    ui, ii, y, c, ws, ul = synth.get_train_instances(train, tn, d2c, u2l, seed=3)
    h = Hyper(learner="adam", lr=0.001)
    dense = Engine(h, p.tb.P, p.tb.R, p.tb.Cat, p.tb.G, max_rows=256, max_label_entries=256 * p.L)
    B, n = 128, len(ui)
    users = np.asarray(ui).astype(np.int32)
    for b in range(n // B):
        s0, s1 = b * B, (b + 1) * B
        spans = [(s0 + k * 8, s0 + (k + 1) * 8, True) for k in range(16)] if b == 0 else [(s0, s1, False)]
        for lo, hi, personal in spans:
            dense.train_step(users[lo:hi], ii[lo:hi], labels=y[lo:hi], categories=c[lo:hi], write_sign=ws[lo:hi],
                             user_one_hot_label=ul[lo:hi], write_personal=personal)
    ic, ulab = side_tables(d2c, u2l, p.I, p.U, p.L)
    res = Engine(h, p.tb.P, p.tb.R, p.tb.Cat, p.tb.G, max_rows=256, item_cats=ic, user_labels=ulab)
    stream = InstanceStream(res, build_instances(train, tn, seed=3))
    assert stream.n == n
    assert stream.run_epoch(B, epoch=0) == n // B - 1 + 16
    ta, tb_ = dense.tables(), res.tables()
    for k in ("P", "R", "Cat", "G"):
        np.testing.assert_array_equal(ta[k], tb_[k], err_msg=k)
    dense.close(); res.close()


def test_feed_prefetch_overlap_gives_identical_results():
    """fr_feed_prefetch stages batch k+1 on the library's copy stream while step k runs; the step that
    consumes the staged image must be indistinguishable from the unstaged host path."""
    from foodrec_b200 import _lib as L
    p = Problem(500, 800, 9, 64, seed=91)
    ea = make_engine(p, learner="adam", lr=0.01, max_rows=1024)
    eb = make_engine(p, learner="adam", lr=0.01, max_rows=1024)
    pin = lambda x, dt: torch.as_tensor(np.ascontiguousarray(np.asarray(x).astype(dt))).pin_memory()
    feeds = []
    for s in range(5):
        f = p.bpr(300, seed=200 + s)
        items = np.stack([f["item_input"], f["neg_item_input"]], 1).reshape(-1)
        cats = np.stack([f["categories"].reshape(-1, 4), f["neg_categories"].reshape(-1, 4)], 1).reshape(-1, 4)
        feeds.append((pin(f["user_input"], np.int32), pin(items, np.int32), pin(cats, np.float32),
                      pin(f["user_one_hot_label"], np.float32)))
    outs_a, outs_b = [], []
    ea.feed_prefetch(L.FR_BPR, 300, feeds[0][0], feeds[0][1], feeds[0][2], None, None, feeds[0][3])
    for s, (u, it, c, ul) in enumerate(feeds):
        if s + 1 < len(feeds):
            n = feeds[s + 1]
            ea.feed_prefetch(L.FR_BPR, 300, n[0], n[1], n[2], None, None, n[3])
        oa = ea.train_step_host(L.FR_BPR, 300, u, it, c, None, None, ul); torch.cuda.synchronize(); outs_a.append(oa.clone())
        ob = eb.train_step_host(L.FR_BPR, 300, u, it, c, None, None, ul); torch.cuda.synchronize(); outs_b.append(ob.clone())
    for oa, ob in zip(outs_a, outs_b):
        assert torch.equal(oa, ob)
    ta, tb_ = ea.tables(), eb.tables()
    for k in ("P", "R", "Cat", "G"):
        np.testing.assert_array_equal(ta[k], tb_[k], err_msg=k)
    ea.close(); eb.close()
