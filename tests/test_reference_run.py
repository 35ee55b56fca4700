"""Traces of the reference's OWN PROGRAM (``tests/golden/reference_run_*.npz``): ``Train_recommender.py``
was executed end to end in the authoring container -- its argparse, ``Dataset``, ``get_train_instances``,
the unmodified ``Model_Recommender.Model`` graph, the batch loop with the personal-write block and
``evaluate_model`` -- with only the ``tensorflow`` module substituted (``tests/golden/tf1_standin``; script
``tests/golden/make_reference_run_golden.py``).  Every ``sess.run`` was recorded: the feed the reference built,
its fetch pattern, and what came back.

CPU tests replay each trace through the oracle (``oracle/recommender_oracle.py``): this is the check that the
oracle's restatement of the graph is what the reference's code actually computes.  The GPU test replays them
through ``foodrec_b200.Model`` / ``Session.run`` -- the drop-in boundary -- with the same fetch lists."""
import glob
import os
import types

import numpy as np
import pytest

from oracle import evaluate_oracle
from oracle.recommender_oracle import Hyper as OHyper, OracleModel
from tests.util import assert_close

GOLD = os.path.join(os.path.dirname(__file__), "golden")
TRACES = sorted(os.path.basename(p)[len("reference_run_"):-4] for p in glob.glob(os.path.join(GOLD, "reference_run_*.npz")))


def load(name):
    z = np.load(os.path.join(GOLD, f"reference_run_{name}.npz"))
    return {k: z[k] for k in z.files}


def runs(t):
    """(kind, feed dict in the reference's placeholder names, recorded outputs) per sess.run."""
    for r in range(len(t["kind"])):
        s = slice(int(t["off"][r]), int(t["off"][r + 1]))
        feed = dict(user_input=t["user"][s], item_input=t["item"][s], labels=t["label"][s],
                    categories=t["cats"][s].reshape(-1, 4, 1), write_sign=t["ws"][s].reshape(-1, 1),
                    user_one_hot_label=t["onehot"][s])
        out = dict(loss=t["out_loss"][r], lr=t["out_lr"][r], personal=t["out_personal"][r], general=t["out_general"][r],
                   personal_at_run_end=t["out_personal_at_run_end"][r], logits=t["logits"][s])
        yield int(t["kind"][r]), feed, out


def test_traces_cover_the_reference_program():
    assert {"adam", "adagrad", "rmsprop", "sgd", "sgd_clipped", "adam_f64", "sgd_clipped_f64", "adagrad_f64", "rmsprop_f64",
            "adam_hyper_f64", "rmsprop_hyper_f64", "adam_defaults_f64"} <= set(TRACES)
    t = load("adam")
    k = t["kind"]
    # Train_recommender.py:169-187: epoch 0 opens with 16 mini-batches of 8 that fetch `personal`
    assert (k[:16] == 1).all() and (np.diff(t["off"])[:16] == 8).all() and (k[16:] != 1).all()
    # :163-166 drops the ragged tail; evaluate.py:35-58 issues one 51-candidate (or fewer, dict-dedup is later) run per test user
    assert (np.diff(t["off"])[k == 0] == int(t["batch_size"])).all()
    assert (k == 2).sum() == 14 * int(t["epochs"]) and (np.diff(t["off"])[k == 2] == 51).all()
    assert int(t["global_step"]) == 0 and int(t["epoch_step"]) == int(t["epochs"])     # :240 passes no global_step
    assert np.all(t["out_lr"][k != 2] == np.float32(t["lr"]))                            # => lr never decays


@pytest.mark.parametrize("name", TRACES)
def test_oracle_reproduces_the_reference_program(name):
    t = load(name)
    wide = str(t["dtype"]) == "float64"
    dt = np.float64 if wide else np.float32
    rtol = 1e-11 if wide else 1e-5
    a, b1, b2, al = (float(x) for x in t["hyper"])
    om = OracleModel(t["P0"], t["R0"], t["Cat0"], t["G0"],
                     OHyper(learner=str(t["learner"]), lr=float(t["lr"]), high_level_score_coefficient=a, beta_1=b1, beta_2=b2,
                            alpha=al), dtype=dt)
    clipped = 0
    for r, (kind, feed, out) in enumerate(runs(t)):
        if kind == 2:
            assert_close(om.scores(feed["user_input"], feed["item_input"], feed["categories"]), out["logits"], rtol,
                         what=f"{name} run {r} logits")
            continue
        o = om.train_step(feed, write_personal=kind == 1)
        clipped += o["scale"] < 1
        assert_close(o["loss"], out["loss"], rtol, what=f"{name} run {r} loss")
        assert float(o["lr"]) == float(out["lr"]) or wide
        # table means are cancelling sums: judged against the size of what is averaged (DESIGN 2)
        assert abs(float(o["general"]) - out["general"]) <= rtol * np.abs(om.G).mean(), f"{name} run {r} general"
        if kind == 1:
            # `personal` (:218) averages the ASSIGN tensor P + bias + general_bias; whether the optimizer's update of
            # the same run is in what TF reads there is a race.  The trace holds both: the fetched value (update not
            # in it) and the mean of the variable once the run was over (what the product reports).
            tol = rtol * np.abs(om.P).mean()
            assert abs(float(o["personal_assign"]) - out["personal"]) <= tol, f"{name} run {r} personal (assign tensor)"
            assert abs(float(o["personal"]) - out["personal_at_run_end"]) <= tol, f"{name} run {r} personal (run end)"
    if "clipped" in name:
        assert clipped > 10, "the trace was built so that clip_by_global_norm(5.0) bites"
    for k in ("P", "R", "Cat", "G"):
        assert_close(getattr(om, k), t[k + "1"], rtol * (1 if wide else 4), what=f"{name} final {k}")
    # the per-user lists the reference's evaluate_model returned in its last epoch
    from foodrec_b200.data import Dataset
    d = Dataset(os.path.join(GOLD, "ref_dataset", "toy"))
    hits, ndcgs, _ = evaluate_oracle.evaluate_model(om, d.testRatings, d.testNegatives, 10, t["item_cats"].astype(np.float32))
    assert [int(h) for h in hits] == t["last_hits"].tolist()
    assert [float(x) for x in ndcgs] == t["last_ndcgs"].tolist()
    assert abs(np.mean(hits) - t["printed_hr_ndcg_loss"][-1][0]) < 5e-5        # what the program printed (%.4f)


@pytest.mark.gpu
@pytest.mark.parametrize("name", TRACES)
def test_dropin_session_reproduces_the_reference_program(name):
    """The same ``sess.run`` calls, in the same order with the same fetch lists, through the drop-in
    ``Model`` / ``Session`` and the CUDA kernels; 1e-5 relative (north_star) on losses, logits and the
    tables the program ends with.  Every trace is replayed, including the ones recorded with the stand-in in
    float64 (the reference's default shapes -- 95 labels, embed_size 200, batch 128 -- and the non-default
    hyper-parameters): there the recorded values are the float64 ground truth of the graph and the CUDA path
    (float32) is judged against them directly."""
    import foodrec_b200 as fb
    from tests.util import assert_close_adam
    t = load(name)
    wide = str(t["dtype"]) == "float64"
    # Adam against a float64 trace: ill-conditioned entries (|summed gradient| ~ eps/sqrt(1-beta2)) are excused only
    # where the float32 numpy oracle, replayed alongside, is itself off by a comparable amount (tests/util.py)
    # The float32 numpy oracle is also the yardstick for the LOSS of a float64 trace: a loss of 1e-4 (scores near 9
    # after a few lr = 0.01 steps) is exp(-s), so the 1e-6 float32 rounding of s alone moves it by 1e-5 relative.
    om32 = None
    if wide:
        a_, b1_, b2_, al_ = (float(x) for x in t["hyper"])
        om32 = OracleModel(t["P0"], t["R0"], t["Cat0"], t["G0"],
                           OHyper(learner=str(t["learner"]), lr=float(t["lr"]), high_level_score_coefficient=a_, beta_1=b1_,
                                  beta_2=b2_, alpha=al_), dtype=np.float32)
    adam32 = om32 if str(t["learner"]) == "adam" else None
    B = int(np.diff(t["off"]).max())
    a, b1, b2, al = (float(x) for x in t["hyper"])
    args = types.SimpleNamespace(learner=str(t["learner"]), num_categories=4, num_users=t["P0"].shape[0],
                                 num_labels=t["G0"].shape[0], embed_size=t["P0"].shape[2], lr=float(t["lr"]),
                                 decay_steps=1000, decay_rate=1.0, high_level_score_coefficient=a,
                                 beta_1=b1, beta_2=b2, alpha=al, batch_size=B)
    model = fb.Model(args, t["P0"], t["R0"], t["Cat0"], t["G0"])
    sess = fb.Session()
    sess.run(fb.global_variables_initializer())
    for r, (kind, feed, out) in enumerate(runs(t)):
        fd = {model.user_input: [str(u) for u in feed["user_input"]],          # str digits, as Dataset.py hands them over
              model.item_input: feed["item_input"].tolist(), model.labels: feed["labels"].tolist(),
              model.categories: feed["categories"].tolist(), model.dropout_keep_prob: 0.8, model.is_training_flag: True}
        if kind == 2:
            (logits,) = sess.run([model.logits], fd)
            assert_close(logits, out["logits"], what=f"{name} run {r} logits")
            continue
        fd[model.user_one_hot_label] = feed["user_one_hot_label"].tolist()
        fd[model.write_sign] = feed["write_sign"].tolist()
        o32 = om32.train_step(feed, write_personal=kind == 1) if om32 is not None else None
        if kind == 1:
            loss, lr, personal, general, _ = sess.run([model.loss_value, model.learning_rate, model.personal, model.general,
                                                       model.train_op], fd)
            # the mean of the variable when the run has ended (see the oracle test for the race in the fetched value)
            assert abs(float(personal) - out["personal_at_run_end"]) <= 1e-5 * np.abs(t["P1"]).mean()
        else:
            loss, lr, general, _ = sess.run([model.loss_value, model.learning_rate, model.general, model.train_op], fd)
        if o32 is not None:
            assert abs(float(loss) - out["loss"]) <= max(1e-5 * abs(out["loss"]), 8 * abs(float(o32["loss"]) - out["loss"])), \
                f"{name} run {r} loss {loss} vs {out['loss']} (float32 oracle {o32['loss']})"
        else:
            assert_close(loss, out["loss"], what=f"{name} run {r} loss")
        assert float(lr) == float(np.float32(out["lr"]))
        assert abs(float(general) - out["general"]) <= 1e-5 * np.abs(t["G1"]).mean()
    assert sess.run(model.epoch_step) == 0          # the replay does not call epoch_increment
    tabs = model.engine.tables()
    for k in ("P", "R", "Cat", "G"):
        if adam32 is not None and k != "G":
            assert_close_adam(tabs[k], t[k + "1"], getattr(adam32, k), what=f"{name} final {k}")
        else:
            assert_close(tabs[k], t[k + "1"], what=f"{name} final {k}")
    # evaluate_model (evaluate.py:13) on the tables the replay ended with: the reference's own per-user lists
    from foodrec_b200.data import Dataset
    d = Dataset(os.path.join(GOLD, "ref_dataset", "toy"))
    d2c = {str(i): [[float(x)] for x in row] for i, row in enumerate(t["item_cats"])}
    hits, ndcgs = fb.evaluate_model(sess, model, d.testRatings, d.testNegatives, 10, d2c)
    assert [int(h) for h in hits] == t["last_hits"].tolist()
    assert [float(x) for x in ndcgs] == t["last_ndcgs"].tolist()
