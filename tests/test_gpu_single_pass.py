"""The single-pass training step (fr_set_shadow; user_fused_kernel in csrc/train_seg.cu): forward + segment reduce +
Adam in one walk over the user-sorted rows, speculating that tf.clip_by_global_norm (Model_Recommender.py:237) is
inactive, on a double-buffered Personal_Memory.  It must give the results of the two-pass step -- whether the
speculation holds or not -- and those of the oracle; readers of the tables must never see a stale row."""
import numpy as np
import pytest
import torch

from oracle.recommender_oracle import Hyper as OHyper
from tests.util import Problem, assert_close, assert_close_adam

pytestmark = pytest.mark.gpu


def engine(p, single_pass, adam_mode="lazy", lr=0.01, max_rows=4096, **hk):
    from foodrec_b200 import Engine, Hyper
    e = Engine(Hyper(learner="adam", lr=lr, **hk), p.tb.P, p.tb.R, p.tb.Cat, p.tb.G, max_rows=max_rows, adam_mode=adam_mode,
               max_label_entries=max_rows * p.L, single_pass=single_pass)
    assert e.single_pass == single_pass
    return e


def step(e, f, bpr, personal=False):
    kw = dict(neg_items=f["neg_item_input"], neg_categories=f["neg_categories"]) if bpr else {}
    e.train_step(f["user_input"], f["item_input"], labels=None if bpr else f["labels"], categories=f["categories"],
                 write_sign=None if bpr else f["write_sign"], user_one_hot_label=f["user_one_hot_label"],
                 write_personal=personal, **kw)
    return e.read_scalars().copy()


def feeds(p, bpr, n, seed, B=700):
    out = []
    for s in range(n):
        users = None
        if s % 3 == 1:
            users = np.repeat(np.arange(10) * 7 % p.U, (B + 9) // 10)[:B]      # long runs: cross many 32-row chunks
        out.append(p.bpr(B, seed=seed + s, users=users) if bpr else p.pointwise(B, seed=seed + s, users=users))
    return out


@pytest.mark.parametrize("bpr", [False, True])
@pytest.mark.parametrize("D,adam_mode", [(4, "lazy"), (64, "lazy"), (128, "lazy"), (128, "lazy_exact"), (132, "lazy"),
                                       (200, "lazy"), (256, "lazy_exact")])
def test_single_pass_equals_two_pass_and_oracle(bpr, D, adam_mode):
    p = Problem(900, 500, 9, D, seed=3 + D)
    a, b = engine(p, True, adam_mode), engine(p, False, adam_mode)
    om = p.oracle(OHyper(learner="adam", lr=0.01))
    om32 = p.oracle(OHyper(learner="adam", lr=0.01), dtype=np.float32)
    for s, f in enumerate(feeds(p, bpr, 6, seed=40)):
        va, vb = step(a, f, bpr), step(b, f, bpr)
        o = om.train_step_bpr(f) if bpr else om.train_step(f)
        (om32.train_step_bpr if bpr else om32.train_step)(f)
        assert va[2] == 1.0 and vb[2] == 1.0                                   # clip inactive: the speculation holds
        for k in (0, 1, 3):
            assert va[k] == pytest.approx(vb[k], rel=2e-6), (s, k)
        assert va[0] == pytest.approx(o["loss"], rel=1e-5) and va[1] == pytest.approx(o["norm"], rel=1e-5)
        assert va[6] == vb[6] and va[7] == vb[7]
        if s == 0:      # same arithmetic, same summation order per row: the first step's tables agree bit for bit
            ta, tb = a.tables(), b.tables()                                    # (flushes: a's rows come back from the shadow copy)
            np.testing.assert_array_equal(ta["P"], tb["P"]); np.testing.assert_array_equal(ta["R"], tb["R"])
    ta, tb = a.tables(), b.tables()
    # (later steps: the dCat / loss partials are summed in sorted-user order instead of batch order, so Cat -- and through
    #  it everything else -- differs in the last bits, which Adam's quotient amplifies (tests/util.py:assert_close_adam):
    #  each side is held to the oracle's 1e-5 rule below; against each other a few of ~1e6 entries reach 1.2e-5)
    for k in ("P", "R", "Cat", "G"):
        assert_close(ta[k], tb[k], rtol=5e-5, what=f"single vs two pass {k}")
        if k == "G":
            assert_close(ta[k], om.G, what="oracle G")
        else:
            assert_close_adam(ta[k], getattr(om, k), getattr(om32, k), what=f"oracle {k}")
    a.close(); b.close()


@pytest.mark.parametrize("bpr", [False, True])
def test_active_clip_falls_back_to_the_true_scale(bpr):
    """Tables 60x larger: the global norm exceeds the clip on some steps and not on others (clip_norm set to the
    median norm of the run).  Where it does, nothing speculative may survive: the step must equal the two-pass step."""
    p = Problem(600, 400, 9, 128, seed=11, scale=6.0)
    fs = feeds(p, bpr, 8, seed=90, B=500)
    probe = engine(p, False)
    norms = [step(probe, f, bpr)[1] for f in fs]
    probe.close()
    clip = float(np.median(norms))
    a, b = engine(p, True, clip_norm=clip), engine(p, False, clip_norm=clip)
    om = p.oracle(OHyper(learner="adam", lr=0.01, clip_norm=clip))
    om32 = p.oracle(OHyper(learner="adam", lr=0.01, clip_norm=clip), dtype=np.float32)
    clipped = 0
    for s, f in enumerate(fs):
        va, vb = step(a, f, bpr), step(b, f, bpr)
        o = om.train_step_bpr(f) if bpr else om.train_step(f)
        (om32.train_step_bpr if bpr else om32.train_step)(f)
        clipped += va[2] != 1.0
        assert va[2] == pytest.approx(vb[2], rel=2e-6) and va[2] == pytest.approx(float(o["scale"]), rel=1e-5)
    assert 2 <= clipped <= 6, clipped
    ta, tb = a.tables(), b.tables()
    for k in ("P", "R", "Cat", "G"):
        assert_close(ta[k], tb[k], rtol=5e-5, what=f"single vs two pass {k}")
        if k != "G":
            assert_close_adam(ta[k], getattr(om, k), getattr(om32, k), what=f"oracle {k}")
    a.close(); b.close()


def test_readers_and_personal_steps_see_current_rows():
    """Between single-pass steps some rows live in the shadow copy.  Scoring, sampled evaluation, the catalog query, a
    personal-write step (two-pass path) and a checkpoint must all see the current rows."""
    from foodrec_b200 import Engine, Hyper
    p = Problem(500, 300, 9, 64, seed=21)
    mk = lambda sp: Engine(Hyper(learner="adam", lr=0.01), p.tb.P, p.tb.R, p.tb.Cat, p.tb.G, max_rows=2048,
                           max_label_entries=2048 * p.L, item_cats=p.item_cats, user_labels=p.user_labels, single_pass=sp)
    a, b = mk(True), mk(False)
    fs = feeds(p, False, 7, seed=300, B=400)
    q = p.pointwise(300, seed=5)
    rng = np.random.default_rng(2)
    cand = rng.integers(0, p.I, (64, 51)).astype(np.int32)
    for s, f in enumerate(fs):
        for e in (a, b):
            step(e, f, False, personal=(s == 3))                # a personal-write step in the middle
        if s in (1, 4):
            sa = a.score(q["user_input"], q["item_input"]).cpu().numpy()
            sb = b.score(q["user_input"], q["item_input"]).cpu().numpy()
            assert_close(sa, sb, rtol=5e-5, what="scores")
            ia, _ = a.eval_sampled_topk(np.arange(64, dtype=np.int32), cand, np.full(64, 51, np.int32), 10)
            ib, _ = b.eval_sampled_topk(np.arange(64, dtype=np.int32), cand, np.full(64, 51, np.int32), 10)
            assert torch.equal(ia, ib)
            ca, _ = a.catalog_topk(n_users=100, K=20); cb, _ = b.catalog_topk(n_users=100, K=20)
            assert torch.equal(ca, cb)
    # checkpoint -> fresh single-pass engine -> continue == uninterrupted
    sd = a.state_dict()
    c = mk(True)
    c.load_state_dict(sd)
    g = p.pointwise(400, seed=999)
    for e in (a, b, c):
        step(e, g, False)
    ta, tb, tc = a.tables(), b.tables(), c.tables()
    # (a test of WHICH rows every reader sees, not of precision: eight lr = 0.01 Adam steps apart, the two step
    #  implementations agree to ~1e-5 on all but a few ill-conditioned entries -- see assert_close_adam; a stale row
    #  would be off by the size of an update, 1e-2)
    for k in ("P", "R", "Cat", "G"):
        assert_close(ta[k], tb[k], rtol=2e-4, what=k)
        assert_close(tc[k], ta[k], rtol=2e-4, what="resumed " + k)
    a.close(); b.close(); c.close()


def test_single_pass_is_deterministic_and_switchable():
    p = Problem(700, 400, 9, 128, seed=8)
    fs = feeds(p, True, 4, seed=70)
    outs = []
    for _ in range(2):
        e = engine(p, True)
        for f in fs:
            step(e, f, True)
        outs.append(e.tables())
        e.close()
    for k in outs[0]:
        np.testing.assert_array_equal(outs[0][k], outs[1][k], err_msg=k)
