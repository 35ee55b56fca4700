"""GPU parity at the REAL configurations (BASELINE.json configs[0] and configs[1]), numeric, against the oracle.

* cfg1, exact shape: 10k users / 5k recipes / 95 labels / D=64, B=128, the reference's user-contiguous instance
  stream (``get_train_instances``, Train_recommender.py:74-96) driven the way its batch loop drives it
  (:163-199: the first batch of epoch 0 is 16 personal-write mini-steps of 8 rows), all four optimizers.
* cfg2, full size: 1M users / 200k recipes / D=128, BPR B=262,144 (the bench's step).  The oracle cannot hold
  1M x 5 x 128 float64 rows plus the TF-1.x dense Adam slots, and does not need to: a step only reads and writes
  the rows its batch touches, and TF's dense Adam leaves a never-touched row (m = v = 0) where it is.  The batches'
  unique users / recipes are therefore remapped to a COMPACT id space, the oracle runs on the gathered rows
  (Adam: its literal every-row sweep over that compact table = TF's behaviour for those rows), and the touched rows
  of the full GPU tables are compared with it; every untouched row must still hold its initial bits.
"""
import numpy as np
import pytest
import torch

from oracle import synth
from oracle.recommender_oracle import Hyper as OHyper, OracleModel
from tests.test_adam_strict_regime import regime_guard, report
from tests.util import assert_close, assert_close_adam

pytestmark = pytest.mark.gpu


# --------------------------------------------------------------------------------------------- cfg1
@pytest.mark.parametrize("learner,lr", [("adam", 0.001), ("adagrad", 0.05), ("rmsprop", 0.001), ("sgd", 0.5)])
def test_cfg1_exact_shape_reference_stream(learner, lr):
    from foodrec_b200 import Engine, Hyper
    U, I, L, D, B = 10_000, 5_000, 95, 64, 128
    tb = synth.make_tables(U, I, L, D, seed=synth.BASE_SEED + 1)
    ic = synth.make_item_categories(I)
    ul = synth.make_user_labels(U, L)
    train, _, tneg = synth.make_reference_dataset(400, I, seed=11)          # the stream is user-contiguous: the first
    d2c, u2l = synth.reference_side_maps(ic, ul)                            # 400 users fill far more than 40 batches
    u_idx, i_idx, labels, cats, sign, ulab = synth.get_train_instances(train, tneg, d2c, u2l, seed=3)
    users = np.asarray(u_idx).astype(np.int64) * 25 + 3                     # spread them over the 10k-row table
    onehot = ul[users]
    items = np.asarray(i_idx, np.int64)
    labels = np.asarray(labels, np.float32)
    cats = np.asarray(cats, np.float32).reshape(-1, 4, 1)
    sign = np.asarray(sign, np.float32).reshape(-1, 1)
    assert len(np.unique(users[:B])) <= 3                                   # 1-2 users per 128-row batch, as in the reference

    e = Engine(Hyper(learner=learner, lr=lr), tb.P, tb.R, tb.Cat, tb.G, max_rows=B, max_label_entries=B * L)
    om = OracleModel(tb.P, tb.R, tb.Cat, tb.G, OHyper(learner=learner, lr=lr), dtype=np.float64)
    om32 = OracleModel(tb.P, tb.R, tb.Cat, tb.G, OHyper(learner=learner, lr=lr), dtype=np.float32) if learner == "adam" else None

    def feed(sl):
        return dict(user_input=users[sl], item_input=items[sl], labels=labels[sl], categories=cats[sl],
                    write_sign=sign[sl], user_one_hot_label=onehot[sl])

    def one(sl, personal):
        f = feed(sl)
        o = om.train_step(f, write_personal=personal)
        if om32 is not None:
            om32.train_step(f, write_personal=personal)
        e.train_step(f["user_input"], f["item_input"], labels=f["labels"], categories=f["categories"],
                     write_sign=f["write_sign"], user_one_hot_label=f["user_one_hot_label"], write_personal=personal)
        v = e.read_scalars()
        assert v[0] == pytest.approx(o["loss"], rel=1e-5)
        assert v[1] == pytest.approx(o["norm"], rel=1e-5)
        assert abs(v[3] - o["general"]) <= 1e-5 * np.abs(om.G).mean()
        if personal:
            assert abs(v[4] - o["personal"]) <= 1e-5 * np.abs(om.P).mean()

    n_batches = 40
    for bi in range(n_batches):
        if bi == 0:                                                          # Train_recommender.py:169-187
            for k in range(16):
                one(slice(8 * k, 8 * k + 8), True)
        else:
            one(slice(bi * B, (bi + 1) * B), False)
    t = e.tables()
    for k in ("P", "R", "Cat", "G"):
        if om32 is not None and k != "G":
            assert_close_adam(t[k], getattr(om, k), getattr(om32, k), what=f"cfg1 {learner} {k}")
        else:
            assert_close(t[k], getattr(om, k), what=f"cfg1 {learner} {k}")
    e.close()


# --------------------------------------------------------------------------------------------- cfg2
CFG2 = dict(U=1_000_000, I=200_000, L=95, D=128)


def _cfg2_problem(dev, seed):
    U, I, L, D = (CFG2[k] for k in "UILD")
    g = torch.Generator(device=dev); g.manual_seed(seed)
    P = torch.randn((U, 5, D), device=dev, generator=g) * 0.1
    R = torch.randn((I, D), device=dev, generator=g) * 0.1
    Cat = torch.randn((4, D), device=dev, generator=g) * 0.1
    G = torch.randn((L, 5, D), device=dev, generator=g) * 0.1
    return P, R, Cat, G, synth.make_item_categories(I), synth.make_user_label_csr(U, L)


def _bpr_batches(B, steps, seed):
    U, I = CFG2["U"], CFG2["I"]
    out = []
    for k in range(steps):
        rng = np.random.default_rng(seed + k)
        users = rng.integers(0, U, B).astype(np.int32)
        pos = synth.zipf_items(rng, I, B)
        neg = rng.integers(0, I, B).astype(np.int32)
        neg[neg == pos] = (neg[neg == pos] + 1) % I
        out.append((users, pos, neg))
    return out


def _run_cfg2(configs, B, steps, seed, adam_eps=1e-8, strict=False):
    """configs: list of (learner, adam_mode, lr) that share ONE oracle run (same learner, same lr).  strict (Adam): every
    touched entry is held to the plain 1e-5 rule, after the regime guard of tests/test_adam_strict_regime.py has checked
    that adam_eps keeps the quotient well conditioned for these gradients."""
    from foodrec_b200 import Engine, Hyper, _lib as L
    dev = torch.device("cuda:0")
    learner, lr = configs[0][0], configs[0][2]
    assert all(c[0] == learner and c[2] == lr for c in configs)
    P, R, Cat, G, ic, lab = _cfg2_problem(dev, seed)
    bs = _bpr_batches(B, steps, 1000 + seed)
    uu = np.unique(np.concatenate([b[0] for b in bs]))
    ui = np.unique(np.concatenate([np.concatenate([b[1], b[2]]) for b in bs]))
    tu, ti = torch.as_tensor(uu).to(dev).long(), torch.as_tensor(ui).to(dev).long()
    P0c, R0c = P[tu].cpu().numpy(), R[ti].cpu().numpy()
    Cat0, G0 = Cat.cpu().numpy(), G.cpu().numpy()
    # checksums of the rows NO batch touches (they must keep their initial bits)
    mu = torch.ones(CFG2["U"], dtype=torch.bool, device=dev); mu[tu] = False
    mi = torch.ones(CFG2["I"], dtype=torch.bool, device=dev); mi[ti] = False
    su0 = P.view(torch.int32)[mu].to(torch.int64).sum().item()
    si0 = R.view(torch.int32)[mi].to(torch.int64).sum().item()

    om = OracleModel(P0c, R0c, Cat0, G0, OHyper(learner=learner, lr=lr, adam_eps=adam_eps), dtype=np.float64)
    om32 = OracleModel(P0c, R0c, Cat0, G0, OHyper(learner=learner, lr=lr, adam_eps=adam_eps),
                       dtype=np.float32) if learner == "adam" else None
    engines = [Engine(Hyper(learner=learner, lr=lr, adam_eps=adam_eps), P.clone(), R.clone(), Cat.clone(), G.clone(),
                      device=dev, max_rows=2 * B, adam_mode=mode, item_cats=ic, user_label_csr=lab, adopt=True) for _, mode, _ in configs]
    del P, R
    for users, pos, neg in bs:
        f = dict(user_input=np.searchsorted(uu, users), item_input=np.searchsorted(ui, pos),
                 neg_item_input=np.searchsorted(ui, neg), categories=ic[pos], neg_categories=ic[neg],
                 user_one_hot_label=synth.csr_rows_dense(lab[0], lab[1], users, CFG2["L"]))
        o = om.train_step_bpr(f)
        if om32 is not None:
            om32.train_step_bpr(f)
        items = torch.as_tensor(np.stack([pos, neg], 1).reshape(-1).copy()).to(dev)
        du = torch.as_tensor(users).to(dev)
        for e in engines:                           # the compact (ids-only) feed: side tables resident, as in the bench
            e._step_dev(L.FR_BPR, B, du, items, None, None, None, None)
            v = e.read_scalars()
            assert v[0] == pytest.approx(o["loss"], rel=1e-5)
            assert v[1] == pytest.approx(o["norm"], rel=1e-5)
            assert v[2] == 1.0 and o["scale"] == 1.0                 # (the clip is inactive at this batch size)
            assert int(v[6]) == len(np.unique(users)) and int(v[7]) == len(np.unique(np.concatenate([pos, neg])))
    if strict:
        regime_guard(om, om32, f"cfg2 B={B} adam_eps={adam_eps:g}")
    for (lrn, mode, _), e in zip(configs, engines):
        e.flush()
        got = {"P": e.P[tu].cpu().numpy(), "R": e.R[ti].cpu().numpy(), "Cat": e.Cat.cpu().numpy(), "G": e.G.cpu().numpy()}
        for k in ("P", "R", "Cat", "G"):
            what = f"cfg2 B={B} {lrn}/{mode} {k}"
            if om32 is not None and k != "G" and not strict:
                assert_close_adam(got[k], getattr(om, k), getattr(om32, k), what=what)
            else:
                assert_close(got[k], getattr(om, k), what=what)
        if strict:
            report(got, om, f"cfg2 B={B} {lrn}/{mode} adam_eps={adam_eps:g}")
        assert e.P.view(torch.int32)[mu].to(torch.int64).sum().item() == su0, "an untouched Personal_Memory row changed"
        assert e.R.view(torch.int32)[mi].to(torch.int64).sum().item() == si0, "an untouched Recipe_Embedding row changed"
        e.close()


def test_cfg2_full_size_numeric_parity_adam_bench_batch():
    """The bench's own step: 1M users x 200k recipes, BPR B = 262,144, two steps (the second one catches up rows the
    first one touched), TF-1.x Adam in both lazy modes against ONE float64 oracle run on the compacted tables."""
    _run_cfg2([("adam", "lazy_exact", 0.001), ("adam", "lazy", 0.001)], B=262_144, steps=2, seed=5)


@pytest.mark.parametrize("learner,lr", [("adagrad", 0.05), ("rmsprop", 0.001), ("sgd", 0.5)])
def test_cfg2_full_size_numeric_parity_sparse_optimizers(learner, lr):
    _run_cfg2([(learner, "dense", lr)], B=65_536, steps=2, seed=6)
