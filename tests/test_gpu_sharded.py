"""GPU parity of the row-sharded step: W ranks emulated in one process on one GPU
(LocalRunner: same kernels, same five phases, collectives as tensor shuffles) must produce
the tables the unsharded engine produces on the same global batches (SURVEY 4, tier iv).
Differences are summation order only: recipe gradients are pre-reduced per rank and loss /
norm partials per rank."""
import numpy as np
import pytest
import torch

from foodrec_b200 import sharded
from oracle.recommender_oracle import Hyper as OHyper
from tests.util import Problem, assert_close

pytestmark = pytest.mark.gpu


def build(p, W, learner, adam_mode, max_rows=2048, cap=None, single_pass=None):
    """single_pass None: the engines' default (on for lazy Adam: the N-rank step then runs the single-pass kernel
    before the all-reduce and commits / redoes the update after it); False: the two-pass phases."""
    from foodrec_b200 import Engine, Hyper
    h = Hyper(learner=learner, lr=0.01)
    single = Engine(h, p.tb.P, p.tb.R, p.tb.Cat, p.tb.G, max_rows=max_rows, adam_mode=adam_mode,
                    max_label_entries=max_rows * p.L, single_pass=False if single_pass is False else None)
    rows, cols = np.nonzero(p.user_labels)
    cnt = np.bincount(rows, minlength=p.U)
    off = np.zeros(p.U + 1, np.int32); off[1:] = np.cumsum(cnt)
    engs = []
    for r in range(W):
        engs.append(sharded.ShardedEngine(
            h, sharded.shard_rows(p.tb.P, r, W), sharded.shard_rows(p.tb.R, r, W), p.tb.Cat, p.tb.G, r, W,
            max_rows=max_rows, cap=cap, adam_mode=adam_mode, item_cats_global=p.item_cats,
            user_label_csr_local=sharded.shard_label_csr(off, cols.astype(np.int32), r, W, p.U),
            max_label_entries=max_rows * p.L, single_pass=single_pass))
    return single, engs


def gather(engs, p):
    W = len(engs)
    for g in engs:
        g.e.flush()
    t = {"P": sharded.unshard_rows([g.e.P.cpu().numpy() for g in engs], p.U),
         "R": sharded.unshard_rows([g.e.R.cpu().numpy() for g in engs], p.I),
         "Cat": engs[0].e.Cat.cpu().numpy(), "G": engs[0].e.G.cpu().numpy()}
    for g in engs[1:]:        # replicated tables must be identical on every rank
        np.testing.assert_array_equal(g.e.Cat.cpu().numpy(), t["Cat"])
        np.testing.assert_array_equal(g.e.G.cpu().numpy(), t["G"])
    return t


@pytest.mark.parametrize("W", [2, 4])
@pytest.mark.parametrize("learner,adam_mode,bpr,single_pass", [
    ("sgd", "dense", False, None), ("adagrad", "dense", True, None), ("adam", "dense", False, None),
    ("adam", "lazy_exact", True, None), ("adam", "lazy", True, None), ("adam", "lazy", False, None),
    ("adam", "lazy", True, False), ("adam", "lazy_exact", False, False)])
def test_sharded_equals_unsharded(W, learner, adam_mode, bpr, single_pass):
    p = Problem(403, 257, 9, 64, seed=61)            # sizes not divisible by W: padded shards
    # W = 2 adds a step whose rows are ~90 % one recipe: each rank's recipe-gradient pre-reduction then holds a run of
    # more than 16 chunks of 32 rows, which seg_combine_long_kernel sums (ItemGradPol, peer or local stores)
    hot = W == 2
    single, engs = build(p, W, learner, adam_mode, max_rows=4096 if hot else 2048, single_pass=single_pass)
    if learner == "adam" and adam_mode != "dense":
        assert all(g.e.single_pass == (single_pass is None) for g in engs)
    run = sharded.LocalRunner(engs)
    for s in range(6 if hot else 5):
        B = 1400 if s == 5 else 300
        users = None
        if s == 2:
            users = np.repeat(np.arange(12), 25)      # duplicate-heavy, runs cross chunks
        f = p.bpr(B, seed=80 + s, users=users) if bpr else p.pointwise(B, seed=80 + s, users=users)
        if s == 5:
            rng = np.random.default_rng(s)
            it = np.where(rng.random(B) < 0.9, 5, f["item_input"]).astype(np.int32)
            f["item_input"], f["categories"] = it, p.item_cats[it].reshape(B, 4, 1).copy()
            if bpr:
                f["neg_item_input"] = np.where(f["neg_item_input"] == it, (it + 1) % p.I, f["neg_item_input"]).astype(np.int32)
                f["neg_categories"] = p.item_cats[f["neg_item_input"]].reshape(B, 4, 1).copy()
        personal = (s == 0)
        # unsharded reference: compact feed so both sides use the same side tables
        kw = dict(neg_items=f["neg_item_input"], neg_categories=f["neg_categories"]) if bpr else {}
        single.train_step(f["user_input"], f["item_input"], labels=None if bpr else f["labels"],
                          categories=f["categories"], user_one_hot_label=f["user_one_hot_label"],
                          write_sign=None, write_personal=personal, **kw)
        v1 = single.read_scalars().copy()
        idx = sharded.route_batch(f["user_input"], W)
        for r, g in enumerate(engs):
            ix = idx[r]
            assert len(ix) > 0
            g.set_batch(f["user_input"][ix] // W, f["item_input"][ix],
                        labels=None if bpr else f["labels"][ix],
                        neg_items=f["neg_item_input"][ix] if bpr else None, global_batch=B)
        outs = run.step(write_personal=personal)
        v = outs[0].cpu().numpy()
        assert v[9] == 0, "capacity/label overflow flag"
        assert v[0] == pytest.approx(v1[0], rel=1e-5) and v[1] == pytest.approx(v1[1], rel=1e-5)   # global loss / norm
        assert v[2] == pytest.approx(v1[2], rel=1e-6)
    ts, tr = gather(engs, p), single.tables()
    rt = 1e-5 if learner != "adam" else 1e-4          # Adam: conditioning (tests/util.py), summation order differs
    for k in ("P", "R", "Cat", "G"):
        assert_close(ts[k], tr[k], rtol=rt, what=f"W={W} {learner}/{adam_mode} {k}")


@pytest.mark.parametrize("learner,adam_mode", [("adam", "lazy"), ("rmsprop", "dense"), ("sgd", "dense")])
def test_rank_without_rows_is_a_first_class_case(learner, adam_mode):
    """The reference's instance stream is user-contiguous and never shuffled (Train_recommender.py:74-96): a
    128-row batch holds one or two users, so with samples routed to the user owner most ranks own NO row of a
    step.  Such a rank must still walk the five phases (serve its peers, take the all-reduced Cat / G update,
    apply the gradient rows it receives); results equal the unsharded engine."""
    W = 4
    p = Problem(203, 157, 9, 64, seed=71)
    single, engs = build(p, W, learner, adam_mode)
    run = sharded.LocalRunner(engs)
    for s in range(4):
        B = 128
        base = 4 * (3 + s) + (s % W)                     # one or two users per batch, like the reference stream
        users = np.where(np.arange(B) < 100, base, base + W * (s % 2)).astype(np.int32)
        f = p.pointwise(B, seed=700 + s, users=users)
        single.train_step(f["user_input"], f["item_input"], labels=f["labels"], categories=f["categories"],
                          user_one_hot_label=f["user_one_hot_label"], write_personal=(s == 0))
        v1 = single.read_scalars().copy()
        idx = sharded.route_batch(f["user_input"], W)
        assert sum(len(ix) == 0 for ix in idx) >= W - 2
        for r, g in enumerate(engs):
            ix = idx[r]
            g.set_batch(f["user_input"][ix] // W, f["item_input"][ix], labels=f["labels"][ix], global_batch=B)
        outs = run.step(write_personal=(s == 0))
        for o in outs:
            v = o.cpu().numpy()
            assert v[9] == 0
            assert v[0] == pytest.approx(v1[0], rel=1e-5) and v[1] == pytest.approx(v1[1], rel=1e-5)
    ts, tr = gather(engs, p), single.tables()
    for k in ("P", "R", "Cat", "G"):
        assert_close(ts[k], tr[k], rtol=1e-5 if learner != "adam" else 1e-4, what=f"{learner} {k}")


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_nccl_sharded_equals_unsharded():
    """The same comparison across real processes: torchrun x2, NCCL all-to-all / all-reduce."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29641", os.path.join(root, "tests", "dist_check.py")],
                         capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0 and out.stdout.count("DIST_CHECK_OK_") == 2, out.stdout[-1500:] + out.stderr[-3000:]


@pytest.mark.parametrize("bpr", [True, False])
def test_unrouted_batches_are_routed_to_their_owners(bpr):
    """Samples arrive on an arbitrary rank (global user ids).  fr_shard_route / one all-to-all / fr_shard_unroute must
    deliver every group to its user's owner: the step then equals the unsharded engine on the concatenated batch."""
    from foodrec_b200 import _lib as L
    W = 4
    p = Problem(403, 257, 9, 64, seed=63)
    single, engs = build(p, W, "adam", "lazy")
    run = sharded.LocalRunner(engs)
    for s in range(3):
        B = 4 * 90
        f = p.bpr(B, seed=180 + s) if bpr else p.pointwise(B, seed=180 + s)
        kw = dict(neg_items=f["neg_item_input"], neg_categories=f["neg_categories"]) if bpr else {}
        # the unsharded engine sees the groups in the order they END UP in: by owner rank, then source rank, then position
        parts = np.array_split(np.arange(B), W)                       # what arrived where
        order = np.concatenate([[i for src in range(W) for i in parts[src] if f["user_input"][i] % W == r] for r in range(W)]).astype(int)
        fo = {k: v[order] for k, v in f.items()}
        kwo = dict(neg_items=fo["neg_item_input"], neg_categories=fo["neg_categories"]) if bpr else {}
        single.train_step(fo["user_input"], fo["item_input"], labels=None if bpr else fo["labels"], categories=fo["categories"],
                          user_one_hot_label=fo["user_one_hot_label"], **kwo)
        v1 = single.read_scalars().copy()
        batches = []
        for r in range(W):
            ix = parts[r]
            items = np.stack([f["item_input"][ix], f["neg_item_input"][ix]], 1).reshape(-1) if bpr else f["item_input"][ix]
            batches.append((f["user_input"][ix], items, None if bpr else f["labels"][ix]))
        ns = run.set_batches_unrouted(L.FR_BPR if bpr else L.FR_POINTWISE, batches, global_batch=B)
        assert ns == [int((f["user_input"] % W == r).sum()) for r in range(W)]
        outs = run.step()
        v = outs[0].cpu().numpy()
        assert v[9] == 0 and v[0] == pytest.approx(v1[0], rel=1e-5) and v[1] == pytest.approx(v1[1], rel=1e-5)
    ts, tr = gather(engs, p), single.tables()
    for k in ("P", "R", "Cat", "G"):
        assert_close(ts[k], tr[k], rtol=1e-4, what=k)
    # capacity: a block too small for what one destination receives is reported, not truncated silently
    with pytest.raises(L.FoodRecError, match="routing"):
        run.set_batches_unrouted(L.FR_BPR if bpr else L.FR_POINTWISE, batches, global_batch=B, rcap=8)


@pytest.mark.parametrize("single_pass", [None, False])
def test_plan_one_step_ahead_equals_sequential(single_pass):
    """fr_shard_plan of step k+1 issued between forward and update of step k (what DistRunner's side stream does): the
    library's two plan slots keep the steps apart -- bit-identical to planning every step in sequence, including a
    personal-write step and a step in which one rank has no rows."""
    W = 4
    p = Problem(403, 257, 9, 64, seed=64)
    _, a = build(p, W, "adam", "lazy", single_pass=single_pass)
    _, b = build(p, W, "adam", "lazy", single_pass=single_pass)
    ra, rb = sharded.LocalRunner(a), sharded.LocalRunner(b)
    feeds = [p.bpr(300, seed=600 + s, users=None if s != 3 else np.repeat(np.arange(0, 48, 4), 25)) for s in range(6)]

    def setter(engs, s):
        def f():
            fd = feeds[s]
            idx = sharded.route_batch(fd["user_input"], W)
            for r, g in enumerate(engs):
                ix = idx[r]
                g.set_batch(fd["user_input"][ix] // W, fd["item_input"][ix], neg_items=fd["neg_item_input"][ix], global_batch=300)
        return f
    for s in range(6):
        setter(a, s)(); oa = ra.step(write_personal=(s == 1))
    setter(b, 0)()
    for s in range(6):
        ob = rb.step(write_personal=(s == 1), plan_ahead=setter(b, s + 1) if s < 5 else None)
    assert all(torch.equal(x, y) for x, y in zip(oa, ob))
    ta, tb_ = gather(a, p), gather(b, p)
    for k in ("P", "R", "Cat", "G"):
        np.testing.assert_array_equal(ta[k], tb_[k], err_msg=k)
    with pytest.raises(Exception, match="plan slots"):
        setter(b, 0)(); b[0].plan(); setter(b, 1)(); b[0].plan(); setter(b, 2)(); b[0].plan()


def test_capacity_overflow_is_reported():
    p = Problem(64, 200, 5, 16, seed=3)
    single, engs = build(p, 2, "sgd", "dense", max_rows=512, cap=4)     # far too small
    run = sharded.LocalRunner(engs)
    f = p.pointwise(200, seed=1)
    idx = sharded.route_batch(f["user_input"], 2)
    for r, g in enumerate(engs):
        g.set_batch(f["user_input"][idx[r]] // 2, f["item_input"][idx[r]], labels=f["labels"][idx[r]], global_batch=200)
    outs = run.step()
    assert outs[0].cpu().numpy()[9] == 2.0


@pytest.mark.parametrize("W", [2, 3])
def test_sharded_catalog_topk_equals_unsharded(W):
    """Item-sharded full-catalog top-K (query rows gathered, per-shard top-K with global ids,
    lists back to the user owners, fr_catalog_merge) == the unsharded engine, bit for bit."""
    from foodrec_b200 import Engine, Hyper
    p = Problem(300, 4001, 9, 128, seed=17)           # 4001 recipes: padded shards
    K, n = 40, 24
    single = Engine(Hyper(), p.tb.P, p.tb.R, p.tb.Cat, p.tb.G, max_rows=256, item_cats=p.item_cats)
    engs = [sharded.ShardedEngine(Hyper(), sharded.shard_rows(p.tb.P, r, W), sharded.shard_rows(p.tb.R, r, W),
                                  p.tb.Cat, p.tb.G, r, W, max_rows=256, item_cats_global=p.item_cats)
            for r in range(W)]
    for g in engs:
        g.catalog_prepare()
    rng = np.random.default_rng(3)
    local_users = [rng.integers(0, len(range(r, p.U, W)), n).astype(np.int32) for r in range(W)]
    outs = sharded.LocalRunner(engs).catalog_topk(local_users, K=K)
    for r in range(W):
        gu = local_users[r].astype(np.int64) * W + r          # global user ids of rank r's queries
        ids, sc = single.catalog_topk(users=gu.astype(np.int32), K=K)
        assert torch.equal(outs[r][0], ids) and torch.equal(outs[r][1], sc), r
    assert int(outs[0][0].max()) < p.I                        # pad rows of the last shard are never returned


@pytest.mark.parametrize("adam_mode", ["lazy_exact", "lazy"])
def test_sharded_checkpoint_resume(tmp_path, adam_mode):
    """Save after 2 sharded steps, restore into FRESH engines, run 2 more == 4 uninterrupted steps (tables, Adam
    slots, stamps and step counter round-trip per rank).  Bit-identical with the step-by-step lazy replay; with the
    closed-form catch-up the checkpoint's flush splits a gap in two, which moves last bits only."""
    W = 2
    p = Problem(203, 157, 9, 64, seed=33)

    def feed(engs, s):
        f = p.bpr(200, seed=300 + s)
        idx = sharded.route_batch(f["user_input"], W)
        for r, g in enumerate(engs):
            ix = idx[r]
            g.set_batch(f["user_input"][ix] // W, f["item_input"][ix], neg_items=f["neg_item_input"][ix], global_batch=200)

    _, a = build(p, W, "adam", adam_mode)
    ra = sharded.LocalRunner(a)
    for s in range(4):
        feed(a, s); ra.step()
    _, b = build(p, W, "adam", adam_mode)
    rb = sharded.LocalRunner(b)
    for s in range(2):
        feed(b, s); rb.step()
    for g in b:
        g.save(str(tmp_path / "ckpt-2"))
    _, c = build(p, W, "adam", adam_mode)
    for g in c:
        g.restore(str(tmp_path / "ckpt-2"))
    rc = sharded.LocalRunner(c)
    for s in range(2, 4):
        feed(c, s); rc.step()
    ta, tc = gather(a, p), gather(c, p)
    for k in ("P", "R", "Cat", "G"):
        if adam_mode == "lazy_exact":
            np.testing.assert_array_equal(ta[k], tc[k], err_msg=k)
        else:
            assert_close(tc[k], ta[k], rtol=1e-6, what=k)
    assert a[0].e.step == c[0].e.step == 4


@pytest.mark.parametrize("W,bpr", [(2, True), (4, False)])
def test_peer_store_exchange_equals_all_to_all(W, bpr):
    """fr_shard_set_peers: gather and gradient kernels store rows straight into the consumer rank's buffer (the
    NVLink P2P path; here the peers are engines of this process).  Bit-identical to the staged all-to-all path."""
    p = Problem(403, 257, 9, 64, seed=62)
    _, a = build(p, W, "adam", "lazy")
    _, b = build(p, W, "adam", "lazy")
    ra, rb = sharded.LocalRunner(a), sharded.LocalRunner(b)
    rb.enable_p2p()
    for s in range(4):
        f = p.bpr(300, seed=500 + s) if bpr else p.pointwise(300, seed=500 + s)
        idx = sharded.route_batch(f["user_input"], W)
        for engs in (a, b):
            for r, g in enumerate(engs):
                ix = idx[r]
                g.set_batch(f["user_input"][ix] // W, f["item_input"][ix], labels=None if bpr else f["labels"][ix],
                            neg_items=f["neg_item_input"][ix] if bpr else None, global_batch=300)
        oa = ra.step(write_personal=(s == 0)); ob = rb.step(write_personal=(s == 0))
        assert torch.equal(oa[0], ob[0])
    ta, tb_ = gather(a, p), gather(b, p)
    for k in ("P", "R", "Cat", "G"):
        np.testing.assert_array_equal(ta[k], tb_[k], err_msg=k)
