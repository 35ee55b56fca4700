"""The row-sharded step (fr_shard_plan / serve / forward / update / apply, W ranks in one process through LocalRunner)
against the fp64 oracle directly, at the shapes and schedules the single-GPU suite covers: every embedding width class
(DV = 1, one lane group, a partial last lane group, NV = 2), every optimizer, bf16 tables, the peer-store exchange, an
active global-norm clip (known only after the all-reduce) and personal-write steps after lazy rows went stale and
single-pass rows moved to the shadow copy.  Also: timing mode, which changes the schedule of a step, computes the same
step bit for bit."""
import numpy as np
import pytest

from foodrec_b200 import sharded
from oracle.recommender_oracle import Hyper as OHyper, OracleModel
from tests.test_gpu_bf16 import check_tables
from tests.util import Problem, assert_close, assert_close_adam

pytestmark = pytest.mark.gpu

HOT = 5                  # the recipe of the step whose rows are ~90 % one recipe
HOT_ROWS = 16 * 32       # a run of more than 16 chunks of 32 rows is summed by seg_combine_long_kernel


def build(p, W, learner, adam_mode="dense", lr=0.01, single_pass=None, table_dtype="float32", max_rows=4096, **hk):
    from foodrec_b200 import Hyper
    h = Hyper(learner=learner, lr=lr, **hk)
    rows, cols = np.nonzero(p.user_labels)
    cnt = np.bincount(rows, minlength=p.U)
    off = np.zeros(p.U + 1, np.int32); off[1:] = np.cumsum(cnt)
    engs = [sharded.ShardedEngine(
        h, sharded.shard_rows(p.tb.P, r, W), sharded.shard_rows(p.tb.R, r, W), p.tb.Cat, p.tb.G, r, W,
        max_rows=max_rows, adam_mode=adam_mode, item_cats_global=p.item_cats,
        user_label_csr_local=sharded.shard_label_csr(off, cols.astype(np.int32), r, W, p.U),
        max_label_entries=max_rows * p.L, single_pass=single_pass, table_dtype=table_dtype) for r in range(W)]
    if learner == "adam" and adam_mode != "dense":
        assert all(g.e.single_pass == (single_pass is None) for g in engs)
    return engs


def gather(engs, p):
    """Global tables (lazy Adam flushed, bf16 widened); the replicated ones must be identical on every rank."""
    ts = [g.e.tables() for g in engs]
    for t in ts[1:]:
        np.testing.assert_array_equal(t["Cat"], ts[0]["Cat"])
        np.testing.assert_array_equal(t["G"], ts[0]["G"])
    return {"P": sharded.unshard_rows([t["P"] for t in ts], p.U), "R": sharded.unshard_rows([t["R"] for t in ts], p.I),
            "Cat": ts[0]["Cat"], "G": ts[0]["G"]}


def close(engs):
    for g in engs:
        g.e.close()


def with_write_sign(f, rng):
    """Pointwise feeds carry the feed's write_sign scaled by a per-row factor: the label-derived sign the kernels use when
    no write_sign is given would then move General_Memory differently, so a write_sign that does not reach the step fails."""
    f["write_sign"] = (f["write_sign"] * rng.uniform(0.5, 1.5, f["write_sign"].shape)).astype(np.float32)
    return f


def make_feed(p, W, kind, bpr, seed):
    rng = np.random.default_rng(seed)
    users = None
    B = 300
    if kind == "dup":             # 16 users on every rank, runs of 40 rows: they cross 32-row chunks
        users = np.repeat(np.arange(16) * 5 % p.U, 40)
        B = users.size
    elif kind == "one_owner":     # every user belongs to rank 1: the other ranks have no rows
        users = 1 + W * rng.integers(0, (p.U - 1) // W, 256)
        B = users.size
    elif kind == "hot":           # ~90 % of the rows hit one recipe: every rank's pre-reduce holds a run of > 16 chunks
        B = 700 * W
    f = p.bpr(B, seed=seed, users=users) if bpr else p.pointwise(B, seed=seed, users=users)
    if kind == "hot":
        it = np.where(rng.random(B) < 0.9, HOT, f["item_input"]).astype(np.int32)
        f["item_input"], f["categories"] = it, p.item_cats[it].reshape(B, 4, 1).copy()
        if bpr:
            f["neg_item_input"] = np.where(f["neg_item_input"] == it, (it + 1) % p.I, f["neg_item_input"]).astype(np.int32)
            f["neg_categories"] = p.item_cats[f["neg_item_input"]].reshape(B, 4, 1).copy()
    if not bpr:
        with_write_sign(f, rng)
    return f


def sharded_step(run, engs, f, bpr, personal=False):
    """Route the global batch to the user owners, run one step; returns every rank's scalars and the routing."""
    W = len(engs)
    B = len(f["user_input"])
    idx = sharded.route_batch(f["user_input"], W)
    for r, g in enumerate(engs):
        ix = idx[r]
        g.set_batch(f["user_input"][ix] // W, f["item_input"][ix], labels=None if bpr else f["labels"][ix],
                    neg_items=f["neg_item_input"][ix] if bpr else None,
                    write_sign=None if bpr else f["write_sign"][ix], global_batch=B)
    return [o.cpu().numpy().copy() for o in run.step(write_personal=personal)], idx


def oracle_step(om, f, bpr, personal=False):
    return om.train_step_bpr(f, write_personal=personal) if bpr else om.train_step(f, write_personal=personal)


def check_scalars(outs, o, om, what):
    """Every rank reports the same loss, norm, clip scale and mean(G) (one all-reduced sum, replicated G), equal to the
    oracle's.  `personal` is not produced by the sharded phases."""
    for r, v in enumerate(outs):
        assert v[9] == 0, f"{what}: rank {r} overflow flag {v[9]}"
        np.testing.assert_array_equal(v[:4], outs[0][:4], err_msg=f"{what}: rank {r} disagrees with rank 0")
    v = outs[0]
    assert v[0] == pytest.approx(float(o["loss"]), rel=1e-5), f"{what}: loss"
    assert v[1] == pytest.approx(float(o["norm"]), rel=1e-5), f"{what}: norm"
    assert v[2] == pytest.approx(float(o["scale"]), rel=1e-5), f"{what}: scale"
    assert v[3] == pytest.approx(float(o["general"]), rel=1e-5, abs=1e-5 * float(np.abs(om.G).mean())), f"{what}: general"


def check_tables_fp32(t, om, om32, what):
    for k in ("P", "R", "Cat", "G"):
        if om32 is not None and k != "G":
            assert_close_adam(t[k], getattr(om, k), getattr(om32, k), what=f"{what} {k}")
        else:
            assert_close(t[k], getattr(om, k), what=f"{what} {k}")


BF16_LR = {"sgd": 0.5, "adagrad": 0.05, "rmsprop": 0.002}      # (as tests/test_gpu_bf16.py: updates above one bf16 ulp)


# D, W, learner, adam_mode, single_pass, bpr, bf16, p2p: pairwise over the axes, not their product
CASES = [
    (4, 2, "sgd", "dense", None, False, False, False),
    (4, 3, "adam", "lazy", None, True, False, False),
    (64, 8, "adagrad", "dense", None, False, False, True),
    (132, 2, "rmsprop", "dense", None, True, False, False),
    (132, 3, "adam", "dense", None, False, False, False),
    (132, 8, "adam", "lazy", False, True, False, False),
    (132, 8, "adagrad", "dense", None, False, True, False),
    (200, 2, "adam", "lazy_exact", None, False, False, True),
    (200, 3, "sgd", "dense", None, True, True, False),
    (200, 3, "rmsprop", "dense", None, False, True, False),
    (200, 8, "adam", "lazy", None, False, False, False),
    (256, 2, "adagrad", "dense", None, True, False, False),
    (256, 3, "sgd", "dense", None, False, False, False),
    (256, 8, "rmsprop", "dense", None, True, False, True),
]


@pytest.mark.parametrize("D,W,learner,adam_mode,single_pass,bpr,bf16,p2p", CASES)
def test_sharded_steps_match_oracle(D, W, learner, adam_mode, single_pass, bpr, bf16, p2p):
    p = Problem(403, 257, 9, D, seed=40 + D + W)          # U, I not divisible by W: padded shards
    lr = BF16_LR[learner] if bf16 else 0.01
    engs = build(p, W, learner, adam_mode, lr=lr, single_pass=single_pass, table_dtype="bf16" if bf16 else "float32")
    run = sharded.LocalRunner(engs)
    if p2p:
        run.enable_p2p()
    oh = OHyper(learner=learner, lr=lr)
    if bf16:        # the bf16 storage rule is defined on float32 arithmetic (tests/test_gpu_bf16.py)
        om, om32 = OracleModel(p.tb.P, p.tb.R, p.tb.Cat, p.tb.G, oh, dtype=np.float32, table_dtype="bf16"), None
    else:
        om = p.oracle(oh)
        om32 = p.oracle(oh, dtype=np.float32) if learner == "adam" else None
    what = f"D={D} W={W} {learner}/{adam_mode} sp={single_pass} bpr={bpr} bf16={bf16} p2p={p2p}"
    # the personal-write step comes after two ordinary steps: lazy rows are stale, single-pass rows in the shadow copy
    schedule = [("plain", False), ("dup", False), ("one_owner", False), ("plain", not bf16), ("hot", False),
                ("plain", False)]
    for s, (kind, personal) in enumerate(schedule):
        f = make_feed(p, W, kind, bpr, seed=1000 * D + 10 * W + s)
        outs, idx = sharded_step(run, engs, f, bpr, personal)
        o = oracle_step(om, f, bpr, personal)
        if om32 is not None:
            oracle_step(om32, f, bpr, personal)
        if kind == "one_owner":
            assert [len(ix) > 0 for ix in idx] == [r == 1 for r in range(W)]
        if kind == "hot":
            rows = [int((f["item_input"][ix] == HOT).sum()) for ix in idx]
            assert min(rows) > HOT_ROWS, rows
        check_scalars(outs, o, om, f"{what} step {s} ({kind})")
    t = gather(engs, p)
    if bf16:
        check_tables(t, om, what)
    else:
        check_tables_fp32(t, om, om32, what)
    close(engs)


@pytest.mark.parametrize("learner,adam_mode,single_pass,D,W,bpr", [
    ("adam", "lazy", None, 132, 2, False),      # single-pass: the speculation fails on clipped steps and is redone
    ("adam", "lazy", None, 256, 3, True),
    ("adam", "lazy", False, 256, 2, False),     # two-pass
    ("adagrad", "dense", None, 132, 3, True),
    ("rmsprop", "dense", None, 256, 3, False),
])
def test_sharded_active_clip_matches_oracle(learner, adam_mode, single_pass, D, W, bpr):
    """Tables 60x larger than elsewhere: the global norm exceeds clip_norm on some steps.  The sharded step knows the
    clip scale only after the all-reduce; finalize applies it to Cat, the user pass redoes a speculative single-pass
    update, and every gradient row a rank sends is scaled before its owner applies it."""
    p = Problem(403, 257, 9, D, seed=11 + D, scale=6.0)
    kinds = ["plain", "dup", "plain", "plain", "dup", "one_owner", "plain", "dup"]
    fs = [make_feed(p, W, k, bpr, seed=90 + s) for s, k in enumerate(kinds)]
    probe = p.oracle(OHyper(learner=learner, lr=0.01, clip_norm=1e30))
    norms = [float(oracle_step(probe, f, bpr)["norm"]) for f in fs]
    clip = float(np.median(norms))
    personal_step = 2 + int(np.argmax(norms[2:]))          # a personal-write step on a step that clips
    oh = OHyper(learner=learner, lr=0.01, clip_norm=clip)
    om = p.oracle(oh)
    om32 = p.oracle(oh, dtype=np.float32) if learner == "adam" else None
    engs = build(p, W, learner, adam_mode, single_pass=single_pass, clip_norm=clip)
    run = sharded.LocalRunner(engs)
    what = f"clip {learner}/{adam_mode} sp={single_pass} D={D} W={W} bpr={bpr}"
    clipped = 0
    for s, f in enumerate(fs):
        personal = s == personal_step
        outs, idx = sharded_step(run, engs, f, bpr, personal)
        o = oracle_step(om, f, bpr, personal)
        if om32 is not None:
            oracle_step(om32, f, bpr, personal)
        # near the threshold the sharded and the oracle sums could disagree about whether the step clips; the seeds are
        # chosen so that no step comes near it (another seed if this fails)
        assert abs(float(o["norm"]) - clip) > 1e-4 * clip, (s, float(o["norm"]), clip)
        check_scalars(outs, o, om, f"{what} step {s}")
        clipped += float(o["scale"]) < 1.0
        if personal:
            assert float(o["scale"]) < 1.0, "the personal-write step should clip"
        if kinds[s] == "one_owner":
            assert sum(len(ix) == 0 for ix in idx) == W - 1
    assert 2 <= clipped <= 6, clipped
    check_tables_fp32(gather(engs, p), om, om32, what)
    close(engs)


@pytest.mark.parametrize("case", ["single_adam_lazy", "single_adagrad", "sharded_adam_lazy"])
def test_timing_mode_computes_the_same_step(case):
    """fr_timing_enable records events between the phases and runs the label pass and finalize in sequence instead of
    beside the forward / single-pass kernel.  The kernels have no atomics on the data path, so the step must be the same
    bit for bit; the events must really have been recorded."""
    from foodrec_b200 import Engine, Hyper
    p = Problem(403, 257, 9, 132, seed=77)
    fs = [p.pointwise(300, seed=700 + s, users=np.repeat(np.arange(10) * 7, 30) if s == 1 else None) for s in range(4)]
    personal = [False, False, True, False]
    if case.startswith("single"):
        learner, mode = ("adam", "lazy") if case == "single_adam_lazy" else ("adagrad", "dense")
        mk = lambda: Engine(Hyper(learner=learner, lr=0.01), p.tb.P, p.tb.R, p.tb.Cat, p.tb.G, max_rows=2048, adam_mode=mode,
                            max_label_entries=2048 * p.L, item_cats=p.item_cats, user_labels=p.user_labels)
        a, b = mk(), mk()
        assert a.single_pass == (learner == "adam")
        b.timing_enable(True)
        for f, pw in zip(fs, personal):
            for e in (a, b):
                e.train_step(f["user_input"], f["item_input"], labels=f["labels"], write_sign=f["write_sign"],
                             write_personal=pw)
            np.testing.assert_array_equal(a.read_scalars(), b.read_scalars())
        ph, n = b.timing_read()
        assert n == len(fs) and ph["fwd"] > 0, (n, ph)
        ta, tb = a.tables(), b.tables()
        a.close(); b.close()
    else:
        W = 2
        ea, eb = build(p, W, "adam", "lazy"), build(p, W, "adam", "lazy")
        ra, rb = sharded.LocalRunner(ea), sharded.LocalRunner(eb)
        for g in eb:
            g.e.timing_enable(True)
        for f, pw in zip(fs, personal):
            oa, _ = sharded_step(ra, ea, f, False, pw)
            ob, _ = sharded_step(rb, eb, f, False, pw)
            for x, y in zip(oa, ob):
                np.testing.assert_array_equal(x, y)
        for g in eb:      # fr_shard_update records its own phases; the others read zero
            ph, _ = g.e.timing_read()
            assert ph["user_chunk"] > 0, ph
        ta, tb = gather(ea, p), gather(eb, p)
        close(ea); close(eb)
    for k in ("P", "R", "Cat", "G"):
        np.testing.assert_array_equal(ta[k], tb[k], err_msg=k)
