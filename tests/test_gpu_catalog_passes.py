"""GPU tests of full-catalog top-K at the configurations only production-sized calls reach, against the oracle for
EVERY row: calls cut into several passes (``max_pass_rows``), every round of the exact fallback and its
self-contained tail, the fallback under recipe shards, and the index rebuilt by itself after training steps.

The exact fallback takes ``fallback_blocks`` rows per round for four rounds (``cat_exact_scores_kernel`` +
``cat_exact_kernel``), then one block per row for the rest (the tail).  Fallback cases therefore send
``4 * fb + fb // 2 + 7`` rows of one pass to it (``fb`` from the sizing rule, asserted against ``catalog_info``).  Oracle:
``tests/catalog_exclude_oracle.catalog_topk_chunked`` (fp64 GEMM form, ties by ascending id), or the exact
per-recipe formula of ``test_catalog_ties_are_broken_by_id`` for tables with exact ties."""
import numpy as np
import pytest
import torch

from oracle import synth
from oracle.recommender_oracle import Hyper as OHyper, OracleModel, health_rows
from tests import catalog_exclude_oracle as xo
from tests.test_gpu_catalog_exclude import random_lists
from tests.util import Problem

pytestmark = pytest.mark.gpu


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def n_fallback_rows(fb):
    return 4 * fb + fb // 2 + 7          # every round full, then the tail


def engine(tb, ic, **kw):
    from foodrec_b200 import Engine, Hyper
    return Engine(kw.pop("hyper", Hyper()), tb.P, tb.R, tb.Cat, tb.G, max_rows=256, item_cats=ic, **kw)


def assert_matches(ids, sc, rid, rsc, rel=1e-12):
    ids = ids.cpu().numpy() if torch.is_tensor(ids) else ids
    sc = sc.cpu().numpy() if torch.is_tensor(sc) else sc
    assert ids.shape == rid.shape
    bad = np.nonzero((ids != rid).any(1))[0]
    assert bad.size == 0, f"{bad.size} of {ids.shape[0]} rows differ, first {bad[:8].tolist()}"
    fin = np.isfinite(rsc)
    assert np.array_equal(fin, np.isfinite(sc))
    if fin.any():
        assert np.abs(sc[fin] - rsc[fin]).max() <= rel * np.abs(rsc[fin]).max()


def in_table(lists, I, id_mul=1, id_add=0):
    """Entries of each list the table (local rows * id_mul + id_add) holds, duplicates counted: what K_eff adds."""
    out = []
    for x in lists:
        x = np.asarray(x, np.int64) - id_add
        out.append(int(((x >= 0) & (x % id_mul == 0) & (x // id_mul < I)).sum()))
    return np.asarray(out)


# ---------------------------------------------------------------------------- 1. calls cut into passes
@pytest.mark.parametrize("prep", [{}, dict(splits=1), dict(cta_group=1)])
def test_multi_pass_calls_match_the_oracle_and_the_one_pass_call(prep):
    """A 2,600-row query cut into 6 passes of 512 rows (ragged last pass of 40): split sweeps (the default for a
    small pass), whole sweeps with the per-pass user sort (splits=1), single-CTA blocks of 128 rows.  Query rows as
    the first n users, as a user list with duplicates in random order, and as dense P rows; with and without
    lists.  Every row equals the oracle, and the ids (and the call's fallback count) equal the one-pass call's."""
    U, I, D, K, mpr = 2600, 4500, 64, 40, 400            # passes of 512 rows (400 rounded up to whole blocks)
    tb = synth.make_tables(U, I, 7, D, seed=71)
    ic = synth.make_item_categories(I, seed=72)
    e = engine(tb, ic)
    om = OracleModel(tb.P, tb.R, tb.Cat, tb.G, OHyper(), dtype=np.float32)
    rng = np.random.default_rng(73)
    users = rng.integers(0, U, U + 300).astype(np.int32)
    users[rng.integers(0, users.size, 200)] = users[:200]                   # duplicates, random order
    rows = e.P[torch.as_tensor(users.astype(np.int64), device=e.device)]
    forms = [("first_n", dict(n_users=U), np.arange(U)), ("users", dict(users=users), users),
             ("P_rows", dict(P_rows=rows), users)]
    results = {}
    for one_pass in (True, False):
        e.catalog_prepare(max_pass_rows=0 if one_pass else mpr, **prep)
        if not one_pass:
            e.timing_enable(True)
            e.catalog_topk(n_users=U, K=K)
            _, passes = e.catalog_timing_read()
            e.timing_enable(False)
            assert passes == 6
        for name, q, uu in forms:
            for with_lists in (False, True):
                excl = random_lists(np.random.default_rng(len(uu)), len(uu), I) if with_lists else None
                ids, sc = e.catalog_topk(K=K, exclude=excl, **q)
                results[one_pass, name, with_lists] = (ids.cpu().numpy(), sc.cpu().numpy(), e.catalog_fallback_rows())
                if not one_pass:
                    assert_matches(ids, sc, *xo.catalog_topk_chunked(om, uu, ic, K, excl))
    for name, _, _ in forms:
        for with_lists in (False, True):
            multi, single = results[False, name, with_lists], results[True, name, with_lists]
            assert np.array_equal(multi[0], single[0]) and multi[2] == single[2], (name, with_lists)
    e.close()


# ---------------------------------------------------------------------------- 2. fallback rows flagged up front
@pytest.mark.parametrize("I,D,K,variant", [
    (1 << 20, 16, 100, "plain"),         # fallback_blocks = 512 MB / (I * 8 B) = 64: the tail starts at row 256
    (1 << 20, 16, 100, "health"),        # health blend: the fallback gathers each user's General_Memory rows
    (200_000, 64, 100, "plain"),         # fallback_blocks = SM count
    (200_000, 64, 100, "P_rows"),        # dense query rows
    (200_000, 64, 256, "plain"),         # largest K: every row with one listed recipe of the table falls back
    (200_000, 64, 100, "pad"),           # lists that leave fewer than K recipes: -1 / -inf padding
])
def test_every_fallback_round_and_the_tail_with_rows_flagged_up_front(I, D, K, variant):
    """Rows whose K + listed recipes of the table exceed 256 go to the exact fallback before the filter runs.  Enough
    of them (interleaved with rows the filter handles) fill all four rounds and reach the tail; lists carry
    duplicates and ids outside the table.  Every row equals the oracle; the call's count equals the flagged rows."""
    from foodrec_b200 import Hyper
    rng = np.random.default_rng(I + D + K)
    fb_expect = min(sm_count(), (512 << 20) // (I * 8))
    n_fb = n_fallback_rows(fb_expect)
    n = U = n_fb + n_fb // 3
    heavy = np.zeros(n, bool)
    heavy[rng.permutation(n)[:n_fb]] = True                                 # interleaved with filter rows
    tb = synth.make_tables(U, I, 7, D, seed=K)
    ic = synth.make_item_categories(I, seed=D)
    lists = []
    for r in range(n):
        if variant == "pad" and r % 97 == 5:
            keep = rng.choice(I, int(rng.integers(0, K)), replace=False)   # fewer than K recipes remain
            x = np.setdiff1d(np.arange(I), keep).tolist()
        elif heavy[r]:
            x = rng.choice(I, int(rng.integers(160, 401)), replace=False).tolist()
            if r % 3 == 0:
                x += x[:20] + [I + int(rng.integers(0, 1000)), -1 - int(rng.integers(0, 100))]
            rng.shuffle(x)
        else:
            x = rng.integers(0, I, int(rng.integers(0, 157 - 100 if K == 100 else 1))).tolist()
            if r % 4 == 0 and K == 256:
                x = [I + 3, -5]                                             # no entry in the table: K_eff = 256
        lists.append(x)
    users = rng.permutation(U).astype(np.int32)
    kw = {}
    om_P = tb.P
    if variant == "health":
        user_labels = synth.make_user_labels(U, 7, seed=4)
        tb.G = (tb.G * 5).astype(np.float32)
        kw = dict(hyper=Hyper(alpha=0.35), user_labels=user_labels)
        om_P = health_rows(tb.P, tb.G, user_labels, 0.35)
    e = engine(tb, ic, **kw)
    if variant == "health":
        e.set_health_blend(True)
    e.catalog_prepare()
    flagged = int((K + in_table(lists, I) > 256).sum())
    assert flagged >= n_fb
    if variant == "P_rows":
        rows = e.P[torch.as_tensor(users.astype(np.int64), device=e.device)]
        ids, sc = e.catalog_topk(P_rows=rows, K=K, exclude=lists)
    else:
        ids, sc = e.catalog_topk(users=users, K=K, exclude=lists)
    assert e.catalog_fallback_rows() == flagged
    assert e.catalog_info()["fallback_blocks"] == fb_expect     # (sized with the first query's workspace)
    om = OracleModel(om_P, tb.R, tb.Cat, tb.G, OHyper(alpha=0.35) if variant == "health" else OHyper(), dtype=np.float32)
    rid, rsc = xo.catalog_topk_chunked(om, users, ic, K, lists)
    assert_matches(ids, sc, rid, rsc)
    if variant == "pad":
        assert (rid == -1).any()
    e.close()


# ---------------------------------------------------------------------------- 3. rows that overflow at the re-rank
def tied_tables(U, I, D, seed):
    """Integer-valued tables with three distinct recipe rows: hundreds of recipes tie exactly at every boundary."""
    rng = np.random.default_rng(seed)
    tb = synth.make_tables(U, I, 7, D, seed=3)
    base = rng.integers(-4, 5, (3, D)).astype(np.float32) / 8
    tb.R[:] = base[rng.integers(0, 3, I)]
    tb.P[:] = rng.integers(-4, 5, tb.P.shape).astype(np.float32) / 8
    tb.Cat[:] = rng.integers(-4, 5, tb.Cat.shape).astype(np.float32) / 8
    return tb


def tied_oracle(tb, ic, users, K):
    """The exact per-recipe fp64 formula (products of multiples of 1/8 sum exactly: identical rows tie exactly)."""
    w = ic.astype(np.float64); w /= w.sum(1, keepdims=True)
    om = OracleModel(tb.P, tb.R, tb.Cat, tb.G, OHyper(), dtype=np.float32)
    a, b = np.float64(om.a), np.float64(om.one_minus_a)
    P, R, Cat = (x.astype(np.float64) for x in (tb.P, tb.R, tb.Cat))
    I = R.shape[0]
    ids = np.empty((len(users), K), np.int64); sc = np.empty((len(users), K))
    for r, u in enumerate(users):
        s = a * (w * (Cat @ P[u, 0])).sum(1) + b * (w * (R @ P[u, 1:].T)).sum(1)
        order = np.lexsort((np.arange(I), -s))[:K]
        ids[r], sc[r] = order, s[order]
    return ids, sc


@pytest.mark.parametrize("prep", [{}, dict(splits=1)])
def test_every_fallback_round_and_the_tail_with_rows_that_overflow(prep):
    """Every row's candidates overflow (detected in the GEMM epilogue with whole sweeps, at the re-rank with split
    sweeps): all of them take the exact fallback, through all four rounds and the tail, ranked by (score, id)."""
    I, D, K = 20_000, 64, 100
    fb = min(sm_count(), (512 << 20) // (I * 8))
    U = n_fallback_rows(fb)
    tb = tied_tables(U, I, D, seed=5)
    ic = synth.make_item_categories(I, seed=9)
    e = engine(tb, ic)
    e.catalog_prepare(**prep)
    ids, sc = e.catalog_topk(n_users=U, K=K)
    assert e.catalog_info()["fallback_blocks"] == fb
    assert e.catalog_fallback_rows() == U
    assert_matches(ids, sc, *tied_oracle(tb, ic, np.arange(U), K))
    e.close()


def test_fallback_count_sums_over_the_passes_and_restarts_with_each_call():
    I, D, K, U = 20_000, 64, 100, 700
    tb = tied_tables(U, I, D, seed=6)
    ic = synth.make_item_categories(I, seed=9)
    e = engine(tb, ic)
    e.catalog_prepare(max_pass_rows=256)                   # 3 passes: 256 + 256 + 188
    ids, sc = e.catalog_topk(n_users=U, K=K)
    assert e.catalog_fallback_rows() == U                  # not just the last pass's 188
    assert_matches(ids, sc, *tied_oracle(tb, ic, np.arange(U), K))
    users = np.arange(U - 1, U - 101, -1).astype(np.int32)
    ids, sc = e.catalog_topk(users=users, K=K)
    assert e.catalog_fallback_rows() == 100                # a new call counts its own rows
    assert_matches(ids, sc, *tied_oracle(tb, ic, users, K))
    e.close()


# ---------------------------------------------------------------------------- 4. recipe shards
def test_recipe_shards_with_fallback_rows_on_some_shards_merge_to_the_unsharded_answer():
    """Lists made so that a row falls back on one shard only, on every shard, only unsharded, or nowhere: the
    fallback writes global ids (local row * W + rank) and the merge equals the unsharded answer."""
    from foodrec_b200 import Engine, Hyper
    U, I, D, K, W = 240, 6001, 128, 50, 3
    tb = synth.make_tables(U, I, 7, D, seed=81)
    ic = synth.make_item_categories(I, seed=82)
    om = OracleModel(tb.P, tb.R, tb.Cat, tb.G, OHyper(), dtype=np.float32)
    rng = np.random.default_rng(83)
    lists = []
    for r in range(U):
        kind = r % 4
        if kind == 0:                                        # 300 recipes of shard r % W: that shard only
            x = (rng.choice(I // W, 300, replace=False) * W + (r // 4) % W).tolist()
        elif kind == 1:                                      # 240 per shard: every shard and unsharded
            x = rng.choice(I, 3 * 240, replace=False).tolist()
        elif kind == 2:                                      # ~150 per shard: unsharded only
            x = rng.choice(I, 450, replace=False).tolist()
        else:
            x = rng.integers(0, I, 40).tolist() + [I + 1, -3]
        lists.append(x)
    e = Engine(Hyper(), tb.P, tb.R, tb.Cat, tb.G, max_rows=256, item_cats=ic)
    ids, sc = e.catalog_topk(K=K, exclude=lists)
    assert e.catalog_fallback_rows() == int((K + in_table(lists, I) > 256).sum())
    rid, rsc = xo.catalog_topk_chunked(om, np.arange(U), ic, K, lists)
    assert_matches(ids, sc, rid, rsc)
    parts_i, parts_s, shard_fb = [], [], []
    for r in range(W):
        sel = np.arange(r, I, W)
        es = Engine(Hyper(), tb.P, tb.R[sel], tb.Cat, tb.G, max_rows=256, item_cats=ic[sel])
        li, ls = es.catalog_topk(K=K, id_mul=W, id_add=r, exclude=lists)
        fb = es.catalog_fallback_rows()
        assert fb == int((K + in_table(lists, len(sel), W, r) > 256).sum()), r
        shard_fb.append(fb)
        parts_i.append(li.clone()); parts_s.append(ls.clone())
        torch.cuda.synchronize()
        es.close()
    assert 0 < min(shard_fb) and max(shard_fb) < U // 2                  # some rows on some shards only
    mi, ms = e.catalog_merge(torch.stack(parts_i), torch.stack(parts_s))
    assert torch.equal(mi, ids)
    assert_matches(mi, ms, rid, rsc)
    e.close()


# ---------------------------------------------------------------------------- 5. index rebuilt after training
def test_engine_rebuilds_the_index_with_the_options_it_was_prepared_with():
    """prepare(max_pass_rows, epi_sets) -> top-K -> a training step -> top-K rebuilds the stale index with the same
    options (same passes, same catalog_info) and answers for the trained tables; a later default prepare needs a
    larger pass workspace, which is re-allocated."""
    from foodrec_b200 import Engine, Hyper
    p = Problem(1000, 3000, 7, 64, seed=91)
    e = Engine(Hyper(learner="sgd", lr=0.05), p.tb.P, p.tb.R, p.tb.Cat, p.tb.G, max_rows=2048,
               max_label_entries=2048 * p.L, item_cats=p.item_cats)
    K = 30

    def check():
        e.timing_enable(True)
        ids, sc = e.catalog_topk(n_users=p.U, K=K)
        _, passes = e.catalog_timing_read()
        e.timing_enable(False)
        t = e.tables()
        om = OracleModel(t["P"], t["R"], t["Cat"], t["G"], OHyper(), dtype=np.float32)
        assert_matches(ids, sc, *xo.catalog_topk_chunked(om, np.arange(p.U), p.item_cats, K))
        return passes

    e.catalog_prepare(max_pass_rows=300, epi_sets=2)       # passes of 512 rows: 2 for 1,000 users
    assert check() == 2
    info = e.catalog_info()
    f = synth.shuffled_bpr_batch(p.U, p.I, 1024, p.item_cats, p.user_labels, seed=4)
    e.train_step(f["user_input"], f["item_input"], categories=f["categories"], neg_items=f["neg_item_input"],
                 neg_categories=f["neg_categories"], user_one_hot_label=f["user_one_hot_label"])
    assert check() == 2
    assert e.catalog_info() == info
    e.catalog_prepare()
    assert check() == 1
    assert e.catalog_info()["epi_sets"] != info["epi_sets"]          # the explicit call's defaults: one epilogue set
    e.close()


@pytest.mark.parametrize("W", [2, 3])
def test_local_runner_rebuilds_each_shards_index_from_its_own_masks(W):
    """Recipe shards that were never prepared, then trained for two steps: every rank's index must be built from
    the masks of ITS rows (local row k = recipe rank + k*W), not from the first rows of the global map.  The
    answer equals the unsharded engine on the same tables, before and after training."""
    from foodrec_b200 import Engine, Hyper, sharded
    p = Problem(300, 4001, 9, 64, seed=17)
    K, n = 40, 24
    h = Hyper(learner="sgd", lr=0.05)
    rows, cols = np.nonzero(p.user_labels)
    off = np.zeros(p.U + 1, np.int32); off[1:] = np.cumsum(np.bincount(rows, minlength=p.U))
    engs = [sharded.ShardedEngine(h, sharded.shard_rows(p.tb.P, r, W), sharded.shard_rows(p.tb.R, r, W),
                                  p.tb.Cat, p.tb.G, r, W, max_rows=2048, item_cats_global=p.item_cats,
                                  user_label_csr_local=sharded.shard_label_csr(off, cols.astype(np.int32), r, W, p.U),
                                  max_label_entries=2048 * p.L)
            for r in range(W)]
    run = sharded.LocalRunner(engs)
    rng = np.random.default_rng(3)
    local_users = [rng.integers(0, len(range(r, p.U, W)), n).astype(np.int32) for r in range(W)]

    def check(tables):
        single = Engine(Hyper(), tables["P"], tables["R"], tables["Cat"], tables["G"], max_rows=256,
                        item_cats=p.item_cats)
        outs = run.catalog_topk(local_users, K=K)
        om = OracleModel(tables["P"], tables["R"], tables["Cat"], tables["G"], OHyper(), dtype=np.float32)
        for r in range(W):
            gu = (local_users[r].astype(np.int64) * W + r).astype(np.int32)
            ids, sc = single.catalog_topk(users=gu, K=K)
            assert torch.equal(outs[r][0], ids) and torch.equal(outs[r][1], sc), r
            assert_matches(ids, sc, *xo.catalog_topk_chunked(om, gu, p.item_cats, K))
        single.close()

    check({"P": p.tb.P, "R": p.tb.R, "Cat": p.tb.Cat, "G": p.tb.G})      # never prepared
    for s in range(2):
        f = p.bpr(300, seed=80 + s)
        idx = sharded.route_batch(f["user_input"], W)
        for r, g in enumerate(engs):
            ix = idx[r]
            g.set_batch(f["user_input"][ix] // W, f["item_input"][ix], neg_items=f["neg_item_input"][ix], global_batch=300)
        run.step()
    for g in engs:
        g.e.flush()
    check({"P": sharded.unshard_rows([g.e.P.cpu().numpy() for g in engs], p.U),
           "R": sharded.unshard_rows([g.e.R.cpu().numpy() for g in engs], p.I),
           "Cat": engs[0].e.Cat.cpu().numpy(), "G": engs[0].e.G.cpu().numpy()})
    for g in engs:
        g.e.close()
