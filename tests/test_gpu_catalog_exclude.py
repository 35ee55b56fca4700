"""GPU tests of full-catalog top-K with per-user exclusion lists (fr_catalog_topk_excluding) against
tests/catalog_exclude_oracle.py: ids exact, fp64 scores to summation-order rounding; empty lists
reproduce fr_catalog_topk bit for bit; heavy lists take the exact fallback; recipe shards take global lists."""
import json
import os

import numpy as np
import pytest
import torch

from foodrec_b200.engine import exclusion_csr
from oracle import evaluate_oracle, synth
from oracle.recommender_oracle import Hyper as OHyper, OracleModel
from tests import catalog_exclude_oracle as xo
from tests.util import Problem, args_ns

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def make(U, I, D, seed, item_cats=None, tables=None, **prep):
    from foodrec_b200 import Engine, Hyper
    tb = tables if tables is not None else synth.make_tables(U, I, 7, D, seed=seed)
    ic = synth.make_item_categories(I, seed=seed + 1) if item_cats is None else item_cats
    e = Engine(Hyper(), tb.P, tb.R, tb.Cat, tb.G, max_rows=256, item_cats=ic)
    e.catalog_prepare(**prep)
    om = OracleModel(tb.P, tb.R, tb.Cat, tb.G, OHyper(), dtype=np.float32)
    return e, om, ic


def check(e, om, ic, K, excl, users=None, U=None, rel=1e-12):
    ids, sc = e.catalog_topk(users=users, n_users=U, K=K, exclude=excl)
    ids, sc = ids.cpu().numpy(), sc.cpu().numpy()
    uu = np.arange(U) if users is None else np.asarray(users)
    rid, rsc = xo.catalog_topk_excluding(om, uu, ic, K, excl)
    assert np.array_equal(ids, rid), f"{int((ids != rid).sum())} of {ids.size} ids differ"
    fin = np.isfinite(rsc)
    assert np.array_equal(fin, np.isfinite(sc))
    if fin.any():
        assert np.abs(sc[fin] - rsc[fin]).max() <= rel * np.abs(rsc[fin]).max()
    return ids, sc


def random_lists(rng, n, I, lo=0, hi=60):
    """0..60 entries per row: recipes of the catalog, duplicates, and ids no table row has."""
    out = []
    for _ in range(n):
        k = int(rng.integers(lo, hi + 1))
        x = rng.integers(0, I, k).tolist()
        if k > 4:
            x += x[:3]                                       # duplicates
            x += [int(rng.integers(I, 2 * I)), -1 - int(rng.integers(0, 100))]
        out.append([int(v) for v in x[:hi]])
    return out


GRID = [
    (300, 3000, 64, 10, {}),
    (300, 5000, 128, 100, {}),
    (260, 4000, 200, 50, {}),
    (700, 9000, 128, 50, dict(splits=1)),
    (1000, 20000, 128, 100, dict(splits=3)),
    (300, 5000, 128, 100, dict(cta_group=1)),
    (300, 5000, 128, 100, dict(epi_sets=2)),
    (300, 5000, 128, 100, dict(epi_sets=4, tile_n=128)),
    (300, 5000, 128, 100, dict(a_split=1)),
    (129, 257, 128, 128, dict(splits=1)),
    (200, 3000, 256, 20, {}),
    (200, 3000, 8, 20, {}),
    (300, 30000, 128, 256, dict(splits=1)),
]


@pytest.mark.parametrize("U,I,D,K,prep", GRID)
def test_empty_lists_are_bit_identical_to_the_plain_call(U, I, D, K, prep):
    e, om, ic = make(U, I, D, seed=31 + U + I, **prep)
    ids, sc = e.catalog_topk(K=K)
    ids, sc = ids.clone(), sc.clone()
    fb = e.catalog_fallback_rows()
    ids2, sc2 = e.catalog_topk(K=K, exclude=(np.zeros(U + 1, np.int32), np.zeros(0, np.int32)))
    assert torch.equal(ids, ids2) and torch.equal(sc, sc2)
    assert e.catalog_fallback_rows() == fb
    e.close()


@pytest.mark.parametrize("U,I,D,K,prep", [
    (300, 5000, 128, 10, {}),
    (300, 5000, 128, 60, dict(cta_group=1)),
    (700, 9000, 128, 50, dict(splits=1)),
    (1000, 20000, 128, 30, dict(splits=3)),
    (300, 5000, 128, 40, dict(epi_sets=4, tile_n=128)),
    (260, 4000, 200, 50, {}),
])
def test_random_lists_match_the_oracle(U, I, D, K, prep):
    e, om, ic = make(U, I, D, seed=7 + U + I, **prep)
    rng = np.random.default_rng(U + K)
    excl = random_lists(rng, U, I)
    check(e, om, ic, K, excl, U=U)
    assert e.catalog_fallback_rows() == 0                   # K + |list| <= 128 everywhere: the filter handled every row
    e.close()


@pytest.mark.parametrize("K,prep", [(50, {}), (100, dict(splits=1)), (20, dict(epi_sets=2))])
def test_excluding_the_users_own_topk_returns_ranks_k1_to_2k(K, prep):
    U, I, D = 200, 6000, 128
    e, om, ic = make(U, I, D, seed=5, **prep)
    full, fsc = evaluate_oracle.catalog_topk(om, np.arange(U), ic, 2 * K)
    ids, sc = e.catalog_topk(K=K, exclude=[full[r, :K][::-1] for r in range(U)])      # any order
    assert np.array_equal(ids.cpu().numpy(), full[:, K:])
    assert np.abs(sc.cpu().numpy() - fsc[:, K:]).max() <= 1e-12 * np.abs(fsc).max()
    e.close()


def test_long_lists_take_the_exact_fallback():
    """K + |list in this table| > 256: flagged to the exact path up front, answer correct, row counted."""
    U, I, D, K = 64, 5000, 64, 40
    e, om, ic = make(U, I, D, seed=12)
    rng = np.random.default_rng(4)
    excl = random_lists(rng, U, I, 0, 40)
    heavy = [3, 17, 40]
    for r in heavy:
        excl[r] = rng.permutation(I)[:400].tolist() + [I + 5] * 50      # 400 in the table (+ ignored ids)
    excl[50] = rng.integers(0, I, 100).tolist()                          # K + 100 <= 256: still the filter
    check(e, om, ic, K, excl, U=U)
    assert e.catalog_fallback_rows() == len(heavy)
    e.close()


def test_lists_covering_almost_the_whole_catalog_pad_with_minus_one():
    U, I, D, K = 16, 3000, 64, 30
    e, om, ic = make(U, I, D, seed=13)
    rng = np.random.default_rng(1)
    excl = [rng.permutation(I)[:I - r].tolist() for r in range(U)]     # row r keeps r recipes
    ids, sc = check(e, om, ic, K, excl, U=U)
    for r in range(U):
        assert (ids[r, :r] >= 0).all() and (ids[r, r:] == -1).all() and np.isneginf(sc[r, r:]).all()
    e.close()


def test_all_equal_scores_return_the_next_lowest_ids():
    U, I, D, K = 40, 3000, 64, 100
    tb = synth.make_tables(U, I, 7, D, seed=3)
    tb.P[:] = 0
    e, om, ic = make(U, I, D, seed=2, tables=tb)
    excl = [list(range(r)) + list(range(r, 2 * r, 2)) for r in range(U)]     # the lowest ids, some of the next
    ids, sc = e.catalog_topk(K=K, exclude=excl)
    for r in range(U):
        want = np.setdiff1d(np.arange(I), excl[r])[:K]
        assert ids[r].cpu().numpy().tolist() == want.tolist(), r
    assert float(sc.abs().max()) == 0.0
    e.close()


def test_health_blend_with_lists_matches_the_oracle():
    from foodrec_b200 import Engine, Hyper
    from oracle.recommender_oracle import health_rows
    p = Problem(300, 4000, 9, 128, seed=44)
    alpha = 0.35
    e = Engine(Hyper(alpha=alpha), p.tb.P, p.tb.R, p.tb.Cat, p.tb.G * 5, max_rows=256, item_cats=p.item_cats,
               user_labels=p.user_labels)
    G = (p.tb.G * 5).astype(np.float32)
    om = OracleModel(health_rows(p.tb.P, G, p.user_labels, alpha), p.tb.R, p.tb.Cat, G, OHyper(alpha=alpha), dtype=np.float32)
    e.set_health_blend(True)
    excl = random_lists(np.random.default_rng(8), p.U, p.I)
    check(e, om, p.item_cats, 20, excl, U=p.U)
    e.close()


def test_dense_query_rows_with_lists_equal_the_users_path():
    U, I, D, K = 500, 4000, 128, 30
    e, om, ic = make(U, I, D, seed=12)
    users = np.array([7, 7, 499, 0, 123, 321, 7], np.int32)
    excl = random_lists(np.random.default_rng(2), len(users), I)
    ids, sc = check(e, om, ic, K, excl, users=users)
    rows = e.P[torch.as_tensor(users.astype(np.int64), device=e.device)]
    off, xi = (torch.as_tensor(x).cuda() for x in exclusion_csr(excl, len(users)))
    ids2, sc2 = e.catalog_topk(P_rows=rows, K=K, exclude=(off, xi))                      # device CSR
    assert np.array_equal(ids2.cpu().numpy(), ids) and np.array_equal(sc2.cpu().numpy(), sc)
    e.close()


def test_recipe_shards_with_global_lists_merge_to_the_unsharded_answer():
    from foodrec_b200 import Engine, Hyper
    U, I, D, K, W = 200, 6001, 128, 50, 3
    e, om, ic = make(U, I, D, seed=21)
    excl = random_lists(np.random.default_rng(6), U, I)
    excl[0] = list(range(0, 150))        # K_eff = 200 unsharded, 100 on every shard: both sides take the filter path
    # (a row the exact fallback ranks sums its fp64 score in another order: same ids, scores equal to rounding only)
    ids, sc = e.catalog_topk(K=K, exclude=excl)
    parts_i, parts_s = [], []
    for r in range(W):
        sel = np.arange(r, I, W)
        es = Engine(Hyper(), om.P, om.R[sel], om.Cat, om.G, max_rows=256, item_cats=ic[sel])
        li, ls = es.catalog_topk(K=K, id_mul=W, id_add=r, exclude=excl)
        parts_i.append(li.clone()); parts_s.append(ls.clone())
        torch.cuda.synchronize()
        es.close()
    mi, ms = e.catalog_merge(torch.stack(parts_i), torch.stack(parts_s))
    assert torch.equal(mi, ids) and torch.equal(ms, sc)
    e.close()


@pytest.mark.parametrize("W", [2, 3])
def test_local_runner_with_lists_equals_unsharded(W):
    from foodrec_b200 import Engine, Hyper, sharded
    p = Problem(300, 4001, 9, 128, seed=17)
    K, n = 40, 24
    single = Engine(Hyper(), p.tb.P, p.tb.R, p.tb.Cat, p.tb.G, max_rows=256, item_cats=p.item_cats)
    engs = [sharded.ShardedEngine(Hyper(), sharded.shard_rows(p.tb.P, r, W), sharded.shard_rows(p.tb.R, r, W),
                                  p.tb.Cat, p.tb.G, r, W, max_rows=256, item_cats_global=p.item_cats)
            for r in range(W)]
    for g in engs:
        g.catalog_prepare()
    rng = np.random.default_rng(3)
    local_users = [rng.integers(0, len(range(r, p.U, W)), n).astype(np.int32) for r in range(W)]
    excl = [random_lists(rng, n, p.I) for _ in range(W)]
    outs = sharded.LocalRunner(engs).catalog_topk(local_users, K=K, exclude=excl)
    for r in range(W):
        gu = local_users[r].astype(np.int64) * W + r
        ids, sc = single.catalog_topk(users=gu.astype(np.int32), K=K, exclude=excl[r])
        assert torch.equal(outs[r][0], ids) and torch.equal(outs[r][1], sc), r
        assert not any(np.isin(outs[r][0][j].cpu().numpy(), excl[r][j]).any() for j in range(n))


def test_full_catalog_evaluation_through_model_matches_the_oracle():
    from foodrec_b200 import Model, evaluate_full_catalog
    from foodrec_b200.data import Dataset
    d = Dataset(os.path.join(GOLD, "ref_dataset", "toy"))
    gi = json.load(open(os.path.join(GOLD, "reference_instances.json")))
    p = Problem(14, 90, 5, 16, seed=17)
    m = Model(args_ns(p), p.tb.P, p.tb.R, p.tb.Cat, p.tb.G)
    from foodrec_b200.data import side_tables
    ic, _ = side_tables(gi["dish_to_category"], gi["user_to_one_hot_label"], 90, 14, 5)
    om = OracleModel(p.tb.P, p.tb.R, p.tb.Cat, p.tb.G, OHyper(), dtype=np.float32)
    for K in (3, 10, 40):
        hits, ndcgs = evaluate_full_catalog(None, m, d.trainMatrix, d.testRatings, K, gi["dish_to_category"])
        rh, rn = xo.evaluate_full_catalog(om, d.trainMatrix, d.testRatings, K, ic)
        assert hits == rh and ndcgs == rn, K
    m.engine.close()


def test_cfg2_with_zipf_histories_matches_the_oracle():
    """cfg2 in full (1M users x 200k recipes, D=128), K=100, every user excluding a Zipf(1.05) history of 20-50
    recipes: 256 sampled users equal the oracle, and no row needs the exact fallback."""
    from foodrec_b200 import Engine, Hyper
    U, I, D, K = 1_000_000, 200_000, 128, 100
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev); g.manual_seed(77)
    P = torch.randn((U, 5, D), generator=g, device=dev) * 0.1
    R = torch.randn((I, D), generator=g, device=dev) * 0.1
    Cat = torch.randn((4, D), generator=g, device=dev) * 0.1
    ic = synth.make_item_categories(I, seed=5)
    e = Engine(Hyper(), P, R, Cat, torch.zeros((7, 5, D)), max_rows=256, item_cats=ic, adopt=True)
    rng = np.random.default_rng(9)
    lens = rng.integers(20, 51, U)
    off = np.zeros(U + 1, np.int64); off[1:] = np.cumsum(lens)
    xi = synth.zipf_items(rng, I, int(off[-1])).astype(np.int32)
    ids, sc = e.catalog_topk(n_users=U, K=K, exclude=(off.astype(np.int32), xi))
    torch.cuda.synchronize()
    assert e.catalog_fallback_rows() == 0
    sample = np.sort(rng.choice(U, 256, replace=False))
    ts = torch.as_tensor(sample).to(dev)
    om = OracleModel(e.P[ts].cpu().numpy(), e.R.cpu().numpy(), e.Cat.cpu().numpy(), np.zeros((7, 5, D), np.float32),
                     OHyper(), dtype=np.float32)
    rid, rsc = xo.catalog_topk_excluding(om, np.arange(len(sample)), ic, K,
                                         [xi[off[u]:off[u + 1]] for u in sample])
    got_i, got_s = ids[ts].cpu().numpy(), sc[ts].cpu().numpy()
    assert np.array_equal(got_i, rid), f"{int((got_i != rid).sum())} ids differ"
    assert np.abs(got_s - rsc).max() <= 1e-12 * np.abs(rsc).max()
    e.close()
