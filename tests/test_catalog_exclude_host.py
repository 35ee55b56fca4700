"""CPU tests of full-catalog top-K with per-user exclusion lists: the filter rule it relies on (widen K by the listed
recipes, drop them after the exact re-rank), the oracle's exclusion and full-ranking evaluation, the host CSR builder,
and the all-gather wiring of the lists in the item-sharded runner."""
import json
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest
import torch

from foodrec_b200.engine import exclusion_csr
from oracle import evaluate_oracle, synth
from oracle.catalog_filter_model import exact_topk, stream_filter
from oracle.recommender_oracle import Hyper as OHyper, OracleModel
from tests import catalog_exclude_oracle as xo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


# ---------------------------------------------------------------------------- the filter rule
def _problem(seed, n=4000, tile=64):
    rng = np.random.default_rng(seed)
    s = rng.normal(0, 1, n)
    s[rng.integers(0, n, 40)] = np.round(s[rng.integers(0, n, 40)], 1)           # exact ties among the top
    tile_of = np.arange(n) // tile
    E = np.full(n // tile + 1, 0.02)
    E[rng.integers(0, E.size)] = 0.6                                              # one tile holds a heavy recipe
    return rng, s, tile_of, E


def _unlisted_topk(s, listed, K):
    keep = np.ones(s.size, bool)
    keep[listed[(listed >= 0) & (listed < s.size)]] = False
    ids = np.nonzero(keep)[0]
    return ids[exact_topk(s[ids], K)]


def _filter_excluding(s_hat, tile_of, E, K, listed, order):
    """What the kernels do: K_eff = K + listed entries in range (duplicates counted), then drop the listed."""
    n_in = int(((listed >= 0) & (listed < s_hat.size)).sum())
    kept = stream_filter(s_hat, tile_of, E, K + n_in, tile_order=order)
    return np.setdiff1d(kept, listed)


@pytest.mark.parametrize("seed", range(8))
@pytest.mark.parametrize("lists", ["true_topk", "random", "top_half_and_junk"])
@pytest.mark.parametrize("errors", ["random", "adversarial_down", "adversarial_up", "boundary"])
def test_widened_filter_keeps_the_unlisted_topk(seed, lists, errors):
    rng, s, tile_of, E = _problem(seed)
    K = 100
    if lists == "true_topk":                  # the user has seen exactly what they would be recommended
        listed = exact_topk(s, K)
    elif lists == "random":                   # duplicates and ids the table cannot return
        listed = np.concatenate([rng.integers(0, s.size, 50), rng.integers(0, s.size, 5), [-1, -7, s.size, s.size + 3]])
        listed = np.concatenate([listed, listed[:6]])
    else:
        listed = np.concatenate([exact_topk(s, K)[::2], rng.integers(-50, s.size + 50, 30)])
    listed = listed.astype(np.int64)
    top = _unlisted_topk(s, listed, K)
    e = E[tile_of]
    if errors == "random":
        err = rng.uniform(-1, 1, s.size) * e
    elif errors == "adversarial_down":        # the unlisted top-K looks as bad as allowed, everything else as good
        err = e.copy(); err[top] = -e[top]
    elif errors == "adversarial_up":
        err = -e.copy(); err[top] = e[top]
    else:
        err = rng.choice([-1.0, 1.0], s.size) * e
    order = rng.permutation(np.unique(tile_of))
    kept = _filter_excluding(s + err, tile_of, E, K, listed, order)
    assert set(top.tolist()) <= set(kept.tolist())
    assert not np.isin(kept, listed).any()
    assert kept.size < s.size // 4


def test_filtering_with_plain_k_would_lose_the_unlisted_topk():
    """Why K is widened: when the list is the true top-K, a filter run at K keeps (almost) only listed recipes."""
    rng, s, tile_of, E = _problem(1)
    E[:] = 0.02
    K = 100
    listed = exact_topk(s, K)
    top = _unlisted_topk(s, listed, K)
    narrow = np.setdiff1d(stream_filter(s, tile_of, E, K), listed)
    assert not set(top.tolist()) <= set(narrow.tolist())
    assert set(top.tolist()) <= set(_filter_excluding(s, tile_of, E, K, listed, None).tolist())


# ---------------------------------------------------------------------------- oracle
def _oracle(U, I, D, seed):
    tb = synth.make_tables(U, I, 7, D, seed=seed)
    ic = synth.make_item_categories(I, seed=seed + 1)
    return OracleModel(tb.P, tb.R, tb.Cat, tb.G, OHyper(), dtype=np.float32), ic


def test_oracle_catalog_topk_exclude_matches_a_masked_scan():
    U, I, D, K = 12, 700, 16, 30
    om, ic = _oracle(U, I, D, seed=5)
    rng = np.random.default_rng(2)
    users = np.array([0, 3, 3, 11, 7, 5])
    base, _ = evaluate_oracle.catalog_topk(om, users, ic, K)
    excl = [base[0][:K].tolist(),                                   # the true top-K
            [],                                                     # nothing
            list(rng.integers(0, I, 40)) * 2 + [-1, I, I + 9],      # duplicates, out of range
            list(range(I - 10)),                                    # nearly the whole catalog: padded
            list(range(I)),                                         # all of it
            base[5][::3].tolist()]
    ids, sc = xo.catalog_topk_excluding(om, users, ic, K, excl)
    ids0, sc0 = xo.catalog_topk_excluding(om, users, ic, K, [[]] * len(users))
    assert np.array_equal(ids0, base)
    w = ic.astype(np.float64); w /= w.sum(1, keepdims=True)
    a, b = np.float64(om.a), np.float64(om.one_minus_a)
    P, R, Cat = (x.astype(np.float64) for x in (om.P, om.R, om.Cat))
    for r, u in enumerate(users):
        s = a * (w @ (Cat @ P[u, 0])) + b * ((R @ P[u, 1:].T) * w).sum(1)
        s[[i for i in excl[r] if 0 <= i < I]] = -np.inf
        order = np.lexsort((np.arange(I), -s))[:K]
        order = order[np.isfinite(s[order])]
        n = order.size
        assert ids[r, :n].tolist() == order.tolist(), r
        assert (ids[r, n:] == -1).all() and np.isneginf(sc[r, n:]).all()
        if n:
            assert np.abs(sc[r, :n] - s[order]).max() <= 1e-12 * np.abs(s[np.isfinite(s)]).max()
    assert (ids[3] >= 0).sum() == 10 and (ids[4] == -1).all()
    assert not np.isin(ids[0], base[0]).any() and ids[1].tolist() == base[1].tolist()


def test_oracle_excluding_the_true_topk_gives_ranks_k1_to_2k():
    U, I, D, K = 6, 900, 16, 25
    om, ic = _oracle(U, I, D, seed=8)
    users = np.arange(U)
    full, fsc = evaluate_oracle.catalog_topk(om, users, ic, 2 * K)
    ids, sc = xo.catalog_topk_excluding(om, users, ic, K, [full[r, :K] for r in range(U)])
    assert np.array_equal(ids, full[:, K:]) and np.array_equal(sc, fsc[:, K:])


@pytest.mark.parametrize("chunk", [1, 4, 32])
def test_chunked_oracle_equals_the_full_sort(chunk):
    """catalog_topk_chunked (partial selection, users in chunks) == the full lexsort of catalog_topk_excluding and
    evaluate_oracle.catalog_topk: lists, padding, and rows where every score ties (all-zero user rows).  Ids exactly;
    scores to the last bits (BLAS may sum a chunk's product in another order than the whole batch's)."""
    def same(a, b):
        assert np.array_equal(a[0], b[0]) and np.array_equal(np.isfinite(a[1]), np.isfinite(b[1]))
        f = np.isfinite(b[1])
        assert np.abs(a[1][f] - b[1][f]).max() <= 1e-14 * np.abs(b[1][f]).max()

    U, I, D, K = 12, 700, 16, 30
    om, ic = _oracle(U, I, D, seed=5)
    om.P[4] = 0                                                      # 700-way tie: lowest ids first
    om.P[9, 1:] = 0                                                  # ties within each category mask
    rng = np.random.default_rng(3)
    users = np.array([0, 3, 3, 11, 7, 5, 4, 9, 4, 9])
    excl = [[], list(range(I - 10)), list(range(I)), list(rng.integers(0, I, 40)) * 2 + [-1, I, I + 9],
            [], [], [], [], list(range(0, 60, 2)), list(range(5))]
    ids, sc = xo.catalog_topk_chunked(om, users, ic, K, excl, chunk=chunk)
    same((ids, sc), xo.catalog_topk_excluding(om, users, ic, K, excl))
    assert (ids[1] >= 0).sum() == 10 and (ids[2] == -1).all() and ids[6].tolist() == list(range(K))
    same(xo.catalog_topk_chunked(om, users, ic, K, chunk=chunk), evaluate_oracle.catalog_topk(om, users, ic, K))


def test_oracle_full_catalog_evaluation_on_the_reference_dataset():
    from foodrec_b200.data import Dataset, side_tables
    d = Dataset(os.path.join(GOLD, "ref_dataset", "toy"))
    gi = json.load(open(os.path.join(GOLD, "reference_instances.json")))
    I, U, Lb, D = 90, 14, 5, 16
    ic, _ = side_tables(gi["dish_to_category"], gi["user_to_one_hot_label"], I, U, Lb)
    tb = synth.make_tables(U, I, Lb, D, seed=17)
    om = OracleModel(tb.P, tb.R, tb.Cat, tb.G, OHyper(), dtype=np.float32)
    seen_hit = set()
    for K in (3, 10, 40):
        hits, ndcgs = xo.evaluate_full_catalog(om, d.trainMatrix, d.testRatings, K, ic)
        assert len(hits) == len(d.testRatings)
        # direct restatement: the catalog top-K with the training items (held-out item kept) excluded
        for r, user in enumerate(d.testRatings):
            h = int(d.testRatings[user][0])
            ex = [int(i) for i in d.trainMatrix.get(user, []) if int(i) != h]
            ids, _ = xo.catalog_topk_excluding(om, [int(user)], ic, K, [ex])
            pos = np.nonzero(ids[0] == h)[0]
            assert hits[r] == (1 if pos.size else 0), (K, user)
            want = np.log(2) / np.log(int(pos[0]) + 2) if pos.size else 0
            assert ndcgs[r] == pytest.approx(want, rel=0, abs=0), (K, user)
            seen_hit.add(hits[r])
    assert seen_hit == {0, 1}                 # the toy data exercises both outcomes


# ---------------------------------------------------------------------------- host CSR builder
def test_exclusion_csr_builds_and_validates():
    off, ids = exclusion_csr([[3, 1, 3], [], [7]], 3)
    assert off.tolist() == [0, 3, 3, 4] and ids.tolist() == [3, 1, 3, 7]
    assert off.dtype == np.int32 and ids.dtype == np.int32
    off2, ids2 = exclusion_csr((torch.tensor([0, 3, 3, 4]), torch.tensor([3, 1, 3, 7])), 3)
    assert off2.tolist() == off.tolist() and ids2.tolist() == ids.tolist()
    off3, ids3 = exclusion_csr((np.zeros(5, np.int64), np.zeros(0, np.int64)), 4)
    assert off3.tolist() == [0] * 5 and ids3.size == 0
    bad = [
        (np.array([0, 2, 3]), np.arange(3)),          # n+1 = 4 entries wanted
        (np.array([1, 2, 3, 3]), np.arange(3)),       # does not start at 0
        (np.array([0, 2, 1, 3]), np.arange(3)),       # decreasing
        (np.array([0, 1, 2, 2]), np.arange(3)),       # does not end at len(ids)
        (np.array([0, 1, 2, 4]), np.arange(3)),       # past the end of ids
    ]
    for o, i in bad:
        with pytest.raises(ValueError):
            exclusion_csr((o, i), 3)
    with pytest.raises(ValueError):
        exclusion_csr([[1], [2]], 3)                  # one list per query row
    with pytest.raises(ValueError):
        exclusion_csr((np.array([0, 1, 1, 1]), np.array([2 ** 31])), 3)     # not an int32
    with pytest.raises(TypeError):
        exclusion_csr((np.array([0, 1, 1, 1]), np.array([1.5])), 3)


# ---------------------------------------------------------------------------- item-sharded wiring
CATALOG_EXCLUDE_WIRING = textwrap.dedent("""
    import os, sys, torch, torch.distributed as dist
    sys.path.insert(0, "__ROOT__")
    from foodrec_b200.sharded import DistRunner
    dist.init_process_group("gloo")
    r, W, n, K, D = dist.get_rank(), dist.get_world_size(), 3, 2, 2
    lists = lambda q: [[1000 * q + 10 * j + t for t in range(j + 2 * q)] for j in range(n)]   # totals differ per rank
    calls = []
    class Stub:
        rank, world = r, W
        def catalog_query_rows(s, users):
            return torch.tensor([[10.0 * r + j] * D for j in range(n)]).view(n, 1, D)
        def catalog_local(s, allrows, K_, exclude=None):
            calls.append(exclude is not None)
            assert allrows[:, 0, 0].tolist() == [10.0 * q + j for q in range(W) for j in range(n)]
            if exclude is not None:               # the gathered rows' lists, in rank order, as one CSR
                off, ids = exclude
                want = [l for q in range(W) for l in lists(q)]
                assert off.tolist() == [0] + [sum(len(l) for l in want[:k + 1]) for k in range(W * n)], off
                assert ids.tolist() == [x for l in want for x in l], ids
            ids = torch.tensor([[1000 * r + int(v), 1000 * r + int(v) + 500] for v in allrows[:, 0, 0]], dtype=torch.int32)
            return ids, ids.double() + 0.25
        def catalog_merge(s, ids, sc):
            for w in range(W):
                assert ids[w, :, 0].tolist() == [1000 * w + 10 * r + j for j in range(n)], ids
            return "merged"
    run = DistRunner(Stub())
    assert run.catalog_topk(None, K=K, exclude=lists(r)) == "merged"
    assert run.catalog_topk(None, K=K) == "merged"
    assert calls == [True, False]
    sys.stdout.write("EXCLUDE_WIRING_OK_%d\\n" % r); sys.stdout.flush()
""")


def test_dist_runner_catalog_exclusion_wiring_gloo_world2(tmp_path):
    """Per-user lists travel with the query rows: lengths and ids all-gathered, one CSR over the W*n rows."""
    script = tmp_path / "exclude_wiring.py"
    script.write_text(CATALOG_EXCLUDE_WIRING.replace("__ROOT__", ROOT))
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29657", str(script)],
                         capture_output=True, text=True, timeout=300, env=env)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert out.stdout.count("EXCLUDE_WIRING_OK_") == 2, out.stdout
