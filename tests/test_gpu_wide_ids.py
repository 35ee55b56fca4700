"""The radix sort, and every step that sorts, at id widths that take three or four passes.

The suite's other cases sort keys of at most 20 bits: one or two passes.  Here:

1. ``fr_sort_pairs`` at 21-32 bits (3 and 4 passes), fused and separate offset scans, key patterns that a wrong
   pass would still turn into a valid permutation, and one sort whose offset scan has more than 4096 blocks -- each
   equal to ``np.argsort(kind="stable")`` bit for bit, with the library's launch count pinned to the restatement in
   tests/test_wide_ids_host.py.
2. The single-GPU step at wide user / recipe ids.  The step depends on ids only through their order: a warp owns 32
   consecutive sorted rows and crossing runs are summed piece by piece in chunk order, so a monotone map of the ids
   leaves every summation order unchanged.  An engine on the wide tables must therefore equal, bit for bit, an engine
   on the compact tables (the batches' rows gathered in id order, sorted in one or two passes), which is checked
   against the fp64 oracle; untouched wide rows keep their initial bits.
3. The row-sharded step and sharded evaluation at the per-rank widths of the 8-GPU legs (23-bit local users, 24-bit
   owner-major recipe keys, 21-bit serve keys), against a run on owner-preserving compact shards.
"""
import numpy as np
import pytest
import torch

from foodrec_b200 import sharded
from oracle.recommender_oracle import Hyper as OHyper, OracleModel
from tests.test_wide_ids_host import (BIG_N, BIG_NBITS, LABEL_CASE_D, SHARD_B, SHARD_IG, SHARD_MAX_ROWS, SHARD_UG,
                                      SHARD_W, SORT_N, SORT_NBITS, SORT_PATTERNS, STEP_CASES, adversarial_ids,
                                      plan_digits, shard_rows_per_rank, sort_launches)
from tests.util import assert_close, assert_close_adam

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")


def cats_of(ids):
    """A deterministic dish_to_category row per recipe id: one or two of the four categories."""
    ids = np.asarray(ids, np.int64)
    c = np.zeros((ids.size, 4), np.float32)
    first = ids % 4
    c[np.arange(ids.size), first] = 1.0
    two = (ids // 4) % 3 == 0
    c[np.arange(ids.size)[two], ((first + 1 + (ids // 12) % 3) % 4)[two]] = 1.0
    return c


def labels_of(users, L):
    """Two distinct health labels per user id (dense [n, L] multi-hot)."""
    users = np.asarray(users, np.int64)
    l1 = users % L
    l2 = (l1 + 1 + (users // L) % (L - 1)) % L
    out = np.zeros((users.size, L), np.float32)
    out[np.arange(users.size), l1] = 1.0
    out[np.arange(users.size), l2] = 1.0
    return out


def dev_tables(U, I, L, D, seed):
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    P = torch.randn((U, 5, D), device=DEV, generator=g) * 0.1
    R = torch.randn((I, D), device=DEV, generator=g) * 0.1
    Cat = torch.randn((4, D), device=DEV, generator=g) * 0.1
    G = torch.randn((L, 5, D), device=DEV, generator=g) * 0.1
    return P, R, Cat, G


def bits_equal(a, b):
    return torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


# ============================================================================================ 1. fr_sort_pairs
@pytest.fixture(scope="module")
def sorter():
    """An engine whose sort workspace holds 2^25 + 2,049 keys (about 6 GB at D = 4)."""
    from foodrec_b200 import Engine, Hyper
    z = np.zeros
    e = Engine(Hyper(learner="sgd"), z((4, 5, 4), np.float32), z((4, 4), np.float32), z((4, 4), np.float32),
               z((1, 5, 4), np.float32), max_rows=BIG_N, max_label_entries=1)
    yield e
    e.close()


def sort_keys(pattern, nbits, n, rng):
    d = plan_digits(nbits)
    top = 1 << nbits
    shifts = np.cumsum((0,) + d[:-1])
    if pattern == "uniform":
        return rng.integers(0, top, n, dtype=np.uint64)
    if pattern == "all_equal":
        return np.full(n, int(rng.integers(0, top)), np.uint64)
    if pattern in ("top_digit", "bottom_digit", "middle_digit"):
        p = {"top_digit": len(d) - 1, "bottom_digit": 0, "middle_digit": 1}[pattern]
        mask = ((1 << d[p]) - 1) << int(shifts[p])
        base = int(rng.integers(0, top)) & ~mask
        return (base | (rng.integers(0, 1 << d[p], n, dtype=np.uint64) << np.uint64(shifts[p]))).astype(np.uint64)
    if pattern == "high_bit":        # keys >= 2^31 (at 32 bits), mixed with a few low ones
        k = rng.integers(0, top, n, dtype=np.uint64)
        if nbits == 32:
            k[rng.random(n) < 0.9] |= np.uint64(1 << 31)
        return k
    if pattern == "descending_dups":  # 37 distinct keys spread over every digit, heavy duplicates, descending
        vals = np.sort(rng.integers(0, top, 37, dtype=np.uint64))[::-1]
        return np.repeat(vals, -(-n // 37))[:n].copy()
    raise ValueError(pattern)


def check_sort(e, keys, nbits):
    n = keys.size
    before = e.lib.fr_launch_count()
    ok, oi = e.sort_pairs(keys, nbits)
    launches = e.lib.fr_launch_count() - before
    assert launches == sort_launches(n, nbits), (n, nbits, launches)
    order = np.argsort(keys.astype(np.uint32), kind="stable")
    np.testing.assert_array_equal(oi, order.astype(np.uint32))
    np.testing.assert_array_equal(ok, keys.astype(np.uint32)[order])


@pytest.mark.parametrize("n", SORT_N)
@pytest.mark.parametrize("nbits", SORT_NBITS)
def test_sort_pairs_three_and_four_passes(sorter, nbits, n):
    rng = np.random.default_rng(nbits * 1_000_003 + n)
    for pattern in SORT_PATTERNS:
        if pattern == "high_bit" and nbits != 32:
            continue
        keys = sort_keys(pattern, nbits, n, rng)
        assert int(keys.max()) < (1 << nbits)
        check_sort(sorter, keys, nbits)


def test_sort_pairs_more_than_4096_scan_blocks(sorter):
    rng = np.random.default_rng(25)
    keys = rng.integers(0, 1 << BIG_NBITS, BIG_N, dtype=np.uint64)
    keys[rng.random(BIG_N) < 0.2] = 12345          # long runs of one key across tiles: stability at scale
    check_sort(sorter, keys, BIG_NBITS)


# ============================================================================================ 2. single-GPU step
def step_feeds(case, steps, seed):
    """Wide-id batches: users and recipes from adversarial_ids (the side with one pass gets the patterns too)."""
    c = STEP_CASES[case]
    B, bpr, L = c["B"], c["bpr"], c["L"]
    out = []
    for s in range(steps):
        rng = np.random.default_rng(seed + s)
        users, _, _ = adversarial_ids(c["U"], rng, B, hot_rows=600 if not bpr else 300)
        n_it = 2 * B if bpr else B
        items, _, _ = adversarial_ids(c["I"], rng, n_it, hot_rows=600)
        f = dict(users=users, ulab=labels_of(users, L))
        if bpr:
            pos, neg = items[:B], items[B:]
            neg = np.where(neg == pos, (neg + 1) % c["I"], neg)
            f.update(items=pos, neg=neg, cats=cats_of(pos), neg_cats=cats_of(neg))
        else:
            lab = (rng.random(B) < 0.5).astype(np.float32)
            ws = (np.where(lab > 0, 1.0, -1.0) * rng.uniform(0.5, 1.5, B)).astype(np.float32)
            f.update(items=items, cats=cats_of(items), labels=lab, ws=ws)
        out.append(f)
    return out


def run_engine(e, f, personal):
    if "neg" in f:
        e.train_step(f["users"], f["items"], categories=f["cats"], neg_items=f["neg"], neg_categories=f["neg_cats"],
                     user_one_hot_label=f["ulab"], write_personal=personal)
    else:
        e.train_step(f["users"], f["items"], labels=f["labels"], categories=f["cats"], write_sign=f["ws"],
                     user_one_hot_label=f["ulab"], write_personal=personal)
    return e.read_scalars().copy()


def run_oracle(om, f, personal):
    feed = dict(user_input=f["users"], item_input=f["items"], categories=f["cats"], user_one_hot_label=f["ulab"])
    if "neg" in f:
        feed.update(neg_item_input=f["neg"], neg_categories=f["neg_cats"])
        return om.train_step_bpr(feed, write_personal=personal)
    feed.update(labels=f["labels"], write_sign=f["ws"].reshape(-1, 1))
    return om.train_step(feed, write_personal=personal)


def check_oracle_scalars(v, o, om, personal, what):
    assert v[0] == pytest.approx(float(o["loss"]), rel=1e-5), f"{what}: loss"
    assert v[1] == pytest.approx(float(o["norm"]), rel=1e-5), f"{what}: norm"
    assert v[2] == pytest.approx(float(o["scale"]), rel=1e-5), f"{what}: scale"
    assert v[3] == pytest.approx(float(o["general"]), rel=1e-5, abs=1e-5 * float(np.abs(om.G).mean())), f"{what}: general"
    if personal:
        assert abs(v[4] - float(o["personal"])) <= 1e-5 * float(np.abs(om.P).mean()), f"{what}: personal"


def check_tables(t, om, om32, what):
    for k in ("P", "R", "Cat", "G"):
        if om32 is not None and k != "G":
            assert_close_adam(t[k], getattr(om, k), getattr(om32, k), what=f"{what} {k}")
        else:
            assert_close(t[k], getattr(om, k), what=f"{what} {k}")


STEP_RUNS = [
    ("a", "adam", "lazy", True, 0.01, ()),          # single-pass
    ("a", "adam", "lazy", False, 0.01, ()),         # two-pass
    ("b", "adagrad", "dense", None, 0.05, (1,)),    # step 1 writes Personal_Memory
    ("b", "rmsprop", "dense", None, 0.001, (1,)),
    ("b", "sgd", "dense", None, 0.5, (1,)),
    ("c", "adam", "lazy_exact", True, 0.01, ()),
    ("c", "sgd", "dense", None, 0.5, ()),
]


@pytest.mark.parametrize("case,learner,adam_mode,single_pass,lr,personal_steps", STEP_RUNS)
def test_wide_id_step_equals_narrow_id_step(case, learner, adam_mode, single_pass, lr, personal_steps):
    from foodrec_b200 import Engine, Hyper
    c = STEP_CASES[case]
    U, I, L, D, B, bpr = c["U"], c["I"], c["L"], c["D"], c["B"], c["bpr"]
    S = 2 * B if bpr else B
    feeds = step_feeds(case, 3, seed=100 * ord(case))
    uu = np.unique(np.concatenate([f["users"] for f in feeds]))
    ui = np.unique(np.concatenate([np.concatenate([f["items"], f.get("neg", f["items"])]) for f in feeds]))
    compact = lambda f: {k: (np.searchsorted(uu, v) if k == "users" else np.searchsorted(ui, v) if k in ("items", "neg")
                             else v) for k, v in f.items()}
    P, R, Cat, G = dev_tables(U, I, L, D, seed=ord(case))
    tu, ti = torch.as_tensor(uu, device=DEV).long(), torch.as_tensor(ui, device=DEV).long()
    P0, R0 = P.clone(), R.clone()
    Pc, Rc = P[tu].clone(), R[ti].clone()
    om = OracleModel(Pc.cpu().numpy(), Rc.cpu().numpy(), Cat.cpu().numpy(), G.cpu().numpy(), OHyper(learner=learner, lr=lr),
                     dtype=np.float64)
    om32 = OracleModel(Pc.cpu().numpy(), Rc.cpu().numpy(), Cat.cpu().numpy(), G.cpu().numpy(),
                       OHyper(learner=learner, lr=lr), dtype=np.float32) if learner == "adam" else None
    mk = lambda P_, R_: Engine(Hyper(learner=learner, lr=lr), P_, R_, Cat.clone(), G.clone(), max_rows=S,
                               max_label_entries=S * L, adam_mode=adam_mode, adopt=True, single_pass=single_pass)
    ew, ec = mk(P, R), mk(Pc, Rc)
    assert ew.single_pass == ec.single_pass == (learner == "adam" and bool(single_pass))
    what = f"case {case} {learner}/{adam_mode} sp={single_pass}"
    for s, f in enumerate(feeds):
        personal = s in personal_steps
        fc = compact(f)
        vw, vc = run_engine(ew, f, personal), run_engine(ec, fc, personal)
        # every scalar but `personal` (the mean over ALL of Personal_Memory, which the compact table does not hold)
        np.testing.assert_array_equal(np.delete(vw, 4), np.delete(vc, 4), err_msg=f"{what} step {s}: scalars")
        assert int(vc[6]) == len(np.unique(fc["users"]))
        o = run_oracle(om, fc, personal)
        if om32 is not None:
            run_oracle(om32, fc, personal)
        check_oracle_scalars(vc, o, om, personal, f"{what} step {s}")
    torch.cuda.synchronize()
    if learner == "adam":                     # stamps (and where the single-pass step left each row) before any flush
        assert torch.equal(ew.last_P[tu], ec.last_P), f"{what}: last_P"
        assert torch.equal(ew.last_R[ti], ec.last_R), f"{what}: last_R"
    ew.flush(); ec.flush()
    assert bits_equal(ew.P[tu], ec.P), f"{what}: P"
    assert bits_equal(ew.R[ti], ec.R), f"{what}: R"
    assert bits_equal(ew.Cat, ec.Cat) and bits_equal(ew.G, ec.G), f"{what}: Cat / G"
    for slots_w, slots_c in ((ew.s1, ec.s1), (ew.s2, ec.s2)):
        for k in slots_w:
            idx = tu if k == "P" else ti if k == "R" else slice(None)
            assert bits_equal(slots_w[k][idx], slots_c[k]), f"{what}: slot {k}"
    mu = torch.ones(U, dtype=torch.bool, device=DEV); mu[tu] = False
    mi = torch.ones(I, dtype=torch.bool, device=DEV); mi[ti] = False
    assert bits_equal(ew.P[mu], P0[mu]), f"{what}: an untouched Personal_Memory row changed"
    assert bits_equal(ew.R[mi], R0[mi]), f"{what}: an untouched Recipe_Embedding row changed"
    # the readers at the top ids: score and sampled evaluation, wide against compact
    rng = np.random.default_rng(5)
    qu = np.concatenate([uu[-8:], uu[:4], rng.choice(uu, 52)])
    qi = np.concatenate([ui[-8:], ui[:4], rng.choice(ui, 52)])
    cu, ci = np.searchsorted(uu, qu), np.searchsorted(ui, qi)
    assert bits_equal(ew.score(qu, qi, cats_of(qi)), ec.score(cu, ci, cats_of(qi))), f"{what}: score"
    cand = np.stack([np.roll(qi, k) for k in range(51)], 1)
    nc = np.full(qu.size, 51, np.int32)
    nc[:3] = [1, 20, 50]
    cc = cats_of(cand.reshape(-1)).reshape(cand.shape + (4,))
    iw, rw, sw = ew.eval_sampled_topk(qu, cand, nc, 10, cand_cats=cc, return_scores=True)
    ic_, rc_, sc_ = ec.eval_sampled_topk(cu, np.searchsorted(ui, cand), nc, 10, cand_cats=cc, return_scores=True)
    icn = ic_.cpu().numpy()
    np.testing.assert_array_equal(iw.cpu().numpy(), np.where(icn >= 0, ui[np.maximum(icn, 0)], icn), err_msg=f"{what}: top-K ids")
    assert torch.equal(rw, rc_) and bits_equal(sw, sc_), f"{what}: gt_rank / scores"
    check_tables(ec.tables(), om, om32, what)
    ew.close(); ec.close()


def test_two_pass_label_sort_with_device_count():
    """1,100 health labels (11-bit keys: two passes) with more than 32,768 label entries: the General_Memory label
    sort takes its key count from the device and runs the separate offset scan."""
    from foodrec_b200 import Engine, Hyper
    c = STEP_CASES["d"]
    U, I, L, D, B = c["U"], c["I"], c["L"], c["D"], c["B"]
    rng = np.random.default_rng(1100)
    P, R, Cat, G = (t.cpu().numpy() for t in dev_tables(U, I, L, D, seed=11))
    # a label pool against LSD sorting of 6 + 5 bits: top digit only, bottom digit only, 0 and L - 1
    pool = np.unique(np.concatenate([7 | (np.arange(0, 18) << 6), (9 << 6) | np.arange(64), [0, L - 1],
                                     rng.integers(0, L, 200)]))
    pool = pool[pool < L]
    om = OracleModel(P, R, Cat, G, OHyper(learner="sgd", lr=0.5), dtype=np.float64)
    e = Engine(Hyper(learner="sgd", lr=0.5), P, R, Cat, G, max_rows=B, max_label_entries=LABEL_CASE_D["max_label_entries"])
    for s in range(3):
        users, _, _ = adversarial_ids(U, rng, B, hot_rows=600)
        items, _, _ = adversarial_ids(I, rng, B, hot_rows=600)
        ulab = np.zeros((B, L), np.float32)
        for r in range(B):
            ulab[r, rng.choice(pool, LABEL_CASE_D["labels_per_row"], replace=False)] = 1.0
        ulab[rng.random(B) < 0.3, L - 1] = 1.0                  # one label in a third of the rows: a long run
        lab = (rng.random(B) < 0.5).astype(np.float32)
        ws = (np.where(lab > 0, 1.0, -1.0) * rng.uniform(0.5, 1.5, B)).astype(np.float32)
        f = dict(users=users, items=items, cats=cats_of(items), ulab=ulab, labels=lab, ws=ws)
        v = run_engine(e, f, False)
        assert int(v[8]) == int(ulab.sum()) > 32_768
        check_oracle_scalars(v, run_oracle(om, f, False), om, False, f"labels step {s}")
    check_tables(e.tables(), om, None, "labels")
    e.close()


# ============================================================================================ 3. row-sharded step
def shard_count(n, r, W=SHARD_W):
    return len(range(r, n, W))


def label_csr(global_users, L):
    """The resident CSR of labels_of: two sorted labels per row."""
    u = np.asarray(global_users, np.int64)
    l1 = u % L
    l2 = (l1 + 1 + (u // L) % (L - 1)) % L
    idx = np.sort(np.stack([l1, l2], 1), axis=1).reshape(-1).astype(np.int32)
    return np.arange(0, 2 * u.size + 1, 2, dtype=np.int32), idx


def build_shards(P_loc, R_loc, Cat, G, user_of_row, ic_global, learner, adam_mode, lr, single_pass, U_global, cap, L):
    """user_of_row[r]: the (wide) global user whose labels local row k of rank r carries."""
    from foodrec_b200 import Hyper
    W = SHARD_W
    return [sharded.ShardedEngine(Hyper(learner=learner, lr=lr), P_loc[r], R_loc[r], Cat.clone(), G.clone(), r, W,
                                  max_rows=SHARD_MAX_ROWS, cap=cap, adam_mode=adam_mode, item_cats_global=ic_global,
                                  user_label_csr_local=label_csr(user_of_row[r], L), max_label_entries=SHARD_MAX_ROWS * 2,
                                  adopt=True, single_pass=single_pass, num_users_global=U_global) for r in range(W)]


def shard_feeds(kind_list, bpr, seed, L):
    W, uloc, ipr = SHARD_W, shard_rows_per_rank(SHARD_UG), shard_rows_per_rank(SHARD_IG)
    out = []
    for s, kind in enumerate(kind_list):
        rng = np.random.default_rng(seed + s)
        B = SHARD_B
        lu, _, _ = adversarial_ids(uloc - 1, rng, B, hot_rows=300)       # local rows every rank holds
        owner = rng.integers(0, W, B)
        if kind == "one_owner":
            owner[:] = 3
        users = lu * W + owner
        if kind != "one_owner":
            users[:2] = [SHARD_UG - 1, 0]
        n_it = 2 * B if bpr else B
        li, _, _ = adversarial_ids(ipr, rng, n_it, hot_rows=600)
        items = li * W + rng.integers(0, W, n_it)
        items[:2] = [SHARD_IG - 1, 0]
        if kind == "hot":                                             # ~90 % of the rows one recipe, top local row
            items = np.where(rng.random(n_it) < 0.9, (ipr - 2) * W + 5, items)
        f = dict(users=users.astype(np.int64), ulab=labels_of(users, L))
        if bpr:
            pos, neg = items[:B], items[B:]
            neg = np.where(neg == pos, (neg + W) % SHARD_IG, neg)
            f.update(items=pos, neg=neg)
        else:
            lab = (rng.random(B) < 0.5).astype(np.float32)
            f.update(items=items, labels=lab,
                     ws=(np.where(lab > 0, 1.0, -1.0) * rng.uniform(0.5, 1.5, B)).astype(np.float32))
        out.append(f)
    return out


def set_batches(engs, f, user_map, item_map):
    W = SHARD_W
    users, items = user_map(f["users"]), item_map(f["items"])
    neg = item_map(f["neg"]) if "neg" in f else None
    B = users.size
    for r, ix in enumerate(sharded.route_batch(users, W)):
        engs[r].set_batch(users[ix] // W, items[ix], labels=f["labels"][ix] if "labels" in f else None,
                          neg_items=None if neg is None else neg[ix], write_sign=f["ws"][ix] if "ws" in f else None,
                          global_batch=B)


SHARD_RUNS = [
    ("bpr", "adam", "lazy", True, 0.01, ["plain", "hot", "one_owner"]),
    ("pointwise", "adagrad", "dense", False, 0.05, ["plain", "plain"]),
]


@pytest.mark.parametrize("mode,learner,adam_mode,single_pass,lr,kinds", SHARD_RUNS)
def test_sharded_wide_ids_equal_compact_shards(mode, learner, adam_mode, single_pass, lr, kinds):
    from foodrec_b200 import Engine, Hyper
    W, L, D = SHARD_W, 9, 4
    bpr = mode == "bpr"
    uloc, ipr = shard_rows_per_rank(SHARD_UG), shard_rows_per_rank(SHARD_IG)
    feeds = shard_feeds(kinds, bpr, seed=700 if bpr else 800, L=L)
    # wide shards, built on the device; padding rows of the last user shards are zero, as shard_rows pads them
    g = torch.Generator(device=DEV); g.manual_seed(31)
    P_w = [torch.randn((uloc, 5, D), device=DEV, generator=g) * 0.1 for _ in range(W)]
    R_w = [torch.randn((ipr, D), device=DEV, generator=g) * 0.1 for _ in range(W)]
    for r in range(W):
        P_w[r][shard_count(SHARD_UG, r):] = 0
    Cat = torch.randn((4, D), device=DEV, generator=g) * 0.1
    G = torch.randn((L, 5, D), device=DEV, generator=g) * 0.1
    P_w0, R_w0 = [t.clone() for t in P_w], [t.clone() for t in R_w]
    # owner-preserving monotone compaction: touched local row k of owner o -> compact global id k * W + o
    all_u = np.unique(np.concatenate([f["users"] for f in feeds]))
    all_i = np.unique(np.concatenate([np.concatenate([f["items"], f.get("neg", f["items"])]) for f in feeds]))
    lu = [all_u[all_u % W == o] // W for o in range(W)]
    li = [all_i[all_i % W == o] // W for o in range(W)]
    mu, mi = max(len(x) for x in lu), max(len(x) for x in li)
    UC, IC = W * mu, W * mi
    cap = min(int(1.1 * SHARD_MAX_ROWS / W) + 256, mi)     # the same request blocks on both runs

    def cmap(loc):
        def f(ids):
            ids = np.asarray(ids, np.int64)
            o = ids % W
            k = np.empty_like(ids)
            for r in range(W):
                m = o == r
                k[m] = np.searchsorted(loc[r], ids[m] // W)
            return k * W + o
        return f
    umap, imap = cmap(lu), cmap(li)

    def gather_rows(tabs, loc, m):
        out = []
        for r in range(W):
            t = torch.zeros((m,) + tuple(tabs[r].shape[1:]), device=DEV)
            t[:len(loc[r])] = tabs[r][torch.as_tensor(loc[r], device=DEV).long()]
            out.append(t)
        return out
    P_c, R_c = gather_rows(P_w, lu, mu), gather_rows(R_w, li, mi)
    wide_u = [np.concatenate([lu[r] * W + r, np.zeros(mu - len(lu[r]), np.int64)]) for r in range(W)]
    ic_c = np.zeros((IC, 4), np.float32)
    for r in range(W):
        ic_c[np.arange(len(li[r])) * W + r] = cats_of(li[r] * W + r)
    # the oracle on the compact global tables
    Pg_c = np.zeros((UC, 5, D), np.float32); Rg_c = np.zeros((IC, D), np.float32)
    for r in range(W):
        Pg_c[r::W] = P_c[r].cpu().numpy(); Rg_c[r::W] = R_c[r].cpu().numpy()
    oh = OHyper(learner=learner, lr=lr)
    om = OracleModel(Pg_c, Rg_c, Cat.cpu().numpy(), G.cpu().numpy(), oh, dtype=np.float64)
    om32 = OracleModel(Pg_c, Rg_c, Cat.cpu().numpy(), G.cpu().numpy(), oh, dtype=np.float32) if learner == "adam" else None

    ic_w = cats_of(np.arange(SHARD_IG))
    ew = build_shards(P_w, R_w, Cat, G, [np.arange(r, W * uloc, W) for r in range(W)], ic_w, learner, adam_mode, lr,
                      single_pass, SHARD_UG, cap, L)
    ec = build_shards(P_c, R_c, Cat, G, wide_u, ic_c, learner, adam_mode, lr, single_pass, UC, cap, L)
    rw, rc = sharded.LocalRunner(ew), sharded.LocalRunner(ec)
    ident = lambda x: np.asarray(x, np.int64)
    what = f"sharded {mode} {learner}/{adam_mode} sp={single_pass}"
    set_batches(ew, feeds[0], ident, ident)
    set_batches(ec, feeds[0], umap, imap)
    for s, f in enumerate(feeds):
        ahead = s == 0 and len(feeds) > 1              # the next step's plan + request exchange under this step
        ow = [o.cpu().numpy().copy() for o in rw.step(plan_ahead=(lambda: set_batches(ew, feeds[1], ident, ident)) if ahead else None)]
        oc = [o.cpu().numpy().copy() for o in rc.step(plan_ahead=(lambda: set_batches(ec, feeds[1], umap, imap)) if ahead else None)]
        for r in range(W):
            assert ow[r][9] == 0, f"{what} step {s}: rank {r} overflow flag {ow[r][9]}"
            np.testing.assert_array_equal(ow[r], oc[r], err_msg=f"{what} step {s}: rank {r} scalars")
        fo = dict(user_input=umap(f["users"]), item_input=imap(f["items"]), categories=cats_of(f["items"]),
                  user_one_hot_label=f["ulab"])
        if bpr:
            fo.update(neg_item_input=imap(f["neg"]), neg_categories=cats_of(f["neg"]))
            o = om.train_step_bpr(fo)
            if om32 is not None:
                om32.train_step_bpr(fo)
        else:
            fo.update(labels=f["labels"], write_sign=f["ws"].reshape(-1, 1))
            o = om.train_step(fo)
        v = oc[0]
        assert v[0] == pytest.approx(float(o["loss"]), rel=1e-5), f"{what} step {s}: loss"
        assert v[1] == pytest.approx(float(o["norm"]), rel=1e-5), f"{what} step {s}: norm"
        assert v[3] == pytest.approx(float(o["general"]), rel=1e-5, abs=1e-5 * float(np.abs(om.G).mean())), f"{what}: general"
        if s + 1 < len(feeds) and not ahead:
            set_batches(ew, feeds[s + 1], ident, ident)
            set_batches(ec, feeds[s + 1], umap, imap)
        if kinds[s] == "one_owner":
            assert [len(ix) > 0 for ix in sharded.route_batch(f["users"], W)] == [r == 3 for r in range(W)]
    torch.cuda.synchronize()
    for r in range(W):
        a, b = ew[r].e, ec[r].e
        tu = torch.as_tensor(lu[r], device=DEV).long(); nu = len(lu[r])
        ti = torch.as_tensor(li[r], device=DEV).long(); ni = len(li[r])
        if learner == "adam":
            assert torch.equal(a.last_P[tu], b.last_P[:nu]) and torch.equal(a.last_R[ti], b.last_R[:ni]), f"{what}: rank {r} stamps"
        a.flush(); b.flush()
        assert bits_equal(a.P[tu], b.P[:nu]) and bits_equal(a.R[ti], b.R[:ni]), f"{what}: rank {r} rows"
        assert bits_equal(a.Cat, b.Cat) and bits_equal(a.G, b.G), f"{what}: rank {r} Cat / G"
        for sw, sc in ((a.s1, b.s1), (a.s2, b.s2)):
            for k in sw:
                if k == "P":
                    ok = bits_equal(sw[k][tu], sc[k][:nu])
                elif k == "R":
                    ok = bits_equal(sw[k][ti], sc[k][:ni])
                else:
                    ok = bits_equal(sw[k], sc[k])
                assert ok, f"{what}: rank {r} slot {k}"
        keep_u = torch.ones(uloc, dtype=torch.bool, device=DEV); keep_u[tu] = False
        keep_i = torch.ones(ipr, dtype=torch.bool, device=DEV); keep_i[ti] = False
        assert bits_equal(a.P[keep_u], P_w0[r][keep_u]), f"{what}: rank {r} an untouched user row changed"
        assert bits_equal(a.R[keep_i], R_w0[r][keep_i]), f"{what}: rank {r} an untouched recipe row changed"
    # the compact run against the oracle
    ts = [g_.e.tables() for g_ in ec]
    got = {"P": sharded.unshard_rows([t["P"] for t in ts], UC), "R": sharded.unshard_rows([t["R"] for t in ts], IC),
           "Cat": ts[0]["Cat"], "G": ts[0]["G"]}
    check_tables(got, om, om32, what)
    for g_ in ec:
        g_.e.close()
    del ec, P_c, R_c, P_w0, R_w0
    # sampled evaluation at the wide ids against one engine on the same global tables
    Pg = torch.zeros((SHARD_UG, 5, D), device=DEV); Rg = torch.zeros((SHARD_IG, D), device=DEV)
    for r in range(W):
        Pg[r::W] = ew[r].e.P[:shard_count(SHARD_UG, r)]
        Rg[r::W] = ew[r].e.R[:shard_count(SHARD_IG, r)]
    single = Engine(Hyper(learner="sgd"), Pg, Rg, ew[0].e.Cat.clone(), ew[0].e.G.clone(), max_rows=256,
                    max_label_entries=256, item_cats=ic_w, adopt=True)
    rng = np.random.default_rng(3)
    parts = []
    for r in range(W):
        nl = shard_count(SHARD_UG, r)
        u = np.concatenate([[uloc - 1, nl - 1, 0], lu[r][-20:], rng.integers(0, nl, 40)]).astype(np.int32)
        top = np.concatenate([[SHARD_IG - 1 - k for k in range(8)], (ipr - 1) * W + np.arange(W)])
        cand = rng.integers(0, SHARD_IG, (u.size, 51))
        cand[:, :top.size] = top[None, :]
        cand[::2] = cand[::2, ::-1]
        nc = np.full(u.size, 51, np.int32)
        parts.append((u, cand.astype(np.int32), nc))
    dev32 = lambda x: torch.as_tensor(np.asarray(x, np.int32), device=DEV)
    outs = rw.eval_sampled_topk([dev32(u) for u, _, _ in parts], [dev32(c) for _, c, _ in parts],
                                [nc for _, _, nc in parts], 10, return_scores=True)
    for r, ((u, c, nc), (ids, rank, sc)) in enumerate(zip(parts, outs)):
        nl = shard_count(SHARD_UG, r)
        gu = np.where(u < nl, u.astype(np.int64) * W + r, -1)
        ids1, rank1, sc1 = single.eval_sampled_topk(dev32(gu), dev32(c), nc, 10, return_scores=True)
        assert torch.equal(ids, ids1), f"{what}: eval rank {r} ids"
        assert torch.equal(rank, rank1), f"{what}: eval rank {r} gt_rank"
        assert bits_equal(sc, sc1), f"{what}: eval rank {r} scores"
    single.close()
    for g_ in ew:
        g_.e.close()
