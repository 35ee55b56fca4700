"""The kernel paths that only production-sized inputs reach, against the oracle.

* Sampled evaluation (eval_sampled_kernel) runs a persistent grid whose warps rank users one after another, with the
  next user's ids and rows fetched while the current one is scored.  At a few hundred users every warp ranks at most
  one, so here every warp ranks at least six, in each of the 16 instantiations (NV x SLOTS x bf16 x EXACT).
* The inference kernel (fwd_score_kernel) carries the current user's row across its 8-row blocks and, above
  8 x 8 warps x 8 CTAs per SM rows, across grid-stride iterations.
* The training step hands a crossing run of more than FR_LONG_CHAIN (16) pieces to seg_combine_long_kernel: recipe runs
  of more than 16 chunks of 32 rows, label runs of more than 16 tiles of 256 entries.  The batches below put runs at
  exactly 16 and 17 pieces, start one at lane 31 (first piece in slot 1) and chain long runs on consecutive ids."""
import numpy as np
import pytest
import torch

from oracle import evaluate_oracle
from oracle.recommender_oracle import Hyper as OHyper, OracleModel, health_rows, round_bf16
from tests.util import Problem, assert_close, assert_close_adam

pytestmark = pytest.mark.gpu

ALPHA = 0.35            # health-blend weight, large enough to reorder rankings (with General_Memory x 5)


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def dev32(x):
    """int32 device tensor: ids passed this way skip the host range check, so the kernels' own checks are tested."""
    return torch.as_tensor(np.ascontiguousarray(x, np.int32), device="cuda")


def outside(rng, n, size):
    """n ids outside [0, size): half past the end, half negative."""
    return np.where(rng.random(n) < 0.5, size + rng.integers(0, 100, n), -1 - rng.integers(0, 100, n))


def inference_setup(p, bf16, health, **hk):
    """An engine over p's tables and the fp64 oracle of what it scores: bf16 storage rounds P and R, the health
    blend scores P[u] + alpha * mean G[labels(u)] (oracle/recommender_oracle.py:health_rows)."""
    from foodrec_b200 import Engine, Hyper
    G = (p.tb.G * 5).astype(np.float32)
    e = Engine(Hyper(learner="sgd", alpha=ALPHA, **hk), p.tb.P, p.tb.R, p.tb.Cat, G, max_rows=256,
               item_cats=p.item_cats, user_labels=p.user_labels, table_dtype="bf16" if bf16 else "float32")
    P, R = (round_bf16(p.tb.P), round_bf16(p.tb.R)) if bf16 else (p.tb.P, p.tb.R)
    if health:
        e.set_health_blend(True)
        P = health_rows(P, G, p.user_labels, ALPHA)
    return e, OracleModel(P, R, p.tb.Cat, G, OHyper(alpha=ALPHA, **hk), dtype=np.float64)


# ---------------------------------------------------------------- sampled evaluation
def eval_feed(rng, n, U, I, stride):
    """n test rows: users drawn with repeats, ~2 % outside Personal_Memory; ragged n_cand (0, 1, 32, 33 and the full
    stride among them); ~1 % of candidates outside the catalog; ~1 % of lists with repeated ids."""
    users = rng.integers(0, U, n)
    bad = rng.random(n) < 0.02
    users[bad] = outside(rng, int(bad.sum()), U)
    cand = rng.integers(0, I, (n, stride))
    bad = rng.random((n, stride)) < 0.01
    cand[bad] = outside(rng, int(bad.sum()), I)
    n_cand = np.where(rng.random(n) < 0.5, rng.choice([0, 1, 32, 33, stride], n), rng.integers(0, stride + 1, n))
    for r in np.nonzero(rng.random(n) < 0.01)[0]:
        n_cand[r] = stride
        k = r % 4
        if k == 0: cand[r, rng.integers(1, stride)] = cand[r, 0]                  # the positive, again
        if k == 1: cand[r, 31] = cand[r, 2]                                       # inside slot 0
        if k == 2: cand[r, stride - 1] = cand[r, rng.integers(0, 32)]             # across slots
        if k == 3: cand[r, 40] = cand[r, 35]; cand[r, 45] = cand[r, 35]           # inside slot 1
    return users, cand, n_cand


def run_eval(e, users, cand, n_cand, K, cand_cats):
    ids, rank, sc = e.eval_sampled_topk(dev32(users), dev32(cand), dev32(n_cand), K, cand_cats=cand_cats,
                                        return_scores=True)
    torch.cuda.synchronize()
    return ids, rank, sc


def check_eval_at_scale(e, om, p, stride, K, cand_cats_given, seed, exact=False):
    n = 6 * 64 * sm_count()           # >= 6 users per warp whatever the occupancy (at most 64 warps per SM)
    rng = np.random.default_rng(seed)
    users, cand, n_cand = eval_feed(rng, n, p.U, p.I, stride)
    cc = p.item_cats[np.clip(cand, 0, p.I - 1)] if cand_cats_given else None
    ids, rank, sc = run_eval(e, users, cand, n_cand, K, cc)
    ids2, rank2, sc2 = run_eval(e, users, cand, n_cand, K, cc)
    assert torch.equal(ids, ids2) and torch.equal(rank, rank2) and torch.equal(sc, sc2), "two calls differ"
    ids, rank, sc = ids.cpu().numpy(), rank.cpu().numpy(), sc.cpu().numpy()
    valid_u = (users >= 0) & (users < p.U)
    valid_c = (cand >= 0) & (cand < p.I)
    live = valid_u[:, None] & valid_c & (np.arange(stride)[None, :] < n_cand[:, None])
    S = evaluate_oracle.catalog_scores(om, np.arange(p.U), p.item_cats)
    ref = S[np.where(valid_u, users, 0)[:, None], np.clip(cand, 0, p.I - 1)]
    assert_close(sc[live], ref[live], what="sampled-evaluation scores")
    assert (sc[~live] == 0).all(), "a score was written for a candidate that is not ranked"
    want, want_rank = evaluate_oracle.sampled_topk(ref, np.where(valid_c, cand, -1), n_cand, K + 1, valid_user=valid_u)
    # the ranking is decided unless two of the top K + 1 distinct scores lie within fp32 rounding of each other
    top = np.where(want >= 0, S[np.where(valid_u, users, 0)[:, None], np.maximum(want, 0)], np.nan)
    gap = top[:, :-1] - top[:, 1:]
    scale = np.abs(np.where(live, ref, 0)).max(1)
    close = (gap <= 1e-6 * scale[:, None]) & (want[:, 1:] >= 0)
    checked = np.ones(n, bool) if exact else ~close.any(1)      # (exact: integer scores, ties are ties in fp32 too)
    want, want_rank = want[:, :K], np.where(want_rank < K, want_rank, -1)
    bad = checked & ((ids != want).any(1) | (rank != want_rank))
    assert not bad.any(), (f"{int(bad.sum())} users ranked differently; first row {np.argmax(bad)}: got "
                           f"{ids[np.argmax(bad)].tolist()} rank {rank[np.argmax(bad)]}, want "
                           f"{want[np.argmax(bad)].tolist()} rank {want_rank[np.argmax(bad)]}")
    assert checked.mean() >= 0.95, f"only {checked.mean():.4f} of the users were checked"
    print(f"[sampled eval] {n} users, {1 - checked.mean():.5f} skipped by the gap rule")


#  D: 4, 64 (NV=1), 128 (NV=1, EXACT), 132, 200 (NV=2), 256 (NV=2, EXACT); stride 51 -> SLOTS=2, 100 -> SLOTS=4
EVAL_GRID = [(4, 51, False, False, 10), (4, 100, True, True, 130), (64, 100, False, True, 1), (64, 51, True, False, 10),
             (128, 51, False, True, 130), (128, 100, False, False, 10), (128, 51, True, False, 1),
             (128, 100, True, True, 10), (132, 51, False, False, 10), (132, 100, True, True, 1),
             (200, 100, False, True, 130), (200, 51, True, True, 10), (256, 51, False, True, 10),
             (256, 100, False, False, 130), (256, 51, True, False, 130), (256, 100, True, True, 10)]


@pytest.mark.parametrize("D,stride,bf16,health,K", EVAL_GRID)
def test_sampled_eval_at_scale_matches_oracle(D, stride, bf16, health, K):
    p = Problem(2500, 5000, 9, D, seed=D + stride)
    e, om = inference_setup(p, bf16, health)
    check_eval_at_scale(e, om, p, stride, K, cand_cats_given=(D + K) % 2 == 0, seed=D * 7 + stride)
    e.close()


@pytest.mark.parametrize("D,stride,bf16", [(256, 51, False), (256, 100, True), (64, 100, False), (128, 51, True)])
def test_sampled_eval_at_scale_dict_semantics_exact(D, stride, bf16):
    """Integer-valued scores (a = 0, one-hot recipe rows, one category per recipe): exact ties everywhere, so ids and
    ranks follow evaluate.py's dict + nlargest bit for bit for every user.  With I = D recipes a list of 100
    candidates repeats ids many times."""
    rng = np.random.default_rng(D + stride)
    p = Problem(2000, D, 3, D, seed=5)
    p.tb.P[:] = 0; p.tb.P[:, 1, :] = rng.integers(-3, 4, (p.U, D)).astype(np.float32)
    p.tb.R[:] = 0; p.tb.R[np.arange(D), np.arange(D)] = 1.0
    p.item_cats[:] = 0; p.item_cats[:, 0] = 1.0
    e, om = inference_setup(p, bf16, False, high_level_score_coefficient=0.0)
    check_eval_at_scale(e, om, p, stride, 10, cand_cats_given=False, seed=stride, exact=True)
    e.close()


# ---------------------------------------------------------------- inference
@pytest.mark.parametrize("D,health,by_item", [(4, False, False), (132, True, True), (256, True, False)])
def test_fwd_score_at_scale_matches_oracle(D, health, by_item):
    """An evaluation-style feed (51 consecutive rows per user) of >= 4 x 512 rows per SM, so every warp walks several
    8-row blocks and grid-stride iterations with the user row in registers; ~0.5 % of rows carry an id outside its
    table (device tensors: NaN score, no row read)."""
    p = Problem(2500, 5000, 9, D, seed=D)
    e, om = inference_setup(p, False, health)
    rng = np.random.default_rng(D)
    groups = -(-4 * 512 * sm_count() // 51) + 7
    users = np.repeat(rng.integers(0, p.U, groups), 51)
    items = rng.integers(0, p.I, users.size)
    bu, bi = rng.random(users.size) < 0.003, rng.random(users.size) < 0.002
    users[bu] = outside(rng, int(bu.sum()), p.U); items[bi] = outside(rng, int(bi.sum()), p.I)
    valid = ~(bu | bi)
    cats = None if by_item else torch.as_tensor(p.item_cats[np.clip(items, 0, p.I - 1)], device="cuda")
    got = e.score(dev32(users), dev32(items), cats).cpu().numpy()
    S = evaluate_oracle.catalog_scores(om, np.arange(p.U), p.item_cats)
    assert np.isnan(got[~valid]).all()
    assert_close(got[valid], S[users[valid], items[valid]], what=f"scores D={D}")
    e.close()


# ---------------------------------------------------------------- training: long segment chains
def placed_counts(rng, n_ids, total, unit, specials):
    """Rows per id such that, sorted by id, the run of each special id starts at a chosen offset within a `unit`-row
    piece and spans exactly a chosen number of pieces: specials = {id: (start offset or None, pieces)}; None starts
    the run right after the previous special id's run, inside the piece where that one ends.  Ids up to the last
    special get 0-7 rows otherwise; the rest of `total` is spread over the ids after it."""
    counts = np.zeros(n_ids, np.int64)
    pos = 0
    last = max(specials)
    for i in range(last + 1):
        if i in specials:
            off, span = specials[i]
            if off is not None:
                d = (off - pos) % unit
                assert d == 0 or (i > 0 and i - 1 not in specials)
                counts[i - 1] += d; pos += d
            end = (pos // unit + span - 1) * unit + int(rng.integers(0, unit - 1))    # never the piece's last row
            counts[i] = end - pos + 1
            pos = end + 1
        else:
            counts[i] = rng.integers(0, 8); pos += counts[i]
    assert pos <= total, (pos, total)
    counts[last + 1:] = rng.multinomial(total - pos, np.full(n_ids - last - 1, 1.0 / (n_ids - last - 1)))
    start = np.cumsum(counts) - counts
    for i, (off, span) in specials.items():        # the layout the test is about
        assert (start[i] + counts[i] - 1) // unit - start[i] // unit + 1 == span
        assert off is None or start[i] % unit == off
    return counts


# recipe pass (pieces = 32-row chunks): 16 pieces (serial combine) next to 17 (long list, first piece in slot 1 and
# sharing the boundary chunk); a long run starting at lane 31; 16 pieces from lane 31; three long runs on consecutive ids
RECIPE_RUNS = {40: (0, 16), 41: (None, 17), 100: (31, 20), 150: (31, 16), 200: (0, 18), 201: (None, 19), 202: (None, 21)}
# label pass (pieces = tiles of 8 x 32 entries): label 1 spans 16 tiles, labels 0 and 2 more than 20
LABEL_RUNS = {0: (0, 22), 1: (None, 16)}
HOT_USER, HOT_ROWS = 17, 3000          # > 90 chunks of one user (serial user-pass combine, FusedUserPol)


def chain_batch(p, bpr, seed):
    """One batch with the run layout above.  BPR: the recipe pass sorts the 2B item rows; the label pass emits one
    entry per item row, so labels are laid out per triple in half-tiles."""
    rng = np.random.default_rng(seed)
    rows = 16000
    B = rows // 2 if bpr else rows
    lab = np.repeat(np.arange(3), placed_counts(rng, 3, B, 128 if bpr else 256, LABEL_RUNS))
    assert (lab == 2).sum() > (21 * 256 if not bpr else 21 * 128)
    items = np.repeat(np.arange(p.I), placed_counts(rng, p.I, rows, 32, RECIPE_RUNS))
    items = rng.permutation(items).astype(np.int32)
    users = rng.integers(0, p.U, B).astype(np.int32)
    users[rng.permutation(B)[:HOT_ROWS]] = HOT_USER
    f = dict(user_input=users, user_one_hot_label=np.eye(3, dtype=np.float32)[rng.permutation(lab)])
    if bpr:
        pos, neg = items[:B].copy(), items[B:].copy()
        while (pos == neg).any():                               # no triple with its positive as its negative
            for c in np.nonzero(pos == neg)[0]:                 # (swaps keep the multiset of recipe rows)
                j = rng.integers(0, B)
                neg[c], neg[j] = neg[j], neg[c]
        f.update(item_input=pos, neg_item_input=neg, categories=p.item_cats[pos].reshape(B, 4, 1),
                 neg_categories=p.item_cats[neg].reshape(B, 4, 1))
    else:
        y = (rng.random(B) < 0.5).astype(np.float32)
        f.update(item_input=items, labels=y, write_sign=np.where(y > 0, 1.0, -1.0).astype(np.float32).reshape(B, 1),
                 categories=p.item_cats[items].reshape(B, 4, 1))
    return f


CHAIN_CASES = [("sgd", 0.5, "dense", None, False, 64, False), ("adagrad", 0.05, "dense", None, True, 200, False),
               ("rmsprop", 0.002, "dense", None, False, 200, False), ("adam", 0.01, "lazy", True, False, 64, False),
               ("adam", 0.01, "lazy", False, True, 200, False), ("adam", 0.01, "lazy_exact", None, False, 200, False),
               ("adam", 0.01, "lazy", True, True, 200, False), ("rmsprop", 0.002, "dense", None, True, 64, True)]


@pytest.mark.parametrize("learner,lr,adam_mode,single_pass,bpr,D,bf16", CHAIN_CASES)
def test_long_segment_chains_match_oracle(learner, lr, adam_mode, single_pass, bpr, D, bf16):
    from foodrec_b200 import Engine, Hyper
    p = Problem(64, 300, 3, D, seed=D + 1)
    e = Engine(Hyper(learner=learner, lr=lr), p.tb.P, p.tb.R, p.tb.Cat, p.tb.G, max_rows=16384,
               max_label_entries=2 * 16384, adam_mode=adam_mode, single_pass=single_pass,
               table_dtype="bf16" if bf16 else "float32")
    if single_pass is not None:
        assert e.single_pass == single_pass
    oh = OHyper(learner=learner, lr=lr)
    om = OracleModel(p.tb.P, p.tb.R, p.tb.Cat, p.tb.G, oh, dtype=np.float32 if bf16 else np.float64,
                     table_dtype="bf16" if bf16 else None)
    om32 = p.oracle(oh, dtype=np.float32) if learner == "adam" else None
    for s in range(3):
        f = chain_batch(p, bpr, seed=100 * D + s)
        kw = dict(neg_items=f["neg_item_input"], neg_categories=f["neg_categories"]) if bpr else {}
        e.train_step(f["user_input"], f["item_input"], labels=None if bpr else f["labels"], categories=f["categories"],
                     write_sign=None if bpr else f["write_sign"], user_one_hot_label=f["user_one_hot_label"], **kw)
        v = e.read_scalars()
        o = om.train_step_bpr(f) if bpr else om.train_step(f)
        if om32 is not None:
            (om32.train_step_bpr if bpr else om32.train_step)(f)
        assert v[0] == pytest.approx(o["loss"], rel=1e-5) and v[1] == pytest.approx(o["norm"], rel=1e-5), s
    t = e.tables()
    if bf16:
        from tests.test_gpu_bf16 import check_tables
        check_tables(t, om, f"bf16 {learner} D={D}")
    else:
        for k in ("P", "R", "Cat", "G"):
            if om32 is not None and k != "G":
                assert_close_adam(t[k], getattr(om, k), getattr(om32, k), what=f"{learner}/{adam_mode} {k}")
            else:
                assert_close(t[k], getattr(om, k), what=f"{learner}/{adam_mode} {k}")
    e.close()
