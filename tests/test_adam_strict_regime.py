"""The well-conditioned Adam regime that tests/test_gpu_adam_strict.py holds every Adam path to, checked on the oracles.

At the TF default adam_eps = 1e-8 the quotient m / (sqrt(v) + eps) is ill-conditioned wherever a summed gradient cancels
to near eps: there the float32 oracle itself misses the float64 one by more than 1e-5, so the Adam table checks at that
eps go through tests/util.py:assert_close_adam, which excuses such rows, lets 0.1 % of entries fail and caps the worst
error only at a multiple of the float32 oracle's worst deviation.  With eps large against the fp32 noise of the summed
gradients the quotient is well conditioned and every entry can be held to the plain 1e-5 rule (assert_close).

This file keeps the schedules of the strict GPU tests, rehearses each one's regime guard on the oracles alone (so an eps
can be chosen without a GPU), and pins the gap the strict rule closes: errors of the size a kernel bug makes that
assert_close_adam accepts at eps 1e-8 and assert_close rejects in the strict regime."""
import numpy as np
import pytest

from oracle.recommender_oracle import Hyper as OHyper
from tests.util import Problem, assert_close, assert_close_adam

GUARD = 4e-6            # float32 vs float64 oracle, every entry, of max(|ref|, rms): 2.5x inside the 1e-5 bound
GAPS = (1, 2, 7, 33, 100)
GROUP = 16              # users (and recipes) per gap group
ALWAYS = 40             # users (and recipes) in every batch


def rel_dev(x, ref):
    """Worst |x - ref| over max(|ref|, rms(ref)): the measure assert_close holds to 1e-5."""
    x = np.asarray(x, np.float64); ref = np.asarray(ref, np.float64)
    rms = float(np.sqrt(np.mean(ref ** 2)))
    return float((np.abs(x - ref) / np.maximum(np.abs(ref), rms)).max())


def gap_feed(p, bpr, s, seed, rows_per_user=3):
    """Step s of the gap schedule: ALWAYS users and recipes are in every batch; the GROUP users and recipes of gap k are
    in the batches of the steps s = 0 (mod k + 1) only, so they sit out exactly k steps before they return.  A group's
    users read only its own recipes, so recipe rows sit out the same gaps."""
    rng = np.random.default_rng(seed + s)
    groups = [(0, ALWAYS)] + [(ALWAYS + g * GROUP, GROUP) for g, k in enumerate(GAPS) if s % (k + 1) == 0]
    users, items = [], []
    for lo, n in groups:
        u = np.repeat(np.arange(lo, lo + n), rows_per_user)
        users.append(u); items.append(lo + rng.integers(0, n, u.size))
    users = np.concatenate(users).astype(np.int32)
    items = np.concatenate(items).astype(np.int32)
    perm = rng.permutation(users.size)
    users, items = users[perm], items[perm]
    B = users.size
    f = p.bpr(B, seed=seed + s, users=users) if bpr else p.pointwise(B, seed=seed + s, users=users)
    f["item_input"], f["categories"] = items, p.item_cats[items].reshape(B, 4, 1).copy()
    if bpr:       # the negative: another recipe of the same group
        lo = np.where(items < ALWAYS, 0, ALWAYS + (items - ALWAYS) // GROUP * GROUP)
        n = np.where(items < ALWAYS, ALWAYS, GROUP)
        neg = (lo + (items - lo + 1 + rng.integers(0, n - 1)) % n).astype(np.int32)
        f["neg_item_input"], f["neg_categories"] = neg, p.item_cats[neg].reshape(B, 4, 1).copy()
    return f


GAP_STEPS = max(GAPS) + 2           # the gap-100 group returns on the last step
PERSONAL_STEP = 50                  # a personal-write step after rows went stale (and moved to the shadow copy)


def gap_schedule(p, bpr, seed, steps=GAP_STEPS, personal=PERSONAL_STEP):
    """[(feed, write_personal)] of the gap schedule."""
    return [(gap_feed(p, bpr, s, seed), s == personal) for s in range(steps)]


def oracle_step(om, f, bpr, personal=False):
    return om.train_step_bpr(f, write_personal=personal) if bpr else om.train_step(f, write_personal=personal)


def quotient_y(om, k):
    """y = sqrt(v) / (sqrt(v) + eps) over the touched (v > 0) entries of table k."""
    q = np.sqrt(om.v[k][om.v[k] > 0])
    return q / (q + om.h.adam_eps)


def regime_guard(om, om32, what):
    """Fails as a set-up error unless (a) the float32 oracle is within GUARD of the float64 one at every entry of P, R
    and Cat -- the well-conditioned regime, where the plain 1e-5 rule holds any float32 implementation -- and (b) the
    touched entries of P and R together span the quotient (some y > 0.5, some y < 0.1), so the catch-up is exercised beyond the
    linear term of its polynomial in y.  Returns the float32 oracle's worst deviation per table."""
    eps = om.h.adam_eps
    dev = {k: rel_dev(getattr(om32, k), getattr(om, k)) for k in ("P", "R", "Cat")}
    for k, d in dev.items():
        if d > GUARD:
            pytest.fail(f"set-up: {what}: the float32 oracle is {d:.2e} off the float64 one in {k} (guard {GUARD:.0e}): "
                        f"adam_eps = {eps:g} is ill-conditioned for these gradients; raise it")
    y = np.concatenate([quotient_y(om, "P"), quotient_y(om, "R")])
    if not ((y > 0.5).any() and (y < 0.1).any()):
        pytest.fail(f"set-up: {what}: y = sqrt(v)/(sqrt(v)+eps) of P and R spans only [{y.min():.3f}, {y.max():.3f}] "
                    f"at adam_eps = {eps:g}: move eps toward the gradients' scale")
    return dev


def report(t, om, what):
    """Print the worst deviation of tables t from the float64 oracle, per table, as a fraction of the 1e-5 bound."""
    print(f"[adam strict] {what}: worst / bound " +
          " ".join(f"{k} {rel_dev(t[k], getattr(om, k)) / 1e-5:.3f}" for k in ("P", "R", "Cat", "G")))


# ---------------------------------------------------------------------------------------- the strict GPU schedules
# (lr, eps) per shape, from the guard.  The Problem shapes at lr 0.01 over ~8 steps: eps 1e-6.  Over the ~100 steps of
# the gap schedule, lr 0.01 moves slice 0 of the always-present users by ~lr per step until their gradients oscillate
# about zero, and the float32 trajectory drifts 2e-5 from the float64 one at any eps; at lr 0.001 it stays within 1.4e-6.
# The long-chain batch (16,000 rows): gradients ~ 1/B, eps scaled down with them (at lr 0.01 Adam's first steps
# move the hot user's row by ~lr and its next gradients cancel: 6e-6).
REGIME = {"gaps": (0.001, 1e-6), "clip": (0.01, 1e-6), "chain": (0.001, 1e-7)}
GAP_D = (4, 64, 128, 132, 200, 256)


def gap_problem(D):
    return Problem(403, 257, 9, D, seed=60 + D)


def clip_problem(D):
    return Problem(403, 257, 9, D, seed=11 + D, scale=6.0)


CLIP_STEPS = 12


def clip_schedule(p, bpr, seed):
    """A shorter gap schedule on tables 60x larger, clip_norm the median norm of the run: the clip is active on some
    steps; a personal-write step falls on one that clips."""
    fs = [gap_feed(p, bpr, s, seed) for s in range(CLIP_STEPS)]
    lr, eps = REGIME["clip"]
    probe = p.oracle(OHyper(learner="adam", lr=lr, adam_eps=eps, clip_norm=1e30))
    norms = [float(oracle_step(probe, f, bpr)["norm"]) for f in fs]
    clip = float(np.median(norms))
    personal = 2 + int(np.argmax(norms[2:]))
    return [(f, s == personal) for s, f in enumerate(fs)], clip


def run_oracles(p, bpr, schedule, lr, eps, clip_norm=5.0):
    oh = OHyper(learner="adam", lr=lr, adam_eps=eps, clip_norm=clip_norm)
    om, om32 = p.oracle(oh), p.oracle(oh, dtype=np.float32)
    outs = []
    for f, personal in schedule:
        outs.append(oracle_step(om, f, bpr, personal))
        oracle_step(om32, f, bpr, personal)
    return om, om32, outs


@pytest.mark.parametrize("bpr", [False, True])
@pytest.mark.parametrize("D", GAP_D)
def test_gap_schedule_regime(D, bpr):
    p = gap_problem(D)
    sched = gap_schedule(p, bpr, seed=D)
    om, om32, _ = run_oracles(p, bpr, sched, *REGIME["gaps"])
    regime_guard(om, om32, f"gaps D={D} bpr={bpr}")


@pytest.mark.parametrize("bpr,D", [(False, 132), (True, 256)])
def test_clip_schedule_regime(bpr, D):
    p = clip_problem(D)
    sched, clip = clip_schedule(p, bpr, seed=90)
    om, om32, outs = run_oracles(p, bpr, sched, *REGIME["clip"], clip_norm=clip)
    clipped = sum(float(o["scale"]) < 1.0 for o in outs)
    assert 2 <= clipped <= CLIP_STEPS - 2, clipped
    regime_guard(om, om32, f"clip D={D} bpr={bpr}")


def chain_problem(D):
    return Problem(64, 300, 3, D, seed=D + 1)


CHAIN_STEPS = 3


def chain_schedule(p, bpr, D):
    from tests.test_gpu_scale_paths import chain_batch
    return [(chain_batch(p, bpr, seed=100 * D + s), False) for s in range(CHAIN_STEPS)]


@pytest.mark.parametrize("bpr,D", [(False, 64), (True, 200), (False, 200)])
def test_chain_schedule_regime(bpr, D):
    p = chain_problem(D)
    om, om32, _ = run_oracles(p, bpr, chain_schedule(p, bpr, D), *REGIME["chain"])
    regime_guard(om, om32, f"chain D={D} bpr={bpr}")


# ---------------------------------------------------------------------------------------- the gap the strict rule closes
def issue_run(eps, steps=8):
    """Problem(403, 257, 9, 132) over 8 pointwise steps at lr 0.01: batches of 300, every third one 16 users x 40 rows.
    Returns both oracles and the P of the float64 one before its last step."""
    p = Problem(403, 257, 9, 132, seed=7)
    oh = OHyper(learner="adam", lr=0.01, adam_eps=eps)
    om, om32 = p.oracle(oh), p.oracle(oh, dtype=np.float32)
    for s in range(steps):
        f = p.pointwise(640, seed=s, users=np.repeat(np.arange(16) * 25, 40)) if s % 3 == 2 else p.pointwise(300, seed=s)
        if s == steps - 1:
            P_before, last = om.P.copy(), f
        om.train_step(f); om32.train_step(f)
    return om, om32, P_before, last


def planted_lane_group(om32, om):
    """The float32 oracle's P with elements 128..131 (the partial last lane group at D = 132) of slice 2 of 50 users
    shifted by 1e-4 of the table's rms -- 10x the bound."""
    x = om32.P.astype(np.float64)
    rms = float(np.sqrt(np.mean(om.P ** 2)))
    x[np.arange(50) * 8, 2, 128:132] += 1e-4 * rms
    return x


def test_assert_close_adam_accepts_a_lane_group_error_at_the_default_eps():
    om, om32, _, _ = issue_run(1e-8)
    assert rel_dev(om32.P, om.P) > 1e-5             # the reason assert_close_adam exists
    assert_close_adam(planted_lane_group(om32, om), om.P, om32.P, what="planted P")


def test_strict_regime_rejects_a_lane_group_error():
    om, om32, _, _ = issue_run(REGIME["clip"][1])
    assert rel_dev(om32.P, om.P) <= GUARD
    assert_close(om32.P, om.P, what="float32 oracle P")
    with pytest.raises(AssertionError, match="entries off"):
        assert_close(planted_lane_group(om32, om), om.P, what="planted P")


def test_strict_regime_rejects_half_an_adam_step_missing():
    """Half of the last step's update undone on one user row that sat out that step (its update is the decay-only step
    a lazy catch-up applies) and on one lane group of a user in the batch: a skipped or duplicated catch-up."""
    om, om32, P_before, last = issue_run(REGIME["clip"][1])
    step = om.P - P_before
    out = np.setdiff1d(np.arange(om.P.shape[0]), last["user_input"])
    u = int(out[np.argmax(np.abs(step[out]).max(axis=(1, 2)))])
    x = om32.P.astype(np.float64)
    x[u] -= 0.5 * step[u]
    with pytest.raises(AssertionError, match="entries off"):
        assert_close(x, om.P, what="catch-up row")
    w = int(last["user_input"][0])
    x = om32.P.astype(np.float64)
    x[w, 0, 128:132] -= 0.5 * step[w, 0, 128:132]
    with pytest.raises(AssertionError, match="entries off"):
        assert_close(x, om.P, what="lane group")
