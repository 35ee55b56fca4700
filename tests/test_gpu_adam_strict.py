"""Every Adam path held to the float64 oracle by the plain 1e-5 rule (tests/util.py:assert_close) at every entry of P,
R, Cat and G, with no exemptions: dense, lazy_exact (step-by-step replay), lazy (closed-form series), the single-pass
kernel with its shadow Personal_Memory and speculative clip, the row-sharded phases and the bench's cfg2 step.

The runs use the well-conditioned regime of tests/test_adam_strict_regime.py: an adam_eps per shape at which the float32
oracle stays within 4e-6 of the float64 one, checked in each test before the kernels are (a set-up failure names the eps
to raise).  The schedules reach the Adam-only code: rows that sit out 1, 2, 7, 33 and 100 steps and return (catch-up
at several gaps, y = sqrt(v)/(sqrt(v)+eps) spread over (0, 1)), a personal-write step after rows went stale, an active
global-norm clip, and the long segment chains of tests/test_gpu_scale_paths.py."""
import numpy as np
import pytest

from foodrec_b200 import sharded
from tests.test_adam_strict_regime import (REGIME, CLIP_STEPS, chain_problem, chain_schedule, clip_problem, clip_schedule,
                                           gap_problem, gap_schedule, oracle_step, regime_guard, report)
from tests.test_gpu_real_configs import _run_cfg2
from tests.test_gpu_sharded_oracle import build, check_scalars as check_sharded_scalars, close, gather, sharded_step
from tests.test_gpu_single_pass import step
from tests.util import assert_close

pytestmark = pytest.mark.gpu


def engine(p, adam_mode, single_pass, lr, eps, max_rows=4096, **hk):
    from foodrec_b200 import Engine, Hyper
    e = Engine(Hyper(learner="adam", lr=lr, adam_eps=eps, **hk), p.tb.P, p.tb.R, p.tb.Cat, p.tb.G, max_rows=max_rows,
               adam_mode=adam_mode, max_label_entries=max_rows * p.L, single_pass=single_pass)
    assert e.single_pass == (adam_mode != "dense" and single_pass is not False)
    return e


def oracles(p, lr, eps, **hk):
    from oracle.recommender_oracle import Hyper as OHyper
    oh = OHyper(learner="adam", lr=lr, adam_eps=eps, **hk)
    return p.oracle(oh), p.oracle(oh, dtype=np.float32)


def check_scalars(v, o, om, what):
    assert v[0] == pytest.approx(float(o["loss"]), rel=1e-5), f"{what}: loss"
    assert v[1] == pytest.approx(float(o["norm"]), rel=1e-5), f"{what}: norm"
    assert v[2] == pytest.approx(float(o["scale"]), rel=1e-5), f"{what}: scale"
    assert v[3] == pytest.approx(float(o["general"]), rel=1e-5, abs=1e-5 * float(np.abs(om.G).mean())), f"{what}: general"


def run(engines, om, om32, schedule, bpr, what):
    """Every engine and both oracles through the schedule; the scalars of every step checked.  Returns the oracle outputs."""
    outs = []
    for s, (f, personal) in enumerate(schedule):
        vs = [step(e, f, bpr, personal) for e in engines]
        o = oracle_step(om, f, bpr, personal)
        oracle_step(om32, f, bpr, personal)
        for v in vs:
            check_scalars(v, o, om, f"{what} step {s}")
        outs.append(o)
    return outs


def check_strict(t, om, om32, what):
    regime_guard(om, om32, what)
    for k in ("P", "R", "Cat", "G"):
        assert_close(t[k], getattr(om, k), what=f"{what} {k}")
    report(t, om, what)


# D covers DV = 1, one lane group, the EXACT width 128, a partial last lane group, NV = 2 and the EXACT width 256;
# adam_mode x single_pass x bpr pairwise over them
GAP_CASES = [(4, "lazy", None, False), (4, "dense", None, True), (64, "lazy_exact", False, True), (64, "lazy", None, False),
             (128, "lazy_exact", None, False), (128, "lazy", False, True), (132, "lazy", None, True),
             (132, "dense", None, False), (132, "lazy_exact", False, False), (200, "lazy", False, False),
             (200, "lazy_exact", None, True), (256, "lazy", None, True), (256, "lazy_exact", False, False),
             (256, "dense", None, True)]


@pytest.mark.parametrize("D,adam_mode,single_pass,bpr", GAP_CASES)
def test_gap_schedule_matches_oracle(D, adam_mode, single_pass, bpr):
    p = gap_problem(D)
    lr, eps = REGIME["gaps"]
    e = engine(p, adam_mode, single_pass, lr, eps)
    om, om32 = oracles(p, lr, eps)
    what = f"gaps D={D} {adam_mode} sp={single_pass} bpr={bpr}"
    run([e], om, om32, gap_schedule(p, bpr, seed=D), bpr, what)
    check_strict(e.tables(), om, om32, what)
    e.close()


@pytest.mark.parametrize("D,adam_mode,bpr", [(4, "lazy", True), (64, "lazy", False), (132, "lazy", False),
                                             (200, "lazy_exact", True), (256, "lazy_exact", False)])
def test_single_pass_equals_two_pass(D, adam_mode, bpr):
    """The single-pass and the two-pass step give the same P and R bit for bit after the first step (same arithmetic,
    same summation order per row).  dCat is summed in sorted-user order instead of batch order, so Cat -- and through it
    everything else on later steps -- differs in the last bits; after the gap schedule the two agree to 2e-6 at every
    entry, as the well-conditioned quotient does not amplify that."""
    p = gap_problem(D)
    lr, eps = REGIME["gaps"]
    a, b = engine(p, adam_mode, True, lr, eps), engine(p, adam_mode, False, lr, eps)
    om, om32 = oracles(p, lr, eps)
    sched = gap_schedule(p, bpr, seed=D)
    what = f"single vs two pass D={D} {adam_mode} bpr={bpr}"
    run([a, b], om, om32, sched[:1], bpr, what)
    ta, tb = a.tables(), b.tables()
    for k in ("P", "R"):
        np.testing.assert_array_equal(ta[k], tb[k], err_msg=f"{what}: step 0 {k}")
    run([a, b], om, om32, sched[1:], bpr, what)
    ta, tb = a.tables(), b.tables()
    for k in ("P", "R", "Cat", "G"):
        assert_close(ta[k], tb[k], rtol=2e-6, what=f"{what} {k}")
    check_strict(ta, om, om32, what + " (single)")
    check_strict(tb, om, om32, what + " (two)")
    a.close(); b.close()


@pytest.mark.parametrize("D,adam_mode,single_pass,bpr", [(132, "lazy", None, False), (132, "lazy_exact", False, False),
                                                         (256, "lazy", None, True), (256, "dense", None, True)])
def test_active_clip_matches_oracle(D, adam_mode, single_pass, bpr):
    """Tables 60x larger, clip_norm the median norm of the run: the clip is active on some steps, where the single-pass
    speculation fails and the step is redone; a personal-write step falls on one that clips."""
    p = clip_problem(D)
    sched, clip = clip_schedule(p, bpr, seed=90)
    lr, eps = REGIME["clip"]
    e = engine(p, adam_mode, single_pass, lr, eps, clip_norm=clip)
    om, om32 = oracles(p, lr, eps, clip_norm=clip)
    what = f"clip D={D} {adam_mode} sp={single_pass} bpr={bpr}"
    outs = run([e], om, om32, sched, bpr, what)
    # (the seeds keep every step's norm away from the threshold, where the two sums could disagree about clipping)
    assert all(abs(float(o["norm"]) - clip) > 1e-4 * clip for o in outs)
    assert 2 <= sum(float(o["scale"]) < 1.0 for o in outs) <= CLIP_STEPS - 2
    assert float(outs[[pw for _, pw in sched].index(True)]["scale"]) < 1.0
    check_strict(e.tables(), om, om32, what)
    e.close()


@pytest.mark.parametrize("D,adam_mode,single_pass,bpr", [(64, "lazy", True, False), (200, "lazy", False, True),
                                                         (200, "lazy_exact", None, False), (200, "lazy", True, True)])
def test_long_segment_chains_match_oracle(D, adam_mode, single_pass, bpr):
    p = chain_problem(D)
    lr, eps = REGIME["chain"]
    e = engine(p, adam_mode, single_pass, lr, eps, max_rows=16384)
    om, om32 = oracles(p, lr, eps)
    what = f"chain D={D} {adam_mode} sp={single_pass} bpr={bpr}"
    run([e], om, om32, chain_schedule(p, bpr, D), bpr, what)
    check_strict(e.tables(), om, om32, what)
    e.close()


# D, W, adam_mode, single_pass, bpr, p2p
SHARDED_CASES = [(132, 2, "lazy", None, False, False), (200, 3, "lazy_exact", None, True, True),
                 (256, 8, "lazy", False, False, False), (64, 8, "lazy", None, True, False),
                 (128, 3, "lazy", None, False, False)]


@pytest.mark.parametrize("D,W,adam_mode,single_pass,bpr,p2p", SHARDED_CASES)
def test_sharded_gap_schedule_matches_oracle(D, W, adam_mode, single_pass, bpr, p2p):
    p = gap_problem(D)
    lr, eps = REGIME["gaps"]
    engs = build(p, W, "adam", adam_mode, lr=lr, single_pass=single_pass, adam_eps=eps)
    runner = sharded.LocalRunner(engs)
    if p2p:
        runner.enable_p2p()
    om, om32 = oracles(p, lr, eps)
    what = f"sharded gaps D={D} W={W} {adam_mode} sp={single_pass} bpr={bpr} p2p={p2p}"
    for s, (f, personal) in enumerate(gap_schedule(p, bpr, seed=D)):
        outs, _ = sharded_step(runner, engs, f, bpr, personal)
        o = oracle_step(om, f, bpr, personal)
        oracle_step(om32, f, bpr, personal)
        check_sharded_scalars(outs, o, om, f"{what} step {s}")
    check_strict(gather(engs, p), om, om32, what)
    close(engs)


@pytest.mark.parametrize("D,W,single_pass,bpr", [(132, 3, None, False), (256, 2, False, True)])
def test_sharded_active_clip_matches_oracle(D, W, single_pass, bpr):
    """The sharded step knows the clip scale only after the all-reduce: the user pass redoes a speculative single-pass
    update and every gradient row a rank sends is scaled before its owner applies it."""
    p = clip_problem(D)
    sched, clip = clip_schedule(p, bpr, seed=90)
    lr, eps = REGIME["clip"]
    engs = build(p, W, "adam", "lazy", lr=lr, single_pass=single_pass, adam_eps=eps, clip_norm=clip)
    runner = sharded.LocalRunner(engs)
    om, om32 = oracles(p, lr, eps, clip_norm=clip)
    what = f"sharded clip D={D} W={W} sp={single_pass} bpr={bpr}"
    clipped = 0
    for s, (f, personal) in enumerate(sched):
        outs, _ = sharded_step(runner, engs, f, bpr, personal)
        o = oracle_step(om, f, bpr, personal)
        oracle_step(om32, f, bpr, personal)
        assert abs(float(o["norm"]) - clip) > 1e-4 * clip, (s, float(o["norm"]), clip)
        check_sharded_scalars(outs, o, om, f"{what} step {s}")
        clipped += float(o["scale"]) < 1.0
    assert 2 <= clipped <= CLIP_STEPS - 2, clipped
    check_strict(gather(engs, p), om, om32, what)
    close(engs)


CFG2_EPS = 3e-8       # gradients ~ 1/B at B = 262,144 and lr 0.001 (the guard checks it)


def test_cfg2_bench_batch_matches_oracle():
    """The bench's step (1M users x 200k recipes, BPR B = 262,144, two steps) in both lazy modes, every touched row of P
    and R held to the plain rule; untouched rows keep their bits."""
    _run_cfg2([("adam", "lazy_exact", 0.001), ("adam", "lazy", 0.001)], B=262_144, steps=2, seed=5, adam_eps=CFG2_EPS,
              strict=True)
