"""CPU tests of full-ranking evaluation on row-sharded tables: the rounds, padding and exclusion lists of
``LocalRunner`` / ``DistRunner.full_ranking`` on stub engines with recognisable payloads (in process, and with a
world_size-2 gloo group), and ``evaluate_full_catalog_sharded`` over stub engines whose catalog is
tests/catalog_exclude_oracle.py, against that file's ``evaluate_full_catalog``."""
import json
import os
import subprocess
import sys
import textwrap
import types

import numpy as np
import pytest
import torch

from foodrec_b200 import _lib as L
from foodrec_b200 import evaluate_full_catalog_sharded, sharded
from oracle import synth
from oracle.recommender_oracle import Hyper as OHyper, OracleModel
from tests import catalog_exclude_oracle as xo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


# ---------------------------------------------------------------------------- recording stubs
# Rank q holds ROWS local rows (the last one of rank 1 is the padding row of the last user shard).  Its test user at
# local row k holds out HELD(q, k) and trained on HIST(q, k): row 0's list is not empty (so a padding row, which must get
# an empty list, differs from a real user at row 0), row 2's is empty, row 1 lists the held-out recipe twice and rows
# k % 3 == 0 once.  Every shard answers the query row (q, k) with a list holding HELD(q, k) at WANT(q, k) (absent at -1).
ROWS, K, RN = 10, 4, 2


def HELD(q, k):
    return 5000 + 100 * q + k


def HIST(q, k):
    if k == 1:
        return [HELD(q, k), 5, HELD(q, k)]
    if k == 2:
        return []
    return [100 * q + 10 * k + t for t in range(1 + k % 4)] + ([HELD(q, k)] if k % 3 == 0 else [])


def WANT(q, k):
    return k % (K + 1) - 1


def hist_csr(q):
    rows = [HIST(q, k) for k in range(ROWS)]
    off = np.zeros(ROWS + 1, np.int32)
    off[1:] = np.cumsum([len(r) for r in rows])
    return off, np.asarray([x for r in rows for x in r], np.int32)


class RecordingShard:
    """The catalog phases of one rank on CPU tensors: a query row carries 100 * rank + local row; catalog_local checks
    the gathered rows and lists of the round against ``users`` (every rank's test users, known to every stub)."""
    device = "cpu"

    def __init__(self, rank, world, users, history_set=True):
        self.rank, self.world, self.users = rank, world, users
        self.U_valid = ROWS - (1 if rank == 1 else 0)
        self.e = types.SimpleNamespace(U=ROWS, _history=tuple(torch.as_tensor(x) for x in hist_csr(rank))
                                       if history_set else None)
        self.rn = max(1, min(RN, max(len(u) for u in users)))        # the round size every rank agrees on
        self.rounds = 0
        self.queried = []

    def catalog_query_rows(self, users_local):
        u = torch.as_tensor(users_local).long()
        self.queried.append(u.tolist())
        return (100.0 * self.rank + u.double()).view(-1, 1, 1)

    def catalog_local(self, allrows, K_, exclude=None):
        a, rn = self.rounds, self.rn
        self.rounds += 1
        want_rows, want_lists = [], []
        for q, us in enumerate(self.users):
            part = [int(x) for x in us[a * rn:(a + 1) * rn]]
            want_rows += [(q, k) for k in part] + [(q, 0)] * (rn - len(part))          # padding: local row 0
            want_lists += [[x for x in HIST(q, k) if x != HELD(q, k)] for k in part] + [[]] * (rn - len(part))
        assert K_ == K and allrows.shape == (len(want_rows), 1, 1)
        assert allrows.view(-1).tolist() == [100.0 * q + k for q, k in want_rows], (a, allrows.view(-1))
        off, ids = (torch.as_tensor(x) for x in exclude)
        got = [ids[off[j]:off[j + 1]].tolist() for j in range(len(want_rows))]
        assert got == want_lists, (a, got, want_lists)
        out = torch.full((len(want_rows), K), -1, dtype=torch.int32)
        for j, (q, k) in enumerate(want_rows):
            out[j] = torch.arange(9000, 9000 + K, dtype=torch.int32)
            if WANT(q, k) >= 0:
                out[j, WANT(q, k)] = HELD(q, k)
        return out, -out.double()

    def catalog_merge(self, ids, sc):              # every shard gave the same list for my users
        assert all(torch.equal(ids[w], ids[0]) for w in range(ids.shape[0]))
        return ids[0], sc[0]


def expected_positions(users):
    return [[WANT(q, int(k)) for k in us] for q, us in enumerate(users)]


# unequal counts, a rank with none, several rounds (RN = 2): every rank walks ceil(max / 2) rounds
CASES = [[[3, 1, 0, 7, 2], [4, 8]], [[0, 6, 9], []], [[], [2, 0, 1, 3]], [[1], [5]]]


@pytest.mark.parametrize("users", CASES)
@pytest.mark.parametrize("given", [True, False])
def test_local_runner_rounds_padding_lists_positions(users, given):
    engs = [RecordingShard(q, 2, users, history_set=not given) for q in range(2)]
    run = sharded.LocalRunner(engs)
    hist = [hist_csr(q) for q in range(2)] if given else None
    pos = run.full_ranking([np.asarray(u, np.int32) for u in users], [[HELD(q, k) for k in u] for q, u in enumerate(users)],
                           K, history=hist, round_users=RN)
    rn = engs[0].rn
    rounds = -(-max(len(u) for u in users) // rn)
    assert all(g.rounds == rounds for g in engs)
    assert [p.tolist() for p in pos] == expected_positions(users)
    assert all(p.dtype == torch.int32 for p in pos)
    for q, g in enumerate(engs):                   # the query rows of each round: own users, then local row 0
        assert g.queried == [(users[q][a * rn:(a + 1) * rn] + [0] * rn)[:rn] for a in range(rounds)]


def test_local_runner_raises_before_any_round():
    users = [[3, 1], [8, 9]]                       # local row 9 of rank 1 is the padding row of the last user shard
    engs = [RecordingShard(q, 2, users) for q in range(2)]
    held = [[HELD(q, k) for k in u] for q, u in enumerate(users)]
    with pytest.raises(IndexError):
        sharded.LocalRunner(engs).full_ranking(users, held, K, round_users=RN)
    with pytest.raises(IndexError):
        sharded.LocalRunner(engs).full_ranking([[3, -1], [8]], [held[0], held[1][:1]], K, round_users=RN)
    engs = [RecordingShard(q, 2, [[3], []], history_set=(q == 0)) for q in range(2)]
    with pytest.raises(L.FoodRecError, match="history"):       # a rank without a history, even one without users
        sharded.LocalRunner(engs).full_ranking([[3], []], [[HELD(0, 3)], []], K)
    assert all(g.rounds == 0 and not g.queried for g in engs)
    with pytest.raises(ValueError):
        sharded.LocalRunner(engs).full_ranking([[3], []], [[1, 2], []], K, history=[hist_csr(0), hist_csr(1)])


def test_round_lists_remove_every_occurrence_of_the_held_out_recipe():
    off, ids = (torch.as_tensor(x) for x in hist_csr(0))
    u = torch.tensor([1, 2, 3, 6, 1], dtype=torch.int64)
    h = torch.tensor([HELD(0, 1), 7, HELD(0, 3), -1, 5], dtype=torch.int64)      # user 1 again, holding out 5
    uu, (xoff, xid) = sharded._round_lists(u, h, (off, ids), 0, 5, 7)
    assert uu.tolist() == [1, 2, 3, 6, 1, 0, 0] and uu.dtype == torch.int32
    want = [[5], [], HIST(0, 3)[:-1], HIST(0, 6), [HELD(0, 1), HELD(0, 1)], [], []]
    assert [xid[xoff[j]:xoff[j + 1]].tolist() for j in range(7)] == want
    assert xoff.dtype == torch.int32 and xid.dtype == torch.int32


# ---------------------------------------------------------------------------- gloo world 2
WIRING = textwrap.dedent("""
    import sys, torch, torch.distributed as dist
    sys.path.insert(0, "__ROOT__")
    from foodrec_b200 import _lib as L
    from foodrec_b200.sharded import DistRunner
    from tests.test_full_ranking_sharded_host import CASES, HELD, K, RN, RecordingShard, expected_positions, hist_csr
    dist.init_process_group("gloo")
    r, W = dist.get_rank(), dist.get_world_size()
    for users in CASES:
        for given in (True, False):
            g = RecordingShard(r, W, users, history_set=not given)
            pos = DistRunner(g).full_ranking(torch.tensor(users[r], dtype=torch.int32), [HELD(r, k) for k in users[r]], K,
                                             history=hist_csr(r) if given else None, round_users=RN)
            assert g.rounds == -(-max(len(u) for u in users) // g.rn), (users, g.rounds)
            assert pos.tolist() == expected_positions(users)[r] and pos.dtype == torch.int32, (users, pos)
    # the padding row of rank 1's shard, and a rank without a history: both ranks raise, before any catalog round
    for users, hist_on in (([[3], [9]], (True, True)), ([[3], []], (True, False))):
        g = RecordingShard(r, W, users, history_set=hist_on[r])
        try:
            DistRunner(g).full_ranking(users[r], [HELD(r, k) for k in users[r]], K, round_users=RN)
            raise SystemExit("no error")
        except (IndexError, L.FoodRecError) as ex:
            assert isinstance(ex, IndexError if hist_on[1] else L.FoodRecError), ex
        assert g.rounds == 0 and not g.queried
    sys.stdout.write("FULL_RANKING_WIRING_OK_%d\\n" % r); sys.stdout.flush()
""")


def test_dist_runner_full_ranking_wiring_gloo_world2(tmp_path):
    """One all-reduce agrees on rounds and errors; per round catalog_topk's all-gather carries the padded rows and
    their lists in rank order; positions come from the merged lists of the rank's own users."""
    script = tmp_path / "full_ranking_wiring.py"
    script.write_text(WIRING.replace("__ROOT__", ROOT))
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29661", str(script)],
                         capture_output=True, text=True, timeout=300, env=env)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert out.stdout.count("FULL_RANKING_WIRING_OK_") == 2, out.stdout


# ---------------------------------------------------------------------------- against the oracle
class OracleShard:
    """Recipe shard ``rank`` (recipe i on rank i % W) of the oracle's catalog on CPU tensors: a query row carries its
    global user, the shard's top-K is catalog_exclude_oracle's with the other shards' recipes and the recipes without a
    category left out (the kernels never return those), and the merge is the (score desc, id asc) top-K of the lists."""
    device = "cpu"

    def __init__(self, om, ic, rank, world, U):
        self.om, self.ic, self.rank, self.world = om, ic, rank, world
        self.U_global = U
        self.U_valid = len(range(rank, U, world))
        self.e = types.SimpleNamespace(U=sharded.local_rows(U, world), _history=None)

    def catalog_query_rows(self, users_local):
        return (torch.as_tensor(users_local).long() * self.world + self.rank).double().view(-1, 1, 1)

    def catalog_local(self, allrows, K_, exclude=None):
        I = self.ic.shape[0]
        skip = np.nonzero((np.arange(I) % self.world != self.rank) | (self.ic.sum(1) == 0))[0]
        off, ids = (np.asarray(x) for x in exclude)
        lists = [np.concatenate([ids[off[j]:off[j + 1]], skip]) for j in range(allrows.shape[0])]
        with np.errstate(invalid="ignore"):              # (recipes without a category score NaN there: left out)
            i, s = xo.catalog_topk_excluding(self.om, allrows.view(-1).long().numpy(), self.ic, K_, lists)
        return torch.as_tensor(i, dtype=torch.int32), torch.as_tensor(s)

    def catalog_merge(self, ids, sc):
        W, n, K_ = ids.shape
        i = ids.permute(1, 0, 2).reshape(n, W * K_).numpy().astype(np.int64)
        s = sc.permute(1, 0, 2).reshape(n, W * K_).numpy()
        out_i, out_s = np.full((n, K_), -1, np.int64), np.full((n, K_), -np.inf)
        for j in range(n):
            live = np.nonzero(i[j] >= 0)[0]
            o = live[np.lexsort((i[j, live], -s[j, live]))][:K_]
            out_i[j, :o.size], out_s[j, :o.size] = i[j, o], s[j, o]
        return torch.as_tensor(out_i, dtype=torch.int32), torch.as_tensor(out_s)


def oracle_runner(U, I, D, W, seed, ic=None):
    tb = synth.make_tables(U, I, 7, D, seed=seed)
    ic = synth.make_item_categories(I, seed=seed + 1) if ic is None else ic
    om = OracleModel(tb.P, tb.R, tb.Cat, tb.G, OHyper(), dtype=np.float32)
    return sharded.LocalRunner([OracleShard(om, ic, r, W, U) for r in range(W)]), om, ic


@pytest.mark.parametrize("W", [1, 2, 3])
@pytest.mark.parametrize("K", [1, 5, 30])
def test_evaluate_full_catalog_sharded_equals_the_oracle_on_the_reference_dataset(W, K):
    from foodrec_b200.data import Dataset, side_tables
    d = Dataset(os.path.join(GOLD, "ref_dataset", "toy"))
    gi = json.load(open(os.path.join(GOLD, "reference_instances.json")))
    ic, _ = side_tables(gi["dish_to_category"], gi["user_to_one_hot_label"], 90, 14, 5)
    run, om, ic = oracle_runner(14, 90, 16, W, seed=17, ic=ic)
    want = xo.evaluate_full_catalog(om, d.trainMatrix, d.testRatings, K, ic)
    assert evaluate_full_catalog_sharded(run, d.trainMatrix, d.testRatings, K) == want
    assert evaluate_full_catalog_sharded(run, d.trainMatrix, d.testRatings, K, round_users=2) == want


@pytest.mark.parametrize("W", [2, 3])
def test_evaluate_full_catalog_sharded_edge_cases_equal_the_oracle(W):
    """Held-out recipes without a category, past the catalog and in the padding of the last recipe shard; one listed
    twice in the history; empty and absent histories; a global CSR for trainMatrix; a rank with few test users."""
    U, I, D, K = 23, 301, 16, 20                    # 301 recipes: the last recipe shard has padding at W = 2 and 3
    rng = np.random.default_rng(W)
    ic = synth.make_item_categories(I, seed=4)
    dead = rng.choice(I, 15, replace=False)
    ic[dead] = 0
    run, om, ic = oracle_runner(U, I, D, W, seed=9, ic=ic)
    train = {str(u): [int(x) for x in rng.integers(0, I, int(rng.integers(0, 40)))] for u in range(U) if u % 5}
    test = {str(u): [int(rng.integers(0, I))] for u in range(U) if u % W != 1 or u in (1, 3)}
    with np.errstate(invalid="ignore"):
        S = np.nan_to_num(xo.catalog_scores(om, np.arange(U), ic), nan=-np.inf)
    for u in range(0, U, 2):                                              # hits: a held-out recipe among the user's best
        if str(u) in test:
            test[str(u)] = [int(np.argsort(-S[u])[rng.integers(0, 12)])]
    test["0"] = [int(dead[0])]                                            # no category
    train["2"] = [test["2"][0]] * 2 + train["2"]                          # held out, and trained on twice
    train["8"] = []                                                       # empty; users 0, 15 and 20 have none at all
    train["12"] = [int(x) for x in np.argsort(-ic.sum(1))[:200]]          # most of the catalog
    outside = {"3": [I + 7], "6": [I]}                                    # past the catalog / in the last shard's padding
    for k in outside:
        test.pop(k)
    want = xo.evaluate_full_catalog(om, train, test, K, ic)
    both = dict(test, **outside)
    got = evaluate_full_catalog_sharded(run, train, both, K, round_users=3)
    keys = list(both)
    assert [got[0][keys.index(k)] for k in test] == want[0] and [got[1][keys.index(k)] for k in test] == want[1]
    assert all(got[0][keys.index(k)] == 0 and got[1][keys.index(k)] == 0 for k in outside)
    assert sum(want[0]) > 0 and want[0][list(test).index("0")] == 0
    off = np.zeros(U + 1, np.int64)
    off[1:] = np.cumsum([len(train.get(str(u), [])) for u in range(U)])
    csr = (off, np.asarray([x for u in range(U) for x in train.get(str(u), [])], np.int64))
    assert evaluate_full_catalog_sharded(run, csr, test, K) == want
    assert all(g.e._history is None for g in run.engs)                   # nothing was set on the engines
    with pytest.raises(IndexError):                                       # a test user past the users
        evaluate_full_catalog_sharded(run, train, dict(test, **{str(U): [1]}), K)
    with pytest.raises(ValueError):
        evaluate_full_catalog_sharded(run, train, dict(test, **{"5": []}), K)
