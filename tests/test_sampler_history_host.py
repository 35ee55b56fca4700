"""The history-aware negative sampler's definition on the CPU (tests/sampler_history_oracle.py): without a history it
is the positive-only sampler of oracle/sampler_oracle.py bit for bit, the vectorised restatement equals a literal loop
over the rule, no draw is in the user's history, and ``history_csr`` builds the CSR the library reads."""
import os

import numpy as np
import pytest

from oracle import sampler_oracle as base
from tests import sampler_history_oracle as so
from tests.sampler_history_cases import KINDS, check_rule, make_history, samples

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def test_no_or_empty_history_is_todays_sampler():
    g = np.load(os.path.join(GOLD, "negative_sampler.npz"))
    args = (g["pos"], int(g["n_neg"]), int(g["num_items"]), int(g["seed"]), int(g["offset"]))
    n = g["pos"].shape[0]
    users = np.random.default_rng(0).integers(0, 40, n)
    empty = (np.zeros(41, np.int32), np.zeros(0, np.int32))
    np.testing.assert_array_equal(so.sample_negatives(*args), g["neg"])
    np.testing.assert_array_equal(base.sample_negatives(*args), g["neg"])
    np.testing.assert_array_equal(so.sample_negatives(*args, users=users, history=empty), g["neg"])
    np.testing.assert_array_equal(so.sample_negatives(*args, users=None, history=make_history("whole", 40, 9, 1)), g["neg"])
    for I in (2, 3, 5, 50):                                     # tiny catalogs: re-draws and the (p + 1) % I fallback
        pos = np.random.default_rng(I).integers(0, I, 3000)
        want = base.sample_negatives(pos, 8, I, seed=7, sample_offset=1 << 33)
        np.testing.assert_array_equal(so.sample_negatives(pos, 8, I, seed=7, sample_offset=1 << 33), want)
        got = so.sample_negatives(pos, 8, I, seed=7, sample_offset=1 << 33, users=np.arange(3000) % 7,
                                  history=(np.zeros(8, np.int32), np.zeros(0, np.int32)))
        np.testing.assert_array_equal(got, want)
        np.testing.assert_array_equal(so.sample_negatives_literal(pos[:300], 8, I, 7, 1 << 33), want[:300])


@pytest.mark.parametrize("I", [2, 5, 5000])
@pytest.mark.parametrize("kind", KINDS)
def test_vectorised_oracle_equals_the_literal_rule(I, kind):
    U = 12
    off, ids = make_history(kind, U, I, seed=I + len(kind))
    users, pos = samples(U, I, 60, seed=3 * I)
    for offset in (0, (1 << 33) + 5):
        got = so.sample_negatives(pos, 8, I, seed=20260105, sample_offset=offset, users=users, history=(off, ids))
        want = so.sample_negatives_literal(pos, 8, I, 20260105, offset, users=users, history=(off, ids))
        np.testing.assert_array_equal(got, want)
        check_rule(got, users, pos, off, ids, I)


def test_step_two_and_three_answers():
    """All but one recipe seen: a draw that is not the free recipe falls to the cyclic walk, which finds it; the whole
    catalog seen: (p + 1) % I."""
    I, U = 5000, 4
    off, ids = make_history("all_but_one", U, I, seed=5)
    free = [int(np.setdiff1d(np.arange(I), ids[off[u]:off[u + 1]])[0]) for u in range(U)]
    users = np.arange(400) % U
    pos = np.array([(free[u] + 1 + s) % I for s, u in enumerate(users)])
    neg = so.sample_negatives(pos, 4, I, seed=1, users=users, history=(off, ids))
    assert (neg == np.array(free)[users][:, None]).all()
    off, ids = make_history("whole", U, I, seed=6)
    neg = so.sample_negatives(pos, 4, I, seed=1, users=users, history=(off, ids))
    assert (neg == ((pos + 1) % I)[:, None]).all()


def test_rows_of_a_shard_draw_what_the_whole_table_draws():
    """A row-sharded rank keeps its users' rows (shard_label_csr) and draws with the global sample index: the ranks'
    draws, together, are the single-table draws."""
    from foodrec_b200 import history_csr
    from foodrec_b200.sharded import shard_label_csr
    I, U, W = 300, 37, 3
    off, ids = make_history("mixed", U, I, seed=11)
    rng = np.random.default_rng(2)
    users = rng.integers(0, U, 500); pos = rng.integers(0, I, 500)
    order = np.argsort(users % W, kind="stable")
    users, pos = users[order], pos[order]
    want = so.sample_negatives(pos, 8, I, seed=3, sample_offset=40, users=users, history=(off, ids))
    start = 0
    for r in range(W):
        m = users % W == r
        loff, lids = shard_label_csr(*history_csr((off, ids), U), r, W, U)
        got = so.sample_negatives(pos[m], 8, I, seed=3, sample_offset=40 + start, users=users[m] // W, history=(loff, lids))
        np.testing.assert_array_equal(got, want[start:start + int(m.sum())])
        start += int(m.sum())


# ---------------------------------------------------------------- history_csr
def test_history_csr_from_a_train_matrix():
    from foodrec_b200 import history_csr
    tm = {"3": [9, 1, 4], "0": [7], "5": [2, 2, 0, 2]}          # any key order; users 1, 2, 4 absent
    off, ids = history_csr(tm, 6)
    assert off.dtype == np.int32 and ids.dtype == np.int32
    assert off.tolist() == [0, 1, 1, 1, 4, 4, 8]
    assert ids.tolist() == [7, 1, 4, 9, 0, 2, 2, 2]
    off2, ids2 = history_csr({3: (4, 9, 1), 0: np.array([7]), 5: [0, 2, 2, 2], 1: []}, 6)     # int keys, empty list
    assert off2.tolist() == off.tolist() and ids2.tolist() == ids.tolist()
    off3, ids3 = history_csr((np.array([0, 1, 1, 1, 4, 4, 8]), np.array([7, 9, 4, 1, 2, 0, 2, 2])), 6)
    assert off3.tolist() == off.tolist() and ids3.tolist() == ids.tolist()
    off4, ids4 = history_csr({}, 3)
    assert off4.tolist() == [0, 0, 0, 0] and ids4.size == 0


def test_history_csr_rejects_what_it_cannot_place():
    from foodrec_b200 import history_csr
    with pytest.raises(IndexError):
        history_csr({"6": [1]}, 6)
    with pytest.raises(IndexError):
        history_csr({"-1": [1]}, 6)
    with pytest.raises(ValueError, match="not an integer"):
        history_csr({"u7": [1]}, 9)
    with pytest.raises(ValueError, match="twice"):
        history_csr({"1": [1], 1: [2]}, 3)
    with pytest.raises(ValueError, match="int32"):
        history_csr({"1": [2**31]}, 3)
    with pytest.raises(TypeError):
        history_csr({"1": [1.5]}, 3)
    with pytest.raises(TypeError):
        history_csr([[1], [2]], 2)
    with pytest.raises(ValueError, match="entries"):
        history_csr((np.array([0, 1]), np.array([3])), 2)
    with pytest.raises(ValueError, match="non-decreasing"):
        history_csr((np.array([0, 2, 1]), np.array([3, 4])), 2)
    with pytest.raises(ValueError, match="start at 0"):
        history_csr((np.array([1, 1, 2]), np.array([3, 4])), 2)
    with pytest.raises(ValueError, match="end at"):
        history_csr((np.array([0, 1, 3]), np.array([3, 4])), 2)
