"""Which radix-sort path each case of tests/test_gpu_wide_ids.py reaches, restated from foodrec_b200/csrc/sort.cu.

The sort splits ``bits_for(n_ids)`` key bits into passes of at most 10 bits (``plan_digits``); a pass whose key count
fits 16 tiles of 2,048 keys derives its offsets inside the scatter kernel (fused), a larger one runs a separate offset
scan.  Every GPU case below is sized to reach a stated (bits, digits, fused) combination; a resized case that no longer
reaches its path fails here, without a GPU.  The GPU sort tests additionally pin this restatement to the library by
counting its launches (``sort_launches``)."""
import numpy as np
import pytest

MAX_DIGIT_BITS = 10          # sort.cu
SORT_TILE = 2048             # internal.h
FUSED_SCAN_MAX_TILES = 16    # sort.cu
SCAN_TILE = 4096             # sort.cu: entries of the offset table one scan block covers


def bits_for(n):
    """ctx.h: bits needed to represent ids in [0, n)."""
    b = 0
    while b < 32 and (1 << b) < n:
        b += 1
    return max(b, 1)


def plan_digits(nbits):
    """sort.cu plan_digits + radix_sort_jobs: the width of every pass's digit, least significant first."""
    nbits = max(nbits, 1)
    passes = (nbits + MAX_DIGIT_BITS - 1) // MAX_DIGIT_BITS
    bpp = (nbits + passes - 1) // passes
    return tuple(max(1, min(bpp, nbits - p * bpp)) for p in range(passes))


def ntiles(n):
    return (n + SORT_TILE - 1) // SORT_TILE


def fused(n):
    return ntiles(n) <= FUSED_SCAN_MAX_TILES


def scan_blocks(n, digit_bits):
    """Blocks of the separate offset scan of a pass over n keys (scan_offsets_kernel)."""
    return ((1 << digit_bits) * ntiles(n) + SCAN_TILE - 1) // SCAN_TILE


def sort_launches(n, nbits):
    """Launches of one fr_sort_pairs call: histogram + scatter per pass, plus the offset scan when not fused."""
    return len(plan_digits(nbits)) * (2 + (0 if fused(n) else 1))


# ------------------------------------------------------------------------------------------- fr_sort_pairs cases
SORT_NBITS = (21, 24, 26, 30, 31, 32)
SORT_N = (32_768, 32_769, 524_288)
SORT_DIGITS = {21: (7, 7, 7), 24: (8, 8, 8), 26: (9, 9, 8), 30: (10, 10, 10), 31: (8, 8, 8, 7), 32: (8, 8, 8, 8)}
SORT_FUSED = {32_768: True, 32_769: False, 524_288: False}
BIG_N, BIG_NBITS = 2**25 + 2_049, 30          # the last scan block's loop over the block sums runs twice
SORT_PATTERNS = ("uniform", "all_equal", "top_digit", "bottom_digit", "middle_digit", "high_bit", "descending_dups")

# ------------------------------------------------------------------------------------------- training-step cases
# U, I: table rows; D; bpr; B groups per step (S = B or 2B item rows); L labels
STEP_CASES = {
    "a": dict(U=2**25 + 3, I=1_000, D=4, bpr=True, B=65_536, L=9),
    "b": dict(U=1_000, I=2**21 + 1, D=4, bpr=False, B=16_384, L=9),
    "c": dict(U=2**20 + 1, I=2**20, D=128, bpr=True, B=32_768, L=9),
    "d": dict(U=4_096, I=4_096, D=4, bpr=False, B=4_096, L=1_100),
}
# the digits of the by-user and by-recipe sorts, and whether their passes fuse the offsets
STEP_EXPECT = {
    "a": dict(users=(9, 9, 8), items=(10,), fused=False),      # the recipe job idles in passes 2-3
    "b": dict(users=(10,), items=(8, 8, 6), fused=True),       # the user job idles in passes 2-3
    "c": dict(users=(7, 7, 7), items=(10, 10), fused=False),   # the recipe job idles in pass 3
    "d": dict(users=(6, 6), items=(6, 6), fused=True),
}
LABEL_CASE_D = dict(max_label_entries=65_536, labels_per_row=12, digits=(6, 5))   # a two-pass label sort, device count

# ------------------------------------------------------------------------------------------- row-sharded cases
SHARD_W = 8
SHARD_UG = SHARD_W * (2**22 + 5) - 3           # global users: the last three ranks hold a padding row
SHARD_IG = SHARD_W * (2**20 + 3)               # global recipes
SHARD_B = 8_192                                # groups per global step
SHARD_MAX_ROWS = 16_384                        # one rank may own every row of a BPR step


def shard_rows_per_rank(n, W=SHARD_W):
    return (n + W - 1) // W


# ------------------------------------------------------------------------------------------- id patterns
def adversarial_ids(n_ids, rng, count, hot_rows=0, top_only=64, scattered_rows=200):
    """``count`` ids in [0, n_ids) laid out against an LSD radix sort of ``bits_for(n_ids)`` bits, shuffled:
    ids that share every digit but the top one, ids that share all but the bottom digit, ids that differ only in
    a middle digit (when there is one), 0 and n_ids - 1, one hot id whose top digit is the largest any id reaches
    (``hot_rows`` copies), one id repeated ``scattered_rows`` times, the rest uniform.  Returns (ids, hot, parts)."""
    digits = plan_digits(bits_for(n_ids))
    top_shift = sum(digits[:-1])
    parts = {}
    if len(digits) > 1:
        low = int(rng.integers(0, 1 << top_shift))
        k = np.arange(0, ((n_ids - 1 - low) >> top_shift) + 1, dtype=np.int64)
        k = k[np.linspace(0, len(k) - 1, min(top_only, len(k))).astype(np.int64)]
        parts["top_digit"] = low | (k << top_shift)
        mid_shift = digits[0]
        if len(digits) > 2:
            base = int(rng.integers(0, n_ids)) & ~(((1 << digits[1]) - 1) << mid_shift)
            m = base | (np.arange(1 << digits[1], dtype=np.int64) << mid_shift)
            parts["middle_digit"] = m[m < n_ids]
    hi = int(rng.integers(0, max(1, n_ids >> digits[0]))) << digits[0]
    b = hi | np.arange(1 << digits[0], dtype=np.int64)
    parts["bottom_digit"] = b[b < n_ids]
    parts["ends"] = np.array([0, n_ids - 1], np.int64)
    top_lo = ((n_ids - 1) >> top_shift) << top_shift
    hot = top_lo + (n_ids - 1 - top_lo) // 2
    parts["hot"] = np.full(hot_rows, hot, np.int64)
    parts["scattered"] = np.full(scattered_rows, int(rng.integers(0, n_ids)), np.int64)
    fixed = np.concatenate(list(parts.values()))
    assert fixed.size <= count, (fixed.size, count)
    ids = np.concatenate([fixed, rng.integers(0, n_ids, count - fixed.size)])
    return ids[rng.permutation(count)], hot, parts


# ------------------------------------------------------------------------------------------- CPU tests
def test_restated_plan_digits():
    assert [bits_for(n) for n in (1, 2, 3, 1000, 1024, 1025, 2**20, 2**20 + 1)] == [1, 1, 2, 10, 10, 11, 20, 21]
    assert plan_digits(20) == (10, 10) and plan_digits(10) == (10,) and plan_digits(11) == (6, 5)
    for nbits in range(1, 33):
        d = plan_digits(nbits)
        assert sum(d) == nbits and max(d) <= MAX_DIGIT_BITS and len(d) == -(-nbits // MAX_DIGIT_BITS)


@pytest.mark.parametrize("nbits", SORT_NBITS)
def test_sort_cases_reach_three_and_four_passes(nbits):
    assert plan_digits(nbits) == SORT_DIGITS[nbits]
    assert len(plan_digits(nbits)) >= 3
    for n in SORT_N:
        assert fused(n) == SORT_FUSED[n]
        assert sort_launches(n, nbits) == len(SORT_DIGITS[nbits]) * (2 if SORT_FUSED[n] else 3)
    assert plan_digits(31)[-1] < plan_digits(31)[0]                 # a short last digit
    assert 524_288 == 2 * 262_144                                     # the bench's rows per step (B = 262,144 BPR)


def test_big_sort_loops_over_more_than_one_scan_tile_of_block_sums():
    d = plan_digits(BIG_NBITS)
    assert d == (10, 10, 10) and not fused(BIG_N)
    nb = scan_blocks(BIG_N, d[0])
    assert nb > SCAN_TILE and -(-nb // SCAN_TILE) == 2                # the last block's loop iterates twice
    # the sort buffers hold that many block sums (ctx.h alloc_sort: RADIX_BINS * ntiles / 4096 + 2)
    assert (1024 * ntiles(BIG_N)) // 4096 + 2 >= nb


@pytest.mark.parametrize("case", sorted(STEP_CASES))
def test_step_cases_reach_their_sort_paths(case):
    c, x = STEP_CASES[case], STEP_EXPECT[case]
    S = c["B"] * (2 if c["bpr"] else 1)
    assert plan_digits(bits_for(c["U"])) == x["users"]
    assert plan_digits(bits_for(c["I"])) == x["items"]
    assert fused(S) == x["fused"]
    if case == "d":
        assert plan_digits(bits_for(c["L"])) == LABEL_CASE_D["digits"]
        assert not fused(LABEL_CASE_D["max_label_entries"])           # n_host of the label sort is its capacity
        assert S * LABEL_CASE_D["labels_per_row"] > FUSED_SCAN_MAX_TILES * SORT_TILE   # keys in more than 16 tiles
    else:
        # one job takes fewer passes than the other: it idles (bits == 0) in the shared launches' later passes
        assert len(x["users"]) != len(x["items"])


def test_sharded_cases_reach_three_passes():
    W = SHARD_W
    uloc, ipr = shard_rows_per_rank(SHARD_UG), shard_rows_per_rank(SHARD_IG)
    assert uloc == 2**22 + 5 and ipr == 2**20 + 3
    assert [len(range(r, SHARD_UG, W)) for r in range(W)] == [uloc] * 5 + [uloc - 1] * 3
    assert plan_digits(bits_for(uloc)) == (8, 8, 7)                   # the by-user sort of the plan
    assert plan_digits(bits_for(W * ipr)) == (8, 8, 8)                # the plan's owner-major recipe keys
    assert plan_digits(bits_for(ipr + 1)) == (7, 7, 7)                # the owners' serve keys
    assert plan_digits(bits_for(W * ipr + 1)) == (8, 8, 8)            # the sharded evaluation plan
    assert 2 * SHARD_B <= SHARD_MAX_ROWS


@pytest.mark.parametrize("n_ids", [2**25 + 3, 2**21 + 1, 2**20 + 1, 2**20, 2**22 + 4, 2**20 + 3, 1_000])
def test_adversarial_ids_hit_every_digit(n_ids):
    rng = np.random.default_rng(n_ids)
    ids, hot, parts = adversarial_ids(n_ids, rng, 20_000, hot_rows=600)
    digits = plan_digits(bits_for(n_ids))
    shifts = np.cumsum((0,) + digits[:-1])
    dig = lambda x, p: (x >> shifts[p]) & ((1 << digits[p]) - 1)
    assert ids.min() >= 0 and ids.max() < n_ids and {0, n_ids - 1} <= set(ids.tolist())
    assert dig(hot, len(digits) - 1) == dig(n_ids - 1, len(digits) - 1)   # the largest top digit any id reaches
    assert (ids == hot).sum() >= 600                                       # > 16 chunks of 32 rows
    if len(digits) > 1:
        t = parts["top_digit"]
        assert len(np.unique(t)) > 1 and len(np.unique(t & ((1 << shifts[-1]) - 1))) == 1
    if len(digits) > 2:
        m = parts["middle_digit"]
        assert len(np.unique(dig(m, 1))) > 1 and len(np.unique(m & ~(((1 << digits[1]) - 1) << shifts[1]))) == 1
    bt = parts["bottom_digit"]
    assert len(np.unique(bt)) > 1 and len(np.unique(bt >> digits[0])) == 1
