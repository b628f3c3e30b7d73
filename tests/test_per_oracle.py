"""CPU: the prioritized replay oracle (oracle/per_oracle.py) against brute-force restatements of its contract."""
import numpy as np
import pytest

from oracle import per_oracle as po


def dyadic_leaves(rng, capacity, T):
    """Priorities k/64 (some 0) with alpha = 1: every partial sum is exact in fp64."""
    leaves = np.zeros(T)
    leaves[:capacity] = rng.integers(0, 65, size=capacity) / 64.
    return leaves


@pytest.mark.parametrize("capacity", [1, 700, 1024, 3000])
def test_descent_equals_searchsorted_of_cumsum(capacity):
    rng = np.random.default_rng(capacity)
    T = po.tree_size(capacity)
    leaves = dyadic_leaves(rng, capacity, T)
    leaves[0] = max(leaves[0], 1 / 64.)
    tree = po.build_tree(leaves, np.add)
    cum = np.cumsum(leaves)
    assert tree[1] == cum[-1]
    total, B = float(tree[1]), 256
    seg = total / B
    masses = [po.draw_uniform(3, 5, b, 0) * seg + float(b) * seg for b in range(B)]       # the stratified draws
    masses += [po.draw_uniform(3, 5, b, a) * total for b in range(64) for a in (1, 2)]   # the redraws
    masses += list(rng.random(200) * total) + list(cum[:20][cum[:20] < total])          # and the edges
    for m in masses:
        assert po.descend(tree, m) == np.searchsorted(cum, m, side="right"), m


def test_build_tree_is_pairwise():
    rng = np.random.default_rng(1)
    leaves = rng.random(2048)
    for op in (np.add, np.minimum):
        t = po.build_tree(leaves, op)
        for j in (1, 2, 3, 1023, 1024, 2047):
            assert t[j] == op(t[2 * j], t[2 * j + 1])


def test_sample_is_proportional_and_skips_unfilled_zero_and_stale():
    """Sampling with rejection: only filled, non-zero, resident leaves come out; the weights follow the contract."""
    cap, T = 40, 1024
    rng = np.random.default_rng(7)
    orc = po.PerOracle(cap, alpha=1.0)
    orc.ingest(30)                                        # slots 30..39 unfilled
    orc.sum_leaves[:30] = orc.min_leaves[:30] = rng.integers(1, 9, size=30) / 8.
    state_step = np.arange(cap, dtype=np.int64)           # slots 0..9 stale at cur_step = 19 with depth 10
    slot12 = orc.sum_leaves[12]
    orc.sum_leaves[12] = orc.min_leaves[12] = 0.          # priority 0 (as after an underflowing pow)
    st, mt = orc.trees()
    idx, pos, w = po.sample(st, mt, orc.leaf_pos, state_step, 30, 19, 10, 512, .4, 11, 1)
    assert (idx >= 10).all() and (idx < 30).all() and (idx != 12).all()
    assert np.array_equal(pos, orc.leaf_pos[idx])
    orc.sum_leaves[12] = orc.min_leaves[12] = slot12
    st, mt = orc.trees()
    idx, pos, w = po.sample(st, mt, orc.leaf_pos, state_step, 30, 19, 10, 512, .4, 11, 1)
    assert (idx >= 10).all() and (idx < 30).all() and (idx == 12).any()
    total = st[1]
    expect = (st[T + idx] / total * 30) ** -.4 / (mt[1] / total * 30) ** -.4
    assert mt[1] == orc.min_leaves[:30].min() > 0            # p_min counts the stale leaves too
    np.testing.assert_array_equal(w, expect)
    counts = np.bincount(idx, minlength=cap)[10:30]       # stratified: close to proportional over resident leaves
    np.testing.assert_allclose(counts / 512, st[T + 10:T + 30] / st[T + 10:T + 30].sum(), atol=.02)
    # a ring that is all stale gives idx = -1 rows with weight 0
    idx, pos, w = po.sample(st, mt, orc.leaf_pos, np.full(cap, po.INT64_MIN), 30, 19, 10, 8, .4, 11, 2)
    assert (idx == -1).all() and (pos == -1).all() and (w == 0).all()


def test_new_records_enter_at_max_priority_and_overwrites_take_it():
    orc = po.PerOracle(8, alpha=.5)
    orc.ingest(5)
    assert (orc.sum_leaves[:5] == 1.).all() and np.isinf(orc.min_leaves[5:]).all() and orc.sum_leaves[5:].sum() == 0
    orc.update([1, 2], [1, 2], [9., 4.])
    assert orc.max_priority == 9. and orc.sum_leaves[1] == 3. and orc.sum_leaves[2] == 2.
    orc.ingest(10)                                        # positions 5..9: slots 5, 6, 7, 0, 1
    assert np.array_equal(orc.leaf_pos, [8, 9, 2, 3, 4, 5, 6, 7])
    assert (orc.sum_leaves[[5, 6, 7, 0, 1]] == 3.).all() and orc.sum_leaves[2] == 2.
    orc.ingest(30)                                        # more than a ring's worth: only the last 8 positions
    assert np.array_equal(orc.leaf_pos, [24, 25, 26, 27, 28, 29, 22, 23])


def test_update_last_wins_skips_and_counts():
    orc = po.PerOracle(16, alpha=1.0)
    orc.ingest(16)
    idx = np.array([3, -1, 3, 5, 7, 3, 9, 9])
    pos = orc.leaf_pos[np.maximum(idx, 0)].copy()
    pos[idx < 0] = -1
    pr = np.array([2., 50., 3., np.nan, 0., 4., 5., -1.])
    orc.ingest(0)                                         # nothing new
    orc.leaf_pos[7] += 16                                 # slot 7 was overwritten after the sample
    orc.update(idx, pos, pr)
    assert orc.sum_leaves[3] == 4.                        # last of three occurrences
    assert orc.sum_leaves[5] == 1. and orc.sum_leaves[7] == 1.  # nan skipped; overwritten skipped (its 0. too)
    assert orc.sum_leaves[9] == 5.                        # the later -1 is skipped, so the earlier 5 stands
    assert orc.n_rejected == 2                            # nan and -1; the overwritten row's 0 is not counted
    assert orc.max_priority == 5.                         # the -1 row's 50 never counts: idx = -1
    assert orc.min_leaves[3] == 4.


def test_max_priority_counts_overridden_duplicates():
    """Every applied priority raises max_priority, also one a later duplicate overrides."""
    orc = po.PerOracle(4, alpha=1.0)
    orc.ingest(4)
    orc.update([2, 2], [2, 2], [7., 3.])
    assert orc.sum_leaves[2] == 3. and orc.max_priority == 7.
    orc.ingest(5)                                         # position 4 -> slot 0
    assert orc.sum_leaves[0] == 7.
