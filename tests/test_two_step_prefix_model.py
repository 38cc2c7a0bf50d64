"""The two-step prefix of the bounded sweep (option 16; tools/bounded_sweep_model.py restates bnd_select, bnd_extend and
bnd_check): a hypothesis pruned after the short stage A is also pruned after the full prefix, so extending only the
survivors S decides every pair as the one-step prefix over k correspondences would, and argmax and the tie replay see
what a full sweep gives them."""
import os
import sys

import numpy as np
from hypothesis import given, settings, strategies as st

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
from bounded_sweep_model import bounded_rule, prefix_points, two_step_rule  # noqa: E402


@st.composite
def two_step_pairs(draw):
    n = draw(st.integers(8, 400))
    k = prefix_points(n, draw(st.integers(1, 1000)) / 1000.0)
    k0 = prefix_points(n, draw(st.integers(1, 1000)) / 1000.0)
    k0 = min(k0, k)
    H = draw(st.integers(1, 80))
    K = draw(st.integers(1, 40))
    # per hypothesis: exact counts over [0, k0), [k0, k), [k, n) and upper bounds of the first two
    e0 = np.array(draw(st.lists(st.integers(0, k0), min_size=H, max_size=H)), np.int64)
    e1 = np.array(draw(st.lists(st.integers(0, k - k0), min_size=H, max_size=H)), np.int64)
    e2 = np.array(draw(st.lists(st.integers(0, n - k), min_size=H, max_size=H)), np.int64)
    if draw(st.booleans()):                       # exact ties with the maximum
        dup = draw(st.lists(st.integers(0, H - 1), max_size=H))
        src = int(np.argmax(e0 + e1 + e2))
        e0[dup], e1[dup], e2[dup] = e0[src], e1[src], e2[src]
    b0 = e0 + np.array([draw(st.integers(0, k0 - v)) for v in e0], np.int64)
    b1 = e1 + np.array([draw(st.integers(0, k - k0 - v)) for v in e1], np.int64)
    return b0, b0 + b1, e0 + e1 + e2, n, k0, k, K


@settings(max_examples=400, deadline=None)
@given(two_step_pairs())
def test_pruned_after_stage_a_is_pruned_after_the_prefix(case):
    pre0, pre, full, n, k0, k, K = case
    t = two_step_rule(pre0, pre, full, n, k0, k, K)
    pruned0 = ~t["cand"] & ~t["live"]
    assert np.all(pre0[pruned0] + (n - k0) < t["L"])
    assert np.all(pre[pruned0] + (n - k) < t["L"])
    assert np.all(full[pruned0] < t["L"])
    # the pair falls back exactly when the one-step rule over k, with the same candidates, finds an escapee
    one = ~t["cand"] & (pre + (n - k) >= t["L"])
    assert t["fallback"] == bool(one.any())
    # a pair certain to fall back after stage A (pre0 is a lower bound of pre) does fall back, and skips stage B
    assert not t["certain"] or t["fallback"]
    assert t["evals_a"] == k0 * len(pre0) and t["evals_b"] == (0 if t["certain"] else t["S"] * (k - k0))


@settings(max_examples=400, deadline=None)
@given(two_step_pairs())
def test_two_step_keeps_winner_and_ties(case):
    pre0, pre, full, n, k0, k, K = case
    seen = two_step_rule(pre0, pre, full, n, k0, k, K)["counts"]
    top = full.max()
    assert seen.max() == top
    assert np.array_equal(np.flatnonzero(seen == top), np.flatnonzero(full == top))
    assert int(np.argmax(seen)) == int(np.argmax(full))


@settings(max_examples=200, deadline=None)
@given(two_step_pairs())
def test_one_step_when_stage_a_covers_the_prefix(case):
    pre0, _, full, n, _, k, K = case
    t = two_step_rule(pre0, pre0, full, n, k, k, K)
    r = bounded_rule(pre0, full, n - k, K)
    assert t["fallback"] == r["fallback"] == t["certain"] and t["escapees"] == r["escapees"] == t["S"]
    assert t["evals_b"] == 0
    assert np.array_equal(t["counts"], r["counts"])
