"""The bounded sweep's pruning rule (tools/bounded_sweep_model.py restates bnd_select / bnd_check): whatever the counts,
the hypotheses it leaves with a prefix count can neither be the first maximum nor tie with it, so argmax and the tie
replay see what a full sweep gives them.  Also the prefix window's arithmetic."""
import os
import sys

import numpy as np
from hypothesis import given, settings, strategies as st

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
from bounded_sweep_model import KSUB, bounded_rule, prefix_points  # noqa: E402


@st.composite
def pairs(draw):
    n = draw(st.integers(8, 400))
    k = prefix_points(n, draw(st.integers(1, 1000)) / 1000.0)
    H = draw(st.integers(1, 80))
    K = draw(st.integers(1, 40))
    rest = n - k
    pre = np.array(draw(st.lists(st.integers(0, k), min_size=H, max_size=H)), np.int64)
    add = np.array(draw(st.lists(st.integers(0, rest), min_size=H, max_size=H)), np.int64)
    if draw(st.booleans()):                       # exact ties with the maximum
        dup = draw(st.lists(st.integers(0, H - 1), max_size=H))
        src = int(np.argmax(pre + add))
        pre[dup], add[dup] = pre[src], add[src]
    return pre, pre + add, rest, K


@settings(max_examples=400, deadline=None)
@given(pairs())
def test_winner_and_ties_are_always_fully_scored(case):
    pre, full, rest, K = case
    r = bounded_rule(pre, full, rest, K)
    seen = r["counts"]
    top = full.max()
    assert seen.max() == top
    assert np.array_equal(np.flatnonzero(seen == top), np.flatnonzero(full == top))
    assert int(np.argmax(seen)) == int(np.argmax(full))
    assert np.all(seen <= full)
    if not r["fallback"]:
        assert np.all(seen[~r["cand"]] < top)


@given(st.integers(1, 200000), st.integers(1, 1000))
def test_prefix_window(n, rho_milli):
    k = prefix_points(n, rho_milli / 1000.0)
    G = (n + KSUB - 1) // KSUB
    assert 0 < k <= n
    assert k >= min(n, rho_milli * n / 1000.0)        # at least the share asked for
    assert k == n or k % (32 * KSUB) == 0             # whole 32-group flag words, or the whole pair
    assert (k + KSUB - 1) // KSUB <= G
