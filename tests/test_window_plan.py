"""The window planner of the windowed forward-backward (engine.plan_windows): no GPU needed."""
import numpy as np
import pytest

from tehmm_b200.engine import plan_windows


@pytest.mark.parametrize("total", [1, 2, 7, 1000, 2_500_001])
@pytest.mark.parametrize("cap", [1, 3, 64, 999, 10 ** 8])
def test_cuts_cover_every_row_once_within_the_cap(total, cap):
    cuts = plan_windows(total, 1, 1 << 62, max_window_steps=cap, min_window_steps=1)
    assert cuts[0] == 0 and cuts[-1] == total
    w = np.diff(cuts)
    assert (w >= 1).all() and (w <= cap).all()         # strictly increasing: no row twice, none skipped
    assert len(w) == -(-total // cap)                   # as few windows as the cap allows
    assert (w[:-1] == cap).all()


def test_budget_from_the_sizes():
    # 3 fp32 lattices of stride 64 + rowmax: 776 bytes per step
    per_step = 3 * 64 * 4 + 8
    kw = dict(min_window_steps=1)
    assert plan_windows(1000, per_step, 1000 * per_step, **kw) is None       # fits: the unwindowed path
    cuts = plan_windows(1000, per_step, 250 * per_step, **kw)
    assert list(cuts) == [0, 250, 500, 750, 1000]
    cuts = plan_windows(1000, per_step, 250 * per_step + per_step - 1, **kw)   # a partial step buys nothing
    assert (np.diff(cuts) <= 250).all()
    # a cap given by the caller is a cap, not a choice of algorithm: the budget still applies
    assert (np.diff(plan_windows(1000, per_step, 100 * per_step, max_window_steps=400, **kw)) <= 100).all()
    assert len(plan_windows(1000, per_step, 10 ** 12, max_window_steps=1000, **kw)) == 2


def test_fit_decided_with_the_unwindowed_lattices():
    # an E-step without posteriors holds 2 lattices unwindowed; a window holds 3
    two, three = 2 * 64 * 4 + 8, 3 * 64 * 4 + 8
    assert plan_windows(1000, three, 1000 * two, fit_bytes_per_step=two, min_window_steps=1) is None
    cuts = plan_windows(1000, three, 999 * two, fit_bytes_per_step=two, min_window_steps=1)
    assert (np.diff(cuts) <= 999 * two // three).all() and cuts[-1] == 1000


def test_too_little_memory_fails_fast():
    # windows below the floor would crawl through millions of launches: refuse with a clear error
    with pytest.raises(MemoryError):
        plan_windows(10 ** 7, 776, 0)
    with pytest.raises(MemoryError):
        plan_windows(10 ** 7, 776, 4095 * 776)
    assert len(plan_windows(10 ** 7, 776, 4096 * 776)) == -(-10 ** 7 // 4096) + 1
    # a caller's cap below the floor is honoured when memory allows it
    assert len(plan_windows(10, 776, 0 + 10 * 776, max_window_steps=1)) == 11
