"""The weight-table grid of tests/weight_tables.py is what it claims, and its inputs reach every regime (no GPU needed).

Without these checks the GPU comparisons at other beta could pass vacuously: a table without zeros, or inputs whose weight sums
never leave div_fast's range, would exercise nothing new."""
import numpy as np
import pytest

from tests import weight_tables as wt


@pytest.mark.parametrize("beta,regime,normal,denormal,zero", wt.GRID, ids=[wt.beta_id(g[0]) for g in wt.GRID])
def test_table_has_the_claimed_regime(beta, regime, normal, denormal, zero):
    lut = wt.table(beta)
    assert lut[256] == 0 and lut[0] == 1.0, regime
    got = []
    for idx in wt.entry_classes(lut):
        if len(idx):
            assert np.array_equal(idx, np.arange(idx[0], idx[-1] + 1)), "%s: entries of one class are not contiguous" % regime
        got.append((int(idx[0]), int(idx[-1]) + 1) if len(idx) else None)
    assert got == [normal, denormal, zero], "%s: normal / denormal / zero index ranges %s, claimed %s" % (regime, got, [normal, denormal, zero])
    # the weights never increase along the table, and never exceed 1 (beta >= 0)
    assert (np.diff(lut[:256]) <= 0).all() and (lut <= 1.0).all()


def test_negative_zero_gives_the_table_of_zero():
    assert np.array_equal(wt.table(-0.0).view(np.uint32), wt.table(0.0).view(np.uint32))
    assert (wt.table(0.0)[:256] == 1.0).all()


def test_grid_spans_the_regimes():
    """The grid holds every kind of table the exact division treats differently."""
    kinds = set()
    for beta, *_ in wt.GRID:
        normal, den, zero = wt.entry_classes(wt.table(beta))
        kinds.add((len(normal) == 256, len(den) > 0, len(zero) > 0, len(normal) == 1))
    assert (True, False, False, False) in kinds          # no denormals, no zeros
    assert (False, True, False, False) in kinds          # denormal tail without zeros
    assert (False, True, True, False) in kinds           # denormals and zeros
    assert (False, False, True, True) in kinds           # w[0] alone


@pytest.mark.parametrize("shape,level,levels", wt.LEVEL_CASES)
@pytest.mark.parametrize("kind", list(wt.INPUTS))
def test_sums_at_beta_zero_count_the_neighbours(kind, shape, level, levels):
    """At beta = 0 every weight is 1, so a free pixel's sum is its number of neighbours inside the level: 2, 3 or 4.  This also
    checks the restated sum order against an independent count."""
    rows, cols = shape
    gray, depth, scribble = wt.level_input(kind, rows, cols, level)
    for beta in (0.0, -0.0):
        s, free = wt.weight_sums(gray, depth, scribble, level, levels - 1, wt.table(beta))
        n = np.full((rows, cols), 4, np.float32)
        n[0, :] -= 1
        n[-1, :] -= 1
        n[:, 0] -= 1
        n[:, -1] -= 1
        assert free.any()
        assert np.array_equal(s[free], n[free])
        assert set(np.unique(s[free]).tolist()) <= {2.0, 3.0, 4.0}


@pytest.mark.parametrize("shape,level,levels", wt.LEVEL_CASES[:2])
@pytest.mark.parametrize("beta", wt.BETAS, ids=wt.beta_id)
def test_gray_steps_reach_every_regime_of_the_table(beta, shape, level, levels):
    """The same non-vacuity guard as `assert tiny.any()` in the pocket test: at every beta the gray-step input has free pixels
    with a weight sum of exactly +0 whenever the table has zeros (beta >= 0.45), and sums in (0, 2^-100) and in (0, 2^-21)
    whenever four of the table's smallest non-zero weight fall below those bounds."""
    rows, cols = shape
    lut = wt.table(beta)
    gray, depth, scribble = wt.level_input("gray-steps", rows, cols, level)
    s, free = wt.weight_sums(gray, depth, scribble, level, levels - 1, lut)
    s = s[free]
    _, den, zero = wt.entry_classes(lut)
    assert bool((s == 0).any()) == (len(zero) > 0) == (beta >= 0.45)
    assert not np.signbit(s).any()                                         # +0 only
    for bound in (wt.TWO_M100, wt.TWO_M21):
        reach = bool(((s > 0) & (s < bound)).any())
        assert reach == wt.table_allows(lut, bound), (bound, reach)
    assert wt.table_allows(lut, wt.TWO_M100) == (0.35 <= beta <= 8.0)
    # sums that are themselves denormal wherever the table has denormals below a quarter of FLT_MIN
    if len(den) and lut[den[-1]] * 4 < wt.FLT_MIN:
        assert ((s > 0) & (s < wt.FLT_MIN)).any()


@pytest.mark.parametrize("kind", ["random", "salt-and-pepper", "gray-steps"])
def test_inputs_with_edges_reach_zero_sums_at_large_beta(kind):
    """At beta = 8, where only w[0..12] are non-zero, each input with grey-level edges has free pixels whose sum is +0: the
    zero-sum path is reached by more than the input built for it.  (The enclosed-zero input has differences of at most 20 grey
    levels on purpose: its point is numerators decaying to zero, not small weights.)"""
    (rows, cols), level, levels = wt.LEVEL_CASES[0]
    gray, depth, scribble = wt.level_input(kind, rows, cols, level)
    s, free = wt.weight_sums(gray, depth, scribble, level, levels - 1, wt.table(8.0))
    assert (s[free] == 0).any()
