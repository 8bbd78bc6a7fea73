"""The reduced golden form (tests/golden_util.py) never passes a result that the whole-array comparison would fail on
the points it can see, and fails on non-finite results wherever they are."""
import numpy as np

from tests import golden_util as G


def reduced(a, exact=False):
    out = {}
    G.reduce_into(out, "x", a, exact)
    return G.load(_Z(out), "x")


class _Z(dict):
    @property
    def files(self):
        return list(self)


def test_non_finite_entries_outside_the_sample_fail():
    want = np.random.default_rng(1).uniform(-1, 1, (64, 8))
    w = reduced(want)
    assert G.rel_err(want, w) == 0.0
    _, _, idx = G._probes(want.shape)
    outside = np.setdiff1d(np.arange(want.size), idx)[[0, -1]]
    for bad in (np.nan, np.inf, -np.inf):
        for at in outside:
            have = want.copy().reshape(-1)
            have[at] = bad
            have = have.reshape(want.shape)
            assert not G.rel_err(have, w) < 1e-11, (bad, at)
            assert not G.rel_err(have, want) < 1e-11, (bad, at)  # the whole-array comparison agrees


def test_reduced_error_is_a_lower_bound_and_sees_large_errors():
    rng = np.random.default_rng(2)
    want = rng.uniform(-1, 1, (512, 128))
    w = reduced(want)
    noise = want + rng.uniform(-1e-13, 1e-13, want.shape)
    assert G.rel_err(noise, w) <= G.rel_err(noise, want) < 1e-11
    one_off = want.copy()
    one_off[300, 17] += 1e-3  # a lone entry off by 1e-3: above rows x cols x tolerance
    assert not G.rel_err(one_off, w) < 1e-11
    spread = want.copy()
    spread[256:] *= 1 + 1e-9  # half of the rows off by 1e-9
    assert not G.rel_err(spread, w) < 1e-11


def test_exact_arrays_compare_by_digest():
    want = np.arange(100, dtype=np.int64)
    w = reduced(want, exact=True)
    assert G.same(want.astype(np.int32), w)
    have = want.copy()
    have[57] += 1
    assert not G.same(have, w) and not G.same(want[:99], w)
