"""The screening's exact top-k (launch_screen_select: a device-wide radix select when p > 16384, launch_topk otherwise or when
the boundary bin is too large) against the rule it implements -- larger utility first, then lower index; the kept
indices ascending; the tie flag set iff more keys equal the k-th than are taken -- and against launch_topk itself."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

DBL_MAX = np.finfo(np.float64).max


def expected(v, k):
    order = np.lexsort((np.arange(v.size), -v))
    sel = np.sort(order[:k])
    kth = v[order[k - 1]]
    tie = int(np.count_nonzero(v == kth) > np.count_nonzero(v[sel] == kth))
    return sel, tie


def utilities(p, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    return rng.standard_normal(p) ** 2 * np.exp(rng.uniform(-6, 6, p))


def case(name):
    rng = np.random.Generator(np.random.PCG64(sum(map(ord, name))))
    if name == "p500k_k5000":
        return utilities(500_000, 1), 5000
    if name == "p500k_k20":
        return utilities(500_000, 2), 20
    if name == "p500k_k1":
        return utilities(500_000, 3), 1
    if name.startswith("p_"):  # p_<p>_<k>: around the one-CTA limit of 16384 keys
        _, p, k = name.split("_")
        return utilities(int(p), int(p)), int(k)
    if name == "all_zero":
        return np.zeros(100_000), 5000
    if name == "eight_values":
        return rng.integers(0, 8, 200_000).astype(np.float64) * 0.5, 5000
    if name == "same_top_16_bits":  # one exponent, the top 8 mantissa bits equal: a boundary bin of ~12 000 keys
        return 1.0 + rng.uniform(0, 2.0 ** -8, 200_000), 5000
    if name == "same_top_24_bits":  # every key in one sub-bin: the fallback decides
        return 1.0 + rng.uniform(0, 2.0 ** -14, 200_000), 5000
    if name == "rounded_ties":  # exact ties spread over the range, several at the boundary
        return np.round(utilities(300_000, 4), 2), 5000
    if name == "pins":
        v = utilities(300_000, 5)
        v[rng.choice(v.size, 30, replace=False)] = DBL_MAX
        return v, 5000
    if name == "pins_more_than_k":
        v = utilities(300_000, 6)
        v[rng.choice(v.size, 30, replace=False)] = DBL_MAX
        return v, 20
    raise KeyError(name)


CASES = ["p500k_k5000", "p500k_k20", "p500k_k1", "p_16383_100", "p_16384_100", "p_16385_100", "p_16385_8192",
         "p_40000_3000", "p_16384_16384", "p_16000_16000", "all_zero", "eight_values", "same_top_16_bits",
         "same_top_24_bits", "rounded_ties", "pins", "pins_more_than_k"]


@pytest.mark.parametrize("name", CASES)
def test_screen_select_matches_rule_and_topk(name):
    from bess_b200 import engine
    v, k = case(name)
    sel, tie = engine.screen_select(v, k)
    exp_sel, exp_tie = expected(v, k)
    assert np.array_equal(sel, exp_sel), name
    assert tie == exp_tie, name
    ref_sel, ref_tie = engine.topk(v, k)
    assert np.array_equal(sel, ref_sel) and tie == ref_tie, name
