"""CPU self-test of the rounding-error checker in tests/grad_bounds.py: float32 sums of random terms in shuffled orders
pass it, and the same sums with one term removed, one term scaled by (1 + 8u), or an error of 1.5x the bound fail it
wherever that change exceeds the bound.  The bound is restated here from its formula, independently of the module,
so a checker loosened by a factor of two fails these tests."""
import numpy as np
import pytest

import grad_bounds as gb

U = 2.0 ** -24


def _literal_bound(n, absum, k):
    m = np.maximum(np.asarray(n, np.float64) - 1 + k, 0)
    return m * U / (1 - m * U) * absum


def _problem(seed, k):
    """Elements with 1..3000 terms (ragged), terms of mixed sign and magnitude; with k > 0 each term is a float32
    product of k + 1 factors (k roundings), and `exact` uses the float64 product of the same factors."""
    rng = np.random.default_rng(seed)
    n = np.concatenate([np.arange(1, 9), rng.integers(1, 3000, 120), [2000, 3000]])
    owner = np.repeat(np.arange(n.size), n)
    factors = [rng.standard_normal(owner.size).astype(np.float32) * np.float32(10.0) ** rng.integers(-3, 3, owner.size)
               .astype(np.float32)]
    for _ in range(k):
        factors.append(rng.uniform(0.0, 1.0, owner.size).astype(np.float32))
    t32 = factors[0]
    t64 = factors[0].astype(np.float64)
    for f in factors[1:]:
        t32 = t32 * f            # float32 product: one rounding per factor
        t64 = t64 * f.astype(np.float64)
    return n, owner, t32, t64


def _sum32(owner, t32, n_elems, rng, order):
    """float32 sums per element in a shuffled order, sequentially ('seq') or as a pairwise tree ('tree')."""
    out = np.zeros(n_elems, np.float32)
    perm = rng.permutation(owner.size)
    o, t = owner[perm], t32[perm]
    srt = np.argsort(o, kind="stable")
    o, t = o[srt], t[srt]
    starts = np.searchsorted(o, np.arange(n_elems))
    ends = np.searchsorted(o, np.arange(n_elems), side="right")
    for e in range(n_elems):
        seg = t[starts[e]:ends[e]]
        if order == "seq":
            acc = np.float32(0.0)
            for v in seg:
                acc = np.float32(acc + v)
            out[e] = acc
        else:
            out[e] = np.sum(seg, dtype=np.float32)  # numpy's pairwise summation
    return out


def _acc(owner, t64, n_elems):
    a = gb.Accumulator(n_elems)
    a.add(owner, t64)
    return a


@pytest.mark.parametrize("k", [0, 3])
@pytest.mark.parametrize("order", ["seq", "tree"])
def test_float32_sums_in_any_order_pass(k, order):
    n, owner, t32, t64 = _problem(1 + k, k)
    rng = np.random.default_rng(7)
    a = _acc(owner, t64, n.size)
    for _ in range(3):
        got = _sum32(owner, t32, n.size, rng, order)
        assert a.check(got, k, f"self-test {order} k={k}")["max_ratio"] <= 1.0


def test_untouched_elements_must_be_positive_zero_and_all_finite():
    a = gb.Accumulator(4)
    a.add([0, 0, 1], [1.0, 2.0, -3.0])
    a.check(np.array([3, -3, 0, 0], np.float32), 0, "zeros")
    with pytest.raises(AssertionError, match="no term reaches"):
        a.check(np.array([3, -3, -0.0, 0], np.float32), 0, "negative zero")
    with pytest.raises(AssertionError, match="no term reaches"):
        a.check(np.array([3, -3, 1e-30, 0], np.float32), 0, "tiny")
    with pytest.raises(AssertionError, match="non-finite"):
        a.check(np.array([np.nan, -3, 0, 0], np.float32), 0, "nan")
    # kAddTo: the initial content is one more term, and untouched elements keep it bit for bit
    init = np.array([1, 1, -0.0, 5], np.float32)
    a.check(np.array([4, -2, -0.0, 5], np.float32), 0, "init", init=init)
    with pytest.raises(AssertionError, match="no term reaches"):
        a.check(np.array([4, -2, 0.0, 5], np.float32), 0, "init sign", init=init)
    with pytest.raises(AssertionError, match="outside the rounding-error bound"):
        a.check(np.array([3, -3, -0.0, 5], np.float32), 0, "init dropped", init=init)


def _verdicts(a, got, k):
    """Per-element verdict of the checker (True: accepted), one element at a time through its public check."""
    ok = np.ones(got.size, bool)
    for e in range(got.size):
        sub = gb.Accumulator(1)
        sub.add_dense(a.exact[e:e + 1], a.absum[e:e + 1], a.count[e:e + 1])
        try:
            sub.check(got[e:e + 1], k, "one")
        except AssertionError:
            ok[e] = False
    return ok


@pytest.mark.parametrize("k", [0, 3])
def test_a_dropped_term_fails_where_it_exceeds_the_bound(k):
    n, owner, t32, t64 = _problem(11 + k, k)
    rng = np.random.default_rng(3)
    # drop one term, chosen at random, of every element
    keep = np.ones(owner.size, bool)
    for e in range(n.size):
        keep[rng.choice(np.flatnonzero(owner == e))] = False
    a = _acc(owner, t64, n.size)
    got = _sum32(owner[keep], t32[keep], n.size, rng, "seq")
    err = np.abs(got.astype(np.float64) - a.exact)
    lit = _literal_bound(a.count, a.absum, k)
    must_fail = err > lit * (1 + 1e-6)
    ok = _verdicts(a, got, k)
    assert not ok[must_fail].any(), "checker accepted a sum with a dropped term whose error exceeds the bound"
    assert must_fail.sum() >= 8, "self-test has no teeth: too few elements where the dropped term is visible"


@pytest.mark.parametrize("k", [0, 3])
def test_a_term_scaled_by_1_plus_8u_fails_where_it_exceeds_the_bound(k):
    n, owner, t32, t64 = _problem(21 + k, k)
    rng = np.random.default_rng(5)
    # scale the term of largest magnitude of every element
    t_bad = t32.copy()
    for e in range(n.size):
        ids = np.flatnonzero(owner == e)
        i = ids[np.argmax(np.abs(t64[ids]))]
        t_bad[i] = np.float32(np.float64(t32[i]) * (1 + 8 * U))
    a = _acc(owner, t64, n.size)
    got = _sum32(owner, t_bad, n.size, rng, "seq")
    err = np.abs(got.astype(np.float64) - a.exact)
    lit = _literal_bound(a.count, a.absum, k)
    must_fail = err > lit * (1 + 1e-6)
    ok = _verdicts(a, got, k)
    assert not ok[must_fail].any(), "checker accepted a sum with a scaled term whose error exceeds the bound"
    assert must_fail[0] and must_fail.sum() >= 3, "single-term and few-term sums must expose a term scaled by (1 + 8u)"


def test_the_bound_is_not_loose():
    """An error of 1.5x the bound fails and one of 0.5x passes, on every element: a checker whose bound were
    loosened by 2x would accept the first."""
    n, owner, t32, t64 = _problem(31, 3)
    a = _acc(owner, t64, n.size)
    lit = _literal_bound(a.count, a.absum, 3)
    ulp = np.spacing(np.abs(a.exact).astype(np.float32)).astype(np.float64)
    usable = lit > 64 * ulp  # the float32 rounding of exact +- c*bound stays on its side of the bound
    assert usable.sum() >= 50
    sign = np.where(np.arange(n.size) % 2, 1.0, -1.0)
    far = (a.exact + sign * 1.5 * lit).astype(np.float32)
    near = (a.exact + sign * 0.5 * lit).astype(np.float32)
    ok_far, ok_near = _verdicts(a, far, 3), _verdicts(a, near, 3)
    assert not ok_far[usable].any(), "an error of 1.5x the bound was accepted"
    assert ok_near[usable].all(), "an error of 0.5x the bound was rejected"
