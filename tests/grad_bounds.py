"""Order-independent rounding-error bound for float32 gradients that the kernels accumulate with atomics.

Every gradient element a backward kernel writes is a float32 sum, in an order nobody controls, of n terms, and each
term is a float32 expression with at most k roundings.  For any summation order (sequential, tree, or atomics in
whatever order they land),

    |got - exact| <= gamma(n - 1 + k) * sum_i |t~_i|,    gamma(m) = m*u / (1 - m*u),   u = 2^-24,

where `exact` is the sum of the terms evaluated in exact arithmetic from the kernel's own float32 branch decisions and
weights, and t~_i is term i evaluated on the absolute values of its operands (Higham, Accuracy and Stability of
Numerical Algorithms, 2nd ed., (3.4) and Lemma 3.3).  A kernel that drops a contribution, uses a wrong weight or a
wrong sign is off by far more than this; a kernel that only sums in another order is not.

`Accumulator` collects the terms per output element in float64 with np.bincount; `Accumulator.check` applies the
bound and the two exact rules: an element no term reaches keeps its initial value bit for bit (+0.0 without one), and
every element is finite.  The float64 terms and sums are themselves rounded; `gamma64(n + k + 2) * sum|t~|` covers
that.  float32 atomic
adds flush subnormal inputs and results to zero (PTX `red.global.add.f32`), so each of the n + k roundings may also
lose up to FLT_MIN in absolute terms; that slack is ~1e-38 and changes no verdict at the magnitudes tested.
"""
from __future__ import annotations

import numpy as np

U = 2.0 ** -24
U64 = 2.0 ** -53
FLT_MIN = float(np.finfo(np.float32).tiny)


def gamma(m, u: float = U) -> np.ndarray:
    m = np.asarray(m, np.float64)
    return m * u / (1.0 - m * u)


def bound(count, absum, k: int) -> np.ndarray:
    """The largest |got - exact| a float32 sum of `count` terms of at most `k` roundings each may show."""
    count = np.asarray(count, np.float64)
    m = np.maximum(count - 1 + k, 0)
    return (gamma(m) + gamma(count + k + 2, U64)) * absum + (count + k) * FLT_MIN


class Accumulator:
    """float64 scatter-add of terms, of their operand-absolute values and of their count, per flat output element."""

    def __init__(self, size: int):
        self.size = int(size)
        self.exact = np.zeros(self.size)
        self.absum = np.zeros(self.size)
        self.count = np.zeros(self.size)

    def add(self, index, terms, abs_terms=None) -> None:
        index = np.asarray(index, np.int64).ravel()
        terms = np.asarray(terms, np.float64).ravel()
        a = np.abs(terms) if abs_terms is None else np.asarray(abs_terms, np.float64).ravel()
        self.exact += np.bincount(index, weights=terms, minlength=self.size)
        self.absum += np.bincount(index, weights=a, minlength=self.size)
        self.count += np.bincount(index, minlength=self.size)

    def add_dense(self, terms, abs_terms, counts) -> None:
        """Terms already summed per element (in float64) by the caller."""
        self.exact += np.asarray(terms, np.float64).ravel()
        self.absum += np.asarray(abs_terms, np.float64).ravel()
        self.count += np.asarray(counts, np.float64).ravel()

    def check(self, got, k: int, name: str, init=None, old_tol=(1e-4, 1e-4)) -> dict:
        """Assert the bound on every element of `got` (float32, any shape with `size` elements).  `init`: the
        buffer's content before an accumulating (kAddTo) call; it enters the sum as one more term.  Returns the
        largest |got - exact| / bound and the median of bound / (atol + rtol * |exact|) of `old_tol` = (rtol, atol)
        over the elements that received terms."""
        got = np.asarray(got)
        assert got.dtype == np.float32 and got.size == self.size, (got.dtype, got.shape, self.size)
        got = got.ravel()
        assert np.isfinite(got).all(), f"{name}: {int((~np.isfinite(got)).sum())} non-finite gradient elements, " \
                                       f"first at {np.flatnonzero(~np.isfinite(got))[:5]}"
        exact, absum, count = self.exact, self.absum, self.count
        untouched = count == 0
        if init is None:
            want0 = np.zeros(self.size, np.float32)
        else:
            want0 = np.asarray(init, np.float32).ravel()
            exact = exact + want0
            absum = absum + np.abs(want0.astype(np.float64))
            count = count + 1
        bad0 = untouched & (got.view(np.uint32) != want0.view(np.uint32))
        assert not bad0.any(), f"{name}: {int(bad0.sum())} elements no term reaches were changed, e.g. " \
                               f"{np.flatnonzero(bad0)[:5]} -> {got[bad0][:5]}"
        hit = ~untouched
        if not hit.any():
            return {"case": name, "max_ratio": 0.0, "median_bound_over_old_tol": None, "elements": 0}
        err = np.abs(got[hit].astype(np.float64) - exact[hit])
        b = bound(count[hit], absum[hit], k)
        ratio = np.divide(err, b, out=np.zeros_like(err), where=b > 0)
        ratio[(b == 0) & (err > 0)] = np.inf
        worst = int(np.argmax(ratio))
        where = np.flatnonzero(hit)[worst]
        assert ratio[worst] <= 1.0, (
            f"{name}: {int((ratio > 1).sum())} of {int(hit.sum())} elements outside the rounding-error bound; worst "
            f"at flat index {where}: got {got[where]!r}, exact {exact[where]!r}, |err| {err[worst]:.3e} > bound "
            f"{b[worst]:.3e} (n={int(count[where])}, k={k})")
        rtol, atol = old_tol
        stats = {"case": name, "max_ratio": float(ratio[worst]),
                 "median_bound_over_old_tol": float(np.median(b / (atol + rtol * np.abs(exact[hit])))),
                 "elements": int(hit.sum()), "max_n": int(count.max())}
        print(f"grad-bound {name}: max |got-exact|/bound = {stats['max_ratio']:.3g}, median bound/old tol = "
              f"{stats['median_bound_over_old_tol']:.3g}, max n = {stats['max_n']}")
        return stats
