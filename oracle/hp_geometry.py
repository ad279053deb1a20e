"""High-precision references for the geometry kernels (test infrastructure).

* ``dlt_*``: the DLT of ``triangulate_multi_view`` (epipolar_matching.py:118-127) against an mpmath SVD at ``DPS``
  digits of the float64 matrix A the kernels build, with the backward (residual) and forward (angle) errors of a
  computed solution expressed in units of eps * sigma_1.
* ``epiline_exact`` / ``line_point_exact`` / ``epipolar_error_exact``: the epipolar distance with every float64 operation
  spelled out and correctly rounded, the fused ones through an exact ``Fraction`` FMA (Python 3.12 has no ``math.fma``).
  The operation order is the one the reference's BLAS calls use and the kernels copy (csrc/common.cuh): ``F @ p``
  accumulates its products in the order 1, 0, 2 (dgemv), ``F.T @ p``, ``np.dot`` and the 2-norm in the order 0, 1, 2.
"""
from __future__ import annotations

import math
from fractions import Fraction

import mpmath as mp
import numpy as np

DPS = 60
EPS = float(np.finfo(np.float64).eps)        # 2^-52


# ---------------------------------------------------------------------------------------------------------------------
# DLT triangulation
# ---------------------------------------------------------------------------------------------------------------------
def dlt_matrix(P, pts):
    """A (2V x 4, float64) exactly as the kernels build it: rows x*P[2] - P[0], y*P[2] - P[1], one rounding per op."""
    P = np.asarray(P, np.float64)
    pts = np.asarray(pts, np.float64)
    A = np.empty((2 * len(P), 4))
    for v in range(len(P)):
        A[2 * v] = pts[v, 0] * P[v, 2] - P[v, 0]        # NumPy never fuses the multiply into the subtraction
        A[2 * v + 1] = pts[v, 1] * P[v, 2] - P[v, 1]
    return A


class DltRef:
    """Singular values (descending) and the unit right singular vector v* of sigma_4 of a float64 A, at DPS digits."""

    def __init__(self, A):
        with mp.workdps(DPS):
            self.A = mp.matrix(np.asarray(A, np.float64).tolist())
            _, S, Vt = mp.svd_r(self.A)
            order = sorted(range(4), key=lambda i: -S[i])
            self.sigma = [S[i] for i in order]
            self.v = [Vt[order[3], j] for j in range(4)]
            if self.v[3] < 0:
                self.v = [-x for x in self.v]
        self.s1 = float(self.sigma[0])
        self.gap = float(self.sigma[2] - self.sigma[3])

    def unit_from_X(self, X):
        """The unit homogeneous vector (X, 1) / ||(X, 1)|| of a computed X, at DPS digits (sign of v*)."""
        with mp.workdps(DPS):
            h = [mp.mpf(float(x)) for x in X] + [mp.mpf(1)]
            nrm = mp.sqrt(mp.fsum(x * x for x in h))
            return [x / nrm for x in h]

    def residual_ratio(self, X):
        """(||A v|| - sigma_4) / (eps sigma_1) for the computed X: the backward error of v in units of eps ||A||."""
        if not np.all(np.isfinite(X)):
            return math.inf
        v = self.unit_from_X(X)
        with mp.workdps(DPS):
            Av = self.A * mp.matrix(v)
            r = mp.sqrt(mp.fsum(x * x for x in Av))
            return float((r - self.sigma[3]) / (EPS * self.sigma[0]))

    def angle_ratio(self, X):
        """sin angle(v, v*) * (sigma_3 - sigma_4) / (eps sigma_1): the forward error against the first-order bound."""
        if not np.all(np.isfinite(X)):
            return math.inf
        v = self.unit_from_X(X)
        with mp.workdps(DPS):
            c = mp.fsum(a * b for a, b in zip(v, self.v))
            s = mp.sqrt(max(mp.mpf(0), 1 - c * c))
            return float(s * (self.sigma[2] - self.sigma[3]) / (EPS * self.sigma[0]))

    def X_star(self):
        with mp.workdps(DPS):
            return [self.v[i] / self.v[3] for i in range(3)]

    def X_ratio(self, X):
        """||X - X*|| / (eps sigma_1 / gap * (1 + ||X*||^2) + eps ||X*||): the error of the dehomogenised point against
        what an angle error of eps sigma_1 / gap and the final division allow (|v*_3| = 1 / sqrt(1 + ||X*||^2))."""
        if not np.all(np.isfinite(X)):
            return math.inf
        with mp.workdps(DPS):
            Xs = self.X_star()
            d = mp.sqrt(mp.fsum((mp.mpf(float(a)) - b) ** 2 for a, b in zip(X, Xs)))
            n2 = mp.fsum(b * b for b in Xs)
            bound = EPS * self.sigma[0] / (self.sigma[2] - self.sigma[3]) * (1 + n2) + EPS * mp.sqrt(n2)
            return float(d / bound)


def numpy_dlt(A):
    """NumPy's answer on the same A: the oracle's triangulate_multi_view after the matrix is built."""
    _, _, Vt = np.linalg.svd(A)
    X = Vt[-1]
    return X[:3] / X[3]


# ---------------------------------------------------------------------------------------------------------------------
# epipolar distance, operation by operation
# ---------------------------------------------------------------------------------------------------------------------
def fma(a, b, c):
    """Correctly rounded a * b + c of three float64 values (float() of a Fraction rounds half to even)."""
    return float(Fraction(a) * Fraction(b) + Fraction(c))


def epiline_exact(F, transpose, x, y):
    """(l, ok): the normalised line F @ (x, y, 1) (transpose 0) or F.T @ (x, y, 1) (transpose 1); ok = norm > 1e-8."""
    F = np.asarray(F, np.float64)
    x, y = float(x), float(y)
    if not transpose:
        l = [fma(float(F[r, 2]), 1.0, fma(float(F[r, 0]), x, float(F[r, 1]) * y)) for r in range(3)]
    else:
        l = [fma(float(F[2, c]), 1.0, fma(float(F[1, c]), y, float(F[0, c]) * x)) for c in range(3)]
    nrm = math.sqrt(fma(l[1], l[1], l[0] * l[0]))
    if nrm > 1e-8:
        return [l[0] / nrm, l[1] / nrm, l[2] / nrm], True
    return l, False


def line_point_exact(l, x, y):
    return abs(fma(l[2], 1.0, fma(l[1], float(y), l[0] * float(x))))


def epipolar_error_exact(F, p1, p2):
    """epipolar_error(pt1, pt2, F) (epipolar_matching.py:5-28), 9999 for a degenerate line."""
    l2, ok2 = epiline_exact(F, 0, p1[0], p1[1])
    l1, ok1 = epiline_exact(F, 1, p2[0], p2[1])
    d1 = line_point_exact(l1, p1[0], p1[1]) if ok1 else 9999.0
    d2 = line_point_exact(l2, p2[0], p2[1]) if ok2 else 9999.0
    return 0.5 * (d1 + d2)
