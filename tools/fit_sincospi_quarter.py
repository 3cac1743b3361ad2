"""Generator of the coefficients of sincospi_quarter (csrc/drt_render.cuh): sin(pi u) and cos(pi u) for |u| <= 1/4 as polynomials in
v = u^2, fitted in float64 with numpy and rounded to float32.

    sin(pi u) = u * S0 + (u v) * (S1 + v (S2 + v S3))        S0 = pi rounded to float32, fixed
    cos(pi u) = 1 + v * (C1 + v (C2 + v (C3 + v C4)))

Each fit is a minimax fit (Lawson's iteratively reweighted least squares on a dense Chebyshev grid of v in [0, 1/16]) of the relative
error of sin and of the absolute error of cos.  tests/test_trace_trim.py checks the float32 evaluation of the stored coefficients
against float64 sin and cos.  Run: python tools/fit_sincospi_quarter.py"""
import numpy as np


def lawson(A, t, iters=300):
    """Coefficients c minimising max |A c - t| (Lawson's algorithm)."""
    w = np.full(len(t), 1.0 / len(t))
    for _ in range(iters):
        sw = np.sqrt(w)
        c = np.linalg.lstsq(A * sw[:, None], t * sw, rcond=None)[0]
        e = np.abs(A @ c - t)
        w = w * e
        w /= w.sum()
    return c


def fit():
    v = (1.0 - np.cos(np.linspace(0.0, np.pi, 6001)))[1:] / 32.0        # (0, 1/16]
    u = np.sqrt(v)
    s0 = float(np.float32(np.pi))
    # sin: relative error of u (S0 + v P(v)), i.e. of S0 + v P(v) against sin(pi u) / u; divide the rows by it to weigh relatively
    ratio = np.sin(np.pi * u) / u
    A = np.stack([v ** (k + 1) for k in range(3)], 1) / ratio[:, None]
    s = lawson(A, (ratio - s0) / ratio)
    # cos: absolute error of 1 + v Q(v)
    A = np.stack([v ** (k + 1) for k in range(4)], 1)
    c = lawson(A, np.cos(np.pi * u) - 1.0)
    return [np.float32(s0)] + [np.float32(x) for x in s], [np.float32(x) for x in c]


if __name__ == "__main__":
    S, Cc = fit()
    for i, x in enumerate(S):
        print(f"S{i} = {float(x).hex()}  /* {float(x):.9e}f */")
    for i, x in enumerate(Cc):
        print(f"C{i + 1} = {float(x).hex()}  /* {float(x):.9e}f */")
