"""Fits the two fp32 polynomials of the equidistant fisheye projection (csrc/egs_math.cuh fisheye_theta_over_r) and
prints them as C literals.  Offline tool: its output is pasted into egs_math.cuh and tests/camera_model_reference.py.

  P(u) ~ atan(sqrt(u)) / sqrt(u)                    on u in [0, 1], P(0) = 1 exactly
  H(u) ~ (1 / (1 + u) - atan(sqrt(u)) / sqrt(u)) / u on u in [0, 1]  (= z^3 g, g = (1/r) d(theta/r)/dr for r <= z)

Each is fitted by weighted least squares on Chebyshev nodes (relative error), one coefficient at a time from the
constant term up: a coefficient is rounded to fp32 and the remaining ones are fitted again around it, so the
rounding of the literals is absorbed by the higher terms.  The printed error is that of an fp32 Horner evaluation
(mul then add, no FMA) against mpmath.

    python scripts/fit_fisheye_theta.py [--degree 11]
"""
from __future__ import annotations

import argparse

import mpmath
import numpy as np

mpmath.mp.dps = 40


def p_exact(u: float) -> float:
    if u == 0:
        return 1.0
    s = mpmath.sqrt(mpmath.mpf(u))
    return float(mpmath.atan(s) / s)


def h_exact(u: float) -> float:
    if u == 0:
        return -2.0 / 3.0
    m = mpmath.mpf(u)
    s = mpmath.sqrt(m)
    return float((1 / (1 + m) - mpmath.atan(s) / s) / m)


def fit(fn, degree: int, c0=None, n_nodes: int = 4000):
    k = np.arange(n_nodes)
    u = 0.5 - 0.5 * np.cos(np.pi * (k + 0.5) / n_nodes)  # Chebyshev nodes on [0, 1]
    f = np.array([fn(x) for x in u])
    coeffs = []
    fixed = 0.0 * u
    if c0 is not None:
        coeffs.append(np.float32(c0))
        fixed = fixed + float(coeffs[0])
    for j in range(len(coeffs), degree + 1):
        cols = np.stack([u ** i for i in range(j, degree + 1)], 1)
        w = 1.0 / np.abs(f)
        sol, *_ = np.linalg.lstsq(cols * w[:, None], (f - fixed) * w, rcond=None)
        cj = np.float32(sol[0])
        coeffs.append(cj)
        fixed = fixed + float(cj) * u ** j
    return np.array(coeffs, dtype=np.float32)


def horner32(c: np.ndarray, u: np.ndarray) -> np.ndarray:
    u = u.astype(np.float32)
    p = np.full_like(u, c[-1])
    for cj in c[-2::-1]:
        p = (p * u).astype(np.float32)
        p = (p + cj).astype(np.float32)
    return p


def report(name: str, c: np.ndarray, fn) -> None:
    u = np.linspace(0.0, 1.0, 20001).astype(np.float32)
    ref = np.array([fn(float(x)) for x in u])
    got = horner32(c, u).astype(np.float64)
    ulp = np.spacing(np.abs(ref).astype(np.float32)).astype(np.float64)
    print(f"// {name}: max |error| {np.max(np.abs(got - ref) / ulp):.3f} ulp (fp32 Horner, u in [0, 1])")
    print(", ".join(f"{float(x)!r}f" for x in c))


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--degree", type=int, default=11)
    args = ap.parse_args()
    report("P", fit(p_exact, args.degree, c0=1.0), p_exact)
    report("H", fit(h_exact, args.degree), h_exact)


if __name__ == "__main__":
    main()
