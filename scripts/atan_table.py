"""Constants of the table-driven arctangent in drone-sim-python_b200/csrc/d2dx_math.cuh (fm::atan2, fm::atan).

atan(t), 0 <= t <= 1, is reduced to the nearest knot c = k/16:  atan(t) = atan(c) + atan(t'),  t' = (t - c) / (1 + c t),
|t'| <= 1/32 plus the error of the 20-bit estimate of t that picks k.  atan(t') = t' (1 + z P(z)), z = t'^2, where P is the
degree-4 Taylor polynomial of (atan(t)/t - 1)/z economised to degree 3 by the shifted Chebyshev polynomial T_4 on [0, a^2].

Prints the 68 table entries (k = 0..16: atan(k/16), then pi/2 - atan(k/16), pi - atan(k/16) and pi/2 + atan(k/16), each rounded to
the nearest double: the four ways the knot enters atan2 in its four half-quadrants) and the four
coefficients of -P (highest power first, the order the kernel evaluates them in), and checks in exact rational arithmetic that
the relative truncation error |1 + z P_double(z) - atan(t')/t'| of the rounded coefficients stays below 2^-56 on the whole interval.

    python scripts/atan_table.py            # prints the constants, exits non-zero if the bound does not hold
"""
from decimal import Decimal, getcontext
from fractions import Fraction as F
import sys

getcontext().prec = 60
N_KNOTS = 16                                   # knots k/16, k = 0..16
A = F(1, 2 * N_KNOTS) + F(1, 2 ** 18)          # |t'| bound: half a knot spacing + the estimate's error (< 2^-19), with margin
BOUND = F(1, 2 ** 56)


def atan_dec(x):
    """atan of a Decimal 0 <= x <= 1 by Euler's series  sum 2^2n (n!)^2 / (2n+1)! x^(2n+1) / (1+x^2)^(n+1) (ratio <= 1/2)."""
    y = x * x / (1 + x * x)
    term = x / (1 + x * x)
    s, n = term, 0
    while abs(term) > Decimal(10) ** -58:
        n += 1
        term = term * y * (2 * n) / (2 * n + 1)
        s += term
    return s


def pi_dec():
    return 4 * (4 * atan_dec(Decimal(1) / 5) - atan_dec(Decimal(1) / 239))


def table():
    pi = pi_dec()
    a = [atan_dec(Decimal(k) / N_KNOTS) for k in range(N_KNOTS + 1)]
    return [float(v) for v in a] + [float(pi / 2 - v) for v in a] + [float(pi - v) for v in a] + [float(pi / 2 + v) for v in a]


def chebyshev_t(n):
    """coefficients (lowest power first) of the Chebyshev polynomial T_n"""
    t0, t1 = [F(1)], [F(0), F(1)]
    if n == 0:
        return t0
    for _ in range(n - 1):
        t2 = [F(0)] + [2 * c for c in t1]
        for i, c in enumerate(t0):
            t2[i] -= c
        t0, t1 = t1, t2
    return t1


def poly_compose_affine(p, alpha, beta):
    """coefficients of p(alpha z + beta) in z (lowest power first)"""
    out = [F(0)] * len(p)
    powk = [F(1)]                                # (alpha z + beta)^k
    for c in p:
        for i, v in enumerate(powk):
            out[i] += c * v
        nxt = [F(0)] * (len(powk) + 1)
        for i, v in enumerate(powk):
            nxt[i] += beta * v
            nxt[i + 1] += alpha * v
        powk = nxt
    return out


def coefficients():
    """P(z) ~ (atan(t)/t - 1)/z: Taylor G(z) = sum_{n=1..5} (-1)^n z^(n-1) / (2n+1), its z^4 term removed with T_4(2z/A^2 - 1)"""
    g = [F((-1) ** n, 2 * n + 1) for n in range(1, 6)]
    a2 = A * A
    t4 = poly_compose_affine(chebyshev_t(4), 2 / a2, F(-1))    # leading coefficient 2^7 (2/a2)^4
    scale = g[4] / t4[4]
    p = [g[i] - scale * t4[i] for i in range(4)]
    return p, abs(scale)                          # |G - P| <= |scale| on [0, A^2]


def poly_eval(c, z):
    v = F(0)
    for x in reversed(c):
        v = v * z + x
    return v


def check(p_double):
    """max over z in [0, A^2] of |z P_double(z) - (atan(t)/t - 1)|, bounded rigorously:
    |z P_double - z G5| on a grid plus the grid spacing times a bound of its derivative, plus the Taylor tail z^6 / 13."""
    g5 = [F((-1) ** n, 2 * n + 1) for n in range(1, 6)]
    d = [F(0)] + [F(pc) - gc for pc, gc in zip(p_double + [0.0], g5)]      # z (P_double(z) - G5(z)), lowest power first
    a2 = A * A
    m = 4096
    grid_max = max(abs(poly_eval(d, a2 * j / m)) for j in range(m + 1))
    dprime = sum(i * abs(c) * a2 ** (i - 1) for i, c in enumerate(d) if i)
    tail = a2 ** 6 / 13
    return grid_max + dprime * a2 / m / 2 + tail


def main():
    tab = table()
    p, econ = coefficients()
    p_double = [float(c) for c in p]
    err = check(p_double)
    print("// atan(k/16), pi/2 - atan(k/16), pi - atan(k/16), pi/2 + atan(k/16), k = 0..16")
    for k in range(0, len(tab), 6):
        print("    " + " ".join(f"{v!r}," for v in tab[k:k + 6]))
    print("// -P, highest power first:", ", ".join(repr(-c) for c in reversed(p_double)))
    print(f"economisation term {float(econ * A * A):.3e}, bound on the relative truncation error {float(err):.3e} "
          f"(2^-56 = {float(BOUND):.3e}), |t'| <= {float(A):.6g}")
    if err >= BOUND:
        sys.exit("bound not met")
    return tab, p_double, err


if __name__ == "__main__":
    main()
