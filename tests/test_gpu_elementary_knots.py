"""The table-driven arctangents of csrc/d2dx_math.cuh at their knots k/16, octant boundaries and signed zeros, and the small-angle
sin / cos of the RK4 stage headings on their whole domain |d| < 2^-5, through d2dx_math_probe."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    import d2d_b200
    return d2d_b200.get_engine()


def _ulp(out, ref):
    return np.abs(out - ref) / np.spacing(np.abs(ref))


def test_atan2_and_atan_at_table_knots(eng):
    knots = np.arange(17) / 16.0
    t = np.concatenate([knots, np.nextafter(knots, np.inf), np.nextafter(knots, -np.inf)])
    t = t[t >= 0]
    # the switch points between knots (odd multiples of 1/32) and their neighbours, inside and outside the diagonal
    mid = (2 * np.arange(16) + 1) / 32.0
    t = np.concatenate([t, mid, np.nextafter(mid, np.inf), np.nextafter(mid, -np.inf)])
    scale = np.array([1.0, 3.7e-3, 41.5, 1e100, 1e-100])
    ax = np.concatenate([np.full_like(t, s) for s in scale])
    ay = np.concatenate([t * s for s in scale])
    # every octant: (|x|, |y|) and the swapped (|y|, |x|) under all four sign combinations
    x = np.concatenate([sx * a for sx in (1, -1) for a in (ax, ay) for _ in (1, -1)])
    y = np.concatenate([sy * b for _ in (1, -1) for b in (ay, ax) for sy in (1, -1)])
    zeros = np.array([0.0, -0.0])
    x = np.concatenate([x, np.repeat(zeros, 2), [1.0, -1.0, 0.0, -0.0, np.nan, 2.0]])
    y = np.concatenate([y, np.tile(zeros, 2), [0.0, -0.0, 2.0, -2.0, 1.0, np.nan]])
    out = eng.math_probe(eng.to_device(x), eng.to_device(y)).cpu().numpy()
    ref2 = np.arctan2(y, x)
    nan = np.isnan(ref2)
    assert np.array_equal(np.isnan(out[2]), nan)
    exact0 = ref2 == 0
    assert np.array_equal(out[2][exact0], ref2[exact0]) and np.array_equal(np.signbit(out[2][exact0]), np.signbit(ref2[exact0]))
    ok = ~nan & ~exact0
    u = _ulp(out[2][ok], ref2[ok])
    assert u.max() <= 4, (u.max(), x[ok][np.argmax(u)], y[ok][np.argmax(u)])
    # atan on the same abscissae (x row), both octants
    v = x[np.isfinite(x)]
    out1 = eng.math_probe(eng.to_device(v), eng.to_device(v)).cpu().numpy()[3]
    ref1 = np.arctan(v)
    nz = ref1 != 0
    assert np.array_equal(out1[~nz], ref1[~nz])
    u1 = _ulp(out1[nz], ref1[nz])
    assert u1.max() <= 4, (u1.max(), v[nz][np.argmax(u1)])
    print("knots: atan2 max ulp %.2f, atan max ulp %.2f" % (u.max(), u1.max()))


def test_sincos_small_on_its_domain(eng):
    rng = np.random.default_rng(5)
    lim = 2.0 ** -5
    d = np.concatenate([rng.uniform(-lim, lim, 1 << 16), np.linspace(-lim, lim, 4097)[1:-1], [0.0, -0.0, 1e-300, np.nextafter(lim, 0)]])
    out = eng.math_probe(eng.to_device(d), eng.to_device(d)).cpu().numpy()
    dl = d.astype(np.longdouble)
    rs, rc = np.sin(dl), np.cos(dl)
    es = np.abs(out[11].astype(np.longdouble) - rs).max()
    # cos d is within an ulp of 1: beyond its rounding to double, the error is the polynomial's (< 3e-17)
    ec = (np.abs(out[12].astype(np.longdouble) - rc) - np.spacing(rc.astype(np.float64)) / 2).max()
    print("sincos_small: |sin err| %.3g, |cos err| beyond rounding %.3g" % (float(es), float(ec)))
    assert es <= 3e-17 and ec <= 3e-17, (float(es), float(ec))
