"""The Riccati warm start of the DFFF rollout on the CPU: csrc/host_check.cu compiles care_gain (d2dx_device.cuh) with its
9-double state -- the previous solution and the last three changes, cubically extrapolated -- and this test runs it along
references of bench.py's C5 population, step by step as the rollout kernel does."""
import ctypes as C
import os

import numpy as np
import pytest

from test_care_math import G, scipy_gain3

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "native", "libd2dx_hostcheck.so")
FAST, LOOP = 2, 1                      # care_gain: straight-line step accepted / fallback loop converged
QR = (1., 0.1, 8., 1.)                 # the default gains: q_pos, q_psi, r_phi, r_v


@pytest.fixture(scope="module")
def host():
    if not os.path.exists(LIB):
        pytest.fail(f"{LIB} is missing: build it with `python __graft_entry__.py` (make -C drone-sim-python_b200/csrc)")
    lib = C.CDLL(LIB)
    dp = C.POINTER(C.c_double)
    lib.d2dx_host_care_gain9.argtypes = [dp, C.c_double, C.c_double, C.c_int, dp, dp]
    return lib


def _ptr(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def c5_reference(n, T, seed, dt=0.01):
    """Air speed and bank of the flat reference (d2d/guidance.py:23-47) along n circles drawn as bench.workload draws them."""
    from bench import workload
    w = workload(n, seed)
    t = np.arange(T) * dt
    for b in range(n):
        om, r = w["v"][b] / w["r"][b], w["r"][b]
        a = om * t + w["a0"][b]
        vax, vay = -om * r * np.sin(a) - w["wind"][b, 0], om * r * np.cos(a) - w["wind"][b, 1]
        va = np.hypot(vax, vay)
        z = (-om ** 2 * r * np.sin(a) * vax + om ** 2 * r * np.cos(a) * vay) / va / G
        yield va, np.arctan(z)


def _run(host, v, phi):
    """care_gain along (v, phi); returns the per-step status, the solutions (C, S, al) and the gains."""
    qr = np.array(QR)
    st, K = np.zeros(9), np.zeros(6)
    res, sol, Ks = [], [], []
    for k in range(len(v)):
        res.append(host.d2dx_host_care_gain9(_ptr(qr), v[k], phi[k], 1 if k == 0 else 0, _ptr(st), _ptr(K)))
        sol.append(st[:3].copy())
        Ks.append(K.copy())
    return np.array(res), np.array(sol), np.array(Ks)


def _converged(host, v, phi):
    qr = np.array(QR)
    out = []
    for k in range(len(v)):
        st, K = np.zeros(9), np.zeros(6)
        assert host.d2dx_host_care_gain9(_ptr(qr), v[k], phi[k], 1, _ptr(st), _ptr(K)) == LOOP
        out.append(st[:3].copy())
    return np.array(out)


def test_cubic_warm_start_along_c5_references(host):
    """One Newton step from the cubic extrapolation: K within 1e-10 of SciPy, the state within 1e-13 of a converged solve,
    and the fallback loop only while the history builds up after the cold start (steps 1-3)."""
    worst_K = worst_x = 0.
    fallbacks = warm = 0
    for v, phi in c5_reference(12, 3000, seed=2024):
        res, sol, Ks = _run(host, v, phi)
        assert (res > 0).all()
        assert (res[1:4] == LOOP).all()                        # history building up: constant, linear, quadratic starts
        fallbacks += int((res[4:] != FAST).sum()); warm += len(res) - 4
        ref = _converged(host, v, phi)
        th, th_ref = np.arctan2(sol[:, 1], sol[:, 0]), np.arctan2(ref[:, 1], ref[:, 0])
        worst_x = max(worst_x, np.abs(th - th_ref).max(), (np.abs(sol[:, 2] - ref[:, 2]) / ref[:, 2]).max())
        for k in range(0, len(v), 97):
            Kref = scipy_gain3(v[k], phi[k], (QR[0], QR[1]), (QR[2], QR[3]))
            worst_K = max(worst_K, np.abs(Ks[k].reshape(2, 3) - Kref).max() / np.abs(Kref).max())
    assert worst_K < 1e-10, worst_K
    assert worst_x < 1e-13, worst_x
    assert fallbacks / warm < 1e-3, (fallbacks, warm)


def test_warm_start_falls_back_at_a_corner_and_rebuilds(host):
    """A jump of the reference (trajectory corner) takes the loop, resets the history, and the straight-line step returns
    once three new changes are known."""
    t = np.arange(0, 20, 0.01)
    v = 10 + 3 * np.sin(0.3 * t); phi = 0.4 * np.sin(0.5 * t)
    v[1200:] += 6.; phi[1200:] -= 0.5
    res, sol, Ks = _run(host, v, phi)
    assert (res > 0).all()
    assert (res[1200:1204] == LOOP).all()
    assert (res[4:1200] == FAST).all() and (res[1204:] == FAST).all()
    for k in list(range(1195, 1210)) + list(range(0, len(t), 53)):
        Kref = scipy_gain3(v[k], phi[k], (QR[0], QR[1]), (QR[2], QR[3]))
        assert np.abs(Ks[k].reshape(2, 3) - Kref).max() / np.abs(Kref).max() < 1e-10

