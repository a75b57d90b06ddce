"""CPU: the FP32 overlap kernel's cell window + closed-form tips (csrc/aai_cell.cuh: aai_tip_window_ok, aai_tip_strips_f32,
compiled for the host by tests/tip_window_host.cpp) against the exact FP64 area of every cell of the footprint box."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def tipmath(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("tipwin") / "libtipwin.so")
    cxx = os.environ.get("CXX", "g++")
    subprocess.run([cxx, "-O2", "-fPIC", "-shared", "-o", so, os.path.join(HERE, "tip_window_host.cpp")], check=True)
    lib = C.CDLL(so)
    lib.aai_test_tip_window_ok.argtypes = [C.c_double] * 3 + [C.c_int]
    lib.aai_test_tip_window_ok.restype = C.c_int
    lib.aai_test_tip_window.argtypes = [C.c_double] * 3 + [C.c_int] + [C.c_void_p] * 6 + [C.c_longlong]
    return lib


def _nmax(c, s, side):
    """The FP32 kernel's translation unit for the shape (aai_f32_maxn)."""
    ext32 = float(np.float32(side / 2 * (c + s) + 0.5 + 2e-6))
    n = math.floor(2.0 * ext32 + 1e-6) + 1
    return 4 if n <= 4 else 5 if n <= 5 else 6 if n <= 6 else 8 if n <= 8 else 0


def _run(lib, c, s, side, nmax, n, seed):
    rng = np.random.default_rng(seed)
    cx, cy = rng.uniform(100, 200, n), rng.uniform(100, 200, n)
    got = np.zeros((n, nmax, nmax))
    want = np.zeros((n, nmax, nmax))
    tip = np.zeros((n, 6))
    ok = np.zeros(n, dtype=np.int32)
    lib.aai_test_tip_window(c, s, side, nmax, cx.ctypes.data, cy.ctypes.data, got.ctypes.data, want.ctypes.data,
                            tip.ctypes.data, ok.ctypes.data, n)
    return got[ok == 1], want[ok == 1], tip[ok == 1]


def _random_shapes(count, seed):
    rng = np.random.default_rng(seed)
    for _ in range(count):
        theta = rng.uniform(5.0, 85.0)
        side = 1.0 / rng.uniform(0.2, 0.7)
        c, s = math.cos(math.radians(theta)), math.sin(math.radians(theta))
        yield theta, side, c, s, _nmax(c, s, side)


def test_benchmark_shapes_pass_the_gate(tipmath):
    for ratio, theta in [(0.37, 17.3), (0.37, 30.0)]:  # BASELINE configs 4 and 2
        c, s = math.cos(math.radians(theta)), math.sin(math.radians(theta))
        assert _nmax(c, s, 1 / ratio) == 5
        assert tipmath.aai_test_tip_window_ok(c, s, 1 / ratio, 5) == 1


def test_window_plus_tips_is_the_exact_box(tipmath):
    """Every shape the gate admits, every MAXN: window cells + tip strips = exact per-cell areas; tips >= 0; sum = L^2."""
    seen = set()
    for k, (theta, side, c, s, nmax) in enumerate(_random_shapes(400, 7)):
        if nmax == 0 or not tipmath.aai_test_tip_window_ok(c, s, side, nmax):
            continue
        seen.add(nmax)
        got, want, tip = _run(tipmath, c, s, side, nmax, 400, k)
        assert len(got) > 300, (theta, side)
        L2 = side * side
        err = np.abs(got - want).max()
        assert err <= 1e-6 * L2, (theta, side, nmax, err)
        assert tip.min() >= -1e-6 * L2, (theta, side, nmax, tip.min())
        assert np.abs(got.sum(axis=(1, 2)) - L2).max() <= 1e-5 * L2, (theta, side, nmax)
    assert seen == {4, 5, 6, 8}


def test_gate_rejects_overlapping_tips(tipmath):
    """Shapes whose tips reach the window's outer corner (or each other) fail the gate, and there window + tips would
    really miss footprint area; every sampled shape where that happens is one the gate rejects."""
    misses = 0
    for k, (theta, side, c, s, nmax) in enumerate(_random_shapes(300, 11)):
        if nmax == 0:
            continue
        got, want, _ = _run(tipmath, c, s, side, nmax, 300, 1000 + k)
        if len(got) and np.abs(got - want).max() > 1e-6 * side * side:
            misses += 1
            assert not tipmath.aai_test_tip_window_ok(c, s, side, nmax), (theta, side, nmax)
    assert misses > 20
    # 45 deg, L = 1.98 (MAXN 4): tips up to 0.8 wide, w (c+s) = 1.13 > L c s = 0.99 -- the two tips meet in the corner
    c = s = math.sqrt(0.5)
    assert _nmax(c, s, 1.98) == 4
    assert not tipmath.aai_test_tip_window_ok(c, s, 1.98, 4)
    got, want, _ = _run(tipmath, c, s, 1.98, 4, 2000, 3)
    assert want[:, 3, 3].max() > 1e-3  # the corner cell beyond both tips' strips holds footprint area
