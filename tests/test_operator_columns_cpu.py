"""The column helpers of tests/common.py without a GPU: on the small geometries of the adjoint's transpose test, where
the dense operator W is cheap, column_window must hold every non-zero of each column and oracle_column must return that
column bitwise -- for every mode, quadrant and expansion factor 1-4.  The full-size GPU tests
(test_operator_columns_gpu.py) trust these helpers for their reference."""
import numpy as np
import pytest

from common import column_window, oracle_column
from test_adjoint_gpu import GEOMS

SMALL = [g for g in GEOMS if g[2] == 1]


@pytest.fixture(scope="module")
def aai(built):
    import area_average_interpolation_b200 as m

    m.lib()
    return m


@pytest.fixture(scope="module")
def oracle(built):
    from oracle import port

    return port


def test_geometries_cover_every_quadrant_and_scale(aai):
    plans = [aai.make_plan(w, h, 1.0, r, iso, a) for w, h, _, r, a, iso in SMALL]
    assert {p.quadrant for p in plans} == {0, 1, 2, 3}
    assert {p.scale for p in plans} == {1, 2, 3, 4}
    assert {p.axis_aligned for p in plans} == {0, 1}


@pytest.mark.parametrize("mode", [1, 2, 3])
@pytest.mark.parametrize("w,h,ch,ratio,angle,iso", SMALL)
def test_column_helper_is_the_dense_operator(aai, oracle, w, h, ch, ratio, angle, iso, mode):
    plan = aai.make_plan(w, h, 1.0, ratio, iso, angle)
    impulse = np.zeros((h, w), dtype=np.uint8)
    for sy in range(h):
        for sx in range(w):
            e = np.zeros((h, w))
            e[sy, sx] = 1.0
            st, dense, _ = oracle.run(e, 1.0, ratio, iso, angle, mode=mode)
            assert st == 0 and dense.shape == (plan.dst_h, plan.dst_w)
            y0, y1, x0, x1 = column_window(plan, sx, sy)
            outside = dense.copy()
            outside[y0:y1, x0:x1] = 0.0
            assert not outside.any(), ("non-zero outside the window", sx, sy, (y0, y1, x0, x1))
            win, col = oracle_column(oracle, impulse, (1.0, ratio, iso, angle), sx, sy, 0, mode)
            assert win == (y0, y1, x0, x1)
            assert np.array_equal(col, dense[y0:y1, x0:x1]), (sx, sy)
    assert not impulse.any()


def test_column_of_one_channel_of_a_multichannel_impulse(aai, oracle):
    w, h, ratio, angle, iso = 16, 12, 1.7, 45.0, (7.5, 5.5)
    impulse = np.zeros((h, w, 3), dtype=np.float32)
    for c in range(3):
        e = np.zeros((h, w))
        e[5, 9] = 1.0
        _, dense, _ = oracle.run(e, 1.0, ratio, iso, angle)
        (y0, y1, x0, x1), col = oracle_column(oracle, impulse, (1.0, ratio, iso, angle), 9, 5, c, 1)
        assert np.array_equal(col, dense[y0:y1, x0:x1]) and col.any()
