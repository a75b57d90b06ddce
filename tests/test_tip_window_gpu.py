"""GPU (-m gpu): shapes whose footprints the FP32 overlap kernel evaluates as a (MAXN-1)^2 cell window plus two tips
(aai_tip_window_ok holds), for every MAXN, against the CPU oracle."""
import numpy as np
import pytest

from common import TOL_F32_REL, f32_err

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def aai(built):
    import area_average_interpolation_b200 as m

    assert m.device_count() >= 1, "no CUDA device: the product has no CPU fallback"
    return m


# (ratio, angle): two shapes per MAXN (4: 0.55-0.7, 5: 0.37-0.45, 6: 0.3-0.33, 8: 0.2) that pass the gate
WINDOW_SHAPES = [(0.6, 37.0), (0.55, 82.0), (0.37, 8.0), (0.45, 52.0), (0.3, 68.0), (0.33, 45.0), (0.2, 23.0),
                 (0.2, 75.0)]


@pytest.mark.parametrize("ratio,angle", WINDOW_SHAPES)
def test_window_kernel_matches_oracle(aai, ratio, angle):
    from oracle import port

    rng = np.random.default_rng(int(ratio * 1000) * 100 + int(angle))
    src = rng.uniform(0.0, 4096.0, size=(203, 251)).astype(np.float32)
    iso = (117.3, 96.8)
    op = aai.AreaAverageInterpolation(arith=aai.ARITH_F32, out_dtype=np.float32)
    before = aai.launch_count()
    r = op.areaAverageInterpolation(src, 1.0, ratio, iso, angle)
    assert r.ok, r.message
    assert aai.launch_count() > before
    st, want, wiso = port.run(src, 1.0, ratio, iso, angle)
    assert st == 0 and want.shape == r.dst.shape and wiso == r.dst_isocenter
    err = f32_err(r.dst, want, 4096.0)
    assert err.max() <= TOL_F32_REL, (float(err.max()), int((err > TOL_F32_REL).sum()))

