"""Adjoint of the resampling operator without a GPU: every refusal of aai_run_device_adjoint happens on the host, before
any CUDA call, with AAI_ERR_ARGUMENT and a message naming the entry point; a failed plan's status passes through; the
torch entry point refuses CPU tensors."""
import ctypes as C

import numpy as np
import pytest

WHO = "aai_run_device_adjoint"


@pytest.fixture(scope="module")
def aai(built):
    import area_average_interpolation_b200 as m

    m.lib()
    return m


@pytest.fixture(scope="module")
def plan(aai):
    return aai.make_plan(40, 30, 1.0, 0.5, (20.0, 15.0), 17.3)


def _img(aai, shape, dtype):
    return aai._host_image(np.zeros(shape, dtype=dtype))


def _refused(aai, plan, canvas, src, mode=1, n=None):
    canvas = canvas if isinstance(canvas, list) else [canvas]
    src = src if isinstance(src, list) else [src]
    with pytest.raises(aai.AaiError) as ei:
        aai.run_device_adjoint(plan, canvas, src, mode=mode)
    assert ei.value.status == aai.ERR_ARGUMENT
    msg = aai.last_error()
    assert msg.startswith(WHO + ":"), msg
    return msg


def test_refusals_are_argument_errors_before_cuda(aai, plan):
    ch, cw = plan.dst_h, plan.dst_w
    good_c, good_s = _img(aai, (ch, cw), np.float64), _img(aai, (30, 40), np.float64)
    L = aai.lib()
    # null pointers and an empty list
    assert L.aai_run_device_adjoint(None, 1, C.byref(good_c), C.byref(good_s), 1, 0, None) == aai.ERR_ARGUMENT
    assert aai.last_error().startswith(WHO + ":")
    assert L.aai_run_device_adjoint(C.byref(plan), 1, None, C.byref(good_s), 1, 0, None) == aai.ERR_ARGUMENT
    assert L.aai_run_device_adjoint(C.byref(plan), 1, C.byref(good_c), None, 1, 0, None) == aai.ERR_ARGUMENT
    assert L.aai_run_device_adjoint(C.byref(plan), 1, C.byref(good_c), C.byref(good_s), 0, 0, None) == aai.ERR_ARGUMENT
    assert aai.last_error().startswith(WHO + ":")
    null_data = aai.Image(*[getattr(good_c, f) for f, _ in aai.Image._fields_])
    null_data.data = None
    _refused(aai, plan, null_data, good_s)
    # the mode
    for mode in (0, 4, -1):
        assert "mode" in _refused(aai, plan, good_c, good_s, mode=mode)
    # element types: integer gradients, mixed float types
    assert "float32 or float64" in _refused(aai, plan, _img(aai, (ch, cw), np.uint8), _img(aai, (30, 40), np.uint8))
    _refused(aai, plan, _img(aai, (ch, cw), np.uint16), _img(aai, (30, 40), np.uint16))
    _refused(aai, plan, good_c, _img(aai, (30, 40), np.float32))
    _refused(aai, plan, _img(aai, (ch, cw), np.float32), good_s)
    # channel counts differ
    assert "channels" in _refused(aai, plan, _img(aai, (ch, cw, 3), np.float64), good_s)
    # not whole images: a band of rows
    band = _img(aai, (ch, cw), np.float64)
    band.y0, band.rows, band.height = 1, ch - 1, ch
    assert "whole" in _refused(aai, plan, band, good_s)
    short = _img(aai, (30, 40), np.float64)
    short.rows = 29
    _refused(aai, plan, good_c, short)
    # sizes that do not match the plan
    assert "does not match the plan" in _refused(aai, plan, _img(aai, (ch + 1, cw), np.float64), good_s)
    _refused(aai, plan, good_c, _img(aai, (30, 41), np.float64))
    # the second image of a list is checked too
    _refused(aai, plan, [good_c, good_c], [good_s, _img(aai, (31, 40), np.float64)])


def test_failed_plan_status_passes_through(aai):
    bad = aai.make_plan(40, 30, -1.0, 0.5, (20.0, 15.0), 17.3)
    assert bad.status not in (aai.AAI_OK, aai.ERR_ARGUMENT)
    c, s = _img(aai, (4, 4), np.float64), _img(aai, (30, 40), np.float64)
    assert aai.lib().aai_run_device_adjoint(C.byref(bad), 1, C.byref(c), C.byref(s), 1, 0, None) == bad.status


def test_torch_entry_refuses_cpu_tensors(aai, plan):
    import torch

    src = torch.zeros((30, 40), dtype=torch.float64)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        aai.resample(src, plan)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        aai.resample_adjoint(torch.zeros((plan.dst_h, plan.dst_w)), plan)


def test_torch_is_not_imported_with_the_package():
    import subprocess
    import sys

    code = ("import sys, area_average_interpolation_b200 as a; from area_average_interpolation_b200 import *; "
            "assert 'torch' not in sys.modules; assert callable(a.resample) and 'torch' in sys.modules")
    import os

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.run([sys.executable, "-c", code], cwd=root, check=True)
