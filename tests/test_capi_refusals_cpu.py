"""C ABI refusals without a GPU: each is decided on the host before any CUDA call, so the exact status and
aai_last_error() text are the same on a box without a device.  Pins the messages of aai_run_device, aai_run_device_batch,
aai_expand_device, the row copies and the host-buffer entry points' image checks."""
import ctypes as C

import numpy as np
import pytest


@pytest.fixture(scope="module")
def aai(built):
    import area_average_interpolation_b200 as m

    m.lib()
    return m


@pytest.fixture(scope="module")
def plan(aai):
    return aai.make_plan(64, 48, 1.0, 0.5, (32, 24), 10.0)


def _img(aai, shape, dtype=np.float32):
    return aai._host_image(np.zeros(shape, dtype=dtype))


def _refusal(aai, status):
    return status, aai.last_error()


def test_run_device_refusals(aai, plan):
    L = aai.lib()
    si, di = _img(aai, (48, 64)), _img(aai, (plan.dst_h, plan.dst_w))
    H, W = plan.dst_h, plan.dst_w

    def run(p, src, dst, mode=aai.MODE_AREA_AVERAGE, arith=aai.ARITH_F32, row0=0, row1=H):
        return _refusal(aai, L.aai_run_device(p, mode, arith, C.byref(src), C.byref(dst), row0, row1, 0, None))

    assert run(None, si, di) == (aai.ERR_ARGUMENT, "aai_run_device: null plan")
    mismatch = (aai.ERR_ARGUMENT, f"aai_run_device: images do not match the plan (src 64x48, canvas {W}x{H})")
    assert run(C.byref(plan), si, _img(aai, (5, 5))) == mismatch
    assert run(C.byref(plan), _img(aai, (48, 63)), di) == mismatch
    assert run(C.byref(plan), si, _img(aai, (H, W, 3))) == mismatch  # channel counts differ
    for mode in (0, 4):
        assert run(C.byref(plan), si, di, mode=mode) == (aai.ERR_ARGUMENT,
                                                        "aai_run_device: interpolation mode must be 1, 2 or 3")
    for arith in (-1, 5):
        assert run(C.byref(plan), si, di, arith=arith) == (aai.ERR_ARGUMENT, f"aai_run_device: unknown arithmetic {arith}")
    assert run(C.byref(plan), si, di, row0=3, row1=H + 1) == (
        aai.ERR_ARGUMENT, f"aai_run_device: rows [3,{H + 1}) outside the destination band")
    band = _img(aai, (10, W))
    band.y0, band.rows, band.height = 4, 10, H
    assert run(C.byref(plan), si, band, row0=2, row1=8) == (
        aai.ERR_ARGUMENT, "aai_run_device: rows [2,8) outside the destination band")
    part = aai.Image(si.data, si.pitch_bytes, si.width, si.height, 0, 8, si.dtype, si.channels)
    _, _, sy0, sy1 = aai.band_source_window(plan, 0, H)
    assert sy1 > 8
    assert run(C.byref(plan), part, di) == (
        aai.ERR_ARGUMENT, f"aai_run_device: source rows [{sy0},{sy1}) needed, [0,8) present")


def test_run_device_batch_bad_argument(aai, plan):
    L = aai.lib()
    si, di = _img(aai, (48, 64)), _img(aai, (plan.dst_h, plan.dst_w))
    want = (aai.ERR_ARGUMENT, "aai_run_device_batch: bad argument")
    for p, s, d, n in [(None, C.byref(si), C.byref(di), 1), (C.byref(plan), None, C.byref(di), 1),
                       (C.byref(plan), C.byref(si), None, 1), (C.byref(plan), C.byref(si), C.byref(di), 0)]:
        assert _refusal(aai, L.aai_run_device_batch(p, 1, aai.ARITH_F32, s, d, n, 0, None)) == want


def test_expand_device_partial_image(aai, plan):
    L = aai.lib()
    want = (aai.ERR_ARGUMENT, f"aai_expand_device: need a whole source image and a whole {plan.mod_w} x {plan.mod_h} "
                              "image of the same type")
    si, mod = _img(aai, (48, 64)), _img(aai, (plan.mod_h, plan.mod_w))
    part = aai.Image(si.data, si.pitch_bytes, si.width, si.height, 0, 47, si.dtype, si.channels)
    assert _refusal(aai, L.aai_expand_device(C.byref(plan), C.byref(part), C.byref(mod), 0, None)) == want
    mod.rows = plan.mod_h - 1
    assert _refusal(aai, L.aai_expand_device(C.byref(plan), C.byref(si), C.byref(mod), 0, None)) == want


def test_image_copy_refusals(aai):
    L = aai.lib()
    a, b = _img(aai, (20, 16)), _img(aai, (20, 16))
    narrow, wide_u8 = _img(aai, (20, 15)), _img(aai, (20, 16), np.uint8)

    def copy_rows(dst, src, y0, y1):
        return _refusal(aai, L.aai_image_copy_rows(C.byref(dst), C.byref(src), y0, y1, 0, None))

    for dst, src in [(a, narrow), (a, wide_u8)]:
        assert copy_rows(dst, src, 0, 5) == (aai.ERR_ARGUMENT,
                                             "aai_image_copy_rows: incompatible images or rows [0,5) not present")
    assert copy_rows(a, b, 3, 21) == (aai.ERR_ARGUMENT,
                                      "aai_image_copy_rows: incompatible images or rows [3,21) not present")
    assert copy_rows(a, b, 5, 4) == (aai.ERR_ARGUMENT,
                                     "aai_image_copy_rows: incompatible images or rows [5,4) not present")

    incompatible = (aai.ERR_ARGUMENT, "aai_image copy: incompatible images")
    assert _refusal(aai, L.aai_image_upload(C.byref(a), C.byref(narrow), 0, None)) == incompatible
    assert _refusal(aai, L.aai_image_download(C.byref(a), C.byref(wide_u8), 0, None)) == incompatible
    # the band (device image of an upload, source of a download) must lie inside the other image's rows
    dev = _img(aai, (10, 16))
    dev.height = 20
    host = _img(aai, (18, 16))
    host.y0, host.height = 2, 20
    assert _refusal(aai, L.aai_image_upload(C.byref(dev), C.byref(host), 0, None)) == (
        aai.ERR_ARGUMENT, "aai_image copy: band rows [0,10) not inside [2,20)")
    assert _refusal(aai, L.aai_image_download(C.byref(host), C.byref(dev), 0, None)) == (
        aai.ERR_ARGUMENT, "aai_image copy: band rows [0,10) not inside [2,20)")


def test_host_entry_points_image_checks(aai, plan):
    L = aai.lib()
    si, di = _img(aai, (48, 64)), _img(aai, (plan.dst_h, plan.dst_w))
    small = _img(aai, (5, 5))
    assert _refusal(aai, L.aai_run_host_band(C.byref(plan), 1, aai.ARITH_F32, C.byref(si), C.byref(small), 0, 1, 0,
                                             None, 1)) == (aai.ERR_ARGUMENT,
                                                           "aai_run_host_band: host images do not match the plan")
    assert _refusal(aai, L.aai_run_host(C.byref(plan), 1, aai.ARITH_F32, C.byref(small), C.byref(di), None, 0)) == (
        aai.ERR_ARGUMENT, "aai_run_host: host images do not match the plan")
    part = aai.Image(si.data, si.pitch_bytes, si.width, si.height, 0, 47, si.dtype, si.channels)
    arr_s, arr_d = (aai.Image * 2)(si, part), (aai.Image * 2)(di, di)
    assert _refusal(aai, L.aai_run_host_batch(C.byref(plan), 1, aai.ARITH_F32, arr_s, arr_d, 2, 0, None, 1)) == (
        aai.ERR_ARGUMENT, "aai_run_host_batch: whole host images expected")
    assert _refusal(aai, L.aai_run_host_batch(C.byref(plan), 1, aai.ARITH_F32, arr_s, arr_d, 0, 0, None, 1)) == (
        aai.ERR_ARGUMENT, "aai_run_host_batch: bad argument")
    assert _refusal(aai, L.aai_run_host_band(C.byref(plan), 1, aai.ARITH_F32, C.byref(si), C.byref(di), 3, 2, 0,
                                             None, 1)) == (aai.ERR_ARGUMENT, "aai_run_host_band: bad rows [3,2)")
