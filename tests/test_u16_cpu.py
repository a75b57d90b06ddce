"""16-bit unsigned images (AAI_U16) without a GPU: the Python mirror of the header enum, the image views of uint16
arrays, the host-side refusal of the unsupported (source, canvas) element-type pairs, and the uint16 synthetic images."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# the four (source, canvas) pairs the library is not compiled for (include/aai.h)
REFUSED = [(np.float64, np.uint16), (np.float32, np.uint16), (np.uint8, np.uint16), (np.uint16, np.uint8)]


@pytest.fixture(scope="module")
def aai(built):
    import area_average_interpolation_b200 as m

    m.lib()
    return m


def test_u16_enum_equals_the_header(aai, tmp_path):
    src = tmp_path / "u16.c"
    src.write_text('#include <stdio.h>\n#include "aai.h"\nint main(void) { printf("%d\\n", (int)AAI_U16); return 0; }\n')
    exe = str(tmp_path / "u16")
    subprocess.run(["gcc", "-std=c99", "-I" + os.path.join(ROOT, "include"), str(src), "-o", exe], check=True)
    out = subprocess.run([exe], capture_output=True, text=True, check=True).stdout
    assert int(out) == aai.U16 == 3


def test_uint16_image_views(aai):
    import torch

    a = np.zeros((7, 11), dtype=np.uint16)
    im = aai._host_image(a)
    assert (im.dtype, im.channels, im.width, im.height, im.pitch_bytes) == (aai.U16, 1, 11, 7, 22)
    rgb = np.zeros((5, 9, 3), dtype=np.uint16)
    im = aai._host_image(rgb)
    assert (im.dtype, im.channels, im.width, im.height, im.pitch_bytes) == (aai.U16, 3, 9, 5, 54)
    padded = np.zeros((6, 16), dtype=np.uint16)[:, :13]   # a column view: only the row pitch is padded
    im = aai._host_image(padded)
    assert (im.width, im.pitch_bytes) == (13, 32)
    t = torch.zeros((4, 10, 3), dtype=torch.uint16)
    ti = aai.tensor_image(t[1:], y0=1, height=4)
    assert (ti.dtype, ti.channels, ti.width, ti.height, ti.y0, ti.rows, ti.pitch_bytes) == (aai.U16, 3, 10, 4, 1, 3, 60)
    assert ti.data == t[1:].data_ptr()
    with pytest.raises(TypeError, match="uint16"):
        aai._host_image(np.zeros((3, 3), dtype=np.int16))


def test_refused_pairs_fail_on_the_host_before_cuda(aai):
    """Every run entry point refuses the four unsupported pairs with AAI_ERR_ARGUMENT and a message naming the pair,
    before any CUDA call -- so the same on a box without a GPU."""
    plan = aai.make_plan(64, 48, 1.0, 0.5, (32, 24), 10.0)
    L = aai.lib()

    def status_of(fn, *a, **k):
        with pytest.raises(aai.AaiError) as ei:
            fn(*a, **k)
        return ei.value.status

    for s_dt, d_dt in REFUSED:
        src = np.zeros((48, 64), dtype=s_dt)
        dst = np.zeros((plan.dst_h, plan.dst_w), dtype=d_dt)
        si, di = aai._host_image(src), aai._host_image(dst)
        pair = f"a {np.dtype(s_dt).name} source cannot write a {np.dtype(d_dt).name} canvas"
        calls = [
            ("aai_run_device", lambda: aai.run_device(plan, si, di)),
            ("aai_run_device_batch", lambda: aai.run_device_batch(plan, [si, si], [di, di])),
            ("aai_run_host", lambda: aai.run_host(plan, src, dst)),
            ("aai_run_host_band", lambda: aai.run_host_band(plan, si, di, 0, plan.dst_h)),
            ("aai_run_host_batch", lambda: aai.run_host_batch(plan, [si, si], [di, di])),
        ]
        for who, call in calls:
            assert status_of(call) == aai.ERR_ARGUMENT, (who, s_dt, d_dt)
            assert aai.last_error().startswith(who) and pair in aai.last_error(), aai.last_error()
        # the peer group checks the pair before it looks at its group
        assert L.aai_peer_run(None, aai.MODE_AREA_AVERAGE, aai.ARITH_F32, C.byref(si), C.byref(di), None, 1) == \
            aai.ERR_ARGUMENT
        assert aai.last_error().startswith("aai_peer_run") and pair in aai.last_error()


def test_supported_uint16_pairs_pass_the_pair_check(aai):
    """u16 -> f64 / f32 / u16 get past the pair check: the next argument error (an unknown mode) is what is reported."""
    plan = aai.make_plan(64, 48, 1.0, 0.5, (32, 24), 10.0)
    si = aai._host_image(np.zeros((48, 64), dtype=np.uint16))
    for d_dt in (np.float64, np.float32, np.uint16):
        di = aai._host_image(np.zeros((plan.dst_h, plan.dst_w), dtype=d_dt))
        with pytest.raises(aai.AaiError) as ei:
            aai.run_device(plan, si, di, mode=4)
        assert ei.value.status == aai.ERR_ARGUMENT and "interpolation mode" in aai.last_error(), aai.last_error()


def test_uint16_synthetic_image(aai):
    """Deterministic, seekable by row, the full range 0..65535 (the top 16 bits of the hash: the top byte is the 8-bit
    image), and the torch generator is bit-identical on the CPU."""
    from area_average_interpolation_b200.synthetic import synthetic_image, synthetic_image_torch

    a = synthetic_image(1024, 1024, np.uint16, 31)
    assert a.dtype == np.uint16
    assert np.array_equal(a, synthetic_image(1024, 1024, np.uint16, 31))
    assert not np.array_equal(a, synthetic_image(1024, 1024, np.uint16, 32))
    assert np.array_equal(a[500:537], synthetic_image(1024, 1024, np.uint16, 31, y0=500, rows=37))
    assert a.min() == 0 and a.max() == 65535
    assert abs(float(a.mean()) - 32767.5) < 100.0
    assert np.array_equal(a >> 8, synthetic_image(1024, 1024, np.uint8, 31))
    rgb = synthetic_image(301, 70, np.uint16, 5, channels=3)
    t = synthetic_image_torch(301, 70, np.uint16, 5, channels=3)
    assert str(t.dtype) == "torch.uint16" and np.array_equal(t.numpy(), rgb)
    band = synthetic_image_torch(301, 70, np.uint16, 5, channels=3, y0=13, rows=20)
    assert np.array_equal(band.numpy(), rgb[13:33])
