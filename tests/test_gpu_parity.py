"""GPU (-m gpu): the CUDA path, called through the C ABI (libaai_b200.so), against the golden vectors of the
compiled reference, against the CPU oracle on seeded inputs, and -- at BASELINE.json's full sizes -- through
size-independent properties plus oracle-checked sample rows."""
import numpy as np
import pytest

from common import TOL_F64_REL, TOL_F32_REL, TOL_U8_ABS, f32_err, golden_source, load_golden, rel_err

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def aai(built):
    import area_average_interpolation_b200 as m

    assert m.device_count() >= 1, "no CUDA device: the product has no CPU fallback"
    return m


@pytest.fixture(scope="module")
def oracle(built):
    from oracle import port

    return port


def _run(aai, src, sres, dres, iso, angle, mode=1, arith=0, out_dtype=np.float64, devices=None):
    op = aai.AreaAverageInterpolation(arith=arith, out_dtype=out_dtype, devices=devices)
    f = op.areaAverageInterpolation if mode == 1 else op.fastAreaAverageInterpolation
    before = aai.launch_count()
    r = f(src, sres, dres, iso, angle)
    assert r.ok, r.message
    assert aai.launch_count() > before, "no CUDA kernel was launched"
    return r


# ---- golden vectors of the compiled reference ----------------------------------------------------------------

def test_golden_vectors_f64(aai):
    z, meta = load_golden()
    for case in meta["cases"]:
        src = golden_source(case)
        r = _run(aai, src, case["src_res"], case["dst_res"], case["iso"], case["angle"], mode=case["mode"])
        want = z[case["name"]]
        assert list(r.dst.shape) == case["dst_shape"], case["name"]
        assert list(r.dst_isocenter) == case["dst_iso"], case["name"]
        if case.get("degenerate"):
            continue  # compared under the conditioning mask below
        err = rel_err(r.dst, want)
        assert err.max() <= TOL_F64_REL, (case["name"], float(err.max()), int((err > TOL_F64_REL).sum()))


def _conditioning_mask(oracle, src, case, want, delta=1e-11):
    """T5: pixels on which the reference's own answer changes when the isocentre moves by 1e-11 (8 directions)."""
    mask = np.zeros(want.shape, dtype=bool)
    for dx, dy in [(1, 1), (-1, -1), (1, 0), (0, 1), (-1, 0), (0, -1), (1, -1), (-1, 1)]:
        iso = (case["iso"][0] + dx * delta, case["iso"][1] + dy * delta)
        st, moved, _ = oracle.run(src, case["src_res"], case["dst_res"], iso, case["angle"], mode=case["mode"])
        mask |= rel_err(moved, want) > TOL_F64_REL
    return mask


def test_degenerate_inputs_match_outside_the_reference_conditioning_mask(aai, oracle):
    """T4: vertices/edges exactly on grid lines.  Every pixel on which the reference is well conditioned must match;
    the ill-conditioned ones (reference flips under a 1e-11 isocentre shift) are counted, not gated."""
    z, meta = load_golden()
    cases = [c for c in meta["cases"] if c.get("degenerate")]
    assert len(cases) >= 7
    for case in cases:
        src = golden_source(case)
        want = z[case["name"]]
        r = _run(aai, src, case["src_res"], case["dst_res"], case["iso"], case["angle"], mode=case["mode"])
        mask = _conditioning_mask(oracle, src, case, want)
        err = rel_err(r.dst, want)
        assert mask.mean() < 0.1, case["name"]
        assert (err[~mask] <= TOL_F64_REL).all(), (case["name"], int(((err > TOL_F64_REL) & ~mask).sum()))
        print(f"{case['name']}: {int(mask.sum())} ill-conditioned reference pixels of {mask.size} masked; "
              f"{int((err[mask] > TOL_F64_REL).sum())} of them differ")


def test_golden_vectors_axis_aligned_are_exact_on_u8(aai):
    # 0.5x / 0 deg on 8-bit data: weights 1/2, 1, 1/2 (or the aligned 2x2 box) -> every operation is exact
    z, meta = load_golden()
    for name in ("cfg1_u8_half_0deg", "cfg1_u8_half_0deg_halfiso"):
        case = next(c for c in meta["cases"] if c["name"] == name)
        r = _run(aai, golden_source(case), case["src_res"], case["dst_res"], case["iso"], case["angle"])
        assert np.array_equal(r.dst, z[name]), name


def test_validation_failures_do_not_touch_the_gpu(aai):
    _, meta = load_golden()
    op = aai.AreaAverageInterpolation()
    for e in meta["errors"]:
        src = np.ones((e["h"], e["w"])) if e["h"] and e["w"] else np.zeros((e["h"], e["w"]))
        before = aai.launch_count()
        r = op.areaAverageInterpolation(src, e["src_res"], e["dst_res"], (1.0, 1.0), 10.0, dstIsocenter=(-7.0, -9.0))
        assert (r.ok, r.message, list(r.dst_isocenter)) == (False, e["message"], e["dst_iso"]), e["name"]
        assert aai.launch_count() == before


# ---- oracle on seeded inputs ------------------------------------------------------------------------------------

SWEEP = [
    # w, h, ratio, angle, iso
    (512, 512, 0.37, 17.3, (256.0, 256.0)),   # cfg4 replica
    (512, 512, 0.37, 30.0, (256.0, 256.0)),   # cfg2 replica (integer isocentre: well conditioned)
    (192, 192, 1.7, 45.0, (95.5, 95.5)),      # cfg3 replica (scale 3, half-integer isocentre)
    (512, 512, 0.5, 0.0, (256.0, 256.0)),     # cfg1 / cfg5 replica
    (300, 200, 0.11, 73.0, (150.0, 100.0)),   # strong downscale: L = 9.09, theta >= 45 branch
    (257, 129, 0.37, 117.3, (100.0, 64.0)),   # quadrant 1, non-square
    (129, 257, 0.45, 200.0, (64.0, 128.0)),   # quadrant 2
    (150, 150, 0.9, 305.5, (0.0, 0.0)),       # quadrant 3, scale 2, isocentre at the corner
    (64, 64, 2.3, 61.0, (32.0, 32.0)),        # scale 4
    (200, 120, 0.2, -12.0, (400.0, -50.0)),   # isocentre far outside the image
    (128, 128, 0.6, 89.0, (64.0, 64.0)),      # nearly 90 degrees
    (128, 128, 0.6, 1.0, (64.0, 64.0)),       # nearly 0 degrees
    (100, 100, 1.0, 180.0, (50.0, 50.0)),     # scale 2, axis aligned
    (100, 80, 0.5, 270.0, (49.5, 40.5)),      # axis aligned, quadrant 3, half-integer isocentre
    (90, 90, 0.70710678, 33.0, (45.0, 45.0)), # ratio*sqrt(2) just below 1
    (31, 17, 0.3, 45.0, (15.2, 8.1)),         # canvas smaller than one tile
]


@pytest.mark.parametrize("w,h,ratio,angle,iso", SWEEP)
def test_f64_kernel_matches_oracle(aai, oracle, w, h, ratio, angle, iso):
    rng = np.random.default_rng(w * 7919 + h)
    src = rng.uniform(0.0, 4096.0, size=(h, w))
    r = _run(aai, src, 1.0, ratio, iso, angle)
    st, want, wiso = oracle.run(src, 1.0, ratio, iso, angle)
    assert st == 0 and want.shape == r.dst.shape and wiso == r.dst_isocenter
    err = rel_err(r.dst, want)
    assert err.max() <= TOL_F64_REL, (float(err.max()), int((err > TOL_F64_REL).sum()))


@pytest.mark.parametrize("w,h,ratio,angle,iso", SWEEP[:8])
def test_fast_mode_matches_oracle(aai, oracle, w, h, ratio, angle, iso):
    """Row f1 (fastAreaAverageInterpolation): a source pixel counts iff its CENTRE is in the footprint, so a centre
    that lies exactly on a footprint edge is a tie the reference itself resolves by rounding noise (its 4-ray test has
    a ~2e-14 px tolerance, below the 1e-13 rounding of its own vertices).  Pixels whose reference value changes under a
    1e-11 isocentre shift are masked (T5); all others must match."""
    rng = np.random.default_rng(w * 31 + h)
    src = rng.uniform(0.0, 4096.0, size=(h, w))
    r = _run(aai, src, 1.0, ratio, iso, angle, mode=2)
    st, want, _ = oracle.run(src, 1.0, ratio, iso, angle, mode=2)
    assert st == 0 and want.shape == r.dst.shape
    bad = rel_err(r.dst, want) > TOL_F64_REL
    if bad.any():
        case = dict(src_res=1.0, dst_res=ratio, iso=iso, angle=angle, mode=2)
        mask = _conditioning_mask(oracle, src, case, want)
        assert not (bad & ~mask).any(), int((bad & ~mask).sum())
        assert bad.mean() < 0.02, float(bad.mean())


@pytest.mark.parametrize("w,h,ratio,angle,iso", SWEEP)
def test_fast_mode_fp32_kernel_matches_oracle(aai, oracle, w, h, ratio, angle, iso):
    """Row f1 in FP32 arithmetic (float / 8-bit images): the inside test is decided in FP32 with a guard band and
    redone in FP64 inside it, so every pixel on which the reference is well conditioned must match to 1e-5."""
    rng = np.random.default_rng(w * 77 + h)
    src = rng.uniform(0.0, 4096.0, size=(h, w)).astype(np.float32)
    r = _run(aai, src, 1.0, ratio, iso, angle, mode=2, arith=aai.ARITH_F32, out_dtype=np.float32)
    st, want, wiso = oracle.run(src, 1.0, ratio, iso, angle, mode=2)
    assert st == 0 and want.shape == r.dst.shape and wiso == r.dst_isocenter
    err = f32_err(r.dst, want, 4096.0)
    bad = err > TOL_F32_REL
    if bad.any():
        case = dict(src_res=1.0, dst_res=ratio, iso=iso, angle=angle, mode=2)
        mask = _conditioning_mask(oracle, src, case, want)
        assert not (bad & ~mask).any(), (int((bad & ~mask).sum()), float(err[~mask].max()))
        assert bad.mean() < 0.02, float(bad.mean())
    # and it agrees with the FP64 fast kernel wherever that one agrees with the oracle
    r64 = _run(aai, src, 1.0, ratio, iso, angle, mode=2, out_dtype=np.float64)
    same = rel_err(r64.dst, want) <= TOL_F64_REL
    assert np.abs(r.dst.astype(np.float64) - r64.dst)[same].max() <= 1e-5 * 4096.0


# ---- FP32 kernel (north star: <= 1e-5 relative on float data, <= 0.5/255 absolute on 8-bit data) ----------------

@pytest.mark.parametrize("w,h,ratio,angle,iso", SWEEP)
def test_f32_kernel_matches_oracle_on_float_data(aai, oracle, w, h, ratio, angle, iso):
    rng = np.random.default_rng(w * 104729 + h)
    src = rng.uniform(0.0, 4096.0, size=(h, w)).astype(np.float32)
    r = _run(aai, src, 1.0, ratio, iso, angle, arith=aai.ARITH_F32, out_dtype=np.float32)
    st, want, wiso = oracle.run(src, 1.0, ratio, iso, angle)
    assert st == 0 and want.shape == r.dst.shape and wiso == r.dst_isocenter
    err = f32_err(r.dst, want, 4096.0)
    assert err.max() <= TOL_F32_REL, (float(err.max()), int((err > TOL_F32_REL).sum()))


def test_f32_kernel_on_8bit_data_and_golden_vectors(aai, oracle):
    z, meta = load_golden()
    for case in meta["cases"]:
        if case.get("degenerate") or case["mode"] != 1:
            continue
        src = golden_source(case)
        if src.dtype == np.float64:
            src = src.astype(np.float32)
        r = _run(aai, src, case["src_res"], case["dst_res"], case["iso"], case["angle"], arith=aai.ARITH_F32,
                 out_dtype=np.float32)
        st, want, _ = oracle.run(src, case["src_res"], case["dst_res"], case["iso"], case["angle"])
        tol = TOL_U8_ABS if src.dtype == np.uint8 else TOL_F32_REL * np.maximum(np.abs(want), float(src.max()) / 256.0)
        assert (np.abs(r.dst - want) <= tol).all(), case["name"]
    rng = np.random.default_rng(12)
    rgb = rng.integers(0, 256, size=(300, 260, 3), dtype=np.uint8)
    for (ratio, angle, iso) in [(0.37, 30.0, (130.0, 150.0)), (1.7, 45.0, (129.5, 149.5)), (0.9, 200.0, (10.0, 10.0))]:
        r = _run(aai, rgb, 1.0, ratio, iso, angle, arith=aai.ARITH_F32, out_dtype=np.float32)
        for c in range(3):
            st, want, _ = oracle.run(rgb, 1.0, ratio, iso, angle, channel=c)
            assert np.abs(r.dst[..., c] - want).max() <= TOL_U8_ABS, (ratio, angle, c)
        r8 = _run(aai, rgb, 1.0, ratio, iso, angle, arith=aai.ARITH_F32, out_dtype=np.uint8)
        assert np.abs(r8.dst.astype(np.float64) - r.dst).max() <= 0.5 + 1e-3  # round half up of the real value


def test_f32_kernel_symmetric_ties_and_near_axis_angles(aai, oracle):
    """Exactly symmetric geometry (cell centres on the footprint's centre lines: sign ties) and angles where the
    FP32 kernel must hand over to FP64 (1/sin or 1/cos > 20)."""
    rng = np.random.default_rng(77)
    src = rng.uniform(0.0, 255.0, size=(256, 256)).astype(np.float32)
    for (ratio, angle, iso) in [(1.7, 45.0, (127.5, 127.5)), (0.5, 45.0, (127.5, 127.5)), (0.6, 1.0, (128.0, 128.0)),
                                (0.6, 88.5, (128.0, 128.0)), (0.6, 5.0, (128.0, 128.0))]:
        r = _run(aai, src, 1.0, ratio, iso, angle, arith=aai.ARITH_F32, out_dtype=np.float32)
        st, want, _ = oracle.run(src, 1.0, ratio, iso, angle)
        err = f32_err(r.dst, want, 255.0)
        assert err.max() <= TOL_F32_REL, (ratio, angle, float(err.max()))


def test_u8_rgb_and_f32_sources(aai, oracle):
    rng = np.random.default_rng(5)
    rgb = rng.integers(0, 256, size=(120, 160, 3), dtype=np.uint8)
    r = _run(aai, rgb, 1.0, 1.7, (79.5, 59.5), 45.0)
    assert r.dst.shape[2] == 3
    for c in range(3):
        st, want, _ = oracle.run(rgb, 1.0, 1.7, (79.5, 59.5), 45.0, channel=c)
        assert np.abs(r.dst[..., c] - want).max() <= TOL_U8_ABS
        assert rel_err(r.dst[..., c], want).max() <= TOL_F64_REL
    f32 = rng.uniform(0, 4096, size=(200, 150)).astype(np.float32)
    r = _run(aai, f32, 1.0, 0.37, (75.0, 100.0), 17.3)
    st, want, _ = oracle.run(f32, 1.0, 0.37, (75.0, 100.0), 17.3)
    assert rel_err(r.dst, want).max() <= TOL_F64_REL
    # float32 / uint8 destinations: the stored value is the rounded real-valued result
    r32 = _run(aai, f32, 1.0, 0.37, (75.0, 100.0), 17.3, out_dtype=np.float32)
    assert np.array_equal(r32.dst, want.astype(np.float32)) or rel_err(r32.dst, want).max() <= 1e-6
    g8 = rng.integers(0, 256, size=(90, 90), dtype=np.uint8)
    r8 = _run(aai, g8, 1.0, 0.37, (45.0, 45.0), 30.0, out_dtype=np.uint8)
    st, want8, _ = oracle.run(g8, 1.0, 0.37, (45.0, 45.0), 30.0)
    # documented store rule: round half up, saturate; ties are measure-zero on this input
    assert np.abs(r8.dst.astype(np.float64) - np.floor(want8 + 0.5)).max() <= 1.0
    assert (r8.dst.astype(np.float64) != np.floor(want8 + 0.5)).mean() < 1e-3


def test_row_bands_are_bitwise_identical_to_one_launch(aai):
    """T6: any band split (the multi-GPU partition) reproduces the single-launch result bit for bit."""
    import torch

    from area_average_interpolation_b200.sharding import all_bands

    w, h, ratio, angle, iso = 700, 500, 0.37, 17.3, (350.0, 250.0)
    plan = aai.make_plan(w, h, 1.0, ratio, iso, angle)
    src = torch.rand(h, w, dtype=torch.float64, device="cuda") * 4096
    whole = torch.empty(plan.dst_h, plan.dst_w, dtype=torch.float64, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    aai.run_device(plan, aai.tensor_image(src), aai.tensor_image(whole), stream=stream)
    for n in (2, 3, 8):
        parts = []
        for band in all_bands(plan, n):
            # the rank holds only its halo rows of the source and only its band of the canvas
            halo = src[band.src_y0:band.src_y1].contiguous()
            out = torch.full((band.rows, plan.dst_w), -1.0, dtype=torch.float64, device="cuda")
            aai.run_device(plan, aai.tensor_image(halo, y0=band.src_y0, height=h),
                           aai.tensor_image(out, y0=band.row0, height=plan.dst_h), band.row0, band.row1,
                           stream=stream)
            parts.append(out)
        torch.cuda.synchronize()
        assert torch.equal(torch.cat(parts, 0), whole), n


@pytest.mark.parametrize("ratio,angle,iso", [(0.9, 305.5, (10.0, 20.0)), (0.37, 117.3, (90.0, 60.0)), (1.7, 200.0, (64.5, 50.5))])
def test_row_bands_with_rotated_quadrants_and_scaled_sources(aai, oracle, ratio, angle, iso):
    """Bands whose source halo is a column range (quadrants 1/3) or a mirrored row range (quadrant 2), scale > 1,
    both kernels: each band equals the single-launch result bit for bit, and the FP64 one matches the oracle."""
    import torch

    from area_average_interpolation_b200.sharding import all_bands

    w, h = 180, 130
    plan = aai.make_plan(w, h, 1.0, ratio, iso, angle)
    rng = np.random.default_rng(9)
    src_np = rng.uniform(0, 4096, size=(h, w)).astype(np.float32)
    src = torch.from_numpy(src_np).cuda()
    stream = torch.cuda.current_stream().cuda_stream
    for arith, dt in ((aai.ARITH_F64, torch.float64), (aai.ARITH_F32, torch.float32)):
        whole = torch.empty(plan.dst_h, plan.dst_w, dtype=dt, device="cuda")
        aai.run_device(plan, aai.tensor_image(src), aai.tensor_image(whole), arith=arith, stream=stream)
        parts = []
        for band in all_bands(plan, 3):
            halo = src[band.src_y0:band.src_y1].contiguous()
            out = torch.full((band.rows, plan.dst_w), -1.0, dtype=dt, device="cuda")
            aai.run_device(plan, aai.tensor_image(halo, y0=band.src_y0, height=h),
                           aai.tensor_image(out, y0=band.row0, height=plan.dst_h), band.row0, band.row1, arith=arith,
                           stream=stream)
            parts.append(out)
        torch.cuda.synchronize()
        assert torch.equal(torch.cat(parts, 0), whole), (arith, angle)
        if arith == aai.ARITH_F64:
            st, want, _ = oracle.run(src_np, 1.0, ratio, iso, angle)
            assert rel_err(whole.cpu().numpy(), want).max() <= TOL_F64_REL


def test_multi_device_host_path_if_available(aai, oracle):
    n = aai.device_count()
    rng = np.random.default_rng(8)
    src = rng.uniform(0, 4096, size=(300, 400))
    one = _run(aai, src, 1.0, 0.37, (200.0, 150.0), 17.3, devices=[0])
    many = _run(aai, src, 1.0, 0.37, (200.0, 150.0), 17.3, devices=list(range(n)) if n > 1 else [0, 0][:1])
    assert np.array_equal(one.dst, many.dst)


def test_batch_of_slices_is_one_launch_and_matches_per_image_runs(aai, oracle):
    """BASELINE config 5 in small: a stack of equally strided slices, 0.5x axis-aligned -> one kernel launch."""
    import torch

    n, w, h = 5, 200, 168
    plan = aai.make_plan(w, h, 1.0, 0.5, (100.0, 84.0), 0.0)
    src = torch.rand(n, h, w, dtype=torch.float32, device="cuda") * 4096
    dst = torch.empty(n, plan.dst_h, plan.dst_w, dtype=torch.float32, device="cuda")
    ref = torch.empty_like(dst)
    stream = torch.cuda.current_stream().cuda_stream
    before = aai.launch_count()
    aai.run_device_batch(plan, [aai.tensor_image(src[k]) for k in range(n)], [aai.tensor_image(dst[k]) for k in range(n)],
                         arith=aai.ARITH_F32, stream=stream)
    assert aai.launch_count() == before + 1
    for k in range(n):
        aai.run_device(plan, aai.tensor_image(src[k]), aai.tensor_image(ref[k]), arith=aai.ARITH_F32, stream=stream)
    torch.cuda.synchronize()
    assert torch.equal(dst, ref)
    st, want, _ = oracle.run(src[3].cpu().numpy(), 1.0, 0.5, (100.0, 84.0), 0.0)
    assert f32_err(dst[3].cpu().numpy(), want, 4096.0).max() <= TOL_F32_REL
    # not equally strided (reversed order): falls back to one launch per image, same results
    order = [4, 2, 0]
    out2 = torch.empty(3, plan.dst_h, plan.dst_w, dtype=torch.float32, device="cuda")
    aai.run_device_batch(plan, [aai.tensor_image(src[k]) for k in order], [aai.tensor_image(out2[i]) for i in range(3)],
                         arith=aai.ARITH_F32, stream=stream)
    torch.cuda.synchronize()
    assert torch.equal(out2, ref[order])


@pytest.mark.parametrize("ratio,angle,iso,dtype,ch,mode,arith", [
    (0.37, 17.3, (60.0, 50.0), "float32", 1, 1, 1),   # FP32 overlap kernel, identity addressing
    (0.37, 117.3, (60.0, 50.0), "float32", 1, 1, 1),  # rotated quadrant: general addressing
    (1.7, 40.0, (59.5, 50.5), "uint8", 3, 1, 1),      # upscaling, RGB: grouped path
    (0.6, 30.0, (60.0, 50.0), "float64", 1, 1, 0),    # unrolled FP64 kernel
    (0.9, 61.0, (10.0, 20.0), "float32", 2, 1, 0),    # two channels: rolled FP64 kernel
    (0.37, 30.0, (60.0, 50.0), "float32", 1, 2, 1),   # fast mode, FP32
    (0.37, 30.0, (60.0, 50.0), "float64", 1, 2, 0),   # fast mode, FP64
    (0.37, 17.3, (60.0, 50.0), "float32", 1, 3, 1),   # exact mode
    (2.0, 90.0, (60.0, 50.0), "float32", 1, 1, 1),    # axis-aligned outside the TMA kernel's preconditions: direct taps
])
def test_batch_of_rotated_slices_is_one_launch(aai, oracle, ratio, angle, iso, dtype, ch, mode, arith):
    """A stack of equally strided slices sharing a ROTATED plan (a CT volume) is one launch with grid.z = slice for
    every kernel of the path, bitwise identical to per-slice launches and within tolerance of the oracle."""
    import torch

    n, w, h = 4, 120, 100
    tdt = {"float32": torch.float32, "float64": torch.float64, "uint8": torch.uint8}[dtype]
    plan = aai.make_plan(w, h, 1.0, ratio, iso, angle)
    tail = (ch,) if ch > 1 else ()
    g = torch.Generator(device="cuda").manual_seed(7)
    if dtype == "uint8":
        src = torch.randint(0, 256, (n, h, w) + tail, dtype=tdt, device="cuda", generator=g)
    else:
        src = (torch.rand((n, h, w) + tail, dtype=torch.float32, device="cuda", generator=g) * 4096).to(tdt)
    odt = torch.float64 if arith == 0 else torch.float32  # (a float32 store would round the FP64 result)
    dst = torch.full((n, plan.dst_h, plan.dst_w) + tail, -1.0, dtype=odt, device="cuda")
    ref = torch.full_like(dst, -2.0)
    stream = torch.cuda.current_stream().cuda_stream
    before = aai.launch_count()
    aai.run_device_batch(plan, [aai.tensor_image(src[k]) for k in range(n)], [aai.tensor_image(dst[k]) for k in range(n)],
                         mode=mode, arith=arith, stream=stream)
    assert aai.launch_count() == before + 1
    for k in range(n):
        aai.run_device(plan, aai.tensor_image(src[k]), aai.tensor_image(ref[k]), mode=mode, arith=arith, stream=stream)
    torch.cuda.synchronize()
    assert torch.equal(dst, ref)
    if mode != 3:  # (exact mode has its own checker, test_exact_mode_matches_its_clipping_checker)
        k = n - 1
        plane = src[k].cpu().numpy().astype(np.float64)
        got = dst[k].cpu().numpy().astype(np.float64)
        for c in range(ch):
            st, want, _ = oracle.run(plane[..., c] if ch > 1 else plane, 1.0, ratio, iso, angle, mode=mode)
            assert st == 0
            gc = got[..., c] if ch > 1 else got
            if dtype == "uint8" and arith == 1:  # north star: 0.5/255 absolute on 8-bit data for the FP32 kernel
                assert np.abs(gc - want).max() <= TOL_U8_ABS
            else:
                err = f32_err(gc, want, 4096.0) if arith == 1 else rel_err(gc, want)
                assert err.max() <= (TOL_F32_REL if arith == 1 else TOL_F64_REL)


def test_device_image_helpers_roundtrip(aai):
    """aai_image_alloc / upload / copy_rows / download: pitched device images and row-range copies."""
    rng = np.random.default_rng(4)
    host = rng.uniform(0, 1, size=(37, 53)).astype(np.float32)
    himg = aai._host_image(host)
    a = aai.image_alloc(0, 53, 37, aai.F32)
    b = aai.image_alloc(0, 53, 37, aai.F32)
    assert a.pitch_bytes % 512 == 0
    aai.image_upload(a, himg)
    aai.image_copy_rows(b, a, 5, 30)
    back = np.zeros_like(host)
    aai.image_download(aai._host_image(back), b)
    import torch

    torch.cuda.synchronize()
    assert np.array_equal(back[5:30], host[5:30])
    with pytest.raises(aai.AaiError):
        aai.image_copy_rows(b, a, 30, 40)
    aai.image_free(a, 0)
    aai.image_free(b, 0)


def test_argument_errors_are_reported_not_crashed(aai):
    import torch

    plan = aai.make_plan(64, 64, 1.0, 0.5, (32, 32), 10.0)
    src = torch.zeros(64, 64, dtype=torch.float32, device="cuda")
    bad = torch.zeros(5, 5, dtype=torch.float32, device="cuda")
    with pytest.raises(aai.AaiError) as ei:
        aai.run_device(plan, aai.tensor_image(src), aai.tensor_image(bad))
    assert ei.value.status == aai.ERR_ARGUMENT
    dst = torch.zeros(plan.dst_h, plan.dst_w, dtype=torch.float32, device="cuda")
    with pytest.raises(aai.AaiError):
        aai.run_device(plan, aai.tensor_image(src), aai.tensor_image(dst), mode=4)
    # a source band that misses rows the canvas band needs is refused
    with pytest.raises(aai.AaiError):
        aai.run_device(plan, aai.tensor_image(src[:8].contiguous(), y0=0, height=64), aai.tensor_image(dst))


# ---- randomised configurations ----------------------------------------------------------------------------------------

def _random_cases(n, seed):
    rng = np.random.default_rng(seed)
    cases = []
    for _ in range(n):
        w, h = int(rng.integers(24, 220)), int(rng.integers(24, 220))
        ratio = float(rng.choice([rng.uniform(0.15, 0.7), rng.uniform(0.7, 1.5), rng.uniform(1.5, 2.8)]))
        # angles away from the axes by at least 0.05 degrees (closer ones are the separable path's business) and away
        # from exact symmetric configurations (conditioning, SURVEY T5)
        angle = float(rng.uniform(-360.0, 720.0))
        if abs((angle % 90.0 + 45.0) % 90.0 - 45.0) < 0.05:
            angle += 1.234
        iso = (float(rng.uniform(-0.2 * w, 1.2 * w)), float(rng.uniform(-0.2 * h, 1.2 * h)))
        cases.append((w, h, round(ratio, 4), round(angle, 3), (round(iso[0], 3), round(iso[1], 3))))
    return cases


@pytest.mark.parametrize("w,h,ratio,angle,iso", _random_cases(36, 20201))
def test_random_configurations_both_kernels(aai, oracle, w, h, ratio, angle, iso):
    """Random sizes, ratios (scale 1..4), angles in all quadrants and isocentres (also outside the image): FP64 kernel
    <= 1e-9 and FP32 kernel <= 1e-5 against the oracle; pixels on which the reference itself is ill-conditioned (its value
    changes under a 1e-11 isocentre shift) are masked, they must stay rare."""
    rng = np.random.default_rng(w * 1009 + h)
    src = rng.uniform(0.0, 4096.0, size=(h, w)).astype(np.float32)
    st, want, wiso = oracle.run(src, 1.0, ratio, iso, angle)
    assert st == 0
    r64 = _run(aai, src, 1.0, ratio, iso, angle, out_dtype=np.float64)
    r32 = _run(aai, src, 1.0, ratio, iso, angle, arith=aai.ARITH_F32, out_dtype=np.float32)
    assert r64.dst.shape == want.shape and r64.dst_isocenter == wiso and r32.dst.shape == want.shape
    bad64 = rel_err(r64.dst, want) > TOL_F64_REL
    e32 = f32_err(r32.dst, want, 4096.0)
    bad32 = e32 > TOL_F32_REL
    if bad64.any() or bad32.any():
        case = dict(src_res=1.0, dst_res=ratio, iso=iso, angle=angle, mode=1)
        mask = _conditioning_mask(oracle, src, case, want)
        assert not (bad64 & ~mask).any(), (int((bad64 & ~mask).sum()), float(rel_err(r64.dst, want)[~mask].max()))
        assert not (bad32 & ~mask).any(), (int((bad32 & ~mask).sum()), float(e32[~mask].max()))
        assert mask.mean() < 0.01


# ---- separable (axis-aligned) path: persistent TMA kernel -----------------------------------------------------------

@pytest.mark.parametrize("w,h,ratio,iso", [
    (1000, 777, 0.37, (500.0, 388.0)),    # L = 2.70: 4 taps, canvas not a multiple of the tile
    (640, 1500, 0.5, (320.5, 750.25)),    # L = 2: 3 taps, tall image: several tiles per strip, fractional isocentre
    (900, 700, 0.23, (450.0, 350.0)),     # L = 4.35: 6 taps
    (1200, 800, 0.125, (600.0, 400.0)),   # L = 8: 9 taps (32-column tiles)
    (333, 4100, 0.7071, (10.0, 4000.0)),  # L = 1.414, canvas narrower than one tile, isocentre near a corner
])
def test_separable_tma_path_matches_oracle(aai, oracle, w, h, ratio, iso):
    """0 degrees, scale 1, one channel: the TMA-staged strip kernel (ring of source windows, producer warp).  FP64 and
    FP32 arithmetic, f64 / f32 / u8 sources, and a split into uneven row bands (bitwise identical to one launch)."""
    import torch

    rng = np.random.default_rng(w + h)
    src = rng.uniform(0.0, 255.0, size=(h, w))
    st, want, wiso = oracle.run(src, 1.0, ratio, iso, 0.0)
    assert st == 0
    r = _run(aai, src, 1.0, ratio, iso, 0.0)
    assert r.dst.shape == want.shape and r.dst_isocenter == wiso
    assert rel_err(r.dst, want).max() <= TOL_F64_REL
    src32 = src.astype(np.float32)
    st, want32, _ = oracle.run(src32, 1.0, ratio, iso, 0.0)
    r32 = _run(aai, src32, 1.0, ratio, iso, 0.0, arith=aai.ARITH_F32, out_dtype=np.float32)
    err = f32_err(r32.dst, want32, 255.0)
    assert err.max() <= TOL_F32_REL, float(err.max())
    src8 = src.astype(np.uint8)
    st, want8, _ = oracle.run(src8, 1.0, ratio, iso, 0.0)
    r8 = _run(aai, src8, 1.0, ratio, iso, 0.0, arith=aai.ARITH_F32, out_dtype=np.float32)
    assert np.abs(r8.dst.astype(np.float64) - want8).max() <= TOL_U8_ABS
    # row bands on the device path
    plan = aai.make_plan(w, h, 1.0, ratio, iso, 0.0)
    s_t = torch.from_numpy(src32).cuda()
    whole = torch.empty((plan.dst_h, plan.dst_w), dtype=torch.float32, device="cuda")
    parts = torch.full_like(whole, -1.0)
    stream = torch.cuda.current_stream().cuda_stream
    aai.run_device(plan, aai.tensor_image(s_t), aai.tensor_image(whole), arith=aai.ARITH_F32, stream=stream)
    cuts = [0, min(7, plan.dst_h), min(7 + 49, plan.dst_h), plan.dst_h]
    for a, b in zip(cuts[:-1], cuts[1:]):
        aai.run_device(plan, aai.tensor_image(s_t), aai.tensor_image(parts), a, b, arith=aai.ARITH_F32, stream=stream)
    torch.cuda.synchronize()
    assert torch.equal(whole, parts)
    # (the host path uses its own pitched buffers, so it may take the other axis-aligned kernel: rounding only)
    assert np.allclose(whole.cpu().numpy(), r32.dst, rtol=2e-6, atol=1e-5)


# ---- rows f3 / f4 of SURVEY 8f ---------------------------------------------------------------------------------------

@pytest.mark.parametrize("ratio,angle", [(0.37, 17.3), (1.7, 117.0), (0.9, 200.0), (2.3, 305.5), (0.5, 0.0)])
def test_expand_device_equals_replicate_and_rot90(aai, ratio, angle):
    """Row f3: modSrc (Source.cpp:157-172) = the source replicated `scale` times, rotated quadrant*90 deg clockwise."""
    import torch

    rng = np.random.default_rng(9)
    for dtype, shape in [(np.float32, (37, 53)), (np.uint8, (37, 53, 3)), (np.float64, (20, 31))]:
        host = (rng.uniform(0, 255, size=shape)).astype(dtype)
        h, w = shape[:2]
        plan = aai.make_plan(w, h, 1.0, ratio, (w / 2.0, h / 2.0), angle)
        src = torch.from_numpy(host).cuda()
        mod = torch.zeros((plan.mod_h, plan.mod_w) + shape[2:], dtype=src.dtype, device="cuda")
        before = aai.launch_count()
        aai.expand_device(plan, aai.tensor_image(src), aai.tensor_image(mod),
                          stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert aai.launch_count() == before + 1
        want = np.repeat(np.repeat(host, plan.scale, axis=0), plan.scale, axis=1)
        want = np.rot90(want, k=-plan.quadrant, axes=(0, 1))  # k*90 degrees clockwise
        assert want.shape == tuple(mod.shape)
        assert np.array_equal(mod.cpu().numpy(), want)


@pytest.mark.parametrize("w,h,ratio,angle,iso", SWEEP[:10])
def test_exact_mode_matches_its_clipping_checker(aai, oracle, w, h, ratio, angle, iso):
    """Row f4 (opt-in, not the reference's arithmetic): areas without the shape-2/4 quirk, against Sutherland-Hodgman
    clipping + shoelace (oracle mode 3), FP64 and FP32 kernels."""
    rng = np.random.default_rng(w * 17 + h)
    src = rng.uniform(0.0, 4096.0, size=(h, w))
    st, want, wiso = oracle.run(src, 1.0, ratio, iso, angle, mode=3)
    assert st == 0
    op = aai.AreaAverageInterpolation()
    r = op.exactAreaAverageInterpolation(src, 1.0, ratio, iso, angle)
    assert r.ok and r.dst.shape == want.shape and r.dst_isocenter == wiso
    err = rel_err(r.dst, want)
    assert err.max() <= TOL_F64_REL, (float(err.max()), int((err > TOL_F64_REL).sum()))
    op32 = aai.AreaAverageInterpolation(arith=aai.ARITH_F32, out_dtype=np.float32)
    r32 = op32.exactAreaAverageInterpolation(src.astype(np.float32), 1.0, ratio, iso, angle)
    st, want32, _ = oracle.run(src.astype(np.float32), 1.0, ratio, iso, angle, mode=3)
    err = f32_err(r32.dst, want32, 4096.0)
    assert err.max() <= TOL_F32_REL, (float(err.max()), int((err > TOL_F32_REL).sum()))


# ---- properties (size independent) + full-size configurations -------------------------------------------------------

def _device_run(aai, plan, src_t, out_dtype, arith=0, mode=1):
    import torch

    dst = torch.empty((plan.dst_h, plan.dst_w) + tuple(src_t.shape[2:]), dtype=out_dtype, device="cuda")
    aai.run_device(plan, aai.tensor_image(src_t), aai.tensor_image(dst), mode=mode, arith=arith,
                   stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return dst


def test_constant_image_and_linearity(aai):
    import torch

    w, h, ratio, angle, iso = 1024, 768, 0.37, 17.3, (512.0, 384.0)
    plan = aai.make_plan(w, h, 1.0, ratio, iso, angle)
    const = torch.full((h, w), 1234.5, dtype=torch.float64, device="cuda")
    out = _device_run(aai, plan, const, torch.float64)
    covered = out != 0
    assert 0.5 < covered.double().mean().item() < 0.75
    assert (out[covered] - 1234.5).abs().max().item() <= 1e-9 * 1234.5  # weights normalise to 1
    a = torch.rand(h, w, dtype=torch.float64, device="cuda")
    b = torch.rand(h, w, dtype=torch.float64, device="cuda")
    fa, fb = _device_run(aai, plan, a, torch.float64), _device_run(aai, plan, b, torch.float64)
    fab = _device_run(aai, plan, 2.0 * a - 3.0 * b, torch.float64)
    assert (fab - (2.0 * fa - 3.0 * fb)).abs().max().item() <= 1e-12


def test_full_size_cfg4_sample_rows_and_properties(aai, oracle):
    """BASELINE config 4: 16384^2 float32, 0.37x, 17.3 deg -> 7591^2.  Whole-image oracle would take ~40 min;
    check sampled rows against the oracle plus the constant-image property on the full canvas."""
    import torch

    from area_average_interpolation_b200.synthetic import synthetic_image

    W = 16384
    plan = aai.make_plan(W, W, 1.0, 0.37, (8192.0, 8192.0), 17.3)
    assert (plan.dst_w, plan.dst_h) == (7591, 7591)
    src = synthetic_image(W, W, np.float32, 20201 + 4)
    src_t = torch.from_numpy(src).cuda()
    out = _device_run(aai, plan, src_t, torch.float64).cpu().numpy()
    out32 = _device_run(aai, plan, src_t, torch.float32, arith=aai.ARITH_F32).cpu().numpy()
    for row in (0, 1, 1700, 3795, 3796, 6000, 7589, 7590):
        st, want, _ = oracle.run(src, 1.0, 0.37, (8192.0, 8192.0), 17.3, rows=(row, row + 1))
        err = rel_err(out[row:row + 1], want)
        assert err.max() <= TOL_F64_REL, (row, float(err.max()))
        e32 = f32_err(out32[row:row + 1], want, 4096.0)
        assert e32.max() <= TOL_F32_REL, (row, float(e32.max()))
    # FP32 and FP64 kernels agree over the WHOLE canvas (the FP64 one is oracle-checked on the sample rows above)
    whole = f32_err(out32, out, 4096.0)
    assert whole.max() <= TOL_F32_REL, float(whole.max())
    frac = (out != 0).mean()
    assert 0.62 < frac < 0.65  # SURVEY §8: covered fraction 0.638
    ones = _device_run(aai, plan, torch.ones(W, W, dtype=torch.float32, device="cuda"), torch.float64)
    nz = ones != 0
    assert (ones[nz] - 1.0).abs().max().item() <= 1e-12
    assert nz.double().mean().item() == pytest.approx(frac, abs=1e-6)


def test_full_size_cfg3_rgb_upscale_sample_rows(aai, oracle):
    """BASELINE config 3 on a quarter-size source (2048^2 RGB u8, 1.7x, 45 deg, scale 3 -> 4924^2 canvas x3):
    sampled rows against the oracle; the full 8192^2 case runs in bench.py --config 3."""
    import torch

    from area_average_interpolation_b200.synthetic import synthetic_image

    W = 2048
    iso = (W / 2 - 0.5, W / 2 - 0.5)
    plan = aai.make_plan(W, W, 1.0, 1.7, iso, 45.0)
    assert plan.scale == 3
    src = synthetic_image(W, W, np.uint8, 20201 + 3, channels=3)
    out = _device_run(aai, plan, torch.from_numpy(src).cuda(), torch.float32).cpu().numpy()
    for row in (0, 2462, 4000, plan.dst_h - 1):
        for c in (0, 2):
            st, want, _ = oracle.run(src, 1.0, 1.7, iso, 45.0, rows=(row, row + 1), channel=c)
            assert np.abs(out[row:row + 1, :, c] - want).max() <= TOL_U8_ABS, (row, c)


def test_full_size_cfg5_slice_axis_aligned(aai, oracle):
    """BASELINE config 5, one 4096^2 float32 slice, 0.5x axis-aligned: 2x2-box / (1/2,1,1/2) taps."""
    import torch

    from area_average_interpolation_b200.synthetic import synthetic_image

    W = 4096
    plan = aai.make_plan(W, W, 1.0, 0.5, (2048.0, 2048.0), 0.0)
    assert plan.axis_aligned == 1 and (plan.dst_w, plan.dst_h) == (2048, 2048)
    src = synthetic_image(W, W, np.float32, 20201 + 5)
    out = _device_run(aai, plan, torch.from_numpy(src).cuda(), torch.float64).cpu().numpy()
    for row in (0, 1, 1024, 2047):
        st, want, _ = oracle.run(src, 1.0, 0.5, (2048.0, 2048.0), 0.0, rows=(row, row + 1))
        assert rel_err(out[row:row + 1], want).max() <= TOL_F64_REL, row
    # closed form for interior pixels: taps (1/2,1,1/2)^2 / 4 around source pixel (2x, 2y)
    s = src.astype(np.float64)
    y, x = 777, 1234
    k = np.array([0.5, 1.0, 0.5])
    want = (s[2 * y - 1:2 * y + 2, 2 * x - 1:2 * x + 2] * np.outer(k, k)).sum() / 4.0
    assert abs(out[y, x] - want) <= 1e-9 * abs(want)


# ---- BASELINE shapes at FULL size on the benchmarked paths (VERDICT r1 "missing" 1) ----------------------------------

def _f32_err(got, want):
    """Error of an FP32-kernel result on the 12-bit synthetic float data (tests/common.py: f32_err)."""
    return f32_err(got, want, 4096.0)


def test_full_size_cfg1_u8_whole_image(aai, oracle):
    """BASELINE config 1 at full size (512^2 8-bit, 0.5x, 0 deg, iso 256): the WHOLE canvas against the oracle --
    FP64 arithmetic bit-exact (weights 1/2, 1, 1/2 are exact), FP32 arithmetic f32 and u8 destinations (the path
    bench.py times: TMA separable kernel, u8 source)."""
    from area_average_interpolation_b200.synthetic import synthetic_image

    src = synthetic_image(512, 512, np.uint8, 20201 + 1)
    st, want, wiso = oracle.run(src, 1.0, 0.5, (256.0, 256.0), 0.0)
    assert st == 0 and want.shape == (256, 256)
    r64 = _run(aai, src, 1.0, 0.5, (256.0, 256.0), 0.0)
    assert r64.dst_isocenter == wiso and np.array_equal(r64.dst, want)
    r32 = _run(aai, src, 1.0, 0.5, (256.0, 256.0), 0.0, arith=aai.ARITH_F32, out_dtype=np.float32)
    assert np.abs(r32.dst.astype(np.float64) - want).max() <= TOL_U8_ABS
    r8 = _run(aai, src, 1.0, 0.5, (256.0, 256.0), 0.0, arith=aai.ARITH_F32, out_dtype=np.uint8)
    assert np.abs(r8.dst.astype(np.float64) - want).max() <= 0.5 + TOL_U8_ABS  # round half up of the real value


def test_full_size_cfg2_u8_whole_image(aai, oracle):
    """BASELINE config 2 at full size (2048^2 8-bit, 0.37x, 30 deg, iso 1024 -> 1035^2): the WHOLE canvas against the
    oracle, FP64 kernel <= 1e-9 relative, FP32 kernel (u8 source; f32 and u8 destinations) <= 0.5/255 absolute."""
    from area_average_interpolation_b200.synthetic import synthetic_image

    src = synthetic_image(2048, 2048, np.uint8, 20201 + 2)
    st, want, wiso = oracle.run(src, 1.0, 0.37, (1024.0, 1024.0), 30.0)
    assert st == 0 and want.shape == (1035, 1035)
    r64 = _run(aai, src, 1.0, 0.37, (1024.0, 1024.0), 30.0)
    assert r64.dst_isocenter == wiso
    e64 = rel_err(r64.dst, want)
    assert e64.max() <= TOL_F64_REL, (float(e64.max()), int((e64 > TOL_F64_REL).sum()))
    r32 = _run(aai, src, 1.0, 0.37, (1024.0, 1024.0), 30.0, arith=aai.ARITH_F32, out_dtype=np.float32)
    e = np.abs(r32.dst.astype(np.float64) - want)
    assert e.max() <= TOL_U8_ABS, (float(e.max()), int((e > TOL_U8_ABS).sum()))
    assert ((r32.dst == 0) == (want == 0)).all()  # the same canvas pixels are covered
    r8 = _run(aai, src, 1.0, 0.37, (1024.0, 1024.0), 30.0, arith=aai.ARITH_F32, out_dtype=np.uint8)
    assert np.abs(r8.dst.astype(np.float64) - want).max() <= 0.5 + TOL_U8_ABS


def test_full_size_cfg3_8192_rgb_u8_sample_rows(aai, oracle):
    """BASELINE config 3 at FULL size: 8192^2 RGB 8-bit, 1.7x, 45 deg -> scale 3, expanded frame 24576^2 (where the 32-bit
    multiply-high division and the int32 offsets live), canvas 19695^2 x 3.  First / middle / last rows, all three
    channels, against the oracle, for the f32 AND the u8 destination (the one bench.py times)."""
    import torch

    from area_average_interpolation_b200.synthetic import synthetic_image

    W = 8192
    iso = (4095.5, 4095.5)
    plan = aai.make_plan(W, W, 1.0, 1.7, iso, 45.0)
    assert plan.scale == 3 and (plan.mod_w, plan.dst_w, plan.dst_h) == (24576, 19695, 19695)
    src = synthetic_image(W, W, np.uint8, 20201 + 3, channels=3)
    src_t = torch.from_numpy(src).cuda()
    rows = (0, 1, 9847, 9848, 13001, plan.dst_h - 2, plan.dst_h - 1)
    out8 = _device_run(aai, plan, src_t, torch.uint8, arith=aai.ARITH_F32)
    got8 = {r: out8[r].cpu().numpy() for r in rows}
    covered8 = int((out8[..., 0] != 0).sum().item())
    del out8
    out32 = _device_run(aai, plan, src_t, torch.float32, arith=aai.ARITH_F32)
    got32 = {r: out32[r].cpu().numpy() for r in rows}
    del out32
    torch.cuda.empty_cache()
    assert 0.49 < covered8 / (plan.dst_w * plan.dst_h) < 0.51  # SURVEY §8: covered fraction 0.500 (u8 zeros are rare)
    for r in rows:
        for c in range(3):
            st, want, _ = oracle.run(src, 1.0, 1.7, iso, 45.0, rows=(r, r + 1), channel=c)
            assert st == 0
            e = np.abs(got32[r][None, :, c].astype(np.float64) - want)
            assert e.max() <= TOL_U8_ABS, (r, c, float(e.max()))
            e8 = np.abs(got8[r][None, :, c].astype(np.float64) - want)
            assert e8.max() <= 0.5 + TOL_U8_ABS, (r, c, float(e8.max()))


def test_full_size_cfg5_fp32_slice_and_64_slice_stack(aai, oracle):
    """BASELINE config 5 on the path bench.py times: FP32 arithmetic, TMA separable kernel.  (a) one full 4096^2 float32
    slice, WHOLE canvas against the oracle; (b) a stack of 64 equally strided slices through aai_run_device_batch (one
    launch, rank-3 tensor map): slices 0 / 31 / 63 x 4 rows against the oracle, and slice 0 bitwise equal to (a)."""
    import torch

    from area_average_interpolation_b200.synthetic import synthetic_image

    W, N = 4096, 64
    iso = (2048.0, 2048.0)
    plan = aai.make_plan(W, W, 1.0, 0.5, iso, 0.0)
    assert plan.axis_aligned == 1 and (plan.dst_w, plan.dst_h) == (2048, 2048)
    base = [synthetic_image(W, W, np.float32, 20201 + 5 + 1000 * k) for k in range(2)]

    def host_slice(k):  # slice k of the stack: a base slice rolled by 37 k rows (cheap to reproduce on the host)
        return np.roll(base[k % 2], 37 * k, axis=0)

    # (a) one slice, whole canvas
    s0 = torch.from_numpy(base[0]).cuda()
    one = _device_run(aai, plan, s0, torch.float32, arith=aai.ARITH_F32)
    st, want, _ = oracle.run(base[0], 1.0, 0.5, iso, 0.0)
    assert st == 0
    e = _f32_err(one.cpu().numpy(), want)
    assert e.max() <= TOL_F32_REL, (float(e.max()), int((e > TOL_F32_REL).sum()))
    # (b) the stack
    dev_base = [torch.from_numpy(b).cuda() for b in base]
    stack = torch.empty((N, W, W), dtype=torch.float32, device="cuda")
    for k in range(N):
        stack[k] = torch.roll(dev_base[k % 2], 37 * k, dims=0)
    dst = torch.full((N, plan.dst_h, plan.dst_w), -1.0, dtype=torch.float32, device="cuda")
    before = aai.launch_count()
    aai.run_device_batch(plan, [aai.tensor_image(stack[k]) for k in range(N)],
                         [aai.tensor_image(dst[k]) for k in range(N)], arith=aai.ARITH_F32,
                         stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert aai.launch_count() == before + 1
    assert torch.equal(dst[0], one)
    for k in (0, 31, 63):
        hs = host_slice(k)
        assert np.array_equal(stack[k, 100:102].cpu().numpy(), hs[100:102])
        got = dst[k].cpu().numpy()
        for row in (0, 777, 1024, 2047):
            st, want, _ = oracle.run(hs, 1.0, 0.5, iso, 0.0, rows=(row, row + 1))
            e = _f32_err(got[row:row + 1], want)
            assert e.max() <= TOL_F32_REL, (k, row, float(e.max()))


# ---- host-buffer copies, very tall canvases, several devices ------------------------------------------------------------

def test_download_into_a_column_view_leaves_the_rest_of_the_array_untouched(aai):
    """ADVICE r1: a host image may be a column view of a wider array; copies must not touch the bytes between rows --
    also when the view's row stride happens to equal the device pitch."""
    import torch

    w, h = 100, 40  # device pitch of 100 floats = 512 bytes = 128 floats
    big = np.full((h, 128), -7.0, dtype=np.float32)
    view = big[:, :w]
    host = np.random.default_rng(3).uniform(0, 1, size=(h, w)).astype(np.float32)
    d = aai.image_alloc(0, w, h, aai.F32)
    assert d.pitch_bytes == big.strides[0]
    aai.image_upload(d, aai._host_image(host))
    aai.image_download(aai._host_image(view), d)
    torch.cuda.synchronize()
    assert np.array_equal(view, host)
    assert (big[:, w:] == -7.0).all()
    # the same through the end-to-end host call: dst is a view into a wider array
    plan = aai.make_plan(64, 64, 1.0, 0.5, (32.0, 32.0), 20.0)
    wide = np.full((plan.dst_h, plan.dst_w + 29), -3.0, dtype=np.float64)
    src = np.random.default_rng(4).uniform(0, 100, size=(64, 64))
    aai.run_host(plan, src, wide[:, :plan.dst_w])
    assert (wide[:, plan.dst_w:] == -3.0).all() and (wide[:, :plan.dst_w] != -3.0).all()
    aai.image_free(d, 0)


def test_canvas_taller_than_the_grid_limit(aai, oracle):
    """ADVICE r1: rows sit on grid.y (<= 65535 CTAs of 8 rows); a line scan with a canvas taller than 524 280 rows is
    cut into several launches instead of failing."""
    import torch

    rng = np.random.default_rng(6)
    tall = rng.uniform(0, 4096, size=(530000, 3)).astype(np.float32)
    wide = np.ascontiguousarray(tall.T)  # a quarter turn makes its canvas as tall
    for angle, mode, arith in ((0.0, 1, aai.ARITH_F32), (0.0, 2, aai.ARITH_F32), (180.0, 1, aai.ARITH_F64),
                               (90.0, 1, aai.ARITH_F32), (90.0, 2, aai.ARITH_F64), (270.0, 1, aai.ARITH_F64),
                               (270.0, 2, aai.ARITH_F32)):
        src = wide if angle in (90.0, 270.0) else tall
        iso = (src.shape[1] / 2 - 0.5, src.shape[0] / 2)
        plan = aai.make_plan(src.shape[1], src.shape[0], 1.0, 1.0, iso, angle)
        assert plan.status == 0 and plan.dst_h > 65535 * 8
        # prefilled with NaN: a row that no slab writes fails below
        out = torch.full((plan.dst_h, plan.dst_w), float("nan"), dtype=torch.float64, device="cuda")
        before = aai.launch_count()
        aai.run_device(plan, aai.tensor_image(torch.from_numpy(src).cuda()), aai.tensor_image(out), mode=mode,
                       arith=arith, stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert aai.launch_count() >= before + 2
        assert not bool(out.isnan().any()), (angle, mode)
        for r0 in (0, 65535 * 8 - 2, plan.dst_h - 3):
            st, want, _ = oracle.run(src, 1.0, 1.0, iso, angle, mode=mode, rows=(r0, r0 + 3))
            assert st == 0
            got = out[r0:r0 + 3].cpu().numpy()
            if mode == 2:  # centre-in ties at exactly symmetric geometry are decided by rounding noise (see fast-mode tests)
                assert (rel_err(got, want) <= 1e-5).mean() > 0.6
            else:
                err = f32_err(got, want, 4096.0) if arith == aai.ARITH_F32 else rel_err(got, want)
                assert err.max() <= (TOL_F32_REL if arith == aai.ARITH_F32 else TOL_F64_REL), (angle, r0)


def test_several_devices_reproduce_one_device_bitwise(aai, oracle):
    """T6 on real hardware: aai_run_host over ALL devices of the box (one band + halo per device, one host thread each)
    is bitwise identical to device 0 alone -- FP64 and FP32 kernels, rotated and axis-aligned.  Needs >= 2 GPUs
    (`gpurun --gpus 2`); the 1-GPU box skips it (bench.py's `verified` flag covers the one-process-per-GPU path)."""
    n = aai.device_count()
    if n < 2:
        pytest.skip("needs at least two CUDA devices")
    rng = np.random.default_rng(8)
    src = rng.uniform(0, 4096, size=(1500, 2000)).astype(np.float32)
    for (ratio, angle, iso) in [(0.37, 17.3, (1000.0, 750.0)), (0.5, 0.0, (1000.0, 750.0)), (1.7, 117.0, (999.5, 749.5))]:
        for arith, od in ((aai.ARITH_F64, np.float64), (aai.ARITH_F32, np.float32)):
            one = _run(aai, src, 1.0, ratio, iso, angle, arith=arith, out_dtype=od, devices=[0])
            many = _run(aai, src, 1.0, ratio, iso, angle, arith=arith, out_dtype=od, devices=list(range(n)))
            assert np.array_equal(one.dst, many.dst), (ratio, angle, arith)
        st, want, _ = oracle.run(src, 1.0, ratio, iso, angle, rows=(700, 704))
        assert f32_err(many.dst[700:704], want, 4096.0).max() <= TOL_F32_REL


@pytest.mark.parametrize("w,h,ratio,angle,iso,dtype,ch", [
    (1500, 1100, 0.37, 17.3, (750.0, 550.0), "float32", 1),   # cfg4 shape: MAXN 5
    (900, 700, 0.37, 30.0, (450.0, 350.0), "uint8", 1),       # cfg2 shape, 8-bit
    (640, 480, 0.6, 61.0, (320.0, 240.0), "float32", 1),      # theta >= 45: MAXN 4
    (800, 600, 0.23, 40.0, (400.0, 300.0), "float32", 1),     # L = 4.35: MAXN 8, large window
    (500, 400, 0.45, 12.0, (10.0, 390.0), "uint8", 3),        # RGB 8-bit, isocentre near a corner
])
def test_tma_staged_overlap_kernel_is_bitwise_the_ldg_kernel(aai, oracle, w, h, ratio, angle, iso, dtype, ch):
    """AAI_ARITH_F32_STAGED (the north star's lay-out: CTA source window staged through shared memory by a 2-D TMA
    tensor map, cells read with LDS) runs the same arithmetic as AAI_ARITH_F32: identical bits, whole canvas, row bands
    and a stack of slices; and within tolerance of the oracle."""
    import torch

    rng = np.random.default_rng(w + h)
    tail = (ch,) if ch > 1 else ()
    host = (rng.integers(0, 256, size=(3, h, w) + tail).astype(np.uint8) if dtype == "uint8"
            else rng.uniform(0, 4096, size=(3, h, w) + tail).astype(np.float32))
    src = torch.from_numpy(host).cuda()
    plan = aai.make_plan(w, h, 1.0, ratio, iso, angle)
    stream = torch.cuda.current_stream().cuda_stream
    outs = {}
    for arith in (aai.ARITH_F32, aai.ARITH_F32_STAGED):
        dst = torch.full((3, plan.dst_h, plan.dst_w) + tail, -1.0, dtype=torch.float32, device="cuda")
        aai.run_device(plan, aai.tensor_image(src[0]), aai.tensor_image(dst[0]), arith=arith, stream=stream)
        outs[arith] = dst
    torch.cuda.synchronize()
    assert torch.equal(outs[aai.ARITH_F32][0], outs[aai.ARITH_F32_STAGED][0])
    # fast mode has the same pair of kernels
    fast = {}
    for arith in (aai.ARITH_F32, aai.ARITH_F32_STAGED):
        fast[arith] = torch.full((plan.dst_h, plan.dst_w) + tail, -1.0, dtype=torch.float32, device="cuda")
        aai.run_device(plan, aai.tensor_image(src[1]), aai.tensor_image(fast[arith]), mode=aai.MODE_FAST, arith=arith,
                       stream=stream)
    torch.cuda.synchronize()
    # (same arithmetic; the 128-bit-load kernel of float images sends a few more pixels next to the right image border
    # through the FP64 path than the staged one does, so those may differ in the last bits)
    fa, fb = fast[aai.ARITH_F32].cpu().numpy(), fast[aai.ARITH_F32_STAGED].cpu().numpy()
    assert (fa == fb).mean() > 0.995 and f32_err(fa, fb, 4096.0).max() <= TOL_F32_REL
    # the persistent, double-buffered form of the staged kernel (AAI_ARITH_F32_RING) runs the same code per tile
    ring = torch.full((plan.dst_h, plan.dst_w) + tail, -1.0, dtype=torch.float32, device="cuda")
    aai.run_device(plan, aai.tensor_image(src[1]), aai.tensor_image(ring), mode=aai.MODE_FAST, arith=aai.ARITH_F32_RING,
                   stream=stream)
    torch.cuda.synchronize()
    assert torch.equal(ring, fast[aai.ARITH_F32_STAGED])
    # row bands (each band holds only its halo rows) and a stack of slices through the staged kernel
    bands = torch.full_like(outs[aai.ARITH_F32][0], -2.0)
    from area_average_interpolation_b200.sharding import all_bands
    for band in all_bands(plan, 3):
        halo = src[0, band.src_y0:band.src_y1].contiguous()
        aai.run_device(plan, aai.tensor_image(halo, y0=band.src_y0, height=h), aai.tensor_image(bands), band.row0,
                       band.row1, arith=aai.ARITH_F32_STAGED, stream=stream)
    stack = torch.full_like(outs[aai.ARITH_F32], -3.0)
    aai.run_device_batch(plan, [aai.tensor_image(src[k]) for k in range(3)], [aai.tensor_image(stack[k]) for k in range(3)],
                         arith=aai.ARITH_F32_STAGED, stream=stream)
    torch.cuda.synchronize()
    assert torch.equal(bands, outs[aai.ARITH_F32][0])
    assert torch.equal(stack[0], outs[aai.ARITH_F32][0])
    ref2 = torch.empty_like(stack[2])
    aai.run_device(plan, aai.tensor_image(src[2]), aai.tensor_image(ref2), arith=aai.ARITH_F32, stream=stream)
    torch.cuda.synchronize()
    assert torch.equal(stack[2], ref2)
    got = outs[aai.ARITH_F32_STAGED][0].cpu().numpy().astype(np.float64)
    for c in range(ch):
        st, want, _ = oracle.run(host[0], 1.0, ratio, iso, angle, channel=c)
        g = got[..., c] if ch > 1 else got
        if dtype == "uint8":
            assert np.abs(g - want).max() <= TOL_U8_ABS
        else:
            assert f32_err(g, want, 4096.0).max() <= TOL_F32_REL


@pytest.mark.parametrize("w,h,ratio,angle,iso,dtype,ch", [
    (640, 480, 0.5, 90.0, (320.0, 240.0), "float32", 1),     # a plain quarter turn
    (640, 480, 0.5, 180.0, (320.5, 239.5), "uint8", 3),      # RGB, half turn, half-integer isocentre
    (333, 517, 0.37, 270.0, (100.0, 400.0), "uint8", 1),     # L = 2.70: 4 taps
    (300, 200, 1.0, 0.0, (150.0, 100.0), "uint8", 3),        # scale 2 (expanded frame), RGB, no rotation
    (300, 200, 2.0, 90.0, (150.0, 100.0), "float32", 1),     # scale 3 + quarter turn
    (500, 400, 0.23, 180.0, (250.0, 200.0), "float32", 3),   # L = 4.35: 6 taps, three float channels
])
def test_axis_aligned_fp32_direct_tap_kernel_matches_oracle(aai, oracle, w, h, ratio, angle, iso, dtype, ch):
    """Axis-aligned cases outside the TMA kernel's preconditions (quadrant pre-rotation Source.cpp:163-168, integer
    expansion, RGB) in FP32 arithmetic: unrolled direct-tap kernel; float and 8-bit canvases; bands bitwise."""
    import torch

    rng = np.random.default_rng(w * 3 + h)
    tail = (ch,) if ch > 1 else ()
    host = (rng.integers(0, 256, size=(h, w) + tail).astype(np.uint8) if dtype == "uint8"
            else rng.uniform(0, 4096, size=(h, w) + tail).astype(np.float32))
    plan = aai.make_plan(w, h, 1.0, ratio, iso, angle)
    assert plan.axis_aligned == 1
    src = torch.from_numpy(host).cuda()
    stream = torch.cuda.current_stream().cuda_stream
    dst = torch.full((plan.dst_h, plan.dst_w) + tail, -1.0, dtype=torch.float32, device="cuda")
    aai.run_device(plan, aai.tensor_image(src), aai.tensor_image(dst), arith=aai.ARITH_F32, stream=stream)
    parts = torch.full_like(dst, -2.0)
    cuts = [0, min(5, plan.dst_h), min(61, plan.dst_h), plan.dst_h]
    for a, b in zip(cuts[:-1], cuts[1:]):
        aai.run_device(plan, aai.tensor_image(src), aai.tensor_image(parts), a, b, arith=aai.ARITH_F32, stream=stream)
    torch.cuda.synchronize()
    assert torch.equal(dst, parts)
    got = dst.cpu().numpy().astype(np.float64)
    for c in range(ch):
        st, want, _ = oracle.run(host, 1.0, ratio, iso, angle, channel=c)
        assert st == 0
        g = got[..., c] if ch > 1 else got
        if dtype == "uint8":
            assert np.abs(g - want).max() <= TOL_U8_ABS, (c, float(np.abs(g - want).max()))
        else:
            assert f32_err(g, want, 4096.0).max() <= TOL_F32_REL, (c, float(f32_err(g, want, 4096.0).max()))
    if dtype == "uint8":
        d8 = torch.zeros((plan.dst_h, plan.dst_w) + tail, dtype=torch.uint8, device="cuda")
        aai.run_device(plan, aai.tensor_image(src), aai.tensor_image(d8), arith=aai.ARITH_F32, stream=stream)
        torch.cuda.synchronize()
        assert np.abs(d8.cpu().numpy().astype(np.float64) - got).max() <= 0.5 + 1e-3
