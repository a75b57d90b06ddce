"""GPU (-m gpu): 16-bit unsigned sources (AAI_U16) through every kernel family, with float32 / float64 / uint16 canvases,
against the CPU oracle on the float64 view of the same full-range data; the store rule of 16-bit canvases; batched, host,
multi-device and peer-group paths bitwise against the device path."""
import os
import re
import sys

import numpy as np
import pytest

from common import TOL_F32_REL, TOL_F64_REL, f32_err, rel_err

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U16_MAX = 65535.0


@pytest.fixture(scope="module")
def aai(built):
    import area_average_interpolation_b200 as m

    assert m.device_count() >= 1, "no CUDA device: the product has no CPU fallback"
    return m


@pytest.fixture(scope="module")
def oracle(built):
    from oracle import port

    return port


def _source(w, h, seed, ch=1):
    from area_average_interpolation_b200.synthetic import synthetic_image

    return synthetic_image(w, h, np.uint16, seed, channels=ch)


# torch's CUDA kernels for uint16 are few: device copies go through the int16 view of the same bits
def _cuda(a):
    import torch

    if a.dtype == np.uint16:
        return torch.from_numpy(np.ascontiguousarray(a).view(np.int16)).cuda().view(torch.uint16)
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _host(t):
    import torch

    if t.dtype == torch.uint16:
        return t.view(torch.int16).cpu().numpy().view(np.uint16)
    return t.cpu().numpy()


def _empty(shape, np_dtype, device="cuda", pin=False):
    import torch

    t_dt = {np.dtype(np.uint16): torch.int16, np.dtype(np.float32): torch.float32, np.dtype(np.float64): torch.float64}
    t = torch.zeros(shape, dtype=t_dt[np.dtype(np_dtype)], device=device)
    if pin:
        t = t.pin_memory()
    return t.view(torch.uint16) if np.dtype(np_dtype) == np.uint16 else t


def _oracle(oracle, src, sres, dres, iso, angle, mode=1, rows=None):
    """The oracle on the float64 view of the data, all channels ([h, w] or [h, w, c])."""
    src = np.asarray(src, dtype=np.float64) if src.dtype == np.uint16 else src
    ch = src.shape[2] if src.ndim == 3 else 1
    outs = []
    for c in range(ch):
        st, want, _ = oracle.run(src, sres, dres, iso, angle, mode=mode, rows=rows, channel=c)
        assert st == 0
        outs.append(want)
    return outs[0] if ch == 1 else np.stack(outs, axis=-1)


def _tie_mask(oracle, src, sres, dres, iso, angle, mode, want, delta=1e-11):
    """Pixels whose reference value changes when the isocentre moves by 1e-11 (fast mode: a source-pixel centre exactly
    on a footprint edge is a tie the reference resolves by rounding noise, see test_gpu_parity)."""
    mask = np.zeros(want.shape, dtype=bool)
    for dx, dy in [(1, 1), (-1, -1), (1, 0), (0, 1), (-1, 0), (0, -1), (1, -1), (-1, 1)]:
        moved = _oracle(oracle, src, sres, dres, (iso[0] + dx * delta, iso[1] + dy * delta), angle, mode)
        mask |= rel_err(moved, want) > TOL_F64_REL
    return mask


def _bad(got, want, arith, canvas):
    """Pixels outside the tolerance of (arithmetic, canvas)."""
    got = np.asarray(got, dtype=np.float64)
    if canvas == np.uint16:  # round half up of the real value: 0.5 + the bound of the arithmetic
        bound = 1e-9 * np.abs(want) if arith == 0 else TOL_F32_REL * np.maximum(np.abs(want), U16_MAX / 256.0)
        return np.abs(got - want) > 0.5 + bound
    if arith == 0:
        return rel_err(got, want) > (TOL_F64_REL if canvas == np.float64 else 1e-7)
    return f32_err(got, want, U16_MAX) > TOL_F32_REL


def _check(oracle, got, want, arith, canvas, src, sres, dres, iso, angle, mode):
    bad = _bad(got, want, arith, canvas)
    if mode == 2 and bad.any():
        mask = _tie_mask(oracle, src, sres, dres, iso, angle, mode, want)
        assert bad.mean() < 0.02, float(bad.mean())
        bad &= ~mask
    assert not bad.any(), (int(bad.sum()), float(np.abs(np.asarray(got, np.float64) - want)[bad].max()))


# ---- every kernel family with a 16-bit source -------------------------------------------------------------------------

# name: (w, h, ratio, angle, iso, channels, mode, arith, kernel that serves the uint16 canvas)
FAMILIES = {
    "f32_ident": (300, 260, 0.37, 17.3, (150.0, 130.0), 1, 1, 1, "overlap_kernel_f32"),
    "f32_general": (300, 260, 0.37, 117.3, (150.0, 130.0), 1, 1, 1, "overlap_kernel_f32"),
    "f32_grouped_rgb": (200, 150, 1.7, 45.0, (99.5, 74.5), 3, 1, 1, "overlap_kernel_f32"),
    "near_axis_f64": (300, 260, 0.37, 1.5, (150.0, 130.0), 1, 1, 1, "overlap_kernel_f64u"),
    "ratio_0p1_rolled": (300, 260, 0.1, 17.3, (150.0, 130.0), 1, 1, 1, "overlap_kernel_f64"),
    "two_channels_rolled": (300, 260, 0.37, 17.3, (150.0, 130.0), 2, 1, 1, "overlap_kernel_f64"),
    "f64_unrolled": (300, 260, 0.37, 17.3, (150.0, 130.0), 1, 1, 0, "overlap_kernel_f64u"),
    "fast_f32": (300, 260, 0.37, 17.3, (150.0, 130.0), 1, 2, 1, "fast_kernel_f32u"),
    "fast_f32_rgb": (300, 260, 0.37, 17.3, (150.0, 130.0), 3, 2, 1, "fast_kernel_f32u"),
    "fast_f64": (300, 260, 0.37, 17.3, (150.0, 130.0), 1, 2, 0, "fast_kernel"),
    "exact_f64": (300, 260, 0.37, 17.3, (150.0, 130.0), 1, 3, 0, "overlap_kernel_f64u"),
    "exact_f32": (300, 260, 0.37, 17.3, (150.0, 130.0), 1, 3, 1, "overlap_kernel_f32"),
    "sep_tma": (320, 256, 0.5, 0.0, (160.0, 128.0), 1, 1, 1, "separable_tma_kernel"),
    "sep_tma_f64": (320, 256, 0.5, 0.0, (160.0, 128.0), 1, 1, 0, "separable_tma_kernel"),
    "sep_direct_90": (300, 260, 0.5, 90.0, (150.0, 130.0), 1, 1, 1, "separable_direct_f32"),
    "sep_direct_scale2_rgb": (120, 90, 2.0, 0.0, (60.0, 45.0), 3, 1, 1, "separable_direct_f32"),
}
CANVASES = [np.float32, np.float64, np.uint16]


def _device_run(aai, plan, src_t, canvas, mode, arith, batch_shape=()):
    import torch

    dst = _empty(batch_shape + (plan.dst_h, plan.dst_w) + tuple(src_t.shape[2 + len(batch_shape):]), canvas)
    aai.run_device(plan, aai.tensor_image(src_t), aai.tensor_image(dst), mode=mode, arith=arith,
                   stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return dst


_WANT = {}


def _family_want(oracle, name):
    if name not in _WANT:
        w, h, ratio, angle, iso, ch, mode, arith, _ = FAMILIES[name]
        src = _source(w, h, 1600 + w + ch, ch)
        _WANT[name] = (src, _oracle(oracle, src, 1.0, ratio, iso, angle, mode))
    return _WANT[name]


@pytest.mark.parametrize("canvas", CANVASES, ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize("name", list(FAMILIES))
def test_every_kernel_family_with_a_16bit_source(aai, oracle, name, canvas):
    w, h, ratio, angle, iso, ch, mode, arith, _ = FAMILIES[name]
    src, want = _family_want(oracle, name)
    plan = aai.make_plan(w, h, 1.0, ratio, iso, angle)
    before = aai.launch_count()
    got = _host(_device_run(aai, plan, _cuda(src), canvas, mode, arith))
    assert aai.launch_count() > before, "no CUDA kernel was launched"
    assert got.dtype == canvas and got.shape == want.shape
    _check(oracle, got, want, arith, canvas, src, 1.0, ratio, iso, angle, mode)
    # the operator passes the uint16 array through natively and gives the same result as the device call
    r = aai.AreaAverageInterpolation(arith=arith, out_dtype=canvas)._run(mode, src, 1.0, ratio, iso, angle, (0.0, 0.0))
    assert r.ok and r.dst.dtype == canvas
    if not (name.startswith("sep_tma") or name == "sep_direct_scale2_rgb"):  # (see test_host_paths_are_bitwise_...)
        assert np.array_equal(r.dst, got)
    else:
        _check(oracle, r.dst, want, arith, canvas, src, 1.0, ratio, iso, angle, mode)


def _kernel_names(run):
    """Names of the CUDA kernels `run` launches (torch.profiler, CUDA activities)."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}


def _has_u16_kernel(names, family):
    # demangled "family<unsigned short, ..." or, if the profiler reports mangled names, "<len>familyIt..."
    pat = re.compile(r"(?<![A-Za-z_])" + family + r"(<unsigned short|It)")
    return any(pat.search(n) for n in names)


def test_each_family_runs_its_uint16_instantiation(aai):
    """The families above (and the STAGED / RING variants) really run kernels instantiated for a uint16 source --
    nothing widens the data on the way."""
    cases = [(n,) + FAMILIES[n][:8] + (FAMILIES[n][8],) for n in FAMILIES]
    # (the staged variants need 16-byte aligned source rows)
    cases += [("staged_overlap", 320, 256, 0.37, 17.3, (160.0, 128.0), 1, 1, 2, "overlap_kernel_f32_tma"),
              ("staged_fast", 320, 256, 0.37, 17.3, (160.0, 128.0), 1, 2, 2, "fast_kernel_f32u_tma"),
              ("ring_fast", 320, 256, 0.37, 17.3, (160.0, 128.0), 1, 2, 4, "fast_kernel_f32u_ring"),
              ("staged_overlap_rgb", 320, 256, 0.37, 17.3, (160.0, 128.0), 3, 1, 2, "overlap_kernel_f32_tma")]
    missing = []
    for name, w, h, ratio, angle, iso, ch, mode, arith, family in cases:
        plan = aai.make_plan(w, h, 1.0, ratio, iso, angle)
        src_t = _cuda(_source(w, h, 7, ch))
        _device_run(aai, plan, src_t, np.uint16, mode, arith)  # warm-up outside the profiled window
        names = _kernel_names(lambda: _device_run(aai, plan, src_t, np.uint16, mode, arith))
        if not _has_u16_kernel(names, family):
            missing.append((name, family, sorted(n[:120] for n in names)))
    assert not missing, missing


# ---- default callers: uint16 through the operator is what float64 was -------------------------------------------------

@pytest.mark.parametrize("mode", [1, 2, 3])
@pytest.mark.parametrize("ratio,angle,iso", [(0.37, 17.3, (150.0, 130.0)), (0.5, 0.0, (160.0, 128.0)),
                                             (0.6, 117.0, (150.0, 130.0))])
def test_default_operator_on_uint16_equals_the_float64_widening(aai, ratio, angle, iso, mode):
    """With ARITH_F64 the native uint16 call is bitwise the call on astype(float64) (what the operator did with uint16
    arrays before it passed them through), and the result type is float64 as before."""
    src = _source(320, 260, 99, 1)
    op = aai.AreaAverageInterpolation()
    a = op._run(mode, src, 1.0, ratio, iso, angle, (0.0, 0.0))
    b = op._run(mode, src.astype(np.float64), 1.0, ratio, iso, angle, (0.0, 0.0))
    assert a.dst.dtype == np.float64 and np.array_equal(a.dst, b.dst)


# ---- store rule of 16-bit canvases ------------------------------------------------------------------------------------

@pytest.mark.parametrize("arith", [0, 1])
def test_u16_canvas_saturates_a_constant_full_scale_image(aai, arith):
    import torch

    w, h = 400, 300
    plan = aai.make_plan(w, h, 1.0, 0.37, (200.0, 150.0), 17.3)
    full = _cuda(np.full((h, w), 65535, dtype=np.uint16))
    got = _host(_device_run(aai, plan, full, np.uint16, 1, arith))
    cover = _host(_device_run(aai, plan, torch.ones((h, w), dtype=torch.float64, device="cuda"), np.float64, 1, 0)) != 0
    assert 0.4 < cover.mean() < 0.9
    assert (got[cover] == 65535).all() and (got[~cover] == 0).all()


def test_u16_canvas_rounds_half_up(aai):
    """0/1 checkerboard at 0 deg, 0.5x: every interior footprint mean is exactly 0.5 (FP64), stored as 1."""
    w, h = 256, 200
    src = ((np.arange(h)[:, None] + np.arange(w)[None, :]) & 1).astype(np.uint16)
    plan = aai.make_plan(w, h, 1.0, 0.5, (128.0, 100.0), 0.0)
    f64 = _host(_device_run(aai, plan, _cuda(src), np.float64, 1, 0))
    assert (f64[1:-1, 1:-1] == 0.5).all()
    got = _host(_device_run(aai, plan, _cuda(src), np.uint16, 1, 0))
    assert (got[1:-1, 1:-1] == 1).all()


# ---- A/B variants ---------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("canvas", [np.float32, np.uint16], ids=lambda d: np.dtype(d).name)
def test_staged_ring_binned_equal_the_default_fp32_kernels(aai, canvas):
    for ch in (1, 3):
        src_t = _cuda(_source(320, 256, 21, ch))  # 16-byte rows: the staged variants apply
        plan = aai.make_plan(320, 256, 1.0, 0.37, (160.0, 128.0), 17.3)
        for mode, variants in ((1, (aai.ARITH_F32_STAGED,)),
                               (2, (aai.ARITH_F32_STAGED, aai.ARITH_F32_RING, aai.ARITH_F32_BINNED))):
            ref = _host(_device_run(aai, plan, src_t, canvas, mode, aai.ARITH_F32))
            for arith in variants:
                assert np.array_equal(_host(_device_run(aai, plan, src_t, canvas, mode, arith)), ref), (ch, mode, arith)


# ---- batches, host paths, several devices, peer group -------------------------------------------------------------------

@pytest.mark.parametrize("canvas", [np.float32, np.uint16], ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize("w,h,ratio,angle,iso", [(300, 260, 0.37, 17.3, (150.0, 130.0)), (640, 512, 0.5, 0.0, (320.0, 256.0))])
def test_u16_stack_is_one_launch_and_equals_per_slice_runs(aai, w, h, ratio, angle, iso, canvas):
    import torch

    n = 5
    src = np.stack([_source(w, h, 300 + k) for k in range(n)])
    src_t = _cuda(src)
    plan = aai.make_plan(w, h, 1.0, ratio, iso, angle)
    dst = _empty((n, plan.dst_h, plan.dst_w), canvas)
    stream = torch.cuda.current_stream().cuda_stream
    before = aai.launch_count()
    aai.run_device_batch(plan, [aai.tensor_image(src_t[k]) for k in range(n)], [aai.tensor_image(dst[k]) for k in range(n)],
                         arith=aai.ARITH_F32, stream=stream)
    torch.cuda.synchronize()
    assert aai.launch_count() == before + 1
    got = _host(dst)
    for k in range(n):
        one = _host(_device_run(aai, plan, src_t[k], canvas, 1, aai.ARITH_F32))
        assert np.array_equal(got[k], one), k


# widths with 16-byte rows: the device path takes the kernels the host path's pitched buffers take
HOST_CASES = [(320, 256, 0.37, 17.3, (160.0, 128.0), 1), (320, 256, 0.5, 0.0, (160.0, 128.0), 1),
              (200, 152, 1.7, 45.0, (99.5, 75.5), 3)]


@pytest.mark.parametrize("canvas", [np.float32, np.uint16], ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize("w,h,ratio,angle,iso,ch", HOST_CASES)
def test_host_paths_are_bitwise_the_device_path(aai, w, h, ratio, angle, iso, ch, canvas):
    import torch

    src = _source(w, h, 77, ch)
    plan = aai.make_plan(w, h, 1.0, ratio, iso, angle)
    want = _host(_device_run(aai, plan, _cuda(src), canvas, 1, aai.ARITH_F32))
    tail = (ch,) if ch > 1 else ()
    # run_host
    dst = np.zeros((plan.dst_h, plan.dst_w) + tail, dtype=canvas)
    aai.run_host(plan, src, dst, arith=aai.ARITH_F32)
    assert np.array_equal(dst, want)
    # run_host_band: pinned buffers, two bands enqueued asynchronously on the caller's stream
    src_p = torch.from_numpy(src.view(np.int16)).pin_memory().view(torch.uint16)
    dst_p = _empty((plan.dst_h, plan.dst_w) + tail, canvas, device="cpu", pin=True)
    stream = torch.cuda.current_stream().cuda_stream
    mid = plan.dst_h // 2
    for r0, r1 in ((0, mid), (mid, plan.dst_h)):
        aai.run_host_band(plan, aai.tensor_image(src_p), aai.tensor_image(dst_p[r0:r1], y0=r0, height=plan.dst_h), r0, r1,
                          arith=aai.ARITH_F32, stream=stream, synchronize=False)
    torch.cuda.synchronize()
    assert np.array_equal(_host(dst_p), want)
    # run_host_batch
    n = 3
    srcs = [_source(w, h, 77 + k, ch) for k in range(n)]
    s_p = [torch.from_numpy(s.view(np.int16)).pin_memory().view(torch.uint16) for s in srcs]
    d_p = [_empty((plan.dst_h, plan.dst_w) + tail, canvas, device="cpu", pin=True) for _ in range(n)]
    aai.run_host_batch(plan, [aai.tensor_image(s) for s in s_p], [aai.tensor_image(d) for d in d_p], arith=aai.ARITH_F32)
    for k in range(n):
        one = _host(_device_run(aai, plan, _cuda(srcs[k]), canvas, 1, aai.ARITH_F32))
        assert np.array_equal(_host(d_p[k]), one), k


def test_two_devices_reproduce_one_device_bitwise(aai):
    if aai.device_count() < 2:
        pytest.skip("needs two devices")
    w, h = 1200, 1000
    src = _source(w, h, 5, 1)
    plan = aai.make_plan(w, h, 1.0, 0.37, (600.0, 500.0), 17.3)
    for canvas in (np.float32, np.uint16):
        one = np.zeros((plan.dst_h, plan.dst_w), dtype=canvas)
        two = np.ones((plan.dst_h, plan.dst_w), dtype=canvas)
        aai.run_host(plan, src, one, arith=aai.ARITH_F32)
        aai.run_host(plan, src, two, arith=aai.ARITH_F32, devices=[0, 1])
        assert np.array_equal(one, two)


PEER = dict(w=400, h=300, ratio=1.7, angle=45.0, iso=(199.5, 149.5), ch=3)
PEER_STEPS = 2


def _peer_rank_main(rank, world, tmpdir):
    sys.path.insert(0, ROOT)
    import torch

    import area_average_interpolation_b200 as aai
    from test_peer_group_gpu import _file_gather

    c = PEER
    device = rank % max(1, torch.cuda.device_count())
    torch.cuda.set_device(device)
    stream = torch.cuda.current_stream().cuda_stream
    plan = aai.make_plan(c["w"], c["h"], 1.0, c["ratio"], c["iso"], c["angle"])
    group = aai.PeerGroup(plan, aai.U16, c["ch"], rank, world, device, _file_gather(tmpdir, "u16", rank, world))
    o0, o1 = group.owned_rows()
    r0, r1 = group.band()
    srcs, dsts = [], []
    for t in range(PEER_STEPS):
        s = _source(c["w"], c["h"], 900 + t, c["ch"])[o0:o1]
        srcs.append(torch.from_numpy(np.ascontiguousarray(s).view(np.int16)).pin_memory().view(torch.uint16))
        dsts.append(_empty((max(r1 - r0, 1), plan.dst_w, c["ch"]), np.uint16, device="cpu", pin=True))
    for t in range(PEER_STEPS):
        group.run(aai.tensor_image(srcs[t], y0=o0, height=c["h"]), aai.tensor_image(dsts[t][:r1 - r0], y0=r0, height=plan.dst_h),
                  arith=aai.ARITH_F32, stream=stream, synchronize=False)
    torch.cuda.synchronize()
    for t in range(PEER_STEPS):
        np.save(os.path.join(tmpdir, f"u16.band{rank}.step{t}.npy"), _host(dsts[t][:r1 - r0]))
    open(os.path.join(tmpdir, f"u16.{rank}.done"), "w").close()
    import time

    t0 = time.time()
    while not all(os.path.exists(os.path.join(tmpdir, f"u16.{p}.done")) for p in range(world)):
        assert time.time() - t0 < 60
        time.sleep(0.005)
    group.close()


def test_peer_group_on_a_u16_rgb_image_equals_one_gpu(aai, tmp_path):
    """Two processes (two devices, or sharing cuda:0): the stitched bands of a uint16 RGB image and a uint16 canvas
    equal the single-process result bit for bit."""
    import torch.multiprocessing as mp

    world = 2
    mp.spawn(_peer_rank_main, args=(world, str(tmp_path)), nprocs=world, join=True)
    c = PEER
    plan = aai.make_plan(c["w"], c["h"], 1.0, c["ratio"], c["iso"], c["angle"])
    bounds = aai.partition_rows(plan, world)
    for t in range(PEER_STEPS):
        want = np.zeros((plan.dst_h, plan.dst_w, c["ch"]), dtype=np.uint16)
        aai.run_host(plan, _source(c["w"], c["h"], 900 + t, c["ch"]), want, arith=aai.ARITH_F32)
        parts = [np.load(tmp_path / f"u16.band{r}.step{t}.npy") for r in range(world)]
        got = np.concatenate([parts[r][:bounds[r + 1] - bounds[r]] for r in range(world)], axis=0)
        assert np.array_equal(got, want), t


# ---- expansion ------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("ratio,angle", [(0.37, 17.3), (1.7, 117.0), (2.3, 305.5), (0.5, 0.0)])
def test_expand_device_on_u16(aai, ratio, angle):
    import torch

    for shape in [(37, 53), (37, 53, 3)]:
        host = _source(shape[1], shape[0], 3, shape[2] if len(shape) == 3 else 1)
        h, w = shape[:2]
        plan = aai.make_plan(w, h, 1.0, ratio, (w / 2.0, h / 2.0), angle)
        mod = _empty((plan.mod_h, plan.mod_w) + shape[2:], np.uint16)
        before = aai.launch_count()
        aai.expand_device(plan, aai.tensor_image(_cuda(host)), aai.tensor_image(mod),
                          stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert aai.launch_count() == before + 1
        want = np.repeat(np.repeat(host, plan.scale, axis=0), plan.scale, axis=1)
        want = np.rot90(want, k=-plan.quadrant, axes=(0, 1))
        assert np.array_equal(_host(mod), want)


# ---- sizes a user runs ------------------------------------------------------------------------------------------------

def test_full_size_16384_u16_to_u16_canvas_sample_rows(aai, oracle):
    """BASELINE config 4's geometry (16384^2, 0.37x, 17.3 deg) on a full-range 16-bit image, FP32 arithmetic, 16-bit
    canvas: three sampled rows against the oracle."""
    import torch

    from area_average_interpolation_b200.synthetic import synthetic_image_torch

    W = 16384
    plan = aai.make_plan(W, W, 1.0, 0.37, (8192.0, 8192.0), 17.3)
    src_t = synthetic_image_torch(W, W, np.uint16, 20201 + 16, device="cuda")
    got = _host(_device_run(aai, plan, src_t, np.uint16, 1, aai.ARITH_F32))
    src32 = _host(src_t).astype(np.float32)  # exact: 16-bit values
    del src_t
    torch.cuda.empty_cache()
    for row in (1, 3795, 7589):
        want = _oracle(oracle, src32, 1.0, 0.37, (8192.0, 8192.0), 17.3, rows=(row, row + 1))
        assert not _bad(got[row:row + 1], want, 1, np.uint16).any(), row
    assert (got[3795] != 0).mean() > 0.5  # the middle row is mostly covered


@pytest.mark.parametrize("mode", [1, 2])
def test_film_scan_with_the_reference_settings(aai, oracle, mode):
    """A 1500 x 1800 RGB 16-bit "film scan" through the reference's shipped settings (150 -> 25.4 dpi, isocentre
    (455, 455), 1.5 deg), whole canvas: FP64 into float64, FP32 into float32 and uint16."""
    src = _source(1500, 1800, 2024, 3)
    args = (150.0, 25.4, (455.0, 455.0), 1.5)
    want = _oracle(oracle, src, *args, mode=mode)
    for arith, canvas in ((0, np.float64), (1, np.float32), (1, np.uint16)):
        op = aai.AreaAverageInterpolation(arith=arith, out_dtype=canvas)
        r = op._run(mode, src, *args, (0.0, 0.0))
        assert r.ok and r.dst.dtype == canvas and r.dst.shape == want.shape
        _check(oracle, r.dst, want, arith, canvas, src, *args, mode)
