"""GPU (-m gpu): the adjoint of the resampling operator (aai_run_device_adjoint) and the differentiable torch entry
point (resample / resample_adjoint).

* transpose of the reference: the dense operator W is built column by column with the CPU oracle on impulse images, and
  the adjoint must equal W^T g;
* the dot-product identity <F v, g> = <v, F^T g> on BASELINE-sized images;
* stacks are one launch and bitwise equal to per-image calls and to non-strided lists; calls are deterministic;
* gradcheck / gradgradcheck of the torch entry point, bitwise agreement with the C ABI, side streams, integer sources.
"""
import numpy as np
import pytest

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


def _stream():
    import torch

    return torch.cuda.current_stream().cuda_stream


def _adjoint(aai, plan, g, mode):
    """F^T g through the C ABI: g is a CUDA tensor [N, dst_h, dst_w, C]; returns [N, src_h, src_w, C]."""
    import torch

    n, _, _, c = g.shape
    out = torch.empty((n, plan.src_h, plan.src_w, c), dtype=g.dtype, device=g.device)
    ci = [aai.tensor_image(g[k]) for k in range(n)]
    si = [aai.tensor_image(out[k]) for k in range(n)]
    aai.run_device_adjoint(plan, ci, si, mode=mode, stream=_stream())
    return out


def _forward(aai, plan, v, mode, arith=0):
    import torch

    n, _, _, c = v.shape
    out = torch.empty((n, plan.dst_h, plan.dst_w, c), dtype=torch.float64 if v.dtype == torch.float64 else torch.float32,
                      device=v.device)
    aai.run_device_batch(plan, [aai.tensor_image(v[k]) for k in range(n)],
                         [aai.tensor_image(out[k]) for k in range(n)], mode=mode, arith=arith, stream=_stream())
    return out


# ---- 1. transpose of the reference ------------------------------------------------------------------------------------

# w, h, channels, ratio, angle, iso
_ROT = [17.3, 30.0, 61.0, 107.3, 197.3, 287.3]
GEOMS = (
    [(21, 17, 1, 0.37, a, (10.0, 8.0)) for a in _ROT]
    + [(21, 17, 1, r, a, (10.0, 8.0)) for r in (1.0, 1.7, 2.3) for a in (17.3, 61.0)]
    + [(21, 17, 1, r, a, (10.0, 8.0)) for r in (0.5, 1.7) for a in (0.0, 90.0, 180.0, 270.0)]
    + [(21, 17, 1, 0.37, 17.3, (-6.0, 25.0)), (21, 17, 1, 1.7, 197.3, (30.0, -4.0)), (21, 17, 1, 0.5, 270.0, (9.5, 7.5))]
    + [(16, 12, 3, 0.37, 30.0, (8.0, 6.0)), (16, 12, 3, 1.7, 45.0, (7.5, 5.5)), (16, 12, 3, 0.5, 0.0, (8.0, 6.0))]
    + [(16, 12, 2, 0.37, 107.3, (8.0, 6.0)), (16, 12, 2, 1.7, 180.0, (7.5, 5.5))]
    + [(16, 12, 4, 1.0, 61.0, (8.3, 5.8)), (16, 12, 4, 0.5, 270.0, (8.0, 6.0))]
)
_W = {}


def _dense_operator(oracle, w, h, ratio, angle, iso, mode):
    """W[p, s]: the oracle's canvas for the impulse at source pixel s (float64, one channel)."""
    key = (w, h, ratio, angle, iso, mode)
    if key not in _W:
        cols = []
        for s in range(w * h):
            e = np.zeros((h, w))
            e.flat[s] = 1.0
            st, out, _ = oracle.run(e, 1.0, ratio, iso, angle, mode=mode)
            assert st == 0
            cols.append(out.ravel())
        _W[key] = np.stack(cols, axis=1)
    return _W[key]


@pytest.mark.parametrize("mode", [1, 2, 3])
@pytest.mark.parametrize("w,h,ch,ratio,angle,iso", GEOMS)
def test_adjoint_is_the_transpose_of_the_reference(aai, oracle, w, h, ch, ratio, angle, iso, mode):
    import torch

    plan = aai.make_plan(w, h, 1.0, ratio, iso, angle)
    assert plan.status == 0
    W = _dense_operator(oracle, w, h, ratio, angle, iso, mode)
    assert W.shape == (plan.dst_h * plan.dst_w, w * h)
    rng = np.random.default_rng(int(1000 * ratio + angle) + mode)
    g = rng.standard_normal((2, plan.dst_h, plan.dst_w, ch))
    want = np.stack([np.stack([(W.T @ g[k, ..., c].ravel()).reshape(h, w) for c in range(ch)], -1) for k in range(2)])
    scale = max(np.abs(want).max(), 1e-300)
    for dt, tol in ((torch.float64, 1e-9), (torch.float32, 1e-5)):
        gt = torch.from_numpy(g).to(dt).cuda()
        got = _adjoint(aai, plan, gt, mode)
        torch.cuda.synchronize()
        ref = want if dt == torch.float64 else np.stack(
            [np.stack([(W.T @ g[k, ..., c].astype(np.float32).astype(np.float64).ravel()).reshape(h, w)
                       for c in range(ch)], -1) for k in range(2)])
        err = np.abs(got.double().cpu().numpy() - ref).max() / scale
        assert err <= tol, (str(dt), err)


# ---- 2. dot-product identity at full size -----------------------------------------------------------------------------

FULL = {
    "cfg4_mode1": (16384, 16384, 1, 0.37, 17.3, (8192.0, 8192.0), 1),
    "cfg4_mode2": (16384, 16384, 1, 0.37, 17.3, (8192.0, 8192.0), 2),
    "cfg3_rgb_mode1": (8192, 8192, 3, 1.7, 45.0, (4095.5, 4095.5), 1),
    "cfg5_slice": (4096, 4096, 1, 0.5, 0.0, (2048.0, 2048.0), 1),
}


@pytest.mark.parametrize("name", list(FULL))
def test_dot_product_identity_at_full_size(aai, name):
    import torch

    w, h, ch, ratio, angle, iso, mode = FULL[name]
    plan = aai.make_plan(w, h, 1.0, ratio, iso, angle)
    gen = torch.Generator(device="cuda").manual_seed(7)
    v = torch.rand((1, h, w, ch), dtype=torch.float64, device="cuda", generator=gen)
    g = torch.rand((1, plan.dst_h, plan.dst_w, ch), dtype=torch.float64, device="cuda", generator=gen) - 0.5
    fv = _forward(aai, plan, v, mode)
    ftg = _adjoint(aai, plan, g, mode)
    lhs = float((fv * g).sum())
    rhs = float((v * ftg).sum())
    bound = 1e-10 * float((fv.abs() * g.abs()).sum())
    assert abs(lhs - rhs) <= bound, (lhs, rhs, bound)
    del v, fv, ftg
    # v = 1, g = 1: the total coverage is the number of canvas pixels the forward writes as non-zero
    ones_src = torch.ones((1, h, w, 1), dtype=torch.float64, device="cuda")
    written = int((_forward(aai, plan, ones_src, mode) != 0).sum())
    cover = _adjoint(aai, plan, torch.ones((1, plan.dst_h, plan.dst_w, 1), dtype=torch.float64, device="cuda"), mode)
    assert abs(float(cover.sum()) - written) <= 1e-9 * written, (float(cover.sum()), written)


# ---- 3. stacks and determinism ----------------------------------------------------------------------------------------

@pytest.mark.parametrize("mode,ratio,angle", [(1, 0.37, 17.3), (2, 0.37, 17.3), (3, 1.7, 107.3), (1, 0.5, 0.0)])
def test_stack_is_one_launch_and_bitwise_per_image(aai, mode, ratio, angle):
    import torch

    w, h, ch, n = 150, 130, 3, 5
    plan = aai.make_plan(w, h, 1.0, ratio, (75.0, 65.0), angle)
    g = torch.randn((n, plan.dst_h, plan.dst_w, ch), dtype=torch.float64, device="cuda")
    before = aai.launch_count()
    _adjoint(aai, plan, g[:1].clone(), mode)
    one = aai.launch_count() - before
    before = aai.launch_count()
    stack = _adjoint(aai, plan, g, mode)
    assert aai.launch_count() - before == one == 2  # normaliser + gather
    per_image = torch.cat([_adjoint(aai, plan, g[k:k + 1].clone(), mode) for k in range(n)])
    # a list that is not an equally strided stack (descending addresses) runs image by image
    parts = [g[k].clone() for k in range(n)]
    outs = [torch.empty((h, w, ch), dtype=g.dtype, device="cuda") for _ in range(n)]
    aai.run_device_adjoint(plan, [aai.tensor_image(p) for p in parts[::-1]], [aai.tensor_image(o) for o in outs[::-1]],
                           mode=mode, stream=_stream())
    again = _adjoint(aai, plan, g, mode)
    torch.cuda.synchronize()
    assert torch.equal(stack, per_image)
    assert torch.equal(stack, torch.stack(outs))
    assert torch.equal(stack, again)


def test_list_mixing_element_types_and_channels(aai):
    """A list (not a stack) may mix float64 / float32 images and channel counts: each image runs with its own element
    type and channel count, bitwise as in a call of its own."""
    import torch

    plan = aai.make_plan(90, 70, 1.0, 0.37, (45.0, 35.0), 17.3)
    shapes = [(torch.float64, 1), (torch.float32, 3), (torch.float64, 4), (torch.float32, 1)]
    gs = [torch.randn((plan.dst_h, plan.dst_w, c), dtype=dt, device="cuda") for dt, c in shapes]
    # each output is the top of a taller buffer: the guard rows below it must stay untouched
    bufs = [torch.full((plan.src_h * 3, plan.src_w, c), 7.0, dtype=dt, device="cuda") for dt, c in shapes]
    outs = [b[:plan.src_h] for b in bufs]
    aai.run_device_adjoint(plan, [aai.tensor_image(g) for g in gs], [aai.tensor_image(o) for o in outs], mode=1,
                           stream=_stream())
    singles = [_adjoint(aai, plan, g[None], 1)[0] for g in gs]
    torch.cuda.synchronize()
    for b, o, one in zip(bufs, outs, singles):
        assert torch.equal(o, one)
        assert bool((b[plan.src_h:] == 7.0).all())


# ---- 4. the torch entry point -----------------------------------------------------------------------------------------

GRAD_PLANS = {
    "rotated": (9, 7, 0.37, 17.3, (4.0, 3.0)),
    "axis": (8, 6, 0.5, 0.0, (4.0, 3.0)),
    "scale3": (6, 5, 1.7, 30.0, (3.0, 2.5)),
}


@pytest.mark.parametrize("ch", [1, 3])
@pytest.mark.parametrize("mode", [1, 2, 3])
@pytest.mark.parametrize("name", list(GRAD_PLANS))
def test_gradcheck_and_gradgradcheck(aai, name, mode, ch):
    import torch

    w, h, ratio, angle, iso = GRAD_PLANS[name]
    plan = aai.make_plan(w, h, 1.0, ratio, iso, angle)
    shape = (2, h, w) if ch == 1 else (2, h, w, ch)
    src = torch.rand(shape, dtype=torch.float64, device="cuda", requires_grad=True)
    fn = lambda x: aai.resample(x, plan, mode=mode)  # noqa: E731
    assert torch.autograd.gradcheck(fn, (src,))
    assert torch.autograd.gradgradcheck(fn, (src,))
    canvas = torch.rand((2, plan.dst_h, plan.dst_w) + (() if ch == 1 else (ch,)), dtype=torch.float64, device="cuda",
                        requires_grad=True)
    assert torch.autograd.gradcheck(lambda c: aai.resample_adjoint(c, plan, mode=mode), (canvas,))


@pytest.mark.parametrize("dtype", ["float64", "float32"])
@pytest.mark.parametrize("rank", [2, 3, 4])
def test_torch_forward_and_backward_are_the_c_abi_bitwise(aai, dtype, rank):
    import torch

    dt = getattr(torch, dtype)
    w, h = 120, 90
    plan = aai.make_plan(w, h, 1.0, 0.37, (60.0, 45.0), 117.3)
    shape = {2: (h, w), 3: (3, h, w), 4: (3, h, w, 2)}[rank]
    src = torch.rand(shape, dtype=dt, device="cuda", requires_grad=True)
    out = aai.resample(src, plan, mode=1)
    assert out.dtype == dt and out.dim() == rank
    stack = src.detach().reshape((-1, h, w, shape[3] if rank == 4 else 1))
    want = _forward(aai, plan, stack, 1)
    torch.cuda.synchronize()
    assert torch.equal(out.detach().reshape(want.shape), want)
    # backward with a grad_output whose rows are not dense
    gout = torch.rand(out.shape[:-1] + (out.shape[-1] * 2,), dtype=dt, device="cuda")[..., ::2]
    out.backward(gout)
    want_g = _adjoint(aai, plan, gout.contiguous().reshape(want.shape), 1)
    torch.cuda.synchronize()
    assert src.grad.shape == src.shape
    assert torch.equal(src.grad.reshape(want_g.shape), want_g)


def test_side_stream(aai):
    import torch

    w, h = 200, 160
    plan = aai.make_plan(w, h, 1.0, 0.37, (100.0, 80.0), 30.0)
    src = torch.rand((4, h, w), dtype=torch.float64, device="cuda", requires_grad=True)
    ref_out = aai.resample(src, plan)
    ref_out.sum().backward()
    ref_grad = src.grad.clone()
    src.grad = None
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        out = aai.resample(src, plan)
        back = aai.resample_adjoint(torch.ones_like(out), plan)
    side.synchronize()
    assert torch.equal(out, ref_out.detach()) and torch.equal(back, ref_grad)


@pytest.mark.parametrize("np_dtype", ["uint8", "uint16"])
def test_integer_sources_are_forward_only(aai, np_dtype):
    import torch

    w, h = 100, 80
    plan = aai.make_plan(w, h, 1.0, 0.37, (50.0, 40.0), 17.3)
    a = np.random.default_rng(3).integers(0, 250, size=(2, h, w)).astype(np_dtype)
    t = torch.from_numpy(a.view(np.int16) if np_dtype == "uint16" else a).cuda()
    t = t.view(torch.uint16) if np_dtype == "uint16" else t
    out = aai.resample(t, plan)
    assert out.dtype == torch.float32 and not out.requires_grad
    want = aai.resample(torch.from_numpy(a.astype(np.float32)).cuda(), plan)
    torch.cuda.synchronize()
    assert torch.allclose(out, want.detach(), rtol=1e-6, atol=1e-4)


def test_plan_errors(aai):
    import torch

    bad = aai.make_plan(40, 30, -1.0, 0.5, (20.0, 15.0), 17.3)
    x = torch.zeros((30, 40), dtype=torch.float64, device="cuda")
    with pytest.raises(aai.AaiError):
        aai.resample(x, bad)
    other = aai.make_plan(41, 30, 1.0, 0.5, (20.0, 15.0), 17.3)
    with pytest.raises(aai.AaiError, match="plan expects"):
        aai.resample(x, other)
    with pytest.raises(aai.AaiError):
        aai.resample_adjoint(torch.zeros((3, 3), dtype=torch.float64, device="cuda"), other)
