"""GPU (-m gpu): the adjoint and the forward against single columns of the reference operator W at full size, and every
launch split of the batched and row-sliced entry points.

* adjoint: F^T g of a random dense g, at ~2000 sampled source pixels s, against sum_p W[p, s] g[p] over the oracle's
  window of column s (tests/common.py: column_window, oracle_column);
* forward: a comb of unit impulses far enough apart that no footprint meets two, so that every non-zero canvas pixel
  holds one pair weight W[p, s]; FP64 and FP32 paths against the oracle over the windows of ~2000 impulses;
* launch splits: row slabs of AAI_MAX_ROWS_PER_LAUNCH rows (forward and both adjoint kernels), the grid.z / grid.y limit
  of 65535 images per launch, and the clamp that keeps a stack's row indices below 2^31.  Outputs are prefilled with
  NaN, so that a row or an image that no launch writes fails.
"""
import numpy as np
import pytest

from common import column_window, f32_err, oracle_column

pytestmark = pytest.mark.gpu

SLAB = 65535 * 8  # AAI_MAX_ROWS_PER_LAUNCH: grid.y limit x tile rows


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
    """F^T g through the C ABI into a NaN-prefilled [N, src_h, src_w, C] tensor; g is [N, dst_h, dst_w, C]."""
    import torch

    n, _, _, c = g.shape
    out = torch.full((n, plan.src_h, plan.src_w, c), float("nan"), dtype=g.dtype, device=g.device)
    aai.run_device_adjoint(plan, [aai.tensor_image(g[k]) for k in range(n)], [aai.tensor_image(out[k]) for k in range(n)],
                           mode=mode, stream=_stream())
    return out


# w, h, channels, ratio, angle, iso, mode; L = footprint side in expanded cells
FULL = {
    "cfg4_mode1": (16384, 16384, 1, 0.37, 17.3, (8192.0, 8192.0), 1),
    "cfg4_mode2": (16384, 16384, 1, 0.37, 17.3, (8192.0, 8192.0), 2),
    "cfg3_rgb": (8192, 8192, 3, 1.7, 45.0, (4095.5, 4095.5), 1),
    "cfg5_slice": (4096, 4096, 1, 0.5, 0.0, (2048.0, 2048.0), 1),
    "down_0.11": (4096, 4096, 1, 0.11, 33.7, (2047.3, 2050.6), 1),          # L = 9.09
    "sqrt2_below_1": (4096, 4096, 1, 0.70706, 45.0, (2047.3, 2050.6), 1),   # scale 1, L = 1.41431 just above sqrt 2
    "sqrt2_below_2": (4096, 4096, 1, 1.41413, 45.0, (2047.3, 2050.6), 3),   # scale 2, L = 1.41433 just above sqrt 2
    "q1_90": (4096, 4096, 1, 0.37, 90.0, (2047.3, 2050.6), 1),
    "q2_180": (4096, 4096, 1, 0.37, 180.0, (2047.3, 2050.6), 2),
    "q3_270": (4096, 4096, 1, 0.37, 270.0, (2047.3, 2050.6), 3),
}
N_SAMPLES = 2000


def _plan(aai, name):
    w, h, ch, ratio, angle, iso, mode = FULL[name]
    plan = aai.make_plan(w, h, 1.0, ratio, iso, angle)
    assert plan.status == 0
    return plan


def test_full_geometries_are_what_they_claim(aai):
    import math

    # the footprint side L in expanded cells just above sqrt 2, the widest a unit cell gets across a footprint row:
    # the adjoint's candidate range 1/2 + (cos + sin) / (2 L) is then almost a whole canvas pixel either way
    for name, scale in (("sqrt2_below_1", 1), ("sqrt2_below_2", 2)):
        p = _plan(aai, name)
        assert p.scale == scale and math.sqrt(2) < p.side < math.sqrt(2) * (1 + 1e-4), name
    assert _plan(aai, "down_0.11").side > 9.0
    assert _plan(aai, "cfg3_rgb").mod_w == 24576 and _plan(aai, "cfg3_rgb").dst_w > 19000
    assert [_plan(aai, n).quadrant for n in ("q1_90", "q2_180", "q3_270")] == [1, 2, 3]


def _source_samples(plan, n, seed):
    """Deterministic source pixels: the four corners, pixels along the four edges (among them the ones whose footprints
    touch the canvas border), pixels on both sides of multiples of the 16 x 8 tile, and a seeded random rest."""
    w, h = int(plan.src_w), int(plan.src_h)
    rng = np.random.default_rng(seed)
    pts = [(0, 0), (w - 1, 0), (0, h - 1), (w - 1, h - 1)]
    for t in np.linspace(0, 1, 40):
        x, y = int(round(t * (w - 1))), int(round(t * (h - 1)))
        pts += [(x, 0), (x, h - 1), (0, y), (w - 1, y)]
    for _ in range(60):
        tx, ty = 16 * int(rng.integers(1, max(2, w // 16))), 8 * int(rng.integers(1, max(2, h // 8)))
        pts += [(min(tx, w - 1), min(ty, h - 1)), (tx - 1, ty - 1), (min(tx, w - 1), ty - 1), (tx - 1, min(ty, h - 1))]
    while len(pts) < n:
        pts.append((int(rng.integers(0, w)), int(rng.integers(0, h))))
    seen, out = set(), []
    for p in pts:
        if p not in seen:
            seen.add(p)
            out.append(p)
    return out


def _windows_to_host(t, wins):
    """t[y0:y1, x0:x1, ...] of every window, gathered on the device and copied back in one transfer."""
    import torch

    idx = []
    for y0, y1, x0, x1 in wins:
        yy, xx = np.meshgrid(np.arange(y0, y1), np.arange(x0, x1), indexing="ij")
        idx.append((yy * t.shape[1] + xx).ravel())
    flat = torch.from_numpy(np.concatenate(idx)).to(t.device)
    vals = t.reshape((t.shape[0] * t.shape[1],) + tuple(t.shape[2:]))[flat].double().cpu().numpy()
    out, k = [], 0
    for (y0, y1, x0, x1), i in zip(wins, idx):
        out.append(vals[k:k + i.size].reshape((y1 - y0, x1 - x0) + tuple(t.shape[2:])))
        k += i.size
    return out


def _ill_conditioned_column(oracle, impulse, args, sx, sy, mode, col, delta=1e-11):
    """T5 (test_gpu_parity._conditioning_mask) on one column's window: the reference's own column changes when the
    isocentre moves by 1e-11 in one of 8 directions."""
    src_res, dst_res, iso, angle = args
    scale = max(np.abs(col).max(), 1e-300)
    for dx, dy in [(1, 1), (-1, -1), (1, 0), (0, 1), (-1, 0), (0, -1), (1, -1), (-1, 1)]:
        moved_iso = (iso[0] + dx * delta, iso[1] + dy * delta)
        _, moved = oracle_column(oracle, impulse, (src_res, dst_res, moved_iso, angle), sx, sy, 0, mode)
        if moved.shape != col.shape or np.abs(moved - col).max() > 1e-9 * scale:
            return True
    return False


# ---- 1. adjoint, pixel by pixel ---------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", list(FULL))
def test_adjoint_columns_at_full_size(aai, oracle, name):
    import torch

    w, h, ch, ratio, angle, iso, mode = FULL[name]
    plan = _plan(aai, name)
    args = (1.0, ratio, iso, angle)
    samples = _source_samples(plan, N_SAMPLES, seed=w + int(100 * ratio))
    wins = [column_window(plan, sx, sy) for sx, sy in samples]
    assert any(y0 == 0 or x0 == 0 or y1 == plan.dst_h or x1 == plan.dst_w for y0, y1, x0, x1 in wins)
    sel = torch.tensor([sy * w + sx for sx, sy in samples], device="cuda")
    gen = torch.Generator(device="cuda").manual_seed(17)
    g64 = torch.rand((1, plan.dst_h, plan.dst_w, ch), dtype=torch.float64, device="cuda", generator=gen) - 0.5
    got, gwin = {}, {}
    for dt in (torch.float64, torch.float32):
        g = g64 if dt == torch.float64 else g64.to(dt)
        out = _adjoint(aai, plan, g, mode)
        assert not bool(out.isnan().any()), "source pixels that no launch wrote"
        got[dt] = out.reshape(h * w, ch)[sel].double().cpu().numpy()
        gwin[dt] = _windows_to_host(g[0], wins)
        del g, out
    del g64
    torch.cuda.empty_cache()
    impulse = np.zeros((h, w), dtype=np.uint8)
    masked = 0
    for k, (sx, sy) in enumerate(samples):
        win, col = oracle_column(oracle, impulse, args, sx, sy, 0, mode)
        assert win == wins[k]
        bad = False
        for dt, tol in ((torch.float64, 1e-9), (torch.float32, 1e-5)):
            gw = gwin[dt][k]
            want = np.einsum("yx,yxc->c", col, gw)
            bound = tol * np.einsum("yx,yxc->c", np.abs(col), np.abs(gw))
            bad |= not (np.abs(got[dt][k] - want) <= bound).all()
        if bad:
            assert _ill_conditioned_column(oracle, impulse, args, sx, sy, mode, col), (
                name, (sx, sy), got[torch.float64][k], np.einsum("yx,yxc->c", col, gwin[torch.float64][k]))
            masked += 1
    assert masked <= len(samples) // 100, (name, masked)


# ---- 2. forward, pair by pair -----------------------------------------------------------------------------------------

def _comb_axis(n, spacing):
    """Impulse positions along one axis: a lattice from 0, and the last index, every two at least `spacing` apart."""
    return np.array(sorted(set(range(0, max(1, n - spacing), spacing)) | {n - 1}))


@pytest.mark.parametrize("name", list(FULL))
def test_forward_columns_at_full_size(aai, oracle, name):
    import torch

    w, h, ch, ratio, angle, iso, mode = FULL[name]
    plan = _plan(aai, name)
    # a footprint spans at most L (cos + sin) expanded cells per axis, i.e. that over scale source pixels: a larger
    # spacing keeps every footprint on one impulse at most
    spacing = int(np.ceil(plan.side * (plan.cos_t + plan.sin_t) / plan.scale)) + 3
    xs, ys = _comb_axis(w, spacing), _comb_axis(h, spacing)
    comb = np.zeros((h, w, ch), dtype=np.uint8)
    for c in range(ch):
        comb[np.ix_(ys, xs, [c])] = c + 1  # channel c carries the impulse c + 1
    rng = np.random.default_rng(5)
    corners = [(xs[0], ys[0]), (xs[-1], ys[0]), (xs[0], ys[-1]), (xs[-1], ys[-1])]
    edges = [(x, y) for x in xs[::max(1, len(xs) // 40)] for y in (ys[0], ys[-1])] + \
            [(x, y) for y in ys[::max(1, len(ys) // 40)] for x in (xs[0], xs[-1])]
    rest = list(zip(rng.choice(xs, N_SAMPLES), rng.choice(ys, N_SAMPLES)))
    samples = list(dict.fromkeys([(int(x), int(y)) for x, y in corners + edges + rest]))[:N_SAMPLES]
    wins = [column_window(plan, sx, sy) for sx, sy in samples]
    src = torch.from_numpy(comb).cuda()
    got = {}
    for arith, dt in ((aai.ARITH_F64, torch.float64), (aai.ARITH_F32, torch.float32)):
        dst = torch.full((plan.dst_h, plan.dst_w, ch), float("nan"), dtype=dt, device="cuda")
        aai.run_device(plan, aai.tensor_image(src), aai.tensor_image(dst), mode=mode, arith=arith, stream=_stream())
        assert not bool(dst.isnan().any()), "canvas pixels that no launch wrote"
        got[arith] = _windows_to_host(dst, wins)
        del dst
    del src
    torch.cuda.empty_cache()
    masked = 0
    for k, ((sx, sy), (y0, y1, x0, x1)) in enumerate(zip(samples, wins)):
        bad = False
        for c in range(ch):
            st, want, _ = oracle.run(comb, 1.0, ratio, iso, angle, mode=mode, rows=(y0, y1), cols=(x0, x1), channel=c,
                                     threads=1)
            assert st == 0
            # an empty column (got must be 0 too): the canvas, whose size is truncated, ends short of a source edge
            top = np.abs(want).max()
            assert top > 0 or sx in (0, w - 1) or sy in (0, h - 1), ("impulse without a column", (sx, sy))
            for arith, tol in ((aai.ARITH_F64, 1e-9), (aai.ARITH_F32, 1e-5)):
                g = got[arith][k][..., c]
                support = ((g != 0) == (want != 0)) | (np.abs(want) < 1e-12 * top)
                bad |= not ((np.abs(g - want) <= tol * top).all() and support.all())
        if bad:
            impulse = np.zeros((h, w), dtype=np.uint8)
            _, col = oracle_column(oracle, impulse, (1.0, ratio, iso, angle), sx, sy, 0, mode)
            assert _ill_conditioned_column(oracle, impulse, (1.0, ratio, iso, angle), sx, sy, mode, col), (name, (sx, sy))
            masked += 1
    assert masked <= len(samples) // 100, (name, masked)


# ---- 3. launch splits -------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("mode", [1, 2])
@pytest.mark.parametrize("angle", [0.0, 90.0, 180.0, 270.0])
def test_adjoint_row_slabs(aai, oracle, angle, mode):
    """A 3 x 530 000 line scan: the gather runs over source rows in slabs of SLAB rows; the normaliser over canvas rows,
    which exceed SLAB at 0 and 180 degrees only."""
    import torch

    w, h, iso = 3, 530000, (1.0, 265000.3)
    plan = aai.make_plan(w, h, 1.0, 1.0, iso, angle)
    assert plan.status == 0 and (plan.dst_h > SLAB) == (angle in (0.0, 180.0))
    g = torch.from_numpy(np.random.default_rng(9).uniform(-0.5, 0.5, (1, plan.dst_h, plan.dst_w, 1))).cuda()
    before = aai.launch_count()
    out = _adjoint(aai, plan, g, mode)
    assert aai.launch_count() - before == (2 if plan.dst_h > SLAB else 1) + 2
    assert not bool(out.isnan().any()), "source pixels that no launch wrote"
    # source rows on both sides of a gather slab boundary, source rows whose canvas rows straddle a normaliser slab
    # boundary, the first and the last rows
    rows = {0, 1, h - 2, h - 1} | set(range(SLAB - 3, SLAB + 3))
    for y in range(SLAB - 8, SLAB + 8):
        for yy in (y, h - 1 - y):  # at 180 degrees canvas row y holds source rows near h - 1 - y
            y0, y1, _, _ = column_window(plan, 1, yy)
            if plan.dst_h > SLAB and y0 <= SLAB <= y1:
                rows.add(yy)
    impulse = np.zeros((h, w), dtype=np.uint8)
    gh = g[0].cpu().numpy()
    got = out[0].cpu().numpy()
    for sy in sorted(rows):
        for sx in range(w):
            (y0, y1, x0, x1), col = oracle_column(oracle, impulse, (1.0, 1.0, iso, angle), sx, sy, 0, mode)
            gw = gh[y0:y1, x0:x1, 0]
            want = float((col * gw).sum())
            assert abs(got[sy, sx, 0] - want) <= 1e-9 * float((np.abs(col) * np.abs(gw)).sum()), (angle, mode, sx, sy)


def _stack_case(aai, angle):
    ratio = 0.37 if angle else 0.5
    plan = aai.make_plan(24, 20, 1.0, ratio, (11.3, 9.7), angle)
    assert plan.status == 0 and plan.axis_aligned == (angle == 0.0)
    return plan, (1.0, ratio, (11.3, 9.7), angle)


@pytest.mark.parametrize("angle", [17.3, 0.0])
def test_stack_beyond_the_grid_limit(aai, oracle, angle):
    """65 537 images of 24 x 20: two forward launches (grid.z; grid.y of the separable TMA kernel on the axis-aligned
    plan, whose 96-byte float rows are 16-byte aligned) and a normaliser plus two gathers for the adjoint.  The images
    on both sides of each cut equal per-image calls bitwise and the oracle."""
    import torch

    n, w, h = 65537, 24, 20
    plan, args = _stack_case(aai, angle)
    gen = torch.Generator(device="cuda").manual_seed(23)
    src = torch.rand((n, h, w), dtype=torch.float32, device="cuda", generator=gen)
    g = torch.rand((n, plan.dst_h, plan.dst_w), dtype=torch.float32, device="cuda", generator=gen) - 0.5
    dst = torch.full((n, plan.dst_h, plan.dst_w), float("nan"), dtype=torch.float32, device="cuda")
    back = torch.full((n, h, w), float("nan"), dtype=torch.float32, device="cuda")
    before = aai.launch_count()
    aai.run_device_batch(plan, [aai.tensor_image(src[k]) for k in range(n)], [aai.tensor_image(dst[k]) for k in range(n)],
                         arith=aai.ARITH_F32, stream=_stream())
    assert aai.launch_count() - before == 2
    before = aai.launch_count()
    aai.run_device_adjoint(plan, [aai.tensor_image(g[k]) for k in range(n)], [aai.tensor_image(back[k]) for k in range(n)],
                           stream=_stream())
    assert aai.launch_count() - before == 1 + 2
    assert not bool(dst.isnan().any()) and not bool(back.isnan().any()), "images that no launch wrote"
    # the torch entry point: the same launches under autograd
    x = src.clone().requires_grad_(True)
    y = aai.resample(x, plan, arith=aai.ARITH_F32)
    y.backward(g)
    torch.cuda.synchronize()
    assert torch.equal(y.detach(), dst) and torch.equal(x.grad, back)
    del x, y
    for k in (0, 65534, 65535, 65536):
        one = torch.full((plan.dst_h, plan.dst_w), float("nan"), dtype=torch.float32, device="cuda")
        aai.run_device(plan, aai.tensor_image(src[k]), aai.tensor_image(one), arith=aai.ARITH_F32, stream=_stream())
        one_back = _adjoint(aai, plan, g[k][None, ..., None], 1)[0, ..., 0]
        torch.cuda.synchronize()
        assert torch.equal(dst[k], one) and torch.equal(back[k], one_back), k
        host = src[k].cpu().numpy()
        st, want, _ = oracle.run(host, *args)
        assert st == 0 and f32_err(dst[k].cpu().numpy(), want, 1.0).max() <= 1e-5, k
        gk = g[k].double().cpu().numpy()
        impulse = np.zeros((h, w), dtype=np.uint8)
        bk = back[k].cpu().numpy()
        for sy in range(h):
            for sx in range(w):
                (y0, y1, x0, x1), col = oracle_column(oracle, impulse, args, sx, sy, 0, 1)
                gw = gk[y0:y1, x0:x1]
                assert abs(bk[sy, sx] - (col * gw).sum()) <= 1e-5 * (np.abs(col) * np.abs(gw)).sum(), (k, sx, sy)
    del src, g, dst, back
    torch.cuda.empty_cache()


def test_stack_rows_beyond_int32(aai, oracle):
    """65 535 width-1 uint8 images of 32 769 rows: the grid.z kernels address the stack as one tall image with int32
    rows, so the batch is cut where the row index would pass 2^31 - 1 (65 534 images in the first launch)."""
    import torch

    n, h = 65535, 32769
    args = (1.0, 0.5, (0.3, 16384.3), 0.0)
    plan = aai.make_plan(1, h, *args)
    assert plan.status == 0 and n * h > 2**31 - 1 and plan.dst_w == 1
    cut = (2**31 - 1) // max(h, int(plan.dst_h))
    assert cut == 65534
    gen = torch.Generator(device="cuda").manual_seed(29)
    src = torch.randint(0, 256, (n, h, 1), dtype=torch.uint8, device="cuda", generator=gen)
    dst = torch.full((n, plan.dst_h, 1), float("nan"), dtype=torch.float32, device="cuda")
    before = aai.launch_count()
    aai.run_device_batch(plan, [aai.tensor_image(src[k]) for k in range(n)], [aai.tensor_image(dst[k]) for k in range(n)],
                         arith=aai.ARITH_F32, stream=_stream())
    assert aai.launch_count() - before == 2
    assert not bool(dst.isnan().any()), "images that no launch wrote"
    for k in (0, cut - 1, cut, n - 1):
        one = torch.full((plan.dst_h, 1), float("nan"), dtype=torch.float32, device="cuda")
        aai.run_device(plan, aai.tensor_image(src[k]), aai.tensor_image(one), arith=aai.ARITH_F32, stream=_stream())
        torch.cuda.synchronize()
        assert torch.equal(dst[k], one), k
        host = src[k].cpu().numpy()
        st, want, _ = oracle.run(host, *args)
        assert st == 0 and np.abs(one.cpu().numpy() - want).max() <= 1e-5 * 255.0, k
    del src, dst
    torch.cuda.empty_cache()
