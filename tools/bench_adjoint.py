#!/usr/bin/env python
"""Device time of the adjoint (aai_run_device_adjoint) against the forward kernels; writes OUTDIR/bench_adjoint.json.

    python tools/bench_adjoint.py OUTDIR [--launches 20]

Shapes (float32 sources, float32 gradients):
    cfg4_mode1   BASELINE config 4 (16384^2, 0.37x, 17.3 deg), area average
    cfg4_mode2   the same in fast mode
    cfg3_rgb     config 3 geometry (8192^2 RGB float32, 1.7x, 45 deg, scale 3), area average
    cfg5         config 5 (256 x 4096^2, 0.5x, 0 deg), area average, every call one launch per kernel
Per shape: the FP64 forward, the FP32 forward and the adjoint, each as CUDA events around `launches` back-to-back calls
after a warm-up (median of 3 rounds, per call); one forward + backward step of `resample` (ARITH_F32 forward); and, from
a separate torch.profiler run, the device time of each adjoint kernel.  Every source is larger than the 126 MB L2.
The card's name, power limit and maximum SM clock are read with one nvidia-smi query in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = {
    "cfg4_mode1": dict(w=16384, h=16384, n=1, ch=1, ratio=0.37, angle=17.3, iso=(8192.0, 8192.0), mode=1),
    "cfg4_mode2": dict(w=16384, h=16384, n=1, ch=1, ratio=0.37, angle=17.3, iso=(8192.0, 8192.0), mode=2),
    "cfg3_rgb": dict(w=8192, h=8192, n=1, ch=3, ratio=1.7, angle=45.0, iso=(4095.5, 4095.5), mode=1),
    "cfg5": dict(w=4096, h=4096, n=256, ch=1, ratio=0.5, angle=0.0, iso=(2048.0, 2048.0), mode=1),
}


def gpu_info() -> dict:
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    first = out.stdout.strip().splitlines()[0] if out.returncode == 0 and out.stdout.strip() else ""
    parts = [p.strip() for p in first.split(",")] if first else []
    return dict(zip(["name", "power_limit", "max_sm_clock"], parts)) if len(parts) == 3 else {"query": out.stdout + out.stderr}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--launches", type=int, default=20)
    ap.add_argument("--shapes", default=",".join(SHAPES))
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile

    import area_average_interpolation_b200 as aai

    if aai.device_count() < 1 or not torch.cuda.is_available():
        raise SystemExit("bench_adjoint: no CUDA device (nothing is measured without one)")
    torch.cuda.set_device(0)
    os.makedirs(args.outdir, exist_ok=True)
    res = {"gpu": gpu_info(), "torch": torch.__version__, "launches": args.launches, "unit": "ms per call",
           "shapes": {}}

    def timed(fn):
        fn()
        torch.cuda.synchronize()
        rounds = []
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.launches):
                fn()
            e1.record()
            torch.cuda.synchronize()
            rounds.append(e0.elapsed_time(e1) / args.launches)
        return statistics.median(rounds)

    for name in args.shapes.split(","):
        s = SHAPES[name]
        plan = aai.make_plan(s["w"], s["h"], 1.0, s["ratio"], s["iso"], s["angle"])
        n, ch, mode = s["n"], s["ch"], s["mode"]
        src = torch.rand((n, s["h"], s["w"], ch), dtype=torch.float32, device="cuda")
        canvas = torch.empty((n, plan.dst_h, plan.dst_w, ch), dtype=torch.float32, device="cuda")
        grad = torch.rand((n, plan.dst_h, plan.dst_w, ch), dtype=torch.float32, device="cuda")
        sgrad = torch.empty_like(src)
        si = [aai.tensor_image(src[k]) for k in range(n)]
        ci = [aai.tensor_image(canvas[k]) for k in range(n)]
        gi = [aai.tensor_image(grad[k]) for k in range(n)]
        oi = [aai.tensor_image(sgrad[k]) for k in range(n)]
        st = torch.cuda.current_stream().cuda_stream
        fwd64 = lambda: aai.run_device_batch(plan, si, ci, mode=mode, arith=aai.ARITH_F64, stream=st)  # noqa: E731
        fwd32 = lambda: aai.run_device_batch(plan, si, ci, mode=mode, arith=aai.ARITH_F32, stream=st)  # noqa: E731
        adj = lambda: aai.run_device_adjoint(plan, gi, oi, mode=mode, stream=st)  # noqa: E731
        before = aai.launch_count()
        adj()
        torch.cuda.synchronize()
        rec = {"source": [n, s["h"], s["w"], ch], "canvas": [n, plan.dst_h, plan.dst_w, ch], "mode": mode,
               "scale": plan.scale, "adjoint_launches_per_call": aai.launch_count() - before,
               "forward_f64_ms": timed(fwd64), "forward_f32_ms": timed(fwd32), "adjoint_ms": timed(adj)}
        rec["adjoint_over_forward_f64"] = rec["adjoint_ms"] / rec["forward_f64_ms"]
        # one training step: forward (FP32 arithmetic) + backward through the adjoint
        x = src.detach().clone().requires_grad_(True)
        src_view = x if ch > 1 else x[..., 0]
        g_view = grad if ch > 1 else grad[..., 0]

        def step():
            x.grad = None
            aai.resample(src_view, plan, mode=mode, arith=aai.ARITH_F32).backward(g_view)

        rec["resample_fwd_bwd_ms"] = timed(step)
        # per-kernel device times, separate profiled run (nothing else in flight when it starts)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA], acc_events=True) as prof:
            for _ in range(5):
                adj()
            torch.cuda.synchronize()
        kern = {}
        for ev in prof.key_averages():
            if "adjoint" in ev.key:
                t = getattr(ev, "device_time", None) or getattr(ev, "cuda_time", 0.0)
                kern[ev.key] = {"avg_ms": t / 1000.0, "count": ev.count}
        rec["adjoint_kernels"] = kern
        res["shapes"][name] = rec
        print(name, json.dumps(rec), flush=True)
        del src, canvas, grad, sgrad, x
        torch.cuda.empty_cache()
    with open(os.path.join(args.outdir, "bench_adjoint.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
