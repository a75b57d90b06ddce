#!/usr/bin/env python
"""16-bit sources against float32 ones on the shapes the library is measured on; writes OUTDIR/bench_u16.json.

    python tools/bench_u16.py OUTDIR [--reps 5] [--lib other/libaai_b200.so --name variant]

W1      BASELINE config 4 geometry (16384^2, 0.37x, 17.3 deg), FP32 area average: f32->f32, u16->f32, u16->u16
W2      the same geometry in fast mode: f32->f32 (128-bit-load kernel) against u16->f32 / u16->u16 (scalar-load kernel)
W3      BASELINE config 5 geometry (256 x 4096^2, 0.5x, 0 deg), ONE batched separable launch: f32->f32, u16->f32,
        u16->u16; achieved bytes/s (source read once + canvas written once) against an HBM copy measured in the same run
W3-e2e  W3's geometry through aai_run_host_batch with pinned host buffers (64 slices: the rate is PCIe-bound)

Kernel times are CUDA events around `launches` back-to-back launches after a warm-up, the variants of a workload
alternated over `reps` rounds, median per launch.  Every source is larger than the 126 MB L2.  The card's name, power
limit and maximum SM clock are read with one nvidia-smi query in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info() -> dict:
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    first = out.stdout.strip().splitlines()[0] if out.returncode == 0 and out.stdout.strip() else ""
    parts = [p.strip() for p in first.split(",")] if first else []
    return dict(zip(["name", "power_limit", "max_sm_clock"], parts)) if len(parts) == 3 else {"query": out.stdout + out.stderr}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--lib", default="", help="another build of libaai_b200.so (A/B of a variant)")
    ap.add_argument("--name", default="bench_u16", help="output file OUTDIR/<name>.json")
    args = ap.parse_args()
    import torch

    import area_average_interpolation_b200 as aai

    if args.lib:
        aai.LIB_PATH = os.path.abspath(args.lib)
    from area_average_interpolation_b200.synthetic import synthetic_image_torch

    if aai.device_count() < 1 or not torch.cuda.is_available():
        raise SystemExit("bench_u16: no CUDA device (nothing is measured without one)")
    torch.cuda.set_device(0)
    stream = torch.cuda.current_stream().cuda_stream
    os.makedirs(args.outdir, exist_ok=True)
    res = {"gpu": gpu_info(), "torch": torch.__version__, "reps": args.reps, "lib": os.path.basename(aai.LIB_PATH)}
    t_dt = {"f32": torch.float32, "u16": torch.int16}

    def empty(shape, kind):  # uint16 through its int16 view (torch's CUDA uint16 kernels are few)
        t = torch.zeros(shape, dtype=t_dt[kind], device="cuda")
        return t.view(torch.uint16) if kind == "u16" else t

    def timed(fn, launches):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(launches):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / launches

    def compare(variants, launches, warmup=2):
        """variants: name -> fn.  Alternated over the rounds; median ms per launch."""
        for fn in variants.values():
            for _ in range(warmup):
                fn()
        torch.cuda.synchronize()
        ms = {k: [] for k in variants}
        for _ in range(args.reps):
            for k, fn in variants.items():
                ms[k].append(timed(fn, launches))
        return {k: {"ms": statistics.median(v), "ms_all": v} for k, v in ms.items()}

    # ---- W1 / W2: config 4 geometry ----
    W = 16384
    plan = aai.make_plan(W, W, 1.0, 0.37, (8192.0, 8192.0), 17.3)
    src = {"f32": synthetic_image_torch(W, W, np.float32, 20201 + 4, device="cuda"),
           "u16": synthetic_image_torch(W, W, np.uint16, 20201 + 4, device="cuda")}
    dst = {"f32": empty((plan.dst_h, plan.dst_w), "f32"), "u16": empty((plan.dst_h, plan.dst_w), "u16")}
    img = {k: aai.tensor_image(v) for k, v in src.items()}
    out = {k: aai.tensor_image(v) for k, v in dst.items()}
    pairs = [("f32", "f32"), ("u16", "f32"), ("u16", "u16")]

    def run1(s, d, mode):
        return lambda: aai.run_device(plan, img[s], out[d], mode=mode, arith=aai.ARITH_F32, stream=stream)

    for wl, mode, launches in (("W1", aai.MODE_AREA_AVERAGE, 10), ("W2", aai.MODE_FAST, 20)):
        r = compare({f"{s}->{d}": run1(s, d, mode) for s, d in pairs}, launches)
        for k, v in r.items():
            v["canvas_mpix_per_s"] = plan.dst_w * plan.dst_h / (v["ms"] * 1e-3) / 1e6
        base = r["f32->f32"]["ms"]
        for k in r:
            r[k]["vs_f32"] = r[k]["ms"] / base
        res[wl] = {"shape": f"{W}x{W} -> {plan.dst_w}x{plan.dst_h}, 0.37x, 17.3 deg, {'fast' if mode == 2 else 'area average'}, "
                            "ARITH_F32", "launches_per_round": launches, "results": r}
    del src, dst, img, out
    torch.cuda.empty_cache()

    # ---- W3: config 5 geometry, one batched launch ----
    n, S = 256, 4096
    plan5 = aai.make_plan(S, S, 1.0, 0.5, (2048.0, 2048.0), 0.0)
    distinct = 8
    stacks = {}
    for kind, np_dt in (("f32", np.float32), ("u16", np.uint16)):
        st = empty((n, S, S), kind)
        for k in range(distinct):
            st[k].view(t_dt[kind]).copy_(synthetic_image_torch(S, S, np_dt, 555 + k, device="cuda").view(t_dt[kind]))
        for k in range(distinct, n):
            st[k].view(t_dt[kind]).copy_(st[k % distinct].view(t_dt[kind]))
        stacks[kind] = st
    canv = {k: empty((n, plan5.dst_h, plan5.dst_w), k) for k in ("f32", "u16")}
    s_imgs = {k: [aai.tensor_image(v[i]) for i in range(n)] for k, v in stacks.items()}
    d_imgs = {k: [aai.tensor_image(v[i]) for i in range(n)] for k, v in canv.items()}

    def run3(s, d):
        return lambda: aai.run_device_batch(plan5, s_imgs[s], d_imgs[d], arith=aai.ARITH_F32, stream=stream)

    before = aai.launch_count()
    run3("u16", "u16")()
    torch.cuda.synchronize()
    launches_per_batch = aai.launch_count() - before
    r = compare({f"{s}->{d}": run3(s, d) for s, d in pairs}, 5)
    # HBM copy rate in the same run: a 4 GiB device-to-device copy (read + write)
    a = torch.empty(1 << 30, dtype=torch.float32, device="cuda")
    b = torch.empty_like(a)
    copy = compare({"copy": lambda: b.copy_(a)}, 5)["copy"]
    copy_gbs = 2 * a.numel() * 4 / (copy["ms"] * 1e-3) / 1e9
    del a, b
    esz = {"f32": 4, "u16": 2}
    base = r["f32->f32"]["ms"]
    for s, d in pairs:
        v = r[f"{s}->{d}"]
        nbytes = n * (S * S * esz[s] + plan5.dst_w * plan5.dst_h * esz[d])
        v["bytes"] = nbytes
        v["bytes_vs_f32"] = nbytes / (n * (S * S * 4 + plan5.dst_w * plan5.dst_h * 4))
        v["achieved_gbs"] = nbytes / (v["ms"] * 1e-3) / 1e9
        v["frac_of_copy"] = v["achieved_gbs"] / copy_gbs
        v["vs_f32"] = v["ms"] / base
    res["W3"] = {"shape": f"{n} x {S}x{S} -> {plan5.dst_w}x{plan5.dst_h}, 0.5x, 0 deg, ARITH_F32, run_device_batch",
                 "launches_per_batch": launches_per_batch, "hbm_copy_gbs": copy_gbs, "hbm_copy_ms": copy["ms"],
                 "results": r}
    del canv, d_imgs
    torch.cuda.empty_cache()

    # ---- W3-e2e: pinned host buffers through aai_run_host_batch ----
    ne = 64
    e2e = {}
    for s, d in pairs:
        hs = torch.empty((ne, S, S), dtype=t_dt[s], pin_memory=True)
        hs.copy_(stacks[s][:ne].view(t_dt[s]))
        hd = torch.zeros((ne, plan5.dst_h, plan5.dst_w), dtype=t_dt[d], pin_memory=True)
        if s == "u16":
            hs = hs.view(torch.uint16)
        if d == "u16":
            hd = hd.view(torch.uint16)
        si, di = [aai.tensor_image(hs[i]) for i in range(ne)], [aai.tensor_image(hd[i]) for i in range(ne)]
        aai.run_host_batch(plan5, si, di, arith=aai.ARITH_F32)  # warm-up (workspace allocation)
        wall = []
        for _ in range(args.reps):
            t0 = time.perf_counter()
            aai.run_host_batch(plan5, si, di, arith=aai.ARITH_F32)
            wall.append((time.perf_counter() - t0) * 1e3)
        nbytes = ne * (S * S * esz[s] + plan5.dst_w * plan5.dst_h * esz[d])
        ms = statistics.median(wall)
        e2e[f"{s}->{d}"] = {"ms": ms, "ms_all": wall, "pcie_bytes": nbytes, "gbs": nbytes / (ms * 1e-3) / 1e9}
        del hs, hd, si, di
    for k in e2e:
        e2e[k]["vs_f32"] = e2e[k]["ms"] / e2e["f32->f32"]["ms"]
    res["W3_e2e"] = {"shape": f"{ne} x {S}x{S} pinned host slices -> host canvases, ARITH_F32, run_host_batch",
                     "timing": "host wall clock around the blocking call, median", "results": e2e}
    path = os.path.join(args.outdir, args.name + ".json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({wl: {k: round(v.get("vs_f32", 0), 3) for k, v in res[wl]["results"].items()}
                      for wl in ("W1", "W2", "W3", "W3_e2e")}))
    print("wrote", path)


if __name__ == "__main__":
    main()
