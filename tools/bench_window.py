#!/usr/bin/env python
"""FP32 overlap kernel: the cell window + tips body against the full MAXN x MAXN body; writes OUTDIR/bench_window.json.

    tools/build_variant.sh no_tip_window -DAAI_TIP_WINDOW=0      # the full body for every plan; prints the .so it built
    python tools/bench_window.py OUTDIR --old <that no_tip_window.so>

Both builds are loaded into one process and alternated (the order flips every round) on BASELINE config 4 (16384^2
float32 -> 7591^2, 0.37x, 17.3 deg) and config 2 (2048^2 u8 -> 1035^2, 0.37x, 30 deg; both pass aai_tip_window_ok,
MAXN 5).  Kernel times are CUDA events around `launches` back-to-back launches after a warm-up, `rounds` rounds, median
per launch.  Config 4's 1 GB source is larger than the 126 MB L2.  For each build, the whole config-4 canvas of the FP32
kernel is compared with the FP64 kernel (max |f32 - f64| / |f64| over the pixels where f64 != 0) on the seeded synthetic
source.  The card's name, power limit and maximum SM clock are read with one nvidia-smi query in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CONFIGS = {  # bench.py's configs 4 and 2
    "cfg4": dict(w=16384, h=16384, dtype="float32", ratio=0.37, angle=17.3, iso=(8192.0, 8192.0), launches=50),
    "cfg2": dict(w=2048, h=2048, dtype="uint8", ratio=0.37, angle=30.0, iso=(1024.0, 1024.0), launches=1000),
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
    ap.add_argument("--old", required=True, help="build of libaai_b200.so with -DAAI_TIP_WINDOW=0")
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    import torch

    import area_average_interpolation_b200 as aai
    from area_average_interpolation_b200.synthetic import synthetic_image

    libs = {}
    for name, path in (("old", os.path.abspath(args.old)), ("new", aai.LIB_PATH)):
        aai.LIB_PATH, aai._lib_handle = path, None
        libs[name] = aai.lib()
    if aai.device_count() < 1 or not torch.cuda.is_available():
        raise SystemExit("bench_window: no CUDA device (nothing is measured without one)")
    torch.cuda.set_device(0)
    stream = torch.cuda.current_stream().cuda_stream
    os.makedirs(args.outdir, exist_ok=True)
    res = {"gpu": gpu_info(), "torch": torch.__version__, "rounds": args.rounds, "old": os.path.basename(args.old)}

    def use(name):
        aai._lib_handle = libs[name]

    for key, cfg in CONFIGS.items():
        plan = aai.make_plan(cfg["w"], cfg["h"], 1.0, cfg["ratio"], cfg["iso"], cfg["angle"])
        if cfg["dtype"] == "uint8":
            src = torch.randint(0, 256, (cfg["h"], cfg["w"]), dtype=torch.uint8, device="cuda")
        else:
            src = torch.rand((cfg["h"], cfg["w"]), dtype=torch.float32, device="cuda") * 4096
        dst = torch.empty((plan.dst_h, plan.dst_w), dtype=src.dtype, device="cuda")
        si, di = aai.tensor_image(src), aai.tensor_image(dst)
        times = {"old": [], "new": []}
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for r in range(args.rounds):
            for name in (("old", "new") if r % 2 == 0 else ("new", "old")):
                use(name)
                for _ in range(3):
                    aai.run_device(plan, si, di, arith=aai.ARITH_F32, stream=stream)
                torch.cuda.synchronize()
                e0.record()
                for _ in range(cfg["launches"]):
                    aai.run_device(plan, si, di, arith=aai.ARITH_F32, stream=stream)
                e1.record()
                torch.cuda.synchronize()
                times[name].append(e0.elapsed_time(e1) / cfg["launches"])
        med = {k: statistics.median(v) for k, v in times.items()}
        res[key] = {"canvas": [plan.dst_w, plan.dst_h], "launches": cfg["launches"], "ms": times,
                    "median_ms": med, "speedup": med["old"] / med["new"]}
        print(key, json.dumps(res[key]), flush=True)
        del src, dst

    # whole config-4 canvas: FP32 kernel of each build against the FP64 kernel
    cfg = CONFIGS["cfg4"]
    plan = aai.make_plan(cfg["w"], cfg["h"], 1.0, cfg["ratio"], cfg["iso"], cfg["angle"])
    src = torch.from_numpy(synthetic_image(cfg["w"], cfg["h"], np.float32, 20205)).cuda()

    def canvas(dt, arith):
        dst = torch.empty(plan.dst_h, plan.dst_w, dtype=dt, device="cuda")
        aai.run_device(plan, aai.tensor_image(src), aai.tensor_image(dst), arith=arith, stream=stream)
        torch.cuda.synchronize()
        return dst

    use("new")
    o64 = canvas(torch.float64, aai.ARITH_F64)
    nz = o64 != 0
    dev = {}
    for name in ("old", "new"):
        use(name)
        o32 = canvas(torch.float32, aai.ARITH_F32).double()
        rel = ((o32 - o64).abs() / o64.abs())[nz]
        dev[name] = {"max_rel_dev_vs_f64": rel.max().item(), "pixels_over_2e-6": int((rel > 2e-6).sum().item())}
        if name == "old":
            old32 = o32
    dev["max_abs_new_minus_old"] = (o32 - old32).abs().max().item()
    res["cfg4_canvas_vs_f64"] = dev
    print("cfg4 canvas vs FP64", json.dumps(dev), flush=True)
    with open(os.path.join(args.outdir, "bench_window.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
