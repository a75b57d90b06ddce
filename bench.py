#!/usr/bin/env python
"""Benchmark of the area-average interpolation hot path (BASELINE.json metric: output Mpixels/s, device-timed).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config 4] [--impl ours|reference] [--no-extra]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path over the whole workload (default: BASELINE config 4, the 16384x16384
float32 slice, 0.37x, 17.3 deg -> 7591x7591 canvas).  With N > 1 (torchrun, one process per GPU) the canvas is
split into row bands balanced by kernel cost; every rank holds its source halo + its band; there is no
data-path collective (bands are independent) -- only the barrier and the max-over-ranks of the timing.

value     = canvas Mpixels/s with the source resident in HBM, CUDA events around exactly K steps (max over ranks)
e2e       = the same metric through the host-buffer C-ABI call: pinned host source -> device, kernel, device ->
            pinned host canvas, all inside the timed region (N = 1: aai_run_host_band, chunk-pipelined; N > 1: the
            peer group of include/aai.h -- every source row crosses PCIe once, halos move over NVLink)
roofline  = the dominant kernel against its bound (FP32 pipe for the rotated clip path, HBM for the separable path);
            peak = the nominal FP32 rate (SMs x 128 lanes x 2 x max clock) resp. the measured HBM copy rate
cpu_baseline = the reference's own CPU implementation (compiled upstream Source.cpp, 1 thread as shipped) on a
            bounded replica of the workload, timed on this box (rank 0, N = 1)
verified  = after the timed regions: the canvas the end-to-end path produced is (a) bitwise equal to the band computed
            from a source generated directly in HBM (independent of the upload / NVLink exchange) and (b) within
            tolerance of the CPU oracle on the first, middle and last row of every rank's band
configs   = the other BASELINE shapes (cfg 1, 2, 3, 5), the FP64 kernel and fast mode on the headline shape, measured
            the same way in the same run outside the headline's timed regions (all ranks take part under torchrun)

--impl reference times the upstream CPU implementation on all host cores (one process per core, one replica image
each per step).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "output Mpixels/s (device-timed)"
UNIT = "Mpix/s"
DUMP_BYTES = 32 << 20  # --dump-outputs: canvas sample size limit

# BASELINE.json configs (SURVEY.md §8d fixes isocentres and generators); index = config number
CONFIGS = {
    1: dict(label="cfg1: 512x512 u8 grayscale, 0.5x, 0 deg", w=512, h=512, dtype="uint8", ch=1, ratio=0.5,
            angle=0.0, iso=(256.0, 256.0), batch=1, replica=512, baseline_replica=512),
    2: dict(label="cfg2: 2048x2048 u8 grayscale, 0.37x, 30 deg", w=2048, h=2048, dtype="uint8", ch=1, ratio=0.37,
            angle=30.0, iso=(1024.0, 1024.0), batch=1, replica=512, baseline_replica=2048),
    3: dict(label="cfg3: 8192x8192 RGB u8, 1.7x, 45 deg", w=8192, h=8192, dtype="uint8", ch=3, ratio=1.7, angle=45.0,
            iso=(4095.5, 4095.5), batch=1, replica=128, baseline_replica=384),
    4: dict(label="cfg4: 16384x16384 float32, 0.37x, 17.3 deg", w=16384, h=16384, dtype="float32", ch=1, ratio=0.37,
            angle=17.3, iso=(8192.0, 8192.0), batch=1, replica=512, baseline_replica=2048),
    5: dict(label="cfg5: 256 x 4096x4096 float32, 0.5x, 0 deg", w=4096, h=4096, dtype="float32", ch=1, ratio=0.5,
            angle=0.0, iso=(2048.0, 2048.0), batch=256, replica=512, baseline_replica=1024),
}


def replica_of(cfg, side):
    """Same ratio / angle / isocentre rule on a smaller source (per-pixel CPU cost is size independent, SURVEY §6)."""
    iso = side / 2.0 - (cfg["w"] / 2.0 - cfg["iso"][0])  # same offset from the image centre
    return dict(w=side, h=side, ratio=cfg["ratio"], angle=cfg["angle"], iso=(iso, iso))


def flops_per_covered_pixel(side, c, s, channels):
    """SURVEY.md §8d contract figure: F = 48 + 128 N_bnd + 2 N_int (+2 per extra channel and touched cell)."""
    n_int = max(0.0, side - c - s) ** 2
    n_all = side * side + 2 * side * (c + s) + 1
    n_bnd = n_all - n_int
    return 48 + 128 * n_bnd + 2 * n_int + 2 * (channels - 1) * n_all


# ---- reference arm -----------------------------------------------------------------------------------------------

def _ref_worker(args):
    side, ratio, angle, iso, seed, kind = args
    sys.path.insert(0, ROOT)
    from area_average_interpolation_b200.synthetic import synthetic_image
    from oracle import port, ref

    src = synthetic_image(side, side, np.float64, seed)
    t0 = time.perf_counter()
    if kind == "reference":
        ok, msg, dst, _, _ = ref.run(src, 1.0, ratio, iso, angle, mode=1)
        assert ok, msg
    else:
        st, dst, _ = port.run(src, 1.0, ratio, iso, angle, mode=1, threads=1)
        assert st == 0
    return dst.size, time.perf_counter() - t0


def cpu_kind():
    from oracle import port, ref

    if ref.available:
        return "reference"
    port.lib()
    return "port"


def _verify_rows(src_rows, src_y0, cfg, mode, rows, channel):
    """Checker leg (outside every timed region): the CPU oracle on canvas rows [rows[0], rows[1]) of the workload.
    `src_rows` holds source rows [src_y0, src_y0 + len) -- everything those canvas rows can touch; the rest of the image
    is never read (untouched virtual memory)."""
    from oracle import port

    full = np.empty((cfg["h"], cfg["w"]) + src_rows.shape[2:], dtype=src_rows.dtype)
    full[src_y0:src_y0 + src_rows.shape[0]] = src_rows
    st, want, _ = port.run(full, 1.0, cfg["ratio"], cfg["iso"], cfg["angle"], mode=mode, rows=rows, channel=channel)
    assert st == 0
    return want


def reference_arm(args, cfg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import multiprocessing as mp

    kind = cpu_kind()
    cores = os.cpu_count() or 1
    rep = replica_of(cfg, cfg["replica"])
    ctx = mp.get_context("spawn")
    with ctx.Pool(cores) as pool:
        tasks = [(rep["w"], rep["ratio"], rep["angle"], rep["iso"], 20201 + k, kind) for k in range(cores)]
        for _ in range(args.warmup):
            pool.map(_ref_worker, tasks)
        t0 = time.perf_counter()
        pixels = 0
        for _ in range(args.steps):
            pixels += sum(n for n, _ in pool.map(_ref_worker, tasks))
        dt = time.perf_counter() - t0
    value = pixels / dt / 1e6
    sample = (f"{cores} processes x one {rep['w']}x{rep['h']} float64 replica of {cfg['label']} per step "
              f"(same ratio/angle; per-pixel CPU cost is size independent)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": cfg["label"], "sample": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ---- clocks ------------------------------------------------------------------------------------------------------------

class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device_uuid):
        self.proc = None
        self.path = None
        self.uuid = device_uuid

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            cmd = ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"]
            if self.uuid:
                cmd += ["-i", self.uuid]
            self.proc = subprocess.Popen(cmd, stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.proc:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        try:
            rows = [r.strip().split(",") for r in open(self.path) if r.strip()]
            os.unlink(self.path)
        except Exception:
            return out
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            if len(r) < 7:
                continue
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except ValueError:
                continue
            for n, v in zip(names, r[3:7]):
                if v.strip().lower().startswith("active"):
                    reasons.add(n)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons),
                       samples=len(sm))
        return out


# ---- our arm -----------------------------------------------------------------------------------------------------------

def bind_to_gpu_numa_node(torch, local):
    """One process per GPU: run on the CPUs of the GPU's own NUMA node, so that the pinned host buffers (first touch)
    and the copy threads sit next to its PCIe root port.  With 8 ranks uploading at once, buffers on the far socket cap
    the upload at ~23 GB/s per rank (measured; 35-50 GB/s from the near socket).  Best effort: any failure leaves the
    affinity as it was."""
    try:
        bus = torch.cuda.get_device_properties(local).pci_bus_id
        dom = getattr(torch.cuda.get_device_properties(local), "pci_domain_id", 0)
        devid = getattr(torch.cuda.get_device_properties(local), "pci_device_id", 0)
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{devid:02x}.0"
        node = int(open(os.path.join(path, "numa_node")).read().strip())
        cpulist = open(os.path.join(path, "local_cpulist")).read().strip()
        cpus = set()
        for part in cpulist.split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        cpus &= os.sched_getaffinity(0)
        if node >= 0 and cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception as exc:  # no sysfs entry, restricted container, ...
        print(f"[bench] NUMA binding skipped: {exc}", file=sys.stderr)
    return None


class Bench:
    """State shared by the measurements of one process (one rank)."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist

        import area_average_interpolation_b200 as aai

        self.torch, self.dist, self.aai, self.args = torch, dist, aai, args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != args.gpus and self.world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N > 1 must be launched with torch.distributed.run (one process per GPU)")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.numa = bind_to_gpu_numa_node(torch, self.local) if self.world > 1 else None
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        # a real (non-default) stream for everything: the C ABI treats stream 0 as "use an internal stream and block"
        self.tstream = torch.cuda.Stream(device=self.dev)
        torch.cuda.set_stream(self.tstream)
        self.stream = self.tstream.cuda_stream
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        self.hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        self.hbm_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
        self.sm_max = float(peaks.get("sm_max_mhz", 1965.0))
        self.n_sm = torch.cuda.get_device_properties(self.local).multi_processor_count
        self.fp32_nominal = self.n_sm * 128 * 2 * self.sm_max * 1e6 / 1e12
        self.fp64_nominal = self.n_sm * 64 * 2 * self.sm_max * 1e6 / 1e12
        self.fp32_probe = None
        try:
            self.uuid = "GPU-" + str(torch.cuda.get_device_properties(self.local).uuid)
        except Exception:
            self.uuid = None
        try:
            self.latest = json.load(open(os.path.join(ROOT, "profiles", "latest.json")))
        except Exception:
            self.latest = {}

    # -- collectives used for TIMING / bookkeeping only (no data-path collective) ------------------------------------
    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def _reduce(self, x, op):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=op)
        return t.item()

    def max_over_ranks(self, x):
        return self._reduce(x, self.dist.ReduceOp.MAX)

    def min_over_ranks(self, x):
        return self._reduce(x, self.dist.ReduceOp.MIN)

    def sum_over_ranks(self, x):
        return self._reduce(x, self.dist.ReduceOp.SUM)

    def gather(self, obj):
        if self.world == 1:
            return [obj]
        out = [None] * self.world
        self.dist.all_gather_object(out, obj)
        return out

    def probe_fp32(self):
        if self.fp32_probe is None:
            try:
                self.fp32_probe = self.aai.measure_fp32_tflops(self.local)
            except Exception as exc:
                print(f"[bench] FP32 probe failed: {exc}", file=sys.stderr)
                self.fp32_probe = 0.0
        return self.fp32_probe

    # -- one workload ----------------------------------------------------------------------------------------------------
    def measure(self, cfg_id, arith_name="auto", mode=1, steps=None, with_e2e=True, with_verify=True,
                with_clocks=True, tag=None, dump_dir=None):
        """Device-timed value, end-to-end value, roofline and verification of one BASELINE shape; with `dump_dir`, the
        canvas of the last timed step is written there (dump_canvas)."""
        torch, aai, args = self.torch, self.aai, self.args
        from area_average_interpolation_b200.sharding import band_for_rank, batch_slice
        from area_average_interpolation_b200.synthetic import synthetic_image_torch

        cfg = CONFIGS[cfg_id]
        steps = steps or args.steps
        warm = max(args.warmup, 3)
        rank, world, local, dev, stream = self.rank, self.world, self.local, self.dev, self.stream
        if arith_name == "auto":
            arith = aai.ARITH_F64 if cfg["dtype"] == "float64" else aai.ARITH_F32
        else:  # f32b / f32r: the opt-in fast-mode kernels (source-side binning, persistent TMA ring), measured beside the default
            arith = {"f32": aai.ARITH_F32, "f32b": aai.ARITH_F32_BINNED, "f32r": aai.ARITH_F32_RING}.get(arith_name,
                                                                                                       aai.ARITH_F64)
        np_dt = np.dtype(cfg["dtype"])
        t_dt = {"uint8": torch.uint8, "float32": torch.float32, "float64": torch.float64}[cfg["dtype"]]
        out_dt = t_dt  # the canvas has the image's own element type (8-bit in -> 8-bit out, round half up)
        W, H, CH = cfg["w"], cfg["h"], cfg["ch"]
        plan = aai.make_plan(W, H, 1.0, cfg["ratio"], cfg["iso"], cfg["angle"])
        assert plan.status == 0, plan.message
        seed = 20201 + cfg_id
        tail = (CH,) if CH > 1 else ()
        esz, osz = np_dt.itemsize, torch.empty((), dtype=out_dt).element_size()
        kw = dict(mode=mode, arith=arith, device=local, stream=stream)
        peer = None
        info = {}

        if cfg["batch"] == 1:
            # bands balanced for THIS kernel (the peer group of the end-to-end leg partitions with the library default)
            band = band_for_rank(plan, rank, world,
                                 None if (world > 1 and with_e2e) else aai.band_empty_weight(plan, mode, arith))
            halo_rows = band.src_y1 - band.src_y0
            # this rank's source halo, generated directly in HBM (bit-identical to the host generator)
            dev_src = synthetic_image_torch(W, H, np_dt, seed, channels=CH, y0=band.src_y0, rows=max(halo_rows, 1),
                                            device=dev)
            si = aai.tensor_image(dev_src[:halo_rows] if halo_rows else dev_src, y0=band.src_y0, height=H)
            dev_dst = torch.empty((band.rows, plan.dst_w) + tail, dtype=out_dt, device=dev)
            di = aai.tensor_image(dev_dst, y0=band.row0, height=plan.dst_h)
            my_pixels = band.rows * plan.dst_w
            resident = dev_src.numel() * esz

            def step():
                aai.run_device(plan, si, di, band.row0, band.row1, **kw)

        else:
            band = None
            lo, hi = batch_slice(cfg["batch"], rank, world)
            n_img = hi - lo
            distinct = min(n_img, 4)  # a few distinct synthetic slices; the device batch is resident
            base = [synthetic_image_torch(W, H, np_dt, seed + 1000 * (lo + k), device=dev) for k in range(distinct)]
            dev_src = torch.empty((n_img, H, W), dtype=t_dt, device=dev)
            for k in range(n_img):
                dev_src[k].copy_(base[k % distinct])
            dev_dst = torch.empty((n_img, plan.dst_h, plan.dst_w), dtype=out_dt, device=dev)
            sis = [aai.tensor_image(dev_src[k]) for k in range(n_img)]
            dis = [aai.tensor_image(dev_dst[k]) for k in range(n_img)]
            my_pixels = n_img * plan.dst_w * plan.dst_h
            resident = dev_src.numel() * esz

            def step():
                aai.run_device_batch(plan, sis, dis, **kw)

        total_pixels = self.sum_over_ranks(float(my_pixels))

        # ---- device-timed region -------------------------------------------------------------------------------------
        for _ in range(warm):
            step()
        torch.cuda.synchronize()
        sampler = ClockSampler(self.uuid) if (rank == 0 and with_clocks) else None
        if sampler:
            sampler.start()
        # untimed pre-load so that the clock sampler sees the loaded state even when K steps are only milliseconds
        t_pre = time.perf_counter()
        while time.perf_counter() - t_pre < (0.6 if with_clocks else 0.05):
            step()
            torch.cuda.synchronize()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        before = aai.launch_count()
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        self.barrier()
        launches = aai.launch_count() - before
        ms_step = self.max_over_ranks(e0.elapsed_time(e1)) / steps
        value = total_pixels / (ms_step * 1e-3) / 1e6
        band_ms = self.gather(e0.elapsed_time(e1) / steps)
        if dump_dir:
            self.dump_canvas(dump_dir, cfg, plan, dev_dst, band.row0 if band is not None else lo * plan.dst_h)

        # ---- end-to-end region (host buffers through the C ABI) --------------------------------------------------
        e2e = None
        host_dst = None
        if with_e2e:
            if cfg["batch"] == 1:
                host_dst = torch.empty((band.rows, plan.dst_w) + tail, dtype=out_dt, pin_memory=True)
                hdi = aai.tensor_image(host_dst, y0=band.row0, height=plan.dst_h)
                d2h = band.rows * plan.dst_w * CH * osz
                if world > 1 and not args.no_peer:
                    if args.peer_chunks:
                        aai.peer_upload_chunks(args.peer_chunks)
                    try:
                        peer = aai.PeerGroup(plan, aai._NP_TO_AAI[np_dt], CH, rank, world, local, self.gather)
                    except Exception as exc:  # IPC unavailable: every rank uploads its own halo from the host
                        print(f"[bench] rank {rank}: peer group unavailable ({exc}); uploading halos from host",
                              file=sys.stderr)
                        peer = None
                    if self.min_over_ranks(1.0 if peer is not None else 0.0) == 0.0 and peer is not None:
                        peer.close()
                        peer = None
                if peer is not None:
                    o0, o1 = peer.owned_rows()
                    host_src = torch.empty((max(o1 - o0, 1), W) + tail, dtype=t_dt, pin_memory=True)
                    if o1 > o0:
                        host_src[:o1 - o0].copy_(synthetic_image_torch(W, H, np_dt, seed, channels=CH, y0=o0,
                                                                       rows=o1 - o0, device=dev))
                    hsi = aai.tensor_image(host_src[:o1 - o0], y0=o0, height=H)
                    h2d = (o1 - o0) * W * CH * esz

                    def e2e_step():
                        peer.run(hsi, hdi, mode=mode, arith=arith, stream=stream, synchronize=False)

                    info["e2e_source"] = ("peer group (include/aai.h): every source row uploaded once by its owner rank in "
                                          "chunks, halos pulled over NVLink as the chunks land (CUDA IPC peer copies, host-"
                                          "driven shared-memory counters), kernel + download chunk-pipelined; no NCCL, no barrier")
                else:
                    host_src = torch.empty((max(halo_rows, 1), W) + tail, dtype=t_dt, pin_memory=True)
                    host_src.copy_(dev_src)
                    hsi = aai.tensor_image(host_src[:halo_rows] if halo_rows else host_src, y0=band.src_y0, height=H)
                    h2d = halo_rows * W * CH * esz

                    def e2e_step():
                        aai.run_host_band(plan, hsi, hdi, band.row0, band.row1, mode=mode, arith=arith, device=local,
                                          stream=stream, synchronize=False)

                    info["e2e_source"] = "each rank uploads its band's source halo from pinned host memory (chunk-pipelined)"
            else:
                host_src = torch.empty((distinct, H, W), dtype=t_dt, pin_memory=True)
                for k in range(distinct):
                    host_src[k].copy_(base[k])
                host_dst = torch.empty((distinct, plan.dst_h, plan.dst_w), dtype=out_dt, pin_memory=True)
                hs_list = [aai.tensor_image(host_src[k % distinct]) for k in range(n_img)]
                hd_list = [aai.tensor_image(host_dst[k % distinct]) for k in range(n_img)]
                h2d = n_img * H * W * esz
                d2h = n_img * plan.dst_w * plan.dst_h * osz

                def e2e_step():
                    aai.run_host_batch(plan, hs_list, hd_list, mode=mode, arith=arith, device=local, stream=stream,
                                       synchronize=False)

                info["e2e_source"] = ("aai_run_host_batch: slices uploaded, resampled (batched launches) and downloaded in "
                                      "a 3-stream pipeline; the host keeps 4 distinct slices")
            for _ in range(2):
                e2e_step()
            self.barrier()
            e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e2.record()
            for _ in range(steps):
                e2e_step()
            e3.record()
            self.barrier()
            e2e_ms = self.max_over_ranks(e2.elapsed_time(e3)) / steps
            e2e = {"value": total_pixels / (e2e_ms * 1e-3) / 1e6, "unit": UNIT,
                   "h2d_bytes_per_step": self.sum_over_ranks(float(h2d)),
                   "d2h_bytes_per_step": self.sum_over_ranks(float(d2h)), "ms_per_step": e2e_ms}
            if peer is not None:  # device-side completion times of the last step's phases, per rank (from its start)
                ph = self.gather(peer.last_timing())
                e2e["phases_ms_per_rank"] = {k: [round(p[k], 3) for p in ph] for k in ph[0]}
        clocks = sampler.stop() if sampler else {}

        # ---- verification (outside the timed regions) ----------------------------------------------------------------
        verify = None
        if with_verify:
            verify = self._verify(cfg, cfg_id, plan, mode, arith, band, dev_dst, host_dst, step, seed,
                                  lo if band is None else 0)

        # ---- roofline of the dominant kernel ------------------------------------------------------------------------
        if cfg["batch"] == 1:
            # covered = canvas pixels whose footprint box meets the image (what the kernels evaluate; plan geometry)
            covered = self.sum_over_ranks(float(aai.covered_pixels(plan, band.row0, band.row1)))
        else:
            covered = total_pixels
        alg_bytes = (W * H * CH * esz + plan.dst_w * plan.dst_h * CH * osz) * cfg["batch"]
        hbm = {"achieved": alg_bytes / world / (ms_step * 1e-3) / 1e9, "peak": self.hbm_peak, "unit": "GB/s",
               "peak_source": self.hbm_src}
        if plan.axis_aligned or mode == 2:
            roofline = {"bound": "hbm", "achieved": hbm["achieved"], "peak": self.hbm_peak, "unit": "GB/s",
                        "frac": hbm["achieved"] / self.hbm_peak, "traffic": None, "peak_source": self.hbm_src,
                        "algorithmic": "each source byte read once + each canvas byte written once (SURVEY 8d)"}
        else:
            F = flops_per_covered_pixel(plan.side, plan.cos_t, plan.sin_t, CH)
            f32 = arith != aai.ARITH_F64
            peak = self.fp32_nominal if f32 else self.fp64_nominal
            achieved = F * covered / world / (ms_step * 1e-3) / 1e12
            roofline = {"bound": "fp32" if f32 else "fp64", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                        "frac": achieved / peak, "traffic": None,
                        "peak_source": f"nominal {self.n_sm} SMs x {128 if f32 else 64} lanes x 2 x {self.sm_max:.0f} MHz "
                                       "(MEASURED_PEAKS.json holds no FP32/FP64 figure)",
                        "algorithmic": f"{F:.0f} flop per covered canvas pixel x {covered / world:.0f} covered pixels per "
                                       "launch (SURVEY 8d contract figure)",
                        "hbm": hbm}
            if f32:
                roofline["peak_measured_ffma_probe"] = self.probe_fp32()
        prof = self.latest.get(tag or f"cfg{cfg_id}", {})
        traffic = prof.get("dram_bytes_per_launch")
        if traffic is not None:
            if "per" in prof:  # profiled per slice of a batched launch: scale to this rank's launch
                traffic = int(traffic * cfg["batch"] / world)
            elif world > 1:
                traffic = None  # captured on the whole canvas; a band's launch was not profiled
        roofline["traffic"] = traffic

        res = {
            "workload": cfg["label"], "mode": {1: "area-average", 2: "fast"}[mode],
            "dtype": "f32" if arith != aai.ARITH_F64 else "f64", "canvas": f"{plan.dst_w}x{plan.dst_h}",
            "canvas_dtype": str(out_dt).replace("torch.", ""), "value": value, "unit": UNIT, "ms_per_step": ms_step,
            "steps": steps, "gpu_launches": int(launches), "roofline": roofline, "covered_pixels": covered,
            "timing": (f"inputs larger than L2 ({resident / 1e6:.0f} MB resident source per rank)" if resident > 130e6
                       else "L2-resident input (source smaller than L2); latency bound"),
        }
        if world > 1:
            res["band_ms"] = [round(v, 4) for v in band_ms]
        if e2e is not None:
            res["e2e"] = e2e
        if verify is not None:
            res["verified"] = verify["ok"]
            res["verify"] = verify
        if with_clocks:
            res["clocks"] = {k: clocks.get(k) for k in ("sm_mhz", "sm_max_mhz", "reasons", "samples")}
        res["_plan"] = plan
        res["_info"] = info
        if peer is not None:
            self.barrier()
            peer.close()
        del dev_src, dev_dst
        torch.cuda.empty_cache()
        return res

    def dump_canvas(self, out_dir, cfg, plan, dev_dst, first_row):
        """Writes `out_dir`/canvas.npy: the canvas rows this workload's timed path produced, as float32 (float64 for a
        float64 canvas), rows ordered over the whole workload (row r of slice k is row k * dst_h + r).  A canvas larger
        than DUMP_BYTES is sampled: a fixed, seeded choice of rows in ascending order, the same for any number of GPUs.
        `dev_dst` holds this rank's rows, starting at workload row `first_row`."""
        torch = self.torch
        local = dev_dst.flatten(0, 1) if cfg["batch"] > 1 else dev_dst
        out_np = np.float64 if dev_dst.dtype == torch.float64 else np.float32
        total = cfg["batch"] * plan.dst_h
        n = min(total, DUMP_BYTES // (plan.dst_w * cfg["ch"] * np.dtype(out_np).itemsize))
        rows = np.arange(total) if n == total else np.sort(np.random.default_rng(0).choice(total, n, replace=False))
        mine = rows[(rows >= first_row) & (rows < first_row + local.shape[0])] - first_row
        part = local[torch.as_tensor(mine, device=self.dev)].cpu().numpy().astype(out_np)
        parts = self.gather(part)  # ranks hold consecutive row ranges in rank order
        if self.rank == 0:
            os.makedirs(out_dir, exist_ok=True)
            np.save(os.path.join(out_dir, "canvas.npy"), np.concatenate(parts, axis=0))

    def _verify(self, cfg, cfg_id, plan, mode, arith, band, dev_dst, host_dst, step, seed, first_image):
        """(a) the end-to-end canvas equals, bit for bit, the canvas computed from the HBM-generated source (the upload /
        NVLink exchange delivered exactly the right bytes to the right rows); (b) first, middle and last row of this rank's
        band (first / last slice of a batch) against the CPU oracle."""
        torch, aai = self.torch, self.aai
        from area_average_interpolation_b200.synthetic import synthetic_image_torch

        np_dt = np.dtype(cfg["dtype"])
        f32 = arith != aai.ARITH_F64
        ok, max_err, checked, same = True, 0.0, 0, None
        try:
            step()
            torch.cuda.synchronize()
            got = dev_dst.cpu()
            if host_dst is not None:
                if band is not None:
                    same = bool(torch.equal(got, host_dst))
                else:  # the host keeps `distinct` canvases; slice k landed in host_dst[k % distinct]
                    n = host_dst.shape[0]
                    same = bool(all(torch.equal(got[k], host_dst[k]) for k in range(n)))
                ok = ok and same
            got = got.numpy()
            u8 = np_dt == np.uint8
            if band is not None:
                rows = sorted({band.row0, (band.row0 + band.row1) // 2, band.row1 - 1}) if band.rows > 0 else []
                for r in rows:
                    _, _, sy0, sy1 = aai.band_source_window(plan, r, r + 1)
                    if sy1 <= sy0:
                        want = np.zeros((1, plan.dst_w))
                        chans = [0]
                    else:
                        src_rows = synthetic_image_torch(cfg["w"], cfg["h"], np_dt, seed, channels=cfg["ch"], y0=sy0,
                                                         rows=sy1 - sy0, device=self.dev).cpu().numpy()
                        chans = [0] if cfg["ch"] == 1 else [0, cfg["ch"] - 1]
                    for c in chans:
                        if sy1 > sy0:
                            want = _verify_rows(src_rows, sy0, cfg, mode, (r, r + 1), c)
                        g = got[r - band.row0][None, ...]
                        g = (g[..., c] if cfg["ch"] > 1 else g).astype(np.float64)
                        err = self._err(g, want, u8, f32)
                        max_err = max(max_err, err)
                        checked += 1
            else:
                for k in sorted({0, got.shape[0] - 1}):
                    src_k = synthetic_image_torch(cfg["w"], cfg["h"], np_dt, seed + 1000 * (first_image + (k % 4)),
                                                  device=self.dev).cpu().numpy()
                    for r in (0, plan.dst_h // 2):
                        want = _verify_rows(src_k, 0, cfg, mode, (r, r + 1), 0)
                        err = self._err(got[k][r][None, :].astype(np.float64), want, u8, f32)
                        max_err = max(max_err, err)
                        checked += 1
            ok = ok and max_err <= 1.0
        except Exception as exc:
            print(f"[bench] rank {self.rank}: verification failed to run: {exc!r}", file=sys.stderr)
            ok = False
        ok_all = self.min_over_ranks(1.0 if ok else 0.0) == 1.0
        return {"ok": bool(ok_all), "e2e_bitwise_equals_device_path": same,
                "oracle_rows_checked_per_rank": checked, "max_error_over_tolerance": self.max_over_ranks(max_err),
                "tolerance": ("0.5 + 0.5/255 absolute (8-bit canvas, round half up)" if np_dt == np.uint8 else
                              ("1e-5 relative to max(|value|, range/256) (FP32 kernel)" if f32 else "1e-9 relative (FP64 arithmetic; float32 canvas "
                                                                        "rounds to 6e-8)"))}

    @staticmethod
    def _err(got, want, u8, f32):
        """max error / tolerance"""
        if u8:
            return float(np.abs(got - want).max() / (0.5 + 0.5 / 255.0))
        if f32:  # relative to max(|want|, range / 256) of the 12-bit synthetic data (tests/common.py: f32_err)
            return float((np.abs(got - want) / np.maximum(np.abs(want), 4096.0 / 256.0)).max() / 1e-5)
        rel = np.abs(got - want) / np.where(want == 0, 1.0, np.abs(want))
        return float(rel.max() / 1e-7)  # (a float32 canvas rounds the FP64 result to 6e-8)


def our_arm(args, cfg_id):
    b = Bench(args)
    cfg = CONFIGS[cfg_id]
    head = b.measure(cfg_id, arith_name=args.arith, mode=args.mode, with_e2e=True, with_verify=not args.no_verify,
                     dump_dir=args.dump_outputs)
    plan, info = head.pop("_plan"), head.pop("_info")
    line = {
        "metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": b.world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": head["ms_per_step"], "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": head["dtype"], "data": "synthetic",
        "config": {"workload": cfg["label"], "canvas": head["canvas"], "canvas_dtype": head["canvas_dtype"],
                   "scale": plan.scale, "footprint_side": plan.side, "mode": head["mode"],
                   "sharding": ("row bands balanced by kernel cost" if cfg["batch"] == 1 else "whole images per rank"),
                   "timing": head["timing"], "covered_pixels": head["covered_pixels"], "numa_node_rank0": b.numa,
                   "e2e_source": info.get("e2e_source")},
        "clocks": head["clocks"], "e2e": head["e2e"], "gpu_launches": head["gpu_launches"],
        "roofline": head["roofline"],
    }
    if "band_ms" in head:
        line["band_ms"] = head["band_ms"]
    if "verified" in head:
        line["verified"] = head["verified"]
        line["verify"] = head["verify"]
    if b.rank == 0 and b.world == 1 and not args.no_cpu_baseline:
        kind = cpu_kind()
        rep = replica_of(cfg, cfg["baseline_replica"])
        n, sec = _ref_worker((rep["w"], rep["ratio"], rep["angle"], rep["iso"], 20201 + cfg_id, kind))
        line["cpu_baseline"] = {
            "value": n / sec / 1e6, "unit": UNIT, "cores": 1, "kind": kind,
            "sample": f"one {rep['w']}x{rep['h']} float64 replica of the workload (same ratio/angle), {sec:.1f} s, "
                      "single thread as the reference ships"}
    # ---- the other named shapes + the FP64 kernel + fast mode, same run, outside the headline's timed regions --------
    if not args.no_extra:
        extra = {}
        k = max(3, min(args.steps, 10))
        todo = [(f"cfg{c}", c, "auto", 1) for c in sorted(CONFIGS) if c != cfg_id]
        todo += [(f"cfg{cfg_id}_f64", cfg_id, "f64", 1), (f"cfg{cfg_id}_fast", cfg_id, "auto", 2)]
        hc = CONFIGS[cfg_id]
        if hc["dtype"] == "float32" and hc["ch"] == 1 and hc["batch"] == 1 and hc["angle"] % 90 != 0:  # the measured alternatives of fast mode
            todo += [(f"cfg{cfg_id}_fast_binned", cfg_id, "f32b", 2), (f"cfg{cfg_id}_fast_ring", cfg_id, "f32r", 2)]
        for name, c, ar, mode in todo:
            try:
                r = b.measure(c, arith_name=ar, mode=mode, steps=k, with_e2e=(b.world == 1 and ar in ("auto", "f64")),
                              with_verify=not args.no_verify, with_clocks=True, tag=name)
                r.pop("_plan")
                r.pop("_info")
                extra[name] = r
            except Exception as exc:
                extra[name] = {"error": repr(exc)}
                print(f"[bench] {name} failed: {exc!r}", file=sys.stderr)
        line["configs"] = extra
    if b.rank == 0:
        print(json.dumps(line), flush=True)
    if b.world > 1:
        b.dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of the headline workload (the `configs` records take min(K, 10), at least 3)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", type=int, default=4, choices=sorted(CONFIGS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--arith", default="auto", choices=["auto", "f64", "f32"],
                    help="auto: FP32 kernel for float32/8-bit images, FP64 kernel for float64 images")
    ap.add_argument("--mode", type=int, default=1, choices=[1, 2], help="1 area average (headline), 2 fast mode")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="headline workload only (skip the `configs` record)")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--peer-chunks", type=int, default=0, help="N>1: upload chunks per owner rank of the peer group (1..8)")
    ap.add_argument("--no-peer", action="store_true",
                    help="N>1: every rank uploads its whole halo from the host instead of NVLink peer copies")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the headline canvas of the last timed step to DIR/canvas.npy (float32; a fixed, seeded "
                         f"sample of rows where the canvas exceeds {DUMP_BYTES >> 20} MiB), to compare two builds; "
                         "--impl ours only: the reference arm times CPU code (the upstream implementation, or the "
                         "oracle restatement where that is absent), not the CUDA path two builds differ in")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the canvas of the CUDA path (--impl ours); the reference arm runs CPU code")
    cfg = CONFIGS[args.config]
    # stdout carries exactly ONE JSON line: libraries that write to file descriptor 1 (NCCL prints its version banner
    # there under torchrun) are sent to stderr; the JSON line is written to the saved descriptor.
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(json_fd, "w")
    if args.impl == "reference":
        return reference_arm(args, cfg)
    return our_arm(args, args.config)


if __name__ == "__main__":
    sys.exit(main())
