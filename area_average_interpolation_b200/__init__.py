"""B200-native area-average interpolation (the hot path of Ishikawa-lab/Area_average_interpolation).

Python mirror of the reference operator interface (``AreaAverageInterpolation::areaAverageInterpolation``,
``Source.cpp:55-583``) on top of the C ABI in ``include/aai.h`` (``libaai_b200.so``, built in-tree by
``__graft_entry__.build()``).  Everything numeric happens in the CUDA library; this module only marshals
buffers.  There is no CPU fallback: without the compiled library or without a GPU the calls raise.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import Optional, Sequence, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libaai_b200.so")  # (developer A/B tools assign another build here before lib() is called)

AAI_OK = 0
ERR_RESOLUTION_XY, ERR_RESOLUTION_NONPOS, ERR_NO_ROWS, ERR_NO_COLUMNS = 1, 2, 3, 4
ERR_ANGLE, ERR_ARGUMENT, ERR_CUDA, ERR_NO_DEVICE = 5, 6, 7, 8
F64, F32, U8, U16 = 0, 1, 2, 3
MODE_AREA_AVERAGE, MODE_FAST, MODE_AREA_AVERAGE_EXACT = 1, 2, 3
ARITH_F64, ARITH_F32, ARITH_F32_STAGED, ARITH_F32_BINNED, ARITH_F32_RING = 0, 1, 2, 3, 4

_NP_TO_AAI = {np.dtype(np.float64): F64, np.dtype(np.float32): F32, np.dtype(np.uint8): U8, np.dtype(np.uint16): U16}
_AAI_TO_NP = {v: k for k, v in _NP_TO_AAI.items()}


class AaiError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"aai status {status}: {message}")
        self.status = status
        self.message = message


class Plan(C.Structure):
    """``struct aai_plan`` (include/aai.h): what the reference decides before its main loop."""
    _fields_ = [
        ("status", C.c_int32), ("scale", C.c_uint32), ("quadrant", C.c_int32), ("axis_aligned", C.c_int32),
        ("src_w", C.c_int64), ("src_h", C.c_int64), ("mod_w", C.c_int64), ("mod_h", C.c_int64),
        ("dst_w", C.c_int64), ("dst_h", C.c_int64),
        ("theta_deg", C.c_double), ("sin_t", C.c_double), ("cos_t", C.c_double),
        ("iso_x", C.c_double), ("iso_y", C.c_double), ("ratio", C.c_double), ("side", C.c_double),
        ("dst_iso_x", C.c_double), ("dst_iso_y", C.c_double), ("off_ix", C.c_double), ("off_iy", C.c_double),
        ("off_x", C.c_double), ("off_y", C.c_double), ("reach", C.c_double),
    ]

    @property
    def message(self) -> str:
        return status_string(self.status)

    @property
    def dst_isocenter(self) -> Tuple[float, float]:
        return (self.dst_iso_x, self.dst_iso_y)


class Image(C.Structure):
    """``struct aai_image``: a pitched image (or a band of rows of one) in host or device memory."""
    _fields_ = [
        ("data", C.c_void_p), ("pitch_bytes", C.c_int64), ("width", C.c_int64), ("height", C.c_int64),
        ("y0", C.c_int64), ("rows", C.c_int64), ("dtype", C.c_int32), ("channels", C.c_int32),
    ]


_lib_handle = None


def lib() -> C.CDLL:
    """Loads the CUDA library; fails loudly when it has not been built."""
    global _lib_handle
    if _lib_handle is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        L.aai_plan_create.restype = C.c_int
        L.aai_plan_create.argtypes = [C.c_int64, C.c_int64] + [C.c_double] * 7 + [C.POINTER(Plan)]
        L.aai_status_string.restype = C.c_char_p
        L.aai_status_string.argtypes = [C.c_int]
        L.aai_last_error.restype = C.c_char_p
        L.aai_partition_rows.restype = C.c_int
        L.aai_partition_rows.argtypes = [C.POINTER(Plan), C.c_int, C.POINTER(C.c_int64)]
        L.aai_partition_rows_weighted.restype = C.c_int
        L.aai_partition_rows_weighted.argtypes = [C.POINTER(Plan), C.c_int, C.c_double, C.POINTER(C.c_int64)]
        L.aai_band_empty_weight.restype = C.c_double
        L.aai_band_empty_weight.argtypes = [C.POINTER(Plan), C.c_int, C.c_int]
        L.aai_band_source_window.restype = C.c_int
        L.aai_band_source_window.argtypes = [C.POINTER(Plan), C.c_int64, C.c_int64] + [C.POINTER(C.c_int64)] * 4
        L.aai_covered_pixels.restype = C.c_int64
        L.aai_covered_pixels.argtypes = [C.POINTER(Plan), C.c_int64, C.c_int64]
        L.aai_device_count.restype = C.c_int
        L.aai_image_alloc.restype = C.c_int
        L.aai_image_alloc.argtypes = [C.POINTER(Image), C.c_int] + [C.c_int64] * 4 + [C.c_int32, C.c_int32]
        L.aai_image_free.restype = C.c_int
        L.aai_image_free.argtypes = [C.POINTER(Image), C.c_int]
        L.aai_image_upload.restype = C.c_int
        L.aai_image_upload.argtypes = [C.POINTER(Image), C.POINTER(Image), C.c_int, C.c_void_p]
        L.aai_image_download.restype = C.c_int
        L.aai_image_download.argtypes = [C.POINTER(Image), C.POINTER(Image), C.c_int, C.c_void_p]
        L.aai_image_copy_rows.restype = C.c_int
        L.aai_image_copy_rows.argtypes = [C.POINTER(Image), C.POINTER(Image), C.c_int64, C.c_int64, C.c_int, C.c_void_p]
        L.aai_ipc_export.restype = C.c_int
        L.aai_ipc_export.argtypes = [C.c_void_p, C.c_char_p]
        L.aai_ipc_open.restype = C.c_int
        L.aai_ipc_open.argtypes = [C.c_char_p, C.c_int, C.POINTER(C.c_void_p)]
        L.aai_ipc_close.restype = C.c_int
        L.aai_ipc_close.argtypes = [C.c_void_p, C.c_int]
        L.aai_measure_fp32_tflops.restype = C.c_int
        L.aai_measure_fp32_tflops.argtypes = [C.c_int, C.POINTER(C.c_double)]
        L.aai_expand_device.restype = C.c_int
        L.aai_expand_device.argtypes = [C.POINTER(Plan), C.POINTER(Image), C.POINTER(Image), C.c_int, C.c_void_p]
        L.aai_run_device.restype = C.c_int
        L.aai_run_device.argtypes = [C.POINTER(Plan), C.c_int, C.c_int, C.POINTER(Image), C.POINTER(Image),
                                     C.c_int64, C.c_int64, C.c_int, C.c_void_p]
        L.aai_run_device_batch.restype = C.c_int
        L.aai_run_device_batch.argtypes = [C.POINTER(Plan), C.c_int, C.c_int, C.POINTER(Image), C.POINTER(Image),
                                           C.c_int, C.c_int, C.c_void_p]
        L.aai_run_device_adjoint.restype = C.c_int
        L.aai_run_device_adjoint.argtypes = [C.POINTER(Plan), C.c_int, C.POINTER(Image), C.POINTER(Image), C.c_int,
                                             C.c_int, C.c_void_p]
        L.aai_run_host.restype = C.c_int
        L.aai_run_host.argtypes = [C.POINTER(Plan), C.c_int, C.c_int, C.POINTER(Image), C.POINTER(Image),
                                   C.POINTER(C.c_int), C.c_int]
        L.aai_run_host_band.restype = C.c_int
        L.aai_run_host_band.argtypes = [C.POINTER(Plan), C.c_int, C.c_int, C.POINTER(Image), C.POINTER(Image),
                                        C.c_int64, C.c_int64, C.c_int, C.c_void_p, C.c_int]
        L.aai_run_host_batch.restype = C.c_int
        L.aai_run_host_batch.argtypes = [C.POINTER(Plan), C.c_int, C.c_int, C.POINTER(Image), C.POINTER(Image),
                                         C.c_int, C.c_int, C.c_void_p, C.c_int]
        L.aai_peer_create.restype = C.c_int
        L.aai_peer_create.argtypes = [C.POINTER(Plan), C.c_int32, C.c_int32, C.c_int, C.c_int, C.c_int,
                                      C.POINTER(C.c_void_p)]
        L.aai_peer_export.restype = C.c_int
        L.aai_peer_export.argtypes = [C.c_void_p, C.c_char_p]
        L.aai_peer_connect.restype = C.c_int
        L.aai_peer_connect.argtypes = [C.c_void_p, C.c_char_p]
        L.aai_peer_owned_rows.restype = C.c_int
        L.aai_peer_owned_rows.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
        L.aai_peer_band.restype = C.c_int
        L.aai_peer_band.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
        L.aai_peer_run.restype = C.c_int
        L.aai_peer_run.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(Image), C.POINTER(Image), C.c_void_p, C.c_int]
        L.aai_peer_device_source.restype = C.c_int
        L.aai_peer_device_source.argtypes = [C.c_void_p, C.POINTER(Image)]
        L.aai_peer_upload_chunks.restype = C.c_int
        L.aai_peer_upload_chunks.argtypes = [C.c_int]
        L.aai_peer_last_timing.restype = C.c_int
        L.aai_peer_last_timing.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
        L.aai_peer_destroy.restype = C.c_int
        L.aai_peer_destroy.argtypes = [C.c_void_p]
        L.aai_launch_count.restype = C.c_int64
        L.aai_last_host_timing.restype = C.c_int
        L.aai_last_host_timing.argtypes = [C.POINTER(C.c_float)] * 3
        _lib_handle = L
    return _lib_handle


def status_string(status: int) -> str:
    return lib().aai_status_string(int(status)).decode()


def last_error() -> str:
    return lib().aai_last_error().decode()


def _check(status: int) -> None:
    if status != AAI_OK:
        msg = status_string(status)
        if status >= ERR_ARGUMENT:
            detail = last_error()
            if detail:
                msg = f"{msg} {detail}"
        raise AaiError(status, msg)


def _pair(v) -> Tuple[float, float]:
    if np.isscalar(v):
        return float(v), float(v)
    return float(v[0]), float(v[1])


def make_plan(src_w: int, src_h: int, src_resolution, dst_resolution, src_isocenter, rotation_angle: float) -> Plan:
    """Source.cpp:112-200 -- never raises for the reference's own validation failures (see ``Plan.status``)."""
    rx, ry = _pair(src_resolution)
    dx, dy = _pair(dst_resolution)
    ix, iy = _pair(src_isocenter)
    p = Plan()
    lib().aai_plan_create(int(src_w), int(src_h), rx, ry, dx, dy, ix, iy, float(rotation_angle), C.byref(p))
    return p


def band_empty_weight(plan: Plan, mode: int = MODE_AREA_AVERAGE, arith: int = ARITH_F32) -> float:
    """``aai_band_empty_weight``: measured cost of an empty canvas pixel relative to a covered one for the kernel that
    (mode, arith) selects on this plan."""
    return float(lib().aai_band_empty_weight(C.byref(plan), int(mode), int(arith)))


def partition_rows(plan: Plan, n_parts: int, empty_weight: Optional[float] = None) -> list:
    """``aai_partition_rows`` (FP32 overlap kernel's weight) or, with ``empty_weight``, ``aai_partition_rows_weighted``."""
    b = (C.c_int64 * (n_parts + 1))()
    if empty_weight is None:
        _check(lib().aai_partition_rows(C.byref(plan), int(n_parts), b))
    else:
        _check(lib().aai_partition_rows_weighted(C.byref(plan), int(n_parts), float(empty_weight), b))
    return list(b)


def band_source_window(plan: Plan, row0: int, row1: int) -> Tuple[int, int, int, int]:
    """(x0, x1, y0, y1): half-open source rectangle (original pixels) that canvas rows [row0,row1) can touch."""
    v = [C.c_int64() for _ in range(4)]
    _check(lib().aai_band_source_window(C.byref(plan), int(row0), int(row1), *[C.byref(a) for a in v]))
    return tuple(a.value for a in v)


def covered_pixels(plan: Plan, row0: int = 0, row1: Optional[int] = None) -> int:
    return int(lib().aai_covered_pixels(C.byref(plan), int(row0), int(plan.dst_h if row1 is None else row1)))


def device_count() -> int:
    return int(lib().aai_device_count())


def launch_count() -> int:
    return int(lib().aai_launch_count())


def last_host_timing() -> dict:
    a, b, c = C.c_float(), C.c_float(), C.c_float()
    _check(lib().aai_last_host_timing(C.byref(a), C.byref(b), C.byref(c)))
    return {"h2d_ms": a.value, "kernel_ms": b.value, "d2h_ms": c.value}


def _host_image(arr: np.ndarray) -> Image:
    if arr.dtype not in _NP_TO_AAI:
        raise TypeError(f"unsupported dtype {arr.dtype}; use float64, float32, uint8 or uint16")
    if arr.ndim == 2:
        h, w = arr.shape
        ch = 1
    elif arr.ndim == 3:
        h, w, ch = arr.shape
    else:
        raise ValueError("image must be [h, w] or [h, w, channels]")
    if arr.strides[-1] != arr.itemsize or (arr.ndim == 3 and arr.strides[1] != ch * arr.itemsize):
        raise ValueError("image rows must be dense (only the row pitch may be padded)")
    return Image(arr.ctypes.data, arr.strides[0], w, h, 0, h, _NP_TO_AAI[arr.dtype], ch)


def tensor_image(t, y0: int = 0, height: Optional[int] = None) -> Image:
    """``aai_image`` view of a CUDA (or pinned host) torch tensor [rows, w] / [rows, w, c] holding rows y0.. of an image."""
    import torch

    dt = {torch.float64: F64, torch.float32: F32, torch.uint8: U8, torch.uint16: U16}[t.dtype]
    if t.dim() == 2:
        rows, w = t.shape
        ch = 1
    else:
        rows, w, ch = t.shape
    if t.stride(-1) != 1 or (t.dim() == 3 and t.stride(1) != ch):
        raise ValueError("tensor rows must be dense")
    return Image(t.data_ptr(), t.stride(0) * t.element_size(), w, int(height if height is not None else rows),
                 int(y0), rows, dt, ch)


def image_alloc(device: int, width: int, height: int, dtype: int, channels: int = 1, y0: int = 0,
                rows: Optional[int] = None) -> Image:
    """``aai_image_alloc``: pitched device image (or a band of rows of one)."""
    img = Image()
    _check(lib().aai_image_alloc(C.byref(img), int(device), int(width), int(height), int(y0),
                                 int(height if rows is None else rows), int(dtype), int(channels)))
    return img


def image_free(img: Image, device: int) -> None:
    _check(lib().aai_image_free(C.byref(img), int(device)))


def image_upload(device_img: Image, host_img: Image, device: int = 0, stream: int = 0) -> None:
    _check(lib().aai_image_upload(C.byref(device_img), C.byref(host_img), int(device), C.c_void_p(stream)))


def image_download(host_img: Image, device_img: Image, device: int = 0, stream: int = 0) -> None:
    _check(lib().aai_image_download(C.byref(host_img), C.byref(device_img), int(device), C.c_void_p(stream)))


def image_copy_rows(dst_img: Image, src_img: Image, y0: int, y1: int, device: int = 0, stream: int = 0) -> None:
    """Device-to-device rows [y0,y1) (a peer device's image goes over NVLink)."""
    _check(lib().aai_image_copy_rows(C.byref(dst_img), C.byref(src_img), int(y0), int(y1), int(device),
                                     C.c_void_p(stream)))


def ipc_export(device_ptr: int) -> bytes:
    buf = C.create_string_buffer(64)
    _check(lib().aai_ipc_export(C.c_void_p(device_ptr), buf))
    return buf.raw


def ipc_open(handle: bytes, device: int) -> int:
    p = C.c_void_p()
    _check(lib().aai_ipc_open(handle, int(device), C.byref(p)))
    return p.value


def ipc_close(device_ptr: int, device: int) -> None:
    _check(lib().aai_ipc_close(C.c_void_p(device_ptr), int(device)))


def measure_fp32_tflops(device: int = 0) -> float:
    """``aai_measure_fp32_tflops``: sustained FP32 FMA rate of the device (roofline denominator of bench.py)."""
    v = C.c_double(0.0)
    _check(lib().aai_measure_fp32_tflops(int(device), C.byref(v)))
    return v.value


def expand_device(plan: Plan, src_img: Image, dst_mod_img: Image, device: int = 0, stream: int = 0) -> None:
    """``aai_expand_device``: the reference's expanded + quadrant-rotated source ``modSrc`` (Source.cpp:157-172)."""
    _check(lib().aai_expand_device(C.byref(plan), C.byref(src_img), C.byref(dst_mod_img), int(device), C.c_void_p(stream)))


def run_device(plan: Plan, src_img: Image, dst_img: Image, row0: int = 0, row1: Optional[int] = None,
               mode: int = MODE_AREA_AVERAGE, arith: int = ARITH_F64, device: int = 0, stream: int = 0) -> None:
    """``aai_run_device``: enqueue the kernels for canvas rows [row0,row1) on ``stream`` of ``device``."""
    _check(lib().aai_run_device(C.byref(plan), int(mode), int(arith), C.byref(src_img), C.byref(dst_img),
                                int(row0), int(plan.dst_h if row1 is None else row1), int(device),
                                C.c_void_p(stream)))


def run_device_batch(plan: Plan, src_imgs: Sequence[Image], dst_imgs: Sequence[Image], mode: int = MODE_AREA_AVERAGE,
                     arith: int = ARITH_F64, device: int = 0, stream: int = 0) -> None:
    """``aai_run_device_batch``: a batch of images sharing one plan (one launch when the images are whole and equally strided)."""
    n = len(src_imgs)
    sa, da = (Image * n)(*src_imgs), (Image * n)(*dst_imgs)
    _check(lib().aai_run_device_batch(C.byref(plan), int(mode), int(arith), sa, da, n, int(device), C.c_void_p(stream)))


def run_device_adjoint(plan: Plan, canvas_imgs: Sequence[Image], src_imgs: Sequence[Image],
                       mode: int = MODE_AREA_AVERAGE, device: int = 0, stream: int = 0) -> None:
    """``aai_run_device_adjoint``: ``src_imgs[k]`` receives the transpose of the resampling operator (FP64 weights)
    applied to ``canvas_imgs[k]``.  Whole float32 / float64 device images, the same type and channel count on both
    sides; one launch per kernel for an equally strided stack."""
    n = len(canvas_imgs)
    if len(src_imgs) != n:
        raise ValueError("run_device_adjoint: as many source images as canvas images")
    ca, sa = (Image * max(n, 1))(*canvas_imgs), (Image * max(n, 1))(*src_imgs)
    _check(lib().aai_run_device_adjoint(C.byref(plan), int(mode), ca, sa, n, int(device), C.c_void_p(stream)))


def run_host(plan: Plan, src: np.ndarray, dst: np.ndarray, mode: int = MODE_AREA_AVERAGE, arith: int = ARITH_F64,
             devices: Optional[Sequence[int]] = None) -> None:
    """``aai_run_host``: the reference call with host buffers (H2D, kernels on per-device streams, D2H)."""
    si, di = _host_image(src), _host_image(dst)
    if devices:
        arr = (C.c_int * len(devices))(*devices)
        n = len(devices)
    else:
        arr, n = None, 0
    _check(lib().aai_run_host(C.byref(plan), int(mode), int(arith), C.byref(si), C.byref(di), arr, n))


def run_host_band(plan: Plan, src_img: Image, dst_img: Image, row0: int, row1: int, mode: int = MODE_AREA_AVERAGE,
                  arith: int = ARITH_F64, device: int = 0, stream: int = 0, synchronize: bool = True) -> None:
    """``aai_run_host_band``: one rank's share of the host-buffer call (halo upload, kernels, band download)."""
    _check(lib().aai_run_host_band(C.byref(plan), int(mode), int(arith), C.byref(src_img), C.byref(dst_img),
                                   int(row0), int(row1), int(device), C.c_void_p(stream), int(bool(synchronize))))


def run_host_batch(plan: Plan, src_imgs: Sequence[Image], dst_imgs: Sequence[Image], mode: int = MODE_AREA_AVERAGE,
                   arith: int = ARITH_F64, device: int = 0, stream: int = 0, synchronize: bool = True) -> None:
    """``aai_run_host_batch``: a batch of whole HOST images sharing one plan, pipelined through the batched kernels."""
    n = len(src_imgs)
    sa, da = (Image * n)(*src_imgs), (Image * n)(*dst_imgs)
    _check(lib().aai_run_host_batch(C.byref(plan), int(mode), int(arith), sa, da, n, int(device), C.c_void_p(stream),
                                    int(bool(synchronize))))


PEER_BLOB_BYTES = 2048


def peer_upload_chunks(n: int = 0) -> int:
    """``aai_peer_upload_chunks``: upload chunks per owner rank of a peer group (1..8, default 4); 0 only queries."""
    return int(lib().aai_peer_upload_chunks(int(n)))


class PeerGroup:
    """``aai_peer_*`` (include/aai.h): ONE large image over one process per GPU, end to end from host buffers -- every
    source row crosses PCIe once, halos move over NVLink as the upload chunks land, no NCCL and no barrier per step.

    ``all_gather(obj) -> list`` is the caller's out-of-band channel (e.g. ``torch.distributed.all_gather_object``), used
    once to exchange the connection blobs."""

    def __init__(self, plan: Plan, dtype: int, channels: int, rank: int, world: int, device: int, all_gather):
        self.plan, self.rank, self.world, self.device = plan, rank, world, device
        self._h = C.c_void_p()
        _check(lib().aai_peer_create(C.byref(plan), int(dtype), int(channels), int(rank), int(world), int(device),
                                     C.byref(self._h)))
        try:
            buf = C.create_string_buffer(PEER_BLOB_BYTES)
            _check(lib().aai_peer_export(self._h, buf))
            blobs = all_gather(buf.raw)
            if len(blobs) != world or any(len(b) != PEER_BLOB_BYTES for b in blobs):
                raise AaiError(ERR_ARGUMENT, "peer group: the gather must return one blob per rank, in rank order")
            _check(lib().aai_peer_connect(self._h, b"".join(blobs)))
        except Exception:
            self.close()
            raise

    def owned_rows(self) -> Tuple[int, int]:
        a, b = C.c_int64(), C.c_int64()
        _check(lib().aai_peer_owned_rows(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def band(self) -> Tuple[int, int]:
        a, b = C.c_int64(), C.c_int64()
        _check(lib().aai_peer_band(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def device_source(self) -> Image:
        img = Image()
        _check(lib().aai_peer_device_source(self._h, C.byref(img)))
        return img

    def run(self, host_src: Image, host_dst: Image, mode: int = MODE_AREA_AVERAGE, arith: int = ARITH_F64,
            stream: int = 0, synchronize: bool = True) -> None:
        _check(lib().aai_peer_run(self._h, int(mode), int(arith), C.byref(host_src), C.byref(host_dst),
                                  C.c_void_p(stream), int(bool(synchronize))))

    def last_timing(self) -> dict:
        """Completion times [ms from the start of the last step] of this rank's upload, pulls, kernels, downloads."""
        ms = (C.c_float * 4)()
        _check(lib().aai_peer_last_timing(self._h, ms))
        return {"upload_ms": ms[0], "pull_ms": ms[1], "kernel_ms": ms[2], "download_ms": ms[3]}

    def close(self) -> None:
        if self._h:
            lib().aai_peer_destroy(self._h)
            self._h = C.c_void_p()


@dataclass
class Result:
    ok: bool
    message: str
    dst: np.ndarray
    dst_isocenter: Tuple[float, float]
    plan: Plan


class AreaAverageInterpolation:
    """Operator with the reference's method names and argument meaning (Source.cpp:52-57, 584-586).

    ``src`` is ``[h, w]`` (the reference's ``IMG``; float64 reproduces it exactly) or, as an extension,
    ``[h, w, c]`` interleaved channels / float32 / uint8 / uint16.  Returns ``Result``: ``ok``/``message`` are the
    reference's ``pair<bool,string>``, ``dst`` its resized output image, ``dst_isocenter`` its out parameter
    (left at ``dst_isocenter_in`` when validation fails, like the reference).

    ``arith=ARITH_F32`` for float32 / uint8 / uint16 images.  The result is float64 for float64 and uint16 sources and
    under ``ARITH_F64``, else float32; ``out_dtype`` overrides that (a uint8 canvas takes any source but uint16, a uint16
    canvas a uint16 source only; integer canvases are rounded half up and saturated).  uint16 sources go to the library
    as they are (2 bytes per value), so ``out_dtype=np.uint16`` or ``np.float32`` keeps every buffer small.
    """

    def __init__(self, arith: int = ARITH_F64, devices: Optional[Sequence[int]] = None, out_dtype=None):
        self.arith = arith
        self.devices = list(devices) if devices else None
        self.out_dtype = out_dtype

    def _run(self, mode, src, srcResolution, dstResolution, srcIsocenter, rotationAngle, dstIsocenter):
        src = np.asarray(src)
        if src.ndim == 1 and src.size == 0:
            src = src.reshape(0, 0)
        if src.ndim not in (2, 3):
            raise ValueError("src must be [h, w] or [h, w, c]")
        h, w = src.shape[0], src.shape[1]
        plan = make_plan(w, h, srcResolution, dstResolution, srcIsocenter, rotationAngle)
        if plan.status != AAI_OK:
            if plan.status > ERR_NO_COLUMNS:
                raise AaiError(plan.status, plan.message)
            return Result(False, plan.message, np.empty((0, 0)), tuple(dstIsocenter), plan)
        if src.dtype not in _NP_TO_AAI:
            src = src.astype(np.float64)
        src = np.ascontiguousarray(src)
        # (uint16 sources keep the float64 result they had when they were widened to float64 before the call)
        out_dtype = np.dtype(self.out_dtype) if self.out_dtype is not None else (
            np.dtype(np.float64) if src.dtype in (np.float64, np.uint16) or self.arith == ARITH_F64
            else np.dtype(np.float32))
        shape = (plan.dst_h, plan.dst_w) + ((src.shape[2],) if src.ndim == 3 else ())
        dst = np.empty(shape, dtype=out_dtype)
        if dst.size:
            run_host(plan, src, dst, mode, self.arith, self.devices)
        return Result(True, "", dst, plan.dst_isocenter, plan)

    def areaAverageInterpolation(self, src, srcResolution, dstResolution, srcIsocenter, rotationAngle,
                                 dstIsocenter=(0.0, 0.0)) -> Result:
        return self._run(MODE_AREA_AVERAGE, src, srcResolution, dstResolution, srcIsocenter, rotationAngle,
                         dstIsocenter)

    def fastAreaAverageInterpolation(self, src, srcResolution, dstResolution, srcIsocenter, rotationAngle,
                                     dstIsocenter=(0.0, 0.0)) -> Result:
        return self._run(MODE_FAST, src, srcResolution, dstResolution, srcIsocenter, rotationAngle, dstIsocenter)

    def exactAreaAverageInterpolation(self, src, srcResolution, dstResolution, srcIsocenter, rotationAngle,
                                      dstIsocenter=(0.0, 0.0)) -> Result:
        """Not in the reference (SURVEY 8f row f4): geometrically exact overlap areas, without the shape-2/4 quirk."""
        return self._run(MODE_AREA_AVERAGE_EXACT, src, srcResolution, dstResolution, srcIsocenter, rotationAngle,
                         dstIsocenter)


def __getattr__(name):
    # the torch entry points live in torch_ops, which imports torch: loaded on first use, not at package import (and
    # left out of __all__, so that `from area_average_interpolation_b200 import *` does not import torch either)
    if name in ("resample", "resample_adjoint"):
        from . import torch_ops

        return getattr(torch_ops, name)
    raise AttributeError(f"module {__name__!r} has no attribute {name!r}")


__all__ = [
    "AreaAverageInterpolation", "Result", "Plan", "Image", "AaiError", "make_plan", "partition_rows",
    "band_source_window", "covered_pixels", "device_count", "launch_count", "last_host_timing", "run_device", "run_device_batch", "run_device_adjoint",
    "expand_device", "measure_fp32_tflops", "image_alloc", "image_free", "image_upload", "image_download", "image_copy_rows",
    "ipc_export", "ipc_open", "ipc_close",
    "run_host", "run_host_band", "run_host_batch", "PeerGroup", "tensor_image", "status_string", "last_error", "lib", "LIB_PATH",
]
