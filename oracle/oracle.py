"""ctypes binding of the CPU oracle (oracle/ssimu2_oracle.c).

TEST INFRASTRUCTURE ONLY.  Importable from tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs; the product package never imports this module.

Every function mirrors one step of the reference's CPU SSIMULACRA2
(/root/reference/crates/ssimulacra2-cuda/examples/cpu.rs) or of its GPU colour front-end
(/root/reference/crates/cuda-colorspace-kernel/src/biplanar.rs); see the C file for file:line.
Planar images are numpy float32 arrays of shape (3, H, W).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libssimu2_oracle.so")

MATRIX = {"bt709": 0, "bt601_525": 1, "bt601_625": 2}


def build(force: bool = False) -> str:
    src = os.path.join(_HERE, "ssimu2_oracle.c")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-B", "libssimu2_oracle.so"],
                              stdout=subprocess.DEVNULL)
    return _SO


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            build()
        _lib = C.CDLL(_SO)
        _lib.oracle_score_from_averages.restype = C.c_double
    return _lib


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def srgb8_lut() -> np.ndarray:
    out = np.zeros(256, np.float32)
    lib().oracle_srgb8_lut(_p(out))
    return out


def weights() -> np.ndarray:
    out = np.zeros(108, np.float64)
    lib().oracle_weights(_p(out))
    return out


def rg_constants() -> np.ndarray:
    out = np.zeros(9, np.float32)
    lib().oracle_rg_constants(_p(out))
    return out


def opsin_constants() -> np.ndarray:
    out = np.zeros(12, np.float32)
    lib().oracle_opsin_constants(_p(out))
    return out


def yuv_coefficients(matrix="bt709", bits=8, full_range=False) -> np.ndarray:
    out = np.zeros(5, np.float32)
    lib().oracle_yuv_coefficients(MATRIX[matrix], bits, int(full_range), _p(out))
    return out


def matrix_kr_kb(matrix="bt709") -> np.ndarray:
    out = np.zeros(2, np.float32)
    lib().oracle_matrix_kr_kb(MATRIX[matrix], _p(out))
    return out


# ---------------------------------------------------------------- front-ends -> planar linear
def linear_from_srgb8(img: np.ndarray) -> np.ndarray:
    """img: (H, W, 3) uint8 (any row stride) -> (3, H, W) float32 linear."""
    assert img.dtype == np.uint8 and img.ndim == 3 and img.shape[2] == 3
    h, w, _ = img.shape
    assert img.strides[1] == 3 and img.strides[2] == 1
    out = np.empty((3, h, w), np.float32)
    lib().oracle_linear_from_srgb8(_p(img), C.c_size_t(img.strides[0]), w, h, _p(out))
    return out


def linear_from_srgb16(img: np.ndarray) -> np.ndarray:
    assert img.dtype == np.uint16 and img.ndim == 3 and img.shape[2] == 3
    h, w, _ = img.shape
    img = np.ascontiguousarray(img)
    out = np.empty((3, h, w), np.float32)
    lib().oracle_linear_from_srgb16(_p(img), C.c_size_t(img.strides[0]), w, h, _p(out))
    return out


def linear_from_srgbf32(img: np.ndarray) -> np.ndarray:
    assert img.dtype == np.float32 and img.ndim == 3 and img.shape[2] == 3
    h, w, _ = img.shape
    img = np.ascontiguousarray(img)
    out = np.empty((3, h, w), np.float32)
    lib().oracle_linear_from_srgbf32(_p(img), C.c_size_t(img.strides[0]), w, h, _p(out))
    return out


def linear_from_linearf32(img: np.ndarray) -> np.ndarray:
    assert img.dtype == np.float32 and img.ndim == 3 and img.shape[2] == 3
    h, w, _ = img.shape
    img = np.ascontiguousarray(img)
    out = np.empty((3, h, w), np.float32)
    lib().oracle_linear_from_linearf32(_p(img), C.c_size_t(img.strides[0]), w, h, _p(out))
    return out


def linear_from_yuv420(buf: np.ndarray, pitch: int, coded_height: int, w: int, h: int, bits: int,
                       matrix="bt709", full_range=False) -> np.ndarray:
    """buf: flat uint8 array holding an NVDEC-style biplanar frame: Y rows at `pitch` bytes,
    UV plane at byte offset pitch*coded_height (cudarse-video/src/dec.rs:299-366).
    bits = 8 (NV12) or 16 (P016)."""
    assert buf.dtype == np.uint8 and buf.ndim == 1 and buf.flags.c_contiguous
    base = buf.ctypes.data
    out = np.empty((3, h, w), np.float32)
    fn = lib().oracle_linear_from_nv12 if bits == 8 else lib().oracle_linear_from_p016
    fn(C.c_void_p(base), C.c_void_p(base + pitch * coded_height), C.c_size_t(pitch),
       MATRIX[matrix], int(full_range), w, h, _p(out))
    return out


# ---------------------------------------------------------------- stages
def downscale_by_2(lin: np.ndarray) -> np.ndarray:
    lin = _f32(lin)
    _, h, w = lin.shape
    out = np.empty((3, (h + 1) // 2, (w + 1) // 2), np.float32)
    lib().oracle_downscale_by_2(_p(lin), w, h, _p(out))
    return out


def linear_to_xyb(lin: np.ndarray) -> np.ndarray:
    lin = _f32(lin)
    _, h, w = lin.shape
    out = np.empty_like(lin)
    lib().oracle_linear_to_xyb(_p(lin), w, h, _p(out))
    return out


def blur_horizontal(plane: np.ndarray) -> np.ndarray:
    plane = _f32(plane)
    h, w = plane.shape
    out = np.empty_like(plane)
    lib().oracle_blur_horizontal(_p(plane), _p(out), w, h)
    return out


def blur_vertical(plane: np.ndarray) -> np.ndarray:
    plane = _f32(plane)
    h, w = plane.shape
    out = np.empty_like(plane)
    lib().oracle_blur_vertical(_p(plane), _p(out), w, h)
    return out


def blur_plane(plane: np.ndarray) -> np.ndarray:
    return blur_vertical(blur_horizontal(plane))


def map_inputs(ref_lin: np.ndarray, dis_lin: np.ndarray, scale: int):
    """Per-pixel inputs of the error maps of one scale (cpu.rs:604-627, :658-662), the f32 values ssim_map and
    edge_diff_map evaluate their maps from: -> (q, a, b), each float32 (3, H_s, W_s): q = the SSIM' quotient
    num_m * num_s / denom_s, a = |x2 - mu2|, b = |x1 - mu1|.  None when the pyramid has no such scale."""
    ref_lin, dis_lin = _f32(ref_lin), _f32(dis_lin)
    assert ref_lin.shape == dis_lin.shape and ref_lin.shape[0] == 3
    _, h, w = ref_lin.shape
    for _ in range(scale):
        w, h = (w + 1) // 2, (h + 1) // 2
    q, a, b = (np.empty((3, h, w), np.float32) for _ in range(3))
    _, h0, w0 = ref_lin.shape
    if lib().oracle_map_inputs(_p(ref_lin), _p(dis_lin), w0, h0, scale, _p(q), _p(a), _p(b)) != 0:
        return None
    return q, a, b


# ---------------------------------------------------------------- whole metric
def ssimu2_linear_planar(ref_lin: np.ndarray, dis_lin: np.ndarray):
    """-> (score, norms[108], nscales).  norms index = c*36 + s*6 + n*3 + m (WEIGHT order)."""
    ref_lin, dis_lin = _f32(ref_lin), _f32(dis_lin)
    assert ref_lin.shape == dis_lin.shape and ref_lin.shape[0] == 3
    _, h, w = ref_lin.shape
    score = C.c_double(0.0)
    norms = np.zeros(108, np.float64)
    ns = lib().oracle_ssimu2_linear_planar(_p(ref_lin), _p(dis_lin), w, h, C.byref(score), _p(norms))
    return score.value, norms, ns


def ssimu2_srgb8(ref: np.ndarray, dis: np.ndarray):
    return ssimu2_linear_planar(linear_from_srgb8(ref), linear_from_srgb8(dis))


def ssimu2_yuv420(ref_buf, dis_buf, pitch, coded_height, w, h, bits, matrix="bt709",
                  full_range=False):
    a = linear_from_yuv420(ref_buf, pitch, coded_height, w, h, bits, matrix, full_range)
    b = linear_from_yuv420(dis_buf, pitch, coded_height, w, h, bits, matrix, full_range)
    return ssimu2_linear_planar(a, b)


def ssimu2_linearf32(ref: np.ndarray, dis: np.ndarray):
    return ssimu2_linear_planar(linear_from_linearf32(ref), linear_from_linearf32(dis))


def score_from_norms(norms: np.ndarray, nscales: int = 6) -> float:
    """Msssim::score (cpu.rs:728-871) on a norms[108] vector in WEIGHT order."""
    norms = np.asarray(norms, np.float64)
    ssim6 = np.zeros((6, 6), np.float64)
    edge12 = np.zeros((6, 12), np.float64)
    for c in range(3):
        for s in range(6):
            for n in range(2):
                ssim6[s, c * 2 + n] = norms[c * 36 + s * 6 + n * 3 + 0]
                edge12[s, c * 4 + n] = norms[c * 36 + s * 6 + n * 3 + 1]
                edge12[s, c * 4 + n + 2] = norms[c * 36 + s * 6 + n * 3 + 2]
    return lib().oracle_score_from_averages(nscales, _p(ssim6), _p(edge12))
