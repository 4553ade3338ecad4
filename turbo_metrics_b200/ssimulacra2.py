"""Host-side mirror of the reference's metric op `Ssimulacra2`
(/root/reference/crates/ssimulacra2-cuda/src/lib.rs:27-291) over the C ABI.

Same call sequence as the reference -- construct once per (width, height), `compute` per pair,
`get_score` afterwards -- with the colour front-end (cuda-colorspace/src/lib.rs:33-169) folded
in: frames are handed over in the layout the decoder / NPP produces (NV12, P016, packed sRGB or
packed linear f32) instead of being converted to linear f32 by a separate op first.

PyTorch is only plumbing here: tensors own device memory, `torch.cuda.current_stream()` supplies
the stream handle.  All arithmetic happens in libssimu2_b200.so.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from enum import IntEnum
from typing import Optional, Sequence

import numpy as np

from . import _lib
from ._lib import Config, Frame, Info, Source, check


class PixelFormat(IntEnum):
    """turbo-metrics/src/lib.rs:125-130 `HwFrame` variants (+ the op's own linear input)."""
    NV12 = 0
    P016 = 1
    SRGB8 = 2
    SRGB16 = 3
    SRGBF32 = 4
    LINEARF32 = 5
    # NVDEC's 4:2:2 / 4:4:4 surfaces (cudaVideoSurfaceFormat_NV16 / _P216 / _YUV444 / _YUV444_16Bit)
    NV16 = 8
    P216 = 9
    YUV444 = 10
    YUV444P16 = 11


YUV_FORMATS = (PixelFormat.NV12, PixelFormat.P016, PixelFormat.NV16, PixelFormat.P216, PixelFormat.YUV444, PixelFormat.YUV444P16)
# the formats SSIMU2_FLAG_P016_DEEP applies to
YUV16_FORMATS = (PixelFormat.P016, PixelFormat.P216, PixelFormat.YUV444P16)


class ColorMatrix(IntEnum):
    """cuda-colorspace/src/lib.rs:8-13."""
    BT709 = 0
    BT601_525 = 1
    BT601_625 = 2


@dataclass
class DeviceFrame:
    """A borrowed frame: device (or host, for compute_from_cpu) addresses + pitch in bytes.
    `keepalive` holds whatever owns the memory (a torch tensor, a numpy array)."""
    plane0: int
    plane1: int
    pitch: int
    keepalive: object = None
    nbytes: int = 0

    def c(self) -> Frame:
        f = Frame()
        f.plane[0] = self.plane0
        f.plane[1] = self.plane1
        f.pitch = self.pitch
        return f

    @staticmethod
    def yuv420(buf, pitch: int, coded_height: int) -> "DeviceFrame":
        """NVDEC layout (cudarse-video/src/dec.rs:299-366): Y at buf, CbCr at buf + pitch*coded_height.
        buf: 1-D uint8 torch tensor (device or pinned host) or numpy array."""
        base = buf.data_ptr() if hasattr(buf, "data_ptr") else buf.ctypes.data
        nbytes = buf.numel() * buf.element_size() if hasattr(buf, "numel") else buf.nbytes
        return DeviceFrame(base, base + pitch * coded_height, pitch, buf, nbytes)

    @staticmethod
    def yuv422(buf, pitch: int, coded_height: int) -> "DeviceFrame":
        """NVDEC NV16 / P216 layout: Y at buf, interleaved CbCr of full height at buf + pitch*coded_height.
        buf: 1-D uint8 torch tensor (device or pinned host) or numpy array.  `nbytes` (what compute_from_cpu copies) is the
        buffer's size, which must reach the end of the last chroma row."""
        return DeviceFrame.yuv420(buf, pitch, coded_height)

    @staticmethod
    def yuv444(buf, pitch: int, coded_height: int) -> "DeviceFrame":
        """NVDEC YUV444 / YUV444_16Bit layout: Y, Cb and Cr planes of `coded_height` rows at `pitch` bytes, one after the other
        (also a contiguous (3, coded_height, pitch) array).  The library finds Cr at plane1 + (plane1 - plane0).
        buf: 1-D uint8 torch tensor (device or pinned host) or numpy array."""
        return DeviceFrame.yuv420(buf, pitch, coded_height)

    @staticmethod
    def packed(img, pitch: Optional[int] = None) -> "DeviceFrame":
        """Packed RGB image (H, W, 3) of u8 / u16 / f32, or its rows as (H, 3 * W): NPP `Image<_, C<3>>` layout.  Rows may be
        padded (a view such as img[:, :w] of a wider image), but the samples of a row must be packed: ValueError otherwise.
        `nbytes` is the span from the first sample to the last, what compute_from_cpu copies."""
        if hasattr(img, "data_ptr"):
            base, esize = img.data_ptr(), img.element_size()
            strides = tuple(s * esize for s in img.stride())
        else:
            base, esize, strides = img.ctypes.data, img.itemsize, tuple(img.strides)
        shape = tuple(img.shape)
        packed = (len(shape) == 3 and shape[2] == 3 and strides[1:] == (3 * esize, esize)) or \
                 (len(shape) == 2 and strides[1] == esize)
        if not packed:
            raise ValueError(f"not a packed RGB image: shape {shape}, byte strides {strides}")
        if pitch is None:
            pitch = strides[0]
        row = int(np.prod(shape[1:])) * esize
        return DeviceFrame(base, 0, pitch, img, (shape[0] - 1) * pitch + row)


def make_config(width, height, fmt, matrix=ColorMatrix.BT709, full_range=False, device=0, batch=0, ring=0,
                pipeline=_lib.PIPELINE_DEFAULT, flags=0, input_group=0, tile=0) -> Config:
    cfg = Config()
    cfg.width, cfg.height, cfg.format, cfg.matrix = width, height, int(fmt), int(matrix)
    cfg.full_range, cfg.device, cfg.batch, cfg.ring = int(full_range), device, batch, ring
    cfg.pipeline, cfg.flags, cfg.input_group, cfg.tile = pipeline, flags, input_group, tile
    return cfg


def make_source(cfg: Config, dis_fmt=None, dis_matrix=None, dis_full_range=None, dis_p016_deep=None, dis_width=None,
                dis_height=None) -> Optional[Source]:
    """ssimu2_source of the distorted frames for a handle whose reference frames `cfg` describes, or None when no dis_*
    argument is given.  A dis_* argument left at None takes the reference's value; the deep flag is the reference's when the
    distorted frames are P016 too.  dis_width / dis_height: the distorted frames' size when they are smaller than the
    reference's (upscaled to it on the GPU); None or 0 = the reference's."""
    if dis_fmt is None and dis_matrix is None and dis_full_range is None and dis_p016_deep is None and \
            dis_width is None and dis_height is None:
        return None
    src = Source()
    src.format = int(cfg.format if dis_fmt is None else dis_fmt)
    src.matrix = int(cfg.matrix if dis_matrix is None else dis_matrix)
    src.full_range = int(cfg.full_range if dis_full_range is None else dis_full_range)
    if dis_p016_deep is None:
        dis_p016_deep = bool(cfg.flags & _lib.FLAG_P016_DEEP) and src.format in YUV16_FORMATS
    src.flags = _lib.FLAG_P016_DEEP if dis_p016_deep else 0
    src.width = int(dis_width or 0)
    src.height = int(dis_height or 0)
    return src


def is_mixed(cfg: Config, src: Optional[Source]) -> bool:
    """Whether ssimu2_create_mixed(cfg, src) makes a mixed handle: the sides differ in format or deep flag, (YUV) in matrix or
    range, or in size (a scaled handle).  Otherwise the handle is an ordinary one."""
    if src is None:
        return False
    deep = _lib.FLAG_P016_DEEP
    yuv = cfg.format in YUV_FORMATS
    return not (src.format == cfg.format and (src.flags & deep) == (cfg.flags & deep) and
                (not yuv or (src.matrix == cfg.matrix and bool(src.full_range) == bool(cfg.full_range))) and
                not is_scaled(cfg, src))


def is_scaled(cfg: Config, src: Optional[Source]) -> bool:
    """Whether the distorted frames `src` describes are smaller than the reference frames (upscaled before scoring)."""
    return src is not None and (src.width or cfg.width, src.height or cfg.height) != (cfg.width, cfg.height)


class Ssimulacra2:
    """`Ssimulacra2::new` (lib.rs:48-107): an instance is valid for one width x height x format."""

    def __init__(self, width: int, height: int, fmt: PixelFormat = PixelFormat.LINEARF32,
                 matrix: ColorMatrix = ColorMatrix.BT709, full_range: bool = False, device: int = 0,
                 batch: int = 0, ring: int = 0, pipeline: Optional[str] = None, score_only: bool = False,
                 input_group: int = 0, timing: bool = True, p016_deep: bool = False, dis_fmt: Optional[PixelFormat] = None,
                 dis_matrix: Optional[ColorMatrix] = None, dis_full_range: Optional[bool] = None,
                 dis_p016_deep: Optional[bool] = None, dis_width: Optional[int] = None, dis_height: Optional[int] = None,
                 tile: int = 0):
        """pipeline: None / "hv" = the product pipeline (front-end, fused H+V kernel, finalize); "split" = development
        pipeline with the H-pass planes in HBM (debug_read(what=1)).
        score_only: SSIMU2_FLAG_SCORE_ONLY -- skip the work whose weights are zero (scores identical, no norms).
        input_group: pairs per front-end launch (0 = whole batch): input frames are consumed sooner, see wait_input().
        p016_deep: SSIMU2_FLAG_P016_DEEP -- P016 / P216 / YUV444P16 samples with more than 10 significant bits (12-bit sources): same results,
        a front-end without the 10-bit memo tables (of the reference frames when the distorted frames are described apart).
        dis_fmt, dis_matrix, dis_full_range, dis_p016_deep: the distorted frames' own description (None = as the reference);
        any of them set creates the handle with ssimu2_create_mixed.  Host frames of a mixed handle are copied with each
        side's own `nbytes`.
        dis_width, dis_height: the distorted frames' size when it is smaller than width x height (e.g. a 720p encode scored
        against its 1080p source): they are upscaled to width x height on the GPU (bicubic Catmull-Rom, ssimu2_source) and
        scored there.  Distorted frames are then given at their own size.
        tile: per-tile scores on a grid of tile x tile pixels (a power of two, 64 .. 32768; 0 = off): get_tile_scores() gives
        a SSIMULACRA2 score per tile, pooled from the frame's own error maps (ssimu2_config.tile)."""
        self._h = C.c_void_p()
        if pipeline not in (None, "hv", "split"):
            raise ValueError(f"unknown pipeline {pipeline!r}")
        flags = (_lib.FLAG_SCORE_ONLY if score_only else 0) | (0 if timing else _lib.FLAG_NO_TIMING) | \
                (_lib.FLAG_P016_DEEP if p016_deep else 0)
        cfg = make_config(width, height, fmt, matrix, full_range, device, batch, ring,
                          _lib.PIPELINE_SPLIT if pipeline == "split" else _lib.PIPELINE_DEFAULT, flags, input_group, tile)
        src = make_source(cfg, dis_fmt, dis_matrix, dis_full_range, dis_p016_deep, dis_width, dis_height)
        if src is None:
            check(_lib.lib().ssimu2_create(C.byref(self._h), C.byref(cfg)), "ssimu2_create")
        else:
            check(_lib.lib().ssimu2_create_mixed(C.byref(self._h), C.byref(cfg), C.byref(src)), "ssimu2_create_mixed")
        self.width, self.height, self.format = width, height, PixelFormat(fmt)
        self.dis_format = self.format if src is None else PixelFormat(src.format)
        self.dis_width = src.width if src is not None and src.width else width
        self.dis_height = src.height if src is not None and src.height else height
        self.mixed = is_mixed(cfg, src)
        self._keep = {}
        self._last = None

    # -- lifetime -------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            _lib.lib().ssimu2_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def mem_usage(self) -> int:
        """`Ssimulacra2::mem_usage` (lib.rs:110-138)."""
        n = C.c_size_t()
        check(_lib.lib().ssimu2_mem_usage(self._h, C.byref(n)), "ssimu2_mem_usage")
        return n.value

    def info(self) -> Info:
        i = Info()
        check(_lib.lib().ssimu2_get_info(self._h, C.byref(i)), "ssimu2_get_info")
        return i

    # -- scoring --------------------------------------------------------------------------
    @staticmethod
    def _stream_handle(stream) -> int:
        if stream is None:
            import torch
            return torch.cuda.current_stream().cuda_stream
        if hasattr(stream, "cuda_stream"):
            return stream.cuda_stream
        return int(stream)

    def compute(self, ref: DeviceFrame, dis: DeviceFrame, stream=None) -> int:
        """`Ssimulacra2::compute` (lib.rs:283-287): asynchronous; returns the pair's ticket."""
        t = C.c_uint64()
        a, b = ref.c(), dis.c()
        check(_lib.lib().ssimu2_submit(self._h, C.byref(a), C.byref(b), C.c_void_p(self._stream_handle(stream)),
                                       C.byref(t)), "ssimu2_submit")
        self._keep[t.value] = (ref, dis)
        self._last = t.value
        return t.value

    def compute_batch(self, refs: Sequence[DeviceFrame], diss: Sequence[DeviceFrame], stream=None) -> range:
        n = len(refs)
        assert n == len(diss)
        A = (Frame * n)(*[f.c() for f in refs])
        B = (Frame * n)(*[f.c() for f in diss])
        t = C.c_uint64()
        check(_lib.lib().ssimu2_submit_batch(self._h, n, A, B, C.c_void_p(self._stream_handle(stream)), C.byref(t)),
              "ssimu2_submit_batch")
        for i in range(n):
            self._keep[t.value + i] = (refs[i], diss[i])
        if n:
            self._last = t.value + n - 1
        return range(t.value, t.value + n)

    def compute_from_cpu(self, ref: DeviceFrame, dis: DeviceFrame) -> int:
        """`Ssimulacra2::compute_from_cpu_srgb_sync` (lib.rs:232-250) without the sync: frames live in
        host memory; the library stages them on the device."""
        t = C.c_uint64()
        a, b = ref.c(), dis.c()
        if self.mixed:
            assert ref.nbytes and dis.nbytes
            check(_lib.lib().ssimu2_submit_host_sized(self._h, 1, C.byref(a), ref.nbytes, C.byref(b), dis.nbytes, C.byref(t)),
                  "ssimu2_submit_host_sized")
        else:
            assert ref.nbytes and ref.nbytes == dis.nbytes
            check(_lib.lib().ssimu2_submit_host(self._h, C.byref(a), C.byref(b), ref.nbytes, C.byref(t)),
                  "ssimu2_submit_host")
        self._keep[t.value] = (ref, dis)
        self._last = t.value
        return t.value

    def compute_from_cpu_batch(self, refs: Sequence[DeviceFrame], diss: Sequence[DeviceFrame]) -> range:
        """n host pairs in one call (`ssimu2_submit_host_batch`; `ssimu2_submit_host_sized` on a mixed handle)."""
        n = len(refs)
        assert n == len(diss) and n > 0
        A = (Frame * n)(*[f.c() for f in refs])
        B = (Frame * n)(*[f.c() for f in diss])
        t = C.c_uint64()
        if self.mixed:
            assert all(f.nbytes == refs[0].nbytes for f in refs) and all(f.nbytes == diss[0].nbytes for f in diss)
            check(_lib.lib().ssimu2_submit_host_sized(self._h, n, A, refs[0].nbytes, B, diss[0].nbytes, C.byref(t)),
                  "ssimu2_submit_host_sized")
        else:
            assert all(f.nbytes == refs[0].nbytes for f in list(refs) + list(diss))
            check(_lib.lib().ssimu2_submit_host_batch(self._h, n, A, B, refs[0].nbytes, C.byref(t)), "ssimu2_submit_host_batch")
        for i in range(n):
            self._keep[t.value + i] = (refs[i], diss[i])
        self._last = t.value + n - 1
        return range(t.value, t.value + n)

    def flush(self):
        check(_lib.lib().ssimu2_flush(self._h), "ssimu2_flush")

    def get_score(self, ticket: Optional[int] = None) -> float:
        """`Ssimulacra2::get_score` (lib.rs:289-291); defaults to the last submitted pair."""
        if ticket is None:
            if self._last is None:
                raise ValueError("get_score() before any compute()")
            ticket = self._last
        s = C.c_double()
        check(_lib.lib().ssimu2_get_score(self._h, ticket, C.byref(s)), "ssimu2_get_score")
        self._release()
        return s.value

    def get_scores(self, tickets: range) -> np.ndarray:
        """Scores of consecutive tickets (`ssimu2_get_scores`): the per-frame score stream in submission order."""
        n = len(tickets)
        out = np.zeros(n, np.float64)
        if n:
            assert tickets.step == 1
            check(_lib.lib().ssimu2_get_scores(self._h, tickets.start, n, out.ctypes.data_as(C.POINTER(C.c_double))), "ssimu2_get_scores")
            self._release()
        return out

    def get_norms(self, ticket: int) -> np.ndarray:
        out = np.zeros(108, np.float64)
        check(_lib.lib().ssimu2_get_norms(self._h, ticket, out.ctypes.data_as(C.POINTER(C.c_double))),
              "ssimu2_get_norms")
        return out

    def tile_grid(self):
        """-> (tile, tiles_x, tiles_y, capacity): the tile size (0 without tiles), the grid, and how many of the most recent
        tickets still have their tile map."""
        t, x, y, cap = C.c_uint32(), C.c_uint32(), C.c_uint32(), C.c_uint64()
        check(_lib.lib().ssimu2_get_tile_grid(self._h, C.byref(t), C.byref(x), C.byref(y), C.byref(cap)), "ssimu2_get_tile_grid")
        return t.value, x.value, y.value, cap.value

    def get_tile_scores(self, ticket: int) -> np.ndarray:
        """The ticket's tile scores, float64 of shape (tiles_y, tiles_x): 100 where nothing differs, lower where it does."""
        _, tx, ty, _ = self.tile_grid()
        out = np.zeros((ty, tx), np.float64)
        check(_lib.lib().ssimu2_get_tile_scores(self._h, ticket, out.ctypes.data_as(C.POINTER(C.c_double)), out.size),
              "ssimu2_get_tile_scores")
        self._release()
        return out

    def compute_sync(self, ref: DeviceFrame, dis: DeviceFrame, stream=None) -> float:
        """`Ssimulacra2::compute_sync` (lib.rs:271-279)."""
        return self.get_score(self.compute(ref, dis, stream))

    def compute_from_cpu_sync(self, ref: DeviceFrame, dis: DeviceFrame) -> float:
        return self.get_score(self.compute_from_cpu(ref, dis))

    def completed(self) -> int:
        """`ssimu2_completed`: every ticket below the returned watermark is done and its frames are no longer read."""
        w = C.c_uint64()
        check(_lib.lib().ssimu2_completed(self._h, C.byref(w)), "ssimu2_completed")
        return w.value

    def _release(self):
        # batches complete out of order across ring slots: only the in-order watermark says which inputs are free
        w = self.completed()
        for k in [k for k in self._keep if k < w]:
            del self._keep[k]

    def stream_wait(self, ticket: int, stream=None):
        """`ssimu2_stream_wait`: make `stream` wait (on the device) for the ticket's batch."""
        check(_lib.lib().ssimu2_stream_wait(self._h, ticket, C.c_void_p(self._stream_handle(stream))), "ssimu2_stream_wait")

    def wait_input(self, ticket: int, stream=None):
        """`ssimu2_stream_wait_input`: make `stream` wait until the ticket's input frames have been consumed -- what a
        decoder needs before it reuses a surface (cudarse-video/src/dec.rs:277-287)."""
        check(_lib.lib().ssimu2_stream_wait_input(self._h, ticket, C.c_void_p(self._stream_handle(stream))),
              "ssimu2_stream_wait_input")

    # -- device-side results / introspection ---------------------------------------------------
    def scores_device(self):
        p, cap = C.c_uint64(), C.c_uint64()
        check(_lib.lib().ssimu2_scores_device(self._h, C.byref(p), C.byref(cap)), "ssimu2_scores_device")
        return p.value, cap.value

    def debug_read(self, ticket: int, what: int, scale: int) -> np.ndarray:
        i = self.info()
        w, h = i.width[scale], i.height[scale]
        planes = 6 if what == 0 else 15
        out = np.zeros((planes, h, w), np.float32)
        check(_lib.lib().ssimu2_debug_read(self._h, ticket, what, scale, out.ctypes.data_as(C.POINTER(C.c_float)),
                                           out.size), "ssimu2_debug_read")
        return out

    def debug_strips(self):
        """-> (strip0[nscales], n_strips[nscales], strip_cols): the rows of each scale in the partial-sum table and the
        columns one strip covers."""
        s0, ns, cols = (C.c_uint32 * 6)(), (C.c_uint32 * 6)(), C.c_uint32()
        check(_lib.lib().ssimu2_debug_strips(self._h, s0, ns, C.byref(cols)), "ssimu2_debug_strips")
        n = self.info().nscales
        return list(s0)[:n], list(ns)[:n], cols.value

    def debug_partials(self, ticket: int) -> list:
        """The pair's per-strip partial sums, one float64 array of shape (n_strips, 3, 6) per scale: channel x {ssim L1,
        ssim L4, artifact L1, artifact L4, detail L1, detail L4} (L1: the strip's sum of the map, L4: of its fourth power).
        Valid until the batch slot that served the ticket is reused, like debug_read."""
        strip0, n_strips, _ = self.debug_strips()
        out = np.zeros((sum(n_strips), 3, 6), np.float64)
        check(_lib.lib().ssimu2_debug_read_partials(self._h, ticket, out.ctypes.data_as(C.POINTER(C.c_double)), out.size),
              "ssimu2_debug_read_partials")
        return [out[s0:s0 + n] for s0, n in zip(strip0, n_strips)]

    def debug_tile_units(self):
        """-> per scale (entry0, units, unit_cols): where the scale starts in the tile table, its column units per tile row
        and the columns of one unit."""
        e0, un, uc = (C.c_uint32 * 6)(), (C.c_uint32 * 6)(), (C.c_uint32 * 6)()
        check(_lib.lib().ssimu2_debug_tile_units(self._h, e0, un, uc), "ssimu2_debug_tile_units")
        return [(e0[s], un[s], uc[s]) for s in range(self.info().nscales)]

    def debug_tile_partials(self, ticket: int) -> list:
        """The pair's per-tile sums, one float64 array of shape (tiles_y, units, 3, 6) per scale (entries as in
        debug_partials; a unit is a tile column, or a 64-column strip of it).  Valid until the batch slot that served the
        ticket is reused, like debug_read."""
        layout = self.debug_tile_units()
        _, _, ty, _ = self.tile_grid()
        n = sum(ty * u for _, u, _ in layout)
        out = np.zeros((n, 3, 6), np.float64)
        check(_lib.lib().ssimu2_debug_read_tile_partials(self._h, ticket, out.ctypes.data_as(C.POINTER(C.c_double)), out.size),
              "ssimu2_debug_read_tile_partials")
        return [out[e0:e0 + ty * u].reshape(ty, u, 3, 6) for e0, u, _ in layout]

    def kernel_ms(self, reset: bool = False):
        """-> (ms_total[4] for frontend/hpass/vpass/finalize, batches, pairs) since the last reset."""
        ms = (C.c_double * 4)()
        b, p = C.c_uint64(), C.c_uint64()
        check(_lib.lib().ssimu2_kernel_ms(self._h, ms, C.byref(b), C.byref(p), int(reset)), "ssimu2_kernel_ms")
        return list(ms), b.value, p.value

    def last_batch_ms(self):
        ms = (C.c_float * 4)()
        check(_lib.lib().ssimu2_last_batch_ms(self._h, ms), "ssimu2_last_batch_ms")
        return list(ms)


class ShardedSsimulacra2:
    """`ssimu2_shard_*`: one scorer per GPU of the box, each driven by its own host thread inside the library; the caller
    sees one ordered score stream (global tickets).  No torch.distributed, no NCCL: pairs are independent
    (ssimulacra2-cuda/README.md:26-27), the reference's single-GPU frame loop is turbo-metrics/src/lib.rs:362-433."""

    def __init__(self, width: int, height: int, fmt: PixelFormat, devices: Sequence[int], matrix: ColorMatrix = ColorMatrix.BT709,
                 full_range: bool = False, batch: int = 0, ring: int = 0, score_only: bool = False,
                 dis_fmt: Optional[PixelFormat] = None, dis_matrix: Optional[ColorMatrix] = None,
                 dis_full_range: Optional[bool] = None, dis_p016_deep: Optional[bool] = None, dis_width: Optional[int] = None,
                 dis_height: Optional[int] = None):
        """dis_*: the distorted frames' own description and size, as for `Ssimulacra2` (every worker's handle is
        ssimu2_create_mixed)."""
        self._s = C.c_void_p()
        flags = _lib.FLAG_SCORE_ONLY if score_only else 0
        cfg = make_config(width, height, fmt, matrix, full_range, 0, batch, ring, _lib.PIPELINE_DEFAULT, flags, 0)
        devs = (C.c_int32 * len(devices))(*devices)
        src = make_source(cfg, dis_fmt, dis_matrix, dis_full_range, dis_p016_deep, dis_width, dis_height)
        if src is None:
            check(_lib.lib().ssimu2_shard_create(C.byref(self._s), C.byref(cfg), devs, len(devices)), "ssimu2_shard_create")
        else:
            check(_lib.lib().ssimu2_shard_create_mixed(C.byref(self._s), C.byref(cfg), C.byref(src), devs, len(devices)),
                  "ssimu2_shard_create_mixed")
        self.mixed = is_mixed(cfg, src)
        self.devices = list(devices)
        self._keep = []
        self._done_upto = 0

    def close(self):
        if getattr(self, "_s", None) is not None and self._s:
            _lib.lib().ssimu2_shard_destroy(self._s)
            self._s = None
            self._keep = []

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def device_of(self, ticket: int) -> int:
        d = C.c_int32()
        check(_lib.lib().ssimu2_shard_device_of(self._s, ticket, C.byref(d)), "ssimu2_shard_device_of")
        return d.value

    def submit_host(self, refs: Sequence[DeviceFrame], diss: Sequence[DeviceFrame]) -> range:
        n = len(refs)
        assert n == len(diss) and n > 0
        A = (Frame * n)(*[f.c() for f in refs])
        B = (Frame * n)(*[f.c() for f in diss])
        t = C.c_uint64()
        if self.mixed:
            check(_lib.lib().ssimu2_shard_submit_host_sized(self._s, n, A, refs[0].nbytes, B, diss[0].nbytes, C.byref(t)),
                  "ssimu2_shard_submit_host_sized")
        else:
            check(_lib.lib().ssimu2_shard_submit_host(self._s, n, A, B, refs[0].nbytes, C.byref(t)), "ssimu2_shard_submit_host")
        self._keep.append((t.value + n, refs, diss))
        return range(t.value, t.value + n)

    def submit_device(self, refs: Sequence[DeviceFrame], diss: Sequence[DeviceFrame], streams: Optional[Sequence[int]] = None) -> range:
        """Frames must live on the device `device_of(ticket)` names for their ticket."""
        n = len(refs)
        assert n == len(diss) and n > 0
        A = (Frame * n)(*[f.c() for f in refs])
        B = (Frame * n)(*[f.c() for f in diss])
        S = None
        if streams is not None:
            S = (C.c_void_p * len(self.devices))(*[C.c_void_p(x) for x in streams])
        t = C.c_uint64()
        check(_lib.lib().ssimu2_shard_submit_device(self._s, n, A, B, S, C.byref(t)), "ssimu2_shard_submit_device")
        self._keep.append((t.value + n, refs, diss))
        return range(t.value, t.value + n)

    def flush(self):
        check(_lib.lib().ssimu2_shard_flush(self._s), "ssimu2_shard_flush")

    def get_scores(self, tickets: range) -> np.ndarray:
        n = len(tickets)
        out = np.zeros(n, np.float64)
        if n:
            check(_lib.lib().ssimu2_shard_get_scores(self._s, tickets.start, n, out.ctypes.data_as(C.POINTER(C.c_double))),
                  "ssimu2_shard_get_scores")
            # a submission's frames are free once every ticket up to its end has been fetched (contiguous watermark)
            if tickets.start <= self._done_upto:
                self._done_upto = max(self._done_upto, tickets.stop)
            self._keep = [k for k in self._keep if k[0] > self._done_upto]
        return out
