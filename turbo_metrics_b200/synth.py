"""Deterministic synthetic frame pairs (SURVEY.md section 8d) for the tests and bench.py.

There is no network, so datasets and bitstreams are replaced by seeded procedural content:
  reference : luma = sinusoid grating x slow cosine + 8-px smooth noise + white noise,
              chroma = two slow gradients around neutral
  distorted : reference passed through a [1 2 1]/4 horizontal blur + additive noise + coarse
              quantisation on every third 16x16 block  (scores spread roughly 30..90)
Layouts match what the decoder / NPP would hand over:
  yuv420 : NVDEC biplanar buffer, Y rows at `pitch` bytes, interleaved CbCr at pitch*coded_height
           (cudarse-video/src/dec.rs:299-366); 8-bit (NV12) or 10-bit in the high bits of u16 (P016)
  yuv422 : the same with an interleaved CbCr plane of full height (NV16 / P216)
  yuv444 : Y, Cb, Cr planes of coded_height rows one after the other (YUV444 / YUV444P16)
  srgb8  : packed RGB u8, (H, W, 3)
Everything is torch so the same code runs on the CPU (tests, oracle inputs) and on the GPU (bench).
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F


def _gen(seed: int, frame: int, device) -> torch.Generator:
    g = torch.Generator(device=device)
    g.manual_seed((0x5551AC2A ^ (seed << 20) ^ frame) & 0x7FFFFFFFFFFF)
    return g


def _smooth_noise(h, w, cell, g, device):
    gh, gw = h // cell + 2, w // cell + 2
    n = torch.rand((1, 1, gh, gw), generator=g, device=device)
    up = F.interpolate(n, size=(gh * cell, gw * cell), mode="bilinear", align_corners=False)
    return up[0, 0, :h, :w] - 0.5


def _base_luma(h, w, frame, g, device, phase=0.0):
    y = torch.arange(h, device=device, dtype=torch.float32)[:, None]
    x = torch.arange(w, device=device, dtype=torch.float32)[None, :]
    lum = 0.5 + 0.25 * torch.sin(2 * math.pi * (3 * x / w + frame / 97.0 + phase)) * torch.cos(2 * math.pi * 2 * y / h)
    lum = lum + 0.30 * _smooth_noise(h, w, 8, g, device)
    lum = lum + 0.03 * (torch.rand((h, w), generator=g, device=device) - 0.5) * 2
    return lum.clamp(0, 1)


def _distort(p, g, device, noise, qstep):
    """p in [0,1] (H, W): blur + noise + blockwise coarse quantisation."""
    h, w = p.shape
    pad = F.pad(p[None, None], (1, 1, 0, 0), mode="replicate")[0, 0]
    blur = 0.25 * pad[:, :-2] + 0.5 * pad[:, 1:-1] + 0.25 * pad[:, 2:]
    out = blur + noise * torch.randn((h, w), generator=g, device=device)
    by = torch.arange(h, device=device)[:, None] // 16
    bx = torch.arange(w, device=device)[None, :] // 16
    coarse = ((by * 7 + bx) % 3) == 0
    q = torch.round(out / qstep) * qstep
    out = torch.where(coarse, q, out)
    return out.clamp(0, 1)


def yuv420_geometry(w: int, h: int, bits: int):
    """NVDEC-like pitch / coded height: pitch = bytes per row rounded up to 256, height to 16... the
    configs of SURVEY.md section 8(d): 1080p NV12 -> pitch 2048, coded_height 1088; 4K P016 -> 7680, 2160."""
    bps = 1 if bits == 8 else 2
    pitch = (w * bps + 255) // 256 * 256
    coded_h = (h + 15) // 16 * 16
    return pitch, coded_h, pitch * coded_h + pitch * ((coded_h + 1) // 2)


def _pack_yuv(yv, cb, cr, w, h, bits, device):
    """yv (H,W), cb/cr (H/2,W/2) floats in [0,1] -> NVDEC buffer (uint8 1-D)."""
    pitch, coded_h, total = yuv420_geometry(w, h, bits)
    ch, cw = (h + 1) // 2, (w + 1) // 2
    if bits == 8:
        yq = torch.round(16 + 219 * yv).clamp(0, 255).to(torch.uint8)
        cbq = torch.round(128 + 224 * (cb - 0.5)).clamp(0, 255).to(torch.uint8)
        crq = torch.round(128 + 224 * (cr - 0.5)).clamp(0, 255).to(torch.uint8)
        buf = torch.zeros(total, dtype=torch.uint8, device=device)
        buf[: pitch * h].view(h, pitch)[:, :w] = yq
        uv = buf[pitch * coded_h: pitch * coded_h + pitch * ch].view(ch, pitch)
        uv[:, 0:2 * cw:2] = cbq
        uv[:, 1:2 * cw:2] = crq
        return buf
    # 10-bit in the high bits of 16 (P016)
    yq = (torch.round(64 + 876 * yv).clamp(0, 1023).to(torch.int32) << 6)
    cbq = (torch.round(512 + 896 * (cb - 0.5)).clamp(0, 1023).to(torch.int32) << 6)
    crq = (torch.round(512 + 896 * (cr - 0.5)).clamp(0, 1023).to(torch.int32) << 6)
    buf16 = torch.zeros(total // 2, dtype=torch.int32, device=device)
    p16 = pitch // 2
    buf16[: p16 * h].view(h, p16)[:, :w] = yq
    uv = buf16[p16 * coded_h: p16 * coded_h + p16 * ch].view(ch, p16)
    uv[:, 0:2 * cw:2] = cbq
    uv[:, 1:2 * cw:2] = crq
    # int32 (values < 65536) -> little-endian u16 bytes
    lo = (buf16 & 0xFF).to(torch.uint8)
    hi = ((buf16 >> 8) & 0xFF).to(torch.uint8)
    return torch.stack([lo, hi], dim=1).reshape(-1).contiguous()


def make_pair_yuv420(w: int, h: int, bits: int = 8, frame: int = 0, seed: int = 1, device="cpu"):
    """-> (ref_buf, dis_buf, pitch, coded_height); buffers are 1-D uint8 tensors on `device`."""
    g = _gen(seed, frame, device)
    ch, cw = (h + 1) // 2, (w + 1) // 2
    lum = _base_luma(h, w, frame, g, device)
    yy = torch.arange(ch, device=device, dtype=torch.float32)[:, None] / max(ch - 1, 1)
    xx = torch.arange(cw, device=device, dtype=torch.float32)[None, :] / max(cw - 1, 1)
    cb = 0.5 + 0.2 * (xx - 0.5) * 2 * torch.cos(2 * math.pi * (yy + frame / 131.0)) + 0.05 * _smooth_noise(ch, cw, 8, g, device)
    cr = 0.5 + 0.2 * (yy - 0.5) * 2 * torch.sin(2 * math.pi * (xx + frame / 171.0)) + 0.05 * _smooth_noise(ch, cw, 8, g, device)
    cb, cr = cb.clamp(0, 1), cr.clamp(0, 1)
    q = 4.0 / 219.0
    lum_d = _distort(lum, g, device, 1.5 / 255.0, q)
    cb_d = _distort(cb, g, device, 0.75 / 255.0, q)
    cr_d = _distort(cr, g, device, 0.75 / 255.0, q)
    pitch, coded_h, _ = yuv420_geometry(w, h, bits)
    return (_pack_yuv(lum, cb, cr, w, h, bits, device), _pack_yuv(lum_d, cb_d, cr_d, w, h, bits, device), pitch, coded_h)


def yuv_geometry(w: int, h: int, bits: int, sub: str):
    """yuv420_geometry for sub = "420", "422" or "444": (pitch, coded_height, total bytes) of an NVDEC-like surface."""
    pitch, coded_h, total = yuv420_geometry(w, h, bits)
    if sub == "420":
        return pitch, coded_h, total
    return pitch, coded_h, pitch * coded_h * (2 if sub == "422" else 3)


def quantize_yuv(yv, cb, cr, bits: int):
    """[0,1] floats -> limited-range integer samples: 8-bit codes, or 10-bit codes in the high bits of u16 (int32 tensors)."""
    if bits == 8:
        return (torch.round(16 + 219 * yv).clamp(0, 255).to(torch.int32),
                torch.round(128 + 224 * (cb - 0.5)).clamp(0, 255).to(torch.int32),
                torch.round(128 + 224 * (cr - 0.5)).clamp(0, 255).to(torch.int32))
    return (torch.round(64 + 876 * yv).clamp(0, 1023).to(torch.int32) << 6,
            torch.round(512 + 896 * (cb - 0.5)).clamp(0, 1023).to(torch.int32) << 6,
            torch.round(512 + 896 * (cr - 0.5)).clamp(0, 1023).to(torch.int32) << 6)


def pack_yuv_samples(yq, cbq, crq, w: int, h: int, bits: int, sub: str, pitch: int, coded_h: int, device="cpu"):
    """Integer samples -> NVDEC-like surface (1-D uint8): Y (h, w); Cb / Cr (h, ceil(w/2)) for "422", (h, w) for "444".
    4:2:2: interleaved CbCr plane at pitch*coded_h; 4:4:4: Cb plane there, Cr plane at 2*pitch*coded_h."""
    bps = 1 if bits == 8 else 2
    n = pitch * coded_h * (2 if sub == "422" else 3) // bps
    buf = torch.zeros(n, dtype=torch.int32, device=device)
    p = pitch // bps
    plane = p * coded_h
    buf[: p * h].view(h, p)[:, :w] = yq
    if sub == "422":
        cw = (w + 1) // 2
        uv = buf[plane: plane + p * h].view(h, p)
        uv[:, 0:2 * cw:2] = cbq
        uv[:, 1:2 * cw:2] = crq
    else:
        buf[plane: plane + p * h].view(h, p)[:, :w] = cbq
        buf[2 * plane: 2 * plane + p * h].view(h, p)[:, :w] = crq
    if bits == 8:
        return buf.to(torch.uint8)
    lo = (buf & 0xFF).to(torch.uint8)
    hi = ((buf >> 8) & 0xFF).to(torch.uint8)
    return torch.stack([lo, hi], dim=1).reshape(-1).contiguous()


def make_pair_yuv(w: int, h: int, bits: int = 8, sub: str = "444", frame: int = 0, seed: int = 1, device="cpu"):
    """make_pair_yuv420's content with chroma at 4:2:2 ("422": ceil(w/2) x h) or 4:4:4 ("444": w x h) resolution.
    -> (ref_buf, dis_buf, pitch, coded_height); buffers are 1-D uint8 tensors on `device` (NV16 / P216 / YUV444 / YUV444P16)."""
    assert sub in ("422", "444")
    g = _gen(seed, frame, device)
    ch, cw = h, (w + 1) // 2 if sub == "422" else w
    lum = _base_luma(h, w, frame, g, device)
    yy = torch.arange(ch, device=device, dtype=torch.float32)[:, None] / max(ch - 1, 1)
    xx = torch.arange(cw, device=device, dtype=torch.float32)[None, :] / max(cw - 1, 1)
    cb = 0.5 + 0.2 * (xx - 0.5) * 2 * torch.cos(2 * math.pi * (yy + frame / 131.0)) + 0.05 * _smooth_noise(ch, cw, 8, g, device)
    cr = 0.5 + 0.2 * (yy - 0.5) * 2 * torch.sin(2 * math.pi * (xx + frame / 171.0)) + 0.05 * _smooth_noise(ch, cw, 8, g, device)
    cb, cr = cb.clamp(0, 1), cr.clamp(0, 1)
    q = 4.0 / 219.0
    lum_d = _distort(lum, g, device, 1.5 / 255.0, q)
    cb_d = _distort(cb, g, device, 0.75 / 255.0, q)
    cr_d = _distort(cr, g, device, 0.75 / 255.0, q)
    pitch, coded_h, _ = yuv_geometry(w, h, bits, sub)
    ref = pack_yuv_samples(*quantize_yuv(lum, cb, cr, bits), w, h, bits, sub, pitch, coded_h, device)
    dis = pack_yuv_samples(*quantize_yuv(lum_d, cb_d, cr_d, bits), w, h, bits, sub, pitch, coded_h, device)
    return ref, dis, pitch, coded_h


def make_pair_srgb8(w: int, h: int, frame: int = 0, seed: int = 1, device="cpu"):
    """-> (ref, dis): uint8 tensors (H, W, 3), contiguous (pitch = 3*W)."""
    g = _gen(seed, frame, device)
    chans, chans_d = [], []
    for c in range(3):
        p = _base_luma(h, w, frame, g, device, phase=0.17 * c)
        chans.append(p)
        chans_d.append(_distort(p, g, device, 1.5 / 255.0, 4.0 / 255.0))
    ref = torch.round(torch.stack(chans, dim=-1) * 255).clamp(0, 255).to(torch.uint8).contiguous()
    dis = torch.round(torch.stack(chans_d, dim=-1) * 255).clamp(0, 255).to(torch.uint8).contiguous()
    return ref, dis


def make_pair_linearf32(w: int, h: int, frame: int = 0, seed: int = 1, device="cpu"):
    """-> (ref, dis): float32 tensors (H, W, 3) of linear RGB in [0,1]."""
    g = _gen(seed, frame, device)
    chans, chans_d = [], []
    for c in range(3):
        p = _base_luma(h, w, frame, g, device, phase=0.17 * c)
        chans.append(p * p)
        d = _distort(p, g, device, 1.5 / 255.0, 4.0 / 255.0)
        chans_d.append(d * d)
    return torch.stack(chans, dim=-1).contiguous(), torch.stack(chans_d, dim=-1).contiguous()


# sample planes of each format (make_pair_scaled): (sample dtype, chroma subsampling or "rgb")
SCALED_FORMATS = {"NV12": ("u8", "420"), "P016": ("u16", "420"), "NV16": ("u8", "422"), "P216": ("u16", "422"),
                  "YUV444": ("u8", "444"), "YUV444P16": ("u16", "444"), "SRGB8": ("u8", "rgb"), "SRGB16": ("u16", "rgb"),
                  "SRGBF32": ("f32", "rgb"), "LINEARF32": ("f32", "rgb")}


def _area(p, h, w):
    """Area-downscale a float plane (H, W) to (h, w) (the identity when the size is unchanged)."""
    if tuple(p.shape) == (h, w):
        return p
    return F.interpolate(p[None, None], size=(h, w), mode="area")[0, 0]


def make_pair_scaled(fmt: str, w: int, h: int, dis_w: int, dis_h: int, frame: int = 0, seed: int = 1):
    """A seeded (reference, lower-resolution distorted) pair of format `fmt` (a SCALED_FORMATS name): the reference content
    at w x h, the distorted frame its area-downscale to dis_w x dis_h (each plane on its own grid) with the distortion of
    the other generators applied.  -> (ref_planes, dis_planes): lists of numpy sample arrays, one per plane, with
    interleaved channels side by side in a row -- YUV 4:2:0 / 4:2:2: [Y (h, w), CbCr (chroma rows, 2 * ceil(w / 2))];
    4:4:4: [Y, Cb, Cr]; packed RGB: [(h, 3 * w)].  8-bit YUV is limited range, 16-bit YUV 10-bit codes in the high bits."""
    dt, sub = SCALED_FORMATS[fmt]
    g = _gen(seed, frame, "cpu")
    q = 4.0 / 219.0
    if sub == "rgb":
        ref, dis = [], []
        for c in range(3):
            p = _base_luma(h, w, frame, g, "cpu", phase=0.17 * c)
            d = _distort(_area(p, dis_h, dis_w), g, "cpu", 1.5 / 255.0, 4.0 / 255.0)
            ref.append(p)
            dis.append(d)

        def pack(chans):
            x = torch.stack(chans, dim=-1)
            if fmt == "LINEARF32":
                x = x * x
            if dt == "f32":
                x = x.float()
            else:
                x = torch.round(x * (255 if dt == "u8" else 65535)).clamp(0, 255 if dt == "u8" else 65535).to(torch.int32)
            return [x.reshape(x.shape[0], -1).numpy().astype({"u8": "uint8", "u16": "uint16", "f32": "float32"}[dt])]
        return pack(ref), pack(dis)
    bits = 8 if dt == "u8" else 16

    def grid(ww, hh):
        return ((hh + 1) // 2 if sub == "420" else hh), ((ww + 1) // 2 if sub != "444" else ww)
    ch, cw = grid(w, h)
    dch, dcw = grid(dis_w, dis_h)
    lum = _base_luma(h, w, frame, g, "cpu")
    yy = torch.arange(ch, dtype=torch.float32)[:, None] / max(ch - 1, 1)
    xx = torch.arange(cw, dtype=torch.float32)[None, :] / max(cw - 1, 1)
    cb = (0.5 + 0.2 * (xx - 0.5) * 2 * torch.cos(2 * math.pi * (yy + frame / 131.0)) + 0.05 * _smooth_noise(ch, cw, 8, g, "cpu")).clamp(0, 1)
    cr = (0.5 + 0.2 * (yy - 0.5) * 2 * torch.sin(2 * math.pi * (xx + frame / 171.0)) + 0.05 * _smooth_noise(ch, cw, 8, g, "cpu")).clamp(0, 1)
    lum_d = _distort(_area(lum, dis_h, dis_w), g, "cpu", 1.5 / 255.0, q)
    cb_d = _distort(_area(cb, dch, dcw), g, "cpu", 0.75 / 255.0, q)
    cr_d = _distort(_area(cr, dch, dcw), g, "cpu", 0.75 / 255.0, q)
    npdt = "uint8" if bits == 8 else "uint16"

    def pack(yv, u, v):
        yq, uq, vq = (t.numpy().astype(npdt) for t in quantize_yuv(yv, u, v, bits))
        if sub == "444":
            return [yq, uq, vq]
        import numpy as np
        uv = np.zeros((uq.shape[0], 2 * uq.shape[1]), npdt)
        uv[:, 0::2], uv[:, 1::2] = uq, vq
        return [yq, uv]
    return pack(lum, cb, cr), pack(lum_d, cb_d, cr_d)


def compact_planes(planes):
    """Sample planes (make_pair_scaled's form) -> (buf: 1-D numpy uint8 array, pitch, plane1 offset or 0): the compact layout
    of a scaled handle's staged frames (pitch = the longest row rounded up to 256 bytes, plane i at i * pitch * h; 4:4:4 Cr at
    plane[1] + (plane[1] - plane[0]))."""
    import numpy as np
    h = planes[0].shape[0]
    pitch = (max(p.shape[1] * p.itemsize for p in planes) + 255) // 256 * 256
    buf = np.zeros(pitch * h * len(planes), np.uint8)
    for i, p in enumerate(planes):
        rows = np.ascontiguousarray(p).view(np.uint8).reshape(p.shape[0], -1)
        buf[i * pitch * h: i * pitch * h + p.shape[0] * pitch].reshape(p.shape[0], pitch)[:, :rows.shape[1]] = rows
    return buf, pitch, (pitch * h if len(planes) > 1 else 0)
