"""Frame layouts: padded, misaligned, split and very large frames against the oracle, bit for bit.

The front-end (k_frontend2) is the only kernel that reads the caller's memory, and it picks its code path per 32x32 region
from the frame's addresses and pitch.  Whatever the layout, the XYB planes must be the oracle's bits and the score and norms
those of the compact layout: the oracle always gets the logical image (a contiguous copy, or the canonical NVDEC buffer).
"One sample" is one channel value: 1 byte for NV12 and sRGB8, 2 for P016 and sRGB16, 4 for sRGB f32 and linear f32.

Layouts (L0-L3 for every format, L4* for NV12 / P016 only):
  L0        compact; NVDEC geometry for YUV (pitch rounded up to 256, chroma at pitch * coded_height)
  L1        pitch padded to a multiple of 512 (keeps the fast path)
  L2        pitch = row bytes + one sample (no fast path; an odd NV12 pitch, a P016 pitch of 2 mod 4)
  L3        plane[0] (and plane[1]) one sample past an aligned base
  L4sep     chroma in a separate allocation
  L4before  chroma placed before luma
  L4coded   coded_height == height
"""
import ctypes as C
from dataclasses import dataclass
from typing import List, Optional, Tuple

import numpy as np
import pytest

OK, E_INVALID = 0, -1
FORMATS = ["NV12", "P016", "SRGB8", "SRGB16", "SRGBF32", "LINEARF32"]
SAMPLE = {"NV12": 1, "P016": 2, "SRGB8": 1, "SRGB16": 2, "SRGBF32": 4, "LINEARF32": 4}
PACKED_LAYOUTS = ["L0", "L1", "L2", "L3"]
YUV_LAYOUTS = PACKED_LAYOUTS + ["L4sep", "L4before", "L4coded"]
SIZES = [(200, 136), (203, 131)]   # interior regions with ragged right / bottom edges; odd sizes (4:2:0 included)


def _up(x, m):
    return (x + m - 1) // m * m


def _is_yuv(fmt):
    return fmt in ("NV12", "P016")


def _layouts(fmt):
    return YUV_LAYOUTS if _is_yuv(fmt) else PACKED_LAYOUTS


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


@dataclass
class Content:
    """The logical image of one side: its planes as rows of bytes, and the oracle's linear planes (3, H, W)."""
    fmt: str
    w: int
    h: int
    planes: List[np.ndarray]           # packed: [(H, 3 W s)]; YUV: [luma (H, W s), chroma (ceil(H/2), 2 ceil(W/2) s)]
    lin: np.ndarray
    img: Optional[np.ndarray] = None   # packed formats: the typed (H, W, 3) image


def _content(oracle, fmt, w, h, side, frame=1, seed=3):
    from turbo_metrics_b200 import synth
    s = SAMPLE[fmt]
    if _is_yuv(fmt):
        bits = 8 if fmt == "NV12" else 16
        rb, db, pitch, ch = synth.make_pair_yuv420(w, h, bits, frame=frame, seed=seed)
        buf = (rb if side == 0 else db).numpy()
        y = buf[: pitch * h].reshape(h, pitch)[:, : w * s]
        chh = (h + 1) // 2
        uv = buf[pitch * ch: pitch * (ch + chh)].reshape(chh, pitch)[:, : (w + 1) // 2 * 2 * s]
        return Content(fmt, w, h, [np.ascontiguousarray(y), np.ascontiguousarray(uv)],
                       oracle.linear_from_yuv420(buf, pitch, ch, w, h, bits))
    if fmt == "LINEARF32":
        img = synth.make_pair_linearf32(w, h, frame=frame, seed=seed)[side].numpy()
        lin = oracle.linear_from_linearf32(img)
    else:
        x = synth.make_pair_srgb8(w, h, frame=frame, seed=seed)[side].numpy()
        if fmt == "SRGB8":
            img = x
            lin = oracle.linear_from_srgb8(img)
        elif fmt == "SRGB16":
            img = np.clip(x.astype(np.int32) * 257 + 5, 0, 65535).astype(np.uint16)
            lin = oracle.linear_from_srgb16(img)
        else:
            img = x.astype(np.float32) / np.float32(255.0)
            lin = oracle.linear_from_srgbf32(img)
    img = np.ascontiguousarray(img)
    return Content(fmt, w, h, [img.view(np.uint8).reshape(h, -1)], lin, img)


@dataclass
class Placed:
    """A frame laid out in byte buffers: plane addresses as (buffer, offset), the pitch, and (host frames) the bytes from
    plane[0] to the end of its last row."""
    buffers: List[np.ndarray]
    p0: Tuple[int, int]
    p1: Optional[Tuple[int, int]]
    pitch: int
    span: int


def _put_rows(buf, off, pitch, rows):
    for i in range(rows.shape[0]):
        buf[off + i * pitch: off + i * pitch + rows.shape[1]] = rows[i]


def _place(c: Content, layout: str) -> Placed:
    s, h = SAMPLE[c.fmt], c.h
    if not _is_yuv(c.fmt):
        rows = c.planes[0]
        row = rows.shape[1]
        pitch = {"L0": row, "L1": _up(row, 512), "L2": row + s, "L3": row}[layout]
        off = s if layout == "L3" else 0
        buf = np.zeros(_up(off + pitch * h, 512), np.uint8)
        _put_rows(buf, off, pitch, rows)
        return Placed([buf], (0, off), None, pitch, (h - 1) * pitch + row)
    y, uv = c.planes
    ry, rc, chh = y.shape[1], uv.shape[1], uv.shape[0]
    nv_pitch, coded = _up(ry, 256), _up(h, 16)
    if layout == "L1":
        pitch = _up(max(ry, rc), 512)
    elif layout == "L2":
        pitch = max(ry + s, rc)
    else:
        pitch = nv_pitch
    o0, o1 = 0, pitch * coded                     # L0, L3 (shifted below)
    if layout in ("L1", "L2", "L4coded"):
        o1 = pitch * h
    elif layout == "L4before":
        o0, o1 = pitch * chh, 0
    elif layout == "L3":
        o0, o1 = s, s + pitch * coded
    if layout == "L4sep":
        ybuf, cbuf = np.zeros(_up(pitch * h, 512), np.uint8), np.zeros(_up(pitch * chh, 512), np.uint8)
        _put_rows(ybuf, 0, pitch, y)
        _put_rows(cbuf, 0, pitch, uv)
        return Placed([ybuf, cbuf], (0, 0), (1, 0), pitch, 0)
    end_y, end_c = o0 + (h - 1) * pitch + ry, o1 + (chh - 1) * pitch + rc
    buf = np.zeros(_up(max(end_y, end_c), 512), np.uint8)
    _put_rows(buf, o0, pitch, y)
    _put_rows(buf, o1, pitch, uv)
    return Placed([buf], (0, o0), (0, o1), pitch, max(end_y, end_c) - o0)


def _frame(p: Placed, where="cuda"):
    """-> DeviceFrame over the placed buffers: "cuda" (device), "pinned" / "pageable" (torch host), "numpy" (host)."""
    import torch
    import turbo_metrics_b200 as tm
    if where == "numpy":
        keep = [b.copy() for b in p.buffers]
        addr = [b.ctypes.data for b in keep]
    else:
        keep = [torch.from_numpy(b.copy()) for b in p.buffers]
        if where == "cuda":
            keep = [t.cuda() for t in keep]
        elif where == "pinned":
            keep = [t.pin_memory() for t in keep]
        addr = [t.data_ptr() for t in keep]
    p1 = addr[p.p1[0]] + p.p1[1] if p.p1 else 0
    return tm.DeviceFrame(addr[p.p0[0]] + p.p0[1], p1, p.pitch, keep, p.span)


def _oracle_xyb(oracle, ref_lin, dis_lin, nscales):
    """XYB planes of every scale (reference then distorted), as _oracle_stages of test_gpu_parity.py builds them."""
    out, a, b = [], ref_lin, dis_lin
    for s in range(nscales):
        if s > 0:
            a, b = oracle.downscale_by_2(a), oracle.downscale_by_2(b)
        out.append(np.concatenate([oracle.linear_to_xyb(a), oracle.linear_to_xyb(b)], axis=0))
    return out


def _fmt(name):
    import turbo_metrics_b200 as tm
    return tm.PixelFormat[name]


def _run(m, a, b):
    """Score one pair on a batch=1, ring=1 handle: (score, norms or None, XYB planes of every scale or None)."""
    t = m.compute(a, b)
    score = m.get_score(t)
    info = m.info()
    norms = None if info.flags & 1 else m.get_norms(t)
    planes = [m.debug_read(t, 0, s) for s in range(info.nscales)] if info.pipeline == 1 else None
    return score, norms, planes


@pytest.fixture(scope="module")
def lib22():
    """ABI 2.2 or later: an older library accepts frames whose loads it cannot align (it would fault on them)."""
    from turbo_metrics_b200 import _lib
    v = _lib.lib().ssimu2_version()
    assert v >= (2 << 16) | 2, f"library ABI {v >> 16}.{v & 0xffff} predates the frame layout rule"
    return _lib


# ------------------------------------------------------------------------------------------ G: CPU only
@pytest.mark.parametrize("dtype", ["uint8", "uint16", "float32"])
def test_packed_frame_reports_the_span_of_padded_views(dtype):
    import torch
    import turbo_metrics_b200 as tm
    h, w, wide = 64, 40, 100
    big = np.zeros((h, wide, 3), dtype)
    es = big.itemsize
    span = (h - 1) * wide * 3 * es + w * 3 * es
    for img in (big[:, :w], torch.from_numpy(big)[:, :w], big[3:, 5:5 + w]):
        f = tm.DeviceFrame.packed(img)
        assert f.pitch == wide * 3 * es
        assert f.nbytes == (img.shape[0] - 1) * wide * 3 * es + w * 3 * es
    assert tm.DeviceFrame.packed(big[:, :w]).nbytes == span          # (64, 40, 3) of (64, 100, 3) u8: 19020, not 7680
    for img in (big, torch.from_numpy(big)):                         # contiguous: the span is the whole image
        assert tm.DeviceFrame.packed(img).nbytes == h * wide * 3 * es
    rows = torch.zeros((h, wide * 3), dtype=getattr(torch, dtype))   # (H, 3 W) rows of samples
    assert tm.DeviceFrame.packed(rows).nbytes == h * wide * 3 * es
    assert tm.DeviceFrame.packed(rows[:, : w * 3]).nbytes == span


def test_packed_frame_rejects_views_whose_pixels_are_not_packed():
    import torch
    import turbo_metrics_b200 as tm
    big = np.zeros((64, 100, 3), np.uint8)
    bad = [big[:, ::2], big[:, :, ::-1], big[:, :, :2], big.transpose(1, 0, 2), np.zeros((64, 100, 4), np.uint8)[:, :, :3],
           torch.from_numpy(big)[:, ::2], torch.from_numpy(big).permute(1, 0, 2), torch.zeros((64, 300))[:, ::3],
           np.zeros((64, 100, 3, 1), np.uint8)]
    for img in bad:
        with pytest.raises(ValueError):
            tm.DeviceFrame.packed(img)


def test_yuv420_frame_is_unchanged():
    import torch
    import turbo_metrics_b200 as tm
    for buf in (torch.zeros(1000, dtype=torch.uint8), np.zeros(1000, np.uint8)):
        f = tm.DeviceFrame.yuv420(buf, 32, 20)
        base = buf.data_ptr() if hasattr(buf, "data_ptr") else buf.ctypes.data
        assert (f.plane0, f.plane1, f.pitch, f.nbytes) == (base, base + 32 * 20, 32, 1000) and f.keepalive is buf


def test_placed_layouts_hold_the_logical_image():
    """The layouts the GPU tests use: every one holds the same rows, with the pitch and plane offsets it names."""
    for fmt in FORMATS:
        s = SAMPLE[fmt]
        for w, h in SIZES:
            rng = np.random.default_rng(1)
            if _is_yuv(fmt):
                planes = [rng.integers(0, 256, (h, w * s), dtype=np.uint8),
                          rng.integers(0, 256, ((h + 1) // 2, (w + 1) // 2 * 2 * s), dtype=np.uint8)]
            else:
                planes = [rng.integers(0, 256, (h, 3 * w * s), dtype=np.uint8)]
            c = Content(fmt, w, h, planes, None)
            for lay in _layouts(fmt):
                p = _place(c, lay)
                row = planes[0].shape[1]
                if lay == "L2":
                    assert p.pitch == max(row + s, planes[-1].shape[1])
                if lay == "L1":
                    assert p.pitch % 512 == 0
                for (bi, off), rows in zip([p.p0] + ([p.p1] if p.p1 else []), planes):
                    got = np.stack([p.buffers[bi][off + i * p.pitch: off + i * p.pitch + rows.shape[1]] for i in range(rows.shape[0])])
                    assert np.array_equal(got, rows), (fmt, w, h, lay)
                if lay == "L3":
                    assert p.p0[1] == s
            if fmt in ("NV12", "P016") and w == 200:   # odd NV12 pitch, P016 pitch of 2 mod 4
                assert _place(c, "L2").pitch % (2 * s) == s


# ------------------------------------------------------------------------------------------ A: layout matrix
pytest_gpu = pytest.mark.gpu


@pytest_gpu
@pytest.mark.parametrize("w,h", SIZES)
@pytest.mark.parametrize("fmt", FORMATS)
def test_layouts_give_the_oracle_planes_and_the_compact_score(lib22, oracle, fmt, w, h):
    """(a) split pipeline: the XYB planes of every scale are the oracle's bits; (b) default pipeline: score and all 108 norms are
    bit-equal to the compact layout's.  The two frames of a pair have different layouts, so both images of one two-side warp
    take different paths."""
    import turbo_metrics_b200 as tm
    ref, dis = _content(oracle, fmt, w, h, 0), _content(oracle, fmt, w, h, 1)
    lays = _layouts(fmt)
    pairs = [(lays[i], lays[(i + 1) % len(lays)]) for i in range(len(lays))] + [("L0", "L0")]
    with tm.Ssimulacra2(w, h, _fmt(fmt), batch=1, ring=1, pipeline="split") as m:
        want = _oracle_xyb(oracle, ref.lin, dis.lin, m.info().nscales)
        for la, lb in pairs:
            _, _, planes = _run(m, _frame(_place(ref, la)), _frame(_place(dis, lb)))
            for s, (got, exp) in enumerate(zip(planes, want)):
                assert np.array_equal(_bits(got), _bits(exp)), f"{la}/{lb}: XYB planes differ at scale {s}"
    with tm.Ssimulacra2(w, h, _fmt(fmt), batch=1, ring=1) as m:
        s0, n0, _ = _run(m, _frame(_place(ref, "L0")), _frame(_place(dis, "L0")))
        for la, lb in pairs:
            score, norms, _ = _run(m, _frame(_place(ref, la)), _frame(_place(dis, lb)))
            assert score == s0 and np.array_equal(norms, n0), (la, lb, score, s0)
    so, no, _ = oracle.ssimu2_linear_planar(ref.lin, dis.lin)
    assert abs(s0 - so) <= 0.01


# ------------------------------------------------------------------------------------------ B: paths mixed in one launch
@pytest_gpu
@pytest.mark.parametrize("group", [0, 3])
@pytest.mark.parametrize("fmt", FORMATS)
def test_one_batch_of_pairs_in_different_layouts(lib22, oracle, fmt, group):
    import turbo_metrics_b200 as tm
    w, h = 200, 136
    ref, dis = _content(oracle, fmt, w, h, 0), _content(oracle, fmt, w, h, 1)
    lays = _layouts(fmt)
    with tm.Ssimulacra2(w, h, _fmt(fmt), batch=8, ring=2, input_group=group) as m:
        s0 = m.compute_sync(_frame(_place(ref, "L0")), _frame(_place(dis, "L0")))
        refs = [_frame(_place(ref, lays[i % len(lays)])) for i in range(8)]
        diss = [_frame(_place(dis, lays[(i + 3) % len(lays)])) for i in range(8)]
        ts = m.compute_batch(refs, diss)
        got = m.get_scores(ts)
    assert np.all(got == s0), (got, s0)


# ------------------------------------------------------------------------------------------ C: one-side front-ends
@pytest_gpu
@pytest.mark.parametrize("ref_fmt,ref_lay,dis_fmt,dis_lay", [("NV12", "L2", "LINEARF32", "L3"), ("SRGB16", "L2", "P016", "L4sep")])
def test_mixed_handle_layouts(lib22, oracle, ref_fmt, ref_lay, dis_fmt, dis_lay):
    """k_frontend2<FMT, kF2Ref / kF2Dis>: each side's planes are the oracle's, and the score is the compact layouts' on the same
    mixed handle."""
    import turbo_metrics_b200 as tm
    w, h = 200, 136
    ref, dis = _content(oracle, ref_fmt, w, h, 0), _content(oracle, dis_fmt, w, h, 1)
    with tm.Ssimulacra2(w, h, _fmt(ref_fmt), dis_fmt=_fmt(dis_fmt), batch=1, ring=1, pipeline="split") as m:
        assert m.mixed
        want = _oracle_xyb(oracle, ref.lin, dis.lin, m.info().nscales)
        s0, n0, p0 = _run(m, _frame(_place(ref, "L0")), _frame(_place(dis, "L0")))
        s1, n1, p1 = _run(m, _frame(_place(ref, ref_lay)), _frame(_place(dis, dis_lay)))
    for s, (exp, a, b) in enumerate(zip(want, p0, p1)):
        assert np.array_equal(_bits(a[:3]), _bits(exp[:3])) and np.array_equal(_bits(a[3:]), _bits(exp[3:])), f"compact, scale {s}"
        assert np.array_equal(_bits(b[:3]), _bits(exp[:3])), f"reference side ({ref_fmt} {ref_lay}) differs at scale {s}"
        assert np.array_equal(_bits(b[3:]), _bits(exp[3:])), f"distorted side ({dis_fmt} {dis_lay}) differs at scale {s}"
    assert s1 == s0 and np.array_equal(n1, n0)


# ------------------------------------------------------------------------------------------ D: offsets beyond 4 GiB
@pytest_gpu
@pytest.mark.parametrize("fmt", ["LINEARF32", "SRGB16", "P016"])
def test_rows_beyond_4gib(oracle, fmt):
    """Both frames of a pair side by side in the rows of one buffer whose pitch keeps the fast path (a multiple of 16): the
    interior region of rows 64-95 straddles the 4 GiB offset, the one of rows 96-127 lies wholly beyond it (for P016 the chroma
    rows sit in the lower half of the buffer, beyond it too).  Planes and score must be the compact copy's bits.
    About 6.8 GB of device memory per case (computed from the pitch, not measured).  Every read stays inside the buffer, so
    this test runs on any library version."""
    import torch
    import turbo_metrics_b200 as tm
    w, h = 192, 136
    pitch = (48 << 20) + 4608
    assert pitch % 16 == 0 and 64 * pitch < (1 << 32) < 95 * pitch and 96 * pitch > (1 << 32)
    ref, dis = _content(oracle, fmt, w, h, 0), _content(oracle, fmt, w, h, 1)
    col = _up(max(p.shape[1] for p in ref.planes), 16)
    chroma_row0 = h // 2
    if torch.cuda.mem_get_info()[0] < pitch * h + (1 << 30):
        pytest.skip("needs about 7 GB of free device memory")
    with tm.Ssimulacra2(w, h, _fmt(fmt), batch=1, ring=1, pipeline="split") as m:
        s0, n0, p0 = _run(m, _frame(_place(ref, "L0")), _frame(_place(dis, "L0")))
        buf = torch.zeros(pitch * h, dtype=torch.uint8, device="cuda")
        rows = buf.view(h, pitch)
        frames = []
        for side, c in enumerate((ref, dis)):
            rows[:, side * col: side * col + c.planes[0].shape[1]] = torch.from_numpy(c.planes[0]).cuda()
            p1 = 0
            if _is_yuv(fmt):
                uv = c.planes[1]
                x1 = (2 + side) * col
                rows[chroma_row0: chroma_row0 + uv.shape[0], x1: x1 + uv.shape[1]] = torch.from_numpy(uv).cuda()
                p1 = buf.data_ptr() + chroma_row0 * pitch + x1
                assert (chroma_row0 + 48) * pitch > (1 << 32)
            frames.append(tm.DeviceFrame(buf.data_ptr() + side * col, p1, pitch, buf, 0))
        s1, n1, p1s = _run(m, frames[0], frames[1])
        del rows, buf, frames
        torch.cuda.empty_cache()
    for s, (a, b) in enumerate(zip(p0, p1s)):
        assert np.array_equal(_bits(a), _bits(b)), f"XYB planes differ at scale {s}"
    assert s1 == s0 and np.array_equal(n1, n0)


# ------------------------------------------------------------------------------------------ E: host frames
@pytest_gpu
@pytest.mark.parametrize("fmt", ["SRGB8", "LINEARF32"])
def test_padded_host_views(lib22, oracle, fmt):
    """Cropped host images (img[:, :w] of a wider image) through compute_from_cpu and compute_from_cpu_batch: torch pinned,
    torch pageable and numpy.  The library copies `nbytes` from plane[0], so that must be the span of the view."""
    import torch
    import turbo_metrics_b200 as tm
    w, h, wide = 200, 136, 237
    ref, dis = _content(oracle, fmt, w, h, 0), _content(oracle, fmt, w, h, 1)
    bigs = []
    for c in (ref, dis):
        big = np.zeros((h, wide, 3), c.img.dtype)
        big[:, :w] = c.img
        bigs.append(big)
    es = ref.img.itemsize
    span = (h - 1) * wide * 3 * es + w * 3 * es
    assert tm.DeviceFrame.packed(bigs[0][:, :w]).nbytes == span
    views = {"numpy": [b[:, :w] for b in bigs], "pageable": [torch.from_numpy(b)[:, :w] for b in bigs],
             "pinned": [torch.from_numpy(b).pin_memory()[:, :w] for b in bigs]}
    assert views["pinned"][0].is_pinned() and not views["pageable"][0].is_pinned()
    with tm.Ssimulacra2(w, h, _fmt(fmt), batch=4, ring=2) as m:
        s0 = m.compute_sync(_frame(_place(ref, "L0")), _frame(_place(dis, "L0")))
        for kind, (rv, dv) in views.items():
            a, b = tm.DeviceFrame.packed(rv), tm.DeviceFrame.packed(dv)
            assert a.nbytes == span and a.pitch == wide * 3 * es
            assert m.get_score(m.compute_from_cpu(a, b)) == s0, kind
            got = m.get_scores(m.compute_from_cpu_batch([a] * 3, [b] * 3))
            assert np.all(got == s0), (kind, got, s0)


@pytest_gpu
@pytest.mark.parametrize("fmt,lay", [("NV12", "L2"), ("P016", "L2"), ("P016", "L4coded"), ("NV12", "L1")])
def test_yuv_host_frames_with_chroma_elsewhere(lib22, oracle, fmt, lay):
    import turbo_metrics_b200 as tm
    w, h = 200, 136
    ref, dis = _content(oracle, fmt, w, h, 0), _content(oracle, fmt, w, h, 1)
    with tm.Ssimulacra2(w, h, _fmt(fmt), batch=2, ring=2) as m:
        s0 = m.compute_sync(_frame(_place(ref, "L0")), _frame(_place(dis, "L0")))
        a, b = _frame(_place(ref, lay), "numpy"), _frame(_place(dis, lay), "numpy")
        assert a.plane1 - a.plane0 != a.pitch * _up(h, 16) and a.nbytes == b.nbytes
        assert m.get_score(m.compute_from_cpu(a, b)) == s0


@pytest_gpu
def test_sized_host_frames_on_a_mixed_handle(lib22, oracle):
    """An NV12 reference with an odd pitch against a cropped sRGB16 view, each copied with its own byte count."""
    import torch
    import turbo_metrics_b200 as tm
    w, h = 200, 136
    ref, dis = _content(oracle, "NV12", w, h, 0), _content(oracle, "SRGB16", w, h, 1)
    big = np.zeros((h, w + 9, 3), np.uint16)
    big[:, :w] = dis.img
    with tm.Ssimulacra2(w, h, tm.PixelFormat.NV12, dis_fmt=tm.PixelFormat.SRGB16, batch=2, ring=2) as m:
        s0 = m.compute_sync(_frame(_place(ref, "L0")), _frame(_place(dis, "L0")))
        a, b = _frame(_place(ref, "L2"), "numpy"), tm.DeviceFrame.packed(torch.from_numpy(big)[:, :w])
        assert a.pitch % 2 == 1 and b.nbytes == (h - 1) * (w + 9) * 6 + w * 6
        assert m.get_score(m.compute_from_cpu(a, b)) == s0
        ts = m.compute_from_cpu_batch([a] * 2, [b] * 2)
        assert np.all(m.get_scores(ts) == s0)


# ------------------------------------------------------------------------------------------ F: rejection
def _cfg(fmt, w=64, h=64, **kw):
    from turbo_metrics_b200.ssimulacra2 import make_config
    return make_config(w, h, _fmt(fmt), batch=kw.pop("batch", 64), ring=1, input_group=0, **kw)


class _Good:
    """A device and a host buffer, and a frame layout over them that every entry point accepts (64x64 frames)."""

    def __init__(self, fmt, w=64, h=64):
        import torch
        self.fmt, self.s, self.yuv = fmt, SAMPLE[fmt], _is_yuv(fmt)
        self.row = row = w * self.s * (1 if self.yuv else 3)
        self.pitch = _up(row, 256)
        self.chroma = self.pitch * h          # plane[1] - plane[0]
        self.size = self.pitch * (2 * h + 8)
        self.dev = torch.zeros(self.size, dtype=torch.uint8, device="cuda")
        self.host = np.zeros(self.size, np.uint8)
        self.span_luma = (h - 1) * self.pitch + row
        self.span = self.chroma + ((h + 1) // 2 - 1) * self.pitch + (w + 1) // 2 * 2 * self.s if self.yuv else self.span_luma

    def frame(self, host=False, d0=0, d1=0, dp=0):
        from turbo_metrics_b200 import _lib
        f = _lib.Frame()
        base = self.host.ctypes.data if host else self.dev.data_ptr()
        f.plane[0] = base + d0
        f.plane[1] = (base + d0 + self.chroma + d1) if self.yuv else 0
        f.pitch = self.pitch + dp
        return f


def _bad_frames(g: _Good):
    """-> [(what, device frame, host frame)] each off by less than one sample; empty for 1-byte samples."""
    if g.s == 1:
        return []
    d = g.s // 2
    out = [("pitch", g.frame(dp=d), g.frame(True, dp=d)), ("plane0", g.frame(d0=d), None)]
    if g.yuv:
        out.append(("plane1", g.frame(d1=d), g.frame(True, d1=d)))
    return out


@pytest_gpu
@pytest.mark.parametrize("fmt", FORMATS)
def test_frames_that_break_the_layout_rule_are_rejected(lib22, fmt):
    """Every entry point returns SSIMU2_E_INVALID for a frame whose plane address, chroma offset or pitch is not a multiple of
    one sample, and for host byte counts one short of the span.  The handle (batch 64, no input groups) is destroyed without a
    flush, wait or fetch, and ssimu2_destroy launches nothing: a frame the library wrongly accepted is never read."""
    lib = lib22.lib()
    g = _Good(fmt)
    h, sh = C.c_void_p(), C.c_void_p()
    t = C.c_uint64()
    assert lib.ssimu2_create(C.byref(h), C.byref(_cfg(fmt))) == OK
    devs = (C.c_int32 * 1)(0)
    assert lib.ssimu2_shard_create(C.byref(sh), C.byref(_cfg(fmt, batch=8)), devs, 1) == OK
    try:
        good, good_h = g.frame(), g.frame(True)
        for what, bad, bad_h in _bad_frames(g):
            for a, b in ((good, bad), (bad, good)):
                assert lib.ssimu2_submit(h, C.byref(a), C.byref(b), None, C.byref(t)) == E_INVALID, what
                assert lib.ssimu2_submit_batch(h, 1, C.byref(a), C.byref(b), None, C.byref(t)) == E_INVALID, what
                assert lib.ssimu2_shard_submit_device(sh, 1, C.byref(a), C.byref(b), None, C.byref(t)) == E_INVALID, what
            if bad_h is None:                  # host frames are staged to aligned memory: their address does not matter
                continue
            for a, b in ((good_h, bad_h), (bad_h, good_h)):
                assert lib.ssimu2_submit_host(h, C.byref(a), C.byref(b), g.size, C.byref(t)) == E_INVALID, what
                assert lib.ssimu2_submit_host_sized(h, 1, C.byref(a), g.size, C.byref(b), g.size, C.byref(t)) == E_INVALID, what
                assert lib.ssimu2_shard_submit_host(sh, 1, C.byref(a), C.byref(b), g.size, C.byref(t)) == E_INVALID, what
                assert lib.ssimu2_shard_submit_host_sized(sh, 1, C.byref(a), g.size, C.byref(b), g.size, C.byref(t)) == E_INVALID, what
        # host byte counts: one short of the span (packed: the last row; YUV: the last chroma row) is refused
        short = g.span - 1
        assert lib.ssimu2_submit_host(h, C.byref(good_h), C.byref(good_h), short, C.byref(t)) == E_INVALID
        assert lib.ssimu2_submit_host_sized(h, 1, C.byref(good_h), g.span, C.byref(good_h), short, C.byref(t)) == E_INVALID
        assert lib.ssimu2_submit_host_sized(h, 1, C.byref(good_h), short, C.byref(good_h), g.span, C.byref(t)) == E_INVALID
        assert lib.ssimu2_shard_submit_host(sh, 1, C.byref(good_h), C.byref(good_h), short, C.byref(t)) == E_INVALID
        assert lib.ssimu2_shard_submit_host_sized(sh, 1, C.byref(good_h), short, C.byref(good_h), g.span, C.byref(t)) == E_INVALID
        if g.yuv:                              # the luma rows alone are not enough
            assert g.span_luma < short
            assert lib.ssimu2_submit_host(h, C.byref(good_h), C.byref(good_h), g.span_luma, C.byref(t)) == E_INVALID
        # nothing was queued; exactly the span is accepted (queued, never launched)
        assert lib.ssimu2_submit_host(h, C.byref(good_h), C.byref(good_h), g.span, C.byref(t)) == OK and t.value == 0
        assert lib.ssimu2_submit_host_sized(h, 1, C.byref(good_h), g.span, C.byref(good_h), g.span, C.byref(t)) == OK
        assert t.value == 1
        # a bad pair at index 3 of 8: the whole call is refused and nothing is queued
        refs = (lib22.Frame * 8)(*[g.frame() for _ in range(8)])
        diss = (lib22.Frame * 8)(*[g.frame() for _ in range(8)])
        refs[3].pitch = g.row - 1 if g.s == 1 else g.pitch + g.s // 2   # a short row, or a misaligned pitch
        assert lib.ssimu2_submit_batch(h, 8, refs, diss, None, C.byref(t)) == E_INVALID
        refs_h = (lib22.Frame * 8)(*[g.frame(True) for _ in range(8)])
        diss_h = (lib22.Frame * 8)(*[g.frame(True) for _ in range(8)])
        diss_h[3].pitch = refs[3].pitch
        assert lib.ssimu2_submit_host_sized(h, 8, refs_h, g.size, diss_h, g.size, C.byref(t)) == E_INVALID
        assert lib.ssimu2_submit(h, C.byref(good), C.byref(good), None, C.byref(t)) == OK and t.value == 2
    finally:
        assert lib.ssimu2_destroy(h) == OK
        assert lib.ssimu2_shard_destroy(sh) == OK


@pytest_gpu
def test_a_shard_rejects_a_bad_frame_and_keeps_scoring(lib22, oracle):
    import turbo_metrics_b200 as tm
    w, h = 200, 136
    ref, dis = _content(oracle, "P016", w, h, 0), _content(oracle, "P016", w, h, 1)
    a, b = _frame(_place(ref, "L0"), "numpy"), _frame(_place(dis, "L0"), "numpy")
    bad = tm.DeviceFrame(a.plane0, a.plane1 + 1, a.pitch, a.keepalive, a.nbytes)
    with tm.Ssimulacra2(w, h, tm.PixelFormat.P016, batch=1, ring=1) as m:
        s0 = m.compute_sync(_frame(_place(ref, "L0")), _frame(_place(dis, "L0")))
    with tm.ShardedSsimulacra2(w, h, tm.PixelFormat.P016, [0], batch=2) as sh:
        with pytest.raises(tm.Ssimu2Error) as e:
            sh.submit_host([a, a, bad], [b, b, b])
        assert e.value.status == E_INVALID
        ts = sh.submit_host([a, a, a], [b, b, b])
        assert ts.start == 0                      # the refused call queued nothing
        sh.flush()
        assert np.all(sh.get_scores(ts) == s0)
