"""Scaled distorted frames (ssimu2_source.width / height): lower-resolution encodes scored against their source.

A scaled handle upscales each distorted frame in its own sample domain to the reference's size (k_resample: bicubic
Catmull-Rom, separable, centre-aligned, clamp-to-edge, f32 with a fixed fmaf chain, u8 / u16 rounded half to even and
clamped) and scores it like an ordinary frame of that format.  So every check compares a scaled handle, bit for bit, with an
unscaled handle scored on a CPU reference's upscale of the same frame (tests/native/resample_ref.c, built here), and for the
formats the oracle converts itself (NV12, P016, the packed RGB formats) also with the oracle's XYB planes.
"""
import ctypes as C
import os
import subprocess
import types

import numpy as np
import pytest

OK, E_INVALID, E_UNSUPPORTED, E_NODEVICE = 0, -1, -2, -4
FORMATS = ["NV12", "P016", "NV16", "P216", "YUV444", "YUV444P16", "SRGB8", "SRGB16", "SRGBF32", "LINEARF32"]
# (reference size, distorted size): 2x (4K from 1080p), 1.5x, fewer than 6 scales, one axis only
SCALES = [((3840, 2160), (1920, 1080)), ((1920, 1080), (1280, 720)), ((203, 131), (101, 67)), ((203, 131), (203, 67))]
SAMPLE = {"NV12": 1, "P016": 2, "NV16": 1, "P216": 2, "YUV444": 1, "YUV444P16": 2, "SRGB8": 1, "SRGB16": 2, "SRGBF32": 4,
          "LINEARF32": 4}
YUV = ("NV12", "P016", "NV16", "P216", "YUV444", "YUV444P16")
MATRICES = ["bt709", "bt601_525", "bt601_625"]


def _up(x, m):
    return (x + m - 1) // m * m


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _fmt(name):
    import turbo_metrics_b200 as tm
    return tm.PixelFormat[name]


# ------------------------------------------------------------------------------------------ the CPU reference resampler
_REF_C = os.path.join(os.path.dirname(os.path.abspath(__file__)), "native", "resample_ref.c")
_RS_TYPE = {np.dtype(np.uint8): 0, np.dtype(np.uint16): 1, np.dtype(np.float32): 2}
_SUB = {"NV12": "420", "P016": "420", "NV16": "422", "P216": "422", "YUV444": "444", "YUV444P16": "444"}


def plane_grids(fmt, w, h):
    """[(width, height, channels)] of each plane of a w x h frame of format `fmt`."""
    sub = _SUB.get(fmt, "rgb")
    if sub == "rgb":
        return [(w, h, 3)]
    if sub == "444":
        return [(w, h, 1)] * 3
    return [(w, h, 1), ((w + 1) // 2, (h + 1) // 2 if sub == "420" else h, 2)]


@pytest.fixture(scope="module")
def rs(tmp_path_factory):
    """tests/native/resample_ref.c, built with the oracle's flags into a temporary directory: .taps(in, out) -> (j0, w);
    .plane(plane, nch, out_w, out_h); .planes(fmt, planes, out_w, out_h) resamples every plane of a frame on its own grid."""
    so = str(tmp_path_factory.mktemp("resample_ref") / "libresample_ref.so")
    subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-std=c11", "-ffp-contract=off", "-fno-fast-math",
                           "-fno-math-errno", "-Wall", "-shared", "-o", so, _REF_C, "-lm"])
    lib = C.CDLL(so)

    def taps(n_in, n_out):
        j0 = np.zeros(n_out, np.int32)
        w = np.zeros((n_out, 4), np.float32)
        lib.rs_ref_taps(n_in, n_out, j0.ctypes.data_as(C.c_void_p), w.ctypes.data_as(C.c_void_p))
        return j0, w

    def plane(a, nch, out_w, out_h):
        a = np.ascontiguousarray(a)
        out = np.zeros((out_h, nch * out_w), a.dtype)
        assert lib.rs_ref_plane(_RS_TYPE[a.dtype], a.ctypes.data_as(C.c_void_p), C.c_size_t(a.strides[0]), a.shape[1] // nch,
                                a.shape[0], nch, out.ctypes.data_as(C.c_void_p), C.c_size_t(out.strides[0]), out_w, out_h) == 0
        return out

    def planes(fmt, ps, out_w, out_h):
        return [plane(p, nch, gw, gh) for p, (gw, gh, nch) in zip(ps, plane_grids(fmt, out_w, out_h))]
    return types.SimpleNamespace(taps=taps, plane=plane, planes=planes)


# ------------------------------------------------------------------------------------------ frames
def _place(planes, layout="compact", pad=0):
    """Sample planes (synth.make_pair_scaled's form) -> (buffer uint8, plane[0] offset, plane[1] offset, pitch, host byte count).
    Planes are one plane stride apart.  compact: pitch rounded up to 256, planes pitch * h apart; padded: pitch rounded up to
    512 plus 64 and 3 spare rows per plane; offset: pitch = row + one sample and every plane one sample past an aligned base."""
    s = planes[0].itemsize
    h = planes[0].shape[0]
    row = max(p.shape[1] * s for p in planes)
    pitch = {"compact": _up(row, 256), "padded": _up(row, 512) + 64, "offset": row + s}[layout]
    coded = h + (3 if layout == "padded" else 0)
    o0 = s if layout == "offset" else 0
    stride = pitch * coded
    last = planes[-1]
    end = o0 + (len(planes) - 1) * stride + (last.shape[0] - 1) * pitch + last.shape[1] * s
    buf = np.zeros(_up(end, 512) + pad, np.uint8)
    for i, p in enumerate(planes):
        rows = np.ascontiguousarray(p).view(np.uint8).reshape(p.shape[0], -1)
        for r in range(rows.shape[0]):
            off = o0 + i * stride + r * pitch
            buf[off: off + rows.shape[1]] = rows[r]
    return buf, o0, (o0 + stride if len(planes) > 1 else 0), pitch, end - o0


def _frame(placed, where="cuda"):
    import torch
    import turbo_metrics_b200 as tm
    buf, o0, o1, pitch, span = placed
    if where == "numpy":
        keep = buf.copy()
        base = keep.ctypes.data
    else:
        keep = torch.from_numpy(buf.copy())
        keep = keep.cuda() if where == "cuda" else (keep.pin_memory() if where == "pinned" else keep)
        base = keep.data_ptr()
    return tm.DeviceFrame(base + o0, base + o1 if o1 else 0, pitch, keep, span)


def _compact_frame(planes, where="cuda"):
    """A frame in the compact layout synth.compact_planes builds (the layout of a scaled handle's staged frames)."""
    from turbo_metrics_b200 import synth
    buf, pitch, p1 = synth.compact_planes(planes)
    return _frame((buf, 0, p1, pitch, buf.size), where)


def _run(m, pairs):
    """Score pairs of frames on a handle: [(score, norms or None, XYB planes of every scale or None)]."""
    ts = [m.compute(a, b) for a, b in pairs]
    info = m.info()
    out = []
    for t in ts:
        score = m.get_score(t)
        norms = None if info.flags & 1 else m.get_norms(t)
        planes = [m.debug_read(t, 0, s) for s in range(info.nscales)] if info.pipeline == 1 else None
        out.append((score, norms, planes))
    return out


def _same(a, b):
    """Bit-equal results of _run."""
    assert len(a) == len(b)
    for (sa, na, pa), (sb, nb, pb) in zip(a, b):
        assert np.float64(sa).view(np.uint64) == np.float64(sb).view(np.uint64), (sa, sb)
        if na is not None and nb is not None:
            assert np.array_equal(na.view(np.uint64), nb.view(np.uint64))
        if pa is not None and pb is not None:
            for s, (x, y) in enumerate(zip(pa, pb)):
                assert np.array_equal(_bits(x), _bits(y)), f"scale {s}: {np.count_nonzero(_bits(x) != _bits(y))} samples differ"


def _oracle_linear(oracle, fmt, planes, w, h, matrix="bt709", full_range=False):
    """The oracle's linear planes of a frame of a format the oracle converts itself (NV12, P016, packed RGB)."""
    if fmt in ("NV12", "P016"):
        from turbo_metrics_b200 import synth
        buf, pitch, p1 = synth.compact_planes(planes)
        return oracle.linear_from_yuv420(buf, pitch, h, w, h, 8 if fmt == "NV12" else 16, matrix, full_range)
    img = planes[0].reshape(h, w, 3)
    return {"SRGB8": oracle.linear_from_srgb8, "SRGB16": oracle.linear_from_srgb16, "SRGBF32": oracle.linear_from_srgbf32,
            "LINEARF32": oracle.linear_from_linearf32}[fmt](img)


def _oracle_xyb(oracle, ref_lin, dis_lin, nscales):
    out, a, b = [], ref_lin, dis_lin
    for s in range(nscales):
        if s > 0:
            a, b = oracle.downscale_by_2(a), oracle.downscale_by_2(b)
        out.append(np.concatenate([oracle.linear_to_xyb(a), oracle.linear_to_xyb(b)], axis=0))
    return out


# ------------------------------------------------------------------------------------------ CPU: arguments
def _create(cfg, src):
    from turbo_metrics_b200 import _lib
    h = C.c_void_p()
    rc = _lib.lib().ssimu2_create_mixed(C.byref(h), C.byref(cfg), C.byref(src))
    if rc == OK:
        _lib.lib().ssimu2_destroy(h)
    return rc


def test_source_struct_keeps_its_size_and_reserved_view():
    from turbo_metrics_b200 import _lib
    s = _lib.Source()
    assert C.sizeof(s) == 32
    s.width, s.height = 1280, 720
    assert list(s.reserved) == [1280, 720, 0, 0]
    assert (s.width, s.height) == (1280, 720)


@pytest.mark.parametrize("size,status", [
    ((1921, 1080), E_UNSUPPORTED), ((1920, 1081), E_UNSUPPORTED), ((4096, 2160), E_UNSUPPORTED),
    ((1280, 0), E_INVALID), ((0, 720), E_INVALID),
    ((1280, 720), E_NODEVICE), ((1, 1), E_NODEVICE), ((1920, 1080), E_NODEVICE), ((0, 0), E_NODEVICE)])
def test_distorted_size_checked_before_any_device_call(size, status):
    import torch
    import turbo_metrics_b200 as tm
    from turbo_metrics_b200.ssimulacra2 import make_config, make_source
    if status == E_NODEVICE and torch.cuda.is_available():
        pytest.skip("a device is present: a valid size creates a handle")
    cfg = make_config(1920, 1080, tm.PixelFormat.NV12)
    src = make_source(cfg, dis_width=size[0], dis_height=size[1])
    assert _create(cfg, src) == status


@pytest.mark.parametrize("word", [2, 3])
def test_reserved_words_after_the_size_must_be_zero(word):
    import turbo_metrics_b200 as tm
    from turbo_metrics_b200.ssimulacra2 import make_config, make_source
    cfg = make_config(1920, 1080, tm.PixelFormat.P016)
    src = make_source(cfg, dis_width=1280, dis_height=720)
    src.reserved[word] = 1
    assert _create(cfg, src) == E_INVALID


def test_python_plumbing_and_is_mixed():
    import turbo_metrics_b200 as tm
    from turbo_metrics_b200.ssimulacra2 import is_mixed, is_scaled, make_config, make_source
    cfg = make_config(1920, 1080, tm.PixelFormat.NV12)
    assert make_source(cfg) is None
    src = make_source(cfg, dis_width=1280, dis_height=720)
    assert (src.format, src.width, src.height) == (int(tm.PixelFormat.NV12), 1280, 720)
    assert is_mixed(cfg, src) and is_scaled(cfg, src)
    # the reference's size, given or left at 0, is an ordinary handle when the descriptions agree
    assert not is_mixed(cfg, make_source(cfg, dis_width=1920, dis_height=1080))
    assert not is_mixed(cfg, make_source(cfg, dis_width=0, dis_height=0))
    assert not is_scaled(cfg, make_source(cfg, dis_fmt=tm.PixelFormat.P016))
    assert is_mixed(cfg, make_source(cfg, dis_fmt=tm.PixelFormat.P016, dis_width=1280, dis_height=720))


def test_classes_pass_the_size_through(monkeypatch):
    import turbo_metrics_b200 as tm
    from turbo_metrics_b200 import _lib, ssimulacra2
    seen = []

    class Fake:
        def __getattr__(self, name):
            def call(*args):
                for a in args:
                    obj = getattr(a, "_obj", None)
                    if isinstance(obj, _lib.Source):
                        seen.append((name, obj.width, obj.height))
                return 0
            return call
    monkeypatch.setattr(_lib, "lib", lambda: Fake())
    monkeypatch.setattr(tm.Ssimulacra2, "info", lambda self: type("I", (), {"batch": 8, "ring": 3})())
    m = tm.Ssimulacra2(1920, 1080, tm.PixelFormat.NV12, dis_width=1280, dis_height=720)
    assert (m.dis_width, m.dis_height, m.mixed) == (1280, 720, True)
    tm.ShardedSsimulacra2(1920, 1080, tm.PixelFormat.NV12, [0], dis_width=960, dis_height=540)
    tm.TurboMetrics(1920, 1080, tm.PixelFormat.NV12, dis_width=640, dis_height=360)
    tm.ShardedTurboMetrics(1920, 1080, tm.PixelFormat.NV12, [0], dis_width=320, dis_height=180)
    assert seen == [("ssimu2_create_mixed", 1280, 720), ("ssimu2_shard_create_mixed", 960, 540),
                    ("ssimu2_create_mixed", 640, 360), ("ssimu2_shard_create_mixed", 320, 180)]
    assert ssimulacra2.Ssimulacra2(1920, 1080, tm.PixelFormat.NV12).dis_width == 1920


# ------------------------------------------------------------------------------------------ CPU: the reference resampler
@pytest.mark.parametrize("dtype", [np.uint8, np.uint16, np.float32])
def test_unchanged_axis_is_a_bitwise_copy(rs, dtype):
    rng = np.random.default_rng(3)
    hi = 1.0 if dtype == np.float32 else np.iinfo(dtype).max
    a = (rng.random((37, 3 * 29)) * hi).astype(dtype)
    same = rs.plane(a, 3, 29, 37)
    assert np.array_equal(same.view(np.uint8), a.view(np.uint8))
    # one axis unchanged: every output column (rows scaled) / row (columns scaled) only mixes along the other axis
    rows = rs.plane(a, 3, 29, 80)
    j0, w = rs.taps(29, 29)
    assert np.array_equal(j0, np.arange(29) - 1) and np.array_equal(w, np.tile([0, 1, 0, 0], (29, 1)).astype(np.float32))
    assert rows.shape == (80, 87)
    cols = rs.plane(a[:1], 3, 64, 1)
    assert cols.shape == (1, 192)


@pytest.mark.parametrize("dtype", [np.uint8, np.uint16])
def test_constant_integer_plane_stays_constant(rs, dtype):
    # (an f32 plane may move by an ulp: the f32 weights sum to 1 only within rounding)
    v = {np.uint8: 201, np.uint16: 40000}[dtype]
    a = np.full((13, 2 * 9), v, dtype)
    out = rs.plane(a, 2, 31, 40)
    assert np.all(out == dtype(v))


@pytest.mark.parametrize("n_in,n_out", [(1, 7), (2, 3), (540, 1080), (720, 1080), (67, 131), (101, 203), (1080, 2160),
                                        (1440, 2160), (541, 1081)])
def test_weights_sum_to_one(rs, n_in, n_out):
    j0, w = rs.taps(n_in, n_out)
    assert np.abs(w.astype(np.float64).sum(axis=1) - 1.0).max() <= 2.0 ** -22
    # taps are centre-aligned: the first tap is floor((x + 0.5) * in / out - 0.5) - 1
    x = np.arange(n_out)
    assert np.array_equal(j0, np.floor((x + 0.5) * (n_in / n_out) - 0.5).astype(np.int32) - 1)


def test_mirror_symmetry(rs):
    rng = np.random.default_rng(11)
    a = rng.random((23, 17)).astype(np.float32)
    out = rs.plane(a, 1, 40, 51)
    flip = rs.plane(np.ascontiguousarray(a[::-1, ::-1]), 1, 40, 51)
    np.testing.assert_allclose(flip[::-1, ::-1], out, rtol=0, atol=2e-6)
    j0, w = rs.taps(17, 40)
    np.testing.assert_allclose(w[::-1, ::-1], w, rtol=0, atol=2e-7)


def test_integer_results_round_half_to_even_and_clamp(rs):
    # a step 0 -> 255 rings below 0 and above 255 in u8 (clamped), and not in f32
    a = np.zeros((4, 8), np.uint8)
    a[:, 4:] = 255
    u8 = rs.plane(a, 1, 29, 4)
    f = rs.plane(a.astype(np.float32), 1, 29, 4)
    assert f.min() < 0 and f.max() > 255
    assert np.array_equal(u8, np.clip(np.rint(f), 0, 255).astype(np.uint8))


# ------------------------------------------------------------------------------------------ GPU
def _handles(fmt, W, H, wd, hd, **kw):
    import turbo_metrics_b200 as tm
    scaled = tm.Ssimulacra2(W, H, _fmt(fmt), batch=kw.pop("batch", 2), ring=1, pipeline="split", dis_width=wd,
                            dis_height=hd, **kw)
    return scaled


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FORMATS)
@pytest.mark.parametrize("sizes", SCALES, ids=lambda s: f"{s[1][0]}x{s[1][1]}-{s[0][0]}x{s[0][1]}")
def test_scaled_equals_unscaled_on_the_reference_upscale(oracle, rs, fmt, sizes):
    import turbo_metrics_b200 as tm
    from turbo_metrics_b200 import synth
    (W, H), (wd, hd) = sizes
    ref, dis = synth.make_pair_scaled(fmt, W, H, wd, hd, frame=2, seed=7)
    up = rs.planes(fmt, dis, W, H)
    with tm.Ssimulacra2(W, H, _fmt(fmt), batch=1, ring=1, pipeline="split", dis_width=wd, dis_height=hd) as m:
        got = _run(m, [(_frame(_place(ref)), _frame(_place(dis)))])
        info = m.info()
        assert info.kernel_launches == 3 + 3   # front-end, k_resample, front-end; k_hpass, k_vpass, k_finalize
    with tm.Ssimulacra2(W, H, _fmt(fmt), batch=1, ring=1, pipeline="split") as m:
        want = _run(m, [(_frame(_place(ref)), _compact_frame(up))])
    _same(got, want)
    if fmt in ("NV12", "P016", "SRGB8", "SRGB16", "SRGBF32", "LINEARF32"):
        xyb = _oracle_xyb(oracle, _oracle_linear(oracle, fmt, ref, W, H), _oracle_linear(oracle, fmt, up, W, H), info.nscales)
        for s, (g, o) in enumerate(zip(got[0][2], xyb)):
            assert np.array_equal(_bits(g), _bits(o)), f"scale {s}: {np.count_nonzero(_bits(g) != _bits(o))} samples differ"


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", YUV)
@pytest.mark.parametrize("matrix", MATRICES)
@pytest.mark.parametrize("full_range", [False, True])
def test_yuv_matrices_and_ranges(rs, fmt, matrix, full_range):
    import turbo_metrics_b200 as tm
    from turbo_metrics_b200 import synth
    (W, H), (wd, hd) = (203, 131), (150, 90)
    ref, dis = synth.make_pair_scaled(fmt, W, H, wd, hd, frame=1, seed=3)
    up = rs.planes(fmt, dis, W, H)
    kw = dict(matrix=tm.ColorMatrix[matrix.upper()], full_range=full_range, batch=1, ring=1, pipeline="split")
    with tm.Ssimulacra2(W, H, _fmt(fmt), dis_width=wd, dis_height=hd, **kw) as m:
        got = _run(m, [(_frame(_place(ref)), _frame(_place(dis)))])
    with tm.Ssimulacra2(W, H, _fmt(fmt), **kw) as m:
        want = _run(m, [(_frame(_place(ref)), _compact_frame(up))])
    _same(got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["P016-4K-NV12-1080p", "SRGB8-1080p-NV12-720p"])
def test_mixed_format_and_size(rs, case):
    import turbo_metrics_b200 as tm
    from turbo_metrics_b200 import synth
    rf, df, (W, H), (wd, hd) = {"P016-4K-NV12-1080p": ("P016", "NV12", (3840, 2160), (1920, 1080)),
                                "SRGB8-1080p-NV12-720p": ("SRGB8", "NV12", (1920, 1080), (1280, 720))}[case]
    ref, _ = synth.make_pair_scaled(rf, W, H, W, H, frame=4, seed=2)
    _, dis = synth.make_pair_scaled(df, W, H, wd, hd, frame=4, seed=2)
    up = rs.planes(df, dis, W, H)
    with tm.Ssimulacra2(W, H, _fmt(rf), batch=1, ring=1, pipeline="split", dis_fmt=_fmt(df), dis_width=wd, dis_height=hd) as m:
        got = _run(m, [(_frame(_place(ref)), _frame(_place(dis)))])
    with tm.Ssimulacra2(W, H, _fmt(rf), batch=1, ring=1, pipeline="split", dis_fmt=_fmt(df)) as m:
        want = _run(m, [(_frame(_place(ref)), _compact_frame(up))])
    _same(got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["P016", "P216", "YUV444P16"])
def test_deep_flag_gives_the_same_bits(fmt):
    import turbo_metrics_b200 as tm
    from turbo_metrics_b200 import synth
    (W, H), (wd, hd) = (640, 360), (427, 240)
    ref, dis = synth.make_pair_scaled(fmt, W, H, wd, hd, frame=3, seed=9)
    res = []
    for deep in (False, True):
        with tm.Ssimulacra2(W, H, _fmt(fmt), batch=1, ring=1, pipeline="split", p016_deep=deep, dis_p016_deep=deep,
                            dis_width=wd, dis_height=hd) as m:
            res.append(_run(m, [(_frame(_place(ref)), _frame(_place(dis)))]))
    _same(res[0], res[1])


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["NV12", "P016", "SRGB8"])
def test_score_only_matches_full_mode(fmt):
    import turbo_metrics_b200 as tm
    from turbo_metrics_b200 import synth
    (W, H), (wd, hd) = (1920, 1080), (1280, 720)
    pairs = [synth.make_pair_scaled(fmt, W, H, wd, hd, frame=f, seed=4) for f in range(3)]
    frames = [(_frame(_place(r)), _frame(_place(d))) for r, d in pairs]
    s = []
    for score_only in (False, True):
        with tm.Ssimulacra2(W, H, _fmt(fmt), batch=2, ring=2, score_only=score_only, dis_width=wd, dis_height=hd) as m:
            s.append(m.get_scores(m.compute_batch([a for a, _ in frames], [b for _, b in frames])))
    assert np.array_equal(s[0].view(np.uint64), s[1].view(np.uint64))


@pytest.mark.gpu
def test_input_groups_with_recycled_surfaces(rs):
    """A decoder-style pool of 2 distorted surfaces, refilled behind wait_input, with input groups of 1 and 3 pairs."""
    import torch
    import turbo_metrics_b200 as tm
    from turbo_metrics_b200 import synth
    fmt, (W, H), (wd, hd) = "NV12", (640, 360), (320, 180)
    pairs = [synth.make_pair_scaled(fmt, W, H, wd, hd, frame=f, seed=6) for f in range(7)]
    with tm.Ssimulacra2(W, H, _fmt(fmt), batch=1, ring=1) as m:
        want = [m.compute_sync(_frame(_place(r)), _compact_frame(rs.planes(fmt, d, W, H)))
                for r, d in pairs]
    for group in (1, 3):
        placed = [_place(d) for _, d in pairs]
        pool = [torch.empty(placed[0][0].size, dtype=torch.uint8, device="cuda") for _ in range(2)]
        refs = [_frame(_place(r)) for r, _ in pairs]
        stream = torch.cuda.Stream()
        with tm.Ssimulacra2(W, H, _fmt(fmt), batch=4, ring=2, input_group=group, dis_width=wd, dis_height=hd) as m:
            tickets = []
            for i, (buf, o0, o1, pitch, span) in enumerate(placed):
                surf = pool[i % 2]
                if i >= 2:
                    m.wait_input(tickets[i - 2], stream)
                with torch.cuda.stream(stream):
                    surf.copy_(torch.from_numpy(buf).pin_memory(), non_blocking=True)
                base = surf.data_ptr()
                tickets.append(m.compute(refs[i], tm.DeviceFrame(base + o0, base + o1, pitch, surf, span), stream))
            m.flush()
            got = [m.get_score(t) for t in tickets]
        assert np.array_equal(np.array(got).view(np.uint64), np.array(want).view(np.uint64)), group


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["NV12", "P016", "YUV444P16", "SRGB16", "LINEARF32"])
def test_distorted_layouts(fmt):
    import turbo_metrics_b200 as tm
    from turbo_metrics_b200 import synth
    (W, H), (wd, hd) = (203, 131), (150, 97)
    ref, dis = synth.make_pair_scaled(fmt, W, H, wd, hd, frame=5, seed=8)
    rf = _frame(_place(ref))
    with tm.Ssimulacra2(W, H, _fmt(fmt), batch=4, ring=1, pipeline="split", dis_width=wd, dis_height=hd) as m:
        res = _run(m, [(rf, _frame(_place(dis, layout))) for layout in ("compact", "padded", "offset")])
    _same(res[:1] * 3, res)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["P016", "YUV444", "SRGBF32"])
def test_distorted_planes_beyond_4gib(fmt):
    """The distorted frame's rows (4:4:4: its Cr plane) lie more than 4 GiB past plane[0]."""
    import torch
    import turbo_metrics_b200 as tm
    from turbo_metrics_b200 import synth
    (W, H), (wd, hd) = (203, 131), (120, 80)
    ref, dis = synth.make_pair_scaled(fmt, W, H, wd, hd, frame=6, seed=1)
    buf, o0, o1, pitch, span = _place(dis)
    rf = _frame(_place(ref))
    gap = (4 << 30) + 4096
    if fmt == "YUV444":
        # planes 2 GiB + a bit apart: Cr lands more than 4 GiB past plane[0]
        stride = gap // 2
        big = torch.zeros(3 * stride, dtype=torch.uint8, device="cuda")
        for i in range(3):
            p = dis[i]
            rows = torch.from_numpy(np.ascontiguousarray(p).view(np.uint8).reshape(p.shape[0], -1)).cuda()
            big[i * stride: i * stride + p.shape[0] * pitch].view(p.shape[0], pitch)[:, :rows.shape[1]] = rows
        base = big.data_ptr()
        df = tm.DeviceFrame(base, base + stride, pitch, big, 0)
    else:
        # a pitch of just over 64 MiB: the last rows lie more than 4 GiB past plane[0]
        bpitch = (64 << 20) + 256
        nrows = [p.shape[0] for p in dis]
        stride = bpitch * nrows[0]
        big = torch.zeros(stride * len(dis), dtype=torch.uint8, device="cuda")
        for i, p in enumerate(dis):
            rows = torch.from_numpy(np.ascontiguousarray(p).view(np.uint8).reshape(p.shape[0], -1)).cuda()
            big[i * stride: i * stride + p.shape[0] * bpitch].view(p.shape[0], bpitch)[:, :rows.shape[1]] = rows
        base = big.data_ptr()
        df = tm.DeviceFrame(base, base + stride if len(dis) > 1 else 0, bpitch, big, 0)
        assert bpitch * (hd - 1) > (4 << 30)
    with tm.Ssimulacra2(W, H, _fmt(fmt), batch=2, ring=1, pipeline="split", dis_width=wd, dis_height=hd) as m:
        res = _run(m, [(rf, _frame((buf, o0, o1, pitch, span))), (rf, df)])
    del big
    torch.cuda.empty_cache()
    _same(res[:1], res[1:])


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["NV12", "P216", "SRGB8"])
def test_host_frames(fmt):
    import turbo_metrics_b200 as tm
    from turbo_metrics_b200 import synth
    (W, H), (wd, hd) = (320, 180), (213, 120)
    pairs = [synth.make_pair_scaled(fmt, W, H, wd, hd, frame=f, seed=5) for f in range(3)]
    with tm.Ssimulacra2(W, H, _fmt(fmt), batch=2, ring=1, dis_width=wd, dis_height=hd) as m:
        want = m.get_scores(m.compute_batch([_frame(_place(r)) for r, _ in pairs], [_frame(_place(d)) for _, d in pairs]))
    for where in ("cpu", "pinned", "numpy"):
        with tm.Ssimulacra2(W, H, _fmt(fmt), batch=2, ring=1, dis_width=wd, dis_height=hd) as m:
            refs = [_frame(_place(r), where) for r, _ in pairs]
            diss = [_frame(_place(d, "padded"), where) for _, d in pairs]
            one = [m.compute_from_cpu(refs[0], diss[0])]
            rest = m.compute_from_cpu_batch(refs[1:], diss[1:])
            got = m.get_scores(range(one[0], rest.stop))
        assert np.array_equal(got.view(np.uint64), want.view(np.uint64)), where


@pytest.mark.gpu
def test_shard_api_and_engine(rs):
    import torch
    import turbo_metrics_b200 as tm
    from turbo_metrics_b200 import synth
    fmt, (W, H), (wd, hd) = "P016", (640, 360), (480, 270)
    pairs = [synth.make_pair_scaled(fmt, W, H, wd, hd, frame=f, seed=12) for f in range(5)]
    with tm.Ssimulacra2(W, H, _fmt(fmt), batch=1, ring=1) as m:
        want = np.array([m.compute_sync(_frame(_place(r)), _compact_frame(rs.planes(fmt, d, W, H)))
                         for r, d in pairs])
    devs = list(range(min(2, torch.cuda.device_count())))
    with tm.ShardedSsimulacra2(W, H, _fmt(fmt), devs, batch=2, dis_width=wd, dis_height=hd) as s:
        refs = [_frame(_place(r), "pinned") for r, _ in pairs]
        diss = [_frame(_place(d), "pinned") for _, d in pairs]
        t = s.submit_host(refs, diss)
        s.flush()
        got = s.get_scores(t)
    assert np.array_equal(got.view(np.uint64), want.view(np.uint64))
    eng = tm.TurboMetrics(W, H, _fmt(fmt), batch=2, ring=2, dis_width=wd, dis_height=hd)
    try:
        res = eng.compute_all([_frame(_place(r)) for r, _ in pairs], [_frame(_place(d)) for _, d in pairs])
    finally:
        eng.close()
    assert np.array_equal(np.array(res.ssimulacra2.scores).view(np.uint64), want.view(np.uint64))


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["NV12", "P016", "YUV444", "SRGB16"])
def test_every_submit_rejects_short_or_misaligned_distorted_frames(fmt):
    """Distorted frames are checked at their own size: a frame right for the reference's size but short or misaligned at
    the distorted size... and a frame right at the distorted size is accepted."""
    import torch
    import turbo_metrics_b200 as tm
    from turbo_metrics_b200 import _lib, synth
    (W, H), (wd, hd) = (320, 180), (200, 120)
    ref, dis = synth.make_pair_scaled(fmt, W, H, wd, hd, frame=0, seed=2)
    s = SAMPLE[fmt]
    good = _place(dis)
    buf, o0, o1, pitch, span = good
    row = max(p.shape[1] * s for p in dis)
    bad = {"short pitch": (buf, o0, o1, row - s, span)}
    if s > 1:
        bad["misaligned pitch"] = (buf, o0, o1, pitch + 1, span)
    bad_host = {"short bytes": (buf, o0, o1, pitch, span - 1)}
    rf_d, rf_h = _frame(_place(ref)), _frame(_place(ref), "numpy")
    lib = _lib.lib()
    with tm.Ssimulacra2(W, H, _fmt(fmt), batch=2, ring=1, dis_width=wd, dis_height=hd) as m:
        for name, p in bad.items():
            f = _frame(p)
            with pytest.raises(_lib.Ssimu2Error) as e:
                m.compute(rf_d, f)
            assert e.value.status == E_INVALID, name
            with pytest.raises(_lib.Ssimu2Error):
                m.compute_batch([rf_d, rf_d], [_frame(good), f])
        for name, p in {**bad, **bad_host}.items():
            f = _frame(p, "numpy")
            with pytest.raises(_lib.Ssimu2Error) as e:
                m.compute_from_cpu(rf_h, f)
            assert e.value.status == E_INVALID, name
            # a batch whose second pair is bad (one byte count per side: the good frame is copied with the bad one's)
            A = (_lib.Frame * 2)(rf_h.c(), rf_h.c())
            B = (_lib.Frame * 2)(_frame(good, "numpy").c(), f.c())
            assert lib.ssimu2_submit_host_sized(m._h, 2, A, rf_h.nbytes, B, f.nbytes, None) == E_INVALID, name
        # nothing of the rejected calls was queued
        t = m.compute(rf_d, _frame(good))
        assert t == 0
        m.get_score(t)
    with tm.ShardedSsimulacra2(W, H, _fmt(fmt), [0], batch=2, dis_width=wd, dis_height=hd) as sh:
        for name, p in {**bad, **bad_host}.items():
            with pytest.raises(_lib.Ssimu2Error) as e:
                sh.submit_host([rf_h], [_frame(p, "numpy")])
            assert e.value.status == E_INVALID, name
        for name, p in bad.items():
            with pytest.raises(_lib.Ssimu2Error) as e:
                sh.submit_device([rf_d], [_frame(p)])
            assert e.value.status == E_INVALID, name
        t = sh.submit_host([rf_h], [_frame(good, "numpy")])
        sh.flush()
        assert np.isfinite(sh.get_scores(t)).all()
    torch.cuda.synchronize()
