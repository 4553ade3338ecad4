"""4:2:2 and 4:4:4 YUV (NVDEC's NV16, P216, YUV444 and YUV444_16Bit surfaces, ABI 2.3) against 4:2:0 and the oracle.

Chroma is sited nearest-neighbour: pixel (x, y) takes chroma (x >> 1, y) in 4:2:2 and (x, y) in 4:4:4, with the per-pixel
arithmetic of NV12 / P016.  So
  - a 4:4:4 frame whose chroma is constant on every 2x2 block, or a 4:2:2 frame whose chroma rows repeat in pairs, must give the
    XYB planes and score of the NV12 / P016 frame holding those chroma samples, bit for bit (no oracle involved);
  - the oracle's value of a 4:4:4 pixel is the oracle's NV12 / P016 value of a pixel with that luma and that chroma: the oracle is
    evaluated on a 2x upscaled 4:2:0 frame (luma repeated on 2x2 blocks, the 4:4:4 chroma as its 4:2:0 chroma) and every second
    pixel of every second row is kept.  4:2:2 is 4:4:4 with each chroma sample repeated across its two pixels.
Layouts: L0 NVDEC geometry (pitch rounded up to 256, planes pitch * coded_height apart, coded_height > height), L1 pitch padded
to a multiple of 512 and coded_height == height, L2 pitch = row bytes + one sample, L3 every plane one sample past an aligned base.
"""
import ctypes as C

import numpy as np
import pytest

OK, E_INVALID, E_UNSUPPORTED, E_NODEVICE = 0, -1, -2, -4
NEW = ["NV16", "P216", "YUV444", "YUV444P16"]
SUB = {"NV16": "422", "P216": "422", "YUV444": "444", "YUV444P16": "444", "NV12": "420", "P016": "420"}
SAMPLE = {"NV16": 1, "P216": 2, "YUV444": 1, "YUV444P16": 2, "NV12": 1, "P016": 2}
SIZES = [(200, 136), (203, 131)]
LAYOUTS = ["L0", "L1", "L2", "L3"]
MATRICES = ["bt709", "bt601_525", "bt601_625"]
E420 = {"NV16": "NV12", "YUV444": "NV12", "P216": "P016", "YUV444P16": "P016"}   # the 4:2:0 format of the same sample size

pytest_gpu = pytest.mark.gpu


def _up(x, m):
    return (x + m - 1) // m * m


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _fmt(name):
    import turbo_metrics_b200 as tm
    return tm.PixelFormat[name]


# ------------------------------------------------------------------------------------------ frames as samples
def _synth(fmt, w, h, side, frame=1, seed=5, deep=False):
    """-> (y, cb, cr) integer sample arrays of one side of a seeded pair: y (h, w); cb / cr at the format's chroma resolution.
    deep: 16-bit samples with non-zero low bits (12-bit content)."""
    from turbo_metrics_b200 import synth
    bits = 8 * SAMPLE[fmt]
    sub = SUB[fmt]
    if sub == "420":
        rb, db, pitch, coded = synth.make_pair_yuv420(w, h, bits, frame=frame, seed=seed)
    else:
        rb, db, pitch, coded = synth.make_pair_yuv(w, h, bits, sub, frame=frame, seed=seed)
    y, cb, cr = _unpack((rb if side == 0 else db).numpy(), fmt, w, h, pitch, coded)
    if deep:
        rng = np.random.default_rng(side + 7)
        y, cb, cr = (a + rng.integers(0, 64, a.shape) for a in (y, cb, cr))
    return y, cb, cr


def _unpack(buf, fmt, w, h, pitch, coded):
    """NVDEC-like surface (1-D uint8) -> (y, cb, cr) as int64 arrays."""
    s, sub = SAMPLE[fmt], SUB[fmt]
    p, plane = pitch // s, pitch * coded // s
    n = 3 * pitch * coded                       # whole rows to the end of the last plane (its last row may be short)
    buf = np.concatenate([buf, np.zeros(max(0, n - buf.size), np.uint8)]) if buf.size < n else buf
    a = buf[: buf.size // s * s].view(np.uint8 if s == 1 else np.uint16).astype(np.int64)
    y = a[: p * h].reshape(h, p)[:, :w]
    if sub == "444":
        return y, a[plane: plane + p * h].reshape(h, p)[:, :w], a[2 * plane: 2 * plane + p * h].reshape(h, p)[:, :w]
    ch, cw = (h + 1) // 2 if sub == "420" else h, (w + 1) // 2
    uv = a[plane: plane + p * ch].reshape(ch, p)
    return y, uv[:, 0:2 * cw:2], uv[:, 1:2 * cw:2]


def _place(fmt, y, cb, cr, layout="L0", pad=0):
    """Samples -> (buffer uint8, plane[0] offset, plane[1] offset, pitch, span of a host frame).  Planes are one plane stride
    apart (4:4:4: Cr at plane[1] + (plane[1] - plane[0])).  pad: extra bytes at the end of the buffer."""
    s, sub = SAMPLE[fmt], SUB[fmt]
    h, w = y.shape
    dt = np.uint8 if s == 1 else np.uint16
    if sub == "444":
        chroma = [cb, cr]
    else:
        uv = np.zeros((cb.shape[0], 2 * cb.shape[1]), np.int64)
        uv[:, 0::2], uv[:, 1::2] = cb, cr
        chroma = [uv]
    row, crow = w * s, chroma[0].shape[1] * s
    pitch = {"L0": _up(row, 256), "L1": _up(max(row, crow), 512), "L2": max(row + s, crow), "L3": _up(row, 256)}[layout]
    coded = _up(h, 16) if layout in ("L0", "L3") else h
    o0 = s if layout == "L3" else 0
    stride = pitch * coded
    planes = [y] + chroma
    end = o0 + (len(planes) - 1) * stride + (planes[-1].shape[0] - 1) * pitch + planes[-1].shape[1] * s
    buf = np.zeros(_up(end, 512) + pad, np.uint8)
    for i, pl in enumerate(planes):
        rows = pl.astype(dt).view(np.uint8).reshape(pl.shape[0], -1)
        for r in range(rows.shape[0]):
            off = o0 + i * stride + r * pitch
            buf[off: off + rows.shape[1]] = rows[r]
    return buf, o0, o0 + stride, pitch, end - o0


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
    return tm.DeviceFrame(base + o0, base + o1, pitch, keep, span)


def oracle_linear(oracle, fmt, y, cb, cr, matrix="bt709", full_range=False):
    """The oracle's linear planes (3, h, w) of a 4:2:0 / 4:2:2 / 4:4:4 frame given as samples (see the module docstring)."""
    sub = SUB[fmt]
    if sub == "420":
        buf, o0, o1, pitch, _ = _place(fmt, y, cb, cr)
        return oracle.linear_from_yuv420(buf[o0:], pitch, (o1 - o0) // pitch, y.shape[1], y.shape[0], 8 * SAMPLE[fmt], matrix,
                                         full_range)
    h, w = y.shape
    if sub == "422":
        cb, cr = np.repeat(cb, 2, axis=1)[:, :w], np.repeat(cr, 2, axis=1)[:, :w]
    s = SAMPLE[fmt]
    dt = np.uint8 if s == 1 else np.uint16
    y2 = np.repeat(np.repeat(y, 2, axis=0), 2, axis=1).astype(dt)
    uv = np.empty((h, 2 * w), dt)
    uv[:, 0::2], uv[:, 1::2] = cb, cr
    buf = np.concatenate([y2.view(np.uint8).ravel(), uv.view(np.uint8).ravel()])
    lin = oracle.linear_from_yuv420(buf, 2 * w * s, 2 * h, 2 * w, 2 * h, 8 * s, matrix, full_range)
    return np.ascontiguousarray(lin[:, ::2, ::2])


def _oracle_xyb(oracle, ref_lin, dis_lin, nscales):
    out, a, b = [], ref_lin, dis_lin
    for s in range(nscales):
        if s > 0:
            a, b = oracle.downscale_by_2(a), oracle.downscale_by_2(b)
        out.append(np.concatenate([oracle.linear_to_xyb(a), oracle.linear_to_xyb(b)], axis=0))
    return out


def _run(m, a, b):
    t = m.compute(a, b)
    score = m.get_score(t)
    info = m.info()
    norms = None if info.flags & 1 else m.get_norms(t)
    planes = [m.debug_read(t, 0, s) for s in range(info.nscales)] if info.pipeline == 1 else None
    return score, norms, planes


@pytest.fixture(scope="module")
def lib23():
    from turbo_metrics_b200 import _lib
    v = _lib.lib().ssimu2_version()
    assert v >= (2 << 16) | 3, f"library ABI {v >> 16}.{v & 0xffff} predates 4:2:2 / 4:4:4"
    return _lib


# ------------------------------------------------------------------------------------------ CPU only
def test_new_formats_are_accepted_up_to_the_device_check(lib23):
    from turbo_metrics_b200.ssimulacra2 import make_config, make_source
    lib = lib23.lib()
    assert lib.ssimu2_version() == (2 << 16) | 3
    gpu = _has_gpu()
    for fmt in [8, 9, 10, 11]:
        for matrix in (0, 1, 2):
            h = C.c_void_p()
            rc = lib.ssimu2_create(C.byref(h), C.byref(make_config(64, 64, fmt, matrix=matrix, full_range=1)))
            assert rc == (OK if gpu else E_NODEVICE), (fmt, rc)
            if rc == OK:
                lib.ssimu2_destroy(h)
        for matrix in (3, 7):                             # still rejected, before the device
            assert lib.ssimu2_create(C.byref(C.c_void_p()), C.byref(make_config(64, 64, fmt, matrix=matrix))) == E_UNSUPPORTED
    for bad in (6, 7, 12, 17, -1):
        assert lib.ssimu2_create(C.byref(C.c_void_p()), C.byref(make_config(64, 64, bad))) == E_UNSUPPORTED, bad
        src = make_source(make_config(64, 64, 0), dis_fmt=0)
        src.format = bad
        assert lib.ssimu2_create_mixed(C.byref(C.c_void_p()), C.byref(make_config(64, 64, 0)), C.byref(src)) == E_UNSUPPORTED


def _has_gpu():
    from conftest import has_gpu
    return has_gpu()


def test_deep_flag_only_on_16_bit_yuv(lib23):
    from turbo_metrics_b200.ssimulacra2 import make_config, make_source
    lib = lib23.lib()
    ok = OK if _has_gpu() else E_NODEVICE
    for fmt in range(12):
        if fmt in (6, 7):
            continue
        want = ok if fmt in (1, 9, 11) else E_UNSUPPORTED
        h = C.c_void_p()
        rc = lib.ssimu2_create(C.byref(h), C.byref(make_config(64, 64, fmt, flags=4)))
        assert rc == want, (fmt, rc)
        if rc == OK:
            lib.ssimu2_destroy(h)
        src = make_source(make_config(64, 64, 0), dis_fmt=fmt, dis_p016_deep=True)
        rc = lib.ssimu2_create_mixed(C.byref(h), C.byref(make_config(64, 64, 0)), C.byref(src))
        assert rc == want, (fmt, rc)
        if rc == OK:
            lib.ssimu2_destroy(h)


def test_pixel_format_names_and_deep_defaults():
    import turbo_metrics_b200 as tm
    from turbo_metrics_b200.ssimulacra2 import is_mixed, make_config, make_source
    assert [(f.name, int(f)) for f in tm.PixelFormat if f >= 8] == [("NV16", 8), ("P216", 9), ("YUV444", 10), ("YUV444P16", 11)]
    cfg = make_config(64, 64, tm.PixelFormat.YUV444P16, flags=4)
    assert make_source(cfg, dis_fmt=tm.PixelFormat.P216).flags == 4        # the reference's deep flag carries over to 16-bit YUV
    assert make_source(cfg, dis_fmt=tm.PixelFormat.YUV444).flags == 0
    assert not is_mixed(cfg, make_source(cfg, dis_fmt=tm.PixelFormat.YUV444P16))
    assert is_mixed(cfg, make_source(cfg, dis_matrix=tm.ColorMatrix.BT601_625))   # matrix matters to every YUV format


def test_yuv422_and_yuv444_frames():
    import torch
    import turbo_metrics_b200 as tm
    for buf in (torch.zeros(3000, dtype=torch.uint8), np.zeros(3000, np.uint8)):
        base = buf.data_ptr() if hasattr(buf, "data_ptr") else buf.ctypes.data
        for ctor in (tm.DeviceFrame.yuv422, tm.DeviceFrame.yuv444):
            f = ctor(buf, 64, 16)
            assert (f.plane0, f.plane1, f.pitch, f.nbytes) == (base, base + 64 * 16, 64, 3000) and f.keepalive is buf
    # a contiguous (3, H, pitch) array is a 4:4:4 frame: Cr at plane1 + (plane1 - plane0)
    planes = np.arange(3 * 16 * 64, dtype=np.uint8).reshape(3, 16, 64)
    f = tm.DeviceFrame.yuv444(planes.reshape(-1), 64, 16)
    assert f.plane1 + (f.plane1 - f.plane0) == planes[2].ctypes.data and f.nbytes == planes.nbytes


def test_synthetic_4_2_2_and_4_4_4_pairs():
    from turbo_metrics_b200 import synth
    for sub, planes in (("422", 2), ("444", 3)):
        for bits in (8, 16):
            r, d, pitch, coded = synth.make_pair_yuv(203, 131, bits, sub, seed=2)
            assert r.numel() == d.numel() == pitch * coded * planes and pitch % 256 == 0 and coded == 144
            r2, _, _, _ = synth.make_pair_yuv(203, 131, bits, sub, seed=2)
            assert (r == r2).all() and not (r == d).all()
            fmt = {("422", 8): "NV16", ("422", 16): "P216", ("444", 8): "YUV444", ("444", 16): "YUV444P16"}[(sub, bits)]
            y, cb, cr = _unpack(r.numpy(), fmt, 203, 131, pitch, coded)
            assert cb.shape == ((131, 102) if sub == "422" else (131, 203))
            if bits == 16:
                assert not any((a & 63).any() for a in (y, cb, cr))   # 10-bit content in the high bits
            assert np.ptp(cb) > 20 * (1 if bits == 8 else 64)   # chroma varies at full resolution


def test_oracle_4_4_4_is_the_per_pixel_formula(oracle):
    """On tiny frames: a 4:4:4 pixel's value is the NV12 / P016 value of a pixel with its own luma and chroma (blocks of
    constant chroma reproduce the 4:2:0 frame), it depends on no other pixel's chroma, and 4:2:2 is 4:4:4 with each chroma
    sample repeated across its two pixels."""
    rng = np.random.default_rng(3)
    for fmt, hi in (("YUV444", 256), ("YUV444P16", 65536)):
        f420 = E420[fmt]
        w, h = 6, 4
        y = rng.integers(0, hi, (h, w))
        cb2, cr2 = rng.integers(0, hi, (2, 3)), rng.integers(0, hi, (2, 3))
        cb, cr = np.repeat(np.repeat(cb2, 2, 0), 2, 1), np.repeat(np.repeat(cr2, 2, 0), 2, 1)
        for matrix in MATRICES:
            for fr in (False, True):
                a = oracle_linear(oracle, fmt, y, cb, cr, matrix, fr)
                b = oracle_linear(oracle, f420, y, cb2, cr2, matrix, fr)
                assert np.array_equal(_bits(a), _bits(b)), (fmt, matrix, fr)
        cb_x = cb.copy()
        cb_x[1, 2] = (cb_x[1, 2] + hi // 3) % hi
        a, b = oracle_linear(oracle, fmt, y, cb, cr), oracle_linear(oracle, fmt, y, cb_x, cr)
        diff = np.any(_bits(a) != _bits(b), axis=0)
        assert diff[1, 2] and diff.sum() == 1
        f422 = "NV16" if fmt == "YUV444" else "P216"
        c422b, c422r = rng.integers(0, hi, (h, 3)), rng.integers(0, hi, (h, 3))
        a = oracle_linear(oracle, f422, y, c422b, c422r)
        b = oracle_linear(oracle, fmt, y, np.repeat(c422b, 2, 1), np.repeat(c422r, 2, 1))
        assert np.array_equal(_bits(a), _bits(b))
    # and a hand-computed pixel: limited-range black and white with neutral chroma are linear 0 and 1
    y = np.array([[16, 235], [235, 16]])
    c = np.full((2, 2), 128)
    lin = oracle_linear(oracle, "YUV444", y, c, c)
    assert np.array_equal(lin[:, 0, 0], [0, 0, 0]) and np.array_equal(lin[:, 0, 1], [1, 1, 1])


def test_placed_layouts_hold_the_samples():
    rng = np.random.default_rng(1)
    for fmt in NEW:
        s, hi = SAMPLE[fmt], 256 ** SAMPLE[fmt]
        for w, h in SIZES:
            cw = w if SUB[fmt] == "444" else (w + 1) // 2
            y, cb, cr = rng.integers(0, hi, (h, w)), rng.integers(0, hi, (h, cw)), rng.integers(0, hi, (h, cw))
            for lay in LAYOUTS:
                buf, o0, o1, pitch, span = _place(fmt, y, cb, cr, lay)
                got = _unpack(buf[o0:], fmt, w, h, pitch, (o1 - o0) // pitch)
                assert all(np.array_equal(a, b) for a, b in zip(got, (y, cb, cr))), (fmt, lay)
                if lay == "L2":
                    assert pitch % (2 * s) == s or pitch == (w + 1) // 2 * 2 * s


# ------------------------------------------------------------------------------------------ GPU: oracle-independent witness
def _witness(fmt, y, cb2, cr2):
    """The 4:2:2 / 4:4:4 frame of `fmt` holding the 4:2:0 chroma (cb2, cr2): chroma repeated on 2x2 blocks (4:4:4) or on row
    pairs (4:2:2)."""
    h, w = y.shape
    if SUB[fmt] == "444":
        return y, np.repeat(np.repeat(cb2, 2, 0), 2, 1)[:h, :w], np.repeat(np.repeat(cr2, 2, 0), 2, 1)[:h, :w]
    return y, np.repeat(cb2, 2, 0)[:h], np.repeat(cr2, 2, 0)[:h]


@pytest_gpu
@pytest.mark.parametrize("w,h", [(203, 131), (1920, 1080)])
@pytest.mark.parametrize("depth", ["8", "16", "deep"])
@pytest.mark.parametrize("sub", ["422", "444"])
def test_subsampled_chroma_gives_the_4_2_0_bits(lib23, sub, depth, w, h):
    import turbo_metrics_b200 as tm
    fmt = {("422", "8"): "NV16", ("444", "8"): "YUV444"}.get((sub, depth), "P216" if sub == "422" else "YUV444P16")
    f420 = E420[fmt]
    deep = depth == "deep"
    sides = [_synth(f420, w, h, side, deep=deep) for side in (0, 1)]
    new = [_witness(fmt, *sd) for sd in sides]
    res = {}
    for name, smp in ((f420, sides), (fmt, new)):
        with tm.Ssimulacra2(w, h, _fmt(name), batch=1, ring=1, pipeline="split", p016_deep=deep) as m:
            res[name] = _run(m, _frame(_place(name, *smp[0])), _frame(_place(name, *smp[1])))
    (s0, n0, p0), (s1, n1, p1) = res[f420], res[fmt]
    for s, (a, b) in enumerate(zip(p0, p1)):
        assert np.array_equal(_bits(a), _bits(b)), f"{fmt}: XYB planes differ from {f420}'s at scale {s}"
    assert s1 == s0 and np.array_equal(n1, n0)
    prod = {}
    for name, smp in ((f420, sides), (fmt, new)):   # the product pipeline too (its sums run in another order than split's)
        with tm.Ssimulacra2(w, h, _fmt(name), batch=2, ring=1, p016_deep=deep) as m:
            prod[name] = _run(m, _frame(_place(name, *smp[0])), _frame(_place(name, *smp[1])))
    assert prod[fmt][0] == prod[f420][0] and np.array_equal(prod[fmt][1], prod[f420][1])


# ------------------------------------------------------------------------------------------ GPU: against the oracle
@pytest_gpu
@pytest.mark.parametrize("w,h", SIZES)
@pytest.mark.parametrize("fmt", NEW)
def test_layouts_against_the_oracle(lib23, oracle, fmt, w, h):
    """Split pipeline: XYB planes of every scale are the oracle's bits in every layout (the two frames of a pair in different
    layouts); default pipeline: score and norms of every layout are the compact layout's, score-only mode gives its score."""
    import turbo_metrics_b200 as tm
    smp = [_synth(fmt, w, h, side) for side in (0, 1)]
    lins = [oracle_linear(oracle, fmt, *sd) for sd in smp]
    pairs = [(LAYOUTS[i], LAYOUTS[(i + 1) % 4]) for i in range(4)] + [("L0", "L0")]
    with tm.Ssimulacra2(w, h, _fmt(fmt), batch=1, ring=1, pipeline="split") as m:
        want = _oracle_xyb(oracle, lins[0], lins[1], m.info().nscales)
        for la, lb in pairs:
            _, _, planes = _run(m, _frame(_place(fmt, *smp[0], la)), _frame(_place(fmt, *smp[1], lb)))
            for s, (got, exp) in enumerate(zip(planes, want)):
                assert np.array_equal(_bits(got), _bits(exp)), f"{la}/{lb}: XYB planes differ at scale {s}"
    with tm.Ssimulacra2(w, h, _fmt(fmt), batch=1, ring=1) as m:
        s0, n0, _ = _run(m, _frame(_place(fmt, *smp[0])), _frame(_place(fmt, *smp[1])))
        for la, lb in pairs:
            score, norms, _ = _run(m, _frame(_place(fmt, *smp[0], la)), _frame(_place(fmt, *smp[1], lb)))
            assert score == s0 and np.array_equal(norms, n0), (la, lb)
    with tm.Ssimulacra2(w, h, _fmt(fmt), batch=1, ring=1, score_only=True) as m:
        assert _run(m, _frame(_place(fmt, *smp[0], "L1")), _frame(_place(fmt, *smp[1])))[0] == s0
    so, no, _ = oracle.ssimu2_linear_planar(*lins)
    assert abs(s0 - so) <= 0.01 and np.max(np.abs(n0 - no) / np.maximum(np.abs(no), 1e-300)) <= 1e-4


@pytest_gpu
@pytest.mark.parametrize("fmt", NEW)
def test_matrices_and_ranges_against_the_oracle(lib23, oracle, fmt):
    import turbo_metrics_b200 as tm
    w, h = 203, 131
    smp = [_synth(fmt, w, h, side) for side in (0, 1)]
    for mi, matrix in enumerate(MATRICES):
        for fr in (False, True):
            lins = [oracle_linear(oracle, fmt, *sd, matrix, fr) for sd in smp]
            with tm.Ssimulacra2(w, h, _fmt(fmt), matrix=tm.ColorMatrix(mi), full_range=fr, batch=1, ring=1, pipeline="split") as m:
                want = _oracle_xyb(oracle, lins[0], lins[1], m.info().nscales)
                score, norms, planes = _run(m, _frame(_place(fmt, *smp[0])), _frame(_place(fmt, *smp[1], "L2")))
            for s, (got, exp) in enumerate(zip(planes, want)):
                assert np.array_equal(_bits(got), _bits(exp)), f"{matrix} full={fr}: XYB planes differ at scale {s}"
            so, no, _ = oracle.ssimu2_linear_planar(*lins)
            assert abs(score - so) <= 0.01 and np.max(np.abs(norms - no) / np.maximum(np.abs(no), 1e-300)) <= 1e-4


@pytest_gpu
@pytest.mark.parametrize("fmt", ["P216", "YUV444P16"])
def test_deep_16_bit_content_against_the_oracle(lib23, oracle, fmt):
    """12-bit content (non-zero low bits): with and without the deep flag, the oracle's planes."""
    import turbo_metrics_b200 as tm
    w, h = 200, 136
    smp = [_synth(fmt, w, h, side, deep=True) for side in (0, 1)]
    lins = [oracle_linear(oracle, fmt, *sd) for sd in smp]
    scores = []
    for deep in (True, False):
        with tm.Ssimulacra2(w, h, _fmt(fmt), batch=1, ring=1, pipeline="split", p016_deep=deep) as m:
            want = _oracle_xyb(oracle, lins[0], lins[1], m.info().nscales)
            score, _, planes = _run(m, _frame(_place(fmt, *smp[0])), _frame(_place(fmt, *smp[1], "L3")))
        for s, (got, exp) in enumerate(zip(planes, want)):
            assert np.array_equal(_bits(got), _bits(exp)), f"deep={deep}: XYB planes differ at scale {s}"
        scores.append(score)
    assert scores[0] == scores[1]


@pytest_gpu
def test_4_4_4_rows_beyond_4gib(lib23, oracle):
    """YUV444P16 planes in the rows of one buffer whose pitch keeps the fast path: luma rows from 0, Cb rows at an offset
    straddling 4 GiB, Cr rows wholly beyond it (Cr = plane[1] + (plane[1] - plane[0])).  Planes and score must be the compact
    copy's bits.  About 6.8 GB of device memory (computed from the pitch, not measured)."""
    import torch
    import turbo_metrics_b200 as tm
    fmt, w, h = "YUV444P16", 192, 136
    pitch = (16 << 20) + 4608
    rows_total = 3 * h
    smp = [_synth(fmt, w, h, side) for side in (0, 1)]
    if torch.cuda.mem_get_info()[0] < pitch * rows_total + (1 << 30):
        pytest.skip("needs about 7 GB of free device memory")
    assert h * pitch < (1 << 32) < 2 * h * pitch and pitch % 16 == 0
    with tm.Ssimulacra2(w, h, _fmt(fmt), batch=1, ring=1, pipeline="split") as m:
        s0, n0, p0 = _run(m, _frame(_place(fmt, *smp[0])), _frame(_place(fmt, *smp[1])))
        buf = torch.zeros(pitch * rows_total, dtype=torch.uint8, device="cuda")
        rows = buf.view(rows_total, pitch)
        col = _up(w * 2, 16)
        frames = []
        for side, (y, cb, cr) in enumerate(smp):
            for i, pl in enumerate((y, cb, cr)):
                rows[i * h: (i + 1) * h, side * col: side * col + 2 * w] = torch.from_numpy(pl.astype(np.uint16).view(np.uint8)).cuda()
            base = buf.data_ptr() + side * col
            frames.append(tm.DeviceFrame(base, base + h * pitch, pitch, buf, 0))
        s1, n1, p1 = _run(m, frames[0], frames[1])
        del rows, buf, frames
        torch.cuda.empty_cache()
    for s, (a, b) in enumerate(zip(p0, p1)):
        assert np.array_equal(_bits(a), _bits(b)), f"XYB planes differ at scale {s}"
    assert s1 == s0 and np.array_equal(n1, n0)


# ------------------------------------------------------------------------------------------ GPU: mixed handles
OTHERS = ["NV12", "P016", "SRGB8", "LINEARF32"]


def _other(oracle, fmt, w, h, side):
    """-> (DeviceFrame on the GPU, oracle linear planes) of one side in a 4:2:0 or packed format."""
    import torch
    import turbo_metrics_b200 as tm
    from turbo_metrics_b200 import synth
    if fmt in ("NV12", "P016"):
        smp = _synth(fmt, w, h, side)
        return _frame(_place(fmt, *smp)), oracle_linear(oracle, fmt, *smp)
    if fmt == "SRGB8":
        img = synth.make_pair_srgb8(w, h, frame=1, seed=5)[side].numpy()
        lin = oracle.linear_from_srgb8(img)
    else:
        img = synth.make_pair_linearf32(w, h, frame=1, seed=5)[side].numpy()
        lin = oracle.linear_from_linearf32(img)
    t = torch.from_numpy(np.ascontiguousarray(img)).cuda()
    return tm.DeviceFrame.packed(t), lin


@pytest_gpu
@pytest.mark.parametrize("other", OTHERS)
@pytest.mark.parametrize("fmt", NEW)
def test_mixed_pairs_against_the_oracle(lib23, oracle, fmt, other):
    """Both orders of (new format, other format) at 203x131: each side's XYB planes are the oracle's, the score is the oracle's."""
    import turbo_metrics_b200 as tm
    w, h = 203, 131
    for new_side in (0, 1):
        smp = _synth(fmt, w, h, new_side)
        fn, ln = _frame(_place(fmt, *smp)), oracle_linear(oracle, fmt, *smp)
        fo, lo = _other(oracle, other, w, h, 1 - new_side)
        (fr, lr), (fd, ld) = ((fn, ln), (fo, lo)) if new_side == 0 else ((fo, lo), (fn, ln))
        rf, df = (fmt, other) if new_side == 0 else (other, fmt)
        with tm.Ssimulacra2(w, h, _fmt(rf), dis_fmt=_fmt(df), batch=1, ring=1, pipeline="split") as m:
            assert m.mixed
            want = _oracle_xyb(oracle, lr, ld, m.info().nscales)
            score, norms, planes = _run(m, fr, fd)
        for s, (got, exp) in enumerate(zip(planes, want)):
            assert np.array_equal(_bits(got), _bits(exp)), f"{rf} vs {df}: XYB planes differ at scale {s}"
        so, no, _ = oracle.ssimu2_linear_planar(lr, ld)
        assert abs(score - so) <= 0.01 and np.max(np.abs(norms - no) / np.maximum(np.abs(no), 1e-300)) <= 1e-4


@pytest_gpu
@pytest.mark.parametrize("fmt,other,w,h", [("YUV444P16", "P016", 3840, 2160), ("NV16", "NV12", 1920, 1080)])
def test_mixed_master_against_its_4_2_0_encode(lib23, fmt, other, w, h):
    """A 4:4:4 / 4:2:2 master (holding the 4:2:0 chroma) against a 4:2:0 encode scores exactly what the 4:2:0 pair scores."""
    import turbo_metrics_b200 as tm
    ref420, dis = _synth(other, w, h, 0), _synth(other, w, h, 1)
    master = _witness(fmt, *ref420)
    with tm.Ssimulacra2(w, h, _fmt(other), batch=2, ring=1) as m:
        s0, n0, _ = _run(m, _frame(_place(other, *ref420)), _frame(_place(other, *dis)))
    with tm.Ssimulacra2(w, h, _fmt(fmt), dis_fmt=_fmt(other), batch=2, ring=1) as m:
        assert m.mixed
        s1, n1, _ = _run(m, _frame(_place(fmt, *master)), _frame(_place(other, *dis)))
        assert m.info().io_bytes_per_pair == w * h * ({"YUV444P16": 6, "NV16": 2}[fmt] + {"P016": 3, "NV12": 1.5}[other]) + 8
    assert s1 == s0 and np.array_equal(n1, n0)


@pytest_gpu
def test_io_bytes_per_pair():
    import turbo_metrics_b200 as tm
    for fmt, bpp in (("NV16", 2), ("P216", 4), ("YUV444", 3), ("YUV444P16", 6)):
        with tm.Ssimulacra2(64, 64, _fmt(fmt), batch=1, ring=1) as m:
            assert m.info().io_bytes_per_pair == 2 * bpp * 64 * 64 + 8, fmt


@pytest_gpu
def test_input_groups_with_recycled_buffers(lib23):
    """Two YUV444 surfaces per side, rewritten on the torch stream behind wait_input: every score is its own content's."""
    import torch
    import turbo_metrics_b200 as tm
    fmt, w, h, n = "YUV444", 200, 136, 12
    placed = [[_place(fmt, *_synth(fmt, w, h, side, frame=f)) for side in (0, 1)] for f in range(3)]
    with tm.Ssimulacra2(w, h, _fmt(fmt), batch=1, ring=1) as m:
        want = [m.compute_sync(_frame(p[0]), _frame(p[1])) for p in placed]
    assert len(set(want)) == 3
    srcs = [[torch.from_numpy(p[side][0]).cuda() for p in placed] for side in (0, 1)]
    pool = [[torch.zeros_like(srcs[side][0]) for _ in range(2)] for side in (0, 1)]
    _, o0, o1, pitch, _ = placed[0][0]
    with tm.Ssimulacra2(w, h, _fmt(fmt), batch=6, ring=2, input_group=1) as m:
        tickets = []
        for i in range(n):
            k = i % 2
            if i >= 2:
                m.wait_input(tickets[i - 2])
            frames = []
            for side in (0, 1):
                pool[side][k].copy_(srcs[side][i % 3])
                b = pool[side][k].data_ptr()
                frames.append(tm.DeviceFrame(b + o0, b + o1, pitch, pool[side][k]))
            tickets.append(m.compute(*frames))
        m.flush()
        got = m.get_scores(range(tickets[0], tickets[-1] + 1))
    assert np.array_equal(got, [want[i % 3] for i in range(n)])


# ------------------------------------------------------------------------------------------ GPU: host frames, shards, engine
@pytest_gpu
@pytest.mark.parametrize("kind", ["pageable", "pinned", "numpy"])
def test_host_frames(lib23, kind):
    """A P216 reference against a YUV444 encode, each copied with its own byte count (ssimu2_submit_host_sized)."""
    import turbo_metrics_b200 as tm
    w, h = 203, 131
    a, b = _place("P216", *_synth("P216", w, h, 0)), _place("YUV444", *_synth("YUV444", w, h, 1), "L2")
    with tm.Ssimulacra2(w, h, tm.PixelFormat.P216, dis_fmt=tm.PixelFormat.YUV444, batch=2, ring=2) as m:
        s0 = m.compute_sync(_frame(a), _frame(b))
        fa, fb = _frame(a, kind), _frame(b, kind)
        assert fa.nbytes != fb.nbytes
        assert m.get_score(m.compute_from_cpu(fa, fb)) == s0
        assert np.all(m.get_scores(m.compute_from_cpu_batch([fa] * 3, [fb] * 3)) == s0)
    for fmt in NEW:   # same-format handles: ssimu2_submit_host with one byte count
        smp = [_synth(fmt, w, h, side) for side in (0, 1)]
        pa, pb = _place(fmt, *smp[0]), _place(fmt, *smp[1])
        with tm.Ssimulacra2(w, h, _fmt(fmt), batch=2, ring=2) as m:
            s0 = m.compute_sync(_frame(pa), _frame(pb))
            assert m.get_score(m.compute_from_cpu(_frame(pa, kind), _frame(pb, kind))) == s0, fmt


@pytest_gpu
def test_shard_stream_equals_the_single_handle_stream(lib23):
    import turbo_metrics_b200 as tm
    fmt, w, h = "YUV444P16", 200, 136
    placed = [[_place(fmt, *_synth(fmt, w, h, side, frame=f)) for side in (0, 1)] for f in range(5)]
    refs = [_frame(p[0], "numpy") for p in placed]
    diss = [_frame(p[1], "numpy") for p in placed]
    with tm.Ssimulacra2(w, h, _fmt(fmt), batch=2, ring=2) as m:
        want = m.get_scores(m.compute_from_cpu_batch(refs, diss))
    with tm.ShardedSsimulacra2(w, h, _fmt(fmt), [0, 0], batch=2) as sh:
        ts = sh.submit_host(refs, diss)
        sh.flush()
        assert np.array_equal(sh.get_scores(ts), want)
    with tm.ShardedSsimulacra2(w, h, _fmt(fmt), [0, 0], batch=2, dis_fmt=tm.PixelFormat.YUV444P16,
                               dis_matrix=tm.ColorMatrix.BT709) as sh:
        ts = sh.submit_host(refs, diss)
        sh.flush()
        assert np.array_equal(sh.get_scores(ts), want)


@pytest_gpu
def test_engine_compute_all_on_a_4_4_4_source(lib23):
    import turbo_metrics_b200 as tm
    fmt, w, h = "YUV444P16", 200, 136
    placed = [[_place(fmt, *_synth(fmt, w, h, side, frame=f)) for side in (0, 1)] for f in range(6)]
    with tm.Ssimulacra2(w, h, _fmt(fmt), batch=1, ring=1) as m:
        want = [m.compute_sync(_frame(p[0]), _frame(p[1])) for p in placed]
    for bit_depth in (10, 12):
        eng = tm.TurboMetrics(w, h, _fmt(fmt), batch=2, ring=2, bit_depth=bit_depth)
        assert bool(eng.ssimulacra2.info().flags & 4) == (bit_depth > 10)
        res = eng.compute_all([_frame(p[0]) for p in placed], [_frame(p[1]) for p in placed])
        eng.close()
        assert res.frame_count == 6 and res.ssimulacra2.scores == want


# ------------------------------------------------------------------------------------------ GPU: rejection
@pytest_gpu
@pytest.mark.parametrize("fmt", NEW)
def test_frames_that_break_the_layout_rule_are_rejected(lib23, fmt):
    """Short host byte counts (4:2:2: the last chroma row; 4:4:4: the last Cr row), misaligned 16-bit planes and a 4:4:4 Cr
    address that wraps are SSIMU2_E_INVALID at the single-GPU and shard entry points; nothing is queued (the handles are
    destroyed without a launch)."""
    from turbo_metrics_b200.ssimulacra2 import make_config
    import torch
    lib = lib23.lib()
    w = hh = 64
    s = SAMPLE[fmt]
    pitch = 256
    planes = 3 if SUB[fmt] == "444" else 2
    span = (planes - 1) * pitch * hh + (hh - 1) * pitch + (w * s if SUB[fmt] == "444" else (w + 1) // 2 * 2 * s)
    host = np.zeros(planes * pitch * hh, np.uint8)
    dev = torch.zeros(planes * pitch * hh, dtype=torch.uint8, device="cuda")
    h, sh, t = C.c_void_p(), C.c_void_p(), C.c_uint64()
    cfg = make_config(w, hh, _fmt(fmt), batch=64, ring=1)
    assert lib.ssimu2_create(C.byref(h), C.byref(cfg)) == OK
    assert lib.ssimu2_shard_create(C.byref(sh), C.byref(make_config(w, hh, _fmt(fmt), batch=8, ring=1)), (C.c_int32 * 1)(0), 1) == OK

    def fr(base, d0=0, d1=0, dp=0):
        f = lib23.Frame()
        f.plane[0], f.plane[1], f.pitch = base + d0, base + pitch * hh + d1, pitch + dp
        return f
    try:
        hb, db = host.ctypes.data, dev.data_ptr()
        good = fr(hb)
        for n in (span - 1, span - pitch):
            assert lib.ssimu2_submit_host(h, C.byref(good), C.byref(good), n, C.byref(t)) == E_INVALID
            assert lib.ssimu2_submit_host_sized(h, 1, C.byref(good), span, C.byref(good), n, C.byref(t)) == E_INVALID
            assert lib.ssimu2_shard_submit_host(sh, 1, C.byref(good), C.byref(good), n, C.byref(t)) == E_INVALID
        bad_dev = []
        if s == 2:
            bad_dev += [fr(db, d0=1), fr(db, d1=1), fr(db, dp=1)]
            for bh in (fr(hb, d1=1), fr(hb, dp=1)):
                assert lib.ssimu2_submit_host(h, C.byref(bh), C.byref(good), span, C.byref(t)) == E_INVALID
        if SUB[fmt] == "444":
            wrap = lib23.Frame()
            wrap.plane[0], wrap.plane[1], wrap.pitch = db, (1 << 63) + db, pitch     # Cr past 2^64
            bad_dev.append(wrap)
            low = lib23.Frame()
            low.plane[0], low.plane[1], low.pitch = db + 4096 * pitch, 4096, pitch   # Cr below address 0
            bad_dev.append(low)
        gd = fr(db)
        for bd in bad_dev:
            for a, b in ((gd, bd), (bd, gd)):
                assert lib.ssimu2_submit(h, C.byref(a), C.byref(b), None, C.byref(t)) == E_INVALID
                assert lib.ssimu2_shard_submit_device(sh, 1, C.byref(a), C.byref(b), None, C.byref(t)) == E_INVALID
        assert lib.ssimu2_submit_host(h, C.byref(good), C.byref(good), span, C.byref(t)) == OK and t.value == 0
        assert lib.ssimu2_submit(h, C.byref(gd), C.byref(gd), None, C.byref(t)) == OK and t.value == 1
    finally:
        assert lib.ssimu2_destroy(h) == OK
        assert lib.ssimu2_shard_destroy(sh) == OK
