"""Mixed sources: a handle whose distorted frames have their own pixel format / matrix / range (ssimu2_create_mixed), the
`compute_one(fref, cc_ref, fdis, cc_dis)` shape of turbo-metrics/src/lib.rs:268-360.

The CPU tests check the argument rules and the Python plumbing; the GPU tests check every ordered format pair, the per-side
XYB bits, the frame-lifetime events, host frames of different sizes, the shard API and the engine against the oracle (which
composes per side: linear_from_*(ref), linear_from_*(dis), ssimu2_linear_planar)."""
import ctypes as C
import itertools

import numpy as np
import pytest

from conftest import has_gpu

OK, E_INVALID, E_UNSUPPORTED, E_NODEVICE = 0, -1, -2, -4
NORM_RTOL = 1e-4
SCORE_ATOL = 0.01


def _src(**kw):
    from turbo_metrics_b200 import _lib
    s = _lib.Source()
    s.format, s.matrix, s.full_range, s.flags = 1, 0, 0, 0
    for k, v in kw.items():
        setattr(s, k, v)
    return s


# ------------------------------------------------------------------------------------------ CPU
def test_source_layout_and_minimum_version():
    """ssimu2_source is 32 bytes and the library has the mixed-source calls of ABI 2.1 (later minor versions only add)."""
    from turbo_metrics_b200 import _lib
    assert C.sizeof(_lib.Source) == 32
    assert _lib.lib().ssimu2_version() >= (2 << 16) | 1


def test_create_mixed_rejects_bad_sources_without_a_device():
    """`dis` is checked before any device call, like `cfg`: on a box without a GPU a bad source is reported as such, not as
    SSIMU2_E_NODEVICE."""
    from turbo_metrics_b200 import _lib
    from turbo_metrics_b200.ssimulacra2 import make_config
    lib = _lib.lib()
    h = C.c_void_p(0)
    cfg = make_config(64, 64, 0)
    assert lib.ssimu2_create_mixed(None, C.byref(cfg), C.byref(_src())) == E_INVALID
    assert lib.ssimu2_create_mixed(C.byref(h), None, C.byref(_src())) == E_INVALID
    for bad in (dict(format=6), dict(format=-1), dict(matrix=3), dict(matrix=-1), dict(flags=1), dict(flags=2), dict(flags=0x80),
                dict(format=0, flags=4), dict(format=2, flags=4)):
        assert lib.ssimu2_create_mixed(C.byref(h), C.byref(cfg), C.byref(_src(**bad))) == E_UNSUPPORTED, bad
        assert not h.value
    s = _src()
    s.reserved[3] = 1
    assert lib.ssimu2_create_mixed(C.byref(h), C.byref(cfg), C.byref(s)) == E_INVALID
    bad_cfg = make_config(64, 64, 17)                    # cfg is still checked first
    assert lib.ssimu2_create_mixed(C.byref(h), C.byref(bad_cfg), C.byref(_src())) == E_UNSUPPORTED
    devs = (C.c_int32 * 2)(0, 1)
    assert lib.ssimu2_shard_create_mixed(None, C.byref(cfg), C.byref(_src()), devs, 2) == E_INVALID
    assert lib.ssimu2_shard_create_mixed(C.byref(h), C.byref(cfg), C.byref(_src(matrix=7)), devs, 2) == E_UNSUPPORTED
    assert lib.ssimu2_submit_host_sized(None, 0, None, 0, None, 0, None) == E_INVALID
    assert lib.ssimu2_shard_submit_host_sized(None, 1, None, 0, None, 16, None) == E_INVALID


@pytest.mark.skipif(has_gpu(), reason="only meaningful on a box without a GPU")
def test_good_source_reaches_the_device_check():
    from turbo_metrics_b200 import _lib
    from turbo_metrics_b200.ssimulacra2 import make_config
    h = C.c_void_p(0)
    cfg = make_config(64, 64, 0)
    assert _lib.lib().ssimu2_create_mixed(C.byref(h), C.byref(cfg), C.byref(_src(format=1, flags=4))) == E_NODEVICE
    assert _lib.lib().ssimu2_create_mixed(C.byref(h), C.byref(cfg), None) == E_NODEVICE


def test_python_source_arguments_and_equal_sides():
    import turbo_metrics_b200 as tm
    from turbo_metrics_b200 import _lib
    from turbo_metrics_b200.ssimulacra2 import is_mixed, make_config, make_source
    P, M = tm.PixelFormat, tm.ColorMatrix
    cfg = make_config(64, 64, P.NV12, M.BT601_525, True, flags=_lib.FLAG_SCORE_ONLY)
    assert make_source(cfg) is None
    s = make_source(cfg, dis_fmt=P.P016, dis_matrix=M.BT709, dis_full_range=False, dis_p016_deep=True)
    assert (s.format, s.matrix, s.full_range, s.flags, list(s.reserved)) == (1, 0, 0, _lib.FLAG_P016_DEEP, [0, 0, 0, 0])
    s = make_source(cfg, dis_fmt=P.P016)                # the rest as the reference
    assert (s.format, s.matrix, s.full_range, s.flags) == (1, 1, 1, 0)
    assert is_mixed(cfg, s)
    # equal sides are an ordinary handle: same format and deep flag, and (YUV) same matrix and range
    assert not is_mixed(cfg, make_source(cfg, dis_fmt=P.NV12))
    assert not is_mixed(cfg, make_source(cfg, dis_matrix=M.BT601_525, dis_full_range=True))
    assert is_mixed(cfg, make_source(cfg, dis_matrix=M.BT709))
    assert is_mixed(cfg, make_source(cfg, dis_full_range=False))
    srgb = make_config(64, 64, P.SRGB8)
    assert not is_mixed(srgb, make_source(srgb, dis_matrix=M.BT601_625, dis_full_range=True))   # packed: matrix / range ignored
    assert is_mixed(srgb, make_source(srgb, dis_fmt=P.SRGB16))
    deep = make_config(64, 64, P.P016, flags=_lib.FLAG_P016_DEEP)
    assert make_source(deep, dis_matrix=M.BT709).flags == _lib.FLAG_P016_DEEP   # P016 on both sides: the reference's flag
    assert make_source(deep, dis_fmt=P.NV12).flags == 0
    assert is_mixed(deep, make_source(deep, dis_p016_deep=False))
    assert not is_mixed(deep, make_source(deep, dis_fmt=P.P016))
    assert not is_mixed(cfg, None)


# ------------------------------------------------------------------------------------------ GPU helpers
def _tm():
    import turbo_metrics_b200 as tm
    return tm


def _assert_norms(norms, ref_norms, score, ref_score):
    ref_norms = np.asarray(ref_norms)
    rel = np.abs(norms - ref_norms) / np.maximum(np.abs(ref_norms), 1e-300)
    rel[ref_norms == 0] = np.abs(norms[ref_norms == 0])
    assert rel.max() <= NORM_RTOL, f"max rel norm err {rel.max():.3e} at {rel.argmax()}"
    assert abs(score - ref_score) <= SCORE_ATOL, (score, ref_score)


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


FORMATS = ["NV12", "P016", "SRGB8", "SRGB16", "SRGBF32", "LINEARF32"]
MATRIX_NAME = {0: "bt709", 1: "bt601_525", 2: "bt601_625"}


def _yuv420(rgb8, bits, sig_bits=None, full=False):
    """Packed sRGB8 (H, W, 3) -> NVDEC-layout 4:2:0 buffer (uint8 torch 1-D) of its BT.709 Y'CbCr, `sig_bits` significant bits
    (P016: 10 by default, MSB-aligned in 16).  -> (buf, pitch, coded_height)"""
    import torch
    from turbo_metrics_b200 import synth
    h, w, _ = rgb8.shape
    x = rgb8.numpy().astype(np.float64) / 255.0
    y = 0.2126 * x[..., 0] + 0.7152 * x[..., 1] + 0.0722 * x[..., 2]
    cb, cr = (x[..., 2] - y) / 1.8556, (x[..., 0] - y) / 1.5748
    ph, pw = (h + 1) // 2 * 2, (w + 1) // 2 * 2

    def sub(c):     # 2x2 mean, edge replicated for odd sizes
        c = np.pad(c, ((0, ph - h), (0, pw - w)), mode="edge")
        return 0.25 * (c[0::2, 0::2] + c[1::2, 0::2] + c[0::2, 1::2] + c[1::2, 1::2])
    cb, cr = sub(cb), sub(cr)
    n = sig_bits or (8 if bits == 8 else 10)
    top = (1 << n) - 1
    if full:
        yq, cbq, crq = y * top, (1 << (n - 1)) + cb * top, (1 << (n - 1)) + cr * top
    else:
        s = 1 << (n - 8)
        yq, cbq, crq = 16 * s + 219 * s * y, 128 * s + 224 * s * cb, 128 * s + 224 * s * cr
    q = lambda v: np.clip(np.round(v), 0, top).astype(np.int64) << (0 if bits == 8 else 16 - n)
    yq, cbq, crq = q(yq), q(cbq), q(crq)
    pitch, ch, total = synth.yuv420_geometry(w, h, bits)
    bps = 1 if bits == 8 else 2
    plane = np.zeros(total // bps, np.uint8 if bits == 8 else np.uint16)
    rows = pitch // bps
    plane[: rows * h].reshape(h, rows)[:, :w] = yq
    uv = plane[rows * ch: rows * ch + rows * ((h + 1) // 2)].reshape((h + 1) // 2, rows)
    uv[:, 0:2 * cb.shape[1]:2] = cbq
    uv[:, 1:2 * cb.shape[1]:2] = crq
    return torch.from_numpy(plane.view(np.uint8).copy()), pitch, ch


def _frame(oracle, fmt, rgb8, matrix=0, full=False, sig_bits=None):
    """One side of a pair in `fmt`, converted from the packed sRGB8 picture rgb8.
    -> (cpu tensor, tensor -> DeviceFrame, oracle linear planes (3, H, W))"""
    import torch
    tm = _tm()
    h, w, _ = rgb8.shape
    if fmt in ("NV12", "P016"):
        bits = 8 if fmt == "NV12" else 16
        buf, pitch, ch = _yuv420(rgb8, bits, sig_bits, full)
        lin = oracle.linear_from_yuv420(buf.numpy(), pitch, ch, w, h, bits, MATRIX_NAME[matrix], full)
        return buf, (lambda t: tm.DeviceFrame.yuv420(t, pitch, ch)), lin
    if fmt == "SRGB8":
        return rgb8, tm.DeviceFrame.packed, oracle.linear_from_srgb8(rgb8.numpy())
    if fmt == "SRGB16":
        t = (rgb8.to(torch.int32) * 257 + 5).clamp(0, 65535).to(torch.int16)
        return t, tm.DeviceFrame.packed, oracle.linear_from_srgb16(t.numpy().view(np.uint16))
    if fmt == "SRGBF32":
        t = rgb8.to(torch.float32) / 255.0
        return t, tm.DeviceFrame.packed, oracle.linear_from_srgbf32(t.numpy())
    t = torch.from_numpy(np.ascontiguousarray(oracle.linear_from_srgb8(rgb8.numpy()).transpose(1, 2, 0)))
    return t, tm.DeviceFrame.packed, oracle.linear_from_linearf32(t.numpy())


def _pair(oracle, w, h, ref_fmt, dis_fmt, frame=1, seed=3, **kw):
    """The distorted picture is the reference picture distorted (synth), each converted to its side's format."""
    from turbo_metrics_b200 import synth
    r8, d8 = synth.make_pair_srgb8(w, h, frame=frame, seed=seed)
    rk = {k[4:]: v for k, v in kw.items() if k.startswith("ref_")}
    dk = {k[4:]: v for k, v in kw.items() if k.startswith("dis_")}
    return _frame(oracle, ref_fmt, r8, **rk), _frame(oracle, dis_fmt, d8, **dk)


def _score(m, a, fa, b, fb):
    t = m.compute(fa(a), fb(b))
    return m.get_score(t), (None if m.info().flags & 1 else m.get_norms(t)), t


def _shard_devices():
    import torch
    n = torch.cuda.device_count()
    return list(range(n)) if n >= 2 else [0, 0]


# ------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("ref_fmt,dis_fmt", [p for p in itertools.permutations(FORMATS, 2)])
def test_every_ordered_format_pair_matches_the_oracle(oracle, ref_fmt, dis_fmt):
    """203x131: interior regions take the fast front-end, the last row / column of regions the general one, on both sides."""
    tm = _tm()
    w, h = 203, 131
    (ra, fa, la), (db, fb, lb) = _pair(oracle, w, h, ref_fmt, dis_fmt)
    so, no, nso = oracle.ssimu2_linear_planar(la, lb)
    with tm.Ssimulacra2(w, h, tm.PixelFormat[ref_fmt], dis_fmt=tm.PixelFormat[dis_fmt], batch=2, ring=2) as m:
        assert m.mixed
        score, norms, _ = _score(m, ra.cuda(), fa, db.cuda(), fb)
        info = m.info()
        assert info.nscales == nso
        assert info.kernel_launches == 4          # two front-end launches (one per side), k_hv, k_finalize
    _assert_norms(norms, no, score, so)
    assert 10 < so < 95                           # a derived picture, not the unrelated-frames regime


@pytest.mark.gpu
@pytest.mark.parametrize("ref_fmt,dis_fmt", [("NV12", "P016"), ("SRGB8", "NV12"), ("P016", "SRGBF32"), ("LINEARF32", "SRGB16"),
                                             ("SRGB16", "NV12")])
def test_each_side_has_the_bits_of_its_own_format(oracle, ref_fmt, dis_fmt):
    """XYB planes of every scale: image 0 equals a same-format handle of the reference format scoring (ref, ref), image 1 a
    same-format handle of the distorted format scoring (dis, dis)."""
    tm = _tm()
    w, h = 203, 131
    (ra, fa, _), (db, fb, _) = _pair(oracle, w, h, ref_fmt, dis_fmt)
    ra, db = ra.cuda(), db.cuda()
    P = tm.PixelFormat
    with tm.Ssimulacra2(w, h, P[ref_fmt], dis_fmt=P[dis_fmt], batch=1, ring=1) as m:
        t = m.compute(fa(ra), fb(db))
        m.get_score(t)
        ns = m.info().nscales
        mixed = [m.debug_read(t, 0, s) for s in range(ns)]
    for side, (fmt, x, f) in enumerate([(ref_fmt, ra, fa), (dis_fmt, db, fb)]):
        with tm.Ssimulacra2(w, h, P[fmt], batch=1, ring=1) as m:
            t = m.compute(f(x), f(x))
            assert m.get_score(t) == 100.0
            for s in range(ns):
                same = m.debug_read(t, 0, s)
                assert np.array_equal(_bits(mixed[s][3 * side: 3 * side + 3]), _bits(same[3 * side: 3 * side + 3])), (side, s)


@pytest.mark.gpu
def test_matrix_and_range_mixing_within_one_format(oracle):
    """Same format, different colour description: one handle holds two memo tables (NV12: 256 x 256, P016: 1024 x 1024)."""
    tm = _tm()
    P, M = tm.PixelFormat, tm.ColorMatrix
    w, h = 320, 180
    cases = [("NV12", M.BT601_525, False, M.BT709, True), ("P016", M.BT709, False, M.BT601_625, False),
             ("P016", M.BT601_525, True, M.BT601_525, False)]
    for fmt, rm, rf, dm, df in cases:
        (ra, fa, la), (db, fb, lb) = _pair(oracle, w, h, fmt, fmt, ref_matrix=int(rm), ref_full=rf, dis_matrix=int(dm), dis_full=df)
        so, no, _ = oracle.ssimu2_linear_planar(la, lb)
        with tm.Ssimulacra2(w, h, P[fmt], matrix=rm, full_range=rf, dis_matrix=dm, dis_full_range=df, batch=1, ring=1) as m:
            assert m.mixed
            score, norms, _ = _score(m, ra.cuda(), fa, db.cuda(), fb)
            assert m.info().kernel_launches == 4
        _assert_norms(norms, no, score, so)


@pytest.mark.gpu
def test_p016_deep_flag_of_the_distorted_side_changes_the_speed_not_the_bits(oracle):
    """NV12 reference against a P016 encode with 12 significant bits: with and without SSIMU2_FLAG_P016_DEEP on the distorted
    side the scores, norms and XYB planes are identical, and match the oracle."""
    tm = _tm()
    P = tm.PixelFormat
    w, h = 256, 168
    (ra, fa, la), (db, fb, lb) = _pair(oracle, w, h, "NV12", "P016", dis_sig_bits=12)
    assert (db.numpy().view(np.uint16) & 0x30).any()      # really 12-bit content
    so, no, _ = oracle.ssimu2_linear_planar(la, lb)
    ra, db = ra.cuda(), db.cuda()
    got = {}
    for deep in (False, True):
        with tm.Ssimulacra2(w, h, P.NV12, dis_fmt=P.P016, dis_p016_deep=deep, batch=1, ring=1) as m:
            score, norms, t = _score(m, ra, fa, db, fb)
            got[deep] = (score, norms, [m.debug_read(t, 0, s) for s in range(m.info().nscales)])
    assert got[False][0] == got[True][0] and np.array_equal(got[False][1], got[True][1])
    for a, b in zip(got[False][2], got[True][2]):
        assert np.array_equal(_bits(a), _bits(b))
    _assert_norms(got[True][1], no, got[True][0], so)


@pytest.mark.gpu
def test_equal_sides_make_an_ordinary_handle(oracle):
    """create_mixed with the same effective description: same score bits and the same kernel launches as ssimu2_create."""
    tm = _tm()
    P, M = tm.PixelFormat, tm.ColorMatrix
    w, h, n = 203, 131, 5
    for fmt, kw in (("SRGB8", dict(dis_fmt=P.SRGB8, dis_matrix=M.BT601_625, dis_full_range=True)),
                    ("NV12", dict(dis_fmt=P.NV12, dis_matrix=M.BT709, dis_full_range=False)),
                    ("P016", dict(dis_p016_deep=False))):
        (ra, fa, _), (db, fb, _) = _pair(oracle, w, h, fmt, fmt)
        ra, db = ra.cuda(), db.cuda()
        res = []
        for extra in ({}, kw):
            with tm.Ssimulacra2(w, h, P[fmt], batch=2, ring=2, **extra) as m:
                assert not m.mixed
                s = m.get_scores(m.compute_batch([fa(ra)] * n, [fb(db)] * n))
                res.append((s, m.info().kernel_launches))
        assert np.array_equal(res[0][0], res[1][0]) and res[0][1] == res[1][1] == 3 * 3, (fmt, res)


@pytest.mark.gpu
def test_score_only_mode_on_a_mixed_handle(oracle):
    tm = _tm()
    P = tm.PixelFormat
    w, h, n = 640, 360, 6
    (ra, fa, _), (db, fb, _) = _pair(oracle, w, h, "SRGB8", "P016")
    ra, db = ra.cuda(), db.cuda()
    out = []
    for so in (False, True):
        with tm.Ssimulacra2(w, h, P.SRGB8, dis_fmt=P.P016, batch=4, ring=2, score_only=so) as m:
            out.append(m.get_scores(m.compute_batch([fa(ra)] * n, [fb(db)] * n)))
    assert np.array_equal(out[0], out[1])


@pytest.mark.gpu
def test_recycled_buffers_on_a_mixed_handle_with_input_groups(oracle):
    """input_group=1: ssimu2_stream_wait_input must wait for the SECOND front-end launch of the group (the distorted side).
    One pair of device buffers serves every pair; each buffer is overwritten right behind wait_input."""
    import torch
    tm = _tm()
    P = tm.PixelFormat
    w, h, n = 320, 192, 13
    pairs = [_pair(oracle, w, h, "SRGB8", "NV12", frame=i, seed=44) for i in range(n)]
    expect = [oracle.ssimu2_linear_planar(a[2], b[2])[0] for a, b in pairs]
    fa, fb = pairs[0][0][1], pairs[0][1][1]
    pinned = [(a[0].pin_memory(), b[0].pin_memory()) for a, b in pairs]
    side = torch.cuda.Stream()
    rg, dg = torch.empty_like(pinned[0][0], device="cuda"), torch.empty_like(pinned[0][1], device="cuda")
    with tm.Ssimulacra2(w, h, P.SRGB8, dis_fmt=P.NV12, batch=8, ring=2, input_group=1) as m:
        ts = []
        with torch.cuda.stream(side):
            for r, d in pinned:
                if ts:
                    m.wait_input(ts[-1], side)
                rg.copy_(r, non_blocking=True)
                dg.copy_(d, non_blocking=True)
                ts.append(m.compute(fa(rg), fb(dg), stream=side))
        got = [m.get_score(t) for t in ts]
    with tm.Ssimulacra2(w, h, P.SRGB8, dis_fmt=P.NV12, batch=8, ring=2) as m:
        dev = [(a.cuda(), b.cuda()) for a, b in pinned]
        straight = m.get_scores(m.compute_batch([fa(a) for a, _ in dev], [fb(b) for _, b in dev]))
    assert np.array_equal(np.array(got), straight)
    assert max(abs(a - b) for a, b in zip(got, expect)) <= SCORE_ATOL
    assert len(set(round(x, 6) for x in got)) == n


@pytest.mark.gpu
def test_host_frames_of_different_sizes(oracle):
    """NV12 reference (1.5 B/px) against P016 (3 B/px) from host memory: each side is copied with its own byte count."""
    import torch
    tm = _tm()
    from turbo_metrics_b200 import _lib
    P = tm.PixelFormat
    w, h, n = 640, 360, 5
    pairs = [_pair(oracle, w, h, "NV12", "P016", frame=i, seed=8) for i in range(n)]
    fa, fb = pairs[0][0][1], pairs[0][1][1]
    with tm.Ssimulacra2(w, h, P.NV12, dis_fmt=P.P016, batch=2, ring=2) as m:
        dev = m.get_scores(m.compute_batch([fa(a[0].cuda()) for a, _ in pairs], [fb(b[0].cuda()) for _, b in pairs]))
        pinned = [(a[0].pin_memory(), b[0].pin_memory()) for a, b in pairs]
        refs, diss = [fa(a) for a, _ in pinned], [fb(b) for _, b in pinned]
        assert refs[0].nbytes != diss[0].nbytes
        host = m.get_scores(m.compute_from_cpu_batch(refs, diss))
        one = m.get_score(m.compute_from_cpu(refs[2], diss[2]))
        lib, t = _lib.lib(), C.c_uint64()
        a, b = refs[0].c(), diss[0].c()
        # one byte count for two sides of different bytes per pixel: refused
        assert lib.ssimu2_submit_host(m._h, C.byref(a), C.byref(b), diss[0].nbytes, C.byref(t)) == E_INVALID
        assert lib.ssimu2_submit_host_batch(m._h, 1, C.byref(a), C.byref(b), diss[0].nbytes, C.byref(t)) == E_INVALID
        # a distorted pitch that holds an NV12 row but not a P016 row: refused (both the host and the device path)
        short = diss[0].c()
        short.pitch = w
        assert lib.ssimu2_submit_host_sized(m._h, 1, C.byref(a), refs[0].nbytes, C.byref(short), diss[0].nbytes, C.byref(t)) == E_INVALID
        assert lib.ssimu2_submit(m._h, C.byref(a), C.byref(short), None, C.byref(t)) == E_INVALID
        # a distorted frame whose CbCr plane lies outside its own byte count: refused
        assert lib.ssimu2_submit_host_sized(m._h, 1, C.byref(a), refs[0].nbytes, C.byref(b), b.plane[1] - b.plane[0], C.byref(t)) == E_INVALID
        torch.cuda.synchronize()
    assert np.array_equal(host, dev) and one == dev[2]
    so = oracle.ssimu2_linear_planar(pairs[0][0][2], pairs[0][1][2])[0]
    assert abs(dev[0] - so) <= SCORE_ATOL


@pytest.mark.gpu
def test_shard_api_with_mixed_sources(oracle):
    tm = _tm()
    P = tm.PixelFormat
    w, h, n, nd = 256, 144, 45, 6
    pairs = [_pair(oracle, w, h, "NV12", "P016", frame=i, seed=61) for i in range(nd)]
    fa, fb = pairs[0][0][1], pairs[0][1][1]
    pinned = [(a[0].pin_memory(), b[0].pin_memory()) for a, b in pairs]
    refs, diss = [fa(pinned[i % nd][0]) for i in range(n)], [fb(pinned[i % nd][1]) for i in range(n)]
    with tm.Ssimulacra2(w, h, P.NV12, dis_fmt=P.P016, batch=8, ring=2) as m:
        single = m.get_scores(m.compute_from_cpu_batch(refs, diss))
    with tm.ShardedSsimulacra2(w, h, P.NV12, devices=_shard_devices(), batch=8, ring=2, dis_fmt=P.P016) as sh:
        assert sh.mixed
        got = sh.get_scores(sh.submit_host(refs, diss))
    assert np.array_equal(got, single), f"{int((got != single).sum())} of {n} scores differ"
    assert abs(got[0] - oracle.ssimu2_linear_planar(pairs[0][0][2], pairs[0][1][2])[0]) <= SCORE_ATOL
    eng = tm.ShardedTurboMetrics(w, h, P.NV12, devices=_shard_devices(), batch=8, ring=2, dis_fmt=P.P016)
    try:
        res = eng.compute_all(iter(refs), iter(diss))
    finally:
        eng.close()
    assert res.ssimulacra2.scores == single.tolist()


@pytest.mark.gpu
def test_engine_with_mixed_sources(oracle):
    """TurboMetrics(..., dis_fmt=...): compute_one and compute_all equal the direct mixed handle."""
    tm = _tm()
    P = tm.PixelFormat
    w, h, n = 320, 192, 9
    pairs = [_pair(oracle, w, h, "SRGB8", "P016", frame=i, seed=33, dis_sig_bits=12) for i in range(n)]
    fa, fb = pairs[0][0][1], pairs[0][1][1]
    dev = [(a[0].cuda(), b[0].cuda()) for a, b in pairs]
    eng = tm.TurboMetrics(w, h, P.SRGB8, dis_fmt=P.P016, dis_bit_depth=12, batch=4, ring=2)
    try:
        assert eng.ssimulacra2.mixed
        one = [eng.compute_one(fa(a), fb(b)).ssimulacra2 for a, b in dev]
        res = eng.compute_all((fa(a) for a, _ in dev), (fb(b) for _, b in dev))
    finally:
        eng.close()
    with tm.Ssimulacra2(w, h, P.SRGB8, dis_fmt=P.P016, batch=4, ring=2) as m:
        direct = m.get_scores(m.compute_batch([fa(a) for a, _ in dev], [fb(b) for _, b in dev]))
    assert one == res.ssimulacra2.scores == direct.tolist()
    assert abs(one[0] - oracle.ssimu2_linear_planar(pairs[0][0][2], pairs[0][1][2])[0]) <= SCORE_ATOL


@pytest.mark.gpu
def test_4k_nv12_against_4k_p016_matches_the_oracle(oracle):
    """4K: an 8-bit source (NV12) against a 10-bit encode of it (P016), the pair in the middle of a full batch."""
    tm = _tm()
    from turbo_metrics_b200 import synth
    P = tm.PixelFormat
    w, h = 3840, 2160
    r8, _, p8, c8 = synth.make_pair_yuv420(w, h, 8, frame=0, seed=1)
    _, d16, p16, c16 = synth.make_pair_yuv420(w, h, 16, frame=0, seed=1)
    so, no, nso = oracle.ssimu2_linear_planar(oracle.linear_from_yuv420(r8.numpy(), p8, c8, w, h, 8),
                                              oracle.linear_from_yuv420(d16.numpy(), p16, c16, w, h, 16))
    r2, _, _, _ = synth.make_pair_yuv420(w, h, 8, frame=1, seed=1, device="cuda")
    _, d2, _, _ = synth.make_pair_yuv420(w, h, 16, frame=1, seed=1, device="cuda")
    fa, fb = (lambda t: tm.DeviceFrame.yuv420(t, p8, c8)), (lambda t: tm.DeviceFrame.yuv420(t, p16, c16))
    with tm.Ssimulacra2(w, h, P.NV12, dis_fmt=P.P016, batch=8, ring=2) as m:
        rg, dg = r8.cuda(), d16.cuda()
        ts = [m.compute(fa(r2), fb(d2)) for _ in range(3)] + [m.compute(fa(rg), fb(dg))] + [m.compute(fa(r2), fb(d2)) for _ in range(4)]
        score, norms = m.get_score(ts[3]), m.get_norms(ts[3])
        assert m.info().nscales == nso == 6
    _assert_norms(norms, no, score, so)


@pytest.mark.gpu
def test_1080p_srgb8_against_1080p_nv12_matches_the_oracle(oracle):
    tm = _tm()
    P = tm.PixelFormat
    w, h = 1920, 1080
    (ra, fa, la), (db, fb, lb) = _pair(oracle, w, h, "SRGB8", "NV12", frame=0, seed=1)
    so, no, _ = oracle.ssimu2_linear_planar(la, lb)
    with tm.Ssimulacra2(w, h, P.SRGB8, dis_fmt=P.NV12, batch=2, ring=2) as m:
        score, norms, _ = _score(m, ra.cuda(), fa, db.cuda(), fb)
    _assert_norms(norms, no, score, so)
