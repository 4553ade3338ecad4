"""Per-tile scores (ssimu2_config.tile): the tile table of k_hv<true> against an exact reference, k_tile_finalize against the
table, and the guarantee that nothing else moves.

The tile sums are the strip sums of tests/test_error_maps.py restricted to a tile footprint: the same f32 terms, pooled
per lane in f32 segments of at most 12 rows (a segment also ends at a tile-row boundary) and in f64 beyond.  So they are
checked with that file's float64 reference (the terms of oracle.map_inputs) and its derived bound, K_L1 = 20 and K_L4 = 34
times 2^-24 * sum|terms|, plus N * 2^-126; where the reference sum is exactly 0 the table must be exactly 0.

Margin of test_one_patch_points_at_its_tile.  The recursive Gaussian is causal with a look-ahead of 4 samples: output n of a
scan reads inputs up to n + 4 (x[n + 4] horizontally, input row t for output row t - 4 vertically), and its poles lie on the
unit circle (DESIGN.md section 2), so what a patch leaves in the filter state does not die out to its right and below it.
Above and to the left of the patch, though, nothing can see it past 4 pixels of a scale, plus the scale-s pixel that holds the
patch's first column or row: 5 x 2^s scale-0 pixels, most at scale 5, so MARGIN = 5 x 32 = 160.  A tile whose footprint ends
MARGIN pixels above or to the left of the patch has identical inputs to every map, every term exactly 0, and scores exactly
100.
"""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from test_error_maps import (K_L1, K_L4, Pair, _oracle, _terms, check_table, lite_scales, patched_srgb8, srgb8_base,
                             srgb8_pair)

MARGIN = 160


def _tm():
    import turbo_metrics_b200 as tm
    return tm


# ------------------------------------------------------------------------------------------ reference
def ref_tile_sums(q, a, b, ts, uc):
    """-> (sums (tiles_y, units, 3, 6), pixels per entry (tiles_y, units)) of one scale: rows in tile rows of ts, columns
    in units of uc, float64."""
    _, h, w = q.shape
    rs, cs = np.arange(0, h, ts), np.arange(0, w, uc)
    out = np.zeros((len(rs), len(cs), 3, 6), np.float64)
    for c in range(3):
        for k, t in enumerate(_terms(q[c], a[c], b[c])):
            out[:, :, c, k] = np.add.reduceat(np.add.reduceat(t, rs, axis=0), cs, axis=1)
    return out, np.minimum(ts, h - rs)[:, None] * np.minimum(uc, w - cs)[None, :]


def map_inputs_all(p, nscales):
    o = _oracle()
    return [o.map_inputs(p.ref_lin, p.dis_lin, s) for s in range(nscales)]


def tile_norms(parts, layout, info, tile, ty, tx):
    """k_tile_finalize's reduction of the table for tile (ty, tx), in its order -> norms[108] in WEIGHT order."""
    norms = np.zeros(108, np.float64)
    for s, p in enumerate(parts):
        ts, uc, units = tile >> s, layout[s][2], p.shape[1]
        u0, u1 = tx * ts // uc, min(units, (tx + 1) * ts // uc)
        tw, th = min(ts, info.width[s] - tx * ts), min(ts, info.height[s] - ty * ts)
        one_per_pixels = 1.0 / float(tw * th)
        for c in range(3):
            for k in range(6):
                acc = 0.0
                for u in range(u0, u1):
                    acc += float(p[ty, u, c, k])
                v = one_per_pixels * acc
                if k & 1:
                    v = math.sqrt(math.sqrt(v))
                norms[c * 36 + s * 6 + (k & 1) * 3 + (k >> 1)] = v
    return norms


def run_tiles(w, h, fmt, pairs, tile, score_only=False, **kw):
    """One batch of `pairs` on one slot -> (per pair: score, norms or None, tile scores, tile table per scale), info, layout."""
    tm = _tm()
    out = []
    with tm.Ssimulacra2(w, h, fmt, batch=len(pairs), ring=1, score_only=score_only, tile=tile, **kw) as m:
        info, layout = m.info(), m.debug_tile_units()
        assert m.tile_grid()[:3] == (tile, -(-w // tile), -(-h // tile))
        ts = [m.compute(p.mk(p.ref), p.mk(p.dis)) for p in pairs]
        for t in ts:
            out.append((m.get_score(t), None if score_only else m.get_norms(t), m.get_tile_scores(t), m.debug_tile_partials(t)))
    return out, info, layout


def linear_base(w, h, seed):
    from turbo_metrics_b200 import synth
    return synth.make_pair_linearf32(w, h, frame=seed, seed=41)[0].numpy()


def linear_pair(ref, dis):
    tm, o = _tm(), _oracle()
    return Pair(torch.from_numpy(ref), torch.from_numpy(dis), tm.DeviceFrame.packed, o.linear_from_linearf32(ref),
                o.linear_from_linearf32(dis))


def patched_linear(ref, patches, seed):
    rng = np.random.default_rng(seed)
    dis = ref.copy()
    for x0, y0, pw, ph in patches:
        dis[y0:y0 + ph, x0:x0 + pw] = rng.random((ph, pw, 3), dtype=np.float32)
    return dis


def tile_patches(w, h, variant):
    """Noise patches on tile corners (multiples of 64, 128 and 256), strip edges of scales 0..2, band edges (output rows
    12 j + 8) and the frame's edges and corners."""
    sets = [
        [(253, 253, 6, 6), (0, 0, 5, 5), (w - 6, h - 6, 6, 6), (125, 17, 6, 6)],
        [(61, 125, 6, 6), (w - 5, 0, 5, 5), (0, h - 7, 7, 7), (509, 91, 6, 6), (w // 2 - 3, h - 4, 6, 4)],
    ]
    return [(min(max(x, 0), w - pw), min(max(y, 0), h - ph), pw, ph) for x, y, pw, ph in sets[variant]]


# ------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["srgb8", "linear"])
@pytest.mark.parametrize("w,h", [(203, 131), (1000, 700), (1920, 1080)])
def test_tile_sums_and_scores_against_the_exact_reference(kind, w, h):
    """Tests 1 and 2: for T in {64, 128, 256}, full and score-only, every entry of the tile table is within the derived
    bound of the float64 reference (exact zeros where it is 0; the skipped SSIM' entries of X and B of lite scales exactly 0),
    and every tile score is the oracle's score of the norms formed from the read-back table, within 1e-12."""
    tm, o = _tm(), _oracle()
    if kind == "srgb8":
        base = srgb8_base(w, h, 5)
        pairs = [srgb8_pair(base, patched_srgb8(base, tile_patches(w, h, v), seed=50 + v)) for v in range(2)]
        fmt = tm.PixelFormat.SRGB8
    else:
        base = linear_base(w, h, 5)
        pairs = [linear_pair(base, patched_linear(base, tile_patches(w, h, v), seed=60 + v)) for v in range(2)]
        fmt = tm.PixelFormat.LINEARF32
    inputs = None
    worst = 0.0
    for tile in (64, 128, 256):
        for score_only in (False, True):
            res, info, layout = run_tiles(w, h, fmt, pairs, tile, score_only)
            ns = info.nscales
            inputs = inputs or [map_inputs_all(p, ns) for p in pairs]
            lite = lite_scales(ns) if score_only else []
            for fi, (score, _, tscores, parts) in enumerate(res):
                for s in range(ns):
                    q, a, b = inputs[fi][s]
                    ref, npx = ref_tile_sums(q, a, b, tile >> s, layout[s][2])
                    assert parts[s].shape == ref.shape, (parts[s].shape, ref.shape)
                    where = f"T={tile}{' score-only' if score_only else ''} frame {fi} scale {s}"
                    worst = max(worst, check_table(parts[s].reshape(-1, 3, 6), ref.reshape(-1, 3, 6), npx.reshape(-1),
                                                   where, lite=s in lite))
                for ty in range(tscores.shape[0]):
                    for tx in range(tscores.shape[1]):
                        want = o.score_from_norms(tile_norms(parts, layout, info, tile, ty, tx), ns)
                        assert abs(tscores[ty, tx] - want) <= 1e-12, (tile, score_only, fi, ty, tx, tscores[ty, tx], want)
    print(f"{kind} {w}x{h}: largest |gpu - ref| / (2^-24 sum|terms|) = {worst:.2f} (K_L1 {K_L1}, K_L4 {K_L4})")


def _yuv_pair(w, h, bits, frame):
    tm = _tm()
    from turbo_metrics_b200 import synth
    rb, db, pitch, ch = synth.make_pair_yuv420(w, h, bits, frame=frame, seed=47)
    return Pair(rb, db, lambda t, p=pitch, c=ch: tm.DeviceFrame.yuv420(t, p, c), None, None)


def _srgb8_dense(w, h, frame):
    tm = _tm()
    from turbo_metrics_b200 import synth
    r, d = synth.make_pair_srgb8(w, h, frame=frame, seed=47)
    return Pair(r, d, tm.DeviceFrame.packed, None, None)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["srgb8_1080p", "p016_4k"])
def test_one_tile_covering_the_frame_is_the_frame(case):
    """Test 3: T = 4096 puts the frame in one tile whose units are the strips: no tile-row boundary falls inside the frame,
    so the tile path repeats the strip path's roundings.  The tile score is bit-identical to the frame score and each
    strip's tile entries to debug_partials."""
    tm = _tm()
    if case == "srgb8_1080p":
        w, h, fmt, pairs = 1920, 1080, tm.PixelFormat.SRGB8, [_srgb8_dense(1920, 1080, f) for f in range(2)]
    else:
        w, h, fmt, pairs = 3840, 2160, tm.PixelFormat.P016, [_yuv_pair(3840, 2160, 16, f) for f in range(2)]
    with tm.Ssimulacra2(w, h, fmt, batch=2, ring=1, tile=4096) as m:
        assert m.tile_grid()[:3] == (4096, 1, 1)
        layout = m.debug_tile_units()
        strip0, n_strips, _ = m.debug_strips()
        ts = [m.compute(p.mk(p.ref), p.mk(p.dis)) for p in pairs]
        for t in ts:
            score, tiles = m.get_score(t), m.get_tile_scores(t)
            parts, strips = m.debug_tile_partials(t), m.debug_partials(t)
            assert tiles.shape == (1, 1) and tiles[0, 0].tobytes() == np.float64(score).tobytes(), (tiles, score)
            for s, p in enumerate(parts):
                assert layout[s][1] == n_strips[s] and layout[s][2] == 64
                assert np.array_equal(p[0].view(np.uint64), strips[s].view(np.uint64)), f"scale {s}"


def _run_plain(w, h, fmt, pairs, tile, score_only=False, **kw):
    tm = _tm()
    with tm.Ssimulacra2(w, h, fmt, batch=len(pairs), ring=1, tile=tile, score_only=score_only, **kw) as m:
        ts = [m.compute(p.mk(p.ref), p.mk(p.dis)) for p in pairs]
        return [(m.get_score(t), None if score_only else m.get_norms(t), m.get_tile_scores(t) if tile else None) for t in ts]


def _same_bits(a, b):
    return np.asarray(a, np.float64).tobytes() == np.asarray(b, np.float64).tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["srgb8", "nv12_1080p", "p016_4k", "mixed", "scaled"])
def test_tiles_move_nothing_else(case):
    """Test 4: frame scores and norms with tiles are bit-identical to the same handle without tiles; tile scores are
    bit-identical between the full and score-only modes."""
    tm = _tm()
    from turbo_metrics_b200 import synth
    P = tm.PixelFormat
    kw = {}
    if case == "srgb8":
        w, h, fmt, pairs = 203, 131, P.SRGB8, [_srgb8_dense(203, 131, f) for f in range(3)]
    elif case == "nv12_1080p":
        w, h, fmt, pairs = 1920, 1080, P.NV12, [_yuv_pair(1920, 1080, 8, f) for f in range(2)]
    elif case == "p016_4k":
        w, h, fmt, pairs = 3840, 2160, P.P016, [_yuv_pair(3840, 2160, 16, f) for f in range(2)]
    elif case == "mixed":
        w, h, fmt = 640, 360, P.SRGB8
        kw = {"dis_fmt": P.LINEARF32}
        pairs = []
        for f in range(2):
            r, _ = synth.make_pair_srgb8(w, h, frame=f, seed=48)
            _, d = synth.make_pair_linearf32(w, h, frame=f, seed=48)
            pairs.append(Pair(r, d, tm.DeviceFrame.packed, None, None))
    else:
        w, h, fmt = 1920, 1080, P.SRGB8
        kw = {"dis_width": 1280, "dis_height": 720}
        pairs = []
        for f in range(2):
            r, _ = synth.make_pair_srgb8(w, h, frame=f, seed=49)
            _, d = synth.make_pair_srgb8(1280, 720, frame=f, seed=49)
            pairs.append(Pair(r, d, tm.DeviceFrame.packed, None, None))
    plain = _run_plain(w, h, fmt, pairs, 0, **kw)
    for tile in (64, 256):
        full = _run_plain(w, h, fmt, pairs, tile, **kw)
        lite = _run_plain(w, h, fmt, pairs, tile, score_only=True, **kw)
        for i, ((s0, n0, _), (s1, n1, t1), (s2, _, t2)) in enumerate(zip(plain, full, lite)):
            assert _same_bits(s0, s1) and _same_bits(n0, n1), (case, tile, i)
            assert _same_bits(s0, s2), (case, tile, i)
            assert _same_bits(t1, t2), (case, tile, i, np.argwhere(t1 != t2)[:4])


@pytest.mark.gpu
def test_identical_frames_score_100_everywhere():
    """Test 5a: identical neighbourhoods make every term exactly 0, so every tile scores exactly 100."""
    tm = _tm()
    p = _srgb8_dense(1000, 700, 0)
    same = Pair(p.ref, p.ref.clone(), p.mk, None, None)
    for tile in (64, 128):
        for score, _, tiles in _run_plain(1000, 700, tm.PixelFormat.SRGB8, [same, same], tile):
            assert score == 100.0 and np.all(tiles == 100.0), tiles[tiles != 100.0][:4]


@pytest.mark.gpu
@pytest.mark.parametrize("tile", [64, 128])
def test_one_patch_points_at_its_tile(tile):
    """Test 5b: one distorted 16x16 patch at 1920x1080.  The lowest tile is the patch's tile, and every tile whose footprint
    ends MARGIN scale-0 pixels above or to the left of the patch scores exactly 100 (see the module docstring)."""
    tm = _tm()
    w, h = 1920, 1080
    base = srgb8_base(w, h, 6)
    x0, y0, pw = 1000, 600, 16
    p = srgb8_pair(base, patched_srgb8(base, [(x0, y0, pw, pw)], seed=70))
    (score, _, tiles), = _run_plain(w, h, tm.PixelFormat.SRGB8, [p], tile)
    assert score < 100.0
    ty, tx = np.unravel_index(np.argmin(tiles), tiles.shape)
    assert (ty, tx) == (y0 // tile, x0 // tile), (ty, tx, tiles.min())
    before = np.zeros(tiles.shape, bool)
    for yy in range(tiles.shape[0]):
        for xx in range(tiles.shape[1]):
            before[yy, xx] = x0 - min(w, (xx + 1) * tile) >= MARGIN or y0 - min(h, (yy + 1) * tile) >= MARGIN
    assert before.sum() > 0 and np.all(tiles[before] == 100.0), tiles[before].min()
    print(f"T={tile}: patch tile {tiles[ty, tx]:.4f}; {before.sum()} tiles above / left of it exactly 100; "
          f"the others >= {tiles[~before].min():.4f}")


@pytest.mark.gpu
def test_plumbing_batches_groups_rings_and_host_frames():
    """Test 6: partial batches, input groups, ring > 1, host frames; a pair repeated at different batch positions keeps its
    tile bits."""
    tm = _tm()
    w, h = 203, 131
    pairs = [_srgb8_dense(w, h, f) for f in range(3)]
    want = [r[2] for r in _run_plain(w, h, tm.PixelFormat.SRGB8, pairs, 64)]
    order = [0, 1, 2, 2, 0, 1, 1, 2, 0, 0, 2]          # 11 pairs: batches of 4 leave a partial batch of 3
    for kw in ({"batch": 4, "ring": 1}, {"batch": 4, "ring": 3}, {"batch": 4, "ring": 2, "input_group": 2}):
        with tm.Ssimulacra2(w, h, tm.PixelFormat.SRGB8, tile=64, **kw) as m:
            ts = [m.compute(pairs[i].mk(pairs[i].ref), pairs[i].mk(pairs[i].dis)) for i in order]
            for t, i in zip(ts, order):
                assert _same_bits(m.get_tile_scores(t), want[i]), (kw, t, i)
    with tm.Ssimulacra2(w, h, tm.PixelFormat.SRGB8, tile=64, batch=4, ring=2) as m:
        host = [(tm.DeviceFrame.packed(p.ref.cpu().numpy()), tm.DeviceFrame.packed(p.dis.cpu().numpy())) for p in pairs]
        ts = m.compute_from_cpu_batch([host[i][0] for i in order], [host[i][1] for i in order])
        for t, i in zip(ts, order):
            assert _same_bits(m.get_tile_scores(t), want[i]), ("host", t, i)


@pytest.mark.gpu
def test_tickets_older_than_the_capacity():
    """Test 6: a ticket older than the capacity, or not submitted yet, is SSIMU2_E_TICKET; the newest are still there."""
    tm = _tm()
    from turbo_metrics_b200._lib import Ssimu2Error
    p = _srgb8_dense(64, 64, 0)
    a, b = p.mk(p.ref), p.mk(p.dis)
    with tm.Ssimulacra2(64, 64, tm.PixelFormat.SRGB8, tile=64, batch=64, ring=1) as m:
        _, tx, ty, cap = m.tile_grid()
        assert (tx, ty) == (1, 1) and cap >= 64
        ts = m.compute_batch([a] * (cap + 70), [b] * (cap + 70))
        last = m.get_tile_scores(ts[-1])
        assert _same_bits(m.get_tile_scores(ts[-cap]), last)
        for t in (ts[0], ts[-cap - 1], ts[-1] + 1):
            with pytest.raises(Ssimu2Error) as e:
                m.get_tile_scores(t)
            assert e.value.status == -5
        assert m.get_score(ts[-cap - 1]) == m.get_score(ts[-1])   # the score ring is longer


# ------------------------------------------------------------------------------------------ without a device
def _create(cfg):
    from turbo_metrics_b200 import _lib
    h = C.c_void_p()
    rc = _lib.lib().ssimu2_create(C.byref(h), C.byref(cfg))
    if rc == 0:
        _lib.lib().ssimu2_destroy(h)
    return rc


@pytest.mark.parametrize("tile", [1, 32, 63, 65, 96, 100, 48000, 65536, 1 << 31])
def test_bad_tile_sizes_are_unsupported(tile):
    from turbo_metrics_b200.ssimulacra2 import make_config
    assert _create(make_config(256, 256, 2, tile=tile)) == -2


def test_tiles_with_the_split_pipeline_are_unsupported():
    from turbo_metrics_b200 import _lib
    from turbo_metrics_b200.ssimulacra2 import make_config
    for tile in (64, 4096):
        assert _create(make_config(256, 256, 2, pipeline=_lib.PIPELINE_SPLIT, tile=tile)) == -2


@pytest.mark.parametrize("tile", [64, 128, 32768])
def test_good_tile_sizes_pass_the_argument_checks(tile):
    """A valid size gets past the checks made before any device call: without a GPU the create fails for want of a device."""
    from conftest import has_gpu
    from turbo_metrics_b200.ssimulacra2 import make_config
    rc = _create(make_config(256, 256, 2, tile=tile))
    assert rc == (0 if has_gpu() else -4)


def test_shards_refuse_tiles():
    from turbo_metrics_b200 import _lib
    from turbo_metrics_b200.ssimulacra2 import make_config, make_source
    cfg = make_config(256, 256, 2, tile=64)
    s, devs = C.c_void_p(), (C.c_int32 * 1)(0)
    assert _lib.lib().ssimu2_shard_create(C.byref(s), C.byref(cfg), devs, 1) == -2
    src = make_source(cfg, dis_fmt=5)
    assert _lib.lib().ssimu2_shard_create_mixed(C.byref(s), C.byref(cfg), C.byref(src), devs, 1) == -2


def test_config_tile_is_the_first_reserved_word():
    from turbo_metrics_b200._lib import Config
    from turbo_metrics_b200.ssimulacra2 import make_config
    assert C.sizeof(Config) == 64
    cfg = make_config(256, 256, 2, tile=128)
    assert cfg.tile == 128 and list(cfg.reserved) == [128, 0, 0, 0, 0]
    cfg.tile = 0
    assert list(cfg.reserved) == [0] * 5 and make_config(256, 256, 2).tile == 0


def test_tile_symbols_are_exported():
    from turbo_metrics_b200 import _lib
    lib = _lib.lib()
    for n in ("ssimu2_get_tile_grid", "ssimu2_get_tile_scores", "ssimu2_debug_read_tile_partials", "ssimu2_debug_tile_units"):
        assert n in _lib.SYMBOLS and hasattr(lib, n)


def test_reference_tile_sums_add_up_to_the_strip_sums(oracle):
    """The reference pooled per tile adds up, over the tiles of each strip, to test_error_maps' per-strip reference."""
    from test_error_maps import ref_strip_sums
    from turbo_metrics_b200 import synth
    r, d = synth.make_pair_srgb8(203, 131, frame=1, seed=43)
    a_lin, b_lin = oracle.linear_from_srgb8(r.numpy()), oracle.linear_from_srgb8(d.numpy())
    for s in range(3):
        q, a, b = oracle.map_inputs(a_lin, b_lin, s)
        strips, spx = ref_strip_sums(q, a, b, 64)
        for tile in (64, 128):
            ts = tile >> s
            uc = min(64, ts)
            tiles, tpx = ref_tile_sums(q, a, b, ts, uc)
            per_strip = np.add.reduceat(tiles.sum(axis=0), np.arange(0, tiles.shape[1], 64 // uc), axis=0)
            assert np.allclose(per_strip, strips, rtol=1e-12, atol=0)
            assert tpx.sum() == spx.sum() == q.shape[1] * q.shape[2]
