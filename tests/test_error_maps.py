"""The error maps, strip by strip, against an exact reference.

The parity tests pin everything up to the blur inputs bit for bit and check what follows -- the V pass, the three error
maps, the f32 band sums, the per-strip f64 partial sums and k_finalize -- only through the 108 pooled norms at 1e-4.  A
norm averages over the whole frame, so one wrong pixel, row or column of a map moves it by ~1/(w*h) of that pixel's
error: far under that bar.  Here the library's partial-sum table (ssimu2_debug_read_partials: per 64-column strip, per
channel, the sums of the SSIM', artifact and detail-lost maps and of their fourth powers) is compared with a float64
evaluation of the same maps, on frames whose error mass sits where kernels go wrong: a small patch of noise on a frame,
strip or band edge makes a strip's sum the work of a few hundred pixels.

Reference.  The algorithm is defined in f32 up to three values per pixel and channel (oracle.map_inputs, the values the
oracle's own map code evaluates): the SSIM' quotient q, a = |x2 - mu2| and b = |x1 - mu1|.  From there the reference is
float64 from the definitions: d = max(1 - q, 0), d^4, d1 = (a - b) / (1 + b), artifact = max(d1, 0), detail = max(-d1, 0)
and their fourth powers (not the (1 + a) / (1 + b) - 1 of cpu.rs: when a and b are ~1e-12 the rounding of 1 + a leaves
few of its digits; see test_reference_sums_reduce_to_the_oracle_norms).  Where ref and dis neighbourhoods are identical,
q is exactly 1 and a == b, so both sides are exactly 0: a strip whose reference sum is 0 must be exactly 0 in the table.

Bound.  Everywhere else |gpu - ref| <= K * 2^-24 * sum|terms| + N * 2^-126 (N = pixels of the strip; the terms are
non-negative, so sum|terms| is the reference sum), with u = 2^-24 and K from the arithmetic of ssimu2_kernels.cuh:
  * accumulation: a lane sums its column over at most 12 rows of a band in f32 (k_hv; k_vpass: 6), the first step being
    exact for an L1 sum and the rounding of the term itself for an L4 sum (fma(d2, d2, 0)), then f2_hsum adds the two
    columns of the lane: at most 13 roundings on the way to f64 -> 13u;
  * f64: at most 181 bands plus 5 shuffle steps per strip, < 2^-45 relative, and the reference's own f64 rounding
    (< h * 2^-53 < 2^-40): together under 1u each -> 2u;
  * per term, L1: SSIM' d = 1 - q is exact for q >= 0.5 and rounded once below -> 1u; edge d1: a - b, 1 + b, the
    rcp.approx + Newton reciprocal (1u + 2^-45: the Newton step squares the seed's 2^-22) and the product -> 4u;
  * per term, L4: d^4 from d carries 4x the error of d, and d2 = d * d one more rounding, doubled by the square:
    SSIM' 4 * 1 + 2 = 6u; edge 4 * 4 + 2 = 18u.
  K_L1 = 13 + 2 + 4 = 19, K_L4 = 13 + 2 + 18 = 33; rounded up to 20 and 34 for the second-order terms.
  * N * 2^-126 covers fourth powers (and any term) that go subnormal or underflow in f32: such a term is below 2^-126.
This bound is derived, not fitted.  Largest observed |gpu - ref| / (2^-24 * sum|terms|) over all cases of this file, on
an NVIDIA B200 at a 1000 W power limit (entries where the N * 2^-126 part of the bound dominates left out):
  hv: 10.1 (score-only: 10.1); split: 9.3.

k_finalize is checked against the same table: the reported norms must be the f64 reduction of the read-back table in the
kernel's order, bit for bit, and the score the oracle's score of those norms within 1e-12 (device pow vs glibc).
"""
import math

import numpy as np
import pytest
import torch

U = 2.0 ** -24
U53 = 2.0 ** -53
TINY = 2.0 ** -126
K_L1, K_L4 = 20, 34
KVEC = np.array([K_L1, K_L4] * 3, np.float64)        # ssim L1, ssim L4, art L1, art L4, det L1, det L4


def _tm():
    import turbo_metrics_b200 as tm
    return tm


# ------------------------------------------------------------------------------------------ reference
def _terms(q, a, b):
    """The six per-pixel terms of one channel in float64: d, d^4, art, art^4, det, det^4."""
    d = 1.0 - q.astype(np.float64)
    d = np.where(d > 0.0, d, 0.0)                    # max(d, 0); NaN -> 0 as in the reference
    a64, b64 = a.astype(np.float64), b.astype(np.float64)
    d1 = (a64 - b64) / (1.0 + b64)
    art, det = np.maximum(d1, 0.0), np.maximum(-d1, 0.0)
    d2, art2, det2 = d * d, art * art, det * det
    return d, d2 * d2, art, art2 * art2, det, det2 * det2


def ref_strip_sums(q, a, b, cols):
    """-> (sums (n_strips, 3, 6), pixels per strip) of the maps of one scale, per `cols`-column strip, in float64."""
    _, h, w = q.shape
    starts = np.arange(0, w, cols)
    out = np.zeros((len(starts), 3, 6), np.float64)
    for c in range(3):
        for k, t in enumerate(_terms(q[c], a[c], b[c])):
            out[:, c, k] = np.add.reduceat(t.sum(axis=0), starts)
    return out, h * np.minimum(cols, w - starts)


def reference_tables(ref_lin, dis_lin, nscales, cols):
    """Reference strip sums of every scale: [(sums, pixels per strip)] from the oracle's per-pixel map inputs."""
    out = []
    for s in range(nscales):
        q, a, b = _oracle().map_inputs(ref_lin, dis_lin, s)
        out.append(ref_strip_sums(q, a, b, cols))
    return out


def _oracle():
    from oracle import oracle
    oracle.build()
    return oracle


def lite_scales(nscales):
    """Scales whose strips run without the SSIM' map of X and B in score-only mode: both SSIM' weights of X and of B are
    zero and those of Y are not (the library's HvArgs::lite == 0b101; weight index ((c * nscales + s) * 2 + n) * 3)."""
    w = _oracle().weights()
    out = []
    for s in range(nscales):
        bits = sum(1 << c for c in range(3) if w[(c * nscales + s) * 6] == 0.0 and w[(c * nscales + s) * 6 + 3] == 0.0)
        if bits == 0b101:
            out.append(s)
    return out


def check_table(gpu, ref, npx, where, lite=False):
    """gpu, ref: (n_strips, 3, 6).  Exact zeros where the reference is 0, the derived bound elsewhere.  lite: the X and B
    SSIM' entries are not computed and must be exactly 0."""
    gpu, ref = gpu.copy(), ref.copy()
    if lite:
        skipped = gpu[:, [0, 2], 0:2]
        assert np.all(skipped == 0.0), f"{where}: lite strip has non-zero X/B SSIM' entries {skipped[skipped != 0][:4]}"
        gpu[:, [0, 2], 0:2] = 0.0
        ref[:, [0, 2], 0:2] = 0.0
    zero = ref == 0.0
    if np.any(gpu[zero] != 0.0):
        i = np.argwhere(zero & (gpu != 0.0))[0]
        raise AssertionError(f"{where}: strip {i[0]} channel {i[1]} entry {i[2]} is {gpu[tuple(i)]!r}, reference exactly 0")
    bound = KVEC * U * ref + npx[:, None, None] * TINY
    err = np.abs(gpu - ref)
    if np.any(err > bound):
        i = np.unravel_index(np.argmax(err / bound), err.shape)
        raise AssertionError(f"{where}: strip {i[0]} channel {i[1]} entry {i[2]}: gpu {gpu[i]!r} ref {ref[i]!r} "
                             f"err {err[i]:.3e} > bound {bound[i]:.3e} ({err[i] / (U * ref[i]) if ref[i] else np.inf:.1f} u)")
    pos = U * ref > npx[:, None, None] * TINY        # the ratio where the relative part of the bound dominates
    return float((err[pos] / (U * ref[pos])).max()) if pos.any() else 0.0


def norms_from_table(parts, info):
    """k_finalize's reduction of the partial-sum table, in its order: sum over strips, (1 / (w * h)) * sum, sqrt(sqrt())
    for L4; -> norms[108] in WEIGHT order (c * 36 + s * 6 + n * 3 + m)."""
    norms = np.zeros(108, np.float64)
    for s, p in enumerate(parts):
        one_per_pixels = 1.0 / float(info.width[s] * info.height[s])
        for c in range(3):
            for k in range(6):
                acc = 0.0
                for i in range(p.shape[0]):
                    acc += float(p[i, c, k])
                v = one_per_pixels * acc
                if k & 1:
                    v = math.sqrt(math.sqrt(v))
                norms[c * 36 + s * 6 + (k & 1) * 3 + (k >> 1)] = v
    return norms


# ------------------------------------------------------------------------------------------ frames
class Pair:
    """One (reference, distorted) pair: device tensors, how to describe them to the library, and the oracle's linear
    planes."""

    def __init__(self, ref, dis, mk, ref_lin, dis_lin):
        self.ref, self.dis, self.mk = ref.cuda(), dis.cuda(), mk
        self.ref_lin, self.dis_lin = ref_lin, dis_lin


def srgb8_base(w, h, seed):
    from turbo_metrics_b200 import synth
    return synth.make_pair_srgb8(w, h, frame=seed, seed=41)[0].numpy()


def srgb8_pair(ref, dis):
    tm, o = _tm(), _oracle()
    return Pair(torch.from_numpy(ref), torch.from_numpy(dis), tm.DeviceFrame.packed, o.linear_from_srgb8(ref),
                o.linear_from_srgb8(dis))


def patched_srgb8(ref, patches, seed):
    """dis = ref except for patches (x0, y0, pw, ph) of seeded noise."""
    rng = np.random.default_rng(seed)
    dis = ref.copy()
    for x0, y0, pw, ph in patches:
        dis[y0:y0 + ph, x0:x0 + pw] = rng.integers(0, 256, (ph, pw, 3), dtype=np.uint8)
    return dis


def clamp_patch(x0, y0, pw, ph, w, h):
    return min(max(x0, 0), w - pw), min(max(y0, 0), h - ph), pw, ph


def edge_patches(w, h, variant):
    """Patch sets on the places kernels go wrong, for one frame of a batch: variant 0..7.  Band edges: k_hv's bands are
    12 input rows, i.e. output rows 12 j - 4 .. 12 j + 7, so a band edge lies between output rows 8 + 12 j - 1 and
    8 + 12 j; strip edges lie between columns 64 k - 1 and 64 k of a scale, i.e. near 64 k 2^s - 1 at scale 0."""
    ns = -(-w // 64)
    last = 64 * (ns - 1)
    sets = [
        [(0, 0, 6, 6)],                                       # top-left corner: first rows, first strip
        [(w - 6, h - 6, 6, 6)],                               # bottom-right corner: last row and column, last strip
        [(61, 17, 6, 6)],                                     # straddles columns 63 | 64 and the band edge 19 | 20
        [(127, 43, 8, 8), (w - 5, 0, 5, 5)],                  # strip edge of scale 1 (columns 63 | 64 there); top-right
        [(0, h - 7, 7, 7)],                                   # bottom-left corner
        [(last - 3, 5, 6, 6)],                                # the last strip's left edge, band edge 7 | 8
        [(w // 2 - 4, h - 4, 8, 4), (w // 3, 0, 8, 4)],       # the last four and the first four output rows
        [(255, 91, 8, 8), (w - 8, h // 2, 8, 4)],             # strip edge of scale 2, band edge 91 | 92; last columns
    ]
    return [clamp_patch(*p, w, h) for p in sets[variant]]


# ------------------------------------------------------------------------------------------ running
def run_batches(tm, w, h, fmt, batches, pipeline, score_only=False):
    """Each batch (a list of Pairs, as many as the handle's batch) goes through ONE batch slot (ring=1), so a later batch
    reuses the slot, its hand-off records and its partial rows.  -> per batch, per pair: (score, norms or None,
    partials per scale); and the handle's info and strip width."""
    kw = {"pipeline": pipeline} if pipeline == "split" else {}
    out = []
    with tm.Ssimulacra2(w, h, fmt, batch=len(batches[0]), ring=1, score_only=score_only, **kw) as m:
        info = m.info()
        _, _, cols = m.debug_strips()
        for pairs in batches:
            ts = [m.compute(p.mk(p.ref), p.mk(p.dis)) for p in pairs]
            res = []
            for t in ts:
                score = m.get_score(t)
                norms = None if score_only else m.get_norms(t)
                res.append((score, norms, m.debug_partials(t)))
            out.append(res)
    return out, info, cols


def check_run(results, batches, info, cols, pipeline, score_only=False, tables=None):
    """Every pair of every batch: partial-sum table against the reference, k_finalize against the table."""
    ns = info.nscales
    lite = lite_scales(ns) if score_only else []
    worst = 0.0
    for bi, (res, pairs) in enumerate(zip(results, batches)):
        for fi, ((score, norms, parts), p) in enumerate(zip(res, pairs)):
            tab = tables[bi][fi] if tables else reference_tables(p.ref_lin, p.dis_lin, ns, cols)
            for s in range(ns):
                ref, npx = tab[s]
                assert parts[s].shape == ref.shape
                worst = max(worst, check_table(parts[s], ref, npx, f"{pipeline} batch {bi} frame {fi} scale {s}",
                                               lite=s in lite))
            from_table = norms_from_table(parts, info)
            if norms is not None:
                assert np.array_equal(norms.view(np.uint64), from_table.view(np.uint64)), \
                    f"batch {bi} frame {fi}: k_finalize norms differ from the table at {np.flatnonzero(norms != from_table)[:6]}"
            assert abs(score - _oracle().score_from_norms(from_table, ns)) <= 1e-12, (score, bi, fi)
    print(f"{pipeline}{' score-only' if score_only else ''}: largest |gpu - ref| / (2^-24 sum|terms|) = {worst:.2f}")
    return worst


# ------------------------------------------------------------------------------------------ GPU cases
# w % 64 in {0, 1, 2, 63, 3}; (h + 4) % 12 in {0, 1, 11, 0, 1}; the last two have fewer than 6 scales (5 and 4)
PATCH_SIZES = [(128, 116), (193, 117), (130, 127), (191, 104), (67, 45)]
MODES = ["hv", "split", "hv_score_only"]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("w,h", PATCH_SIZES)
def test_patches_on_strip_band_and_frame_edges(w, h, mode):
    """Two batches of four frames on one slot, each frame with its patches elsewhere (corners, the last row and column,
    columns 63 | 64 and the last strip, band edges, the first and last four rows, a patch across two strips and two
    bands); the second batch moves every patch, so state left by the first batch, or by another frame of the batch,
    shows as a non-zero entry where the reference is exactly 0."""
    tm = _tm()
    pipeline = mode.replace("_score_only", "")
    score_only = mode.endswith("_score_only")
    base = srgb8_base(w, h, 1)
    batches = [[srgb8_pair(base, patched_srgb8(base, edge_patches(w, h, 4 * b + f), seed=10 * b + f)) for f in range(4)]
               for b in range(2)]
    results, info, cols = run_batches(tm, w, h, tm.PixelFormat.SRGB8, batches, pipeline, score_only)
    if score_only and info.nscales == 6:
        assert lite_scales(6) == [0]
    check_run(results, batches, info, cols, pipeline, score_only)


@pytest.mark.gpu
def test_patches_at_1080p_on_every_scale():
    """1920x1080, both pipelines: patches on the strip edges of scales 0..4 (columns 64 * 2^s - 1 at scale 0), at band
    edges of the deeper scales, and at the corners; then a batch with the patches moved."""
    tm = _tm()
    w, h = 1920, 1080
    base = srgb8_base(w, h, 2)
    sets = [[(64 * (1 << s) - 3, (8 + 12 * (s + 1)) * (1 << s) - 3, 6, 6)] for s in range(5)] + \
           [[(0, 0, 4, 4), (w - 4, h - 4, 4, 4)], [(w - 8, 0, 8, 8), (0, h - 8, 8, 8)],
            [(64 * 7 * 2 - 2, h - 4, 8, 4)]]
    batches = [[srgb8_pair(base, patched_srgb8(base, [clamp_patch(*p, w, h) for p in sets[4 * b + f]], seed=20 + 4 * b + f))
                for f in range(4)] for b in range(2)]
    tables = None
    for pipeline in ("hv", "split"):
        results, info, cols = run_batches(tm, w, h, tm.PixelFormat.SRGB8, batches, pipeline)
        if tables is None:   # the same frames for both pipelines
            tables = [[reference_tables(p.ref_lin, p.dis_lin, info.nscales, cols) for p in pairs] for pairs in batches]
        check_run(results, batches, info, cols, pipeline, tables=tables)


def _dense_pair(kind, w, h, frame):
    tm, o = _tm(), _oracle()
    from turbo_metrics_b200 import synth
    if kind == "srgb8":
        r, d = synth.make_pair_srgb8(w, h, frame=frame, seed=43)
        return srgb8_pair(r.numpy(), d.numpy())
    if kind == "linear":
        r, d = synth.make_pair_linearf32(w, h, frame=frame, seed=43)
        return Pair(r, d, tm.DeviceFrame.packed, o.linear_from_linearf32(r.numpy()), o.linear_from_linearf32(d.numpy()))
    bits = 8 if kind == "nv12" else 16
    rb, db, pitch, ch = synth.make_pair_yuv420(w, h, bits, frame=frame, seed=43)
    mk = lambda t, p=pitch, c=ch: tm.DeviceFrame.yuv420(t, p, c)
    return Pair(rb, db, mk, o.linear_from_yuv420(rb.numpy(), pitch, ch, w, h, bits),
                o.linear_from_yuv420(db.numpy(), pitch, ch, w, h, bits))


FORMATS = {"srgb8": "SRGB8", "nv12": "NV12", "p016": "P016", "linear": "LINEARF32"}


@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(FORMATS))
@pytest.mark.parametrize("w,h", [(203, 131), (1920, 1080)])
def test_dense_content(kind, w, h):
    """Seeded content distorted everywhere: both pipelines at the small size (4:2:0 frames there are 202x131, they have
    even widths), the product pipeline at 1080p; different pairs in one batch."""
    tm = _tm()
    if kind in ("nv12", "p016"):
        w &= ~1
    n = 4 if w < 1000 else 2
    batches = [[_dense_pair(kind, w, h, f) for f in range(n)]]
    tables = None
    for pipeline in (["hv", "split"] if w < 1000 else ["hv"]):
        results, info, cols = run_batches(tm, w, h, tm.PixelFormat[FORMATS[kind]], batches, pipeline)
        if tables is None:
            tables = [[reference_tables(p.ref_lin, p.dis_lin, info.nscales, cols) for p in batches[0]]]
        check_run(results, batches, info, cols, pipeline, tables=tables)


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", ["hv", "split"])
def test_near_identical_pairs(pipeline):
    """dis = ref +- 1 code value at a few pixels: most terms are tiny (fourth powers far below 2^-126), which is where
    the N * 2^-126 allowance and the exact-zero rule meet."""
    tm = _tm()
    w, h = 203, 131
    rng = np.random.default_rng(7)
    base = srgb8_base(w, h, 3)
    pairs = []
    for f in range(4):
        dis = base.copy()
        for _ in range(3 + f):
            y, x, c = rng.integers(0, h), rng.integers(0, w), rng.integers(0, 3)
            v = int(dis[y, x, c])
            dis[y, x, c] = v + 1 if v < 255 else v - 1
        pairs.append(srgb8_pair(base, dis))
    pairs[3] = srgb8_pair(base, base.copy())          # identical: every entry exactly 0
    results, info, cols = run_batches(tm, w, h, tm.PixelFormat.SRGB8, [pairs], pipeline)
    check_run(results, [pairs], info, cols, pipeline)
    assert all(np.all(p == 0.0) for p in results[0][3][2])


@pytest.mark.gpu
def test_4k_p016_patches():
    """3840x2160 P016 (60 strips x 181 bands per chain at scale 0, the longest hand-off chain): a batch of four with two
    patched frames and two identical pairs between them (all-zero tables), on the product pipeline."""
    tm, o = _tm(), _oracle()
    from turbo_metrics_b200 import synth
    w, h = 3840, 2160
    rb, _, pitch, ch = synth.make_pair_yuv420(w, h, 16, frame=0, seed=45)
    mk = lambda t: tm.DeviceFrame.yuv420(t, pitch, ch)
    ref_lin = o.linear_from_yuv420(rb.numpy(), pitch, ch, w, h, 16)

    def patched(patches, seed):
        rng = np.random.default_rng(seed)
        buf = rb.numpy().copy()
        y = buf[: pitch * h].view(np.uint16).reshape(h, pitch // 2)
        for x0, y0, pw, ph in patches:
            y[y0:y0 + ph, x0:x0 + pw] = rng.integers(64, 941, (ph, pw), dtype=np.uint16) << 6
        return Pair(rb, torch.from_numpy(buf), mk, ref_lin, o.linear_from_yuv420(buf, pitch, ch, w, h, 16))

    same = Pair(rb, rb.clone(), mk, ref_lin, ref_lin)
    a = patched([(0, 0, 6, 6), (64 * 32 - 3, 8 * 16 - 3, 8, 8), (w - 6, h - 6, 6, 6)], 1)
    b = patched([(w - 8, 0, 8, 8), (64 * 59 - 2, h - 4, 8, 4), (64 * 2 * 8 - 3, 12 * 90 - 5, 8, 8)], 2)
    batch = [a, same, b, same]
    results, info, cols = run_batches(tm, w, h, tm.PixelFormat.P016, [batch], "hv")
    assert cols == 64 and info.nscales == 6
    # identical pairs: the reference is exactly 0 everywhere (q == 1, a == b), no need to run the oracle on them
    tables = [[reference_tables(p.ref_lin, p.dis_lin, 6, cols) if p is not same else
               [(np.zeros_like(t), np.ones(t.shape[0])) for t in res[2]] for p, res in zip(batch, results[0])]]
    check_run(results, [batch], info, cols, "hv", tables=tables)


# ------------------------------------------------------------------------------------------ CPU: the reference and the export
def _oracle_form_bound(a, b):
    """Per-pixel bound on |d1_oracle - d1| for the oracle's (1 + a) / (1 + b) - 1 in f64 (fl(1 + a), fl(1 + b), the
    quotient: 3 roundings relative to R = (1 + a) / (1 + b); the subtraction: one relative to d1) and d1 itself."""
    a64, b64 = a.astype(np.float64), b.astype(np.float64)
    d1 = (a64 - b64) / (1.0 + b64)
    return 4.0 * U53 * ((1.0 + a64) / (1.0 + b64) + np.abs(d1)), d1


@pytest.mark.parametrize("case", ["dense", "patches", "near_identical", "small"])
def test_reference_sums_reduce_to_the_oracle_norms(oracle, case):
    """Without a device: the reference strip sums of every scale, reduced to norms, agree with the oracle's pooled norms.
    Bounds: both sides sum non-negative terms in f64 ((2 n + 12) * 2^-53 * sum|terms| covers both summations and the
    per-term roundings); the L4 norms are compared as norm^4 (two sqrt and the power: 10 * 2^-53 relative).  The edge
    maps differ by the form: the oracle's (1 + a) / (1 + b) - 1 loses up to 4 * 2^-53 * ((1 + a) / (1 + b) + |d1|) per
    pixel ("oracle form bound"), 4 (|d1| + e)^3 e in the fourth power; where a and b are tiny this is the larger term."""
    from turbo_metrics_b200 import synth
    if case == "dense":
        r, d = synth.make_pair_srgb8(203, 131, frame=1, seed=43)
        r, d = r.numpy(), d.numpy()
    elif case == "small":
        r, d = synth.make_pair_srgb8(67, 45, frame=2, seed=43)
        r, d = r.numpy(), d.numpy()
    else:
        r = synth.make_pair_srgb8(193, 117, frame=1, seed=41)[0].numpy()
        if case == "patches":
            d = patched_srgb8(r, edge_patches(193, 117, 2) + edge_patches(193, 117, 7), seed=3)
        else:
            d = r.copy()
            for y, x, c in ((40, 100, 1), (7, 3, 0), (116, 192, 2)):
                d[y, x, c] = d[y, x, c] + 1 if d[y, x, c] < 255 else 254
    a_lin, b_lin = oracle.linear_from_srgb8(r), oracle.linear_from_srgb8(d)
    _, no, ns = oracle.ssimu2_linear_planar(a_lin, b_lin)
    assert oracle.map_inputs(a_lin, b_lin, ns) is None
    for s in range(ns):
        q, a, b = oracle.map_inputs(a_lin, b_lin, s)
        sums, _ = ref_strip_sums(q, a, b, 64)
        total = sums.sum(axis=0)                                    # (3, 6)
        n = q.shape[1] * q.shape[2]
        form = np.zeros((3, 6))
        for c in range(3):
            e, d1 = _oracle_form_bound(a[c], b[c])
            for k, sign in ((2, 1.0), (4, -1.0)):
                t = np.maximum(sign * d1, 0.0)
                form[c, k] = e.sum()
                form[c, k + 1] = (4.0 * (t + e) ** 3 * e).sum()
        for c in range(3):
            for k in range(6):
                mean = total[c, k] / n
                bound = ((2 * n + 12) * U53 * total[c, k] + form[c, k]) / n
                got = no[c * 36 + s * 6 + (k & 1) * 3 + (k >> 1)]
                if k & 1:
                    got = got ** 4
                    bound += 10 * U53 * mean
                assert abs(got - mean) <= bound, (case, s, c, k, got, mean, bound)
