"""Host-side mirror of the reference's per-pair driver `TurboMetrics`
(/root/reference/crates/turbo-metrics/src/lib.rs:188-433) for the SSIMULACRA2 metric, plus the frame
sharding the reference does not have (it is single-GPU: device 0 is hard-coded, lib.rs:442).

* `TurboMetrics.compute_one(fref, fdis)`  -- same contract as lib.rs:268-360: one pair in, `FrameScores` out,
  host-synchronous (the score is fetched before returning).
* `TurboMetrics.compute_all(pairs)`       -- the frame loop of lib.rs:362-433 re-done for throughput: pairs are
  submitted ahead (batch x ring in flight) and scores are collected in submission order.
* `ShardedTurboMetrics.compute_all(...)`   -- the same loop over ALL GPUs of the box from one process (north_star 3): host frames
  go through `ssimu2_shard_submit_host`, the library's per-device worker threads copy and score them, one ordered score stream.
* `shard_range / gather_scores`           -- the one-process-per-GPU form (torchrun): each rank scores a contiguous shard; only
  scalar scores are exchanged (ordered gather to rank 0).  No data-path collective.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Iterable, List, Optional, Sequence, Tuple

from .ssimulacra2 import YUV16_FORMATS, ColorMatrix, DeviceFrame, PixelFormat, ShardedSsimulacra2, Ssimulacra2


@dataclass
class FrameScores:
    """turbo-metrics/src/lib.rs:114-123 restricted to the metric of this path (serde skips the `None` metrics, so a
    reference run with only --ssimulacra2 serialises exactly this)."""
    ssimulacra2: Optional[float] = None


@dataclass
class MetricAggregate:
    """turbo-metrics/src/lib.rs:56-70."""
    scores: List[float]
    stats: "Stats"


@dataclass
class MetricsResults:
    """turbo-metrics/src/lib.rs:72-84 restricted to ssimulacra2."""
    frame_count: int
    ssimulacra2: Optional[MetricAggregate]


@dataclass
class Options:
    """turbo-metrics/src/lib.rs:40-54: frame selection of `compute_all`."""
    every: int = 1
    skip: int = 0
    skip_ref: int = 0
    skip_dis: int = 0
    frames: int = 0  # 0 = all


def select_frames(n_ref: int, n_dis: int, opt: Options) -> List[Tuple[int, int]]:
    """Index pairs (ref_idx, dis_idx) the reference loop scores (lib.rs:385-400): skip `skip + skip_ref` reference
    frames and `skip + skip_dis` distorted frames; with k counting the frames decoded after that, score k when
    `k % every == 0`, and stop at the first scored candidate with `k >= frames` (`frames` bounds the DECODE count)."""
    r0, d0 = opt.skip + opt.skip_ref, opt.skip + opt.skip_dis
    out = []
    k = 0
    while r0 + k < n_ref and d0 + k < n_dis:
        if opt.every > 1 and k != 0 and k % opt.every != 0:
            k += 1
            continue
        if opt.frames > 0 and k >= opt.frames:
            break
        out.append((r0 + k, d0 + k))
        k += 1
    return out


def shard_range(n: int, rank: int, world: int) -> range:
    """Contiguous shard of `n` frame pairs for `rank` of `world` (sizes differ by at most one)."""
    base, rem = divmod(n, world)
    start = rank * base + min(rank, rem)
    return range(start, start + base + (1 if rank < rem else 0))


def gather_scores(local: Sequence[float], n_total: int, rank: int, world: int, group=None) -> Optional[List[float]]:
    """Ordered per-frame score stream on rank 0 (None elsewhere).  Only 8 bytes per frame cross the process
    boundary; works on any torch.distributed backend (nccl on GPUs, gloo in the CPU tests)."""
    if world == 1:
        return list(local)
    import torch
    import torch.distributed as dist
    dev = "cuda" if dist.get_backend(group) == "nccl" else "cpu"
    sizes = [len(shard_range(n_total, r, world)) for r in range(world)]
    mx = max(sizes)
    buf = torch.full((mx,), float("nan"), dtype=torch.float64, device=dev)
    buf[: len(local)] = torch.tensor(list(local), dtype=torch.float64, device=dev)
    out = [torch.empty_like(buf) for _ in range(world)] if rank == 0 else None
    dist.gather(buf, out, dst=0, group=group)
    if rank != 0:
        return None
    res: List[float] = []
    for r in range(world):
        res.extend(out[r][: sizes[r]].cpu().tolist())
    return res


class TurboMetrics:
    """`TurboMetrics::new(width, height, &Metrics)` (lib.rs:201-251) for metrics = {ssimulacra2}."""

    def __init__(self, width: int, height: int, fmt: PixelFormat, matrix: ColorMatrix = ColorMatrix.BT709,
                 full_range: bool = False, device: int = 0, batch: int = 0, ring: int = 0, score_only: bool = True,
                 bit_depth: Optional[int] = None, dis_fmt: Optional[PixelFormat] = None, dis_matrix: Optional[ColorMatrix] = None,
                 dis_full_range: Optional[bool] = None, dis_bit_depth: Optional[int] = None, dis_width: Optional[int] = None,
                 dis_height: Optional[int] = None):
        """score_only: the engine only ever hands out scores (`FrameScores`), so it asks the scorer for nothing else
        (SSIMU2_FLAG_SCORE_ONLY: same score bits, ~8 % faster).  bit_depth: of the decoded stream (the reference reads it from the
        stream's colour info, turbo-metrics/src/lib.rs:185-199); P016 / P216 / YUV444P16 frames of a stream deeper than 10 bits select the
        front-end without the 10-bit memo tables (SSIMU2_FLAG_P016_DEEP).
        dis_fmt, dis_matrix, dis_full_range, dis_bit_depth: the distorted source's own frame format and colour characteristics
        (None = as the reference), the `compute_one(fref, cc_ref, fdis, cc_dis)` shape of lib.rs:268-360; `bit_depth` then
        applies to the reference side and `dis_bit_depth` to the distorted side.
        dis_width, dis_height: the distorted source's frame size when it is a lower rung of an encoding ladder (smaller than
        width x height): its frames are upscaled to the reference's size on the GPU before they are scored."""
        deep = fmt in YUV16_FORMATS and bit_depth is not None and bit_depth > 10
        dfmt = fmt if dis_fmt is None else dis_fmt
        dis_deep = None if dis_bit_depth is None else (dfmt in YUV16_FORMATS and dis_bit_depth > 10)
        self.ssimulacra2 = Ssimulacra2(width, height, fmt, matrix, full_range, device, batch, ring, score_only=score_only,
                                       p016_deep=deep, dis_fmt=dis_fmt, dis_matrix=dis_matrix, dis_full_range=dis_full_range,
                                       dis_p016_deep=dis_deep, dis_width=dis_width, dis_height=dis_height)
        info = self.ssimulacra2.info()
        self.window = info.batch * info.ring

    def close(self):
        self.ssimulacra2.close()

    def compute_one(self, fref: DeviceFrame, fdis: DeviceFrame, stream=None) -> FrameScores:
        """lib.rs:268-360."""
        return FrameScores(ssimulacra2=self.ssimulacra2.compute_sync(fref, fdis, stream))

    def compute_all(self, frames_ref: Iterable[DeviceFrame], frames_dis: Iterable[DeviceFrame], opts: Optional[Options] = None,
                    stream=None) -> MetricsResults:
        """The frame loop of lib.rs:362-433 with the same `Options` semantics (lib.rs:385-400): skip `skip + skip_ref` /
        `skip + skip_dis` frames of the two sources, then walk them in lockstep; with `decode_count` counting the pairs seen,
        score a pair unless `every > 1 and decode_count != 0 and decode_count % every != 0`, stop at the first candidate
        with `decode_count >= frames` (frames > 0), or when either source ends.  Re-done for throughput: up to
        batch x ring pairs are in flight, scores are collected in submission order.

        LIFETIME: a yielded frame is read when its batch is launched, not when it is submitted -- every frame must own
        its memory until its score has been collected (this loop keeps the DeviceFrame objects alive for that long);
        a source that recycles a small buffer pool has to order the reuse with `Ssimulacra2.wait_input(ticket, stream)`."""
        opts = opts or Options()
        it_ref, it_dis = iter(frames_ref), iter(frames_dis)
        for _ in range(opts.skip_ref + opts.skip):       # FrameSource::skip_frames
            next(it_ref, None)
        for _ in range(opts.skip_dis + opts.skip):
            next(it_dis, None)
        scores: List[float] = []
        pending: List[int] = []
        decode_count = 0
        for fref, fdis in zip(it_ref, it_dis):
            if opts.every > 1 and decode_count != 0 and decode_count % opts.every != 0:
                decode_count += 1
                continue
            if opts.frames > 0 and decode_count >= opts.frames:
                break
            decode_count += 1
            pending.append(self.ssimulacra2.compute(fref, fdis, stream))
            if len(pending) >= self.window:
                scores.append(self.ssimulacra2.get_score(pending.pop(0)))
        self.ssimulacra2.flush()
        scores.extend(self.ssimulacra2.get_score(t) for t in pending)
        from .stats import Stats
        return MetricsResults(len(scores), MetricAggregate(scores, Stats.compute(scores)) if scores else None)


class ShardedTurboMetrics:
    """The frame loop over every GPU of the box, one process (the reference drives device 0 only, lib.rs:438-456).  Frames are
    HOST frames (decoded / loaded on the CPU: turbo-metrics/src/input_image.rs:206-228 copies each frame itself)."""

    def __init__(self, width: int, height: int, fmt: PixelFormat, devices: Sequence[int], matrix: ColorMatrix = ColorMatrix.BT709,
                 full_range: bool = False, batch: int = 0, ring: int = 0, score_only: bool = True,
                 dis_fmt: Optional[PixelFormat] = None, dis_matrix: Optional[ColorMatrix] = None, dis_full_range: Optional[bool] = None,
                 dis_width: Optional[int] = None, dis_height: Optional[int] = None):
        """dis_fmt, dis_matrix, dis_full_range: the distorted source's own description (None = as the reference); dis_width,
        dis_height: its frame size when smaller than the reference's (upscaled on the GPU)."""
        self.sharded = ShardedSsimulacra2(width, height, fmt, devices, matrix, full_range, batch, ring, score_only,
                                          dis_fmt=dis_fmt, dis_matrix=dis_matrix, dis_full_range=dis_full_range,
                                          dis_width=dis_width, dis_height=dis_height)
        self.chunk = max(1, (batch or 8) * len(devices))
        self.window = self.chunk * max(2, ring or 3)

    def close(self):
        self.sharded.close()

    def compute_all(self, frames_ref: Iterable[DeviceFrame], frames_dis: Iterable[DeviceFrame], opts: Optional[Options] = None) -> MetricsResults:
        """Same `Options` semantics as `TurboMetrics.compute_all`; pairs are submitted in chunks of one batch per GPU and at most
        `window` pairs are in flight.  Every yielded frame must own its (host) memory until its score has been collected."""
        opts = opts or Options()
        it_ref, it_dis = iter(frames_ref), iter(frames_dis)
        for _ in range(opts.skip_ref + opts.skip):
            next(it_ref, None)
        for _ in range(opts.skip_dis + opts.skip):
            next(it_dis, None)
        scores: List[float] = []
        pending: List[range] = []
        inflight = 0
        cr: List[DeviceFrame] = []
        cd: List[DeviceFrame] = []

        def push():
            nonlocal inflight
            if cr:
                pending.append(self.sharded.submit_host(list(cr), list(cd)))
                inflight += len(cr)
                cr.clear(); cd.clear()
            while inflight > self.window and pending:
                t = pending.pop(0)
                scores.extend(self.sharded.get_scores(t).tolist())
                inflight -= len(t)
        decode_count = 0
        for fref, fdis in zip(it_ref, it_dis):
            if opts.every > 1 and decode_count != 0 and decode_count % opts.every != 0:
                decode_count += 1
                continue
            if opts.frames > 0 and decode_count >= opts.frames:
                break
            decode_count += 1
            cr.append(fref); cd.append(fdis)
            if len(cr) >= self.chunk:
                push()
        push()
        self.sharded.flush()
        for t in pending:
            scores.extend(self.sharded.get_scores(t).tolist())
        from .stats import Stats
        return MetricsResults(len(scores), MetricAggregate(scores, Stats.compute(scores)) if scores else None)
