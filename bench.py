#!/usr/bin/env python
"""bench.py -- SSIMULACRA2 frame-pairs/s on B200 (BASELINE.json metric), one JSON line on stdout.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload 4k|1080p|512|1080p_srgb8] [--impl ours|reference]
                  [--dump-outputs DIR]
  N > 1:  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...
          (or, one process for all GPUs through the C ABI's own sharding: python bench.py --gpus N --shard-api)

A "step" is one pass of the hot path over the workload's frame sequence (300 synthetic pairs per GPU,
SURVEY.md section 8d).  Frames are sharded over the ranks with no data-path collective (weak scaling:
every rank scores its own 300 pairs); only scalar scores leave a GPU.

  value      pairs/s with the frames already resident in HBM when the timed region starts
             (device frames through the C ABI, ssimu2_submit_batch + ssimu2_get_scores)
  e2e        the same metric through the host-frame entry point of the C ABI (ssimu2_submit_host):
             pinned HOST buffers, host->device copies and the score read-back inside the timed region;
             beside it the raw host->device rate of the same buffers with no kernels (what the link gives)
  roofline   frac = B_alg (the contract's two-global-pass traffic model, SURVEY 8d) x measured pairs/s / measured HBM peak
             -- the figure BASELINE.json's ">= 60 % of the HBM roofline" is stated in.  What actually binds each kernel
             (FP64 pipe + issue in the front-end, FP32 pipe in k_hv), its achieved fraction of THAT resource and its real
             DRAM rate are under roofline.kernels; every number is recomputable from this line + profiles/.
  parity     the first pair of the timed sequence against the CPU oracle (108 norms <= 1e-4 relative, score <= 0.01);
             the run FAILS above the bar
  workloads  the other BASELINE.json configs (1080p NV12, 512x512 batch, 1080p sRGB8) measured in the same run
  cpu_baseline  the CPU oracle (a port of the reference's examples/cpu.rs; the Rust reference cannot be
             built here) on the host cores, one pair per thread, bounded sample
--impl reference times that oracle alone, on the same config, as the reference arm.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (w, h, kind, bits, description)
    "4k": (3840, 2160, "yuv", 16, "4K 10-bit YUV420 (P016) BT.709 limited, 300 synthetic pairs per GPU (BASELINE configs[2]/[3])"),
    "1080p": (1920, 1080, "yuv", 8, "1080p 8-bit YUV420 (NV12) BT.709 limited, 300 synthetic pairs per GPU (BASELINE configs[1])"),
    "512": (512, 512, "srgb8", 8, "512 synthetic 512x512 sRGB8 pairs in one submission, small-frame path (BASELINE configs[4])"),
    "1080p_srgb8": (1920, 1080, "srgb8", 8, "1920x1080 sRGB8 pairs (BASELINE configs[0] is one such pair through the CPU reference)"),
}
PAIRS_PER_STEP = {"4k": 300, "1080p": 300, "512": 512, "1080p_srgb8": 64}
DISTINCT = {"4k": 32, "1080p": 64, "512": 128, "1080p_srgb8": 32}   # distinct pairs cycled through a step (>> 126 MB L2)
BATCH = {"4k": 16, "1080p": 32, "512": 128, "1080p_srgb8": 32}
IN0 = {"4k": 6, "1080p": 3, "512": 6, "1080p_srgb8": 6}             # input bytes per pixel pair

# FP32-pipe operations of k_hv per pyramid pixel PAIR and channel (DESIGN.md section 4 counts them): 5 products, 5 x 12
# (horizontal filter step), 5 x 9 (vertical step), 22 (SSIM' map incl. the division), 13 (edge maps)
HV_FP32_OPS_PER_PX = 3 * (5 + 60 + 45 + 22 + 13)
# FP64-pipe operations of the front-end: 13 per cube root x 3 per XYB value, per image; 18 per transfer function (YUV only)
FE_FP64_PER_XYB, FE_FP64_PER_EOTF = 39, 18


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p))["hbm_gbs"], "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def kernel_source_hash():
    h = hashlib.sha256()
    for f in ("ssimu2_kernels.cuh", "exact_math.cuh"):
        h.update(open(os.path.join(ROOT, "turbo_metrics_b200", "csrc", f), "rb").read())
    return h.hexdigest()[:16]


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", os.environ.get("BENCH_SMI_MS", "100")], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        # the samples span idle gaps too: take the median of the upper half as "under load"
        load = sm[len(sm) // 2:] if sm else []
        return {"sm_mhz": load[len(load) // 2] if load else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def bind_to_gpu_numa(index):
    """Pin this process to the CPUs of the NUMA node the GPU hangs off, so that the pinned host buffers allocated afterwards
    (first touch) and the copy threads live next to the GPU's PCIe root.  Pure /sys reads; a no-op where unavailable."""
    out = {"node": None, "bound": False}
    try:
        import torch
        props = torch.cuda.get_device_properties(index)
        bdf = f"{props.pci_domain_id:04x}:{props.pci_bus_id:02x}:{props.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
        out["pci"] = bdf
        if node < 0:
            return out
        out["node"] = node
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            out["bound"], out["cpus"] = True, len(cpus)
    except Exception as e:   # measurement aid only
        out["error"] = repr(e)[:120]
    return out


# ------------------------------------------------------------------------------------------ CPU oracle arm
def oracle_pairs_per_s(workload, n_pairs, threads, frames=None):
    """Score n_pairs synthetic pairs (all copies of frame 0, seed 1 = the first pair rank 0 times on the GPU) with the CPU
    oracle, one pair per thread; returns (pairs/s, seconds, (score, norms[108]) of that pair)."""
    import torch  # noqa: F401
    from oracle import oracle
    from turbo_metrics_b200 import synth
    w, h, kind, bits, _ = WORKLOADS[workload]
    oracle.lib()
    # frames: the very bytes the GPU scored (copied back from the device: torch's device and host generators are not
    # bit-identical in sin/cos, so a host re-generation of "the same" frame differs in a few samples)
    if kind == "yuv":
        if frames is None:
            rb, db, pitch, ch = synth.make_pair_yuv420(w, h, bits, frame=0, seed=1)
            rn, dn = rb.numpy(), db.numpy()
        else:
            rn, dn, pitch, ch = frames
        job = lambda: oracle.ssimu2_yuv420(rn, dn, pitch, ch, w, h, bits)[:2]
    else:
        if frames is None:
            r, d = synth.make_pair_srgb8(w, h, frame=0, seed=1)
            rn, dn = r.numpy(), d.numpy()
        else:
            rn, dn = frames
        job = lambda: oracle.ssimu2_srgb8(rn, dn)[:2]
    out = [None] * n_pairs
    idx = iter(range(n_pairs))
    lock = threading.Lock()

    def worker():
        while True:
            with lock:
                i = next(idx, None)
            if i is None:
                return
            out[i] = job()
    ts = [threading.Thread(target=worker) for _ in range(min(threads, n_pairs))]
    t0 = time.perf_counter()
    [t.start() for t in ts]
    [t.join() for t in ts]
    dt = time.perf_counter() - t0
    return n_pairs / dt, dt, out[0]


def run_reference(args, rank, world):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    threads = min(cores, 32)
    w, h, kind, bits, desc = WORKLOADS[args.workload]
    sample = threads if args.workload != "512" else threads * 8
    for _ in range(args.warmup):
        oracle_pairs_per_s(args.workload, max(1, min(sample, 2)), threads)
    vals, secs = [], 0.0
    for _ in range(args.steps):
        v, dt, _ = oracle_pairs_per_s(args.workload, sample, threads)
        vals.append(v); secs += dt
    value = sample * args.steps / secs
    line = {
        "impl": "reference", "metric": "ssimulacra2_frame_pairs_per_s", "value": value, "unit": "pairs/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * secs / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32+f64", "data": "synthetic",
        "config": {"workload": desc, "width": w, "height": h, "note": "reference Rust crate cannot be built here (no rustc); "
                   "this is the C port of its examples/cpu.rs + biplanar.rs (oracle/), one pair per host thread"},
        "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": threads, "kind": "port",
                         "sample": f"{sample} pairs per step x {args.steps} steps of the same {w}x{h} workload"},
        "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------------ GPU arm
class Ctx:
    pass


def parity_block(norms_gpu, score_gpu, o_score, o_norms, what):
    import numpy as np
    nz = o_norms != 0
    rel = np.zeros(108)
    rel[nz] = np.abs(norms_gpu[nz] - o_norms[nz]) / np.abs(o_norms[nz])
    rel[~nz] = np.abs(norms_gpu[~nz])
    p = {"pair": what, "score_gpu": float(score_gpu), "score_oracle": float(o_score), "dscore": float(abs(score_gpu - o_score)),
         "max_rel_norm": float(rel.max()), "bar": {"dscore": 0.01, "max_rel_norm": 1e-4}}
    assert p["dscore"] <= 0.01 and p["max_rel_norm"] <= 1e-4, p
    return p


def measure(c, workload, steps, warmup, batch, ring, e2e_steps, with_clocks=True, score_only=None, outputs=False):
    """One workload on this rank's GPU: device-resident throughput, e2e from pinned host buffers + the raw H2D rate, per-kernel
    device times (ring = 1), the first pair's score + norms.  Returns a dict (times are max over ranks).
    e2e_steps = 0 skips the host-buffer legs (used for the score-only sub-result, whose e2e is the same PCIe-bound figure).
    outputs = True also returns the scores and (outside score-only mode) the norms of every pair of the last timed step."""
    score_only = c.args.score_only if score_only is None else score_only
    torch, tm, synth, dist = c.torch, c.tm, c.synth, c.dist
    w, h, kind, bits, desc = WORKLOADS[workload]
    n_pairs, n_distinct = PAIRS_PER_STEP[workload], DISTINCT[workload]
    fmt = {("yuv", 8): tm.PixelFormat.NV12, ("yuv", 16): tm.PixelFormat.P016, ("srgb8", 8): tm.PixelFormat.SRGB8}[(kind, bits)]
    dev = c.dev
    # ---- synthetic frames, resident in HBM (each rank its own shard: seed includes the rank)
    dev_frames = []
    pitch = ch = None
    for i in range(n_distinct):
        if kind == "yuv":
            rb, db, pitch, ch = synth.make_pair_yuv420(w, h, bits, frame=i, seed=1 + c.rank, device=dev)
        else:
            rb, db = synth.make_pair_srgb8(w, h, frame=i, seed=1 + c.rank, device=dev)
        dev_frames.append((rb, db))
    mk = (lambda t: tm.DeviceFrame.yuv420(t, pitch, ch)) if kind == "yuv" else tm.DeviceFrame.packed
    n_host = min(n_distinct, 16)
    host_frames = [(dev_frames[i][0].cpu().pin_memory(), dev_frames[i][1].cpu().pin_memory()) for i in range(n_host)]
    frame_bytes = dev_frames[0][0].numel() * dev_frames[0][0].element_size()
    refs = [mk(dev_frames[i % n_distinct][0]) for i in range(n_pairs)]
    diss = [mk(dev_frames[i % n_distinct][1]) for i in range(n_pairs)]
    hrefs = [mk(host_frames[i % n_host][0]) for i in range(n_pairs)]
    hdiss = [mk(host_frames[i % n_host][1]) for i in range(n_pairs)]

    m = tm.Ssimulacra2(w, h, fmt, device=c.local_rank, batch=batch, ring=ring, score_only=score_only)
    info = m.info()
    stream = torch.cuda.current_stream()

    # A step = submit the step's pairs, then fetch their scores.  Like the reference's frame loop (compute() is asynchronous,
    # get_score() comes later), the timed loop fetches the scores of step i after step i+1 has been submitted, so the
    # batch ring never drains between steps; every submit and every fetch of the K steps is inside the timed region.
    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, nsteps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        t0 = time.perf_counter()
        e0.record(stream)
        prev = None
        for _ in range(nsteps):
            ts = fn()
            if prev is not None:
                m.get_scores(prev)
            prev = ts
        timed.tickets, timed.scores = prev, m.get_scores(prev)
        # get_scores() has synchronised every batch stream with the host; mark the end on the device clock
        e1.record(stream)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        barrier()
        ms_event = max(e0.elapsed_time(e1), 0.0)
        # every batch stream waits on the submit stream (so all work starts after e0) and get_scores() has synchronised every
        # batch with the host before e1 is recorded: the CUDA-event interval covers the whole region; the host clock around
        # the same synchronised region is kept as a cross-check, the larger one wins
        ms = max(ms_event, wall * 1000.0)
        timed.last = {"event_ms": ms_event, "wall_ms": wall * 1000.0}
        if dist is not None:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    submit_device = lambda: m.compute_batch(refs, diss, stream)
    submit_host = lambda: m.compute_from_cpu_batch(hrefs, hdiss)
    for _ in range(warmup):
        m.get_scores(submit_device())
    l0 = m.info().kernel_launches
    sampler = ClockSampler(c.local_rank).start() if (with_clocks and c.rank == 0 and not os.environ.get("BENCH_NO_CLOCKS")) else None
    ms = timed(submit_device, steps)
    timing = dict(timed.last)
    clocks = sampler.stop() if sampler else None
    launches = m.info().kernel_launches - l0
    value = c.world * n_pairs * steps / (ms / 1000.0)
    last_step = None
    if outputs:
        import numpy as np
        last_step = {"scores": timed.scores}
        if not score_only:
            # the library keeps the results of its last 16384 tickets on the host: no device work after the timed region
            last_step["norms"] = np.stack([m.get_norms(t) for t in timed.tickets])

    e2e = None
    # ---- e2e: host frames through the C ABI, and the raw H2D rate of the same buffers (no kernels) for comparison
    for _ in range(max(1, warmup // 2) if e2e_steps else 0):
        m.get_scores(submit_host())
    stage = None
    if e2e_steps:
        ms_e2e = timed(submit_host, e2e_steps)
        e2e_value = c.world * n_pairs * e2e_steps / (ms_e2e / 1000.0)
        stage = [torch.empty_like(dev_frames[0][0]) for _ in range(4)]
        n_raw = min(n_pairs, 128)

        def raw_h2d():
            for i in range(n_raw):
                stage[(2 * i) % 4].copy_(host_frames[i % n_host][0], non_blocking=True)
                stage[(2 * i + 1) % 4].copy_(host_frames[i % n_host][1], non_blocking=True)
        raw_h2d()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream); raw_h2d(); e1.record(stream)
        torch.cuda.synchronize()
        raw_ms = e0.elapsed_time(e1)
        if dist is not None:
            t = torch.tensor([raw_ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            raw_ms = float(t.item())
        raw_gbs = c.world * 2 * frame_bytes * n_raw / (raw_ms / 1e3) / 1e9
        e2e = {"value": e2e_value, "unit": "pairs/s", "h2d_bytes_per_step": 2 * frame_bytes * n_pairs,
               "d2h_bytes_per_step": 8 * n_pairs * (1 if score_only else 109), "steps": e2e_steps,
               "h2d_gbs": e2e_value * 2 * frame_bytes / 1e9, "h2d_gbs_raw": raw_gbs,
               "note": "ssimu2_submit_host_batch from pinned host buffers (aggregate over all ranks); h2d_gbs_raw = the same buffers "
                       "copied with no kernels running, all ranks at once: when the two agree the limiter is the host->device path"}

    # ---- score + norms of the first pair of the sequence (for the parity block)
    ts_chk = submit_device()
    sc = m.get_scores(ts_chk)
    s_first, s_last = float(sc[0]), float(sc[-1])
    assert 0.0 < s_first <= 100.0 and 0.0 < s_last <= 100.0, (s_first, s_last)
    norms_first = None if score_only else m.get_norms(ts_chk[0])
    m.close()

    # ---- per-kernel device time without cross-stream overlap: same batch size, ring = 1
    m1 = tm.Ssimulacra2(w, h, fmt, device=c.local_rank, batch=batch, ring=1, score_only=score_only)
    for _ in range(2):
        m1.get_scores(m1.compute_batch(refs[:2 * batch], diss[:2 * batch], stream))
    m1.kernel_ms(reset=True)
    sc1 = m1.get_scores(m1.compute_batch(refs, diss, stream))
    kms, kbatches, kpairs = m1.kernel_ms()
    m1.close()
    assert float(sc1[0]) == s_first, "score depends on the batch slot"
    del dev_frames, host_frames, stage
    torch.cuda.empty_cache()
    return {"workload": workload, "desc": desc, "w": w, "h": h, "kind": kind, "bits": bits, "value": value, "ms": ms, "steps": steps,
            "warmup": warmup, "timing": timing, "clocks": clocks, "launches": int(launches), "e2e": e2e, "info": info,
            "frame_bytes": frame_bytes, "n_pairs": n_pairs, "n_distinct": n_distinct, "kms": kms, "kbatches": kbatches, "kpairs": kpairs,
            "s_first": s_first, "s_last": s_last, "norms_first": norms_first, "pitch": pitch, "ch": ch,
            "last_step": last_step}


def roofline_block(c, r):
    """The contract's block (bound / achieved / peak / frac / traffic) + what really binds each kernel."""
    info, world = r["info"], c.world
    peak, peak_src = peaks()
    alg, io = info.alg_bytes_per_pair, info.io_bytes_per_pair
    px = [info.width[s] * info.height[s] for s in range(info.nscales)]
    pairs_per_launch = r["kpairs"] / r["kbatches"]
    ms_fe, ms_hv, _, ms_fin = [x / r["kbatches"] for x in r["kms"]]
    group_ms = ms_fe + ms_hv + ms_fin
    per_gpu = r["value"] / world
    achieved = alg * per_gpu / 1e9
    clk_mhz = (r["clocks"] or {}).get("sm_mhz") or (r["clocks"] or {}).get("sm_max_mhz") or 1965.0
    sms = c.torch.cuda.get_device_properties(c.local_rank).multi_processor_count
    # ---- measured DRAM bytes per pair per kernel: from the committed ncu capture, valid only for the same kernel source
    tr, tr_note = {}, "no ncu capture committed for this workload"
    tf = os.path.join(ROOT, "profiles", "traffic_r2.json")
    if os.path.exists(tf):
        ent = json.load(open(tf)).get(r["workload"])
        if ent:
            tr = ent.get("dram_bytes_per_pair", {})
            tr_note = f"ncu --set full capture {ent.get('report')} (profiles/{ent.get('summary')}), kernel source {ent.get('source_hash')}"
            if ent.get("source_hash") != kernel_source_hash():
                tr_note += f" -- STALE: the kernels have changed since (now {kernel_source_hash()})"
    in0 = IN0[r["workload"]]
    pass_bytes = 60 * sum(px) + in0 * px[0] + 24 * sum(px[1:])
    kalg = {"k_frontend2": 24 * sum(px[1:]), "k_hv": 2 * pass_bytes}
    assert sum(kalg.values()) == alg, (kalg, alg)
    fe_fp64 = 2 * (FE_FP64_PER_XYB * sum(px) + (FE_FP64_PER_EOTF * px[0] if r["kind"] == "yuv" else 0))
    hv_fp32 = HV_FP32_OPS_PER_PX * sum(px)
    lanes32, lanes64 = sms * 128 * clk_mhz * 1e6, sms * 64 * clk_mhz * 1e6
    kernels = {
        "k_frontend2": {
            "ms_per_launch": ms_fe, "share_of_launch_group": ms_fe / group_ms,
            "bound": "fp64_pipe latency + issue (bit-exact cbrtf / powf: 23-cycle FP64 dependent-issue latency, 4 warps per scheduler at 128 registers)",
            "fp64_ops_per_pair": fe_fp64, "fp64_pipe_frac": fe_fp64 * pairs_per_launch / (ms_fe / 1e3) / lanes64,
            "alg_bytes_per_pair": kalg["k_frontend2"], "dram_bytes_per_pair_ncu": tr.get("k_frontend2"),
            "dram_frac_real": (tr["k_frontend2"] * pairs_per_launch / (ms_fe / 1e3) / 1e9 / peak) if tr.get("k_frontend2") else None},
        "k_hv": {
            "ms_per_launch": ms_hv, "share_of_launch_group": ms_hv / group_ms,
            "bound": "fp32_pipe (packed FFMA2/FADD2/FMUL2 are half rate: 128 lane-ops per clock per SM either way)",
            "fp32_ops_per_pair": hv_fp32, "fp32_pipe_frac": hv_fp32 * pairs_per_launch / (ms_hv / 1e3) / lanes32,
            "alg_bytes_per_pair": kalg["k_hv"], "dram_bytes_per_pair_ncu": tr.get("k_hv"),
            "dram_frac_real": (tr["k_hv"] * pairs_per_launch / (ms_hv / 1e3) / 1e9 / peak) if tr.get("k_hv") else None},
        "k_finalize": {"ms_per_launch": ms_fin, "share_of_launch_group": ms_fin / group_ms},
    }
    dom = "k_hv" if ms_hv >= ms_fe else "k_frontend2"
    real = sum(v for v in tr.values()) if tr else None
    return {
        "bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
        "traffic": (tr[dom] * pairs_per_launch) if tr.get(dom) else None, "peak_source": peak_src,
        "basis": "contract figure: B_alg (SURVEY 8d, the DRAM traffic of the prescribed two-global-pass design) x measured pairs/s per GPU "
                 "of the timed loop / measured HBM copy peak.  It is a throughput yardstick, NOT this design's limiter: the fused kernels "
                 "move far fewer bytes (dram_bytes_per_pair_real) and are bound by arithmetic pipes (kernels.*.bound)",
        "alg_bytes_per_pair": alg, "io_bytes_per_pair": io, "dram_bytes_per_pair_real": real,
        "dram_frac_real": (real * per_gpu / 1e9 / peak) if real else None, "traffic_source": tr_note,
        "launch_group": {"pairs_per_launch": pairs_per_launch, "ms": group_ms, "pairs_per_s_no_overlap": pairs_per_launch / (group_ms / 1e3),
                         "frac_no_overlap": alg * pairs_per_launch / (group_ms / 1e3) / 1e9 / peak,
                         "note": "CUDA-event times of the three kernels of one launch group, ring = 1 (no cross-batch overlap)"},
        "sm_clock_mhz_used": clk_mhz, "sms": sms, "kernels": kernels,
    }


def run_shard_api(args):
    """One process, N GPUs, through ssimu2_shard_* (one handle + host thread per device inside the library): no torch.distributed."""
    import torch
    import turbo_metrics_b200 as tm
    from turbo_metrics_b200 import synth
    n = args.gpus
    assert torch.cuda.device_count() >= n, f"--shard-api needs {n} visible GPUs"
    workload = args.workload
    w, h, kind, bits, desc = WORKLOADS[workload]
    fmt = {("yuv", 8): tm.PixelFormat.NV12, ("yuv", 16): tm.PixelFormat.P016, ("srgb8", 8): tm.PixelFormat.SRGB8}[(kind, bits)]
    batch = args.batch or BATCH[workload]
    # device frames must live on the GPU their ticket is routed to ((ticket / batch) % n): a step of a whole number of
    # batch x n rounds keeps that routing identical from step to step
    n_pairs, n_distinct = -(-PAIRS_PER_STEP[workload] * n // (batch * n)) * batch * n, DISTINCT[workload]
    devs = list(range(n))
    frames = {}
    pitch = ch = None
    for d in devs:
        frames[d] = []
        for i in range(n_distinct):
            if kind == "yuv":
                rb, db, pitch, ch = synth.make_pair_yuv420(w, h, bits, frame=i, seed=1, device=f"cuda:{d}")
            else:
                rb, db = synth.make_pair_srgb8(w, h, frame=i, seed=1, device=f"cuda:{d}")
            frames[d].append((rb, db))
        torch.cuda.synchronize(d)
    mk = (lambda t: tm.DeviceFrame.yuv420(t, pitch, ch)) if kind == "yuv" else tm.DeviceFrame.packed
    n_host = 16
    host = [(frames[0][i][0].cpu().pin_memory(), frames[0][i][1].cpu().pin_memory()) for i in range(n_host)]
    frame_bytes = host[0][0].numel() * host[0][0].element_size()
    with tm.ShardedSsimulacra2(w, h, fmt, devices=devs, batch=batch, ring=args.ring, score_only=args.score_only) as sh:
        refs = [mk(frames[sh.device_of(g)][g % n_distinct][0]) for g in range(n_pairs)]
        diss = [mk(frames[sh.device_of(g)][g % n_distinct][1]) for g in range(n_pairs)]
        hrefs = [mk(host[g % n_host][0]) for g in range(n_pairs)]
        hdiss = [mk(host[g % n_host][1]) for g in range(n_pairs)]

        def run(fn, steps):
            prev = None
            t0 = time.perf_counter()
            for _ in range(steps):
                ts = fn()
                if prev is not None:
                    sh.get_scores(prev)
                prev = ts
            sc = sh.get_scores(prev)
            return time.perf_counter() - t0, sc
        for _ in range(args.warmup):
            run(lambda: sh.submit_device(refs, diss), 1)
        sampler = ClockSampler(0).start()
        dt, sc = run(lambda: sh.submit_device(refs, diss), args.steps)
        clocks = sampler.stop()
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"scores": sc})
        run(lambda: sh.submit_host(hrefs, hdiss), 1)
        e2e_steps = max(1, min(args.steps, 2))
        dt_h, sc_h = run(lambda: sh.submit_host(hrefs, hdiss), e2e_steps)
    value = n_pairs * args.steps / dt
    peak, peak_src = peaks()
    with tm.Ssimulacra2(w, h, fmt, device=0, batch=1, ring=1) as m0:
        alg = m0.info().alg_bytes_per_pair
    emit({
        "metric": "ssimulacra2_frame_pairs_per_s", "value": value, "unit": "pairs/s", "n_gpus": n, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 (+f64 seed/tails)", "data": "synthetic",
        "config": {"workload": desc, "width": w, "height": h, "pairs_per_step": n_pairs, "batch": batch, "ring": args.ring,
                   "parallelism": f"ssimu2_shard_*: ONE process, {n} GPUs, one handle + host thread per device inside the library, no collective",
                   "timing": "host wall clock around submit + ordered fetch (the shard API has no single device stream to put events on)"},
        "e2e": {"value": n_pairs * e2e_steps / dt_h, "unit": "pairs/s", "h2d_bytes_per_step": 2 * frame_bytes * n_pairs,
                "d2h_bytes_per_step": 8 * n_pairs * 109, "steps": e2e_steps},
        "gpu_launches": None, "clocks": clocks,
        "roofline": {"bound": "hbm", "achieved": alg * value / n / 1e9, "peak": peak, "unit": "GB/s", "frac": alg * value / n / 1e9 / peak,
                     "traffic": None, "peak_source": peak_src, "basis": "B_alg x pairs/s per GPU / HBM peak (contract figure)"},
        "scores": {"first": float(sc[0]), "last": float(sc[-1]), "host_first": float(sc_h[0])},
    })


def run_ours(args, rank, world, local_rank):
    import torch
    import turbo_metrics_b200 as tm
    from turbo_metrics_b200 import synth
    c = Ctx()
    c.args, c.rank, c.world, c.local_rank, c.torch, c.tm, c.synth = args, rank, world, local_rank, torch, tm, synth
    c.dist = None
    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa(local_rank) if not args.no_numa_bind else {"bound": False, "note": "--no-numa-bind"}
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        c.dist = dist
    c.dev = torch.device("cuda", local_rank)
    workload = args.workload
    w, h, kind, bits, desc = WORKLOADS[workload]
    batch = args.batch or BATCH[workload]
    r = measure(c, workload, args.steps, args.warmup, batch, args.ring, max(1, min(args.steps, 3)), outputs=bool(args.dump_outputs))
    if args.dump_outputs:
        suffix = "" if world == 1 else f"_rank{rank}"
        dump_outputs(args.dump_outputs, {k + suffix: v for k, v in r["last_step"].items()})

    # ---- the other BASELINE configs, measured in the same run (fewer steps: they are sub-results, not the headline)
    subs = {}
    if not args.no_workloads and workload == "4k":
        for wl in ("1080p", "512", "1080p_srgb8"):
            subs[wl] = measure(c, wl, 3, 3, BATCH[wl], args.ring, 2, with_clocks=True)
    # ---- the same workload with SSIMU2_FLAG_SCORE_ONLY (the reference's API returns the score only; the flag drops the
    # filters and maps whose weights are zero): device-resident throughput, and the score must have the same BITS
    somode = None
    if not args.score_only and not args.no_workloads:
        somode = measure(c, workload, 3, 3, batch, args.ring, 0, with_clocks=False, score_only=True)
        assert somode["s_first"] == r["s_first"] and somode["s_last"] == r["s_last"], "score-only mode changed a score"
    if rank != 0:
        return

    roof = roofline_block(c, r)
    cores = os.cpu_count() or 1
    threads = min(cores, 32)
    parity = None
    if args.no_cpu_baseline:
        cpu = {"value": None, "unit": "pairs/s", "cores": threads, "kind": "port", "sample": "skipped (--no-cpu-baseline)"}
    else:
        # the first pair of the timed sequence: regenerate its device buffers (same seed => same bytes) and copy them back
        def first_pair(wl):
            ww, hh, kk, bb, _ = WORKLOADS[wl]
            if kk == "yuv":
                rb, db, pitch, ch = synth.make_pair_yuv420(ww, hh, bb, frame=0, seed=1 + rank, device=c.dev)
                return (rb.cpu().numpy(), db.cpu().numpy(), pitch, ch)
            rb, db = synth.make_pair_srgb8(ww, hh, frame=0, seed=1 + rank, device=c.dev)
            return (rb.cpu().numpy(), db.cpu().numpy())
        sample = max(2, min(threads, 16)) if workload != "512" else threads * 8
        cv, cdt, (o_score, o_norms) = oracle_pairs_per_s(workload, sample, threads, first_pair(workload))
        cpu = {"value": cv, "unit": "pairs/s", "cores": min(threads, sample), "kind": "port",
               "sample": f"{sample} pairs of the same {w}x{h} workload, one pair per thread, {cdt:.1f} s"}
        what = "first pair of the timed sequence (frame 0, seed 1), the device buffers copied back for the oracle"
        if r["norms_first"] is not None:
            parity = parity_block(r["norms_first"], r["s_first"], o_score, o_norms, what)
        else:
            parity = {"pair": what, "score_gpu": r["s_first"], "score_oracle": float(o_score), "dscore": abs(r["s_first"] - o_score),
                      "max_rel_norm": None, "note": "score-only mode: no norms"}
            assert parity["dscore"] <= 0.01, parity
        for wl, sr in subs.items():
            _, _, (so, no) = oracle_pairs_per_s(wl, 1, 1, first_pair(wl))
            sr["parity"] = parity_block(sr["norms_first"], sr["s_first"], so, no, what) if sr["norms_first"] is not None else \
                {"dscore": abs(sr["s_first"] - so), "score_gpu": sr["s_first"], "score_oracle": float(so)}

    # ---- the reference's GPU design (NPP + per-sample kernels + one graph launch and one host sync per pair) restated in
    # baseline/refgpu and timed on this GPU on a bounded sample of the same frames: measurement tooling (SURVEY 8f row 3)
    refdesign = None
    if kind == "yuv" and not args.no_refgpu and world == 1:
        try:
            from baseline.refgpu import refgpu
            if os.path.exists(refgpu.SO_PATH):
                n_ref = 64 if workload == "4k" else 128
                fr = [synth.make_pair_yuv420(w, h, bits, frame=i, seed=1, device=c.dev) for i in range(8)]
                with refgpu.RefGpu(w, h, bits) as rg:
                    for i in range(4):
                        rg.compute(fr[i % 8][0], fr[i % 8][1], fr[0][2], fr[0][3])
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    rs = [rg.compute(fr[i % 8][0], fr[i % 8][1], fr[0][2], fr[0][3])[0] for i in range(n_ref)]
                    rdt = time.perf_counter() - t0
                    rinfo = rg.info()
                refdesign = {"value": n_ref / rdt, "unit": "pairs/s", "sample": f"{n_ref} pairs of the same workload, device frames",
                             "kernel_nodes_per_pair": rinfo["kernel_nodes"] + 2, "workspace_bytes": rinfo["bytes"],
                             "score_first": rs[0], "speedup_of_value": r["value"] / (n_ref / rdt),
                             "note": "baseline/refgpu: the reference's design (ssimulacra2-cuda/src/lib.rs:140-447) restated with NPP "
                                     "on this GPU; host sync per pair like TurboMetrics::compute_one; not the product path"}
        except Exception as e:   # tooling must never take the bench line down
            refdesign = {"unavailable": repr(e)[:200]}

    workloads = {}
    for wl, sr in subs.items():
        sroof = roofline_block(c, sr)
        workloads[wl] = {"desc": sr["desc"], "value": sr["value"], "unit": "pairs/s", "ms_per_step": sr["ms"] / sr["steps"], "steps": sr["steps"],
                         "warmup": sr["warmup"], "pairs_per_step_per_gpu": sr["n_pairs"], "batch": sr["info"].batch, "e2e": sr["e2e"],
                         "roofline_frac": sroof["frac"], "alg_bytes_per_pair": sr["info"].alg_bytes_per_pair,
                         "kernel_ms_per_launch": {k: v["ms_per_launch"] for k, v in sroof["kernels"].items()},
                         "fp32_pipe_frac_k_hv": sroof["kernels"]["k_hv"]["fp32_pipe_frac"], "clocks": sr["clocks"], "parity": sr.get("parity"),
                         "us_per_pair": 1e6 / (sr["value"] / world), "gpu_launches": sr["launches"]}
    info = r["info"]
    line = {
        "metric": "ssimulacra2_frame_pairs_per_s", "value": r["value"], "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": r["ms"] / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 (+f64 seed/tails)", "data": "synthetic",
        "config": {"workload": desc, "width": w, "height": h, "pairs_per_step_per_gpu": r["n_pairs"], "distinct_pairs": r["n_distinct"],
                   "batch": info.batch, "ring": info.ring, "score_only": bool(args.score_only),
                   "l2": f"inputs cycle through {r['n_distinct']} distinct pairs = {2 * r['frame_bytes'] * r['n_distinct'] / 1e6:.0f} MB per GPU "
                         "(> 126 MB L2); XYB planes + strip hand-off records are 0.33 GB per pair",
                   "step_pipelining": "scores of step i are fetched after step i+1 is submitted (all K submits and K fetches "
                                      "are inside the timed region)",
                   "parallelism": f"frame-sharded x{world}, no collective", "numa": numa},
        "e2e": r["e2e"],
        "gpu_launches": r["launches"],
        "clocks": r["clocks"],
        "roofline": roof,
        "cpu_baseline": cpu,
        "parity": parity,
        "workloads": workloads,
        "score_only_mode": None if somode is None else {
            "value": somode["value"], "unit": "pairs/s", "ms_per_step": somode["ms"] / somode["steps"], "steps": somode["steps"], "warmup": somode["warmup"],
            "roofline_frac": roofline_block(c, somode)["frac"],
            "kernel_ms_per_launch": {k: v["ms_per_launch"] for k, v in roofline_block(c, somode)["kernels"].items()},
            "scores_bit_equal_to_full_mode": True,
            "note": "same workload and timed loop as `value` with ssimu2_config.flags = SSIMU2_FLAG_SCORE_ONLY: the 54 zero-weight norms "
                    "are not computed (no ssimu2_get_norms); the run asserts the first and last score equal the full mode's bit for bit"},
        "gpu_reference_design": refdesign,
        "timing": r["timing"],
        "scores": {"first": r["s_first"], "last": r["s_last"]},
    }
    emit(line)


def dump_outputs(d, arrays):
    """Writes each array as d/<name>.npy in float64.  The inputs are seeded, so two builds run with the same arguments
    can be compared output for output."""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(d, name + ".npy"), np.asarray(a, dtype=np.float64))


_REAL_STDOUT = None


def _guard_stdout():
    """Libraries (NCCL's version banner, torchrun) write to fd 1; the contract is ONE JSON line on stdout.  Point fd 1 at
    stderr for the run and keep the real stdout for the final line."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, data)
    else:
        sys.stdout.write(data.decode()); sys.stdout.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="4k", choices=list(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="pairs per launch group (default: 16 at 4K, 32 at 1080p, 128 for 512x512)")
    ap.add_argument("--ring", type=int, default=3)
    ap.add_argument("--score-only", action="store_true", help="SSIMU2_FLAG_SCORE_ONLY: skip the zero-weight SSIM work (no norms)")
    ap.add_argument("--shard-api", action="store_true", help="one process for all --gpus through ssimu2_shard_* (no torchrun)")
    ap.add_argument("--no-workloads", action="store_true", help="skip the 1080p / 512 / sRGB8 sub-results")
    ap.add_argument("--no-numa-bind", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-refgpu", action="store_true", help="skip the reference-design GPU baseline (baseline/refgpu)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the scores of the last timed step to DIR/scores.npy and, "
                    "except with --score-only or --shard-api, their 108 norms each to DIR/norms.npy "
                    "(DIR/<name>_rank<r>.npy per rank under torchrun)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computed; --impl reference has no GPU path")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    _guard_stdout()
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.shard_api:
        if rank == 0:
            run_shard_api(args)
        return
    if args.gpus != world and world == 1 and args.gpus > 1:
        # convenience: re-launch under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", "29533", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd, stdout=_REAL_STDOUT))
    run_ours(args, rank, world, local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
