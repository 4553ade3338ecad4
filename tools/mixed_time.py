"""Throughput and per-kernel device time of mixed-source handles (ssimu2_create_mixed) beside the same-format handles of
their two sides.  Prints one JSON line.

Workloads: 4K NV12/NV12, P016/P016 and NV12 -> P016 (an 8-bit source against a 10-bit encode); 1080p SRGB8/SRGB8, NV12/NV12 and
SRGB8 -> NV12.  Each configuration scores 32 distinct seeded pairs (the 4K working set, 0.8-1.6 GB, is far larger than L2)
with the default batch and ring; every handle is warmed up first, then the configurations of a size take turns in timed
windows of >= `--window` seconds (`--rounds` turns each), and the median window is reported.  Per-kernel times come from a
second handle of each configuration with ring = 1: with several ring slots the kernels of other slots run between a slot's
timing events, so those events do not isolate a kernel.  Front-end time per pair of a mixed handle covers both of its launches;
`fe_vs_mean` is that time over the mean of the two same-format front-end times.
usage: python tools/mixed_time.py [--window 1.0] [--rounds 3] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import turbo_metrics_b200 as tm
from turbo_metrics_b200 import synth

P = tm.PixelFormat
N_PAIRS = 32


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, sm = [x.strip() for x in q[0].split(",")]
    return {"name": name, "power_limit": power, "clocks_max_sm": sm}


def frames(w, h, kind):
    """32 distinct pairs of one source kind on the device -> (refs, diss) per side format"""
    out = {}
    if kind == "yuv":
        for bits, fmt in ((8, "NV12"), (16, "P016")):
            ps = [synth.make_pair_yuv420(w, h, bits, frame=i, seed=1, device="cuda") for i in range(N_PAIRS)]
            pitch, ch = ps[0][2], ps[0][3]
            mk = lambda t, p=pitch, c=ch: tm.DeviceFrame.yuv420(t, p, c)
            out[fmt] = ([mk(r) for r, _, _, _ in ps], [mk(d) for _, d, _, _ in ps])
    else:
        ps = [synth.make_pair_srgb8(w, h, frame=i, seed=1, device="cuda") for i in range(N_PAIRS)]
        out["SRGB8"] = ([tm.DeviceFrame.packed(r) for r, _ in ps], [tm.DeviceFrame.packed(d) for _, d in ps])
        ps = [synth.make_pair_yuv420(w, h, 8, frame=i, seed=1, device="cuda") for i in range(N_PAIRS)]
        pitch, ch = ps[0][2], ps[0][3]
        out["NV12"] = ([tm.DeviceFrame.yuv420(r, pitch, ch) for r, _, _, _ in ps], [tm.DeviceFrame.yuv420(d, pitch, ch) for _, d, _, _ in ps])
    return out


def window(m, refs, diss, min_s):
    """pairs/s over >= min_s seconds of back-to-back batches, ending in a device synchronise (the last ring of batches)"""
    i = m.info()
    tail = i.batch * i.ring
    t0 = time.perf_counter()
    n, last = 0, None
    while True:
        last = m.compute_batch(refs, diss)
        n += len(last)
        if time.perf_counter() - t0 >= min_s:
            break
    stop = last.stop
    m.get_scores(range(max(stop - tail, stop - n), stop))
    return n / (time.perf_counter() - t0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--window", type=float, default=1.0)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    res = {"gpu": gpu_info(), "pairs": N_PAIRS, "window_s": a.window, "rounds": a.rounds, "workloads": {}}
    for size, (w, h), kind, cfgs in (("4k", (3840, 2160), "yuv", [("NV12", "NV12"), ("P016", "P016"), ("NV12", "P016")]),
                                     ("1080p", (1920, 1080), "rgb", [("SRGB8", "SRGB8"), ("NV12", "NV12"), ("SRGB8", "NV12")])):
        fr = frames(w, h, kind)
        handles = {}
        for rf, df in cfgs:
            kw = {} if rf == df else {"dis_fmt": P[df]}
            m = tm.Ssimulacra2(w, h, P[rf], **kw)
            refs, diss = fr[rf][0], fr[df][1]
            for _ in range(2):                       # warm-up: module load, every ring slot, staging of the frame tables
                m.get_scores(m.compute_batch(refs, diss))
            m.kernel_ms(reset=True)
            handles[(rf, df)] = (m, refs, diss)
        rates = {c: [] for c in cfgs}
        for _ in range(a.rounds):
            for c in cfgs:                           # the configurations take turns
                m, refs, diss = handles[c]
                rates[c].append(window(m, refs, diss, a.window))
        out = {}
        for c in cfgs:
            m, refs, diss = handles[c]
            i = m.info()
            m.close()
            kw = {} if c[0] == c[1] else {"dis_fmt": P[c[1]]}
            with tm.Ssimulacra2(w, h, P[c[0]], ring=1, **kw) as m1:   # isolated kernels: one slot, one stream
                m1.get_scores(m1.compute_batch(refs, diss))
                m1.kernel_ms(reset=True)
                for _ in range(4):
                    m1.get_scores(m1.compute_batch(refs, diss))
                ms, batches, pairs = m1.kernel_ms()
            out[f"{c[0]}->{c[1]}" if c[0] != c[1] else f"{c[0]}/{c[1]}"] = {
                "pairs_per_s": float(np.median(rates[c])), "pairs_per_s_windows": [round(x, 1) for x in rates[c]],
                "batch": i.batch, "ring": i.ring, "kernel_launches_per_batch": 4 if c[0] != c[1] else 3,
                "ms_per_pair": {"k_frontend2": ms[0] / pairs, "k_hv": ms[1] / pairs, "k_finalize": ms[3] / pairs},
                "timed_batches": batches}
        (a0, b0), (a1, b1), (mr, md) = cfgs
        same = [out[f"{a0}/{b0}"], out[f"{a1}/{b1}"]]
        mix = out[f"{mr}->{md}"]
        mean_fe = 0.5 * (same[0]["ms_per_pair"]["k_frontend2"] + same[1]["ms_per_pair"]["k_frontend2"])
        mean_hv = 0.5 * (same[0]["ms_per_pair"]["k_hv"] + same[1]["ms_per_pair"]["k_hv"])
        mix["fe_vs_mean"] = mix["ms_per_pair"]["k_frontend2"] / mean_fe
        mix["hv_vs_mean"] = mix["ms_per_pair"]["k_hv"] / mean_hv
        mix["fe_within_10pct_of_mean"] = abs(mix["fe_vs_mean"] - 1.0) <= 0.10
        res["workloads"][size] = out
        del fr, handles
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
