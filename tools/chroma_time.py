"""Throughput and front-end device time of the 4:2:2 / 4:4:4 formats (NV16, P216, YUV444, YUV444P16) beside NV12 and P016 on
the same GPU, at 4K and 1080p.  Prints one JSON line.

Each configuration is a same-format handle with the default batch and ring scoring N_PAIRS distinct seeded pairs
(synth.make_pair_yuv420 / make_pair_yuv; the 4K working sets, 0.4-3.2 GB, are far larger than L2).  Every handle is warmed up
first, then the configurations of a size take turns in timed windows of >= `--window` seconds (`--rounds` turns each) and the
median window is reported.  Per-kernel times come from a second handle of each configuration with ring = 1 (with several ring
slots the kernels of other slots run between a slot's timing events); with no input groups there is one front-end launch per
batch, so `k_frontend2_ms_per_launch` is the front-end time of one batch.  `fe_vs_p016` / `fe_vs_nv12` divide a format's front-end
time per pair by that of the 4:2:0 format of its sample size.
usage: python tools/chroma_time.py [--window 1.0] [--rounds 3] [--out FILE]"""
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
N_PAIRS = 16
FORMATS = [("NV12", 8, "420"), ("P016", 16, "420"), ("NV16", 8, "422"), ("P216", 16, "422"), ("YUV444", 8, "444"),
           ("YUV444P16", 16, "444")]
BASE = {"NV16": "NV12", "YUV444": "NV12", "P216": "P016", "YUV444P16": "P016"}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, sm = [x.strip() for x in q[0].split(",")]
    return {"name": name, "power_limit": power, "clocks_max_sm": sm}


def frames(w, h, bits, sub):
    """N_PAIRS distinct device pairs of one format -> (refs, diss)"""
    if sub == "420":
        ps = [synth.make_pair_yuv420(w, h, bits, frame=i, seed=1, device="cuda") for i in range(N_PAIRS)]
        mk = tm.DeviceFrame.yuv420
    else:
        ps = [synth.make_pair_yuv(w, h, bits, sub, frame=i, seed=1, device="cuda") for i in range(N_PAIRS)]
        mk = tm.DeviceFrame.yuv422 if sub == "422" else tm.DeviceFrame.yuv444
    pitch, ch = ps[0][2], ps[0][3]
    return [mk(r, pitch, ch) for r, _, _, _ in ps], [mk(d, pitch, ch) for _, d, _, _ in ps]


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
    for size, (w, h) in (("4k", (3840, 2160)), ("1080p", (1920, 1080))):
        handles = {}
        for fmt, bits, sub in FORMATS:
            refs, diss = frames(w, h, bits, sub)
            m = tm.Ssimulacra2(w, h, P[fmt])
            for _ in range(2):                       # warm-up: module load, every ring slot, staging of the frame tables
                m.get_scores(m.compute_batch(refs, diss))
            handles[fmt] = (m, refs, diss)
        rates = {f: [] for f, _, _ in FORMATS}
        for _ in range(a.rounds):
            for fmt, _, _ in FORMATS:                # the configurations take turns
                m, refs, diss = handles[fmt]
                rates[fmt].append(window(m, refs, diss, a.window))
        out = {}
        for fmt, _, _ in FORMATS:
            m, refs, diss = handles[fmt]
            i = m.info()
            m.close()
            with tm.Ssimulacra2(w, h, P[fmt], ring=1) as m1:   # isolated kernels: one slot, one stream
                m1.get_scores(m1.compute_batch(refs, diss))
                m1.kernel_ms(reset=True)
                for _ in range(4):
                    m1.get_scores(m1.compute_batch(refs, diss))
                ms, batches, pairs = m1.kernel_ms()
                b1 = m1.info().batch
            out[fmt] = {"pairs_per_s": float(np.median(rates[fmt])), "pairs_per_s_windows": [round(x, 1) for x in rates[fmt]],
                        "batch": i.batch, "ring": i.ring, "io_bytes_per_pair": int(i.io_bytes_per_pair),
                        "k_frontend2_ms_per_launch": ms[0] / batches, "launch_batch": b1,
                        "ms_per_pair": {"k_frontend2": ms[0] / pairs, "k_hv": ms[1] / pairs, "k_finalize": ms[3] / pairs},
                        "timed_batches": batches}
        for fmt, base in BASE.items():
            out[fmt][f"fe_vs_{base.lower()}"] = out[fmt]["ms_per_pair"]["k_frontend2"] / out[base]["ms_per_pair"]["k_frontend2"]
        res["workloads"][size] = out
        del handles
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
