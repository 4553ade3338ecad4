"""Throughput of scaled handles (distorted frames smaller than the reference, upscaled by k_resample) beside the same-size handle
of the reference format, and k_resample's device time beside the front-end's.  Prints one JSON line.

Workloads: a 4K P016 reference against 1080p, 1440p and 720p P016 encodes, and a 1080p NV12 reference against 720p and 540p NV12
encodes.  Each handle has the default batch and ring and scores N_PAIRS distinct seeded pairs (synth.make_pair_scaled; the
same-size handle scores synth.make_pair_yuv420 pairs of the reference's size).  Every handle is warmed up first, then the handles
of a reference size take turns in timed windows of >= `--window` seconds (`--rounds` turns each) and the median is reported.
Kernel times come from a separate phase under torch.profiler (CUDA activity), on handles with ring = 1 and no input groups, so
each batch is one launch group of front-end (reference), k_resample, front-end (distorted): `k_resample_ms_per_launch` and
`k_frontend2_ms_per_group` (both front-end launches) are averages over the profiled batches, `resample_vs_frontend` their ratio.
usage: python tools/scaled_time.py [--window 1.0] [--rounds 3] [--out FILE] [--trace-dir DIR]"""
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
N_PAIRS = 8
WORKLOADS = [("P016", (3840, 2160), [(1920, 1080), (2560, 1440), (1280, 720)]),
             ("NV12", (1920, 1080), [(1280, 720), (960, 540)])]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, sm = [x.strip() for x in q[0].split(",")]
    return {"name": name, "power_limit": power, "clocks_max_sm": sm}


def device_frame(planes):
    """Sample planes -> a device frame: planes pitch * h apart, pitch rounded up to 256 bytes."""
    buf, pitch, p1 = synth.compact_planes(planes)
    t = torch.from_numpy(buf).cuda()
    return tm.DeviceFrame(t.data_ptr(), t.data_ptr() + p1, pitch, t, buf.size)


def window(m, refs, diss, min_s):
    """pairs/s over >= min_s seconds of back-to-back batches, ending in a device synchronise"""
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
    ap.add_argument("--trace-dir", default=None, help="where torch.profiler writes its trace (default: none written)")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    res = {"gpu": gpu_info(), "pairs": N_PAIRS, "window_s": a.window, "rounds": a.rounds, "workloads": {}}
    for fmt, (w, h), dis_sizes in WORKLOADS:
        bits = 8 if fmt == "NV12" else 16
        ps = [synth.make_pair_yuv420(w, h, bits, frame=i, seed=1, device="cuda") for i in range(N_PAIRS)]
        pitch, ch = ps[0][2], ps[0][3]
        refs = [tm.DeviceFrame.yuv420(r, pitch, ch) for r, _, _, _ in ps]
        same = [tm.DeviceFrame.yuv420(d, pitch, ch) for _, d, _, _ in ps]
        configs = {"same_size": (dict(), refs, same)}
        for wd, hd in dis_sizes:
            diss = [device_frame(synth.make_pair_scaled(fmt, w, h, wd, hd, frame=i, seed=1)[1]) for i in range(N_PAIRS)]
            configs[f"{wd}x{hd}"] = (dict(dis_width=wd, dis_height=hd), refs, diss)
        handles = {}
        for name, (kw, r, d) in configs.items():
            m = tm.Ssimulacra2(w, h, P[fmt], **kw)
            for _ in range(2):                       # warm-up: module load, every ring slot
                m.get_scores(m.compute_batch(r, d))
            handles[name] = m
        rates = {n: [] for n in configs}
        for _ in range(a.rounds):
            for name, (kw, r, d) in configs.items():   # the configurations take turns
                rates[name].append(window(handles[name], r, d, a.window))
        out = {}
        for name, m in handles.items():
            i = m.info()
            out[name] = {"pairs_per_s": float(np.median(rates[name])), "pairs_per_s_windows": [round(x, 1) for x in rates[name]],
                         "batch": i.batch, "ring": i.ring, "io_bytes_per_pair": int(i.io_bytes_per_pair),
                         "device_bytes": m.mem_usage()}
            m.close()
        for name in configs:
            out[name]["vs_same_size"] = out[name]["pairs_per_s"] / out["same_size"]["pairs_per_s"]
        # kernel times: a phase of its own under the profiler
        for name, (kw, r, d) in configs.items():
            if not kw:
                continue
            with tm.Ssimulacra2(w, h, P[fmt], ring=1, **kw) as m1:
                m1.get_scores(m1.compute_batch(r, d))
                batches = 4
                with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                    for _ in range(batches):
                        m1.get_scores(m1.compute_batch(r, d))
                if a.trace_dir:
                    os.makedirs(a.trace_dir, exist_ok=True)
                    prof.export_chrome_trace(os.path.join(a.trace_dir, f"scaled_{fmt}_{name}.pt.trace.json"))
                rs_us = fe_us = 0.0
                rs_n = 0
                for e in prof.key_averages():
                    if "k_resample" in e.key:
                        rs_us += e.device_time_total
                        rs_n += e.count
                    elif "k_frontend2" in e.key:
                        fe_us += e.device_time_total
                assert rs_n == batches, rs_n
                out[name].update({"k_resample_ms_per_launch": rs_us / 1e3 / rs_n, "k_frontend2_ms_per_group": fe_us / 1e3 / rs_n,
                                  "resample_vs_frontend": rs_us / fe_us, "profiled_launch_groups": rs_n,
                                  "pairs_per_group": m1.info().batch})
        res["workloads"][f"{fmt}_{w}x{h}"] = out
        del handles, configs, refs, same, ps
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
