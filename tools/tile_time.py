"""Cost of per-tile scores (ssimu2_config.tile): pairs/s and k_hv device time per launch with tiles off, T = 64 and T = 256, in
the full and the score-only mode.  Prints one JSON line.

Workloads: 4K P016 and 1080p NV12, N_PAIRS distinct seeded pairs (synth.make_pair_yuv420) per handle, default batch and ring.
Every handle is warmed up first; then, per workload, the six handles take turns in timed windows of >= `--window` seconds
(`--rounds` turns each) and the median is reported.  Kernel times are the library's CUDA events on each batch's own stream
(ssimu2_kernel_ms, summed over the batches of the timed windows): `k_hv_ms_per_launch` is k_hv alone, `finalize_ms_per_launch`
k_finalize plus, with tiles, k_tile_finalize.  The card's name and power limit are read in the same run.
usage: python tools/tile_time.py [--window 1.0] [--rounds 3] [--out FILE]"""
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
WORKLOADS = [("P016", 16, (3840, 2160)), ("NV12", 8, (1920, 1080))]
TILES = [0, 64, 256]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, sm = [x.strip() for x in q[0].split(",")]
    return {"name": name, "power_limit": power, "clocks_max_sm": sm}


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
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    res = {"gpu": gpu_info(), "pairs": N_PAIRS, "window_s": a.window, "rounds": a.rounds, "workloads": {}}
    for fmt, bits, (w, h) in WORKLOADS:
        ps = [synth.make_pair_yuv420(w, h, bits, frame=i, seed=1, device="cuda") for i in range(N_PAIRS)]
        pitch, ch = ps[0][2], ps[0][3]
        refs = [tm.DeviceFrame.yuv420(r, pitch, ch) for r, _, _, _ in ps]
        diss = [tm.DeviceFrame.yuv420(d, pitch, ch) for _, d, _, _ in ps]
        handles = {}
        for score_only in (False, True):
            for tile in TILES:
                name = f"{'score_only' if score_only else 'full'}_tile{tile}"
                m = tm.Ssimulacra2(w, h, P[fmt], score_only=score_only, tile=tile)
                for _ in range(2):                   # warm-up: module load, every ring slot
                    m.get_scores(m.compute_batch(refs, diss))
                m.kernel_ms(reset=True)
                handles[name] = m
        rates = {n: [] for n in handles}
        for _ in range(a.rounds):
            for name, m in handles.items():         # the configurations take turns
                rates[name].append(window(m, refs, diss, a.window))
        out = {}
        for name, m in handles.items():
            i = m.info()
            ms, batches, pairs = m.kernel_ms()
            out[name] = {"pairs_per_s": float(np.median(rates[name])), "pairs_per_s_windows": [round(x, 1) for x in rates[name]],
                         "k_hv_ms_per_launch": ms[1] / batches, "finalize_ms_per_launch": ms[3] / batches,
                         "timed_batches": batches, "batch": i.batch, "ring": i.ring,
                         "device_bytes": m.mem_usage(), "tile_grid": list(m.tile_grid())}
            m.close()
        for name in handles:
            base = out[name.rsplit("_tile", 1)[0] + "_tile0"]
            out[name]["vs_tiles_off"] = out[name]["pairs_per_s"] / base["pairs_per_s"]
            out[name]["k_hv_vs_tiles_off"] = out[name]["k_hv_ms_per_launch"] / base["k_hv_ms_per_launch"]
        res["workloads"][f"{fmt}_{w}x{h}"] = out
        del handles, refs, diss, ps
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
