#!/usr/bin/env python
"""Pixel selection for new keyframes: dmv_ct_make_new_traces (device) against what a caller does on the CPU today, the single-thread
oracle's FrameHessian::makeImages + PixelSelector::makeMaps + ImmaturePoint constructor loop, on the same seeded frames.

  python tools/bench_select.py --frames 30 --out /tmp/bench_select.json

Cases: 640x480 (density 1500, the potential carried over a seeded frame sequence) and 512x512.  Reports the median wall time of a
synchronised dmv_ct_make_new_traces call (the frame is already resident), the summed kernel time per call from torch.profiler (CUDA
activities, a separate pass), launches per call and bytes moved over PCIe per call, the card name and its power limit."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import dmvio_b200.capi as capi  # noqa: E402
import select_cases as S  # noqa: E402
from oracle import orc, orc_select  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return q.stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def run_case(w, h, nframes, seed0):
    frames = [S.smooth(w, h, seed0 + i) for i in range(nframes)]
    g = capi.CT(w, h, 4, max_points=1024)
    L = capi.lib()
    # device: warm up, then the timed pass, the potential carried frame to frame
    g.upload_new_image(frames[0])
    g.make_new_traces(1500)
    wall, counts, launches, d2h = [], [], [], []
    pot = 3
    for img in frames:
        g.upload_new_image(img)
        L.dmv_ct_get_ref(g.h, 0, capi.C.byref(capi.C.c_int(0)), None, None, None, None)   # synchronises the handle's stream: the upload is done
        n0 = capi.C.c_longlong(0)
        L.dmv_ct_kernel_launch_count(g.h, capi.C.byref(n0))
        t = time.perf_counter()
        P, sub, pot_new = g.make_new_traces(1500, potential=pot)
        wall.append(time.perf_counter() - t)
        n1 = capi.C.c_longlong(0)
        L.dmv_ct_kernel_launch_count(g.h, capi.C.byref(n1))
        launches.append(n1.value - n0.value)
        passes = 1 + (pot_new != pot and sub > 0)
        m = len(P["u"])
        d2h.append(32 * passes + 32 + 4 + 25 * 4 * m)   # pick counts per pass, the sub-sample count, the compacted count, the point list
        counts.append(m)
        pot = pot_new
    # kernel time: a separate pass under torch.profiler
    kernel_ms = None
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.init()
        pot = 3
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for img in frames:
                g.upload_new_image(img)
                _, _, pot = g.make_new_traces(1500, potential=pot)
        names = ("ps_", "ip_init_kernel")
        tot = sum(e.device_time_total for e in prof.key_averages() if any(e.key.startswith(n) or n in e.key for n in names))
        kernel_ms = tot / 1000.0 / len(frames)
    except Exception as e:  # noqa: BLE001
        kernel_ms = f"not measured ({e})"
    g.close()
    # CPU: the single-thread oracle doing makeImages + makeMaps + the constructor loop
    cpu = []
    pot = 3
    for img in frames:
        t = time.perf_counter()
        lv = orc.make_images(img, S.K640)
        _, _, pot = orc_select.make_new_traces(lv, 1500, potential=pot)
        cpu.append(time.perf_counter() - t)
    return dict(w=w, h=h, frames=nframes, points_median=int(np.median(counts)), device_wall_ms_median=1e3 * float(np.median(wall)),
                device_kernel_ms_per_call=kernel_ms, launches_per_call=int(np.median(launches)), d2h_bytes_per_call_median=int(np.median(d2h)),
                h2d_bytes_per_call=0, cpu_oracle_ms_median=1e3 * float(np.median(cpu)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=30)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if capi.lib().dmv_device_count() < 1:
        raise SystemExit("bench_select: no CUDA device")
    res = dict(card=card(), cases=[run_case(640, 480, a.frames, 100), run_case(512, 512, a.frames, 200)])
    for c in res["cases"]:
        c["device_faster"] = c["device_wall_ms_median"] < c["cpu_oracle_ms_median"]
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
