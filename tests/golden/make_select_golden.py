#!/usr/bin/env python
"""Records tests/golden/ref_select.npz: the reference's own PixelSelector::makeMaps (oracle/_ref/libdso_ref_select.so, built by
oracle/ref_select_build.sh from the reference's sources) on every case of tests/select_cases.py, and FullSystem::makeNewTraces' point list for the TRACE_CASES (the
reference's map filtered to [patternPadding+1, dim-patternPadding-2) in raster order and fed to the reference's ImmaturePoint constructor,
points with a non-finite energyTH dropped).  Maps are stored whole as uint8, so that a failing test names pixels.

Run from the repo root, with the reference build present:  python tests/golden/make_select_golden.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import select_cases as S  # noqa: E402
from oracle import ref, ref_select  # noqa: E402

GOLDEN = os.path.join(HERE, "ref_select.npz")


def new_traces_list(dI0, m, K):
    """FullSystem::makeNewTraces' loop (FullSystem.cpp:L1652-1664) over the reference's map, through the reference's constructor"""
    h, w = m.shape
    ys, xs = np.nonzero(m[3:h - 4, 3:w - 4])
    u, v = (xs + 3).astype(np.int32), (ys + 3).astype(np.int32)   # np.nonzero walks in raster order
    P = ref.ip_init(dI0, w, h, K, u, v)
    keep = P["ok"].astype(bool)
    return dict(u=u[keep], v=v[keep], type=m[v, u][keep].astype(np.float32), color=P["color"][keep], weights=P["weights"][keep],
                gradH=P["gradH"][keep], energyTH=P["energyTH"][keep])


def main():
    out = {}

    def run(img, c):
        m, n, pot, lv = ref_select.make_maps(img, S.K640, c["density"], c["recursionsLeft"], c["thFactor"], c["potential"], c["B"], c["settings"])
        return m, n, pot, lv, img

    res = S.run_cases(run)
    for name, (m, n, pot, lv, img) in res.items():
        out[f"{name}/map"] = m
        out[f"{name}/numHaveSub"] = np.int64(n)
        out[f"{name}/potential"] = np.int64(pot)
        out[f"{name}/image_sha256"] = np.array(S.sha(img))
        if name in S.TRACE_CASES:
            for k, a in new_traces_list(lv[0], m, S.K640).items():
                out[f"{name}/traces/{k}"] = a
        print(f"{name}: numHaveSub {n}, potential {S.resolve(name, 0)['potential']} -> {pot}")
    np.savez_compressed(GOLDEN, **out)
    print(f"{GOLDEN}: {os.path.getsize(GOLDEN) / 1024:.0f} KiB")


if __name__ == "__main__":
    main()
