"""The frames and makeMaps arguments of the pixel-selection tests (tests/test_ref_pin_select.py, tests/test_gpu_select.py), the recording script
tests/golden/make_select_golden.py and tools/bench_select.py.

Frames are generated with integer and float32 arithmetic only (no libm), so they are bit-identical on every machine; the golden file stores
their SHA-256 to prove it."""
import hashlib

import numpy as np

K640 = (500.0, 500.0, 319.5, 239.5)


def _lcg(seed, n):
    """n uint32 values of a 32-bit LCG (Numerical Recipes constants), as float32 in [0, 1)."""
    out = np.empty(n, np.uint32)
    x = np.uint64(seed * 2654435761 % 2**32)
    a, c, m = np.uint64(1664525), np.uint64(1013904223), np.uint64(2**32)
    for i in range(n):
        x = (a * x + c) % m
        out[i] = x
    return (out >> np.uint32(8)).astype(np.float32) / np.float32(2**24)


def _value_noise(w, h, cell, seed):
    gw, gh = w // cell + 2, h // cell + 2
    g = _lcg(seed, gw * gh).reshape(gh, gw)
    ys, xs = np.divmod(np.arange(h * w, dtype=np.int64), w)
    fy = (ys % cell).astype(np.float32) / np.float32(cell)
    fx = (xs % cell).astype(np.float32) / np.float32(cell)
    y0, x0 = ys // cell, xs // cell
    top = g[y0, x0] * (np.float32(1) - fx) + g[y0, x0 + 1] * fx
    bot = g[y0 + 1, x0] * (np.float32(1) - fx) + g[y0 + 1, x0 + 1] * fx
    return (top * (np.float32(1) - fy) + bot * fy).reshape(h, w).astype(np.float32)


def smooth(w, h, seed):
    """two octaves of bilinear value noise, intensities in [20, 235]"""
    a = _value_noise(w, h, 32, seed) * np.float32(150) + _value_noise(w, h, 8, seed + 1000) * np.float32(65)
    return (a + np.float32(20)).astype(np.float32)


def quantised(w, h, seed):
    return np.floor(smooth(w, h, seed) + np.float32(0.5)).astype(np.float32)


def stripes(w, h, seed):
    """integer image: regions of purely vertical stripes (dy == 0), purely horizontal stripes (dx == 0) and quantised noise"""
    img = quantised(w, h, seed)
    ys, xs = np.mgrid[0:h, 0:w]
    v = np.where((xs // 6) % 2 == 0, 60.0, 140.0).astype(np.float32)   # depends on x only
    hz = np.where((ys // 7) % 2 == 0, 70.0, 170.0).astype(np.float32)  # depends on y only
    img = np.where((xs < w // 3) & (ys < 2 * h // 3), v, img)
    img = np.where((xs >= 2 * w // 3) & (ys >= h // 3), hz, img)
    return img.astype(np.float32)


IMAGES = {
    "smooth640": lambda: smooth(640, 480, 1),
    "quant640": lambda: quantised(640, 480, 2),
    "smooth512": lambda: smooth(512, 512, 3),
    "stripes640": lambda: stripes(640, 480, 4),
    "seq640_0": lambda: smooth(640, 480, 11),
    "seq640_1": lambda: smooth(640, 480, 12),
    "seq640_2": lambda: smooth(640, 480, 13),
}


def gamma_B():
    """a non-identity CalibHessian::B: a gamma curve 255 * (i / 255)^0.6"""
    i = np.arange(256, dtype=np.float64)
    return (255.0 * (i / 255.0) ** 0.6).astype(np.float32)


# name -> dict(img, density, recursionsLeft, thFactor, potential, B, settings); "potential": None = carried from the previous case
CASES = {
    "smooth640": dict(img="smooth640", density=1500),
    "quant640": dict(img="quant640", density=1500),
    "smooth512": dict(img="smooth512", density=1500),
    "stripes640": dict(img="stripes640", density=1500),
    "setfirst_smooth640": dict(img="smooth640", density=0.03 * 640 * 480, thFactor=2.0),
    "setfirst_stripes640": dict(img="stripes640", density=0.03 * 640 * 480, thFactor=2.0),
    "more_points": dict(img="quant640", density=20000),        # quotia > 1.25: potential down
    "fewer_points": dict(img="smooth640", density=150),        # quotia < 0.25: potential up
    "no_recursion_subsample": dict(img="quant640", density=1200, recursionsLeft=0),   # quotia < 0.95 subsample at potential 3
    "no_recursion_many": dict(img="stripes640", density=40000, recursionsLeft=0),
    "pot1_subsample": dict(img="stripes640", density=15000, potential=1),
    "no_direction": dict(img="quant640", density=1500, settings=(0.5, 7.0, 0.75, 0)),
    "no_direction_stripes": dict(img="stripes640", density=1500, settings=(0.5, 7.0, 0.75, 0)),
    "gamma_B": dict(img="smooth640", density=1500, B="gamma"),
    "gamma_B_stripes": dict(img="stripes640", density=1500, B="gamma"),
    "seq_0": dict(img="seq640_0", density=1500, potential=3),
    "seq_1": dict(img="seq640_1", density=1500, potential=None),
    "seq_2": dict(img="seq640_2", density=1500, potential=None),
}
# the makeNewTraces cases (density 1500, thFactor 1, recursionsLeft 1)
TRACE_CASES = ("smooth640", "stripes640", "fewer_points", "gamma_B")


def resolve(name, prev_potential=None):
    c = dict(recursionsLeft=1, thFactor=1.0, potential=3, B=None, settings=None)
    c.update(CASES[name])
    if c["potential"] is None:
        c["potential"] = prev_potential
    if isinstance(c["B"], str):
        c["B"] = gamma_B()
    return c


def run_cases(fn):
    """fn(image, case) -> (map, numHaveSub, potential_after, ...); returns {name: result}, carrying the potential between sequence cases."""
    out, pot = {}, None
    for name in CASES:
        c = resolve(name, pot)
        r = fn(IMAGES[c["img"]](), c)
        pot = r[2]
        out[name] = r
    return out


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def direction_dependent_cells(dI0, ag0, pot, thFactor, minGradHistCut=0.5, minGradHistAdd=7.0):
    """pot-cells whose level-0 pick depends on the block direction for a reason read off the input alone: at least one pixel passes
    PixelSelector::select's level-0 threshold and every passing pixel has dx == 0 or every one has dy == 0 (then |g . d| == 0 for
    d = (1, 0) or d = (0, 1) and > 0 for the other).  Thresholds are makeHists' (PixelSelector2.cpp:L94-157), restated in numpy."""
    h, w = ag0.shape
    nbW, nbH = w // 16, h // 16
    g = np.minimum(np.sqrt(ag0).astype(np.int64), 48)
    valid = np.zeros((h, w), bool)
    valid[1:h - 1, 1:w - 1] = True
    ths = np.zeros((nbH, nbW), np.float32)
    for by in range(nbH):
        for bx in range(nbW):
            sl = (slice(16 * by, 16 * by + 16), slice(16 * bx, 16 * bx + 16))
            hist = np.bincount(g[sl][valid[sl]], minlength=49)
            th = int(np.float32(valid[sl].sum()) * np.float32(minGradHistCut) + np.float32(0.5))
            q = 90
            for i in range(90):
                th -= int(hist[i]) if i < 49 else 0
                if th < 0:
                    q = i
                    break
            ths[by, bx] = np.float32(q) + np.float32(minGradHistAdd)
    sm = np.zeros_like(ths)
    for by in range(nbH):
        for bx in range(nbW):
            nb = ths[max(by - 1, 0):by + 2, max(bx - 1, 0):bx + 2]
            m = np.float32(nb.sum(dtype=np.float32)) / np.float32(nb.size)
            sm[by, bx] = m * m
    ys, xs = np.mgrid[0:h, 0:w]
    inside = (xs >= 4) & (xs < w - 5) & (ys >= 4) & (ys <= h - 4)
    passing = inside & (ag0 > sm[ys // 16, xs // 16] * np.float32(thFactor))
    dx, dy = dI0[..., 1], dI0[..., 2]
    n = 0
    for cy in range(0, h, pot):
        for cx in range(0, w, pot):
            p = passing[cy:cy + pot, cx:cx + pot]
            if not p.any():
                continue
            if (dx[cy:cy + pot, cx:cx + pot][p] == 0).all() or (dy[cy:cy + pot, cx:cx + pot][p] == 0).all():
                n += 1
    return n
