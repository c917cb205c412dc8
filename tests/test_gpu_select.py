"""Pixel selection for new keyframes on the device (dmv_ct_select_pixels, dmv_ct_make_new_traces) against the CPU oracle, which
tests/test_ref_pin_select.py pins to the reference bit for bit.  Bar: BIT-EXACT (maps, counts, potentials, point lists in order)."""
import numpy as np
import pytest

import select_cases as S
from oracle import orc_select

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def capi():
    import dmvio_b200.capi as c
    if c.lib().dmv_device_count() < 1:
        pytest.skip("no CUDA device")
    return c


def _oracle(orc, img, c):
    lv = orc.make_images(img, S.K640)
    return orc_select.make_maps(lv, c["density"], c["recursionsLeft"], c["thFactor"], c["potential"], c["B"], c["settings"]), lv


@pytest.mark.parametrize("upload", ["image", "levels"])
def test_select_pixels_bit_exact(capi, orc, upload):
    handles = {}

    def run(img, c):
        h, w = img.shape
        if (w, h) not in handles:
            handles[(w, h)] = capi.CT(w, h, 4, max_points=1024)
        g = handles[(w, h)]
        (m_o, n_o, p_o), lv = _oracle(orc, img, c)
        if upload == "image":
            g.upload_new_image(img)
        else:
            for l in range(4):
                g.upload_new(l, lv[l] if l < 3 else orc.make_images(img, S.K640)[l])
        m_g, n_g, p_g = g.select_pixels(c["density"], c["recursionsLeft"], c["thFactor"], c["potential"], c["B"], c["settings"])
        return m_g, n_g, p_g, m_o, n_o, p_o

    res = S.run_cases(run)
    for name, (m_g, n_g, p_g, m_o, n_o, p_o) in res.items():
        bad = np.argwhere(m_g != m_o)
        assert bad.size == 0, f"{name}: {len(bad)} pixels differ, first (y, x) {bad[:8].tolist()}"
        assert (n_g, p_g) == (n_o, p_o), name
    for g in handles.values():
        g.close()


@pytest.mark.parametrize("name", S.TRACE_CASES)
def test_make_new_traces_bit_exact(capi, orc, name):
    c = S.resolve(name, 3)
    img = S.IMAGES[c["img"]]()
    lv = orc.make_images(img, S.K640)
    P_o, sub_o, pot_o = orc_select.make_new_traces(lv, c["density"], c["recursionsLeft"], c["thFactor"], c["potential"], c["B"], c["settings"])
    g = capi.CT(img.shape[1], img.shape[0], 4, max_points=1024)
    g.upload_new_image(img)
    P_g, sub_g, pot_g = g.make_new_traces(c["density"], c["recursionsLeft"], c["thFactor"], c["potential"], c["B"], c["settings"])
    assert (sub_g, pot_g) == (sub_o, pot_o)
    assert len(P_g["u"]) == len(P_o["u"]) > 0
    for k in ("u", "v", "type", "color", "weights", "gradH", "energyTH"):
        a, b = P_g[k], P_o[k]
        assert np.array_equal(a.view(np.uint32) if a.dtype == np.float32 else a, b.view(np.uint32) if b.dtype == np.float32 else b), k
    # the same call again: identical bytes; the map of dmv_ct_select_pixels with the same arguments is the one the list was made from
    P_2, sub_2, pot_2 = g.make_new_traces(c["density"], c["recursionsLeft"], c["thFactor"], c["potential"], c["B"], c["settings"])
    assert (sub_2, pot_2) == (sub_g, pot_g)
    for k in P_g:
        assert P_2[k].tobytes() == P_g[k].tobytes(), k
    m1 = g.select_pixels(c["density"], c["recursionsLeft"], c["thFactor"], c["potential"], c["B"], c["settings"])[0]
    m2 = g.select_pixels(c["density"], c["recursionsLeft"], c["thFactor"], c["potential"], c["B"], c["settings"])[0]
    assert m1.tobytes() == m2.tobytes()
    assert m1[P_g["v"], P_g["u"]].tolist() == P_g["type"].astype(np.uint8).tolist()
    g.close()


def test_select_errors(capi):
    DMV_ERR_INVALID, DMV_ERR_STATE = -1, -4
    L = capi.lib()
    img = S.IMAGES["smooth640"]()

    def rc_select(g, **kw):
        a, keep = g._ps_args(kw.get("density", 1500), 1, 1.0, kw.get("potential", 3), None, None)
        r = capi.PSResult()
        return L.dmv_ct_select_pixels(g.h, capi.C.byref(a), None, capi.C.byref(r))

    g = capi.CT(640, 480, 4, max_points=1024)
    assert rc_select(g) == DMV_ERR_STATE                 # no frame resident yet
    g.upload_new(0, np.zeros((480, 640, 3), np.float32))
    assert rc_select(g) == DMV_ERR_STATE                 # levels 1 and 2 missing
    g.upload_new_image(img)
    assert rc_select(g) == 0
    assert rc_select(g, density=0) == DMV_ERR_INVALID
    assert rc_select(g, potential=0) == DMV_ERR_INVALID
    # cap smaller than the list: only the needed count is written
    P, _, _ = g.make_new_traces(1500)
    a, keep = g._ps_args(1500, 1, 1.0, 3, None, None)
    n, r = capi.C.c_int(0), capi.PSResult(-7, -7)
    u = np.full(4, -5, np.int32)
    rest = [np.zeros(4 * k, np.float32) for k in (1, 1, 8, 8, 4, 1)]   # v, type, color8, weights8, gradH4, energyTH
    rc = L.dmv_ct_make_new_traces(g.h, capi.C.byref(a), 4, capi.C.byref(n), u.ctypes.data, *[x.ctypes.data for x in rest], capi.C.byref(r))
    assert rc == DMV_ERR_INVALID and n.value == len(P["u"]) > 4
    assert (u == -5).all() and (r.numHaveSub, r.currentPotential) == (-7, -7)
    g.close()
    g = capi.CT(640, 480, 2, max_points=1024)            # fewer than 3 levels
    g.upload_new_image(img)
    assert rc_select(g) == DMV_ERR_INVALID
    g.close()
    g = capi.CT(648, 480, 4, max_points=1024)            # w not divisible by 16
    g.upload_new_image(np.zeros((480, 648), np.float32))
    assert rc_select(g) == DMV_ERR_INVALID
    g.close()
