"""GPU parity tests of the coarse direct-image-alignment kernel (CoarseTracker::calcRes + calcGSSSE fused) vs the CPU oracle.

Tolerances: counters (numTermsInE, saturated, n_warped) exact up to points whose |residual| is within 1e-3 of the cutoff or
whose projection is within 1e-3 px of the image border; energies rel 1e-4 (the oracle sums in fp32 sequentially, the GPU in
fp32 per thread + fp64 across threads); H and b (fp64-accumulated oracle) ||d||_F/||.||_F <= 2e-5 / 2e-4."""
import numpy as np
import pytest

from helpers import rel

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def capi():
    import dmvio_b200.capi as c
    if c.lib().dmv_device_count() < 1:
        pytest.fail("no CUDA device visible: GPU tests must run on the B200 box")
    return c


def _setup(capi, orc, synth, levels, seed=4321):
    T = synth.make_tracking_pair(seed=seed, levels=levels)
    oct_ = orc.CoarseTracker(T["w"], T["h"], T["K"], levels)
    oct_.make_coarse_depth(T["Ku"], T["Kv"], T["new_idepth"], T["HdiF"], T["pyr_ref"])
    oct_.set_new_frame(T["pyr_new"])
    L = oct_.levels
    g = capi.CT(T["w"], T["h"], L, max_points=65536)
    for l in range(L):
        k, wh = oct_.K(l)
        g.set_K(l, *[float(x) for x in k])
        p = oct_.ref_points(l)
        g.set_ref(l, p["u"], p["v"], p["idepth"], p["color"])
        g.upload_new(l, T["pyr_new"][l])
    return T, oct_, g


def _pose_args(synth, oct_, lvl, R, t, a, b):
    import dmvio_b200.hostmath as hm
    k, _ = oct_.K(lvl)
    Ki = hm.inv3_cofactor_f32(np.array([[k[0], 0, k[2]], [0, k[1], k[3]], [0, 0, 1]], np.float32))  # K[lvl].inverse() as the reference rounds it
    RKi = hm.mm3_f32(R.astype(np.float32), Ki)
    affLL = np.array([np.exp(a), b], np.float32)  # ref aff_g2l = (0,0), exposures 1
    return RKi, t.astype(np.float32), affLL


@pytest.mark.parametrize("levels", [0, 5])
def test_calc_res_gs_parity(capi, orc, synth, levels):
    T, oct_, g = _setup(capi, orc, synth, levels)
    R, t = synth.se3_mul(*synth.se3_exp(np.array([0.003, -0.002, 0.001, 0.001, -0.001, 0.001])), T["R_true"], T["t_true"])
    a, b = T["a_new"] + 0.01, T["b_new"] - 0.3
    for lvl in range(oct_.levels):
        r_o = oct_.calc_res(lvl, R, t, a, b, cutoff=20.0)
        H_o, b_o = oct_.calc_gs(lvl, a, b, 1)
        n_o = oct_.warped().shape[1]
        RKi, tf, affLL = _pose_args(synth, oct_, lvl, R, t, a, b)
        r_g, H_g, b_g, n_g = g.calc_res_gs(lvl, RKi, tf, affLL, 0.0, 20.0, True)
        assert abs(r_g[1] - r_o[1]) <= 2 and abs(n_g - n_o) <= 4, (lvl, r_g, r_o, n_g, n_o)
        assert abs(r_g[0] - r_o[0]) <= 2e-4 * abs(r_o[0]) + 2 * 391.0
        if lvl == 0:
            np.testing.assert_allclose(r_g[[2, 4]], r_o[[2, 4]], rtol=1e-4)
        assert abs(r_g[5] - r_o[5]) < 2e-3
        if n_g == n_o and r_g[1] == r_o[1]:
            assert rel(H_g, H_o) < 2e-5, (lvl, rel(H_g, H_o))
            assert rel(b_g, b_o) < 2e-4, (lvl, rel(b_g, b_o))
        assert np.abs(H_g - H_g.T).max() <= 1e-12 * np.abs(H_g).max()
    g.close()


def test_track_abort_returns_input_pose(capi, orc, synth):
    """dmv_ct_track aborted at its first level (minResForAbort = 0): status 2, not good, and R, t, a, b exactly as passed in, like the
    reference's early `return false`; lastResiduals of the aborted level as the oracle's, the levels never reached stay NaN."""
    T, oct_, g = _setup(capi, orc, synth, 0)
    R0, t0, a0, b0 = np.eye(3), np.zeros(3), 0.0, 0.0
    r_o = oct_.track(R0, t0, a0, b0, coarsest=3, minRes=np.zeros(5))
    r_g = g.track(R0, t0, a0, b0, coarsest=3, minRes=np.zeros(5))
    assert r_g["status"] == 2 and r_g["good"] == 0
    np.testing.assert_array_equal(r_g["R"], R0)
    np.testing.assert_array_equal(r_g["t"], t0)
    assert r_g["a"] == a0 and r_g["b"] == b0
    np.testing.assert_allclose(r_g["lastResiduals"][3], r_o["lastResiduals"][3], rtol=2e-3)
    assert np.isnan(r_g["lastResiduals"][[0, 1, 2, 4]]).all()
    g.close()


def test_device_pyramid_matches_host(capi, orc, synth):
    """dmv_ct_upload_new_image (FrameHessian::makeImages on the device) gives the same calcRes/GS as uploading host pyramids."""
    T, oct_, g = _setup(capi, orc, synth, 0)
    R, t, a, b = T["R_true"], T["t_true"], T["a_new"], T["b_new"]
    out_host = [g.calc_res_gs(l, *_pose_args(synth, oct_, l, R, t, a, b), 0.0, 20.0, True) for l in range(oct_.levels)]
    g.upload_new_image(T["img_new"])
    for l in range(oct_.levels):
        r2, H2, b2, n2 = g.calc_res_gs(l, *_pose_args(synth, oct_, l, R, t, a, b), 0.0, 20.0, True)
        r1, H1, b1, n1 = out_host[l]
        assert n1 == n2
        np.testing.assert_allclose(r2, r1, rtol=1e-6)
        np.testing.assert_allclose(H2, H1, rtol=1e-9, atol=1e-9 * np.abs(H1).max())
    g.close()


def test_edge_cases(capi, orc, synth):
    T, oct_, g = _setup(capi, orc, synth, 0)
    # everything out of bounds: huge translation -> no terms, NaN mean energy handled by the caller like the reference
    RKi, tf, affLL = _pose_args(synth, oct_, 0, np.eye(3), np.array([1e3, 0, 0.0]), 0.0, 0.0)
    r, H, b, n = g.calc_res_gs(0, RKi, tf, affLL, 0.0, 20.0, True)
    assert r[1] == 0 and n == 0
    # empty reference list
    g.set_ref(1, np.zeros(0, np.float32), np.zeros(0, np.float32), np.zeros(0, np.float32), np.zeros(0, np.float32))
    r, H, b, n = g.calc_res_gs(1, RKi, tf, affLL, 0.0, 20.0, True)
    assert r[1] == 0 and n == 0
    g.close()


@pytest.mark.parametrize("cfg", [dict(seed=4321), dict(seed=77, w=160, h=120, npts=400), dict(seed=5, npts=6000)], ids=["640x480", "160x120", "dense"])
def test_make_coarse_depth_on_device_bit_exact(capi, orc, synth, cfg):
    """dmv_ct_make_coarse_depth == makeCoarseDepthL0: the pc_u / pc_v / pc_idepth / pc_color lists of every level equal the oracle's
    (itself equal to the reference's compiled code) in values AND order."""
    T = synth.make_tracking_pair(**cfg)
    oct_ = orc.CoarseTracker(T["w"], T["h"], T["K"], 0)
    oct_.make_coarse_depth(T["Ku"], T["Kv"], T["new_idepth"], T["HdiF"], T["pyr_ref"])
    L = oct_.levels
    g = capi.CT(T["w"], T["h"], L, max_points=65536)
    for l in range(L):
        g.upload_new(l, T["pyr_ref"][l])                  # the reference frame is the resident frame
    pc_n = g.make_coarse_depth(T["Ku"], T["Kv"], T["new_idepth"], T["HdiF"])
    for l in range(L):
        po, pg = oct_.ref_points(l), g.get_ref(l)
        assert pc_n[l] == len(po["u"])
        for k in po:
            np.testing.assert_array_equal(pg[k], po[k], err_msg=f"lvl{l} pc_{k}")
    # colliding splats (several residuals in one pixel) are folded in input order
    Ku = np.concatenate([T["Ku"], T["Ku"][:50], T["Ku"][:50], T["Ku"][:20]]); Kv = np.concatenate([T["Kv"], T["Kv"][:50], T["Kv"][:50], T["Kv"][:20]])
    nid = np.concatenate([T["new_idepth"], T["new_idepth"][:50] * 1.1, T["new_idepth"][:50] * 0.9, T["new_idepth"][:20] * 1.3]).astype(np.float32)
    Hd = np.concatenate([T["HdiF"], T["HdiF"][:50] * 2, T["HdiF"][:50] * 0.5, T["HdiF"][:20] * 3]).astype(np.float32)
    oct_.make_coarse_depth(Ku, Kv, nid, Hd, T["pyr_ref"])
    g.make_coarse_depth(Ku, Kv, nid, Hd)
    for l in range(L):
        po, pg = oct_.ref_points(l), g.get_ref(l)
        for k in po:
            np.testing.assert_array_equal(pg[k], po[k], err_msg=f"collisions lvl{l} pc_{k}")
    g.close()
