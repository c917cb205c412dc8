"""GPU tests of the C++ host adapters (dmvio_b200::WindowBA / CoarseTracker) that mirror the reference's C++ surface:
the whole FullSystem::optimize GN/LM loop and CoarseTracker::trackNewestCoarse against the CPU oracle."""
import numpy as np
import pytest

from helpers import rel

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def hostapi():
    import dmvio_b200.capi as c
    if c.lib().dmv_device_count() < 1:
        pytest.fail("no CUDA device visible: GPU tests must run on the B200 box")
    import dmvio_b200.hostapi as h
    return h


def test_host_tables_match_oracle(hostapi, orc, synth):
    W = synth.make_window(nf=5, npts=300, seed=3)
    ow = orc.Window(W)
    hw = hostapi.WindowBA(W)
    pc, adH, adT = hw.tables()
    np.testing.assert_allclose(pc, ow.precalc(), rtol=2e-6, atol=1e-4)
    a_o, t_o = ow.adjoints()
    np.testing.assert_allclose(adH, a_o, rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(adT, t_o, rtol=1e-12, atol=1e-12)
    hw.close()


@pytest.mark.parametrize("cfg", [dict(nf=4, npts=600, seed=13), dict(nf=7, npts=2000, seed=1234)], ids=["nf4", "nf7"])
def test_optimize_matches_oracle(hostapi, orc, synth, cfg):
    """FullSystem::optimize on the GPU (fused gn_step per iteration) vs the oracle's optimize: same accept/reject sequence,
    energies within 1e-4 relative, final frame states within 1e-5 absolute (unscaled state units), depths within 1e-4 relative."""
    W = synth.make_window(state_noise=2e-3, **cfg)
    ow = orc.Window(W)
    n_o, log_o = ow.optimize(6, precision=1)
    hw = hostapi.WindowBA(W)
    n_g, log_g = hw.optimize(6)
    assert n_g == n_o
    assert len(log_g) == len(log_o)
    # energies AFTER a step inherit the fp32 differences of the solved increment (the reduced system is conditioned ~1e7): 3e-4, the first
    # (pure linearisation) entry 2e-5
    assert abs(log_g[0] - log_o[0]) <= 2e-5 * abs(log_o[0])
    np.testing.assert_allclose(log_g, log_o, rtol=3e-4)
    st_g, id_g, th_g = hw.states()
    st_o = ow.frame_states()
    assert np.abs(st_g - st_o).max() < 2e-5
    id_o = ow.point_outputs()["idepth"]
    np.testing.assert_allclose(id_g, id_o, rtol=2e-3, atol=2e-4)
    np.testing.assert_allclose(th_g, ow.frame_tables()["frameEnergyTH"], rtol=2e-3)
    assert log_g[-1] < 0.6 * log_g[0]
    hw.close()


def test_device_pyramid_frames(hostapi, orc, synth):
    """frames uploaded as raw images (level-0 [I,dx,dy] built on the device) give the same linearisation as host-built dI."""
    W = synth.make_window(nf=3, npts=300, seed=8)
    a = hostapi.WindowBA(W, use_device_pyramid=False)
    b = hostapi.WindowBA(W, use_device_pyramid=True)
    ea, eb = a.linearize(), b.linearize()
    assert abs(ea - eb) <= 1e-6 * abs(ea)
    a.close(); b.close()


@pytest.mark.parametrize("device_lm", [False, True], ids=["host_lm", "device_lm"])
@pytest.mark.parametrize("levels", [4, 5])
@pytest.mark.parametrize("npts", [2000, 12000])
def test_track_newest_coarse(hostapi, orc, synth, npts, levels, device_lm):
    """npts=12000 puts 54 195 reference points on level 0: more than a 16-CTA cluster keeps in registers (16 384), so dmv_ct_track
    streams the rest of the level from global memory."""
    T = synth.make_tracking_pair(seed=4321, levels=levels if levels == 5 else 0, npts=npts)
    oct_ = orc.CoarseTracker(T["w"], T["h"], T["K"], levels if levels == 5 else 0)
    oct_.make_coarse_depth(T["Ku"], T["Kv"], T["new_idepth"], T["HdiF"], T["pyr_ref"])
    oct_.set_new_frame(T["pyr_new"])
    r_o = oct_.track(np.eye(3), np.zeros(3), 0.0, 0.0)
    g = hostapi.CoarseTracker(T["w"], T["h"], T["K"], levels)
    counts = g.set_ref(T["Ku"], T["Kv"], T["new_idepth"], T["HdiF"], T["pyr_ref"])
    assert counts == [len(oct_.ref_points(l)["u"]) for l in range(levels)]
    g.set_new_image(T["img_new"])
    r_g = g.track(np.eye(3), np.zeros(3), 0.0, 0.0, device_lm=device_lm)
    assert r_g["evaluations"] >= r_g["iterations"] >= levels
    assert r_g["good"] == r_o["good"]
    assert np.abs(r_g["R"] - r_o["R"]).max() < 2e-5
    assert np.abs(r_g["t"] - r_o["t"]).max() < 2e-5
    assert abs(r_g["a"] - r_o["a"]) < 1e-3 and abs(r_g["b"] - r_o["b"]) < 5e-2
    np.testing.assert_allclose(r_g["lastResiduals"][:levels], r_o["lastResiduals"][:levels], rtol=2e-3)
    assert abs(r_g["iterations"] - r_o["iterations"]) <= 2
    assert np.linalg.norm(r_g["t"] - T["t_true"]) < 5e-4
    g.close()


def test_track_with_device_built_reference(hostapi, orc, synth):
    """setCoarseTrackingRef entirely on the device (raw keyframe image in, pc_* lists never leave the GPU) gives the same track as the host-built reference."""
    T = synth.make_tracking_pair(seed=4321)
    L = T["levels"]
    a = hostapi.CoarseTracker(T["w"], T["h"], T["K"], L)
    b = hostapi.CoarseTracker(T["w"], T["h"], T["K"], L)
    ca = a.set_ref(T["Ku"], T["Kv"], T["new_idepth"], T["HdiF"], T["pyr_ref"])
    cb = b.set_ref_device(T["Ku"], T["Kv"], T["new_idepth"], T["HdiF"], T["img_ref"])
    assert ca == cb
    a.set_new_image(T["img_new"]); b.set_new_image(T["img_new"])
    ra, rb = a.track(np.eye(3), np.zeros(3), 0.0, 0.0), b.track(np.eye(3), np.zeros(3), 0.0, 0.0)
    np.testing.assert_array_equal(ra["R"], rb["R"]); np.testing.assert_array_equal(ra["t"], rb["t"])
    assert ra["iterations"] == rb["iterations"]
    a.close(); b.close()


def test_marginalize_points_after_optimize(hostapi, orc, synth):
    """makeKeyFrame's point marginalisation through the C++ adapter (WindowBA::marginalizePointsF): after the same optimize() on both
    sides the marginalisation prior HM/bM matches the oracle's marginalizePointsF (tolerances: those of the optimised states it is
    linearised at), the listed points and their residuals are gone, and the smaller window keeps optimising."""
    W = synth.make_window(nf=5, npts=800, seed=17, state_noise=2e-3)
    ow = orc.Window(W)
    ow.optimize(4, precision=1)
    hw = hostapi.WindowBA(W)
    hw.optimize(4)
    po = ow.point_outputs()
    idepth_hessian = np.where(po["HdiF"] > 0, 1.0 / np.maximum(po["HdiF"], 1e-30), 0.0)
    rng = np.random.default_rng(0)
    well = np.nonzero(idepth_hessian > 200)[0]                      # far from setting_minIdepthH_marg = 50: both sides marginalise all of them
    marg = np.sort(rng.choice(well, len(well) // 3, replace=False)).astype(np.int32)
    rest = np.setdiff1d(np.arange(len(W["host"])), marg)
    drop = np.sort(rng.choice(rest, 20, replace=False)).astype(np.int32)
    o = ow.marginalize(marg, precision=1)
    g = hw.marginalize_points(marg, drop)
    assert g["npts"] == len(W["host"]) - len(marg) - len(drop)
    assert g["nres"] == int((~np.isin(W["res_point"], np.concatenate([marg, drop]))).sum())
    assert abs(g["resInM"] - o["resInM"]) <= max(2, o["resInM"] // 500)
    assert rel(g["HM"], o["HM"]) < 2e-3
    assert rel(g["bM"], o["bM"]) < 2e-2     # signed sums of res_toZeroF at slightly different optima
    assert np.allclose(g["HM"], g["HM"].T, rtol=1e-9, atol=1e-9 * np.abs(g["HM"]).max())
    e0 = hw.linearize()
    assert np.isfinite(e0) and e0 > 0
    n, log = hw.optimize(3)
    assert n >= 1 and np.all(np.isfinite(log))
    hw.close()


def test_finish_optimize_matches_oracle(hostapi, orc, synth):
    """The tail of FullSystem::optimize (FullSystemOptimize.cpp:L591-609) through WindowBA::finishOptimize: setEvalPT of the newest frame,
    linearizeAll(true) with its bookkeeping (maxRelBaseline, numGoodResiduals, deletion of the residuals that are not IN), and a second
    optimize() on the thinned window (resetOOB on the device, deleted residuals stay out) against the oracle."""
    W = synth.make_window(nf=5, npts=600, seed=21, state_noise=2e-3)
    nres = len(W["res_point"])
    ow = orc.Window(W)
    ow.optimize(4, precision=1)
    E_o, rem_o = ow.finish_optimize()
    hw = hostapi.WindowBA(W)
    hw.optimize(4)
    E_g, rem_g = hw.finish_optimize()
    assert abs(E_g - E_o) <= 2e-4 * abs(E_o)
    ties = np.setxor1d(rem_o, rem_g)
    assert len(ties) <= max(2, nres // 500), ties                     # identical up to energy-threshold ties
    assert hw.nres == nres - len(rem_g)
    touched = np.unique(np.asarray(W["res_point"])[ties]) if len(ties) else np.zeros(0, int)
    ok = np.ones(len(W["host"]), bool); ok[touched] = False
    ps_o, ps_g = ow.point_stats(), hw.point_stats()
    np.testing.assert_array_equal(ps_g["numGoodResiduals"][ok], ps_o["numGoodResiduals"][ok])
    np.testing.assert_allclose(ps_g["maxRelBaseline"][ok], ps_o["maxRelBaseline"][ok], rtol=2e-3, atol=1e-6)
    st_g, _, th_g = hw.states()
    st_o = ow.frame_states()
    assert np.all(st_g[-1, :6] == 0)                                  # the newest frame's pose now lives in its evaluation point
    assert np.abs(st_g - st_o).max() < 2e-5
    np.testing.assert_allclose(th_g, ow.frame_tables()["frameEnergyTH"], rtol=2e-3)
    if len(ties) == 0:
        n_o, log_o = ow.optimize(3, precision=1)
        n_g, log_g = hw.optimize(3)
        assert abs(n_g - n_o) <= 1                                    # near the optimum the convergence test can fire one iteration apart
        m = min(len(log_g), len(log_o))
        np.testing.assert_allclose(log_g[:m], log_o[:m], rtol=5e-4)
    hw.close()


def test_flag_points_for_removal_rules(hostapi, orc, synth):
    """WindowBA::flagPointsForRemoval (FullSystem.cpp:L785-879 with PointHessian::isOOB / isInlierNew) against a numpy restatement of the
    rules on the adapter's own bookkeeping, then the flagged points go through marginalizePointsF."""
    W = synth.make_window(nf=6, npts=500, seed=29, state_noise=1e-3, hosts="all")
    hw = hostapi.WindowBA(W)
    hw.optimize(3)
    for _ in range(4):                                                # numGoodResiduals grows by the active residuals at every keyframe optimisation
        E, rem = hw.finish_optimize()
        # the adapter compacts its residual list: track it the same way
        W["res_point"] = np.asarray(W["res_point"])[np.setdiff1d(np.arange(len(W["res_point"])), rem)]
        W["res_target"] = np.asarray(W["res_target"])[np.setdiff1d(np.arange(len(W["res_target"])), rem)]
    npts = len(W["host"])
    rng = np.random.default_rng(4)
    last_t = np.tile(np.asarray(W["frameID"])[[-1, -2]], (npts, 1)).astype(np.int32)
    last_s = rng.choice([0, 1, 2], (npts, 2), p=[0.8, 0.1, 0.1]).astype(np.int32)
    hw.set_last_residuals(last_t, last_s)
    flagged = [0]
    marg, drop = hw.flag_points(flagged)
    _, idepth, _ = hw.states()
    ps = hw.point_stats()
    nres_p = np.bincount(W["res_point"], minlength=npts)
    vis = np.bincount(W["res_point"][np.isin(W["res_target"], flagged)], minlength=npts)     # every remaining residual is IN after linearizeAll(true)
    exp_m, exp_d = [], []
    for i in range(npts):
        if idepth[i] < 0.02 or nres_p[i] == 0:
            exp_d.append(i); continue
        oob = (nres_p[i] >= 3 and ps["numGoodResiduals"][i] > 14 and nres_p[i] - vis[i] < 3)
        if not oob:
            oob = last_s[i, 0] == 1 or (nres_p[i] >= 2 and last_s[i, 0] == 2 and last_s[i, 1] == 2)
        if not oob and W["host"][i] != 0:
            continue
        (exp_m if (nres_p[i] >= 3 and ps["numGoodResiduals"][i] >= 4) else exp_d).append(i)
    np.testing.assert_array_equal(marg, np.asarray(exp_m, np.int32))
    np.testing.assert_array_equal(drop, np.asarray(exp_d, np.int32))
    assert len(marg) > 20 and len(drop) > 0
    g = hw.marginalize_points(marg, drop)
    assert g["npts"] == npts - len(drop) - len(marg) and g["resInM"] > 0
    assert np.isfinite(hw.linearize())
    hw.close()


def test_keyframe_turnover_flow(hostapi, orc, synth):
    """The makeKeyFrame sequence on the adapter: optimize -> tail -> flagPointsForRemoval(frame 0) -> marginalizePointsF -> marginalizeFrame(0)
    (FullSystemMarginalize.cpp:L156-219 + EnergyFunctional.cpp:L522-675).  The prior that comes out is exactly host/marg_frame.h applied to
    the prior after the point marginalisation (that function is pinned to the reference through the oracle on the CPU); the window of
    nf - 1 frames keeps optimising with the prior in place."""
    nf = 6
    W = synth.make_window(nf=nf, npts=500, seed=31, state_noise=1e-3, hosts="all")
    prior0 = orc.Window(W).frame_tables()["prior"][0]
    hw = hostapi.WindowBA(W)
    hw.optimize(3)
    hw.finish_optimize()
    marg, drop = hw.flag_points([0])
    assert len(marg) > 10
    g = hw.marginalize_points(marg, drop)
    assert g["resInM"] > 0 and np.abs(g["HM"]).max() > 0
    st, _, _ = hw.states()
    exp_H, exp_b = hostapi.marginalize_frame_hm(g["HM"], g["bM"], nf, 0, prior0, st[0][:8])
    nres_before = hw.nres
    m = hw.marginalize_frame(0)
    assert m["nf"] == nf - 1 and m["HM"].shape == (8 * (nf - 1) + 4,) * 2
    assert rel(m["HM"], exp_H) < 1e-12 and rel(m["bM"], exp_b) < 1e-12
    assert m["nres"] < nres_before                                   # the observations in the marginalised frame are gone
    e = hw.linearize()
    assert np.isfinite(e) and e > 0
    eL, eM = hw.energies_LM()
    assert eM != 0                                                    # the prior is active: the window sits off the marginalisation point
    n, log = hw.optimize(3)
    eL1, eM1 = hw.energies_LM()
    # what the LM loop minimises (FullSystemOptimize.cpp:L548-551); log[0] / log[-1] are the photometric energies at the same two states
    assert log[-1] + eL1 + eM1 <= (log[0] + eL + eM) * (1 + 1e-9)
    # the log holds the photometric energy only; steps are accepted on photometric + prior energies (L + M), so with the marginalisation
    # prior in place the photometric part may give a little while the total goes down
    assert n >= 1 and np.all(np.isfinite(log)) and log[-1] <= log[0] * 1.01
    st2, _, _ = hw.states()
    assert st2.shape[0] == nf - 1
    hw.close()


def test_ba_adopts_the_frame_resident_in_the_tracker_handle(orc, synth):
    """SURVEY §8f-1: a frame crosses PCIe once.  dmv_ba_adopt_frame (device-to-device copy of the level-0 plane the coarse-tracker handle built
    when the frame arrived) gives bit-identical BA results to uploading the image to the BA handle a second time."""
    import dmvio_b200.capi as capi
    W = synth.make_window(nf=3, npts=400, seed=23)
    ow = orc.Window(W)

    def load(ba):
        ba.set_window(W["nf"])
        ba.set_points(W["host"], W["u"], W["v"], W["idepth"], W["idepth_zero"], W["color"], W["weights"])
        ba.set_residuals(W["res_point"], W["res_target"])
        ba.set_adjoints(*ow.adjoints())
        ba.set_state(ow.calib()["k8"], ow.precalc(), ow.frame_tables()["frameEnergyTH"])
        r = ba.linearize(); ba.apply_res()
        return r, ba.accumulate()

    ba1 = capi.BA(W["w"], W["h"], max_frames=3, max_points=len(W["host"]))
    for k in range(3):
        ba1.upload_image(k, W["images"][k])
    ct = capi.CT(W["w"], W["h"], synth.pyr_levels(W["w"], W["h"]), max_points=1024)
    ba2 = capi.BA(W["w"], W["h"], max_frames=3, max_points=len(W["host"]))
    for k in range(3):
        ct.upload_new_image(W["images"][k])   # the tracker receives the frame (H2D + device pyramid) ...
        ba2.adopt_frame(k, ct)                # ... the mapper takes its level-0 plane from there
    r1, a1 = load(ba1)
    r2, a2 = load(ba2)
    assert r1["energy"] == r2["energy"] and r1["n_in"] == r2["n_in"]
    for k in ("HA", "bA", "Hsc", "bsc"):
        np.testing.assert_array_equal(a1[k], a2[k])
    ba1.close(); ba2.close(); ct.close()
