"""Multi-rank GPU tests of the sharded BA path (2, 4 and 8 ranks; each is skipped when the box has fewer GPUs): one process per GPU,
points sharded (dmvio_b200.sharding), systems all-reduced (a) inside ba_fused_kernel over NVLink peer memory and (b) by NCCL.
Checks: every rank ends with the bit-identical system; it equals the UNSHARDED oracle system within the single-GPU tolerances
(shard-sum invariance, reference AccumulatedSCHessian.cpp:L62-76)."""
import os
import socket

import numpy as np
import pytest

from helpers import rel

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, cfg, mode, q):
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import torch.distributed as dist
    import dmvio_b200.capi as capi
    import dmvio_b200.hostmath as hm
    import dmvio_b200.synth as synth
    from dmvio_b200.sharding import shard_window
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    W = synth.make_window(**cfg)
    S = shard_window(W, rank, world)
    ba = capi.BA(W["w"], W["h"], max_frames=W["nf"], max_points=len(S["host"]), device=rank)
    for k in range(W["nf"]):
        ba.upload_frame(k, S["dI"][k])
    ba.set_window(W["nf"])
    ba.set_points(S["host"], S["u"], S["v"], S["idepth"], S["idepth_zero"], S["color"], S["weights"])
    ba.set_residuals(S["res_point"], S["res_target"])
    ba.set_adjoints(*hm.adjoints(S))
    k8, pc, TH = hm.calib8(S["K"]), hm.precalc_table(S), S["frameEnergyTH"]
    if mode == "p2p":
        handles = [None] * world
        dist.all_gather_object(handles, ba.p2p_export())
        ba.p2p_import(world, rank, handles)
    else:
        uid = [capi.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ba.comm_init(world, rank, uid[0])
    ba.set_state(k8, pc, TH)
    out = []
    r = ba.linearize()
    states = (S["shard_res_index"], ba.residual_outputs()["newState"])
    ba.apply_res()
    a = ba.accumulate()
    out.append((r["energy"], r["n_in"], a["HA"].copy(), a["bA"].copy(), a["Hsc"].copy(), a["bsc"].copy()))
    # sharded point marginalisation: every rank marginalises ITS share of the flagged points, the partial M / Msc are summed in the launch
    from oracle import orc as _orc
    ow = _orc.Window(W)
    flagged = np.arange(0, len(W["host"]), 3)
    keep = np.nonzero((np.arange(len(W["host"])) % world) == rank)[0]            # dmvio_b200.sharding.shard_points
    local = np.nonzero(np.isin(keep, flagged))[0].astype(np.int32)
    g = ba.marginalize_points(local, ow.adHTdeltaF(), ow.calib()["cDeltaF"])
    marg = (g["M"].copy(), g["Msc"].copy(), g["Mb"].copy(), g["Mbsc"].copy(), g["resInM"])
    # a few fused GN steps: exercises the parity double-buffering of the inbox
    HL, bL = hm.prior_system(W)
    ba.backup_points()
    for _ in range(5):
        x = hm.solve_reduced(a["HA"], a["bA"], a["Hsc"], a["bsc"], HL, bL, lam=1e-5)
        r = ba.gn_step(x, k8, pc, TH)
        ba.apply_res()
        a = ba.accumulate()
        ba.backup_points()
    out.append((r["energy"], r["n_in"], a["HA"].copy(), a["bA"].copy(), a["Hsc"].copy(), a["bsc"].copy()))
    q.put((rank, out + [states, marg]))
    dist.barrier()
    ba.close()
    dist.destroy_process_group()


@pytest.mark.parametrize("world,mode", [(2, "p2p"), (2, "nccl"), (4, "p2p"), (8, "p2p"), (8, "nccl")])
def test_sharded_exchange(orc, synth, world, mode):
    import dmvio_b200.capi as capi
    if capi.lib().dmv_device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    import torch.multiprocessing as mp
    cfg = dict(nf=5, npts=901, seed=17) if world == 2 else dict(nf=7, npts=250 * world + 3, seed=17 + world)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, cfg, mode, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=300) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for it in range(2):
        e0, n0, *m0 = res[0][it]
        for rk in range(1, world):
            e1, n1, *m1 = res[rk][it]
            assert e0 == e1 and n0 == n1
            for a, b in zip(m0, m1):
                np.testing.assert_array_equal(a, b)  # bit-identical on every rank
    W = synth.make_window(**cfg)
    ow = orc.Window(W)
    ow.linearize_all(update_th=False)
    full = np.zeros(ow.nres, np.int32)
    for rk in range(world):   # the ranks' classifications, imposed on the oracle (threshold ties): the comparison below is unconditional
        idx, ns = res[rk][2]
        full[idx] = ns
    E, _, unfixable = ow.override_new_states(full)
    assert unfixable == 0
    ow.apply_res()
    a = ow.accumulate(1)
    # sharded marginalisation: identical on every rank, equal to the unsharded oracle's marginalizePointsF of the same points
    for rk in range(1, world):
        for x, y in zip(res[0][3][:4], res[rk][3][:4]):
            np.testing.assert_array_equal(x, y)
    om = orc.Window(W).marginalize(np.arange(0, len(W["host"]), 3).astype(np.int32), precision=1)
    M, Msc, Mb, Mbsc, nM = res[0][3]
    assert nM == om["resInM"]
    assert rel(M, om["M"]) < 1e-5 and rel(Msc, om["Msc"]) < 1e-5 and rel(Mb, om["Mb"]) < 2e-4 and rel(Mbsc, om["Mbsc"]) < 2e-4
    e0, n0, HA, bA, Hsc, bsc = res[0][0]
    assert abs(e0 - E) <= 2e-5 * abs(E)
    assert rel(HA, a["HA"]) < 1e-5 and rel(Hsc, a["Hsc"]) < 1e-5
    assert rel(bA, a["bA"]) < 1e-4 and rel(bsc, a["bsc"]) < 1e-4


def _flow(hw, nf):
    """the makeKeyFrame sequence on the adapter (as tests/test_gpu_host.py::test_keyframe_turnover_flow)"""
    out = {}
    n1, log1 = hw.optimize(4)
    E_tail, removed = hw.finish_optimize()
    marg, drop = hw.flag_points([0])
    g = hw.marginalize_points(marg, drop)
    m = hw.marginalize_frame(0)
    n2, log2 = hw.optimize(3)
    st, idd, th = hw.states()
    out.update(n1=n1, log1=log1, E_tail=E_tail, removed=removed, marg=marg, drop=drop, resInM=g["resInM"], HM=m["HM"], bM=m["bM"], nres=m["nres"],
               n2=n2, log2=log2, st=st, idepth=idd, th=th)
    return out


def _worker_window(rank, world, port, cfg, mode, q):
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import torch
    import torch.distributed as dist
    import dmvio_b200.capi as capi
    import dmvio_b200.hostapi as hostapi
    import dmvio_b200.synth as synth
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)

    def allgather(data):   # the application's host communicator (here gloo)
        t = torch.frombuffer(bytearray(data), dtype=torch.uint8)
        outs = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(outs, t)
        return b"".join(o.numpy().tobytes() for o in outs)

    W = synth.make_window(**cfg)
    shard = dict(rank=rank, nranks=world, allgather=allgather, exchange=mode)
    if mode == "nccl":
        uid = [capi.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        shard["uid"] = uid[0]
    hw = hostapi.WindowBA(W, device=rank, shard=shard)
    out = _flow(hw, W["nf"])
    q.put((rank, out))
    dist.barrier()
    hw.close()
    dist.destroy_process_group()


@pytest.mark.parametrize("world,mode", [(2, "p2p"), (2, "nccl"), (4, "p2p")])
def test_window_ba_sharded(synth, world, mode):
    """The C++ adapter in sharded mode (WindowBA::setSharding): every rank runs the SAME host logic on the all-reduced system; per-point read-backs
    are gathered through the application's host allgather.  The whole makeKeyFrame flow (optimize, tail with residual removal, flagPointsForRemoval,
    marginalizePointsF, marginalizeFrame, optimize again) must take the same decisions as the unsharded adapter and end in the same state."""
    import dmvio_b200.capi as capi
    import dmvio_b200.hostapi as hostapi
    if capi.lib().dmv_device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    import torch.multiprocessing as mp
    cfg = dict(nf=6, npts=500 + world, seed=31, state_noise=1e-3, hosts="all")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker_window, args=(r, world, port, cfg, mode, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=300) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    ref = _flow(hostapi.WindowBA(synth.make_window(**cfg)), cfg["nf"])
    for rk in range(world):
        o = res[rk]
        # identical host decisions on every rank and the unsharded adapter
        assert (o["n1"], o["n2"], o["resInM"], o["nres"]) == (ref["n1"], ref["n2"], ref["resInM"], ref["nres"])
        np.testing.assert_array_equal(o["marg"], ref["marg"]); np.testing.assert_array_equal(o["drop"], ref["drop"])
        np.testing.assert_array_equal(o["removed"], ref["removed"])
        np.testing.assert_allclose(o["log1"], ref["log1"], rtol=3e-4)
        np.testing.assert_allclose(o["log2"], ref["log2"], rtol=3e-4)
        assert abs(o["E_tail"] - ref["E_tail"]) <= 3e-4 * abs(ref["E_tail"])
        assert rel(o["HM"], ref["HM"]) < 1e-4 and rel(o["bM"], ref["bM"]) < 1e-3
        assert np.abs(o["st"] - ref["st"]).max() < 2e-5
        np.testing.assert_allclose(o["idepth"], ref["idepth"], rtol=2e-3, atol=2e-4)
        np.testing.assert_allclose(o["th"], ref["th"], rtol=2e-3)
    for rk in range(1, world):   # the ranks agree bit for bit (same all-reduced system, same host arithmetic)
        np.testing.assert_array_equal(res[rk]["st"], res[0]["st"])
        np.testing.assert_array_equal(res[rk]["HM"], res[0]["HM"])
        np.testing.assert_array_equal(res[rk]["idepth"], res[0]["idepth"])
