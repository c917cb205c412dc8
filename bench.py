#!/usr/bin/env python
"""bench.py — headline benchmark of the DM-VIO photometric BA hot path on B200 (BASELINE.json metric).

One "step" = one Gauss-Newton iteration of the hot path on the 7-keyframe / 2000-point / 640x480 synthetic window
(SURVEY.md §8d): resubstitute(x) + point step, residual/Jacobian evaluation of every active point-residual, per-pair
Hessian blocks, per-point Schur complement, adjoint products to the dense (8nf+4)^2 system — ONE kernel launch
(ba_fused_kernel); the dense host solve is excluded, as in the metric's definition.

  value      device-resident throughput: all inputs in HBM, CUDA-event time of the launch, L2 scrubbed between steps
  e2e        the same step through the C ABI call a DM-VIO host makes (dmv_ba_gn_step + dmv_ba_apply_res):
             host buffers in, H/b out, host<->device traffic and the stream synchronisation inside the timed region
  roofline   algorithmic bytes of ba_fused_kernel / its CUDA-event duration vs the measured HBM peak
  roofline_batched   the same kernel body over B independent windows in ONE launch (planes of B windows exceed L2): the
             regime in which the HBM roofline is meaningful (SURVEY.md §8d "batched variant")
  parity     H_A, b_A, H_sc, b_sc of the first step (all-reduced over the ranks) vs the UNSHARDED CPU oracle, outside the
             timed region; the run fails above 1e-5 / 1e-4
  cpu_baseline   the CPU oracle (restatement of the reference's SSE path) on this host (N = 1 only)

N > 1 (torchrun): the headline is weak scaling — every rank owns 2000 points of one N*2000-point window (images and tables
replicated), the system is all-reduced inside the kernel over NVLink peer memory.  The same line also carries
  strong     2000 points in total split over the N ranks (BASELINE's metric window at N GPUs)
  config4    BASELINE config 4: 8000 points in total split over the N ranks
`--impl reference` times the CPU path only (rank 0), same metric/config.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "point-residuals/sec per GN iter (7 KF, 2000 pts, 640x480)"
UNIT = "point-residuals/s"
NF, NPTS, W_, H_ = 7, 2000, 640, 480
PARITY_TOL = {"HA": 1e-5, "Hsc": 1e-5, "bA": 1e-4, "bsc": 1e-4, "energy": 2e-5}


class ClockSampler:
    """SM clock + clock-event reasons sampled WHILE the timed regions run (NVML in a thread, 2 ms period; the timed regions of
    this benchmark last only tens of milliseconds, so the 100-200 ms nvidia-smi loop of B200_PROFILING.md would see nothing)."""

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.samples = []   # (t, sm_mhz, reasons_bitmask, power_w)
        self.stop_flag = False
        self.t = None
        self.h = None
        self.smax = None
        self.windows = []   # (t0, t1) of the timed regions

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)  # NVML index == CUDA ordinal on the gpurun boxes
            self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.h = None
            return
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def _run(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                mhz = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                rs = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                try:
                    pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                except Exception:
                    pw = float("nan")
                self.samples.append((time.perf_counter(), mhz, rs, pw))
            except Exception:
                pass
            time.sleep(0.002)

    def mark(self, t0, t1):
        self.windows.append((t0, t1))

    def stop(self):
        if self.h is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"], "samples": 0}
        self.stop_flag = True
        self.t.join(timeout=1)
        nv = self.nv
        inside = [s for s in self.samples if any(a <= s[0] <= b for a, b in self.windows)]
        use = inside if len(inside) >= 3 else self.samples
        names = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap,
                 "hw_power_brake": nv.nvmlClocksEventReasonHwPowerBrakeSlowdown}
        reasons = sorted(n for n, bit in names.items() if any(s[2] & bit for s in use))
        sm = [s[1] for s in use]
        pw = [s[3] for s in use if s[3] == s[3]]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.smax, "reasons": reasons, "samples": len(use),
                "samples_scope": "inside the timed regions" if use is inside else "whole run (timed regions too short to sample)",
                "power_w_max": max(pw) if pw else None}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(pattern="*_ba_fused_summary.md"):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the newest committed `ncu --set full` capture of the kernel
    (profiles/<pattern>, written by tools/summarize_profiles.py); None if there is none."""
    import glob
    import re
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", pattern)))
    if not files:
        return None, None
    rd = wr = None
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    for line in open(files[-1]):
        m = re.match(r"\| dram__bytes_(read|write)\.sum \| ([0-9.]+) \| (\w+) \|", line)
        if m:
            v = float(m.group(2)) * unit.get(m.group(3), 1.0)
            if m.group(1) == "read" and rd is None:
                rd = v
            if m.group(1) == "write" and wr is None:
                wr = v
    if rd is None:
        return None, None
    return rd + (wr or 0.0), os.path.relpath(files[-1], ROOT)


def algorithmic_bytes(nres, npts, nf):
    """SURVEY.md §8d: B_alg = 436*nres + 112*npts + 8*(8nf+4)(8nf+5)."""
    N = 8 * nf + 4
    return 436 * nres + 112 * npts + 8 * N * (N + 1)


# ----------------------------------------------------------------------------------------------------------------- CPU legs
def _pin(threads):
    """pin the process (and the worker threads it creates) to `threads` logical CPUs: less migration noise on a shared host"""
    try:
        cpus = sorted(os.sched_getaffinity(0))
        if len(cpus) > threads:
            os.sched_setaffinity(0, set(cpus[:threads]))
            return cpus[:threads]
    except Exception:
        pass
    return None


def _unpin(all_cpus):
    try:
        os.sched_setaffinity(0, all_cpus)
    except Exception:
        pass


def cpu_rate(W, seconds, threads, kind="port", blocks=5, pin=True):
    """times the CPU path's hot iteration (accumulate + stitch, resubstitute, step, linearizeAll, applyRes) for >= `seconds` in `blocks`
    blocks; returns median-of-blocks rate.  kind = "port": the oracle restatement; "reference": the reference's own translation units
    (oracle/_ref/libdso_ref.so, built from /root/reference over stand-in Eigen headers — slower than the port, DESIGN.md §2)."""
    all_cpus = os.sched_getaffinity(0)
    pinned = _pin(threads) if pin else None
    try:
        if kind == "reference":
            from oracle import ref
            ow = ref.Window(W, nthreads=threads)
        else:
            from oracle import orc
            ow = orc.Window(W, nthreads=threads)
        ow.linearize_all(update_th=False)
        ow.apply_res()
        x, _, _ = ow.solve(0, 1e-5, 0)
        for _ in range(3):
            ow.hot_iteration(x, 0)
        rates, total = [], 0
        for _ in range(blocks):
            t0 = time.perf_counter()
            n = 0
            while True:
                ow.hot_iteration(x, 0)
                n += 1
                if time.perf_counter() - t0 >= seconds / blocks:
                    break
            rates.append(ow.nres * n / (time.perf_counter() - t0))
            total += n
        return {"rate": float(np.median(rates)), "rate_min": float(min(rates)), "rate_max": float(max(rates)), "iters": total,
                "ms_per_iter": ow.nres / float(np.median(rates)) * 1e3, "pinned_cpus": len(pinned) if pinned else None, "nres": ow.nres}
    finally:
        _unpin(all_cpus)


def pick_threads(W, candidates=(6, 12, 24, 48), seconds=1.0):
    """the reference hard-codes NUM_THREADS = 6 (util/settings.h); its worker pool restated in the oracle takes any count, so the
    CPU arm is given the best of a few counts on this host (favouring the baseline)."""
    best = (0.0, 6)
    ncpu = os.cpu_count() or 1
    rates = {}
    for t in candidates:
        if t > ncpu:
            continue
        r = cpu_rate(W, seconds, t, blocks=2)["rate"]
        rates[t] = r
        if r > best[0]:
            best = (r, t)
    return best[1], rates


def run_ref_courtesy(npts):
    """child process of run_reference: the reference's OWN translation units (oracle/_ref) on the same window, 6 threads"""
    import dmvio_b200.synth as synth
    W = synth.make_window(nf=NF, npts=npts, w=W_, h=H_, seed=1234)
    rr = cpu_rate(W, 2.0, 6, kind="reference", blocks=2)
    print(json.dumps({"value": rr["rate"], "cores": 6, "kind": "reference", "iters": rr["iters"], "ms_per_iter": rr["ms_per_iter"],
                      "what": "ref_win_hot_iteration of oracle/_ref/libdso_ref.so = the reference's own sources compiled over stand-in Eigen/Sophus headers "
                              "(their heap temporaries make it slower than real Eigen would be): the lower bound of 'the reference's CPU path', the port is the upper one"}))


def run_reference(args, rank, world):
    if rank != 0:
        return
    import dmvio_b200.synth as synth
    W = synth.make_window(nf=NF, npts=NPTS * world, w=W_, h=H_, seed=1234)
    threads, rates = pick_threads(W)
    # a bounded sample that is long enough to mean something on a shared host: >= 4 s in 5 blocks, median (the driver's --steps is a
    # lower bound on the iteration count, not the sample size: 20 steps = 0.1 s measured anything between 2.4 and 3.5 M/s in round 1)
    seconds = max(4.0, args.steps * 0.005)
    r = cpu_rate(W, seconds, threads)
    val = r["rate"]
    ref_courtesy = None
    try:  # in a child process: the reference's objects print to stdout and abort() on paths the harness does not cover
        import subprocess
        if os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libdso_ref.so")):
            cp = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--ref-courtesy", "--points", str(NPTS * world)],
                                capture_output=True, text=True, timeout=120)
            last = [ln for ln in cp.stdout.splitlines() if ln.startswith("{")]
            ref_courtesy = json.loads(last[-1]) if last else {"unavailable": f"child rc={cp.returncode}"}
        else:
            ref_courtesy = {"unavailable": "oracle/_ref/libdso_ref.so not built"}
    except Exception as e:  # the courtesy number must never break the arm
        ref_courtesy = {"unavailable": str(e)[:200]}
    out = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": world, "steps": r["iters"], "warmup": 3,
        "ms_per_step": r["ms_per_iter"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"sliding window {NF} KF / {NPTS * world} pts / {W_}x{H_}, pattern 8, {r['nres']} point-residuals, one GN iteration "
                               "of the hot path per step (host solve excluded)"},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "value_min_block": r["rate_min"], "value_max_block": r["rate_max"],
                         "value_at_NUM_THREADS_6": rates.get(6),
                         "sample": f"{r['iters']} full GN iterations of the window in {seconds:.1f} s (5 blocks, median; process pinned to {r['pinned_cpus']} CPUs); oracle = CPU "
                                   f"restatement of the reference's SSE path, g++ -O3 (no -march, as the reference's CMakeLists), {threads} worker threads = best of "
                                   f"{{{', '.join(f'{t}: {v / 1e6:.2f} M/s' for t, v in rates.items())}}} on this {os.cpu_count()}-thread host (the reference hard-codes NUM_THREADS=6)",
                         "reference_sources_courtesy": ref_courtesy},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out))


# ----------------------------------------------------------------------------------------------------------------- GPU arm
class Dist:
    """torch.distributed plumbing (NCCL backend for the bootstrap, barriers and max-over-ranks; the data plane is the kernel's own)."""

    def __init__(self, world, local_rank):
        self.world = world
        self.dist = None
        if world > 1:
            import torch
            import torch.distributed as dist
            torch.cuda.set_device(local_rank)
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            self.dist, self.torch = dist, torch

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def max(self, v):
        if self.dist is None:
            return v
        t = self.torch.tensor([v], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def min_int(self, v):
        if self.dist is None:
            return v
        t = self.torch.tensor([v], device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
        return int(t.item())

    def gather(self, obj):
        if self.dist is None:
            return [obj]
        out = [None] * self.world
        self.dist.all_gather_object(out, obj)
        return out

    def bcast(self, obj, src=0):
        if self.dist is None:
            return obj
        box = [obj]
        self.dist.broadcast_object_list(box, src=src)
        return box[0]

    def close(self):
        if self.dist is not None:
            self.dist.destroy_process_group()


class Case:
    """one window (npts_total points in total) sharded over the ranks, loaded into a BA handle"""

    def __init__(self, D, rank, world, local_rank, npts_total, chunk, exchange, seed=1234):
        import dmvio_b200.capi as capi
        import dmvio_b200.hostmath as hm
        import dmvio_b200.synth as synth
        from dmvio_b200.sharding import shard_window
        self.D, self.rank, self.world = D, rank, world
        self.Wfull = synth.make_window(nf=NF, npts=npts_total, w=W_, h=H_, seed=seed)
        Wr = self.Wr = shard_window(self.Wfull, rank, world)
        self.nres_local, self.nres_total = len(Wr["res_point"]), len(self.Wfull["res_point"])
        ba = self.ba = capi.BA(W_, H_, max_frames=NF, max_points=len(Wr["host"]), device=local_rank, chunk_points=chunk)
        for k in range(NF):
            ba.upload_frame(k, Wr["dI"][k])
        ba.set_window(NF)
        ba.set_points(Wr["host"], Wr["u"], Wr["v"], Wr["idepth"], Wr["idepth_zero"], Wr["color"], Wr["weights"])
        ba.set_residuals(Wr["res_point"], Wr["res_target"])
        adH, adT = hm.adjoints(Wr)
        ba.set_adjoints(adH, adT)
        self.k8, self.precalc, self.TH = hm.calib8(Wr["K"]), hm.precalc_table(Wr), Wr["frameEnergyTH"].copy()
        self.exchange = "none"
        if world > 1:
            self.exchange = exchange
            if exchange == "p2p":
                try:
                    mine = ba.p2p_export()
                    handles = D.gather(mine)   # doubles as the barrier after every inbox has been zeroed
                    ba.p2p_import(world, rank, handles)
                    ok = 1
                except Exception as e:  # no peer access between these GPUs: fall back to NCCL on ALL ranks
                    sys.stderr.write(f"[rank {rank}] peer-memory exchange unavailable ({e}); using NCCL\n")
                    ok = 0
                if D.min_int(ok) == 0:
                    self.exchange = "nccl"
                    try:
                        ba.p2p_import(1, 0, [mine])  # nranks = 1 switches the peer exchange off again
                    except Exception:
                        pass
            if self.exchange == "nccl":
                ba.comm_init(world, rank, D.bcast(capi.nccl_unique_id() if rank == 0 else None))
        ba.set_state(self.k8, self.precalc, self.TH)
        self.r0 = ba.linearize()
        self.g0 = ba.residual_outputs()
        ba.apply_res()
        self.acc = ba.accumulate()
        HL, bL = hm.prior_system(Wr)
        self.x = hm.solve_reduced(self.acc["HA"], self.acc["bA"], self.acc["Hsc"], self.acc["bsc"], HL, bL, lam=1e-5)
        ba.backup_points()

    def parity(self):
        """first step vs the UNSHARDED oracle (test infrastructure, outside every timed region): the ranks' classifications are gathered and
        imposed on the oracle (threshold ties), then the all-reduced system every rank holds is compared on rank 0"""
        states = self.D.gather((self.Wr.get("shard_res_index"), self.g0["newState"]))
        if self.rank != 0:
            return None
        from oracle import orc
        full = np.zeros(self.nres_total, np.int32)
        for idx, ns in states:
            if idx is None:
                full[:] = ns
            else:
                full[idx] = ns
        ow = orc.Window(self.Wfull, nthreads=min(16, os.cpu_count() or 1))
        ow.linearize_all(update_th=False)
        E, nch, bad = ow.override_new_states(full)
        ow.apply_res()
        a = ow.accumulate(1)
        rel = lambda g, o: float(np.linalg.norm(np.asarray(g) - o) / max(np.linalg.norm(o), 1e-300))
        out = {k: rel(self.acc[k], a[k]) for k in ("HA", "bA", "Hsc", "bsc")}
        out["energy"] = abs(self.r0["energy"] - E) / abs(E)
        out["threshold_ties_imposed"] = nch
        out["unfixable_oob_ties"] = bad
        out["n_in"] = [int(self.r0["n_in"]), int(a["resInA"])]
        out["ok"] = bool(bad == 0 and all(out[k] <= PARITY_TOL[k] for k in PARITY_TOL) and int(self.r0["n_in"]) == int(a["resInA"]))
        out["tolerance"] = PARITY_TOL
        return out

    def outputs(self):
        """what the last GN step through the C ABI left for its caller: the committed system (dmv_ba_accumulate), the per-residual and
        per-point results and the updated depths; integer outputs as float64"""
        ba = self.ba
        out = ba.accumulate()
        out.update(ba.residual_outputs())
        out.update({"pt_" + k: v for k, v in ba.point_outputs().items()})
        out["idepth"], out["idepth_zero"] = ba.get_idepth()
        return {k: np.asarray(v, np.float64 if np.asarray(v).dtype.kind in "iub" else None) for k, v in out.items()}

    def measure(self, steps, warmup, sampler=None, dump=None):
        ba, D, x = self.ba, self.D, self.x
        for _ in range(max(3, warmup)):
            ba.gn_step(x, self.k8, self.precalc, self.TH)
            ba.apply_res()
        ba.bench_device(x, iters=max(3, warmup), flush_l2=True)
        launches0 = ba.launch_count()
        # ---- value: device-resident, CUDA events, L2 scrubbed between steps
        D.barrier()
        tw0 = time.perf_counter()
        ms_iter, ms_kernel, done = 0.0, 0.0, 0
        while done < steps:  # dmv_ba_bench_device takes at most 4096 iterations per call
            n = min(2048, steps - done)
            a, b_ = ba.bench_device(x, iters=n, flush_l2=True)
            ms_iter += a * n; ms_kernel += b_ * n; done += n
        ms_iter /= steps; ms_kernel /= steps
        D.barrier()
        if sampler:
            sampler.mark(tw0, time.perf_counter())
        ms_iter = D.max(ms_iter)
        # ---- e2e: the C ABI call with host buffers (tables in, kernel, H/b out, sync), wall clock
        D.barrier()
        tw0 = time.perf_counter()
        e2e_ms_c = ba.bench_e2e(x, self.k8, self.precalc, self.TH, iters=steps)  # the C ABI calls issued from C (what a C++ host pays)
        D.barrier()
        if sampler:
            sampler.mark(tw0, time.perf_counter())
        if dump is not None:
            dump.update(self.outputs())
        e2e_ms = D.max(e2e_ms_c)
        launches = int(ba.launch_count() - launches0)
        ba.set_timing(True)
        ba.gn_step(x, self.k8, self.precalc, self.TH)
        ba.apply_res()
        tm = ba.last_timing()
        ba.set_timing(False)
        h2d, d2h = ba.io_bytes()
        return {"ms_iter": ms_iter, "ms_kernel": ms_kernel, "e2e_ms": e2e_ms, "launches": launches, "device_ms_last_step": float(tm[0]),
                "h2d": h2d, "d2h": d2h, "value": self.nres_total / (ms_iter * 1e-3), "e2e_value": self.nres_total / (e2e_ms * 1e-3)}

    def close(self):
        self.ba.close()


def batched_roofline(B, steps, warmup, chunk, local_rank, peak):
    """B independent windows (different images / points) in ONE ba_fused_batch_kernel launch; planes of B windows = B x 34 MB > L2."""
    import dmvio_b200.capi as capi
    import dmvio_b200.hostmath as hm
    import dmvio_b200.synth as synth
    bas, xs, states, nres, balg = [], [], [], 0, 0
    for i in range(B):
        W = synth.make_window(nf=NF, npts=NPTS, w=W_, h=H_, seed=1234 + 17 * i)
        ba = capi.BA(W_, H_, max_frames=NF, max_points=len(W["host"]), device=local_rank, chunk_points=chunk)
        for k in range(NF):
            ba.upload_frame(k, W["dI"][k])
        ba.set_window(NF)
        ba.set_points(W["host"], W["u"], W["v"], W["idepth"], W["idepth_zero"], W["color"], W["weights"])
        ba.set_residuals(W["res_point"], W["res_target"])
        ba.set_adjoints(*hm.adjoints(W))
        st = (hm.calib8(W["K"]), hm.precalc_table(W), W["frameEnergyTH"].copy())
        ba.set_state(*st)
        ba.linearize(); ba.apply_res()
        a = ba.accumulate()
        HL, bL = hm.prior_system(W)
        xs.append(hm.solve_reduced(a["HA"], a["bA"], a["Hsc"], a["bsc"], HL, bL, lam=1e-5))
        ba.backup_points()
        bas.append(ba); states.append(st)
        nres += len(W["res_point"]); balg += algorithmic_bytes(len(W["res_point"]), len(W["host"]), NF)
    batch = capi.BABatch(bas)
    ms, e2e_ms, identical = batch.bench(xs, states, iters=steps, warmup=max(3, warmup))
    ach = balg / (ms * 1e-3) / 1e9
    traffic, src = ncu_traffic("*_ba_fused_batch_summary.md")
    out = {"bound": "hbm", "kernel": f"ba_fused_batch_kernel ({B} windows / launch)", "windows": B, "point_residuals": nres, "achieved": ach, "peak": peak, "unit": "GB/s",
           "frac": ach / peak, "traffic": traffic, "traffic_source": src, "algorithmic_bytes_per_launch": balg, "kernel_ms": ms,
           "value": nres / (ms * 1e-3), "e2e_value": nres / (e2e_ms * 1e-3), "e2e_ms": e2e_ms, "unit_value": UNIT,
           "l2": f"no scrub: the {B} windows' level-0 planes ({B} x 34 MB as float4) exceed the 126 MB L2",
           "results_identical_to_single_window_launches": identical}
    batch.close()
    for b in bas:
        b.close()
    return out


def config5_stream(D, rank, world, local_rank):
    """BASELINE config 5: TUM-VI-shaped 512x512 stream, 10 GN iterations per keyframe, IMU factors stubbed (host LDL^T); every rank runs an
    independent replica (the path does not shard below a window: 'replicas only'), keyframes/s add up."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import bench_stream
    r = bench_stream.run_stream(keyframes=14, its=10, cpu_keyframes=(3 if (rank == 0 and world == 1) else 0), size=512, device=local_rank)
    rates = D.gather(r["gpu_keyframes_per_s"])
    if rank != 0:
        return None
    out = {"workload": "512x512 stream, 7 KF window, 2000 pts, exactly 10 GN iterations per keyframe, one replica per GPU", "scaling": "replicas",
           "keyframes_per_s": float(sum(rates)), "keyframes_per_s_per_gpu": [float(x) for x in rates], "gpu_ms_per_keyframe": r["gpu_ms_per_keyframe"],
           "gn_iterations_per_keyframe": r["gpu_gn_iterations_per_keyframe"], "timed_gpu": r["timed_gpu"],
           "gpu_ms_setup_per_keyframe": r.get("gpu_ms_setup_per_keyframe"), "gpu_us_per_iteration": r.get("gpu_us_per_iteration")}
    if world == 1:
        out.update(cpu_keyframes_per_s=r["cpu_keyframes_per_s"], cpu_threads=r["cpu_threads"], timed_cpu=r["timed_cpu"])
    return out


def coarse_record(local_rank, peak):
    """BASELINE config 2: CoarseTracker 5-level alignment of a 640x480 pair (one cluster launch per frame) + its roofline (64 B per point and
    evaluation: SURVEY.md section 8d) + the single-threaded CPU oracle (the reference's tracker is single-threaded)."""
    import dmvio_b200.hostapi as hostapi
    import dmvio_b200.synth as synth
    from oracle import orc
    out = {}
    for levels in (5, 0):
        T = synth.make_tracking_pair(seed=4321, levels=levels)
        L = T["levels"]
        g = hostapi.CoarseTracker(T["w"], T["h"], T["K"], L, device=local_rank)
        counts = g.set_ref_device(T["Ku"], T["Kv"], T["new_idepth"], T["HdiF"], T["img_ref"])
        g.set_new_image(T["img_new"])
        R0, t0 = np.eye(3), np.zeros(3)
        for _ in range(5):
            r = g.track(R0, t0, 0.0, 0.0)
        n = 200
        tw = time.perf_counter()
        for _ in range(n):
            r = g.track(R0, t0, 0.0, 0.0)
        ms = (time.perf_counter() - tw) / n * 1e3
        tw = time.perf_counter()
        for _ in range(n):
            g.set_new_image(T["img_new"]); g.track(R0, t0, 0.0, 0.0)
        ms_frame = (time.perf_counter() - tw) / n * 1e3
        ev = r["evaluations"]
        # point-evaluations per frame: every evaluation of a level touches all its reference points
        pe = float(r.get("point_evaluations", 0)) or float(ev) * float(np.mean(counts))
        ct = orc.CoarseTracker(T["w"], T["h"], T["K"], levels)
        ct.make_coarse_depth(T["Ku"], T["Kv"], T["new_idepth"], T["HdiF"], T["pyr_ref"])
        ct.set_new_frame(T["pyr_new"])
        tw = time.perf_counter()
        for _ in range(3):
            ct.track(np.eye(3), np.zeros(3), 0.0, 0.0)
        cpu_ms = (time.perf_counter() - tw) / 3 * 1e3
        key = f"L{L}"
        out[key] = {"levels": L, "ref_points_per_level": [int(c) for c in counts], "track_only_ms": ms, "frame_ms_incl_h2d_and_pyramid": ms_frame, "evaluations": int(ev),
                    "us_per_evaluation": ms * 1e3 / max(1, ev), "cpu_oracle_track_ms_1_thread": cpu_ms, "speedup_track_only": cpu_ms / ms,
                    "roofline": {"bound": "hbm", "kernel": "ct_track_cluster_kernel", "algorithmic_bytes": 64.0 * pe, "achieved": 64.0 * pe / (ms * 1e-3) / 1e9, "peak": peak,
                                 "unit": "GB/s", "frac": 64.0 * pe / (ms * 1e-3) / 1e9 / peak,
                                 "note": "a sequential LM chain of ~%d dependent evaluations of <= 10 k points each: latency-bound by construction (DESIGN.md section 5)" % ev}}
        g.close()
    return out


DUMP_BYTES = 64 << 20


def dump_outputs(d, arrays):
    """writes each array as d/<name>.npy (float32 / float64).  Above DUMP_BYTES in all, every array is cut to the same fixed, seeded
    sample of rows (its first axis), and the sampled row indices are written beside it as <name>_rows.npy (float64 indices take at most
    twice the bytes of the rows they index, hence a third of the budget for the rows themselves)."""
    os.makedirs(d, exist_ok=True)
    total = sum(a.nbytes for a in arrays.values())
    for name, a in sorted(arrays.items()):
        if total > DUMP_BYTES and a.ndim > 0 and a.shape[0] > 1:
            k = max(1, int(a.shape[0] * DUMP_BYTES / (3 * total)))
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], k, replace=False))
            a = a[rows]
            np.save(os.path.join(d, f"{name}_rows.npy"), rows.astype(np.float64))
        np.save(os.path.join(d, f"{name}.npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--chunk", type=int, default=0, help="points per thread block (16/32, 0 = library default)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--points", type=int, default=0,
                    help="points per GPU of the headline line; default 2000 = BASELINE.json configs[1].  Other values relabel the metric")
    ap.add_argument("--batch", type=int, default=8, help="windows per launch of the batched roofline record (N = 1 only); 0 = skip")
    ap.add_argument("--no-extras", action="store_true", help="skip the strong-scaling / config-4 / batched side records")
    ap.add_argument("--ref-courtesy", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of the headline window returned to its caller as DIR/<name>.npy (rank 0)")
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "nccl"],
                    help="N>1: all-reduce of the system inside the kernel over NVLink peer memory (CUDA IPC) or by NCCL behind it")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    args.steps = max(1, args.steps)
    global NPTS, METRIC
    if args.points > 0:
        NPTS = args.points
        METRIC = METRIC.replace("2000 pts", f"{NPTS} pts")
    if args.ref_courtesy:
        run_ref_courtesy(args.points or NPTS)
        return
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    D = Dist(world, local_rank)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    peak, peak_src = measured_peak()

    # ---------------- headline: weak scaling, NPTS points per rank
    C = Case(D, rank, world, local_rank, NPTS * world, args.chunk, args.exchange)
    parity = C.parity()
    dump = {} if args.dump_outputs and rank == 0 else None
    m = C.measure(args.steps, args.warmup, sampler, dump)
    if dump is not None:
        dump_outputs(args.dump_outputs, dump)
    balg = algorithmic_bytes(C.nres_local, len(C.Wr["host"]), NF)
    exchange, r0, nres_total, nres_local = C.exchange, C.r0, C.nres_total, C.nres_local
    Wfull = C.Wfull
    C.close()

    extras = {}
    if not args.no_extras:
        side_steps = max(50, min(args.steps, 300))
        if world > 1:
            for name, total in (("strong", NPTS), ("config4", 8000)):
                Cx = Case(D, rank, world, local_rank, total, args.chunk, args.exchange)
                px = Cx.parity()
                mx = Cx.measure(side_steps, min(args.warmup, 10))
                if rank == 0:
                    extras[name] = {"workload": f"{NF} KF / {total} pts in total ({total // world} per GPU) / {W_}x{H_}, {Cx.nres_total} point-residuals", "scaling": "strong",
                                    "value": mx["value"], "ms_per_step": mx["ms_iter"], "e2e_value": mx["e2e_value"], "e2e_ms_per_step": mx["e2e_ms"], "unit": UNIT,
                                    "steps": side_steps, "parity": px,
                                    "roofline_frac": algorithmic_bytes(Cx.nres_local, len(Cx.Wr["host"]), NF) / (mx["ms_kernel"] * 1e-3) / 1e9 / peak}
                Cx.close()
        else:
            Cx = Case(D, rank, world, local_rank, 8000, args.chunk, args.exchange)
            px = Cx.parity()
            mx = Cx.measure(side_steps, min(args.warmup, 10))
            extras["config4_one_gpu"] = {"workload": f"{NF} KF / 8000 pts / {W_}x{H_} on ONE GPU, {Cx.nres_total} point-residuals", "value": mx["value"],
                                         "ms_per_step": mx["ms_iter"], "e2e_value": mx["e2e_value"], "unit": UNIT, "steps": side_steps, "parity": px,
                                         "roofline_frac": algorithmic_bytes(Cx.nres_local, 8000, NF) / (mx["ms_kernel"] * 1e-3) / 1e9 / peak}
            Cx.close()
            try:
                extras["config2_coarse"] = coarse_record(local_rank, peak)
            except Exception as e:
                extras["config2_coarse"] = {"error": str(e)[:300]}
            if args.batch > 0:
                try:
                    tw0 = time.perf_counter()
                    extras["roofline_batched"] = batched_roofline(args.batch, side_steps, min(args.warmup, 10), args.chunk, local_rank, peak)
                    sampler.mark(tw0, time.perf_counter())
                except Exception as e:
                    extras["roofline_batched"] = {"error": str(e)[:300]}

    if not args.no_extras:
        try:
            c5 = config5_stream(D, rank, world, local_rank)
        except Exception as e:
            c5 = {"error": str(e)[:300]}
            D.gather(0.0) if world > 1 and "gather" not in str(e) else None
        if rank == 0:
            extras["config5_stream"] = c5
    clocks = sampler.stop() if rank == 0 else None
    traffic, traffic_src = ncu_traffic()
    ach = balg / (m["ms_kernel"] * 1e-3) / 1e9

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads, rates = pick_threads(Wfull)
        r = cpu_rate(Wfull, args.cpu_seconds, threads)
        cpu = {"value": r["rate"], "unit": UNIT, "cores": threads, "kind": "port", "ms_per_iter": r["ms_per_iter"],
               "value_min_block": r["rate_min"], "value_max_block": r["rate_max"], "value_at_reference_NUM_THREADS_6": rates.get(6),
               "sample": f"{r['iters']} full GN iterations of the same window in ~{args.cpu_seconds:.0f} s (5 blocks, median), oracle (g++ -O3, no -march), "
                         f"{threads} worker threads pinned to {r['pinned_cpus']} CPUs (best of {sorted(rates)}; the reference hard-codes NUM_THREADS=6); host has {os.cpu_count()} logical cores"}

    if rank == 0:
        xdesc = {"p2p": ", all-reduce of H,b per step inside ba_fused_kernel (LL packets over NVLink peer memory, CUDA IPC)", "nccl": ", NCCL all-reduce of H,b per step", "none": ""}[exchange]
        out = {
            "metric": METRIC, "value": m["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": m["ms_iter"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"sliding window {NF} KF / {NPTS * world} pts / {W_}x{H_}, pattern 8, {nres_total} point-residuals "
                                   f"({nres_local}/GPU), one GN iteration of the hot path per step (host solve excluded)",
                       "parallelism": f"points sharded over {world} GPU(s), images replicated" + xdesc,
                       "l2": "L2 scrubbed (256 MiB write) between timed steps of `value`", "chunk_points": args.chunk or 16,
                       "n_in": r0["n_in"], "n_oob": r0["n_oob"], "n_outlier": r0["n_outlier"]},
            "e2e": {"value": m["e2e_value"], "unit": UNIT, "ms_per_step": m["e2e_ms"], "h2d_bytes_per_step": m["h2d"], "d2h_bytes_per_step": m["d2h"],
                    "device_ms_last_step": m["device_ms_last_step"],
                    "timed": "steps x {dmv_ba_gn_step(host x, host tables) ; dmv_ba_apply_res()} issued from C, wall clock, incl. host<->device traffic + sync"},
            "gpu_launches": m["launches"],
            "parity": parity,
            "roofline": {"bound": "hbm", "kernel": "ba_fused_kernel (the whole GN linearisation: one cooperative launch)", "achieved": ach, "peak": peak, "unit": "GB/s",
                         "frac": ach / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": balg, "kernel_ms": m["ms_kernel"],
                         "note": "one 7-KF window is a latency-bound dependent chain (launch, gather round trip, reductions, grid barrier) on an L2-sized "
                                 "working set: see roofline_batched for the bandwidth regime (DESIGN.md section 6)"},
            "clocks": clocks,
        }
        out.update(extras)
        if cpu:
            out["cpu_baseline"] = cpu
        print(json.dumps(out))
        if parity is not None and not parity["ok"]:
            sys.stderr.write(f"PARITY FAILURE vs the unsharded oracle: {parity}\n")
            D.close()
            sys.exit(3)
    D.close()


if __name__ == "__main__":
    main()
