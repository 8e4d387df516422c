#!/usr/bin/env python
"""bench.py - headline measurement of the B200 hot path (contract: see DESIGN.md "Measurement").

Workload (BASELINE.json configs[1]): Kajita2003 preview control, 4096 random straight/circle footstep walks turned into
5 ms ZMP references by ZMPDiscretization (the product's kernel in the CUDA arm, the oracle's restatement in the reference
arm; both pinned to the TestKajita2003 datrefs), 320-tap preview window.  A "step" of the bench is --passes-per-step passes (default
160, so that 20 steps time >= 1 s) of the hot path over the whole batch (every preview step of every walk); the metric unit is
one preview step = one OneIterationOfPreview call for both axes (PreviewControl.cpp:324-374).

  python bench.py [--gpus N] [--steps K] [--warmup W]            the CUDA path through the C ABI
                  [--dump-outputs DIR]                           + the last timed pass's outputs as DIR/*.npy
  python bench.py --impl reference [...]                         the reference's CPU path on the host cores: its own
                                                                 PreviewControl object code (oracle/_ref), one process per core

With N > 1 (torchrun) every rank runs the same 4096-walk batch shape on its own GPU with its own seed
(instances are independent: weak scaling, no data-path collective); value = all steps of all ranks / max time.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "Kajita preview steps/s (batched; Herdt2010 QP solves/s reported under 'herdt')"
UNIT = "preview steps/s"
WORKLOAD = "kajita2003_preview_batched_4096_footstep_walks_zmpdiscretization_320tap"
FLOP_PER_STEP = 1360.0          # SURVEY 8d: both axes, 2*(2*320 + 40)
FIR_FLOP_PER_STEP = 1280.0      # the 2x320-tap window MACs, the part the FIR kernel executes
BYTES_PER_STEP = 80.0           # streaming minimum: 16 B in, 48 B CoM + 16 B ZMP out


class ClockSampler:
    """Samples SM clock / throttle reasons with nvidia-smi while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for (t, line) in self.rows:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                clk, mx = float(f[0]), float(f[1])
            except ValueError:
                continue
            smax = mx
            if t0 - 0.05 <= t <= t1 + 0.05:
                sm.append(clk)
                for nme, v in zip(names, f[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
        if not sm:  # region shorter than the sampling period: use the nearest samples
            sm = [float(r[1].split(",")[0]) for r in self.rows[-3:] if r[1].split(",")[0].strip().replace(".", "").isdigit()]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


def reduce_over_ranks(dist, times, units, device="cuda"):
    """Multi-GPU reduction of the measurements (the data path itself has no collective): element-wise MAX of the times,
    SUM of the unit counts.  dist = torch.distributed (nccl on the GPUs, gloo in the CPU tests) or None."""
    if dist is None:
        return list(times), list(units)
    import torch
    t = torch.tensor(list(times), dtype=torch.float64, device=device)
    u = torch.tensor(list(units), dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dist.all_reduce(u, op=dist.ReduceOp.SUM)
    return [float(v) for v in t], [float(v) for v in u]


def ncu_traffic(kernel, walks):
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        e = t[kernel]
        if int(e.get("walks", walks)) != int(walks):
            return {"traffic": None}
        return {"traffic": float(e["dram_bytes_per_launch"]), "traffic_unit": "bytes per launch", "traffic_source": e["source"]}
    except (OSError, KeyError, ValueError):
        return {"traffic": None}


def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_preview_rate(offsets, z, seconds=10.0):
    """cpu_baseline of the main line: the reference arm (below) timed on a bounded sample - whole passes over the first
    walks of the batch, grown until one pass takes a few seconds."""
    B = len(offsets) - 1
    cores = host_cores()
    nb = min(B, max(cores * 4, 64))
    while True:
        arm = ReferencePreviewArm(offsets[:nb + 1], z[:int(offsets[nb])])
        arm.one_pass()                                     # warm-up: workers start, pin, build their PreviewControl
        steps, dt = arm.one_pass()
        arm.close()
        if dt >= seconds / 3 or nb >= B:
            break
        nb = min(B, int(nb * max(2.0, (seconds / 2) / max(dt, 1e-3))))
    return {"value": steps / dt, "unit": UNIT, "cores": arm.procs, "kind": arm.kind,
            "sample": f"first {nb} of {B} walks ({steps} preview steps in {dt:.2f} s); " + arm.describe(nb, steps)}


# ---- reference arm: the reference's OWN PreviewControl object code, one process per core ----------------
_REF_JOB = {}


def _ref_worker(i):
    """Worker i of P (forked: offsets / z are inherited copy-on-write): pins itself to one core on first use, builds its
    own PreviewControl object of the reference (oracle/_ref) and runs OneIterationOfPreview over walks i, i+P, ...
    exactly as the reference's caller does (one call at lindex 0 per tick, then pop_front)."""
    import preview_ref as pr
    J = _REF_JOB
    if "rp" not in J:
        try:
            cpus = sorted(os.sched_getaffinity(0))
            os.sched_setaffinity(0, {cpus[i % len(cpus)]})
        except (AttributeError, OSError):
            pass
        rp = pr.RefPreview(1, False)
        if J["own_gains"] and pr.lapack_available():
            rp.compute_weights(0.005, 1.6, 0.814, 1)          # the reference's own dgges_ Riccati solve
        else:
            g = J["gains"]
            rp.set_gains(0.005, 1.6, 0.814, g.Kx, g.Ks, g.F)
        J["rp"] = rp
        n = int(J["offsets"][-1])
        J["com"] = np.zeros((n, 6)); J["zmp"] = np.zeros((n, 2))   # only this worker's rows are ever touched
    B = len(J["offsets"]) - 1
    st = np.zeros((B, 8))
    t = time.perf_counter()
    steps = J["rp"].run_batch(J["offsets"], J["z"], st, J["com"], J["zmp"], b0=i, b1=B, stride=J["P"])
    return int(steps), time.perf_counter() - t


class ReferencePreviewArm:
    """bench.py --impl reference and the cpu_baseline leg: PreviewControl::OneIterationOfPreview of the reference
    (its own source compiled into oracle/_ref; falls back to the oracle port when that library is absent), one walking
    problem per call chain, one PROCESS per host core (BASELINE.md: one instance per core)."""

    def __init__(self, offsets, z, procs=None):
        import multiprocessing as mp
        import oracle_lib as ol
        import preview_ref as pr
        self.procs = procs or host_cores()
        self.kind = "reference" if pr.lib() is not None else "port"
        self.offsets, self.z = offsets, z
        self.gains = ol.OracleGains(0.005, 1.6, 0.814, 1)
        self.own_gains = False
        if self.kind == "reference":
            self.own_gains = pr.lapack_available()
            _REF_JOB.clear()
            _REF_JOB.update(offsets=offsets, z=z, P=self.procs, gains=self.gains, own_gains=self.own_gains)
            self.pool = mp.get_context("fork").Pool(self.procs)
        else:
            self.pool = None

    def one_pass(self):
        """-> (preview steps, wall seconds) of one pass over every walk."""
        t = time.perf_counter()
        if self.pool is not None:
            res = self.pool.map(_ref_worker, range(self.procs), chunksize=1)
            steps = sum(r[0] for r in res)
        else:
            import oracle_lib as ol
            st = np.zeros((len(self.offsets) - 1, 8))
            _, _, steps = ol.oracle_preview_batch(self.gains, self.offsets, self.z, st, threads=self.procs, want_out=False)
        return steps, time.perf_counter() - t

    def describe(self, walks, steps):
        what = ("the reference's own PreviewControl.cpp object code (oracle/_ref), std::deque<ZMPPosition> popped per tick"
                if self.kind == "reference" else "oracle port of PreviewControl::OneIterationOfPreview over std::deque<ZMPPosition>")
        gains = "gains from the reference's own dgges_ Riccati solve" if self.own_gains else "gains from the oracle's Riccati fixed point"
        return f"each step = all {walks} walks ({steps} preview steps), one process per core pinned with sched_setaffinity; {what}; {gains}"

    def close(self):
        if self.pool is not None:
            self.pool.terminate()
            self.pool.join()


def herdt_cpu_inputs(n_sims=48, periods=30, seed=7):
    """Closed-loop QP inputs for the CPU Herdt leg of the reference arm, generated on the CPU by the oracle's
    TestHerdt2010 harness (no GPU on this path): n_sims walks under random velocity references (the distribution of
    BASELINE configs[2]), `periods` QP periods each."""
    import herdt_oracle as ho
    rng = np.random.default_rng(seed)
    ins = []
    for k in range(n_sims):
        sim = ho.Sim(textbook=True, logging=True)
        sim.steps_before_stop(2)
        sim.vel_ref(float(rng.uniform(-0.2, 0.3)), float(rng.uniform(-0.15, 0.15)), float(rng.uniform(-0.2, 0.2)))
        for _ in range(20 * periods):
            sim.tick()
        ins.append(sim.log()[0].copy())
        sim.close()
    return np.concatenate(ins)


def _oracle_discretize_worker(job):
    import zmpdisc_oracle as zo
    zp = zo.default_params()
    out = []
    for st, f in job:
        o = zo.run(zp, st.astype(zo.REL_STEP_DTYPE), f)
        out.append(np.ascontiguousarray(o["zmp"][:, :2]))
    return out


def headline_workload_cpu(walks, seed):
    """configs[1] for the reference arm (no GPU there): the footstep walks of workloads.kajita_steps_batch through the ORACLE's
    ZMPDiscretization (pinned to the four TestKajita2003 datrefs), one process per core -> (offsets, zmpref [total][2])."""
    import multiprocessing as mp
    from jrl_walkgen_b200 import workloads
    off, steps, feet = workloads.kajita_steps_batch(walks, seed=seed)
    procs = host_cores()
    jobs = [[] for _ in range(procs)]
    for b in range(walks):
        jobs[b % procs].append((steps[off[b]:off[b + 1]].copy(), feet[b].copy()))
    with mp.get_context("fork").Pool(procs) as pool:
        res = pool.map(_oracle_discretize_worker, jobs)
    zs = [None] * walks
    for p, r in enumerate(res):
        for k, z in enumerate(r):
            zs[p + k * procs] = z
    lens = np.array([len(z) for z in zs], dtype=np.int64)
    return np.concatenate([[0], np.cumsum(lens)]).astype(np.int64), np.ascontiguousarray(np.concatenate(zs))


def headline_workload_gpu(ctx, walks, seed):
    """configs[1] for the CUDA arm: the same footstep walks through the product's own ZMPDiscretization kernel
    (wg_zmpdisc_run_batch), downloaded once - the ZMP references the preview kernel is then timed on."""
    from jrl_walkgen_b200 import workloads
    off, steps, feet = workloads.kajita_steps_batch(walks, seed=seed)
    kp = ctx.kajita_plan(off, steps, feet)
    offsets = np.ascontiguousarray(kp.sample_offsets, dtype=np.int64).copy()
    z = np.zeros((int(offsets[-1]), 2))
    kp.discretize(zmpref_xy=z)
    kp.destroy()
    return offsets, z


def run_reference(args):
    rank, _, world = dist_env()
    if rank != 0:
        return
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "liboracle.so"], check=True)
    offsets, z = headline_workload_cpu(args.walks, seed=0)
    arm = ReferencePreviewArm(offsets, z)
    ms, steps = [], 0
    for it in range(args.warmup + args.steps):
        steps, dt = arm.one_pass()
        if it >= args.warmup:
            ms.append(dt * 1e3)
    arm.close()
    value = float(steps * len(ms) / (sum(ms) * 1e-3))
    sample = arm.describe(args.walks, steps)
    herdt = None
    if not args.no_herdt:
        qin = herdt_cpu_inputs()
        herdt = cpu_herdt_rate(qin, seconds=max(2.0, args.cpu_seconds / 2))
        herdt["workload"] = HERDT_WORKLOAD
        herdt["inputs"] = f"{len(qin)} closed-loop QPs of 48 oracle walks under random velocity references (CPU-generated)"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(np.mean(ms)), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "walks_per_gpu": args.walks, "NL": 320, "T": 0.005,
                       "preview_steps_per_pass_per_gpu": int(steps)},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": arm.procs, "kind": arm.kind, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "herdt": herdt, "herdt_qp_solves_per_s": None if herdt is None else herdt["value"],
            "gpu_launches": 0}
    emit_line(line)


# ------------------------------------------------------------------------------------------------
# Herdt2010 leg (BASELINE configs[2]: 16 384 random velocity references on one B200)
# ------------------------------------------------------------------------------------------------
HERDT_WORKLOAD = "herdt2010_qp_16384_random_velocity_refs_N16"


def herdt_flop_model(n, m, iters):
    """SURVEY 8d: flops of the reference algorithm for one solve (assembly + Cholesky + active-set iterations)."""
    return 1.2e4 + (2.0 / 3.0) * n ** 3 + iters * (2.0 * m * n + 6.0 * n * n)


def _cpu_qld_worker(args):
    import ctypes as C
    import herdt_oracle as ho
    ins_bytes, n, seconds = args
    ins = np.frombuffer(ins_bytes, dtype=ho.QP_INPUT_DTYPE)
    p = ho.default_params()
    out = np.zeros(n, dtype=ho.QP_OUTPUT_DTYPE)
    done = 0
    t0 = time.perf_counter()
    while True:
        ho.lib().oracle_herdt_solve_qp_batch(C.byref(p), n, ins.ctypes.data, out.ctypes.data, 0)
        done += n
        if time.perf_counter() - t0 >= seconds:
            break
    return done, time.perf_counter() - t0, int((out["fail"] != 0).sum())


def cpu_herdt_rate(qin, seconds=5.0, procs=None):
    """The reference's own QLD (oracle/_ref object code) + the oracle's restated assembly, one PROCESS per core
    (QLD keeps its locals static, qld.cpp:403-412: threads are unsafe), each on its own slice of the inputs."""
    import multiprocessing as mp
    import herdt_oracle as ho
    procs = procs or host_cores()
    kind = "reference" if ho.lib().oracle_herdt_have_ref_qld() == 1 else "port"
    per = max(64, min(512, len(qin) // procs))
    jobs = [(qin[(i * per) % max(1, len(qin) - per):][:per].tobytes(), per, seconds) for i in range(procs)]
    with mp.get_context("fork").Pool(procs) as pool:
        res = pool.map(_cpu_qld_worker, jobs)
    total = sum(r[0] for r in res)
    wall = max(r[1] for r in res)
    return {"value": total / wall, "unit": "QP solves/s", "cores": procs, "kind": kind,
            "sample": f"{procs} processes x {per} captured closed-loop QPs repeated for {seconds:.0f} s "
                      f"({total} solves): oracle assembly (generator-vel-ref.cpp restated) + "
                      + ("the reference's own ql0001_ object code" if kind == "reference" else "textbook solver"),
            "us_per_solve_per_core": 1e6 * wall * procs / total, "failures": sum(r[2] for r in res)}


def herdt_leg(ctx, wg, args, rank, fp64_peak, want_cpu):
    import ctypes as C
    B = args.herdt_instances
    rng = np.random.default_rng([7, rank])
    v = np.column_stack([rng.uniform(-0.2, 0.3, B), rng.uniform(-0.15, 0.15, B), rng.uniform(-0.2, 0.2, B)])
    ctx.herdt_set_params()
    ctx.herdt_mpc_set_params()
    d_st = ctx.herdt_mpc_init(B, device=True)
    d_v = ctx.to_device(v)
    d_qin = ctx.alloc(B * wg.QP_INPUT_DTYPE.itemsize)
    d_out = ctx.alloc(B * wg.QP_OUTPUT_DTYPE.itemsize)
    d_flush = ctx.alloc(256 << 20)
    lib, h = ctx.lib, ctx.h
    ST, QI = wg.MPC_STATE_DTYPE.itemsize, wg.QP_INPUT_DTYPE.itemsize

    def mpc(off, n, periods, qin=False):
        ctx._check(lib.wg_herdt_mpc_run_batch(h, wg.WG_MEM_DEVICE, n, periods, C.c_void_p(d_st.ptr + off * ST),
                                              C.c_void_p(d_v.ptr + off * 24), None, None,
                                              C.c_void_p(d_qin.ptr + off * QI) if qin else None))

    # warm-up rollout: 16 slices advanced by 40..55 periods so that the batch covers every phase of the step cycle
    sl = (B + 15) // 16
    for j in range(16):
        a = j * sl
        n = min(sl, B - a)
        if n > 0:
            mpc(a, n, 40 + j)
    ctx.sync()
    # ---- closed loop: K launches of `periods` QP periods over the whole batch
    periods = args.herdt_periods
    for _ in range(2):
        mpc(0, B, periods)
    ctx.sync()
    # CUDA events on the context stream around the K launches (a period is three kernels by default: FSM + assemble,
    # herdt_qp_kernel, interpolate + state update; WG_HERDT_MPC_SPLIT=0 selects the fused single kernel)
    ctx.timer_start()
    for _ in range(args.steps):
        mpc(0, B, periods)
    mpc_ms = ctx.timer_stop_ms() / args.steps
    mpc_rate = B * periods / (mpc_ms * 1e-3)
    # ---- open loop on the captured QP inputs of the last period (device resident, L2 flushed between launches)
    mpc(0, B, 1, qin=True)
    ctx.sync()
    for _ in range(3):
        ctx.herdt_qp_solve(d_qin, d_out, mem=wg.WG_MEM_DEVICE, count=B)
    ctx.sync()
    ctx.prof_begin(2 * args.steps + 8)
    for _ in range(args.steps):
        ctx._check(lib.wg_memset_device(h, d_flush.ptr, 0, 256 << 20))
        ctx.herdt_qp_solve(d_qin, d_out, mem=wg.WG_MEM_DEVICE, count=B)
    prof = ctx.prof_end()
    qp_ms = prof[2][1] / prof[2][0]
    qp_rate = B / (qp_ms * 1e-3)
    out = d_out.download(wg.QP_OUTPUT_DTYPE, (B,))
    qin = d_qin.download(wg.QP_INPUT_DTYPE, (B,))
    st = d_st.download(wg.MPC_STATE_DTYPE, (B,))
    iters = out["iterations"].astype(np.float64)
    flops = float(np.sum(herdt_flop_model(out["n_vars"].astype(np.float64), out["n_rows"].astype(np.float64), iters)))
    ach = flops / (qp_ms * 1e-3) / 1e12
    # ---- end to end: host records in, host records out through the C ABI
    pin_in = ctx.pinned((B,), wg.QP_INPUT_DTYPE); pin_in[:] = qin
    pin_out = ctx.pinned((B,), wg.QP_OUTPUT_DTYPE)
    for _ in range(2):
        ctx.herdt_qp_solve(pin_in, pin_out)
    n_e2e = max(3, min(args.steps, 10))
    te = time.perf_counter()
    for _ in range(n_e2e):
        ctx.herdt_qp_solve(pin_in, pin_out)
    e2e_s = time.perf_counter() - te
    res = {"workload": HERDT_WORKLOAD, "instances": B,
           "qp_solves_per_s": qp_rate, "qp_ms_per_launch": qp_ms,
           "closed_loop_qp_solves_per_s": mpc_rate, "closed_loop_ms_per_launch": mpc_ms,
           "closed_loop_periods_per_launch": periods,
           "iterations_mean": float(iters.mean()), "iterations_max": int(iters.max()),
           "n_prw_steps_hist": [int((qin["sup_step"][:, 16] == k).sum()) for k in range(3)],
           "failures": int((out["fail"] != 0).sum()), "closed_loop_failures": int(st["fail_count"].sum()),
           "roofline": {"kernel": "herdt_qp_kernel", "bound": "fp64", "achieved": ach, "peak": fp64_peak,
                        "unit": "TFLOP/s", "frac": ach / fp64_peak, "traffic": None,
                        "algorithmic_flop_per_solve_mean": flops / B,
                        "note": "flop model of the reference algorithm (SURVEY 8d) with the measured active-set "
                                "iteration counts; the kernel is latency/divergence bound, not pipe bound"},
           "e2e": {"value": B * n_e2e / e2e_s, "unit": "QP solves/s", "h2d_bytes_per_step": int(qin.nbytes),
                   "d2h_bytes_per_step": int(out.nbytes), "api": "wg_herdt_qp_solve_batch(WG_MEM_HOST), pinned host records"}}
    if want_cpu:
        res["cpu_baseline"] = cpu_herdt_rate(qin, seconds=max(2.0, args.cpu_seconds / 2))
    for b in (d_st, d_v, d_qin, d_out, d_flush):
        b.free()
    return res, {"herdt_qp_kernel": {"launches": args.steps, "avg_ms": qp_ms},
                 "herdt_mpc (pre + herdt_qp_kernel + post per period)": {"launches": args.steps, "avg_ms": mpc_ms}}


# ------------------------------------------------------------------------------------------------
# Kajita front end + preview (SURVEY 8f rank 1): footsteps -> 5 ms ZMP reference + feet -> CoM without leaving the GPU
# ------------------------------------------------------------------------------------------------
def kajita_leg(ctx, wg, args, rank, hbm_peak):
    from jrl_walkgen_b200 import workloads
    B = args.walks
    off, steps, feet = workloads.kajita_steps_batch(B, seed=1000 * rank)
    plan = ctx.kajita_plan(off, steps, feet)
    n, nsteps = plan.total_samples, plan.total_steps
    dst = ctx.to_device(np.zeros((B, 8)))
    dcom = ctx.alloc(n * 48); dzmp = ctx.alloc(n * 16); dref = ctx.alloc(n * 16)
    dl = ctx.alloc(n * 48); dr = ctx.alloc(n * 48)
    for _ in range(3):
        plan.run(dst, dcom, dzmp, dref, dl, dr, True, mem=wg.WG_MEM_DEVICE)
    ctx.sync()
    ctx.prof_begin(4 * args.steps + 8)
    ctx.timer_start()
    for _ in range(args.steps):
        plan.set_steps(steps, feet)                       # a new batch of footstep plans: the H2D copy of a real caller
        plan.run(dst, dcom, dzmp, dref, dl, dr, True, mem=wg.WG_MEM_DEVICE)
    ms = ctx.timer_stop_ms() / args.steps
    prof = ctx.prof_end()
    zd_ms = prof[7][1] / prof[7][0] if 7 in prof else None
    # end to end: host step lists in, host CoM/ZMP/ZMP-reference/feet out
    com = ctx.pinned((n, 6)); zmp = ctx.pinned((n, 2)); ref = ctx.pinned((n, 2))
    st = ctx.pinned((B, 8))
    n_e2e = max(2, min(args.steps, 4))
    st[:] = 0.0
    plan.run(st, com, zmp, ref, None, None, True, mem=wg.WG_MEM_HOST)
    te = time.perf_counter()
    for _ in range(n_e2e):
        st[:] = 0.0
        plan.set_steps(steps, feet)
        plan.run(st, com, zmp, ref, None, None, True, mem=wg.WG_MEM_HOST)
    ctx.sync()
    e2e_s = time.perf_counter() - te
    res = {"workload": "kajita2003_footsteps_to_com_%d_walks" % B, "walks": B, "footsteps": int(len(steps)),
           "samples": int(n), "preview_steps": int(nsteps), "ms_per_pass": ms,
           "preview_steps_per_s": nsteps / (ms * 1e-3),
           "zmpdisc_ms_per_launch": zd_ms,
           # the front-end kernel is store bound: ZMP reference (16 B) + two feet (2 x 48 B) per 5 ms sample
           "zmpdisc_roofline": None if zd_ms is None else {
               "kernel": "zmpdisc_kernel", "bound": "hbm", "achieved": 112.0 * n / (zd_ms * 1e-3) / 1e9, "peak": hbm_peak,
               "unit": "GB/s", "frac": 112.0 * n / (zd_ms * 1e-3) / 1e9 / hbm_peak, "traffic": None,
               "algorithmic_bytes_per_sample": 112.0},
           "e2e": {"value": nsteps * n_e2e / e2e_s, "unit": "preview steps/s", "h2d_bytes_per_step": int(steps.nbytes + feet.nbytes + st.nbytes),
                   "d2h_bytes_per_step": int(com.nbytes + zmp.nbytes + ref.nbytes + st.nbytes),
                   "api": "wg_kajita_plan_set_steps + wg_kajita_run_batch(WG_MEM_HOST): step lists in, CoM/ZMP/ZMP reference out"}}
    for b in (dst, dcom, dzmp, dref, dl, dr):
        b.free()
    plan.destroy()
    return res, ({"zmpdisc_kernel": {"launches": int(prof[7][0]), "avg_ms": zd_ms}} if zd_ms is not None else {})


# ------------------------------------------------------------------------------------------------
# Mixed sweep (BASELINE configs[4]): 10^6 Herdt2010 MPC instances x 100 control periods, instance i -> rank i mod G
# ------------------------------------------------------------------------------------------------
SWEEP_WORKLOAD = "herdt2010_mpc_sweep_1M_instances_x_100_periods"


def sweep_leg(ctx, wg, args, rank, world, dist):
    """Strong scaling: the 10^6 instances are dealt round-robin to the ranks (SURVEY 8e); every rank advances its share
    by 100 QP periods (10 s of walking: start from rest in double support, constant random velocity reference per
    instance, seed = instance index order) without leaving the device.  No data-path collective; the times are reduced
    with one MAX all-reduce."""
    import ctypes as C
    total, periods, chunk = args.sweep_instances, args.sweep_periods, 10
    mine = np.arange(rank, total, world)
    B = len(mine)
    rng = np.random.default_rng(2010)
    v_all = np.column_stack([rng.uniform(-0.2, 0.3, total), rng.uniform(-0.15, 0.15, total), rng.uniform(-0.2, 0.2, total)])
    v = np.ascontiguousarray(v_all[mine])
    ctx.herdt_set_params()
    ctx.herdt_mpc_set_params()
    d_st = ctx.herdt_mpc_init(B, device=True)
    d_v = ctx.to_device(v)
    lib, h = ctx.lib, ctx.h
    # warm the kernel on a throw-away copy of a small slice
    d_w = ctx.herdt_mpc_init(min(B, 4096), device=True)
    ctx._check(lib.wg_herdt_mpc_run_batch(h, wg.WG_MEM_DEVICE, min(B, 4096), 2, C.c_void_p(d_w.ptr), C.c_void_p(d_v.ptr),
                                          None, None, None))
    ctx.sync(); d_w.free()
    if dist is not None:
        dist.barrier()
    ctx.reset_launches()
    ctx.timer_start()
    done = 0
    while done < periods:
        n = min(chunk, periods - done)
        ctx._check(lib.wg_herdt_mpc_run_batch(h, wg.WG_MEM_DEVICE, B, n, C.c_void_p(d_st.ptr),
                                              C.c_void_p(d_v.ptr) if done == 0 else None, None, None, None))
        done += n
    ms = ctx.timer_stop_ms()
    launches = ctx.launches
    st = d_st.download(wg.MPC_STATE_DTYPE, (B,))
    fails = int(st["fail_count"].sum()); solves = int(st["qp_count"].sum())
    d_st.free(); d_v.free()
    (ms_max,), (solves_all, fails_all) = reduce_over_ranks(dist, [ms], [float(solves), float(fails)])
    return {"workload": SWEEP_WORKLOAD, "instances_total": total, "instances_per_rank": B, "periods": periods,
            "n_gpus": world, "scaling": "strong", "sharding": "instance i -> rank i mod G, no collective on the data path",
            "seconds": ms_max * 1e-3, "qp_solves": int(solves_all), "qp_solves_per_s": solves_all / (ms_max * 1e-3),
            "failures": int(fails_all), "launches_per_rank": int(launches),
            "state_bytes_per_rank": int(B * wg.MPC_STATE_DTYPE.itemsize)}


def pin_to_gpu_numa_node(index):
    """Best effort: restrict this rank to the CPUs of its GPU's NUMA node BEFORE any pinned buffer is allocated (first touch
    then places the staging buffers next to the GPU's PCIe root).  Returns what happened, for the bench line."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(index)],
                             capture_output=True, text=True, timeout=10).stdout.strip().lower()
        bus = out[-12:] if len(out) >= 12 else out            # 0000:1b:00.0
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        if node < 0:
            return {"gpu_numa_node": node, "pinned": False, "why": "the platform reports no NUMA node for the GPU"}
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0)
        use = cpus & allowed
        if not use:
            return {"gpu_numa_node": node, "pinned": False, "allowed_cpus": len(allowed),
                    "why": "none of the node's CPUs is in this process's cpuset"}
        os.sched_setaffinity(0, use)
        return {"gpu_numa_node": node, "pinned": True, "cpus": len(use)}
    except Exception as e:                                        # noqa: BLE001
        return {"pinned": False, "why": str(e)[:120]}


def library_multi_leg(wg, args, world):
    """configs[4] through wg_multi_herdt_mpc_sweep on devices 0 .. world-1 from ONE process."""
    total, periods = args.sweep_instances, args.sweep_periods
    rng = np.random.default_rng(2010)
    v_all = np.column_stack([rng.uniform(-0.2, 0.3, total), rng.uniform(-0.15, 0.15, total), rng.uniform(-0.2, 0.2, total)])
    m = wg.MultiContext((1 << world) - 1)
    try:
        m.herdt_set_params()
        m.herdt_mpc_sweep(v_all[:4096 * world], 2)                        # warm-up
        r = m.herdt_mpc_sweep(v_all, periods, chunk=10)
    finally:
        m.close()
    return {"api": "wg_multi_create + wg_multi_herdt_mpc_sweep (one process, one host thread per device)",
            "devices": r["devices"], "seconds": r["seconds"], "qp_solves": int(r["qp_solves"]),
            "qp_solves_per_s": r["qp_solves"] / r["seconds"], "failures": int(r["failures"]),
            "reduced_by_nccl": r["reduced_by_nccl"], "nccl_version": r["nccl_version"], "device_ms": r["device_ms"],
            "device_instances": r["device_instances"]}


# ------------------------------------------------------------------------------------------------
# Dimitrov PLDP leg (BASELINE configs[3]: 16 384 constrained CoP QPs)
# ------------------------------------------------------------------------------------------------
PLDP_WORKLOAD = "dimitrov_pldp_16384_constrained_cop_qps_N16"


def _cpu_pldp_worker(args):
    import ctypes as C
    import pldp_oracle as po
    from jrl_walkgen_b200 import workloads
    blob, n, seconds = args
    K = workloads.DimitrovConstants()
    pb = {k: (np.frombuffer(v[0], dtype=v[1]).reshape(v[2]) if isinstance(v, tuple) else v) for k, v in blob.items()}
    L = po.lib()
    L.oracle_pldp_solve_batch.restype = C.c_long
    X = np.zeros((n, 32)); its = np.zeros(n, dtype=np.int32)
    done = 0; fails = 0
    t0 = time.perf_counter()
    while True:
        fails = L.oracle_pldp_solve_batch(C.c_int(16), C.c_void_p(K.iPu.ctypes.data), C.c_void_p(K.Px.ctypes.data),
                                          C.c_void_p(K.Pu.ctypes.data), C.c_int(n), C.c_void_p(pb["D"].ctypes.data),
                                          C.c_void_p(pb["m"].ctypes.data), C.c_void_p(pb["DPu"].ctypes.data),
                                          C.c_long(int(pb["dpu_stride"])), C.c_void_p(pb["DPx"].ctypes.data),
                                          C.c_long(int(pb["dpx_stride"])), C.c_void_p(pb["ZMPRef"].ctypes.data),
                                          C.c_void_p(pb["XkYk"].ctypes.data), C.c_void_p(X.ctypes.data),
                                          C.c_void_p(its.ctypes.data))
        done += n
        if time.perf_counter() - t0 >= seconds:
            break
    return done, time.perf_counter() - t0, int(fails)


def cpu_pldp_rate(pb, seconds=5.0, procs=None):
    """Oracle port of PLDPSolver::SolveProblem (bitwise equal to the reference's object code, tests/test_pldp_oracle.py;
    the port is used because a reference solver object cannot be reused across unrelated problems: its hot start would
    re-activate the previous problem's constraints), cold start, one process per core."""
    import multiprocessing as mp
    procs = procs or host_cores()
    n = min(256, len(pb["m"]))
    jobs = []
    for i in range(procs):
        a = (i * n) % max(1, len(pb["m"]) - n)
        blob = {k: ((np.ascontiguousarray(v[a:a + n]).tobytes(), v.dtype, (n,) + v.shape[1:]) if isinstance(v, np.ndarray) else v)
                for k, v in pb.items()}
        jobs.append((blob, n, seconds))
    with mp.get_context("fork").Pool(procs) as pool:
        res = pool.map(_cpu_pldp_worker, jobs)
    total = sum(r[0] for r in res); wall = max(r[1] for r in res)
    return {"value": total / wall, "unit": "PLDP solves/s", "cores": procs, "kind": "port",
            "sample": f"{procs} processes x {n} problems repeated for {seconds:.0f} s ({total} solves), cold start, "
                      "oracle port of PLDPSolver::SolveProblem (bitwise pinned to the reference object code)",
            "us_per_solve_per_core": 1e6 * wall * procs / total, "failures": sum(r[2] for r in res)}


def pldp_leg(ctx, wg, args, rank, fp64_peak, want_cpu):
    """configs[3]: 16 384 DISTINCT cold-started constrained CoP QPs, through both entry points: wg_pldp_solve_batch (the
    dense (m+1) x 32 matrix the reference hands to SolveProblem) and wg_pldp_solve_batch_ranked (rows as (A_r(0), A_r(1),
    i_r): the structure every reference call has); results are bitwise equal (tests/test_pldp_gpu.py)."""
    from jrl_walkgen_b200 import workloads
    B = args.pldp_instances
    K, pb = workloads.pldp_batch(B, seed=100 + rank)
    small = {k: (v[:2048] if isinstance(v, np.ndarray) else v) for k, v in pb.items()}
    ctx.pldp_set_constants(K.iPu, K.Px, K.Pu)
    dev = {k: (ctx.to_device(v) if isinstance(v, np.ndarray) else v) for k, v in pb.items()}
    dX = ctx.alloc(B * 32 * 8); dinfo = ctx.alloc(B * wg.PLDP_INFO_DTYPE.itemsize)
    d_flush = ctx.alloc(256 << 20)
    ms = {}
    for ranked in (False, True):
        for _ in range(3):
            ctx.pldp_solve(dev, mem=wg.WG_MEM_DEVICE, B=B, X=dX, info=dinfo, ranked=ranked)
        ctx.sync()
        ctx.prof_begin(args.steps + 4)
        for _ in range(args.steps):
            ctx._check(ctx.lib.wg_memset_device(ctx.h, d_flush.ptr, 0, 256 << 20))      # L2 flush between launches
            ctx.pldp_solve(dev, mem=wg.WG_MEM_DEVICE, B=B, X=dX, info=dinfo, ranked=ranked)
        prof = ctx.prof_end()
        ms[ranked] = prof[4][1] / prof[4][0]
    info = dinfo.download(wg.PLDP_INFO_DTYPE, (B,))
    it = info["iterations"].astype(np.float64); k = info["n_active"].astype(np.float64); m = pb["m"].astype(np.float64)
    u = 32.0
    # SURVEY 8d: F = 2u^2 (v0) + I (2 k u 2 + 2 k^2 + 2 m u) + sum_k (2 k u + k^2); k averaged as k_final / 2 over the run
    flops = float(np.sum(2 * u * u + it * (4 * (k / 2) * u + 2 * (k / 2) ** 2 + 2 * m * u) + k * (k * u + k * k / 3)))
    # end to end with pinned host buffers, both entries
    n_e2e = max(3, min(args.steps, 8))
    pin = {}
    for k_, v_ in pb.items():
        if isinstance(v_, np.ndarray):
            pin[k_] = ctx.pinned(v_.shape, v_.dtype); pin[k_][...] = v_
        else:
            pin[k_] = v_
    pX = ctx.pinned((B, 32)); pinfo = ctx.pinned((B,), wg.PLDP_INFO_DTYPE)
    e2e = {}
    for ranked in (False, True):
        ctx.pldp_solve(pin, X=pX, info=pinfo, ranked=ranked)
        te = time.perf_counter()
        for _ in range(n_e2e):
            ctx.pldp_solve(pin, X=pX, info=pinfo, ranked=ranked)
        e2e[ranked] = B * n_e2e / (time.perf_counter() - te)
        assert int(((pinfo["rc"] != 0) | (pinfo["status"] != 0)).sum()) == 0
    common = sum(pb[k_].nbytes for k_ in ("D", "m", "DPx", "ZMPRef", "XkYk"))
    h2d = {False: common + pb["DPu"].nbytes, True: common + pb["a0"].nbytes + pb["a1"].nbytes + pb["ri"].nbytes}
    d2h = int(B * (256 + wg.PLDP_INFO_DTYPE.itemsize))

    def roof(t_ms, note):
        ach = flops / (t_ms * 1e-3) / 1e12
        return {"kernel": "pldp_kernel", "bound": "fp64", "achieved": ach, "peak": fp64_peak, "unit": "TFLOP/s",
                "frac": ach / fp64_peak, "traffic": None, "algorithmic_flop_per_solve_mean": flops / B, "note": note}
    res = {"workload": PLDP_WORKLOAD, "instances": B, "distinct_problems": B,
           "pldp_solves_per_s": B / (ms[True] * 1e-3), "ms_per_launch": ms[True], "entry": "wg_pldp_solve_batch_ranked",
           "iterations_mean": float(it.mean()), "iterations_max": int(it.max()), "active_mean": float(k.mean()),
           "constraints_mean": float(m.mean()), "failures": int(((info["rc"] != 0) | (info["status"] != 0)).sum()),
           "roofline": roof(ms[True], "non-fused FP64 in the reference's serial summation order (bitwise parity): latency bound by "
                                      "design; rank-structured rows, no constraint matrix in memory"),
           "e2e": {"value": e2e[True], "unit": "PLDP solves/s", "h2d_bytes_per_step": int(h2d[True]), "d2h_bytes_per_step": d2h,
                   "api": "wg_pldp_solve_batch_ranked(WG_MEM_HOST), pinned host buffers, 4 pipelined chunks"},
           "dense_entry": {"entry": "wg_pldp_solve_batch", "pldp_solves_per_s": B / (ms[False] * 1e-3), "ms_per_launch": ms[False],
                           "roofline": roof(ms[False], "dense (m+1) x 32 matrix re-read from L2 every iteration"),
                           "e2e": {"value": e2e[False], "unit": "PLDP solves/s", "h2d_bytes_per_step": int(h2d[False]),
                                   "d2h_bytes_per_step": d2h,
                                   "api": "wg_pldp_solve_batch(WG_MEM_HOST), pinned host buffers, 4 pipelined chunks"}}}
    if want_cpu:
        res["cpu_baseline"] = cpu_pldp_rate(small, seconds=max(2.0, args.cpu_seconds / 2))
    for v in list(dev.values()) + [dX, dinfo, d_flush]:
        if hasattr(v, "free"):
            v.free()
    return res, {"pldp_kernel<ranked>": {"launches": args.steps, "avg_ms": ms[True]},
                 "pldp_kernel<dense>": {"launches": args.steps, "avg_ms": ms[False]}}


# ------------------------------------------------------------------------------------------------
# Dimitrov2008 front to back (SURVEY 8a rows a19-a21 in closed loop): footsteps -> feet -> support polygons ->
# per-period constraint matrices -> PLDP -> LIPM, CoM/ZMP at 5 ms, without leaving the GPU
# ------------------------------------------------------------------------------------------------
def _cpu_dimitrov_worker(args):
    import dimitrov_oracle as do
    import zmpdisc_oracle as zo
    walks, feet, seconds = args
    par = do.default_params()
    par.cold_restart = 1
    par.merge_duplicate_rows = 1
    zp = zo.default_params()
    periods = 0; done_walks = 0
    t0 = time.perf_counter()
    while True:
        for st, f in zip(walks, feet):
            o = zo.run(zp, st.astype(zo.REL_STEP_DTYPE), f)
            out = do.run(o["left"], o["right"], o["types"][:, 1].copy(), par)
            periods += len(out["periods"]); done_walks += 1
            if time.perf_counter() - t0 >= seconds:
                return periods, done_walks, time.perf_counter() - t0
        if not walks:
            return 0, 0, 1.0


def cpu_dimitrov_rate(off, steps, feet, seconds=5.0, procs=None):
    """The oracle chain (ZMPDiscretization, FootConstraintsAsLinearSystem, BuildConstraintMatrices, PLDP, LIPM
    restatements; hull/polygons/PLDP bitwise pinned to the reference's object code), one process per core."""
    import multiprocessing as mp
    procs = procs or host_cores()
    B = len(off) - 1
    jobs = []
    for i in range(procs):
        idx = [(i * 8 + k) % B for k in range(8)]
        jobs.append(([steps[off[b]:off[b + 1]].copy() for b in idx], [feet[b].copy() for b in idx], seconds))
    with mp.get_context("fork").Pool(procs) as pool:
        res = pool.map(_cpu_dimitrov_worker, jobs)
    total = sum(r[0] for r in res); wall = max(r[2] for r in res)
    return {"value": total / wall, "unit": "QP periods/s", "cores": procs, "kind": "port",
            "sample": f"{procs} processes x up to 8 walks repeated for {seconds:.0f} s ({total} periods, "
                      f"{sum(r[1] for r in res)} walks): oracle chain footsteps -> CoM, cold_restart = 1",
            "us_per_period_per_core": 1e6 * wall * procs / max(1, total)}


def dimitrov_leg(ctx, wg, args, rank, want_cpu):
    import ctypes as C
    from jrl_walkgen_b200 import workloads, _capi
    B = args.dimitrov_walks
    off, steps, feet = workloads.kajita_steps_batch(B, seed=2000 + 1000 * rank)
    par = wg.dimitrov_default_params()
    plan = ctx.kajita_plan(off, steps, feet)
    # one untimed pass with the reference's exact semantics (defaults): how many walks the reference itself would finish
    ctx.dimitrov_set_params(par)
    f_stat = np.zeros(B, dtype=np.int32); f_done = np.zeros(B, dtype=np.int32)
    t_ref_sem = None
    for rep in range(3):                                  # the last two repetitions are timed (wall clock, sync inside the call)
        if rep == 1:
            t_ref_sem = time.perf_counter()
        ctx._check(ctx.lib.wg_dimitrov_run_batch(ctx.h, plan.h, wg.WG_MEM_HOST, None, None, None, None, None, None,
                                                 f_stat.ctypes.data, f_done.ctypes.data))
    t_ref_sem = (time.perf_counter() - t_ref_sem) / 2
    par.cold_restart = 1
    par.merge_duplicate_rows = 1
    ctx.dimitrov_set_params(par)
    n = plan.total_samples
    so = plan.sample_offsets
    pc = np.array([ctx.lib.wg_dimitrov_period_count(C.byref(par), int(so[b + 1] - so[b])) for b in range(B)], dtype=np.int64)
    dcom = ctx.alloc(n * 48); dzmp = ctx.alloc(n * 16); dl = ctx.alloc(n * 48); dr = ctx.alloc(n * 48)
    dstat = ctx.alloc(B * 4); ddone = ctx.alloc(B * 4)

    def run_dev():
        ctx._check(ctx.lib.wg_dimitrov_run_batch(ctx.h, plan.h, wg.WG_MEM_DEVICE, dcom.ptr, dzmp.ptr, dl.ptr, dr.ptr, None,
                                                 None, dstat.ptr, ddone.ptr))
    for _ in range(2):
        run_dev()
    ctx.sync()
    reps = max(2, min(args.steps, 5))
    ctx.prof_begin(4 * reps + 8)
    ctx.timer_start()
    for _ in range(reps):
        plan.set_steps(steps, feet)
        run_dev()
    ms = ctx.timer_stop_ms() / reps
    prof = ctx.prof_end()
    status = dstat.download(np.int32, (B,)); done = ddone.download(np.int32, (B,))
    periods = int(done.sum())
    kern = {}
    for kid, name in ((7, "zmpdisc_kernel"), (8, "fcals_kernel"), (9, "dimitrov_kernel")):
        if kid in prof:
            kern[name] = {"launches": int(prof[kid][0]), "avg_ms": prof[kid][1] / prof[kid][0]}
    # end to end: host step lists in, host CoM / ZMP out
    com = ctx.pinned((n, 6)); zmp = ctx.pinned((n, 2))
    hstat = np.zeros(B, dtype=np.int32); hdone = np.zeros(B, dtype=np.int32)

    def run_host():
        plan.set_steps(steps, feet)
        ctx._check(ctx.lib.wg_dimitrov_run_batch(ctx.h, plan.h, wg.WG_MEM_HOST, com.ctypes.data, zmp.ctypes.data, None, None,
                                                 None, None, hstat.ctypes.data, hdone.ctypes.data))
    run_host()
    n_e2e = 2
    te = time.perf_counter()
    for _ in range(n_e2e):
        run_host()
    e2e_s = time.perf_counter() - te
    assert (hdone == done).all()
    res = {"workload": "dimitrov2008_footsteps_to_com_%d_walks_N16_pldp" % B, "walks": B, "samples": int(n),
           "qp_periods": periods, "qp_periods_if_all_walks_completed": int(pc.sum()), "ms_per_pass": ms,
           "qp_periods_per_s": periods / (ms * 1e-3), "walks_per_s": B / (ms * 1e-3),
           "walks_completed": int((status == 0).sum()), "walks_stopped": int((status != 0).sum()),
           "reference_semantics": {"walks_completed": int((f_stat == 0).sum()), "walks_stopped": int((f_stat != 0).sum()),
                                   "qp_periods_before_the_stops": int(f_done.sum()),
                                   "qp_periods_per_s": float(f_done.sum()) / t_ref_sem, "ms_per_pass": t_ref_sem * 1e3,
                                   "note": "defaults = the reference bit for bit: a walk stops where the reference calls "
                                           "exit(0) (m_tol drift of a hot start) or returns IFAIL (NaN on a duplicated half-plane)"},
           "note": "timed with cold_restart = 1 and merge_duplicate_rows = 1 (both off by default, both outside the "
                   "reference): infeasible hot starts are solved again from the cold start point, half-planes that repeat "
                   "their predecessor are dropped",
           "kernels": kern,
           "e2e": {"value": periods * n_e2e / e2e_s, "unit": "QP periods/s", "h2d_bytes_per_step": int(steps.nbytes + feet.nbytes),
                   "d2h_bytes_per_step": int(com.nbytes + zmp.nbytes + hstat.nbytes + hdone.nbytes),
                   "api": "wg_kajita_plan_set_steps + wg_dimitrov_run_batch(WG_MEM_HOST): step lists in, CoM/ZMP at 5 ms out"}}
    if want_cpu:
        res["cpu_baseline"] = cpu_dimitrov_rate(off, steps, feet, seconds=max(2.0, args.cpu_seconds / 2))
    for b in (dcom, dzmp, dl, dr, dstat, ddone):
        b.free()
    plan.destroy()
    return res, kern


def _cpu_wieber_worker(args):
    import wieber_oracle as wo
    import zmpdisc_oracle as zo
    walks, feet, seconds = args
    zp = zo.default_params()
    periods = 0
    t0 = time.perf_counter()
    while True:
        for st, f in zip(walks, feet):
            w = zo.run(zp, st.astype(zo.REL_STEP_DTYPE), f)
            budget = max(8, int((seconds - (time.perf_counter() - t0)) / 0.004))      # ~4 ms per QP: stop inside a walk
            k, _, _, _ = wo.run(w, max_periods=budget)
            periods += max(int(k), 0)
            if time.perf_counter() - t0 >= seconds:
                return periods, time.perf_counter() - t0


def cpu_wieber_rate(off, steps, feet, seconds=5.0, procs=None):
    """The oracle chain of the Wieber2006 generator (bitwise the reference's ZMPQPWithConstraint object code, tests/test_wieber.py)
    with the reference's own ql0001_ object code as the solver, one process per core (QLD is not re-entrant)."""
    import multiprocessing as mp
    procs = procs or host_cores()
    B = len(off) - 1
    jobs = []
    for i in range(procs):
        idx = [(i * 4 + k) % B for k in range(4)]
        jobs.append(([steps[off[b]:off[b + 1]].copy() for b in idx], [feet[b].copy() for b in idx], seconds))
    with mp.get_context("fork").Pool(procs) as pool:
        res = pool.map(_cpu_wieber_worker, jobs)
    total = sum(r[0] for r in res); wall = max(r[1] for r in res)
    return {"value": total / wall, "unit": "QP periods/s", "cores": procs, "kind": "reference",
            "sample": f"{procs} processes, walks of the batch for {seconds:.0f} s ({total} QPs of n = 150, m = 300..304): oracle "
                      "assembly (bitwise the reference object) + the reference's own ql0001_ object code",
            "us_per_qp_per_core": 1e6 * wall * procs / max(1, total)}


def wieber_leg(ctx, wg, args, rank, want_cpu, hbm_peak):
    """BASELINE configs[3] names 'Dimitrov ZMPQPWithConstraint ...': ZMPQPWithConstraint is the Wieber2006 generator (SURVEY 8f
    rank 3).  The straight / arc walks of configs[1] through wg_wieber_run_batch: one dense QP (n = 150, m = 300..304) per 20 ms."""
    from jrl_walkgen_b200 import workloads
    B = args.wieber_walks
    off, steps, feet = workloads.kajita_steps_batch(B, seed=3000 + 1000 * rank)
    ctx.wieber_set_params()
    plan = ctx.kajita_plan(off, steps, feet)
    n = plan.total_samples
    dcom = ctx.alloc(n * 48); dzmp = ctx.alloc(n * 16)
    dstat = ctx.alloc(B * 4); ddone = ctx.alloc(B * 4); dit = ctx.alloc(B * 8)

    def run_dev():
        ctx._check(ctx.lib.wg_wieber_run_batch(ctx.h, plan.h, wg.WG_MEM_DEVICE, dcom.ptr, dzmp.ptr, None, None, dstat.ptr,
                                               ddone.ptr, dit.ptr))
    run_dev()
    ctx.sync()
    reps = 2
    ctx.reset_launches()
    ctx.prof_begin(20000)
    ctx.timer_start()
    for _ in range(reps):
        run_dev()
    ms = ctx.timer_stop_ms() / reps
    prof = ctx.prof_end()
    launches = ctx.launches // reps
    status = dstat.download(np.int32, (B,)); done = ddone.download(np.int32, (B,)); its = dit.download(np.int64, (B,))
    periods = int(done.sum())
    kern = {}
    for kid, name in ((10, "qld_kernel"), (11, "wieber_pre_kernel + wieber_post_kernel")):
        if kid in prof:
            kern[name] = {"launches": int(prof[kid][0]), "avg_ms": prof[kid][1] / prof[kid][0], "total_ms": prof[kid][1]}
    com = ctx.pinned((n, 6)); zmp = ctx.pinned((n, 2))
    hstat = np.zeros(B, dtype=np.int32); hdone = np.zeros(B, dtype=np.int32)
    te = time.perf_counter()
    plan.set_steps(steps, feet)
    ctx._check(ctx.lib.wg_wieber_run_batch(ctx.h, plan.h, wg.WG_MEM_HOST, com.ctypes.data, zmp.ctypes.data, None, None,
                                           hstat.ctypes.data, hdone.ctypes.data, None))
    e2e_s = time.perf_counter() - te
    qld_ms = prof[10][1] / reps if 10 in prof else None
    # per QP the solver streams the m x n constraint matrix once per violation scan (iterations + 1 scans) plus once for the row norms
    m_mean, nvar = 300.0, 150
    scans = float(its.sum()) / max(periods, 1) + 2.0
    traffic_model = periods * m_mean * nvar * 8.0 * scans
    res = {"workload": "wieber2006_zmpqpwithconstraint_%d_straight_and_arc_walks_N75_T20ms" % B, "walks": B, "samples": int(n),
           "qp_periods": periods, "ms_per_pass": ms, "qp_periods_per_s": periods / (ms * 1e-3),
           "walks_completed": int((status == 0).sum()), "walks_stopped": int((status != 0).sum()),
           "active_set_changes_per_qp": float(its.sum()) / max(periods, 1), "launches_per_pass": int(launches),
           "kernels": kern,
           "roofline": None if qld_ms is None else {
               "kernel": "qld_kernel", "bound": "hbm", "achieved": traffic_model / (qld_ms * 1e-3) / 1e9, "peak": hbm_peak,
               "unit": "GB/s", "frac": traffic_model / (qld_ms * 1e-3) / 1e9 / hbm_peak, "traffic": None,
               "note": "model: every violation scan (active-set changes + 2 per QP) streams the 300 x 150 constraint matrix "
                       "(360 KB) of its QP; the kernel's other operands (the factor of the shared Hessian, the basis of the "
                       "active rows) are L2 resident"},
           "e2e": {"value": periods / e2e_s, "unit": "QP periods/s", "h2d_bytes_per_step": int(steps.nbytes + feet.nbytes),
                   "d2h_bytes_per_step": int(com.nbytes + zmp.nbytes + hstat.nbytes + hdone.nbytes),
                   "api": "wg_kajita_plan_set_steps + wg_wieber_run_batch(WG_MEM_HOST): step lists in, CoM/ZMP at 5 ms out"}}
    if want_cpu:
        res["cpu_baseline"] = cpu_wieber_rate(off, steps, feet, seconds=max(2.0, args.cpu_seconds / 2))
    for b in (dcom, dzmp, dstat, ddone, dit):
        b.free()
    plan.destroy()
    return res, kern


DUMP_ROWS = 1 << 19          # preview steps sampled by --dump-outputs: 512 Ki rows of CoM + ZMP = 32 MB


def dump_preview_outputs(out_dir, dcom, dzmp, ds, B, n):
    """--dump-outputs: what the last timed pass hands its caller, as float64 .npy files - the CoM [n][6] and ZMP [n][2]
    rows at a fixed, seeded sample of the n preview steps (every row when n <= DUMP_ROWS), the sampled row indices, and
    the final [B][8] state of every walk.  The workload is seeded, so two builds can be compared file by file."""
    os.makedirs(out_dir, exist_ok=True)
    com = dcom.download(np.float64, (n, 6))
    zmp = dzmp.download(np.float64, (n, 2))
    rows = np.arange(n) if n <= DUMP_ROWS else np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))
    np.save(os.path.join(out_dir, "preview_com.npy"), com[rows])
    np.save(os.path.join(out_dir, "preview_zmp.npy"), zmp[rows])
    np.save(os.path.join(out_dir, "preview_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "preview_state.npy"), ds.download(np.float64, (B, 8)))


def run_cuda(args):
    rank, local_rank, world = dist_env()
    import jrl_walkgen_b200 as wg
    from jrl_walkgen_b200 import workloads
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        # host-side barrier for the one leg in which rank 0 drives every GPU itself: an NCCL barrier would park a spinning
        # kernel on the other ranks' GPUs (measured: 2.2x slower sweep on the GPU whose rank waits in dist.barrier())
        cpu_group = dist.new_group(backend="gloo")
    numa_note = pin_to_gpu_numa_node(local_rank) if world > 1 else \
        {"pinned": False, "why": "single rank: affinity left alone (the CPU baseline legs use every core)"}
    ctx = wg.Context(local_rank)
    gains = wg.preview_gains(0.005, 1.6, 0.814, wg.MODE_WITHOUT_INITIALPOS)
    ctx.preview_set_gains(gains)
    offsets, z = headline_workload_gpu(ctx, args.walks, seed=1000 * rank)
    B = args.walks
    n = int(offsets[-1])
    plan = ctx.preview_plan(offsets)
    steps_per_pass = int(plan.total_steps)

    # ---- device-resident leg (value) -------------------------------------------------------
    dz = ctx.to_device(z)
    st0 = np.zeros((B, 8))                      # every pass starts from rest: the states are reset on the device (memset)
    ds = ctx.to_device(st0)
    dcom = ctx.alloc(n * 48); dzmp = ctx.alloc(n * 16)

    def barrier():
        ctx.sync()
        if dist is not None:
            dist.barrier()

    def one_pass():
        ctx._check(ctx.lib.wg_memset_device(ctx.h, ds.ptr, 0, st0.nbytes))  # reset 256 KB of states (all zero) on the device
        plan.run(dz, ds, dcom, dzmp, True, mem=wg.WG_MEM_DEVICE)

    # A bench "step" is `passes` passes over the 4096-walk batch (default 160: K = 20 steps time ~1.2 s of kernels, so that
    # clocks and throttle reasons are sampled under sustained load; one pass alone is 0.39 ms).  Every pass re-reads the
    # 254 MB input and rewrites the 1.0 GB output, far above the 126 MB L2: nothing is served from cache between passes.
    passes = max(1, args.passes_per_step)
    for _ in range(max(args.warmup, 3)):
        for _ in range(passes):
            one_pass()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.25)
    ctx.reset_launches()
    ctx.prof_begin(passes * args.steps + 8)
    barrier()
    t0 = time.time()
    ctx.timer_start()
    for _ in range(args.steps * passes):
        one_pass()
    ms_total = ctx.timer_stop_ms()
    t1 = time.time()
    barrier()
    launches = ctx.launches
    prof = ctx.prof_end()
    sum_mode, fit_resid = ctx.preview_sum_info()
    if args.dump_outputs and rank == 0:
        # before the direct-sum leg below reuses the same output buffers
        dump_preview_outputs(args.dump_outputs, dcom, dzmp, ds, B, n)

    # ---- the same pass with the preview sum evaluated directly (the 320-tap FIR of preview_fused_kernel, FP64-pipe bound):
    # the kernel the recursive evaluation replaced as the default, timed beside it on the same inputs
    direct = None
    if sum_mode == wg.PREVIEW_SUM_RECURSIVE:
        ctx.preview_set_sum_mode(wg.PREVIEW_SUM_DIRECT)
        dpasses = max(8, passes // 4)
        for _ in range(4):
            one_pass()
        barrier()
        ctx.prof_begin(dpasses * max(1, args.steps // 4) + 8)
        ctx.timer_start()
        for _ in range(max(1, args.steps // 4) * dpasses):
            one_pass()
        d_ms = ctx.timer_stop_ms()
        dprof = ctx.prof_end()
        barrier()
        ctx.preview_set_sum_mode(wg.PREVIEW_SUM_AUTO)
        direct = {"ms_total": d_ms, "passes": max(1, args.steps // 4) * dpasses, "kernel_avg_ms": dprof[6][1] / dprof[6][0]}

    # ---- end-to-end leg: host buffers through the C ABI (H2D + kernels + D2H inside) ---------
    zp = ctx.pinned(z.shape); zp[:] = z
    stp = ctx.pinned((B, 8))
    comp = ctx.pinned((n, 6)); zmpp = ctx.pinned((n, 2))
    e2e_steps = max(args.steps, args.e2e_passes)          # ~21 ms per pass: 48 passes time ~1 s
    for _ in range(2):
        stp[:] = 0.0
        plan.run(zp, stp, comp, zmpp, True, mem=wg.WG_MEM_HOST)
    barrier()
    te = time.perf_counter()
    for _ in range(e2e_steps):
        stp[:] = 0.0
        plan.run(zp, stp, comp, zmpp, True, mem=wg.WG_MEM_HOST)
    ctx.sync()
    e2e_s = time.perf_counter() - te
    # output selection (wg_preview_run_batch_pos): a caller that only consumes the CoM position moves 16 + 16 B per step
    posp = ctx.pinned((n, 2))
    for _ in range(2):
        stp[:] = 0.0
        plan.run_pos(zp, stp, posp, True, mem=wg.WG_MEM_HOST)
    barrier()
    te = time.perf_counter()
    for _ in range(e2e_steps):
        stp[:] = 0.0
        plan.run_pos(zp, stp, posp, True, mem=wg.WG_MEM_HOST)
    ctx.sync()
    e2e_pos_s = time.perf_counter() - te
    clocks = sampler.stop(t0, t1)
    h2d = z.nbytes + stp.nbytes
    d2h = comp.nbytes + zmpp.nbytes + stp.nbytes

    # ---- host link probe: what the e2e leg is bounded by.  Every rank copies 256 MB pinned <-> device at the same time
    # (after a barrier); the per-rank rates are summed over the ranks.  On one GPU this is the PCIe link; at N > 1 the sum
    # shows whether the box's host side (root complex / host DRAM / virtualised IOMMU path) scales with the GPU count.
    link = {}
    nb_probe = 256 << 20
    dprobe = ctx.alloc(nb_probe)
    hprobe = ctx.pinned((nb_probe // 8,))
    hprobe[:] = 1.0
    for name, fn in (("h2d", lambda: ctx._check(ctx.lib.wg_memcpy_h2d(ctx.h, dprobe.ptr, hprobe.ctypes.data, nb_probe))),
                     ("d2h", lambda: ctx._check(ctx.lib.wg_memcpy_d2h(ctx.h, hprobe.ctypes.data, dprobe.ptr, nb_probe)))):
        fn(); ctx.sync()
        barrier()
        tp = time.perf_counter()
        for _ in range(4):
            fn()
        ctx.sync()
        link[name] = 4 * nb_probe / (time.perf_counter() - tp) / 1e9
    dprobe.free()
    (_, _), (h2d_sum, d2h_sum) = reduce_over_ranks(dist, [0.0, 0.0], [link["h2d"], link["d2h"]])
    link = {"h2d_gbs_sum_over_ranks": h2d_sum, "d2h_gbs_sum_over_ranks": d2h_sum, "ranks": world,
            "how": "4 x 256 MB pinned copies per direction per rank, all ranks at once"}

    # ---- max over ranks ----------------------------------------------------------------------
    d_ms_all = direct["ms_total"] if direct else 0.0
    (ms_total, e2e_s, e2e_pos_s, d_ms_all), (total_steps_all,) = reduce_over_ranks(dist, [ms_total, e2e_s, e2e_pos_s, d_ms_all], [float(steps_per_pass)])
    ms_per_step = ms_total / args.steps
    value = total_steps_all * passes / (ms_per_step * 1e-3)
    e2e_value = total_steps_all * e2e_steps / e2e_s
    for b_ in (dz, ds, dcom, dzmp):
        b_.free()
    launches_preview = launches
    herdt = herdt_kern = None
    if not args.no_herdt:
        fp64_peak_all = ctx.fp64_peak_tflops()
        ctx.reset_launches()
        herdt, herdt_kern = herdt_leg(ctx, wg, args, rank, fp64_peak_all, want_cpu=(rank == 0 and world == 1))
        if dist is not None:
            import torch
            t = torch.tensor([1.0 / herdt["qp_solves_per_s"], 1.0 / herdt["closed_loop_qp_solves_per_s"]],
                             dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)          # slowest rank
            herdt["qp_solves_per_s"] = world / float(t[0])
            herdt["closed_loop_qp_solves_per_s"] = world / float(t[1])
            herdt["instances"] = herdt["instances"] * world
    pldp = None
    if not args.no_pldp:
        pldp, pldp_kern = pldp_leg(ctx, wg, args, rank, ctx.fp64_peak_tflops(), want_cpu=(rank == 0 and world == 1))
        herdt_kern = dict(herdt_kern or {}, **pldp_kern)
        if dist is not None:
            import torch
            t = torch.tensor([1.0 / pldp["pldp_solves_per_s"]], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            pldp["pldp_solves_per_s"] = world / float(t[0])
            pldp["instances"] = pldp["instances"] * world

    kajita = None
    if not args.no_kajita:
        try:
            hbm_pk = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs", 6650.0))
        except OSError:
            hbm_pk = 6650.0
        kajita, kj_kern = kajita_leg(ctx, wg, args, rank, hbm_pk)
        herdt_kern = dict(herdt_kern or {}, **kj_kern)
        if dist is not None:
            (t_k,), (s_k,) = reduce_over_ranks(dist, [kajita["ms_per_pass"]], [float(kajita["preview_steps"])])
            kajita["preview_steps_per_s"] = s_k / (t_k * 1e-3)
            kajita["walks"] = kajita["walks"] * world
    dimitrov = None
    if not args.no_dimitrov:
        dimitrov, dm_kern = dimitrov_leg(ctx, wg, args, rank, want_cpu=(rank == 0 and world == 1))
        herdt_kern = dict(herdt_kern or {}, **dm_kern)
        if dist is not None:
            (t_d,), (p_d, w_d) = reduce_over_ranks(dist, [dimitrov["ms_per_pass"]], [float(dimitrov["qp_periods"]), float(dimitrov["walks"])])
            dimitrov["qp_periods_per_s"] = p_d / (t_d * 1e-3)
            dimitrov["walks_per_s"] = w_d / (t_d * 1e-3)
            dimitrov["walks"] = int(w_d)
    wieber = None
    if not args.no_wieber:
        try:
            hbm_pk2 = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs", 6650.0))
        except OSError:
            hbm_pk2 = 6650.0
        wieber, wb_kern = wieber_leg(ctx, wg, args, rank, want_cpu=(rank == 0 and world == 1), hbm_peak=hbm_pk2)
        herdt_kern = dict(herdt_kern or {}, **wb_kern)
        if dist is not None:
            (t_w,), (p_w, w_w) = reduce_over_ranks(dist, [wieber["ms_per_pass"]], [float(wieber["qp_periods"]), float(wieber["walks"])])
            wieber["qp_periods_per_s"] = p_w / (t_w * 1e-3)
            wieber["walks"] = int(w_w)
    sweep = None
    if not args.no_sweep:
        sweep = sweep_leg(ctx, wg, args, rank, world, dist)
        # the same sweep through the LIBRARY's own sharding driver (wg_multi: one process, a host thread per device, NCCL
        # all-reduce of the statistics): rank 0 drives all `world` devices while the other ranks wait at the barrier below
        if dist is not None:
            torch.cuda.synchronize()
            dist.barrier(group=cpu_group)
        if rank == 0:
            try:
                sweep["library_multi_gpu"] = library_multi_leg(wg, args, world)
            except Exception as e:                                       # noqa: BLE001 - reported, not fatal for the line
                sweep["library_multi_gpu"] = {"error": str(e)}
        if dist is not None:
            dist.barrier(group=cpu_group)

    if rank == 0:
        # roofline of the dominant kernel (largest share of the timed region)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        hbm_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
        fp64_peak = ctx.fp64_peak_tflops()
        launches = launches_preview
        names = {6: "preview_fused_kernel", 2: "herdt_qp_kernel", 3: "herdt_mpc_kernel", 4: "pldp_kernel"}
        kern = {names.get(k, str(k)): {"launches": v[0], "avg_ms": v[1] / v[0]} for k, v in prof.items()}
        dom = max(kern.items(), key=lambda kv: kv[1]["avg_ms"] * kv[1]["launches"])
        dom_name, dom_ms = dom[0], dom[1]["avg_ms"]
        fp64_src = ("measured live: register-resident DFMA chains on all SMs (wg_measure_fp64_peak); "
                    "MEASURED_PEAKS.json has no FP64 entry")
        if sum_mode == wg.PREVIEW_SUM_RECURSIVE:
            # the window sum as a backward linear recurrence (~170 FMA per step for everything): the kernel streams 16 B in
            # and 64 B out per step and is bounded by HBM, SURVEY 8(d)'s 80 B per step.  A device-resident batch of >= 2048
            # walks runs one warp per trajectory (preview_rec_warp_kernel), smaller ones preview_rec_kernel (preview.cu)
            shape_env = os.environ.get("WG_PREVIEW_SHAPE")
            one_warp = (int(shape_env) == 2) if shape_env is not None else args.walks >= 2048
            dom_name = "preview_rec_warp_kernel" if one_warp else "preview_rec_kernel"
            kern = {dom_name: kern.pop("preview_fused_kernel")}
            ach = BYTES_PER_STEP * steps_per_pass / (dom_ms * 1e-3) / 1e9
            roof = {"kernel": dom_name, "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                    "frac": ach / hbm_peak, "traffic": None, "peak_source": hbm_src + ", burst copy figure",
                    "algorithmic_bytes_per_step": BYTES_PER_STEP,
                    "fp64_frac_on_the_direct_sum_flop_model": FLOP_PER_STEP * steps_per_pass / (dom_ms * 1e-3) / 1e12 / fp64_peak,
                    "note": "the direct-sum flop model (1360 flop per step) no longer describes the work: the recursive "
                            "evaluation executes ~340 flop per step; see direct_sum for the FIR kernel on the same inputs"}
        else:
            fl = (FIR_FLOP_PER_STEP if dom_name == "preview_fir_kernel" else FLOP_PER_STEP)
            ach = fl * steps_per_pass / (dom_ms * 1e-3) / 1e12
            roof = {"kernel": dom_name, "bound": "fp64", "achieved": ach, "peak": fp64_peak, "unit": "TFLOP/s",
                    "frac": ach / fp64_peak, "traffic": None,
                    "peak_source": fp64_src, "algorithmic_flop_per_step": fl}
        roof["hbm_frac_streaming_minimum"] = BYTES_PER_STEP * steps_per_pass * passes / (ms_per_step * 1e-3) / 1e9 / hbm_peak
        roof["algorithmic_bytes_per_launch"] = BYTES_PER_STEP * steps_per_pass
        # dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of this (seeded, deterministic) workload: not
        # measurable from inside the process, so it is read from the committed summary of the round's `ncu --set full`
        # capture of this same command (profiles/ncu_traffic.json, written by tools/ncu_summary.py --traffic); null when
        # that file has no entry for this kernel and batch size.
        roof.update(ncu_traffic(dom_name, args.walks))
        direct_line = None
        if direct:
            d_ms_pass = d_ms_all / direct["passes"]
            d_ach = FLOP_PER_STEP * steps_per_pass / (direct["kernel_avg_ms"] * 1e-3) / 1e12
            direct_line = {"kernel": "preview_fused_kernel", "value": total_steps_all / (d_ms_pass * 1e-3), "unit": UNIT,
                           "ms_per_pass": d_ms_pass, "passes": direct["passes"],
                           "roofline": dict({"bound": "fp64", "achieved": d_ach, "peak": fp64_peak, "unit": "TFLOP/s",
                                             "frac": d_ach / fp64_peak, "peak_source": fp64_src,
                                             "algorithmic_flop_per_step": FLOP_PER_STEP},
                                            **ncu_traffic("preview_fused_kernel", args.walks)),
                           "how": "wg_preview_set_sum_mode(WG_PREVIEW_SUM_DIRECT): the 320-tap sum as written in "
                                  "PreviewControl.cpp:346-352, same inputs, device resident"}
        cpu = None
        if world == 1:
            subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "liboracle.so"], check=True)
            cpu = cpu_preview_rate(offsets, z, seconds=args.cpu_seconds)
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": WORKLOAD, "walks_per_gpu": B, "NL": 320, "T": 0.005,
                           "preview_steps_per_pass_per_gpu": steps_per_pass, "passes_per_step": passes,
                           "l2": "inputs+outputs per pass (%.2f GB) exceed the 126 MB L2" % ((n * 80) / 1e9)},
                "roofline": roof, "preview_sum": {"mode": "recursive" if sum_mode == wg.PREVIEW_SUM_RECURSIVE else "direct",
                                                  "fit_residual_relative": fit_resid, "direct_sum": direct_line},
                "kernels": dict(kern, **(herdt_kern or {})), "fp64_peak_tflops_measured": fp64_peak,
                "herdt": herdt, "pldp": pldp, "kajita_front_end": kajita, "dimitrov_front_to_back": dimitrov, "wieber_front_to_back": wieber, "sweep": sweep,
                "herdt_qp_solves_per_s": None if herdt is None else herdt["qp_solves_per_s"],
                "herdt_qp_solves_per_s_e2e": None if herdt is None else herdt["e2e"]["value"],
                "cpu_baseline": cpu,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                        "passes": e2e_steps, "api": "wg_preview_run_batch(WG_MEM_HOST), pinned host buffers",
                        "com_position_only": {"value": total_steps_all * e2e_steps / e2e_pos_s, "unit": UNIT,
                                              "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(posp.nbytes + stp.nbytes),
                                              "api": "wg_preview_run_batch_pos(WG_MEM_HOST): output selection, 16 B per step out"},
                        "numa": numa_note,
                        "host_link": link,
                        "bound": "host link: %.0f B per preview step cross PCIe (16 in, 64 out); at the probed D2H rate the "
                                 "64 B/step alone cap the leg at %.2f G steps/s" % (BYTES_PER_STEP, d2h_sum / 64.0)},
                "gpu_launches": int(launches), "clocks": clocks}
        emit_line(line)
    plan.destroy()
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()


_STDOUT_FD = None


def emit_line(line):
    """The bench's JSON line, on the process's real stdout."""
    sys.stdout.flush()
    if _STDOUT_FD is not None:
        os.dup2(_STDOUT_FD, 1)
    print(json.dumps(line), flush=True)
    if _STDOUT_FD is not None:
        os.dup2(2, 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--walks", type=int, default=4096)
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--herdt-instances", type=int, default=16384)
    ap.add_argument("--herdt-periods", type=int, default=10)
    ap.add_argument("--no-herdt", action="store_true")
    ap.add_argument("--pldp-instances", type=int, default=16384)
    ap.add_argument("--no-pldp", action="store_true")
    ap.add_argument("--no-kajita", action="store_true")
    ap.add_argument("--dimitrov-walks", type=int, default=4096)
    ap.add_argument("--no-dimitrov", action="store_true")
    ap.add_argument("--wieber-walks", type=int, default=888)   # 3 x 296 resident CTAs of the dense QP kernel
    ap.add_argument("--no-wieber", action="store_true")
    ap.add_argument("--sweep", action="store_true", help="(default since round 2; kept for old command lines)")
    ap.add_argument("--no-sweep", action="store_true", help="skip BASELINE configs[4]: 1M MPC instances x 100 periods")
    ap.add_argument("--passes-per-step", type=int, default=160,
                    help="passes over the batch per bench step (timed region = steps x passes x 0.39 ms: >= 1 s at the default 20 steps)")
    ap.add_argument("--e2e-passes", type=int, default=48)
    ap.add_argument("--sweep-instances", type=int, default=1000000)
    ap.add_argument("--sweep-periods", type=int, default=100)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the CoM / ZMP / state outputs of the last timed pass as DIR/*.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "cuda":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl cuda)")
    # stdout carries the ONE JSON line and nothing else: libraries that print to file descriptor 1 on their own (NCCL announces
    # its version there when the box sets NCCL_DEBUG) are sent to stderr for the run; emit_line() puts the descriptor back
    global _STDOUT_FD
    sys.stdout.flush()
    _STDOUT_FD = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_cuda(args)


if __name__ == "__main__":
    main()
