"""Plans of the on-line Herdt2010 generator (wg_herdt_online_tick_plan) against the plain tick, device-resident.

  ticks      at each --batch size B, the aligned and staggered handles of bench_herdt_online.py (every robot starting at
             tick 0, so all fire on one tick in 20; robot b starting at tick b mod 20, so B/20 fire every tick).  Legs: tick
             and tick_plan (plans and plan_tick to device buffers), alternating pass by pass; a pass is --ticks ticks, 20 per
             call, rows and running flags to device buffers, timed with CUDA events on the context stream.
  kernel     device ms of online_plan_kernel alone on a tick where every robot fires and on one where none does (aligned
             handle), from torch.profiler's CUDA kernel records in a separate pass; bytes from the shapes (1888 B of plan
             written, 784 B of QP record and 960 B of QP output read per firing robot) and GB/s.
  lookahead  the cycle of bench_herdt_online_fork.py (--live robots, --branches K each: copy, 20 branch ticks under candidate
             velocities, 20 live ticks), with and without plans on the branch ticks, alternating; ms per decision.
Card name and power limit are read in the same command.  Prints one JSON line (and writes it to --out).

    python tools/bench_herdt_online_plan.py [--batch 16384 1000000] [--ticks 2000] [--reps 3] [--out FILE]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import jrl_walkgen_b200 as wg  # noqa: E402
from bench_herdt_online import Bench, CHUNK, card  # noqa: E402
from bench_herdt_online_fork import staggered  # noqa: E402

PLAN = 1888
PLAN_READ = 784 + 960   # QP record and QP output of a firing robot


def plan_pass(bench, h, d_plans, d_pt, nticks):
    ctx = bench.ctx
    ctx.sync()
    ctx.timer_start()
    for _ in range(nticks // CHUNK):
        h.tick_plan_device(CHUNK, d_plans, bench.d_cmd, bench.d_rows, bench.d_run, d_pt)
    return ctx.timer_stop_ms()


def plan_kernel_ms(bench, d_plans, d_pt):
    """(all-fire ms, none-fire ms, robots fired) of online_plan_kernel on the aligned handle, from torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    ctx, h = bench.ctx, bench.aligned
    q = h.states()
    phase = int(round((q["upper_time_limit"][0] - q["clock"][0]) / 0.005))   # ticks until the next QP instant
    for _ in range(phase - 1 if phase > 0 else 19):
        h.tick_plan_device(1, d_plans, bench.d_cmd, None, None, d_pt)
    ctx.sync()
    q0 = h.states()["qp_count"].sum()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:   # the firing tick, then a tick without any QP
        h.tick_plan_device(1, d_plans, bench.d_cmd, None, None, d_pt)
        ctx.sync()
        fired = int(h.states()["qp_count"].sum() - q0)
        h.tick_plan_device(1, d_plans, bench.d_cmd, None, None, d_pt)
        ctx.sync()
        torch.cuda.synchronize()
    ev = sorted((e for e in prof.events() if "online_plan_kernel" in e.name), key=lambda e: e.time_range.start)
    if len(ev) != 2:                          # a record was lost: the two cannot be told apart
        return None, None, fired
    res = [e.time_range.elapsed_us() / 1e3 for e in ev]
    return res[0], res[1], fired


def lookahead(ctx, live_n, K, decisions):
    nb = live_n * K
    live = staggered(ctx, live_n)
    br = ctx.herdt_online(nb)
    rng = np.random.default_rng(3)
    cand = np.column_stack([np.linspace(0.0, 0.3, K), np.zeros(K), np.linspace(-0.2, 0.2, K)])
    bcmd = np.zeros((20, nb), dtype=wg.HERDT_COMMAND_DTYPE)
    bcmd["vel"] = np.tile(cand, (live_n, 1))[None, :, :]
    bcmd["flags"] = wg.CMD_VEL
    lcmd = np.zeros((20, live_n), dtype=wg.HERDT_COMMAND_DTYPE)
    lcmd["vel"] = np.column_stack([rng.uniform(0.0, 0.3, live_n), rng.uniform(-0.1, 0.1, live_n),
                                   rng.uniform(-0.2, 0.2, live_n)])[None, :, :]
    lcmd["flags"] = wg.CMD_VEL
    d_bcmd, d_lcmd = ctx.to_device(bcmd), ctx.to_device(lcmd)
    d_rows, d_run = ctx.alloc(20 * live_n * wg.TICK_DTYPE.itemsize), ctx.alloc(20 * live_n)
    d_plans, d_pt = ctx.alloc(nb * PLAN), ctx.alloc(nb * 4)
    src = np.repeat(np.arange(live_n, dtype=np.int32), K)

    def decision(plans):
        br.copy_from(live, src_idx=src)
        if plans:
            br.tick_plan_device(20, d_plans, d_bcmd, None, None, d_pt)
        else:
            br.tick_device(20, d_bcmd)
        live.tick_device(20, d_lcmd, d_rows, d_run)

    out = {False: [], True: []}
    for rep in range(4):
        for plans in (False, True):
            decision(plans)
            ctx.sync()
            ctx.timer_start()
            for _ in range(decisions):
                decision(plans)
            ms = ctx.timer_stop_ms() / decisions
            if rep:
                out[plans].append(ms)
    for d in (d_bcmd, d_lcmd, d_rows, d_run, d_plans, d_pt):
        d.free()
    live.destroy(); br.destroy()
    base, withp = float(np.median(out[False])), float(np.median(out[True]))
    return {"live": live_n, "branches_per_robot": K, "decisions": decisions, "ms_per_decision": round(base, 4),
            "ms_per_decision_with_plans": round(withp, 4), "plans_over_plain": round(withp / base, 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, nargs="+", default=[16384, 1000000])
    ap.add_argument("--ticks", type=int, default=2000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--live", type=int, default=16384)
    ap.add_argument("--branches", type=int, default=8)
    ap.add_argument("--decisions", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert a.ticks % CHUNK == 0
    ctx = wg.Context(0)
    ctx.herdt_set_params()
    ctx.herdt_mpc_set_params()
    out = {"card": card(), "ticks_per_pass": a.ticks, "ticks_per_call": CHUNK, "reps": a.reps, "results": []}
    for B in a.batch:
        bench = Bench(ctx, B)
        d_plans, d_pt = ctx.alloc(B * PLAN), ctx.alloc(B * 4)
        legs = {}
        for mode in ("aligned", "staggered"):
            h = getattr(bench, mode)
            legs[mode + "_tick"] = (lambda h=h: bench.online_pass(h, a.ticks)[0])
            legs[mode + "_tick_plan"] = (lambda h=h: plan_pass(bench, h, d_plans, d_pt, a.ticks))
        ms = {k: [] for k in legs}
        for rep in range(a.reps + 1):            # rep 0 warms every leg up
            for k, f in legs.items():
                v = f()
                if rep:
                    ms[k].append(v)
        r = {"B": B}
        for k, v in ms.items():
            r[k] = {"ms_median": round(float(np.median(v)), 3), "ms_min": round(min(v), 3), "ms_max": round(max(v), 3)}
        for mode in ("aligned", "staggered"):
            r[mode + "_plan_over_tick"] = round(r[mode + "_tick_plan"]["ms_median"] / r[mode + "_tick"]["ms_median"], 4)
        all_ms, none_ms, fired = plan_kernel_ms(bench, d_plans, d_pt)
        nbytes = fired * (PLAN + PLAN_READ)
        r["plan_kernel"] = {"robots_fired": fired, "all_fire_ms": all_ms, "none_fire_ms": none_ms, "bytes": nbytes,
                            "GB_per_s": round(nbytes / (all_ms * 1e-3) / 1e9, 1) if all_ms else None}
        out["results"].append(r)
        print(json.dumps(r), flush=True)
        d_plans.free(); d_pt.free()
        bench.free()
    out["lookahead"] = lookahead(ctx, a.live, a.branches, a.decisions)
    print(json.dumps(out["lookahead"]), flush=True)
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
