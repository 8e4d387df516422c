"""The on-line Kajita generator one control tick at a time (wg_kajita_online_*), device-resident rows, NL = 320.

At each --batch size B, for each start leg and each number of ticks per call, one handle of B walks (walk b starts with its
support-foot step and two steps of 0.2 m, then refills from its empty stack with the default in-place step, no commands):
  all       every walk started at tick 0: the walks refill together, on one tick in 160;
  stagger   walk b started at tick b mod 160: B/160 walks refill on every tick.
The start phase (ticks 0..159, the walks of the stagger leg started one group per tick) is not timed.  Then --ticks ticks
in calls of N ticks (--calls-of) into device rows [N][B]: walk-ticks/s from a host clock around the window and the
synchronise after it, device ms per call from CUDA events around the window, host ms per call from a host clock around
each call (the call returns before the device is done: this is the host's replay of the tick rules, O(B * N), and the
enqueue), launches per call with and without a refill.  Prints one JSON line with the card's name and power limit (and
writes it to --out).

    python tools/bench_kajita_online.py [--batch 4096 65536] [--ticks 2000] [--calls-of 1 20]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import jrl_walkgen_b200 as wg  # noqa: E402
from bench_kajita_stream import card  # noqa: E402

FEET = np.array([0.00949035, 0.095, 0.0, 0.00949035, -0.095, 0.0])


def start_steps():
    s = np.zeros(3, dtype=wg.REL_STEP_DTYPE)
    s["sy"] = [-0.095, 0.19, -0.19]
    s["sx"] = [0.0, 0.2, 0.2]
    s["ss_time"], s["ds_time"], s["step_type"] = 0.78, 0.02, 1
    return s


def leg(ctx, B, stagger, N, nticks):
    h = ctx.kajita_online(B)
    d_rows, d_run = ctx.alloc(N * B * wg.KAJITA_TICK_DTYPE.itemsize), ctx.alloc(N * B)
    st = start_steps()
    try:
        for t in range(160):                      # start phase, untimed
            idx = np.arange(t, B, 160) if stagger else (np.arange(B) if t == 0 else np.arange(0))
            if len(idx):
                h.start(idx, [st] * len(idx), np.tile(FEET, (len(idx), 1)))
            h.tick_device(1, None, d_rows, d_run)
        ctx.sync()
        calls = nticks // N
        host_ms, launches = [], []
        ctx.timer_start()
        t0 = time.perf_counter()
        for _ in range(calls):
            l0 = ctx.launches
            a = time.perf_counter()
            h.tick_device(N, None, d_rows, d_run)
            host_ms.append((time.perf_counter() - a) * 1e3)
            launches.append(ctx.launches - l0)
        dev_ms = ctx.timer_stop_ms()
        wall = time.perf_counter() - t0
        launches = np.array(launches)
        assert h.state()[2].all()
        return {"B": B, "start": "stagger" if stagger else "all", "ticks_per_call": N, "calls": calls,
                "walk_ticks_per_s": B * calls * N / wall, "wall_ms_per_call": 1e3 * wall / calls,
                "device_ms_per_call": dev_ms / calls, "host_ms_per_call": float(np.mean(host_ms)),
                "host_ms_per_call_p50": float(np.median(host_ms)),
                "launches_per_call": float(launches.mean()),
                "launch_counts": sorted(set(int(x) for x in launches)),
                "calls_with_refill": int((launches > 1).sum()), "ring_rows": h.ring_rows}
    finally:
        h.destroy()
        d_rows.free(); d_run.free()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, nargs="+", default=[4096, 65536])
    ap.add_argument("--ticks", type=int, default=2000)
    ap.add_argument("--calls-of", type=int, nargs="+", default=[1, 20])
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    ctx = wg.Context(0)
    ctx.preview_set_gains(wg.preview_gains(0.005, 1.6, 0.814, wg.MODE_WITHOUT_INITIALPOS))
    res = {"card": card(), "legs": []}
    try:
        leg(ctx, 256, True, 20, 200)              # warm-up: module load, first allocations
        for B in a.batch:
            for stagger in (False, True):
                for N in a.calls_of:
                    r = leg(ctx, B, stagger, N, a.ticks)
                    print(json.dumps(r), file=sys.stderr)
                    res["legs"].append(r)
    finally:
        ctx.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
