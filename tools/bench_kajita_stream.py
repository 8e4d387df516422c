"""Footsteps -> CoM on 4096 walks of workloads.kajita_steps_batch, off-line against on-line:
  (a) wg_kajita_run_batch over the whole walks;
  (b) wg_kajita_stream: one append + run holding the whole walks (START | FINISH);
  (c) wg_kajita_stream: one step per walk per run, until every walk has finished.
Outputs stay on the device; each pass is timed with CUDA events on the context stream (host planning of the appends
included), and the three alternate pass by pass in one process.  Prints one JSON line (and writes it to --out).

    python tools/bench_kajita_stream.py [--walks 4096] [--reps 7] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import jrl_walkgen_b200 as wg  # noqa: E402
from jrl_walkgen_b200 import workloads as W  # noqa: E402


def card():
    """Name and power limit of GPU 0 (read only)."""
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        name, power, clock = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:       # the numbers still stand, the card is then unknown
        return {"name": f"unknown ({e})"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--walks", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    B = a.walks
    ctx = wg.Context(0)
    ctx.preview_set_gains(wg.preview_gains(0.005, 1.6, 0.814, wg.MODE_WITHOUT_INITIALPOS))
    off, steps, feet = W.kajita_steps_batch(B)
    lens = np.diff(off)
    plan = ctx.kajita_plan(off, steps, feet)
    n, total_steps = plan.total_samples, plan.total_steps
    d_state, d_com, d_zmp = ctx.alloc(B * 64), ctx.alloc(n * 48), ctx.alloc(n * 16)

    # (b): the whole walks in one append
    sb = ctx.kajita_stream(B)
    flags_b = np.full(B, wg.STREAM_START | wg.STREAM_FINISH, dtype=np.int32)
    # (c): run r appends step r of every walk that has one
    sc = ctx.kajita_stream(B)
    runs_c = []
    for r in range(int(lens.max())):
        has = (lens > r).astype(np.int64)
        o = np.concatenate([[0], np.cumsum(has)]).astype(np.int64)
        st = np.ascontiguousarray(steps[off[:-1][lens > r] + r])
        fl = np.where(has > 0, (wg.STREAM_START if r == 0 else 0) | np.where(lens - 1 == r, wg.STREAM_FINISH, 0), 0)
        runs_c.append((o, st, fl.astype(np.int32)))

    def pass_a():
        ctx.sync()
        ctx.timer_start()
        plan.run(d_state, d_com, d_zmp, mem=wg.WG_MEM_DEVICE)
        return ctx.timer_stop_ms(), 1, total_steps

    def pass_b():
        ctx.sync()
        ctx.timer_start()
        sb.append(off, steps, flags_b, feet)
        sb.run(com_out=d_com, zmp_out=d_zmp, mem=wg.WG_MEM_DEVICE)
        return ctx.timer_stop_ms(), 1, int(sb.com_counts.sum())

    def pass_c():
        ctx.sync()
        ctx.timer_start()
        k = 0
        for o, st, fl in runs_c:
            sc.append(o, st, fl, feet)
            assert sc.com_offsets[-1] <= n
            sc.run(com_out=d_com, zmp_out=d_zmp, mem=wg.WG_MEM_DEVICE)
            k += int(sc.com_counts.sum())
        return ctx.timer_stop_ms(), len(runs_c), k

    legs = {"a_run_batch": pass_a, "b_stream_whole": pass_b, "c_stream_one_step": pass_c}
    res = {k: {"ms": [], "launches": 0, "runs": 0, "steps": 0} for k in legs}
    for rep in range(a.reps + 1):                      # rep 0 warms every leg up
        for k, f in legs.items():
            l0 = ctx.launches
            ms, runs, k_steps = f()
            if rep == 0:
                continue
            res[k]["ms"].append(ms)
            res[k]["launches"] = (ctx.launches - l0) / runs
            res[k]["runs"] = runs
            res[k]["steps"] = k_steps
    # one profiled pass per leg (after the timed ones): device time of the front-end and preview kernels
    kern = {}
    for k, f in legs.items():
        ctx.sync()
        ctx.prof_begin(4 * len(runs_c) + 8)
        f()
        prof = ctx.prof_end()
        kern[k] = {"front_end_ms": round(prof[7][1], 4) if 7 in prof else None,
                   "preview_ms": round(prof[6][1], 4) if 6 in prof else None}
    out = {"workload": f"kajita_steps_batch({B})", "walks": B, "samples": int(n), "preview_steps": int(total_steps),
           "card": card(), "reps": a.reps}
    for k, r in res.items():
        assert r["steps"] == total_steps, (k, r["steps"], total_steps)
        med = float(np.median(r["ms"]))
        out[k] = {"ms_median": round(med, 4), "ms_min": round(min(r["ms"]), 4), "ms_max": round(max(r["ms"]), 4),
                  "preview_steps_per_s": round(total_steps / (med * 1e-3), 1), "runs_per_pass": r["runs"],
                  "ms_per_run": round(med / r["runs"], 4), "launches_per_run": r["launches"], "kernels_per_pass": kern[k]}
    out["b_over_a"] = round(out["b_stream_whole"]["ms_median"] / out["a_run_batch"]["ms_median"], 4)
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")
    for s in (sb, sc):
        s.destroy()
    plan.destroy()
    ctx.close()


if __name__ == "__main__":
    main()
