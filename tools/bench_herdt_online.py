"""The on-line Herdt2010 generator (wg_herdt_online_*) at B robots, device-resident, against the period API:
  aligned    every robot starts at tick 0, so all of them fire on the same tick (one tick in 20);
  staggered  robot b starts at tick b mod 20, so about B/20 fire on every tick;
  periods    wg_herdt_mpc_run_batch, one QP period (20 ticks of rows) per call, every instance firing.
Every tick applies a velocity command to every robot (WG_CMD_VEL, the robot's own reference) and writes the popped rows and
running flags to device buffers.  The three legs alternate pass by pass in one process; a pass is --ticks ticks (periods:
--ticks / 20 periods) timed with CUDA events on the context stream.  After the timed passes, single ticks are timed one by
one (events around each call) and then profiled per kernel, split into ticks on which robots fire and ticks on which none
does.  Prints one JSON line (and writes it to --out).

    python tools/bench_herdt_online.py [--batch 16384 1000000] [--ticks 2000] [--reps 2] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import jrl_walkgen_b200 as wg  # noqa: E402

CHUNK = 20    # ticks per wg_herdt_online_tick call in the timed passes


def card():
    """Name and power limit of GPU 0 (read only)."""
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        name, power, clock = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:       # the numbers still stand, the card is then unknown
        return {"name": f"unknown ({e})"}


class Bench:
    def __init__(self, ctx, B, seed=1):
        self.ctx, self.B = ctx, B
        rng = np.random.default_rng(seed)
        self.vel = np.column_stack([rng.uniform(0.0, 0.3, B), rng.uniform(-0.1, 0.1, B), rng.uniform(-0.2, 0.2, B)])
        cmd = np.zeros((CHUNK, B), dtype=wg.HERDT_COMMAND_DTYPE)
        cmd["vel"] = self.vel[None, :, :]
        cmd["flags"] = wg.CMD_VEL
        self.d_cmd = ctx.to_device(cmd)
        del cmd
        self.d_rows = ctx.alloc(CHUNK * B * wg.TICK_DTYPE.itemsize)
        self.d_run = ctx.alloc(CHUNK * B)
        self.d_stats = ctx.alloc(4 * 8)
        # the two on-line handles
        self.aligned = ctx.herdt_online(B)
        self.aligned.start(np.arange(B, dtype=np.int32))
        self.staggered = ctx.herdt_online(B)
        for t in range(20):
            self.staggered.start(np.arange(t, B, 20, dtype=np.int32))
            self.tick(self.staggered, 1)
        # the period API
        self.d_states = ctx.herdt_mpc_init(B, device=True)
        self.d_vel = ctx.to_device(self.vel)
        self.ctx.herdt_mpc_run_device(self.d_states, B, 1, d_vel_ref=self.d_vel)

    def tick(self, h, n):
        self.ctx._check(self.ctx.lib.wg_herdt_online_tick(h.h, wg.WG_MEM_DEVICE, int(n), C.c_void_p(self.d_cmd.ptr),
                                                          C.c_void_p(self.d_rows.ptr), C.c_void_p(self.d_run.ptr)))

    def qp_count(self, d_states_ptr):
        self.ctx._check(self.ctx.lib.wg_herdt_mpc_stats(self.ctx.h, self.B, C.c_void_p(d_states_ptr), C.c_void_p(self.d_stats.ptr)))
        return float(self.d_stats.download(np.float64, (4,))[0])

    def online_pass(self, h, nticks):
        q0 = self.qp_count(h.d_states)
        l0 = self.ctx.launches
        self.ctx.sync()
        self.ctx.timer_start()
        for _ in range(nticks // CHUNK):
            self.tick(h, CHUNK)
        ms = self.ctx.timer_stop_ms()
        return ms, self.ctx.launches - l0, self.qp_count(h.d_states) - q0

    def period_pass(self, nticks):
        q0 = self.qp_count(self.d_states.ptr)
        l0 = self.ctx.launches
        self.ctx.sync()
        self.ctx.timer_start()
        for _ in range(nticks // 20):
            self.ctx.herdt_mpc_run_device(self.d_states, self.B, 1, d_ticks=self.d_rows)
        ms = self.ctx.timer_stop_ms()
        return ms, self.ctx.launches - l0, self.qp_count(self.d_states.ptr) - q0

    def single_ticks(self, h, n):
        """n ticks, one call each: (ms, robots that fired) per tick, then the per-kernel device ms of the same kind of ticks."""
        out = []
        for _ in range(n):
            q0 = self.qp_count(h.d_states)
            self.ctx.sync()
            self.ctx.timer_start()
            self.tick(h, 1)
            ms = self.ctx.timer_stop_ms()
            out.append((ms, self.qp_count(h.d_states) - q0))
        prof = []
        for _ in range(n):
            q0 = self.qp_count(h.d_states)
            self.ctx.sync()
            self.ctx.prof_begin(16)
            self.tick(h, 1)
            p = self.ctx.prof_end()
            prof.append((p, self.qp_count(h.d_states) - q0))
        return out, prof

    def free(self):
        for h in (self.aligned, self.staggered):
            h.destroy()
        for d in (self.d_cmd, self.d_rows, self.d_run, self.d_stats, self.d_states, self.d_vel):
            d.free()


def summarize_ticks(samples, prof):
    res = {}
    for kind, sel in (("firing", lambda f: f > 0), ("non_firing", lambda f: f == 0)):
        ms = [m for m, f in samples if sel(f)]
        if not ms:
            continue
        ks = [p for p, f in prof if sel(f)]
        qp = [p[2][1] for p in ks if 2 in p]
        mpc = [p[3][1] for p in ks if 3 in p]
        res[kind] = {"ticks": len(ms), "ms_median": round(float(np.median(ms)), 4), "ms_min": round(min(ms), 4),
                     "robots_fired_median": float(np.median([f for _, f in samples if sel(f)])),
                     "qp_kernel_ms_median": round(float(np.median(qp)), 4) if qp else None,
                     "tick_post_merge_kernels_ms_median": round(float(np.median(mpc)), 4) if mpc else None}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, nargs="+", default=[16384, 1000000])
    ap.add_argument("--ticks", type=int, default=2000)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--single", type=int, default=40, help="ticks timed one by one per mode")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert a.ticks % CHUNK == 0
    ctx = wg.Context(0)
    ctx.herdt_set_params()
    ctx.herdt_mpc_set_params()
    out = {"card": card(), "ticks_per_pass": a.ticks, "reps": a.reps, "results": []}
    for B in a.batch:
        bench = Bench(ctx, B)
        legs = {"aligned": lambda: bench.online_pass(bench.aligned, a.ticks),
                "staggered": lambda: bench.online_pass(bench.staggered, a.ticks),
                "periods": lambda: bench.period_pass(a.ticks)}
        res = {k: {"ms": [], "launches": 0, "solves": 0.0} for k in legs}
        for rep in range(a.reps + 1):                  # rep 0 warms every leg up
            for k, f in legs.items():
                ms, launches, solves = f()
                if rep == 0:
                    continue
                res[k]["ms"].append(ms); res[k]["launches"] = launches; res[k]["solves"] = solves
        r = {"B": B}
        for k, v in res.items():
            med = float(np.median(v["ms"]))
            r[k] = {"ms_median": round(med, 3), "ms_min": round(min(v["ms"]), 3), "ms_max": round(max(v["ms"]), 3),
                    "robot_ticks_per_s": round(B * a.ticks / (med * 1e-3), 1),
                    "qp_solves_per_s": round(v["solves"] / (med * 1e-3), 1),
                    "launches_per_tick": v["launches"] / a.ticks, "qp_solves_per_pass": v["solves"]}
        for mode in ("aligned", "staggered"):
            samples, prof = bench.single_ticks(getattr(bench, mode), a.single)
            r[mode]["single_ticks"] = summarize_ticks(samples, prof)
        r["staggered_over_periods"] = round(r["staggered"]["ms_median"] / r["periods"]["ms_median"], 4)
        r["aligned_over_periods"] = round(r["aligned"]["ms_median"] / r["periods"]["ms_median"], 4)
        out["results"].append(r)
        print(json.dumps(r), flush=True)
        bench.free()
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
