"""Whole robots of the on-line Herdt2010 generator (wg_herdt_online_save / restore / copy), device-resident.

  records    at each --batch size B: one handle of B robots (staggered starts, so the rings hold different counts at
             different heads), a second handle of B robots and a device array of B records.  Device ms per call of
             copy (handle to handle), save and restore (its check kernel included), from per-kernel CUDA events over --reps
             calls with NULL index arrays; bytes moved from the shapes (a record is 8448 B, a robot in a handle 8440 B:
             ring 7424, state 1000, slot 16), GB/s and the fraction of 7.7 TB/s.  Whole-call ms separately: a host clock
             around one call with a permuted index array and the synchronise after it (host validation and index upload
             included).  Every working set is larger than the 126 MB L2 (two copies of B robots: 169 MB at 10^4).
  lookahead  --live robots (staggered starts), --branches K scratch robots each.  One decision: copy every live robot into
             its K branches (one call, source indices repeated), tick the branches 20 ticks, branch k of every robot under
             candidate velocity k on every tick (no rows kept), then tick the live robots 20 ticks (rows and running flags
             to device buffers).  ms per decision from events around --decisions decisions in a row; then each phase alone
             (events around it) for the copy's share and the cost of the 20 live ticks alone.
Every leg is run once before it is timed.  Prints one JSON line (and writes it to --out).

    python tools/bench_herdt_online_fork.py [--batch 10000 100000 1000000] [--reps 10] [--live 16384] [--branches 8]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import jrl_walkgen_b200 as wg  # noqa: E402
from bench_herdt_online import card  # noqa: E402

HBM_TBPS = 7.7          # HGX B200 data sheet, one GPU
REC = 8448              # sizeof(wg_herdt_online_robot)
ROBOT = 29 * 256 + 1000 + 16   # what a robot occupies in a handle: ring, state, slot
K_MPC = 3               # profiler id of the on-line kernels (WG_K_HERDT_MPC)


def staggered(ctx, B, vel=None):
    """A handle of B robots, robot b started at tick b mod 20, 20 ticks run: every robot running, rings at all phases."""
    h = ctx.herdt_online(B)
    for t in range(20):
        h.start(np.arange(t, B, 20, dtype=np.int32))
        h.tick_device(1)
    ctx.sync()
    return h


def device_ms(ctx, call, reps):
    """Per-call device ms of the library's kernels over reps calls (per-kernel events) -> (ms per call, launches per call)."""
    ctx.sync()
    ctx.prof_begin(4 * reps + 8)
    for _ in range(reps):
        call()
    p = ctx.prof_end()
    n, ms = p.get(K_MPC, (0, 0.0))
    return ms / reps, n / reps


def whole_ms(ctx, call, reps):
    out = []
    for _ in range(reps):
        ctx.sync()
        t0 = time.perf_counter()
        call()
        ctx.sync()
        out.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(out))


def records_leg(ctx, B, reps):
    lib = ctx.lib
    src = staggered(ctx, B)
    dst = ctx.herdt_online(B)
    d_rec = ctx.alloc(B * REC)
    perm = np.random.default_rng(B).permutation(B).astype(np.int32)
    pp = perm.ctypes.data
    calls = {
        "copy": (lambda: ctx._check(lib.wg_herdt_online_copy(dst.h, B, None, src.h, None)),
                 lambda: ctx._check(lib.wg_herdt_online_copy(dst.h, B, pp, src.h, pp)), 2 * ROBOT),
        "save": (lambda: src.save_device(B, d_rec),
                 lambda: ctx._check(lib.wg_herdt_online_save(src.h, wg.WG_MEM_DEVICE, B, pp, C.c_void_p(d_rec.ptr))),
                 REC + ROBOT),
        "restore": (lambda: dst.restore_device(B, d_rec),
                    lambda: ctx._check(lib.wg_herdt_online_restore(dst.h, wg.WG_MEM_DEVICE, B, pp, C.c_void_p(d_rec.ptr))),
                    REC + ROBOT),
    }
    res = {"B": B}
    for name, (plain, indexed, per_robot) in calls.items():
        plain(); indexed(); ctx.sync()                     # warm-up
        ms, launches = device_ms(ctx, plain, reps)
        nbytes = per_robot * B
        gbs = nbytes / (ms * 1e-3) / 1e9
        res[name] = {"device_ms": round(ms, 4), "launches_per_call": launches, "bytes": nbytes,
                     "GB_per_s": round(gbs, 1), "of_7_7_TBps": round(gbs / (HBM_TBPS * 1e3), 3),
                     "lower_bound_ms": round(nbytes / (HBM_TBPS * 1e12) * 1e3, 4),
                     "whole_call_ms_indexed": round(whole_ms(ctx, indexed, max(3, reps // 2)), 4)}
    # the records the legs moved mean what they should: dst now holds src's robots, bitwise
    n = min(B, 256)
    assert dst.save(np.arange(n)).tobytes() == src.save(np.arange(n)).tobytes()
    d_rec.free(); src.destroy(); dst.destroy()
    return res


def lookahead_leg(ctx, live_n, K, decisions):
    lib = ctx.lib
    nb = live_n * K
    live = staggered(ctx, live_n)
    br = ctx.herdt_online(nb)
    rng = np.random.default_rng(3)
    cand = np.column_stack([np.linspace(0.0, 0.3, K), np.zeros(K), np.linspace(-0.2, 0.2, K)])   # candidate (dx, dy, dyaw)
    bcmd = np.zeros((20, nb), dtype=wg.HERDT_COMMAND_DTYPE)
    bcmd["vel"] = np.tile(cand, (live_n, 1))[None, :, :]
    bcmd["flags"] = wg.CMD_VEL
    lcmd = np.zeros((20, live_n), dtype=wg.HERDT_COMMAND_DTYPE)
    lcmd["vel"] = np.column_stack([rng.uniform(0.0, 0.3, live_n), rng.uniform(-0.1, 0.1, live_n),
                                   rng.uniform(-0.2, 0.2, live_n)])[None, :, :]
    lcmd["flags"] = wg.CMD_VEL
    d_bcmd, d_lcmd = ctx.to_device(bcmd), ctx.to_device(lcmd)
    d_rows = ctx.alloc(20 * live_n * wg.TICK_DTYPE.itemsize)
    d_run = ctx.alloc(20 * live_n)
    src_idx = np.repeat(np.arange(live_n, dtype=np.int32), K)
    sp = src_idx.ctypes.data

    def copy():
        ctx._check(lib.wg_herdt_online_copy(br.h, nb, None, live.h, sp))

    def branches():
        br.tick_device(20, d_bcmd)

    def live_ticks():
        live.tick_device(20, d_lcmd, d_rows, d_run)

    def decision():
        copy(); branches(); live_ticks()

    for _ in range(2):
        decision()                                  # warm-up
    ctx.sync()
    ctx.timer_start()
    for _ in range(decisions):
        decision()
    per_decision = ctx.timer_stop_ms() / decisions
    phases = {}
    for name, f in (("copy", copy), ("branch_ticks", branches), ("live_ticks", live_ticks)):
        ms = []
        for _ in range(decisions):
            ctx.sync()
            ctx.timer_start()
            f()
            ms.append(ctx.timer_stop_ms())
        phases[name] = round(float(np.median(ms)), 4)
    copy_whole = whole_ms(ctx, copy, decisions)
    for d in (d_bcmd, d_lcmd, d_rows, d_run):
        d.free()
    live.destroy(); br.destroy()
    return {"live": live_n, "branches_per_robot": K, "branch_robots": nb, "decisions": decisions,
            "ms_per_decision": round(per_decision, 4), "phase_ms": phases,
            "copy_share_of_decision": round(phases["copy"] / per_decision, 4),
            "copy_whole_call_ms": round(copy_whole, 4), "copy_bytes": nb * 2 * ROBOT,
            "decision_over_live_ticks_alone": round(per_decision / phases["live_ticks"], 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, nargs="+", default=[10000, 100000, 1000000])
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--live", type=int, default=16384)
    ap.add_argument("--branches", type=int, default=8)
    ap.add_argument("--decisions", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    ctx = wg.Context(0)
    ctx.herdt_set_params()
    ctx.herdt_mpc_set_params()
    out = {"card": card(), "hbm_TBps_datasheet": HBM_TBPS, "records": [], "lookahead": None}
    for B in a.batch:
        r = records_leg(ctx, B, a.reps)
        out["records"].append(r)
        print(json.dumps(r), flush=True)
    out["lookahead"] = lookahead_leg(ctx, a.live, a.branches, a.decisions)
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
