"""Whole walks of the on-line Kajita generator one tick at a time (wg_kajita_online_save / restore / copy), device-resident,
NL = 320, max_step_time = 0.8 s (ring of 1922 rows, 430 KB per walk).

  records    --batch walks (7 GB of rings at 16 384) started with three steps of workloads.kajita_steps_batch and advanced
             --advance ticks, so their queues hold what a walk holds mid-walk; a second handle and device arrays of the
             records, carries and queues.  Device ms per call of save, restore and copy (handle to handle) from per-kernel
             CUDA events over --reps calls with NULL index arrays, with a 256 MB fill between calls that leaves nothing of
             the working set in the 126 MB L2.  The byte lower bound comes from R and the walks' actual queued counts: save
             reads the queued rows and the stream part and writes whole queues (R rows), records and carries; restore reads
             records, carries and queued rows and writes the stream part and queued rows; copy reads and writes the stream
             part and the queued rows.  GB/s and the fraction of 7.7 TB/s.
  lookahead  --live walks advanced as above, --branches K branch walks each in a second handle.  One decision: copy every
             live walk into its K branches (one call, source indices repeated), push one candidate step per branch, tick the
             branches 2 NL + one segment (800 ticks, device outputs off) so that the candidate's rows are popped, then push
             the chosen step to the live walks and tick them once.  ms per decision from events around --decisions
             decisions; the copy alone for its share.
Every leg runs once before it is timed.  Prints one JSON line with the card's name and power limit (and writes it to --out).

    python tools/bench_kajita_online_fork.py [--batch 16384] [--reps 5] [--live 4096] [--branches 4]
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
from jrl_walkgen_b200 import workloads as W  # noqa: E402
from bench_kajita_stream import card  # noqa: E402

HBM_TBPS = 7.7                 # HGX B200 data sheet, one GPU
REC, CARRY, ROW = 624, 319 * 16, 224
WALK = 496 + 64 + CARRY        # the stream part of a walk on the device: state record, preview state, carry
K_ZD = 7                       # profiler id of the zmpdisc kernels (WG_K_ZMPDISC)
BASE = W.kajita_steps_batch(4096)


def started(ctx, B, advance):
    off, steps, feet = BASE
    h = ctx.kajita_online(B)
    first = np.arange(B) % 4096
    for c0 in range(0, B, 4096):
        idx = np.arange(c0, min(B, c0 + 4096))
        h.start(idx, [steps[off[first[b]]:off[first[b]] + 3] for b in idx], feet[first[idx]])
    for t in range(0, advance, 160):
        h.tick_device(min(160, advance - t))
    ctx.sync()
    return h


def device_ms(ctx, call, reps, flush):
    ctx.sync()
    ctx.prof_begin(4 * reps + 8)
    for _ in range(reps):
        flush()
        call()
    p = ctx.prof_end()
    n, ms = p.get(K_ZD, (0, 0.0))
    return ms / reps, n / reps


def records_leg(ctx, B, reps, advance, scrub):
    src = started(ctx, B, advance)
    dst = ctx.kajita_online(B)
    R = src.ring_rows
    d_w, d_c, d_q = ctx.alloc(B * REC), ctx.alloc(B * CARRY), ctx.alloc(B * R * ROW)
    stacks = {}

    def flush():
        ctx.lib.wg_memset_device(ctx.h, scrub.ptr, 0, scrub.nbytes)

    def save():
        stacks["s"] = src.save_device(B, d_w, d_c, d_q)

    q = int(src.state()[0].sum())
    calls = {
        "save": (save, B * (WALK + 24 + 64 + REC + CARRY + R * ROW) + q * ROW),
        "restore": (lambda: dst.restore_device(B, d_w, d_c, d_q, stacks["s"]), B * (REC + CARRY + WALK) + 2 * q * ROW),
        "copy": (lambda: dst.copy_from(src), B * 2 * WALK + 2 * q * ROW),
    }
    res = {"B": B, "ring_rows": R, "ring_GB": round(B * R * ROW / 1e9, 2), "queued_rows_mean": round(q / B, 1)}
    for name, (f, nbytes) in calls.items():
        f(); ctx.sync()
        ms, launches = device_ms(ctx, f, reps, flush)
        gbs = nbytes / (ms * 1e-3) / 1e9
        res[name] = {"device_ms_l2_flushed": round(ms, 4), "launches_per_call": launches, "bytes": nbytes,
                     "GB_per_s": round(gbs, 1), "of_7_7_TBps": round(gbs / (HBM_TBPS * 1e3), 3),
                     "lower_bound_ms": round(nbytes / (HBM_TBPS * 1e12) * 1e3, 4)}
    n = min(B, 64)
    a, b = dst.save(np.arange(n)), src.save(np.arange(n))
    assert all(x.tobytes() == y.tobytes() for x, y in zip(a[:3], b[:3]))
    d_w.free(); d_c.free(); d_q.free(); src.destroy(); dst.destroy()
    return res


def lookahead_leg(ctx, live_n, K, decisions, advance):
    nb = live_n * K
    NL = ctx.gains.NL
    live = started(ctx, live_n, advance)
    br = ctx.kajita_online(nb)
    cand = np.zeros(K, dtype=wg.KAJITA_COMMAND_DTYPE)
    cand["flags"] = wg.KAJITA_PUSH
    cand["step"]["sx"] = np.linspace(0.05, 0.25, K)
    cand["step"]["theta"] = np.linspace(-10.0, 10.0, K)
    cand["step"]["ss_time"], cand["step"]["ds_time"], cand["step"]["step_type"] = 0.78, 0.02, 1
    src_idx = np.repeat(np.arange(live_n, dtype=np.int32), K)
    side = {"s": 1.0}
    horizon = 2 * NL + 160

    def copy():
        br.copy_from(live, src_idx=src_idx)

    def decision():
        copy()
        c = np.tile(cand, nb // K).reshape(1, nb)
        c["step"]["sy"] = side["s"] * 0.19
        br.tick_device(1, c)
        for t in range(1, horizon, 160):
            br.tick_device(min(160, horizon - t))
        lc = np.repeat(cand[:1], live_n).reshape(1, live_n)
        lc["step"]["sy"] = side["s"] * 0.19
        live.tick_device(1, lc)
        side["s"] = -side["s"]

    for _ in range(2):
        decision()
    ctx.sync()
    ctx.timer_start()
    for _ in range(decisions):
        decision()
    per_decision = ctx.timer_stop_ms() / decisions
    cm = []
    for _ in range(decisions):
        ctx.sync()
        ctx.timer_start()
        copy()
        cm.append(ctx.timer_stop_ms())
    copy_ms = float(np.median(cm))
    assert br.state()[2].all() and live.state()[2].all()
    live.destroy(); br.destroy()
    return {"live": live_n, "branches_per_walk": K, "branch_walks": nb, "ticks_per_branch": horizon, "decisions": decisions,
            "ms_per_decision": round(per_decision, 3), "copy_ms": round(copy_ms, 4),
            "copy_share_of_decision": round(copy_ms / per_decision, 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, nargs="+", default=[16384])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--advance", type=int, default=400)
    ap.add_argument("--live", type=int, default=4096)
    ap.add_argument("--branches", type=int, default=4)
    ap.add_argument("--decisions", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    ctx = wg.Context(0)
    ctx.preview_set_gains(wg.preview_gains(0.005, 1.6, 0.814, wg.MODE_WITHOUT_INITIALPOS))
    assert ctx.gains.NL == 320
    scrub = ctx.alloc(256 << 20)
    out = {"card": card(), "records": [records_leg(ctx, B, a.reps, a.advance, scrub) for B in a.batch],
           "lookahead": lookahead_leg(ctx, a.live, a.branches, a.decisions, a.advance)}
    scrub.free()
    ctx.close()
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
