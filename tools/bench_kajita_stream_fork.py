"""Whole walks of the on-line Kajita generator (wg_kajita_stream_save / restore / copy), device-resident, NL = 320.

  records    at each --batch size B: one stream of B started walks (walk b is walk b mod 4096 of workloads.kajita_steps_batch
             after its support-foot step and two more: the lead-in and two segments emitted, the carry full), a second stream
             of B walks and device arrays of B records and B carries.  Device ms per call of copy (stream to stream), save and
             restore (its check kernel included), from per-kernel CUDA events over --reps calls with NULL index arrays, once
             back to back and once with a 256 MB fill between calls, which leaves nothing of the working set in the 126 MB L2
             (at 4096 walks the back-to-back working set, 46 MB, is L2-resident).  Bytes moved from the shapes, read plus
             written: a record is 576 B and a carry 5104 B (5680 B per walk); a walk in a stream is its 496-B state record,
             its 64-B preview state and its carry (5664 B); save also reads 24 B of host counters per walk.  GB/s and the
             fraction of 7.7 TB/s.  Whole-call ms separately: a host clock around one call with a permuted index array and
             the synchronise after it (host checks, staging and, for the device restore, the read-back of the check).
  lookahead  --live walks of kajita_steps_batch started and advanced three steps, --branches K branch walks each in a
             second stream.  One decision: copy every live walk into its K branches (one call, source indices repeated),
             append one candidate step to every branch (K step lengths and yaws), run the branches with device outputs,
             append the chosen step to the live walks, run them.  ms per decision from events around --decisions decisions
             in a row; then each phase alone (events around it) for the copy's share.
Every leg is run once before it is timed.  Prints one JSON line with the card's name and power limit (and writes it to --out).

    python tools/bench_kajita_stream_fork.py [--batch 4096 65536 262144] [--reps 10] [--live 4096] [--branches 4]
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
from jrl_walkgen_b200 import workloads as W  # noqa: E402
from bench_kajita_stream import card  # noqa: E402

HBM_TBPS = 7.7                 # HGX B200 data sheet, one GPU
L2_BYTES = 126 << 20
REC, CARRY = 576, 319 * 16     # sizeof(wg_kajita_stream_walk), one walk's carry at NL = 320
WALK = 496 + 64 + CARRY        # what a walk occupies in a stream: state record, preview state, carry
K_ZD = 7                       # profiler id of the zmpdisc kernels (WG_K_ZMPDISC)
CHUNK = 32768                  # walks started per run when a stream is filled
BASE = W.kajita_steps_batch(4096)


def started(ctx, B, nsteps=3):
    """A stream of B walks, walk b = walk b mod 4096 of kajita_steps_batch started with its first nsteps steps."""
    off, steps, feet = BASE
    s = ctx.kajita_stream(B)
    first = np.arange(B) % 4096
    for c0 in range(0, B, CHUNK):
        c1 = min(B, c0 + CHUNK)
        n = np.zeros(B, dtype=np.int64)
        n[c0:c1] = nsteps
        o = np.concatenate([[0], np.cumsum(n)]).astype(np.int64)
        st = steps[(off[first[c0:c1]][:, None] + np.arange(nsteps)).reshape(-1)]
        fl = np.where(n > 0, wg.STREAM_START, 0).astype(np.int32)
        s.append(o, st, fl, feet[first])
        out = {k: ctx.alloc(max(16, int(s.sample_offsets[-1] if k == "zmpref_xy" else s.com_offsets[-1]) * w))
               for k, w in (("zmpref_xy", 16), ("com_out", 48), ("zmp_out", 16))}
        s.run(**out, mem=wg.WG_MEM_DEVICE)
        ctx.sync()
        for b in out.values():
            b.free()
    return s


def device_ms(ctx, call, reps, flush=None):
    """Per-call device ms of the zmpdisc kernels over reps calls (per-kernel events) -> (ms per call, launches per call)."""
    ctx.sync()
    ctx.prof_begin(4 * reps + 8)
    for _ in range(reps):
        if flush:
            flush()
        call()
    p = ctx.prof_end()
    n, ms = p.get(K_ZD, (0, 0.0))
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


def records_leg(ctx, B, reps, scrub):
    lib = ctx.lib
    src = started(ctx, B)
    dst = ctx.kajita_stream(B)
    d_w, d_c = ctx.alloc(B * REC), ctx.alloc(B * CARRY)
    wp, cp = C.c_void_p(d_w.ptr), C.c_void_p(d_c.ptr)
    perm = np.random.default_rng(B).permutation(B).astype(np.int32)
    pp = perm.ctypes.data
    D = wg.WG_MEM_DEVICE

    def flush():
        lib.wg_memset_device(ctx.h, scrub.ptr, 0, scrub.nbytes)

    calls = {
        "copy": (lambda: dst.copy_from(src),
                 lambda: ctx._check(lib.wg_kajita_stream_copy(dst.h, B, pp, src.h, pp)), 2 * WALK),
        "save": (lambda: src.save_device(B, d_w, d_c),
                 lambda: ctx._check(lib.wg_kajita_stream_save(src.h, D, B, pp, wp, cp)), WALK + 24 + REC + CARRY),
        "restore": (lambda: dst.restore_device(B, d_w, d_c),
                    lambda: ctx._check(lib.wg_kajita_stream_restore(dst.h, D, B, pp, wp, cp)), REC + CARRY + WALK),
    }
    res = {"B": B, "working_set_MB": round(2 * WALK * B / 1e6, 1), "back_to_back_fits_L2": 2 * WALK * B < L2_BYTES}
    for name, (plain, indexed, per_walk) in calls.items():
        plain(); indexed(); ctx.sync()                     # warm-up
        ms, launches = device_ms(ctx, plain, reps)
        ms_cold, _ = device_ms(ctx, plain, reps, flush)
        nbytes = per_walk * B
        gbs = nbytes / (ms_cold * 1e-3) / 1e9
        res[name] = {"device_ms": round(ms, 4), "device_ms_l2_flushed": round(ms_cold, 4), "launches_per_call": launches,
                     "bytes": nbytes, "GB_per_s_l2_flushed": round(gbs, 1), "of_7_7_TBps": round(gbs / (HBM_TBPS * 1e3), 3),
                     "lower_bound_ms": round(nbytes / (HBM_TBPS * 1e12) * 1e3, 4),
                     "whole_call_ms_indexed": round(whole_ms(ctx, indexed, max(3, reps // 2)), 4)}
    # the records the legs moved mean what they should: dst holds src's walks, bitwise
    n = min(B, 256)
    a, b = dst.save(np.arange(n)), src.save(np.arange(n))
    assert a[0].tobytes() == b[0].tobytes() and a[1].tobytes() == b[1].tobytes()
    d_w.free(); d_c.free(); src.destroy(); dst.destroy()
    return res


def lookahead_leg(ctx, live_n, K, decisions):
    nb = live_n * K
    live = started(ctx, live_n)
    br = ctx.kajita_stream(nb)
    off, steps, _ = BASE
    last_sy = steps["sy"][off[np.arange(live_n) % 4096] + 2]
    cand = np.zeros(K, dtype=wg.REL_STEP_DTYPE)
    cand["sx"] = np.linspace(0.05, 0.25, K)
    cand["theta"] = np.linspace(-10.0, 10.0, K)
    cand["ss_time"], cand["ds_time"], cand["step_type"] = 0.78, 0.02, 1

    def steps_for(sign):
        """(branch steps [nb], live steps [live_n]) when the walks' next step goes to side `sign` (per live walk)."""
        b = np.tile(cand, live_n)
        b["sy"] = np.repeat(sign * 0.2, K)
        l = np.repeat(cand[:1], live_n)
        l["sy"] = sign * 0.2
        return b, l

    sides = [steps_for(-np.sign(last_sy)), steps_for(np.sign(last_sy))]      # the side alternates from one step to the next
    src_idx = np.repeat(np.arange(live_n, dtype=np.int32), K)
    ob, ol = np.arange(nb + 1, dtype=np.int64), np.arange(live_n + 1, dtype=np.int64)
    rows = 319 + 160                                                          # carry + one step, per walk and run
    bout = {k: ctx.alloc(nb * rows * w) for k, w in (("zmpref_xy", 16), ("com_out", 48), ("zmp_out", 16))}
    lout = {k: ctx.alloc(live_n * rows * w) for k, w in (("zmpref_xy", 16), ("com_out", 48), ("zmp_out", 16))}
    state = {"i": 0}

    def copy():
        br.copy_from(live, src_idx=src_idx)

    def branches():
        br.append(ob, sides[state["i"] % 2][0])
        br.run(**bout, mem=wg.WG_MEM_DEVICE)

    def live_step():
        live.append(ol, sides[state["i"] % 2][1])
        live.run(**lout, mem=wg.WG_MEM_DEVICE)
        state["i"] += 1

    def decision():
        copy(); branches(); live_step()

    for _ in range(2):
        decision()                                  # warm-up
    ctx.sync()
    ctx.timer_start()
    for _ in range(decisions):
        decision()
    per_decision = ctx.timer_stop_ms() / decisions
    phases = {n: [] for n in ("copy", "branch_append_run", "live_append_run")}
    for _ in range(decisions):
        for name, f in (("copy", copy), ("branch_append_run", branches), ("live_append_run", live_step)):
            ctx.sync()
            ctx.timer_start()
            f()
            phases[name].append(ctx.timer_stop_ms())
    phases = {k: round(float(np.median(v)), 4) for k, v in phases.items()}
    copy_whole = whole_ms(ctx, copy, decisions)
    assert int(br.com_counts.sum()) > 0 and int(live.com_counts.sum()) > 0
    for d in list(bout.values()) + list(lout.values()):
        d.free()
    live.destroy(); br.destroy()
    return {"live": live_n, "branches_per_walk": K, "branch_walks": nb, "decisions": decisions,
            "ms_per_decision": round(per_decision, 4), "phase_ms": phases,
            "copy_share_of_decision": round(phases["copy"] / per_decision, 4),
            "copy_whole_call_ms": round(copy_whole, 4), "copy_bytes": nb * 2 * WALK}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, nargs="+", default=[4096, 65536, 262144])
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--live", type=int, default=4096)
    ap.add_argument("--branches", type=int, default=4)
    ap.add_argument("--decisions", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    ctx = wg.Context(0)
    ctx.preview_set_gains(wg.preview_gains(0.005, 1.6, 0.814, wg.MODE_WITHOUT_INITIALPOS))
    scrub = ctx.alloc(256 << 20)
    out = {"card": card(), "hbm_TBps_datasheet": HBM_TBPS, "records": [], "lookahead": None}
    for B in a.batch:
        r = records_leg(ctx, B, a.reps, scrub)
        out["records"].append(r)
        print(json.dumps(r), file=sys.stderr, flush=True)
    out["lookahead"] = lookahead_leg(ctx, a.live, a.branches, a.decisions)
    scrub.free()
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
