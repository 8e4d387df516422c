"""The one-warp recursive preview kernel (CTA shape 2) writes a walk's CoM rows from row o on, 48 bytes each, so where its
tiles fall against 128-byte lines depends on o mod 8; whole tiles and a walk's last, partial tile take different store
paths.  These tests run walks at every o mod 8, with step counts just under and just over 128 and 256 ticks, into an
output array with guard rows on both sides, and check:
  * the rows are bitwise the pinned ones (SHA-256 of the rows): a change of the store path must not change a bit;
  * no guard row, and no row past a walk's last step, is written.
"""
import ctypes as C
import hashlib

import numpy as np
import pytest

NL = 320
GUARD = 37                      # guard rows before and after the output (odd: the array itself starts at 48 * 37 bytes)
SENTINEL = np.float64(-1234.5)
# step counts: just under / over 128 and 256 ticks, then one and several whole tiles plus a partial one
BASE_STEPS = (120, 129, 248, 257, 512, 1100)

# SHA-256 of the output rows (all walks' rows, guards excluded), measured on a B200 with the one-warp kernel that stages each
# lane's CoM rows for one cp.async.bulk per lane and tile.
PINNED_SHA = {
    "sim": "63a5d77296ef80e336448c203a0df2cff25eab2452f2eefb63e5993bf8d1574d",
    "nosim": "706bb72cc9f3fc5fb155029ebdb4b1cf271e38d308fa4741da17c0305e61e5ed",
    "stage2": "d429fd345a666f6a0aff8db60744c38316de53d467ad76b3f0d2b032f0cd6b67",
}


def walk_offsets():
    """24 walks; walk i starts at a row with o mod 8 == i mod 8, each step count a base of BASE_STEPS plus 0..7."""
    lens, o = [], 0
    for i in range(24):
        base = BASE_STEPS[i % len(BASE_STEPS)]
        L = base + NL - 1
        L += ((i + 1) % 8 - (o + L)) % 8        # next walk starts at residue (i + 1) mod 8
        lens.append(L)
        o += L
    return np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)


def inputs(offsets):
    rng = np.random.default_rng(7)
    n = int(offsets[-1])
    z = np.cumsum(rng.normal(scale=2e-3, size=(n, 2)), axis=0)
    st = rng.normal(scale=1e-2, size=(len(offsets) - 1, 8))
    com1 = rng.normal(scale=1e-1, size=(n, 6))
    return z, st, com1


def run_guarded(ctx, kind, shape=2):
    """Run one batch (kind: 'sim', 'nosim' or 'stage2') from device buffers into an output with GUARD rows on both sides;
    return (offsets, the whole guarded output array)."""
    import jrl_walkgen_b200 as wg
    gains = wg.preview_gains(0.005, 1.6, 0.814, wg.MODE_WITHOUT_INITIALPOS)
    ctx.preview_set_gains(gains)
    ctx.preview_set_cta_shape(shape)
    offsets = walk_offsets()
    n = int(offsets[-1])
    z, st, com1 = inputs(offsets)
    plan = ctx.preview_plan(offsets)
    out = np.full((GUARD + n + GUARD, 6), SENTINEL)
    bufs = [ctx.to_device(a) for a in (z, st, com1, out)]
    dz, ds, dc1, do = bufs
    rows = C.c_void_p(do.ptr + 48 * GUARD)
    try:
        if kind == "stage2":
            rc = ctx.lib.wg_preview_stage2_run_batch(ctx.h, plan.h, wg.WG_MEM_DEVICE, C.c_void_p(dz.ptr), C.c_void_p(dc1.ptr),
                                                     C.c_void_p(ds.ptr), rows, None)
        else:
            rc = ctx.lib.wg_preview_run_batch(ctx.h, plan.h, wg.WG_MEM_DEVICE, C.c_void_p(dz.ptr), C.c_void_p(ds.ptr), rows,
                                              None, int(kind == "sim"))
        assert rc == 0, ctx.lib.wg_last_error(ctx.h)
        ctx.sync()
        return offsets, do.download(np.float64, out.shape)
    finally:
        for b in bufs:
            b.free()
        plan.destroy()
        ctx.preview_set_cta_shape(-1)


def digests(ctx):
    return {k: hashlib.sha256(run_guarded(ctx, k)[1][GUARD:-GUARD].tobytes()).hexdigest() for k in PINNED_SHA}


def test_walks_cover_every_row_alignment():
    offsets = walk_offsets()
    assert sorted(set(int(o) % 8 for o in offsets[:-1])) == list(range(8))
    steps = np.diff(offsets) - NL + 1
    for lo, hi in ((120, 127), (129, 136), (248, 255), (257, 264)):
        assert ((steps >= lo) & (steps <= hi)).any()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["sim", "nosim", "stage2"])
def test_rec_warp_rows_bitwise_and_guards_untouched(ctx, kind):
    offsets, out = run_guarded(ctx, kind)
    assert (out[:GUARD] == SENTINEL).all() and (out[-GUARD:] == SENTINEL).all()
    rows = out[GUARD:-GUARD]
    for b in range(len(offsets) - 1):
        o, L = int(offsets[b]), int(offsets[b + 1] - offsets[b])
        ns = L - NL + 1
        assert not (rows[o:o + ns] == SENTINEL).any(), b
        assert (rows[o + ns:o + L] == SENTINEL).all(), b        # rows past the last step stay as they were
    assert hashlib.sha256(rows.tobytes()).hexdigest() == PINNED_SHA[kind]

