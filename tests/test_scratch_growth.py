"""Host-buffer entry points stage their batches in device scratch that a context keeps and grows with the batch size.
A call with a larger batch after a smaller one on the same context must give bitwise what the same call gives on a fresh
context: the grown buffers are reallocated and, where the entry relies on it, cleared as on first use."""
import numpy as np
import pytest

from jrl_walkgen_b200 import workloads as W

SMALL = 37
LARGE = 9000        # > 2 x 4096: the host-buffer Herdt QP pipelines it in two chunks


def two_contexts():
    import jrl_walkgen_b200 as wg
    return wg.Context(0), wg.Context(0)


def velocity_refs(B, seed):
    rng = np.random.default_rng(seed)
    return np.column_stack([rng.uniform(-0.2, 0.3, B), rng.uniform(-0.15, 0.15, B), rng.uniform(-0.2, 0.2, B)])


@pytest.mark.gpu
def test_gpu_herdt_qp_host_batch_grown_on_one_context_equals_fresh_context(ctx):
    ctx.herdt_set_params()
    ctx.herdt_mpc_set_params()
    st = ctx.herdt_mpc_init(LARGE)
    _, _, qin = ctx.herdt_mpc_run(st, 12, vel_ref=velocity_refs(LARGE, 1), qp_in=True)
    grown, fresh = two_contexts()
    try:
        grown.herdt_set_params(); fresh.herdt_set_params()
        grown.herdt_qp_solve(qin[:SMALL])
        a = grown.herdt_qp_solve(qin)
        b = fresh.herdt_qp_solve(qin)
        assert (a["fail"] == 0).all()
        assert a.tobytes() == b.tobytes()
        # the warm-start entry shares the input / output staging and grows its own active-set buffer
        grown.herdt_qp_solve_warm(qin[:SMALL])
        a, a_act = grown.herdt_qp_solve_warm(qin[:2 * SMALL])
        b, b_act = fresh.herdt_qp_solve_warm(qin[:2 * SMALL])
        assert a.tobytes() == b.tobytes() and a_act.tobytes() == b_act.tobytes()
    finally:
        grown.close(); fresh.close()


@pytest.mark.gpu
def test_gpu_herdt_mpc_host_batch_grown_on_one_context_equals_fresh_context():
    grown, fresh = two_contexts()
    try:
        for c in (grown, fresh):
            c.herdt_set_params()
            c.herdt_mpc_set_params()
        v = velocity_refs(LARGE, 2)
        st0 = grown.herdt_mpc_init(LARGE)
        small = st0[:SMALL].copy()
        grown.herdt_mpc_run(small, 5, vel_ref=v[:SMALL], ticks=True, steps=True, qp_in=True)
        a = st0.copy()
        ta, sa, qa = grown.herdt_mpc_run(a, 20, vel_ref=v, ticks=True, steps=True, qp_in=True)
        b = st0.copy()
        tb, sb, qb = fresh.herdt_mpc_run(b, 20, vel_ref=v, ticks=True, steps=True, qp_in=True)
        assert (a["qp_count"] == 20).all()
        assert a.tobytes() == b.tobytes()
        assert ta.tobytes() == tb.tobytes() and sa.tobytes() == sb.tobytes() and qa.tobytes() == qb.tobytes()
    finally:
        grown.close(); fresh.close()


@pytest.mark.gpu
def test_gpu_pldp_host_batch_grown_on_one_context_equals_fresh_context():
    import jrl_walkgen_b200 as wg
    K = W.DimitrovConstants()
    _, base = W.pldp_batch(1024, seed=41, K=K)
    reps = 5                                       # 5120 problems: two pipelined chunks
    pb = {k: (np.tile(v, (reps,) + (1,) * (v.ndim - 1)) if isinstance(v, np.ndarray) else v) for k, v in base.items()}
    B = 1024 * reps
    small = {k: (v[:SMALL] if isinstance(v, np.ndarray) else v) for k, v in pb.items()}
    grown, fresh = two_contexts()
    try:
        for c in (grown, fresh):
            c.pldp_set_constants(K.iPu, K.Px, K.Pu)
        grown.pldp_solve(small, hot=np.zeros(SMALL, dtype=wg.PLDP_STATE_DTYPE), starting=np.ones(SMALL, np.int32))
        hot_a = np.zeros(B, dtype=wg.PLDP_STATE_DTYPE)
        Xa, ia = grown.pldp_solve(pb, hot=hot_a, starting=np.ones(B, np.int32))
        hot_b = np.zeros(B, dtype=wg.PLDP_STATE_DTYPE)
        Xb, ib = fresh.pldp_solve(pb, hot=hot_b, starting=np.ones(B, np.int32))
        assert (ia["rc"] == 0).all()
        assert Xa.tobytes() == Xb.tobytes() and ia.tobytes() == ib.tobytes() and hot_a.tobytes() == hot_b.tobytes()
    finally:
        grown.close(); fresh.close()
