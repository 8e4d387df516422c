"""Write tests/golden/pldp_ref.npz: what the reference's PLDPSolver.cpp / OptCholesky.cpp object code returns on the
seeded inputs of tests/test_pldp_oracle.py, so that those tests compare against stored vectors.

The reference's sources are not part of this repository.  The vectors are computed by the oracle port
(oracle/oracle_pldp.cpp), which the same tests held BITWISE equal to the reference's object code on exactly these
inputs (X, L and the return code) while that object code was built beside it; a vector that differs from the
reference's in any bit would have failed them.
    python tests/golden/make_pldp_ref.py            (after `make -C oracle liboracle.so`)
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))

import pldp_oracle as po                       # noqa: E402
from jrl_walkgen_b200 import workloads as W    # noqa: E402

HOT_SEQS, HOT_T = 4, 25


def optcholesky():
    """L after adding 10 rows, for the two (mode, nb, cu) cases of test_oracle_optcholesky_equals_reference_object_code."""
    rng = np.random.default_rng(1)
    out = {}
    for mode, nb, cu in ((0, 12, 15), (1, 20, 32)):
        A = rng.uniform(0.0, 1.0, size=(nb, cu)) if mode == 0 else rng.uniform(-1.0, 1.0, size=(cu, nb + 1))
        A = np.ascontiguousarray(A)
        rows = rng.permutation(nb)[:10].astype(np.int32)
        L = np.zeros((nb, nb))
        po.lib().oracle_optcholesky_add_rows(mode, nb, cu, nb, A.ctypes.data, rows.ctypes.data, 0, 10, L.ctypes.data)
        out["optchol_L%d" % mode] = L
    return out


def pldp_cold_and_hot():
    """X of 20 cold solves of pldp_batch(40, seed=3), and X of the hot-started sequences, NaN after a sequence ends."""
    K, pb = W.pldp_batch(40, seed=3)
    cold = np.stack([po.oracle_solve(K, pb, b, hot=None, starting=True)[0] for b in range(20)])
    hot = np.full((HOT_SEQS, HOT_T, 32), np.nan)
    for seq in range(HOT_SEQS):
        rng = np.random.default_rng([9, seq])
        polys = W._support_polygons(rng, K.N, K.T, count=K.N + 25)
        xk = np.zeros(6); xk[0], xk[3] = polys[0][0]
        state = np.zeros(1, dtype=po.STATE)
        n_removed = 0
        for t in range(HOT_T):
            p = W.pldp_problem_from(K, polys[t:t + K.N], xk)
            X, info, _ = po.oracle_solve(K, W.pldp_pack(K, [p]), 0, hot=state, starting=(t == 0), n_removed=n_removed)
            if info[1] == 2:
                break
            hot[seq, t] = X
            n_removed = p["n_first"]
            xk = W.pldp_advance(K, xk, X)
    return {"cold_X": cold, "hot_X": hot}


def pldp_similar():
    """X with consistent SimilarConstraints flags, and X / return code with the seeded inconsistent ones (NaN and -1
    where the solve is not clean: the reference would exit(0) there)."""
    K, pb = W.pldp_batch(24, seed=11)
    ok = np.zeros((24, 32)); bad = np.full((24, 32), np.nan); bad_rc = np.full(24, -1, dtype=np.int32)
    for b in range(24):
        m = int(pb["m"][b])
        ok[b] = po.oracle_solve(K, pb, b, starting=True, similar=np.ascontiguousarray(pb["similar"][b]))[0]
        rng = np.random.default_rng([11, b])
        sim_bad = np.zeros(128, dtype=np.int32)
        for li in range(1, m):
            if rng.random() < 0.3:
                sim_bad[li] = -int(rng.integers(1, min(li, 5) + 1))
        X2, i2, _ = po.oracle_solve(K, pb, b, starting=True, similar=sim_bad)
        if i2[1] == 0:
            bad[b], bad_rc[b] = X2, i2[0]
    return {"similar_X": ok, "similar_bad_X": bad, "similar_bad_rc": bad_rc}


def main():
    out = dict(**optcholesky(), **pldp_cold_and_hot(), **pldp_similar())
    np.savez_compressed(os.path.join(HERE, "pldp_ref.npz"), **out)
    print("written pldp_ref.npz:", {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main()
