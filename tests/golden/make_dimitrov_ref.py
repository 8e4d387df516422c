"""Write tests/golden/dimitrov_ref.npz: what the reference's ConvexHull.cpp, FootConstraintsAsLinearSystem.cpp and
PLDPSolver.cpp object code returns on the seeded inputs of three tests in tests/test_dimitrov.py (the convex hulls of 400 stored point sets, the
support polygons of the four TestKajita2003 profiles, and the PLDP solutions of the first 17 periods of the straight
walk), so that those tests compare against stored vectors.

The reference's sources are not part of this repository.  The vectors are computed by the oracle's restatements
(oracle/oracle_dimitrov.cpp, oracle/oracle_pldp.cpp), which the same tests held BITWISE equal to the reference's object
code on exactly these inputs while that object code was built beside it.
    python tests/golden/make_dimitrov_ref.py        (after `make -C oracle liboracle.so`)
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))

import dimitrov_oracle as do                   # noqa: E402
import pldp_oracle as po                       # noqa: E402
import zmpdisc_oracle as zo                    # noqa: E402

LCI_FIELDS = ("rows", "similar", "A", "B", "center", "t_start", "t_end")   # what the reference's builder reports
PROFILES = ("StraightWalking", "Circle", "PbFlorentSeq1", "PbFlorentSeq2")


def feet_of(name):
    o = zo.run(zo.default_params(), zo.profile_steps(name))
    return o["left"], o["right"], o["types"][:, 1].copy()


def hull_trials():
    """400 seeded point sets: two feet with the same or different headings, random points, and points with exact ties."""
    rng = np.random.default_rng(7)
    trials = []
    for trial in range(400):
        kind = trial % 4
        if kind == 0:      # two feet, same heading (collinear corners: 4 or 6 vertices)
            th = rng.uniform(-0.5, 0.5) if trial % 8 else 0.0
            feet = [(rng.uniform(-0.2, 0.2), 0.095, th), (rng.uniform(-0.2, 0.2), -0.095, th)]
        elif kind == 1:    # two feet, different headings (up to 8 vertices)
            feet = [(rng.uniform(-0.2, 0.2), 0.095, rng.uniform(-0.6, 0.6)), (rng.uniform(-0.2, 0.2), -0.095, rng.uniform(-0.6, 0.6))]
        else:
            feet = None
        if feet:
            pts = []
            for (x, y, th) in feet:
                c, s = np.cos(th), np.sin(th)
                for lx, ly in ((1, -1), (1, 1), (-1, 1), (-1, -1)):
                    pts.append((x + lx * 0.085 * c - ly * 0.03 * s, y + lx * 0.085 * s + ly * 0.03 * c))
            pts = np.array(pts)
        else:
            pts = rng.uniform(-1, 1, (rng.integers(3, 9), 2))
            if kind == 3:
                pts = np.round(pts * 4) / 4      # many exact ties and collinear triples
                if len(np.unique(pts, axis=0)) < 3:
                    continue
        trials.append(pts)
    return trials


def hulls():
    """The point sets of test_oracle_convex_hull_equals_reference_object_code (stored: their trigonometry runs through
    numpy, whose last bits depend on the CPU) and the vertices of their hulls, NaN-padded."""
    trials = hull_trials()
    pts = np.full((len(trials), 8, 2), np.nan)
    npts = np.zeros(len(trials), dtype=np.int32)
    out = np.full((len(trials), 16, 2), np.nan)
    count = np.zeros(len(trials), dtype=np.int32)
    for k, p in enumerate(trials):
        h = do.hull(p)
        pts[k, :len(p)], npts[k] = p, len(p)
        out[k, :len(h)], count[k] = h, len(h)
    return {"hull_points": pts, "hull_npts": npts, "hull": out, "hull_count": count}


def polygons():
    out = {}
    for name in PROFILES:
        left, right, lt = feet_of(name)
        P = do.fcals(left, right, lt)
        for f in LCI_FIELDS:
            out["fcals_%s_%s" % (name, f)] = P[f]
    return out


def straight_walk_solutions():
    """X of the 17 hot-started PLDP solves before the straight walk's stop, solver memory carried period to period."""
    left, right, lt = feet_of("StraightWalking")
    par = do.default_params()
    per = do.run(left, right, lt, par)["periods"]
    K = do.Constants(par)
    P = do.fcals(left, right, lt, par)
    state = np.zeros(1, dtype=po.STATE)
    X = np.zeros((17, 32))
    removed, st = 0, 0.0
    for li in range(17):
        pb = do.build_constraints(K, P, st, per["xk"][li].copy())
        packed = {"m": np.array([pb["m"]]), "DPu": pb["DPu"][None], "DPx": pb["DPx"][None], "D": pb["D"][None],
                  "ZMPRef": pb["ZMPRef"][None], "XkYk": pb["XkYk"][None]}
        X[li], info, _ = po.oracle_solve(K, packed, 0, hot=state, starting=(li == 0), n_removed=removed)
        assert info[0] == 0 and info[1] == 0, (li, info)
        removed = pb["n_first"]
        st += par.T
    return {"loop_X": X}


def main():
    out = dict(**hulls(), **polygons(), **straight_walk_solutions())
    np.savez_compressed(os.path.join(HERE, "dimitrov_ref.npz"), **out)
    print("written dimitrov_ref.npz:", len(out), "arrays")


if __name__ == "__main__":
    main()
