"""Write tests/golden/preview_ref.npz: what the reference's PreviewControl::OneIterationOfPreview object code returns,
with the product's gains, on the seeded inputs of test_gpu_preview_vs_reference_object and
test_gpu_one_iteration_vs_reference_object (tests/test_preview_ref.py), so that those tests compare against stored
vectors.  Walks are sampled at SAMPLE fixed, seeded rows each (first and last included); final states are stored whole.

The reference's sources are not part of this repository.  The vectors are computed by the oracle's restatement
(oracle/oracle_preview.cpp), which test_oracle_recursion_is_bitwise_the_reference held BITWISE equal to the
reference's object code, given the same gains, while that object code was built beside it.
    python tests/golden/make_preview_ref.py         (after build(): the gains come from the product's host solve)
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))

import jrl_walkgen_b200 as wg                  # noqa: E402
import oracle_lib as ol                        # noqa: E402
import test_preview_ref as tp                  # noqa: E402

SAMPLE = 96
T, TP, ZC = 0.005, 1.6, 0.807709


def product_gains():
    """The product's Kx / Ks / F with the oracle's A / B / C for (T, zc): what RefPreview.set_gains hands the reference."""
    g = wg.preview_gains(T, TP, ZC, 1)
    o = ol.OracleGains(T, TP, ZC, 1)
    o.Kx = np.array(g.Kx[:]); o.Ks = g.Ks; o.F = np.array(g.F[:g.NL]); o.NL = g.NL
    return o


def run(o, z, st, simulation):
    st = st.copy()
    com, zmp, steps = ol.oracle_preview_batch(o, [0, len(z)], z, st, simulation)
    return com[:steps], zmp[:steps], st


def main():
    o = product_gains()
    walks, st0 = tp.gpu_preview_inputs()
    out = {}
    for simulation in (True, False):
        tag = "sim" if simulation else "nosim"
        rows, com, zmp, state = [], [], [], []
        for b, w in enumerate(walks):
            c, zm, st = run(o, w, st0[b], simulation)
            r = tp.sample_rows(len(c), b, SAMPLE)
            rows.append(r); com.append(c[r][:, [0, 3]]); zmp.append(zm[r]); state.append(st[:6])
        out["%s_rows" % tag] = np.stack(rows); out["%s_com_x_y" % tag] = np.stack(com)
        out["%s_zmp" % tag] = np.stack(zmp); out["%s_state" % tag] = np.stack(state)
    z = tp.straight_walking_zmpref()[600:600 + 320 + 200]
    c, zm, _ = run(o, z, np.zeros(8), True)
    out["one_iteration_com"], out["one_iteration_zmp"] = c[:200], zm[:200]
    np.savez_compressed(os.path.join(HERE, "preview_ref.npz"), **out)
    print("written preview_ref.npz:", {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main()
