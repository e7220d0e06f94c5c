"""Spread that sets the tolerances of tests/test_gpu_x_ring.py: on the lattices of that test, relative L2 difference of x
between two m = 2 solves (the data term's atomics make runs differ) and between m = 4 / 8 and m = 2, for every iteration
count the test uses.  One JSON line per (lattice, precision, iteration count), then one summary line per precision."""
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import field_interpolation_b200 as fi
from test_gpu_x_ring import ITERS, lattice_2d, lattice_3d, rel


def solve(f, ring, P, its):
    os.environ["FI_B200_X_RING"] = str(ring)
    x, s = f.solve(fi.solve_options(P, its, 1e-30, check_every=8))
    return np.asarray(x, np.float64), s["iterations"]


worst = {}
for lname, make in (("3d", lattice_3d), ("2d", lattice_2d)):
    f = make(fi)
    for prec, P in (("f32", fi.FI_F32), ("f64", fi.FI_F64)):
        for its in ITERS:
            a, ia = solve(f, 2, P, its)
            b, ib = solve(f, 2, P, its)
            line = {"lattice": lname, "prec": prec, "iters": its, "m2_vs_m2": rel(a, b)}
            for ring in (4, 8):
                c, ic = solve(f, ring, P, its)
                line[f"m{ring}_vs_m2"] = rel(c, a)
                line[f"m{ring}_iterations_equal"] = ic == ia == ib == its
            print(json.dumps(line), flush=True)
            w = worst.setdefault(prec, {"spread_m2_vs_m2": 0.0, "max_m4_m8_vs_m2": 0.0})
            w["spread_m2_vs_m2"] = max(w["spread_m2_vs_m2"], line["m2_vs_m2"])
            w["max_m4_m8_vs_m2"] = max(w["max_m4_m8_vs_m2"], line["m4_vs_m2"], line["m8_vs_m2"])
os.environ.pop("FI_B200_X_RING", None)
for prec, w in worst.items():
    print(json.dumps({"summary": prec, **w}), flush=True)
