"""CUDA-event times of the fused Jacobi-PCG iteration for every x ring (FI_B200_X_RING=2|4|8) on the bench cloud
(sphere + torus, 1M points): the update kernel in its skip form, in its flush form, in the mix the solve runs (m-1 skip
launches and one flush per m iterations), the stencil kernel and the whole iteration, per launch.  One JSON line per
(lattice, precision, m).

    python scripts/time_x_ring.py [--sizes 512,1024] [--iters 200]

1024^3 runs in fp32 only (one fp64 vector is 8.6 GB)."""
import argparse
import json
import os
import sys
from statistics import median

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import field_interpolation_b200 as fi
from field_interpolation_b200 import workloads as W

RINGS = (2, 4, 8)


def per_launch(f, opt, iters):
    f.time_iterations(20, opt)
    t = f.time_iterations(iters, opt)
    return {k: v / iters for k, v in t.items() if k.endswith("_ms")}, t["x_ring"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="512,1024")
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--points", type=int, default=1_000_000)
    args = ap.parse_args()
    cloud = W.sphere_torus_3d(args.points, seed=0)
    up = torch.from_numpy(cloud["unit_pos"]).cuda()
    nr = torch.from_numpy(cloud["normals"]).cuda()
    gpu = torch.cuda.get_device_name(0)
    for n in (int(s) for s in args.sizes.split(",")):
        f = fi.sdf_from_points([n] * 3, fi.Weights(), up * (n - 1.0), nr)
        for prec, name, B in ((fi.FI_F32, "f32", 4), (fi.FI_F64, "f64", 8)):
            if n > 512 and name == "f64":
                continue
            cells = n ** 3
            for m in RINGS:
                os.environ["FI_B200_X_RING"] = str(m)
                opt = fi.solve_options(prec, 0, 1e-6)
                mix, ran = per_launch(f, opt, args.iters)
                # the forms alone, from calls of m-1 iterations (skip launches only) and of m (one ring: the skip launches and
                # the flush); median of 11 calls each, since one call times only a few launches
                skip = median(f.time_iterations(m - 1, opt)["update_ms"] / (m - 1) for _ in range(11))
                flush = median(f.time_iterations(m, opt)["update_ms"] for _ in range(11)) - (m - 1) * skip
                upd_bytes = (20 + 8 / m) * B / 4
                print(json.dumps({
                    "gpu": gpu, "n": n, "points": args.points, "prec": name, "x_ring": ran,
                    "iteration_ms": round(mix["iteration_ms"], 4), "update_ms": round(mix["update_ms"], 4),
                    "update_skip_ms": round(skip, 4), "update_flush_ms": round(flush, 4),
                    "stencil_ms": round(mix["stencil_ms"], 4), "data_term_ms": round(mix["data_term_ms"], 4),
                    "update_model_bytes_per_cell": upd_bytes,
                    "update_GBs_model": round(upd_bytes * cells / (mix["update_ms"] * 1e-3) / 1e9, 1),
                    "Gcell_iters_per_s": round(cells / (mix["iteration_ms"] * 1e-3) / 1e9, 2)}), flush=True)
        del f
        torch.cuda.empty_cache()
    os.environ.pop("FI_B200_X_RING", None)


if __name__ == "__main__":
    main()
