"""Summarises the bench lines of scripts/x_ring_gpu.sh: `value` of each arm (default x ring against FI_B200_X_RING=2), the
C2..C4 Jacobi-PCG ms per iteration, and the --dump-outputs of the arms against each other and against a second m = 2 run.

    python scripts/x_ring_compare.py DIR [f64]"""
import glob
import json
import os
import sys
from statistics import median

import numpy as np

d = sys.argv[1]
tag = "_f64" if len(sys.argv) > 2 and sys.argv[2] == "f64" else ""


def line(path):
    try:
        with open(path) as fh:
            rows = [r for r in fh.read().splitlines() if r.startswith("{")]
        return json.loads(rows[-1])
    except (OSError, IndexError, ValueError):
        return None


arms = {}
for arm in ("m2", "default"):
    rows = [line(p) for p in sorted(glob.glob(os.path.join(d, f"x_ring_bench{tag}_{arm}_*.json")))]
    arms[arm] = [r for r in rows if r]
    vals = [r["value"] for r in arms[arm]]
    if not vals:
        print(arm, "no bench line")
        continue
    it = [r["kernels"]["iteration"]["ms_per_iteration"] for r in arms[arm] if r.get("kernels")]
    print(json.dumps({"arm": arm, "prec": tag[1:] or "f32", "values_G": [round(v / 1e9, 2) for v in vals], "median_G": round(median(vals) / 1e9, 2),
                      "spread_pct": round((max(vals) - min(vals)) / median(vals) * 100, 2),
                      "ms_per_iteration": [round(v, 4) for v in it],
                      "update_ms": [round(r["kernels"]["update_kernel"]["avg_launch_ms"], 4) for r in arms[arm] if r.get("kernels")]}))
    cfg = {}
    for r in arms[arm]:
        for c in ("C2_interpolate2d_512_10k", "C3_sdf2d_2048_200k", "C4_sdf3d_256_1M"):
            j = ((r.get("configs") or {}).get(c) or {}).get("jacobi_pcg")
            if j:
                cfg.setdefault(c, []).append(round(j["ms_per_iteration"], 5))
    if cfg:
        print(json.dumps({"arm": arm, "configs_ms_per_iteration": cfg}))
if arms.get("m2") and arms.get("default"):
    a, b = median(r["value"] for r in arms["m2"]), median(r["value"] for r in arms["default"])
    print(json.dumps({"prec": tag[1:] or "f32", "default_over_m2_pct": round((b / a - 1) * 100, 2)}))

if not tag:
    def load(k):
        p = os.path.join(d, k)
        if not os.path.isdir(p):
            return None
        return {f[:-4]: np.load(os.path.join(p, f)).astype(np.float64) for f in os.listdir(p) if f.endswith(".npy")}

    def rel(a, b):
        return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))

    ref = load("dump_m2_1")
    for k in ("dump_m2_2", "dump_m2_3", "dump_def_1", "dump_def_2", "dump_def_3"):
        o = load(k)
        if ref is None or o is None:
            continue
        print(json.dumps({"vs": "dump_m2_1", "run": k, "iterations": [float(ref["iterations"]), float(o["iterations"])],
                          "field_rel_l2": rel(o["field"], ref["field"]), "field_max_abs": float(np.abs(o["field"] - ref["field"]).max()),
                          "relative_residual": [float(ref["relative_residual"]), float(o["relative_residual"])]}))
