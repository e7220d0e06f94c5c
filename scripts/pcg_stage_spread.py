"""Worst error / bound ratio of every per-entry bound of tests/test_gpu_pcg_stages.py, per stage and case, with the inputs
and bounds the tests use.  A ratio above 1 is a bug or a wrong bound; one far below 1e-3 a bound too loose to catch
anything.  One JSON line per (case, precision, stage), then one summary line with the worst and best ratio per check.
    python scripts/pcg_stage_spread.py [--emu]"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
if "--emu" in sys.argv:
    os.environ["FI_B200_TEST_EMU"] = "1"
    import conftest  # noqa: E402
    conftest.use_emulated_library()

import field_interpolation_b200 as fi  # noqa: E402
import test_gpu_pcg_stages as T  # noqa: E402

F32, F64 = T.F32, T.F64
summary = {}


def emit(name, prec, stage, ratios, report=None):
    line = {"case": name, "precision": "fp32" if prec == F32 else "fp64", "stage": stage, "ratios": ratios}
    if report is not None:
        line["report"] = report
    print(json.dumps(line), flush=True)
    for k, v in ratios.items():
        lo, hi = summary.get(k, (v, v))
        summary[k] = (min(lo, v), max(hi, v))


for name, (kw, precs) in T.STENCIL_CASES.items():
    c = T.case(fi, name, **kw)
    for prec in precs:
        for iters, par in [(0, 0), (3, 0), (4, 1)]:
            emit(name, prec, f"stencil it{iters} par{par}", T.run_stencil(fi, c, prec, 1, par, iters, seed=iters), list(T.expected_stencil(c, prec, 1)))
        if c.D == 3:
            emit(name, prec, "stencil tiled", T.run_stencil(fi, c, prec, 2, 1, 5, seed=7), list(T.expected_stencil(c, prec, 2)))
for name, kw in T.DATA_CASES.items():
    c = T.case(fi, "data_" + name, **kw)
    for prec in (F32, F64):
        emit(name, prec, "data", T.run_data(fi, c, prec))
c = T.case(fi, "update", **T.UPDATE_CASE)
for prec in (F32, F64):
    for m in (2, 4, 8):
        for pos in range(m):
            emit("update", prec, f"update m{m} pos{pos}", T.run_update(fi, c, prec, m, pos))
        for count in range(1, m):
            emit("update", prec, f"pending flush m{m} count{count}", T.run_flush(fi, c, prec, m, count))
for name, kw in [("1d", T.sc([257], [dict(model_1=0.2)], npts=100)), ("3d_x33", T.sc([33, 9, 8], [dict()], npts=150))]:
    c = T.case(fi, "unfused_" + name, **kw)
    for prec in (F32, F64):
        for par in (0, 1):
            emit(name, prec, f"unfused par{par}", T.run_unfused(fi, c, prec, par))
if not T.EMU:
    import numpy as np  # noqa: F401
    from field_interpolation_b200 import workloads as W
    sizes = [512, 512, 512]
    cloud = W.sphere_torus_3d(1_000_000, seed=0)
    c = T.case(fi, "full_512", sizes=sizes, models=[dict()], cloud=(W.to_lattice(cloud["unit_pos"], sizes), cloud["normals"]))
    emit("full_512", F32, "stencil", T.run_stencil(fi, c, F32, 1, 1, 3, device=True), list(T.expected_stencil(c, F32, 1)))
    emit("full_512", F32, "data", T.run_data(fi, c, F32))
    emit("full_512", F32, "update m2 pos1", T.run_update(fi, c, F32, 2, 1))
print(json.dumps({"summary": {k: {"worst": hi, "best": lo} for k, (lo, hi) in sorted(summary.items())}}), flush=True)
