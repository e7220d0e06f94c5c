"""Spread that sets the smoother and cycle tolerances of tests/test_gpu_multigrid_operator.py: on every case of that file,
the relative L2 difference of the library's fp32 SMOOTH (every smoothed level, from zero and from a given e) and CYCLE
(every cycle configuration of the file) from the fp64 restatement of tests/mg_reference.py, the same inputs the tests
use; plus lmax / lambda_max per level and the lambda(BA) range of the cycles on the lattices where B is formed.  One
JSON line per (case, check), then one summary line."""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import scipy.linalg as sla  # noqa: E402

import field_interpolation_b200 as fi  # noqa: E402
import mg_reference as R  # noqa: E402
import test_gpu_multigrid_operator as T  # noqa: E402
from field_interpolation_b200 import _lib as L  # noqa: E402
from oracle import oracle as O  # noqa: E402


class Env:  # the tests' monkeypatch, for a script
    def setenv(self, k, v):
        os.environ[k] = v

    def delenv(self, k, raising=False):
        os.environ.pop(k, None)


port, env = O.port(), Env()
worst = {"smooth": 0.0, "cycle": 0.0}
for name in T.CASES:
    prob, f, info, H = T.field_and_reference(fi, port, name, env)
    rng = np.random.default_rng(5)  # test_smoother's inputs
    for l in range(info["levels"] - 1):
        n = H.A[l].shape[0]
        r, e = rng.normal(size=(2, n)), rng.normal(size=(2, n))
        z0 = f.mg_stage(L.FI_MG_SMOOTH, l, r, None, options=T.mg_opts(fi))
        z1 = f.mg_stage(L.FI_MG_SMOOTH, l, r, e, options=T.mg_opts(fi))
        d = max(max(T.rel(z0[k], H.smooth(l, r[k])), T.rel(z1[k], H.smooth(l, r[k], e[k]))) for k in range(2))
        lam = T.lambda_max(H.A[l])
        print(json.dumps({"case": name, "check": "smooth", "level": l, "rel_l2": d, "lmax_over_lambda_max": info["lmax"][l] / lam}), flush=True)
        worst["smooth"] = max(worst["smooth"], d)
    for cycle in T.CYCLES:
        prob, f, info, H = T.field_and_reference(fi, port, name, env, cycle)
        r = np.random.default_rng(6).normal(size=(3, prob.n))  # test_cycle_matches_reference's inputs
        z = f.mg_stage(L.FI_MG_CYCLE, 0, r, options=T.mg_opts(fi))
        d = max(T.rel(z[k], H.cycle(r[k])) for k in range(3))
        line = {"case": name, "check": "cycle", "cycle": cycle, "levels": info["levels"], "rel_l2": d}
        if name in T.EXPLICIT and cycle in ("V", "W3"):
            B = f.mg_stage(L.FI_MG_CYCLE, 0, np.eye(prob.n), options=T.mg_opts(fi)).astype(np.float64).T
            C = np.linalg.cholesky(H.A[0].toarray())
            lam = sla.eigvalsh(C.T @ (0.5 * (B + B.T)) @ C)
            line.update(lambda_BA_min=float(lam.min()), lambda_BA_max=float(lam.max()), asym=float(np.abs(B - B.T).max() / np.abs(B).max()))
        print(json.dumps(line), flush=True)
        worst["cycle"] = max(worst["cycle"], d)
for k in T.MG_ENV:
    os.environ.pop(k, None)
print(json.dumps({"summary": "worst relative L2 against fp64", **worst}), flush=True)
