"""Times the exact nearest-point search (fi_nearest_point_distance) and the border-distance builder
(fi_field_add_border_distance) on the device.

  builder     fi_field_add_border_distance at 256^3 and 512^3 with the bench cloud (1M sphere-and-torus points), a fresh
              field per call, from host and from device positions.  Split with public calls on device arrays:
              build = fi_nearest_point_distance with one query (copy-free structure build); search = the same call
              with the border nodes' coordinates as queries, minus build; append = the device-position builder call
              minus both (distance copy to the host and the host append of the rows).
  queries     fi_nearest_point_distance against the same 1M cloud at 512^3: 1M and 16M uniform queries in the lattice,
              and the marching-cubes vertices of the solved 512^3 field (near-surface queries); distances and indices,
              device-resident, every call building its structure.
  brute       the tests' chunked torch brute force (tests/nearest_port.py) on 65 536 queries of each set on the same
              device, scaled linearly to the set's size (its cost is exactly linear in the number of queries).
  host loop   the caller's loop (one thread, C++ -O2 without FMA contraction, compiled into a temporary directory) on
              every border node of 128^3 with 100k points: one run.  Its distances are checked against the device's.
  solve       time to a 1e-6 true residual at 512^3 of sdf_from_points with and without border rows, one solve each:
              MG-PCG (fp32) without rows and with rows of weight 0.5, 0.05 and 0.005 (caller rows cost the multigrid its
              fused finest-level step, and the coarse levels do not see them), and Jacobi-PCG (fp64) without rows and
              with rows of weight 0.5.

Every time is the median of 10 calls after 2 warm-up calls, each call ending in a device synchronise (host clock),
except the brute force (median of 3), the host loop and the solves (one run each).  --parts picks a subset of
builder, queries, hostloop, solve.  The card's name and power limit are read in the
same run.  Usage: time_nearest_points.py [--out FILE] [--parts LIST] (appends)"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

HOST_LOOP = r"""
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <limits>
extern "C" void border_loop(int64_t nq, const float* q, int64_t n, const float* p, float* out)
{
	for (int64_t j = 0; j < nq; ++j) {
		float closest = std::numeric_limits<float>::infinity();
		for (int64_t i = 0; i < n; ++i) {
			const float dx = p[3 * i] - q[3 * j], dy = p[3 * i + 1] - q[3 * j + 1], dz = p[3 * i + 2] - q[3 * j + 2];
			closest = std::min(closest, dx * dx + dy * dy + dz * dz);
		}
		out[j] = std::sqrt(closest);
	}
}
"""


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (r.stdout.strip().splitlines()[0].split(", ") + ["?"])[:2] if r.returncode == 0 else ("?", "?")
    return {"gpu": name, "power_limit": power}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--parts", default="builder,queries,hostloop,solve", help="comma-separated subset of the cases to run")
    args = ap.parse_args()
    parts = set(args.parts.split(","))
    import torch
    import field_interpolation_b200 as fi
    import nearest_port as P
    from field_interpolation_b200 import _lib as L
    from field_interpolation_b200 import workloads as W
    if not torch.cuda.is_available():
        raise SystemExit("time_nearest_points.py needs a CUDA device")
    info = card()
    dll = L.lib()
    lines = []

    def timed(fn, reps=10, warm=2, setup=None):
        ts = []
        for r in range(warm + reps):
            arg = setup() if setup else None
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn(arg)
            torch.cuda.synchronize()
            if r >= warm:
                ts.append((time.perf_counter() - t0) * 1e3)
        return float(np.median(ts))

    def emit(line):
        line.update(info)
        lines.append(line)
        print(json.dumps(line), flush=True)

    def nearest(dp, dq, want_index=True):
        d = torch.empty(dq.shape[0], dtype=torch.float32, device="cuda")
        k = torch.empty(dq.shape[0], dtype=torch.int64, device="cuda") if want_index else None
        st = dll.fi_nearest_point_distance(3, dp.shape[0], C.c_void_p(dp.data_ptr()), dq.shape[0], C.c_void_p(dq.data_ptr()), L.FI_DEVICE,
                                           C.c_void_p(d.data_ptr()), C.c_void_p(k.data_ptr()) if want_index else None)
        assert st == L.FI_OK
        return d, k

    def brute_ms(dp, qs):
        pick = qs[torch.randperm(qs.shape[0], generator=torch.Generator().manual_seed(0))[:65536].cuda()].contiguous()
        return timed(lambda _: P.torch_nearest(dp, pick), reps=3, warm=1), pick.shape[0]

    cloud = W.sphere_torus_3d(1_000_000, seed=0)

    # ---- the builder at 256^3 and 512^3 ----
    if "builder" in parts:
        for n in (256, 512):
            sizes = [n, n, n]
            pos = W.to_lattice(cloud["unit_pos"], sizes)
            dp = torch.from_numpy(pos).cuda()
            nodes, q = P.border_nodes(sizes)
            dq = torch.from_numpy(q).cuda()
            fresh = lambda: fi.LatticeField(sizes)  # noqa: E731
            ms_host = timed(lambda f: fi.add_border_distance_constraints(f, 0.5, pos), setup=fresh)
            ms_dev = timed(lambda f: fi.add_border_distance_constraints(f, 0.5, dp), setup=fresh)
            ms_build = timed(lambda _: nearest(dp, dq[:1], False))
            ms_build_search = timed(lambda _: nearest(dp, dq, False))
            line = {"what": "fi_field_add_border_distance", "n": n, "points": len(pos), "border_nodes": int(nodes.size), "ms_host_positions": ms_host,
                    "ms_device_positions": ms_dev, "ms_build": ms_build, "ms_search": ms_build_search - ms_build,
                    "ms_copy_and_append": ms_dev - ms_build_search, "target_ms_512": 50.0}
            if n == 512:
                bms, bq = brute_ms(dp, dq)
                line.update({"torch_brute_ms_65536": bms, "torch_brute_ms_scaled": bms * nodes.size / bq,
                             "search_speedup_vs_brute": bms * nodes.size / bq / (ms_build_search - ms_build),
                             "call_speedup_vs_brute": bms * nodes.size / bq / ms_build_search})
            emit(line)
            del dq
            torch.cuda.empty_cache()

    # ---- arbitrary queries at 512^3 ----
    if "queries" in parts:
        n = 512
        sizes = [n, n, n]
        pos = W.to_lattice(cloud["unit_pos"], sizes)
        dp = torch.from_numpy(pos).cuda()
        g = torch.Generator(device="cuda").manual_seed(0)
        f = fi.sdf_from_points(sizes, fi.Weights(), pos, cloud["normals"])
        out = torch.zeros(n ** 3, dtype=torch.float32, device="cuda")
        _, st0 = f.solve(fi.solve_options(fi.FI_F32, 300, 1e-6, preconditioner=fi.FI_PRECOND_MULTIGRID), out=out)
        verts, _ = fi.marching_cubes(out.view(n, n, n), 0.0)
        sets = {"uniform_1M": torch.rand((1_000_000, 3), generator=g, device="cuda") * (n - 1),
                "uniform_16M": torch.rand((16_000_000, 3), generator=g, device="cuda") * (n - 1),
                "mc_vertices_512": verts.contiguous()}
        ms_build = timed(lambda _: nearest(dp, sets["uniform_1M"][:1]))
        for name, qs in sets.items():
            ms = timed(lambda _: nearest(dp, qs))
            bms, bq = brute_ms(dp, qs)
            d, _ = nearest(dp, qs)
            emit({"what": "fi_nearest_point_distance", "n": n, "points": len(pos), "queries": name, "num_queries": qs.shape[0], "ms_call": ms,
                  "ms_build": ms_build, "ms_search": ms - ms_build, "queries_per_s": qs.shape[0] / (ms - ms_build) * 1e3,
                  "torch_brute_ms_65536": bms, "torch_brute_ms_scaled": bms * qs.shape[0] / bq,
                  "search_speedup_vs_brute": bms * qs.shape[0] / bq / (ms - ms_build), "call_speedup_vs_brute": bms * qs.shape[0] / bq / ms,
                  "median_distance": float(d.median()), "max_distance": float(d.max())})
        del sets, verts, f
        torch.cuda.empty_cache()

    # ---- the caller's host loop at 128^3, 100k points ----
    if "hostloop" in parts:
        n = 128
        sizes = [n, n, n]
        pos = np.ascontiguousarray(W.to_lattice(W.sphere_torus_3d(100_000, seed=0)["unit_pos"], sizes), np.float32)
        nodes, q = P.border_nodes(sizes)
        with tempfile.TemporaryDirectory() as tmp:
            src, so = os.path.join(tmp, "loop.cpp"), os.path.join(tmp, "loop.so")
            open(src, "w").write(HOST_LOOP)
            subprocess.run([os.environ.get("CXX", "g++"), "-O2", "-ffp-contract=off", "-shared", "-fPIC", src, "-o", so], check=True)
            lib = C.CDLL(so)
            host = np.empty(nodes.size, np.float32)
            t0 = time.perf_counter()
            lib.border_loop(C.c_int64(nodes.size), q.ctypes.data_as(C.c_void_p), C.c_int64(len(pos)), pos.ctypes.data_as(C.c_void_p),
                            host.ctypes.data_as(C.c_void_p))
            ms_loop = (time.perf_counter() - t0) * 1e3
        fresh = lambda: fi.LatticeField(sizes)  # noqa: E731
        ms_call = timed(lambda f: fi.add_border_distance_constraints(f, 1.0, pos), setup=fresh)
        fl = fi.LatticeField(sizes)
        fi.add_border_distance_constraints(fl, 1.0, pos)
        same = bool(np.array_equal(fl.eq.rhs.view(np.uint32), host.view(np.uint32)))
        emit({"what": "caller host loop vs fi_field_add_border_distance", "n": n, "points": len(pos), "border_nodes": int(nodes.size),
              "evaluations": int(nodes.size) * len(pos), "ms_host_loop_one_thread": ms_loop, "ms_call_host_positions": ms_call,
              "speedup": ms_loop / ms_call, "bit_identical": same})

    # ---- time to 1e-6 at 512^3 with and without border rows ----
    if "solve" in parts:
        n = 512
        sizes = [n, n, n]
        pos = W.to_lattice(cloud["unit_pos"], sizes)
        # MG-PCG without and with border rows (weights 0.5, 0.05, 0.005: whether the stall follows the rows' strength),
        # Jacobi-PCG in fp64 with and without them (the solver that sees the rows through its diagonal)
        cases = [("multigrid", fi.FI_F32, fi.FI_PRECOND_MULTIGRID, 500, None), ("multigrid", fi.FI_F32, fi.FI_PRECOND_MULTIGRID, 500, 0.5),
                 ("multigrid", fi.FI_F32, fi.FI_PRECOND_MULTIGRID, 500, 0.05), ("multigrid", fi.FI_F32, fi.FI_PRECOND_MULTIGRID, 500, 0.005),
                 ("jacobi_f64", fi.FI_F64, fi.FI_PRECOND_JACOBI, 60000, None), ("jacobi_f64", fi.FI_F64, fi.FI_PRECOND_JACOBI, 60000, 0.5)]
        for name, prec, pre, iters, weight in cases:
            f = fi.sdf_from_points(sizes, fi.Weights(), pos, cloud["normals"])
            if weight is not None:
                fi.add_border_distance_constraints(f, weight, pos)
            opt = fi.solve_options(prec, iters, 1e-6, preconditioner=pre)
            out = torch.zeros(n ** 3, dtype=torch.float32, device="cuda")
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            _, st = f.solve(opt, out=out)
            torch.cuda.synchronize()
            ms = (time.perf_counter() - t0) * 1e3
            emit({"what": "PCG time to 1e-6, one solve", "solver": name, "n": n, "points": len(pos), "border_rows_weight": weight,
                  "max_iterations": iters, "ms_solve_with_setup": ms, "iterations": st["iterations"], "true_residual": st["true_residual"],
                  "converged": st["converged"], "setup_ms": st["setup_ms"], "solve_ms": st["solve_ms"], "generic_rows": st["generic_rows"]})
            del f, out
            torch.cuda.empty_cache()

    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as h:
            for line in lines:
                h.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
