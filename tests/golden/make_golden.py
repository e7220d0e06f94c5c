"""Generates tests/golden/*.npz from the REFERENCE ITSELF (oracle/_ref/libfi_ref.so = the reference's
field_interpolation.cpp compiled unmodified, see oracle/Makefile).  Run in the build container, where
/root/reference exists:   python tests/golden/make_golden.py
The fixtures travel to the GPU box (which has no /root/reference); tests compare the CPU port and the
CUDA path against them.  Solutions are fp64 direct solves (scipy) of the normal equations of the
reference-assembled rows — the stand-in for solve_sparse_linear_exact (Eigen is not available).

vs_ref.npz holds what the reference returns on the inputs of tests/test_oracle_vs_ref.py.

    python tests/golden/make_golden.py --vs-ref-from-port

writes only vs_ref.npz, from the port instead of the reference.  The committed vs_ref.npz was written that way,
because the reference's source tree is not part of the repository.  The port, its build flags and the input
generators are unchanged since commit 4f549c6, where test_oracle_vs_ref ran green against the reference on exactly
these inputs, and test_oracle_golden still holds the port bit for bit to the fixtures the reference wrote.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import oracle as O  # noqa: E402
from field_interpolation_b200 import workloads as W  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
WKEYS = ["data_pos", "data_gradient", "model_0", "model_1", "model_2", "model_3", "model_4", "gradient_smoothness",
         "value_kernel", "gradient_kernel"]


def wdict(w):
    return np.array([getattr(w, k) for k in WKEYS], dtype=np.float64)


def save(name, sys_, n, **extra):
    sol = O.exact_solve(sys_, n) if extra.pop("solve", True) else np.zeros(0)
    np.savez_compressed(os.path.join(OUT, name), rows=sys_.rows, cols=sys_.cols, vals=sys_.vals, rhs=sys_.rhs,
                        solution=sol, **extra)
    print(f"{name}: {sys_.num_rows} rows, {sys_.num_triplets} triplets")


def vs_ref(lib):
    """tests/golden/vs_ref.npz: what `lib` returns on the inputs of tests/test_oracle_vs_ref.py."""
    sys.path.insert(0, os.path.dirname(OUT))
    import test_oracle_vs_ref as T
    out = {}
    for sizes in T.SDF_SIZES:
        for vk in (0, 1):
            for gk in (0, 1, 2):
                out.update(T.sdf_from_points_outputs(lib, sizes, vk, gk))
    for make in (T.single_point_builder_outputs, T.upscale_and_error_map_outputs, T.iso_surface_outputs):
        out.update(make(lib))
    np.savez_compressed(os.path.join(OUT, "vs_ref"), **T.stored_form(out))
    print(f"vs_ref: {len(out)} outputs")


def main():
    if "--vs-ref-from-port" in sys.argv:
        vs_ref(O.port())
        return
    ref = O.reference()
    assert ref is not None, "build oracle/_ref first (make -C oracle)"

    # KAT-1: the README's 1D system on the real library (SURVEY.md §8c)
    f = ref.field([6])
    ret = [f.add_value_constraint([0.0], 4.0, 1.0), f.add_value_constraint([5.0], 2.0, 1.0),
           f.add_gradient_constraint([0.0], [1.0], 1.0, O.GRAD_NEAREST),
           f.add_gradient_constraint([5.0], [-1.0], 1.0, O.GRAD_NEAREST)]
    f.add_field_constraints(O.make_weights(model_2=1.0))
    save("kat1_readme_1d", f.system(), 6, returns=np.array(ret))

    # KAT-2 / C1: field_1d.cpp defaults at resolution 12 and 100 (data rows first, then model rows)
    for res in (12, 100):
        c = W.field_1d(res)
        w = O.make_weights()
        f = ref.field(c["sizes"])
        for p, v, g in zip(c["pos"], c["value"], c["gradient"]):
            f.add_value_constraint(p, float(v), w.data_pos)
            f.add_gradient_constraint(p, g, w.data_gradient, w.gradient_kernel)
        f.add_field_constraints(w)
        save(f"kat2_field_1d_res{res}", f.system(), res)

    # KAT-3: structure counts, 3D default weights, 1000 points strictly inside
    counts = []
    for n in (8, 16, 32):
        rng = np.random.default_rng(n)
        pos = rng.uniform(0.01, n - 1.01, size=(1000, 3)).astype(np.float32)
        nrm = rng.normal(size=(1000, 3)).astype(np.float32)
        s = ref.sdf_from_points([n] * 3, O.make_weights(), pos, nrm).system()
        counts.append([n, s.num_rows, s.num_triplets])
    np.savez_compressed(os.path.join(OUT, "kat3_counts"), counts=np.array(counts))
    print("kat3_counts:", counts)

    # KAT-4: every weight on, 7x6x9 lattice, no points
    w = O.make_weights(model_0=0.1, model_1=0.2, model_2=0.5, model_3=0.3, model_4=0.25, gradient_smoothness=0.15)
    f = ref.field([7, 6, 9])
    f.add_field_constraints(w)
    save("kat4_all_weights_7x6x9", f.system(), 7 * 6 * 9, weights=wdict(w))

    # Randomised differential cases: every dimension x value kernel x gradient kernel, points on / over every
    # boundary, exact-lattice hits, per-point weights (some zero).
    case = 0
    for sizes in ([11], [7, 6], [5, 4, 6]):
        D = len(sizes)
        for vk in (O.VALUE_NEAREST, O.VALUE_LINEAR):
            for gk in (O.GRAD_NEAREST, O.GRAD_CELL_EDGES, O.GRAD_LINEAR):
                pos, nrm = W.random_cloud(D, 40, sizes, seed=100 + case)
                pw = np.random.default_rng(case).uniform(0.0, 2.0, 40).astype(np.float32)
                pw[::7] = 0.0
                w = O.make_weights(model_0=0.05, model_1=0.1 * (case % 2), model_2=0.5, model_3=0.2 * (case % 3 == 0),
                                   model_4=0.1 * (case % 4 == 1), gradient_smoothness=0.1 * (D > 1 and case % 2),
                                   data_pos=1.5, data_gradient=0.75, value_kernel=vk, gradient_kernel=gk)
                s = ref.sdf_from_points(sizes, w, pos, nrm, pw).system()
                save(f"rand_{D}d_v{vk}_g{gk}", s, int(np.prod(sizes)), sizes=np.array(sizes), weights=wdict(w),
                     positions=pos, normals=nrm, point_weights=pw)
                case += 1

    # values-only cloud (normals == null) and a caller-appended generic row (sdf_field.cpp:239-241 pattern)
    sizes = [9, 8]
    pos, _ = W.random_cloud(2, 30, sizes, seed=7)
    w = O.make_weights(model_1=0.1, model_2=1.0)
    f = ref.sdf_from_points(sizes, w, pos, None, None)
    f.add_equation(0.001, 3.25, [5], [1.0])
    f.add_equation(0.5, -1.0, [0, 71], [1.0, -1.0])
    save("values_only_plus_rows_2d", f.system(), 72, sizes=np.array(sizes), weights=wdict(w), positions=pos)

    # upscale_field (field_interpolation.cpp:431-485) and generate_error_map (:402-429)
    rng = np.random.default_rng(3)
    for small, large in (([5], [12]), ([4, 5], [9, 13]), ([3, 4, 5], [7, 9, 11]), ([4, 4, 4], [8, 8, 8])):
        src = rng.normal(size=int(np.prod(small))).astype(np.float32)
        np.savez_compressed(os.path.join(OUT, f"upscale_{len(small)}d_{'x'.join(map(str, large))}"),
                            small=src, small_sizes=np.array(small), large_sizes=np.array(large),
                            large=ref.upscale_field(src, small, large))
    s = ref.sdf_from_points([7, 6], O.make_weights(), *W.random_cloud(2, 25, [7, 6], seed=5)).system()
    sol = rng.normal(size=42).astype(np.float32)
    save("error_map_2d", s, 42, solve=False, sol_in=sol, heat=ref.generate_error_map(s, sol))

    # iso-surface helpers (SURVEY.md §8f rank 4): emilib::marching_squares / calc_area from the reference's own
    # marching_squares.cpp, bicubic_upsample / iso_surface (src/sdf_field.cpp:555-614) around the reference's emath.
    def iso_case(name, field, upsample, iso):
        field = np.ascontiguousarray(field, np.float32)
        lines = ref.marching_squares(field)
        up = ref.bicubic_upsample(field, upsample)
        zero_up = ref.iso_surface(up, 0.0)
        np.savez_compressed(os.path.join(OUT, name), field=field, lines=lines, area=np.float32(ref.calc_area(lines)),
                            upsample=np.int32(upsample), upsampled=up, zero_lines_up=zero_up, area_up=np.float32(ref.calc_area(zero_up)),
                            iso=np.float32(iso), iso_lines_up=ref.iso_surface(up, iso), iso_lines=ref.iso_surface(field, iso))
        print(f"{name}: {field.shape} -> {len(lines)} segments, x{upsample}: {up.shape} -> {len(zero_up)} segments")

    sizes = [44, 37]
    cloud = W.circles_2d(600, seed=5)
    pos = W.to_lattice(cloud["unit_pos"], sizes)
    s = ref.sdf_from_points(sizes, O.make_weights(), pos, cloud["normals"]).system()
    iso_case("iso_sdf_2d_44x37", O.exact_solve(s, 44 * 37).astype(np.float32).reshape(37, 44), 3, 0.7)
    rng = np.random.default_rng(11)
    noise = rng.standard_normal((33, 20)).astype(np.float32)
    noise[rng.random((33, 20)) < 0.15] = 0.0      # exact zeros: corners sitting on the contour (>= 0 counts as outside)
    noise[5:9, 3:8] = np.float32(-0.0)
    iso_case("iso_random_33x20", noise, 2, -0.25)
    yy, xx = np.mgrid[0:75, 0:61].astype(np.float32)
    iso_case("iso_saddles_61x75", (np.sin(xx * np.float32(0.9)) * np.sin(yy * np.float32(1.1)) + np.float32(0.05)).astype(np.float32), 3, 0.3)
    iso_case("iso_2x2", np.array([[-1.0, 1.0], [1.0, -2.0]], np.float32), 5, 0.5)
    iso_case("iso_1x7", np.linspace(-1, 1, 7, dtype=np.float32).reshape(1, 7), 2, 0.0)   # no cells at all
    iso_case("iso_9x2", np.linspace(-1, 1, 18, dtype=np.float32).reshape(9, 2), 3, 0.1)

    vs_ref(ref)


if __name__ == "__main__":
    main()
