// A C++ caller of b200::add_border_distance_constraints (include/field_interpolation/field_interpolation.hpp), built
// against the drop-in headers and libraries.  It builds the 2D demo field of the reference's SDF caller
// (src/sdf_field.cpp:212-249: sdf_from_points, then one add_equation per border node with the brute-force nearest
// distance) three ways in one process, each with a row appended by hand before the border rows:
//   A  the demo's hand loop with add_equation;
//   B  b200::add_border_distance_constraints;
//   C  the same on a deferred field, materialised afterwards.
// It exits 1 unless the three field.eq are bit-identical.  Usage: border_driver IN OUT.  IN: int32 width, height,
// float boundary_weight, int64 n, then n*2 unit position floats and n*2 normal floats.  OUT: int64 rows, triplets,
// then B's triplets (row, col int32, value float each) and rhs floats.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <limits>
#include <vector>

#include "field_interpolation/field_interpolation.hpp"

using namespace field_interpolation;

static bool same(const LinearEquation& a, const LinearEquation& b)
{
	if (a.triplets.size() != b.triplets.size() || a.rhs.size() != b.rhs.size()) { return false; }
	return std::memcmp(a.triplets.data(), b.triplets.data(), a.triplets.size() * sizeof(Triplet)) == 0 &&
	       std::memcmp(a.rhs.data(), b.rhs.data(), a.rhs.size() * sizeof(float)) == 0;
}

int main(int argc, char** argv)
{
	if (argc != 3) { return 2; }
	std::FILE* in = std::fopen(argv[1], "rb");
	if (!in) { return 2; }
	int32_t wh[2] = {0, 0};
	float   bw    = 0;
	int64_t n     = 0;
	if (std::fread(wh, 4, 2, in) != 2 || std::fread(&bw, 4, 1, in) != 1 || std::fread(&n, 8, 1, in) != 1 || n < 1) { return 2; }
	std::vector<float> unit(static_cast<size_t>(n) * 2), nrm(unit.size());
	if (std::fread(unit.data(), 4, unit.size(), in) != unit.size() || std::fread(nrm.data(), 4, nrm.size(), in) != nrm.size()) { return 2; }
	std::fclose(in);
	const int w = wh[0], h = wh[1], npts = static_cast<int>(n);
	std::vector<float> pos(unit.size());
	for (int i = 0; i < npts; ++i) {  // on_lattice, src/sdf_field.cpp:198-210
		pos[2 * i]     = unit[2 * i] * (w - 1.0f);
		pos[2 * i + 1] = unit[2 * i + 1] * (h - 1.0f);
	}
	const Weights weights;

	LatticeField a = sdf_from_points({w, h}, weights, npts, pos.data(), nrm.data(), nullptr);
	add_equation(&a.eq, Weight{2.0f}, Rhs{0.5f}, {{1, 1.0f}, {3, -0.5f}});
	for (int y = 0; y < h; ++y) {
		for (int x = 0; x < w; ++x) {
			if (!(x == 0 || x == w - 1 || y == 0 || y == h - 1)) { continue; }
			float closest = std::numeric_limits<float>::infinity();
			for (int i = 0; i < npts; ++i) {
				const float dx = pos[2 * i] - x, dy = pos[2 * i + 1] - y;
				closest        = std::min(closest, dx * dx + dy * dy);
			}
			add_equation(&a.eq, Weight{bw}, {std::sqrt(closest)}, {{y * w + x, 1.0f}});
		}
	}

	LatticeField b = sdf_from_points({w, h}, weights, npts, pos.data(), nrm.data(), nullptr);
	add_equation(&b.eq, Weight{2.0f}, Rhs{0.5f}, {{1, 1.0f}, {3, -0.5f}});
	const long long added = b200::add_border_distance_constraints(&b, bw, npts, pos.data());

	LatticeField c{{w, h}};
	b200::defer_triplets(&c, true);
	add_field_constraints(&c, weights);
	add_points(&c, weights.data_pos, weights.value_kernel, weights.data_gradient, weights.gradient_kernel, npts, pos.data(), nrm.data(), nullptr);
	add_equation(&c.eq, Weight{2.0f}, Rhs{0.5f}, {{1, 1.0f}, {3, -0.5f}});
	if (b200::add_border_distance_constraints(&c, bw, npts, pos.data()) != added || !b200::materialize(&c)) { return 1; }

	LatticeField bad{{w, h}};
	if (b200::add_border_distance_constraints(&bad, bw, 0, pos.data()) != -1) { return 1; }  // no points

	std::vector<float>   dist;
	std::vector<int64_t> near;
	const float          q[4] = {0.0f, 0.0f, static_cast<float>(w - 1), static_cast<float>(h - 1)};
	if (!b200::nearest_point_distance(2, n, pos.data(), 2, q, &dist, &near) || dist.size() != 2 || near.size() != 2) { return 1; }

	if (added != 2 * (w + h) - 4 || !same(a.eq, b.eq) || !same(a.eq, c.eq)) {
		std::fprintf(stderr, "border rows differ: added %lld\n", added);
		return 1;
	}
	// the first and last border rows are those of corners (0, 0) and (w - 1, h - 1)
	if (dist[0] * bw != b.eq.rhs[b.eq.rhs.size() - static_cast<size_t>(added)] || dist[1] * bw != b.eq.rhs.back()) { return 1; }
	std::FILE* out = std::fopen(argv[2], "wb");
	if (!out) { return 2; }
	const int64_t counts[2] = {static_cast<int64_t>(b.eq.rhs.size()), static_cast<int64_t>(b.eq.triplets.size())};
	std::fwrite(counts, 8, 2, out);
	std::fwrite(b.eq.triplets.data(), sizeof(Triplet), b.eq.triplets.size(), out);
	std::fwrite(b.eq.rhs.data(), 4, b.eq.rhs.size(), out);
	std::fclose(out);
	return 0;
}
