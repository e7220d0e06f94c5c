// A C++ caller of b200::generate_error_map (include/field_interpolation/field_interpolation.hpp) on a deferred
// LatticeField, built against the drop-in headers and libraries.  Usage: error_map_driver IN OUT.  IN: int32 D,
// int32 sizes[D], int64 n, then n*D position floats, n*D normal floats and prod(sizes) solution floats.  The field is
// add_field_constraints(Weights()) + add_points of the points with the default weights and kernels + one row appended
// by hand with add_equation.  OUT: the heat map (prod(sizes) floats), then the model, point and caller row sums (3
// doubles).
#include <cstdint>
#include <cstdio>
#include <vector>

#include "field_interpolation/field_interpolation.hpp"

int main(int argc, char** argv)
{
	using namespace field_interpolation;
	if (argc != 3) { return 2; }
	std::FILE* in = std::fopen(argv[1], "rb");
	if (!in) { return 2; }
	int32_t D = 0;
	int64_t n = 0;
	if (std::fread(&D, 4, 1, in) != 1 || D < 1 || D > 3) { return 2; }
	std::vector<int> sizes(static_cast<size_t>(D));
	size_t           cells = 1;
	for (int d = 0; d < D; ++d) {
		int32_t s = 0;
		if (std::fread(&s, 4, 1, in) != 1) { return 2; }
		sizes[static_cast<size_t>(d)] = s;
		cells *= static_cast<size_t>(s);
	}
	if (std::fread(&n, 8, 1, in) != 1) { return 2; }
	std::vector<float> pos(static_cast<size_t>(n) * D), nrm(pos.size()), x(cells);
	if (std::fread(pos.data(), 4, pos.size(), in) != pos.size() || std::fread(nrm.data(), 4, nrm.size(), in) != nrm.size() ||
	    std::fread(x.data(), 4, x.size(), in) != x.size()) {
		return 2;
	}
	std::fclose(in);

	LatticeField field{sizes};
	b200::defer_triplets(&field, true);
	const Weights w;
	add_field_constraints(&field, w);
	add_points(&field, w.data_pos, w.value_kernel, w.data_gradient, w.gradient_kernel, static_cast<int>(n), pos.data(), nrm.data(), nullptr);
	add_equation(&field.eq, Weight{2.0f}, Rhs{0.5f}, {{1, 1.0f}, {3, -0.5f}});
	if (!field.eq.triplets.empty() && field.eq.triplets.size() != 2) { return 3; }  // deferred: only the hand-written row is in eq

	b200::ErrorSums          sums;
	const std::vector<float> heat = b200::generate_error_map(&field, x, &sums);
	if (heat.size() != cells) {
		std::fprintf(stderr, "generate_error_map failed\n");
		return 1;
	}
	std::FILE* out = std::fopen(argv[2], "wb");
	if (!out) { return 2; }
	const double s[3] = {sums.model_rows, sums.point_rows, sums.caller_rows};
	std::fwrite(heat.data(), 4, heat.size(), out);
	std::fwrite(s, 8, 3, out);
	std::fclose(out);
	return 0;
}
