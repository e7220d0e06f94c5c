// Host side of include/emilib/marching_squares.hpp, include/field_interpolation/iso_surface.hpp and
// b200::marching_cubes: thin C++ over the C ABI (fi_marching_squares, fi_calc_area, fi_bicubic_upsample,
// fi_marching_cubes).  No arithmetic happens here.
#include "../../include/emilib/marching_squares.hpp"
#include "../../include/field_interpolation/field_interpolation.hpp"
#include "../../include/field_interpolation/iso_surface.hpp"

#include <cstdint>
#include <utility>

#include "../../include/fi_b200.h"

namespace {

std::vector<float> contour(int width, int height, const float* values, float iso)
{
	if (width < 1 || height < 1 || values == nullptr) { return {}; }
	int64_t n = 0;
	if (fi_marching_squares(width, height, values, iso, FI_HOST, nullptr, 0, &n, nullptr) != FI_OK || n == 0) { return {}; }
	std::vector<float> lines(static_cast<size_t>(n) * 4);
	if (fi_marching_squares(width, height, values, iso, FI_HOST, lines.data(), n, &n, nullptr) != FI_OK) { return {}; }
	return lines;
}

}  // namespace

namespace emilib {

std::vector<float> marching_squares(std::size_t width, std::size_t height, const float* iso)
{
	return contour(static_cast<int>(width), static_cast<int>(height), iso, 0.0f);
}

float calc_area(std::size_t num_line_segments, const float* xy)
{
	float area = 0.0f;
	if (fi_calc_area(static_cast<int64_t>(num_line_segments), xy, FI_HOST, &area) != FI_OK) { return 0.0f; }
	return area;
}

}  // namespace emilib

namespace field_interpolation {

std::vector<float> bicubic_upsample(int* io_width, int* io_height, const float* values, int upsample)
{
	if (!io_width || !io_height || !values || upsample <= 1 || *io_width < 1 || *io_height < 1) { return {}; }
	const int64_t lw = static_cast<int64_t>(upsample) * *io_width - upsample + 1, lh = static_cast<int64_t>(upsample) * *io_height - upsample + 1;
	std::vector<float> large(static_cast<size_t>(lw * lh));
	if (fi_bicubic_upsample(*io_width, *io_height, values, upsample, large.data(), FI_HOST) != FI_OK) { return {}; }
	*io_width  = static_cast<int>(lw);
	*io_height = static_cast<int>(lh);
	return large;
}

std::vector<float> iso_surface(int width, int height, const float* values, float iso) { return contour(width, height, values, iso); }

}  // namespace field_interpolation

namespace field_interpolation {
namespace b200 {

bool marching_cubes(const std::vector<int>& sizes, const float* values, float iso, bool want_normals, Mesh* mesh)
{
	if (mesh == nullptr) { return false; }
	*mesh = Mesh();
	if (sizes.size() != 3 || values == nullptr) { return false; }
	const int32_t sz[3] = {sizes[0], sizes[1], sizes[2]};
	int64_t       nv = 0, nt = 0;
	if (fi_marching_cubes(sz, values, iso, FI_HOST, nullptr, nullptr, 0, nullptr, 0, &nv, &nt) != FI_OK) { return false; }
	if (nv == 0) { return true; }
	Mesh out;
	out.positions.resize(static_cast<size_t>(nv) * 3);
	if (want_normals) { out.normals.resize(static_cast<size_t>(nv) * 3); }
	out.triangles.resize(static_cast<size_t>(nt) * 3);
	static_assert(sizeof(int) == sizeof(int32_t), "triangles are int32 in the C ABI");
	if (fi_marching_cubes(sz, values, iso, FI_HOST, out.positions.data(), want_normals ? out.normals.data() : nullptr, nv,
	                      reinterpret_cast<int32_t*>(out.triangles.data()), nt, &nv, &nt) != FI_OK) {
		return false;
	}
	*mesh = std::move(out);
	return true;
}

}  // namespace b200
}  // namespace field_interpolation
