// A C++ caller of b200::marching_cubes (include/field_interpolation/field_interpolation.hpp), built against the drop-in
// headers and libraries.  Usage: mesh_driver IN OUT.  IN: int32 nx ny nz, float iso, int32 want_normals, then nx*ny*nz
// floats.  OUT: int64 V, int64 T, then V*3 positions, V*3 normals (when asked for), T*3 int32 triangles.
#include <cstdint>
#include <cstdio>
#include <vector>

#include "field_interpolation/field_interpolation.hpp"

int main(int argc, char** argv)
{
	if (argc != 3) { return 2; }
	std::FILE* in = std::fopen(argv[1], "rb");
	if (!in) { return 2; }
	int32_t sizes[3];
	float   iso;
	int32_t want_normals;
	if (std::fread(sizes, 4, 3, in) != 3 || std::fread(&iso, 4, 1, in) != 1 || std::fread(&want_normals, 4, 1, in) != 1) { return 2; }
	std::vector<float> values(static_cast<size_t>(sizes[0]) * sizes[1] * sizes[2]);
	if (std::fread(values.data(), 4, values.size(), in) != values.size()) { return 2; }
	std::fclose(in);

	field_interpolation::b200::Mesh mesh;
	if (!field_interpolation::b200::marching_cubes({sizes[0], sizes[1], sizes[2]}, values.data(), iso, want_normals != 0, &mesh)) {
		std::fprintf(stderr, "marching_cubes failed\n");
		return 1;
	}
	std::FILE* out = std::fopen(argv[2], "wb");
	if (!out) { return 2; }
	const int64_t nv = static_cast<int64_t>(mesh.positions.size() / 3), nt = static_cast<int64_t>(mesh.triangles.size() / 3);
	std::fwrite(&nv, 8, 1, out);
	std::fwrite(&nt, 8, 1, out);
	std::fwrite(mesh.positions.data(), 4, mesh.positions.size(), out);
	std::fwrite(mesh.normals.data(), 4, mesh.normals.size(), out);
	std::fwrite(mesh.triangles.data(), 4, mesh.triangles.size(), out);
	std::fclose(out);
	return 0;
}
