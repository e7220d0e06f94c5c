// TEST INFRASTRUCTURE — NOT PRODUCT CODE.  Sequential CPU port of fi_marching_cubes (include/fi_b200.h): one pass over
// the nodes in index order numbers the vertices, one pass over the cells in index order writes the triangles from the
// generated case table (field_interpolation_b200/csrc/mc_table.cuh).  Built with -ffp-contract=off: the same scalar
// fp32 expressions as the -fmad=false CUDA build, so vertices, normals and indices agree bit for bit.
#include <cmath>
#include <cstdint>
#include <vector>

#include "../field_interpolation_b200/csrc/mc_table.cuh"

namespace {

float gradient(const float* v, int64_t i, int64_t c, int64_t n, int64_t st)
{
	if (c == 0) { return v[i + st] - v[i]; }
	if (c + 1 == n) { return v[i] - v[i - st]; }
	return 0.5f * (v[i + st] - v[i - st]);
}

}  // namespace

// sizes: nx ny nz.  Writes the counts; fills the non-null outputs (sized by a previous count-only call).
extern "C" void mcp_marching_cubes(const int32_t* sizes, const float* v, float iso, float* vertices, float* normals, int32_t* triangles,
                                   int64_t* num_vertices, int64_t* num_triangles)
{
	*num_vertices = *num_triangles = 0;
	const int64_t n[3] = {sizes[0], sizes[1], sizes[2]};
	if (n[0] < 2 || n[1] < 2 || n[2] < 2) { return; }
	const int64_t st[3] = {1, n[0], n[0] * n[1]}, nodes = n[0] * n[1] * n[2];
	std::vector<uint8_t> side(static_cast<size_t>(nodes));
	for (int64_t i = 0; i < nodes; ++i) { side[i] = v[i] - iso >= 0.0f; }
	std::vector<int64_t> first(static_cast<size_t>(nodes), -1);  // first vertex of each node
	int64_t nv = 0;
	for (int64_t z = 0; z < n[2]; ++z) {
		for (int64_t y = 0; y < n[1]; ++y) {
			for (int64_t x = 0; x < n[0]; ++x) {
				const int64_t c[3] = {x, y, z}, i = x + st[1] * y + st[2] * z;
				for (int e = 0; e < 3; ++e) {
					if (c[e] + 1 >= n[e] || side[i] == side[i + st[e]]) { continue; }
					if (first[i] < 0) { first[i] = nv; }
					const float a = v[i] - iso, b = v[i + st[e]] - iso;
					const float t = a / (a - b);
					if (vertices) {
						for (int d = 0; d < 3; ++d) { vertices[3 * nv + d] = d == e ? static_cast<float>(c[d]) + t : static_cast<float>(c[d]); }
					}
					if (normals) {
						float g[3];
						for (int d = 0; d < 3; ++d) {
							const float lo = gradient(v, i, c[d], n[d], st[d]);
							const float hi = gradient(v, i + st[e], c[d] + (d == e ? 1 : 0), n[d], st[d]);
							g[d]           = lo + t * (hi - lo);
						}
						const float len = std::sqrt(g[0] * g[0] + g[1] * g[1] + g[2] * g[2]);
						for (int d = 0; d < 3; ++d) { normals[3 * nv + d] = len > 0.0f ? g[d] / len : 0.0f; }
					}
					++nv;
				}
			}
		}
	}
	// vertex of the edge along `axis` starting at node (x, y, z): the node's first vertex plus its crossed lower-axis edges
	auto vertex = [&](int64_t x, int64_t y, int64_t z, int axis) {
		const int64_t c[3] = {x, y, z}, i = x + st[1] * y + st[2] * z;
		int64_t       id   = first[i];
		for (int b = 0; b < axis; ++b) { id += (c[b] + 1 < n[b] && side[i] != side[i + st[b]]) ? 1 : 0; }
		return id;
	};
	int64_t nt = 0;
	for (int64_t z = 0; z + 1 < n[2]; ++z) {
		for (int64_t y = 0; y + 1 < n[1]; ++y) {
			for (int64_t x = 0; x + 1 < n[0]; ++x) {
				int cfg = 0;
				for (int k = 0; k < 8; ++k) { cfg |= side[(x + (k & 1)) + st[1] * (y + ((k >> 1) & 1)) + st[2] * (z + (k >> 2))] << k; }
				for (int t = 0; t < 3 * fi_mc::kTriCount[cfg]; ++t) {
					const int e = fi_mc::kTriEdges[cfg][t], k = fi_mc::kEdgeCorner[e];
					if (triangles) { triangles[3 * nt + t] = static_cast<int32_t>(vertex(x + (k & 1), y + ((k >> 1) & 1), z + (k >> 2), e >> 2)); }
				}
				nt += fi_mc::kTriCount[cfg];
			}
		}
	}
	*num_vertices  = nv;
	*num_triangles = nt;
}
