// field_interpolation/field_interpolation.hpp — B200 drop-in for the header of the same name in
// emilk/field_interpolation (reference field_interpolation/field_interpolation.hpp:44-183): lattice fields,
// the constraint builders and the point-cloud helpers, with the reference's names, signatures, defaults and
// return conventions.  Callers written against the reference (its src/field_1d.cpp, src/interpolate_2d.cpp,
// src/sdf_field.cpp ...) compile unchanged.
//
// Implementation: field_interpolation_b200/host/field_interpolation.cpp — host C++ over the C ABI of
// libfi_b200.so (include/fi_b200.h).  Every builder records the constraint in the device-resident structured
// description (field->eq.structured) and, unless triplet mirroring was switched off with
// b200::defer_triplets, appends the rows it produced — bit-identical to the reference's — to field->eq so the
// triplet list stays observable and appendable exactly as before.
#pragma once

#include <cstdint>
#include <vector>

#include "sparse_linear.hpp"

namespace field_interpolation {

const int MAX_DIM = 3;  // reference :44

enum class ValueKernel  // reference :47-51
{
	kNearestNeighbor,
	kLinearInterpolation,
};

enum class GradientKernel  // reference :54-59
{
	kNearestNeighbor,
	kCellEdges,
	kLinearInterpolation,
};

struct Weights  // reference :75-95, same order and defaults
{
	float data_pos      = 1.00f;
	float data_gradient = 1.00f;
	float model_0       = 0.00f;
	float model_1       = 0.00f;
	float model_2       = 0.50f;
	float model_3       = 0.00f;
	float model_4       = 0.00f;
	float gradient_smoothness = 0.0f;

	ValueKernel    value_kernel    = ValueKernel::kLinearInterpolation;
	GradientKernel gradient_kernel = GradientKernel::kCellEdges;
};

struct LatticeField  // reference :97-114
{
	LinearEquation   eq;       ///< Accumulated equations.
	std::vector<int> sizes;    ///< sizes[d] == size of dimension `d`
	std::vector<int> strides;  ///< strides[d] == distance between adjacent values along dimension `d` (x fastest)

	LatticeField() = default;
	explicit LatticeField(const std::vector<int>& sizes_arg) : sizes(sizes_arg)
	{
		int stride = 1;
		for (int size : sizes) {
			strides.push_back(stride);
			stride *= size;
		}
	}

	int num_dim() const { return static_cast<int>(sizes.size()); }
};

/// Add equations describing the model: a smooth field on a lattice.  (reference field_interpolation.cpp:326-341)
void add_field_constraints(LatticeField* field, const Weights& weights);

/// f(pos) = value.  Returns false if the position was ignored (outside, or weight == 0).  (reference :57-80)
bool add_value_constraint(LatticeField* field, const float pos[], float value, float weight);

/// f(pos) = value applied at the nearest lattice point with a gradient offset.  Returns false iff the point
/// is outside of the field.  (reference :82-107)
bool add_value_constraint_nearest_neighbor(LatticeField* field, const float pos[], const float gradient[], float value, float weight);

/// grad f(pos) = gradient.  Returns false if the position was ignored.  (reference :123-240)
bool add_gradient_constraint(LatticeField* field, const float pos[], const float gradient[], float weight, GradientKernel kernel);

/// add_value_constraint* and add_gradient_constraint for every point.  (reference :343-371)
void add_points(LatticeField* field, float value_weight, ValueKernel value_kernel, float gradient_weight, GradientKernel gradient_kernel,
                const int num_points, const float positions[], const float* normals, const float* point_weights);

/// Signed distance field from oriented points.  (reference :373-400)
LatticeField sdf_from_points(const std::vector<int>& sizes, const Weights& weights, const int num_points, const float positions[],
                             const float* normals, const float* point_weights);

/// (Ax - b)^2 distributed onto the solution space, a heat map of blame.  (reference :402-429)
std::vector<float> generate_error_map(const std::vector<Triplet>& triplets, const std::vector<float>& solution,
                                      const std::vector<float>& rhs);

/// Multilinear interpolation of a small lattice onto a large one.  (reference :431-485)
std::vector<float> upscale_field(const float* field, const std::vector<int>& small_sizes, const std::vector<int>& large_sizes);

// ---- B200 extensions ---------------------------------------------------------------------------------------
namespace b200 {

/// Stops (or resumes) mirroring the rows of builder calls into field->eq.  With mirroring off nothing of size
/// O(rows) ever exists on the host: this is how lattices whose triplet list would not fit the reference's
/// int32 rows (1024^3: 3.2e9 model rows) are built.  Call before the first builder.
void defer_triplets(LatticeField* field, bool deferred);

/// Brings field->eq up to date with everything recorded so far (no-op unless mirroring was deferred).
/// Returns false when the system does not fit the int32 triplet view.
bool materialize(LatticeField* field);

/// Number of equations / triplets recorded, whether or not they are mirrored in field->eq.
void counts(const LatticeField& field, long long* num_rows, long long* num_triplets);

struct CascadeStats
{
	int                    levels = 0;
	std::vector<long long> level_cells, level_iterations;
	std::vector<double>    level_ms, level_initial_residual;
	double                 total_ms = 0;
	SolveStats             finest;
};

/// Coarse-to-fine SDF solve, the recipe of the reference demo (src/sdf_field.cpp:251-304) applied recursively:
/// positions in unit coordinates are scaled per level by (size - 1), every level is re-assembled with the same
/// weights and unscaled normals, the coarser solution is upscaled, multiplied by the size ratio and refined by
/// PCG.  Returns {} on failure.
std::vector<float> sdf_solve_cascade(const std::vector<int>& sizes, const Weights& weights, int num_points, const float unit_positions[],
                                     const float* normals, const float* point_weights, Precision precision, int max_iterations,
                                     double tolerance, int factor, int coarsest_size, double coarse_tolerance, CascadeStats* stats);

/// Triangle mesh in lattice coordinates (x y z per vertex; three vertex indices per triangle).
struct Mesh
{
	std::vector<float> positions, normals;  ///< 3 floats per vertex; normals empty unless asked for
	std::vector<int>   triangles;           ///< 3 per triangle, (P1 - P0) x (P2 - P0) toward values >= iso
};

/// Marching cubes of the surface values == iso of a 3D lattice (sizes = {nx, ny, nz}, x fastest, host values) on the
/// GPU: fi_marching_cubes (include/fi_b200.h) states the contract.  Returns false on failure (mesh left empty).
bool marching_cubes(const std::vector<int>& sizes, const float* values, float iso, bool want_normals, Mesh* mesh);

/// Value (and gradient) of a lattice field (sizes = {nx[, ny[, nz]]}, x fastest, host values) at num_points host
/// positions (D interleaved floats each, lattice coordinates), on the GPU: fi_sample_field (include/fi_b200.h) states
/// the contract.  values receives num_points floats; gradients (with want_gradients) D per point, computed with
/// `kernel`.  NaN where the reference would emit no row.  Returns false on failure (outputs left empty).
bool sample_field(const std::vector<int>& sizes, const float* field, int64_t num_points, const float* positions, GradientKernel kernel,
                  bool want_gradients, std::vector<float>* values, std::vector<float>* gradients);

/// Sum over rows of err^2 (err = rhs - row . solution in fp32, squared and summed in fp64), by kind of row: the
/// least-squares objective the solve minimises, term by term.
struct ErrorSums
{
	double model_rows = 0, point_rows = 0, caller_rows = 0;
};

/// generate_error_map of the field's own system, on the GPU and without its triplet list: bit-identical to
/// generate_error_map(field->eq.triplets, solution, field->eq.rhs) of a materialised field, and also defined for
/// deferred fields and systems beyond the int32 triplet view.  Rows appended to field->eq by hand are forwarded first,
/// as the builders do.  fi_field_error_map (include/fi_b200.h) states the contract.  Returns {} on failure.
std::vector<float> generate_error_map(LatticeField* field, const std::vector<float>& solution, ErrorSums* sums = nullptr);

}  // namespace b200

}  // namespace field_interpolation
