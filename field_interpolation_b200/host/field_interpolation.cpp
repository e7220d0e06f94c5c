// Host C++ implementation of include/field_interpolation/field_interpolation.hpp over the C ABI of
// libfi_b200.so.  Each function cites the reference function whose behaviour it reproduces
// (field_interpolation/field_interpolation.cpp of the reference tree); the arithmetic itself runs in the CUDA
// kernels of csrc/assembly.cu.
#include <cmath>
#include <cstring>
#include <utility>

#include "structured.hpp"

namespace field_interpolation {

namespace b200 {

static fi_weights to_c(const Weights& w)
{
	fi_weights c;
	c.data_pos            = w.data_pos;
	c.data_gradient       = w.data_gradient;
	c.model_0             = w.model_0;
	c.model_1             = w.model_1;
	c.model_2             = w.model_2;
	c.model_3             = w.model_3;
	c.model_4             = w.model_4;
	c.gradient_smoothness = w.gradient_smoothness;
	c.value_kernel        = static_cast<int32_t>(w.value_kernel);
	c.gradient_kernel     = static_cast<int32_t>(w.gradient_kernel);
	return c;
}

Forwarded forward_tail_rows(const LinearEquation& eq, Structured* st)
{
	if (eq.rhs.size() == st->eq_rows && eq.triplets.size() == st->eq_triplets) { return Forwarded::kOk; }
	// the list shrank (clear(), resize, assignment from a shorter system): what the handle holds is not a prefix of it any more
	if (eq.rhs.size() < st->eq_rows || eq.triplets.size() < st->eq_triplets) { return Forwarded::kInconsistent; }
	const size_t nrows = eq.rhs.size() - st->eq_rows, ntrip = eq.triplets.size() - st->eq_triplets;
	std::vector<int32_t> r(ntrip), c(ntrip);
	std::vector<float>   v(ntrip);
	bool sorted = true;
	for (size_t k = 0; k < ntrip; ++k) {
		const Triplet& t = eq.triplets[st->eq_triplets + k];
		const long long rel = static_cast<long long>(t.row) - static_cast<long long>(st->eq_rows);
		if (rel < 0 || rel >= static_cast<long long>(nrows)) { return Forwarded::kInconsistent; }
		r[k] = static_cast<int32_t>(rel);
		c[k] = t.col;
		v[k] = t.value;
		sorted = sorted && (k == 0 || r[k - 1] <= r[k]);
	}
	if (!sorted) {  // rows appended by hand need not be grouped; a stable counting sort keeps duplicates in order
		std::vector<size_t> start(nrows + 1, 0);
		for (size_t k = 0; k < ntrip; ++k) { ++start[r[k] + 1]; }
		for (size_t i = 0; i < nrows; ++i) { start[i + 1] += start[i]; }
		std::vector<int32_t> r2(ntrip), c2(ntrip);
		std::vector<float>   v2(ntrip);
		for (size_t k = 0; k < ntrip; ++k) {
			const size_t at = start[r[k]]++;
			r2[at] = r[k];
			c2[at] = c[k];
			v2[at] = v[k];
		}
		r.swap(r2);
		c.swap(c2);
		v.swap(v2);
	}
	// fi_field_add_rows validates before it stores anything: a refused call leaves the handle as it was
	if (fi_field_add_rows(st->handle, static_cast<int64_t>(nrows), static_cast<int64_t>(ntrip), r.data(), c.data(), v.data(),
	                      eq.rhs.data() + st->eq_rows) != FI_OK) {
		return Forwarded::kError;
	}
	st->eq_rows     = eq.rhs.size();
	st->eq_triplets = eq.triplets.size();
	return Forwarded::kOk;
}

std::shared_ptr<Structured> clone_description(const Structured& src)
{
	auto st = std::make_shared<Structured>();
	if (fi_field_clone(src.handle, &st->handle) != FI_OK) { return nullptr; }
	st->sizes       = src.sizes;
	st->deferred    = src.deferred;
	st->eq_rows     = src.eq_rows;
	st->eq_triplets = src.eq_triplets;
	return st;
}

std::shared_ptr<Structured> description_from_triplets(const LinearEquation& eq, const std::vector<int>& sizes)
{
	if (sizes.empty() || static_cast<int>(sizes.size()) > MAX_DIM) { return nullptr; }
	auto st   = std::make_shared<Structured>();
	st->sizes = sizes;
	std::vector<int32_t> sz(sizes.begin(), sizes.end());
	if (fi_field_create(static_cast<int32_t>(sz.size()), sz.data(), &st->handle) != FI_OK) { return nullptr; }
	if (forward_tail_rows(eq, st.get()) != Forwarded::kOk) { return nullptr; }
	return st;
}

Structured* structured_for_append(LatticeField* field)
{
	LinearEquation& eq = field->eq;
	if (!eq.structured) {
		if (field->sizes.empty() || static_cast<int>(field->sizes.size()) > MAX_DIM) { return nullptr; }
		auto st   = std::make_shared<Structured>();
		st->sizes = field->sizes;
		std::vector<int32_t> sz(field->sizes.begin(), field->sizes.end());
		if (fi_field_create(static_cast<int32_t>(sz.size()), sz.data(), &st->handle) != FI_OK) { return nullptr; }
		eq.structured = st;
	}
	// a copied LatticeField / LinearEquation shares the description with its source until one of them is written to
	if (eq.structured.use_count() > 1) {
		auto own = clone_description(*eq.structured);
		if (!own) { return nullptr; }
		eq.structured = own;
	}
	Structured*     st  = eq.structured.get();
	const Forwarded fwd = forward_tail_rows(eq, st);
	if (fwd == Forwarded::kInconsistent && !st->deferred) {
		// the caller rewrote eq (cleared it, assigned another system): the triplet list is the truth, start again from it
		auto fresh = description_from_triplets(eq, field->sizes);
		if (!fresh) { return nullptr; }
		eq.structured = fresh;
		return fresh.get();
	}
	return fwd == Forwarded::kOk ? st : nullptr;
}

bool mirror_new_rows(LinearEquation* eq, Structured* st, long long rows_before, long long trips_before)
{
	int64_t rows = 0, trips = 0;
	if (fi_field_counts(st->handle, &rows, &trips) != FI_OK) { return false; }
	if (st->deferred || (rows == rows_before && trips == trips_before)) { return true; }
	const size_t nr = static_cast<size_t>(rows - rows_before), nt = static_cast<size_t>(trips - trips_before);
	static_assert(sizeof(Triplet) == sizeof(fi_triplet), "Triplet must be layout-identical to fi_triplet");
	const size_t r0 = eq->rhs.size(), t0 = eq->triplets.size();
	eq->rhs.resize(r0 + nr);
	eq->triplets.resize(t0 + nt);
	if (fi_field_export_rows(st->handle, rows_before, reinterpret_cast<fi_triplet*>(eq->triplets.data() + t0), eq->rhs.data() + r0) != FI_OK) {
		eq->rhs.resize(r0);
		eq->triplets.resize(t0);
		return false;
	}
	st->eq_rows     = eq->rhs.size();
	st->eq_triplets = eq->triplets.size();
	return true;
}

// One builder call: forward pending hand-written rows, run `call` on the handle, mirror what it added.
// Returns the number of equations added, or -1 on error.
template <typename F>
static long long build(LatticeField* field, F&& call)
{
	Structured* st = structured_for_append(field);
	if (!st) { return -1; }
	int64_t rows0 = 0, trips0 = 0;
	if (fi_field_counts(st->handle, &rows0, &trips0) != FI_OK) { return -1; }
	if (call(st->handle) != FI_OK) { return -1; }
	int64_t rows1 = 0, trips1 = 0;
	if (fi_field_counts(st->handle, &rows1, &trips1) != FI_OK) { return -1; }
	if (!mirror_new_rows(&field->eq, st, rows0, trips0)) { return -1; }
	return rows1 - rows0;
}

void defer_triplets(LatticeField* field, bool deferred)
{
	Structured* st = structured_for_append(field);
	if (!st) { return; }
	if (st->deferred && !deferred) { materialize(field); }
	st->deferred = deferred;
}

bool materialize(LatticeField* field)
{
	Structured* st = structured_for_append(field);
	if (!st) { return false; }
	int64_t rows = 0, trips = 0;
	if (fi_field_counts(st->handle, &rows, &trips) != FI_OK) { return false; }
	if (static_cast<size_t>(rows) == field->eq.rhs.size() && static_cast<size_t>(trips) == field->eq.triplets.size()) { return true; }
	std::vector<Triplet> t(static_cast<size_t>(trips));
	std::vector<float>   b(static_cast<size_t>(rows));
	if (fi_field_export(st->handle, reinterpret_cast<fi_triplet*>(t.data()), b.data()) != FI_OK) { return false; }
	field->eq.triplets.swap(t);
	field->eq.rhs.swap(b);
	st->eq_rows     = field->eq.rhs.size();
	st->eq_triplets = field->eq.triplets.size();
	return true;
}

void counts(const LatticeField& field, long long* num_rows, long long* num_triplets)
{
	int64_t r = static_cast<int64_t>(field.eq.rhs.size()), t = static_cast<int64_t>(field.eq.triplets.size());
	if (field.eq.structured) {
		int64_t hr = 0, ht = 0;
		if (fi_field_counts(field.eq.structured->handle, &hr, &ht) == FI_OK) {
			// rows appended by hand and not forwarded yet come on top of what the handle holds
			r = hr + static_cast<int64_t>(field.eq.rhs.size() - field.eq.structured->eq_rows);
			t = ht + static_cast<int64_t>(field.eq.triplets.size() - field.eq.structured->eq_triplets);
		}
	}
	if (num_rows) { *num_rows = r; }
	if (num_triplets) { *num_triplets = t; }
}

std::vector<float> sdf_solve_cascade(const std::vector<int>& sizes, const Weights& weights, int num_points, const float unit_positions[],
                                     const float* normals, const float* point_weights, Precision precision, int max_iterations,
                                     double tolerance, int factor, int coarsest_size, double coarse_tolerance, CascadeStats* stats)
{
	fi_cascade_options o;
	std::memset(&o, 0, sizeof(o));
	fi_solve_options_default(&o.fine);
	o.fine.precision      = static_cast<int32_t>(precision);
	o.fine.max_iterations = max_iterations;
	o.fine.tolerance      = tolerance;
	o.factor              = factor;
	o.coarsest_size       = coarsest_size;
	o.coarse_tolerance    = coarse_tolerance;
	size_t n = 1;
	for (int s : sizes) { n *= static_cast<size_t>(s); }
	std::vector<float>   out(n);
	std::vector<int32_t> sz(sizes.begin(), sizes.end());
	const fi_weights     w = to_c(weights);
	fi_cascade_stats     cs;
	if (fi_sdf_solve_cascade(static_cast<int32_t>(sz.size()), sz.data(), &w, num_points, unit_positions, normals, point_weights, &o, out.data(),
	                         FI_HOST, &cs) != FI_OK) {
		return {};
	}
	if (stats) {
		stats->levels = cs.levels;
		stats->level_cells.assign(cs.level_cells, cs.level_cells + cs.levels);
		stats->level_iterations.assign(cs.level_iterations, cs.level_iterations + cs.levels);
		stats->level_ms.assign(cs.level_ms, cs.level_ms + cs.levels);
		stats->level_initial_residual.assign(cs.level_initial_residual, cs.level_initial_residual + cs.levels);
		stats->total_ms                 = cs.total_ms;
		stats->finest.iterations        = cs.finest.iterations;
		stats->finest.relative_residual = cs.finest.relative_residual;
		stats->finest.true_residual     = cs.finest.true_residual;
		stats->finest.initial_residual  = cs.finest.initial_residual;
		stats->finest.setup_ms          = cs.finest.setup_ms;
		stats->finest.solve_ms          = cs.finest.solve_ms;
		stats->finest.converged         = cs.finest.converged != 0;
		stats->finest.occupied_cells    = cs.finest.occupied_cells;
		stats->finest.generic_rows      = cs.finest.generic_rows;
	}
	return out;
}

bool sample_field(const std::vector<int>& sizes, const float* field, int64_t num_points, const float* positions, GradientKernel kernel,
                  bool want_gradients, std::vector<float>* values, std::vector<float>* gradients)
{
	if (values) { values->clear(); }
	if (gradients) { gradients->clear(); }
	if (values == nullptr || (want_gradients && gradients == nullptr) || sizes.empty() || sizes.size() > 3 || num_points < 0) { return false; }
	const int32_t              ndim = static_cast<int32_t>(sizes.size());
	const std::vector<int32_t> sz(sizes.begin(), sizes.end());
	std::vector<float>         v(static_cast<size_t>(num_points)), g(want_gradients ? static_cast<size_t>(num_points) * ndim : 0);
	if (fi_sample_field(ndim, sz.data(), field, num_points, positions, static_cast<int32_t>(kernel), FI_HOST, v.data(),
	                    want_gradients ? g.data() : nullptr) != FI_OK) {
		return false;
	}
	*values = std::move(v);
	if (want_gradients) { *gradients = std::move(g); }
	return true;
}

std::vector<float> generate_error_map(LatticeField* field, const std::vector<float>& solution, ErrorSums* sums)
{
	if (field == nullptr) { return {}; }
	Structured* st = structured_for_append(field);  // forwards rows appended to field->eq by hand since the last builder call
	if (!st) { return {}; }
	size_t n = 1;
	for (int s : field->sizes) { n *= static_cast<size_t>(s); }
	if (solution.size() != n) { return {}; }
	std::vector<float> heat(n);
	double             s[3] = {0, 0, 0};
	if (fi_field_error_map(st->handle, solution.data(), FI_HOST, heat.data(), s) != FI_OK) { return {}; }
	if (sums) {
		sums->model_rows  = s[0];
		sums->point_rows  = s[1];
		sums->caller_rows = s[2];
	}
	return heat;
}

}  // namespace b200

using b200::build;
using b200::to_c;

// reference field_interpolation.cpp:326-341
void add_field_constraints(LatticeField* field, const Weights& weights)
{
	const fi_weights w = to_c(weights);
	build(field, [&](fi_field* h) { return fi_field_add_model(h, &w); });
}

// reference :57-80 — false when weight == 0 or no corner of the containing cell is inside the lattice
bool add_value_constraint(LatticeField* field, const float pos[], float value, float weight)
{
	return build(field, [&](fi_field* h) {
		       return fi_field_add_points(h, weight, FI_VALUE_LINEAR_INTERPOLATION, 0.0f, FI_GRADIENT_CELL_EDGES, 1, pos, nullptr, nullptr, &value,
		                                  FI_HOST, nullptr);
	       }) > 0;
}

// reference :82-107 — false iff the nearest lattice point is outside; a zero weight still returns true (the
// row is dropped inside add_equation)
bool add_value_constraint_nearest_neighbor(LatticeField* field, const float pos[], const float gradient[], float value, float weight)
{
	for (int d = 0; d < field->num_dim(); ++d) {
		const int nearest = static_cast<int>(std::round(pos[d]));  // :91 (half away from zero)
		if (nearest < 0 || field->sizes[d] <= nearest) { return false; }
	}
	return build(field, [&](fi_field* h) {
		       return fi_field_add_points(h, weight, FI_VALUE_NEAREST_NEIGHBOR, 0.0f, FI_GRADIENT_CELL_EDGES, 1, pos, gradient, nullptr, &value,
		                                  FI_HOST, nullptr);
	       }) >= 0;
}

// reference :123-240
bool add_gradient_constraint(LatticeField* field, const float pos[], const float gradient[], float weight, GradientKernel kernel)
{
	return build(field, [&](fi_field* h) {
		       return fi_field_add_points(h, 0.0f, FI_VALUE_LINEAR_INTERPOLATION, weight, static_cast<int32_t>(kernel), 1, pos, gradient, nullptr,
		                                  nullptr, FI_HOST, nullptr);
	       }) > 0;
}

// reference :343-371
void add_points(LatticeField* field, float value_weight, ValueKernel value_kernel, float gradient_weight, GradientKernel gradient_kernel,
                const int num_points, const float positions[], const float* normals, const float* point_weights)
{
	build(field, [&](fi_field* h) {
		return fi_field_add_points(h, value_weight, static_cast<int32_t>(value_kernel), gradient_weight, static_cast<int32_t>(gradient_kernel),
		                           num_points, positions, normals, point_weights, nullptr, FI_HOST, nullptr);
	});
}

// reference :373-400
LatticeField sdf_from_points(const std::vector<int>& sizes, const Weights& weights, const int num_points, const float positions[],
                             const float* normals, const float* point_weights)
{
	LatticeField field{sizes};
	add_field_constraints(&field, weights);
	add_points(&field, weights.data_pos, weights.value_kernel, weights.data_gradient, weights.gradient_kernel, num_points, positions, normals,
	           point_weights);
	return field;
}

// reference :402-429
std::vector<float> generate_error_map(const std::vector<Triplet>& triplets, const std::vector<float>& solution, const std::vector<float>& rhs)
{
	std::vector<float> heatmap(solution.size(), 0.0f);
	if (fi_error_map(static_cast<int64_t>(triplets.size()), reinterpret_cast<const fi_triplet*>(triplets.data()),
	                 static_cast<int64_t>(solution.size()), solution.data(), static_cast<int64_t>(rhs.size()), rhs.data(), heatmap.data()) != FI_OK) {
		return {};
	}
	return heatmap;
}

// reference :431-485
std::vector<float> upscale_field(const float* field, const std::vector<int>& small_sizes, const std::vector<int>& large_sizes)
{
	size_t n = 1;
	for (int s : large_sizes) { n *= static_cast<size_t>(s); }
	std::vector<float>   out(n);
	std::vector<int32_t> ss(small_sizes.begin(), small_sizes.end()), ls(large_sizes.begin(), large_sizes.end());
	if (ss.size() != ls.size() || fi_upscale_field(static_cast<int32_t>(ss.size()), ss.data(), ls.data(), field, out.data(), FI_HOST) != FI_OK) {
		return {};
	}
	return out;
}

}  // namespace field_interpolation
