// A C++ caller of b200::sample_field (include/field_interpolation/field_interpolation.hpp), built against the drop-in
// headers and libraries.  Usage: sample_driver IN OUT.  IN: int32 D, int32 sizes[D], int32 kernel (-1: values only),
// int64 N, then prod(sizes) field floats and N*D position floats.  OUT: N values, then N*D gradients (when asked for).
#include <cstdint>
#include <cstdio>
#include <vector>

#include "field_interpolation/field_interpolation.hpp"

int main(int argc, char** argv)
{
	if (argc != 3) { return 2; }
	std::FILE* in = std::fopen(argv[1], "rb");
	if (!in) { return 2; }
	int32_t D = 0, kernel = 0;
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
	if (std::fread(&kernel, 4, 1, in) != 1 || std::fread(&n, 8, 1, in) != 1) { return 2; }
	std::vector<float> field(cells), pos(static_cast<size_t>(n) * D);
	if (std::fread(field.data(), 4, field.size(), in) != field.size() || std::fread(pos.data(), 4, pos.size(), in) != pos.size()) { return 2; }
	std::fclose(in);

	const bool         want = kernel >= 0;
	std::vector<float> values, gradients;
	if (!field_interpolation::b200::sample_field(sizes, field.data(), n, pos.data(),
	                                             static_cast<field_interpolation::GradientKernel>(want ? kernel : 0), want, &values, &gradients)) {
		std::fprintf(stderr, "sample_field failed\n");
		return 1;
	}
	std::FILE* out = std::fopen(argv[2], "wb");
	if (!out) { return 2; }
	std::fwrite(values.data(), 4, values.size(), out);
	std::fwrite(gradients.data(), 4, gradients.size(), out);
	std::fclose(out);
	return 0;
}
