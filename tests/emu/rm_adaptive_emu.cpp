// rm_adaptive_emu.cpp -- DEV/TEST TOOL, not part of the product and never loaded by it.
//
// rm::adaptive_mark (rusty_marcher_b200/csrc/rm_math.cuh), the per-pixel test of adaptive_mark_kernel, compiled for the
// host, so that the tests can hold it against a numpy restatement of the normative mask without a GPU.
#include <cstddef>

#include "../../rusty_marcher_b200/csrc/rm_math.cuh"

// rgb: (hi - lo, width, 3) floats and id: (hi - lo, width) of the frame rows [lo, hi); mask: (rows, width) bytes for the rows
// [row_begin, row_begin + rows), which must lie in [lo, hi)
extern "C" int emu_adaptive_mark(const float* rgb, const int* id, int width, int lo, int hi, int row_begin, int rows, float k,
                                 int all, unsigned char* mask) {
    if (row_begin < lo || row_begin + rows > hi) return -3;
    for (int r = 0; r < rows; r++)
        for (int x = 0; x < width; x++)
            mask[(size_t)r * width + x] = rm::adaptive_mark(rgb, id, width, lo, hi, x, row_begin + r, k, all != 0) ? 1 : 0;
    return 0;
}
