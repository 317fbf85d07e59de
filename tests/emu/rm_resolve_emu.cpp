// rm_resolve_emu.cpp -- DEV/TEST TOOL, not part of the product and never loaded by it.
//
// rm::resolve_box (rusty_marcher_b200/csrc/rm_math.cuh), the per-pixel arithmetic of resolve_box_kernel, compiled for the
// host, so that the tests can hold it against a numpy restatement of the normative order without a GPU.
#include <cstddef>

#include "../../rusty_marcher_b200/csrc/rm_math.cuh"

namespace {
template <int S> void resolve(const float* sub, int width, int rows, float* out) {
    const size_t sub_row = (size_t)S * width * 3;
    for (int y = 0; y < rows; y++)
        for (int x = 0; x < width; x++) {
            const float* p = sub + (size_t)S * y * sub_row + (size_t)S * 3 * x;
            rm::resolve_box<S>([&](int i, float (&r)[3 * S]) {
                for (int k = 0; k < 3 * S; k++) r[k] = p[i * sub_row + k];
            }, out + ((size_t)y * width + x) * 3);
        }
}
}  // namespace

// sub: (samples * rows, samples * width, 3) floats; out: (rows, width, 3)
extern "C" int emu_resolve_box(const float* sub, int samples, int width, int rows, float* out) {
    switch (samples) {
        case 1: resolve<1>(sub, width, rows, out); return 0;
        case 2: resolve<2>(sub, width, rows, out); return 0;
        case 3: resolve<3>(sub, width, rows, out); return 0;
        case 4: resolve<4>(sub, width, rows, out); return 0;
        case 5: resolve<5>(sub, width, rows, out); return 0;
        case 6: resolve<6>(sub, width, rows, out); return 0;
        case 7: resolve<7>(sub, width, rows, out); return 0;
        case 8: resolve<8>(sub, width, rows, out); return 0;
        default: return -3;
    }
}
