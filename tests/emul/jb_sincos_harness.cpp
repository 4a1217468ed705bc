// TEST INFRASTRUCTURE ONLY -- see jb_emul_shim.h.  Exports the hot path's inline `jb_sincos` (jiminy_b200/csrc/jb_device.cuh)
// over an array, compiled for the host from the unchanged device source, so that tests/test_kernel_paths.py can measure
// its accuracy against long double.  Build with -ffp-contract=off: the function is written with explicit fma(), products
// and exact subtractions only, so the host build then rounds every operation exactly as the device build does.
#include "jb_emul_shim.h"
#include "jb_device.cuh"

// definitions the device header refers to (never used by jb_sincos; the emulator library defines them for real)
thread_local EmulDim3 threadIdx, blockIdx, blockDim, gridDim;
thread_local double* emul_smem = nullptr;
namespace emul {
thread_local Warp* warp = nullptr;
thread_local int lane_id = 0;
}  // namespace emul
namespace jb { KParams g_kp_host; }

extern "C" void jb_sincos_array(const double* x, double* s, double* c, long long n) {
    for (long long i = 0; i < n; ++i) jb::jb_sincos(x[i], s + i, c + i);
}
