// emul_aov.cpp — TEST INFRASTRUCTURE (tests/test_denoise.py).  k_aov's per-path body (rt_device.cuh aov_path) compiled for the host
// and run over the host-flattened DeviceScene (rt_debug_host_scene), with the kernel's round-to-nearest-even fixed-point sums, so the
// device code of rt_render_aov is checked against the oracle on machines without a GPU.
#include "cuda_shim.h"

#include "../../include/rtb200.h"
#include "../../ray_tracing_series_rust_b200/csrc/cuda/rt_device.cuh"

using namespace rtb;

extern "C" {

uint64_t emul_aov_sizeof_device_scene(void) { return sizeof(DeviceScene); }

// samples [s0, s1) of every pixel of rows [0, rows); wide: the 4-wide walk, as k_aov takes it when the scene carries nodes4
int32_t emul_render_aov(const void* scene, int32_t W, int32_t H, int32_t rows, int32_t spp_total, int32_t s0, int32_t s1, uint64_t seed, int32_t wide,
                        int64_t* albedo, int64_t* normal) {
    const DeviceScene& S = *static_cast<const DeviceScene*>(scene);
    if (wide && !S.nodes4) return -1;
    auto fix = [](double x) { return (int64_t)std::nearbyint(x * 4294967296.0); };
    for (int32_t j = 0; j < rows; ++j)
        for (int32_t ii = 0; ii < W; ++ii)
            for (int32_t sl = s0; sl < s1; ++sl) {
                const uint32_t pixel = (uint32_t)j * (uint32_t)W + (uint32_t)ii;
                const uint64_t path_id = (uint64_t)pixel * (uint64_t)spp_total + (uint64_t)sl;
                D3 a, n;
                if (wide) aov_path<true>(S, ii, j, W, H, seed, path_id, a, n);
                else aov_path<false>(S, ii, j, W, H, seed, path_id, a, n);
                const size_t e = (size_t)pixel * 3;
                albedo[e] += fix(a.x); albedo[e + 1] += fix(a.y); albedo[e + 2] += fix(a.z);
                normal[e] += fix(n.x); normal[e + 1] += fix(n.y); normal[e + 2] += fix(n.z);
            }
    return 0;
}

} // extern "C"
