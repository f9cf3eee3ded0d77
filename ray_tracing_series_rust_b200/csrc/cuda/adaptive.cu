// adaptive.cu — the device side of rt_render_adaptive / rt_render_adaptive_multi (sm_100a): convergence test, dilation, ordered
// compaction of the active pixel list, and the resolve with per-pixel sample counts.  The render rounds themselves are launch_render
// over a pixel list (kernels.cu, shard_pixel); the error test and the resolve read the half accumulators of every GPU (AdaptiveShards).
//
// Every decision is made from integer sums with correctly rounded f64 operations (the library is built with -fmad=false), so the
// active set of every round is the one ray_tracing_series_rust_b200/adaptive.py computes on the host, whatever the render mode.
#include <cub/device/device_select.cuh>

#include <algorithm>
#include <cstdint>

#include "kernels.h"

namespace rtb {

__global__ void k_adaptive_iota(uint32_t* __restrict__ list, uint32_t n) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) list[i] = i;
}

// The int64 components of pixel p summed over the shards, 128 bits per load where the 24-byte pixel allows it (even p: 16 + 8 bytes,
// odd p: 8 + 16).  ld.cg: a shard may be a peer GPU's memory, rewritten by its renders between check points.
__device__ __forceinline__ void shard_pixel_sum(const int64_t* const* P, int32_t n, uint32_t p, long long& r, long long& g, long long& b) {
    r = 0; g = 0; b = 0;
    const size_t e = 3 * (size_t)p;
    for (int32_t k = 0; k < n; ++k) {
        const long long* q = reinterpret_cast<const long long*>(P[k] + e);
        if (!(p & 1u)) {
            const longlong2 v = __ldcg(reinterpret_cast<const longlong2*>(q));
            r += v.x; g += v.y; b += __ldcg(q + 2);
        } else {
            const longlong2 v = __ldcg(reinterpret_cast<const longlong2*>(q + 1));
            r += __ldcg(q); g += v.x; b += v.y;
        }
    }
}

// U[p] = 1 for every active pixel p whose half-buffer error is not below tau (NaN included).  h = samples in each of A and B.  A and B
// are the sums over the shards: integer, so the f64 arithmetic below sees the same values for any shard count.
__global__ void k_adaptive_error(const AdaptiveShards H, const uint32_t* __restrict__ list, uint32_t n_active, int32_t h, double tau,
                                 uint8_t* __restrict__ U) {
    const double S = (double)h * 4294967296.0;
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < n_active; q += gridDim.x * blockDim.x) {
        const uint32_t p = list[q];
        long long sar, sag, sab, sbr, sbg, sbb;
        shard_pixel_sum(H.a, H.n, p, sar, sag, sab);
        shard_pixel_sum(H.b, H.n, p, sbr, sbg, sbb);
        const double ar = (double)sar, ag = (double)sag, ab = (double)sab;
        const double br = (double)sbr, bg = (double)sbg, bb = (double)sbb;
        const double d = (fabs(ar - br) + fabs(ag - bg)) + fabs(ab - bb);
        const double t = ((ar + br) + (ag + bg)) + (ab + bb);
        const double err = (d / S) / sqrt(1e-4 + t / (2.0 * S));
        U[p] = !(err < tau) ? 1 : 0;
    }
}

// An active pixel stays active iff some pixel of U lies within Chebyshev distance `radius` on a rendered row; a pixel that leaves
// gets its final sample count n.  keep[q] is the flag of list position q for the compaction.
__global__ void k_adaptive_keep(const uint32_t* __restrict__ list, uint32_t n_active, const uint8_t* __restrict__ U, int32_t W, int32_t rows,
                                int32_t radius, int32_t n, uint8_t* __restrict__ keep, int32_t* __restrict__ samples) {
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < n_active; q += gridDim.x * blockDim.x) {
        const uint32_t p = list[q];
        const int32_t y = (int32_t)(p / (uint32_t)W), x = (int32_t)(p - (uint32_t)y * (uint32_t)W);
        const int32_t y0 = max(0, y - radius), y1 = min(rows - 1, y + radius);
        const int32_t x0 = max(0, x - radius), x1 = min(W - 1, x + radius);
        bool hit = false;
        for (int32_t yy = y0; yy <= y1 && !hit; ++yy)
            for (int32_t xx = x0; xx <= x1; ++xx)
                if (U[(size_t)yy * W + xx]) { hit = true; break; }
        keep[q] = hit ? 1 : 0;
        if (!hit) samples[p] = n;
    }
}

__global__ void k_adaptive_fill(const uint32_t* __restrict__ list, uint32_t n_active, int32_t n, int32_t* __restrict__ samples) {
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < n_active; q += gridDim.x * blockDim.x) samples[list[q]] = n;
}

// accum_out = the sum of every shard's A + B; the Screen bytes with k_resolve's arithmetic and the pixel's own sample count (0 samples:
// an unrendered compat_threads row, black).  Pairs of channels: 16-byte loads, as in k_reduce_resolve.
__global__ void __launch_bounds__(256) k_resolve_adaptive(const AdaptiveShards H, const int32_t* __restrict__ samples, int64_t* __restrict__ accum_out,
                                                          uint8_t* __restrict__ screen_u8, int32_t W, int32_t Hgt) {
    const int64_t n = (int64_t)W * Hgt * 3, n2 = (n + 1) >> 1;
    for (int64_t i2 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i2 < n2; i2 += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = 2 * i2;
        const bool pair = i + 1 < n;
        long long s[2] = {0, 0};
        for (int32_t g = 0; g < H.n; ++g) {
            if (pair) {
                const longlong2 a = __ldcg(reinterpret_cast<const longlong2*>(H.a[g] + i)), b = __ldcg(reinterpret_cast<const longlong2*>(H.b[g] + i));
                s[0] += a.x + b.x; s[1] += a.y + b.y;
            } else {
                s[0] += __ldcg(reinterpret_cast<const long long*>(H.a[g] + i)) + __ldcg(reinterpret_cast<const long long*>(H.b[g] + i));
            }
        }
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            if (k == 1 && !pair) break;
            const int64_t e = i + k;
            const int32_t np = samples[e / 3];
            double out = 0.0;
            if (np > 0) {
                const double sum = (double)s[k] * (1.0 / 4294967296.0);
                double c = sqrt(sum * (1.0 / (double)np));
                c = c < 0.0 ? 0.0 : (c > 1.0 ? 1.0 : c);     // mutil.rs:1-9 (NaN passes through)
                const double q = 255.9 * c;
                out = (q != q) ? 0.0 : (double)(int32_t)q;    // `as i32`: truncation, NaN -> 0
            }
            accum_out[e] = s[k];
            screen_u8[e] = (uint8_t)out;
        }
    }
}

// the kernels' 128-bit loads need every shard 16-byte aligned: a misaligned one is refused here instead of faulting the context
static bool shards_aligned(const AdaptiveShards& sh) {
    for (int32_t g = 0; g < sh.n; ++g)
        if ((reinterpret_cast<uintptr_t>(sh.a[g]) | reinterpret_cast<uintptr_t>(sh.b[g])) & 15u) return false;
    return true;
}

static int grid_for(uint64_t n, int per_block) { return (int)std::max<uint64_t>(1, std::min<uint64_t>((n + per_block - 1) / per_block, 148ull * 16ull)); }

cudaError_t launch_adaptive_iota(uint32_t* d_list, uint32_t n, cudaStream_t stream) {
    k_adaptive_iota<<<grid_for(n, 256), 256, 0, stream>>>(d_list, n);
    return cudaGetLastError();
}

size_t adaptive_select_temp_bytes(uint32_t max_items) {
    size_t bytes = 0;
    cub::DeviceSelect::Flagged(nullptr, bytes, (const uint32_t*)nullptr, (const uint8_t*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr, (int)max_items);
    return bytes;
}

cudaError_t launch_adaptive_check(const AdaptiveCheck& c, cudaStream_t stream) {
    if (!shards_aligned(c.shards)) return cudaErrorMisalignedAddress;
    cudaError_t e;
    if ((e = cudaMemsetAsync(c.d_u, 0, (size_t)c.W * c.rows, stream)) != cudaSuccess) return e;
    const int g = grid_for(c.n_active, 256);
    k_adaptive_error<<<g, 256, 0, stream>>>(c.shards, c.d_list_in, c.n_active, c.n / 2, c.threshold, c.d_u);
    k_adaptive_keep<<<g, 256, 0, stream>>>(c.d_list_in, c.n_active, c.d_u, c.W, c.rows, c.radius, c.n, c.d_keep, c.d_samples);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    size_t bytes = c.temp_bytes;
    // stable: the next list keeps ascending pixel order (coherent primary rays in the next rounds)
    return cub::DeviceSelect::Flagged(c.d_temp, bytes, c.d_list_in, c.d_keep, c.d_list_out, c.count_out, (int)c.n_active, stream);
}

cudaError_t launch_adaptive_fill(const uint32_t* d_list, uint32_t n_active, int32_t n, int32_t* d_samples, cudaStream_t stream) {
    if (n_active == 0) return cudaSuccess;
    k_adaptive_fill<<<grid_for(n_active, 256), 256, 0, stream>>>(d_list, n_active, n, d_samples);
    return cudaGetLastError();
}

cudaError_t launch_resolve_adaptive(const AdaptiveShards& shards, const int32_t* d_samples, int64_t* d_accum_out, uint8_t* d_screen_u8, int32_t W,
                                    int32_t H, cudaStream_t stream) {
    if (!shards_aligned(shards)) return cudaErrorMisalignedAddress;
    k_resolve_adaptive<<<grid_for(((uint64_t)W * H * 3 + 1) / 2, 256), 256, 0, stream>>>(shards, d_samples, d_accum_out, d_screen_u8, W, H);
    return cudaGetLastError();
}

} // namespace rtb
