// denoise.cu — the device side of rt_render_aov and rt_render_denoised (sm_100a): the first-hit feature pass (k_aov) and the
// feature-guided a-trous filter over two half accumulators (k_dn_*).  The half renders themselves are launch_render over sample ranges.
//
// k_aov adds integers, so its sums do not depend on scheduling.  The filter gathers from the previous pass's buffers, one thread per
// pixel, with no atomics, in the order ray_tracing_series_rust_b200/denoise.py states; the library is built with -fmad=false, so the
// only differences from that reference are the last bits of exp and sqrt.
#include <algorithm>
#include <cstdint>

#include "kernels.h"
#include "rt_device.cuh"

namespace rtb {

// ---------------------------------------------------------------- feature pass
// One thread per path, sample-major like the render (index = local sample * pixels + pixel), grid-stride.
RT_DEV void add_fixed(int64_t* __restrict__ sums, size_t e, double x) {
    atomicAdd(reinterpret_cast<unsigned long long*>(sums + e), (unsigned long long)__double2ll_rn(x * 4294967296.0));
}

template <bool WIDE>
__global__ void __launch_bounds__(128) k_aov(const __grid_constant__ DeviceScene S, int32_t W, int32_t H, uint32_t npix, int32_t spp_total,
                                             int32_t sample_begin, uint64_t total, uint64_t seed, int64_t* __restrict__ albedo,
                                             int64_t* __restrict__ normal) {
    for (uint64_t L = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; L < total; L += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t s_local = L / npix;
        const uint32_t pix = (uint32_t)(L - s_local * npix);
        const int32_t j = (int32_t)(pix / (uint32_t)W), ii = (int32_t)(pix - (uint32_t)j * (uint32_t)W);
        const uint64_t path_id = (uint64_t)pix * (uint64_t)spp_total + (uint64_t)sample_begin + s_local;
        D3 a, n;
        aov_path<WIDE>(S, ii, j, W, H, seed, path_id, a, n);
        const size_t e = (size_t)pix * 3;
        if (albedo) { add_fixed(albedo, e, a.x); add_fixed(albedo, e + 1, a.y); add_fixed(albedo, e + 2, a.z); }
        if (normal) { add_fixed(normal, e, n.x); add_fixed(normal, e + 1, n.y); add_fixed(normal, e + 2, n.z); }
    }
}

cudaError_t launch_aov(const DeviceScene& scene, const RenderJob& job, int64_t* d_albedo, int64_t* d_normal, cudaStream_t stream) {
    const uint32_t npix = (uint32_t)job.width * (uint32_t)job.rows;
    const uint64_t total = (uint64_t)npix * (uint64_t)(job.sample_end - job.sample_begin);
    if (total == 0) return cudaSuccess;
    const int blocks = (int)std::min<uint64_t>((total + 127) / 128, 148ull * 32ull);
    if (scene.nodes4 != nullptr)
        k_aov<true><<<blocks, 128, 0, stream>>>(scene, job.width, job.height, npix, job.spp_total, job.sample_begin, total, job.seed, d_albedo, d_normal);
    else
        k_aov<false><<<blocks, 128, 0, stream>>>(scene, job.width, job.height, npix, job.spp_total, job.sample_begin, total, job.seed, d_albedo, d_normal);
    return cudaGetLastError();
}

// ---------------------------------------------------------------- filter
RT_DEV double lum(double r, double g, double b) { return (0.2126 * r + 0.7152 * g) + 0.0722 * b; }

// Inputs of the filter: the mean c = ((A+B) 2^-32)(1/n), the noise of the mean v = (lA - lB)^2 hA hB / n^2 from the half means' luminances,
// the feature means albedo 2^-32 / m and normal 2^-32 / m; accum_out = A + B.  Unrendered rows: zeros.
__global__ void k_dn_init(const DenoiseJob J, double kv) {
    const int64_t npix = (int64_t)J.W * J.H;
    const double inv_n = 1.0 / (double)(J.hA + J.hB), inv_a = 1.0 / (double)J.hA, inv_b = 1.0 / (double)J.hB, S = 1.0 / 4294967296.0;
    for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < npix; p += (int64_t)gridDim.x * blockDim.x) {
        const bool on = p / J.W < J.rows;
        double c[3], ma[3], mb[3];
        for (int k = 0; k < 3; ++k) {
            const int64_t a = J.a[3 * p + k], b = J.b[3 * p + k];
            if (J.accum_out) J.accum_out[3 * p + k] = a + b;
            c[k] = ((double)(a + b) * S) * inv_n;
            ma[k] = ((double)a * S) * inv_a;
            mb[k] = ((double)b * S) * inv_b;
            J.c[0][3 * p + k] = on ? c[k] : 0.0;
            J.feat[6 * p + k] = on ? ((double)J.albedo[3 * p + k] * S) / (double)J.m : 0.0;
            J.feat[6 * p + 3 + k] = on ? ((double)J.normal[3 * p + k] * S) / (double)J.m : 0.0;
        }
        const double d = lum(ma[0], ma[1], ma[2]) - lum(mb[0], mb[1], mb[2]);
        J.v[0][p] = on ? (d * d) * kv : 0.0;
    }
}

// vbar = 3x3 blur of v, weights (1/4, 1/2, 1/4) per axis, renormalised over the taps on rendered rows inside the image
__global__ void k_dn_vblur(const double* __restrict__ v, double* __restrict__ vbar, int32_t W, int32_t rows) {
    const int64_t npix = (int64_t)W * rows;
    const double g[3] = {0.25, 0.5, 0.25};
    for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < npix; p += (int64_t)gridDim.x * blockDim.x) {
        const int32_t y = (int32_t)(p / W), x = (int32_t)(p - (int64_t)y * W);
        double s = 0.0, ws = 0.0;
#pragma unroll
        for (int dy = -1; dy <= 1; ++dy) {
            const int32_t qy = y + dy;
            if (qy < 0 || qy >= rows) continue;
#pragma unroll
            for (int dx = -1; dx <= 1; ++dx) {
                const int32_t qx = x + dx;
                if (qx < 0 || qx >= W) continue;
                const double w = g[dy + 1] * g[dx + 1];
                s += w * v[(int64_t)qy * W + qx];
                ws += w;
            }
        }
        vbar[p] = s / ws;
    }
}

// One a-trous pass at step `step`: 25 taps p + step (dx, dy), kernel h = (1/16, 1/4, 3/8, 1/4, 1/16) per axis times the edge stops
// exp(-(|lum(c_p) - lum(c_q)| / (sigma_c sqrt(vbar_p) + 1e-10) + |a_p - a_q|^2 / sigma_a^2 + |n_p - n_q|^2 / sigma_n^2)).
// c' = sum w c_q / sum w, v' = sum w^2 v_q / (sum w)^2; dy outer, dx inner, both ascending.
__global__ void k_dn_atrous(const double* __restrict__ c, const double* __restrict__ v, const double* __restrict__ vbar,
                            const double* __restrict__ feat, double* __restrict__ c_out, double* __restrict__ v_out, int32_t W, int32_t rows,
                            int32_t step, double sigma_c, double sa2, double sn2) {
    const int64_t npix = (int64_t)W * rows;
    const double h[5] = {1.0 / 16.0, 1.0 / 4.0, 3.0 / 8.0, 1.0 / 4.0, 1.0 / 16.0};
    for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < npix; p += (int64_t)gridDim.x * blockDim.x) {
        const int32_t y = (int32_t)(p / W), x = (int32_t)(p - (int64_t)y * W);
        const double cr = c[3 * p], cg = c[3 * p + 1], cb = c[3 * p + 2];
        const double lp = lum(cr, cg, cb);
        const double den = sigma_c * sqrt(vbar[p]) + 1e-10;
        const double* fp = feat + 6 * p;
        const double a0 = fp[0], a1 = fp[1], a2 = fp[2], n0 = fp[3], n1 = fp[4], n2 = fp[5];
        double sw = 0.0, sr = 0.0, sg = 0.0, sb = 0.0, sv = 0.0;
#pragma unroll
        for (int dy = -2; dy <= 2; ++dy) {
            const int32_t qy = y + dy * step;
            if (qy < 0 || qy >= rows) continue;
#pragma unroll
            for (int dx = -2; dx <= 2; ++dx) {
                const int32_t qx = x + dx * step;
                if (qx < 0 || qx >= W) continue;
                const int64_t q = (int64_t)qy * W + qx;
                const double qr = c[3 * q], qg = c[3 * q + 1], qb = c[3 * q + 2];
                const double* fq = feat + 6 * q;
                const double da0 = a0 - fq[0], da1 = a1 - fq[1], da2 = a2 - fq[2];
                const double dn0 = n0 - fq[3], dn1 = n1 - fq[4], dn2 = n2 - fq[5];
                const double da = (da0 * da0 + da1 * da1) + da2 * da2;
                const double dn = (dn0 * dn0 + dn1 * dn1) + dn2 * dn2;
                const double e = (fabs(lp - lum(qr, qg, qb)) / den + da / sa2) + dn / sn2;
                const double w = (h[dx + 2] * h[dy + 2]) * exp(-e);
                sw += w;
                sr += w * qr; sg += w * qg; sb += w * qb;
                sv += (w * w) * v[q];
            }
        }
        c_out[3 * p] = sr / sw; c_out[3 * p + 1] = sg / sw; c_out[3 * p + 2] = sb / sw;
        v_out[p] = sv / (sw * sw);
    }
}

// the filtered mean and its Screen bytes (screen_value, as every resolve); unrendered rows stay 0
__global__ void k_dn_out(const double* __restrict__ c, double* __restrict__ linear_out, uint8_t* __restrict__ screen_u8, int32_t W, int32_t H, int32_t rows) {
    const int64_t n = (int64_t)W * H * 3, rendered = (int64_t)W * rows * 3;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double x = i < rendered ? c[i] : 0.0;
        if (linear_out) linear_out[i] = x;
        if (screen_u8) screen_u8[i] = (uint8_t)(i < rendered ? screen_value(x) : 0.0);
    }
}

static int grid_for(uint64_t n, int per_block) { return (int)std::max<uint64_t>(1, std::min<uint64_t>((n + per_block - 1) / per_block, 148ull * 16ull)); }

cudaError_t launch_denoise(const DenoiseJob& j, cudaStream_t stream) {
    const uint64_t npix = (uint64_t)j.W * j.H, rendered = (uint64_t)j.W * j.rows;
    const int64_t n = (int64_t)j.hA + j.hB;
    const double kv = (double)((int64_t)j.hA * j.hB) / (double)(n * n);
    k_dn_init<<<grid_for(npix, 256), 256, 0, stream>>>(j, kv);
    const double sa2 = j.sigma_albedo * j.sigma_albedo, sn2 = j.sigma_normal * j.sigma_normal;
    for (int32_t it = 0; it < j.iterations && rendered > 0; ++it) {
        const int cur = it & 1;
        k_dn_vblur<<<grid_for(rendered, 256), 256, 0, stream>>>(j.v[cur], j.vbar, j.W, j.rows);
        k_dn_atrous<<<grid_for(rendered, 128), 128, 0, stream>>>(j.c[cur], j.v[cur], j.vbar, j.feat, j.c[cur ^ 1], j.v[cur ^ 1], j.W, j.rows, 1 << it,
                                                               j.sigma_color, sa2, sn2);
    }
    k_dn_out<<<grid_for(npix * 3, 256), 256, 0, stream>>>(j.c[j.iterations & 1], j.linear_out, j.screen_u8, j.W, j.H, j.rows);
    return cudaGetLastError();
}

} // namespace rtb
