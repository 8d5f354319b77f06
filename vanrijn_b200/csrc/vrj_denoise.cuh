// vrj_denoise.cuh -- the edge-avoiding a-trous filter of vrj_denoise, guided by the per-pixel variance of the mean Y.
// include/vanrijn_cuda.h states the filter operation by operation; these kernels follow it in that order, so a caller can
// replay it (tests/test_gpu_denoise.py does, in numpy).
//
// Per pixel the filter keeps (X, Y, Z, var) as one double4 (32 bytes) and ping-pongs two such buffers.  An invalid pixel
// (header: n < 2, or c / var not finite) is marked by var = -1: a valid var is never negative (v is clamped at 0 and the
// weights are positive), so the mark costs no extra array and every tap tests it with the load it needs anyway.
#pragma once
#include "vrj_device.cuh"

namespace vrj {

struct DenoiseGuides {
    const double *normal; // 3 per pixel
    const double *depth;
    const int32_t *material;
};

// c = s * (1/n), var = v * (1/n) with adaptive_converged's v
static __global__ void k_denoise_init(const double *__restrict__ sum, const double *__restrict__ weight, const double *__restrict__ ysq,
                               uint32_t npix, double4 *__restrict__ out) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= npix) return;
    const double n = weight[p], sx = sum[3 * (size_t)p], sy = sum[3 * (size_t)p + 1], sz = sum[3 * (size_t)p + 2], q = ysq[p];
    const double inv = 1.0 / n;
    const double cx = sx * inv, cy = sy * inv, cz = sz * inv;
    const double m = sy * inv;
    double v = (q - sy * m) / (n - 1.0);
    if (v < 0.0) v = 0.0;
    double var = v * inv;
    if (!(n >= 2.0) || !isfinite(cx) || !isfinite(cy) || !isfinite(cz) || !isfinite(var)) var = -1.0;
    out[p] = make_double4(cx, cy, cz, var);
}

// the B3-spline taps h = {1/16, 1/4, 3/8, 1/4, 1/16} at offset -2..2 (a function, not an array: no local-memory stack frame)
__device__ __forceinline__ double atrous_h(int d) { return d == 0 ? 3.0 / 8.0 : (d == 1 || d == -1) ? 1.0 / 4.0 : 1.0 / 16.0; }

// one iteration at `step`.  A block of 256 threads covers 32 x 8 pixels (blocks_x of them per row of blocks), so its taps
// share cache lines in both directions; one grid dimension keeps any tile shape within the launch limits.
static __global__ void __launch_bounds__(256) k_denoise_step(const double4 *__restrict__ in, double4 *__restrict__ out, DenoiseGuides g,
                                                             uint32_t tw, uint32_t th, uint32_t blocks_x, int step, double sigma_l,
                                                             double sigma_n, double sigma_z) {
    const uint32_t by = blockIdx.x / blocks_x, bx = blockIdx.x - by * blocks_x;
    const uint32_t x = bx * 32 + (threadIdx.x & 31), y = by * 8 + (threadIdx.x >> 5);
    if (x >= tw || y >= th) return;
    const size_t p = (size_t)y * tw + x;
    const double4 cp = in[p];
    if (cp.w < 0.0) { // invalid: keeps its input colour
        out[p] = cp;
        return;
    }
    const int32_t id_p = g.material[p];
    const D3 n_p = d3(g.normal[3 * p], g.normal[3 * p + 1], g.normal[3 * p + 2]);
    const double z_p = g.depth[p];
    const double lum_den = sigma_l * sqrt(cp.w) + 1e-10;
    double W = 0.0, Cx = 0.0, Cy = 0.0, Cz = 0.0, V = 0.0;
#pragma unroll 1
    for (int dy = -2; dy <= 2; dy++) {
        const long long qy = (long long)y + (long long)step * dy;
        if (qy < 0 || qy >= (long long)th) continue;
#pragma unroll 1
        for (int dx = -2; dx <= 2; dx++) {
            const long long qx = (long long)x + (long long)step * dx;
            if (qx < 0 || qx >= (long long)tw) continue;
            const size_t q = (size_t)qy * tw + (size_t)qx;
            const double4 cq = in[q];
            if (cq.w < 0.0) continue;
            double w = atrous_h(dx) * atrous_h(dy);
            if (q != p) {
                if (g.material[q] != id_p) continue;
                if (id_p >= 0) {
                    const D3 n_q = d3(g.normal[3 * q], g.normal[3 * q + 1], g.normal[3 * q + 2]);
                    w = w * pow(fmax(0.0, dot(n_p, n_q)), sigma_n);
                    const int dist = max(abs(dx), abs(dy));
                    w = w * exp(-fabs(z_p - g.depth[q]) / (((sigma_z * z_p) * (double)step) * (double)dist));
                }
                w = w * exp(-fabs(cp.y - cq.y) / lum_den);
            }
            W = W + w;
            Cx = Cx + w * cq.x, Cy = Cy + w * cq.y, Cz = Cz + w * cq.z;
            V = V + (w * w) * cq.w;
        }
    }
    const double inv = 1.0 / W;
    out[p] = make_double4(Cx * inv, Cy * inv, Cz * inv, V * (1.0 / (W * W)));
}

// the colours of the last iteration, 3 doubles per pixel
static __global__ void k_denoise_colour(const double4 *__restrict__ in, uint32_t npix, double *__restrict__ colour) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= npix) return;
    const double4 c = in[p];
    colour[3 * (size_t)p] = c.x, colour[3 * (size_t)p + 1] = c.y, colour[3 * (size_t)p + 2] = c.z;
}

} // namespace vrj
