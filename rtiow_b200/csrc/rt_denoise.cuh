// rt_denoise.cuh — rtiow_denoise: an edge-avoiding a-trous wavelet filter (Dammertz et al., HPG 2010) over the buffers
// rtiow_render_aov writes, guided by the first hit's albedo, normal and depth.
//
// Every value the filter computes is pinned by include/rtiow_cuda.h: each operation is one correctly rounded fp32 add, sub,
// mul or div (the _rn intrinsics, so nothing contracts into an FMA), min or max, in a fixed order, and the paper's Gaussians are
// Cauchy weights 1 / (1 + D k).  So tests/np_denoise.py restates every output bit in numpy float32.
//
// Three kernels over one pixel per thread: prepare (range checks, demodulation by the albedo, guides packed as float4), one
// level per a-trous step ping-ponging between two float4 buffers, and finish (remodulation, and the frame's own quantisation).
// At 1200x675 the working set (40 B/px in, 48 B/px of float4 buffers) sits in the 126 MB L2, so the level is a plain
// global-memory stencil.
//
// The kernels are templates instantiated only in rt_denoise.cu (denoise_launch): ptxas numbers every function of a module in
// emission order, and kernels added to capi.cu's module shift that numbering and change the SASS of existing render kernels.
#pragma once
#include "rt_device.cuh"

namespace rt {

constexpr float kDenoiseAlbedoFloor = 0x1p-8f;    // demodulation divides by max(albedo, 2^-8)
constexpr float kDenoiseDepthFloor = 0x1p-16f;    // the depth term divides by s max(z_p, z_q, 2^-16)

// 1 / (1 + d k): the edge-stopping weight of a squared distance d at inverse squared width k (0 when k d overflows)
__device__ __forceinline__ float denoise_cauchy(float d, float k) { return __fdiv_rn(1.0f, __fadd_rn(1.0f, __fmul_rn(d, k))); }

// in: colour [n][3], albedo [n][3], normal [n][3], depth [n], as rtiow_render_aov writes them.  Sets *bad when a value lies
// outside the range the AOVs can take (NaN included); writes x = colour / max(albedo, 2^-8) and the guides (normal, depth).
template <int kBlock> __global__ void __launch_bounds__(kBlock) denoise_prepare_kernel(const float* __restrict__ in, size_t n, float4* __restrict__ x,
                                                                          float4* __restrict__ guide, uint32_t* __restrict__ bad)
{
    const size_t i = (size_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= n) return;
    const float* color = in; const float* albedo = in + 3 * n; const float* normal = in + 6 * n; const float* depth = in + 9 * n;
    float xv[3], nv[3];
    bool ok = true;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float col = color[3 * i + c], alb = albedo[3 * i + c], nrm = normal[3 * i + c];
        ok = ok && col >= 0.0f && col <= 4294967296.0f && alb >= 0.0f && alb <= 1.0f && nrm >= -1.0f && nrm <= 1.0f;   // false on NaN
        xv[c] = __fdiv_rn(col, fmaxf(alb, kDenoiseAlbedoFloor));
        nv[c] = nrm;
    }
    const float z = depth[i];
    ok = ok && ((z >= 0.0f && z <= 65536.0f) || z == __int_as_float(0x7f800000));
    if (!ok) *bad = 1u;
    x[i] = make_float4(xv[0], xv[1], xv[2], 0.0f);
    guide[i] = make_float4(nv[0], nv[1], nv[2], z);
}

// One a-trous level at step s: out(p) = sum_q w(p, q) x(q) / sum_q w(p, q) over the 5x5 taps q = p + s (dx, dy) inside the
// image, dy outer and dx inner, w = ((h wc) wn) wz (include/rtiow_cuda.h).  kc, kn, kz: the level's inverse squared widths.
template <int kBlock> __global__ void __launch_bounds__(kBlock) denoise_level_kernel(const float4* __restrict__ xin, const float4* __restrict__ guide,
                                                                        float4* __restrict__ xout, uint32_t width, uint32_t height, uint32_t step,
                                                                        float kc, float kn, float kz)
{
    constexpr float h1[5] = { 0.0625f, 0.25f, 0.375f, 0.25f, 0.0625f };
    const size_t n = (size_t)width * height;
    const size_t i = (size_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= n) return;
    const int64_t px = (int64_t)(i % width), py = (int64_t)(i / width);
    const float4 xp = xin[i], gp = guide[i];
    const float sf = (float)step;
    const bool p_inf = isinf(gp.w);
    float nr = 0.0f, ng = 0.0f, nb = 0.0f, den = 0.0f;
#pragma unroll
    for (int dy = -2; dy <= 2; ++dy) {
        const int64_t qy = py + (int64_t)dy * step;
        if (qy < 0 || qy >= (int64_t)height) continue;
#pragma unroll
        for (int dx = -2; dx <= 2; ++dx) {
            const int64_t qx = px + (int64_t)dx * step;
            if (qx < 0 || qx >= (int64_t)width) continue;
            const size_t q = (size_t)qy * width + (size_t)qx;
            const float4 xq = xin[q], gq = guide[q];
            float d = __fsub_rn(xp.x, xq.x);
            float dc = __fmul_rn(d, d);
            d = __fsub_rn(xp.y, xq.y); dc = __fadd_rn(dc, __fmul_rn(d, d));
            d = __fsub_rn(xp.z, xq.z); dc = __fadd_rn(dc, __fmul_rn(d, d));
            d = __fsub_rn(gp.x, gq.x);
            float dn = __fmul_rn(d, d);
            d = __fsub_rn(gp.y, gq.y); dn = __fadd_rn(dn, __fmul_rn(d, d));
            d = __fsub_rn(gp.z, gq.z); dn = __fadd_rn(dn, __fmul_rn(d, d));
            const bool q_inf = isinf(gq.w);
            float wz;
            if (p_inf || q_inf) {
                wz = p_inf && q_inf ? 1.0f : 0.0f;                  // sky never blends into geometry
            } else {
                const float t = __fdiv_rn(__fsub_rn(gp.w, gq.w), __fmul_rn(sf, fmaxf(fmaxf(gp.w, gq.w), kDenoiseDepthFloor)));
                wz = denoise_cauchy(__fmul_rn(t, t), kz);
            }
            const float h = h1[dy + 2] * h1[dx + 2];                 // exact: a constant product of powers of two and 3/8
            const float w = __fmul_rn(__fmul_rn(__fmul_rn(h, denoise_cauchy(dc, kc)), denoise_cauchy(dn, kn)), wz);
            nr = __fadd_rn(nr, __fmul_rn(w, xq.x));
            ng = __fadd_rn(ng, __fmul_rn(w, xq.y));
            nb = __fadd_rn(nb, __fmul_rn(w, xq.z));
            den = __fadd_rn(den, w);
        }
    }
    xout[i] = make_float4(__fdiv_rn(nr, den), __fdiv_rn(ng, den), __fdiv_rn(nb, den), 0.0f);     // den >= 9/64: the centre tap
}

// y = x max(albedo, 2^-8) into out_color ([n][3], may be NULL) and, quantised as a frame's epilogue quantises a pixel of one
// sample (to_rgba, vec3.rs:404-420), into out_rgba (may be NULL)
template <int kBlock> __global__ void __launch_bounds__(kBlock) denoise_finish_kernel(const float4* __restrict__ x, const float* __restrict__ albedo, size_t n,
                                                                         uint32_t alpha, float* __restrict__ out_color, uint32_t* __restrict__ out_rgba)
{
    const size_t i = (size_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= n) return;
    const float4 v = x[i];
    const float y0 = __fmul_rn(v.x, fmaxf(albedo[3 * i + 0], kDenoiseAlbedoFloor));
    const float y1 = __fmul_rn(v.y, fmaxf(albedo[3 * i + 1], kDenoiseAlbedoFloor));
    const float y2 = __fmul_rn(v.z, fmaxf(albedo[3 * i + 2], kDenoiseAlbedoFloor));
    if (out_color) { out_color[3 * i + 0] = y0; out_color[3 * i + 1] = y1; out_color[3 * i + 2] = y2; }
    if (out_rgba) out_rgba[i] = to_rgba<double>(mk<double>(y0, y1, y2), alpha, 1);
}

// The whole filter on `st` (rt_denoise.cu): prepare, `levels` level kernels and finish.  in: the four input buffers back to
// back (10 n floats); work: 3 n float4 (the ping-pong pair, then the guides); *bad is set when an input is out of range.  The
// sigmas are already narrowed to float; out_color and out_rgba are device buffers or NULL.
cudaError_t denoise_launch(const float* in, float4* work, uint32_t* bad, uint32_t width, uint32_t height, uint32_t levels, float sigma_color,
                           float sigma_normal, float sigma_depth, uint32_t alpha, float* out_color, uint32_t* out_rgba, cudaStream_t st);

}  // namespace rt
