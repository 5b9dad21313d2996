// rt_denoise.cu — the launches of rtiow_denoise's kernels (rt_denoise.cuh), in a module of their own so that capi.cu's
// kernels compile to the same SASS as without them.
#include "rt_denoise.cuh"

#include <cmath>

namespace rt {

static const int kDenoiseBlock = 256;          // threads per block of the denoise kernels, one pixel each

// 1 / (s s) in float: the inverse squared width of an edge-stopping term (0 for s = +inf)
static float denoise_k(float s) { const float s2 = s * s; return 1.0f / s2; }

cudaError_t denoise_launch(const float* in, float4* work, uint32_t* bad, uint32_t width, uint32_t height, uint32_t levels, float sigma_color,
                           float sigma_normal, float sigma_depth, uint32_t alpha, float* out_color, uint32_t* out_rgba, cudaStream_t st)
{
    const size_t n = (size_t)width * height;
    const unsigned blocks = (unsigned)((n + kDenoiseBlock - 1) / kDenoiseBlock);
    float4* const buf[2] = { work, work + n };
    float4* const guide = work + 2 * n;
    const float kn = denoise_k(sigma_normal), kz = denoise_k(sigma_depth);
    denoise_prepare_kernel<kDenoiseBlock><<<blocks, kDenoiseBlock, 0, st>>>(in, n, buf[0], guide, bad);
    for (uint32_t i = 0; i < levels; ++i) {
        const float kc = denoise_k(sigma_color * std::ldexp(1.0f, -(int)i));      // the colour width halves with every level
        denoise_level_kernel<kDenoiseBlock><<<blocks, kDenoiseBlock, 0, st>>>(buf[i & 1], guide, buf[(i + 1) & 1], width, height, 1u << i, kc, kn, kz);
    }
    denoise_finish_kernel<kDenoiseBlock><<<blocks, kDenoiseBlock, 0, st>>>(buf[levels & 1], in + 3 * n, n, alpha, out_color, out_rgba);
    return cudaGetLastError();
}

}  // namespace rt
