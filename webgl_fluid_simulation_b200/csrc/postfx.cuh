// postfx.cuh — the display-side post-FX of render() (SURVEY §8f rank 1, second half): bloom
// (applyBloom S:1350-1394; shaders S:614-674) and sunrays (applySunrays + blur S:1396-1419; shaders
// S:461-494, S:676-724) and the full display shader with SHADING + BLOOM + SUNRAYS (S:549-612).
//
// Every kernel is one reference blit: one thread per target texel, sources fetched through the
// GL_LINEAR formula of passes.cuh (linear_fetch4).  Arithmetic order follows the GLSL; with the
// library's --fmad=false / IEEE div+sqrt build everything is bit-identical to the CPU oracle except
// the display's pow() (linearToGamma), which is tolerance-checked like splat's exp().
//
// The kernels are templated over the texture storage: float4 / float (fp32 storage) or hs::h4 /
// hs::h1 (FLUID_FLAG_HALF_STORAGE).  The reference creates the bloom FBO, the bloom pyramid and both
// sunrays FBOs with ext.halfFloatTexType (S:1012-1043) and draws the mask into the RGBA16F dye.write
// (S:1300), so in that mode every texel is widened exactly when fetched and every blit's output is
// rounded to fp16 (RN-even, hs::st) when stored; the arithmetic in between is the same fp32 code.
// The dithering texture and the final target are fp32 in both modes.
#pragma once
#include <cuda_runtime.h>

#include "half_passes.cuh"
#include "passes.cuh"

namespace fk {

// texel access by storage type: fp32 as stored; fp16 widened exactly / rounded to nearest even
__device__ __forceinline__ float tex_ld(const float* __restrict__ t, size_t k) { return __ldg(t + k); }
__device__ __forceinline__ float tex_ld(const hs::h1* __restrict__ t, size_t k) { return hs::ld(t + k, 0); }
__device__ __forceinline__ float4 tex_ld(const hs::h4* __restrict__ t, size_t k) { return hs::ld(t + k, 0); }
__device__ __forceinline__ void tex_st(float4* t, size_t k, float4 v) { t[k] = v; }
__device__ __forceinline__ void tex_st(float* t, size_t k, float v) { t[k] = v; }
__device__ __forceinline__ void tex_st(hs::h4* t, size_t k, float4 v) { hs::st(t + k, 0, v); }
__device__ __forceinline__ void tex_st(hs::h1* t, size_t k, float v) { hs::st(t + k, 0, v); }
// the destination texel of an additive blit (blendFunc(ONE, ONE)): a plain load, the thread overwrites it
__device__ __forceinline__ float4 dst_ld(const float4* t, size_t k) { return t[k]; }
__device__ __forceinline__ float4 dst_ld(const hs::h4* t, size_t k) {
    const hs::h4 v = t[k];
    const float2 a = __half22float2(v.a), b = __half22float2(v.b);
    return make_float4(a.x, a.y, b.x, b.y);
}

// linear_fetch4 of passes.cuh on an fp16 RGBA texture: the same taps, weights and add order
__device__ __forceinline__ float4 linear_fetch4(const hs::h4* __restrict__ tex, int W, int H, float uvx, float uvy) {
    const float u = uvx * (float)W - 0.5f, v = uvy * (float)H - 0.5f;
    const float fi = floorf(u), fj = floorf(v);
    const float a = u - fi, b = v - fj;
    const int i0 = texel_index(fi, W), i1 = texel_index(fi + 1.0f, W);
    const int j0 = texel_index(fj, H), j1 = texel_index(fj + 1.0f, H);
    const float w00 = (1.0f - a) * (1.0f - b), w10 = a * (1.0f - b), w01 = (1.0f - a) * b, w11 = a * b;
    const float4 t00 = tex_ld(tex, (size_t)j0 * W + i0), t10 = tex_ld(tex, (size_t)j0 * W + i1);
    const float4 t01 = tex_ld(tex, (size_t)j1 * W + i0), t11 = tex_ld(tex, (size_t)j1 * W + i1);
    float4 r;
    r.x = ((w00 * t00.x + w10 * t10.x) + w01 * t01.x) + w11 * t11.x;
    r.y = ((w00 * t00.y + w10 * t10.y) + w01 * t01.y) + w11 * t11.y;
    r.z = ((w00 * t00.z + w10 * t10.z) + w01 * t01.z) + w11 * t11.z;
    r.w = ((w00 * t00.w + w10 * t10.w) + w01 * t01.w) + w11 * t11.w;
    return r;
}

template <typename T1>
__device__ __forceinline__ float linear_fetch1(const T1* __restrict__ tex, int W, int H, float uvx, float uvy) {
    const float u = uvx * (float)W - 0.5f, v = uvy * (float)H - 0.5f;
    const float fi = floorf(u), fj = floorf(v);
    const float a = u - fi, b = v - fj;
    const int i0 = texel_index(fi, W), i1 = texel_index(fi + 1.0f, W);
    const int j0 = texel_index(fj, H), j1 = texel_index(fj + 1.0f, H);
    const float w00 = (1.0f - a) * (1.0f - b), w10 = a * (1.0f - b), w01 = (1.0f - a) * b, w11 = a * b;
    return ((w00 * tex_ld(tex, (size_t)j0 * W + i0) + w10 * tex_ld(tex, (size_t)j0 * W + i1)) +
            w01 * tex_ld(tex, (size_t)j1 * W + i0)) + w11 * tex_ld(tex, (size_t)j1 * W + i1);
}

// REPEAT-wrapped LINEAR fetch of the first channel of an RGB (3 floats / texel) texture: the
// dithering texture (createTextureAsync S:1128-1158: LINEAR, REPEAT).
__device__ __forceinline__ float linear_fetch_rgb_r_repeat(const float* __restrict__ tex, int W, int H, float uvx, float uvy) {
    const float u = uvx * (float)W - 0.5f, v = uvy * (float)H - 0.5f;
    const float fi = floorf(u), fj = floorf(v);
    const float a = u - fi, b = v - fj;
    long long i0 = (long long)fi % W, j0 = (long long)fj % H;
    if (i0 < 0) i0 += W;
    if (j0 < 0) j0 += H;
    const long long i1 = (i0 + 1) % W, j1 = (j0 + 1) % H;
    const float w00 = (1.0f - a) * (1.0f - b), w10 = a * (1.0f - b), w01 = (1.0f - a) * b, w11 = a * b;
    return ((w00 * __ldg(&tex[((size_t)j0 * W + i0) * 3]) + w10 * __ldg(&tex[((size_t)j0 * W + i1) * 3])) +
            w01 * __ldg(&tex[((size_t)j1 * W + i0) * 3])) + w11 * __ldg(&tex[((size_t)j1 * W + i1) * 3]);
}

// bloomPrefilterShader S:614-631
template <typename T4>
__global__ void __launch_bounds__(256) bloom_prefilter_kernel(const T4* __restrict__ dye, int Wd, int Hd,
                                                              T4* __restrict__ out, int w, int h, float curve0,
                                                              float curve1, float curve2, float threshold) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y * blockDim.y + threadIdx.y;
    if (i >= w || j >= h) return;
    const float uvx = ((float)i + 0.5f) / (float)w, uvy = ((float)j + 0.5f) / (float)h;
    const float4 c = linear_fetch4(dye, Wd, Hd, uvx, uvy);
    const float br = fmaxf(c.x, fmaxf(c.y, c.z));
    float rq = fminf(fmaxf(br - curve0, 0.0f), curve1);
    rq = (curve2 * rq) * rq;
    const float f = fmaxf(rq, br - threshold) / fmaxf(br, 0.0001f);
    tex_st(out, (size_t)j * w + i, make_float4(c.x * f, c.y * f, c.z * f, 0.0f));
}

// bloomBlurShader S:633-651 / bloomFinalShader S:653-674; add = blendFunc(ONE, ONE) (S:1374-1375)
template <typename T4>
__global__ void __launch_bounds__(256) box4_kernel(const T4* __restrict__ src, int ws, int hs,
                                                   T4* __restrict__ dst, int w, int h, float scale, int add) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y * blockDim.y + threadIdx.y;
    if (i >= w || j >= h) return;
    const float tsx = (float)(1.0 / (double)ws), tsy = (float)(1.0 / (double)hs);
    const float uvx = ((float)i + 0.5f) / (float)w, uvy = ((float)j + 0.5f) / (float)h;
    const float4 L = linear_fetch4(src, ws, hs, uvx - tsx, uvy), R = linear_fetch4(src, ws, hs, uvx + tsx, uvy);
    const float4 T = linear_fetch4(src, ws, hs, uvx, uvy + tsy), B = linear_fetch4(src, ws, hs, uvx, uvy - tsy);
    float4 s;
    s.x = ((((0.0f + L.x) + R.x) + T.x) + B.x) * 0.25f * scale;
    s.y = ((((0.0f + L.y) + R.y) + T.y) + B.y) * 0.25f * scale;
    s.z = ((((0.0f + L.z) + R.z) + T.z) + B.z) * 0.25f * scale;
    s.w = ((((0.0f + L.w) + R.w) + T.w) + B.w) * 0.25f * scale;
    const size_t o = (size_t)j * w + i;
    if (add) { const float4 d = dst_ld(dst, o); s.x = s.x + d.x; s.y = s.y + d.y; s.z = s.z + d.z; s.w = s.w + d.w; }
    tex_st(dst, o, s);
}

// sunraysMaskShader S:676-691 (target = dye.write, like the reference: S:1300)
template <typename T4>
__global__ void __launch_bounds__(256) sunrays_mask_kernel(const T4* __restrict__ dye, T4* __restrict__ mask,
                                                           int Wd, int Hd) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y * blockDim.y + threadIdx.y;
    if (i >= Wd || j >= Hd) return;
    const float uvx = ((float)i + 0.5f) / (float)Wd, uvy = ((float)j + 0.5f) / (float)Hd;
    float4 c = linear_fetch4(dye, Wd, Hd, uvx, uvy);
    const float br = fmaxf(c.x, fmaxf(c.y, c.z));
    c.w = 1.0f - fminf(fmaxf(br * 20.0f, 0.0f), 0.8f);
    tex_st(mask, (size_t)j * Wd + i, c);
}

// sunraysShader S:693-724
template <typename T4, typename T1>
__global__ void __launch_bounds__(256) sunrays_kernel(const T4* __restrict__ mask, int Wm, int Hm,
                                                      T1* __restrict__ out, int w, int h, float weight) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y * blockDim.y + threadIdx.y;
    if (i >= w || j >= h) return;
    const float Density = 0.3f, Decay = 0.95f, Exposure = 0.7f;
    const float f = (float)(1.0 / 16.0) * Density;
    const float uvx = ((float)i + 0.5f) / (float)w, uvy = ((float)j + 0.5f) / (float)h;
    float cx = uvx, cy = uvy;
    float dx = uvx - 0.5f, dy = uvy - 0.5f;
    dx = dx * f; dy = dy * f;
    float illum = 1.0f;
    float color = linear_fetch4(mask, Wm, Hm, uvx, uvy).w;
#pragma unroll 1
    for (int k = 0; k < 16; ++k) {
        cx = cx - dx; cy = cy - dy;
        const float col = linear_fetch4(mask, Wm, Hm, cx, cy).w;
        color = color + (col * illum) * weight;
        illum = illum * Decay;
    }
    tex_st(out, (size_t)j * w + i, color * Exposure);
}

// blurShader S:478-494 + blurVertexShader S:461-476 on the one-channel sunrays texture
template <typename T1>
__global__ void __launch_bounds__(256) blur3_kernel(const T1* __restrict__ src, T1* __restrict__ dst, int w, int h,
                                                    float tsx, float tsy) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y * blockDim.y + threadIdx.y;
    if (i >= w || j >= h) return;
    const float off = 1.33333333f;
    const float uvx = ((float)i + 0.5f) / (float)w, uvy = ((float)j + 0.5f) / (float)h;
    const float c = linear_fetch1(src, w, h, uvx, uvy);
    const float l = linear_fetch1(src, w, h, uvx - tsx * off, uvy - tsy * off);
    const float r = linear_fetch1(src, w, h, uvx + tsx * off, uvy + tsy * off);
    float sum = c * 0.29411764f;
    sum = sum + l * 0.35294117f;
    sum = sum + r * 0.35294117f;
    tex_st(dst, (size_t)j * w + i, sum);
}

// displayShaderSource S:549-612 with SHADING + BLOOM + SUNRAYS over drawColor, premultiplied blend;
// the target is fp32 in both storage modes (the unquantised frame fluid_render returns)
template <typename T4, typename T1>
__global__ void __launch_bounds__(256) display_full_kernel(const T4* __restrict__ dye, int Wd, int Hd,
                                                           const T4* __restrict__ bloom, int bw, int bh,
                                                           const T1* __restrict__ sun, int sw, int sh,
                                                           const float* __restrict__ dither, int dw, int dh,
                                                           float4* __restrict__ out, int w, int h, float br_, float bg_,
                                                           float bb_, int bg_mode, float aspect, float4 ts) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y * blockDim.y + threadIdx.y;
    if (i >= w || j >= h) return;
    const float tsx = ts.x, tsy = ts.y;     // 1/width, 1/height (S:1337) and getTextureScale (S:1626-1631): JS doubles, narrowed on the host
    const float dsx = ts.z, dsy = ts.w;
    const float uvx = ((float)i + 0.5f) / (float)w, uvy = ((float)j + 0.5f) / (float)h;
    const float4 c = linear_fetch4(dye, Wd, Hd, uvx, uvy);
    const float4 lc = linear_fetch4(dye, Wd, Hd, uvx - tsx, uvy), rc = linear_fetch4(dye, Wd, Hd, uvx + tsx, uvy);
    const float4 tc = linear_fetch4(dye, Wd, Hd, uvx, uvy + tsy), bc = linear_fetch4(dye, Wd, Hd, uvx, uvy - tsy);
    const float dx = len3(rc) - len3(lc), dy = len3(tc) - len3(bc);
    const float nz = sqrtf(tsx * tsx + tsy * tsy);
    const float nl = sqrtf((dx * dx + dy * dy) + nz * nz);
    const float d = ((dx / nl) * 0.0f + (dy / nl) * 0.0f) + (nz / nl) * 1.0f;
    const float diffuse = fminf(fmaxf(d + 0.7f, 0.7f), 1.0f);
    const float4 bl = linear_fetch4(bloom, bw, bh, uvx, uvy);
    const float s = linear_fetch1(sun, sw, sh, uvx, uvy);
    const float noise = linear_fetch_rgb_r_repeat(dither, dw, dh, uvx * dsx, uvy * dsy) * 2.0f - 1.0f;
    const float cin[3] = {c.x, c.y, c.z}, bin[3] = {bl.x, bl.y, bl.z};
    float cc[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float ck = (cin[k] * diffuse) * s;
        float bk = bin[k] * s;
        bk = bk + noise / 255.0f;
        bk = fmaxf(bk, 0.0f);
        bk = fmaxf(1.055f * powf(bk, 0.416666667f) - 0.055f, 0.0f);     // linearToGamma S:565-568
        cc[k] = ck + bk;
    }
    const float a = fmaxf(cc[0], fmaxf(cc[1], cc[2]));
    out[(size_t)j * w + i] = blend_over_background(cc[0], cc[1], cc[2], a, bg_mode, br_, bg_, bb_, aspect, uvx, uvy);
}

}  // namespace fk
