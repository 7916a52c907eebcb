// Bandwidth-bound small-channel 3x3 convolutions (3->64 stem, 64->3 heads, 3->3r^2 sub-pixel, 3->3 + add).
// Reference call sites: conv1 (WindowTransformer/model.py:200,244; FastTransformer/model.py:202,251;
// ResidualTransformer/model.py:83,128), decoder_conv2 (W:222,298; F:229,313; R:112,157),
// up1_conv = BasicConv 64->3 no-bias + ReLU (FastTransformer/utils.py:13-40; model.py:208,265),
// final_upscale = Upsampler(n_feats=3) (utils.py:43-98; model.py:211,316), final_upscale_conv + sum
// + clamp (model.py:212,317-327).
#include "tu_common.cuh"
#include "tc/tc_api.cuh"

namespace tu {

// ------------------------------------------------------------------ conv1: 3 -> 64, + ReLU
// NCHW image (TI) -> NHWC features (T).  16x16 pixel tile per CTA, one pixel per thread, the 27x64
// filter bank broadcast from shared memory.
template <typename TI, typename T>
__global__ void __launch_bounds__(256) stem_conv_kernel(const TI *__restrict__ x, const float *__restrict__ w,
                                                        const float *__restrict__ bias, T *__restrict__ out, int H, int W) {
    __shared__ float ws[27 * 64];
    __shared__ float bs[64];
    __shared__ float in_s[3][18][19];
    const int tid = threadIdx.x;
    const int b = blockIdx.z;
    const int y0 = blockIdx.y * 16, x0 = blockIdx.x * 16;
    for (int i = tid; i < 27 * 64; i += 256) ws[i] = w[i];
    if (tid < 64) bs[tid] = bias[tid];
    for (int i = tid; i < 3 * 18 * 18; i += 256) {
        int c = i / 324, r = (i % 324) / 18, cc = i % 18;
        int y = y0 + r - 1, xx = x0 + cc - 1;
        float v = 0.f;
        if (y >= 0 && y < H && xx >= 0 && xx < W) v = to_f(x[(((long)b * 3 + c) * H + y) * W + xx]);
        in_s[c][r][cc] = v;
    }
    __syncthreads();
    const int ly = tid >> 4, lx = tid & 15;
    const int y = y0 + ly, xx = x0 + lx;
    if (y >= H || xx >= W) return;
    float v[27];
#pragma unroll
    for (int ky = 0; ky < 3; ++ky)
#pragma unroll
        for (int kx = 0; kx < 3; ++kx)
#pragma unroll
            for (int c = 0; c < 3; ++c) v[(ky * 3 + kx) * 3 + c] = in_s[c][ly + ky][lx + kx];
    T *o = out + (((long)b * H + y) * W + xx) * 64;
#pragma unroll 1
    for (int g = 0; g < 4; ++g) {
        float acc[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) acc[j] = 0.f;
#pragma unroll
        for (int t = 0; t < 27; ++t) {
#pragma unroll
            for (int j = 0; j < 16; ++j) acc[j] = fmaf(v[t], ws[t * 64 + g * 16 + j], acc[j]);
        }
#pragma unroll
        for (int j = 0; j < 16; j += 4) {
            float4 r = make_float4(fmaxf(acc[j] + bs[g * 16 + j], 0.f), fmaxf(acc[j + 1] + bs[g * 16 + j + 1], 0.f),
                                   fmaxf(acc[j + 2] + bs[g * 16 + j + 2], 0.f), fmaxf(acc[j + 3] + bs[g * 16 + j + 3], 0.f));
            store4(o + g * 16 + j, r);
        }
    }
}

// ------------------------------------------------------------------ 64 -> 3 (decoder_conv2, up1_conv)
// NHWC(64) T -> planar fp32 (B,3,H,W).  One pixel per thread; weights [tap][ci][3] in shared memory.
template <typename T>
__global__ void __launch_bounds__(128) conv64to3_kernel(const T *__restrict__ in, const float *__restrict__ w,
                                                        const float *__restrict__ bias, float *__restrict__ out, int H, int W,
                                                        int relu) {
    __shared__ float ws[9 * 64 * 3];
    for (int i = threadIdx.x; i < 9 * 64 * 3; i += 128) ws[i] = w[i];
    __syncthreads();
    const int b = blockIdx.z;
    const int y = blockIdx.y;
    const int x = blockIdx.x * 128 + threadIdx.x;
    if (x >= W) return;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f;
#pragma unroll 1
    for (int tap = 0; tap < 9; ++tap) {
        int iy = y + tap / 3 - 1, ix = x + tap % 3 - 1;
        if (iy < 0 || iy >= H || ix < 0 || ix >= W) continue;
        const T *p = in + (((long)b * H + iy) * W + ix) * 64;
        const float *wt = ws + tap * 192;
#pragma unroll
        for (int c = 0; c < 64; c += 4) {
            float4 v = load4(p + c);
            a0 = fmaf(v.x, wt[(c + 0) * 3 + 0], a0); a1 = fmaf(v.x, wt[(c + 0) * 3 + 1], a1); a2 = fmaf(v.x, wt[(c + 0) * 3 + 2], a2);
            a0 = fmaf(v.y, wt[(c + 1) * 3 + 0], a0); a1 = fmaf(v.y, wt[(c + 1) * 3 + 1], a1); a2 = fmaf(v.y, wt[(c + 1) * 3 + 2], a2);
            a0 = fmaf(v.z, wt[(c + 2) * 3 + 0], a0); a1 = fmaf(v.z, wt[(c + 2) * 3 + 1], a1); a2 = fmaf(v.z, wt[(c + 2) * 3 + 2], a2);
            a0 = fmaf(v.w, wt[(c + 3) * 3 + 0], a0); a1 = fmaf(v.w, wt[(c + 3) * 3 + 1], a1); a2 = fmaf(v.w, wt[(c + 3) * 3 + 2], a2);
        }
    }
    if (bias) { a0 += bias[0]; a1 += bias[1]; a2 += bias[2]; }
    if (relu) { a0 = fmaxf(a0, 0.f); a1 = fmaxf(a1, 0.f); a2 = fmaxf(a2, 0.f); }
    long plane = (long)H * W, o = (long)b * 3 * plane + (long)y * W + x;
    out[o] = a0; out[o + plane] = a1; out[o + 2 * plane] = a2;
}

// ------------------------------------------------------------------ 3 -> 3 r^2 + PixelShuffle(r)
// planar fp32 (B,3,H,W) -> planar fp32 (B,3,rH,rW).  One OUTPUT (high-res) pixel per thread:
// out[c, y*r+i, x*r+j] = b[c*r*r+i*r+j] + sum_{tap,ci} w[tap*3+ci][c*r*r+i*r+j] * in[ci, y+ky-1, x+kx-1].
__global__ void __launch_bounds__(256) conv3_ps_kernel(const float *__restrict__ in, const float *__restrict__ w,
                                                       const float *__restrict__ bias, float *__restrict__ out, int H, int W, int r) {
    extern __shared__ float ws[];   // 27 * 3r^2 weights + 3r^2 bias
    const int nco = 3 * r * r;
    for (int i = threadIdx.x; i < 27 * nco; i += 256) ws[i] = w[i];
    for (int i = threadIdx.x; i < nco; i += 256) ws[27 * nco + i] = bias[i];
    __syncthreads();
    const int b = blockIdx.z;
    const int oH = H * r, oW = W * r;
    const int ox = blockIdx.x * 64 + (threadIdx.x & 63);
    const int oy = blockIdx.y * 4 + (threadIdx.x >> 6);
    if (ox >= oW || oy >= oH) return;
    const int y = oy / r, i = oy % r, x = ox / r, j = ox % r;
    float v[27];
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) {
        int iy = y + tap / 3 - 1, ix = x + tap % 3 - 1;
        bool ok = iy >= 0 && iy < H && ix >= 0 && ix < W;
#pragma unroll
        for (int c = 0; c < 3; ++c) v[tap * 3 + c] = ok ? in[(((long)b * 3 + c) * H + iy) * W + ix] : 0.f;
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        int co = c * r * r + i * r + j;
        float acc = 0.f;
#pragma unroll
        for (int t = 0; t < 27; ++t) acc = fmaf(v[t], ws[t * nco + co], acc);
        out[(((long)b * 3 + c) * oH + oy) * oW + ox] = acc + ws[27 * nco + co];
    }
}

// ------------------------------------------------------------------ 3 -> 3 conv + addend (+ clamp) -> image
template <typename TO>
__global__ void __launch_bounds__(256) final_conv_add_kernel(const float *__restrict__ in, const float *__restrict__ w,
                                                             const float *__restrict__ bias, const float *__restrict__ addend,
                                                             TO *__restrict__ out, int H, int W, int clamp) {
    __shared__ float ws[27 * 3 + 3];
    if (threadIdx.x < 81) ws[threadIdx.x] = w[threadIdx.x];
    if (threadIdx.x < 3) ws[81 + threadIdx.x] = bias[threadIdx.x];
    __syncthreads();
    const int b = blockIdx.z;
    const int x = blockIdx.x * 64 + (threadIdx.x & 63);
    const int y = blockIdx.y * 4 + (threadIdx.x >> 6);
    if (x >= W || y >= H) return;
    float a[3] = {0.f, 0.f, 0.f};
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) {
        int iy = y + tap / 3 - 1, ix = x + tap % 3 - 1;
        if (iy < 0 || iy >= H || ix < 0 || ix >= W) continue;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            float v = in[(((long)b * 3 + c) * H + iy) * W + ix];
#pragma unroll
            for (int co = 0; co < 3; ++co) a[co] = fmaf(v, ws[(tap * 3 + c) * 3 + co], a[co]);
        }
    }
#pragma unroll
    for (int co = 0; co < 3; ++co) {
        long o = (((long)b * 3 + co) * H + y) * W + x;
        // reference: out = upscaled_input + (conv + bias)   (FastTransformer/model.py:320)
        float r = addend[o] + (a[co] + ws[81 + co]);
        if (clamp) r = fminf(fmaxf(r, 0.f), 1.f);
        out[o] = from_f<TO>(r);
    }
}

}  // namespace tu

using namespace tu;

extern "C" int tu_stem_conv(const void *x, int in_dtype, const float *w27x64, const void *w64, const float *b, void *out,
                            int dtype, int B, int H, int W, void *stream) {
    TU_CHECK_ARG(x && w27x64 && b && out && B > 0 && H > 0 && W > 0, "stem_conv: bad argument");
    TU_CHECK_ARG(in_dtype == TU_F32 || in_dtype == TU_BF16 || in_dtype == TU_F16 || in_dtype == TU_U8, "stem_conv: bad input dtype");
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == TU_BF16 && w64 && tc_enabled()) {
        int rc = tc_stem_conv(x, in_dtype, (const bf16 *)w64, b, (bf16 *)out, B, H, W, st);
        if (rc != TU_TC_UNSUPPORTED) return rc;
    }
    dim3 grid(ceil_div(W, 16), ceil_div(H, 16), B);
    if (in_dtype == TU_F32 && dtype == TU_F32)
        stem_conv_kernel<float, float><<<grid, 256, 0, st>>>((const float *)x, w27x64, b, (float *)out, H, W);
    else if (in_dtype == TU_F32 && dtype == TU_BF16)
        stem_conv_kernel<float, bf16><<<grid, 256, 0, st>>>((const float *)x, w27x64, b, (bf16 *)out, H, W);
    else if (in_dtype == TU_BF16 && dtype == TU_BF16)
        stem_conv_kernel<bf16, bf16><<<grid, 256, 0, st>>>((const bf16 *)x, w27x64, b, (bf16 *)out, H, W);
    else if (in_dtype == TU_BF16 && dtype == TU_F32)
        stem_conv_kernel<bf16, float><<<grid, 256, 0, st>>>((const bf16 *)x, w27x64, b, (float *)out, H, W);
    else if (in_dtype == TU_U8 && dtype == TU_F32)
        stem_conv_kernel<uint8_t, float><<<grid, 256, 0, st>>>((const uint8_t *)x, w27x64, b, (float *)out, H, W);
    else if (in_dtype == TU_U8 && dtype == TU_BF16)
        stem_conv_kernel<uint8_t, bf16><<<grid, 256, 0, st>>>((const uint8_t *)x, w27x64, b, (bf16 *)out, H, W);
    else if (in_dtype == TU_F16 && dtype == TU_F32)
        stem_conv_kernel<f16, float><<<grid, 256, 0, st>>>((const f16 *)x, w27x64, b, (float *)out, H, W);
    else if (in_dtype == TU_F16 && dtype == TU_BF16)
        stem_conv_kernel<f16, bf16><<<grid, 256, 0, st>>>((const f16 *)x, w27x64, b, (bf16 *)out, H, W);
    else
        TU_CHECK_ARG(false, "stem_conv: bad dtype");
    TU_CHECK_LAUNCH("stem_conv");
    return TU_OK;
}

extern "C" int tu_conv3x3_c64_to3(const void *in, int dtype, const float *w, const void *w16, const float *b, float *out, int B,
                                  int H, int W, int relu, void *stream) {
    TU_CHECK_ARG(in && w && out && B > 0 && H > 0 && W > 0, "conv3x3_c64_to3: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == TU_BF16 && w16 && tc_enabled()) {
        int rc = tc_conv3x3_c64_to3((const bf16 *)in, (const bf16 *)w16, b, out, B, H, W, relu, st);
        if (rc != TU_TC_UNSUPPORTED) return rc;
    }
    dim3 grid(ceil_div(W, 128), H, B);
    if (dtype == TU_F32)
        conv64to3_kernel<float><<<grid, 128, 0, st>>>((const float *)in, w, b, out, H, W, relu);
    else if (dtype == TU_BF16)
        conv64to3_kernel<bf16><<<grid, 128, 0, st>>>((const bf16 *)in, w, b, out, H, W, relu);
    else
        TU_CHECK_ARG(false, "conv3x3_c64_to3: bad dtype");
    TU_CHECK_LAUNCH("conv3x3_c64_to3");
    return TU_OK;
}

extern "C" int tu_conv3x3_c3_ps(const float *in, const float *w, const float *b, float *out, int B, int H, int W, int r,
                                void *stream) {
    TU_CHECK_ARG(in && w && b && out && B > 0 && H > 0 && W > 0 && r >= 1 && r <= 6, "conv3x3_c3_ps: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    dim3 grid(ceil_div(W * r, 64), ceil_div(H * r, 4), B);
    size_t smem = (size_t)(28 * 3 * r * r) * sizeof(float);
    conv3_ps_kernel<<<grid, 256, smem, st>>>(in, w, b, out, H, W, r);
    TU_CHECK_LAUNCH("conv3x3_c3_ps");
    return TU_OK;
}

extern "C" int tu_final_conv_add(const float *in, const float *w, const float *b, const float *addend, void *out,
                                 int out_dtype, int B, int H, int W, int clamp, void *stream) {
    TU_CHECK_ARG(in && w && b && addend && out && B > 0 && H > 0 && W > 0, "final_conv_add: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    dim3 grid(ceil_div(W, 64), ceil_div(H, 4), B);
    if (out_dtype == TU_F32)
        final_conv_add_kernel<float><<<grid, 256, 0, st>>>(in, w, b, addend, (float *)out, H, W, clamp);
    else if (out_dtype == TU_BF16)
        final_conv_add_kernel<bf16><<<grid, 256, 0, st>>>(in, w, b, addend, (bf16 *)out, H, W, clamp);
    else if (out_dtype == TU_U8)
        final_conv_add_kernel<uint8_t><<<grid, 256, 0, st>>>(in, w, b, addend, (uint8_t *)out, H, W, clamp);
    else if (out_dtype == TU_F16)
        final_conv_add_kernel<f16><<<grid, 256, 0, st>>>(in, w, b, addend, (f16 *)out, H, W, clamp);
    else
        TU_CHECK_ARG(false, "final_conv_add: bad dtype");
    TU_CHECK_LAUNCH("final_conv_add");
    return TU_OK;
}
