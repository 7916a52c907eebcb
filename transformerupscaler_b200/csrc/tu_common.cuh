// Shared device/host helpers for libtu_b200 (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>
#include <string>

#include "../../include/tu_b200.h"

namespace tu {

typedef __nv_bfloat16 bf16;
typedef __half f16;

// ---- error plumbing (host) -------------------------------------------------------------------
void set_error(const std::string &msg);
int cuda_fail(cudaError_t e, const char *what);
void count_launch();   // every kernel launch of the library is counted (tu_launch_count)
// checks B NV12 / P010 frame surfaces (resample.cu): TU_ERR_ARG with the frame index and field in the message
int check_yuv420_planes(const TuFramePlanes *frames, int code, int B, int H, int W, const char *op);
// the same for B planar YUV frames (every planar code: TuFramePlanes3)
int check_yuvp_frames(const TuFramePlanes3 *frames, int code, int B, int H, int W, const char *op);
// the same for B semi-planar 4:2:2 frames (NV16 / P210: TuFramePlanes with H chroma rows)
int check_yuv422sp_frames(const TuFramePlanes *frames, int code, int B, int H, int W, const char *op);
// the same for B packed 4:2:2 frames (yuyv422 / uyvy422 / y210: TuFramePacked)
int check_packed422_frames(const TuFramePacked *frames, int code, int B, int H, int W, const char *op);

#define TU_CHECK_ARG(cond, msg)                         \
    do {                                                \
        if (!(cond)) {                                  \
            ::tu::set_error(std::string("tu: ") + msg); \
            return TU_ERR_ARG;                          \
        }                                               \
    } while (0)

#define TU_CHECK_LAUNCH(what)                                   \
    do {                                                        \
        cudaError_t _e = cudaGetLastError();                    \
        if (_e != cudaSuccess) return ::tu::cuda_fail(_e, what); \
        ::tu::count_launch();                                   \
    } while (0)

// ---- per-device launch state (host) ------------------------------------------------------------------------------
// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) and the SM count belong to a DEVICE, not to the process: a host that runs
// on cuda:0 and later on cuda:1 must raise the limit on both.  Launchers key their "attribute already set" flags and the
// SM count by the current device ordinal (lock-free: setting an attribute twice from two threads is harmless).
inline int current_device() {
    int d = 0;
    cudaGetDevice(&d);
    return d;
}
struct PerDeviceFlag {
    std::atomic<unsigned long long> bits[4] = {};      // 256 device ordinals
    bool is_set() const {
        const int d = current_device() & 255;
        return (bits[d >> 6].load(std::memory_order_acquire) >> (d & 63)) & 1ull;
    }
    void set() {
        const int d = current_device() & 255;
        bits[d >> 6].fetch_or(1ull << (d & 63), std::memory_order_release);
    }
};
struct PerDeviceMax {                                   // high-water mark of a per-device attribute (dynamic shared memory)
    std::atomic<int> v[256] = {};
    int get() const { return v[current_device() & 255].load(std::memory_order_acquire); }
    void set(int x) { v[current_device() & 255].store(x, std::memory_order_release); }
};
inline int device_sm_count() {                          // SM count of the CURRENT device
    static std::atomic<int> cache[256] = {};
    const int d = current_device();
    int n = cache[d & 255].load(std::memory_order_relaxed);
    if (!n) {
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, d);
        cache[d & 255].store(n, std::memory_order_relaxed);
    }
    return n;
}

// ---- scalar load/store with dtype conversion --------------------------------------------------
__device__ __forceinline__ float to_f(float v) { return v; }
__device__ __forceinline__ float to_f(bf16 v) { return __bfloat162float(v); }
__device__ __forceinline__ float to_f(f16 v) { return __half2float(v); }      // exact: every fp16 value is an fp32 value
// uint8 frames: ToTensor semantics on the way in (x / 255 in fp32, inference.py:65-70, app_overlay.py:298) and
// (out * 255).clamp(0, 255).to(uint8) on the way out (truncation, app_overlay.py:383)
// exact uint8 -> float without the conversion pipe: 2^23 + v has v in its low mantissa bits
__device__ __forceinline__ float u8_to_float(uint32_t v) { return __uint_as_float(0x4B000000u | v) - 8388608.f; }
__device__ __forceinline__ float to_f(uint8_t v) { return u8_to_float(v) / 255.f; }
template <typename T> __device__ __forceinline__ T from_f(float v);
template <> __device__ __forceinline__ float from_f<float>(float v) { return v; }
template <> __device__ __forceinline__ bf16 from_f<bf16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ f16 from_f<f16>(float v) { return __float2half_rn(v); }
// trunc(clamp(v * 255, 0, 255)): adding 2^23 with round-down leaves floor(t) in the low mantissa bits (t >= 0)
template <> __device__ __forceinline__ uint8_t from_f<uint8_t>(float v) {
    return (uint8_t)(__float_as_uint(__fadd_rd(fminf(fmaxf(v * 255.f, 0.f), 255.f), 8388608.f)) & 0xFFu);
}

// ---- uint8 frame layouts at the boundary ---------------------------------------------------------------------------
// A dtype code of the image input / output may carry a layout in bits 8..: TU_U8 | TU_LAYOUT_HWC (interleaved RGB, what PIL /
// OpenCV hand over: inference.py:65-70) or TU_U8 | TU_LAYOUT_HWC_BGR (channel order reversed: app_overlay.py:384-386).
// TU_U8 | TU_LAYOUT_NV12 (4:2:0 video frames) may add the colour bits TU_YUV_BT601 / TU_YUV_FULL_RANGE in bits 12..13.
// TU_U16 | TU_LAYOUT_P010 (10-bit 4:2:0 frames) may add the same bits, or TU_YUV_BT2020 (bit 14) instead of TU_YUV_BT601.
__host__ __device__ __forceinline__ int dtype_base(int d) { return d & 0xFF; }
// the layout bits are an enumeration (0 CHW, 1 HWC, 2 HWC_BGR, 3 RGBA, 4 NV12, 5 BGRA, 6 YUV420P, 7 YUV444P, 8 P010, 9 YUV422P, 10 NV16,
// 11 YUYV, 12 UYVY), and dtype_layout keeps the colour bits
// above them: compare whole values, never bits (0x500 = BGRA shares a bit with NV12, 0x300 = RGBA two bits with HWC / HWC_BGR)
__host__ __device__ __forceinline__ int dtype_layout(int d) { return d >> 8; }
__host__ __device__ __forceinline__ bool layout_is_px4(int l) { return l == 3 || l == 5; }          // RGBA / BGRA: 4-byte pixels
__host__ __device__ __forceinline__ bool layout_is_interleaved(int l) { return l == 1 || l == 2 || layout_is_px4(l); }
__host__ __device__ __forceinline__ bool dtype_is_px4(int d) {                          // TU_U8 | TU_LAYOUT_RGBA or TU_U8 | TU_LAYOUT_BGRA
    return d == (TU_U8 | TU_LAYOUT_RGBA) || d == (TU_U8 | TU_LAYOUT_BGRA);
}
__host__ __device__ __forceinline__ bool dtype_is_nv12(int d) {                        // TU_U8 | TU_LAYOUT_NV12 [| colour bits]
    return (d & ~(TU_YUV_BT601 | TU_YUV_FULL_RANGE)) == (TU_U8 | TU_LAYOUT_NV12);
}
__host__ __device__ __forceinline__ bool dtype_is_p010(int d) {                        // TU_U16 | TU_LAYOUT_P010 [| colour bits]
    const int c = d & (TU_YUV_BT601 | TU_YUV_BT2020 | TU_YUV_FULL_RANGE);
    return (d & ~c) == (TU_U16 | TU_LAYOUT_P010) && (c & (TU_YUV_BT601 | TU_YUV_BT2020)) != (TU_YUV_BT601 | TU_YUV_BT2020);
}
__host__ __device__ __forceinline__ bool dtype_is_yuv420(int d) { return dtype_is_nv12(d) || dtype_is_p010(d); }
// planar YUV (three planes Y, U, V): layout 6 yuv420p (TU_U8 only), 7 yuv444p (TU_U8) / yuv444p16 (TU_U16, the code in the high 10
// bits); the 8-bit codes take NV12's colour bits, the 16-bit one P010's
__host__ __device__ __forceinline__ bool dtype_is_yuv420p(int d) {                     // TU_U8 | TU_LAYOUT_YUV420P [| colour bits]
    return (d & ~(TU_YUV_BT601 | TU_YUV_FULL_RANGE)) == (TU_U8 | TU_LAYOUT_YUV420P);
}
__host__ __device__ __forceinline__ bool dtype_is_yuv444p(int d) {                     // TU_U8 | TU_LAYOUT_YUV444P [| colour bits]
    return (d & ~(TU_YUV_BT601 | TU_YUV_FULL_RANGE)) == (TU_U8 | TU_LAYOUT_YUV444P);
}
__host__ __device__ __forceinline__ bool dtype_is_yuv444p16(int d) {                   // TU_U16 | TU_LAYOUT_YUV444P [| colour bits]
    const int c = d & (TU_YUV_BT601 | TU_YUV_BT2020 | TU_YUV_FULL_RANGE);
    return (d & ~c) == (TU_U16 | TU_LAYOUT_YUV444P) && (c & (TU_YUV_BT601 | TU_YUV_BT2020)) != (TU_YUV_BT601 | TU_YUV_BT2020);
}
// 4:2:2 (layout 9 yuv422p: three planes, 10 NV16: Y then interleaved (U, V) rows) and the LSB-aligned 10-bit planar codes (TU_U16 |
// planar layout | TU_YUV_LSB10: the code in the low 10 bits).  8-bit codes take NV12's colour bits, 16-bit codes P010's
__host__ __device__ __forceinline__ bool yuv8_code_is(int d, int base) { return (d & ~(TU_YUV_BT601 | TU_YUV_FULL_RANGE)) == base; }
__host__ __device__ __forceinline__ bool yuv16_code_is(int d, int base) {
    const int c = d & (TU_YUV_BT601 | TU_YUV_BT2020 | TU_YUV_FULL_RANGE);
    return (d & ~c) == base && (c & (TU_YUV_BT601 | TU_YUV_BT2020)) != (TU_YUV_BT601 | TU_YUV_BT2020);
}
__host__ __device__ __forceinline__ bool dtype_is_yuv422p(int d) { return yuv8_code_is(d, TU_U8 | TU_LAYOUT_YUV422P); }
__host__ __device__ __forceinline__ bool dtype_is_nv16(int d) { return yuv8_code_is(d, TU_U8 | TU_LAYOUT_NV16); }
__host__ __device__ __forceinline__ bool dtype_is_p210(int d) { return yuv16_code_is(d, TU_U16 | TU_LAYOUT_NV16); }
__host__ __device__ __forceinline__ bool dtype_is_yuv420p10(int d) { return yuv16_code_is(d, TU_U16 | TU_LAYOUT_YUV420P | TU_YUV_LSB10); }
__host__ __device__ __forceinline__ bool dtype_is_yuv422p10(int d) { return yuv16_code_is(d, TU_U16 | TU_LAYOUT_YUV422P | TU_YUV_LSB10); }
__host__ __device__ __forceinline__ bool dtype_is_yuv444p10(int d) { return yuv16_code_is(d, TU_U16 | TU_LAYOUT_YUV444P | TU_YUV_LSB10); }
__host__ __device__ __forceinline__ bool dtype_is_lsb10(int d) { return dtype_is_yuv420p10(d) || dtype_is_yuv422p10(d) || dtype_is_yuv444p10(d); }
// semi-planar 4:2:2 (TuFramePlanes surfaces with H chroma rows)
__host__ __device__ __forceinline__ bool dtype_is_yuv422sp(int d) { return dtype_is_nv16(d) || dtype_is_p210(d); }
// every planar code (TuFramePlanes3 surfaces)
__host__ __device__ __forceinline__ bool dtype_is_yuvp(int d) {
    return dtype_is_yuv420p(d) || dtype_is_yuv444p(d) || dtype_is_yuv444p16(d) || dtype_is_yuv422p(d) || dtype_is_lsb10(d);
}
// packed 4:2:2 (layout 11 YUYV: Y0 U Y1 V, 12 UYVY: U Y0 V Y1; one plane, TuFramePacked surfaces): yuyv422 and uyvy422 (TU_U8, NV12's
// colour bits) and y210 (TU_U16 | TU_LAYOUT_YUYV, the code in the high 10 bits, P010's colour bits)
__host__ __device__ __forceinline__ bool dtype_is_yuyv422(int d) { return yuv8_code_is(d, TU_U8 | TU_LAYOUT_YUYV); }
__host__ __device__ __forceinline__ bool dtype_is_uyvy422(int d) { return yuv8_code_is(d, TU_U8 | TU_LAYOUT_UYVY); }
__host__ __device__ __forceinline__ bool dtype_is_y210(int d) { return yuv16_code_is(d, TU_U16 | TU_LAYOUT_YUYV); }
__host__ __device__ __forceinline__ bool dtype_is_packed422(int d) { return dtype_is_yuyv422(d) || dtype_is_uyvy422(d) || dtype_is_y210(d); }
// every YUV frame code: converted to / from a planar fp16 (8-bit) or fp32 (16-bit) RGB frame at the ends of the forward
__host__ __device__ __forceinline__ bool dtype_is_yuv(int d) {
    return dtype_is_yuv420(d) || dtype_is_yuvp(d) || dtype_is_yuv422sp(d) || dtype_is_packed422(d);
}
// one RGB pixel of frame b -> out, in the requested layout.  pix = y * W + x, plane = H * W
template <typename TO>
__device__ __forceinline__ void store_rgb(TO *out, long b, long plane, long pix, int layout, float r, float g, float bl) {
    if (layout == 0) {
        TO *o = out + b * 3 * plane + pix;
        o[0] = from_f<TO>(r); o[plane] = from_f<TO>(g); o[2 * plane] = from_f<TO>(bl);
    } else {
        TO *o = out + (b * plane + pix) * 3;
        o[layout == 2 ? 2 : 0] = from_f<TO>(r); o[1] = from_f<TO>(g); o[layout == 2 ? 0 : 2] = from_f<TO>(bl);
    }
}
// one 4-byte pixel (layout 3: R G B A, 5: B G R A) at pixel index pix of a (B, H, W, 4) frame batch, written once; its alpha is byte pix of
// the (B, H, W) plane `alpha`, or 255 when there is none
__device__ __forceinline__ void store_px4(uint8_t *out, long pix, int layout, float r, float g, float bl, const uint8_t *alpha) {
    const uint32_t cr = from_f<uint8_t>(r), cg = from_f<uint8_t>(g), cb = from_f<uint8_t>(bl);
    const uint32_t a = alpha ? (uint32_t)alpha[pix] : 255u;
    reinterpret_cast<uint32_t *>(out)[pix] = (layout == 5 ? cb | cr << 16 : cr | cb << 16) | cg << 8 | a << 24;
}

// internal forms of two output ops that also take the alpha plane of a 4-byte output (NULL: alpha 255); the exported functions
// (tu_bicubic_add_clamp, tu_subpixel_conv_add) are these with NULL
int bicubic_add_clamp_alpha(const void *x, int in_dtype, int H, int W, const float *res, int rH, int rW, void *out, int out_dtype, int B,
                            int outH, int outW, int clamp, const uint8_t *alpha, cudaStream_t st);
int subpixel_conv_add_alpha(const float *in, const float *w_ps, const float *b_ps, int r, const float *host_fin_wb, const float *addend,
                            void *out, int out_dtype, int B, int H, int W, int clamp, const uint8_t *alpha, cudaStream_t st);

// 4 consecutive elements -> float4 (pointer must be aligned to 4 elements)
__device__ __forceinline__ float4 load4(const float *p) { return *reinterpret_cast<const float4 *>(p); }
__device__ __forceinline__ float4 load4(const bf16 *p) {
    uint2 u = *reinterpret_cast<const uint2 *>(p);
    __nv_bfloat162 a = *reinterpret_cast<__nv_bfloat162 *>(&u.x);
    __nv_bfloat162 b = *reinterpret_cast<__nv_bfloat162 *>(&u.y);
    float2 fa = __bfloat1622float2(a), fb = __bfloat1622float2(b);
    return make_float4(fa.x, fa.y, fb.x, fb.y);
}
__device__ __forceinline__ void store4(float *p, float4 v) { *reinterpret_cast<float4 *>(p) = v; }
__device__ __forceinline__ void store4(bf16 *p, float4 v) {
    __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y);
    __nv_bfloat162 b = __floats2bfloat162_rn(v.z, v.w);
    uint2 u;
    u.x = *reinterpret_cast<uint32_t *>(&a);
    u.y = *reinterpret_cast<uint32_t *>(&b);
    *reinterpret_cast<uint2 *>(p) = u;
}

// ---- programmatic dependent launch (PDL) -----------------------------------------------------------------------
// Every kernel of a forward is launched with programmatic stream serialization: it may become resident (and run its prologue:
// barrier init, TMEM allocation, tensor-map prefetch) while the previous kernel of the stream is draining.  pdl_wait() blocks
// until that kernel has completed and its writes are visible, so it must precede EVERY access to global memory; kernels call
// pdl_trigger() first thing so that their own successor can be scheduled early.  Both are no-ops for ordinary launches.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

extern thread_local int g_use_pdl;      // api.cu (debug key "pdl")
extern thread_local int g_ga_shape;      // transformer_simt.cu (debug key "ga_shape")
extern thread_local int g_bicubic_pair; // resample.cu (debug key "bicubic_pair")
extern thread_local int g_bicubic_tile; // resample.cu (debug key "bicubic_tile")
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args &&...args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = g_use_pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f)); }

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
static inline size_t dtype_size(int dtype) {
    const int d = dtype & 0xFF;
    return d == TU_BF16 || d == TU_F16 || d == TU_U16 ? 2 : d == TU_U8 ? 1 : 4;
}

}  // namespace tu
