// Memory-bound resampling kernels.
//  * fused  out = clamp( bicubic(x) + bicubic(residual) )  — replaces two F.interpolate(mode='bicubic',
//    align_corners=False) calls, the add and the clamp (WindowTransformer/model.py:241,301,304-305;
//    ResidualTransformer/model.py:125,160,163-164) with one pass: x and residual read once, out written once.
//    Tap arithmetic follows ATen bit-for-bit in fp32 (ATen/native/UpSample.h:259-312,400-448):
//    scale = (float)in/out, src = fma(scale, dst+0.5, -0.5), i = floor(src), t = src - i,
//    Keys cubic A = -0.75, taps clamped to [0, in-1].
//  * antialiased bilinear resize (torchvision Resize on a tensor = ATen _upsample_bilinear2d_aa), used by
//    FastTransformer when the integer factor overshoots res_out (FastTransformer/model.py:323-325).
#include <cuda.h>

#include <algorithm>
#include <type_traits>

#include "tc/ptx.cuh"
#include "tc/tc_api.cuh"
#include "tu_common.cuh"

namespace tu {

struct Cubic {
    int idx[4];
    float w[4];
};

__device__ __forceinline__ float cubic1(float x, float A) { return ((A + 2.f) * x - (A + 3.f)) * x * x + 1.f; }
__device__ __forceinline__ float cubic2(float x, float A) { return ((A * x - 5.f * A) * x + 8.f * A) * x - 4.f * A; }

__device__ __forceinline__ Cubic cubic_taps(int dst, int in_size, int out_size) {
    const float scale = (float)in_size / (float)out_size;
    const float src = fmaf(scale, (float)dst + 0.5f, -0.5f);
    int i0 = min((int)floorf(src), in_size - 1);
    float t = fminf(fmaxf(src - (float)i0, 0.f), 1.f);
    const float A = -0.75f;
    Cubic c;
    c.w[0] = cubic2(t + 1.f, A);
    c.w[1] = cubic1(t, A);
    const float u = 1.f - t;
    c.w[2] = cubic1(u, A);
    c.w[3] = cubic2(u + 1.f, A);
#pragma unroll
    for (int j = 0; j < 4; ++j) c.idx[j] = min(max(i0 + j - 1, 0), in_size - 1);
    return c;
}

// A thread owns one output column of a 32-row strip and slides a 4-row window of horizontally-resampled source rows
// down the strip, for the 3 channels and both sources at once.  A source row is resampled horizontally exactly once
// per strip, the per-row vertical taps come from a small shared table computed once per CTA.  Operation order per
// output is ATen's: horizontal 4-tap sum inside each source row, then the vertical 4-tap sum.
//
// Source pixels come from one of two places:
//   * TMA variant (row pitch of both sources a multiple of 16 bytes): one thread issues two cp.async.bulk.tensor loads
//     that bring the whole source footprint of the tile (3 channels x rows x cols) into shared memory; out-of-image
//     parts are rewritten with the border pixel (replicate padding == clamped taps), so a thread's four taps are four
//     contiguous elements and the strip walk runs at shared-memory latency with almost no address arithmetic.
//   * direct variant (any shape): taps are read from global memory.
constexpr int BS_W = 128, BS_H = 32;

// element as stored -> float, and the factor applied once per 4-tap sum (uint8 frames: 1/255, ToTensor)
__device__ __forceinline__ float raw_f(float v) { return v; }
__device__ __forceinline__ float raw_f(bf16 v) { return __bfloat162float(v); }
__device__ __forceinline__ float raw_f(f16 v) { return __half2float(v); }
__device__ __forceinline__ float raw_f(uint8_t v) { return u8_to_float(v); }
template <typename TS> __device__ __forceinline__ float src_scale(float t) { return t; }
template <> __device__ __forceinline__ float src_scale<uint8_t>(float t) { return t * 0.00392156862745098f; }

template <typename TS>
struct GlobalSrc {          // image of one frame: (3, H, W); taps and rows clamped to the image like ATen
    const TS *img;
    long plane;
    int H, W;
    __device__ __forceinline__ float hrow(int ch, int row, const Cubic &cx) const {
        const TS *p = img + ch * plane + (long)min(max(row, 0), H - 1) * W;
        float t = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) t += raw_f(p[cx.idx[j]]) * cx.w[j];
        return src_scale<TS>(t);
    }
};
// slide the 3-channel window so that it covers source rows base-1 .. base+2
template <typename Src>
__device__ __forceinline__ void slide(float (&win)[3][4], int &cur, int base, const Src &src, const Cubic &cx) {
    if (cur != base) {
        const int step = base - cur;
        if (step < 0 || step > 3) {
#pragma unroll
            for (int c = 0; c < 3; ++c)
#pragma unroll
                for (int i = 0; i < 4; ++i) win[c][i] = src.hrow(c, base - 1 + i, cx);
        } else {
            for (int s = 0; s < step; ++s) {
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    win[c][0] = win[c][1]; win[c][1] = win[c][2]; win[c][2] = win[c][3];
                    win[c][3] = src.hrow(c, cur + s + 3, cx);
                }
            }
        }
        cur = base;
    }
}

// The TMA zero-fills the parts of the box that lie outside the image; bicubic taps clamp to the border instead.
// Rewrite those columns / rows with the nearest image pixel so that a thread's four taps are always contiguous.
template <typename TS>
__device__ __forceinline__ void replicate_pad(TS *s, int r0, int c0, int nr, int nc, int H, int W) {
    const int padL = max(0, -c0), padR = max(0, c0 + nc - W), padT = max(0, -r0), padB = max(0, r0 + nr - H);
    if ((padL | padR | padT | padB) == 0) return;           // interior tile (uniform across the CTA)
    if (padL | padR) {
        for (int e = threadIdx.x; e < 3 * nr; e += blockDim.x) {
            TS *p = s + e * nc;
            const TS l = p[min(padL, nc - 1)], r = p[max(nc - 1 - padR, 0)];
            for (int c = 0; c < padL; ++c) p[c] = l;
            for (int c = nc - padR; c < nc; ++c) p[c] = r;
        }
        __syncthreads();
    }
    if (padT | padB) {
        for (int e = threadIdx.x; e < 3 * nc; e += blockDim.x) {
            TS *p = s + (e / nc) * nr * nc + (e % nc);
            const TS tp = p[min(padT, nr - 1) * nc], bt = p[max(nr - 1 - padB, 0) * nc];
            for (int r = 0; r < padT; ++r) p[r * nc] = tp;
            for (int r = nr - padB; r < nr; ++r) p[r * nc] = bt;
        }
    }
    __syncthreads();
}

__device__ __forceinline__ int src_floor(int dst, int in_size, int out_size) {
    const float scale = (float)in_size / (float)out_size;
    return min((int)floorf(fmaf(scale, (float)dst + 0.5f, -0.5f)), in_size - 1);
}

struct BicubicTileGeom {
    int xr, xc, rr, rc;             // TMA box sizes: rows / cols of the x tile and of the residual tile
    float sxh, sxw, srh, srw;       // (float)in / (float)out per axis and source, divided once on the host (same IEEE quotient)
};
__device__ __forceinline__ int src_floor_s(int dst, float scale, int in_size) {
    return min((int)floorf(fmaf(scale, (float)dst + 0.5f, -0.5f)), in_size - 1);
}

// shared-memory element -> float with an immediate byte offset (the four taps of a row are contiguous)
template <int OFF> __device__ __forceinline__ float lds_raw(uint32_t a, float) {
    float v;
    asm("ld.shared.f32 %0, [%1+%2];" : "=f"(v) : "r"(a), "n"(OFF * 4));
    return v;
}
template <int OFF> __device__ __forceinline__ float lds_raw(uint32_t a, bf16) {
    unsigned short h;
    asm("ld.shared.u16 %0, [%1+%2];" : "=h"(h) : "r"(a), "n"(OFF * 2));
    return __uint_as_float((uint32_t)h << 16);
}
template <int OFF> __device__ __forceinline__ float lds_raw(uint32_t a, f16) {
    unsigned short h;
    asm("ld.shared.u16 %0, [%1+%2];" : "=h"(h) : "r"(a), "n"(OFF * 2));
    return __half2float(__ushort_as_half(h));
}
template <int OFF> __device__ __forceinline__ float lds_raw(uint32_t a, uint8_t) {
    unsigned short h;
    asm("ld.shared.u8 %0, [%1+%2];" : "=h"(h) : "r"(a), "n"(OFF));
    return u8_to_float(h);
}
// 4-tap horizontal sum of one source row of the replicate-padded tile (ATen's left-to-right order)
template <typename TS>
__device__ __forceinline__ float hrow_tile(uint32_t a, const float (&w)[4]) {
    float t = 0.f;
    t += lds_raw<0>(a, TS()) * w[0];
    t += lds_raw<1>(a, TS()) * w[1];
    t += lds_raw<2>(a, TS()) * w[2];
    t += lds_raw<3>(a, TS()) * w[3];
    return src_scale<TS>(t);
}
// slide a 3-channel window of horizontally resampled rows to source rows base-1 .. base+2; ca[] = per-channel shared
// address of the thread's first tap in tile row 0, trow0 = tile row of source row 0 (= -r0)
template <typename TS>
__device__ __forceinline__ void slide_tile(float (&win)[3][4], int &cur, int base, const uint32_t (&ca)[3], int trow0, uint32_t pitchB,
                                           const float (&w)[4]) {
    if (base == cur) return;
    if (base == cur + 1) {                  // the only step an up-scaling strip ever takes after its first row
        const uint32_t ro = (uint32_t)(base + 2 + trow0) * pitchB;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            win[c][0] = win[c][1]; win[c][1] = win[c][2]; win[c][2] = win[c][3];
            win[c][3] = hrow_tile<TS>(ca[c] + ro, w);
        }
    } else {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const uint32_t ro = (uint32_t)(base - 1 + i + trow0) * pitchB;
#pragma unroll
            for (int c = 0; c < 3; ++c) win[c][i] = hrow_tile<TS>(ca[c] + ro, w);
        }
    }
    cur = base;
}

// MODE 0: taps from global memory (any shape, residual optional at run time); MODE 1 / 2: TMA-staged tile with / without
// the residual source (compile-time, so the strip loop has no dead branches).  PX4: 4-byte uint8 pixels (layout 3 / 5) whose alpha
// comes from the plane `alpha` (NULL: 255); the other instantiations never read `alpha`
template <typename TI, typename TO, int MODE, bool PX4 = false>
__global__ void __launch_bounds__(BS_W) bicubic_add_clamp_strip_kernel(const __grid_constant__ CUtensorMap tmap_x,
                                                                       const __grid_constant__ CUtensorMap tmap_r,
                                                                       const BicubicTileGeom g, const TI *__restrict__ x, int H, int W,
                                                                       const float *__restrict__ res, int rH, int rW,
                                                                       TO *__restrict__ out, int oH, int oW, int clamp, int layout,
                                                                       const uint8_t *__restrict__ alpha) {
    pdl_trigger();
    pdl_wait();          // the residual image is written by the previous kernel of the stream
    __shared__ float yw[2][BS_H][4];
    __shared__ int ybase[2][BS_H];
    __shared__ __align__(8) uint64_t bar;
    extern __shared__ uint8_t tile_dyn[];
    uint8_t *tile_raw = tile_dyn + ((128u - (ptx::smem_u32(tile_dyn) & 127u)) & 127u);     // TMA destinations are 128-byte aligned
    constexpr bool TMA = MODE != 0;
    if (MODE == 2) res = nullptr;
    const int t = threadIdx.x;
    const int ox0 = blockIdx.x * BS_W, ox = ox0 + t, oy0 = blockIdx.y * BS_H, b = blockIdx.z;
    int xr0 = 0, xc0 = 0, rr0 = 0, rc0 = 0;
    const uint32_t x_bytes = 3u * g.xr * g.xc * sizeof(TI);
    const uint32_t x_bytes_al = (x_bytes + 127u) & ~127u;
    if (TMA) {
        // the innermost box coordinate must start on a 16-byte boundary (measured: tools/probes/tma_probe.cu): round the
        // first column down to a multiple of 16 / sizeof(element); the box is that much wider (see the host side)
        constexpr int XA = 16 / (int)sizeof(TI);
        xr0 = src_floor(oy0, H, oH) - 1; xc0 = (src_floor(ox0, W, oW) - 1) & ~(XA - 1);
        if (res) { rr0 = src_floor(oy0, rH, oH) - 1; rc0 = (src_floor(ox0, rW, oW) - 1) & ~3; }
        if (t == 0) {
            const uint32_t bar_a = ptx::smem_u32(&bar);
            ptx::mbar_init(bar_a, 1);
            ptx::fence_barrier_init();
            ptx::mbar_expect_tx(bar_a, x_bytes + (res ? 3u * g.rr * g.rc * 4u : 0u));
            ptx::tma_load_4d(ptx::smem_u32(tile_raw), &tmap_x, bar_a, xc0, xr0, 0, b);
            if (res) ptx::tma_load_4d(ptx::smem_u32(tile_raw) + x_bytes_al, &tmap_r, bar_a, rc0, rr0, 0, b);
        }
    }
    if (t < 2 * BS_H) {
        const int s = t / BS_H, r = t % BS_H;
        const int in_size = s ? rH : H;
        const float scale = (float)in_size / (float)oH;
        const float src = fmaf(scale, (float)min(oy0 + r, oH - 1) + 0.5f, -0.5f);
        const int i0 = min((int)floorf(src), in_size - 1);
        const float tt = fminf(fmaxf(src - (float)i0, 0.f), 1.f), u = 1.f - tt;
        const float A = -0.75f;
        ybase[s][r] = i0;
        yw[s][r][0] = cubic2(tt + 1.f, A); yw[s][r][1] = cubic1(tt, A); yw[s][r][2] = cubic1(u, A); yw[s][r][3] = cubic2(u + 1.f, A);
    }
    __syncthreads();
    if (TMA) {
        ptx::mbar_wait(ptx::smem_u32(&bar), 0);
        replicate_pad(reinterpret_cast<TI *>(tile_raw), xr0, xc0, g.xr, g.xc, H, W);
        if (res) replicate_pad(reinterpret_cast<float *>(tile_raw + x_bytes_al), rr0, rc0, g.rr, g.rc, rH, rW);
    }
    if (ox >= oW) return;
    const Cubic cx = cubic_taps(ox, W, oW);
    Cubic cr = cx;
    if (res) cr = cubic_taps(ox, rW, oW);
    const long xplane = (long)H * W, rplane = (long)rH * rW, oplane = (long)oH * oW;
    TO *ob = out + (long)b * 3 * oplane + ox;
    float wx[3][4], wr[3][4];
    int curx = -1000000, curr = -1000000;
    const int nrows = min(BS_H, oH - oy0);
    auto run = [&](const auto &sx, const auto &sr) {
        for (int r = 0; r < nrows; ++r) {
            slide(wx, curx, ybase[0][r], sx, cx);
            if (res) slide(wr, curr, ybase[1][r], sr, cr);
            const float4 a = *reinterpret_cast<const float4 *>(yw[0][r]);
            const float4 gg = *reinterpret_cast<const float4 *>(yw[1][r]);
#pragma unroll
            float v3[3];
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                float v = 0.f;
                v += wx[c][0] * a.x; v += wx[c][1] * a.y; v += wx[c][2] * a.z; v += wx[c][3] * a.w;
                if (res) {
                    float u = 0.f;
                    u += wr[c][0] * gg.x; u += wr[c][1] * gg.y; u += wr[c][2] * gg.z; u += wr[c][3] * gg.w;
                    v += u;
                }
                if (clamp) v = fminf(fmaxf(v, 0.f), 1.f);
                v3[c] = v;
            }
            if constexpr (PX4) store_px4(out, b * oplane + (long)(oy0 + r) * oW + ox, layout, v3[0], v3[1], v3[2], alpha);
            else store_rgb<TO>(out, b, oplane, (long)(oy0 + r) * oW + ox, layout, v3[0], v3[1], v3[2]);
        }
    };
    if (TMA) {
        // ---- fast path: explicit shared-memory addresses, immediate tap offsets, running output pointers
        constexpr bool RES = MODE == 1;
        const uint32_t xpitch = g.xc * sizeof(TI), rpitch = g.rc * 4u;
        const uint32_t xs = ptx::smem_u32(tile_raw) + (uint32_t)(src_floor(ox, W, oW) - 1 - xc0) * (uint32_t)sizeof(TI);
        const uint32_t xa[3] = {xs, xs + g.xr * xpitch, xs + 2u * g.xr * xpitch};
        uint32_t ra[3] = {0u, 0u, 0u};
        if (RES) {
            const uint32_t rs = ptx::smem_u32(tile_raw) + x_bytes_al + (uint32_t)(src_floor(ox, rW, oW) - 1 - rc0) * 4u;
            ra[0] = rs; ra[1] = rs + g.rr * rpitch; ra[2] = rs + 2u * g.rr * rpitch;
        }
        TO *o0 = ob + (long)oy0 * oW, *o1 = o0 + oplane, *o2 = o1 + oplane;
        for (int r = 0; r < nrows; ++r) {
            slide_tile<TI>(wx, curx, ybase[0][r], xa, -xr0, xpitch, cx.w);
            if (RES) slide_tile<float>(wr, curr, ybase[1][r], ra, -rr0, rpitch, cr.w);
            const float4 a = *reinterpret_cast<const float4 *>(yw[0][r]);
            const float4 gg = *reinterpret_cast<const float4 *>(yw[1][r]);
            float v[3];
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                v[c] = 0.f;
                v[c] += wx[c][0] * a.x; v[c] += wx[c][1] * a.y; v[c] += wx[c][2] * a.z; v[c] += wx[c][3] * a.w;
                if (RES) {
                    float u = 0.f;
                    u += wr[c][0] * gg.x; u += wr[c][1] * gg.y; u += wr[c][2] * gg.z; u += wr[c][3] * gg.w;
                    v[c] += u;
                }
                if (clamp) v[c] = fminf(fmaxf(v[c], 0.f), 1.f);
            }
            if constexpr (PX4) {
                store_px4(out, b * oplane + (long)(oy0 + r) * oW + ox, layout, v[0], v[1], v[2], alpha);
            } else if (layout == 0) {
                *o0 = from_f<TO>(v[0]); *o1 = from_f<TO>(v[1]); *o2 = from_f<TO>(v[2]);
                o0 += oW; o1 += oW; o2 += oW;
            } else {
                store_rgb<TO>(out, b, oplane, (long)(oy0 + r) * oW + ox, layout, v[0], v[1], v[2]);
            }
        }
    } else {
        const GlobalSrc<TI> sx{x + (long)b * 3 * xplane, xplane, H, W};
        const GlobalSrc<float> sr{res ? res + (long)b * 3 * rplane : nullptr, rplane, rH, rW};
        run(sx, sr);
    }
}

// ---- two output columns per thread -----------------------------------------------------------------------------------
// The strip kernel above is bound by instruction issue (145 instructions per output pixel, 81 % issue slots, 29 % of the HBM
// bandwidth).  Here a thread owns TWO adjacent output columns: the horizontal and vertical 4-tap sums of the pair run on packed
// fp32 pairs (FFMA2: one issue slot for both columns, bit-identical to the scalar FMAs in the same order), the per-row vertical
// weights, row bookkeeping and window shifts are shared by the pair, and the pair leaves as one 4-byte (bf16) / 8-byte (fp32) /
// 2-byte (uint8) store.  TMA-staged tiles only (PAIR_H x 128 outputs per 64-thread CTA), even output width.
constexpr int PAIR_H = 36;

template <typename TS>
__device__ __forceinline__ ptx::f32x2 hrow_pair(uint32_t aA, uint32_t aB, const ptx::f32x2 (&w)[4]) {
    ptx::f32x2 t = ptx::mul2(ptx::pk2(lds_raw<0>(aA, TS()), lds_raw<0>(aB, TS())), w[0]);
    t = ptx::fma2(ptx::pk2(lds_raw<1>(aA, TS()), lds_raw<1>(aB, TS())), w[1], t);
    t = ptx::fma2(ptx::pk2(lds_raw<2>(aA, TS()), lds_raw<2>(aB, TS())), w[2], t);
    t = ptx::fma2(ptx::pk2(lds_raw<3>(aA, TS()), lds_raw<3>(aB, TS())), w[3], t);
    if (sizeof(TS) == 1) t = ptx::mul2(t, ptx::pk2(0.00392156862745098f, 0.00392156862745098f));
    return t;
}
template <typename TS>
__device__ __forceinline__ void slide_pair(ptx::f32x2 (&win)[3][4], int &cur, int base, const uint32_t (&caA)[3], const uint32_t (&caB)[3],
                                           int trow0, uint32_t pitchB, const ptx::f32x2 (&w)[4]) {
    if (base == cur) return;
    if (base == cur + 1) {                  // the only step an up-scaling strip ever takes after its first row
        const uint32_t ro = (uint32_t)(base + 2 + trow0) * pitchB;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            win[c][0] = win[c][1]; win[c][1] = win[c][2]; win[c][2] = win[c][3];
            win[c][3] = hrow_pair<TS>(caA[c] + ro, caB[c] + ro, w);
        }
    } else {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const uint32_t ro = (uint32_t)(base - 1 + i + trow0) * pitchB;
#pragma unroll
            for (int c = 0; c < 3; ++c) win[c][i] = hrow_pair<TS>(caA[c] + ro, caB[c] + ro, w);
        }
    }
    cur = base;
}
__device__ __forceinline__ void store_pair(float *o, float a, float b) { *reinterpret_cast<float2 *>(o) = make_float2(a, b); }
__device__ __forceinline__ void store_pair(bf16 *o, float a, float b) { *reinterpret_cast<__nv_bfloat162 *>(o) = __floats2bfloat162_rn(a, b); }
__device__ __forceinline__ void store_pair(f16 *o, float a, float b) { *reinterpret_cast<__half2 *>(o) = __floats2half2_rn(a, b); }
__device__ __forceinline__ void store_pair(uint8_t *o, float a, float b) {
    *reinterpret_cast<unsigned short *>(o) = (unsigned short)((unsigned)from_f<uint8_t>(a) | ((unsigned)from_f<uint8_t>(b) << 8));
}

// PX4: 4-byte uint8 pixels (layout 3 / 5), the pair's two pixels one 8-byte store, alpha from the plane `alpha` (NULL: 255)
template <typename TI, typename TO, bool RES, bool PX4 = false>
__global__ void __launch_bounds__(BS_W / 2) bicubic_add_clamp_pair_kernel(const __grid_constant__ CUtensorMap tmap_x,
                                                                          const __grid_constant__ CUtensorMap tmap_r,
                                                                          const BicubicTileGeom g, int H, int W, int rH, int rW,
                                                                          TO *__restrict__ out, int oH, int oW, int clamp, int layout,
                                                                          const uint8_t *__restrict__ alpha) {
    pdl_trigger();
    pdl_wait();          // the residual image is written by the previous kernel of the stream
    __shared__ __align__(16) float yw[2][PAIR_H][4];
    __shared__ int ybase[2][PAIR_H];
    __shared__ __align__(8) uint64_t bar;
    extern __shared__ uint8_t tile_dyn[];
    uint8_t *tile_raw = tile_dyn + ((128u - (ptx::smem_u32(tile_dyn) & 127u)) & 127u);     // TMA destinations are 128-byte aligned
    const int t = threadIdx.x;
    const int ox0 = blockIdx.x * BS_W, ox = ox0 + 2 * t, oy0 = blockIdx.y * PAIR_H, b = blockIdx.z;
    const uint32_t x_bytes = 3u * g.xr * g.xc * sizeof(TI);
    const uint32_t x_bytes_al = (x_bytes + 127u) & ~127u;
    constexpr int XA = 16 / (int)sizeof(TI);       // the innermost box coordinate must start on a 16-byte boundary
    const int xr0 = src_floor(oy0, H, oH) - 1, xc0 = (src_floor(ox0, W, oW) - 1) & ~(XA - 1);
    int rr0 = 0, rc0 = 0;
    if (RES) { rr0 = src_floor(oy0, rH, oH) - 1; rc0 = (src_floor(ox0, rW, oW) - 1) & ~3; }
    if (t == 0) {
        const uint32_t bar_a = ptx::smem_u32(&bar);
        ptx::mbar_init(bar_a, 1);
        ptx::fence_barrier_init();
        ptx::mbar_expect_tx(bar_a, x_bytes + (RES ? 3u * g.rr * g.rc * 4u : 0u));
        ptx::tma_load_4d(ptx::smem_u32(tile_raw), &tmap_x, bar_a, xc0, xr0, 0, b);
        if (RES) ptx::tma_load_4d(ptx::smem_u32(tile_raw) + x_bytes_al, &tmap_r, bar_a, rc0, rr0, 0, b);
    }
    for (int i = t; i < 2 * PAIR_H; i += BS_W / 2) {
        const int s = i / PAIR_H, r = i % PAIR_H;
        const int in_size = s ? rH : H;
        const float scale = (float)in_size / (float)oH;
        const float src = fmaf(scale, (float)min(oy0 + r, oH - 1) + 0.5f, -0.5f);
        const int i0 = min((int)floorf(src), in_size - 1);
        const float tt = fminf(fmaxf(src - (float)i0, 0.f), 1.f), u = 1.f - tt;
        const float A = -0.75f;
        ybase[s][r] = i0;
        yw[s][r][0] = cubic2(tt + 1.f, A); yw[s][r][1] = cubic1(tt, A); yw[s][r][2] = cubic1(u, A); yw[s][r][3] = cubic2(u + 1.f, A);
    }
    __syncthreads();
    ptx::mbar_wait(ptx::smem_u32(&bar), 0);
    replicate_pad(reinterpret_cast<TI *>(tile_raw), xr0, xc0, g.xr, g.xc, H, W);
    if (RES) replicate_pad(reinterpret_cast<float *>(tile_raw + x_bytes_al), rr0, rc0, g.rr, g.rc, rH, rW);
    if (ox >= oW) return;           // oW is even: a pair is inside or outside as a whole
    const Cubic cA = cubic_taps(ox, W, oW), cB = cubic_taps(ox + 1, W, oW);
    ptx::f32x2 wxp[4], wrp[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) wxp[j] = ptx::pk2(cA.w[j], cB.w[j]);
    const uint32_t xpitch = g.xc * sizeof(TI), rpitch = g.rc * 4u;
    const uint32_t tile_a = ptx::smem_u32(tile_raw);
    const uint32_t xsA = tile_a + (uint32_t)(src_floor(ox, W, oW) - 1 - xc0) * (uint32_t)sizeof(TI);
    const uint32_t xsB = tile_a + (uint32_t)(src_floor(ox + 1, W, oW) - 1 - xc0) * (uint32_t)sizeof(TI);
    const uint32_t xaA[3] = {xsA, xsA + g.xr * xpitch, xsA + 2u * g.xr * xpitch};
    const uint32_t xaB[3] = {xsB, xsB + g.xr * xpitch, xsB + 2u * g.xr * xpitch};
    uint32_t raA[3] = {0u, 0u, 0u}, raB[3] = {0u, 0u, 0u};
    if (RES) {
        const Cubic rA = cubic_taps(ox, rW, oW), rB = cubic_taps(ox + 1, rW, oW);
#pragma unroll
        for (int j = 0; j < 4; ++j) wrp[j] = ptx::pk2(rA.w[j], rB.w[j]);
        const uint32_t rsA = tile_a + x_bytes_al + (uint32_t)(src_floor(ox, rW, oW) - 1 - rc0) * 4u;
        const uint32_t rsB = tile_a + x_bytes_al + (uint32_t)(src_floor(ox + 1, rW, oW) - 1 - rc0) * 4u;
        raA[0] = rsA; raA[1] = rsA + g.rr * rpitch; raA[2] = rsA + 2u * g.rr * rpitch;
        raB[0] = rsB; raB[1] = rsB + g.rr * rpitch; raB[2] = rsB + 2u * g.rr * rpitch;
    }
    const long oplane = (long)oH * oW;
    TO *o0 = out + (long)b * 3 * oplane + (long)oy0 * oW + ox, *o1 = o0 + oplane, *o2 = o1 + oplane;
    ptx::f32x2 wx[3][4], wr[3][4];
    int curx = -1000000, curr = -1000000;
    const int nrows = min(PAIR_H, oH - oy0);
    for (int r = 0; r < nrows; ++r) {
        slide_pair<TI>(wx, curx, ybase[0][r], xaA, xaB, -xr0, xpitch, wxp);
        if (RES) slide_pair<float>(wr, curr, ybase[1][r], raA, raB, -rr0, rpitch, wrp);
        const float4 a = *reinterpret_cast<const float4 *>(yw[0][r]);
        const float4 gg = *reinterpret_cast<const float4 *>(yw[1][r]);
        const ptx::f32x2 a0 = ptx::pk2(a.x, a.x), a1 = ptx::pk2(a.y, a.y), a2 = ptx::pk2(a.z, a.z), a3 = ptx::pk2(a.w, a.w);
        float lo[3], hi[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            ptx::f32x2 v = ptx::mul2(wx[c][0], a0);
            v = ptx::fma2(wx[c][1], a1, v); v = ptx::fma2(wx[c][2], a2, v); v = ptx::fma2(wx[c][3], a3, v);
            if (RES) {
                ptx::f32x2 u = ptx::mul2(wr[c][0], ptx::pk2(gg.x, gg.x));
                u = ptx::fma2(wr[c][1], ptx::pk2(gg.y, gg.y), u); u = ptx::fma2(wr[c][2], ptx::pk2(gg.z, gg.z), u);
                u = ptx::fma2(wr[c][3], ptx::pk2(gg.w, gg.w), u);
                v = ptx::add2(v, u);
            }
            ptx::up2(v, lo[c], hi[c]);
            if (clamp) { lo[c] = fminf(fmaxf(lo[c], 0.f), 1.f); hi[c] = fminf(fmaxf(hi[c], 0.f), 1.f); }
        }
        if constexpr (PX4) {
            // the pair's two pixels are eight consecutive bytes (ox even, the buffer 8-byte aligned: host); their alphas two bytes
            const long pix = ((long)b * oH + oy0 + r) * oW + ox;
            const uint32_t a2 = alpha ? (uint32_t)*reinterpret_cast<const unsigned short *>(alpha + pix) : 0xFFFFu;
            const int c0 = layout == 5 ? 2 : 0, c2 = 2 - c0;
            uint2 px;
            px.x = (uint32_t)from_f<uint8_t>(lo[c0]) | (uint32_t)from_f<uint8_t>(lo[1]) << 8 | (uint32_t)from_f<uint8_t>(lo[c2]) << 16 | (a2 & 0xFFu) << 24;
            px.y = (uint32_t)from_f<uint8_t>(hi[c0]) | (uint32_t)from_f<uint8_t>(hi[1]) << 8 | (uint32_t)from_f<uint8_t>(hi[c2]) << 16 |
                   (a2 >> 8) << 24;
            *reinterpret_cast<uint2 *>(out + pix * 4) = px;
        } else if (layout == 0) {
            store_pair(o0, lo[0], hi[0]); store_pair(o1, lo[1], hi[1]); store_pair(o2, lo[2], hi[2]);
            o0 += oW; o1 += oW; o2 += oW;
        } else {
            // interleaved frames: the pair's two pixels are six consecutive elements (ox is even: 2-element aligned)
            const int c0 = layout == 2 ? 2 : 0, c2 = 2 - c0;
            TO *o = out + (((long)b * oH + oy0 + r) * oW + ox) * 3;
            store_pair(o, lo[c0], lo[1]); store_pair(o + 2, lo[c2], hi[c0]); store_pair(o + 4, hi[1], hi[c2]);
        }
    }
}

// pair store of values already clamped to [0, 1]: from_f<uint8_t> without its (then no-op) clamp to [0, 255] — the same product
// and the same round-down add, the two result bytes packed by one permute; other output types store as usual
template <typename T> __device__ __forceinline__ void store_pair_unit(T *o, float a, float b) { store_pair(o, a, b); }
template <> __device__ __forceinline__ void store_pair_unit<uint8_t>(uint8_t *o, float a, float b) {
    const uint32_t ua = __float_as_uint(__fadd_rd(__fmul_rn(a, 255.f), 8388608.f)), ub = __float_as_uint(__fadd_rd(__fmul_rn(b, 255.f), 8388608.f));
    *reinterpret_cast<unsigned short *>(o) = (unsigned short)__byte_perm(ua, ub, 0x0040);
}

// clamp a pair to [0, 1] and store it.  bf16: the conversion clamps below (cvt.rn.relu) and one packed min clamps above — rounding is
// monotonic and 1.0 is a bf16, so min(bf16(relu(v)), 1) == bf16(clamp(v, 0, 1)) bit for bit — which takes the two saturating adds off
// the FMA pipe, the busy one in these kernels; other types: saturate, then store
template <typename T> __device__ __forceinline__ void clamp_store_pair(T *o, float lo, float hi) {
    store_pair_unit(o, fminf(fmaxf(lo, 0.f), 1.f), fminf(fmaxf(hi, 0.f), 1.f));
}
template <> __device__ __forceinline__ void clamp_store_pair<bf16>(bf16 *o, float lo, float hi) {
    uint32_t d;
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    asm("min.bf16x2 %0, %0, %1;" : "+r"(d) : "r"(0x3f803f80u));
    *reinterpret_cast<uint32_t *>(o) = d;
}
// fp16: the same identity (1.0 = 0x3c00 is an fp16 and rounding to fp16 is monotonic as well)
template <> __device__ __forceinline__ void clamp_store_pair<f16>(f16 *o, float lo, float hi) {
    uint32_t d;
    asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    asm("min.f16x2 %0, %0, %1;" : "+r"(d) : "r"(0x3c003c00u));
    *reinterpret_cast<uint32_t *>(o) = d;
}

// one value already clamped to [0, 1] -> the output element (uint8: the same product and round-down add as from_f<uint8_t>, whose clamp
// is a no-op here; the low byte of the sum is the result)
template <typename T> __device__ __forceinline__ T unit_to_u8(float v) { return from_f<T>(v); }
template <> __device__ __forceinline__ uint8_t unit_to_u8<uint8_t>(float v) {
    return (uint8_t)__float_as_uint(__fadd_rd(__fmul_rn(v, 255.f), 8388608.f));
}

// ---- periodic row schedules: x at 3:2 with the residual at 3:1 (720p -> 1080p, every x1.5 output), x at n:1 with the residual at 2n:1
// for n = 2, 3, 4, 6 (720p -> 4K is n = 3) ----------------------------------------------------------------------------------------
// The pair kernel spends more than half of its issue slots on bookkeeping: window moves (28 MOVs per source row), per-row
// compare / branch chains, 16-bit tap loads with one shift each, and a local-memory round trip of the pixel values.  When
// outH = 3/2 H = 3 rH (or n H = 2n rH) the source-row schedule is periodic (RowSched below; checked on the host with the same fp32
// coordinate arithmetic, row_pattern), so the strip loop unrolls over one period of output rows (12, or 8n)
// with the four window rows in FIXED registers (a circular window: no moves, no compares).  Taps are fetched as aligned words:
// the two columns of a pair need at most six consecutive source elements starting at an even index (three 32-bit loads for
// bf16, three 16-bit loads for uint8) against 6-entry weight vectors padded with zeros — fma(e, 0, t) == t, so every sum is
// bitwise the pair kernel's.  Vertical weights enter the packed FMAs as broadcast scalars; a thread works on one channel.
// Planar output, clamp on, outH a multiple of the period (a CTA's rows are whole unrolled periods).

template <typename TS> __device__ __forceinline__ void ld6(uint32_t a, float (&e)[6]);
template <> __device__ __forceinline__ void ld6<bf16>(uint32_t a, float (&e)[6]) {
    uint32_t w0, w1, w2;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w0) : "r"(a));
    asm volatile("ld.shared.u32 %0, [%1+4];" : "=r"(w1) : "r"(a));
    asm volatile("ld.shared.u32 %0, [%1+8];" : "=r"(w2) : "r"(a));
    // low half by a byte permute (ALU pipe; a shift may be issued as an integer multiply on the FMA pipe, which is the busy one here)
    e[0] = __uint_as_float(__byte_perm(w0, 0u, 0x1044)); e[1] = __uint_as_float(w0 & 0xffff0000u);
    e[2] = __uint_as_float(__byte_perm(w1, 0u, 0x1044)); e[3] = __uint_as_float(w1 & 0xffff0000u);
    e[4] = __uint_as_float(__byte_perm(w2, 0u, 0x1044)); e[5] = __uint_as_float(w2 & 0xffff0000u);
}
// fp16: the same three aligned words, each half converted exactly (cvt.f32.f16; fp16 -> fp32 never rounds)
template <> __device__ __forceinline__ void ld6<f16>(uint32_t a, float (&e)[6]) {
    uint32_t w0, w1, w2;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w0) : "r"(a));
    asm volatile("ld.shared.u32 %0, [%1+4];" : "=r"(w1) : "r"(a));
    asm volatile("ld.shared.u32 %0, [%1+8];" : "=r"(w2) : "r"(a));
    const float2 f0 = __half22float2(*reinterpret_cast<const __half2 *>(&w0));
    const float2 f1 = __half22float2(*reinterpret_cast<const __half2 *>(&w1));
    const float2 f2 = __half22float2(*reinterpret_cast<const __half2 *>(&w2));
    e[0] = f0.x; e[1] = f0.y; e[2] = f1.x; e[3] = f1.y; e[4] = f2.x; e[5] = f2.y;
}
template <> __device__ __forceinline__ void ld6<uint8_t>(uint32_t a, float (&e)[6]) {
    unsigned short h0, h1, h2;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(h0) : "r"(a));
    asm volatile("ld.shared.u16 %0, [%1+2];" : "=h"(h1) : "r"(a));
    asm volatile("ld.shared.u16 %0, [%1+4];" : "=h"(h2) : "r"(a));
    // byte -> 0x4B0000bb (2^23 + b) with one byte permute, minus 2^23: u8_to_float
    e[0] = __uint_as_float(__byte_perm(h0, 0x4B000000u, 0x7440)) - 8388608.f; e[1] = __uint_as_float(__byte_perm(h0, 0x4B000000u, 0x7441)) - 8388608.f;
    e[2] = __uint_as_float(__byte_perm(h1, 0x4B000000u, 0x7440)) - 8388608.f; e[3] = __uint_as_float(__byte_perm(h1, 0x4B000000u, 0x7441)) - 8388608.f;
    e[4] = __uint_as_float(__byte_perm(h2, 0x4B000000u, 0x7440)) - 8388608.f; e[5] = __uint_as_float(__byte_perm(h2, 0x4B000000u, 0x7441)) - 8388608.f;
}
// horizontal sums of a column pair over one staged source row: six elements from an aligned address, zero-padded weights
template <typename TS>
__device__ __forceinline__ ptx::f32x2 hsum6(uint32_t a, const ptx::f32x2 (&w)[6]) {
    float e[6];
    ld6<TS>(a, e);
    ptx::f32x2 t = ptx::mul2(w[0], ptx::pk2(e[0], e[0]));
#pragma unroll
    for (int j = 1; j < 6; ++j) t = ptx::fma2(w[j], ptx::pk2(e[j], e[j]), t);
    if (sizeof(TS) == 1) t = ptx::mul2(t, ptx::pk2(0.00392156862745098f, 0.00392156862745098f));
    return t;
}
// the same over a fp32 row (residual): five elements from the first tap of the left column
__device__ __forceinline__ ptx::f32x2 hsum5(uint32_t a, const ptx::f32x2 (&w)[5]) {
    float e[5];
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(e[0]) : "r"(a));
    asm volatile("ld.shared.f32 %0, [%1+4];" : "=f"(e[1]) : "r"(a));
    asm volatile("ld.shared.f32 %0, [%1+8];" : "=f"(e[2]) : "r"(a));
    asm volatile("ld.shared.f32 %0, [%1+12];" : "=f"(e[3]) : "r"(a));
    asm volatile("ld.shared.f32 %0, [%1+16];" : "=f"(e[4]) : "r"(a));
    ptx::f32x2 t = ptx::mul2(w[0], ptx::pk2(e[0], e[0]));
#pragma unroll
    for (int j = 1; j < 5; ++j) t = ptx::fma2(w[j], ptx::pk2(e[j], e[j]), t);
    return t;
}
// w[k] of a 4-tap filter, zero outside 0..3 (k is a compile-time constant after unrolling: no branches, selects only)
__device__ __forceinline__ float tap_or_zero(const float (&w)[4], int k) { return (k >= 0 && k < 4) ? w[k] : 0.f; }

// A thread is (channel, column pair): 192 threads share the staged tile of a 36 x 128 output block — three times the warps of a
// three-channels-per-thread layout for the same shared memory, which is what hides the FMA-chain and shared-memory latencies
// (measured: 2 warps per CTA, 12 per SM -> issue slots 50 % busy).  The per-column filters (four cubic_taps per pair: two
// columns x two sources) are computed once per CTA by 256 tasks spread over the threads and handed over in shared memory, so
// the three channels do not repeat them.
constexpr int R32_T = 3 * (BS_W / 2);

// Row schedules of the tile kernel: over a period of P output rows (a multiple of the 4-row window rotation for both sources), does
// x / the residual step to a new source row before output row q?  PAT 0: outH = 3/2 H = 3 rH (720p -> 1080p; x 3:2, residual 3:1).
// PAT n = 2, 3, 4, 6: outH = n H = 2n rH (inference.py's --scale values on a 2x-downsampled residual; 3 = 720p -> 4K): the source
// coordinate (2 oy + 1 - n) / (2n) passes an integer before oy = n m + n / 2 (n even; n odd: AT oy = n m + (n - 1) / 2, where the
// fp32 rounding decides — the host checks every row), and likewise at ratio 2n for the residual.  A CTA covers whole periods of rows:
// TILE, or BIG when the larger tiles still give every SM a CTA (the per-tile set-up — column filters, vertical
// table, four window rows per source — is 30 % of the instructions at TILE rows; measured at 3:2 / 3:1, profiles/r3_ab_bicubic_tile_rows.log:
// 36 / 48 / 60 / 72 rows = 0.574 / 0.550 / 0.550 / 0.575 of the pair kernel's time, 72 rows leave three CTAs per SM).
template <int PAT> struct RowSched {
    static constexpr int P = 8 * PAT, TILE = PAT == 2 ? 48 : P, BIG = PAT == 2 ? 80 : PAT == 3 ? 72 : 96;
    static constexpr bool xstep(int q) { return q % PAT == PAT / 2; }
    static constexpr bool rstep(int q) { return q % (2 * PAT) == PAT; }
};
template <> struct RowSched<0> {
    static constexpr int P = 12, TILE = 36, BIG = 60;
    static constexpr bool xstep(int q) { return q % 3 != 0; }
    static constexpr bool rstep(int q) { return q % 3 == 1; }
};
template <int PAT> constexpr int sched_relx(int q) { int n = 0; for (int i = 0; i <= q; ++i) n += RowSched<PAT>::xstep(i) ? 1 : 0; return n; }
template <int PAT> constexpr int sched_relr(int q) { int n = 0; for (int i = 0; i <= q; ++i) n += RowSched<PAT>::rstep(i) ? 1 : 0; return n; }
static_assert(sched_relx<0>(11) == 8 && sched_relr<0>(11) == 4 && sched_relx<2>(15) == 8 && sched_relr<2>(15) == 4 &&
                  sched_relx<3>(23) == 8 && sched_relr<3>(23) == 4 && sched_relx<4>(31) == 8 && sched_relr<4>(31) == 4 &&
                  sched_relx<6>(47) == 8 && sched_relr<6>(47) == 4,
              "a period must rotate both 4-row windows a whole number of times");
constexpr int R32_MAXTILE = 96;
static inline int sched_tile(int pat, bool big) {
    switch (pat) {
        case 0: return big ? RowSched<0>::BIG : RowSched<0>::TILE;
        case 2: return big ? RowSched<2>::BIG : RowSched<2>::TILE;
        case 3: return big ? RowSched<3>::BIG : RowSched<3>::TILE;
        case 4: return big ? RowSched<4>::BIG : RowSched<4>::TILE;
        default: return big ? RowSched<6>::BIG : RowSched<6>::TILE;
    }
}

// PX (uint8 frames only when not 0): 0 planar; 3 interleaved output pixels, `layout` 1 = RGB, 2 = BGR, a thread stores its channel's
// two bytes; 4 four-byte pixels, `layout` 3 = RGBA, 5 = BGRA: the three channels of a pixel belong to three warps, so each period of
// rows is staged in shared memory (PX4_STAGE bytes behind the tile) and written as whole pixels, with the alpha of the plane `alpha`
// (NULL: 255).  PX 0 / 3 never read `alpha`.
template <int PAT> constexpr int px4_stage_bytes() { return RowSched<PAT>::P * BS_W * 4; }
template <typename TI, typename TO, int PAT, int PX>
__global__ void __launch_bounds__(R32_T, 5) bicubic_add_clamp_r32_kernel(const __grid_constant__ CUtensorMap tmap_x,
                                                                         const __grid_constant__ CUtensorMap tmap_r,
                                                                         const BicubicTileGeom g, int H, int W, int rH, int rW,
                                                                         TO *__restrict__ out, int oH, int oW, int layout, int TILE,
                                                                         const uint8_t *__restrict__ alpha) {
    constexpr bool HWC = PX == 3;
    pdl_trigger();
    pdl_wait();          // the residual image is written by the previous kernel of the stream
    constexpr int P = RowSched<PAT>::P;             // TILE (rows per CTA, a multiple of P, <= R32_MAXTILE) is chosen per launch
    __shared__ __align__(16) float yw[2][R32_MAXTILE][4];
    __shared__ float tapw[4][4][BS_W / 2];       // [x left, x right, residual left, residual right][tap][pair]
    __shared__ int tapi[4][BS_W / 2];            // source column of the second tap (floor of the source coordinate)
    __shared__ __align__(8) uint64_t bar;
    extern __shared__ uint8_t tile_dyn[];
    uint8_t *tile_raw = tile_dyn + ((128u - (ptx::smem_u32(tile_dyn) & 127u)) & 127u);     // TMA destinations are 128-byte aligned
    const int t = threadIdx.x;
    const int ox0 = blockIdx.x * BS_W, oy0 = blockIdx.y * TILE, b = blockIdx.z;
    const uint32_t x_bytes = 3u * g.xr * g.xc * sizeof(TI);
    const uint32_t x_bytes_al = (x_bytes + 127u) & ~127u;
    constexpr int XA = 16 / (int)sizeof(TI);       // the innermost box coordinate must start on a 16-byte boundary
    const int xr0 = src_floor_s(oy0, g.sxh, H) - 1, xc0 = (src_floor_s(ox0, g.sxw, W) - 1) & ~(XA - 1);
    const int rr0 = src_floor_s(oy0, g.srh, rH) - 1, rc0 = (src_floor_s(ox0, g.srw, rW) - 1) & ~3;
    if (t == 0) {
        const uint32_t bar_a = ptx::smem_u32(&bar);
        ptx::mbar_init(bar_a, 1);
        ptx::fence_barrier_init();
        ptx::mbar_expect_tx(bar_a, x_bytes + 3u * g.rr * g.rc * 4u);
        ptx::tma_load_4d(ptx::smem_u32(tile_raw), &tmap_x, bar_a, xc0, xr0, 0, b);
        ptx::tma_load_4d(ptx::smem_u32(tile_raw) + x_bytes_al, &tmap_r, bar_a, rc0, rr0, 0, b);
    }
    const float A = -0.75f;
    if (t < 2 * TILE) {                             // vertical filters of the block's rows, both sources (2 * TILE <= 192 threads)
        const int s = t / TILE, r = t % TILE;
        const int in_size = s ? rH : H;
        const float scale = s ? g.srh : g.sxh;
        const float src = fmaf(scale, (float)min(oy0 + r, oH - 1) + 0.5f, -0.5f);
        const int i0 = min((int)floorf(src), in_size - 1);
        const float tt = fminf(fmaxf(src - (float)i0, 0.f), 1.f), u = 1.f - tt;
        yw[s][r][0] = cubic2(tt + 1.f, A); yw[s][r][1] = cubic1(tt, A); yw[s][r][2] = cubic1(u, A); yw[s][r][3] = cubic2(u + 1.f, A);
    }
    for (int i = t; i < 4 * (BS_W / 2); i += R32_T) {       // horizontal filters: (source, left / right column) x pair
        const int which = i / (BS_W / 2), pair = i % (BS_W / 2);
        const int in_size = (which & 2) ? rW : W;
        const float scale = (which & 2) ? g.srw : g.sxw;
        const float src = fmaf(scale, (float)(ox0 + 2 * pair + (which & 1)) + 0.5f, -0.5f);
        const int i0 = min((int)floorf(src), in_size - 1);
        const float tt = fminf(fmaxf(src - (float)i0, 0.f), 1.f), u = 1.f - tt;
        tapi[which][pair] = i0;
        tapw[which][0][pair] = cubic2(tt + 1.f, A); tapw[which][1][pair] = cubic1(tt, A);
        tapw[which][2][pair] = cubic1(u, A); tapw[which][3][pair] = cubic2(u + 1.f, A);
    }
    __syncthreads();
    ptx::mbar_wait(ptx::smem_u32(&bar), 0);
    replicate_pad(reinterpret_cast<TI *>(tile_raw), xr0, xc0, g.xr, g.xc, H, W);
    replicate_pad(reinterpret_cast<float *>(tile_raw + x_bytes_al), rr0, rc0, g.rr, g.rc, rH, rW);
    const int ch = t / (BS_W / 2), pair = t % (BS_W / 2), ox = ox0 + 2 * pair;
    // oW is even: a pair is inside or outside as a whole.  PX 4: every thread stays for the block barriers of the staging; a pair
    // right of the image computes from clamped taps inside the tile, and its pixels are not written
    if (PX != 4 && ox >= oW) return;

    // ---- horizontal filters of the pair: six (x) / five (residual) consecutive elements, zero-padded weights
    const uint32_t xpitch = g.xc * sizeof(TI), rpitch = g.rc * 4u;
    ptx::f32x2 wx6[6], wr5[5];
    uint32_t px, pr;                // shared addresses of the pair's first element in tile row 0 of the thread's channel
    {
        float wA[4], wB[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) { wA[k] = tapw[0][k][pair]; wB[k] = tapw[1][k][pair]; }
        const int iA = tapi[0][pair], iB = tapi[1][pair];
        const int p0 = (iA - 1) & ~1;                           // even source column (the tile starts on an even column too)
        const int offA = iA - 1 - p0, offB = iB - 1 - p0;         // 0..1, 0..2
#pragma unroll
        for (int j = 0; j < 6; ++j) {
            const float a = offA ? tap_or_zero(wA, j - 1) : tap_or_zero(wA, j);
            const float bb = offB == 0 ? tap_or_zero(wB, j) : offB == 1 ? tap_or_zero(wB, j - 1) : tap_or_zero(wB, j - 2);
            wx6[j] = ptx::pk2(a, bb);
        }
        px = ptx::smem_u32(tile_raw) + (uint32_t)(p0 - xc0) * (uint32_t)sizeof(TI) + (uint32_t)ch * g.xr * xpitch;
#pragma unroll
        for (int k = 0; k < 4; ++k) { wA[k] = tapw[2][k][pair]; wB[k] = tapw[3][k][pair]; }
        const int jA = tapi[2][pair], d = tapi[3][pair] - jA;       // d = 0 or 1
#pragma unroll
        for (int j = 0; j < 5; ++j) wr5[j] = ptx::pk2(tap_or_zero(wA, j), d ? tap_or_zero(wB, j - 1) : tap_or_zero(wB, j));
        pr = ptx::smem_u32(tile_raw) + x_bytes_al + (uint32_t)(jA - 1 - rc0) * 4u + (uint32_t)ch * g.rr * rpitch;
    }
    const long oplane = (long)oH * oW;
    // planar: the channel's plane; interleaved: the channel's byte inside the pixel (reversed for BGR), three bytes per pixel
    TO *o = HWC ? out + (((long)b * oH + oy0) * oW + ox) * 3 + (layout == 2 ? 2 - ch : ch) : out + ((long)b * 3 + ch) * oplane + (long)oy0 * oW + ox;
    const int orow = HWC ? 3 * oW : oW;
    const int nrows = min(TILE, oH - oy0);
    // PX 4: the staged period, [row q][column 0..127][byte]; the thread's channel byte (reversed for BGRA) of its pair in row 0
    const uint32_t stage = ptx::smem_u32(tile_raw) + x_bytes_al + ((3u * g.rr * g.rc * 4u + 15u) & ~15u);
    const uint32_t sbyte = stage + (uint32_t)(2 * pair) * 4u + (uint32_t)(layout == 5 ? 2 - ch : ch);

    // window rows live in fixed registers: tile row n of a source sits in slot n & 3
    ptx::f32x2 wx[4], wr[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        wx[i] = hsum6<TI>(px + i * xpitch, wx6);
        wr[i] = hsum5(pr + i * rpitch, wr5);
    }
    px += 4u * xpitch;
    pr += 4u * rpitch;
    const float *ywx = &yw[0][0][0], *ywr = &yw[1][0][0];
#pragma unroll 1
    for (int r0 = 0; r0 < nrows; r0 += P) {
#pragma unroll
        for (int q = 0; q < P; ++q) {
            const int relx = sched_relx<PAT>(q);    // first tile row of the x window (a whole number of rotations per period: slots unchanged)
            const int relr = sched_relr<PAT>(q);    // first tile row of the residual window
            if (RowSched<PAT>::xstep(q)) {
                wx[(relx + 3) & 3] = hsum6<TI>(px, wx6);
                px += xpitch;
            }
            if (RowSched<PAT>::rstep(q)) {
                wr[(relr + 3) & 3] = hsum5(pr, wr5);
                pr += rpitch;
            }
            const float4 a = *reinterpret_cast<const float4 *>(ywx + (r0 + q) * 4);
            const float4 gg = *reinterpret_cast<const float4 *>(ywr + (r0 + q) * 4);
            ptx::f32x2 v = ptx::mul2(wx[relx & 3], ptx::pk2(a.x, a.x));
            v = ptx::fma2(wx[(relx + 1) & 3], ptx::pk2(a.y, a.y), v);
            v = ptx::fma2(wx[(relx + 2) & 3], ptx::pk2(a.z, a.z), v);
            v = ptx::fma2(wx[(relx + 3) & 3], ptx::pk2(a.w, a.w), v);
            ptx::f32x2 u = ptx::mul2(wr[relr & 3], ptx::pk2(gg.x, gg.x));
            u = ptx::fma2(wr[(relr + 1) & 3], ptx::pk2(gg.y, gg.y), u);
            u = ptx::fma2(wr[(relr + 2) & 3], ptx::pk2(gg.z, gg.z), u);
            u = ptx::fma2(wr[(relr + 3) & 3], ptx::pk2(gg.w, gg.w), u);
            v = ptx::add2(v, u);
            float lo, hi;
            ptx::up2(v, lo, hi);
            if constexpr (PX == 4) {
                const uint32_t q_lo = unit_to_u8<TO>(fminf(fmaxf(lo, 0.f), 1.f)), q_hi = unit_to_u8<TO>(fminf(fmaxf(hi, 0.f), 1.f));
                asm volatile("st.shared.u8 [%0], %1;" ::"r"(sbyte + (uint32_t)q * BS_W * 4u), "r"(q_lo) : "memory");
                asm volatile("st.shared.u8 [%0], %1;" ::"r"(sbyte + (uint32_t)q * BS_W * 4u + 4u), "r"(q_hi) : "memory");
            } else {
                if (HWC) { o[0] = unit_to_u8<TO>(fminf(fmaxf(lo, 0.f), 1.f)); o[3] = unit_to_u8<TO>(fminf(fmaxf(hi, 0.f), 1.f)); }
                else clamp_store_pair(o, lo, hi);       // outH % P == 0 (host): whole periods of rows
                o += orow;
            }
        }
        if constexpr (PX == 4) {        // the period's pixels, each written once as a 32-bit word with its alpha
            __syncthreads();
            for (int i = t; i < P * BS_W; i += R32_T) {
                const int q = i / BS_W, x = ox0 + (i % BS_W);
                if (x >= oW) continue;
                const long pix = ((long)b * oH + oy0 + r0 + q) * oW + x;
                uint32_t w;
                asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w) : "r"(stage + (uint32_t)i * 4u) : "memory");
                reinterpret_cast<uint32_t *>(out)[pix] = (w & 0x00FFFFFFu) | (alpha ? (uint32_t)alpha[pix] : 255u) << 24;
            }
            __syncthreads();            // the next period overwrites the stage
        }
    }
}

// ---- the same, streaming ---------------------------------------------------------------------------------------------------
// The tile kernel pays its set-up (column filters, vertical table, four window rows per source, the wait for the tile) once per
// 36 output rows: 30 % of its instructions.  Here a CTA walks DOWN a 128-column strip for up to 16 blocks of 12 output rows; the
// window registers simply carry over, and the source rows arrive through a ring of three small stages (8 x rows + 4 residual rows
// = the new rows of one block), loaded by TMA two blocks ahead.  full[] barriers carry the TMA bytes, empty[] barriers count one
// arrival per warp; warp 0 refills the stage released one block earlier.  Load 0 is the window's initial four rows (an 8-row x
// box whose upper half is not used, so that every box has the same shape).  The grid is sized to be co-resident: strips x
// segments <= 5 CTAs per SM.
constexpr int R32S_NST = 3, R32S_MAXBLK = 16;

template <typename TI, typename TO>
__global__ void __launch_bounds__(R32_T, 5) bicubic_add_clamp_r32s_kernel(const __grid_constant__ CUtensorMap tmap_x,
                                                                          const __grid_constant__ CUtensorMap tmap_r, int xc, int rc,
                                                                          int H, int W, int rH, int rW, TO *__restrict__ out, int oH,
                                                                          int oW, int blocks_per_seg) {
    pdl_trigger();
    pdl_wait();          // the residual image is written by the previous kernel of the stream
    __shared__ __align__(16) float yw[2][R32S_MAXBLK * 12][4];
    __shared__ float tapw[4][4][BS_W / 2];       // [x left, x right, residual left, residual right][tap][pair]
    __shared__ int tapi[4][BS_W / 2];            // source column of the second tap (floor of the source coordinate)
    __shared__ __align__(8) uint64_t full[R32S_NST], empty[R32S_NST];
    extern __shared__ uint8_t tile_dyn[];
    uint8_t *tile_raw = tile_dyn + ((128u - (ptx::smem_u32(tile_dyn) & 127u)) & 127u);     // TMA destinations are 128-byte aligned
    const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
    const int ox0 = blockIdx.x * BS_W, b = blockIdx.z;
    const int kb0 = blockIdx.y * blocks_per_seg, nblk = min(blocks_per_seg, oH / 12 - kb0), oy0 = kb0 * 12;
    const int X0 = 8 * kb0 - 6, R0 = 4 * kb0 - 2;   // first source rows of load 0: the window of output row oy0 is x rows 8 kb0 - 2 .. + 1
    constexpr int XA = 16 / (int)sizeof(TI);       // the innermost box coordinate must start on a 16-byte boundary
    const int xc0 = (src_floor(ox0, W, oW) - 1) & ~(XA - 1), rc0 = (src_floor(ox0, rW, oW) - 1) & ~3;
    const uint32_t xpitch = xc * sizeof(TI), rpitch = rc * 4u;
    const uint32_t x_bytes = 3u * 8u * xpitch, r_bytes = 3u * 4u * rpitch;
    const uint32_t xst = (x_bytes + 127u) & ~127u, stage_bytes = xst + ((r_bytes + 127u) & ~127u);
    const uint32_t ring = ptx::smem_u32(tile_raw), full_a = ptx::smem_u32(&full[0]), empty_a = ptx::smem_u32(&empty[0]);
    const int total = nblk + 1;
    auto issue = [&](int L) {
        const uint32_t st = (uint32_t)(L % R32S_NST), bar_a = full_a + 8u * st;
        ptx::mbar_expect_tx(bar_a, x_bytes + r_bytes);
        ptx::tma_load_4d(ring + st * stage_bytes, &tmap_x, bar_a, xc0, X0 + 8 * L, 0, b);
        ptx::tma_load_4d(ring + st * stage_bytes + xst, &tmap_r, bar_a, rc0, R0 + 4 * L, 0, b);
    };
    if (t == 0) {
        for (int i = 0; i < R32S_NST; ++i) { ptx::mbar_init(full_a + 8u * i, 1); ptx::mbar_init(empty_a + 8u * i, R32_T / 32); }
        ptx::fence_barrier_init();
        for (int L = 0; L < R32S_NST && L < total; ++L) issue(L);
    }
    const float A = -0.75f;
    for (int i = t; i < 2 * 12 * nblk; i += R32_T) {      // vertical filters of the segment's rows, both sources
        const int s = i / (12 * nblk), r = i % (12 * nblk);
        const int in_size = s ? rH : H;
        const float scale = (float)in_size / (float)oH;
        const float src = fmaf(scale, (float)(oy0 + r) + 0.5f, -0.5f);
        const int i0 = min((int)floorf(src), in_size - 1);
        const float tt = fminf(fmaxf(src - (float)i0, 0.f), 1.f), u = 1.f - tt;
        yw[s][r][0] = cubic2(tt + 1.f, A); yw[s][r][1] = cubic1(tt, A); yw[s][r][2] = cubic1(u, A); yw[s][r][3] = cubic2(u + 1.f, A);
    }
    for (int i = t; i < 4 * (BS_W / 2); i += R32_T) {       // horizontal filters: (source, left / right column) x pair
        const int which = i / (BS_W / 2), pair = i % (BS_W / 2);
        const int in_size = (which & 2) ? rW : W;
        const float scale = (float)in_size / (float)oW;
        const float src = fmaf(scale, (float)(ox0 + 2 * pair + (which & 1)) + 0.5f, -0.5f);
        const int i0 = min((int)floorf(src), in_size - 1);
        const float tt = fminf(fmaxf(src - (float)i0, 0.f), 1.f), u = 1.f - tt;
        tapi[which][pair] = i0;
        tapw[which][0][pair] = cubic2(tt + 1.f, A); tapw[which][1][pair] = cubic1(tt, A);
        tapw[which][2][pair] = cubic1(u, A); tapw[which][3][pair] = cubic2(u + 1.f, A);
    }
    __syncthreads();
    const int ch = t / (BS_W / 2), pair = t % (BS_W / 2), ox = ox0 + 2 * pair;
    const bool active = ox < oW;    // oW is even: a pair is inside or outside as a whole; idle threads keep the barrier counts

    // ---- horizontal filters of the pair: six (x) / five (residual) consecutive elements, zero-padded weights
    ptx::f32x2 wx6[6], wr5[5];
    uint32_t pxo, pro;              // byte offsets of the pair's first element inside a stage, in tile row 0 of the thread's channel
    {
        float wA[4], wB[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) { wA[k] = tapw[0][k][pair]; wB[k] = tapw[1][k][pair]; }
        const int iA = tapi[0][pair], iB = tapi[1][pair];
        const int p0 = (iA - 1) & ~1;                           // even source column (the tile starts on an even column too)
        const int offA = iA - 1 - p0, offB = iB - 1 - p0;         // 0..1, 0..2
#pragma unroll
        for (int j = 0; j < 6; ++j) {
            const float a = offA ? tap_or_zero(wA, j - 1) : tap_or_zero(wA, j);
            const float bb = offB == 0 ? tap_or_zero(wB, j) : offB == 1 ? tap_or_zero(wB, j - 1) : tap_or_zero(wB, j - 2);
            wx6[j] = ptx::pk2(a, bb);
        }
        pxo = (active ? (uint32_t)(p0 - xc0) * (uint32_t)sizeof(TI) : 0u) + (uint32_t)ch * 8u * xpitch;
#pragma unroll
        for (int k = 0; k < 4; ++k) { wA[k] = tapw[2][k][pair]; wB[k] = tapw[3][k][pair]; }
        const int jA = tapi[2][pair], d = tapi[3][pair] - jA;       // d = 0 or 1
#pragma unroll
        for (int j = 0; j < 5; ++j) wr5[j] = ptx::pk2(tap_or_zero(wA, j), d ? tap_or_zero(wB, j - 1) : tap_or_zero(wB, j));
        pro = xst + (active ? (uint32_t)(jA - 1 - rc0) * 4u : 0u) + (uint32_t)ch * 4u * rpitch;
    }
    const long oplane = (long)oH * oW;
    TO *o = out + ((long)b * 3 + ch) * oplane + (long)oy0 * oW + (active ? ox : 0);
    // loads whose boxes reach outside the image (uniform over the CTA): every one of a strip at the left / right edge, else the
    // first ones of the top segment and the last ones of the bottom segment
    int kpad_lo = 0, kpad_hi = total;
    if (xc0 < 0 || xc0 + xc > W || rc0 < 0 || rc0 + rc > rW) kpad_lo = total;
    else {
        while (kpad_lo < total && (X0 + 8 * kpad_lo < 0 || R0 + 4 * kpad_lo < 0)) ++kpad_lo;
        while (kpad_hi > kpad_lo && (X0 + 8 * (kpad_hi - 1) + 8 > H || R0 + 4 * (kpad_hi - 1) + 4 > rH)) --kpad_hi;
    }

    // window rows live in fixed registers: row n of a source (counted from the window's first row at oy0) sits in slot n & 3
    ptx::f32x2 wx[4], wr[4];
    const float *ywx = &yw[0][0][0], *ywr = &yw[1][0][0];
#pragma unroll 1
    for (int k = 0; k < total; ++k) {
        const uint32_t st = (uint32_t)(k % R32S_NST);
        if (warp == 0 && k >= 1 && k - 1 + R32S_NST < total) {      // refill the stage every warp released one block ago
            ptx::mbar_wait(empty_a + 8u * (uint32_t)((k - 1) % R32S_NST), (uint32_t)((k - 1) / R32S_NST) & 1u);
            if (lane == 0) issue(k - 1 + R32S_NST);
        }
        ptx::mbar_wait(full_a + 8u * st, (uint32_t)(k / R32S_NST) & 1u);
        const bool pad = k < kpad_lo || k >= kpad_hi;
        if (pad) {          // the TMA zero-fills outside the image; bicubic taps clamp to the border
            replicate_pad(reinterpret_cast<TI *>(tile_raw + st * stage_bytes), X0 + 8 * k, xc0, 8, xc, H, W);
            replicate_pad(reinterpret_cast<float *>(tile_raw + st * stage_bytes + xst), R0 + 4 * k, rc0, 4, rc, rH, rW);
        }
        uint32_t px = ring + st * stage_bytes + pxo, pr = ring + st * stage_bytes + pro;
        if (k == 0) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                wx[i] = hsum6<TI>(px + (4 + i) * xpitch, wx6);
                wr[i] = hsum5(pr + i * rpitch, wr5);
            }
        } else {
            const int r0 = (k - 1) * 12;
#pragma unroll
            for (int q = 0; q < 12; ++q) {
                const int kk = q / 3, j = q % 3;
                const int relx = 2 * kk + j;            // first row of the x window (8 rows per block: slots unchanged)
                const int relr = kk + (j >= 1 ? 1 : 0); // first row of the residual window
                if (j != 0) {                           // x steps one source row on two output rows of three
                    wx[(relx + 3) & 3] = hsum6<TI>(px, wx6);
                    px += xpitch;
                }
                if (j == 1) {                           // the residual steps on one of three
                    wr[(relr + 3) & 3] = hsum5(pr, wr5);
                    pr += rpitch;
                }
                const float4 a = *reinterpret_cast<const float4 *>(ywx + (r0 + q) * 4);
                const float4 gg = *reinterpret_cast<const float4 *>(ywr + (r0 + q) * 4);
                ptx::f32x2 v = ptx::mul2(wx[relx & 3], ptx::pk2(a.x, a.x));
                v = ptx::fma2(wx[(relx + 1) & 3], ptx::pk2(a.y, a.y), v);
                v = ptx::fma2(wx[(relx + 2) & 3], ptx::pk2(a.z, a.z), v);
                v = ptx::fma2(wx[(relx + 3) & 3], ptx::pk2(a.w, a.w), v);
                ptx::f32x2 u = ptx::mul2(wr[relr & 3], ptx::pk2(gg.x, gg.x));
                u = ptx::fma2(wr[(relr + 1) & 3], ptx::pk2(gg.y, gg.y), u);
                u = ptx::fma2(wr[(relr + 2) & 3], ptx::pk2(gg.z, gg.z), u);
                u = ptx::fma2(wr[(relr + 3) & 3], ptx::pk2(gg.w, gg.w), u);
                v = ptx::add2(v, u);
                float lo, hi;
                ptx::up2(v, lo, hi);
                lo = fminf(fmaxf(lo, 0.f), 1.f); hi = fminf(fmaxf(hi, 0.f), 1.f);
                if (active) store_pair_unit(o, lo, hi);
                o += oW;
            }
        }
        __syncwarp();
        if (pad) ptx::fence_proxy_async();      // the stage was rewritten through the generic proxy; the next writer is the TMA
        if (lane == 0) ptx::mbar_arrive(empty_a + 8u * st);
    }
}

// The tile kernel's row schedule, checked with the device's own fp32 coordinate arithmetic (ATen's): the source row of output row oy
// must be the exact-arithmetic floor on every row — schedule 0: floor((4 oy - 1) / 6) for x (3:2) and floor((oy - 1) / 3) for the
// residual (3:1); schedule n: floor((2 oy + 1 - n) / 2n) for x (n:1) and floor((2 oy + 1 - 2n) / 4n) for the residual (2n:1).  Where
// the exact coordinate is an integer (every third row at 3:1) the rounding of scale = (float)in / out decides which side the floor falls.
// Returns the schedule, or -1 (the pair kernel handles everything else).
static int floor_div(int a, int b) { return (a >= 0 ? a : a - b + 1) / b; }
static int row_pattern(int H, int rH, int oH) {
    int pat = -1;
    if ((long)H * 3 == (long)oH * 2 && (long)rH * 3 == (long)oH) pat = 0;
    else if (H > 0 && oH % H == 0 && (long)rH * 2 * (oH / H) == (long)oH) pat = oH / H;
    if (!(pat == 0 || pat == 2 || pat == 3 || pat == 4 || pat == 6) || oH % (pat ? 8 * pat : 12) != 0) return -1;
    static thread_local int key[3] = {0, 0, 0}, val = -1;
    if (key[0] == H && key[1] == rH && key[2] == oH) return val;
    const float sx = (float)H / (float)oH, sr = (float)rH / (float)oH;
    bool ok = true;
    for (int oy = 0; oy < oH && ok; ++oy) {
        int ix = (int)floorf(fmaf(sx, (float)oy + 0.5f, -0.5f));
        int ir = (int)floorf(fmaf(sr, (float)oy + 0.5f, -0.5f));
        if (ix > H - 1) ix = H - 1;
        if (ir > rH - 1) ir = rH - 1;
        const int ex = pat == 0 ? floor_div(4 * oy - 1, 6) : floor_div(2 * oy + 1 - pat, 2 * pat);
        const int er = pat == 0 ? floor_div(oy - 1, 3) : floor_div(2 * oy + 1 - 2 * pat, 4 * pat);
        ok = ix == ex && ir == er;
    }
    key[0] = H; key[1] = rH; key[2] = oH; val = ok ? pat : -1;
    return val;
}

// triangle-filter taps for one output index: [lo, lo+n) and the normalisation 1/sum
__device__ __forceinline__ void aa_range(int dst, int in_size, int out_size, int &lo, int &n, float &center, float &inv,
                                         float &norm) {
    const float scale = (float)in_size / (float)out_size;
    const float support = scale >= 1.f ? scale : 1.f;
    center = scale * ((float)dst + 0.5f);
    inv = scale >= 1.f ? 1.f / scale : 1.f;
    lo = max((int)(center - support + 0.5f), 0);
    n = min((int)(center + support + 0.5f), in_size) - lo;
    float tot = 0.f;
    for (int j = 0; j < n; ++j) tot += fmaxf(0.f, 1.f - fabsf(((float)(j + lo) - center + 0.5f) * inv));
    norm = tot != 0.f ? 1.f / tot : 0.f;
}

// one output value of one plane p (the same operations, in the same order, for every output form)
template <typename T>
__device__ __forceinline__ float resize_aa_value(const T *__restrict__ p, int W, int ylo, int yn, float yc, float yi, float ynorm, int xlo,
                                                 int xn, float xc, float xi, float xnorm) {
    float acc = 0.f;
    for (int a = 0; a < yn; ++a) {
        const float wy = fmaxf(0.f, 1.f - fabsf(((float)(a + ylo) - yc + 0.5f) * yi)) * ynorm;
        float t = 0.f;
        for (int c = 0; c < xn; ++c) {
            const float wx = fmaxf(0.f, 1.f - fabsf(((float)(c + xlo) - xc + 0.5f) * xi)) * xnorm;
            t = fmaf(wx, to_f(p[(long)(a + ylo) * W + c + xlo]), t);
        }
        acc = fmaf(wy, t, acc);
    }
    return acc;
}

// PX4 = false: a thread per (plane = b * 3 + c, pixel); PX4 = true (4-byte uint8 pixels, layout 3 / 5): a thread per (frame b, pixel)
// computes the three planes and writes the pixel once, its alpha from the plane `alpha` (NULL: 255)
template <typename T, typename TO, bool PX4 = false>
__global__ void __launch_bounds__(256) resize_aa_kernel(const T *__restrict__ in, TO *__restrict__ out, int H, int W, int oH,
                                                        int oW, int clamp, int layout, const uint8_t *__restrict__ alpha) {
    const int ox = blockIdx.x * 64 + (threadIdx.x & 63);
    const int oy = blockIdx.y * 4 + (threadIdx.x >> 6);
    const long plane = blockIdx.z;
    if (ox >= oW || oy >= oH) return;
    int ylo, yn, xlo, xn;
    float yc, yi, ynorm, xc, xi, xnorm;
    aa_range(oy, H, oH, ylo, yn, yc, yi, ynorm);
    aa_range(ox, W, oW, xlo, xn, xc, xi, xnorm);
    if constexpr (PX4) {
        float v[3];
#pragma unroll 1
        for (int c = 0; c < 3; ++c) {
            v[c] = resize_aa_value(in + (plane * 3 + c) * H * W, W, ylo, yn, yc, yi, ynorm, xlo, xn, xc, xi, xnorm);
            if (clamp) v[c] = fminf(fmaxf(v[c], 0.f), 1.f);
        }
        store_px4(out, (plane * oH + oy) * oW + ox, layout, v[0], v[1], v[2], alpha);
        return;
    }
    float acc = resize_aa_value(in + plane * H * W, W, ylo, yn, yc, yi, ynorm, xlo, xn, xc, xi, xnorm);
    if (clamp) acc = fminf(fmaxf(acc, 0.f), 1.f);
    if (layout == 0) {
        out[(plane * oH + oy) * oW + ox] = from_f<TO>(acc);
    } else {
        const long b = plane / 3;
        const int c = (int)(plane - 3 * b);
        out[((b * oH + oy) * oW + ox) * 3 + (layout == 2 ? 2 - c : c)] = from_f<TO>(acc);
    }
}

// interleaved uint8 frames (B,H,W,PX) -> planar RGB (B,3,H,W): four pixels per thread, 4 PX bytes in, 3 x 4 bytes out.  PX = 3: RGB /
// BGR; PX = 4: RGBA / BGRA, one aligned 32-bit load per pixel, the alpha bytes are not read into the result
template <int PX>
__global__ void __launch_bounds__(256) frames_to_planar_kernel(const uint8_t *__restrict__ in, uint8_t *__restrict__ out, long plane,
                                                               int swap) {
    pdl_trigger();
    pdl_wait();
    const long b = blockIdx.y;
    const long q = ((long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (q >= plane) return;
    const uint8_t *src = in + (b * plane + q) * PX;
    uint8_t *dst = out + b * 3 * plane + q;
    const int c0 = swap ? 2 : 0, c2 = 2 - c0;
    if (q + 4 <= plane && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst) | (uintptr_t)plane) & 3) == 0) {
        const uint32_t w0 = reinterpret_cast<const uint32_t *>(src)[0], w1 = reinterpret_cast<const uint32_t *>(src)[1],
                       w2 = reinterpret_cast<const uint32_t *>(src)[2];
        uint32_t ch0, ch1, ch2;
        if constexpr (PX == 3) {
            // bytes: w0 = p0c0 p0c1 p0c2 p1c0 | w1 = p1c1 p1c2 p2c0 p2c1 | w2 = p2c2 p3c0 p3c1 p3c2
            ch0 = __byte_perm(__byte_perm(w0, w1, 0x0630), w2, 0x5210);      // p0c0 p1c0 p2c0 p3c0
            ch1 = __byte_perm(__byte_perm(w0, w1, 0x0741), w2, 0x6210);      // p0c1 p1c1 p2c1 p3c1
            ch2 = __byte_perm(__byte_perm(w0, w1, 0x0052), w2, 0x7410);      // p0c2 p1c2 p2c2 p3c2
        } else {
            // word i = pixel i: pic0 pic1 pic2 alpha; channel c of pixels 0, 1 and of pixels 2, 3, then the two halves
            const uint32_t w3 = reinterpret_cast<const uint32_t *>(src)[3];
            ch0 = __byte_perm(__byte_perm(w0, w1, 0x0040), __byte_perm(w2, w3, 0x0040), 0x5410);
            ch1 = __byte_perm(__byte_perm(w0, w1, 0x0051), __byte_perm(w2, w3, 0x0051), 0x5410);
            ch2 = __byte_perm(__byte_perm(w0, w1, 0x0062), __byte_perm(w2, w3, 0x0062), 0x5410);
        }
        reinterpret_cast<uint32_t *>(dst + c0 * plane)[0] = ch0;
        reinterpret_cast<uint32_t *>(dst + plane)[0] = ch1;
        reinterpret_cast<uint32_t *>(dst + c2 * plane)[0] = ch2;
    } else {
        for (int i = 0; i < 4 && q + i < plane; ++i) {
            dst[c0 * plane + i] = src[PX * i];
            dst[plane + i] = src[PX * i + 1];
            dst[c2 * plane + i] = src[PX * i + 2];
        }
    }
}

// ---- the alpha plane of 4-byte frames, resampled (bicubic, ATen's taps and weights; include/tu_b200.h: tu_resample_alpha) -------
// Every step is one correctly rounded fp32 operation, the tap weights included: they are the fp32 tensor arithmetic of
// oracle/upscaler_oracle.py::_cubic_taps, operation for operation, so that a CPU evaluation gives the same bits.
__device__ __forceinline__ float cubic1_rn(float x) {          // ((A + 2) x - (A + 3)) x x + 1, A = -0.75
    return __fadd_rn(__fmul_rn(__fmul_rn(__fadd_rn(__fmul_rn(1.25f, x), -2.25f), x), x), 1.f);
}
__device__ __forceinline__ float cubic2_rn(float x) {          // ((A x - 5 A) x + 8 A) x - 4 A
    return __fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(-0.75f, x), 3.75f), x), -6.f), x), 3.f);
}
__device__ __forceinline__ void cubic_taps_rn(int dst, int in_size, float scale, int (&idx)[4], float (&w)[4]) {
    const float src = fmaf(scale, (float)dst + 0.5f, -0.5f);
    const int i0 = min((int)floorf(src), in_size - 1);
    const float t = fminf(fmaxf(__fadd_rn(src, -(float)i0), 0.f), 1.f), u = __fadd_rn(1.f, -t);
    w[0] = cubic2_rn(__fadd_rn(t, 1.f)); w[1] = cubic1_rn(t); w[2] = cubic1_rn(u); w[3] = cubic2_rn(__fadd_rn(u, 1.f));
#pragma unroll
    for (int j = 0; j < 4; ++j) idx[j] = min(max(i0 + j - 1, 0), in_size - 1);
}

// A thread writes four consecutive output bytes of one row (one 32-bit store where the row allows it).  Memory bound: the 16 taps
// of an output are mostly L1 / L2 hits of the 4-byte input pixels (only their alpha byte is used).
constexpr int RA_X = 64, RA_Y = 4;
__global__ void __launch_bounds__(RA_X * RA_Y) resample_alpha_kernel(const uint8_t *__restrict__ in, uint8_t *__restrict__ out, int H, int W,
                                                                     int oH, int oW, float sy, float sx) {
    pdl_trigger();
    pdl_wait();
    const int ox0 = (blockIdx.x * RA_X + threadIdx.x) * 4, oy = blockIdx.y * RA_Y + threadIdx.y;
    const long b = blockIdx.z;
    if (ox0 >= oW || oy >= oH) return;
    int ty[4], tx[4];
    float wy[4], wx[4];
    cubic_taps_rn(oy, H, sy, ty, wy);
    const uint8_t *f = in + b * H * W * 4 + 3;
    uint32_t word = 0;
    const int n = min(4, oW - ox0);
    for (int k = 0; k < n; ++k) {
        cubic_taps_rn(ox0 + k, W, sx, tx, wx);
        float a = 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const uint8_t *row = f + (long)ty[i] * W * 4;
            float acc = 0.f;
#pragma unroll
            for (int j = 0; j < 4; ++j) acc = __fadd_rn(acc, __fmul_rn(u8_to_float(row[tx[j] * 4]), wx[j]));
            a = __fadd_rn(a, __fmul_rn(acc, wy[i]));
        }
        const uint32_t code = (uint32_t)fminf(fmaxf(floorf(__fadd_rn(a, 0.5f)), 0.f), 255.f);
        word |= code << (8 * k);
    }
    uint8_t *o = out + (b * oH + oy) * oW + ox0;
    if (n == 4 && (reinterpret_cast<uintptr_t>(o) & 3) == 0) {
        *reinterpret_cast<uint32_t *>(o) = word;
    } else {
        for (int k = 0; k < n; ++k) o[k] = (uint8_t)(word >> (8 * k));
    }
}

// ---- 4:2:0 video frames (NV12 / P010, type-0 chroma siting) <-> planar RGB (fp16 / fp32) ------------------------------------------
// Every step is one correctly rounded fp32 operation (__fmul_rn / __fadd_rn / __fdiv_rn: -O3 would contract a*b+c into an FMA), in
// the order include/tu_b200.h states, so that the kernels give the bits of a plain fp32 evaluation of the formulas.
struct YuvCoef {
    float yo, ys, cs;                   // y' = (Y - yo) / ys, c' = (C - mid) / cs (mid: Yuv420<TS>::mid)
    float a_rv, a_gu, a_gv, a_bu;       // YUV -> RGB
    float kr, kg, kb;                   // RGB -> Y'
    float cb_r, cb_g, cr_g, cr_b;       // RGB -> Cb', Cr' (the 0.5 terms are exact); codes: ys Y' + yo, cs C' + mid
};

// coefficients of a colour code, each computed in double and rounded once to float.  P010 codes (TU_U16) take the 10-bit offsets
// and scales, and may name the BT.2020 matrix
static YuvCoef yuv_coef(int code) {
    const bool bt601 = code & TU_YUV_BT601, bt2020 = code & TU_YUV_BT2020, full = code & TU_YUV_FULL_RANGE;
    const bool p010 = dtype_base(code) == TU_U16;
    const double kr = bt2020 ? 0.2627 : bt601 ? 0.299 : 0.2126, kb = bt2020 ? 0.0593 : bt601 ? 0.114 : 0.0722, kg = 1.0 - kr - kb;
    YuvCoef k;
    k.yo = full ? 0.f : p010 ? 64.f : 16.f;
    k.ys = full ? (p010 ? 1023.f : 255.f) : p010 ? 876.f : 219.f;
    k.cs = full ? (p010 ? 1023.f : 255.f) : p010 ? 896.f : 224.f;
    k.a_rv = (float)(2.0 * (1.0 - kr));
    k.a_bu = (float)(2.0 * (1.0 - kb));
    k.a_gu = (float)(-2.0 * (1.0 - kb) * kb / kg);
    k.a_gv = (float)(-2.0 * (1.0 - kr) * kr / kg);
    k.kr = (float)kr;
    k.kg = (float)kg;
    k.kb = (float)kb;
    k.cb_r = (float)(-kr / (2.0 * (1.0 - kb)));
    k.cb_g = (float)(-kg / (2.0 * (1.0 - kb)));
    k.cr_g = (float)(-kg / (2.0 * (1.0 - kr)));
    k.cr_b = (float)(-kb / (2.0 * (1.0 - kr)));
    return k;
}

// sample formats: NV12 holds one 8-bit code per byte; P010 one 10-bit code in the high bits of a little-endian uint16 word (the low
// 6 bits are ignored on read and zero on write).  A pair of samples (two luma, or U then V) is one 2-byte / 4-byte access.
template <typename TS> struct Yuv420;
template <> struct Yuv420<uint8_t> {
    typedef uchar2 Pair;
    static constexpr int shift = 0;
    static constexpr float mid = 128.f, cmax = 255.f;
    static __device__ __forceinline__ Pair pair(uint8_t a, uint8_t b) { return make_uchar2(a, b); }
};
template <> struct Yuv420<uint16_t> {
    typedef ushort2 Pair;
    static constexpr int shift = 6;
    static constexpr float mid = 512.f, cmax = 1023.f;
    static __device__ __forceinline__ Pair pair(uint16_t a, uint16_t b) { return make_ushort2(a, b); }
};

// Frame addressing of the 4:2:0 kernels: where row r of a frame's luma and chroma planes starts.  blockIdx.y is the frame of the launch
// (the RGB side is always a dense (B, 3, H, W) batch indexed by it).  Param is the kernel parameter that carries the frames.
// Dense: one (B, 3H/2, W) buffer, row pitch W samples, the chroma plane right after the luma plane, frame b at b * 3HW/2.
template <typename TS> struct Dense420 {
    typedef TS *__restrict__ Param;
    TS *y, *uv;
    int W;
    static __device__ __forceinline__ Dense420 frame(Param p, int H, int W) {
        const long plane = (long)H * W;
        TS *f = p + (long)blockIdx.y * (plane + plane / 2);
        return {f, f + plane, W};
    }
    __device__ __forceinline__ TS *yrow(int r) const { return y + (long)r * W; }
    __device__ __forceinline__ TS *uvrow(int r) const { return uv + (long)r * W; }
};
// Surfaces: frame blockIdx.y of a table of up to kPlanesPerLaunch TuFramePlanes passed by value in the kernel parameters (no copy of
// descriptors to the device, so a captured graph needs no host memory alive); a larger batch is several launches.  64 x 32 bytes keeps
// the parameters of a launch at about 2 KB, within the classic 4 KB limit.
constexpr int kPlanesPerLaunch = 64;
template <typename TS> struct Planes420 {
    struct Param { TuFramePlanes f[kPlanesPerLaunch]; };
    TS *y, *uv;
    long long yp, uvp;
    static __device__ __forceinline__ Planes420 frame(const Param &p, int, int) {
        const TuFramePlanes &d = p.f[blockIdx.y];
        return {(TS *)d.y, (TS *)d.uv, d.y_pitch, d.uv_pitch};
    }
    __device__ __forceinline__ TS *yrow(int r) const { return (TS *)((char *)y + (long long)r * yp); }
    __device__ __forceinline__ TS *uvrow(int r) const { return (TS *)((char *)uv + (long long)r * uvp); }
};

__device__ __forceinline__ float clamp01(float v) { return fminf(fmaxf(v, 0.f), 1.f); }
// two horizontally adjacent RGB values of one plane (an aligned half2 / float2)
__device__ __forceinline__ void store_rgb2(f16 *p, float a, float b) { *reinterpret_cast<__half2 *>(p) = __floats2half2_rn(a, b); }
__device__ __forceinline__ void store_rgb2(float *p, float a, float b) { *reinterpret_cast<float2 *>(p) = make_float2(a, b); }
__device__ __forceinline__ float2 load_rgb2(const f16 *p) { return __half22float2(*reinterpret_cast<const __half2 *>(p)); }
__device__ __forceinline__ float2 load_rgb2(const float *p) { return *reinterpret_cast<const float2 *>(p); }

// One thread per chroma sample (i, j): the 2x2 luma block rows 2i..2i+1, columns 2j..2j+1.  Bilinear chroma: luma row 2i takes
// (C[i-1] + 3 C[i]) / 4, row 2i+1 (3 C[i] + C[i+1]) / 4; column 2j takes chroma column j, column 2j+1 the mean of j and j+1 (edges
// clamped).  These are integer sums (at most 8 * 1023) times 1/4 or 1/8: exact in fp32.
template <typename TS, typename TR, typename A>
__global__ void __launch_bounds__(256) yuv420_to_rgb_kernel(typename A::Param in, TR *__restrict__ out, int H, int W, YuvCoef k) {
    typedef Yuv420<TS> F;
    typedef typename F::Pair P;
    constexpr int s = F::shift;
    pdl_trigger();
    pdl_wait();
    const int Hc = H >> 1, Wc = W >> 1;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= Hc * Wc) return;
    const int i = t / Wc, j = t - i * Wc;
    const long plane = (long)H * W;
    const A f = A::frame(in, H, W);
    const int im = max(i - 1, 0), ip = min(i + 1, Hc - 1), jp = min(j + 1, Wc - 1);
    const P cm0 = *reinterpret_cast<const P *>(f.uvrow(im) + 2 * j), cm1 = *reinterpret_cast<const P *>(f.uvrow(im) + 2 * jp);
    const P c00 = *reinterpret_cast<const P *>(f.uvrow(i) + 2 * j), c01 = *reinterpret_cast<const P *>(f.uvrow(i) + 2 * jp);
    const P cp0 = *reinterpret_cast<const P *>(f.uvrow(ip) + 2 * j), cp1 = *reinterpret_cast<const P *>(f.uvrow(ip) + 2 * jp);
    // vertical sums (x4) of U and V for the top (2i) and bottom (2i+1) luma rows, at chroma columns j and j+1
    const int ut0 = (cm0.x >> s) + 3 * (c00.x >> s), ut1 = (cm1.x >> s) + 3 * (c01.x >> s);
    const int ub0 = 3 * (c00.x >> s) + (cp0.x >> s), ub1 = 3 * (c01.x >> s) + (cp1.x >> s);
    const int vt0 = (cm0.y >> s) + 3 * (c00.y >> s), vt1 = (cm1.y >> s) + 3 * (c01.y >> s);
    const int vb0 = 3 * (c00.y >> s) + (cp0.y >> s), vb1 = 3 * (c01.y >> s) + (cp1.y >> s);
    const int us[4] = {2 * ut0, ut0 + ut1, 2 * ub0, ub0 + ub1}, vs[4] = {2 * vt0, vt0 + vt1, 2 * vb0, vb0 + vb1};   // x8
    const P y0 = *reinterpret_cast<const P *>(f.yrow(2 * i) + 2 * j);
    const P y1 = *reinterpret_cast<const P *>(f.yrow(2 * i + 1) + 2 * j);
    const int ys[4] = {y0.x >> s, y0.y >> s, y1.x >> s, y1.y >> s};
    float r[4], g[4], bl[4];
#pragma unroll
    for (int p = 0; p < 4; ++p) {
        const float yn = __fdiv_rn(__fadd_rn((float)ys[p], -k.yo), k.ys);
        const float un = __fdiv_rn(__fadd_rn(__fmul_rn((float)us[p], 0.125f), -F::mid), k.cs);
        const float vn = __fdiv_rn(__fadd_rn(__fmul_rn((float)vs[p], 0.125f), -F::mid), k.cs);
        r[p] = clamp01(__fadd_rn(yn, __fmul_rn(k.a_rv, vn)));
        g[p] = clamp01(__fadd_rn(__fadd_rn(yn, __fmul_rn(k.a_gu, un)), __fmul_rn(k.a_gv, vn)));
        bl[p] = clamp01(__fadd_rn(yn, __fmul_rn(k.a_bu, un)));
    }
    TR *o = out + (long)blockIdx.y * 3 * plane + (long)(2 * i) * W + 2 * j;
    store_rgb2(o, r[0], r[1]);
    store_rgb2(o + W, r[2], r[3]);
    store_rgb2(o + plane, g[0], g[1]);
    store_rgb2(o + plane + W, g[2], g[3]);
    store_rgb2(o + 2 * plane, bl[0], bl[1]);
    store_rgb2(o + 2 * plane + W, bl[2], bl[3]);
}

template <typename TS>
__device__ __forceinline__ TS yuv_code(float v) {         // min(max(floor(v + 0.5), 0), cmax), stored << shift
    return (TS)((int)fminf(fmaxf(floorf(__fadd_rn(v, 0.5f)), 0.f), Yuv420<TS>::cmax) << Yuv420<TS>::shift);
}

// One thread per chroma sample (i, j): its (U, V) pair and its 2x2 luma block.  Chroma filter (type-0 siting): the column sums
// v(c) = P[2i][c] + P[2i+1][c] weighted 1, 2, 1 over columns 2j-1 (clamped at 0), 2j, 2j+1, times 1/8, per channel.
template <typename TR, typename TS, typename A>
__global__ void __launch_bounds__(256) rgb_to_yuv420_kernel(const TR *__restrict__ in, typename A::Param out, int H, int W, YuvCoef k) {
    typedef Yuv420<TS> F;
    typedef typename F::Pair P;
    pdl_trigger();
    pdl_wait();
    const int Hc = H >> 1, Wc = W >> 1;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= Hc * Wc) return;
    const int i = t / Wc, j = t - i * Wc;
    const long plane = (long)H * W;
    const TR *src = in + (long)blockIdx.y * 3 * plane + (long)(2 * i) * W;
    const int cl = max(2 * j - 1, 0);
    float px[3][4], bar[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const TR *s = src + c * plane;
        const float2 a = load_rgb2(s + 2 * j);
        const float2 b = load_rgb2(s + W + 2 * j);
        const float v0 = __fadd_rn(to_f(s[cl]), to_f(s[W + cl]));
        const float v1 = __fadd_rn(a.x, b.x), v2 = __fadd_rn(a.y, b.y);
        px[c][0] = a.x; px[c][1] = a.y; px[c][2] = b.x; px[c][3] = b.y;
        bar[c] = __fmul_rn(__fadd_rn(__fadd_rn(v0, __fmul_rn(2.f, v1)), v2), 0.125f);
    }
    TS yq[4];
#pragma unroll
    for (int p = 0; p < 4; ++p) {
        const float yl = __fadd_rn(__fadd_rn(__fmul_rn(k.kr, px[0][p]), __fmul_rn(k.kg, px[1][p])), __fmul_rn(k.kb, px[2][p]));
        yq[p] = yuv_code<TS>(__fadd_rn(__fmul_rn(k.ys, yl), k.yo));
    }
    const float cb = __fadd_rn(__fadd_rn(__fmul_rn(k.cb_r, bar[0]), __fmul_rn(k.cb_g, bar[1])), __fmul_rn(0.5f, bar[2]));
    const float cr = __fadd_rn(__fadd_rn(__fmul_rn(0.5f, bar[0]), __fmul_rn(k.cr_g, bar[1])), __fmul_rn(k.cr_b, bar[2]));
    const A f = A::frame(out, H, W);
    *reinterpret_cast<P *>(f.yrow(2 * i) + 2 * j) = F::pair(yq[0], yq[1]);
    *reinterpret_cast<P *>(f.yrow(2 * i + 1) + 2 * j) = F::pair(yq[2], yq[3]);
    *reinterpret_cast<P *>(f.uvrow(i) + 2 * j) =
        F::pair(yuv_code<TS>(__fadd_rn(__fmul_rn(k.cs, cb), F::mid)), yuv_code<TS>(__fadd_rn(__fmul_rn(k.cs, cr), F::mid)));
}

}  // namespace tu

using namespace tu;

thread_local int tu::g_bicubic_tile = 0;      // debug key "bicubic_tile": rows per CTA of the row-schedule kernel: 0 = by grid size (default), 1 = the smaller tile, 2 = the larger
thread_local int tu::g_bicubic_pair = 2;      // debug key "bicubic_pair": 2 = two output columns per thread + the unrolled fixed-row-pattern kernel where it applies (default), 3 = the same with the streaming form of that kernel (measured slower), 1 = the pair kernel only, 0 = the one-column strip kernel

// (W, H, 3, B) view of an NCHW image of dtype code `dtype` for the tile loads; box = (cols, rows, 3, 1)
static bool encode_image_map(CUtensorMap *tm, const void *ptr, int dtype, int B, int H, int W, int box_rows, int box_cols) {
    TcEncodeFn enc = tc_encode_fn();
    const int elem_bytes = (int)dtype_size(dtype);
    if (!enc || box_rows > 256 || box_cols > 256) return false;
    cuuint64_t dims[4] = {(cuuint64_t)W, (cuuint64_t)H, 3, (cuuint64_t)B};
    cuuint64_t strides[3] = {(cuuint64_t)W * elem_bytes, (cuuint64_t)H * W * elem_bytes, (cuuint64_t)3 * H * W * elem_bytes};
    cuuint32_t box[4] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows, 3, 1}, es[4] = {1, 1, 1, 1};
    return enc(tm, tc_image_map_dtype(dtype), 4, (void *)ptr, dims, strides,
               box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

int tu::bicubic_add_clamp_alpha(const void *x, int in_dtype, int H, int W, const float *res, int rH, int rW, void *out, int out_dtype,
                                int B, int outH, int outW, int clamp, const uint8_t *alpha, cudaStream_t st) {
    TU_CHECK_ARG(x && out && B > 0 && H > 0 && W > 0 && outH > 0 && outW > 0, "bicubic_add_clamp: bad argument");
    const int layout = dtype_layout(out_dtype);
    out_dtype = dtype_base(out_dtype);
    TU_CHECK_ARG((in_dtype == TU_F32 || in_dtype == TU_BF16 || in_dtype == TU_F16 || in_dtype == TU_U8) &&
                     (out_dtype == TU_F32 || out_dtype == TU_BF16 || out_dtype == TU_F16 || out_dtype == TU_U8),
                 "bicubic_add_clamp: bad dtype");
    TU_CHECK_ARG(layout == 0 || (out_dtype == TU_U8 && layout_is_interleaved(layout)), "bicubic_add_clamp: interleaved layouts are for uint8 frames");
    const bool px4 = layout_is_px4(layout);
    TU_CHECK_ARG(!px4 || (reinterpret_cast<uintptr_t>(out) & 3) == 0, "bicubic_add_clamp: a 4-byte (RGBA / BGRA) output must be 4-byte aligned");
    if (!px4) alpha = nullptr;
    const int eb = (int)dtype_size(in_dtype), ob = (int)dtype_size(out_dtype);
    BicubicTileGeom g;
    g.sxh = (float)H / (float)outH; g.sxw = (float)W / (float)outW;
    g.srh = res ? (float)rH / (float)outH : 0.f; g.srw = res ? (float)rW / (float)outW : 0.f;
    size_t tile_bytes = 0;
    CUtensorMap tx, tr;
    // source footprint of a bh x 128 output tile (+4 taps, +2 for fp32 rounding of the coordinates), cols padded to 16 bytes
    auto plan = [&](int bh) -> bool {
        g.xr = (int)((long)(bh - 1) * H / outH) + 6;
        g.xc = ((int)((long)(BS_W - 1) * W / outW) + 8 + (16 / eb - 1) + 15) & ~15;        // + alignment slack of the first column
        g.rr = res ? (int)((long)(bh - 1) * rH / outH) + 6 : 0;
        g.rc = res ? ((int)((long)(BS_W - 1) * rW / outW) + 8 + 3 + 3) & ~3 : 0;
        const size_t x_bytes = ((size_t)3 * g.xr * g.xc * eb + 127) & ~(size_t)127;
        tile_bytes = x_bytes + (size_t)3 * g.rr * g.rc * 4;
        memset(&tx, 0, sizeof(tx));
        memset(&tr, 0, sizeof(tr));
        bool ok = tile_bytes <= 96 * 1024 && ((size_t)W * eb) % 16 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0 &&
                  (!res || (((size_t)rW * 4) % 16 == 0 && (reinterpret_cast<uintptr_t>(res) & 15) == 0));
        return ok && encode_image_map(&tx, x, in_dtype, B, H, W, g.xr, g.xc) && (!res || encode_image_map(&tr, res, TU_F32, B, rH, rW, g.rr, g.rc));
    };
    // two output columns per thread: TMA tiles, even output width, pair stores aligned
    const bool pair = g_bicubic_pair && (outW % 2) == 0 && (reinterpret_cast<uintptr_t>(out) % (px4 ? 8 : 2 * ob)) == 0 && plan(PAIR_H);
    // periodic row schedules (x1.5 outputs such as 720p -> 1080p, x3 outputs such as 720p -> 4K): the unrolled circular-window kernel
    const int pat = pair && g_bicubic_pair >= 2 && res && clamp && (in_dtype == TU_BF16 || in_dtype == TU_F16 || in_dtype == TU_U8) &&
                            W <= outW && rW <= outW
                        ? row_pattern(H, rH, outH)
                        : -1;
    // rows per CTA: the larger tile as soon as it still gives every SM a CTA (measured at 720p -> 1080p, profiles/r3_ab_bicubic_tile_rows.log:
    // 1 / 2 / 4 / 8 frames = 16.3 -> 14.8, 23.1 -> 21.8, 34.1 -> 34.7, 63.3 -> 59.2 us), else the smaller one
    int tile_rows = 0;
    bool r32 = false;
    if (pat >= 0) {
        const long ctas_big = (long)ceil_div(outW, BS_W) * ceil_div(outH, sched_tile(pat, true)) * B;
        tile_rows = sched_tile(pat, g_bicubic_tile ? g_bicubic_tile == 2 : ctas_big >= (long)device_sm_count());
        if (!(r32 = plan(tile_rows))) plan(PAIR_H);            // or back to the pair kernel's plan
    }
    static_assert(RowSched<0>::BIG <= R32_MAXTILE && RowSched<2>::BIG <= R32_MAXTILE && RowSched<3>::BIG <= R32_MAXTILE &&
                      RowSched<4>::BIG <= R32_MAXTILE && RowSched<6>::BIG <= R32_MAXTILE && 2 * R32_MAXTILE <= R32_T,
                  "the vertical table is filled in one pass of the CTA's threads");
    const bool tma = pair || plan(BS_H);
    dim3 grid(ceil_div(outW, BS_W), ceil_div(outH, pair ? PAIR_H : BS_H), B);
#define TU_BIC_PAIR(TI, TO, PX4)                                                                                                \
    do {                                                                                                                        \
        static PerDeviceFlag attr_done;                                                                                          \
        if (!attr_done.is_set()) {                                                                                                       \
            cudaError_t e = cudaFuncSetAttribute(bicubic_add_clamp_pair_kernel<TI, TO, true, PX4>,                             \
                                                 cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);                      \
            if (e == cudaSuccess)                                                                                               \
                e = cudaFuncSetAttribute(bicubic_add_clamp_pair_kernel<TI, TO, false, PX4>,                                    \
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);                              \
            if (e != cudaSuccess) return cuda_fail(e, "bicubic smem attribute");                                                \
            attr_done.set();                                                                                                   \
        }                                                                                                                       \
        if (res)                                                                                                                \
            launch_pdl(bicubic_add_clamp_pair_kernel<TI, TO, true, PX4>, grid, dim3(BS_W / 2), tile_bytes + 128, st, tx, tr, g, H, W, rH, \
                       rW, (TO *)out, outH, outW, clamp, layout, alpha);                                                       \
        else                                                                                                                    \
            launch_pdl(bicubic_add_clamp_pair_kernel<TI, TO, false, PX4>, grid, dim3(BS_W / 2), tile_bytes + 128, st, tx, tr, g, H, W, rH, \
                       rW, (TO *)out, outH, outW, clamp, layout, alpha);                                                       \
    } while (0)
#define TU_BIC(TI, TO, PX4)                                                                                                     \
    do {                                                                                                                        \
        if (tma) {                                                                                                              \
            static PerDeviceFlag attr_done;                                                                                      \
            if (!attr_done.is_set()) {                                                                                                   \
                cudaError_t e = cudaFuncSetAttribute(bicubic_add_clamp_strip_kernel<TI, TO, 1, PX4>,                         \
                                                     cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);                  \
                if (e == cudaSuccess)                                                                                           \
                    e = cudaFuncSetAttribute(bicubic_add_clamp_strip_kernel<TI, TO, 2, PX4>,                                    \
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);                          \
                if (e != cudaSuccess) return cuda_fail(e, "bicubic smem attribute");                                            \
                attr_done.set();                                                                                               \
            }                                                                                                                   \
            if (res)                                                                                                            \
                launch_pdl(bicubic_add_clamp_strip_kernel<TI, TO, 1, PX4>, grid, dim3(BS_W), tile_bytes + 128, st, tx, tr, g, (const TI *)x, \
                           H, W, res, rH, rW, (TO *)out, outH, outW, clamp, layout, alpha);                                 \
            else                                                                                                                \
                launch_pdl(bicubic_add_clamp_strip_kernel<TI, TO, 2, PX4>, grid, dim3(BS_W), tile_bytes + 128, st, tx, tr, g, (const TI *)x, \
                           H, W, res, rH, rW, (TO *)out, outH, outW, clamp, layout, alpha);                                 \
        } else {                                                                                                                \
            bicubic_add_clamp_strip_kernel<TI, TO, 0, PX4><<<grid, BS_W, 0, st>>>(tx, tr, g, (const TI *)x, H, W, res, rH, rW, \
                                                                                       (TO *)out, outH, outW, clamp, layout, alpha); \
        }                                                                                                                       \
    } while (0)
#define TU_BIC2_A(TI, TO, PX4)        \
    do {                              \
        if (pair) TU_BIC_PAIR(TI, TO, PX4); \
        else TU_BIC(TI, TO, PX4);     \
    } while (0)
#define TU_BIC2(TI, TO) TU_BIC2_A(TI, TO, false)
#define TU_BIC_R32_P(TI, TO, PAT, PX)                                                                                           \
    do {                                                                                                                        \
        static PerDeviceFlag attr_done;                                                                                          \
        if (!attr_done.is_set()) {                                                                                               \
            cudaError_t e = cudaFuncSetAttribute(bicubic_add_clamp_r32_kernel<TI, TO, PAT, PX>,                                 \
                                                 cudaFuncAttributeMaxDynamicSharedMemorySize, (PX == 4 ? 128 : 96) * 1024);     \
            if (e != cudaSuccess) return cuda_fail(e, "bicubic smem attribute");                                                \
            attr_done.set();                                                                                                    \
        }                                                                                                                       \
        launch_pdl(bicubic_add_clamp_r32_kernel<TI, TO, PAT, PX>, dim3(grid.x, ceil_div(outH, tile_rows), B), dim3(R32_T),      \
                   tile_bytes + 128 + (PX == 4 ? px4_stage_bytes<PAT>() + 16 : 0), st, tx, tr, g, H, W, rH, rW, (TO *)out, outH, outW, \
                   layout, tile_rows, alpha);                                                                                   \
    } while (0)
#define TU_BIC_R32_L(TI, TO, PX)                                                                                                \
    do {                                                                                                                        \
        if (pat == 0) TU_BIC_R32_P(TI, TO, 0, PX);                                                                              \
        else if (pat == 2) TU_BIC_R32_P(TI, TO, 2, PX);                                                                         \
        else if (pat == 3) TU_BIC_R32_P(TI, TO, 3, PX);                                                                         \
        else if (pat == 4) TU_BIC_R32_P(TI, TO, 4, PX);                                                                         \
        else TU_BIC_R32_P(TI, TO, 6, PX);                                                                                       \
    } while (0)
#define TU_BIC_R32(TI, TO) TU_BIC_R32_L(TI, TO, 0)
    if (r32 && pat == 0 && layout == 0 && g_bicubic_pair >= 3 && in_dtype != TU_F16 && out_dtype != TU_F16) {
        // streaming variant: strips x segments co-resident (5 CTAs per SM), <= 16 blocks of 12 rows per segment
        const int nblk = outH / 12, strips = (int)grid.x * B;
        const size_t stage = (((size_t)3 * 8 * g.xc * eb + 127) & ~(size_t)127) + (((size_t)3 * 4 * g.rc * 4 + 127) & ~(size_t)127);
        const size_t ring_bytes = R32S_NST * stage + 128;
        // CTAs per SM: 5 by registers (64 x 192 threads), fewer if the ring + 12 KB of static tables + 1 KB reserved do not fit 227 KB
        const int per_sm = (int)std::max<size_t>(1, std::min<size_t>(5, (size_t)227 * 1024 / (ring_bytes + 13 * 1024)));
        int nseg = std::max(1, std::min(nblk, device_sm_count() * per_sm / std::max(strips, 1)));
        int bps = std::min(std::max(ceil_div(nblk, nseg), std::min(3, nblk)), R32S_MAXBLK);      // at least 36 rows per CTA
        nseg = ceil_div(nblk, bps);
        CUtensorMap sx, sr;
        memset(&sx, 0, sizeof(sx));
        memset(&sr, 0, sizeof(sr));
        if (ring_bytes <= 96 * 1024 && encode_image_map(&sx, x, in_dtype, B, H, W, 8, g.xc) && encode_image_map(&sr, res, TU_F32, B, rH, rW, 4, g.rc)) {
            dim3 sgrid(grid.x, nseg, B);
#define TU_BIC_R32S(TI, TO)                                                                                                     \
    do {                                                                                                                        \
        static PerDeviceFlag attr_done;                                                                                          \
        if (!attr_done.is_set()) {                                                                                               \
            cudaError_t e = cudaFuncSetAttribute(bicubic_add_clamp_r32s_kernel<TI, TO>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                                 96 * 1024);                                                                    \
            if (e != cudaSuccess) return cuda_fail(e, "bicubic smem attribute");                                                \
            attr_done.set();                                                                                                    \
        }                                                                                                                       \
        launch_pdl(bicubic_add_clamp_r32s_kernel<TI, TO>, sgrid, dim3(R32_T), ring_bytes, st, sx, sr, g.xc, g.rc, H, W, rH, rW,   \
                   (TO *)out, outH, outW, bps);                                                                                 \
    } while (0)
            if (in_dtype == TU_BF16 && out_dtype == TU_BF16) TU_BIC_R32S(bf16, bf16);
            else if (in_dtype == TU_BF16 && out_dtype == TU_F32) TU_BIC_R32S(bf16, float);
            else if (in_dtype == TU_BF16) TU_BIC_R32S(bf16, uint8_t);
            else if (out_dtype == TU_U8) TU_BIC_R32S(uint8_t, uint8_t);
            else if (out_dtype == TU_BF16) TU_BIC_R32S(uint8_t, bf16);
            else TU_BIC_R32S(uint8_t, float);
#undef TU_BIC_R32S
            TU_CHECK_LAUNCH("bicubic_add_clamp");
            return TU_OK;
        }
    }
    if (r32 && px4) {                   // 4-byte uint8 frames
        if (in_dtype == TU_BF16) TU_BIC_R32_L(bf16, uint8_t, 4);
        else if (in_dtype == TU_F16) TU_BIC_R32_L(f16, uint8_t, 4);
        else TU_BIC_R32_L(uint8_t, uint8_t, 4);
    } else if (r32 && layout != 0) {    // interleaved uint8 frames (layouts are accepted for uint8 output only)
        if (in_dtype == TU_BF16) TU_BIC_R32_L(bf16, uint8_t, 3);
        else if (in_dtype == TU_F16) TU_BIC_R32_L(f16, uint8_t, 3);
        else TU_BIC_R32_L(uint8_t, uint8_t, 3);
    } else if (px4) {
        if (in_dtype == TU_F32) TU_BIC2_A(float, uint8_t, true);
        else if (in_dtype == TU_BF16) TU_BIC2_A(bf16, uint8_t, true);
        else if (in_dtype == TU_F16) TU_BIC2_A(f16, uint8_t, true);
        else TU_BIC2_A(uint8_t, uint8_t, true);
    } else if (r32) {
        if (in_dtype == TU_BF16 && out_dtype == TU_BF16) TU_BIC_R32(bf16, bf16);
        else if (in_dtype == TU_BF16 && out_dtype == TU_F32) TU_BIC_R32(bf16, float);
        else if (in_dtype == TU_BF16 && out_dtype == TU_F16) TU_BIC_R32(bf16, f16);
        else if (in_dtype == TU_BF16) TU_BIC_R32(bf16, uint8_t);
        else if (in_dtype == TU_F16 && out_dtype == TU_F16) TU_BIC_R32(f16, f16);
        else if (in_dtype == TU_F16 && out_dtype == TU_F32) TU_BIC_R32(f16, float);
        else if (in_dtype == TU_F16 && out_dtype == TU_BF16) TU_BIC_R32(f16, bf16);
        else if (in_dtype == TU_F16) TU_BIC_R32(f16, uint8_t);
        else if (out_dtype == TU_U8) TU_BIC_R32(uint8_t, uint8_t);
        else if (out_dtype == TU_BF16) TU_BIC_R32(uint8_t, bf16);
        else if (out_dtype == TU_F16) TU_BIC_R32(uint8_t, f16);
        else TU_BIC_R32(uint8_t, float);
    } else
    if (in_dtype == TU_F32 && out_dtype == TU_F32) TU_BIC2(float, float);
    else if (in_dtype == TU_F32 && out_dtype == TU_BF16) TU_BIC2(float, bf16);
    else if (in_dtype == TU_BF16 && out_dtype == TU_F32) TU_BIC2(bf16, float);
    else if (in_dtype == TU_BF16 && out_dtype == TU_BF16) TU_BIC2(bf16, bf16);
    else if (in_dtype == TU_U8 && out_dtype == TU_U8) TU_BIC2(uint8_t, uint8_t);
    else if (in_dtype == TU_U8 && out_dtype == TU_F32) TU_BIC2(uint8_t, float);
    else if (in_dtype == TU_U8 && out_dtype == TU_BF16) TU_BIC2(uint8_t, bf16);
    else if (in_dtype == TU_F32 && out_dtype == TU_U8) TU_BIC2(float, uint8_t);
    else if (in_dtype == TU_F16 && out_dtype == TU_F16) TU_BIC2(f16, f16);
    else if (in_dtype == TU_F16 && out_dtype == TU_F32) TU_BIC2(f16, float);
    else if (in_dtype == TU_F16 && out_dtype == TU_BF16) TU_BIC2(f16, bf16);
    else if (in_dtype == TU_F16 && out_dtype == TU_U8) TU_BIC2(f16, uint8_t);
    else if (in_dtype == TU_F32 && out_dtype == TU_F16) TU_BIC2(float, f16);
    else if (in_dtype == TU_BF16 && out_dtype == TU_F16) TU_BIC2(bf16, f16);
    else if (in_dtype == TU_U8 && out_dtype == TU_F16) TU_BIC2(uint8_t, f16);
    else TU_BIC2(bf16, uint8_t);
#undef TU_BIC2
#undef TU_BIC2_A
#undef TU_BIC_R32
#undef TU_BIC_R32_P
#undef TU_BIC_R32_L
#undef TU_BIC_PAIR
#undef TU_BIC
    TU_CHECK_LAUNCH("bicubic_add_clamp");
    return TU_OK;
}

extern "C" int tu_bicubic_add_clamp(const void *x, int in_dtype, int H, int W, const float *res, int rH, int rW, void *out,
                                    int out_dtype, int B, int outH, int outW, int clamp, void *stream) {
    return bicubic_add_clamp_alpha(x, in_dtype, H, W, res, rH, rW, out, out_dtype, B, outH, outW, clamp, nullptr, (cudaStream_t)stream);
}

extern "C" int tu_bicubic_row_schedule(int H, int rH, int outH) { return H > 0 && rH > 0 && outH > 0 ? row_pattern(H, rH, outH) : -1; }

extern "C" int tu_resize_bilinear_aa_to_alpha(const void *in, int in_dtype, const void *alpha, void *out, int out_dtype, int B, int H, int W,
                                              int outH, int outW, int clamp, void *stream) {
    TU_CHECK_ARG(in && out && B > 0 && H > 0 && W > 0 && outH > 0 && outW > 0, "resize_bilinear_aa: bad argument");
    const int layout = dtype_layout(out_dtype);
    out_dtype = dtype_base(out_dtype);
    TU_CHECK_ARG(layout == 0 || (out_dtype == TU_U8 && layout_is_interleaved(layout)), "resize_bilinear_aa: interleaved layouts are for uint8 frames");
    const bool px4 = layout_is_px4(layout);
    TU_CHECK_ARG(!px4 || (reinterpret_cast<uintptr_t>(out) & 3) == 0, "resize_bilinear_aa: a 4-byte (RGBA / BGRA) output must be 4-byte aligned");
    TU_CHECK_ARG(px4 || !alpha, "resize_bilinear_aa: an alpha plane needs a 4-byte (RGBA / BGRA) output");
    TU_CHECK_ARG(!px4 || B <= 65535, "resize_bilinear_aa: too many frames");
    cudaStream_t st = (cudaStream_t)stream;
    dim3 grid(ceil_div(outW, 64), ceil_div(outH, 4), px4 ? B : B * 3);
    const uint8_t *ap = (const uint8_t *)alpha;
#define TU_RS(TI, TO) resize_aa_kernel<TI, TO><<<grid, 256, 0, st>>>((const TI *)in, (TO *)out, H, W, outH, outW, clamp, layout, nullptr)
#define TU_RS4(TI) resize_aa_kernel<TI, uint8_t, true><<<grid, 256, 0, st>>>((const TI *)in, (uint8_t *)out, H, W, outH, outW, clamp, layout, ap)
    if (px4 && in_dtype == TU_F32) TU_RS4(float);
    else if (px4 && in_dtype == TU_BF16) TU_RS4(bf16);
    else if (px4 && in_dtype == TU_F16) TU_RS4(f16);
    else if (px4) TU_CHECK_ARG(false, "resize_bilinear_aa: bad dtype");
    else if (in_dtype == TU_F32 && out_dtype == TU_F32) TU_RS(float, float);
    else if (in_dtype == TU_BF16 && out_dtype == TU_BF16) TU_RS(bf16, bf16);
    else if (in_dtype == TU_F32 && out_dtype == TU_BF16) TU_RS(float, bf16);
    else if (in_dtype == TU_BF16 && out_dtype == TU_F32) TU_RS(bf16, float);
    else if (in_dtype == TU_F32 && out_dtype == TU_U8) TU_RS(float, uint8_t);
    else if (in_dtype == TU_BF16 && out_dtype == TU_U8) TU_RS(bf16, uint8_t);
    else if (in_dtype == TU_F16 && out_dtype == TU_F16) TU_RS(f16, f16);
    else if (in_dtype == TU_F16 && out_dtype == TU_F32) TU_RS(f16, float);
    else if (in_dtype == TU_F16 && out_dtype == TU_BF16) TU_RS(f16, bf16);
    else if (in_dtype == TU_F16 && out_dtype == TU_U8) TU_RS(f16, uint8_t);
    else if (in_dtype == TU_F32 && out_dtype == TU_F16) TU_RS(float, f16);
    else if (in_dtype == TU_BF16 && out_dtype == TU_F16) TU_RS(bf16, f16);
    else TU_CHECK_ARG(false, "resize_bilinear_aa: bad dtype");
#undef TU_RS
#undef TU_RS4
    TU_CHECK_LAUNCH("resize_bilinear_aa");
    return TU_OK;
}

extern "C" int tu_resize_bilinear_aa_to(const void *in, int in_dtype, void *out, int out_dtype, int B, int H, int W, int outH, int outW,
                                        int clamp, void *stream) {
    return tu_resize_bilinear_aa_to_alpha(in, in_dtype, nullptr, out, out_dtype, B, H, W, outH, outW, clamp, stream);
}

extern "C" int tu_resize_bilinear_aa(const void *in, int dtype, void *out, int B, int H, int W, int outH, int outW,
                                     int clamp, void *stream) {
    TU_CHECK_ARG(dtype == TU_F32 || dtype == TU_BF16 || dtype == TU_F16, "resize_bilinear_aa: bad dtype");
    return tu_resize_bilinear_aa_to(in, dtype, out, dtype, B, H, W, outH, outW, clamp, stream);
}

extern "C" int tu_frames_to_planar(const void *in, int layout, void *out, int B, int H, int W, void *stream) {
    TU_CHECK_ARG(in && out && B > 0 && H > 0 && W > 0, "frames_to_planar: bad argument");
    TU_CHECK_ARG(layout == TU_LAYOUT_HWC || layout == TU_LAYOUT_HWC_BGR || layout == TU_LAYOUT_RGBA || layout == TU_LAYOUT_BGRA,
                 "frames_to_planar: layout must be TU_LAYOUT_HWC, TU_LAYOUT_HWC_BGR, TU_LAYOUT_RGBA or TU_LAYOUT_BGRA");
    const long plane = (long)H * W;
    dim3 grid((unsigned)((plane + 1023) / 1024), B);
    const int swap = layout == TU_LAYOUT_HWC_BGR || layout == TU_LAYOUT_BGRA ? 1 : 0;
    if (layout_is_px4(layout >> 8))
        launch_pdl(frames_to_planar_kernel<4>, grid, dim3(256), 0, (cudaStream_t)stream, (const uint8_t *)in, (uint8_t *)out, plane, swap);
    else
        launch_pdl(frames_to_planar_kernel<3>, grid, dim3(256), 0, (cudaStream_t)stream, (const uint8_t *)in, (uint8_t *)out, plane, swap);
    TU_CHECK_LAUNCH("frames_to_planar");
    return TU_OK;
}

extern "C" int tu_resample_alpha(const void *frames, int code, void *alpha, int B, int H, int W, int outH, int outW, void *stream) {
    TU_CHECK_ARG(frames && alpha && B > 0 && B <= 65535 && H > 0 && W > 0 && outH > 0 && outW > 0, "resample_alpha: bad argument");
    TU_CHECK_ARG(dtype_is_px4(code), "resample_alpha: code must be TU_U8 | TU_LAYOUT_RGBA or TU_U8 | TU_LAYOUT_BGRA");
    TU_CHECK_ARG((long)H * W * 4 < (1L << 31) && (long)outH * outW < (1L << 31), "resample_alpha: frame too large");
    const dim3 grid((unsigned)ceil_div(ceil_div(outW, 4), RA_X), (unsigned)ceil_div(outH, RA_Y), (unsigned)B);
    launch_pdl(resample_alpha_kernel, grid, dim3(RA_X, RA_Y), 0, (cudaStream_t)stream, (const uint8_t *)frames, (uint8_t *)alpha, H, W, outH,
               outW, (float)H / (float)outH, (float)W / (float)outW);
    TU_CHECK_LAUNCH("resample_alpha");
    return TU_OK;
}

// NV12: code TU_U8 | TU_LAYOUT_NV12 [| colour bits], RGB fp16; P010: code TU_U16 | TU_LAYOUT_P010 [| colour bits], RGB fp32
static int check_yuv420_args(const void *frames, int code, bool p010, const void *rgb, int B, int H, int W, const char *op) {
    const std::string fmt = p010 ? "P010" : "NV12";
    TU_CHECK_ARG(frames && rgb && B > 0 && B <= 65535 && H > 0 && W > 0, std::string(op) + ": bad argument");
    if (p010)
        TU_CHECK_ARG(dtype_is_p010(code), std::string(op) + ": code must be TU_U16 | TU_LAYOUT_P010 [| TU_YUV_BT601 or TU_YUV_BT2020] "
                                                            "[| TU_YUV_FULL_RANGE]");
    else
        TU_CHECK_ARG(dtype_is_nv12(code), std::string(op) + ": code must be TU_U8 | TU_LAYOUT_NV12 [| TU_YUV_BT601] [| TU_YUV_FULL_RANGE]");
    TU_CHECK_ARG(H % 2 == 0 && W % 2 == 0, std::string(op) + ": " + fmt + " frames need an even height and width");
    TU_CHECK_ARG((long)H * W * 3 < (1L << 31), std::string(op) + ": frame too large");
    const uintptr_t fa = p010 ? 3 : 1, ra = p010 ? 7 : 3;      // a pair of samples / of RGB values is one access
    TU_CHECK_ARG((reinterpret_cast<uintptr_t>(frames) & fa) == 0 && (reinterpret_cast<uintptr_t>(rgb) & ra) == 0,
                 std::string(op) + (p010 ? ": buffers must be 4-byte (P010) and 8-byte (fp32) aligned"
                                         : ": buffers must be 2-byte (NV12) and 4-byte (fp16) aligned"));
    return TU_OK;
}

extern "C" int tu_nv12_to_rgb(const void *nv12, int code, void *rgb_f16, int B, int H, int W, void *stream) {
    if (int rc = check_yuv420_args(nv12, code, false, rgb_f16, B, H, W, "nv12_to_rgb")) return rc;
    const int n = (H / 2) * (W / 2);
    launch_pdl(yuv420_to_rgb_kernel<uint8_t, f16, Dense420<const uint8_t>>, dim3((unsigned)ceil_div(n, 256), B), dim3(256), 0, (cudaStream_t)stream,
               (const uint8_t *)nv12, (f16 *)rgb_f16, H, W, yuv_coef(code));
    TU_CHECK_LAUNCH("nv12_to_rgb");
    return TU_OK;
}

extern "C" int tu_rgb_to_nv12(const void *rgb_f16, void *nv12, int code, int B, int H, int W, void *stream) {
    if (int rc = check_yuv420_args(nv12, code, false, rgb_f16, B, H, W, "rgb_to_nv12")) return rc;
    const int n = (H / 2) * (W / 2);
    launch_pdl(rgb_to_yuv420_kernel<f16, uint8_t, Dense420<uint8_t>>, dim3((unsigned)ceil_div(n, 256), B), dim3(256), 0, (cudaStream_t)stream,
               (const f16 *)rgb_f16, (uint8_t *)nv12, H, W, yuv_coef(code));
    TU_CHECK_LAUNCH("rgb_to_nv12");
    return TU_OK;
}

extern "C" int tu_p010_to_rgb(const void *p010, int code, void *rgb_f32, int B, int H, int W, void *stream) {
    if (int rc = check_yuv420_args(p010, code, true, rgb_f32, B, H, W, "p010_to_rgb")) return rc;
    const int n = (H / 2) * (W / 2);
    launch_pdl(yuv420_to_rgb_kernel<uint16_t, float, Dense420<const uint16_t>>, dim3((unsigned)ceil_div(n, 256), B), dim3(256), 0, (cudaStream_t)stream,
               (const uint16_t *)p010, (float *)rgb_f32, H, W, yuv_coef(code));
    TU_CHECK_LAUNCH("p010_to_rgb");
    return TU_OK;
}

extern "C" int tu_rgb_to_p010(const void *rgb_f32, void *p010, int code, int B, int H, int W, void *stream) {
    if (int rc = check_yuv420_args(p010, code, true, rgb_f32, B, H, W, "rgb_to_p010")) return rc;
    const int n = (H / 2) * (W / 2);
    launch_pdl(rgb_to_yuv420_kernel<float, uint16_t, Dense420<uint16_t>>, dim3((unsigned)ceil_div(n, 256), B), dim3(256), 0, (cudaStream_t)stream,
               (const float *)rgb_f32, (uint16_t *)p010, H, W, yuv_coef(code));
    TU_CHECK_LAUNCH("rgb_to_p010");
    return TU_OK;
}

// B frame surfaces of an NV12 (code TU_U8 | TU_LAYOUT_NV12 ...) or P010 (TU_U16 | TU_LAYOUT_P010 ...) side: host-side checks of the
// code, the sizes and every descriptor, made before anything is enqueued (tu_forward_planes runs them ahead of its first kernel)
int tu::check_yuv420_planes(const TuFramePlanes *frames, int code, int B, int H, int W, const char *op) {
    TU_CHECK_ARG(frames && B > 0 && H > 0 && W > 0, std::string(op) + ": bad argument");
    TU_CHECK_ARG(dtype_is_yuv420(code), std::string(op) + ": frame planes are for NV12 (TU_U8 | TU_LAYOUT_NV12 [| colour bits]) or P010 "
                                                          "(TU_U16 | TU_LAYOUT_P010 [| colour bits]) frames only");
    const bool p010 = dtype_is_p010(code);
    const std::string fmt = p010 ? "P010" : "NV12";
    TU_CHECK_ARG(H % 2 == 0 && W % 2 == 0, std::string(op) + ": " + fmt + " frames need an even height and width");
    TU_CHECK_ARG((long)H * W * 3 < (1L << 31), std::string(op) + ": frame too large");
    const long long row = (long long)W * (p010 ? 2 : 1);
    const uintptr_t al = p010 ? 4 : 2;                              // a pair of samples is one access
    const char *al_msg = p010 ? "a multiple of 4 bytes (P010)" : "a multiple of 2 bytes (NV12)";
    for (int b = 0; b < B; ++b) {
        const TuFramePlanes &d = frames[b];
        const std::string at = std::string(op) + ": frame " + std::to_string(b) + ": ";
        TU_CHECK_ARG(d.y, at + "y is NULL");
        TU_CHECK_ARG(d.uv, at + "uv is NULL");
        TU_CHECK_ARG(d.y_pitch >= row, at + "y_pitch " + std::to_string(d.y_pitch) + " is smaller than W samples (" + std::to_string(row) + " bytes)");
        TU_CHECK_ARG(d.uv_pitch >= row, at + "uv_pitch " + std::to_string(d.uv_pitch) + " is smaller than W samples (" + std::to_string(row) + " bytes)");
        TU_CHECK_ARG(reinterpret_cast<uintptr_t>(d.y) % al == 0, at + "y must be " + al_msg);
        TU_CHECK_ARG(reinterpret_cast<uintptr_t>(d.uv) % al == 0, at + "uv must be " + al_msg);
        TU_CHECK_ARG(d.y_pitch % (long long)al == 0, at + "y_pitch must be " + al_msg);
        TU_CHECK_ARG(d.uv_pitch % (long long)al == 0, at + "uv_pitch must be " + al_msg);
    }
    return TU_OK;
}

// one launch per kPlanesPerLaunch frames; the RGB side is the dense batch, offset to the first frame of the launch
template <typename TS, typename TR, bool ToRgb>
static int launch_planes(const TuFramePlanes *frames, int code, TR *rgb, int B, int H, int W, cudaStream_t st, const char *what) {
    typedef Planes420<typename std::conditional<ToRgb, const TS, TS>::type> A;
    const int n = (H / 2) * (W / 2);
    const long frame = 3L * H * W;
    for (int b0 = 0; b0 < B; b0 += kPlanesPerLaunch) {
        const int nb = std::min(kPlanesPerLaunch, B - b0);
        typename A::Param p = {};
        for (int b = 0; b < nb; ++b) p.f[b] = frames[b0 + b];
        const dim3 grid((unsigned)ceil_div(n, 256), nb);
        if constexpr (ToRgb)
            launch_pdl(yuv420_to_rgb_kernel<TS, TR, A>, grid, dim3(256), 0, st, p, rgb + b0 * frame, H, W, yuv_coef(code));
        else
            launch_pdl(rgb_to_yuv420_kernel<TR, TS, A>, grid, dim3(256), 0, st, (const TR *)rgb + b0 * frame, p, H, W,
                       yuv_coef(code));
        TU_CHECK_LAUNCH(what);
    }
    return TU_OK;
}

extern "C" int tu_yuv420_planes_to_rgb(const TuFramePlanes *frames, int code, void *rgb, int B, int H, int W, void *stream) {
    if (int rc = check_yuv420_planes(frames, code, B, H, W, "yuv420_planes_to_rgb")) return rc;
    const bool p010 = dtype_is_p010(code);
    TU_CHECK_ARG(rgb && (reinterpret_cast<uintptr_t>(rgb) & (p010 ? 7 : 3)) == 0,
                 std::string(p010 ? "yuv420_planes_to_rgb: the fp32 RGB buffer must be non-NULL and 8-byte aligned"
                                  : "yuv420_planes_to_rgb: the fp16 RGB buffer must be non-NULL and 4-byte aligned"));
    cudaStream_t st = (cudaStream_t)stream;
    return p010 ? launch_planes<uint16_t, float, true>(frames, code, (float *)rgb, B, H, W, st, "p010_to_rgb")
                : launch_planes<uint8_t, f16, true>(frames, code, (f16 *)rgb, B, H, W, st, "nv12_to_rgb");
}

extern "C" int tu_rgb_to_yuv420_planes(const void *rgb, const TuFramePlanes *frames, int code, int B, int H, int W, void *stream) {
    if (int rc = check_yuv420_planes(frames, code, B, H, W, "rgb_to_yuv420_planes")) return rc;
    const bool p010 = dtype_is_p010(code);
    TU_CHECK_ARG(rgb && (reinterpret_cast<uintptr_t>(rgb) & (p010 ? 7 : 3)) == 0,
                 std::string(p010 ? "rgb_to_yuv420_planes: the fp32 RGB buffer must be non-NULL and 8-byte aligned"
                                  : "rgb_to_yuv420_planes: the fp16 RGB buffer must be non-NULL and 4-byte aligned"));
    cudaStream_t st = (cudaStream_t)stream;
    return p010 ? launch_planes<uint16_t, float, false>(frames, code, (float *)rgb, B, H, W, st, "rgb_to_p010")
                : launch_planes<uint8_t, f16, false>(frames, code, (f16 *)rgb, B, H, W, st, "rgb_to_nv12");
}
