// FastTransformer's image tail in one kernel: the last sub-pixel stage of `final_upscale` (Conv2d 3 -> 3 r^2 + PixelShuffle(r),
// FastTransformer/utils.py:43-98 with n_feats = 3; model.py:211,316), `final_upscale_conv` (Conv2d 3 -> 3, model.py:212,317),
// `out = upscaled_input + residual_up` (model.py:320) and the clamp (model.py:327).
//
// Unfused, the three steps move the high-resolution 3-channel image through HBM four times and ran at 4 % of the copy
// bandwidth (one thread per output pixel, every tap a global load).  Here a CTA owns a 36 x 30r tile of the OUTPUT image:
//   1. the low-resolution residual under the tile (+ halo) is staged in shared memory (zero outside the image = the first
//      conv's padding);
//   2. the sub-pixel conv is evaluated into a shared-memory tile of the intermediate high-resolution image, 38 rows x 32r
//      columns x 3 channels (zero outside the image = the second conv's padding).  A warp owns one intermediate row (one
//      sub-pixel row phase i, so its filter rows are warp-uniform and are read as broadcast 128-bit loads), a lane one
//      low-resolution pixel: 27 inputs in registers, 3r outputs of 27 FMAs each;
//   3. a thread slides a 3x3x3 register window down a column of the intermediate tile (9 shared loads per pixel) and
//      applies the 3 -> 3 filter, whose 84 coefficients ride in the kernel parameters (constant-bank operands of the FMAs),
//      adds the other branch and writes the clamped image in its final dtype.
// Arithmetic is fp32 throughout (this kernel also serves the 1e-4 fp32 path), on packed pairs (fma.rn.f32x2 = FFMA2: two IEEE FMAs per issue
// slot) in the sub-pixel convolution: even and odd taps accumulate in the two halves of a pair, added at the end.  The 3 -> 3 convolution
// stays scalar: its 81 coefficients are constant-bank operands of FFMA, while FFMA2 takes its pair from (uniform) registers -- 45 pairs
// exceed the uniform register file and spill (measured: 800 bytes of spills at 64 registers).
#include "tc/ptx.cuh"
#include "tu_common.cuh"

namespace tu {

namespace {

// output rows per tile (a multiple of r: tiles start on a low-res row).  36 rows, but 18 at r = 6, where the 36-row intermediate
// tile (87 KB) allowed only two CTAs per SM (ncu: 20 % warps active, issue slots 49 % busy)
template <int R> constexpr int tile_rows() { return R == 6 ? 18 : 36; }
constexpr int TLX = 30;         // low-res columns per tile -> 30 r output columns; + 2 halo columns = 32 lanes
constexpr int NT = 256;

// [(ky*3+kx)*3+ci][co], bias.  THREE identical copies of the filter: the row loop of step 3 is unrolled three times (rotating window rows) and a
// coefficient that is read by all three copies would be hoisted into a register by the compiler (81 registers: spills); a copy per unrolled
// body keeps every coefficient a constant-bank operand of exactly one FFMA.
struct FinFilter { float w[3][81]; float b[3]; };

// PX4: 4-byte uint8 pixels (layout 3 / 5), each written once with its alpha from the plane `alpha` (NULL: 255); the other
// instantiations never read `alpha`
template <int R, typename TO, bool PX4 = false>
__global__ void __launch_bounds__(NT, 4)
subpixel_tail_kernel(const float *__restrict__ in, const float *__restrict__ wps, const float *__restrict__ bps,
                     const float *__restrict__ addend, TO *__restrict__ out, int H, int W, int clamp, int layout,
                     const FinFilter fin, const uint8_t *__restrict__ alpha) {
    constexpr int NCO = 3 * R * R;
    constexpr int TH = tile_rows<R>(), IR = TH + 2;     // IR = intermediate rows held
    constexpr int NLR = TH / R + 4;            // low-res rows staged: ly0 - 2 .. ly0 + TH/R + 1
    constexpr int LRW = TLX + 4;               // low-res columns staged: lx0 - 2 .. lx0 + 31
    constexpr int IW = 32 * R;                 // intermediate columns held: (lx0 - 1) r .. (lx0 + 31) r - 1
    extern __shared__ float sm[];
    float *w_s = sm;                           // [NCO][28] (27 taps, padded for 128-bit reads)
    float *b_s = w_s + NCO * 28;               // [NCO] (+ pad to 4)
    float *lr_s = b_s + ((NCO + 3) & ~3);      // [3][NLR][LRW]
    float *im_s = lr_s + 3 * NLR * LRW;        // [3][IR][IW]
    pdl_trigger();
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int b = blockIdx.z;
    const int oy0 = blockIdx.y * TH, lx0 = blockIdx.x * TLX;
    const int ly0 = oy0 / R;
    const int oH = H * R, oW = W * R;
    pdl_wait();

    // Staging: all of a thread's global loads are issued before the first shared store, so that their latencies overlap (ncu
    // on the first version: half of the stall samples of the kernel sat on these loads, one exposed round trip per element)
    {
        constexpr int NLRE = 3 * NLR * LRW, KLR = (NLRE + NT - 1) / NT;
        constexpr int NWE = NCO * 27, KW = (NWE + NT - 1) / NT;
        float tl[KLR], tw[KW];
#pragma unroll
        for (int k = 0; k < KLR; ++k) {
            const int i = tid + k * NT;
            const int c = i / (NLR * LRW), rem = i - c * (NLR * LRW);
            const int ry = rem / LRW, rx = rem - ry * LRW;
            const int y = ly0 - 2 + ry, x = lx0 - 2 + rx;
            tl[k] = (i < NLRE && y >= 0 && y < H && x >= 0 && x < W) ? __ldg(in + (((long)b * 3 + c) * H + y) * W + x) : 0.f;
        }
#pragma unroll
        for (int k = 0; k < KW; ++k) {
            const int i = tid + k * NT;
            tw[k] = i < NWE ? __ldg(wps + i) : 0.f;
        }
        const float bv = tid < NCO ? __ldg(bps + tid) : 0.f;
#pragma unroll
        for (int k = 0; k < KLR; ++k) {
            const int i = tid + k * NT;
            if (i < NLRE) lr_s[i] = tl[k];
        }
#pragma unroll
        for (int k = 0; k < KW; ++k) {
            const int i = tid + k * NT;
            if (i < NWE) {
                const int t = i / NCO, o = i - t * NCO;
                w_s[o * 28 + t] = tw[k];
            }
        }
        if (tid < NCO) {
            b_s[tid] = bv;
            w_s[tid * 28 + 27] = 0.f;
        }
    }
    __syncthreads();

    // ---- step 2: intermediate rows hy = oy0 - 1 + hr; lane = low-res column lx0 - 1 + lane
    for (int hr = warp; hr < IR; hr += NT / 32) {
        const int hy = oy0 - 1 + hr;
        float *dst = im_s + hr * IW + lane * R;
        const int lx = lx0 - 1 + lane;
        if (hy < 0 || hy >= oH || lx < 0 || lx >= W) {          // outside the image: the 3 -> 3 conv's zero padding
#pragma unroll
            for (int c = 0; c < 3; ++c)
#pragma unroll
                for (int j = 0; j < R; ++j) dst[c * IR * IW + j] = 0.f;
            continue;
        }
        const int ly = hy / R, i = hy - ly * R;
        const float *src = lr_s + (ly - ly0 + 1) * LRW + lane;       // tap (ky, kx) -> row ly - 1 + ky, column lx - 1 + kx
        float v[28];
#pragma unroll
        for (int ky = 0; ky < 3; ++ky)
#pragma unroll
            for (int kx = 0; kx < 3; ++kx)
#pragma unroll
                for (int c = 0; c < 3; ++c) v[(ky * 3 + kx) * 3 + c] = src[c * NLR * LRW + ky * LRW + kx];
        v[27] = 0.f;
        ptx::f32x2 vp[14];                                   // (tap 2k, tap 2k + 1)
#pragma unroll
        for (int k = 0; k < 14; ++k) vp[k] = ptx::pk2(v[2 * k], v[2 * k + 1]);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
#pragma unroll
            for (int j = 0; j < R; ++j) {
                const int o = c * R * R + i * R + j;
                const ulonglong2 *wr = reinterpret_cast<const ulonglong2 *>(w_s + o * 28);      // warp-uniform: broadcast 128-bit loads
                ptx::f32x2 acc = ptx::pk2(b_s[o], 0.f);       // even taps (+ bias) | odd taps
#pragma unroll
                for (int q = 0; q < 7; ++q) {
                    const ulonglong2 ww = wr[q];
                    acc = ptx::fma2(vp[2 * q], ww.x, acc);
                    acc = ptx::fma2(vp[2 * q + 1], ww.y, acc);
                }
                float lo, hi;
                ptx::up2(acc, lo, hi);
                dst[c * IR * IW + j] = lo + hi;
            }
        }
    }
    __syncthreads();

    // ---- step 3: 3 -> 3 conv + addend (+ clamp); a thread walks down one output column of the tile
    constexpr int TW = TLX * R;
    constexpr int G = NT / TW >= 1 ? NT / TW : 1;      // row groups
    constexpr int RPG = (TH + G - 1) / G;
    const int cx = tid % TW, g = tid / TW;
    if (g >= G) return;
    const int ox = lx0 * R + cx;
    if (ox >= oW) return;
    const int r0 = g * RPG, r1 = min(min(r0 + RPG, TH), oH - oy0);
    if (r0 >= r1) return;
    // output row oy0 + ry reads intermediate rows ry .. ry + 2, columns cx + R - 1 .. cx + R + 1
    const float *col = im_s + cx + R - 1;
    // a row of the 3 x 3 x 3 window = nine values e = kx * 3 + ci; the three rows live in three register sets whose roles rotate
    // (the row loop is unrolled three times, so no window moves: they were 18 of the ~130 instructions per pixel of this step)
#define TU_TAIL_LOAD_ROW(row, ir)                                                                           \
    do {                                                                                                    \
        _Pragma("unroll") for (int kx = 0; kx < 3; ++kx)                                                    \
            _Pragma("unroll") for (int c = 0; c < 3; ++c) row[kx * 3 + c] = col[c * IR * IW + (ir) * IW + kx]; \
    } while (0)
    const long plane = (long)oH * oW;
    long o = (long)b * 3 * plane + (long)(oy0 + r0) * oW + ox;
    float ad[3];                                        // the other branch, fetched one row ahead of its use
#pragma unroll
    for (int co = 0; co < 3; ++co) ad[co] = addend[o + co * plane];
    // one output pixel of the 3 -> 3 convolution from the three window rows (the filter's coefficients are constant-bank operands of the
    // FMAs), + the other branch (+ clamp), stored in its final dtype.  Macros, not lambdas: with lambdas the three unrolled copies kept
    // the window rows in local memory (ptxas: 400 bytes of stack, 700 bytes of spills).
#define TU_TAIL_ROW(top, mid, bot, ry, cp)                                                                     \
    do {                                                                                                    \
        float a[3] = {0.f, 0.f, 0.f}, adn[3];                                                               \
        const long on = (ry) + 1 < r1 ? o + oW : o;                                                         \
        _Pragma("unroll") for (int co = 0; co < 3; ++co) adn[co] = addend[on + co * plane];                 \
        _Pragma("unroll") for (int e = 0; e < 9; ++e)                                                       \
            _Pragma("unroll") for (int co = 0; co < 3; ++co) a[co] = fmaf(top[e], fin.w[cp][e * 3 + co], a[co]);      \
        _Pragma("unroll") for (int e = 0; e < 9; ++e)                                                       \
            _Pragma("unroll") for (int co = 0; co < 3; ++co) a[co] = fmaf(mid[e], fin.w[cp][(9 + e) * 3 + co], a[co]); \
        _Pragma("unroll") for (int e = 0; e < 9; ++e)                                                       \
            _Pragma("unroll") for (int co = 0; co < 3; ++co) a[co] = fmaf(bot[e], fin.w[cp][(18 + e) * 3 + co], a[co]); \
        float rgb[3];                                                                                       \
        _Pragma("unroll") for (int co = 0; co < 3; ++co) {                                                  \
            /* reference: out = upscaled_input + (conv + bias)   (FastTransformer/model.py:320) */          \
            float r = ad[co] + (a[co] + fin.b[co]);                                                         \
            if (clamp) r = fminf(fmaxf(r, 0.f), 1.f);                                                       \
            rgb[co] = r;                                                                                    \
            ad[co] = adn[co];                                                                               \
        }                                                                                                   \
        if constexpr (PX4) {                                                                                \
            store_px4(out, (long)b * plane + (long)(oy0 + (ry)) * oW + ox, layout, rgb[0], rgb[1], rgb[2], alpha); \
        } else if (layout == 0) {                                                                           \
            _Pragma("unroll") for (int co = 0; co < 3; ++co) out[o + co * plane] = from_f<TO>(rgb[co]);     \
        } else {                                                                                            \
            store_rgb<TO>(out, b, plane, (long)(oy0 + (ry)) * oW + ox, layout, rgb[0], rgb[1], rgb[2]);     \
        }                                                                                                   \
        o += oW;                                                                                            \
    } while (0)
    float ra[9], rb[9], rc[9];
    TU_TAIL_LOAD_ROW(ra, r0);
    TU_TAIL_LOAD_ROW(rb, r0 + 1);
#pragma unroll 1
    for (int ry = r0; ry < r1; ry += 3) {
        TU_TAIL_LOAD_ROW(rc, ry + 2);
        TU_TAIL_ROW(ra, rb, rc, ry, 0);
        if (ry + 1 < r1) {
            TU_TAIL_LOAD_ROW(ra, ry + 3);
            TU_TAIL_ROW(rb, rc, ra, ry + 1, 1);
        }
        if (ry + 2 < r1) {
            TU_TAIL_LOAD_ROW(rb, ry + 4);
            TU_TAIL_ROW(rc, ra, rb, ry + 2, 2);
        }
    }
}
#undef TU_TAIL_LOAD_ROW
#undef TU_TAIL_ROW

template <int R>
constexpr size_t tail_smem() {
    constexpr int TH = tile_rows<R>(), IR = TH + 2;
    return sizeof(float) * (3 * R * R * 28 + ((3 * R * R + 3) & ~3) + 3 * (TH / R + 4) * (TLX + 4) + 3 * IR * 32 * R);
}

template <int R, typename TO, bool PX4>
int launch_tail(const float *in, const float *wps, const float *bps, const float *addend, TO *out, int B, int H, int W, int clamp, int layout,
                const FinFilter &fin, const uint8_t *alpha, cudaStream_t st) {
    static PerDeviceFlag attr;
    constexpr size_t smem = tail_smem<R>();
    if (!attr.is_set() && smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(subpixel_tail_kernel<R, TO, PX4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return cuda_fail(e, "subpixel_tail smem attribute");
        attr.set();
    }
    dim3 grid(ceil_div(W, TLX), ceil_div(H * R, tile_rows<R>()), B);
    launch_pdl(subpixel_tail_kernel<R, TO, PX4>, grid, dim3(NT), smem, st, in, wps, bps, addend, out, H, W, clamp, layout, fin, alpha);
    TU_CHECK_LAUNCH("subpixel_tail");
    return TU_OK;
}

template <typename TO, bool PX4 = false>
int tail_by_r(int r, const float *in, const float *wps, const float *bps, const float *addend, TO *out, int B, int H, int W, int clamp, int layout,
              const FinFilter &fin, cudaStream_t st, const uint8_t *alpha = nullptr) {
    switch (r) {
        case 2: return launch_tail<2, TO, PX4>(in, wps, bps, addend, out, B, H, W, clamp, layout, fin, alpha, st);
        case 3: return launch_tail<3, TO, PX4>(in, wps, bps, addend, out, B, H, W, clamp, layout, fin, alpha, st);
        case 6: return launch_tail<6, TO, PX4>(in, wps, bps, addend, out, B, H, W, clamp, layout, fin, alpha, st);
    }
    set_error("tu: subpixel_conv_add: r must be 2, 3 or 6");
    return TU_ERR_ARG;
}

}  // namespace

}  // namespace tu

using namespace tu;

int tu::subpixel_conv_add_alpha(const float *in, const float *w_ps, const float *b_ps, int r, const float *host_fin_wb, const float *addend,
                                void *out, int out_dtype, int B, int H, int W, int clamp, const uint8_t *alpha, cudaStream_t st) {
    TU_CHECK_ARG(in && w_ps && b_ps && host_fin_wb && addend && out && B > 0 && H > 0 && W > 0, "subpixel_conv_add: bad argument");
    TU_CHECK_ARG((long)B * 3 * H * r * W * r < (1L << 31), "subpixel_conv_add: image too large for 32-bit pixel indexing");
    const int layout = dtype_layout(out_dtype);
    out_dtype = dtype_base(out_dtype);
    TU_CHECK_ARG(layout == 0 || (out_dtype == TU_U8 && layout_is_interleaved(layout)), "subpixel_conv_add: interleaved layouts are for uint8 frames");
    TU_CHECK_ARG(out_dtype == TU_F32 || out_dtype == TU_BF16 || out_dtype == TU_U8 || out_dtype == TU_F16, "subpixel_conv_add: bad dtype");
    const bool px4 = layout_is_px4(layout);
    TU_CHECK_ARG(!px4 || (reinterpret_cast<uintptr_t>(out) & 3) == 0, "subpixel_conv_add: a 4-byte (RGBA / BGRA) output must be 4-byte aligned");
    FinFilter fin;
    for (int cp = 0; cp < 3; ++cp)
        for (int i = 0; i < 81; ++i) fin.w[cp][i] = host_fin_wb[i];
    for (int i = 0; i < 3; ++i) fin.b[i] = host_fin_wb[81 + i];
    if (px4) return tail_by_r<uint8_t, true>(r, in, w_ps, b_ps, addend, (uint8_t *)out, B, H, W, clamp, layout, fin, st, alpha);
    if (out_dtype == TU_F32) return tail_by_r<float>(r, in, w_ps, b_ps, addend, (float *)out, B, H, W, clamp, layout, fin, st);
    if (out_dtype == TU_BF16) return tail_by_r<bf16>(r, in, w_ps, b_ps, addend, (bf16 *)out, B, H, W, clamp, layout, fin, st);
    if (out_dtype == TU_U8) return tail_by_r<uint8_t>(r, in, w_ps, b_ps, addend, (uint8_t *)out, B, H, W, clamp, layout, fin, st);
    if (out_dtype == TU_F16) return tail_by_r<f16>(r, in, w_ps, b_ps, addend, (f16 *)out, B, H, W, clamp, layout, fin, st);
    TU_CHECK_ARG(false, "subpixel_conv_add: bad dtype");
}

extern "C" int tu_subpixel_conv_add(const float *in, const float *w_ps, const float *b_ps, int r, const float *host_fin_wb,
                                    const float *addend, void *out, int out_dtype, int B, int H, int W, int clamp, void *stream) {
    return subpixel_conv_add_alpha(in, w_ps, b_ps, r, host_fin_wb, addend, out, out_dtype, B, H, W, clamp, nullptr, (cudaStream_t)stream);
}
