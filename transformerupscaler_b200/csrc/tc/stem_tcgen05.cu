// conv1 (3 -> 64, 3x3, pad 1, + ReLU) on the tensor cores: NCHW image in, NHWC bf16 features out.
// Reference: conv1 + relu (WindowTransformer/model.py:200,244; FastTransformer/model.py:202,251;
// ResidualTransformer/model.py:83,128).
//
// The op is HBM-bound on its 128-byte-per-pixel output (K = 27 only), so the point of using tcgen05 here is to
// take the 1728 FMAs per pixel off the CUDA cores: four "builder" warps write the im2col rows (27 taps padded to
// 32 bf16 = four 16-byte chunks per pixel) straight into a 128-byte-swizzled K-major operand tile in shared
// memory, one thread issues two 128x64x16 UMMAs per 128-pixel row segment, and four epilogue warps drain TMEM
// (+bias, ReLU, bf16) into full 128-byte pixel stores.  Tiles are row segments of 128 pixels; the CTA is
// persistent and double-buffers both the operand tile and the accumulator.
#include <cuda.h>
#include <string.h>

#include "ptx.cuh"
#include "tc_api.cuh"

namespace tu {

namespace {

constexpr int NUM_THREADS = 288;      // warps 0-3 epilogue, 4-7 builders, 8 MMA / TMEM / weight TMA
constexpr int ROWS = 4;               // image rows per tile (halo rows are loaded once for all four)
constexpr int A_BYTES = 128 * 128;    // one operand tile: 128 pixels x 128-byte rows
constexpr int W_BYTES = 64 * 128;     // 64 output channels x (64 k, 27 real)
constexpr int STG_BYTES = 4 * 4096;       // epilogue staging: 4 warps x (32 pixels x 128 B), source of the TMA stores
constexpr int NRAW_MAX = 3;               // raw input tiles in flight (TMA variant)
constexpr int RAW_BUDGET = 20 * 1024;     // bytes reserved for them
constexpr int SMEM_BYTES = ROWS * A_BYTES + W_BYTES + STG_BYTES + RAW_BUDGET + 256 + 256 + 1024;
// raw input tile of the TMA variant: (3 channels, ROWS + 2 rows, RW columns) of the image element type; the box starts
// PADL = 16 / sizeof(element) pixels left of the tile (the innermost TMA start coordinate must be 16-byte aligned), so image
// pixel x0 + d sits in column PADL + d
template <typename TI> struct RawGeom {
    static constexpr int PADL = 16 / (int)sizeof(TI);
    static constexpr int RW = 128 + 2 * PADL;
    static constexpr int BYTES = ((3 * (ROWS + 2) * RW * (int)sizeof(TI)) + 127) & ~127;
    static constexpr int NRAW = (NRAW_MAX * BYTES <= RAW_BUDGET) ? NRAW_MAX : 2;
    static_assert(NRAW * BYTES <= RAW_BUDGET, "raw tiles exceed their shared-memory budget");
};

struct StemParams {
    int B, H, W, tiles_x, tiles_y, total_tiles;
    const float *bias;
    bf16 *out;
};

struct Barriers {
    uint64_t a_full, a_empty, acc_full[ROWS], acc_empty[ROWS], w_full, raw_full[NRAW_MAX];
    uint32_t tmem_base;
};

// image element -> float for the bf16 operand (uint8 frames: x * (1/255); the product is rounded to bf16 right after)
__device__ __forceinline__ float ldx(float v) { return v; }
__device__ __forceinline__ float ldx(bf16 v) { return __bfloat162float(v); }
__device__ __forceinline__ float ldx(f16 v) { return __half2float(v); }
__device__ __forceinline__ float ldx(uint8_t v) { return u8_to_float(v) * 0.00392156862745098f; }

// (lo, hi) -> bf16x2 with ReLU in the same instruction
__device__ __forceinline__ uint32_t pack2_relu(float lo, float hi) {
    uint32_t d;
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    return d;
}

__device__ __forceinline__ uint32_t pack2(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t *>(&h);
}

// RAWTMA: the image footprint of a tile arrives by TMA (zero-filled outside the image = the convolution's padding), NRAW tiles
// ahead, so the builders never wait on global-memory latency; otherwise (row pitch not a multiple of 16 bytes) they load
// their pixels through registers one tile ahead.
template <typename TI, bool RAWTMA>
__global__ void __launch_bounds__(NUM_THREADS, 2)
stem_tc_kernel(const __grid_constant__ CUtensorMap tmap_w, const __grid_constant__ CUtensorMap tmap_out,
               const __grid_constant__ CUtensorMap tmap_x, const TI *__restrict__ x, const StemParams p) {
    pdl_trigger();
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem0 = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t *smem_al = smem_raw + (smem0 - ptx::smem_u32(smem_raw));
    const uint32_t a_sm = smem0, w_sm = smem0 + ROWS * A_BYTES;
    const uint32_t stg_sm = w_sm + W_BYTES;        // 1024-byte aligned
    uint8_t *raw_al = smem_al + ROWS * A_BYTES + W_BYTES + STG_BYTES;      // 1024-byte aligned
    const uint32_t raw_sm = stg_sm + STG_BYTES;
    Barriers *bars = reinterpret_cast<Barriers *>(smem_al + ROWS * A_BYTES + W_BYTES + STG_BYTES + RAW_BUDGET + 256);
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // provably warp-uniform

    if (threadIdx.x == 0) {
        ptx::mbar_init(ptx::smem_u32(&bars->a_full), 128);
        ptx::mbar_init(ptx::smem_u32(&bars->a_empty), 1);
        for (int i = 0; i < ROWS; ++i) {
            ptx::mbar_init(ptx::smem_u32(&bars->acc_full[i]), 1);
            ptx::mbar_init(ptx::smem_u32(&bars->acc_empty[i]), 4);
        }
        ptx::mbar_init(ptx::smem_u32(&bars->w_full), 1);
        for (int i = 0; i < NRAW_MAX; ++i) ptx::mbar_init(ptx::smem_u32(&bars->raw_full[i]), 1);
        ptx::fence_barrier_init();
    }
    if (warp == 8) {
        ptx::tmem_alloc(ptx::smem_u32(&bars->tmem_base), 256);
        ptx::tmem_relinquish();
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = bars->tmem_base;
    pdl_wait();

    if (warp == 8) {
        // ================================ weights + MMA issuer (whole warp converged, elected lane issues) ================================
        const uint32_t leader = ptx::elect_one();
        if (leader) {
            ptx::mbar_expect_tx(ptx::smem_u32(&bars->w_full), W_BYTES);
            ptx::tma_load_2d(w_sm, &tmap_w, ptx::smem_u32(&bars->w_full), 0, 0);
        }
        __syncwarp();
        ptx::mbar_wait(ptx::smem_u32(&bars->w_full), 0);
        // fold the bias into the contraction: operand columns k = 27, 28 are constant 1, filter columns 27, 28 hold the
        // bias split into bf16 hi + lo parts (fp32 accuracy), so the epilogue is a single convert-with-ReLU per pair
#pragma unroll
        for (int co = lane; co < 64; co += 32) {
            const float bv = p.bias[co];
            const bf16 hi = __float2bfloat16_rn(bv), lo = __float2bfloat16_rn(bv - __bfloat162float(hi));
            bf16 *row = reinterpret_cast<bf16 *>(smem_al + ROWS * A_BYTES + co * 128 + ((3 ^ (co & 7)) << 4));
            row[3] = hi;      // k = 27
            row[4] = lo;      // k = 28
        }
        ptx::fence_proxy_async();
        __syncwarp();
        const uint32_t idesc = ptx::make_idesc_bf16(128, 64);
        const uint32_t a_lo = ptx::sdesc_lo(a_sm), w_lo = ptx::sdesc_lo(w_sm);
        uint32_t ph = 0;
        for (int t = blockIdx.x; t < p.total_tiles; t += gridDim.x, ph ^= 1) {
            ptx::mbar_wait(ptx::smem_u32(&bars->a_full), ph);
            ptx::tc_fence_after();
#pragma unroll
            for (int r = 0; r < ROWS; ++r) {
                ptx::mbar_wait(ptx::smem_u32(&bars->acc_empty[r]), ph ^ 1);
                ptx::tc_fence_after();
                // k = 0..31 (27 taps + 5 zeros); chunks 4-7 of a row are never read
                ptx::umma_bf16_lo<0>(tmem_base + r * 64, a_lo + ((r * A_BYTES) >> 4), w_lo, idesc, leader);
                ptx::umma_bf16_lo<1>(tmem_base + r * 64, a_lo + ((r * A_BYTES + 32) >> 4), w_lo + 2, idesc, leader);
                ptx::umma_commit_pred(ptx::smem_u32(&bars->acc_full[r]), leader);
            }
            ptx::umma_commit_pred(ptx::smem_u32(&bars->a_empty), leader);
        }
    } else if (warp >= 4) {
        // ================================ builders: im2col rows -> swizzled smem ================================
        const int i = (warp - 4) * 32 + lane;            // pixel of the segment = operand row
        float v[3][ROWS + 2][3];                         // [channel][input row][kx]
        auto load_tile = [&](int t) {
            const int tx = t % p.tiles_x;
            int rem = t / p.tiles_x;
            const int ty = rem % p.tiles_y, b = rem / p.tiles_y;
            const int px = tx * 128 + i, y0 = ty * ROWS;
#pragma unroll
            for (int c = 0; c < 3; ++c)
#pragma unroll
                for (int r = 0; r < ROWS + 2; ++r) {
                    const int iy = y0 + r - 1;
                    const bool rowok = iy >= 0 && iy < p.H;
                    const TI *row = x + (((long)b * 3 + c) * p.H + (rowok ? iy : 0)) * p.W;
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx) {
                        const int ix = px + kx - 1;
                        v[c][r][kx] = (rowok && ix >= 0 && ix < p.W) ? ldx(row[ix]) : 0.f;
                    }
                }
        };
        // one L2 prefetch per thread and tile, two tiles ahead: thread i touches row segment i % 18 = (channel, input row) at
        // pixel 18 * (i / 18), so every 128-byte line of the tile's footprint is requested; the register loads of the next
        // iteration then pay L2 latency instead of DRAM latency
        auto prefetch_tile = [&](int t) {
            const int tx = t % p.tiles_x;
            int rem = t / p.tiles_x;
            const int ty = rem % p.tiles_y, b = rem / p.tiles_y;
            const int seg = i % 18, c = seg / 6, r = seg % 6;
            const int iy = min(max(ty * ROWS + r - 1, 0), p.H - 1), ix = min(tx * 128 + (i / 18) * 18, p.W - 1);
            const TI *a = x + (((long)b * 3 + c) * p.H + iy) * p.W + ix;
            asm volatile("prefetch.global.L2 [%0];" ::"l"(a));
        };
        // im2col rows of the four image rows of a tile -> swizzled operand tiles (k = (ky*3+kx)*3 + c; k = 27, 28 = 1 for the bias)
        auto build = [&]() {
#pragma unroll
            for (int r = 0; r < ROWS; ++r) {
                uint8_t *rowp = smem_al + r * A_BYTES + i * 128;
                float k[32];
#pragma unroll
                for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx)
#pragma unroll
                        for (int c = 0; c < 3; ++c) k[(ky * 3 + kx) * 3 + c] = v[c][r + ky][kx];
#pragma unroll
                for (int z = 27; z < 32; ++z) k[z] = z < 29 ? 1.f : 0.f;       // k = 27, 28 multiply the bias columns
#pragma unroll
                for (int ch = 0; ch < 4; ++ch) {
                    uint4 u;
                    u.x = pack2(k[ch * 8 + 0], k[ch * 8 + 1]);
                    u.y = pack2(k[ch * 8 + 2], k[ch * 8 + 3]);
                    u.z = pack2(k[ch * 8 + 4], k[ch * 8 + 5]);
                    u.w = pack2(k[ch * 8 + 6], k[ch * 8 + 7]);
                    *reinterpret_cast<uint4 *>(rowp + ((ch ^ (i & 7)) << 4)) = u;      // 128-byte swizzle: chunk ^= row % 8
                }
            }
            ptx::fence_proxy_async();        // generic-proxy writes -> visible to the tensor core (async proxy)
            ptx::mbar_arrive(ptx::smem_u32(&bars->a_full));
        };
        uint32_t ph = 0;
        if (RAWTMA) {
            using G = RawGeom<TI>;
            auto issue = [&](int t, int stage) {          // one thread: TMA of tile t's footprint into raw stage `stage`
                const int tx = t % p.tiles_x;
                int rem = t / p.tiles_x;
                const int ty = rem % p.tiles_y, b = rem / p.tiles_y;
                const uint32_t fb = ptx::smem_u32(&bars->raw_full[stage]);
                ptx::mbar_expect_tx(fb, 3 * (ROWS + 2) * G::RW * (int)sizeof(TI));
                ptx::tma_load_4d(raw_sm + stage * G::BYTES, &tmap_x, fb, tx * 128 - G::PADL, ty * ROWS - 1, 0, b);
            };
            if (i == 0)
                for (int s = 0; s < G::NRAW; ++s)
                    if (blockIdx.x + s * gridDim.x < p.total_tiles) issue(blockIdx.x + s * gridDim.x, s);
            int stage = 0;
            uint32_t rph = 0;
            for (int t = blockIdx.x; t < p.total_tiles; t += gridDim.x, ph ^= 1) {
                ptx::mbar_wait(ptx::smem_u32(&bars->raw_full[stage]), rph);
                const TI *raw = reinterpret_cast<const TI *>(raw_al + stage * G::BYTES) + (G::PADL - 1 + i);
#pragma unroll
                for (int c = 0; c < 3; ++c)
#pragma unroll
                    for (int r = 0; r < ROWS + 2; ++r)
#pragma unroll
                        for (int kx = 0; kx < 3; ++kx) v[c][r][kx] = ldx(raw[(c * (ROWS + 2) + r) * G::RW + kx]);
                asm volatile("bar.sync 2, 128;" ::: "memory");          // all builders have read the stage: refill it
                if (i == 0 && t + G::NRAW * gridDim.x < p.total_tiles) issue(t + G::NRAW * gridDim.x, stage);
                if (++stage == G::NRAW) { stage = 0; rph ^= 1; }
                ptx::mbar_wait(ptx::smem_u32(&bars->a_empty), ph ^ 1);
                build();
            }
        } else {
            if (blockIdx.x < p.total_tiles) load_tile(blockIdx.x);
            if (blockIdx.x + gridDim.x < p.total_tiles) prefetch_tile(blockIdx.x + gridDim.x);
            for (int t = blockIdx.x; t < p.total_tiles; t += gridDim.x, ph ^= 1) {
                ptx::mbar_wait(ptx::smem_u32(&bars->a_empty), ph ^ 1);
                build();
                if (t + gridDim.x < p.total_tiles) load_tile(t + gridDim.x);   // next tile's pixels fly while this one is consumed
                if (t + 2 * gridDim.x < p.total_tiles) prefetch_tile(t + 2 * gridDim.x);
            }
        }
    } else {
        // ================================ epilogue ================================
        // TMEM -> (+bias, ReLU, bf16) -> the pixel's 128 bytes into a swizzled staging buffer -> one TMA store per 32-pixel
        // row segment and warp (a thread storing its own pixel would touch 32 different cache lines per instruction).
        const int q = warp;
        uint32_t ph = 0;
        uint8_t *stg_w = smem_al + ROWS * A_BYTES + W_BYTES + q * 4096;
        const uint32_t stg_w_sm = stg_sm + q * 4096;
        for (int t = blockIdx.x; t < p.total_tiles; t += gridDim.x, ph ^= 1) {
            const int tx = t % p.tiles_x;
            int rem = t / p.tiles_x;
            const int ty = rem % p.tiles_y, b = rem / p.tiles_y;
            const int px0 = tx * 128 + q * 32;
#pragma unroll 1
            for (int r = 0; r < ROWS; ++r) {
                const int y = ty * ROWS + r;
                ptx::mbar_wait(ptx::smem_u32(&bars->acc_full[r]), ph);
                ptx::tc_fence_after();
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + r * 64;
                uint32_t v0[32], v1[32];
                ptx::tmem_ld_x32(taddr, v0);
                ptx::tmem_ld_x32(taddr + 32, v1);
                ptx::tmem_ld_wait();
                ptx::tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                    ptx::mbar_arrive(ptx::smem_u32(&bars->acc_empty[r]));   // values are in registers now
                    ptx::bulk_wait_read<0>();                               // the previous row's store has read the staging buffer
                }
                __syncwarp();
                uint8_t *rowp = stg_w + lane * 128;
#pragma unroll
                for (int c = 0; c < 64; c += 8) {
                    const uint32_t *v = c < 32 ? &v0[c] : &v1[c - 32];
                    uint4 u;
                    u.x = pack2_relu(__uint_as_float(v[0]), __uint_as_float(v[1]));
                    u.y = pack2_relu(__uint_as_float(v[2]), __uint_as_float(v[3]));
                    u.z = pack2_relu(__uint_as_float(v[4]), __uint_as_float(v[5]));
                    u.w = pack2_relu(__uint_as_float(v[6]), __uint_as_float(v[7]));
                    *reinterpret_cast<uint4 *>(rowp + (((c >> 3) ^ (lane & 7)) << 4)) = u;      // 128-byte swizzle: chunk ^= row % 8
                }
                ptx::fence_proxy_async();
                __syncwarp();
                if (lane == 0) {
                    if (y < p.H && px0 < p.W) ptx::tma_store_4d(&tmap_out, stg_w_sm, 0, px0, y, b);
                    ptx::bulk_commit();
                }
            }
        }
        if (lane == 0) ptx::bulk_wait<0>();
        __syncwarp();
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 8) ptx::tmem_dealloc(tmem_base, 256);
}

PerDeviceFlag g_attr_set;

}  // namespace

// w64: bf16 (64 co, 64 k) with k = (ky*3+kx)*3 + ci for k < 27 and zeros above
int tc_stem_conv(const void *x, int in_dtype, const bf16 *w64, const float *bias, bf16 *out, int B, int H, int W, cudaStream_t st) {
    TcEncodeFn enc = tc_encode_fn();
    if (!enc || (reinterpret_cast<uintptr_t>(w64) & 127) || (reinterpret_cast<uintptr_t>(out) & 15)) return TU_TC_UNSUPPORTED;
    const int g_sm_count = device_sm_count();
    if (!g_attr_set.is_set()) {
        cudaError_t e = cudaSuccess;
#define TU_STEM_ATTR(TI, R) \
    if (e == cudaSuccess) e = cudaFuncSetAttribute(stem_tc_kernel<TI, R>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES)
        TU_STEM_ATTR(float, false); TU_STEM_ATTR(float, true);
        TU_STEM_ATTR(bf16, false); TU_STEM_ATTR(bf16, true);
        TU_STEM_ATTR(uint8_t, false); TU_STEM_ATTR(uint8_t, true);
        TU_STEM_ATTR(f16, false); TU_STEM_ATTR(f16, true);
#undef TU_STEM_ATTR
        if (e != cudaSuccess) return cuda_fail(e, "stem_tc smem attribute");
        g_attr_set.set();
    }
    CUtensorMap tw;
    cuuint64_t wd[2] = {64, 64}, ws[1] = {128};
    cuuint32_t wb[2] = {64, 64}, we[2] = {1, 1};
    CUresult r = enc(&tw, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void *)w64, wd, ws, wb, we, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("tu: cuTensorMapEncodeTiled(stem weights) failed with code " + std::to_string((int)r));
        return TU_ERR_CUDA;
    }
    CUtensorMap to;
    {
        cuuint64_t od[4] = {64, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B}, os[3] = {128, (cuuint64_t)W * 128, (cuuint64_t)H * W * 128};
        cuuint32_t ob[4] = {64, 32, 1, 1}, oe[4] = {1, 1, 1, 1};
        r = enc(&to, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, (void *)out, od, os, ob, oe, CU_TENSOR_MAP_INTERLEAVE_NONE,
                CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) {
            set_error("tu: cuTensorMapEncodeTiled(stem output) failed with code " + std::to_string((int)r));
            return TU_ERR_CUDA;
        }
    }
    StemParams p;
    p.B = B; p.H = H; p.W = W;
    p.tiles_x = ceil_div(W, 128);
    p.tiles_y = ceil_div(H, ROWS);
    p.total_tiles = p.tiles_x * p.tiles_y * B;
    p.bias = bias; p.out = out;
    const int grid = p.total_tiles < 2 * g_sm_count ? p.total_tiles : 2 * g_sm_count;
    // raw image tiles by TMA when the row pitch allows it: (W, H, 3, B) view, box (RW, ROWS + 2, 3, 1)
    const int eb = (int)dtype_size(in_dtype);
    const int rw = 128 + 2 * (16 / eb);
    CUtensorMap tx;
    memset(&tx, 0, sizeof(tx));
    bool raw_tma = ((size_t)W * eb) % 16 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0;
    if (raw_tma) {
        cuuint64_t xd[4] = {(cuuint64_t)W, (cuuint64_t)H, 3, (cuuint64_t)B};
        cuuint64_t xs[3] = {(cuuint64_t)W * eb, (cuuint64_t)H * W * eb, (cuuint64_t)3 * H * W * eb};
        cuuint32_t xb[4] = {(cuuint32_t)rw, ROWS + 2, 3, 1}, xe[4] = {1, 1, 1, 1};
        raw_tma = enc(&tx, tc_image_map_dtype(in_dtype),
                      4, const_cast<void *>(x), xd, xs, xb, xe, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                      CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
    }
#define TU_STEM_LAUNCH(TI)                                                                                         \
    do {                                                                                                           \
        if (raw_tma)                                                                                               \
            launch_pdl(stem_tc_kernel<TI, true>, dim3(grid), dim3(NUM_THREADS), SMEM_BYTES, st, tw, to, tx, (const TI *)x, p);   \
        else                                                                                                       \
            launch_pdl(stem_tc_kernel<TI, false>, dim3(grid), dim3(NUM_THREADS), SMEM_BYTES, st, tw, to, tx, (const TI *)x, p);  \
    } while (0)
    if (in_dtype == TU_F32) TU_STEM_LAUNCH(float);
    else if (in_dtype == TU_U8) TU_STEM_LAUNCH(uint8_t);
    else if (in_dtype == TU_F16) TU_STEM_LAUNCH(f16);
    else TU_STEM_LAUNCH(bf16);
#undef TU_STEM_LAUNCH
    TU_CHECK_LAUNCH("stem_tc");
    return TU_OK;
}

}  // namespace tu
