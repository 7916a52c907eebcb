// conv1 (3 -> 64, 3x3, + ReLU) FUSED INTO conv2 (64 -> 64, 3x3, + ReLU): the 64-channel full-resolution output of conv1
// (944 MB for eight 720p frames, written once and read once: 0.185 ms of HBM time) never leaves the SM.
//
// Reference: `feat = relu(conv1(x)); feat = relu(conv2(feat))` (WindowTransformer/model.py:244-245,
// FastTransformer/model.py:251-252, ResidualTransformer/model.py:128-129).
//
// conv2 is the streaming ky-stacked kernel of conv3x3_stream_tcgen05.cu (a work item = a strip of 128 pixels x R rows; one
// input row per step; a ring of row accumulators in TMEM).  There, a TMA load fills each input-row slot (136 pixels x 128 B,
// 128-byte swizzled).  Here the slot is PRODUCED ON CHIP, one conv1 row per step, by the stem pipeline of stem_tcgen05.cu:
//   warp 0      raw-image TMA producer: one image row (3 channels x 128 + 2 PADL pixels, zero-filled outside = conv1's
//               padding) per step into a 4-stage ring; also loads both filter banks once
//   warps 12-15 builders: a thread owns pixel x0 + i, keeps a 3x3x3 register window sliding down the strip and writes its
//               im2col row (27 taps + the two bias columns, bf16) into the swizzled operand tile
//   warp 1      MMA issuer: per step two 128x64x16 stem MMAs (three rows AHEAD of the conv2 row they feed) into one of two
//               stem accumulators, then conv2's 12 (or 24) ky-stacked MMAs of the current row
//   warps 8-11  stem epilogue: accumulator -> ReLU -> bf16 -> rows 1..128 of the conv2 input slot (zero outside the image =
//               conv2's padding), exactly the bytes TMA would have put there
//   warps 2-3   halo: the strip needs conv1 at x0-1 and x0+128 too; 2 pixels x 64 channels x 27 taps per row are cheaper on
//               the CUDA cores (one warp per side, two channels per lane, filter in registers) than a second MMA
//   warps 4-7   conv2 epilogue (unchanged): accumulator -> +bias, ReLU -> bf16 -> swizzled staging -> TMA store
// TMEM: columns [0,384) six conv2 row accumulators, [384,512) two stem accumulators.
#include <cuda.h>
#include <string.h>

#include "ptx.cuh"
#include "tc_api.cuh"

namespace tu {

namespace {

constexpr int TILE_M = 128, BOXW = 136;
constexpr int UNIT_BYTES = BOXW * 128;        // one conv2 input row slot
constexpr int RING = 4;
constexpr int NACC = 6;                       // conv2 row accumulators (64 columns each)
constexpr int STEM_COL0 = NACC * 64;          // 384
constexpr int W2_BLK = 64 * 128, W2_KX = 3 * W2_BLK, W2_BYTES = 3 * W2_KX;     // 73728
constexpr int W1_BYTES = 64 * 128;
constexpr int A1_BYTES = 128 * 128;
constexpr int STG_BYTES = 4 * 2 * 4096;
constexpr int NRAW = 4;
constexpr int STEM_LEAD = 3;                   // conv1 rows the stem MMAs run ahead of the conv2 row they feed (ring of 4 slots)
constexpr int RAW_STAGE = 1664;               // >= 3 * (128 + 2 PADL) * sizeof(TI) for every TI, multiple of 128
constexpr int OFF_RING = W2_BYTES;
constexpr int OFF_A1 = OFF_RING + RING * UNIT_BYTES;
constexpr int OFF_W1 = OFF_A1 + A1_BYTES;
constexpr int OFF_STG = OFF_W1 + W1_BYTES;
constexpr int OFF_RAW = OFF_STG + STG_BYTES;
constexpr int OFF_BAR = OFF_RAW + NRAW * RAW_STAGE;
constexpr int SMEM_BYTES = OFF_BAR + 640 + 1024;
constexpr int NUM_THREADS = 512;
static_assert(OFF_A1 % 1024 == 0 && OFF_W1 % 1024 == 0 && OFF_STG % 1024 == 0 && SMEM_BYTES <= 232448, "shared memory layout");

template <typename TI> struct RawRow {
    static constexpr int PADL = 16 / (int)sizeof(TI);        // the innermost TMA start coordinate must be 16-byte aligned
    static constexpr int RW = 128 + 2 * PADL;
    static constexpr int BYTES = 3 * RW * (int)sizeof(TI);
    static_assert(BYTES <= RAW_STAGE, "raw row exceeds its stage");
};

struct FusedParams {
    int B, H, W, relu;
    int R;                  // conv2 output rows per work item
    int tiles_x, chunks_y, total_items;
    const float *bias1, *bias2;
    const bf16 *w64;        // conv1 filter (64 co, 64 k) for the halo warps
};

struct FusedBarriers {
    uint64_t full[RING], empty[RING];
    uint64_t acc_full[NACC], acc_empty[NACC];
    uint64_t s_full[2], s_empty[2];
    uint64_t raw_full[NRAW], raw_empty[NRAW];
    uint64_t a_full, a_empty, w_full;
    uint32_t tmem_base;
};
static_assert(sizeof(FusedBarriers) <= 384, "barrier block too large (the last 256 bytes of its 640-byte area hold conv2's bias)");

__device__ __forceinline__ float ldx(float v) { return v; }
__device__ __forceinline__ float ldx(bf16 v) { return __bfloat162float(v); }
__device__ __forceinline__ float ldx(f16 v) { return __half2float(v); }
__device__ __forceinline__ float ldx(uint8_t v) { return u8_to_float(v) * 0.00392156862745098f; }
__device__ __forceinline__ uint32_t pack2_relu(float lo, float hi) {
    uint32_t d;
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    return d;
}
__device__ __forceinline__ uint32_t pack2(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t *>(&h);
}
__device__ __forceinline__ float bf16_round(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }

template <typename TI>
__global__ void __launch_bounds__(NUM_THREADS, 1)
conv12_fused_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_w1,
                    const __grid_constant__ CUtensorMap tmap_w2, const __grid_constant__ CUtensorMap tmap_out, const FusedParams p) {
    using G = RawRow<TI>;
    pdl_trigger();
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem0 = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t *sm = smem_raw + (smem0 - ptx::smem_u32(smem_raw));
    FusedBarriers *bars = reinterpret_cast<FusedBarriers *>(sm + OFF_BAR);
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        for (int i = 0; i < RING; ++i) {
            ptx::mbar_init(ptx::smem_u32(&bars->full[i]), 6);          // 4 stem-epilogue warps + 2 halo warps
            ptx::mbar_init(ptx::smem_u32(&bars->empty[i]), 1);
        }
        for (int i = 0; i < NACC; ++i) {
            ptx::mbar_init(ptx::smem_u32(&bars->acc_full[i]), 1);
            ptx::mbar_init(ptx::smem_u32(&bars->acc_empty[i]), 4);
        }
        for (int i = 0; i < 2; ++i) {
            ptx::mbar_init(ptx::smem_u32(&bars->s_full[i]), 1);
            ptx::mbar_init(ptx::smem_u32(&bars->s_empty[i]), 4);
        }
        for (int i = 0; i < NRAW; ++i) {
            ptx::mbar_init(ptx::smem_u32(&bars->raw_full[i]), 1);
            ptx::mbar_init(ptx::smem_u32(&bars->raw_empty[i]), 6);     // 4 builder warps + 2 halo warps
        }
        ptx::mbar_init(ptx::smem_u32(&bars->a_full), 128);
        ptx::mbar_init(ptx::smem_u32(&bars->a_empty), 1);
        ptx::mbar_init(ptx::smem_u32(&bars->w_full), 1);
        ptx::fence_barrier_init();
    }
    if (warp == 2) {
        ptx::tmem_alloc(ptx::smem_u32(&bars->tmem_base), 512);
        ptx::tmem_relinquish();
    }
    if (warp == 0 && lane == 0) {
        ptx::prefetch_tmap(&tmap_x);
        ptx::prefetch_tmap(&tmap_w1);
        ptx::prefetch_tmap(&tmap_w2);
        ptx::prefetch_tmap(&tmap_out);
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = bars->tmem_base;
    pdl_wait();

    auto item_geom = [&](int it, int &b, int &y0, int &rows, int &x0) {
        const int tx = it % p.tiles_x;
        int rem = it / p.tiles_x;
        const int cy = rem % p.chunks_y;
        b = rem / p.chunks_y;
        y0 = cy * p.R;
        rows = min(p.R, p.H - y0);
        x0 = tx * TILE_M;
    };

    if (warp == 0) {
        if (lane == 0) {
            // ================================ TMA producer: filter banks once, then one raw image row per step ================================
            ptx::mbar_expect_tx(ptx::smem_u32(&bars->w_full), W2_BYTES + W1_BYTES);
            for (int kx = 0; kx < 3; ++kx)
                for (int j = 0; j < 3; ++j)       // conv2 bank as [kx][ky = 2, 1, 0][co][ci]
                    ptx::tma_load_2d(smem0 + kx * W2_KX + j * W2_BLK, &tmap_w2, ptx::smem_u32(&bars->w_full), 0, ((2 - j) * 3 + kx) * 64);
            ptx::tma_load_2d(smem0 + OFF_W1, &tmap_w1, ptx::smem_u32(&bars->w_full), 0, 0);
            int stage = 0;
            uint32_t phase = 0;
            for (int it = blockIdx.x; it < p.total_items; it += gridDim.x) {
                int b, y0, rows, x0;
                item_geom(it, b, y0, rows, x0);
                for (int j = 0; j < rows + 4; ++j) {           // image rows y0 - 2 .. y0 + rows + 1
                    ptx::mbar_wait(ptx::smem_u32(&bars->raw_empty[stage]), phase ^ 1);
                    const uint32_t fb = ptx::smem_u32(&bars->raw_full[stage]);
                    ptx::mbar_expect_tx(fb, G::BYTES);
                    ptx::tma_load_4d(smem0 + OFF_RAW + stage * RAW_STAGE, &tmap_x, fb, x0 - G::PADL, y0 - 2 + j, 0, b);
                    if (++stage == NRAW) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ================================ MMA issuer (whole warp converged, elected lane issues) ================================
        const uint32_t leader = ptx::elect_one();
        ptx::mbar_wait(ptx::smem_u32(&bars->w_full), 0);
        // conv1's bias rides in the contraction: operand columns k = 27, 28 are 1, filter columns 27, 28 hold the bias as bf16 hi + lo
#pragma unroll
        for (int co = lane; co < 64; co += 32) {
            const float bv = p.bias1[co];
            const bf16 hi = __float2bfloat16_rn(bv), lo = __float2bfloat16_rn(bv - __bfloat162float(hi));
            bf16 *row = reinterpret_cast<bf16 *>(sm + OFF_W1 + co * 128 + ((3 ^ (co & 7)) << 4));
            row[3] = hi;      // k = 27
            row[4] = lo;      // k = 28
        }
        ptx::fence_proxy_async();
        __syncwarp();
        const uint32_t w2_lo = ptx::sdesc_lo(smem0), ring_lo = ptx::sdesc_lo(smem0 + OFF_RING);
        const uint32_t a1_lo = ptx::sdesc_lo(smem0 + OFF_A1), w1_lo = ptx::sdesc_lo(smem0 + OFF_W1);
        const uint32_t idesc1 = ptx::make_idesc_bf16(128, 64);
        // the stem runs over the flat sequence of conv1 rows of all this CTA's items, STEM_LEAD rows ahead of conv2
        long stem_total = 0;
        for (int it = blockIdx.x; it < p.total_items; it += gridDim.x) {
            int b, y0, rows, x0;
            item_geom(it, b, y0, rows, x0);
            stem_total += rows + 2;
        }
        long stem_issued = 0;
        uint32_t aph = 0;
        auto issue_stem = [&]() {
            const uint32_t set = (uint32_t)stem_issued & 1u, sph = ((uint32_t)stem_issued >> 1) & 1u;
            ptx::mbar_wait(ptx::smem_u32(&bars->a_full), aph);
            ptx::mbar_wait(ptx::smem_u32(&bars->s_empty[set]), sph ^ 1);
            ptx::tc_fence_after();
            const uint32_t d = tmem_base + STEM_COL0 + set * 64;
            ptx::umma_bf16_lo<0>(d, a1_lo, w1_lo, idesc1, leader);                 // k = 0..15
            ptx::umma_bf16_lo<1>(d, a1_lo + 2, w1_lo + 2, idesc1, leader);         // k = 16..31 (27 taps, 2 bias columns, 3 zeros)
            ptx::umma_commit_pred(ptx::smem_u32(&bars->s_full[set]), leader);
            ptx::umma_commit_pred(ptx::smem_u32(&bars->a_empty), leader);
            aph ^= 1;
            ++stem_issued;
        };
        for (int k = 0; k < STEM_LEAD && stem_issued < stem_total; ++k) issue_stem();
        uint32_t rs = 0;                                   // conv2 input rows consumed so far (ring slot = rs % RING)
        uint32_t g0 = 0;                                   // running index of the item's first output row
        for (int it = blockIdx.x; it < p.total_items; it += gridDim.x) {
            int b, y0, rows, x0;
            item_geom(it, b, y0, rows, x0);
            for (int u = 0; u < rows + 2; ++u, ++rs) {
                if (stem_issued < stem_total) issue_stem();
                const int slot = rs % RING;
                const uint32_t phase = (rs / RING) & 1;
                const int lo = max(u - 2, 0), hi = min(u, rows - 1);
                ptx::mbar_wait(ptx::smem_u32(&bars->full[slot]), phase);
                if (u <= rows - 1) {                       // row u opens: its accumulator must have been drained and cleared
                    const uint32_t g = g0 + u;
                    ptx::mbar_wait(ptx::smem_u32(&bars->acc_empty[g % NACC]), (g / NACC) & 1);
                }
                ptx::tc_fence_after();
                const uint32_t a_lo = ring_lo + ((uint32_t)(slot * UNIT_BYTES) >> 4);
                const int n = hi - lo + 1, blk0 = 2 - (u - lo);
                const int s0 = (g0 + lo) % NACC;
                const int n1 = min(n, NACC - s0), n2 = n - n1;
                const uint32_t d1 = tmem_base + s0 * 64, b1 = w2_lo + ((uint32_t)(blk0 * W2_BLK) >> 4);
                const uint32_t id1 = ptx::make_idesc_bf16(TILE_M, 64 * n1);
                if (n2 == 0) {
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx)
#pragma unroll
                        for (int k4 = 0; k4 < 4; ++k4)
                            ptx::umma_bf16_lo<1>(d1, a_lo + ((kx * 128 + k4 * 32) >> 4), b1 + ((kx * W2_KX + k4 * 32) >> 4), id1, leader);
                } else {
                    const uint32_t b2 = b1 + ((uint32_t)(n1 * W2_BLK) >> 4), id2 = ptx::make_idesc_bf16(TILE_M, 64 * n2);
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx)
#pragma unroll
                        for (int k4 = 0; k4 < 4; ++k4) {
                            ptx::umma_bf16_lo<1>(d1, a_lo + ((kx * 128 + k4 * 32) >> 4), b1 + ((kx * W2_KX + k4 * 32) >> 4), id1, leader);
                            ptx::umma_bf16_lo<1>(tmem_base, a_lo + ((kx * 128 + k4 * 32) >> 4), b2 + ((kx * W2_KX + k4 * 32) >> 4), id2, leader);
                        }
                }
                ptx::umma_commit_pred(ptx::smem_u32(&bars->empty[slot]), leader);
                if (u >= 2) ptx::umma_commit_pred(ptx::smem_u32(&bars->acc_full[(g0 + u - 2) % NACC]), leader);
            }
            g0 += rows;
        }
    } else if (warp == 2 || warp == 3) {
        // ================================ halo pixels x0 - 1 (warp 2) and x0 + 128 (warp 3) on the CUDA cores ================================
        const int side = warp - 2;
        float wf[2][27], bsv[2];
#pragma unroll
        for (int c2 = 0; c2 < 2; ++c2) {
            const int co = 2 * lane + c2;
            bsv[c2] = p.bias1[co];
#pragma unroll
            for (int k = 0; k < 27; ++k) wf[c2][k] = __bfloat162float(p.w64[co * 64 + k]);
        }
        float v[3][3][3];                                  // [row][kx][c], bf16-rounded like the tensor-core operand
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int kx = 0; kx < 3; ++kx)
#pragma unroll
                for (int c = 0; c < 3; ++c) v[r][kx][c] = 0.f;
        int stage = 0;
        uint32_t rphase = 0, rs = 0;
        for (int it = blockIdx.x; it < p.total_items; it += gridDim.x) {
            int b, y0, rows, x0;
            item_geom(it, b, y0, rows, x0);
            const int px = side ? x0 + 128 : x0 - 1;
            const int col = G::PADL + (side ? 128 : -1) - 1;               // raw column of tap kx = 0
            for (int j = 0; j < rows + 4; ++j) {
                ptx::mbar_wait(ptx::smem_u32(&bars->raw_full[stage]), rphase);
                const TI *raw = reinterpret_cast<const TI *>(sm + OFF_RAW + stage * RAW_STAGE);
#pragma unroll
                for (int kx = 0; kx < 3; ++kx)
#pragma unroll
                    for (int c = 0; c < 3; ++c) {
                        v[0][kx][c] = v[1][kx][c];
                        v[1][kx][c] = v[2][kx][c];
                        v[2][kx][c] = bf16_round(ldx(raw[c * G::RW + col + kx]));
                    }
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive(ptx::smem_u32(&bars->raw_empty[stage]));
                if (++stage == NRAW) { stage = 0; rphase ^= 1; }
                if (j < 2) continue;
                const int y = y0 - 1 + (j - 2);                             // conv1 row held by the window's middle row
                float a0 = bsv[0], a1 = bsv[1];
#pragma unroll
                for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx)
#pragma unroll
                        for (int c = 0; c < 3; ++c) {
                            a0 = fmaf(v[ky][kx][c], wf[0][(ky * 3 + kx) * 3 + c], a0);
                            a1 = fmaf(v[ky][kx][c], wf[1][(ky * 3 + kx) * 3 + c], a1);
                        }
                const bool inside = y >= 0 && y < p.H && px >= 0 && px < p.W;
                const uint32_t val = inside ? pack2_relu(a0, a1) : 0u;
                const int slot = rs % RING;
                ptx::mbar_wait(ptx::smem_u32(&bars->empty[slot]), ((rs / RING) & 1) ^ 1);
                const int row = side ? 129 : 0;
                *reinterpret_cast<uint32_t *>(sm + OFF_RING + slot * UNIT_BYTES + row * 128 + (((lane >> 2) ^ (row & 7)) << 4) + (lane & 3) * 4) = val;
                ptx::fence_proxy_async();
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive(ptx::smem_u32(&bars->full[slot]));
                ++rs;
            }
        }
    } else if (warp >= 12) {
        // ================================ builders: im2col row of pixel x0 + i -> swizzled operand tile ================================
        const int i = (warp - 12) * 32 + lane;
        float v[3][3][3];                                  // [row][kx][c]
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int kx = 0; kx < 3; ++kx)
#pragma unroll
                for (int c = 0; c < 3; ++c) v[r][kx][c] = 0.f;
        int stage = 0;
        uint32_t rphase = 0, aph = 0;
        uint8_t *rowp = sm + OFF_A1 + i * 128;
        for (int it = blockIdx.x; it < p.total_items; it += gridDim.x) {
            int b, y0, rows, x0;
            item_geom(it, b, y0, rows, x0);
            for (int j = 0; j < rows + 4; ++j) {
                ptx::mbar_wait(ptx::smem_u32(&bars->raw_full[stage]), rphase);
                const TI *raw = reinterpret_cast<const TI *>(sm + OFF_RAW + stage * RAW_STAGE) + (G::PADL - 1 + i);
#pragma unroll
                for (int kx = 0; kx < 3; ++kx)
#pragma unroll
                    for (int c = 0; c < 3; ++c) {
                        v[0][kx][c] = v[1][kx][c];
                        v[1][kx][c] = v[2][kx][c];
                        v[2][kx][c] = ldx(raw[c * G::RW + kx]);
                    }
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive(ptx::smem_u32(&bars->raw_empty[stage]));
                if (++stage == NRAW) { stage = 0; rphase ^= 1; }
                if (j < 2) continue;
                ptx::mbar_wait(ptx::smem_u32(&bars->a_empty), aph ^ 1);           // the stem MMAs of the previous row have read the tile
                aph ^= 1;
                float k[32];
#pragma unroll
                for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx)
#pragma unroll
                        for (int c = 0; c < 3; ++c) k[(ky * 3 + kx) * 3 + c] = v[ky][kx][c];
#pragma unroll
                for (int z = 27; z < 32; ++z) k[z] = z < 29 ? 1.f : 0.f;
#pragma unroll
                for (int ch = 0; ch < 4; ++ch) {
                    uint4 u;
                    u.x = pack2(k[ch * 8 + 0], k[ch * 8 + 1]);
                    u.y = pack2(k[ch * 8 + 2], k[ch * 8 + 3]);
                    u.z = pack2(k[ch * 8 + 4], k[ch * 8 + 5]);
                    u.w = pack2(k[ch * 8 + 6], k[ch * 8 + 7]);
                    *reinterpret_cast<uint4 *>(rowp + ((ch ^ (i & 7)) << 4)) = u;
                }
                ptx::fence_proxy_async();
                ptx::mbar_arrive(ptx::smem_u32(&bars->a_full));
            }
        }
    } else if (warp >= 8) {
        // ================================ stem epilogue: conv1 row -> rows 1..128 of the conv2 input slot ================================
        const int q = warp - 8;
        uint32_t su = 0;                                   // conv1 rows drained so far (= conv2 input rows produced)
        for (int it = blockIdx.x; it < p.total_items; it += gridDim.x) {
            int b, y0, rows, x0;
            item_geom(it, b, y0, rows, x0);
            const int px = x0 + q * 32 + lane;
#pragma unroll 1
            for (int u = 0; u < rows + 2; ++u, ++su) {
                const int y = y0 - 1 + u;
                const uint32_t set = su & 1u;
                ptx::mbar_wait(ptx::smem_u32(&bars->s_full[set]), (su >> 1) & 1);
                ptx::tc_fence_after();
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + STEM_COL0 + set * 64;
                uint32_t v0[32], v1[32];
                ptx::tmem_ld_x32(taddr, v0);
                ptx::tmem_ld_x32(taddr + 32, v1);
                ptx::tmem_ld_wait();
                ptx::tc_fence_before();
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive(ptx::smem_u32(&bars->s_empty[set]));
                const int slot = su % RING;
                ptx::mbar_wait(ptx::smem_u32(&bars->empty[slot]), ((su / RING) & 1) ^ 1);       // conv2 has consumed the slot's previous row
                const bool inside = y >= 0 && y < p.H && px < p.W;
                const int row = 1 + q * 32 + lane;
                uint8_t *rowp = sm + OFF_RING + slot * UNIT_BYTES + row * 128;
#pragma unroll
                for (int c = 0; c < 64; c += 8) {
                    const uint32_t *v = c < 32 ? &v0[c] : &v1[c - 32];
                    uint4 o;
                    o.x = inside ? pack2_relu(__uint_as_float(v[0]), __uint_as_float(v[1])) : 0u;
                    o.y = inside ? pack2_relu(__uint_as_float(v[2]), __uint_as_float(v[3])) : 0u;
                    o.z = inside ? pack2_relu(__uint_as_float(v[4]), __uint_as_float(v[5])) : 0u;
                    o.w = inside ? pack2_relu(__uint_as_float(v[6]), __uint_as_float(v[7])) : 0u;
                    *reinterpret_cast<uint4 *>(rowp + (((c >> 3) ^ (row & 7)) << 4)) = o;
                }
                ptx::fence_proxy_async();
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive(ptx::smem_u32(&bars->full[slot]));
            }
        }
    } else {
        // ================================ conv2 epilogue (warps 4-7): one output row at a time ================================
        const int q = warp - 4;
        uint32_t g = 0, nstore = 0;
        // conv2's bias is folded into the accumulators: a row accumulator is "cleared" to the bias vector, so the drain is only
        // ReLU + convert (it used to issue 64 bias loads per row and thread on a kernel bound by the load/store and
        // shared-memory pipes).  The vector is staged once in shared memory and re-read (8 x 128 bit) for every clear.
        float *bias_s = reinterpret_cast<float *>(sm + OFF_BAR + 384);
        if (q == 0) {
            bias_s[lane] = p.bias2 ? p.bias2[lane] : 0.f;
            bias_s[lane + 32] = p.bias2 ? p.bias2[lane + 32] : 0.f;
        }
        asm volatile("bar.sync 3, 128;" ::: "memory");
        auto store_bias = [&](uint32_t taddr) {           // 64 columns of this warp's 32 lanes <- bias
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                uint32_t t[32];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    uint4 u;
                    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(u.x), "=r"(u.y), "=r"(u.z), "=r"(u.w)
                                 : "r"(ptx::smem_u32(bias_s + h * 32 + j * 4)));
                    t[j * 4 + 0] = u.x; t[j * 4 + 1] = u.y; t[j * 4 + 2] = u.z; t[j * 4 + 3] = u.w;
                }
                ptx::tmem_st_x32(taddr + h * 32, t);
            }
        };
        for (int sl = 0; sl < NACC; ++sl) store_bias(tmem_base + ((uint32_t)(q * 32) << 16) + sl * 64);
        ptx::tmem_st_wait();
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0)
            for (int sl = 0; sl < NACC; ++sl) ptx::mbar_arrive(ptx::smem_u32(&bars->acc_empty[sl]));
        uint8_t *stg_w = sm + OFF_STG + q * 8192;
        const uint32_t stg_w_sm = smem0 + OFF_STG + q * 8192;
        for (int it = blockIdx.x; it < p.total_items; it += gridDim.x) {
            int b, y0, rows, x0;
            item_geom(it, b, y0, rows, x0);
            const int px0 = x0 + q * 32;
#pragma unroll 1
            for (int m = 0; m < rows; ++m, ++g) {
                const int sl = g % NACC;
                ptx::mbar_wait(ptx::smem_u32(&bars->acc_full[sl]), (g / NACC) & 1);
                ptx::tc_fence_after();
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + sl * 64;
                uint32_t v0[32], v1[32];
                ptx::tmem_ld_x32(taddr, v0);
                ptx::tmem_ld_x32(taddr + 32, v1);
                ptx::tmem_ld_wait();
                store_bias(taddr);                      // "clear" the slot for the row that opens it next
                ptx::tmem_st_wait();
                ptx::tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                    ptx::mbar_arrive(ptx::smem_u32(&bars->acc_empty[sl]));
                    ptx::bulk_wait_read<1>();
                }
                __syncwarp();
                const uint32_t buf = nstore & 1;
                uint8_t *rowp = stg_w + buf * 4096 + lane * 128;
#pragma unroll
                for (int c = 0; c < 64; c += 8) {
                    const uint32_t *v = c < 32 ? &v0[c] : &v1[c - 32];
                    uint4 uu;      // conv2 is always followed by ReLU (W:245, F:252, R:129): one convert-with-ReLU per channel pair
                    uu.x = pack2_relu(__uint_as_float(v[0]), __uint_as_float(v[1]));
                    uu.y = pack2_relu(__uint_as_float(v[2]), __uint_as_float(v[3]));
                    uu.z = pack2_relu(__uint_as_float(v[4]), __uint_as_float(v[5]));
                    uu.w = pack2_relu(__uint_as_float(v[6]), __uint_as_float(v[7]));
                    *reinterpret_cast<uint4 *>(rowp + ((((c >> 3) ^ (lane & 7))) << 4)) = uu;
                }
                ptx::fence_proxy_async();
                __syncwarp();
                if (lane == 0) {
                    if (px0 < p.W) ptx::tma_store_4d(&tmap_out, stg_w_sm + buf * 4096, 0, px0, y0 + m, b);
                    ptx::bulk_commit();
                }
                ++nstore;
            }
        }
        if (lane == 0) ptx::bulk_wait<0>();
        __syncwarp();
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 2) ptx::tmem_dealloc(tmem_base, 512);
}

PerDeviceFlag g_attr_set_c;
thread_local int g_enable_fused = 1;

}  // namespace

void tc_set_conv12_fused(int on) { g_enable_fused = on; }

// relu(conv2(relu(conv1(x)))): NCHW image (fp32 | bf16 | fp16 | uint8) -> NHWC bf16 (B,H,W,64).  w64: conv1 filter bf16 (64 co, 64 k);
// w2: conv2 filter bf16 [9 taps][64 co][64 ci].  Needs an image row pitch that is a multiple of 16 bytes (raw rows arrive by TMA).
int tc_conv12_fused(const void *x, int in_dtype, const bf16 *w64, const float *bias1, const bf16 *w2, const float *bias2, bf16 *out,
                    int B, int H, int W, cudaStream_t st) {
    if (!g_enable_fused) return TU_TC_UNSUPPORTED;
    const int eb = (int)dtype_size(in_dtype);
    if (((size_t)W * eb) % 16 || (reinterpret_cast<uintptr_t>(x) & 15) || (reinterpret_cast<uintptr_t>(w64) & 127) ||
        (reinterpret_cast<uintptr_t>(w2) & 127) || (reinterpret_cast<uintptr_t>(out) & 15))
        return TU_TC_UNSUPPORTED;
    TcEncodeFn enc = tc_encode_fn();
    if (!enc) return TU_TC_UNSUPPORTED;
    const int g_sm_count_c = device_sm_count();
    if (!g_attr_set_c.is_set()) {
        cudaError_t e = cudaFuncSetAttribute(conv12_fused_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(conv12_fused_kernel<bf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(conv12_fused_kernel<uint8_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(conv12_fused_kernel<f16>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
        if (e != cudaSuccess) return cuda_fail(e, "conv12_fused smem attribute");
        g_attr_set_c.set();
    }
    CUtensorMap tm_x, tm_w1, tm_w2, tm_out;
    {
        const int rw = 128 + 2 * (16 / eb);
        cuuint64_t xd[4] = {(cuuint64_t)W, (cuuint64_t)H, 3, (cuuint64_t)B};
        cuuint64_t xs[3] = {(cuuint64_t)W * eb, (cuuint64_t)H * W * eb, (cuuint64_t)3 * H * W * eb};
        cuuint32_t xb[4] = {(cuuint32_t)rw, 1, 3, 1}, e1[4] = {1, 1, 1, 1};
        CUresult r = enc(&tm_x, tc_image_map_dtype(in_dtype), 4, const_cast<void *>(x), xd, xs, xb, e1, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        cuuint64_t w1d[2] = {64, 64}, wst[1] = {128};
        cuuint32_t wb[2] = {64, 64};
        if (r == CUDA_SUCCESS)
            r = enc(&tm_w1, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void *)w64, w1d, wst, wb, e1, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        cuuint64_t w2d[2] = {64, 9 * 64};
        if (r == CUDA_SUCCESS)
            r = enc(&tm_w2, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void *)w2, w2d, wst, wb, e1, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        cuuint32_t ob[4] = {64, 32, 1, 1};
        cuuint64_t od[4] = {64, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
        cuuint64_t os[3] = {128, (cuuint64_t)W * 128, (cuuint64_t)H * W * 128};
        if (r == CUDA_SUCCESS)
            r = enc(&tm_out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, (void *)out, od, os, ob, e1, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) {
            set_error("tu: cuTensorMapEncodeTiled(conv12 fused) failed with code " + std::to_string((int)r));
            return TU_ERR_CUDA;
        }
    }
    FusedParams p;
    p.B = B; p.H = H; p.W = W; p.relu = 1;
    p.tiles_x = ceil_div(W, TILE_M);
    int bestR = H < 8 ? H : 8;
    double best = 1e30;
    for (int R = 8; R <= 64 && R <= (H > 8 ? H : 8); ++R) {
        const long items = (long)p.tiles_x * ceil_div(H, R) * B;
        const long waves = (items + g_sm_count_c - 1) / g_sm_count_c;
        const double cost = (double)waves * (R + 2);
        if (cost < best - 1e-9) { best = cost; bestR = R; }
    }
    p.R = bestR;
    p.chunks_y = ceil_div(H, p.R);
    p.total_items = p.tiles_x * p.chunks_y * B;
    p.bias1 = bias1; p.bias2 = bias2; p.w64 = w64;
    const int grid = p.total_items < g_sm_count_c ? p.total_items : g_sm_count_c;
    if (in_dtype == TU_F32) launch_pdl(conv12_fused_kernel<float>, dim3(grid), dim3(NUM_THREADS), SMEM_BYTES, st, tm_x, tm_w1, tm_w2, tm_out, p);
    else if (in_dtype == TU_BF16) launch_pdl(conv12_fused_kernel<bf16>, dim3(grid), dim3(NUM_THREADS), SMEM_BYTES, st, tm_x, tm_w1, tm_w2, tm_out, p);
    else if (in_dtype == TU_F16) launch_pdl(conv12_fused_kernel<f16>, dim3(grid), dim3(NUM_THREADS), SMEM_BYTES, st, tm_x, tm_w1, tm_w2, tm_out, p);
    else launch_pdl(conv12_fused_kernel<uint8_t>, dim3(grid), dim3(NUM_THREADS), SMEM_BYTES, st, tm_x, tm_w1, tm_w2, tm_out, p);
    TU_CHECK_LAUNCH("conv12_fused");
    return TU_OK;
}

}  // namespace tu
