// ResidualTransformer's TransformerBlock (ResidualTransformer/model.py:22-50) around its global attention, in TWO fused kernels per
// layer instead of six (LayerNorm, qkv, proj, LayerNorm, fc1, fc2 were separate launches of 5-12 us each on 57 tiles of 128 tokens:
// 64 us per layer of latency for 3 us of math):
//
//   resid_pre_kernel    x -> LN1 -> in_proj (q | k | v, q pre-scaled) -> bf16 qkv rows in global memory
//   [global attention:  transformer_simt.cu::global_attn_mma_kernel or tc/global_attn_tcgen05.cu]
//   resid_post_kernel   x += out_proj(att);  x += fc2(GELU(fc1(LN2(x))))            (x: the fp32 token stream, in place)
//
// Both are the window-stack kernel (window_stack_tcgen05.cu) with the window attention taken out: a CTA takes 128 tokens, the fp32
// residual stream lives in TMEM columns [0,128) (out_proj and fc2 accumulate straight onto it, their biases ride in offset vectors
// added on read), LayerNorm output / attention output / GELU output are 128-byte-swizzled K-major A operands in shared memory, the
// weights stream as pre-packed [128 n x 64 k] slabs through a TMA ring in MMA consumption order (6 slabs for the pre kernel, 18 for
// the post kernel: the same 24-slab order per layer the window stack uses).  Token rows past M (3600 tokens per frame is not a
// multiple of 128) are loaded as zeros and never stored.
// Roles: warps 0-15 math (thread = token row x column quarter), warp 16 TMA producer, warp 17 MMA issuer + TMEM allocation.
#include <cuda.h>

#include "ptx.cuh"
#include "tc_api.cuh"

namespace tu {

namespace {

constexpr int DIM = 128;
constexpr int NMATH = 16;
constexpr int NUM_THREADS = (NMATH + 2) * 32;    // 576
constexpr int SLAB = 128 * 128;                 // 16 KB: 128 rows x 64 bf16
constexpr int NRING = 5;
constexpr int SLABS_PER_LAYER = 24, SLABS_PRE = 6;
constexpr int OFF_A32 = 0;
constexpr int OFF_HID = 2 * SLAB;               // GELU(fc1) half-tiles: 4 slabs
constexpr int OFF_RING = OFF_HID + 4 * SLAB;
constexpr int OFF_PAR = OFF_RING + NRING * SLAB;
constexpr int PAR_FLOATS = 1664 + 128;          // c0 | ln1w | ln1b | qkvb(384) | c1 | ln2w | ln2b | fc1b(512) | c_final
constexpr int OFF_STAT = OFF_PAR + PAR_FLOATS * 4;
constexpr int OFF_BAR = OFF_STAT + 128 * 4 * 8;
constexpr int SMEM_BYTES = OFF_BAR + 256 + 1024;
constexpr int P_C0 = 0, P_LN1W = 128, P_LN1B = 256, P_QKVB = 384, P_C1 = 768, P_LN2W = 896, P_LN2B = 1024, P_FC1B = 1152, P_CFIN = 1664;
static_assert(OFF_RING % 1024 == 0 && SMEM_BYTES <= 232448, "shared memory layout");

struct ResidParams {
    float *tok;            // (M, 128) fp32 token stream; the post kernel updates it in place
    bf16 *tok16;           // post kernel, optional: bf16 copy of the result
    bf16 *qkv;             // pre kernel: (M, 384) bf16 out
    const bf16 *att;       // post kernel: (M, 128) bf16 attention output
    const float *par;      // this layer's PAR_FLOATS parameters
    int M, n_tiles, slab0; // first weight slab of this launch in the packed stream
};

enum { ACC_0 = 0, ACC_1, ACC_2, ACC_PROJ, ACC_FC1A0, ACC_FC1A1, ACC_FC1B0, ACC_FC1B1, ACC_FC2B, NACC };

struct Barriers {
    uint64_t full[NRING], empty[NRING];
    uint64_t a_ready;
    uint64_t acc[NACC];
    uint32_t tmem_base;
};

__device__ __forceinline__ void math_barrier() { asm volatile("bar.sync 1, 512;" ::: "memory"); }
__device__ __forceinline__ uint32_t pk(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t *>(&h);
}
using ptx::f32x2;
__device__ __forceinline__ uint32_t pk_pair(f32x2 v) {
    float lo, hi;
    ptx::up2(v, lo, hi);
    return pk(lo, hi);
}
// GELU(x) = 0.5 x (1 + tanh(p(x))), p the odd polynomial fitted to atanh(erf(x / sqrt 2)) (|error| <= 2.6e-5; tools/fit_gelu.py)
__device__ __forceinline__ f32x2 gelu_fast2(f32x2 x) {
    float a, b;
    ptx::up2(ptx::mul2(x, x), a, b);
    const f32x2 x2 = ptx::pk2(fminf(a, 64.f), fminf(b, 64.f));
    f32x2 q = ptx::fma2(ptx::pk2(-0.0003515167826820022f, -0.0003515167826820022f), x2, ptx::pk2(0.03700564597780192f, 0.03700564597780192f));
    q = ptx::fma2(q, x2, ptx::pk2(0.7975078843613885f, 0.7975078843613885f));
    float u0, u1, t0, t1;
    ptx::up2(ptx::mul2(x, q), u0, u1);
    asm("tanh.approx.f32 %0, %1;" : "=f"(t0) : "f"(u0));
    asm("tanh.approx.f32 %0, %1;" : "=f"(t1) : "f"(u1));
    const f32x2 h = ptx::mul2(x, ptx::pk2(0.5f, 0.5f));
    return ptx::fma2(h, ptx::pk2(t0, t1), h);
}

// LayerNorm of this thread's 32 columns of row i; statistics shared with the three partner threads of the row; result -> A32, swizzled
__device__ __forceinline__ void layernorm_to_a32(f32x2 (&x)[16], const float *gam, const float *bet, float2 *stat, uint8_t *a32, int i, int part) {
    // one exchange: every thread publishes the mean and M2 = sum (x - mean)^2 of its own 32 columns (two passes over registers);
    // Chan's combination M2 = sum M2_p + 32 sum (mean_p - mean)^2 keeps the variance exact for rows whose channels share an offset
    // far above their spread, where E[x^2] - mean^2 in fp32 cancels away
    f32x2 s2 = ptx::pk2(0.f, 0.f), q2 = ptx::pk2(0.f, 0.f);
#pragma unroll
    for (int j = 0; j < 16; ++j) s2 = ptx::add2(s2, x[j]);
    float s_lo, s_hi, q_lo, q_hi;
    ptx::up2(s2, s_lo, s_hi);
    const float pmean = (s_lo + s_hi) * (1.0f / 32);
    const f32x2 npm = ptx::pk2(-pmean, -pmean);
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const f32x2 d = ptx::add2(x[j], npm);
        q2 = ptx::fma2(d, d, q2);
    }
    ptx::up2(q2, q_lo, q_hi);
    stat[i * 4 + part] = make_float2(pmean, q_lo + q_hi);
    math_barrier();
    const float4 p01 = *reinterpret_cast<const float4 *>(stat + i * 4), p23 = *reinterpret_cast<const float4 *>(stat + i * 4 + 2);
    const float mean = ((p01.x + p01.z) + (p23.x + p23.z)) * 0.25f;
    const float d0 = p01.x - mean, d1 = p01.z - mean, d2 = p23.x - mean, d3 = p23.z - mean;
    const float m2 = ((p01.y + p01.w) + (p23.y + p23.w)) + 32.0f * ((d0 * d0 + d1 * d1) + (d2 * d2 + d3 * d3));
    const float rstd = rsqrtf(m2 * (1.0f / DIM) + 1e-5f);
    const f32x2 nmean = ptx::pk2(-mean, -mean), rs = ptx::pk2(rstd, rstd);
    uint8_t *rowp = a32 + (part >> 1) * SLAB + i * 128;
#pragma unroll
    for (int ch = 0; ch < 4; ++ch) {
        uint32_t w[4];
#pragma unroll
        for (int e = 0; e < 4; ++e)
            w[e] = pk_pair(ptx::fma2(ptx::mul2(ptx::add2(x[ch * 4 + e], nmean), rs), ptx::ld2(gam + ch * 8 + 2 * e), ptx::ld2(bet + ch * 8 + 2 * e)));
        uint4 u;
        u.x = w[0]; u.y = w[1]; u.z = w[2]; u.w = w[3];
        *reinterpret_cast<uint4 *>(rowp + ((((part & 1) * 4 + ch) ^ (i & 7)) << 4)) = u;
    }
}

// POST == false: LN1 + in_proj -> qkv.   POST == true: out_proj + residual, LN2, MLP + residual.
template <bool POST>
__global__ void __launch_bounds__(NUM_THREADS, 1) resid_block_kernel(const __grid_constant__ CUtensorMap tmap_w, const ResidParams p) {
    pdl_trigger();
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem0 = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t *sm = smem_raw + (smem0 - ptx::smem_u32(smem_raw));
    Barriers *bars = reinterpret_cast<Barriers *>(sm + OFF_BAR);
    float *par = reinterpret_cast<float *>(sm + OFF_PAR);
    float2 *stat = reinterpret_cast<float2 *>(sm + OFF_STAT);
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    constexpr int NSLAB = POST ? SLABS_PER_LAYER - SLABS_PRE : SLABS_PRE;

    if (threadIdx.x == 0) {
        for (int i = 0; i < NRING; ++i) {
            ptx::mbar_init(ptx::smem_u32(&bars->full[i]), 1);
            ptx::mbar_init(ptx::smem_u32(&bars->empty[i]), 1);
        }
        ptx::mbar_init(ptx::smem_u32(&bars->a_ready), NMATH);
        for (int i = 0; i < NACC; ++i) ptx::mbar_init(ptx::smem_u32(&bars->acc[i]), 1);
        ptx::fence_barrier_init();
    }
    if (warp == NMATH + 1) {
        ptx::tmem_alloc(ptx::smem_u32(&bars->tmem_base), 512);
        ptx::tmem_relinquish();
    }
    if (warp == NMATH && lane == 0) ptx::prefetch_tmap(&tmap_w);
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = bars->tmem_base;
    const uint32_t TX = tmem_base, TACC = tmem_base + 128;
    pdl_wait();

    if (warp == NMATH) {
        if (lane == 0) {
            // ================================ TMA producer: this launch's weight slabs, once per tile ================================
            int stage = 0;
            uint32_t phase = 0;
            for (int t = blockIdx.x; t < p.n_tiles; t += gridDim.x)
                for (int s = 0; s < NSLAB; ++s) {
                    ptx::mbar_wait(ptx::smem_u32(&bars->empty[stage]), phase ^ 1);
                    const uint32_t fb = ptx::smem_u32(&bars->full[stage]);
                    ptx::mbar_expect_tx(fb, SLAB);
                    ptx::tma_load_2d(smem0 + OFF_RING + stage * SLAB, &tmap_w, fb, 0, (p.slab0 + s) * 128);
                    if (++stage == NRING) { stage = 0; phase ^= 1; }
                }
        }
    } else if (warp == NMATH + 1) {
        // ================================ MMA issuer ================================
        const uint32_t leader = ptx::elect_one();
        const uint32_t idesc = ptx::make_idesc_bf16(128, 128);
        const uint32_t ring_lo = ptx::sdesc_lo(smem0 + OFF_RING);
        int stage = 0;
        uint32_t phase = 0, aph = 0;
        auto slab_mma = [&](uint32_t d_tmem, uint32_t a_lo, bool first_clears) {
            ptx::mbar_wait(ptx::smem_u32(&bars->full[stage]), phase);
            ptx::tc_fence_after();
            const uint32_t w_lo = ring_lo + ((stage * SLAB) >> 4);
            ptx::umma_bf16_lo_rt(d_tmem, a_lo, w_lo, idesc, first_clears ? 0u : 1u, leader);
#pragma unroll
            for (int k4 = 1; k4 < 4; ++k4) ptx::umma_bf16_lo<1>(d_tmem, a_lo + k4 * 2, w_lo + k4 * 2, idesc, leader);
            ptx::umma_commit_pred(ptx::smem_u32(&bars->empty[stage]), leader);
            if (++stage == NRING) { stage = 0; phase ^= 1; }
        };
        auto wait_a = [&]() {
            ptx::mbar_wait(ptx::smem_u32(&bars->a_ready), aph);
            aph ^= 1;
            ptx::tc_fence_after();
        };
        const uint32_t a32 = ptx::sdesc_lo(smem0 + OFF_A32), hid = ptx::sdesc_lo(smem0 + OFF_HID);
        constexpr uint32_t SL = SLAB >> 4;
        for (int t = blockIdx.x; t < p.n_tiles; t += gridDim.x) {
            if (!POST) {
                wait_a();                                       // LN1 output in A32
                for (int nc = 0; nc < 3; ++nc) {
                    for (int ks = 0; ks < 2; ++ks) slab_mma(TACC + nc * 128, a32 + ks * SL, ks == 0);
                    ptx::umma_commit_pred(ptx::smem_u32(&bars->acc[ACC_0 + nc]), leader);
                }
            } else {
                wait_a();                                       // X in TMEM, attention output in A32
                for (int ks = 0; ks < 2; ++ks) slab_mma(TX, a32 + ks * SL, false);            // x += att Wo^T
                ptx::umma_commit_pred(ptx::smem_u32(&bars->acc[ACC_PROJ]), leader);
                wait_a();                                       // LN2 output in A32
                for (int nc = 0; nc < 2; ++nc) {
                    for (int ks = 0; ks < 2; ++ks) slab_mma(TACC + nc * 128, a32 + ks * SL, ks == 0);   // fc1, half 0
                    ptx::umma_commit_pred(ptx::smem_u32(&bars->acc[ACC_FC1A0 + nc]), leader);
                }
                wait_a();                                       // GELU(half 0) in HID
                for (int ks = 0; ks < 4; ++ks) slab_mma(TX, hid + ks * SL, false);            // x += h0 W2[:, h0]^T
                for (int nc = 0; nc < 2; ++nc) {
                    for (int ks = 0; ks < 2; ++ks) slab_mma(TACC + nc * 128, a32 + ks * SL, ks == 0);   // fc1, half 1
                    ptx::umma_commit_pred(ptx::smem_u32(&bars->acc[ACC_FC1B0 + nc]), leader);
                }
                wait_a();                                       // GELU(half 1) in HID
                for (int ks = 0; ks < 4; ++ks) slab_mma(TX, hid + ks * SL, false);
                ptx::umma_commit_pred(ptx::smem_u32(&bars->acc[ACC_FC2B]), leader);
            }
        }
    } else {
        // ================================ math warps ================================
        const int q = warp & 3, part = warp >> 2;           // TMEM lane quadrant, column quarter
        const int i = q * 32 + lane;                        // token row of the tile == TMEM lane
        const uint32_t lane_base = (uint32_t)(q * 32) << 16;
        const int mt = threadIdx.x;
        uint8_t *a32 = sm + OFF_A32, *hidp = sm + OFF_HID;
        uint32_t cph = 0;             // every acc barrier in use completes exactly once per tile: one shared phase bit
        auto wait_acc = [&](int which) {
            ptx::mbar_wait(ptx::smem_u32(&bars->acc[which]), cph);
            ptx::tc_fence_after();
        };
        auto signal_a = [&]() {
            ptx::fence_proxy_async();
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(ptx::smem_u32(&bars->a_ready));
        };
        // this layer's parameters -> smem, once
        {
            const float4 *g = reinterpret_cast<const float4 *>(p.par);
            float4 *d = reinterpret_cast<float4 *>(par);
            for (int e = mt; e < PAR_FLOATS / 4; e += NMATH * 32) d[e] = g[e];
        }
        math_barrier();
        for (int t = blockIdx.x; t < p.n_tiles; t += gridDim.x) {
            const long row = (long)t * 128 + i;
            const bool valid = row < p.M;
            const float *src = p.tok + row * DIM + part * 32;
            if (!POST) {
                // ---- LN1(x) -> A32 (x straight from global memory: the pre kernel needs no residual stream in TMEM)
                {
                    f32x2 x[16];
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        const float4 f = valid ? __ldcg(reinterpret_cast<const float4 *>(src + j)) : make_float4(0.f, 0.f, 0.f, 0.f);
                        x[j / 2] = ptx::pk2(f.x, f.y);
                        x[j / 2 + 1] = ptx::pk2(f.z, f.w);
                    }
                    layernorm_to_a32(x, par + P_LN1W + part * 32, par + P_LN1B + part * 32, stat, a32, i, part);
                }
                signal_a();
                // ---- in_proj epilogue: ACC -> (+bias) -> bf16 qkv rows in global memory, one column third at a time
                bf16 *dst = p.qkv + row * (3 * DIM);
#pragma unroll
                for (int nc = 0; nc < 3; ++nc) {
                    wait_acc(ACC_0 + nc);
                    uint32_t v[32];
                    const int col = nc * 128 + part * 32;
                    ptx::tmem_ld_x32(TACC + lane_base + col, v);
                    ptx::tmem_ld_wait();
                    const float *qb = par + P_QKVB + col;
#pragma unroll
                    for (int j = 0; j < 32; j += 8) {
                        uint4 u;
                        u.x = pk_pair(ptx::add2(ptx::pk2u(v[j + 0], v[j + 1]), ptx::ld2(qb + j + 0)));
                        u.y = pk_pair(ptx::add2(ptx::pk2u(v[j + 2], v[j + 3]), ptx::ld2(qb + j + 2)));
                        u.z = pk_pair(ptx::add2(ptx::pk2u(v[j + 4], v[j + 5]), ptx::ld2(qb + j + 4)));
                        u.w = pk_pair(ptx::add2(ptx::pk2u(v[j + 6], v[j + 7]), ptx::ld2(qb + j + 6)));
                        if (valid) *reinterpret_cast<uint4 *>(dst + col + j) = u;
                    }
                }
                ptx::tc_fence_before();
                cph ^= 1;
                math_barrier();       // A32 and the accumulators are free for the next tile
            } else {
                // ---- x -> TMEM X; attention output -> A32
                {
                    uint32_t v[32];
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        const float4 f = valid ? __ldcg(reinterpret_cast<const float4 *>(src + j)) : make_float4(0.f, 0.f, 0.f, 0.f);
                        v[j] = __float_as_uint(f.x); v[j + 1] = __float_as_uint(f.y); v[j + 2] = __float_as_uint(f.z); v[j + 3] = __float_as_uint(f.w);
                    }
                    ptx::tmem_st_x32(TX + lane_base + part * 32, v);
                    const bf16 *as = p.att + row * DIM + part * 32;
                    uint8_t *rowp = a32 + (part >> 1) * SLAB + i * 128;
#pragma unroll
                    for (int ch = 0; ch < 4; ++ch) {
                        const uint4 u = valid ? __ldcg(reinterpret_cast<const uint4 *>(as + ch * 8)) : make_uint4(0, 0, 0, 0);
                        *reinterpret_cast<uint4 *>(rowp + ((((part & 1) * 4 + ch) ^ (i & 7)) << 4)) = u;
                    }
                    ptx::tmem_st_wait();
                }
                signal_a();
                // ---- LN2(x + c1) -> A32 (after out_proj has been accumulated onto X)
                wait_acc(ACC_PROJ);
                {
                    uint32_t v[32];
                    ptx::tmem_ld_x32(TX + lane_base + part * 32, v);
                    ptx::tmem_ld_wait();
                    f32x2 x[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) x[j] = ptx::add2(ptx::pk2u(v[2 * j], v[2 * j + 1]), ptx::ld2(par + P_C1 + part * 32 + 2 * j));
                    layernorm_to_a32(x, par + P_LN2W + part * 32, par + P_LN2B + part * 32, stat, a32, i, part);
                }
                signal_a();
                // ---- MLP: two halves of the hidden layer: ACC -> +bias -> GELU -> bf16 HID slabs
#pragma unroll 1
                for (int half = 0; half < 2; ++half) {
#pragma unroll
                    for (int nc = 0; nc < 2; ++nc) {
                        wait_acc((half ? ACC_FC1B0 : ACC_FC1A0) + nc);
                        const int col = nc * 128 + part * 32;
                        uint8_t *rowp = hidp + (col >> 6) * SLAB + i * 128;
                        uint32_t v[32];
                        ptx::tmem_ld_x32(TACC + lane_base + col, v);
                        ptx::tmem_ld_wait();
                        const float *bb = par + P_FC1B + half * 256 + col;
#pragma unroll
                        for (int j = 0; j < 32; j += 8) {
                            uint4 u;
                            u.x = pk_pair(gelu_fast2(ptx::add2(ptx::pk2u(v[j + 0], v[j + 1]), ptx::ld2(bb + j + 0))));
                            u.y = pk_pair(gelu_fast2(ptx::add2(ptx::pk2u(v[j + 2], v[j + 3]), ptx::ld2(bb + j + 2))));
                            u.z = pk_pair(gelu_fast2(ptx::add2(ptx::pk2u(v[j + 4], v[j + 5]), ptx::ld2(bb + j + 4))));
                            u.w = pk_pair(gelu_fast2(ptx::add2(ptx::pk2u(v[j + 6], v[j + 7]), ptx::ld2(bb + j + 6))));
                            const int ch = ((col & 63) + j) >> 3;
                            *reinterpret_cast<uint4 *>(rowp + ((ch ^ (i & 7)) << 4)) = u;
                        }
                    }
                    signal_a();
                }
                wait_acc(ACC_FC2B);      // fc2 of the second half accumulated: X holds the block output (minus the folded biases)
                cph ^= 1;
                // ---- X + c_final -> global (fp32 stream, optional bf16 copy)
                {
                    float *dst = p.tok + row * DIM + part * 32;
                    bf16 *dst16 = p.tok16 ? p.tok16 + row * DIM + part * 32 : nullptr;
                    const float *cfin = par + P_CFIN + part * 32;
                    uint32_t v[32];
                    ptx::tmem_ld_x32(TX + lane_base + part * 32, v);
                    ptx::tmem_ld_wait();
                    if (valid) {
#pragma unroll
                        for (int j = 0; j < 32; j += 4) {
                            float4 f;
                            f.x = __uint_as_float(v[j]) + cfin[j];
                            f.y = __uint_as_float(v[j + 1]) + cfin[j + 1];
                            f.z = __uint_as_float(v[j + 2]) + cfin[j + 2];
                            f.w = __uint_as_float(v[j + 3]) + cfin[j + 3];
                            *reinterpret_cast<float4 *>(dst + j) = f;
                            if (dst16) {
                                uint2 u;
                                u.x = pk(f.x, f.y); u.y = pk(f.z, f.w);
                                *reinterpret_cast<uint2 *>(dst16 + j) = u;
                            }
                        }
                    }
                    ptx::tc_fence_before();
                }
                math_barrier();       // X, A32 and HID are free for the next tile
            }
        }
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == NMATH + 1) ptx::tmem_dealloc(tmem_base, 512);
}

PerDeviceFlag g_rb_attr;
thread_local int g_rb_enable = 1;

}  // namespace

void tc_set_resid_fused(int on) { g_rb_enable = on; }

static int resid_launch(bool post, const ResidParams &p0, const bf16 *stack_w, int n_layers, cudaStream_t st) {
    TcEncodeFn enc = tc_encode_fn();
    if (!enc) return TU_TC_UNSUPPORTED;
    if (!g_rb_attr.is_set()) {
        cudaError_t e = cudaFuncSetAttribute(resid_block_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(resid_block_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
        if (e != cudaSuccess) return cuda_fail(e, "resid_block smem attribute");
        g_rb_attr.set();
    }
    CUtensorMap tw;
    cuuint64_t wd[2] = {64, (cuuint64_t)n_layers * SLABS_PER_LAYER * 128}, ws[1] = {128};
    cuuint32_t wb[2] = {64, 128}, we[2] = {1, 1};
    CUresult r = enc(&tw, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void *)stack_w, wd, ws, wb, we, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("tu: cuTensorMapEncodeTiled(residual block weights) failed with code " + std::to_string((int)r));
        return TU_ERR_CUDA;
    }
    const int sms = device_sm_count();
    const int grid = p0.n_tiles < sms ? p0.n_tiles : sms;
    if (post) launch_pdl(resid_block_kernel<true>, dim3(grid), dim3(NUM_THREADS), (size_t)SMEM_BYTES, st, tw, p0);
    else launch_pdl(resid_block_kernel<false>, dim3(grid), dim3(NUM_THREADS), (size_t)SMEM_BYTES, st, tw, p0);
    TU_CHECK_LAUNCH(post ? "resid_post" : "resid_pre");
    return TU_OK;
}

// stack_w: bf16 (n_layers * 24 * 128, 64) weight slabs (the window stack's order per layer); stack_p: fp32 n_layers * 1792
// (c0 = 0 | ln1 w,b | in_proj bias (q part pre-scaled) | c1 = out_proj bias | ln2 w,b | fc1 bias | c_final = out_proj bias + fc2 bias)
int tc_resid_pre(const float *tok, bf16 *qkv, int M, int layer, int n_layers, const bf16 *stack_w, const float *stack_p, cudaStream_t st) {
    if (!g_rb_enable || !stack_w || !stack_p || (reinterpret_cast<uintptr_t>(stack_w) & 127) || (reinterpret_cast<uintptr_t>(tok) & 15) ||
        (reinterpret_cast<uintptr_t>(qkv) & 15))
        return TU_TC_UNSUPPORTED;
    ResidParams p;
    p.tok = const_cast<float *>(tok); p.tok16 = nullptr; p.qkv = qkv; p.att = nullptr;
    p.par = stack_p + (size_t)layer * PAR_FLOATS;
    p.M = M; p.n_tiles = ceil_div(M, 128); p.slab0 = layer * SLABS_PER_LAYER;
    return resid_launch(false, p, stack_w, n_layers, st);
}

int tc_resid_post(float *tok, bf16 *tok16, const bf16 *att, int M, int layer, int n_layers, const bf16 *stack_w, const float *stack_p,
                  cudaStream_t st) {
    if (!g_rb_enable || !stack_w || !stack_p || (reinterpret_cast<uintptr_t>(stack_w) & 127) || (reinterpret_cast<uintptr_t>(tok) & 15) ||
        (reinterpret_cast<uintptr_t>(att) & 15))
        return TU_TC_UNSUPPORTED;
    ResidParams p;
    p.tok = tok; p.tok16 = tok16; p.qkv = nullptr; p.att = att;
    p.par = stack_p + (size_t)layer * PAR_FLOATS;
    p.M = M; p.n_tiles = ceil_div(M, 128); p.slab0 = layer * SLABS_PER_LAYER + SLABS_PRE;
    return resid_launch(true, p, stack_w, n_layers, st);
}

}  // namespace tu
