// The whole window-transformer stack (all blocks) of WindowTransformer in ONE persistent kernel.
//
// Reference: the loop `for block in self.window_blocks: tokens_windows = block(tokens_windows)`
// (WindowTransformer/model.py:272-273) over WindowTransformerBlock (model.py:133-170) with WindowAttention
// (model.py:63-131).  Windows are never shifted, so a window's 64 tokens only ever interact with each other:
// a CTA takes 128 tokens (two windows) through all 8 blocks without touching HBM in between.
//
// On-chip data layout (dim = 128):
//   TMEM columns [0,128)   X: the fp32 residual stream, one TMEM lane per token.  proj and fc2 are issued with
//                          accumulate=1 straight onto X, so the two residual adds of a block cost nothing; their
//                          constant biases are folded into a running offset vector c that LayerNorm adds on read.
//   TMEM columns [128,384) two accumulator slots of 128 columns: q and k, then the fc1 chunks of the MLP.
//   TMEM columns [384,512) v's accumulators, then two HID buffers of 64 columns: GELU(fc1 chunk) as bf16 pairs, lane = token row --
//                          the A operand of fc2 straight from tensor memory (tcgen05.mma TS form).
//   smem A32  (32 KB)      LayerNorm output / attention output as a 128-byte-swizzled K-major UMMA A operand.
//   smem STG  (99 KB)      q,k,v of the 128 tokens in bf16 for the attention (mma.sync).
//   smem ring (5 x 16 KB)  weight slabs [128 n x 64 k] streamed by TMA in exactly the order the MMAs consume them
//                          (24 slabs = 384 KB per block, pre-packed on the host).
// Roles: warps 0-15 "math" (LN, epilogues, attention; thread = token row x column quarter: warp w may only touch TMEM
// lanes 32*(w%4).., so the four warps of a lane quadrant split the columns), warp 16 TMA producer, warp 17 MMA issuer
// + TMEM allocation.  Hand-offs are mbarriers: a_ready / a_half / g_ready (math -> MMA), acc[] (MMA -> math, one per commit point).
// DESIGN.md section 3.4 has the measured timeline of a block and the experiments that shaped this layout.
#include <cuda.h>

#include "ptx.cuh"
#include "stack_split.cuh"
#include "tc_api.cuh"

namespace tu {

namespace {

constexpr int DIM = 128, HEADS = 8, HID = 512;
constexpr int NMATH = 16;                        // math warps
constexpr int NUM_THREADS = (NMATH + 2) * 32;    // 576
constexpr int SLAB = 128 * 128;                 // 16 KB: 128 rows x 64 bf16
constexpr int NRING = 5;
constexpr int SLABS_PER_BLOCK = 24;
constexpr int STG_PITCH = 3 * DIM * 2 + 16;     // 784 B per token row (conflict-free fragment loads)
constexpr int OFF_A32 = 0;
constexpr int OFF_STG = 2 * SLAB;               // 32768
constexpr int STG_BYTES = 99 * 1024;            // >= 128 * 784 = 100352 and >= 4 slabs (HID)
constexpr int OFF_RING = OFF_STG + STG_BYTES;
constexpr int OFF_PAR = OFF_RING + NRING * SLAB;
constexpr int PAR_FLOATS = 1664;                // c0 | ln1w | ln1b | qkvb(384) | c1 | ln2w | ln2b | fc1b(512)
constexpr int OFF_STAT = OFF_PAR + PAR_FLOATS * 4;
constexpr int OFF_BAR = OFF_STAT + 2 * 128 * 4 * 8;      // two (sum, sumsq) tables: LN1 and LN2 alternate, so no barrier guards reuse
constexpr int SMEM_BYTES = OFF_BAR + 256 + 1024;
constexpr int P_C0 = 0, P_LN1W = 128, P_LN1B = 256, P_QKVB = 384, P_C1 = 768, P_LN2W = 896, P_LN2B = 1024, P_FC1B = 1152;

struct StackParams {
    float *tok;            // (M, 128) fp32 token stream, window-ordered; updated in place
    bf16 *tok16;           // optional bf16 copy of the result
    const float *par;      // nblocks * PAR_FLOATS + 128 (final offset vector)
    const float *rel_bias; // nblocks x (8, 4096) fp32 relative-position bias in mma C-fragment order (packing.py::frag_rel_bias)
    int n_tiles, n_blocks;
    int rev;               // token tiles are walked last to first (debug key "snake", bit 2)
    int var;               // debug variants (tu_debug_set("stack_var", mask))
    int *tile_flags;       // optional: tile_flags[t] = 1 once tile t's tokens are written and fenced (consumed by the unembed kernel)
    // Block-level work split (seg_flags != nullptr, zeroed by the caller): the n_tiles * n_blocks (tile, block) units are dealt out in
    // equal contiguous shares, so a CTA may take a tile through its first blocks only and hand the residual stream (raw TMEM X, fp32,
    // through the token buffer) to the next CTA, which continues it: 240 tiles x 8 blocks on 148 SMs = 13 units per SM instead of
    // two whole tiles (16).  seg_flags[t] = 1 once the first part of tile t is stored and fenced.
    int *seg_flags;
    int units_per_cta;
    unsigned long long *trace;      // debug (tu_debug_trace)
    unsigned int trace_cap;
};


// commit points of one block, in issue order: qkv column thirds, proj, then the MLP in four 128-column chunks of the hidden layer
// through two ACC slots and two HID buffers IN TENSOR MEMORY: fc1 chunks 0-1, then per chunk c {fc2 chunk c, fc1 chunk c + 2}.
// A part's epilogue starts while the MMAs of the next part are still running.
enum { ACC_QKV0 = 0, ACC_QKV1, ACC_QKV2, ACC_PROJ, ACC_FC1_0, ACC_FC1_1, ACC_FC1_2, ACC_FC1_3, ACC_FC2_3, NACC };

struct Barriers {
    uint64_t full[NRING], empty[NRING];
    uint64_t a_ready;
    uint64_t a_half;             // math -> MMA: attention output of heads 0-3 stored (its own barrier: no MMA result is awaited between
                                 // this arrival and the next one on a_ready, so a fast warp could otherwise arrive twice in one phase)
    uint64_t g_ready[2];         // math -> MMA: GELU(chunk c) stored in HID buffer c & 1 (alternating: consecutive chunks have no MMA
                                 // result between their arrivals)
    uint64_t acc[NACC];          // MMA -> math, one barrier per commit point of a block (each completes once per block)
    uint32_t tmem_base;
};

__device__ __forceinline__ void math_barrier() { asm volatile("bar.sync 1, 512;" ::: "memory"); }

__device__ __forceinline__ uint32_t pk(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t *>(&h);
}

// GELU(x) = x * Phi(x) with Phi(x) = 0.5 (1 + tanh(p(x))), p the odd polynomial fitted (minimax over |x| <= 8) to
// atanh(erf(x / sqrt 2)): |error| <= 2.6e-5 against the exact erf form in exact arithmetic, plus tanh.approx's 2^-11
// relative error -- both far below the bf16 resolution of the stored activation (tools/fit_gelu.py reproduces the fit).
__device__ __forceinline__ float gelu_fast(float x) {
    const float x2 = fminf(x * x, 64.f);            // beyond |x| = 8 the tanh is saturated; keeps p monotone
    float q = fmaf(-0.0003515167826820022f, x2, 0.03700564597780192f);
    q = fmaf(q, x2, 0.7975078843613885f);
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(x * q));
    const float h = 0.5f * x;
    return fmaf(h, t, h);
}

// ---- packed-fp32 (FFMA2 / FMUL2 / FADD2) forms of the element-wise math: same IEEE operations, half the issue slots
using ptx::f32x2;
// softmax: single-instruction exp2 / reciprocal (2 ulp; arguments are <= 0 resp. >= 1, the results are rounded to bf16)
__device__ __forceinline__ float ex2_fast(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_fast(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ uint32_t pk_pair(f32x2 v) {          // (lo, hi) -> bf16x2
    float lo, hi;
    ptx::up2(v, lo, hi);
    return pk(lo, hi);
}
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

__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// LayerNorm of this thread's 32 columns of row i (x already includes the folded bias offset); statistics are shared
// with the three partner threads holding the rest of the row; result -> A32 slab part/2, swizzled.
__device__ __forceinline__ void layernorm_to_a32(f32x2 (&x)[16], const float *gam, const float *bet, float2 *stat, uint8_t *a32,
                                                 int i, int part) {
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
    asm volatile("bar.sync %0, 128;" ::"r"(2 + (i >> 5)) : "memory");      // only the four warps holding this row's quarters
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
        f32x2 gm[4], bt[4];
        ptx::ld4(gam + ch * 8, gm[0], gm[1]); ptx::ld4(gam + ch * 8 + 4, gm[2], gm[3]);
        ptx::ld4(bet + ch * 8, bt[0], bt[1]); ptx::ld4(bet + ch * 8 + 4, bt[2], bt[3]);
#pragma unroll
        for (int e = 0; e < 4; ++e)      // ((x - mean) * rstd) * gamma + beta, two columns per instruction
            w[e] = pk_pair(ptx::fma2(ptx::mul2(ptx::add2(x[ch * 4 + e], nmean), rs), gm[e], bt[e]));
        uint4 u;
        u.x = w[0]; u.y = w[1]; u.z = w[2]; u.w = w[3];
        *reinterpret_cast<uint4 *>(rowp + ((((part & 1) * 4 + ch) ^ (i & 7)) << 4)) = u;
    }
}

__global__ void __launch_bounds__(NUM_THREADS, 1)
window_stack_kernel(const __grid_constant__ CUtensorMap tmap_w, const StackParams p) {
    pdl_trigger();
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem0 = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t *sm = smem_raw + (smem0 - ptx::smem_u32(smem_raw));
    Barriers *bars = reinterpret_cast<Barriers *>(sm + OFF_BAR);
    float *par = reinterpret_cast<float *>(sm + OFF_PAR);
    float2 *stat = reinterpret_cast<float2 *>(sm + OFF_STAT);
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // provably warp-uniform

    if (threadIdx.x == 0) {
        for (int i = 0; i < NRING; ++i) {
            ptx::mbar_init(ptx::smem_u32(&bars->full[i]), 1);
            ptx::mbar_init(ptx::smem_u32(&bars->empty[i]), 1);
        }
        ptx::mbar_init(ptx::smem_u32(&bars->a_ready), NMATH);
        ptx::mbar_init(ptx::smem_u32(&bars->a_half), NMATH);
        ptx::mbar_init(ptx::smem_u32(&bars->g_ready[0]), NMATH);
        ptx::mbar_init(ptx::smem_u32(&bars->g_ready[1]), NMATH);
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
    const uint32_t TX = tmem_base, TACC = tmem_base + 128, THID = tmem_base + 384;      // X 128 | ACC slots 2 x 128 | HID 2 x 64 (= third qkv slot)
    pdl_wait();

    if (warp == NMATH) {
        if (lane == 0) {
            // ================================ TMA producer: weight slabs in consumption order ================================
            int stage = 0;
            uint32_t phase = 0;
            Seg sg;
            for (int k = 0; get_seg(p.n_tiles, p.n_blocks, p.seg_flags != nullptr, p.units_per_cta, k, sg); ++k)
                for (int s = sg.lo * SLABS_PER_BLOCK; s < sg.hi * SLABS_PER_BLOCK; ++s) {
                    // packed order of the MLP slab pairs (packing.py): fc1 c0, fc1 c1, fc2 c0, fc2 c1, fc1 c2, fc1 c3, fc2 c2, fc2 c3;
                    // consumed as fc1 c0, fc1 c1, fc2 c0, fc1 c2, fc2 c1, fc1 c3, fc2 c2, fc2 c3
                    const int sb = s % SLABS_PER_BLOCK;
                    int src = s;
                    if (sb >= 8) src = s - sb + 8 + ((0x76534210u >> (((sb - 8) >> 1) * 4)) & 7) * 2 + (sb & 1);
                    ptx::mbar_wait(ptx::smem_u32(&bars->empty[stage]), phase ^ 1);
                    const uint32_t fb = ptx::smem_u32(&bars->full[stage]);
                    ptx::mbar_expect_tx(fb, SLAB);
                    ptx::tma_load_2d(smem0 + OFF_RING + stage * SLAB, &tmap_w, fb, 0, src * 128);
                    if (++stage == NRING) { stage = 0; phase ^= 1; }
                }
        }
    } else if (warp == NMATH + 1) {
        // ================================ MMA issuer (whole warp converged, elected lane issues) ================================
        const uint32_t leader = ptx::elect_one();
        const uint32_t idesc = ptx::make_idesc_bf16(128, 128);
        const uint32_t ring_lo = ptx::sdesc_lo(smem0 + OFF_RING);
        int stage = 0;
        uint32_t phase = 0, aph = 0, hph = 0, gph = 0;
        // one weight slab: D[128 x 128] (+)= A_slab[128 x 64] * W_slab[128 x 64]^T
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
        const uint32_t a32 = ptx::sdesc_lo(smem0 + OFF_A32);
        constexpr uint32_t SL = SLAB >> 4;
        Seg sg;
        for (int k = 0; get_seg(p.n_tiles, p.n_blocks, p.seg_flags != nullptr, p.units_per_cta, k, sg); ++k)
            for (int bk = sg.lo; bk < sg.hi; ++bk) {
                wait_a();                                       // LN1 output in A32
                for (int nc = 0; nc < 3; ++nc) {
                    for (int ks = 0; ks < 2; ++ks) slab_mma(TACC + nc * 128, a32 + ks * SL, ks == 0);
                    ptx::umma_commit_pred(ptx::smem_u32(&bars->acc[ACC_QKV0 + nc]), leader);
                }
                ptx::mbar_wait(ptx::smem_u32(&bars->a_half), hph);      // attention output of heads 0-3 in A32 K-slab 0
                hph ^= 1;
                ptx::tc_fence_after();
                slab_mma(TX, a32, false);                       // x += att Wp^T, first K half
                wait_a();                                       // heads 4-7 in K-slab 1
                slab_mma(TX, a32 + SL, false);
                ptx::umma_commit_pred(ptx::smem_u32(&bars->acc[ACC_PROJ]), leader);
                wait_a();                                       // LN2 output in A32
                for (int c = 0; c < 2; ++c) {                   // fc1 chunks 0, 1 into the two ACC slots
                    for (int ks = 0; ks < 2; ++ks) slab_mma(TACC + c * 128, a32 + ks * SL, ks == 0);
                    ptx::umma_commit_pred(ptx::smem_u32(&bars->acc[ACC_FC1_0 + c]), leader);
                }
                for (int c = 0; c < 4; ++c) {
                    ptx::mbar_wait(ptx::smem_u32(&bars->g_ready[c & 1]), (gph >> (c & 1)) & 1);       // GELU(chunk c) in HID buffer c & 1
                    gph ^= 1u << (c & 1);
                    ptx::tc_fence_after();
                    // x += h_c W2[:, chunk c]^T with the A operand in TENSOR MEMORY (lane = token row, one column = two consecutive hidden
                    // units as a bf16 pair): the MMA reads only the weight slab from shared memory, half the port load of the SS form
                    for (int ks = 0; ks < 2; ++ks) {
                        ptx::mbar_wait(ptx::smem_u32(&bars->full[stage]), phase);
                        ptx::tc_fence_after();
                        const uint32_t w_lo = ring_lo + ((stage * SLAB) >> 4);
#pragma unroll
                        for (int k4 = 0; k4 < 4; ++k4)
                            ptx::umma_bf16_ts_lo<1>(TX, THID + (c & 1) * 64 + ks * 32 + k4 * 8, w_lo + k4 * 2, idesc, leader);
                        ptx::umma_commit_pred(ptx::smem_u32(&bars->empty[stage]), leader);
                        if (++stage == NRING) { stage = 0; phase ^= 1; }
                    }
                    if (c + 2 < 4) {                            // ACC slot c & 1 is drained: fc1 chunk c + 2
                        for (int ks = 0; ks < 2; ++ks) slab_mma(TACC + (c & 1) * 128, a32 + ks * SL, ks == 0);
                        ptx::umma_commit_pred(ptx::smem_u32(&bars->acc[ACC_FC1_0 + c + 2]), leader);      // (also: fc2 of chunk c has read HID buffer c & 1)
                    }
                }
                ptx::umma_commit_pred(ptx::smem_u32(&bars->acc[ACC_FC2_3]), leader);
            }
    } else {
        // ================================ math warps ================================
        const int q = warp & 3, part = warp >> 2;           // TMEM lane quadrant, column quarter
        const int i = q * 32 + lane;                        // token row of the tile == TMEM lane
        const uint32_t lane_base = (uint32_t)(q * 32) << 16;
        const int mt = threadIdx.x;                          // 0..511
        uint8_t *a32 = sm + OFF_A32, *stg = sm + OFF_STG;
        uint32_t cph = 0;             // every acc barrier completes exactly once per block: one shared phase bit
        auto wait_acc = [&](int which) {
            ptx::mbar_wait(ptx::smem_u32(&bars->acc[which]), cph);
            ptx::tc_fence_after();
        };
        auto signal_a = [&]() {       // every thread orders its own writes, one lane per warp arrives
            ptx::fence_proxy_async();
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(ptx::smem_u32(&bars->a_ready));
        };
        // x row quarter (+ offset vector) -> registers
        auto load_x = [&](f32x2 (&x)[16], const float *cvec) {
            uint32_t v[32];
            ptx::tmem_ld_x32(TX + lane_base + part * 32, v);
            ptx::tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 16; j += 2) {
                f32x2 c0v, c1v;
                ptx::ld4(cvec + part * 32 + 2 * j, c0v, c1v);
                x[j] = ptx::add2(ptx::pk2u(v[2 * j], v[2 * j + 1]), c0v);
                x[j + 1] = ptx::add2(ptx::pk2u(v[2 * j + 2], v[2 * j + 3]), c1v);
            }
        };

        Seg sg;
        int tr_t = 0, tr_b = 0;
        auto phase_ev = [&](int ph) {      // debug (tu_debug_trace): phase boundaries of warps 0 and 15
            if (p.trace && (mt == 0 || mt == 480)) trace_event(p.trace, p.trace_cap, mt == 0 ? 10 : 11, (unsigned)(tr_t * 256 + tr_b * 16 + ph));
        };
        for (int k = 0; get_seg(p.n_tiles, p.n_blocks, p.seg_flags != nullptr, p.units_per_cta, k, sg); ++k) {
            const int t = p.rev ? p.n_tiles - 1 - sg.tile : sg.tile;
            tr_t = t;
            if (sg.lo > 0) {          // the CTA that ran blocks [0, lo) of this tile has stored and fenced the raw residual stream
                if (mt == 0) wait_flag_acquire(p.seg_flags + t);
                math_barrier();
            }
            if (mt == 0) trace_event(p.trace, p.trace_cap, 1, (unsigned)t);          // tile begins
            // ---- tokens (or the raw residual stream of a tile in progress) -> TMEM X
            {
                const float *src = p.tok + ((long)t * 128 + i) * DIM + part * 32;
                uint32_t v[32];
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    const float4 f = __ldcg(reinterpret_cast<const float4 *>(src + j));
                    v[j] = __float_as_uint(f.x); v[j + 1] = __float_as_uint(f.y); v[j + 2] = __float_as_uint(f.z); v[j + 3] = __float_as_uint(f.w);
                }
                ptx::tmem_st_x32(TX + lane_base + part * 32, v);
                ptx::tmem_st_wait();
                ptx::tc_fence_before();
            }
            // per-block parameters -> smem: the first block's here, the next block's while the last fc2 of a block runs
            auto load_params = [&](int bk) {
                math_barrier();       // everyone is done with the previous parameters
                const float4 *g = reinterpret_cast<const float4 *>(p.par + (long)bk * PAR_FLOATS);
                float4 *d = reinterpret_cast<float4 *>(par);
                for (int e = mt; e < PAR_FLOATS / 4; e += NMATH * 32) d[e] = g[e];
            };
            load_params(sg.lo);
            for (int bk = sg.lo; bk < sg.hi; ++bk) {
                math_barrier();       // parameters (and the X stores of a new tile) are visible
                ptx::tc_fence_after();
                tr_b = bk;
                phase_ev(0);
                // relative-position bias of this thread's 2 rows x 16 columns: a warp's four attention tasks are (head hw, window 0),
                // (hw, window 1), (hw + 4, window 0), (hw + 4, window 1) with the same 16-row group, so two fetches serve four tasks;
                // the first is issued here, before LayerNorm (64 KB per SM: half a microsecond of the SM's L2 read path, which
                // delays everything else that returns through it -- issued next to the qkv MMAs it held up their completion wait), the second right after the first's last use
                // (fragment order, packing.py::frag_rel_bias: one coalesced 16-byte load per lane and key octet -- the dense layout cost
                // sixteen 8-byte loads per lane, each warp instruction touching eight cache lines: ~1.3 us per block of L1 tag lookups)
                const ulonglong2 *relb = reinterpret_cast<const ulonglong2 *>(p.rel_bias) + (long)bk * HEADS * 1024;
                f32x2 ba[8], bb[8];
                auto load_bias = [&](int h) {
                    const ulonglong2 *bp = relb + (h * 4 + (warp & 3)) * 256 + lane;
#pragma unroll
                    for (int n = 0; n < 8; ++n) {
                        const ulonglong2 v = __ldg(bp + n * 32);
                        ba[n] = v.x;
                        bb[n] = v.y;
                    }
                };
                if (!(p.var & 1)) load_bias(warp >> 2);
                // ---- LN1(x + c0) -> A32
                {
                    f32x2 x[16];
                    load_x(x, par + P_C0);
                    layernorm_to_a32(x, par + P_LN1W + part * 32, par + P_LN1B + part * 32, stat, a32, i, part);
                }
                signal_a();
                phase_ev(1);
                // ---- qkv epilogue: ACC -> (+bias) -> bf16 staging rows, one column third at a time as its MMAs retire
                {
                    uint8_t *rowp = stg + i * STG_PITCH;
#pragma unroll
                    for (int nc = 0; nc < 3; ++nc) {
                        wait_acc(ACC_QKV0 + nc);
                        if (nc == 0) { phase_ev(2); if (p.var & 1) load_bias(warp >> 2); }
                        uint32_t v[32];
                        const int col = nc * 128 + part * 32;
                        ptx::tmem_ld_x32(TACC + lane_base + col, v);
                        ptx::tmem_ld_wait();
                        const float *qb = par + P_QKVB + col;
#pragma unroll
                        for (int j = 0; j < 32; j += 8) {
                            uint4 u;
                            f32x2 b0v, b1v, b2v, b3v;
                            ptx::ld4(qb + j, b0v, b1v); ptx::ld4(qb + j + 4, b2v, b3v);
                            u.x = pk_pair(ptx::add2(ptx::pk2u(v[j + 0], v[j + 1]), b0v));
                            u.y = pk_pair(ptx::add2(ptx::pk2u(v[j + 2], v[j + 3]), b1v));
                            u.z = pk_pair(ptx::add2(ptx::pk2u(v[j + 4], v[j + 5]), b2v));
                            u.w = pk_pair(ptx::add2(ptx::pk2u(v[j + 6], v[j + 7]), b3v));
                            *reinterpret_cast<uint4 *>(rowp + (col + j) * 2) = u;
                        }
                    }
                }
                math_barrier();
                phase_ev(3);
                // ---- window attention: 2 windows x 8 heads x 4 row groups = 64 warp tasks, 4 per warp
                {
                    const int g = lane >> 2, tq = lane & 3;
#pragma unroll 1
                    for (int tk = 0; tk < 4; ++tk) {
                        const int win = tk & 1, h = (warp >> 2) + 4 * (tk >> 1), rg = warp & 3;
                        const uint8_t *wbase = stg + (win * 64) * STG_PITCH;
                        const int r0 = rg * 16 + g;
                        uint32_t qa[4];
                        qa[0] = *reinterpret_cast<const uint32_t *>(wbase + r0 * STG_PITCH + (h * 16 + tq * 2) * 2);
                        qa[1] = *reinterpret_cast<const uint32_t *>(wbase + (r0 + 8) * STG_PITCH + (h * 16 + tq * 2) * 2);
                        qa[2] = *reinterpret_cast<const uint32_t *>(wbase + r0 * STG_PITCH + (h * 16 + tq * 2 + 8) * 2);
                        qa[3] = *reinterpret_cast<const uint32_t *>(wbase + (r0 + 8) * STG_PITCH + (h * 16 + tq * 2 + 8) * 2);
                        float s[8][4];
#pragma unroll
                        for (int n = 0; n < 8; ++n) {
                            const uint8_t *kp = wbase + (n * 8 + g) * STG_PITCH + (DIM + h * 16 + tq * 2) * 2;
                            const uint32_t b0 = *reinterpret_cast<const uint32_t *>(kp), b1 = *reinterpret_cast<const uint32_t *>(kp + 16);
                            ptx::up2(ba[n], s[n][0], s[n][1]);          // accumulators start at the relative-position bias
                            ptx::up2(bb[n], s[n][2], s[n][3]);
                            mma16816(s[n], qa, b0, b1);
                        }
                        float m0 = -INFINITY, m1 = -INFINITY;
                        f32x2 sa[8], sb[8];                       // (row r0: columns c, c+1), (row r0 + 8: columns c, c+1)
#pragma unroll
                        for (int n = 0; n < 8; ++n) {
                            sa[n] = ptx::pk2(s[n][0], s[n][1]);
                            sb[n] = ptx::pk2(s[n][2], s[n][3]);
                            m0 = fmaxf(m0, fmaxf(s[n][0], s[n][1]));
                            m1 = fmaxf(m1, fmaxf(s[n][2], s[n][3]));
                        }
                        if (tk == 1) load_bias((warp >> 2) + 4);       // the second head's bias flies during this task's softmax and PV
                        if (tk == 2) {                                 // heads 0-3 of both windows are in A32 K-slab 0: proj starts on it
                            ptx::fence_proxy_async();
                            ptx::tc_fence_before();
                            __syncwarp();
                            if (lane == 0) ptx::mbar_arrive(ptx::smem_u32(&bars->a_half));
                        }
                        m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1)); m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 2));
                        m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1)); m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 2));
                        const float L2E = 1.4426950408889634f;
                        const float mm0 = m0 * L2E, mm1 = m1 * L2E;
                        const f32x2 l2e2 = ptx::pk2(L2E, L2E), nm0 = ptx::pk2(-mm0, -mm0), nm1 = ptx::pk2(-mm1, -mm1);
#pragma unroll
                        for (int n = 0; n < 8; ++n) {
                            float e0, e1, e2, e3;
                            ptx::up2(ptx::fma2(sa[n], l2e2, nm0), e0, e1);
                            ptx::up2(ptx::fma2(sb[n], l2e2, nm1), e2, e3);
                            s[n][0] = ex2_fast(e0); s[n][1] = ex2_fast(e1);
                            s[n][2] = ex2_fast(e2); s[n][3] = ex2_fast(e3);
                        }
                        // row sums come from the tensor core as well: P times a column of ones (exactly the bf16 probabilities PV uses,
                        // summed in fp32; every column of the result holds the row sum, so no shuffles)
                        float ls[4] = {0.f, 0.f, 0.f, 0.f};
                        float o[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
#pragma unroll
                        for (int kt = 0; kt < 4; ++kt) {
                            uint32_t pa[4];
                            pa[0] = pk(s[2 * kt][0], s[2 * kt][1]);
                            pa[1] = pk(s[2 * kt][2], s[2 * kt][3]);
                            pa[2] = pk(s[2 * kt + 1][0], s[2 * kt + 1][1]);
                            pa[3] = pk(s[2 * kt + 1][2], s[2 * kt + 1][3]);
                            uint32_t v0, v1, v2, v3;
                            const uint32_t addr = ptx::smem_u32(wbase + (kt * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * STG_PITCH +
                                                                (2 * DIM + h * 16 + (lane >> 4) * 8) * 2);
                            asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                                         : "=r"(v0), "=r"(v1), "=r"(v2), "=r"(v3)
                                         : "r"(addr));
                            mma16816(o[0], pa, v0, v1);
                            mma16816(o[1], pa, v2, v3);
                            mma16816(ls, pa, 0x3f803f80u, 0x3f803f80u);
                        }
                        const float i0 = rcp_fast(ls[0]), i1 = rcp_fast(ls[2]);      // l >= 1: the row maximum contributes exp2(0)
                        // attention output -> A32 (row = token of the tile, column = h*16 + d), swizzled
                        const int row0 = win * 64 + r0, row1 = row0 + 8;
#pragma unroll
                        for (int nt = 0; nt < 2; ++nt) {
                            const int col = h * 16 + nt * 8 + tq * 2;
                            const int ks = col >> 6, ch = (col & 63) >> 3, bo = (col & 7) * 2;
                            *reinterpret_cast<uint32_t *>(a32 + ks * SLAB + row0 * 128 + ((ch ^ (row0 & 7)) << 4) + bo) = pk_pair(ptx::mul2(ptx::pk2(o[nt][0], o[nt][1]), ptx::pk2(i0, i0)));
                            *reinterpret_cast<uint32_t *>(a32 + ks * SLAB + row1 * 128 + ((ch ^ (row1 & 7)) << 4) + bo) = pk_pair(ptx::mul2(ptx::pk2(o[nt][2], o[nt][3]), ptx::pk2(i1, i1)));
                        }
                    }
                }
                signal_a();
                phase_ev(4);
                // ---- LN2(x + c1) -> A32 (after proj has been accumulated onto X)
                wait_acc(ACC_PROJ);
                phase_ev(5);
                {
                    f32x2 x[16];
                    load_x(x, par + P_C1);
                    layernorm_to_a32(x, par + P_LN2W + part * 32, par + P_LN2B + part * 32, stat + 128 * 4, a32, i, part);
                }
                signal_a();
                phase_ev(6);
                // ---- MLP: four 128-column chunks of the hidden layer: ACC slot c & 1 -> +bias -> GELU -> bf16 pairs into HID buffer c & 1
                // in tensor memory (tcgen05.st: no swizzle arithmetic, no proxy fence, no shared-memory traffic).  fc1 of chunk c + 2 is
                // committed behind fc2 of chunk c, so its arrival also frees the HID buffer this chunk writes.
#pragma unroll 1
                for (int c = 0; c < 4; ++c) {
                    wait_acc(ACC_FC1_0 + c);
                    if (c == 0) phase_ev(7);
                    uint32_t v[32];
                    ptx::tmem_ld_x32(TACC + lane_base + (c & 1) * 128 + part * 32, v);
                    ptx::tmem_ld_wait();
                    const float *bb = par + P_FC1B + c * 128 + part * 32;
#pragma unroll
                    for (int j = 0; j < 32; j += 8) {
                        f32x2 b0v, b1v, b2v, b3v;
                        ptx::ld4(bb + j, b0v, b1v); ptx::ld4(bb + j + 4, b2v, b3v);
                        const uint32_t h0 = pk_pair(gelu_fast2(ptx::add2(ptx::pk2u(v[j + 0], v[j + 1]), b0v)));
                        const uint32_t h1 = pk_pair(gelu_fast2(ptx::add2(ptx::pk2u(v[j + 2], v[j + 3]), b1v)));
                        const uint32_t h2 = pk_pair(gelu_fast2(ptx::add2(ptx::pk2u(v[j + 4], v[j + 5]), b2v)));
                        const uint32_t h3 = pk_pair(gelu_fast2(ptx::add2(ptx::pk2u(v[j + 6], v[j + 7]), b3v)));
                        ptx::tmem_st_x4(THID + lane_base + (c & 1) * 64 + part * 16 + j / 2, h0, h1, h2, h3);
                    }
                    ptx::tmem_st_wait();
                    ptx::tc_fence_before();
                    __syncwarp();
                    if (lane == 0) ptx::mbar_arrive(ptx::smem_u32(&bars->g_ready[c & 1]));
                    phase_ev(8 + c);
                }
                if (bk + 1 < sg.hi) load_params(bk + 1);
                wait_acc(ACC_FC2_3);      // the last fc2 is accumulated: X holds the block output (minus folded biases)
                phase_ev(12);
                cph ^= 1;
            }
            if (sg.hi < p.n_blocks) {
                // ---- tile in progress: raw X -> global (the folded bias offsets are NOT applied: the next CTA continues exactly here)
                float *dst = p.tok + ((long)t * 128 + i) * DIM + part * 32;
                uint32_t v[32];
                ptx::tmem_ld_x32(TX + lane_base + part * 32, v);
                ptx::tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 32; j += 4)
                    *reinterpret_cast<float4 *>(dst + j) = make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
                ptx::tc_fence_before();
                __threadfence();
                math_barrier();
                if (mt == 0) atomicExch(p.seg_flags + t, 1);
                continue;
            }
            // ---- X (+ final offset) -> global
            {
                const float *cfin = p.par + (long)p.n_blocks * PAR_FLOATS + part * 32;
                float *dst = p.tok + ((long)t * 128 + i) * DIM + part * 32;
                bf16 *dst16 = p.tok16 ? p.tok16 + ((long)t * 128 + i) * DIM + part * 32 : nullptr;
                uint32_t v[32];
                ptx::tmem_ld_x32(TX + lane_base + part * 32, v);
                ptx::tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    float4 f;
                    f.x = __uint_as_float(v[j]) + __ldg(cfin + j);
                    f.y = __uint_as_float(v[j + 1]) + __ldg(cfin + j + 1);
                    f.z = __uint_as_float(v[j + 2]) + __ldg(cfin + j + 2);
                    f.w = __uint_as_float(v[j + 3]) + __ldg(cfin + j + 3);
                    *reinterpret_cast<float4 *>(dst + j) = f;
                    if (dst16) {
                        uint2 u;
                        u.x = pk(f.x, f.y); u.y = pk(f.z, f.w);
                        *reinterpret_cast<uint2 *>(dst16 + j) = u;
                    }
                }
                ptx::tc_fence_before();
                if (p.tile_flags) {       // publish the tile: every thread fences its own stores, then one thread raises the flag
                    __threadfence();
                    math_barrier();
                    if (mt == 0) atomicExch(p.tile_flags + t, 1);
                }
                if (mt == 0) trace_event(p.trace, p.trace_cap, 2, (unsigned)t);      // tile stored (and published)
            }
        }
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == NMATH + 1) ptx::tmem_dealloc(tmem_base, 512);
}

PerDeviceFlag g_attr_set;
thread_local int g_stack_var = 0;
thread_local int g_stack_split = 0;       // measured (profiles/r05c_ab.log): 342 -> 290 us serialised, but inside a forward the unembed overlap already uses
                             // the SMs the whole-tile schedule leaves idle: 1.2605 -> 1.2637 ms (dim 128), 2.0515 -> 2.0694 ms (dim 192)

}  // namespace

void tc_set_stack_split(int on) { g_stack_split = on; }
void tc_set_stack_var(int mask) { g_stack_var = mask; }
int tc_stack_var() { return g_stack_var; }
bool tc_stack_split_enabled() { return g_stack_split != 0; }

// stack_w: bf16 (n_blocks * 24 * 128, 64) weight slabs in consumption order; stack_p: fp32 n_blocks*1664 + 128;
// rel_bias: fp32 n_blocks x (8,4096) in fragment order.  tok: (M,128) fp32 with M % 128 == 0.
int tc_window_stack(float *tok, bf16 *tok16, int M, int n_blocks, const bf16 *stack_w, const float *stack_p,
                    const float *rel_bias, int *tile_flags, int *seg_flags, cudaStream_t st) {
    TcEncodeFn enc = tc_encode_fn();
    if (!enc || !stack_w || !stack_p || !rel_bias || (M % 128) || (reinterpret_cast<uintptr_t>(stack_w) & 127) ||
        (reinterpret_cast<uintptr_t>(tok) & 15))
        return TU_TC_UNSUPPORTED;
    const int g_sm_count = device_sm_count();
    if (!g_attr_set.is_set()) {
        cudaError_t e = cudaFuncSetAttribute(window_stack_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
        if (e != cudaSuccess) return cuda_fail(e, "window_stack smem attribute");
        g_attr_set.set();
    }
    CUtensorMap tw;
    cuuint64_t wd[2] = {64, (cuuint64_t)n_blocks * SLABS_PER_BLOCK * 128}, ws[1] = {128};
    cuuint32_t wb[2] = {64, 128}, we[2] = {1, 1};
    CUresult r = enc(&tw, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void *)stack_w, wd, ws, wb, we, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("tu: cuTensorMapEncodeTiled(window stack weights) failed with code " + std::to_string((int)r));
        return TU_ERR_CUDA;
    }
    StackParams p;
    p.tok = tok; p.tok16 = tok16; p.par = stack_p; p.rel_bias = rel_bias;
    p.n_tiles = M / 128; p.n_blocks = n_blocks; p.tile_flags = tile_flags;
    p.rev = (g_snake_mask >> 2) & 1;
    p.var = g_stack_var;
    p.trace = g_trace_buf; p.trace_cap = g_trace_cap;
    const int grid = p.n_tiles < g_sm_count ? p.n_tiles : g_sm_count;
    // split tiles between CTAs at block boundaries only when whole tiles do not divide evenly (and the caller provided flags)
    p.seg_flags = (seg_flags && g_stack_split && p.n_tiles % grid != 0) ? seg_flags : nullptr;
    p.units_per_cta = ceil_div(p.n_tiles * n_blocks, grid);
    launch_pdl(window_stack_kernel, dim3(grid), dim3(NUM_THREADS), SMEM_BYTES, st, tw, p);
    TU_CHECK_LAUNCH("window_stack");
    return TU_OK;
}

}  // namespace tu
