// The whole window-transformer stack of FastTransformer (dim 192, 12 heads, hidden 768) in ONE persistent kernel.
//
// Reference: `for block in self.window_blocks: tokens_windows = block(tokens_windows)` (FastTransformer/model.py:288-289) over
// WindowTransformerBlock (model.py:135-172) with WindowAttention (model.py:65-133).  Same idea as window_stack_tcgen05.cu
// (dim 128): windows are never shifted, so a CTA takes 128 tokens (two windows) through all blocks on-chip.  With dim 192
// neither the qkv activations (128 x 576) nor an MLP half fit beside the residual stream, so the block is cut finer:
//
//   TMEM columns [0,192)    X: fp32 residual stream (one lane per token); proj and fc2 accumulate straight onto it, their
//                           biases folded into offset vectors added on read (c0 before LN1, c1 before LN2, c_final at the end)
//   TMEM columns [192,448)  two accumulator slots of 128 columns: one qkv head-group (96 columns) at a time, then the fc1 chunks
//   TMEM columns [448,512)  HID of the even MLP chunks: GELU(fc1 chunk) as bf16 pairs, the A operand of fc2 in tensor memory
//   smem A32  (48 KB)       LayerNorm output: three 128 x 64 swizzled K-slabs (A operand of qkv and fc1)
//   smem AO   (48 KB)       attention output (A operand of proj); later its first 32 KB hold HID of the odd MLP chunks
//   smem STG  (27 KB)       q | k | v (32 + 32 + 32 columns, bf16) of the CURRENT group of two heads, 128 token rows
//   smem ring (84 KB)       weight slabs streamed by TMA in consumption order (packing.py), packed back to back (byte-granular ring,
//                           layout planned on the host: plan_ring): per block 18 slabs [96 n x 64 k] (qkv: 6 head-groups x 3 K-slabs,
//                           rows q|k|v of the group), 3 slabs [192 n x 64 k] (proj), then the MLP in six chunks of 128 hidden units:
//                           fc1 chunk = 3 slabs [128 n x 64 k], fc2 chunk = 2 slabs [192 n x 64 k]; order fc1 c0, fc1 c1, then per
//                           chunk c: fc2 c, fc1 c+2
// Head-group pipeline: the qkv MMAs of group g+1 run while the math warps do the attention of group g (one (window, head,
// 16-row) task per warp: mma.sync QK^T seeded with the bias, softmax, PV and the row sums on the tensor core).
// Roles: warps 0-15 math (thread = token row x column quarter), warp 16 TMA producer, warp 17 MMA issuer + TMEM allocation.
// DESIGN.md section 3.4 has the measured timeline of a block.
#include <cuda.h>

#include "ptx.cuh"
#include "stack_split.cuh"
#include "tc_api.cuh"

namespace tu {

namespace {

constexpr int DIM = 192, HEADS = 12, HID = 768;
constexpr int NGROUP = 6, NCHUNK = 6;               // qkv head groups; MLP chunks of 128 hidden units
constexpr int NMATH = 16;
constexpr int NUM_THREADS = (NMATH + 2) * 32;     // 576
constexpr int SLAB_A = 128 * 128;                 // activation K-slab: 128 rows x 64 bf16
constexpr int SLAB_W = 192 * 128;                 // weight slab slot: up to 192 rows x 64 bf16
constexpr int NRING = 8;                          // weight slabs in flight at most (barrier pairs)
constexpr int RING_BYTES = 84 * 1024;             // byte-granular weight ring: slabs of 12 / 16 / 24 KB are packed back to back
constexpr int STG_PITCH = 96 * 2 + 16;            // 208 B per token row (conflict-free fragment loads)
constexpr int OFF_A32 = 0;
constexpr int OFF_AO = 3 * SLAB_A;                // 49152
constexpr int OFF_STG = OFF_AO + 3 * SLAB_A;      // 98304
constexpr int STG_BYTES = 27 * 1024;              // >= 128 * 208 = 26624
constexpr int OFF_RING = OFF_STG + STG_BYTES;     // 125952 = 123 * 1024
constexpr int OFF_PAR = OFF_RING + RING_BYTES;
constexpr int PAR_FLOATS = 2496;                  // c0 | ln1w | ln1b | qkvb(576, group-major) | c1 | ln2w | ln2b | fc1b(768)
constexpr int P_C0 = 0, P_LN1W = 192, P_LN1B = 384, P_QKVB = 576, P_C1 = 1152, P_LN2W = 1344, P_LN2B = 1536, P_FC1B = 1728;
constexpr int OFF_STAT = OFF_PAR + PAR_FLOATS * 4;
constexpr int OFF_BAR = OFF_STAT + 2 * 128 * 4 * 8;
constexpr int SMEM_BYTES = OFF_BAR + 384 + 1024;
static_assert(SMEM_BYTES <= 232448 && OFF_RING % 1024 == 0, "shared memory layout");
constexpr int SLABS96 = NGROUP * 3;                                  // qkv: 18 slabs of 96 rows
constexpr int SLABS_PER_BLOCK = SLABS96 + 3 + NCHUNK * 5;            // + proj 3 x 192 rows + per MLP chunk fc1 3 x 128 rows and fc2 2 x 192 rows = 51
constexpr int ROWS_PER_BLOCK = SLABS96 * 96 + 3 * 192 + NCHUNK * (3 * 128 + 2 * 192);       // 6912 rows of 64 bf16
// rows of the s-th slab of a block in consumption order (packing.py::_pack_fused_stack192): qkv, proj, fc1 c0, fc1 c1, then per
// chunk c: fc2 c (2 slabs), fc1 c + 2 (3 slabs, c < 4)
__device__ __forceinline__ int slab_rows(int s) {
    if (s < SLABS96) return 96;
    if (s < SLABS96 + 3) return 192;
    if (s < SLABS96 + 9) return 128;
    const int t = s - (SLABS96 + 9);
    return (t >= 20 || t % 5 < 2) ? 192 : 128;
}

// Byte-granular weight ring.  Slab n of `bytes` goes to the current head, or to offset 0 when it would not fit before the end of the
// ring (the tail stays unused for that lap); every block starts at offset 0 again, so the layout is the same for all blocks and the
// host can tell the producer which older slabs each load overwrites (plan_ring).
struct RingPos {
    int head = 0;
    __device__ __forceinline__ int place(int bytes) {
        if (head + bytes > RING_BYTES) head = 0;
        const int off = head;
        head += bytes;
        return off;
    }
};

enum { ACC_QKV0 = 0, ACC_PROJ = NGROUP, ACC_FC1_0, ACC_FC2L = ACC_FC1_0 + NCHUNK, NACC };

struct Stack192Params {
    float *tok;            // (M, 192) fp32 token stream, window-ordered; updated in place
    bf16 *tok16;           // optional bf16 copy of the result
    const float *par;      // nblocks * PAR_FLOATS + 192 (final offset vector)
    const float *rel_bias; // nblocks x (12, 4096) fp32 relative-position bias in mma C-fragment order (packing.py::frag_rel_bias)
    int n_tiles, n_blocks;
    int *tile_flags;       // optional: tile_flags[t] = 1 once tile t's tokens are written and fenced (consumed by the unembed kernel)
    int *seg_flags;        // optional: block-level work split (stack_split.cuh); seg_flags[t] = 1 once the first part of tile t is stored
    int units_per_cta;
    int var;               // debug variants (tu_debug_set("stack_var", mask)); none at the moment
    // byte-granular weight ring, the same for every block (the ring restarts at offset 0 with a block's first slab): offset of slab s
    // in KB, and the newest slab -- index relative to the block, negative = a slab of the previous block -- that must have been released
    // before slab s may be loaded (computed on the host: plan_ring)
    unsigned char w_off[64];
    signed char w_need[64];
    unsigned long long *trace;      // debug (tu_debug_trace)
    unsigned int trace_cap;
};

struct Barriers {
    uint64_t full[NRING], empty[NRING];
    uint64_t a_ready;
    uint64_t g_ready[2];         // math -> MMA: GELU(chunk c) stored in HID buffer c & 1
    uint64_t acc[NACC];
    uint32_t tmem_base;
};
static_assert(sizeof(Barriers) <= 384, "barrier block too large");

__device__ __forceinline__ void math_barrier() { asm volatile("bar.sync 1, 512;" ::: "memory"); }

__device__ __forceinline__ uint32_t pk(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t *>(&h);
}

// same fitted GELU as window_stack_tcgen05.cu (tools/fit_gelu.py)
__device__ __forceinline__ float gelu_fast(float x) {
    const float x2 = fminf(x * x, 64.f);
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

// 48 consecutive TMEM columns of this thread's lane -> registers (32 + 16)
__device__ __forceinline__ void tmem_ld48(uint32_t taddr, uint32_t (&v)[48]) {
    uint32_t a[32], b[16];
    ptx::tmem_ld_x32(taddr, a);
    ptx::tmem_ld_x16(taddr + 32, b);
    ptx::tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = a[j];
#pragma unroll
    for (int j = 0; j < 16; ++j) v[32 + j] = b[j];
}

// byte offset of the 16-byte chunk holding columns [col, col+8) of row i inside a stack of swizzled 128 x 64 K-slabs
__device__ __forceinline__ int slab_chunk_off(int col, int i) { return (col >> 6) * SLAB_A + i * 128 + ((((col & 63) >> 3) ^ (i & 7)) << 4); }

// LayerNorm of this thread's 48 columns of row i (x already includes the folded offset) -> A32, swizzled
__device__ __forceinline__ void layernorm_to_a32(f32x2 (&x)[24], const float *gam, const float *bet, float2 *stat, uint8_t *a32, int i,
                                                 int part) {
    // one exchange: every thread publishes the mean and M2 = sum (x - mean)^2 of its own 48 columns (two passes over registers);
    // Chan's combination M2 = sum M2_p + 48 sum (mean_p - mean)^2 keeps the variance exact for rows whose channels share an offset
    // far above their spread, where E[x^2] - mean^2 in fp32 cancels away
    f32x2 s2 = ptx::pk2(0.f, 0.f), q2 = ptx::pk2(0.f, 0.f);
#pragma unroll
    for (int j = 0; j < 24; ++j) s2 = ptx::add2(s2, x[j]);
    float s_lo, s_hi, q_lo, q_hi;
    ptx::up2(s2, s_lo, s_hi);
    const float pmean = (s_lo + s_hi) * (1.0f / 48);
    const f32x2 npm = ptx::pk2(-pmean, -pmean);
#pragma unroll
    for (int j = 0; j < 24; ++j) {
        const f32x2 d = ptx::add2(x[j], npm);
        q2 = ptx::fma2(d, d, q2);
    }
    ptx::up2(q2, q_lo, q_hi);
    stat[i * 4 + part] = make_float2(pmean, q_lo + q_hi);
    asm volatile("bar.sync %0, 128;" ::"r"(2 + (i >> 5)) : "memory");      // only the four warps holding this row's quarters
    const float4 p01 = *reinterpret_cast<const float4 *>(stat + i * 4), p23 = *reinterpret_cast<const float4 *>(stat + i * 4 + 2);
    const float mean = ((p01.x + p01.z) + (p23.x + p23.z)) * 0.25f;
    const float d0 = p01.x - mean, d1 = p01.z - mean, d2 = p23.x - mean, d3 = p23.z - mean;
    const float m2 = ((p01.y + p01.w) + (p23.y + p23.w)) + 48.0f * ((d0 * d0 + d1 * d1) + (d2 * d2 + d3 * d3));
    const float rstd = rsqrtf(m2 * (1.0f / DIM) + 1e-5f);
    const f32x2 nmean = ptx::pk2(-mean, -mean), rs = ptx::pk2(rstd, rstd);
#pragma unroll
    for (int ch = 0; ch < 6; ++ch) {
        uint32_t w[4];
        f32x2 gm[4], bt[4];
        ptx::ld4(gam + ch * 8, gm[0], gm[1]); ptx::ld4(gam + ch * 8 + 4, gm[2], gm[3]);
        ptx::ld4(bet + ch * 8, bt[0], bt[1]); ptx::ld4(bet + ch * 8 + 4, bt[2], bt[3]);
#pragma unroll
        for (int e = 0; e < 4; ++e)      // ((x - mean) * rstd) * gamma + beta, two columns per instruction
            w[e] = pk_pair(ptx::fma2(ptx::mul2(ptx::add2(x[ch * 4 + e], nmean), rs), gm[e], bt[e]));
        uint4 u;
        u.x = w[0]; u.y = w[1]; u.z = w[2]; u.w = w[3];
        *reinterpret_cast<uint4 *>(a32 + slab_chunk_off(part * 48 + ch * 8, i)) = u;
    }
}

__global__ void __launch_bounds__(NUM_THREADS, 1)
window_stack192_kernel(const __grid_constant__ CUtensorMap tmap_w96, const __grid_constant__ CUtensorMap tmap_w128,
                       const __grid_constant__ CUtensorMap tmap_w192, const Stack192Params p) {
    pdl_trigger();
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem0 = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t *sm = smem_raw + (smem0 - ptx::smem_u32(smem_raw));
    Barriers *bars = reinterpret_cast<Barriers *>(sm + OFF_BAR);
    float *par = reinterpret_cast<float *>(sm + OFF_PAR);
    float2 *stat = reinterpret_cast<float2 *>(sm + OFF_STAT);
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        for (int i = 0; i < NRING; ++i) {
            ptx::mbar_init(ptx::smem_u32(&bars->full[i]), 1);
            ptx::mbar_init(ptx::smem_u32(&bars->empty[i]), 1);
        }
        ptx::mbar_init(ptx::smem_u32(&bars->a_ready), NMATH);
        ptx::mbar_init(ptx::smem_u32(&bars->g_ready[0]), NMATH);
        ptx::mbar_init(ptx::smem_u32(&bars->g_ready[1]), NMATH);
        for (int i = 0; i < NACC; ++i) ptx::mbar_init(ptx::smem_u32(&bars->acc[i]), 1);
        ptx::fence_barrier_init();
    }
    if (warp == NMATH + 1) {
        ptx::tmem_alloc(ptx::smem_u32(&bars->tmem_base), 512);
        ptx::tmem_relinquish();
    }
    if (warp == NMATH && lane == 0) {
        ptx::prefetch_tmap(&tmap_w96);
        ptx::prefetch_tmap(&tmap_w128);
        ptx::prefetch_tmap(&tmap_w192);
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = bars->tmem_base;
    const uint32_t TX = tmem_base, TACC = tmem_base + DIM, THID = tmem_base + DIM + 256;      // X 192 | two accumulator slots 256 | HID 64
    pdl_wait();

    if (warp == NMATH) {
        if (lane == 0) {
            // ================================ TMA producer: weight slabs in consumption order ================================
            // In flight: slabs [tail_n, n), laid out circularly in allocation order.  Before slab n is loaded, every older slab whose bytes it
            // would overwrite must have been released by the MMAs (releases arrive in order), and at most NRING slabs are in flight
            // (barrier pair n % NRING, parity (n / NRING) & 1).
            int nb0 = 0, tail_n = 0;          // slab number of the current block's first slab; slabs [tail_n, ..) may still be unreleased
            Seg sg;
            for (int k = 0; get_seg(p.n_tiles, p.n_blocks, p.seg_flags != nullptr, p.units_per_cta, k, sg); ++k)
                for (int bk = sg.lo; bk < sg.hi; ++bk, nb0 += SLABS_PER_BLOCK) {
                    int row = bk * ROWS_PER_BLOCK;
                    for (int s = 0; s < SLABS_PER_BLOCK; ++s) {
                        const int nr = slab_rows(s), n = nb0 + s;
                        for (const int need = nb0 + p.w_need[s]; tail_n <= need; ++tail_n)      // releases arrive in order
                            ptx::mbar_wait(ptx::smem_u32(&bars->empty[tail_n % NRING]), (uint32_t)(tail_n / NRING) & 1);
                        const uint32_t fb = ptx::smem_u32(&bars->full[n % NRING]);
                        ptx::mbar_expect_tx(fb, nr * 128);
                        ptx::tma_load_2d(smem0 + OFF_RING + p.w_off[s] * 1024, nr == 96 ? &tmap_w96 : nr == 128 ? &tmap_w128 : &tmap_w192, fb, 0, row);
                        row += nr;
                    }
                }
        }
    } else if (warp == NMATH + 1) {
        // ================================ MMA issuer (whole warp converged, elected lane issues) ================================
        const uint32_t leader = ptx::elect_one();
        const uint32_t id96 = ptx::make_idesc_bf16(128, 96), id128 = ptx::make_idesc_bf16(128, 128), id192 = ptx::make_idesc_bf16(128, 192);
        const uint32_t ring_lo = ptx::sdesc_lo(smem0 + OFF_RING);
        RingPos ring;
        int n = 0;                    // running slab number: barrier pair n % NRING, parity (n / NRING) & 1
        uint32_t aph = 0, gph = 0;
        // next weight slab (nrows x 64 k) of the ring: waits for it and returns the low descriptor word of its first byte
        auto next_slab = [&](int nrows) -> uint32_t {
            const int off = ring.place(nrows * 128);
            ptx::mbar_wait(ptx::smem_u32(&bars->full[n % NRING]), (uint32_t)(n / NRING) & 1);
            ptx::tc_fence_after();
            return ring_lo + (off >> 4);
        };
        auto release_slab = [&]() {
            ptx::umma_commit_pred(ptx::smem_u32(&bars->empty[n % NRING]), leader);
            ++n;
        };
        // one weight slab: D[128 x N] (+)= A_slab[128 x 64] * W_slab[N x 64]^T
        auto slab_mma = [&](uint32_t d_tmem, uint32_t a_lo, uint32_t idesc, int nrows, bool first_clears) {
            const uint32_t w_lo = next_slab(nrows);
            ptx::umma_bf16_lo_rt(d_tmem, a_lo, w_lo, idesc, first_clears ? 0u : 1u, leader);
#pragma unroll
            for (int k4 = 1; k4 < 4; ++k4) ptx::umma_bf16_lo<1>(d_tmem, a_lo + k4 * 2, w_lo + k4 * 2, idesc, leader);
            release_slab();
        };
        auto wait_a = [&]() {
            ptx::mbar_wait(ptx::smem_u32(&bars->a_ready), aph);
            aph ^= 1;
            ptx::tc_fence_after();
        };
        auto commit = [&](int which) { ptx::umma_commit_pred(ptx::smem_u32(&bars->acc[which]), leader); };
        const uint32_t a32 = ptx::sdesc_lo(smem0 + OFF_A32), ao = ptx::sdesc_lo(smem0 + OFF_AO);
        constexpr uint32_t SL = SLAB_A >> 4;
        Seg sg;
        for (int k = 0; get_seg(p.n_tiles, p.n_blocks, p.seg_flags != nullptr, p.units_per_cta, k, sg); ++k)
            for (int bk = sg.lo; bk < sg.hi; ++bk) {
                ring.head = 0;                                  // every block lays its slabs out from offset 0
                for (int g = 0; g < NGROUP; ++g) {
                    wait_a();                                   // g = 0: LN1 output in A32; g > 0: ACC drained by the previous group
                    for (int ks = 0; ks < 3; ++ks) slab_mma(TACC, a32 + ks * SL, id96, 96, ks == 0);
                    commit(ACC_QKV0 + g);
                }
                wait_a();                                       // attention output of all heads in AO
                for (int ks = 0; ks < 3; ++ks) slab_mma(TX, ao + ks * SL, id192, 192, false);          // x += att Wp^T
                commit(ACC_PROJ);
                wait_a();                                       // LN2 output in A32
                for (int c = 0; c < 2; ++c) {                   // fc1 chunks 0, 1 into the two accumulator slots
                    for (int ks = 0; ks < 3; ++ks) slab_mma(TACC + c * 128, a32 + ks * SL, id128, 128, ks == 0);
                    commit(ACC_FC1_0 + c);
                }
                for (int c = 0; c < NCHUNK; ++c) {
                    ptx::mbar_wait(ptx::smem_u32(&bars->g_ready[c & 1]), (gph >> (c & 1)) & 1);       // GELU(chunk c) in HID buffer c & 1
                    gph ^= 1u << (c & 1);
                    ptx::tc_fence_after();
                    // x += h_c W2[:, chunk c]^T.  Even chunks: A = GELU(chunk c) in TENSOR MEMORY (columns [448, 512): lane = token row, one
                    // column = two consecutive hidden units as a bf16 pair): the MMA reads only the weight slab from shared memory -- half
                    // the port load of the SS form -- and the math warps store the activation with tcgen05.st.  Tensor memory has room for
                    // one such buffer beside X and the two accumulator slots, so odd chunks keep the shared-memory buffer (SS form).
                    if (c & 1) {
                        for (int ks = 0; ks < 2; ++ks) slab_mma(TX, ao + ks * SL, id192, 192, false);
                    } else {
                        for (int ks = 0; ks < 2; ++ks) {
                            const uint32_t w_lo = next_slab(192);
#pragma unroll
                            for (int k4 = 0; k4 < 4; ++k4) ptx::umma_bf16_ts_lo<1>(TX, THID + ks * 32 + k4 * 8, w_lo + k4 * 2, id192, leader);
                            release_slab();
                        }
                    }
                    if (c + 2 < NCHUNK) {                       // accumulator slot c & 1 is drained: fc1 chunk c + 2
                        for (int ks = 0; ks < 3; ++ks) slab_mma(TACC + (c & 1) * 128, a32 + ks * SL, id128, 128, ks == 0);
                        commit(ACC_FC1_0 + c + 2);              // (its arrival also says: fc2 of chunk c has read HID buffer c & 1)
                    }
                }
                commit(ACC_FC2L);
            }
    } else {
        // ================================ math warps ================================
        const int q = warp & 3, part = warp >> 2;           // TMEM lane quadrant, column quarter (48 columns)
        const int i = q * 32 + lane;                        // token row of the tile == TMEM lane
        const uint32_t lane_base = (uint32_t)(q * 32) << 16;
        const int mt = threadIdx.x;                          // 0..511
        uint8_t *a32 = sm + OFF_A32, *aout = sm + OFF_AO, *stg = sm + OFF_STG;
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
        auto load_x = [&](f32x2 (&x)[24], const float *cvec) {
            uint32_t v[48];
            tmem_ld48(TX + lane_base + part * 48, v);
#pragma unroll
            for (int j = 0; j < 24; j += 2) {
                f32x2 c0v, c1v;
                ptx::ld4(cvec + part * 48 + 2 * j, c0v, c1v);
                x[j] = ptx::add2(ptx::pk2u(v[2 * j], v[2 * j + 1]), c0v);
                x[j + 1] = ptx::add2(ptx::pk2u(v[2 * j + 2], v[2 * j + 3]), c1v);
            }
        };

        Seg sg;
        for (int k = 0; get_seg(p.n_tiles, p.n_blocks, p.seg_flags != nullptr, p.units_per_cta, k, sg); ++k) {
            const int t = sg.tile;
            if (sg.lo > 0) {          // the CTA that ran blocks [0, lo) of this tile has stored and fenced the raw residual stream
                if (mt == 0) wait_flag_acquire(p.seg_flags + t);
                math_barrier();
            }
            // ---- tokens (or the raw residual stream of a tile in progress) -> TMEM X
            {
                const float *src = p.tok + ((long)t * 128 + i) * DIM + part * 48;
                uint32_t v[32], w[16];
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    const float4 f = __ldcg(reinterpret_cast<const float4 *>(src + j));
                    v[j] = __float_as_uint(f.x); v[j + 1] = __float_as_uint(f.y); v[j + 2] = __float_as_uint(f.z); v[j + 3] = __float_as_uint(f.w);
                }
#pragma unroll
                for (int j = 0; j < 16; j += 4) {
                    const float4 f = __ldcg(reinterpret_cast<const float4 *>(src + 32 + j));
                    w[j] = __float_as_uint(f.x); w[j + 1] = __float_as_uint(f.y); w[j + 2] = __float_as_uint(f.z); w[j + 3] = __float_as_uint(f.w);
                }
                ptx::tmem_st_x32(TX + lane_base + part * 48, v);
                ptx::tmem_st_x16(TX + lane_base + part * 48 + 32, w);
                ptx::tmem_st_wait();
                ptx::tc_fence_before();
            }
            // per-block parameters -> smem: the first block's here, the next block's while the last fc2 of a block runs
            auto load_params = [&](int bk) {
                math_barrier();       // everyone is done with the previous parameters
                const float4 *g4 = reinterpret_cast<const float4 *>(p.par + (long)bk * PAR_FLOATS);
                float4 *d = reinterpret_cast<float4 *>(par);
                for (int e = mt; e < PAR_FLOATS / 4; e += NMATH * 32) d[e] = g4[e];
            };
            int tr_b = 0;
            auto phase_ev = [&](int ph) {      // debug (tu_debug_trace): phase boundaries of warp 0
                if (p.trace && mt == 0) trace_event(p.trace, p.trace_cap, 10, (unsigned)(t * 256 + tr_b * 16 + ph));
            };
            load_params(sg.lo);
            for (int bk = sg.lo; bk < sg.hi; ++bk) {
                math_barrier();       // parameters (and the X stores of a new tile) are visible
                ptx::tc_fence_after();
                tr_b = bk;
                phase_ev(0);
                // ---- LN1(x + c0) -> A32
                {
                    f32x2 x[24];
                    load_x(x, par + P_C0);
                    layernorm_to_a32(x, par + P_LN1W + part * 48, par + P_LN1B + part * 48, stat, a32, i, part);
                }
                signal_a();
                phase_ev(1);
                // ---- six groups of two heads: qkv epilogue of group g, then its attention while the MMAs of g+1 run
                const ulonglong2 *relb = reinterpret_cast<const ulonglong2 *>(p.rel_bias) + (long)bk * HEADS * 1024;
                // relative-position bias of this thread's 2 rows x 16 columns of head (2g + hl): fetched one group ahead of its
                // use (the 17 KB of L1 left beside the shared memory cannot hold it, so every fetch is an L2 round trip); stored in
                // mma C-fragment order (packing.py::frag_rel_bias): one coalesced 16-byte load per lane and key octet
                f32x2 ba[8], bb2[8];
                auto load_bias = [&](int g) {
                    const int hl = (warp >> 2) & 1, rg = warp & 3;
                    const ulonglong2 *bp = relb + ((g * 2 + hl) * 4 + rg) * 256 + lane;
#pragma unroll
                    for (int n = 0; n < 8; ++n) {
                        const ulonglong2 v = __ldg(bp + n * 32);
                        ba[n] = v.x;
                        bb2[n] = v.y;
                    }
                };
                load_bias(0);
#pragma unroll 1
                for (int g = 0; g < NGROUP; ++g) {
                    wait_acc(ACC_QKV0 + g);
                    if (g == 0) phase_ev(2);
                    if (g > 0) math_barrier();            // every warp is done reading the previous group's q, k, v
                    if (part < 3) {                       // 96 columns: q | k | v of the group, 32 columns per part
                        uint32_t v[32];
                        ptx::tmem_ld_x32(TACC + lane_base + part * 32, v);
                        ptx::tmem_ld_wait();
                        const float *bb = par + P_QKVB + g * 96 + part * 32;
                        uint8_t *rowp = stg + i * STG_PITCH + part * 64;
#pragma unroll
                        for (int j = 0; j < 32; j += 8) {
                            uint4 u;
                            f32x2 b0v, b1v, b2v, b3v;
                            ptx::ld4(bb + j, b0v, b1v); ptx::ld4(bb + j + 4, b2v, b3v);
                            u.x = pk_pair(ptx::add2(ptx::pk2u(v[j + 0], v[j + 1]), b0v));
                            u.y = pk_pair(ptx::add2(ptx::pk2u(v[j + 2], v[j + 3]), b1v));
                            u.z = pk_pair(ptx::add2(ptx::pk2u(v[j + 4], v[j + 5]), b2v));
                            u.w = pk_pair(ptx::add2(ptx::pk2u(v[j + 6], v[j + 7]), b3v));
                            *reinterpret_cast<uint4 *>(rowp + j * 2) = u;
                        }
                    }
                    if (g + 1 < NGROUP) signal_a();       // ACC is drained: the MMAs of the next group may run
                    math_barrier();                       // q, k, v of the group are staged
                    // ---- attention: 2 windows x 2 heads x 4 row groups = 16 warp tasks, one per warp
                    {
                        const int gq = lane >> 2, tq = lane & 3;
                        const int win = warp >> 3, hl = (warp >> 2) & 1, rg = warp & 3;
                        const int h = g * 2 + hl;
                        const uint8_t *wbase = stg + (win * 64) * STG_PITCH;
                        const int r0 = rg * 16 + gq;
                        uint32_t qa[4];
                        qa[0] = *reinterpret_cast<const uint32_t *>(wbase + r0 * STG_PITCH + (hl * 16 + tq * 2) * 2);
                        qa[1] = *reinterpret_cast<const uint32_t *>(wbase + (r0 + 8) * STG_PITCH + (hl * 16 + tq * 2) * 2);
                        qa[2] = *reinterpret_cast<const uint32_t *>(wbase + r0 * STG_PITCH + (hl * 16 + tq * 2 + 8) * 2);
                        qa[3] = *reinterpret_cast<const uint32_t *>(wbase + (r0 + 8) * STG_PITCH + (hl * 16 + tq * 2 + 8) * 2);
                        float s[8][4];
#pragma unroll
                        for (int n = 0; n < 8; ++n) {
                            const uint8_t *kp = wbase + (n * 8 + gq) * STG_PITCH + (32 + hl * 16 + tq * 2) * 2;
                            const uint32_t b0 = *reinterpret_cast<const uint32_t *>(kp), b1 = *reinterpret_cast<const uint32_t *>(kp + 16);
                            ptx::up2(ba[n], s[n][0], s[n][1]);          // accumulators start at the relative-position bias
                            ptx::up2(bb2[n], s[n][2], s[n][3]);
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
                        if (g + 1 < NGROUP) load_bias(g + 1);         // in flight during softmax, PV and the next group's epilogue
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
                                                                (64 + hl * 16 + (lane >> 4) * 8) * 2);
                            asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                                         : "=r"(v0), "=r"(v1), "=r"(v2), "=r"(v3)
                                         : "r"(addr));
                            mma16816(o[0], pa, v0, v1);
                            mma16816(o[1], pa, v2, v3);
                            mma16816(ls, pa, 0x3f803f80u, 0x3f803f80u);
                        }
                        const float i0 = rcp_fast(ls[0]), i1 = rcp_fast(ls[2]);      // l >= 1: the row maximum contributes exp2(0)
                        // attention output -> AO (row = token of the tile, column = h*16 + d), swizzled K-slabs
                        const int row0 = win * 64 + r0, row1 = row0 + 8;
#pragma unroll
                        for (int nt = 0; nt < 2; ++nt) {
                            const int col = h * 16 + nt * 8 + tq * 2;
                            const int bo = (col & 7) * 2;
                            *reinterpret_cast<uint32_t *>(aout + slab_chunk_off(col, row0) + bo) = pk_pair(ptx::mul2(ptx::pk2(o[nt][0], o[nt][1]), ptx::pk2(i0, i0)));
                            *reinterpret_cast<uint32_t *>(aout + slab_chunk_off(col, row1) + bo) = pk_pair(ptx::mul2(ptx::pk2(o[nt][2], o[nt][3]), ptx::pk2(i1, i1)));
                        }
                    }
                }
                signal_a();                               // attention output of all 12 heads is in AO
                phase_ev(3);
                // ---- LN2(x + c1) -> A32 (after proj has been accumulated onto X)
                wait_acc(ACC_PROJ);
                phase_ev(4);
                {
                    f32x2 x[24];
                    load_x(x, par + P_C1);
                    layernorm_to_a32(x, par + P_LN2W + part * 48, par + P_LN2B + part * 48, stat + 128 * 4, a32, i, part);
                }
                signal_a();
                phase_ev(5);
                // ---- MLP: six chunks of 128 hidden units: accumulator slot c & 1 -> +bias -> GELU -> bf16 HID (even chunks: tensor memory,
                // odd chunks: 32 KB of the idle AO region).  fc1 of chunk c + 2 is committed behind fc2 of chunk c, so its arrival also
                // frees the HID buffer this chunk writes.
#pragma unroll 1
                for (int c = 0; c < NCHUNK; ++c) {
                    wait_acc(ACC_FC1_0 + c);
                    if (c == 0) phase_ev(6);
                    uint32_t v[32];
                    ptx::tmem_ld_x32(TACC + lane_base + (c & 1) * 128 + part * 32, v);
                    ptx::tmem_ld_wait();
                    const float *bb = par + P_FC1B + c * 128 + part * 32;
#pragma unroll
                    for (int j = 0; j < 32; j += 8) {
                        uint4 u;
                        f32x2 b0v, b1v, b2v, b3v;
                        ptx::ld4(bb + j, b0v, b1v); ptx::ld4(bb + j + 4, b2v, b3v);
                        u.x = pk_pair(gelu_fast2(ptx::add2(ptx::pk2u(v[j + 0], v[j + 1]), b0v)));
                        u.y = pk_pair(gelu_fast2(ptx::add2(ptx::pk2u(v[j + 2], v[j + 3]), b1v)));
                        u.z = pk_pair(gelu_fast2(ptx::add2(ptx::pk2u(v[j + 4], v[j + 5]), b2v)));
                        u.w = pk_pair(gelu_fast2(ptx::add2(ptx::pk2u(v[j + 6], v[j + 7]), b3v)));
                        if (c & 1) *reinterpret_cast<uint4 *>(aout + slab_chunk_off(part * 32 + j, i)) = u;      // odd chunks: shared-memory buffer
                        else ptx::tmem_st_x4(THID + lane_base + part * 16 + j / 2, u.x, u.y, u.z, u.w);          // even chunks: tensor memory
                    }
                    if (c & 1) ptx::fence_proxy_async();
                    else ptx::tmem_st_wait();
                    ptx::tc_fence_before();
                    __syncwarp();
                    if (lane == 0) ptx::mbar_arrive(ptx::smem_u32(&bars->g_ready[c & 1]));
                    if (c < 4) phase_ev(7 + c);
                }
                if (bk + 1 < sg.hi) load_params(bk + 1);
                wait_acc(ACC_FC2L);      // fc2 of the last quarter accumulated: X holds the block output (minus folded biases)
                phase_ev(11);
                cph ^= 1;
            }
            if (sg.hi < p.n_blocks) {
                // ---- tile in progress: raw X -> global (the folded bias offsets are NOT applied: the next CTA continues exactly here)
                float *dst = p.tok + ((long)t * 128 + i) * DIM + part * 48;
                uint32_t v[48];
                tmem_ld48(TX + lane_base + part * 48, v);
#pragma unroll
                for (int j = 0; j < 48; j += 4)
                    *reinterpret_cast<float4 *>(dst + j) = make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
                ptx::tc_fence_before();
                __threadfence();
                math_barrier();
                if (mt == 0) atomicExch(p.seg_flags + t, 1);
                continue;
            }
            // ---- X (+ final offset) -> global
            {
                const float *cfin = p.par + (long)p.n_blocks * PAR_FLOATS + part * 48;
                float *dst = p.tok + ((long)t * 128 + i) * DIM + part * 48;
                bf16 *dst16 = p.tok16 ? p.tok16 + ((long)t * 128 + i) * DIM + part * 48 : nullptr;
                uint32_t v[48];
                tmem_ld48(TX + lane_base + part * 48, v);
#pragma unroll
                for (int j = 0; j < 48; j += 4) {
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
            }
        }
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == NMATH + 1) ptx::tmem_dealloc(tmem_base, 512);
}

PerDeviceFlag g_attr_set;

int host_slab_rows(int s) {
    if (s < SLABS96) return 96;
    if (s < SLABS96 + 3) return 192;
    if (s < SLABS96 + 9) return 128;
    const int t = s - (SLABS96 + 9);
    return (t >= 20 || t % 5 < 2) ? 192 : 128;
}
// layout of a block's slabs in the ring and, per slab, the newest older slab its bytes (or its barrier pair) still belong to
void plan_ring(Stack192Params &p) {
    int off[2 * SLABS_PER_BLOCK], len[2 * SLABS_PER_BLOCK];
    for (int blk = 0; blk < 2; ++blk) {
        int head = 0;
        for (int s = 0; s < SLABS_PER_BLOCK; ++s) {
            const int b = host_slab_rows(s) * 128;
            if (head + b > RING_BYTES) head = 0;
            off[blk * SLABS_PER_BLOCK + s] = head;
            len[blk * SLABS_PER_BLOCK + s] = b;
            head += b;
        }
    }
    for (int s = 0; s < SLABS_PER_BLOCK; ++s) {          // steady state = the second block
        const int n = SLABS_PER_BLOCK + s;
        int need = n - NRING;                             // its barrier pair was last used by slab n - NRING
        for (int m = n - 1; m > need && m >= 0; --m)
            if (off[m] < off[n] + len[n] && off[n] < off[m] + len[m]) { need = m; break; }
        p.w_off[s] = (unsigned char)(off[n] / 1024);
        p.w_need[s] = (signed char)(need - SLABS_PER_BLOCK);
    }
}

}  // namespace

// stack_w: bf16 (n_blocks * 6912, 64) weight slabs in consumption order; stack_p: fp32 n_blocks*2496 + 192;
// rel_bias: fp32 n_blocks x (12,4096) in fragment order.  tok: (M,192) fp32 with M % 128 == 0.
int tc_window_stack192(float *tok, bf16 *tok16, int M, int n_blocks, const bf16 *stack_w, const float *stack_p,
                       const float *rel_bias, int *tile_flags, int *seg_flags, cudaStream_t st) {
    TcEncodeFn enc = tc_encode_fn();
    if (!enc || !stack_w || !stack_p || !rel_bias || (M % 128) || (reinterpret_cast<uintptr_t>(stack_w) & 127) ||
        (reinterpret_cast<uintptr_t>(tok) & 15))
        return TU_TC_UNSUPPORTED;
    const int g_sm_count = device_sm_count();
    if (!g_attr_set.is_set()) {
        cudaError_t e = cudaFuncSetAttribute(window_stack192_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
        if (e != cudaSuccess) return cuda_fail(e, "window_stack192 smem attribute");
        g_attr_set.set();
    }
    CUtensorMap t96, t128, t192;
    cuuint64_t wd[2] = {64, (cuuint64_t)n_blocks * ROWS_PER_BLOCK}, ws[1] = {128};
    cuuint32_t b96[2] = {64, 96}, b128[2] = {64, 128}, b192[2] = {64, 192}, we[2] = {1, 1};
    CUresult r = enc(&t96, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void *)stack_w, wd, ws, b96, we, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r == CUDA_SUCCESS)
        r = enc(&t128, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void *)stack_w, wd, ws, b128, we, CU_TENSOR_MAP_INTERLEAVE_NONE,
                CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r == CUDA_SUCCESS)
        r = enc(&t192, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void *)stack_w, wd, ws, b192, we, CU_TENSOR_MAP_INTERLEAVE_NONE,
                CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("tu: cuTensorMapEncodeTiled(window stack 192 weights) failed with code " + std::to_string((int)r));
        return TU_ERR_CUDA;
    }
    Stack192Params p;
    p.tok = tok; p.tok16 = tok16; p.par = stack_p; p.rel_bias = rel_bias;
    p.trace = g_trace_buf; p.trace_cap = g_trace_cap;
    p.var = tc_stack_var();
    plan_ring(p);
    p.n_tiles = M / 128; p.n_blocks = n_blocks; p.tile_flags = tile_flags;
    const int grid = p.n_tiles < g_sm_count ? p.n_tiles : g_sm_count;
    p.seg_flags = (seg_flags && tc_stack_split_enabled() && p.n_tiles % grid != 0) ? seg_flags : nullptr;
    p.units_per_cta = ceil_div(p.n_tiles * n_blocks, grid);
    launch_pdl(window_stack192_kernel, dim3(grid), dim3(NUM_THREADS), SMEM_BYTES, st, t96, t128, t192, p);
    TU_CHECK_LAUNCH("window_stack192");
    return TU_OK;
}

}  // namespace tu
