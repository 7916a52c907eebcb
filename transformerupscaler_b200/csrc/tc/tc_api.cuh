// Internal interface between the C-ABI layer and the tcgen05 (5th-gen tensor core) kernels.
#pragma once
#include <cuda.h>

#include "../tu_common.cuh"

namespace tu {

constexpr int TU_TC_UNSUPPORTED = 1;   // shape not covered by the tensor-core kernel: caller falls back to SIMT

// 1 when the tcgen05 kernels were compiled in and may be used on this device.
int tc_available();
// tc_available() and not switched off by tu_set_bf16_tcgen05(0)
bool tc_enabled();
// debug: 0 = UMMA descriptor base_offset 0, 1 = base_offset (addr>>7)&7 for row-shifted operand views
void tc_set_base_off_mode(int m);
// debug: reversed work-item order per kernel (bit mask, see conv3x3_tcgen05.cu)
extern thread_local int g_snake_mask;
void tc_set_snake(int mask);

// debug: device buffer of (time, tag) event pairs written by the window stack and the unembed GEMM (tu_debug_trace); word 0 = count
extern thread_local unsigned long long *g_trace_buf;
extern thread_local unsigned int g_trace_cap;
__device__ __forceinline__ void trace_event(unsigned long long *buf, unsigned int cap, unsigned int kind, unsigned int value) {
    if (!buf) return;
    unsigned long long t;
    unsigned int sm;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    asm volatile("mov.u32 %0, %%smid;" : "=r"(sm));
    const unsigned long long i = atomicAdd(buf, 1ULL);
    if (i < cap) {
        buf[1 + 2 * i] = t;
        buf[2 + 2 * i] = ((unsigned long long)kind << 48) | ((unsigned long long)sm << 32) | value;
    }
}

// cuTensorMapEncodeTiled resolved through the runtime (no link-time dependency on libcuda); nullptr without a driver
typedef CUresult (*TcEncodeFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                               const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
TcEncodeFn tc_encode_fn();
// TMA element type of an image at the boundary, chosen by dtype code: fp16 and bf16 are both 2 bytes wide and must not share it
static inline CUtensorMapDataType tc_image_map_dtype(int dtype) {
    switch (dtype_base(dtype)) {
        case TU_F32: return CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
        case TU_BF16: return CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
        case TU_F16: return CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
        default: return CU_TENSOR_MAP_DATA_TYPE_UINT8;
    }
}

// C = A W^T GEMMs of the transformer part (gemm_tcgen05.cu).  All return TU_OK, an error, or TU_TC_UNSUPPORTED.
//   out != nullptr : out[M][N] = act(A W^T + bias) as bf16 (act 0 none, 2 exact GELU)
//   resid_x != nullptr : resid_x[M][N] += A W^T + bias (fp32), and resid_bf16 (optional) receives a bf16 copy
int tc_linear(const bf16 *A, const bf16 *W, const float *bias, int M, int N, int K, int act, bf16 *out, float *resid_x,
              bf16 *resid_bf16, cudaStream_t st);
int tc_patch_embed(const bf16 *feat, const bf16 *W, const float *bias, const float *pos, float *tok, int B, int H, int Wd,
                   int Ht, int Wt, int dim, int window, cudaStream_t st);
void tc_set_unembed_areuse(int on);
// patch embed at dim 128 with one tile per CTA and two CTAs per SM (embed_tcgen05.cu): same contract as tc_patch_embed
int tc_patch_embed_pair(const bf16 *feat, const bf16 *W, const float *bias, const float *pos, float *tok, int B, int H, int Wd,
                        int Ht, int Wt, int dim, int window, cudaStream_t st);
void tc_set_embed_pair(int on);
int tc_patch_unembed(const bf16 *tok_bf16, const bf16 *W, const float *bias, const bf16 *skip, int skipH, int skipW, bf16 *out,
                     int B, int Ht, int Wt, int Hc, int Wc, int dim, int window, int *dyn_ctr, const int *tile_flags, cudaStream_t st);

// 3x3 / pad 1 convolution, 64 input channels, NHWC bf16, fp32 accumulation in TMEM.
// w: [chunk][tap][co 64][ci 64] bf16.  Returns TU_OK, an error code, or TU_TC_UNSUPPORTED.
int tc_conv3x3_c64(const bf16 *in, const bf16 *w, const float *bias, bf16 *out, int B, int H, int W, int stride, int relu,
                   int nchunk, int ps_r, cudaStream_t st);

// the same convolution on a CTA pair (tcgen05 cta_group::2, conv3x3_2cta_tcgen05.cu): plain 64 -> 64 only
int tc_conv3x3_c64_pair(const bf16 *in, const bf16 *w, const float *bias, bf16 *out, int B, int H, int W, int stride, int relu,
                        cudaStream_t st);
void tc_set_conv_2cta(int on);
// the same convolution streaming down the image with the three ky taps stacked into N = 192 (conv3x3_stream_tcgen05.cu):
// plain 64 -> 64, stride 1
int tc_conv3x3_c64_stream(const bf16 *in, const bf16 *w, const float *bias, bf16 *out, int B, int H, int W, int relu, int nchunk,
                          int ps_r, cudaStream_t st);
void tc_set_conv_stream(int on);

// decoder_conv2(relu(decoder_conv1(x))) in one kernel (dec12_fused_tcgen05.cu): NHWC bf16 -> planar fp32 (B, 3, H, W); w1 = the
// 64 -> 64 bank of tc_conv3x3_c64, w16 = the head bank of tc_conv3x3_c64_to3.  The pixels shared by two 128-pixel strips are
// accumulated with atomicAdd: tc_dec12_zero_seams must run on the same stream beforehand (anywhere before the launch)
int tc_dec12_fused(const bf16 *in, const bf16 *w1, const float *bias1, const bf16 *w16, const float *bias2, float *out3, int B, int H,
                   int W, cudaStream_t st);
int tc_dec12_zero_seams(float *out3, int B, int H, int W, cudaStream_t st);
void tc_set_dec12_fused(int on);
bool tc_dec12_fused_enabled();

// relu(conv2(relu(conv1(x)))) in one kernel (conv12_fused_tcgen05.cu): NCHW image -> NHWC bf16; conv1's output stays on chip
int tc_conv12_fused(const void *x, int in_dtype, const bf16 *w64, const float *bias1, const bf16 *w2, const float *bias2, bf16 *out,
                    int B, int H, int W, cudaStream_t st);
void tc_set_conv12_fused(int on);

// conv1 3 -> 64 + ReLU, NCHW (fp32|bf16) -> NHWC bf16 (stem_tcgen05.cu)
int tc_stem_conv(const void *x, int in_dtype, const bf16 *w64, const float *bias, bf16 *out, int B, int H, int W, cudaStream_t st);

// 64 -> 3 head (decoder_conv2 / up1_conv): w16 = bf16 [3 ky][16 rows n = kx*4 + co (co < 3)][64 ci]; planar fp32 (B,3,H,W) out
int tc_conv3x3_c64_to3(const bf16 *in, const bf16 *w16, const float *bias, float *out, int B, int H, int W, int relu,
                       cudaStream_t st);

// folded last up1 stage + up1_conv (upfold_stream_tcgen05.cu): NHWC bf16 -> planar fp32 (B,3,rH,rW), ReLU applied
int tc_upfold(const bf16 *in, const TuUpFold *f, float *out, int B, int H, int W, cudaStream_t st);

// 64 -> 3 head on the streaming kernel (3x3 instance of upfold_stream_tcgen05.cu); wst / bias16 as packed by packing.py
int tc_conv3x3_c64_to3_stream(const bf16 *in, const bf16 *wst, const float *bias16, float *out, int B, int H, int W, int relu,
                              cudaStream_t st);

// all window-transformer blocks in one persistent kernel (dim 128; window_stack_tcgen05.cu)
// tile_flags (optional, zeroed by the caller): tile_flags[t] is set once the 128 tokens of tile t are final and fenced
// seg_flags (optional, zeroed by the caller, one int per tile): allows a tile to be handed from one CTA to the next at a block
// boundary, so that the (tile, block) units are dealt out evenly when the tiles do not fill whole waves of SMs
int tc_window_stack(float *tok, bf16 *tok16, int M, int n_blocks, const bf16 *stack_w, const float *stack_p,
                    const float *rel_bias, int *tile_flags, int *seg_flags, cudaStream_t st);
void tc_set_stack_split(int on);
void tc_set_stack_var(int mask);      // debug variants of the stack kernels
int tc_stack_var();
bool tc_stack_split_enabled();

// the same for FastTransformer (dim 192, 12 heads; window_stack192_tcgen05.cu)
int tc_window_stack192(float *tok, bf16 *tok16, int M, int n_blocks, const bf16 *stack_w, const float *stack_p,
                       const float *rel_bias, int *tile_flags, int *seg_flags, cudaStream_t st);

// ResidualTransformer's global attention on tcgen05 (global_attn_tcgen05.cu): qkv (B*S, 3*dim) bf16 with q pre-scaled -> out (B*S, dim)
// bf16.  vt: B*dim*S bf16 scratch (V transposed), scratch: tc_global_attention_scratch_bytes() of fp32 partials
size_t tc_global_attention_scratch_bytes(int B, int S, int heads);
int tc_global_attention(const bf16 *qkv, bf16 *out, bf16 *vt, float *scratch, size_t scratch_bytes, int B, int S, int heads,
                        cudaStream_t st);
void tc_set_global_attn(int on);
// workspace of one transformer block including the scratch of the tcgen05 global attention (window == 0)
size_t block_workspace_bytes_ex(int M, int dim, int dtype, int window, int S);

// ResidualTransformer's block around the attention in two fused kernels (residual_block_tcgen05.cu): LN1 + in_proj -> qkv, and
// out_proj + residual + LN2 + MLP + residual in place on the fp32 stream.  stack_w / stack_p as packed for TU_MODEL_RESIDUAL.
int tc_resid_pre(const float *tok, bf16 *qkv, int M, int layer, int n_layers, const bf16 *stack_w, const float *stack_p, cudaStream_t st);
int tc_resid_post(float *tok, bf16 *tok16, const bf16 *att, int M, int layer, int n_layers, const bf16 *stack_w, const float *stack_p,
                  cudaStream_t st);
void tc_set_resid_fused(int on);
// one ResidualTransformer layer through the two fused kernels and the global attention (transformer_simt.cu); workspace as for
// transformer_block_ex.  TU_TC_UNSUPPORTED when the fused kernels cannot run.
int resid_layer_fused(float *x, const TuModelWeights *w, int layer, int M, int S, void *workspace, size_t workspace_bytes, bf16 *x_bf16_out,
                      cudaStream_t st);

// one pre-LN transformer block (transformer_simt.cu); x_bf16_out optionally receives a bf16 copy of the output stream
int transformer_block_ex(float *x, const TuBlockWeights *w, int M, int dim, int heads, int window, int S, int dtype,
                         void *workspace, size_t workspace_bytes, bf16 *x_bf16_out, cudaStream_t st);

}  // namespace tu
