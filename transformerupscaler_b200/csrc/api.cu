// C-ABI entry points of libtu_b200: error plumbing, the GEMM-shaped single ops, and the whole-model
// forward drivers that enqueue every kernel of a TransformerModel.forward on the caller's stream.
#include <string.h>

#include <algorithm>
#include <atomic>
#include <mutex>
#include <vector>

#include "gemm_simt.cuh"
#include "tc/tc_api.cuh"

namespace tu {

thread_local int g_use_pdl = 1;            // programmatic dependent launch of the forward's kernels (debug key "pdl")
static thread_local std::string g_err;
static thread_local int g_use_tc = 1;
static thread_local int g_unembed_overlap = 1;   // unembed starts on the SMs the window stack's last wave leaves idle (debug switch "unembed_overlap")
static thread_local int g_head_stream = 0; // 64 -> 3 heads on the streaming kernel (debug switch "head_stream"): measured slower than the tile kernel
static thread_local int g_fold_up1 = 1;    // FastTransformer: folded last up1 stage + up1_conv (debug switch "fold_up1")
static thread_local int g_use_stack = 1;   // fused window-transformer stack kernel (debug switch "fused_stack")
static thread_local int g_frame_chunk = 0;  // debug switch "frame_chunk": conv1+conv2 and the downsample run in chunks of this many frames (0 = whole batch)

static std::atomic<long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

// bench-only kernel timing hook (see tu_profile_enable in tu_b200.h): every launch of tu_forward is bracketed by a
// pair of CUDA events on the caller's stream and tagged with the name of the reference op it implements
static thread_local int g_prof_on = 0;
static std::mutex g_prof_mu;
struct ProfRec { const char *name; cudaEvent_t a, b; };
static std::vector<ProfRec> g_prof_events;
static thread_local cudaEvent_t g_prof_open = nullptr;
static thread_local const char *g_prof_name = nullptr;      // the op about to be launched (set by TU_STEP)
static inline bool prof_wanted() {
    return g_prof_on >= 2 || (g_prof_on == 1 && g_prof_name && (!strcmp(g_prof_name, "conv2") || !strcmp(g_prof_name, "conv1_conv2")));
}
static void prof_begin(cudaStream_t st) {
    if (!prof_wanted()) return;
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) return;
    cudaEventRecord(e, st);
    g_prof_open = e;
}
static void prof_end(cudaStream_t st, const char *name) {
    if (!g_prof_open) return;
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) return;
    cudaEventRecord(e, st);
    std::lock_guard<std::mutex> lk(g_prof_mu);
    g_prof_events.push_back({name, g_prof_open, e});
    g_prof_open = nullptr;
}
// run one launcher call, bracketed when profiling is on
#define TU_STEP(name, call)            \
    do {                               \
        g_prof_name = name;            \
        prof_begin(st);                \
        rc = (call);                   \
        prof_end(st, name);            \
        if (rc) return rc;             \
    } while (0)

void set_error(const std::string &msg) { g_err = msg; }
int cuda_fail(cudaError_t e, const char *what) {
    g_err = std::string("tu: CUDA error in ") + what + ": " + cudaGetErrorString(e);
    return TU_ERR_CUDA;
}

bool tc_enabled() { return g_use_tc && tc_available(); }
static inline bool tc_on(int dtype) { return dtype == TU_BF16 && tc_enabled(); }

// ------------------------------------------------------------------ op launchers (typed)
template <typename T>
static int conv3x3_c64(const T *in, const T *w, const float *b, T *out, int B, int H, int W, int stride, int relu,
                       int nchunk, int ps_r, cudaStream_t st) {
    const int Ho = (H - 1) / stride + 1, Wo = (W - 1) / stride + 1;
    const int M = B * Ho * Wo;
    AConv3x3<T> a{in, M, H, W, Ho, Wo, stride};
    WDesc<T> wd{w, 64, 64L * 64, 9L * 64 * 64};
    EpiConv<T> e{out, b, Ho, Wo, relu, ps_r, nchunk * 64};
    return launch_gemm_simt<T>(a, wd, M, nchunk * 64, 576, e, st, "conv3x3_c64");
}

template <typename T>
static int patch_embed(const T *feat, const T *w, const float *b, const float *pos, float *tok, int B, int H, int W,
                       int Ht, int Wt, int dim, int window, int reflect, cudaStream_t st) {
    const int M = B * Ht * Wt;
    APatch<T> a{feat, M, H, W, Ht, Wt, reflect};
    WDesc<T> wd{w, 4096, 0, 64L * 4096};
    EpiEmbed e{tok, b, pos, Ht, Wt, dim, window, (Ht + 7) / 8, (Wt + 7) / 8};
    return launch_gemm_simt<T>(a, wd, M, dim, 4096, e, st, "patch_embed");
}

template <typename T>
static int patch_unembed(const float *tok, const T *w, const float *b, const T *skip, int skipH, int skipW, T *out, int B,
                         int Ht, int Wt, int Hc, int Wc, int dim, int window, cudaStream_t st) {
    const int M = B * Ht * Wt;
    ATokens a{tok, M, Ht, Wt, dim, window, (Ht + 7) / 8, (Wt + 7) / 8};
    WDesc<T> wd{w, dim, 0, 64L * dim};
    EpiUnembed<T> e{out, b, skip, Ht, Wt, Hc, Wc, skipH, skipW};
    return launch_gemm_simt<T>(a, wd, M, 4096, dim, e, st, "patch_unembed");
}

// fp16 frame -> fp32 frame (exact).  Used where an fp16 frame's rows cannot be addressed by TMA but fp32 rows can (W % 8 == 4), so
// that the frame takes the fused conv1+conv2 kernel like the fp32 frame of the same values, and gives its bits.
__global__ void __launch_bounds__(256) widen_f16_kernel(const f16 *__restrict__ in, float *__restrict__ out, long n) {
    pdl_trigger();
    pdl_wait();
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) out[i] = __half2float(in[i]);
}

// ------------------------------------------------------------------ workspace arena
struct Arena {
    char *base;
    size_t off, cap;
    bool dry;
    void *get(size_t bytes) {
        size_t o = off;
        off += align_up(bytes, 1024);
        return dry ? (void *)nullptr : (void *)(base + o);
    }
};

static int scale_slot(int s) { return s == 2 ? 0 : s == 3 ? 1 : s == 4 ? 2 : s == 6 ? 3 : -1; }

// Runs (or, with a.dry, only sizes) one forward.  TI/TO are handled by dtype codes in the leaf launchers.
// xf / of: the input / output frame surfaces of an NV12 / P010 side, or NULL for the dense buffer x / out.
template <typename T>
static int forward_impl(const TuModelWeights *w, const void *x, const TuFramePlanes *xf, int in_dtype, void *out, const TuFramePlanes *of,
                        int out_dtype, int B, int H, int W, int outH, int outW, int scale, int clamp, Arena &a, cudaStream_t st) {
    const int dt = sizeof(T) == 2 ? TU_BF16 : TU_F32;
    const bool dry = a.dry;
    const int model = w->model, dim = w->dim, heads = w->heads;
    const bool fast = model == TU_MODEL_FAST, window = model != TU_MODEL_RESIDUAL;
    int rc;
    void *stv = (void *)st;

    if (fast && scale_slot(scale) < 0) {
        set_error("Requested scale=" + std::to_string(scale) + " was not built.");
        return TU_ERR_SCALE;
    }
    // feature-map geometry
    const int Hd = fast ? H : (H - 1) / 2 + 1, Wd = fast ? W : (W - 1) / 2 + 1;   // grid the tokens come from
    const int Ht = fast ? (H + 7) / 8 : Hd / 8, Wt = fast ? (W + 7) / 8 : Wd / 8;  // Fast reflect-pads up, others floor
    if (Ht < 1 || Wt < 1) {
        set_error("tu: input too small for an 8x8 patch grid");
        return TU_ERR_ARG;
    }
    if (model == TU_MODEL_RESIDUAL) {
        if (Ht * Wt != 3600) {
            set_error("The size of tensor a (" + std::to_string(Ht * Wt) +
                      ") must match the size of tensor b (3600) at non-singleton dimension 1");
            return TU_ERR_TOKENS;
        }
        if (Hd != 8 * Ht || Wd != 8 * Wt) {
            set_error("tu: ResidualTransformer skip connection needs a feature map that is a multiple of 8");
            return TU_ERR_ARG;
        }
    }
    const int nWy = (Ht + 7) / 8, nWx = (Wt + 7) / 8;
    const int Mtok = window ? B * nWy * nWx * 64 : B * Ht * Wt;
    const int Hc = fast ? H : min(Hd, 8 * Ht), Wc = fast ? W : min(Wd, 8 * Wt);

    // NV12 frames are converted to planar fp16 first: from then on the frame is an fp16 frame (the W % 8 == 4 widening below
    // included), and the final bicubic reads the same buffer
    if (dtype_is_nv12(in_dtype)) {
        f16 *rgb = (f16 *)a.get((size_t)B * 3 * H * W * sizeof(f16));
        if (!dry) TU_STEP("nv12_to_rgb", xf ? tu_yuv420_planes_to_rgb(xf, in_dtype, rgb, B, H, W, stv) : tu_nv12_to_rgb(x, in_dtype, rgb, B, H, W, stv));
        x = rgb;
        in_dtype = TU_F16;
    } else if (dtype_is_p010(in_dtype)) {
        // P010 frames are converted to planar fp32 (fp16 cannot hold every 10-bit step exactly): the forward is then the fp32-input one
        float *rgb = (float *)a.get((size_t)B * 3 * H * W * sizeof(float));
        if (!dry) TU_STEP("p010_to_rgb", xf ? tu_yuv420_planes_to_rgb(xf, in_dtype, rgb, B, H, W, stv) : tu_p010_to_rgb(x, in_dtype, rgb, B, H, W, stv));
        x = rgb;
        in_dtype = TU_F32;
    }
    // NV12 / P010 output: the last image kernel writes planar fp16 / fp32 here, and tu_rgb_to_nv12 / tu_rgb_to_p010 writes `out` from it
    const bool nv12_out = dtype_is_nv12(out_dtype), p010_out = dtype_is_p010(out_dtype);
    void *img = nv12_out ? a.get((size_t)B * 3 * outH * outW * sizeof(f16))
                : p010_out ? a.get((size_t)B * 3 * outH * outW * sizeof(float)) : out;
    const int img_dtype = nv12_out ? TU_F16 : p010_out ? TU_F32 : out_dtype;
#define TU_YUV_OUT()                                                                                                    \
    if (of) TU_STEP(nv12_out ? "rgb_to_nv12" : "rgb_to_p010", tu_rgb_to_yuv420_planes(img, of, out_dtype, B, outH, outW, stv)); \
    else if (nv12_out) TU_STEP("rgb_to_nv12", tu_rgb_to_nv12(img, out, out_dtype, B, outH, outW, stv));                    \
    else if (p010_out) TU_STEP("rgb_to_p010", tu_rgb_to_p010(img, out, out_dtype, B, outH, outW, stv))

    // interleaved uint8 frames (HWC RGB / BGR, RGBA / BGRA) are made planar once; the stem and the final bicubic both read the planar copy
    uint8_t *xplanar = (uint8_t *)a.get((size_t)B * 3 * H * W);
    // 4-byte frames on both sides: the input alpha, resampled to the output size, is the output alpha (read by the last image kernel)
    const bool alpha_io = dtype_is_px4(in_dtype) && dtype_is_px4(out_dtype);
    uint8_t *aplane = alpha_io ? (uint8_t *)a.get((size_t)B * outH * outW) : nullptr;
    if (!dry && alpha_io) TU_STEP("resample_alpha", tu_resample_alpha(x, in_dtype, aplane, B, H, W, outH, outW, stv));
    if (!dry && dtype_layout(in_dtype)) {
        if ((rc = tu_frames_to_planar(x, dtype_layout(in_dtype) << 8, xplanar, B, H, W, stv))) return rc;
        x = xplanar;
        in_dtype = TU_U8;
    }
    // (sized on every pass whose width needs it: the workspace queries do not know the input dtype)
    float *xwide = (W % 8) == 4 ? (float *)a.get((size_t)B * 3 * H * W * sizeof(float)) : nullptr;
    if (!dry && xwide && dtype_base(in_dtype) == TU_F16 && tc_on(dt) && w->conv1_w64) {
        const long n = (long)B * 3 * H * W;
        const cudaError_t e = launch_pdl(widen_f16_kernel, dim3((unsigned)std::min<long>((n + 255) / 256, 4096)), dim3(256), 0, st,
                                         (const f16 *)x, xwide, n);
        if (e != cudaSuccess) return cuda_fail(e, "widen_f16");
        count_launch();
        x = xwide;
        in_dtype = TU_F32;
    }
    const size_t full = (size_t)B * H * W * 64 * sizeof(T);
    T *f1 = (T *)a.get(full);
    T *f2 = (T *)a.get(full);
    T *fd = fast ? f2 : (T *)a.get((size_t)B * Hd * Wd * 64 * sizeof(T));
    float *tok = (float *)a.get((size_t)Mtok * dim * sizeof(float));
    bf16 *tok16 = (bf16 *)a.get((size_t)Mtok * dim * sizeof(bf16));   // bf16 copy of the final stream (tensor-core unembed)
    const size_t bws = block_workspace_bytes_ex(Mtok, dim, dt, window ? 1 : 0, Ht * Wt);
    void *blk = a.get(bws);
    T *comb = (T *)a.get((size_t)B * Hc * Wc * 64 * sizeof(T));
    T *dec = (T *)a.get((size_t)B * Hc * Wc * 64 * sizeof(T));
    float *res = (float *)a.get((size_t)B * 3 * Hc * Wc * sizeof(float));
    // tile hand-off between the fused window stack and the unembed GEMM: word 0 = tile counter, words 16.. = one flag per 128 tokens
    // ... and, behind them, one flag per tile for the hand-over of a tile between two CTAs of the stack kernel (block-level split)
    const int n_tok_tiles = Mtok / 128 + 1;
    const size_t sync_bytes = (size_t)(16 + 2 * n_tok_tiles) * sizeof(int);
    int *sync_words = (int *)a.get(sync_bytes);
    const bool overlap = g_unembed_overlap && window && tc_on(dt) && w->stack_w && g_use_stack && (Mtok % 128) == 0;
    const bool stack_flags = window && tc_on(dt) && w->stack_w && g_use_stack && (Mtok % 128) == 0;

    // decoder_conv1 + decoder_conv2 in one kernel: the pixels two of its strips share are accumulated atomically and are
    // zeroed here, ahead of the whole forward, so that no memset sits between two kernels chained by programmatic launch
    const bool fuse_dec = tc_on(dt) && w->dec2_w16 && w->dec1_b && w->dec2_b && tc_dec12_fused_enabled();
    if (!dry && fuse_dec && (rc = tc_dec12_zero_seams(res, B, Hc, Wc, st))) return rc;

    // ---- encoder
    if (!dry && (overlap || stack_flags)) {
        cudaError_t e = cudaMemsetAsync(sync_words, 0, sync_bytes, st);
        if (e != cudaSuccess) return cuda_fail(e, "memset tile flags");
    }
    if (!dry) {
        // conv1 fused into conv2 (its 64-channel output never reaches HBM) when the tensor-core path and the image pitch allow it.
        // "frame_chunk" = c > 0 runs {conv1+conv2, downsample} c frames at a time: the downsample then reads what conv2 just wrote while
        // (part of) it is still in the 126 MB L2 (one 720p map is 118 MB)
        const int chunk = (!fast && g_frame_chunk > 0 && g_frame_chunk < B) ? g_frame_chunk : B;
        for (int b0 = 0; b0 < B; b0 += chunk) {
            const int nb = min(chunk, B - b0);
            const void *xb = (const char *)x + (size_t)b0 * 3 * H * W * dtype_size(in_dtype);
            T *f1b = f1 + (size_t)b0 * H * W * 64, *f2b = f2 + (size_t)b0 * H * W * 64, *fdb = fd + (size_t)b0 * Hd * Wd * 64;
            rc = TU_TC_UNSUPPORTED;
            if (tc_on(dt) && w->conv1_w64) {
                g_prof_name = "conv1_conv2";
                prof_begin(st);
                rc = tc_conv12_fused(xb, in_dtype, (const bf16 *)w->conv1_w64, w->conv1_b, (const bf16 *)w->conv2_w, w->conv2_b, (bf16 *)f2b, nb, H, W, st);
                if (rc == TU_OK) prof_end(st, "conv1_conv2");
                else if (g_prof_open) { cudaEventDestroy(g_prof_open); g_prof_open = nullptr; }
                if (rc != TU_OK && rc != TU_TC_UNSUPPORTED) return rc;
            }
            if (rc == TU_TC_UNSUPPORTED) {
                TU_STEP("conv1", tu_stem_conv(xb, in_dtype, w->conv1_w, w->conv1_w64, w->conv1_b, f1b, dt, nb, H, W, stv));
                TU_STEP("conv2", tu_conv3x3_c64(f1b, w->conv2_w, w->conv2_b, f2b, dt, nb, H, W, 1, 1, 1, 0, stv));
            }
            if (!fast) TU_STEP("downsample", tu_conv3x3_c64(f2b, w->down_w, w->down_b, fdb, dt, nb, H, W, 2, 0, 1, 0, stv));
        }
    }

    // ---- FastTransformer branch A: sub-pixel upsample of feat, then 64->3 (+ReLU)
    float *upA = nullptr;
    if (fast) {
        const int slot = scale_slot(scale);
        const int nst = scale == 4 ? 2 : 1;
        const T *cur = f2;
        int ch = H, cw = W;
        const TuUpFold *fold = &w->upfold[slot];
        // fold the last stage with up1_conv when the folded filter is packed and the output row pitch suits TMA
        const int last_r = w->up1[slot][nst - 1].r;
        const int lw = nst == 2 ? W * w->up1[slot][0].r : W;
        const bool use_fold = g_fold_up1 && tc_on(dt) && fold->r == last_r && fold->w && (lw * last_r) % 4 == 0;
        for (int s = 0; s < nst; ++s) {
            const TuUpsamplerStage &sg = w->up1[slot][s];
            const int r = sg.r;
            if (use_fold && s == nst - 1) break;
            T *nxt = (T *)a.get((size_t)B * ch * r * cw * r * 64 * sizeof(T));
            if (!dry) TU_STEP("up1", tu_conv3x3_c64(cur, sg.w, sg.b, nxt, dt, B, ch, cw, 1, 0, r * r, r, stv));
            cur = nxt;
            ch *= r;
            cw *= r;
        }
        if (use_fold) {
            upA = (float *)a.get((size_t)B * 3 * ch * last_r * cw * last_r * sizeof(float));
            if (!dry) TU_STEP("up1_folded", tu_upfold_conv(cur, fold, upA, B, ch, cw, stv));
        } else {
            upA = (float *)a.get((size_t)B * 3 * ch * cw * sizeof(float));
            if (!dry) {
                g_prof_name = "up1_conv";
                prof_begin(st);
                rc = TU_TC_UNSUPPORTED;
                if (tc_on(dt) && g_head_stream) rc = tc_conv3x3_c64_to3_stream((const bf16 *)cur, (const bf16 *)w->up1conv_wst, w->up1conv_b16, upA, B, ch, cw, 1, st);
                if (rc == TU_TC_UNSUPPORTED) rc = tu_conv3x3_c64_to3(cur, dt, w->up1conv_w, w->up1conv_w16, nullptr, upA, B, ch, cw, 1, stv);
                prof_end(st, "up1_conv");
                if (rc) return rc;
            }
        }
    }

    // ---- tokens
    if (!dry) {
        if (window && (Ht % 8 || Wt % 8)) {
            cudaError_t e = cudaMemsetAsync(tok, 0, (size_t)Mtok * dim * sizeof(float), st);   // zero pad tokens
            if (e != cudaSuccess) return cuda_fail(e, "memset tokens");
        }
        TU_STEP("patch_embed", tu_patch_embed(fd, dt, w->embed_w, w->embed_b, w->pos_embed, tok, B, Hd, Wd, Ht, Wt, dim, window ? 1 : 0,
                                              fast ? 1 : 0, stv));
        const bool tc = tc_on(dt);
        g_prof_name = "transformer_blocks";
        prof_begin(st);
        rc = TU_TC_UNSUPPORTED;
        if (tc && window && dim == 128 && w->stack_w && g_use_stack)
            rc = tc_window_stack(tok, tok16, Mtok, w->n_blocks, (const bf16 *)w->stack_w, w->stack_p, w->stack_rel,
                                 overlap ? sync_words + 16 : nullptr, stack_flags ? sync_words + 16 + n_tok_tiles : nullptr, st);
        else if (tc && window && dim == 192 && w->stack_w && g_use_stack)
            rc = tc_window_stack192(tok, tok16, Mtok, w->n_blocks, (const bf16 *)w->stack_w, w->stack_p, w->stack_rel,
                                    overlap ? sync_words + 16 : nullptr, stack_flags ? sync_words + 16 + n_tok_tiles : nullptr, st);
        if (rc != TU_TC_UNSUPPORTED && rc != TU_OK) return rc;
        const bool stack_done = rc == TU_OK;
        for (int i = 0; i < w->n_blocks && !stack_done; ++i) {
            bf16 *x16 = (tc && i == w->n_blocks - 1) ? tok16 : nullptr;
            rc = TU_TC_UNSUPPORTED;
            if (tc && !window && w->stack_w) rc = resid_layer_fused(tok, w, i, Mtok, Ht * Wt, blk, bws, x16, st);      // two fused kernels + attention
            if (rc == TU_TC_UNSUPPORTED)
                rc = transformer_block_ex(tok, &w->blocks[i], Mtok, dim, heads, window ? 1 : 0, Ht * Wt, dt, blk, bws, x16, st);
            if (rc) return rc;
        }
        prof_end(st, "transformer_blocks");
        g_prof_name = "patch_unembed";
        prof_begin(st);
        rc = TU_TC_UNSUPPORTED;
        if (tc && overlap && stack_done && !g_prof_open)       // (the per-kernel profiling events would serialise the two kernels)
            rc = tc_patch_unembed(tok16, (const bf16 *)w->unembed_w, w->unembed_b, (const bf16 *)fd, Hd, Wd, (bf16 *)comb, B, Ht, Wt,
                                  Hc, Wc, dim, 1, sync_words, sync_words + 16, st);
        if (tc && rc == TU_TC_UNSUPPORTED)
            rc = tc_patch_unembed(tok16, (const bf16 *)w->unembed_w, w->unembed_b, (const bf16 *)fd, Hd, Wd, (bf16 *)comb, B, Ht, Wt,
                                  Hc, Wc, dim, window ? 1 : 0, nullptr, nullptr, st);
        if (rc == TU_TC_UNSUPPORTED)
            rc = tu_patch_unembed(tok, w->unembed_w, w->unembed_b, fd, Hd, Wd, comb, dt, B, Ht, Wt, Hc, Wc, dim, window ? 1 : 0, stv);
        prof_end(st, "patch_unembed");
        if (rc) return rc;
        // ---- decoder
        rc = TU_TC_UNSUPPORTED;
        if (fuse_dec) {
            g_prof_name = "decoder_fused";
            prof_begin(st);
            rc = tc_dec12_fused((const bf16 *)comb, (const bf16 *)w->dec1_w, w->dec1_b, (const bf16 *)w->dec2_w16, w->dec2_b, res, B, Hc, Wc, st);
            if (rc == TU_OK) prof_end(st, "decoder_fused");
            else if (g_prof_open) { cudaEventDestroy(g_prof_open); g_prof_open = nullptr; }
            if (rc != TU_OK && rc != TU_TC_UNSUPPORTED) return rc;
        }
        if (rc == TU_TC_UNSUPPORTED) {
        TU_STEP("decoder_conv1", tu_conv3x3_c64(comb, w->dec1_w, w->dec1_b, dec, dt, B, Hc, Wc, 1, 1, 1, 0, stv));
        {   // 64 -> 3 head: streaming kernel when packed and the row pitch suits its TMA stores, else the tile kernel
            g_prof_name = "decoder_conv2";
            prof_begin(st);
            rc = TU_TC_UNSUPPORTED;
            if (tc && g_head_stream) rc = tc_conv3x3_c64_to3_stream((const bf16 *)dec, (const bf16 *)w->dec2_wst, w->dec2_b16, res, B, Hc, Wc, 0, st);
            if (rc == TU_TC_UNSUPPORTED) rc = tu_conv3x3_c64_to3(dec, dt, w->dec2_w, w->dec2_w16, w->dec2_b, res, B, Hc, Wc, 0, stv);
            prof_end(st, "decoder_conv2");
            if (rc) return rc;
        }
        }
    }

    if (!fast) {
        if (!dry) {
            TU_STEP("bicubic_add_clamp", bicubic_add_clamp_alpha(x, in_dtype, H, W, res, Hc, Wc, img, img_dtype, B, outH, outW, clamp, aplane, st));
            TU_YUV_OUT();
        }
        return TU_OK;
    }
    // ---- FastTransformer branch B: sub-pixel upsample of the residual image, 3->3 conv, sum, clamp
    {
        const int slot = scale_slot(scale);
        const int nst = scale == 4 ? 2 : 1;
        const float *cur = res;
        int ch = H, cw = W;
        const bool fuse_tail = w->host_finconv_wb != nullptr;     // last sub-pixel stage + 3->3 conv + sum + clamp in one kernel
        for (int s = 0; s < nst; ++s) {
            const TuUpsamplerStage &sg = w->fin[slot][s];
            const int r = sg.r;
            if (fuse_tail && s == nst - 1) {
                if (!dry) {
                    if (ch * r != outH || cw * r != outW) {
                        set_error("tu: FastTransformer output buffer must be (scale*H, scale*W)");
                        return TU_ERR_ARG;
                    }
                    TU_STEP("final_upscale_conv_add", subpixel_conv_add_alpha(cur, (const float *)sg.w, sg.b, r, w->host_finconv_wb, upA, img,
                                                                              img_dtype, B, ch, cw, clamp, aplane, st));
                    TU_YUV_OUT();
                }
                return TU_OK;
            }
            float *nxt = (float *)a.get((size_t)B * 3 * ch * r * cw * r * sizeof(float));
            if (!dry) TU_STEP("final_upscale", tu_conv3x3_c3_ps(cur, (const float *)sg.w, sg.b, nxt, B, ch, cw, r, stv));
            cur = nxt;
            ch *= r;
            cw *= r;
        }
        if (!dry) {
            if (ch != outH || cw != outW) {
                set_error("tu: FastTransformer output buffer must be (scale*H, scale*W)");
                return TU_ERR_ARG;
            }
            TU_STEP("final_conv_add", tu_final_conv_add(cur, w->finconv_w, w->finconv_b, upA, img, img_dtype, B, ch, cw, clamp, stv));
            TU_YUV_OUT();
        }
    }
    return TU_OK;
#undef TU_YUV_OUT
}

}  // namespace tu

using namespace tu;

extern "C" int tu_version(void) { return 100; }
extern "C" const char *tu_last_error(void) { return g_err.c_str(); }
extern "C" int tu_bf16_uses_tcgen05(void) { return g_use_tc && tc_available(); }
extern "C" void tu_set_bf16_tcgen05(int enable) { g_use_tc = enable; }
extern "C" int tu_debug_set(const char *key, int value) {
    if (key && !strcmp(key, "tc_base_off_mode")) {
        tc_set_base_off_mode(value);
        return TU_OK;
    }
    if (key && !strcmp(key, "pdl")) {
        g_use_pdl = value;
        return TU_OK;
    }
    if (key && !strcmp(key, "conv_stream")) {
        tc_set_conv_stream(value);
        return TU_OK;
    }
    if (key && !strcmp(key, "conv_2cta")) {
        tc_set_conv_2cta(value);
        return TU_OK;
    }
    if (key && !strcmp(key, "unembed_overlap")) {
        g_unembed_overlap = value;
        return TU_OK;
    }
    if (key && !strcmp(key, "head_stream")) {
        g_head_stream = value;
        return TU_OK;
    }
    if (key && !strcmp(key, "fuse_conv12")) {
        tc_set_conv12_fused(value);
        return TU_OK;
    }
    if (key && !strcmp(key, "fold_up1")) {
        g_fold_up1 = value;
        return TU_OK;
    }
    if (key && !strcmp(key, "unembed_areuse")) {
        tc_set_unembed_areuse(value);
        return TU_OK;
    }
    if (key && !strcmp(key, "stack_split")) {
        tc_set_stack_split(value);
        return TU_OK;
    }
    if (key && !strcmp(key, "ga_shape")) {
        g_ga_shape = value;
        return TU_OK;
    }
    if (key && !strcmp(key, "stack_var")) {
        tc_set_stack_var(value);
        return TU_OK;
    }
    if (key && !strcmp(key, "embed_pair")) {
        tc_set_embed_pair(value);
        return TU_OK;
    }
    if (key && !strcmp(key, "bicubic_pair")) {
        g_bicubic_pair = value;
        return TU_OK;
    }
    if (key && !strcmp(key, "bicubic_tile")) {
        g_bicubic_tile = value;
        return TU_OK;
    }
    if (key && !strcmp(key, "fuse_dec12")) {
        tc_set_dec12_fused(value);
        return TU_OK;
    }
    if (key && !strcmp(key, "snake")) {
        tc_set_snake(value);
        return TU_OK;
    }
    if (key && !strcmp(key, "global_attn_tc")) {
        tc_set_global_attn(value);
        return TU_OK;
    }
    if (key && !strcmp(key, "resid_fused")) {
        tc_set_resid_fused(value);
        return TU_OK;
    }
    if (key && !strcmp(key, "frame_chunk")) {
        g_frame_chunk = value;
        return TU_OK;
    }
    if (key && !strcmp(key, "fused_stack")) {
        g_use_stack = value;
        return TU_OK;
    }
    set_error("tu: unknown debug key");
    return TU_ERR_ARG;
}
thread_local unsigned long long *tu::g_trace_buf = nullptr;
thread_local unsigned int tu::g_trace_cap = 0;
extern "C" int tu_debug_trace(void *device_buffer, unsigned int capacity_events) {
    tu::g_trace_buf = (unsigned long long *)device_buffer;
    tu::g_trace_cap = device_buffer ? capacity_events : 0;
    return TU_OK;
}
extern "C" long long tu_launch_count(void) { return g_launches.load(); }
extern "C" void tu_profile_enable(int on) { g_prof_on = on; }
// waits for the recorded events (the only calls in the library that wait on the device)
extern "C" int tu_profile_collect(const char *name, double *total_ms, int *launches) {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    double tot = 0.0;
    int n = 0;
    for (auto &pr : g_prof_events) {
        if (name && strcmp(name, pr.name)) continue;
        float ms = 0.f;
        if (cudaEventSynchronize(pr.b) == cudaSuccess && cudaEventElapsedTime(&ms, pr.a, pr.b) == cudaSuccess) {
            tot += ms;
            ++n;
        }
    }
    if (total_ms) *total_ms = tot;
    if (launches) *launches = n;
    return TU_OK;
}
extern "C" int tu_profile_report(char *buf, size_t cap) {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    std::vector<const char *> names;
    std::vector<double> ms;
    std::vector<int> cnt;
    for (auto &pr : g_prof_events) {
        float t = 0.f;
        if (cudaEventSynchronize(pr.b) != cudaSuccess || cudaEventElapsedTime(&t, pr.a, pr.b) != cudaSuccess) continue;
        size_t i = 0;
        for (; i < names.size(); ++i)
            if (!strcmp(names[i], pr.name)) break;
        if (i == names.size()) { names.push_back(pr.name); ms.push_back(0.0); cnt.push_back(0); }
        ms[i] += t;
        cnt[i] += 1;
    }
    std::string out;
    for (size_t i = 0; i < names.size(); ++i) {
        char line[160];
        snprintf(line, sizeof(line), "%s %.6f %d\n", names[i], ms[i], cnt[i]);
        out += line;
    }
    if (!buf || cap == 0) return (int)out.size() + 1;
    snprintf(buf, cap, "%s", out.c_str());
    return TU_OK;
}
extern "C" void tu_profile_reset(void) {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    for (auto &pr : g_prof_events) {
        cudaEventDestroy(pr.a);
        cudaEventDestroy(pr.b);
    }
    g_prof_events.clear();
}

extern "C" int tu_conv3x3_c64(const void *in, const void *w, const float *b, void *out, int dtype, int B, int H, int W,
                              int stride, int relu, int nchunk, int ps_r, void *stream) {
    TU_CHECK_ARG(in && w && out && B > 0 && H > 0 && W > 0, "conv3x3_c64: bad argument");
    TU_CHECK_ARG(stride == 1 || stride == 2, "conv3x3_c64: stride must be 1 or 2");
    TU_CHECK_ARG(nchunk >= 1 && (ps_r == 0 || (ps_r * ps_r == nchunk && stride == 1)), "conv3x3_c64: bad chunking");
    cudaStream_t st = (cudaStream_t)stream;
    if (tc_on(dtype)) {
        int rc = TU_TC_UNSUPPORTED;
        if (stride == 1) rc = tc_conv3x3_c64_stream((const bf16 *)in, (const bf16 *)w, b, (bf16 *)out, B, H, W, relu, nchunk, ps_r, st);
        if (rc == TU_TC_UNSUPPORTED && nchunk == 1 && ps_r == 0)
            rc = tc_conv3x3_c64_pair((const bf16 *)in, (const bf16 *)w, b, (bf16 *)out, B, H, W, stride, relu, st);
        if (rc == TU_TC_UNSUPPORTED)
            rc = tc_conv3x3_c64((const bf16 *)in, (const bf16 *)w, b, (bf16 *)out, B, H, W, stride, relu, nchunk, ps_r, st);
        if (rc != TU_TC_UNSUPPORTED) return rc;
    }
    if (dtype == TU_F32)
        return conv3x3_c64<float>((const float *)in, (const float *)w, b, (float *)out, B, H, W, stride, relu, nchunk, ps_r, st);
    if (dtype == TU_BF16)
        return conv3x3_c64<bf16>((const bf16 *)in, (const bf16 *)w, b, (bf16 *)out, B, H, W, stride, relu, nchunk, ps_r, st);
    TU_CHECK_ARG(false, "conv3x3_c64: bad dtype");
}

extern "C" int tu_conv3x3_c64_to3_stream(const void *in, const void *wst, const float *b16, float *out, int B, int H, int W, int relu,
                                         void *stream) {
    TU_CHECK_ARG(in && wst && b16 && out && B > 0 && H > 0 && W > 0, "conv3x3_c64_to3_stream: bad argument");
    TU_CHECK_ARG(tc_enabled(), "conv3x3_c64_to3_stream: tcgen05 kernels are unavailable or switched off");
    int rc = tc_conv3x3_c64_to3_stream((const bf16 *)in, (const bf16 *)wst, b16, out, B, H, W, relu, (cudaStream_t)stream);
    TU_CHECK_ARG(rc != TU_TC_UNSUPPORTED, "conv3x3_c64_to3_stream: unsupported alignment (W % 4 must be 0)");
    return rc;
}

extern "C" int tu_dec12_fused(const void *in, const void *w1, const float *b1, const void *w16, const float *b2, float *out, int B, int H,
                              int W, void *stream) {
    TU_CHECK_ARG(in && w1 && b1 && w16 && b2 && out && B > 0 && H > 0 && W > 0, "dec12_fused: bad argument");
    TU_CHECK_ARG(tc_enabled(), "dec12_fused: tcgen05 kernels are unavailable or switched off");
    int rc = tc_dec12_zero_seams(out, B, H, W, (cudaStream_t)stream);
    if (rc) return rc;
    rc = tc_dec12_fused((const bf16 *)in, (const bf16 *)w1, b1, (const bf16 *)w16, b2, out, B, H, W, (cudaStream_t)stream);
    TU_CHECK_ARG(rc != TU_TC_UNSUPPORTED, "dec12_fused: unsupported alignment or switched off");
    return rc;
}

extern "C" int tu_conv12_fused(const void *x, int in_dtype, const void *w64, const float *b1, const void *w2, const float *b2, void *out,
                               int B, int H, int W, void *stream) {
    TU_CHECK_ARG(x && w64 && b1 && w2 && out && B > 0 && H > 0 && W > 0, "conv12_fused: bad argument");
    TU_CHECK_ARG(in_dtype == TU_F32 || in_dtype == TU_BF16 || in_dtype == TU_F16 || in_dtype == TU_U8, "conv12_fused: bad input dtype");
    TU_CHECK_ARG(tc_enabled(), "conv12_fused: tcgen05 kernels are unavailable or switched off");
    int rc = tc_conv12_fused(x, in_dtype, (const bf16 *)w64, b1, (const bf16 *)w2, b2, (bf16 *)out, B, H, W, (cudaStream_t)stream);
    TU_CHECK_ARG(rc != TU_TC_UNSUPPORTED, "conv12_fused: unsupported alignment (image row pitch must be a multiple of 16 bytes) or switched off");
    return rc;
}

extern "C" int tu_upfold_conv(const void *in, const TuUpFold *f, float *out, int B, int H, int W, void *stream) {
    TU_CHECK_ARG(in && f && out && B > 0 && H > 0 && W > 0, "upfold_conv: bad argument");
    TU_CHECK_ARG(f->w && f->b && f->ring_w && f->ring_b && (f->r == 2 || f->r == 3 || f->r == 6), "upfold_conv: folded filter not packed");
    TU_CHECK_ARG(tc_enabled(), "upfold_conv: tcgen05 kernels are unavailable or switched off");
    TU_CHECK_ARG((long)B * 3 * H * f->r * W * f->r < (1L << 31), "upfold_conv: image too large for 32-bit indexing");
    int rc = tc_upfold((const bf16 *)in, f, out, B, H, W, (cudaStream_t)stream);
    TU_CHECK_ARG(rc != TU_TC_UNSUPPORTED, "upfold_conv: unsupported shape or alignment ((W*r) % 4 must be 0)");
    return rc;
}

extern "C" int tu_window_stack(float *tokens, const TuModelWeights *w, int M, void *stream) {
    TU_CHECK_ARG(tokens && w && M > 0 && M % 64 == 0, "window_stack: bad argument");
    TU_CHECK_ARG(w->stack_w && w->stack_p && w->stack_rel, "window_stack: the model has no fused-stack weights (bf16 WindowTransformer / FastTransformer only)");
    TU_CHECK_ARG(tc_enabled(), "window_stack: tcgen05 kernels are unavailable or switched off");
    cudaStream_t st = (cudaStream_t)stream;
    int rc = TU_TC_UNSUPPORTED;
    if (w->dim == 128) rc = tc_window_stack(tokens, nullptr, M, w->n_blocks, (const bf16 *)w->stack_w, w->stack_p, w->stack_rel, nullptr, nullptr, st);
    else if (w->dim == 192) rc = tc_window_stack192(tokens, nullptr, M, w->n_blocks, (const bf16 *)w->stack_w, w->stack_p, w->stack_rel, nullptr, nullptr, st);
    TU_CHECK_ARG(rc != TU_TC_UNSUPPORTED, "window_stack: unsupported shape (token count must be a multiple of 128)");
    return rc;
}

extern "C" int tu_resid_pre(const float *tokens, void *qkv, const TuModelWeights *w, int layer, int M, void *stream) {
    TU_CHECK_ARG(tokens && qkv && w && M > 0 && layer >= 0 && layer < w->n_blocks, "resid_pre: bad argument");
    TU_CHECK_ARG(w->model == TU_MODEL_RESIDUAL && w->dim == 128 && w->stack_w && w->stack_p,
                 "resid_pre: the model has no fused-layer weights (bf16 ResidualTransformer only)");
    TU_CHECK_ARG(tc_enabled(), "resid_pre: tcgen05 kernels are unavailable or switched off");
    int rc = tc_resid_pre(tokens, (bf16 *)qkv, M, layer, w->n_blocks, (const bf16 *)w->stack_w, w->stack_p, (cudaStream_t)stream);
    TU_CHECK_ARG(rc != TU_TC_UNSUPPORTED, "resid_pre: unsupported alignment (16-byte aligned tokens and qkv) or switched off");
    return rc;
}

extern "C" int tu_resid_post(float *tokens, const void *att, const TuModelWeights *w, int layer, int M, void *stream) {
    TU_CHECK_ARG(tokens && att && w && M > 0 && layer >= 0 && layer < w->n_blocks, "resid_post: bad argument");
    TU_CHECK_ARG(w->model == TU_MODEL_RESIDUAL && w->dim == 128 && w->stack_w && w->stack_p,
                 "resid_post: the model has no fused-layer weights (bf16 ResidualTransformer only)");
    TU_CHECK_ARG(tc_enabled(), "resid_post: tcgen05 kernels are unavailable or switched off");
    int rc = tc_resid_post(tokens, nullptr, (const bf16 *)att, M, layer, w->n_blocks, (const bf16 *)w->stack_w, w->stack_p,
                           (cudaStream_t)stream);
    TU_CHECK_ARG(rc != TU_TC_UNSUPPORTED, "resid_post: unsupported alignment (16-byte aligned tokens and att) or switched off");
    return rc;
}

extern "C" int tu_patch_embed(const void *feat, int dtype, const void *w, const float *b, const float *pos_embed,
                              float *tokens, int B, int H, int W, int Ht, int Wt, int dim, int window, int reflect,
                              void *stream) {
    TU_CHECK_ARG(feat && w && b && tokens && B > 0 && Ht > 0 && Wt > 0, "patch_embed: bad argument");
    TU_CHECK_ARG(reflect ? (8 * Ht - H < 8 && 8 * Wt - W < 8 && 8 * Ht >= H && 8 * Wt >= W) : (8 * Ht <= H && 8 * Wt <= W),
                 "patch_embed: token grid does not match the feature map");
    TU_CHECK_ARG(!reflect || ((8 * Ht - H) < H && (8 * Wt - W) < W), "patch_embed: reflect pad larger than the input");
    cudaStream_t st = (cudaStream_t)stream;
    if (tc_on(dtype) && (!reflect || (H % 8 == 0 && W % 8 == 0))) {
        int rc = tc_patch_embed_pair((const bf16 *)feat, (const bf16 *)w, b, pos_embed, tokens, B, H, W, Ht, Wt, dim, window, st);
        if (rc == TU_TC_UNSUPPORTED)
            rc = tc_patch_embed((const bf16 *)feat, (const bf16 *)w, b, pos_embed, tokens, B, H, W, Ht, Wt, dim, window, st);
        if (rc != TU_TC_UNSUPPORTED) return rc;
    }
    if (dtype == TU_F32)
        return patch_embed<float>((const float *)feat, (const float *)w, b, pos_embed, tokens, B, H, W, Ht, Wt, dim, window, reflect, st);
    if (dtype == TU_BF16)
        return patch_embed<bf16>((const bf16 *)feat, (const bf16 *)w, b, pos_embed, tokens, B, H, W, Ht, Wt, dim, window, reflect, st);
    TU_CHECK_ARG(false, "patch_embed: bad dtype");
}

extern "C" int tu_patch_unembed(const float *tokens, const void *w, const float *b, const void *skip, int skipH, int skipW,
                                void *out, int dtype, int B, int Ht, int Wt, int Hc, int Wc, int dim, int window,
                                void *stream) {
    TU_CHECK_ARG(tokens && w && b && skip && out && B > 0 && Ht > 0 && Wt > 0, "patch_unembed: bad argument");
    TU_CHECK_ARG(Hc <= skipH && Wc <= skipW && Hc <= 8 * Ht && Wc <= 8 * Wt, "patch_unembed: crop larger than its sources");
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == TU_F32)
        return patch_unembed<float>(tokens, (const float *)w, b, (const float *)skip, skipH, skipW, (float *)out, B, Ht, Wt, Hc, Wc, dim, window, st);
    if (dtype == TU_BF16)
        return patch_unembed<bf16>(tokens, (const bf16 *)w, b, (const bf16 *)skip, skipH, skipW, (bf16 *)out, B, Ht, Wt, Hc, Wc, dim, window, st);
    TU_CHECK_ARG(false, "patch_unembed: bad dtype");
}

static int check_forward_args(const TuModelWeights *w, int B, int H, int W, int outH, int outW, int compute_dtype) {
    TU_CHECK_ARG(w, "forward: null weights");
    TU_CHECK_ARG(w->model >= 0 && w->model <= 2, "forward: bad model id");
    TU_CHECK_ARG(B > 0 && H > 0 && W > 0 && outH > 0 && outW > 0, "forward: bad shape");
    TU_CHECK_ARG(compute_dtype == TU_F32 || compute_dtype == TU_BF16, "forward: bad compute dtype");
    TU_CHECK_ARG((long)B * H * W < (1L << 31) / 64 * 16, "forward: batch too large for 32-bit pixel indexing");
    return TU_OK;
}

extern "C" size_t tu_forward_workspace_bytes(int model, int B, int H, int W, int outH, int outW, int scale,
                                             int compute_dtype) {
    TuModelWeights w;
    memset(&w, 0, sizeof(w));
    w.model = model;
    w.dim = model == TU_MODEL_FAST ? 192 : 128;
    w.heads = w.dim / 16;
    w.n_blocks = model == TU_MODEL_FAST ? 6 : 8;
    for (int s = 0; s < 4; ++s) {
        const int r0 = s == 0 ? 2 : s == 1 ? 3 : s == 2 ? 2 : 6;
        w.up1[s][0].r = w.fin[s][0].r = r0;
        w.up1[s][1].r = w.fin[s][1].r = 2;
    }
    if (check_forward_args(&w, B, H, W, outH, outW, compute_dtype)) return 0;
    Arena a{nullptr, 0, 0, true};
    int rc = compute_dtype == TU_F32
                 ? forward_impl<float>(&w, nullptr, nullptr, TU_F32, nullptr, nullptr, TU_F32, B, H, W, outH, outW, scale, 1, a, 0)
                 : forward_impl<bf16>(&w, nullptr, nullptr, TU_F32, nullptr, nullptr, TU_F32, B, H, W, outH, outW, scale, 1, a, 0);
    return rc == TU_OK ? a.off : 0;
}

extern "C" size_t tu_forward_workspace_bytes_for(const TuModelWeights *w, int B, int H, int W, int outH, int outW, int scale,
                                                 int compute_dtype) {
    if (check_forward_args(w, B, H, W, outH, outW, compute_dtype)) return 0;
    Arena a{nullptr, 0, 0, true};
    int rc = compute_dtype == TU_F32
                 ? forward_impl<float>(w, nullptr, nullptr, TU_F32, nullptr, nullptr, TU_F32, B, H, W, outH, outW, scale, 1, a, 0)
                 : forward_impl<bf16>(w, nullptr, nullptr, TU_F32, nullptr, nullptr, TU_F32, B, H, W, outH, outW, scale, 1, a, 0);
    return rc == TU_OK ? a.off : 0;
}

// 4:2:0 codes: TU_U8 | TU_LAYOUT_NV12 [| TU_YUV_BT601] [| TU_YUV_FULL_RANGE], or TU_U16 | TU_LAYOUT_P010 [| TU_YUV_BT601 or
// TU_YUV_BT2020] [| TU_YUV_FULL_RANGE].  TU_U16 is a P010 word and nothing else.  Such frames have an even height and width.
// 4-byte frames: exactly TU_U8 | TU_LAYOUT_RGBA or TU_U8 | TU_LAYOUT_BGRA.  Other codes have a layout nibble below 4 and no colour bit.
static bool plain_code(int d) {
    const int nib = (d >> 8) & 0xF;
    return dtype_is_px4(d) || (!(d & (TU_YUV_BT601 | TU_YUV_BT2020 | TU_YUV_FULL_RANGE)) && nib < 4 && dtype_base(d) != TU_U16);
}
static int check_yuv420_codes(int in_dtype, int out_dtype, int H, int W, int outH, int outW) {
    const bool in420 = dtype_is_yuv420(in_dtype), out420 = dtype_is_yuv420(out_dtype);
    for (int d : {in_dtype, out_dtype})
        TU_CHECK_ARG(dtype_is_px4(d) || !layout_is_px4((d >> 8) & 0xF),
                     "forward: TU_LAYOUT_RGBA / TU_LAYOUT_BGRA are for uint8 frames (TU_U8) only, without colour bits");
    TU_CHECK_ARG(in420 || plain_code(in_dtype),
                 "forward: TU_LAYOUT_NV12 is for uint8 frames (TU_U8), TU_LAYOUT_P010 for 16-bit words (TU_U16, P010 only), and the "
                 "colour bits TU_YUV_* go with them only (TU_YUV_BT2020 with P010, never with TU_YUV_BT601) (input)");
    TU_CHECK_ARG(out420 || plain_code(out_dtype),
                 "forward: TU_LAYOUT_NV12 is for uint8 frames (TU_U8), TU_LAYOUT_P010 for 16-bit words (TU_U16, P010 only), and the "
                 "colour bits TU_YUV_* go with them only (TU_YUV_BT2020 with P010, never with TU_YUV_BT601) (output)");
    TU_CHECK_ARG(!in420 || (H % 2 == 0 && W % 2 == 0),
                 std::string("forward: ") + (dtype_is_p010(in_dtype) ? "P010" : "NV12") + " input frames need an even height and width");
    TU_CHECK_ARG(!out420 || (outH % 2 == 0 && outW % 2 == 0),
                 std::string("forward: ") + (dtype_is_p010(out_dtype) ? "P010" : "NV12") + " output frames need an even height and width");
    return TU_OK;
}

extern "C" size_t tu_forward_workspace_bytes_io(const TuModelWeights *w, int B, int H, int W, int outH, int outW, int scale,
                                                int compute_dtype, int in_dtype, int out_dtype) {
    if (check_forward_args(w, B, H, W, outH, outW, compute_dtype) || check_yuv420_codes(in_dtype, out_dtype, H, W, outH, outW)) return 0;
    // only the NV12 / P010 sides and a 4-byte pair of sides (its alpha plane) change the arena; every other code sizes exactly as
    // tu_forward_workspace_bytes_for
    const bool alpha_io = dtype_is_px4(in_dtype) && dtype_is_px4(out_dtype);
    in_dtype = dtype_is_yuv420(in_dtype) || alpha_io ? in_dtype : TU_F32;
    out_dtype = dtype_is_yuv420(out_dtype) || alpha_io ? out_dtype : TU_F32;
    Arena a{nullptr, 0, 0, true};
    int rc = compute_dtype == TU_F32
                 ? forward_impl<float>(w, nullptr, nullptr, in_dtype, nullptr, nullptr, out_dtype, B, H, W, outH, outW, scale, 1, a, 0)
                 : forward_impl<bf16>(w, nullptr, nullptr, in_dtype, nullptr, nullptr, out_dtype, B, H, W, outH, outW, scale, 1, a, 0);
    return rc == TU_OK ? a.off : 0;
}

extern "C" int tu_forward_planes(const TuModelWeights *w, const void *x, const TuFramePlanes *x_frames, int in_dtype, void *out,
                                 const TuFramePlanes *out_frames, int out_dtype, int B, int H, int W, int outH, int outW, int scale,
                                 int compute_dtype, int clamp, void *workspace, size_t workspace_bytes, void *stream) {
    int rc = check_forward_args(w, B, H, W, outH, outW, compute_dtype);
    if (rc) return rc;
    TU_CHECK_ARG((x || x_frames) && (out || out_frames) && workspace, "forward: null buffer");
    TU_CHECK_ARG(!(x && x_frames), "forward: give the input as either x or x_frames, not both");
    TU_CHECK_ARG(!(out && out_frames), "forward: give the output as either out or out_frames, not both");
    if ((rc = check_yuv420_codes(in_dtype, out_dtype, H, W, outH, outW))) return rc;
    TU_CHECK_ARG(!x_frames || dtype_is_yuv420(in_dtype), "forward: x_frames (frame planes) are for NV12 / P010 input only");
    TU_CHECK_ARG(!out_frames || dtype_is_yuv420(out_dtype), "forward: out_frames (frame planes) are for NV12 / P010 output only");
    // every descriptor is checked here, before the first kernel of the forward is enqueued
    if (x_frames && (rc = check_yuv420_planes(x_frames, in_dtype, B, H, W, "forward: x_frames"))) return rc;
    if (out_frames && (rc = check_yuv420_planes(out_frames, out_dtype, B, outH, outW, "forward: out_frames"))) return rc;
    {
        const int ib = dtype_base(in_dtype), ob = dtype_base(out_dtype);
        const int il = dtype_is_yuv420(in_dtype) ? 0 : dtype_layout(in_dtype), ol = dtype_is_yuv420(out_dtype) ? 0 : dtype_layout(out_dtype);
        // (TU_U16 has passed check_yuv420_codes only as a P010 word)
        TU_CHECK_ARG((ib == TU_F32 || ib == TU_BF16 || ib == TU_F16 || ib == TU_U8 || ib == TU_U16) &&
                         (ob == TU_F32 || ob == TU_BF16 || ob == TU_F16 || ob == TU_U8 || ob == TU_U16),
                     "forward: bad i/o dtype");
        TU_CHECK_ARG((il == 0 || (ib == TU_U8 && layout_is_interleaved(il))) && (ol == 0 || (ob == TU_U8 && layout_is_interleaved(ol))),
                     "forward: interleaved layouts (TU_LAYOUT_HWC / TU_LAYOUT_HWC_BGR / TU_LAYOUT_RGBA / TU_LAYOUT_BGRA) are for uint8 frames");
        TU_CHECK_ARG(!layout_is_px4(ol) || (reinterpret_cast<uintptr_t>(out) & 3) == 0, "forward: a 4-byte (RGBA / BGRA) output must be 4-byte aligned");
    }
    TU_CHECK_ARG(w->blocks && w->n_blocks > 0 && w->dim == w->heads * 16, "forward: bad transformer configuration");
    // size pass, then the real pass
    Arena dry{nullptr, 0, 0, true};
    rc = compute_dtype == TU_F32
             ? forward_impl<float>(w, x, x_frames, in_dtype, out, out_frames, out_dtype, B, H, W, outH, outW, scale, clamp, dry, 0)
             : forward_impl<bf16>(w, x, x_frames, in_dtype, out, out_frames, out_dtype, B, H, W, outH, outW, scale, clamp, dry, 0);
    if (rc) return rc;
    if (dry.off > workspace_bytes) {
        set_error("tu: forward workspace too small: need " + std::to_string(dry.off) + " bytes");
        return TU_ERR_WORKSPACE;
    }
    Arena a{(char *)workspace, 0, workspace_bytes, false};
    cudaStream_t st = (cudaStream_t)stream;
    return compute_dtype == TU_F32
               ? forward_impl<float>(w, x, x_frames, in_dtype, out, out_frames, out_dtype, B, H, W, outH, outW, scale, clamp, a, st)
               : forward_impl<bf16>(w, x, x_frames, in_dtype, out, out_frames, out_dtype, B, H, W, outH, outW, scale, clamp, a, st);
}

extern "C" int tu_forward(const TuModelWeights *w, const void *x, int in_dtype, void *out, int out_dtype, int B, int H,
                          int W, int outH, int outW, int scale, int compute_dtype, int clamp, void *workspace,
                          size_t workspace_bytes, void *stream) {
    return tu_forward_planes(w, x, nullptr, in_dtype, out, nullptr, out_dtype, B, H, W, outH, outW, scale, compute_dtype, clamp, workspace,
                             workspace_bytes, stream);
}
