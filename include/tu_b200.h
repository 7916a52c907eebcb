/*
 * tu_b200.h — C ABI of libtu_b200.so, the B200 (sm_100a) engine for the forward pass of
 * TransformerUpscaler's models.  This is the drop-in boundary for the hot path: everything the
 * reference's `models/<Name>/model.py::TransformerModel.forward` computes through torch ops
 * (reference: models/WindowTransformer/model.py:224-305, models/FastTransformer/model.py:231-327,
 * models/ResidualTransformer/model.py:114-165) is reachable through these entry points.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless named host_*;
 *   - the caller owns every buffer; the library never allocates or frees device memory, never
 *     synchronises the device, and enqueues all work on `stream` (a cudaStream_t passed as void*);
 *   - return value 0 = success, negative = error; tu_last_error() gives the message (thread-local);
 *   - dtype codes: TU_F32 = 0, TU_BF16 = 1, TU_U8 = 2 and TU_F16 = 3 (both image input / output only), TU_U16 = 4 (P010,
 *     P210, yuv444p16 and the TU_YUV_LSB10 frames only);
 *   - activations inside the engine are NHWC (64 channels); images at the boundary are NCHW, like
 *     the reference's tensors.
 */
#ifndef TU_B200_H
#define TU_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TU_F32 0
#define TU_BF16 1
#define TU_U8 2   /* image I/O only (in_dtype / out_dtype of tu_forward, tu_stem_conv, tu_bicubic_add_clamp,        */
                  /* tu_final_conv_add): uint8 frames, x/255 on read (ToTensor), trunc(clamp(v*255,0,255)) on write  */
#define TU_F16 3  /* image I/O only (in_dtype / out_dtype of tu_forward, tu_stem_conv, tu_conv12_fused, tu_bicubic_add_clamp,  */
                  /* tu_subpixel_conv_add, tu_final_conv_add, tu_resize_bilinear_aa[_to]); never a compute dtype: an fp16    */
                  /* model runs on the TU_BF16 (or TU_F32) path.  Read exactly into fp32 registers; the fp32 result is        */
                  /* rounded to fp16 once, at the store, so fp16 output == (the fp32-output call on the same values).half() */

/* uint8 frame layouts (OR-ed into TU_U8 for the image input / output of tu_forward, and for the output of tu_bicubic_add_clamp,
 * tu_subpixel_conv_add and tu_resize_bilinear_aa_to): planar CHW is the default (the reference's tensors); HWC is what PIL /
 * OpenCV frames are (inference.py:65-70: ToTensor reads HWC RGB); HWC_BGR reverses the channel order on the way
 * (app_overlay.py:382-386: permute(1,2,0) then [..., [2,1,0]]).  (B,H,W,3) uint8 either way. */
#define TU_LAYOUT_HWC 0x100
#define TU_LAYOUT_HWC_BGR 0x200
#define TU_U8_HWC (TU_U8 | TU_LAYOUT_HWC)
#define TU_U8_HWC_BGR (TU_U8 | TU_LAYOUT_HWC_BGR)
/* 32-bit pixels with an alpha byte (OR-ed into TU_U8 for the image input and / or output of tu_forward, the output of
 * tu_bicubic_add_clamp, tu_subpixel_conv_add and tu_resize_bilinear_aa_to[_alpha], and the input of tu_frames_to_planar and
 * tu_resample_alpha): (B,H,W,4) uint8, bytes R G B A (TU_LAYOUT_RGBA) or B G R A (TU_LAYOUT_BGRA: DXGI_FORMAT_B8G8R8A8_UNORM, what
 * screen capture returns).  Alpha is straight (not premultiplied).  R, G, B are read and written exactly as TU_LAYOUT_HWC /
 * TU_LAYOUT_HWC_BGR read and write them; the alpha bytes never reach the network.  A 4-byte output buffer must be 4-byte aligned.
 * The alpha byte of an output pixel is the input alpha resampled to the output size when the input is 4-byte too (tu_resample_alpha),
 * 255 otherwise; a 4-byte input going to an output without alpha loses its alpha.  TU_U8 only; never with colour bits.
 * The layout bits 8..11 are an enumeration: 0 CHW, 1 HWC, 2 HWC_BGR, 3 RGBA, 4 NV12, 5 BGRA, 6 YUV420P, 7 YUV444P, 8 P010, 9 YUV422P,
 * 10 NV16, 11 YUYV, 12 UYVY. */
#define TU_LAYOUT_RGBA 0x300
#define TU_LAYOUT_BGRA 0x500
#define TU_U8_RGBA (TU_U8 | TU_LAYOUT_RGBA)
#define TU_U8_BGRA (TU_U8 | TU_LAYOUT_BGRA)
/* NV12 video frames (OR-ed into TU_U8 for the image input and / or output of tu_forward, and the code of tu_nv12_to_rgb /
 * tu_rgb_to_nv12): one uint8 buffer of (3H/2) x W bytes per frame, (B, 3H/2, W) for a batch.  Rows 0..H-1 are the Y plane, the next
 * H/2 rows hold interleaved chroma pairs (U first) of the 4:2:0 "type 0" siting: chroma co-sited with even luma columns, midway
 * between luma rows 2i and 2i+1.  H and W must be even.  The colour bits below are valid with TU_LAYOUT_NV12 only, and the input and
 * output codes carry their own; neither bit = BT.709 limited range.  The frame is converted to / from planar fp16 RGB (the TU_F16
 * image I/O path) at both ends of the forward. */
#define TU_LAYOUT_NV12 0x400
#define TU_YUV_BT601 0x1000         /* BT.601 matrix (Kr, Kb = 0.299, 0.114) instead of BT.709 (0.2126, 0.0722) */
#define TU_YUV_FULL_RANGE 0x2000    /* full range (Y, C in 0..255) instead of limited (Y 16..235, C 16..240) */
#define TU_U8_NV12 (TU_U8 | TU_LAYOUT_NV12)
/* P010 video frames (10-bit 4:2:0; TU_U16 | TU_LAYOUT_P010 for the image input and / or output of tu_forward, and the code of
 * tu_p010_to_rgb / tu_rgb_to_p010): one buffer of (3H/2) x W little-endian uint16 words per frame, (B, 3H/2, W) for a batch, laid
 * out and sited like NV12 (Y plane, then H/2 rows of interleaved (U, V) pairs, U first; H and W even).  A word holds its 10-bit
 * code in the HIGH 10 bits, as video decoders write it and encoders read it: the code is word >> 6 on read (the low 6 bits are
 * ignored) and code << 6 on write (the low 6 bits are zero).  TU_U16 is valid with TU_LAYOUT_P010 only, and never a compute dtype.
 * The colour bits: TU_YUV_BT601 or TU_YUV_BT2020 (not both), TU_YUV_FULL_RANGE; none = BT.709 limited range.  Limited range is
 * Y 64..940, C 64..960; full range (BT.2100) is Y, C 0..1023.  The frame is converted to / from planar fp32 RGB (the TU_F32 image
 * I/O path) at both ends of the forward: fp16 would move a 10-bit output code by one on many bright samples.  RGB values outside
 * [0, 1] are clamped on the way in, which matters for wide-gamut BT.2020 content. */
#define TU_U16 4
#define TU_LAYOUT_P010 0x800
#define TU_YUV_BT2020 0x4000        /* BT.2020 non-constant-luminance matrix (Kr, Kb = 0.2627, 0.0593); with TU_LAYOUT_P010 only */
#define TU_U16_P010 (TU_U16 | TU_LAYOUT_P010)
/* Planar YUV frames: three separate planes Y, U, V (FFmpeg's yuv420p / yuv444p / yuv444p16, NVDEC's YUV444 / YUV444_16Bit surfaces)
 * for the image input and / or output of tu_forward / tu_forward_frames, and the code of tu_yuvp_to_rgb / tu_rgb_to_yuvp.
 *   TU_U8 | TU_LAYOUT_YUV420P (I420): one uint8 buffer of 3HW/2 bytes per frame, (B, 3H/2, W) for a batch: the Y plane (H x W), then
 *        the U plane (H/2 x W/2), then the V plane (H/2 x W/2), each row-major and contiguous.  H and W even; sited, filtered and
 *        converted exactly as NV12 (the results are bitwise those of the NV12 frame with U and V interleaved).
 *   TU_U8 | TU_LAYOUT_YUV444P: (B, 3, H, W) uint8, planes Y, U, V at full resolution; any H and W.
 *   TU_U16 | TU_LAYOUT_YUV444P (yuv444p16): (B, 3, H, W) little-endian uint16 words with the 10-bit code in the HIGH 10 bits, as P010
 *        (word >> 6 on read, code << 6 on write); any H and W.
 * Colour bits: TU_YUV_BT601 and TU_YUV_FULL_RANGE on each; TU_YUV_BT2020 (not with TU_YUV_BT601) on yuv444p16 only.  8-bit frames
 * convert through planar fp16 RGB, yuv444p16 through planar fp32 RGB.  4:4:4 has no chroma filter: each pixel is converted with its own
 * (U, V), by NV12's / P010's formulas (u' = (U - mid) / cs, ...; Cb', Cr' from the pixel's own R, G, B).  Buffers and planes need the
 * alignment of their accesses: 2 bytes for a yuv420p Y plane and its pitch (a pair of luma samples is one access), 2 bytes for every
 * yuv444p16 plane and pitch; U / V planes of yuv420p and every yuv444p plane may sit at any address.  The 4:4:4 kernels move four
 * samples per access where a row's four samples are 4-sample aligned (planes and pitches that are multiples of 4 samples, or dense
 * frames) and single samples elsewhere. */
#define TU_LAYOUT_YUV420P 0x600
#define TU_LAYOUT_YUV444P 0x700
#define TU_U8_YUV420P (TU_U8 | TU_LAYOUT_YUV420P)
#define TU_U8_YUV444P (TU_U8 | TU_LAYOUT_YUV444P)
#define TU_U16_YUV444P16 (TU_U16 | TU_LAYOUT_YUV444P)
/* 4:2:2 frames (chroma at full height and half width, co-sited with the even luma columns of every row: MPEG-2 / H.264 4:2:2 siting)
 * and LSB-aligned 10-bit planar frames, for the image input and / or output of tu_forward / tu_forward_frames:
 *   TU_U8 | TU_LAYOUT_YUV422P (yuv422p, MJPEG's yuvj422p with full-range BT.601): (B, 2H, W) uint8: the Y plane (H x W), then the U and V
 *        planes (H x W/2 each); surfaces are TuFramePlanes3.
 *   TU_U8 | TU_LAYOUT_NV16 (nv16): (B, 2H, W) uint8: the Y plane, then H rows of W/2 interleaved (U, V) pairs; surfaces are TuFramePlanes.
 *   TU_U16 | TU_LAYOUT_NV16 (p210, P216 holding 10-bit content): as nv16 with 16-bit words, the code in the HIGH 10 bits as P010.
 *   TU_YUV_LSB10, OR-ed into TU_U16 with one of the planar layouts: FFmpeg's yuv420p10le ((B, 3H/2, W), as yuv420p), yuv422p10le
 *        ((B, 2H, W), as yuv422p) and yuv444p10le ((B, 3, H, W), as yuv444p16): the 10-bit code in the LOW 10 bits of each little-endian
 *        word.  A word above 1023 reads as 1023 (a stray high bit saturates); a write stores the code with the top 6 bits zero.  Valid
 *        with TU_U16 and TU_LAYOUT_YUV420P / TU_LAYOUT_YUV422P / TU_LAYOUT_YUV444P only.  TU_U16 | TU_LAYOUT_YUV420P and TU_U16 |
 *        TU_LAYOUT_YUV422P without it are TU_ERR_ARG; TU_U16 | TU_LAYOUT_YUV444P without it is yuv444p16.
 * Colour bits: 8-bit codes take NV12's, 16-bit codes P010's (TU_YUV_BT2020 allowed, never with TU_YUV_BT601) and its 10-bit offsets and
 * scales.  8-bit frames convert through planar fp16 RGB, 16-bit frames through planar fp32 RGB.  4:2:2 needs an even W (any H), yuv420p10le
 * an even H and W, yuv444p10le takes any size.  4:2:2 is converted with the NV12 formulas on one row instead of a row pair:
 *   to RGB:  column 2j takes C[j], column 2j+1 (C[j] + C[j+1]) / 2 (j+1 clamped to W/2 - 1), then the NV12 per-pixel sequence;
 *   to YUV:  Y' per pixel as NV12; per channel bar = ((P[2j-1] + 2 P[2j]) + P[2j+1]) * 0.25 (column 2j-1 clamped at 0), Cb', Cr' from
 *            bar as NV12.  An image whose rows come in equal pairs gives chroma rows 2i and 2i+1 equal to NV12 chroma row i.
 * Alignment: a pair of luma samples is one access, so the Y plane and its pitch of nv16 / yuv422p are 2-byte and of the 16-bit 4:2:0 /
 * 4:2:2 codes 4-byte aligned; an nv16 / p210 (U, V) pair is one access too (2 / 4 bytes); every other 16-bit plane is 2-byte aligned. */
#define TU_LAYOUT_YUV422P 0x900
#define TU_LAYOUT_NV16 0xA00
#define TU_YUV_LSB10 0x10000       /* bit 16 (bit 15, 0x8000, is a flag of no code) */
#define TU_U8_YUV422P (TU_U8 | TU_LAYOUT_YUV422P)
#define TU_U8_NV16 (TU_U8 | TU_LAYOUT_NV16)
#define TU_U16_P210 (TU_U16 | TU_LAYOUT_NV16)
#define TU_U16_YUV420P10 (TU_U16 | TU_LAYOUT_YUV420P | TU_YUV_LSB10)
#define TU_U16_YUV422P10 (TU_U16 | TU_LAYOUT_YUV422P | TU_YUV_LSB10)
#define TU_U16_YUV444P10 (TU_U16 | TU_LAYOUT_YUV444P | TU_YUV_LSB10)
/* Packed 4:2:2 frames (luma and chroma interleaved in one plane, as webcams, capture cards and D3D11 / VAAPI decoders hand them out), for
 * the image input and / or output of tu_forward / tu_forward_frames and the code of tu_packed422_to_rgb / tu_rgb_to_packed422:
 *   TU_U8 | TU_LAYOUT_YUYV (yuyv422, YUY2): (B, H, W, 2) uint8, each row W/2 macropixels of the bytes Y0 U Y1 V.
 *   TU_U8 | TU_LAYOUT_UYVY (uyvy422, UYVY, DeckLink's 8-bit YUV): (B, H, W, 2) uint8, macropixels U Y0 V Y1.
 *   TU_U16 | TU_LAYOUT_YUYV (y210, DXGI_FORMAT_Y210): (B, H, W, 2) little-endian uint16 words Y0 U Y1 V, the 10-bit code in the HIGH
 *        10 bits as P010 (word >> 6 on read: the low 6 bits are ignored; code << 6 on write: the low 6 bits are zero).
 * Every other code with these layouts is TU_ERR_ARG (TU_U16 | TU_LAYOUT_UYVY, float dtypes, TU_YUV_LSB10).  Colour bits: the 8-bit codes
 * take NV12's, y210 P010's (TU_YUV_BT2020 allowed, never with TU_YUV_BT601).  A packed frame holds the samples of an nv16 (8-bit) or p210
 * (y210) frame -- macropixel j of row i is Y[i][2j], Y[i][2j+1], U[i][j], V[i][j] -- and converts bitwise as that frame does, in both
 * directions: 4:2:2 siting and formulas as above, planar fp16 RGB for the 8-bit codes and planar fp32 RGB for y210.  W even, any H.
 * A macropixel is one access: the buffer (dense) or each frame's data pointer and pitch (TuFramePacked) are multiples of 4 bytes (8-bit)
 * or 8 bytes (y210).  A write touches only the 2W samples of each row. */
#define TU_LAYOUT_YUYV 0xB00
#define TU_LAYOUT_UYVY 0xC00
#define TU_U8_YUYV422 (TU_U8 | TU_LAYOUT_YUYV)
#define TU_U8_UYVY422 (TU_U8 | TU_LAYOUT_UYVY)
#define TU_U16_Y210 (TU_U16 | TU_LAYOUT_YUYV)

#define TU_OK 0
#define TU_ERR_ARG (-1)      /* bad argument (shape / dtype / null pointer)              */
#define TU_ERR_SCALE (-2)    /* FastTransformer scale not in {2,3,4,6} (utils.py:96-97)   */
#define TU_ERR_TOKENS (-3)   /* ResidualTransformer token count != 3600 (model.py:140)    */
#define TU_ERR_WORKSPACE (-4)/* workspace too small                                       */
#define TU_ERR_CUDA (-5)     /* a CUDA launch failed                                      */

#define TU_MODEL_WINDOW 0
#define TU_MODEL_FAST 1
#define TU_MODEL_RESIDUAL 2

int tu_version(void);
const char *tu_last_error(void);
/* 1 if the tcgen05 (tensor-core) kernels are used for compute dtype TU_BF16, 0 if the CUDA-core path. */
int tu_bf16_uses_tcgen05(void);
void tu_set_bf16_tcgen05(int enable);
/* number of kernels this library has launched in the calling process (monotonic) */
long long tu_launch_count(void);
/* Measurement hook for bench.py: tu_profile_enable(1) brackets the dominant kernel ("conv2") of every tu_forward with CUDA
 * events on the caller's stream (two event records per forward: cheap enough for the timed region); tu_profile_enable(2)
 * brackets EVERY kernel, tagged with the reference op it implements ("conv1", "conv2" (or "conv1_conv2" when fused), "downsample", "patch_embed",
 * "transformer_blocks", "patch_unembed", "decoder_conv1", "decoder_conv2", "bicubic_add_clamp", "up1", "up1_conv",
 * "final_upscale", "final_conv_add", and "nv12_to_rgb" / "rgb_to_nv12" at an NV12 end, "p010_to_rgb" / "rgb_to_p010" at a P010 end, "yuv420p_to_rgb" / "rgb_to_yuv420p", "yuv444p_to_rgb" / "rgb_to_yuv444p", "yuv444p16_to_rgb" / "rgb_to_yuv444p16", "yuv420p10le_to_rgb" / "rgb_to_yuv420p10le", "yuv422p_to_rgb" / "rgb_to_yuv422p", "yuv422p10le_to_rgb" / "rgb_to_yuv422p10le", "yuv444p10le_to_rgb" / "rgb_to_yuv444p10le" at a planar YUV end, "nv16_to_rgb" / "rgb_to_nv16", "p210_to_rgb" / "rgb_to_p210" at a semi-planar 4:2:2 end, "yuyv422_to_rgb" / "rgb_to_yuyv422", "uyvy422_to_rgb" / "rgb_to_uyvy422", "y210_to_rgb" / "rgb_to_y210" at a packed 4:2:2 end, "resample_alpha" when both ends are RGBA / BGRA).  tu_profile_collect / tu_profile_report synchronise those events (the only
 * calls in the library that wait on the device): collect sums the milliseconds and launches recorded under `name`
 * (NULL = all); report writes "name total_ms launches\n" lines into buf (returns the needed size when buf is NULL);
 * tu_profile_reset drops the records. */
void tu_profile_enable(int on);
int tu_profile_collect(const char *name, double *total_ms, int *launches);
int tu_profile_report(char *buf, size_t cap);
void tu_profile_reset(void);
/* bring-up / A-B switches (not part of the stable interface): "tc_base_off_mode" {0,1}, "fused_stack" {0,1} (fused window
 * stack vs per-layer kernels), "conv_2cta" {0,1} (CTA-pair convolution, default off), "conv_stream" {0,1} (streaming ky-stacked N=192 convolution, default on),
 * "unembed_overlap" {0,1} (unembed starts tile by tile behind the fused window stack, default on), "head_stream" {0,1} (64->3 heads on the streaming kernel; default off: measured slower than the tile kernel), "fuse_conv12" {0,1} (conv1 fused into conv2, default on), "fold_up1" {0,1} (FastTransformer: folded up1 stage + up1_conv, default on; 0 = the unfolded op graph), "fuse_dec12" {0,1} (decoder_conv1 + decoder_conv2 in one kernel, default on), "unembed_areuse" {0,1} (unembed behind the stack: the token tile is loaded once per M tile, default off), "stack_split" {0,1} (window stack: tiles handed between CTAs at block boundaries; default off: bitwise neutral, measured slower together with the unembed overlap), "embed_pair" bit mask (patch embed: 1 one tile per CTA and two CTAs per SM [default, dim 128], 2 filter stages multicast in clusters of two, +4 also at dim 192, +8 L2 prefetch of patch rows), "bicubic_pair" {0..3} (bicubic kernel: 0 one output column per thread, 1 two columns per thread, 2 [default] the same plus the unrolled circular-window kernel, one 36-row tile per CTA and one (channel, column pair) per thread, where the row schedule is periodic: outH = 3/2 H = 3 rH as in 720p -> 1080p, or outH = n H = 2n rH with n = 2, 3, 4, 6 (720p -> 4K is n = 3), 3 the streaming form (x1.5 outputs only) of that kernel: a CTA walks down a column strip through a ring of TMA stages; measured slower), "bicubic_tile" {0,1,2} (rows per CTA of that kernel: 0 [default] the larger tile when it still gives every SM a CTA, 1 the smaller tile, 2 the larger), "resid_fused" {0,1} (ResidualTransformer: LN1 + in_proj and out_proj + LN2 + MLP as two fused kernels per layer, default on; 0 = six kernels), "global_attn_tc" {0,1} (ResidualTransformer: tcgen05 flash attention instead of the mma.sync kernel; default off: measured 6 % / 26 % slower at 2 / 16 frames), "snake" bit mask (reversed work-item order per kernel: 1 downsample, 2 the 64->3 head, 4 window stack + unembed; default 0, measured neutral), "ga_shape" (ResidualTransformer mma.sync attention: -1 automatic by CTA count [default], 0 / 1 / 2 / 3 CTA shapes 4x32 / 2x32 / 4x16 / 8x16 queries, 4 / 5 balanced launches with 64- / 128-query tiles and merged partials; these need the workspace), "stack_var" bit mask (experiments of the dim-128 window stack: 1 = first relative-position bias fetch after the first qkv third instead of before LayerNorm 1) */
int tu_debug_set(const char *key, int value);
/* debug only: while device_buffer != NULL the window stack and the unembed GEMM append (globaltimer ns, kind << 48 | smid << 32 | value)
 * pairs behind a 64-bit event counter in word 0 (caller zeroes it); capacity in events; buffer of (1 + 2 * capacity) * 8 bytes */
int tu_debug_trace(void *device_buffer, unsigned int capacity_events);

/* ---- packed weights -------------------------------------------------------------------------
 * All pointers are device pointers to tensors repacked by the host side
 * (transformerupscaler_b200/packing.py documents each layout).  `T` = the compute dtype of the
 * call (float for TU_F32, bf16 for TU_BF16); biases, LayerNorm affine, the dense relative-position
 * bias and pos_embed are always fp32.
 */
typedef struct TuBlockWeights {
    const float *ln1_w, *ln1_b, *ln2_w, *ln2_b;       /* (dim)                                   */
    const void *qkv_w;  const float *qkv_b;           /* T (3dim, dim); rows [q;k;v], q rows and  */
                                                      /*   q bias pre-scaled by head_dim^-0.5     */
    const void *proj_w; const float *proj_b;          /* T (dim, dim)                             */
    const void *fc1_w;  const float *fc1_b;           /* T (4dim, dim)                            */
    const void *fc2_w;  const float *fc2_b;           /* T (dim, 4dim)                            */
    const float *rel_bias;                            /* (heads, 64 query i, 64 key j) or NULL    */
} TuBlockWeights;

typedef struct TuUpsamplerStage {
    const void *w;      /* T: (r*r phase chunks, 9 taps, 64 co, 64 ci) for the 64-ch branch               */
                        /* float: (27, 3*r*r) for the 3-ch branch (tap-major, out-channel minor)  */
    const float *b;     /* same out-channel order as w's last dim(s)                              */
    int r;              /* PixelShuffle factor of this stage                                      */
} TuUpsamplerStage;

/* the last up1 stage (Conv2d 64 -> 64 r^2 + PixelShuffle(r)) folded with up1_conv (Conv2d 64 -> 3, no bias) into one
 * 5x5 convolution 64 -> 3 r^2 (packing.py::fold_up1; tc/upfold_stream_tcgen05.cu).  bf16 tensor-core path only. */
typedef struct TuUpFold {
    const void *w;          /* bf16 (nchunk, 5 kx, 5 ky-blocks holding ky = 4..0, NO rows, 64 ci); row n of a chunk =      */
                            /*   ((c*r + i) - chunk*RPC)*r + j; (NO, RPC, nchunk) = (16,6,1) r=2, (32,9,1) r=3, (48,6,3) r=6 */
    const float *b;         /* fp32 (nchunk*NO), zero in unused rows                                                        */
    const float *ring_w;    /* fp32 (9 border cases vy*3+vx, 3r^2 outputs o=(c*r+i)*r+j, 25 taps dy*5+dx, 64 ci)             */
    const float *ring_b;    /* fp32 (9, 3r^2)                                                                               */
    int r;                  /* PixelShuffle factor of the folded stage; 0 = not packed                                       */
} TuUpFold;

typedef struct TuModelWeights {
    int model;                  /* TU_MODEL_*                                                     */
    int dim, heads, n_blocks;   /* 128/8/8 (Window, Residual), 192/12/6 (Fast)                    */
    const float *conv1_w;       /* (27, 64) fp32: [(ky*3+kx)*3+ci][co]                            */
    const float *conv1_b;
    const void *conv1_w64;      /* bf16 (64 co, 64 k): k = (ky*3+kx)*3+ci for k < 27, zero above; tensor-core stem, or NULL */
    const void *conv2_w;        /* T (9, 64 cout, 64 cin)  [tap][co][ci]                          */
    const float *conv2_b;
    const void *down_w;         /* T (9,64,64) or NULL (Fast)                                     */
    const float *down_b;
    const void *embed_w;        /* T (dim, 4096) with K ordered (ky, kx, ci)                      */
    const float *embed_b;
    const float *pos_embed;     /* fp32 (3600, dim) or NULL                                       */
    const TuBlockWeights *blocks; /* HOST pointer to n_blocks structs                             */
    /* fused window-transformer stack (bf16, tcgen05) or NULL: layouts per dim in packing.py / window_stack{,192}_tcgen05.cu.           */
    /* TU_MODEL_RESIDUAL (bf16): the same 24 slabs per layer for tc/residual_block_tcgen05.cu; stack_p then holds 1792 floats per layer */
    /* (c0 = 0 | ln1 w,b | in_proj bias | c1 = out_proj bias | ln2 w,b | fc1 bias | c_final = out_proj bias + fc2 bias), stack_rel NULL   */
    const void *stack_w;        /* bf16 (n_blocks*24*128, 64): weight slabs [128 n][64 k] in consumption order   */
    const float *stack_p;       /* fp32 n_blocks*1664 + 128: per block c0|ln1w|ln1b|qkvb|c1|ln2w|ln2b|fc1b, then c_final */
    const float *stack_rel;     /* fp32 (n_blocks, heads, 4096) relative-position bias in mma C-fragment order: */
                                /* [rg 4][n 8][lane 32][half 2][e 2] = bias[rg*16+half*8+lane/4][n*8+(lane%4)*2+e] */
    const void *unembed_w;      /* T (4096, dim): row n = (ky*8+kx)*64 + co                       */
    const float *unembed_b;     /* (64)                                                           */
    const void *dec1_w;         /* T (9,64,64)                                                    */
    const float *dec1_b;
    const float *dec2_w;        /* fp32 (9, 64 ci, 3 co)                                          */
    const float *dec2_b;        /* (3)                                                            */
    const void *dec2_w16;       /* bf16 (3 ky, 16 rows n = kx*4 + co [co < 3, rest zero], 64 ci) for the tensor-core head, or NULL */
    const void *dec2_wst;       /* bf16 (3 kx, 3 blocks ky = 2..0, 16 rows co [co < 3, rest zero], 64 ci): streaming head, or NULL  */
    const float *dec2_b16;      /* fp32 (16): bias padded with zeros (streaming head)                                          */
    /* FastTransformer only */
    TuUpsamplerStage up1[4][2];     /* indexed by scale slot {2,3,4,6} -> 0..3, stage 0/1         */
    TuUpsamplerStage fin[4][2];
    const float *up1conv_w;     /* fp32 (9, 64, 3), no bias                                       */
    const void *up1conv_w16;    /* bf16 (3, 16, 64), same layout, or NULL                          */
    const void *up1conv_wst;    /* bf16 (3, 3, 16, 64) streaming-head layout, or NULL; its bias vector is 16 zeros */
    const float *up1conv_b16;
    const float *finconv_w;     /* fp32 (27, 3)                                                   */
    const float *finconv_b;     /* (3)                                                            */
    TuUpFold upfold[4];         /* per scale slot: folded last up1 stage + up1_conv (r = 0: absent)   */
    const float *host_finconv_wb; /* HOST pointer: the 81 finconv_w values then the 3 finconv_b values (they ride in the  */
                                /* parameters of the fused tail kernel, tu_subpixel_conv_add), or NULL                  */
} TuModelWeights;

/* ---- packing a state dict on the host side, without Python (csrc/pack_weights.cu) -----------------------------------------
 * tensors: the model's state_dict as HOST arrays under the reference's parameter names (fp32, contiguous, the reference's shapes;
 * `attn.relative_position_index` buffers are int64 and optional).  tu_pack_weights repacks them into the layouts above, uploads them
 * with one cudaMemcpyAsync on `stream` into `device_buf` (caller-owned, tu_packed_weights_bytes() bytes) and fills `out`, a
 * caller-allocated host struct: out->w is the TuModelWeights to hand to tu_forward.  out->w.blocks and out->w.host_finconv_wb point
 * INSIDE *out: keep the struct where it is.  Same results as transformerupscaler_b200/packing.py (which the PyTorch classes use). */
#define TU_MAX_BLOCKS 16
typedef struct TuNamedTensor {
    const char *name;       /* e.g. "window_blocks.3.attn.qkv.weight"                                          */
    const void *data;       /* host pointer: float32 (int64 for relative_position_index), contiguous           */
    long long numel;        /* number of elements                                                              */
} TuNamedTensor;
typedef struct TuPackedModel {
    TuModelWeights w;
    TuBlockWeights blocks[TU_MAX_BLOCKS];
    float host_finconv_wb[84];
    size_t device_bytes_used;
} TuPackedModel;
size_t tu_packed_weights_bytes(int model, int dim, int n_blocks, int compute_dtype);
int tu_pack_weights(int model, const TuNamedTensor *tensors, int n_tensors, int compute_dtype, void *device_buf, size_t device_bytes,
                    TuPackedModel *out, void *stream);

/* ---- whole-model forward (what TransformerModel.forward calls) --------------------------------
 * x:   (B,3,H,W) NCHW, dtype in_dtype.     out: (B,3,outH,outW) NCHW, dtype out_dtype, clamped to [0,1]
 *      (or un-clamped when clamp == 0; tests compare pre-clamp tensors).
 * compute_dtype: TU_F32 (exact fp32 FFMA path) or TU_BF16 (bf16 operands, fp32 accumulate); TU_F16 is rejected (TU_ERR_ARG,
 *      and a workspace size of 0).  in_dtype / out_dtype: TU_F32, TU_BF16, TU_F16 or TU_U8 [| layout] for either compute dtype.
 *      TU_U8 | TU_LAYOUT_NV12 [| colour bits]: x is (B, 3H/2, W) and / or out is (B, 3 outH/2, outW), H, W (outH, outW) even; the
 *      frame is converted to planar fp16 first (the forward is then the TU_F16 one) / the last image kernel writes planar fp16 that
 *      is converted last (codes saturate at 0 / 255 with clamp == 0 too).  Size the workspace with tu_forward_workspace_bytes_io.
 *      TU_U16 | TU_LAYOUT_P010 [| colour bits]: the same with 16-bit words and planar fp32: a P010 input is converted to planar fp32
 *      first (the forward is then the TU_F32-input one), a P010 output is the converted TU_F32 output (codes saturate at 0 / 1023
 *      with clamp == 0 too).  Either side may be NV12, P010 or any other code independently of the other.
 *      TU_U8 | TU_LAYOUT_RGBA / TU_LAYOUT_BGRA: (B,H,W,4) frames on either side; an input is read as the same pixels given as
 *      TU_LAYOUT_HWC / TU_LAYOUT_HWC_BGR.  With 4-byte frames on BOTH sides the output alpha is the input alpha resampled
 *      (tu_resample_alpha; the workspace of tu_forward_workspace_bytes_io then holds that (B, outH, outW) plane), else 255.
 *      TU_U8 | TU_LAYOUT_YUV420P / TU_LAYOUT_YUV444P, TU_U16 | TU_LAYOUT_YUV444P (planar YUV, above): as NV12 (8-bit: planar fp16) and
 *      P010 (16-bit: planar fp32) on either side; the workspace holds the planar RGB frame of each such side.  The 4:2:2 codes
 *      (TU_LAYOUT_YUV422P, TU_LAYOUT_NV16), the TU_YUV_LSB10 codes and the packed 4:2:2 codes (TU_LAYOUT_YUYV, TU_LAYOUT_UYVY; above)
 *      likewise.
 * scale: FastTransformer integer factor (ignored by the others).  For FastTransformer the library
 *      writes the (scale*H, scale*W) image; an antialiased Resize to res_out, when required, is
 *      tu_resize_bilinear_aa.
 */
/* one NV12 / P010 frame as a video decoder maps it or an encoder registers it: two planes, each with its own row pitch, anywhere in
 * device memory.  A sample is 1 byte (NV12) or one 2-byte word (P010, the code in the high 10 bits as above).
 *   y:  H rows of W samples; row r starts at y + r * y_pitch bytes;
 *   uv: H/2 rows of W samples (W/2 interleaved (U, V) pairs, U first); row r starts at uv + r * uv_pitch bytes;
 *   y_pitch, uv_pitch: bytes between rows, >= W samples.
 * The kernels access a pair of samples at a time, so both plane pointers and both pitches must be multiples of 2 bytes (NV12) or
 * 4 bytes (P010).  A write touches only the W samples of each row: pitch padding and the bytes between or after the planes are never
 * written.  The surfaces of one call must not overlap each other or the other side's buffers; the library does not check that. */
typedef struct TuFramePlanes {
    void *y;
    void *uv;
    long long y_pitch;
    long long uv_pitch;
} TuFramePlanes;
/* one planar YUV frame (yuv420p / yuv444p / yuv444p16 codes): three planes, each with its own row pitch in bytes, anywhere in device
 * memory, as an FFmpeg AVFrame (data[0..2], linesize[0..2]) or an NVDEC 4:4:4 surface holds it.
 *   y:    H rows of W samples;  u, v: H/2 rows of W/2 samples (yuv420p) or H rows of W samples (4:4:4);
 *   *_pitch: bytes between rows, >= the row's samples.
 * A YV12 surface (V plane before U) is this descriptor with u and v pointing at its U and V planes.  Alignment: see TU_LAYOUT_YUV420P
 * above.  A write touches only the valid samples of each row.  The surfaces of one call must not overlap each other or the other side's
 * buffers; the library does not check that. */
typedef struct TuFramePlanes3 {
    void *y, *u, *v;
    long long y_pitch, u_pitch, v_pitch;
} TuFramePlanes3;
/* one packed 4:2:2 frame (yuyv422 / uyvy422 / y210 codes): one plane of H rows of 2W samples (W/2 macropixels), row r starting at
 * data + r * pitch bytes, as a V4L2 / Media Foundation buffer, a DeckLink / NDI frame or a D3D11 / VAAPI surface holds it.  pitch >= 2W
 * samples; data and pitch are multiples of 4 bytes (8-bit) or 8 bytes (y210).  A write touches only the 2W samples of each row.  The
 * surfaces of one call must not overlap each other or the other side's buffers; the library does not check that. */
typedef struct TuFramePacked {
    void *data;
    long long pitch;
} TuFramePacked;

size_t tu_forward_workspace_bytes(int model, int B, int H, int W, int outH, int outW, int scale, int compute_dtype);
/* the same, sized from the packed weights actually used (non-default dim / heads / n_blocks; which fused kernels are packed) */
size_t tu_forward_workspace_bytes_for(const TuModelWeights *w, int B, int H, int W, int outH, int outW, int scale, int compute_dtype);
/* the same for the image input / output codes of the call: equal to tu_forward_workspace_bytes_for for every code pair without a YUV
 * side, larger by the planar fp16 frames of the side(s) that are NV12, yuv420p or yuv444p and the planar fp32 frames of the side(s)
 * that are P010 or yuv444p16, and by the (B, outH, outW) alpha plane when both sides are RGBA / BGRA (tu_forward needs it then); 0 for a
 * bad code */
size_t tu_forward_workspace_bytes_io(const TuModelWeights *w, int B, int H, int W, int outH, int outW, int scale, int compute_dtype,
                                     int in_dtype, int out_dtype);
int tu_forward(const TuModelWeights *w, const void *x, int in_dtype, void *out, int out_dtype,
               int B, int H, int W, int outH, int outW, int scale, int compute_dtype, int clamp,
               void *workspace, size_t workspace_bytes, void *stream);
/* tu_forward with per-frame decoder / encoder surfaces on an NV12 or P010 side.  On each side exactly one of the dense buffer (x, out)
 * and x_frames / out_frames, a HOST array of B TuFramePlanes, is non-NULL; a frames array is valid only when that side's code is NV12 or
 * P010.  Frame b of the batch is x_frames[b] / out_frames[b].  The arrays are read during the call (the descriptors travel in kernel
 * parameters), so the caller may reuse them once it returns, and a captured CUDA graph replays the same surfaces.  Every descriptor is
 * checked before anything is enqueued (TU_ERR_ARG, with the frame index and field in tu_last_error).  The workspace is the one
 * tu_forward_workspace_bytes_io gives for the same codes: surfaces do not change it.  The results are bitwise those of tu_forward on the
 * dense frames of the same contents.  tu_forward(...) is tu_forward_planes with both arrays NULL. */
int tu_forward_planes(const TuModelWeights *w, const void *x, const TuFramePlanes *x_frames, int in_dtype, void *out,
                      const TuFramePlanes *out_frames, int out_dtype, int B, int H, int W, int outH, int outW, int scale,
                      int compute_dtype, int clamp, void *workspace, size_t workspace_bytes, void *stream);
/* tu_forward_planes for every kind of YUV side: x_frames / out_frames is a HOST array of B descriptors whose element type the side's
 * code chooses -- TuFramePlanes for NV12 / P010 / NV16 / P210 (4:2:2: uv holds H rows), TuFramePlanes3 for the planar codes (yuv420p,
 * yuv422p, yuv444p, yuv444p16 and the TU_YUV_LSB10 ones; 4:2:2: u and v hold H rows of W/2 samples), TuFramePacked for yuyv422 /
 * uyvy422 / y210 (tu_forward_planes rejects a frames array on such a side) -- and otherwise follows the rules of
 * tu_forward_planes (exactly one of dense buffer and array per side, every descriptor checked before anything is enqueued, workspace of
 * tu_forward_workspace_bytes_io, results bitwise those of the dense frames).  The two sides are independent: NV12 surfaces in and
 * yuv444p surfaces out is one call.  tu_forward_planes(...) is this function. */
int tu_forward_frames(const TuModelWeights *w, const void *x, const void *x_frames, int in_dtype, void *out, const void *out_frames,
                      int out_dtype, int B, int H, int W, int outH, int outW, int scale, int compute_dtype, int clamp, void *workspace,
                      size_t workspace_bytes, void *stream);

/* ---- single ops (exported for the per-op parity tests and for composition) ---------------------- */
/* conv1: 3->64 3x3 p1 + ReLU, NCHW in -> NHWC out.  w64 (optional, bf16 (64,64)) enables the tensor-core kernel
 * for dtype TU_BF16. */
int tu_stem_conv(const void *x, int in_dtype, const float *w27x64, const void *w64, const float *b, void *out, int dtype,
                 int B, int H, int W, void *stream);
/* 64->(64*nchunk) 3x3 p1 conv on NHWC, stride 1|2, optional ReLU, optional PixelShuffle(r) store
 * (then nchunk = r*r and chunk p holds phase (i,j) = (p/r, p%r) for all 64 channels). */
int tu_conv3x3_c64(const void *in, const void *w, const float *b, void *out, int dtype,
                   int B, int H, int W, int stride, int relu, int nchunk, int ps_r, void *stream);
/* 64->3 3x3 p1 conv, NHWC in -> planar fp32 (B,3,H,W) out.  w16 (optional, bf16 (3 ky, 16 n = kx*4+co, 64 ci)) enables the
 * tensor-core kernel for dtype TU_BF16; w (fp32 (9,64,3)) is always required. */
int tu_conv3x3_c64_to3(const void *in, int dtype, const float *w, const void *w16, const float *b, float *out,
                       int B, int H, int W, int relu, void *stream);
/* the same 64->3 convolution on the streaming tensor-core kernel (bf16 NHWC in, planar fp32 out): wst = bf16 (3 kx, 3 blocks
 * ky = 2..0, 16 rows co, 64 ci), b16 = fp32 (16, zero padded).  Needs the tcgen05 path and W % 4 == 0. */
int tu_conv3x3_c64_to3_stream(const void *in, const void *wst, const float *b16, float *out, int B, int H, int W, int relu,
                              void *stream);
/* 3->3r^2 3x3 conv + PixelShuffle(r) on planar fp32 */
int tu_conv3x3_c3_ps(const float *in, const float *w, const float *b, float *out, int B, int H, int W, int r,
                     void *stream);
/* out = clamp?(conv3x3_3to3(in) + addend) -> NCHW image of out_dtype */
int tu_final_conv_add(const float *in, const float *w, const float *b, const float *addend, void *out,
                      int out_dtype, int B, int H, int W, int clamp, void *stream);
/* relu(conv2(relu(conv1(x)))) in one kernel (bf16 tensor-core path): NCHW image (in_dtype) -> NHWC bf16 (B,H,W,64); w64 = conv1
 * filter bf16 (64 co, 64 k), w2 = conv2 filter bf16 (9, 64 co, 64 ci).  conv1's output never reaches HBM.  W:244-245, F:251-252,
 * R:128-129.  Needs an image row pitch that is a multiple of 16 bytes. */
int tu_conv12_fused(const void *x, int in_dtype, const void *w64, const float *b1, const void *w2, const float *b2, void *out,
                    int B, int H, int W, void *stream);
/* decoder_conv2(relu(decoder_conv1(in))) in one kernel (bf16 tensor-core path): NHWC bf16 (B,H,W,64) -> planar fp32 (B,3,H,W);
 * w1 = decoder_conv1 filter bf16 (9, 64 co, 64 ci), w16 = decoder_conv2 filter bf16 (3 ky, 16 rows n = kx*4 + co, 64 ci), b1 (64)
 * and b2 (3) fp32.  The 64-channel map between the two convolutions never reaches HBM.  W:297-298, F:312-313, R:156-157.
 * out is written with plain stores except for the columns two 128-pixel strips share (atomicAdd onto zeros: the op zeroes
 * them itself, on the same stream). */
int tu_dec12_fused(const void *in, const void *w1, const float *b1, const void *w16, const float *b2, float *out, int B, int H,
                   int W, void *stream);
/* relu(up1_conv(PixelShuffle_r(up1_stage(in)))) through the folded 5x5 filter: NHWC bf16 (B,H,W,64) -> planar fp32
 * (B,3,rH,rW).  FastTransformer/model.py:264-265.  Needs the tcgen05 path and (W*r) % 4 == 0. */
int tu_upfold_conv(const void *in, const TuUpFold *f, float *out, int B, int H, int W, void *stream);
/* the last sub-pixel stage of final_upscale, final_upscale_conv, the sum with the other branch and the clamp in one kernel:
 * out = clamp?(conv3x3_3to3(PixelShuffle_r(conv3x3_3to3r^2(in))) + addend); in (B,3,H,W) and addend (B,3,rH,rW) planar fp32,
 * w_ps fp32 (27, 3r^2), b_ps (3r^2), r in {2,3,6}; host_fin_wb is a HOST pointer to the 3->3 filter, (27,3) then bias (3).
 * FastTransformer/model.py:316-327. */
int tu_subpixel_conv_add(const float *in, const float *w_ps, const float *b_ps, int r, const float *host_fin_wb,
                         const float *addend, void *out, int out_dtype, int B, int H, int W, int clamp, void *stream);
/* patch embed (Conv2d k8 s8) as GEMM; reflect-pads feat to x8 when reflect != 0; writes fp32 tokens
 * window-ordered into zero-initialised (B*nWy*nWx*64, dim) (window != 0) or row-major + pos_embed. */
int tu_patch_embed(const void *feat, int dtype, const void *w, const float *b, const float *pos_embed,
                   float *tokens, int B, int H, int W, int Ht, int Wt, int dim, int window, int reflect,
                   void *stream);
/* patch unembed (ConvTranspose2d k8 s8) + crop + skip add -> NHWC (B,Hc,Wc,64) */
int tu_patch_unembed(const float *tokens, const void *w, const float *b, const void *skip, int skipH, int skipW,
                     void *out, int dtype, int B, int Ht, int Wt, int Hc, int Wc, int dim, int window,
                     void *stream);
/* one pre-LN transformer block in place on the fp32 token stream x (M, dim).
 * window != 0: M = nWin*64, 8x8 window attention with rel_bias; else global attention over S tokens per frame. */
size_t tu_block_workspace_bytes(int M, int dim, int dtype);
/* the same including the scratch of the tcgen05 global attention (window == 0, S tokens per frame, TU_BF16): with only
 * tu_block_workspace_bytes() the block falls back to the mma.sync attention kernel */
size_t tu_block_workspace_bytes_for(int M, int dim, int dtype, int window, int S);
int tu_transformer_block(float *x, const TuBlockWeights *w, int M, int dim, int heads, int window, int S,
                         int dtype, void *workspace, size_t workspace_bytes, void *stream);
/* all window-transformer blocks of a bf16 WindowTransformer / FastTransformer in one fused kernel, in place on the fp32
 * window-ordered token stream (M, dim), M a multiple of 128 (`for block in self.window_blocks`, W:272-273, F:288-289) */
int tu_window_stack(float *tokens, const TuModelWeights *w, int M, void *stream);
/* the two fused kernels of one bf16 ResidualTransformer layer (`layer` of w->n_blocks), around its global attention (R:22-50):
 * tu_resid_pre: LN1 + in_proj of the fp32 tokens (M, 128) -> bf16 q | k | v rows (M, 384) with q pre-scaled by head_dim^-0.5;
 * tu_resid_post: tokens += out_proj(att), then tokens += fc2(GELU(fc1(LN2(tokens)))) in place, att (M, 128) bf16.
 * Rows past M are neither read nor written. */
int tu_resid_pre(const float *tokens, void *qkv, const TuModelWeights *w, int layer, int M, void *stream);
int tu_resid_post(float *tokens, const void *att, const TuModelWeights *w, int layer, int M, void *stream);
/* window attention alone: softmax(q k^T + rel_bias) v per 8x8 window and head (head_dim 16) on qkv rows (nWin*64, 3*dim) with q
 * pre-scaled; rel_bias dense (heads,64,64) fp32; out (nWin*64, dim).  WindowTransformer/model.py:104-127 between qkv and proj. */
int tu_window_attention(const void *qkv, const float *rel_bias, void *out, int nWin, int dim, int heads, int dtype, void *stream);
/* global attention alone (ResidualTransformer/model.py:31,44 between in_proj and out_proj): softmax(q k^T) v over the S tokens of a
 * frame per head (head_dim 16) on qkv rows (B*S, 3*heads*16) bf16 with q pre-scaled; out (B*S, heads*16) bf16.  With a workspace of
 * tu_global_attention_workspace_bytes() AND tu_debug_set("global_attn_tc", 1) the tcgen05 kernel runs (S % 8 == 0, S >= 128), otherwise
 * the mma.sync kernel (the default: measured faster at head_dim 16). */
size_t tu_global_attention_workspace_bytes(int B, int S, int heads);
int tu_global_attention(const void *qkv, void *out, int B, int S, int heads, void *workspace, size_t workspace_bytes, void *stream);
/* Host-side query, no GPU needed: the periodic row schedule tu_bicubic_add_clamp's unrolled kernel would use for these heights
 * (WindowTransformer/model.py:241,301: x H rows and the decoder's residual rH rows, both resampled to outH): 0 for outH = 3/2 H = 3 rH
 * (720p -> 1080p), n = 2, 3, 4, 6 for outH = n H = 2n rH (3: 720p -> 4K), -1 when the heights have no such schedule OR when ATen's
 * fp32 source-row arithmetic deviates from it on some output row (the general kernel runs then). */
int tu_bicubic_row_schedule(int H, int rH, int outH);
/* out = clamp?(bicubic(x -> outH,outW) + bicubic(res -> outH,outW)); res may be NULL */
int tu_bicubic_add_clamp(const void *x, int in_dtype, int H, int W, const float *res, int rH, int rW,
                         void *out, int out_dtype, int B, int outH, int outW, int clamp, void *stream);
/* antialiased bilinear resize (torchvision Resize on a tensor) of an NCHW image, then optional clamp */
int tu_resize_bilinear_aa(const void *in, int dtype, void *out, int B, int H, int W, int outH, int outW,
                          int clamp, void *stream);
/* the same with an output dtype of its own (TU_F32 / TU_BF16 / TU_U8 [| layout]): FastTransformer's Resize as the LAST op of a
 * uint8-frame forward (FastTransformer/model.py:323-327 followed by app_overlay.py:382-386); a 4-byte layout gets alpha 255 */
int tu_resize_bilinear_aa_to(const void *in, int in_dtype, void *out, int out_dtype, int B, int H, int W, int outH, int outW,
                             int clamp, void *stream);
/* the same with the alpha byte of a 4-byte output (TU_U8 | TU_LAYOUT_RGBA / TU_LAYOUT_BGRA) taken from `alpha`, a (B, outH, outW) uint8
 * plane (tu_resample_alpha); alpha == NULL writes 255.  tu_resize_bilinear_aa_to is this function with alpha == NULL. */
int tu_resize_bilinear_aa_to_alpha(const void *in, int in_dtype, const void *alpha, void *out, int out_dtype, int B, int H, int W,
                                   int outH, int outW, int clamp, void *stream);
/* uint8 frames (B,H,W,3) interleaved (layout TU_LAYOUT_HWC or TU_LAYOUT_HWC_BGR), or (B,H,W,4) with alpha (TU_LAYOUT_RGBA or
 * TU_LAYOUT_BGRA; the alpha is dropped) -> planar RGB (B,3,H,W) uint8; tu_forward does this itself for an in_dtype that carries a
 * layout (into its workspace) */
int tu_frames_to_planar(const void *in, int layout, void *out, int B, int H, int W, void *stream);
/* the alpha bytes of 4-byte frames (B,H,W,4), code TU_U8 | TU_LAYOUT_RGBA or TU_U8 | TU_LAYOUT_BGRA, resampled to a (B, outH, outW) uint8
 * plane: bicubic, ATen's F.interpolate(mode="bicubic", align_corners=False) -- A = -0.75, half-pixel centres, taps clamped to the
 * edge, the taps ty_i / tx_j and weights wy_i / wx_j of the engine's bicubic kernels (scale = (float)in / out,
 * src = fma(scale, dst + 0.5, -0.5) in fp32) -- on the codes 0..255 as floats, every step one correctly rounded fp32 operation
 * (no contraction), sums left to right from 0:
 *   acc_i = sum_j A[ty_i, tx_j] * wx_j,   a = sum_i acc_i * wy_i,   alpha = min(max(floor(a + 0.5), 0), 255).
 * A constant plane stays exactly constant.  tu_forward runs this on its input when both sides are 4-byte frames (into its workspace). */
int tu_resample_alpha(const void *frames, int code, void *alpha, int B, int H, int W, int outH, int outW, void *stream);
/* NV12 frames (B, 3H/2, W) uint8 -> planar RGB (B, 3, H, W) fp16, and back.  code = TU_U8 | TU_LAYOUT_NV12 | colour bits (anything else,
 * an odd H or W, or B > 65535: TU_ERR_ARG).  Every step is one correctly rounded fp32 operation (no contraction), so the results are exactly
 * those of the formulas below, with (yo, ys, cs) = (16, 219, 224) limited / (0, 255, 255) full range, Kg = 1 - Kr - Kb and every
 * coefficient computed in double and rounded once to float:
 *   to RGB:  chroma upsampled bilinearly (type-0 siting, edges clamped), y' = (Y - yo) / ys, u' = (U - 128) / cs, v' = (V - 128) / cs,
 *            R = y' + a_rv v', G = (y' + a_gu u') + a_gv v', B = y' + a_bu u', each clamped to [0, 1] and rounded to fp16;
 *   to NV12: Y' = (Kr R + Kg G) + Kb B per pixel; chroma from the 2-row column sums v(c) filtered (v(2j-1) + 2 v(2j) + v(2j+1)) / 8
 *            (column 2j-1 clamped at 0), Cb' = (cbR R + cbG G) + 0.5 B, Cr' = (0.5 R + crG G) + crB B; a code is
 *            min(max(floor(s Y' + o + 0.5), 0), 255) with (s, o) = (219, 16) / (224, 128) limited, (255, 0) / (255, 128) full range. */
int tu_nv12_to_rgb(const void *nv12, int code, void *rgb_f16, int B, int H, int W, void *stream);
int tu_rgb_to_nv12(const void *rgb_f16, void *nv12, int code, int B, int H, int W, void *stream);
/* P010 frames (B, 3H/2, W) of uint16 words -> planar RGB (B, 3, H, W) fp32, and back.  code = TU_U16 | TU_LAYOUT_P010 | colour bits
 * (anything else, an odd H or W, or B > 65535: TU_ERR_ARG); the P010 buffer must be 4-byte and the RGB buffer 8-byte aligned.  The
 * formulas are those of the NV12 ops above, on 10-bit codes (Y = word >> 6, and so on) with chroma midpoint 512 instead of 128,
 * (yo, ys, cs) = (64, 876, 896) limited / (0, 1023, 1023) full range, and (Kr, Kb) = (0.2627, 0.0593) for TU_YUV_BT2020:
 *   to RGB:  y' = (Y - yo) / ys, u' = (U - 512) / cs, v' = (V - 512) / cs, R, G, B as for NV12, each clamped to [0, 1] (fp32 out);
 *   to P010: Y', Cb', Cr' as for NV12; a code is min(max(floor(s Y' + o + 0.5), 0), 1023) with (s, o) = (876, 64) / (896, 512)
 *            limited, (1023, 0) / (1023, 512) full range, stored as code << 6. */
int tu_p010_to_rgb(const void *p010, int code, void *rgb_f32, int B, int H, int W, void *stream);
int tu_rgb_to_p010(const void *rgb_f32, void *p010, int code, int B, int H, int W, void *stream);
/* the four ops above on per-frame surfaces: frames is a HOST array of B TuFramePlanes (see tu_forward_planes), read during the call.
 * code = TU_U8 | TU_LAYOUT_NV12 [| colour bits] with planar fp16 RGB (4-byte aligned), or TU_U16 | TU_LAYOUT_P010 [| colour bits] with
 * planar fp32 RGB (8-byte aligned); rgb is a dense (B, 3, H, W) buffer.  Same bits as the dense ops on the same frame contents. */
int tu_yuv420_planes_to_rgb(const TuFramePlanes *frames, int code, void *rgb, int B, int H, int W, void *stream);
int tu_rgb_to_yuv420_planes(const void *rgb, const TuFramePlanes *frames, int code, int B, int H, int W, void *stream);
/* planar YUV frames <-> planar RGB (B, 3, H, W): fp16 RGB for TU_U8 | TU_LAYOUT_YUV420P / TU_LAYOUT_YUV444P codes, fp32 RGB for
 * TU_U16 | TU_LAYOUT_YUV444P (colour bits as above; anything else, an odd H or W for yuv420p, or B > 65535: TU_ERR_ARG).  Exactly one of
 * `dense` (the (B, 3H/2, W) or (B, 3, H, W) batch) and `frames` (a HOST array of B TuFramePlanes3, read during the call) is non-NULL.
 * yuv420p gives the bits of tu_nv12_to_rgb / tu_rgb_to_nv12 on the same samples; 4:4:4 follows the same formulas per pixel without the
 * chroma filter.  The RGB buffer is 4-byte aligned (yuv420p) or aligned to its element (4:4:4). */
int tu_yuvp_to_rgb(const void *dense, const TuFramePlanes3 *frames, int code, void *rgb, int B, int H, int W, void *stream);
int tu_rgb_to_yuvp(const void *rgb, void *dense, const TuFramePlanes3 *frames, int code, int B, int H, int W, void *stream);
/* The same two ops also take TU_U8 | TU_LAYOUT_YUV422P (fp16 RGB) and the TU_YUV_LSB10 codes (fp32 RGB): yuv420p10le gives the bits of
 * P010 with every word shifted left by 6, yuv444p10le those of yuv444p16 likewise; yuv422p follows the 4:2:2 formulas above.  The RGB
 * buffer is 4-byte (fp16) / 8-byte (fp32) aligned for 4:2:0 and 4:2:2, aligned to its element for 4:4:4.
 * Semi-planar 4:2:2 frames <-> planar RGB (B, 3, H, W): code TU_U8 | TU_LAYOUT_NV16 with fp16 RGB (4-byte aligned), or TU_U16 |
 * TU_LAYOUT_NV16 (p210) with fp32 RGB (8-byte aligned), colour bits as above (anything else, an odd W, or B > 65535: TU_ERR_ARG).  Exactly
 * one of `dense` (the (B, 2H, W) batch) and `frames` (a HOST array of B TuFramePlanes whose uv planes hold H rows, read during the call)
 * is non-NULL.  yuv422p gives the bits of nv16 on the same samples. */
int tu_yuv422sp_to_rgb(const void *dense, const TuFramePlanes *frames, int code, void *rgb, int B, int H, int W, void *stream);
int tu_rgb_to_yuv422sp(const void *rgb, void *dense, const TuFramePlanes *frames, int code, int B, int H, int W, void *stream);
/* Packed 4:2:2 frames <-> planar RGB (B, 3, H, W): code TU_U8 | TU_LAYOUT_YUYV / TU_LAYOUT_UYVY with fp16 RGB (4-byte aligned), or
 * TU_U16 | TU_LAYOUT_YUYV (y210) with fp32 RGB (8-byte aligned), colour bits as above (anything else, an odd W, B > 65535, a NULL or a
 * misaligned buffer: TU_ERR_ARG, before any launch).  Exactly one of `dense` (the (B, H, W, 2) batch) and `frames` (a HOST array of B
 * TuFramePacked, read during the call) is non-NULL.  Bitwise tu_yuv422sp_to_rgb / tu_rgb_to_yuv422sp on the nv16 / p210 frame of the
 * same samples. */
int tu_packed422_to_rgb(const void *dense, const TuFramePacked *frames, int code, void *rgb, int B, int H, int W, void *stream);
int tu_rgb_to_packed422(const void *rgb, void *dense, const TuFramePacked *frames, int code, int B, int H, int W, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* TU_B200_H */
