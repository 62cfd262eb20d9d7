/*
 * t2v.h -- C ABI of libt2v_b200.so: the sm_100a kernels behind txt2vid's GAN training step.
 *
 * The reference (miguelmartin75/txt2vid) has no FFI of its own: its "plugin" boundary is Python
 * reflection (txt2vid/util/reflection.py:12-50) and every FLOP is an ATen call inside
 * txt2vid/models/ and txt2vid/gan/.  Each entry point below replaces the ATen call sites named in its
 * comment (file:line relative to the reference tree).  The Python host side (txt2vid_b200/) binds
 * these with ctypes; see INTEGRATION.md for the binding a maintainer of the reference would add.
 *
 * Conventions
 *   - plain pointers and sizes only; all pointers are DEVICE pointers unless named host_*;
 *   - every call enqueues work on `stream` (a cudaStream_t passed as void*), never synchronises,
 *     never allocates device memory and never throws; returns T2V_OK (0) or a negative T2V_ERR_*;
 *   - "CL" = channels-last activation layout [N][D][H][W][C] (2-D feature maps use D = 1);
 *     activations are bf16, accumulation is fp32, master weights / gradients of weights are fp32;
 *   - conv weights are [Cout][kd][kh][kw][Cin] ("channels-last" memory of the reference's
 *     (Cout,Cin,kd,kh,kw) parameter), so a weight gradient written by the kernels IS the parameter
 *     gradient's memory.
 */
#ifndef T2V_H_
#define T2V_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define T2V_OK 0
#define T2V_ERR_ARG (-1)      /* unsupported shape / null pointer / misalignment */
#define T2V_ERR_LAUNCH (-2)   /* CUDA reported an error at launch */
#define T2V_ERR_DRIVER (-3)   /* driver entry point (tensor-map encode) unavailable */

/* algo selector for the convolution engine */
#define T2V_ALGO_AUTO 0   /* tcgen05 implicit GEMM when the shape allows it, else SIMT */
#define T2V_ALGO_TC 1     /* force the tcgen05/TMEM/TMA kernel (error if shape unsupported) */
#define T2V_ALGO_SIMT 2   /* force the CUDA-core kernels of t2v_gconv_* (cross-check + odd shapes) */
#define T2V_ALGO_TC_GENERIC 3 /* force the generic tcgen05 implicit GEMM (skip the halo-resident 64-channel kernels) */
#define T2V_ALGO_SIMT_F32 4   /* t2v_conv_wgrad only: dy and x are fp32 CL, on the kernel of t2v_gconv_wgrad_f32:
                               * exact fp32 FMAs (fp32 parity mode) */

/* epilogue flags of t2v_conv_fprop */
#define T2V_EPI_RELU 1u       /* y = max(y, 0) after bias/residual */
#define T2V_EPI_OUT_F32 2u    /* y is fp32 CL instead of bf16 CL */
#define T2V_EPI_RELU_MASK 4u  /* the `residual` pointer is a ReLU reference r (bf16 CL, output-shaped): instead of
                               * adding it, zero the output where r <= 0 -- the backward of the ReLU that produced the
                               * convolution's input, fused into the data-gradient epilogue (layers.py:230-232) */
#define T2V_EPI_IN_F32 16u    /* fp32 PARITY mode: x / residual are fp32 CL and w is fp32 [Cout][taps][Cin]; the
                               * convolution runs on the kernel of t2v_gconv_fprop_f32 as exact fp32 FMAs, flushed
                               * once per tap (the reference's numerics; the tensor pipe's truncating fp32 accumulator
                               * cannot reach 1e-6 on K ~ 1e4), y fp32 */

/* Stride-1, "same"-padded convolution geometry (every conv on the TGANv2 path:
 * models/layers.py:174,177,183,231,233,237,251; models/resnet3d.py:12-17; 1x1(x1) convs of the
 * attention blocks layers.py:16-19,45-48; nn.Linear is the k=1, D=H=W=1 case). */
typedef struct {
  int32_t N, D, H, W;    /* batch (or merged batch*frames) and spatial extents            */
  int32_t Cin, Cout;     /* channels; both multiples of 16 (pad with zeros otherwise)      */
  int32_t kd, kh, kw;    /* kernel extents, each 1 or 3; padding is k/2                     */
} t2v_conv_geom;

/* library / bookkeeping ------------------------------------------------------------------- */
int t2v_version(void);
/* number of kernels launched by this library since load (bench.py: "gpu_launches") */
unsigned long long t2v_launch_count(void);
/* optional CUDA-event timing of every conv-engine launch (bench.py roofline); read returns
 * host_out6 = {fprop+dgrad ms, useful FLOPs, launches, wgrad ms, useful FLOPs, launches} and resets */
int t2v_profile_enable(int on);
int t2v_profile_read(double* host_out6);
/* same, split by kernel: {generic fprop/dgrad, generic wgrad, halo-resident fprop/dgrad, halo-resident wgrad} x
 * {ms, useful FLOPs, launches} */
int t2v_profile_read4(double* host_out12);
/* same with the direct RGB-stem kernels as kinds 4 (fprop) and 5 (wgrad) */
int t2v_profile_read6(double* host_out18);
/* fraction of the NEXT profiled launch's channel products that are real (zero channel padding excluded from the
 * roofline's FLOP count); resets to 1 after that launch */
int t2v_profile_next_scale(double real_fraction);

/* convolution engine (tcgen05 implicit GEMM; replaces F.conv2d/conv3d/linear = cuDNN/cuBLAS)  */
/* y[n,d,h,w,co] = sum_{taps,ci} x[n,d+a-pd,h+b-ph,w+c-pw,ci] * w[co,a,b,c,ci] + bias[co] (+ residual)
 * x: bf16 CL, w: bf16 [Cout][taps][Cin], bias: fp32[Cout] or NULL, residual: bf16 CL [..,Cout] or NULL */
int t2v_conv_fprop(const t2v_conv_geom* g, const void* x, const void* w, const float* bias,
                   const void* residual, void* y, uint32_t epi_flags, int algo, void* stream);
/* y = conv(x, w) + conv1x1x1(x2, w2) + bias: a residual block's identity_map convolution fused into the main path's
 * last convolution as extra K of the same implicit GEMM (DownBlock, models/layers.py:224-243): the skip tensor is never
 * written or re-read.  x2 bf16 CL (N,D,H,W,Cin2), w2 bf16 [Cout][Cin2]; Cin and Cin2 multiples of 64.          */
int t2v_conv_fprop_skip(const t2v_conv_geom* g, const void* x, const void* w, const float* bias, const void* x2,
                        const void* w2, int32_t Cin2, void* y, uint32_t epi_flags, void* stream);
/* dx = conv_transpose(dy, w): same engine, fed with the weight pack made by t2v_pack_dgrad_weight:
 * wT bf16 [Cin][taps (flipped)][Cout]; g is the FORWARD geometry. */
int t2v_conv_dgrad(const t2v_conv_geom* g, const void* dy, const void* wT, const void* residual,
                   void* dx, uint32_t epi_flags, int algo, void* stream);
/* dw[co,tap,ci] (+)= sum_pos dy[pos,co] * x[pos+tap,ci]   (fp32, layout [Cout][taps][Cin]).
 * accumulate = 0 overwrites dw, 1 adds into it.                                              */
int t2v_conv_wgrad(const t2v_conv_geom* g, const void* dy, const void* x, float* dw,
                   int accumulate, int algo, void* stream);
/* ONE ConvLSTM step (models/conv_lstm.py:32-38, zero peepholes :46-49) as one tcgen05 implicit GEMM whose EPILOGUE is
 * the cell update: gates = conv(x, w) + b on the tensor pipe (x = the input at step 0, h_{t-1} afterwards; g->Cout =
 * 4 * hidden), then per output row sigmoid / tanh, c_t = f c_{t-1} + i g, h_t = o tanh(c_t) straight from TMEM.
 * w_il / bias_il are GATE-INTERLEAVED along Cout: row blk * 128 + gate * 32 + j holds gate `gate` (i, f, g, o) of hidden
 * unit blk * 32 + j, so one 128-column accumulator tile carries all four gates of 32 units.  Writes gates (fp32
 * [P][4 hidden], standard [i|f|g|o] order, pre-activation: the backward pass's input), c_out (fp32 [P][hidden]), h_out
 * (bf16 [P][hidden], the next step's operand) and h_t into its slot of the merged (b, t) frame map h_merged
 * (bf16 [(n * steps + t) * D*H*W + pos][hidden], tganv2_cond/gen.py:75-76).  c_prev may be NULL (zeros).            */
int t2v_conv_lstm_step(const t2v_conv_geom* g, const void* x, const void* w_il, const float* bias_il,
                       const float* c_prev, float* gates, float* c_out, void* h_out, void* h_merged, int32_t t,
                       int32_t steps, void* stream);
/* Convolution with stride (2,1,1), kernel 3x3x3, padding 1, 64 -> 64 channels: the second convolution of the
 * discriminator stem (models/resnet3d.py:15) is followed by AvgPool3d((1,2,2), 2) (resnet3d.py:16: kernel 1,
 * stride 2 along d), which never reads its odd output planes; computing only the even planes is the same
 * function at half the MACs.  g = geometry of x (D even, H >= 16, W >= 8); y / dy are (N, D/2, H, W, 64).
 * dgrad takes the flipped pack of t2v_pack_dgrad_weight and an optional ReLU reference (NULL or x-shaped, see
 * T2V_EPI_RELU_MASK); wgrad writes [Cout][27][Cin] fp32 like t2v_conv_wgrad. */
int t2v_conv_sd2_supported(const t2v_conv_geom* g);
int t2v_conv_fprop_sd2(const t2v_conv_geom* g, const void* x, const void* w, const float* bias, void* y,
                       uint32_t epi_flags, void* stream);
int t2v_conv_dgrad_sd2(const t2v_conv_geom* g, const void* dy, const void* wT, const void* relu_ref, void* dx,
                       uint32_t epi_flags, void* stream);
int t2v_conv_wgrad_sd2(const t2v_conv_geom* g, const void* dy, const void* x, float* dw, int accumulate,
                       void* stream);
/* RGB stem of the discriminator on the tensor cores without an im2col tensor in memory
 * (models/resnet3d.py:12-13: Conv3d(3 -> 64, 3, padding 1) + ReLU): the im2col tile is gathered into shared memory.
 *   xc  bf16 CL (N, D, H, W, cpv), cpv = 4 or 16 channels per voxel: RGB in channels 0..2, zeros elsewhere
 *       (t2v_rgb_to_cl; 4-channel rows make the gather's 8-byte loads contiguous across a warp)
 *   wp  bf16 [64][128]: wp[co][tap*4 + c] = w[co][c][tap] for c < 3, zero elsewhere (tap = (a_d*3 + a_h)*3 + a_w)
 *   y   bf16 CL (N, D, H, W, 64) = [relu](conv + bias);   dw fp32 [64][27][3] (+)= sum_pos dy[pos,co] x[pos+tap,c] */
int t2v_stem_fprop(const void* xc, int32_t cpv, const void* wp, const float* bias, void* y, int64_t N, int32_t D,
                   int32_t H, int32_t W, int32_t relu, void* stream);
int t2v_stem_wgrad(const void* dy, const void* xc, int32_t cpv, float* dw, int64_t N, int32_t D, int32_t H, int32_t W,
                   int32_t accumulate, void* stream);
/* Small-channel (1,3,3) weight gradients on position pairs: run t2v_conv_wgrad on x viewed as (N,1,H,W/2,2*Cin) and
 * dy as (N,1,H,W/2,2*Cout) (128-byte rows for Cin = 32), then fold dw2 fp32 [2*Cout][9][2*Cin] into
 * dw fp32 [Cout][9][Cin] (accumulate = 1: dw += ...).  Generator levels 2-3 (models/layers.py:174-183,251).        */
int t2v_wgrad_fold_pairs(const float* dw2, float* dw, int32_t Cout, int32_t Cin, int32_t accumulate, void* stream);
/* General convolution geometry (any kernel / stride / zero padding; 1-D and 2-D use unit extents):
 * the TGAN / TCWYT layers that are not stride-1 "same" convolutions -- Conv3d/Conv2d k4 s2 p1
 * (models/tcwyt/video_discrim.py:12-27, frame_discrim.py:8-19), k(1,3,3) and k2 s2 heads
 * (video_discrim.py:41,46; frame_discrim.py:49), and every ConvTranspose1d/2d/3d (models/tgan/gen.py:21-25,
 * tgan/temporal_gen.py:16-20, tcwyt/gen.py:14-30).  Do = (Di + 2*pd - kd)/sd + 1, etc.                */
typedef struct {
  int32_t N, Di, Hi, Wi, Do, Ho, Wo;
  int32_t Cin, Cout;           /* channels of the convolution's input / output                      */
  int32_t kd, kh, kw, sd, sh, sw, pd, ph, pw;
} t2v_gconv_geom;
/* y[N,Do,Ho,Wo,Cout] = conv(x[N,Di,Hi,Wi,Cin], w[Cout][taps][Cin]) + bias; y bf16 or fp32 CL        */
int t2v_gconv_fprop(const t2v_gconv_geom* g, const void* x, const void* w, const float* bias, void* y,
                    int32_t out_f32, void* stream);
/* dx[N,Di,Hi,Wi,Cin] = conv_transpose(dy[N,Do,Ho,Wo,Cout], w) (+ bias[Cin]): the data gradient of the
 * convolution AND the forward of nn.ConvTranspose*d(Cout -> Cin) with the same weight memory           */
int t2v_gconv_dgrad(const t2v_gconv_geom* g, const void* dy, const void* w, const float* bias, void* dx,
                    int32_t out_f32, void* stream);
/* dw[Cout][taps][Cin] (+)= sum_pos dy[pos,co] * x[in(pos,tap),ci]  (fp32)                              */
int t2v_gconv_wgrad(const t2v_gconv_geom* g, const void* dy, const void* x, float* dw, int32_t accumulate,
                    void* stream);
/* On-device input pipeline (SURVEY 8 f1).
 * t2v_moving_digits: frames of data/synthetic/generate.py:18-47: black RGB frames with the oh x ow grey patch
 *   bank[digit[b]] pasted at pos[b][t] = (x, y) (host-computed, int32 [B][T][2]); out uint8 as stored or (out_f32) fp32
 *   through ToTensor + Normalize(0.5, 0.5) (data/__init__.py:362-364); layout 0 = (B,T,3,H,W), 1 = (B,3,T,H,W).
 * t2v_grammar_tokens: int64 tokens [B][8] of "digit {cls} is {a} and {b}." as Vocab.tokenize + collate_fn produce them
 *   (data/__init__.py:260-355); table int64[23] = {START, "digit", "0".."9", "is", "and", END, 4 x (a, b)}, move =
 *   horizontal * 2 + forward (generate.py:144-166).
 * t2v_u8_normalize: dst = (src / 255 - 0.5) / 0.5 with IEEE division (the values of the reference's CPU transform). */
int t2v_moving_digits(const void* bank, const int32_t* digit, const int32_t* pos, void* out, int32_t B, int32_t T,
                      int32_t H, int32_t W, int32_t oh, int32_t ow, int32_t out_f32, int32_t layout, void* stream);
int t2v_grammar_tokens(const int32_t* cls, const int32_t* move, const int64_t* table, int64_t* tokens, int32_t B,
                       void* stream);
int t2v_u8_normalize(const void* src, float* dst, int64_t n, void* stream);
/* Stride-2 convolutions / transposed convolutions of the TGAN and TCWYT families on the tcgen05 engine
 * (models/tcwyt/video_discrim.py:12-25, tcwyt/frame_discrim.py:9-21, tcwyt/gen.py:18-26, tgan/gen.py:20-23,
 * tgan/temporal_gen.py:112-115).  A kernel-4 / stride-2 / padding-1 axis reads inputs 2o-1 .. 2o+2 for output o: with
 * the input grouped in blocks of two samples aligned at odd positions (block b = samples 2b-1, 2b; b = 0..O) output
 * o reads exactly blocks o and o+1 -- a DENSE kernel-2 stride-1 convolution over a block tensor with 2^s * C channels.
 * Per axis `m`: 2 = kernel 4 / stride 2 / padding 1 (even extent), 1 = kernel 1 / stride 1 / padding 0.
 *   t2v_s2d_shift: x (N,D,H,W,C) -> xs (N,D',H',W',Cp), D' = D/2+1 on a strided axis, channel = phase * creal + c for
 *     the creal <= C real channels, phase = ((pd * 2) + ph) * 2 + pw over the strided axes; channels >= 2^s * creal and
 *     samples outside x are zero.  elem_bytes = 2 (bf16) or 4 (fp32).  t2v_d2s_shift is the inverse (channels
 *     >= creal of x are zeroed): a bit-exact index kernel pair.                                                    */
int t2v_s2d_shift(const void* x, void* xs, int64_t N, int32_t D, int32_t H, int32_t W, int32_t C, int32_t creal,
                  int32_t md, int32_t mh, int32_t mw, int32_t Cp, int32_t elem_bytes, void* stream);
int t2v_d2s_shift(const void* xs, void* x, int64_t N, int32_t D, int32_t H, int32_t W, int32_t C, int32_t creal,
                  int32_t md, int32_t mh, int32_t mw, int32_t Cp, int32_t elem_bytes, void* stream);
/* w bf16 [Co][k taps][Ci] (k = 4 per strided axis) -> the block convolution's operand: bf16 [Co][3^s taps][Cp]
 * (engine tap t = block offset + 1; tap 0 of a strided axis stays zero and is never read), or with transposed = 1 the
 * data-gradient / transposed-convolution operand bf16 [Cp][3^s taps reversed][Co]                                 */
int t2v_s2d_embed_weight(const void* w, void* we, int32_t Co, int32_t Ci, int32_t creal, int32_t Cp, int32_t md,
                         int32_t mh, int32_t mw, int32_t transposed, void* stream);
/* dwe fp32 [Co][3^s][Cp] (t2v_conv_wgrad_win on the block tensor) -> dw fp32 [Co][k taps][Ci]                     */
int t2v_s2d_extract_wgrad(const float* dwe, float* dw, int32_t Co, int32_t Ci, int32_t creal, int32_t Cp, int32_t md,
                          int32_t mh, int32_t mw, void* stream);
/* bf16 [Co][taps][Ci] -> bf16 [Ci][taps reversed][Co]: operand of the data gradient / transposed convolution of a
 * stride-1 layer made from the bf16 forward pack (tgan/gen.py:24 ConvTranspose2d k3 s1 p1, tcwyt/gen.py:14,30)   */
int t2v_transpose_flip_bf16(const void* w, void* wT, int32_t Co, int32_t taps, int32_t Ci, void* stream);
/* rows [N][kd*kh*kw*C] <- x[:, :kd, :kh, :kw, :] of x (N,D,H,W,C) (scatter = 0), or x <- zeros with the window
 * written back from rows (scatter = 1): the single-output-position head convolutions of the TCWYT / TGAN critics
 * (tcwyt/frame_discrim.py:55, motion_discrim.py:19, video_discrim.py:46) become Linear layers on the engine      */
int t2v_window_rows(void* x, void* rows, int64_t N, int32_t D, int32_t H, int32_t W, int32_t C, int32_t kd, int32_t kh,
                    int32_t kw, int32_t elem_bytes, int32_t scatter, void* stream);
/* out fp32 [Cp]: out[ph * creal + c] = bias[c] for ph < phases, zero beyond (bias of a transposed convolution in block form) */
int t2v_s2d_tile_bias(const float* bias, float* out, int32_t creal, int32_t phases, int32_t Cp, void* stream);
/* Windowed implicit GEMM on the generic tcgen05 kernels: g = geometry of the OUTPUT positions (fprop) / of dy
 * (wgrad); win9 = {iD, iH, iW, lo_d, hi_d, lo_h, hi_h, lo_w, hi_w}: extents of the tensor the taps read (x) and the live
 * tap range per axis (tap t reads coordinate o + t - k/2, out-of-range coordinates read zero).  Weight layouts as in
 * t2v_conv_fprop / t2v_conv_wgrad (all k taps present in memory, only the live ones touched).  epi_flags: T2V_EPI_RELU,
 * T2V_EPI_OUT_F32.                                                                                                 */
int t2v_conv_fprop_win(const t2v_conv_geom* g, const int32_t* win9, const void* x, const void* w, const float* bias,
                       void* y, uint32_t epi_flags, void* stream);
int t2v_conv_wgrad_win(const t2v_conv_geom* g, const int32_t* win9, const void* dy, const void* x, float* dw,
                       int accumulate, void* stream);
/* fp32 master weight [Cout][taps][Cin] -> bf16 same layout (fprop operand)                    */
int t2v_cast_f32_to_bf16(const float* src, void* dst, int64_t n, void* stream);
int t2v_cast_bf16_to_f32(const void* src, float* dst, int64_t n, void* stream);
/* fp32 master weight [Cout][taps][Cin] -> bf16 [CinP][taps reversed][CoutP] (dgrad operand); the
 * destination must be pre-zeroed when CinP > Cin or CoutP > Cout                                 */
int t2v_pack_dgrad_weight(const float* w, void* wT, int32_t Cout, int32_t taps, int32_t Cin, int32_t CoutP,
                          void* stream);
/* channel-padded operand packs for the convs whose channel count is not a multiple of 16
 * (RGB stem conv resnet3d.py:12,17; render conv layers.py:251; attention 1x1 convs)              */
int t2v_pack_weight_padded(const float* w, void* dst, int32_t Cout, int32_t taps, int32_t Cin, int32_t CinP,
                           void* stream);
int t2v_unpack_wgrad_padded(const float* src, float* dst, int32_t Cout, int32_t taps, int32_t Cin, int32_t CinP,
                            void* stream);

/* activations / pooling / layout (HBM-bound; all tensors bf16 CL unless noted) ---------------- */
/* nn.ReLU: layers.py:172,176,230,232,250; n = element count (multiple of 8)                      */
int t2v_relu_fwd(const void* x, void* y, int64_t n, void* stream);
/* dx = dy * (ref > 0); ref = the ReLU's input or output                                          */
int t2v_relu_bwd(const void* dy, const void* ref, void* dx, int64_t n, void* stream);
/* nn.LeakyReLU(slope) (models/tcwyt/gen.py:16, video_discrim.py:9) and tanh on CL bf16 tensors
 * (models/tgan/temporal_gen.py:33); n elements, multiple of 8; bwd: ref = x or y, y = tanh output     */
int t2v_leaky_relu_fwd(const void* x, void* y, int64_t n, float slope, void* stream);
int t2v_leaky_relu_bwd(const void* dy, const void* ref, void* dx, int64_t n, float slope, void* stream);
int t2v_tanh_fwd(const void* x, void* y, int64_t n, void* stream);
int t2v_tanh_bwd(const void* dy, const void* y, void* dx, int64_t n, void* stream);
/* F.avg_pool3d, count_include_pad, kernel <= stride (layers.py:202-217, resnet3d.py:16,18);
 * in_shape = {N,D,H,W,C}; y = pool(x) (+ residual, y-shaped, may be NULL)                        */
int t2v_avgpool_fwd(const void* x, const void* residual, void* y, const int32_t* in_shape, const int32_t* kernel,
                    const int32_t* stride, const int32_t* pad, void* stream);
int t2v_avgpool_bwd(const void* dy, void* dx, const int32_t* in_shape, const int32_t* kernel, const int32_t* stride,
                    const int32_t* pad, void* stream);
/* nn.Upsample(scale_factor=2) nearest on (N,H,W,C) (layers.py:168,180) and its adjoint            */
int t2v_upsample2x_fwd(const void* x, void* y, int32_t N, int32_t H, int32_t W, int32_t C, void* stream);
int t2v_upsample2x_bwd(const void* dy, void* dx, int32_t N, int32_t H, int32_t W, int32_t C, void* stream);
/* fp32 (N,C,S) <-> bf16 (N,S,Cp) with zero channel padding (D input / G output boundary)         */
int t2v_nchw_to_cl(const float* x, void* y, int64_t N, int32_t C, int64_t S, int32_t Cp, void* stream);
/* RGB clip fp32 (N,3,S) -> bf16 (N,S,16) (y16) and bf16 (N,S,4) (y4), zero padded; either output may be NULL.
 * The discriminator's input boundary: 16-channel rows feed the TMA boxes of the skip path, 4-channel rows the
 * gather of t2v_stem_fprop / t2v_stem_wgrad.                                                          */
int t2v_rgb_to_cl(const float* x, void* y16, void* y4, int64_t N, int64_t S, void* stream);
int t2v_cl_to_nchw(const void* x, float* y, int64_t N, int32_t C, int64_t S, int32_t Cp, void* stream);
/* RGB stem of the discriminator (resnet3d.py:12, Conv3d(C<=4 -> 64, 3^3)) as im2col + 1x1x1 GEMM:
 * col bf16 (N,D,H,W,Kp), col[pos][tap*C+c] = x[c][pos+tap-1] (zero padded; Kp >= 27*C, multiple of 8);
 * t2v_col2im3 is its adjoint (fp32 (N,C,D,H,W) out) for the gradient penalty's d/dx.                */
int t2v_im2col3(const float* x, void* col, int64_t N, int32_t C, int32_t D, int32_t H, int32_t W, int32_t Kp,
                void* stream);
int t2v_col2im3(const void* dcol, float* dx, int64_t N, int32_t C, int32_t D, int32_t H, int32_t W, int32_t Kp,
                void* stream);
/* out[c] = sum_rows x[row,c] (bias gradients)                                                    */
int t2v_sum_rows(const void* x, float* out, int64_t P, int32_t C, void* stream);
/* same, out += column sums (no memset): bias gradients accumulated straight into the parameter's gradient buffer */
int t2v_sum_rows_acc(const void* x, float* out, int64_t P, int32_t C, void* stream);
/* torch.sum(x,[2,3,4]) resnet3d.py:48: out fp32 (N,C) = sum_s x (N,S,C); and its adjoint          */
int t2v_sum_spatial(const void* x, float* out, int64_t N, int64_t S, int32_t C, void* stream);
int t2v_broadcast_spatial(const float* g, void* y, int64_t N, int64_t S, int32_t C, void* stream);

/* BatchNorm2d in train() fused with ReLU and nearest x2 (layers.py:171-173,175-176,249-250) ---- */
/* stats fp32 [2C] = {sum, sum of squares} over P rows                                            */
int t2v_bn_stats(const void* x, float* stats, int64_t P, int32_t C, void* stream);
/* mean_invstd [2C], scale_shift [2C]; updates running stats in place (NULL to skip)               */
int t2v_bn_finalize(const float* stats, const float* gamma, const float* beta, float* running_mean,
                    float* running_var, float* mean_invstd, float* scale_shift, int32_t C, int64_t count,
                    float eps, float momentum, void* stream);
/* y (N,up*H,up*W,C) = act(x*scale+shift) nearest-upsampled by up in {1,2};
 * relu: 0 = identity, 1 = ReLU, 2 = LeakyReLU(0.2) (BatchNorm3d + LeakyReLU of the models/tcwyt files)   */
int t2v_bn_apply(const void* x, const float* scale_shift, void* y, int64_t N, int32_t H, int32_t W, int32_t C,
                 int32_t relu, int32_t up, void* stream);
/* red fp32 [2C] = {dbeta, dgamma}; dx (N,H,W,C)                                                   */
int t2v_bn_bwd(const void* dy, const void* x, const float* scale_shift, const float* mean_invstd, float* red,
               void* dx, int64_t N, int32_t H, int32_t W, int32_t C, int32_t relu, int32_t up, void* stream);
/* double backward of t2v_bn_bwd (up == 1) seen as (dy, x, gamma) -> (dx, dgamma, dbeta), for second-order graphs
 * (the critics' gradient penalty).  x, dy (P,C) CL with the same scale_shift / mean_invstd; upstream gradients
 * ggx (P,C) w.r.t. dx and ggamma / ggbeta fp32 [C] w.r.t. dgamma / dbeta (NULL = zero).  Writes gx (P,C), the
 * gradient w.r.t. x; gdy (P,C), the gradient w.r.t. dy (activation mask applied, as in t2v_bn_bwd); dgamma_out fp32
 * [C], the gradient w.r.t. gamma; red fp32 [5C] receives the per-channel sums {g, g*xhat, ggx, ggx*xhat, ggx*g}
 * (g = masked dy).  Float atomics, no scratch allocation.  T2V_ERR_ARG for up != 1 or C % 8 != 0.            */
int t2v_bn_bwd_bwd(const void* dy, const void* x, const void* ggx, const float* ggamma, const float* ggbeta,
                   const float* scale_shift, const float* mean_invstd, float* red, void* gx, void* gdy,
                   float* dgamma_out, int64_t P, int32_t C, int32_t relu, int32_t up, void* stream);

/* Fused core of the non-local block (models/layers.py:23-36,52-68): o = softmax(theta . maxpool(phi)^T) . maxpool(g)
 * per map, max-pool (1,2,2); theta/phi (N,D,H,W,C8p) and g/o (N,D,H,W,C2p) bf16 CL with c8 <= 8, c2 <= 16 real
 * channels (the rest zero padding); H, W even.  The attention matrix is never materialised.  bwd writes
 * d theta, d phi, d g (full resolution: the pooled gradients land on the arg-max voxel of each window).   */
int t2v_attention_fwd(const void* theta, const void* phi, const void* g, void* o, int64_t N, int32_t D, int32_t H,
                      int32_t W, int32_t c8, int32_t c2, int32_t C8p, int32_t C2p, void* stream);
int t2v_attention_bwd(const void* theta, const void* phi, const void* g, const void* dout, void* dtheta, void* dphi,
                      void* dg, int64_t N, int32_t D, int32_t H, int32_t W, int32_t c8, int32_t c2, int32_t C8p,
                      int32_t C2p, void* stream);
/* the same for maps beyond one CTA of the backward kernel (2 * pooled keys > 512; c8 = 4, c2 = 16, rows padded to 16;
 * up to 2560 pooled keys): two launches (thread = query, then thread = key x query quarter), deterministic;
 * stats_ws = fp32 workspace [N * D*H*W * 3] (softmax maximum, 1 / sum, D_q per query).  BASELINE configs[4]: the
 * generator's block sits on a 64 x 64 map (4096 queries x 1024 keys) there.                                        */
int t2v_attention_bwd_large(const void* theta, const void* phi, const void* g, const void* dout, void* dtheta, void* dphi,
                            void* dg, float* stats_ws, int64_t N, int32_t D, int32_t H, int32_t W, int32_t c8, int32_t c2,
                            int32_t C8p, int32_t C2p, void* stream);

/* RenderBlock tail: tanh + (B*T,H,W,Cp) bf16 -> (B,C,T,H,W) fp32 (layers.py:252, gen.py:116-119)  */
int t2v_render_fwd(const void* pre, float* y, int32_t B, int32_t T, int32_t H, int32_t W, int32_t C, int32_t Cp,
                   void* stream);
int t2v_render_bwd(const float* dy, const float* y, void* dpre, int32_t B, int32_t T, int32_t H, int32_t W,
                   int32_t C, int32_t Cp, void* stream);

/* bit-exact index kernels -------------------------------------------------------------------
 * bt_dev (may be NULL): device int32 holding the frame offset, read by the kernel instead of `bt` so that a
 * captured CUDA graph can be replayed with a fresh draw; the caller then guarantees that the output frame
 * count computed from `bt` holds for every value *bt_dev may take (even T).                       */
/* Subsample x[::sn, :, bt::st] (layers.py:106-111) on merged-frame maps of frame_bytes each;
 * scatter = 1 runs the adjoint (y = zero-filled source-shaped gradient)                           */
int t2v_gather_frames(const void* x, void* y, int32_t B, int32_t T, int64_t frame_bytes, int32_t sn, int32_t st,
                      int32_t bt, const int32_t* bt_dev, int32_t scatter, void* stream);
/* one level of the real-video pyramid (gan/trainer.py:131-165): fp32 (B,C,T,H,W) ->
 * (ceil(B/sn), C, ceil((T-bt)/st), Ho, Wo) with nearest resize src = floor(dst*in/out)            */
int t2v_pyramid_level(const float* x, float* y, const int32_t* in_shape, int32_t Ho, int32_t Wo, int32_t sn,
                      int32_t st, int32_t bt, const int32_t* bt_dev, void* stream);

/* LSTM cell update (conv_lstm.py:32-38; txt/basic.py:56 nn.LSTM): gates fp32 (P,4H) = [i|f|g|o]   */
int t2v_lstm_cell_fwd(const float* gates, const float* c_prev, float* c, void* h, float* h32, int64_t P, int32_t Hd,
                      void* stream);
int t2v_lstm_cell_bwd(const float* gates, const float* c_prev, const float* c, const float* dh, const float* dc_next,
                      void* dgates, float* dc_prev, int64_t P, int32_t Hd, void* stream);

/* torch.optim.Adam (train/gan.py:93-94), multi-tensor: host arrays of `count` device pointers;
 * dyn_dev (may be NULL): device {lr/(1-b1^t), 1/sqrt(1-b2^t)} overriding `step` for CUDA-graph replays   */
int t2v_adam_step(int32_t count, float* const* host_params, const float* const* host_grads, float* const* host_m,
                  float* const* host_v, const int64_t* host_sizes, float lr, float beta1, float beta2, float eps,
                  int32_t step, float grad_scale, const float* dyn_dev, void* stream);

/* gradient bucket pack / unpack for the data-parallel all-reduce (fp32, memory order): dst[i][:] = src[i][:]  */
int t2v_multi_copy(int32_t count, const float* const* host_src, float* const* host_dst, const int64_t* host_sizes,
                   void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * fp32 ACTIVATION STORAGE (the "fp32 parity mode": BASELINE north_star, 1e-3 relative on losses and gradients).
 * Every entry point above whose activations are bf16 CL has a twin with the suffix _f32 and the SAME signature
 * in which those tensors are fp32 CL (same kernels instantiated for float storage; arithmetic is fp32 in both).
 * Convolutions on fp32 storage bypass the bf16 tensor pipe and run as exact fp32 FMAs on the CUDA cores, all on the
 * kernels of the t2v_gconv_*_f32 entry points below: an accumulator per tap (FMA chains of at most Cin terms) added
 * into the total in ascending tap order, and in the weight gradient a flush every 1024 positions.
 * t2v_conv_fprop / t2v_conv_dgrad with T2V_EPI_IN_F32 and t2v_conv_wgrad with T2V_ALGO_SIMT_F32 reach the same
 * kernels for their stride-1 "same" geometry.                                                                  */
int t2v_relu_fwd_f32(const void* x, void* y, int64_t n, void* stream);
int t2v_relu_bwd_f32(const void* dy, const void* ref, void* dx, int64_t n, void* stream);
int t2v_leaky_relu_fwd_f32(const void* x, void* y, int64_t n, float slope, void* stream);
int t2v_leaky_relu_bwd_f32(const void* dy, const void* ref, void* dx, int64_t n, float slope, void* stream);
int t2v_tanh_fwd_f32(const void* x, void* y, int64_t n, void* stream);
int t2v_tanh_bwd_f32(const void* dy, const void* y, void* dx, int64_t n, void* stream);
int t2v_avgpool_fwd_f32(const void* x, const void* residual, void* y, const int32_t* in_shape, const int32_t* kernel,
                        const int32_t* stride, const int32_t* pad, void* stream);
int t2v_avgpool_bwd_f32(const void* dy, void* dx, const int32_t* in_shape, const int32_t* kernel,
                        const int32_t* stride, const int32_t* pad, void* stream);
int t2v_upsample2x_fwd_f32(const void* x, void* y, int32_t N, int32_t H, int32_t W, int32_t C, void* stream);
int t2v_upsample2x_bwd_f32(const void* dy, void* dx, int32_t N, int32_t H, int32_t W, int32_t C, void* stream);
int t2v_nchw_to_cl_f32(const float* x, void* y, int64_t N, int32_t C, int64_t S, int32_t Cp, void* stream);
int t2v_cl_to_nchw_f32(const void* x, float* y, int64_t N, int32_t C, int64_t S, int32_t Cp, void* stream);
int t2v_im2col3_f32(const float* x, void* col, int64_t N, int32_t C, int32_t D, int32_t H, int32_t W, int32_t Kp,
                    void* stream);
int t2v_col2im3_f32(const void* dcol, float* dx, int64_t N, int32_t C, int32_t D, int32_t H, int32_t W, int32_t Kp,
                    void* stream);
int t2v_sum_rows_f32(const void* x, float* out, int64_t P, int32_t C, void* stream);
int t2v_sum_rows_acc_f32(const void* x, float* out, int64_t P, int32_t C, void* stream);
int t2v_sum_spatial_f32(const void* x, float* out, int64_t N, int64_t S, int32_t C, void* stream);
int t2v_broadcast_spatial_f32(const float* g, void* y, int64_t N, int64_t S, int32_t C, void* stream);
int t2v_bn_stats_f32(const void* x, float* stats, int64_t P, int32_t C, void* stream);
int t2v_bn_apply_f32(const void* x, const float* scale_shift, void* y, int64_t N, int32_t H, int32_t W, int32_t C,
                     int32_t relu, int32_t up, void* stream);
int t2v_bn_bwd_f32(const void* dy, const void* x, const float* scale_shift, const float* mean_invstd, float* red,
                   void* dx, int64_t N, int32_t H, int32_t W, int32_t C, int32_t relu, int32_t up, void* stream);
int t2v_bn_bwd_bwd_f32(const void* dy, const void* x, const void* ggx, const float* ggamma, const float* ggbeta,
                       const float* scale_shift, const float* mean_invstd, float* red, void* gx, void* gdy,
                       float* dgamma_out, int64_t P, int32_t C, int32_t relu, int32_t up, void* stream);
int t2v_render_fwd_f32(const void* pre, float* y, int32_t B, int32_t T, int32_t H, int32_t W, int32_t C, int32_t Cp,
                       void* stream);
int t2v_render_bwd_f32(const float* dy, const float* y, void* dpre, int32_t B, int32_t T, int32_t H, int32_t W,
                       int32_t C, int32_t Cp, void* stream);
int t2v_lstm_cell_fwd_f32(const float* gates, const float* c_prev, float* c, void* h, float* h32, int64_t P,
                          int32_t Hd, void* stream);
int t2v_lstm_cell_bwd_f32(const float* gates, const float* c_prev, const float* c, const float* dh,
                          const float* dc_next, void* dgates, float* dc_prev, int64_t P, int32_t Hd, void* stream);
/* general convolution with fp32 x / w / dy (CUDA-core FMA: exact fp32) */
int t2v_gconv_fprop_f32(const t2v_gconv_geom* g, const void* x, const void* w, const float* bias, void* y,
                        int32_t out_f32, void* stream);
int t2v_gconv_dgrad_f32(const t2v_gconv_geom* g, const void* dy, const void* w, const float* bias, void* dx,
                        int32_t out_f32, void* stream);
int t2v_gconv_wgrad_f32(const t2v_gconv_geom* g, const void* dy, const void* x, float* dw, int32_t accumulate,
                        void* stream);

/* scale / add / dot on CL activations (bf16; _f32 twins): the non-local block's gamma * o + x
 * (models/layers.py:36,68) with its gradients, and the gradient penalty's sum ||g||^2 (gan/losses.py:180-186).
 * s, out: ONE fp32 on the device.  n elements, multiple of 8.                                                 */
int t2v_scale(const void* x, const float* s, void* y, int64_t n, void* stream);                  /* y = s * x       */
int t2v_scale_add(const void* o, const void* x, const float* s, void* y, int64_t n, void* stream); /* y = s*o + x (s NULL: 1) */
int t2v_dot(const void* a, const void* b, float* out, int64_t n, void* stream);                 /* out = sum a*b   */
int t2v_scale_f32(const void* x, const float* s, void* y, int64_t n, void* stream);
int t2v_scale_add_f32(const void* o, const void* x, const float* s, void* y, int64_t n, void* stream);
int t2v_dot_f32(const void* a, const void* b, float* out, int64_t n, void* stream);
/* CL [rows][Cp] -> fp32 [rows][c] (first c channels), and its adjoint (zero padding) */
int t2v_cl_slice_f32(const void* x, float* y, int64_t rows, int32_t Cp, int32_t c, void* stream);
int t2v_f32_pad_cl(const float* x, void* y, int64_t rows, int32_t Cp, int32_t c, void* stream);
int t2v_cl_slice_f32_f32(const void* x, float* y, int64_t rows, int32_t Cp, int32_t c, void* stream);
int t2v_f32_pad_cl_f32(const float* x, void* y, int64_t rows, int32_t Cp, int32_t c, void* stream);

/* Non-local block core as differentiable fp32 primitives (models/layers.py:23-36, 52-68): replaces F.max_pool2d/3d,
 * torch.bmm and F.softmax on the discriminator's block, which the gradient penalty differentiates twice.
 * x fp32 [maps][H][W][c] (maps = N*D; pooling window (1,2,2)), idx u8 = arg-max voxel 0..3 of each window.     */
int t2v_maxpool122_fwd(const float* x, float* y, void* idx, int64_t maps, int32_t H, int32_t W, int32_t c,
                       void* stream);
int t2v_pool122_gather(const float* x, const void* idx, float* y, int64_t maps, int32_t H, int32_t W, int32_t c,
                       void* stream);
int t2v_pool122_scatter(const float* dy, const void* idx, float* dx, int64_t maps, int32_t H, int32_t W, int32_t c,
                        void* stream);
/* C[b] (M x N) = op(A[b]) op(B[b]), row-major fp32; trans_a: A[b] stored K x M; trans_b: B[b] stored N x K       */
int t2v_bmm_f32(const float* A, const float* B, float* C, int32_t batch, int32_t M, int32_t N, int32_t K,
                int32_t trans_a, int32_t trans_b, void* stream);
/* row softmax; dS = beta * (dbeta - <beta, dbeta>); and the derivative of that map against a cotangent u
 * (g_beta / g_dbeta may be NULL)                                                                               */
int t2v_softmax_fwd(const float* S, float* out, int64_t rows, int32_t cols, void* stream);
int t2v_softmax_bwd(const float* beta, const float* dbeta, float* dS, int64_t rows, int32_t cols, void* stream);
int t2v_softmax_bwd_bwd(const float* beta, const float* dbeta, const float* u, float* g_beta, float* g_dbeta,
                        int64_t rows, int32_t cols, void* stream);

/* The discriminator's Linear(F [+ E], 1) heads (models/resnet3d.py:50-55) on fp32 features (B,F) [and captions
 * (B,E), may be NULL]: out[b] = [feat | cond][b] . w + bias;  data gradient (outer product);  weight / bias gradient
 * (accumulate = 1 adds into dw / db).  Each is the derivative of another, so the penalty's double backward stays on
 * these kernels.                                                                                               */
int t2v_head_fwd(const float* feat, const float* cond, const float* w, const float* bias, float* out, int32_t B,
                 int32_t F, int32_t E, void* stream);
int t2v_head_bwd_data(const float* dpred, const float* w, float* dfeat, float* dcond, int32_t B, int32_t F, int32_t E,
                      void* stream);
int t2v_head_bwd_weight(const float* dpred, const float* feat, const float* cond, float* dw, float* db, int32_t B,
                        int32_t F, int32_t E, int32_t accumulate, void* stream);
/* Loss reduction over all (level, prediction pair) entries in one launch (gan/cond_gan.py:51-61,108-112):
 * out = sum_e weight_e / n_e * sum_j f(b_e[j] - a_e[j]); mode 0: f = softplus (RSGANLoss, gan/losses.py:74-85),
 * mode 1: f = identity (WassersteinGanLoss, losses.py:55-68).  bwd ADDS into da / db (entries may share tensors;
 * NULL = not needed); gout = d(out) on the device.  At most 24 entries.                                         */
int t2v_rel_loss_fwd(int32_t count, const float* const* host_a, const float* const* host_b, const int32_t* host_n,
                     const float* host_weight, int32_t mode, float* out, void* stream);
int t2v_rel_loss_bwd(int32_t count, const float* const* host_a, const float* const* host_b, float* const* host_da,
                     float* const* host_db, const int32_t* host_n, const float* host_weight, int32_t mode,
                     const float* gout, void* stream);
/* x_hat[b] = alpha[b] * real[b] + (1 - alpha[b]) * fake[b]  (gan/losses.py:140-145), fp32 (B, S)                 */
int t2v_lerp_rows(const float* real, const float* fake, const float* alpha, float* out, int64_t B, int64_t S,
                  void* stream);
/* Non-zero-centred penalty of a single-scale critic (gan/losses.py:180-186, combine = mean) on g fp32 (B, S), 16-byte
 * aligned: norms[b] = ||g_b||_2, out = mean_b (norms[b] - 1)^2, reduced in a fixed order (bit-identical across calls).
 * partials: caller-provided fp32 scratch of B * splits (splits >= 1: blocks per sample).  bwd: dg = gout * 2 (n_b - 1)
 * / (n_b B) * g, 0 on rows with n_b = 0; gout on the device.  T2V_ERR_ARG for B < 1 or S % 4 != 0.             */
int t2v_gp_norm_fwd(const float* g, float* partials, float* norms, float* out, int64_t B, int64_t S, int32_t splits,
                    void* stream);
int t2v_gp_norm_bwd(const float* g, const float* norms, const float* gout, float* dg, int64_t B, int64_t S,
                    void* stream);

/* Caption encoder / decoder recurrence (models/txt/basic.py:18-19,49-101: nn.Embedding + nn.LSTM on a
 * PackedSequence), replacing cuDNN.  gx fp32 [B][L][ndir][4H] = W_ih x + b_ih + b_hh (one GEMM on the engine);
 * whhT fp32 [ndir][H][4H] from t2v_lstm_pack_whh(whh [ndir][4H][H]); lengths int32 [B] (descending as
 * pack_padded_sequence requires); h0 / c0 fp32 [ndir][B][H] or NULL.  out / hprev: CL storage type [B][L][ndir*H]
 * (zeros at padded steps; hprev = the state entering each step, NULL to skip); gates / cells: fp32 saved for
 * backward (NULL to skip); hn / cn fp32 [ndir][B][H].  bwd: dgates [B][L][ndir*4H] storage type.                 */
int t2v_lstm_pack_whh(const float* whh, float* whhT, int32_t ndir, int32_t H, void* stream);
int t2v_lstm_seq_fwd(const float* gx, const float* whhT, const int32_t* lengths, const float* h0, const float* c0,
                     void* out, void* hprev, float* gates, float* cells, float* hn, float* cn, int32_t B, int32_t L,
                     int32_t H, int32_t ndir, void* stream);
int t2v_lstm_seq_bwd(const float* whh, const int32_t* lengths, const float* c0, const float* gates,
                     const float* cells, const void* dout, const float* dhn, const float* dcn, void* dgates,
                     float* dh0, float* dc0, int32_t B, int32_t L, int32_t H, int32_t ndir, void* stream);
int t2v_lstm_seq_fwd_f32(const float* gx, const float* whhT, const int32_t* lengths, const float* h0, const float* c0,
                         void* out, void* hprev, float* gates, float* cells, float* hn, float* cn, int32_t B,
                         int32_t L, int32_t H, int32_t ndir, void* stream);
int t2v_lstm_seq_bwd_f32(const float* whh, const int32_t* lengths, const float* c0, const float* gates,
                         const float* cells, const void* dout, const float* dhn, const float* dcn, void* dgates,
                         float* dh0, float* dc0, int32_t B, int32_t L, int32_t H, int32_t ndir, void* stream);
/* nn.Embedding: out[row] = weight[tokens[row]] (int64 tokens, bit-exact gather) and its weight gradient       */
int t2v_embedding_fwd(const int64_t* tokens, const float* weight, void* out, int64_t rows, int32_t E, void* stream);
int t2v_embedding_bwd(const int64_t* tokens, const void* dout, float* dweight, int64_t rows, int32_t E, int64_t V,
                      void* stream);
int t2v_embedding_fwd_f32(const int64_t* tokens, const float* weight, void* out, int64_t rows, int32_t E,
                          void* stream);
int t2v_embedding_bwd_f32(const int64_t* tokens, const void* dout, float* dweight, int64_t rows, int32_t E, int64_t V,
                          void* stream);

#ifdef __cplusplus
}
#endif
#endif /* T2V_H_ */
