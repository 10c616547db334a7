/*
 * flowdiff.h -- C ABI of libflowdiff.so, the sm_100a kernel library behind the
 * flow_diffuser hot path of davidfang00/opticalflowdiffusion.
 *
 * Conventions (all entry points):
 *   - plain pointers and sizes, no torch / C++ types;
 *   - every pointer is DEVICE memory owned by the caller (PyTorch); kernels are enqueued on
 *     `stream` (a cudaStream_t passed as void*), never synchronise and never allocate;
 *   - return 0 on success, a negative FD_E* code otherwise; fd_last_error() gives a
 *     thread-local message;
 *   - fp32 image-space tensors are NCHW contiguous (the reference's layout); UNet activations
 *     are bf16 NHWC ("pixel rows" of C channels), weights are packed bf16 [Cout][K].
 *
 * Each group cites the reference code (file:line under the reference repo) it replaces.
 */
#ifndef FLOWDIFF_H_
#define FLOWDIFF_H_

#include <stddef.h>
#include <stdint.h>

#if defined(FD_BUILDING_LIB)
#define FD_API __attribute__((visibility("default")))
#else
#define FD_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define FD_OK 0
#define FD_EINVAL (-1)   /* bad argument / unsupported shape */
#define FD_ECUDA (-2)    /* CUDA runtime / driver error */
#define FD_EARCH (-3)    /* device is not sm_100 */

/* ---- library info ------------------------------------------------------------------ */
FD_API int fd_version(void);                 /* 100 * major + minor */
FD_API const char* fd_arch(void);            /* "sm_100a" */
FD_API const char* fd_last_error(void);
FD_API int fd_device_check(void);            /* FD_OK iff the current device is compute capability 10.x */
FD_API int fd_num_sms(void);
FD_API unsigned long long fd_launch_count(void);   /* kernels launched by the library so far (this process) */

/* ---- backward bilinear warp:  warp.py:95-119 (warp_backward_flow) --------------------
 * flow channel 0 = dy, channel 1 = dx (the reference flips).  out is NOT multiplied by mask.
 * The coordinate / weight / accumulation sequence is the one torch's CPU grid_sample performs
 * (see oracle/flowdiff_oracle.py:backwarp) and is bit-exact against it. */
FD_API int fd_backwarp_fwd(const float* image, const float* flow, float* out, float* mask,
                    int B, int C, int H, int W, void* stream);
/* grads of sum(out * gout): gimage (B,C,H,W) is zero-filled by the call; either may be NULL */
FD_API int fd_backwarp_bwd(const float* image, const float* flow, const float* gout,
                    float* gimage, float* gflow, int B, int C, int H, int W, void* stream);

/* Backward passes with a caller-provided workspace (fd_warp_bwd_workspace_floats(B, H, W) floats, 16-byte aligned): on
 * three-channel frames with W % 4 == 0 the gradient of the sampled frame is accumulated pixel-interleaved in the workspace
 * with ONE 128-bit reduction per bilinear tap (4 instead of 12 L2 reduction operations per pixel; the gathers read the frame
 * from TMA-staged shared-memory windows) and converted to the planar gradient by a second launch.  Same arguments and
 * results as fd_backwarp_bwd / fd_backwarp_photo_epe_bwd, which serve every other shape (and a NULL workspace). */
FD_API size_t fd_warp_bwd_workspace_floats(int B, int H, int W);
FD_API int fd_backwarp_bwd_ws(const float* image, const float* flow, const float* gout, float* gimage, float* gflow,
                     float* workspace, int B, int C, int H, int W, void* stream);
FD_API int fd_backwarp_photo_epe_bwd_ws(const float* frame1, const float* frame2, const float* flow, const float* flow_gt,
                     const float* sums, float g_photo, float g_epe, float* gflow, float* gframe2, float* workspace,
                     int B, int C, int H, int W, void* stream);

/* Self-test of the warp kernels' division: the normalisation `2 v / (W - 1)` of warp.py:107-108 is computed with the
 * reciprocal half of `__fdiv_rn`'s own instruction sequence hoisted out of the pixel loop (fd_warp_common.cuh:bw_div_rn);
 * this runs ALL 2^32 numerator bit patterns for one divisor against `__fdiv_rn` and counts the differences (expected: 0). */
FD_API int fd_warp_div_selftest(float divisor, unsigned long long* mismatches, void* stream);

/* fused warp + Charbonnier photometric + end-point error (BASELINE config #4):
 *   warped, mask = backwarp(frame2, flow)
 *   sums[0] = sum(mask * sqrt((frame1-warped)^2 + 1e-6))   losses.py:3-6,46-47
 *   sums[1] = sum(mask)                                     (over B*C*H*W, like the reference's mask)
 *   sums[2] = sum_px sqrt(du^2 + dv^2),  sums[3] = B*H*W
 * partials: workspace of fd_photo_epe_workspace_floats(B,H,W) floats, 4-byte aligned, ANY contents on entry (the kernel's
 * last-block ticket is a {launch tag, count} word that it claims and clears itself; one workspace per call in flight).
 * Deterministic. */
FD_API size_t fd_photo_epe_workspace_floats(int B, int H, int W);
FD_API int fd_backwarp_photo_epe_fwd(const float* frame1, const float* frame2, const float* flow,
                              const float* flow_gt, float* sums, float* partials,
                              int B, int C, int H, int W, void* stream);
/* backward of  L = g_photo * sums[0]/sums[1] + g_epe * sums[2]/sums[3]  (mask treated as constant,
 * as autograd does through the reference's thresholding): gflow (B,2,H,W), gframe2 (B,C,H,W, zero-filled) */
FD_API int fd_backwarp_photo_epe_bwd(const float* frame1, const float* frame2, const float* flow,
                              const float* flow_gt, const float* sums, float g_photo, float g_epe,
                              float* gflow, float* gframe2, int B, int C, int H, int W, void* stream);

/* ---- forward splat: softsplat_new.py:352-423 / 489-565 / 600-700 ----------------------
 * flow channel 0 = dx, channel 1 = dy.  out is (B,C,H/scale,W/scale) and is zero-filled by the call. */
FD_API int fd_splat_fwd(const float* in, const float* flow, float* out,
                 int B, int C, int H, int W, int scale, int off_x, int off_y, void* stream);
FD_API int fd_splat_ingrad(const float* flow, const float* gout, float* gin,
                    int B, int C, int H, int W, int scale, int off_x, int off_y, void* stream);
FD_API int fd_splat_flowgrad(const float* in, const float* flow, const float* gout, float* gflow,
                      int B, int C, int H, int W, int scale, int off_x, int off_y, void* stream);
/* warp_forward_flow pre-processing (warp.py:122-126 + softsplat_new.py:301-302, mode linear_unn):
 * ten_in (B,C+1,HW): [:C] = nan_to_zero(first) * w, [C] = w, w = any_c(isnan(first)) ? 0 : 1 */
FD_API int fd_splat_prepare(const float* first, float* ten_in, int B, int C, int HW, void* stream);
/* warp_forward_flow post-processing (warp.py:139-156): img[b,c] = splat[b,C]>0 ? splat[b,c] : NaN; splat is (B,C+1,HW) */
FD_API int fd_splat_finish(const float* splat, float* img, int B, int C, int HW, int set_nans, void* stream);
/* fd_splat_fwd with a caller-provided workspace (fd_splat_fwd_workspace_floats floats, 16-byte aligned): for C = 3 or 4 the
 * splat is accumulated pixel-interleaved with one 128-bit reduction per tap and copied out to the planar `out`; every other
 * channel count (or a NULL workspace) runs fd_splat_fwd.  Same results up to the order of the atomics. */
FD_API size_t fd_splat_fwd_workspace_floats(int B, int H, int W, int scale);
FD_API int fd_splat_fwd_ws(const float* in, const float* flow, float* out, float* workspace, int B, int C, int H, int W,
                     int scale, int off_x, int off_y, void* stream);
/* warp_forward_flow(warp_style='sum') for THREE-channel images in two launches (warp.py:121-156; prepare + splat + finish
 * fused): `acc` is a caller-provided workspace of 4*B*(H/scale)*(W/scale) floats, 16-byte aligned, in which the splat is
 * accumulated pixel-interleaved (r, g, b, weight) so that a tap is one 128-bit vector reduction; img (B,3,H/s,W/s) receives
 * the image (holes -> NaN when set_nans), wsum (B,1,H/s,W/s, may be NULL) the splatted weight, ten_in (B,4,H,W, may be
 * NULL) the prepared splat input for the backward kernels (fd_splat_ingrad / fd_splat_flowgrad). */
FD_API int fd_forward_warp_sum3(const float* first, const float* flow, float* ten_in, float* acc, float* img, float* wsum,
                     int B, int H, int W, int scale, int off_x, int off_y, int set_nans, void* stream);

/* ---- NaN-aware MSE: warp.py:260-271 + torch.nanmean (denoising_diffusion.py:908,973) --------
 * sums[0] = sum over non-NaN pairs of (pred-target)^2, sums[1] = count, sums[2] = their ratio; strided channel-slice views:
 * element (b, c, i) lives at ptr[b*bstride + c*HW + i], c < C. */
FD_API int fd_nan_mse_fwd(const float* pred, const float* target, float* sums, float* partials,
                   int B, int C, int HW, long pred_bstride, long target_bstride, void* stream);
FD_API size_t fd_nan_mse_workspace_floats(int B, int C, int HW);
/* gpred = gscale * 2 (pred-target) on non-NaN pairs else 0, gscale = upstream / count */
FD_API int fd_nan_mse_bwd(const float* pred, const float* target, const float* sums, float upstream,
                   float* gpred, int B, int C, int HW, long pred_bstride, long target_bstride,
                   long gpred_bstride, void* stream);

/* ---- scheduler: denoising_diffusion.py:806-812 (q_sample), 653-656 + 752-767 (DDIM),
 *      666-698 + 613-623 (DDPM ancestral) ---------------------------------------------------- */
/* out = a[t_b] * x0 + s[t_b] * noise ; t int64 (B), tables fp32 device (T) */
FD_API int fd_q_sample(const float* x0, const float* noise, const int64_t* t, const float* sqrt_ac,
                const float* sqrt_1mac, float* out, int B, long per_sample, void* stream);
/* x0 = clamp(model_out,-1,1); eps = (recip*x - x0)/recipm1;
 * last ? x_next = x0 : x_next = x0*sqrt_alpha_next + c*eps + sigma*noise (noise may be NULL iff sigma==0).
 * x0_out optional. In-place (x_next == x) allowed. */
FD_API int fd_ddim_step(const float* x, const float* model_out, const float* noise, float* x_next, float* x0_out,
                 long n, float recip, float recipm1, float sqrt_alpha_next, float c, float sigma,
                 int last, void* stream);
/* DPM-Solver++ multistep step (data prediction, orders 1-3; not in the reference):
 * D0 = clamp(model_out,-1,1); d_out = D0;
 * last ? x_next = D0 : x_next = ((cx*x + c0*D0) + c1*d_hist1) + c2*d_hist2, fp32, no FMA, in that order.
 * A term with a zero coefficient is not evaluated (NaN in unused history does not leak); d_hist1 / d_hist2 may be
 * NULL when c1 / c2 == 0. Aliasing: x_next == x and d_out == d_hist2 are allowed (each element is read before it
 * is written), so two rotating history buffers suffice for order 3; no other pair may overlap. */
FD_API int fd_dpmpp_step(const float* x, const float* model_out, const float* d_hist1, const float* d_hist2,
                  float* x_next, float* d_out, long n, float cx, float c0, float c1, float c2, int last,
                  void* stream);
/* x0 = clamp(model_out,-1,1); x_next = coef1*x0 + coef2*x + (noise ? sigma*noise : 0) */
FD_API int fd_ddpm_step(const float* x, const float* model_out, const float* noise, float* x_next, float* x0_out,
                 long n, float coef1, float coef2, float sigma, void* stream);

/* ---- UNet building blocks: denoising_diffusion.py:81-417 ---------------------------------- */
/* Unet.forward input assembly (:367-368 cat + flow_diffuser.py:39-45 NaN mask) for the 7x7 init conv
 * (:297,374), emitted as the 7-tap "row-im2col" tensor packed[b,h,w, kx*Cpad + c] = in[b,c,h,w+kx-3]
 * (bf16, 64 channels per pixel, zero outside the image / above Cpad*7).  x:(B,Cx,H,W) cond:(B,Cc,H,W)
 * fp32 NCHW; if nan_mask: NaNs of x become 0 and a channel any_c(isnan(x)) is inserted after x.
 * Ctot = Cx + nan_mask + Cc must be <= 9.
 * x / cond are H0 x W0 planes that sit at (pad_top, pad_left) inside the H x W frame the UNet runs on
 * (H, W multiples of 8: three pixel-unshuffle downsamples, :95-99); the border is replicate-padded on the fly, i.e.
 * InputPadder(mode='sintel') (future/raft_utils.py:7-25) folded into the packing: 436x1024 -> 440x1024 costs no pass. */
FD_API int fd_pack_input_pad(const float* x, const float* cond, void* packed, int B, int Cx, int Cc, int H0, int W0,
                      int pad_top, int pad_left, int H, int W, int nan_mask, void* stream);
/* More than 9 input channels (latent mode: flow_diffuser.py:98-110 builds the UNet over latent_dim + ... = 33-35 channels,
 * flow_pred.py:31-37 the decoder over latent_dim + 3): same NaN / mask / replicate-pad semantics, packed as plain bf16
 * (B,H,W,64) with the channels zero-padded to 64; init_conv then runs as a 49-tap fd_conv_igemm with kind-3 weights. */
FD_API int fd_pack_input_wide(const float* x, const float* cond, void* packed, int B, int Cx, int Cc, int H0, int W0,
                      int pad_top, int pad_left, int H, int W, int nan_mask, void* stream);

/* Weight preparation.  w: fp32 [Cout][Cin][KH][KW] (torch layout) -> bf16 [Cout][K] K-major.
 * kind 0: K index = (ky*KW+kx)*Cin + ci                       (implicit-GEMM tap-major order)
 * kind 1: pixel-unshuffle 1x1 (:95-99): Cin = 4*C, torch channel c*4+p1*2+p2 -> K = (p1*2+p2)*C + c
 * kind 2: 7x7 init conv as 7 taps of 64: K = ky*64 + kx*Cin + ci, zero padded
 * kind 3: tap-major over an input zero-padded to 64 channels: K = (ky*KW+kx)*64 + ci (Cin <= 64; the wide init conv)
 * standardize != 0 applies WeightStandardizedConv2d (:106-114) with eps before packing. */
FD_API int fd_prep_weight(const float* w, void* packed, int Cout, int Cin, int KH, int KW, int kind,
                   int standardize, float eps, void* stream);

/* Implicit-GEMM convolution on tcgen05 tensor cores (the nn.Conv2d / WeightStandardizedConv2d calls
 * at :92,98,114,200,222,225,253,254,297,339,354).  Activations bf16 NHWC.
 *   out[n,h,w,co] = bias[co] + sum_{tap,ci} src[n, h+dy(tap), w+dx(tap), ci] * wpacked[co][tap*Cin+ci]
 *                   (+ residual[n,h,w,co])
 * src = channel-concatenation of src0 (C0 ch) and src1 (C1 ch, may be NULL) -- the skip concat of
 * :405,408,414 without materialising it.  C0, C1 multiples of 64; Cout multiple of 64 (<=256 or a
 * multiple of 128/192/256 tiles).
 * mode 0: KHxKW taps, zero padding (pad_h, pad_w), stride 1; H,W = spatial size of src and out.
 * mode 1: pixel-unshuffle + 1x1: src is (N, 2H, 2W, C0), taps (p1,p2), out (N,H,W,Cout).
 * gn_stats (optional): double [N][8][2]; (sum, sum of squares) of the fp32 results per sample and
 *   GroupNorm group are atomically accumulated (caller zero-fills) -- the statistics pass of
 *   Block.forward's GroupNorm (:176,181) fused into the producer.
 * 1x1 convolutions without statistics treat the whole batch as one row of pixels (any H, W). */
FD_API int fd_conv_igemm(const void* src0, int C0, const void* src1, int C1, const void* wpacked,
                  const float* bias, const void* residual, void* out, double* gn_stats,
                  int N, int H, int W, int Cout, int KH, int KW, int pad_h, int pad_w, int mode,
                  void* stream);

/* fd_conv_igemm with an output mode.  out_mode 0: as fd_conv_igemm.  out_mode 1 (the data gradient of
 * Downsample, :95-99): a 1x1 conv whose Cout = 4*Cq channels are stored pixel-shuffled, channel
 * (p1*2+p2)*Cq + c of pixel (h, w) -> pixel (2h+p1, 2w+p2), channel c of out (N, 2H, 2W, Cq); Cout % 256 == 0,
 * no residual / statistics. */
FD_API int fd_conv_igemm_ex(const void* src0, int C0, const void* src1, int C1, const void* wpacked,
                     const float* bias, const void* residual, void* out, double* gn_stats,
                     int N, int H, int W, int Cout, int KH, int KW, int pad_h, int pad_w, int mode,
                     int out_mode, void* stream);
/* Upsample (:89-93): nearest x2 + 3x3 conv (pad 1) WITHOUT materialising the up-sampled tensor: four 2x2 convolutions on the
 * low-resolution grid, one per output phase, with the coinciding taps' weights added (2.25x fewer MACs).
 * fd_prep_weight_upconv: w fp32 [Cout][Cin][3][3] -> packed bf16 [4 phases][Cout][4*Cin].
 * fd_conv_igemm_up: src bf16 (N,H,W,Cin) -> out bf16 (N,2H,2W,Cout), bias fp32 [Cout] or NULL. */
FD_API int fd_prep_weight_upconv(const float* w, void* packed, int Cout, int Cin, void* stream);
FD_API int fd_conv_igemm_up(const void* src, int Cin, const void* wpacked4, const float* bias, void* out, int N, int H, int W,
                     int Cout, void* stream);

/* fd_conv_igemm whose residual input is a RAW conv output h2 that still needs its GroupNorm(8) + SiLU
 * (ResnetBlock with a res_conv, :212-214: out = res_conv(x) + silu(GroupNorm(h2))): the epilogue folds
 * res_stats ([N][8][2] sum / sum of squares of h2, as accumulated by the producing conv), gamma, beta into per-channel
 * coefficients and applies them to the residual on the fly -- the activated tensor never goes through HBM. */
FD_API int fd_conv_igemm_rt(const void* src0, int C0, const void* src1, int C1, const void* wpacked, const float* bias,
                     const void* residual_raw, const double* res_stats, const float* res_gamma, const float* res_beta,
                     float eps, void* out, int N, int H, int W, int Cout, int KH, int KW, int pad_h, int pad_w, void* stream);

/* The UNet's last two lines in one launch (Unet.forward, denoising_diffusion.py:414-417: the final ResnetBlock's
 * res_conv + residual, then final_conv 1x1 64 -> out_dim): fd_conv_igemm_rt for a 1x1 conv with Cout = 64 whose epilogue
 * applies final_conv (head_w fp32 [head_n][64], head_b fp32 [head_n], head_n <= 4) to the fp32 tile and writes
 * out_nchw fp32 (N, head_n, H0, W0) = the H0 x W0 window at (pad_top, pad_left) of the padded H x W grid
 * (InputPadder.unpad).  The 64-channel activation never goes through HBM. */
FD_API int fd_conv_igemm_rt_head(const void* src0, int C0, const void* src1, int C1, const void* wpacked, const float* bias,
                     const void* residual_raw, const double* res_stats, const float* res_gamma, const float* res_beta,
                     float eps, const float* head_w, const float* head_b, int head_n, float* out_nchw, int N, int H, int W,
                     int H0, int W0, int pad_top, int pad_left, void* stream);


/* 3x3 / pad 1 / 64 -> 64 channel convolution whose INPUT is activated on the fly:
 *   out = conv3x3(silu(GroupNorm(src) * (scale + 1) + shift)) (+ bias, + residual, + GroupNorm statistics of out)
 * i.e. fd_gn_silu (Block.forward, denoising_diffusion.py:176-187) fused into the consuming block2.proj convolution
 * (ResnetBlock.forward :202-214): the activated tensor is never written to memory.  in_stats are the (sum, sum of squares)
 * statistics of src as produced by the convolution that wrote it; the other arguments as fd_gn_silu / fd_conv_igemm.
 * Same folded coefficients as fd_gn_silu; the in-kernel SiLU uses tanh.approx (within 2^-10 of fd_silu before the bf16
 * rounding of the activation).  Needs W >= 64. */
FD_API int fd_conv3x3_gnsilu_in(const void* src, const double* in_stats, const float* in_gamma, const float* in_beta,
                                const float* in_scale_shift, long in_ss_stride, float in_eps, const void* wpacked,
                                const float* bias, const void* residual, void* out, double* gn_stats, int N, int H, int W,
                                void* stream);

/* Weight gradient of the same convolutions (autograd of the nn.Conv2d calls above) on tcgen05, K = pixels:
 *   dw[co][tap*Cin + ci] += sum_{n,h,w} src[n, h+dy(tap), w+dx(tap), ci] * dy[n,h,w,co]      (fp32, packed order of
 * fd_prep_weight kind 0 / 1; caller zero-fills).  src = concat(src0, src1) as in fd_conv_igemm; mode as there
 * (mode 1: src is (N, 2H, 2W, C0), dy (N,H,W,Cout), taps (p1,p2)).  fp32 atomics: summation order is not fixed. */
FD_API int fd_conv_wgrad(const void* src0, int C0, const void* src1, int C1, const void* dy, float* dw,
                  int N, int H, int W, int Cout, int KH, int KW, int pad_h, int pad_w, int mode, void* stream);

/* GroupNorm(8) apply + optional (scale+1, shift) + SiLU (+ optional residual add), bf16 NHWC:
 * Block.forward :181-187 and ResnetBlock's "+ res_conv(x)" :214.  stats from fd_conv_igemm.
 * scale_shift: fp32, row n at scale_shift + n*ss_stride holds [scale(C) | shift(C)] (time_emb.chunk(2), :208)
 * or NULL.  gn_stats: double [N][8][2] as accumulated by fd_conv_igemm. */
FD_API int fd_gn_silu(const void* x, const double* gn_stats, const float* gamma, const float* beta,
               const float* scale_shift, long ss_stride, const void* residual, void* out,
               int N, int HW, int C, float eps, void* stream);
/* The same transform with SiLU as h + h tanh(h), h = z/2 (one tanh.approx per element, within 2^-10 of fd_gn_silu before
 * the bf16 rounding): what the inference forward (sampling) calls; the fused forms of this transform (fd_conv3x3_gnsilu_in,
 * fd_conv_igemm_rt) use the same expression. */
FD_API int fd_gn_silu_fast(const void* x, const double* gn_stats, const float* gamma, const float* beta,
               const float* scale_shift, long ss_stride, const void* residual, void* out,
               int N, int HW, int C, float eps, void* stream);

/* channel LayerNorm (:116-125) over C per pixel, out = (x-mean)*rsqrt(var+eps)*g (+ residual) */
FD_API int fd_chan_layernorm(const void* x, const float* g, const void* residual, void* out,
                      long npix, int C, float eps, void* stream);

/* nearest 2x upsample (:91), bf16 NHWC (N,H,W,C) -> (N,2H,2W,C) */
FD_API int fd_upsample2x(const void* x, void* out, int N, int H, int W, int C, void* stream);

/* SinusoidalPosEmb + time_mlp (:144-151, 319-324): t int64 (B) -> temb fp32 (B,256) */
FD_API int fd_time_embed(const int64_t* t, const float* w1, const float* b1, const float* w2, const float* b2,
                  float* temb, int B, int dim, int time_dim, void* stream);
/* ResnetBlock.mlp (:193-196, 206): out[b][j] = bias[j] + sum_k silu(temb[b][k]) * w[j][k] ; w [J][time_dim] */
FD_API int fd_time_proj(const float* temb, const float* w, const float* bias, float* out, int B, int time_dim,
                 int J, void* stream);

/* LinearAttention core (:229-243) on qkv bf16 (N, HW, 384) [q | k | v, each heads*32]:
 *   q softmax over d, *scale; k softmax over pixels; v / HW; ctx = k v^T; out = ctx^T q  -> bf16 (N,HW,128).
 * workspace floats: fd_linattn_workspace_floats(N, HW). */
FD_API size_t fd_linattn_workspace_floats(int N, int HW);
FD_API int fd_linattn(const void* qkv, void* out, float* workspace, int N, int HW, void* stream);
/* the context half of fd_linattn: kv rows = [k(128) | v(128)] bf16, row_stride elements apart -> ctx_t bf16
 * [N][4][32 e][32 d] (softmax_n(k) v^T / HW, with the 32^-0.5 q scale folded in); workspace as fd_linattn_workspace_floats. */
FD_API int fd_linattn_context(const void* kv, int row_stride, void* ctx_t, float* workspace, int N, int HW, void* stream);

/* Residual(PreNorm(LinearAttention)) (:81-87,127-135,216-244) for C in {64,128} on tcgen05 / TMEM / TMA: two passes over
 * x, no intermediate tensor in HBM (csrc/fd_linattn_tc.cu).
 * fd_linattn_tc_prep (once per weight update): to_qkv.weight fp32 [384][C] and the PreNorm gain g1[C] ->
 *   wq, wk bf16 [128][C] (rows scaled by g1 and log2 e), sq, sk fp32 [128] (their row sums), mk fp32 [128] (upper bound of
 *   the k logit = the pixel-softmax shift), wv fp32 [128][C].
 * fd_linattn_tc: x, out bf16 (N,HW,C); wout fp32 [C][128], bout fp32 [C] (to_out.0), g2 fp32 [C] (to_out.1.g);
 *   workspace: fd_linattn_tc_workspace_floats(N, HW, C) floats. */
FD_API size_t fd_linattn_tc_workspace_floats(int N, int HW, int C);
FD_API int fd_linattn_tc_prep(const float* wqkv, const float* g1, void* wq, float* sq, void* wk, float* sk, float* mk,
                       float* wv, int C, void* stream);
FD_API int fd_linattn_tc(const void* x, const void* wk, const float* sk, const float* mk, const void* wq, const float* sq,
                  const float* wv, const float* wout, const float* bout, const float* g2, void* out, float* workspace,
                  int N, int HW, int C, float eps, void* stream);

/* Attention core (:256-267): softmax(q^T k * 32^-0.5) v, flash-style, bf16 (N,HW,384) -> (N,HW,128) */
FD_API int fd_attention(const void* qkv, void* out, int N, int HW, void* stream);

/* Logging reductions of training_step / validation_step (flow_diffuser.py:221-232, 262-282) in one pass: x fp32 (B, inner)
 * -> out4 = {torch.min(x), torch.max(x), torch.mean(x), torch.mean(torch.std(x, dim=0))} (unbiased std over the batch axis;
 * NaN propagation as torch).  workspace: fd_tensor_stats_workspace_floats(inner) floats.  Deterministic, no host sync. */
FD_API size_t fd_tensor_stats_workspace_floats(long inner);
FD_API int fd_tensor_stats(const float* x, int B, long inner, float* out4, float* workspace, void* stream);

/* final 1x1 conv (:361,417) 64 -> Cout (<= 64; four output channels per launch) on a bf16 NHWC (N,H,W,64) frame, writing
 * only the H0 x W0 window at (pad_top, pad_left) as fp32 (N,Cout,H0,W0): the InputPadder.unpad crop
 * (future/raft_utils.py:20-25) folded into the store. */
FD_API int fd_final_conv_crop(const void* x, const float* w, const float* bias, float* out, int N, int H, int W, int Cin,
                       int Cout, int pad_top, int pad_left, int H0, int W0, void* stream);

/* ==== backward pass: the autograd graph `loss.backward()` walks in training_step (flow_diffuser.py:217-235,
 *      exp_base.py:193-214) for the modules above ================================================ */

/* Attention core that also saves the log2-domain log-sum-exp of the scaled scores, lse fp32 [N][4][HW] (may be NULL) */
FD_API int fd_attention_lse(const void* qkv, void* out, float* lse, int N, int HW, void* stream);
/* backward of fd_attention: out / dout bf16 (N,HW,128), dqkv bf16 (N,HW,384); deterministic (no atomics).
 * workspace floats: fd_attention_bwd_workspace_floats(N, HW). */
FD_API size_t fd_attention_bwd_workspace_floats(int N, int HW);
FD_API int fd_attention_bwd(const void* qkv, const void* out, const void* dout, const float* lse, void* dqkv,
                     float* workspace, int N, int HW, void* stream);

/* fp32 statistics of LinearAttention's k softmax: stats [N][ max(128) | sum-exp(128) | ctx(4*32*32) ];
 * workspace as fd_linattn_workspace_floats. */
FD_API int fd_linattn_stats(const void* kv, int row_stride, float* stats, float* workspace, int N, int HW, void* stream);
/* fd_linattn that also writes those statistics (N * fd_linattn_stats_floats() floats) from the same partial sums */
FD_API size_t fd_linattn_stats_floats(void);
FD_API int fd_linattn_save(const void* qkv, void* out, float* stats, float* workspace, int N, int HW, void* stream);
/* backward of fd_linattn: dout bf16 (N,HW,128) -> dqkv bf16 (N,HW,384); saved_stats from fd_linattn_save or NULL
 * (then they are recomputed); workspace fd_linattn_bwd_workspace_floats */
FD_API size_t fd_linattn_bwd_workspace_floats(int N, int HW);
FD_API int fd_linattn_bwd(const void* qkv, const void* dout, void* dqkv, const float* saved_stats, float* workspace,
                   int N, int HW, void* stream);

/* backward of fd_gn_silu (Block.forward :181-187): h = the conv output the forward normalised, da = gradient of the
 * activation output -> dh (bf16), and ACCUMULATES (+=, fp32) dgamma[C], dbeta[C], dbias[C] (the producing conv's bias
 * gradient = sum over pixels of dh; may be NULL); writes dscale_shift rows like scale_shift (NULL iff scale_shift NULL).
 * workspace floats: fd_gn_silu_bwd_workspace_floats(N, C). */
FD_API size_t fd_gn_silu_bwd_workspace_floats(int N, int C);
FD_API int fd_gn_silu_bwd(const void* h, const void* da, const double* gn_stats, const float* gamma, const float* beta,
                   const float* scale_shift, long ss_stride, void* dh, float* dgamma, float* dbeta,
                   float* dscale_shift, float* dbias, float* workspace, int N, int HW, int C, float eps, void* stream);
/* backward of fd_chan_layernorm: dx = LN'(dy) (+ add, bf16, may be NULL), dg[C] += sum_px dy * xhat */
FD_API int fd_chan_layernorm_bwd(const void* x, const float* g, const void* dy, const void* add, void* dx, float* dg,
                          long npix, int C, float eps, void* stream);
/* backward of fd_upsample2x: dy (N,2H,2W,C) -> dx (N,H,W,C) */
FD_API int fd_upsample2x_bwd(const void* dy, void* dx, int N, int H, int W, int C, void* stream);
/* out = a + b over n bf16 elements (n % 8 == 0); out may alias a or b */
FD_API int fd_add_bf16(const void* a, const void* b, void* out, long n, void* stream);
/* db[C] += sum over pixels of dy (bf16 [npix][C]) */
FD_API int fd_bias_grad(const void* dy, float* db, long npix, int C, void* stream);
/* backward of fd_final_conv_crop over the whole frame: dout fp32 NCHW (N,Cout,HW) -> dx bf16 (N,HW,64); dw[Cout][64], db[Cout] += */
FD_API int fd_final_conv_bwd(const void* x, const float* w, const float* dout, void* dx, float* dw, float* db,
                      int N, int HW, int Cin, int Cout, void* stream);
/* dgrad weights from the forward's packed weights: wd[ci][(T-1-tap)*Cout + co] = wpacked[co][tap*Cin + ci]
 * (for kind 1 use T = 1, Cin = 4*C).  The data gradient is then fd_conv_igemm(_ex) on dy with wd. */
FD_API int fd_prep_weight_dgrad(const void* wpacked, void* wd, int Cout, int Cin, int taps, void* stream);
/* Batched forms: ONE launch for all the layers of a model (a training step re-packs ~80 weight tensors; 230 launches of
 * 5-13 us each otherwise).  `table` is a DEVICE array of n_layers records of 8 x int64:
 *   fd_prep_weight_batch        {w (float*), packed (bf16*), 0, Cout, Cin, KH, KW, kind | standardize << 8}
 *   fd_prep_weight_dgrad_batch  {wpacked, wd, 0, Cout, Cin, taps, 0, 0}
 *   fd_prep_weight_bwd_batch    {g, w, dw, Cout, Cin, KH, KW, kind | standardize << 8}
 * with the per-layer arguments of the single-layer functions; `blk_start` is a DEVICE int32[n_layers + 1] array of prefix sums
 * of the layers' block counts (Cout blocks per layer; ceil(Cin/32) * ceil(Cout/32) * taps for the dgrad form) and
 * total_blocks = blk_start[n_layers]. */
FD_API int fd_prep_weight_batch(const long long* table, const int* blk_start, int n_layers, int total_blocks, float eps,
                                void* stream);
FD_API int fd_prep_weight_dgrad_batch(const long long* table, const int* blk_start, int n_layers, int total_blocks,
                                      void* stream);
FD_API int fd_prep_weight_bwd_batch(const long long* table, const int* blk_start, int n_layers, int total_blocks, float eps,
                                    void* stream);
/* fd_conv_wgrad result (fp32 packed [Cout][K]) -> parameter gradient dw (+=, torch layout), through the
 * weight-standardisation backward when standardize != 0 (arguments as fd_prep_weight). */
FD_API int fd_prep_weight_bwd(const float* g, const float* w, float* dw, int Cout, int Cin, int KH, int KW, int kind,
                       int standardize, float eps, void* stream);
/* small fp32 dense layers of the time path (:319-324, :193-196); act 0 none, 1 SiLU, 2 GELU(erf):
 *   bwd_w: dW[J][K] += sum_b dY[b][j] act(X[b][k]), db[J] += sum_b dY[b][j] (db may be NULL)
 *   bwd_x: dX[b][k] = act'(A[b][k]) * sum_j dY[b][j] W[j][k] */
FD_API int fd_linear_bwd_w(const float* dY, long dy_stride, const float* X, long x_stride, float* dW, float* db,
                    int B, int J, int K, int act, void* stream);
FD_API int fd_linear_bwd_x(const float* dY, long dy_stride, const float* W, const float* A, long a_stride, float* dX,
                    long dx_stride, int B, int J, int K, int act, void* stream);
/* fd_time_embed that also saves its intermediates for the backward: pe fp32 (B,dim), pre fp32 (B,time_dim) = the
 * pre-GELU activations (either may be NULL) */
FD_API int fd_time_embed_save(const int64_t* t, const float* w1, const float* b1, const float* w2, const float* b2,
                       float* temb, float* pe, float* pre, int B, int dim, int time_dim, void* stream);

/* optimiser (flow_diffuser.py:129-134 torch.optim.Adam with L2-in-gradient weight decay; Lightning's
 * gradient_clip_val, exp_base.py:192,205): out[0] += sum of squares of g; then one fused update over flat buffers:
 *   g' = g * grad_scale * min(1, max_norm / (grad_scale * sqrt(*grad_sumsq) + 1e-6)) + wd * p ;  Adam(m, v, step) */
FD_API int fd_sumsq(const float* g, long n, float* out, void* stream);
FD_API int fd_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long n, float lr,
                 float beta1, float beta2, float eps, float weight_decay, int step, const float* grad_sumsq,
                 float max_norm, float grad_scale, void* stream);

/* ---- training augmentation on the GPU: augmentation.py:6-76 (torchvision ColorJitter / Grayscale / GaussianBlur(3) /
 *      flips / RandomResizedCrop, applied item by item in the reference).  fp32 NCHW images in [0,1].
 * frame tables have 2B rows (item*2 + {0: img, 1: tgt}):
 *   frame_ints  [8] = {jitter_on, op0..op3 (0 brightness, 1 contrast, 2 saturation, 3 hue, applied in this order),
 *                      gray_on, blur_on, -};   frame_floats [8] = {brightness, contrast, saturation, hue, k_edge, k_center, -, -}
 * item_ints [8] = {hflip, vflip, crop_on, top, left, crop_h, crop_w, -}.
 * photometric: frames_out (B,2,3,H,W) = Grayscale?(ColorJitter?(frame)); means: 2B floats of scratch.
 * blur3: blurred[f] = GaussianBlur3(frames[f]) for the frames with blur_on (others untouched).
 * geometric: reads frame f from `blurred` if blur_on else from `frames`; hflip negates the LAST flow channel, vflip the
 *   second-last; the crop scales the flow by (crop_h/H, crop_w/W) and resamples all 8 channels bilinearly
 *   (align_corners = False, no antialias) back to (H, W). */
FD_API int fd_aug_photometric(const float* img, const float* tgt, const int* frame_ints, const float* frame_floats,
                       float* means, float* frames_out, int B, int HW, void* stream);
FD_API int fd_aug_blur3(const float* frames, const int* frame_ints, const float* frame_floats, float* blurred,
                 int B, int H, int W, void* stream);
FD_API int fd_aug_geometric(const float* frames, const float* blurred, const float* flow, const int* frame_ints,
                     const int* item_ints, float* out_img, float* out_tgt, float* out_flow, int B, int H, int W,
                     void* stream);

/* ---- FlowLearner objective: flow_learner.py:133-222 -------------------------------------------------
 * soft_charb: one (level, offset) term.  S, T (B, C+1, HW) are the RAW soft splats (softsplat_new.py:306-307 before the
 * normalisation): warped = S[:C] / (S[C] + 1e-7), NaN where S[C] is not > 0 (fill_holes_nan, warp.py:273-276),
 * target = T[:C] / (T[C] + 1e-7); sums = {sum of sqrt((target - warped)^2 + 1e-6) over non-NaN pairs, count, mean}
 * (nan_charbonnier, warp.py:281-287).  bwd: gS = d(upstream[0] * mean)/dS.  partials: fd_loss_workspace_floats(B*HW). */
FD_API size_t fd_loss_workspace_floats(long items);
FD_API int fd_soft_charb_fwd(const float* S, const float* T, float* sums, float* partials, int B, int C, int HW, void* stream);
FD_API int fd_soft_charb_bwd(const float* S, const float* T, const float* sums, const float* upstream, float* gS,
                      int B, int C, int HW, void* stream);
/* All scale^2 offsets of one pyramid level at once (the loop of flow_learner.py:184-196): offset index k = a*scale + b
 * <-> offset = [a, b].  The stacked splats and their gradients are PIXEL-INTERLEAVED, (K, B, H/scale, W/scale, 4) with the four
 * channels (r, g, b, weight) of a cell adjacent (16-byte aligned), so that a bilinear tap is one 128-bit reduction / load: the
 * splat input has C = 4 channels, soft_charb_multi takes C = 3 (+ the weight).  splat_*_multi: the per-offset arithmetic of
 * fd_splat_fwd / _ingrad / _flowgrad, the two gradient kernels summing over k.
 * soft_charb_multi: sums [K][3], out[0] = mean_k mean_k; bwd: gS = d(upstream[0] * out[0])/dS. */
FD_API int fd_splat_fwd_multi(const float* in, const float* flow, float* out, int B, int C, int H, int W, int scale, void* stream);
FD_API int fd_splat_ingrad_multi(const float* flow, const float* gout, float* gin, int B, int C, int H, int W, int scale,
                          void* stream);
FD_API int fd_splat_flowgrad_multi(const float* in, const float* flow, const float* gout, float* gflow, int B, int C,
                            int H, int W, int scale, void* stream);
FD_API size_t fd_soft_charb_multi_workspace_floats(int B, int HW, int K);
FD_API int fd_soft_charb_multi_fwd(const float* S, const float* T, float* sums, float* out, float* partials, int B, int C,
                            int HW, int K, void* stream);
FD_API int fd_soft_charb_multi_bwd(const float* S, const float* T, const float* sums, const float* upstream, float* gS,
                            int B, int C, int HW, int K, void* stream);
/* edgeaware_smoothness1 (warp.py:289-303): out[0] = loss; bwd: gflow = upstream[0] * dloss/dflow (image has no gradient) */
FD_API int fd_edge_smooth_fwd(const float* img, const float* flow, float* out, float* partials, int B, int Ci, int Cf,
                       int H, int W, void* stream);
FD_API int fd_edge_smooth_bwd(const float* img, const float* flow, const float* upstream, float* gflow, int B, int Ci,
                       int Cf, int H, int W, void* stream);

/* debug / test helpers: fp32 NCHW <-> bf16 NHWC */
FD_API int fd_nchw_to_nhwc_bf16(const float* x, void* out, int N, int C, int HW, void* stream);
FD_API int fd_nhwc_bf16_to_nchw(const void* x, float* out, int N, int C, int HW, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FLOWDIFF_H_ */
