/*
 * gap_b200.h — C ABI of the B200-native conv hot path for GAN-AUG-PFA (Pix2Pix U-Net generator,
 * PatchGAN discriminator, Siamese U-Net reuse).
 *
 * The reference (Affi-Amine/GAN-AUG-PFA) is pure Python and defines no FFI of its own: its hot path
 * is whatever torch dispatches for the nn.* modules built in models.py.  Every entry point below
 * therefore cites the reference call site whose torch library kernel it replaces (file:line into
 * the reference tree).  INTEGRATION.md shows the ctypes stub a maintainer adds to models.py.
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless the name says host; the caller owns every buffer
 *     (including workspaces); the library never allocates or frees device memory;
 *   - activations are NHWC bf16 (pixel stride `ld` in elements, so a tensor may live in a channel
 *     slot of a wider concat buffer); weights are packed bf16 K-major matrices (gap_pack_weights);
 *     gradients of weights, BatchNorm statistics, losses and optimizer state are fp32/fp64;
 *   - every function enqueues work on `stream` (a cudaStream_t passed as void*) and returns
 *     without synchronising;
 *   - return value: 0 = ok, negative = gap_status (bad argument / unsupported configuration),
 *     positive = cudaError_t.  gap_last_error_string() describes the last failure of the calling
 *     thread.  There is no CPU fallback and no cuDNN/cuBLAS fallback.
 */
#ifndef GAP_B200_H
#define GAP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum gap_status {
  GAP_OK = 0,
  GAP_ERR_BAD_ARG = -1,
  GAP_ERR_UNSUPPORTED = -2,
  GAP_ERR_ALIGNMENT = -3,
  GAP_ERR_DRIVER = -4
};

enum gap_act {
  GAP_ACT_NONE = 0,
  GAP_ACT_LRELU = 1, /* LeakyReLU(0.2)   models.py:178,223,232,240 */
  GAP_ACT_RELU = 2,  /* ReLU             models.py:180,11,14,37   */
  GAP_ACT_TANH = 3,  /* Tanh             models.py:186             */
  GAP_ACT_SIGMOID = 4 /* Sigmoid          models.py:34              */
};

const char* gap_last_error_string(void);
int gap_version(void);
/* Number of SMs the persistent kernels size their grids for (148 on B200). */
int gap_sm_count(void);

/* ------------------------------------------------------------------------------------------------
 * Implicit-GEMM convolution engine (tcgen05 / TMEM / TMA).
 *
 * One call computes, for every phase p = (ph, pw), every image n and every grid point (gy, gx):
 *
 *   acc[co] = sum over taps (th, tw), sources s, channels c of
 *             src_s[n, gy*in_stride + in_off_h[ph] + th, gx*in_stride + in_off_w[pw] + tw, c]
 *             * wpk[p][co][(th*taps_w + tw)*ctot + chan_off(s) + c]
 *   v = acc[co] + bias[co];  stats[co] += v, stats[n_out+co] += v*v   (fp64, optional)
 *   out [n, gy*out_stride + ph, gx*out_stride + pw, co] = act (v)   (bf16)
 *   out2[same pixel, co]                                 = act2(v)   (bf16, optional)
 *
 * Out-of-range source coordinates read as zero (that is the convolution padding).  With the right
 * taps / offsets / packed weights this one contraction is Conv2d forward (models.py:177,223,230,
 * 238,243,9,12,22,27,32,90), Conv2d dgrad, ConvTranspose2d forward (models.py:184,189,194) and
 * ConvTranspose2d dgrad; the named wrappers further down fill this struct.
 * ---------------------------------------------------------------------------------------------- */
typedef struct gap_conv_gemm_args {
  /* A operand: one or two NHWC bf16 sources concatenated along channels (torch.cat, models.py:208) */
  const void* src[2];
  int src_c[2];      /* channels taken from each source; multiple of 64; src_c[1] = 0 if unused */
  int64_t src_ld[2]; /* pixel stride in elements (>= src_c, multiple of 8) */
  int n, ih, iw;     /* source images / rows / cols */
  /* M iteration space */
  int gh, gw;    /* grid rows / cols per image per phase */
  int n_phase;   /* 1, or 4 for the stride-2 transposed geometry */
  int taps_h, taps_w;
  int in_stride;
  int in_off_h[2], in_off_w[2];
  int out_stride;
  /* B operand: packed weights, bf16, [n_phase][w_rows][taps_h*taps_w*ctot] */
  const void* wpk;
  int w_rows; /* rows present in wpk per phase (>= n_out) */
  /* epilogue */
  int n_out; /* valid output channels */
  int oh, ow; /* full output rows / cols */
  void* out;
  int64_t out_ld;
  int act;
  void* out2; /* may be NULL */
  int64_t out2_ld;
  int act2;
  const float* bias; /* may be NULL */
  double* stats;     /* may be NULL; [2*n_out] */
  int out_f32;       /* 1: `out` is fp32 instead of bf16 (out2 must be NULL) */
  /* Backward-fused epilogue (bwd_y != NULL; dgrad calls): the GEMM result g = dL/d(activation output) is turned
   * into the gradient at the BatchNorm output before it is stored, for output channels c >= bwd_c0:
   *     mask = (bwd_y[pix][c'] * bwd_scale[c'] + bwd_shift[c'] > 0),  c' = c - bwd_c0   (scale NULL: mask = bwd_y > 0)
   *     d    = mask ? g + bwd_g2[pix][c'] : bwd_slope * g                       (LeakyReLU / ReLU backward, with the
   *            U-Net skip gradient g2 that only flows through the ReLU'd copy; models.py:178,180,208)
   *     stats[c'] += d,  stats[(n_out - bwd_c0) + c'] += d * bwd_y[pix][c']     (BatchNorm backward sums, fp64)
   *     out[pix][c] = d
   * Channels below bwd_c0 are stored unchanged.  Needs act = NONE, no bias / out2, a 32-byte aligned output. */
  const void* bwd_y;
  int64_t bwd_y_ld;
  const float* bwd_scale;
  const float* bwd_shift;
  const void* bwd_g2; /* may be NULL */
  int64_t bwd_g2_ld;
  float bwd_slope;
  int bwd_c0;
  /* Optional per-channel multiplier applied to the accumulator before the bias: v = acc*scale[co] + bias[co].
   * Eval-mode BatchNorm (generate_synthetic_data.py:55, train.py:151, evaluate.py:146) folds into the conv this way
   * (scale = gamma/sqrt(running_var+eps), bias = beta - running_mean*scale), so no normalisation pass runs. */
  const float* scale;
  /* 1: out[pix][co] = act(v) + out[pix][co] instead of a plain store -- a gradient buffer that collects several
   * contributions (autograd's accumulation for a tensor with more than one consumer: the Siamese skips, gate inputs
   * and concatenated decoder inputs, models.py:104-135).  Excludes out2, stats and the backward-fused epilogue. */
  int accumulate;
} gap_conv_gemm_args;

int gap_conv_gemm(const gap_conv_gemm_args* args, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Weight-gradient contraction (tcgen05, MN-major operands, split-K with fp32 red.add):
 *
 *   out[m*ld_m + tap*ld_tap + c] += sum over images and grid points (gy, gx) of
 *        mop[img, gy, gx, m] * nop[img, gy*stride + off_h + th, gx*stride + off_w + tw, c]
 *
 * Conv2d wgrad (autograd of models.py:177,223,230,238,243,9,12,...): mop = dY, nop = X,
 * out = dW viewed as [Cout][kh*kw][Cin].  ConvTranspose2d wgrad (models.py:184,189,194):
 * mop = X, nop = dY, out = dW viewed as [Cin][kh*kw][Cout].  The caller zeroes `out` (that is
 * optimizer.zero_grad(), train_gan.py:55,64); concatenated inputs are handled by one call per
 * source with `out` offset to the source's channel range.
 * ---------------------------------------------------------------------------------------------- */
typedef struct gap_wgrad_args {
  const void* mop; /* NHWC bf16 [n, gh, gw, m_c] */
  int m_c;
  int m_rows; /* rows of `out` that exist (<= m_c); rows beyond are not written */
  int64_t m_ld;
  const void* nop; /* NHWC bf16 [n, nh, nw, n_c] */
  int n_c;
  int64_t n_ld;
  int n, gh, gw, nh, nw;
  int taps_h, taps_w, stride, off_h, off_w;
  float* out;
  int64_t ld_m, ld_tap;
} gap_wgrad_args;

int gap_conv_wgrad(const gap_wgrad_args* args, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Model-boundary layout conversion (replaces the implicit NCHW fp32 contract of models.py:163,246)
 * ---------------------------------------------------------------------------------------------- */
int gap_nchw_f32_to_nhwc_bf16(const float* x, void* out, int n, int c, int h, int w, int64_t out_ld,
                              void* stream);
/* writes channels [c_off, c_off+c) of an NCHW fp32 tensor that has c_total channels */
int gap_nhwc_to_nchw_f32(const void* x, int x_is_f32, float* out, int n, int c, int h, int w, int64_t x_ld,
                         int c_total, int c_off, void* stream);
/* Tanh backward at the model boundary (models.py:186): dpre = gout * (1 - y^2), NCHW fp32 -> NHWC bf16 */
int gap_tanh_bwd(const float* gout_nchw, const float* y_nhwc, int64_t ld_y, void* dpre, int64_t ld_p, int n, int c,
                 int h, int w, void* stream);

/* L1Loss(fake, real) * lambda (train_gan.py:43,68) fused with the Tanh backward:
 * loss_acc += sum|fake-real|; dpre = (dfake_d + l1_scale*sign(fake-real)) * (1 - fake^2). */
int gap_gen_out_bwd(const float* fake, int64_t ld_f, const float* real_nchw, int64_t hw, const float* dfake_d,
                    int64_t ld_d, float l1_scale, void* dpre, int64_t ld_p, int64_t pixels, int c,
                    double* loss_acc, void* stream);
/* Same with real_B as the raw uint8 HWC image [pixel][c], normalised in the kernel exactly like the dataset does
 * ((x/255)*2-1 in fp32, dataset.py:28-29,155-159): the device-side input pipeline of the training loop. */
int gap_gen_out_bwd_u8(const float* fake, int64_t ld_f, const uint8_t* real_hwc, int64_t hw, const float* dfake_d,
                       int64_t ld_d, float l1_scale, void* dpre, int64_t ld_p, int64_t pixels, int c,
                       double* loss_acc, void* stream);

/* BCEWithLogitsLoss against ones / zeros (train_gan.py:42,58,60,67): loss_acc += sum l(x, t);
 * dlogits[i*ld_d] = grad_scale * (sigmoid(x) - t) in bf16 (dlogits may be NULL). */
int gap_bce_logits_const(const float* logits, int64_t count, float target, float grad_scale, void* dlogits,
                         int64_t ld_d, double* loss_acc, void* stream);

/* Same loss with an fp32 gradient and the bias gradient of the conv that produced the logits
 * (dbias += sum dlogits; dlogits / dbias may be NULL). */
int gap_bce_logits_const_f32(const float* logits, int64_t count, float target, float grad_scale, float* dlogits,
                             double* loss_acc, float* dbias, void* stream);
/* out[0] += sum x[i] (fp32) */
int gap_sum_f32(const float* x, int64_t count, float* out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Conv2d(C -> 1, k4, s1, pad) + bias: the PatchGAN's last layer (models.py:243) as direct warp-MMA
 * kernels that read every activation once (the layer is HBM-bound: 8192 MACs per 1 KiB pixel).
 *   fwd:   z_ws[pix][16] = x[pix][:] . w[tap][:]  then  logits[n][oy][ox] = bias + sum_taps z[...]
 *   dgrad: gx[pix][c]  = sum_taps dlogits[n][y-kh+pad][x-kw+pad] * w[tap][c]            (bf16 out)
 *   wgrad: dw[tap][c] += sum_pix  dlogits[n][y-kh+pad][x-kw+pad] * x[pix][c]            (fp32)
 * x / gx: NHWC bf16 (pixel stride ld, multiple of 8; 16-byte aligned); w: bf16 [16][c] ([kh][kw][c], the packed
 * forward operand; 16-byte aligned); logits / dlogits: fp32 [n][oh][ow]; z_ws: fp32 workspace [n*ih*iw*16].
 * c % 64 == 0.  Up to c = 512 (and 2^31 pixels, 0 <= in_slope <= 1) forward and wgrad run as streaming kernels (per-warp
 * cp.async rings, one CTA per SM); other shapes take the general kernels -- same results, same contract.
 * in_scale / in_shift (fp32 [c], both or neither; c <= 512) + in_slope: x is then the RAW conv output of the layer below
 * and the kernels form LeakyReLU_slope(x*in_scale + in_shift) while staging it -- the BatchNorm apply + activation of
 * models.py:239-240 fused into its consumer, so the activated tensor never makes an HBM round trip.
 * ---------------------------------------------------------------------------------------------- */
int gap_cout1_conv_fwd(const void* x, int64_t ld_x, int n, int ih, int iw, int c, const void* w, const float* bias,
                       int ksize, int pad, float* z_ws, float* logits, const float* in_scale, const float* in_shift,
                       float in_slope, void* stream);
int gap_cout1_conv_dgrad(const float* dlogits, int n, int oh, int ow, const void* w, int ksize, int pad, int c, void* gx,
                         int64_t ld_gx, int ih, int iw, void* stream);
/* The same dgrad with the activation backward of the layer below and its BatchNorm-backward sums fused into the
 * copy-out: gx = (y*scale+shift > 0) ? g : slope*g;  sums[0..c) += sum gx, sums[c..2c) += sum gx*y (fp64, of the stored
 * bf16 values) -- the contract of gap_conv_gemm's bwd_* epilogue, finished by gap_bn_bwd_finalize + gap_bn_bwd_apply. */
int gap_cout1_conv_dgrad_bwd(const float* dlogits, int n, int oh, int ow, const void* w, int ksize, int pad, int c, void* gx,
                             int64_t ld_gx, int ih, int iw, const void* y, int64_t ld_y, const float* scale,
                             const float* shift, float slope, double* sums, void* stream);
int gap_cout1_conv_wgrad(const float* dlogits, int n, int oh, int ow, const void* x, int64_t ld_x, int ih, int iw, int c,
                         int ksize, int pad, float* dw, const float* in_scale, const float* in_shift, float in_slope,
                         void* stream);

/* ------------------------------------------------------------------------------------------------
 * Thin-input Conv2d(k4, s2, p1) as one fused warp-MMA kernel (no im2col buffer): the generator's first
 * conv (models.py:177, outermost block), the discriminator's first conv over cat(A, B) (models.py:223,
 * train_gan.py:57,59,66) and the input gradient of the generator's last ConvTranspose2d (models.py:184).
 *   out1[pix][co] = act1(bias[co] + sum_{tap,slot} in[2*pix+tap-1][slot] * wpk[co][tap*CT + slot]),  out2 likewise
 * src0 / src1: NHWC bf16 with 4 channel slots used per pixel (1..4 channels, the rest zero slots; ld % 4 == 0);
 * src1 == NULL -> CT = 4, else CT = 8 with src1's slots at 4..7.  wpk: bf16 [cw][16*CT]; cw = 64 or 128;
 * activations: none / LeakyReLU / ReLU.  out2 may be NULL.
 * The kernel sums over every slot, so it serves any channel count of up to 4 per source provided BOTH the packed
 * weights of unused slots AND the unused activation slots are zero (0 * NaN = NaN): every producer of a 4-slot image
 * tensor (the converters below, gap_nchw_f32_to_nhwc_bf16 on zero-initialised buffers, gap_thin_convT_fwd[_c],
 * gap_gen_out_bwd[_u8]) leaves the slots past its channel count zero.
 * ---------------------------------------------------------------------------------------------- */
int gap_thin_conv_fwd(const void* src0, int64_t ld0, const void* src1, int64_t ld1, int n, int h, int w, const void* wpk,
                      const float* bias, int cw, void* out1, int64_t ldo1, int act1, void* out2, int64_t ldo2, int act2,
                      void* stream);

/* Weight (and bias) gradient of the same thin layers, accumulated straight into the fp32 master layout
 * [cw][(kh*4+kw)*c + ch] (row stride ld_m, c = 3 or 6):
 *   dw[cw][tap][ch] += sum_pix wide[pix][cw] * thin[2*pix+tap-1][ch];   dbias[cw] += sum_pix wide[pix][cw]
 * wide: NHWC bf16 [n, h/2, w/2, cw] (dY of the first convs; X of the generator's last ConvTranspose2d, whose
 * weight (Cin, 3, 4, 4) has this same form with thin = dY); thin sources as in gap_thin_conv_fwd.
 * dbias may be NULL. */
int gap_thin_conv_wgrad(const void* wide, int64_t ld_w, const void* src0, int64_t ld0, const void* src1, int64_t ld1,
                        int n, int h, int w, int cw, float* dw, int64_t ld_m, float* dbias, void* stream);
/* The same with c0 / c1 channels in source 0 / source 1 (c0 = 1..4; c1 = 1..4 with src1, 0 without): slots past a
 * source's channel count are dropped and slot s of source 1 is master channel c0 + s, in the layout
 * [cw][(kh*4+kw)*(c0+c1) + ch].  gap_thin_conv_wgrad is c0 = 3, c1 = src1 ? 3 : 0. */
int gap_thin_conv_wgrad_c(const void* wide, int64_t ld_w, const void* src0, int64_t ld0, int c0, const void* src1,
                          int64_t ld1, int c1, int n, int h, int w, int cw, float* dw, int64_t ld_m, float* dbias,
                          void* stream);

/* Thin-output ConvTranspose2d(cw -> 3, k4, s2, p1) (+bias, Tanh): the generator's last layer
 * (models.py:184,186), and — with the first conv's weights — the input gradient of the discriminator's first
 * conv (models.py:223).  wide: NHWC bf16 [n, ih, iw, cw]; wcol: bf16 [48 = (kh*4+kw)*3 + co][cw]; outputs
 * [n, 2ih, 2iw, 4 slots] in bf16 and / or fp32 (slot 3 is written as zero); act = GAP_ACT_NONE or GAP_ACT_TANH. */
int gap_thin_convT_fwd(const void* wide, int64_t ld_w, int n, int ih, int iw, int cw, const void* wcol, const float* bias,
                       int act, void* out_bf16, int64_t ld_bf, float* out_f32, int64_t ld_f, uint8_t* out_u8, void* stream);
/* ConvTranspose2d(cw -> co, k4, s2, p1) for co = 1..4: wcol bf16 [16*co = (kh*4+kw)*co + c][cw], bias [co] (may be
 * NULL), outputs [n, 2ih, 2iw, 4 slots] with slots >= co written as zero, out_u8 [n][2ih][2iw][co].
 * gap_thin_convT_fwd is co = 3. */
int gap_thin_convT_fwd_c(const void* wide, int64_t ld_w, int n, int ih, int iw, int cw, int co, const void* wcol,
                         const float* bias, int act, void* out_bf16, int64_t ld_bf, float* out_f32, int64_t ld_f,
                         uint8_t* out_u8, void* stream);
/* SURVEY.md §8(f) ranks 1-2 (the I/O either side of the generator): out_u8 above, if not NULL, receives the image
 * generate_synthetic_data.py:69-88 writes to PNG — uint8 [n][2ih][2iw][3] = byte((v*0.5 + 0.5) * 255) — straight from
 * the last layer's epilogue; gap_u8_hwc_to_nhwc_bf16 is dataset.py's ToTensor + Normalize(0.5, 0.5) (dataset.py:155-159)
 * on the device: uint8 HWC [pixels][3] -> NHWC bf16 with 4 channel slots, x*(2/255) - 1. */
int gap_u8_hwc_to_nhwc_bf16(const uint8_t* x, void* out, int64_t out_ld, int64_t pixels, void* stream);
/* The same for c = 1..4 channels per pixel (uint8 HWC [pixels][c]); slots >= c are written as zero. */
int gap_u8_hwc_to_nhwc_bf16_c(const uint8_t* x, int c, void* out, int64_t out_ld, int64_t pixels, void* stream);
/* The same with dataset.py's JointResize in front (dataset.py:136-153; ToTensor -> resize(BILINEAR) -> Normalize): uint8
 * HWC [n][ih][iw][3] -> antialiased bilinear resize (torchvision's tensor path = F.interpolate(mode="bilinear",
 * align_corners=False, antialias=True)) -> x*2 - 1 -> NHWC bf16 [n][oh][ow][4 slots] and / or (out_nchw_f32) the fp32
 * [n][3][oh][ow] tensor the reference's DataLoader yields (either output may be NULL).  gap_resize_nearest_i64 is the
 * label half of JointResize (InterpolationMode.NEAREST on the int64 {0,1} map, dataset.py:143-146). */
int gap_resize_u8_to_nhwc_bf16(const uint8_t* x, int n, int ih, int iw, int oh, int ow, void* out, int64_t out_ld,
                               float* out_nchw_f32, void* stream);
/* The same for c = 1..4 channels per pixel (uint8 HWC [n][ih][iw][c]; out_nchw_f32 [n][c][oh][ow]); bf16 slots >= c are
 * written as zero.  gap_resize_u8_to_nhwc_bf16 is c = 3. */
int gap_resize_u8_to_nhwc_bf16_c(const uint8_t* x, int c, int n, int ih, int iw, int oh, int ow, void* out,
                                 int64_t out_ld, float* out_nchw_f32, void* stream);
int gap_resize_nearest_i64(const int64_t* x, int n, int ih, int iw, int oh, int ow, int64_t* out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Siamese U-Net extras (models.py:47-145, train.py:34-128); NHWC bf16 activations, 8-channel vectors
 * (channels and pixel strides multiples of 8); single-channel maps (psi, final logits) are fp32 [pixels].
 * ---------------------------------------------------------------------------------------------- */
/* im2col of Conv2d(3 -> C, k3, s1, p1) (models.py:9 through :54): col[pix][(kh*3+kw)*3 + c], padded to 64 */
int gap_im2col_k3s1p1_c3(const void* x, int64_t ld, void* col, int n, int h, int w, void* stream);
/* The same for c = 1..4 input channels: col[pix][(kh*3+kw)*c + ch], 9*c values padded to 64 (gap_im2col_k3s1p1_c3 is
 * c = 3) */
int gap_im2col_k3s1p1_c(const void* x, int64_t ld, int c, void* col, int n, int h, int w, void* stream);
/* nn.MaxPool2d(2) (models.py:58).  Backward sends the gradient to the first maximum in scan order. */
int gap_maxpool2x2_fwd(const void* x, int64_t ldx, void* out, int64_t ldo, int n, int h, int w, int c, void* stream);
int gap_maxpool2x2_bwd(const void* x, int64_t ldx, const void* gout, int64_t ldg, void* gin, int64_t ldi, int n, int h,
                       int w, int c, int accumulate, void* stream);
/* nn.Upsample(scale_factor=2, mode='bilinear', align_corners=True) (models.py:64); h, w = INPUT size */
int gap_upsample_bilinear2x_fwd(const void* x, int64_t ldx, void* out, int64_t ldo, int n, int h, int w, int c,
                                void* stream);
int gap_upsample_bilinear2x_bwd(const void* gout, int64_t ldg, void* gin, int64_t ldi, int n, int h, int w, int c,
                                int accumulate, void* stream);
/* nn.Dropout(p) of UnetSkipConnectionBlock(use_dropout=True) (models.py:197-198), in place: x = keep ? x/(1-p) : 0 with
 * keep = hash(seed, offset + element index) — forward and backward call it with the same (seed, offset), on the
 * activation and on its gradient.  Not bit-compatible with torch's Philox stream (statistical parity only). */
int gap_dropout_bf16(void* x, int64_t ld, int64_t pixels, int c, float p_drop, uint64_t seed, uint64_t offset, void* stream);
/* AttentionGate (models.py:18-44): s = ReLU(BN(yg) + BN(yx)) (dense [pixels][c]); d = (s > 0) ? gs : 0;
 * psi = Sigmoid(BN(ypsi)), out = x * psi;  gate backward: gx (+)= gout * psi, dz = (sum_c gout * x) * psi * (1 - psi) */
int gap_att_add_relu_fwd(const void* yg, const float* scale_g, const float* shift_g, const void* yx, const float* scale_x,
                         const float* shift_x, void* s, int64_t pixels, int c, void* stream);
int gap_relu_bwd(const void* s, const void* gs, void* d, int64_t count, void* stream);
/* LeakyReLU backward on NHWC bf16 channel slices: d (+)= (y > 0) ? g : slope*g.  Used by the stand-alone
 * UnetSkipConnectionBlock path (models.py:178,208: the block's skip output is LeakyReLU(x) itself). */
int gap_lrelu_bwd_bf16(const void* y, int64_t ldy, const void* g, int64_t ldg, float slope, void* d, int64_t ldd,
                       int64_t pixels, int c, int accumulate, void* stream);
int gap_att_gate_fwd(const float* ypsi, const float* scale, const float* shift, float* psi, const void* x, int64_t ldx,
                     void* out, int64_t ldo, int64_t pixels, int c, void* stream);
int gap_att_gate_bwd(const void* gout, int64_t ldg, const void* x, int64_t ldx, const float* psi, void* gx, int64_t ldgx,
                     int accumulate, float* dz, int64_t pixels, int c, void* stream);
/* single-channel BatchNorm2d(1) (models.py:33): stats[0] += sum y, stats[1] += sum y^2 (then gap_bn_finalize, c = 1);
 * backward: sums[0..1] accumulate sum dz, sum dz*xhat; dy = scale * (dz - sums[0]/n - xhat * sums[1]/n) */
int gap_vec_stats(const float* y, int64_t n, double* stats, void* stream);
int gap_vec_bn_bwd(const float* y, const float* dz, int64_t n, const float* scale, const float* mean, const float* invstd,
                   double* sums, float* dy, void* stream);
/* Conv2d(C -> 1, k1) + bias (models.py:32, :90): out[pix] = bias + x[pix] . w;  gx[pix][c] = dl[pix] * w[c];
 * dw[c] += sum_pix dl[pix] * x[pix][c], db += sum dl.  w is the fp32 master (rounded to bf16 in the kernel). */
int gap_conv1x1_cout1_fwd(const void* x, int64_t ldx, const float* w, const float* bias, float* out, int64_t pixels, int c,
                          void* stream);
int gap_conv1x1_cout1_dgrad(const float* dl, const float* w, void* gx, int64_t ldg, int64_t pixels, int c, void* stream);
int gap_conv1x1_cout1_wgrad(const float* dl, const void* x, int64_t ldx, int64_t pixels, int c, float* dw, float* db,
                            void* stream);
/* Segmentation losses on fp32 logits vs int64 {0,1} labels (train.py:34-128):
 *   mode 0 CombinedLoss  = w_point * BCEWithLogits(pos_weight) + w_dice * Dice(smooth)      (train.py:82-105)
 *   mode 1 FocalDiceLoss = w_point * Focal(gamma, focal_alpha) + w_dice * Dice(smooth)     (train.py:108-128)
 * loss[0] is written; grad (may be NULL) = grad_scale * d(loss)/d(logit); sums4 is a 4-double workspace. */
int gap_seg_loss(const float* logits, const int64_t* labels, int64_t n, int mode, float w_point, float w_dice,
                 float pos_weight, float smooth, float gamma, float focal_alpha, double* sums4, float* grad,
                 float grad_scale, double* loss, void* stream);

/* Multi-class head of SiameseUNet(n_channels, n_classes), K = n_classes = 1..16 (seg_head.cu).
 * Layout: logits and their gradient are fp32 class planes [n][K][hw] (NCHW: what nn.CrossEntropyLoss and
 * torch.argmax(dim=1) take; for K = 1 the same memory as the [n][hw] map of the single-class path).  The head input
 * x is the NHWC bf16 output of dconv_last, [n*hw][64] with row stride ldx (a multiple of 8); w is the fp32 master
 * conv_last.weight [K][64] (rounded to bf16 in the kernels), bias [K].
 *   fwd:   out[n][c][p] = bias[c] + sum_ch w[c][ch] * x[pix][ch];  pred (optional, uint8 [n][hw]) = argmax over c
 *          (ties to the lowest index, NaN above everything, as torch.argmax)
 *   dgrad: gx[pix][ch] = sum_c dl[c][pix] * w[c][ch], bf16, written (not accumulated) into channels 0..63 of rows ldg apart
 *   wgrad: dw[c][ch] += sum_pix dl[c][pix] * x[pix][ch], db[c] += sum_pix dl[c][pix] (db optional) */
int gap_conv1x1_ck_fwd(const void* x, int64_t ldx, const float* w, const float* bias, int k, int n, int64_t hw,
                       float* out, uint8_t* pred, void* stream);
int gap_conv1x1_ck_dgrad(const float* dl, const float* w, int k, int n, int64_t hw, void* gx, int64_t ldg, void* stream);
int gap_conv1x1_ck_wgrad(const float* dl, const void* x, int64_t ldx, int k, int n, int64_t hw, float* dw, float* db,
                         void* stream);
/* nn.CrossEntropyLoss(weight=class_weight, ignore_index, reduction="mean") over the K planes against int64 labels
 * [n][hw]: loss[0] = sum w[y] * (logsumexp - x[y]) / sum w[y] over labels != ignore_index (NaN when there are none);
 * grad (may be NULL) = grad_scale * d(loss)/d(logits) in the plane layout.  class_weight fp32 [K] or NULL (all 1).
 * A label outside [0, K) that is not ignore_index contributes nothing and adds 1 to *bad_labels (never zeroed here).
 * sums2 is a 2-double workspace.  No host synchronisation. */
int gap_seg_ce_loss(const float* logits, const int64_t* labels, int k, int n, int64_t hw, const float* class_weight,
                    int64_t ignore_index, double* sums2, int64_t* bad_labels, float* grad, float grad_scale,
                    double* loss, void* stream);
/* Softmax point term + multi-class Dice over the K = 2..16 planes against int64 labels [n][hw], p = softmax(logits):
 *   loss[0] = w_point * Point + (1 - w_point) * Dice,  Dice = 1 - 1/(K-1) sum_{k=1..K-1} (2 I_k + s) / (P_k + T_k + s)
 * with I_k = sum p_k [y=k], P_k = sum p_k, T_k = sum [y=k] over the counted pixels of the whole batch (y != ignore_index,
 * 0 <= y < K; class 0 is not a Dice class) and s = smooth > 0.
 *   mode 0: Point = nn.CrossEntropyLoss(weight=class_weight, ignore_index) (weighted mean, normalised by sum w[y])
 *   mode 1: Point = sum a[y] (1 - p_y)^gamma (-log p_y) / (counted pixels), a = class_weight (NULL: all 1), gamma >= 0
 * grad (may be NULL) = grad_scale * d(loss)/d(logits), zero at pixels that are not counted.  An all-ignored batch gives a
 * NaN loss and a zero gradient.  A label outside [0, K) that is not ignore_index adds 1 to *bad_labels (never zeroed
 * here).  sums is a fp64 workspace of 3(K-1)+2 doubles.  0 <= w_point <= 1.  No host synchronisation. */
int gap_seg_softmax_dice(const float* logits, const int64_t* labels, int k, int n, int64_t hw, int mode, float w_point,
                         float gamma, float smooth, const float* class_weight, int64_t ignore_index, double* sums,
                         int64_t* bad_labels, float* grad, float grad_scale, double* loss, void* stream);
/* Per-sample K x K confusion matrix: counts[n][label][argmax_c logits] += 1 (int64, accumulated: the caller zeroes it
 * once); pixels whose label is ignore_index or outside [0, K) are skipped.  n < 65536. */
int gap_seg_confusion_ck(const float* logits, const int64_t* labels, int k, int n, int64_t hw, int64_t ignore_index,
                         int64_t* counts, void* stream);

/* Sliding-window inference over a whole scene (scene.cu, SiameseEngine.predict_scene).  Each axis of the tile grid is
 * (len, ext, step, n): the scene length, the tile extent (a multiple of 16), the step between tile origins and the tile
 * count; tile i of an axis starts at n == 1 ? 0 : min(i*step, len - ext) (n == 1 needs len <= ext and reads past len
 * clamp to the last row / column; n > 1 needs len > ext).  Tiles are numbered row-major, t = ty*nx + tx.  Blending
 * window w = g(ty) g(tx), g(t) = exp(-(t + 0.5 - ext/2)^2 / (2 (ext/8)^2)).
 * gather: tiles tile0 .. tile0+batch-1 of both scenes -> NHWC bf16 [batch][ey][ex][4 slots] (out1 / out2, dense);
 *   src_u8: uint8 HWC [h][w][c] normalised as gap_u8_hwc_to_nhwc_bf16_c, else fp32 CHW [c][h][w] rounded as
 *   gap_nchw_f32_to_nhwc_bf16; slots >= c and tiles >= ny*nx (padding of the last batch) are written as zero.
 *   out1 / out2 must be 8-byte aligned: each 4-slot pixel is one 8-byte store. */
int gap_scene_gather(const void* img1, const void* img2, int src_u8, int c, int h, int w, int ey, int ex, int sy, int sx,
                     int ny, int nx, int tile0, int batch, void* out1, void* out2, void* stream);
/* blend: logits fp32 [batch][k][ey][ex] (k = 1: sigmoid, else softmax over the k planes) of tiles tile0 .. -> for every
 * scene pixel, over the covering tiles of this batch in ascending index: acc[c][pixel] += w * p_c, wsum[pixel] += w
 * (fp32 [k][h][w] and [h][w]).  A pixel whose first covering tile of the grid is in this batch starts from zero, so the
 * accumulators need no clearing when the batches run in order.  No floating-point atomics: deterministic. */
int gap_scene_blend(const float* logits, int k, int h, int w, int ey, int ex, int sy, int sx, int ny, int nx, int tile0,
                    int batch, float* acc, float* wsum, void* stream);
/* finalize: p = acc / wsum over `pixels`; pred (uint8) = argmax_c p (ties to the lowest class) or, k = 1, p > 0.5;
 * write_probs: acc is overwritten with p.  labels (int64, optional, with counts): counts += k > 1 ? [label][pred] (k*k)
 * : [TP, FP, FN, TN] (label 1 positive, 0 negative); ignore_index and labels outside [0, k) ({0, 1} for k = 1) are not
 * counted.  The caller zeroes counts. */
int gap_scene_finalize(float* acc, const float* wsum, int k, int64_t pixels, uint8_t* pred, int write_probs,
                       const int64_t* labels, int64_t ignore_index, int64_t* counts, void* stream);
/* The generator's scene kernels (GeneratorEngine.translate_scene), on the same tile grid and window.
 * gather_one: tiles tile0 .. tile0+batch-1 of one scene -> NHWC bf16 [batch][ey][ex][4 slots] (out, dense, 8-byte
 *   aligned), with the values, zero slots and zero padding tiles of gap_scene_gather. */
int gap_scene_gather_one(const void* img, int src_u8, int c, int h, int w, int ey, int ex, int sy, int sx, int ny,
                         int nx, int tile0, int batch, void* out, void* stream);
/* blend_image: the generator's fp32 output of tiles tile0 .. , fake [batch][ey][ex][4 slots] (16-byte aligned) ->
 *   for every scene pixel, over the covering tiles of this batch in ascending index: acc[ch][pixel] += w * v_ch for
 *   ch < c, wsum[pixel] += w (fp32 [c][h][w] and [h][w]); c = 1..4.  Same start-from-zero rule as gap_scene_blend, no
 *   floating-point atomics.  ey + ex <= 12288 (the window table lives in shared memory). */
int gap_scene_blend_image(const float* fake, int c, int h, int w, int ey, int ex, int sy, int sx, int ny, int nx,
                          int tile0, int batch, float* acc, float* wsum, void* stream);
/* finalize_image: v = acc / wsum over `pixels`; image (uint8 [pixels][c]) = uint8(clamp((v*0.5 + 0.5)*255, 0, 255)),
 *   truncated; write_float: acc is overwritten with v.  c = 1..4. */
int gap_scene_finalize_image(float* acc, const float* wsum, int c, int64_t pixels, uint8_t* image, int write_float,
                             void* stream);

/* evaluate.py:34-64 calculate_metrics, device side: per-sample counts[n][4] += [TP, FP, FN, TN] of
 * (sigmoid(logits) > 0.5) against {0,1} labels (int64 when labels_are_i64, else fp32); logits are [n][hw] fp32.
 * The caller zeroes counts once and may accumulate several batches; the ratios are formed on the host. */
int gap_seg_confusion(const float* logits, const void* labels, int labels_are_i64, int n, int64_t hw, int64_t* counts,
                      void* stream);

/* nn.BatchNorm2d training bookkeeping (models.py:179,181,231,239): statistics -> scale/shift,
 * saved mean / inv-std, running stats (momentum, unbiased var, `repeat` identical updates),
 * num_batches_tracked += repeat.  Re-zeroes `stats`. */
int gap_bn_finalize(double* stats, int c, double count, const float* gamma, const float* beta, float eps,
                    float momentum, int repeat, float* running_mean, float* running_var, int64_t* nbt,
                    float* scale, float* shift, float* save_mean, float* save_invstd, void* stream);
/* eval-mode BatchNorm (generate_synthetic_data.py:55): scale/shift from the running statistics */
int gap_bn_eval_scale_shift(int c, const float* gamma, const float* beta, const float* running_mean,
                            const float* running_var, float eps, float* scale, float* shift, void* stream);
/* out1 = act1(y*scale+shift), out2 = act2(y*scale+shift) (optional): BatchNorm apply fused with
 * LeakyReLU / ReLU and the U-Net skip write into the concat buffer (models.py:178-181,208). */
int gap_bn_act(const void* y, int64_t ld_y, const float* scale, const float* shift, int64_t pixels, int c,
               void* out1, int64_t ld1, int act1, void* out2, int64_t ld2, int act2, void* stream);
/* BatchNorm + activation backward, pass 1 (per-channel sums) and pass 2 (apply); see elementwise.cu.
 * scale == NULL in gap_bn_bwd_apply selects the activation-only mode. */
int gap_bn_bwd_reduce(const void* y, int64_t ld_y, const void* g1, int64_t ld_g1, const void* g2, int64_t ld_g2,
                      float slope, const float* scale, const float* shift, const float* mean,
                      const float* invstd, int64_t pixels, int c, double* sums, void* stream);
int gap_bn_bwd_apply(const void* y, int64_t ld_y, const void* g1, int64_t ld_g1, const void* g2, int64_t ld_g2,
                     float slope, const float* scale, const float* shift, const float* mean, const float* invstd,
                     int64_t pixels, int c, const double* sums, double count, void* dy, int64_t ld_dy,
                     void* stream);
int gap_bn_param_grads(double* sums, int c, float* dgamma, float* dbeta, void* stream);
/* After a backward-fused dgrad epilogue: raw = [sum d, sum d*y] (fp64, re-zeroed here) ->
 * sums = [sum d, sum d*xhat] with xhat = (y - mean) * invstd, for gap_bn_bwd_apply (slope 1, no g2);
 * dbeta += sum d, dgamma += sum d*xhat (either may be NULL). */
int gap_bn_bwd_finalize(double* raw, const float* mean, const float* invstd, int c, float* dgamma, float* dbeta,
                        double* sums, void* stream);
/* bias gradient: out[c] += sum over pixels of x[pixel][c] */
int gap_colsum_bf16(const void* x, int64_t ld, int64_t pixels, int c, float* out, void* stream);

/* nn.InstanceNorm2d(affine=False, track_running_stats=False) (models.py:173-191 with norm_layer=nn.InstanceNorm2d):
 * statistics per (image, channel) over hw = H*W >= 2 pixels, the same in train and eval mode (instance_norm.cu).
 * y / g1 / g2 / outputs are NHWC bf16 [n][hw][>= c] with pixel strides that are multiples of 8, c % 8 == 0, c <= 2048.
 * Per-(n,c) vectors are [N][C]; fp64 sums are [2][N*C], so gap_bn_finalize(sums, N*C, H*W, NULL, NULL, eps, 0, 1, NULL,
 * NULL, NULL, scale, shift, mean, invstd) turns the forward sums into scale = invstd, shift = -mean*invstd (and re-zeroes
 * them); gap_bn_param_grads(sums, N*C, NULL, NULL) re-zeroes the backward sums after gap_in_bwd_apply. */
/* sums[0][n*C+c] += sum y, sums[1][n*C+c] += sum y^2 */
int gap_in_stats(const void* y, int64_t ld, int n, int64_t hw, int c, double* sums, void* stream);
/* out1 = act1(y*scale[n][c] + shift[n][c]), out2 = act2(same) (optional); act = NONE / LRELU / RELU */
int gap_in_act(const void* y, int64_t ld, int n, int64_t hw, int c, const float* scale, const float* shift, void* out1,
               int64_t ld1, int act1, void* out2, int64_t ld2, int act2, void* stream);
/* xhat = y*scale + shift; d = xhat > 0 ? g1 + g2 : slope*g1 (g2 optional); sums[0] += sum d, sums[1] += sum d*xhat */
int gap_in_bwd_reduce(const void* y, int64_t ld, const void* g1, int64_t ld_g1, const void* g2, int64_t ld_g2, float slope,
                      const float* scale, const float* shift, int n, int64_t hw, int c, double* sums, void* stream);
/* dy = scale * (d - sums[0]/hw - xhat*sums[1]/hw) (bf16); dbias (optional) += the per-channel sum of the fp32 dy over
 * all images and pixels: the gradient of a conv bias in front of the norm */
int gap_in_bwd_apply(const void* y, int64_t ld, const void* g1, int64_t ld_g1, const void* g2, int64_t ld_g2, float slope,
                     const float* scale, const float* shift, int n, int64_t hw, int c, const double* sums, void* dy,
                     int64_t ld_dy, float* dbias, void* stream);

/* optim.Adam / optim.AdamW step on a flat fp32 buffer (train_gan.py:140-141,63,71; train.py:295,144).
 * grad_scale folds the 1/world_size of the data-parallel gradient all-reduce. */
int gap_adam_flat(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                  float eps, float weight_decay, int decoupled, int step, float grad_scale, void* stream);

/* Same step with the step counter kept in device memory (*step_dev is incremented, then used for the bias
 * corrections), so that a captured CUDA graph of the whole iteration can be replayed. */
int gap_adam_flat_devstep(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                          float eps, float weight_decay, int decoupled, int* step_dev, float grad_scale, void* stream);

/* loss_D = (loss_D_real + loss_D_fake) * 0.5 and loss_G = loss_G_GAN + lambda * loss_G_L1 (train_gan.py:61,68-69)
 * from the four fp64 sums the loss kernels accumulated: acc4 = [sum BCE(D(real),1), sum BCE(D(fake),0),
 * sum BCE(D(fake'),1), sum |fake-real|], count = logits per pass, numel = elements of fake.  out2 = [loss_D, loss_G];
 * acc4 is re-zeroed. */
int gap_gan_losses(double* acc4, double count, double l1_weight, double numel, double* out2, void* stream);

/* fp32 master weights (arbitrary strides) -> bf16 K-major GEMM operand; modes in elementwise.cu. */
int gap_pack_weights(const float* w, void* out, int mode, int n_phase, int rows, int rows_pad, int taps_h,
                     int taps_w, int c, int c_pad, int krow, int64_t s_r, int64_t s_c, int64_t s_kh, int64_t s_kw,
                     int kdim, void* stream);

/* All operands of a network in one launch.  `table` lives in DEVICE memory; the host fills tile_begin
 * (exclusive prefix sum of n_phase*taps_h*taps_w*tiles_r*tiles_c), tiles_r = ceil(rows/64),
 * tiles_c = ceil(c/64).  Same element mapping as gap_pack_weights modes 0-2, except that padding
 * elements (c >= C, rows >= R, k >= taps*c_pad) are not written: zero the operand buffers once. */
typedef struct gap_pack_entry {
  const float* w;
  void* out;
  int mode, n_phase, rows, rows_pad, taps_h, taps_w, c, c_pad, krow;
  int tile_begin, tiles_r, tiles_c;
  int64_t s_r, s_c, s_kh, s_kw;
} gap_pack_entry;
int gap_pack_weights_multi(const gap_pack_entry* table, int n_entries, int total_tiles, void* stream);

/* Debug knobs for bring-up (descriptor conventions); not part of the stable surface. */
int gap_debug_set(const char* key, int value);

#ifdef __cplusplus
}
#endif
#endif /* GAP_B200_H */
