/* nirgan_b200 -- C ABI of the B200 (sm_100a) NIR-GAN hot-path library.
 *
 * Every entry point takes plain device pointers, explicit sizes and an opaque CUDA stream
 * (cudaStream_t passed as void*).  No torch / C++ types cross this boundary.  The caller owns
 * every buffer; the library allocates nothing persistent apart from cached TMA descriptors.
 *
 * All compute entry points return 0 on success, a negative NG_E_* code for argument / shape /
 * alignment errors and a positive value (cudaError_t) for CUDA failures.  ng_last_error()
 * returns a thread-local human-readable message for the last non-zero status.  There is NO
 * CPU fallback: on a device that is not sm_100 the compute entry points return NG_E_ARCH.
 *
 * Tensor layouts used on the device
 *   activation  : NHWC, element type `dtype`, optional materialised halo:
 *                 [B][H + 2*pad][W + 2*pad][C]            ("haloed buffer", pad >= 0)
 *   pre-norm    : NHWC compact [B][H][W][C] (conv output before InstanceNorm)
 *   weights     : packed [tap = kh*KW + kw][n][k]  (k contiguous; n = output channel of the op)
 *   stats       : float [B][C][2] = (mean, rstd)
 *
 * Reference interfaces replaced (paths relative to the NIR-GAN repository):
 *   ng_conv2d          nn.Conv2d / nn.ConvTranspose2d call sites  model/networks.py:342,349,360-363,367,
 *                      405-427 (ResnetBlock), 559-579 (NLayerDiscriminator) and their autograd dgrad
 *   ng_conv2d_wgrad    autograd weight gradient of the same call sites (model/pix2pix.py:165-257)
 *   ng_in_stats / ng_in_stats_finalize / ng_in_apply / ng_memset_zero
 *                      nn.InstanceNorm2d + ReLU/LeakyReLU + residual add + ReflectionPad2d
 *                      model/networks.py:29-30,341-344,350-351,405-434,567-576; the SatCLIP
 *                      injection x*(1+s*e) model/generator_inject.py:113-127
 *   ng_prep_input / ng_prep_input_s2d
 *                      F.pad(..., mode='reflect') model/pix2pix.py:91-93, ReflectionPad2d(3)
 *                      model/networks.py:341, torch.cat((rgb, pred),1) model/pix2pix.py:197,202,216
 *   ng_linear          self.fc(embeds) model/generator_inject.py:110
 *   ng_lsgan_loss      GANLoss('lsgan') model/networks.py:232-233,268-270
 *   ng_adam_step / ng_adam_multi
 *                      torch.optim.Adam model/pix2pix.py:486-487 (one launch per optimizer over a flat arena)
 *   ng_in_bwd          autograd of the InstanceNorm / inject / activation / residual / halo unit above
 *   ng_stem_conv / ng_prep_stem
 *                      F.pad(reflect) + ReflectionPad2d(3) + Conv2d(3, 64, 7) straight from the fp32 tiles
 *                      (model/pix2pix.py:91-93, model/networks.py:341-342); ng_prep_stem: the row-merged tensor the
 *                      stem's weight gradient contracts over
 *   ng_head_conv / ng_tap_gather / ng_tap_scatter / ng_head_bwd_prep
 *                      the single-output-channel layers: Conv2d(64, 1, 7) + Tanh head (model/networks.py:366-368) and the
 *                      PatchGAN logit Conv2d(512, 1, 4, 1, 1) (model/networks.py:574-576) in one kernel; the two-kernel
 *                      form of the head and the adjoints, incl. the wrapper's crop
 *   ng_rs_pixel_losses / ng_rs_index
 *                      L1Loss model/pix2pix.py:60,222 + all six RemoteSensingIndices, criterion l1 / l2,
 *                      loss / logging / index modes utils/remote_sensing_indices.py:23-319 (forward and d/dpred)
 *   ng_ssim_loss / ng_emd_loss
 *                      utils/losses.py:10-29,64-78 (ssim_loss; emd_loss = pix2pix.py's hist_loss)
 *   ng_image_metrics   utils/calculate_metrics.py:6-37 (L1, L2, PSNR, SSIM)
 *   ng_resize_plane / ng_hist_match / ng_sort_segments
 *                      F.interpolate + skimage.exposure.match_histograms, create_synthetic_dataset.py:34-52,111-118
 *   ng_scene_tiles / ng_scene_blend / ng_scene_tile_valid / ng_scene_blend_masked / ng_scene_blend_indices
 *                      the per-tile `model(hr)` loop of create_synthetic_dataset.py:100-118 over pre-cut files plus the
 *                      cutting and stitching a user writes around it for a whole scene (the reference has neither)
 *   ng_satclip_encode  SatClIP_wrapper.predict model/satclip/satclip_wrapper.py:29-34 (location_encoder.py:73-151,
 *                      267-275; positional_encoding/spherical_harmonics.py:27-42)
 *   ng_grad_scale_pow2 / ng_unpack_weight_grad* / ng_grad_to_nchw / ng_inject_bwd / ng_nonfinite_flag
 *                      plumbing of the training step (fp16 gradient scale, gradient export in the reference layout)
 */
#ifndef NIRGAN_B200_H_
#define NIRGAN_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NG_VERSION 102

/* element types (NG_U16: unsigned 16-bit digital numbers, scene input of ng_scene_tiles only) */
enum { NG_F32 = 0, NG_F16 = 1, NG_BF16 = 2, NG_U16 = 3 };
/* conv implementations */
enum { NG_IMPL_SIMT = 0,   /* CUDA-core fp32-accumulate implicit GEMM (verification mode, any dtype) */
       NG_IMPL_TC = 1 };   /* tcgen05 / TMEM / TMA implicit GEMM (f16 or bf16 operands) */
/* conv forms */
enum { NG_FORM_GATHER = 0,     /* out[y] = sum_k in[y*stride + sgn*k - sgn*pad] * w[k]   (conv, dgrad of convT / s1 conv) */
       NG_FORM_PHASED = 1,     /* out[stride*i + a] = sum_{k == a+pad (mod stride)} in[i + (a+pad-k)/stride] * w[k]
                                  (ConvTranspose2d, dgrad of a strided conv) */
       NG_FORM_PHASED_MERGED = 2 };
                               /* the same ConvTranspose2d(k3, s2, p1, op1) with the four output-parity phases merged into
                                  the GEMM-N dimension: N = 4*Cout virtual channels (phase-major), K = 4 input shifts
                                  (0/1 rows x 0/1 columns) x Cin; weights packed by ng_pack_weight_phasemerged (zeros
                                  where a phase does not use a shift).  Each input tile is fetched once per shift instead
                                  of once per (phase, tap) and every MMA is N >= 256 wide.  TC only. */
/* epilogues */
enum { NG_EPI_RAW = 0,        /* store pre-norm output (+ per-tile sum / sum-of-squares partials) */
       NG_EPI_BIAS_ACT = 1,   /* out = act(acc + bias) stored as `dtype` NHWC */
       NG_EPI_HEAD = 2 };     /* single output channel: out = act(acc + bias) stored fp32 [B][H-2c][W-2c] */
/* activations */
enum { NG_ACT_NONE = 0, NG_ACT_RELU = 1, NG_ACT_LRELU = 2, NG_ACT_TANH = 3 };
/* halo modes */
enum { NG_HALO_ZERO = 0, NG_HALO_REFLECT = 1 };
/* injection styles (model/generator_inject.py:122-127) */
enum { NG_INJECT_NONE = 0, NG_INJECT_ADD = 1, NG_INJECT_MUL_SCALED = 2, NG_INJECT_MUL = 3 };

/* error codes */
enum { NG_OK = 0, NG_E_ARG = -1, NG_E_SHAPE = -2, NG_E_ALIGN = -3, NG_E_ARCH = -4, NG_E_UNSUPPORTED = -5,
       NG_E_DRIVER = -6 };

typedef struct ng_conv_args {
  int32_t dtype;        /* NG_F32 / NG_F16 / NG_BF16: element type of x, w and (for RAW / BIAS_ACT) y */
  int32_t impl;         /* NG_IMPL_* */
  int32_t form;         /* NG_FORM_* */
  int32_t sgn;          /* +1 (correlation) or -1 (flipped taps; dgrad of a stride-1 conv). GATHER only */
  int32_t B, Hin, Win, Cin;   /* input interior; Cin is the stored (padded) channel count */
  int32_t in_pad;       /* halo rows materialised above/below the input interior */
  int32_t in_pad_w;     /* halo columns materialised left/right (usually == in_pad) */
  int32_t Cout;         /* stored output channels (multiple of 8; HEAD: 16, of which channel 0 is real) */
  int32_t KH, KW, stride;
  int32_t pad;          /* logical padding along H */
  int32_t pad_w;        /* logical padding along W (usually == pad) */
  int32_t Hout, Wout;
  int32_t epilogue;     /* NG_EPI_* */
  int32_t act;          /* NG_ACT_* (BIAS_ACT / HEAD) */
  float   slope;        /* LeakyReLU slope */
  int32_t crop;         /* HEAD: rows/cols cropped from every border of the output */
  int32_t reserved;
  const void* x;        /* [B][Hin+2*in_pad][Win+2*in_pad][Cin] */
  const void* w;        /* packed [KH*KW][Cout][Cin] */
  const float* bias;    /* [Cout] or NULL */
  void* y;              /* RAW/BIAS_ACT: [B][Hout][Wout][Cout] dtype; HEAD: float [B][Hout-2c][Wout-2c] */
  float* stat_partials; /* RAW + TC: [B][ng_conv_stat_slots][Cout][2] (sum, sumsq) or NULL */
  /* optional fused InstanceNorm finalisation (TC + RAW + stat_partials): the CTA that completes the last tile of an
   * image reduces that image's partials in a fixed order and writes (mean, rstd) itself, so no separate
   * ng_in_stats_finalize launch is needed.  tile_counters: [B] int32, zero before the first launch (the kernel leaves
   * them zero again); mean_rstd: [B][Cout][2]; both NULL = off. */
  float* mean_rstd;
  int32_t* tile_counters;
  /* optional fixed-point statistics accumulators (TC + RAW): [B][Cout][2] int64, ZERO before the launch
   * (ng_memset_zero).  Every tile adds its per-channel sum * 2^NG_STAT_SUM_SHIFT and sum of squares *
   * 2^NG_STAT_SQ_SHIFT with 64-bit integer atomics -- integer addition is associative, so the totals do not depend
   * on the order in which tiles finish (deterministic, bit-identical across batch slices and shardings) -- and
   * ng_in_apply turns them into (mean, rstd) itself: no ng_in_stats_finalize launch, stat_partials may be NULL. */
  int64_t* stat_acc;
} ng_conv_args;

#define NG_STAT_SUM_SHIFT 24
#define NG_STAT_SQ_SHIFT 20

int         ng_version(void);
const char* ng_last_error(void);
/* 0 when `device` is an sm_100 GPU usable by this library */
int         ng_device_check(int device);

/* number of per-image partial-statistics slots ng_conv2d(TC, RAW) writes for this geometry */
int ng_conv_stat_slots(const ng_conv_args* a);
int ng_conv2d(const ng_conv_args* a, void* stream);

/* weight gradient: dw[tap][n][k] (fp32, packed layout) = sum_pixels dy[.., n] * x[.. shifted by tap .., k]
 * with the geometry of the forward op described by `a` (a->x = forward input, a->y = dY compact).
 * impl == NG_IMPL_TC with 16-bit operands, Cin in {64,128,256} and Cout % 64 == 0 runs the tcgen05 split-K kernel
 * (MN-major operands straight from the NHWC tensors; deterministic two-stage reduction) and needs a caller-provided
 * workspace of ng_conv2d_wgrad_workspace_bytes(a) bytes; other geometries (and workspace == NULL) use the CUDA-core
 * kernel.  dbias (optional) = per-channel sum of dy. */
int64_t ng_conv2d_wgrad_workspace_bytes(const ng_conv_args* a);
int ng_conv2d_wgrad(const ng_conv_args* a, float* dw_packed, float* dbias, void* workspace, int64_t workspace_bytes,
                    void* stream);

/* pack an fp32 weight (4-D, [d0][d1][KH][KW]) into [tap][n][k]; n_axis selects which of d0/d1 is n.
 * k is zero-padded to k_pad, n to n_pad. */
int ng_pack_weight(const float* src, int32_t d0, int32_t d1, int32_t KH, int32_t KW, int32_t n_axis,
                   int32_t n_pad, int32_t k_pad, int32_t dtype, void* dst, void* stream);
/* inverse for gradients: dst[d0][d1][KH][KW] = beta * dst + scale * dev_scale[0] * packed[tap][n_pad][k_pad]  (fp32;
 * undoes the loss scaling: `scale` is the host-known static part, dev_scale (device pointer, may be NULL) the adaptive
 * part written by ng_grad_scale_pow2; beta = 0 overwrites -- dst is not read --, beta = 1 accumulates like autograd's
 * AccumulateGrad when a parameter is reached twice in one backward pass or .grad was not cleared) */
int ng_unpack_weight_grad(const float* packed, int32_t d0, int32_t d1, int32_t KH, int32_t KW, int32_t n_axis,
                          int32_t n_pad, int32_t k_pad, float scale, const float* dev_scale, float beta, float* dst,
                          void* stream);

/* weights for NG_FORM_PHASED_MERGED: ConvTranspose2d weight fp32 [Cin][Cout][3][3] ->
 * [shift = sy*2+sx][n = phase*Cout + co][Cin], phase = (oy&1)*2 + (ox&1); entry = w[ci][co][pa+1-2sy][pb+1-2sx] or 0 */
int ng_pack_weight_phasemerged(const float* src, int32_t Cin, int32_t Cout, int32_t dtype, void* dst, void* stream);

/* Generator stem input in "row-merged" form: NCHW fp32 -> [B][H+2*wrap+2*halo][W+2*wrap][64] `dtype`, where element
 * (kw*8 + c) of output pixel (y, x) is channel c of the reflect-padded image at (y, x + kw)  (kw < KW <= 8, c < cin <= 8,
 * zero elsewhere).  A KHxKW convolution over cin channels then becomes a KHx1 convolution over 64 "channels" whose
 * GEMM-K rows are 128 contiguous bytes (one TMA / UMMA swizzle row).  Replaces ReflectionPad2d(3) + the im2col half of
 * Conv2d(3->64, k7) (model/networks.py:341-342) and Px2Px_PL.forward's F.pad (model/pix2pix.py:91-93). */
int ng_prep_stem(const float* src, int32_t cin, int32_t B, int32_t H, int32_t W, int32_t wrap_pad, int32_t halo,
                 int32_t KW, int32_t dtype, void* dst, void* stream);
/* weights for the row-merged stem: fp32 [O][I][KH][KW] -> [kh][O][kw*c_slots + c] (c_slots = 8: zero padded to 64
 * elements, the ng_prep_stem layout; c_slots = 4: 32 elements, the ng_stem_conv layout; I <= c_slots, KW <= 8) */
int ng_pack_weight_rowmerged(const float* src, int32_t O, int32_t I, int32_t KH, int32_t KW, int32_t c_slots,
                             int32_t dtype, void* dst, void* stream);
/* The generator stem -- F.pad(reflect, wrap_pad) + ReflectionPad2d(3) + Conv2d(cin -> 64, k7) (model/pix2pix.py:91-93,
 * model/networks.py:341-342) -- straight from the caller's NCHW fp32 tiles on the tensor cores: src [B][cin][H][W]
 * (cin <= 4) -> y [B][H+2*wrap_pad][W+2*wrap_pad][64] pre-norm `dtype` (+ InstanceNorm statistics as for ng_conv2d:
 * stat_partials [B][ng_stem_conv_stat_slots][64][2] and / or stat_acc [B][64][2], either may be NULL).  The im2col tile
 * (row-merged, 32 elements per pixel) is assembled in shared memory inside the kernel: no intermediate tensor.
 * w_packed: ng_pack_weight_rowmerged(..., c_slots = 4, ...) = [7][64][32].  The conv bias is not applied (it cancels in
 * the InstanceNorm that follows). */
int ng_stem_conv(const float* src, int32_t cin, int32_t B, int32_t H, int32_t W, int32_t wrap_pad, const void* w_packed,
                 int32_t dtype, void* y, float* stat_partials, int64_t* stat_acc, void* stream);
int ng_stem_conv_stat_slots(int32_t H, int32_t W, int32_t wrap_pad);
/* inverse for gradients: fp32 [kh][O][64] -> fp32 [O][I][KH][KW], dst = beta * dst + scale * dev_scale[0] * packed */
int ng_unpack_weight_grad_rowmerged(const float* packed, int32_t O, int32_t I, int32_t KH, int32_t KW, float scale,
                                    const float* dev_scale, float beta, float* dst, void* stream);

/* Single-output-channel KHxKW convolution as "tap GEMM + gather": z = [B][Hz][Wz][zc] holds, per input pixel, the
 * dot product of its channels with each of the KH*KW taps (a 1x1 ng_conv2d with Cout = zc >= KH*KW);
 * out[n][y][x] = act(bias + sum_{kh,kw} z[n][y+kh][x+kw][kh*KW+kw]) for the (Hz-KH+1-2*crop) x (Wz-KW+1-2*crop)
 * cropped output.  Replaces Conv2d(64->1, k7) + Tanh (model/networks.py:366-368) without the 49x im2col re-read. */
int ng_tap_gather(const void* z, int32_t dtype, int32_t B, int32_t Hz, int32_t Wz, int32_t zc, int32_t KH, int32_t KW,
                  const float* bias, int32_t act, int32_t crop, float* out, void* stream);

/* Single-output-channel convolution in ONE kernel (16-bit storage): the generator head Conv2d(64 -> 1, k7) + Tanh
 * (model/networks.py:366-368; C = 64, K = 7) and the PatchGAN's last layer Conv2d(512 -> 1, k4, p1)
 * (model/networks.py:574-576; C = 512, K = 4).  Per 8 x 16 output patch the haloed (8+K-1) x (16+K-1) x C input patch is
 * fetched once by TMA (64 channels per pipeline stage), the tap GEMM z[pixel][tap] of the whole patch runs on tcgen05 into
 * TMEM, and the K*K shifted taps are summed from a shared-memory z tile -- z never goes to HBM (the ng_conv2d tap GEMM +
 * ng_tap_gather pair writes and re-reads it; the im2col form re-reads the input once per tap).
 * H x W: the convolution's output; pad: its padding (3 / 1); halo (<= pad): the part of the padding that is materialised
 * in the buffer, x_haloed = [B][H+K-1-2*(pad-halo)][W+K-1-2*(pad-halo)][C] (the head's reflect halo of 3 is written by
 * ng_in_apply; the PatchGAN buffers carry none: the rest of the padding is zeros by TMA out-of-bounds fill),
 * w_taps: [taps stored (64 for K = 7, 16 for K = 4)][C] as packed by ng_pack_weight for the tap GEMM,
 * out: fp32 [B][H-2*crop][W-2*crop] = act(bias + conv). */
int ng_head_conv(const void* x_haloed, int32_t dtype, int32_t B, int32_t H, int32_t W, int32_t C, int32_t K, int32_t pad,
                 int32_t halo, const void* w_taps, const float* bias, int32_t act, int32_t crop, float* out, void* stream);

/* Backward of ng_tap_gather: dz[n][yy][xx][kh*KW+kw] = scale * dev_scale[0] * dout[n][yy-kh-crop][xx-kw-crop] * act'(out)
 * (zero outside the cropped output window; taps >= KH*KW zero).  With dz, the weight gradient of the single-channel
 * convolution is a 1x1 ng_conv2d_wgrad (dW[tap][k] = sum_px dz[px][tap] x[px][k]) and its data gradient a 1x1
 * ng_conv2d over dz -- both on the tensor cores.  Autograd of Conv2d(64->1, k7) + Tanh (model/networks.py:366-368). */
int ng_tap_scatter(const float* dout, const float* out, int32_t B, int32_t Hz, int32_t Wz, int32_t zc, int32_t KH,
                   int32_t KW, int32_t act, int32_t crop, float scale, const float* dev_scale, int32_t dtype, void* dz,
                   void* stream);

/* NCHW fp32 (one or two sources concatenated on C) -> haloed NHWC `dtype` with channels zero-padded to c_pad.
 * wrap_pad: reflect padding applied first (Px2Px_PL.forward, padding_amount); halo: second reflect (or zero) halo. */
int ng_prep_input(const float* src_a, int32_t ca, const float* src_b, int32_t cb, int32_t B, int32_t H, int32_t W,
                  int32_t wrap_pad, int32_t halo, int32_t halo_mode, int32_t c_pad, int32_t dtype, void* dst,
                  void* stream);

/* Space-to-depth form of the PatchGAN input layer Conv2d(4 -> 64, k4, s2, p1) (model/networks.py:559): the zero-padded
 * (pad 1) channel concatenation of src_a / src_b is written as [B][(H+2)/2][(W+2)/2][(py*2+px)*16 + c] `dtype` (H, W even,
 * ca + cb <= 16, 16-bit), on which the layer is a 2x2 STRIDE-1 convolution over 64 stored channels -- kernel position
 * (kh, kw) = (2*dy + py, 2*dx + px), a bijection -- i.e. an ordinary ng_conv2d / ng_conv2d_wgrad with KH = KW = 2, pad 0.
 * ng_pack_weight_s2d packs the fp32 [O][I][4][4] master as [tap = dy*2+dx][O][64] (transpose 0) or [tap][64][O]
 * (transpose 1: the data gradient's operand); ng_unpack_weight_grad_s2d is the inverse for the weight gradient. */
int ng_prep_input_s2d(const float* src_a, int32_t ca, const float* src_b, int32_t cb, int32_t B, int32_t H, int32_t W,
                      int32_t dtype, void* dst, void* stream);
int ng_pack_weight_s2d(const float* src, int32_t O, int32_t I, int32_t transpose, int32_t dtype, void* dst, void* stream);
int ng_unpack_weight_grad_s2d(const float* packed, int32_t O, int32_t I, float scale, const float* dev_scale, float beta,
                              float* dst, void* stream);

/* per-(n,c) mean / rstd (eps 1e-5, biased variance) of a compact NHWC tensor */
int ng_in_stats(const void* y, int32_t dtype, int32_t B, int32_t HW, int32_t C, float* mean_rstd, void* stream);
/* same from the conv epilogue partial sums */
int ng_in_stats_finalize(const float* partials, int32_t B, int32_t slots, int32_t C, int32_t count,
                         float* mean_rstd, void* stream);

/* out = act( inject( (y - mean) * rstd ) ) + residual, written with a halo of out_pad.
 * Statistics: mean_rstd ([B][C][2] floats) when given; else stat_acc ([B][C][2] int64 fixed-point sums written by
 * ng_conv2d, see ng_conv_args.stat_acc) from which every block derives mean = S/(H*W), rstd = rsqrt(Q/(H*W) - mean^2 +
 * 1e-5) for its channels -- and, when mean_rstd_out is given, the first block of each image also stores them as floats
 * for the backward pass; both NULL skips the normalisation (y is used as is). */
int ng_in_apply(const void* y, int32_t dtype, int32_t B, int32_t H, int32_t W, int32_t C, const float* mean_rstd,
                const int64_t* stat_acc, float* mean_rstd_out, int32_t act, float slope, const void* residual,
                int32_t res_pad, const float* inject_e, int32_t inject_mode, const float* inject_scale, void* out,
                int32_t out_pad, int32_t halo_mode, void* stream);
/* cudaMemsetAsync(ptr, 0, bytes) on `stream` (the statistics accumulators of a whole plan are cleared by one call) */
int ng_memset_zero(void* ptr, int64_t bytes, void* stream);

/* Backward of the unit computed by ng_in_apply (autograd of InstanceNorm2d / ReLU / LeakyReLU / residual add /
 * ReflectionPad2d / the SatCLIP injection; model/pix2pix.py:165-257 runs it through torch autograd):
 *   g_halo : dL/d(haloed output buffer) [B][H+2*g_pad][W+2*g_pad][C] or NULL (halo folded back per halo_mode).
 *            CONSUMED: with 16-bit storage and a reflect halo the fold is done in place (the halo contributions are added
 *            into the interior pixels next to the border before the two passes stream the interior), so the buffer
 *            must not be handed to a second ng_in_bwd call without being produced again.
 *   g_skip : dL/d(output interior) from a skip connection, compact [B][H][W][C], or NULL
 *   y, mean_rstd : the forward's pre-norm tensor and statistics (mean_rstd NULL = unit without normalisation)
 *   dy     : dL/dy compact [B][H][W][C];  do_out (optional): dL/d(output interior) for the residual path
 *   dscale / de_map (optional): accumulated dL/d(scale_param) (1 float, caller zero-initialised) and
 *   dL/d(bilinear embedding map) [B][H][W] for the injection.   sums_scratch: ng_in_bwd_scratch_floats(B,H,W,C)
 *   floats (per-block partial sums, added in a fixed order by the second pass: no atomics, deterministic). */
int64_t ng_in_bwd_scratch_floats(int32_t B, int32_t H, int32_t W, int32_t C);
int ng_in_bwd(void* g_halo, int32_t g_pad, int32_t halo_mode, const void* g_skip, const void* y, int32_t dtype,
              int32_t B, int32_t H, int32_t W, int32_t C, const float* mean_rstd, int32_t act, float slope,
              const float* inject_e, int32_t inject_mode, const float* inject_scale, float* sums_scratch, void* dy,
              void* do_out, float* dscale, float* de_map, void* stream);
/* Adaptive power-of-two gradient scale for the 16-bit backward pass: out4[0] = f = 2^floor(log2(target / max|g|))
 * (1 if g is all zero or not finite), out4[1] = 1/f, out4[2..3] scratch.  The backward plan is linear in the incoming
 * gradient, so entering with g*f and leaving with (1/f) is exact; it keeps the largest gradient element at `target`
 * whatever the loss weights, batch size or singular pixels of the spectral-index losses. No host synchronisation. */
int ng_grad_scale_pow2(const float* g, int64_t n, float target, float* out4, void* stream);
/* dst[B][H][W][c_pad] (dtype): channel 0 = scale * dev_scale[0] * dout * act'(out) inside the crop window, zero
 * elsewhere.  dout/out: fp32 [B][H-2*crop][W-2*crop] (the fp32 single-channel head output and its gradient).
 * dev_scale: device pointer or NULL. */
int ng_head_bwd_prep(const float* dout, const float* out, int32_t B, int32_t H, int32_t W, int32_t crop, int32_t act,
                     float scale, const float* dev_scale, int32_t c_pad, int32_t dtype, void* dst, void* stream);
/* gradient export: channels [c0, c0 + c) of NHWC [B][H][W][c_pad] (dtype) -> NCHW fp32 [B][c][H][W], times
 * scale * dev_scale[0]  (the G pass needs dL/d(pred) only: channel 3 of the PatchGAN's (rgb, pred) input).
 * s2d != 0: the source is in the space-to-depth layout of ng_prep_input_s2d (c_pad = channel slots per parity). */
int ng_grad_to_nchw(const void* src, int32_t dtype, int32_t B, int32_t H, int32_t W, int32_t c_pad, int32_t c0, int32_t c,
                    int32_t s2d, float scale, const float* dev_scale, float* dst, void* stream);
/* SatCLIP injection backward: adjoint of the bilinear resize (128x128 -> HxW) then of fc:
 * dfc_w[16384][256] = (scale * A^T de_map)^T embeds, dfc_b[16384].  de128_scratch: [B][16384] floats. */
int ng_inject_bwd(const float* de_map, int32_t B, int32_t H, int32_t W, float scale, const float* dev_scale,
                  const float* embeds, float* de128_scratch, float* dfc_w, float* dfc_b, void* stream);

/* y[b][n] = sum_k x[b][k] * w[n][k] + bias[n]   (fp32) */
int ng_linear(const float* x, const float* w, const float* bias, int32_t B, int32_t K, int32_t N, float* y,
              void* stream);

/* mean((p - target)^2) over n elements -> loss[0] (+= when accumulate); loss must have room for 2 floats
 * (loss[1] is scratch); grad (optional) = gscale*2*(p-target)/n */
int ng_lsgan_loss(const float* p, int64_t n, float target, float* loss, int32_t accumulate, float* grad,
                  float gscale, void* stream);

/* Every term of RemoteSensingIndices (utils/remote_sensing_indices.py:84-319) plus the pix2pix L1 term in one pass over
 * NCHW fp32 planes.  Term order (= the reference's iteration order, :45-52): 0 L1(pred, nir), 1 NDVI, 2 NDWI, 3 GNDVI,
 * 4 SAVI, 5 MSAVI, 6 EVI; out8[k] = mean criterion of term k for the terms selected by bit k of `mask` (0 otherwise;
 * out8 has room for 8 floats).  criterion 0 = l1, 1 = l2 (F.mse_loss) for the six indices.  dpred (optional) =
 * d( sum_k w[k] * term_k ) / dpred with w = weights7_dev (7 floats on the device: the upstream gradient of every term as
 * autograd delivers it) when given, else the host array weights7.  scratch: >= 8*1024 floats. */
int ng_rs_pixel_losses(const float* rgb, const float* nir, const float* pred, int32_t B, int32_t HW,
                       const float* weights7, const float* weights7_dev, int32_t criterion, int32_t mask, float* out8,
                       float* dpred, float* scratch, void* stream);
/* 'index' mode: the index maps of the target and of the prediction (which = 1..6 as above); loss_eps != 0 keeps the
 * loss-mode epsilons, 0 gives the index-mode formulas (remote_sensing_indices.py:101,137,304-316) */
int ng_rs_index(const float* rgb, const float* nir, const float* pred, int32_t B, int32_t HW, int32_t which,
                int32_t loss_eps, float* out_target, float* out_pred, void* stream);

/* Adam (torch defaults: eps 1e-8, no weight decay, bias-corrected) on a flat fp32 parameter vector */
int ng_adam_step(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                 float eps, int32_t step, float grad_scale, void* stream);

/* Multi-tensor Adam: one launch for every parameter of an optimizer.  params_dev / offsets_dev / numel_dev: device
 * arrays of `ntensors` parameter pointers, their element offsets into the flat gradient / moment arenas g, m, v (`total`
 * elements, slots may be padded for alignment) and their element counts (arena elements at or beyond a tensor's count are
 * padding and are never written through).  step_counter_dev: device int32 holding the number of updates applied so far (advanced here, used for the
 * bias corrections).  skip_flag (device, optional): a non-zero value makes the whole call a no-op (see
 * ng_nonfinite_flag) -- torch.cuda.amp-style step skipping without a host round trip. */
int ng_adam_multi(void* const* params_dev, const int64_t* offsets_dev, const int64_t* numel_dev, int32_t ntensors,
                  const float* g, float* m, float* v, int64_t total, float lr, float beta1, float beta2, float eps, int32_t* step_counter_dev,
                  float grad_scale, const int32_t* skip_flag, void* stream);
/* flag[0] = 1 if any of the n floats is inf or NaN, else 0 */
int ng_nonfinite_flag(const float* x, int64_t n, int32_t* flag, void* stream);

/* ---- post-processing after the generator (create_synthetic_dataset.py:34-52,111-118; SURVEY.md 8f rank 1) ---------- */
/* plane resize with F.interpolate semantics: mode 0 'nearest' (the scale_factor=4 upsampling of the Sentinel-2 NIR,
 * create_synthetic_dataset.py:111), mode 1 'bilinear' align_corners=False (histogram_match, :37).  fp32 planes. */
int ng_resize_plane(const float* src, int32_t planes, int32_t h, int32_t w, int32_t H, int32_t W, int32_t mode,
                    float* dst, void* stream);
/* per-tile histogram matching = skimage.exposure.match_histograms(img, ref, channel_axis=None) for every tile of a
 * batch (create_synthetic_dataset.py:41-47): image [B][N], reference [B][M] fp32; out [B][N] as NG_F32 or NG_F16 (the
 * reference stores float16, :116).  Segmented radix sort of both arrays + three binary searches per pixel. */
int64_t ng_hist_match_workspace_bytes(int32_t B, int32_t N, int32_t M);
int ng_hist_match(const float* image, const float* reference, int32_t B, int32_t N, int32_t M, int32_t out_dtype,
                  void* out, void* workspace, int64_t workspace_bytes, void* stream);
/* the building block on its own: ascending sort of `segs` segments of n floats (-0.0 == +0.0);
 * workspace >= segs*n*8 + segs*ceil(n/4096)*1024 bytes */
int ng_sort_segments(const float* src, int32_t segs, int32_t n, float* sorted_out, void* workspace,
                     int64_t workspace_bytes, void* stream);

/* ---- whole-scene inference (nirgan_b200/scene.py) ------------------------------------------------------------------ */
/* Cut n windows of T x T out of a scene into the generator's input layout: scene [C][rows][W] holds scene rows
 * [row0, row0 + rows) (a band may be resident instead of the whole scene) as NG_F32 reflectance or NG_U16 digital
 * numbers, origins [n][2] int32 (device, 8-byte aligned) the windows' (y0, x0) in scene coordinates, dst [n][C][T][T]
 * fp32 (16-byte aligned when T % 4 == 0).  NG_U16 values become (float)dn / dn_scale (IEEE division); a window that is
 * not inside the resident rows is written as NaN.  One pass: conversion and cut. */
int ng_scene_tiles(const void* scene, int32_t dtype, int32_t C, int32_t rows, int32_t W, int32_t row0,
                   const int32_t* origins, int32_t n, int32_t T, float dn_scale, float* dst, void* stream);
/* Weighted blend of a grid of tile predictions into output rows [y0, y1) of a W-wide band: pred [ny*nx][T][T] fp32 is
 * the prediction of the tile at (oy[ky], ox[kx]) at index ky*nx + kx; oy [ny] and ox [nx] (device int32, ascending)
 * must cover rows [y0, y1) and columns [0, W).  out [y1-y0][W] fp32 =
 *   sum_t w_t p_t / sum_t w_t  over the covering tiles in ascending (ky, kx) order, fp32,
 *   w(i, j) = w1(i) w1(j),  w1(i) = min(i + 1, T - i, overlap + 1) / (overlap + 1)
 * (evaluated as the exact integers (overlap + 1)^2 w, the factor cancels), and exactly p_t where a single tile covers the pixel; an uncovered pixel is NaN.  Every pixel is written once (gather
 * form, no atomics): deterministic, and bit-identical whichever band computes it. */
int ng_scene_blend(const float* pred, const int32_t* oy, int32_t ny, const int32_t* ox, int32_t nx, int32_t T,
                   int32_t overlap, int32_t W, int32_t y0, int32_t y1, float* out, void* stream);
/* Nodata (GDAL's per-dataset mask): a pixel is nodata when every channel equals `nodata` -- NG_F32: v == nodata, and NaN
 * matches NaN; NG_U16: the raw digital number compared as an exact float.  Valid pixels of each of n windows:
 * scene / dtype / C / rows / W / row0 / origins as in ng_scene_tiles; counts [n] int32 (device) gets the number of
 * valid pixels of the window, or -1 for a window not inside the resident rows.  An integer reduction without atomics
 * (deterministic); reads C T^2 elements per window. */
int ng_scene_tile_valid(const void* scene, int32_t dtype, int32_t C, int32_t rows, int32_t W, int32_t row0,
                        const int32_t* origins, int32_t n, int32_t T, float nodata, int32_t* counts, void* stream);
/* ng_scene_blend over a compacted prediction buffer, with nodata pixels written as nodata_out: tile ky*nx + kx is row
 * slot[ky*nx + kx] (device int32) of pred, or skipped when the slot is -1 (a tile without a valid pixel; no valid pixel
 * reads it).  scene [C][rows][W] (NG_F32 or NG_U16) holds scene rows [row0, row0 + rows), which must contain [y0, y1);
 * a pixel that is nodata there (rule above) is nodata_out, every other pixel is exactly what ng_scene_blend gives for
 * the uncompacted grid. */
int ng_scene_blend_masked(const float* pred, const int32_t* slot, const int32_t* oy, int32_t ny, const int32_t* ox,
                          int32_t nx, int32_t T, int32_t overlap, int32_t W, int32_t y0, int32_t y1, const void* scene,
                          int32_t dtype, int32_t C, int32_t rows, int32_t row0, float nodata, float nodata_out,
                          float* out, void* stream);
/* ng_scene_blend (slot NULL) or ng_scene_blend_masked (slot given), followed by k index bands:
 * out [1 + k][y1-y0][W] fp32 (16-byte aligned when W % 4 == 0), plane 0 the blended NIR, bit-identical to what those
 * entry points give, plane 1 + i index which[i] (host int32 [k], 1 <= k <= 6, values 1..6: NDVI, NDWI, GNDVI, SAVI,
 * MSAVI, EVI, utils/remote_sensing_indices.py's order) in index mode -- bit-identical to ng_rs_index(loss_eps = 0) of
 * that NIR.  R, G, B are channels 0, 1, 2 of scene [C][rows][W] (NG_F32 as is, NG_U16 as (float)dn / dn_scale, the
 * values ng_scene_tiles cuts), which holds scene rows [row0, row0 + rows) and must contain [y0, y1); C >= 3.  With
 * use_nodata != 0 a nodata pixel (rule above) is nodata_out in every plane, without it no pixel is masked (slot may
 * still be given).  Each element is written once. */
int ng_scene_blend_indices(const float* pred, const int32_t* slot, const int32_t* oy, int32_t ny, const int32_t* ox,
                           int32_t nx, int32_t T, int32_t overlap, int32_t W, int32_t y0, int32_t y1, const void* scene,
                           int32_t dtype, int32_t C, int32_t rows, int32_t row0, float dn_scale, int32_t use_nodata,
                           float nodata, float nodata_out, const int32_t* which, int32_t k, float* out, void* stream);

/* Optional generator losses (utils/losses.py:10-29 ssim_loss, :64-78 emd_loss -- pix2pix.py:12-13,233-242), forward and
 * d/dpred (dpred may be NULL).  ssim_loss: out1[0] = 1 - mean(kornia.metrics.ssim(pred, target, window)); planes = B*C;
 * scratch: ng_ssim_loss_scratch_floats() floats, 16-byte aligned.  emd_loss: per sample softmax over the N = C*H*W
 * entries, cumulative sums, out1[0] = mean |cdf_pred - cdf_target| over B*N; scratch: B doubles. */
int64_t ng_ssim_loss_scratch_floats(int32_t planes, int32_t H, int32_t W);
int ng_ssim_loss(const float* pred, const float* target, int32_t planes, int32_t H, int32_t W, int32_t window,
                 float max_val, float* out1, float* dpred, float* scratch, void* stream);
int ng_emd_loss(const float* pred, const float* target, int32_t B, int32_t N, float* out1, float* dpred,
                double* scratch, void* stream);

/* SatCLIP location encoder (model/satclip/satclip_wrapper.py:29-34, location_encoder.py:73-151,267-275,
 * positional_encoding/spherical_harmonics.py:27-42 + spherical_harmonics_closed_form.py:8-40): lonlat [B][2] degrees
 * (float64) -> L*L real spherical harmonics -> SIREN MLP -> out [B][dim_out] float32; float64 arithmetic like the
 * reference.  params_t: float64 blob, per hidden layer W^T [in][hidden] then bias [hidden], then W_last^T [hidden][dim_out]
 * and bias [dim_out] (transposed so the reads coalesce). */
int ng_satclip_encode(const double* lonlat, int32_t B, int32_t L, const double* params_t, int32_t hidden,
                      int32_t num_layers, int32_t dim_out, double w0_initial, double w0, float* out, void* stream);

/* Validation metrics (utils/calculate_metrics.py:6-37): out4 = { F.l1_loss, F.mse_loss, kornia.metrics.psnr(.., max_val),
 * kornia.metrics.ssim(.., window, max_val).mean() } over `planes` = B*C fp32 planes of HxW.  window odd, <= 11 (5 in
 * calculate_metrics, 11 in utils/losses.py::ssim_loss).  scratch: ng_image_metrics_scratch_floats() floats. */
int64_t ng_image_metrics_scratch_floats(int32_t planes, int32_t H, int32_t W);
int ng_image_metrics(const float* pred, const float* target, int32_t planes, int32_t H, int32_t W, int32_t window,
                     float max_val, float* out4, float* scratch, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NIRGAN_B200_H_ */
