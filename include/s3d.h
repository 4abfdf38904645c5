/*
 * s3d.h -- C ABI of libs3d_b200.so, the B200 (sm_100a) hot path for the
 * Stereo2Voxel / Stereo2Point inference pipeline.
 *
 * Boundary contract (SURVEY.md 8(b)):
 *   - plain C: raw DEVICE pointers, integer shapes, a cudaStream_t passed as void*;
 *     no torch types, no allocation, no synchronisation, no global state except the
 *     last-error slot; every entry point enqueues on the caller's stream and returns
 *     0 on success or a negative S3D_ERR_* code (never throws across the ABI);
 *   - all memory (inputs, outputs, workspaces) is owned by the caller (PyTorch);
 *   - there is NO CPU fallback: on a box without a CUDA device every compute entry
 *     point returns S3D_ERR_CUDA.
 *
 * What each entry point replaces in the reference.  The reference's model code is on
 * the upstream Stereo2Voxel / Stereo2Point branches (/root/reference/README.md:5,56,62)
 * and is NOT on disk, so the only citable reference interfaces are
 *   - extensions/chamfer_dist (README.md:62-65)  -> s3d_chamfer_forward
 *   - runner.py --test --weights (README.md:91)  -> the nn.Module forwards in
 *     stereo_3d_reconstruction_b200/, which call the s3d_* entry points below where
 *     upstream calls torch.nn.functional conv2d / conv3d / conv_transpose3d / softmax
 *     (torch>=1.4.0, requirements.txt:8).
 *
 * Tensor layout: activations are channels-last, 5-D [N, D, H, W, C] (2-D maps have D=1),
 * dense, C padded to a multiple of 16 (bf16) / 8 (fp32).
 */
#ifndef S3D_H_
#define S3D_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define S3D_OK                0
#define S3D_ERR_INVALID      -1   /* bad argument / unsupported shape            */
#define S3D_ERR_CUDA         -2   /* CUDA runtime / driver error (s3d_last_error) */
#define S3D_ERR_UNSUPPORTED  -3   /* device is not sm_100                         */

#define S3D_DTYPE_F32   0
#define S3D_DTYPE_BF16  1
/* Split bf16 pair ('bf16x3' precision mode): a value v is stored as hi = bf16(v) and lo = bf16(v - hi), v ~= hi + lo to
 * 2^-17 relative.  A tensor with C logical channels has 2*C bf16 channels per position, [hi(C) | lo(C)]; weights are
 * [rows][Cout][hi(Cin) | lo(Cin)].  The tensor-core engines compute x*w as hi*hi + lo*hi + hi*lo: three kind::f16 MMAs
 * per K step into the same fp32 TMEM accumulator (~2^-16 per product, i.e. fp32-grade results at the bf16 MMA rate / 3;
 * no split kernel, no partial sums through HBM).  Channel counts and strides of such tensors are in bf16 ELEMENTS of
 * the physical tensor; S3dConvParams.Cin / Cout stay LOGICAL. */
#define S3D_DTYPE_BF16X2 2

#define S3D_ACT_NONE     0
#define S3D_ACT_RELU     1
#define S3D_ACT_LEAKY    2   /* slope = act_param                       */
#define S3D_ACT_SIGMOID  3
#define S3D_ACT_TANH     4   /* act_param * tanh(x)                     */

#define S3D_MAX_TAPS 64

/* One convolution-like layer as an implicit GEMM:
 *   out[n*osN + (z*omz+ooz)*osD + (y*omy+ooy)*osH + (x*omx+oox)*osW + co*osC] =
 *     act( bias[co] + sum_{t<ntaps} sum_{ci<Cin}
 *            in[n, z*sz+dz[t], y*sy+dy[t], x*sx+dx[t], ci] * w[cls*ntaps+t, co, ci]  (+ residual) )
 * for (z,y,x) in the logical output grid oD x oH x oW; out-of-range input samples read 0.
 * Ordinary convs use n_classes=1, om*=1, oo*=0 and d*[t] = k - pad.  A stride-2
 * ConvTranspose3d(k4,p1) is n_classes=8 sub-pixel classes of 8 taps each; class bits
 * (cz,cy,cx) select oo* = (cz,cy,cx) with om*=2, and use tap rows cls*ntaps .. +ntaps. */
typedef struct S3dConvParams {
  int32_t N, iD, iH, iW, Cin;       /* input  [N,iD,iH,iW,Cin]                          */
  int32_t oD, oH, oW, Cout;         /* logical output grid per class, padded Cout (GEMM N) */
  int32_t sz, sy, sx;               /* input stride per output step (1 or 2)            */
  int32_t ntaps, n_classes;         /* taps per class; 1 or 8 classes                   */
  int8_t  dz[S3D_MAX_TAPS], dy[S3D_MAX_TAPS], dx[S3D_MAX_TAPS]; /* [n_classes*ntaps]   */
  int64_t osN, osD, osH, osW;       /* output element strides of n, z, y, x              */
  int64_t osC;                      /* output channel stride (1 = channels-last; h*w etc. = planar) */
  int64_t os_lo;                    /* out_dtype BF16X2: element offset from a channel's hi to its lo part (0 = Cout) */
  int32_t omz, omy, omx;            /* output coordinate multiplier                     */
  int32_t cout_store;               /* channels actually written (<= Cout)              */
  int32_t in_dtype, out_dtype;      /* S3D_DTYPE_*; weights have in_dtype.  BF16X2 in: bf16 / fp32 / BF16X2 out  */
  int32_t act;  float act_param;
  int32_t tw, th, td, tn;           /* M-tile box, powers of two, tw*th*td*tn == 128    */
  int32_t bn;                       /* GEMM N tile: multiple of 16, <= 256, divides Cout */
  /* Optional fused 1x1 projection (may be NULL): after the activation, channel `proj_channel` of every output
   * position is overwritten with proj_act(sum_{c<16} proj_w[c] * out[c]) (proj_w: 16 fp32 DEVICE values, zeros
   * beyond the real channels).  Needs Cout == 16 (one accumulator group).  Used to fold the decoder's final
   * 1x1x1 transposed conv + sigmoid into the last deconv layer.  Supported by s3d_conv_igemm's generic engine
   * and by s3d_conv_direct. */
  const float* proj_w;
  int32_t proj_channel, proj_act;
  /* Optional (may be NULL): weights of a stride-1 3x3x3 layer with Cout <= 64 pre-stacked for the plane-scatter
   * kernel (csrc/conv_scatter.cu), a DEVICE tensor [4][9][3*Cout][Cin] in the layer's dtype.  Rotation r = 0..2
   * (used for input plane p with p % 3 == r), in-plane tap kyx: row block s = 0..2 holds W[kz = (r+1-s) mod 3, kyx]
   * (the slice that carries input plane p into output plane z = p+1-kz, which accumulates in slot z % 3 == s).
   * Rotation 3 is rotation 0 with block 2 zeroed (p = 0: there is no output plane -1). */
  const void* w_nstack;
  /* Optional constant-region descriptor (dz_nref = 0: none), used by the plane-scatter kernel with bf16 operands and
   * ignored by every other engine.  The input is N = 2 * dz_nref volumes descending from a concat cost volume (in the
   * order of s3d_cost_volume_concat: [0, dz_nref) left-referenced, [dz_nref, N) right-referenced), and input plane z of
   * pixel column x is the same, bit for bit, for every z in [xr + dz_c, iD - 1 - dz_e], xr = x (left-referenced) or
   * iW - 1 - x (right-referenced).  The output then repeats along z on [xr + dz_c + 2, oD - 2 - dz_e]; the kernel computes
   * such a run once per column and stores it as copies (same results, fewer MMAs).  Not used with z-split columns.
   * dz_sched (may be NULL): int32 DEVICE table that pairs the columns for the CTA pairs of the kernel and balances their
   * planes, dz_pairs pairs: [dz_pairs + 1 offsets into the items][items x 2 column indices]; column index
   * (n * ceil(oH / 32) + y0 / 32) * ceil(oW / 8) + x0 / 8 for the 32 x 8 patch at (y0, x0), an index >= the column
   * count is an empty column.  Built by layers.py (dz_schedule); every column must appear exactly once.
   * dz_planes (may be NULL): int64 DEVICE counter, ADDED the number of input planes the kernel's CTAs marched. */
  int32_t dz_nref, dz_c, dz_e, dz_pairs;
  const int32_t* dz_sched;
  long long* dz_planes;
} S3dConvParams;

const char* s3d_version(void);
/* Human-readable text of the last error seen on this thread ("" if none). */
const char* s3d_last_error(void);
/* 0 if device `dev` is usable (compute capability 10.x), else a negative code. */
int s3d_device_check(int dev);
/* A/B switches of the launchers ("no_scatter", "scatter_no_pair", "scatter_generic", "scatter_tps3", "scatter_ring",
 * "scatter_res_transpose", "scatter_no_transpose", "no_corr_tc", "scatter_zsplit", "scatter_no_rm", "igemm_ts1", "igemm_one_cta", "scatter_one_cta", "no_conv_first_tc", "chamfer_sym", "chamfer_sym_r", "no_dz_skip"; all 0 by default = the shipped path).  They are
 * initialised ONCE from the environment variables S3D_<NAME> when the library is first used and are never read from
 * the environment on the launch path; s3d_set_knob overrides one at run time.  Process-wide, not thread-safe against
 * concurrent launches. */
int s3d_set_knob(const char* name, int value);
int s3d_get_knob(const char* name);

/* --- convolution engines ------------------------------------------------------------ */
/* tcgen05/TMEM/TMA implicit GEMM (bf16 -> kind::f16, fp32 -> kind::tf32), fp32 accumulate.
 * bias: fp32[Cout] or NULL; residual: NULL or a tensor addressed exactly like `out` (same dtype, strides, os_lo).
 * `residual` MAY alias `out` (in-place accumulation): every thread reads the residual of exactly the elements it
 * stores, before it stores them. */
int s3d_conv_igemm(const S3dConvParams* p, const void* in, const void* w, const float* bias,
                   const void* residual, void* out, void* stream);
/* Same contract, plain fp32 SIMT FMA loop (exact-fp32 validation mode; in/out dtype free). */
int s3d_conv_direct(const S3dConvParams* p, const void* in, const void* w, const float* bias,
                    const void* residual, void* out, void* stream);

/* Stride-1 3x3 2-D convolution, bf16, 32 / 64 input and output channels, in halo-once form (csrc/conv2d_halo.cu): the feature
 * encoder's conv1 / conv3 / conv4 / conv5.  in: [nimg,h,w,cin] channels-last; w: the layer's packed weights [9][cout][cin]
 * (tap order ky*3+kx); bias fp32[cout]; residual: NULL or bf16 addressed like out; out: bf16, element strides osN / osH / osW
 * of image / row / pixel (channels contiguous; a slice of a wider buffer is allowed); relu: 0 / 1.  Same arithmetic as
 * s3d_conv_igemm on the same operands (bf16 products, fp32 accumulate, one rounding of the output). */
int s3d_conv2d_halo(const void* in, const void* w, const float* bias, const void* residual, void* out, int nimg, int h, int wd,
                    int cin, int cout, int64_t osN, int64_t osH, int64_t osW, int relu, void* stream);

/* --- input staging ------------------------------------------------------------------ */
/* NCHW fp32 image [B,3,H,W] (+ optional fp32 disparity plane [B,H,W], scaled by disp_scale
 * into channel 3) -> channels-last [B,1,H,W,Cpad], zero padded channels. */
int s3d_pack_image(const float* img, const float* disp, float disp_scale, void* out,
                   int B, int H, int W, int Cpad, int out_dtype, void* stream);

/* Same, from decoded 8-bit images (the reference's inputs are PNG renders, README.md:73-74): img is uint8 HWC
 * [B,H,W,3]; channels 0-2 = img * img_scale (1/255 for [0,1] images), channel 3 = disp * disp_scale. */
int s3d_pack_image_u8(const uint8_t* img, const float* disp, float disp_scale, float img_scale, void* out,
                      int B, int H, int W, int Cpad, int out_dtype, void* stream);

/* First layer of the 2-D encoders, direct: Conv2d(cin, Cout, 3, stride 2, pad 1) + bias + activation straight from the
 * raw image -- img fp32 NCHW [B,3,H,W] (img_u8 = 0) or uint8 HWC [B,H,W,3] scaled by 1/255 (img_u8 = 1), plus for
 * cin = 4 the channel disp[B,H,W] * disp_scale -- to channels-last [B,1,oH,oW,cout_pad] (oH = (H-1)/2+1) of `dtype`.
 * w: the layer's packed weights [9][cout_pad][cin_pad] of `dtype` (only ci < cin is read); bias fp32[cout_pad] or NULL.
 * Same arithmetic as s3d_pack_image + s3d_conv_igemm (inputs/weights rounded to `dtype`, fp32 accumulate).
 * dtype BF16X2: w is [9][cout_pad][hi(cin_pad) | lo(cin_pad)], the image is not rounded, out is [.., hi | lo]. */
int s3d_conv_first(const void* img, int img_u8, const float* disp, float disp_scale, const void* w, const float* bias,
                   void* out, int B, int H, int W, int cin, int cin_pad, int cout_pad, int dtype, int act,
                   float act_param, void* stream);

/* --- cost volume / disparity (rows V, S) ---------------------------------------------- */
/* Cost volume + first aggregation layer fused (csrc/conv_scatter_concat.cu): the stride-1 3x3x3 conv `p` (N = 2B volumes,
 * iD = D, Cin = 2C, Cout <= 64, w_nstack set) over the concat volume of s3d_cost_volume_concat, WITHOUT materialising it.
 * feat: channels-last feature maps [2B, h, feat_pitch, C] whose real pixels start at column feat_pad and whose margins
 * (>= D-1 pixels on both sides) are ZERO; left images first.  Bit-identical to s3d_cost_volume_concat + s3d_conv_igemm. */
int s3d_conv_concat_volume(const S3dConvParams* p, const void* feat, int feat_pitch, int feat_pad, const float* bias,
                           void* out, void* stream);
/* The same layer in REFERENCE-ONCE form (bf16 only; Cout = 64, ReLU, dense output, CTA pairs).  The reference half of the
 * concat volume is the same feature map on every disparity plane, so its contribution R = ref (*) sum_kz W[kz, :, ref ch]
 * is computed once per column and added to every plane by the epilogue; the planes run the tensor cores on the TARGET half
 * only (half the MMA work of the layer) and the two border planes get ref (*) -W[kz=0] / -W[kz=2] added.
 * w_refonce: bf16 DEVICE tensor [3][9][Cout][C] = [sum_kz W[kz] | -W[kz=0] | -W[kz=2]] over the reference channels
 * (in-plane tap order ky*3+kx).  Same result as s3d_conv_concat_volume up to bf16 rounding of the summed weights and
 * the fp32 accumulation order (NOT bit-identical). */
int s3d_conv_concat_volume_ro(const S3dConvParams* p, const void* feat, int feat_pitch, int feat_pad, const void* w_refonce,
                              const float* bias, void* out, void* stream);
/* The same layer in SHEARED form (bf16, Cout = 64, ReLU): in the coordinate u = x -/+ d the target half of the volume is
 * the same feature map on every plane, so the layer is a few 2-D convolutions (maps, computed by s3d_conv_igemm from
 * weight sets packed by the host: layers.py, PackedConv.gonce_convs) and this streaming pass, which adds
 *   bias + Psum[y,x] + G[y,u]  (+ the dz = -1 / +1 maps on the two border planes, + the edge-column maps at x = w-1 / 0),
 * applies the ReLU and writes out bf16 [2B,D,h,w,64] (left-referenced volumes first).  maps_l / maps_r: fp32
 * [B,h,map_w = w+4,384] from the left / right images, channels [Psum | Pm | Pp | G | Hm | Hp], map column j <-> u = j-2;
 * a volume takes its reference maps from its own image and its target maps from the other one.  edge_l / edge_r: fp32
 * [B,h,D,256] = [Ge | Gem | Gep | unused].  out_dtype BF16X2 ('bf16x3'): out is [2B,D,h,w, hi(64) | lo(64)].  Not bit-identical to s3d_conv_concat_volume (weights summed before the bf16 rounding,
 * different summation order). */
int s3d_concat_gonce_assemble(const float* maps_l, const float* maps_r, const float* edge_l, const float* edge_r,
                              const float* bias, void* out, int B, int D, int h, int w, int map_w, int out_dtype, void* stream);
/* The map convolutions of that form on their own engine (csrc/map_conv.cu): in bf16 [nimg,h,in_w,32] (feature rows with their
 * zero margins), w bf16 [3*ntx][cout][32] (taps dy = -1..1 major, ex = 0..ntx-1 minor; ntx = 3 or 5; cout a multiple of 128),
 * out fp32 [nimg,h,ow,cout]:  out[n,y,j,co] = sum_{dy,ex,ci} in[n, y+dy, j+off+ex, ci] * w[(dy+1)*ntx+ex, co, ci]  (zero outside
 * the input).  One TMA box per output tile (patch + halo), every tap a descriptor offset into it.  dtype BF16X2: in is
 * [nimg,h,in_w, hi(32) | lo(32)], w is [3*ntx][cout][hi(32) | lo(32)], three MMAs per product (fp32-grade maps). */
int s3d_map_conv(const void* in, const void* w, float* out, int nimg, int h, int in_w, int ow, int off, int ntx, int cout,
                 int dtype, void* stream);
/* feat: [2B,1,h,w,C] (left maps first, then right).  vol: [2B,D,h,w,2C]; entries [0,B) are
 * left-referenced (target sampled at x-d), [B,2B) right-referenced (target at x+d).
 * dtype BF16X2: feat [.., hi(C) | lo(C)] -> vol [.., hi(2C) | lo(2C)] (C logical channels). */
int s3d_cost_volume_concat(const void* feat, void* vol, int B, int h, int w, int C, int D,
                           int dtype, void* stream);
/* cost: fp32 [N,D,h,w] -> disp fp32 [N,h,w] = sum_d d*softmax_d(sign*cost).  sign=-1: soft-argmin. */
int s3d_soft_argmin(const float* cost, float* disp, int N, int D, int h, int w, float sign,
                    void* stream);

/* --- disparity uncertainty ------------------------------------------------------------------------------------------------
 * The four soft-argmin calls below (tap_gather, cls, conv_cls, corr) take disp_std_q fp32 [N,h,w] right after disp; NULL means
 * "do not compute it".  When it is set they write the same disp bit for bit, and into disp_std_q the standard deviation of
 * each pixel's soft-argmin distribution, in planes: with p_d = softmax_d(sign * cost_d) the weights whose mean is disp_q,
 *   sigma_q = sqrt(sum_d p_d (d - disp_q)^2)     (fp32, >= 0; NaN where disp_q is not finite).
 * The corr kernels include the cost-0 planes outside the image, as for the mean.  Accuracy: |sigma_q - sigma_ref| <= 1e-4 *
 * (1 + sigma_ref) against sigma_ref computed in fp64 from the same costs, also for sharp peaks at large d (the online kernels
 * accumulate the moments about the running arg-max plane, the corr kernels take a second pass about the mean). */

/* Cout=1 3x3x3 classifier conv + soft-argmin from per-tap planes.  taps: fp32, line-planar [N,D,h,tap_stride,w] with
 * taps[n,z,y,(kz*3+ky)*3+kx,x] = W[kz,ky,kx,:] . in[n,z,y,x,:] (a pointwise GEMM done by s3d_conv_igemm with osC=w);
 * cost[z,y,x] = sum_t taps[z+kz-1, y+ky-1, x+kx-1, t] (zero outside), disp = sum_z z*softmax_z(sign*cost).
 * cost_out may be NULL (debug: fp32 [N,D,h,w]). */
int s3d_tap_gather_soft_argmin(const float* taps, float* disp, float* disp_std_q, float* cost_out, int N, int D, int h, int w,
                               int tap_stride, float sign, void* stream);
/* The same classifier + soft-argmin in ONE pass over the aggregated volume, no per-tap tensor (csrc/cls_fused.cu):
 * x: bf16 channels-last [N,D,h,w,C], C in {16,32,64}; w_taps: bf16 [32][C], row t = (kz*3+ky)*3+kx holds W[kz,ky,kx,:]
 * (rows 27..31 zero) -- the weight tensor of the pointwise layer above; disp: fp32 [N,h,w]. */
int s3d_cls_soft_argmin(const void* x, const void* w_taps, float* disp, float* disp_std_q, int N, int D, int h, int w, int C,
                        float sign, void* stream);
/* Last aggregation layer + classifier + soft-argmin WITHOUT the layer's output volume (csrc/conv_scatter_cls.cu): `p` is the
 * bf16 stride-1 3x3x3 64 -> 64 ReLU layer (w_nstack set) over in [N,D,h,w,64]; its output Y is projected on the 27 classifier
 * taps w_taps (bf16 [32][64], as for s3d_cls_soft_argmin) on the tensor core, scattered into per-CTA partial cost planes in
 * `workspace` (s3d_conv_cls_workspace_bytes(N, D, h, w) bytes, fp32) and a second kernel adds the partial sums in a fixed order
 * and runs the soft-argmin: disp fp32 [N,h,w].  Same arithmetic as s3d_conv_igemm + s3d_cls_soft_argmin (Y rounded to bf16 as
 * the stored tensor would be) up to the fp32 summation order of the 27 taps.  Needs N * ceil(h/32) * ceil(w/8) >= 2. */
int64_t s3d_conv_cls_workspace_bytes(int N, int D, int h, int w);
int s3d_conv_cls_soft_argmin(const S3dConvParams* p, const void* in, const float* bias, const void* w_taps, void* workspace,
                             float* disp, float* disp_std_q, float sign, void* stream);
/* Fused correlation + soft-argmax; the [2B,D,h,w] cost is never materialised.
 * feat: [2B,1,h,w,C] with C the PADDED channel count (row pitch); cost = (1/c_real) * sum_c ref*tgt over the real
 * channels (padded channels must be zero; c_real = 0 means C).
 * disp: fp32 [2B,h,w]; cost_out may be NULL (debug: fp32 [2B,D,h,w]). */
int s3d_corr_soft_argmin(const void* feat, float* disp, float* disp_std_q, float* cost_out, int B, int h, int w,
                         int C, int c_real, int D, int dtype, void* stream);
/* disp_q fp32 [N,h,w] (1/4-res units) -> fp32 [N,H,W] = bilinear(scale*disp_q), align_corners=False. */
int s3d_upsample_disp(const float* disp_q, float* disp, int N, int h, int w, int H, int W,
                      float scale, void* stream);
/* s3d_upsample_disp + per-pixel evaluation, in one launch.  disp_q fp32 [2B,h,w] (left-referenced first), disp fp32 [2B,H,W]
 * (written bit-identically to s3d_upsample_disp).  Three optional groups, each on when its lead pointer is set: gt comes with
 * disp_stats, lr_mask with lr_stats, disp_std_q with disp_std (both or neither).  A call with no group on is rejected: the
 * plain upsampling is s3d_upsample_disp.  Every stats tensor is ACCUMULATED (the caller zeroes it).  thresholds: T <= 8 fp32
 * HOST values; T sets the row length of every stats tensor, also when gt == NULL (then lr_stats and unc_stats get column 0
 * only).
 *
 * GT (gt, disp_stats): gt fp32 [B,2,H,W] (view 0 = left-referenced, 1 = right-referenced), disp_stats int64 [B,2,2+T]:
 *   [n_valid, sum_valid q(|disp - gt|), count_valid(|disp - gt| > thresholds[t]) for t < T]
 * valid: gt finite and 0 <= gt < max_gt.  q(e) = round-half-even(e * 65536) of the fp32 error (fixed point, 2^-16 px).
 * Range: q < 2^26 per pixel while disparities are below 1024 px, so one image's sum stays below 2^50 for H*W <= 2^24 and
 * int64 holds the sums of more than 2^12 such images.  Integer counters, one atomic per counter per block and no block
 * spans two images: the stats do not depend on the launch order, batch split or number of GPUs.
 *
 * LR check (lr_mask, lr_stats): the left-right consistency check of the two views.  With D0 / D1 the
 * left- / right-referenced maps of a sample and d = Dv[y,x] finite, k = round-half-even(d), xo = x - k (view 0) or x + k
 * (view 1): the pixel is KEPT iff 0 <= xo < W and |d - D(1-v)[y,xo]| <= lr_thresh (fp32 subtraction, one rounding; a NaN
 * on the other side is not kept).  A non-finite d is not kept; |d| >= W + 1 is out of range.  lr_mask uint8 [B,2,H,W]
 * (1 = kept).  lr_stats int64 [B,2,3+T]:
 *   [n_kept, n_valid_kept, sum_{valid & kept} q(|disp - gt|), count_{valid & kept}(|disp - gt| > thresholds[t]) for t < T]
 * lr_thresh must be >= 0.
 *
 * Uncertainty (disp_std_q, disp_std; unc_thresh, K, unc_stats): disp_std_q fp32 [2B,h,w] (from a soft-argmin call) ->
 * disp_std fp32 [B,2,H,W] (view 0 = left-referenced) = bilinear(scale * disp_std_q), bit-identical to
 * s3d_upsample_disp(disp_std_q, scale) of the image where both take the same (16-byte or scalar) path: W % 4 == 0 and 16-byte
 * aligned outputs, or neither.  unc_thresh: K <= 4 HOST values in input pixels, finite and >= 0 (K > 0 needs disp_std_q).
 * unc_stats int64 [B,2,K,3+T]: per view and threshold k, over the CONFIDENT pixels (disp_std <= unc_thresh[k] in fp32; a
 * non-finite disp_std never is)
 *   [n_conf, n_valid_conf, sum_{valid & conf} q(|disp - gt|), count_{valid & conf}(|disp - gt| > thresholds[t]) for t < T]
 * (the range argument above holds for these sums, which run over fewer pixels). */
int s3d_upsample_disp_eval(const float* disp_q, float* disp, int B, int h, int w, int H, int W, float scale,
                           const float* gt, const float* thresholds, int T, float max_gt, long long* disp_stats,
                           uint8_t* lr_mask, float lr_thresh, long long* lr_stats,
                           const float* disp_std_q, float* disp_std, const float* unc_thresh, int K, long long* unc_stats,
                           void* stream);

/* --- decoder glue (rows X, D, F, M) ---------------------------------------------------- */
/* adaptive average pool [N,1,H,W,C] -> [N,1,L,L,C], then the NCHW .view(N,C*L*L/8,2,2,2)
 * re-indexing of the oracle, written channels-last as [N,2,2,2,C*L*L/8].
 * (This and the next two accept dtype BF16X2: split tensors in and out, C / 64 / Cpad = LOGICAL channels.) */
int s3d_latent_to_vox(const void* x, void* out, int N, int H, int W, int C, int L, int dtype,
                      void* stream);
/* Generic adaptive average pool, channels-last [N,1,H,W,C] -> [N,1,L,L,C]. */
int s3d_avg_pool(const void* x, void* out, int N, int H, int W, int C, int L, int dtype,
                 void* stream);
/* Depth-to-space after a transposed conv computed as a blocked stride-1 conv: in [N,d,h,w,64] with channel
 * (class, c) = (cz*4 + cy*2 + cx)*8 + c  ->  out [N,2d,2h,2w,Cpad], out[n, 2z+cz, 2y+cy, 2x+cx, c] for c < 8.
 * If Cpad > 8: channel 8 = proj_act(sum_c proj_w[c] * feature c) (proj_w: 8 fp32 DEVICE values; NULL -> 0), channels
 * 9.. = 0 -- the decoder's final 1x1x1 transposed conv + sigmoid. */
int s3d_depth_to_space(const void* in, void* out, const float* proj_w, int proj_act, int N, int d, int h, int w,
                       int Cpad, int dtype, void* stream);
/* Operand split of the 'tf32x3' precision mode: hi = x with the low 13 mantissa bits cleared (exactly representable
 * in TF32), lo = x - hi (exact).  conv(x, w) ~= conv(hi, w_hi) + conv(lo, w_hi) + conv(hi, w_lo) on kind::tf32 tensor
 * cores with fp32 accumulation reproduces fp32 to ~1e-6 relative.  n (elements) must be a multiple of 4. */
int s3d_split_tf32(const float* x, float* hi, float* lo, int64_t n, void* stream);
/* fp32 [npix, C] <-> split bf16 pairs [npix, hi(C) | lo(C)] (S3D_DTYPE_BF16X2): hi = bf16(x), lo = bf16(x - hi);
 * unsplit returns hi + lo.  Hand-off between 'bf16x3' tensors and the kernels that take fp32. */
int s3d_split_bf16(const float* x, void* out, int64_t npix, int C, void* stream);
int s3d_unsplit_bf16(const void* x, float* out, int64_t npix, int C, void* stream);
/* Context-aware fusion epilogue + IoU.  score, vol: [V*B, 32^3] planes with element strides
 * score_stride / vol_stride (view-major); fused[b,v] = clamp(sum_v softmax_v(score)*vol, 0, 1).
 * gt (uint8 [B,32^3]) and iou (int64 [B,T,2] = intersection, union) may be NULL.
 * dtype BF16X2: score_lo / vol_lo are the element offsets from a value's hi part to its lo part (0 for other dtypes). */
int s3d_fuse_views(const void* score, int64_t score_stride, const void* vol, int64_t vol_stride,
                   int dtype, float* fused, int B, int V, int nvox, const uint8_t* gt,
                   const float* thresholds, int T, long long* iou, int64_t score_lo, int64_t vol_lo, void* stream);
/* Voxel-surface metrics of predicted occupancy against GT occupancy: exact voxel-face Chamfer and F-score counters.
 * fused fp32 [B,n,n,n], gt uint8 [B,n,n,n]; 1 <= n <= 64.  Occupied: fused >= thresholds[t] in fp32 (NaN is empty, as for
 * the IoU of s3d_fuse_views), gt != 0; outside the grid is empty.  Surface = the centres of the faces between an occupied and
 * an empty voxel, in doubled integer coordinates (voxel centre 2i+1, a face at an even coordinate 0..2n on its axis), so each
 * is a site of the (2n+1)^3 lattice.  s = squared distance in doubled units to the nearest point of the other surface, an
 * integer <= 3 (2n)^2: exact, no ties problem.  stats int64 [B,T,2,3+F] is ADDED to (caller zeroes); per sample, t and
 * direction (0: predicted -> GT, 1: GT -> predicted)
 *   [ n_pts, sum s, sum q(sqrt_rn(s)), count(s < kbound[f]) for f < F ]
 * q(x) = round-half-even(x * 2^32) (exact product), sqrt_rn = the correctly rounded fp32 square root of (float)s.  When the
 * other surface is empty only n_pts is counted.  kbound: F <= 8 HOST ints in [0, 3 (2n)^2 + 1]; an F-score threshold tau in
 * unit-cube units (the grid spans a unit cube) is kbound = min(ceil((2n tau)^2), 3 (2n)^2 + 1).  thresholds: T <= 8 HOST
 * values.  workspace: >= s3d_voxel_surface_workspace_bytes(B, T, n) bytes, 8-byte aligned (one uint16 distance grid per
 * sample and surface).  Two kernels: the in-plane passes of the distance transform, then the third pass at the query sites
 * fused with the counters (one atomic per counter per block, no block spanning two slices: the sums do not depend on the
 * launch order or the batch split). */
int64_t s3d_voxel_surface_workspace_bytes(int B, int T, int n);
int s3d_voxel_surface_eval(const float* fused, const uint8_t* gt, int B, int n, const float* thresholds, int T,
                           const int* kbound, int F, long long* stats, void* workspace, int64_t workspace_bytes, void* stream);
/* Triangle mesh of an occupancy grid: marching cubes at iso-level t, closed and consistently oriented.
 * vol fp32 [B,n,n,n] (sample b is vol[b,k,j,i], x along i), 1 <= n <= 64, padded with one layer of 0 on every side; the
 * padded field is clamped (NaN -> 0, then min(max(v, 0), 1)) and a corner is inside when v >= t; t finite, 0 < t <= 1, so
 * the padding is outside and every mesh is closed.  Cells: the (n+1)^3 cubes of the padded lattice, case table
 * csrc/mc_table.cuh (generated with its rule by stereo_3d_reconstruction_b200/mc_table.py; faces with inside corners on a
 * diagonal separate them).  One vertex per crossing lattice edge, id = its rank in (padded corner linear index, axis x < y
 * < z) order; with a, b the values at its lower corner p and at p + e_axis, s = (t - a) / (b - a) and the coordinate along
 * the axis is ((float)p + 0.5f + s) / n, the other two (q + 0.5f) / n (fp32, round to nearest, left to right): the grid
 * spans the unit cube.  Faces: 0-based per-sample vertex ids, in cell linear order then table order, each oriented so that
 * (v1 - v0) x (v2 - v0) points from occupied to empty.  verts fp32 [B,max_verts,3], faces int32 [B,max_faces,3], counts
 * int32 [B,2] = (n_verts, n_faces); rows past the counts are not written.  max_verts / max_faces must be at least the
 * worst case of s3d_voxel_mesh_bounds.  One kernel, one block per sample, no atomics: the output is deterministic. */
int s3d_voxel_mesh_bounds(int n, int* max_verts, int* max_faces);    /* 3 (n+1)(n+2)^2 and 5 (n+1)^3 */
int s3d_voxel_mesh(const float* vol, int B, int n, float t, float* verts, int max_verts, int* faces, int max_faces,
                   int* counts, void* stream);
/* Threshold-free occupancy evaluation: per-sample probability histograms split by GT label, and BCE / Brier sums, from which
 * the IoU at every threshold k / K, the precision-recall curve and the calibration follow.  fused fp32 [B,nvox], gt uint8
 * [B,nvox], 1 <= nvox <= 2^24, 0 <= B; K a power of two in [2, 1024].  Per voxel: v = fused clamped as for s3d_voxel_mesh
 * (NaN -> 0, then min(max(v, 0), 1)), g = (gt != 0), bin k = min(floor(v * K), K - 1) in fp32 (v * K is exact, so bin >= k
 * exactly when v >= k / K), q(x) = round-half-even(x * 2^20) in fp64.  Per sample b (written, not added; no zeroing needed):
 *   hist int64 [B,3,K]: row 0 the voxels with g = 0 in bin k, row 1 those with g = 1, row 2 sum q(v) over bin k (both);
 *   loss int64 [B,2]:   sum q(bce), bce = -max(log(v), -100) if g else -max(log(1 - v), -100) (PyTorch's BCELoss clamp;
 *                       1 - v and log in fp64 on the fp32 v), then sum q((v - g)^2) (fp64).
 * Overflow: a voxel adds at most 100 * 2^20 to a counter, so at n = 32 (32768 voxels) a sample's counters stay below 2^42
 * and an int64 sum over samples holds more than 2M samples even if every voxel hits the BCE clamp.  One kernel, one cluster
 * of blocks per sample reducing through distributed shared memory: integer sums, no global atomics, deterministic. */
int s3d_occupancy_curves(const float* fused, const uint8_t* gt, int B, int nvox, int K, int64_t* hist, int64_t* loss,
                         void* stream);

/* --- Chamfer distance (row C; replaces extensions/chamfer_dist, README.md:62-65) ------- */
/* xyz1 fp32 [B,N,3], xyz2 fp32 [B,M,3] -> dist1 fp32 [B,N], idx1 int32 [B,N] (nearest in
 * xyz2), dist2 fp32 [B,M], idx2 int32 [B,M] (nearest in xyz1).  Squared L2, computed as
 * ((x1-x2)^2 + (y1-y2)^2) + (z1-z2)^2 with round-to-nearest mul/add and no FMA contraction;
 * ties resolve to the lowest index. */
int s3d_chamfer_forward(const float* xyz1, const float* xyz2, float* dist1, int32_t* idx1,
                        float* dist2, int32_t* idx2, int B, int N, int M, void* stream);
/* The same forward with a caller-owned device workspace (8-byte aligned, s3d_chamfer_workspace_bytes(B, N, M) bytes; that
 * is 0 when the problem is too small for it).  With the workspace every point pair is evaluated ONCE for both directions
 * (d(i, j) is the same fp32 number either way round): row minima in registers, column minima merged through 64-bit
 * atomicMin keys in the workspace, indices recovered by rescanning one 32- / 256-point chunk.  Results are bit-identical
 * to s3d_chamfer_forward (which is this call with workspace = NULL: one search per direction). */
int64_t s3d_chamfer_workspace_bytes(int B, int N, int M);
int s3d_chamfer_forward_ws(const float* xyz1, const float* xyz2, float* dist1, int32_t* idx1,
                           float* dist2, int32_t* idx2, int B, int N, int M, void* workspace,
                           int64_t workspace_bytes, void* stream);
/* Chamfer search of s3d_chamfer_forward_ws (same dist / idx outputs, bit for bit) + per-sample point-cloud metrics.
 * xyz1 = predicted [B,N,3], xyz2 = GT [B,M,3].  stats int64 [B,2,3+T] is ADDED to (caller zeroes):
 *   direction 0 = xyz1 -> xyz2 (dist1), direction 1 = xyz2 -> xyz1 (dist2); per direction
 *   [ sum q(d), sum q(sqrt_rn(d)), n_out, count(sqrt_rn(d) < tau_t) for t < T ]   over the points with d in range.
 * d is the squared distance written to dist1 / dist2.  In range: d finite and d < 2^8; every other point (a NaN point gets
 * d = +inf) counts in n_out only.  q(x) = round-half-even(x * 2^32) as int64 (the product is exact in fp32); sqrt_rn is the
 * correctly rounded fp32 square root.  A point counts at tau_t when sqrt_rn(d) < tau_t in fp32, strictly: the thresholds
 * are Euclidean distances in the points' units.  tau: T <= 8 HOST values, each finite and > 0.  N, M < 2^22, so a
 * (sample, direction) sum of q < 2^40 stays inside int64.  The counters are integers summed with one atomic per counter
 * per block, no block spanning two (sample, direction) slices: they do not depend on the launch order or batch split.
 * One kernel after the search, over the distances it has just written. */
int s3d_chamfer_eval(const float* xyz1, const float* xyz2, float* dist1, int32_t* idx1, float* dist2, int32_t* idx2,
                     int B, int N, int M, const float* tau, int T, long long* stats,
                     void* workspace, int64_t workspace_bytes, void* stream);

/* Measurement aid (bench.py): a launch of independent fp32 FMA chains that is bound by the FMA issue rate only;
 * *fma_count (HOST) receives the number of thread-level FMAs the launch executes.  Timed with CUDA events it gives the
 * MEASURED fp32 SIMT peak the Chamfer kernel's pair rate is quoted against.  sink: any device float. */
int s3d_fma_probe(float* sink, int iters, int64_t* fma_count, void* stream);

#ifdef __cplusplus
}
#endif
#endif  /* S3D_H_ */
