// Shared host/device helpers for libs3d_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/s3d.h"

namespace s3d {

void set_error(const char* fmt, ...);

#define S3D_CHECK_ARG(cond, ...)                         \
  do {                                                   \
    if (!(cond)) {                                       \
      s3d::set_error(__VA_ARGS__);                       \
      return S3D_ERR_INVALID;                            \
    }                                                    \
  } while (0)

#define S3D_CUDA(expr)                                                              \
  do {                                                                              \
    cudaError_t _e = (expr);                                                        \
    if (_e != cudaSuccess) {                                                        \
      s3d::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return S3D_ERR_CUDA;                                                          \
    }                                                                               \
  } while (0)

#define S3D_LAUNCH_CHECK() S3D_CUDA(cudaGetLastError())

int num_sms();   // SM count of the current device (cached)

// A/B switches of the launchers.  Read ONCE from the S3D_* environment variables (first use), never per launch;
// s3d_set_knob() overrides them at run time (tests, A/B scripts).  All default to 0 = the shipped path.
struct Knobs {
  int no_scatter;             // S3D_NO_SCATTER: 3x3x3 layers take the generic per-tap engine instead of conv_scatter
  int scatter_tps3;           // S3D_SCATTER_TPS3: 3-tap weight stages where 9-tap ones are the default
  int scatter_no_pair;        // S3D_SCATTER_NO_PAIR: single-CTA kernels instead of cta_group::2 pairs
  int scatter_ring;           // S3D_SCATTER_RING=n: force the plane ring depth (0 = automatic)
  int scatter_res_transpose;  // S3D_SCATTER_RES_TRANSPOSE: coalesced residual group loads + second shuffle transpose
  int scatter_no_transpose;   // S3D_SCATTER_NO_TRANSPOSE: per-pixel stores instead of the transposed epilogue
  int scatter_generic;        // S3D_SCATTER_GENERIC: all-in-one kernel instead of the lean per-shape ones
  int no_corr_tc;             // S3D_NO_CORR_TC: SIMT correlation kernel even where the tensor-core one applies
  int scatter_zsplit;         // S3D_SCATTER_ZSPLIT=n: force n z-chunks per column (-1: never split; 0 = automatic)
  int igemm_ts1;              // S3D_IGEMM_TS1: one tap per pipeline stage in the generic engine (conv_igemm.cu)
  int igemm_one_cta;          // S3D_IGEMM_ONE_CTA: one CTA per SM in the generic engine even where two fit
  int scatter_one_cta;        // S3D_SCATTER_ONE_CTA: one CTA per SM for the narrow plane-scatter layers too
  int no_conv_first_tc;       // S3D_NO_CONV_FIRST_TC: SIMT first layers (conv_first.cu) instead of the tensor-core ones
  int chamfer_sym;            // S3D_CHAMFER_SYM: 1 = symmetric one-pass Chamfer kernel at every size (given a workspace), -1 = never (0: when it fills the chip)
  int chamfer_sym_r;          // S3D_CHAMFER_SYM_R: resident points per lane of the symmetric Chamfer kernel, 4 or 8 (0: automatic)
  int scatter_no_rm;          // S3D_SCATTER_NO_RM: residual added by the epilogue threads instead of an identity tap on the tensor core
  int no_dz_skip;             // S3D_NO_DZ_SKIP: the plane-scatter kernel ignores S3dConvParams' constant-region descriptor (dz_nref)
};
Knobs& knobs();

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

// Thresholds of the in-kernel evaluation counters (IoU in fuse_views, bad-pixel rates in upsample_disp_eval), passed by value.
namespace {
constexpr int kMaxThresh = 8;
struct Thresh { float t[kMaxThresh]; };
// Distance-histogram edges of the point / surface evaluations (s3d_chamfer_eval_hist, s3d_voxel_surface_eval_hist), passed
// by value: 4 KB of kernel parameters, copied to shared memory by each block.
constexpr int kMaxBins = 1024;
}  // namespace

template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// NaN-propagating max / min (FMNMX.NAN, one instruction like fmaxf): fmaxf(NaN, 0) is 0, which would scrub a NaN
// accumulator (corrupt checkpoint, inf - inf) out of every tensor-core layer while PyTorch and the fp32 engine keep it.
__device__ __forceinline__ float fmax_nan(float a, float b) { float d; asm("max.NaN.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(b)); return d; }
__device__ __forceinline__ float fmin_nan(float a, float b) { float d; asm("min.NaN.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(b)); return d; }

__device__ __forceinline__ float apply_act(float v, int act, float a) {
  switch (act) {
    case S3D_ACT_RELU:    return fmax_nan(v, 0.f);
    case S3D_ACT_LEAKY:   return v > 0.f ? v : v * a;
    case S3D_ACT_SIGMOID: return 1.f / (1.f + expf(-v));
    case S3D_ACT_TANH:    return a * tanhf(v);
    default:              return v;
  }
}

// Out-of-line copy for epilogues that must stay small: 16 calls instead of 16 inlined switch bodies.
static __device__ __noinline__ float apply_act_slow(float v, int act, float a) { return apply_act(v, act, a); }

// 8-bit colour of an fp32 image channel (s3d_disp_cloud, s3d_disp_wls): rint(clamp(c, 0, 1) * 255), NaN -> 0.
__device__ __forceinline__ unsigned colour_f32(float c) {
  const float u = fminf(fmaxf(c, 0.f), 1.f);                             // NaN -> 0 (fmaxf)
  return (unsigned)__float2int_rn(__fmul_rn(u, 255.f));                  // round half to even
}

// sigma_q = sqrt(var) of a soft-argmin distribution; a non-finite mean gives NaN.
__device__ __forceinline__ float soft_std(float var, float mu) {
  return isfinite(mu) ? sqrtf(fmaxf(var, 0.f)) : __int_as_float(0x7fffffff);
}

// Spread of the soft-argmin distribution for the online (max, sum e, sum e*d) marches: the first and second moments of the
// weights about the running arg-max plane r, s1 = sum e (d - r), s2 = sum e (d - r)^2, shifted when the max moves.  About 0,
// sum e d^2 / sum e - mu^2 cancels in fp32 when mu is large and the peak sharp (D = 128, peak at 120, sigma 0.05: wrong in the
// second digit).  About r it cannot: p_r >= 1/D, so s2 / s <= (D + 1) var.
struct SoftSpread {
  float s1 = 0.f, s2 = 0.f;
  int r = 0;
  // the max moved to plane z and s1, s2 and s (the sum of the weights) were rescaled to it
  __device__ __forceinline__ void move(int z, float s) {
    const float dl = (float)(r - z);
    s2 = fmaf(dl * dl, s, fmaf(2.f * dl, s1, s2));
    s1 = fmaf(dl, s, s1);
    r = z;
  }
  __device__ __forceinline__ void scale(float sc) { s1 *= sc;  s2 *= sc; }
  __device__ __forceinline__ void add(float e, int z) {
    const float dz = (float)(z - r);
    s1 = fmaf(e, dz, s1);
    s2 = fmaf(e * dz, dz, s2);
  }
  __device__ __forceinline__ float sigma(float mu, float s) const {
    const float a = s1 / s;
    return soft_std(s2 / s - a * a, mu);
  }
};

}  // namespace s3d
