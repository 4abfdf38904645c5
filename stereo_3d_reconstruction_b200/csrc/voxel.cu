// Glue kernels around the conv engine: input staging, latent re-indexing, pooling, and the
// context-aware fusion epilogue fused with the IoU statistics (rows X, F, M).  All bandwidth-bound
// elementwise / small-reduction kernels.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>
#include "common.cuh"

namespace s3d {

// ---- error slot / device info (library-wide) -------------------------------------------------
static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
int num_sms() {
  // per call: one process may drive several devices (cudaDeviceGetAttribute is a cached host-side lookup)
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
    n = 148;
  return n;
}

namespace {
struct KnobName { const char* name; const char* env; int Knobs::*field; };
const KnobName kKnobNames[] = {
    {"no_scatter", "S3D_NO_SCATTER", &Knobs::no_scatter},
    {"scatter_tps3", "S3D_SCATTER_TPS3", &Knobs::scatter_tps3},
    {"scatter_no_pair", "S3D_SCATTER_NO_PAIR", &Knobs::scatter_no_pair},
    {"scatter_ring", "S3D_SCATTER_RING", &Knobs::scatter_ring},
    {"scatter_res_transpose", "S3D_SCATTER_RES_TRANSPOSE", &Knobs::scatter_res_transpose},
    {"scatter_no_transpose", "S3D_SCATTER_NO_TRANSPOSE", &Knobs::scatter_no_transpose},
    {"scatter_generic", "S3D_SCATTER_GENERIC", &Knobs::scatter_generic},
    {"no_corr_tc", "S3D_NO_CORR_TC", &Knobs::no_corr_tc},
    {"scatter_zsplit", "S3D_SCATTER_ZSPLIT", &Knobs::scatter_zsplit},
    {"scatter_no_rm", "S3D_SCATTER_NO_RM", &Knobs::scatter_no_rm},
    {"igemm_ts1", "S3D_IGEMM_TS1", &Knobs::igemm_ts1},
    {"no_conv_first_tc", "S3D_NO_CONV_FIRST_TC", &Knobs::no_conv_first_tc},
    {"scatter_one_cta", "S3D_SCATTER_ONE_CTA", &Knobs::scatter_one_cta},
    {"igemm_one_cta", "S3D_IGEMM_ONE_CTA", &Knobs::igemm_one_cta},
    {"chamfer_sym", "S3D_CHAMFER_SYM", &Knobs::chamfer_sym},
    {"chamfer_sym_r", "S3D_CHAMFER_SYM_R", &Knobs::chamfer_sym_r},
    {"no_dz_skip", "S3D_NO_DZ_SKIP", &Knobs::no_dz_skip},
};
}  // namespace

Knobs& knobs() {
  static Knobs k = [] {
    Knobs v;
    memset(&v, 0, sizeof(v));
    for (const KnobName& n : kKnobNames)
      if (const char* e = getenv(n.env)) { const int x = atoi(e); v.*(n.field) = x != 0 ? x : 1; }   // "S3D_X=" or "=yes" -> 1 (negative values are kept)
    return v;
  }();
  return k;
}

namespace {

template <typename T>
__global__ void pack_image_kernel(const float* __restrict__ img, const float* __restrict__ disp, float disp_scale,
                                  T* __restrict__ out, int B, int H, int W, int Cpad) {
  const int64_t plane = (int64_t)H * W, total = plane * B;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = i / plane, pix = i % plane;
    const float* ip = img + b * 3 * plane + pix;
    const float c0 = ip[0], c1 = ip[plane], c2 = ip[2 * plane], c3 = disp ? disp[i] * disp_scale : 0.f;
    T* o = out + i * Cpad;
    if (sizeof(T) == 2 && (Cpad & 7) == 0) {
      // 16-byte stores: channels 0-3 real, the rest zero
      uint4 v0 = make_uint4(0, 0, 0, 0);
      __nv_bfloat162 p01 = __floats2bfloat162_rn(c0, c1), p23 = __floats2bfloat162_rn(c2, c3);
      v0.x = *reinterpret_cast<uint32_t*>(&p01);
      v0.y = *reinterpret_cast<uint32_t*>(&p23);
      uint4* o4 = reinterpret_cast<uint4*>(o);
      o4[0] = v0;
      for (int c = 1; c < Cpad / 8; ++c) o4[c] = make_uint4(0, 0, 0, 0);
    } else if (sizeof(T) == 4 && (Cpad & 3) == 0) {
      float4* o4 = reinterpret_cast<float4*>(o);
      o4[0] = make_float4(c0, c1, c2, c3);
      for (int c = 1; c < Cpad / 4; ++c) o4[c] = make_float4(0.f, 0.f, 0.f, 0.f);
    } else {
      o[0] = from_f32<T>(c0);  o[1] = from_f32<T>(c1);  o[2] = from_f32<T>(c2);  o[3] = from_f32<T>(c3);
      for (int c = 4; c < Cpad; ++c) o[c] = from_f32<T>(0.f);
    }
  }
}

// uint8 HWC input (decoded PNG): 3 bytes per pixel, coalesced enough through L1; same output layout as above.
template <typename T>
__global__ void pack_image_u8_kernel(const uint8_t* __restrict__ img, const float* __restrict__ disp, float disp_scale,
                                     float img_scale, T* __restrict__ out, int64_t total, int Cpad) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const uint8_t* ip = img + i * 3;
    const float c0 = (float)ip[0] * img_scale, c1 = (float)ip[1] * img_scale, c2 = (float)ip[2] * img_scale;
    const float c3 = disp ? disp[i] * disp_scale : 0.f;
    T* o = out + i * Cpad;
    if (sizeof(T) == 2 && (Cpad & 7) == 0) {
      uint4 v0 = make_uint4(0, 0, 0, 0);
      __nv_bfloat162 p01 = __floats2bfloat162_rn(c0, c1), p23 = __floats2bfloat162_rn(c2, c3);
      v0.x = *reinterpret_cast<uint32_t*>(&p01);
      v0.y = *reinterpret_cast<uint32_t*>(&p23);
      uint4* o4 = reinterpret_cast<uint4*>(o);
      o4[0] = v0;
      for (int c = 1; c < Cpad / 8; ++c) o4[c] = make_uint4(0, 0, 0, 0);
    } else {
      o[0] = from_f32<T>(c0);  o[1] = from_f32<T>(c1);  o[2] = from_f32<T>(c2);  o[3] = from_f32<T>(c3);
      for (int c = 4; c < Cpad; ++c) o[c] = from_f32<T>(0.f);
    }
  }
}

__device__ __forceinline__ void pool_bin(int i, int in, int out, int& s, int& e) {
  s = (i * in) / out;
  e = ((i + 1) * in + out - 1) / out;
}

// [N,H,W,C] -> pooled [N,L,L,C]; if to_vox, written as [N,2,2,2,C*L*L/8] with the NCHW .view order.
template <typename T>
__global__ void pool_kernel(const T* __restrict__ x, T* __restrict__ out, int N, int H, int W, int C, int L, int to_vox) {
  const int64_t total = (int64_t)N * L * L * C;
  const int K = C * L * L / 8;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = i;
    const int c = (int)(r % C);  r /= C;
    const int px = (int)(r % L);  r /= L;
    const int py = (int)(r % L);  r /= L;
    const int n = (int)r;
    int ys, ye, xs, xe;
    pool_bin(py, H, L, ys, ye);
    pool_bin(px, W, L, xs, xe);
    float acc = 0.f;
    for (int yy = ys; yy < ye; ++yy)
      for (int xx = xs; xx < xe; ++xx) acc += to_f32(x[(((int64_t)n * H + yy) * W + xx) * C + c]);
    acc /= (float)((ye - ys) * (xe - xs));
    if (to_vox) {
      const int f = (c * L + py) * L + px;
      const int k = f >> 3, cell = f & 7;           // cell = z*4 + y*2 + x of the 2x2x2 grid
      out[((int64_t)n * 8 + cell) * K + k] = from_f32<T>(acc);
    } else {
      out[i] = from_f32<T>(acc);
    }
  }
}

// Split (BF16X2) variant: x [N,H,W, hi(C) | lo(C)], the mean is taken over hi + lo in fp32 and written split again
// ([N,L,L, hi(C) | lo(C)], or [N,2,2,2, hi(K) | lo(K)] with K = C*L*L/8 for to_vox).
__global__ void pool_split_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ out, int N, int H, int W, int C,
                                  int L, int to_vox) {
  const int64_t total = (int64_t)N * L * L * C;
  const int K = C * L * L / 8;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = i;
    const int c = (int)(r % C);  r /= C;
    const int px = (int)(r % L);  r /= L;
    const int py = (int)(r % L);  r /= L;
    const int n = (int)r;
    int ys, ye, xs, xe;
    pool_bin(py, H, L, ys, ye);
    pool_bin(px, W, L, xs, xe);
    float acc = 0.f;
    for (int yy = ys; yy < ye; ++yy)
      for (int xx = xs; xx < xe; ++xx) {
        const __nv_bfloat16* q = x + (((int64_t)n * H + yy) * W + xx) * 2 * C + c;
        acc += __bfloat162float(q[0]) + __bfloat162float(q[C]);
      }
    acc /= (float)((ye - ys) * (xe - xs));
    const __nv_bfloat16 hi = __float2bfloat16_rn(acc), lo = __float2bfloat16_rn(acc - __bfloat162float(hi));
    if (to_vox) {
      const int f = (c * L + py) * L + px;
      const int k = f >> 3, cell = f & 7;
      __nv_bfloat16* o = out + ((int64_t)n * 8 + cell) * 2 * K + k;
      o[0] = hi;  o[K] = lo;
    } else {
      __nv_bfloat16* o = out + (i / C) * 2 * C + c;
      o[0] = hi;  o[C] = lo;
    }
  }
}

template <typename T>
__global__ void __launch_bounds__(256)
fuse_views_kernel(const T* __restrict__ score, int64_t sstride, const T* __restrict__ vol, int64_t vstride,
                  float* __restrict__ fused, int B, int V, int nvox, const uint8_t* __restrict__ gt, Thresh th, int nT,
                  unsigned long long* __restrict__ iou, int64_t score_lo, int64_t vol_lo) {
  // score_lo / vol_lo != 0: split (BF16X2) tensors, value = [e] + [e + lo offset]
  auto ld = [](const T* p, int64_t lo) { return lo ? to_f32(p[0]) + to_f32(p[lo]) : to_f32(p[0]); };
  const int b = blockIdx.y;
  unsigned inter[kMaxThresh], uni[kMaxThresh];
#pragma unroll
  for (int t = 0; t < kMaxThresh; ++t) { inter[t] = 0; uni[t] = 0; }
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nvox; i += gridDim.x * blockDim.x) {
    float m = -INFINITY;
    for (int v = 0; v < V; ++v) m = fmaxf(m, ld(score + (((int64_t)v * B + b) * nvox + i) * sstride, score_lo));
    float s = 0.f, acc = 0.f;
    for (int v = 0; v < V; ++v) {
      const int64_t e = ((int64_t)v * B + b) * nvox + i;
      const float w = expf(ld(score + e * sstride, score_lo) - m);
      s += w;
      acc += w * ld(vol + e * vstride, vol_lo);
    }
    float f = acc / s;
    f = fminf(fmaxf(f, 0.f), 1.f);
    fused[(int64_t)b * nvox + i] = f;
    if (gt) {
      const bool g = gt[(int64_t)b * nvox + i] != 0;
#pragma unroll
      for (int t = 0; t < kMaxThresh; ++t)
        if (t < nT) { const bool p = f >= th.t[t]; inter[t] += (p && g); uni[t] += (p || g); }
    }
  }
  if (gt && iou) {
    // warp shuffle -> shared-memory counters -> ONE global atomic per counter per block (per-warp global atomics on the 2T
    // counters of a sample serialised: 35 us of a 0.7 ms batch-1 forward)
    __shared__ unsigned blk[2 * kMaxThresh];
    if (threadIdx.x < 2 * kMaxThresh) blk[threadIdx.x] = 0;
    __syncthreads();
#pragma unroll
    for (int t = 0; t < kMaxThresh; ++t) {
      if (t >= nT) break;
      unsigned a = inter[t], u = uni[t];
      for (int o = 16; o > 0; o >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); u += __shfl_xor_sync(0xffffffffu, u, o); }
      if ((threadIdx.x & 31) == 0) {
        if (a) atomicAdd(&blk[2 * t], a);
        if (u) atomicAdd(&blk[2 * t + 1], u);
      }
    }
    __syncthreads();
    if ((int)threadIdx.x < 2 * nT && blk[threadIdx.x])
      atomicAdd(iou + (int64_t)b * nT * 2 + threadIdx.x, (unsigned long long)blk[threadIdx.x]);
  }
}

int grid_for(int64_t total, int threads) {
  int64_t blocks = ceil_div64(total, threads);
  const int64_t cap = (int64_t)num_sms() * 16;
  return (int)(blocks > cap ? cap : (blocks < 1 ? 1 : blocks));
}

}  // namespace
}  // namespace s3d

using namespace s3d;

extern "C" const char* s3d_version(void) { return "s3d_b200 0.1 (sm_100a)"; }
extern "C" const char* s3d_last_error(void) { return g_err; }

extern "C" int s3d_set_knob(const char* name, int value) {
  if (!name) { set_error("s3d_set_knob: null name"); return S3D_ERR_INVALID; }
  for (const KnobName& n : kKnobNames)
    if (strcmp(name, n.name) == 0) { knobs().*(n.field) = value; return S3D_OK; }
  set_error("s3d_set_knob: unknown knob '%s'", name);
  return S3D_ERR_INVALID;
}
extern "C" int s3d_get_knob(const char* name) {
  if (name)
    for (const KnobName& n : kKnobNames)
      if (strcmp(name, n.name) == 0) return knobs().*(n.field);
  set_error("s3d_get_knob: unknown knob");
  return S3D_ERR_INVALID;
}

extern "C" int s3d_device_check(int dev) {
  cudaDeviceProp prop;
  cudaError_t e = cudaGetDeviceProperties(&prop, dev);
  if (e != cudaSuccess) { set_error("s3d_device_check: %s", cudaGetErrorString(e)); cudaGetLastError(); return S3D_ERR_CUDA; }
  if (prop.major != 10) { set_error("s3d_device_check: device %d is sm_%d%d, need sm_100", dev, prop.major, prop.minor); return S3D_ERR_UNSUPPORTED; }
  return S3D_OK;
}

extern "C" int s3d_pack_image(const float* img, const float* disp, float disp_scale, void* out, int B, int H, int W,
                              int Cpad, int out_dtype, void* stream) {
  if (!img || !out) { set_error("pack_image: null argument"); return S3D_ERR_INVALID; }
  S3D_CHECK_ARG(B > 0 && H > 0 && W > 0 && Cpad >= 4, "pack_image: bad shape");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t total = (int64_t)B * H * W;
  if (out_dtype == S3D_DTYPE_BF16)
    pack_image_kernel<__nv_bfloat16><<<grid_for(total, 256), 256, 0, st>>>(img, disp, disp_scale, static_cast<__nv_bfloat16*>(out), B, H, W, Cpad);
  else if (out_dtype == S3D_DTYPE_F32)
    pack_image_kernel<float><<<grid_for(total, 256), 256, 0, st>>>(img, disp, disp_scale, static_cast<float*>(out), B, H, W, Cpad);
  else { set_error("pack_image: bad dtype"); return S3D_ERR_INVALID; }
  S3D_LAUNCH_CHECK();
  return S3D_OK;
}

extern "C" int s3d_pack_image_u8(const uint8_t* img, const float* disp, float disp_scale, float img_scale, void* out,
                                 int B, int H, int W, int Cpad, int out_dtype, void* stream) {
  if (!img || !out) { set_error("pack_image_u8: null argument"); return S3D_ERR_INVALID; }
  S3D_CHECK_ARG(B > 0 && H > 0 && W > 0 && Cpad >= 4, "pack_image_u8: bad shape");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t total = (int64_t)B * H * W;
  if (out_dtype == S3D_DTYPE_BF16)
    pack_image_u8_kernel<__nv_bfloat16><<<grid_for(total, 256), 256, 0, st>>>(img, disp, disp_scale, img_scale, static_cast<__nv_bfloat16*>(out), total, Cpad);
  else if (out_dtype == S3D_DTYPE_F32)
    pack_image_u8_kernel<float><<<grid_for(total, 256), 256, 0, st>>>(img, disp, disp_scale, img_scale, static_cast<float*>(out), total, Cpad);
  else { set_error("pack_image_u8: bad dtype"); return S3D_ERR_INVALID; }
  S3D_LAUNCH_CHECK();
  return S3D_OK;
}

// Depth-to-space after a blocked transposed conv (layers.py::from_deconv_k4s2p1_blocked): in[n, j, (class, c)] ->
// out[n, 2j + class, c], c < 8, plus an optional 1x1x1 projection of the 8 features into channel 8 and zeros above.
template <typename T>
__global__ void depth_to_space_kernel(const T* __restrict__ in, T* __restrict__ out, const float* __restrict__ proj_w,
                                      int proj_act, int N, int d, int h, int w, int Cpad) {
  const int64_t total = (int64_t)N * d * h * w * 8;
  float pw[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) pw[c] = proj_w ? __ldg(proj_w + c) : 0.f;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    // consecutive threads = consecutive 16-byte (bf16) chunks of the input: coalesced reads
    const int cls = (int)(i & 7);
    int64_t r = i >> 3;
    const int x = (int)(r % w);  r /= w;
    const int y = (int)(r % h);  r /= h;
    const int z = (int)(r % d);  r /= d;
    const int n = (int)r;
    float f[8];
    const T* ip = in + i * 8;
    const int oz = 2 * z + (cls >> 2), oy = 2 * y + ((cls >> 1) & 1), ox = 2 * x + (cls & 1);
    T* op = out + ((((int64_t)n * 2 * d + oz) * 2 * h + oy) * 2 * w + ox) * Cpad;
    if (sizeof(T) == 2 && Cpad == 16) {
      // bf16, 16 output channels: one 16-byte load, two 16-byte stores
      const uint4 raw = __ldg(reinterpret_cast<const uint4*>(ip));
      const __nv_bfloat162* hp = reinterpret_cast<const __nv_bfloat162*>(&raw);
      float pr = 0.f;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const float2 g = __bfloat1622float2(hp[c]);
        pr = fmaf(g.x, pw[2 * c], pr);  pr = fmaf(g.y, pw[2 * c + 1], pr);
      }
      uint4 hi = make_uint4(0, 0, 0, 0);
      const __nv_bfloat16 pb = __float2bfloat16_rn(proj_w ? apply_act(pr, proj_act, 1.f) : 0.f);
      hi.x = (uint32_t)(*reinterpret_cast<const unsigned short*>(&pb));
      reinterpret_cast<uint4*>(op)[0] = raw;
      reinterpret_cast<uint4*>(op)[1] = hi;
      continue;
    }
    if (sizeof(T) == 4 && Cpad == 16) {
      // fp32, 16 output channels: two 16-byte loads, four 16-byte stores
      const float4 a = __ldg(reinterpret_cast<const float4*>(ip)), b = __ldg(reinterpret_cast<const float4*>(ip) + 1);
      float pr = a.x * pw[0];
      pr = fmaf(a.y, pw[1], pr);  pr = fmaf(a.z, pw[2], pr);  pr = fmaf(a.w, pw[3], pr);
      pr = fmaf(b.x, pw[4], pr);  pr = fmaf(b.y, pw[5], pr);  pr = fmaf(b.z, pw[6], pr);  pr = fmaf(b.w, pw[7], pr);
      float4* o4 = reinterpret_cast<float4*>(op);
      o4[0] = a;  o4[1] = b;
      o4[2] = make_float4(proj_w ? apply_act(pr, proj_act, 1.f) : 0.f, 0.f, 0.f, 0.f);
      o4[3] = make_float4(0.f, 0.f, 0.f, 0.f);
      continue;
    }
#pragma unroll
    for (int c = 0; c < 8; ++c) f[c] = to_f32(ip[c]);
#pragma unroll
    for (int c = 0; c < 8; ++c) op[c] = from_f32<T>(f[c]);
    if (Cpad > 8) {
      float pr = 0.f;
#pragma unroll
      for (int c = 0; c < 8; ++c) pr = fmaf(f[c], pw[c], pr);
      op[8] = from_f32<T>(proj_w ? apply_act(pr, proj_act, 1.f) : 0.f);
      for (int c = 9; c < Cpad; ++c) op[c] = from_f32<T>(0.f);
    }
  }
}

// Split (BF16X2) variant: in [N,d,h,w, hi(64) | lo(64)] -> out [N,2d,2h,2w, hi(16) | lo(16)]; the projection is computed
// from hi + lo in fp32 and stored split in channel 8.
__global__ void depth_to_space_split_kernel(const __nv_bfloat16* __restrict__ in, __nv_bfloat16* __restrict__ out,
                                            const float* __restrict__ proj_w, int proj_act, int N, int d, int h, int w) {
  const int64_t total = (int64_t)N * d * h * w * 8;
  float pw[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) pw[c] = proj_w ? __ldg(proj_w + c) : 0.f;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int cls = (int)(i & 7);
    int64_t r = i >> 3;
    const int64_t pix = r;
    const int x = (int)(r % w);  r /= w;
    const int y = (int)(r % h);  r /= h;
    const int z = (int)(r % d);  r /= d;
    const int n = (int)r;
    const __nv_bfloat16* ip = in + pix * 128 + cls * 8;
    const uint4 rh = __ldg(reinterpret_cast<const uint4*>(ip)), rl = __ldg(reinterpret_cast<const uint4*>(ip + 64));
    const __nv_bfloat162* ph = reinterpret_cast<const __nv_bfloat162*>(&rh);
    const __nv_bfloat162* pl = reinterpret_cast<const __nv_bfloat162*>(&rl);
    float pr = 0.f;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const float2 gh = __bfloat1622float2(ph[c]), gl = __bfloat1622float2(pl[c]);
      pr = fmaf(gh.x + gl.x, pw[2 * c], pr);  pr = fmaf(gh.y + gl.y, pw[2 * c + 1], pr);
    }
    pr = proj_w ? apply_act(pr, proj_act, 1.f) : 0.f;
    const __nv_bfloat16 prh = __float2bfloat16_rn(pr), prl = __float2bfloat16_rn(pr - __bfloat162float(prh));
    const int oz = 2 * z + (cls >> 2), oy = 2 * y + ((cls >> 1) & 1), ox = 2 * x + (cls & 1);
    __nv_bfloat16* op = out + ((((int64_t)n * 2 * d + oz) * 2 * h + oy) * 2 * w + ox) * 32;
    uint4 zh = make_uint4(0, 0, 0, 0), zl = make_uint4(0, 0, 0, 0);
    zh.x = (uint32_t)(*reinterpret_cast<const unsigned short*>(&prh));
    zl.x = (uint32_t)(*reinterpret_cast<const unsigned short*>(&prl));
    reinterpret_cast<uint4*>(op)[0] = rh;  reinterpret_cast<uint4*>(op)[1] = zh;      // hi: 8 features, projection, zeros
    reinterpret_cast<uint4*>(op)[2] = rl;  reinterpret_cast<uint4*>(op)[3] = zl;      // lo
  }
}

extern "C" int s3d_depth_to_space(const void* in, void* out, const float* proj_w, int proj_act, int N, int d, int h, int w,
                                  int Cpad, int dtype, void* stream) {
  if (!in || !out) { set_error("depth_to_space: null argument"); return S3D_ERR_INVALID; }
  S3D_CHECK_ARG(N > 0 && d > 0 && h > 0 && w > 0 && Cpad >= 8 && (Cpad == 8 || Cpad >= 9), "depth_to_space: bad shape");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t total = (int64_t)N * d * h * w * 8;
  if (dtype == S3D_DTYPE_BF16X2) {
    S3D_CHECK_ARG(Cpad == 16, "depth_to_space (split): Cpad must be 16");
    depth_to_space_split_kernel<<<grid_for(total, 256), 256, 0, st>>>(static_cast<const __nv_bfloat16*>(in),
        static_cast<__nv_bfloat16*>(out), proj_w, proj_act, N, d, h, w);
  } else if (dtype == S3D_DTYPE_BF16)
    depth_to_space_kernel<__nv_bfloat16><<<grid_for(total, 256), 256, 0, st>>>(static_cast<const __nv_bfloat16*>(in),
        static_cast<__nv_bfloat16*>(out), proj_w, proj_act, N, d, h, w, Cpad);
  else if (dtype == S3D_DTYPE_F32)
    depth_to_space_kernel<float><<<grid_for(total, 256), 256, 0, st>>>(static_cast<const float*>(in), static_cast<float*>(out),
        proj_w, proj_act, N, d, h, w, Cpad);
  else { set_error("depth_to_space: bad dtype"); return S3D_ERR_INVALID; }
  S3D_LAUNCH_CHECK();
  return S3D_OK;
}

// x = hi + lo with hi exactly representable in TF32 (low 13 mantissa bits cleared) and lo = x - hi (exact in fp32):
// the operand split of the 3-pass 'tf32x3' precision mode (hi*hi + lo*hi + hi*lo on kind::tf32 MMAs, fp32 accumulation).
__global__ void split_tf32_kernel(const float4* __restrict__ x, float4* __restrict__ hi, float4* __restrict__ lo, int64_t n4) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 v = __ldg(x + i);
    float4 h, l;
    h.x = __uint_as_float(__float_as_uint(v.x) & 0xFFFFE000u);  l.x = v.x - h.x;
    h.y = __uint_as_float(__float_as_uint(v.y) & 0xFFFFE000u);  l.y = v.y - h.y;
    h.z = __uint_as_float(__float_as_uint(v.z) & 0xFFFFE000u);  l.z = v.z - h.z;
    h.w = __uint_as_float(__float_as_uint(v.w) & 0xFFFFE000u);  l.w = v.w - h.w;
    hi[i] = h;  lo[i] = l;
  }
}

extern "C" int s3d_split_tf32(const float* x, float* hi, float* lo, int64_t n, void* stream) {
  if (!x || !hi || !lo) { set_error("split_tf32: null argument"); return S3D_ERR_INVALID; }
  S3D_CHECK_ARG(n > 0 && n % 4 == 0, "split_tf32: element count must be a positive multiple of 4");
  S3D_CHECK_ARG(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(hi) | reinterpret_cast<uintptr_t>(lo)) & 15) == 0,
                "split_tf32: pointers must be 16-byte aligned");
  split_tf32_kernel<<<grid_for(n / 4, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const float4*>(x), reinterpret_cast<float4*>(hi), reinterpret_cast<float4*>(lo), n / 4);
  S3D_LAUNCH_CHECK();
  return S3D_OK;
}

// Split (BF16X2) tensor [npix, hi(C) | lo(C)] <-> fp32 [npix, C] (hand-off to / from the kernels that take plain fp32).
__global__ void unsplit_kernel(const __nv_bfloat16* __restrict__ x, float* __restrict__ out, int64_t npix, int C) {
  const int64_t total = npix * C;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t pix = i / C;  const int c = (int)(i % C);
    const __nv_bfloat16* q = x + pix * 2 * C + c;
    out[i] = __bfloat162float(q[0]) + __bfloat162float(q[C]);
  }
}
__global__ void split_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ out, int64_t npix, int C) {
  const int64_t total = npix * C;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t pix = i / C;  const int c = (int)(i % C);
    const float v = x[i];
    const __nv_bfloat16 hi = __float2bfloat16_rn(v);
    __nv_bfloat16* q = out + pix * 2 * C + c;
    q[0] = hi;  q[C] = __float2bfloat16_rn(v - __bfloat162float(hi));
  }
}

extern "C" int s3d_split_bf16(const float* x, void* out, int64_t npix, int C, void* stream) {
  if (!x || !out) { set_error("split_bf16: null argument"); return S3D_ERR_INVALID; }
  S3D_CHECK_ARG(npix > 0 && C > 0, "split_bf16: bad shape");
  split_kernel<<<grid_for(npix * C, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, static_cast<__nv_bfloat16*>(out), npix, C);
  S3D_LAUNCH_CHECK();
  return S3D_OK;
}
extern "C" int s3d_unsplit_bf16(const void* x, float* out, int64_t npix, int C, void* stream) {
  if (!x || !out) { set_error("unsplit_bf16: null argument"); return S3D_ERR_INVALID; }
  S3D_CHECK_ARG(npix > 0 && C > 0, "unsplit_bf16: bad shape");
  unsplit_kernel<<<grid_for(npix * C, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const __nv_bfloat16*>(x), out, npix, C);
  S3D_LAUNCH_CHECK();
  return S3D_OK;
}

static int pool_launch(const void* x, void* out, int N, int H, int W, int C, int L, int dtype, int to_vox, void* stream) {
  if (!x || !out) { set_error("pool: null argument"); return S3D_ERR_INVALID; }
  S3D_CHECK_ARG(N > 0 && H > 0 && W > 0 && C > 0 && L > 0, "pool: bad shape");
  S3D_CHECK_ARG(!to_vox || (C * L * L) % 8 == 0, "latent_to_vox: C*L*L must be a multiple of 8");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t total = (int64_t)N * L * L * C;
  if (dtype == S3D_DTYPE_BF16X2)
    pool_split_kernel<<<grid_for(total, 256), 256, 0, st>>>(static_cast<const __nv_bfloat16*>(x), static_cast<__nv_bfloat16*>(out), N, H, W, C, L, to_vox);
  else if (dtype == S3D_DTYPE_BF16)
    pool_kernel<__nv_bfloat16><<<grid_for(total, 256), 256, 0, st>>>(static_cast<const __nv_bfloat16*>(x), static_cast<__nv_bfloat16*>(out), N, H, W, C, L, to_vox);
  else if (dtype == S3D_DTYPE_F32)
    pool_kernel<float><<<grid_for(total, 256), 256, 0, st>>>(static_cast<const float*>(x), static_cast<float*>(out), N, H, W, C, L, to_vox);
  else { set_error("pool: bad dtype"); return S3D_ERR_INVALID; }
  S3D_LAUNCH_CHECK();
  return S3D_OK;
}

extern "C" int s3d_latent_to_vox(const void* x, void* out, int N, int H, int W, int C, int L, int dtype, void* stream) {
  return pool_launch(x, out, N, H, W, C, L, dtype, 1, stream);
}
extern "C" int s3d_avg_pool(const void* x, void* out, int N, int H, int W, int C, int L, int dtype, void* stream) {
  return pool_launch(x, out, N, H, W, C, L, dtype, 0, stream);
}

extern "C" int s3d_fuse_views(const void* score, int64_t score_stride, const void* vol, int64_t vol_stride, int dtype,
                              float* fused, int B, int V, int nvox, const uint8_t* gt, const float* thresholds, int T,
                              long long* iou, int64_t score_lo, int64_t vol_lo, void* stream) {
  if (!score || !vol || !fused) { set_error("fuse_views: null argument"); return S3D_ERR_INVALID; }
  S3D_CHECK_ARG(B > 0 && V > 0 && nvox > 0 && T >= 0 && T <= kMaxThresh, "fuse_views: bad shape (T<=8)");
  S3D_CHECK_ARG(!gt || (thresholds && iou), "fuse_views: gt needs thresholds and iou");
  Thresh th;
  for (int t = 0; t < kMaxThresh; ++t) th.t[t] = (gt && t < T) ? thresholds[t] : 2.f;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  dim3 grid(ceil_div(nvox, 256 * 4), B);
  S3D_CHECK_ARG(dtype == S3D_DTYPE_BF16X2 ? (score_lo > 0 && vol_lo > 0) : (score_lo == 0 && vol_lo == 0),
                "fuse_views: score_lo / vol_lo are the lo-part offsets of split (BF16X2) tensors, 0 otherwise");
  if (dtype == S3D_DTYPE_BF16 || dtype == S3D_DTYPE_BF16X2)
    fuse_views_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(static_cast<const __nv_bfloat16*>(score), score_stride, static_cast<const __nv_bfloat16*>(vol), vol_stride, fused, B, V, nvox, gt, th, T, reinterpret_cast<unsigned long long*>(iou), score_lo, vol_lo);
  else if (dtype == S3D_DTYPE_F32)
    fuse_views_kernel<float><<<grid, 256, 0, st>>>(static_cast<const float*>(score), score_stride, static_cast<const float*>(vol), vol_stride, fused, B, V, nvox, gt, th, T, reinterpret_cast<unsigned long long*>(iou), 0, 0);
  else { set_error("fuse_views: bad dtype"); return S3D_ERR_INVALID; }
  S3D_LAUNCH_CHECK();
  return S3D_OK;
}
