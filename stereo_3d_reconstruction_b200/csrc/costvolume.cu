// Rows V and S: disparity cost volume and soft-argmin regression.  All HBM-bound kernels.
//
//   cost_volume_concat   one CTA per (volume, image row): the reference row and the target row
//                        are staged once in shared memory, then D planes of 2C channels are
//                        streamed out with 16 B coalesced stores.  Bytes: read 2*C*w*e, write
//                        D*2C*w*e per row -- write-bound.
//   soft_argmin          lanes along x (coalesced planes), online softmax over d in registers.
//   corr_soft_argmin     fused correlation + soft-argmax: the [D,h,w] cost never reaches HBM.
//                        Rows staged (transposed, zero padded by D) in shared memory; each thread
//                        owns a 4(x) x 8(d) register tile, the disparity axis is finished with
//                        warp-shuffle (max, sum, weighted-sum) reductions.
#include "common.cuh"

namespace s3d {
namespace {

// ------------------------------------------------------------------------------------------
// concat volume
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
concat_volume_kernel(const uint4* __restrict__ feat, uint4* __restrict__ vol, int B, int h, int w,
                     int vpp /* 16-B vectors per pixel of one feature map */, int D) {
  extern __shared__ uint4 srow[];          // [2][w*vpp]: ref row, tgt row
  const int n = blockIdx.x / h, y = blockIdx.x % h;
  const bool left_ref = n < B;
  const int tgt_n = left_ref ? n + B : n - B;
  const int rowv = w * vpp;
  const uint4* ref_g = feat + ((int64_t)n * h + y) * rowv;
  const uint4* tgt_g = feat + ((int64_t)tgt_n * h + y) * rowv;
  for (int i = threadIdx.x; i < rowv; i += blockDim.x) {
    srow[i] = __ldg(ref_g + i);
    srow[rowv + i] = __ldg(tgt_g + i);
  }
  __syncthreads();
  const int outv = 2 * rowv;               // vectors per (d, row) output line
  const uint4 zero = make_uint4(0, 0, 0, 0);
  for (int d = 0; d < D; ++d) {
    uint4* o = vol + (((int64_t)n * D + d) * h + y) * outv;
    for (int i = threadIdx.x; i < outv; i += blockDim.x) {
      const int x = i / (2 * vpp), j = i % (2 * vpp);
      uint4 v;
      if (j < vpp) {
        v = srow[x * vpp + j];
      } else {
        const int xs = left_ref ? x - d : x + d;
        v = (xs >= 0 && xs < w) ? srow[rowv + xs * vpp + (j - vpp)] : zero;
      }
      __stcs(o + i, v);                    // streaming store: the volume is consumed much later
    }
  }
}

// Split (BF16X2) features [.., hi(C) | lo(C)] -> split volume [.., hi(ref C, tgt C) | lo(ref C, tgt C)]: the hi halves and the
// lo halves each form the plain concat volume, so a 2C-channel split layer reads it like any other split tensor.
__global__ void __launch_bounds__(256)
concat_volume_split_kernel(const uint4* __restrict__ feat, uint4* __restrict__ vol, int B, int h, int w,
                           int vpp /* 16-B vectors per pixel of one HALF of a feature map */, int D) {
  extern __shared__ uint4 srow[];          // [2][w * 2 vpp]: ref row, tgt row (physical pixels)
  const int n = blockIdx.x / h, y = blockIdx.x % h;
  const bool left_ref = n < B;
  const int tgt_n = left_ref ? n + B : n - B;
  const int rowv = w * 2 * vpp;
  const uint4* ref_g = feat + ((int64_t)n * h + y) * rowv;
  const uint4* tgt_g = feat + ((int64_t)tgt_n * h + y) * rowv;
  for (int i = threadIdx.x; i < rowv; i += blockDim.x) {
    srow[i] = __ldg(ref_g + i);
    srow[rowv + i] = __ldg(tgt_g + i);
  }
  __syncthreads();
  const int outv = 2 * rowv;               // vectors per (d, row) output line: 4 vpp per pixel
  const uint4 zero = make_uint4(0, 0, 0, 0);
  for (int d = 0; d < D; ++d) {
    uint4* o = vol + (((int64_t)n * D + d) * h + y) * outv;
    for (int i = threadIdx.x; i < outv; i += blockDim.x) {
      const int x = i / (4 * vpp), j = i % (4 * vpp);
      const int part = j / vpp, jj = j % vpp;          // part: 0 ref hi, 1 tgt hi, 2 ref lo, 3 tgt lo
      const int half = part >> 1;
      uint4 v;
      if ((part & 1) == 0) {
        v = srow[x * 2 * vpp + half * vpp + jj];
      } else {
        const int xs = left_ref ? x - d : x + d;
        v = (xs >= 0 && xs < w) ? srow[rowv + xs * 2 * vpp + half * vpp + jj] : zero;
      }
      __stcs(o + i, v);
    }
  }
}

// ------------------------------------------------------------------------------------------
// standalone soft-argmin over a [N,D,h,w] fp32 cost
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
soft_argmin_kernel(const float* __restrict__ cost, float* __restrict__ disp, int64_t npix_total, int64_t plane,
                   int D, float sign) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= npix_total) return;
  const int64_t n = i / plane, pix = i % plane;
  const float* c = cost + n * D * plane + pix;
  float m = -INFINITY, s = 0.f, t = 0.f;
  int d = 0;
  for (; d + 8 <= D; d += 8) {                 // 8 independent plane loads in flight per thread
    float v[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = sign * __ldcs(c + (int64_t)(d + k) * plane);
    float mm = v[0];
#pragma unroll
    for (int k = 1; k < 8; ++k) mm = fmaxf(mm, v[k]);
    if (mm > m) { const float sc = expf(m - mm); s *= sc; t *= sc; m = mm; }
#pragma unroll
    for (int k = 0; k < 8; ++k) { const float e = expf(v[k] - m); s += e; t += e * (float)(d + k); }
  }
  for (; d < D; ++d) {
    const float v = sign * __ldcs(c + (int64_t)d * plane);
    if (v > m) { const float sc = expf(m - v); s *= sc; t *= sc; m = v; }
    const float e = expf(v - m);  s += e;  t += e * (float)d;
  }
  disp[i] = t / s;
}

// Four pixels per thread (one 16-byte load per plane, 8 planes = 128 bytes in flight per thread): the one-pixel kernel
// above reaches 0.45-0.67 of the HBM peak on this 20-60 us stream; wider loads keep more bytes in flight per warp and
// quarter the instruction count.  Needs plane % 4 == 0 (a vector never straddles two volumes) and 16-byte aligned cost.
__global__ void __launch_bounds__(256)
soft_argmin_v4_kernel(const float4* __restrict__ cost, float4* __restrict__ disp, int64_t nvec_total, int64_t plane4,
                      int D, float sign) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= nvec_total) return;
  const int64_t n = i / plane4, pix = i % plane4;
  const float4* c = cost + n * D * plane4 + pix;
  const float sl = sign * 1.4426950408889634f;           // softmax in the base-2 domain: one MUFU.EX2 per value
  float m[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY}, s[4] = {0.f, 0.f, 0.f, 0.f}, t[4] = {0.f, 0.f, 0.f, 0.f};
  int d = 0;
  for (; d + 8 <= D; d += 8) {
    float4 q[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) q[k] = __ldcs(c + (int64_t)(d + k) * plane4);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float v[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) v[k] = sl * (j == 0 ? q[k].x : j == 1 ? q[k].y : j == 2 ? q[k].z : q[k].w);
      float mm = v[0];
#pragma unroll
      for (int k = 1; k < 8; ++k) mm = fmaxf(mm, v[k]);
      if (mm > m[j]) { const float sc = exp2f(m[j] - mm); s[j] *= sc; t[j] *= sc; m[j] = mm; }
#pragma unroll
      for (int k = 0; k < 8; ++k) { const float e = exp2f(v[k] - m[j]); s[j] += e; t[j] += e * (float)(d + k); }
    }
  }
  for (; d < D; ++d) {
    const float4 q = __ldcs(c + (int64_t)d * plane4);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float v = sl * (j == 0 ? q.x : j == 1 ? q.y : j == 2 ? q.z : q.w);
      if (v > m[j]) { const float sc = exp2f(m[j] - v); s[j] *= sc; t[j] *= sc; m[j] = v; }
      const float e = exp2f(v - m[j]);  s[j] += e;  t[j] += e * (float)d;
    }
  }
  disp[i] = make_float4(t[0] / s[0], t[1] / s[1], t[2] / s[2], t[3] / s[3]);
}

// ------------------------------------------------------------------------------------------
// tap-plane gather + soft-argmin: the Cout = 1 classifier conv of the aggregation stack.
// A 3x3x3 conv with ONE output channel wastes a 128-row tensor-core tile per tap, so it is computed
// as a pointwise GEMM P[pix][t] = W_t . x[pix] (27 taps = 27 output "channels", one pass over the
// activations, tensor cores) followed by this gather: cost[z,y,x] = sum_t P[z+kz-1, y+ky-1, x+kx-1][t],
// fused with the soft-argmin over z so the cost volume itself never reaches HBM.
// One thread per (n, y, x); marching over the input plane z' it keeps the three partial sums of the
// output planes z'-1, z', z'+1 in registers and retires plane z'-1 into an online softmax.
// kStd: also the distribution's standard deviation -> std_q (common.cuh, SoftSpread).
// ------------------------------------------------------------------------------------------
template <bool kStd>
__global__ void __launch_bounds__(128)
tap_gather_soft_argmin_kernel(const float* __restrict__ P, float* __restrict__ disp, float* __restrict__ cost_out,
                              int N, int D, int h, int w, int ts, float sign, float* __restrict__ std_q) {
  // taps are LINE-PLANAR: P[n][z][y][t][x]: for a fixed tap the lanes of a warp (consecutive x) read
  // consecutive floats (one coalesced wavefront per load, neighbours reuse L1), while the producer
  // writes each image line as one contiguous ts*w*4-byte block (DRAM-friendly).
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y, n = blockIdx.z;
  if (x >= w) return;
  const int64_t plane = (int64_t)h * w;
  const float* Pn = P + (int64_t)n * D * ts * plane;
  const int64_t tstride = w, lstride = (int64_t)ts * w;      // tap stride, line stride
  float m = -INFINITY, s = 0.f, t = 0.f;
  SoftSpread u;
  float c0 = 0.f, c1 = 0.f, c2 = 0.f;            // partial costs of output planes z'-1, z', z'+1
  auto retire = [&](int z, float c) {
    if (cost_out) cost_out[((int64_t)n * D + z) * plane + (int64_t)y * w + x] = c;
    const float v = sign * c;
    if (v > m) {
      const float sc = expf(m - v); s *= sc; t *= sc; m = v;
      if (kStd) { u.scale(sc);  u.move(z, s); }
    }
    const float e = expf(v - m);  s += e;  t += e * (float)z;
    if (kStd) u.add(e, z);
  };
  for (int zi = 0; zi < D; ++zi) {
    const float* Pz = Pn + (int64_t)zi * ts * plane;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f;          // contributions of input plane zi with kz = 2, 1, 0
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
      const int yy = y + ky - 1;
      if (yy < 0 || yy >= h) continue;
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        const int xx = x + kx - 1;
        if (xx < 0 || xx >= w) continue;
        const float* p = Pz + (int64_t)yy * lstride + (int64_t)(ky * 3 + kx) * tstride + xx;
        a0 += __ldg(p + 18 * tstride);   // kz = 2: input plane zi feeds output plane zi - 1
        a1 += __ldg(p + 9 * tstride);    // kz = 1: output plane zi
        a2 += __ldg(p);                // kz = 0: output plane zi + 1
      }
    }
    c0 += a0;  c1 += a1;  c2 += a2;
    if (zi >= 1) retire(zi - 1, c0);
    c0 = c1;  c1 = c2;  c2 = 0.f;
  }
  retire(D - 1, c0);
  disp[(int64_t)n * plane + (int64_t)y * w + x] = t / s;
  if (kStd) std_q[(int64_t)n * plane + (int64_t)y * w + x] = u.sigma(t / s, s);
}

// ------------------------------------------------------------------------------------------
// fused correlation + soft-argmax
// ------------------------------------------------------------------------------------------
constexpr int kXG = 4;   // x per thread
constexpr int kDG = 8;   // d per thread

// kStd: also the standard deviation of each pixel's distribution -> std_row, in a second pass over the held costs about the
// mean the first pass reduced (exact two-pass variance: one more value in the warp-shuffle reduction).
template <typename T, bool kLeftRef, bool kStd>
__device__ __forceinline__ void corr_row(const T* __restrict__ ref_g, const T* __restrict__ tgt_g,
                                         float* __restrict__ disp_row, float* __restrict__ cost_row,
                                         int64_t cost_plane, int w, int C, int D, float inv_c, float* smem,
                                         float* __restrict__ std_row) {
  const int WP = ((w + 3) & ~3);
  const int rs = WP + 4;                       // ref row stride (floats); +4 spreads banks
  const int ts = WP + D + 12 + 4;              // tgt row stride: zero pad D + window slack
  float* refT = smem;                          // [C][rs]
  float* tgtT = smem + C * rs;                 // [C][ts]
  // zero fill (padding must read as 0), then transposed fill
  for (int i = threadIdx.x; i < C * ts; i += blockDim.x) tgtT[i] = 0.f;
  for (int i = threadIdx.x; i < C * rs; i += blockDim.x) refT[i] = 0.f;
  __syncthreads();
  const int shift = kLeftRef ? D : 0;
  for (int i = threadIdx.x; i < w * C; i += blockDim.x) {
    const int x = i / C, c = i % C;
    refT[c * rs + x] = to_f32(ref_g[i]);
    tgtT[c * ts + x + shift] = to_f32(tgt_g[i]);
  }
  __syncthreads();

  const int ndg = D / kDG;                     // lanes sharing one x-group (power of two <= 16)
  const int nxg = WP / kXG;
  const int groups_per_pass = blockDim.x / ndg;
  const int dgi = threadIdx.x % ndg;
  const int d0 = dgi * kDG;
  for (int xg0 = 0; xg0 < nxg; xg0 += groups_per_pass) {
    const int xg = xg0 + threadIdx.x / ndg;
    const bool active = xg < nxg;
    const int x0 = (active ? xg : 0) * kXG;
    const int base = kLeftRef ? (x0 - d0 - 8 + D) : (x0 + d0);
    float acc[kXG][kDG];
#pragma unroll
    for (int i = 0; i < kXG; ++i)
#pragma unroll
      for (int j = 0; j < kDG; ++j) acc[i][j] = 0.f;
    for (int c = 0; c < C; ++c) {
      const float4 r4 = *reinterpret_cast<const float4*>(refT + c * rs + x0);
      const float4* tp = reinterpret_cast<const float4*>(tgtT + c * ts + base);
      const float4 t0 = tp[0], t1 = tp[1], t2 = tp[2];
      const float r[4] = {r4.x, r4.y, r4.z, r4.w};
      const float t[12] = {t0.x, t0.y, t0.z, t0.w, t1.x, t1.y, t1.z, t1.w, t2.x, t2.y, t2.z, t2.w};
#pragma unroll
      for (int i = 0; i < kXG; ++i)
#pragma unroll
        for (int j = 0; j < kDG; ++j) acc[i][j] = fmaf(r[i], t[kLeftRef ? (8 + i - j) : (i + j)], acc[i][j]);
    }
    float res[kXG], sd[kXG];
#pragma unroll
    for (int i = 0; i < kXG; ++i) {
      float m = -INFINITY;
#pragma unroll
      for (int j = 0; j < kDG; ++j) { acc[i][j] *= inv_c; m = fmaxf(m, acc[i][j]); }
      for (int o = ndg >> 1; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
      float s = 0.f, tt = 0.f;
#pragma unroll
      for (int j = 0; j < kDG; ++j) { const float e = __expf(acc[i][j] - m); s += e; tt += e * (float)(d0 + j); }
      for (int o = ndg >> 1; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        tt += __shfl_xor_sync(0xffffffffu, tt, o);
      }
      res[i] = tt / s;
      if (kStd) {
        float v2 = 0.f;
#pragma unroll
        for (int j = 0; j < kDG; ++j) {
          const float dd = (float)(d0 + j) - res[i];
          v2 = fmaf(__expf(acc[i][j] - m) * dd, dd, v2);
        }
        for (int o = ndg >> 1; o > 0; o >>= 1) v2 += __shfl_xor_sync(0xffffffffu, v2, o);
        sd[i] = soft_std(v2 / s, res[i]);
      }
    }
    if (active) {
      if (dgi == 0) {
#pragma unroll
        for (int i = 0; i < kXG; ++i) if (x0 + i < w) disp_row[x0 + i] = res[i];
        if (kStd) {
#pragma unroll
          for (int i = 0; i < kXG; ++i) if (x0 + i < w) std_row[x0 + i] = sd[i];
        }
      }
      if (cost_row) {
#pragma unroll
        for (int i = 0; i < kXG; ++i)
#pragma unroll
          for (int j = 0; j < kDG; ++j)
            if (x0 + i < w) cost_row[(int64_t)(d0 + j) * cost_plane + x0 + i] = acc[i][j];
      }
    }
  }
}

template <typename T, bool kStd>
__global__ void __launch_bounds__(256)
corr_soft_argmin_kernel(const T* __restrict__ feat, float* __restrict__ disp, float* __restrict__ cost_out,
                        int B, int h, int w, int C, int D, float inv_c, float* __restrict__ std_q) {
  extern __shared__ float smem_f[];
  const int n = blockIdx.x / h, y = blockIdx.x % h;
  const bool left_ref = n < B;
  const int tgt_n = left_ref ? n + B : n - B;
  const T* ref_g = feat + ((int64_t)n * h + y) * w * C;
  const T* tgt_g = feat + ((int64_t)tgt_n * h + y) * w * C;
  float* disp_row = disp + ((int64_t)n * h + y) * w;
  const int64_t plane = (int64_t)h * w;
  float* cost_row = cost_out ? cost_out + (int64_t)n * D * plane + (int64_t)y * w : nullptr;
  float* std_row = kStd ? std_q + ((int64_t)n * h + y) * w : nullptr;
  if (left_ref) corr_row<T, true, kStd>(ref_g, tgt_g, disp_row, cost_row, plane, w, C, D, inv_c, smem_f, std_row);
  else          corr_row<T, false, kStd>(ref_g, tgt_g, disp_row, cost_row, plane, w, C, D, inv_c, smem_f, std_row);
}

// ------------------------------------------------------------------------------------------
// bilinear upsample (align_corners = False), PyTorch index / weight convention.  The formula lives in the two helpers
// below, shared by the plain kernels and the evaluating ones, so both write the same bits.
// ------------------------------------------------------------------------------------------
struct UpRow { const float* p0; const float* p1; float ly, hy; };    // the two source rows of one output row + their weights

__device__ __forceinline__ UpRow up_row(const float* __restrict__ q_img, int Y, int h, int w, float ry) {
  float sy = ((float)Y + 0.5f) * ry - 0.5f;  if (sy < 0.f) sy = 0.f;
  const int y0 = (int)sy, y1 = y0 + (y0 < h - 1 ? 1 : 0);
  const float ly = sy - (float)y0;
  return {q_img + (int64_t)y0 * w, q_img + (int64_t)y1 * w, ly, 1.f - ly};
}

__device__ __forceinline__ float up_px(const UpRow& r, int X, int w, float rx, float scale) {
  float sx = ((float)X + 0.5f) * rx - 0.5f;  if (sx < 0.f) sx = 0.f;
  const int x0 = (int)sx, x1 = x0 + (x0 < w - 1 ? 1 : 0);
  const float lx = sx - (float)x0, hx = 1.f - lx;
  const float v = r.hy * (hx * __ldg(r.p0 + x0) + lx * __ldg(r.p0 + x1)) + r.ly * (hx * __ldg(r.p1 + x0) + lx * __ldg(r.p1 + x1));
  return v * scale;
}

// up_px with its roundings spelled out: the contraction ptxas picks for upsample_disp_kernel.  Inlined next to other work it may
// contract the same expression the other way round (1 ulp apart), so the scalar kStd path uses this to stay bit-identical.
__device__ __forceinline__ float up_px_rn(const UpRow& r, int X, int w, float rx, float scale) {
  float sx = ((float)X + 0.5f) * rx - 0.5f;  if (sx < 0.f) sx = 0.f;
  const int x0 = (int)sx, x1 = x0 + (x0 < w - 1 ? 1 : 0);
  const float lx = sx - (float)x0, hx = 1.f - lx;
  const float a = __fmaf_rn(lx, __ldg(r.p0 + x1), __fmul_rn(hx, __ldg(r.p0 + x0)));
  const float b = __fmaf_rn(lx, __ldg(r.p1 + x1), __fmul_rn(hx, __ldg(r.p1 + x0)));
  return __fmul_rn(__fmaf_rn(r.hy, a, __fmul_rn(r.ly, b)), scale);
}

__global__ void upsample_disp_kernel(const float* __restrict__ q, float* __restrict__ out, int N, int h, int w,
                                     int H, int W, float scale) {
  const int64_t total = (int64_t)N * H * W;
  const float ry = (float)h / (float)H, rx = (float)w / (float)W;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int X = (int)(i % W), Y = (int)((i / W) % H);
    const int64_t n = i / ((int64_t)W * H);
    out[i] = up_px(up_row(q + n * h * w, Y, h, w, ry), X, w, rx, scale);
  }
}

// The same, four consecutive outputs per thread (one 16-byte store), 32-bit index arithmetic: the scalar kernel spends its time
// in 64-bit divisions (0.051 ms for 33.5 MB at B = 64, 8x its HBM time).  Same formula per output, bit-identical results.
__global__ void __launch_bounds__(256)
upsample_disp_v4_kernel(const float* __restrict__ q, float4* __restrict__ out, uint32_t total4, int h, int w, int H, int W4,
                        float ry, float rx, float scale) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  const uint32_t X4 = i % (uint32_t)W4, row = i / (uint32_t)W4;
  const uint32_t Y = row % (uint32_t)H, n = row / (uint32_t)H;
  const UpRow r = up_row(q + (int64_t)n * h * w, (int)Y, h, w, ry);
  float o[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) o[k] = up_px(r, 4 * (int)X4 + k, w, rx, scale);
  out[i] = make_float4(o[0], o[1], o[2], o[3]);
}

// ------------------------------------------------------------------------------------------
// upsample + evaluation against GT disparity (kEval) and / or the left-right consistency check (kLR).  Each block covers
// part of ONE (sample, view) image (blockIdx.y = image), so its counters belong to one row of `stats` / `lr_stats`; the
// per-thread counters are integers, reduced by warp shuffle -> shared memory -> one 64-bit atomic per counter per block:
// any order of atomics gives the same sums.
// ------------------------------------------------------------------------------------------
struct DispCounters {
  unsigned n_valid = 0;
  unsigned long long epe_fx = 0;                 // sum of round-half-even(|disp - gt| * 2^16)
  unsigned bad[kMaxThresh] = {};

  __device__ __forceinline__ void add(float d, float g, float max_gt, const Thresh& th, int nT) {
    if (!(isfinite(g) && g >= 0.f && g < max_gt)) return;
    const float e = fabsf(__fsub_rn(d, g));      // the stored value: no contraction with the multiply that produced d
    ++n_valid;
    epe_fx += (unsigned long long)__float2ll_rn(e * 65536.f);    // exact scaling by 2^16, then round half to even
#pragma unroll
    for (int t = 0; t < kMaxThresh; ++t)
      if (t < nT) bad[t] += e > th.t[t];
  }

  // -> dst[0 .. n) of the block's image, n <= kLead + 2 + nT, as [lead (kLead = 1 only), n_valid, epe_fx, bad...]; every
  // thread of the block calls it.  The shared array belongs to the instantiation, so a kernel may flush a <0> and a <1> set
  // back to back.
  template <int kLead = 0>
  __device__ __forceinline__ void flush(unsigned long long* __restrict__ dst, int n, unsigned lead = 0) {
    constexpr int kN = kLead + 2 + kMaxThresh;
    __shared__ unsigned long long blk[kN];
    if (threadIdx.x < kN) blk[threadIdx.x] = 0;
    __syncthreads();
    unsigned long long v[kN];
    v[0] = lead;
    v[kLead] = n_valid;  v[kLead + 1] = epe_fx;
#pragma unroll
    for (int t = 0; t < kMaxThresh; ++t) v[kLead + 2 + t] = bad[t];
#pragma unroll
    for (int k = 0; k < kN; ++k) {
      if (k >= n) break;
      unsigned long long a = v[k];
      for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
      if ((threadIdx.x & 31) == 0 && a) atomicAdd(&blk[k], a);
    }
    __syncthreads();
    if ((int)threadIdx.x < n && blk[threadIdx.x]) atomicAdd(dst + threadIdx.x, blk[threadIdx.x]);
  }
};

// Confidence-filtered counters (kStd): per threshold k < nU, the pixels whose upsampled standard deviation is <= ut.t[k]
// (a non-finite one never is), and with kEval the disparity counters over those of them with valid GT.
constexpr int kMaxUnc = 4;
struct UncCounters {
  unsigned n_conf[kMaxUnc] = {};
  DispCounters c[kMaxUnc];

  template <bool kEval>
  __device__ __forceinline__ void add(float sd, float d, float g, const Thresh& ut, int nU, float max_gt, const Thresh& th,
                                      int nT) {
#pragma unroll
    for (int k = 0; k < kMaxUnc; ++k) {
      if (k < nU && sd <= ut.t[k]) {
        ++n_conf[k];
        if (kEval) c[k].add(d, g, max_gt, th, nT);
      }
    }
  }

  // -> rows [k][3 + nT] of the block's image, [n_conf, n_valid_conf, epe_fx, bad...] (column 0 only without kEval)
  template <bool kEval>
  __device__ __forceinline__ void flush(unsigned long long* __restrict__ dst, int nU, int nT) {
#pragma unroll
    for (int k = 0; k < kMaxUnc; ++k)
      if (k < nU) c[k].flush<1>(dst + k * (3 + nT), kEval ? 3 + nT : 1, n_conf[k]);
  }
};

// image n of [2B]: view = n / B (0 = left-referenced), sample b = n % B; gt / lr_mask / disp_std [B,2,H,W], stats
// [B,2,2+nT], lr_stats [B,2,3+nT], unc_stats [B,2,nU,3+nT]
__device__ __forceinline__ int64_t eval_image_index(int n, int B) { return (int64_t)(n % B) * 2 + n / B; }

// Left-right consistency of the pixel at column X whose stored disparity is d (include/s3d.h, s3d_upsample_disp_eval).  `ro`:
// the OTHER view's source rows of the same output row, so up_px gives the value the other image's blocks store at xo.
// dir = -1 for view 0 (xo = X - k), +1 for view 1 (xo = X + k).
__device__ __forceinline__ bool lr_kept(float d, int X, const UpRow& ro, int w, int W, float rx, float scale, int dir,
                                        float tau) {
  if (!(fabsf(d) < (float)(W + 1))) return false;       // NaN / inf, or |k| > W: xo out of range (and no int overflow)
  const int xo = X + dir * __float2int_rn(d);            // round half to even
  if (xo < 0 || xo >= W) return false;
  return fabsf(__fsub_rn(d, up_px(ro, xo, w, rx, scale))) <= tau;     // NaN on the other side: not kept
}

// kStd: the same interpolation of the standard deviation std_q -> std_out, and the confidence-filtered counters (UncCounters).
template <bool kEval, bool kLR, bool kStd>
__global__ void __launch_bounds__(256)
upsample_disp_eval_v4_kernel(const float* __restrict__ q, float4* __restrict__ out, const float4* __restrict__ gt, int B, int h,
                             int w, int H, int W4, float ry, float rx, float scale, Thresh th, int nT, float max_gt,
                             unsigned long long* __restrict__ stats, uint32_t* __restrict__ lr_mask, float lr_thresh,
                             unsigned long long* __restrict__ lr_stats, const float* __restrict__ std_q,
                             float4* __restrict__ std_out, Thresh ut, int nU, unsigned long long* __restrict__ unc_stats) {
  const int n = blockIdx.y;
  const int64_t img4 = (int64_t)H * W4;
  const float* q_img = q + (int64_t)n * h * w;
  const int64_t q_other = (int64_t)(n < B ? B : -B) * h * w;        // the other view's 1/4-res image, relative to q_img
  const int dir = n < B ? -1 : 1;
  float4* out_img = out + n * img4;
  const float4* gt_img = kEval ? gt + eval_image_index(n, B) * img4 : nullptr;
  uint32_t* mask_img = kLR ? lr_mask + eval_image_index(n, B) * img4 : nullptr;
  const float* std_img = kStd ? std_q + (int64_t)n * h * w : nullptr;
  float4* std_out_img = kStd ? std_out + eval_image_index(n, B) * img4 : nullptr;
  DispCounters c, kc;                                               // all pixels / the kept ones (kLR)
  UncCounters uc;                                                   // the confident ones (kStd)
  unsigned n_kept = 0;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < (uint32_t)img4; i += gridDim.x * blockDim.x) {
    const uint32_t X4 = i % (uint32_t)W4, Y = i / (uint32_t)W4;
    float4 g4 = {};
    if (kEval) g4 = __ldcs(gt_img + i);                             // read once: keep it out of L2
    const UpRow r = up_row(q_img, (int)Y, h, w, ry);
    float o[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) o[k] = up_px(r, 4 * (int)X4 + k, w, rx, scale);
    out_img[i] = make_float4(o[0], o[1], o[2], o[3]);
    const float g[4] = {g4.x, g4.y, g4.z, g4.w};
    if (kEval) {
#pragma unroll
      for (int k = 0; k < 4; ++k) c.add(o[k], g[k], max_gt, th, nT);
    }
    if (kLR) {
      const UpRow ro = {r.p0 + q_other, r.p1 + q_other, r.ly, r.hy};  // same output row Y, same weights
      uint32_t m = 0;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const bool keep = lr_kept(o[k], 4 * (int)X4 + k, ro, w, 4 * W4, rx, scale, dir, lr_thresh);
        m |= (uint32_t)keep << (8 * k);
        n_kept += keep;
        if (kEval && keep) kc.add(o[k], g[k], max_gt, th, nT);
      }
      mask_img[i] = m;                                              // four mask bytes, one 32-bit store
    }
    if (kStd) {
      const UpRow rs = up_row(std_img, (int)Y, h, w, ry);
      float sd[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) sd[k] = up_px(rs, 4 * (int)X4 + k, w, rx, scale);
      std_out_img[i] = make_float4(sd[0], sd[1], sd[2], sd[3]);
#pragma unroll
      for (int k = 0; k < 4; ++k) uc.add<kEval>(sd[k], o[k], g[k], ut, nU, max_gt, th, nT);
    }
  }
  if (kEval) c.flush(stats + eval_image_index(n, B) * (2 + nT), 2 + nT);
  if (kLR) kc.flush<1>(lr_stats + eval_image_index(n, B) * (3 + nT), kEval ? 3 + nT : 1, n_kept);
  if (kStd) uc.flush<kEval>(unc_stats + eval_image_index(n, B) * nU * (3 + nT), nU, nT);
}

template <bool kEval, bool kLR, bool kStd>
__global__ void __launch_bounds__(256)
upsample_disp_eval_kernel(const float* __restrict__ q, float* __restrict__ out, const float* __restrict__ gt, int B, int h, int w,
                          int H, int W, float scale, Thresh th, int nT, float max_gt, unsigned long long* __restrict__ stats,
                          uint8_t* __restrict__ lr_mask, float lr_thresh, unsigned long long* __restrict__ lr_stats,
                          const float* __restrict__ std_q, float* __restrict__ std_out, Thresh ut, int nU,
                          unsigned long long* __restrict__ unc_stats) {
  const int n = blockIdx.y;
  const int img = H * W;                                            // < 2^31 (checked by the launcher)
  const float ry = (float)h / (float)H, rx = (float)w / (float)W;
  const float* q_img = q + (int64_t)n * h * w;
  const int64_t q_other = (int64_t)(n < B ? B : -B) * h * w;
  const int dir = n < B ? -1 : 1;
  float* out_img = out + (int64_t)n * img;
  const float* gt_img = kEval ? gt + eval_image_index(n, B) * img : nullptr;
  uint8_t* mask_img = kLR ? lr_mask + eval_image_index(n, B) * img : nullptr;
  const float* std_img = kStd ? std_q + (int64_t)n * h * w : nullptr;
  float* std_out_img = kStd ? std_out + eval_image_index(n, B) * img : nullptr;
  DispCounters c, kc;
  UncCounters uc;
  unsigned n_kept = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < img; i += gridDim.x * blockDim.x) {
    const int X = i % W, Y = i / W;
    const UpRow r = up_row(q_img, Y, h, w, ry);
    const float d = up_px(r, X, w, rx, scale);
    out_img[i] = d;
    const float g = kEval ? __ldcs(gt_img + i) : 0.f;
    if (kEval) c.add(d, g, max_gt, th, nT);
    if (kLR) {
      const UpRow ro = {r.p0 + q_other, r.p1 + q_other, r.ly, r.hy};
      const bool keep = lr_kept(d, X, ro, w, W, rx, scale, dir, lr_thresh);
      mask_img[i] = keep;
      n_kept += keep;
      if (kEval && keep) kc.add(d, g, max_gt, th, nT);
    }
    if (kStd) {
      const float sd = up_px_rn(up_row(std_img, Y, h, w, ry), X, w, rx, scale);
      std_out_img[i] = sd;
      uc.add<kEval>(sd, d, g, ut, nU, max_gt, th, nT);
    }
  }
  if (kEval) c.flush(stats + eval_image_index(n, B) * (2 + nT), 2 + nT);
  if (kLR) kc.flush<1>(lr_stats + eval_image_index(n, B) * (3 + nT), kEval ? 3 + nT : 1, n_kept);
  if (kStd) uc.flush<kEval>(unc_stats + eval_image_index(n, B) * nU * (3 + nT), nU, nT);
}

// The arguments of one s3d_upsample_disp_eval call, checked there.  The pointers of a group that is off are NULL.
struct UpsampleEvalArgs {
  const float* disp_q = nullptr;
  float* disp = nullptr;
  int B = 0, h = 0, w = 0, H = 0, W = 0;
  float scale = 0.f;
  const float* gt = nullptr;                     // kEval
  Thresh th = {};
  int T = 0;
  float max_gt = 0.f;
  long long* disp_stats = nullptr;
  uint8_t* lr_mask = nullptr;                    // kLR
  float lr_thresh = 0.f;
  long long* lr_stats = nullptr;
  const float* std_q = nullptr;                  // kStd
  float* std_out = nullptr;
  Thresh ut = {};
  int K = 0;
  long long* unc_stats = nullptr;
};

template <bool kEval, bool kLR, bool kStd>
int launch_upsample_eval(const UpsampleEvalArgs& a, cudaStream_t s) {
  const int64_t img = (int64_t)a.H * a.W;
  auto* st = reinterpret_cast<unsigned long long*>(a.disp_stats);
  auto* lst = reinterpret_cast<unsigned long long*>(a.lr_stats);
  auto* ust = reinterpret_cast<unsigned long long*>(a.unc_stats);
  if (a.W % 4 == 0 &&
      ((reinterpret_cast<uintptr_t>(a.disp) | reinterpret_cast<uintptr_t>(a.gt) | reinterpret_cast<uintptr_t>(a.std_out)) & 15) == 0 &&
      (reinterpret_cast<uintptr_t>(a.lr_mask) & 3) == 0) {
    // 16 outputs per thread: 4x fewer blocks (and counter atomics) than one vector per thread
    const dim3 grid((unsigned)ceil_div64(img / 4, 256 * 4), 2 * a.B);
    upsample_disp_eval_v4_kernel<kEval, kLR, kStd><<<grid, 256, 0, s>>>(
        a.disp_q, reinterpret_cast<float4*>(a.disp), reinterpret_cast<const float4*>(a.gt), a.B, a.h, a.w, a.H, a.W / 4,
        (float)a.h / (float)a.H, (float)a.w / (float)a.W, a.scale, a.th, a.T, a.max_gt, st, reinterpret_cast<uint32_t*>(a.lr_mask),
        a.lr_thresh, lst, a.std_q, reinterpret_cast<float4*>(a.std_out), a.ut, a.K, ust);
    S3D_LAUNCH_CHECK();
    return S3D_OK;
  }
  upsample_disp_eval_kernel<kEval, kLR, kStd><<<dim3((unsigned)ceil_div64(img, 256 * 4), 2 * a.B), 256, 0, s>>>(
      a.disp_q, a.disp, a.gt, a.B, a.h, a.w, a.H, a.W, a.scale, a.th, a.T, a.max_gt, st, a.lr_mask, a.lr_thresh, lst, a.std_q,
      a.std_out, a.ut, a.K, ust);
  S3D_LAUNCH_CHECK();
  return S3D_OK;
}

}  // namespace
}  // namespace s3d

using namespace s3d;

namespace s3d {
bool corr_tc_eligible(int w, int C, int D, int dtype);
int corr_tc_launch(const void* feat, float* disp, float* std_q, int B, int h, int w, int C, int D, float inv_c, cudaStream_t stream);
}

extern "C" int s3d_cost_volume_concat(const void* feat, void* vol, int B, int h, int w, int C, int D, int dtype,
                                      void* stream) {
  if (!feat || !vol) { set_error("cost_volume_concat: null argument"); return S3D_ERR_INVALID; }
  S3D_CHECK_ARG(dtype == S3D_DTYPE_F32 || dtype == S3D_DTYPE_BF16 || dtype == S3D_DTYPE_BF16X2, "cost_volume_concat: bad dtype");
  const int esz = dtype == S3D_DTYPE_F32 ? 4 : 2;
  S3D_CHECK_ARG(B > 0 && h > 0 && w > 0 && D > 0 && C > 0 && (C * esz) % 16 == 0,
                "cost_volume_concat: C*elem must be a multiple of 16 B");
  const int vpp = C * esz / 16;
  const bool split = dtype == S3D_DTYPE_BF16X2;
  const size_t smem = (size_t)(split ? 4 : 2) * w * vpp * sizeof(uint4);
  S3D_CHECK_ARG(smem <= 200 * 1024, "cost_volume_concat: row too large for shared memory");
  if (split) {
    S3D_CUDA(cudaFuncSetAttribute(concat_volume_split_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    concat_volume_split_kernel<<<2 * B * h, 256, smem, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const uint4*>(feat), static_cast<uint4*>(vol), B, h, w, vpp, D);
    S3D_LAUNCH_CHECK();
    return S3D_OK;
  }
  S3D_CUDA(cudaFuncSetAttribute(concat_volume_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  concat_volume_kernel<<<2 * B * h, 256, smem, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const uint4*>(feat), static_cast<uint4*>(vol), B, h, w, vpp, D);
  S3D_LAUNCH_CHECK();
  return S3D_OK;
}

extern "C" int s3d_soft_argmin(const float* cost, float* disp, int N, int D, int h, int w, float sign, void* stream) {
  if (!cost || !disp) { set_error("soft_argmin: null argument"); return S3D_ERR_INVALID; }
  S3D_CHECK_ARG(N > 0 && D > 0 && h > 0 && w > 0, "soft_argmin: bad shape");
  const int64_t plane = (int64_t)h * w, total = plane * N;
  if (plane % 4 == 0 && ((reinterpret_cast<uintptr_t>(cost) | reinterpret_cast<uintptr_t>(disp)) & 15) == 0) {
    soft_argmin_v4_kernel<<<(unsigned)ceil_div64(total / 4, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        reinterpret_cast<const float4*>(cost), reinterpret_cast<float4*>(disp), total / 4, plane / 4, D, sign);
    S3D_LAUNCH_CHECK();
    return S3D_OK;
  }
  soft_argmin_kernel<<<(unsigned)ceil_div64(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      cost, disp, total, plane, D, sign);
  S3D_LAUNCH_CHECK();
  return S3D_OK;
}

extern "C" int s3d_corr_soft_argmin(const void* feat, float* disp, float* std_q, float* cost_out, int B, int h, int w, int C,
                                    int c_real, int D, int dtype, void* stream) {
  if (!feat || !disp) { set_error("corr_soft_argmin: null argument"); return S3D_ERR_INVALID; }
  S3D_CHECK_ARG(dtype == S3D_DTYPE_F32 || dtype == S3D_DTYPE_BF16, "corr_soft_argmin: bad dtype");
  S3D_CHECK_ARG(B > 0 && h > 0 && w > 0 && C > 0 && D > 0, "corr_soft_argmin: bad shape");
  S3D_CHECK_ARG(c_real >= 0 && c_real <= C, "corr_soft_argmin: c_real must be in [0, C] (0 = C)");
  // the mean runs over the REAL feature channels; the padded ones are zero and only widen the rows
  const float inv_c = 1.f / (float)(c_real > 0 ? c_real : C);
  // bf16 features, rows of up to 64 pixels, no debug cost output: Gram-matrix kernel on the tensor cores (corr_tc.cu)
  if (!cost_out && corr_tc_eligible(w, C, D, dtype))
    return corr_tc_launch(feat, disp, std_q, B, h, w, C, D, inv_c, static_cast<cudaStream_t>(stream));
  S3D_CHECK_ARG(D >= 8 && D <= 128 && (D & (D - 1)) == 0, "corr_soft_argmin (SIMT path): D must be a power of two in [8,128]");
  const int WP = (w + 3) & ~3;
  const size_t smem = (size_t)C * ((WP + 4) + (WP + D + 16)) * sizeof(float);
  S3D_CHECK_ARG(smem <= 200 * 1024, "corr_soft_argmin: row too large for shared memory");
  const int ndg = D / kDG;
  int threads = (WP / kXG) * ndg;
  threads = ((threads + 31) / 32) * 32;
  if (threads > 256) threads = 256;
  if (threads < 32) threads = 32;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  auto launch = [&](auto kern, const auto* f) -> int {
    S3D_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    kern<<<2 * B * h, threads, smem, st>>>(f, disp, cost_out, B, h, w, C, D, inv_c, std_q);
    S3D_LAUNCH_CHECK();
    return S3D_OK;
  };
  if (dtype == S3D_DTYPE_BF16) {
    const auto* f = static_cast<const __nv_bfloat16*>(feat);
    return std_q ? launch(corr_soft_argmin_kernel<__nv_bfloat16, true>, f) : launch(corr_soft_argmin_kernel<__nv_bfloat16, false>, f);
  }
  const auto* f = static_cast<const float*>(feat);
  return std_q ? launch(corr_soft_argmin_kernel<float, true>, f) : launch(corr_soft_argmin_kernel<float, false>, f);
}

extern "C" int s3d_upsample_disp(const float* disp_q, float* disp, int N, int h, int w, int H, int W, float scale,
                                 void* stream) {
  if (!disp_q || !disp) { set_error("upsample_disp: null argument"); return S3D_ERR_INVALID; }
  S3D_CHECK_ARG(N > 0 && h > 0 && w > 0 && H > 0 && W > 0, "upsample_disp: bad shape");
  const int64_t total = (int64_t)N * H * W;
  if (W % 4 == 0 && total / 4 < (1ll << 31) && (reinterpret_cast<uintptr_t>(disp) & 15) == 0) {
    const uint32_t total4 = (uint32_t)(total / 4);
    upsample_disp_v4_kernel<<<(total4 + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(
        disp_q, reinterpret_cast<float4*>(disp), total4, h, w, H, W / 4, (float)h / (float)H, (float)w / (float)W, scale);
    S3D_LAUNCH_CHECK();
    return S3D_OK;
  }
  int64_t blocks = ceil_div64(total, 256);
  if (blocks > (int64_t)num_sms() * 16) blocks = (int64_t)num_sms() * 16;
  upsample_disp_kernel<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(disp_q, disp, N, h, w, H, W, scale);
  S3D_LAUNCH_CHECK();
  return S3D_OK;
}

extern "C" int s3d_upsample_disp_eval(const float* disp_q, float* disp, int B, int h, int w, int H, int W, float scale,
                                      const float* gt, const float* thresholds, int T, float max_gt, long long* disp_stats,
                                      uint8_t* lr_mask, float lr_thresh, long long* lr_stats, const float* disp_std_q,
                                      float* disp_std, const float* unc_thresh, int K, long long* unc_stats, void* stream) {
  if (!disp_q || !disp || (gt && T > 0 && !thresholds) || (K > 0 && (!unc_thresh || !unc_stats))) {
    set_error("upsample_disp_eval: null argument");
    return S3D_ERR_INVALID;
  }
  S3D_CHECK_ARG(gt || lr_mask || disp_std_q,
                "upsample_disp_eval: gt, lr_mask and disp_std_q are all NULL (the plain upsampling is s3d_upsample_disp)");
  S3D_CHECK_ARG(!gt == !disp_stats, "upsample_disp_eval: gt and disp_stats must be both set or both NULL");
  S3D_CHECK_ARG(!lr_mask == !lr_stats, "upsample_disp_eval: lr_mask and lr_stats must be both set or both NULL");
  S3D_CHECK_ARG(!disp_std_q == !disp_std, "upsample_disp_eval: disp_std_q and disp_std must be both set or both NULL");
  S3D_CHECK_ARG(B > 0 && 2 * B < 65536 && h > 0 && w > 0 && H > 0 && W > 0 && (int64_t)H * W < (1ll << 31),
                "upsample_disp_eval: bad shape");
  S3D_CHECK_ARG(T >= 0 && T <= kMaxThresh, "upsample_disp_eval: T must be in [0, 8]");
  S3D_CHECK_ARG(K >= 0 && K <= kMaxUnc, "upsample_disp_eval: K must be in [0, 4]");
  S3D_CHECK_ARG(disp_std_q || K == 0, "upsample_disp_eval: unc_thresh needs disp_std_q");
  S3D_CHECK_ARG(!lr_mask || lr_thresh >= 0.f, "upsample_disp_eval: lr_thresh must be >= 0 (and not NaN)");
  S3D_CHECK_ARG(!gt || max_gt > 0.f, "upsample_disp_eval: max_gt must be > 0");
  UpsampleEvalArgs a;
  a.disp_q = disp_q;  a.disp = disp;  a.B = B;  a.h = h;  a.w = w;  a.H = H;  a.W = W;  a.scale = scale;
  a.gt = gt;  a.T = T;  a.max_gt = max_gt;  a.disp_stats = disp_stats;
  for (int t = 0; t < kMaxThresh; ++t) a.th.t[t] = gt && t < T ? thresholds[t] : 0.f;
  a.lr_mask = lr_mask;  a.lr_thresh = lr_thresh;  a.lr_stats = lr_stats;
  a.std_q = disp_std_q;  a.std_out = disp_std;  a.K = K;  a.unc_stats = unc_stats;
  for (int k = 0; k < K; ++k) {
    S3D_CHECK_ARG(unc_thresh[k] >= 0.f && unc_thresh[k] < INFINITY, "upsample_disp_eval: unc_thresh must be finite and >= 0");
    a.ut.t[k] = unc_thresh[k];
  }
  // one instantiation per combination of groups that are on
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (!disp_std_q) {
    if (!lr_mask) return launch_upsample_eval<true, false, false>(a, s);
    return gt ? launch_upsample_eval<true, true, false>(a, s) : launch_upsample_eval<false, true, false>(a, s);
  }
  if (gt && lr_mask) return launch_upsample_eval<true, true, true>(a, s);
  if (gt) return launch_upsample_eval<true, false, true>(a, s);
  if (lr_mask) return launch_upsample_eval<false, true, true>(a, s);
  return launch_upsample_eval<false, false, true>(a, s);
}

extern "C" int s3d_tap_gather_soft_argmin(const float* taps, float* disp, float* std_q, float* cost_out, int N, int D, int h,
                                          int w, int tap_stride, float sign, void* stream) {
  if (!taps || !disp) { set_error("tap_gather_soft_argmin: null argument"); return S3D_ERR_INVALID; }
  S3D_CHECK_ARG(N > 0 && D > 0 && h > 0 && w > 0 && tap_stride >= 27 && h < 65536 && N < 65536,
                "tap_gather_soft_argmin: bad shape");
  const int threads = w <= 32 ? 32 : (w <= 64 ? 64 : 128);
  dim3 grid(ceil_div(w, threads), h, N);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (std_q)
    tap_gather_soft_argmin_kernel<true><<<grid, threads, 0, st>>>(taps, disp, cost_out, N, D, h, w, tap_stride, sign, std_q);
  else
    tap_gather_soft_argmin_kernel<false><<<grid, threads, 0, st>>>(taps, disp, cost_out, N, D, h, w, tap_stride, sign, nullptr);
  S3D_LAUNCH_CHECK();
  return S3D_OK;
}
