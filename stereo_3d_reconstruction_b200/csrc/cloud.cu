// Coloured point clouds of the two disparity maps (s3d_disp_cloud): back-projection with the camera, the kept-pixel filter
// and the compaction into one cloud per sample.  Definitions (which pixels are kept, the point, the colour, the order) in
// include/s3d.h.
//
// Two launches, both streaming:
//   1. cloud_count_kernel: a warp per row (r = v * H + y of sample b), lanes on 4 consecutive pixels (16-byte loads of disp and
//      disp_std, 4-byte loads of the mask when W % 4 == 0 and the pointers allow it).  A ballot and popc per 32 pixels give
//      the row's kept count, written to the workspace int32 [B, 2H] (rows in output order: view 0, then view 1).
//   2. cloud_write_kernel: a block per band of rows of one sample.  Its base is the sum of the row counts before the band
//      (a block reduction over at most 2H ints, read from L2).  The band is walked in tiles of 4 pixels per thread; ranks
//      within a tile come from ballot and popc prefixes plus a scan of the warp totals.  The colours are loaded with the maps
//      (16-byte loads per fp32 plane, 4-byte loads of the uint8 pixels), before the filter is known, so no load waits on
//      another.  The tile's points and colours are staged in shared memory at the offset their global destination has in a
//      16-byte word and copied out as one contiguous run of floats and one of bytes with 16-byte stores.
//   The block holding row 0 of a sample also writes its counts.  Positions come from counts only, no atomics: the output is
//   deterministic and does not depend on the batch split.
#include "common.cuh"

namespace s3d {
namespace {

constexpr int kCloudThreads = 256;
constexpr int kCloudWarps = kCloudThreads / 32;
constexpr int kCloudTile = 4 * kCloudThreads;            // pixels per tile of the write pass
constexpr int kCloudBandPixels = 1024;                   // target pixels per band of the write pass

struct CloudIn {
  const float* disp;       // [2B,H,W], view-major
  const uint8_t* mask;     // [B,2,H,W] or NULL
  const float* std;        // [B,2,H,W] or NULL
  float max_std, min_disp;
  int B, H, W;
};

// The filter of include/s3d.h: d finite, d + doffs >= min_disp (fp32 add), mask == 1, spread <= max_std (a NaN spread compares
// false); m and s are ignored without their tensor (m = 1, s = 0 then).
__device__ __forceinline__ bool kept(const CloudIn& a, float d, float doffs, unsigned m, float s) {
  return isfinite(d) && __fadd_rn(d, doffs) >= a.min_disp && m == 1u && (!a.std || s <= a.max_std);
}

// Kept bits (bit j: pixel x + j) and disparities of pixels x .. x+3 of row y of view v of sample b.  VEC: W % 4 == 0 and the
// pointers are aligned, so the four pixels are one 16-byte (4-byte for the mask) load each; otherwise pixels past W are not
// kept and not read.
template <bool VEC>
__device__ __forceinline__ unsigned load_keep4(const CloudIn& a, int b, int v, int y, int x, float doffs, float d[4]) {
  const int64_t pd = ((int64_t)(v * a.B + b) * a.H + y) * a.W + x;          // disp
  const int64_t pm = ((int64_t)(b * 2 + v) * a.H + y) * a.W + x;            // mask / std
  float s[4] = {0.f, 0.f, 0.f, 0.f};
  unsigned m4 = 0x01010101u, live = 0xfu;
  if (VEC) {
    const float4 dv = __ldg(reinterpret_cast<const float4*>(a.disp + pd));
    d[0] = dv.x;  d[1] = dv.y;  d[2] = dv.z;  d[3] = dv.w;
    if (a.mask) m4 = __ldg(reinterpret_cast<const unsigned*>(a.mask + pm));
    if (a.std) {
      const float4 sv = __ldg(reinterpret_cast<const float4*>(a.std + pm));
      s[0] = sv.x;  s[1] = sv.y;  s[2] = sv.z;  s[3] = sv.w;
    }
  } else {
    live = 0u;
    m4 = 0u;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      d[j] = 0.f;
      if (x + j < a.W) {
        live |= 1u << j;
        d[j] = __ldg(a.disp + pd + j);
        m4 |= (a.mask ? (unsigned)__ldg(a.mask + pm + j) : 1u) << (8 * j);
        if (a.std) s[j] = __ldg(a.std + pm + j);
      }
    }
  }
  unsigned k = 0;
#pragma unroll
  for (int j = 0; j < 4; ++j)
    k |= (unsigned)(((live >> j) & 1u) && kept(a, d[j], doffs, (m4 >> (8 * j)) & 0xffu, s[j])) << j;
  return k;
}

// The same for the one pixel x of row y of view v of sample b.
__device__ __forceinline__ bool load_keep1(const CloudIn& a, int b, int v, int y, int x, float doffs, float& d) {
  const int64_t pm = ((int64_t)(b * 2 + v) * a.H + y) * a.W + x;
  d = __ldg(a.disp + ((int64_t)(v * a.B + b) * a.H + y) * a.W + x);
  return kept(a, d, doffs, a.mask ? __ldg(a.mask + pm) : 1u, a.std ? __ldg(a.std + pm) : 0.f);
}

template <bool VEC>
__global__ void __launch_bounds__(kCloudThreads)
cloud_count_kernel(CloudIn a, const float* __restrict__ camera, int* __restrict__ row_counts) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * kCloudWarps + (threadIdx.x >> 5);
  if (row >= (int64_t)a.B * 2 * a.H) return;
  const int b = (int)(row / (2 * a.H)), r = (int)(row % (2 * a.H));
  const int v = r >= a.H, y = r - v * a.H;
  const float doffs = __ldg(camera + b * 5 + 4);
  int n = 0;
#pragma unroll 2
  for (int x0 = 0; x0 < a.W; x0 += 128) {
    const int x = x0 + 4 * lane;
    float d[4];
    const unsigned k = x < a.W ? load_keep4<VEC>(a, b, v, y, x, doffs, d) : 0u;
#pragma unroll
    for (int j = 0; j < 4; ++j) n += __popc(__ballot_sync(0xffffffffu, (k >> j) & 1u));
  }
  if (lane == 0) row_counts[row] = n;
}

__device__ __forceinline__ int block_sum(int s, int* red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  __syncthreads();                                                        // red is reused
  if (lane == 0) red[warp] = s;
  __syncthreads();
  int t = 0;
#pragma unroll
  for (int w = 0; w < kCloudWarps; ++w) t += red[w];
  return t;
}

// Colours of pixels x .. x+3 of row y of image `img` of sample b (one row, x % 4 == 0, aligned rows), packed r | g << 8 |
// b << 16: three 4-byte loads of the uint8 HWC pixels, or one 16-byte load per fp32 channel plane.
template <bool U8>
__device__ __forceinline__ void load_rgb4(const void* img, int b, int y, int x, int H, int W, unsigned c[4]) {
  const int64_t HW = (int64_t)H * W, pix = (int64_t)y * W + x;
  if (U8) {
    const unsigned* p = reinterpret_cast<const unsigned*>(static_cast<const uint8_t*>(img) + ((int64_t)b * HW + pix) * 3);
    const unsigned w0 = __ldg(p), w1 = __ldg(p + 1), w2 = __ldg(p + 2);   // r0 g0 b0 r1 | g1 b1 r2 g2 | b2 r3 g3 b3
    c[0] = w0 & 0xffffffu;
    c[1] = (w0 >> 24) | (w1 & 0xffffu) << 8;
    c[2] = (w1 >> 16) | (w2 & 0xffu) << 16;
    c[3] = w2 >> 8;
  } else {
    const float* p = static_cast<const float*>(img) + (int64_t)b * 3 * HW + pix;
    const float4 r = __ldg(reinterpret_cast<const float4*>(p)), g = __ldg(reinterpret_cast<const float4*>(p + HW)),
                 bl = __ldg(reinterpret_cast<const float4*>(p + 2 * HW));
    c[0] = colour_f32(r.x) | colour_f32(g.x) << 8 | colour_f32(bl.x) << 16;
    c[1] = colour_f32(r.y) | colour_f32(g.y) << 8 | colour_f32(bl.y) << 16;
    c[2] = colour_f32(r.z) | colour_f32(g.z) << 8 | colour_f32(bl.z) << 16;
    c[3] = colour_f32(r.w) | colour_f32(g.w) << 8 | colour_f32(bl.w) << 16;
  }
}

// Copies the staged run s[pad, pad + n) to d[0, n), where pad = (address of d / sizeof(T)) % (16 / sizeof(T)) so that the
// staged and the global element share their position in a 16-byte word: 16-byte stores from 16-byte shared loads, with
// element-wise head and tail.  s is 16-byte aligned.
template <typename T>
__device__ __forceinline__ void copy_run(T* d, const T* s, int pad, int n) {
  constexpr int V = 16 / sizeof(T);
  const int u0 = pad, u1 = pad + n, q0 = (u0 + V - 1) / V, q1 = u1 / V;
  T* base = d - pad;                                                      // element u of the run is base[u]
  for (int u = u0 + threadIdx.x; u < min(q0 * V, u1); u += kCloudThreads) base[u] = s[u];
  for (int q = q0 + threadIdx.x; q < q1; q += kCloudThreads)
    reinterpret_cast<uint4*>(base)[q] = reinterpret_cast<const uint4*>(s)[q];
  for (int u = max(q1, q0) * V + threadIdx.x; u < u1; u += kCloudThreads) base[u] = s[u];
}

// 5 blocks of 256 threads an SM (at most 51 registers): the occupancy hides the two load round trips of a band better than
// the 63 registers the compiler would take (measured on a B200: 70 against 75 us for the write pass at B = 64, 256^2)
template <bool VEC, bool U8>
__global__ void __launch_bounds__(kCloudThreads, 5)
cloud_write_kernel(CloudIn a, const void* __restrict__ left, const void* __restrict__ right, const float* __restrict__ camera,
                   const int* __restrict__ row_counts, int rows_per_band, int n_bands, float* __restrict__ xyz,
                   uint8_t* __restrict__ rgb, int* __restrict__ counts) {
  __shared__ __align__(16) float sxyz[kCloudTile * 3 + 4];
  __shared__ __align__(16) uint8_t srgb[kCloudTile * 3 + 16];
  __shared__ int red[kCloudWarps];                                        // block_sum
  __shared__ int wtot[kCloudWarps];                                       // kept points of each warp in the tile
  __shared__ int wbase[kCloudWarps + 1];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int b = blockIdx.x / n_bands, band = blockIdx.x % n_bands;
  const int H = a.H, W = a.W, R2 = 2 * H;
  const int r0 = band * rows_per_band, r1 = min(r0 + rows_per_band, R2);
  const int* rc = row_counts + (int64_t)b * R2;
  const float* cam = camera + b * 5;
  const float f = __ldg(cam), cx = __ldg(cam + 1), cy = __ldg(cam + 2), bl = __ldg(cam + 3), doffs = __ldg(cam + 4);
  const int64_t P = (int64_t)(r1 - r0) * W;                               // pixels of the band, rows r0.. in raster order
  // VEC: a thread's 4 pixels p .. p+3 are in one row; their maps and colours (loaded with the maps, not after the filter)
  unsigned k = 0, col[4] = {0u, 0u, 0u, 0u};
  float d[4];
  auto load_tile = [&](int64_t p) {
    k = 0;
    if (VEC && p < P) {
      const int r = r0 + (int)(p / W), x = (int)(p % W), v = r >= H, y = r - v * H;
      k = load_keep4<true>(a, b, v, y, x, doffs, d);
      load_rgb4<U8>(v ? right : left, b, y, x, H, W, col);
    }
  };
  load_tile(4 * threadIdx.x);                                             // the first tile's loads overlap the reduction
  // base of the band: the kept points of the rows before it
  int s = 0;
  for (int r = threadIdx.x; r < r0; r += kCloudThreads) s += rc[r];
  const int base = block_sum(s, red);
  if (band == 0) {                                                        // counts of the sample, once
    int c0 = 0, c1 = 0;
    for (int r = threadIdx.x; r < R2; r += kCloudThreads) (r < H ? c0 : c1) += rc[r];
    c0 = block_sum(c0, red);
    c1 = block_sum(c1, red);
    if (threadIdx.x == 0) { counts[2 * b] = c0;  counts[2 * b + 1] = c1; }
  }
  const float fb = __fmul_rn(f, bl);
  const int64_t HW = (int64_t)H * W;
  float* xo = xyz + ((int64_t)b * 2 * HW + base) * 3;
  uint8_t* co = rgb + ((int64_t)b * 2 * HW + base) * 3;
  int px = (int)((reinterpret_cast<uintptr_t>(xo) >> 2) & 3), pc = (int)(reinterpret_cast<uintptr_t>(co) & 15);
  const unsigned lt = (1u << lane) - 1u;
  for (int64_t p0 = 0; p0 < P; p0 += kCloudTile) {
    const int64_t p = p0 + 4 * threadIdx.x;                               // first of this thread's 4 pixels
    if (p0 > 0) load_tile(p);
    // VEC: loaded above.  Otherwise a thread's pixels may wrap to the next row: take them one by one.
    unsigned m[4];
    int before = 0, total = 0;
    if (VEC) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        m[j] = __ballot_sync(0xffffffffu, (k >> j) & 1u);
        before += __popc(m[j] & lt);
        total += __popc(m[j]);
      }
    } else {
      // scalar form: pixel p + j lives in row r0 + (p + j) / W
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int64_t q = p + j;
        unsigned kj = 0;
        if (q < P) {
          const int rj = r0 + (int)(q / W), xj = (int)(q % W);
          const int vj = rj >= H;
          kj = load_keep1(a, b, vj, rj - vj * H, xj, doffs, d[j]);
        }
        k |= kj << j;
        m[j] = __ballot_sync(0xffffffffu, kj);
        before += __popc(m[j] & lt);
        total += __popc(m[j]);
      }
    }
    if (lane == 0) wtot[warp] = total;
    __syncthreads();
    if (threadIdx.x == 0) {
      int t = 0;
      for (int w = 0; w < kCloudWarps; ++w) { wbase[w] = t;  t += wtot[w]; }
      wbase[kCloudWarps] = t;
    }
    __syncthreads();
    int o = wbase[warp] + before;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (!((k >> j) & 1u)) continue;
      const int64_t q = p + j;
      const int rj = r0 + (int)(q / W), xj = (int)(q % W);
      const int vj = rj >= H, yj = rj - vj * H;
      const float den = __fadd_rn(d[j], doffs);
      const float z = __fdiv_rn(fb, den), sc = __fdiv_rn(z, f);
      float X = __fmul_rn(__fsub_rn((float)xj, cx), sc);
      if (vj) X = __fadd_rn(X, bl);
      sxyz[px + 3 * o] = X;
      sxyz[px + 3 * o + 1] = __fmul_rn(__fsub_rn((float)yj, cy), sc);
      sxyz[px + 3 * o + 2] = z;
      unsigned c = col[j];
      if (!VEC) {
        const int64_t pix = (int64_t)yj * W + xj;
        if (U8) {
          const uint8_t* im = static_cast<const uint8_t*>(vj ? right : left) + ((int64_t)b * HW + pix) * 3;
          c = (unsigned)__ldg(im) | (unsigned)__ldg(im + 1) << 8 | (unsigned)__ldg(im + 2) << 16;
        } else {
          const float* im = static_cast<const float*>(vj ? right : left) + (int64_t)b * 3 * HW + pix;
          c = colour_f32(__ldg(im)) | colour_f32(__ldg(im + HW)) << 8 | colour_f32(__ldg(im + 2 * HW)) << 16;
        }
      }
      srgb[pc + 3 * o] = (uint8_t)c;
      srgb[pc + 3 * o + 1] = (uint8_t)(c >> 8);
      srgb[pc + 3 * o + 2] = (uint8_t)(c >> 16);
      ++o;
    }
    __syncthreads();
    const int n3 = 3 * wbase[kCloudWarps];
    copy_run(xo, sxyz, px, n3);
    copy_run(co, srgb, pc, n3);
    xo += n3;
    co += n3;
    px = (px + n3) & 3;
    pc = (pc + n3) & 15;
    __syncthreads();                                                      // the staging buffers are reused
  }
}

bool aligned(const void* p, int n) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) % n) == 0; }

}  // namespace
}  // namespace s3d

using namespace s3d;

extern "C" int64_t s3d_disp_cloud_workspace_bytes(int B, int H) {
  if (B < 0 || H < 0) return 0;
  return (int64_t)B * 2 * H * (int64_t)sizeof(int);
}

extern "C" int s3d_disp_cloud(const float* disp, int B, int H, int W, const void* left, const void* right, int img_u8,
                              const uint8_t* lr_mask, const float* disp_std, float max_std, const float* camera,
                              float min_disp, float* xyz, uint8_t* rgb, int* counts, void* workspace,
                              int64_t workspace_bytes, void* stream) {
  if (!disp || !left || !right || !camera || !xyz || !rgb || !counts) {
    set_error("disp_cloud: null argument");
    return S3D_ERR_INVALID;
  }
  S3D_CHECK_ARG(B >= 0 && H >= 1 && W >= 1, "disp_cloud: need B >= 0, H >= 1, W >= 1, got %d %d %d", B, H, W);
  S3D_CHECK_ARG(2 * (int64_t)H * W <= 0x7fffffff, "disp_cloud: 2 H W must fit in int32, got H = %d, W = %d", H, W);
  S3D_CHECK_ARG(img_u8 == 0 || img_u8 == 1, "disp_cloud: img_u8 must be 0 or 1, got %d", img_u8);
  S3D_CHECK_ARG(isfinite(min_disp) && min_disp > 0.f, "disp_cloud: min_disp must be finite and > 0, got %g", (double)min_disp);
  S3D_CHECK_ARG(!disp_std || (isfinite(max_std) && max_std >= 0.f),
                "disp_cloud: max_std must be finite and >= 0, got %g", (double)max_std);
  const int64_t need = s3d_disp_cloud_workspace_bytes(B, H);
  S3D_CHECK_ARG(workspace_bytes >= need && (need == 0 || workspace),
                "disp_cloud: workspace of %lld bytes, need %lld", (long long)workspace_bytes, (long long)need);
  S3D_CHECK_ARG(aligned(workspace, 4), "disp_cloud: workspace must be 4-byte aligned");
  if (B == 0) return S3D_OK;
  const CloudIn in{disp, lr_mask, disp_std, max_std, min_disp, B, H, W};
  const bool vec = W % 4 == 0 && aligned(disp, 16) && aligned(disp_std, 16) && aligned(lr_mask, 4) &&
                   aligned(left, img_u8 ? 4 : 16) && aligned(right, img_u8 ? 4 : 16);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int* rc = static_cast<int*>(workspace);
  const int64_t rows = (int64_t)B * 2 * H;
  const int64_t gc = (rows + kCloudWarps - 1) / kCloudWarps;
  const int rpb = W >= kCloudBandPixels ? 1 : kCloudBandPixels / W;
  const int nb = (2 * H + rpb - 1) / rpb;
  S3D_CHECK_ARG(gc <= 0x7fffffff && (int64_t)B * nb <= 0x7fffffff, "disp_cloud: too many rows (B = %d, H = %d)", B, H);
  if (vec) cloud_count_kernel<true><<<(unsigned)gc, kCloudThreads, 0, st>>>(in, camera, rc);
  else     cloud_count_kernel<false><<<(unsigned)gc, kCloudThreads, 0, st>>>(in, camera, rc);
  S3D_LAUNCH_CHECK();
  const unsigned gw = (unsigned)((int64_t)B * nb);
  if (vec && img_u8)  cloud_write_kernel<true, true><<<gw, kCloudThreads, 0, st>>>(in, left, right, camera, rc, rpb, nb, xyz, rgb, counts);
  else if (vec)       cloud_write_kernel<true, false><<<gw, kCloudThreads, 0, st>>>(in, left, right, camera, rc, rpb, nb, xyz, rgb, counts);
  else if (img_u8)    cloud_write_kernel<false, true><<<gw, kCloudThreads, 0, st>>>(in, left, right, camera, rc, rpb, nb, xyz, rgb, counts);
  else                cloud_write_kernel<false, false><<<gw, kCloudThreads, 0, st>>>(in, left, right, camera, rc, rpb, nb, xyz, rgb, counts);
  S3D_LAUNCH_CHECK();
  return S3D_OK;
}
