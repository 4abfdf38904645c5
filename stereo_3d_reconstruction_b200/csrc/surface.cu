// Voxel surfaces evaluated against each other (s3d_voxel_surface_eval): exact voxel-face Chamfer L2 / L1 and F-score
// counters of predicted occupancy (fused >= t) against GT occupancy (gt != 0), in integers.
//
// Surface = the centres of the faces between an occupied and an empty voxel (outside the grid is empty).  In doubled
// coordinates a voxel centre is 2i+1 and a face sits at an even coordinate on its axis and odd ones on the other two, so
// every surface point is a site of the (2n+1)^3 lattice; s = squared distance in doubled units to the nearest site of the
// other surface, an integer <= 3 (2n)^2 < 2^16.  The distance transform is separable (squared Euclidean = sum over axes):
//   surface_plane_kernel   one block per (sample, grid, lattice plane z): pass 1 along x (nearest site in the row), pass 2
//                          along y (lower envelope of parabolas) in shared memory -> uint16 plane of the caller's workspace;
//                          blocks z < n also bit-pack voxel row j = z of their grid along z (one uint64 per (j, i) column).
//   surface_count_kernel   pass 3 along z, only on the lattice columns holding query sites of the other surface, fused with
//                          the counters: registers -> warp shuffle -> shared memory -> one 64-bit atomic per counter per
//                          block; no block spans two (sample, t, direction) slices, so the sums do not depend on launch order.
// Grid 0 of a sample is the GT surface, grid 1 + t the prediction at threshold t.  Both lower envelopes are the integer
// form of Felzenszwalb & Huttenlocher's (Meijster et al.'s separation): exact, O(2n+1) per line.
#include "common.cuh"

namespace s3d {
namespace {

constexpr int kSurfThreads = 128;
constexpr int kSurfMaxN = 64;
constexpr unsigned kNoSite = 0xFFFFu;     // workspace value: no site on this line / plane

struct KBound { int k[kMaxThresh]; };

// Lower envelope of the parabolas (x - u)^2 + f(u) over u in [0, m) with f(u) != kNoSite.  Stack entry e (in st[e * stride])
// = f << 16 | start << 8 | u: parabola u is the lowest for integer x in [start, next entry's start).  -> entries.
template <typename Load>
__device__ __forceinline__ int envelope(Load f, int m, uint32_t* st, int stride) {
  int k = 0;
  for (int u = 0; u < m; ++u) {
    const int fu = (int)f(u);
    if (fu == (int)kNoSite) continue;
    int w = 0;
    while (k > 0) {
      const uint32_t e = st[(k - 1) * stride];
      const int v = e & 0xFF, tv = (e >> 8) & 0xFF, fv = (int)(e >> 16);
      if ((tv - v) * (tv - v) + fv < (tv - u) * (tv - u) + fu) {
        // v is strictly lower at its start: the last x where v is still <= u (the numerator is >= tv * den >= 0)
        w = 1 + (u * u - v * v + fu - fv) / (2 * (u - v));
        break;
      }
      --k;
    }
    if (k == 0 || w < m) { st[k * stride] = (uint32_t)fu << 16 | (uint32_t)(k == 0 ? 0 : w) << 8 | (uint32_t)u;  ++k; }
  }
  return k;
}

__device__ __forceinline__ bool occupied(const float* fused, const uint8_t* gt, int grid, const Thresh& th, int64_t i) {
  return grid == 0 ? gt[i] != 0 : fused[i] >= th.t[grid - 1];          // NaN >= t is false: empty, as for the IoU
}

__global__ void __launch_bounds__(kSurfThreads)
surface_plane_kernel(const float* __restrict__ fused, const uint8_t* __restrict__ gt, int n, int G, Thresh th,
                     unsigned long long* __restrict__ pack, uint16_t* __restrict__ dt) {
  extern __shared__ uint32_t smem[];
  const int m = 2 * n + 1, nn = n * n;
  const int z = blockIdx.x % m, grid = (blockIdx.x / m) % G, b = blockIdx.x / (m * G);
  const int64_t vox0 = (int64_t)b * nn * n;
  const float* fb = fused + vox0;
  const uint8_t* gb = gt + vox0;
  uint8_t* occ = reinterpret_cast<uint8_t*>(smem);                     // [2][n][n]: voxel slices z/2 - 1 and z/2 (z even),
  uint16_t* g1 = reinterpret_cast<uint16_t*>(occ + ((2 * nn + 3) & ~3));  // (z - 1)/2 (z odd); then [m][m] pass 1
  uint32_t* st = reinterpret_cast<uint32_t*>(g1 + ((m * m + 1) & ~1));  // [m][threads] envelope stacks
  const int k0 = (z & 1) ? (z - 1) / 2 : z / 2 - 1;                     // slice in occ[0]; occ[1] = k0 + 1 (z even)
  for (int e = threadIdx.x; e < 2 * nn; e += blockDim.x) {
    const int k = k0 + e / nn;
    occ[e] = (k >= 0 && k < n) ? occupied(fb, gb, grid, th, (int64_t)k * nn + e % nn) : 0;
  }
  if (z < n) {                                                          // bit-pack voxel row j = z along the column axis
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      unsigned long long w = 0;
      for (int k = 0; k < n; ++k) w |= (unsigned long long)occupied(fb, gb, grid, th, ((int64_t)k * n + z) * n + i) << k;
      pack[((int64_t)b * G + grid) * nn + (int64_t)z * n + i] = w;
    }
  }
  __syncthreads();
  // face site at (z, y, x) of this plane: exactly one even coordinate, the voxels on its two sides differ
  auto site = [&](int y, int x) -> bool {
    if (z & 1) {
      if ((y & 1) == (x & 1)) return false;
      const uint8_t* s = occ;
      if (y & 1) { const int j = y >> 1, i = x >> 1; return (i > 0 ? s[j * n + i - 1] : 0) != (i < n ? s[j * n + i] : 0); }
      const int j = y >> 1, i = x >> 1;
      return (j > 0 ? s[(j - 1) * n + i] : 0) != (j < n ? s[j * n + i] : 0);
    }
    if (!((y & 1) && (x & 1))) return false;
    const int e = (y >> 1) * n + (x >> 1);
    return occ[e] != occ[nn + e];
  };
  // pass 1, along x: squared distance to the nearest site of the row
  for (int y = threadIdx.x; y < m; y += blockDim.x) {
    uint16_t* row = g1 + y * m;
    int last = -1;
    for (int x = 0; x < m; ++x) {
      if (site(y, x)) last = x;
      row[x] = last < 0 ? (uint16_t)kNoSite : (uint16_t)((x - last) * (x - last));
    }
    int next = -1;
    for (int x = m - 1; x >= 0; --x) {
      if (row[x] == 0) next = x;
      if (next >= 0 && (next - x) * (next - x) < row[x]) row[x] = (uint16_t)((next - x) * (next - x));
    }
  }
  __syncthreads();
  // pass 2, along y: lower envelope of g1[., x] -> the plane's squared distances, <= 2 (2n)^2 < kNoSite
  uint16_t* out = dt + (((int64_t)b * G + grid) * m + z) * m * m;
  for (int x = threadIdx.x; x < m; x += blockDim.x) {
    uint32_t* s = st + threadIdx.x;
    const int k = envelope([&](int y) { return g1[y * m + x]; }, m, s, blockDim.x);
    int j = 0;
    for (int y = 0; y < m; ++y) {
      unsigned v = kNoSite;
      if (k) {
        while (j + 1 < k && (int)((s[(j + 1) * blockDim.x] >> 8) & 0xFF) <= y) ++j;
        const uint32_t e = s[j * blockDim.x];
        const int u = e & 0xFF;
        v = (unsigned)((y - u) * (y - u)) + (e >> 16);
      }
      out[y * m + x] = (uint16_t)v;
    }
  }
}

// Query sites of column (y, x) of a packed grid: bit k of *bits = site at z = 2k + par; *top = the site at z = 2n (par 0).
__device__ __forceinline__ int column_sites(const unsigned long long* P, int n, int y, int x, unsigned long long* bits, int* top) {
  *top = 0;
  *bits = 0;
  if ((y & 1) && (x & 1)) {                                             // z-faces between voxels k - 1 and k, k = 0..n
    const unsigned long long w = P[(y >> 1) * n + (x >> 1)];
    *bits = (w ^ (w << 1)) & (n == 64 ? ~0ull : (1ull << n) - 1);
    *top = (int)((w >> (n - 1)) & 1);
    return 0;
  }
  if ((y & 1) == (x & 1)) return 0;
  const int j = y >> 1, i = x >> 1;
  if (y & 1) *bits = (i > 0 ? P[j * n + i - 1] : 0) ^ (i < n ? P[j * n + i] : 0);   // x-faces
  else       *bits = (j > 0 ? P[(j - 1) * n + i] : 0) ^ (j < n ? P[j * n + i] : 0); // y-faces
  return 1;
}

__global__ void __launch_bounds__(kSurfThreads)
surface_count_kernel(const unsigned long long* __restrict__ pack, const uint16_t* __restrict__ dt, int n, int T, int nchunk,
                     KBound kb, int F, unsigned long long* __restrict__ stats) {
  extern __shared__ uint32_t smem[];
  const int m = 2 * n + 1, G = T + 1;
  const int chunk = blockIdx.x % nchunk;
  const int slice = blockIdx.x / nchunk;                                 // (b, t, dir)
  const int dir = slice & 1, t = (slice >> 1) % T, b = (slice >> 1) / T;
  const int qg = dir == 0 ? 1 + t : 0, sg = dir == 0 ? 0 : 1 + t;        // query surface, searched surface
  unsigned long long sum_s = 0, sum_q = 0;
  unsigned npts = 0, cnt[kMaxThresh] = {};
  const int c = chunk * blockDim.x + threadIdx.x;
  if (c < m * m) {
    const int y = c / m, x = c % m;
    unsigned long long bits;
    int top;
    const int par = column_sites(pack + ((int64_t)b * G + qg) * n * n, n, y, x, &bits, &top);
    if (bits || top) {
      npts = __popcll(bits) + top;
      const uint16_t* col = dt + ((int64_t)b * G + sg) * m * m * m + c;
      uint32_t* s = smem + threadIdx.x;
      const int k = envelope([&](int zz) { return col[(int64_t)zz * m * m]; }, m, s, blockDim.x);
      if (k) {                                                           // else the other surface is empty: n_pts only
        int j = 0;
        while (bits || top) {                                            // the sites in increasing z
          int z;
          if (bits) { z = 2 * (__ffsll((long long)bits) - 1) + par;  bits &= bits - 1; }
          else { z = 2 * n;  top = 0; }
          while (j + 1 < k && (int)((s[(j + 1) * blockDim.x] >> 8) & 0xFF) <= z) ++j;
          const uint32_t e = s[j * blockDim.x];
          const int u = e & 0xFF;
          const unsigned d = (unsigned)((z - u) * (z - u)) + (e >> 16);
          sum_s += d;
          sum_q += (unsigned long long)__float2ll_rn(__fsqrt_rn((float)d) * 4294967296.f);   // exact product in fp32
#pragma unroll
          for (int f = 0; f < kMaxThresh; ++f)
            if (f < F) cnt[f] += (int)d < kb.k[f];
        }
      }
    }
  }
  constexpr int kN = 3 + kMaxThresh;
  __shared__ unsigned long long acc[kN];
  if (threadIdx.x < kN) acc[threadIdx.x] = 0;
  __syncthreads();
  unsigned long long v[kN];
  v[0] = npts;  v[1] = sum_s;  v[2] = sum_q;
#pragma unroll
  for (int f = 0; f < kMaxThresh; ++f) v[3 + f] = cnt[f];
  const int nc = 3 + F;
#pragma unroll
  for (int i = 0; i < kN; ++i) {
    if (i >= nc) break;
    unsigned long long a = v[i];
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if ((threadIdx.x & 31) == 0 && a) atomicAdd(&acc[i], a);
  }
  __syncthreads();
  if ((int)threadIdx.x < nc && acc[threadIdx.x]) atomicAdd(stats + (int64_t)slice * nc + threadIdx.x, acc[threadIdx.x]);
}

int64_t pack_bytes(int B, int T, int n) { return (int64_t)B * (T + 1) * n * n * 8; }
int64_t grid_bytes(int B, int T, int n) { const int64_t m = 2 * n + 1; return (int64_t)B * (T + 1) * m * m * m * 2; }

}  // namespace
}  // namespace s3d

using namespace s3d;

extern "C" int64_t s3d_voxel_surface_workspace_bytes(int B, int T, int n) {
  if (B < 0 || T < 0 || n < 1 || n > kSurfMaxN) return -1;
  return pack_bytes(B, T, n) + grid_bytes(B, T, n);
}

extern "C" int s3d_voxel_surface_eval(const float* fused, const uint8_t* gt, int B, int n, const float* thresholds, int T,
                                      const int* kbound, int F, long long* stats, void* workspace, int64_t workspace_bytes,
                                      void* stream) {
  if (!fused || !gt || !stats || (T > 0 && !thresholds) || (F > 0 && !kbound)) {
    set_error("voxel_surface_eval: null argument");
    return S3D_ERR_INVALID;
  }
  S3D_CHECK_ARG(n >= 1 && n <= kSurfMaxN, "voxel_surface_eval: n must be in [1, %d], got %d", kSurfMaxN, n);
  S3D_CHECK_ARG(B >= 0, "voxel_surface_eval: B must be >= 0, got %d", B);
  S3D_CHECK_ARG(T >= 0 && T <= kMaxThresh, "voxel_surface_eval: T must be in [0, %d], got %d", kMaxThresh, T);
  S3D_CHECK_ARG(F >= 0 && F <= kMaxThresh, "voxel_surface_eval: F must be in [0, %d], got %d", kMaxThresh, F);
  const int kmax = 3 * (2 * n) * (2 * n) + 1;
  Thresh th;
  KBound kb;
  for (int i = 0; i < kMaxThresh; ++i) {
    th.t[i] = i < T ? thresholds[i] : 0.f;
    kb.k[i] = i < F ? kbound[i] : 0;
    S3D_CHECK_ARG(i >= F || (kb.k[i] >= 0 && kb.k[i] <= kmax), "voxel_surface_eval: kbound[%d] must be in [0, %d], got %d",
                  i, kmax, kb.k[i]);
  }
  const int64_t need = s3d_voxel_surface_workspace_bytes(B, T, n);
  if (B == 0 || T == 0) return S3D_OK;
  S3D_CHECK_ARG(workspace && workspace_bytes >= need, "voxel_surface_eval: workspace of %lld bytes, need %lld",
                (long long)workspace_bytes, (long long)need);
  S3D_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 7) == 0, "voxel_surface_eval: workspace must be 8-byte aligned");
  const int m = 2 * n + 1, G = T + 1;
  S3D_CHECK_ARG((int64_t)B * G * m < (1ll << 31), "voxel_surface_eval: grid too large");
  auto* pack = static_cast<unsigned long long*>(workspace);
  auto* dt = reinterpret_cast<uint16_t*>(static_cast<char*>(workspace) + pack_bytes(B, T, n));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int stack_bytes = m * kSurfThreads * 4;
  const int smem1 = ((2 * n * n + 3) & ~3) + ((m * m + 1) & ~1) * 2 + stack_bytes;
  S3D_CUDA(cudaFuncSetAttribute(surface_plane_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem1));
  surface_plane_kernel<<<(unsigned)((int64_t)B * G * m), kSurfThreads, smem1, st>>>(fused, gt, n, G, th, pack, dt);
  S3D_LAUNCH_CHECK();
  const int nchunk = ceil_div(m * m, kSurfThreads);
  S3D_CHECK_ARG((int64_t)B * T * 2 * nchunk < (1ll << 31), "voxel_surface_eval: grid too large");
  S3D_CUDA(cudaFuncSetAttribute(surface_count_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, stack_bytes));
  surface_count_kernel<<<(unsigned)((int64_t)B * T * 2 * nchunk), kSurfThreads, stack_bytes, st>>>(
      pack, dt, n, T, nchunk, kb, F, reinterpret_cast<unsigned long long*>(stats));
  S3D_LAUNCH_CHECK();
  return S3D_OK;
}
