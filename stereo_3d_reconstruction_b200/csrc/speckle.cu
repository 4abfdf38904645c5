// Speckle filter of the two disparity maps (s3d_speckle_filter): the connected components of every map's candidate pixels,
// their sizes, and the mask of the pixels whose component is larger than max_size, with the counters of the kept pixels.
// Definitions (candidate, adjacency, region, mask, counters) in include/s3d.h.
//
// Block-based union-find (Playne & Hawick; Allegretti et al.'s BUF), four launches.  The workspace holds a label (a parent
// index inside the map, -1 for a non-candidate) and a size slot per pixel.  A parent only ever decreases and stays inside its
// component, so whatever order the unions run in, every root ends as its component's smallest index: the partition, the
// sizes and every counter are unique, and the result does not depend on scheduling or on the batch split.
//   1. speckle_local_kernel: a block per 32 x 32 tile of one map.  The tile's disparities and labels go to shared memory,
//      its 4-neighbour edges are united there (lock-free: link the larger root to the smaller with atomicMin, retry when
//      another thread moved it first), and each pixel's tile root, as a map index, is written to the labels.  The tile roots
//      zero their size slots: only they can be roots after the merge.
//   2. speckle_border_kernel: a thread per 4-neighbour edge that crosses a tile border, the same union on the global labels.
//   3. speckle_size_kernel: each candidate finds its root, stores it, and adds 1 to the root's size; the adds of a warp are
//      aggregated per root with __match_any_sync, so a map that is one region costs one atomic per warp, not per pixel.
//   4. speckle_finish_kernel: the mask and the counters.  No block spans two maps: per-thread integer counters, reduced over
//      the block, then one 64-bit atomic per counter per block.
#include "common.cuh"

namespace s3d {
namespace {

constexpr int kTile = 32;                      // side of a tile of the local pass
constexpr int kThreads = 256;
constexpr int kTileRows = kThreads / kTile;    // thread rows of a local block: a thread takes every kTileRows-th row
constexpr int kPix = 4;                        // pixels per thread of the size pass
constexpr int kFinPix = 8;                     // pixels per thread of the finish pass
constexpr int kNumCounters = 5 + kMaxThresh;   // [n_kept, n_valid_kept, epe_fx, bad_t x 8, n_speckles, n_speckle_px]

struct SpeckleIn {
  const float* disp;     // [2B,H,W], view-major: map m = v * B + b
  const uint8_t* lr;     // [B,2,H,W] or NULL
  int B, H, W;
  float max_diff;
};

__device__ __forceinline__ bool adjacent(float a, float b, float max_diff) {
  return fabsf(__fsub_rn(a, b)) <= max_diff;                 // one rounding, no contraction
}

// Root of x: the parents are followed to a fixed point.  Volatile: other threads lower parents while this one reads.
__device__ __forceinline__ int find_root(const volatile int* L, int x) {
  int p = L[x];
  while (p != x) {
    x = p;
    p = L[x];
  }
  return x;
}

// Lock-free union of the components of a and b (shared or global labels).  atomicMin links the larger root to the smaller;
// when the larger one stopped being a root first, atomicMin returns its new parent and the union goes on from there.
__device__ __forceinline__ void unite(int* L, int a, int b) {
  for (;;) {
    a = find_root(L, a);
    b = find_root(L, b);
    if (a == b) return;
    if (a > b) {
      const int t = a;
      a = b;
      b = t;
    }
    const int old = atomicMin(L + b, a);
    if (old == b) return;
    b = old;
  }
}

// A warp per tile row (lane = column).  Horizontal links come from ballots: each pixel starts labelled with the first pixel of
// its run (the pixels linked to their left neighbours), so a row costs no atomics.  A vertical edge is united only where it
// starts a stretch: when the edge at x - 1 is linked and x is linked to x - 1 in both rows, the edge at x joins nothing new.
// A constant tile so takes 31 unions instead of 1984.
__global__ void __launch_bounds__(kThreads)
speckle_local_kernel(SpeckleIn a, int tiles_x, int* __restrict__ labels, int* __restrict__ sizes) {
  __shared__ int sl[kTile * kTile];            // tile-local labels, -1 for a non-candidate
  __shared__ float sd[kTile * kTile];
  __shared__ unsigned sc[kTile], sh[kTile];    // per row: candidate bits, bits of the pixels linked to their left neighbour
  const int m = blockIdx.y, b = m % a.B, v = m / a.B;
  const int tx0 = (blockIdx.x % tiles_x) * kTile, ty0 = (blockIdx.x / tiles_x) * kTile;
  const int lx = threadIdx.x % kTile, ly0 = threadIdx.x / kTile, x = tx0 + lx;
  const unsigned upto = lx == 31 ? 0xffffffffu : (2u << lx) - 1u;         // bits 0 .. lx
  const int64_t HW = (int64_t)a.H * a.W;
  const float* dm = a.disp + m * HW;
  const uint8_t* lm = a.lr ? a.lr + ((int64_t)b * 2 + v) * HW : nullptr;
#pragma unroll
  for (int ly = ly0; ly < kTile; ly += kTileRows) {
    const int y = ty0 + ly, i = ly * kTile + lx;
    float d = 0.f;
    bool c = false;
    if (x < a.W && y < a.H) {
      const int64_t p = (int64_t)y * a.W + x;
      d = __ldg(dm + p);
      c = isfinite(d) && (!lm || __ldg(lm + p) == 1);
    }
    const float dl = __shfl_up_sync(0xffffffffu, d, 1);
    const unsigned cb = __ballot_sync(0xffffffffu, c);
    const unsigned hb = __ballot_sync(0xffffffffu, lx > 0 && c && ((cb >> (lx - 1)) & 1u) && adjacent(d, dl, a.max_diff));
    sd[i] = d;
    sl[i] = c ? ly * kTile + 31 - __clz(~hb & upto) : -1;                // the highest unlinked pixel at or left of lx
    if (lx == 0) {
      sc[ly] = cb;
      sh[ly] = hb;
    }
  }
  __syncthreads();
#pragma unroll
  for (int ly = ly0; ly < kTile; ly += kTileRows) {
    if (ly == 0) continue;
    const int i = ly * kTile + lx;
    const unsigned vb = __ballot_sync(0xffffffffu, ((sc[ly] & sc[ly - 1]) >> lx) & 1u &&
                                                   adjacent(sd[i], sd[i - kTile], a.max_diff));
    const unsigned redundant = vb & (vb << 1) & sh[ly] & sh[ly - 1];
    if (((vb & ~redundant) >> lx) & 1u) unite(sl, i, i - kTile);
  }
  __syncthreads();
#pragma unroll
  for (int ly = ly0; ly < kTile; ly += kTileRows) {
    const int y = ty0 + ly, i = ly * kTile + lx;
    if (x >= a.W || y >= a.H) continue;
    const int64_t p = (int64_t)y * a.W + x;
    int g = -1;
    if (sl[i] >= 0) {
      const int r = find_root(sl, i);
      g = (ty0 + r / kTile) * a.W + tx0 + r % kTile;    // raster order inside the tile is raster order in the map
      if (r == i) sizes[m * HW + p] = 0;
    }
    labels[m * HW + p] = g;
  }
}

// Edge e of a map: e < n_vert crosses a vertical border (pixel at x = k * kTile, k >= 1, and its left neighbour), the others
// a horizontal one (pixel at y = k * kTile and its upper neighbour).
__global__ void __launch_bounds__(kThreads)
speckle_border_kernel(SpeckleIn a, int tiles_x, int64_t n_vert, int64_t n_edges, int* __restrict__ labels) {
  const int64_t e = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (e >= n_edges) return;
  const int m = blockIdx.y;
  int p, q;
  if (e < n_vert) {
    const int y = (int)(e / (tiles_x - 1)), k = (int)(e % (tiles_x - 1)) + 1;
    p = y * a.W + k * kTile;
    q = p - 1;
  } else {
    const int64_t f = e - n_vert;
    const int k = (int)(f / a.W) + 1, x = (int)(f % a.W);
    p = k * kTile * a.W + x;
    q = p - a.W;
  }
  const int64_t HW = (int64_t)a.H * a.W;
  int* L = labels + m * HW;
  if (((const volatile int*)L)[p] < 0 || ((const volatile int*)L)[q] < 0) return;
  const float* dm = a.disp + m * HW;
  if (!adjacent(__ldg(dm + p), __ldg(dm + q), a.max_diff)) return;
  unite(L, p, q);
}

__global__ void __launch_bounds__(kThreads)
speckle_size_kernel(int64_t HW, int* __restrict__ labels, int* __restrict__ sizes) {
  const int m = blockIdx.y;
  int* L = labels + m * HW;
  int* S = sizes + m * HW;
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int j = 0; j < kPix; ++j) {
    const int64_t p = ((int64_t)blockIdx.x * kPix + j) * kThreads + threadIdx.x;
    int r = -1;
    if (p < HW) {
      const int l = L[p];
      if (l >= 0) {
        r = find_root(L, l);                   // no union runs now: the roots are final
        if (r != l) L[p] = r;
      }
    }
    const unsigned peers = __match_any_sync(0xffffffffu, r);
    if (r >= 0 && lane == __ffs(peers) - 1) atomicAdd(S + r, __popc(peers));
  }
}

__global__ void __launch_bounds__(kThreads)
speckle_finish_kernel(SpeckleIn a, const float* __restrict__ gt, Thresh th, int nT, float max_gt, int max_size,
                      const int* __restrict__ labels, const int* __restrict__ sizes, uint8_t* __restrict__ mask,
                      unsigned long long* __restrict__ stats) {
  __shared__ unsigned long long blk[kNumCounters];
  const int m = blockIdx.y, b = m % a.B, v = m / a.B;
  const int64_t HW = (int64_t)a.H * a.W, img = ((int64_t)b * 2 + v) * HW;
  const int* L = labels + m * HW;
  const int* S = sizes + m * HW;
  unsigned n_kept = 0, n_valid = 0, n_spk = 0, n_spk_px = 0, bad[kMaxThresh] = {};
  unsigned long long epe = 0;
  // every load of the block's pixels is issued before any result is needed: labels, then the roots' sizes, then GT and disp
  int64_t p[kFinPix];
  int r[kFinPix], sz[kFinPix];
  float g[kFinPix], d[kFinPix];
#pragma unroll
  for (int j = 0; j < kFinPix; ++j) {
    p[j] = ((int64_t)blockIdx.x * kFinPix + j) * kThreads + threadIdx.x;
    r[j] = p[j] < HW ? __ldg(L + p[j]) : -1;                             // the root, stored by the size pass
  }
#pragma unroll
  for (int j = 0; j < kFinPix; ++j) {
    sz[j] = r[j] >= 0 ? __ldg(S + r[j]) : 0;
    g[j] = gt && p[j] < HW ? __ldg(gt + img + p[j]) : 0.f;
    d[j] = gt && p[j] < HW ? __ldg(a.disp + m * HW + p[j]) : 0.f;
  }
#pragma unroll
  for (int j = 0; j < kFinPix; ++j) {
    if (p[j] >= HW) break;
    const bool kept = r[j] >= 0 && sz[j] > max_size;
    if (r[j] >= 0 && !kept) {
      ++n_spk_px;
      n_spk += r[j] == p[j];                     // a region's root is its smallest index: counted once
    }
    mask[img + p[j]] = kept;
    if (!kept) continue;
    ++n_kept;
    if (!gt || !(isfinite(g[j]) && g[j] >= 0.f && g[j] < max_gt)) continue;
    const float e = fabsf(__fsub_rn(d[j], g[j]));
    ++n_valid;
    epe += (unsigned long long)__float2ll_rn(e * 65536.f);      // exact scaling by 2^16, then round half to even
#pragma unroll
    for (int t = 0; t < kMaxThresh; ++t)
      if (t < nT) bad[t] += e > th.t[t];
  }
  if (threadIdx.x < kNumCounters) blk[threadIdx.x] = 0;
  __syncthreads();
  unsigned long long c[kNumCounters];
  c[0] = n_kept;  c[1] = n_valid;  c[2] = epe;
#pragma unroll
  for (int t = 0; t < kMaxThresh; ++t) c[3 + t] = bad[t];
  c[3 + kMaxThresh] = n_spk;  c[4 + kMaxThresh] = n_spk_px;
#pragma unroll
  for (int k = 0; k < kNumCounters; ++k) {
    if (k >= 3 + nT && k < 3 + kMaxThresh) continue;
    unsigned long long s = c[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0 && s) atomicAdd(&blk[k], s);
  }
  __syncthreads();
  // counter k -> column k of the row [n_kept, n_valid_kept, epe_fx, bad_t x nT, n_speckles, n_speckle_px]
  const int k = threadIdx.x;
  if (k < kNumCounters && blk[k] && (k < 3 + nT || k >= 3 + kMaxThresh)) {
    const int col = k < 3 + nT ? k : k - kMaxThresh + nT;
    atomicAdd(stats + ((int64_t)b * 2 + v) * (5 + nT) + col, blk[k]);
  }
}

bool aligned(const void* p, int n) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) % n) == 0; }

}  // namespace
}  // namespace s3d

using namespace s3d;

extern "C" int64_t s3d_speckle_filter_workspace_bytes(int B, int H, int W) {
  if (B < 0 || H < 0 || W < 0) return 0;
  return (int64_t)2 * B * H * (int64_t)W * 2 * (int64_t)sizeof(int);        // labels + sizes, int32 per pixel each
}

extern "C" int s3d_speckle_filter(const float* disp, int B, int H, int W, const uint8_t* lr_mask, int max_size,
                                  float max_diff, const float* gt, const float* thresholds, int T, float max_gt,
                                  uint8_t* mask, long long* stats, void* workspace, int64_t workspace_bytes, void* stream) {
  if (!disp || !mask || !stats || (T > 0 && !thresholds)) {
    set_error("speckle_filter: null argument");
    return S3D_ERR_INVALID;
  }
  S3D_CHECK_ARG(B >= 0 && 2 * (int64_t)B < 65536 && H >= 1 && W >= 1,
                "speckle_filter: need 0 <= B < 32768, H >= 1, W >= 1, got %d %d %d", B, H, W);
  S3D_CHECK_ARG((int64_t)H * W < (1ll << 31), "speckle_filter: H W must be < 2^31, got H = %d, W = %d", H, W);
  S3D_CHECK_ARG(max_size >= 0, "speckle_filter: max_size must be >= 0, got %d", max_size);
  S3D_CHECK_ARG(isfinite(max_diff) && max_diff >= 0.f, "speckle_filter: max_diff must be finite and >= 0, got %g",
                (double)max_diff);
  S3D_CHECK_ARG(T >= 0 && T <= kMaxThresh, "speckle_filter: T must be in [0, 8], got %d", T);
  S3D_CHECK_ARG(!gt || max_gt > 0.f, "speckle_filter: max_gt must be > 0 with gt");
  const int64_t need = s3d_speckle_filter_workspace_bytes(B, H, W);
  S3D_CHECK_ARG(workspace_bytes >= need && (need == 0 || workspace),
                "speckle_filter: workspace of %lld bytes, need %lld", (long long)workspace_bytes, (long long)need);
  S3D_CHECK_ARG(aligned(workspace, 4), "speckle_filter: workspace must be 4-byte aligned");
  if (B == 0) return S3D_OK;
  Thresh th;
  for (int t = 0; t < kMaxThresh; ++t) th.t[t] = gt && t < T ? thresholds[t] : 0.f;
  const SpeckleIn in{disp, lr_mask, B, H, W, max_diff};
  const int64_t HW = (int64_t)H * W;
  int* labels = static_cast<int*>(workspace);
  int* sizes = labels + 2 * B * HW;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int tiles_x = ceil_div(W, kTile), tiles_y = ceil_div(H, kTile);
  const unsigned maps = 2u * (unsigned)B;
  speckle_local_kernel<<<dim3((unsigned)tiles_x * tiles_y, maps), kThreads, 0, st>>>(in, tiles_x, labels, sizes);
  S3D_LAUNCH_CHECK();
  const int64_t n_vert = (int64_t)(tiles_x - 1) * H, n_edges = n_vert + (int64_t)(tiles_y - 1) * W;
  const int64_t gb = n_edges > 0 ? ceil_div64(n_edges, kThreads) : 1;       // a tile-sized map has no border: 4 launches still
  speckle_border_kernel<<<dim3((unsigned)gb, maps), kThreads, 0, st>>>(in, tiles_x, n_vert, n_edges, labels);
  S3D_LAUNCH_CHECK();
  const dim3 grid((unsigned)ceil_div64(HW, kPix * kThreads), maps);
  speckle_size_kernel<<<grid, kThreads, 0, st>>>(HW, labels, sizes);
  S3D_LAUNCH_CHECK();
  speckle_finish_kernel<<<dim3((unsigned)ceil_div64(HW, kFinPix * kThreads), maps), kThreads, 0, st>>>(in, gt, th, T, max_gt, max_size, labels, sizes, mask,
                                                   reinterpret_cast<unsigned long long*>(stats));
  S3D_LAUNCH_CHECK();
  return S3D_OK;
}
