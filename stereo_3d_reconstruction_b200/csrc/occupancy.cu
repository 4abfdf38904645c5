// Threshold-free occupancy evaluation (s3d_occupancy_curves): per-sample histograms of the clamped prediction split by GT
// label, and fixed-point BCE / Brier sums.  Definitions in include/s3d.h.
//
// One cluster of kOccSplit blocks per sample.  Each block takes one contiguous slice of the sample, streams it with 16-byte
// loads (kOccUnroll in flight per thread) and builds a partial histogram in its shared memory.  The predictions of one sample
// often fall into one or two bins, so the updates are warp-aggregated: lanes with the same (bin, label) find each other with
// __match_any_sync, and one lane per group adds the group's count and its summed q(v) (at most 32 * 2^20, 32 bits), so a
// warp makes at most one shared atomic per distinct key instead of 32 on one address.  A block's per-bin sum of q(v) can
// exceed 32 bits; a 64-bit shared atomicAdd is a CAS loop on this architecture, so the sum is kept as two 32-bit words: the
// native 32-bit add returns the old low word, and the lane that wraps it adds the carry to the high word.  After a cluster
// barrier, block r sums bins r * blockDim + t over the cluster's shared memories (DSMEM) and writes them; block 0 writes the
// two loss sums.
// Every counter is written, not added: no global atomics, no zeroing, one launch, integer sums (deterministic).
#include <cooperative_groups.h>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace s3d {
namespace {

constexpr int kOccThreads = 256;
constexpr int kOccSplit = 8;            // blocks (one cluster) per sample
constexpr int kOccUnroll = 4;           // units loaded per thread before any is processed
constexpr int kOccMaxBins = 1024;
constexpr double kOccFx = 1048576.0;    // 2^20

struct OccAcc {
  long long bce = 0, brier = 0;
};

// one voxel: c clamped value, g GT label; valid is warp-divergent, the warp calls this together
__device__ __forceinline__ void occ_voxel(float v, bool g, bool valid, int K, unsigned* cnt, unsigned* qlo, unsigned* qhi,
                                          OccAcc& acc) {
  const float c = fminf(fmaxf(v, 0.f), 1.f);                             // NaN -> 0 (fmaxf), then [0, 1]
  const int k = min((int)(c * (float)K), K - 1);                         // c * K is exact: K is a power of two
  const int key = valid ? (k << 1 | (int)g) : -1;
  const unsigned grp = __match_any_sync(0xffffffffu, key);
  const double cd = (double)c;
  const unsigned q = valid ? (unsigned)__double2int_rn(__dmul_rn(cd, kOccFx)) : 0u;
  const unsigned s = __reduce_add_sync(grp, q);
  if (!valid) return;
  if ((threadIdx.x & 31) == __ffs(grp) - 1) {
    atomicAdd(cnt + (g ? K : 0) + k, (unsigned)__popc(grp));
    if (atomicAdd(qlo + k, s) > ~s) atomicAdd(qhi + k, 1u);          // old + s wraps past 2^32
  }
  const double x = g ? cd : __dsub_rn(1.0, cd);                          // exact in fp64
  const double bce = -fmax(log(x), -100.0);                              // PyTorch's BCELoss clamp; log(0) = -inf
  acc.bce += __double2ll_rn(__dmul_rn(bce, kOccFx));
  const double d = __dsub_rn(cd, g ? 1.0 : 0.0);
  acc.brier += __double2ll_rn(__dmul_rn(__dmul_rn(d, d), kOccFx));
}

__device__ __forceinline__ long long warp_sum_ll(long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// kVec: 4 voxels per unit (float4 + uchar4 loads; nvox % 4 == 0, aligned pointers), else 1
template <bool kVec>
__global__ void __cluster_dims__(kOccSplit, 1, 1) __launch_bounds__(kOccThreads)
occupancy_curves_kernel(const float* __restrict__ fused, const uint8_t* __restrict__ gt, int nvox, int K,
                        long long* __restrict__ hist, long long* __restrict__ loss) {
  constexpr int W = kVec ? 4 : 1;
  extern __shared__ unsigned occ_smem[];
  unsigned* qlo = occ_smem;                                              // [K]   sum q(v) per bin: low 32 bits
  unsigned* qhi = qlo + K;                                               // [K]   and the carries out of them
  unsigned* cnt = qhi + K;                                               // [2K]  counts, label 0 then label 1
  __shared__ long long part[2][kOccThreads / 32];
  __shared__ long long blk_loss[2];
  cg::cluster_group cluster = cg::this_cluster();
  const int r = (int)cluster.block_rank();
  const int b = blockIdx.x / kOccSplit;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int e = threadIdx.x; e < 4 * K; e += blockDim.x) occ_smem[e] = 0;
  __syncthreads();

  // this block's slice of the sample, in units of W voxels
  const int units = nvox / W;
  const int per = (units + kOccSplit - 1) / kOccSplit;
  const int u0 = min(r * per, units), u1 = min(u0 + per, units);
  const float* f = fused + (int64_t)b * nvox;
  const uint8_t* g8 = gt + (int64_t)b * nvox;
  OccAcc acc;
  for (int base = u0; base < u1; base += kOccUnroll * kOccThreads) {   // trip count uniform over the block
    float v[kOccUnroll][W];
    unsigned gl[kOccUnroll];
#pragma unroll
    for (int j = 0; j < kOccUnroll; ++j) {
      const int u = base + j * kOccThreads + threadIdx.x;
      if (u < u1) {
        if constexpr (kVec) {
          const float4 x = __ldg(reinterpret_cast<const float4*>(f) + u);
          v[j][0] = x.x;  v[j][1] = x.y;  v[j][2] = x.z;  v[j][3] = x.w;
          gl[j] = __ldg(reinterpret_cast<const unsigned*>(g8) + u);
        } else {
          v[j][0] = __ldg(f + u);
          gl[j] = __ldg(g8 + u);
        }
      } else {
#pragma unroll
        for (int e = 0; e < W; ++e) v[j][e] = 0.f;
        gl[j] = 0;
      }
    }
#pragma unroll
    for (int j = 0; j < kOccUnroll; ++j) {
      const bool valid = base + j * kOccThreads + (int)threadIdx.x < u1;
#pragma unroll
      for (int e = 0; e < W; ++e) occ_voxel(v[j][e], ((gl[j] >> (8 * e)) & 0xffu) != 0, valid, K, cnt, qlo, qhi, acc);
    }
  }
  const long long sb = warp_sum_ll(acc.bce), sr = warp_sum_ll(acc.brier);
  if (lane == 0) { part[0][warp] = sb;  part[1][warp] = sr; }
  __syncthreads();
  if (threadIdx.x < 2) {
    long long s = 0;
    for (int w = 0; w < kOccThreads / 32; ++w) s += part[threadIdx.x][w];
    blk_loss[threadIdx.x] = s;
  }
  cluster.sync();                                                        // every partial histogram of the sample is done

  long long* h = hist + (int64_t)b * 3 * K;
  for (int k = r * kOccThreads + threadIdx.x; k < K; k += kOccSplit * kOccThreads) {
    long long c0 = 0, c1 = 0, s = 0;
#pragma unroll
    for (int q = 0; q < kOccSplit; ++q) {
      const unsigned* sm = cluster.map_shared_rank(occ_smem, q);
      s += (long long)sm[K + k] << 32 | sm[k];
      c0 += sm[2 * K + k];  c1 += sm[3 * K + k];
    }
    h[k] = c0;  h[K + k] = c1;  h[2 * K + k] = s;
  }
  if (r == 0 && threadIdx.x < 2) {
    long long s = 0;
#pragma unroll
    for (int q = 0; q < kOccSplit; ++q) s += *cluster.map_shared_rank(&blk_loss[threadIdx.x], q);
    loss[2 * b + threadIdx.x] = s;
  }
  cluster.sync();                                                        // no block leaves while its memory is read
}

}  // namespace
}  // namespace s3d

using namespace s3d;

extern "C" int s3d_occupancy_curves(const float* fused, const uint8_t* gt, int B, int nvox, int K, int64_t* hist,
                                    int64_t* loss, void* stream) {
  if (!fused || !gt || !hist || !loss) {
    set_error("occupancy_curves: null argument");
    return S3D_ERR_INVALID;
  }
  S3D_CHECK_ARG(B >= 0 && B <= INT32_MAX / kOccSplit, "occupancy_curves: B must be in [0, %d], got %d",
                INT32_MAX / kOccSplit, B);
  S3D_CHECK_ARG(nvox >= 1 && nvox <= (1 << 24), "occupancy_curves: nvox must be in [1, 2^24], got %d", nvox);
  S3D_CHECK_ARG(K >= 2 && K <= kOccMaxBins && (K & (K - 1)) == 0,
                "occupancy_curves: K must be a power of two in [2, %d], got %d", kOccMaxBins, K);
  if (B == 0) return S3D_OK;
  const size_t smem = (size_t)K * 4 * sizeof(unsigned);
  const bool vec = nvox % 4 == 0 && reinterpret_cast<uintptr_t>(fused) % 16 == 0 && reinterpret_cast<uintptr_t>(gt) % 4 == 0;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  long long* h = reinterpret_cast<long long*>(hist);
  long long* l = reinterpret_cast<long long*>(loss);
  if (vec)
    occupancy_curves_kernel<true><<<B * kOccSplit, kOccThreads, smem, st>>>(fused, gt, nvox, K, h, l);
  else
    occupancy_curves_kernel<false><<<B * kOccSplit, kOccThreads, smem, st>>>(fused, gt, nvox, K, h, l);
  S3D_LAUNCH_CHECK();
  return S3D_OK;
}
