// Row C: Chamfer nearest-neighbour search (forward), replacing the reference's
// extensions/chamfer_dist CUDA extension (/root/reference/README.md:62-65; its source is on the
// upstream Stereo2Point branch and not on disk).
//
// For every query point: min over the other set of ((dx*dx + dy*dy) + dz*dz), with explicit
// round-to-nearest mul/add (no FMA contraction) so the distances -- and therefore the argmin --
// are bit-identical to the C oracle (oracle/chamfer_ref.c).  Ties go to the lowest index.
//
// Tiled shared-memory min-reduction: the "other" set streams through shared memory in tiles of
// kTile points (float4, broadcast reads); every thread keeps kQ query points and their running
// (best distance, best index) in registers; S lanes of a warp split each tile between them and
// finish with a warp-shuffle lexicographic (distance, index) argmin.  Bound by the fp32 ALU issue
// rate (about 11 instructions per point pair), not by HBM: B*(N+M)*20 bytes move in total.
//
// Symmetric one-pass search (chamfer_sym_kernel, used when the caller provides a workspace and the problem fills the
// chip).  d(i, j) is the same fp32 number in both directions -- (a - b) and (b - a) differ in sign only and are squared --
// so every pair is evaluated ONCE and feeds the row minimum (nearest streamed point of a resident point) and the column
// minimum (nearest resident point of a streamed point):
//   * a lane keeps 8 consecutive points of the LARGER set in registers, packed two to a 64-bit register (FADD2 / FMUL2:
//     8 packed instructions per two pairs); the smaller set streams through shared memory, 8 points per step (broadcast
//     LDS.128), so a step is 64 pairs per lane;
//   * only the minimum VALUES are tracked in the loop (3-input FMNMX3: half an instruction per pair and direction).  Row
//     minima stay in registers; every 32 streamed points a lane notes which rows improved, and at the end of a tile it
//     rescans only that 32-point chunk of each row for the lowest index that attains the minimum (strict '<' between
//     chunks + lowest match inside the chunk = the oracle's scan order);
//   * column minima of a step are reduced over the warp's 256 resident points with a halving shuffle butterfly (9 SHFL +
//     9 FMNMX per 64 pairs) and merged across warps with one 64-bit atomicMin per streamed point on the key
//     (distance bits << 32 | 256-point block): non-negative floats order like their bit patterns, so the key's minimum is
//     the minimum distance at the lowest block; chamfer_sym_finish_kernel rescans that one block for the lowest index.
// About 9.6 issued instructions per pair for BOTH directions against 2 x 11, and 8 of them are the exact arithmetic.
#include <cmath>

#include "common.cuh"

namespace s3d {
namespace {

constexpr int kQ = 4;        // queries per thread
constexpr int kTile = 1024;  // reference points per shared-memory tile
constexpr int kThreads = 256;

__global__ void __launch_bounds__(kThreads)
chamfer_nn_kernel(const float* __restrict__ q_xyz, const float* __restrict__ r_xyz, float* __restrict__ dist,
                  int32_t* __restrict__ idx, int nq, int nr, int S, int blocks_per_batch) {
  __shared__ float4 tile[kTile];
  const int b = blockIdx.x / blocks_per_batch;
  const int blk = blockIdx.x % blocks_per_batch;
  const int s = threadIdx.x % S;                       // slice of the tile this lane scans
  const int group = threadIdx.x / S;                   // query group within the block
  const int groups = kThreads / S;
  const int q0 = (blk * groups + group) * kQ;          // first query of this thread
  const float* qb = q_xyz + (int64_t)b * nq * 3;
  const float* rb = r_xyz + (int64_t)b * nr * 3;

  float qx[kQ], qy[kQ], qz[kQ], best[kQ];
  int bi[kQ];
#pragma unroll
  for (int k = 0; k < kQ; ++k) {
    const int qi = min(q0 + k, nq - 1);
    qx[k] = qb[qi * 3 + 0];  qy[k] = qb[qi * 3 + 1];  qz[k] = qb[qi * 3 + 2];
    best[k] = INFINITY;  bi[k] = 0x7fffffff;
  }

  for (int j0 = 0; j0 < nr; j0 += kTile) {
    const int cnt = min(kTile, nr - j0);
    __syncthreads();
    for (int i = threadIdx.x; i < cnt; i += kThreads) {
      const float* p = rb + (int64_t)(j0 + i) * 3;
      tile[i] = make_float4(p[0], p[1], p[2], 0.f);
    }
    __syncthreads();
#pragma unroll 4
    for (int j = s; j < cnt; j += S) {
      const float4 r = tile[j];
#pragma unroll
      for (int k = 0; k < kQ; ++k) {
        const float dx = __fsub_rn(qx[k], r.x), dy = __fsub_rn(qy[k], r.y), dz = __fsub_rn(qz[k], r.z);
        const float d = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
        if (d < best[k]) { best[k] = d; bi[k] = j0 + j; }
      }
    }
  }
  // lexicographic (distance, index) argmin across the S lanes of the group
#pragma unroll
  for (int k = 0; k < kQ; ++k) {
    for (int o = S >> 1; o > 0; o >>= 1) {
      const float od = __shfl_xor_sync(0xffffffffu, best[k], o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi[k], o);
      if (od < best[k] || (od == best[k] && oi < bi[k])) { best[k] = od; bi[k] = oi; }
    }
    if (s == 0 && q0 + k < nq) {
      dist[(int64_t)b * nq + q0 + k] = best[k];
      idx[(int64_t)b * nq + q0 + k] = bi[k] == 0x7fffffff ? 0 : bi[k];     // nothing compared less (all NaN / +inf): index 0, never out of range
    }
  }
}

// ---- symmetric one-pass search ---------------------------------------------------------------------------------------
constexpr int kSymRMax = 8;              // resident points per lane (template parameter R: 8, or 4 for twice the warps)
constexpr int kSymWarps = 2;             // warps per CTA (they share the staged tile of the streamed set)
constexpr int kSymTile = 2048;           // streamed points per shared-memory tile
constexpr int kSymChunk = 32;            // streamed points between two "which rows improved" checks

__device__ __forceinline__ unsigned long long pack2(float lo, float hi) {
  unsigned long long r;  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));  return r;
}
__device__ __forceinline__ void unpack2(unsigned long long v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ unsigned long long sub2(unsigned long long a, unsigned long long b) {
  unsigned long long r;  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));  return r;
}
// a + b as fma(a, 1, b) with a ONE THE COMPILER CANNOT SEE (a kernel argument): ptxas 12.9 contracts mul.rn.f32x2 +
// add.rn.f32x2 into FFMA2 even with --fmad=false (it honours .rn only on the scalar forms), which would round the sum of
// squares once instead of twice and break bit-exactness.  a * 1 is exact, so this is the add, in one instruction.
__device__ __forceinline__ unsigned long long add2(unsigned long long a, unsigned long long b, unsigned long long one) {
  unsigned long long r;  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(one), "l"(b));  return r;
}
__device__ __forceinline__ unsigned long long mul2(unsigned long long a, unsigned long long b) {
  unsigned long long r;  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));  return r;
}
// min ignoring NaN operands (like the oracle's `d < best`, which a NaN distance never passes)
__device__ __forceinline__ float min3(float a, float b, float c) { float r;  asm("min.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));  return r; }

// Exact distance of one pair, the same operations as the packed ones (IEEE round-to-nearest per lane, no contraction).
__device__ __forceinline__ float pair_dist(float ax, float ay, float az, float bx, float by, float bz) {
  const float dx = __fsub_rn(ax, bx), dy = __fsub_rn(ay, by), dz = __fsub_rn(az, bz);
  return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}

// res_xyz [B, nr, 3]: resident set (rows), str_xyz [B, ns, 3]: streamed set (columns).  Writes the rows' results
// (res_dist, res_idx) and merges the columns' (distance, block) keys into keys[B, ns] (pre-set to all ones).
template <int kSymR>
__global__ void __launch_bounds__(32 * kSymWarps)
chamfer_sym_kernel(const float* __restrict__ res_xyz, const float* __restrict__ str_xyz, float* __restrict__ res_dist,
                   int32_t* __restrict__ res_idx, unsigned long long* __restrict__ keys, int nr, int ns, int ctas_per_batch, float one_arg) {
  constexpr int kSymBlock = 32 * kSymR;  // resident points per warp
  static_assert(kSymChunk == 32, "the cooperative rescan maps lane j to point j of a chunk");
  __shared__ __align__(16) float sx[kSymTile], sy[kSymTile], sz[kSymTile];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int b = blockIdx.x / ctas_per_batch;
  const int rblk = (blockIdx.x % ctas_per_batch) * kSymWarps + warp;       // 256-point block of the resident set
  const int r0 = rblk * kSymBlock + lane * kSymR;
  const float* rb = res_xyz + (int64_t)b * nr * 3;
  const float* sb = str_xyz + (int64_t)b * ns * 3;
  const float nanf_ = __int_as_float(0x7fc00000);
  const unsigned long long one = pack2(one_arg, one_arg);

  // resident points: rows 2p (lo) and 2p + 1 (hi) share a register pair; rows beyond nr are NaN (they never win a minimum)
  unsigned long long qx[kSymR / 2], qy[kSymR / 2], qz[kSymR / 2];
  float best[kSymR], seen[kSymR];
  int cid[kSymR], bidx[kSymR];
#pragma unroll
  for (int p = 0; p < kSymR / 2; ++p) {
    float c[6];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int r = r0 + 2 * p + h;
#pragma unroll
      for (int a = 0; a < 3; ++a) c[3 * h + a] = r < nr ? rb[(int64_t)r * 3 + a] : nanf_;
    }
    qx[p] = pack2(c[0], c[3]);  qy[p] = pack2(c[1], c[4]);  qz[p] = pack2(c[2], c[5]);
  }
#pragma unroll
  for (int k = 0; k < kSymR; ++k) { best[k] = INFINITY;  seen[k] = INFINITY;  bidx[k] = 0; }

  for (int t0 = 0; t0 < ns; t0 += kSymTile) {
    const int cnt = min(kSymTile, ns - t0);
    const int cnt_pad = (cnt + kSymChunk - 1) / kSymChunk * kSymChunk;     // NaN padding to whole chunks
    __syncthreads();
    for (int i = threadIdx.x; i < cnt_pad; i += 32 * kSymWarps) {
      const float* p = sb + (int64_t)(t0 + i) * 3;
      const bool ok = i < cnt;
      sx[i] = ok ? p[0] : nanf_;  sy[i] = ok ? p[1] : nanf_;  sz[i] = ok ? p[2] : nanf_;
    }
    __syncthreads();
    if (rblk * kSymBlock < nr) {                                           // (warp-uniform; a CTA's last warp may have no rows)
#pragma unroll
      for (int k = 0; k < kSymR; ++k) cid[k] = -1;
      // The column minima of a step are reduced ONE STEP LATER (pm / pcol): the shuffle butterfly is a chain of five
      // ~25-cycle round trips, and in the same loop body as the next step's arithmetic it hides behind it.
      float pm[8];
      int pcol = -1;                                                       // first column of the pending step (-1: none)
#pragma unroll
      for (int i = 0; i < 8; ++i) pm[i] = INFINITY;
      auto reduce_pending = [&]() {
        // halve the values a lane carries while doubling the lanes they cover: 9 SHFL + 9 FMNMX for 8 columns x 256 rows
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const bool up = lane & 16;
          const float other = __shfl_xor_sync(0xffffffffu, up ? pm[i] : pm[i + 4], 16);
          pm[i] = fminf(up ? pm[i + 4] : pm[i], other);                    // lanes 16-31 keep columns 4-7
        }
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const bool up = lane & 8;
          const float other = __shfl_xor_sync(0xffffffffu, up ? pm[i] : pm[i + 2], 8);
          pm[i] = fminf(up ? pm[i + 2] : pm[i], other);
        }
        {
          const bool up = lane & 4;
          const float other = __shfl_xor_sync(0xffffffffu, up ? pm[0] : pm[1], 4);
          pm[0] = fminf(up ? pm[1] : pm[0], other);
        }
        pm[0] = fminf(pm[0], __shfl_xor_sync(0xffffffffu, pm[0], 2));
        pm[0] = fminf(pm[0], __shfl_xor_sync(0xffffffffu, pm[0], 1));
        const int col = pcol + (lane >> 2);                                // column of this lane group: bits 4,3,2 of the lane
        if ((lane & 3) == 0 && pcol >= 0 && col < cnt)
          atomicMin(keys + (int64_t)b * ns + t0 + col, ((unsigned long long)__float_as_uint(pm[0]) << 32) | (unsigned)rblk);
      };
      for (int c0 = 0; c0 < cnt_pad; c0 += kSymChunk) {
#pragma unroll 1
        for (int s0 = c0; s0 < c0 + kSymChunk; s0 += 8) {
          float px[8], py[8], pz[8], cm[8];
          *reinterpret_cast<float4*>(px) = *reinterpret_cast<const float4*>(sx + s0);
          *reinterpret_cast<float4*>(px + 4) = *reinterpret_cast<const float4*>(sx + s0 + 4);
          *reinterpret_cast<float4*>(py) = *reinterpret_cast<const float4*>(sy + s0);
          *reinterpret_cast<float4*>(py + 4) = *reinterpret_cast<const float4*>(sy + s0 + 4);
          *reinterpret_cast<float4*>(pz) = *reinterpret_cast<const float4*>(sz + s0);
          *reinterpret_cast<float4*>(pz + 4) = *reinterpret_cast<const float4*>(sz + s0 + 4);
          reduce_pending();
#pragma unroll
          for (int s = 0; s < 8; s += 2) {
            const unsigned long long ax = pack2(px[s], px[s]), ay = pack2(py[s], py[s]), az = pack2(pz[s], pz[s]);
            const unsigned long long bx = pack2(px[s + 1], px[s + 1]), by = pack2(py[s + 1], py[s + 1]), bz = pack2(pz[s + 1], pz[s + 1]);
#pragma unroll
            for (int p = 0; p < kSymR / 2; ++p) {
              unsigned long long dx = sub2(qx[p], ax), dy = sub2(qy[p], ay), dz = sub2(qz[p], az);
              const unsigned long long da = add2(add2(mul2(dx, dx), mul2(dy, dy), one), mul2(dz, dz), one);
              dx = sub2(qx[p], bx);  dy = sub2(qy[p], by);  dz = sub2(qz[p], bz);
              const unsigned long long db = add2(add2(mul2(dx, dx), mul2(dy, dy), one), mul2(dz, dz), one);
              float a0, a1, b0, b1;
              unpack2(da, a0, a1);  unpack2(db, b0, b1);
              best[2 * p] = min3(best[2 * p], a0, b0);
              best[2 * p + 1] = min3(best[2 * p + 1], a1, b1);
              cm[s] = p == 0 ? fminf(a0, a1) : min3(cm[s], a0, a1);
              cm[s + 1] = p == 0 ? fminf(b0, b1) : min3(cm[s + 1], b0, b1);
            }
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) pm[i] = cm[i];
          pcol = s0;
        }
#pragma unroll
        for (int k = 0; k < kSymR; ++k)
          if (best[k] < seen[k]) { seen[k] = best[k];  cid[k] = c0; }
      }
      reduce_pending();                                                    // the tile's last step
      // Rows whose minimum fell inside this tile: lowest streamed index of the noted 32-point chunk that attains it.  The warp
      // serves one (lane, row) at a time -- lane j evaluates point j of that chunk (conflict-free shared-memory reads; a lane
      // walking its own chunk would collide with 31 others on one bank), a ballot finds the lowest match.
#pragma unroll
      for (int k = 0; k < kSymR; ++k) {
        float ax, ay, az, hx, hy, hz;
        unpack2(qx[k >> 1], ax, hx);  unpack2(qy[k >> 1], ay, hy);  unpack2(qz[k >> 1], az, hz);
        if (k & 1) { ax = hx;  ay = hy;  az = hz; }
        unsigned need = __ballot_sync(0xffffffffu, cid[k] >= 0);
        while (need) {
          const int L = __ffs(need) - 1;
          need &= need - 1;
          const int c = __shfl_sync(0xffffffffu, cid[k], L);
          const float bx = __shfl_sync(0xffffffffu, ax, L), by = __shfl_sync(0xffffffffu, ay, L), bz = __shfl_sync(0xffffffffu, az, L);
          const float bb = __shfl_sync(0xffffffffu, best[k], L);
          const unsigned hit = __ballot_sync(0xffffffffu, pair_dist(bx, by, bz, sx[c + lane], sy[c + lane], sz[c + lane]) == bb);
          if (lane == L && hit) bidx[k] = t0 + c + __ffs(hit) - 1;
        }
      }
    }
  }
#pragma unroll
  for (int k = 0; k < kSymR; ++k) {
    if (r0 + k < nr) {
      res_dist[(int64_t)b * nr + r0 + k] = best[k];
      res_idx[(int64_t)b * nr + r0 + k] = bidx[k];         // best == +inf (nothing compared less): index 0, as the oracle
    }
  }
}

// One warp per streamed point: decode its key, rescan the 256 resident points of the winning block for the lowest index.
__global__ void __launch_bounds__(256)
chamfer_sym_finish_kernel(const float* __restrict__ res_xyz, const float* __restrict__ str_xyz, const unsigned long long* __restrict__ keys,
                          float* __restrict__ str_dist, int32_t* __restrict__ str_idx, int nr, int ns, int64_t total, int kSymBlock) {
  const int lane = threadIdx.x & 31;
  const int64_t i = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);      // b * ns + s
  if (i >= total) return;
  const int b = (int)(i / ns);
  const unsigned long long key = keys[i];
  float best = key == ~0ull ? INFINITY : __uint_as_float((unsigned)(key >> 32));
  if (!(best < INFINITY)) best = INFINITY;                 // all-NaN column: the oracle's untouched +inf / index 0
  int idx = 0x7fffffff;
  if (best < INFINITY) {
    const float ax = str_xyz[i * 3], ay = str_xyz[i * 3 + 1], az = str_xyz[i * 3 + 2];
    const int j0 = (int)(key & 0xffffffffu) * kSymBlock;
    const float* rb = res_xyz + (int64_t)b * nr * 3;
    for (int j = j0 + kSymBlock - 32 + lane; j >= j0; j -= 32)
      if (j < nr && pair_dist(rb[(int64_t)j * 3], rb[(int64_t)j * 3 + 1], rb[(int64_t)j * 3 + 2], ax, ay, az) == best) idx = j;
  }
  idx = __reduce_min_sync(0xffffffffu, idx);
  if (lane == 0) {
    str_dist[i] = best;
    str_idx[i] = idx == 0x7fffffff ? 0 : idx;
  }
}

// fp32 issue-rate probe: every thread runs 8 independent FFMA chains, so the FMA pipe is the only limit.  bench.py times it
// with CUDA events to get the MEASURED fp32 SIMT peak (instructions/s) that the Chamfer kernel's pair rate is quoted against.
__global__ void __launch_bounds__(256) fma_probe_kernel(float* __restrict__ sink, int iters, float a, float b) {
  float r[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) r[k] = (float)(threadIdx.x + k);
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int k = 0; k < 8; ++k) r[k] = fmaf(r[k], a, b);
  }
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < 8; ++k) s += r[k];
  if (s == 12345.678f) sink[0] = s;                    // never true in practice; keeps the chains alive
}

int launch_dir(const float* q, const float* r, float* dist, int32_t* idx, int B, int nq, int nr, cudaStream_t st) {
  // lanes per query group: enough threads to fill the chip (~2 waves of 2048 threads / SM)
  const int64_t want = (int64_t)num_sms() * 2048 * 2;
  int S = 1;
  while (S < 32 && (int64_t)B * ceil_div(nq, kQ) * S < want && S * 2 <= nr) S <<= 1;
  const int groups = kThreads / S;
  const int blocks_per_batch = ceil_div(nq, groups * kQ);
  chamfer_nn_kernel<<<B * blocks_per_batch, kThreads, 0, st>>>(q, r, dist, idx, nq, nr, S, blocks_per_batch);
  S3D_LAUNCH_CHECK();
  return S3D_OK;
}

// ---- point-cloud metrics over the search's distances (s3d_chamfer_eval) ------------------------------------------------
// A separate pass over dist1 / dist2 (just written, read from L2), so the search kernels above stay as they are.  Blocks
// [0, B * c0) cover direction 0 (dist1, c0 blocks per sample), the rest direction 1 (dist2, c1 per sample); a block never
// spans two (sample, direction) slices.  Integer counters: warp shuffle -> shared memory -> one 64-bit atomic per counter
// per block, so the sums do not depend on the launch order.
constexpr int kEvalThreads = 256;
constexpr int kEvalPts = 4 * kEvalThreads;   // distances per block
constexpr float kEvalMaxD = 256.f;           // in range: d finite and d < 2^8, so q(d) < 2^40
constexpr float kFx = 4294967296.f;          // 2^32: q(x) = round-half-even(x * 2^32), the product exact in fp32

__global__ void __launch_bounds__(kEvalThreads)
chamfer_eval_kernel(const float* __restrict__ dist1, const float* __restrict__ dist2, int N, int M, int c0, int c1, int B,
                    Thresh th, int nT, unsigned long long* __restrict__ stats) {
  const int64_t blk0 = (int64_t)B * c0;
  const bool d1 = blockIdx.x < blk0;
  const int64_t k = d1 ? blockIdx.x : blockIdx.x - blk0;
  const int c = d1 ? c0 : c1, n = d1 ? N : M;
  const int b = (int)(k / c), chunk = (int)(k % c);
  const float* d = (d1 ? dist1 : dist2) + (int64_t)b * n;
  unsigned long long sum_d = 0, sum_s = 0;
  unsigned n_out = 0, cnt[kMaxThresh] = {};
#pragma unroll
  for (int j = 0; j < kEvalPts / kEvalThreads; ++j) {
    const int i = chunk * kEvalPts + j * kEvalThreads + threadIdx.x;
    if (i >= n) break;
    const float v = d[i];
    if (!(v < kEvalMaxD)) { ++n_out; continue; }                 // +inf (NaN point or nothing compared less), NaN, >= 2^8
    const float s = __fsqrt_rn(v);
    sum_d += (unsigned long long)__float2ll_rn(v * kFx);
    sum_s += (unsigned long long)__float2ll_rn(s * kFx);
#pragma unroll
    for (int t = 0; t < kMaxThresh; ++t)
      if (t < nT) cnt[t] += s < th.t[t];
  }
  constexpr int kN = 3 + kMaxThresh;
  __shared__ unsigned long long acc[kN];
  if (threadIdx.x < kN) acc[threadIdx.x] = 0;
  __syncthreads();
  unsigned long long v[kN];
  v[0] = sum_d;  v[1] = sum_s;  v[2] = n_out;
#pragma unroll
  for (int t = 0; t < kMaxThresh; ++t) v[3 + t] = cnt[t];
  const int nc = 3 + nT;
#pragma unroll
  for (int j = 0; j < kN; ++j) {
    if (j >= nc) break;
    unsigned long long a = v[j];
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if ((threadIdx.x & 31) == 0 && a) atomicAdd(&acc[j], a);
  }
  __syncthreads();
  if ((int)threadIdx.x < nc && acc[threadIdx.x])
    atomicAdd(stats + ((int64_t)b * 2 + (d1 ? 0 : 1)) * nc + threadIdx.x, acc[threadIdx.x]);
}

}  // namespace
}  // namespace s3d

extern "C" int s3d_fma_probe(float* sink, int iters, int64_t* fma_count, void* stream) {
  using namespace s3d;
  if (!sink || !fma_count) { set_error("fma_probe: null argument"); return S3D_ERR_INVALID; }
  S3D_CHECK_ARG(iters > 0, "fma_probe: iters");
  const int blocks = num_sms() * 8;
  fma_probe_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(sink, iters, 1.0000001f, 1e-7f);
  S3D_LAUNCH_CHECK();
  *fma_count = (int64_t)blocks * 256 * 8 * iters;       // thread-level FMAs executed by the launch
  return S3D_OK;
}

// The symmetric kernel wants enough 256-point blocks of the larger set to fill the chip (or knob chamfer_sym = 1).
static bool sym_eligible(int B, int N, int M) {
  const int k = s3d::knobs().chamfer_sym;
  if (k < 0) return false;
  if (k > 0) return true;
  const int nr = N > M ? N : M;
  return (int64_t)B * s3d::ceil_div(nr, 32 * s3d::kSymRMax) >= 2 * (int64_t)s3d::num_sms();
}

extern "C" int64_t s3d_chamfer_workspace_bytes(int B, int N, int M) {
  if (B <= 0 || N <= 0 || M <= 0 || !sym_eligible(B, N, M)) return 0;
  return (int64_t)B * (N < M ? N : M) * 8;
}

extern "C" int s3d_chamfer_forward_ws(const float* xyz1, const float* xyz2, float* dist1, int32_t* idx1, float* dist2,
                                      int32_t* idx2, int B, int N, int M, void* workspace, int64_t workspace_bytes, void* stream) {
  using namespace s3d;
  if (!xyz1 || !xyz2 || !dist1 || !idx1 || !dist2 || !idx2) { set_error("chamfer: null argument"); return S3D_ERR_INVALID; }
  S3D_CHECK_ARG(B >= 0 && N > 0 && M > 0, "chamfer: empty point set (N=%d, M=%d)", N, M);
  if (B == 0) return S3D_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t need = s3d_chamfer_workspace_bytes(B, N, M);
  if (workspace && need > 0 && workspace_bytes >= need) {
    S3D_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 7) == 0, "chamfer: workspace must be 8-byte aligned");
    // resident (rows, in registers) = the larger set, streamed (columns, shared memory) = the smaller one
    const bool swap = N > M;
    const float *res = swap ? xyz1 : xyz2, *str = swap ? xyz2 : xyz1;
    float *res_d = swap ? dist1 : dist2, *str_d = swap ? dist2 : dist1;
    int32_t *res_i = swap ? idx1 : idx2, *str_i = swap ? idx2 : idx1;
    const int nr = swap ? N : M, ns = swap ? M : N;
    unsigned long long* keys = static_cast<unsigned long long*>(workspace);
    S3D_CUDA(cudaMemsetAsync(keys, 0xff, (size_t)need, st));
    // 8 resident points per lane amortise the per-step column reduction best; with fewer than ~24 warps per SM at that size
    // 4 per lane (twice the warps) hide the dependent-issue latency better
    const int R = (knobs().chamfer_sym_r == 4 || knobs().chamfer_sym_r == 8) ? knobs().chamfer_sym_r
                : ((int64_t)B * ceil_div(nr, 32 * 8) >= 24 * (int64_t)num_sms() ? 8 : 4);
    const int blk = 32 * R;
    const int ctas_per_batch = ceil_div(ceil_div(nr, blk), kSymWarps);
    S3D_CHECK_ARG((int64_t)B * ctas_per_batch < (1ll << 31), "chamfer: grid too large");
    if (R == 8) chamfer_sym_kernel<8><<<B * ctas_per_batch, 32 * kSymWarps, 0, st>>>(res, str, res_d, res_i, keys, nr, ns, ctas_per_batch, 1.0f);
    else        chamfer_sym_kernel<4><<<B * ctas_per_batch, 32 * kSymWarps, 0, st>>>(res, str, res_d, res_i, keys, nr, ns, ctas_per_batch, 1.0f);
    S3D_LAUNCH_CHECK();
    const int64_t total = (int64_t)B * ns;
    chamfer_sym_finish_kernel<<<(unsigned)ceil_div64(total, 8), 256, 0, st>>>(res, str, keys, str_d, str_i, nr, ns, total, blk);
    S3D_LAUNCH_CHECK();
    return S3D_OK;
  }
  int rc = launch_dir(xyz1, xyz2, dist1, idx1, B, N, M, st);
  if (rc != S3D_OK) return rc;
  return launch_dir(xyz2, xyz1, dist2, idx2, B, M, N, st);
}

extern "C" int s3d_chamfer_eval(const float* xyz1, const float* xyz2, float* dist1, int32_t* idx1, float* dist2, int32_t* idx2,
                                int B, int N, int M, const float* tau, int T, long long* stats, void* workspace,
                                int64_t workspace_bytes, void* stream) {
  using namespace s3d;
  if (!stats || (T > 0 && !tau)) { set_error("chamfer_eval: null argument"); return S3D_ERR_INVALID; }
  S3D_CHECK_ARG(T >= 0 && T <= kMaxThresh, "chamfer_eval: T must be in [0, %d], got %d", kMaxThresh, T);
  Thresh th;
  for (int t = 0; t < kMaxThresh; ++t) {
    th.t[t] = t < T ? tau[t] : 0.f;
    S3D_CHECK_ARG(t >= T || (std::isfinite(th.t[t]) && th.t[t] > 0.f),"chamfer_eval: threshold %d must be finite and > 0", t);
  }
  S3D_CHECK_ARG(N < (1 << 22) && M < (1 << 22), "chamfer_eval: N and M must be below 2^22 (N=%d, M=%d)", N, M);
  const int c0 = N > 0 ? ceil_div(N, kEvalPts) : 0, c1 = M > 0 ? ceil_div(M, kEvalPts) : 0;
  S3D_CHECK_ARG((int64_t)B * (c0 + c1) < (1ll << 31), "chamfer_eval: grid too large");
  const int rc = s3d_chamfer_forward_ws(xyz1, xyz2, dist1, idx1, dist2, idx2, B, N, M, workspace, workspace_bytes, stream);
  if (rc != S3D_OK || B == 0) return rc;
  chamfer_eval_kernel<<<(unsigned)((int64_t)B * (c0 + c1)), kEvalThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      dist1, dist2, N, M, c0, c1, B, th, T, reinterpret_cast<unsigned long long*>(stats));
  S3D_LAUNCH_CHECK();
  return S3D_OK;
}

extern "C" int s3d_chamfer_forward(const float* xyz1, const float* xyz2, float* dist1, int32_t* idx1, float* dist2,
                                   int32_t* idx2, int B, int N, int M, void* stream) {
  return s3d_chamfer_forward_ws(xyz1, xyz2, dist1, idx1, dist2, idx2, B, N, M, nullptr, 0, stream);
}
