// Fused correlation + soft-argmax on the tensor cores (rows V+S, correlation variant).
//
// The SIMT kernel in costvolume.cu is compute-bound (2*C*D flop per pixel against 2*C*e bytes: D/4
// flop/B in fp32, beyond the fp32 ridge for D >= 32).  The correlation of one image row is a Gram
// matrix, S = X_ref [w x C] . X_tgt^T [C x w], whose band S[x, x -/+ d] is the cost volume -- a dense
// contraction, so it goes to tcgen05:
//   tile      two image rows (y, y+1) of one stereo pair: M = 128 reference pixels (2 x 64, x padded to 64
//             by TMA zero fill), N = 128 target pixels of the same two rows, K = C.  One TMA box per
//             image and K chunk, loaded ONCE for both views: the left-reference accumulator is L . R^T, the
//             right-reference one R . L^T (a second MMA with the operands exchanged).  Accumulators
//             [128 x 128] fp32 live in TMEM (four buffers).
//             Only the two 64 x 64 diagonal blocks are used (the off-diagonal blocks pair different
//             image rows), and of those only the band -- the tensor pipe has ~50x headroom here.
//   epilogue  thread = reference pixel (TMEM lane).  It reads the <= 64 target columns of its own row
//             block, keeps those with 0 <= d < D, adds the closed-form contribution of the out-of-image
//             disparities (cost 0, as in the oracle), and finishes softmax / expectation in registers.
//             The cost volume never exists anywhere: per pixel 2*C*e bytes in, 4 bytes out.
// Restrictions: bf16 features (fp32 features keep the exact SIMT kernel), w <= 64, C*2 a multiple of 32 B.
#include <cuda.h>
#include <string.h>
#include <stdlib.h>
#include "common.cuh"
#include "ptx.cuh"
#include "epilogue.cuh"

namespace s3d {
namespace {

constexpr int kGroups = 4;         // epilogue warp groups; group g owns TMEM accumulator buffer g
constexpr int kThreads = 128 + kGroups * 128;   // warps 0-3: TMA / MMA / TMEM alloc / idle; then 4 warps per group
constexpr int kWP = 64;            // padded row width
constexpr int kRows = 2;           // image rows per tile
constexpr int kM = kWP * kRows;    // 128
constexpr int kMaxStages = 6;
constexpr int kTmemCols = kGroups * kM;   // 512
static_assert(kGroups == 4, "the epilogue maps group g to buffer g, pair tiles g >> 1, g >> 1 + 2, ..., alternating views");

struct CorrArgs {
  float* disp;
  int B, h, w, C, D;
  int row_bytes, kc, nchunks;
  int op_bytes;        // bytes of one operand tile per chunk: 128 * row_bytes
  int stage_bytes;     // 2 * op_bytes
  int stages;
  int tiles_per_img, pair_tiles;   // pair tile = (stereo pair, two image rows): one load, two accumulators (left / right reference)
  float inv_c;
  uint32_t idesc;
  float* std_q;        // kStd: the distribution's standard deviation [2B,h,w]
};

struct CorrCtrl {
  uint64_t full[kMaxStages], empty[kMaxStages];
  uint64_t acc_full[kGroups], acc_empty[kGroups];
  uint32_t tmem_base;
};

// MUFU.EX2 as one instruction (exp2f() wraps it in range tests and two scalings for denormal results, which a softmax
// weight does not need): <= 2 ulp, results below 2^-126 flush to zero.
__device__ __forceinline__ float ex2_approx(float x) { float r;  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));  return r; }

// kStd: also the standard deviation of each pixel's distribution, from a third pass over the held exponentials about the mean
// (exact two-pass variance; the zero-cost tail in closed form).
template <bool kStd>
__global__ void __launch_bounds__(kThreads, 1)
corr_tc_kernel(const __grid_constant__ CUtensorMap map_f, const __grid_constant__ CorrArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ CorrCtrl ctrl;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) ptx::prefetch_tensormap(&map_f);
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < kMaxStages; ++s) { ptx::mbar_init(&ctrl.full[s], 1); ptx::mbar_init(&ctrl.empty[s], 2); }
    for (int b = 0; b < kGroups; ++b) { ptx::mbar_init(&ctrl.acc_full[b], 1); ptx::mbar_init(&ctrl.acc_empty[b], 128); }
    ptx::fence_barrier_init();
  }
  if (warp == 2) ptx::tmem_alloc(&ctrl.tmem_base, kTmemCols);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = ctrl.tmem_base;

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;  uint32_t phase = 0;
      // a pair tile (stereo pair b, rows y0, y0+1) loads the LEFT and the RIGHT feature rows once; both views' accumulators
      // are built from that one stage (S_right = S_left^T, formed by a second MMA with the operands exchanged): half the
      // TMA rows per disparity map -- the loads, at ~2-4 cycles per 64-byte row, were what the epilogue warps waited for
      for (int pt = blockIdx.x; pt < a.pair_tiles; pt += gridDim.x) {
        const int n = pt / a.tiles_per_img, y0 = (pt % a.tiles_per_img) * kRows;
        for (int ch = 0; ch < a.nchunks; ++ch) {
          ptx::mbar_wait(&ctrl.empty[stage], phase ^ 1);
          uint8_t* s = smem + stage * a.stage_bytes;
          ptx::mbar_arrive_expect_tx(&ctrl.full[stage], a.stage_bytes);
          ptx::tma_load_5d(s, &map_f, &ctrl.full[stage], ch * a.kc, 0, y0, n, 0);    // ONE box: [view][row][x][c] = L tile, R tile
          if (++stage == a.stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1 || warp == 2) {
    // TWO MMA issuers, one per view (warp 1: left image is the reference, A = left rows; warp 2: right).  An item is only
    // 2-4 MMAs, but around them sit ~800 cycles of serial barrier waits, fences and commits (clock64 timeline,
    // profiles/r2_corr_tc_timeline.txt): with one issuer that chain, 28 items long, WAS the kernel.  Both issuers wait on the
    // same `full` barrier of a stage and both commit to its `empty` barrier (count 2).
    const int view = warp - 1;                             // buffer parity j of this issuer's items (buffers j, j + 2)
    int stage = 0;  uint32_t phase = 0;
    int buf = view;  uint32_t acc_phase = 0;
    int kt = 0;                                            // running pair-tile index of this CTA
    const int kper = a.row_bytes >> 5;
    const uint64_t hi = ptx::make_smem_desc(0, a.row_bytes) & 0xFFFFFFFF00000000ull;
    const uint32_t smem_u = ptx::smem_u32(smem);
    for (int pt = blockIdx.x; pt < a.pair_tiles; pt += gridDim.x, ++kt) {
      // which view lands in which buffer flips every second pair tile (v = j ^ bit 1 of the pair-tile index), so that an
      // epilogue group alternates between the two views (see the epilogue)
      const int v = view ^ ((kt >> 1) & 1);
      ptx::mbar_wait(&ctrl.acc_empty[buf], acc_phase ^ 1);
      const uint32_t d_tmem = tmem_base + buf * kM;
      for (int ch = 0; ch < a.nchunks; ++ch) {
        ptx::mbar_wait(&ctrl.full[stage], phase);
        ptx::tc_fence_after();
        const uint32_t sa = smem_u + stage * a.stage_bytes;
        const uint64_t ldesc = hi | ((sa >> 4) | (1u << 16));
        const uint64_t rdesc = hi | (((sa + a.op_bytes) >> 4) | (1u << 16));
        if (ptx::elect_one()) {
          for (int k = 0; k < kper; ++k)
            ptx::mma_bf16(d_tmem, (v ? rdesc : ldesc) + 2 * k, (v ? ldesc : rdesc) + 2 * k, a.idesc, (ch | k) != 0);
          ptx::tc_commit(&ctrl.empty[stage]);              // the stage is free once BOTH views have read it
          if (ch == a.nchunks - 1) ptx::tc_commit(&ctrl.acc_full[buf]);
        }
        __syncwarp();
        if (++stage == a.stages) { stage = 0; phase ^= 1; }
      }
      buf += 2;
      if (buf >= kGroups) { buf = view; acc_phase ^= 1; }
    }
  } else if (warp >= 4) {
    const int q = warp & 3;
    const int rowblk = q >> 1;                 // image row of the tile this warp serves
    const int x = (q & 1) * 32 + lane;         // reference pixel of this thread
    const int xw0 = (q & 1) * 32;              // first x of the warp
    const int D = a.D, w = a.w;
    const float scale2 = a.inv_c * 1.4426950408889634f;     // 1/C * log2(e)
    // kGroups epilogue groups take the items round-robin; item i = (pair tile k, buffer parity j) uses accumulator buffer
    // 2 (k & 1) + j = its group's.  The VIEW of an item is v = j ^ bit 1 of k, so a group ALTERNATES between left- and
    // right-referenced items: a warp's band covers 2 chunks of 16 target columns for one view and 4 for the other (x < 32 /
    // x >= 32), and with a fixed view per group the 4-chunk warps paced their group while the 2-chunk warps idled (third timeline
    // in profiles/r2_corr_tc_timeline.txt).  One max over all columns first, then 16-way independent ex2 + four partial sums per
    // chunk (no online softmax); tile indices advance incrementally (no division in the loop).
    const int grp = (warp - 4) >> 2;
    const int buf = grp;  uint32_t acc_phase = 0;
    const uint32_t taddr = tmem_base + buf * kM + rowblk * kWP + (static_cast<uint32_t>(q * 32) << 16);
    const int step = 2 * (int)gridDim.x;
    const int step_img = step / a.tiles_per_img, step_row = step % a.tiles_per_img;
    int pt = blockIdx.x + (grp >> 1) * gridDim.x;
    int img = pt / a.tiles_per_img, yt = pt % a.tiles_per_img;
    int mi = 0;                                             // this group's item counter: pair tile k = (grp >> 1) + 2 mi
    for (; pt < a.pair_tiles; pt += step, ++mi) {
      const bool left_ref = ((grp ^ mi) & 1) == 0;
      // target columns this warp needs: left-ref xt in [xw0-D+1, xw0+31], right-ref xt in [xw0, xw0+31+D-1]
      const int lo = left_ref ? max(0, xw0 - D + 1) : xw0;
      const int hi_ = left_ref ? xw0 + 31 : min(kWP - 1, xw0 + 31 + D - 1);
      const int c_lo = lo >> 4, c_hi = hi_ >> 4;            // 16-column chunks, warp-uniform
      // out-of-image disparities keep cost 0 (oracle semantics): d in [dz0, D) where
      //   left-ref : x - d < 0   <=>  d > x            right-ref: x + d >= w  <=>  d >= w - x
      const int dz0 = left_ref ? min(D, x + 1) : min(D, max(0, w - x));
      // the target columns inside the window as a 64-bit mask (bit xt): left xt in [x - dz0 + 1, x], right xt in [x, x + dz0 - 1]
      const uint64_t ones = dz0 >= 64 ? ~0ull : ((1ull << dz0) - 1ull);
      const uint64_t win = left_ref ? ones << (x - dz0 + 1) : ones << x;
      const float m0 = dz0 < D ? 0.f : -1e30f;               // the zero-cost tail takes part in the max; else a finite floor
      const float tail_cnt = (float)(D - dz0), tail_d = 0.5f * (float)(dz0 + D - 1);
      const float xs = left_ref ? (float)x : -(float)x, sgn = left_ref ? -1.f : 1.f;
      const int n = img + (left_ref ? 0 : a.B), y = yt * kRows + rowblk;
      ptx::mbar_wait(&ctrl.acc_full[buf], acc_phase);
      ptx::tc_fence_after();
      // all the columns this warp needs go to registers and the accumulator buffer is handed back at once: the MMA of the
      // group's next item then runs under this item's arithmetic
      uint32_t u[4][16];
#pragma unroll
      for (int c = 0; c < 4; ++c)
        if (c >= c_lo && c <= c_hi) ptx::tmem_ld16(taddr + c * 16, u[c]);
      ptx::tmem_ld_wait();
      ptx::tc_fence_before();
      ptx::mbar_arrive(&ctrl.acc_empty[buf]);
      acc_phase ^= 1;
      // pass 1: columns outside the window become -inf (they drop out of the max, and ex2(-inf * scale2 - m) = 0); one max
      float mx = -INFINITY;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        if (c >= c_lo && c <= c_hi) {
          const uint32_t mb = (uint32_t)(win >> (16 * c));
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const float v = (mb >> i) & 1u ? __uint_as_float(u[c][i]) : -INFINITY;
            u[c][i] = __float_as_uint(v);
            mx = fmaxf(mx, v);
          }
        }
      }
      const float m = fmaxf(m0, mx * scale2);               // scale2 > 0: max commutes with the scaling
      // pass 2: base-2 exponentials IN PLACE, the 16 MUFU.EX2 of a chunk issued back to back (volatile: ptxas otherwise sinks
      // each one next to its consumer -- with 64 accumulator values live it has no spare registers to look ahead -- and the warp
      // stalls on every MUFU result); chunk c's sums are taken while chunk c+1's exponentials are in flight
      float s4[4] = {0.f, 0.f, 0.f, 0.f}, t4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int c = 0; c <= 4; ++c) {
        if (c < 4 && c >= c_lo && c <= c_hi) {
#pragma unroll
          for (int i = 0; i < 16; ++i) u[c][i] = __float_as_uint(fmaf(__uint_as_float(u[c][i]), scale2, -m));
#pragma unroll
          for (int i = 0; i < 16; ++i) asm volatile("ex2.approx.ftz.f32 %0, %0;" : "+r"(u[c][i]));
        }
        if (c >= 1 && c - 1 >= c_lo && c - 1 <= c_hi) {
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const float e = __uint_as_float(u[c - 1][i]);
            s4[i & 3] += e;
            t4[i & 3] = fmaf(e, (float)((c - 1) * 16 + i), t4[i & 3]);
          }
        }
      }
      float s = (s4[0] + s4[1]) + (s4[2] + s4[3]);
      const float tx = (t4[0] + t4[1]) + (t4[2] + t4[3]);
      float t = fmaf(xs, s, sgn * tx);                      // sum e * d  (d = x - xt for the left view, xt - x for the right)
      if (dz0 < D) {                                        // (D - dz0) terms of cost 0 at d = dz0 .. D-1
        const float e0 = ex2_approx(-m) * tail_cnt;
        s += e0;
        t = fmaf(e0, tail_d, t);
      }
      if (x < w && y < a.h) a.disp[((int64_t)n * a.h + y) * w + x] = __fdividef(t, s);
      if (kStd) {
        // sum e (d - mu)^2 with d = x - xt (left view) or xt - x (right view): the same (xt - x - sgn mu)^2 for both
        const float mu = __fdividef(t, s), c0 = (float)x + sgn * mu;
        float v4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          if (c >= c_lo && c <= c_hi) {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float dd = (float)(c * 16 + i) - c0;
              v4[i & 3] = fmaf(__uint_as_float(u[c][i]) * dd, dd, v4[i & 3]);
            }
          }
        }
        float v2 = (v4[0] + v4[1]) + (v4[2] + v4[3]);
        if (dz0 < D) {                                      // the tail: tail_cnt planes, mean tail_d, variance (cnt^2 - 1) / 12
          const float dt = tail_d - mu;
          v2 = fmaf(ex2_approx(-m) * tail_cnt, fmaf(dt, dt, (tail_cnt * tail_cnt - 1.f) * (1.f / 12.f)), v2);
        }
        if (x < w && y < a.h) a.std_q[((int64_t)n * a.h + y) * w + x] = soft_std(v2 / s, mu);
      }
      img += step_img;  yt += step_row;
      if (yt >= a.tiles_per_img) { yt -= a.tiles_per_img;  ++img; }
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, kTmemCols);
  }
}

}  // namespace

bool corr_tc_eligible(int w, int C, int D, int dtype) {
  return dtype == S3D_DTYPE_BF16 && w <= kWP && (C * 2) % 32 == 0 && C <= 6 * 64 && D >= 1 && !knobs().no_corr_tc;
}

int corr_tc_launch(const void* feat, float* disp, float* std_q, int B, int h, int w, int C, int D, float inv_c, cudaStream_t stream) {
  CorrArgs a;
  memset(&a, 0, sizeof(a));
  a.disp = disp;  a.std_q = std_q;  a.B = B;  a.h = h;  a.w = w;  a.C = C;  a.D = D;
  const int cb = C * 2;
  a.row_bytes = cb % 128 == 0 ? 128 : (cb % 64 == 0 ? 64 : 32);
  a.kc = a.row_bytes / 2;
  a.nchunks = cb / a.row_bytes;
  a.op_bytes = kM * a.row_bytes;
  a.stage_bytes = 2 * a.op_bytes;
  a.stages = (200 * 1024) / a.stage_bytes;
  if (a.stages > kMaxStages) a.stages = kMaxStages;
  S3D_CHECK_ARG(a.nchunks <= a.stages, "corr_tc: C = %d needs %d K chunks resident at once (at most %d)", C, a.nchunks, a.stages);
  a.tiles_per_img = ceil_div(h, kRows);
  const int64_t total = (int64_t)B * a.tiles_per_img;
  S3D_CHECK_ARG(total > 0 && total < (1ll << 30), "corr_tc: tile count out of range");
  a.pair_tiles = (int)total;
  a.inv_c = inv_c;
  a.idesc = ptx::make_instr_desc(1, kM, kM);
  const CUtensorMapSwizzle sw = a.row_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                              : a.row_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B;
  CUtensorMap map_f;
  // feat [2B, h, w, C] seen as (C, w, h, pair, view): one box {kc, 64, 2 rows, 1, 2 views} fetches the left AND the right rows of
  // a pair tile -- issuing a tiled TMA costs the producer thread ~390 cycles whatever its size (clock64 timeline), so the op
  // count per CTA, not the bytes, set the pace of the loads
  cuuint32_t box[5] = {(cuuint32_t)a.kc, kWP, kRows, 1, 2};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  int rc = encode_act_map(&map_f, feat, 2, false, C, w, h, B, 2, box, estr, sw);
  if (rc != S3D_OK) return rc;
  const int smem_bytes = a.stages * a.stage_bytes + 1024;
  auto kern = std_q ? corr_tc_kernel<true> : corr_tc_kernel<false>;
  S3D_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
  int grid = num_sms();
  if (grid > a.pair_tiles) grid = a.pair_tiles;
  kern<<<grid, kThreads, smem_bytes, stream>>>(map_f, a);
  S3D_LAUNCH_CHECK();
  return S3D_OK;
}

}  // namespace s3d
