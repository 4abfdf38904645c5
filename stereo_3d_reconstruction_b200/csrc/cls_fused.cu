// Fused disparity classifier: the Cout = 1 3x3x3 convolution at the end of the cost aggregation AND the soft-argmin
// over the disparity planes, in one pass over the aggregated volume (bf16 channels-last [N,D,h,w,C]).
//
// The unfused path (s3d_conv_igemm as a 27-tap pointwise GEMM + s3d_tap_gather_soft_argmin) writes and re-reads a
// [N,D,h,32,w] fp32 tensor of per-tap projections -- 2 x 2.1 GB at the benchmark shape, more than the volume itself.
// Here a CTA owns a 32(y) x 8(x) pixel patch and marches over the disparity planes:
//   1. TMA stages input plane p of the patch with its halo (34 x 10 pixels, zero fill outside the image).
//   2. tcgen05: T[halo pixel, tap] = X_p[halo pixel, :] . W[tap, :] for all 27 taps at once (M = 128 pixels x 3
//      tiles, N = 32, K = C); the 2 KB weight matrix stays in shared memory for the whole kernel.
//   3. The projections go TMEM -> registers -> shared memory as T[tap][halo pixel] (fp32, 37 KB).
//   4. Every output pixel gathers its 27 neighbours' taps: the kz = 2 / 1 / 0 sums of plane p belong to output planes
//      p-1 / p / p+1, held in three registers; plane p-1 is then complete and retires into an online softmax
//      (running max, sum, disparity-weighted sum).  After the last plane the expectation is the disparity.
// HBM traffic = one read of the volume (+ 4 bytes per pixel out); the kernel is bound by that read.
//
// Warp roles: 0 TMA producer, 1 MMA issuer, 2 TMEM allocator, 4-11 projection staging + gather (one thread per pixel).
#include <cuda.h>
#include <stdlib.h>
#include <string.h>
#include "common.cuh"
#include "ptx.cuh"
#include "epilogue.cuh"

namespace s3d {
namespace {

constexpr int kThreads = 384;
constexpr int kTX = 8, kHX = kTX + 2;
constexpr int kTY = 32, kHY = kTY + 2;
constexpr int kRows = kHX * kHY;               // 340 halo pixels
constexpr int kTiles = 3;                      // 3 x 128 MMA rows cover them (rows 340..383 are never read back)
constexpr int kN = 32;                         // 27 taps padded to the UMMA N granule
constexpr int kTaps = 27;
constexpr int kTS = 352;                       // floats per tap line of the projection buffer
constexpr int kMaxRing = 4;
constexpr int kTmemCols = 256;                 // two accumulator buffers of 3 x 32 columns, 128 apart

struct ClsArgs {
  float* disp;
  float sign;
  int N, D, h, w;
  int row_bytes, slot_bytes, ring;
  int cols_x, cols_y, total_cols;
  uint32_t idesc;
  float* std_q;        // kStd: the distribution's standard deviation [N,h,w]
};

struct ClsCtrl {
  uint64_t plane_full[kMaxRing], plane_empty[kMaxRing];
  uint64_t acc_full[2], acc_empty[2];
  uint64_t w_full;
  uint32_t tmem_base;
};

struct Col { int n, y0, x0; };
__device__ __forceinline__ Col decode_col(const ClsArgs& a, int c) {
  Col r;
  r.x0 = (c % a.cols_x) * kTX;  c /= a.cols_x;
  r.y0 = (c % a.cols_y) * kTY;  c /= a.cols_y;
  r.n = c;
  return r;
}

template <int kPer, bool kStd>                   // MMAs per tile = row_bytes / 32; kStd: also write std_q (common.cuh, SoftSpread)
__global__ void __launch_bounds__(kThreads, 1)
cls_fused_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w,
                 const __grid_constant__ ClsArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_w = smem + a.ring * a.slot_bytes;                       // [32][row_bytes], swizzled like the planes
  float* T = reinterpret_cast<float*>(smem_w + 4096);                   // [27][kTS]
  __shared__ ClsCtrl ctrl;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int D = a.D, ring = a.ring;
  const int rb = a.row_bytes;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&map_x);
    ptx::prefetch_tensormap(&map_w);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < kMaxRing; ++s) { ptx::mbar_init(&ctrl.plane_full[s], 1); ptx::mbar_init(&ctrl.plane_empty[s], 1); }
    for (int b = 0; b < 2; ++b) { ptx::mbar_init(&ctrl.acc_full[b], 1); ptx::mbar_init(&ctrl.acc_empty[b], 8); }
    ptx::mbar_init(&ctrl.w_full, 1);
    ptx::fence_barrier_init();
  }
  if (warp == 2) ptx::tmem_alloc(&ctrl.tmem_base, kTmemCols);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = ctrl.tmem_base;
  const int ncols = (a.total_cols - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  if (warp == 0) {
    // ================= TMA producer =================
    const uint32_t planes_u32 = ptx::smem_u32(smem);
    const uint32_t bar_pf = ptx::smem_u32(&ctrl.plane_full[0]), bar_pe = ptx::smem_u32(&ctrl.plane_empty[0]);
    const int plane_tx = kRows * rb;
    if (ptx::elect_one()) {
      ptx::mbar_arrive_expect_tx_u32(ptx::smem_u32(&ctrl.w_full), kN * rb);
      ptx::tma_load_3d_u32(ptx::smem_u32(smem_w), &map_w, ptx::smem_u32(&ctrl.w_full), 0, 0, 0);
    }
    __syncwarp();
    int slot = 0;  uint32_t phase = 0;
    for (int ci = 0; ci < ncols; ++ci) {
      const Col c = decode_col(a, blockIdx.x + ci * gridDim.x);
      for (int p = 0; p < D; ++p) {
        ptx::mbar_wait_u32(bar_pe + 8 * slot, phase ^ 1);
        if (ptx::elect_one()) {
          ptx::mbar_arrive_expect_tx_u32(bar_pf + 8 * slot, plane_tx);
          ptx::tma_load_5d_u32(planes_u32 + slot * a.slot_bytes, &map_x, bar_pf + 8 * slot, 0, c.x0 - 1, c.y0 - 1, p, c.n);
        }
        __syncwarp();
        if (++slot == ring) { slot = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer: 3 tiles x kPer MMAs per plane =================
    const uint32_t bar_pf = ptx::smem_u32(&ctrl.plane_full[0]), bar_pe = ptx::smem_u32(&ctrl.plane_empty[0]);
    const uint32_t bar_af = ptx::smem_u32(&ctrl.acc_full[0]), bar_ae = ptx::smem_u32(&ctrl.acc_empty[0]);
    const uint64_t layout = rb == 128 ? 2ull : (rb == 64 ? 4ull : 6ull);
    const uint64_t hi = (static_cast<uint64_t>((8 * rb) >> 4) << 32) | (1ull << 46) | (layout << 61);   // dense rows
    const uint32_t x_lo0 = ((ptx::smem_u32(smem) & 0x3FFFF) >> 4) | (1u << 16);
    const uint64_t wdesc = hi | (((ptx::smem_u32(smem_w) & 0x3FFFF) >> 4) | (1u << 16));
    const uint32_t slot_step = a.slot_bytes >> 4, tile_step = (128 * rb) >> 4;
    ptx::mbar_wait_u32(ptx::smem_u32(&ctrl.w_full), 0);
    int slot = 0;  uint32_t phase = 0;
    int buf = 0;   uint32_t aphase = 0;
    const int nplanes = ncols * D;
    for (int gp = 0; gp < nplanes; ++gp) {
      ptx::mbar_wait_u32(bar_pf + 8 * slot, phase);
      ptx::mbar_wait_u32(bar_ae + 8 * buf, aphase ^ 1);
      ptx::tc_fence_after();
      const uint64_t xdesc = hi | (x_lo0 + slot * slot_step);
      const uint32_t d = tmem_base + buf * 128;
      if (ptx::elect_one()) {
#pragma unroll
        for (int t = 0; t < kTiles; ++t) {
#pragma unroll
          for (int k = 0; k < kPer; ++k)
            ptx::mma_bf16(d + t * kN, xdesc + t * tile_step + 2 * k, wdesc + 2 * k, a.idesc, k ? 1u : 0u);
        }
        ptx::tc_commit_u32(bar_af + 8 * buf);
        ptx::tc_commit_u32(bar_pe + 8 * slot);
      }
      __syncwarp();
      if (++slot == ring) { slot = 0; phase ^= 1; }
      if (++buf == 2) { buf = 0; aphase ^= 1; }
    }
  } else if (warp >= 4) {
    // ================= projections -> shared memory -> gather + online softmax =================
    const int ew = warp - 4;                       // 0..7; TMEM lane quarter = warp % 4 = ew % 4
    const int q = ew & 3;
    // output pixel of this thread inside the patch.  A warp takes rows b, b+4, b+8, b+12 (not 4 consecutive rows): a tap
    // line of the projection buffer has a pitch of 10 floats, so rows 4 apart start 8 banks apart and the warp's 27 gather
    // loads are conflict-free (4 consecutive rows overlap on 6 banks: 2 wavefronts per load)
    const int xl = lane & 7;
    const int yl = (ew & 3) + 16 * (ew >> 2) + 4 * (lane >> 3);
    const uint32_t bar_af = ptx::smem_u32(&ctrl.acc_full[0]), bar_ae = ptx::smem_u32(&ctrl.acc_empty[0]);
    const float* Tg = T + yl * kHX + xl;           // tap (ky,kx) of this pixel: Tg[tap * kTS + ky * kHX + kx]
    int buf = 0;  uint32_t aphase = 0;
    for (int ci = 0; ci < ncols; ++ci) {
      const Col c = decode_col(a, blockIdx.x + ci * gridDim.x);
      float m = -INFINITY, s = 0.f, t = 0.f;
      SoftSpread u;
      float c0 = 0.f, c1 = 0.f, c2 = 0.f;          // partial costs of output planes p-1, p, p+1
      auto retire = [&](int z, float cst) {
        const float v = a.sign * cst;
        if (v > m) {
          const float sc = expf(m - v); s *= sc; t *= sc; m = v;
          if (kStd) { u.scale(sc);  u.move(z, s); }
        }
        const float e = expf(v - m);  s += e;  t += e * (float)z;
        if (kStd) u.add(e, z);
      };
      for (int p = 0; p < D; ++p) {
        ptx::mbar_wait_u32(bar_af + 8 * buf, aphase);
        ptx::tc_fence_after();
        // this warp's lane quarter of tiles (ew >> 2) and (ew >> 2) + 2
        uint32_t v0[2][16], v1[2][16];
        const int tile0 = ew >> 2, tile1 = tile0 + 2;
        const uint32_t ta = tmem_base + buf * 128 + (static_cast<uint32_t>(q * 32) << 16);
        ptx::tmem_ld16(ta + tile0 * kN, v0[0]);
        ptx::tmem_ld16(ta + tile0 * kN + 16, v0[1]);
        if (tile1 < kTiles) {
          ptx::tmem_ld16(ta + tile1 * kN, v1[0]);
          ptx::tmem_ld16(ta + tile1 * kN + 16, v1[1]);
        }
        ptx::tmem_ld_wait();
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive_u32(bar_ae + 8 * buf);
        // everyone has finished gathering the previous plane before its projections are overwritten
        asm volatile("bar.sync 1, 256;" ::: "memory");
        const int r0 = tile0 * 128 + q * 32 + lane, r1 = tile1 * 128 + q * 32 + lane;
#pragma unroll
        for (int tp = 0; tp < kTaps; ++tp) T[tp * kTS + r0] = __uint_as_float(v0[tp >> 4][tp & 15]);
        if (tile1 < kTiles && r1 < kRows) {
#pragma unroll
          for (int tp = 0; tp < kTaps; ++tp) T[tp * kTS + r1] = __uint_as_float(v1[tp >> 4][tp & 15]);
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");
        float a0 = 0.f, a1 = 0.f, a2 = 0.f;        // contributions of input plane p through kz = 2, 1, 0
#pragma unroll
        for (int ky = 0; ky < 3; ++ky) {
#pragma unroll
          for (int kx = 0; kx < 3; ++kx) {
            const float* pp = Tg + (ky * 3 + kx) * kTS + ky * kHX + kx;
            a0 += pp[18 * kTS];
            a1 += pp[9 * kTS];
            a2 += pp[0];
          }
        }
        c0 += a0;  c1 += a1;  c2 += a2;
        if (p >= 1) retire(p - 1, c0);
        c0 = c1;  c1 = c2;  c2 = 0.f;
        if (++buf == 2) { buf = 0; aphase ^= 1; }
      }
      retire(D - 1, c0);
      const int y = c.y0 + yl, x = c.x0 + xl;
      if (y < a.h && x < a.w) {
        a.disp[((int64_t)c.n * a.h + y) * a.w + x] = t / s;
        if (kStd) a.std_q[((int64_t)c.n * a.h + y) * a.w + x] = u.sigma(t / s, s);
      }
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
}  // namespace s3d

extern "C" int s3d_cls_soft_argmin(const void* x, const void* w_taps, float* disp, float* std_q, int N, int D, int h, int w,
                                   int C, float sign, void* stream) {
  using namespace s3d;
  if (!x || !w_taps || !disp) { set_error("cls_soft_argmin: null argument"); return S3D_ERR_INVALID; }
  S3D_CHECK_ARG(N > 0 && D > 0 && h > 0 && w > 0, "cls_soft_argmin: bad shape");
  S3D_CHECK_ARG(C == 16 || C == 32 || C == 64, "cls_soft_argmin: C must be 16, 32 or 64 (bf16 rows of 32 / 64 / 128 bytes)");
  S3D_CHECK_ARG((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(w_taps) & 15) == 0,
                "cls_soft_argmin: pointers must be 16-byte aligned");
  ClsArgs a;
  memset(&a, 0, sizeof(a));
  a.disp = disp;  a.std_q = std_q;  a.sign = sign;  a.N = N;  a.D = D;  a.h = h;  a.w = w;
  a.row_bytes = C * 2;
  a.slot_bytes = kTiles * 128 * a.row_bytes;                // 384 rows; multiple of 1024
  const int fixed = 4096 + kTaps * kTS * 4 + 1024;          // weights + projection buffer + alignment slack
  int ring = (227 * 1024 - 512 - fixed) / a.slot_bytes;
  if (ring > kMaxRing) ring = kMaxRing;
  S3D_CHECK_ARG(ring >= 2, "cls_soft_argmin: not enough shared memory");
  a.ring = ring;
  a.cols_x = ceil_div(w, kTX);  a.cols_y = ceil_div(h, kTY);
  const int64_t total = (int64_t)N * a.cols_x * a.cols_y;
  S3D_CHECK_ARG(total < (1ll << 31), "cls_soft_argmin: column count out of range");
  a.total_cols = (int)total;
  a.idesc = ptx::make_instr_desc(1, 128, kN);

  const CUtensorMapSwizzle sw = a.row_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                              : a.row_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B;
  CUtensorMap map_x, map_w;
  cuuint32_t box[5] = {(cuuint32_t)C, kHX, kHY, 1, 1};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  int rc = encode_act_map(&map_x, x, 2, false, C, w, h, D, N, box, estr, sw);
  if (rc != S3D_OK) return rc;
  rc = encode_weight_map(&map_w, w_taps, 2, false, C, kN, 1, C, kN, sw, 1);
  if (rc != S3D_OK) return rc;
  const int smem_bytes = a.ring * a.slot_bytes + fixed;
  auto kern = std_q ? (a.row_bytes == 128 ? cls_fused_kernel<4, true> : (a.row_bytes == 64 ? cls_fused_kernel<2, true> : cls_fused_kernel<1, true>))
                    : (a.row_bytes == 128 ? cls_fused_kernel<4, false> : (a.row_bytes == 64 ? cls_fused_kernel<2, false> : cls_fused_kernel<1, false>));
  S3D_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
  int grid = num_sms();
  if (grid > a.total_cols) grid = a.total_cols;
  kern<<<grid, kThreads, smem_bytes, static_cast<cudaStream_t>(stream)>>>(map_x, map_w, a);
  S3D_LAUNCH_CHECK();
  return S3D_OK;
}
