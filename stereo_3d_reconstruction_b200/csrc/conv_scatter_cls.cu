// Last aggregation layer + disparity classifier in ONE march: cls_a (3x3x3, 64 -> 64, BN, ReLU; the plane-scatter kernel of
// conv_scatter.cuh) whose output volume is never written.  The unfused pair wrote 2.1 GB (B = 64) from cls_a's epilogue and read
// it back one kernel later in cls_fused.cu -- a round trip of ~0.8 ms of HBM time per step, and 0.48 ms of kernel.
//
// The classifier cls_b is a Cout = 1 3x3x3 conv: cost[zc, yc, xc] = sum_{kz,ky,kx} Wb[kz,ky,kx,:] . Y[zc+kz-1, yc+ky-1, xc+kx-1, :]
// with Y = cls_a's output.  Fusing it as a gather would need the 3x3 halo of Y that OTHER CTAs compute (recomputing it costs a
// third M tile, +50 % MMAs).  So it runs in SCATTER form, per drained output plane z of the CTA's 32x8 patch:
//   1. the epilogue (thread = pixel) finishes Y = bf16(relu(acc + bias)) -- the same rounding as the stored tensor -- and writes it
//      to shared memory as a K-major 128-byte-row operand tile (128B swizzle; pixels outside the image are written as zero);
//   2. the issuer runs the PROJECTION on the tensor core: P[pixel, tap] = Y[pixel, :] . Wb[tap, :], 4 MMAs of N = 32 per tile into
//      the tile's spare TMEM columns [192, 224) (+4.6 % tensor work); Wb (4 KB) stays in shared memory;
//   3. one plane later the epilogue reads P back (27 values per pixel), stages it as T[tap][pixel] and every cell of the patch PLUS
//      ITS HALO RING (34 x 10 = 340 cells) gathers the taps of its <= 9 in-patch neighbours: the kz = 2 / 1 / 0 sums of plane z
//      belong to cost planes z-1 / z / z+1, held in three registers per cell (as in cls_fused.cu);
//   4. a finished cost plane is stored as the CTA's PARTIAL sums: partials[column][zc][340] fp32.  Interior cells are complete,
//      cells on the patch edge and in the ring also receive terms from the neighbouring patches' CTAs.
// A second small kernel adds, per pixel, the partial sums of the <= 4 patches that touch it IN A FIXED ORDER (deterministic, no
// atomics) and runs the soft-argmin: it reads 1.33 x N D h w x 4 bytes (89 MB at B = 64) instead of the 2.1 GB volume.
//
// Pipeline: drain d (global index over the CTA's planes) -> Y(d) -> projection(d) issued in the middle of input plane d + 2 ->
// P(d) consumed at drain d + 1's event, right after that plane's accumulator hand-back (which stays first, so the conv's MMA
// schedule is the plain kernel's).  Y(d) and T share one 32 KB buffer: three named barriers per event order the epilogue warps.
#include "conv_scatter.cuh"

namespace s3d {
namespace scatter {

constexpr int kCells = kHX * kHY;            // 340 cells of the halo'd patch
constexpr int kPCol = 192;                   // TMEM column of the projections inside a tile's 256
constexpr int kYBytes = 256 * 128;           // Y tile pair / T buffer (27 x 256 fp32 = 27 KB fits inside)

struct ClCtrl {
  ScCtrl c;
  uint64_t y_full[2], p_full[2], wb_full;
};

struct ClArgs {
  ScArgs a;
  float* partials;
};

struct ClIss {
  uint32_t y_u32, wb_u32;
  uint32_t bar_yf, bar_pf, bar_wb;
  uint32_t idesc_p;
};

// 4 MMAs (K = 64 channels) of tile t's Y against the classifier taps; D = the tile's projection columns.
template <bool kPair>
__device__ __forceinline__ void cl_project(const ScIssue& z, const ClIss& x, int t, uint32_t d) {
  ptx::mbar_wait_u32(x.bar_yf + 8 * t, d & 1u);
  ptx::tc_fence_after();
  const uint64_t hi = desc_hi(8 * 128, 128);
  const uint64_t yd = hi | desc_lo(x.y_u32 + t * (128 * 128)), wd = hi | desc_lo(x.wb_u32);
  if (ptx::elect_one()) {
#pragma unroll
    for (int k = 0; k < 4; ++k)
      sc_mma<false, kPair>(z.tmem_base + t * kTileCols + kPCol, yd + 2 * k, wd + 2 * k, x.idesc_p, k ? 1u : 0u);
    sc_commit<kPair>(x.bar_pf + 8 * t);
  }
  __syncwarp();
}

// sc_issue<bf16, TPS = 1, kPer = 4> + the projections: the one of drain gp - 2 goes out late in global plane gp (groups 6 / 7 of
// 9), when its Y tile has long been written, and is finished well before the plane's own drain event needs the result.
template <bool kPair>
__device__ __forceinline__ void cl_issue(const ScIssue& z, const ClIss& x) {
  constexpr int G = 9;
  int ws = 0;  uint32_t wphase = 0;
  int pw = 0;  uint32_t pwphase = 0;
  uint32_t aphase = 0;
  const uint32_t w_lo0 = desc_lo(z.w_u32), w_lo_step = z.w_bytes >> 4;
  const uint32_t x_lo0 = desc_lo(z.planes_u32), x_lo_step = z.slot_bytes >> 4;
  const uint32_t d0 = z.tmem_base, d1 = z.tmem_base + kTileCols;
  ptx::mbar_wait_u32(x.bar_wb, 0);
  const int nplanes = z.ncols * z.D;
  int gp = 0;
  for (int ci = 0; ci < z.ncols; ++ci) {
    for (int p = 0; p < z.D; ++p, ++gp) {
      ptx::mbar_wait_u32(z.bar_pf + 8 * pw, pwphase);
      const uint64_t xd0 = z.x_hi | (x_lo0 + pw * x_lo_step);
      const uint64_t xd1 = xd0 + z.tile_off;
      const uint32_t first = p == 0 ? 0u : 1u;
      int ws_prev = 0;
#pragma unroll
      for (int g = 0; g <= G; ++g) {
        if (g < G) {
          ptx::mbar_wait_u32(z.bar_wf + 8 * ws, wphase);
          if (g == 0) ptx::mbar_wait_u32(z.bar_ae, aphase ^ 1);
          ptx::tc_fence_after();
          const uint64_t wd = z.w_hi | (w_lo0 + ws * w_lo_step);
          if (ptx::elect_one()) {
            sc_issue_group<false, 1, 4, kPair, 1, false>(z, d0, xd0, wd, g, first);
            if (g == G - 1) sc_commit<kPair>(z.bar_af);
          }
          __syncwarp();
          if (g == 6 && gp >= 2) cl_project<kPair>(z, x, 0, (uint32_t)(gp - 2));
        }
        if (g >= 1) {
          if (g == 1) { ptx::mbar_wait_u32(z.bar_ae + 8, aphase ^ 1); ptx::tc_fence_after(); }
          const uint64_t wd = z.w_hi | (w_lo0 + ws_prev * w_lo_step);
          if (ptx::elect_one()) {
            sc_issue_group<false, 1, 4, kPair, 1, false>(z, d1, xd1, wd, g - 1, first);
            sc_commit<kPair>(z.bar_we + 8 * ws_prev);
            if (g == G) { sc_commit<kPair>(z.bar_af + 8); sc_commit<kPair>(z.bar_pe + 8 * pw); }
          }
          __syncwarp();
          if (g == 7 && gp >= 2) cl_project<kPair>(z, x, 1, (uint32_t)(gp - 2));
        }
        if (g < G) {
          ws_prev = ws;
          if (++ws == z.w_stages) { ws = 0; wphase ^= 1; }
        }
      }
      aphase ^= 1;
      if (++pw == z.ring) { pw = 0; pwphase ^= 1; }
    }
  }
  // the last two drains of the CTA have no later plane to ride on
  for (int d = nplanes >= 2 ? nplanes - 2 : 0; d < nplanes; ++d) {
    cl_project<kPair>(z, x, 0, (uint32_t)d);
    cl_project<kPair>(z, x, 1, (uint32_t)d);
  }
}

__device__ __forceinline__ void cl_bar() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

// Epilogue: warps 4-7 tile 0, 8-11 tile 1 (thread = pixel = TMEM lane), see the file header.
__device__ __forceinline__ void cl_epilogue(const ClArgs& ca, ClCtrl& ctrl, uint32_t tmem_base, uint8_t* ybuf, int warp, int lane) {
  const ScArgs& a = ca.a;
  constexpr int CP = 64;
  const int t = (warp - 4) >> 2, q = warp & 3;
  const uint32_t bar_af = ptx::smem_u32(&ctrl.c.acc_full[t]), bar_ae = ptx::smem_u32(&ctrl.c.acc_empty[t]);
  const uint32_t bar_yf = ptx::smem_u32(&ctrl.y_full[t]), bar_pf = ptx::smem_u32(&ctrl.p_full[t]);
  const uint32_t tbase = tmem_base + t * kTileCols + (static_cast<uint32_t>(q * 32) << 16);
  const int row = q * 32 + lane;                          // row of the tile's Y operand = TMEM lane
  const int yl = t * kTileY + (row >> 3), xl = row & 7;   // pixel inside the patch; its index in T is t * 128 + row = yl * 8 + xl
  float* T = reinterpret_cast<float*>(ybuf);
  uint8_t* yrow = ybuf + t * (128 * 128) + row * 128;
  const int D = a.dl;
  const int ncols = cta_cols(a);
  // the (up to two) cells this thread gathers: cell c = (yc + 1) * 10 + (xc + 1), yc in [-1, 32], xc in [-1, 8]
  const int et = (warp - 4) * 32 + lane;
  int cbase[2];  uint32_t cmask[2];
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int c = et + 256 * k;
    const int yc = c / kHX - 1, xc = c % kHX - 1;
    cbase[k] = (yc - 1) * 8 + (xc - 1);
    uint32_t m = 0;
#pragma unroll
    for (int ky = 0; ky < 3; ++ky)
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        const int py = yc + ky - 1, px = xc + kx - 1;
        if (c < kCells && py >= 0 && py < kTY && px >= 0 && px < kTX) m |= 1u << (ky * 3 + kx);
      }
    cmask[k] = m;
  }
  float cc[2][3] = {{0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}};    // partial costs of planes z-1, z, z+1 of the column being consumed
  bool have_prev = false;
  int prev_col = 0, prev_z = 0;
  uint32_t dcount = 0;                                    // global drain index of this CTA
  uint32_t aphase = 0;

  // consume P of drain d (column prev_col, plane prev_z): TMEM -> T -> gather -> partial cost planes
  auto consume = [&](uint32_t d) {
    ptx::mbar_wait_u32(bar_pf, d & 1u);
    ptx::tc_fence_after();
    uint32_t pr[2][16];
    ptx::tmem_ld16(tbase + kPCol, pr[0]);
    ptx::tmem_ld16(tbase + kPCol + 16, pr[1]);
    ptx::tmem_ld_wait();
    ptx::tc_fence_before();
    cl_bar();                                             // both tiles' Y have been read by the projection MMAs: the buffer is T now
#pragma unroll
    for (int tp = 0; tp < 27; ++tp) T[tp * 256 + t * 128 + row] = __uint_as_float(pr[tp >> 4][tp & 15]);
    cl_bar();
    const bool colok = prev_col < a.total_cols;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      if (k == 1 && et >= kCells - 256) break;
      float a0 = 0.f, a1 = 0.f, a2 = 0.f;                 // plane prev_z through kz = 2, 1, 0
#pragma unroll
      for (int j = 0; j < 9; ++j) {
        if ((cmask[k] >> j) & 1u) {
          const float* pp = T + j * 256 + cbase[k] + (j / 3) * 8 + (j % 3);
          a0 += pp[18 * 256];
          a1 += pp[9 * 256];
          a2 += pp[0];
        }
      }
      cc[k][0] += a0;  cc[k][1] += a1;  cc[k][2] += a2;
      float* dst = ca.partials + ((int64_t)prev_col * D) * kCells + et + 256 * k;
      if (prev_z >= 1 && colok) dst[(int64_t)(prev_z - 1) * kCells] = cc[k][0];
      cc[k][0] = cc[k][1];  cc[k][1] = cc[k][2];  cc[k][2] = 0.f;
      if (prev_z == D - 1) {
        if (colok) dst[(int64_t)(D - 1) * kCells] = cc[k][0];
        cc[k][0] = 0.f;  cc[k][1] = 0.f;
      }
    }
    cl_bar();                                             // everyone is done reading T: the buffer takes the next Y
  };

  for (int ci = 0; ci < ncols; ++ci) {
    const int colidx = blockIdx.x + ci * gridDim.x;
    const Col c = decode_col(a, colidx);
    const bool pixok = c.n < a.p.N && c.y0 + yl < a.p.oH && c.x0 + xl < a.p.oW;
    int slot = 0, z = 0;
    for (int p = 0; p < D; ++p) {
      const int ndrain = (p >= 1 ? 1 : 0) + (p == D - 1 ? 1 : 0);
      ptx::mbar_wait_u32(bar_af, aphase);
      ptx::tc_fence_after();
      if (ndrain == 0) {
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) { if (a.pair) ptx::mbar_arrive_cluster_u32(bar_ae, 0); else ptx::mbar_arrive_u32(bar_ae); }
      }
      for (int i = 0; i < ndrain; ++i) {
        uint32_t yb[CP / 2];                              // the pixel's 64 outputs as bf16 pairs
        {
          uint32_t v[CP / 16][16];
          const uint32_t taddr = tbase + slot * CP;
#pragma unroll
          for (int j = 0; j < CP / 16; ++j) ptx::tmem_ld16(taddr + 16 * j, v[j]);
          ptx::tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < CP / 16; ++j) ptx::tmem_st16_zero(taddr + 16 * j);
          ptx::tmem_st_wait();
          if (i == ndrain - 1) {                          // hand the tile back before anything else
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) { if (a.pair) ptx::mbar_arrive_cluster_u32(bar_ae, 0); else ptx::mbar_arrive_u32(bar_ae); }
          }
#pragma unroll
          for (int j = 0; j < CP / 16; ++j) {
            const float4* b4 = reinterpret_cast<const float4*>(a.bias + 16 * j);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float4 b = __ldg(b4 + e);
              const float f0 = fmax_nan(__uint_as_float(v[j][4 * e]) + b.x, 0.f), f1 = fmax_nan(__uint_as_float(v[j][4 * e + 1]) + b.y, 0.f);
              const float f2 = fmax_nan(__uint_as_float(v[j][4 * e + 2]) + b.z, 0.f), f3 = fmax_nan(__uint_as_float(v[j][4 * e + 3]) + b.w, 0.f);
              const __nv_bfloat162 h0 = __floats2bfloat162_rn(f0, f1), h1 = __floats2bfloat162_rn(f2, f3);
              yb[8 * j + 2 * e] = pixok ? *reinterpret_cast<const uint32_t*>(&h0) : 0u;
              yb[8 * j + 2 * e + 1] = pixok ? *reinterpret_cast<const uint32_t*>(&h1) : 0u;
            }
          }
        }
        if (have_prev) consume(dcount - 1);
        // Y(dcount): 8 chunks of 16 bytes, chunk j of row r at (j ^ (r & 7)) -- the 128B swizzle of the UMMA descriptor
#pragma unroll
        for (int j = 0; j < 8; ++j)
          *reinterpret_cast<uint4*>(yrow + ((j ^ (row & 7)) << 4)) = make_uint4(yb[4 * j], yb[4 * j + 1], yb[4 * j + 2], yb[4 * j + 3]);
        ptx::fence_proxy_async();
        __syncwarp();
        if (lane == 0) { if (a.pair) ptx::mbar_arrive_cluster_u32(bar_yf, 0); else ptx::mbar_arrive_u32(bar_yf); }
        have_prev = true;  prev_col = colidx;  prev_z = z;
        ++dcount;  ++z;
        if (++slot == 3) slot = 0;
      }
      aphase ^= 1;
    }
  }
  if (have_prev) consume(dcount - 1);
}

template <bool kPair>
__global__ void __launch_bounds__(kThreads, 1)
conv_scatter_cls_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w,
                        const __grid_constant__ CUtensorMap map_wb, const __grid_constant__ ClArgs ca) {
  const ScArgs& a = ca.a;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_w = smem + a.ring * a.slot_bytes;
  uint8_t* smem_y = smem_w + a.w_stages * a.w_bytes;          // Y tiles / T
  uint8_t* smem_wb = smem_y + kYBytes;                        // this CTA's classifier taps: [32 or 16 (pair)][128 B]
  __shared__ ClCtrl ctrl;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&map_x);  ptx::prefetch_tensormap(&map_w);  ptx::prefetch_tensormap(&map_wb);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < kMaxRing; ++s) { ptx::mbar_init(&ctrl.c.plane_full[s], 1); ptx::mbar_init(&ctrl.c.plane_empty[s], 1); }
    for (int s = 0; s < kMaxW; ++s) { ptx::mbar_init(&ctrl.c.w_full[s], 1); ptx::mbar_init(&ctrl.c.w_empty[s], 1); }
    for (int b = 0; b < 2; ++b) {
      ptx::mbar_init(&ctrl.c.acc_full[b], 1);  ptx::mbar_init(&ctrl.c.acc_empty[b], kPair ? 8 : 4);
      ptx::mbar_init(&ctrl.y_full[b], kPair ? 8 : 4);  ptx::mbar_init(&ctrl.p_full[b], 1);
    }
    ptx::mbar_init(&ctrl.wb_full, 1);
    ptx::fence_barrier_init();
  }
  if (warp == 2) { if (kPair) ptx::tmem_alloc_2sm(&ctrl.c.tmem_base, kTmemCols); else ptx::tmem_alloc(&ctrl.c.tmem_base, kTmemCols); }
  ptx::tc_fence_before();
  __syncthreads();
  if (kPair) ptx::cluster_sync_all();
  ptx::tc_fence_after();
  const uint32_t tmem_base = ctrl.c.tmem_base;

  if (warp == 0) {
    sc_produce<1, kPair>(a, ctrl.c, ptx::smem_u32(smem), ptx::smem_u32(smem_w), &map_x, &map_w);
  } else if (warp == 3) {
    // classifier taps, once: rows [16 rank, +16) of the [32][64] tap matrix in pair mode (each CTA holds half of B's N rows)
    const uint32_t bar = ptx::smem_u32(&ctrl.wb_full);
    if (ptx::elect_one()) {
      if (kPair) {
        const int crank = (int)ptx::cluster_ctarank();
        if (crank == 0) ptx::mbar_arrive_expect_tx_u32(bar, 2 * 16 * 128);
        ptx::tma_load_3d_2sm_u32(ptx::smem_u32(smem_wb), &map_wb, bar, 0, 16 * crank, 0);
      } else {
        ptx::mbar_arrive_expect_tx_u32(bar, 32 * 128);
        ptx::tma_load_3d_u32(ptx::smem_u32(smem_wb), &map_wb, bar, 0, 0, 0);
      }
    }
    __syncwarp();
  } else if (warp == 1 && (!kPair || ptx::cluster_ctarank() == 0)) {
    const int rb = a.row_bytes;
    const ScIssue zi = {tmem_base, ptx::smem_u32(smem), ptx::smem_u32(smem_w),
                        ptx::smem_u32(&ctrl.c.plane_full[0]), ptx::smem_u32(&ctrl.c.plane_empty[0]), ptx::smem_u32(&ctrl.c.w_full[0]),
                        ptx::smem_u32(&ctrl.c.w_empty[0]), ptx::smem_u32(&ctrl.c.acc_full[0]), ptx::smem_u32(&ctrl.c.acc_empty[0]),
                        desc_hi(kHX * rb, rb), desc_hi(8 * rb, rb), a.slot_bytes, a.w_bytes, a.w_stages, a.ring,
                        (uint32_t)(rb >> 4), (uint32_t)(((kPair ? 3 * a.cp / 2 : 3 * a.cp) * rb) >> 4), (uint32_t)((kTileY * kHX * rb) >> 4),
                        (uint32_t)(a.chunk_stride >> 4), a.idesc, a.dl, cta_cols(a)};
    const ClIss xi = {ptx::smem_u32(smem_y), ptx::smem_u32(smem_wb), ptx::smem_u32(&ctrl.y_full[0]), ptx::smem_u32(&ctrl.p_full[0]),
                      ptx::smem_u32(&ctrl.wb_full), ptx::make_instr_desc(1, kPair ? 256 : 128, 32)};
    cl_issue<kPair>(zi, xi);
  } else if (warp >= 4) {
    cl_epilogue(ca, ctrl, tmem_base, smem_y, warp, lane);
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (kPair) ptx::cluster_sync_all();
  if (warp == 2) {
    ptx::tc_fence_after();
    if (kPair) ptx::tmem_dealloc_2sm(tmem_base, kTmemCols); else ptx::tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ---- partial cost planes -> disparity -------------------------------------------------------------------------------------------
// One thread per pixel: cost[z] = own patch's cell + the cells of the neighbouring patches whose halo ring covers the pixel (left /
// right, up / down, diagonal -- always in this order), then the online soft-argmin over z (cls_fused.cu's arithmetic).
// kStd: also the distribution's standard deviation -> std_q (common.cuh, SoftSpread); disp is the same either way.
template <bool kStd>
__global__ void __launch_bounds__(256)
partials_soft_argmin_kernel(const float* __restrict__ partials, float* __restrict__ disp, int N, int D, int h, int w, int cols_x,
                            int cols_y, float sign, float* __restrict__ std_q) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)N * h * w) return;
  const int x = (int)(idx % w), y = (int)((idx / w) % h), n = (int)(idx / ((int64_t)w * h));
  const int px = x / kTX, py = y / kTY, xi = x % kTX, yi = y % kTY;
  const int dxn = xi == 0 ? -1 : (xi == kTX - 1 ? 1 : 0), dyn = yi == 0 ? -1 : (yi == kTY - 1 ? 1 : 0);
  const bool hx = dxn != 0 && px + dxn >= 0 && px + dxn < cols_x, hy = dyn != 0 && py + dyn >= 0 && py + dyn < cols_y;
  auto cell_ptr = [&](int ppy, int ppx, int yc, int xc) {
    const int64_t col = ((int64_t)n * cols_y + ppy) * cols_x + ppx;
    return partials + col * D * kCells + (yc + 1) * kHX + (xc + 1);
  };
  const float* p0 = cell_ptr(py, px, yi, xi);
  // in the neighbour's coordinates the pixel sits one step outside the patch: xc = -1 (right neighbour) or 8 (left neighbour)
  const float* p1 = hx ? cell_ptr(py, px + dxn, yi, dxn > 0 ? -1 : kTX) : nullptr;
  const float* p2 = hy ? cell_ptr(py + dyn, px, dyn > 0 ? -1 : kTY, xi) : nullptr;
  const float* p3 = (hx && hy) ? cell_ptr(py + dyn, px + dxn, dyn > 0 ? -1 : kTY, dxn > 0 ? -1 : kTX) : nullptr;
  float m = -INFINITY, s = 0.f, tt = 0.f;
  SoftSpread u;
  for (int z = 0; z < D; ++z) {
    const int64_t o = (int64_t)z * kCells;
    float c = p0[o];
    if (p1) c += p1[o];
    if (p2) c += p2[o];
    if (p3) c += p3[o];
    const float v = sign * c;
    if (v > m) {
      const float sc = expf(m - v); s *= sc; tt *= sc; m = v;
      if (kStd) { u.scale(sc);  u.move(z, s); }
    }
    const float e = expf(v - m);  s += e;  tt += e * (float)z;
    if (kStd) u.add(e, z);
  }
  disp[idx] = tt / s;
  if (kStd) std_q[idx] = u.sigma(tt / s, s);
}

}  // namespace scatter
}  // namespace s3d

extern "C" int64_t s3d_conv_cls_workspace_bytes(int N, int D, int h, int w) {
  using namespace s3d::scatter;
  return (int64_t)N * ((h + kTY - 1) / kTY) * ((w + kTX - 1) / kTX) * D * kCells * 4;
}

extern "C" int s3d_conv_cls_soft_argmin(const S3dConvParams* p_in, const void* in, const float* bias, const void* w_taps,
                                        void* workspace, float* disp, float* std_q, float sign, void* stream) {
  using namespace s3d;
  using namespace s3d::scatter;
  if (!p_in || !in || !bias || !w_taps || !workspace || !disp) { set_error("conv_cls_soft_argmin: null argument"); return S3D_ERR_INVALID; }
  const S3dConvParams& p = *p_in;
  S3D_CHECK_ARG(p.w_nstack != nullptr, "conv_cls_soft_argmin: the layer needs host-packed rotations (w_nstack)");
  S3D_CHECK_ARG(plane_scatter_layer(p) && p.in_dtype == S3D_DTYPE_BF16 && p.Cin == 64 && p.Cout == 64 && p.act == S3D_ACT_RELU,
                "conv_cls_soft_argmin: needs a bf16 stride-1 3x3x3 64 -> 64 ReLU layer in canonical tap order");
  S3D_CHECK_ARG(((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(w_taps) | reinterpret_cast<uintptr_t>(workspace)) & 15) == 0,
                "conv_cls_soft_argmin: pointers must be 16-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);

  ClArgs ca;
  memset(&ca, 0, sizeof(ca));
  ScArgs& a = ca.a;
  a.p = p;  a.bias = bias;  a.residual = nullptr;  a.out = nullptr;
  ca.partials = static_cast<float*>(workspace);
  const int64_t total = plane_geometry(a, 128, 64, 1);
  a.cp = 64;  a.tps = 1;
  S3D_CHECK_ARG(total >= 2 && total < (1ll << 31), "conv_cls_soft_argmin: needs at least two columns (CTA pairs)");
  a.pair = 1;
  const int grid = deal_columns(a, total, num_sms());
  const int w_rows = 3 * a.cp / 2;
  a.w_tx = w_rows * 128;
  a.w_bytes = align1024(a.w_tx);
  const int extra = kYBytes + 2048;
  const int budget = 227 * 1024 - 1024 - 640 - extra;
  a.ring = 3;
  a.w_stages = (budget - a.ring * a.slot_bytes) / a.w_bytes;
  if (a.w_stages > kMaxW) a.w_stages = kMaxW;
  S3D_CHECK_ARG(a.w_stages >= 3, "conv_cls_soft_argmin: not enough shared memory");
  a.idesc = ptx::make_instr_desc(1, 256, 3 * a.cp);
  a.fast_store = 1;  a.res_direct = 1;

  CUtensorMap map_x, map_w, map_wb;
  cuuint32_t box[5] = {64, kHX, kHY, 1, 1};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  int rc = encode_act_map(&map_x, in, 2, false, 64, p.iW, p.iH, p.iD, p.N, box, estr, CU_TENSOR_MAP_SWIZZLE_128B);
  if (rc != S3D_OK) return rc;
  rc = encode_weight_map(&map_w, p.w_nstack, 2, false, 64, 3 * a.cp, 36, 64, w_rows, CU_TENSOR_MAP_SWIZZLE_128B, 1);
  if (rc != S3D_OK) return rc;
  rc = encode_weight_map(&map_wb, w_taps, 2, false, 64, 32, 1, 64, 16, CU_TENSOR_MAP_SWIZZLE_128B, 1);
  if (rc != S3D_OK) return rc;

  const int smem_bytes = a.ring * a.slot_bytes + a.w_stages * a.w_bytes + extra + 1024;
  rc = launch_plane_scatter(conv_scatter_cls_kernel<true>, grid, smem_bytes, a.pair, st, map_x, map_w, map_wb, ca);
  if (rc != S3D_OK) return rc;
  const int64_t npix = (int64_t)p.N * p.oH * p.oW;
  const unsigned blocks = (unsigned)((npix + 255) / 256);
  if (std_q)
    partials_soft_argmin_kernel<true><<<blocks, 256, 0, st>>>(ca.partials, disp, p.N, p.oD, p.oH, p.oW, a.cols_x, a.cols_y, sign, std_q);
  else
    partials_soft_argmin_kernel<false><<<blocks, 256, 0, st>>>(ca.partials, disp, p.N, p.oD, p.oH, p.oW, a.cols_x, a.cols_y, sign,
                                                               nullptr);
  S3D_LAUNCH_CHECK();
  return S3D_OK;
}
