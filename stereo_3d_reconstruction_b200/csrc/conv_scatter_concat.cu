// Cost volume + first aggregation layer in one kernel: the plane-scatter 3x3x3 conv (conv_scatter.cuh) reading a concat
// volume that is never written.  Plane d of volume n is [ ref(y, x) | tgt(y, x -/+ d) ] (SURVEY 8 row V; the reference half
// is the SAME feature map for every d, the target half is the other view shifted by d, zero outside the image), so
//   * the reference half of a 32x8 patch is staged ONCE per column (two buffers, so the next column's is in flight) and is
//     the K-chunk 0 operand of all D planes;
//   * the target half of plane d is one TMA box of the other view's feature map through a SKEWED tensor map: the map's X
//     and D dimensions have the same stride (one pixel), i.e. coordinate (x, d) addresses pixel x + d (right reference)
//     or, with d counted downwards from a base moved D-1 pixels left, pixel x - d (left reference).  X keeps its real
//     bound, so both conv halos are TMA zero fill; the shifted-out pixels land in the zero margins the feature rows are
//     stored with (pad >= D-1 pixels on both sides).  Checked stand-alone with scripts/tma_skew.cu.
// The 2.1 GB volume (B = 64), its write (0.34 ms at 96 % of HBM peak) and its read by the conv disappear; the MMA
// sequence is the K-chunked one of conv_scatter.cuh (chunk 0 = reference channels, chunk 1 = target channels), so the
// result is bit-identical to concat_volume_kernel + conv_scatter_kernel.
#include "conv_scatter.cuh"

namespace s3d {
namespace scatter {

struct CcCtrl {
  ScCtrl c;
  uint64_t ref_full[2], ref_empty[2];
};

struct CcArgs {
  ScArgs a;
  int n_half;          // B: volumes [0, B) are left-referenced, [B, 2B) right-referenced
  int D;
};

template <bool kPair>
__device__ __forceinline__ void cc_produce(const CcArgs& ca, CcCtrl& ctrl, uint32_t ref_u32, uint32_t planes_u32, uint32_t w_u32,
                                           const CUtensorMap* map_ref, const CUtensorMap* map_tl, const CUtensorMap* map_tr,
                                           const CUtensorMap* map_w) {
  const ScArgs& a = ca.a;
  constexpr int G = 9;                             // one weight stage per tap: [reference-channel rows][target-channel rows]
  const uint32_t bar_pf = ptx::smem_u32(&ctrl.c.plane_full[0]), bar_pe = ptx::smem_u32(&ctrl.c.plane_empty[0]);
  const uint32_t bar_wf = ptx::smem_u32(&ctrl.c.w_full[0]), bar_we = ptx::smem_u32(&ctrl.c.w_empty[0]);
  const uint32_t bar_rf = ptx::smem_u32(&ctrl.ref_full[0]), bar_re = ptx::smem_u32(&ctrl.ref_empty[0]);
  const int D = ca.D, ring = a.ring, w_stages = a.w_stages, ncols = cta_cols(a);
  const int slot_bytes = a.slot_bytes, w_bytes = a.w_bytes, w_tx = a.w_tx, kc = a.kc, B = ca.n_half;
  const int crank = kPair ? (int)ptx::cluster_ctarank() : 0;
  const bool leader = crank == 0;
  const int w_row0 = kPair ? crank * (3 * a.cp / 2) : 0;
  const int plane_tx = kPlaneRows * a.row_bytes;
  const uint32_t mult = kPair ? 2u : 1u;           // the leader's barriers collect the bytes of both CTAs
  int ws = 0;  uint32_t wphase = 0;
  int pslot = 0;  uint32_t pphase = 0;
  int pci = 0, pj = 0, issued = 0;
  Col pc = decode_col(a, blockIdx.x);
  auto load = [&](uint32_t dst, const CUtensorMap* m, uint32_t bf, int c1, int c2, int c3, int c4) {
    if (kPair) ptx::tma_load_5d_2sm_u32(dst, m, bf, 0, c1, c2, c3, c4);
    else       ptx::tma_load_5d_u32(dst, m, bf, 0, c1, c2, c3, c4);
  };
  auto issue_plane = [&](bool blocking) -> bool {
    if (pci >= ncols) return false;
    if (pj == 0) {
      // first plane of a column: its reference half goes out first (buffer pci & 1, free once column pci-2 is done);
      // only when called blocking, so that an opportunistic call never stalls the weight stream on it
      const int rb_ = pci & 1;
      const uint32_t rpar = ((uint32_t)(pci >> 1) & 1u) ^ 1u;
      if (blocking) ptx::mbar_wait_u32(bar_re + 8 * rb_, rpar);
      else if (!ptx::mbar_test_wait_u32(bar_re + 8 * rb_, rpar)) return false;
    }
    const uint32_t be = bar_pe + 8 * pslot, bf = bar_pf + 8 * pslot;
    if (blocking) ptx::mbar_wait_u32(be, pphase ^ 1);
    else if (!ptx::mbar_test_wait_u32(be, pphase ^ 1)) return false;
    if (ptx::elect_one()) {
      if (pj == 0) {
        const uint32_t rf = bar_rf + 8 * (pci & 1);
        if (leader) ptx::mbar_arrive_expect_tx_u32(rf, mult * plane_tx);
        load(ref_u32 + (pci & 1) * slot_bytes, map_ref, rf, pc.x0 - 1, pc.y0 - 1, 0, pc.n);          // dims (C, X, Y, 1, 2B)
      }
      if (leader) ptx::mbar_arrive_expect_tx_u32(bf, mult * plane_tx);
      // target half: dims (C, X, D, Y, B).  Left reference: pixel x - d = (x, D-1-d) on the map based D-1 pixels to the left
      if (pc.n < B) load(planes_u32 + pslot * slot_bytes, map_tl, bf, pc.x0 - 1, D - 1 - pj, pc.y0 - 1, pc.n);
      else          load(planes_u32 + pslot * slot_bytes, map_tr, bf, pc.x0 - 1, pj, pc.y0 - 1, pc.n - B);
    }
    __syncwarp();
    ++issued;
    if (++pslot == ring) { pslot = 0; pphase ^= 1; }
    if (++pj == D) {
      pj = 0;  ++pci;
      if (pci < ncols) pc = decode_col(a, blockIdx.x + pci * gridDim.x);
    }
    return true;
  };
  int gp = 0;
  for (int ci = 0; ci < ncols; ++ci) {
    int rot = 3;
    for (int p = 0; p < D; ++p, ++gp) {
      while (issued <= gp) issue_plane(true);
      const int ahead = gp + ring;
#pragma unroll
      for (int g = 0; g < G; ++g) {
        if (issued < ahead) issue_plane(false);
        const uint32_t be = bar_we + 8 * ws, bf = bar_wf + 8 * ws;
        ptx::mbar_wait_u32(be, wphase ^ 1);
        if (ptx::elect_one()) {
          if (leader) ptx::mbar_arrive_expect_tx_u32(bf, mult * w_tx);
#pragma unroll
          for (int ch = 0; ch < 2; ++ch) {
            if (kPair) ptx::tma_load_3d_2sm_u32(w_u32 + ws * w_bytes + ch * (w_tx >> 1), map_w, bf, ch * kc, w_row0, rot * 9 + g);
            else       ptx::tma_load_3d_u32(w_u32 + ws * w_bytes + ch * (w_tx >> 1), map_w, bf, ch * kc, 0, rot * 9 + g);
          }
        }
        __syncwarp();
        if (++ws == w_stages) { ws = 0; wphase ^= 1; }
      }
      rot = (p == 0) ? 1 : (rot == 2 ? 0 : rot + 1);
    }
  }
}

struct CcIssue {
  ScIssue z;
  uint32_t ref_u32, bar_rf, bar_re;
};

// One tap = one weight stage: kPer MMAs on the reference buffer (K chunk 0), then kPer on the target slot (K chunk 1).
template <bool kTF32, int kPer, bool kPair>
__device__ __forceinline__ void cc_issue_group(const ScIssue& z, uint32_t d_tmem, uint64_t rdesc, uint64_t xdesc, uint64_t wdesc, int g,
                                               uint32_t first) {
  const uint32_t xoff = ((g / 3) * kHX + (g % 3)) * z.rb16;
#pragma unroll
  for (int ch = 0; ch < 2; ++ch) {
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
      const uint32_t acc = (g == 0 && ch == 0 && k == 0) ? first : 1u;
      const uint64_t ad = (ch ? xdesc : rdesc) + xoff + 2 * k, bd = wdesc + ch * z.chunk_step + 2 * k;
      if (kPair) { if (kTF32) ptx::mma_tf32_2sm(d_tmem, ad, bd, z.idesc, acc); else ptx::mma_bf16_2sm(d_tmem, ad, bd, z.idesc, acc); }
      else       { if (kTF32) ptx::mma_tf32(d_tmem, ad, bd, z.idesc, acc);     else ptx::mma_bf16(d_tmem, ad, bd, z.idesc, acc); }
    }
  }
}

// Same schedule as sc_issue (tile 1 trails tile 0 by one weight stage); K chunk 0 of every tap reads the column's
// reference buffer, chunk 1 the plane's target slot.
template <bool kTF32, int kPer, bool kPair>
__device__ __forceinline__ void cc_issue(const CcIssue& ci_) {
  const ScIssue& z = ci_.z;
  constexpr int G = 9;
  int ws = 0;  uint32_t wphase = 0;
  int pw = 0;  uint32_t pwphase = 0;
  uint32_t aphase = 0;
  const uint32_t w_lo0 = desc_lo(z.w_u32), w_lo_step = z.w_bytes >> 4;
  const uint32_t x_lo0 = desc_lo(z.planes_u32), x_lo_step = z.slot_bytes >> 4;
  const uint32_t r_lo0 = desc_lo(ci_.ref_u32);
  const uint32_t d0 = z.tmem_base, d1 = z.tmem_base + kTileCols;
  for (int ci = 0; ci < z.ncols; ++ci) {
    const int rbuf = ci & 1;
    ptx::mbar_wait_u32(ci_.bar_rf + 8 * rbuf, (uint32_t)(ci >> 1) & 1u);
    const uint64_t rd0 = z.x_hi | (r_lo0 + rbuf * x_lo_step), rd1 = rd0 + z.tile_off;
    for (int p = 0; p < z.D; ++p) {
      ptx::mbar_wait_u32(z.bar_pf + 8 * pw, pwphase);
      const uint64_t xd0 = z.x_hi | (x_lo0 + pw * x_lo_step), xd1 = xd0 + z.tile_off;
      const uint32_t first = p == 0 ? 0u : 1u;
      const bool last_plane = p == z.D - 1;
      int ws_prev = 0;
#pragma unroll
      for (int g = 0; g <= G; ++g) {
        if (g < G) {
          ptx::mbar_wait_u32(z.bar_wf + 8 * ws, wphase);
          if (g == 0) ptx::mbar_wait_u32(z.bar_ae, aphase ^ 1);
          ptx::tc_fence_after();
          const uint64_t wd = z.w_hi | (w_lo0 + ws * w_lo_step);
          if (ptx::elect_one()) {
            cc_issue_group<kTF32, kPer, kPair>(z, d0, rd0, xd0, wd, g, first);
            if (g == G - 1) sc_commit<kPair>(z.bar_af);
          }
          __syncwarp();
        }
        if (g >= 1) {
          if (g == 1) { ptx::mbar_wait_u32(z.bar_ae + 8, aphase ^ 1); ptx::tc_fence_after(); }
          const uint64_t wd = z.w_hi | (w_lo0 + ws_prev * w_lo_step);
          if (ptx::elect_one()) {
            cc_issue_group<kTF32, kPer, kPair>(z, d1, rd1, xd1, wd, g - 1, first);
            sc_commit<kPair>(z.bar_we + 8 * ws_prev);
            if (g == G) {
              sc_commit<kPair>(z.bar_af + 8);
              sc_commit<kPair>(z.bar_pe + 8 * pw);
              if (last_plane) sc_commit<kPair>(ci_.bar_re + 8 * rbuf);      // the column's reference buffer is free
            }
          }
          __syncwarp();
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
}

template <bool kTF32, bool kPair, int kPer, bool kLean>
__global__ void __launch_bounds__(kThreads, 1)
conv_scatter_concat_kernel(const __grid_constant__ CUtensorMap map_ref, const __grid_constant__ CUtensorMap map_tl,
                           const __grid_constant__ CUtensorMap map_tr, const __grid_constant__ CUtensorMap map_w,
                           const __grid_constant__ CcArgs ca) {
  const ScArgs& a = ca.a;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_planes = smem + 2 * a.slot_bytes;              // [ref 0][ref 1][target ring][weights]
  uint8_t* smem_w = smem_planes + a.ring * a.slot_bytes;
  __shared__ CcCtrl ctrl;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&map_ref);  ptx::prefetch_tensormap(&map_tl);
    ptx::prefetch_tensormap(&map_tr);   ptx::prefetch_tensormap(&map_w);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < kMaxRing; ++s) { ptx::mbar_init(&ctrl.c.plane_full[s], 1); ptx::mbar_init(&ctrl.c.plane_empty[s], 1); }
    for (int s = 0; s < kMaxW; ++s) { ptx::mbar_init(&ctrl.c.w_full[s], 1); ptx::mbar_init(&ctrl.c.w_empty[s], 1); }
    for (int b = 0; b < 2; ++b) {
      ptx::mbar_init(&ctrl.c.acc_full[b], 1);  ptx::mbar_init(&ctrl.c.acc_empty[b], kPair ? 8 : 4);
      ptx::mbar_init(&ctrl.ref_full[b], 1);    ptx::mbar_init(&ctrl.ref_empty[b], 1);
    }
    ptx::fence_barrier_init();
  }
  if (warp == 2) { if (kPair) ptx::tmem_alloc_2sm(&ctrl.c.tmem_base, kTmemCols); else ptx::tmem_alloc(&ctrl.c.tmem_base, kTmemCols); }
  ptx::tc_fence_before();
  __syncthreads();
  if (kPair) ptx::cluster_sync_all();
  ptx::tc_fence_after();
  const uint32_t tmem_base = ctrl.c.tmem_base;

  if (warp == 0) {
    cc_produce<kPair>(ca, ctrl, ptx::smem_u32(smem), ptx::smem_u32(smem_planes), ptx::smem_u32(smem_w), &map_ref, &map_tl, &map_tr,
                      &map_w);
  } else if (warp == 1 && (!kPair || ptx::cluster_ctarank() == 0)) {
    const int rb = a.row_bytes;
    const CcIssue zi = {{tmem_base, ptx::smem_u32(smem_planes), ptx::smem_u32(smem_w),
                         ptx::smem_u32(&ctrl.c.plane_full[0]), ptx::smem_u32(&ctrl.c.plane_empty[0]), ptx::smem_u32(&ctrl.c.w_full[0]),
                         ptx::smem_u32(&ctrl.c.w_empty[0]), ptx::smem_u32(&ctrl.c.acc_full[0]), ptx::smem_u32(&ctrl.c.acc_empty[0]),
                         desc_hi(kHX * rb, rb), desc_hi(8 * rb, rb), a.slot_bytes, a.w_bytes, a.w_stages, a.ring,
                         (uint32_t)(rb >> 4), 0u, (uint32_t)((kTileY * kHX * rb) >> 4), (uint32_t)(a.w_tx >> 5), a.idesc, ca.D, cta_cols(a)},
                        ptx::smem_u32(smem), ptx::smem_u32(&ctrl.ref_full[0]), ptx::smem_u32(&ctrl.ref_empty[0])};
    cc_issue<kTF32, kPer, kPair>(zi);
  } else if (warp >= 4) {
    if constexpr (kLean) sc_epilogue<64, __nv_bfloat16, true, 0, 0>(a, ctrl.c, tmem_base, warp, lane);
    else if (a.cp == 64) sc_epilogue_dispatch<64>(a, ctrl.c, tmem_base, warp, lane);
    else if (a.cp == 48) sc_epilogue_dispatch<48>(a, ctrl.c, tmem_base, warp, lane);
    else if (a.cp == 32) sc_epilogue_dispatch<32>(a, ctrl.c, tmem_base, warp, lane);
    else sc_epilogue_dispatch<16>(a, ctrl.c, tmem_base, warp, lane);
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (kPair) ptx::cluster_sync_all();
  if (warp == 2) {
    ptx::tc_fence_after();
    if (kPair) ptx::tmem_dealloc_2sm(tmem_base, kTmemCols); else ptx::tmem_dealloc(tmem_base, kTmemCols);
  }
}

// =====================================================================================================================
// Reference-once mode.  The reference half of the concat volume is the SAME feature map on every disparity plane, so its
// contribution to output plane z is a 2-D convolution that does not depend on z (for interior planes):
//     out[z] = sum_kz ( ref (*) W[kz, :, ref ch] + tgt_{z+kz-1} (*) W[kz, :, tgt ch] )   over the planes z+kz-1 inside [0, D)
//            = R + (plane-scatter conv over the TARGET half only),      R = ref (*) sum_kz W[kz, :, ref ch]
// with the two border planes missing one kz each: out[0] has no kz = 0 term, out[D-1] no kz = 2 term.  So per column
//   1. R is computed ONCE (9 taps x kPer MMAs per tile, N = Cout) into the tile's spare TMEM columns [3 Cout, 4 Cout); the
//      epilogue folds the bias into it (R' = R + bias, written back with tcgen05.st) when the column's first plane is done;
//   2. the D planes run the plane-scatter MMAs on the target half only: K = C instead of 2C, HALF the tensor-core work of
//      the layer (this layer is 15 % of the forward);
//   3. the epilogue adds R' to every drained plane instead of the bias: no extra arithmetic, no bias loads;
//   4. the border corrections are more MMAs into the border planes' own accumulator slots: ref (*) (-W[kz=0]) into the slot
//      of out[0] after input plane 0, ref (*) (-W[kz=2]) into the slot of out[D-1] after input plane D-1.
// The three small weight sets [sum_kz W | -W[kz=0] | -W[kz=2]] x 9 taps x [Cout][C] are packed by the host
// (s3d_conv_concat_volume_ro's w_refonce) and stream through the same weight ring as extra stages.  Per column that is 27 taps
// of N = Cout MMAs on top of D x 9 taps of N = 3 Cout ones: ~5 % at D = 32.  Not bit-identical to the unfused path (sum_kz W is
// rounded to bf16 once, and the accumulation order differs); tests hold it to the engine's tolerance instead.
//
// With K halved a weight stage of ONE tap is only kPer MMAs per tile (192 tensor cycles at C = 32): the first version of this
// kernel ran the tensor pipe at 58 % because the issuer's per-stage overhead (barrier wait, election, commit) and the one-stage
// lead of tile 0 over tile 1 no longer hid behind the MMAs (ncu: profiles/r2_ncu_summary.md).  So a stage here holds kTps = 3
// taps, and the two tiles are interleaved as T0g0 T0g1 T1g0 T0g2 T1g1 T1g2: BOTH tiles get two groups (12 kPer MMAs) of the
// other tile's work between their last MMA of plane p and their first of plane p+1 to hide the accumulator hand-back.
constexpr int kTps = 3;                  // in-plane taps per weight stage
constexpr int kGr = 9 / kTps;            // stages (groups) per plane

struct RoArgs {
  CcArgs c;
  int w_tx_r;          // bytes of one special weight stage per CTA
  uint32_t idesc_r;    // instruction descriptor of the N = Cout MMAs
};

template <bool kPair>
__device__ __forceinline__ void ro_produce(const RoArgs& ra, CcCtrl& ctrl, uint32_t ref_u32, uint32_t planes_u32, uint32_t w_u32,
                                           const CUtensorMap* map_ref, const CUtensorMap* map_tl, const CUtensorMap* map_tr,
                                           const CUtensorMap* map_w, const CUtensorMap* map_wr) {
  const CcArgs& ca = ra.c;
  const ScArgs& a = ca.a;
  const uint32_t bar_pf = ptx::smem_u32(&ctrl.c.plane_full[0]), bar_pe = ptx::smem_u32(&ctrl.c.plane_empty[0]);
  const uint32_t bar_wf = ptx::smem_u32(&ctrl.c.w_full[0]), bar_we = ptx::smem_u32(&ctrl.c.w_empty[0]);
  const uint32_t bar_rf = ptx::smem_u32(&ctrl.ref_full[0]), bar_re = ptx::smem_u32(&ctrl.ref_empty[0]);
  const int D = ca.D, ring = a.ring, w_stages = a.w_stages, ncols = cta_cols(a);
  const int slot_bytes = a.slot_bytes, w_bytes = a.w_bytes, w_tx = a.w_tx, kc = a.kc, B = ca.n_half;
  const int crank = kPair ? (int)ptx::cluster_ctarank() : 0;
  const bool leader = crank == 0;
  const int w_row0 = kPair ? crank * (3 * a.cp / 2) : 0;
  const int w_row0_r = kPair ? crank * (a.cp / 2) : 0;
  const int plane_tx = kPlaneRows * a.row_bytes;
  const uint32_t mult = kPair ? 2u : 1u;
  int ws = 0;  uint32_t wphase = 0;
  int pslot = 0;  uint32_t pphase = 0;
  int pci = 0, pj = 0, issued = 0;
  Col pc = decode_col(a, blockIdx.x);
  auto load = [&](uint32_t dst, const CUtensorMap* m, uint32_t bf, int c1, int c2, int c3, int c4) {
    if (kPair) ptx::tma_load_5d_2sm_u32(dst, m, bf, 0, c1, c2, c3, c4);
    else       ptx::tma_load_5d_u32(dst, m, bf, 0, c1, c2, c3, c4);
  };
  auto issue_plane = [&](bool blocking) -> bool {
    if (pci >= ncols) return false;
    if (pj == 0) {
      const int rb_ = pci & 1;
      const uint32_t rpar = ((uint32_t)(pci >> 1) & 1u) ^ 1u;
      if (blocking) ptx::mbar_wait_u32(bar_re + 8 * rb_, rpar);
      else if (!ptx::mbar_test_wait_u32(bar_re + 8 * rb_, rpar)) return false;
    }
    const uint32_t be = bar_pe + 8 * pslot, bf = bar_pf + 8 * pslot;
    if (blocking) ptx::mbar_wait_u32(be, pphase ^ 1);
    else if (!ptx::mbar_test_wait_u32(be, pphase ^ 1)) return false;
    if (ptx::elect_one()) {
      if (pj == 0) {
        const uint32_t rf = bar_rf + 8 * (pci & 1);
        if (leader) ptx::mbar_arrive_expect_tx_u32(rf, mult * plane_tx);
        load(ref_u32 + (pci & 1) * slot_bytes, map_ref, rf, pc.x0 - 1, pc.y0 - 1, 0, pc.n);
      }
      if (leader) ptx::mbar_arrive_expect_tx_u32(bf, mult * plane_tx);
      if (pc.n < B) load(planes_u32 + pslot * slot_bytes, map_tl, bf, pc.x0 - 1, D - 1 - pj, pc.y0 - 1, pc.n);
      else          load(planes_u32 + pslot * slot_bytes, map_tr, bf, pc.x0 - 1, pj, pc.y0 - 1, pc.n - B);
    }
    __syncwarp();
    ++issued;
    if (++pslot == ring) { pslot = 0; pphase ^= 1; }
    if (++pj == D) {
      pj = 0;  ++pci;
      if (pci < ncols) pc = decode_col(a, blockIdx.x + pci * gridDim.x);
    }
    return true;
  };
  // one weight stage: kTps taps of the stacked rotation (target-channel columns only) or of a special set
  auto stage = [&](const CUtensorMap* m, int c0, int row0, int tap, int tx) {
    const uint32_t be = bar_we + 8 * ws, bf = bar_wf + 8 * ws;
    ptx::mbar_wait_u32(be, wphase ^ 1);
    if (ptx::elect_one()) {
      if (leader) ptx::mbar_arrive_expect_tx_u32(bf, mult * tx);
      if (kPair) ptx::tma_load_3d_2sm_u32(w_u32 + ws * w_bytes, m, bf, c0, row0, tap);
      else       ptx::tma_load_3d_u32(w_u32 + ws * w_bytes, m, bf, c0, row0, tap);
    }
    __syncwarp();
    if (++ws == w_stages) { ws = 0; wphase ^= 1; }
  };
  auto emit_special = [&](int set) {
#pragma unroll 1
    for (int g = 0; g < kGr; ++g) stage(map_wr, 0, w_row0_r, set * 9 + g * kTps, ra.w_tx_r);
  };
  int gp = 0;
  for (int ci = 0; ci < ncols; ++ci) {
    while (issued <= gp) issue_plane(true);          // the column's reference buffer (+ plane 0) goes out BEFORE its weights
    emit_special(0);                                 // sum_kz W[kz]: the issuer computes R first
    int rot = 3;
    for (int p = 0; p < D; ++p, ++gp) {
      while (issued <= gp) issue_plane(true);
      const int ahead = gp + ring;
#pragma unroll
      for (int g = 0; g < kGr; ++g) {
        if (issued < ahead) issue_plane(false);
        stage(map_w, kc, w_row0, rot * 9 + g * kTps, w_tx);
      }
      if (p == 0) emit_special(1);                   // -W[kz=0] into out[0]
      if (p == D - 1) emit_special(2);               // -W[kz=2] into out[D-1]
      rot = (p == 0) ? 1 : (rot == 2 ? 0 : rot + 1);
    }
  }
}

struct RoIssue {
  CcIssue c;
  uint32_t idesc_r;
  int cp;
  uint32_t tap_step_r;     // 16-byte units between the taps of a special stage
};

// One group = kTps taps x kPer MMAs of one tile; tap_step = z.tap_step (plane stages) or the special stages' own.
template <int kPer, bool kPair>
__device__ __forceinline__ void ro_group(const ScIssue& z, uint32_t d_tmem, uint64_t adesc, uint64_t wdesc, int g, uint32_t tap_step,
                                         uint32_t idesc, uint32_t acc0) {
#pragma unroll
  for (int tt = 0; tt < kTps; ++tt) {
    const int kyx = g * kTps + tt;
    const uint32_t xoff = ((kyx / 3) * kHX + (kyx % 3)) * z.rb16;
#pragma unroll
    for (int k = 0; k < kPer; ++k)
      sc_mma<false, kPair>(d_tmem, adesc + xoff + 2 * k, wdesc + tt * tap_step + 2 * k, idesc, (tt == 0 && k == 0) ? acc0 : 1u);
  }
}

template <int kPer, bool kPair>
__device__ __forceinline__ void ro_issue(const RoIssue& ri) {
  const CcIssue& ci_ = ri.c;
  const ScIssue& z = ci_.z;
  static_assert(kGr == 3, "the tile interleave below is written out for three groups per plane");
  int ws = 0;  uint32_t wphase = 0;
  int pw = 0;  uint32_t pwphase = 0;
  uint32_t aphase = 0;
  const uint32_t w_lo0 = desc_lo(z.w_u32), w_lo_step = z.w_bytes >> 4;
  const uint32_t x_lo0 = desc_lo(z.planes_u32), x_lo_step = z.slot_bytes >> 4;
  const uint32_t r_lo0 = desc_lo(ci_.ref_u32);
  const uint32_t d0 = z.tmem_base, d1 = z.tmem_base + kTileCols;
  // three special stages: N = Cout MMAs of the column's reference buffer into TMEM columns `col` of both tiles
  auto special = [&](uint64_t rd0, uint64_t rd1, uint32_t col, bool overwrite) {
#pragma unroll
    for (int g = 0; g < kGr; ++g) {
      ptx::mbar_wait_u32(z.bar_wf + 8 * ws, wphase);
      ptx::tc_fence_after();
      const uint64_t wd = z.w_hi | (w_lo0 + ws * w_lo_step);
      if (ptx::elect_one()) {
        const uint32_t acc0 = (overwrite && g == 0) ? 0u : 1u;
        ro_group<kPer, kPair>(z, d0 + col, rd0, wd, g, ri.tap_step_r, ri.idesc_r, acc0);
        ro_group<kPer, kPair>(z, d1 + col, rd1, wd, g, ri.tap_step_r, ri.idesc_r, acc0);
        sc_commit<kPair>(z.bar_we + 8 * ws);
      }
      __syncwarp();
      if (++ws == z.w_stages) { ws = 0; wphase ^= 1; }
    }
  };
  for (int ci = 0; ci < z.ncols; ++ci) {
    const int rbuf = ci & 1;
    ptx::mbar_wait_u32(ci_.bar_rf + 8 * rbuf, (uint32_t)(ci >> 1) & 1u);
    const uint64_t rd0 = z.x_hi | (r_lo0 + rbuf * x_lo_step), rd1 = rd0 + z.tile_off;
    // R into the spare columns: both tiles' epilogues must have finished with the previous column's R' (they hand the last
    // plane of a column back only after reading it)
    ptx::mbar_wait_u32(z.bar_ae, aphase ^ 1);
    ptx::mbar_wait_u32(z.bar_ae + 8, aphase ^ 1);
    ptx::tc_fence_after();
    special(rd0, rd1, 3u * ri.cp, true);
    for (int p = 0; p < z.D; ++p) {
      ptx::mbar_wait_u32(z.bar_pf + 8 * pw, pwphase);
      const uint64_t xd0 = z.x_hi | (x_lo0 + pw * x_lo_step), xd1 = xd0 + z.tile_off;
      const uint32_t first = p == 0 ? 0u : 1u;
      const bool last_plane = p == z.D - 1;
      const bool border = p == 0 || last_plane;       // accumulator hand-over is delayed until the corrections are in
      // the plane's three weight stages (ring positions ws, ws+1, ws+2); order T0g0 T0g1 T1g0 T0g2 T1g1 T1g2
      uint32_t wsl[3], wph[3];
      {
        int s = ws;  uint32_t ph = wphase;
#pragma unroll
        for (int g = 0; g < 3; ++g) { wsl[g] = s; wph[g] = ph; if (++s == z.w_stages) { s = 0; ph ^= 1; } }
        ws = s;  wphase = ph;
      }
      auto wdesc = [&](int g) { return z.w_hi | (w_lo0 + wsl[g] * w_lo_step); };
      // T0g0
      ptx::mbar_wait_u32(z.bar_wf + 8 * wsl[0], wph[0]);
      ptx::mbar_wait_u32(z.bar_ae, aphase ^ 1);
      ptx::tc_fence_after();
      if (ptx::elect_one()) ro_group<kPer, kPair>(z, d0, xd0, wdesc(0), 0, z.tap_step, z.idesc, first);
      __syncwarp();
      // T0g1, T1g0
      ptx::mbar_wait_u32(z.bar_wf + 8 * wsl[1], wph[1]);
      ptx::mbar_wait_u32(z.bar_ae + 8, aphase ^ 1);
      ptx::tc_fence_after();
      if (ptx::elect_one()) {
        ro_group<kPer, kPair>(z, d0, xd0, wdesc(1), 1, z.tap_step, z.idesc, 1u);
        ro_group<kPer, kPair>(z, d1, xd1, wdesc(0), 0, z.tap_step, z.idesc, first);
        sc_commit<kPair>(z.bar_we + 8 * wsl[0]);
      }
      __syncwarp();
      // T0g2, T1g1, T1g2
      ptx::mbar_wait_u32(z.bar_wf + 8 * wsl[2], wph[2]);
      ptx::tc_fence_after();
      if (ptx::elect_one()) {
        ro_group<kPer, kPair>(z, d0, xd0, wdesc(2), 2, z.tap_step, z.idesc, 1u);
        if (!border) sc_commit<kPair>(z.bar_af);
        ro_group<kPer, kPair>(z, d1, xd1, wdesc(1), 1, z.tap_step, z.idesc, 1u);
        sc_commit<kPair>(z.bar_we + 8 * wsl[1]);
        ro_group<kPer, kPair>(z, d1, xd1, wdesc(2), 2, z.tap_step, z.idesc, 1u);
        sc_commit<kPair>(z.bar_we + 8 * wsl[2]);
        if (!border) sc_commit<kPair>(z.bar_af + 8);
        sc_commit<kPair>(z.bar_pe + 8 * pw);
      }
      __syncwarp();
      if (border) {
        if (p == 0) special(rd0, rd1, 0u, false);                                        // out[0] lives in slot 0
        if (last_plane) special(rd0, rd1, (uint32_t)((z.D - 1) % 3) * ri.cp, false);      // out[D-1] in slot (D-1) % 3
        if (ptx::elect_one()) {
          sc_commit<kPair>(z.bar_af);
          sc_commit<kPair>(z.bar_af + 8);
          if (last_plane) sc_commit<kPair>(ci_.bar_re + 8 * rbuf);                        // the column's reference buffer is free
        }
        __syncwarp();
      }
      aphase ^= 1;
      if (++pw == z.ring) { pw = 0; pwphase ^= 1; }
    }
  }
}

// Epilogue of the reference-once kernel (Cout = 64, bf16 out, ReLU, transposed coalesced stores; cf. sc_epilogue<64, bf16, true>).
// The tile's TMEM columns [192, 256) hold R; when the column's first plane is done this thread adds the bias to its pixel's R and
// writes R' back; every drained plane is then acc + R'.  R' is read in two halves AFTER the accumulator hand-back (the issuer
// only rewrites it for the next column), except for the last plane of a column, which hands back once R' is in registers.
__device__ __forceinline__ void ro_pack16(const uint32_t (&v)[16], const uint32_t (&r)[16], uint4& c0, uint4& c1) {
  float f[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) f[i] = fmax_nan(__uint_as_float(v[i]) + __uint_as_float(r[i]), 0.f);
  __nv_bfloat162* h0 = reinterpret_cast<__nv_bfloat162*>(&c0);
  __nv_bfloat162* h1 = reinterpret_cast<__nv_bfloat162*>(&c1);
#pragma unroll
  for (int i = 0; i < 4; ++i) { h0[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);  h1[i] = __floats2bfloat162_rn(f[8 + 2 * i], f[9 + 2 * i]); }
}

__device__ __forceinline__ void ro_epilogue(const ScArgs& a, ScCtrl& ctrl, uint32_t tmem_base, int warp, int lane) {
  constexpr int CP = 64, NCH = 8;
  const int t = (warp - 4) >> 2, q = warp & 3;
  const uint32_t bar_af = ptx::smem_u32(&ctrl.acc_full[t]), bar_ae = ptx::smem_u32(&ctrl.acc_empty[t]);
  const uint32_t tbase = tmem_base + t * kTileCols + (static_cast<uint32_t>(q * 32) << 16);
  const uint32_t raddr = tbase + 3 * CP;
  const int yl = t * kTileY + q * 4 + (lane >> 3);       // a transpose group = the 8 pixels of one tile row
  const int D = a.dl;
  const int osW = (int)a.p.osW;
  uint32_t aphase = 0;
  const int ncols = cta_cols(a);
  auto hand_back = [&]() {
    ptx::tc_fence_before();
    __syncwarp();
    if (lane == 0) { if (a.pair) ptx::mbar_arrive_cluster_u32(bar_ae, 0); else ptx::mbar_arrive_u32(bar_ae); }
  };
  for (int ci = 0; ci < ncols; ++ci) {
    const Col c = decode_col(a, blockIdx.x + ci * gridDim.x);
    const bool rowok = c.y0 + yl < a.p.oH && c.n < a.p.N;
    const int64_t grp_off = (int64_t)c.n * a.p.osN + (int64_t)(c.y0 + yl) * a.p.osH + (int64_t)c.x0 * a.p.osW;
    uint32_t okmask = 0;
#pragma unroll
    for (int k = 0; k < NCH; ++k) okmask |= (rowok && c.x0 + k < a.p.oW) ? (1u << k) : 0u;
    int slot = 0, z = 0;
    for (int p = 0; p < D; ++p) {
      const int ndrain = (p >= 1 ? 1 : 0) + (p == D - 1 ? 1 : 0);
      ptx::mbar_wait_u32(bar_af, aphase);
      ptx::tc_fence_after();
      if (p == 0) {                                      // R is complete (it was issued before plane 0): R' = R + bias
#pragma unroll
        for (int j = 0; j < CP / 16; ++j) {
          uint32_t r[16];
          ptx::tmem_ld16(raddr + 16 * j, r);
          ptx::tmem_ld_wait();
          const float4* b4 = reinterpret_cast<const float4*>(a.bias + 16 * j);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float4 b = __ldg(b4 + i);
            r[4 * i] = __float_as_uint(__uint_as_float(r[4 * i]) + b.x);          r[4 * i + 1] = __float_as_uint(__uint_as_float(r[4 * i + 1]) + b.y);
            r[4 * i + 2] = __float_as_uint(__uint_as_float(r[4 * i + 2]) + b.z);  r[4 * i + 3] = __float_as_uint(__uint_as_float(r[4 * i + 3]) + b.w);
          }
          ptx::tmem_st16(raddr + 16 * j, r);
        }
        ptx::tmem_st_wait();
      }
      if (ndrain == 0) hand_back();
      for (int i = 0; i < ndrain; ++i) {
        uint32_t v[CP / 16][16];
        const uint32_t taddr = tbase + slot * CP;
#pragma unroll
        for (int j = 0; j < CP / 16; ++j) ptx::tmem_ld16(taddr + 16 * j, v[j]);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < CP / 16; ++j) ptx::tmem_st16_zero(taddr + 16 * j);
        ptx::tmem_st_wait();
        const bool last_of_col = p == D - 1 && i == ndrain - 1;
        if (i == ndrain - 1 && !last_of_col) hand_back();
        uint32_t ra[16], rb[16];
        uint4 cc[NCH];
        ptx::tmem_ld16(raddr, ra);  ptx::tmem_ld16(raddr + 16, rb);
        ptx::tmem_ld_wait();
        ro_pack16(v[0], ra, cc[0], cc[1]);
        ro_pack16(v[1], rb, cc[2], cc[3]);
        ptx::tmem_ld16(raddr + 32, ra);  ptx::tmem_ld16(raddr + 48, rb);
        ptx::tmem_ld_wait();
        if (last_of_col) hand_back();
        ro_pack16(v[2], ra, cc[4], cc[5]);
        ro_pack16(v[3], rb, cc[6], cc[7]);
        chunk_transpose<NCH>(cc, lane);
        const uint32_t om = z < a.p.oD ? okmask : 0u;
        __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(a.out) + grp_off + (int64_t)z * a.p.osD + (lane & (NCH - 1)) * 8;
#pragma unroll
        for (int k = 0; k < NCH; ++k)
          if ((om >> k) & 1u) *reinterpret_cast<uint4*>(o + k * osW) = cc[k];
        ++z;
        if (++slot == 3) slot = 0;
      }
      aphase ^= 1;
    }
  }
}

template <bool kPair, int kPer>
__global__ void __launch_bounds__(kThreads, 1)
conv_scatter_concat_ro_kernel(const __grid_constant__ CUtensorMap map_ref, const __grid_constant__ CUtensorMap map_tl,
                              const __grid_constant__ CUtensorMap map_tr, const __grid_constant__ CUtensorMap map_w,
                              const __grid_constant__ CUtensorMap map_wr, const __grid_constant__ RoArgs ra) {
  const CcArgs& ca = ra.c;
  const ScArgs& a = ca.a;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_planes = smem + 2 * a.slot_bytes;
  uint8_t* smem_w = smem_planes + a.ring * a.slot_bytes;
  __shared__ CcCtrl ctrl;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&map_ref);  ptx::prefetch_tensormap(&map_tl);  ptx::prefetch_tensormap(&map_tr);
    ptx::prefetch_tensormap(&map_w);    ptx::prefetch_tensormap(&map_wr);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < kMaxRing; ++s) { ptx::mbar_init(&ctrl.c.plane_full[s], 1); ptx::mbar_init(&ctrl.c.plane_empty[s], 1); }
    for (int s = 0; s < kMaxW; ++s) { ptx::mbar_init(&ctrl.c.w_full[s], 1); ptx::mbar_init(&ctrl.c.w_empty[s], 1); }
    for (int b = 0; b < 2; ++b) {
      ptx::mbar_init(&ctrl.c.acc_full[b], 1);  ptx::mbar_init(&ctrl.c.acc_empty[b], kPair ? 8 : 4);
      ptx::mbar_init(&ctrl.ref_full[b], 1);    ptx::mbar_init(&ctrl.ref_empty[b], 1);
    }
    ptx::fence_barrier_init();
  }
  if (warp == 2) { if (kPair) ptx::tmem_alloc_2sm(&ctrl.c.tmem_base, kTmemCols); else ptx::tmem_alloc(&ctrl.c.tmem_base, kTmemCols); }
  ptx::tc_fence_before();
  __syncthreads();
  if (kPair) ptx::cluster_sync_all();
  ptx::tc_fence_after();
  const uint32_t tmem_base = ctrl.c.tmem_base;

  if (warp == 0) {
    ro_produce<kPair>(ra, ctrl, ptx::smem_u32(smem), ptx::smem_u32(smem_planes), ptx::smem_u32(smem_w), &map_ref, &map_tl, &map_tr,
                      &map_w, &map_wr);
  } else if (warp == 1 && (!kPair || ptx::cluster_ctarank() == 0)) {
    const int rb = a.row_bytes;
    const int w_rows = kPair ? 3 * a.cp / 2 : 3 * a.cp, w_rows_r = kPair ? a.cp / 2 : a.cp;
    const RoIssue zi = {{{tmem_base, ptx::smem_u32(smem_planes), ptx::smem_u32(smem_w),
                          ptx::smem_u32(&ctrl.c.plane_full[0]), ptx::smem_u32(&ctrl.c.plane_empty[0]), ptx::smem_u32(&ctrl.c.w_full[0]),
                          ptx::smem_u32(&ctrl.c.w_empty[0]), ptx::smem_u32(&ctrl.c.acc_full[0]), ptx::smem_u32(&ctrl.c.acc_empty[0]),
                          desc_hi(kHX * rb, rb), desc_hi(8 * rb, rb), a.slot_bytes, a.w_bytes, a.w_stages, a.ring,
                          (uint32_t)(rb >> 4), (uint32_t)((w_rows * rb) >> 4), (uint32_t)((kTileY * kHX * rb) >> 4), 0u, a.idesc, ca.D,
                          cta_cols(a)},
                         ptx::smem_u32(smem), ptx::smem_u32(&ctrl.ref_full[0]), ptx::smem_u32(&ctrl.ref_empty[0])},
                        ra.idesc_r, a.cp, (uint32_t)((w_rows_r * rb) >> 4)};
    ro_issue<kPer, kPair>(zi);
  } else if (warp >= 4) {
    ro_epilogue(a, ctrl.c, tmem_base, warp, lane);
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (kPair) ptx::cluster_sync_all();
  if (warp == 2) {
    ptx::tc_fence_after();
    if (kPair) ptx::tmem_dealloc_2sm(tmem_base, kTmemCols); else ptx::tmem_dealloc(tmem_base, kTmemCols);
  }
}

// =====================================================================================================================
// Reference-once mode on SPLIT (BF16X2, 'bf16x3') operands: feature rows are [hi(C) | lo(C)] (C = 32: 128 bytes), every
// product runs as hi*hi + lo*hi + hi*lo.  Same column march as above; per tap and tile 6 MMAs instead of 2, so a weight stage
// is ONE tap again (the plain split kernel's pacing) and the tiles keep sc_issue's one-group stagger.
//   planes / reference buffers   340 rows x 128 B (128B swizzle): hi half at +0, lo half at +64 B of every row
//   plane weight stage           target-channel columns of the stacked rotation, hi part and lo part as two 64-byte-row tiles
//                                (64B swizzle): [w_hi: 96 rows x 64 B][w_lo: 96 rows x 64 B]
//   special weight stage         [32 rows][hi(32) | lo(32)] = 128-byte rows (128B swizzle) of w_refonce
// The epilogue adds R' (R + bias, folded once per column) and writes hi = bf16(v), lo = bf16(v - hi) as two transposed passes.
struct RosIssue {
  CcIssue c;
  uint64_t w64_hi;         // descriptor high part of the 64-byte-row weight tiles
  uint32_t wlo_off;        // 16-byte units from the w_hi tile to the w_lo tile of a plane stage
  uint32_t idesc_r;
  int cp;
};

template <bool kPair>
__device__ __forceinline__ void ros_produce(const RoArgs& ra, CcCtrl& ctrl, uint32_t ref_u32, uint32_t planes_u32, uint32_t w_u32,
                                            const CUtensorMap* map_ref, const CUtensorMap* map_tl, const CUtensorMap* map_tr,
                                            const CUtensorMap* map_w, const CUtensorMap* map_wr) {
  const CcArgs& ca = ra.c;
  const ScArgs& a = ca.a;
  const uint32_t bar_pf = ptx::smem_u32(&ctrl.c.plane_full[0]), bar_pe = ptx::smem_u32(&ctrl.c.plane_empty[0]);
  const uint32_t bar_wf = ptx::smem_u32(&ctrl.c.w_full[0]), bar_we = ptx::smem_u32(&ctrl.c.w_empty[0]);
  const uint32_t bar_rf = ptx::smem_u32(&ctrl.ref_full[0]), bar_re = ptx::smem_u32(&ctrl.ref_empty[0]);
  const int D = ca.D, ring = a.ring, w_stages = a.w_stages, ncols = cta_cols(a);
  const int slot_bytes = a.slot_bytes, w_bytes = a.w_bytes, w_tx = a.w_tx, kc = a.kc, B = ca.n_half;
  const int crank = kPair ? (int)ptx::cluster_ctarank() : 0;
  const bool leader = crank == 0;
  const int w_row0 = kPair ? crank * (3 * a.cp / 2) : 0;
  const int w_row0_r = kPair ? crank * (a.cp / 2) : 0;
  const int plane_tx = kPlaneRows * a.row_bytes;
  const uint32_t mult = kPair ? 2u : 1u;
  int ws = 0;  uint32_t wphase = 0;
  int pslot = 0;  uint32_t pphase = 0;
  int pci = 0, pj = 0, issued = 0;
  Col pc = decode_col(a, blockIdx.x);
  auto load = [&](uint32_t dst, const CUtensorMap* m, uint32_t bf, int c1, int c2, int c3, int c4) {
    if (kPair) ptx::tma_load_5d_2sm_u32(dst, m, bf, 0, c1, c2, c3, c4);
    else       ptx::tma_load_5d_u32(dst, m, bf, 0, c1, c2, c3, c4);
  };
  auto issue_plane = [&](bool blocking) -> bool {
    if (pci >= ncols) return false;
    if (pj == 0) {
      const int rb_ = pci & 1;
      const uint32_t rpar = ((uint32_t)(pci >> 1) & 1u) ^ 1u;
      if (blocking) ptx::mbar_wait_u32(bar_re + 8 * rb_, rpar);
      else if (!ptx::mbar_test_wait_u32(bar_re + 8 * rb_, rpar)) return false;
    }
    const uint32_t be = bar_pe + 8 * pslot, bf = bar_pf + 8 * pslot;
    if (blocking) ptx::mbar_wait_u32(be, pphase ^ 1);
    else if (!ptx::mbar_test_wait_u32(be, pphase ^ 1)) return false;
    if (ptx::elect_one()) {
      if (pj == 0) {
        const uint32_t rf = bar_rf + 8 * (pci & 1);
        if (leader) ptx::mbar_arrive_expect_tx_u32(rf, mult * plane_tx);
        load(ref_u32 + (pci & 1) * slot_bytes, map_ref, rf, pc.x0 - 1, pc.y0 - 1, 0, pc.n);
      }
      if (leader) ptx::mbar_arrive_expect_tx_u32(bf, mult * plane_tx);
      if (pc.n < B) load(planes_u32 + pslot * slot_bytes, map_tl, bf, pc.x0 - 1, D - 1 - pj, pc.y0 - 1, pc.n);
      else          load(planes_u32 + pslot * slot_bytes, map_tr, bf, pc.x0 - 1, pj, pc.y0 - 1, pc.n - B);
    }
    __syncwarp();
    ++issued;
    if (++pslot == ring) { pslot = 0; pphase ^= 1; }
    if (++pj == D) {
      pj = 0;  ++pci;
      if (pci < ncols) pc = decode_col(a, blockIdx.x + pci * gridDim.x);
    }
    return true;
  };
  auto plane_stage = [&](int tap) {
    const uint32_t be = bar_we + 8 * ws, bf = bar_wf + 8 * ws;
    ptx::mbar_wait_u32(be, wphase ^ 1);
    if (ptx::elect_one()) {
      if (leader) ptx::mbar_arrive_expect_tx_u32(bf, mult * w_tx);
      const uint32_t dst = w_u32 + ws * w_bytes;
      // physical weight row: [hi(ref C | tgt C) | lo(ref C | tgt C)] -> target-hi at column C, target-lo at column 3 C
      if (kPair) { ptx::tma_load_3d_2sm_u32(dst, map_w, bf, kc, w_row0, tap);  ptx::tma_load_3d_2sm_u32(dst + (w_tx >> 1), map_w, bf, 3 * kc, w_row0, tap); }
      else       { ptx::tma_load_3d_u32(dst, map_w, bf, kc, w_row0, tap);      ptx::tma_load_3d_u32(dst + (w_tx >> 1), map_w, bf, 3 * kc, w_row0, tap); }
    }
    __syncwarp();
    if (++ws == w_stages) { ws = 0; wphase ^= 1; }
  };
  auto emit_special = [&](int set) {
#pragma unroll 1
    for (int g = 0; g < 9; ++g) {
      const uint32_t be = bar_we + 8 * ws, bf = bar_wf + 8 * ws;
      ptx::mbar_wait_u32(be, wphase ^ 1);
      if (ptx::elect_one()) {
        if (leader) ptx::mbar_arrive_expect_tx_u32(bf, mult * ra.w_tx_r);
        if (kPair) ptx::tma_load_3d_2sm_u32(w_u32 + ws * w_bytes, map_wr, bf, 0, w_row0_r, set * 9 + g);
        else       ptx::tma_load_3d_u32(w_u32 + ws * w_bytes, map_wr, bf, 0, w_row0_r, set * 9 + g);
      }
      __syncwarp();
      if (++ws == w_stages) { ws = 0; wphase ^= 1; }
    }
  };
  int gp = 0;
  for (int ci = 0; ci < ncols; ++ci) {
    while (issued <= gp) issue_plane(true);
    emit_special(0);
    int rot = 3;
    for (int p = 0; p < D; ++p, ++gp) {
      while (issued <= gp) issue_plane(true);
      const int ahead = gp + ring;
#pragma unroll 1
      for (int g = 0; g < 9; ++g) {
        if (issued < ahead) issue_plane(false);
        plane_stage(rot * 9 + g);
      }
      if (p == 0) emit_special(1);
      if (p == D - 1) emit_special(2);
      rot = (p == 0) ? 1 : (rot == 2 ? 0 : rot + 1);
    }
  }
}

// One tap of one tile on split operands: (x_hi, w_hi), (x_lo, w_hi), (x_hi, w_lo); the lo half of an A row starts 64 bytes in.
template <bool kPair>
__device__ __forceinline__ void ros_tap(uint32_t d_tmem, uint64_t ad, uint64_t wd_hi, uint64_t wd_lo, uint32_t idesc, uint32_t acc0) {
#pragma unroll
  for (int k = 0; k < 2; ++k) sc_mma<false, kPair>(d_tmem, ad + 2 * k, wd_hi + 2 * k, idesc, k == 0 ? acc0 : 1u);
#pragma unroll
  for (int k = 0; k < 2; ++k) sc_mma<false, kPair>(d_tmem, ad + 4 + 2 * k, wd_hi + 2 * k, idesc, 1u);
#pragma unroll
  for (int k = 0; k < 2; ++k) sc_mma<false, kPair>(d_tmem, ad + 2 * k, wd_lo + 2 * k, idesc, 1u);
}

template <bool kPair>
__device__ __forceinline__ void ros_issue(const RosIssue& ri) {
  const CcIssue& ci_ = ri.c;
  const ScIssue& z = ci_.z;
  constexpr int G = 9;
  int ws = 0;  uint32_t wphase = 0;
  int pw = 0;  uint32_t pwphase = 0;
  uint32_t aphase = 0;
  const uint32_t w_lo0 = desc_lo(z.w_u32), w_lo_step = z.w_bytes >> 4;
  const uint32_t x_lo0 = desc_lo(z.planes_u32), x_lo_step = z.slot_bytes >> 4;
  const uint32_t r_lo0 = desc_lo(ci_.ref_u32);
  const uint32_t d0 = z.tmem_base, d1 = z.tmem_base + kTileCols;
  auto tap_off = [&](int g) { return (uint32_t)(((g / 3) * kHX + (g % 3)) * z.rb16); };
  // nine special stages (128-byte-row tile: w_hi at +0, w_lo at +64 B) of the column's reference buffer into columns `col`
  auto special = [&](uint64_t rd0, uint64_t rd1, uint32_t col, bool overwrite) {
#pragma unroll 1
    for (int g = 0; g < G; ++g) {
      ptx::mbar_wait_u32(z.bar_wf + 8 * ws, wphase);
      ptx::tc_fence_after();
      const uint64_t wd = z.w_hi | (w_lo0 + ws * w_lo_step);
      if (ptx::elect_one()) {
        const uint32_t acc0 = (overwrite && g == 0) ? 0u : 1u;
        const uint32_t xo = tap_off(g);
        ros_tap<kPair>(d0 + col, rd0 + xo, wd, wd + 4, ri.idesc_r, acc0);
        ros_tap<kPair>(d1 + col, rd1 + xo, wd, wd + 4, ri.idesc_r, acc0);
        sc_commit<kPair>(z.bar_we + 8 * ws);
      }
      __syncwarp();
      if (++ws == z.w_stages) { ws = 0; wphase ^= 1; }
    }
  };
  for (int ci = 0; ci < z.ncols; ++ci) {
    const int rbuf = ci & 1;
    ptx::mbar_wait_u32(ci_.bar_rf + 8 * rbuf, (uint32_t)(ci >> 1) & 1u);
    const uint64_t rd0 = z.x_hi | (r_lo0 + rbuf * x_lo_step), rd1 = rd0 + z.tile_off;
    ptx::mbar_wait_u32(z.bar_ae, aphase ^ 1);
    ptx::mbar_wait_u32(z.bar_ae + 8, aphase ^ 1);
    ptx::tc_fence_after();
    special(rd0, rd1, 3u * ri.cp, true);
    for (int p = 0; p < z.D; ++p) {
      ptx::mbar_wait_u32(z.bar_pf + 8 * pw, pwphase);
      const uint64_t xd0 = z.x_hi | (x_lo0 + pw * x_lo_step), xd1 = xd0 + z.tile_off;
      const uint32_t first = p == 0 ? 0u : 1u;
      const bool last_plane = p == z.D - 1;
      const bool border = p == 0 || last_plane;
      int ws_prev = 0;
#pragma unroll
      for (int g = 0; g <= G; ++g) {
        if (g < G) {
          ptx::mbar_wait_u32(z.bar_wf + 8 * ws, wphase);
          if (g == 0) ptx::mbar_wait_u32(z.bar_ae, aphase ^ 1);
          ptx::tc_fence_after();
          const uint64_t wd = ri.w64_hi | (w_lo0 + ws * w_lo_step);
          if (ptx::elect_one()) {
            ros_tap<kPair>(d0, xd0 + tap_off(g), wd, wd + ri.wlo_off, z.idesc, g == 0 ? first : 1u);
            if (g == G - 1 && !border) sc_commit<kPair>(z.bar_af);
          }
          __syncwarp();
        }
        if (g >= 1) {
          if (g == 1) { ptx::mbar_wait_u32(z.bar_ae + 8, aphase ^ 1); ptx::tc_fence_after(); }
          const uint64_t wd = ri.w64_hi | (w_lo0 + ws_prev * w_lo_step);
          if (ptx::elect_one()) {
            ros_tap<kPair>(d1, xd1 + tap_off(g - 1), wd, wd + ri.wlo_off, z.idesc, g == 1 ? first : 1u);
            sc_commit<kPair>(z.bar_we + 8 * ws_prev);
            if (g == G) {
              if (!border) sc_commit<kPair>(z.bar_af + 8);
              sc_commit<kPair>(z.bar_pe + 8 * pw);
            }
          }
          __syncwarp();
        }
        if (g < G) {
          ws_prev = ws;
          if (++ws == z.w_stages) { ws = 0; wphase ^= 1; }
        }
      }
      if (border) {
        if (p == 0) special(rd0, rd1, 0u, false);
        if (last_plane) special(rd0, rd1, (uint32_t)((z.D - 1) % 3) * ri.cp, false);
        if (ptx::elect_one()) {
          sc_commit<kPair>(z.bar_af);
          sc_commit<kPair>(z.bar_af + 8);
          if (last_plane) sc_commit<kPair>(ci_.bar_re + 8 * rbuf);
        }
        __syncwarp();
      }
      aphase ^= 1;
      if (++pw == z.ring) { pw = 0; pwphase ^= 1; }
    }
  }
}

// ro_epilogue on split outputs: [hi(64) | lo(64)] bf16 per pixel, lo parts os_lo elements after the hi parts.
__device__ __forceinline__ void ros_epilogue(const ScArgs& a, ScCtrl& ctrl, uint32_t tmem_base, int warp, int lane) {
  constexpr int CP = 64, NCH = 8;
  const int t = (warp - 4) >> 2, q = warp & 3;
  const uint32_t bar_af = ptx::smem_u32(&ctrl.acc_full[t]), bar_ae = ptx::smem_u32(&ctrl.acc_empty[t]);
  const uint32_t tbase = tmem_base + t * kTileCols + (static_cast<uint32_t>(q * 32) << 16);
  const uint32_t raddr = tbase + 3 * CP;
  const int yl = t * kTileY + q * 4 + (lane >> 3);
  const int D = a.dl;
  const int osW = (int)a.p.osW;
  const int64_t os_lo = a.os_lo;
  uint32_t aphase = 0;
  const int ncols = cta_cols(a);
  auto hand_back = [&]() {
    ptx::tc_fence_before();
    __syncwarp();
    if (lane == 0) { if (a.pair) ptx::mbar_arrive_cluster_u32(bar_ae, 0); else ptx::mbar_arrive_u32(bar_ae); }
  };
  for (int ci = 0; ci < ncols; ++ci) {
    const Col c = decode_col(a, blockIdx.x + ci * gridDim.x);
    const bool rowok = c.y0 + yl < a.p.oH && c.n < a.p.N;
    const int64_t grp_off = (int64_t)c.n * a.p.osN + (int64_t)(c.y0 + yl) * a.p.osH + (int64_t)c.x0 * a.p.osW;
    uint32_t okmask = 0;
#pragma unroll
    for (int k = 0; k < NCH; ++k) okmask |= (rowok && c.x0 + k < a.p.oW) ? (1u << k) : 0u;
    int slot = 0, z = 0;
    for (int p = 0; p < D; ++p) {
      const int ndrain = (p >= 1 ? 1 : 0) + (p == D - 1 ? 1 : 0);
      ptx::mbar_wait_u32(bar_af, aphase);
      ptx::tc_fence_after();
      if (p == 0) {                                      // R' = R + bias
#pragma unroll
        for (int j = 0; j < CP / 16; ++j) {
          uint32_t r[16];
          ptx::tmem_ld16(raddr + 16 * j, r);
          ptx::tmem_ld_wait();
          const float4* b4 = reinterpret_cast<const float4*>(a.bias + 16 * j);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float4 b = __ldg(b4 + i);
            r[4 * i] = __float_as_uint(__uint_as_float(r[4 * i]) + b.x);          r[4 * i + 1] = __float_as_uint(__uint_as_float(r[4 * i + 1]) + b.y);
            r[4 * i + 2] = __float_as_uint(__uint_as_float(r[4 * i + 2]) + b.z);  r[4 * i + 3] = __float_as_uint(__uint_as_float(r[4 * i + 3]) + b.w);
          }
          ptx::tmem_st16(raddr + 16 * j, r);
        }
        ptx::tmem_st_wait();
      }
      if (ndrain == 0) hand_back();
      for (int i = 0; i < ndrain; ++i) {
        uint32_t v[CP / 16][16];
        const uint32_t taddr = tbase + slot * CP;
#pragma unroll
        for (int j = 0; j < CP / 16; ++j) ptx::tmem_ld16(taddr + 16 * j, v[j]);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < CP / 16; ++j) ptx::tmem_st16_zero(taddr + 16 * j);
        ptx::tmem_st_wait();
        const bool last_of_col = p == D - 1 && i == ndrain - 1;
        if (i == ndrain - 1 && !last_of_col) hand_back();
        // v <- relu(v + R') as fp32 bits, R' read in two halves
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          uint32_t ra[16], rb[16];
          ptx::tmem_ld16(raddr + 32 * hh, ra);  ptx::tmem_ld16(raddr + 32 * hh + 16, rb);
          ptx::tmem_ld_wait();
          if (hh == 1 && last_of_col) hand_back();
#pragma unroll
          for (int e = 0; e < 16; ++e) {
            v[2 * hh][e] = __float_as_uint(fmax_nan(__uint_as_float(v[2 * hh][e]) + __uint_as_float(ra[e]), 0.f));
            v[2 * hh + 1][e] = __float_as_uint(fmax_nan(__uint_as_float(v[2 * hh + 1][e]) + __uint_as_float(rb[e]), 0.f));
          }
        }
        const uint32_t om = z < a.p.oD ? okmask : 0u;
        __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(a.out) + grp_off + (int64_t)z * a.p.osD + (lane & (NCH - 1)) * 8;
#pragma unroll
        for (int half = 0; half < 2; ++half) {           // 0: hi parts, 1: lo parts
          uint4 cc[NCH];
#pragma unroll
          for (int jg = 0; jg < CP / 16; ++jg) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              uint32_t w4[4];
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                uint32_t hi, lo;
                split_bf16x2(__uint_as_float(v[jg][8 * h + 2 * e]), __uint_as_float(v[jg][8 * h + 2 * e + 1]), hi, lo);
                w4[e] = half == 0 ? hi : lo;
              }
              cc[2 * jg + h] = make_uint4(w4[0], w4[1], w4[2], w4[3]);
            }
          }
          chunk_transpose<NCH>(cc, lane);
          __nv_bfloat16* oh = o + (half == 0 ? (int64_t)0 : os_lo);
#pragma unroll
          for (int k = 0; k < NCH; ++k)
            if ((om >> k) & 1u) *reinterpret_cast<uint4*>(oh + k * osW) = cc[k];
        }
        ++z;
        if (++slot == 3) slot = 0;
      }
      aphase ^= 1;
    }
  }
}

template <bool kPair>
__global__ void __launch_bounds__(kThreads, 1)
conv_scatter_concat_ros_kernel(const __grid_constant__ CUtensorMap map_ref, const __grid_constant__ CUtensorMap map_tl,
                               const __grid_constant__ CUtensorMap map_tr, const __grid_constant__ CUtensorMap map_w,
                               const __grid_constant__ CUtensorMap map_wr, const __grid_constant__ RoArgs ra) {
  const CcArgs& ca = ra.c;
  const ScArgs& a = ca.a;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_planes = smem + 2 * a.slot_bytes;
  uint8_t* smem_w = smem_planes + a.ring * a.slot_bytes;
  __shared__ CcCtrl ctrl;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&map_ref);  ptx::prefetch_tensormap(&map_tl);  ptx::prefetch_tensormap(&map_tr);
    ptx::prefetch_tensormap(&map_w);    ptx::prefetch_tensormap(&map_wr);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < kMaxRing; ++s) { ptx::mbar_init(&ctrl.c.plane_full[s], 1); ptx::mbar_init(&ctrl.c.plane_empty[s], 1); }
    for (int s = 0; s < kMaxW; ++s) { ptx::mbar_init(&ctrl.c.w_full[s], 1); ptx::mbar_init(&ctrl.c.w_empty[s], 1); }
    for (int b = 0; b < 2; ++b) {
      ptx::mbar_init(&ctrl.c.acc_full[b], 1);  ptx::mbar_init(&ctrl.c.acc_empty[b], kPair ? 8 : 4);
      ptx::mbar_init(&ctrl.ref_full[b], 1);    ptx::mbar_init(&ctrl.ref_empty[b], 1);
    }
    ptx::fence_barrier_init();
  }
  if (warp == 2) { if (kPair) ptx::tmem_alloc_2sm(&ctrl.c.tmem_base, kTmemCols); else ptx::tmem_alloc(&ctrl.c.tmem_base, kTmemCols); }
  ptx::tc_fence_before();
  __syncthreads();
  if (kPair) ptx::cluster_sync_all();
  ptx::tc_fence_after();
  const uint32_t tmem_base = ctrl.c.tmem_base;

  if (warp == 0) {
    ros_produce<kPair>(ra, ctrl, ptx::smem_u32(smem), ptx::smem_u32(smem_planes), ptx::smem_u32(smem_w), &map_ref, &map_tl, &map_tr,
                       &map_w, &map_wr);
  } else if (warp == 1 && (!kPair || ptx::cluster_ctarank() == 0)) {
    const int rb = a.row_bytes;                            // 128
    const RosIssue zi = {{{tmem_base, ptx::smem_u32(smem_planes), ptx::smem_u32(smem_w),
                           ptx::smem_u32(&ctrl.c.plane_full[0]), ptx::smem_u32(&ctrl.c.plane_empty[0]), ptx::smem_u32(&ctrl.c.w_full[0]),
                           ptx::smem_u32(&ctrl.c.w_empty[0]), ptx::smem_u32(&ctrl.c.acc_full[0]), ptx::smem_u32(&ctrl.c.acc_empty[0]),
                           desc_hi(kHX * rb, rb), desc_hi(8 * rb, rb), a.slot_bytes, a.w_bytes, a.w_stages, a.ring,
                           (uint32_t)(rb >> 4), 0u, (uint32_t)((kTileY * kHX * rb) >> 4), 0u, a.idesc, ca.D, cta_cols(a)},
                          ptx::smem_u32(smem), ptx::smem_u32(&ctrl.ref_full[0]), ptx::smem_u32(&ctrl.ref_empty[0])},
                         desc_hi(8 * 64, 64), (uint32_t)(a.w_tx >> 5), ra.idesc_r, a.cp};
    ros_issue<kPair>(zi);
  } else if (warp >= 4) {
    ros_epilogue(a, ctrl.c, tmem_base, warp, lane);
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (kPair) ptx::cluster_sync_all();
  if (warp == 2) {
    ptx::tc_fence_after();
    if (kPair) ptx::tmem_dealloc_2sm(tmem_base, kTmemCols); else ptx::tmem_dealloc(tmem_base, kTmemCols);
  }
}

static int encode5(CUtensorMap* m, const void* base, bool f32, const cuuint64_t dims[5], const cuuint64_t strides[4],
                   const cuuint32_t box[5], CUtensorMapSwizzle sw) {
  const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  return encode_tiled_cached(m, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, base, dims, strides, box,
                             estr, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, "concat view");
}

}  // namespace scatter
}  // namespace s3d

// Split (BF16X2) operands: reference-once form only.  feat: [2B, h, pitch, hi(C) | lo(C)], out: [2B, D, h, w, hi(64) | lo(64)].
static int launch_concat_ros(const S3dConvParams& p, const void* feat, int feat_pitch, int feat_pad, const void* w_refonce,
                             const float* bias, void* out, void* stream) {
  using namespace s3d;
  using namespace s3d::scatter;
  S3D_CHECK_ARG(w_refonce != nullptr, "conv_concat_volume: split (BF16X2) operands need the reference-once form (s3d_conv_concat_volume_ro)");
  S3D_CHECK_ARG(p.w_nstack != nullptr && bias != nullptr, "conv_concat_volume_ro: the layer needs host-packed rotations (w_nstack) and a bias");
  S3D_CHECK_ARG(plane_scatter_layer(p), "conv_concat_volume_ro: not a stride-1 3x3x3 layer in canonical tap order");
  S3D_CHECK_ARG(p.N % 2 == 0 && p.Cin == 64 && p.Cout == 64 && p.cout_store == 64 && p.out_dtype == S3D_DTYPE_BF16X2 && p.act == S3D_ACT_RELU,
                "conv_concat_volume_ro (split): needs C = 32 feature channels, Cout = 64, a split output and ReLU");
  const int C = 32, B = p.N / 2, D = p.iD, h = p.iH, w = p.iW, rb = 128;
  S3D_CHECK_ARG(feat_pad >= D - 1 && feat_pitch >= w + 2 * feat_pad, "conv_concat_volume_ro: feature rows need >= D-1 zero pixels on both sides");
  S3D_CHECK_ARG(((reinterpret_cast<uintptr_t>(feat) | reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(w_refonce)) & 15) == 0,
                "conv_concat_volume_ro: pointer alignment");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  RoArgs ra;
  memset(&ra, 0, sizeof(ra));
  CcArgs& ca = ra.c;
  ScArgs& a = ca.a;
  a.p = p;  a.bias = bias;  a.residual = nullptr;  a.out = out;
  a.split = 1;  a.os_lo = p.os_lo ? p.os_lo : (int64_t)p.Cout;
  ca.n_half = B;  ca.D = D;
  const int64_t total = plane_geometry(a, rb, C, 1);
  a.cp = 64;  a.tps = 1;
  S3D_CHECK_ARG(total >= 2 && total < (1ll << 31), "conv_concat_volume_ro: column count out of range");
  a.pair = 1;
  const int grid = deal_columns(a, total, num_sms());
  const int w_rows = 3 * a.cp / 2;
  a.w_tx = 2 * w_rows * 64;                                     // [w_hi | w_lo] tiles of 64-byte rows
  a.w_bytes = align1024(a.w_tx);
  ra.w_tx_r = (a.cp / 2) * 128;
  ra.idesc_r = ptx::make_instr_desc(1, 256, a.cp);
  const int budget = 227 * 1024 - 1024 - 640;
  a.ring = 2;
  a.w_stages = (budget - (2 + a.ring) * a.slot_bytes) / a.w_bytes;
  if (a.w_stages > kMaxW) a.w_stages = kMaxW;
  S3D_CHECK_ARG(a.w_stages >= 3, "conv_concat_volume_ro (split): not enough shared memory");
  a.idesc = ptx::make_instr_desc(1, 256, 3 * a.cp);
  a.res_direct = 1;
  a.fast_store = coalesced_store_ok(p, bias, out, nullptr, 2) && (a.os_lo * 2) % 16 == 0;
  S3D_CHECK_ARG(a.fast_store, "conv_concat_volume_ro (split): output strides must be multiples of 16 bytes");
  const uint8_t* fb = static_cast<const uint8_t*>(feat);
  const cuuint64_t px = 2 * C * 2, row = (cuuint64_t)feat_pitch * px, img = (cuuint64_t)h * row;
  CUtensorMap map_ref, map_tl, map_tr, map_w, map_wr;
  {
    const cuuint64_t dims[5] = {(cuuint64_t)(2 * C), (cuuint64_t)w, (cuuint64_t)h, 1, (cuuint64_t)p.N};
    const cuuint64_t strides[4] = {px, row, img, img};
    const cuuint32_t box[5] = {(cuuint32_t)(2 * C), kHX, kHY, 1, 1};
    int rc = encode5(&map_ref, fb + (size_t)feat_pad * px, false, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc != S3D_OK) return rc;
  }
  {
    const cuuint64_t dims[5] = {(cuuint64_t)(2 * C), (cuuint64_t)w, (cuuint64_t)D, (cuuint64_t)h, (cuuint64_t)B};
    const cuuint64_t strides[4] = {px, px, row, img};
    const cuuint32_t box[5] = {(cuuint32_t)(2 * C), kHX, 1, kHY, 1};
    int rc = encode5(&map_tl, fb + (size_t)B * img + (size_t)(feat_pad - (D - 1)) * px, false, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc != S3D_OK) return rc;
    rc = encode5(&map_tr, fb + (size_t)feat_pad * px, false, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc != S3D_OK) return rc;
  }
  // stacked rotations, physical rows [hi(2C) | lo(2C)]: boxes of C channels (64 bytes) x this CTA's rows
  int rc = encode_weight_map(&map_w, p.w_nstack, 2, false, 4 * C, 3 * a.cp, 36, C, w_rows, CU_TENSOR_MAP_SWIZZLE_64B, 1);
  if (rc != S3D_OK) return rc;
  rc = encode_weight_map(&map_wr, w_refonce, 2, false, 2 * C, a.cp, 27, 2 * C, a.cp / 2, CU_TENSOR_MAP_SWIZZLE_128B, 1);
  if (rc != S3D_OK) return rc;
  const int smem_bytes = (2 + a.ring) * a.slot_bytes + a.w_stages * a.w_bytes + 1024;
  return launch_plane_scatter(conv_scatter_concat_ros_kernel<true>, grid, smem_bytes, a.pair, st, map_ref, map_tl, map_tr, map_w,
                              map_wr, ra);
}

// w_refonce != nullptr: reference-once mode (bf16, CTA pairs, Cout = 64, ReLU, coalesced stores only).
static int launch_concat(const S3dConvParams* p_in, const void* feat, int feat_pitch, int feat_pad, const void* w_refonce,
                         const float* bias, void* out, void* stream) {
  using namespace s3d;
  using namespace s3d::scatter;
  if (!p_in || !feat || !out) { set_error("conv_concat_volume: null argument"); return S3D_ERR_INVALID; }
  const S3dConvParams& p = *p_in;
  if (p.in_dtype == S3D_DTYPE_BF16X2) return launch_concat_ros(p, feat, feat_pitch, feat_pad, w_refonce, bias, out, stream);
  const bool ro = w_refonce != nullptr;
  const bool tf32 = p.in_dtype == S3D_DTYPE_F32;
  const int esz = tf32 ? 4 : 2;
  S3D_CHECK_ARG(p.w_nstack != nullptr, "conv_concat_volume: the layer needs host-packed rotations (w_nstack)");
  S3D_CHECK_ARG(plane_scatter_layer(p), "conv_concat_volume: not a stride-1 3x3x3 layer in canonical tap order");
  S3D_CHECK_ARG(p.N % 2 == 0 && p.Cin % 2 == 0, "conv_concat_volume: N = 2B volumes, Cin = 2C channels");
  const int C = p.Cin / 2, B = p.N / 2, D = p.iD, h = p.iH, w = p.iW;
  const int rb = C * esz;
  S3D_CHECK_ARG(rb == 32 || rb == 64 || rb == 128, "conv_concat_volume: C * element size must be 32, 64 or 128 bytes");
  S3D_CHECK_ARG(!(tf32 && rb == 32), "conv_concat_volume: fp32 features need C >= 16");
  S3D_CHECK_ARG(p.Cout <= 64 && p.Cout % 16 == 0, "conv_concat_volume: Cout");
  S3D_CHECK_ARG(feat_pad >= D - 1 && feat_pitch >= w + 2 * feat_pad, "conv_concat_volume: feature rows need >= D-1 zero pixels on both sides");
  S3D_CHECK_ARG((reinterpret_cast<uintptr_t>(feat) & 15) == 0, "conv_concat_volume: feat alignment");
  S3D_CHECK_ARG(p.cout_store >= 1 && p.cout_store <= p.Cout, "conv_concat_volume: cout_store");
  cudaStream_t st = static_cast<cudaStream_t>(stream);

  CcArgs ca;
  memset(&ca, 0, sizeof(ca));
  ScArgs& a = ca.a;
  a.p = p;  a.bias = bias;  a.residual = nullptr;  a.out = out;
  ca.n_half = B;  ca.D = D;
  const int64_t total = plane_geometry(a, rb, C, 2);          // (no z-split here: small batches take the unfused path)
  a.slot_bytes = a.chunk_stride;                               // a slot holds ONE half (reference buffers / target ring)
  a.cp = p.Cout;  a.tps = 1;
  S3D_CHECK_ARG(total > 0 && total < (1ll << 31), "conv_concat_volume: column count out of range");
  int grid = num_sms();
  a.pair = ((3 * a.cp / 2) % 8 == 0 && total >= 2 && grid >= 2 && !knobs().scatter_no_pair) ? 1 : 0;
  grid = deal_columns(a, total, grid);
  const int w_rows = a.pair ? 3 * a.cp / 2 : 3 * a.cp;
  // one stage = one tap, both K chunks; reference-once: kTps taps of the target chunk
  a.w_tx = ro ? kTps * w_rows * rb : 2 * w_rows * rb;
  a.w_bytes = align1024(a.w_tx);
  const int budget = 227 * 1024 - 1024 - 640;
  int ring = 4;
  while (ring > 2 && (2 + ring) * a.slot_bytes + 4 * a.w_bytes > budget) --ring;
  a.ring = ring;
  a.w_stages = (budget - (2 + a.ring) * a.slot_bytes) / a.w_bytes;
  if (a.w_stages > kMaxW) a.w_stages = kMaxW;
  S3D_CHECK_ARG(a.w_stages >= 2 && (a.pair || rb < 128), "conv_concat_volume: not enough shared memory (128-byte halves need CTA pairs)");
  a.idesc = ptx::make_instr_desc(tf32 ? 2 : 1, a.pair ? 256 : 128, 3 * a.cp);
  a.res_direct = 1;
  a.fast_store = coalesced_store_ok(p, bias, out, nullptr, p.out_dtype == S3D_DTYPE_BF16 ? 2 : 4);

  const CUtensorMapSwizzle sw = rb == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : rb == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B;
  const uint8_t* fb = static_cast<const uint8_t*>(feat);
  const cuuint64_t px = (cuuint64_t)C * esz, row = (cuuint64_t)feat_pitch * px, img = (cuuint64_t)h * row;
  CUtensorMap map_ref, map_tl, map_tr, map_w;
  {
    // reference half: plain view of the real pixels, dims (C, X, Y, 1, 2B)
    const cuuint64_t dims[5] = {(cuuint64_t)C, (cuuint64_t)w, (cuuint64_t)h, 1, (cuuint64_t)p.N};
    const cuuint64_t strides[4] = {px, row, img, img};
    const cuuint32_t box[5] = {(cuuint32_t)C, kHX, kHY, 1, 1};
    int rc = encode5(&map_ref, fb + (size_t)feat_pad * px, tf32, dims, strides, box, sw);
    if (rc != S3D_OK) return rc;
  }
  {
    // target halves: skewed views, dims (C, X, D, Y, B) with stride(X) == stride(D) == one pixel
    const cuuint64_t dims[5] = {(cuuint64_t)C, (cuuint64_t)w, (cuuint64_t)D, (cuuint64_t)h, (cuuint64_t)B};
    const cuuint64_t strides[4] = {px, px, row, img};
    const cuuint32_t box[5] = {(cuuint32_t)C, kHX, 1, kHY, 1};
    // left-referenced volumes read the RIGHT images (feat[B..2B)) at x - d: coordinate (x, D-1-d) from a base D-1 pixels left
    int rc = encode5(&map_tl, fb + (size_t)B * img + (size_t)(feat_pad - (D - 1)) * px, tf32, dims, strides, box, sw);
    if (rc != S3D_OK) return rc;
    // right-referenced volumes read the LEFT images (feat[0..B)) at x + d: coordinate (x, d)
    rc = encode5(&map_tr, fb + (size_t)feat_pad * px, tf32, dims, strides, box, sw);
    if (rc != S3D_OK) return rc;
  }
  int rc = encode_weight_map(&map_w, p.w_nstack, esz, tf32, p.Cin, 3 * a.cp, 36, C, w_rows, sw, ro ? kTps : 1);
  if (rc != S3D_OK) return rc;

  const int smem_bytes = (2 + a.ring) * a.slot_bytes + a.w_stages * a.w_bytes + 1024;
  if (ro) {
    const bool simple = a.pair && !tf32 && p.out_dtype == S3D_DTYPE_BF16 && a.fast_store && a.cp == 64 && p.act == S3D_ACT_RELU;
    S3D_CHECK_ARG(simple && rb <= 64 && a.w_stages >= 4,
                  "conv_concat_volume_ro: needs bf16 in/out, C <= 32, Cout = 64, ReLU, dense 16-byte aligned output, >= 2 columns");
    S3D_CHECK_ARG((reinterpret_cast<uintptr_t>(w_refonce) & 15) == 0, "conv_concat_volume_ro: w_refonce alignment");
    RoArgs ra;
    memset(&ra, 0, sizeof(ra));
    ra.c = ca;
    ra.w_tx_r = kTps * (a.cp / 2) * rb;
    ra.idesc_r = ptx::make_instr_desc(1, 256, a.cp);
    CUtensorMap map_wr;
    rc = encode_weight_map(&map_wr, w_refonce, esz, false, C, a.cp, 27, C, a.cp / 2, sw, kTps);
    if (rc != S3D_OK) return rc;
    typedef void (*KernR)(CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, RoArgs);
    KernR kern = rb == 64 ? conv_scatter_concat_ro_kernel<true, 2> : conv_scatter_concat_ro_kernel<true, 1>;
    return launch_plane_scatter(kern, grid, smem_bytes, a.pair, st, map_ref, map_tl, map_tr, map_w, map_wr, ra);
  }
  typedef void (*Kern)(CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CcArgs);
  const bool lean = a.pair && !tf32 && p.out_dtype == S3D_DTYPE_BF16 && a.fast_store && a.cp == 64 && p.act == S3D_ACT_RELU && rb == 64;
  Kern kern = nullptr;
  if (lean) kern = conv_scatter_concat_kernel<false, true, 2, true>;
  else if (a.pair) {
    kern = tf32 ? (rb == 128 ? conv_scatter_concat_kernel<true, true, 4, false> : conv_scatter_concat_kernel<true, true, 2, false>)
                : (rb == 128 ? conv_scatter_concat_kernel<false, true, 4, false> : rb == 64 ? conv_scatter_concat_kernel<false, true, 2, false>
                                                                                            : conv_scatter_concat_kernel<false, true, 1, false>);
  } else {
    // a single CTA cannot hold two weight stages of 128-byte halves (checked above through w_stages), so no kPer = 4 here
    kern = tf32 ? conv_scatter_concat_kernel<true, false, 2, false>
                : (rb == 64 ? conv_scatter_concat_kernel<false, false, 2, false> : conv_scatter_concat_kernel<false, false, 1, false>);
  }
  return launch_plane_scatter(kern, grid, smem_bytes, a.pair, st, map_ref, map_tl, map_tr, map_w, ca);
}

extern "C" int s3d_conv_concat_volume(const S3dConvParams* p, const void* feat, int feat_pitch, int feat_pad, const float* bias,
                                      void* out, void* stream) {
  return launch_concat(p, feat, feat_pitch, feat_pad, nullptr, bias, out, stream);
}

extern "C" int s3d_conv_concat_volume_ro(const S3dConvParams* p, const void* feat, int feat_pitch, int feat_pad, const void* w_refonce,
                                         const float* bias, void* out, void* stream) {
  if (!w_refonce) { s3d::set_error("conv_concat_volume_ro: null w_refonce"); return S3D_ERR_INVALID; }
  return launch_concat(p, feat, feat_pitch, feat_pad, w_refonce, bias, out, stream);
}
