// Plane-scatter implicit GEMM for stride-1 3x3x3 convolutions with Cout <= 64 (the five 64-wide cost-aggregation
// layers = two thirds of the forward pass, and the fusion scorer's narrow 3-D layers).
//
// conv_halo.cu's z-stacked tile (two output planes x 64 channels on the M side) spends a quarter of its MMA rows on
// structural zeros: of the four input planes a plane pair reads, the first and the last only feed one of the two
// output planes.  Here the roles are turned round.  An INPUT plane p feeds exactly three output planes
// (z = p+1, p, p-1 through kz = 0, 1, 2), so the pixels go on the M side (128 per tile) and the three kz slices of
// the weights are stacked on the N side:
//
//     D[pixel, (slot, co)] += sum_ci X_p[pixel + (ky,kx), ci] * Wrot[(slot, co), ci]        N = 3 * Cout (192)
//
// Every MMA row and column is a useful product; an N = 192 MMA issues at the full tensor rate (96 cycles, measured
// with scripts/mma_rate.cu, operands distinct per instruction).  The three 64-column accumulator "slots" of a tile
// form a ring over output planes: out plane z lives in slot z % 3, receives input planes z-1, z, z+1 and is then
// complete.  Which kz lands in which slot depends on p % 3, so the host packs three rotations of the stacked
// weights (plus a fourth for p = 0 whose non-existent z = -1 block is zero, so that the first MMA of a column can
// overwrite all three slots): S3dConvParams.w_nstack, [4][9][3*Cout][Cin].
//
//   CTA work item   a column: one volume n, a 32(y) x 8(x) patch = two tiles of 16 x 8 = 128 pixels, marching over z.
//   plane slot      input plane p of the patch with halo (34 x 10 rows, one 5-D TMA box, zero fill outside); each
//                   plane is fetched once per column and is the A operand of 9 taps x 2 tiles (descriptor start
//                   moved by (ky*10 + kx) rows, 8-row groups one halo line apart -- as in conv_halo.cu).
//   weights         one stage = TPS of the 9 in-plane taps of the current rotation (24 KB for 64 -> 64), used by
//                   BOTH tiles, so the L2 -> SM weight stream is the same 32 B/clk/SM as the z-stacked kernel's.
//   accumulators    TMEM columns [256 t + 64 s, +64) for tile t, slot s.
//   epilogue        thread = pixel (TMEM lane).  When input plane p is done, out plane p-1 is complete: its slot is
//                   read into registers, ZEROED (tcgen05.st; the slot's next user accumulates from its first MMA)
//                   and handed back at once; bias / residual / activation / store then run from registers while
//                   the tensor core is already on the next plane.  Tile 1 trails tile 0 by one weight stage so
//                   that each tile's hand-back is hidden behind the other tile's MMAs.
//
// Warp roles: 0 TMA producer, 1 MMA issuer, 2 TMEM allocator, 4-7 epilogue of tile 0, 8-11 epilogue of tile 1.
#pragma once
#include <cuda.h>
#include <stdlib.h>
#include <string.h>
#include "common.cuh"
#include "ptx.cuh"
#include "epilogue.cuh"

// Device code of the plane-scatter kernel.  Included by conv_scatter.cu (host launcher + the all-in-one kernels) and by
// conv_scatter_spec.cu (the lean per-layer-shape kernels), which are separate translation units only so that they
// compile in parallel.
namespace s3d {
namespace scatter {

constexpr int kThreads = 384;
constexpr int kTX = 8, kHX = kTX + 2;
constexpr int kTY = 32, kHY = kTY + 2;
constexpr int kTileY = 16;                     // rows of one M = 128 tile
constexpr int kPlaneRows = kHX * kHY;          // 340
constexpr int kMaxRing = 6;
constexpr int kMaxW = 12;
constexpr int kTmemCols = 512;
constexpr int kTileCols = 256;                 // TMEM column pitch between the two tiles

struct ScArgs {
  S3dConvParams p;
  const float* bias;
  const void* residual;
  void* out;
  int row_bytes;      // bytes of one K chunk of a pixel row: 32 / 64 / 128
  int kc;             // channels per K chunk
  int nchunks;        // K chunks per row: 1, or 2 for 256-byte rows (64 fp32 channels: the tf32 aggregation layers)
  int chunk_stride;   // bytes between the chunks of a plane slot
  int slot_bytes;     // one input plane with halo, rounded to 1024
  int ring;           // plane slots
  int cp;             // accumulator columns per output plane (= Cout, multiple of 16)
  int tps;            // in-plane taps per weight stage: 1, 3 or 9
  int w_stages, w_bytes, w_tx;
  int cols_x, cols_y, total_cols;
  int pair;           // 1: CTA pairs (cta_group::2, M = 256): each CTA keeps its own pixels, half of the weight rows
  int ncols_max;      // pair mode: columns every CTA walks (phantom columns beyond total_cols compute on zeros)
  uint32_t idesc;
  int fast_store;     // epilogue may use the transposed (coalesced) store path
  int res_direct;
  // Split (BF16X2, 'bf16x3' precision) operands: rows are [hi(Cin) | lo(Cin)] bf16, weights [hi | lo] likewise, and every tap
  // issues (x_hi, w_hi), (x_lo, w_hi), (x_hi, w_lo) into the same accumulator.  64 / 128-byte physical rows are ONE K chunk
  // (the lo half starts row_bytes / 2 into the swizzle atom); 256-byte rows are two chunks as in the fp32 case, with one
  // weight stage per (tap, hi | lo weights).  The output is split as well: lo parts os_lo elements after the hi parts.
  int split;
  int64_t os_lo;
  // z-split (small batches): with fewer columns than SMs a column of D planes is a serial chain on a fraction of the chip,
  // so a column is cut into nz chunks of zc output planes.  A chunk marches over the zc + 2 input planes z0-1 .. z0+zc
  // exactly like a whole column (planes outside the volume are TMA zero fill) and only STORES its own zc output planes:
  // the first and last local output plane of a chunk are incomplete and dropped.  nz <= 1: no split (dl = D).
  int nz, zc, dl;     // chunks per column, output planes per chunk, local planes marched per work item
};

struct ScCtrl {
  uint64_t plane_full[kMaxRing], plane_empty[kMaxRing];
  uint64_t w_full[kMaxW], w_empty[kMaxW];
  uint64_t acc_full[2], acc_empty[2];
  uint64_t res_full, res_empty;                  // residual-by-MMA kernels (conv_scatter_rm.cu): one staged residual plane
  uint32_t tmem_base;
};

// Residual through the tensor core (conv_scatter_rm.cu): the residual plane of the 32x8 patch (256 pixels x 128 bytes, no halo)
// is staged by TMA and added to the accumulators as one more "tap" whose weight matrix is the identity.
struct ScRes {
  const CUtensorMap* map_r;
  uint32_t res_u32;        // staged residual plane: [tile][128 pixels][128 B], 128B swizzle
  uint32_t ident_u32;      // identity rows of this CTA: [Cout / 2 (pair)][128 B], 128B swizzle
  uint32_t bar_rf, bar_re;
  uint32_t idesc_r;        // N = Cout
  int cp;
};
constexpr int kResBytes = 256 * 128;

struct Col { int n, y0, x0, zb; };             // zb: global z of local plane 0 (0, or z0 - 1 of a z-chunk)

__device__ __forceinline__ Col decode_col(const ScArgs& a, int c) {
  Col r;
  r.zb = 0;
  if (a.nz > 1) { r.zb = (c % a.nz) * a.zc - 1;  c /= a.nz; }
  r.x0 = (c % a.cols_x) * kTX;  c /= a.cols_x;
  r.y0 = (c % a.cols_y) * kTY;  c /= a.cols_y;
  r.n = c;
  return r;
}

// Columns this CTA walks.  The two CTAs of a pair run the same MMAs, so in pair mode every CTA walks ncols_max
// columns (or its pair's list in the schedule table, include/s3d.h dz_sched); a column index >= total_cols decodes to
// n >= N (TMA zero fill, nothing stored).
__device__ __forceinline__ int cta_cols(const ScArgs& a) {
  if (a.p.dz_sched) return __ldg(a.p.dz_sched + (blockIdx.x >> 1) + 1) - __ldg(a.p.dz_sched + (blockIdx.x >> 1));
  return a.pair ? a.ncols_max : (a.total_cols - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
}

// Constant-region skip (include/s3d.h, dz_nref).  Output planes [zs, zs + J] of a work item are equal: once input plane
// zs + 1 is done (out plane zs drained), the slots of out planes zs + 1 and zs + 2 hold exactly the partial sums that out
// planes zs + 1 + J and zs + 2 + J need (their input planes are the same), so the march continues at input plane
// zs + 2 + J and the epilogue stores plane zs J more times.  J % 3 == 0 keeps every slot (z % 3) and weight rotation
// (p % 3) where it was.  The two CTAs of a pair issue the same MMAs: both take the intersection of their columns' runs.
struct Item { Col c; int zs, J; };

__device__ __forceinline__ int dz_first(const ScArgs& a, const Col& c) {      // first plane of the column's repeating run
  if (c.n >= a.p.N) return 0;                                                 // empty column: no constraint
  const int xr = c.n < a.p.dz_nref ? min(c.x0 + kTX - 1, a.p.oW - 1) : a.p.oW - 1 - c.x0;
  return xr + a.p.dz_c + 2;
}

__device__ __forceinline__ Item cta_item(const ScArgs& a, int ci) {
  int mine, other;
  if (a.p.dz_sched) {
    const int r = blockIdx.x & 1;
    const int32_t* e = a.p.dz_sched + a.p.dz_pairs + 1 + 2 * (__ldg(a.p.dz_sched + (blockIdx.x >> 1)) + ci);
    mine = __ldg(e + r);  other = __ldg(e + (r ^ 1));
  } else {
    mine = blockIdx.x + ci * gridDim.x;  other = a.pair ? (mine ^ 1) : mine;   // pair mode: grid even, partner = blockIdx ^ 1
  }
  Item it;
  it.c = decode_col(a, mine);
  it.zs = 0;  it.J = 0;
  if (a.p.dz_nref > 0) {
    const int zs = max(dz_first(a, it.c), dz_first(a, decode_col(a, other))), ze = a.p.oD - 2 - a.p.dz_e;
    it.zs = zs;
    it.J = ze - zs >= 3 ? (ze - zs) / 3 * 3 : 0;
  }
  return it;
}

// The input planes of a work item, in march order: 0 .. D-1 with zs + 2 .. zs + 1 + J left out.
__device__ __forceinline__ int next_plane(const Item& it, int p) { return p == it.zs + 1 ? p + 1 + it.J : p + 1; }

__device__ __forceinline__ uint64_t desc_hi(uint32_t sbo, int row_bytes) {
  const uint64_t layout = row_bytes == 128 ? 2ull : (row_bytes == 64 ? 4ull : 6ull);
  return (static_cast<uint64_t>(sbo >> 4) << 32) | (1ull << 46) | (layout << 61);
}
__device__ __forceinline__ uint32_t desc_lo(uint32_t addr) { return ((addr & 0x3FFFF) >> 4) | (1u << 16); }

// ---- TMA producer: warp-uniform, incremental ring counters, TMA issue under small elect_one regions -----------------
template <int TPS, bool kPair, int NK = 1, bool kRM = false>       // NK = 2: 256-byte rows as two 128-byte K chunks, one weight stage per (tap, chunk)
__device__ __forceinline__ void sc_produce(const ScArgs& a, ScCtrl& ctrl, uint32_t planes_u32, uint32_t w_u32,
                                           const CUtensorMap* map_x, const CUtensorMap* map_w, const ScRes* rs = nullptr) {
  constexpr int G = 9 * NK / TPS;
  const uint32_t bar_pf = ptx::smem_u32(&ctrl.plane_full[0]), bar_pe = ptx::smem_u32(&ctrl.plane_empty[0]);
  const uint32_t bar_wf = ptx::smem_u32(&ctrl.w_full[0]), bar_we = ptx::smem_u32(&ctrl.w_empty[0]);
  const int D = a.dl, ring = a.ring, w_stages = a.w_stages, ncols = cta_cols(a);
  const int slot_bytes = a.slot_bytes, w_bytes = a.w_bytes, w_tx = a.w_tx;
  // pair mode: this CTA stages its own planes and ITS half of the weight rows; every load signals the leader's `full`
  // barrier, on which the leader's producer expects the bytes of both CTAs
  const int crank = kPair ? (int)ptx::cluster_ctarank() : 0;
  const bool leader = crank == 0;
  const int w_row0 = kPair ? crank * (3 * a.cp / 2) : 0;
  const int plane_tx = NK * kPlaneRows * a.row_bytes;
  const int kc = a.kc, chunk_stride = a.chunk_stride;
  int ws = 0;  uint32_t wphase = 0;
  int pslot = 0;  uint32_t pphase = 0;
  int pci = 0, pj = 0, issued = 0;
  Item pit{};
  if (ncols > 0) pit = cta_item(a, 0);
  const Col& pc = pit.c;
  auto issue_plane = [&](bool blocking) -> bool {
    if (pci >= ncols) return false;
    const uint32_t be = bar_pe + 8 * pslot, bf = bar_pf + 8 * pslot;
    if (blocking) ptx::mbar_wait_u32(be, pphase ^ 1);
    else if (!ptx::mbar_test_wait_u32(be, pphase ^ 1)) return false;
    if (ptx::elect_one()) {
      if (kPair) {
        if (leader) ptx::mbar_arrive_expect_tx_u32(bf, 2 * plane_tx);
#pragma unroll
        for (int ch = 0; ch < NK; ++ch)
          ptx::tma_load_5d_2sm_u32(planes_u32 + pslot * slot_bytes + ch * chunk_stride, map_x, bf, ch * kc, pc.x0 - 1, pc.y0 - 1, pc.zb + pj, pc.n);
      } else {
        ptx::mbar_arrive_expect_tx_u32(bf, plane_tx);
#pragma unroll
        for (int ch = 0; ch < NK; ++ch)
          ptx::tma_load_5d_u32(planes_u32 + pslot * slot_bytes + ch * chunk_stride, map_x, bf, ch * kc, pc.x0 - 1, pc.y0 - 1, pc.zb + pj, pc.n);
      }
    }
    __syncwarp();
    ++issued;
    if (++pslot == ring) { pslot = 0; pphase ^= 1; }
    pj = next_plane(pit, pj);
    if (pj >= D) {
      pj = 0;  ++pci;
      if (pci < ncols) pit = cta_item(a, pci);
    }
    return true;
  };
  int gp = 0;                                    // global index of the current plane
  [[maybe_unused]] uint32_t rphase = 0;
  // Residual of output plane p (kRM): one staged plane, added by the issuer in the MIDDLE of plane p's taps.  The load for
  // plane p + 1 goes out after plane p's weight stages: the weight ring (< 9 stages) keeps this warp less than a plane ahead
  // of the issuer, so plane p's residual MMAs have retired (or are about to) and the wait is short, and the data arrives
  // most of a plane before it is needed.
  [[maybe_unused]] auto load_res = [&](const Col& rc, int p) {
    ptx::mbar_wait_u32(rs->bar_re, rphase ^ 1);
    if (ptx::elect_one()) {
      if (kPair) {
        if (leader) ptx::mbar_arrive_expect_tx_u32(rs->bar_rf, 2 * kResBytes);
        ptx::tma_load_5d_2sm_u32(rs->res_u32, rs->map_r, rs->bar_rf, 0, rc.x0, rc.y0, rc.zb + p, rc.n);
      } else {
        ptx::mbar_arrive_expect_tx_u32(rs->bar_rf, kResBytes);
        ptx::tma_load_5d_u32(rs->res_u32, rs->map_r, rs->bar_rf, 0, rc.x0, rc.y0, rc.zb + p, rc.n);
      }
    }
    __syncwarp();
    rphase ^= 1;
  };
  for (int ci = 0; ci < ncols; ++ci) {
    int rot = 3;                                 // weight rotation: 3 for p = 0, then p % 3 (a skip keeps p % 3)
    const Item it = cta_item(a, ci);
    [[maybe_unused]] const Col& rc = it.c;
    if constexpr (kRM) load_res(rc, 0);
    for (int p = 0; p < D; p = next_plane(it, p), ++gp) {
      while (issued <= gp) issue_plane(true);
      const int ahead = gp + ring;               // planes that may be in flight while plane gp is being read
#pragma unroll
      for (int g = 0; g < G; ++g) {
        if (issued < ahead) issue_plane(false);
        const uint32_t be = bar_we + 8 * ws, bf = bar_wf + 8 * ws;
        ptx::mbar_wait_u32(be, wphase ^ 1);
        if (ptx::elect_one()) {
          // NK = 2: group g = (tap g / 2, chunk g % 2)
          const int tap = rot * 9 + (NK == 2 ? g / 2 : g * TPS), c0 = NK == 2 ? (g & 1) * kc : 0;
          if (kPair) {
            if (leader) ptx::mbar_arrive_expect_tx_u32(bf, 2 * w_tx);
            ptx::tma_load_3d_2sm_u32(w_u32 + ws * w_bytes, map_w, bf, c0, w_row0, tap);
          } else {
            ptx::mbar_arrive_expect_tx_u32(bf, w_tx);
            ptx::tma_load_3d_u32(w_u32 + ws * w_bytes, map_w, bf, c0, 0, tap);
          }
        }
        __syncwarp();
        if (++ws == w_stages) { ws = 0; wphase ^= 1; }
      }
      if constexpr (kRM) { const int pn = next_plane(it, p); if (pn < D) load_res(rc, pn); }       // one plane ahead (see load_res)
      rot = (p == 0) ? 1 : (rot == 2 ? 0 : rot + 1);
    }
  }
  if (a.p.dz_planes) {
    if (ptx::elect_one()) atomicAdd(reinterpret_cast<unsigned long long*>(a.p.dz_planes), (unsigned long long)issued);
    __syncwarp();
  }
}

// ---- MMA issuer -------------------------------------------------------------------------------------------------
// Per input plane the weight groups g = 0..G-1 are issued as  T0g0, [T0g1, T1g0], [T0g2, T1g1], ..., T1g(G-1):
// tile 1 trails tile 0 by one group, so a tile's accumulator hand-back (epilogue reads + zeroes the finished slot)
// overlaps the other tile's MMAs.  Everything is warp-uniform; only MMAs and commits sit under elect_one, in small
// straight-line regions with compile-time operand offsets (the cheap tcgen05.mma encoding, see conv_halo.cu).
struct ScIssue {
  uint32_t tmem_base, planes_u32, w_u32;
  uint32_t bar_pf, bar_pe, bar_wf, bar_we, bar_af, bar_ae;
  uint64_t x_hi, w_hi;
  int slot_bytes, w_bytes, w_stages, ring;
  uint32_t rb16, tap_step, tile_off, chunk_step; // 16-byte units
  uint32_t idesc;
  int D, ncols;
  const ScArgs* args = nullptr;                  // work items (cta_item); only sc_issue reads it
};

template <bool kPair>
__device__ __forceinline__ void sc_commit(uint32_t bar) {
  if (kPair) ptx::tc_commit_2sm_u32(bar, 3);       // same barrier in both CTAs of the pair
  else       ptx::tc_commit_u32(bar);
}

template <bool kTF32, bool kPair>
__device__ __forceinline__ void sc_mma(uint32_t d_tmem, uint64_t ad, uint64_t bd, uint32_t idesc, uint32_t acc) {
  if (kPair) { if (kTF32) ptx::mma_tf32_2sm(d_tmem, ad, bd, idesc, acc); else ptx::mma_bf16_2sm(d_tmem, ad, bd, idesc, acc); }
  else       { if (kTF32) ptx::mma_tf32(d_tmem, ad, bd, idesc, acc);     else ptx::mma_bf16(d_tmem, ad, bd, idesc, acc); }
}

// kPer = MMAs (of 32 K bytes) per operand HALF in split mode, per chunk otherwise.
template <bool kTF32, int TPS, int kPer, bool kPair, int NK, bool kSplit>
__device__ __forceinline__ void sc_issue_group(const ScIssue& z, uint32_t d_tmem, uint64_t xdesc, uint64_t wdesc, int g,
                                               uint32_t first) {
#pragma unroll
  for (int tt = 0; tt < TPS; ++tt) {
    const int kyx = NK == 2 ? g / 2 : g * TPS + tt;
    const uint32_t xrow = ((kyx / 3) * kHX + (kyx % 3)) * z.rb16;
    if constexpr (!kSplit) {
      const uint32_t xoff = xrow + (NK == 2 ? (g & 1) * z.chunk_step : 0u);
#pragma unroll
      for (int k = 0; k < kPer; ++k) {
        const uint32_t acc = (g == 0 && tt == 0 && k == 0) ? first : 1u;
        sc_mma<kTF32, kPair>(d_tmem, xdesc + xoff + 2 * k, wdesc + tt * z.tap_step + 2 * k, z.idesc, acc);
      }
    } else if constexpr (NK == 2) {
      // 256-byte rows: chunk 0 = hi, chunk 1 = lo; stage g = (tap g / 2, hi weights | lo weights)
      if ((g & 1) == 0) {
#pragma unroll
        for (int k = 0; k < kPer; ++k)               // x_hi * w_hi
          sc_mma<kTF32, kPair>(d_tmem, xdesc + xrow + 2 * k, wdesc + 2 * k, z.idesc, (g == 0 && k == 0) ? first : 1u);
#pragma unroll
        for (int k = 0; k < kPer; ++k)               // x_lo * w_hi
          sc_mma<kTF32, kPair>(d_tmem, xdesc + xrow + z.chunk_step + 2 * k, wdesc + 2 * k, z.idesc, 1u);
      } else {
#pragma unroll
        for (int k = 0; k < kPer; ++k)               // x_hi * w_lo
          sc_mma<kTF32, kPair>(d_tmem, xdesc + xrow + 2 * k, wdesc + 2 * k, z.idesc, 1u);
      }
    } else {
      // one physical chunk [hi | lo]: the lo half starts kPer MMA steps (32 bytes each) into the row
      const uint64_t wd = wdesc + tt * z.tap_step;
#pragma unroll
      for (int k = 0; k < kPer; ++k)                 // x_hi * w_hi
        sc_mma<kTF32, kPair>(d_tmem, xdesc + xrow + 2 * k, wd + 2 * k, z.idesc, (g == 0 && tt == 0 && k == 0) ? first : 1u);
#pragma unroll
      for (int k = 0; k < kPer; ++k)                 // x_lo * w_hi
        sc_mma<kTF32, kPair>(d_tmem, xdesc + xrow + 2 * (kPer + k), wd + 2 * k, z.idesc, 1u);
#pragma unroll
      for (int k = 0; k < kPer; ++k)                 // x_hi * w_lo
        sc_mma<kTF32, kPair>(d_tmem, xdesc + xrow + 2 * k, wd + 2 * (kPer + k), z.idesc, 1u);
    }
  }
}

// The residual plane as one more tap with identity weights: K = Cout channels = CP / 16 MMAs of N = CP into the slot of the
// plane's own output (kz = 1 block: slot p % 3).
template <bool kPair, int CP>
__device__ __forceinline__ void sc_res_mma(const ScRes& rs, uint32_t d_tmem, uint64_t adesc, uint64_t idd) {
#pragma unroll
  for (int k = 0; k < CP / 16; ++k) sc_mma<false, kPair>(d_tmem, adesc + 2 * k, idd + 2 * k, rs.idesc_r, 1u);
}

template <bool kTF32, int TPS, int kPer, bool kPair, int NK = 1, bool kSplit = false, bool kRM = false, int kTP = kTileCols>
__device__ __forceinline__ void sc_issue(const ScIssue& z, const ScRes* rs = nullptr) {
  constexpr int G = 9 * NK / TPS;
  int ws = 0;  uint32_t wphase = 0;
  int pw = 0;  uint32_t pwphase = 0;
  uint32_t aphase = 0;
  [[maybe_unused]] uint32_t rphase = 0;
  [[maybe_unused]] uint64_t rdesc = 0, idd = 0;
  if constexpr (kRM) {
    const uint64_t hi = desc_hi(8 * 128, 128);
    rdesc = hi | desc_lo(rs->res_u32);
    idd = hi | desc_lo(rs->ident_u32);
  }
  const uint32_t w_lo0 = desc_lo(z.w_u32), w_lo_step = z.w_bytes >> 4;
  const uint32_t x_lo0 = desc_lo(z.planes_u32), x_lo_step = z.slot_bytes >> 4;
  const uint32_t d0 = z.tmem_base, d1 = z.tmem_base + kTP;
  for (int ci = 0; ci < z.ncols; ++ci) {
    const Item it = cta_item(*z.args, ci);
    for (int p = 0; p < z.D; p = next_plane(it, p)) {
      ptx::mbar_wait_u32(z.bar_pf + 8 * pw, pwphase);
      const uint64_t xd0 = z.x_hi | (x_lo0 + pw * x_lo_step);
      const uint64_t xd1 = xd0 + z.tile_off;
      const uint32_t first = p == 0 ? 0u : 1u;     // the first MMA of a column overwrites all three slots
      int ws_prev = 0;
#pragma unroll
      for (int g = 0; g <= G; ++g) {
        if (g < G) {                               // tile 0, group g
          ptx::mbar_wait_u32(z.bar_wf + 8 * ws, wphase);
          if (g == 0) ptx::mbar_wait_u32(z.bar_ae, aphase ^ 1);
          ptx::tc_fence_after();
          const uint64_t wd = z.w_hi | (w_lo0 + ws * w_lo_step);
          if constexpr (kRM) { if (g == G / 2) { ptx::mbar_wait_u32(rs->bar_rf, rphase); ptx::tc_fence_after(); } }
          if (ptx::elect_one()) {
            sc_issue_group<kTF32, TPS, kPer, kPair, NK, kSplit>(z, d0, xd0, wd, g, first);
            if constexpr (kRM) { if (g == G / 2) sc_res_mma<kPair, 64>(*rs, d0 + (uint32_t)(p % 3) * rs->cp, rdesc, idd); }
            if (g == G - 1) sc_commit<kPair>(z.bar_af);
          }
          __syncwarp();
        }
        if (g >= 1) {                              // tile 1, group g-1 (its stage was awaited one iteration ago)
          if (g == 1) { ptx::mbar_wait_u32(z.bar_ae + 8, aphase ^ 1); ptx::tc_fence_after(); }
          const uint64_t wd = z.w_hi | (w_lo0 + ws_prev * w_lo_step);
          if (ptx::elect_one()) {
            sc_issue_group<kTF32, TPS, kPer, kPair, NK, kSplit>(z, d1, xd1, wd, g - 1, first);
            sc_commit<kPair>(z.bar_we + 8 * ws_prev);
            if constexpr (kRM) {
              if (g == G / 2 + 1) {                // tile 1's pixels are the second 16 KB of the staged residual plane
                sc_res_mma<kPair, 64>(*rs, d1 + (uint32_t)(p % 3) * rs->cp, rdesc + (128 * 128 >> 4), idd);
                sc_commit<kPair>(rs->bar_re);
              }
            }
            if (g == G) { sc_commit<kPair>(z.bar_af + 8); sc_commit<kPair>(z.bar_pe + 8 * pw); }
          }
          __syncwarp();
        }
        if (g < G) {
          ws_prev = ws;
          if (++ws == z.w_stages) { ws = 0; wphase ^= 1; }
        }
      }
      aphase ^= 1;
      if constexpr (kRM) rphase ^= 1;
      if (++pw == z.ring) { pw = 0; pwphase ^= 1; }
    }
  }
}

// ---- epilogue ------------------------------------------------------------------------------------------------------
// A thread owns one pixel (TMEM lane) and all of its channels, i.e. a 128-byte run of the channels-last output; stored
// directly, one warp instruction would touch 32 different lines with 16 bytes each.  ncu showed those scattered
// stores filling 40 % of the L1 data pipe that also feeds the tensor core its shared-memory operands (56 %), which
// cost 25 % of the kernel.  So the 16-byte chunks are transposed inside each group of NCH lanes first (butterfly of
// warp shuffles): lane j of a group then holds chunk j of every pixel of the group, and one instruction writes whole
// pixels contiguously (4 lines per instruction instead of 32).  Residual reads go the same way round.
template <int NCH>
__device__ __forceinline__ void chunk_transpose(uint4 (&c)[NCH], int lane) {
#pragma unroll
  for (int s = NCH / 2; s >= 1; s >>= 1) {
    const bool up = (lane & s) != 0;
#pragma unroll
    for (int a = 0; a < NCH; ++a) {
      if (a & s) continue;
      const uint4 send = up ? c[a] : c[a | s];
      uint4 recv;
      recv.x = __shfl_xor_sync(0xffffffffu, send.x, s);
      recv.y = __shfl_xor_sync(0xffffffffu, send.y, s);
      recv.z = __shfl_xor_sync(0xffffffffu, send.z, s);
      recv.w = __shfl_xor_sync(0xffffffffu, send.w, s);
      if (up) c[a] = recv; else c[a | s] = recv;
    }
  }
}

struct ScEpi {
  const float* bias;  const void* residual;  void* out;
  float slope;                 // none / ReLU / LeakyReLU as max(v,0) + slope * min(v,0)
  int osW;
  int res_direct;              // residual read per own pixel (no transpose) instead of per transpose group
};

// Coalesced read of the residual chunks of this lane's group of pixels (then transposed back to "my pixel").
template <int NCH, typename TOut>
__device__ __forceinline__ void sc_res_load(const ScEpi& e, int64_t grp_off, int osW, int lane, uint32_t okmask, uint4 (&r)[NCH]) {
  const int j = lane & (NCH - 1);
  if (e.res_direct) {
    const int own = (lane & 7) & (NCH - 1);            // this lane's pixel inside its group
    const TOut* rs = reinterpret_cast<const TOut*>(e.residual) + grp_off + own * osW;
    const bool ok = (okmask >> own) & 1u;
#pragma unroll
    for (int k = 0; k < NCH; ++k)
      r[k] = ok ? __ldg(reinterpret_cast<const uint4*>(rs) + k) : make_uint4(0, 0, 0, 0);
    return;
  }
  const TOut* rs = reinterpret_cast<const TOut*>(e.residual) + grp_off + j * (16 / (int)sizeof(TOut));
#pragma unroll
  for (int k = 0; k < NCH; ++k)
    r[k] = ((okmask >> k) & 1u) ? __ldg(reinterpret_cast<const uint4*>(rs + k * osW)) : make_uint4(0, 0, 0, 0);
}

// kAct: 0 ReLU, 2 general slope (none / leaky).  (An identity variant that skips the three slope instructions was
// measured SLOWER on the residual layer, 2.85 vs 2.70 ms, and grew the kernel; it is not instantiated.)
// ncopy > 0: the same values are stored again at ncopy more planes, zstep elements apart.
template <int CP, typename TOut, bool kRes, int kAct>
__device__ __forceinline__ void sc_fast_store(const ScEpi& e, int64_t grp_off, int lane, uint32_t okmask,
                                              const uint32_t (&v)[CP / 16][16], uint4 (&r)[CP * sizeof(TOut) / 16],
                                              int ncopy = 0, int64_t zstep = 0) {
  constexpr int NCH = CP * sizeof(TOut) / 16;
  constexpr int CPC = 16 / sizeof(TOut);          // channels per chunk
  uint4 c[NCH];
  if (kRes && !e.res_direct) chunk_transpose<NCH>(r, lane);
#pragma unroll
  for (int jg = 0; jg < CP / 16; ++jg) {
    float f[16];
    const float4* b4 = reinterpret_cast<const float4*>(e.bias + 16 * jg);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 b = __ldg(b4 + i);
      f[4 * i] = __uint_as_float(v[jg][4 * i]) + b.x;          f[4 * i + 1] = __uint_as_float(v[jg][4 * i + 1]) + b.y;
      f[4 * i + 2] = __uint_as_float(v[jg][4 * i + 2]) + b.z;  f[4 * i + 3] = __uint_as_float(v[jg][4 * i + 3]) + b.w;
    }
    if (kRes) {
      if (sizeof(TOut) == 2) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const __nv_bfloat162* hp = reinterpret_cast<const __nv_bfloat162*>(&r[2 * jg + h]);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float2 g = __bfloat1622float2(hp[i]);
            f[8 * h + 2 * i] += g.x;  f[8 * h + 2 * i + 1] += g.y;
          }
        }
      } else {
#pragma unroll
        for (int h = 0; h < 4; ++h) {
          const float4 g = *reinterpret_cast<const float4*>(&r[4 * jg + h]);
          f[4 * h] += g.x;  f[4 * h + 1] += g.y;  f[4 * h + 2] += g.z;  f[4 * h + 3] += g.w;
        }
      }
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) f[i] = kAct == 0 ? fmax_nan(f[i], 0.f) : (kAct == 1 ? f[i] : fmax_nan(f[i], 0.f) + e.slope * fmin_nan(f[i], 0.f));
    if (sizeof(TOut) == 2) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        __nv_bfloat162* hp = reinterpret_cast<__nv_bfloat162*>(&c[2 * jg + h]);
#pragma unroll
        for (int i = 0; i < 4; ++i) hp[i] = __floats2bfloat162_rn(f[8 * h + 2 * i], f[8 * h + 2 * i + 1]);
      }
    } else {
#pragma unroll
      for (int h = 0; h < 4; ++h) c[4 * jg + h] = *reinterpret_cast<const uint4*>(&f[4 * h]);
    }
  }
  chunk_transpose<NCH>(c, lane);
  const int j = lane & (NCH - 1);
  TOut* o = reinterpret_cast<TOut*>(e.out) + grp_off + j * CPC;
  for (int i = 0; i <= ncopy; ++i, o += zstep) {
#pragma unroll
    for (int k = 0; k < NCH; ++k)
      if ((okmask >> k) & 1u) *reinterpret_cast<uint4*>(o + k * e.osW) = c[k];
  }
}

// One drained plane: residual chunks `r` (already loaded, still in group order) + accumulators -> coalesced stores.
template <int CP, typename TOut>
__device__ __forceinline__ void sc_fast_plane(const ScEpi& e, int64_t grp_off, int lane, uint32_t okmask,
                                              const uint32_t (&v)[CP / 16][16], uint4 (&r)[CP * sizeof(TOut) / 16],
                                              int ncopy, int64_t zstep) {
  if (e.slope == 0.f) {                             // ReLU (the aggregation layers): one instruction per value
    if (e.residual) sc_fast_store<CP, TOut, true, 0>(e, grp_off, lane, okmask, v, r, ncopy, zstep);
    else            sc_fast_store<CP, TOut, false, 0>(e, grp_off, lane, okmask, v, r, ncopy, zstep);
  } else {
    if (e.residual) sc_fast_store<CP, TOut, true, 2>(e, grp_off, lane, okmask, v, r, ncopy, zstep);
    else            sc_fast_store<CP, TOut, false, 2>(e, grp_off, lane, okmask, v, r, ncopy, zstep);
  }
}

// kFast: transposed stores (needs a power-of-two chunk count per pixel).  kSRes / kSAct >= 0: residual / activation fixed at
// compile time (the specialised kernels below), -1: decided at run time.
template <int CP, typename TOut, bool kFast, int kSRes = -1, int kSAct = -1, int kTP = kTileCols>
__device__ __forceinline__ void sc_epilogue(const ScArgs& a, ScCtrl& ctrl, uint32_t tmem_base, int warp, int lane) {
  constexpr int NCH = kFast ? CP * (int)sizeof(TOut) / 16 : 1;     // 16-byte chunks per pixel
  const int t = (warp - 4) >> 2, q = warp & 3;
  const EpiParams ep = {a.bias, a.residual, a.out, a.p.cout_store, sizeof(TOut) == 2, a.p.act, a.p.act_param, 1, nullptr, 0, 0};
  const ScEpi fe = {a.bias, a.residual, a.out,
                    a.p.act == S3D_ACT_NONE ? 1.f : (a.p.act == S3D_ACT_LEAKY ? a.p.act_param : 0.f), (int)a.p.osW, a.res_direct};
  const uint32_t bar_af = ptx::smem_u32(&ctrl.acc_full[t]), bar_ae = ptx::smem_u32(&ctrl.acc_empty[t]);
  const uint32_t tbase = tmem_base + t * kTP + (static_cast<uint32_t>(q * 32) << 16);
  const int yl = t * kTileY + q * 4 + (lane >> 3), xl = lane & 7;      // TMEM lane = 8 * row + x inside the tile
  const int D = a.dl;                                 // local planes per work item (= oD unless z-split)
  const int zs0 = a.nz > 1 ? 1 : 0, zs1 = a.nz > 1 ? a.zc + 1 : D;     // local output planes a work item stores
  const int xb = xl & ~(NCH - 1);                     // first pixel of this lane's transpose group
  uint32_t aphase = 0;
  const int ncols = cta_cols(a);
  for (int ci = 0; ci < ncols; ++ci) {
    const Item it = cta_item(a, ci);
    const Col& c = it.c;
    const bool rowok = c.y0 + yl < a.p.oH && c.n < a.p.N;
    const bool ok = rowok && c.x0 + xl < a.p.oW;
    const int64_t row_off = (int64_t)c.n * a.p.osN + (int64_t)(c.y0 + yl) * a.p.osH + (int64_t)c.x0 * a.p.osW;
    const int64_t pix_off = row_off + (int64_t)xl * a.p.osW;
    const int64_t grp_off = row_off + (int64_t)xb * a.p.osW;
    uint32_t okmask = 0;                              // which pixels of the group exist
#pragma unroll
    for (int k = 0; k < NCH; ++k) okmask |= (rowok && c.x0 + xb + k < a.p.oW) ? (1u << k) : 0u;
    int slot = 0, z = 0;                              // next output plane to drain and its slot (z % 3)
    for (int p = 0; p < D; p = next_plane(it, p)) {
      // input plane p done => out plane p-1 is complete; after the last input plane so is out plane D-1
      const int ndrain = (p >= 1 ? 1 : 0) + (p == D - 1 ? 1 : 0);
      uint4 r[NCH];
      if constexpr (kFast) {                          // residual of the plane about to be drained: in flight during the wait
        if (a.residual && ndrain)
          sc_res_load<NCH, TOut>(fe, grp_off + (int64_t)(c.zb + z) * a.p.osD, fe.osW, lane,
                                 (z >= zs0 && z < zs1 && c.zb + z < a.p.oD) ? okmask : 0u, r);
      }
      ptx::mbar_wait_u32(bar_af, aphase);
      ptx::tc_fence_after();
      if (ndrain == 0) {
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) { if (a.pair) ptx::mbar_arrive_cluster_u32(bar_ae, 0); else ptx::mbar_arrive_u32(bar_ae); }
      }
      for (int i = 0; i < ndrain; ++i) {
        uint32_t v[CP / 16][16];
        const uint32_t taddr = tbase + slot * CP;
#pragma unroll
        for (int j = 0; j < CP / 16; ++j) ptx::tmem_ld16(taddr + 16 * j, v[j]);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < CP / 16; ++j) ptx::tmem_st16_zero(taddr + 16 * j);
        ptx::tmem_st_wait();
        if (i == ndrain - 1) {                        // hand the tile back before the arithmetic / stores
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) { if (a.pair) ptx::mbar_arrive_cluster_u32(bar_ae, 0); else ptx::mbar_arrive_u32(bar_ae); }
        }
        const int64_t zo = (int64_t)(c.zb + z) * a.p.osD;
        const bool stz = z >= zs0 && z < zs1 && c.zb + z < a.p.oD;       // z-split: a chunk's border planes are not stored
        const uint32_t om = stz ? okmask : 0u;
        const int ncopy = z == it.zs ? it.J : 0;      // out planes zs + 1 .. zs + J are copies of plane zs (never z-split)
        if constexpr (kFast) {
          // (second drain of the last plane: its residual could not be prefetched)
          if (i == 1 && a.residual) sc_res_load<NCH, TOut>(fe, grp_off + zo, fe.osW, lane, om, r);
          if constexpr (kSRes >= 0) sc_fast_store<CP, TOut, kSRes != 0, kSAct>(fe, grp_off + zo, lane, om, v, r, ncopy, a.p.osD);
          else sc_fast_plane<CP, TOut>(fe, grp_off + zo, lane, om, v, r, ncopy, a.p.osD);
        } else {
          if (ok && stz) {
            for (int k = 0; k <= ncopy; ++k) {
#pragma unroll
              for (int j = 0; j < CP / 16; ++j) epilogue_store16(ep, pix_off + zo + k * a.p.osD, 16 * j, v[j]);
            }
          }
        }
        z += ncopy;                                   // ncopy % 3 == 0: the slot stays
        ++z;
        if (++slot == 3) slot = 0;
      }
      aphase ^= 1;
    }
  }
}

template <int CP>
__device__ __forceinline__ void sc_epilogue_dispatch(const ScArgs& a, ScCtrl& ctrl, uint32_t tmem_base, int warp, int lane) {
  constexpr bool kPow2_16 = CP == 16 || CP == 32 || CP == 64;      // bf16: CP / 8 chunks
  constexpr bool kPow2_32 = CP == 16 || CP == 32;                  // fp32: CP / 4 chunks, at most 8
  if (a.p.out_dtype == S3D_DTYPE_BF16) {
    if (kPow2_16 && a.fast_store) sc_epilogue<CP, __nv_bfloat16, kPow2_16>(a, ctrl, tmem_base, warp, lane);
    else sc_epilogue<CP, __nv_bfloat16, false>(a, ctrl, tmem_base, warp, lane);
  } else {
    if (kPow2_32 && a.fast_store) sc_epilogue<CP, float, kPow2_32>(a, ctrl, tmem_base, warp, lane);
    else sc_epilogue<CP, float, false>(a, ctrl, tmem_base, warp, lane);
  }
}

// ---- split (BF16X2) epilogue -------------------------------------------------------------------------------------------
// Output and residual are [hi(CP) | lo(CP)] bf16 per pixel (lo parts os_lo elements after the hi parts).  The value is
// finished in fp32 (bias, residual = hi + lo, activation), written back over the accumulator registers, and stored as
// two transposed (coalesced) passes: hi = bf16(v), then lo = bf16(v - hi).  With three MMA passes per tap the tensor core
// spends 3x longer on a plane than in the bf16 kernel, so this epilogue has slack the bf16 one does not.
template <int NCH>
__device__ __forceinline__ void sc_res_load_split(const ScEpi& e, int64_t os_lo, int64_t grp_off, int lane, uint32_t okmask,
                                                  uint4 (&rh)[NCH], uint4 (&rl)[NCH]) {
  const int own = (lane & 7) & (NCH - 1);              // this lane's pixel inside its transpose group
  const __nv_bfloat16* rs = reinterpret_cast<const __nv_bfloat16*>(e.residual) + grp_off + (int64_t)own * e.osW;
  const bool ok = (okmask >> own) & 1u;
#pragma unroll
  for (int k = 0; k < NCH; ++k) {
    rh[k] = ok ? __ldg(reinterpret_cast<const uint4*>(rs) + k) : make_uint4(0, 0, 0, 0);
    rl[k] = ok ? __ldg(reinterpret_cast<const uint4*>(rs + os_lo) + k) : make_uint4(0, 0, 0, 0);
  }
}

template <int CP, bool kRes, int kAct>
__device__ __forceinline__ void sc_split_store(const ScEpi& e, int64_t os_lo, int64_t grp_off, int lane, uint32_t okmask,
                                               uint32_t (&v)[CP / 16][16], const uint4 (&rh)[CP / 8], const uint4 (&rl)[CP / 8]) {
  constexpr int NCH = CP / 8;                           // 16-byte chunks of one half of a pixel
  // pass 0: v <- act(v + bias (+ residual)) as fp32 bits
#pragma unroll
  for (int jg = 0; jg < CP / 16; ++jg) {
    const float4* b4 = reinterpret_cast<const float4*>(e.bias + 16 * jg);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 b = __ldg(b4 + i);
      float f0 = __uint_as_float(v[jg][4 * i]) + b.x, f1 = __uint_as_float(v[jg][4 * i + 1]) + b.y;
      float f2 = __uint_as_float(v[jg][4 * i + 2]) + b.z, f3 = __uint_as_float(v[jg][4 * i + 3]) + b.w;
      if (kRes) {
        // channels 16 jg + 4 i .. + 3 = halves (2 i) % 4, (2 i + 1) % 4 of chunk 2 jg + i / 2
        const __nv_bfloat162* ph = reinterpret_cast<const __nv_bfloat162*>(&rh[2 * jg + (i >> 1)]) + 2 * (i & 1);
        const __nv_bfloat162* pl = reinterpret_cast<const __nv_bfloat162*>(&rl[2 * jg + (i >> 1)]) + 2 * (i & 1);
        const float2 h0 = __bfloat1622float2(ph[0]), h1 = __bfloat1622float2(ph[1]);
        const float2 l0 = __bfloat1622float2(pl[0]), l1 = __bfloat1622float2(pl[1]);
        f0 += h0.x + l0.x;  f1 += h0.y + l0.y;  f2 += h1.x + l1.x;  f3 += h1.y + l1.y;
      }
      if (kAct == 0) { f0 = fmax_nan(f0, 0.f); f1 = fmax_nan(f1, 0.f); f2 = fmax_nan(f2, 0.f); f3 = fmax_nan(f3, 0.f); }
      else if (kAct == 2) {
        f0 = fmax_nan(f0, 0.f) + e.slope * fmin_nan(f0, 0.f);  f1 = fmax_nan(f1, 0.f) + e.slope * fmin_nan(f1, 0.f);
        f2 = fmax_nan(f2, 0.f) + e.slope * fmin_nan(f2, 0.f);  f3 = fmax_nan(f3, 0.f) + e.slope * fmin_nan(f3, 0.f);
      }
      v[jg][4 * i] = __float_as_uint(f0);      v[jg][4 * i + 1] = __float_as_uint(f1);
      v[jg][4 * i + 2] = __float_as_uint(f2);  v[jg][4 * i + 3] = __float_as_uint(f3);
    }
  }
  const int j = lane & (NCH - 1);
  __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(e.out) + grp_off + j * 8;
#pragma unroll
  for (int half = 0; half < 2; ++half) {               // 0: hi parts, 1: lo parts
    uint4 c[NCH];
#pragma unroll
    for (int jg = 0; jg < CP / 16; ++jg) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        uint32_t w[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          uint32_t hi, lo;
          split_bf16x2(__uint_as_float(v[jg][8 * h + 2 * i]), __uint_as_float(v[jg][8 * h + 2 * i + 1]), hi, lo);
          w[i] = half == 0 ? hi : lo;
        }
        c[2 * jg + h] = make_uint4(w[0], w[1], w[2], w[3]);
      }
    }
    chunk_transpose<NCH>(c, lane);
    __nv_bfloat16* oh = o + (half == 0 ? (int64_t)0 : os_lo);
#pragma unroll
    for (int k = 0; k < NCH; ++k)
      if ((okmask >> k) & 1u) *reinterpret_cast<uint4*>(oh + k * e.osW) = c[k];
  }
}

template <int CP, int kSRes = -1, int kSAct = -1>
__device__ __forceinline__ void sc_epilogue_split(const ScArgs& a, ScCtrl& ctrl, uint32_t tmem_base, int warp, int lane) {
  constexpr int NCH = CP / 8;
  const int t = (warp - 4) >> 2, q = warp & 3;
  const ScEpi fe = {a.bias, a.residual, a.out,
                    a.p.act == S3D_ACT_NONE ? 1.f : (a.p.act == S3D_ACT_LEAKY ? a.p.act_param : 0.f), (int)a.p.osW, 1};
  const int64_t os_lo = a.os_lo;
  const uint32_t bar_af = ptx::smem_u32(&ctrl.acc_full[t]), bar_ae = ptx::smem_u32(&ctrl.acc_empty[t]);
  const uint32_t tbase = tmem_base + t * kTileCols + (static_cast<uint32_t>(q * 32) << 16);
  const int yl = t * kTileY + q * 4 + (lane >> 3), xl = lane & 7;
  const int D = a.dl;
  const int zs0 = a.nz > 1 ? 1 : 0, zs1 = a.nz > 1 ? a.zc + 1 : D;
  const int xb = xl & ~(NCH - 1);
  uint32_t aphase = 0;
  const int ncols = cta_cols(a);
  for (int ci = 0; ci < ncols; ++ci) {
    const Col c = decode_col(a, blockIdx.x + ci * gridDim.x);
    const bool rowok = c.y0 + yl < a.p.oH && c.n < a.p.N;
    const int64_t row_off = (int64_t)c.n * a.p.osN + (int64_t)(c.y0 + yl) * a.p.osH + (int64_t)c.x0 * a.p.osW;
    const int64_t grp_off = row_off + (int64_t)xb * a.p.osW;
    uint32_t okmask = 0;
#pragma unroll
    for (int k = 0; k < NCH; ++k) okmask |= (rowok && c.x0 + xb + k < a.p.oW) ? (1u << k) : 0u;
    int slot = 0, z = 0;
    for (int p = 0; p < D; ++p) {
      const int ndrain = (p >= 1 ? 1 : 0) + (p == D - 1 ? 1 : 0);
      uint4 rh[NCH], rl[NCH];
      if (a.residual && ndrain)
        sc_res_load_split<NCH>(fe, os_lo, grp_off + (int64_t)(c.zb + z) * a.p.osD, lane,
                               (z >= zs0 && z < zs1 && c.zb + z < a.p.oD) ? okmask : 0u, rh, rl);
      ptx::mbar_wait_u32(bar_af, aphase);
      ptx::tc_fence_after();
      if (ndrain == 0) {
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) { if (a.pair) ptx::mbar_arrive_cluster_u32(bar_ae, 0); else ptx::mbar_arrive_u32(bar_ae); }
      }
      for (int i = 0; i < ndrain; ++i) {
        uint32_t v[CP / 16][16];
        const uint32_t taddr = tbase + slot * CP;
#pragma unroll
        for (int j = 0; j < CP / 16; ++j) ptx::tmem_ld16(taddr + 16 * j, v[j]);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < CP / 16; ++j) ptx::tmem_st16_zero(taddr + 16 * j);
        ptx::tmem_st_wait();
        if (i == ndrain - 1) {
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) { if (a.pair) ptx::mbar_arrive_cluster_u32(bar_ae, 0); else ptx::mbar_arrive_u32(bar_ae); }
        }
        const int64_t zo = (int64_t)(c.zb + z) * a.p.osD;
        const uint32_t om = (z >= zs0 && z < zs1 && c.zb + z < a.p.oD) ? okmask : 0u;
        if (i == 1 && a.residual) sc_res_load_split<NCH>(fe, os_lo, grp_off + zo, lane, om, rh, rl);
        if constexpr (kSRes >= 0) {
          sc_split_store<CP, kSRes != 0, kSAct>(fe, os_lo, grp_off + zo, lane, om, v, rh, rl);
        } else if (fe.slope == 0.f) {
          if (a.residual) sc_split_store<CP, true, 0>(fe, os_lo, grp_off + zo, lane, om, v, rh, rl);
          else            sc_split_store<CP, false, 0>(fe, os_lo, grp_off + zo, lane, om, v, rh, rl);
        } else {
          if (a.residual) sc_split_store<CP, true, 2>(fe, os_lo, grp_off + zo, lane, om, v, rh, rl);
          else            sc_split_store<CP, false, 2>(fe, os_lo, grp_off + zo, lane, om, v, rh, rl);
        }
        ++z;
        if (++slot == 3) slot = 0;
      }
      aphase ^= 1;
    }
  }
}

// Taps per weight stage.  Narrow layers take all 9 in-plane taps in one stage when that fits 28 KB: a tile's accumulator
// hand-back hides behind the OTHER tile's current stage, and a stage of 3 one-MMA taps (~180 cycles) is too short for
// it (fusion scorer: 0.148 -> 0.100 ms per layer).
__host__ __device__ constexpr int spec_tps(int rb, int cp) {
  return rb == 128 ? 1 : (9 * (3 * cp / 2) * rb <= 28 * 1024 ? 9 : 3);
}

// RB != 0: a kernel specialised for ONE layer shape (bf16 rows of RB bytes, CP output channels, residual, activation).
// Every variant of producer / issuer / epilogue is inlined into the kernel, and the kernel is sensitive to its own code
// size (measured: two more epilogue variants in the all-in-one kernel cost 4 % of the whole forward), so the layer
// shapes of the network each get a kernel that contains only their own code.  RB == 0: all-in-one, run-time dispatch.
// kSplit: BF16X2 operands and output (see ScArgs::split).  RB is then the PHYSICAL row (64 / 128 bytes: one chunk; 256: two).
// kTwo: a narrow layer shape (3 * CP <= 128 accumulator columns per tile) that leaves room for TWO CTAs per SM -- half the
// TMEM columns (tile pitch 128), half the shared memory, <= 85 registers.  Its planes are too short (9 one-MMA taps per tile)
// to hide the accumulator hand-back behind the other tile; a second resident CTA fills the bubbles (fusion scorer layers).
template <bool kTF32, bool kPair, int RB = 0, int CP = 0, int kSRes = -1, int kSAct = -1, bool kSplit = false, bool kTwo = false>
__global__ void __launch_bounds__(kThreads, kTwo ? 2 : 1)
conv_scatter_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w,
                    const __grid_constant__ ScArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_w = smem + a.ring * a.slot_bytes;
  __shared__ ScCtrl ctrl;
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&map_x);
    ptx::prefetch_tensormap(&map_w);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < kMaxRing; ++s) { ptx::mbar_init(&ctrl.plane_full[s], 1); ptx::mbar_init(&ctrl.plane_empty[s], 1); }
    for (int s = 0; s < kMaxW; ++s) { ptx::mbar_init(&ctrl.w_full[s], 1); ptx::mbar_init(&ctrl.w_empty[s], 1); }
    // accumulator hand-back: one arrival per epilogue warp of the tile -- of both CTAs in pair mode (on the leader's barrier)
    for (int b = 0; b < 2; ++b) { ptx::mbar_init(&ctrl.acc_full[b], 1); ptx::mbar_init(&ctrl.acc_empty[b], kPair ? 8 : 4); }
    ptx::fence_barrier_init();
  }
  constexpr int kTP = kTwo ? 128 : kTileCols;
  if (warp == 2) { if (kPair) ptx::tmem_alloc_2sm(&ctrl.tmem_base, 2 * kTP); else ptx::tmem_alloc(&ctrl.tmem_base, 2 * kTP); }
  ptx::tc_fence_before();
  __syncthreads();
  if (kPair) ptx::cluster_sync_all();              // the peer's barriers exist before anything is signalled at them
  ptx::tc_fence_after();
  const uint32_t tmem_base = ctrl.tmem_base;

  if (warp == 0) {
    const uint32_t planes_u32 = ptx::smem_u32(smem), w_u32 = ptx::smem_u32(smem_w);
    if constexpr (RB == 256) sc_produce<1, kPair, 2>(a, ctrl, planes_u32, w_u32, &map_x, &map_w);
    else if constexpr (RB == 128) sc_produce<1, kPair>(a, ctrl, planes_u32, w_u32, &map_x, &map_w);
    else if constexpr (RB != 0) sc_produce<spec_tps(RB, CP), kPair>(a, ctrl, planes_u32, w_u32, &map_x, &map_w);
    else if (a.nchunks == 2) sc_produce<1, kPair, 2>(a, ctrl, planes_u32, w_u32, &map_x, &map_w);
    else if (a.tps == 1) sc_produce<1, kPair>(a, ctrl, planes_u32, w_u32, &map_x, &map_w);
    else if (a.tps == 3) sc_produce<3, kPair>(a, ctrl, planes_u32, w_u32, &map_x, &map_w);
    else sc_produce<9, kPair>(a, ctrl, planes_u32, w_u32, &map_x, &map_w);
  } else if (warp == 1 && (!kPair || ptx::cluster_ctarank() == 0)) {      // pair mode: the leader issues for both CTAs
    const int rb = a.row_bytes;
    const ScIssue zi = {tmem_base, ptx::smem_u32(smem), ptx::smem_u32(smem_w),
                        ptx::smem_u32(&ctrl.plane_full[0]), ptx::smem_u32(&ctrl.plane_empty[0]), ptx::smem_u32(&ctrl.w_full[0]),
                        ptx::smem_u32(&ctrl.w_empty[0]), ptx::smem_u32(&ctrl.acc_full[0]), ptx::smem_u32(&ctrl.acc_empty[0]),
                        desc_hi(kHX * rb, rb), desc_hi(8 * rb, rb), a.slot_bytes, a.w_bytes, a.w_stages, a.ring,
                        (uint32_t)(rb >> 4), (uint32_t)(((kPair ? 3 * a.cp / 2 : 3 * a.cp) * rb) >> 4), (uint32_t)((kTileY * kHX * rb) >> 4), (uint32_t)(a.chunk_stride >> 4), a.idesc,
                        a.dl, cta_cols(a), &a};
    if constexpr (kSplit) {
      // kPer counts the MMAs of one operand HALF here
      if constexpr (RB == 256) sc_issue<false, 1, 4, kPair, 2, true>(zi);
      else if constexpr (RB == 128) sc_issue<false, 1, 2, kPair, 1, true>(zi);
      else if constexpr (RB == 64) sc_issue<false, spec_tps(RB, CP), 1, kPair, 1, true>(zi);
      else if (a.nchunks == 2) sc_issue<false, 1, 4, kPair, 2, true>(zi);
      else if (rb == 128) sc_issue<false, 1, 2, kPair, 1, true>(zi);
      else if (a.tps == 9) sc_issue<false, 9, 1, kPair, 1, true>(zi);
      else sc_issue<false, 3, 1, kPair, 1, true>(zi);
    }
    else if constexpr (RB == 128) sc_issue<kTF32, 1, 4, kPair>(zi);
    else if constexpr (RB == 64) sc_issue<kTF32, spec_tps(RB, CP), 2, kPair>(zi);
    else if constexpr (RB == 32) sc_issue<kTF32, spec_tps(RB, CP), 1, kPair, 1, false, false, kTP>(zi);
    else if (a.nchunks == 2) sc_issue<kTF32, 1, 4, kPair, 2>(zi);
    else if (rb == 128) sc_issue<kTF32, 1, 4, kPair>(zi);
    else if (rb == 64 && a.tps == 9) sc_issue<kTF32, 9, 2, kPair>(zi);
    else if (rb == 64) sc_issue<kTF32, 3, 2, kPair>(zi);
    else if (a.tps == 3) sc_issue<kTF32, 3, 1, kPair>(zi);
    else sc_issue<kTF32, 9, 1, kPair>(zi);
  } else if (warp >= 4) {
    if constexpr (kSplit) {
      if constexpr (RB != 0) sc_epilogue_split<CP, kSRes, kSAct>(a, ctrl, tmem_base, warp, lane);
      else if (a.cp == 64) sc_epilogue_split<64>(a, ctrl, tmem_base, warp, lane);
      else if (a.cp == 32) sc_epilogue_split<32>(a, ctrl, tmem_base, warp, lane);
      else sc_epilogue_split<16>(a, ctrl, tmem_base, warp, lane);
    }
    else if constexpr (RB != 0) sc_epilogue<CP, __nv_bfloat16, true, kSRes, kSAct, kTP>(a, ctrl, tmem_base, warp, lane);
    else if (a.cp == 64) sc_epilogue_dispatch<64>(a, ctrl, tmem_base, warp, lane);
    else if (a.cp == 48) sc_epilogue_dispatch<48>(a, ctrl, tmem_base, warp, lane);
    else if (a.cp == 32) sc_epilogue_dispatch<32>(a, ctrl, tmem_base, warp, lane);
    else sc_epilogue_dispatch<16>(a, ctrl, tmem_base, warp, lane);
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (kPair) ptx::cluster_sync_all();              // no CTA leaves while its peer may still signal its barriers
  if (warp == 2) {
    ptx::tc_fence_after();
    if (kPair) ptx::tmem_dealloc_2sm(tmem_base, 2 * kTP); else ptx::tmem_dealloc(tmem_base, 2 * kTP);
  }
}


typedef void (*KernFn)(CUtensorMap, CUtensorMap, ScArgs);
// conv_scatter_spec.cu: the lean kernel for this layer shape (bf16, CTA pairs, coalesced epilogue), or nullptr
KernFn spec_kernel(int row_bytes, int cp, bool residual, bool relu, bool two_ctas = false);
// conv_scatter_split.cu: kernels for split (BF16X2) operands -- lean per-shape ones (CTA pairs; phys_row_bytes = bytes of a
// [hi | lo] pixel row) or, with lean = false, the all-in-one kernel for the given pairing
KernFn split_kernel(bool lean, bool pair, int phys_row_bytes, int cp, bool residual, bool relu);
// conv_scatter_rm.cu: the 64 -> 64 bf16 layer with its residual added on the tensor core (CTA pairs, no activation / ReLU)
typedef void (*KernFnR)(CUtensorMap, CUtensorMap, CUtensorMap, ScArgs);
KernFnR rm_kernel(bool relu);

// ---- host side: the decisions every plane-scatter launcher shares (conv_scatter.cu, conv_scatter_concat.cu,
// conv_scatter_cls.cu).  Shared-memory budgets, ring depths, weight stages and kernel choices stay with each launcher.

// Plane slots, weight stages and the kernels' shared-memory base are 1024-byte aligned (the 128B-swizzle atom pattern).
inline int align1024(int bytes) { return (bytes + 1023) / 1024 * 1024; }

// A layer the plane-scatter kernels compute: stride 1, the 27 taps of a 3x3x3 kernel in canonical order (dz major, dx
// fastest), output grid = input grid, one class, and a plain output (no coordinate multipliers, projection or planar
// channel stride).
inline bool plane_scatter_layer(const S3dConvParams& p) {
  if (p.n_classes != 1 || p.sx != 1 || p.sy != 1 || p.sz != 1 || p.ntaps != 27) return false;
  if (p.omx != 1 || p.omy != 1 || p.omz != 1 || p.osC != 1 || p.proj_w) return false;
  if (p.oD != p.iD || p.oH != p.iH || p.oW != p.iW) return false;
  for (int t = 0; t < 27; ++t)
    if (p.dz[t] != t / 9 - 1 || p.dy[t] != (t % 9) / 3 - 1 || p.dx[t] != t % 3 - 1) return false;
  return true;
}

// Plane slots of nchunks K chunks of row_bytes bytes (kc channels) each, the kTY x kTX columns of a.p's output grid and
// no z-split (a work item marches its whole column).  -> the column count.
inline int64_t plane_geometry(ScArgs& a, int row_bytes, int kc, int nchunks) {
  a.row_bytes = row_bytes;  a.kc = kc;  a.nchunks = nchunks;
  a.chunk_stride = align1024(kPlaneRows * row_bytes);
  a.slot_bytes = nchunks * a.chunk_stride;
  a.cols_x = ceil_div(a.p.oW, kTX);  a.cols_y = ceil_div(a.p.oH, kTY);
  a.nz = 1;  a.zc = a.p.oD;  a.dl = a.p.oD;
  return (int64_t)a.p.N * a.cols_x * a.cols_y;
}

// Deals `total` work items to at most `grid` CTAs (a.pair decided): CTA pairs take an even grid and each walks
// ncols_max items (cta_cols), single CTAs stride over the items.  -> the grid to launch.
inline int deal_columns(ScArgs& a, int64_t total, int grid) {
  a.total_cols = (int)total;
  if (a.pair) {
    if ((int64_t)grid > total) grid = (int)((total + 1) / 2 * 2);
    grid -= grid % 2;
    a.ncols_max = (int)((total + grid - 1) / grid);
  } else if ((int64_t)grid > total) grid = (int)total;
  return grid;
}

// The transposed (coalesced) epilogue stores: 16-byte aligned out / residual (nullptr: none), 16-byte multiples as
// pixel strides, osW < 2^24, a bias, every channel stored, a none / ReLU / LeakyReLU activation.
inline bool coalesced_store_ok(const S3dConvParams& p, const float* bias, const void* out, const void* residual, int out_elem_size) {
  const bool simple_act = p.act == S3D_ACT_NONE || p.act == S3D_ACT_RELU || p.act == S3D_ACT_LEAKY;
  auto aligned = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
  auto dense16 = [&](int64_t st) { return (st * out_elem_size) % 16 == 0; };
  return simple_act && bias != nullptr && p.cout_store == p.Cout && aligned(out) && aligned(residual) &&
         dense16(p.osW) && dense16(p.osH) && dense16(p.osD) && dense16(p.osN) && p.osW < (1ll << 24);
}

// Launches a plane-scatter kernel with `smem` bytes of dynamic shared memory: as clusters of two CTAs when `pair`
// (cta_group::2), plainly otherwise.
template <typename... KArgs, typename... Args>
int launch_plane_scatter(void (*kern)(KArgs...), int grid, int smem, bool pair, cudaStream_t stream, const Args&... args) {
  S3D_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  if (pair) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(grid);  cfg.blockDim = dim3(kThreads);  cfg.dynamicSmemBytes = smem;  cfg.stream = stream;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeClusterDimension;
    attr.val.clusterDim.x = 2;  attr.val.clusterDim.y = 1;  attr.val.clusterDim.z = 1;
    cfg.attrs = &attr;  cfg.numAttrs = 1;
    S3D_CUDA(cudaLaunchKernelEx(&cfg, kern, args...));
  } else {
    kern<<<grid, kThreads, smem, stream>>>(args...);
  }
  S3D_LAUNCH_CHECK();
  return S3D_OK;
}

}  // namespace scatter
}  // namespace s3d
