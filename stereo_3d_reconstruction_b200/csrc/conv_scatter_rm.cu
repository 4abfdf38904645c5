// Plane-scatter 3x3x3 conv, 64 -> 64 bf16, with the RESIDUAL added on the tensor core (conv_scatter.cuh for the design).
//
// The residual layer of the aggregation (dres1b) cost 0.45 ms more than its siblings: every epilogue thread read its pixel's
// 128 residual bytes as eight scattered 16-byte loads (32 lines per warp instruction, 2048 L1 wavefronts per plane on the
// data pipe the tensor core reads its operands through); coalesced loads + a second shuffle transpose and TMA-staged tiles
// read back with LDS were both measured slower.  Here the residual never touches a thread: the plane of the 32x8 patch
// (256 pixels x 128 B, no halo) is staged by ONE TMA box per plane and added to the accumulators as one more "tap" whose
// weight matrix is the identity -- 4 MMAs of N = 64 per tile into the slot of the plane's own output (+6 % tensor work,
// exact: bf16 x 1.0 accumulated in fp32).  The epilogue is the plain one of the non-residual layers.
// Costs: 32 KB + 4 KB of shared memory, i.e. three weight stages (8 -> 5).
#include "conv_scatter.cuh"

namespace s3d {
namespace scatter {

template <int kSAct>
__global__ void __launch_bounds__(kThreads, 1)
conv_scatter_rm_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w,
                       const __grid_constant__ CUtensorMap map_r, const __grid_constant__ ScArgs a) {
  constexpr bool kPair = true;
  constexpr int CP = 64;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_w = smem + a.ring * a.slot_bytes;
  uint8_t* smem_res = smem_w + a.w_stages * a.w_bytes;
  uint8_t* smem_id = smem_res + kResBytes;
  __shared__ ScCtrl ctrl;
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&map_x);
    ptx::prefetch_tensormap(&map_w);
    ptx::prefetch_tensormap(&map_r);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < kMaxRing; ++s) { ptx::mbar_init(&ctrl.plane_full[s], 1); ptx::mbar_init(&ctrl.plane_empty[s], 1); }
    for (int s = 0; s < kMaxW; ++s) { ptx::mbar_init(&ctrl.w_full[s], 1); ptx::mbar_init(&ctrl.w_empty[s], 1); }
    for (int b = 0; b < 2; ++b) { ptx::mbar_init(&ctrl.acc_full[b], 1); ptx::mbar_init(&ctrl.acc_empty[b], 8); }
    ptx::mbar_init(&ctrl.res_full, 1);  ptx::mbar_init(&ctrl.res_empty, 1);
    ptx::fence_barrier_init();
  }
  if (warp == 2) ptx::tmem_alloc_2sm(&ctrl.tmem_base, kTmemCols);
  if (warp == 3) {
    // this CTA's half of the 64 x 64 identity (rows = output channels 32 * rank .. + 32), K-major 128-byte rows in the
    // 128B-swizzled layout the UMMA descriptor expects: 16-byte chunk c of row r sits at chunk c ^ (r % 8)
    uint4* z4 = reinterpret_cast<uint4*>(smem_id);
    for (int i = lane; i < (CP / 2) * 128 / 16; i += 32) z4[i] = make_uint4(0, 0, 0, 0);
    __syncwarp();
    const int r = lane, ci = (int)ptx::cluster_ctarank() * (CP / 2) + lane;
    *reinterpret_cast<__nv_bfloat16*>(smem_id + (r >> 3) * 1024 + (r & 7) * 128 + (((ci >> 3) ^ (r & 7)) << 4) + (ci & 7) * 2) =
        __float2bfloat16_rn(1.f);
    ptx::fence_proxy_async();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync_all();
  ptx::tc_fence_after();
  const uint32_t tmem_base = ctrl.tmem_base;
  const ScRes rs = {&map_r, ptx::smem_u32(smem_res), ptx::smem_u32(smem_id), ptx::smem_u32(&ctrl.res_full),
                    ptx::smem_u32(&ctrl.res_empty), ptx::make_instr_desc(1, 256, CP), CP};

  if (warp == 0) {
    sc_produce<1, kPair, 1, true>(a, ctrl, ptx::smem_u32(smem), ptx::smem_u32(smem_w), &map_x, &map_w, &rs);
  } else if (warp == 1 && ptx::cluster_ctarank() == 0) {
    const int rb = a.row_bytes;
    const ScIssue zi = {tmem_base, ptx::smem_u32(smem), ptx::smem_u32(smem_w),
                        ptx::smem_u32(&ctrl.plane_full[0]), ptx::smem_u32(&ctrl.plane_empty[0]), ptx::smem_u32(&ctrl.w_full[0]),
                        ptx::smem_u32(&ctrl.w_empty[0]), ptx::smem_u32(&ctrl.acc_full[0]), ptx::smem_u32(&ctrl.acc_empty[0]),
                        desc_hi(kHX * rb, rb), desc_hi(8 * rb, rb), a.slot_bytes, a.w_bytes, a.w_stages, a.ring,
                        (uint32_t)(rb >> 4), (uint32_t)(((3 * a.cp / 2) * rb) >> 4), (uint32_t)((kTileY * kHX * rb) >> 4),
                        (uint32_t)(a.chunk_stride >> 4), a.idesc, a.dl, cta_cols(a), &a};
    sc_issue<false, 1, 4, kPair, 1, false, true>(zi, &rs);
  } else if (warp >= 4) {
    sc_epilogue<CP, __nv_bfloat16, true, 0, kSAct>(a, ctrl, tmem_base, warp, lane);
  }

  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync_all();
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc_2sm(tmem_base, kTmemCols);
  }
}

KernFnR rm_kernel(bool relu) { return relu ? conv_scatter_rm_kernel<0> : conv_scatter_rm_kernel<2>; }

}  // namespace scatter
}  // namespace s3d
