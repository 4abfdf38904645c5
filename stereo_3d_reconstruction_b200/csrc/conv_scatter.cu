// Host side of the plane-scatter kernel (see conv_scatter.cuh for the design) + its all-in-one instantiations.
#include "conv_scatter.cuh"

namespace s3d {
using namespace scatter;

// stride-1 3x3x3, pad 1, canonical tap order, Cout <= 64, one K chunk per row, channels-last output, host-packed
// rotations present.
bool conv_scatter_eligible(const S3dConvParams* p) {
  const int esz = p->in_dtype == S3D_DTYPE_F32 ? 4 : 2;
  const bool split = p->in_dtype == S3D_DTYPE_BF16X2;
  if (!p->w_nstack || knobs().no_scatter) return false;
  // split operands: [hi | lo] rows of 64 / 128 / 256 bytes, split output, transposed stores (Cout a power of two)
  if (split && (p->out_dtype != S3D_DTYPE_BF16X2 || p->Cin > 64 || (p->Cout != 16 && p->Cout != 32 && p->Cout != 64) ||
                p->cout_store != p->Cout)) return false;
  if (!split && p->out_dtype == S3D_DTYPE_BF16X2) return false;
  if (p->n_classes != 1 || p->sx != 1 || p->sy != 1 || p->sz != 1 || p->ntaps != 27) return false;
  if (p->omx != 1 || p->omy != 1 || p->omz != 1 || p->osC != 1 || p->proj_w) return false;
  if (p->oD != p->iD || p->oH != p->iH || p->oW != p->iW) return false;
  for (int t = 0; t < 27; ++t)
    if (p->dz[t] != t / 9 - 1 || p->dy[t] != (t % 9) / 3 - 1 || p->dx[t] != t % 3 - 1) return false;
  const int cin_bytes = (split ? 2 : 1) * p->Cin * esz;
  if (split && cin_bytes == 32) return false;
  if (cin_bytes != 32 && cin_bytes != 64 && cin_bytes != 128 && cin_bytes != 256) return false;
  if (p->Cout > 64 || p->Cout % 16 != 0) return false;
  return true;
}

int conv_scatter_launch(const S3dConvParams* p_in, const void* in, const float* bias, const void* residual, void* out,
                        cudaStream_t stream) {
  const S3dConvParams& p = *p_in;
  const bool tf32 = p.in_dtype == S3D_DTYPE_F32;
  const bool split = p.in_dtype == S3D_DTYPE_BF16X2;
  const int esz = tf32 ? 4 : 2;
  const int cin_phys = split ? 2 * p.Cin : p.Cin;            // channels of a physical pixel row ([hi | lo] when split)
  S3D_CHECK_ARG(p.cout_store >= 1 && p.cout_store <= p.Cout, "scatter: cout_store");
  ScArgs a;
  memset(&a, 0, sizeof(a));
  a.p = p;  a.bias = bias;  a.residual = residual;  a.out = out;
  a.split = split ? 1 : 0;
  a.os_lo = p.os_lo ? p.os_lo : (int64_t)p.Cout;
  a.nchunks = cin_phys * esz == 256 ? 2 : 1;
  a.row_bytes = cin_phys * esz / a.nchunks;
  a.kc = cin_phys / a.nchunks;
  a.chunk_stride = (kPlaneRows * a.row_bytes + 1023) / 1024 * 1024;
  a.slot_bytes = a.nchunks * a.chunk_stride;
  a.cp = p.Cout;
  a.tps = spec_tps(a.row_bytes, a.cp);
  if (knobs().scatter_tps3 && a.tps == 9) a.tps = 3;
  a.cols_x = ceil_div(p.oW, kTX);  a.cols_y = ceil_div(p.oH, kTY);
  int64_t total = (int64_t)p.N * a.cols_x * a.cols_y;
  S3D_CHECK_ARG(total > 0 && total < (1ll << 31), "scatter: column count out of range");
  // z-split for small batches (conv_scatter.cuh, ScArgs::nz): as many chunks as fill the chip in ONE wave, each at least 4
  // output planes deep (a chunk marches over 2 extra planes)
  a.nz = 1;  a.zc = p.oD;  a.dl = p.oD;
  {
    const int sms = num_sms();
    int nz = knobs().scatter_zsplit > 0 ? knobs().scatter_zsplit : (knobs().scatter_zsplit < 0 ? 1 : (int)(sms / total));
    if (nz > p.oD / 4) nz = p.oD / 4;
    if (nz > 1) {
      a.zc = ceil_div(p.oD, nz);
      a.nz = ceil_div(p.oD, a.zc);
      a.dl = a.zc + 2;
      if (a.nz > 1) total *= a.nz; else { a.nz = 1; a.zc = p.oD; a.dl = p.oD; }
    }
  }
  a.total_cols = (int)total;
  // CTA pairs (cta_group::2): the two SMs of a TPC run one M = 256 MMA, each on its own 128 pixels, and each keeps only
  // HALF of the weight rows in shared memory.  That halves the B-operand reads and the weight TMA writes per SM -- the
  // single-CTA kernel saturates the shared-memory pipe (A 4 KB + B 6 KB per 96-cycle MMA, plus the TMA fills).
  int grid = num_sms();
  a.pair = ((3 * a.cp / 2) % 8 == 0 && total >= 2 && grid >= 2 && !knobs().scatter_no_pair) ? 1 : 0;
  // coalesced (transposed) store path: needed by every lean kernel
  bool fast_ok;
  {
    const int oesz = p.out_dtype == S3D_DTYPE_F32 ? 4 : 2;
    const bool simple_act = p.act == S3D_ACT_NONE || p.act == S3D_ACT_RELU || p.act == S3D_ACT_LEAKY;
    auto aligned = [&](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
    auto dense16 = [&](int64_t st) { return (st * oesz) % 16 == 0; };
    fast_ok = simple_act && bias != nullptr && p.cout_store == p.Cout && aligned(out) && aligned(residual) &&
              dense16(p.osW) && dense16(p.osH) && dense16(p.osD) && dense16(p.osN) && p.osW < (1ll << 24) &&
              (split || !knobs().scatter_no_transpose);
  }
  // narrow lean shapes: two CTAs per SM (conv_scatter.cuh, kTwo) when there is work for both
  const bool two = fast_ok && a.pair && !tf32 && !split && a.nchunks == 1 && p.out_dtype == S3D_DTYPE_BF16 && residual == nullptr &&
                   spec_kernel(a.row_bytes, a.cp, false, p.act == S3D_ACT_RELU, true) != nullptr && total > grid &&
                   !knobs().scatter_generic && !knobs().scatter_one_cta && !knobs().scatter_tps3 && !knobs().scatter_ring;
  if (two) grid *= 2;
  if (a.pair) {
    if ((int64_t)grid > total) grid = (int)((total + 1) / 2 * 2);
    grid -= grid % 2;
    a.ncols_max = (int)((total + grid - 1) / grid);
  } else if ((int64_t)grid > total) grid = (int)total;
  // constant-region skip (include/s3d.h dz_nref; conv_scatter.cuh, Item): bf16 operands and whole columns only -- a z-split
  // chunk marches its own few planes, so the skip is off there.  The schedule table replaces the round-robin column order
  // of CTA pairs and sets the grid; single CTAs skip on their own columns without it.
  const bool dz = p.dz_nref > 0 && !tf32 && !split && a.nz == 1 && !knobs().no_dz_skip;
  if (dz) S3D_CHECK_ARG(p.N == 2 * p.dz_nref && p.dz_c >= 0 && p.dz_e >= 0, "scatter: constant-region descriptor");
  if (!dz) a.p.dz_nref = 0;
  if (!dz || !a.pair) a.p.dz_sched = nullptr;
  if (a.p.dz_sched) {
    S3D_CHECK_ARG(p.dz_pairs >= 1, "scatter: dz_pairs");
    grid = 2 * p.dz_pairs;
  }
  const int w_rows = a.pair ? 3 * a.cp / 2 : 3 * a.cp;          // weight rows staged per CTA
  a.w_tx = a.tps * w_rows * a.row_bytes;
  a.w_bytes = (a.w_tx + 1023) / 1024 * 1024;
  const int budget = two ? 110 * 1024 : 227 * 1024 - 1024 - 512;   // dynamic shared memory minus alignment slack and ScCtrl
  // big planes: 2 slots and the rest for weight stages (weight latency is what stalls); small planes: a deeper ring
  // (a plane is then consumed faster than its TMA round trip), keeping at least 4 weight stages
  int ring = (budget - 4 * a.w_bytes) / a.slot_bytes;
  if (ring > kMaxRing) ring = kMaxRing;
  if (ring < 2) ring = 2;
  if (a.row_bytes == 128 && ring > (a.pair && a.nchunks == 1 ? 3 : 2)) ring = a.pair && a.nchunks == 1 ? 3 : 2;
  if (const int r = knobs().scatter_ring) { if (r >= 2 && r <= kMaxRing) ring = r; }
  a.ring = ring;
  a.w_stages = (budget - a.ring * a.slot_bytes) / a.w_bytes;
  if (a.w_stages > kMaxW) a.w_stages = kMaxW;
  S3D_CHECK_ARG(a.w_stages >= 2, "scatter: not enough shared memory for the weight ring");   // 2 works (no prefetch), >= 3 is the norm
  a.idesc = ptx::make_instr_desc(tf32 ? 2 : 1, a.pair ? 256 : 128, 3 * a.cp);
  // residual: each thread reads its own pixel's 128 bytes directly (measured 2.58 vs 2.71 ms on the residual layer against
  // coalesced group loads + a second shuffle transpose -- with CTA pairs the L1 data pipe has room for the scattered reads;
  // staging the residual tiles in shared memory by TMA was tried too: 2.66 vs 2.55 ms, it costs three weight stages)
  a.res_direct = !knobs().scatter_res_transpose;
  {
    auto dense16 = [&](int64_t st) { return (st * 2) % 16 == 0; };
    a.fast_store = fast_ok;
    if (split) {
      S3D_CHECK_ARG(a.fast_store && dense16(a.os_lo) && a.os_lo >= p.Cout,
                    "scatter (split operands): needs a bias, a none / ReLU / LeakyReLU activation and 16-byte aligned out / residual / strides");
      a.res_direct = 1;
    }
  }

  const CUtensorMapSwizzle sw = a.row_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                              : a.row_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B;
  CUtensorMap map_x, map_w;
  cuuint32_t box[5] = {(cuuint32_t)a.kc, kHX, kHY, 1, 1};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  int rc = encode_act_map(&map_x, in, esz, tf32, cin_phys, p.iW, p.iH, p.iD, p.N, box, estr, sw);
  if (rc != S3D_OK) return rc;
  rc = encode_weight_map(&map_w, p.w_nstack, esz, tf32, cin_phys, 3 * a.cp, 36, a.kc, w_rows, sw, a.tps);
  if (rc != S3D_OK) return rc;

  // the 64 -> 64 bf16 residual layers: residual staged by TMA and added as an identity tap on the tensor core
  // (conv_scatter_rm.cu); the residual must be a dense channels-last tensor of the output's shape
  const bool rm = residual != nullptr && a.pair && !tf32 && !split && a.nchunks == 1 && a.row_bytes == 128 && a.cp == 64 &&
                  p.out_dtype == S3D_DTYPE_BF16 && a.fast_store && a.tps == 1 && (p.act == S3D_ACT_RELU || p.act == S3D_ACT_NONE) &&
                  p.osW == 64 && p.osH == (int64_t)p.oW * 64 && p.osD == (int64_t)p.oH * p.osH && p.osN == (int64_t)p.oD * p.osD &&
                  !knobs().scatter_no_rm && !knobs().scatter_generic;
  if (rm) {
    const int extra = kResBytes + 32 * 128;
    a.w_stages = (budget - a.ring * a.slot_bytes - extra) / a.w_bytes;
    if (a.w_stages > kMaxW) a.w_stages = kMaxW;
    S3D_CHECK_ARG(a.w_stages >= 3, "scatter: not enough shared memory for the residual stage");
    CUtensorMap map_r;
    cuuint32_t rbox[5] = {64, kTX, kTY, 1, 1};
    rc = encode_act_map(&map_r, residual, 2, false, 64, p.oW, p.oH, p.oD, p.N, rbox, estr, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc != S3D_OK) return rc;
    a.residual = nullptr;                                     // the epilogue is the plain one
    const int smem_rm = a.ring * a.slot_bytes + a.w_stages * a.w_bytes + extra + 1024;
    KernFnR kr = rm_kernel(p.act == S3D_ACT_RELU);
    S3D_CUDA(cudaFuncSetAttribute(kr, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_rm));
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(grid);  cfg.blockDim = dim3(kThreads);  cfg.dynamicSmemBytes = smem_rm;  cfg.stream = stream;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeClusterDimension;
    attr.val.clusterDim.x = 2;  attr.val.clusterDim.y = 1;  attr.val.clusterDim.z = 1;
    cfg.attrs = &attr;  cfg.numAttrs = 1;
    S3D_CUDA(cudaLaunchKernelEx(&cfg, kr, map_x, map_w, map_r, a));
    S3D_LAUNCH_CHECK();
    return S3D_OK;
  }

  const int smem_bytes = a.ring * a.slot_bytes + a.w_stages * a.w_bytes + 1024;
  KernFn kern = a.pair ? (tf32 ? conv_scatter_kernel<true, true> : conv_scatter_kernel<false, true>)
                       : (tf32 ? conv_scatter_kernel<true, false> : conv_scatter_kernel<false, false>);
  if (split) {
    const bool lean = a.pair && a.tps == spec_tps(a.row_bytes, a.cp) && !knobs().scatter_generic;
    kern = split_kernel(lean, a.pair != 0, cin_phys * esz, a.cp, residual != nullptr, p.act == S3D_ACT_RELU);
  }
  // the network's own layer shapes (bf16, CTA pairs, coalesced epilogue) each have a lean kernel
  else if (a.pair && !tf32 && a.nchunks == 1 && p.out_dtype == S3D_DTYPE_BF16 && a.fast_store && a.tps == spec_tps(a.row_bytes, a.cp) &&
      !knobs().scatter_generic) {
    const bool relu = p.act == S3D_ACT_RELU;        // anything else: slope formula
    if (KernFn k = spec_kernel(a.row_bytes, a.cp, residual != nullptr, relu, two && a.fast_store)) kern = k;
    else if (two) { set_error("scatter: the two-CTA kernel needs the coalesced store path"); return S3D_ERR_INVALID; }
  }
  S3D_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
  if (a.pair) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(grid);  cfg.blockDim = dim3(kThreads);  cfg.dynamicSmemBytes = smem_bytes;  cfg.stream = stream;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeClusterDimension;
    attr.val.clusterDim.x = 2;  attr.val.clusterDim.y = 1;  attr.val.clusterDim.z = 1;
    cfg.attrs = &attr;  cfg.numAttrs = 1;
    S3D_CUDA(cudaLaunchKernelEx(&cfg, kern, map_x, map_w, a));
  } else {
    kern<<<grid, kThreads, smem_bytes, stream>>>(map_x, map_w, a);
  }
  S3D_LAUNCH_CHECK();
  return S3D_OK;
}

}  // namespace s3d
