// Confidence-weighted WLS filter of the two disparity maps (s3d_disp_wls): the fast global smoother of Min et al. (2014),
// guided by each view's own image, applied to the map weighted by its confidence and to the confidence, then divided.
// Definitions (confidence, edge weights, schedule, the line solve, output, counters) in include/s3d.h.
//
// Six launches, one per line pass, each a thread per line (a serial Thomas elimination: one reciprocal per pixel):
//   1. wls_row_kernel<FIRST>: a warp per 32 rows of one map.  The two streams are read from disp and the mask (f = c ? d : 0)
//      and run through the first horizontal pass; the edge weights are looked up once, here, and kept in the workspace, so
//      that no later pass has a dependent table load on its chain.  Rows are walked in 32-column chunks staged in shared memory, so that every
//      global load and store is a coalesced row segment (lane = column) while each lane runs the elimination of its own row
//      (lane = row).  The forward sweep writes y(f) to `out`, y(c) and g to the workspace; the backward sweep turns them
//      into u(f), u(c) in place.
//   2. wls_col_kernel: a thread per column of one map (lanes on consecutive columns: coalesced).  Steps are loaded in
//      chunks of kStep, the next chunk's loads issued before the current chunk is solved.
//   3.-5. the same row and column kernels at lam_1 and lam_2.
//   6. wls_col_kernel<LAST>: its backward sweep also writes out = u(f) / u(c) and counts.  No block spans two maps:
//      per-thread integer counters, reduced over the block, then one 64-bit atomic per counter per block.
// Every pixel is one fixed sequence of fp32 round-to-nearest operations that no launch geometry changes: the result does not
// depend on scheduling or on the batch split.  The passes keep the two streams, g and the two edge weights (20 bytes a pixel)
// in `out` and the workspace.
#include "common.cuh"

namespace s3d {
namespace {

constexpr int kRowTile = 32;                    // rows of a row-pass block (one warp) and columns of a chunk
constexpr int kColThreads = 64;                 // columns of a column-pass block
constexpr int kStep = 8;                        // rows of a column-pass chunk
constexpr int kFirstRows = 8;                   // rows whose loads the first row pass issues together
constexpr int kNumCounters = 4 + kMaxThresh;    // [n_finite, n_valid_finite, epe_fx, bad_t x 8, n_conf]

struct WlsIn {
  const float* disp;     // [2B,H,W], view-major: map m = v * B + b
  const void* left;      // guides: uint8 HWC [B,H,W,3] or fp32 NCHW [B,3,H,W]
  const void* right;
  const uint8_t* mask;   // [B,2,H,W] or NULL
  const float* lut;      // [3 * 255^2 + 1]
  int B, H, W;
};

// Colour of pixel (y, x) of the guide of map m, packed r | g << 8 | b << 16.
template <bool U8>
__device__ __forceinline__ unsigned guide_colour(const WlsIn& a, int m, int y, int x) {
  const int b = m % a.B, v = m / a.B;
  const int64_t HW = (int64_t)a.H * a.W, pix = (int64_t)y * a.W + x;
  if (U8) {
    const uint8_t* p = static_cast<const uint8_t*>(v ? a.right : a.left) + ((int64_t)b * HW + pix) * 3;
    return (unsigned)__ldg(p) | (unsigned)__ldg(p + 1) << 8 | (unsigned)__ldg(p + 2) << 16;
  }
  const float* p = static_cast<const float*>(v ? a.right : a.left) + (int64_t)b * 3 * HW + pix;
  return colour_f32(__ldg(p)) | colour_f32(__ldg(p + HW)) << 8 | colour_f32(__ldg(p + 2 * HW)) << 16;
}

// lut[s], s = the sum over the channels of the squared 8-bit colour differences (an exact integer in [0, 3 * 255^2]).
__device__ __forceinline__ float edge_weight(const float* lut, unsigned c0, unsigned c1) {
  int s = 0;
#pragma unroll
  for (int ch = 0; ch < 3; ++ch) {
    const int d = (int)((c0 >> (8 * ch)) & 0xffu) - (int)((c1 >> (8 * ch)) & 0xffu);
    s += d * d;
  }
  return __ldg(lut + s);
}

// The confidence of disp value d with mask value mk (1 without a mask).
__device__ __forceinline__ bool confident(float d, unsigned mk) { return isfinite(d) && mk == 1u; }

// One forward step of the elimination (include/s3d.h): kl = k_{i-1} and g, yf, yc of pixel i-1 in, those of pixel i out.
struct Sweep {
  float kl = 0.f, g = 0.f, yf = 0.f, yc = 0.f;
  __device__ __forceinline__ void step(float kr, float f, float c) {
    const float den = __fsub_rn(__fadd_rn(__fadd_rn(1.f, kl), kr), __fmul_rn(kl, g));
    const float r = __frcp_rn(den);                                      // == __fdiv_rn(1, den): both correctly rounded
    g = __fmul_rn(kr, r);
    yf = __fmul_rn(__fadd_rn(f, __fmul_rn(kl, yf)), r);
    yc = __fmul_rn(__fadd_rn(c, __fmul_rn(kl, yc)), r);
    kl = kr;
  }
};

// u_i = y_i + g_i u_{i+1}; the last pixel of a line keeps u = y.
__device__ __forceinline__ float back(float y, float g, float un, bool last) { return last ? y : __fadd_rn(y, __fmul_rn(g, un)); }

// FIRST: the streams come from disp and the mask, and the edge weights from the guide; they are kept in WH (edge to the
// right neighbour, 0 in the last column) and WV (edge to the neighbour below, 0 in the last row) for the later passes.
template <bool U8, bool FIRST>
__global__ void __launch_bounds__(kRowTile)
wls_row_kernel(WlsIn a, float lam, float* __restrict__ F, float* __restrict__ C, float* __restrict__ G,
               float* __restrict__ WH, float* __restrict__ WV) {
  __shared__ float sf[kRowTile][kRowTile + 1], sc[kRowTile][kRowTile + 1], sg[kRowTile][kRowTile + 1];
  const int m = blockIdx.y, y0 = blockIdx.x * kRowTile, lane = threadIdx.x;
  const int H = a.H, W = a.W;
  const int64_t HW = (int64_t)H * W, base = (int64_t)m * HW;
  const uint8_t* mk = FIRST && a.mask ? a.mask + ((int64_t)(m % a.B) * 2 + m / a.B) * HW : nullptr;
  const int rows = min(kRowTile, H - y0);
  Sweep s;                                                              // lane = row y0 + lane
  for (int x0 = 0; x0 < W; x0 += kRowTile) {
    const int x = x0 + lane, xc = min(x, W - 1);
    // the loads of a group of rows are all issued before any is used: clamped addresses, no branch between them
    if (FIRST) {
#pragma unroll 1
      for (int j0 = 0; j0 < kRowTile; j0 += kFirstRows) {
        float d[kFirstRows];
        unsigned col[kFirstRows], below[kFirstRows], right[kFirstRows], mv[kFirstRows];
#pragma unroll
        for (int jj = 0; jj < kFirstRows; ++jj) {
          const int y = y0 + min(j0 + jj, rows - 1);
          const int64_t p = (int64_t)y * W + xc;
          d[jj] = __ldg(a.disp + base + p);
          mv[jj] = mk ? (unsigned)__ldg(mk + p) : 1u;
          col[jj] = guide_colour<U8>(a, m, y, xc);
          below[jj] = guide_colour<U8>(a, m, min(y + 1, H - 1), xc);
          right[jj] = guide_colour<U8>(a, m, y, min(x + 1, W - 1));
        }
#pragma unroll
        for (int jj = 0; jj < kFirstRows; ++jj) {
          const int j = j0 + jj;
          const bool in = j < rows && x < W, cf = in && confident(d[jj], mv[jj]);
          const float wh = x + 1 < W ? edge_weight(a.lut, col[jj], right[jj]) : 0.f;
          const float wv = y0 + j + 1 < H ? edge_weight(a.lut, col[jj], below[jj]) : 0.f;
          if (in) {
            const int64_t p = base + (int64_t)(y0 + j) * W + x;
            WH[p] = wh;
            WV[p] = wv;
          }
          sf[j][lane] = cf ? d[jj] : 0.f;
          sc[j][lane] = cf ? 1.f : 0.f;
          sg[j][lane] = __fmul_rn(lam, in ? wh : 0.f);
        }
      }
    } else {
      float rf[kRowTile], rc[kRowTile], rw[kRowTile];
#pragma unroll
      for (int j = 0; j < kRowTile; ++j) {
        const int64_t p = base + (int64_t)(y0 + min(j, rows - 1)) * W + xc;
        rf[j] = F[p];
        rc[j] = C[p];
        rw[j] = WH[p];
      }
#pragma unroll
      for (int j = 0; j < kRowTile; ++j) {
        const bool in = j < rows && x < W;
        sf[j][lane] = in ? rf[j] : 0.f;
        sc[j][lane] = in ? rc[j] : 0.f;
        sg[j][lane] = __fmul_rn(lam, in ? rw[j] : 0.f);
      }
    }
    __syncwarp();
    const int n = min(kRowTile, W - x0);
    if (lane < rows) {
      for (int i = 0; i < n; ++i) {                                     // lane = row: the elimination
        s.step(sg[lane][i], sf[lane][i], sc[lane][i]);
        sf[lane][i] = s.yf;
        sc[lane][i] = s.yc;
        sg[lane][i] = s.g;
      }
    }
    __syncwarp();
    if (x < W) {
#pragma unroll
      for (int j = 0; j < kRowTile; ++j) {
        if (j >= rows) break;
        const int64_t p = base + (int64_t)(y0 + j) * W + x;
        F[p] = sf[j][lane];
        C[p] = sc[j][lane];
        G[p] = sg[j][lane];
      }
    }
    __syncwarp();
  }
  float uf = 0.f, uc = 0.f;
  for (int x0 = (W - 1) / kRowTile * kRowTile; x0 >= 0; x0 -= kRowTile) {
    const int x = x0 + lane, xc = min(x, W - 1);
    float rf[kRowTile], rc[kRowTile], rg[kRowTile];
#pragma unroll
    for (int j = 0; j < kRowTile; ++j) {                                // clamped: all loads in flight at once
      const int64_t p = base + (int64_t)(y0 + min(j, rows - 1)) * W + xc;
      rf[j] = F[p];
      rc[j] = C[p];
      rg[j] = G[p];
    }
#pragma unroll
    for (int j = 0; j < kRowTile; ++j) {
      sf[j][lane] = rf[j];
      sc[j][lane] = rc[j];
      sg[j][lane] = rg[j];
    }
    __syncwarp();
    const int n = min(kRowTile, W - x0);
    if (lane < rows) {
      for (int i = n - 1; i >= 0; --i) {
        const bool last = x0 + i == W - 1;
        uf = back(sf[lane][i], sg[lane][i], uf, last);
        uc = back(sc[lane][i], sg[lane][i], uc, last);
        sf[lane][i] = uf;
        sc[lane][i] = uc;
      }
    }
    __syncwarp();
    if (x < W) {
#pragma unroll
      for (int j = 0; j < kRowTile; ++j) {
        if (j >= rows) break;
        const int64_t p = base + (int64_t)(y0 + j) * W + x;
        F[p] = sf[j][lane];
        C[p] = sc[j][lane];
      }
    }
    __syncwarp();
  }
}

struct WlsEval {
  const float* gt;       // [B,2,H,W] or NULL
  Thresh th;
  int nT;
  float max_gt;
  unsigned long long* stats;
};

template <bool LAST>
__global__ void __launch_bounds__(kColThreads)
wls_col_kernel(WlsIn a, float lam, float* __restrict__ F, float* __restrict__ C, float* __restrict__ G,
               const float* __restrict__ WV, WlsEval e) {
  const int m = blockIdx.y, x = blockIdx.x * kColThreads + threadIdx.x;
  const int H = a.H, W = a.W;
  const int64_t HW = (int64_t)H * W, base = (int64_t)m * HW;
  const bool live = x < W;
  const int xc = live ? x : W - 1;                  // dead lanes shadow the last column and store nothing
  // forward sweep, chunks of kStep rows; the next chunk's loads are issued before the current one is solved
  float f[kStep], c[kStep], w[kStep];
  auto load_fwd = [&](int y0, float* ff, float* cc, float* ww) {
#pragma unroll
    for (int j = 0; j < kStep; ++j) {
      const int64_t p = base + (int64_t)min(y0 + j, H - 1) * W + xc;
      ff[j] = F[p];
      cc[j] = C[p];
      ww[j] = WV[p];                                                    // 0 in the last row
    }
  };
  Sweep s;
  load_fwd(0, f, c, w);
  for (int y0 = 0; y0 < H; y0 += kStep) {
    float fn[kStep], cn[kStep], wn[kStep];
    if (y0 + kStep < H) load_fwd(y0 + kStep, fn, cn, wn);
#pragma unroll
    for (int j = 0; j < kStep; ++j) {
      const int y = y0 + j;
      if (y >= H) break;
      s.step(__fmul_rn(lam, w[j]), f[j], c[j]);
      if (live) {
        const int64_t p = base + (int64_t)y * W + x;
        F[p] = s.yf;
        C[p] = s.yc;
        G[p] = s.g;
      }
    }
#pragma unroll
    for (int j = 0; j < kStep; ++j) { f[j] = fn[j];  c[j] = cn[j];  w[j] = wn[j]; }
  }
  // backward sweep, chunks of kStep rows from the bottom
  float g[kStep], d[kStep], gtv[kStep];
  unsigned mk[kStep];
  const int64_t img = ((int64_t)(m % a.B) * 2 + m / a.B) * HW;
  auto load_bwd = [&](int y1, float* ff, float* cc, float* gg, float* dd, float* tt, unsigned* mm) {
#pragma unroll
    for (int j = 0; j < kStep; ++j) {                                   // rows y1 - j, clamped at 0
      const int64_t p = (int64_t)max(y1 - j, 0) * W + xc;
      ff[j] = F[base + p];
      cc[j] = C[base + p];
      gg[j] = G[base + p];
      if (LAST) {
        dd[j] = __ldg(a.disp + base + p);
        mm[j] = a.mask ? (unsigned)__ldg(a.mask + img + p) : 1u;
        tt[j] = e.gt ? __ldg(e.gt + img + p) : 0.f;
      }
    }
  };
  unsigned n_fin = 0, n_valid = 0, n_conf = 0, bad[kMaxThresh] = {};
  unsigned long long epe = 0;
  float uf = 0.f, uc = 0.f;
  load_bwd(H - 1, f, c, g, d, gtv, mk);
  for (int y1 = H - 1; y1 >= 0; y1 -= kStep) {
    float fn[kStep], cn[kStep], gn[kStep], dn[kStep], tn[kStep];
    unsigned mn[kStep];
    if (y1 - kStep >= 0) load_bwd(y1 - kStep, fn, cn, gn, dn, tn, mn);
#pragma unroll
    for (int j = 0; j < kStep; ++j) {
      const int y = y1 - j;
      if (y < 0) break;
      uf = back(f[j], g[j], uf, y == H - 1);
      uc = back(c[j], g[j], uc, y == H - 1);
      if (!live) continue;
      const int64_t p = base + (int64_t)y * W + x;
      if (!LAST) {
        F[p] = uf;
        C[p] = uc;
        continue;
      }
      const float o = uc > 0.f ? __fdiv_rn(uf, uc) : __int_as_float(0x7fffffff);
      F[p] = o;
      n_conf += confident(d[j], mk[j]);
      if (!isfinite(o)) continue;
      ++n_fin;
      const float t = gtv[j];
      if (!e.gt || !(isfinite(t) && t >= 0.f && t < e.max_gt)) continue;
      const float err = fabsf(__fsub_rn(o, t));
      ++n_valid;
      epe += (unsigned long long)__float2ll_rn(err * 65536.f);     // exact scaling by 2^16, then round half to even
#pragma unroll
      for (int q = 0; q < kMaxThresh; ++q)
        if (q < e.nT) bad[q] += err > e.th.t[q];
    }
#pragma unroll
    for (int j = 0; j < kStep; ++j) {
      f[j] = fn[j];  c[j] = cn[j];  g[j] = gn[j];
      if (LAST) { d[j] = dn[j];  gtv[j] = tn[j];  mk[j] = mn[j]; }
    }
  }
  if (!LAST) return;
  __shared__ unsigned long long blk[kNumCounters];
  if (threadIdx.x < kNumCounters) blk[threadIdx.x] = 0;
  __syncthreads();
  unsigned long long cnt[kNumCounters];
  cnt[0] = n_fin;  cnt[1] = n_valid;  cnt[2] = epe;
#pragma unroll
  for (int q = 0; q < kMaxThresh; ++q) cnt[3 + q] = bad[q];
  cnt[3 + kMaxThresh] = n_conf;
#pragma unroll
  for (int k = 0; k < kNumCounters; ++k) {
    if (k >= 3 + e.nT && k < 3 + kMaxThresh) continue;
    unsigned long long v = cnt[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(&blk[k], v);
  }
  __syncthreads();
  // counter k -> column k of the row [n_finite, n_valid_finite, epe_fx, bad_t x nT, n_conf]
  const int k = threadIdx.x;
  if (k < kNumCounters && blk[k] && (k < 3 + e.nT || k == 3 + kMaxThresh)) {
    const int cl = k < 3 + e.nT ? k : 3 + e.nT;
    atomicAdd(e.stats + img / HW * (4 + e.nT) + cl, blk[k]);
  }
}

bool aligned(const void* p, int n) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) % n) == 0; }

void launch_passes(const WlsIn& in, bool u8, const float lam[3], float* F, float* ws, const WlsEval& ev, cudaStream_t st) {
  const unsigned maps = 2u * (unsigned)in.B;
  const int64_t n = (int64_t)2 * in.B * in.H * in.W;
  float *C = ws, *G = ws + n, *WH = ws + 2 * n, *WV = ws + 3 * n;
  const dim3 rg((unsigned)ceil_div(in.H, kRowTile), maps), cg((unsigned)ceil_div(in.W, kColThreads), maps);
  const WlsEval none{nullptr, {}, 0, 0.f, nullptr};
  if (u8) wls_row_kernel<true, true><<<rg, kRowTile, 0, st>>>(in, lam[0], F, C, G, WH, WV);
  else    wls_row_kernel<false, true><<<rg, kRowTile, 0, st>>>(in, lam[0], F, C, G, WH, WV);
  wls_col_kernel<false><<<cg, kColThreads, 0, st>>>(in, lam[0], F, C, G, WV, none);
  wls_row_kernel<true, false><<<rg, kRowTile, 0, st>>>(in, lam[1], F, C, G, WH, WV);
  wls_col_kernel<false><<<cg, kColThreads, 0, st>>>(in, lam[1], F, C, G, WV, none);
  wls_row_kernel<true, false><<<rg, kRowTile, 0, st>>>(in, lam[2], F, C, G, WH, WV);
  wls_col_kernel<true><<<cg, kColThreads, 0, st>>>(in, lam[2], F, C, G, WV, ev);
}

}  // namespace
}  // namespace s3d

using namespace s3d;

extern "C" int64_t s3d_disp_wls_workspace_bytes(int B, int H, int W) {
  if (B < 0 || H < 0 || W < 0) return 0;
  return (int64_t)2 * B * H * (int64_t)W * 4 * (int64_t)sizeof(float);     // U(c), g and the two edge weights, fp32 each
}

extern "C" int s3d_disp_wls(const float* disp, int B, int H, int W, const void* left, const void* right, int img_u8,
                            const uint8_t* mask, const float* lut, float lambda, const float* gt, const float* thresholds,
                            int T, float max_gt, float* out, long long* stats, void* workspace, int64_t workspace_bytes,
                            void* stream) {
  if (!disp || !left || !right || !lut || !out || !stats || (T > 0 && !thresholds)) {
    set_error("disp_wls: null argument");
    return S3D_ERR_INVALID;
  }
  S3D_CHECK_ARG(B >= 0 && 2 * (int64_t)B < 65536 && H >= 1 && W >= 1,
                "disp_wls: need 0 <= B < 32768, H >= 1, W >= 1, got %d %d %d", B, H, W);
  S3D_CHECK_ARG((int64_t)H * W < (1ll << 31), "disp_wls: H W must be < 2^31, got H = %d, W = %d", H, W);
  S3D_CHECK_ARG(img_u8 == 0 || img_u8 == 1, "disp_wls: img_u8 must be 0 or 1, got %d", img_u8);
  S3D_CHECK_ARG(isfinite(lambda) && lambda > 0.f, "disp_wls: lambda must be finite and > 0, got %g", (double)lambda);
  S3D_CHECK_ARG(T >= 0 && T <= kMaxThresh, "disp_wls: T must be in [0, 8], got %d", T);
  S3D_CHECK_ARG(!gt || max_gt > 0.f, "disp_wls: max_gt must be > 0 with gt");
  S3D_CHECK_ARG(out != disp, "disp_wls: out must not be disp");
  const int64_t need = s3d_disp_wls_workspace_bytes(B, H, W);
  S3D_CHECK_ARG(workspace_bytes >= need && (need == 0 || workspace),
                "disp_wls: workspace of %lld bytes, need %lld", (long long)workspace_bytes, (long long)need);
  S3D_CHECK_ARG(aligned(workspace, 4), "disp_wls: workspace must be 4-byte aligned");
  if (B == 0) return S3D_OK;
  WlsEval ev{gt, {}, T, max_gt, reinterpret_cast<unsigned long long*>(stats)};
  for (int t = 0; t < kMaxThresh; ++t) ev.th.t[t] = gt && t < T ? thresholds[t] : 0.f;
  float lam[3];
  for (int t = 0; t < 3; ++t) lam[t] = (float)((double)lambda * pow(0.25, t));
  const WlsIn in{disp, left, right, mask, lut, B, H, W};
  launch_passes(in, img_u8 == 1, lam, out, static_cast<float*>(workspace), ev, static_cast<cudaStream_t>(stream));
  S3D_LAUNCH_CHECK();
  return S3D_OK;
}
