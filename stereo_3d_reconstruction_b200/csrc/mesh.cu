// Triangle mesh of an occupancy grid (s3d_voxel_mesh): marching cubes at iso-level t over the zero-padded, clamped field,
// with the generated case table of mc_table.cuh.  Definitions (vertex ids, coordinates, face order) in include/s3d.h.
//
// One block per sample, four phases separated by block barriers:
//   1. the inside mask of every grid row (k, j) is bit-packed into shared memory (one uint64 per row, bit i; a warp per row,
//      coalesced loads and a ballot).  Padding rows are 0.
//   2. per lattice row (k, j), k, j in -1..n-1 (a warp per row): the crossing edges of the row along x, y and z are three
//      masks of xors of neighbouring rows, so the row's vertex count is a sum of popcounts; its face count is the sum of
//      the table's triangle counts over the row's n+1 cells.  Rows with k = n or j = n hold neither.
//   3. block-wide exclusive scan of both counts over the (n+1)^2 rows: each row's first vertex id and first face.
//   4. per row again (a warp per row, lanes along i): a warp scan places each lane's vertices and faces.  A vertex reads the
//      two field values of its edge from global memory (L2-resident); a face's vertex id is its row's first id plus the
//      popcounts of the row's crossing masks below it.
// Positions come from scans only, no atomics: the output is deterministic.
#include "common.cuh"
#include "mc_table.cuh"

namespace s3d {
namespace {

constexpr int kMeshThreads = 1024;
constexpr int kMeshWarps = kMeshThreads / 32;
constexpr int kMeshMaxN = 64;

struct MeshSmem {
  const unsigned long long* m;   // [n][n] inside masks of the grid rows
  int n;
  __device__ __forceinline__ unsigned long long row(int k, int j) const {
    return (k >= 0 && k < n && j >= 0 && j < n) ? m[k * n + j] : 0ull;
  }
};

// crossing masks of lattice row (k, j): bit i of x / y / z = the edge from (k, j, i) along that axis crosses (i in 0..n-1);
// x1 = the x edge from i = -1 (padding) to i = 0
struct RowCross {
  unsigned long long x, y, z;
  int x1;
};

__device__ __forceinline__ RowCross row_cross(const MeshSmem& s, int k, int j) {
  const unsigned long long c = s.row(k, j);
  RowCross r;
  r.x = c ^ (c >> 1);
  r.y = c ^ s.row(k, j + 1);
  r.z = c ^ s.row(k + 1, j);
  r.x1 = (int)(c & 1);
  return r;
}

__device__ __forceinline__ unsigned long long below(int i) { return i <= 0 ? 0ull : (~0ull >> (64 - i)); }

__device__ __forceinline__ int bit(unsigned long long w, int i) { return (i >= 0 && i < 64) ? (int)((w >> i) & 1) : 0; }

// inside bits of the cell with lower corner (k, j, i): case = sum inside(c) << c, c = cx | cy << 1 | cz << 2
__device__ __forceinline__ int cell_case(unsigned long long r00, unsigned long long r10, unsigned long long r01,
                                         unsigned long long r11, int i) {
  // r<dy><dz>: rows (k + dz, j + dy); bits past the grid (i = -1, i + 1 = n) are 0 since the masks hold n bits
  return bit(r00, i) | bit(r00, i + 1) << 1 | bit(r10, i) << 2 | bit(r10, i + 1) << 3 |
         bit(r01, i) << 4 | bit(r01, i + 1) << 5 | bit(r11, i) << 6 | bit(r11, i + 1) << 7;
}

__device__ __forceinline__ float clamp01(float v) { return fminf(fmaxf(v, 0.f), 1.f); }   // NaN -> 0 (fmaxf)

__device__ __forceinline__ int warp_incl_scan(int v) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int u = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += u;
  }
  return v;
}

__global__ void __launch_bounds__(kMeshThreads)
voxel_mesh_kernel(const float* __restrict__ vol, int n, float t, float* __restrict__ verts, int max_verts,
                  int* __restrict__ faces, int max_faces, int* __restrict__ counts) {
  extern __shared__ unsigned long long mesh_smem[];
  const int b = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nn = n * n, n1 = n + 1, R = n1 * n1;
  unsigned long long* masks = mesh_smem;                                   // [n * n]
  int* vbase = reinterpret_cast<int*>(masks + nn);                         // [R] vertex count, then first id
  int* fbase = vbase + R;                                                  // [R] face count, then first face
  uint8_t* tcnt = reinterpret_cast<uint8_t*>(fbase + R);                   // [256]
  uint8_t* tedg = tcnt + 256;                                              // [256][15]
  __shared__ int wsum[2][kMeshWarps];
  __shared__ int total[2];
  const float* v = vol + (int64_t)b * nn * n;
  const MeshSmem S{masks, n};

  for (int e = threadIdx.x; e < 256; e += blockDim.x) tcnt[e] = kMcTriCount[e];
  for (int e = threadIdx.x; e < 256 * 3 * kMcMaxTri; e += blockDim.x) tedg[e] = (&kMcTriEdges[0][0])[e];
  // 1. inside masks
  for (int r = warp; r < nn; r += kMeshWarps) {
    const float* row = v + (int64_t)r * n;
    const bool in0 = lane < n && clamp01(__ldg(row + lane)) >= t;
    const bool in1 = lane + 32 < n && clamp01(__ldg(row + lane + 32)) >= t;
    const unsigned lo = __ballot_sync(0xffffffffu, in0), hi = __ballot_sync(0xffffffffu, in1);
    if (lane == 0) masks[r] = (unsigned long long)hi << 32 | lo;
  }
  __syncthreads();
  // 2. vertex and face count per lattice row
  for (int r = warp; r < R; r += kMeshWarps) {
    const int k = r / n1 - 1, j = r % n1 - 1;
    const unsigned long long r00 = S.row(k, j), r10 = S.row(k, j + 1), r01 = S.row(k + 1, j), r11 = S.row(k + 1, j + 1);
    int f = 0;
    for (int i = lane - 1; i < n; i += 32) f += tcnt[cell_case(r00, r10, r01, r11, i)];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) f += __shfl_xor_sync(0xffffffffu, f, o);
    if (lane == 0) {
      const RowCross c = row_cross(S, k, j);
      vbase[r] = c.x1 + __popcll(c.x) + __popcll(c.y) + __popcll(c.z);
      fbase[r] = f;
    }
  }
  __syncthreads();
  // 3. exclusive scan over the rows: thread t owns rows [t * per, (t + 1) * per)
  {
    const int per = (R + blockDim.x - 1) / blockDim.x;
    const int r0 = min((int)threadIdx.x * per, R), r1 = min(r0 + per, R);
    int sv = 0, sf = 0;
    for (int r = r0; r < r1; ++r) { sv += vbase[r];  sf += fbase[r]; }
    const int iv = warp_incl_scan(sv), jf = warp_incl_scan(sf);
    if (lane == 31) { wsum[0][warp] = iv;  wsum[1][warp] = jf; }
    __syncthreads();
    if (warp == 0) {
      const int a = warp_incl_scan(wsum[0][lane]), c = warp_incl_scan(wsum[1][lane]);
      wsum[0][lane] = a - wsum[0][lane];
      wsum[1][lane] = c - wsum[1][lane];
      if (lane == 31) { total[0] = a;  total[1] = c; }
    }
    __syncthreads();
    int ov = wsum[0][warp] + iv - sv, of = wsum[1][warp] + jf - sf;
    for (int r = r0; r < r1; ++r) {
      const int cv = vbase[r], cf = fbase[r];
      vbase[r] = ov;  fbase[r] = of;
      ov += cv;  of += cf;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) { counts[2 * b] = total[0];  counts[2 * b + 1] = total[1]; }
  float* vout = verts + (int64_t)b * max_verts * 3;
  int* fout = faces + (int64_t)b * max_faces * 3;
  const float fn = (float)n;
  auto field = [&](int k, int j, int i) -> float {
    return (k >= 0 && k < n && j >= 0 && j < n && i >= 0 && i < n) ? clamp01(__ldg(v + ((int64_t)k * n + j) * n + i)) : 0.f;
  };
  // vertex id of the edge from (k, j, i) along `axis` (a crossing edge, so k, j <= n - 1)
  auto vid = [&](int k, int j, int i, int axis) -> int {
    const int r = (k + 1) * n1 + (j + 1);
    if (i < 0) return vbase[r];                                            // the x edge from the padding
    const RowCross c = row_cross(S, k, j);
    const unsigned long long lo = below(i);
    return vbase[r] + c.x1 + __popcll(c.x & lo) + __popcll(c.y & lo) + __popcll(c.z & lo) +
           (axis > 0 ? bit(c.x, i) : 0) + (axis > 1 ? bit(c.y, i) : 0);
  };
  // 4. emit
  for (int r = warp; r < R; r += kMeshWarps) {
    const int k = r / n1 - 1, j = r % n1 - 1;
    const RowCross c = row_cross(S, k, j);
    int vb = vbase[r], fb = fbase[r];
    const unsigned long long r00 = S.row(k, j), r10 = S.row(k, j + 1), r01 = S.row(k + 1, j), r11 = S.row(k + 1, j + 1);
    for (int i0 = -1; i0 < n; i0 += 32) {                                 // lanes along i = i0 + lane
      const int i = i0 + lane;
      const bool live = i < n;
      const int bx = live ? (i < 0 ? c.x1 : bit(c.x, i)) : 0;
      const int by = live ? bit(c.y, i) : 0, bz = live ? bit(c.z, i) : 0;
      const int nv = bx + by + bz;
      const int ev = warp_incl_scan(nv);
      int id = vb + ev - nv;
      if (nv) {
        const float a = field(k, j, i);
        const float q[3] = {__fdiv_rn(__fadd_rn((float)i, 0.5f), fn), __fdiv_rn(__fadd_rn((float)j, 0.5f), fn),
                            __fdiv_rn(__fadd_rn((float)k, 0.5f), fn)};
        const float p[3] = {(float)i, (float)j, (float)k};
#pragma unroll
        for (int ax = 0; ax < 3; ++ax) {
          if (!(ax == 0 ? bx : ax == 1 ? by : bz)) continue;
          const float bv = ax == 0 ? field(k, j, i + 1) : ax == 1 ? field(k, j + 1, i) : field(k + 1, j, i);
          const float s = __fdiv_rn(__fsub_rn(t, a), __fsub_rn(bv, a));
          float* o = vout + (int64_t)id * 3;
          o[0] = ax == 0 ? __fdiv_rn(__fadd_rn(__fadd_rn(p[0], 0.5f), s), fn) : q[0];
          o[1] = ax == 1 ? __fdiv_rn(__fadd_rn(__fadd_rn(p[1], 0.5f), s), fn) : q[1];
          o[2] = ax == 2 ? __fdiv_rn(__fadd_rn(__fadd_rn(p[2], 0.5f), s), fn) : q[2];
          ++id;
        }
      }
      vb = __shfl_sync(0xffffffffu, vb + ev, 31);
      const int cs = live ? cell_case(r00, r10, r01, r11, i) : 0;
      const int nf = tcnt[cs];
      const int ef = warp_incl_scan(nf);
      int* fo = fout + (int64_t)(fb + ef - nf) * 3;
      for (int tr = 0; tr < nf; ++tr) {
#pragma unroll
        for (int q = 0; q < 3; ++q) {
          const int e = tedg[cs * 3 * kMcMaxTri + tr * 3 + q];
          const int ax = e >> 2, b0 = e & 1, b1 = (e >> 1) & 1;
          const int dx = ax == 0 ? 0 : b0, dy = ax == 0 ? b0 : ax == 1 ? 0 : b1, dz = ax == 2 ? 0 : b1;
          fo[tr * 3 + q] = vid(k + dz, j + dy, i + dx, ax);
        }
      }
      fb = __shfl_sync(0xffffffffu, fb + ef, 31);
    }
  }
}

int64_t mesh_smem_bytes(int n) {
  const int64_t R = (int64_t)(n + 1) * (n + 1);
  return (int64_t)n * n * 8 + 2 * R * 4 + 256 + 256 * 3 * kMcMaxTri;
}

}  // namespace
}  // namespace s3d

using namespace s3d;

extern "C" int s3d_voxel_mesh_bounds(int n, int* max_verts, int* max_faces) {
  if (!max_verts || !max_faces) {
    set_error("voxel_mesh_bounds: null argument");
    return S3D_ERR_INVALID;
  }
  S3D_CHECK_ARG(n >= 1 && n <= kMeshMaxN, "voxel_mesh_bounds: n must be in [1, %d], got %d", kMeshMaxN, n);
  *max_verts = 3 * (n + 1) * (n + 2) * (n + 2);
  *max_faces = 5 * (n + 1) * (n + 1) * (n + 1);
  return S3D_OK;
}

extern "C" int s3d_voxel_mesh(const float* vol, int B, int n, float t, float* verts, int max_verts, int* faces,
                              int max_faces, int* counts, void* stream) {
  if (!vol || !verts || !faces || !counts) {
    set_error("voxel_mesh: null argument");
    return S3D_ERR_INVALID;
  }
  S3D_CHECK_ARG(n >= 1 && n <= kMeshMaxN, "voxel_mesh: n must be in [1, %d], got %d", kMeshMaxN, n);
  S3D_CHECK_ARG(B >= 0, "voxel_mesh: B must be >= 0, got %d", B);
  S3D_CHECK_ARG(isfinite(t) && t > 0.f && t <= 1.f, "voxel_mesh: t must be finite and in (0, 1], got %g", (double)t);
  int mv = 0, mf = 0;
  s3d_voxel_mesh_bounds(n, &mv, &mf);
  S3D_CHECK_ARG(max_verts >= mv, "voxel_mesh: max_verts must be >= %d for n = %d, got %d", mv, n, max_verts);
  S3D_CHECK_ARG(max_faces >= mf, "voxel_mesh: max_faces must be >= %d for n = %d, got %d", mf, n, max_faces);
  if (B == 0) return S3D_OK;
  const int smem = (int)mesh_smem_bytes(n);
  S3D_CUDA(cudaFuncSetAttribute(voxel_mesh_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  voxel_mesh_kernel<<<B, kMeshThreads, smem, static_cast<cudaStream_t>(stream)>>>(vol, n, t, verts, max_verts, faces,
                                                                                 max_faces, counts);
  S3D_LAUNCH_CHECK();
  return S3D_OK;
}
