// deftet.cu — B200 implementation of Kaolin's DefTet volumetric renderer operators
// (SURVEY.md §8f rank 3):
//   deftet_sparse_render_forward_cuda   kaolin/csrc/render/mesh/deftet_cuda.cu:31-194
//   deftet_sparse_render_backward_cuda  kaolin/csrc/render/mesh/deftet_cuda.cu:238-430
// behind the C ABI of include/dibr_b200.h.
//
// Semantics (reference kernel): for every query point (x0, y0) with depth range [dmin, dmax)
// visit the faces of its view in INDEX ORDER; a face is recorded when the point is inside its
// bbox (half-open), all three eps-normalised barycentric weights are >= 0 and the interpolated
// depth lies in the range; the first `knum` such faces are written (face id, depth, w0, w1),
// the rest of the (B,P,K) arrays is -1 / 0.  The reference scans ALL faces for every point
// (O(P*F) bbox tests, one warp per point).  Here:
//   * the faces of a view are binned once into a uniform G x G grid laid over the bounding box of
//     the query points (count -> scan -> fill; faces that cover more than kMaxCells cells go to a
//     short per-view "wide" list instead);
//   * one warp per point reads only its cell's faces + the wide list, 32 candidates per step, the
//     hits are compacted with a ballot into shared memory, sorted by face index (they are few) and
//     written in that order — the reference's order;
//   * a point with more than kHitCap hits (never on real scenes) falls back to the reference's
//     in-order scan so that the first-knum rule stays exact.
// Per-hit arithmetic follows the compiled operation tree of the rasterizer (dibr_math.cuh),
// which shares its source expressions with this kernel (deftet_cuda.cu:131-153).
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/dibr_b200.h"
#include "dibr_math.cuh"

namespace {

using namespace dibr;

// Any tensor pointer not DIBR_B200_ALIGNMENT-byte aligned (NULL is aligned): bboxes are read as
// float4, coordinates as float2.
template <typename... P>
bool misaligned(P... p) { return ((((uintptr_t)p) | ... | (uintptr_t)0) & (DIBR_B200_ALIGNMENT - 1)) != 0; }

constexpr int kMaxCells = 16;     // cells a face may be inserted in; wider faces -> the view's wide list
constexpr int kHitCap = 128;      // hits a point can collect before it takes the ordered scan
constexpr int kWarps = 8;         // points per CTA
constexpr unsigned kFull = 0xffffffffu;

struct Grid {
  int B, F, P, G;
  const float* bounds;   // [B][4] xmin, ymin, 1/cell_w, 1/cell_h
  int* cnt;              // [B][G*G + 1] (last: wide list length)
  int* off;              // [B][G*G + 1]
  int* entries;          // [B][F*kMaxCells]
  int* wide;             // [B][F]
};

__global__ void deftet_bounds_kernel(int B, int P, int G, const float* __restrict__ pix, float* __restrict__ bounds) {
  const int b = blockIdx.x;
  float x0 = INFINITY, y0 = INFINITY, x1 = -INFINITY, y1 = -INFINITY;
  for (int i = threadIdx.x; i < P; i += blockDim.x) {
    const float2 p = __ldg(reinterpret_cast<const float2*>(pix) + (size_t)b * P + i);
    x0 = fminf(x0, p.x); x1 = fmaxf(x1, p.x); y0 = fminf(y0, p.y); y1 = fmaxf(y1, p.y);
  }
  __shared__ float s[4][32];
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    x0 = fminf(x0, __shfl_xor_sync(kFull, x0, d)); y0 = fminf(y0, __shfl_xor_sync(kFull, y0, d));
    x1 = fmaxf(x1, __shfl_xor_sync(kFull, x1, d)); y1 = fmaxf(y1, __shfl_xor_sync(kFull, y1, d));
  }
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { s[0][w] = x0; s[1][w] = y0; s[2][w] = x1; s[3][w] = y1; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < (int)(blockDim.x >> 5); ++i) {
      x0 = fminf(x0, s[0][i]); y0 = fminf(y0, s[1][i]); x1 = fmaxf(x1, s[2][i]); y1 = fmaxf(y1, s[3][i]);
    }
    if (!(x1 >= x0) || !(y1 >= y0)) { x0 = y0 = 0.f; x1 = y1 = 1.f; }   // no finite point
    const float wx = fmaxf(x1 - x0, 1e-20f), wy = fmaxf(y1 - y0, 1e-20f);
    float* o = bounds + 4 * b;
    o[0] = x0; o[1] = y0; o[2] = (float)G / wx; o[3] = (float)G / wy;
  }
}

__device__ __forceinline__ int cell_of(float v, float lo, float inv, int G) {
  const float c = (v - lo) * inv;
  // NaN -> 0; the clamp keeps points on the upper border (and anything outside) in range
  return (int)fminf(fmaxf(c, 0.f), (float)(G - 1));
}

// cells whose points can pass the half-open bbox test  x0 >= xmin && x0 < xmax  (conservative)
__device__ __forceinline__ bool face_cells(const Grid& g, int b, int64_t face, const float* bbox, int& cx0, int& cx1,
                                           int& cy0, int& cy1) {
  const float4 bb = __ldg(reinterpret_cast<const float4*>(bbox) + face);
  const float* bd = g.bounds + 4 * b;
  if (!(bb.z > bb.x) || !(bb.w > bb.y)) return false;   // empty or NaN box: no point can be inside
  cx0 = cell_of(bb.x, bd[0], bd[2], g.G); cx1 = cell_of(bb.z, bd[0], bd[2], g.G);
  cy0 = cell_of(bb.y, bd[1], bd[3], g.G); cy1 = cell_of(bb.w, bd[1], bd[3], g.G);
  return true;
}

template <bool FILL>
__global__ void __launch_bounds__(256) deftet_bin_kernel(Grid g, const float* __restrict__ bbox) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)g.B * g.F) return;
  const int b = (int)(i / g.F), f = (int)(i - (int64_t)b * g.F);
  int cx0, cx1, cy0, cy1;
  if (!face_cells(g, b, i, bbox, cx0, cx1, cy0, cy1)) return;
  const int ncell = g.G * g.G;
  int* cnt = g.cnt + (size_t)b * (ncell + 1);
  if ((cx1 - cx0 + 1) * (cy1 - cy0 + 1) > kMaxCells) {
    const int pos = atomicAdd(cnt + ncell, 1);
    if (FILL) g.wide[(size_t)b * g.F + pos] = f;
    return;
  }
  for (int cy = cy0; cy <= cy1; ++cy)
    for (int cx = cx0; cx <= cx1; ++cx) {
      const int c = cy * g.G + cx;
      const int pos = atomicAdd(cnt + c, 1);
      if (FILL) g.entries[(size_t)b * g.F * kMaxCells + g.off[(size_t)b * (ncell + 1) + c] + pos] = f;
    }
}

// exclusive scan of the G*G cell counters of one view (the wide-list counter is only reset)
__global__ void __launch_bounds__(1024) deftet_scan_kernel(Grid g) {
  __shared__ int warp_sums[32];
  __shared__ int carry;
  const int ncell = g.G * g.G;
  int* cnt = g.cnt + (size_t)blockIdx.x * (ncell + 1);
  int* off = g.off + (size_t)blockIdx.x * (ncell + 1);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) { carry = 0; off[ncell] = cnt[ncell]; cnt[ncell] = 0; }   // off[ncell] keeps the wide length
  __syncthreads();
  for (int base = 0; base < ncell; base += 1024) {
    const int i = base + tid;
    const int v = i < ncell ? cnt[i] : 0;
    int x = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const int y = __shfl_up_sync(kFull, x, d); if (lane >= d) x += y; }
    if (lane == 31) warp_sums[warp] = x;
    __syncthreads();
    if (warp == 0) {
      int w = warp_sums[lane];
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) { const int y = __shfl_up_sync(kFull, w, d); if (lane >= d) w += y; }
      warp_sums[lane] = w;
    }
    __syncthreads();
    const int excl = carry + (warp ? warp_sums[warp - 1] : 0) + x - v;
    if (i < ncell) { off[i] = excl; cnt[i] = 0; }
    __syncthreads();
    if (tid == 1023) carry = excl + v;
    __syncthreads();
  }
}

struct Hit { int face; float w0, w1, depth; };

// deftet_cuda.cu:118-160 for one (point, face): bbox, weights, depth, range.
__device__ __forceinline__ bool deftet_test(const float* __restrict__ fvz, const float* __restrict__ fvi,
                                            const float* __restrict__ bbox, int64_t face, float x0, float y0,
                                            float dmin, float dmax, float eps, Hit& h) {
  const float4 bb = __ldg(reinterpret_cast<const float4*>(bbox) + face);
  if (!(x0 >= bb.x && x0 < bb.z && y0 >= bb.y && y0 < bb.w)) return false;
  const float2* p = reinterpret_cast<const float2*>(fvi + face * 6);
  const float2 a = __ldg(p), b = __ldg(p + 1), c = __ldg(p + 2);
  const float aex = fsub(a.x, x0), aey = fsub(a.y, y0), bex = fsub(b.x, x0), bey = fsub(b.y, y0);
  const float cex = fsub(c.x, x0), cey = fsub(c.y, y0);
  const float u0 = ffma(bex, cey, -fmul(bey, cex));
  const float u1 = ffma(cex, aey, -fmul(cey, aex));
  const float u2 = ffma(aex, bey, -fmul(aey, bex));
  const float norm = fadd(fadd(u0, u1), u2);
  const float norm_eps = copysignf(eps, norm);          // copysignf((double)eps, (double)norm) -> float
  const float den = fadd(norm, norm_eps);
  const float w0 = fdiv(u0, den), w1 = fdiv(u1, den), w2 = fdiv(u2, den);
  if (!(w0 >= 0.f && w1 >= 0.f && w2 >= 0.f)) return false;
  const float* z = fvz + face * 3;
  const float depth = ffma(w2, __ldg(z + 2), ffma(w1, __ldg(z + 1), fmul(w0, __ldg(z))));
  if (!(depth < dmax && depth >= dmin)) return false;
  h.w0 = w0; h.w1 = w1; h.depth = depth;
  return true;
}

struct FwdArgs {
  Grid g;
  int knum;
  float eps;
  const float* fvz; const float* fvi; const float* bbox; const float* pix; const float* ranges;
  int64_t* face_idx; float* depth; float* w0; float* w1;
};

__global__ void __launch_bounds__(kWarps * 32) deftet_render_kernel(const __grid_constant__ FwdArgs a) {
  __shared__ Hit hits[kWarps][kHitCap];
  const Grid& g = a.g;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t pt = (int64_t)blockIdx.x * kWarps + warp;
  if (pt >= (int64_t)g.B * g.P) return;
  const int b = (int)(pt / g.P);
  const float2 xy = __ldg(reinterpret_cast<const float2*>(a.pix) + pt);
  const float2 rg = __ldg(reinterpret_cast<const float2*>(a.ranges) + pt);
  const float x0 = xy.x, y0 = xy.y, dmin = rg.x, dmax = rg.y;
  const int64_t fbase = (int64_t)b * g.F;
  const int ncell = g.G * g.G;
  const float* bd = g.bounds + 4 * b;
  const int cell = cell_of(y0, bd[1], bd[3], g.G) * g.G + cell_of(x0, bd[0], bd[2], g.G);
  Hit* mine = hits[warp];
  int n = 0;

  auto visit = [&](const int* list, int len) {
    for (int base = 0; base < len; base += 32) {
      Hit h; h.face = -1;
      bool hit = false;
      if (base + lane < len) {
        h.face = __ldg(list + base + lane);
        hit = deftet_test(a.fvz, a.fvi, a.bbox, fbase + h.face, x0, y0, dmin, dmax, a.eps, h);
      }
      const unsigned m = __ballot_sync(kFull, hit);
      if (hit) {
        const int pos = n + __popc(m & ((1u << lane) - 1u));
        if (pos < kHitCap) mine[pos] = h;
      }
      n += __popc(m);
    }
  };
  const int* cnt = g.cnt + (size_t)b * (ncell + 1);
  const int* off = g.off + (size_t)b * (ncell + 1);
  visit(g.entries + (size_t)b * g.F * kMaxCells + off[cell], cnt[cell]);
  visit(g.wide + (size_t)b * g.F, off[ncell]);
  __syncwarp();

  const int64_t out0 = pt * a.knum;
  int written = 0;
  if (n <= kHitCap) {
    // sort by face index: rank sort (n is small; the keys are distinct)
    for (int i = lane; i < n; i += 32) {
      const Hit h = mine[i];
      int rank = 0;
      for (int j = 0; j < n; ++j) rank += mine[j].face < h.face ? 1 : 0;
      if (rank < a.knum) {
        a.face_idx[out0 + rank] = h.face; a.depth[out0 + rank] = h.depth;
        a.w0[out0 + rank] = h.w0; a.w1[out0 + rank] = h.w1;
      }
    }
    written = min(n, a.knum);
  } else {
    // the reference's own ordered scan (deftet_cuda.cu:96-187), for this point only
    int num = 0;
    for (int base = 0; base < g.F && num < a.knum; base += 32) {
      Hit h; h.face = base + lane;
      const bool hit = h.face < g.F && deftet_test(a.fvz, a.fvi, a.bbox, fbase + h.face, x0, y0, dmin, dmax, a.eps, h);
      const unsigned m = __ballot_sync(kFull, hit);
      if (hit) {
        const int pos = num + __popc(m & ((1u << lane) - 1u));
        if (pos < a.knum) {
          a.face_idx[out0 + pos] = h.face; a.depth[out0 + pos] = h.depth; a.w0[out0 + pos] = h.w0; a.w1[out0 + pos] = h.w1;
        }
      }
      num += __popc(m);
    }
    written = min(num, a.knum);
  }
  // padding (the reference's at::full(-1) / at::full(-inf) / at::zeros, deftet.cpp:88-95)
  for (int k = written + lane; k < a.knum; k += 32) {
    a.face_idx[out0 + k] = -1; a.depth[out0 + k] = -INFINITY; a.w0[out0 + k] = 0.f; a.w1[out0 + k] = 0.f;
  }
}

// deftet_cuda.cu:238-430: one thread per (point, k) entry; the same derivative tree as the
// rasterizer's backward (raster_backward_geom / _feature), scattered with vector reductions.
struct BwdArgs {
  int64_t n; int P, K, F, D;
  const float* grad; const int64_t* face_idx; const float* weights; const float* fvi; const float* ff;
  float eps;
  float* g_xy; float* g_ff;
};

__global__ void __launch_bounds__(256) deftet_backward_kernel(const __grid_constant__ BwdArgs a) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  const int64_t f = a.face_idx[i];
  if (f < 0) return;
  const int64_t b = i / ((int64_t)a.P * a.K);
  const int64_t face = b * a.F + f;
  const float w0 = __ldg(a.weights + i * 3), w1 = __ldg(a.weights + i * 3 + 1), w2 = __ldg(a.weights + i * 3 + 2);
  const float2* pp = reinterpret_cast<const float2*>(a.fvi + face * 6);
  const float2 pa = __ldg(pp), pb = __ldg(pp + 1), pc = __ldg(pp + 2);
  const float p[6] = {pa.x, pa.y, pb.x, pb.y, pc.x, pc.y};
  RasterBwdGeom G;
  raster_backward_geom(p, w0, w1, w2, a.eps, G);
  float v[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  const float* cf = a.ff + face * 3 * a.D;
  float* gf = a.g_ff + face * 3 * a.D;
  for (int d = 0; d < a.D; ++d) {
    const float g = __ldg(a.grad + i * a.D + d);
    float t6[6];
    raster_backward_feature(G, g, __ldg(cf + d), __ldg(cf + a.D + d), __ldg(cf + 2 * a.D + d), t6);
#pragma unroll
    for (int j = 0; j < 6; ++j) v[j] += t6[j];
    atomicAdd(gf + d, g * w0); atomicAdd(gf + a.D + d, g * w1); atomicAdd(gf + 2 * a.D + d, g * w2);
  }
  float2* gx = reinterpret_cast<float2*>(a.g_xy + face * 6);
  atomicAdd(gx, make_float2(v[0], v[1]));
  atomicAdd(gx + 1, make_float2(v[2], v[3]));
  atomicAdd(gx + 2, make_float2(v[4], v[5]));
}

int grid_side(int F) {
  int G = 8;
  while (G < 256 && (int64_t)G * G < F) G += 8;   // ~1 face per cell before overlaps
  return G;
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct Layout { size_t bounds, cnt, off, entries, wide, total; };
Layout layout_for(int B, int F) {
  const int G = grid_side(F);
  Layout L;
  L.bounds = align_up((size_t)B * 4 * sizeof(float), 256);
  L.cnt = align_up((size_t)B * (G * G + 1) * sizeof(int), 256);
  L.off = L.cnt;
  L.entries = align_up((size_t)B * (size_t)(F > 0 ? F : 1) * kMaxCells * sizeof(int), 256);
  L.wide = align_up((size_t)B * (size_t)(F > 0 ? F : 1) * sizeof(int), 256);
  L.total = L.bounds + L.cnt + L.off + L.entries + L.wide + 256;
  return L;
}

}  // namespace

extern "C" {

size_t dibr_b200_deftet_workspace_bytes(int batch, int num_faces) {
  if (batch <= 0 || num_faces < 0) return 0;
  return layout_for(batch, num_faces).total;
}

int dibr_b200_deftet_sparse_render_forward(int batch, int num_faces, int num_pixels, int knum,
                                           const float* face_vertices_z, const float* face_vertices_image,
                                           const float* face_bboxes, const float* pixel_coords,
                                           const float* render_ranges, float eps, int64_t* face_idx,
                                           float* pixel_depth, float* w0, float* w1, void* workspace,
                                           size_t workspace_bytes, dibr_b200_stream_t stream) {
  if (batch <= 0 || num_faces < 0 || num_pixels < 0 || knum <= 0) return DIBR_B200_EINVAL;
  if (!pixel_coords || !render_ranges || !face_idx || !pixel_depth || !w0 || !w1 || !workspace) return DIBR_B200_EINVAL;
  if (num_faces > 0 && (!face_vertices_z || !face_vertices_image || !face_bboxes)) return DIBR_B200_EINVAL;
  if (misaligned(face_vertices_z, face_vertices_image, face_bboxes, pixel_coords, render_ranges, face_idx,
                 pixel_depth, w0, w1))
    return DIBR_B200_EINVAL;
  if ((int64_t)batch * num_pixels * knum >= (int64_t)1 << 40 || (int64_t)num_faces * kMaxCells >= 0x7fffffffLL) return DIBR_B200_ESIZE;
  const Layout L = layout_for(batch, num_faces);
  char* p = (char*)align_up((size_t)workspace, 256);
  if (workspace_bytes < L.total || p + L.total - 256 > (char*)workspace + workspace_bytes) return DIBR_B200_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  if (num_pixels == 0) return 0;
  FwdArgs a;
  Grid& g = a.g;
  g.B = batch; g.F = num_faces; g.P = num_pixels; g.G = grid_side(num_faces);
  g.bounds = (float*)p; p += L.bounds;
  g.cnt = (int*)p; p += L.cnt;
  g.off = (int*)p; p += L.off;
  g.entries = (int*)p; p += L.entries;
  g.wide = (int*)p;
  cudaError_t e = cudaMemsetAsync(g.cnt, 0, L.cnt, st);
  if (e != cudaSuccess) return (int)e;
  deftet_bounds_kernel<<<batch, 256, 0, st>>>(batch, num_pixels, g.G, pixel_coords, const_cast<float*>(g.bounds));
  const int64_t nf = (int64_t)batch * num_faces;
  if (nf > 0) {
    deftet_bin_kernel<false><<<(unsigned)((nf + 255) / 256), 256, 0, st>>>(g, face_bboxes);
    deftet_scan_kernel<<<batch, 1024, 0, st>>>(g);
    deftet_bin_kernel<true><<<(unsigned)((nf + 255) / 256), 256, 0, st>>>(g, face_bboxes);
  } else {
    e = cudaMemsetAsync(g.off, 0, L.off, st);
    if (e != cudaSuccess) return (int)e;
  }
  a.knum = knum; a.eps = eps; a.fvz = face_vertices_z; a.fvi = face_vertices_image; a.bbox = face_bboxes;
  a.pix = pixel_coords; a.ranges = render_ranges; a.face_idx = face_idx; a.depth = pixel_depth; a.w0 = w0; a.w1 = w1;
  const int64_t npt = (int64_t)batch * num_pixels;
  deftet_render_kernel<<<(unsigned)((npt + kWarps - 1) / kWarps), kWarps * 32, 0, st>>>(a);
  return (int)cudaGetLastError();
}

int dibr_b200_deftet_sparse_render_backward(int batch, int num_faces, int num_pixels, int knum, int feat_dim,
                                            const float* grad_interpolated_features, const int64_t* face_idx,
                                            const float* weights, const float* face_vertices_image,
                                            const float* face_features, float eps,
                                            float* grad_face_vertices_image, float* grad_face_features,
                                            dibr_b200_stream_t stream) {
  if (batch <= 0 || num_faces < 0 || num_pixels < 0 || knum <= 0 || feat_dim < 0) return DIBR_B200_EINVAL;
  if (!grad_face_vertices_image || (feat_dim > 0 && !grad_face_features)) return DIBR_B200_EINVAL;
  if (misaligned(grad_interpolated_features, face_idx, weights, face_vertices_image, face_features,
                 grad_face_vertices_image, grad_face_features))
    return DIBR_B200_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t nf = (int64_t)batch * num_faces;
  cudaError_t e = cudaMemsetAsync(grad_face_vertices_image, 0, (size_t)nf * 6 * sizeof(float), st);
  if (e != cudaSuccess) return (int)e;
  if (feat_dim > 0) {
    e = cudaMemsetAsync(grad_face_features, 0, (size_t)nf * 3 * feat_dim * sizeof(float), st);
    if (e != cudaSuccess) return (int)e;
  }
  const int64_t n = (int64_t)batch * num_pixels * knum;
  if (n == 0 || nf == 0 || feat_dim == 0) return 0;
  if (!grad_interpolated_features || !face_idx || !weights || !face_vertices_image || !face_features) return DIBR_B200_EINVAL;
  BwdArgs a;
  a.n = n; a.P = num_pixels; a.K = knum; a.F = num_faces; a.D = feat_dim;
  a.grad = grad_interpolated_features; a.face_idx = face_idx; a.weights = weights; a.fvi = face_vertices_image;
  a.ff = face_features; a.eps = eps; a.g_xy = grad_face_vertices_image; a.g_ff = grad_face_features;
  deftet_backward_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(a);
  return (int)cudaGetLastError();
}

}  // extern "C"
