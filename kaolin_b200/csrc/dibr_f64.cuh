// dibr_f64.cuh — the float64 instantiation of the DIB-R path (SURVEY.md §8 a11: the reference
// dispatches float and double, rasterization_cuda.cu:218/427, dibr_soft_mask_cuda.cu:205/376).
// Included inside dibr_b200.cu's unnamed namespace: it reuses the binning infrastructure.
//
// Double callers are rare (the reference's tests parametrise the dtype; training runs in fp32), so
// this path is built for exactness, not speed:
//   * f64_prep_kernel turns the double vertices into CONSERVATIVE float bboxes (mins rounded down,
//     maxes rounded up, tight and enlarged) + a validity byte per face; the fp32 binning kernels
//     (bin pyramid, exact integer rectangles of those float boxes) then enumerate a superset of the
//     faces every pixel has to look at;
//   * dibr_f64_fwd_kernel: one thread per pixel walks the bins of its tile and decides every
//     candidate with the reference's own double arithmetic (dibr_math_f64.cuh): the half-open bbox
//     test on the double bbox, the DMUL/DFMA edge functions, eps by copysign, IEEE divisions, strict
//     '>' with ties to the lowest index; the soft mask visits the tile's candidates in index order
//     (the shared-memory sort of the fp32 path) and applies the double enlarged-bbox test, the
//     first knum hits count;
//   * dibr_f64_bwd_kernel: the same walk, gradients scattered with native double atomics.
// The four operators run the same device code in double natively (f64_raster_op_kernel,
// f64_raster_bwd_op_kernel, f64_soft_op_kernel, f64_soft_bwd_op_kernel): their bbox tests read the
// caller's boxes, xy comes multiplied, and the soft-mask K-lists are outputs / inputs.
#include "dibr_math_f64.cuh"

struct F64Args {
  Scene s;
  int D, K, mode;
  float eps, sigmainv, multiplier;
  double margin;                                          // boxlen * multiplier, in double
  const double* xy; const double* z; const double* feat;  // (NF,3,2) unscaled, (NF,3), (NF,3,D)
  double* out_feat; int64_t* idx; double* out_w; double* out_soft;
  const double* g_feat; const double* g_soft; const double* soft;
  double* g_xy; double* g_ff;
};

__global__ void __launch_bounds__(256) f64_prep_kernel(int64_t NF, const double* __restrict__ xy, const double* __restrict__ fnz,
                                                       const uint8_t* __restrict__ valid_in, float multiplier, double margin,
                                                       float* __restrict__ xyf, float* __restrict__ bt, float* __restrict__ bl,
                                                       uint8_t* __restrict__ valid) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= NF) return;
  const double m = (double)multiplier;
  double v[6];
#pragma unroll
  for (int k = 0; k < 6; ++k) { v[k] = __dmul_rn(xy[i * 6 + k], m); xyf[i * 6 + k] = (float)v[k]; }
  const double xmin = fmin(fmin(v[0], v[2]), v[4]), ymin = fmin(fmin(v[1], v[3]), v[5]);
  const double xmax = fmax(fmax(v[0], v[2]), v[4]), ymax = fmax(fmax(v[1], v[3]), v[5]);
  reinterpret_cast<float4*>(bt)[i] = make_float4(__double2float_rd(xmin), __double2float_rd(ymin),
                                                 __double2float_ru(xmax), __double2float_ru(ymax));
  reinterpret_cast<float4*>(bl)[i] = make_float4(__double2float_rd(xmin - margin), __double2float_rd(ymin - margin),
                                                 __double2float_ru(xmax + margin), __double2float_ru(ymax + margin));
  bool ok = true;
  if (fnz) ok = ok && fnz[i] >= 0.0;
  if (valid_in) ok = ok && valid_in[i] != 0;
  valid[i] = ok ? 1 : 0;
}

__device__ __forceinline__ void f64_face(const F64Args& a, int64_t g, double m, double v[6], double bb[4]) {
#pragma unroll
  for (int k = 0; k < 6; ++k) v[k] = __dmul_rn(__ldg(a.xy + g * 6 + k), m);   // face_vertices_image * multiplier (torch, double)
  bb[0] = fmin(fmin(v[0], v[2]), v[4]); bb[1] = fmin(fmin(v[1], v[3]), v[5]);
  bb[2] = fmax(fmax(v[0], v[2]), v[4]); bb[3] = fmax(fmax(v[1], v[3]), v[5]);
}

// Visits, in face-index order, the soft-mask candidates of the calling thread's pixel (CTA-collective:
// every thread of the tile calls it).  inside(face, v[6]) loads the face's multiplied xy into v and
// returns whether its double enlarged bbox holds the pixel; hit(face, v[6]) is invoked for those faces
// and returns false to stop (knum reached).
template <typename SM, typename Inside, typename Hit>
__device__ __forceinline__ void f64_soft_walk_by(const Scene& s, const TileCtx& c, SM& sm, bool uncovered,
                                                 Inside inside, Hit hit) {
  const int maxf = s.F;
  bool want = uncovered;
  int lo = -1;
  while (true) {
    int hi;
    const int n = soft_window(s, c, sm, lo, maxf, hi);
    soft_sort(sm, n);
    for (int j = 0; j < n; ++j) {
      const unsigned long long key = sm.sorted[j];
      if (want && (((uint32_t)key) & c.sel) == c.sel) {
        const int f = (int)(key >> 32);
        double v[6];
        if (inside(f, v)) want = hit(f, v);
      }
    }
    const bool all_done = __syncthreads_and(!want);
    if (hi == 0x7fffffff || all_done) break;
    lo = hi;
  }
}

// The fused path's walk: enlarged bboxes recomputed from the vertices (dibr.py:33-39 in double:
// [min - boxlen*m, max + boxlen*m]; dibr_soft_mask_cuda.cu:95).
template <typename Hit>
__device__ __forceinline__ void f64_soft_walk(const F64Args& a, const TileCtx& c, TileSmem& sm, bool uncovered,
                                              double x0, double y0, Hit hit) {
  const double m = (double)a.multiplier;
  f64_soft_walk_by(a.s, c, sm, uncovered, [&](int f, double* v) {
    double bb[4];
    f64_face(a, c.fbase + f, m, v, bb);
    return !(x0 < bb[0] - a.margin || x0 >= bb[2] + a.margin || y0 < bb[1] - a.margin || y0 >= bb[3] + a.margin);
  }, hit);
}

// The reference's double rasterize decision (rasterization_cuda.cu:85-188) for the calling thread's pixel
// over the tight bins of its tile: face(f, v[6], bb[4]) loads face f's multiplied xy and the bbox its
// half-open test reads.  Returns the winning face (relative to the view, -1: none) and its weights.
template <typename SM, typename Face>
__device__ __forceinline__ int f64_raster_pixel(const Scene& s, const TileCtx& c, const SM& sm, float eps,
                                                const double* z, double x0, double y0, Face face,
                                                double& b0, double& b1, double& b2) {
  int best = -1;
  double bz = -INFINITY;
  b0 = 0.0; b1 = 0.0; b2 = 0.0;
  for (int l = 0; l < s.L; ++l) {
    const BinRef bin = sm.bin[0][l];
    for (int i = 0; i < bin.n; ++i) {
      const int4 e = __ldg(bin.ptr + i);
      const int x_lo = e.y & 0xffff, x_hi = (int)((unsigned)e.y >> 16), y_lo = e.z & 0xffff, y_hi = (int)((unsigned)e.z >> 16);
      if (c.px < x_lo || c.px >= x_hi || c.py < y_lo || c.py >= y_hi) continue;
      double v[6], bb[4];
      face(c.fbase + e.x, v, bb);
      if (x0 < bb[0] || x0 >= bb[2] || y0 < bb[1] || y0 >= bb[3]) continue;
      double w0, w1, w2;
      if (!dibr64::raster_weights((double)eps, x0, y0, v[0], v[1], v[2], v[3], v[4], v[5], w0, w1, w2)) continue;
      const double* zp = z + (c.fbase + e.x) * 3;
      const double zv = dibr64::raster_interp(__ldg(zp), __ldg(zp + 1), __ldg(zp + 2), w0, w1, w2);
      if (!(zv <= bz) || (zv == bz && e.x < best)) { bz = zv; best = e.x; b0 = w0; b1 = w1; b2 = w2; }
    }
  }
  return best;
}

// face_idx, weights and interpolated features of pixel `pix` (feat: the faces of its view from fbase).
__device__ __forceinline__ void f64_raster_store(int64_t pix, int64_t fbase, int best, double b0, double b1,
                                                 double b2, int D, const double* feat, int64_t* idx,
                                                 double* out_w, double* out_feat) {
  idx[pix] = (int64_t)best;
  double* wp = out_w + pix * 3;
  wp[0] = b0; wp[1] = b1; wp[2] = b2;
  double* fp = out_feat + pix * D;
  const double* ff = feat + (fbase + max(best, 0)) * 3 * D;
  for (int d = 0; d < D; ++d)
    fp[d] = best >= 0 ? dibr64::raster_interp(__ldg(ff + d), __ldg(ff + D + d), __ldg(ff + 2 * D + d), b0, b1, b2) : 0.0;
}

// Rasterize backward of one covered pixel (rasterization_cuda.cu:266-399 with scalar_t = double): a.xy is
// UNSCALED (rasterization.py:360-368), `face` the global face id; double atomics into a.g_xy / a.g_ff.
__device__ __forceinline__ void f64_raster_backward_pixel(const F64Args& a, int64_t face, int64_t pix) {
  double p[6];
#pragma unroll
  for (int k = 0; k < 6; ++k) p[k] = __ldg(a.xy + face * 6 + k);
  const double* wp = a.out_w + pix * 3;
  const double w0 = wp[0], w1 = wp[1], w2 = wp[2];
  dibr64::BwdGeom G;
  dibr64::raster_backward_geom(p, w0, w1, w2, a.eps, G);
  double vsum[6] = {0, 0, 0, 0, 0, 0};
  const double* cf = a.feat + face * 3 * a.D;
  double* gf = a.g_ff + face * 3 * a.D;
  for (int d = 0; d < a.D; ++d) {
    const double g = a.g_feat[pix * a.D + d];
    double t6[6];
    dibr64::raster_backward_feature(G, g, __ldg(cf + d), __ldg(cf + a.D + d), __ldg(cf + 2 * a.D + d), t6);
#pragma unroll
    for (int j = 0; j < 6; ++j) vsum[j] += t6[j];
    atomicAdd(gf + d, g * w0); atomicAdd(gf + a.D + d, g * w1); atomicAdd(gf + 2 * a.D + d, g * w2);
  }
#pragma unroll
  for (int j = 0; j < 6; ++j) atomicAdd(a.g_xy + face * 6 + j, vsum[j]);
}

template <bool BWD>
__global__ void __launch_bounds__(kThreads) dibr_f64_kernel(const __grid_constant__ F64Args a) {
  __shared__ __align__(128) TileSmem sm;
  const Scene& s = a.s;
  const TileCtx c = make_tile_ctx(s);
  load_bin_table(s, c, sm);
  __syncthreads();
  const double x0 = (double)c.x0, y0 = (double)c.y0;     // computed in float, widened (rasterization_cuda.cu:85-86)
  const double m = (double)a.multiplier;
  int best = -1;
  if (!BWD && (a.mode & DIBR_B200_RASTER)) {
    double b0, b1, b2;
    best = f64_raster_pixel(s, c, sm, a.eps, a.z, x0, y0,
                            [&](int64_t g, double* v, double* bb) { f64_face(a, g, m, v, bb); }, b0, b1, b2);
    if (c.in_img) f64_raster_store(c.pix, c.fbase, best, b0, b1, b2, a.D, a.feat, a.idx, a.out_w, a.out_feat);
  } else {
    best = c.in_img ? (int)a.idx[c.pix] : 0;
  }
  const bool uncovered = c.in_img && best < 0;

  if (!BWD) {
    if (!(a.mode & DIBR_B200_SOFT_MASK)) return;
    double allprob = 1.0;
    int kid = 0;
    if (__syncthreads_or(uncovered)) {
      f64_soft_walk(a, c, sm, uncovered, x0, y0, [&](int, const double* v) {
        int edgeid;
        const double d2 = dibr64::soft_min_dist(x0, y0, v, a.multiplier, edgeid);
        allprob = dibr::dmul(allprob, dibr::dsub(1.0, dibr64::soft_prob(d2, a.sigmainv, a.multiplier)));
        return ++kid < a.K;
      });
    }
    if (c.in_img) a.out_soft[c.pix] = uncovered ? dibr::dsub(1.0, allprob) : 1.0;
    return;
  }

  // ---- backward
  if (a.g_feat && c.in_img && best >= 0) f64_raster_backward_pixel(a, c.fbase + best, c.pix);
  if (a.g_soft && __syncthreads_or(uncovered)) {
    const double dLdp = uncovered ? a.g_soft[c.pix] : 0.0;
    const double allprob = uncovered ? a.soft[c.pix] : 0.0;
    int kid = 0;
    f64_soft_walk(a, c, sm, uncovered, x0, y0, [&](int f, const double* v) {
      int edgeid;
      const double d2 = dibr64::soft_min_dist(x0, y0, v, a.multiplier, edgeid);
      const double prob = dibr64::soft_prob(d2, a.sigmainv, a.multiplier);
      double g[6];
      dibr64::soft_backward_terms(x0, y0, v, edgeid, prob, allprob, dLdp, a.sigmainv, a.multiplier, g);
      double* gp = a.g_xy + (c.fbase + f) * 6;
#pragma unroll
      for (int j = 0; j < 6; ++j)
        if (g[j] != 0.0) atomicAdd(gp + j, g[j]);
      return ++kid < a.K;
    });
  }
}

// ---------------------------------------------------------------------------
// The four operators in double (rasterization_cuda.cu / dibr_soft_mask_cuda.cu with scalar_t = double).
// Unlike the fused path they take the caller's tensors as given: xy already multiplied, the half-open
// bbox tests read the caller's (tight | enlarged) boxes, every face is valid, and the soft-mask
// K-lists are outputs of the forward and inputs of the backward.
struct F64OpArgs {
  Scene s;
  int D, K;
  float eps, sigmainv, multiplier;
  const double* xy; const double* z; const double* feat;  // xy: (NF,3,2) multiplied; z (NF,3); feat (NF,3,D)
  const double* box;                                      // (NF,4) the caller's bboxes [xmin,ymin,xmax,ymax]
  double* out_feat; int64_t* idx; double* out_w; double* out_soft;
  double* prob; int64_t* cidx; uint8_t* ctype;             // K-lists (all or none)
};

// The bins of an operator call: the caller's double boxes rounded outward to float, so that the fp32
// binning enumerates a superset of the faces the double test accepts; xy to float only because the
// binning kernel loads it (it reads the given boxes, not the vertices).
__global__ void __launch_bounds__(256) f64_op_prep_kernel(int64_t NF, const double* __restrict__ xy,
                                                          const double* __restrict__ box, float* __restrict__ xyf,
                                                          float* __restrict__ boxf) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= NF) return;
#pragma unroll
  for (int k = 0; k < 6; ++k) xyf[i * 6 + k] = (float)xy[i * 6 + k];
  const double* b = box + i * 4;
  reinterpret_cast<float4*>(boxf)[i] = make_float4(__double2float_rd(b[0]), __double2float_rd(b[1]),
                                                   __double2float_ru(b[2]), __double2float_ru(b[3]));
}

__device__ __forceinline__ void f64_op_face(const F64OpArgs& a, int64_t g, double v[6], double bb[4]) {
#pragma unroll
  for (int k = 0; k < 6; ++k) v[k] = __ldg(a.xy + g * 6 + k);
#pragma unroll
  for (int k = 0; k < 4; ++k) bb[k] = __ldg(a.box + g * 4 + k);
}

struct F64BinSmem { BinRef bin[2][kMaxLevels]; };

// packed_rasterize_forward: one thread per pixel over its tile's tight bins (Scene.first: packed meshes).
__global__ void __launch_bounds__(kThreads) f64_raster_op_kernel(const __grid_constant__ F64OpArgs a) {
  __shared__ F64BinSmem sm;
  const Scene& s = a.s;
  const TileCtx c = make_tile_ctx(s);
  load_bin_table(s, c, sm);
  __syncthreads();
  if (!c.in_img) return;
  double b0, b1, b2;
  const int best = f64_raster_pixel(s, c, sm, a.eps, a.z, (double)c.x0, (double)c.y0,
                                    [&](int64_t g, double* v, double* bb) { f64_op_face(a, g, v, bb); }, b0, b1, b2);
  f64_raster_store(c.pix, c.fbase, best, b0, b1, b2, a.D, a.feat, a.idx, a.out_w, a.out_feat);
}

// rasterize_backward: one thread per pixel of the (B,H,W) image; selected_face_idx relative to the view of
// a.s.F faces.
__global__ void __launch_bounds__(256) f64_raster_bwd_op_kernel(const __grid_constant__ F64Args a) {
  const int64_t pix = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t HW = (int64_t)a.s.H * a.s.W;
  if (pix >= a.s.B * HW) return;
  const int64_t f = a.idx[pix];
  if (f >= 0) f64_raster_backward_pixel(a, (pix / HW) * a.s.F + f, pix);
}

// dibr_soft_mask_forward: the first knum faces by index whose enlarged box holds each uncovered pixel.
__global__ void __launch_bounds__(kThreads) f64_soft_op_kernel(const __grid_constant__ F64OpArgs a) {
  __shared__ __align__(128) TileSmem sm;
  const Scene& s = a.s;
  const TileCtx c = make_tile_ctx(s);
  load_bin_table(s, c, sm);
  __syncthreads();
  const double x0 = (double)c.x0, y0 = (double)c.y0;
  const bool uncovered = c.in_img && a.idx[c.pix] < 0;
  double allprob = 1.0;
  int kid = 0;
  if (__syncthreads_or(uncovered)) {
    f64_soft_walk_by(s, c, sm, uncovered, [&](int f, double* v) {
      double bb[4];
      f64_op_face(a, c.fbase + f, v, bb);
      return !(x0 < bb[0] || x0 >= bb[2] || y0 < bb[1] || y0 >= bb[3]);
    }, [&](int f, const double* v) {
      int edgeid;
      const double d2 = dibr64::soft_min_dist(x0, y0, v, a.multiplier, edgeid);
      const double prob = dibr64::soft_prob(d2, a.sigmainv, a.multiplier);
      allprob = dibr::dmul(allprob, dibr::dsub(1.0, prob));
      if (a.cidx) {
        const int64_t o = c.pix * a.K + kid;
        a.prob[o] = prob; a.cidx[o] = f; a.ctype[o] = (uint8_t)(edgeid + 1);
      }
      return ++kid < a.K;
    });
  }
  if (!c.in_img) return;
  a.out_soft[c.pix] = uncovered ? dibr::dsub(1.0, allprob) : 1.0;
  if (a.cidx) {   // padding the reference gets from at::zeros / at::full(-1)
    for (int k = kid; k < a.K; ++k) {
      const int64_t o = c.pix * a.K + k;
      a.prob[o] = 0.0; a.cidx[o] = -1; a.ctype[o] = 0;
    }
  }
}

// dibr_soft_mask_backward: walks each uncovered pixel's stored list up to the first idx < 0, with the
// stored prob and dist_type and the geometry recomputed from the multiplied xy
// (dibr_soft_mask_cuda.cu:266-349).
struct F64SoftBwdArgs {
  int B, H, W, F, K;
  PixelGrid grid;
  float sigmainv, multiplier;
  const double* grad_soft; const double* soft; const int64_t* idx;
  const double* prob; const int64_t* cidx; const uint8_t* ctype; const double* xy;
  double* grad_xy;
};

__global__ void __launch_bounds__(256) f64_soft_bwd_op_kernel(const __grid_constant__ F64SoftBwdArgs a) {
  const int64_t pix = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= (int64_t)a.B * a.H * a.W || a.idx[pix] >= 0) return;
  const int ix = (int)(pix % a.W), iy = (int)((pix / a.W) % a.H);
  const int64_t b = pix / ((int64_t)a.W * a.H);
  const double x0 = (double)pix_x(a.grid, ix), y0 = (double)pix_y(a.grid, iy);
  const double dLdp = a.grad_soft[pix], allprob = a.soft[pix];
  for (int k = 0; k < a.K; ++k) {
    const int64_t f = a.cidx[pix * a.K + k];
    if (f < 0) break;
    const int64_t base = (b * a.F + f) * 6;
    double v[6], g[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) v[i] = __ldg(a.xy + base + i);
    dibr64::soft_backward_terms(x0, y0, v, (int)a.ctype[pix * a.K + k] - 1, a.prob[pix * a.K + k], allprob, dLdp,
                                a.sigmainv, a.multiplier, g);
#pragma unroll
    for (int i = 0; i < 6; ++i)
      if (g[i] != 0.0) atomicAdd(a.grad_xy + base + i, g[i]);
  }
}

struct F64Layout { size_t base, xyf, bt, bl, valid, total; };
F64Layout f64_layout(int B, int64_t NF, int H, int W) {
  F64Layout L;
  const size_t n = (size_t)(NF > 0 ? NF : 1);
  L.base = align_up(layout_for(B, NF, H, W).base, 256);
  L.xyf = align_up(n * 6 * sizeof(float), 256);
  L.bt = align_up(n * 4 * sizeof(float), 256);
  L.bl = L.bt;
  L.valid = align_up(n, 256);
  L.total = L.base + L.xyf + L.bt + L.bl + L.valid + 256;
  return L;
}

// Lays out the float scene of a double call in the workspace: bins, then xy, tight and enlarged boxes and
// a validity byte per face, all float.
struct F64Scratch { float* xyf; float* bt; float* bl; uint8_t* valid; };
int f64_scene(Scene& s, int B, int64_t NF, int F, int H, int W, float multiplier, void* ws, size_t ws_bytes,
              F64Scratch& o) {
  const F64Layout L = f64_layout(B, NF, H, W);
  char* p = (char*)align_up((size_t)ws, 256);
  if (!ws || ws_bytes < L.total || p + L.total - 256 > (char*)ws + ws_bytes) return DIBR_B200_EWORKSPACE;
  int rc = setup_scene(s, B, NF, F, H, W, multiplier, 0.f, 0, p, L.base);
  if (rc) return rc;
  o.xyf = (float*)(p + L.base);
  o.bt = (float*)(p + L.base + L.xyf);
  o.bl = (float*)(p + L.base + L.xyf + L.bt);
  o.valid = (uint8_t*)(p + L.base + L.xyf + L.bt + L.bl);
  s.first = nullptr; s.xy = o.xyf; s.z = nullptr; s.premultiplied = 1; s.fnz = nullptr; s.valid = nullptr;
  s.bbox_tight = o.bt; s.bbox_large = o.bl;
  return 0;
}

// Prepares the float scene (conservative bboxes) + bins for a double call.
int f64_setup(F64Args& a, int B, int F, int H, int W, const double* fvi, const double* fnz, const uint8_t* valid,
              float multiplier, double margin, int sets, bool rebuild, void* ws, size_t ws_bytes, cudaStream_t st) {
  const int64_t NF = (int64_t)B * F;
  F64Scratch o;
  int rc = f64_scene(a.s, B, NF, F, H, W, multiplier, ws, ws_bytes, o);
  if (rc) return rc;
  Scene& s = a.s;
  s.valid = o.valid;
  if (rebuild) {
    if (NF > 0)
      f64_prep_kernel<<<(unsigned)((NF + 255) / 256), 256, 0, st>>>(NF, fvi, fnz, valid, multiplier, margin, o.xyf,
                                                                    o.bt, o.bl, o.valid);
    rc = build_bins(s, sets, st);     // with no faces: zeroed counters, every pixel takes the empty path
    if (rc) return rc;
  }
  return 0;
}

// Scene + bins of an operator call from the caller's boxes: set 1 = tight (rasterize), 2 = enlarged (soft mask).
int f64_op_setup(F64OpArgs& a, int B, int64_t NF, int F, int H, int W, const int64_t* first, float multiplier,
                 int set, void* ws, size_t ws_bytes, cudaStream_t st) {
  F64Scratch o;
  int rc = f64_scene(a.s, B, NF, F, H, W, multiplier, ws, ws_bytes, o);
  if (rc) return rc;
  Scene& s = a.s;
  s.first = first;
  float* boxf = set == 1 ? o.bt : o.bl;
  s.bbox_tight = set == 1 ? boxf : nullptr;
  s.bbox_large = set == 2 ? boxf : nullptr;
  if (NF > 0) {
    Span sp("f64_op_prep_kernel", st);
    f64_op_prep_kernel<<<(unsigned)((NF + 255) / 256), 256, 0, st>>>(NF, a.xy, a.box, o.xyf, boxf);
  }
  return build_bins(s, set, st);
}
