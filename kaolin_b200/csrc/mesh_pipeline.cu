// mesh_pipeline.cu — the steps immediately before and after the DIB-R rasterizer in every
// caller (SURVEY.md §8f rank 1 and 2), as single sm_100a kernels behind the C ABI of
// include/dibr_b200.h:
//
//   prepare_vertices   kaolin/render/mesh/utils.py:129-175 = camera transform
//                      (camera/legacy.py:22-37 or padded @ camera_transform), perspective
//                      divide (camera/legacy.py:120-138), index_vertices_by_faces x2
//                      (ops/mesh/mesh.py:54-76) and unit face normals
//                      (ops/mesh/trianglemesh.py:314-338): the reference runs ~8 PyTorch
//                      kernels and materialises (B,V,3), (B,V,2) intermediates; here one
//                      kernel gathers the 3 vertices of a face, transforms them in registers
//                      and writes the three per-face tensors; the backward scatters straight
//                      to the (B,V,3) camera-space vertex gradient.
//   texture_mapping    kaolin/render/mesh/utils.py:22-79 (clamp, [0,1] -> [-1,1], y flip,
//                      grid_sample(align_corners=False, padding_mode='border')) forward and
//                      backward (wrt the texture and wrt the coordinates).
//   mask_iou           kaolin/metrics/render.py:18-41 forward (per-view sums, one pass) and
//                      backward (element-wise).
// All of it is HBM-bound streaming work: coalesced loads/stores, no shared-memory staging
// needed, grids sized by the element count.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/dibr_b200.h"

namespace {

// Any tensor pointer not DIBR_B200_ALIGNMENT-byte aligned (NULL is aligned).  Texture coordinates
// and their gradient are read and written as float2; the rule is the same for every entry point.
template <typename... P>
bool misaligned(P... p) { return ((((uintptr_t)p) | ... | (uintptr_t)0) & (DIBR_B200_ALIGNMENT - 1)) != 0; }

// ---------------------------------------------------------------------------
// prepare_vertices
struct Cam {
  // mode 0: vc = [p, 1] @ T (T: 4x3 row-major);  mode 1: vc = R (p - t)
  int mode;
  const float* transform;  // (B,4,3)
  const float* rot;        // (B,3,3)
  const float* trans;      // (B,3)
  float px, py, pz;        // camera_proj (3,1)
};

__device__ __forceinline__ void cam_point(const Cam& c, int b, const float p[3], float vc[3]) {
  if (c.mode == 0) {
    const float* T = c.transform + (size_t)b * 12;
#pragma unroll
    for (int j = 0; j < 3; ++j)
      vc[j] = __fmaf_rn(p[2], __ldg(T + 6 + j), __fmaf_rn(p[1], __ldg(T + 3 + j), __fmaf_rn(p[0], __ldg(T + j), __ldg(T + 9 + j))));
  } else {
    const float* R = c.rot + (size_t)b * 9;
    const float* t = c.trans + (size_t)b * 3;
    const float d0 = p[0] - __ldg(t), d1 = p[1] - __ldg(t + 1), d2 = p[2] - __ldg(t + 2);
#pragma unroll
    for (int j = 0; j < 3; ++j)   // translated @ R^T  ->  vc_j = sum_i d_i R[j][i]
      vc[j] = __fmaf_rn(d2, __ldg(R + 3 * j + 2), __fmaf_rn(d1, __ldg(R + 3 * j + 1), d0 * __ldg(R + 3 * j)));
  }
}

__global__ void __launch_bounds__(256) prepare_vertices_fwd_kernel(
    int B, int V, int F, const float* __restrict__ vertices, const int64_t* __restrict__ faces, Cam cam,
    float* __restrict__ fvc, float* __restrict__ fvi, float* __restrict__ fn) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)B * F) return;
  const int b = (int)(i / F), f = (int)(i - (int64_t)b * F);
  float vc[3][3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const int64_t vid = __ldg(faces + (int64_t)f * 3 + k);
    const float* vp = vertices + ((int64_t)b * V + vid) * 3;
    const float p[3] = {__ldg(vp), __ldg(vp + 1), __ldg(vp + 2)};
    cam_point(cam, b, p, vc[k]);
  }
  float* o = fvc + i * 9;
#pragma unroll
  for (int k = 0; k < 3; ++k) { o[3 * k] = vc[k][0]; o[3 * k + 1] = vc[k][1]; o[3 * k + 2] = vc[k][2]; }
  float* o2 = fvi + i * 6;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    // perspective_camera: (p * proj).xy / (p * proj).z
    const float zz = vc[k][2] * cam.pz;
    o2[2 * k] = __fdiv_rn(vc[k][0] * cam.px, zz);
    o2[2 * k + 1] = __fdiv_rn(vc[k][1] * cam.py, zz);
  }
  // face_normals(unit=True): cross(v1 - v0, v2 - v0) / (|.| + 1e-10)
  const float e0[3] = {vc[1][0] - vc[0][0], vc[1][1] - vc[0][1], vc[1][2] - vc[0][2]};
  const float e1[3] = {vc[2][0] - vc[0][0], vc[2][1] - vc[0][1], vc[2][2] - vc[0][2]};
  const float cx = e0[1] * e1[2] - e0[2] * e1[1];
  const float cy = e0[2] * e1[0] - e0[0] * e1[2];
  const float cz = e0[0] * e1[1] - e0[1] * e1[0];
  const float len = sqrtf(cx * cx + cy * cy + cz * cz) + 1e-10f;
  float* o3 = fn + i * 3;
  o3[0] = __fdiv_rn(cx, len); o3[1] = __fdiv_rn(cy, len); o3[2] = __fdiv_rn(cz, len);
}

// Gradient wrt the CAMERA-SPACE vertices (B,V,3), scattered with float atomics (a vertex is
// shared by ~6 faces); the linear map back to world-space vertices / camera parameters is a
// (B,V,3) x (3,3) product the host does with a library GEMM.
__global__ void __launch_bounds__(256) prepare_vertices_bwd_kernel(
    int B, int V, int F, const float* __restrict__ vertices, const int64_t* __restrict__ faces, Cam cam,
    const float* __restrict__ g_fvc, const float* __restrict__ g_fvi, const float* __restrict__ g_fn,
    float* __restrict__ g_vc) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)B * F) return;
  const int b = (int)(i / F), f = (int)(i - (int64_t)b * F);
  float vc[3][3];
  int64_t vid[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    vid[k] = __ldg(faces + (int64_t)f * 3 + k);
    const float* vp = vertices + ((int64_t)b * V + vid[k]) * 3;
    const float p[3] = {__ldg(vp), __ldg(vp + 1), __ldg(vp + 2)};
    cam_point(cam, b, p, vc[k]);
  }
  float g[3][3];
#pragma unroll
  for (int k = 0; k < 3; ++k) { g[k][0] = 0.f; g[k][1] = 0.f; g[k][2] = 0.f; }
  if (g_fvc) {
    const float* gp = g_fvc + i * 9;
#pragma unroll
    for (int k = 0; k < 3; ++k) { g[k][0] += __ldg(gp + 3 * k); g[k][1] += __ldg(gp + 3 * k + 1); g[k][2] += __ldg(gp + 3 * k + 2); }
  }
  if (g_fvi) {
    const float* gp = g_fvi + i * 6;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const float gx = __ldg(gp + 2 * k), gy = __ldg(gp + 2 * k + 1);
      const float zz = vc[k][2] * cam.pz;
      const float inv = 1.0f / zz;
      const float x2 = vc[k][0] * cam.px * inv, y2 = vc[k][1] * cam.py * inv;
      g[k][0] += gx * cam.px * inv;
      g[k][1] += gy * cam.py * inv;
      g[k][2] -= (gx * x2 + gy * y2) * cam.pz * inv;
    }
  }
  if (g_fn) {
    const float e0[3] = {vc[1][0] - vc[0][0], vc[1][1] - vc[0][1], vc[1][2] - vc[0][2]};
    const float e1[3] = {vc[2][0] - vc[0][0], vc[2][1] - vc[0][1], vc[2][2] - vc[0][2]};
    const float c[3] = {e0[1] * e1[2] - e0[2] * e1[1], e0[2] * e1[0] - e0[0] * e1[2], e0[0] * e1[1] - e0[1] * e1[0]};
    const float L = sqrtf(c[0] * c[0] + c[1] * c[1] + c[2] * c[2]);
    const float Le = L + 1e-10f;
    const float gn[3] = {__ldg(g_fn + i * 3), __ldg(g_fn + i * 3 + 1), __ldg(g_fn + i * 3 + 2)};
    // n = c / (L + eps):  g_c = g_n / (L+eps) - c (c . g_n) / (L (L+eps)^2)
    const float dot = c[0] * gn[0] + c[1] * gn[1] + c[2] * gn[2];
    const float k2 = L > 0.f ? dot / (L * Le * Le) : 0.f;
    const float gc[3] = {gn[0] / Le - c[0] * k2, gn[1] / Le - c[1] * k2, gn[2] / Le - c[2] * k2};
    // c = e0 x e1:  g_e0 = e1 x g_c,  g_e1 = g_c x e0
    const float ge0[3] = {e1[1] * gc[2] - e1[2] * gc[1], e1[2] * gc[0] - e1[0] * gc[2], e1[0] * gc[1] - e1[1] * gc[0]};
    const float ge1[3] = {gc[1] * e0[2] - gc[2] * e0[1], gc[2] * e0[0] - gc[0] * e0[2], gc[0] * e0[1] - gc[1] * e0[0]};
#pragma unroll
    for (int j = 0; j < 3; ++j) { g[1][j] += ge0[j]; g[2][j] += ge1[j]; g[0][j] -= ge0[j] + ge1[j]; }
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    float* o = g_vc + ((int64_t)b * V + vid[k]) * 3;
    atomicAdd(o, g[k][0]); atomicAdd(o + 1, g[k][1]); atomicAdd(o + 2, g[k][2]);
  }
}

// ---------------------------------------------------------------------------
// texture_mapping: coordinates (B,N,2) in [0,1] (OpenGL: y up), texture (B,C,Ht,Wt), out (B,N,C).
__device__ __forceinline__ void tex_source(float u, float v, int Wt, int Ht, float& ix, float& iy, bool& in_u, bool& in_v) {
  // utils.py:66-69: clamp to [0,1], *2-1, flip y; grid_sample unnormalise (align_corners=False):
  // ((g + 1) * size - 1) / 2, then 'border' padding clips to [0, size-1]
  in_u = u > 0.f && u < 1.f;       // d clamp / du (torch.clamp passes the gradient inside the open interval... and at the bounds)
  in_v = v > 0.f && v < 1.f;
  const float cu = fminf(fmaxf(u, 0.f), 1.f), cv = fminf(fmaxf(v, 0.f), 1.f);
  const float gx = cu * 2.f - 1.f, gy = -(cv * 2.f - 1.f);
  ix = ((gx + 1.f) * (float)Wt - 1.f) * 0.5f;
  iy = ((gy + 1.f) * (float)Ht - 1.f) * 0.5f;
}

template <bool NEAREST>
__global__ void __launch_bounds__(256) texture_mapping_fwd_kernel(int B, int64_t N, int C, int Ht, int Wt,
                                                                 const float* __restrict__ uv,
                                                                 const float* __restrict__ tex,
                                                                 float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)B * N) return;
  const int b = (int)(i / N);
  const float2 t = __ldg(reinterpret_cast<const float2*>(uv) + i);
  float ix, iy; bool iu, iv;
  tex_source(t.x, t.y, Wt, Ht, ix, iy, iu, iv);
  ix = fminf(fmaxf(ix, 0.f), (float)(Wt - 1));
  iy = fminf(fmaxf(iy, 0.f), (float)(Ht - 1));
  const float* tb = tex + (size_t)b * C * Ht * Wt;
  float* o = out + i * C;
  if (NEAREST) {
    const int x = (int)nearbyintf(ix), y = (int)nearbyintf(iy);
    for (int c = 0; c < C; ++c) o[c] = __ldg(tb + ((size_t)c * Ht + y) * Wt + x);
  } else {
    const float fx = floorf(ix), fy = floorf(iy);
    const int x0 = (int)fx, y0 = (int)fy;
    const int x1 = min(x0 + 1, Wt - 1), y1 = min(y0 + 1, Ht - 1);
    const float wx1 = ix - fx, wy1 = iy - fy, wx0 = 1.f - wx1, wy0 = 1.f - wy1;
    for (int c = 0; c < C; ++c) {
      const float* p = tb + (size_t)c * Ht * Wt;
      const float a = __ldg(p + (size_t)y0 * Wt + x0), bb = __ldg(p + (size_t)y0 * Wt + x1);
      const float cc = __ldg(p + (size_t)y1 * Wt + x0), d = __ldg(p + (size_t)y1 * Wt + x1);
      o[c] = a * (wx0 * wy0) + bb * (wx1 * wy0) + cc * (wx0 * wy1) + d * (wx1 * wy1);
    }
  }
}

template <bool NEAREST>
__global__ void __launch_bounds__(256) texture_mapping_bwd_kernel(int B, int64_t N, int C, int Ht, int Wt,
                                                                 const float* __restrict__ uv,
                                                                 const float* __restrict__ tex,
                                                                 const float* __restrict__ g_out,
                                                                 float* __restrict__ g_tex,
                                                                 float* __restrict__ g_uv) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)B * N) return;
  const int b = (int)(i / N);
  const float2 t = __ldg(reinterpret_cast<const float2*>(uv) + i);
  float ix, iy; bool iu, iv;
  tex_source(t.x, t.y, Wt, Ht, ix, iy, iu, iv);
  // 'border' clip: gradient passes only strictly inside (grid_sample's clip_coordinates_set_grad)
  const bool cx_in = ix > 0.f && ix < (float)(Wt - 1), cy_in = iy > 0.f && iy < (float)(Ht - 1);
  ix = fminf(fmaxf(ix, 0.f), (float)(Wt - 1));
  iy = fminf(fmaxf(iy, 0.f), (float)(Ht - 1));
  const size_t plane = (size_t)Ht * Wt;
  const float* tb = tex + (size_t)b * C * plane;
  float* gb = g_tex ? g_tex + (size_t)b * C * plane : nullptr;
  const float* go = g_out + i * C;
  if (NEAREST) {
    const int x = (int)nearbyintf(ix), y = (int)nearbyintf(iy);
    if (gb) for (int c = 0; c < C; ++c) atomicAdd(gb + c * plane + (size_t)y * Wt + x, __ldg(go + c));
    if (g_uv) reinterpret_cast<float2*>(g_uv)[i] = make_float2(0.f, 0.f);
    return;
  }
  const float fx = floorf(ix), fy = floorf(iy);
  const int x0 = (int)fx, y0 = (int)fy;
  const int x1 = min(x0 + 1, Wt - 1), y1 = min(y0 + 1, Ht - 1);
  const bool x1_in = x0 + 1 <= Wt - 1, y1_in = y0 + 1 <= Ht - 1;   // grid_sample drops out-of-range corners
  const float wx1 = ix - fx, wy1 = iy - fy, wx0 = 1.f - wx1, wy0 = 1.f - wy1;
  float gix = 0.f, giy = 0.f;
  for (int c = 0; c < C; ++c) {
    const float g = __ldg(go + c);
    const float* p = tb + c * plane;
    const float a = __ldg(p + (size_t)y0 * Wt + x0);
    const float bb = x1_in ? __ldg(p + (size_t)y0 * Wt + x1) : 0.f;
    const float cc = y1_in ? __ldg(p + (size_t)y1 * Wt + x0) : 0.f;
    const float d = (x1_in && y1_in) ? __ldg(p + (size_t)y1 * Wt + x1) : 0.f;
    gix += g * ((bb - a) * wy0 + (d - cc) * wy1);
    giy += g * ((cc - a) * wx0 + (d - bb) * wx1);
    if (gb) {
      float* q = gb + c * plane;
      atomicAdd(q + (size_t)y0 * Wt + x0, g * wx0 * wy0);
      if (x1_in) atomicAdd(q + (size_t)y0 * Wt + x1, g * wx1 * wy0);
      if (y1_in) atomicAdd(q + (size_t)y1 * Wt + x0, g * wx0 * wy1);
      if (x1_in && y1_in) atomicAdd(q + (size_t)y1 * Wt + x1, g * wx1 * wy1);
    }
  }
  if (g_uv) {
    // d ix / du = 2 * Wt / 2 = Wt (inside the clamp and the border clip); d iy / dv = -Ht
    const float du = (iu && cx_in) ? gix * (float)Wt : 0.f;
    const float dv = (iv && cy_in) ? -giy * (float)Ht : 0.f;
    reinterpret_cast<float2*>(g_uv)[i] = make_float2(du, dv);
  }
}

// ---------------------------------------------------------------------------
// mask_iou: per-view sums of lhs*rhs and lhs+rhs-lhs*rhs (one streaming pass, warp shuffle +
// one atomic per CTA), then the scalar loss; backward is element-wise.
__global__ void __launch_bounds__(256) mask_iou_sums_kernel(int64_t HW, const float* __restrict__ lhs,
                                                           const float* __restrict__ rhs, float* __restrict__ sums) {
  const int b = blockIdx.y;
  const float* l = lhs + (size_t)b * HW;
  const float* r = rhs + (size_t)b * HW;
  float up = 0.f, down = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < HW; i += (int64_t)gridDim.x * blockDim.x) {
    const float a = __ldg(l + i), c = __ldg(r + i);
    const float m = a * c;
    up += m;
    down += (a + c) - m;
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) { up += __shfl_xor_sync(0xffffffffu, up, d); down += __shfl_xor_sync(0xffffffffu, down, d); }
  __shared__ float su[8], sd[8];
  if ((threadIdx.x & 31) == 0) { su[threadIdx.x >> 5] = up; sd[threadIdx.x >> 5] = down; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float u = 0.f, d = 0.f;
    for (int w = 0; w < 8; ++w) { u += su[w]; d += sd[w]; }
    atomicAdd(sums + 2 * b, u);
    atomicAdd(sums + 2 * b + 1, d);
  }
}

__global__ void mask_iou_loss_kernel(int B, const float* __restrict__ sums, float* __restrict__ loss) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    float acc = 0.f;
    for (int b = 0; b < B; ++b) acc += sums[2 * b] / (sums[2 * b + 1] + 1e-10f);
    *loss = 1.0f - acc / (float)B;
  }
}

// d loss / d lhs = -(1/B) * (rhs * (down+eps) - up * (1 - rhs)) / (down+eps)^2
__global__ void __launch_bounds__(256) mask_iou_bwd_kernel(int B, int64_t HW, const float* __restrict__ lhs,
                                                          const float* __restrict__ rhs,
                                                          const float* __restrict__ sums,
                                                          const float* __restrict__ g_loss,
                                                          float* __restrict__ g_lhs, float* __restrict__ g_rhs) {
  const int b = blockIdx.y;
  const float up = sums[2 * b], de = sums[2 * b + 1] + 1e-10f;
  const float k = -__ldg(g_loss) / ((float)B * de * de);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < HW; i += (int64_t)gridDim.x * blockDim.x) {
    const size_t o = (size_t)b * HW + i;
    const float a = __ldg(lhs + o), c = __ldg(rhs + o);
    if (g_lhs) g_lhs[o] = k * (c * de - up * (1.f - c));
    if (g_rhs) g_rhs[o] = k * (a * de - up * (1.f - a));
  }
}

}  // namespace

extern "C" {

static int make_cam(Cam& c, const float* camera_transform, const float* camera_rot, const float* camera_trans,
                    const float* camera_proj_host) {
  if (!camera_proj_host) return DIBR_B200_EINVAL;
  if (camera_transform) {
    if (camera_rot || camera_trans) return DIBR_B200_EINVAL;
    c.mode = 0;
  } else {
    if (!camera_rot || !camera_trans) return DIBR_B200_EINVAL;
    c.mode = 1;
  }
  c.transform = camera_transform; c.rot = camera_rot; c.trans = camera_trans;
  c.px = camera_proj_host[0]; c.py = camera_proj_host[1]; c.pz = camera_proj_host[2];
  return 0;
}

int dibr_b200_prepare_vertices_forward(int batch, int num_vertices, int num_faces, const float* vertices,
                                       const int64_t* faces, const float* camera_transform,
                                       const float* camera_rot, const float* camera_trans,
                                       const float* camera_proj_host, float* face_vertices_camera,
                                       float* face_vertices_image, float* face_normals,
                                       dibr_b200_stream_t stream) {
  if (batch <= 0 || num_vertices <= 0 || num_faces < 0) return DIBR_B200_EINVAL;
  if (!vertices || !faces || !face_vertices_camera || !face_vertices_image || !face_normals) return DIBR_B200_EINVAL;
  if (misaligned(vertices, faces, camera_transform, camera_rot, camera_trans, face_vertices_camera,
                 face_vertices_image, face_normals))
    return DIBR_B200_EINVAL;
  Cam c;
  const int rc = make_cam(c, camera_transform, camera_rot, camera_trans, camera_proj_host);
  if (rc) return rc;
  const int64_t n = (int64_t)batch * num_faces;
  if (n == 0) return 0;
  prepare_vertices_fwd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      batch, num_vertices, num_faces, vertices, faces, c, face_vertices_camera, face_vertices_image, face_normals);
  return (int)cudaGetLastError();
}

int dibr_b200_prepare_vertices_backward(int batch, int num_vertices, int num_faces, const float* vertices,
                                        const int64_t* faces, const float* camera_transform,
                                        const float* camera_rot, const float* camera_trans,
                                        const float* camera_proj_host, const float* grad_face_vertices_camera,
                                        const float* grad_face_vertices_image, const float* grad_face_normals,
                                        float* grad_vertices_camera, dibr_b200_stream_t stream) {
  if (batch <= 0 || num_vertices <= 0 || num_faces < 0) return DIBR_B200_EINVAL;
  if (!vertices || !faces || !grad_vertices_camera) return DIBR_B200_EINVAL;
  if (misaligned(vertices, faces, camera_transform, camera_rot, camera_trans, grad_face_vertices_camera,
                 grad_face_vertices_image, grad_face_normals, grad_vertices_camera))
    return DIBR_B200_EINVAL;
  Cam c;
  const int rc = make_cam(c, camera_transform, camera_rot, camera_trans, camera_proj_host);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(grad_vertices_camera, 0, (size_t)batch * num_vertices * 3 * sizeof(float), st);
  if (e != cudaSuccess) return (int)e;
  const int64_t n = (int64_t)batch * num_faces;
  if (n == 0) return 0;
  prepare_vertices_bwd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(
      batch, num_vertices, num_faces, vertices, faces, c, grad_face_vertices_camera, grad_face_vertices_image,
      grad_face_normals, grad_vertices_camera);
  return (int)cudaGetLastError();
}

int dibr_b200_texture_mapping_forward(int batch, int64_t num_points, int channels, int tex_height, int tex_width,
                                      const float* texture_coordinates, const float* texture_maps, int nearest,
                                      float* out, dibr_b200_stream_t stream) {
  if (batch <= 0 || num_points < 0 || channels <= 0 || tex_height <= 0 || tex_width <= 0) return DIBR_B200_EINVAL;
  if (!texture_coordinates || !texture_maps || !out) return DIBR_B200_EINVAL;
  if (misaligned(texture_coordinates, texture_maps, out)) return DIBR_B200_EINVAL;
  const int64_t n = (int64_t)batch * num_points;
  if (n == 0) return 0;
  const unsigned blocks = (unsigned)((n + 255) / 256);
  if (nearest) texture_mapping_fwd_kernel<true><<<blocks, 256, 0, (cudaStream_t)stream>>>(batch, num_points, channels, tex_height, tex_width, texture_coordinates, texture_maps, out);
  else texture_mapping_fwd_kernel<false><<<blocks, 256, 0, (cudaStream_t)stream>>>(batch, num_points, channels, tex_height, tex_width, texture_coordinates, texture_maps, out);
  return (int)cudaGetLastError();
}

int dibr_b200_texture_mapping_backward(int batch, int64_t num_points, int channels, int tex_height, int tex_width,
                                       const float* texture_coordinates, const float* texture_maps, int nearest,
                                       const float* grad_out, float* grad_texture_maps,
                                       float* grad_texture_coordinates, dibr_b200_stream_t stream) {
  if (batch <= 0 || num_points < 0 || channels <= 0 || tex_height <= 0 || tex_width <= 0) return DIBR_B200_EINVAL;
  if (!texture_coordinates || !texture_maps || !grad_out) return DIBR_B200_EINVAL;
  if (misaligned(texture_coordinates, texture_maps, grad_out, grad_texture_maps, grad_texture_coordinates))
    return DIBR_B200_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  if (grad_texture_maps) {
    cudaError_t e = cudaMemsetAsync(grad_texture_maps, 0, (size_t)batch * channels * tex_height * tex_width * sizeof(float), st);
    if (e != cudaSuccess) return (int)e;
  }
  const int64_t n = (int64_t)batch * num_points;
  if (n == 0) return 0;
  const unsigned blocks = (unsigned)((n + 255) / 256);
  if (nearest) texture_mapping_bwd_kernel<true><<<blocks, 256, 0, st>>>(batch, num_points, channels, tex_height, tex_width, texture_coordinates, texture_maps, grad_out, grad_texture_maps, grad_texture_coordinates);
  else texture_mapping_bwd_kernel<false><<<blocks, 256, 0, st>>>(batch, num_points, channels, tex_height, tex_width, texture_coordinates, texture_maps, grad_out, grad_texture_maps, grad_texture_coordinates);
  return (int)cudaGetLastError();
}

int dibr_b200_mask_iou_forward(int batch, int64_t pixels_per_view, const float* lhs_mask, const float* rhs_mask,
                               float* sums, float* loss, dibr_b200_stream_t stream) {
  if (batch <= 0 || batch > 65535 || pixels_per_view <= 0 || !lhs_mask || !rhs_mask || !sums || !loss) return DIBR_B200_EINVAL;
  if (misaligned(lhs_mask, rhs_mask, sums, loss)) return DIBR_B200_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(sums, 0, (size_t)batch * 2 * sizeof(float), st);
  if (e != cudaSuccess) return (int)e;
  int64_t bx = (pixels_per_view + 256 * 8 - 1) / (256 * 8);
  if (bx > 1184) bx = 1184;   // 148 SMs x 8
  mask_iou_sums_kernel<<<dim3((unsigned)bx, (unsigned)batch), 256, 0, st>>>(pixels_per_view, lhs_mask, rhs_mask, sums);
  mask_iou_loss_kernel<<<1, 32, 0, st>>>(batch, sums, loss);
  return (int)cudaGetLastError();
}

int dibr_b200_mask_iou_backward(int batch, int64_t pixels_per_view, const float* lhs_mask, const float* rhs_mask,
                                const float* sums, const float* grad_loss, float* grad_lhs, float* grad_rhs,
                                dibr_b200_stream_t stream) {
  if (batch <= 0 || batch > 65535 || pixels_per_view <= 0 || !lhs_mask || !rhs_mask || !sums || !grad_loss) return DIBR_B200_EINVAL;
  if (misaligned(lhs_mask, rhs_mask, sums, grad_loss, grad_lhs, grad_rhs)) return DIBR_B200_EINVAL;
  int64_t bx = (pixels_per_view + 256 * 8 - 1) / (256 * 8);
  if (bx > 1184) bx = 1184;
  mask_iou_bwd_kernel<<<dim3((unsigned)bx, (unsigned)batch), 256, 0, (cudaStream_t)stream>>>(
      batch, pixels_per_view, lhs_mask, rhs_mask, sums, grad_loss, grad_lhs, grad_rhs);
  return (int)cudaGetLastError();
}

}  // extern "C"
