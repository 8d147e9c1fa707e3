// INTEGRATION.md "Option A", built for real: the host wrappers a Kaolin maintainer would put in
// place of kaolin/csrc/render/mesh/rasterization.cpp:49-168 and dibr_soft_mask.cpp:48-183 so that
// the four operators registered in kaolin/csrc/bindings.cpp:111-115 run on libdibr_b200.so.
//
// Same names, argument order, argument checks (same GPU, contiguous, sizes), return structure and
// allocation policy (outputs from the first input's options(), owned by the caching allocator) as
// the reference wrappers; the only difference is what is called after the checks: the C ABI of
// include/dibr_b200.h with raw pointers on the current CUDA stream instead of *_cuda_impl.
// Outputs are allocated with at::empty (every element is written by the kernels).
//
// Built by integration/build_binding.py (g++ against the torch headers, linked to
// kaolin_b200/csrc/libdibr_b200.so) into integration/_build/kaolin_b200_binding.so and exercised
// by tests/test_reference_wrappers.py.
#include <torch/extension.h>
#include <c10/cuda/CUDAGuard.h>
#include <c10/cuda/CUDAStream.h>

#include <vector>

#include "dibr_b200.h"

namespace {

// AT_DISPATCH_FLOATING_TYPES: true for double, false for float; any other type is refused in the
// reference's wording.  The other tensors' data_ptr<scalar_t>() then refuses a mixed float/double call.
bool is_double(const char* fn, const at::Tensor& t) {
  TORCH_CHECK(t.scalar_type() == at::kFloat || t.scalar_type() == at::kDouble, "\"", fn, "\" not implemented for '",
              toString(t.scalar_type()), "'");
  return t.scalar_type() == at::kDouble;
}

void check_status(const char* fn, int st) {
  TORCH_CHECK(st == 0, fn, " failed with status ", st,
              st < 0 ? " (argument error detected on the host)" : " (cudaError_t)");
}

dibr_b200_stream_t current_stream() {
  return reinterpret_cast<dibr_b200_stream_t>(at::cuda::getCurrentCUDAStream().stream());
}

// include/dibr_b200.h: every tensor pointer 16-byte aligned.  A contiguous view at a storage
// offset passes the reference's checks, so such an input is copied first.
at::Tensor aligned(const at::Tensor& t) {
  return reinterpret_cast<uintptr_t>(t.data_ptr()) % DIBR_B200_ALIGNMENT ? t.clone(at::MemoryFormat::Contiguous) : t;
}

at::Tensor workspace(const at::Tensor& like, int batch, int64_t faces, int height, int width, bool f64 = false) {
  const size_t n = f64 ? dibr_b200_workspace_bytes_f64(batch, faces, height, width)
                       : dibr_b200_workspace_bytes(batch, faces, height, width);
  TORCH_CHECK(n > 0, "libdibr_b200: unsupported problem size");
  return at::empty({static_cast<int64_t>(n)}, like.options().dtype(at::kByte));
}

}  // namespace

namespace kaolin {

// rasterization.h:23-32
std::vector<at::Tensor> packed_rasterize_forward_cuda(
    const int height, const int width, const at::Tensor face_vertices_z, const at::Tensor face_vertices_image,
    const at::Tensor face_bboxes, const at::Tensor face_features, const at::Tensor first_idx_face_per_mesh,
    const float multiplier, const float eps) {
  at::TensorArg z_arg{face_vertices_z, "face_vertices_z", 3}, xy_arg{face_vertices_image, "face_vertices_image", 4},
      bb_arg{face_bboxes, "face_bboxes", 5}, ff_arg{face_features, "face_features", 6},
      first_arg{first_idx_face_per_mesh, "first_idx_face_per_mesh", 7};
  at::checkAllSameGPU(__func__, {z_arg, xy_arg, bb_arg, ff_arg, first_arg});
  at::checkAllContiguous(__func__, {z_arg, xy_arg, bb_arg, ff_arg, first_arg});
  const int64_t num_faces = face_vertices_z.size(0);
  const int batch = static_cast<int>(first_idx_face_per_mesh.size(0)) - 1;
  const int D = static_cast<int>(face_features.size(2));
  at::checkSize(__func__, z_arg, {num_faces, 3});
  at::checkSize(__func__, xy_arg, {num_faces, 3, 2});
  at::checkSize(__func__, bb_arg, {num_faces, 4});
  at::checkSize(__func__, ff_arg, {num_faces, 3, D});
  at::checkSize(__func__, first_arg, {batch + 1});
  const bool f64 = is_double(__func__, face_vertices_z);
  const at::cuda::OptionalCUDAGuard guard(at::device_of(face_vertices_z));
  const at::Tensor z = aligned(face_vertices_z), xy = aligned(face_vertices_image), bb = aligned(face_bboxes),
                   ff = aligned(face_features), first = aligned(first_idx_face_per_mesh);
  auto opt = face_vertices_z.options();
  at::Tensor idx = at::empty({batch, height, width}, opt.dtype(at::kLong));
  at::Tensor w = at::empty({batch, height, width, 3}, opt);
  at::Tensor out = at::empty({batch, height, width, D}, opt);
  at::Tensor ws = workspace(face_vertices_z, batch, num_faces, height, width, f64);
  if (f64) {
    check_status(__func__, dibr_b200_packed_rasterize_forward_f64(
        batch, num_faces, height, width, D, z.data_ptr<double>(), xy.data_ptr<double>(),
        bb.data_ptr<double>(), ff.data_ptr<double>(), first.data_ptr<int64_t>(),
        multiplier, eps, out.data_ptr<double>(), idx.data_ptr<int64_t>(), w.data_ptr<double>(), ws.data_ptr(),
        static_cast<size_t>(ws.numel()), current_stream()));
    return {out, idx, w};
  }
  check_status(__func__, dibr_b200_packed_rasterize_forward(
      batch, num_faces, height, width, D, z.data_ptr<float>(), xy.data_ptr<float>(),
      bb.data_ptr<float>(), ff.data_ptr<float>(), first.data_ptr<int64_t>(),
      multiplier, eps, out.data_ptr<float>(), idx.data_ptr<int64_t>(), w.data_ptr<float>(), ws.data_ptr(),
      static_cast<size_t>(ws.numel()), current_stream()));
  return {out, idx, w};
}

// rasterization.h:34-41
std::vector<at::Tensor> rasterize_backward_cuda(
    const at::Tensor grad_interpolated_features, const at::Tensor interpolated_features,
    const at::Tensor selected_face_idx, const at::Tensor output_weights, const at::Tensor face_vertices_image,
    const at::Tensor face_features, const float eps) {
  at::TensorArg g_arg{grad_interpolated_features, "grad_interpolated_features", 1},
      i_arg{interpolated_features, "interpolated_features", 2}, idx_arg{selected_face_idx, "selected_face_idx", 3},
      w_arg{output_weights, "output_weights", 4}, xy_arg{face_vertices_image, "face_vertices_image", 5},
      ff_arg{face_features, "face_features", 6};
  at::checkAllSameGPU(__func__, {g_arg, i_arg, idx_arg, w_arg, xy_arg, ff_arg});
  at::checkAllContiguous(__func__, {g_arg, i_arg, idx_arg, w_arg, xy_arg, ff_arg});
  const int batch = static_cast<int>(grad_interpolated_features.size(0));
  const int height = static_cast<int>(grad_interpolated_features.size(1));
  const int width = static_cast<int>(grad_interpolated_features.size(2));
  const int D = static_cast<int>(grad_interpolated_features.size(3));
  const int F = static_cast<int>(face_vertices_image.size(1));
  at::checkSize(__func__, i_arg, {batch, height, width, D});
  at::checkSize(__func__, idx_arg, {batch, height, width});
  at::checkSize(__func__, w_arg, {batch, height, width, 3});
  at::checkSize(__func__, xy_arg, {batch, F, 3, 2});
  at::checkSize(__func__, ff_arg, {batch, F, 3, D});
  const bool f64 = is_double(__func__, grad_interpolated_features);
  const at::cuda::OptionalCUDAGuard guard(at::device_of(grad_interpolated_features));
  const at::Tensor g = aligned(grad_interpolated_features), idx = aligned(selected_face_idx),
                   w = aligned(output_weights), xy = aligned(face_vertices_image), ff = aligned(face_features);
  at::Tensor g_xy = at::empty_like(face_vertices_image);
  at::Tensor g_ff = at::empty_like(face_features);
  if (f64) {
    check_status(__func__, dibr_b200_rasterize_backward_f64(
        batch, F, height, width, D, g.data_ptr<double>(), idx.data_ptr<int64_t>(), w.data_ptr<double>(),
        xy.data_ptr<double>(), ff.data_ptr<double>(), eps, g_xy.data_ptr<double>(), g_ff.data_ptr<double>(),
        current_stream()));
    return {g_xy, g_ff};
  }
  // the fused entry point with a workspace takes the row-walk scatter kernel
  at::Tensor ws = workspace(face_vertices_image, batch, static_cast<int64_t>(batch) * F, height, width);
  check_status(__func__, dibr_b200_backward(
      batch, F, height, width, D, g.data_ptr<float>(), nullptr,
      idx.data_ptr<int64_t>(), w.data_ptr<float>(), nullptr,
      xy.data_ptr<float>(), ff.data_ptr<float>(), 1.f, eps, 0.f, 0.f, 0,
      g_xy.data_ptr<float>(), g_ff.data_ptr<float>(), ws.data_ptr(), static_cast<size_t>(ws.numel()), 0,
      current_stream()));
  return {g_xy, g_ff};
}

// dibr_soft_mask.h:23-30
std::vector<at::Tensor> dibr_soft_mask_forward_cuda(
    const at::Tensor face_vertices_image, const at::Tensor face_large_bboxes, const at::Tensor selected_face_idx,
    const float sigmainv, const int knum, const float multiplier) {
  at::TensorArg xy_arg{face_vertices_image, "face_vertices_image", 1}, bb_arg{face_large_bboxes, "face_bboxes", 2},
      idx_arg{selected_face_idx, "selected_face_idx", 3};
  at::checkAllSameGPU(__func__, {xy_arg, bb_arg, idx_arg});
  at::checkAllContiguous(__func__, {xy_arg, bb_arg, idx_arg});
  const int batch = static_cast<int>(face_vertices_image.size(0));
  const int F = static_cast<int>(face_vertices_image.size(1));
  const int height = static_cast<int>(selected_face_idx.size(1));
  const int width = static_cast<int>(selected_face_idx.size(2));
  at::checkSize(__func__, xy_arg, {batch, F, 3, 2});
  at::checkSize(__func__, bb_arg, {batch, F, 4});
  at::checkSize(__func__, idx_arg, {batch, height, width});
  const bool f64 = is_double(__func__, face_vertices_image);
  const at::cuda::OptionalCUDAGuard guard(at::device_of(face_vertices_image));
  const at::Tensor xy = aligned(face_vertices_image), bb = aligned(face_large_bboxes), idx = aligned(selected_face_idx);
  auto opt = face_vertices_image.options();
  at::Tensor soft = at::empty({batch, height, width}, opt);
  at::Tensor prob = at::empty({batch, height, width, knum}, opt);
  at::Tensor cidx = at::empty({batch, height, width, knum}, opt.dtype(at::kLong));
  at::Tensor ctype = at::empty({batch, height, width, knum}, opt.dtype(at::kByte));
  at::Tensor ws = workspace(face_vertices_image, batch, static_cast<int64_t>(batch) * F, height, width, f64);
  if (f64) {
    check_status(__func__, dibr_b200_soft_mask_forward_f64(
        batch, F, height, width, knum, xy.data_ptr<double>(), bb.data_ptr<double>(),
        idx.data_ptr<int64_t>(), sigmainv, multiplier, soft.data_ptr<double>(), prob.data_ptr<double>(),
        cidx.data_ptr<int64_t>(), ctype.data_ptr<uint8_t>(), ws.data_ptr(), static_cast<size_t>(ws.numel()),
        current_stream()));
    return {soft, prob, cidx, ctype};
  }
  check_status(__func__, dibr_b200_soft_mask_forward(
      batch, F, height, width, knum, xy.data_ptr<float>(), bb.data_ptr<float>(),
      idx.data_ptr<int64_t>(), sigmainv, multiplier, soft.data_ptr<float>(), prob.data_ptr<float>(),
      cidx.data_ptr<int64_t>(), ctype.data_ptr<uint8_t>(), ws.data_ptr(), static_cast<size_t>(ws.numel()),
      current_stream()));
  return {soft, prob, cidx, ctype};
}

// dibr_soft_mask.h:32-42
at::Tensor dibr_soft_mask_backward_cuda(
    const at::Tensor grad_soft_mask, const at::Tensor soft_mask, const at::Tensor selected_face_idx,
    const at::Tensor close_face_prob, const at::Tensor close_face_idx, const at::Tensor close_face_dist_type,
    const at::Tensor face_vertices_image, const float sigmainv, const float multiplier) {
  at::TensorArg g_arg{grad_soft_mask, "grad_soft_mask", 1}, s_arg{soft_mask, "soft_mask", 2},
      idx_arg{selected_face_idx, "selected_face_idx", 3}, p_arg{close_face_prob, "close_face_prob", 4},
      ci_arg{close_face_idx, "close_face_idx", 5}, ct_arg{close_face_dist_type, "close_face_dist_type", 6},
      xy_arg{face_vertices_image, "face_vertices_image", 7};
  at::checkAllSameGPU(__func__, {g_arg, s_arg, idx_arg, p_arg, ci_arg, ct_arg, xy_arg});
  at::checkAllContiguous(__func__, {g_arg, s_arg, idx_arg, p_arg, ci_arg, ct_arg, xy_arg});
  const int batch = static_cast<int>(face_vertices_image.size(0));
  const int F = static_cast<int>(face_vertices_image.size(1));
  const int height = static_cast<int>(selected_face_idx.size(1));
  const int width = static_cast<int>(selected_face_idx.size(2));
  const int knum = static_cast<int>(close_face_idx.size(3));
  at::checkSize(__func__, g_arg, {batch, height, width});
  at::checkSize(__func__, s_arg, {batch, height, width});
  at::checkSize(__func__, idx_arg, {batch, height, width});
  at::checkSize(__func__, p_arg, {batch, height, width, knum});
  at::checkSize(__func__, ci_arg, {batch, height, width, knum});
  at::checkSize(__func__, ct_arg, {batch, height, width, knum});
  at::checkSize(__func__, xy_arg, {batch, F, 3, 2});
  const bool f64 = is_double(__func__, face_vertices_image);
  const at::cuda::OptionalCUDAGuard guard(at::device_of(grad_soft_mask));
  const at::Tensor g = aligned(grad_soft_mask), soft = aligned(soft_mask), idx = aligned(selected_face_idx),
                   prob = aligned(close_face_prob), cidx = aligned(close_face_idx),
                   ctype = aligned(close_face_dist_type), xy = aligned(face_vertices_image);
  at::Tensor g_xy = at::empty_like(face_vertices_image);
  if (f64) {
    check_status(__func__, dibr_b200_soft_mask_backward_f64(
        batch, F, height, width, knum, g.data_ptr<double>(), soft.data_ptr<double>(),
        idx.data_ptr<int64_t>(), prob.data_ptr<double>(), cidx.data_ptr<int64_t>(),
        ctype.data_ptr<uint8_t>(), xy.data_ptr<double>(), sigmainv, multiplier,
        g_xy.data_ptr<double>(), current_stream()));
    return g_xy;
  }
  check_status(__func__, dibr_b200_soft_mask_backward(
      batch, F, height, width, knum, g.data_ptr<float>(), soft.data_ptr<float>(),
      idx.data_ptr<int64_t>(), prob.data_ptr<float>(), cidx.data_ptr<int64_t>(),
      ctype.data_ptr<uint8_t>(), xy.data_ptr<float>(), sigmainv, multiplier,
      g_xy.data_ptr<float>(), current_stream()));
  return g_xy;
}

}  // namespace kaolin

// kaolin/csrc/bindings.cpp:111-115
PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
  m.def("packed_rasterize_forward_cuda", &kaolin::packed_rasterize_forward_cuda);
  m.def("rasterize_backward_cuda", &kaolin::rasterize_backward_cuda);
  m.def("dibr_soft_mask_forward_cuda", &kaolin::dibr_soft_mask_forward_cuda);
  m.def("dibr_soft_mask_backward_cuda", &kaolin::dibr_soft_mask_backward_cuda);
}
