// bpc_baseline_b200._C -- the thin PyTorch C++ extension over the C ABI of include/bpc_b200.h.
//
// Every operator checks its tensors (TORCH_CHECK: dtype, shape, device, contiguity -> RuntimeError), allocates its
// outputs and scratch with the caching allocator, looks up the current CUDA stream and calls ONE extern "C" launcher
// of libbpc_b200.so.  Nothing here computes, allocates outside torch, or synchronises, so the operators are safe to
// capture into CUDA graphs.  They are registered with the dispatcher (torch.ops.bpc_b200.*, CUDA + Meta kernels), so
// FakeTensor / torch.compile tracing sees shapes and dtypes without running anything.
//
// Reference call surface each op stands for: see the comments of include/bpc_b200.h (file:line under /root/reference).
#include <ATen/ATen.h>
#include <c10/cuda/CUDAGuard.h>
#include <c10/cuda/CUDAStream.h>
#include <torch/library.h>

#include <cmath>
#include <tuple>
#include <vector>

#include "bpc_b200.h"

namespace {

using at::Tensor;

void chk(const Tensor& t, at::ScalarType dt, const char* name, int64_t ndim = -1) {
    TORCH_CHECK(t.is_cuda(), name, " must be a CUDA tensor (the hot path has no CPU fallback)");
    TORCH_CHECK(t.scalar_type() == dt, name, " must be ", c10::toString(dt), ", got ", c10::toString(t.scalar_type()));
    TORCH_CHECK(t.is_contiguous(), name, " must be contiguous");
    TORCH_CHECK(ndim < 0 || t.dim() == ndim, name, " must have ", ndim, " dimensions, got ", t.dim());
}

void rc_check(int rc, const char* what) { TORCH_CHECK(rc == BPC_OK, what, ": ", bpc_error_string(rc), " (", rc, ")"); }

void* cur_stream(const Tensor& t) { return (void*)c10::cuda::getCurrentCUDAStream(t.device().index()).stream(); }

Tensor scratch(const Tensor& like, size_t bytes) {
    return at::empty({(int64_t)(bytes ? bytes : 16)}, like.options().dtype(at::kByte));
}

// ---- PoseEstimator._match for S scenes (process_pose.py:144-188) --------------------------------------------------
std::tuple<Tensor, Tensor, Tensor, Tensor, Tensor, Tensor> match_triangulate(const Tensor& Ks, const Tensor& RTs, const Tensor& centers,
                                                                             const Tensor& counts, double threshold,
                                                                             c10::optional<double> reproj_thresh, bool want_F) {
    chk(Ks, at::kFloat, "Ks", 4); chk(RTs, at::kDouble, "RTs", 4); chk(centers, at::kDouble, "centers", 4); chk(counts, at::kInt, "counts", 2);
    const int64_t S = centers.size(0), D = centers.size(2);
    TORCH_CHECK(Ks.sizes() == at::IntArrayRef({S, 3, 3, 3}) && RTs.sizes() == at::IntArrayRef({S, 3, 4, 4}) &&
                centers.sizes() == at::IntArrayRef({S, 3, D, 2}) && counts.sizes() == at::IntArrayRef({S, 3}),
                "expected Ks [S,3,3,3], RTs [S,3,4,4], centers [S,3,Dmax,2], counts [S,3]");
    TORCH_CHECK(D >= 1 && D <= BPC_MAX_DET, "Dmax must be in 1..", BPC_MAX_DET);
    const c10::cuda::CUDAGuard guard(Ks.device());
    const auto oi = counts.options();
    Tensor idx = at::empty({S, D, 3}, oi), n = at::empty({S}, oi);
    Tensor cost = at::empty({S, D}, Ks.options());
    Tensor X = at::empty({S, D, 3}, RTs.options()), reproj = at::empty({S, D, 3}, RTs.options());
    Tensor F = want_F ? at::empty({S, 3, 3, 3}, RTs.options()) : at::empty({0}, RTs.options());
    const size_t wsb = bpc_match_workspace_bytes((int)S, (int)D);
    Tensor ws = scratch(Ks, wsb);
    rc_check(bpc_match_triangulate(Ks.data_ptr<float>(), RTs.data_ptr<double>(), centers.data_ptr<double>(), counts.data_ptr<int32_t>(),
                                   (int)S, (int)D, (float)threshold, reproj_thresh.has_value() ? 1 : 0, reproj_thresh.value_or(0.0),
                                   idx.data_ptr<int32_t>(), n.data_ptr<int32_t>(), cost.data_ptr<float>(), X.data_ptr<double>(),
                                   reproj.data_ptr<double>(), want_F ? F.data_ptr<double>() : nullptr,
                                   wsb ? ws.data_ptr() : nullptr, wsb, cur_stream(Ks)),
             "bpc_match_triangulate");
    return {idx, n, cost, X, reproj, F};
}

std::tuple<Tensor, Tensor, Tensor, Tensor, Tensor, Tensor> match_triangulate_meta(const Tensor& Ks, const Tensor& RTs, const Tensor& centers,
                                                                                  const Tensor& counts, double, c10::optional<double>, bool want_F) {
    const auto S = centers.sym_size(0), D = centers.sym_size(2);
    const auto oi = counts.options();
    return {at::empty_symint({S, D, 3}, oi), at::empty_symint({S}, oi), at::empty_symint({S, D}, Ks.options()),
            at::empty_symint({S, D, 3}, RTs.options()), at::empty_symint({S, D, 3}, RTs.options()),
            want_F ? at::empty_symint({S, 3, 3, 3}, RTs.options()) : at::empty({0}, RTs.options())};
}

// ---- centres of int boxes (process_pose.py:134-136) ----------------------------------------------------------------
Tensor box_centers(const Tensor& boxes) {
    chk(boxes, at::kInt, "boxes");
    TORCH_CHECK(boxes.dim() >= 1 && boxes.size(-1) == 4, "boxes must be [..., 4]");
    const c10::cuda::CUDAGuard guard(boxes.device());
    auto shape = boxes.sizes().vec();
    shape.back() = 2;
    Tensor out = at::empty(shape, boxes.options().dtype(at::kDouble));
    rc_check(bpc_box_centers(boxes.data_ptr<int32_t>(), (int)(boxes.numel() / 4), out.data_ptr<double>(), cur_stream(boxes)), "bpc_box_centers");
    return out;
}

Tensor box_centers_meta(const Tensor& boxes) {
    auto shape = boxes.sym_sizes().vec();
    shape.back() = 2;
    return at::empty_symint(shape, boxes.options().dtype(at::kDouble));
}

// ---- ROI list of every matched detection (process_pose.py:195-201) -------------------------------------------------
std::tuple<Tensor, Tensor> build_rois(const Tensor& boxes, const Tensor& idx, const Tensor& n, const Tensor& image_of_scene) {
    chk(boxes, at::kInt, "boxes", 4); chk(idx, at::kInt, "idx", 3); chk(n, at::kInt, "n", 1); chk(image_of_scene, at::kInt, "image_of_scene", 2);
    const int64_t S = boxes.size(0), D = boxes.size(2), K = idx.size(1);
    TORCH_CHECK(boxes.size(1) == 3 && boxes.size(3) == 4 && idx.size(0) == S && idx.size(2) == 3 && n.size(0) == S &&
                image_of_scene.size(0) == S && image_of_scene.size(1) == 3, "expected boxes [S,3,Dmax,4], idx [S,Kmax,3], n [S], image_of_scene [S,3]");
    const c10::cuda::CUDAGuard guard(boxes.device());
    Tensor rois = at::empty({S * K * 3, 5}, boxes.options()), offs = at::empty({S + 1}, boxes.options());
    rc_check(bpc_build_rois(boxes.data_ptr<int32_t>(), idx.data_ptr<int32_t>(), n.data_ptr<int32_t>(), image_of_scene.data_ptr<int32_t>(),
                            (int)S, (int)D, (int)K, offs.data_ptr<int32_t>(), rois.data_ptr<int32_t>(), cur_stream(boxes)), "bpc_build_rois");
    return {rois, offs};
}

std::tuple<Tensor, Tensor> build_rois_meta(const Tensor& boxes, const Tensor& idx, const Tensor&, const Tensor&) {
    return {at::empty_symint({boxes.sym_size(0) * idx.sym_size(1) * 3, 5}, boxes.options()), at::empty_symint({boxes.sym_size(0) + 1}, boxes.options())};
}

// ---- to_tensor + normalize as a table (process_pose.py:207-209) ----------------------------------------------------
Tensor normalise_lut(at::ArrayRef<double> mean, at::ArrayRef<double> std_, at::Device device) {
    TORCH_CHECK(mean.size() == 3 && std_.size() == 3, "mean and std must have three entries");
    TORCH_CHECK(device.is_cuda(), "device must be a CUDA device");
    const c10::cuda::CUDAGuard guard(device);
    Tensor lut = at::empty({3, 256}, at::TensorOptions().dtype(at::kFloat).device(device));
    const float m[3] = {(float)mean[0], (float)mean[1], (float)mean[2]}, s[3] = {(float)std_[0], (float)std_[1], (float)std_[2]};
    rc_check(bpc_normalise_lut(m, s, lut.data_ptr<float>(), cur_stream(lut)), "bpc_normalise_lut");
    return lut;
}

// ---- crop -> letterbox -> RGB -> normalise (data_utils.py:34-44, process_pose.py:199-209) --------------------------
void crop_common(const Tensor& images, const Tensor& rois, int64_t T, at::ArrayRef<int64_t> fill, const c10::optional<Tensor>& n_rois) {
    chk(images, at::kByte, "images", 4); chk(rois, at::kInt, "rois", 2);
    TORCH_CHECK(images.size(3) == 3 && rois.size(1) == 5, "images must be [B,H,W,3] and rois [R,5]");
    TORCH_CHECK(T >= 1 && T <= BPC_MAX_TARGET, "target size must be in 1..", BPC_MAX_TARGET);
    TORCH_CHECK(fill.size() == 3, "fill must have three entries");
    if (n_rois.has_value()) chk(*n_rois, at::kInt, "n_rois");
}

std::tuple<Tensor, Tensor> roi_crop(const Tensor& images, const Tensor& rois, int64_t T, at::ArrayRef<int64_t> fill, bool swap_rb, const Tensor& lut,
                                    const c10::optional<Tensor>& n_rois, int64_t roi_first, const c10::optional<Tensor>& out_) {
    crop_common(images, rois, T, fill, n_rois);
    chk(lut, at::kFloat, "lut", 2);
    TORCH_CHECK(lut.size(0) == 3 && lut.size(1) == 256, "lut must be [3,256]");
    const int64_t R = rois.size(0);
    const c10::cuda::CUDAGuard guard(images.device());
    Tensor out;
    if (out_.has_value()) {
        out = *out_;
        chk(out, at::kFloat, "out", 4);
        TORCH_CHECK(out.size(0) >= R && out.size(1) == 3 && out.size(2) == T && out.size(3) == T, "out must be [>=R,3,T,T]");
    } else {
        out = at::empty({R, 3, T, T}, lut.options());
    }
    Tensor status = at::empty({R}, rois.options());
    const uint8_t f[3] = {(uint8_t)fill[0], (uint8_t)fill[1], (uint8_t)fill[2]};
    const int64_t step = 32768;                                           // bounds the scratch (tap descriptors per ROI)
    const size_t wsb = bpc_roi_crop_workspace_bytes((int)std::min(R, step), (int)T);
    Tensor ws = scratch(images, wsb);
    for (int64_t lo = 0; lo < R; lo += step) {
        const int64_t r = std::min(step, R - lo);
        rc_check(bpc_roi_crop(images.data_ptr<uint8_t>(), (int)images.size(0), (int)images.size(1), (int)images.size(2),
                              rois.data_ptr<int32_t>() + lo * 5, (int)r, n_rois.has_value() ? n_rois->data_ptr<int32_t>() : nullptr,
                              (int)(roi_first + lo), (int)T, f, swap_rb ? 1 : 0, lut.data_ptr<float>(), out.data_ptr<float>() + lo * 3 * T * T,
                              status.data_ptr<int32_t>() + lo, ws.data_ptr(), wsb, cur_stream(images)), "bpc_roi_crop");
    }
    return {out, status};
}

std::tuple<Tensor, Tensor> roi_crop_meta(const Tensor& images, const Tensor& rois, int64_t T, at::ArrayRef<int64_t>, bool, const Tensor& lut,
                                         const c10::optional<Tensor>&, int64_t, const c10::optional<Tensor>& out_) {
    Tensor out = out_.has_value() ? *out_ : at::empty_symint({rois.sym_size(0), 3, T, T}, lut.options());
    return {out, at::empty_symint({rois.sym_size(0)}, rois.options())};
}

// bfloat16 channels-last variant: logical shape [R,3,T,T], memory [R,T,T,3] (what a bf16 tensor-core pose head reads)
std::tuple<Tensor, Tensor> roi_crop_bf16(const Tensor& images, const Tensor& rois, int64_t T, at::ArrayRef<int64_t> fill, bool swap_rb,
                                         const Tensor& lut, const c10::optional<Tensor>& n_rois, int64_t roi_first) {
    crop_common(images, rois, T, fill, n_rois);
    chk(lut, at::kFloat, "lut", 2);
    TORCH_CHECK(lut.size(0) == 3 && lut.size(1) == 256, "lut must be [3,256]");
    const int64_t R = rois.size(0);
    const c10::cuda::CUDAGuard guard(images.device());
    Tensor out = at::empty({R, 3, T, T}, lut.options().dtype(at::kBFloat16), at::MemoryFormat::ChannelsLast);
    Tensor status = at::empty({R}, rois.options());
    const uint8_t f[3] = {(uint8_t)fill[0], (uint8_t)fill[1], (uint8_t)fill[2]};
    const int64_t step = 32768;
    const size_t wsb = bpc_roi_crop_workspace_bytes((int)std::min(R, step), (int)T);
    Tensor ws = scratch(images, wsb);
    for (int64_t lo = 0; lo < R; lo += step) {
        const int64_t r = std::min(step, R - lo);
        rc_check(bpc_roi_crop_bf16(images.data_ptr<uint8_t>(), (int)images.size(0), (int)images.size(1), (int)images.size(2),
                                   rois.data_ptr<int32_t>() + lo * 5, (int)r, n_rois.has_value() ? n_rois->data_ptr<int32_t>() : nullptr,
                                   (int)(roi_first + lo), (int)T, f, swap_rb ? 1 : 0, lut.data_ptr<float>(),
                                   static_cast<char*>(out.data_ptr()) + lo * 3 * T * T * 2, status.data_ptr<int32_t>() + lo, ws.data_ptr(), wsb,
                                   cur_stream(images)), "bpc_roi_crop_bf16");
    }
    return {out, status};
}

std::tuple<Tensor, Tensor> roi_crop_bf16_meta(const Tensor& images, const Tensor& rois, int64_t T, at::ArrayRef<int64_t>, bool, const Tensor& lut,
                                              const c10::optional<Tensor>&, int64_t) {
    return {at::empty_symint({rois.sym_size(0), 3, T, T}, lut.options().dtype(at::kBFloat16)), at::empty_symint({rois.sym_size(0)}, rois.options())};
}

std::tuple<Tensor, Tensor> roi_crop_u8(const Tensor& images, const Tensor& rois, int64_t T, at::ArrayRef<int64_t> fill,
                                       const c10::optional<Tensor>& n_rois, int64_t roi_first) {
    crop_common(images, rois, T, fill, n_rois);
    const int64_t R = rois.size(0);
    const c10::cuda::CUDAGuard guard(images.device());
    Tensor out = at::empty({R, T, T, 3}, images.options());
    Tensor status = at::empty({R}, rois.options());
    const uint8_t f[3] = {(uint8_t)fill[0], (uint8_t)fill[1], (uint8_t)fill[2]};
    const int64_t step = 32768;
    const size_t wsb = bpc_roi_crop_workspace_bytes((int)std::min(R, step), (int)T);
    Tensor ws = scratch(images, wsb);
    for (int64_t lo = 0; lo < R; lo += step) {
        const int64_t r = std::min(step, R - lo);
        rc_check(bpc_roi_crop_u8(images.data_ptr<uint8_t>(), (int)images.size(0), (int)images.size(1), (int)images.size(2),
                                 rois.data_ptr<int32_t>() + lo * 5, (int)r, n_rois.has_value() ? n_rois->data_ptr<int32_t>() : nullptr,
                                 (int)(roi_first + lo), (int)T, f, out.data_ptr<uint8_t>() + lo * T * T * 3, status.data_ptr<int32_t>() + lo,
                                 ws.data_ptr(), wsb, cur_stream(images)), "bpc_roi_crop_u8");
    }
    return {out, status};
}

std::tuple<Tensor, Tensor> roi_crop_u8_meta(const Tensor& images, const Tensor& rois, int64_t T, at::ArrayRef<int64_t>,
                                            const c10::optional<Tensor>&, int64_t) {
    return {at::empty_symint({rois.sym_size(0), T, T, 3}, images.options()), at::empty_symint({rois.sym_size(0)}, rois.options())};
}

// ---- training-side ColorJitter + to_tensor + normalize (bpc/utils/data_utils.py, torchvision ColorJitter) -----------
Tensor color_jitter(const Tensor& canvases, const Tensor& order, const Tensor& factors, bool swap_rb, const Tensor& lut) {
    chk(canvases, at::kByte, "canvases", 4); chk(order, at::kInt, "order", 2); chk(factors, at::kFloat, "factors", 2); chk(lut, at::kFloat, "lut", 2);
    const int64_t n = canvases.size(0), T = canvases.size(1);
    TORCH_CHECK(canvases.size(2) == T && canvases.size(3) == 3 && order.size(0) == n && order.size(1) == 4 && factors.size(0) == n &&
                factors.size(1) == 4, "expected canvases [n,T,T,3], order [n,4] and factors [n,4]");
    TORCH_CHECK(T >= 1 && T <= BPC_MAX_TARGET, "target size must be in 1..", BPC_MAX_TARGET);
    TORCH_CHECK(lut.size(0) == 3 && lut.size(1) == 256, "lut must be [3,256]");
    TORCH_CHECK(order.device() == canvases.device() && factors.device() == canvases.device() && lut.device() == canvases.device(),
                "canvases, order, factors and lut must be on the same device");
    const c10::cuda::CUDAGuard guard(canvases.device());
    Tensor out = at::empty({n, 3, T, T}, lut.options());
    rc_check(bpc_color_jitter(canvases.data_ptr<uint8_t>(), (int)n, (int)T, order.data_ptr<int32_t>(), factors.data_ptr<float>(), swap_rb ? 1 : 0,
                              lut.data_ptr<float>(), out.data_ptr<float>(), cur_stream(canvases)), "bpc_color_jitter");
    return out;
}

Tensor color_jitter_meta(const Tensor& canvases, const Tensor&, const Tensor&, bool, const Tensor& lut) {
    return at::empty_symint({canvases.sym_size(0), 3, canvases.sym_size(1), canvases.sym_size(2)}, lut.options());
}

// ---- pose records for the final gather (SURVEY.md 8e) --------------------------------------------------------------
Tensor pack_records(const Tensor& idx, const Tensor& n, const Tensor& cost, const Tensor& X, const Tensor& reproj, const Tensor& scene_offset,
                    int64_t offset_div) {
    chk(idx, at::kInt, "idx", 3); chk(n, at::kInt, "n", 1); chk(cost, at::kFloat, "cost", 2); chk(X, at::kDouble, "X", 3);
    chk(reproj, at::kDouble, "reproj", 3); chk(scene_offset, at::kInt, "scene_offset", 1);
    const int64_t S = idx.size(0), K = idx.size(1);
    TORCH_CHECK(scene_offset.size(0) == S + 1 && n.size(0) == S && cost.size(0) == S && cost.size(1) == K, "shape mismatch");
    const c10::cuda::CUDAGuard guard(idx.device());
    Tensor buf = at::empty({(int64_t)bpc_pack_records_bytes((int)S, (int)K)}, idx.options().dtype(at::kByte));
    rc_check(bpc_pack_records(idx.data_ptr<int32_t>(), n.data_ptr<int32_t>(), cost.data_ptr<float>(), X.data_ptr<double>(), reproj.data_ptr<double>(),
                              scene_offset.data_ptr<int32_t>(), (int)offset_div, (int)S, (int)K, buf.data_ptr(), cur_stream(idx)), "bpc_pack_records");
    return buf;
}

Tensor fundamental(const Tensor& Ks, const Tensor& RTs) {
    chk(Ks, at::kFloat, "Ks", 4); chk(RTs, at::kDouble, "RTs", 4);
    const int64_t S = Ks.size(0);
    TORCH_CHECK(Ks.sizes() == at::IntArrayRef({S, 3, 3, 3}) && RTs.sizes() == at::IntArrayRef({S, 3, 4, 4}), "expected Ks [S,3,3,3], RTs [S,3,4,4]");
    const c10::cuda::CUDAGuard guard(Ks.device());
    Tensor F = at::empty({S, 3, 3, 3}, RTs.options());
    rc_check(bpc_fundamental(Ks.data_ptr<float>(), RTs.data_ptr<double>(), (int)S, F.data_ptr<double>(), cur_stream(Ks)), "bpc_fundamental");
    return F;
}

int64_t abi_version() { return bpc_abi_version(); }

}  // namespace

TORCH_LIBRARY(bpc_b200, m) {
    m.def("match_triangulate(Tensor Ks, Tensor RTs, Tensor centers, Tensor counts, float threshold=30., float? reproj_thresh=None, "
          "bool want_F=False) -> (Tensor, Tensor, Tensor, Tensor, Tensor, Tensor)");
    m.def("box_centers(Tensor boxes) -> Tensor");
    m.def("build_rois(Tensor boxes, Tensor idx, Tensor n, Tensor image_of_scene) -> (Tensor, Tensor)");
    m.def("normalise_lut(float[] mean, float[] std, Device device) -> Tensor", &normalise_lut);
    m.def("roi_crop(Tensor images, Tensor rois, int T, int[] fill, bool swap_rb, Tensor lut, Tensor? n_rois=None, int roi_first=0, "
          "Tensor(a!)? out=None) -> (Tensor(a!), Tensor)");
    m.def("roi_crop_u8(Tensor images, Tensor rois, int T, int[] fill, Tensor? n_rois=None, int roi_first=0) -> (Tensor, Tensor)");
    m.def("roi_crop_bf16(Tensor images, Tensor rois, int T, int[] fill, bool swap_rb, Tensor lut, Tensor? n_rois=None, int roi_first=0) -> (Tensor, Tensor)");
    m.def("color_jitter(Tensor canvases, Tensor order, Tensor factors, bool swap_rb, Tensor lut) -> Tensor");
    m.def("pack_records(Tensor idx, Tensor n, Tensor cost, Tensor X, Tensor reproj, Tensor scene_offset, int offset_div=3) -> Tensor");
    m.def("fundamental(Tensor Ks, Tensor RTs) -> Tensor");
    m.def("abi_version() -> int", &abi_version);
}

TORCH_LIBRARY_IMPL(bpc_b200, CUDA, m) {
    m.impl("match_triangulate", &match_triangulate);
    m.impl("box_centers", &box_centers);
    m.impl("build_rois", &build_rois);
    m.impl("roi_crop", &roi_crop);
    m.impl("roi_crop_u8", &roi_crop_u8);
    m.impl("roi_crop_bf16", &roi_crop_bf16);
    m.impl("color_jitter", &color_jitter);
    m.impl("pack_records", &pack_records);
    m.impl("fundamental", &fundamental);
}

TORCH_LIBRARY_IMPL(bpc_b200, Meta, m) {
    m.impl("match_triangulate", &match_triangulate_meta);
    m.impl("box_centers", &box_centers_meta);
    m.impl("build_rois", &build_rois_meta);
    m.impl("roi_crop", &roi_crop_meta);
    m.impl("roi_crop_u8", &roi_crop_u8_meta);
    m.impl("roi_crop_bf16", &roi_crop_bf16_meta);
    m.impl("color_jitter", &color_jitter_meta);
}
