// class Frame -- "Holds the processed data from a time t: original frames, 3d points, edge map" (reference
// include/Frame.h:5,41, where the class is an empty shell, Frame.h:42-46).  Here it has a body: one device-resident
// slot holding the frame's edge points (ref role, get_aX standalone/utils.cpp:201-281) and its normalised edge
// distance transform (now role, get_distance_transform utils.cpp:38-83), at every pyramid level.
#pragma once
#include <stdexcept>
#include <string>
#include <vector>

#include "../ea_cabi.h"
#include "Mat.h"

namespace ea {

inline void check(int rc, const char* what) {
  if (rc != EA_OK) throw std::runtime_error(std::string(what) + ": " + ea_last_error());
}

// One CUDA context shared by the facade objects of a thread (created on first use; device from EA_DEVICE or 0).
inline ea_context* default_context(int device = -1) {
  static thread_local ea_context* ctx = nullptr;
  if (!ctx) check(ea_create(device < 0 ? 0 : device, &ctx), "ea_create");
  return ctx;
}

}  // namespace ea

class Frame {
 public:
  Frame() = default;                                   // reference signature (include/Frame.h:45)
  explicit Frame(const ea_frame_params& p, ea_context* ctx = nullptr) { init(p, ctx); }
  Frame(const Frame&) = delete;
  Frame& operator=(const Frame&) = delete;
  ~Frame() { if (fs_) ea_frameset_destroy(fs_); }

  void init(const ea_frame_params& p, ea_context* ctx = nullptr) {
    if (fs_) { ea_frameset_destroy(fs_); fs_ = nullptr; }
    ctx_ = ctx ? ctx : ea::default_context();
    params_ = p;
    ea::check(ea_frameset_create(ctx_, &p, 1, &fs_), "ea_frameset_create");
  }
  bool valid() const { return fs_ != nullptr; }
  const ea_frame_params& params() const { return params_; }
  ea_frameset* handle() const { return fs_; }
  ea_context* context() const { return ctx_; }

  // rgb: 8UC3 (BGR as cv::imread gives it) or 8UC1 (gray / IR; preprocessed exactly as the BGR image (g, g, g)); any other
  // type throws.  depth: 16UC1 raw units or 32FC1 metres (SolveEA.cpp:27,68), converted to the frameset's own depth_type
  // when they differ; depth may be null for a now-only frame.  The "Z==0 -> 1.0" rule of SolveEA.cpp:69 is a frameset
  // parameter (zero_depth_to_one) applied on the device.
  template <class MatT>
  void set(const MatT& rgb, const MatT* depth, int roles) {
    if (!fs_) throw std::runtime_error("Frame::set before init");
    if (rgb.rows != params_.height || rgb.cols != params_.width) throw std::runtime_error("Frame::set: image size differs from ea_frame_params");
    const int type = rgb.type();
    if (type != ea::U8C3 && type != ea::U8C1) throw std::runtime_error("Frame::set: the image must be 8UC3 (BGR) or 8UC1 (gray)");
    const size_t W = size_t(params_.width), H = size_t(params_.height);
    const void* dptr = nullptr;
    if (depth && depth->data) {
      const bool want_f32 = params_.depth_type == EA_DEPTH_F32, have_f32 = depth->type() == ea::F32C1;
      depth_.resize(W * H * (want_f32 ? 4 : 2));
      for (size_t y = 0; y < H; ++y) {
        const unsigned char* row = depth->data + y * size_t(depth->step);
        for (size_t x = 0; x < W; ++x) {
          if (want_f32) {
            const float z = have_f32 ? reinterpret_cast<const float*>(row)[x] : float(double(reinterpret_cast<const uint16_t*>(row)[x]) / params_.depth_scale);
            reinterpret_cast<float*>(depth_.data())[y * W + x] = z;
          } else {
            uint16_t v;
            if (have_f32) { const double r = double(reinterpret_cast<const float*>(row)[x]) * params_.depth_scale + 0.5; v = r <= 0 ? 0 : (r >= 65535.0 ? 65535 : uint16_t(r)); }
            else v = reinterpret_cast<const uint16_t*>(row)[x];
            reinterpret_cast<uint16_t*>(depth_.data())[y * W + x] = v;
          }
        }
      }
      dptr = depth_.data();
    }
    const int32_t slot = 0;
    // the rows are read where they lie: the upload skips the padding between them
    const ea_image_layout layout{type == ea::U8C3 ? EA_IMAGE_BGR8 : EA_IMAGE_GRAY8, 0, int64_t(size_t(rgb.step)), 0};
    ea::check(ea_frameset_preprocess_image_host(fs_, 1, &slot, &layout, rgb.data, dptr, nullptr, nullptr, roles),
              "ea_frameset_preprocess_image_host");
    ea::check(ea_sync(ctx_), "ea_sync");
  }

  int numEdgePoints(int level = 0) const { int n = 0; ea::check(ea_frameset_get_num_points(fs_, 0, level, &n), "get_num_points"); return n; }
  // list_edge_ref as {u, v, depth (raw units or metres per depth_type), 1} rows (reference: 3xN X,Y,Z doubles, SolveEA.h:63)
  std::vector<float> edgePoints(int level = 0) const {
    int n = numEdgePoints(level);
    std::vector<float> p(size_t(n) * 4);
    if (n) ea::check(ea_frameset_get_points(fs_, 0, level, p.data(), n, &n), "get_points");
    return p;
  }
  // now_dist_transform (SolveEA.h:59) at the given level, row-major
  std::vector<float> distanceTransform(int level = 0) const {
    int w = 0, h = 0;
    ea::check(ea_frameset_level_geometry(fs_, level, &w, &h, nullptr), "level_geometry");
    std::vector<float> d(size_t(w) * h);
    ea::check(ea_frameset_get_dt(fs_, 0, level, d.data()), "get_dt");
    return d;
  }

 private:
  ea_context* ctx_ = nullptr;
  ea_frameset* fs_ = nullptr;
  ea_frame_params params_{};
  std::vector<unsigned char> depth_;
};
