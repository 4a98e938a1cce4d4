// api.cu -- the C-ABI of libkvfe.so (include/kvfe.h): context set-up, host-side constant tables
// and the kernel sequences behind every entry point.  No CPU compute path exists here: every
// function either launches the CUDA kernels or fails.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <random>
#include <map>
#include <limits>
#include <vector>

#include <cuda.h>           // CUtensorMap types only: the encoder is resolved through the runtime, libcuda is not linked

#include "kvfe_internal.h"

static thread_local char g_create_err[512] = "";
// The pipeline keeps one CUDA stream per camera stream busy (kvfe_pipeline: 32 streams at the benchmark
// batch).  The driver multiplexes streams onto CUDA_DEVICE_MAX_CONNECTIONS hardware work queues (default
// 8): with more busy streams than queues, step graphs queued on different streams serialise behind each
// other (measured on B200: 1.28 ms per 32-stream pass at 8 queues, 0.68 ms at 32).  The variable is read
// when the CUDA context is created, so it is set when the library is loaded, unless the caller chose a value.
__attribute__((constructor)) static void kvfe_on_load() { setenv("CUDA_DEVICE_MAX_CONNECTIONS", "32", 0); }


static int set_err(kvfe_ctx* ctx, int code, const char* fmt, ...) {
  char* dst = ctx ? ctx->err : g_create_err;
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(dst, 512, fmt, ap);
  va_end(ap);
  return code;
}
int kvfe_set_err(kvfe_ctx* ctx, int code, const char* fmt, ...) {
  char* dst = ctx ? ctx->err : g_create_err;
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(dst, 512, fmt, ap);
  va_end(ap);
  return code;
}

#define CU(call)                                                                              \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess)                                                                    \
      return set_err(ctx, KVFE_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                     __FILE__, __LINE__);                                                     \
  } while (0)

template <typename T>
static cudaError_t dmalloc(T** p, size_t n) {
  cudaError_t e = cudaMalloc((void**)p, n * sizeof(T));
  if (e == cudaSuccess) e = cudaMemset(*p, 0, n * sizeof(T));
  return e;
}

extern "C" void kvfe_config_default(kvfe_config* c) {
  memset(c, 0, sizeof(*c));
  c->width = 752; c->height = 480; c->batch = 1; c->max_keypoints = 0;
  // params/Euroc/FrontendParams.yaml
  c->klt_win_size = 24; c->klt_max_iter = 30; c->klt_max_level = 4; c->klt_eps = 0.1;
  c->max_feature_track_age = 25;
  c->min_nr_mono_inliers = 10; c->min_nr_stereo_inliers = 5;
  c->ransac_threshold_mono = 1e-6; c->ransac_threshold_stereo = 1.0;
  c->ransac_max_iterations = 100; c->ransac_probability = 0.995; c->ransac_randomize = 0;
  c->ransac_use_1point_stereo = 1; c->ransac_use_2point_mono = 1; c->pose_2d2d_algorithm = 1;
  c->optical_flow_predictor_type = 1; c->disparity_threshold = 0.5; c->rnd_libstdcxx = 0;
  c->max_features_per_frame = 300; c->enable_subpixel_corner_refinement = 1;
  c->subpix_max_iters = 40; c->subpix_epsilon = 0.001; c->subpix_window_size = 10; c->subpix_zero_zone = -1;
  c->enable_non_max_suppression = 1; c->non_max_suppression_type = 6; c->min_distance = 20;
  c->max_nr_keypoints_before_anms = 2000; c->nr_horizontal_bins = 7; c->nr_vertical_bins = 5;
  for (int i = 0; i < 64; ++i) c->binning_mask[i] = 1;
  c->quality_level = 0.001; c->block_size = 3; c->use_harris_detector = 0; c->k = 0.04;
  c->sobel_cpu_tail_start = -1;
  c->tolerance_template_matching = 0.15; c->templ_cols = 101; c->templ_rows = 11; c->stripe_extra_rows = 0;
  c->min_point_dist = 0.5; c->max_point_dist = 10.0; c->subpixel_refinement_stereo = 0;
  c->min_intra_keyframe_time_ns = 200000000LL; c->max_intra_keyframe_time_ns = 5000000000LL;
  c->min_number_features = 0; c->use_stereo_tracking = 1; c->use_ransac = 1;
  c->max_disparity_since_lkf = 1000.0;
  c->mesh_2d = 0; c->subdiv_bounding_factor = 0.f;
  c->optimize_2d2d_pose_from_inliers = 0; c->optimize_3d3d_pose_from_inliers = 0; c->equalize_image = 0; c->frontend_type = 0;
  // CameraParams::DepthParams defaults (CameraParams.h:136-145), metric float depth
  c->depth.depth_type = KVFE_DEPTH_F32; c->depth.virtual_baseline = 1.0e-2f; c->depth.depth_to_meters = 1.0f;
  c->depth.min_depth = 0.0f; c->depth.max_depth = 10.0f;
}

static int check_depth_params(kvfe_ctx* ctx, const kvfe_depth_params* dp);
// DepthFrame.cpp:76-77: the cv::inRange bounds in float; for a CV_16UC1 image static_cast<uint16_t> (clamped here)
static void depth_mask_bounds(const kvfe_depth_params& dp, float* lo, float* hi, unsigned int* lo16, unsigned int* hi16) {
  *lo = dp.min_depth * 1.0f / dp.depth_to_meters; *hi = dp.max_depth * 1.0f / dp.depth_to_meters;
  auto to_u16 = [](float v) -> unsigned int { return !(v > 0.f) ? 0u : (v >= 65535.f ? 65535u : (unsigned int)v); };
  *lo16 = to_u16(*lo); *hi16 = to_u16(*hi);
}

static size_t round_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// P[:, :3] * R with cv::gemm's 3x3 path, then cv::invert's 3x3 cofactor formula
static void make_cam(CamModel& c, const double* K, const double* D, const double* R, const double* P, int model) {
  c.model = model; c.pad = 0;
  c.fx = K[0]; c.fy = K[4]; c.cx = K[2]; c.cy = K[5];
  c.k1 = D[0]; c.k2 = D[1]; c.p1 = D[2]; c.p2 = D[3];
  for (int i = 0; i < 9; ++i) c.R[i] = R[i];
  for (int i = 0; i < 12; ++i) c.P[i] = P[i];
  for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) c.PP[3 * i + j] = P[4 * i + j];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j)
      c.RP[3 * i + j] = (c.PP[3 * i] * R[j] + c.PP[3 * i + 1] * R[3 + j]) + c.PP[3 * i + 2] * R[6 + j];
  const double* S = c.RP;
  double d = S[0] * (S[4] * S[8] - S[5] * S[7]) - S[1] * (S[3] * S[8] - S[5] * S[6]) + S[2] * (S[3] * S[7] - S[4] * S[6]);
  d = 1.0 / d;
  double* t = c.iR;
  t[0] = (S[4] * S[8] - S[5] * S[7]) * d; t[1] = (S[2] * S[7] - S[1] * S[8]) * d; t[2] = (S[1] * S[5] - S[2] * S[4]) * d;
  t[3] = (S[5] * S[6] - S[3] * S[8]) * d; t[4] = (S[0] * S[8] - S[2] * S[6]) * d; t[5] = (S[2] * S[3] - S[0] * S[5]) * d;
  t[6] = (S[3] * S[7] - S[4] * S[6]) * d; t[7] = (S[1] * S[6] - S[0] * S[7]) * d; t[8] = (S[0] * S[4] - S[1] * S[3]) * d;
}

static void packet_layout(int cap, bool mesh, size_t* off, size_t* total) {
  // per keypoint-capacity unit; the mesh holds up to 2 * cap triangles of 6 floats
  const size_t sz[KVFE_PACKET_ARRAYS] = {4, 4, 8, 4, 8, 24, 4, 4, 4, 4, 4, 4, 8, 24, 4, 4, 8, 8, 8, 8, mesh ? 48u : 0u};
  size_t o = round_up(sizeof(kvfe_packet_header), 16);
  for (int i = 0; i < KVFE_PACKET_ARRAYS; ++i) { off[i] = o; o = round_up(o + sz[i] * (size_t)cap, 16); }
  *total = o;
}

static std::vector<float> subpix_mask_table(int win) {
  // cv::cornerSubPix: mask[i][j] = (float)(exp(-y*y) * exp(-x*x)), float math (host libm expf)
  int ww = 2 * win + 1;
  std::vector<float> m((size_t)ww * ww);
  for (int i = 0; i < ww; ++i) {
    float y = (float)(i - win) / win;
    float vy = std::exp(-y * y);
    for (int j = 0; j < ww; ++j) {
      float x = (float)(j - win) / win;
      m[(size_t)i * ww + j] = (float)(vy * std::exp(-x * x));
    }
  }
  return m;
}

static std::vector<int> circle_half_widths(int r) {
  // cv::circle(..., FILLED) raster (FillCircle / Circle with fill): per-row half width
  std::vector<int> hw(2 * r + 1, -1);
  int err = 0, dx = r, dy = 0, plus = 1, minus = (r << 1) - 1;
  while (dx >= dy) {
    hw[r + dy] = std::max(hw[r + dy], dx); hw[r - dy] = std::max(hw[r - dy], dx);
    hw[r + dx] = std::max(hw[r + dx], dy); hw[r - dx] = std::max(hw[r - dx], dy);
    dy++; err += plus; plus += 2;
    int mask = (err <= 0) - 1;
    err -= minus & mask; dx += mask; minus -= mask & 2;
  }
  return hw;
}

// kvfe_create's failure path: the message goes where the caller can read it (kvfe_last_error(NULL)) and
// everything allocated so far is released
#define CUC(call)                                                                               \
  do {                                                                                          \
    cudaError_t e_ = (call);                                                                    \
    if (e_ != cudaSuccess) {                                                                    \
      set_err(nullptr, KVFE_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_),   \
              __FILE__, __LINE__);                                                              \
      kvfe_destroy(ctx);                                                                        \
      return KVFE_ERR_CUDA;                                                                     \
    }                                                                                           \
  } while (0)
// Tensor maps of the pyramid levels for the LK patch boxes (lk.cu, lk_kernel_tma): per pyramid slot and level
// one 3-D u8 tensor (x: level width, y: level height, z: stream) with row pitch lvl_pitch and stream pitch
// pyr_stride, box 48 x 28 x 1, no swizzle, zero fill outside.  cuTensorMapEncodeTiled is a driver entry point:
// it is looked up through cudaGetDriverEntryPoint.  On failure the maps stay null and LK runs lk_kernel_col.
static const void* build_lk_tensor_maps(const DevCfg& dc, unsigned char* const pyr[2]) {
  typedef CUresult (*EncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn ||
      qres != cudaDriverEntryPointSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  EncodeTiled encode = reinterpret_cast<EncodeTiled>(fn);
  std::vector<CUtensorMap> maps(2 * KVFE_MAX_LEVELS);
  memset(maps.data(), 0, maps.size() * sizeof(CUtensorMap));
  for (int slot = 0; slot < 2; ++slot)
    for (int l = 0; l < dc.n_levels; ++l) {
      const cuuint64_t dims[3] = {(cuuint64_t)dc.lvl_w[l], (cuuint64_t)dc.lvl_h[l], (cuuint64_t)dc.B};
      const cuuint64_t strides[2] = {(cuuint64_t)dc.lvl_pitch[l], (cuuint64_t)dc.pyr_stride};
      const cuuint32_t box[3] = {48, 28, 1}, estr[3] = {1, 1, 1};   // LKT_BOXW x LKT_BOXH of lk.cu
      CUresult r = encode(&maps[slot * KVFE_MAX_LEVELS + l], CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, pyr[slot] + dc.lvl_off[l], dims,
                          strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                          CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) return nullptr;
    }
  // handed to the kernel as a __grid_constant__ parameter (the documented way to give a tensor map to the TMA
  // unit); the host copy lives as long as the context
  void* h = aligned_alloc(128, maps.size() * sizeof(CUtensorMap));
  if (h) memcpy(h, maps.data(), maps.size() * sizeof(CUtensorMap));
  return h;
}

extern "C" void kvfe_destroy(kvfe_ctx* ctx);
extern "C" int kvfe_create(const kvfe_config* cfg, const kvfe_rig* rig, kvfe_ctx** out) {
  kvfe_ctx* ctx = nullptr;
  if (!cfg || !rig || !out) return set_err(nullptr, KVFE_ERR_INVALID_ARG, "null argument");
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return set_err(nullptr, KVFE_ERR_NO_DEVICE, "no CUDA device: libkvfe has no CPU path");
  const kvfe_config& c = *cfg;
  if (c.width < 64 || c.height < 64 || c.batch < 1) return set_err(nullptr, KVFE_ERR_INVALID_ARG, "bad geometry");
  if (c.klt_win_size < 3 || c.klt_win_size > 32) return set_err(nullptr, KVFE_ERR_INVALID_ARG, "klt_win_size must be in [3,32]");
  if (c.block_size != 3 || c.use_harris_detector) return set_err(nullptr, KVFE_ERR_INVALID_ARG, "only GFTT min-eigenvalue, block_size 3");
  if (c.enable_non_max_suppression && c.non_max_suppression_type != 0 && c.non_max_suppression_type != 6)
    return set_err(nullptr, KVFE_ERR_INVALID_ARG, "non_max_suppression_type must be 0 (TopN) or 6 (Binning)");
  if (c.nr_horizontal_bins * c.nr_vertical_bins > 64 || c.nr_horizontal_bins < 1 || c.nr_vertical_bins < 1)
    return set_err(nullptr, KVFE_ERR_INVALID_ARG, "at most 64 bins");
  if (c.ransac_randomize) return set_err(nullptr, KVFE_ERR_INVALID_ARG, "ransac_randomize must be 0");
  if (c.enable_subpixel_corner_refinement && (c.subpix_window_size < 1 || c.subpix_window_size > 12 || c.subpix_zero_zone >= 0))
    return set_err(nullptr, KVFE_ERR_INVALID_ARG, "subpix window must be in [1,12], zero zone -1");
  if (c.max_nr_keypoints_before_anms < 1 || c.max_nr_keypoints_before_anms > 4096)
    return set_err(nullptr, KVFE_ERR_INVALID_ARG, "max_nr_keypoints_before_anms must be in [1,4096]");
  if (c.ransac_max_iterations < 1 || c.ransac_max_iterations > KVFE_MAX_RANSAC_ITERS)
    return set_err(nullptr, KVFE_ERR_INVALID_ARG, "ransac_max_iterations out of range");
  if ((c.templ_cols & 1) == 0 || (c.templ_rows & 1) == 0) return set_err(nullptr, KVFE_ERR_INVALID_ARG, "template size must be odd");
  if (c.pose_2d2d_algorithm != 1) return set_err(nullptr, KVFE_ERR_INVALID_ARG, "pose_2d2d_algorithm must be 1 (NISTER)");
  if (c.klt_max_level < 0 || c.klt_max_level >= KVFE_MAX_LEVELS) return set_err(nullptr, KVFE_ERR_INVALID_ARG, "klt_max_level must be in [0,%d]", KVFE_MAX_LEVELS - 1);
  if (c.min_distance < 0) return set_err(nullptr, KVFE_ERR_INVALID_ARG, "min_distance must be >= 0");
  if (c.frontend_type < 0 || c.frontend_type > 2) return set_err(nullptr, KVFE_ERR_INVALID_ARG, "frontend_type must be 0 (stereo), 1 (mono) or 2 (RGB-D)");
  if (rig->distortion_model != KVFE_DISTORTION_RADTAN && rig->distortion_model != KVFE_DISTORTION_EQUIDISTANT)
    return set_err(nullptr, KVFE_ERR_INVALID_ARG, "kvfe_rig.distortion_model must be KVFE_DISTORTION_RADTAN or KVFE_DISTORTION_EQUIDISTANT (omni is not supported)");
  if (c.frontend_type == 1 && c.mesh_2d) return set_err(nullptr, KVFE_ERR_INVALID_ARG, "the 2-D mesh needs stereo matches: not available with the mono front-end");
  if (c.optimize_2d2d_pose_from_inliers || c.optimize_3d3d_pose_from_inliers)
    return set_err(nullptr, KVFE_ERR_INVALID_ARG, "optimize_{2d2d,3d3d}_pose_from_inliers (nonlinear refinement of the RANSAC pose) is not implemented");
  if (c.frontend_type == 2) {
    if (check_depth_params(nullptr, &c.depth) != KVFE_OK) return KVFE_ERR_INVALID_ARG;
    // the fake stereo camera (stereo RANSAC) and the fill (virtual disparity) must agree on fx * b (RgbdCamera.cpp:87-101)
    if (rig->baseline != (double)c.depth.virtual_baseline)
      return set_err(nullptr, KVFE_ERR_INVALID_ARG, "RGB-D: kvfe_rig.baseline (%.17g) must equal (double)depth.virtual_baseline (%.17g)",
                     rig->baseline, (double)c.depth.virtual_baseline);
    if (c.mesh_2d) return set_err(nullptr, KVFE_ERR_INVALID_ARG, "RGB-D: the 2-D mesh is not available with the RGB-D front-end");
    if (rig->distortion_model != KVFE_DISTORTION_RADTAN)
      return set_err(nullptr, KVFE_ERR_INVALID_ARG, "RGB-D: only the radial-tangential camera model is supported");
  }

  ctx = new kvfe_ctx();
  memset(ctx, 0, sizeof(*ctx));
  ctx->cfg = c; ctx->rig = *rig;
  DevCfg& dc = ctx->dc;
  DevBuf& db = ctx->db;
  dc.W = c.width; dc.H = c.height; dc.pitch = (int)round_up(c.width, 16); dc.B = c.batch;
  const int nbins = c.nr_horizontal_bins * c.nr_vertical_bins;
  int cap = c.max_keypoints;
  if (cap <= 0) {
    // a frame holds the survivors of the previous frame (<= max_features + nbins valid ones, and the
    // RANSAC outliers stay in place with landmark -1) plus up to need + nbins new corners
    cap = c.enable_non_max_suppression ? 2 * (c.max_features_per_frame + nbins) + 16
                                       : 2 * std::max(c.max_nr_keypoints_before_anms, c.max_features_per_frame) + 16;
  }
  cap = (int)round_up(cap, 32);
  dc.cap = cap;
  // pyramid geometry (cv::buildOpticalFlowPyramid stopping rule)
  {
    int w = dc.W, h = dc.H, lv = 0;
    size_t off = 0;
    for (int level = 0; level <= c.klt_max_level && level < KVFE_MAX_LEVELS; ++level) {
      dc.lvl_w[level] = w; dc.lvl_h[level] = h; dc.lvl_pitch[level] = (int)round_up(w, 16);
      dc.lvl_off[level] = off;
      off = round_up(off + (size_t)dc.lvl_pitch[level] * h, 256);
      lv = level + 1;
      w = (w + 1) / 2; h = (h + 1) / 2;
      if (w <= c.klt_win_size || h <= c.klt_win_size) break;
    }
    dc.n_levels = lv;
    dc.pyr_stride = off;
  }
  dc.img_stride = round_up((size_t)dc.pitch * dc.H, 256);
  dc.win = c.klt_win_size;
  dc.max_iter = std::min(std::max(c.klt_max_iter, 0), 100);
  { double e = std::min(std::max(c.klt_eps, 0.), 10.); dc.eps2 = e * e; }
  dc.min_eig_thr = (float)1e-4;
  dc.max_age = c.max_feature_track_age; dc.pred_type = c.optical_flow_predictor_type;
  dc.max_features = c.max_features_per_frame; dc.max_before_anms = c.max_nr_keypoints_before_anms;
  dc.min_distance = c.min_distance; dc.nms_enabled = c.enable_non_max_suppression; dc.nms_type = c.non_max_suppression_type;
  dc.hbins = c.nr_horizontal_bins; dc.vbins = c.nr_vertical_bins; dc.n_active_bins = 0;
  for (int i = 0; i < 64; ++i) { dc.bin_mask[i] = i < nbins ? c.binning_mask[i] : 0; if (i < nbins && c.binning_mask[i]) dc.n_active_bins++; }
  dc.quality = c.quality_level;          // GFTTDetector keeps a double: maxVal * qualityLevel in double, rounded to float once
  dc.subpix_enabled = c.enable_subpixel_corner_refinement; dc.subpix_win = c.subpix_window_size;
  dc.subpix_iters = std::min(std::max(c.subpix_max_iters, 1), 100); dc.subpix_zero = c.subpix_zero_zone;
  { double e = std::max(c.subpix_epsilon, 0.); dc.subpix_eps2 = e * e; }
  dc.sobel_tail_start = c.sobel_cpu_tail_start;
  // every interior pixel can be a candidate (a flat plateau of the response passes the 3x3 max test), and
  // cv::goodFeaturesToTrack keeps them all; a power of two because the min_distance < 1 path sorts the list
  // in place, padded to the next power of two
  {
    size_t want = (size_t)(dc.W - 2) * (dc.H - 2), p = 8192;
    while (p < want) p <<= 1;
    if (p > ((size_t)1 << 30)) { delete ctx; return set_err(nullptr, KVFE_ERR_INVALID_ARG, "image too large for the corner candidate list"); }
    dc.cand_cap = (int)p;
  }
  // rectified calibration: Cal3_S2Stereo from P1 (StereoCamera.cpp:75-82)
  dc.fx = rig->P1[0]; dc.fy = rig->P1[5]; dc.cxr = rig->P1[2]; dc.cyr = rig->P1[6]; dc.baseline = rig->baseline;
  // stereo stripe geometry (StereoMatcher.cpp:214-231)
  dc.templ_cols = c.templ_cols; dc.templ_rows = c.templ_rows;
  dc.stripe_rows = c.templ_rows + c.stripe_extra_rows;
  {
    int sc = (int)std::round(dc.fx * dc.baseline / c.min_point_dist) + c.templ_cols + 4;
    if (sc % 2 != 1) sc += 1;
    if (sc > dc.W) sc = dc.W;
    dc.stripe_cols = sc;
  }
  if (dc.stripe_cols < dc.templ_cols || dc.stripe_rows < dc.templ_rows) {
    delete ctx; return set_err(nullptr, KVFE_ERR_INVALID_ARG, "stripe smaller than template");
  }
  dc.min_depth = c.min_point_dist; dc.max_depth = c.max_point_dist; dc.fx_b = dc.fx * dc.baseline;
  dc.tol_templ = (float)c.tolerance_template_matching; dc.subpix_stereo = c.subpixel_refinement_stereo;
  dc.ransac_iters = c.ransac_max_iterations; dc.thr_mono = c.ransac_threshold_mono; dc.thr_stereo = c.ransac_threshold_stereo;
  dc.ransac_prob = c.ransac_probability; dc.min_mono_inl = c.min_nr_mono_inliers; dc.min_stereo_inl = c.min_nr_stereo_inliers;
  dc.use_2pt = c.ransac_use_2point_mono; dc.use_1pt = c.ransac_use_1point_stereo; dc.use_ransac = c.use_ransac;
  dc.use_stereo_tracking = c.use_stereo_tracking; dc.disparity_thr = c.disparity_threshold; dc.max_disparity = c.max_disparity_since_lkf;
  dc.min_kf_ns = c.min_intra_keyframe_time_ns; dc.max_kf_ns = c.max_intra_keyframe_time_ns; dc.min_features = c.min_number_features;

  make_cam(ctx->cam[0], rig->K_left, rig->D_left, rig->R1, rig->P1, rig->distortion_model);
  make_cam(ctx->cam[1], rig->K_right, rig->D_right, rig->R2, rig->P2, rig->distortion_model);

  CUC(cudaGetDevice(&ctx->device));
  CUC(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  const size_t B = dc.B;
  CUC(dmalloc(&ctx->d_cam, 2));
  CUC(cudaMemcpy(ctx->d_cam, ctx->cam, sizeof(CamModel) * 2, cudaMemcpyHostToDevice));
  for (int k = 0; k < 2; ++k) CUC(dmalloc(&db.pyr[k], B * dc.pyr_stride));
  static_assert(sizeof(CUtensorMap) == 128, "lk_kernel_tma indexes the tensor maps with a 128-byte stride");
  db.lk_tmaps = build_lk_tensor_maps(dc, db.pyr);
  CUC(dmalloc(&db.right_raw, B * dc.img_stride));
  // fixed-point remap tables (cv::convertMaps-style: integer source pixel + 5+5 fractional bits),
  // computed once per rig from the in-register f64 map model
  for (int k = 0; k < 2; ++k) {
    CUC(dmalloc(&db.rmap[k], (size_t)dc.W * dc.H));
    launch_rmap_table(dc, ctx->d_cam, k, db.rmap[k], ctx->stream);
  }
  CUC(cudaStreamSynchronize(ctx->stream));
  CUC(cudaGetLastError());
  CUC(dmalloc(&db.rectL, B * dc.img_stride));
  CUC(dmalloc(&db.rectR, B * dc.img_stride));
  CUC(dmalloc(&db.mask, B * dc.img_stride));
  CUC(dmalloc(&db.eig, B * (size_t)dc.W * dc.H));
  CUC(dmalloc(&db.eig_max, B));
  CUC(dmalloc(&db.cand, B * (size_t)dc.cand_cap));
  CUC(dmalloc(&db.cand_n, B));
  CUC(dmalloc(&db.cand_hist, B * 2048));
  CUC(dmalloc(&db.cand_sel, B * 16384));
  CUC(dmalloc(&db.cand_sel_n, B));
  CUC(dmalloc(&db.greedy_redo, B));
  CUC(dmalloc(&db.force_kf, B));
  CUC(dmalloc(&db.corner_idx, B * (size_t)dc.max_before_anms));
  CUC(dmalloc(&db.corner_n, B));
  CUC(dmalloc(&db.new_x, B * cap)); CUC(dmalloc(&db.new_y, B * cap)); CUC(dmalloc(&db.new_n, B));
  {
    int cell = std::max(dc.min_distance, 1);
    size_t ncells = (size_t)((dc.W + cell - 1) / cell) * ((dc.H + cell - 1) / cell);
    // sort_greedy_kernel's global sections: cstart[ncells+1] | head[ncells] | newacc[ncells] | state[cand_cap bytes] |
    // tmp[cand_cap u64]; the RANSAC kernels use 5 * (iters + 1) + cap ints of the same block
    const size_t greedy = 3 * ncells + 8 + (size_t)dc.cand_cap / 4 + 2 + 2 * (size_t)dc.cand_cap;
    db.scratch_stride = round_up(std::max(greedy, 3 * (size_t)dc.cand_cap + ncells) + 64 + 5 * (size_t)(dc.ransac_iters + 1) + cap, 64);
    CUC(dmalloc(&db.scratch_i, B * db.scratch_stride));
  }
  // all-equal-keys std::sort permutations (cv::sortIdx descending): perm(N) at offset N(N-1)/2
  {
    int M = dc.max_before_anms;
    std::vector<unsigned short> tab((size_t)M * (M + 1) / 2 + 1);
    std::vector<int> keys, idx;
    for (int N = 1; N <= M; ++N) {
      keys.assign(N, 0); idx.resize(N);
      std::iota(idx.begin(), idx.end(), 0);
      std::sort(idx.begin(), idx.end(), [&](int a, int b) { return keys[a] < keys[b]; });
      std::reverse(idx.begin(), idx.end());
      for (int i = 0; i < N; ++i) tab[(size_t)N * (N - 1) / 2 + i] = (unsigned short)idx[i];
    }
    CUC(dmalloc(&db.sort_perm, tab.size()));
    CUC(cudaMemcpy(db.sort_perm, tab.data(), tab.size() * sizeof(unsigned short), cudaMemcpyHostToDevice));
  }
  // OpenGV rnd(): uniform_int_distribution<int>(0, INT_MAX)(mt19937(12345)), both libstdc++ algorithms
  {
    int n = 16 * (dc.ransac_iters + 1) + 1024;
    std::vector<int> tab(n);
    std::mt19937 alg; alg.seed(12345u);
    for (int i = 0; i < n;) {
      unsigned int r = alg();
      if (c.rnd_libstdcxx == 0) tab[i++] = (int)(r >> 1);
      else if (r < 0x80000000u) tab[i++] = (int)r;
    }
    db.rnd_n = n;
    CUC(dmalloc(&db.rnd_table, n));
    CUC(cudaMemcpy(db.rnd_table, tab.data(), n * sizeof(int), cudaMemcpyHostToDevice));
  }
  {
    std::vector<float> m = subpix_mask_table(std::max(dc.subpix_win, 1));
    CUC(dmalloc(&db.subpix_mask, m.size()));
    CUC(cudaMemcpy(db.subpix_mask, m.data(), m.size() * sizeof(float), cudaMemcpyHostToDevice));
    std::vector<float> m2 = subpix_mask_table(10);
    CUC(dmalloc(&db.subpix_mask_stereo, m2.size()));
    CUC(cudaMemcpy(db.subpix_mask_stereo, m2.data(), m2.size() * sizeof(float), cudaMemcpyHostToDevice));
  }
  {
    int r = std::max(dc.min_distance, 0);
    std::vector<int> hw = circle_half_widths(r);
    ctx->circle_r = r;
    CUC(dmalloc(&ctx->circle_hw, hw.size()));
    CUC(cudaMemcpy(ctx->circle_hw, hw.data(), hw.size() * sizeof(int), cudaMemcpyHostToDevice));
  }
  CUC(dmalloc(&db.lk_px, B * cap)); CUC(dmalloc(&db.lk_py, B * cap));
  CUC(dmalloc(&db.lk_qx, B * cap)); CUC(dmalloc(&db.lk_qy, B * cap));
  CUC(dmalloc(&db.lk_pred_x, B * cap)); CUC(dmalloc(&db.lk_pred_y, B * cap));
  CUC(dmalloc(&db.lk_src, B * cap)); CUC(dmalloc(&db.lk_status, B * cap));
  CUC(dmalloc(&db.m_ref, B * cap)); CUC(dmalloc(&db.m_cur, B * cap)); CUC(dmalloc(&db.m_n, B));
  CUC(dmalloc(&db.inl, B * cap)); CUC(dmalloc(&db.inl_n, B));
  db.rs_stride = round_up(6 * (size_t)cap + 12 * (size_t)std::max(dc.ransac_iters + 1, 32) + 16 * (size_t)cap, 32);
  CUC(dmalloc(&db.rs_d, B * db.rs_stride));
  {
    FrameSoA& f = db.fr;
    size_t n = B * 3 * cap;
    CUC(dmalloc(&f.n, B * 3)); CUC(dmalloc(&f.timestamp, B * 3)); CUC(dmalloc(&f.frame_id, B * 3));
    CUC(dmalloc(&f.kx, n)); CUC(dmalloc(&f.ky, n)); CUC(dmalloc(&f.lmk, n)); CUC(dmalloc(&f.age, n));
    CUC(dmalloc(&f.versor, 3 * n)); CUC(dmalloc(&f.lstat, n)); CUC(dmalloc(&f.lrx, n)); CUC(dmalloc(&f.lry, n));
    CUC(dmalloc(&f.rstat, n)); CUC(dmalloc(&f.mstat, n)); CUC(dmalloc(&f.rrx, n)); CUC(dmalloc(&f.rry, n)); CUC(dmalloc(&f.depth, n));
    CUC(dmalloc(&f.p3d, 3 * n)); CUC(dmalloc(&f.rkx, n)); CUC(dmalloc(&f.rky, n));
  }
  CUC(dmalloc(&db.st, B));
  dc.mesh_on = c.mesh_2d ? 1 : 0;
  dc.equalize = c.equalize_image ? 1 : 0;
  dc.mono = c.frontend_type == 1 ? 1 : 0;
  dc.rgbd = c.frontend_type == 2 ? 1 : 0;
  if (dc.rgbd) {
    const kvfe_depth_params& dp = c.depth;
    dc.depth_type = dp.depth_type;
    dc.depth_row = (size_t)dc.W * (dp.depth_type == KVFE_DEPTH_F32 ? 4 : 2);
    dc.depth_stride = round_up(dc.depth_row * dc.H, 256);
    dc.depth_to_m = dp.depth_to_meters; dc.depth_min = dp.min_depth;
    depth_mask_bounds(dp, &dc.depth_lo, &dc.depth_hi, &dc.depth_lo16, &dc.depth_hi16);
    dc.depth_fx_b = ctx->cam[0].fx * (double)dp.virtual_baseline;      // RgbdFrame.cpp:66
    CUC(dmalloc(&db.depth, B * dc.depth_stride));
  }
  dc.subdiv_factor = c.subdiv_bounding_factor > 0.f ? c.subdiv_bounding_factor : 6.f;
  packet_layout(cap, dc.mesh_on != 0, db.pk_off, &db.packet_bytes);
  launch_mesh_init(dc);
  if (!mesh_fits_smem(dc)) CUC(dmalloc(&db.mesh_ws, (dc.mesh_on ? B : 1) * mesh_global_ws_ints(dc)));
  CUC(dmalloc(&db.packets, B * db.packet_bytes));
  CUC(cudaMallocHost((void**)&ctx->h_stage, 2 * B * dc.img_stride));
  CUC(cudaMallocHost((void**)&ctx->h_packets, B * db.packet_bytes));
  ctx->io_pk_off = (B * (sizeof(long long) + 9 * sizeof(double)) + 255) & ~(size_t)255;
  for (int i = 0; i < 2; ++i) {
    CUC(cudaMallocHost((void**)&ctx->h_io[i], ctx->io_pk_off + B * db.packet_bytes));
    CUC(cudaEventCreateWithFlags(&ctx->pipe_done[i], cudaEventDisableTiming));
  }
  CUC(cudaMallocHost((void**)&ctx->h_ts, KVFE_IN_SLOTS * B * sizeof(long long)));
  CUC(cudaMallocHost((void**)&ctx->h_Rin, KVFE_IN_SLOTS * B * 9 * sizeof(double)));
  for (int i = 0; i < KVFE_IN_SLOTS; ++i) CUC(cudaEventCreateWithFlags(&ctx->in_ev[i], cudaEventDisableTiming));
  ctx->in_bytes = B * (sizeof(long long) + 9 * sizeof(double));
  CUC(dmalloc(&ctx->d_in, ctx->in_bytes));
  ctx->d_ts = reinterpret_cast<long long*>(ctx->d_in);
  ctx->d_Rin = reinterpret_cast<double*>(ctx->d_in + B * sizeof(long long));
  ctx->launches += launch_reset(dc, db, ctx->stream);
  CUC(cudaStreamSynchronize(ctx->stream));
  ctx->cur_slot = 0;
  {
    const char* e = getenv("KVFE_NO_GRAPH");
    ctx->use_graph = !(e && e[0] == '1');
    // opt-in: measured 4.5x SLOWER with 32 concurrent step graphs on B200 / CUDA 12.9 (graphs holding
    // conditional nodes do not overlap across streams the way flat kernel graphs do), see DESIGN.md
    const char* c = getenv("KVFE_GRAPH_COND");
    ctx->use_cond = (c && c[0] == '1');
  }
  CUC(dmalloc(&ctx->d_kf_steps, 1));
  CUC(dmalloc(&ctx->d_pub_count, 2));
  CUC(cudaMemset(ctx->d_pub_count, 0, 2 * sizeof(unsigned int)));
  for (int i = 0; i < 2; ++i) {
    const size_t bytes = KVFE_STEPIO_ARRAYS + B * (sizeof(long long) + 9 * sizeof(double));
    CUC(cudaMallocHost((void**)&ctx->pio[i], bytes));
    memset(ctx->pio[i], 0, bytes);
  }
  *out = ctx;
  return KVFE_OK;
}

extern "C" void kvfe_destroy(kvfe_ctx* ctx) {
  if (!ctx) return;
  cudaStreamSynchronize(ctx->stream);
  DevBuf& db = ctx->db;
  for (int i = 0; i < 2; ++i) {
    if (ctx->pipe_graph_ready[i]) cudaGraphExecDestroy(ctx->pipe_graph[i]);
    if (ctx->pipe_split_ready[i]) { cudaGraphExecDestroy(ctx->pipe_graph_a[i]); cudaGraphExecDestroy(ctx->pipe_graph_kf[i]); cudaGraphExecDestroy(ctx->pipe_graph_nokf[i]); }
    if (ctx->pio[i]) cudaFreeHost(ctx->pio[i]);
  }
  free(const_cast<void*>(db.lk_tmaps));
  if (ctx->side) cudaStreamDestroy(ctx->side);
  if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
  if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
  void* ptrs[] = {db.depth, db.force_kf, db.cand_hist, db.cand_sel, db.cand_sel_n, db.greedy_redo, db.stage_img[0], db.stage_img[1], db.stage_seq, db.mesh_ws, ctx->d_pub_count, ctx->d_kf_steps, ctx->d_cam, db.pyr[0], db.pyr[1], db.right_raw, db.rmap[0], db.rmap[1], db.rectL, db.rectR, db.mask, db.eig, db.eig_max,
                  db.cand, db.cand_n, db.corner_idx, db.corner_n, db.new_x, db.new_y, db.new_n, db.scratch_i,
                  db.sort_perm, db.rnd_table, db.subpix_mask, db.subpix_mask_stereo, ctx->circle_hw, db.lk_px,
                  db.lk_py, db.lk_qx, db.lk_qy, db.lk_pred_x, db.lk_pred_y, db.lk_src, db.lk_status, db.m_ref,
                  db.m_cur, db.m_n, db.inl, db.inl_n, db.rs_d, db.fr.n, db.fr.timestamp, db.fr.frame_id, db.fr.kx,
                  db.fr.ky, db.fr.lmk, db.fr.age, db.fr.versor, db.fr.lstat, db.fr.lrx, db.fr.lry, db.fr.rstat, db.fr.mstat,
                  db.fr.rrx, db.fr.rry, db.fr.depth, db.fr.p3d, db.fr.rkx, db.fr.rky, db.st, ctx->own_packets ? ctx->own_packets : db.packets, ctx->d_in};
  for (void* p : ptrs) if (p) cudaFree(p);
  if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
  if (ctx->h_packets) cudaFreeHost(ctx->h_packets);
  for (int i = 0; i < 2; ++i) {
    if (ctx->h_io[i]) cudaFreeHost(ctx->h_io[i]);
    if (ctx->host_graph_ready[i]) cudaGraphExecDestroy(ctx->host_graph[i]);
    if (ctx->pipe_done[i]) cudaEventDestroy(ctx->pipe_done[i]);
  }

  if (ctx->h_ts) cudaFreeHost(ctx->h_ts);
  if (ctx->h_Rin) cudaFreeHost(ctx->h_Rin);
  for (int i = 0; i < KVFE_IN_SLOTS; ++i) if (ctx->in_ev[i]) cudaEventDestroy(ctx->in_ev[i]);
  for (int i = 0; i < 2; ++i) if (ctx->graph_ready[i]) cudaGraphExecDestroy(ctx->step_graph[i]);
  cudaStreamDestroy(ctx->stream);
  delete ctx;
}

extern "C" const char* kvfe_last_error(const kvfe_ctx* ctx) { return ctx ? ctx->err : g_create_err; }
extern "C" int kvfe_max_keypoints(const kvfe_ctx* ctx) { return ctx ? ctx->dc.cap : 0; }
// kernels launched so far: host-side count of everything outside the conditional keyframe part
// plus (executions of that part, counted on the device) x (its kernels)
extern "C" int kvfe_kernel_launches(const kvfe_ctx* ctx) {
  if (!ctx) return 0;
  int kf = 0;
  if (ctx->d_kf_steps) {
    cudaStreamSynchronize(ctx->stream);
    cudaMemcpy(&kf, ctx->d_kf_steps, sizeof(int), cudaMemcpyDeviceToHost);
  }
  return (int)(ctx->launches + (long long)kf * ctx->graph_launches_kf);
}
extern "C" size_t kvfe_packet_bytes(const kvfe_ctx* ctx) { return ctx ? ctx->db.packet_bytes : 0; }
extern "C" int kvfe_packet_offsets(const kvfe_ctx* ctx, size_t* offsets, int max_entries) {
  if (!ctx || !offsets) return KVFE_ERR_INVALID_ARG;
  int n = std::min(max_entries, KVFE_PACKET_ARRAYS);
  for (int i = 0; i < n; ++i) offsets[i] = ctx->db.pk_off[i];
  return n;
}
extern "C" void* kvfe_cuda_stream(kvfe_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }
extern "C" int kvfe_sync(kvfe_ctx* ctx) {
  if (!ctx) return KVFE_ERR_INVALID_ARG;
  CU(cudaStreamSynchronize(ctx->stream));
  return KVFE_OK;
}

// ---- helpers for the stage-level calls: they drive stream 0 with an explicit mode ----------------
static int set_stage_state(kvfe_ctx* ctx, int mode, int need, int n_frame) {
  StreamState st;
  memset(&st, 0, sizeof(st));
  st.mode = mode; st.slot_k = 0; st.slot_km1 = 1; st.slot_lkf = 1; st.need = need; st.frame_count = 1;
  for (int i = 0; i < 9; ++i) { st.kf_R_ref[i] = st.kf_R_cur[i] = st.ref_R_cur[i] = (i % 4 == 0) ? 1.0 : 0.0; }
  CU(cudaMemcpyAsync(ctx->db.st, &st, sizeof(st), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(ctx->db.fr.n, &n_frame, sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));   // st / n_frame live on this stack frame
  return KVFE_OK;
}
// every other stream must be idle (mode with no stage bit set) during a stage call
static int park_other_streams(kvfe_ctx* ctx) {
  if (ctx->dc.B <= 1) return KVFE_OK;
  std::vector<StreamState> h(ctx->dc.B);
  CU(cudaMemcpy(h.data(), ctx->db.st, sizeof(StreamState) * ctx->dc.B, cudaMemcpyDeviceToHost));
  for (int b = 1; b < ctx->dc.B; ++b) h[b].mode = 7;
  CU(cudaMemcpy(ctx->db.st, h.data(), sizeof(StreamState) * ctx->dc.B, cudaMemcpyHostToDevice));
  return KVFE_OK;
}

// image copies: a single contiguous transfer when both sides are densely packed (the common case:
// pitch == width), else a strided 2-D copy
static int copy_image(kvfe_ctx* ctx, void* dst, size_t dst_pitch, const void* src, size_t src_pitch,
                      cudaMemcpyKind kind) {
  const size_t W = ctx->dc.W, H = ctx->dc.H;
  if (dst_pitch == W && src_pitch == W) CU(cudaMemcpyAsync(dst, src, W * H, kind, ctx->stream));
  else CU(cudaMemcpy2DAsync(dst, dst_pitch, src, src_pitch, W, H, kind, ctx->stream));
  return KVFE_OK;
}
static int upload_image(kvfe_ctx* ctx, unsigned char* dst, int dst_pitch, const uint8_t* src, size_t pitch) {
  return copy_image(ctx, dst, dst_pitch, src, pitch, cudaMemcpyHostToDevice);
}
static int download_image(kvfe_ctx* ctx, uint8_t* dst, size_t pitch, const unsigned char* src, int src_pitch) {
  CU(cudaMemcpy2DAsync(dst, pitch, src, src_pitch, ctx->dc.W, ctx->dc.H, cudaMemcpyDeviceToHost, ctx->stream));
  return KVFE_OK;
}
#define RET(call) do { int r_ = (call); if (r_ != KVFE_OK) return r_; } while (0)
#define CHECK_LAUNCH() CU(cudaGetLastError())

extern "C" int kvfe_rectify_pair(kvfe_ctx* ctx, const uint8_t* left, const uint8_t* right, size_t pitch,
                                 uint8_t* left_rect, uint8_t* right_rect, size_t out_pitch) {
  if (!ctx || !left || !right || !left_rect || !right_rect) return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  const DevCfg& dc = ctx->dc; DevBuf& db = ctx->db;
  unsigned char* L = db.pyr[0] + dc.lvl_off[0];
  RET(upload_image(ctx, L, dc.pitch, left, pitch));
  RET(upload_image(ctx, db.right_raw, dc.pitch, right, pitch));
  ctx->launches += launch_rectify(dc, db.rmap[0], L, dc.pyr_stride, db.rectL, dc.img_stride, 1, nullptr, 0, ctx->stream);
  ctx->launches += launch_rectify(dc, db.rmap[1], db.right_raw, dc.img_stride, db.rectR, dc.img_stride, 1, nullptr, 0, ctx->stream);
  CHECK_LAUNCH();
  RET(download_image(ctx, left_rect, out_pitch, db.rectL, dc.pitch));
  RET(download_image(ctx, right_rect, out_pitch, db.rectR, dc.pitch));
  CU(cudaStreamSynchronize(ctx->stream));
  return KVFE_OK;
}

extern "C" int kvfe_rectify_maps(kvfe_ctx* ctx, int cam, float* map_x, float* map_y) {
  if (!ctx || !map_x || !map_y || cam < 0 || cam > 1) return set_err(ctx, KVFE_ERR_INVALID_ARG, "bad argument");
  const DevCfg& dc = ctx->dc;
  size_t n = (size_t)dc.W * dc.H;
  float* d = ctx->db.eig;    // reuse the response buffer (W*H floats per stream) + a temporary
  float* d2 = nullptr;
  CU(cudaMalloc((void**)&d2, n * sizeof(float)));
  ctx->launches += launch_maps(dc, ctx->d_cam, cam, d, d2, ctx->stream);
  CHECK_LAUNCH();
  CU(cudaMemcpyAsync(map_x, d, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaMemcpyAsync(map_y, d2, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  cudaFree(d2);
  return KVFE_OK;
}

extern "C" int kvfe_pyramid(kvfe_ctx* ctx, const uint8_t* img, size_t pitch, uint8_t* levels_out,
                            size_t levels_out_bytes, int* n_levels) {
  if (!ctx || !img || !levels_out || !n_levels) return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  const DevCfg& dc = ctx->dc; DevBuf& db = ctx->db;
  RET(upload_image(ctx, db.pyr[0] + dc.lvl_off[0], dc.pitch, img, pitch));
  ctx->launches += launch_pyramid(dc, db.pyr[0], 1, ctx->stream);
  CHECK_LAUNCH();
  size_t o = 0;
  for (int l = 1; l < dc.n_levels; ++l) {
    size_t sz = (size_t)dc.lvl_w[l] * dc.lvl_h[l];
    if (o + sz > levels_out_bytes) return set_err(ctx, KVFE_ERR_CAPACITY, "levels_out too small");
    CU(cudaMemcpy2DAsync(levels_out + o, dc.lvl_w[l], db.pyr[0] + dc.lvl_off[l], dc.lvl_pitch[l], dc.lvl_w[l],
                         dc.lvl_h[l], cudaMemcpyDeviceToHost, ctx->stream));
    o += sz;
  }
  CU(cudaStreamSynchronize(ctx->stream));
  *n_levels = dc.n_levels;
  return KVFE_OK;
}

extern "C" int kvfe_min_eigen_response(kvfe_ctx* ctx, const uint8_t* img, size_t pitch, float* response) {
  if (!ctx || !img || !response) return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  const DevCfg& dc = ctx->dc; DevBuf& db = ctx->db;
  RET(park_other_streams(ctx));
  RET(set_stage_state(ctx, 2, 0, 0));
  unsigned char* I = db.pyr[0] + dc.lvl_off[0];
  RET(upload_image(ctx, I, dc.pitch, img, pitch));
  ctx->launches += launch_min_eig(dc, db, I, dc.pyr_stride, 1 << 2, ctx->stream);
  CHECK_LAUNCH();
  CU(cudaMemcpyAsync(response, db.eig, (size_t)dc.W * dc.H * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return KVFE_OK;
}

static int load_existing(kvfe_ctx* ctx, const float* x, const float* y, const int64_t* lmk, int n) {
  DevBuf& db = ctx->db;
  if (n > ctx->dc.cap) return set_err(ctx, KVFE_ERR_CAPACITY, "n_existing %d exceeds capacity %d", n, ctx->dc.cap);
  if (n > 0) {
    CU(cudaMemcpyAsync(db.fr.kx, x, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(db.fr.ky, y, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(db.fr.lmk, lmk, n * sizeof(long long), cudaMemcpyHostToDevice, ctx->stream));
  }
  return KVFE_OK;
}

static int detect_common(kvfe_ctx* ctx, const uint8_t* img, size_t pitch, const float* ex, const float* ey,
                         const int64_t* el, int n_existing, int need, bool raw, const uint8_t* mask = nullptr, size_t mask_pitch = 0) {
  const DevCfg& dc = ctx->dc; DevBuf& db = ctx->db;
  RET(park_other_streams(ctx));
  RET(set_stage_state(ctx, 2, need, n_existing));
  RET(load_existing(ctx, ex, ey, el, n_existing));
  unsigned char* I = db.pyr[0] + dc.lvl_off[0];
  RET(upload_image(ctx, I, dc.pitch, img, pitch));
  if (mask) RET(upload_image(ctx, db.mask, dc.pitch, mask, mask_pitch));      // Frame::detection_mask_
  ctx->launches += launch_gftt(dc, db, I, dc.pyr_stride, ctx->circle_hw, ctx->circle_r, 1 << 2, ctx->stream, mask ? 1 : 0);
  if (!raw) ctx->launches += launch_select(dc, db, I, dc.pyr_stride, ctx->d_cam, 1 << 2, 0, ctx->stream);
  CHECK_LAUNCH();
  return KVFE_OK;
}

extern "C" int kvfe_detect(kvfe_ctx* ctx, const uint8_t* img, size_t pitch, const float* existing_x,
                           const float* existing_y, const int64_t* existing_lmk, int n_existing, int need,
                           float* out_x, float* out_y, int* n_out) {
  if (!ctx || !img || !out_x || !out_y || !n_out) return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  RET(detect_common(ctx, img, pitch, existing_x, existing_y, existing_lmk, n_existing, need, false));
  int n = 0;
  CU(cudaMemcpyAsync(&n, ctx->db.new_n, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  if (n > 0) {
    CU(cudaMemcpy(out_x, ctx->db.new_x, n * sizeof(float), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(out_y, ctx->db.new_y, n * sizeof(float), cudaMemcpyDeviceToHost));
  }
  *n_out = n;
  return KVFE_OK;
}

extern "C" int kvfe_detect_masked(kvfe_ctx* ctx, const uint8_t* img, size_t pitch, const uint8_t* detection_mask, size_t mask_pitch,
                                  const float* existing_x, const float* existing_y, const int64_t* existing_lmk, int n_existing,
                                  int need, float* out_x, float* out_y, int* n_out) {
  if (!ctx || !img || !detection_mask || !out_x || !out_y || !n_out) return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  RET(detect_common(ctx, img, pitch, existing_x, existing_y, existing_lmk, n_existing, need, false, detection_mask, mask_pitch));
  int n = 0;
  CU(cudaMemcpyAsync(&n, ctx->db.new_n, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  if (n > 0) {
    CU(cudaMemcpy(out_x, ctx->db.new_x, n * sizeof(float), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(out_y, ctx->db.new_y, n * sizeof(float), cudaMemcpyDeviceToHost));
  }
  *n_out = n;
  return KVFE_OK;
}

extern "C" int kvfe_detect_raw(kvfe_ctx* ctx, const uint8_t* img, size_t pitch, const float* existing_x,
                               const float* existing_y, const int64_t* existing_lmk, int n_existing,
                               float* out_x, float* out_y, float* out_response, int* n_out) {
  if (!ctx || !img || !out_x || !out_y || !n_out) return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  RET(detect_common(ctx, img, pitch, existing_x, existing_y, existing_lmk, n_existing, 0, true));
  const DevCfg& dc = ctx->dc;
  int n = 0;
  CU(cudaMemcpyAsync(&n, ctx->db.corner_n, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  std::vector<int> idx(std::max(n, 1));
  std::vector<float> eig((size_t)dc.W * dc.H);
  if (n > 0) CU(cudaMemcpy(idx.data(), ctx->db.corner_idx, n * sizeof(int), cudaMemcpyDeviceToHost));
  if (out_response) CU(cudaMemcpy(eig.data(), ctx->db.eig, eig.size() * sizeof(float), cudaMemcpyDeviceToHost));
  for (int i = 0; i < n; ++i) {
    out_x[i] = (float)(idx[i] % dc.W); out_y[i] = (float)(idx[i] / dc.W);
    if (out_response) out_response[i] = eig[idx[i]];
  }
  *n_out = n;
  return KVFE_OK;
}

extern "C" int kvfe_track(kvfe_ctx* ctx, const uint8_t* ref_img, const uint8_t* cur_img, size_t pitch,
                          const double* ref_R_cur, const float* ref_x, const float* ref_y, int n,
                          float* pred_x, float* pred_y, float* cur_x, float* cur_y, uint8_t* status) {
  if (!ctx || !ref_img || !cur_img || !ref_R_cur || !cur_x || !cur_y || !status)
    return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  const DevCfg& dc = ctx->dc; DevBuf& db = ctx->db;
  if (n > dc.cap) return set_err(ctx, KVFE_ERR_CAPACITY, "n %d exceeds capacity %d", n, dc.cap);
  RET(park_other_streams(ctx));
  // frame slot 1 (km1) holds the reference keypoints; prep computes the homography from
  // keyframe_R_ref = I, keyframe_R_cur = ref_R_cur
  StreamState st;
  memset(&st, 0, sizeof(st));
  st.frame_count = 1; st.slot_km1 = 1; st.slot_lkf = 1; st.slot_k = 0; st.mode = 1;
  for (int i = 0; i < 9; ++i) st.kf_R_ref[i] = (i % 4 == 0) ? 1.0 : 0.0;
  CU(cudaMemcpy(db.st, &st, sizeof(st), cudaMemcpyHostToDevice));
  std::vector<long long> lm(std::max(n, 1));
  std::iota(lm.begin(), lm.end(), 0LL);
  std::vector<int> age(std::max(n, 1), 1);
  int ns[3] = {0, n, 0};
  CU(cudaMemcpy(db.fr.n, ns, sizeof(ns), cudaMemcpyHostToDevice));
  if (n > 0) {
    CU(cudaMemcpy(db.fr.kx + dc.cap, ref_x, n * sizeof(float), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(db.fr.ky + dc.cap, ref_y, n * sizeof(float), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(db.fr.lmk + dc.cap, lm.data(), n * sizeof(long long), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(db.fr.age + dc.cap, age.data(), n * sizeof(int), cudaMemcpyHostToDevice));
  }
  long long ts = 0;
  CU(cudaMemcpy(ctx->d_ts, &ts, sizeof(ts), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(ctx->d_Rin, ref_R_cur, 9 * sizeof(double), cudaMemcpyHostToDevice));
  RET(upload_image(ctx, db.pyr[0] + dc.lvl_off[0], dc.pitch, ref_img, pitch));
  RET(upload_image(ctx, db.pyr[1] + dc.lvl_off[0], dc.pitch, cur_img, pitch));
  ctx->launches += launch_pyramid(dc, db.pyr[0], 1, ctx->stream);
  ctx->launches += launch_pyramid(dc, db.pyr[1], 1, ctx->stream);
  ctx->launches += launch_prep(dc, db, ctx->d_cam, ctx->d_ts, ctx->d_Rin, nullptr, ctx->stream);
  ctx->launches += launch_track_pre(dc, db, ctx->stream);
  ctx->launches += launch_lk(dc, db, 0, 1, ctx->stream);
  CHECK_LAUNCH();
  CU(cudaStreamSynchronize(ctx->stream));
  if (n > 0) {
    if (pred_x) CU(cudaMemcpy(pred_x, db.lk_pred_x, n * sizeof(float), cudaMemcpyDeviceToHost));
    if (pred_y) CU(cudaMemcpy(pred_y, db.lk_pred_y, n * sizeof(float), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(cur_x, db.lk_qx, n * sizeof(float), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(cur_y, db.lk_qy, n * sizeof(float), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(status, db.lk_status, n, cudaMemcpyDeviceToHost));
  }
  ctx->launches += launch_reset(dc, db, ctx->stream);
  CU(cudaStreamSynchronize(ctx->stream));
  return KVFE_OK;
}

extern "C" int kvfe_undistort_keypoints(kvfe_ctx* ctx, int cam, int use_R, int use_P, const float* x,
                                        const float* y, int n, float* out_x, float* out_y) {
  if (!ctx || !x || !y || !out_x || !out_y || cam < 0 || cam > 1) return set_err(ctx, KVFE_ERR_INVALID_ARG, "bad argument");
  if (n <= 0) return KVFE_OK;
  float* d = nullptr;
  CU(cudaMalloc((void**)&d, 4 * (size_t)n * sizeof(float)));
  CU(cudaMemcpyAsync(d, x, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(d + n, y, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  ctx->launches += launch_undistort(ctx->dc, ctx->d_cam, cam, use_R, use_P, d, d + n, n, d + 2 * n, d + 3 * n, ctx->stream);
  CHECK_LAUNCH();
  CU(cudaMemcpyAsync(out_x, d + 2 * n, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaMemcpyAsync(out_y, d + 3 * n, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  cudaFree(d);
  return KVFE_OK;
}

extern "C" int kvfe_bearing_vectors(kvfe_ctx* ctx, const float* x, const float* y, int n, double* versors) {
  if (!ctx || !x || !y || !versors) return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  if (n <= 0) return KVFE_OK;
  float* d = nullptr; double* dv = nullptr;
  CU(cudaMalloc((void**)&d, 2 * (size_t)n * sizeof(float)));
  CU(cudaMalloc((void**)&dv, 3 * (size_t)n * sizeof(double)));
  CU(cudaMemcpyAsync(d, x, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(d + n, y, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  ctx->launches += launch_bearing(ctx->dc, ctx->d_cam, d, d + n, n, dv, ctx->stream);
  CHECK_LAUNCH();
  CU(cudaMemcpyAsync(versors, dv, 3 * (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  cudaFree(d); cudaFree(dv);
  return KVFE_OK;
}

extern "C" int kvfe_sparse_stereo(kvfe_ctx* ctx, const uint8_t* left, const uint8_t* right, size_t pitch,
                                  const float* kp_x, const float* kp_y, const double* versors, int n,
                                  kvfe_stereo_out* out, uint8_t* left_rect, uint8_t* right_rect, size_t rect_pitch) {
  if (!ctx || !left || !right || !kp_x || !kp_y || !versors || !out) return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  const DevCfg& dc = ctx->dc; DevBuf& db = ctx->db;
  if (n > dc.cap) return set_err(ctx, KVFE_ERR_CAPACITY, "n %d exceeds capacity %d", n, dc.cap);
  if (n <= 0) return set_err(ctx, KVFE_ERR_INVALID_ARG, "Call feature detection on left frame first...");
  RET(park_other_streams(ctx));
  RET(set_stage_state(ctx, 2, 0, n));
  CU(cudaMemcpyAsync(db.fr.kx, kp_x, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(db.fr.ky, kp_y, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(db.fr.versor, versors, 3 * (size_t)n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  unsigned char* L = db.pyr[0] + dc.lvl_off[0];
  RET(upload_image(ctx, L, dc.pitch, left, pitch));
  RET(upload_image(ctx, db.right_raw, dc.pitch, right, pitch));
  ctx->launches += launch_rectify(dc, db.rmap[0], L, dc.pyr_stride, db.rectL, dc.img_stride, 1, nullptr, 0, ctx->stream);
  ctx->launches += launch_rectify(dc, db.rmap[1], db.right_raw, dc.img_stride, db.rectR, dc.img_stride, 1, nullptr, 0, ctx->stream);
  ctx->launches += launch_sparse_stereo(dc, db, ctx->d_cam, 1 << 2, 0, ctx->stream);
  CHECK_LAUNCH();
  CU(cudaStreamSynchronize(ctx->stream));
  const FrameSoA& f = db.fr;
  if (out->left_status) CU(cudaMemcpy(out->left_status, f.lstat, n * sizeof(int), cudaMemcpyDeviceToHost));
  if (out->left_rect_x) CU(cudaMemcpy(out->left_rect_x, f.lrx, n * sizeof(float), cudaMemcpyDeviceToHost));
  if (out->left_rect_y) CU(cudaMemcpy(out->left_rect_y, f.lry, n * sizeof(float), cudaMemcpyDeviceToHost));
  if (out->right_status) CU(cudaMemcpy(out->right_status, f.rstat, n * sizeof(int), cudaMemcpyDeviceToHost));
  if (out->right_rect_x) CU(cudaMemcpy(out->right_rect_x, f.rrx, n * sizeof(float), cudaMemcpyDeviceToHost));
  if (out->right_rect_y) CU(cudaMemcpy(out->right_rect_y, f.rry, n * sizeof(float), cudaMemcpyDeviceToHost));
  if (out->depth) CU(cudaMemcpy(out->depth, f.depth, n * sizeof(double), cudaMemcpyDeviceToHost));
  if (out->points_3d) CU(cudaMemcpy(out->points_3d, f.p3d, 3 * (size_t)n * sizeof(double), cudaMemcpyDeviceToHost));
  if (out->right_x) CU(cudaMemcpy(out->right_x, f.rkx, n * sizeof(float), cudaMemcpyDeviceToHost));
  if (out->right_y) CU(cudaMemcpy(out->right_y, f.rky, n * sizeof(float), cudaMemcpyDeviceToHost));
  if (left_rect) RET(download_image(ctx, left_rect, rect_pitch, db.rectL, dc.pitch));
  if (right_rect) RET(download_image(ctx, right_rect, rect_pitch, db.rectR, dc.pitch));
  CU(cudaStreamSynchronize(ctx->stream));
  return KVFE_OK;
}

// ---- boundary completion: the remaining public methods of UndistorterRectifier / StereoCamera / StereoMatcher /
// Tracker as stage-level calls (host buffers, synchronous, stream 0 of the context as scratch) -------------
namespace {
// n floats / ints of several host arrays through one device allocation
struct StageScratch {
  unsigned char* p = nullptr;
  cudaError_t alloc(size_t bytes) { return cudaMalloc((void**)&p, bytes ? bytes : 16); }
  ~StageScratch() { if (p) cudaFree(p); }
};
}  // namespace

extern "C" int kvfe_check_rectified_keypoints(kvfe_ctx* ctx, int cam, const float* distorted_x, const float* distorted_y,
                                              const float* rectified_x, const float* rectified_y, int n, float pixel_tolerance,
                                              int32_t* status, float* out_x, float* out_y) {
  if (!ctx || !distorted_x || !distorted_y || !rectified_x || !rectified_y || !status || !out_x || !out_y || cam < 0 || cam > 1)
    return set_err(ctx, KVFE_ERR_INVALID_ARG, "bad argument");
  if (n <= 0) return KVFE_OK;
  StageScratch d;
  CU(d.alloc(7 * (size_t)n * 4));
  float* f = reinterpret_cast<float*>(d.p);
  const float* src[4] = {distorted_x, distorted_y, rectified_x, rectified_y};
  for (int k = 0; k < 4; ++k) CU(cudaMemcpyAsync(f + (size_t)k * n, src[k], n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  int* dst = reinterpret_cast<int*>(f + 4 * (size_t)n);
  ctx->launches += launch_check_rect_raw(ctx->dc, ctx->d_cam, cam, f, f + n, f + 2 * (size_t)n, f + 3 * (size_t)n, n, pixel_tolerance, dst,
                                         f + 5 * (size_t)n, f + 6 * (size_t)n, ctx->stream);
  CHECK_LAUNCH();
  CU(cudaMemcpyAsync(status, dst, n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaMemcpyAsync(out_x, f + 5 * (size_t)n, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaMemcpyAsync(out_y, f + 6 * (size_t)n, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return KVFE_OK;
}

extern "C" int kvfe_distort_unrectify_keypoints(kvfe_ctx* ctx, int cam, const int32_t* status, const float* x, const float* y,
                                                int n, float* out_x, float* out_y) {
  if (!ctx || !status || !x || !y || !out_x || !out_y || cam < 0 || cam > 1) return set_err(ctx, KVFE_ERR_INVALID_ARG, "bad argument");
  if (n <= 0) return KVFE_OK;
  StageScratch d;
  CU(d.alloc(5 * (size_t)n * 4));
  float* f = reinterpret_cast<float*>(d.p);
  int* ds = reinterpret_cast<int*>(f + 4 * (size_t)n);
  CU(cudaMemcpyAsync(f, x, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(f + n, y, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(ds, status, n * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  ctx->launches += launch_distort_unrectify_raw(ctx->dc, ctx->d_cam, cam, ds, f, f + n, n, f + 2 * (size_t)n, f + 3 * (size_t)n, ctx->stream);
  CHECK_LAUNCH();
  CU(cudaMemcpyAsync(out_x, f + 2 * (size_t)n, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaMemcpyAsync(out_y, f + 3 * (size_t)n, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return KVFE_OK;
}

// ---- RGB-D, stage level (rgbd.cu) ---------------------------------------------------------------------------------
static int check_depth_params(kvfe_ctx* ctx, const kvfe_depth_params* dp) {
  if (dp->depth_type != KVFE_DEPTH_U16 && dp->depth_type != KVFE_DEPTH_F32)
    return set_err(ctx, KVFE_ERR_INVALID_ARG, "depth_type must be KVFE_DEPTH_U16 or KVFE_DEPTH_F32");
  if (!(dp->virtual_baseline > 0.f)) return set_err(ctx, KVFE_ERR_INVALID_ARG, "virtual_baseline must be positive");   // CameraParams.cpp:344
  return KVFE_OK;
}

// depth image (W x H, u16 or f32) to the device, densely packed
static int upload_depth(kvfe_ctx* ctx, const void* depth, size_t pitch_bytes, int depth_type, unsigned char** out, size_t* row_bytes) {
  const size_t es = depth_type == KVFE_DEPTH_F32 ? 4 : 2;
  *row_bytes = (size_t)ctx->dc.W * es;
  if (pitch_bytes < *row_bytes) return set_err(ctx, KVFE_ERR_INVALID_ARG, "depth pitch %zu smaller than a row (%zu bytes)", pitch_bytes, *row_bytes);
  CU(cudaMalloc((void**)out, *row_bytes * ctx->dc.H));
  cudaError_t e = cudaMemcpy2DAsync(*out, *row_bytes, depth, pitch_bytes, *row_bytes, ctx->dc.H, cudaMemcpyHostToDevice, ctx->stream);
  if (e != cudaSuccess) { cudaFree(*out); *out = nullptr; return set_err(ctx, KVFE_ERR_CUDA, "depth upload: %s", cudaGetErrorString(e)); }
  return KVFE_OK;
}

extern "C" int kvfe_depth_detection_mask(kvfe_ctx* ctx, const void* depth, size_t depth_pitch_bytes, const kvfe_depth_params* dp,
                                         uint8_t* mask, size_t mask_pitch) {
  if (!ctx || !depth || !dp || !mask) return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  RET(check_depth_params(ctx, dp));
  if (mask_pitch < (size_t)ctx->dc.W) return set_err(ctx, KVFE_ERR_INVALID_ARG, "mask pitch smaller than the width");
  float lo, hi; unsigned int lo16, hi16;
  depth_mask_bounds(*dp, &lo, &hi, &lo16, &hi16);
  unsigned char* d_depth = nullptr; size_t rb = 0;
  RET(upload_depth(ctx, depth, depth_pitch_bytes, dp->depth_type, &d_depth, &rb));
  StageScratch m;
  cudaError_t e = m.alloc((size_t)ctx->dc.W * ctx->dc.H);
  if (e == cudaSuccess) {
    ctx->launches += launch_depth_mask(ctx->dc, d_depth, rb, dp->depth_type, lo, hi, lo16, hi16, m.p, ctx->dc.W, ctx->stream);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaMemcpy2DAsync(mask, mask_pitch, m.p, ctx->dc.W, ctx->dc.W, ctx->dc.H, cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  cudaFree(d_depth);
  if (e != cudaSuccess) return set_err(ctx, KVFE_ERR_CUDA, "kvfe_depth_detection_mask: %s", cudaGetErrorString(e));
  return KVFE_OK;
}

extern "C" int kvfe_rgbd_fill_stereo_frame(kvfe_ctx* ctx, const void* depth, size_t depth_pitch_bytes, const kvfe_depth_params* dp,
                                           const float* kp_x, const float* kp_y, const int32_t* left_status, const float* left_x,
                                           const float* left_y, const double* versors, int n, int32_t* right_status, float* right_x,
                                           float* right_y, double* keypoints_depth, double* keypoints_3d, float* right_kp_x,
                                           float* right_kp_y) {
  if (!ctx || !depth || !dp) return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  RET(check_depth_params(ctx, dp));
  if (n <= 0) return KVFE_OK;                         // "no features": every output stays empty (testRgbdFrame.cpp:108-117)
  if (!kp_x || !kp_y || !left_status || !left_x || !left_y || !versors || !right_status || !right_x || !right_y || !keypoints_depth ||
      !keypoints_3d || !right_kp_x || !right_kp_y)
    return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  unsigned char* d_depth = nullptr; size_t rb = 0;
  RET(upload_depth(ctx, depth, depth_pitch_bytes, dp->depth_type, &d_depth, &rb));
  // doubles first (8-byte alignment): versors 3n | depth n | p3d 3n ; then 4-byte arrays: 4 in f32 + status in, 5 out
  StageScratch d;
  const size_t N = (size_t)n;
  cudaError_t e = d.alloc(7 * N * 8 + 10 * N * 4);
  if (e != cudaSuccess) { cudaFree(d_depth); return set_err(ctx, KVFE_ERR_CUDA, "cudaMalloc: %s", cudaGetErrorString(e)); }
  double* dv = reinterpret_cast<double*>(d.p);
  double* dd = dv + 3 * N;
  double* dp3 = dd + N;
  float* f = reinterpret_cast<float*>(dp3 + 3 * N);
  float *d_kx = f, *d_ky = f + N, *d_lx = f + 2 * N, *d_ly = f + 3 * N;
  int* d_ls = reinterpret_cast<int*>(f + 4 * N);
  int* d_rs = reinterpret_cast<int*>(f + 5 * N);
  float *d_rx = f + 6 * N, *d_ry = f + 7 * N, *d_rkx = f + 8 * N, *d_rky = f + 9 * N;
  cudaStream_t s = ctx->stream;
  const struct { void* dst; const void* src; size_t bytes; } ups[] = {
      {dv, versors, 3 * N * 8}, {d_kx, kp_x, N * 4}, {d_ky, kp_y, N * 4}, {d_lx, left_x, N * 4}, {d_ly, left_y, N * 4}, {d_ls, left_status, N * 4}};
  for (const auto& u : ups)
    if (e == cudaSuccess) e = cudaMemcpyAsync(u.dst, u.src, u.bytes, cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) {
    const double fx_b = ctx->cam[0].fx * (double)dp->virtual_baseline;        // RgbdFrame.cpp:66
    ctx->launches += launch_rgbd_fill(ctx->dc, ctx->d_cam, d_depth, rb, dp->depth_type, dp->depth_to_meters, dp->min_depth, fx_b, d_kx, d_ky,
                                      d_ls, d_lx, d_ly, dv, n, d_rs, d_rx, d_ry, dd, dp3, d_rkx, d_rky, s);
    e = cudaGetLastError();
  }
  const struct { void* dst; const void* src; size_t bytes; } downs[] = {
      {right_status, d_rs, N * 4}, {right_x, d_rx, N * 4}, {right_y, d_ry, N * 4}, {keypoints_depth, dd, N * 8},
      {keypoints_3d, dp3, 3 * N * 8}, {right_kp_x, d_rkx, N * 4}, {right_kp_y, d_rky, N * 4}};
  for (const auto& u : downs)
    if (e == cudaSuccess) e = cudaMemcpyAsync(u.dst, u.src, u.bytes, cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  cudaFree(d_depth);
  if (e != cudaSuccess) return set_err(ctx, KVFE_ERR_CUDA, "kvfe_rgbd_fill_stereo_frame: %s", cudaGetErrorString(e));
  return KVFE_OK;
}

// the frame-level stereo kernels work on frame slot 0 of stream 0: a stage call fills the fields a kernel reads
static int stage_frame_begin(kvfe_ctx* ctx, int n) {
  if (n > ctx->dc.cap) return set_err(ctx, KVFE_ERR_CAPACITY, "n %d exceeds capacity %d", n, ctx->dc.cap);
  if (ctx->n_submitted != ctx->n_waited) return set_err(ctx, KVFE_ERR_STATE, "stage call with frame-level steps in flight");
  RET(park_other_streams(ctx));
  return set_stage_state(ctx, 2, 0, n);
}

extern "C" int kvfe_undistort_rectify_left_keypoints(kvfe_ctx* ctx, const float* x, const float* y, int n, int32_t* status,
                                                     float* rect_x, float* rect_y) {
  if (!ctx || !x || !y || !status || !rect_x || !rect_y) return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  if (n <= 0) return KVFE_OK;
  RET(stage_frame_begin(ctx, n));
  const FrameSoA& f = ctx->db.fr;
  CU(cudaMemcpyAsync(f.kx, x, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(f.ky, y, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  ctx->launches += launch_sparse_stereo_part(ctx->dc, ctx->db, ctx->d_cam, 1 << 2, 0, ctx->stream);
  CHECK_LAUNCH();
  CU(cudaMemcpyAsync(status, f.lstat, n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaMemcpyAsync(rect_x, f.lrx, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaMemcpyAsync(rect_y, f.lry, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return KVFE_OK;
}

extern "C" int kvfe_right_keypoints_rectified(kvfe_ctx* ctx, const uint8_t* left_rectified, const uint8_t* right_rectified, size_t pitch,
                                              const int32_t* left_status, const float* left_x, const float* left_y, int n,
                                              int32_t* right_status, float* right_x, float* right_y) {
  if (!ctx || !left_rectified || !right_rectified || !left_status || !left_x || !left_y || !right_status || !right_x || !right_y)
    return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  if (n <= 0) return KVFE_OK;
  RET(stage_frame_begin(ctx, n));
  const DevCfg& dc = ctx->dc; DevBuf& db = ctx->db;
  const FrameSoA& f = db.fr;
  RET(upload_image(ctx, db.rectL, dc.pitch, left_rectified, pitch));
  RET(upload_image(ctx, db.rectR, dc.pitch, right_rectified, pitch));
  CU(cudaMemcpyAsync(f.lstat, left_status, n * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(f.lrx, left_x, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(f.lry, left_y, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  ctx->launches += launch_sparse_stereo_part(dc, db, ctx->d_cam, 1 << 2, 1, ctx->stream);
  CHECK_LAUNCH();
  CU(cudaMemcpyAsync(right_status, f.rstat, n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaMemcpyAsync(right_x, f.rrx, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaMemcpyAsync(right_y, f.rry, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return KVFE_OK;
}

extern "C" int kvfe_depth_from_rectified_matches(kvfe_ctx* ctx, const int32_t* left_status, const float* left_x,
                                                 int32_t* right_status, const float* right_x, int n, double* depth) {
  if (!ctx || !left_status || !left_x || !right_status || !right_x || !depth) return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  if (n <= 0) return KVFE_OK;
  RET(stage_frame_begin(ctx, n));
  const DevCfg& dc = ctx->dc; DevBuf& db = ctx->db;
  const FrameSoA& f = db.fr;
  CU(cudaMemcpyAsync(f.lstat, left_status, n * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(f.lrx, left_x, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(f.rstat, right_status, n * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(f.rrx, right_x, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemsetAsync(f.rry, 0, n * sizeof(float), ctx->stream));
  CU(cudaMemsetAsync(f.versor, 0, 3 * (size_t)n * sizeof(double), ctx->stream));
  ctx->launches += launch_sparse_stereo_part(dc, db, ctx->d_cam, 1 << 2, 2, ctx->stream);
  CHECK_LAUNCH();
  CU(cudaMemcpyAsync(right_status, f.rstat, n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaMemcpyAsync(depth, f.depth, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return KVFE_OK;
}

extern "C" int kvfe_compute_median_disparity(kvfe_ctx* ctx, const float* ref_x, const float* ref_y, int n_ref, const float* cur_x,
                                             const float* cur_y, int n_cur, const int32_t* match_ref, const int32_t* match_cur,
                                             int n_matches, double* median, int* ok) {
  if (!ctx || !ref_x || !ref_y || !cur_x || !cur_y || !median || !ok || (n_matches > 0 && (!match_ref || !match_cur)))
    return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  const DevCfg& dc = ctx->dc; DevBuf& db = ctx->db;
  if (n_ref > dc.cap || n_cur > dc.cap || n_matches > dc.cap) return set_err(ctx, KVFE_ERR_CAPACITY, "more keypoints than capacity %d", dc.cap);
  for (int i = 0; i < n_matches; ++i)
    if (match_ref[i] < 0 || match_ref[i] >= n_ref || match_cur[i] < 0 || match_cur[i] >= n_cur) return set_err(ctx, KVFE_ERR_INVALID_ARG, "match index out of range");
  *median = 0.0; *ok = 0;
  if (n_matches <= 0) return KVFE_OK;                 // Tracker.cpp:995-999: false, nothing computed
  RET(stage_frame_begin(ctx, n_cur));
  const FrameSoA& f = db.fr;
  CU(cudaMemcpyAsync(f.kx, cur_x, n_cur * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));                   // slot 0 = cur
  CU(cudaMemcpyAsync(f.ky, cur_y, n_cur * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(f.kx + dc.cap, ref_x, n_ref * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));          // slot 1 = ref
  CU(cudaMemcpyAsync(f.ky + dc.cap, ref_y, n_ref * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(db.m_ref, match_ref, n_matches * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(db.m_cur, match_cur, n_matches * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  StageScratch d;
  CU(d.alloc(2 * sizeof(double)));
  ctx->launches += launch_median_disparity_raw(dc, db, n_matches, reinterpret_cast<double*>(d.p), ctx->stream);
  CHECK_LAUNCH();
  double h[2] = {0, 0};
  CU(cudaMemcpyAsync(h, d.p, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  *median = h[0]; *ok = h[1] != 0.0;
  return KVFE_OK;
}

extern "C" int kvfe_point3_and_covariance(kvfe_ctx* ctx, const float* left_x, const float* right_x, const float* left_y,
                                          const double* points_3d, int n, const double* R, double* out_points, double* out_cov) {
  if (!ctx || !left_x || !right_x || !left_y || !points_3d || !out_points || !out_cov) return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  if (n <= 0) return KVFE_OK;
  StageScratch d;
  const size_t fbytes = 3 * (size_t)n * sizeof(float), pbytes = 3 * (size_t)n * sizeof(double);
  const size_t off_p = (fbytes + 15) & ~(size_t)15, off_R = off_p + pbytes, off_op = off_R + 16 * sizeof(double), off_cov = off_op + pbytes;
  CU(d.alloc(off_cov + 9 * (size_t)n * sizeof(double)));
  float* f = reinterpret_cast<float*>(d.p);
  double* dp = reinterpret_cast<double*>(d.p + off_p);
  double* dR = reinterpret_cast<double*>(d.p + off_R);
  double* dop = reinterpret_cast<double*>(d.p + off_op);
  double* dcov = reinterpret_cast<double*>(d.p + off_cov);
  CU(cudaMemcpyAsync(f, left_x, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(f + n, right_x, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(f + 2 * (size_t)n, left_y, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(dp, points_3d, pbytes, cudaMemcpyHostToDevice, ctx->stream));
  if (R) CU(cudaMemcpyAsync(dR, R, 9 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  ctx->launches += launch_point3_cov_raw(ctx->dc, f, f + n, f + 2 * (size_t)n, dp, n, R ? dR : nullptr, dop, dcov, ctx->stream);
  CHECK_LAUNCH();
  CU(cudaMemcpyAsync(out_points, dop, pbytes, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaMemcpyAsync(out_cov, dcov, 9 * (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return KVFE_OK;
}

// Tracker::findMatchingKeypoints (Tracker.cpp:919-946): (ref index, cur index) of the keypoints that observe the same
// landmark, in the order of the current frame; a landmark id seen twice in the reference frame resolves to its last
// position (std::map assignment).  Host logic, as in the reference (the frame-level step does it on the device:
// matches.cuh).  match_ref / match_cur must hold n_cur entries.
extern "C" int kvfe_find_matching_keypoints(const int64_t* ref_landmarks, int n_ref, const int64_t* cur_landmarks, int n_cur,
                                            int32_t* match_ref, int32_t* match_cur, int* n_matches) {
  if (n_ref < 0 || n_cur < 0 || (n_ref > 0 && !ref_landmarks) || (n_cur > 0 && (!cur_landmarks || !match_ref || !match_cur)) || !n_matches)
    return KVFE_ERR_INVALID_ARG;
  std::map<int64_t, int32_t> ref_index;
  for (int i = 0; i < n_ref; ++i) if (ref_landmarks[i] != -1) ref_index[ref_landmarks[i]] = i;
  int m = 0;
  for (int i = 0; i < n_cur; ++i) {
    if (cur_landmarks[i] == -1) continue;
    auto it = ref_index.find(cur_landmarks[i]);
    if (it != ref_index.end()) { match_ref[m] = it->second; match_cur[m] = i; ++m; }
  }
  *n_matches = m;
  return KVFE_OK;
}
// Tracker::findMatchingStereoKeypoints (Tracker.cpp:948-989): the mono matches whose right keypoints are VALID in both
// frames.  match_ref / match_cur may alias the inputs.
extern "C" int kvfe_find_matching_stereo_keypoints(const int32_t* ref_right_status, int n_ref, const int32_t* cur_right_status, int n_cur,
                                                   const int32_t* mono_match_ref, const int32_t* mono_match_cur, int n_mono,
                                                   int32_t* match_ref, int32_t* match_cur, int* n_matches) {
  if (n_mono < 0 || !n_matches || (n_mono > 0 && (!ref_right_status || !cur_right_status || !mono_match_ref || !mono_match_cur || !match_ref || !match_cur)))
    return KVFE_ERR_INVALID_ARG;
  int m = 0;
  for (int i = 0; i < n_mono; ++i) {
    const int ir = mono_match_ref[i], ic = mono_match_cur[i];
    if (ir < 0 || ir >= n_ref || ic < 0 || ic >= n_cur) return KVFE_ERR_INVALID_ARG;
    if (ref_right_status[ir] == KVFE_KP_VALID && cur_right_status[ic] == KVFE_KP_VALID) { match_ref[m] = ir; match_cur[m] = ic; ++m; }
  }
  *n_matches = m;
  return KVFE_OK;
}
// StereoVisionImuFrontend::getSmartStereoMeasurements (StereoVisionImuFrontend.cpp:485-531; use_right =
// use_stereo_tracking_) and RgbdVisionImuFrontend::fillSmartStereoMeasurements (RgbdVisionImuFrontend.cpp:368-395;
// use_right = 1): one (landmark, uL, uR, v) per keypoint with a landmark, uR = NaN unless the right keypoint is VALID.
extern "C" int kvfe_smart_stereo_measurements(const int64_t* landmarks, const float* left_x, const float* left_y,
                                              const int32_t* right_status, const float* right_x, int n, int use_right,
                                              int64_t* out_landmarks, double* out_uL, double* out_uR, double* out_v, int* n_out) {
  if (n < 0 || !n_out || (n > 0 && (!landmarks || !left_x || !left_y || !right_status || !right_x || !out_landmarks || !out_uL || !out_uR || !out_v)))
    return KVFE_ERR_INVALID_ARG;
  int m = 0;
  for (int i = 0; i < n; ++i) {
    if (landmarks[i] == -1) continue;
    out_landmarks[m] = landmarks[i];
    out_uL[m] = (double)left_x[i];
    out_v[m] = (double)left_y[i];
    out_uR[m] = (use_right && right_status[i] == KVFE_KP_VALID) ? (double)right_x[i] : std::numeric_limits<double>::quiet_NaN();
    ++m;
  }
  *n_out = m;
  return KVFE_OK;
}

// VisionImuFrontend::shouldBeKeyframe (VisionImuFrontend.cpp:175-232) from the quantities the caller holds: the two
// timestamps, Frame::getNrValidKeypoints, the median disparity of computeMedianDisparity over findMatchingKeypoints(lkf,
// frame) (0.0 when there is no match, Tracker.cpp:1004-1008), kfTrackingStatus_mono_ and Frame::isKeyframe_.  The
// frame-level step takes the same decision on the device (fsm.cu: decide_kernel).
extern "C" int kvfe_should_be_keyframe(const kvfe_config* cfg, int64_t timestamp_ns, int64_t lkf_timestamp_ns, int nr_valid_features,
                                       double median_disparity, int mono_status, int user_keyframe, int* is_keyframe) {
  if (!cfg || !is_keyframe) return KVFE_ERR_INVALID_ARG;
  const int64_t kf_diff_ns = timestamp_ns - lkf_timestamp_ns;
  const bool min_time_elapsed = kf_diff_ns >= cfg->min_intra_keyframe_time_ns;
  const bool max_time_elapsed = kf_diff_ns >= cfg->max_intra_keyframe_time_ns;
  const bool nr_features_low = nr_valid_features <= cfg->min_number_features;
  const bool is_disparity_low = median_disparity < cfg->disparity_threshold;
  const bool disparity_low_first_time = is_disparity_low && !(mono_status == KVFE_TRK_LOW_DISPARITY);
  const bool enough_disparity = !is_disparity_low;
  const bool max_disparity_reached = median_disparity > cfg->max_disparity_since_lkf;
  const bool disparity_flipped = (enough_disparity || disparity_low_first_time) && min_time_elapsed;
  *is_keyframe = (max_time_elapsed || max_disparity_reached || disparity_flipped || nr_features_low || user_keyframe) ? 1 : 0;
  return KVFE_OK;
}

// Tracker::findOutliers (Tracker.cpp:836-853): the match indices that are not in the (sorted or unsorted) inlier list,
// ascending.  Host logic: the reference's own implementation is a std::set_difference on the host.
extern "C" int kvfe_find_outliers(int n_matches, const int32_t* inliers, int n_inliers, int32_t* outliers, int* n_outliers) {
  if (n_matches < 0 || n_inliers < 0 || (n_inliers > 0 && !inliers) || !outliers || !n_outliers) return KVFE_ERR_INVALID_ARG;
  std::vector<char> in(n_matches, 0);
  for (int i = 0; i < n_inliers; ++i) if (inliers[i] >= 0 && inliers[i] < n_matches) in[inliers[i]] = 1;
  int m = 0;
  for (int i = 0; i < n_matches; ++i) if (!in[i]) outliers[m++] = i;
  *n_outliers = m;
  return KVFE_OK;
}
// Tracker::removeOutliersMono (Tracker.cpp:856-882): landmarks of the outlier matches become -1 in both frames and the
// match list is reduced to the inliers (in inlier-list order).
extern "C" int kvfe_remove_outliers_mono(const int32_t* inliers, int n_inliers, int64_t* ref_landmarks, int n_ref,
                                         int64_t* cur_landmarks, int n_cur, int32_t* match_ref, int32_t* match_cur, int* n_matches) {
  if (!ref_landmarks || !cur_landmarks || !match_ref || !match_cur || !n_matches || (n_inliers > 0 && !inliers)) return KVFE_ERR_INVALID_ARG;
  const int nm = *n_matches;
  std::vector<int32_t> out(nm > 0 ? nm : 1);
  int no = 0;
  int rc = kvfe_find_outliers(nm, inliers, n_inliers, out.data(), &no);
  if (rc != KVFE_OK) return rc;
  for (int k = 0; k < no; ++k) {
    const int ir = match_ref[out[k]], ic = match_cur[out[k]];
    if (ir < 0 || ir >= n_ref || ic < 0 || ic >= n_cur) return KVFE_ERR_INVALID_ARG;
    ref_landmarks[ir] = -1; cur_landmarks[ic] = -1;
  }
  std::vector<int32_t> mr(n_inliers > 0 ? n_inliers : 1), mc(n_inliers > 0 ? n_inliers : 1);
  for (int k = 0; k < n_inliers; ++k) {
    if (inliers[k] < 0 || inliers[k] >= nm) return KVFE_ERR_INVALID_ARG;
    mr[k] = match_ref[inliers[k]]; mc[k] = match_cur[inliers[k]];
  }
  for (int k = 0; k < n_inliers; ++k) { match_ref[k] = mr[k]; match_cur[k] = mc[k]; }
  *n_matches = n_inliers;
  return KVFE_OK;
}
// Tracker::removeOutliersStereo (Tracker.cpp:884-917): outlier matches get right status FAILED_ARUN, depth 0 and a
// zero 3-D point in both frames; the match list is reduced to the inliers.
extern "C" int kvfe_remove_outliers_stereo(const int32_t* inliers, int n_inliers, int32_t* ref_right_status, double* ref_depth,
                                           double* ref_points_3d, int n_ref, int32_t* cur_right_status, double* cur_depth,
                                           double* cur_points_3d, int n_cur, int32_t* match_ref, int32_t* match_cur, int* n_matches) {
  if (!ref_right_status || !ref_depth || !ref_points_3d || !cur_right_status || !cur_depth || !cur_points_3d || !match_ref || !match_cur ||
      !n_matches || (n_inliers > 0 && !inliers)) return KVFE_ERR_INVALID_ARG;
  const int nm = *n_matches;
  std::vector<int32_t> out(nm > 0 ? nm : 1);
  int no = 0;
  int rc = kvfe_find_outliers(nm, inliers, n_inliers, out.data(), &no);
  if (rc != KVFE_OK) return rc;
  for (int k = 0; k < no; ++k) {
    const int ir = match_ref[out[k]], ic = match_cur[out[k]];
    if (ir < 0 || ir >= n_ref || ic < 0 || ic >= n_cur) return KVFE_ERR_INVALID_ARG;
    ref_right_status[ir] = KVFE_KP_FAILED_ARUN; ref_depth[ir] = 0.0;
    cur_right_status[ic] = KVFE_KP_FAILED_ARUN; cur_depth[ic] = 0.0;
    for (int a = 0; a < 3; ++a) { ref_points_3d[3 * (size_t)ir + a] = 0.0; cur_points_3d[3 * (size_t)ic + a] = 0.0; }
  }
  std::vector<int32_t> mr(n_inliers > 0 ? n_inliers : 1), mc(n_inliers > 0 ? n_inliers : 1);
  for (int k = 0; k < n_inliers; ++k) {
    if (inliers[k] < 0 || inliers[k] >= nm) return KVFE_ERR_INVALID_ARG;
    mr[k] = match_ref[inliers[k]]; mc[k] = match_cur[inliers[k]];
  }
  for (int k = 0; k < n_inliers; ++k) { match_ref[k] = mr[k]; match_cur[k] = mc[k]; }
  *n_matches = n_inliers;
  return KVFE_OK;
}

extern "C" int kvfe_equalize_hist(kvfe_ctx* ctx, const uint8_t* img, size_t pitch, uint8_t* out, size_t out_pitch) {
  if (!ctx || !img || !out) return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  if (ctx->n_submitted != ctx->n_waited) return set_err(ctx, KVFE_ERR_STATE, "stage call with frame-level steps in flight");
  const DevCfg& dc = ctx->dc; DevBuf& db = ctx->db;
  unsigned char* L = db.pyr[0] + dc.lvl_off[0];
  RET(upload_image(ctx, L, dc.pitch, img, pitch));
  ctx->launches += launch_equalize(dc, L, dc.pyr_stride, 1, nullptr, 0, ctx->stream);
  CHECK_LAUNCH();
  RET(download_image(ctx, out, out_pitch, L, dc.pitch));
  CU(cudaStreamSynchronize(ctx->stream));
  return KVFE_OK;
}

extern "C" int kvfe_mesh_2d(kvfe_ctx* ctx, const float* kp_x, const float* kp_y, int n, float* triangles, int max_triangles,
                            int* n_triangles) {
  if (!ctx || !kp_x || !kp_y || !triangles || !n_triangles || max_triangles < 0) return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  const DevCfg& dc = ctx->dc;
  if (n < 0 || n > dc.cap) return set_err(ctx, KVFE_ERR_CAPACITY, "n %d exceeds capacity %d", n, dc.cap);
  *n_triangles = 0;
  if (n == 0) return KVFE_OK;                     // Mesher.cpp:1716
  float* d = nullptr;
  const size_t mt = (size_t)std::min(max_triangles, 2 * n + 8);
  CU(cudaMalloc((void**)&d, (2 * (size_t)n + 6 * mt + 2) * sizeof(float)));
  float* dtri = d + 2 * n; int* dn = reinterpret_cast<int*>(dtri + 6 * mt);
  CU(cudaMemcpyAsync(d, kp_x, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(d + n, kp_y, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  ctx->launches += launch_mesh_raw(dc, ctx->db, d, d + n, n, dtri, (int)mt, dn, ctx->stream);
  CHECK_LAUNCH();
  int nt = 0;
  CU(cudaMemcpyAsync(&nt, dn, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  const size_t copy = std::min((size_t)nt, mt);
  if (copy) CU(cudaMemcpy(triangles, dtri, copy * 6 * sizeof(float), cudaMemcpyDeviceToHost));
  cudaFree(d);
  *n_triangles = nt;
  return KVFE_OK;
}

// ---- RANSAC stage calls ---------------------------------------------------------------------------
struct DevScratch {
  void* p = nullptr;
  ~DevScratch() { if (p) cudaFree(p); }
};

static int compact_inliers(const std::vector<int>& flags, int n, int32_t* inliers, int* n_inliers) {
  int m = 0;
  for (int i = 0; i < n; ++i) if (flags[i]) inliers[m++] = i;
  *n_inliers = m;
  return KVFE_OK;
}

extern "C" int kvfe_ransac_mono(kvfe_ctx* ctx, const double* f_ref, const double* f_cur, int n, const double* R12,
                                int32_t* inliers, int* n_inliers, double* pose, int* status) {
  if (!ctx || !f_ref || !f_cur || !inliers || !n_inliers || !pose || !status) return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  const DevCfg& dc = ctx->dc;
  if (n > dc.cap || n < 0) return set_err(ctx, KVFE_ERR_CAPACITY, "n %d exceeds capacity %d", n, dc.cap);
  if (n == 0) { *n_inliers = 0; *status = KVFE_TRK_INVALID; for (int i = 0; i < 12; ++i) pose[i] = (i % 5 == 0); return KVFE_OK; }
  DevScratch sc;
  size_t bytes = sizeof(double) * (6 * (size_t)n + 9 + 12) + sizeof(int) * ((size_t)n + 2);
  CU(cudaMalloc(&sc.p, bytes));
  double* d_a = (double*)sc.p; double* d_b = d_a + 3 * n; double* d_R = d_b + 3 * n; double* d_pose = d_R + 9;
  int* d_inl = (int*)(d_pose + 12); int* d_n = d_inl + n; int* d_st = d_n + 1;
  CU(cudaMemcpyAsync(d_a, f_ref, 3 * (size_t)n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(d_b, f_cur, 3 * (size_t)n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  if (R12) CU(cudaMemcpyAsync(d_R, R12, 9 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  ctx->launches += launch_ransac_mono_raw(dc, ctx->db, d_a, d_b, n, R12 ? d_R : nullptr, R12 ? 1 : 0, d_inl, d_n, d_pose, d_st, ctx->stream);
  CHECK_LAUNCH();
  std::vector<int> flags(n);
  CU(cudaMemcpyAsync(flags.data(), d_inl, n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaMemcpyAsync(pose, d_pose, 12 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaMemcpyAsync(status, d_st, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return compact_inliers(flags, n, inliers, n_inliers);
}

extern "C" int kvfe_ransac_stereo_3pt(kvfe_ctx* ctx, const double* ref_3d, const double* cur_3d, int n,
                                      int32_t* inliers, int* n_inliers, double* pose, int* status) {
  if (!ctx || !ref_3d || !cur_3d || !inliers || !n_inliers || !pose || !status) return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  const DevCfg& dc = ctx->dc;
  if (n > dc.cap || n < 0) return set_err(ctx, KVFE_ERR_CAPACITY, "n %d exceeds capacity %d", n, dc.cap);
  if (n == 0) { *n_inliers = 0; *status = KVFE_TRK_INVALID; for (int i = 0; i < 12; ++i) pose[i] = (i % 5 == 0); return KVFE_OK; }
  DevScratch sc;
  size_t bytes = sizeof(double) * (6 * (size_t)n + 12) + sizeof(int) * ((size_t)n + 2);
  CU(cudaMalloc(&sc.p, bytes));
  double* d_a = (double*)sc.p; double* d_b = d_a + 3 * n; double* d_pose = d_b + 3 * n;
  int* d_inl = (int*)(d_pose + 12); int* d_n = d_inl + n; int* d_st = d_n + 1;
  CU(cudaMemcpyAsync(d_a, ref_3d, 3 * (size_t)n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(d_b, cur_3d, 3 * (size_t)n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  ctx->launches += launch_ransac_3pt_raw(dc, ctx->db, d_a, d_b, n, d_inl, d_n, d_pose, d_st, ctx->stream);
  CHECK_LAUNCH();
  std::vector<int> flags(n);
  CU(cudaMemcpyAsync(flags.data(), d_inl, n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaMemcpyAsync(pose, d_pose, 12 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaMemcpyAsync(status, d_st, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return compact_inliers(flags, n, inliers, n_inliers);
}

extern "C" int kvfe_ransac_stereo_1pt(kvfe_ctx* ctx, const float* ref_left_xy, const float* ref_right_xy,
                                      const float* cur_left_xy, const float* cur_right_xy, const double* ref_3d,
                                      const double* cur_3d, int n, const double* R, int32_t* inliers,
                                      int* n_inliers, double* pose, double* info, int* status) {
  if (!ctx || !ref_left_xy || !ref_right_xy || !cur_left_xy || !cur_right_xy || !ref_3d || !cur_3d || !R || !inliers ||
      !n_inliers || !pose || !info || !status)
    return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  const DevCfg& dc = ctx->dc;
  if (n > dc.cap || n < 0) return set_err(ctx, KVFE_ERR_CAPACITY, "n %d exceeds capacity %d", n, dc.cap);
  if (n == 0) { *n_inliers = 0; *status = KVFE_TRK_INVALID; for (int i = 0; i < 12; ++i) pose[i] = (i % 5 == 0); for (int i = 0; i < 9; ++i) info[i] = 0; return KVFE_OK; }
  DevScratch sc;
  size_t bytes = sizeof(double) * (6 * (size_t)n + 9 + 12 + 9) + sizeof(float) * 8 * (size_t)n + sizeof(int) * ((size_t)n + 2);
  CU(cudaMalloc(&sc.p, bytes));
  double* d_a = (double*)sc.p; double* d_b = d_a + 3 * n; double* d_R = d_b + 3 * n; double* d_pose = d_R + 9; double* d_info = d_pose + 12;
  float* d_rl = (float*)(d_info + 9); float* d_rr = d_rl + 2 * n; float* d_cl = d_rr + 2 * n; float* d_cr = d_cl + 2 * n;
  int* d_inl = (int*)(d_cr + 2 * n); int* d_n = d_inl + n; int* d_st = d_n + 1;
  CU(cudaMemcpyAsync(d_a, ref_3d, 3 * (size_t)n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(d_b, cur_3d, 3 * (size_t)n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(d_R, R, 9 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(d_rl, ref_left_xy, 2 * (size_t)n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(d_rr, ref_right_xy, 2 * (size_t)n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(d_cl, cur_left_xy, 2 * (size_t)n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(d_cr, cur_right_xy, 2 * (size_t)n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  ctx->launches += launch_ransac_1pt_raw(dc, ctx->db, d_rl, d_rr, d_cl, d_cr, d_a, d_b, n, d_R, d_inl, d_n, d_pose, d_info, d_st, ctx->stream);
  CHECK_LAUNCH();
  std::vector<int> flags(n);
  CU(cudaMemcpyAsync(flags.data(), d_inl, n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaMemcpyAsync(pose, d_pose, 12 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaMemcpyAsync(info, d_info, 9 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaMemcpyAsync(status, d_st, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return compact_inliers(flags, n, inliers, n_inliers);
}

// ---- frame-level step ---------------------------------------------------------------------------
// The packets of the frame-level steps are assembled by finalize_kernel directly in `packets_dev` (batch *
// kvfe_packet_bytes() bytes of device memory owned by the caller, e.g. the send buffer of an NCCL gather: the optional
// gather of the keypoint packets to rank 0 then needs no pack / copy kernel).  NULL restores the internal buffer.
// The captured step graphs hold the buffer address: they are rebuilt on the next step.
extern "C" int kvfe_frontend_bind_packets(kvfe_ctx* ctx, uint8_t* packets_dev) {
  if (!ctx) return KVFE_ERR_INVALID_ARG;
  if (ctx->n_submitted != ctx->n_waited) return set_err(ctx, KVFE_ERR_STATE, "bind_packets with steps in flight");
  CU(cudaStreamSynchronize(ctx->stream));
  if (!ctx->own_packets) ctx->own_packets = ctx->db.packets;
  ctx->db.packets = packets_dev ? packets_dev : ctx->own_packets;
  for (int i = 0; i < 2; ++i) {
    if (ctx->graph_ready[i]) { cudaGraphExecDestroy(ctx->step_graph[i]); ctx->graph_ready[i] = 0; }
    if (ctx->host_graph_ready[i]) { cudaGraphExecDestroy(ctx->host_graph[i]); ctx->host_graph_ready[i] = 0; }
  }
  return KVFE_OK;
}

extern "C" int kvfe_frontend_force_keyframe(kvfe_ctx* ctx, const int32_t* flags) {
  if (!ctx || !flags) return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  // consumed (and cleared) by the next step's keyframe decision; enqueued on the context's stream like the step itself
  std::vector<int> h(flags, flags + ctx->dc.B);
  for (int& v : h) v = v ? 1 : 0;
  CU(cudaMemcpy(ctx->db.force_kf, h.data(), h.size() * sizeof(int), cudaMemcpyHostToDevice));
  return KVFE_OK;
}

extern "C" int kvfe_frontend_reset(kvfe_ctx* ctx) {
  if (!ctx) return KVFE_ERR_INVALID_ARG;
  ctx->launches += launch_reset(ctx->dc, ctx->db, ctx->stream);
  CU(cudaGetLastError());
  CU(cudaStreamSynchronize(ctx->stream));
  ctx->cur_slot = 0;
  return KVFE_OK;
}

// The stereo / mono frame-level entry points take no depth image: an RGB-D context goes through kvfe_frontend_step_rgbd
// or kvfe_pipeline_push_rgbd
static int refuse_rgbd(kvfe_ctx* ctx, const char* fn) {
  return set_err(ctx, KVFE_ERR_INVALID_ARG, "%s: this is an RGB-D context (frontend_type 2): use kvfe_frontend_step_rgbd or "
                 "kvfe_pipeline_push_rgbd", fn);
}

// The fixed kernel sequence of one step; images of the current frame already sit in
// pyr[cur_slot] level 0 (left) and right_raw (right).  Three parts: (1) tracking up to the keyframe
// decision, (2) the keyframe / detection part (every kernel of it exits at entry for a stream in
// plain tracking mode), (3) packet assembly.
static int enqueue_part_track(kvfe_ctx* ctx, unsigned long long cond, long long* n_launch, const StepIO* io = nullptr) {
  const DevCfg& dc = ctx->dc; DevBuf& db = ctx->db; cudaStream_t s = ctx->stream;
  const int cur = ctx->cur_slot, prev = cur ^ 1;
  long long n = 0;
  n += launch_prep(dc, db, ctx->d_cam, ctx->in_ts ? ctx->in_ts : ctx->d_ts, ctx->in_R ? ctx->in_R : ctx->d_Rin, io, s);
  if (dc.equalize) {       // what the reference's data provider does at load time (UtilsOpenCV.cpp:390-403)
    n += launch_equalize(dc, db.pyr[cur] + dc.lvl_off[0], dc.pyr_stride, dc.B, nullptr, 0, s);
    if (!dc.rgbd) n += launch_equalize(dc, db.right_raw, dc.img_stride, dc.B, nullptr, 0, s);   // RGB-D: never the depth
  }
  n += launch_pyramid(dc, db.pyr[cur], dc.B, s);
  n += launch_track_pre(dc, db, s);
  n += launch_lk(dc, db, prev, cur, s);
  n += launch_track_post(dc, db, ctx->d_cam, s);
  n += launch_decide(dc, db, cond, s);
  *n_launch += n;
  CU(cudaGetLastError());
  return KVFE_OK;
}

static int enqueue_part_keyframe(kvfe_ctx* ctx, int* kf_counter, long long* n_launch, const StepIO* io = nullptr) {
  const DevCfg& dc = ctx->dc; DevBuf& db = ctx->db; cudaStream_t s = ctx->stream;
  const int cur = ctx->cur_slot;
  const int M_BOOT = 1 << 0, M_KF = 1 << 2, M_LOST = 1 << 3;
  unsigned char* Lcur = db.pyr[cur] + dc.lvl_off[0];
  long long n = 0;
  // pipeline step: the right image crosses the host link only when the frame is a keyframe (or the first frame)
  if (io) n += launch_fetch_right_io(dc, db, io, cur, M_KF | M_BOOT, s);
  if (dc.rgbd) {
    // RgbdVisionImuFrontend::processFirstFrame / handleKeyframe (RgbdVisionImuFrontend.cpp:183-209, :300-368): the depth
    // image crosses the host link only now, for the streams that need it
    if (io) n += launch_fetch_depth_io(dc, db, io, M_BOOT | M_KF, s);
    n += launch_ransac_mono(dc, db, M_KF, s);
    // Camera::undistortKeypoints of the tracked keypoints (left_rect_kernel with R1 = I, P1 = [K | 0]); the reference does it
    // right after tracking, which is the same: mono RANSAC changes landmarks, not keypoints
    n += launch_sparse_stereo_part(dc, db, ctx->d_cam, M_KF, 0, s);
    n += launch_rgbd_fill_batch(dc, db, ctx->d_cam, M_KF, s);
    n += launch_ransac_stereo(dc, db, M_KF, s);                 // fake stereo camera; INVALID without use_stereo_tracking
    // detection with the depth mask (the circles of the tracked keypoints are drawn into it), then undistortKeypoints and
    // fillStereoFrame again over ALL keypoints
    n += launch_detect_pre(dc, db, M_BOOT | M_KF, kf_counter, s);
    n += launch_depth_mask_batch(dc, db, M_BOOT | M_KF, s);
    n += launch_gftt(dc, db, Lcur, dc.pyr_stride, ctx->circle_hw, ctx->circle_r, M_BOOT | M_KF, s, 1);
    n += launch_select(dc, db, Lcur, dc.pyr_stride, ctx->d_cam, M_BOOT | M_KF, 1, s);
    n += launch_sparse_stereo_part(dc, db, ctx->d_cam, M_BOOT | M_KF, 0, s);
    n += launch_rgbd_fill_batch(dc, db, ctx->d_cam, M_BOOT | M_KF, s);
    *n_launch += n;
    CU(cudaGetLastError());
    return KVFE_OK;
  }
  if (dc.mono) {
    // MonoVisionImuFrontend::processFrame (MonoVisionImuFrontend.cpp:271-316): mono RANSAC, detection,
    // Camera::undistortKeypoints (left_rect_kernel with R1 = I, P1 = [K | 0]); no stereo half
    n += launch_ransac_mono(dc, db, M_KF, s);
    n += launch_detect_pre(dc, db, M_BOOT | M_KF, kf_counter, s);
    n += launch_gftt(dc, db, Lcur, dc.pyr_stride, ctx->circle_hw, ctx->circle_r, M_BOOT | M_KF, s);
    n += launch_select(dc, db, Lcur, dc.pyr_stride, ctx->d_cam, M_BOOT | M_KF, 1, s);
    n += launch_sparse_stereo_part(dc, db, ctx->d_cam, M_BOOT | M_KF, 0, s);
    *n_launch += n;
    CU(cudaGetLastError());
    return KVFE_OK;
  }
  // keyframe: mono RANSAC -> sparse stereo -> stereo RANSAC
  n += launch_ransac_mono(dc, db, M_KF, s);
  n += launch_rectify(dc, db.rmap[0], Lcur, dc.pyr_stride, db.rectL, dc.img_stride, dc.B, db.st, M_KF | M_BOOT, s);
  n += launch_rectify(dc, db.rmap[1], db.right_raw, dc.img_stride, db.rectR, dc.img_stride, dc.B, db.st, M_KF | M_BOOT, s);
  n += launch_sparse_stereo(dc, db, ctx->d_cam, M_KF, 0, s);
  n += launch_ransac_stereo(dc, db, M_KF, s);
  // detection (bootstrap, keyframe, all-tracks-lost)
  n += launch_detect_pre(dc, db, M_BOOT | M_KF | M_LOST, kf_counter, s);
  n += launch_gftt(dc, db, Lcur, dc.pyr_stride, ctx->circle_hw, ctx->circle_r, M_BOOT | M_KF | M_LOST, s);
  n += launch_select(dc, db, Lcur, dc.pyr_stride, ctx->d_cam, M_BOOT | M_KF | M_LOST, 1, s);
  // sparse stereo over all keypoints incl. the new ones (the second remap of the reference is
  // idempotent -- same raw images, same maps -- and is therefore not repeated)
  n += launch_sparse_stereo(dc, db, ctx->d_cam, M_BOOT | M_KF, 1, s);
  *n_launch += n;
  CU(cudaGetLastError());
  return KVFE_OK;
}

__global__ void kvfe_empty_kernel() {}

static int enqueue_part_finalize(kvfe_ctx* ctx, long long* n_launch) {
  *n_launch += launch_finalize(ctx->dc, ctx->db, ctx->stream);
  if (ctx->dc.mesh_on) *n_launch += launch_mesh(ctx->dc, ctx->db, ctx->stream);
  if (const char* e = getenv("KVFE_EXTRA_LAUNCHES"))      // diagnostic: dispatch-rate sensitivity
    for (int i = 0; i < atoi(e); ++i) kvfe_empty_kernel<<<1, 32, 0, ctx->stream>>>();
  CU(cudaGetLastError());
  return KVFE_OK;
}

static int enqueue_step_kernels(kvfe_ctx* ctx, long long* n_launch) {
  *n_launch = 0;
  RET(enqueue_part_track(ctx, 0ull, n_launch));
  RET(enqueue_part_keyframe(ctx, nullptr, n_launch));
  return enqueue_part_finalize(ctx, n_launch);
}
// the same sequence with the step inputs taken from a pipeline I/O block (pipeline.cu)
int kvfe_enqueue_step_kernels(kvfe_ctx* ctx, const StepIO* io, long long* n_launch) {
  *n_launch = 0;
  RET(enqueue_part_track(ctx, 0ull, n_launch, io));
  RET(enqueue_part_keyframe(ctx, nullptr, n_launch, io));
  return enqueue_part_finalize(ctx, n_launch);
}

// the pieces of a pipeline step for the split graphs (pipeline.cu)
int kvfe_enqueue_step_part(kvfe_ctx* ctx, StepIO* io, int part, long long* n_launch) {
  *n_launch = 0;
  if (part == 0) {
    RET(enqueue_part_track(ctx, 0ull, n_launch, io));
    *n_launch += launch_publish_decision(ctx->db, io, ctx->stream);
    return KVFE_OK;
  }
  if (part == 1) RET(enqueue_part_keyframe(ctx, nullptr, n_launch, io));
  return enqueue_part_finalize(ctx, n_launch);
}

// The kernel sequence of a step is identical from step to step (all arguments are by-value structs
// of device pointers; only the pyramid slot alternates), so it is built once per slot as a CUDA
// graph and replayed: one cudaGraphLaunch per step.  The keyframe part is the body of an IF node
// whose condition the decision kernel sets on the device (cudaGraphSetConditional): a step in which
// no stream of the batch is at a keyframe dispatches 10 kernels instead of 32, still without any
// host round trip.  That variant is opt-in (KVFE_GRAPH_COND=1): with many step graphs in flight on
// separate streams it measured far slower than the flat captured graph, which is the default;
// KVFE_NO_GRAPH=1 falls back to plain stream launches.
static int build_step_graph(kvfe_ctx* ctx, cudaGraphExec_t* exec, long long* n_track, long long* n_kf) {
  cudaStream_t s = ctx->stream;
  const cudaStreamCaptureMode mode = cudaStreamCaptureModeThreadLocal;
  cudaGraph_t g = nullptr, gout = nullptr;
  long long na = 0, nb = 0, nc = 0;
  if (!ctx->use_cond) {
    CU(cudaStreamBeginCapture(s, mode));
    int rc = enqueue_step_kernels(ctx, &na);
    cudaError_t e = cudaStreamEndCapture(s, &g);
    if (rc != KVFE_OK) return rc;
    if (e != cudaSuccess) return set_err(ctx, KVFE_ERR_CUDA, "graph capture failed: %s", cudaGetErrorString(e));
    CU(cudaGraphInstantiate(exec, g, 0));
    cudaGraphDestroy(g);
    *n_track = na; *n_kf = 0;
    return KVFE_OK;
  }
  CU(cudaGraphCreate(&g, 0));
  cudaGraphConditionalHandle cond;
  CU(cudaGraphConditionalHandleCreate(&cond, g, 0, cudaGraphCondAssignDefault));
  // (1) tracking part
  CU(cudaStreamBeginCaptureToGraph(s, g, nullptr, nullptr, 0, mode));
  int rc = enqueue_part_track(ctx, (unsigned long long)cond, &na);
  cudaError_t e = cudaStreamEndCapture(s, &gout);
  if (rc != KVFE_OK) return rc;
  if (e != cudaSuccess) return set_err(ctx, KVFE_ERR_CUDA, "graph capture (tracking part) failed: %s", cudaGetErrorString(e));
  // its last node: the only node without an outgoing edge (the part is a linear chain)
  size_t nn = 0, ne = 0;
  CU(cudaGraphGetNodes(g, nullptr, &nn));
  std::vector<cudaGraphNode_t> nodes(nn);
  CU(cudaGraphGetNodes(g, nodes.data(), &nn));
  CU(cudaGraphGetEdges(g, nullptr, nullptr, &ne));
  std::vector<cudaGraphNode_t> from(ne), to(ne);
  if (ne) CU(cudaGraphGetEdges(g, from.data(), to.data(), &ne));
  cudaGraphNode_t tail = nullptr;
  int n_tail = 0;
  for (cudaGraphNode_t nd : nodes) {
    bool has_out = false;
    for (size_t i = 0; i < ne; ++i) has_out |= from[i] == nd;
    if (!has_out) { tail = nd; ++n_tail; }
  }
  if (n_tail != 1) return set_err(ctx, KVFE_ERR_CUDA, "step graph: expected one tail node, found %d", n_tail);
  // (2) IF node + keyframe part as its body
  cudaGraphNodeParams cp = {};
  cp.type = cudaGraphNodeTypeConditional;
  cp.conditional.handle = cond;
  cp.conditional.type = cudaGraphCondTypeIf;
  cp.conditional.size = 1;
  cudaGraphNode_t cnode = nullptr;
  CU(cudaGraphAddNode(&cnode, g, &tail, 1, &cp));
  cudaGraph_t body = cp.conditional.phGraph_out[0];
  CU(cudaStreamBeginCaptureToGraph(s, body, nullptr, nullptr, 0, mode));
  rc = enqueue_part_keyframe(ctx, ctx->d_kf_steps, &nb);
  e = cudaStreamEndCapture(s, &gout);
  if (rc != KVFE_OK) return rc;
  if (e != cudaSuccess) return set_err(ctx, KVFE_ERR_CUDA, "graph capture (keyframe part) failed: %s", cudaGetErrorString(e));
  // (3) packet assembly after the IF node
  CU(cudaStreamBeginCaptureToGraph(s, g, &cnode, nullptr, 1, mode));
  rc = enqueue_part_finalize(ctx, &nc);
  e = cudaStreamEndCapture(s, &gout);
  if (rc != KVFE_OK) return rc;
  if (e != cudaSuccess) return set_err(ctx, KVFE_ERR_CUDA, "graph capture (finalize part) failed: %s", cudaGetErrorString(e));
  CU(cudaGraphInstantiate(exec, g, 0));
  cudaGraphDestroy(g);
  *n_track = na + nc; *n_kf = nb;
  return KVFE_OK;
}

static int enqueue_step(kvfe_ctx* ctx) {
  const int cur = ctx->cur_slot;
  if (ctx->use_graph) {
    if (!ctx->graph_ready[cur]) {
      RET(build_step_graph(ctx, &ctx->step_graph[cur], &ctx->graph_launches, &ctx->graph_launches_kf));
      ctx->graph_ready[cur] = 1;
    }
    CU(cudaGraphLaunch(ctx->step_graph[cur], ctx->stream));
    // launches of the IF body are counted by the device (StreamState::kf_steps, read at kvfe_kernel_launches)
    ctx->launches += ctx->graph_launches;
  } else {
    long long n = 0;
    RET(enqueue_step_kernels(ctx, &n));
    ctx->launches += n;
  }
  ctx->cur_slot ^= 1;
  return KVFE_OK;
}

// Step inputs (timestamps, rotations) go through a ring of pinned slots so that consecutive steps
// can be enqueued without waiting for the previous one (no host sync on the steady-state path).
static int stage_inputs(kvfe_ctx* ctx, const int64_t* timestamps, const double* keyframe_R_cur) {
  const size_t B = ctx->dc.B;
  const int slot = ctx->in_slot;
  ctx->in_slot = (slot + 1) % KVFE_IN_SLOTS;
  if (ctx->in_used[slot]) CU(cudaEventSynchronize(ctx->in_ev[slot]));
  long long* hts = ctx->h_ts + (size_t)slot * B;
  double* hR = ctx->h_Rin + (size_t)slot * B * 9;
  memcpy(hts, timestamps, B * sizeof(long long));
  memcpy(hR, keyframe_R_cur, B * 9 * sizeof(double));
  CU(cudaMemcpyAsync(ctx->d_ts, hts, B * sizeof(long long), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(ctx->d_Rin, hR, B * 9 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaEventRecord(ctx->in_ev[slot], ctx->stream));
  ctx->in_used[slot] = 1;
  return KVFE_OK;
}

extern "C" int kvfe_frontend_step_dev(kvfe_ctx* ctx, const uint8_t* left_dev, const uint8_t* right_dev, size_t pitch,
                                      const int64_t* timestamps, const double* keyframe_R_cur) {
  if (!ctx || !left_dev || !right_dev || !timestamps || !keyframe_R_cur) return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  if (ctx->dc.rgbd) return refuse_rgbd(ctx, "kvfe_frontend_step_dev");
  const DevCfg& dc = ctx->dc; DevBuf& db = ctx->db; cudaStream_t s = ctx->stream;
  const size_t B = dc.B;
  RET(stage_inputs(ctx, timestamps, keyframe_R_cur));
  // device-to-device placement into the pyramid slot / right buffer (strided destination)
  if (pitch == (size_t)dc.W && dc.pitch == dc.W) {
    // densely packed images: one strided copy per camera for the whole batch (row = one image)
    // (an SM copy kernel, not two copy-engine operations: those share in-order queues across contexts)
    const size_t img = (size_t)dc.W * dc.H;
    ctx->launches += launch_fetch(left_dev, right_dev, db.pyr[ctx->cur_slot] + dc.lvl_off[0], dc.pyr_stride, db.right_raw,
                                  dc.img_stride, img, (int)B, s);
    CU(cudaGetLastError());
  } else {
    for (size_t b = 0; b < B; ++b) {
      RET(copy_image(ctx, db.pyr[ctx->cur_slot] + b * dc.pyr_stride + dc.lvl_off[0], dc.pitch,
                     left_dev + b * pitch * dc.H, pitch, cudaMemcpyDeviceToDevice));
      RET(copy_image(ctx, db.right_raw + b * dc.img_stride, dc.pitch, right_dev + b * pitch * dc.H, pitch,
                     cudaMemcpyDeviceToDevice));
    }
  }
  return enqueue_step(ctx);
}

// H2D of one batch of host images: one 2-D copy per side when the batch is contiguous in host memory
// (image b at left[0] + b*W*H), else one copy per image.
static int upload_batch(kvfe_ctx* ctx, const uint8_t* const* left, const uint8_t* const* right, size_t pitch) {
  const DevCfg& dc = ctx->dc; DevBuf& db = ctx->db;
  const size_t B = dc.B, img = (size_t)dc.W * dc.H;
  bool contig = (pitch == (size_t)dc.W && (size_t)dc.pitch == pitch);
  for (size_t b = 1; b < B && contig; ++b)
    contig = left[b] == left[0] + b * img && right[b] == right[0] + b * img;
  unsigned char* dl = db.pyr[ctx->cur_slot] + dc.lvl_off[0];
  if (contig && B > 1) {
    CU(cudaMemcpy2DAsync(dl, dc.pyr_stride, left[0], img, img, B, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpy2DAsync(db.right_raw, dc.img_stride, right[0], img, img, B, cudaMemcpyHostToDevice, ctx->stream));
    return KVFE_OK;
  }
  for (size_t b = 0; b < B; ++b) {
    RET(copy_image(ctx, dl + b * dc.pyr_stride, dc.pitch, left[b], pitch, cudaMemcpyHostToDevice));
    RET(copy_image(ctx, db.right_raw + b * dc.img_stride, dc.pitch, right[b], pitch, cudaMemcpyHostToDevice));
  }
  return KVFE_OK;
}

// Common tail of a submit (the caller has already enqueued the image copies on ctx->stream): write the
// step inputs into the pinned I/O block of this pyramid slot and launch the host-step graph: the kernel
// sequence reading its inputs straight from that (mapped) block, then publish_kernel storing the
// packets into it.  No copy-engine operation is involved besides the image uploads, and a step
// costs the host one graph launch and one event record.
static int launch_host_step(kvfe_ctx* ctx, const int64_t* timestamps, const double* keyframe_R_cur, uint8_t* packets) {
  const size_t B = ctx->dc.B;
  const int slot = ctx->cur_slot, ps = (int)(ctx->n_submitted & 1);
  unsigned char* io = ctx->h_io[slot];
  memcpy(io, timestamps, B * sizeof(long long));
  memcpy(io + B * sizeof(long long), keyframe_R_cur, B * 9 * sizeof(double));
  const size_t pk_bytes = B * ctx->db.packet_bytes;
  // pinned allocations are mapped into the device address space (unified addressing)
  ctx->in_ts = reinterpret_cast<const long long*>(io);
  ctx->in_R = reinterpret_cast<const double*>(io + B * sizeof(long long));
  int rc = KVFE_OK;
  if (ctx->use_graph) {
    if (!ctx->host_graph_ready[slot]) {
      cudaGraph_t g = nullptr;
      long long n = 0;
      cudaError_t e = cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal);
      if (e == cudaSuccess) {
        rc = enqueue_step_kernels(ctx, &n);
        n += launch_publish(io + ctx->io_pk_off, ctx->db.packets, pk_bytes, ctx->stream);
        e = cudaStreamEndCapture(ctx->stream, &g);
      }
      if (rc == KVFE_OK && e != cudaSuccess) rc = set_err(ctx, KVFE_ERR_CUDA, "host-step graph capture failed: %s", cudaGetErrorString(e));
      if (rc == KVFE_OK && cudaGraphInstantiate(&ctx->host_graph[slot], g, 0) != cudaSuccess) rc = set_err(ctx, KVFE_ERR_CUDA, "host-step graph instantiation failed");
      if (g) cudaGraphDestroy(g);
      if (rc == KVFE_OK) { ctx->host_graph_ready[slot] = 1; ctx->host_graph_launches = n; }
    }
    if (rc == KVFE_OK && cudaGraphLaunch(ctx->host_graph[slot], ctx->stream) != cudaSuccess) rc = set_err(ctx, KVFE_ERR_CUDA, "cudaGraphLaunch failed");
    if (rc == KVFE_OK) ctx->launches += ctx->host_graph_launches;
  } else {
    long long n = 0;
    rc = enqueue_step_kernels(ctx, &n);
    if (rc == KVFE_OK) n += launch_publish(io + ctx->io_pk_off, ctx->db.packets, pk_bytes, ctx->stream);
    ctx->launches += n;
  }
  ctx->in_ts = nullptr; ctx->in_R = nullptr;
  if (rc != KVFE_OK) return rc;
  ctx->cur_slot ^= 1;
  CU(cudaEventRecord(ctx->pipe_done[ps], ctx->stream));
  ctx->pipe_user[ps] = packets; ctx->pipe_io_slot[ps] = slot;
  ++ctx->n_submitted;
  return KVFE_OK;
}

extern "C" int kvfe_frontend_submit(kvfe_ctx* ctx, const uint8_t* const* left, const uint8_t* const* right, size_t pitch,
                                    const int64_t* timestamps, const double* keyframe_R_cur, uint8_t* packets) {
  if (!ctx || !left || !right || !timestamps || !keyframe_R_cur) return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  if (ctx->dc.rgbd) return refuse_rgbd(ctx, "kvfe_frontend_submit");
  if (ctx->n_submitted - ctx->n_waited >= 2) return set_err(ctx, KVFE_ERR_INVALID_ARG, "submit: two steps already in flight, call kvfe_frontend_wait first");
  RET(upload_batch(ctx, left, right, pitch));
  return launch_host_step(ctx, timestamps, keyframe_R_cur, packets);
}

// submit with the images already in device memory (densely packed batch: image b at left_dev +
// b*W*H): an SM copy kernel places them, then the host-step graph runs.  No copy-engine operation at
// all, so contexts never queue behind each other; same pipelining rules as kvfe_frontend_submit.
extern "C" int kvfe_frontend_submit_dev(kvfe_ctx* ctx, const uint8_t* left_dev, const uint8_t* right_dev, size_t pitch,
                                        const int64_t* timestamps, const double* keyframe_R_cur, uint8_t* packets) {
  if (!ctx || !left_dev || !right_dev || !timestamps || !keyframe_R_cur) return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  if (ctx->dc.rgbd) return refuse_rgbd(ctx, "kvfe_frontend_submit_dev");
  if (ctx->n_submitted - ctx->n_waited >= 2) return set_err(ctx, KVFE_ERR_INVALID_ARG, "submit: two steps already in flight, call kvfe_frontend_wait first");
  const DevCfg& dc = ctx->dc; DevBuf& db = ctx->db;
  if (pitch != (size_t)dc.W || dc.pitch != dc.W) return set_err(ctx, KVFE_ERR_INVALID_ARG, "submit_dev: images must be densely packed (pitch == width)");
  ctx->launches += launch_fetch(left_dev, right_dev, db.pyr[ctx->cur_slot] + dc.lvl_off[0], dc.pyr_stride, db.right_raw,
                                dc.img_stride, (size_t)dc.W * dc.H, dc.B, ctx->stream);
  CU(cudaGetLastError());
  return launch_host_step(ctx, timestamps, keyframe_R_cur, packets);
}

// ---- staged uploads: frames of a group of contexts travel in ONE H2D copy per camera ----------------
struct kvfe_upload {
  int n = 0;
  std::vector<kvfe_ctx*> ctx;
  size_t B = 0, img = 0;
  unsigned char* stage[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};   // [ring slot][camera]
  cudaStream_t stream = nullptr;
  cudaEvent_t up_done[2] = {nullptr, nullptr};
  std::vector<cudaEvent_t> taken[2];            // [ring slot][member]: the member's slice copies are done
  std::vector<char> taken_used[2];
  std::vector<unsigned long long> consumed;     // uploads consumed per member
  unsigned long long uploaded = 0;
};

extern "C" void kvfe_upload_destroy(kvfe_upload* u) {
  if (!u) return;
  if (u->stream) cudaStreamSynchronize(u->stream);
  for (kvfe_ctx* c : u->ctx) if (c) cudaStreamSynchronize(c->stream);
  for (int s = 0; s < 2; ++s) {
    for (int k = 0; k < 2; ++k) if (u->stage[s][k]) cudaFree(u->stage[s][k]);
    if (u->up_done[s]) cudaEventDestroy(u->up_done[s]);
    for (cudaEvent_t e : u->taken[s]) if (e) cudaEventDestroy(e);
  }
  if (u->stream) cudaStreamDestroy(u->stream);
  delete u;
}

extern "C" int kvfe_upload_create(kvfe_ctx* const* ctxs, int n, kvfe_upload** out) {
  if (!ctxs || n <= 0 || !out || !ctxs[0]) return KVFE_ERR_INVALID_ARG;
  kvfe_ctx* ctx = ctxs[0];                               // error sink of the CU() macro
  const DevCfg& d0 = ctx->dc;
  if (d0.pitch != d0.W) return set_err(ctx, KVFE_ERR_INVALID_ARG, "upload: the device row pitch must equal the width");
  for (int i = 0; i < n; ++i)
    if (ctxs[i] && ctxs[i]->dc.rgbd) return refuse_rgbd(ctx, "kvfe_upload_create");
  for (int i = 0; i < n; ++i)
    if (!ctxs[i] || ctxs[i]->dc.W != d0.W || ctxs[i]->dc.H != d0.H || ctxs[i]->dc.B != d0.B)
      return set_err(ctx, KVFE_ERR_INVALID_ARG, "upload: contexts must share image size and batch");
  kvfe_upload* u = new kvfe_upload();
  u->n = n; u->ctx.assign(ctxs, ctxs + n); u->B = d0.B; u->img = (size_t)d0.W * d0.H;
  u->consumed.assign(n, 0);
  const size_t bytes = (size_t)n * u->B * u->img;
  cudaError_t e = cudaStreamCreateWithFlags(&u->stream, cudaStreamNonBlocking);
  for (int s = 0; s < 2 && e == cudaSuccess; ++s) {
    for (int k = 0; k < 2 && e == cudaSuccess; ++k) e = cudaMalloc((void**)&u->stage[s][k], bytes);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&u->up_done[s], cudaEventDisableTiming);
    u->taken[s].assign(n, nullptr); u->taken_used[s].assign(n, 0);
    for (int i = 0; i < n && e == cudaSuccess; ++i) e = cudaEventCreateWithFlags(&u->taken[s][i], cudaEventDisableTiming);
  }
  if (e != cudaSuccess) { kvfe_upload_destroy(u); return set_err(ctx, KVFE_ERR_CUDA, "upload_create: %s", cudaGetErrorString(e)); }
  *out = u;
  return KVFE_OK;
}

extern "C" int kvfe_upload_frames(kvfe_upload* u, const uint8_t* left, const uint8_t* right, size_t pitch) {
  if (!u) return KVFE_ERR_INVALID_ARG;
  kvfe_ctx* ctx = u->ctx[0];
  if (!left || !right) return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  if (ctx->dc.rgbd) return refuse_rgbd(ctx, "kvfe_upload_frames");
  if (pitch != (size_t)ctx->dc.W) return set_err(ctx, KVFE_ERR_INVALID_ARG, "upload_frames: images must be densely packed (pitch == width)");
  const unsigned long long seq = u->uploaded;
  const int slot = (int)(seq & 1);
  for (int i = 0; i < u->n; ++i) {
    if (seq >= 2 && u->consumed[i] + 1 < seq)
      return set_err(ctx, KVFE_ERR_INVALID_ARG, "upload_frames: two uploads are already waiting for member %d", i);
    // the ring slot may be overwritten once every member has taken its slice of the upload before last
    if (u->taken_used[slot][i]) CU(cudaStreamWaitEvent(u->stream, u->taken[slot][i], 0));
  }
  const size_t bytes = (size_t)u->n * u->B * u->img;
  CU(cudaMemcpyAsync(u->stage[slot][0], left, bytes, cudaMemcpyHostToDevice, u->stream));
  CU(cudaMemcpyAsync(u->stage[slot][1], right, bytes, cudaMemcpyHostToDevice, u->stream));
  CU(cudaEventRecord(u->up_done[slot], u->stream));
  ++u->uploaded;
  return KVFE_OK;
}

extern "C" int kvfe_frontend_submit_uploaded(kvfe_ctx* ctx, kvfe_upload* u, int member, const int64_t* timestamps,
                                             const double* keyframe_R_cur, uint8_t* packets) {
  if (!ctx || !u || !timestamps || !keyframe_R_cur) return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  if (member < 0 || member >= u->n || u->ctx[member] != ctx) return set_err(ctx, KVFE_ERR_INVALID_ARG, "submit_uploaded: not a member of this upload group");
  if (ctx->dc.rgbd) return refuse_rgbd(ctx, "kvfe_frontend_submit_uploaded");
  if (ctx->n_submitted - ctx->n_waited >= 2) return set_err(ctx, KVFE_ERR_INVALID_ARG, "submit: two steps already in flight, call kvfe_frontend_wait first");
  const unsigned long long seq = u->consumed[member];
  if (seq >= u->uploaded) return set_err(ctx, KVFE_ERR_INVALID_ARG, "submit_uploaded: no uploaded frames left for this member");
  const int slot = (int)(seq & 1);
  const DevCfg& dc = ctx->dc; DevBuf& db = ctx->db;
  const size_t B = u->B, img = u->img, off = (size_t)member * B * img;
  CU(cudaStreamWaitEvent(ctx->stream, u->up_done[slot], 0));
  // slice -> pyramid slot / right buffer with an SM copy kernel: copy-engine operations of different
  // contexts share in-order queues, a kernel does not
  ctx->launches += launch_fetch(u->stage[slot][0] + off, u->stage[slot][1] + off, db.pyr[ctx->cur_slot] + dc.lvl_off[0],
                                dc.pyr_stride, db.right_raw, dc.img_stride, img, (int)B, ctx->stream);
  CU(cudaGetLastError());
  CU(cudaEventRecord(u->taken[slot][member], ctx->stream));
  u->taken_used[slot][member] = 1;
  ++u->consumed[member];
  return launch_host_step(ctx, timestamps, keyframe_R_cur, packets);
}

extern "C" int kvfe_frontend_wait(kvfe_ctx* ctx) {
  if (!ctx) return KVFE_ERR_INVALID_ARG;
  if (ctx->n_waited == ctx->n_submitted) return set_err(ctx, KVFE_ERR_INVALID_ARG, "wait: nothing in flight");
  const int ps = (int)(ctx->n_waited & 1);
  CU(cudaEventSynchronize(ctx->pipe_done[ps]));
  const int slot = ctx->pipe_io_slot[ps];
  if (ctx->pipe_user[ps])
    memcpy(ctx->pipe_user[ps], ctx->h_io[slot] + ctx->io_pk_off, (size_t)ctx->dc.B * ctx->db.packet_bytes);
  ctx->last_io_slot = slot;
  ++ctx->n_waited;
  return KVFE_OK;
}

extern "C" int kvfe_frontend_ready(kvfe_ctx* ctx) {
  if (!ctx) return KVFE_ERR_INVALID_ARG;
  if (ctx->n_waited == ctx->n_submitted) return 0;
  cudaError_t e = cudaEventQuery(ctx->pipe_done[ctx->n_waited & 1]);
  if (e == cudaSuccess) return 1;
  if (e == cudaErrorNotReady) { cudaGetLastError(); return 0; }
  return set_err(ctx, KVFE_ERR_CUDA, "cudaEventQuery failed: %s", cudaGetErrorString(e));
}

extern "C" const uint8_t* kvfe_frontend_packets_view(const kvfe_ctx* ctx) {
  return ctx ? ctx->h_io[ctx->last_io_slot] + ctx->io_pk_off : nullptr;
}

extern "C" int kvfe_frontend_step_multi(kvfe_ctx* const* ctxs, int n, const uint8_t* const* const* left,
                                        const uint8_t* const* const* right, size_t pitch,
                                        const int64_t* const* timestamps, const double* const* keyframe_R_cur,
                                        uint8_t* const* packets) {
  if (!ctxs || n <= 0 || !left || !right || !timestamps || !keyframe_R_cur || !packets) return KVFE_ERR_INVALID_ARG;
  for (int i = 0; i < n; ++i)
    RET(kvfe_frontend_submit(ctxs[i], left[i], right[i], pitch, timestamps[i], keyframe_R_cur[i], packets[i]));
  for (int i = 0; i < n; ++i) RET(kvfe_frontend_wait(ctxs[i]));
  return KVFE_OK;
}

extern "C" int kvfe_frontend_step_dev_multi(kvfe_ctx* const* ctxs, int n, const uint8_t* const* left_dev,
                                            const uint8_t* const* right_dev, size_t pitch,
                                            const int64_t* const* timestamps, const double* const* keyframe_R_cur) {
  if (!ctxs || n <= 0 || !left_dev || !right_dev || !timestamps || !keyframe_R_cur) return KVFE_ERR_INVALID_ARG;
  for (int i = 0; i < n; ++i) {
    int rc = kvfe_frontend_step_dev(ctxs[i], left_dev[i], right_dev[i], pitch, timestamps[i], keyframe_R_cur[i]);
    if (rc != KVFE_OK) return rc;
  }
  return KVFE_OK;
}

extern "C" int kvfe_frontend_step_dev_timed(kvfe_ctx* ctx, const uint8_t* left_dev, const uint8_t* right_dev,
                                            size_t pitch, const int64_t* timestamps, const double* keyframe_R_cur,
                                            float* stage_ms) {
  if (!ctx || !left_dev || !right_dev || !timestamps || !keyframe_R_cur || !stage_ms) return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  if (ctx->dc.mono || ctx->dc.rgbd) return set_err(ctx, KVFE_ERR_INVALID_ARG, "the per-stage timing pass is written for the stereo front-end");
  const DevCfg& dc = ctx->dc; DevBuf& db = ctx->db; cudaStream_t s = ctx->stream;
  const size_t B = dc.B;
  RET(stage_inputs(ctx, timestamps, keyframe_R_cur));
  if (pitch == (size_t)dc.W && dc.pitch == dc.W) {
    // densely packed images: one strided copy per camera for the whole batch (row = one image)
    // (an SM copy kernel, not two copy-engine operations: those share in-order queues across contexts)
    const size_t img = (size_t)dc.W * dc.H;
    ctx->launches += launch_fetch(left_dev, right_dev, db.pyr[ctx->cur_slot] + dc.lvl_off[0], dc.pyr_stride, db.right_raw,
                                  dc.img_stride, img, (int)B, s);
    CU(cudaGetLastError());
  } else {
    for (size_t b = 0; b < B; ++b) {
      RET(copy_image(ctx, db.pyr[ctx->cur_slot] + b * dc.pyr_stride + dc.lvl_off[0], dc.pitch,
                     left_dev + b * pitch * dc.H, pitch, cudaMemcpyDeviceToDevice));
      RET(copy_image(ctx, db.right_raw + b * dc.img_stride, dc.pitch, right_dev + b * pitch * dc.H, pitch,
                     cudaMemcpyDeviceToDevice));
    }
  }
  const int cur = ctx->cur_slot, prev = cur ^ 1;
  const int M_BOOT = 1 << 0, M_KF = 1 << 2, M_LOST = 1 << 3;
  unsigned char* Lcur = db.pyr[cur] + dc.lvl_off[0];
  cudaEvent_t ev[KVFE_N_STAGES + 3];
  for (auto& e : ev) CU(cudaEventCreate(&e));
  long long n = 0;
  CU(cudaEventRecord(ev[0], s));
  n += launch_prep(dc, db, ctx->d_cam, ctx->d_ts, ctx->d_Rin, nullptr, s);
  if (dc.equalize) {
    n += launch_equalize(dc, db.pyr[cur] + dc.lvl_off[0], dc.pyr_stride, dc.B, nullptr, 0, s);
    n += launch_equalize(dc, db.right_raw, dc.img_stride, dc.B, nullptr, 0, s);
  }
  n += launch_pyramid(dc, db.pyr[cur], dc.B, s);
  CU(cudaEventRecord(ev[1], s));
  n += launch_track_pre(dc, db, s);
  CU(cudaEventRecord(ev[9], s));
  n += launch_lk(dc, db, prev, cur, s);
  CU(cudaEventRecord(ev[10], s));
  n += launch_track_post(dc, db, ctx->d_cam, s);
  CU(cudaEventRecord(ev[2], s));
  n += launch_decide(dc, db, 0ull, s);
  n += launch_ransac_mono(dc, db, M_KF, s);
  CU(cudaEventRecord(ev[3], s));
  n += launch_rectify(dc, db.rmap[0], Lcur, dc.pyr_stride, db.rectL, dc.img_stride, dc.B, db.st, M_KF | M_BOOT, s);
  n += launch_rectify(dc, db.rmap[1], db.right_raw, dc.img_stride, db.rectR, dc.img_stride, dc.B, db.st, M_KF | M_BOOT, s);
  CU(cudaEventRecord(ev[4], s));
  n += launch_sparse_stereo(dc, db, ctx->d_cam, M_KF, 0, s);
  n += launch_ransac_stereo(dc, db, M_KF, s);
  CU(cudaEventRecord(ev[5], s));
  n += launch_detect_pre(dc, db, M_BOOT | M_KF | M_LOST, nullptr, s);
  n += launch_gftt(dc, db, Lcur, dc.pyr_stride, ctx->circle_hw, ctx->circle_r, M_BOOT | M_KF | M_LOST, s);
  CU(cudaEventRecord(ev[6], s));
  n += launch_select(dc, db, Lcur, dc.pyr_stride, ctx->d_cam, M_BOOT | M_KF | M_LOST, 1, s);
  CU(cudaEventRecord(ev[7], s));
  n += launch_sparse_stereo(dc, db, ctx->d_cam, M_BOOT | M_KF, 1, s);
  n += launch_finalize(dc, db, s);
  if (dc.mesh_on) n += launch_mesh(dc, db, s);
  CU(cudaEventRecord(ev[8], s));
  CU(cudaGetLastError());
  CU(cudaStreamSynchronize(s));
  for (int i = 0; i < 8; ++i) CU(cudaEventElapsedTime(&stage_ms[i], ev[i], ev[i + 1]));
  CU(cudaEventElapsedTime(&stage_ms[8], ev[9], ev[10]));
  for (auto& e : ev) cudaEventDestroy(e);
  ctx->launches += n;
  ctx->cur_slot ^= 1;
  return KVFE_OK;
}

extern "C" int kvfe_frontend_step(kvfe_ctx* ctx, const uint8_t* const* left, const uint8_t* const* right, size_t pitch,
                                  const int64_t* timestamps, const double* keyframe_R_cur, uint8_t* packets,
                                  uint8_t* const* rect_left, uint8_t* const* rect_right, size_t rect_pitch) {
  if (!ctx || !left || !right || !timestamps || !keyframe_R_cur || !packets) return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  if (ctx->dc.rgbd) return refuse_rgbd(ctx, "kvfe_frontend_step");
  const DevCfg& dc = ctx->dc; DevBuf& db = ctx->db; cudaStream_t s = ctx->stream;
  const size_t B = dc.B;
  if (ctx->n_submitted != ctx->n_waited) return set_err(ctx, KVFE_ERR_INVALID_ARG, "step: submitted steps still in flight");
  RET(stage_inputs(ctx, timestamps, keyframe_R_cur));
  RET(upload_batch(ctx, left, right, pitch));
  RET(enqueue_step(ctx));
  CU(cudaMemcpyAsync(ctx->h_packets, db.packets, B * db.packet_bytes, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  memcpy(packets, ctx->h_packets, B * db.packet_bytes);
  if (rect_left && rect_right) {
    for (size_t b = 0; b < B; ++b) {
      const kvfe_packet_header* h = reinterpret_cast<const kvfe_packet_header*>(ctx->h_packets + b * db.packet_bytes);
      if (!h->is_keyframe || !rect_left[b] || !rect_right[b]) continue;
      CU(cudaMemcpy2DAsync(rect_left[b], rect_pitch, db.rectL + b * dc.img_stride, dc.pitch, dc.W, dc.H, cudaMemcpyDeviceToHost, s));
      CU(cudaMemcpy2DAsync(rect_right[b], rect_pitch, db.rectR + b * dc.img_stride, dc.pitch, dc.W, dc.H, cudaMemcpyDeviceToHost, s));
    }
    CU(cudaStreamSynchronize(s));
  }
  return KVFE_OK;
}

// RGB-D host-buffer step: intensity images to pyramid level 0, depth images to db.depth (every frame: the keyframe decision
// is only known on the device), then the step graph and the packets back
extern "C" int kvfe_frontend_step_rgbd(kvfe_ctx* ctx, const uint8_t* const* img, size_t pitch, const void* const* depth,
                                       size_t depth_pitch_bytes, const int64_t* timestamps, const double* keyframe_R_cur,
                                       uint8_t* packets) {
  if (!ctx || !img || !depth || !timestamps || !keyframe_R_cur || !packets) return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  const DevCfg& dc = ctx->dc; DevBuf& db = ctx->db; cudaStream_t s = ctx->stream;
  if (!dc.rgbd) return set_err(ctx, KVFE_ERR_INVALID_ARG, "kvfe_frontend_step_rgbd: not an RGB-D context (frontend_type 2)");
  if (ctx->n_submitted != ctx->n_waited) return set_err(ctx, KVFE_ERR_INVALID_ARG, "step: submitted steps still in flight");
  if (pitch < (size_t)dc.W) return set_err(ctx, KVFE_ERR_INVALID_ARG, "pitch %zu smaller than the width", pitch);
  if (depth_pitch_bytes < dc.depth_row)
    return set_err(ctx, KVFE_ERR_INVALID_ARG, "depth pitch %zu smaller than a row (%zu bytes)", depth_pitch_bytes, dc.depth_row);
  const size_t B = dc.B;
  for (size_t b = 0; b < B; ++b)
    if (!img[b] || !depth[b]) return set_err(ctx, KVFE_ERR_INVALID_ARG, "null image of stream %zu", b);
  RET(stage_inputs(ctx, timestamps, keyframe_R_cur));
  for (size_t b = 0; b < B; ++b) {
    RET(copy_image(ctx, db.pyr[ctx->cur_slot] + b * dc.pyr_stride + dc.lvl_off[0], dc.pitch, img[b], pitch, cudaMemcpyHostToDevice));
    CU(cudaMemcpy2DAsync(db.depth + b * dc.depth_stride, dc.depth_row, depth[b], depth_pitch_bytes, dc.depth_row, dc.H,
                         cudaMemcpyHostToDevice, s));
  }
  RET(enqueue_step(ctx));
  CU(cudaMemcpyAsync(ctx->h_packets, db.packets, B * db.packet_bytes, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  memcpy(packets, ctx->h_packets, B * db.packet_bytes);
  return KVFE_OK;
}

extern "C" int kvfe_frontend_read_packets(kvfe_ctx* ctx, uint8_t* packets) {
  if (!ctx || !packets) return set_err(ctx, KVFE_ERR_INVALID_ARG, "null argument");
  const size_t bytes = (size_t)ctx->dc.B * ctx->db.packet_bytes;
  CU(cudaMemcpyAsync(ctx->h_packets, ctx->db.packets, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  memcpy(packets, ctx->h_packets, bytes);
  return KVFE_OK;
}

extern "C" int kvfe_frontend_read_rectified(kvfe_ctx* ctx, int stream, uint8_t* rect_left, uint8_t* rect_right, size_t rect_pitch) {
  if (!ctx || !rect_left || !rect_right || stream < 0 || stream >= ctx->dc.B) return set_err(ctx, KVFE_ERR_INVALID_ARG, "bad argument");
  const DevCfg& dc = ctx->dc;
  RET(download_image(ctx, rect_left, rect_pitch, ctx->db.rectL + (size_t)stream * dc.img_stride, dc.pitch));
  RET(download_image(ctx, rect_right, rect_pitch, ctx->db.rectR + (size_t)stream * dc.img_stride, dc.pitch));
  CU(cudaStreamSynchronize(ctx->stream));
  return KVFE_OK;
}

extern "C" int kvfe_debug_lk(kvfe_ctx* ctx, int stream, float* pred_x, float* pred_y, float* next_x, float* next_y,
                             uint8_t* status, int* n) {
  if (!ctx || stream < 0 || stream >= ctx->dc.B || !n) return set_err(ctx, KVFE_ERR_INVALID_ARG, "bad argument");
  const DevCfg& dc = ctx->dc; DevBuf& db = ctx->db;
  CU(cudaStreamSynchronize(ctx->stream));
  StreamState st;
  CU(cudaMemcpy(&st, db.st + stream, sizeof(st), cudaMemcpyDeviceToHost));
  int m = st.n_ref;
  size_t o = (size_t)stream * dc.cap;
  if (m > 0) {
    if (pred_x) CU(cudaMemcpy(pred_x, db.lk_pred_x + o, m * sizeof(float), cudaMemcpyDeviceToHost));
    if (pred_y) CU(cudaMemcpy(pred_y, db.lk_pred_y + o, m * sizeof(float), cudaMemcpyDeviceToHost));
    if (next_x) CU(cudaMemcpy(next_x, db.lk_qx + o, m * sizeof(float), cudaMemcpyDeviceToHost));
    if (next_y) CU(cudaMemcpy(next_y, db.lk_qy + o, m * sizeof(float), cudaMemcpyDeviceToHost));
    if (status) CU(cudaMemcpy(status, db.lk_status + o, m, cudaMemcpyDeviceToHost));
  }
  *n = m;
  return KVFE_OK;
}
