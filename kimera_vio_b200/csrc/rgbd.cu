// rgbd.cu -- row f2 (RGB-D): the two functions that are specific to the RGB-D front-end
// (reference src/frontend/RgbdVisionImuFrontend.cpp:183-209, :313-366):
//   * DepthFrame::getDetectionMask (src/frontend/DepthFrame.cpp:75-98): cv::inRange of the raw depth image against
//     [min_depth, max_depth] / depth_to_meters -> the detection mask FeatureDetector::featureDetection takes;
//   * RgbdFrame::fillStereoFrame (src/frontend/RgbdFrame.cpp:52-115): the "hallucinated" right frame -- per left
//     keypoint the depth at the truncated raw pixel (DepthFrame::getDepthAtPoint, DepthFrame.cpp:39-73), the virtual
//     disparity fx * virtual_baseline / depth, the right rectified keypoint, keypoints_depth_, keypoints_3d_ =
//     versor * depth / versor.z, and RgbdCamera::distortKeypoints (RgbdCamera.cpp:81-85) for right_frame_.keypoints_.
// Each has a stage-level launch (one image / keypoint list, kvfe_depth_detection_mask / kvfe_rgbd_fill_stereo_frame) and
// a batched, mode-gated launch over frame slot k of every stream (the frame-level RGB-D step, api.cu); both run the same
// per-pixel / per-keypoint device functions.  Everything else the RGB-D front-end does per frame (tracking,
// Camera::undistortKeypoints, 2-point / 5-point and 1-point / 3-point outlier rejection on the fake stereo camera,
// detection) is the mono / stereo kernels; PnP (Tracker.cpp:1064-1288) is not built.
// Float arithmetic follows the reference expression by expression (float depth, double fx_b, float disparity).
#include "common.cuh"

// depth_type: 0 = CV_16UC1, 1 = CV_32FC1.  255 when the raw value of pixel x of `row` lies in the range
__device__ __forceinline__ unsigned char depth_in_range(const unsigned char* row, int x, int depth_type, float lo, float hi,
                                                        unsigned int lo16, unsigned int hi16) {
  bool in;
  if (depth_type == 1) {
    const float v = reinterpret_cast<const float*>(row)[x];
    in = (v >= lo) && (v <= hi);                       // NaN fails both, as in cv::inRange
  } else {
    const unsigned int v = reinterpret_cast<const unsigned short*>(row)[x];
    in = (v >= lo16) && (v <= hi16);
  }
  return in ? 255 : 0;
}

__global__ void __launch_bounds__(256) depth_mask_kernel(const unsigned char* __restrict__ depth, size_t pitch_bytes, int depth_type,
                                                         int W, int H, float lo, float hi, unsigned int lo16, unsigned int hi16,
                                                         unsigned char* __restrict__ mask, size_t mask_pitch) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
  if (x >= W) return;
  mask[(size_t)y * mask_pitch + x] = depth_in_range(depth + (size_t)y * pitch_bytes, x, depth_type, lo, hi, lo16, hi16);
}

// grid ((W + 255) / 256, H, B): Frame::detection_mask_ of every stream at a bootstrap / keyframe, into db.mask
__global__ void __launch_bounds__(256) depth_mask_batch_kernel(DevCfg dc, DevBuf db, int mode_mask) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, b = blockIdx.z;
  if (x >= dc.W || !mode_on(db.st[b].mode, mode_mask)) return;
  const unsigned char* row = db.depth + (size_t)b * dc.depth_stride + (size_t)y * dc.depth_row;
  db.mask[(size_t)b * dc.img_stride + (size_t)y * dc.pitch + x] =
      depth_in_range(row, x, dc.depth_type, dc.depth_lo, dc.depth_hi, dc.depth_lo16, dc.depth_hi16);
}

// DepthFrame::getDepthAtPoint: static_cast<int> truncation of the raw keypoint, NaN outside the image or below min_depth
__device__ __forceinline__ float depth_at_point(const unsigned char* depth, size_t pitch_bytes, int depth_type, int W, int H,
                                                float px, float py, float depth_to_meters, float min_depth) {
  const float nan = __int_as_float(0x7fc00000);
  const int x = (int)px, y = (int)py;
  if (x < 0 || x >= W || y < 0 || y >= H) return nan;
  const unsigned char* row = depth + (size_t)y * pitch_bytes;
  float d = (depth_type == 1) ? reinterpret_cast<const float*>(row)[x] : (float)reinterpret_cast<const unsigned short*>(row)[x];
  d *= depth_to_meters;
  if (d < min_depth) return nan;
  return d;
}

struct RgbdFillOut {
  int rs; float rx, ry;                // right_keypoints_rectified_
  double d, X, Y, Z;                   // keypoints_depth_, keypoints_3d_
  float dx, dy;                        // right_frame_.keypoints_
};

// fillStereoFrame + distortKeypoints for one keypoint (raw kx, ky; left rectified status / position; versor v)
__device__ __forceinline__ RgbdFillOut rgbd_fill_point(const DevCfg& dc, const CamModel& cam, const unsigned char* depth,
                                                       size_t pitch_bytes, int depth_type, float depth_to_meters, float min_depth,
                                                       double fx_b, float kx, float ky, int lstat, float lx, float ly,
                                                       const double* v) {
  RgbdFillOut o;
  o.rs = lstat; o.rx = 0.f; o.ry = 0.f;
  o.d = 0.0; o.X = 0.0; o.Y = 0.0; o.Z = 0.0;
  if (o.rs == KVFE_KP_VALID) {
    const float kd = depth_at_point(depth, pitch_bytes, depth_type, dc.W, dc.H, kx, ky, depth_to_meters, min_depth);
    o.rs = KVFE_KP_NO_DEPTH;
    if (isfinite(kd)) {
      const float disparity = (float)(fx_b / (double)kd);
      const float uR = lx - disparity;
      if (!(uR < 0.0f)) {
        o.rs = KVFE_KP_VALID;
        o.rx = uR; o.ry = ly;
        o.d = (double)kd;
        const double vz = v[2];
        o.X = v[0] * o.d / vz; o.Y = v[1] * o.d / vz; o.Z = vz * o.d / vz;
      }
    }
  }
  // RgbdCamera::distortKeypoints -> UndistorterRectifier::distortUnrectifyKeypoints (UndistorterRectifier.cpp:213-228)
  o.dx = 0.f; o.dy = 0.f;
  if (o.rs == KVFE_KP_VALID) {
    const int xx = clampi((int)roundf(o.rx), 0, dc.W - 1), yy = clampi((int)roundf(o.ry), 0, dc.H - 1);
    rect_map_at(cam, xx, yy, &o.dx, &o.dy);
  }
  return o;
}

__global__ void __launch_bounds__(128) rgbd_fill_kernel(DevCfg dc, const CamModel* __restrict__ cams, const unsigned char* __restrict__ depth,
                                                        size_t pitch_bytes, int depth_type, float depth_to_meters, float min_depth,
                                                        double fx_b, const float* __restrict__ kp_x, const float* __restrict__ kp_y,
                                                        const int* __restrict__ left_status, const float* __restrict__ left_x,
                                                        const float* __restrict__ left_y, const double* __restrict__ versors, int n,
                                                        int* __restrict__ right_status, float* __restrict__ right_x,
                                                        float* __restrict__ right_y, double* __restrict__ depth_out,
                                                        double* __restrict__ p3d, float* __restrict__ right_kp_x,
                                                        float* __restrict__ right_kp_y) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const RgbdFillOut o = rgbd_fill_point(dc, cams[0], depth, pitch_bytes, depth_type, depth_to_meters, min_depth, fx_b, kp_x[i], kp_y[i],
                                        left_status[i], left_x[i], left_y[i], versors + 3 * i);
  right_status[i] = o.rs; right_x[i] = o.rx; right_y[i] = o.ry;
  depth_out[i] = o.d;
  p3d[3 * i] = o.X; p3d[3 * i + 1] = o.Y; p3d[3 * i + 2] = o.Z;
  right_kp_x[i] = o.dx; right_kp_y[i] = o.dy;
}

// grid ((cap + 127) / 128, B): every keypoint of frame slot k.  It reads kx/ky, lstat/lrx/lry (Camera::undistortKeypoints,
// left_rect_kernel) and the versors, and rewrites the whole right half -- also the keypoints the stereo RANSAC of this
// keyframe marked FAILED_ARUN, as the reference's second fillStereoFrame over all keypoints does (RgbdVisionImuFrontend.cpp:358)
__global__ void __launch_bounds__(128) rgbd_fill_batch_kernel(DevCfg dc, DevBuf db, const CamModel* __restrict__ cams, int mode_mask) {
  const int b = blockIdx.y;
  const StreamState& s = db.st[b];
  if (!mode_on(s.mode, mode_mask)) return;
  const int fs = b * 3 + s.slot_k;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= db.fr.n[fs]) return;
  const size_t k = (size_t)fs * dc.cap + i;
  const RgbdFillOut o = rgbd_fill_point(dc, cams[0], db.depth + (size_t)b * dc.depth_stride, dc.depth_row, dc.depth_type, dc.depth_to_m,
                                        dc.depth_min, dc.depth_fx_b, db.fr.kx[k], db.fr.ky[k], db.fr.lstat[k], db.fr.lrx[k],
                                        db.fr.lry[k], db.fr.versor + 3 * k);
  db.fr.rstat[k] = o.rs; db.fr.rrx[k] = o.rx; db.fr.rry[k] = o.ry;
  db.fr.depth[k] = o.d;
  db.fr.p3d[3 * k] = o.X; db.fr.p3d[3 * k + 1] = o.Y; db.fr.p3d[3 * k + 2] = o.Z;
  db.fr.rkx[k] = o.dx; db.fr.rky[k] = o.dy;
}

int launch_depth_mask(const DevCfg& dc, const unsigned char* depth, size_t pitch_bytes, int depth_type, float lo, float hi,
                      unsigned int lo16, unsigned int hi16, unsigned char* mask, size_t mask_pitch, cudaStream_t s) {
  dim3 grid((dc.W + 255) / 256, dc.H);
  depth_mask_kernel<<<grid, 256, 0, s>>>(depth, pitch_bytes, depth_type, dc.W, dc.H, lo, hi, lo16, hi16, mask, mask_pitch);
  return 1;
}

int launch_rgbd_fill(const DevCfg& dc, const CamModel* d_cam, const unsigned char* depth, size_t pitch_bytes, int depth_type,
                     float depth_to_meters, float min_depth, double fx_b, const float* kp_x, const float* kp_y, const int* left_status,
                     const float* left_x, const float* left_y, const double* versors, int n, int* right_status, float* right_x,
                     float* right_y, double* depth_out, double* p3d, float* right_kp_x, float* right_kp_y, cudaStream_t s) {
  rgbd_fill_kernel<<<(n + 127) / 128, 128, 0, s>>>(dc, d_cam, depth, pitch_bytes, depth_type, depth_to_meters, min_depth, fx_b, kp_x, kp_y,
                                                    left_status, left_x, left_y, versors, n, right_status, right_x, right_y, depth_out,
                                                    p3d, right_kp_x, right_kp_y);
  return 1;
}

int launch_depth_mask_batch(const DevCfg& dc, const DevBuf& db, int mode_mask, cudaStream_t s) {
  depth_mask_batch_kernel<<<dim3((dc.W + 255) / 256, dc.H, dc.B), 256, 0, s>>>(dc, db, mode_mask);
  return 1;
}

int launch_rgbd_fill_batch(const DevCfg& dc, const DevBuf& db, const CamModel* d_cam, int mode_mask, cudaStream_t s) {
  rgbd_fill_batch_kernel<<<dim3((dc.cap + 127) / 128, dc.B), 128, 0, s>>>(dc, db, d_cam, mode_mask);
  return 1;
}
