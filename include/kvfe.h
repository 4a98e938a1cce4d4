/* kvfe.h -- C-ABI of libkvfe.so: the B200-native stereo visual front-end hot path of Kimera-VIO.
 *
 * Every entry point replaces one method (or a sequence of methods) of the reference's C++ classes;
 * the reference interface each one stands in for is cited as file:line relative to the reference
 * tree.  Only plain pointers, sizes and POD structs cross this boundary (no torch / cv / gtsam
 * types).  All functions return 0 on success and a negative kvfe_status on failure; the reason is
 * available through kvfe_last_error().  Nothing here ever falls back to a CPU implementation: if
 * no CUDA device is usable kvfe_create() fails with KVFE_ERR_NO_DEVICE.
 *
 * Conventions: images are 8-bit, row-major, `pitch` bytes per row, HOST pointers unless the
 * function name ends in `_dev`.  Keypoint arrays are SoA (separate x / y arrays) exactly like the
 * reference's parallel std::vectors (include/kimera-vio/frontend/Frame.h:160-186,
 * StereoFrame.h:141-171).  Rotation matrices and camera matrices are row-major doubles.
 */
#ifndef KVFE_H_
#define KVFE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KVFE_VERSION 3

typedef struct kvfe_ctx kvfe_ctx;

typedef enum {
  KVFE_OK = 0,
  KVFE_ERR_INVALID_ARG = -1,
  KVFE_ERR_NO_DEVICE = -2,
  KVFE_ERR_CUDA = -3,
  KVFE_ERR_CAPACITY = -4,
  KVFE_ERR_STATE = -5
} kvfe_status;

/* KeypointStatus -- include/kimera-vio/common/vio_types.h:38-44 */
typedef enum {
  KVFE_KP_VALID = 0,
  KVFE_KP_NO_LEFT_RECT = 1,
  KVFE_KP_NO_RIGHT_RECT = 2,
  KVFE_KP_NO_DEPTH = 3,
  KVFE_KP_FAILED_ARUN = 4
} kvfe_keypoint_status;

/* TrackingStatus -- include/kimera-vio/frontend/Tracker-definitions.h:124-130 */
typedef enum {
  KVFE_TRK_VALID = 0,
  KVFE_TRK_LOW_DISPARITY = 1,
  KVFE_TRK_FEW_MATCHES = 2,
  KVFE_TRK_INVALID = 3,
  KVFE_TRK_DISABLED = 4
} kvfe_tracking_status;

/* CameraParams::DepthParams (include/kimera-vio/frontend/CameraParams.h:131-155) as parsed by parseDepthParams
 * (src/frontend/CameraParams.cpp:342-349).  The depth image has the context's width x height; it must already be
 * registered to the intensity camera (is_registered: cv::rgbd::registerDepth is not built). */
#define KVFE_DEPTH_U16 0   /* CV_16UC1 */
#define KVFE_DEPTH_F32 1   /* CV_32FC1 */
typedef struct {
  int32_t depth_type;        /* KVFE_DEPTH_U16 / KVFE_DEPTH_F32 */
  float virtual_baseline;    /* virtual_baseline_ (also the baseline of RgbdCamera::getFakeStereoCamera) */
  float depth_to_meters;     /* depth_to_meters_ */
  float min_depth;           /* min_depth_ */
  float max_depth;           /* max_depth_ */
} kvfe_depth_params;

/* Mirrors the YAML keys parsed by TrackerParams (src/frontend/VisionImuTrackerParams.cpp:84-135),
 * FeatureDetectorParams (src/frontend/feature-detector/FeatureDetectorParams.cpp:105-222),
 * StereoMatchingParams (src/frontend/StereoMatchingParams.cpp:80-90) and FrontendParams
 * (src/frontend/VisionImuFrontendParams.cpp:80-112). */
typedef struct {
  /* geometry of the batch */
  int32_t width, height;          /* image size (all streams) */
  int32_t batch;                  /* number of independent camera-stream slots */
  int32_t max_keypoints;          /* capacity of every per-frame keypoint array; 0 = derive */
  /* tracker */
  int32_t klt_win_size, klt_max_iter, klt_max_level;
  double klt_eps;
  int32_t max_feature_track_age;
  int32_t min_nr_mono_inliers, min_nr_stereo_inliers;
  double ransac_threshold_mono, ransac_threshold_stereo;
  int32_t ransac_max_iterations;
  double ransac_probability;
  int32_t ransac_randomize;             /* must be 0: deterministic seed 12345 (Euroc default) */
  int32_t ransac_use_1point_stereo, ransac_use_2point_mono;
  int32_t pose_2d2d_algorithm;          /* 1 = NISTER (only value on the graded path) */
  int32_t optical_flow_predictor_type;  /* 0 static, 1 rotational */
  double disparity_threshold;
  int32_t rnd_libstdcxx;                /* 0: libstdc++ >= 11 (Lemire), 1: libstdc++ < 11 */
  /* detector */
  int32_t max_features_per_frame;
  int32_t enable_subpixel_corner_refinement;
  int32_t subpix_max_iters;
  double subpix_epsilon;
  int32_t subpix_window_size, subpix_zero_zone;
  int32_t enable_non_max_suppression;
  int32_t non_max_suppression_type;     /* 0 TopN, 6 Binning (others: KVFE_ERR_INVALID_ARG) */
  int32_t min_distance;
  int32_t max_nr_keypoints_before_anms;
  int32_t nr_horizontal_bins, nr_vertical_bins;
  uint8_t binning_mask[64];             /* row-major nr_vertical_bins x nr_horizontal_bins, 0/1 */
  double quality_level;
  int32_t block_size;                   /* 3 only */
  int32_t use_harris_detector;          /* 0 only */
  double k;
  int32_t sobel_cpu_tail_start;         /* first column where the reference host's scalar Sobel
                                           tail (non-FMA) applies; -1 = none (SURVEY App. A.2) */
  /* stereo matching */
  double tolerance_template_matching;
  int32_t templ_cols, templ_rows, stripe_extra_rows;
  double min_point_dist, max_point_dist;
  int32_t subpixel_refinement_stereo;
  /* front-end FSM */
  int64_t min_intra_keyframe_time_ns, max_intra_keyframe_time_ns;
  int32_t min_number_features;
  int32_t use_stereo_tracking, use_ransac;
  double max_disparity_since_lkf;
  /* Mesher (next row downstream of the packet): Mesher::createMesh2dStereo + createMesh2dImpl
   * (src/mesh/Mesher.cpp:1849-1886, :1712-1817) on every keyframe -- cv::Subdiv2D Delaunay triangulation of the
   * keypoints with a VALID right match and a live landmark; the triangle list joins the packet. */
  int32_t mesh_2d;                      /* 0 off (default), 1 on */
  float subdiv_bounding_factor;         /* cv::Subdiv2D::initDelaunay: outer triangle at factor * max(w, h);
                                           0 = 6 (OpenCV 4.13, this repo's oracle); OpenCV <= 4.5 used 3 */
  /* keys the reference parses that change the results when set: carried so that they are REJECTED or honoured,
   * never silently ignored */
  int32_t optimize_2d2d_pose_from_inliers;  /* VisionImuTrackerParams.cpp:119-122: nonlinear refinement of the RANSAC */
  int32_t optimize_3d3d_pose_from_inliers;  /* pose (opengv optimize_nonlinear); must be 0: KVFE_ERR_INVALID_ARG otherwise */
  int32_t frontend_type;                /* 0: StereoVisionImuFrontend (default); 1: MonoVisionImuFrontend
                                           (src/frontend/MonoVisionImuFrontend.cpp:194-371) -- the same kernels without the
                                           stereo half: no rectification, stereo matching or stereo RANSAC; statuses reset on
                                           every frame (mono INVALID, stereo DISABLED); the keyframe's keypoints_undistorted_
                                           (Camera::undistortKeypoints, P = K, R = I) travel in left_status / left_rect_*.
                                           The rig is kvfe_rig with R1 = I, P1 = [K | 0]; right images are ignored.
                                           2: RgbdVisionImuFrontend (src/frontend/RgbdVisionImuFrontend.cpp:183-395) -- the
                                           mono front-end plus a registered depth image per frame: detection masked by the
                                           depth range, RgbdFrame::fillStereoFrame (the "hallucinated" right keypoints,
                                           depth, 3-D points) and stereo RANSAC on the fake stereo camera; statuses reset
                                           to INVALID (mono and stereo) on every frame, no "all tracks lost" shortcut.  The
                                           rig is kvfe_rig with R1 = I, P1 = [K | 0], baseline = depth.virtual_baseline,
                                           radial-tangential only; frames go through kvfe_frontend_step_rgbd /
                                           kvfe_pipeline_push_rgbd, and mesh_2d must be 0 */
  int32_t equalize_image;               /* StereoMatchingParams.cpp:80-90 "equalizeImage": cv::equalizeHist on both raw
                                           images (UtilsOpenCV::ReadAndConvertToGrayScale, UtilsOpenCV.cpp:390-403),
                                           done on the device as the first kernels of a step (RGB-D: the intensity image
                                           only, never the depth) */
  kvfe_depth_params depth;              /* frontend_type 2 only (ignored otherwise): the camera's depth block */
} kvfe_config;

/* Stereo rig after cv::stereoRectify -- what StereoCamera::StereoCamera hands to its two
 * UndistorterRectifiers (src/frontend/StereoCamera.cpp:34-94,
 * src/frontend/UndistorterRectifier.cpp:26-31, :230-292). Pinhole cameras with the radial-tangential or the
 * equidistant (cv::fisheye) distortion model (CameraParams.cpp:125-140); the omni model is not supported. */
#define KVFE_DISTORTION_RADTAN 0        /* cv::stereoRectify / initUndistortRectifyMap / undistortPoints */
#define KVFE_DISTORTION_EQUIDISTANT 1   /* cv::fisheye::stereoRectify / initUndistortRectifyMap / undistortPoints
                                           (StereoCamera.cpp:350-373, UndistorterRectifier.cpp:49-56, :260-268) */
typedef struct {
  double K_left[9], K_right[9];
  double D_left[4], D_right[4];   /* radtan: k1 k2 p1 p2; equidistant: k1 k2 k3 k4 */
  double R1[9], R2[9];
  double P1[12], P2[12];
  double baseline;                /* 1 / Q(3,2), StereoCamera.cpp:70-72 */
  int32_t distortion_model;       /* KVFE_DISTORTION_*; both cameras share it (StereoCamera.cpp:328 switches on the left one) */
  int32_t reserved;               /* 0 */
} kvfe_rig;

/* Fills every field with the reference's struct defaults / the Euroc YAML. */
void kvfe_config_default(kvfe_config* cfg);

int kvfe_create(const kvfe_config* cfg, const kvfe_rig* rig, kvfe_ctx** out);
void kvfe_destroy(kvfe_ctx* ctx);
const char* kvfe_last_error(const kvfe_ctx* ctx);   /* ctx may be NULL: last create() error */
int kvfe_max_keypoints(const kvfe_ctx* ctx);
int kvfe_kernel_launches(const kvfe_ctx* ctx);       /* kernels launched by this ctx so far */

/* ---------------------------------------------------------------------------------------------
 * Stage-level entry points (one camera stream; host buffers; synchronous).
 * ------------------------------------------------------------------------------------------- */

/* UndistorterRectifier::undistortRectifyImage x2 == StereoCamera::undistortRectifyStereoFrame
 * (src/frontend/UndistorterRectifier.cpp:115-128, src/frontend/StereoCamera.cpp:269-290).
 * cv::remap INTER_LINEAR / BORDER_REPLICATE with the float maps recomputed in registers. */
int kvfe_rectify_pair(kvfe_ctx* ctx, const uint8_t* left, const uint8_t* right, size_t pitch,
                      uint8_t* left_rect, uint8_t* right_rect, size_t out_pitch);

/* The CV_32FC1 maps of UndistorterRectifier::initUndistortRectifyMaps (UndistorterRectifier.cpp:
 * 230-292) for camera `cam` (0 left, 1 right), written densely (width floats per row). */
int kvfe_rectify_maps(kvfe_ctx* ctx, int cam, float* map_x, float* map_y);

/* cv::buildOpticalFlowPyramid as used inside cv::calcOpticalFlowPyrLK (Tracker.cpp:137-146):
 * returns levels 1..klt_max_level densely packed one after the other (diagnostics / tests). */
int kvfe_pyramid(kvfe_ctx* ctx, const uint8_t* img, size_t pitch, uint8_t* levels_out,
                 size_t levels_out_bytes, int* n_levels);

/* cv::cornerMinEigenVal(img, blockSize 3, ksize 3) -- the response map inside
 * cv::goodFeaturesToTrack (FeatureDetector.cpp:165-172); diagnostics / tests. */
int kvfe_min_eigen_response(kvfe_ctx* ctx, const uint8_t* img, size_t pitch, float* response);

/* FeatureDetector::featureDetection(const Frame&, int need_n_corners)
 * (src/frontend/feature-detector/FeatureDetector.cpp:174-299): mask of tracked keypoints,
 * GFTT, non-max suppression (NonMaximumSuppression.cpp:33-169), cv::cornerSubPix.
 * existing_*: the frame's current keypoints_ / landmarks_ (landmark -1 = not masked). */
int kvfe_detect(kvfe_ctx* ctx, const uint8_t* img, size_t pitch, const float* existing_x,
                const float* existing_y, const int64_t* existing_lmk, int n_existing, int need,
                float* out_x, float* out_y, int* n_out);
/* Same with a caller-supplied Frame::detection_mask_ (FeatureDetector.cpp:186-189; the RGB-D front-end fills it):
 * 255 = consider, 0 = do not; the circles around the tracked keypoints are drawn into it like the reference does. */
int kvfe_detect_masked(kvfe_ctx* ctx, const uint8_t* img, size_t pitch, const uint8_t* detection_mask, size_t mask_pitch,
                       const float* existing_x, const float* existing_y, const int64_t* existing_lmk, int n_existing,
                       int need, float* out_x, float* out_y, int* n_out);
/* Same, but stops after cv::GFTTDetector::detect (FeatureDetector::rawFeatureDetection,
 * FeatureDetector.cpp:165-172): corners in descending-response order. */
int kvfe_detect_raw(kvfe_ctx* ctx, const uint8_t* img, size_t pitch, const float* existing_x,
                    const float* existing_y, const int64_t* existing_lmk, int n_existing,
                    float* out_x, float* out_y, float* out_response, int* n_out);

/* The optical-flow half of Tracker::featureTracking (src/frontend/Tracker.cpp:117-148):
 * RotationalOpticalFlowPredictor::predictSparseFlow (optical-flow/OpticalFlowPredictor.cpp:70-126)
 * followed by cv::calcOpticalFlowPyrLK with OPTFLOW_USE_INITIAL_FLOW.  ref_R_cur row-major 3x3. */
int kvfe_track(kvfe_ctx* ctx, const uint8_t* ref_img, const uint8_t* cur_img, size_t pitch,
               const double* ref_R_cur, const float* ref_x, const float* ref_y, int n,
               float* pred_x, float* pred_y, float* cur_x, float* cur_y, uint8_t* status);

/* UndistorterRectifier::UndistortRectifyKeypoints (UndistorterRectifier.cpp:33-68).
 * cam: 0 left, 1 right; use_R / use_P select R1|R2 and P1|P2 or identity. */
int kvfe_undistort_keypoints(kvfe_ctx* ctx, int cam, int use_R, int use_P, const float* x,
                             const float* y, int n, float* out_x, float* out_y);
/* UndistorterRectifier::GetBearingVector (UndistorterRectifier.cpp:73-113), left camera, R = R1. */
int kvfe_bearing_vectors(kvfe_ctx* ctx, const float* x, const float* y, int n, double* versors);

/* StereoMatcher::sparseStereoReconstruction(StereoFrame*) (src/frontend/StereoMatcher.cpp:123-175):
 * rectify both images, StereoCamera::undistortRectifyLeftKeypoints (StereoCamera.cpp:236-260),
 * getRightKeypointsRectified (:196-281), getDepthFromRectifiedMatches (:425-483),
 * distortUnrectifyRightKeypoints (StereoCamera.cpp:262-267), keypoints_3d (:157-174). */
typedef struct {
  int32_t* left_status;  float* left_rect_x;  float* left_rect_y;
  int32_t* right_status; float* right_rect_x; float* right_rect_y;
  double* depth;         /* n   */
  double* points_3d;     /* n*3 */
  float* right_x;  float* right_y;   /* right_frame_.keypoints_ */
} kvfe_stereo_out;
int kvfe_sparse_stereo(kvfe_ctx* ctx, const uint8_t* left, const uint8_t* right, size_t pitch,
                       const float* kp_x, const float* kp_y, const double* versors, int n,
                       kvfe_stereo_out* out, uint8_t* left_rect, uint8_t* right_rect,
                       size_t rect_pitch);

/* ---- the remaining public methods of the replaced classes, one call each (stage level) ------------------------- */
/* UndistorterRectifier::checkUndistortedRectifiedLeftKeypoints (include/kimera-vio/frontend/UndistorterRectifier.h:106,
 * src/frontend/UndistorterRectifier.cpp:138-211): crop the undistorted-rectified keypoint to the image, look the
 * rectification maps up at its rounded position and compare with the distorted keypoint; status VALID or NO_LEFT_RECT,
 * out = the cropped rectified keypoint.  cam: 0 left maps, 1 right maps.  The reference's default tolerance is 2.0. */
int kvfe_check_rectified_keypoints(kvfe_ctx* ctx, int cam, const float* distorted_x, const float* distorted_y,
                                   const float* rectified_x, const float* rectified_y, int n, float pixel_tolerance,
                                   int32_t* status, float* out_x, float* out_y);
/* UndistorterRectifier::distortUnrectifyKeypoints (UndistorterRectifier.h:113, .cpp:213-228) /
 * StereoCamera::distortUnrectifyRightKeypoints (StereoCamera.cpp:262-267, cam = 1): maps at the rounded rectified
 * position for VALID keypoints, (0, 0) otherwise. */
int kvfe_distort_unrectify_keypoints(kvfe_ctx* ctx, int cam, const int32_t* status, const float* x, const float* y,
                                     int n, float* out_x, float* out_y);
/* StereoCamera::undistortRectifyLeftKeypoints (StereoCamera.cpp:236-260): cv::undistortPoints(K, D, R1, P1) followed
 * by the check above with the default tolerance. */
int kvfe_undistort_rectify_left_keypoints(kvfe_ctx* ctx, const float* x, const float* y, int n, int32_t* status,
                                          float* rect_x, float* rect_y);
/* StereoMatcher::getRightKeypointsRectified (include/kimera-vio/frontend/StereoMatcher.h:81, .cpp:196-281): the
 * epipolar template search of every VALID rectified left keypoint on an already rectified image pair. */
int kvfe_right_keypoints_rectified(kvfe_ctx* ctx, const uint8_t* left_rectified, const uint8_t* right_rectified, size_t pitch,
                                   const int32_t* left_status, const float* left_x, const float* left_y, int n,
                                   int32_t* right_status, float* right_x, float* right_y);
/* StereoMatcher::getDepthFromRectifiedMatches (StereoMatcher.h:89, .cpp:425-483): depth = fx * baseline / disparity
 * inside [minPointDist, maxPointDist]; right_status is updated in place (NO_DEPTH, or the left status). */
int kvfe_depth_from_rectified_matches(kvfe_ctx* ctx, const int32_t* left_status, const float* left_x, int32_t* right_status,
                                      const float* right_x, int n, double* depth);
/* Tracker::computeMedianDisparity (include/kimera-vio/frontend/Tracker.h:215, .cpp:991-1018): *ok = 0 and nothing
 * computed when there is no match. */
int kvfe_compute_median_disparity(kvfe_ctx* ctx, const float* ref_x, const float* ref_y, int n_ref, const float* cur_x,
                                  const float* cur_y, int n_cur, const int32_t* match_ref, const int32_t* match_cur,
                                  int n_matches, double* median, int* ok);
/* Tracker::getPoint3AndCovariance (Tracker.h:221, .cpp:772-818) for n rectified stereo points at once, with
 * stereo_point_covariance = identity (what its caller passes, Tracker.cpp:560-563): out_points = R * p (p when R is
 * NULL), out_cov = (R J)(R J)^T with J the Jacobian of gtsam::StereoCamera::backproject2 at (uL, uR, v). */
int kvfe_point3_and_covariance(kvfe_ctx* ctx, const float* left_x, const float* right_x, const float* left_y,
                               const double* points_3d, int n, const double* R, double* out_points, double* out_cov);
/* Tracker::findOutliers / removeOutliersMono / removeOutliersStereo (Tracker.h:150-172, .cpp:836-917): pure
 * bookkeeping on the caller's vectors (host logic, no device work -- the frame-level path does the same on the GPU). */
int kvfe_find_outliers(int n_matches, const int32_t* inliers, int n_inliers, int32_t* outliers, int* n_outliers);
int kvfe_remove_outliers_mono(const int32_t* inliers, int n_inliers, int64_t* ref_landmarks, int n_ref, int64_t* cur_landmarks,
                              int n_cur, int32_t* match_ref, int32_t* match_cur, int* n_matches);
int kvfe_remove_outliers_stereo(const int32_t* inliers, int n_inliers, int32_t* ref_right_status, double* ref_depth,
                                double* ref_points_3d, int n_ref, int32_t* cur_right_status, double* cur_depth,
                                double* cur_points_3d, int n_cur, int32_t* match_ref, int32_t* match_cur, int* n_matches);

/* Tracker::findMatchingKeypoints (include/kimera-vio/frontend/Tracker.h:195, src/frontend/Tracker.cpp:919-946): pairs
 * (ref index, cur index) observing the same landmark, in current-frame order.  Host bookkeeping (no ctx), like the
 * reference's; match arrays sized n_cur. */
int kvfe_find_matching_keypoints(const int64_t* ref_landmarks, int n_ref, const int64_t* cur_landmarks, int n_cur,
                                 int32_t* match_ref, int32_t* match_cur, int* n_matches);
/* Tracker::findMatchingStereoKeypoints (Tracker.h:199-208, Tracker.cpp:948-989): the mono matches with a VALID right
 * keypoint in both frames. */
int kvfe_find_matching_stereo_keypoints(const int32_t* ref_right_status, int n_ref, const int32_t* cur_right_status, int n_cur,
                                        const int32_t* mono_match_ref, const int32_t* mono_match_cur, int n_mono,
                                        int32_t* match_ref, int32_t* match_cur, int* n_matches);
/* StereoVisionImuFrontend::getSmartStereoMeasurements (src/frontend/StereoVisionImuFrontend.cpp:485-531; use_right =
 * use_stereo_tracking_) / RgbdVisionImuFrontend::fillSmartStereoMeasurements (src/frontend/RgbdVisionImuFrontend.cpp:
 * 368-395; use_right = 1): (landmark, uL, uR, v) per keypoint with a landmark; uR = NaN without a VALID right keypoint.
 * Output arrays sized n.  (The frame-level step assembles the same list in the packet: smart_* arrays.) */
int kvfe_smart_stereo_measurements(const int64_t* landmarks, const float* left_x, const float* left_y,
                                   const int32_t* right_status, const float* right_x, int n, int use_right,
                                   int64_t* out_landmarks, double* out_uL, double* out_uR, double* out_v, int* n_out);

/* VisionImuFrontend::shouldBeKeyframe (src/frontend/VisionImuFrontend.cpp:175-232) for a front-end composed at the stage
 * level (mono / RGB-D): thresholds from cfg, median_disparity from kvfe_compute_median_disparity over
 * kvfe_find_matching_keypoints(lkf, frame) (0.0 without matches), mono_status = kfTrackingStatus_mono_ (KVFE_TRK_*),
 * user_keyframe = Frame::isKeyframe_.  Host logic. */
int kvfe_should_be_keyframe(const kvfe_config* cfg, int64_t timestamp_ns, int64_t lkf_timestamp_ns, int nr_valid_features,
                            double median_disparity, int mono_status, int user_keyframe, int* is_keyframe);

/* cv::equalizeHist as UtilsOpenCV::ReadAndConvertToGrayScale applies it (src/utils/UtilsOpenCV.cpp:390-403), one image. */
int kvfe_equalize_hist(kvfe_ctx* ctx, const uint8_t* img, size_t pitch, uint8_t* out, size_t out_pitch);

/* ---- RGB-D (row f2, stage level): the two functions RgbdVisionImuFrontend adds to the mono / stereo ones ----------
 * (kvfe_depth_params is defined above kvfe_config.) */
/* DepthFrame::getDetectionMask (src/frontend/DepthFrame.cpp:75-98): cv::inRange(depth, min_depth / depth_to_meters,
 * max_depth / depth_to_meters) -> 255 / 0 (CV_16UC1: the bounds truncated to uint16, clamped to [0, 65535]); the mask
 * kvfe_detect_masked takes (RgbdVisionImuFrontend.cpp:196-198, :354-356).  pitch in BYTES. */
int kvfe_depth_detection_mask(kvfe_ctx* ctx, const void* depth, size_t depth_pitch_bytes, const kvfe_depth_params* dp,
                              uint8_t* mask, size_t mask_pitch);
/* RgbdFrame::fillStereoFrame (src/frontend/RgbdFrame.cpp:52-115) for the n keypoints of a frame:
 *   kp_x/kp_y         left_frame_.keypoints_ (raw pixels; DepthFrame::getDepthAtPoint truncates them, DepthFrame.cpp:39-73)
 *   left_status/x/y   left_keypoints_rectified_ (Camera::undistortKeypoints == kvfe_undistort_rectify_left_keypoints
 *                     on a mono rig)
 *   versors           left_frame_.versors_ (3 doubles each)
 * out: right_keypoints_rectified_ (status: the left status when it is not VALID, NO_DEPTH for a non-finite depth, a depth
 * below min_depth or uR < 0), keypoints_depth_, keypoints_3d_ (versor * depth / versor.z) and right_frame_.keypoints_
 * (RgbdCamera::distortKeypoints, RgbdCamera.cpp:81-85).  fx is K_left's. */
int kvfe_rgbd_fill_stereo_frame(kvfe_ctx* ctx, const void* depth, size_t depth_pitch_bytes, const kvfe_depth_params* dp,
                                const float* kp_x, const float* kp_y, const int32_t* left_status, const float* left_x,
                                const float* left_y, const double* versors, int n, int32_t* right_status, float* right_x,
                                float* right_y, double* keypoints_depth, double* keypoints_3d, float* right_kp_x,
                                float* right_kp_y);

/* Mesher::createMesh2dImpl (src/mesh/Mesher.cpp:1712-1817): cv::Subdiv2D(rect(0, 0, width, height)), insert the
 * keypoints that lie inside the image, getTriangleList, keep the triangles with all vertices inside.  triangles:
 * 6 floats each (x0 y0 x1 y1 x2 y2) in cv::Subdiv2D's order; n_triangles may exceed max_triangles (then only the
 * first max_triangles were written).  One mesh is inherently sequential (incremental insertion); the frame-level
 * path builds the meshes of all streams of a batch concurrently (cfg.mesh_2d). */
int kvfe_mesh_2d(kvfe_ctx* ctx, const float* kp_x, const float* kp_y, int n, float* triangles, int max_triangles,
                 int* n_triangles);

/* Tracker::geometricOutlierRejection2d2d (src/frontend/Tracker.cpp:213-319) on matched bearing
 * pairs: 2-point (TranslationOnlySacProblem, R12 given) or 5-point Nister (R12 == NULL).
 * inliers: ascending match indices; pose: row-major 3x4 [R|t]; status: kvfe_tracking_status. */
int kvfe_ransac_mono(kvfe_ctx* ctx, const double* f_ref, const double* f_cur, int n,
                     const double* R12, int32_t* inliers, int* n_inliers, double* pose,
                     int* status);
/* Tracker::geometricOutlierRejection3d3dGivenRotation (Tracker.cpp:382-632): 1-point voting. */
int kvfe_ransac_stereo_1pt(kvfe_ctx* ctx, const float* ref_left_xy, const float* ref_right_xy,
                           const float* cur_left_xy, const float* cur_right_xy,
                           const double* ref_3d, const double* cur_3d, int n, const double* R,
                           int32_t* inliers, int* n_inliers, double* pose, double* info,
                           int* status);
/* Tracker::geometricOutlierRejection3d3d (Tracker.cpp:667-742): 3-point Arun. */
int kvfe_ransac_stereo_3pt(kvfe_ctx* ctx, const double* ref_3d, const double* cur_3d, int n,
                           int32_t* inliers, int* n_inliers, double* pose, int* status);

/* ---------------------------------------------------------------------------------------------
 * Frame-level entry points: the whole hot path for `batch` independent streams per call, with
 * the per-stream front-end state (previous pyramid, km1 / lkf keypoint SoA, landmark-id counter)
 * resident in HBM.  One call == VisionImuFrontend::spinOnce for every stream
 * (src/frontend/VisionImuFrontend.cpp:50-64 -> StereoVisionImuFrontend.cpp:67-100 / :283-481).
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  int32_t n;                 /* keypoints in the output StereoFrame */
  int32_t is_keyframe;
  int32_t mono_status, stereo_status;      /* TrackerStatusSummary (kvfe_tracking_status) */
  int32_t n_smart;           /* smart stereo measurements (keyframes only) */
  int32_t nr_tracked;        /* DebugTrackerInfo::nrTrackerFeatures_ */
  int32_t nr_mono_putatives, nr_mono_inliers, nr_stereo_putatives, nr_stereo_inliers;
  int32_t nr_valid_rkp, nr_no_left_rect_rkp, nr_no_right_rect_rkp, nr_no_depth_rkp,
      nr_failed_arun_rkp;    /* StereoFrame::checkStatusRightKeypoints (StereoFrame.cpp:106-143) */
  int32_t mode;              /* 0 bootstrap, 1 nominal non-keyframe, 2 keyframe, 3 all tracks lost */
  int64_t frame_id, timestamp;
  double lkf_T_k_mono[12], lkf_T_k_stereo[12], info_stereo[9];
  double median_disparity;
  int32_t n_mesh_triangles;  /* cfg.mesh_2d: triangles of the keyframe's 2-D mesh (0 otherwise) */
  int32_t reserved;
} kvfe_packet_header;

/* Byte layout of one stream's packet in the flat output buffer (cap = kvfe_max_keypoints()):
 * header, then arrays in this order (each `cap` entries):
 *   kp_x f32, kp_y f32, landmark i64, age i32, score f64 (always 0), versor f64 x3,
 *   left_status i32, left_rect_x f32, left_rect_y f32, right_status i32, right_rect_x f32,
 *   right_rect_y f32, depth f64, point3d f64 x3, right_x f32, right_y f32,
 *   smart_lmk i64, smart_uL f64, smart_uR f64, smart_v f64,
 *   mesh_tri f32 x6 (x0 y0 x1 y1 x2 y2 per triangle, 2*cap triangles; empty unless cfg.mesh_2d).
 * kvfe_packet_bytes() gives the stride; kvfe_packet_offsets() the KVFE_PACKET_ARRAYS offsets in that order. */
#define KVFE_PACKET_ARRAYS 21
size_t kvfe_packet_bytes(const kvfe_ctx* ctx);
int kvfe_packet_offsets(const kvfe_ctx* ctx, size_t* offsets, int max_entries);

int kvfe_frontend_reset(kvfe_ctx* ctx);
/* Multi-GPU (SURVEY 8(e), the optional gather of the keypoint packets to rank 0): the frame-level steps assemble their
 * packets directly in `packets_dev` -- batch * kvfe_packet_bytes() bytes of caller-owned DEVICE memory, typically the
 * send buffer of an NCCL gather -- so the collective needs no pack or copy kernel.  NULL restores the internal buffer. */
int kvfe_frontend_bind_packets(kvfe_ctx* ctx, uint8_t* packets_dev);
/* Frame::isKeyframe_ (include/kimera-vio/frontend/Frame.h:172): flags[b] != 0 makes the NEXT step's frame of stream b a
 * keyframe whatever the other criteria say (VisionImuFrontend::shouldBeKeyframe, VisionImuFrontend.cpp:207-209). */
int kvfe_frontend_force_keyframe(kvfe_ctx* ctx, const int32_t* flags /* batch */);

/* Host-buffer step: copies the batch's images H2D, runs the step, copies the packets (and, when
 * rect_left/right are non-NULL, the rectified images of keyframes) D2H.  left/right: `batch`
 * pointers; timestamps: batch; keyframe_R_cur: batch x 9 (camLrectLkf_R_camLrectK from the IMU,
 * StereoVisionImuFrontend.cpp:149-150); packets: batch * kvfe_packet_bytes(). */
int kvfe_frontend_step(kvfe_ctx* ctx, const uint8_t* const* left, const uint8_t* const* right,
                       size_t pitch, const int64_t* timestamps, const double* keyframe_R_cur,
                       uint8_t* packets, uint8_t* const* rect_left, uint8_t* const* rect_right,
                       size_t rect_pitch);

/* Host-buffer step of an RGB-D context (frontend_type 2): VisionImuFrontend::spinOnce of RgbdVisionImuFrontend for every
 * stream (bootstrapSpin / nominalSpin, RgbdVisionImuFrontend.cpp:183-298).  img: `batch` intensity images (`pitch`
 * bytes per row); depth: `batch` registered depth images of cfg.depth.depth_type (`depth_pitch_bytes` per row);
 * timestamps, keyframe_R_cur and packets as in kvfe_frontend_step.  Synchronous.  The packet of a keyframe carries
 *   left_status / left_rect_*    left_keypoints_rectified_ (Camera::undistortKeypoints, P = K, R = I)
 *   right_status / right_rect_*  right_keypoints_rectified_ (RgbdFrame::fillStereoFrame)
 *   depth, point3d               keypoints_depth_, keypoints_3d_
 *   right_x / right_y            right_frame_.keypoints_ (RgbdCamera::distortKeypoints)
 *   nr_*_rkp                     checkStatusRightKeypoints of right_keypoints_rectified_
 *   smart_*                      fillSmartStereoMeasurements (:370-399): uR whenever the right keypoint is VALID,
 *                                whatever use_stereo_tracking says;
 * a non-keyframe packet follows the convention of the other front-ends: status fields -1, coordinates, depth and points 0.
 * The stereo / mono entry points (kvfe_frontend_step*, _submit*, kvfe_upload_*, kvfe_pipeline_push[_many]) refuse an
 * RGB-D context with KVFE_ERR_INVALID_ARG, and the RGB-D ones refuse the other front-ends. */
int kvfe_frontend_step_rgbd(kvfe_ctx* ctx, const uint8_t* const* img, size_t pitch, const void* const* depth,
                            size_t depth_pitch_bytes, const int64_t* timestamps, const double* keyframe_R_cur,
                            uint8_t* packets);

/* Device-resident step: images already in HBM (batch-major, `pitch` bytes per row, one image
 * after the other); packets stay in HBM until kvfe_frontend_read_packets. Asynchronous on the
 * context's stream; kvfe_sync() waits. */
int kvfe_frontend_step_dev(kvfe_ctx* ctx, const uint8_t* left_dev, const uint8_t* right_dev,
                           size_t pitch, const int64_t* timestamps, const double* keyframe_R_cur);
/* Same as kvfe_frontend_step_dev but synchronous, without the CUDA graph, with CUDA events around
 * the stages; stage_ms receives KVFE_N_STAGES durations in milliseconds (measurement aid for
 * bench.py's roofline line): 0 prep+pyramid, 1 LK tracking (track_pre, lk, track_post), 2 decide +
 * mono RANSAC, 3 rectification, 4 sparse stereo #1 + stereo RANSAC, 5 GFTT (mask, response,
 * selection), 6 NMS + sub-pixel + append, 7 sparse stereo #2 + finalize, 8 the LK kernel alone. */
#define KVFE_N_STAGES 9
int kvfe_frontend_step_dev_timed(kvfe_ctx* ctx, const uint8_t* left_dev, const uint8_t* right_dev,
                                 size_t pitch, const int64_t* timestamps, const double* keyframe_R_cur,
                                 float* stage_ms);
/* Pipelined host-buffer step (the asynchronous input/output queues of the reference's
 * PipelineModule around the frontend, pipeline/PipelineModule.h:190-215 spin(), :359-416
 * SIMOPipelineModule input queue): submit enqueues the H2D
 * copies, the step and the packet D2H copy and returns; wait blocks until the oldest submitted step
 * is done and `packets` (given at submit; owned by the library until wait returns) is filled.  At
 * most two steps may be in flight per context.  The step inputs, the kernel sequence and the
 * packet D2H copy are one CUDA graph over a pinned I/O block owned by the context, so a step costs
 * the host the image copies, one graph launch and one event record.  `packets` may be NULL: the
 * packets of the last waited step are then read in place through kvfe_frontend_packets_view()
 * (valid until the second next submit on this context).  With several contexts one or a few
 * dispatcher threads keep the host link and the GPU busy: wait(k-1) then submit(k), round-robin. */
int kvfe_frontend_submit(kvfe_ctx* ctx, const uint8_t* const* left, const uint8_t* const* right,
                         size_t pitch, const int64_t* timestamps, const double* keyframe_R_cur,
                         uint8_t* packets);
int kvfe_frontend_wait(kvfe_ctx* ctx);
/* 1 when the oldest submitted step is complete (kvfe_frontend_wait will not block), 0 when it is still
 * running or nothing is in flight, < 0 on error.  Streams are independent and a keyframe step takes
 * about three times as long as a tracking step, so a dispatcher that serves contexts in COMPLETION order
 * (poll, collect, resubmit) keeps all of them busy; serving them in a fixed order makes every context
 * advance at the pace of the slowest one of each round. */
int kvfe_frontend_ready(kvfe_ctx* ctx);
const uint8_t* kvfe_frontend_packets_view(const kvfe_ctx* ctx);
/* kvfe_frontend_submit with the batch's images already in device memory (densely packed: image b at
 * left_dev + b * width * height). */
int kvfe_frontend_submit_dev(kvfe_ctx* ctx, const uint8_t* left_dev, const uint8_t* right_dev, size_t pitch,
                             const int64_t* timestamps, const double* keyframe_R_cur, uint8_t* packets);

/* Staged uploads.  Copies of a few hundred KB reach well under half of the host link rate, copies of
 * several MB reach it; and the frames of step k+1 do not depend on the results of step k (only the
 * IMU rotation does).  A kvfe_upload couples n contexts (same image size and batch) to a two-slot
 * device staging ring: kvfe_upload_frames enqueues ONE H2D copy per camera for the n * batch
 * densely packed images of the next step of every member (member 0's batch first) and returns at
 * once -- it may run one step ahead of the members -- and kvfe_frontend_submit_uploaded is
 * kvfe_frontend_submit with the images taken from the member's slice of the oldest upload it has
 * not consumed yet (device-side copy).  Uploads are issued by one thread; every member must
 * consume upload s before upload s+2 is issued. */
typedef struct kvfe_upload kvfe_upload;
int kvfe_upload_create(kvfe_ctx* const* ctxs, int n, kvfe_upload** out);
void kvfe_upload_destroy(kvfe_upload* u);      /* before the member contexts */
int kvfe_upload_frames(kvfe_upload* u, const uint8_t* left, const uint8_t* right, size_t pitch);
int kvfe_frontend_submit_uploaded(kvfe_ctx* ctx, kvfe_upload* u, int member, const int64_t* timestamps,
                                  const double* keyframe_R_cur, uint8_t* packets);
/* submit on each of n contexts, then wait on each (one blocking call for n sub-batches). */
int kvfe_frontend_step_multi(kvfe_ctx* const* ctxs, int n, const uint8_t* const* const* left,
                             const uint8_t* const* const* right, size_t pitch,
                             const int64_t* const* timestamps, const double* const* keyframe_R_cur,
                             uint8_t* const* packets);
/* Enqueues one kvfe_frontend_step_dev on each of n contexts (sub-batches that run concurrently on
 * their own CUDA streams) with a single host call; arrays are indexed by context. */
int kvfe_frontend_step_dev_multi(kvfe_ctx* const* ctxs, int n, const uint8_t* const* left_dev,
                                 const uint8_t* const* right_dev, size_t pitch,
                                 const int64_t* const* timestamps, const double* const* keyframe_R_cur);
int kvfe_frontend_read_packets(kvfe_ctx* ctx, uint8_t* packets);
int kvfe_frontend_read_rectified(kvfe_ctx* ctx, int stream, uint8_t* rect_left,
                                 uint8_t* rect_right, size_t rect_pitch);
int kvfe_sync(kvfe_ctx* ctx);
void* kvfe_cuda_stream(kvfe_ctx* ctx);   /* cudaStream_t the context launches on */

/* ---------------------------------------------------------------------------------------------
 * Pipeline: the queue-in / queue-out shape the reference puts around its front-end
 * (include/kimera-vio/pipeline/PipelineModule.h:190-232 spin(): getInputPacket -> spinOnce ->
 * pushOutputPacket; :359-416 the SIMO module's input queue and output callbacks), for `n_streams`
 * independent camera streams served by native dispatcher threads inside the library.
 *
 *   push   enqueues one stereo frame of one stream (FrontendInputPacketBase: images, timestamp and the
 *          rotation the IMU front-end integrated) and returns at once;
 *   pop    returns finished frames in COMPLETION order: the output packet (kvfe_packet_header + SoA
 *          arrays, exactly the layout of kvfe_frontend_step) and, for keyframes, the rectified image
 *          pair the reference materialises inside the StereoFrame (StereoFrame.h:71-87) -- all in
 *          pinned host memory owned by the pipeline until kvfe_pipeline_release.
 *
 * One stream == one device-resident context; a frame costs the host one ~100-byte write into a
 * mapped I/O block and ONE cudaGraphLaunch.  Images in pinned (cudaHostAlloc / cudaHostRegister'ed)
 * memory are read by the SMs over the host link (zero-copy: no copy-engine queue between streams);
 * images in pageable memory are staged through a pinned slot first; device pointers are read in
 * place.  Input images must stay valid until the frame's output has been popped.  Outputs travel as
 * SM stores into mapped host memory; completion is a sequence number the last kernel publishes, so
 * the dispatchers issue no CUDA call besides the graph launch.
 *
 * rotation_mode 0: R = camLrectLkf_R_camLrectK (StereoVisionImuFrontend.cpp:149-150), which the caller
 *   can only form after it has seen frame k-1's keyframe decision (one frame in flight per stream);
 * rotation_mode 1: R = camLrectKm1_R_camLrectK, the rotation integrated between two consecutive frames;
 *   the front-end accumulates it since the last keyframe itself, as the reference's front-end does with
 *   the IMU measurements of its input packet (StereoVisionImuFrontend.cpp:140-150, :196-203), so
 *   frames can be queued ahead without a host round trip.
 * ------------------------------------------------------------------------------------------- */
typedef struct kvfe_pipeline kvfe_pipeline;
typedef struct {
  int32_t n_streams;        /* independent camera streams (cfg->batch is ignored: one context per stream) */
  int32_t n_workers;        /* dispatcher threads (0 = default) */
  int32_t queue_depth;      /* input queue capacity per stream (frames) */
  int32_t output_slots;     /* output buffers per stream (>= 2); a stream stalls when all are unreleased */
  int32_t want_rectified;   /* deliver the rectified image pair of every keyframe */
  int32_t rotation_mode;    /* 0 / 1, see above */
  int32_t checksum_outputs; /* the dispatcher reads every delivered byte (packet, rectified images) and
                               returns a 64-bit checksum with the output */
  int32_t max_in_flight;    /* steps in flight per stream on the GPU, 1 or 2 (0 = default 2) */
  int32_t prefetch;         /* > 0: when a stream's NEXT frame is already queued at launch time (dense rows, 16-byte
                               aligned, device or pinned memory), its images are pulled into a staging slot by a side
                               branch of the current step's graph.  Off by default: with 32 streams on one B200 the
                               forked graphs measured slower than the plain chain (see pipeline.cu) */
  int32_t split_graphs;     /* 0 = default (on), < 0 = off.  On: the step is two graph launches -- [fetch .. keyframe decision], then, once the dispatcher
                               has seen the decision in the mapped I/O block, EITHER the keyframe kernels + packet assembly OR
                               the packet assembly alone (13 kernel launches for a tracking frame instead of 36) */
} kvfe_pipeline_config;
typedef struct {
  int32_t stream, slot;     /* slot: pass back to kvfe_pipeline_release */
  uint64_t tag;             /* the tag given at push */
  int32_t is_keyframe, n_keypoints;
  uint64_t checksum;        /* checksum_outputs: sum of the 64-bit words of the used part of the packet
                               (+ the rectified images of a keyframe) */
  const uint8_t* packet;    /* kvfe_pipeline_packet_bytes() bytes */
  const uint8_t* rect_left; /* width*height dense, NULL unless want_rectified and is_keyframe */
  const uint8_t* rect_right;
} kvfe_pipeline_output;
typedef struct {
  int64_t frames_pushed, frames_done, graph_launches, kernel_launches;
  double launch_seconds;    /* host time spent inside the launch path (I/O block write + cudaGraphLaunch) */
  int64_t staged_copies;    /* frames whose images were in pageable memory and had to be staged */
} kvfe_pipeline_stats;
int kvfe_pipeline_create(const kvfe_config* cfg, const kvfe_rig* rig, const kvfe_pipeline_config* pc,
                         kvfe_pipeline** out);
void kvfe_pipeline_destroy(kvfe_pipeline* p);
const char* kvfe_pipeline_last_error(const kvfe_pipeline* p);
size_t kvfe_pipeline_packet_bytes(const kvfe_pipeline* p);
int kvfe_pipeline_packet_offsets(const kvfe_pipeline* p, size_t* offsets, int max_entries);
int kvfe_pipeline_max_keypoints(const kvfe_pipeline* p);
/* KVFE_ERR_CAPACITY when the stream's input queue is full (nothing enqueued; retry later). */
int kvfe_pipeline_push(kvfe_pipeline* p, int stream, const uint8_t* left, const uint8_t* right, size_t pitch,
                       int64_t timestamp, const double* R, uint64_t tag);
/* n frames with one call; returns the number accepted (stops at the first full queue) or < 0. */
int kvfe_pipeline_push_many(kvfe_pipeline* p, int n, const int32_t* streams, const uint8_t* const* left,
                            const uint8_t* const* right, size_t pitch, const int64_t* timestamps,
                            const double* R, const uint64_t* tags);
/* RGB-D pipeline (frontend_type 2): one intensity image and its registered depth image (cfg.depth.depth_type,
 * depth_pitch_bytes per row).  Depth may sit in pageable, pinned or device memory, with the same rules as the images; it
 * crosses the host link only for the first frame and keyframes (fetched after the keyframe decision), so a frame moves
 * W*H*(1 + rho*elem) bytes with rho the keyframe share and elem 2 or 4.  No rectified pair is delivered.  The prefetch
 * option does not apply. */
int kvfe_pipeline_push_rgbd(kvfe_pipeline* p, int stream, const uint8_t* img, size_t pitch, const void* depth,
                            size_t depth_pitch_bytes, int64_t timestamp, const double* R, uint64_t tag);
/* Frame::isKeyframe_ = true (user-enforced keyframe, VisionImuFrontend.cpp:207-209) for the next frame pushed on `stream`. */
int kvfe_pipeline_force_keyframe(kvfe_pipeline* p, int stream);
/* Up to max_n finished frames; blocks up to timeout_ms (0: poll) while none is ready.  Returns the count. */
int kvfe_pipeline_pop(kvfe_pipeline* p, kvfe_pipeline_output* outs, int max_n, int timeout_ms);
int kvfe_pipeline_release(kvfe_pipeline* p, const kvfe_pipeline_output* outs, int n);
/* All streams back to the bootstrap state; the pipeline must be idle (every pushed frame popped). */
int kvfe_pipeline_reset(kvfe_pipeline* p);
int kvfe_pipeline_get_stats(kvfe_pipeline* p, kvfe_pipeline_stats* st);

/* Debug taps of the last step for parity tests (stream-major, cap entries per stream). */
int kvfe_debug_lk(kvfe_ctx* ctx, int stream, float* pred_x, float* pred_y, float* next_x,
                  float* next_y, uint8_t* status, int* n);

#ifdef __cplusplus
}
#endif
#endif /* KVFE_H_ */
