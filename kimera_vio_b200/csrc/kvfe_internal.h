// kvfe_internal.h -- device-side data layout and kernel launchers shared by the .cu files.
//
// Data layout in HBM (one context, B streams, cap = keypoint capacity):
//   * image pyramids: 2 slots (previous / current frame) x B streams; each stream-slot is one
//     contiguous block holding levels 0..L (level l at lvl_off[l], row pitch lvl_pitch[l]).
//   * right raw image, rectified left/right images, GFTT response map, detection mask: B images.
//   * frame SoA: 3 frame slots per stream (km1, lkf, k may alias), every field a flat array
//     indexed by (stream*3 + slot)*cap + i.
//   * per-stream FSM state (StreamState) and the packed output packets.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/kvfe.h"

#define KVFE_MAX_LEVELS 8
#define KVFE_MAX_RANSAC_ITERS 1024
#define KVFE_IN_SLOTS 8

struct CamModel {        // one camera of the rig, everything the kernels need (f64)
  double fx, fy, cx, cy;
  double k1, k2, p1, p2;
  double R[9];           // rectification rotation (R1 / R2)
  double P[12];          // new projection (P1 / P2)
  double PP[9];          // P[:, :3]
  double RP[9];          // P[:, :3] * R   (cv::gemm 3x3 fast path: (a0*b0 + a1*b1) + a2*b2)
  double iR[9];          // inv(RP), cv::invert 3x3 cofactor formula -- for map recomputation
  int model;             // 0 radial-tangential (k1 k2 p1 p2), 1 equidistant / cv::fisheye (k1..k4 held in k1 k2 p1 p2)
  int pad;
};

struct FrameSoA {        // flat arrays, index (stream*3 + slot)*cap + i
  int* n;                // [B*3]
  float *kx, *ky;
  long long* lmk;
  int* age;
  double* versor;        // *3
  int* lstat; float *lrx, *lry;
  int* rstat; float *rrx, *rry;
  int* mstat;            // status right after template matching (before depth / RANSAC rewrite it)
  double* depth;
  double* p3d;           // *3
  float *rkx, *rky;
  long long* timestamp;  // [B*3]
  long long* frame_id;   // [B*3]
};

struct StreamState {     // one per stream, device resident
  int frame_count;
  int slot_km1, slot_lkf, slot_k;
  int mode;              // 0 bootstrap, 1 nominal non-KF, 2 keyframe, 3 all tracks lost
  int mono_status, stereo_status;
  int need;              // corners needed by the detector this step
  int n_existing;
  int use_pred;          // rotational prediction active this step
  int n_ref;             // keypoints fed to LK
  int n_new;             // corners appended by the detector
  long long lmk_next;    // FeatureDetector.cpp:141 static counter (one per stream == per process)
  long long timestamp;
  double kf_R_ref[9];    // keyframe_R_ref_frame_
  double kf_R_cur[9];    // input of this step
  double ref_R_cur[9];
  float H[9];            // K * R^T * K^-1 (float, cv::Matx33f semantics)
  double pose_mono[12], pose_stereo[12], info_stereo[9];
  double median_disparity;
  int given_rot;
  int nr_tracked, nr_mono_put, nr_mono_inl, nr_stereo_put, nr_stereo_inl;
  double acc_R[9];       // rotation input mode 1 (frame-to-frame rotations): lkf_R_km1 accumulated on the
                         // device like the IMU front-end's preintegration (reset at every keyframe)
};

// Per-step I/O block in pinned, mapped host memory (one per pyramid slot of a context): the host fills
// it and launches the pipeline step graph; the first kernels of the graph read their inputs -- image
// source pointers included -- straight from it, the last one stores the outputs through the pointers it
// names and then publishes `done_seq`.  Layout: this header, then at KVFE_STEPIO_ARRAYS: ts[B] (i64),
// R[B*9] (f64).
#define KVFE_STEPIO_ARRAYS 256
struct StepIO {
  const unsigned char* srcL;     // batch images, image b at srcL + b * src_pitch * H (device or mapped host memory)
  const unsigned char* srcR;
  unsigned long long src_pitch;
  unsigned char* dst_packets;    // B * packet_bytes (mapped host memory), may be null
  unsigned char* dst_rectL;      // B * W * H dense: rectified images of the keyframes of this step, may be null
  unsigned char* dst_rectR;
  unsigned long long seq;        // echoed into done_seq by the last kernel of the step
  int rot_mode;                  // 0: R = lkf_R_cur (StereoVisionImuFrontend.cpp:149-150); 1: R = km1_R_cur
  int force_kf;                  // Frame::isKeyframe_ of this frame (user-enforced keyframe, VisionImuFrontend.cpp:209)
  const unsigned char* next_srcL;   // images of the stream's NEXT frame when it is already queued (dense rows, 16-byte
  const unsigned char* next_srcR;   // aligned), else null: pulled into the staging slot while this step computes
  const unsigned char* srcD;     // RGB-D: the frame's depth image (device or mapped host memory), srcD_pitch bytes per row
  unsigned long long srcD_pitch;
  unsigned long long pad1[4];
  volatile unsigned long long done_seq;   // device -> host, own 64-byte line
  unsigned long long pad2[7];
  volatile unsigned long long decided_seq;  // split step graphs: published right after the keyframe decision, own line
  volatile int decided_mode;                // StreamState::mode of the frame (1 = tracking frame: no keyframe kernels needed)
};
static_assert(sizeof(StepIO) <= KVFE_STEPIO_ARRAYS, "StepIO header must fit before the arrays");

struct DevCfg {          // passed by value to kernels
  int W, H, pitch;       // level-0 geometry; pitch in bytes (multiple of 16)
  int B, cap;
  int n_levels;          // pyramid levels actually used by LK (maxLevel + 1)
  int lvl_w[KVFE_MAX_LEVELS], lvl_h[KVFE_MAX_LEVELS], lvl_pitch[KVFE_MAX_LEVELS];
  size_t lvl_off[KVFE_MAX_LEVELS];
  size_t pyr_stride;     // bytes per stream-slot pyramid
  size_t img_stride;     // bytes per full-res u8 image (pitch * H)
  // tracker
  int win, max_iter; double eps2; float min_eig_thr;
  int max_age;
  int pred_type;
  // detector
  int max_features, max_before_anms, min_distance, nms_enabled, nms_type;
  int hbins, vbins; unsigned char bin_mask[64]; int n_active_bins;
  double quality;        // quality_level as given: cv::GFTTDetector keeps it a double
  int subpix_enabled, subpix_win, subpix_iters, subpix_zero; double subpix_eps2;
  int sobel_tail_start;
  int cand_cap;          // candidate list capacity per stream
  // stereo
  int templ_cols, templ_rows, stripe_cols, stripe_rows;
  double min_depth, max_depth, fx_b; float tol_templ;
  int subpix_stereo;
  // ransac / fsm
  int ransac_iters; double thr_mono, thr_stereo, ransac_prob;
  int min_mono_inl, min_stereo_inl, use_2pt, use_1pt, use_ransac, use_stereo_tracking;
  double disparity_thr, max_disparity;
  long long min_kf_ns, max_kf_ns; int min_features;
  // rectified calibration
  double fx, fy, cxr, cyr, baseline;
  // mesher
  int mesh_on; float subdiv_factor;
  int mono;              // frontend_type 1: MonoVisionImuFrontend (no stereo half)
  // frontend_type 2: RgbdVisionImuFrontend -- the depth image of stream b at DevBuf::depth + b * depth_stride, depth_row bytes
  // per row (W * 2 or W * 4); kvfe_depth_params as the kernels use them
  int rgbd, depth_type;
  size_t depth_row, depth_stride;
  float depth_to_m, depth_min;                  // getDepthAtPoint
  float depth_lo, depth_hi; unsigned int depth_lo16, depth_hi16;   // getDetectionMask bounds (f32 / u16 images)
  double depth_fx_b;                            // fx * virtual_baseline (RgbdFrame.cpp:66)
  // ingest
  int equalize;          // cv::equalizeHist on both raw images before anything else (stereo_matching_params.equalize_image)
};

struct DevBuf {
  unsigned char* pyr[2];       // B * pyr_stride each
  unsigned char* right_raw;    // B * img_stride
  uint2* rmap[2];              // per camera W*H: {ix | iy << 16 (int16 each), fx | fy << 5}
  unsigned char* rectL;        // B * img_stride
  unsigned char* rectR;
  unsigned char* mask;         // B * img_stride (u8 0/255)
  unsigned char* depth;        // RGB-D: B * depth_stride (null otherwise)
  float* eig;                  // B * W*H
  unsigned int* eig_max;       // B (ordered-int encoded float)
  unsigned long long* cand;    // B * cand_cap  (float bits << 32 | pixel index)
  int* cand_n;                 // B
  int* cand_hist;              // B * 2048: histogram of the candidates' float bits below the maximum (top-K prefilter)
  unsigned long long* cand_sel;  // B * 16384: the best candidates, compacted (unordered)
  int* cand_sel_n;             // B
  int* greedy_redo;            // B: the prefix did not reach maxCorners, the full list decides
  int* corner_idx;             // B * max_before_anms: accepted GFTT corners (pixel index), in order
  int* corner_n;               // B
  float *new_x, *new_y;        // B * cap: corners after NMS / subpix
  int* new_n;                  // B
  int* scratch_i;              // B * scratch_stride ints (cell lists, states, ...)
  size_t scratch_stride;
  unsigned short* sort_perm;   // all-equal-keys std::sort permutations, triangular: perm(N) at N*(N-1)/2
  int* rnd_table;              // OpenGV rnd() sequence
  int rnd_n;
  // LK staging
  float *lk_px, *lk_py;        // ref points fed to LK   (B*cap)
  float *lk_qx, *lk_qy;        // predicted / tracked    (B*cap)
  float *lk_pred_x, *lk_pred_y;
  int* lk_src;                 // index in the ref frame (B*cap)
  unsigned char* lk_status;    // B*cap
  // matches / ransac staging
  int *m_ref, *m_cur;          // B*cap
  int* m_n;                    // B
  int* inl;                    // B*cap (inlier flags / lists)
  int* inl_n;                  // B
  float* subpix_mask;          // (2*win+1)^2 Gaussian weights of cv::cornerSubPix (host expf)
  float* subpix_mask_stereo;   // same for the hard-coded stereo refinement window (10)
  double* rs_d;                // B * rs_stride doubles
  size_t rs_stride;
  FrameSoA fr;
  StreamState* st;             // B
  unsigned char* packets;      // B * packet_bytes
  size_t packet_bytes;
  size_t pk_off[32];
  int* force_kf;               // B: user-enforced keyframe (Frame::isKeyframe_) for the next step, cleared by decide_kernel
  int* mesh_ws;                // quad-edge workspace of the mesh kernel when it does not fit shared memory
  unsigned char* stage_img[2]; // pipeline prefetch staging, per pyramid slot: [cam][B] dense images, img_stride apart (or null)
  unsigned long long* stage_seq; // [2]: sequence number of the frame held by stage_img[slot] (0: none)
  const void* lk_tmaps;        // HOST pointer (never dereferenced on the device): CUtensorMap[2 pyramid slots][KVFE_MAX_LEVELS],
                               // (x, y, stream) u8 tensors of the pyramid levels, box 48 x 28 x 1 -- launch_lk passes them
                               // to lk_kernel_tma as a __grid_constant__ parameter; null when they could not be built
};

struct kvfe_ctx {
  kvfe_config cfg;
  kvfe_rig rig;
  DevCfg dc;
  DevBuf db;
  CamModel cam[2];
  CamModel* d_cam;             // device copy [2]
  cudaStream_t stream;
  int cur_slot;                // pyramid slot of the frame being processed
  long long launches;
  char err[512];
  // pinned staging for the host-buffer step
  unsigned char* h_stage;      // 2 * B * img_stride
  unsigned char* h_packets;
  // submit/wait pipeline (depth KVFE_PIPE_DEPTH): pinned packet staging per in-flight step
  cudaEvent_t pipe_done[2]; unsigned char* pipe_user[2]; int pipe_io_slot[2]; int last_io_slot;
  // pinned I/O block per pyramid slot: [ts: B x i64][R: B x 9 f64][pad][packets]; the host-step graph
  // (host_graph) holds the H2D copy of the inputs, the kernel sequence and the D2H copy of the packets
  unsigned char* h_io[2]; size_t in_bytes, io_pk_off;
  unsigned char* d_in;         // device copy of the inputs (d_ts / d_Rin point into it)
  cudaGraphExec_t host_graph[2]; int host_graph_ready[2]; long long host_graph_launches;
  unsigned long long n_submitted, n_waited;
  long long* d_ts; double* d_Rin;        // step inputs
  const long long* in_ts; const double* in_R;   // what prep_kernel reads: d_ts/d_Rin, or the mapped pinned I/O block
  long long* h_ts; double* h_Rin;        // KVFE_IN_SLOTS pinned slots each
  cudaEvent_t in_ev[KVFE_IN_SLOTS]; int in_used[KVFE_IN_SLOTS]; int in_slot;
  cudaGraphExec_t step_graph[2];   // captured kernel sequence of one step, per pyramid slot
  int graph_ready[2];
  int use_graph, use_cond;
  long long graph_launches, graph_launches_kf;   // per step: always / inside the IF body
  int* d_kf_steps;             // device counter: executions of the IF body
  int* circle_hw;              // device: half widths of the filled-circle raster rows (2r+1)
  int circle_r;
  int device;                  // CUDA device the context lives on
  // pipeline step (pipeline.cu): I/O blocks in mapped pinned memory, one graph per pyramid slot
  unsigned char* pio[2];
  cudaGraphExec_t pipe_graph[2]; int pipe_graph_ready[2]; long long pipe_graph_launches;
  // split variant: [fetch .. decide, publish_decision] | host picks | [keyframe kernels, finalize, publish] or [finalize, publish]
  cudaGraphExec_t pipe_graph_a[2], pipe_graph_kf[2], pipe_graph_nokf[2]; int pipe_split_ready[2];
  long long pipe_launches_a, pipe_launches_kf, pipe_launches_nokf;
  unsigned int* d_pub_count;   // last-block-done counters: [0] publish_io_kernel, [1] prefetch_io_kernel
  unsigned char* own_packets;  // the internal packet buffer while kvfe_frontend_bind_packets points db.packets elsewhere
  cudaStream_t side;           // capture-time fork of the pipeline step graph (prefetch branch); no work is ever queued on it
  cudaEvent_t ev_fork, ev_join;
};

// ---- launchers (each returns the number of kernels it launched) ------------------------------
// rectify.cu
int launch_rectify(const DevCfg& dc, const uint2* rmap, const unsigned char* src, size_t src_stride,
                   unsigned char* dst, size_t dst_stride, int nimg, const StreamState* st, int mode_mask,
                   cudaStream_t s);
int launch_rmap_table(const DevCfg& dc, const CamModel* d_cam, int cam, uint2* rmap, cudaStream_t s);
int launch_maps(const DevCfg& dc, const CamModel* d_cam, int cam, float* mx, float* my, cudaStream_t s);
// pyramid.cu
int launch_pyramid(const DevCfg& dc, unsigned char* pyr, int nimg, cudaStream_t s);
// lk.cu
int launch_lk(const DevCfg& dc, const DevBuf& db, int prev_slot, int cur_slot, cudaStream_t s);
// gftt.cu
int launch_gftt(const DevCfg& dc, const DevBuf& db, const unsigned char* img, size_t img_stride,
                const int* circle_hw, int circle_r, int mode_mask, cudaStream_t s, int keep_mask = 0);
int launch_min_eig(const DevCfg& dc, const DevBuf& db, const unsigned char* img, size_t img_stride,
                   int mode_mask, cudaStream_t s);
// select.cu (ANMS + subpix + append)
int launch_select(const DevCfg& dc, const DevBuf& db, const unsigned char* img, size_t img_stride,
                  const CamModel* d_cam, int mode_mask, int append, cudaStream_t s);
// stereo.cu
int launch_sparse_stereo(const DevCfg& dc, const DevBuf& db, const CamModel* d_cam, int mode_mask,
                         int reuse_tracked, cudaStream_t s);
int launch_undistort(const DevCfg& dc, const CamModel* d_cam, int cam, int use_R, int use_P,
                     const float* x, const float* y, int n, float* ox, float* oy, cudaStream_t s);
int launch_bearing(const DevCfg& dc, const CamModel* d_cam, const float* x, const float* y, int n,
                   double* versors, cudaStream_t s);
int launch_check_rect_raw(const DevCfg& dc, const CamModel* d_cam, int cam, const float* dx, const float* dy, const float* ux,
                          const float* uy, int n, float tol, int* status, float* ox, float* oy, cudaStream_t s);
int launch_distort_unrectify_raw(const DevCfg& dc, const CamModel* d_cam, int cam, const int* status, const float* x,
                                 const float* y, int n, float* ox, float* oy, cudaStream_t s);
int launch_sparse_stereo_part(const DevCfg& dc, const DevBuf& db, const CamModel* d_cam, int mode_mask, int which, cudaStream_t s);
// ransac.cu
int launch_median_disparity_raw(const DevCfg& dc, const DevBuf& db, int m, double* out, cudaStream_t s);
int launch_point3_cov_raw(const DevCfg& dc, const float* ul, const float* ur, const float* v, const double* p3d, int n,
                          const double* Rm, double* op, double* ocov, cudaStream_t s);
int launch_ransac_mono(const DevCfg& dc, const DevBuf& db, int mode_mask, cudaStream_t s);
int launch_ransac_stereo(const DevCfg& dc, const DevBuf& db, int mode_mask, cudaStream_t s);
int launch_ransac_mono_raw(const DevCfg& dc, const DevBuf& db, const double* f_ref, const double* f_cur,
                           int n, const double* R12, int use_2pt, int* inl, int* n_inl, double* pose,
                           int* status, cudaStream_t s);
int launch_ransac_1pt_raw(const DevCfg& dc, const DevBuf& db, const float* rl, const float* rr,
                          const float* cl, const float* cr, const double* p_ref, const double* p_cur,
                          int n, const double* R, int* inl, int* n_inl, double* pose, double* info,
                          int* status, cudaStream_t s);
int launch_ransac_3pt_raw(const DevCfg& dc, const DevBuf& db, const double* p_ref, const double* p_cur,
                          int n, int* inl, int* n_inl, double* pose, int* status, cudaStream_t s);
// fsm.cu
int launch_prep(const DevCfg& dc, const DevBuf& db, const CamModel* d_cam, const long long* ts,
                const double* Rin, const StepIO* io, cudaStream_t s);
int launch_fetch_io(const DevCfg& dc, const DevBuf& db, const StepIO* io, int cur_slot, cudaStream_t s);
int launch_fetch_right_io(const DevCfg& dc, const DevBuf& db, const StepIO* io, int cur_slot, int mode_mask, cudaStream_t s);
int launch_fetch_depth_io(const DevCfg& dc, const DevBuf& db, const StepIO* io, int mode_mask, cudaStream_t s);
int launch_prefetch_io(const DevCfg& dc, const DevBuf& db, const StepIO* io, int cur_slot, unsigned int* counter, cudaStream_t s);
int launch_publish_io(const DevCfg& dc, const DevBuf& db, StepIO* io, unsigned int* counter, cudaStream_t s);
int launch_track_pre(const DevCfg& dc, const DevBuf& db, cudaStream_t s);
int launch_track_post(const DevCfg& dc, const DevBuf& db, const CamModel* d_cam, cudaStream_t s);
int launch_fetch(const unsigned char* srcL, const unsigned char* srcR, unsigned char* dstL, size_t dstL_stride,
                 unsigned char* dstR, size_t dstR_stride, size_t img, int B, cudaStream_t s);
int launch_publish(void* dst_host, const void* src_dev, size_t bytes, cudaStream_t s);
int launch_decide(const DevCfg& dc, const DevBuf& db, unsigned long long cond, cudaStream_t s);
int launch_detect_pre(const DevCfg& dc, const DevBuf& db, int mode_mask, int* kf_counter, cudaStream_t s);
int launch_finalize(const DevCfg& dc, const DevBuf& db, cudaStream_t s);
int launch_reset(const DevCfg& dc, const DevBuf& db, cudaStream_t s);
// ingest.cu
int launch_equalize(const DevCfg& dc, unsigned char* imgs, size_t img_stride, int nimg, const StreamState* st, int mode_mask,
                    cudaStream_t s);
// rgbd.cu
int launch_depth_mask(const DevCfg& dc, const unsigned char* depth, size_t pitch_bytes, int depth_type, float lo, float hi,
                      unsigned int lo16, unsigned int hi16, unsigned char* mask, size_t mask_pitch, cudaStream_t s);
int launch_rgbd_fill(const DevCfg& dc, const CamModel* d_cam, const unsigned char* depth, size_t pitch_bytes, int depth_type,
                     float depth_to_meters, float min_depth, double fx_b, const float* kp_x, const float* kp_y, const int* left_status,
                     const float* left_x, const float* left_y, const double* versors, int n, int* right_status, float* right_x,
                     float* right_y, double* depth_out, double* p3d, float* right_kp_x, float* right_kp_y, cudaStream_t s);
// the same two on frame slot k of every stream whose mode is in mode_mask (frame-level RGB-D step)
int launch_depth_mask_batch(const DevCfg& dc, const DevBuf& db, int mode_mask, cudaStream_t s);
int launch_rgbd_fill_batch(const DevCfg& dc, const DevBuf& db, const CamModel* d_cam, int mode_mask, cudaStream_t s);
// mesh.cu
bool mesh_fits_smem(const DevCfg& dc);
size_t mesh_global_ws_ints(const DevCfg& dc);
int launch_mesh_init(const DevCfg& dc);
int launch_mesh(const DevCfg& dc, const DevBuf& db, cudaStream_t s);
int launch_mesh_raw(const DevCfg& dc, const DevBuf& db, const float* x, const float* y, int n, float* tri, int max_tri,
                    int* n_tri, cudaStream_t s);
// api.cu (shared with pipeline.cu)
int kvfe_set_err(kvfe_ctx* ctx, int code, const char* fmt, ...);
int kvfe_enqueue_step_kernels(kvfe_ctx* ctx, const StepIO* io, long long* n_launch);
int kvfe_enqueue_step_part(kvfe_ctx* ctx, StepIO* io, int part, long long* n_launch);   // 0 track + decision, 1 keyframe + finalize, 2 finalize
int launch_publish_decision(const DevBuf& db, StepIO* io, cudaStream_t s);
