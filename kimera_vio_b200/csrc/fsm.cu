// fsm.cu -- the per-stream front-end state machine, device resident: one CTA (or one thread) per
// camera stream per stage, no host round trip inside a step.
//   prep         StereoVisionImuFrontend::processStereoFrame preamble (reference
//                src/frontend/StereoVisionImuFrontend.cpp:283-310): frame slot for k, ref_R_cur,
//                RotationalOpticalFlowPredictor homography (optical-flow/OpticalFlowPredictor.cpp:70-92)
//   track_pre    Tracker::featureTracking :102-129 (valid reference keypoints + predicted flow)
//   track_post   Tracker::featureTracking :162-189 (survivors, landmark invalidation in the ref frame,
//                bearing vectors)
//   decide       VisionImuFrontend::shouldBeKeyframe (src/frontend/VisionImuFrontend.cpp:175-232) and
//                the "all tracks lost" branch (StereoVisionImuFrontend.cpp:312-323; stereo only)
//   detect_pre   FeatureDetector::featureDetection(Frame*, R) :98-115 (ages, n_existing, need)
//   finalize     slot rotation, keyframe_R_ref_frame_ update (:462-475), getSmartStereoMeasurements
//                (:485-531), StereoFrame::checkStatusRightKeypoints (StereoFrame.cpp:106-143), packing.
#include <cstdlib>
#include "common.cuh"
#include "tma.cuh"
#include "matches.cuh"


__global__ void reset_kernel(DevCfg dc, DevBuf db) {
  int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= dc.B) return;
  StreamState& s = db.st[b];
  s.frame_count = 0; s.slot_km1 = 0; s.slot_lkf = 0; s.slot_k = 0; s.mode = 0;
  s.mono_status = KVFE_TRK_INVALID; s.stereo_status = KVFE_TRK_INVALID;
  s.lmk_next = 0; s.need = 0; s.n_existing = 0; s.n_ref = 0; s.n_new = 0; s.use_pred = 0; s.given_rot = 0;
  s.nr_tracked = s.nr_mono_put = s.nr_mono_inl = s.nr_stereo_put = s.nr_stereo_inl = 0;
  s.median_disparity = 0;
  for (int i = 0; i < 9; ++i) { s.kf_R_ref[i] = (i % 4 == 0) ? 1.0 : 0.0; s.acc_R[i] = s.kf_R_ref[i]; s.info_stereo[i] = 0; }
  for (int i = 0; i < 12; ++i) { s.pose_mono[i] = (i % 5 == 0) ? 1.0 : 0.0; s.pose_stereo[i] = s.pose_mono[i]; }
  for (int k = 0; k < 3; ++k) db.fr.n[b * 3 + k] = 0;
}

// `io` (may be null): the step inputs come from the pipeline's mapped I/O block instead of ts / Rin; with
// io->rot_mode == 1 the rotation given is km1_R_cur (what the gyroscope integrates between two frames) and
// keyframe_R_cur is accumulated here, exactly like the IMU front-end's preintegration that the reference's
// front-end owns and resets at keyframes (StereoVisionImuFrontend.cpp:140-150, :196-203).
__global__ void prep_kernel(DevCfg dc, DevBuf db, const CamModel* __restrict__ cams,
                            const long long* __restrict__ ts, const double* __restrict__ Rin,
                            const StepIO* __restrict__ io) {
  int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= dc.B) return;
  StreamState& s = db.st[b];
  int rot_mode = 0;
  if (io) {
    const unsigned char* arr = reinterpret_cast<const unsigned char*>(io) + KVFE_STEPIO_ARRAYS;
    ts = reinterpret_cast<const long long*>(arr);
    Rin = reinterpret_cast<const double*>(arr + (size_t)dc.B * sizeof(long long));
    rot_mode = io->rot_mode;
    if (io->force_kf) db.force_kf[b] = 1;
  }
  s.timestamp = ts[b];
  if (rot_mode == 1) {
    double Rk[9];
    for (int i = 0; i < 9; ++i) Rk[i] = Rin[9 * b + i];
    matmul3(s.acc_R, Rk, s.kf_R_cur);
  } else {
    for (int i = 0; i < 9; ++i) s.kf_R_cur[i] = Rin[9 * b + i];
  }
  s.n_ref = 0; s.n_new = 0;
  if (s.frame_count == 0) {
    s.mode = 0; s.slot_k = 0; s.slot_km1 = 0; s.slot_lkf = 0;
    s.use_pred = 0; s.given_rot = 0;
  } else {
    int k = 0;
    while (k == s.slot_km1 || k == s.slot_lkf) ++k;
    s.slot_k = k;
    s.mode = 1;
    // ref_frame_R_cur_frame = keyframe_R_ref_frame_.inverse().compose(keyframe_R_cur_frame)
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j)
        s.ref_R_cur[3 * i + j] = s.kf_R_ref[i] * s.kf_R_cur[j] +
                                 (s.kf_R_ref[3 + i] * s.kf_R_cur[3 + j] + s.kf_R_ref[6 + i] * s.kf_R_cur[6 + j]);
    // given_rot = !keyframe_R_cur_frame.equals(Rot3(), 1e-9)
    bool ident = true;
    for (int i = 0; i < 9; ++i) {
      double e = (i % 4 == 0) ? 1.0 : 0.0;
      if (!(fabs(s.kf_R_cur[i] - e) <= 1e-9)) ident = false;
    }
    s.given_rot = ident ? 0 : 1;
    // Eigen::Quaterniond(R).w()
    const double* R = s.ref_R_cur;
    double t = R[0] + (R[4] + R[8]);
    double qw;
    if (t > 0) qw = 0.5 * sqrt(t + 1.0);
    else {
      int i = 0;
      if (R[4] > R[0]) i = 1;
      if (R[8] > R[4 * i]) i = 2;
      int j = (i + 1) % 3, kk = (i + 2) % 3;
      double tt = sqrt(R[4 * i] - R[4 * j] - R[4 * kk] + 1.0);
      qw = (R[3 * kk + j] - R[3 * j + kk]) * (0.5 / tt);
    }
    s.use_pred = (dc.pred_type == 1) && !(fabs(1.0 - fabs(qw)) < 1e-4);
    // H = K * R^T * K^-1 in float (cv::Matx33f): s = 0; s += a(i,k) * b(k,j)
    float K[9] = {(float)cams[0].fx, 0.f, (float)cams[0].cx, 0.f, (float)cams[0].fy, (float)cams[0].cy, 0.f, 0.f, 1.f};
    float Rt[9];
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) Rt[3 * i + j] = (float)R[3 * j + i];
    float Ki[9];
    {
      const float* a = K;
      float d = a[0] * (a[4] * a[8] - a[7] * a[5]) - a[1] * (a[3] * a[8] - a[6] * a[5]) + a[2] * (a[3] * a[7] - a[6] * a[4]);
      d = 1.f / d;
      Ki[0] = (a[4] * a[8] - a[5] * a[7]) * d; Ki[1] = (a[2] * a[7] - a[1] * a[8]) * d; Ki[2] = (a[1] * a[5] - a[2] * a[4]) * d;
      Ki[3] = (a[5] * a[6] - a[3] * a[8]) * d; Ki[4] = (a[0] * a[8] - a[2] * a[6]) * d; Ki[5] = (a[2] * a[3] - a[0] * a[5]) * d;
      Ki[6] = (a[3] * a[7] - a[4] * a[6]) * d; Ki[7] = (a[1] * a[6] - a[0] * a[7]) * d; Ki[8] = (a[0] * a[4] - a[1] * a[3]) * d;
    }
    float T[9];
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) {
        float acc = 0.f;
        for (int q = 0; q < 3; ++q) acc += K[3 * i + q] * Rt[3 * q + j];
        T[3 * i + j] = acc;
      }
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) {
        float acc = 0.f;
        for (int q = 0; q < 3; ++q) acc += T[3 * i + q] * Ki[3 * q + j];
        s.H[3 * i + j] = acc;
      }
  }
  const int fs = b * 3 + s.slot_k;
  db.fr.n[fs] = 0;
  db.fr.timestamp[fs] = ts[b];
  db.fr.frame_id[fs] = s.frame_count;
}

// CTA-wide ordered compaction helper: returns the output position of `keep` elements (or -1)
__device__ __forceinline__ int block_compact_pos(int keep, int* s_total, int* wsum, int* s_chunk) {
  unsigned bal = __ballot_sync(KVFE_FULL_MASK, keep);
  int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) wsum[warp] = __popc(bal);
  __syncthreads();
  if (warp == 0) {
    int v = (lane < (blockDim.x >> 5)) ? wsum[lane] : 0, incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int t = __shfl_up_sync(KVFE_FULL_MASK, incl, o);
      if (lane >= o) incl += t;
    }
    wsum[lane] = incl - v;
    if (lane == 31) *s_chunk = incl;
  }
  __syncthreads();
  int pos = *s_total + wsum[warp] + __popc(bal & ((1u << lane) - 1));
  __syncthreads();
  if (threadIdx.x == 0) *s_total += *s_chunk;
  __syncthreads();
  return keep ? pos : -1;
}

__global__ void __launch_bounds__(256) track_pre_kernel(DevCfg dc, DevBuf db) {
  const int b = blockIdx.x;
  StreamState& s = db.st[b];
  if (s.mode == 0) return;
  __shared__ int s_total, s_chunk, wsum[32];
  if (threadIdx.x == 0) s_total = 0;
  __syncthreads();
  const int fs = b * 3 + s.slot_km1;
  const int n = db.fr.n[fs];
  const float Wf = (float)dc.W, Hf = (float)dc.H;
  for (int base = 0; base < n; base += blockDim.x) {
    int i = base + threadIdx.x;
    int keep = (i < n) && db.fr.lmk[(size_t)fs * dc.cap + i] != -1;
    int pos = block_compact_pos(keep, &s_total, wsum, &s_chunk);
    if (keep) {
      size_t g = (size_t)b * dc.cap + pos;
      float x = db.fr.kx[(size_t)fs * dc.cap + i], y = db.fr.ky[(size_t)fs * dc.cap + i];
      db.lk_px[g] = x; db.lk_py[g] = y; db.lk_src[g] = i;
      float nx = x, ny = y;
      if (s.use_pred) {
        const float* H = s.H;
        float p0 = 0.f, p1 = 0.f, p2 = 0.f;
        p0 += H[0] * x; p0 += H[1] * y; p0 += H[2] * 1.0f;
        p1 += H[3] * x; p1 += H[4] * y; p1 += H[5] * 1.0f;
        p2 += H[6] * x; p2 += H[7] * y; p2 += H[8] * 1.0f;
        float qx = x, qy = y;
        if (p2 > 0.0f) { qx = p0 / p2; qy = p1 / p2; }
        if (qx >= 0.f && qx < Wf && qy >= 0.f && qy < Hf) { nx = qx; ny = qy; }
      }
      db.lk_qx[g] = nx; db.lk_qy[g] = ny;
      db.lk_pred_x[g] = nx; db.lk_pred_y[g] = ny;
    }
  }
  if (threadIdx.x == 0) s.n_ref = s_total;
}

__global__ void __launch_bounds__(256) track_post_kernel(DevCfg dc, DevBuf db, const CamModel* __restrict__ cams) {
  const int b = blockIdx.x;
  StreamState& s = db.st[b];
  if (s.mode == 0) return;
  __shared__ int s_total, s_chunk, wsum[32];
  if (threadIdx.x == 0) s_total = 0;
  __syncthreads();
  const int fr = b * 3 + s.slot_km1, fk = b * 3 + s.slot_k;
  const int n = s.n_ref;
  for (int base = 0; base < n; base += blockDim.x) {
    int j = base + threadIdx.x;
    int keep = 0, src = 0;
    size_t g = (size_t)b * dc.cap + j;
    if (j < n) {
      src = db.lk_src[g];
      size_t kr = (size_t)fr * dc.cap + src;
      if (!db.lk_status[g] || db.fr.age[kr] > dc.max_age) db.fr.lmk[kr] = -1;   // Tracker.cpp:174-179
      else keep = 1;
    }
    int pos = block_compact_pos(keep, &s_total, wsum, &s_chunk);
    if (keep) {
      size_t kr = (size_t)fr * dc.cap + src, kk = (size_t)fk * dc.cap + pos;
      float x = db.lk_qx[g], y = db.lk_qy[g];
      db.fr.lmk[kk] = db.fr.lmk[kr];
      db.fr.age[kk] = db.fr.age[kr];
      db.fr.kx[kk] = x; db.fr.ky[kk] = y;
      float ux, uy;
      undistort_point(cams[0], x, y, 1, &ux, &uy);
      double v0 = (double)ux, v1 = (double)uy, v2 = 1.0;
      double n2 = v0 * v0 + (v1 * v1 + v2 * v2);
      double nrm = sqrt(n2);
      if (n2 > 0) { v0 = v0 / nrm; v1 = v1 / nrm; v2 = v2 / nrm; }
      db.fr.versor[3 * kk] = v0; db.fr.versor[3 * kk + 1] = v1; db.fr.versor[3 * kk + 2] = v2;
      // stereo fields of frame k are undefined until sparseStereoReconstruction runs
      db.fr.lstat[kk] = KVFE_KP_VALID; db.fr.rstat[kk] = KVFE_KP_NO_RIGHT_RECT;
    }
  }
  if (threadIdx.x == 0) { db.fr.n[fk] = s_total; s.nr_tracked = s_total; }
}

// `cond` (0 = none): conditional handle of the step graph; set to 1 as soon as any stream of the
// batch needs the keyframe / detection part (bootstrap, keyframe, all tracks lost), which otherwise
// is skipped as a whole (a CUDA-graph IF node around ~20 kernels that would all exit at entry).
__global__ void __launch_bounds__(256) decide_kernel(DevCfg dc, DevBuf db, cudaGraphConditionalHandle cond) {
  const int b = blockIdx.x;
  StreamState& s = db.st[b];
  if (s.mode == 0) {
    if (threadIdx.x == 0) { db.force_kf[b] = 0; if (cond) cudaGraphSetConditional(cond, 1); }
    return;
  }
  const int fk = b * 3 + s.slot_k, fl = b * 3 + s.slot_lkf;
  const int nk = db.fr.n[fk];
  if ((dc.mono || dc.rgbd) && threadIdx.x == 0) {   // reset on every frame, before the decision:
    s.mono_status = KVFE_TRK_INVALID;                // MonoVisionImuFrontend.cpp:266-267 (stereo DISABLED),
    s.stereo_status = dc.mono ? KVFE_TRK_DISABLED : KVFE_TRK_INVALID;   // RgbdVisionImuFrontend.cpp:271-272 (both INVALID)
  }
  __syncthreads();
  if (nk == 0 && !dc.mono && !dc.rgbd) {   // StereoVisionImuFrontend.cpp:312-323 (mono and RGB-D have no such shortcut)
    if (threadIdx.x == 0) { s.mode = 3; db.force_kf[b] = 0; if (cond) cudaGraphSetConditional(cond, 1); }
    return;
  }
  int* m_ref = db.m_ref + (size_t)b * dc.cap;
  int* m_cur = db.m_cur + (size_t)b * dc.cap;
  const int nm = block_find_matches(dc, db, fl, fk, false, m_ref, m_cur, db.scratch_i + (size_t)b * db.scratch_stride);
  double* tmp = db.rs_d + (size_t)b * db.rs_stride;
  double med = block_median_disparity(dc, db, fl, fk, m_ref, m_cur, nullptr, nm, tmp);
  // nr valid keypoints of frame k
  __shared__ int s_valid;
  if (threadIdx.x == 0) s_valid = 0;
  __syncthreads();
  int c = 0;
  for (int i = threadIdx.x; i < nk; i += blockDim.x) c += db.fr.lmk[(size_t)fk * dc.cap + i] != -1;
  if (c) atomicAdd(&s_valid, c);
  __syncthreads();
  if (threadIdx.x == 0) {
    double disparity = med < 0.0 ? 0.0 : med;
    s.median_disparity = disparity;
    long long kf_diff = db.fr.timestamp[fk] - db.fr.timestamp[fl];
    bool min_time = kf_diff >= dc.min_kf_ns, max_time = kf_diff >= dc.max_kf_ns;
    bool nr_low = s_valid <= dc.min_features;
    bool is_low = disparity < dc.disparity_thr;
    bool low_first = is_low && !(s.mono_status == KVFE_TRK_LOW_DISPARITY);
    bool enough = !is_low;
    bool max_disp = disparity > dc.max_disparity;
    bool flipped = (enough || low_first) && min_time;
    const bool forced = db.force_kf[b] != 0;          // frame.isKeyframe_ (VisionImuFrontend.cpp:207-209), one shot
    db.force_kf[b] = 0;
    bool kf = max_time || max_disp || flipped || nr_low || forced;
    s.mode = kf ? 2 : 1;
    if (kf) {
      // StereoVisionImuFrontend.cpp:345-346, :402-404; RGB-D the same (RgbdVisionImuFrontend.cpp:313-345): stereo_ransac_kernel
      // overwrites the stereo status, and leaves it INVALID without use_stereo_tracking
      s.mono_status = dc.use_ransac ? KVFE_TRK_INVALID : KVFE_TRK_DISABLED;
      s.stereo_status = dc.mono ? KVFE_TRK_DISABLED : (dc.use_ransac ? KVFE_TRK_INVALID : KVFE_TRK_DISABLED);
      if (cond) cudaGraphSetConditional(cond, 1);
    }
  }
}

// kf_counter (may be null): counts executions of the conditional keyframe part (launch accounting)
__global__ void __launch_bounds__(256) detect_pre_kernel(DevCfg dc, DevBuf db, int mode_mask, int* kf_counter) {
  const int b = blockIdx.x;
  if (kf_counter && b == 0 && threadIdx.x == 0) atomicAdd(kf_counter, 1);
  StreamState& s = db.st[b];
  if (!mode_on(s.mode, mode_mask)) return;
  const int fk = b * 3 + s.slot_k;
  const int n = db.fr.n[fk];
  __shared__ int s_cnt;
  if (threadIdx.x == 0) s_cnt = 0;
  __syncthreads();
  int c = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    size_t k = (size_t)fk * dc.cap + i;
    c += db.fr.lmk[k] != -1;
    db.fr.age[k] += 1;
  }
  if (c) atomicAdd(&s_cnt, c);
  __syncthreads();
  if (threadIdx.x == 0) {
    s.n_existing = s_cnt;
    int need = dc.max_features - s_cnt;
    s.need = need > 0 ? need : 0;
  }
}

__global__ void __launch_bounds__(256) finalize_kernel(DevCfg dc, DevBuf db) {
  const int b = blockIdx.x;
  StreamState& s = db.st[b];
  const int fk = b * 3 + s.slot_k;
  const int n = db.fr.n[fk];
  const int mode = s.mode;
  const bool is_kf = (mode == 0 || mode == 2);
  unsigned char* pk = db.packets + (size_t)b * db.packet_bytes;
  kvfe_packet_header* h = reinterpret_cast<kvfe_packet_header*>(pk);
  const size_t* off = db.pk_off;
  float* o_kx = (float*)(pk + off[0]); float* o_ky = (float*)(pk + off[1]);
  long long* o_lmk = (long long*)(pk + off[2]); int* o_age = (int*)(pk + off[3]);
  double* o_score = (double*)(pk + off[4]); double* o_ver = (double*)(pk + off[5]);
  int* o_ls = (int*)(pk + off[6]); float* o_lx = (float*)(pk + off[7]); float* o_ly = (float*)(pk + off[8]);
  int* o_rs = (int*)(pk + off[9]); float* o_rx = (float*)(pk + off[10]); float* o_ry = (float*)(pk + off[11]);
  double* o_depth = (double*)(pk + off[12]); double* o_p3d = (double*)(pk + off[13]);
  float* o_rkx = (float*)(pk + off[14]); float* o_rky = (float*)(pk + off[15]);
  long long* o_sl = (long long*)(pk + off[16]); double* o_suL = (double*)(pk + off[17]);
  double* o_suR = (double*)(pk + off[18]); double* o_sv = (double*)(pk + off[19]);
  __shared__ int cnt[5];
  __shared__ int s_total, s_chunk, wsum[32];
  if (threadIdx.x < 5) cnt[threadIdx.x] = 0;
  if (threadIdx.x == 0) s_total = 0;
  __syncthreads();
  const bool stereo_valid = (mode == 0 || mode == 2);
  for (int base = 0; base < n; base += blockDim.x) {
    int i = base + threadIdx.x;
    int keep = 0;
    size_t k = (size_t)fk * dc.cap + i;
    if (i < n) {
      o_kx[i] = db.fr.kx[k]; o_ky[i] = db.fr.ky[k]; o_lmk[i] = db.fr.lmk[k]; o_age[i] = db.fr.age[k];
      o_score[i] = 0.0;
      o_ver[3 * i] = db.fr.versor[3 * k]; o_ver[3 * i + 1] = db.fr.versor[3 * k + 1]; o_ver[3 * i + 2] = db.fr.versor[3 * k + 2];
      if (stereo_valid) {
        int rs = dc.mono ? -1 : db.fr.rstat[k];          // mono: no right camera; left_* = keypoints_undistorted_
        o_ls[i] = db.fr.lstat[k]; o_lx[i] = db.fr.lrx[k]; o_ly[i] = db.fr.lry[k];
        if (dc.mono) { db.fr.rrx[k] = 0.f; db.fr.rry[k] = 0.f; db.fr.depth[k] = 0.0; db.fr.p3d[3 * k] = db.fr.p3d[3 * k + 1] = db.fr.p3d[3 * k + 2] = 0.0; db.fr.rkx[k] = db.fr.rky[k] = 0.f; }
        o_rs[i] = rs; o_rx[i] = db.fr.rrx[k]; o_ry[i] = db.fr.rry[k];
        o_depth[i] = db.fr.depth[k];
        o_p3d[3 * i] = db.fr.p3d[3 * k]; o_p3d[3 * i + 1] = db.fr.p3d[3 * k + 1]; o_p3d[3 * i + 2] = db.fr.p3d[3 * k + 2];
        o_rkx[i] = db.fr.rkx[k]; o_rky[i] = db.fr.rky[k];
        if (rs >= 0 && rs < 5) atomicAdd(&cnt[rs], 1);
        keep = (mode == 2) && db.fr.lmk[k] != -1;      // smart measurements: keyframes of the nominal spin
      } else {
        o_ls[i] = -1; o_rs[i] = -1; o_lx[i] = o_ly[i] = o_rx[i] = o_ry[i] = 0.f; o_depth[i] = 0.0;
        o_p3d[3 * i] = o_p3d[3 * i + 1] = o_p3d[3 * i + 2] = 0.0; o_rkx[i] = o_rky[i] = 0.f;
      }
    }
    int pos = block_compact_pos(keep, &s_total, wsum, &s_chunk);
    if (keep) {
      o_sl[pos] = db.fr.lmk[k];
      o_suL[pos] = (double)db.fr.lrx[k];
      o_sv[pos] = (double)db.fr.lry[k];
      // RGB-D: uR whenever the right keypoint is VALID, use_stereo_tracking or not (RgbdVisionImuFrontend.cpp:370-399)
      o_suR[pos] = (!dc.mono && (dc.use_stereo_tracking || dc.rgbd) && db.fr.rstat[k] == KVFE_KP_VALID) ? (double)db.fr.rrx[k]
                                                                                : __longlong_as_double(0x7ff8000000000000LL);
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    h->n = n; h->is_keyframe = is_kf ? 1 : 0;
    h->mono_status = s.mono_status; h->stereo_status = s.stereo_status;
    h->n_smart = s_total;
    h->nr_tracked = (mode == 0) ? 0 : s.nr_tracked;
    h->nr_mono_putatives = s.nr_mono_put; h->nr_mono_inliers = s.nr_mono_inl;
    h->nr_stereo_putatives = s.nr_stereo_put; h->nr_stereo_inliers = s.nr_stereo_inl;
    h->nr_valid_rkp = cnt[0]; h->nr_no_left_rect_rkp = cnt[1]; h->nr_no_right_rect_rkp = cnt[2];
    h->nr_no_depth_rkp = cnt[3]; h->nr_failed_arun_rkp = cnt[4];
    h->mode = mode;
    h->frame_id = s.frame_count; h->timestamp = s.timestamp;
    for (int i = 0; i < 12; ++i) { h->lkf_T_k_mono[i] = s.pose_mono[i]; h->lkf_T_k_stereo[i] = s.pose_stereo[i]; }
    for (int i = 0; i < 9; ++i) h->info_stereo[i] = s.info_stereo[i];
    h->median_disparity = s.median_disparity;
    h->n_mesh_triangles = 0; h->reserved = 0;          // mesh_kernel fills it in on keyframes (cfg.mesh_2d)
    // rotation accumulated since the last keyframe (rotation input mode 1)
    for (int i = 0; i < 9; ++i) s.acc_R[i] = is_kf ? ((i % 4 == 0) ? 1.0 : 0.0) : s.kf_R_cur[i];
    // state update (StereoVisionImuFrontend.cpp:268-271, :317-319, :447-475)
    if (mode == 0) { s.slot_km1 = s.slot_k; s.slot_lkf = s.slot_k; }
    else if (mode == 3) { s.slot_km1 = s.slot_k; }
    else {
      if (mode == 2) {
        s.slot_lkf = s.slot_k;
        for (int i = 0; i < 9; ++i) s.kf_R_ref[i] = (i % 4 == 0) ? 1.0 : 0.0;
      } else {
        for (int i = 0; i < 9; ++i) s.kf_R_ref[i] = s.kf_R_cur[i];
      }
      s.slot_km1 = s.slot_k;
    }
    s.frame_count += 1;
  }
}

int launch_reset(const DevCfg& dc, const DevBuf& db, cudaStream_t s) {
  reset_kernel<<<(dc.B + 63) / 64, 64, 0, s>>>(dc, db);
  return 1;
}
int launch_prep(const DevCfg& dc, const DevBuf& db, const CamModel* d_cam, const long long* ts,
                const double* Rin, const StepIO* io, cudaStream_t s) {
  prep_kernel<<<(dc.B + 63) / 64, 64, 0, s>>>(dc, db, d_cam, ts, Rin, io);
  return 1;
}
int launch_track_pre(const DevCfg& dc, const DevBuf& db, cudaStream_t s) {
  track_pre_kernel<<<dc.B, 256, 0, s>>>(dc, db);
  return 1;
}
int launch_track_post(const DevCfg& dc, const DevBuf& db, const CamModel* d_cam, cudaStream_t s) {
  track_post_kernel<<<dc.B, 256, 0, s>>>(dc, db, d_cam);
  return 1;
}
int launch_decide(const DevCfg& dc, const DevBuf& db, unsigned long long cond, cudaStream_t s) {
  decide_kernel<<<dc.B, 256, 0, s>>>(dc, db, (cudaGraphConditionalHandle)cond);
  return 1;
}
int launch_detect_pre(const DevCfg& dc, const DevBuf& db, int mode_mask, int* kf_counter, cudaStream_t s) {
  detect_pre_kernel<<<dc.B, 256, 0, s>>>(dc, db, mode_mask, kf_counter);
  return 1;
}
// SM-driven copy of the packets into mapped pinned host memory (16-byte stores over the host link).
// A memcpy node / cudaMemcpyAsync would sit in the copy engine's in-order queue behind the D2H copies
// of contexts submitted earlier whose (three times longer) keyframe steps are still running, so
// every context would complete at the pace of the slowest one; a kernel has no such queue.
__global__ void __launch_bounds__(256) publish_kernel(uint4* __restrict__ dst, const uint4* __restrict__ src, size_t n16) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) dst[i] = src[i];
}
int launch_publish(void* dst_host, const void* src_dev, size_t bytes, cudaStream_t s) {
  const size_t n16 = bytes / 16;
  int blocks = (int)((n16 + 255) / 256);
  if (blocks > 64) blocks = 64;
  if (blocks < 1) blocks = 1;
  publish_kernel<<<blocks, 256, 0, s>>>(reinterpret_cast<uint4*>(dst_host), reinterpret_cast<const uint4*>(src_dev), n16);
  return 1;
}
// SM-driven placement of a sub-batch's images (contiguous in a device staging area) into the pyramid
// slot (level 0, stride pyr_stride) and the right-image buffer: one launch instead of two strided
// copy-engine operations.  grid (x, B, 2): y = image of the batch, z = camera.
__global__ void __launch_bounds__(256) fetch_kernel(const unsigned char* __restrict__ srcL, const unsigned char* __restrict__ srcR,
                                                    unsigned char* __restrict__ dstL, size_t dstL_stride,
                                                    unsigned char* __restrict__ dstR, size_t dstR_stride, size_t img) {
  const unsigned char* src = (blockIdx.z ? srcR : srcL) + (size_t)blockIdx.y * img;
  unsigned char* dst = blockIdx.z ? dstR + (size_t)blockIdx.y * dstR_stride : dstL + (size_t)blockIdx.y * dstL_stride;
  const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (size_t)gridDim.x * blockDim.x;
  if ((((size_t)src | (size_t)dst) & 15) == 0) {
    const size_t n16 = img / 16;
    for (size_t i = tid; i < n16; i += nth) reinterpret_cast<uint4*>(dst)[i] = reinterpret_cast<const uint4*>(src)[i];
    for (size_t i = n16 * 16 + tid; i < img; i += nth) dst[i] = src[i];
  } else {
    for (size_t i = tid; i < img; i += nth) dst[i] = src[i];
  }
}
int launch_fetch(const unsigned char* srcL, const unsigned char* srcR, unsigned char* dstL, size_t dstL_stride,
                 unsigned char* dstR, size_t dstR_stride, size_t img, int B, cudaStream_t s) {
  fetch_kernel<<<dim3(24, B, 2), 256, 0, s>>>(srcL, srcR, dstL, dstL_stride, dstR, dstR_stride, img);
  return 1;
}
// ---- pipeline step: image fetch and output publication through the mapped I/O block -----------------
// The source pointers are read from the I/O block, so ONE captured graph serves every step.  A source in
// pinned host memory is pulled over the host link by the SM's TMA unit (zero-copy): no copy-engine
// operation, hence no in-order copy queue shared between contexts and no small-copy inefficiency (a 361 KB
// cudaMemcpyAsync reaches well under half of the link rate).
//
// Bulk asynchronous copies (cp.async.bulk, tma.cuh): ONE warp per CTA streams its share of the image through a
// two-stage 8 KB shared-memory ring -- global/host -> shared on an mbarrier, shared -> global as a bulk
// group.  The first version of this kernel parked 44 CTAs x 256 threads per stream on 16-byte loads over the
// host link; with 32 streams in flight those threads took the SM slots of the compute kernels (measured on
// B200, 32 streams: 0.91 -> 0.83 ms per pass just by shrinking that grid to 8 CTAs).  grid (x, B, 2):
// y = image of the batch, z = camera; chunk c is handled by CTA c % gridDim.x.
#define FETCH_CHUNK 8192
#define FETCH_STAGES 2
struct BulkRing {
  unsigned char buf[FETCH_STAGES][FETCH_CHUNK];
  unsigned long long bar[FETCH_STAGES];
};
// one thread: initialise the ring's barriers (once per kernel)
__device__ __forceinline__ void bulk_ring_init(BulkRing& r) {
  for (int st = 0; st < FETCH_STAGES; ++st) tma::mbar_init(reinterpret_cast<uint64_t*>(&r.bar[st]), 1);
  tma::fence_barrier_init();
}
// one thread: copies chunks first, first + stride, ... of [src, src + total) to dst through the ring.
// `uses` counts the completed phases of every stage's barrier across calls (phase parity of the next wait).
__device__ __forceinline__ void bulk_stream_copy(BulkRing& r, unsigned int (&uses)[FETCH_STAGES], unsigned char* dst,
                                                 const unsigned char* src, size_t total, int first, int stride) {
  const int nchunks = (int)((total + FETCH_CHUNK - 1) / FETCH_CHUNK);
  const int n_my = first < nchunks ? (nchunks - first + stride - 1) / stride : 0;
  auto chunk_off = [&](int i) { return (size_t)(first + i * stride) * FETCH_CHUNK; };
  auto chunk_bytes = [&](int i) { const size_t o = chunk_off(i); return (uint32_t)(total - o < FETCH_CHUNK ? total - o : FETCH_CHUNK); };
  auto load = [&](int i) {
    uint64_t* bar = reinterpret_cast<uint64_t*>(&r.bar[i % FETCH_STAGES]);
    tma::mbar_expect_tx(bar, chunk_bytes(i));
    tma::bulk_g2s(r.buf[i % FETCH_STAGES], src + chunk_off(i), chunk_bytes(i), bar);
  };
  for (int i = 0; i < FETCH_STAGES && i < n_my; ++i) load(i);
  for (int i = 0; i < n_my; ++i) {
    const int st = i % FETCH_STAGES;
    tma::mbar_wait(reinterpret_cast<uint64_t*>(&r.bar[st]), uses[st] & 1u);
    ++uses[st];
    tma::bulk_s2g(dst + chunk_off(i), r.buf[st], chunk_bytes(i));
    tma::bulk_commit();
    if (i + FETCH_STAGES < n_my) {
      tma::bulk_wait_read<0>();            // the store has drained this stage: refill it
      load(i + FETCH_STAGES);
    }
  }
  tma::bulk_wait<0>();                     // every global write of this thread's bulk groups performed
  asm volatile("fence.proxy.async;" ::: "memory");
}

// Head of the step graph: the frame's images go to pyramid level 0 / the right raw image -- from the staging slot
// when the previous step's prefetch branch already pulled them (stage_seq == this step's sequence number: an
// HBM -> HBM copy), else straight from the source the I/O block names.
// cam_base: grid z = 0 handles camera cam_base, z = 1 camera cam_base + 1.  The head of the step graph fetches the LEFT
// image only (grid z extent 1, cam_base 0); the RIGHT image is needed by keyframes alone (rectification, stereo
// matching: "the right image is not touched by the reference on non-keyframes", SURVEY 8(d)), so it is fetched after
// the keyframe decision by the same kernel with cam_base 1 and the keyframe mode mask (st != null): three frames out of
// four move half the bytes over the host link.  cam 2 is the depth image of an RGB-D context (rows of dc.depth_row bytes,
// dense destination dstR = db.depth), fetched the same way after the decision: only bootstraps and keyframes read it.
__global__ void __launch_bounds__(32) fetch_io_kernel(DevCfg dc, const StepIO* __restrict__ io, unsigned char* __restrict__ dstL,
                                                      unsigned char* __restrict__ dstR, const unsigned char* __restrict__ stage,
                                                      const unsigned long long* __restrict__ stage_seq, int cam_base,
                                                      const StreamState* __restrict__ st, int mode_mask) {
  __shared__ __align__(128) BulkRing ring;
  if (st && !mode_on(st[blockIdx.y].mode, mode_mask)) return;
  const int cam = cam_base + (int)blockIdx.z;
  const bool dep = cam == 2;
  const size_t row = dep ? dc.depth_row : (size_t)dc.W;           // bytes per row
  const bool staged = !dep && stage != nullptr && *stage_seq == io->seq;
  const size_t sp = staged ? row : (size_t)(dep ? io->srcD_pitch : io->src_pitch);
  const unsigned char* src = staged ? stage + ((size_t)cam * dc.B + blockIdx.y) * dc.img_stride
                                    : (dep ? io->srcD : cam ? io->srcR : io->srcL) + (size_t)blockIdx.y * sp * dc.H;
  const size_t dp = dep ? row : (size_t)dc.pitch;                  // destination row pitch
  unsigned char* dst = dep ? dstR + (size_t)blockIdx.y * dc.depth_stride
                           : cam ? dstR + (size_t)blockIdx.y * dc.img_stride : dstL + (size_t)blockIdx.y * dc.pyr_stride;
  const size_t img = row * dc.H;
  if (sp == row && dp == row && ((((size_t)src | (size_t)dst) | img) & 15) == 0) {
    if (threadIdx.x == 0) {
      unsigned int uses[FETCH_STAGES] = {0};
      bulk_ring_init(ring);
      bulk_stream_copy(ring, uses, dst, src, img, blockIdx.x, gridDim.x);
    }
  } else {
    // row pitch or alignment the bulk unit cannot take: plain byte copy by the warp (rare: ROI views)
    for (size_t i = (size_t)blockIdx.x * 32 + threadIdx.x; i < img; i += (size_t)gridDim.x * 32) {
      const size_t y = i / row, x = i - y * row;
      dst[y * dp + x] = src[y * sp + x];
    }
  }
}
// Side branch of the step graph (runs beside the step's kernels): the NEXT frame's images, when that frame is
// already queued, are pulled over the host link into the other staging slot; the last CTA publishes the
// sequence number the next step's head looks for.  next_src* are dense and 16-byte aligned (the host checks).
__global__ void __launch_bounds__(32) prefetch_io_kernel(DevCfg dc, const StepIO* __restrict__ io, unsigned char* __restrict__ stage,
                                                         unsigned long long* __restrict__ stage_seq, unsigned int* counter) {
  __shared__ __align__(128) BulkRing ring;
  const unsigned char* sL = io->next_srcL;
  const unsigned char* sR = io->next_srcR;
  if (!sL || !sR) return;                          // grid-uniform: nobody touches the counter
  const size_t img = (size_t)dc.W * dc.H;
  const unsigned char* src = (blockIdx.z ? sR : sL) + (size_t)blockIdx.y * img;
  unsigned char* dst = stage + ((size_t)blockIdx.z * dc.B + blockIdx.y) * dc.img_stride;
  if (threadIdx.x == 0) {
    unsigned int uses[FETCH_STAGES] = {0};
    bulk_ring_init(ring);
    bulk_stream_copy(ring, uses, dst, src, img, blockIdx.x, gridDim.x);
    __threadfence();
    const unsigned int total = gridDim.x * gridDim.y * gridDim.z;
    if (atomicAdd(counter, 1u) == total - 1) {
      *counter = 0;
      __threadfence();
      *stage_seq = io->seq + 1;
    }
  }
}
// CTAs per image of `bytes` bytes
static int bulk_grid_bytes(size_t bytes) {
  const int nchunks = (int)((bytes + FETCH_CHUNK - 1) / FETCH_CHUNK);
  static const int env_ctas = getenv("KVFE_FETCH_CTAS") ? atoi(getenv("KVFE_FETCH_CTAS")) : 0;   // diagnostic
  // measured on B200, 32 streams x 752x480 (45 chunks): 4 CTAs per image 0.80 ms per pass end to end, 11 CTAs
  // 0.91, 22 CTAs 0.97 -- a few resident warps per image keep the host link busy, more only crowd the SMs
  const int g = env_ctas > 0 ? env_ctas : nchunks / 11;
  return g < 2 ? 2 : (g > 16 ? 16 : g);
}
static int bulk_grid(const DevCfg& dc) { return bulk_grid_bytes((size_t)dc.W * dc.H); }
int launch_fetch_io(const DevCfg& dc, const DevBuf& db, const StepIO* io, int cur_slot, cudaStream_t s) {
  // left image now; the right one after the keyframe decision (launch_fetch_right_io) -- unless the images are equalised
  // (then both are conditioned up front like the reference's data provider does) or there is no right camera
  const int both = dc.equalize && !dc.mono && !dc.rgbd;
  fetch_io_kernel<<<dim3(bulk_grid(dc), dc.B, both ? 2 : 1), 32, 0, s>>>(dc, io, db.pyr[cur_slot] + dc.lvl_off[0], db.right_raw,
                                                                        db.stage_img[cur_slot], db.stage_seq ? db.stage_seq + cur_slot : nullptr,
                                                                        0, nullptr, 0);
  return 1;
}
int launch_fetch_right_io(const DevCfg& dc, const DevBuf& db, const StepIO* io, int cur_slot, int mode_mask, cudaStream_t s) {
  if (dc.mono || dc.rgbd || dc.equalize) return 0;
  fetch_io_kernel<<<dim3(bulk_grid(dc), dc.B, 1), 32, 0, s>>>(dc, io, db.pyr[cur_slot] + dc.lvl_off[0], db.right_raw,
                                                              db.stage_img[cur_slot], db.stage_seq ? db.stage_seq + cur_slot : nullptr,
                                                              1, db.st, mode_mask);
  return 1;
}
// RGB-D: the depth image, after the keyframe decision, for the streams in mode_mask (never equalised, never prefetched)
int launch_fetch_depth_io(const DevCfg& dc, const DevBuf& db, const StepIO* io, int mode_mask, cudaStream_t s) {
  fetch_io_kernel<<<dim3(bulk_grid_bytes(dc.depth_row * dc.H), dc.B, 1), 32, 0, s>>>(dc, io, nullptr, db.depth, nullptr, nullptr, 2,
                                                                                     db.st, mode_mask);
  return 1;
}
int launch_prefetch_io(const DevCfg& dc, const DevBuf& db, const StepIO* io, int cur_slot, unsigned int* counter, cudaStream_t s) {
  prefetch_io_kernel<<<dim3(bulk_grid(dc), dc.B, 2), 32, 0, s>>>(dc, io, db.stage_img[cur_slot ^ 1], db.stage_seq + (cur_slot ^ 1), counter);
  return 1;
}

// Last kernel of a pipeline step: the packets and -- for the streams whose frame became a keyframe -- the
// rectified image pair (part of the output StereoFrame, include/kimera-vio/frontend/StereoFrame.h:71-87) go
// into the mapped host buffers the I/O block names; the last CTA to finish fences and publishes the step's
// sequence number, which is all the dispatcher polls.  CTA 0: packets (only the entries in use), 16-byte
// stores by 128 threads.  CTAs 1..: rectified images, one warp each, bulk copies through the same ring as the
// fetch (HBM -> shared -> host).
__global__ void __launch_bounds__(128) publish_io_kernel(DevCfg dc, DevBuf db, StepIO* io, unsigned int* counter) {
  __shared__ __align__(128) BulkRing ring;
  if (blockIdx.x == 0) {
    if (io->dst_packets) {
      // header, then of every array only the entries in use (a packet's capacity is ~2.3x its typical content)
      const unsigned sz[KVFE_PACKET_ARRAYS] = {4, 4, 8, 4, 8, 24, 4, 4, 4, 4, 4, 4, 8, 24, 4, 4, 8, 8, 8, 8, 24};
      for (int b = 0; b < dc.B; ++b) {
        const unsigned char* src = db.packets + (size_t)b * db.packet_bytes;
        unsigned char* dst = io->dst_packets + (size_t)b * db.packet_bytes;
        const kvfe_packet_header* h = reinterpret_cast<const kvfe_packet_header*>(src);
        const int n = h->n, ns = h->n_smart, nt = h->n_mesh_triangles;
        for (int a = -1; a < KVFE_PACKET_ARRAYS; ++a) {
          const size_t off = a < 0 ? 0 : db.pk_off[a];
          const size_t bytes = a < 0 ? sizeof(kvfe_packet_header) : (size_t)sz[a] * (size_t)(a == 20 ? nt : a >= 16 ? ns : n);
          const size_t n16 = (bytes + 15) / 16;       // arrays start 16-byte aligned and are padded to 16 bytes
          const uint4* s4 = reinterpret_cast<const uint4*>(src + off);
          uint4* d4 = reinterpret_cast<uint4*>(dst + off);
          for (size_t i = threadIdx.x; i < n16; i += blockDim.x) d4[i] = s4[i];
        }
      }
    }
  } else if (io->dst_rectL && io->dst_rectR && !dc.mono && !dc.rgbd) {
    const size_t img = (size_t)dc.W * dc.H;
    const int part = blockIdx.x - 1, nparts = gridDim.x - 1;
    unsigned int uses[FETCH_STAGES] = {0};
    if (threadIdx.x == 0) bulk_ring_init(ring);
    for (int b = 0; b < dc.B; ++b) {
      const int mode = db.st[b].mode;
      if (!(mode == 0 || mode == 2)) continue;
      for (int cam = 0; cam < 2; ++cam) {
        const unsigned char* src = (cam ? db.rectR : db.rectL) + (size_t)b * dc.img_stride;
        unsigned char* dst = (cam ? io->dst_rectR : io->dst_rectL) + (size_t)b * img;
        if (dc.pitch == dc.W && ((((size_t)dst | (size_t)src) | img) & 15) == 0) {
          if (threadIdx.x == 0) bulk_stream_copy(ring, uses, dst, src, img, part, nparts);
        } else {
          for (size_t i = (size_t)part * blockDim.x + threadIdx.x; i < img; i += (size_t)nparts * blockDim.x) {
            const size_t y = i / dc.W, x = i - y * dc.W;
            dst[i] = src[y * dc.pitch + x];
          }
        }
      }
    }
  }
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int done = atomicAdd(counter, 1u);
    if (done == gridDim.x - 1) {
      *counter = 0;
      __threadfence_system();
      io->done_seq = io->seq;
      __threadfence_system();
    }
  }
}
int launch_publish_io(const DevCfg& dc, const DevBuf& db, StepIO* io, unsigned int* counter, cudaStream_t s) {
  publish_io_kernel<<<1 + bulk_grid(dc), 128, 0, s>>>(dc, db, io, counter);
  return 1;
}
// split step graphs (pipeline.cu): the keyframe decision of the (single) stream of a pipeline context goes to the mapped
// I/O block as soon as it exists, so that the dispatcher launches the keyframe kernels only for the frames that need them
__global__ void publish_decision_kernel(DevBuf db, StepIO* io) {
  if (threadIdx.x == 0) {
    io->decided_mode = db.st[0].mode;
    __threadfence_system();
    io->decided_seq = io->seq;
    __threadfence_system();
  }
}
int launch_publish_decision(const DevBuf& db, StepIO* io, cudaStream_t s) {
  publish_decision_kernel<<<1, 32, 0, s>>>(db, io);
  return 1;
}
int launch_finalize(const DevCfg& dc, const DevBuf& db, cudaStream_t s) {
  finalize_kernel<<<dc.B, 256, 0, s>>>(dc, db);
  return 1;
}
