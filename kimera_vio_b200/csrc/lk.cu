// lk.cu -- row a9: cv::calcOpticalFlowPyrLK as called by Tracker::featureTracking
// (reference src/frontend/Tracker.cpp:117-148; winSize 24, maxLevel 4, criteria(COUNT+EPS, 30, 0.1),
// OPTFLOW_USE_INITIAL_FLOW, minEigThreshold 1e-4).
//
// One warp per keypoint, levels maxLevel..0 inside the kernel.  Per level:
//   1. a (win+3)^2 patch of the PREVIOUS image level (BORDER_REFLECT_101 padding semantics) is
//      staged in shared memory; Scharr derivatives are computed from it on the fly (zero outside
//      the image, like the zero-padded derivative buffer of OpenCV) -- no derivative image is ever
//      written to HBM;
//   2. the fixed-point window I / Ix / Iy (14-bit bilinear weights) and the structure tensor are
//      formed; the float accumulations reproduce OpenCV's SIMD128 lane order exactly (bit-exact
//      with cv2 for windows that are a multiple of 8, e.g. the Euroc 24);
//   3. <= maxCount Gauss-Newton iterations, each staging a (win+1)^2 patch of the NEXT image level.
// All float scalar arithmetic follows LKTrackerInvoker's scalar code path operation by operation.
#include <cstdlib>

#include "common.cuh"
#include "tma.cuh"

#define LK_MAX_WIN 32
#define LK_WARPS 4

// per-warp shared-memory carve-up (sizes depend on the runtime window):
//   P (win+3)^2 u8 | J (win+1)^2 u8 | Dx, Dy (win+1)^2 i16 | I, Ix, Iy win^2 i16
struct LkSmem {
  unsigned char* P; unsigned char* J;
  short *Dx, *Dy, *I, *Ix, *Iy;
};
__host__ __device__ inline size_t lk_warp_bytes(int win) {
  size_t a = ((size_t)(win + 3) * (win + 3) + 15) & ~(size_t)15;
  size_t b = ((size_t)(win + 1) * (win + 1) + 15) & ~(size_t)15;
  size_t d = (2 * (size_t)(win + 1) * (win + 1) + 15) & ~(size_t)15;
  size_t w = (2 * (size_t)win * win + 15) & ~(size_t)15;
  return a + b + 2 * d + 3 * w;
}

__device__ __forceinline__ int descale(int x, int n) { return (x + (1 << (n - 1))) >> n; }

// grid (ceil(cap / LK_WARPS), B)
__global__ void __launch_bounds__(LK_WARPS * 32) lk_kernel(DevCfg dc, DevBuf db, int prev_slot, int cur_slot) {
  extern __shared__ __align__(16) unsigned char lk_smem_raw[];
  const int b = blockIdx.y;
  const StreamState& st = db.st[b];
  if (st.mode == 0) return;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int pt = blockIdx.x * LK_WARPS + warp;
  if (pt >= st.n_ref) return;
  LkSmem s;
  {
    const int w_ = dc.win;
    unsigned char* base = lk_smem_raw + (size_t)warp * lk_warp_bytes(w_);
    size_t a = ((size_t)(w_ + 3) * (w_ + 3) + 15) & ~(size_t)15;
    size_t bq = ((size_t)(w_ + 1) * (w_ + 1) + 15) & ~(size_t)15;
    size_t d = (2 * (size_t)(w_ + 1) * (w_ + 1) + 15) & ~(size_t)15;
    size_t ww = (2 * (size_t)w_ * w_ + 15) & ~(size_t)15;
    s.P = base; s.J = base + a;
    s.Dx = reinterpret_cast<short*>(base + a + bq); s.Dy = reinterpret_cast<short*>(base + a + bq + d);
    s.I = reinterpret_cast<short*>(base + a + bq + 2 * d);
    s.Ix = reinterpret_cast<short*>(base + a + bq + 2 * d + ww);
    s.Iy = reinterpret_cast<short*>(base + a + bq + 2 * d + 2 * ww);
  }
  const size_t gi = (size_t)b * dc.cap + pt;
  const unsigned char* prevPyr = db.pyr[prev_slot] + (size_t)b * dc.pyr_stride;
  const unsigned char* nextPyr = db.pyr[cur_slot] + (size_t)b * dc.pyr_stride;
  const int win = dc.win;
  const float halfWin = (win - 1) * 0.5f;
  const float px0 = db.lk_px[gi], py0 = db.lk_py[gi];
  float nx = db.lk_qx[gi], ny = db.lk_qy[gi];     // running nextPts[ptidx]
  bool status = true;
  const int maxLevel = dc.n_levels - 1;
  const float FLT_SCALE = 1.f / (1 << 20);
  const int pw = win + 3, jw = win + 1, dw = win + 1;

  for (int level = maxLevel; level >= 0; --level) {
    const int cols = dc.lvl_w[level], rows = dc.lvl_h[level], pitch = dc.lvl_pitch[level];
    const unsigned char* I = prevPyr + dc.lvl_off[level];
    const unsigned char* Jimg = nextPyr + dc.lvl_off[level];
    const float scl = (float)(1. / (1 << level));
    float ppx = px0 * scl, ppy = py0 * scl;
    if (level == maxLevel) { nx = nx * scl; ny = ny * scl; }   // OPTFLOW_USE_INITIAL_FLOW
    else { nx = nx * 2.f; ny = ny * 2.f; }
    ppx -= halfWin; ppy -= halfWin;
    const int ipx = cv_floor(ppx), ipy = cv_floor(ppy);
    if (ipx < -win || ipx >= cols || ipy < -win || ipy >= rows) {
      if (level == 0) status = false;
      continue;
    }
    // ---- stage prev patch rows ipy-1 .. ipy+win+1, cols ipx-1 .. ipx+win+1 (reflect101 padding)
    for (int i = lane; i < pw * pw; i += 32) {
      int r = i / pw, c = i - r * pw;
      int yy = reflect101(ipy - 1 + r, rows), xx = reflect101(ipx - 1 + c, cols);
      s.P[i] = I[(size_t)yy * pitch + xx];
    }
    __syncwarp();
    // ---- Scharr derivatives at the (win+1)^2 tap positions; zero outside the image
    for (int i = lane; i < dw * dw; i += 32) {
      int r = i / dw, c = i - r * dw;
      int X = ipx + c, Y = ipy + r;
      short dx = 0, dy = 0;
      if (X >= 0 && X < cols && Y >= 0 && Y < rows) {
        const unsigned char* p = s.P + (r + 1) * pw + (c + 1);
        int a00 = p[-pw - 1], a01 = p[-pw], a02 = p[-pw + 1];
        int a10 = p[-1], a12 = p[1];
        int a20 = p[pw - 1], a21 = p[pw], a22 = p[pw + 1];
        dx = (short)(3 * (a02 - a00) + 10 * (a12 - a10) + 3 * (a22 - a20));
        dy = (short)(3 * (a20 - a00) + 10 * (a21 - a01) + 3 * (a22 - a02));
      }
      s.Dx[i] = dx; s.Dy[i] = dy;
    }
    __syncwarp();
    // ---- window of I, Ix, Iy with 14-bit bilinear weights; structure tensor
    float a = ppx - ipx, bb = ppy - ipy;
    int iw00 = cv_round((1.f - a) * (1.f - bb) * (1 << 14));
    int iw01 = cv_round(a * (1.f - bb) * (1 << 14));
    int iw10 = cv_round((1.f - a) * bb * (1 << 14));
    int iw11 = (1 << 14) - iw00 - iw01 - iw10;
    for (int i = lane; i < win * win; i += 32) {
      int y = i / win, x = i - y * win;
      const unsigned char* p = s.P + (y + 1) * pw + (x + 1);
      int ival = descale(p[0] * iw00 + p[1] * iw01 + p[pw] * iw10 + p[pw + 1] * iw11, 14 - 5);
      const short* d = s.Dx + y * dw + x;
      int ixval = descale(d[0] * iw00 + d[1] * iw01 + d[dw] * iw10 + d[dw + 1] * iw11, 14);
      d = s.Dy + y * dw + x;
      int iyval = descale(d[0] * iw00 + d[1] * iw01 + d[dw] * iw10 + d[dw + 1] * iw11, 14);
      s.I[i] = (short)ival; s.Ix[i] = (short)ixval; s.Iy[i] = (short)iyval;
    }
    __syncwarp();
    // Structure tensor with OpenCV's SIMD128 accumulation order (pinned against cv2: scratch probe,
    // 2400/2400 points bit-exact): within each window row, pixels x < win & ~3 go to four float lanes
    // (x -> lane x % 4, sequential float accumulation per lane over the rows), the rest of the row to a
    // scalar float sum; final tail + ((L0 + L2) + (L1 + L3)).  Lanes 0..11 = 3 sums x 4 chains, lanes
    // 12..14 the three tails (zero when win is a multiple of 4).
    float A11, A12, A22;
    {
      float acc = 0.f;
      const int nv = win & ~3;
      if (lane < 15) {
        const int q = lane < 12 ? lane >> 2 : lane - 12, c = lane & 3;
        const short* u = (q == 2) ? s.Iy : s.Ix;
        const short* v = (q == 0) ? s.Ix : s.Iy;
        for (int y = 0; y < win; ++y) {
          const int r = y * win;
          if (lane < 12) { for (int x = c; x < nv; x += 4) acc = acc + (float)((int)u[r + x] * (int)v[r + x]); }
          else { for (int x = nv; x < win; ++x) acc = acc + (float)((int)u[r + x] * (int)v[r + x]); }
        }
      }
      float l2 = __shfl_down_sync(KVFE_FULL_MASK, acc, 2);
      float l1 = __shfl_down_sync(KVFE_FULL_MASK, acc, 1);
      float l3 = __shfl_down_sync(KVFE_FULL_MASK, acc, 3);
      float tot = (acc + l2) + (l1 + l3);          // valid in lanes 0, 4, 8
      A11 = (__shfl_sync(KVFE_FULL_MASK, acc, 12) + __shfl_sync(KVFE_FULL_MASK, tot, 0)) * FLT_SCALE;
      A12 = (__shfl_sync(KVFE_FULL_MASK, acc, 13) + __shfl_sync(KVFE_FULL_MASK, tot, 4)) * FLT_SCALE;
      A22 = (__shfl_sync(KVFE_FULL_MASK, acc, 14) + __shfl_sync(KVFE_FULL_MASK, tot, 8)) * FLT_SCALE;
    }
    float D = A11 * A22 - A12 * A12;
    float minEig = (A22 + A11 - sqrtf((A11 - A22) * (A11 - A22) + 4.f * A12 * A12)) / (float)(2 * win * win);
    if (minEig < dc.min_eig_thr || D < 1.1920929e-07f) {
      if (level == 0) status = false;
      continue;
    }
    D = 1.f / D;
    float qx = nx - halfWin, qy = ny - halfWin;
    float pdx = 0.f, pdy = 0.f;
    for (int j = 0; j < dc.max_iter; ++j) {
      const int iqx = cv_floor(qx), iqy = cv_floor(qy);
      if (iqx < -win || iqx >= cols || iqy < -win || iqy >= rows) {
        if (level == 0) status = false;
        break;
      }
      a = qx - iqx; bb = qy - iqy;
      iw00 = cv_round((1.f - a) * (1.f - bb) * (1 << 14));
      iw01 = cv_round(a * (1.f - bb) * (1 << 14));
      iw10 = cv_round((1.f - a) * bb * (1 << 14));
      iw11 = (1 << 14) - iw00 - iw01 - iw10;
      for (int i = lane; i < jw * jw; i += 32) {
        int r = i / jw, c = i - r * jw;
        int yy = reflect101(iqy + r, rows), xx = reflect101(iqx + c, cols);
        s.J[i] = Jimg[(size_t)yy * pitch + xx];
      }
      __syncwarp();
      // residuals into shared memory (reuses the Dx tap buffer: (win+1)^2 >= win^2 shorts)
      short* diffv = s.Dx;
      for (int i = lane; i < win * win; i += 32) {
        int y = i / win, x = i - y * win;
        const unsigned char* p = s.J + y * jw + x;
        diffv[i] = (short)(descale(p[0] * iw00 + p[1] * iw01 + p[jw] * iw10 + p[jw + 1] * iw11, 14 - 5) - s.I[i]);
      }
      __syncwarp();
      // OpenCV's SIMD128 order for the mismatch vector (pinned against cv2): within each window row, groups
      // of 8 pixels x < win & ~7; chain m in 0..3 accumulates float(int32(d[k]*G[k] + d[k+4]*G[k+4])),
      // k = 8g + m; the rest of the row goes to a scalar float sum; final tail + ((c0 + c2) + (c1 + c3)).
      // Lanes 0..7 = 2 sums x 4 chains, lanes 8..9 the two tails (zero when win is a multiple of 8).
      float b1, b2;
      {
        float acc = 0.f;
        const int nv = win & ~7;
        if (lane < 10) {
          const short* G = (lane < 4 || lane == 8) ? s.Ix : s.Iy;
          const int m = lane & 3;
          for (int y = 0; y < win; ++y) {
            const int r = y * win;
            if (lane < 8) {
              for (int k = r + m; k < r + nv; k += 8)
                acc = acc + (float)((int)diffv[k] * (int)G[k] + (int)diffv[k + 4] * (int)G[k + 4]);
            } else {
              for (int k = r + nv; k < r + win; ++k) acc = acc + (float)((int)diffv[k] * (int)G[k]);
            }
          }
        }
        float l2 = __shfl_down_sync(KVFE_FULL_MASK, acc, 2);
        float l1 = __shfl_down_sync(KVFE_FULL_MASK, acc, 1);
        float l3 = __shfl_down_sync(KVFE_FULL_MASK, acc, 3);
        float tot = (acc + l2) + (l1 + l3);        // valid in lanes 0 and 4
        b1 = (__shfl_sync(KVFE_FULL_MASK, acc, 8) + __shfl_sync(KVFE_FULL_MASK, tot, 0)) * FLT_SCALE;
        b2 = (__shfl_sync(KVFE_FULL_MASK, acc, 9) + __shfl_sync(KVFE_FULL_MASK, tot, 4)) * FLT_SCALE;
      }
      __syncwarp();
      float dxv = (float)((A12 * b2 - A22 * b1) * D);
      float dyv = (float)((A12 * b1 - A11 * b2) * D);
      qx += dxv; qy += dyv;
      nx = qx + halfWin; ny = qy + halfWin;
      if ((double)dxv * (double)dxv + (double)dyv * (double)dyv <= (double)dc.eps2) break;
      if (j > 0 && fabsf(dxv + pdx) < 0.01 && fabsf(dyv + pdy) < 0.01) {
        nx -= dxv * 0.5f; ny -= dyv * 0.5f;
        break;
      }
      pdx = dxv; pdy = dyv;
    }
  }
  if (status) {
    // the error pass of calcOpticalFlowPyrLK (level 0, `err` requested as the reference does,
    // Tracker.cpp:137-146): a FINAL position whose window origin left the image clears the status
    // (the iteration loop only tests the position it starts an iteration from)
    const int fx = cv_floor(nx - halfWin), fy = cv_floor(ny - halfWin);
    if (fx < -win || fx >= dc.lvl_w[0] || fy < -win || fy >= dc.lvl_h[0]) status = false;
  }
  if (lane == 0) {
    db.lk_qx[gi] = nx; db.lk_qy[gi] = ny;
    db.lk_status[gi] = status ? 1 : 0;
  }
}

// ------------------------------------------------------------------------------------------------
// Column-per-lane specialisation for windows that are a multiple of 8 (Euroc: 24): lane x owns
// column x of the window.  Patch columns are loaded one row at a time (a coalesced <=27-byte row per
// instruction), right-hand neighbours come from warp shuffles, the fixed-point window I / Ix / Iy is
// kept in shared memory (conflict-free column access) so that the row loops stay rolled: small code
// (no instruction-cache thrash), few registers, high occupancy.  Arithmetic identical to lk_kernel.
// ------------------------------------------------------------------------------------------------
#define LKC_WARPS 4
#define LKC_CHUNK 6      // window rows per software-pipelined chunk of J loads

template <int WIN>
__global__ void __launch_bounds__(LKC_WARPS * 32) lk_kernel_col(DevCfg dc, DevBuf db, int prev_slot, int cur_slot) {
  constexpr int PW = WIN + 3, TW = WIN + 1;
  static_assert(WIN % LKC_CHUNK == 0 || WIN % 8 == 0, "window must be a multiple of 8");
  __shared__ short sI[LKC_WARPS][WIN * WIN], sIx[LKC_WARPS][WIN * WIN], sIy[LKC_WARPS][WIN * WIN];
  __shared__ float sP[LKC_WARPS][3][WIN * WIN];     // structure-tensor products (xx, xy, yy)
  const int b = blockIdx.y;
  const StreamState& st = db.st[b];
  if (st.mode == 0) return;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int pt = blockIdx.x * LKC_WARPS + warp;
  if (pt >= st.n_ref) return;
  short* wI = sI[warp]; short* wIx = sIx[warp]; short* wIy = sIy[warp];
  float (*wP)[WIN * WIN] = sP[warp];
  const int xl = min(lane, WIN - 1);               // window column of this lane (lanes >= WIN idle copies)
  const size_t gi = (size_t)b * dc.cap + pt;
  const unsigned char* prevPyr = db.pyr[prev_slot] + (size_t)b * dc.pyr_stride;
  const unsigned char* nextPyr = db.pyr[cur_slot] + (size_t)b * dc.pyr_stride;
  const float halfWin = (WIN - 1) * 0.5f;
  const float px0 = db.lk_px[gi], py0 = db.lk_py[gi];
  float nx = db.lk_qx[gi], ny = db.lk_qy[gi];
  bool status = true;
  const int maxLevel = dc.n_levels - 1;
  const float FLT_SCALE = 1.f / (1 << 20);
  const int m4 = lane & 3;

  for (int level = maxLevel; level >= 0; --level) {
    const int cols = dc.lvl_w[level], rows = dc.lvl_h[level], pitch = dc.lvl_pitch[level];
    const unsigned char* I = prevPyr + dc.lvl_off[level];
    const unsigned char* Jimg = nextPyr + dc.lvl_off[level];
    const float scl = (float)(1. / (1 << level));
    float ppx = px0 * scl, ppy = py0 * scl;
    if (level == maxLevel) { nx = nx * scl; ny = ny * scl; }
    else { nx = nx * 2.f; ny = ny * 2.f; }
    ppx -= halfWin; ppy -= halfWin;
    const int ipx = cv_floor(ppx), ipy = cv_floor(ppy);
    if (ipx < -WIN || ipx >= cols || ipy < -WIN || ipy >= rows) {
      if (level == 0) status = false;
      continue;
    }
    float a = ppx - ipx, bb = ppy - ipy;
    int iw00 = cv_round((1.f - a) * (1.f - bb) * (1 << 14));
    int iw01 = cv_round(a * (1.f - bb) * (1 << 14));
    int iw10 = cv_round((1.f - a) * bb * (1 << 14));
    int iw11 = (1 << 14) - iw00 - iw01 - iw10;
    __syncwarp();
    // ---- window of I, Ix, Iy streamed over the (WIN+3) patch rows; structure tensor products on the fly
    {
      const int colx = reflect101(ipx - 1 + min(lane, PW - 1), cols);
      const bool xin = (ipx + lane) >= 0 && (ipx + lane) < cols;
      int C0 = 0, R0 = 0, C1 = 0, R1 = 0;
      int h0 = 0, h1 = 0, s0 = 0, s1 = 0;          // per row: horizontal difference R - L and smoothing 3L + 10C + 3R
      int dxp = 0, dyp = 0, dxpn = 0, dypn = 0;
      // one patch row: L2 = pixel of image row (ipy - 1 + r) at this lane's column
      auto patch_row = [&](const int r, const int L2) {
        const int C2 = __shfl_down_sync(KVFE_FULL_MASK, L2, 1);
        const int R2 = __shfl_down_sync(KVFE_FULL_MASK, L2, 2);
        const int h2 = R2 - L2, s2 = 3 * (L2 + R2) + 10 * C2;
        if (r >= 2) {
          const int d = r - 2;
          // Scharr: dx = [3 10 3]^T (rows) x [-1 0 1] (cols), dy = [-1 0 1]^T x [3 10 3]
          int dx = 3 * (h0 + h2) + 10 * h1;
          int dy = s2 - s0;
          const bool yin = (ipy + d) >= 0 && (ipy + d) < rows;
          if (!(xin && yin)) { dx = 0; dy = 0; }
          const int dxn = __shfl_down_sync(KVFE_FULL_MASK, dx, 1);
          const int dyn = __shfl_down_sync(KVFE_FULL_MASK, dy, 1);
          if (d >= 1) {
            const int y = d - 1;
            const int iv = descale(C0 * iw00 + R0 * iw01 + C1 * iw10 + R1 * iw11, 14 - 5);
            const int ix = descale(dxp * iw00 + dxpn * iw01 + dx * iw10 + dxn * iw11, 14);
            const int iy = descale(dyp * iw00 + dypn * iw01 + dy * iw10 + dyn * iw11, 14);
            if (lane < WIN) {
              const int o = y * WIN + lane;
              wI[o] = (short)iv; wIx[o] = (short)ix; wIy[o] = (short)iy;
              wP[0][o] = (float)(ix * ix); wP[1][o] = (float)(ix * iy); wP[2][o] = (float)(iy * iy);
            }
          }
          dxp = dx; dyp = dy; dxpn = dxn; dypn = dyn;
        }
        h0 = h1; h1 = h2; s0 = s1; s1 = s2;
        C0 = C1; R0 = R1; C1 = C2; R1 = R2;
      };
      if (ipy - 1 >= 0 && ipy - 1 + PW <= rows) {
        // all patch rows inside the image: running 32-bit offset, no reflection
        unsigned int o = (unsigned int)(ipy - 1) * (unsigned int)pitch + (unsigned int)colx;
        int Lnext = I[o];
#pragma unroll 3
        for (int r = 0; r < PW; ++r) {
          const int L2 = Lnext;
          o += (unsigned int)pitch;
          if (r + 1 < PW) Lnext = I[o];                                                 // prefetch next row
          patch_row(r, L2);
        }
      } else {
        int Lnext = I[(size_t)reflect101(ipy - 1, rows) * pitch + colx];
#pragma unroll 3
        for (int r = 0; r < PW; ++r) {
          const int L2 = Lnext;
          if (r + 1 < PW) Lnext = I[(size_t)reflect101(ipy + r, rows) * pitch + colx];   // prefetch next row
          patch_row(r, L2);
        }
      }
    }
    __syncwarp();
    float A11, A12, A22;
    {
      // OpenCV lane c = i % 4, sequential float accumulation; 12 chains (3 sums x 4 lanes) on lanes 0..11
      float acc = 0.f;
      if (lane < 12) {
        const float* P = wP[lane >> 2];
#pragma unroll 8
        for (int i = m4; i < WIN * WIN; i += 4) acc = acc + P[i];
      }
      // (L0 + L2) + (L1 + L3)
      const float tot = (acc + __shfl_down_sync(KVFE_FULL_MASK, acc, 2)) +
                        (__shfl_down_sync(KVFE_FULL_MASK, acc, 1) + __shfl_down_sync(KVFE_FULL_MASK, acc, 3));
      A11 = __shfl_sync(KVFE_FULL_MASK, tot, 0) * FLT_SCALE;
      A12 = __shfl_sync(KVFE_FULL_MASK, tot, 4) * FLT_SCALE;
      A22 = __shfl_sync(KVFE_FULL_MASK, tot, 8) * FLT_SCALE;
    }
    float D = A11 * A22 - A12 * A12;
    float minEig = (A22 + A11 - sqrtf((A11 - A22) * (A11 - A22) + 4.f * A12 * A12)) / (float)(2 * WIN * WIN);
    if (minEig < dc.min_eig_thr || D < 1.1920929e-07f) {
      if (level == 0) status = false;
      continue;
    }
    D = 1.f / D;
    float qx = nx - halfWin, qy = ny - halfWin;
    float pdx = 0.f, pdy = 0.f;
    for (int j = 0; j < dc.max_iter; ++j) {
      const int iqx = cv_floor(qx), iqy = cv_floor(qy);
      if (iqx < -WIN || iqx >= cols || iqy < -WIN || iqy >= rows) {
        if (level == 0) status = false;
        break;
      }
      a = qx - iqx; bb = qy - iqy;
      iw00 = cv_round((1.f - a) * (1.f - bb) * (1 << 14));
      iw01 = cv_round(a * (1.f - bb) * (1 << 14));
      iw10 = cv_round((1.f - a) * bb * (1 << 14));
      iw11 = (1 << 14) - iw00 - iw01 - iw10;
      const int colx = reflect101(iqx + min(lane, TW - 1), cols);
      const bool inner = iqy >= 0 && iqy + TW <= rows;
      float bacc = 0.f;                            // lanes 0..3: b1 chains, lanes 4..7: b2 chains
      const int m8 = lane & 7;
      int jprev, jprevR;
      // LKC_CHUNK window rows whose J pixels (rows y0+1 .. y0+LKC_CHUNK of the patch) were loaded together
      auto consume = [&](const int (&Jr)[LKC_CHUNK], const int y0) {
#pragma unroll
        for (int u = 0; u < LKC_CHUNK; ++u) {
          const int y = y0 + u;
          const int jn = Jr[u];
          const int jnR = __shfl_down_sync(KVFE_FULL_MASK, jn, 1);
          const int diff = descale(jprev * iw00 + jprevR * iw01 + jn * iw10 + jnR * iw11, 14 - 5) - wI[y * WIN + xl];
          jprev = jn; jprevR = jnR;
          const int t1 = diff * wIx[y * WIN + xl], t2 = diff * wIy[y * WIN + xl];
          // pixel pairs (x, x + 4): the Ix pair sum lands on lanes with (x & 4) == 0, the Iy pair sum
          // on lanes with (x & 4) != 0, so that ONE gather shuffle per group feeds both chain sets
          const int s1 = t1 + __shfl_down_sync(KVFE_FULL_MASK, t1, 4);
          const int s2 = t2 + __shfl_up_sync(KVFE_FULL_MASK, t2, 4);
          const float g = (float)((lane & 4) ? s2 : s1);
#pragma unroll
          for (int q = 0; q < WIN / 8; ++q) bacc = bacc + __shfl_sync(KVFE_FULL_MASK, g, m8 + 8 * q);
        }
      };
      if (inner) {
        // patch rows inside the image: running 32-bit offset from the (warp-uniform) level base
        unsigned int o = (unsigned int)iqy * (unsigned int)pitch + (unsigned int)colx;
        jprev = Jimg[o];
        jprevR = __shfl_down_sync(KVFE_FULL_MASK, jprev, 1);
#pragma unroll 1
        for (int y0 = 0; y0 < WIN; y0 += LKC_CHUNK) {
          int Jr[LKC_CHUNK];
#pragma unroll
          for (int u = 0; u < LKC_CHUNK; ++u) { o += (unsigned int)pitch; Jr[u] = Jimg[o]; }
          consume(Jr, y0);
        }
      } else {
        jprev = Jimg[(size_t)reflect101(iqy, rows) * pitch + colx];
        jprevR = __shfl_down_sync(KVFE_FULL_MASK, jprev, 1);
#pragma unroll 1
        for (int y0 = 0; y0 < WIN; y0 += LKC_CHUNK) {
          int Jr[LKC_CHUNK];
#pragma unroll
          for (int u = 0; u < LKC_CHUNK; ++u)
            Jr[u] = Jimg[(size_t)reflect101(iqy + y0 + u + 1, rows) * pitch + colx];
          consume(Jr, y0);
        }
      }
      float b1, b2;
      {
        // per sum: (c0 + c2) + (c1 + c3)
        const float tot = (bacc + __shfl_down_sync(KVFE_FULL_MASK, bacc, 2)) +
                          (__shfl_down_sync(KVFE_FULL_MASK, bacc, 1) + __shfl_down_sync(KVFE_FULL_MASK, bacc, 3));
        b1 = __shfl_sync(KVFE_FULL_MASK, tot, 0) * FLT_SCALE;
        b2 = __shfl_sync(KVFE_FULL_MASK, tot, 4) * FLT_SCALE;
      }
      float dxv = (float)((A12 * b2 - A22 * b1) * D);
      float dyv = (float)((A12 * b1 - A11 * b2) * D);
      qx += dxv; qy += dyv;
      nx = qx + halfWin; ny = qy + halfWin;
      if ((double)dxv * (double)dxv + (double)dyv * (double)dyv <= (double)dc.eps2) break;
      if (j > 0 && fabsf(dxv + pdx) < 0.01 && fabsf(dyv + pdy) < 0.01) {
        nx -= dxv * 0.5f; ny -= dyv * 0.5f;
        break;
      }
      pdx = dxv; pdy = dyv;
    }
  }
  if (status) {
    // the error pass of calcOpticalFlowPyrLK (level 0, `err` requested as the reference does,
    // Tracker.cpp:137-146): a FINAL position whose window origin left the image clears the status
    // (the iteration loop only tests the position it starts an iteration from)
    const int fx = cv_floor(nx - halfWin), fy = cv_floor(ny - halfWin);
    if (fx < -WIN || fx >= dc.lvl_w[0] || fy < -WIN || fy >= dc.lvl_h[0]) status = false;
  }
  if (lane == 0) {
    db.lk_qx[gi] = nx; db.lk_qy[gi] = ny;
    db.lk_status[gi] = status ? 1 : 0;
  }
}

// ------------------------------------------------------------------------------------------------
// TMA-staged specialisation (sm_100a): the same arithmetic as lk_kernel_col, restructured around the
// tensor-memory-accelerator so that no lane ever waits on a global load inside the row loops.
//   * every (keypoint, level) patch is ONE cp.async.bulk.tensor.3d box of 48 x 28 u8 (x origin a multiple of 16) (tensor maps per pyramid
//     slot and level over (x, y, stream), built in kvfe_create): the previous-image box of level L-1 is in
//     flight while level L is processed, the next-image box is issued before the window of its level is
//     built and is re-used by the Gauss-Newton iterations as long as the window stays inside it;
//     BORDER_REFLECT_101 is an index remap into the box (the box is placed so that it holds the reflected
//     rows / columns), out-of-image elements are zero-filled by the unit and never read;
//   * patches that lie inside the image (most of levels 0-2) build the window from U = the bilinear
//     interpolation of the PIXELS (4 multiply-adds) and apply Scharr to U -- integer-exact linearity:
//     sum_w w * Scharr(P) == Scharr(sum_w w * P) -- instead of interpolating I, dx and dy separately (12);
//   * the window lives in shared memory as one 8-byte entry per pixel (I | A << 16, B) with (A, B) = (Ix, Iy)
//     or (Iy, Ix) by lane so that the mismatch pair sums need one shuffle and no select per row; the
//     structure-tensor products of 4 window rows at a time are laid out per accumulation chain, read back
//     with 128-bit loads.
// ------------------------------------------------------------------------------------------------
#define LKT_WARPS 4
#define LKT_BOXW 48                    // the unit needs the innermost box coordinate 16-byte aligned (u8: x % 16 == 0;
                                       // measured on B200: any other x raises "illegal instruction"), so a box is 3 x 16 columns
#define LKT_BOXH 28
#define LKT_BOX_BYTES (LKT_BOXW * LKT_BOXH)
#define LKT_BOX_SMEM 1408              // 1344 rounded up to the 128-byte alignment of a TMA destination
#define LKT_PROD_ROWS 4
#define LKT_PSTR 24                    // floats between the 4 chains of one sum: conflict-free stores ((x & 3) * 24 mod 32 distinct)
#define LKT_SSTR 100                   // floats between the 3 sums
#define LKT_J_SLACK_X 3
#define LKT_J_SLACK_Y 1

struct __align__(128) LktWarp {
  unsigned char ibox[2][LKT_BOX_SMEM];
  unsigned char jbox[LKT_BOX_SMEM];
  int2 win[24 * 24];
  float prod[3 * LKT_SSTR];
  unsigned long long bar[3];
};

// lowest in-image coordinate among reflect101(c0 + k, n), k in [0, nw)
__device__ __forceinline__ int lkt_lo(int c0, int nw, int n) {
  const int c1 = c0 + nw - 1;
  if (c0 < 0) return 0;
  return c1 < n ? c0 : min(c0, 2 * (n - 1) - c1);
}
// does [b0, b0 + extent) hold every in-image coordinate reflect101(c0 + k, n), k in [0, nw)?
__device__ __forceinline__ bool lkt_box_covers(int b0, int extent, int c0, int nw, int n) {
  const int c1 = c0 + nw - 1;
  int lo = max(c0, 0), hi = min(c1, n - 1);
  if (c0 < 0) hi = max(hi, -c0);
  if (c1 >= n) lo = min(lo, 2 * (n - 1) - c1);
  return lo >= b0 && hi <= b0 + extent - 1;
}

struct __align__(64) LktMaps { unsigned char m[2][KVFE_MAX_LEVELS][128]; };      // CUtensorMap is 128 bytes, 64-byte aligned

template <int WIN>
__global__ void __launch_bounds__(LKT_WARPS * 32) lk_kernel_tma(const __grid_constant__ LktMaps maps, DevCfg dc, DevBuf db,
                                                                int prev_slot, int cur_slot) {
  static_assert(WIN == 24, "lane mapping and chain layout are written for the 24-pixel window");
  constexpr int PW = WIN + 3, TW = WIN + 1;
  __shared__ LktWarp sm[LKT_WARPS];
  const int b = blockIdx.y;
  const StreamState& st = db.st[b];
  if (st.mode == 0) return;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int pt = blockIdx.x * LKT_WARPS + warp;
  if (pt >= st.n_ref) return;
  LktWarp& w = sm[warp];
  uint64_t* bars = reinterpret_cast<uint64_t*>(w.bar);
  const char* mapP = reinterpret_cast<const char*>(&maps.m[prev_slot][0][0]);
  const char* mapN = reinterpret_cast<const char*>(&maps.m[cur_slot][0][0]);
  if (lane == 0) {
    tma::mbar_init(&bars[0], 1); tma::mbar_init(&bars[1], 1); tma::mbar_init(&bars[2], 1);
    tma::fence_barrier_init();
  }
  __syncwarp();
  unsigned ph = 0;                                   // bit i: parity of the next completion of barrier i
  auto issue = [&](int bi, unsigned char* dst, const char* map, int x, int y) {
    if (lane == 0) {
      tma::mbar_expect_tx(&bars[bi], LKT_BOX_BYTES);
      tma::tensor_g2s_3d(dst, map, x, y, b, &bars[bi]);
    }
  };
  auto wait = [&](int bi) {
    tma::mbar_wait(&bars[bi], (ph >> bi) & 1u);
    ph ^= 1u << bi;
  };
  const int xl = min(lane, WIN - 1);
  const size_t gi = (size_t)b * dc.cap + pt;
  const float halfWin = (WIN - 1) * 0.5f;
  const float px0 = db.lk_px[gi], py0 = db.lk_py[gi];
  float nx = db.lk_qx[gi], ny = db.lk_qy[gi];
  bool status = true;
  const int maxLevel = dc.n_levels - 1;
  const float FLT_SCALE = 1.f / (1 << 20);
  const int m4 = lane & 3, m8 = lane & 7;
  const bool hi4 = (lane & 4) != 0;

  // previous-image box of a level: window origin, validity and box origin
  auto prev_geom = [&](int level, int& ipx, int& ipy, float& ppx, float& ppy) -> bool {
    const float scl = (float)(1. / (1 << level));
    ppx = px0 * scl - halfWin; ppy = py0 * scl - halfWin;
    ipx = cv_floor(ppx); ipy = cv_floor(ppy);
    return !(ipx < -WIN || ipx >= dc.lvl_w[level] || ipy < -WIN || ipy >= dc.lvl_h[level]);
  };
  int i_bx = 0, i_by = 0;                            // origin of the previous-image box of the current level
  {
    int ipx, ipy; float fx, fy;
    if (prev_geom(maxLevel, ipx, ipy, fx, fy)) {
      i_bx = lkt_lo(ipx - 1, PW, dc.lvl_w[maxLevel]) & ~15;
      i_by = lkt_lo(ipy - 1, PW, dc.lvl_h[maxLevel]);
      issue(maxLevel & 1, w.ibox[maxLevel & 1], mapP + maxLevel * 128, i_bx, i_by);
    }
  }
  int j_state = 0;                                   // next-image box: 0 none, 1 in flight, 2 landed
  int j_bx = 0, j_by = 0;

  for (int level = maxLevel; level >= 0; --level) {
    const int cols = dc.lvl_w[level], rows = dc.lvl_h[level];
    __syncwarp();
    if (level == maxLevel) { const float scl = (float)(1. / (1 << level)); nx = nx * scl; ny = ny * scl; }
    else { nx = nx * 2.f; ny = ny * 2.f; }
    int ipx, ipy; float ppx, ppy;
    const bool okI = prev_geom(level, ipx, ipy, ppx, ppy);
    const int cur_bx = i_bx, cur_by = i_by;
    // previous-image box of the next (finer) level: in flight while this level is processed
    if (level > 0) {
      int npx, npy; float fx, fy;
      if (prev_geom(level - 1, npx, npy, fx, fy)) {
        i_bx = lkt_lo(npx - 1, PW, dc.lvl_w[level - 1]) & ~15;
        i_by = lkt_lo(npy - 1, PW, dc.lvl_h[level - 1]);
        __syncwarp();
        issue((level - 1) & 1, w.ibox[(level - 1) & 1], mapP + (level - 1) * 128, i_bx, i_by);
      }
    }
    if (!okI) {
      if (level == 0) status = false;
      continue;
    }
    // next-image box for the first iteration of this level
    if (j_state == 1) wait(2);
    j_state = 0;
    {
      const int iqx = cv_floor(nx - halfWin), iqy = cv_floor(ny - halfWin);
      if (!(iqx < -WIN || iqx >= cols || iqy < -WIN || iqy >= rows)) {
        j_bx = (lkt_lo(iqx, TW, cols) - LKT_J_SLACK_X) & ~15;
        j_by = lkt_lo(iqy, TW, rows) - LKT_J_SLACK_Y;
        __syncwarp();
        issue(2, w.jbox, mapN + level * 128, j_bx, j_by);
        j_state = 1;
      }
    }
    float a = ppx - ipx, bb = ppy - ipy;
    int iw00 = cv_round((1.f - a) * (1.f - bb) * (1 << 14));
    int iw01 = cv_round(a * (1.f - bb) * (1 << 14));
    int iw10 = cv_round((1.f - a) * bb * (1 << 14));
    int iw11 = (1 << 14) - iw00 - iw01 - iw10;
    wait(level & 1);
    const unsigned char* IB = w.ibox[level & 1];
    float acc = 0.f;                                 // lanes 0..11: structure-tensor chain (sum lane >> 2, chain lane & 3)
    auto store_px = [&](const int y, const int iv, const int ix, const int iy) {
      if (lane < WIN) {
        const int A = hi4 ? iy : ix, Bv = hi4 ? ix : iy;
        w.win[y * WIN + lane] = make_int2((iv & 0xffff) | (A << 16), Bv);
        float* pp = w.prod + m4 * LKT_PSTR + (y & (LKT_PROD_ROWS - 1)) * (WIN / 4) + (lane >> 2);
        pp[0] = (float)(ix * ix); pp[LKT_SSTR] = (float)(ix * iy); pp[2 * LKT_SSTR] = (float)(iy * iy);
      }
    };
    auto chain_rows = [&]() {
      // OpenCV lane c = i % 4, sequential float accumulation; 12 chains (3 sums x 4 lanes) on lanes 0..11
      __syncwarp();
      if (lane < 12) {
        const float4* q = reinterpret_cast<const float4*>(w.prod + (lane >> 2) * LKT_SSTR + m4 * LKT_PSTR);
#pragma unroll
        for (int k = 0; k < LKT_PROD_ROWS * (WIN / 4) / 4; ++k) {
          const float4 v = q[k];
          acc = acc + v.x; acc = acc + v.y; acc = acc + v.z; acc = acc + v.w;
        }
      }
      __syncwarp();
    };
    const bool interior = ipx >= 1 && ipy >= 1 && ipx + WIN + 1 <= cols - 1 && ipy + WIN + 1 <= rows - 1;
    if (interior) {
      // patch row r, column c at IB[(ipy - 1 - cur_by + r) * LKT_BOXW + (ipx - 1 - cur_bx + c)]
      const unsigned char* col = IB + (ipy - 1 - cur_by) * LKT_BOXW + (ipx - 1 - cur_bx) + min(lane, PW - 1);
      int Lp = 0, LpR = 0, H0 = 0, H1 = 0, S0 = 0, S1 = 0, UcPrev = 0;
      auto row_fast = [&](const int r) {
        const int L = col[r * LKT_BOXW];
        const int LR = __shfl_down_sync(KVFE_FULL_MASK, L, 1);
        if (r >= 1) {
          const int U = Lp * iw00 + LpR * iw01 + L * iw10 + LR * iw11;       // U(r - 1, lane), exact
          const int Uc = __shfl_down_sync(KVFE_FULL_MASK, U, 1);
          const int Ur = __shfl_down_sync(KVFE_FULL_MASK, U, 2);
          const int H2 = Ur - U, S2 = 3 * (U + Ur) + 10 * Uc;
          if (r >= 3) store_px(r - 3, descale(UcPrev, 14 - 5), descale(3 * (H0 + H2) + 10 * H1, 14), descale(S2 - S0, 14));
          H0 = H1; H1 = H2; S0 = S1; S1 = S2; UcPrev = Uc;
        }
        Lp = L; LpR = LR;
      };
      row_fast(0); row_fast(1); row_fast(2);
#pragma unroll 1
      for (int c = 0; c < WIN / LKT_PROD_ROWS; ++c) {
#pragma unroll 4
        for (int u = 0; u < LKT_PROD_ROWS; ++u) row_fast(3 + c * LKT_PROD_ROWS + u);
        chain_rows();
      }
    } else {
      const int cidx = clampi(reflect101(ipx - 1 + min(lane, PW - 1), cols) - cur_bx, 0, LKT_BOXW - 1);
      const bool xin = (ipx + lane) >= 0 && (ipx + lane) < cols;
      int C0 = 0, R0 = 0, C1 = 0, R1 = 0;
      int h0 = 0, h1 = 0, s0 = 0, s1 = 0;
      int dxp = 0, dyp = 0, dxpn = 0, dypn = 0;
      auto row_border = [&](const int r) {
        const int ridx = clampi(reflect101(ipy - 1 + r, rows) - cur_by, 0, LKT_BOXH - 1);
        const int L2 = IB[ridx * LKT_BOXW + cidx];
        const int C2 = __shfl_down_sync(KVFE_FULL_MASK, L2, 1);
        const int R2 = __shfl_down_sync(KVFE_FULL_MASK, L2, 2);
        const int h2 = R2 - L2, s2 = 3 * (L2 + R2) + 10 * C2;
        if (r >= 2) {
          const int d = r - 2;
          int dx = 3 * (h0 + h2) + 10 * h1;
          int dy = s2 - s0;
          const bool yin = (ipy + d) >= 0 && (ipy + d) < rows;
          if (!(xin && yin)) { dx = 0; dy = 0; }
          const int dxn = __shfl_down_sync(KVFE_FULL_MASK, dx, 1);
          const int dyn = __shfl_down_sync(KVFE_FULL_MASK, dy, 1);
          if (d >= 1)
            store_px(d - 1, descale(C0 * iw00 + R0 * iw01 + C1 * iw10 + R1 * iw11, 14 - 5),
                     descale(dxp * iw00 + dxpn * iw01 + dx * iw10 + dxn * iw11, 14),
                     descale(dyp * iw00 + dypn * iw01 + dy * iw10 + dyn * iw11, 14));
          dxp = dx; dyp = dy; dxpn = dxn; dypn = dyn;
        }
        h0 = h1; h1 = h2; s0 = s1; s1 = s2;
        C0 = C1; R0 = R1; C1 = C2; R1 = R2;
      };
      row_border(0); row_border(1); row_border(2);
#pragma unroll 1
      for (int c = 0; c < WIN / LKT_PROD_ROWS; ++c) {
#pragma unroll 2
        for (int u = 0; u < LKT_PROD_ROWS; ++u) row_border(3 + c * LKT_PROD_ROWS + u);
        chain_rows();
      }
    }
    float A11, A12, A22;
    {
      // (L0 + L2) + (L1 + L3)
      const float tot = (acc + __shfl_down_sync(KVFE_FULL_MASK, acc, 2)) +
                        (__shfl_down_sync(KVFE_FULL_MASK, acc, 1) + __shfl_down_sync(KVFE_FULL_MASK, acc, 3));
      A11 = __shfl_sync(KVFE_FULL_MASK, tot, 0) * FLT_SCALE;
      A12 = __shfl_sync(KVFE_FULL_MASK, tot, 4) * FLT_SCALE;
      A22 = __shfl_sync(KVFE_FULL_MASK, tot, 8) * FLT_SCALE;
    }
    float D = A11 * A22 - A12 * A12;
    float minEig = (A22 + A11 - sqrtf((A11 - A22) * (A11 - A22) + 4.f * A12 * A12)) / (float)(2 * WIN * WIN);
    if (minEig < dc.min_eig_thr || D < 1.1920929e-07f) {
      if (level == 0) status = false;
      continue;
    }
    D = 1.f / D;
    float qx = nx - halfWin, qy = ny - halfWin;
    float pdx = 0.f, pdy = 0.f;
    for (int j = 0; j < dc.max_iter; ++j) {
      const int iqx = cv_floor(qx), iqy = cv_floor(qy);
      if (iqx < -WIN || iqx >= cols || iqy < -WIN || iqy >= rows) {
        if (level == 0) status = false;
        break;
      }
      a = qx - iqx; bb = qy - iqy;
      iw00 = cv_round((1.f - a) * (1.f - bb) * (1 << 14));
      iw01 = cv_round(a * (1.f - bb) * (1 << 14));
      iw10 = cv_round((1.f - a) * bb * (1 << 14));
      iw11 = (1 << 14) - iw00 - iw01 - iw10;
      if (j_state == 1) { wait(2); j_state = 2; }
      if (!(j_state == 2 && lkt_box_covers(j_bx, LKT_BOXW, iqx, TW, cols) && lkt_box_covers(j_by, LKT_BOXH, iqy, TW, rows))) {
        j_bx = (lkt_lo(iqx, TW, cols) - LKT_J_SLACK_X) & ~15;
        j_by = lkt_lo(iqy, TW, rows) - LKT_J_SLACK_Y;
        __syncwarp();
        issue(2, w.jbox, mapN + level * 128, j_bx, j_by);
        wait(2);
        j_state = 2;
      }
      const unsigned char* JB = w.jbox;
      const int jc = clampi(reflect101(iqx + min(lane, TW - 1), cols) - j_bx, 0, LKT_BOXW - 1);
      const bool inner = iqx >= 0 && iqy >= 0 && iqx + TW <= cols && iqy + TW <= rows;
      float bacc = 0.f;                            // lanes 0..3: b1 chains, lanes 4..7: b2 chains
      int jprev, jprevR;
      auto row_iter = [&](const int y, const int jn) {
        const int jnR = __shfl_down_sync(KVFE_FULL_MASK, jn, 1);
        const int2 e = w.win[y * WIN + xl];
        const int diff = descale(jprev * iw00 + jprevR * iw01 + jn * iw10 + jnR * iw11, 14 - 5) - (int)(short)(e.x & 0xffff);
        jprev = jn; jprevR = jnR;
        // own = the product whose pair sum lands on this lane (Ix on lanes with (x & 4) == 0, Iy on the others),
        // sent = the product the partner lane x ^ 4 needs: ONE exchange per row feeds both chain sets
        const int own = diff * (e.x >> 16), sent = diff * e.y;
        const float g = (float)(own + __shfl_xor_sync(KVFE_FULL_MASK, sent, 4));
#pragma unroll
        for (int q = 0; q < WIN / 8; ++q) bacc = bacc + __shfl_sync(KVFE_FULL_MASK, g, m8 + 8 * q);
      };
      if (inner) {
        const unsigned char* p = JB + (iqy - j_by) * LKT_BOXW + jc;
        jprev = p[0];
        jprevR = __shfl_down_sync(KVFE_FULL_MASK, jprev, 1);
#pragma unroll 6
        for (int y = 0; y < WIN; ++y) row_iter(y, p[(y + 1) * LKT_BOXW]);
      } else {
        jprev = JB[clampi(reflect101(iqy, rows) - j_by, 0, LKT_BOXH - 1) * LKT_BOXW + jc];
        jprevR = __shfl_down_sync(KVFE_FULL_MASK, jprev, 1);
#pragma unroll 2
        for (int y = 0; y < WIN; ++y)
          row_iter(y, JB[clampi(reflect101(iqy + y + 1, rows) - j_by, 0, LKT_BOXH - 1) * LKT_BOXW + jc]);
      }
      float b1, b2;
      {
        // per sum: (c0 + c2) + (c1 + c3)
        const float tot = (bacc + __shfl_down_sync(KVFE_FULL_MASK, bacc, 2)) +
                          (__shfl_down_sync(KVFE_FULL_MASK, bacc, 1) + __shfl_down_sync(KVFE_FULL_MASK, bacc, 3));
        b1 = __shfl_sync(KVFE_FULL_MASK, tot, 0) * FLT_SCALE;
        b2 = __shfl_sync(KVFE_FULL_MASK, tot, 4) * FLT_SCALE;
      }
      float dxv = (float)((A12 * b2 - A22 * b1) * D);
      float dyv = (float)((A12 * b1 - A11 * b2) * D);
      qx += dxv; qy += dyv;
      nx = qx + halfWin; ny = qy + halfWin;
      if ((double)dxv * (double)dxv + (double)dyv * (double)dyv <= (double)dc.eps2) break;
      if (j > 0 && fabsf(dxv + pdx) < 0.01 && fabsf(dyv + pdy) < 0.01) {
        nx -= dxv * 0.5f; ny -= dyv * 0.5f;
        break;
      }
      pdx = dxv; pdy = dyv;
    }
  }
  if (j_state == 1) wait(2);                         // nothing may land in this CTA's shared memory after it exits
  if (status) {
    const int fx = cv_floor(nx - halfWin), fy = cv_floor(ny - halfWin);
    if (fx < -WIN || fx >= dc.lvl_w[0] || fy < -WIN || fy >= dc.lvl_h[0]) status = false;
  }
  if (lane == 0) {
    db.lk_qx[gi] = nx; db.lk_qy[gi] = ny;
    db.lk_status[gi] = status ? 1 : 0;
  }
}

int launch_lk(const DevCfg& dc, const DevBuf& db, int prev_slot, int cur_slot, cudaStream_t s) {
  // the TMA kernel needs the tensor maps (kvfe_create) and single-bounce reflection at the coarsest level
  static const int lk_mode = getenv("KVFE_LK") ? atoi(getenv("KVFE_LK")) : 2;      // diagnostic: 1 = lk_kernel_col
  const int top = dc.n_levels - 1;
  if (dc.win == 24 && db.lk_tmaps && lk_mode == 2 && dc.lvl_w[top] >= 28 && dc.lvl_h[top] >= 28) {
    lk_kernel_tma<24><<<dim3((dc.cap + LKT_WARPS - 1) / LKT_WARPS, dc.B), LKT_WARPS * 32, 0, s>>>(
        *reinterpret_cast<const LktMaps*>(db.lk_tmaps), dc, db, prev_slot, cur_slot);
    return 1;
  }
  dim3 gridc((dc.cap + LKC_WARPS - 1) / LKC_WARPS, dc.B);
  if (dc.win == 24) { lk_kernel_col<24><<<gridc, LKC_WARPS * 32, 0, s>>>(dc, db, prev_slot, cur_slot); return 1; }
  size_t sm = LK_WARPS * lk_warp_bytes(dc.win);
  static size_t attr = 0;
  if (sm > 48 * 1024 && sm > attr) {
    cudaFuncSetAttribute(lk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    attr = sm;
  }
  lk_kernel<<<dim3((dc.cap + LK_WARPS - 1) / LK_WARPS, dc.B), LK_WARPS * 32, sm, s>>>(dc, db, prev_slot, cur_slot);
  return 1;
}
