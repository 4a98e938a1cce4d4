// gftt.cu -- row a3: cv::goodFeaturesToTrack as called by FeatureDetector::rawFeatureDetection
// (reference src/frontend/feature-detector/FeatureDetector.cpp:165-203, GFTTDetector :71-82).
//
//   mask     : 255 image minus filled circles of radius min_distance at every keypoint with a
//              valid landmark (FeatureDetector.cpp:185-203; cv::circle raster, App. A.2)
//   response : cv::cornerMinEigenVal(blockSize 3, ksize 3, BORDER_REFLECT_101), bit-exact:
//              Sobel with OpenCV's FMA op-order, f32 products, 3-tap f64 row sums and the
//              HISTORY-DEPENDENT f64 running column sum of cv::boxFilter (one lane per column,
//              marching down the rows), min-eigenvalue formula in f32.
//   select   : max over mask, threshold (quality * max), 3x3 non-max ("== dilate"), sort by
//              (value desc, address desc), greedy min-distance on a cell grid (parallel fixed
//              point that reproduces the sequential result), stop at maxCorners.
//
// HBM traffic per keyframe image: image 1 B/px (L2 hits for the 3-row window), mask 1 B/px write
// + read, response 4 B/px write + 9 reads served by L1/L2.  Non-compulsory (SURVEY 8(d)).
#include <cstdio>
#include <cstdlib>

#include "common.cuh"

#define GREEDY_TOPK 12288        // candidates the first selection pass looks at (top-K prefilter)
#define GREEDY_SEL_CAP 16384
#define CAND_HIST_BINS 2048

// ------------------------------------------------------------------------------------------------
// mask
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) mask_fill_kernel(DevCfg dc, unsigned char* __restrict__ mask,
                                                        const StreamState* __restrict__ st, int mode_mask) {
  const int b = blockIdx.y;
  if (st && !mode_on(st[b].mode, mode_mask)) return;
  uint4* p = reinterpret_cast<uint4*>(mask + (size_t)b * dc.img_stride);
  size_t n16 = dc.img_stride / 16;
  const uint4 v = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x)
    p[i] = v;
}

// grid (ceil(cap / 8), B), one warp per keypoint; hw[dy + r] = half width of the raster row
__global__ void __launch_bounds__(256) mask_circles_kernel(DevCfg dc, DevBuf db, const int* __restrict__ hw, int r,
                                                           int mode_mask) {
  const int b = blockIdx.y;
  const StreamState& s = db.st[b];
  if (!mode_on(s.mode, mode_mask)) return;
  const int fs = b * 3 + s.slot_k;
  const int n = db.fr.n[fs];
  unsigned char* m = db.mask + (size_t)b * dc.img_stride;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int i = blockIdx.x * 8 + warp;
  if (i >= n) return;
  size_t k = (size_t)fs * dc.cap + i;
  if (db.fr.lmk[k] == -1) return;
  // cv::Point(Point2f): saturate_cast<int>(float) == cvRound
  int cx = cv_round(db.fr.kx[k]), cy = cv_round(db.fr.ky[k]);
  for (int dy = -r; dy <= r; ++dy) {
    int y = cy + dy;
    if (y < 0 || y >= dc.H) continue;
    int h = hw[dy + r];
    int xa = max(cx - h, 0), xb = min(cx + h, dc.W - 1);
    for (int x = xa + lane; x <= xb; x += 32) m[(size_t)y * dc.pitch + x] = 0;
  }
}

// ------------------------------------------------------------------------------------------------
// response map
// ------------------------------------------------------------------------------------------------
struct RT { float r, t; };

__device__ __forceinline__ RT rt_from(float im, float i0, float ip, float s, float s2, bool tail) {
  RT o;
  o.r = ip - im;                                   // exact
  if (!tail) o.t = fmaf(ip, s, fmaf(i0, s2, s * im));
  else o.t = (s * im + s2 * i0) + s * ip;          // host scalar loop tail: no FMA
  return o;
}

#define MINEIG_ROWS 32     // rows staged per batch
#define MINEIG_TW 48       // staged tile width in bytes (12 aligned words >= 2 + 34 + 3)

// grid (ceil(ngroups/4), B); block 128 = 4 warps, each warp owns 30 output columns (+2 halo lanes).
// Each batch of 32 image rows (and the 32 mask rows of the outputs) is first staged into shared
// memory with one row per lane (12 independent 32-bit loads per lane in flight -> the DRAM/L2 latency
// is paid once per batch instead of once per row), then the warp marches down the staged rows.
__global__ void __launch_bounds__(128) mineig_kernel(DevCfg dc, DevBuf db, const unsigned char* __restrict__ imgs,
                                                     size_t img_stride, int mode_mask, int use_mask) {
  __shared__ __align__(16) unsigned char tile[4][MINEIG_ROWS][MINEIG_TW];
  __shared__ __align__(16) unsigned char mtile[4][MINEIG_ROWS][MINEIG_TW];
  const int b = blockIdx.y;
  if (!mode_on(db.st[b].mode, mode_mask)) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int group = blockIdx.x * 4 + warp;
  const int x0 = group * 30;
  const int W = dc.W, H = dc.H;
  if (x0 >= W) return;
  const unsigned char* img = imgs + (size_t)b * img_stride;
  const unsigned char* msk = db.mask + (size_t)b * dc.img_stride;
  float* eig = db.eig + (size_t)b * W * H;
  const int cx = x0 - 1 + lane;                 // lanes 0 and 31 are halo
  int c = reflect101(cx, W);
  c = clampi(c, 0, W - 1);                      // lanes beyond the reflected border are inactive
  const int cm = reflect101(c - 1, W), cp = reflect101(c + 1, W);
  const bool writer = lane >= 1 && lane <= 30 && cx < W;
  const float s = (float)(1.0 / 3060.0), s2 = 2.0f * s;
  const bool tail = dc.sobel_tail_start >= 0 && c >= dc.sobel_tail_start;
  const int pitch = dc.pitch;                   // multiple of 16, rows are 16-byte aligned
  const int xs = max(x0 - 2, 0) & ~3;           // tile origin (aligned); covers [x0-2, x0+32]
  // offsets into the staged tile (lanes past the reflected border are inactive: clamp them)
  const int oc = clampi(c - xs, 0, MINEIG_TW - 1), om = clampi(cm - xs, 0, MINEIG_TW - 1),
            op = clampi(cp - xs, 0, MINEIG_TW - 1), ox = clampi(cx - xs, 0, MINEIG_TW - 1);
  unsigned char (*T)[MINEIG_TW] = tile[warp];
  unsigned char (*M)[MINEIG_TW] = mtile[warp];

  RT a, m;
  {
    const unsigned char* r1 = img + (size_t)reflect101(-1, H) * pitch;
    a = rt_from((float)r1[cm], (float)r1[c], (float)r1[cp], s, s2, tail);       // row p-1
    m = rt_from((float)img[cm], (float)img[c], (float)img[cp], s, s2, tail);    // row p
  }
  double sum0 = 0, sum1 = 0, sum2 = 0;             // running column sums (xx, xy, yy)
  double rm2_0 = 0, rm2_1 = 0, rm2_2 = 0;          // R(p-2)
  double rm1_0 = 0, rm1_1 = 0, rm1_2 = 0;          // R(p-1)
  float vmax = -INFINITY;

  for (int p0 = 0; p0 <= H; p0 += MINEIG_ROWS) {
    // ---- stage: lane u loads image row reflect(p0+u+1) and mask row (p0+u-1), 12 words each
    {
      const int p = p0 + lane;
      const int yr = reflect101(min(p + 1, H), H);
      const unsigned int* src = reinterpret_cast<const unsigned int*>(img + (size_t)yr * pitch + xs);
      const int ym = clampi(p - 1, 0, H - 1);
      const unsigned int* msrc = reinterpret_cast<const unsigned int*>(msk + (size_t)ym * pitch + xs);
      const int nw = min(MINEIG_TW / 4, (pitch - xs) / 4);
      unsigned int v[MINEIG_TW / 4], w[MINEIG_TW / 4];
#pragma unroll
      for (int q = 0; q < MINEIG_TW / 4; ++q) {
        v[q] = (q < nw) ? src[q] : 0u;
        w[q] = (use_mask && q < nw) ? msrc[q] : 0xffffffffu;
      }
      __syncwarp();
#pragma unroll
      for (int q = 0; q < MINEIG_TW / 4; ++q) {
        reinterpret_cast<unsigned int*>(T[lane])[q] = v[q];
        reinterpret_cast<unsigned int*>(M[lane])[q] = w[q];
      }
      __syncwarp();
    }
#pragma unroll 4
    for (int u = 0; u < MINEIG_ROWS; ++u) {
      const int p = p0 + u;
      if (p > H) break;
      double r0, r1, r2;
      if (p < H) {
        RT n = rt_from((float)T[u][om], (float)T[u][oc], (float)T[u][op], s, s2, tail);   // row p+1
        // cv::Sobel column pass: Dx = fma(r(y-1) + r(y+1), s, (2s) * r(y)); Dy = t(y+1) - t(y-1)
        float dx = fmaf(a.r + n.r, s, s2 * m.r);
        float dy = n.t - a.t;
        float pxx = dx * dx, pxy = dx * dy, pyy = dy * dy;
        // RowSum<float,double>, ksize 3: (S[x-1] + S[x]) + S[x+1]
        float l0 = __shfl_up_sync(KVFE_FULL_MASK, pxx, 1), g0 = __shfl_down_sync(KVFE_FULL_MASK, pxx, 1);
        float l1 = __shfl_up_sync(KVFE_FULL_MASK, pxy, 1), g1 = __shfl_down_sync(KVFE_FULL_MASK, pxy, 1);
        float l2 = __shfl_up_sync(KVFE_FULL_MASK, pyy, 1), g2 = __shfl_down_sync(KVFE_FULL_MASK, pyy, 1);
        r0 = ((double)l0 + (double)pxx) + (double)g0;
        r1 = ((double)l1 + (double)pxy) + (double)g1;
        r2 = ((double)l2 + (double)pyy) + (double)g2;
        a = m;
        m = n;
      } else {
        r0 = rm2_0; r1 = rm2_1; r2 = rm2_2;            // R(H) = R(H-2) (reflect)
      }
      if (p == 1) {                                    // ColumnSum init: SUM = (0 + R(-1)) + R(0), R(-1) = R(1)
        sum0 = (0.0 + r0) + rm1_0;
        sum1 = (0.0 + r1) + rm1_1;
        sum2 = (0.0 + r2) + rm1_2;
      }
      if (p >= 1) {
        const int y = p - 1;
        // s0 = SUM + R(y+1); out = (float)s0; SUM = s0 - R(y-1)   (R(-1) = R(1))
        double s0 = sum0 + r0, s1 = sum1 + r1, s2d = sum2 + r2;
        double o0 = (y == 0) ? r0 : rm2_0, o1 = (y == 0) ? r1 : rm2_1, o2 = (y == 0) ? r2 : rm2_2;
        sum0 = s0 - o0; sum1 = s1 - o1; sum2 = s2d - o2;
        if (writer) {
          float A = (float)s0 * 0.5f, Bv = (float)s1, C = (float)s2d * 0.5f;
          float e = (A + C) - sqrtf((A - C) * (A - C) + Bv * Bv);
          eig[(size_t)y * W + cx] = e;
          if (M[u][ox]) vmax = fmaxf(vmax, e);
        }
      }
      rm2_0 = rm1_0; rm2_1 = rm1_1; rm2_2 = rm1_2;
      rm1_0 = r0; rm1_1 = r1; rm1_2 = r2;
    }
    __syncwarp();
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) vmax = fmaxf(vmax, __shfl_xor_sync(KVFE_FULL_MASK, vmax, o));
  if (lane == 0 && vmax > -INFINITY) atomicMax(&db.eig_max[b], f2ord(vmax));
}

// ------------------------------------------------------------------------------------------------
// Response map, warp-specialised: the same arithmetic as mineig_kernel, with the row-parallel part (Sobel,
// products, f64 row sums) taken off the serial column scan.  One CTA per stripe of 30 output columns:
//   warps 0..2  producers: chunks of 8 rows (chunk c -> warp c % 3); per row the three f64 row sums R(p) of the
//               stripe go into a 32-row shared-memory ring;
//   warp 3      scanner: the history-dependent running column sums (2 dependent f64 adds per sum and row) and
//               nothing else; the sums of every output row go into a second ring as floats;
//   warps 4..7  finishers (chunk k -> warp k % 4): min-eigenvalue formula, store, masked maximum.
// The warp that carries the serial chain executes ~20 instructions per row instead of ~120 interleaved with the
// image loads.  Hand-over through shared-memory sequence numbers per 8-row chunk (ready / scanned / finished).
// ------------------------------------------------------------------------------------------------
#define ME_RING 32
#define ME_CHUNK 8
#define ME_PRODUCERS 3
#define ME_FINISHERS 4
#define ME_SLOTS (ME_RING / ME_CHUNK)
struct MeRing {
  double r0[ME_RING][32], r1[ME_RING][32], r2[ME_RING][32];   // producers -> scanner: f64 row sums R(p)
  float s0[ME_RING][32], s1[ME_RING][32], s2[ME_RING][32];    // scanner -> finishers: (float) column sums of output row y
  int ready[ME_SLOTS];                // chunk index + 1 once the chunk's R rows are in the ring
  int scanned[ME_SLOTS];              // chunk index + 1 once the chunk's column sums are in the ring
  int finished[ME_SLOTS];             // chunk index + 1 once a finisher is done with the chunk's column sums
  int cons_row;                       // R rows the scanner is done with
};

__global__ void __launch_bounds__(32 * (ME_PRODUCERS + 1 + ME_FINISHERS))
mineig_pipe_kernel(DevCfg dc, DevBuf db, const unsigned char* __restrict__ imgs, size_t img_stride, int mode_mask, int use_mask) {
  __shared__ MeRing ring;
  const int b = blockIdx.y;
  if (!mode_on(db.st[b].mode, mode_mask)) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int x0 = blockIdx.x * 30;
  const int W = dc.W, H = dc.H;
  if (x0 >= W) return;
  const unsigned char* img = imgs + (size_t)b * img_stride;
  const int cx = x0 - 1 + lane;                 // lanes 0 and 31 are halo
  int c = reflect101(cx, W);
  c = clampi(c, 0, W - 1);                      // lanes beyond the reflected border are inactive
  const int pitch = dc.pitch;
  if (threadIdx.x < ME_SLOTS) { ring.ready[threadIdx.x] = 0; ring.scanned[threadIdx.x] = 0; ring.finished[threadIdx.x] = 0; }
  if (threadIdx.x == 0) ring.cons_row = 0;
  __syncthreads();
  volatile int* ready = ring.ready;
  volatile int* scanned = ring.scanned;
  volatile int* finished = ring.finished;
  volatile int* cons_row = &ring.cons_row;

  if (warp < ME_PRODUCERS) {
    // ---- producers: Sobel, products, f64 row sums of chunk rows p0 .. p0 + 7
    const int cm = reflect101(c - 1, W), cp = reflect101(c + 1, W);
    const float s = (float)(1.0 / 3060.0), s2 = 2.0f * s;
    const bool tail = dc.sobel_tail_start >= 0 && c >= dc.sobel_tail_start;
    for (int p0 = warp * ME_CHUNK; p0 < H; p0 += ME_PRODUCERS * ME_CHUNK) {
      // image rows p0 - 1 .. p0 + ME_CHUNK (reflected), three columns each: independent loads, issued up front
      float im[ME_CHUNK + 2], i0[ME_CHUNK + 2], ip[ME_CHUNK + 2];
#pragma unroll
      for (int u = 0; u < ME_CHUNK + 2; ++u) {
        const int y = reflect101(min(p0 - 1 + u, H), H);
        const unsigned char* row = img + (size_t)y * pitch;
        im[u] = (float)row[cm]; i0[u] = (float)row[c]; ip[u] = (float)row[cp];
      }
      RT rt[ME_CHUNK + 2];
#pragma unroll
      for (int u = 0; u < ME_CHUNK + 2; ++u) rt[u] = rt_from(im[u], i0[u], ip[u], s, s2, tail);
      // the ring slots of this chunk are free once the scanner is past row p0 + ME_CHUNK - 1 - ME_RING
      while (*cons_row <= p0 + ME_CHUNK - 1 - ME_RING) __nanosleep(64);
      __threadfence_block();
#pragma unroll
      for (int u = 0; u < ME_CHUNK; ++u) {
        const int p = p0 + u;
        if (p < H) {
          // cv::Sobel column pass: Dx = fma(r(y-1) + r(y+1), s, (2s) * r(y)); Dy = t(y+1) - t(y-1)
          const float dx = fmaf(rt[u].r + rt[u + 2].r, s, s2 * rt[u + 1].r);
          const float dy = rt[u + 2].t - rt[u].t;
          const float pxx = dx * dx, pxy = dx * dy, pyy = dy * dy;
          // RowSum<float,double>, ksize 3: (S[x-1] + S[x]) + S[x+1]
          const float l0 = __shfl_up_sync(KVFE_FULL_MASK, pxx, 1), g0 = __shfl_down_sync(KVFE_FULL_MASK, pxx, 1);
          const float l1 = __shfl_up_sync(KVFE_FULL_MASK, pxy, 1), g1 = __shfl_down_sync(KVFE_FULL_MASK, pxy, 1);
          const float l2 = __shfl_up_sync(KVFE_FULL_MASK, pyy, 1), g2 = __shfl_down_sync(KVFE_FULL_MASK, pyy, 1);
          const int slot = p & (ME_RING - 1);
          ring.r0[slot][lane] = ((double)l0 + (double)pxx) + (double)g0;
          ring.r1[slot][lane] = ((double)l1 + (double)pxy) + (double)g1;
          ring.r2[slot][lane] = ((double)l2 + (double)pyy) + (double)g2;
        }
      }
      __syncwarp();
      __threadfence_block();
      if (lane == 0) ready[(p0 / ME_CHUNK) & (ME_SLOTS - 1)] = p0 / ME_CHUNK + 1;
    }
    return;
  }

  if (warp == ME_PRODUCERS) {
    // ---- scanner: the history-dependent running column sums, nothing else.  Iteration p consumes R(p) and emits the
    // sums of output row y = p - 1 into ring slot y % ME_RING; output chunk k = rows 8k .. 8k + 7.
    double sum0 = 0, sum1 = 0, sum2 = 0;             // running column sums (xx, xy, yy)
    double rm2_0 = 0, rm2_1 = 0, rm2_2 = 0;          // R(p-2)
    double rm1_0 = 0, rm1_1 = 0, rm1_2 = 0;          // R(p-1)
    for (int p0 = 0; p0 <= H; p0 += ME_CHUNK) {
      if (p0 < H) {                                      // one wait per chunk: its 8 rows then pipeline freely
        while (ready[(p0 / ME_CHUNK) & (ME_SLOTS - 1)] != p0 / ME_CHUNK + 1) __nanosleep(32);
        // output rows p0 .. p0 + 7 reuse the slots of rows p0 - 32 ..: their finisher must be done
        if (p0 >= ME_RING) while (finished[(p0 / ME_CHUNK) & (ME_SLOTS - 1)] != p0 / ME_CHUNK - ME_SLOTS + 1) __nanosleep(32);
        __threadfence_block();
      }
      double q0[ME_CHUNK], q1[ME_CHUNK], q2[ME_CHUNK];
#pragma unroll
      for (int u = 0; u < ME_CHUNK; ++u) {
        const int slot = (p0 + u) & (ME_RING - 1);
        q0[u] = ring.r0[slot][lane]; q1[u] = ring.r1[slot][lane]; q2[u] = ring.r2[slot][lane];
      }
#pragma unroll
      for (int u = 0; u < ME_CHUNK; ++u) {
        const int p = p0 + u;
        if (p > H) break;
        double r0, r1, r2;
        if (p < H) {
          r0 = q0[u]; r1 = q1[u]; r2 = q2[u];
        } else {
          r0 = rm2_0; r1 = rm2_1; r2 = rm2_2;            // R(H) = R(H-2) (reflect)
        }
        if (p == 1) {                                    // ColumnSum init: SUM = (0 + R(-1)) + R(0), R(-1) = R(1)
          sum0 = (0.0 + r0) + rm1_0;
          sum1 = (0.0 + r1) + rm1_1;
          sum2 = (0.0 + r2) + rm1_2;
        }
        if (p >= 1) {
          const int y = p - 1;
          // s0 = SUM + R(y+1); out = (float)s0; SUM = s0 - R(y-1)   (R(-1) = R(1))
          const double s0 = sum0 + r0, s1 = sum1 + r1, s2d = sum2 + r2;
          const double o0 = (y == 0) ? r0 : rm2_0, o1 = (y == 0) ? r1 : rm2_1, o2 = (y == 0) ? r2 : rm2_2;
          sum0 = s0 - o0; sum1 = s1 - o1; sum2 = s2d - o2;
          const int slot = y & (ME_RING - 1);
          ring.s0[slot][lane] = (float)s0; ring.s1[slot][lane] = (float)s1; ring.s2[slot][lane] = (float)s2d;
          if ((y & (ME_CHUNK - 1)) == ME_CHUNK - 1 || y == H - 1) {     // output chunk complete (warp-uniform)
            __syncwarp();
            __threadfence_block();
            if (lane == 0) scanned[(y / ME_CHUNK) & (ME_SLOTS - 1)] = y / ME_CHUNK + 1;
          }
        }
        rm2_0 = rm1_0; rm2_1 = rm1_1; rm2_2 = rm1_2;
        rm1_0 = r0; rm1_1 = r1; rm1_2 = r2;
      }
      __syncwarp();
      if (lane == 0) *cons_row = min(p0 + ME_CHUNK, H);   // every lane has read the R rows below this
    }
    return;
  }

  // ---- finishers: min-eigenvalue formula, store, masked maximum of output chunk k (rows 8k .. 8k + 7)
  const int fw = warp - ME_PRODUCERS - 1;
  const unsigned char* msk = db.mask + (size_t)b * dc.img_stride;
  float* eig = db.eig + (size_t)b * W * H;
  const bool writer = lane >= 1 && lane <= 30 && cx < W;
  const int cxw = clampi(cx, 0, W - 1);
  float vmax = -INFINITY;
  for (int k = fw; k * ME_CHUNK < H; k += ME_FINISHERS) {
    const int y0 = k * ME_CHUNK;
    unsigned char mk[ME_CHUNK];
#pragma unroll
    for (int u = 0; u < ME_CHUNK; ++u) mk[u] = use_mask ? msk[(size_t)min(y0 + u, H - 1) * pitch + cxw] : (unsigned char)255;
    while (scanned[k & (ME_SLOTS - 1)] != k + 1) __nanosleep(64);
    __threadfence_block();
    float a0[ME_CHUNK], a1[ME_CHUNK], a2[ME_CHUNK];
#pragma unroll
    for (int u = 0; u < ME_CHUNK; ++u) {
      const int slot = (y0 + u) & (ME_RING - 1);
      a0[u] = ring.s0[slot][lane]; a1[u] = ring.s1[slot][lane]; a2[u] = ring.s2[slot][lane];
    }
    __syncwarp();
    if (lane == 0) finished[k & (ME_SLOTS - 1)] = k + 1;       // every lane holds the chunk in registers
#pragma unroll
    for (int u = 0; u < ME_CHUNK; ++u) {
      const int y = y0 + u;
      if (writer && y < H) {
        const float A = a0[u] * 0.5f, Bv = a1[u], C = a2[u] * 0.5f;
        const float e = (A + C) - sqrtf((A - C) * (A - C) + Bv * Bv);
        eig[(size_t)y * W + cx] = e;
        if (mk[u]) vmax = fmaxf(vmax, e);
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) vmax = fmaxf(vmax, __shfl_xor_sync(KVFE_FULL_MASK, vmax, o));
  if (lane == 0 && vmax > -INFINITY) atomicMax(&db.eig_max[b], f2ord(vmax));
}

// grid B, block 256
__global__ void gftt_init_kernel(DevCfg dc, DevBuf db, int mode_mask) {
  const int b = blockIdx.x;
  if (!mode_on(db.st[b].mode, mode_mask)) return;
  if (threadIdx.x == 0) {
    db.eig_max[b] = f2ord(-INFINITY);
    db.cand_n[b] = 0;
    db.corner_n[b] = 0;
    db.cand_sel_n[b] = 0;
    db.greedy_redo[b] = 0;
  }
  for (int i = threadIdx.x; i < CAND_HIST_BINS; i += blockDim.x) db.cand_hist[(size_t)b * CAND_HIST_BINS + i] = 0;
}

// ------------------------------------------------------------------------------------------------
// candidates: interior pixels with eig > thr, eig == 3x3 max, mask != 0
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) cand_kernel(DevCfg dc, DevBuf db, int mode_mask) {
  const int b = blockIdx.z;
  if (!mode_on(db.st[b].mode, mode_mask)) return;
  const int W = dc.W, H = dc.H;
  const int x = blockIdx.x * 32 + (threadIdx.x & 31);
  const float* e = db.eig + (size_t)b * W * H;
  float maxv = ord2f(db.eig_max[b]);
  if (!(maxv > -INFINITY)) maxv = 0.f;              // empty mask: minMaxLoc leaves maxVal = 0
  const float thr = (float)((double)maxv * dc.quality);   // cv::threshold(eig, eig, maxVal * qualityLevel, ...)
  for (int k = 0; k < 8; ++k) {
    const int y = blockIdx.y * 64 + k * 8 + (threadIdx.x >> 5);
    if (x < 1 || y < 1 || x > W - 2 || y > H - 2) continue;
    const float v = e[(size_t)y * W + x];
    if (!(v > thr)) continue;
    if (!db.mask[(size_t)b * dc.img_stride + (size_t)y * dc.pitch + x]) continue;
    const float* r0 = e + (size_t)(y - 1) * W + x;
    const float* r1 = r0 + W;
    const float* r2 = r1 + W;
    float nb = fmaxf(fmaxf(fmaxf(r0[-1], r0[0]), fmaxf(r0[1], r1[-1])), fmaxf(fmaxf(r1[1], r2[-1]), fmaxf(r2[0], r2[1])));
    if (v < nb) continue;
    int slot = atomicAdd(&db.cand_n[b], 1);
    if (slot < dc.cand_cap)
      db.cand[(size_t)b * dc.cand_cap + slot] =
          ((unsigned long long)__float_as_uint(v) << 32) | ((unsigned int)y << 16) | (unsigned int)x;   // (y, x) orders like y * W + x
  }
}

// ------------------------------------------------------------------------------------------------
// Top-K prefilter of the candidate list.  cv::goodFeaturesToTrack walks the candidates in descending order and
// stops after maxCorners acceptances, and a candidate's fate depends only on BETTER candidates: the greedy
// selection over the best K candidates decides them exactly as the full run would, and when it already yields
// maxCorners corners the rest of the list is never looked at.  A 4K keyframe has > 10^5 candidates at
// quality_level 0.001 but needs 2000 corners: the single-CTA selection over all of them took 18.7 ms; over the
// best ~12 k it runs out of shared memory like the 752 x 480 case.  When the prefix does NOT reach maxCorners
// the selection is repeated over the full list (second launch, exits at entry otherwise): always exact.
//   cand_hist_kernel     histogram of the candidates' float bits relative to the maximum (128 bins per binade)
//   cand_compact_kernel  threshold bin for >= GREEDY_TOPK candidates, compaction into cand_sel
// ------------------------------------------------------------------------------------------------

__device__ __forceinline__ int cand_bin(unsigned long long key, unsigned int maxbits) {
  const int d = (int)(maxbits >> 16) - (int)((unsigned int)(key >> 32) >> 16);
  return d < 0 ? 0 : (d > CAND_HIST_BINS - 1 ? CAND_HIST_BINS - 1 : d);
}

// grid (x, B)
__global__ void __launch_bounds__(256) cand_hist_kernel(DevCfg dc, DevBuf db, int mode_mask) {
  __shared__ int h[CAND_HIST_BINS];
  const int b = blockIdx.y;
  if (!mode_on(db.st[b].mode, mode_mask)) return;
  const int n = min(db.cand_n[b], dc.cand_cap);
  if (n <= GREEDY_TOPK) return;                     // small list: the selection reads it as it is
  for (int i = threadIdx.x; i < CAND_HIST_BINS; i += blockDim.x) h[i] = 0;
  __syncthreads();
  const unsigned long long* gk = db.cand + (size_t)b * dc.cand_cap;
  const unsigned int maxbits = __float_as_uint(ord2f(db.eig_max[b]));
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) atomicAdd(&h[cand_bin(gk[i], maxbits)], 1);
  __syncthreads();
  int* gh = db.cand_hist + (size_t)b * CAND_HIST_BINS;
  for (int i = threadIdx.x; i < CAND_HIST_BINS; i += blockDim.x) if (h[i]) atomicAdd(&gh[i], h[i]);
}

// grid (x, B): every CTA finds the threshold bin from the finished histogram, then compacts its slice
__global__ void __launch_bounds__(256) cand_compact_kernel(DevCfg dc, DevBuf db, int mode_mask) {
  __shared__ int s_t;
  const int b = blockIdx.y;
  if (!mode_on(db.st[b].mode, mode_mask)) return;
  const int n = min(db.cand_n[b], dc.cand_cap);
  if (n <= GREEDY_TOPK) return;
  const int* gh = db.cand_hist + (size_t)b * CAND_HIST_BINS;
  if (threadIdx.x < 32) {                           // smallest t with count(bin <= t) >= GREEDY_TOPK
    int carry = 0, t = CAND_HIST_BINS - 1;
    bool found = false;
    for (int base = 0; base < CAND_HIST_BINS && !found; base += 32) {
      const int v = gh[base + threadIdx.x];
      int incl = v;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int u = __shfl_up_sync(KVFE_FULL_MASK, incl, o);
        if ((int)threadIdx.x >= o) incl += u;
      }
      const unsigned hit = __ballot_sync(KVFE_FULL_MASK, carry + incl >= GREEDY_TOPK);
      if (hit) { t = base + __ffs(hit) - 1; found = true; }
      carry += __shfl_sync(KVFE_FULL_MASK, incl, 31);
    }
    if (threadIdx.x == 0) s_t = t;
  }
  __syncthreads();
  const int t = s_t;
  const unsigned long long* gk = db.cand + (size_t)b * dc.cand_cap;
  unsigned long long* sel = db.cand_sel + (size_t)b * GREEDY_SEL_CAP;
  const unsigned int maxbits = __float_as_uint(ord2f(db.eig_max[b]));
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const unsigned long long key = gk[i];
    if (cand_bin(key, maxbits) <= t) {
      const int pos = atomicAdd(&db.cand_sel_n[b], 1);
      if (pos < GREEDY_SEL_CAP) sel[pos] = key;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// greedy min-distance selection, one CTA per stream.  The sequential OpenCV loop accepts a
// candidate iff no BETTER (higher value, ties: higher address) already-accepted candidate lies in
// the 3x3 neighbouring cells within minDistance.  "Better" is a comparison of the 64-bit keys, so no
// global sort is needed for the decision: candidates are bucketed into the cell grid and a parallel
// fixed point (accept when every better conflicting neighbour is rejected, reject when one is
// accepted) reproduces the sequential result; only the accepted corners (<= a few thousand) are
// sorted at the end to produce OpenCV's output order and the maxCorners cut.
// ------------------------------------------------------------------------------------------------
__device__ void bitonic_desc(unsigned long long* k, int P) {
  for (int size = 2; size <= P; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = threadIdx.x; t < (P >> 1); t += blockDim.x) {
        int lo = 2 * t - (t & (stride - 1));
        int hi = lo + stride;
        bool desc = ((lo & size) == 0);
        unsigned long long a = k[lo], c = k[hi];
        if ((a < c) == desc) { k[lo] = c; k[hi] = a; }
      }
      __syncthreads();
    }
  }
}

__device__ int getenv_dbg = 0;
#define GREEDY_ACC_MAX 2048
#define GREEDY_SMEM_CELLS 4096

// Layout of the dynamic shared memory: skey[smem_keys] (candidates ordered by (cell, key desc)),
// then acc[GREEDY_ACC_MAX].  When the candidates do not fit, skey lives in the global candidate
// buffer instead (same code path, slower).
// pass 0: the top-K prefix when the prefilter produced one (else the full list); pass 1: the full list, only for the
// streams whose prefix did not reach maxCorners (greedy_redo)
__global__ void __launch_bounds__(1024, 1) sort_greedy_kernel(DevCfg dc, DevBuf db, int mode_mask, int smem_keys, int pass) {
  extern __shared__ unsigned long long skeys[];
  const int b = blockIdx.x;
  if (!mode_on(db.st[b].mode, mode_mask)) return;
  const int W = dc.W, H = dc.H;
  const int n_all = min(db.cand_n[b], dc.cand_cap);
  const int n_sel = db.cand_sel_n[b];
  const bool prefix = pass == 0 && n_all > GREEDY_TOPK && n_sel <= GREEDY_SEL_CAP;
  if (pass == 1 && !db.greedy_redo[b]) return;
  const int n = prefix ? n_sel : n_all;
  unsigned long long* gk = prefix ? db.cand_sel + (size_t)b * GREEDY_SEL_CAP : db.cand + (size_t)b * dc.cand_cap;
  int* corner = db.corner_idx + (size_t)b * dc.max_before_anms;
  __shared__ int s_total, s_chunk, wsum[32];
  const int md = dc.min_distance;
  const int tid = threadIdx.x;

  if (md < 1) {                             // no min-distance: plain top-maxCorners (needs the full sort)
    int P = 2;
    while (P < n) P <<= 1;
    unsigned long long* k = (P <= smem_keys) ? skeys : gk;
    for (int i = tid; i < P; i += blockDim.x) k[i] = (i < n) ? gk[i] : 0ull;
    __syncthreads();
    bitonic_desc(k, P);
    int m = min(n, dc.max_before_anms);
    for (int i = tid; i < m; i += blockDim.x) { const unsigned int lo = (unsigned int)(k[i] & 0xffffffffu); corner[i] = (int)(lo >> 16) * W + (int)(lo & 0xffffu); }
    if (tid == 0) db.corner_n[b] = m;
    return;
  }

  int* sc = db.scratch_i + (size_t)b * db.scratch_stride;
  // cells of k * minDistance (any cell >= minDistance keeps every conflict inside the 3x3 neighbourhood): the
  // smallest k whose grid fits the shared-memory bookkeeping -- 1 at 752x480 / 20 px, 3 at 3840x2160
  int cell = md;                            // cvRound(minDistance), minDistance is an int parameter
  while ((long long)((W + cell - 1) / cell) * ((H + cell - 1) / cell) + 1 > GREEDY_SMEM_CELLS && cell < 64 * md) cell += md;
  const int gw = (W + cell - 1) / cell, gh = (H + cell - 1) / cell;
  const int ncells = gw * gh;
  // bookkeeping arrays: shared memory when the grid and the candidate list fit, else global scratch
  unsigned char* sm_tail = reinterpret_cast<unsigned char*>(skeys + smem_keys + GREEDY_ACC_MAX);
  const bool small = (ncells + 1 <= GREEDY_SMEM_CELLS) && (n <= smem_keys);
  // global-scratch sections are sized from the cell grid (min_distance 1 gives one cell per pixel);
  // kvfe_create sizes scratch_stride with the same formula (greedy_scratch_ints)
  const int o_head = (ncells + 1 + 3) & ~3, o_new = o_head + ncells, o_state = o_new + ncells;
  const int o_tmp = (o_state + dc.cand_cap / 4 + 1) & ~1;
  int* cstart = small ? reinterpret_cast<int*>(sm_tail) : sc;                                   // [ncells + 1]
  int* head = small ? cstart + GREEDY_SMEM_CELLS : sc + o_head;                                 // [ncells]
  int* newacc = small ? head + GREEDY_SMEM_CELLS : sc + o_new;                                  // [ncells]
  unsigned char* state = small ? reinterpret_cast<unsigned char*>(newacc + GREEDY_SMEM_CELLS)
                               : reinterpret_cast<unsigned char*>(sc + o_state);                // [n]
  unsigned long long* tmp = reinterpret_cast<unsigned long long*>(sc + o_tmp);                  // [cand_cap] keys by cell
  unsigned long long* sk = (n <= smem_keys) ? skeys : gk;
  // ---- 1. bucket by cell (counting sort) into tmp
  for (int i = tid; i <= ncells; i += blockDim.x) cstart[i] = 0;
  __syncthreads();
  for (int i = tid; i < n; i += blockDim.x) {
    const unsigned int lo = (unsigned int)(gk[i] & 0xffffffffu);
    int y = (int)(lo >> 16), x = (int)(lo & 0xffffu);
    atomicAdd(&cstart[(y / cell) * gw + (x / cell) + 1], 1);
  }
  __syncthreads();
  if (tid < 32) {                           // exclusive scan of the cell counts by one warp
    int carry = 0;
    for (int base = 0; base <= ncells; base += 32) {
      int i = base + tid;
      int v = (i <= ncells) ? cstart[i] : 0, incl = v;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(KVFE_FULL_MASK, incl, o);
        if (tid >= o) incl += t;
      }
      if (i <= ncells) cstart[i] = carry + incl - v;
      carry += __shfl_sync(KVFE_FULL_MASK, incl, 31);
    }
  }
  __syncthreads();
  for (int i = tid; i < n; i += blockDim.x) {        // cstart[c+1] = cursor of cell c
    unsigned long long key = gk[i];
    const unsigned int lo = (unsigned int)(key & 0xffffffffu);
    int y = (int)(lo >> 16), x = (int)(lo & 0xffffu);
    int pos = atomicAdd(&cstart[(y / cell) * gw + (x / cell) + 1], 1);
    tmp[pos] = key;
  }
  __syncthreads();
  // now cell c spans [cstart[c], cstart[c+1]) in tmp
  // ---- 2. order every cell by key descending (rank by counting inside the cell)
  for (int i = tid; i < n; i += blockDim.x) {
    unsigned long long key = tmp[i];
    const unsigned int lo = (unsigned int)(key & 0xffffffffu);
    int y = (int)(lo >> 16), x = (int)(lo & 0xffffu);
    int c = (y / cell) * gw + (x / cell);
    int a0 = cstart[c], a1 = cstart[c + 1], rank = 0;
    for (int q = a0; q < a1; ++q) rank += tmp[q] > key;
    sk[a0 + rank] = key;
    state[i] = 0;
  }
  for (int c = tid; c < ncells; c += blockDim.x) { head[c] = cstart[c]; newacc[c] = -1; }
  __syncthreads();
  // ---- 3. rounds: only the best undecided candidate of each cell ("head") is examined
  const int md2 = md * md;
  volatile unsigned char* vst = state;
  volatile int* vhead = head;
  // Asynchronous relaxation, one WARP per cell: the warps draw cells from a shared counter and decide a cell's
  // successive heads; the 32 lanes test the candidates of the three neighbouring cell rows in parallel (a row's
  // three cells are contiguous in the cell-ordered array).  An accepted head immediately rejects the undecided
  // candidates within minDistance.  States only move 0 -> 1/2, readers of a stale 0 merely wait, and two
  // conflicting heads can never both be accepted (the worse one always sees the better one as undecided or
  // accepted; "rejected" wins over "wait": an accepted better neighbour within minDistance is final).
  // (Round 1 gave every cell to one THREAD: the critical path was the busiest thread's serial scan -- 49 % of
  // the samples sat in the barrier behind it, profiles/r02_ncu_kf.txt.)
  __shared__ int s_next_cell;
  const int lane = tid & 31;
  for (int round = 0; round < 100000; ++round) {
    int active = 0;
    if (tid == 0) s_next_cell = 0;
    __syncthreads();
    for (;;) {
      int c = 0;
      if (lane == 0) c = atomicAdd(&s_next_cell, 1);
      c = __shfl_sync(KVFE_FULL_MASK, c, 0);
      if (c >= ncells) break;
      const int e = cstart[c + 1];
      int h = vhead[c];
      if (h >= e) continue;
      const int cxl = c % gw, cyl = c / gw;
      const int x1 = max(cxl - 1, 0), x2 = min(cxl + 1, gw - 1), y1 = max(cyl - 1, 0), y2 = min(cyl + 1, gh - 1);
      for (int attempt = 0; attempt < 64; ++attempt) {
        while (h < e && vst[h] != 0) ++h;              // skip decided entries (warp-uniform)
        if (h >= e) break;
        const unsigned long long kh = sk[h];
        const unsigned int lo = (unsigned int)(kh & 0xffffffffu);
        const int y = (int)(lo >> 16), x = (int)(lo & 0xffffu);
        bool rej = false, wait = false;
        for (int yy = y1; yy <= y2; ++yy) {
          const int qa = cstart[yy * gw + x1], qb = cstart[yy * gw + x2 + 1];
          for (int q = qa + lane; q < qb; q += 32) {
            const unsigned long long kq = sk[q];
            if (kq <= kh) continue;                       // only better candidates matter (kq == kh: the head itself)
            const int sq = vst[q];
            if (sq == 2) continue;
            const unsigned int jlo = (unsigned int)(kq & 0xffffffffu);
            const int ddx = x - (int)(jlo & 0xffffu), ddy = y - (int)(jlo >> 16);
            if (ddx * ddx + ddy * ddy < md2) { if (sq == 1) rej = true; else wait = true; }
          }
        }
        rej = __any_sync(KVFE_FULL_MASK, rej);
        wait = __any_sync(KVFE_FULL_MASK, wait);
        if (!rej && wait) { active = 1; break; }        // blocked by an undecided better neighbour
        if (lane == 0) vst[h] = rej ? (unsigned char)2 : (unsigned char)1;
        __syncwarp();
        if (!rej) {
          __threadfence_block();
          for (int yy = y1; yy <= y2; ++yy) {           // reject the undecided candidates within minDistance
            const int qa = cstart[yy * gw + x1], qb = cstart[yy * gw + x2 + 1];
            for (int q = qa + lane; q < qb; q += 32) {
              if (vst[q] != 0) continue;
              const unsigned int jlo = (unsigned int)(sk[q] & 0xffffffffu);
              const int ddx = x - (int)(jlo & 0xffffu), ddy = y - (int)(jlo >> 16);
              if (ddx * ddx + ddy * ddy < md2) vst[q] = 2;
            }
          }
          __syncwarp();
        }
      }
      while (h < e && vst[h] != 0) ++h;
      if (lane == 0) vhead[c] = h;
      if (h < e) active = 1;
    }
    if (!__syncthreads_or(active)) { if (tid == 0 && getenv_dbg) printf("greedy b=%d pass=%d n=%d ncells=%d cell=%d rounds=%d\n", b, pass, n, ncells, cell, round + 1); break; }
  }
  __syncthreads();
  // ---- 4. gather accepted keys, sort them descending, emit the first maxCorners
  // (shared memory when they fit, else the -- now free -- global bucket buffer)
  int my_acc = 0;
  for (int i = tid; i < n; i += blockDim.x) my_acc += (state[i] == 1);
  if (tid == 0) s_total = 0;
  __syncthreads();
  if (my_acc) atomicAdd(&s_total, my_acc);
  __syncthreads();
  const int acc_cap = (s_total <= GREEDY_ACC_MAX) ? GREEDY_ACC_MAX : dc.cand_cap;
  unsigned long long* acc = (s_total <= GREEDY_ACC_MAX) ? (skeys + smem_keys) : tmp;
  __syncthreads();
  if (tid == 0) s_total = 0;
  __syncthreads();
  for (int base = 0; base < n; base += blockDim.x) {
    int i = base + tid;
    int a = (i < n && state[i] == 1) ? 1 : 0;
    unsigned bal = __ballot_sync(KVFE_FULL_MASK, a);
    int lane = tid & 31, warp = tid >> 5;
    if (lane == 0) wsum[warp] = __popc(bal);
    __syncthreads();
    if (warp == 0) {
      int v = wsum[lane], incl = v;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(KVFE_FULL_MASK, incl, o);
        if (lane >= o) incl += t;
      }
      wsum[lane] = incl - v;
      if (lane == 31) s_chunk = incl;
    }
    __syncthreads();
    int pos = s_total + wsum[warp] + __popc(bal & ((1u << lane) - 1));
    if (a && pos < acc_cap) acc[pos] = sk[i];
    __syncthreads();
    if (tid == 0) s_total += s_chunk;
    __syncthreads();
  }
  const int na = min(s_total, acc_cap);
  int P = 2;
  while (P < na) P <<= 1;
  for (int i = na + tid; i < P; i += blockDim.x) acc[i] = 0ull;
  __syncthreads();
  bitonic_desc(acc, P);
  const int m = min(na, dc.max_before_anms);
  if (prefix && na < dc.max_before_anms) {
    // the best-K prefix does not fill maxCorners: the full list decides (pass 1)
    if (tid == 0) db.greedy_redo[b] = 1;
    return;
  }
  for (int i = tid; i < m; i += blockDim.x) { const unsigned int lo = (unsigned int)(acc[i] & 0xffffffffu); corner[i] = (int)(lo >> 16) * W + (int)(lo & 0xffffu); }
  if (tid == 0) { db.corner_n[b] = m; db.greedy_redo[b] = 0; }
  (void)H;
}

static int launch_mineig_any(const DevCfg& dc, const DevBuf& db, const unsigned char* img, size_t img_stride, int mode_mask,
                             int use_mask, cudaStream_t s) {
  static const int mode = getenv("KVFE_MINEIG") ? atoi(getenv("KVFE_MINEIG")) : 2;      // diagnostic: 1 = mineig_kernel
  const int groups = (dc.W + 29) / 30;
  if (mode == 2) mineig_pipe_kernel<<<dim3(groups, dc.B), 32 * (ME_PRODUCERS + 1 + ME_FINISHERS), 0, s>>>(dc, db, img, img_stride, mode_mask, use_mask);
  else mineig_kernel<<<dim3((groups + 3) / 4, dc.B), 128, 0, s>>>(dc, db, img, img_stride, mode_mask, use_mask);
  return 1;
}

int launch_min_eig(const DevCfg& dc, const DevBuf& db, const unsigned char* img, size_t img_stride,
                   int mode_mask, cudaStream_t s) {
  int n = 0;
  gftt_init_kernel<<<dc.B, 256, 0, s>>>(dc, db, mode_mask); ++n;
  n += launch_mineig_any(dc, db, img, img_stride, mode_mask, 0, s);
  return n;
}

int launch_gftt(const DevCfg& dc, const DevBuf& db, const unsigned char* img, size_t img_stride,
                const int* circle_hw, int circle_r, int mode_mask, cudaStream_t s, int keep_mask) {
  int n = 0;
  gftt_init_kernel<<<dc.B, 256, 0, s>>>(dc, db, mode_mask); ++n;
  // keep_mask: db.mask already holds the caller's Frame::detection_mask_ (FeatureDetector.cpp:186-189)
  if (!keep_mask) { mask_fill_kernel<<<dim3(64, dc.B), 256, 0, s>>>(dc, db.mask, db.st, mode_mask); ++n; }
  mask_circles_kernel<<<dim3((dc.cap + 7) / 8, dc.B), 256, 0, s>>>(dc, db, circle_hw, circle_r, mode_mask); ++n;
  n += launch_mineig_any(dc, db, img, img_stride, mode_mask, 1, s);
  cand_kernel<<<dim3((dc.W + 31) / 32, (dc.H + 63) / 64, dc.B), 256, 0, s>>>(dc, db, mode_mask); ++n;
  int smem_keys = 16384;
  const int smem_bytes = (smem_keys + GREEDY_ACC_MAX) * 8 + 3 * GREEDY_SMEM_CELLS * 4 + smem_keys;
  static bool attr_set = false;
  if (!attr_set) {
    cudaFuncSetAttribute(sort_greedy_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
    attr_set = true;
  }
  { static int once = 0; if (!once) { once = 1; if (getenv("KVFE_GREEDY_DEBUG")) { int one = 1; cudaMemcpyToSymbol(getenv_dbg, &one, sizeof(int)); } } }
  cand_hist_kernel<<<dim3(32, dc.B), 256, 0, s>>>(dc, db, mode_mask); ++n;
  cand_compact_kernel<<<dim3(32, dc.B), 256, 0, s>>>(dc, db, mode_mask); ++n;
  sort_greedy_kernel<<<dc.B, 1024, smem_bytes, s>>>(dc, db, mode_mask, smem_keys, 0); ++n;
  sort_greedy_kernel<<<dc.B, 1024, smem_bytes, s>>>(dc, db, mode_mask, smem_keys, 1); ++n;
  return n;
}
