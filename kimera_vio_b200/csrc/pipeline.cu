// pipeline.cu -- kvfe_pipeline_*: native dispatcher threads serving `n_streams` independent camera
// streams (one device-resident context each) through input / output queues, the shape the reference
// puts around its front-end (include/kimera-vio/pipeline/PipelineModule.h:190-232, :359-416).
//
// Host cost of one frame: a ~100-byte write into the context's mapped I/O block and ONE
// cudaGraphLaunch.  Everything else happens on the device: fetch_io_kernel pulls the images (from
// pinned host memory over the host link, or from HBM) through the pointers in the I/O block, the
// step kernels run, publish_io_kernel stores the packet (and a keyframe's rectified images) into the
// pinned output slot and publishes the step's sequence number, which is all a dispatcher polls.
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <mutex>
#include <thread>
#include <vector>

#include <sched.h>
#include <time.h>

#include "kvfe_internal.h"

namespace {

struct PipeIn {
  const unsigned char* L; const unsigned char* R; size_t pitch;
  const unsigned char* D; size_t dpitch;       // RGB-D: depth image (null otherwise)
  long long ts; double Rm[9]; unsigned long long tag;
  int force_kf;
};
struct PipeOutSlot { unsigned char* packet; unsigned char* rectL; unsigned char* rectR; };
struct PipeFlight { int out_slot, io_slot; unsigned long long seq, tag; int phase; };   // phase 0: decision pending (split graphs)

struct PipeStream {
  kvfe_ctx* ctx = nullptr;
  std::mutex mu;                      // guards `in` and `free_out`
  std::deque<PipeIn> in;
  std::vector<int> free_out;
  std::vector<PipeOutSlot> out;
  unsigned char* out_block = nullptr; // one pinned allocation behind `out`
  unsigned char* stage[2] = {nullptr, nullptr};   // pinned staging of pageable inputs, per I/O slot (lazy)
  unsigned char* dstage[2] = {nullptr, nullptr};  // the same for a pageable depth image (RGB-D)
  bool force_next = false;            // kvfe_pipeline_force_keyframe: Frame::isKeyframe_ of the next pushed frame (under mu)
  // dispatcher-private
  std::deque<PipeFlight> fl;
  unsigned long long seq = 0;
};

inline double now_s() {
  timespec t; clock_gettime(CLOCK_MONOTONIC, &t);
  return (double)t.tv_sec + 1e-9 * (double)t.tv_nsec;
}

}  // namespace

struct kvfe_pipeline {
  kvfe_pipeline_config pc{};
  int W = 0, H = 0, device = 0;
  size_t packet_bytes = 0, img = 0;
  size_t pk_off[KVFE_PACKET_ARRAYS] = {0};
  int cap = 0;
  std::vector<PipeStream*> streams;
  std::vector<std::thread> workers;
  std::atomic<bool> stop{false};
  std::mutex out_mu; std::condition_variable out_cv; std::deque<kvfe_pipeline_output> outq;
  std::mutex wk_mu; std::condition_variable wk_cv;
  std::atomic<long long> n_pushed{0}, n_done{0}, n_graph{0}, n_kernels{0}, n_staged{0};
  std::atomic<long long> launch_ns{0};
  std::atomic<int> failed{0};
  std::mutex err_mu; char err[512] = "";
  bool split = false;                 // split step graphs (keyframe kernels launched only for keyframes)
  bool rgbd = false;                  // frontend_type 2: frames come with a depth image (kvfe_pipeline_push_rgbd)
  size_t depth_row = 0;               // bytes per depth row (W * 2 or W * 4)
};

static thread_local char g_pipe_create_err[512] = "";

// KVFE_ERR_INVALID_ARG with a message, without marking the pipeline failed (nothing was enqueued)
static int pipe_refuse(kvfe_pipeline* p, const char* msg) {
  std::lock_guard<std::mutex> g(p->err_mu);
  snprintf(p->err, sizeof(p->err), "%s", msg);
  return KVFE_ERR_INVALID_ARG;
}

static int pipe_fail(kvfe_pipeline* p, int code, const char* msg) {
  if (p) {
    std::lock_guard<std::mutex> g(p->err_mu);
    snprintf(p->err, sizeof(p->err), "%s", msg);
    p->failed.store(code);
  } else {
    snprintf(g_pipe_create_err, sizeof(g_pipe_create_err), "%s", msg);
  }
  return code;
}

// one graph per pyramid slot: fetch (indirect) -> the step kernels -> publish (indirect)
static int build_pipe_graph(kvfe_ctx* ctx, int slot) {
  cudaGraph_t g = nullptr;
  long long n = 0;
  ctx->cur_slot = slot;
  StepIO* io = reinterpret_cast<StepIO*>(ctx->pio[slot]);
  cudaError_t e = cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal);
  if (e != cudaSuccess) return kvfe_set_err(ctx, KVFE_ERR_CUDA, "pipeline graph capture: %s", cudaGetErrorString(e));
  long long k = 0;
  if (ctx->db.stage_img[0]) {
    // fork: the prefetch of the next frame's images runs beside the whole step and joins at its end
    cudaEventRecord(ctx->ev_fork, ctx->stream);
    cudaStreamWaitEvent(ctx->side, ctx->ev_fork, 0);
    n += launch_prefetch_io(ctx->dc, ctx->db, io, slot, ctx->d_pub_count + 1, ctx->side);
    cudaEventRecord(ctx->ev_join, ctx->side);
  }
  n += launch_fetch_io(ctx->dc, ctx->db, io, slot, ctx->stream);
  int rc = kvfe_enqueue_step_kernels(ctx, io, &k);
  n += k;
  n += launch_publish_io(ctx->dc, ctx->db, io, ctx->d_pub_count, ctx->stream);
  if (ctx->db.stage_img[0]) cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0);
  e = cudaStreamEndCapture(ctx->stream, &g);
  if (rc != KVFE_OK) { if (g) cudaGraphDestroy(g); return rc; }
  if (e != cudaSuccess) return kvfe_set_err(ctx, KVFE_ERR_CUDA, "pipeline graph capture: %s", cudaGetErrorString(e));
  e = cudaGraphInstantiate(&ctx->pipe_graph[slot], g, 0);
  cudaGraphDestroy(g);
  if (e != cudaSuccess) return kvfe_set_err(ctx, KVFE_ERR_CUDA, "pipeline graph instantiation: %s", cudaGetErrorString(e));
  ctx->pipe_graph_ready[slot] = 1;
  ctx->pipe_graph_launches = n;
  return KVFE_OK;
}

// Split variant: three graphs per pyramid slot.  A = fetch(left) .. decide + publish_decision; then the dispatcher, which
// polls the decision in the mapped I/O block, launches EITHER the keyframe graph (fetch(right), RANSAC, rectification,
// stereo, detection, finalize, publish) OR the two-kernel tracking tail (finalize, publish).  A tracking frame -- three out
// of four -- costs 13 launches instead of 36; the price is one host reaction per frame, hidden by the other streams.
static int capture_exec(kvfe_ctx* ctx, cudaGraphExec_t* exec, int (*body)(kvfe_ctx*, StepIO*, int, long long*), StepIO* io, int arg,
                        long long* n) {
  cudaGraph_t g = nullptr;
  cudaError_t e = cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal);
  if (e != cudaSuccess) return kvfe_set_err(ctx, KVFE_ERR_CUDA, "pipeline graph capture: %s", cudaGetErrorString(e));
  const int rc = body(ctx, io, arg, n);
  e = cudaStreamEndCapture(ctx->stream, &g);
  if (rc != KVFE_OK) { if (g) cudaGraphDestroy(g); return rc; }
  if (e != cudaSuccess) return kvfe_set_err(ctx, KVFE_ERR_CUDA, "pipeline graph capture: %s", cudaGetErrorString(e));
  e = cudaGraphInstantiate(exec, g, 0);
  cudaGraphDestroy(g);
  if (e != cudaSuccess) return kvfe_set_err(ctx, KVFE_ERR_CUDA, "pipeline graph instantiation: %s", cudaGetErrorString(e));
  return KVFE_OK;
}
static int body_a(kvfe_ctx* ctx, StepIO* io, int slot, long long* n) {
  long long k = 0;
  *n = launch_fetch_io(ctx->dc, ctx->db, io, slot, ctx->stream);
  const int rc = kvfe_enqueue_step_part(ctx, io, 0, &k);
  *n += k;
  return rc;
}
static int body_tail(kvfe_ctx* ctx, StepIO* io, int part, long long* n) {
  long long k = 0;
  const int rc = kvfe_enqueue_step_part(ctx, io, part, &k);
  *n = k + launch_publish_io(ctx->dc, ctx->db, io, ctx->d_pub_count, ctx->stream);
  return rc;
}
static int build_split_graphs(kvfe_ctx* ctx, int slot) {
  ctx->cur_slot = slot;
  StepIO* io = reinterpret_cast<StepIO*>(ctx->pio[slot]);
  int rc = capture_exec(ctx, &ctx->pipe_graph_a[slot], body_a, io, slot, &ctx->pipe_launches_a);
  if (rc == KVFE_OK) rc = capture_exec(ctx, &ctx->pipe_graph_kf[slot], body_tail, io, 1, &ctx->pipe_launches_kf);
  if (rc == KVFE_OK) rc = capture_exec(ctx, &ctx->pipe_graph_nokf[slot], body_tail, io, 2, &ctx->pipe_launches_nokf);
  if (rc == KVFE_OK) ctx->pipe_split_ready[slot] = 1;
  return rc;
}

// sum of the 64-bit words of [p, p + bytes) (bytes is a multiple of 8 for every range used here)
static inline unsigned long long sum64(const unsigned char* p, size_t bytes) {
  const unsigned long long* q = reinterpret_cast<const unsigned long long*>(p);
  const size_t n = bytes / 8;
  unsigned long long a = 0, b = 0, c = 0, d = 0;
  size_t i = 0;
  for (; i + 4 <= n; i += 4) { a += q[i]; b += q[i + 1]; c += q[i + 2]; d += q[i + 3]; }
  for (; i < n; ++i) a += q[i];
  unsigned long long tail = 0;
  if (bytes & 7) memcpy(&tail, p + n * 8, bytes & 7);
  return a + b + c + d + tail;
}

static unsigned long long packet_checksum(const kvfe_pipeline* p, const unsigned char* pk) {
  static const size_t sz[KVFE_PACKET_ARRAYS] = {4, 4, 8, 4, 8, 24, 4, 4, 4, 4, 4, 4, 8, 24, 4, 4, 8, 8, 8, 8, 24};
  const kvfe_packet_header* h = reinterpret_cast<const kvfe_packet_header*>(pk);
  unsigned long long s = sum64(pk, sizeof(kvfe_packet_header));
  const int n = h->n < 0 ? 0 : (h->n > p->cap ? p->cap : h->n);
  const int ns = h->n_smart < 0 ? 0 : (h->n_smart > p->cap ? p->cap : h->n_smart);
  const int nt = h->n_mesh_triangles < 0 ? 0 : (h->n_mesh_triangles > 2 * p->cap ? 2 * p->cap : h->n_mesh_triangles);
  for (int i = 0; i < KVFE_PACKET_ARRAYS; ++i) s += sum64(pk + p->pk_off[i], sz[i] * (size_t)(i == 20 ? nt : i >= 16 ? ns : n));
  return s;
}

static void emit(kvfe_pipeline* p, int sidx, PipeStream* s, const PipeFlight& f) {
  kvfe_pipeline_output o;
  memset(&o, 0, sizeof(o));
  const PipeOutSlot& os = s->out[f.out_slot];
  const kvfe_packet_header* h = reinterpret_cast<const kvfe_packet_header*>(os.packet);
  o.stream = sidx; o.slot = f.out_slot; o.tag = f.tag;
  o.is_keyframe = h->is_keyframe; o.n_keypoints = h->n;
  o.packet = os.packet;
  if (p->pc.want_rectified && h->is_keyframe) { o.rect_left = os.rectL; o.rect_right = os.rectR; }
  if (p->pc.checksum_outputs) {
    unsigned long long c = packet_checksum(p, os.packet);
    if (o.rect_left) c += sum64(os.rectL, p->img) + sum64(os.rectR, p->img);
    o.checksum = c;
  }
  {
    std::lock_guard<std::mutex> g(p->out_mu);
    p->outq.push_back(o);
  }
  p->out_cv.notify_one();
  p->n_done.fetch_add(1, std::memory_order_relaxed);
}

// device-visible address of a user image buffer: pinned host memory and device memory are read in
// place, pageable memory is staged through a pinned slot
static const unsigned char* resolve_src(kvfe_pipeline* p, PipeStream* s, int io_slot, int cam, const unsigned char* ptr,
                                        size_t pitch, size_t* out_pitch, bool force_stage = false) {
  cudaPointerAttributes a;
  cudaError_t e = cudaPointerGetAttributes(&a, ptr);
  if (e == cudaSuccess && (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged)) { *out_pitch = pitch; return ptr; }
  if (e == cudaSuccess && a.type == cudaMemoryTypeHost && a.devicePointer && !force_stage) {
    *out_pitch = pitch;
    return static_cast<const unsigned char*>(a.devicePointer);
  }
  if (e != cudaSuccess) cudaGetLastError();
  if (!s->stage[io_slot]) {
    if (cudaMallocHost((void**)&s->stage[io_slot], 2 * p->img) != cudaSuccess) return nullptr;
  }
  unsigned char* d = s->stage[io_slot] + (size_t)cam * p->img;
  if (pitch == (size_t)p->W) memcpy(d, ptr, p->img);
  else for (int y = 0; y < p->H; ++y) memcpy(d + (size_t)y * p->W, ptr + (size_t)y * pitch, p->W);
  if (cam == 0) p->n_staged.fetch_add(1, std::memory_order_relaxed);
  *out_pitch = p->W;
  return d;
}

// the same for a depth image (RGB-D): in place when the SMs can read it, else staged densely through a pinned slot
static const unsigned char* resolve_depth(kvfe_pipeline* p, PipeStream* s, int io_slot, const unsigned char* ptr, size_t pitch,
                                          size_t* out_pitch) {
  cudaPointerAttributes a;
  cudaError_t e = cudaPointerGetAttributes(&a, ptr);
  if (e == cudaSuccess && (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged)) { *out_pitch = pitch; return ptr; }
  if (e == cudaSuccess && a.type == cudaMemoryTypeHost && a.devicePointer) {
    *out_pitch = pitch;
    return static_cast<const unsigned char*>(a.devicePointer);
  }
  if (e != cudaSuccess) cudaGetLastError();
  const size_t rb = p->depth_row;
  if (!s->dstage[io_slot] && cudaMallocHost((void**)&s->dstage[io_slot], rb * p->H) != cudaSuccess) return nullptr;
  unsigned char* d = s->dstage[io_slot];
  if (pitch == rb) memcpy(d, ptr, rb * p->H);
  else for (int y = 0; y < p->H; ++y) memcpy(d + (size_t)y * rb, ptr + (size_t)y * pitch, rb);
  p->n_staged.fetch_add(1, std::memory_order_relaxed);
  *out_pitch = rb;
  return d;
}

// device-visible address of a buffer the SMs can read in place (device memory, or pinned mapped host memory); null otherwise
static const unsigned char* direct_src(const unsigned char* ptr) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, ptr) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  if (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) return ptr;
  if (a.type == cudaMemoryTypeHost && a.devicePointer) return static_cast<const unsigned char*>(a.devicePointer);
  return nullptr;
}

static void worker_main(kvfe_pipeline* p, int widx) {
  cudaSetDevice(p->device);
  std::vector<int> mine;
  for (int i = widx; i < (int)p->streams.size(); i += p->pc.n_workers) mine.push_back(i);
  const int depth = p->pc.max_in_flight;
  const bool split = p->split;
  int idle = 0;
  while (!p->stop.load(std::memory_order_acquire)) {
    bool progress = false;
    long long inflight_total = 0;
    for (int si : mine) {
      PipeStream* s = p->streams[si];
      kvfe_ctx* ctx = s->ctx;
      // completions, oldest first
      while (!s->fl.empty()) {
        const PipeFlight& f = s->fl.front();
        const StepIO* io = reinterpret_cast<const StepIO*>(ctx->pio[f.io_slot]);
        if (f.phase == 0 || io->done_seq != f.seq) break;
        std::atomic_thread_fence(std::memory_order_acquire);
        emit(p, si, s, f);
        s->fl.pop_front();
        progress = true;
      }
      // split graphs: the frame whose keyframe decision has arrived gets its second graph (at most one frame per
      // stream is in that phase, and it is the newest one)
      if (split && !s->fl.empty() && s->fl.back().phase == 0) {
        PipeFlight& f = s->fl.back();
        const StepIO* io = reinterpret_cast<const StepIO*>(ctx->pio[f.io_slot]);
        if (io->decided_seq == f.seq) {
          std::atomic_thread_fence(std::memory_order_acquire);
          const double t0 = now_s();
          const bool kf = io->decided_mode != 1;
          cudaError_t e = cudaGraphLaunch(kf ? ctx->pipe_graph_kf[f.io_slot] : ctx->pipe_graph_nokf[f.io_slot], ctx->stream);
          if (e != cudaSuccess) { pipe_fail(p, KVFE_ERR_CUDA, cudaGetErrorString(e)); break; }
          f.phase = 1;
          const long long nk = kf ? ctx->pipe_launches_kf : ctx->pipe_launches_nokf;
          ctx->launches += nk;
          p->n_graph.fetch_add(1, std::memory_order_relaxed);
          p->n_kernels.fetch_add(nk, std::memory_order_relaxed);
          p->launch_ns.fetch_add((long long)((now_s() - t0) * 1e9), std::memory_order_relaxed);
          progress = true;
        }
      }
      // launches (split graphs: not while the newest frame still waits for its second graph -- stream order)
      while ((int)s->fl.size() < depth && !(split && !s->fl.empty() && s->fl.back().phase == 0)) {
        PipeIn in, nxt; int oslot = -1;
        bool have_next = false;
        {
          std::lock_guard<std::mutex> g(s->mu);
          if (s->in.empty() || s->free_out.empty()) break;
          in = s->in.front(); s->in.pop_front();
          oslot = s->free_out.back(); s->free_out.pop_back();
          if (p->pc.prefetch != 0 && !s->in.empty()) { nxt = s->in.front(); have_next = true; }
        }
        const double t0 = now_s();
        const int io_slot = ctx->cur_slot;
        StepIO* io = reinterpret_cast<StepIO*>(ctx->pio[io_slot]);
        size_t pl = 0, pr = 0;
        const unsigned char* L = resolve_src(p, s, io_slot, 0, in.L, in.pitch, &pl);
        const unsigned char* R = resolve_src(p, s, io_slot, 1, in.R, in.pitch, &pr);
        if (L && R && pl != pr) {      // one side pageable (staged densely), the other pinned with a row pitch
          L = resolve_src(p, s, io_slot, 0, in.L, in.pitch, &pl, true);
          R = resolve_src(p, s, io_slot, 1, in.R, in.pitch, &pr, true);
        }
        if (!L || !R || pl != pr) { pipe_fail(p, KVFE_ERR_CUDA, "pipeline: cannot stage the input images"); break; }
        io->srcL = L; io->srcR = R; io->src_pitch = pl;
        io->srcD = nullptr; io->srcD_pitch = 0;
        if (p->rgbd) {
          size_t pd = 0;
          const unsigned char* D = resolve_depth(p, s, io_slot, in.D, in.dpitch, &pd);
          if (!D) { pipe_fail(p, KVFE_ERR_CUDA, "pipeline: cannot stage the depth image"); break; }
          io->srcD = D; io->srcD_pitch = pd;
        }
        io->next_srcL = nullptr; io->next_srcR = nullptr;
        if (have_next) {
          const unsigned char* nl = direct_src(nxt.L);
          const unsigned char* nr = direct_src(nxt.R);
          if (nl && nr && nxt.pitch == (size_t)p->W && ((((size_t)nl | (size_t)nr) | p->img) & 15) == 0) { io->next_srcL = nl; io->next_srcR = nr; }
        }
        io->dst_packets = s->out[oslot].packet;
        io->dst_rectL = p->pc.want_rectified ? s->out[oslot].rectL : nullptr;
        io->dst_rectR = p->pc.want_rectified ? s->out[oslot].rectR : nullptr;
        io->seq = ++s->seq;
        io->rot_mode = p->pc.rotation_mode;
        io->force_kf = in.force_kf;
        unsigned char* arr = ctx->pio[io_slot] + KVFE_STEPIO_ARRAYS;
        memcpy(arr, &in.ts, sizeof(long long));
        memcpy(arr + sizeof(long long), in.Rm, 9 * sizeof(double));
        std::atomic_thread_fence(std::memory_order_release);
        cudaError_t e = cudaGraphLaunch(split ? ctx->pipe_graph_a[io_slot] : ctx->pipe_graph[io_slot], ctx->stream);
        if (e != cudaSuccess) { pipe_fail(p, KVFE_ERR_CUDA, cudaGetErrorString(e)); break; }
        ctx->cur_slot ^= 1;
        const long long nl = split ? ctx->pipe_launches_a : ctx->pipe_graph_launches;
        ctx->launches += nl;
        s->fl.push_back(PipeFlight{oslot, io_slot, s->seq, in.tag, split ? 0 : 1});
        p->n_graph.fetch_add(1, std::memory_order_relaxed);
        p->n_kernels.fetch_add(nl, std::memory_order_relaxed);
        p->launch_ns.fetch_add((long long)((now_s() - t0) * 1e9), std::memory_order_relaxed);
        progress = true;
      }
      inflight_total += (long long)s->fl.size();
    }
    if (progress) { idle = 0; continue; }
    ++idle;
    if (inflight_total > 0) {
      // work is running on the GPU: poll the mapped sequence numbers, politely
      if (idle > 64) sched_yield();
    } else {
      // nothing in flight and nothing launchable: sleep until a push or a release wakes us
      std::unique_lock<std::mutex> lk(p->wk_mu);
      p->wk_cv.wait_for(lk, std::chrono::microseconds(200));
      idle = 0;
    }
  }
}

extern "C" const char* kvfe_pipeline_last_error(const kvfe_pipeline* p) { return p ? p->err : g_pipe_create_err; }
extern "C" size_t kvfe_pipeline_packet_bytes(const kvfe_pipeline* p) { return p ? p->packet_bytes : 0; }
extern "C" int kvfe_pipeline_max_keypoints(const kvfe_pipeline* p) { return p ? p->cap : 0; }
extern "C" int kvfe_pipeline_packet_offsets(const kvfe_pipeline* p, size_t* offsets, int max_entries) {
  if (!p || !offsets) return KVFE_ERR_INVALID_ARG;
  const int n = max_entries < KVFE_PACKET_ARRAYS ? max_entries : KVFE_PACKET_ARRAYS;
  for (int i = 0; i < n; ++i) offsets[i] = p->pk_off[i];
  return n;
}

extern "C" void kvfe_pipeline_destroy(kvfe_pipeline* p) {
  if (!p) return;
  p->stop.store(true, std::memory_order_release);
  p->wk_cv.notify_all();
  for (std::thread& t : p->workers) if (t.joinable()) t.join();
  for (PipeStream* s : p->streams) {
    if (!s) continue;
    if (s->ctx) { cudaStreamSynchronize(s->ctx->stream); kvfe_destroy(s->ctx); }
    if (s->out_block) cudaFreeHost(s->out_block);
    for (int i = 0; i < 2; ++i) if (s->stage[i]) cudaFreeHost(s->stage[i]);
    for (int i = 0; i < 2; ++i) if (s->dstage[i]) cudaFreeHost(s->dstage[i]);
    delete s;
  }
  delete p;
}

extern "C" int kvfe_pipeline_create(const kvfe_config* cfg, const kvfe_rig* rig, const kvfe_pipeline_config* pc,
                                    kvfe_pipeline** out) {
  if (!cfg || !rig || !pc || !out) return pipe_fail(nullptr, KVFE_ERR_INVALID_ARG, "null argument");
  *out = nullptr;
  if (pc->n_streams < 1 || pc->n_streams > 4096) return pipe_fail(nullptr, KVFE_ERR_INVALID_ARG, "n_streams out of range");
  if (pc->rotation_mode != 0 && pc->rotation_mode != 1) return pipe_fail(nullptr, KVFE_ERR_INVALID_ARG, "rotation_mode must be 0 or 1");
  kvfe_pipeline* p = new kvfe_pipeline();
  p->pc = *pc;
  if (p->pc.n_workers <= 0) p->pc.n_workers = pc->n_streams >= 16 ? 4 : (pc->n_streams >= 4 ? 2 : 1);
  if (p->pc.n_workers > pc->n_streams) p->pc.n_workers = pc->n_streams;
  if (p->pc.queue_depth <= 0) p->pc.queue_depth = 4;
  if (p->pc.output_slots < 2) p->pc.output_slots = 4;
  if (p->pc.max_in_flight <= 0 || p->pc.max_in_flight > 2) p->pc.max_in_flight = 2;
  // opt-in: measured SLOWER on B200 with 32 streams (device-resident 0.63 -> 0.75 ms per pass, host buffers 0.81 ->
  // 0.87): a step graph with a parallel branch costs twice the launch time on the host and the branches of 32
  // graphs compete for the 32 hardware work queues; the overlap across streams already hides the transfer
  p->pc.prefetch = pc->prefetch > 0 ? 1 : 0;
  p->rgbd = cfg->frontend_type == 2;
  if (p->rgbd) {
    p->pc.prefetch = 0;            // the prefetch branch pulls the two 8-bit images of the next frame, not a depth image
    p->pc.want_rectified = 0;      // no rectified pair: outputs carry null rect_left / rect_right
    p->depth_row = (size_t)cfg->width * (cfg->depth.depth_type == KVFE_DEPTH_F32 ? 4 : 2);
  }
  {
    // KVFE_PIPE_SPLIT=0/1 overrides (diagnostic); the prefetch branch lives in the single-graph variant only
    const char* e = getenv("KVFE_PIPE_SPLIT");
    p->split = e ? (e[0] == '1') : (pc->split_graphs >= 0);      // library default: on (measured below)
    if (p->pc.prefetch) p->split = false;
  }
  p->W = cfg->width; p->H = cfg->height; p->img = (size_t)cfg->width * cfg->height;
  kvfe_config c1 = *cfg;
  c1.batch = 1;
  for (int i = 0; i < pc->n_streams; ++i) {
    PipeStream* s = new PipeStream();
    p->streams.push_back(s);
    int rc = kvfe_create(&c1, rig, &s->ctx);
    if (rc != KVFE_OK) {
      pipe_fail(nullptr, rc, kvfe_last_error(nullptr));
      kvfe_pipeline_destroy(p);
      return rc;
    }
    if (p->pc.prefetch != 0) {
      // staging of the next frame's images (two slots, like the pyramid) + the fork stream / events of the capture
      kvfe_ctx* c = s->ctx;
      bool ok = true;
      for (int k = 0; k < 2 && ok; ++k) ok = cudaMalloc((void**)&c->db.stage_img[k], 2 * (size_t)c->dc.B * c->dc.img_stride) == cudaSuccess;
      ok = ok && cudaMalloc((void**)&c->db.stage_seq, 2 * sizeof(unsigned long long)) == cudaSuccess;
      ok = ok && cudaMemset(c->db.stage_seq, 0, 2 * sizeof(unsigned long long)) == cudaSuccess;
      ok = ok && cudaStreamCreateWithFlags(&c->side, cudaStreamNonBlocking) == cudaSuccess;
      ok = ok && cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming) == cudaSuccess;
      ok = ok && cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming) == cudaSuccess;
      if (!ok) {
        pipe_fail(nullptr, KVFE_ERR_CUDA, "pipeline: prefetch staging allocation failed");
        kvfe_pipeline_destroy(p);
        return KVFE_ERR_CUDA;
      }
    }
    for (int slot = 1; slot >= 0; --slot) {      // slot 0 last: cur_slot ends at 0
      rc = p->split ? build_split_graphs(s->ctx, slot) : build_pipe_graph(s->ctx, slot);
      if (rc != KVFE_OK) {
        pipe_fail(nullptr, rc, kvfe_last_error(s->ctx));
        kvfe_pipeline_destroy(p);
        return rc;
      }
    }
    s->ctx->cur_slot = 0;
    if (i == 0) {
      p->device = s->ctx->device;
      p->packet_bytes = s->ctx->db.packet_bytes;
      p->cap = s->ctx->dc.cap;
      for (int k = 0; k < KVFE_PACKET_ARRAYS; ++k) p->pk_off[k] = s->ctx->db.pk_off[k];
    }
    const size_t pkb = (p->packet_bytes + 255) & ~(size_t)255, imb = (p->img + 255) & ~(size_t)255;
    const size_t per = pkb + (p->pc.want_rectified ? 2 * imb : 0);
    if (cudaMallocHost((void**)&s->out_block, per * p->pc.output_slots) != cudaSuccess) {
      pipe_fail(nullptr, KVFE_ERR_CUDA, "pipeline: pinned output allocation failed");
      kvfe_pipeline_destroy(p);
      return KVFE_ERR_CUDA;
    }
    memset(s->out_block, 0, per * p->pc.output_slots);
    for (int k = 0; k < p->pc.output_slots; ++k) {
      unsigned char* b = s->out_block + (size_t)k * per;
      s->out.push_back(PipeOutSlot{b, p->pc.want_rectified ? b + pkb : nullptr, p->pc.want_rectified ? b + pkb + imb : nullptr});
      s->free_out.push_back(k);
    }
  }
  for (int w = 0; w < p->pc.n_workers; ++w) p->workers.emplace_back(worker_main, p, w);
  *out = p;
  return KVFE_OK;
}

static int push_one(kvfe_pipeline* p, int stream, const uint8_t* left, const uint8_t* right, size_t pitch,
                    int64_t timestamp, const double* R, uint64_t tag, bool notify, const void* depth = nullptr,
                    size_t depth_pitch = 0) {
  if (p && !right && !p->streams.empty() && p->streams[0]->ctx->dc.mono) right = left;      // mono front-end: no right camera
  if (!p || !left || !right || !R) return KVFE_ERR_INVALID_ARG;
  if (p->rgbd != (depth != nullptr))        // wrong entry point for the front-end: refused, the pipeline stays usable
    return pipe_refuse(p, p->rgbd ? "push: an RGB-D pipeline (frontend_type 2) takes kvfe_pipeline_push_rgbd"
                                                      : "push_rgbd: not an RGB-D pipeline (frontend_type 2)");
  if (stream < 0 || stream >= (int)p->streams.size() || pitch < (size_t)p->W) return pipe_fail(p, KVFE_ERR_INVALID_ARG, "push: bad stream or pitch");
  if (depth && depth_pitch < p->depth_row) return pipe_refuse(p, "push_rgbd: depth pitch smaller than a row");
  if (int f = p->failed.load()) return f;
  PipeStream* s = p->streams[stream];
  PipeIn in;
  in.L = left; in.R = right; in.pitch = pitch; in.ts = timestamp; in.tag = tag; in.force_kf = 0;
  in.D = static_cast<const unsigned char*>(depth); in.dpitch = depth_pitch;
  memcpy(in.Rm, R, sizeof(in.Rm));
  {
    std::lock_guard<std::mutex> g(s->mu);
    if ((int)s->in.size() >= p->pc.queue_depth) return KVFE_ERR_CAPACITY;
    in.force_kf = s->force_next ? 1 : 0;
    s->force_next = false;
    s->in.push_back(in);
  }
  p->n_pushed.fetch_add(1, std::memory_order_relaxed);
  if (notify) p->wk_cv.notify_all();
  return KVFE_OK;
}

extern "C" int kvfe_pipeline_push(kvfe_pipeline* p, int stream, const uint8_t* left, const uint8_t* right, size_t pitch,
                                  int64_t timestamp, const double* R, uint64_t tag) {
  return push_one(p, stream, left, right, pitch, timestamp, R, tag, true);
}

// RGB-D: the intensity image stands in for the (absent) right image, like the mono front-end's
extern "C" int kvfe_pipeline_push_rgbd(kvfe_pipeline* p, int stream, const uint8_t* img, size_t pitch, const void* depth,
                                       size_t depth_pitch_bytes, int64_t timestamp, const double* R, uint64_t tag) {
  if (!p || !img || !depth || !R) return KVFE_ERR_INVALID_ARG;
  return push_one(p, stream, img, img, pitch, timestamp, R, tag, true, depth, depth_pitch_bytes);
}

extern "C" int kvfe_pipeline_push_many(kvfe_pipeline* p, int n, const int32_t* streams, const uint8_t* const* left,
                                       const uint8_t* const* right, size_t pitch, const int64_t* timestamps,
                                       const double* R, const uint64_t* tags) {
  if (!p || n < 0 || !streams || !left || !right || !timestamps || !R) return KVFE_ERR_INVALID_ARG;
  int i = 0;
  for (; i < n; ++i) {
    int rc = push_one(p, streams[i], left[i], right[i], pitch, timestamps[i], R + 9 * (size_t)i, tags ? tags[i] : 0, (i & 63) == 0);
    if (rc == KVFE_ERR_CAPACITY) break;
    if (rc != KVFE_OK) { p->wk_cv.notify_all(); return rc; }
  }
  p->wk_cv.notify_all();
  return i;
}

// Frame::isKeyframe_ (user-enforced keyframe, VisionImuFrontend.cpp:207-209) for the NEXT frame pushed on `stream`
extern "C" int kvfe_pipeline_force_keyframe(kvfe_pipeline* p, int stream) {
  if (!p || stream < 0 || stream >= (int)p->streams.size()) return KVFE_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> g(p->streams[stream]->mu);
  p->streams[stream]->force_next = true;
  return KVFE_OK;
}

extern "C" int kvfe_pipeline_pop(kvfe_pipeline* p, kvfe_pipeline_output* outs, int max_n, int timeout_ms) {
  if (!p || !outs || max_n < 1) return KVFE_ERR_INVALID_ARG;
  std::unique_lock<std::mutex> lk(p->out_mu);
  if (p->outq.empty() && timeout_ms > 0) {
    const auto deadline = std::chrono::steady_clock::now() + std::chrono::milliseconds(timeout_ms);
    while (p->outq.empty() && !p->failed.load()) {
      if (p->out_cv.wait_until(lk, deadline) == std::cv_status::timeout) break;
    }
  }
  if (p->outq.empty()) { int f = p->failed.load(); return f ? f : 0; }
  int n = 0;
  while (n < max_n && !p->outq.empty()) { outs[n++] = p->outq.front(); p->outq.pop_front(); }
  return n;
}

extern "C" int kvfe_pipeline_release(kvfe_pipeline* p, const kvfe_pipeline_output* outs, int n) {
  if (!p || (!outs && n > 0)) return KVFE_ERR_INVALID_ARG;
  for (int i = 0; i < n; ++i) {
    const int si = outs[i].stream;
    if (si < 0 || si >= (int)p->streams.size()) return pipe_fail(p, KVFE_ERR_INVALID_ARG, "release: bad stream");
    PipeStream* s = p->streams[si];
    if (outs[i].slot < 0 || outs[i].slot >= (int)s->out.size()) return pipe_fail(p, KVFE_ERR_INVALID_ARG, "release: bad slot");
    std::lock_guard<std::mutex> g(s->mu);
    s->free_out.push_back(outs[i].slot);
  }
  p->wk_cv.notify_all();
  return KVFE_OK;
}

extern "C" int kvfe_pipeline_reset(kvfe_pipeline* p) {
  if (!p) return KVFE_ERR_INVALID_ARG;
  if (p->n_pushed.load() != p->n_done.load()) return pipe_fail(p, KVFE_ERR_STATE, "reset: frames still in flight");
  {
    std::lock_guard<std::mutex> g(p->out_mu);
    if (!p->outq.empty()) return pipe_fail(p, KVFE_ERR_STATE, "reset: outputs not popped");
  }
  // the dispatchers touch a context only when its input queue is non-empty; every queue is empty here
  for (PipeStream* s : p->streams) {
    cudaStreamSynchronize(s->ctx->stream);
    const int slot = s->ctx->cur_slot;
    int rc = kvfe_frontend_reset(s->ctx);
    if (rc != KVFE_OK) return pipe_fail(p, rc, kvfe_last_error(s->ctx));
    s->ctx->cur_slot = slot;      // the graphs are tied to the pyramid slots, not to the frame count
  }
  return KVFE_OK;
}

extern "C" int kvfe_pipeline_get_stats(kvfe_pipeline* p, kvfe_pipeline_stats* st) {
  if (!p || !st) return KVFE_ERR_INVALID_ARG;
  st->frames_pushed = p->n_pushed.load(); st->frames_done = p->n_done.load();
  st->graph_launches = p->n_graph.load(); st->kernel_launches = p->n_kernels.load();
  st->launch_seconds = 1e-9 * (double)p->launch_ns.load();
  st->staged_copies = p->n_staged.load();
  return KVFE_OK;
}
